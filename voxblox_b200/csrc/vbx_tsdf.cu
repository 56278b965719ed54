// TSDF integration on the device: the Simple / Merged / Fast integrators of
// voxblox/src/integrator/tsdf_integrator.cc re-designed as a data-parallel pipeline.
//
//   k_point_keys     transform + validate every point, key it by its end voxel
//                    (bundleRays, cc:340-371)
//   sort             stable radix sort of the point keys: bundles become runs, in the
//                    reference's point order inside a run
//   k_heads          dense list of bundle heads
//   k_merge          one WARP per bundle: 32 members prefetched per step, the
//                    reference's sequential weighted mean (integrateVoxel cc:387-405)
//                    evaluated in order on the prefetched registers
//   k_rays_count     one thread per ray: DDA walk (RayCaster) that creates missing
//                    blocks in the device hash and counts the voxels it will update
//                    (allocateStorageAndGetVoxelPtr cc:91-134)
//   scan + k_assign  offsets of every ray's update records; pool slots for new blocks
//   k_rays_emit      second DDA walk writing (voxel id, ray id) records
//   sort             stable radix sort by voxel id: every voxel's updates become one
//                    run, ordered by ray rank
//   k_apply_short /  updateTsdfVoxel (cc:150-209) applied sequentially per voxel --
//   k_apply_long     clamp-after-every-update semantics preserved exactly, with no
//                    locks and no atomics on voxels.  Runs longer than 32 updates
//                    (free space near the sensor) continue in a warp-per-run kernel.
//
// Update order.  The reference applies a voxel's updates in whatever order its
// threads reach the voxel's mutex (cc:186); with one thread that is point order for
// Simple / Fast and unordered_map iteration order for Merged.  The device applies
// them in ray-rank order, and the rank IS the reference's one-thread order: point
// order (integration_order_mode) for Simple / Fast; for Merged the iteration order
// of the reference's libstdc++ unordered_map (k_bundle_order, vbx_order.cuh), normal
// bundles before clearing bundles (cc:323-335).  See DESIGN.md "update order".
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <unordered_map>  // std::__detail::_Prime_rehash_policy: the growth schedule the reference's map follows

#include <cooperative_groups.h>

#include "vbx_engine.h"
#include "vbx_hash.cuh"
#include "vbx_sort.cuh"
#include "vbx_order.cuh"

namespace cg = cooperative_groups;

namespace vbx {

constexpr int kShortRun = 32;  // updates a single thread applies before handing the run to a warp

struct ScanParams {
  Pose T;
  F3 origin;
  float voxel_size, voxel_size_inv;
  float trunc, min_ray, max_ray;
  UpdateParams up;
  int L;  // log2(voxels per side)
  int kind;
  int freespace, use_const_weight, allow_clear, carving, anti_grazing;
  int order_mode;      // 0 mixed, 1 sorted (order array)
  uint32_t n;          // points in the cloud
  uint32_t n_groups;   // n / 1024 (MixedThreadSafeIndex)
  float start_inv;     // start_voxel_subsampling_factor * voxel_size_inv
  int max_collisions;
  uint32_t set_epoch;  // generation tag of the Fast integrator's approximate sets
  uint32_t epoch;      // call id
  uint64_t max_updates;
  // block-ownership sharding (multi-GPU, one map over the GPUs of a box): this rank applies the
  // updates of the voxels in blocks it owns (block_owner() == own_rank) and creates only those
  // blocks; everything before the apply is identical on all ranks
  int own_world, own_rank;
  // the number of voxels a ray updates is known from its DDA set-up alone (no anti-grazing, not the
  // Fast integrator): one walk that creates blocks AND writes the update records
  int single_walk;
  // a call whose update records do not fit max_updates_per_pass is emitted and applied in several
  // passes over contiguous ray-slot ranges [emit_lo, emit_hi); emit_base = off[emit_lo]
  uint32_t emit_lo, emit_hi, emit_base;
};

// MixedThreadSafeIndex::getNextIndexImpl, integrator_utils.cc:54-63
__device__ __forceinline__ uint32_t point_order(const ScanParams& P, const uint32_t* order, uint32_t s) {
  if (P.order_mode == 1) return order[s];
  if (P.n_groups * 1024u <= s) return s;
  return (s % P.n_groups) * 1024u + s / P.n_groups;
}

__device__ __forceinline__ F3 load_point(const float* xyz, uint32_t idx) {
  return f3(__ldg(xyz + 3 * idx), __ldg(xyz + 3 * idx + 1), __ldg(xyz + 3 * idx + 2));
}
__device__ __forceinline__ uint32_t load_color(const uint8_t* rgba, uint32_t idx) {
  return __ldg(reinterpret_cast<const uint32_t*>(rgba) + idx);
}

// ------------------------------------------------------- block ownership (multi-GPU)
// One map over the GPUs of a box: rank r owns the blocks with block_owner() == r -- a 2 x 2 x 2
// brick pattern for 8 ranks, so the blocks around the sensor (where most updates land) spread
// over all ranks.  See DESIGN.md "multi-GPU".
__device__ __forceinline__ bool owns_block(const ScanParams& P, int bx, int by, int bz) {
  return P.own_world <= 1 || block_owner(bx, by, bz, P.own_world) == P.own_rank;
}
// An update record's key: (touched id of the block in this call, voxel inside the block) -- e.g.
// 6 + 12 bits when a scan touches ~50 blocks, so the record sort runs three 8-bit passes whatever
// the size of the map.  Records of blocks another rank owns keep their place in the ray's record
// range (offsets are fixed before the walk) under the key 0xffffffff, which sorts behind every
// real key and is skipped by the apply.
constexpr uint32_t kNotOwned = 0xfffffffeu;
constexpr uint32_t kSkipRecord = 0xffffffffu;
__device__ __forceinline__ uint32_t record_key(uint32_t touched_id, uint32_t lin, int L) {
  return touched_id >= kNotOwned ? kSkipRecord : ((touched_id << (3 * L)) | lin);
}

// ------------------------------------------------------------------ bundle keys
// key = [clearing | z | y | x] with the voxel coordinates taken relative to the bounding box of
// the scan's valid points' voxels (k_point_bounds), each axis in exactly the bits its extent
// needs.  Any scan fits 64 bits (|voxel coordinate| < 2^20: at most 21 bits per axis + 1), a
// 640 x 480 room scan needs ~22 -- and the sort only runs the radix passes those bits span.
// Ascending key order = (clearing, z, y, x).
constexpr uint32_t kBoundBias = 1u << 30;
struct KeyLayout {
  int minx, miny, minz;
  int bx, by, bz;  // bits per axis
  bool any;        // the scan has at least one valid point
};
__device__ __forceinline__ int bits_of(uint32_t extent) { return 32 - __clz(extent); }
__device__ __forceinline__ KeyLayout key_layout(const ScanState* st) {
  KeyLayout k;
  const uint32_t mx = st->kb_max[0];
  k.any = mx != 0u;
  k.minx = (int)(0xffffffffu - st->kb_min[0] - kBoundBias);
  k.miny = (int)(0xffffffffu - st->kb_min[1] - kBoundBias);
  k.minz = (int)(0xffffffffu - st->kb_min[2] - kBoundBias);
  k.bx = k.any ? bits_of((uint32_t)((int)(mx - kBoundBias) - k.minx)) : 0;
  k.by = k.any ? bits_of((uint32_t)((int)(st->kb_max[1] - kBoundBias) - k.miny)) : 0;
  k.bz = k.any ? bits_of((uint32_t)((int)(st->kb_max[2] - kBoundBias) - k.minz)) : 0;
  return k;
}
__device__ __forceinline__ uint64_t make_point_key(const KeyLayout& k, I3 v, bool clearing, bool* in_range) {
  const int rx = v.x - k.minx, ry = v.y - k.miny, rz = v.z - k.minz;
  *in_range = k.any && rx >= 0 && ry >= 0 && rz >= 0 && (rx >> k.bx) == 0 && (ry >> k.by) == 0 && (rz >> k.bz) == 0;
  return (uint64_t)(uint32_t)rx | ((uint64_t)(uint32_t)ry << k.bx) | ((uint64_t)(uint32_t)rz << (k.bx + k.by)) |
         ((uint64_t)clearing << (k.bx + k.by + k.bz));
}
// the key a NORMAL bundle ending in voxel v would have (anti-grazing lookup)
__device__ __forceinline__ uint64_t normal_key_of(const KeyLayout& k, int x, int y, int z, bool* in_range) {
  return make_point_key(k, i3(x, y, z), false, in_range);
}
__device__ __forceinline__ bool key_is_clearing(const KeyLayout& k, uint64_t key) {
  return ((key >> (k.bx + k.by + k.bz)) & 1ull) != 0;
}
// the voxel a bundle key stands for
__device__ __forceinline__ I3 key_voxel(const KeyLayout& k, uint64_t key) {
  return i3((int)(key & ((1ull << k.bx) - 1ull)) + k.minx, (int)((key >> k.bx) & ((1ull << k.by) - 1ull)) + k.miny,
            (int)((key >> (k.bx + k.by)) & ((1ull << k.bz) - 1ull)) + k.minz);
}

// ------------------------------------------------------------------- kernels
// Merged, pass 1 over the cloud: the bounding box of the valid points' voxels (and their count).
// Grid-stride over the points, one set of atomics per thread block.
__global__ void __launch_bounds__(256)
k_point_bounds(ScanParams P, const float* __restrict__ xyz, uint32_t* __restrict__ first_bits, SortPlan* plan,
               uint32_t* __restrict__ scan_status, uint32_t scan_words, ScanState* st) {
  __shared__ uint32_t s_red[7];
  if (threadIdx.x < 7) s_red[threadIdx.x] = 0u;
  const uint32_t words2 = 2u * ((P.n + 31u) >> 5);
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < words2; w += gridDim.x * blockDim.x) {
    first_bits[w] = 0u;  // the first-occurrence bitmaps k_heads fills
  }
  // (the first kernel of the front half also clears what later kernels of its lane count in: the point sort's
  // plan and the status words of the offset scan)
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < (uint32_t)(sizeof(SortPlan) / 4); w += gridDim.x * blockDim.x) {
    reinterpret_cast<uint32_t*>(plan)[w] = 0u;
  }
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < scan_words; w += gridDim.x * blockDim.x) scan_status[w] = 0u;
  __syncthreads();
  // both ends encoded so that the zero-initialised status block means "empty" and atomicMax serves both
  uint32_t hi_x = 0, hi_y = 0, hi_z = 0, lo_x = 0, lo_y = 0, lo_z = 0, n_valid = 0;
  const int lim = kCoordBias - 1;
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < P.n; s += gridDim.x * blockDim.x) {
    const F3 p = load_point(xyz, s);  // (the bounding box does not depend on the point order)
    if (classify_point(p, P.min_ray, P.max_ray, P.allow_clear != 0, P.freespace != 0) == 0) continue;
    const I3 v = grid_index(transform(P.T, p), P.voxel_size_inv);
    if (v.x < -lim || v.x > lim || v.y < -lim || v.y > lim || v.z < -lim || v.z > lim) {
      atomicOr(&st->error, kErrCoordRange);
      continue;
    }
    ++n_valid;
    hi_x = max(hi_x, (uint32_t)v.x + kBoundBias);
    hi_y = max(hi_y, (uint32_t)v.y + kBoundBias);
    hi_z = max(hi_z, (uint32_t)v.z + kBoundBias);
    lo_x = max(lo_x, 0xffffffffu - ((uint32_t)v.x + kBoundBias));
    lo_y = max(lo_y, 0xffffffffu - ((uint32_t)v.y + kBoundBias));
    lo_z = max(lo_z, 0xffffffffu - ((uint32_t)v.z + kBoundBias));
  }
  hi_x = __reduce_max_sync(0xffffffffu, hi_x);
  hi_y = __reduce_max_sync(0xffffffffu, hi_y);
  hi_z = __reduce_max_sync(0xffffffffu, hi_z);
  lo_x = __reduce_max_sync(0xffffffffu, lo_x);
  lo_y = __reduce_max_sync(0xffffffffu, lo_y);
  lo_z = __reduce_max_sync(0xffffffffu, lo_z);
  n_valid = __reduce_add_sync(0xffffffffu, n_valid);
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&s_red[0], hi_x);
    atomicMax(&s_red[1], hi_y);
    atomicMax(&s_red[2], hi_z);
    atomicMax(&s_red[3], lo_x);
    atomicMax(&s_red[4], lo_y);
    atomicMax(&s_red[5], lo_z);
    atomicAdd(&s_red[6], n_valid);
  }
  __syncthreads();
  if (threadIdx.x < 3 && s_red[threadIdx.x]) atomicMax(&st->kb_max[threadIdx.x], s_red[threadIdx.x]);
  if (threadIdx.x >= 3 && threadIdx.x < 6 && s_red[threadIdx.x]) atomicMax(&st->kb_min[threadIdx.x - 3], s_red[threadIdx.x]);
  if (threadIdx.x == 6 && s_red[6]) atomicAdd(&st->n_valid_points, s_red[6]);
}

// Merged, pass 2: key every point by its end voxel (bundleRays, cc:340-371), in the reference's
// point order (position s of that order holds point point_order(s)).
template <typename KeyT>
__global__ void k_point_keys(ScanParams P, const float* __restrict__ xyz, const uint32_t* __restrict__ order,
                             KeyT* __restrict__ keys, uint32_t* __restrict__ vals, ScanState* st) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  const KeyLayout kl = key_layout(st);
  if (s == 0) st->key_bits = (uint32_t)(kl.bx + kl.by + kl.bz + 1);
  if (s < P.n) {
    const uint32_t idx = point_order(P, order, s);
    const F3 p = load_point(xyz, idx);
    const int cls = classify_point(p, P.min_ray, P.max_ray, P.allow_clear != 0, P.freespace != 0);
    KeyT key = (KeyT)~(KeyT)0;
    if (cls != 0) {
      const I3 v = grid_index(transform(P.T, p), P.voxel_size_inv);
      bool in_range;
      const uint64_t k = make_point_key(kl, v, cls == 2, &in_range);
      if (in_range) key = (KeyT)k;  // (out of range only beyond +-2^20 voxels: flagged by k_point_bounds)
    }
    keys[s] = key;
    vals[s] = idx;
  }
}

// "sorted" integration order: key = |p|^2 (float, widened to double like
// SortedThreadSafeIndex, integrator_utils.cc:24-37); non-negative doubles order as integers.
__global__ void k_sqnorm_keys(uint32_t n, const float* __restrict__ xyz, uint64_t* __restrict__ keys,
                              uint32_t* __restrict__ vals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const F3 p = load_point(xyz, i);
  const double d = (double)dot3(p, p);
  keys[i] = (uint64_t)__double_as_longlong(d);
  vals[i] = i;
}

// point index -> its position in the reference's point order (the inverse of point_order)
__device__ __forceinline__ uint32_t point_order_inv(const ScanParams& P, const uint32_t* order_inv, uint32_t idx) {
  if (P.order_mode == 1) return order_inv[idx];
  if (P.n_groups * 1024u <= idx) return idx;
  return (idx % 1024u) * P.n_groups + idx / 1024u;
}
__global__ void k_invert_order(uint32_t n, const uint32_t* __restrict__ order, uint32_t* __restrict__ order_inv) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n) order_inv[order[s]] = s;
}

// A bundle's id is its position j in head_list (unordered, dense): the per-ray tables (ray_p / ray_a /
// ray_c / cnt) are indexed by j, update records carry j, and ray_list[rank] = j gives the order.
constexpr uint32_t kBigBundle = 256;         // members from which a bundle is folded before the others
constexpr uint32_t kHeadBig = 0x80000000u;   // head_list entry: sorted position of the head | this flag

// Dense (unordered) list of bundle heads, and the first-occurrence bitmaps: bit t of map m
// (0 normal, 1 clearing) is set when the point at position t of the reference's point order is the
// first of its bundle, i.e. the point whose operator[] inserts the bundle's key into the reference's
// voxel_map / clear_map (bundleRays, cc:340-371).  k_bundle_order turns them into the maps'
// iteration order.
template <typename KeyT>
__global__ void k_heads(ScanParams P, const KeyT* __restrict__ keys, const uint32_t* __restrict__ vals,
                        const uint32_t* __restrict__ order_inv, uint32_t* __restrict__ head_list,
                        uint32_t* __restrict__ big_list, uint32_t* __restrict__ first_bits, uint32_t* __restrict__ cnt,
                        ScanState* st) {
  const uint32_t n = P.n;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const KeyLayout kl = key_layout(st);
  bool head = false;
  if (i <= n) cnt[i] = 0;
  if (i < n) {
    const KeyT key = keys[i];
    head = key != (KeyT)~(KeyT)0 && (i == 0 || keys[i - 1] != key);
    if (head) {
      // the stable sort keeps point order inside a bundle: its first member is its first occurrence
      const uint32_t t0 = point_order_inv(P, order_inv, vals[i]);
      const uint32_t words = (n + 31u) >> 5;
      atomicOr(first_bits + (key_is_clearing(kl, (uint64_t)key) ? words : 0u) + (t0 >> 5), 1u << (t0 & 31u));
    }
  }
  const unsigned b = __ballot_sync(0xffffffffu, head);
  if (b) {
    const int lane = threadIdx.x & 31;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(&st->n_ray_list, (uint32_t)__popc(b));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (head) {
      // the fold of a bundle is one dependent chain: the long ones are started first (k_merge)
      const bool big = i + kBigBundle < n && keys[i + kBigBundle] == keys[i];
      const uint32_t j = base + __popc(b & ((1u << lane) - 1u));
      head_list[j] = i | (big ? kHeadBig : 0u);
      if (big) big_list[atomicAdd(&st->n_big, 1u)] = j;
    }
  }
}

// LongIndexHash, core/block_hash.h:52-64 (32-bit wrap of x + 17191 y + 17191^2 z)
__device__ __forceinline__ uint32_t long_index_hash(int x, int y, int z) {
  return (uint32_t)x + (uint32_t)y * 17191u + (uint32_t)z * 295530481u;
}
// ---- The reference's bundle order (vbx_order.cuh) in three kernels:
//   k_order_prefix  per-word popcount prefixes of the two first-occurrence bitmaps (one thread block);
//                   the bundle counts B0 (normal map) and B1 (clearing map)
//   k_order_heads   one thread per bundle: its insertion index e into the reference's map (= number of
//                   earlier first occurrences), LongIndexHash of its voxel -> h[map][e], head_of[map][e]
//   k_bundle_order  the iteration order of each map; writes ray_list[rank] = bundle id.  Ranks are
//                   dense: normal bundles 0 .. B0-1 in voxel_map's iteration order, clearing bundles
//                   B0 .. B0+B1-1 in clear_map's (integrateRays(false) runs before integrateRays(true),
//                   cc:323-335).  When a map's tables fit shared memory (16-bit tables: up to ~18 k
//                   bundles; 640 x 480 scans have a few thousand) one block does everything alone -- an
//                   ordinary one-block launch when recent scans say so, see launch_bundle_order; larger
//                   maps (LiDAR: ~50 k bundles) run their late rehash stages grid-wide on global tables
//                   (cooperative launch), the early (small) stages still in block 0's shared memory.
// The clearing map's arrays follow the normal map's at offset g.cap.
__global__ void __launch_bounds__(kOrderThreads)
k_order_prefix(uint32_t n, const uint32_t* __restrict__ first_bits, OrderScratch g, ScanState* st) {
  __shared__ uint32_t warp_sums[33];
  const uint32_t tid = threadIdx.x;
  const uint32_t words = (n + 31u) >> 5;
  const uint32_t per = (words + kOrderThreads - 1) / kOrderThreads;
  const uint32_t lo = min(tid * per, words), hi = min(lo + per, words);
  for (int mp = 0; mp < 2; ++mp) {
    const uint32_t* bits = first_bits + (mp ? words : 0u);
    uint32_t* wp = g.wp + (mp ? words : 0u);
    uint32_t sum = 0;
    for (uint32_t w = lo; w < hi; ++w) sum += (uint32_t)__popc(bits[w]);  // (independent loads: all in flight together)
    uint32_t total;
    uint32_t run = order_block_scan(sum, warp_sums, &total);
    for (uint32_t w = lo; w < hi; ++w) {
      wp[w] = run;
      run += (uint32_t)__popc(bits[w]);
    }
    if (tid == 0) {
      if (mp == 0) st->n_rays = total; else st->n_clear_rays = total;
    }
  }
}

template <typename KeyT>
__global__ void k_order_heads(ScanParams P, const KeyT* __restrict__ keys, const uint32_t* __restrict__ vals,
                              const uint32_t* __restrict__ order_inv, const uint32_t* __restrict__ head_list,
                              const uint32_t* __restrict__ first_bits, OrderScratch g, const ScanState* st) {
  const uint32_t words = (P.n + 31u) >> 5;
  const uint32_t n_heads = st->n_ray_list;
  const KeyLayout kl = key_layout(st);
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_heads; j += gridDim.x * blockDim.x) {
    const uint32_t i = head_list[j] & ~kHeadBig;
    const uint64_t key = (uint64_t)keys[i];
    const uint32_t mp = key_is_clearing(kl, key) ? 1u : 0u;
    const uint32_t t0 = point_order_inv(P, order_inv, vals[i]);
    const uint32_t w = (mp ? words : 0u) + (t0 >> 5);
    const uint32_t e = g.wp[w] + (uint32_t)__popc(first_bits[w] & ((1u << (t0 & 31u)) - 1u));
    if (e >= g.cap) continue;  // (cannot happen: cap = max_points_per_scan)
    const I3 v = key_voxel(kl, key);
    g.h[mp * g.cap + e] = long_index_hash(v.x, v.y, v.z);
    g.head_of[mp * g.cap + e] = j;
  }
}

// A one-block grid needs no cooperative launch: its grid barrier is the block barrier.
__device__ __forceinline__ void order_grid_sync(cg::grid_group& grid) {
  if (gridDim.x == 1) {
    __syncthreads();
  } else {
    grid.sync();
  }
}

// grid-wide version of order_positions (vbx_order.cuh) on global tables; every block of the cooperative
// grid calls it.  cta_tot: one word per block.
__device__ void order_positions_grid(cg::grid_group& grid, const uint32_t* h, const uint32_t* tau, uint32_t* tau_out,
                                     uint32_t* next, uint32_t* bkt, uint32_t* A, uint32_t* bhead, uint32_t m, uint32_t n,
                                     uint32_t tag, uint32_t B, uint32_t* cta_tot, uint32_t* warp_sums) {
  const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gthreads = gridDim.x * blockDim.x;
  const uint32_t tg = tag << 20;
  for (uint32_t b = gtid; b < m; b += gthreads) {
    const uint32_t gb = h[b] % n;
    bkt[b] = gb;
    const uint32_t old = atomicExch(&bhead[gb], tg | b);
    next[b] = (old >> 20) == tag ? (old & 0xfffffu) : kOrderNil;
  }
  order_grid_sync(grid);
  for (uint32_t b = gtid; b < m; b += gthreads) {
    const uint32_t tb = __ldcg(&tau[b]);
    uint32_t cmin = kOrderNil, size = 0;
    for (uint32_t c = __ldcg(&bhead[bkt[b]]) & 0xfffffu; c != kOrderNil; c = __ldcg(&next[c])) {
      cmin = min(cmin, __ldcg(&tau[c]));
      ++size;
    }
    A[tb] = cmin == tb ? size : 0u;
  }
  order_grid_sync(grid);
  // exclusive suffix sum of A over times: block c owns a contiguous range of times (block 0 the highest),
  // thread t of it a contiguous run inside
  {
    const uint32_t per_cta = (m + gridDim.x - 1) / gridDim.x;
    const uint32_t chi = m > blockIdx.x * per_cta ? m - blockIdx.x * per_cta : 0u;
    const uint32_t clo = chi > per_cta ? chi - per_cta : 0u;
    const uint32_t per = (per_cta + kOrderThreads - 1) / kOrderThreads;
    const uint32_t hi = chi > clo + threadIdx.x * per ? chi - threadIdx.x * per : clo;
    const uint32_t lo = hi > clo + per ? hi - per : clo;
    uint32_t sum = 0;
    for (uint32_t t = lo; t < hi; ++t) sum += __ldcg(&A[t]);
    uint32_t total;
    uint32_t run = order_block_scan(sum, warp_sums, &total);
    if (threadIdx.x == 0) cta_tot[blockIdx.x] = total;
    order_grid_sync(grid);
    uint32_t above = 0;  // elements at times above this block's range
    for (uint32_t c = 0; c < blockIdx.x; ++c) above += __ldcg(&cta_tot[c]);
    run += above;
    for (uint32_t t = hi; t-- > lo;) {
      const uint32_t v = __ldcg(&A[t]);
      A[t] = run;
      run += v;
    }
  }
  order_grid_sync(grid);
  for (uint32_t b = gtid; b < B; b += gthreads) {
    if (b >= m) {  // inserted after this rehash: the insertion index stays its time
      tau_out[b] = b;
      continue;
    }
    const uint32_t tb = __ldcg(&tau[b]);
    uint32_t cmin = kOrderNil, later = 0;
    for (uint32_t c = __ldcg(&bhead[bkt[b]]) & 0xfffffu; c != kOrderNil; c = __ldcg(&next[c])) {
      const uint32_t tc = __ldcg(&tau[c]);
      cmin = min(cmin, tc);
      later += tc > tb ? 1u : 0u;
    }
    tau_out[b] = __ldcg(&A[cmin]) + later;
  }
  order_grid_sync(grid);
}

__global__ void __launch_bounds__(kOrderThreads)
k_bundle_order(RehashSchedule rs, OrderScratch g, uint32_t smem_words, uint32_t* __restrict__ ray_list, uint32_t* cta_tot,
               ScanState* st) {
  extern __shared__ uint32_t order_smem[];
  __shared__ uint32_t warp_sums[33];
  cg::grid_group grid = cg::this_grid();
  const uint32_t tid = threadIdx.x;
  const uint32_t B_of[2] = {st->n_rays, st->n_clear_rays};
  uint32_t n_of[2];
  bool small = true, bad = false;
  for (int mp = 0; mp < 2; ++mp) {
    uint32_t nf = 1;
    for (int k = 0; k < rs.count && rs.m[k] < B_of[mp]; ++k) nf = rs.n[k];
    n_of[mp] = nf;
    if (order_smem_words_needed(B_of[mp], nf) > smem_words) small = false;
    // bucket heads pack the element into 20 bits; cap = max_points_per_scan
    if (B_of[mp] > g.cap || B_of[mp] > (1u << 20) || nf > g.bucket_cap) bad = true;
  }
  if (bad) {
    if (blockIdx.x == 0 && tid == 0) atomicOr(&st->error, kErrUpdatesFull);
    return;
  }
  if (small && blockIdx.x != 0) return;  // (every block takes the same decision: nobody waits at a grid barrier)
  uint32_t base_rank = 0;
  for (int mp = 0; mp < 2; ++mp) {
    const uint32_t B = B_of[mp], n_final = n_of[mp];
    if (B == 0) continue;
    const uint32_t* gh = g.h + mp * g.cap;
    const uint32_t* head_of = g.head_of + mp * g.cap;
    uint32_t *h = order_smem, *tau = h, *tau2 = h, *next = h, *bkt = h, *A = h, *bhead = h;
    if (small) {
      // one block, 16-bit tables in shared memory (the hashes are read from global memory, once per stage)
      const uint32_t pad = (B + 1u) & ~1u;
      uint16_t* t16 = reinterpret_cast<uint16_t*>(order_smem);
      bhead = order_smem + 5u * pad / 2u;
      const uint16_t* pos = order_run<uint16_t>(rs, B, gh, t16, t16 + pad, t16 + 2u * pad, t16 + 3u * pad, t16 + 4u * pad, bhead,
                                                n_final, warp_sums);
      for (uint32_t e = tid; e < B; e += kOrderThreads) ray_list[base_rank + pos[e]] = head_of[e];
      __syncthreads();
      base_rank += B;
      continue;
    }
    // ---- a large map.  Stages whose tables fit shared memory run in block 0 alone ...
    int k_small = 0;       // rehash events [0, k_small) are handled in shared memory
    uint32_t m_small = 0;  // elements present at the last of them
    uint32_t n_small = 1;  // bucket count after it
    for (int k = 0; k < rs.count && rs.m[k] < B; ++k) {
      if (6u * rs.m[k] + (k > 0 ? rs.n[k - 1] : 1u) > smem_words) break;
      k_small = k + 1;
      m_small = rs.m[k];
      n_small = rs.n[k];
    }
    uint32_t* cur = g.tau;   // global arrays of the grid-wide stages
    uint32_t* oth = g.tau2;
    if (blockIdx.x == 0) {
      // the first m_small elements through rehash events 0 .. k_small-1: order_run's loop on a prefix
      h = order_smem;
      tau = h + m_small;
      tau2 = tau + m_small;
      next = tau2 + m_small;
      bkt = next + m_small;
      A = bkt + m_small;
      bhead = A + m_small;
      for (uint32_t e = tid; e < m_small; e += kOrderThreads) {
        h[e] = gh[e];
        tau[e] = e;
      }
      const uint32_t n_clear = k_small > 1 ? rs.n[k_small - 2] : 1u;
      for (uint32_t j = tid; j < n_clear; j += kOrderThreads) bhead[j] = 0u;
      __syncthreads();
      uint32_t n_cur = 1, tag = 1;
      uint32_t* c0 = tau;
      uint32_t* c1 = tau2;
      for (int k = 0; k < k_small; ++k) {
        const uint32_t mk = rs.m[k];
        if (mk > 0) {
          order_positions<uint32_t>(h, c0, c1, next, bkt, A, bhead, mk, n_cur, tag++, warp_sums);
          for (uint32_t e = mk + tid; e < m_small; e += kOrderThreads) c1[e] = e;
          __syncthreads();
          uint32_t* t = c0;
          c0 = c1;
          c1 = t;
        }
        n_cur = rs.n[k];
      }
      for (uint32_t e = tid; e < m_small; e += kOrderThreads) cur[e] = c0[e];
    }
    // ... the rest grid-wide.  Times of elements not yet inserted = their insertion index.
    const uint32_t gtid = blockIdx.x * blockDim.x + tid, gthreads = gridDim.x * blockDim.x;
    for (uint32_t e = m_small + gtid; e < B; e += gthreads) cur[e] = e;
    for (uint32_t j = gtid; j < n_final; j += gthreads) g.bhead[j] = 0u;
    order_grid_sync(grid);
    uint32_t n_cur = n_small, tag = 1;
    for (int k = k_small; k < rs.count && rs.m[k] < B; ++k) {
      order_positions_grid(grid, gh, cur, oth, g.next, g.bkt, g.A, g.bhead, rs.m[k], n_cur, tag++, B, cta_tot, warp_sums);
      uint32_t* t = cur;
      cur = oth;
      oth = t;
      n_cur = rs.n[k];
    }
    order_positions_grid(grid, gh, cur, oth, g.next, g.bkt, g.A, g.bhead, B, n_cur, tag, B, cta_tot, warp_sums);
    for (uint32_t e = gtid; e < B; e += gthreads) ray_list[base_rank + __ldcg(&oth[e])] = head_of[e];
    order_grid_sync(grid);  // the arrays are reused by the other map
    base_rank += B;
  }
}

// Correctly rounded a / b in three dependent operations, given y = RN(1 / b):
//   q = RN(a y);  r = a - q b (exact, one FMA);  a / b = RN(q + r y)
// (Markstein's division step; checked against IEEE division on 8e8 random and adversarial
// operand pairs by tests/exact_div_check.c).  It is only trusted for operands in a
// comfortable exponent band with a non-zero dividend (sign of zero) and a divisor whose
// mantissa is not all ones; anything else is flagged and the bundle is folded again with the
// IEEE division instruction.
__device__ __forceinline__ bool exact_div_operand_ok(float v) {
  const float a = fabsf(v);
  return a > 1e-18f && a < 1e18f;
}
__device__ __forceinline__ float recip_for_exact_div(float b, bool* ok) {
  *ok = exact_div_operand_ok(b) && (__float_as_uint(b) & 0x7fffffu) != 0x7fffffu;
  return __frcp_rn(b);
}

constexpr int kStageStride = 9;  // float4 per staged member (8 roles + 1 pad: conflict-free stores)

// One member's step of the fold for this lane's role:
//   t = state * A + B;   mean lanes: state = t / C;   colour lanes: state = round(t)
// kIeee = false uses the three-operation division with D = RN(1/C) and records operands it does
// not trust in *suspect; kIeee = true is the plain reference arithmetic.
template <bool kIeee>
__device__ __forceinline__ float fold_step(float state, float4 abcd, bool is_mean, bool* suspect) {
  const float tt = fadd(fmul(state, abcd.x), abcd.y);
  float quot;
  if (kIeee) {
    quot = is_mean ? fdiv(tt, abcd.z) : 0.f;
  } else {
    const float q = __fmul_rn(tt, abcd.w);
    quot = __fmaf_rn(__fmaf_rn(-q, abcd.z, tt), abcd.w, q);
    *suspect |= is_mean && !exact_div_operand_ok(tt);
  }
  // C round() (half away from zero) of t in [0, 2^22): nearest-even via the 2^23 trick, then
  // bump exact ties that went down
  const float m = fadd(fadd(tt, 8388608.0f), -8388608.0f);
  const float rnd = (fsub(tt, m) == 0.5f) ? fadd(m, 1.0f) : m;
  return is_mean ? quot : rnd;
}

// The two halves of fold_step as separate chains (k_merge runs them in separate warps, so that neither
// pays for the other's instructions): the running mean's  state = (state*A + B) / C  with the
// three-operation division, and a colour channel's  state = round(state*A + B).
__device__ __forceinline__ float fold_step_mean(float state, float4 abcd, bool* suspect) {
  const float tt = fadd(fmul(state, abcd.x), abcd.y);
  const float q = __fmul_rn(tt, abcd.w);
  *suspect |= !exact_div_operand_ok(tt);
  return __fmaf_rn(__fmaf_rn(-q, abcd.z, tt), abcd.w, q);
}
__device__ __forceinline__ float fold_step_colour(float state, float4 abcd) {
  const float tt = fadd(fmul(state, abcd.x), abcd.y);
  const float m = fadd(fadd(tt, 8388608.0f), -8388608.0f);
  return (fsub(tt, m) == 0.5f) ? fadd(m, 1.0f) : m;
}

// Fold one bundle (a run of equal keys starting at sorted position i) with one warp.
// Members are loaded 32 at a time (keys coalesced, points gathered, next chunk prefetched) and
// folded in list order with the reference's running weighted mean
//   merged = (merged * W + p * w) / (W + w); colour blended; W += w            (cc:387-405)
// Lanes 0-2 carry x, y, z of the mean, lanes 3-6 the colour channels (floats holding exact
// integers 0..255).  Returns true if the fast division met an operand it does not trust.
template <typename KeyT, bool kIeee>
__device__ bool fold_bundle(const ScanParams& P, const float* __restrict__ xyz, const uint8_t* __restrict__ rgba,
                            const KeyT* __restrict__ keys, const uint32_t* __restrict__ vals, uint32_t i,
                            float4* stage_warp, F3* out_mp, float* out_mw, uint32_t* out_col, const ScanState* st) {
  const int lane = threadIdx.x & 31;
  const KeyT key = keys[i];
  const bool clearing = key_is_clearing(key_layout(st), (uint64_t)key);
  float mw = 0.0f;
  bool done = false;
  bool suspect = false;
  float state = 0.f;
  const int role = lane < 7 ? lane : 7;  // lanes 7.. mirror a benign slot
  const bool is_mean = lane < 3;
  uint32_t j0 = i;
  bool in;
  F3 p = f3(0.f, 0.f, 0.f);
  uint32_t col = 0u;
  // Three-deep load pipeline: while chunk c is folded, the points of chunk c+1 are gathered (their
  // keys / point indices arrived one iteration ago) and the keys / indices of chunk c+2 are
  // requested -- no load is waited for right after it was issued.
  KeyT k_next;
  uint32_t idx_next;
  bool inb_next;
  {
    const uint32_t jj = j0 + lane;
    const bool inb = jj < P.n;
    const KeyT kk = inb ? keys[jj] : (KeyT)~(KeyT)0;
    const uint32_t idx = inb ? vals[jj] : 0u;
    j0 += 32;
    const uint32_t jn = j0 + lane;
    inb_next = jn < P.n;
    k_next = inb_next ? keys[jn] : (KeyT)~(KeyT)0;
    idx_next = inb_next ? vals[jn] : 0u;
    in = inb && kk == key;
    if (in) {
      p = load_point(xyz, idx);
      col = load_color(rgba, idx);
    }
  }
  while (!done) {
    const int cnt = __popc(__ballot_sync(0xffffffffu, in));  // members form a prefix
    const F3 pc = p;
    const uint32_t colc = col;
    const bool inc = in;
    if (cnt == 32) {
      in = inb_next && k_next == key;
      if (in) {
        p = load_point(xyz, idx_next);
        col = load_color(rgba, idx_next);
      }
      j0 += 32;
      const uint32_t jn = j0 + lane;
      inb_next = jn < P.n;
      k_next = inb_next ? keys[jn] : (KeyT)~(KeyT)0;
      idx_next = inb_next ? vals[jn] : 0u;
    }
    const float w = inc ? point_weight(pc.z, P.use_const_weight != 0) : 0.f;
    // (1) the weight chain W <- W + w is the only part every member depends on.  Lane L needs
    //     the W its member sees = mw + w_0 + ... + w_{L-1} added in list order (members below
    //     kEpsilon are skipped, cc:391-393: adding +0.0f is the identity).
    const float wl = (inc && !(w < VBX_EPS)) ? w : 0.f;
    float wb = mw;
#pragma unroll
    for (int k = 0; k < 31; ++k) {
      const float wk = __shfl_sync(0xffffffffu, wl, k);
      if (k < lane) wb = fadd(wb, wk);
    }
    float mw_run = __shfl_sync(0xffffffffu, fadd(wb, wl), 31);
    // (2) everything that does not depend on the running state, in parallel per lane, staged
    //     per role as (A, B, C, D = RN(1/C))
    const float tot = fadd(wb, w);
    const F3 pw = scale3(pc, w);
    float w1 = 0.f, w2 = 0.f, rtot = 1.f;
    if (wl != 0.f) {
      w1 = fdiv(wb, tot);  // blendTwoColors' normalised weights, core/common.h:112-113
      w2 = fdiv(w, tot);
      bool ok;
      rtot = recip_for_exact_div(tot, &ok);
      suspect |= !ok;
    }
    float4* st_row = stage_warp + lane * kStageStride;
    __syncwarp();  // the previous chunk's readers are done
    st_row[0] = make_float4(wb, pw.x, tot, rtot);
    st_row[1] = make_float4(wb, pw.y, tot, rtot);
    st_row[2] = make_float4(wb, pw.z, tot, rtot);
    st_row[3] = make_float4(w1, fmul((float)(int)(colc & 0xffu), w2), 1.f, 1.f);
    st_row[4] = make_float4(w1, fmul((float)(int)((colc >> 8) & 0xffu), w2), 1.f, 1.f);
    st_row[5] = make_float4(w1, fmul((float)(int)((colc >> 16) & 0xffu), w2), 1.f, 1.f);
    st_row[6] = make_float4(w1, fmul((float)(int)(colc >> 24), w2), 1.f, 1.f);
    st_row[7] = make_float4(0.f, 1.f, 1.f, 1.f);
    __syncwarp();
    // (3) the dependent chain, in list order, over the members that carry weight
    unsigned live = __ballot_sync(0xffffffffu, wl != 0.f);
    const float4* st_col = stage_warp + role;
    if (clearing && live) {  // "only take first point when clearing", cc:401-404
      const int k = __ffs(live) - 1;
      live = 1u << k;
      mw_run = fadd(__shfl_sync(0xffffffffu, wb, k), __shfl_sync(0xffffffffu, w, k));
      done = true;
    }
    if (live == 0xffffffffu) {
      float4 cur = st_col[0];
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float4 nxt = st_col[((k + 1) & 31) * kStageStride];
        state = fold_step<kIeee>(state, cur, is_mean, &suspect);
        cur = nxt;
      }
    } else {
      for (unsigned m = live; m; m &= m - 1) {
        state = fold_step<kIeee>(state, st_col[(__ffs(m) - 1) * kStageStride], is_mean, &suspect);
      }
    }
    mw = mw_run;
    if (cnt < 32) done = true;
  }
  *out_mp = f3(__shfl_sync(0xffffffffu, state, 0), __shfl_sync(0xffffffffu, state, 1),
               __shfl_sync(0xffffffffu, state, 2));
  *out_col = ((uint32_t)(int)__shfl_sync(0xffffffffu, state, 3) & 0xffu) |
             (((uint32_t)(int)__shfl_sync(0xffffffffu, state, 4) & 0xffu) << 8) |
             (((uint32_t)(int)__shfl_sync(0xffffffffu, state, 5) & 0xffu) << 16) |
             (((uint32_t)(int)__shfl_sync(0xffffffffu, state, 6) & 0xffu) << 24);
  *out_mw = mw;
  return __any_sync(0xffffffffu, suspect);
}

// Per-ray records.  ray_p (point_G, flags) feeds the two DDA walks; ray_a (point_G - origin and
// its norm, the per-ray half of computeDistance cc:216-228) and ray_c (colour, weight) feed the
// apply kernels, so that an update costs one division and no square root.
__device__ __forceinline__ void store_ray(const ScanParams& P, uint32_t i, F3 point_G, float weight, uint32_t color,
                                          bool clearing, float4* ray_p, float4* ray_a, uint2* ray_c) {
  const F3 po = sub3(point_G, P.origin);
  ray_p[i] = make_float4(point_G.x, point_G.y, point_G.z, __uint_as_float(clearing ? 1u : 0u));
  ray_a[i] = make_float4(po.x, po.y, po.z, norm3(po));
  ray_c[i] = make_uint2(color, __float_as_uint(weight));
}

// One chunk (up to 32 consecutive members of one bundle) handed from the producer warp to the
// consumer warp of a pair through shared memory.
struct ChunkDesc {
  uint32_t live;   // members that carry weight, in list order
  uint32_t head;   // sorted position of the bundle's first member
  uint32_t slot;   // the bundle's ray slot = its rank in the reference's bundle order
  uint32_t flags;
  float mw;        // merged weight after this chunk (final on the bundle's last chunk)
};
constexpr uint32_t kChunkFirst = 1u, kChunkLast = 2u, kChunkSuspect = 4u, kChunkEnd = 8u;

// named barriers of one warp triple (producer, mean consumer, colour consumer): ids 1 / 2 = the chunk
// hand-over of triple 0 / 1 (96 threads), ids 3 / 4 = the two consumers among themselves (64 threads);
// 0 is __syncthreads'.  Literal ids so that ptxas reserves five barriers, not all sixteen.
__device__ __forceinline__ void pair_barrier(int triple_in_block) {
  if (triple_in_block == 0) {
    asm volatile("bar.sync 1, 96;" ::: "memory");
  } else {
    asm volatile("bar.sync 2, 96;" ::: "memory");
  }
}
__device__ __forceinline__ void consumer_barrier(int triple_in_block) {
  if (triple_in_block == 0) {
    asm volatile("bar.sync 3, 64;" ::: "memory");
  } else {
    asm volatile("bar.sync 4, 64;" ::: "memory");
  }
}

// The merge of integrateVoxel (cc:384-407): every bundle's points folded in list order.  The fold
// is one dependent chain per bundle, so the kernel's duration is the largest bundle's chain (up to
// ~3000 points on this workload).  Warps work in TRIPLES on a stream of 32-member chunks:
//   producer         loads the members (three-deep load pipeline), walks the weight chain W <- W + w
//                    (the only thing a chunk needs from its predecessor besides the running state),
//                    computes everything else that does not depend on the running mean -- p*w, W+w,
//                    RN(1/(W+w)), blendTwoColors' normalised weights -- and stages it per role
//   mean consumer    runs the dependent chain state = (state*A + B) / C over the staged operands (lanes 0-2: x, y, z)
//   colour consumer  runs state = round(state*A + B) (lanes 0-3: r, g, b, a)
// so the preparation of chunk c+1 overlaps the chains of chunk c (two shared-memory slots, one
// named barrier per chunk), also across bundle boundaries, and each chain issues only its own
// instructions (~5 dependent operations per member for the mean, ~7 for a colour channel).
template <typename KeyT>
__global__ void __launch_bounds__(192)
k_merge(ScanParams P, const float* __restrict__ xyz, const uint8_t* __restrict__ rgba,
        const KeyT* __restrict__ keys, const uint32_t* __restrict__ vals, const uint32_t* __restrict__ head_list,
        const uint32_t* __restrict__ big_list,
        float4* __restrict__ ray_p, float4* __restrict__ ray_a, uint2* __restrict__ ray_c, uint32_t* __restrict__ cnt,
        ScanState* st) {
  __shared__ float4 stage[2][2][32 * kStageStride];  // [pair in block][slot][member][role]
  __shared__ ChunkDesc desc[2][2];
  const int lane = threadIdx.x & 31;
  __shared__ uint32_t s_col[2];
  const int warp_in_block = threadIdx.x >> 5;
  const int pair_in_block = warp_in_block / 3;  // (the triple this warp belongs to)
  const int warp_role = warp_in_block % 3;      // 0 producer, 1 mean consumer, 2 colour consumer
  const bool producer = warp_role == 0;
  const int bar_id = pair_in_block;
  const uint32_t n_bundles = st->n_ray_list;
  const uint32_t n_big = st->n_big;
  const KeyLayout kl = key_layout(st);
  uint32_t seq = 0;
  if (producer) {
    // Work is handed out by ticket: first the big bundles (their chains bound the kernel's duration, so
    // they start at once), then every other bundle in head_list order.
    while (true) {
      uint32_t ticket = 0;
      if (lane == 0) ticket = atomicAdd(&st->merge_ticket, 1u);
      ticket = __shfl_sync(0xffffffffu, ticket, 0);
      if (ticket >= n_big + n_bundles) break;
      uint32_t b, hl;
      if (ticket < n_big) {
        b = big_list[ticket];
        hl = head_list[b];
      } else {
        b = ticket - n_big;
        hl = head_list[b];
        if (hl & kHeadBig) continue;  // folded through the big list
      }
      const uint32_t i = hl & ~kHeadBig;
      const KeyT key = keys[i];
      const bool clearing = key_is_clearing(kl, (uint64_t)key);
      float mw = 0.0f;
      bool done = false, first = true;
      uint32_t j0 = i;
      bool in;
      F3 p = f3(0.f, 0.f, 0.f);
      uint32_t col = 0u;
      // three-deep load pipeline: while chunk c is prepared, the points of chunk c+1 are gathered
      // (their keys / point indices arrived one iteration ago) and the keys of chunk c+2 requested
      KeyT k_next;
      uint32_t idx_next;
      bool inb_next;
      {
        const uint32_t jj = j0 + lane;
        const bool inb = jj < P.n;
        const KeyT kk = inb ? keys[jj] : (KeyT)~(KeyT)0;
        const uint32_t idx = inb ? vals[jj] : 0u;
        j0 += 32;
        const uint32_t jn = j0 + lane;
        inb_next = jn < P.n;
        k_next = inb_next ? keys[jn] : (KeyT)~(KeyT)0;
        idx_next = inb_next ? vals[jn] : 0u;
        in = inb && kk == key;
        if (in) {
          p = load_point(xyz, idx);
          col = load_color(rgba, idx);
        }
      }
      while (!done) {
        const int n_in = __popc(__ballot_sync(0xffffffffu, in));  // members form a prefix
        const F3 pc = p;
        const uint32_t colc = col;
        const bool inc = in;
        if (n_in == 32) {
          in = inb_next && k_next == key;
          if (in) {
            p = load_point(xyz, idx_next);
            col = load_color(rgba, idx_next);
          }
          j0 += 32;
          const uint32_t jn = j0 + lane;
          inb_next = jn < P.n;
          k_next = inb_next ? keys[jn] : (KeyT)~(KeyT)0;
          idx_next = inb_next ? vals[jn] : 0u;
        }
        const float w = inc ? point_weight(pc.z, P.use_const_weight != 0) : 0.f;
        // the weight chain: lane L needs the W its member sees = mw + w_0 + ... + w_{L-1} added in
        // list order (members below kEpsilon are skipped, cc:391-393: adding +0.0f is the identity)
        const float wl = (inc && !(w < VBX_EPS)) ? w : 0.f;
        float wb = mw;
#pragma unroll
        for (int k = 0; k < 31; ++k) {
          const float wk = __shfl_sync(0xffffffffu, wl, k);
          if (k < lane) wb = fadd(wb, wk);
        }
        float mw_run = __shfl_sync(0xffffffffu, fadd(wb, wl), 31);
        const float tot = fadd(wb, w);
        const F3 pw = scale3(pc, w);
        float w1 = 0.f, w2 = 0.f, rtot = 1.f;
        bool bad = false;
        if (wl != 0.f) {
          w1 = fdiv(wb, tot);  // blendTwoColors' normalised weights, core/common.h:112-113
          w2 = fdiv(w, tot);
          bool ok;
          rtot = recip_for_exact_div(tot, &ok);
          bad = !ok;
        }
        unsigned live = __ballot_sync(0xffffffffu, wl != 0.f);
        if (clearing && live) {  // "only take first point when clearing", cc:401-404
          const int k = __ffs(live) - 1;
          live = 1u << k;
          mw_run = fadd(__shfl_sync(0xffffffffu, wb, k), __shfl_sync(0xffffffffu, w, k));
          done = true;
        }
        if (n_in < 32) done = true;
        const bool any_bad = __any_sync(0xffffffffu, bad);
        // (the slot was released by the consumer two barriers ago)
        const int slot = (int)(seq & 1u);
        float4* st_row = stage[pair_in_block][slot] + lane * kStageStride;
        st_row[0] = make_float4(wb, pw.x, tot, rtot);
        st_row[1] = make_float4(wb, pw.y, tot, rtot);
        st_row[2] = make_float4(wb, pw.z, tot, rtot);
        st_row[3] = make_float4(w1, fmul((float)(int)(colc & 0xffu), w2), 1.f, 1.f);
        st_row[4] = make_float4(w1, fmul((float)(int)((colc >> 8) & 0xffu), w2), 1.f, 1.f);
        st_row[5] = make_float4(w1, fmul((float)(int)((colc >> 16) & 0xffu), w2), 1.f, 1.f);
        st_row[6] = make_float4(w1, fmul((float)(int)(colc >> 24), w2), 1.f, 1.f);
        st_row[7] = make_float4(0.f, 1.f, 1.f, 1.f);
        if (lane == 0) {
          ChunkDesc d;
          d.live = live;
          d.head = i;
          d.slot = b;
          d.flags = (first ? kChunkFirst : 0u) | (done ? kChunkLast : 0u) | (any_bad ? kChunkSuspect : 0u);
          d.mw = mw_run;
          desc[pair_in_block][slot] = d;
        }
        pair_barrier(bar_id);
        ++seq;
        first = false;
        mw = mw_run;
      }
    }
    if (lane == 0) {
      ChunkDesc d;
      d.live = 0u;
      d.head = 0u;
      d.slot = 0u;
      d.flags = kChunkEnd;
      d.mw = 0.f;
      desc[pair_in_block][seq & 1u] = d;
    }
    pair_barrier(bar_id);
  } else if (warp_role == 2) {
    // ---- colour consumer: lanes 0-3 carry r, g, b, a (floats holding exact integers 0..255)
    const int role = 3 + (lane < 4 ? lane : 3);
    float state = 0.f;
    for (;; ++seq) {
      pair_barrier(bar_id);
      const int slot = (int)(seq & 1u);
      const ChunkDesc d = desc[pair_in_block][slot];
      if (d.flags & kChunkEnd) break;
      if (d.flags & kChunkFirst) state = 0.f;
      const float4* st_col = stage[pair_in_block][slot] + role;
      if (d.live == 0xffffffffu) {
        float4 cur = st_col[0];
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const float4 nxt = st_col[((k + 1) & 31) * kStageStride];
          state = fold_step_colour(state, cur);
          cur = nxt;
        }
      } else if (d.live) {
        unsigned m = d.live;
        float4 cur = st_col[(__ffs(m) - 1) * kStageStride];
        while (m) {
          m &= m - 1;
          const float4 nxt = st_col[(m ? __ffs(m) - 1 : 0) * kStageStride];
          state = fold_step_colour(state, cur);
          cur = nxt;
        }
      }
      if (d.flags & kChunkLast) {
        const uint32_t mcol = ((uint32_t)(int)__shfl_sync(0xffffffffu, state, 0) & 0xffu) |
                              (((uint32_t)(int)__shfl_sync(0xffffffffu, state, 1) & 0xffu) << 8) |
                              (((uint32_t)(int)__shfl_sync(0xffffffffu, state, 2) & 0xffu) << 16) |
                              (((uint32_t)(int)__shfl_sync(0xffffffffu, state, 3) & 0xffu) << 24);
        if (lane == 0) s_col[pair_in_block] = mcol;
        consumer_barrier(pair_in_block);  // the mean consumer picks the colour up and finishes the bundle
      }
    }
  } else {
    // ---- mean consumer: lanes 0-2 carry x, y, z of the running mean; it also finishes every bundle
    const int role = lane < 3 ? lane : 2;
    float state = 0.f;
    bool suspect = false;
    for (;; ++seq) {
      pair_barrier(bar_id);
      const int slot = (int)(seq & 1u);
      const ChunkDesc d = desc[pair_in_block][slot];
      if (d.flags & kChunkEnd) break;
      if (d.flags & kChunkFirst) {
        state = 0.f;
        suspect = false;
      }
      suspect |= (d.flags & kChunkSuspect) != 0u;
      const float4* st_col = stage[pair_in_block][slot] + role;
      if (d.live == 0xffffffffu) {
        float4 cur = st_col[0];
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const float4 nxt = st_col[((k + 1) & 31) * kStageStride];
          state = fold_step_mean(state, cur, &suspect);
          cur = nxt;
        }
      } else if (d.live) {
        unsigned m = d.live;
        float4 cur = st_col[(__ffs(m) - 1) * kStageStride];
        while (m) {
          m &= m - 1;
          const float4 nxt = st_col[(m ? __ffs(m) - 1 : 0) * kStageStride];  // the next operand's load overlaps the step
          state = fold_step_mean(state, cur, &suspect);
          cur = nxt;
        }
      }
      if (d.flags & kChunkLast) {
        consumer_barrier(pair_in_block);  // the colour consumer is done with this slot and has published the colour
        const uint32_t i = d.head;
        F3 mp;
        float mw = d.mw;
        uint32_t mcol = s_col[pair_in_block];
        if (__any_sync(0xffffffffu, suspect)) {
          // the fast division met an operand it does not trust: fold this bundle again with the
          // IEEE division (this warp alone, the slot just consumed as its staging area)
          fold_bundle<KeyT, true>(P, xyz, rgba, keys, vals, i, stage[pair_in_block][slot], &mp, &mw, &mcol, st);
          if (lane == 0) {
            atomicAdd(&st->n_refold, 1u);
            uint32_t lo = i, hi = P.n;  // first sorted position with a larger key
            const KeyT k = keys[i];
            while (lo < hi) {
              const uint32_t mid = (lo + hi) >> 1;
              if (keys[mid] <= k) lo = mid + 1; else hi = mid;
            }
            atomicAdd(&st->refold_members, lo - i);
          }
        } else {
          mp = f3(__shfl_sync(0xffffffffu, state, 0), __shfl_sync(0xffffffffu, state, 1),
                  __shfl_sync(0xffffffffu, state, 2));
        }
        if (lane == 0) {
          const bool clearing = key_is_clearing(kl, (uint64_t)keys[i]);
          const F3 pg = transform(P.T, mp);
          store_ray(P, d.slot, pg, mw, mcol, clearing, ray_p, ray_a, ray_c);
          if (P.single_walk) {
            Dda dd;
            dda_setup(dd, P.origin, pg, clearing, P.carving != 0, P.max_ray, P.voxel_size_inv, P.trunc, true);
            cnt[d.slot] = dd.len + 1u;  // RayCaster emits ray_length_in_steps_ + 1 voxels (integrator_utils.cc:111-125)
          }
        }
      }
    }
  }
}

// binary search over the sorted point keys: is there a NORMAL bundle ending in this voxel?
// (the voxel_map.find() of the anti-grazing test, cc:415-422)
template <typename KeyT>
__device__ bool bundle_exists(const KeyT* keys, uint32_t n, KeyT key) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (keys[mid] < key) {
      lo = mid + 1;
    } else {
      hi = mid;
    }
  }
  return lo < n && keys[lo] == key;
}

template <typename KeyT>
__device__ __forceinline__ bool grazing_skip(const ScanParams& P, const KeyLayout& kl, const KeyT* keys, KeyT own,
                                             bool clearing, int x, int y, int z) {
  bool in_range;
  const KeyT vkey = (KeyT)normal_key_of(kl, x, y, z, &in_range);
  if (!in_range) return false;
  const KeyT own_normal = clearing ? (KeyT)~(KeyT)0 : own;
  return (clearing || vkey != own_normal) && bundle_exists<KeyT>(keys, P.n, vkey);
}

// ApproxHashSet::replaceHash, utils/approx_hash_array.h:125-134.  The generation tag in
// the upper word plays the role of the reference's sliding offset (h:155-168).
__device__ __forceinline__ bool replace_hash(unsigned long long* set, uint32_t h, uint32_t epoch) {
  const unsigned long long tag = ((unsigned long long)epoch << 32) | h;
  const unsigned long long old = atomicExch(set + (h & 0xfffffu), tag);
  return old != tag;
}

// One thread per ray: first DDA walk.  Merged rays come from k_merge's records through the
// dense ray list; Simple / Fast build their ray from point slot i (integrateFunction,
// cc:269-305 / :488-553).
template <typename KeyT>
__global__ void k_rays_count(ScanParams P, Tables tab, const float* __restrict__ xyz,
                             const uint8_t* __restrict__ rgba, const uint32_t* __restrict__ order,
                             const KeyT* __restrict__ keys, const uint32_t* __restrict__ head_list,
                             float4* __restrict__ ray_p, float4* __restrict__ ray_a, uint2* __restrict__ ray_c,
                             uint32_t* __restrict__ cnt,
                             unsigned long long* set_start, unsigned long long* set_observed, ScanState* st) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t i;
  F3 point_G;
  bool clearing;
  KeyT own = 0;
  if (P.kind == VBX_MERGED) {
    if (t >= st->n_ray_list) return;
    i = t;  // bundle id j (the count does not depend on the order); head_list[j] = sorted position of its head
    const float4 rp = ray_p[i];
    point_G = f3(rp.x, rp.y, rp.z);
    clearing = (__float_as_uint(rp.w) & 1u) != 0;
    own = keys[head_list[t] & ~kHeadBig];
  } else {
    i = t;
    if (i > P.n) return;
    if (i == P.n) {
      cnt[i] = 0;
      return;
    }
    const uint32_t idx = point_order(P, order, i);
    const F3 p = load_point(xyz, idx);
    const int cls = classify_point(p, P.min_ray, P.max_ray, P.allow_clear != 0, P.freespace != 0);
    if (cls == 0) {
      cnt[i] = 0;
      return;
    }
    point_G = transform(P.T, p);
    clearing = (cls == 2);
    if (P.kind == VBX_FAST) {
      // start-voxel subsampling, cc:507-519
      const I3 g = grid_index(point_G, P.start_inv);
      if (!replace_hash(set_start, long_index_hash(g.x, g.y, g.z), P.set_epoch)) {
        cnt[i] = 0;
        return;
      }
    }
    store_ray(P, i, point_G, point_weight(p.z, P.use_const_weight != 0), load_color(rgba, idx), clearing, ray_p,
              ray_a, ray_c);
  }
  if (P.kind != VBX_MERGED) atomicAdd(clearing ? &st->n_clear_rays : &st->n_rays, 1u);  // (Merged: k_bundle_order)

  Dda d;
  dda_setup(d, P.origin, point_G, clearing, P.carving != 0, P.max_ray, P.voxel_size_inv, P.trunc,
            P.kind != VBX_FAST);
  if (P.single_walk) {
    cnt[i] = d.len + 1u;
    return;
  }
  uint32_t count = 0;
  int collisions = 0;
  int lbx = INT_MIN, lby = INT_MIN, lbz = INT_MIN;
  const int lim = (kCoordBias - 1) << P.L;
  for (unsigned int s = 0; s <= d.len; ++s, dda_advance(d)) {
    if (P.kind == VBX_MERGED && P.anti_grazing) {
      if (grazing_skip<KeyT>(P, key_layout(st), keys, own, clearing, d.cx, d.cy, d.cz)) continue;
    }
    if (P.kind == VBX_FAST) {
      // cc:531-543: stop once the ray runs through voxels other rays already observed
      if (!replace_hash(set_observed, long_index_hash(d.cx, d.cy, d.cz), P.set_epoch)) {
        ++collisions;
      } else {
        collisions = 0;
      }
      if (collisions > P.max_collisions) break;
    }
    if (d.cx < -lim || d.cx > lim || d.cy < -lim || d.cy > lim || d.cz < -lim || d.cz > lim) {
      atomicOr(&st->error, kErrCoordRange);
      break;
    }
    const int bx = d.cx >> P.L, by = d.cy >> P.L, bz = d.cz >> P.L;
    if ((bx != lbx || by != lby || bz != lbz) && owns_block(P, bx, by, bz)) {
      const uint32_t hp = ensure_block(tab, pack3(bx, by, bz), st);
      if (hp == 0xffffffffu) break;
      touch_block(tab, hp, P.epoch, st);
    }
    lbx = bx;
    lby = by;
    lbz = bz;
    ++count;
  }
  cnt[i] = count;
}

// A call that is applied in several passes (K > max_updates_per_pass): before each pass.  Blocks
// created by earlier passes already own their slots; the apply work lists restart.
__global__ void k_pass_begin(ScanState* st, unsigned long long pass_updates) {
  st->error &= ~kErrUpdatesFull;
  st->total_updates = st->error ? 0ull : pass_updates;
  st->n_new = 0;
  st->n_long = 0;
  st->n_verify = 0;
}

// First kernel of an asynchronously submitted scan's back half (walk stream: submission order).
__global__ void k_back_begin(ScanState* st, uint32_t* hold) {
  if (*hold) {
    st->error |= kSkipped;  // queued behind a scan that must be redone: do nothing, the host redoes both in order
    st->total_updates = 0;
  } else if (st->error & kErrUpdatesFull) {
    *hold = 1u;
  }
}

// After the last walk that can create blocks: pool slots for the blocks created by this call
// (updateLayerWithStoredBlocks, cc:137-147); a new block is born with all updated bits set (cc:128).
__global__ void k_assign(Tables tab, const uint32_t* __restrict__ nb_in, uint32_t* __restrict__ nb_out, SortPlan* record_plan,
                         ScanState* st) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < (uint32_t)(sizeof(SortPlan) / 4)) reinterpret_cast<uint32_t*>(record_plan)[j] = 0u;  // for the record sort that follows
  const uint32_t n_blocks_before = *nb_in;
  const uint32_t n_new = min(st->n_new, tab.max_blocks);
  if (j < n_new) {
    const uint32_t slot = n_blocks_before + j;
    if (slot < tab.max_blocks) {
      const uint32_t hp = tab.new_list[j];
      tab.hslot[hp] = (int32_t)slot;
      tab.slot_key[slot] = tab.hkeys[hp];
      tab.slot_updated[slot] = kTouchedBits;
    } else {
      atomicOr(&st->error, kErrPoolFull);
    }
  }
  if (j == 0) {
    const uint32_t after = min(n_blocks_before + st->n_new, tab.max_blocks);
    st->n_blocks = after;
    *nb_out = after;
    // what the record sort has to look at: voxel bits + the bits of the touched ids handed out
    uint32_t vb = 0;
    while ((tab.vox_per_block >> vb) > 1u) ++vb;
    st->rec_key_bits = vb + (uint32_t)(32 - __clz(st->n_touch_ids));
  }
}

// One ray, walked sequentially by the calling thread: RayCaster's loop (integrator_utils.cc:106-125)
// with allocateStorageAndGetVoxelPtr's find-or-create per block change (cc:91-134).
template <typename KeyT>
__device__ void emit_ray_sequential(const ScanParams& P, const Tables& tab, const KeyT* __restrict__ keys, uint32_t i,
                                    uint32_t rank, uint32_t head_pos, const float4* __restrict__ ray_p,
                                    const uint32_t* __restrict__ cnt,
                                    const uint32_t* __restrict__ off, uint32_t* __restrict__ ckeys,
                                    uint32_t* __restrict__ cvals, ScanState* st) {
  const uint32_t c = cnt[i];
  if (c == 0 || st->total_updates == 0) return;  // (a failed / to-be-redone call emits nothing)
  if (rank < P.emit_lo || rank >= P.emit_hi) return;   // (not in this pass)
  const float4 rp = ray_p[i];
  const bool clearing = (__float_as_uint(rp.w) & 1u) != 0;
  const F3 point_G = f3(rp.x, rp.y, rp.z);
  Dda d;
  dda_setup(d, P.origin, point_G, clearing, P.carving != 0, P.max_ray, P.voxel_size_inv, P.trunc,
            P.kind != VBX_FAST);
  const KeyT own = (P.kind == VBX_MERGED) ? keys[head_pos] : (KeyT)0;
  uint32_t emitted = 0;
  int lbx = INT_MIN, lby = INT_MIN, lbz = INT_MIN;
  uint32_t hp = 0, tid = 0;
  const uint32_t base = off[rank] - P.emit_base;
  const int mask = (1 << P.L) - 1;
  const int lim = (kCoordBias - 1) << P.L;
  for (unsigned int s = 0; s <= d.len && emitted < c; ++s, dda_advance(d)) {
    if (P.kind == VBX_MERGED && P.anti_grazing) {
      if (grazing_skip<KeyT>(P, key_layout(st), keys, own, clearing, d.cx, d.cy, d.cz)) continue;
    }
    const int bx = d.cx >> P.L, by = d.cy >> P.L, bz = d.cz >> P.L;
    if (bx != lbx || by != lby || bz != lbz) {
      if (!owns_block(P, bx, by, bz)) {
        hp = kNotOwned;  // another rank's block: the record keeps its place and is skipped by the apply
      } else if (P.single_walk) {
        // the only walk of this ray: allocateStorageAndGetVoxelPtr's find-or-create, cc:91-134
        if (d.cx < -lim || d.cx > lim || d.cy < -lim || d.cy > lim || d.cz < -lim || d.cz > lim) {
          atomicOr(&st->error, kErrCoordRange);
          hp = 0xffffffffu;
        } else {
          hp = ensure_block(tab, pack3(bx, by, bz), st);
        }
      } else {
        hp = find_block(tab, pack3(bx, by, bz));
      }
      tid = hp;  // (the two sentinels pass through)
      if (hp != 0xffffffffu && hp != kNotOwned) {
        tid = touch_block(tab, hp, P.epoch, st);
        const int32_t slot = tab.hslot[hp];
        if (slot >= 0) tab.slot_updated[slot] = kTouchedBits;  // (*last_block)->updated().set(), cc:128
      }
      lbx = bx;
      lby = by;
      lbz = bz;
    }
    const uint32_t lin = (uint32_t)(d.cx & mask) | ((uint32_t)(d.cy & mask) << P.L) |
                         ((uint32_t)(d.cz & mask) << (2 * P.L));
    // a record = (hash position of the block, voxel inside the block) -> ray.  A ray whose block
    // could not be created still fills its slots so that offsets stay valid; the error flag set
    // above stops the apply kernels.
    ckeys[base + emitted] = record_key(tid, lin, P.L);
    cvals[base + emitted] = i;
    ++emitted;
  }
}

template <typename KeyT>
__global__ void k_rays_emit(ScanParams P, Tables tab, const KeyT* __restrict__ keys,
                            const uint32_t* __restrict__ ray_list, const uint32_t* __restrict__ head_list,
                            const float4* __restrict__ ray_p, const uint32_t* __restrict__ cnt,
                            const uint32_t* __restrict__ off, uint32_t* __restrict__ ckeys,
                            uint32_t* __restrict__ cvals, ScanState* st) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t i;
  uint32_t head_pos = 0;
  if (P.kind == VBX_MERGED) {
    if (t >= st->n_ray_list) return;
    i = ray_list[t];  // rank t -> bundle id
    head_pos = head_list[i] & ~kHeadBig;
  } else {
    i = t;
    if (i >= P.n) return;
  }
  emit_ray_sequential<KeyT>(P, tab, keys, i, t, head_pos, ray_p, cnt, off, ckeys, cvals, st);
}

// The same walk cast by a WARP per ray (single-walk modes of the Merged integrator: a few thousand
// rays of 100-300 steps each, far too few threads for a thread-per-ray walk).  The walk is the
// stable three-way merge of the per-axis boundary-crossing chains (vbx_math.cuh, dda_rank):
//   1. lanes 0-2 build the chains T_a(k+1) = RN(T_a(k) + dt_a) in shared memory -- the only
//      sequential part, and plain additions;
//   2. all lanes rank the chain elements (two binary searches each) and scatter the voxel each
//      step reaches into a shared walk list;
//   3. the walk list is turned into records 32 at a time: block changes are found by comparing
//      neighbouring lanes, only the first lane of each block run does the hash find-or-create,
//      and the records leave the warp coalesced.
// Bit-identical to the sequential walk (tests/dda_merge_check.cc proves the merge against
// dda_advance on the host); rays the merge form does not cover (axis-parallel components,
// non-finite increments, more than kChainCap crossings on an axis) are walked by lane 0.
constexpr int kChainCap = 256;
constexpr int kWalkCap = 3 * kChainCap;

template <typename KeyT>
__global__ void __launch_bounds__(128)
k_rays_emit_warp(ScanParams P, Tables tab, const KeyT* __restrict__ keys, const uint32_t* __restrict__ ray_list,
                 const uint32_t* __restrict__ head_list, const float4* __restrict__ ray_p, const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ off,
                 uint32_t* __restrict__ ckeys, uint32_t* __restrict__ cvals, ScanState* st) {
  __shared__ float chain_s[4][3][kChainCap];
  __shared__ uint32_t walk_s[4][kWalkCap];
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t n_rays = st->n_ray_list;
  if (st->total_updates == 0) return;  // (a failed / to-be-redone call emits nothing)
  const int mask = (1 << P.L) - 1;
  const int lim = (kCoordBias - 1) << P.L;
  for (uint32_t b = warp; b < n_rays; b += n_warps) {
    const uint32_t i = ray_list[b];  // rank b in the reference's bundle order -> bundle id
    const uint32_t c = cnt[i];
    if (c == 0 || b < P.emit_lo || b >= P.emit_hi) continue;
    const float4 rp = ray_p[i];
    const bool clearing = (__float_as_uint(rp.w) & 1u) != 0;
    Dda d;
    dda_setup(d, P.origin, f3(rp.x, rp.y, rp.z), clearing, P.carving != 0, P.max_ray, P.voxel_size_inv, P.trunc, true);
    const unsigned int len = d.len;
    int K[3];
    K[0] = (int)dda_chain_len(d.nx, len);
    K[1] = (int)dda_chain_len(d.ny, len);
    K[2] = (int)dda_chain_len(d.nz, len);
    bool merge_ok = dda_is_regular(d) && K[0] <= kChainCap && K[1] <= kChainCap && K[2] <= kChainCap &&
                    len + 1u <= (unsigned int)kWalkCap && c == len + 1u;
    if (merge_ok) {
      // 1. the chains
      if (lane < 3) {
        float t = lane == 0 ? d.tx : (lane == 1 ? d.ty : d.tz);
        const float dt = lane == 0 ? d.dx : (lane == 1 ? d.dy : d.dz);
        const int kk = K[lane];
        float* dst = chain_s[w][lane];
        for (int k = 0; k < kk; ++k) {
          dst[k] = t;
          t = fadd(t, dt);
        }
      }
      if (lane == 0) walk_s[w][0] = 0u;
      __syncwarp();
      // 2. rank every chain element, scatter the voxel it leads to
      const float* const T[3] = {chain_s[w][0], chain_s[w][1], chain_s[w][2]};
      const int total = K[0] + K[1] + K[2];
      unsigned int emitted = 0;
      bool trusted_all = true;
      for (int e = lane; e < total; e += 32) {
        const int a = e < K[0] ? 0 : (e < K[0] + K[1] ? 1 : 2);
        const int k = e - (a == 0 ? 0 : (a == 1 ? K[0] : K[0] + K[1]));
        unsigned int rank;
        int c3[3];
        const bool trusted = dda_rank(T, K, len, a, k, &rank, c3);
        if (rank < len) {
          trusted_all &= trusted;
          walk_s[w][rank + 1u] = (uint32_t)c3[0] | ((uint32_t)c3[1] << 10) | ((uint32_t)c3[2] << 20);
          ++emitted;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) emitted += __shfl_xor_sync(0xffffffffu, emitted, o);
      merge_ok = __all_sync(0xffffffffu, trusted_all) && emitted == len;
      __syncwarp();
    }
    if (!merge_ok) {
      if (lane == 0) {
        emit_ray_sequential<KeyT>(P, tab, keys, i, b, head_list[i] & ~kHeadBig, ray_p, cnt, off, ckeys, cvals, st);
      }
      __syncwarp();
      continue;
    }
    // 3. records, 32 steps at a time
    const uint32_t base = off[b] - P.emit_base;
    int cbx = INT_MIN, cby = INT_MIN, cbz = INT_MIN;  // block of the previous chunk's last step
    uint32_t chp = 0u;
    for (unsigned int r0 = 0; r0 <= len; r0 += 32u) {
      const unsigned int r = r0 + (unsigned int)lane;
      const bool valid = r <= len;
      const uint32_t pk = valid ? walk_s[w][r] : 0u;
      const int vx = d.cx + d.sx * (int)(pk & 1023u);
      const int vy = d.cy + d.sy * (int)((pk >> 10) & 1023u);
      const int vz = d.cz + d.sz * (int)(pk >> 20);
      const int bx = vx >> P.L, by = vy >> P.L, bz = vz >> P.L;
      int pbx = __shfl_up_sync(0xffffffffu, bx, 1), pby = __shfl_up_sync(0xffffffffu, by, 1),
          pbz = __shfl_up_sync(0xffffffffu, bz, 1);
      if (lane == 0) {
        pbx = cbx;
        pby = cby;
        pbz = cbz;
      }
      const bool head = valid && (bx != pbx || by != pby || bz != pbz);
      uint32_t hp = 0u;
      if (head) {
        // the first step inside a block: allocateStorageAndGetVoxelPtr's find-or-create, cc:91-134
        if (!owns_block(P, bx, by, bz)) {
          hp = kNotOwned;
        } else if (vx < -lim || vx > lim || vy < -lim || vy > lim || vz < -lim || vz > lim) {
          atomicOr(&st->error, kErrCoordRange);
          hp = 0xffffffffu;
        } else {
          hp = ensure_block(tab, pack3(bx, by, bz), st);
        }
        if (hp != 0xffffffffu && hp != kNotOwned) {
          const int32_t slot = tab.hslot[hp];
          if (slot >= 0) tab.slot_updated[slot] = kTouchedBits;  // (*last_block)->updated().set(), cc:128
          hp = touch_block(tab, hp, P.epoch, st);      // from here on: the block's touched id
        }
      }
      const unsigned int heads = __ballot_sync(0xffffffffu, head);
      const unsigned int below = heads & (0xffffffffu >> (31 - lane));  // heads at or below this lane
      const int src = below ? 31 - __clz(below) : 0;
      const uint32_t hp_run = __shfl_sync(0xffffffffu, hp, src);
      const uint32_t hp_l = below ? hp_run : chp;
      if (valid) {
        const uint32_t lin = (uint32_t)(vx & mask) | ((uint32_t)(vy & mask) << P.L) | ((uint32_t)(vz & mask) << (2 * P.L));
        ckeys[base + r] = record_key(hp_l, lin, P.L);
        cvals[base + r] = i;
      }
      // carry the last step's block into the next chunk (a full chunk whenever there is a next one)
      cbx = __shfl_sync(0xffffffffu, bx, 31);
      cby = __shfl_sync(0xffffffffu, by, 31);
      cbz = __shfl_sync(0xffffffffu, bz, 31);
      chp = __shfl_sync(0xffffffffu, hp_l, 31);
    }
    __syncwarp();  // the walk list is reused by this warp's next ray
  }
}

// ----------------------------------------------------------------------- apply
struct VoxelRef {
  TsdfVoxel* ptr;
  F3 vo;  // voxel centre - sensor origin
};

__device__ __forceinline__ VoxelRef locate_voxel(const ScanParams& P, const Tables& tab, uint32_t key) {
  const uint32_t hp = tab.touched_list[key >> (3 * P.L)];  // touched id -> hash position
  const uint32_t lin = key & ((1u << (3 * P.L)) - 1u);
  int bx, by, bz;
  unpack3(tab.hkeys[hp], &bx, &by, &bz);
  const int mask = (1 << P.L) - 1;
  const int vx = (bx << P.L) + (int)(lin & mask);
  const int vy = (by << P.L) + (int)((lin >> P.L) & mask);
  const int vz = (bz << P.L) + (int)(lin >> (2 * P.L));
  VoxelRef r;
  // (a block that found no pool slot -- kErrPoolFull -- has hslot < 0: nothing to update)
  const int32_t slot = tab.hslot[hp];
  r.ptr = slot >= 0 ? tab.tsdf + (((size_t)slot) << (3 * P.L)) + lin : nullptr;
  const F3 c = f3(center_coord(vx, P.voxel_size), center_coord(vy, P.voxel_size), center_coord(vz, P.voxel_size));
  r.vo = sub3(c, P.origin);
  return r;
}

// computeDistance (cc:216-228) with both sides hoisted: vo = voxel centre - origin (per voxel),
// ra = (point_G - origin, |point_G - origin|) (per ray):  sdf = |po| - (vo . po) / |po|
__device__ __forceinline__ float sdf_from(F3 vo, float4 ra) {
  return fsub(ra.w, fdiv(dot3(vo, f3(ra.x, ra.y, ra.z)), ra.w));
}

// The sorted update records as the apply kernels see them: with the library sort the host knows
// which buffer holds the result and how many records there are; with the engine's own sort both
// live in device memory (SortPlan::final_buf, ScanState::total_updates).
struct RecordView {
  const uint32_t* keys[2];
  const uint32_t* vals[2];
  const SortPlan* plan;                 // nullptr: buffer 0 holds the sorted records
  const unsigned long long* d_total;    // nullptr: total_fixed
  unsigned long long total_fixed;
};
__device__ __forceinline__ void open_records(const RecordView& rv, const uint32_t** ckeys, const uint32_t** cvals,
                                             unsigned long long* total) {
  const uint32_t sel = rv.plan ? rv.plan->final_buf : 0u;
  *ckeys = rv.keys[sel];
  *cvals = rv.vals[sel];
  *total = rv.d_total ? *rv.d_total : rv.total_fixed;
}

// Voxel runs longer than kShortRun updates.  state: 0 = apply sequentially (k_apply_long),
// 1 = candidate for the parallel fixed-point check, |2 = the check failed.
constexpr unsigned long long kVerifyItem = 256;  // 8 records per lane: short dependent chains, many items
struct LongRuns {
  unsigned long long* start;   // first record after the prefix the head thread applied
  unsigned long long* end;     // one past the run's last record (state != 0)
  uint32_t* state;
  uint32_t* item_run;          // work items of k_apply_verify
  unsigned long long* item_start;
  float* rec_sdf;              // per sorted record: sdf and effective weight, written by
  float* rec_w;                // k_apply_short's parallel phase, read by the long-run kernels
};

// One warp per work item: do all updates in [start, start + kVerifyItem) of a saturated voxel's
// run map (+T, max_weight) onto itself?  An update does when its sdf >= T (no colour blend), the
// new distance clamps back to +T and the weight clamps back to max_weight -- evaluated with the
// reference's own arithmetic, so "unchanged" is exact, not approximate.
__global__ void k_apply_verify(ScanParams P, Tables tab, RecordView rv, const float4* __restrict__ ray_a,
                               const uint2* __restrict__ ray_c, LongRuns lr, const ScanState* st) {
  const uint32_t* ckeys;
  const uint32_t* cvals;
  unsigned long long total;
  open_records(rv, &ckeys, &cvals, &total);
  if (st->error & kFatalErrors) return;
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t n_items = st->n_verify;
  const float T = P.up.trunc, W = P.up.max_weight;
  for (uint32_t it = warp; it < n_items; it += n_warps) {
    const uint32_t q = lr.item_run[it];
    const unsigned long long a = lr.item_start[it];
    const unsigned long long b = min(a + kVerifyItem, lr.end[q]);
    bool ok = true;
#pragma unroll
    for (int k = 0; k < (int)(kVerifyItem / 32); ++k) {
      const unsigned long long j = a + lane + 32ull * k;
      if (j >= b) continue;
      const float sdf = lr.rec_sdf[j], w = lr.rec_w[j];
      const float nw = fadd(W, w);
      bool keeps = sdf >= T && !(nw < VBX_EPS) && !(nw < W);
      if (keeps) {
        const float ns = fdiv(fadd(fmul(sdf, w), fmul(T, W)), nw);
        keeps = (ns > 0.0f) && !(ns < T);
      }
      ok = ok && keeps;
    }
    if (!__all_sync(0xffffffffu, ok) && lane == 0) atomicOr(&lr.state[q], 2u);
  }
}

// One thread per run head applies the first kShortRun updates of its voxel in order
// (updateTsdfVoxel, cc:150-209); longer runs are queued for k_apply_long.
__global__ void __launch_bounds__(256)
k_apply_short(ScanParams P, Tables tab, RecordView rv, const float4* __restrict__ ray_a,
              const uint2* __restrict__ ray_c, LongRuns lr, ScanState* st) {
  // Phase 1 (every thread): one record each -- gather its ray, form sdf and weight.  This is the
  // expensive, perfectly parallel part; results are staged in shared memory.
  // Phase 2 (run heads): the read-modify-write chain of updateTsdfVoxel over the staged values.
  __shared__ uint32_t s_key[256];
  __shared__ float s_sdf[256];
  __shared__ float s_w[256];
  __shared__ uint32_t s_col[256];
  const uint32_t* ckeys;
  const uint32_t* cvals;
  unsigned long long total;
  open_records(rv, &ckeys, &cvals, &total);
  if (st->error & kFatalErrors) return;
  const unsigned long long n_tiles = (total + 255ull) / 256ull;
  for (unsigned long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const unsigned long long base = tile * 256ull;
    const unsigned long long e = base + threadIdx.x;
    bool head = false;
    uint32_t key = 0xffffffffu;
    VoxelRef vr;
    vr.ptr = nullptr;
    vr.vo = f3(0.f, 0.f, 0.f);
    if (e < total) key = ckeys[e];
    if (key != kSkipRecord) {  // (records of blocks this rank does not own sort to the end and are skipped)
      head = (e == 0) || (ckeys[e - 1] != key);
      const uint32_t r = cvals[e];
      const float4 ra = ray_a[r];
      const uint2 rc = ray_c[r];
      vr = locate_voxel(P, tab, key);
      const float sdf = sdf_from(vr.vo, ra);
      const float w = update_weight(sdf, __uint_as_float(rc.y), P.up);
      s_sdf[threadIdx.x] = sdf;
      s_w[threadIdx.x] = w;
      s_col[threadIdx.x] = rc.x;
      lr.rec_sdf[e] = sdf;
      lr.rec_w[e] = w;
    }
    s_key[threadIdx.x] = key;
    __syncthreads();
    head = head && vr.ptr != nullptr;
    if (head) {
      TsdfVoxel v = *vr.ptr;
      unsigned long long j = e;
      int k = 0;
      // inside this tile: staged values
      for (; k < kShortRun && j < base + 256ull && s_key[j - base] == key; ++k, ++j) {
        apply_update(v, s_sdf[j - base], s_w[j - base], s_col[j - base], P.up);
      }
      // a run that crosses the tile boundary continues from global memory
      if (j == base + 256ull) {
        for (; k < kShortRun && j < total && ckeys[j] == key; ++k, ++j) {
          const uint32_t r = cvals[j];  // (the next tile's staged values are not visible here)
          const float sdf = sdf_from(vr.vo, ray_a[r]);
          const uint2 rc = ray_c[r];
          apply_update(v, sdf, update_weight(sdf, __uint_as_float(rc.y), P.up), rc.x, P.up);
        }
      }
      *vr.ptr = v;
      if (j < total && ckeys[j] == key) {
        const uint32_t q = atomicAdd(&st->n_long, 1u);
        lr.start[q] = j;
        // A voxel resting at (+T, max_weight) -- free space seen many times -- stays there as
        // long as every remaining update maps that state onto itself, which can be checked
        // record by record, in parallel (k_apply_verify).  Find the end of the run (records are
        // sorted) and cut it into work items.
        const bool saturated = v.distance == P.up.trunc && v.weight == P.up.max_weight && P.up.max_weight >= VBX_EPS;
        uint32_t state = 0u;
        if (saturated) {
          unsigned long long lo = j, hi = total;  // first record past the run
          while (lo < hi) {
            const unsigned long long mid = (lo + hi) >> 1;
            if (ckeys[mid] <= key) {
              lo = mid + 1;
            } else {
              hi = mid;
            }
          }
          lr.end[q] = lo;
          for (unsigned long long a = j; a < lo; a += kVerifyItem) {
            const uint32_t it = atomicAdd(&st->n_verify, 1u);
            lr.item_run[it] = q;
            lr.item_start[it] = a;
          }
          state = 1u;
        }
        lr.state[q] = state;
      }
    }
    const unsigned b = __ballot_sync(0xffffffffu, head);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(&st->n_voxels, (uint32_t)__popc(b));
    __syncthreads();  // the staging arrays are reused by the next tile
  }
}

// One warp per long run.  32 updates are prefetched per step (records coalesced, ray data
// gathered, sdf and weight computed in parallel); the read-modify-write chain is then
// evaluated in order.  Free space far in front of any surface is the common long run:
// there every update has sdf >= T and the voxel already sits at +T, so after computing the
// exact sequential weight chain each lane checks that ITS update maps +T to +T; if all do,
// the sequential result is (+T, chained weight) without walking the distance chain.
__global__ void k_apply_long(ScanParams P, Tables tab, RecordView rv, const float4* __restrict__ ray_a,
                             const uint2* __restrict__ ray_c, LongRuns lr, const ScanState* st) {
  const uint32_t* ckeys;
  const uint32_t* cvals;
  unsigned long long total;
  open_records(rv, &ckeys, &cvals, &total);
  if (st->error & kFatalErrors) return;
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t n_long = st->n_long;
  const float T = P.up.trunc;
  for (uint32_t q = warp; q < n_long; q += n_warps) {
    if (lr.state[q] == 1u) continue;  // verified: every remaining update keeps (+T, max_weight)
    unsigned long long j0 = lr.start[q];
    const uint32_t key = ckeys[j0];
    const VoxelRef vr = locate_voxel(P, tab, key);
    TsdfVoxel v = *vr.ptr;
    bool done = false;
    // sdf and weight of every record were computed by k_apply_short's parallel phase; the chain
    // only streams them.  Four 32-record chunks are loaded per step (and the next four are
    // prefetched) so that the loads of a step are all in flight together; colours are gathered
    // on the rare chunks that need the full update.
    constexpr int kG = 4;
    bool in_n[kG];
    float sdf_n[kG], w_n[kG];
#pragma unroll
    for (int g = 0; g < kG; ++g) {
      const unsigned long long j = j0 + 32ull * g + lane;
      in_n[g] = j < total && ckeys[j] == key;
      sdf_n[g] = in_n[g] ? lr.rec_sdf[j] : 0.f;
      w_n[g] = in_n[g] ? lr.rec_w[j] : 0.f;
    }
    while (!done) {
      bool in_c[kG];
      float sdf_c[kG], w_c[kG];
#pragma unroll
      for (int g = 0; g < kG; ++g) {
        in_c[g] = in_n[g];
        sdf_c[g] = sdf_n[g];
        w_c[g] = w_n[g];
      }
      const bool more = __all_sync(0xffffffffu, in_c[kG - 1]);  // the run may continue past these records
      if (more) {
#pragma unroll
        for (int g = 0; g < kG; ++g) {
          const unsigned long long j = j0 + 32ull * (kG + g) + lane;
          in_n[g] = j < total && ckeys[j] == key;
          sdf_n[g] = in_n[g] ? lr.rec_sdf[j] : 0.f;
          w_n[g] = in_n[g] ? lr.rec_w[j] : 0.f;
        }
      }
      // The common long run -- free space far in front of any surface, the voxel already at +T -- is decided
      // for all kG chunks at once: ONE exact in-order weight chain over the step's records, then every
      // lane checks that its updates map +T onto +T, one vote.  (Same arithmetic as the per-chunk path
      // below, which remains for everything else and redoes the step from the unchanged voxel if a
      // check fails.)
      bool step_done = false;
      {
        bool ff = true;
        float wl[kG];
#pragma unroll
        for (int g = 0; g < kG; ++g) {
          ff = ff && (!in_c[g] || sdf_c[g] >= T);
          wl[g] = in_c[g] ? w_c[g] : 0.f;
        }
        if (__all_sync(0xffffffffu, ff) && v.distance == T) {
          float ws = (wl[0] + wl[1]) + (wl[2] + wl[3]);  // any-order sum, used only as a bound
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) ws += __shfl_xor_sync(0xffffffffu, ws, o);
          const bool saturated = v.weight == P.up.max_weight && P.up.max_weight >= VBX_EPS;
          const bool no_clamp = v.weight >= VBX_EPS && (v.weight + ws) * 1.0001f < P.up.max_weight;
          float mb[kG];
          float w_end = v.weight;
          bool have = true;
          if (saturated) {
            // W + w >= max_weight for every w >= 0: the clamp returns max_weight at every step
#pragma unroll
            for (int g = 0; g < kG; ++g) mb[g] = v.weight;
          } else if (no_clamp) {
            // neither the 1e-6 guard nor the max_weight clamp can fire: the chain is plain in-order addition
            bool ints = v.weight == truncf(v.weight) && (v.weight + ws) < 16777216.0f;
#pragma unroll
            for (int g = 0; g < kG; ++g) ints = ints && wl[g] == truncf(wl[g]);
            if (__all_sync(0xffffffffu, ints)) {
              // integer-valued weights (use_const_weight: a bundle's weight is its point count) on an
              // integer-valued W, everything below 2^24: every partial sum is exact, so any order gives
              // the in-order chain -- a warp scan per chunk
              float base = v.weight;
#pragma unroll
              for (int g = 0; g < kG; ++g) {
                float inc = wl[g];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                  const float t = __shfl_up_sync(0xffffffffu, inc, o);
                  if (lane >= o) inc += t;
                }
                mb[g] = base + (inc - wl[g]);
                base = base + __shfl_sync(0xffffffffu, inc, 31);
              }
              w_end = base;
            } else {
              float base = v.weight;
#pragma unroll
              for (int g = 0; g < kG; ++g) {
                float before = base;
#pragma unroll
                for (int k = 0; k < 31; ++k) {
                  const float wk = __shfl_sync(0xffffffffu, wl[g], k);
                  if (k < lane) before = fadd(before, wk);
                }
                mb[g] = before;
                base = __shfl_sync(0xffffffffu, fadd(before, wl[g]), 31);
              }
              w_end = base;
            }
          } else {
            have = false;
          }
          if (have) {
            bool keeps_T = true;
#pragma unroll
            for (int g = 0; g < kG; ++g) {
              if (in_c[g]) {
                const float nw = fadd(mb[g], w_c[g]);
                if (!(nw < VBX_EPS)) {
                  const float ns = fdiv(fadd(fmul(sdf_c[g], w_c[g]), fmul(T, mb[g])), nw);
                  const float clamped = (ns > 0.0f) ? ((ns < T) ? ns : T) : ((-T < ns) ? ns : -T);
                  keeps_T = keeps_T && (clamped == T);
                }
              }
            }
            if (__all_sync(0xffffffffu, keeps_T)) {
              v.weight = w_end;
              step_done = true;
            }
          }
        }
      }
#pragma unroll
      for (int g = 0; g < kG; ++g) {
        if (step_done) break;
        const bool in = in_c[g];
        const float sdf = sdf_c[g], w = w_c[g];
        const int cnt = __popc(__ballot_sync(0xffffffffu, in));
        if (cnt == 0) break;
        const bool far_free = !in || sdf >= T;
        bool fast = __all_sync(0xffffffffu, far_free) && v.distance == T;
        float w_end = v.weight;
        if (fast) {
          // exact sequential weight chain: W <- min(W + w, max_weight) unless W + w < 1e-6
          float my_before = 0.f;
          float wsum = in ? w : 0.f;  // any-order sum, used only as a bound
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
          const bool no_clamp = v.weight >= VBX_EPS && (v.weight + wsum) * 1.0001f < P.up.max_weight;
          if (v.weight == P.up.max_weight && P.up.max_weight >= VBX_EPS) {
            // the weight already sits at max_weight: W + w >= max_weight for every w >= 0, so the
            // clamp returns max_weight at every step
            my_before = v.weight;
          } else if (no_clamp && v.weight < 4194304.0f && v.weight == truncf(v.weight) &&
                     __all_sync(0xffffffffu, !in || w == 1.0f)) {
            // constant weights (use_const_weight) on an integer-valued W below 2^22: every partial
            // sum is an integer that float represents exactly, so the in-order chain is W + k
            my_before = v.weight + (float)lane;
            w_end = v.weight + (float)cnt;
          } else if (no_clamp) {
            // neither the 1e-6 guard nor the max_weight clamp can fire in this chunk: the
            // chain is plain in-order addition; lane L forms its own prefix
            const float wl = in ? w : 0.f;
            my_before = v.weight;
#pragma unroll
            for (int k = 0; k < 31; ++k) {
              const float wk = __shfl_sync(0xffffffffu, wl, k);
              if (k < lane) my_before = fadd(my_before, wk);
            }
            w_end = __shfl_sync(0xffffffffu, fadd(my_before, wl), 31);
          } else {
            for (int k = 0; k < cnt; ++k) {
              const float wk = __shfl_sync(0xffffffffu, w, k);
              if (lane == k) my_before = w_end;
              const float nw = fadd(w_end, wk);
              w_end = (nw < VBX_EPS) ? w_end : ((nw < P.up.max_weight) ? nw : P.up.max_weight);
            }
          }
          bool keeps_T = true;
          if (in) {
            const float nw = fadd(my_before, w);
            if (!(nw < VBX_EPS)) {
              const float ns = fdiv(fadd(fmul(sdf, w), fmul(T, my_before)), nw);
              const float clamped = (ns > 0.0f) ? ((ns < T) ? ns : T) : ((-T < ns) ? ns : -T);
              keeps_T = (clamped == T);
            }
          }
          fast = __all_sync(0xffffffffu, keeps_T);
        }
        if (fast) {
          v.weight = w_end;
        } else {
          const uint32_t col = in ? ray_c[cvals[j0 + 32ull * g + lane]].x : 0u;
          for (int k = 0; k < cnt; ++k) {
            apply_update(v, __shfl_sync(0xffffffffu, sdf, k), __shfl_sync(0xffffffffu, w, k),
                         __shfl_sync(0xffffffffu, col, k), P.up);
          }
        }
      }
      j0 += 32ull * kG;
      if (!more) done = true;
    }
    if (lane == 0) *vr.ptr = v;
  }
}

// --------------------------------------------------------------------- host side
// The growth schedule of a default-constructed std::unordered_map (max_load_factor 1) under
// one-by-one insertion, taken from the C++ library's own policy object: operator[] asks
// _M_need_rehash(bucket_count, element_count, 1) before every insertion of a new key
// (bits/hashtable.h _M_insert_unique_node).
int init_bundle_order(vbx_ctx* c) {
  RehashSchedule& rs = c->rehash;
  std::memset(&rs, 0, sizeof(rs));
  std::__detail::_Prime_rehash_policy pol;
  size_t buckets = 1;
  size_t e = 0;
  const size_t limit = (size_t)c->max_points + 1;
  while (e < limit && rs.count < 30) {
    const auto r = pol._M_need_rehash(buckets, e, 1);
    if (r.first) {
      buckets = r.second;
      rs.m[rs.count] = (uint32_t)e;
      rs.n[rs.count] = (uint32_t)buckets;
      ++rs.count;
    }
    // no rehash can happen before the element count exceeds the policy's next threshold
    const size_t next = (size_t)pol._M_next_resize;
    e = std::max(e + 1, next);
  }
  if (e < limit) return fail(c, VBX_E_INVALID, "unordered_map growth schedule longer than expected");
  int dev = 0, max_optin = 0;
  VBX_CUDA(c, cudaGetDevice(&dev));
  VBX_CUDA(c, cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  c->order_smem_bytes = (size_t)std::max(0, max_optin - 2048) & ~(size_t)15;
  VBX_CUDA(c, cudaFuncSetAttribute(k_bundle_order, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->order_smem_bytes));
  return VBX_OK;
}

static inline unsigned int grid_for(uint64_t n, int block) { return (unsigned int)((n + block - 1) / block); }

static int check_state_errors(vbx_ctx* c, const ScanState& h) {
  const uint32_t err = h.error & kFatalErrors;
  if (!err) return VBX_OK;
  if (err & kErrPoolFull) {
    // the surplus hash entries of this call have no pool slot: drop them, or later calls would find them
    if (h.n_blocks) c->n_blocks = h.n_blocks;
    rebuild_hash(c);
  }
  std::string m = "device reported:";
  if (err & kErrPoolFull) m += " block pool full (raise vbx_engine_options.max_blocks);";
  if (err & kErrHashFull) m += " block hash full;";
  if (err & kErrCoordRange) m += " voxel coordinate outside +-2^20 blocks;";
  if (err & kErrUpdatesFull) m += " ray-voxel updates exceed max_updates_per_pass;";
  return fail(c, VBX_E_CAPACITY, m);
}

namespace {
struct Marks {
  vbx_ctx* c;
  cudaStream_t s;
  bool on;  // stage profiling (vbx_set_stage_profiling); pipelined scans run without: the events would serialise the streams
  int n = 0;
  int stage[20];
  void begin() {
    if (on) cudaEventRecord(c->sev[0], s);
  }
  void mark(int stage_just_finished) {
    if (on && n < 19) {
      cudaEventRecord(c->sev[n + 1], s);
      stage[n++] = stage_just_finished;
    }
  }
  void collect() {
    for (int m = 0; m < n; ++m) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, c->sev[m], c->sev[m + 1]) == cudaSuccess) {
        c->stage_ms[stage[m]] += ms;
        c->stage_calls[stage[m]] += 1;
      }
    }
  }
};

// Where the back half of a scan runs: the ray walk and block creation on `walk`, the record sort on `sort`,
// the apply kernels on `apply`.  A stage on another stream than the one before it waits for the hand-off
// event (`walked`, `sorted`); synchronous calls run all three on the main stream without hand-off events.
struct Stages {
  cudaStream_t walk, sort, apply;
  cudaEvent_t walked, sorted;
};

// the map's tables as one scan's kernels see them: with the hand-off set's own touched-block list
Tables scan_tables(const vbx_ctx* c, const vbx_ctx::ScratchSet& S) {
  Tables t = c->tab;
  t.touched_list = S.touched_list;
  return t;
}
}  // namespace

// The engine's own stable radix sort (vbx_sort.cuh): one launch on stream s.  n lives on the device (d_n) or
// is n_fixed; n_hint sizes the grid (tiles are handed out by ticket, so any grid sorts any n).  result_in_a: the
// sorted pairs end in buffer A whatever the number of passes (otherwise SortPlan::final_buf says where they are).
template <typename KeyT>
static int own_sort(vbx_ctx* c, cudaStream_t s, SortPlan* plan, uint32_t* status, uint32_t tiles_cap, KeyT* keys_a,
                    uint32_t* vals_a, KeyT* keys_b, uint32_t* vals_b, const unsigned long long* d_n, uint32_t n_fixed,
                    uint64_t n_hint, int key_bits, bool result_in_a, uint64_t* launches,
                    const uint32_t* d_key_bits = nullptr, bool plan_cleared = false) {
  const int passes = std::min(kMaxPasses, (key_bits + 7) / 8);
  if (!plan_cleared) VBX_CUDA(c, cudaMemsetAsync(plan, 0, sizeof(SortPlan), s));  // (else: an earlier kernel of the stream did)
  const uint64_t tiles_hint = std::max<uint64_t>(1, (n_hint + kSortTile - 1) / kSortTile);
  const unsigned int grid = (unsigned int)std::min<uint64_t>(std::min<uint64_t>(tiles_cap, tiles_hint), (uint64_t)c->grid_sms * 2);
  k_sort<KeyT><<<grid, kSortThreads, 0, s>>>(keys_a, vals_a, keys_b, vals_b, d_n, n_fixed, passes, d_key_bits, plan, status,
                                              tiles_cap, result_in_a ? 1 : 0);
  *launches += 1;
  return VBX_OK;
}

// k_order_prefix, k_order_heads, k_bundle_order on stream `so` (see the kernels).
constexpr int kOrderGrid = 32;  // blocks of the cooperative k_bundle_order launch (only large maps use more than one)
// The shared memory asked for is what the bundle count of recent scans needs (plus a margin), not the whole
// SM: a block that wants 200 KB can only start on an SM that holds nothing else, and in the pipelined path
// -- every SM busy with other scans' kernels -- it waits for one to drain.  A scan with more bundles than the
// request covers is still ordered correctly: the kernel falls back to its global-memory stages.
template <typename KeyT>
static int launch_bundle_order(vbx_ctx* c, vbx_ctx::ScratchSet& S, vbx_ctx::FrontLane& F, cudaStream_t so,
                               const ScanParams& P, const KeyT* keys, const uint32_t* vals) {
  k_order_prefix<<<1, kOrderThreads, 0, so>>>(P.n, F.first_bits, F.order_scratch, S.d_state);
  k_order_heads<KeyT><<<std::min<unsigned int>(grid_for(P.n, 256), 148 * 2), 256, 0, so>>>(
      P, keys, vals, c->order_inv, S.head_list, F.first_bits, F.order_scratch, S.d_state);
  RehashSchedule rs = c->rehash;
  size_t smem_bytes = c->order_smem_bytes;
  unsigned int grid = kOrderGrid;
  if (c->bundle_hint) {
    const uint32_t B = (uint32_t)std::min<uint64_t>(c->bundle_hint + c->bundle_hint / 4 + 512, P.n);
    uint32_t nf = 1;
    for (int k = 0; k < rs.count && rs.m[k] < B; ++k) nf = rs.n[k];
    const uint32_t words = order_smem_words_needed(B, nf);
    const size_t need = ((size_t)words * 4 + 1023) & ~(size_t)1023;
    if (words != 0xffffffffu && need <= c->order_smem_bytes) {
      smem_bytes = need;
      grid = 1;  // the single-block form; block 0 is the only one that would work
    }
  }
  OrderScratch g = F.order_scratch;
  uint32_t smem_words = (uint32_t)(smem_bytes / 4);
  uint32_t* ray_list = S.ray_list;
  uint32_t* cta_tot = F.order_scratch.cta_tot;
  ScanState* st = S.d_state;
  void* args[] = {&rs, &g, &smem_words, &ray_list, &cta_tot, &st};
  if (grid == 1) {
    // an ordinary launch: nothing about it has to be co-scheduled
    k_bundle_order<<<1, kOrderThreads, smem_bytes, so>>>(rs, g, smem_words, ray_list, cta_tot, st);
  } else {
    VBX_CUDA(c, cudaLaunchCooperativeKernel((void*)k_bundle_order, dim3(grid), dim3(kOrderThreads), args, smem_bytes, so));
  }
  return VBX_OK;
}

// Stages up to and including k_assign: everything that decides WHICH voxels are updated.
template <typename KeyT>
static int front_half(vbx_ctx* c, vbx_ctx::ScratchSet& S, vbx_ctx::FrontLane& F, cudaStream_t s, ScanParams& P,
                      const float* d_xyz, const uint8_t* d_rgba, const uint32_t* order, Marks& mk, uint64_t* launches,
                      const KeyT** keys_out) {
  const uint32_t n = P.n;
  const int TB = 256;
  const Tables tab = scan_tables(c, S);
  const KeyT* keys = nullptr;
  const uint32_t* vals = nullptr;
  const uint32_t* scan_perm = nullptr;
  const uint32_t* scan_limit = nullptr;
  if (P.kind == VBX_MERGED) {
    KeyT* k0 = reinterpret_cast<KeyT*>(S.pkeys0);
    KeyT* k1 = reinterpret_cast<KeyT*>(F.pkeys1);
    k_point_bounds<<<std::min<unsigned int>(grid_for(n, TB), 148 * 4), TB, 0, s>>>(
        P, d_xyz, F.first_bits, F.sort_plan0, F.scan_status, (n + 1 + kScanTile - 1) / kScanTile + 1, S.d_state);
    k_point_keys<KeyT><<<grid_for(n, TB), TB, 0, s>>>(P, d_xyz, order, k0, F.pvals[0], S.d_state);
    mk.mark(0);
    // the bits in use are known on the device only (ScanState::key_bits): passes beyond them exit at once
    if (int rc = own_sort<KeyT>(c, s, F.sort_plan0, F.sort_status0, c->sort_tiles_cap[0], k0, F.pvals[0], k1, F.pvals[1],
                                nullptr, n, n, 8 * (int)sizeof(KeyT), true, launches, &S.d_state->key_bits,
                                /*plan_cleared=*/true)) {
      return rc;
    }
    keys = k0;
    vals = F.pvals[0];
    mk.mark(1);
    k_heads<KeyT><<<grid_for((uint64_t)n + 1, TB), TB, 0, s>>>(P, keys, vals, c->order_inv, S.head_list, F.big_list,
                                                               F.first_bits, S.cnt, S.d_state);
    // The reference's bundle order (ray_list[rank] = bundle id, vbx_order.cuh) is one thread block's work
    // and the fold (k_merge) does not need it: the two run side by side.  (With stage profiling on they
    // run one after the other so that each gets its own time.)
    cudaStream_t so = mk.on ? s : F.side;
    if (so != s) {
      VBX_CUDA(c, cudaEventRecord(F.ev_fork, s));
      VBX_CUDA(c, cudaStreamWaitEvent(so, F.ev_fork, 0));
    }
    if (int rc = launch_bundle_order<KeyT>(c, S, F, so, P, keys, vals)) return rc;
    if (so != s) VBX_CUDA(c, cudaEventRecord(F.ev_join, so));
    mk.mark(12);
    k_merge<KeyT><<<c->grid_sms * 4, 192, 0, s>>>(P, d_xyz, d_rgba, keys, vals, S.head_list, F.big_list, S.ray_p, S.ray_a,
                                           S.ray_c, S.cnt, S.d_state);
    mk.mark(8);
    *launches += 8;
    if (!P.single_walk) {
      // the bundle count is only known on the device: launch for the worst case (every
      // point its own bundle); surplus threads exit on the first load
      k_rays_count<KeyT><<<grid_for(n, 128), 128, 0, s>>>(P, tab, d_xyz, d_rgba, order, keys, S.head_list,
                                                           S.ray_p, S.ray_a, S.ray_c, S.cnt, c->set_start,
                                                           c->set_observed, S.d_state);
      *launches += 1;
    }
    if (so != s) VBX_CUDA(c, cudaStreamWaitEvent(s, F.ev_join, 0));
    // record offsets in RANK order: off[rank] = sum of cnt[ray_list[r]] over r < rank
    scan_perm = S.ray_list;
    scan_limit = &S.d_state->n_ray_list;
  } else {
    k_rays_count<KeyT><<<grid_for((uint64_t)n + 1, 128), 128, 0, s>>>(P, tab, d_xyz, d_rgba, order, keys,
                                                                       S.head_list, S.ray_p, S.ray_a, S.ray_c, S.cnt,
                                                                       c->set_start, c->set_observed, S.d_state);
    *launches += 1;
  }
  mk.mark(2);
  {
    // record offsets; the scan's last position also settles the call's update count (total_found, total_updates,
    // kErrUpdatesFull: too many for one pass; nothing downstream runs on a call that failed)
    const uint32_t tiles = (n + 1 + kScanTile - 1) / kScanTile;
    if (P.kind != VBX_MERGED) VBX_CUDA(c, cudaMemsetAsync(F.scan_status, 0, (size_t)(tiles + 1) * sizeof(uint32_t), s));  // (Merged: k_point_bounds did)
    k_exclusive_scan<<<std::min<uint32_t>(tiles, 148 * 4), kSortThreads, 0, s>>>(
        S.cnt, scan_perm, scan_limit, S.off, n + 1, F.scan_status + 1, F.scan_status, &S.d_state->total_found,
        &S.d_state->total_updates, &S.d_state->error, (unsigned long long)c->max_updates, kErrUpdatesFull);
  }
  mk.mark(3);
  *launches += 1;
  *keys_out = keys;
  return VBX_OK;
}

// update-record sort + the apply kernels
static int sort_and_apply(vbx_ctx* c, vbx_ctx::ScratchSet& S, const Stages& st, const ScanParams& P, unsigned long long K,
                          uint32_t n_touched, Marks& mk, uint64_t* launches) {
  RecordView rv;
  {
    // K and the number of touched blocks are only known on the device: sort on every bit a
    // record key can have; passes whose digit is uniform are skipped on the device
    const int key_bits = 32;
    if (st.walked) {
      // pipelined submission: the record sort works on buffers private to this scan, so it leaves
      // the walk stream (which the next scan's ray walk is waiting for)
      VBX_CUDA(c, cudaEventRecord(st.walked, st.walk));
      VBX_CUDA(c, cudaStreamWaitEvent(st.sort, st.walked, 0));
    }
    if (int rc = own_sort<uint32_t>(c, st.sort, S.sort_plan1, S.sort_status1, c->sort_tiles_cap[1], S.ckeys[0], S.cvals[0],
                                     S.ckeys[1], S.cvals[1], &S.d_state->total_updates, 0, c->record_hint, key_bits, false,
                                     launches, &S.d_state->rec_key_bits, /*plan_cleared=*/true)) {
      return rc;
    }
    rv.keys[0] = S.ckeys[0];
    rv.keys[1] = S.ckeys[1];
    rv.vals[0] = S.cvals[0];
    rv.vals[1] = S.cvals[1];
    rv.plan = S.sort_plan1;
    rv.d_total = &S.d_state->total_updates;
    rv.total_fixed = 0;
  }
  mk.mark(6);
  if (st.sorted) {
    // pipelined submission: the apply kernels run on their own stream behind the sort, so the
    // next scan's ray walk can start while this scan's voxels are still being written
    VBX_CUDA(c, cudaEventRecord(st.sorted, st.sort));
    VBX_CUDA(c, cudaStreamWaitEvent(st.apply, st.sorted, 0));
  }
  cudaStream_t s = st.apply;
  const Tables tab = scan_tables(c, S);
  const unsigned int g_short = c->grid_sms * 8;
  LongRuns lr;
  lr.start = c->long_list;
  lr.end = c->long_end;
  lr.state = c->long_state;
  lr.item_run = c->verify_run;
  lr.item_start = c->verify_start;
  lr.rec_sdf = c->rec_sdf;
  lr.rec_w = c->rec_w;
  k_apply_short<<<g_short, 256, 0, s>>>(P, tab, rv, S.ray_a, S.ray_c, lr, S.d_state);
  k_apply_verify<<<c->grid_sms * 8, 128, 0, s>>>(P, tab, rv, S.ray_a, S.ray_c, lr, S.d_state);
  k_apply_long<<<c->grid_sms * 4, 128, 0, s>>>(P, tab, rv, S.ray_a, S.ray_c, lr, S.d_state);
  mk.mark(7);
  *launches += 3;
  return VBX_OK;
}

template <typename KeyT>
static int back_half(vbx_ctx* c, vbx_ctx::ScratchSet& S, const Stages& st, const ScanParams& P, const KeyT* keys,
                     unsigned long long K, uint32_t n_touched, Marks& mk, uint64_t* launches) {
  cudaStream_t s = st.walk;
  const uint32_t n = P.n;
  const Tables tab = scan_tables(c, S);
  if (P.kind == VBX_MERGED && P.single_walk) {
    // a few thousand bundles of 100-300 steps: one warp per ray
    k_rays_emit_warp<KeyT><<<c->grid_sms * 8, 128, 0, s>>>(P, tab, keys, S.ray_list, S.head_list, S.ray_p, S.cnt, S.off,
                                                   S.ckeys[0], S.cvals[0], S.d_state);
  } else {
    k_rays_emit<KeyT><<<grid_for(n, 128), 128, 0, s>>>(P, tab, keys, S.ray_list, S.head_list, S.ray_p, S.cnt, S.off,
                                                        S.ckeys[0], S.cvals[0], S.d_state);
  }
  mk.mark(5);
  k_assign<<<grid_for(std::max<uint32_t>(c->tab.max_blocks, 1024), 256), 256, 0, s>>>(
      tab, c->d_nblocks + c->nb_cur, c->d_nblocks + (c->nb_cur ^ 1), S.sort_plan1, S.d_state);
  c->nb_cur ^= 1;
  mk.mark(4);
  *launches += 2;
  return sort_and_apply(c, S, st, P, K, n_touched, mk, launches);
}

// The back half of a call whose K exceeds max_updates_per_pass, in passes (see integrate_device).
template <typename KeyT>
static int apply_in_passes(vbx_ctx* c, vbx_ctx::ScratchSet& S, const Stages& st, ScanParams P, const KeyT* keys, Marks& mk,
                           uint64_t* launches) {
  cudaStream_t s = st.walk;
  const uint32_t n = P.n;
  std::vector<uint32_t> off(n + 1);
  VBX_CUDA(c, cudaMemcpyAsync(off.data(), S.off, (size_t)(n + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  if (P.kind == VBX_MERGED) {
    // the scan wrote the offsets of the bundles and, at [n], the total; ranks past the last bundle hold nothing
    const uint32_t nr = std::min(S.h_state->n_ray_list, n);
    for (uint32_t i = nr + 1; i < n; ++i) off[i] = off[n];
  }
  uint32_t lo = 0, passes = 0;
  while (lo < n) {
    // the longest slot range starting at lo whose records fit
    const uint64_t room = (uint64_t)off[lo] + c->max_updates;
    uint32_t hi = (uint32_t)(std::upper_bound(off.begin() + lo, off.end(), room,
                                              [](uint64_t v, uint32_t o) { return v < (uint64_t)o; }) -
                             off.begin());
    hi = hi > 0 ? hi - 1 : 0;  // off[hi] <= room
    if (hi <= lo) return fail(c, VBX_E_CAPACITY, "a single ray has more updates than max_updates_per_pass");
    const unsigned long long kp = (unsigned long long)off[hi] - off[lo];
    if (kp > 0) {
      P.emit_lo = lo;
      P.emit_hi = hi;
      P.emit_base = off[lo];
      k_pass_begin<<<1, 1, 0, s>>>(S.d_state, kp);
      *launches += 1;
      if (int rc = back_half<KeyT>(c, S, st, P, keys, kp, 0, mk, launches)) return rc;
      ++passes;
    }
    lo = hi;
  }
  c->last_passes = passes;
  return VBX_OK;
}

static void fill_params(vbx_ctx* c, int kind, const float q[4], const float t[3], uint32_t n, int freespace,
                        ScanParams& P) {
  const vbx_tsdf_config& cfg = c->cfg;
  std::memset(&P, 0, sizeof(P));
  P.T.w = q[0];
  P.T.x = q[1];
  P.T.y = q[2];
  P.T.z = q[3];
  P.T.t = f3(t[0], t[1], t[2]);
  P.origin = P.T.t;  // T_G_C.getPosition()
  P.voxel_size = c->voxel_size;
  P.voxel_size_inv = c->voxel_size_inv;
  P.trunc = cfg.default_truncation_distance;
  P.min_ray = cfg.min_ray_length_m;
  P.max_ray = cfg.max_ray_length_m;
  P.up.trunc = cfg.default_truncation_distance;
  P.up.max_weight = cfg.max_weight;
  P.up.voxel_size = c->voxel_size;
  P.up.use_weight_dropoff = cfg.use_weight_dropoff;
  P.up.use_sparsity = cfg.use_sparsity_compensation_factor;
  P.up.sparsity_factor = cfg.sparsity_compensation_factor;
  P.L = c->L;
  P.kind = kind;
  P.freespace = freespace;
  P.use_const_weight = cfg.use_const_weight;
  P.allow_clear = cfg.allow_clear;
  P.carving = cfg.voxel_carving_enabled;
  P.anti_grazing = cfg.enable_anti_grazing;
  P.order_mode = cfg.integration_order_mode;
  P.n = n;
  P.n_groups = n / 1024u;
  P.start_inv = cfg.start_voxel_subsampling_factor * c->voxel_size_inv;
  P.max_collisions = cfg.max_consecutive_ray_collisions;
  P.max_updates = c->max_updates;
  c->epoch += 1;
  P.epoch = c->epoch;
  if (kind == VBX_FAST) {
    // resetApproxSet every clear_checks_every_n_frames calls (cc:563-568)
    if ((++c->fast_reset_counter) >= cfg.clear_checks_every_n_frames) {
      c->fast_reset_counter = 0;
      c->set_epoch += 1;
    }
  }
  P.set_epoch = c->set_epoch;
  P.own_world = c->opt.world_size > 1 ? c->opt.world_size : 1;
  P.own_rank = c->opt.rank;
  P.emit_lo = 0;
  P.emit_hi = 0xffffffffu;
  P.emit_base = 0;
  P.single_walk = (kind != VBX_FAST && !(kind == VBX_MERGED && cfg.enable_anti_grazing)) ? 1 : 0;
}

int integrate_device(vbx_ctx* c, int kind, const float q[4], const float t[3], const float* d_xyz,
                     const uint8_t* d_rgba, uint64_t n64, int freespace) {
  if (kind < VBX_SIMPLE || kind > VBX_FAST) return fail(c, VBX_E_INVALID, "Unknown TSDF integrator type");
  if (n64 > c->max_points) return fail(c, VBX_E_CAPACITY, "cloud larger than max_points_per_scan");
  const uint32_t n = (uint32_t)n64;
  // synchronous calls work on hand-off set 0 and front lane 0, every stage on the main stream
  vbx_ctx::ScratchSet& S = c->set[0];
  vbx_ctx::FrontLane& F = c->lane[0];
  cudaStream_t s = c->stream_main;
  const Stages st{s, s, s, nullptr, nullptr};
  const vbx_tsdf_config& cfg = c->cfg;
  std::memset(c->counters, 0, sizeof(c->counters));
  uint64_t launches = 0;

  ScanParams P;
  fill_params(c, kind, q, t, n, freespace, P);

  VBX_CUDA(c, cudaEventRecord(c->ev0, s));
  VBX_CUDA(c, cudaMemsetAsync(S.d_state, 0, sizeof(ScanState), s));
  if (n == 0) {
    VBX_CUDA(c, cudaEventRecord(c->ev1, s));
    VBX_CUDA(c, cudaStreamSynchronize(s));
    c->last_ms = 0.f;
    return VBX_OK;
  }
  const int TB = 256;
  Marks mk{c, s, c->profiling};
  mk.begin();

  const uint32_t* order = nullptr;
  if (cfg.integration_order_mode == 1) {
    // SortedThreadSafeIndex: ascending |p|^2 (stable here; std::sort leaves ties unspecified)
    k_sqnorm_keys<<<grid_for(n, TB), TB, 0, s>>>(n, d_xyz, S.pkeys0, F.pvals[0]);
    if (int rc = own_sort<uint64_t>(c, s, F.sort_plan0, F.sort_status0, c->sort_tiles_cap[0], S.pkeys0, F.pvals[0], F.pkeys1,
                                    F.pvals[1], nullptr, n, n, 64, true, &launches)) {
      return rc;
    }
    VBX_CUDA(c, cudaMemcpyAsync(c->order, F.pvals[0], n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
    k_invert_order<<<grid_for(n, TB), TB, 0, s>>>(n, c->order, c->order_inv);
    order = c->order;
    launches += 2;
  }

  uint32_t chunk_blocks_before = 0;
  bool chunked = false;
  const uint64_t* keys64 = nullptr;
  unsigned long long K = 0;
  uint32_t n_touched = 0;
  if (int rc = front_half<uint64_t>(c, S, F, s, P, d_xyz, d_rgba, order, mk, &launches, &keys64)) return rc;
  {
    // own sort: K stays on the device, the whole call is enqueued without a host round trip
    if (int rc = back_half<uint64_t>(c, S, st, P, keys64, 0, 0, mk, &launches)) return rc;
    VBX_CUDA(c, cudaEventRecord(c->ev1, s));
    VBX_CUDA(c, cudaMemcpyAsync(S.h_state, S.d_state, sizeof(ScanState), cudaMemcpyDeviceToHost, s));
    VBX_CUDA(c, cudaStreamSynchronize(s));
    if (S.h_state->error == kErrUpdatesFull) {
      // More update records than one pass holds.  Nothing was emitted or applied; the per-ray
      // tables, counts and offsets of the front half stand.  Apply the call in passes over
      // contiguous ray-slot ranges: every voxel still sees its updates in ray-rank order, so
      // the result is the one-pass result bit for bit.
      chunk_blocks_before = c->n_blocks;
      if (int rc = apply_in_passes<uint64_t>(c, S, st, P, keys64, mk, &launches)) return rc;
      chunked = true;
      VBX_CUDA(c, cudaEventRecord(c->ev1, s));
      VBX_CUDA(c, cudaMemcpyAsync(S.h_state, S.d_state, sizeof(ScanState), cudaMemcpyDeviceToHost, s));
      VBX_CUDA(c, cudaStreamSynchronize(s));
    }
    if (int rc = check_state_errors(c, *S.h_state)) return rc;
    c->n_blocks = S.h_state->n_blocks;
    K = S.h_state->total_found;
    n_touched = S.h_state->n_touched;
  }
  VBX_CUDA(c, cudaEventRecord(c->ev1, s));
  VBX_CUDA(c, cudaMemcpyAsync(S.h_state, S.d_state, sizeof(ScanState), cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  VBX_CUDA(c, cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
  mk.collect();
  c->launches += launches;
  c->counters[0] = S.h_state->n_rays;
  if (kind == VBX_MERGED) c->bundle_hint = std::max(S.h_state->n_rays, S.h_state->n_clear_rays);
  c->counters[1] = S.h_state->n_clear_rays;
  c->counters[2] = K;
  if (K) c->record_hint = K;
  c->counters[3] = S.h_state->n_voxels;
  c->counters[4] = n_touched;
  c->counters[5] = chunked ? (uint64_t)(c->n_blocks - chunk_blocks_before) : (uint64_t)S.h_state->n_new;
  c->counters[11] = chunked ? c->last_passes : 1;
  c->counters[9] = S.h_state->n_refold;
  c->counters[10] = S.h_state->refold_members;
  c->counters[12] = S.h_state->key_bits;
  c->counters[6] = (kind == VBX_MERGED) ? S.h_state->n_valid_points
                                        : (uint64_t)S.h_state->n_rays + S.h_state->n_clear_rays;
  c->counters[7] = launches;
  return VBX_OK;
}

// ------------------------------------------------------------- asynchronous submission
// integratePointCloud without the host round trip: the call enqueues the scan and returns.  A scan
// passes through three stages on separate streams:
//   front   keys, bundle sort, bundle fold, record offsets -- touches nothing of the map; two front
//           lanes alternate, so two front halves can run side by side
//   walk    ray walk with block creation, slot assignment (stream_e)
//   sort    record sort on scan-private buffers (two sort streams alternate)
//   apply   the per-voxel updates (main stream)
// Stages that touch the map run in submission order (one stream each; the walk of scan i+1 only
// inserts new hash entries and never moves existing ones, so it can overlap the apply of scan i).
// Up to kSets scans are in flight, each with its own hand-off buffers; results (counters, errors)
// of a scan are collected when its set is reused or at the next synchronous call / vbx_sync.
int integrate_async(vbx_ctx* c, int kind, const float q[4], const float t[3], const float* xyz, const uint8_t* rgba,
                    uint64_t n64, int freespace, int on_device) {
  if (kind < VBX_SIMPLE || kind > VBX_FAST) return fail(c, VBX_E_INVALID, "Unknown TSDF integrator type");
  if (n64 > c->max_points) return fail(c, VBX_E_CAPACITY, "cloud larger than max_points_per_scan");
  const vbx_tsdf_config& cfg = c->cfg;
  const bool overlappable = kind != VBX_FAST && !(kind == VBX_MERGED && cfg.enable_anti_grazing) &&
                            cfg.integration_order_mode == 0 && n64 > 0;
  if (!overlappable) {
    // configurations whose front half touches the map or the Fast integrator's sets run in order
    if (int rc = drain_async(c)) return rc;
    const float* dx = xyz;
    const uint8_t* dr = rgba;
    if (!on_device && n64) {
      vbx_ctx::ScratchSet& S0 = c->set[0];
      VBX_CUDA(c, cudaMemcpyAsync(S0.d_xyz, xyz, n64 * 3 * sizeof(float), cudaMemcpyHostToDevice, c->stream_main));
      VBX_CUDA(c, cudaMemcpyAsync(S0.d_rgba, rgba, n64 * 4, cudaMemcpyHostToDevice, c->stream_main));
      dx = S0.d_xyz;
      dr = S0.d_rgba;
    }
    return integrate_device(c, kind, q, t, dx, dr, n64, freespace);
  }
  if (int rc = ensure_async(c)) return rc;
  const uint32_t n = (uint32_t)n64;
  vbx_ctx::ScratchSet& S = c->set[c->async_seq % c->sets_in_use];
  vbx_ctx::FrontLane& F = c->lane[c->async_seq % c->lanes_in_use];
  const auto t_enter = std::chrono::steady_clock::now();
  if (S.in_flight) {  // bounded run-ahead: wait for the scan that used this hand-off set
    VBX_CUDA(c, cudaEventSynchronize(S.back_done));
    c->async_wait_ns += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t_enter).count();
    harvest_async(c, S);
    if (S.redo) {
      // it (and every scan queued behind it) did not run its back half: redo them now, in order
      if (int rc = drain_async(c)) return rc;
    }
  }
  ScanParams P;
  fill_params(c, kind, q, t, n, freespace, P);
  uint64_t launches = 0;
  Marks mk{c, F.stream, false};  // no stage profiling: the events would serialise the streams
  // ---- front half on this scan's front lane
  const float* dx = xyz;
  const uint8_t* dr = rgba;
  if (!on_device) {
    // the copy engine works ahead of the front half on a stream of its own
    // (two copy streams alternate, so two scans' clouds can be in flight on the copy engines at once)
    cudaStream_t sc = (c->async_seq & 1u) ? c->stream_c2 : c->stream_c;
    if (cudaMemcpyAsync(S.d_xyz, xyz, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, sc) != cudaSuccess ||
        cudaMemcpyAsync(S.d_rgba, rgba, (size_t)n * 4, cudaMemcpyHostToDevice, sc) != cudaSuccess ||
        cudaEventRecord(S.copy_done, sc) != cudaSuccess ||
        cudaStreamWaitEvent(F.stream, S.copy_done, 0) != cudaSuccess) {
      return fail(c, VBX_E_CUDA, "asynchronous host-to-device copy failed");
    }
    dx = S.d_xyz;
    dr = S.d_rgba;
  }
  const uint64_t* keys64 = nullptr;
  if (cudaMemsetAsync(S.d_state, 0, sizeof(ScanState), F.stream) != cudaSuccess) return fail(c, VBX_E_CUDA, "cudaMemsetAsync");
  if (c->timeline) cudaEventRecord(S.front_start, F.stream);
  if (int rc = front_half<uint64_t>(c, S, F, F.stream, P, dx, dr, nullptr, mk, &launches, &keys64)) return rc;
  if (cudaEventRecord(S.front_done, F.stream) != cudaSuccess) return fail(c, VBX_E_CUDA, "cudaEventRecord");
  // ---- walk + record sort on stream_e, apply on the main stream
  if (cudaStreamWaitEvent(c->stream_e, S.front_done, 0) != cudaSuccess) return fail(c, VBX_E_CUDA, "cudaStreamWaitEvent");
  // Scans run their map-touching stages in submission order on this stream.  A scan that cannot be
  // applied asynchronously (more update records than one pass holds) raises the context's hold
  // flag here; every scan queued behind it then skips its back half, and the host redoes all of
  // them synchronously, in order, from the retained inputs (recover_async, vbx_capi.cu).
  k_back_begin<<<1, 1, 0, c->stream_e>>>(S.d_state, c->d_hold);
  launches += 1;
  const Stages st{c->stream_e, c->stream_s[c->async_seq % vbx_ctx::kSortStreams], c->stream_main, S.walked, S.sorted};
  if (int rc = back_half<uint64_t>(c, S, st, P, keys64, 0, 0, mk, &launches)) return rc;
  // the status block travels on a stream of its own: a copy between two scans' apply kernels would make the
  // apply stream (the pace setter of the pipeline) hop between the compute and the copy engine for every scan
  if (cudaEventRecord(S.applied, c->stream_main) != cudaSuccess || cudaStreamWaitEvent(c->stream_h, S.applied, 0) != cudaSuccess ||
      cudaMemcpyAsync(S.h_state, S.d_state, sizeof(ScanState), cudaMemcpyDeviceToHost, c->stream_h) != cudaSuccess ||
      cudaEventRecord(S.back_done, c->stream_h) != cudaSuccess) {
    return fail(c, VBX_E_CUDA, "enqueueing the result read-back failed");
  }
  S.in_flight = true;
  S.kind = kind;
  S.launches = launches;
  S.seq = c->async_seq;
  S.redo = false;
  std::memcpy(S.q, q, sizeof(S.q));
  std::memcpy(S.t, t, sizeof(S.t));
  S.n = n64;
  S.freespace = freespace;
  S.in_xyz = dx;   // (the set's private copy of a host cloud, or the caller's device buffers)
  S.in_rgba = dr;
  c->async_submit_ns += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t_enter).count();
  c->launches += launches;
  c->async_seq += 1;
  if (c->deferred_rc) {
    const int rc = c->deferred_rc;
    c->err = c->deferred_msg;
    c->deferred_rc = 0;
    return rc;
  }
  return VBX_OK;
}

// ------------------------------------------------------------------ test hooks
// k_bundle_order on caller-supplied hashes (element e = e-th inserted key, hash hashes[e]): out[p] = the
// element at iteration position p.  tests/test_order_gpu.py compares it with a real std::unordered_map.
// force_global: pretend there is no shared memory, i.e. run every stage grid-wide on the global tables.
__global__ void k_debug_order_setup(OrderScratch g, uint32_t n, ScanState* st) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) g.head_of[e] = e;
  if (e == 0) {
    st->n_rays = n;
    st->n_clear_rays = 0;
  }
}

int debug_bundle_order(vbx_ctx* c, const uint32_t* hashes, uint32_t n, int force_global, uint32_t* out) {
  cudaStream_t s = c->stream_main;
  vbx_ctx::ScratchSet& S = c->set[0];
  const OrderScratch& g0 = c->lane[0].order_scratch;
  if (n > c->max_points) return fail(c, VBX_E_CAPACITY, "debug_bundle_order: n > max_points_per_scan");
  if (n == 0) return VBX_OK;
  VBX_CUDA(c, cudaMemsetAsync(S.d_state, 0, sizeof(ScanState), s));
  VBX_CUDA(c, cudaMemcpyAsync(g0.h, hashes, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  k_debug_order_setup<<<grid_for(n, 256), 256, 0, s>>>(g0, n, S.d_state);
  RehashSchedule rs = c->rehash;
  OrderScratch g = g0;
  uint32_t smem_words = force_global ? 0u : (uint32_t)(c->order_smem_bytes / 4);
  uint32_t* ray_list = S.ray_list;
  uint32_t* cta_tot = g0.cta_tot;
  ScanState* st = S.d_state;
  void* args[] = {&rs, &g, &smem_words, &ray_list, &cta_tot, &st};
  VBX_CUDA(c, cudaLaunchCooperativeKernel((void*)k_bundle_order, dim3(kOrderGrid), dim3(kOrderThreads), args,
                                          c->order_smem_bytes, s));
  VBX_CUDA(c, cudaMemcpyAsync(out, S.ray_list, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaMemcpyAsync(S.h_state, S.d_state, sizeof(ScanState), cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  if (S.h_state->error) return fail(c, VBX_E_CAPACITY, "debug_bundle_order: table capacity");
  return VBX_OK;
}

__global__ void k_iota(uint32_t* v, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) v[i] = i;
}

// Sorts n host keys with the engine's radix sort and returns the sorted keys and the permutation
// (tests/test_sort_gpu.py checks it against a stable host sort).  key_bytes 4 uses the update-
// record buffers with the count in device memory, 8 the point-key buffers with a host count.
int debug_sort(vbx_ctx* c, const void* keys, int key_bytes, uint32_t n, int key_bits, void* keys_out,
               uint32_t* vals_out) {
  cudaStream_t s = c->stream_main;
  vbx_ctx::ScratchSet& S = c->set[0];
  vbx_ctx::FrontLane& F = c->lane[0];
  uint64_t launches = 0;
  if (key_bytes == 4) {
    if (n > c->max_updates) return fail(c, VBX_E_CAPACITY, "debug_sort: n > max_updates_per_pass");
    VBX_CUDA(c, cudaMemcpyAsync(S.ckeys[0], keys, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    k_iota<<<148, 256, 0, s>>>(S.cvals[0], n);
    VBX_CUDA(c, cudaMemsetAsync(S.d_state, 0, sizeof(ScanState), s));
    const unsigned long long nn = n;
    VBX_CUDA(c, cudaMemcpyAsync(&S.d_state->total_updates, &nn, sizeof(nn), cudaMemcpyHostToDevice, s));
    if (int rc = own_sort<uint32_t>(c, s, S.sort_plan1, S.sort_status1, c->sort_tiles_cap[1], S.ckeys[0], S.cvals[0],
                                     S.ckeys[1], S.cvals[1], &S.d_state->total_updates, 0, n, key_bits, true, &launches)) {
      return rc;
    }
    VBX_CUDA(c, cudaMemcpyAsync(keys_out, S.ckeys[0], (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    VBX_CUDA(c, cudaMemcpyAsync(vals_out, S.cvals[0], (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  } else if (key_bytes == 8) {
    if (n > c->max_points) return fail(c, VBX_E_CAPACITY, "debug_sort: n > max_points_per_scan");
    VBX_CUDA(c, cudaMemcpyAsync(S.pkeys0, keys, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    k_iota<<<148, 256, 0, s>>>(F.pvals[0], n);
    if (int rc = own_sort<uint64_t>(c, s, F.sort_plan0, F.sort_status0, c->sort_tiles_cap[0], S.pkeys0, F.pvals[0], F.pkeys1,
                                     F.pvals[1], nullptr, n, n, key_bits, true, &launches)) {
      return rc;
    }
    VBX_CUDA(c, cudaMemcpyAsync(keys_out, S.pkeys0, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    VBX_CUDA(c, cudaMemcpyAsync(vals_out, F.pvals[0], (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  } else {
    return fail(c, VBX_E_INVALID, "debug_sort: key_bytes must be 4 or 8");
  }
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  return VBX_OK;
}

// exclusive prefix sum of n host uint32 through the engine's scan kernel
int debug_scan(vbx_ctx* c, const uint32_t* in, uint32_t n, uint32_t* out) {
  cudaStream_t s = c->stream_main;
  vbx_ctx::ScratchSet& S = c->set[0];
  uint32_t* scan_status = c->lane[0].scan_status;
  if (n > c->max_points + 1) return fail(c, VBX_E_CAPACITY, "debug_scan: n > max_points_per_scan + 1");
  VBX_CUDA(c, cudaMemcpyAsync(S.cnt, in, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  const uint32_t tiles = (n + kScanTile - 1) / kScanTile;
  VBX_CUDA(c, cudaMemsetAsync(scan_status, 0, (size_t)(tiles + 1) * sizeof(uint32_t), s));
  if (n) {
    k_exclusive_scan<<<std::min<uint32_t>(tiles, 148 * 4), kSortThreads, 0, s>>>(S.cnt, nullptr, nullptr, S.off, n,
                                                                               scan_status + 1, scan_status, nullptr,
                                                                               nullptr, nullptr, 0ull, 0u);
  }
  VBX_CUDA(c, cudaMemcpyAsync(out, S.off, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  return VBX_OK;
}

}  // namespace vbx
