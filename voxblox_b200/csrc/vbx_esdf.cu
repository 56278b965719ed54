// ESDF update on the device: EsdfIntegrator::updateFromTsdfLayer / ...Batch
// (voxblox/src/integrator/esdf_integrator.cc:94-530) over the same block hash and pool
// slots as the TSDF layer.
//
// The reference is a single-threaded queue algorithm: (1) a streaming pass classifies every
// voxel of every updated TSDF block against its stored ESDF voxel (new / lower / raise / sign
// flip, cc:136-287) and fills a FIFO raise queue and a bucketed open queue, (2) the raise
// queue invalidates the descendants of raised voxels through their parent pointers
// (cc:305-369), (3) the open queue relaxes 26-neighbourhoods until no distance can be lowered
// (cc:371-496).  On the device the three steps become
//   k_esdf_propagate   one thread per voxel of every listed block (streaming, coalesced)
//   k_esdf_seed        incremental only: updateVoxelFromNeighbors for new free voxels (cc:498-530)
//   k_esdf_raise       persistent cooperative kernel, level-synchronous BFS over the parent tree
//   k_esdf_lower       persistent cooperative kernel, wavefront relaxation with atomicMin on the
//                      distance word; one warp per frontier voxel, one lane per neighbour
//   k_esdf_parents     parent direction of every voxel the wavefront lowered, recomputed from the
//                      converged distances
// Distances are compared and lowered through their integer bit patterns: for two floats of the
// same sign the one nearer zero has the smaller signed-integer pattern, so "closer to the
// surface" is atomicMin on both sides of the surface.
//
// With min_diff_m = 0 (what the reference's own tests use, test_sdf_integrators.cc:200) the
// converged distances are the unique least fixed point of the relaxation rule and do not
// depend on visiting order; see DESIGN.md "ESDF" for what is and is not order dependent.
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "vbx_engine.h"
#include "vbx_hash.cuh"

namespace cg = cooperative_groups;

namespace vbx {

// src/utils/neighbor_tools.cc:24-30: 6 faces, 12 edges, 8 corners, in this order
__constant__ int8_t kOff[26][3] = {
    {-1, 0, 0},  {1, 0, 0},   {0, -1, 0},  {0, 1, 0},  {0, 0, -1},  {0, 0, 1},  {-1, -1, 0}, {-1, 1, 0}, {1, -1, 0},
    {1, 1, 0},   {0, -1, -1}, {0, -1, 1},  {0, 1, -1}, {0, 1, 1},   {-1, 0, -1}, {1, 0, -1}, {-1, 0, 1}, {1, 0, 1},
    {-1, -1, -1}, {-1, -1, 1}, {-1, 1, -1}, {-1, 1, 1}, {1, -1, -1}, {1, -1, 1}, {1, 1, -1},  {1, 1, 1}};

struct EsdfParams {
  int L;
  float voxel_size;
  float max_distance, min_distance, default_distance, min_diff, min_weight;
  int full_euclidean, multi_queue, add_occupied_crust;
  int incremental;
  float d1, d2, d3;  // kDistances * voxel_size (1, sqrtf(2), sqrtf(3)), neighbor_tools.cc:8-21
  float u1, u2, u3;  // kDistances unscaled (used by updateVoxelFromNeighbors, cc:508)
  uint32_t cap;      // frontier capacity
};

// the four bools of EsdfVoxel as bits of one word (each bool byte holds 0 or 1); kBitLowered is a
// scratch mark that lives only inside one update call
constexpr uint32_t kFlagObserved = 0x00000001u, kFlagHallucinated = 0x00000100u, kFlagInQueue = 0x00010000u,
                   kFlagFixed = 0x01000000u, kBitLowered = 0x00020000u;
constexpr uint32_t kBitObserved = kFlagObserved, kBitHallucinated = kFlagHallucinated, kBitInQueue = kFlagInQueue,
                   kBitFixed = kFlagFixed;

// EsdfVoxel viewed as five 32-bit words: distance, flags (4 bools), parent x, y, z
struct EsdfWords {
  float distance;
  uint32_t flags;
  int32_t px, py, pz;
};
static_assert(sizeof(EsdfWords) == sizeof(EsdfVoxel), "EsdfVoxel words");

__device__ __forceinline__ int signum_d(float v) { return (v == 0.0f) ? 0 : (v < 0.0f ? -1 : 1); }
__device__ __forceinline__ float nbr_dist(const EsdfParams& E, int i) { return i < 6 ? E.d1 : (i < 18 ? E.d2 : E.d3); }
__device__ __forceinline__ float nbr_dist_unscaled(const EsdfParams& E, int i) {
  return i < 6 ? E.u1 : (i < 18 ? E.u2 : E.u3);
}

// (slot, lin) of the neighbour of voxel (slot, lin) in direction i, or ~0 if its ESDF block does
// not exist (Layer::getVoxelPtrByGlobalIndex returning nullptr, core/layer.h:228-239)
__device__ __forceinline__ uint32_t neighbor_ref(const Tables& tab, int L, uint32_t ref, int i) {
  const uint32_t slot = ref >> (3 * L), lin = ref & ((1u << (3 * L)) - 1u);
  const int mask = (1 << L) - 1;
  int x = (int)(lin & mask) + kOff[i][0];
  int y = (int)((lin >> L) & mask) + kOff[i][1];
  int z = (int)(lin >> (2 * L)) + kOff[i][2];
  uint32_t nslot = slot;
  if ((x | y | z) & ~mask) {  // leaves the block
    int bx, by, bz;
    unpack3(tab.slot_key[slot], &bx, &by, &bz);
    bx += x >> L;
    by += y >> L;
    bz += z >> L;
    x &= mask;
    y &= mask;
    z &= mask;
    uint32_t hp = hash64(pack3(bx, by, bz)) & tab.hmask;
    nslot = 0xffffffffu;
    for (uint32_t probe = 0; probe <= tab.hmask; ++probe) {
      const uint64_t k = tab.hkeys[hp];
      if (k == pack3(bx, by, bz)) {
        nslot = (uint32_t)tab.hslot[hp];
        break;
      }
      if (k == kEmptyKey) break;
      hp = (hp + 1) & tab.hmask;
    }
    if (nslot == 0xffffffffu) return 0xffffffffu;
  }
  if (!tab.slot_has_esdf[nslot]) return 0xffffffffu;
  return (nslot << (3 * L)) | (uint32_t)(x | (y << L) | (z << (2 * L)));
}

// the wavefront changed a voxel of this block: mark it for the incremental host mirror (the reference flags only
// the blocks it propagates, cc:147; the blocks its queues reach stay unflagged there)
__device__ __forceinline__ void mark_mirror(const Tables& tab, int L, uint32_t ref) {
  uint8_t* f = tab.slot_esdf_updated + (ref >> (3 * L));
  if (!(*f & 8)) *f |= 8;  // (every concurrent writer stores the same bit)
}

__device__ __forceinline__ void push(uint32_t* list, uint32_t* count, uint32_t cap, uint32_t ref, ScanState* st) {
  const uint32_t j = atomicAdd(count, 1u);
  if (j < cap) {
    list[j] = ref;
  } else {
    atomicOr(&st->error, kErrUpdatesFull);
  }
}

// The level-synchronous kernels below keep THREE counters per queue and rotate through them: sweep k
// reads counter k % 3, appends to counter (k + 1) % 3 and zeroes counter (k + 2) % 3 (last read one
// sweep ago, next written one sweep ahead), so a sweep needs a single grid-wide barrier.
__device__ __forceinline__ uint32_t* frontier_cnt(ScanState* st, uint32_t k) {
  return k % 3u == 2u ? &st->frontier_n2 : &st->frontier_n[k % 3u];
}
__device__ __forceinline__ uint32_t* raise_cnt(ScanState* st, uint32_t k) {
  return k % 3u == 2u ? &st->raise_n2 : &st->raise_n[k % 3u];
}

// Step (1), esdf_integrator.cc:136-287, for ONE voxel: the stored ESDF voxel `ev` against its TSDF voxel `tv`.
// Returns false when the voxel is left alone (unobserved in the TSDF, cc:153-164); otherwise ev holds the new
// voxel and the flags say which queues it joins.  kind: 0 none, 1 lower, 2 raise, 3 new (the VLOG counters).
struct EsdfClass {
  bool to_open, to_raise, to_seed;
  int kind;
};
__device__ __forceinline__ bool esdf_classify(const EsdfParams& E, const TsdfVoxel& tv, EsdfWords& ev, EsdfClass& k) {
  k.to_open = k.to_raise = k.to_seed = false;
  k.kind = 0;
  if (tv.weight < E.min_weight) {  // unobserved in the TSDF, cc:153-164
    if (!E.incremental && E.add_occupied_crust) {
      ev.distance = -E.default_distance;
      ev.flags = (ev.flags & ~(kFlagObserved | kFlagHallucinated | kFlagFixed)) | kBitObserved | kBitHallucinated;
      return true;
    }
    return false;
  }
  const bool observed = (ev.flags & kFlagObserved) != 0, halluc = (ev.flags & kFlagHallucinated) != 0;
  bool fixed = (ev.flags & kFlagFixed) != 0, in_queue = (ev.flags & kFlagInQueue) != 0;
  const bool tfixed = fabsf(tv.distance) < E.min_distance;  // isFixed, esdf_integrator.h:131-133
  const float sgn_default = (float)signum_d(tv.distance) * E.default_distance;
  const float md = E.min_diff;
  bool reset_parent = false;
  if (!observed || halluc) {  // nothing there before, cc:174-200
    if (halluc) k.to_raise = true;
    if (tfixed) {
      ev.distance = tv.distance;
      fixed = true;
      k.to_open = true;
    } else {
      ev.distance = sgn_default;
      fixed = false;
      if (E.incremental) k.to_seed = true;
    }
    reset_parent = true;
    k.kind = 3;
  } else if (tfixed || fixed) {  // cc:211-262
    if (!tfixed) {
      ev.distance = sgn_default;
      reset_parent = true;
      fixed = false;
      k.to_raise = true;
      k.to_open = true;
      k.kind = 2;
    } else if ((ev.distance > 0.0f && tv.distance + md < ev.distance) ||
               (ev.distance <= 0.0f && tv.distance - md > ev.distance)) {
      fixed = tfixed;
      ev.distance = fixed ? tv.distance : sgn_default;
      reset_parent = true;
      k.to_open = true;
      k.kind = 1;
    } else if ((ev.distance > 0.0f && tv.distance - md > ev.distance) ||
               (ev.distance <= 0.0f && tv.distance + md < ev.distance)) {
      fixed = tfixed;
      ev.distance = fixed ? tv.distance : sgn_default;
      reset_parent = true;
      k.to_raise = true;
      k.to_open = true;
      k.kind = 2;
    }
  } else if (signum_d(tv.distance) != signum_d(ev.distance)) {  // cc:263-282
    if (tv.distance < ev.distance) {
      ev.distance = sgn_default;
      reset_parent = true;
      k.to_open = true;
      k.kind = 1;
    } else {
      ev.distance = sgn_default;
      reset_parent = true;
      k.to_raise = true;
      k.kind = 2;
    }
  }
  if (k.to_open) in_queue = true;
  if (reset_parent) ev.px = ev.py = ev.pz = 0;
  // esdf_voxel.observed = true; hallucinated = false, cc:285-286
  ev.flags = kBitObserved | (in_queue ? kBitInQueue : 0u) | (fixed ? kBitFixed : 0u);
  return true;
}

// one queue append per warp instead of one per voxel
__device__ __forceinline__ void push_warp(bool want, uint32_t* list, uint32_t* count, uint32_t cap, uint32_t ref, ScanState* st) {
  const unsigned m = __ballot_sync(0xffffffffu, want);
  if (!m) return;
  const int lane = threadIdx.x & 31;
  uint32_t base = 0;
  if (lane == __ffs(m) - 1) base = atomicAdd(count, (uint32_t)__popc(m));
  base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
  if (want) {
    const uint32_t j = base + (uint32_t)__popc(m & ((1u << lane) - 1u));
    if (j < cap) {
      list[j] = ref;
    } else {
      atomicOr(&st->error, kErrUpdatesFull);
    }
  }
}

// ---- TMA helpers (PTX: mbarrier + cp.async.bulk, the bulk-copy path of the tensor memory accelerator)
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared, completion signalled on the mbarrier (bytes: multiple of 16, both addresses 16-byte aligned)
__device__ __forceinline__ void tma_load_bulk(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_addr(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
// shared -> global
__device__ __forceinline__ void tma_store_bulk(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_addr(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit_and_wait() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Step (1) over every listed block: "HOT LOOP 1" of SURVEY.md 3.3 -- a stream of whole blocks, 12 B in and
// 20 B in/out per voxel.  One thread block per voxel block: the TSDF slab (48 KiB at 16^3) and the ESDF slab
// (80 KiB) are staged into shared memory by two TMA bulk copies, classified from there (every thread a few
// voxels), and the ESDF slab goes back with one bulk store.  Queue appends are warp-aggregated, the VLOG
// counters block-aggregated.  esdf_counts: [1] lower [2] raise [3] new.
__global__ void __launch_bounds__(1024)
k_esdf_propagate(EsdfParams E, Tables tab, const uint32_t* __restrict__ block_list, uint32_t n_blocks,
                 uint32_t* open_list, uint32_t* raise_list, uint32_t* seed_list, ScanState* st) {
  extern __shared__ __align__(128) unsigned char slab[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t s_cnt[4];
  const uint32_t vpb = 1u << (3 * E.L);
  if (blockIdx.x >= min(n_blocks, st->esdf_counts[0])) return;  // (n_blocks is the launch's upper bound)
  const uint32_t slot = block_list[blockIdx.x];
  TsdfVoxel* s_tsdf = reinterpret_cast<TsdfVoxel*>(slab);
  EsdfWords* s_esdf = reinterpret_cast<EsdfWords*>(slab + (size_t)vpb * sizeof(TsdfVoxel));
  EsdfWords* g_esdf = reinterpret_cast<EsdfWords*>(tab.esdf) + (size_t)slot * vpb;
  const uint32_t tsdf_bytes = vpb * (uint32_t)sizeof(TsdfVoxel), esdf_bytes = vpb * (uint32_t)sizeof(EsdfVoxel);
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_async_smem();
  }
  if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0u;
  __syncthreads();
  const bool bulk = (tsdf_bytes & 15u) == 0u && (esdf_bytes & 15u) == 0u;  // (not for one-voxel blocks)
  if (bulk) {
    if (threadIdx.x == 0) {
      mbar_expect_tx(&bar, tsdf_bytes + esdf_bytes);
      tma_load_bulk(s_tsdf, tab.tsdf + (size_t)slot * vpb, tsdf_bytes, &bar);
      tma_load_bulk(s_esdf, g_esdf, esdf_bytes, &bar);
    }
    mbar_wait(&bar, 0);
  } else {
    for (uint32_t lin = threadIdx.x; lin < vpb; lin += blockDim.x) {
      s_tsdf[lin] = tab.tsdf[(size_t)slot * vpb + lin];
      s_esdf[lin] = g_esdf[lin];
    }
    __syncthreads();
  }
  uint32_t n_kind[4] = {0, 0, 0, 0};
  for (uint32_t lin0 = 0; lin0 < vpb; lin0 += blockDim.x) {
    const uint32_t lin = lin0 + threadIdx.x;
    EsdfClass k;
    k.to_open = k.to_raise = k.to_seed = false;
    k.kind = 0;
    if (lin < vpb) {
      EsdfWords ev = s_esdf[lin];
      if (esdf_classify(E, s_tsdf[lin], ev, k)) s_esdf[lin] = ev;
      n_kind[k.kind] += 1;
    }
    const uint32_t ref = (slot << (3 * E.L)) | lin;
    push_warp(k.to_open, open_list, &st->frontier_n[0], E.cap, ref, st);
    push_warp(k.to_raise, raise_list, &st->raise_n[0], E.cap, ref, st);
    push_warp(k.to_seed, seed_list, &st->seed_n, E.cap, ref, st);
  }
#pragma unroll
  for (int q = 1; q < 4; ++q) {
    const uint32_t w = __reduce_add_sync(0xffffffffu, n_kind[q]);
    if ((threadIdx.x & 31) == 0 && w) atomicAdd(&s_cnt[q], w);
  }
  fence_async_smem();  // the slab written through the generic proxy is read by the bulk store (async proxy)
  __syncthreads();
  if (bulk) {
    if (threadIdx.x == 0) {
      tma_store_bulk(g_esdf, s_esdf, esdf_bytes);
      tma_store_commit_and_wait();
    }
  } else {
    for (uint32_t lin = threadIdx.x; lin < vpb; lin += blockDim.x) g_esdf[lin] = s_esdf[lin];
  }
  if (threadIdx.x >= 1 && threadIdx.x < 4 && s_cnt[threadIdx.x]) atomicAdd(&st->esdf_counts[threadIdx.x], s_cnt[threadIdx.x]);
}

// updateVoxelFromNeighbors (cc:498-530) for the new free-space voxels of an incremental update:
// first neighbour in table order that is observed, inside +-max_distance, of the same sign and
// closer; the distance added is the UNSCALED table entry (cc:508).  Candidates are read in
// their post-classification state (the reference sees neighbours seeded earlier in its own
// loop order as well; see DESIGN.md).
__global__ void k_esdf_seed(EsdfParams E, Tables tab, const uint32_t* __restrict__ seed_list, uint32_t* open_list,
                            float* seed_val, ScanState* st) {
  const uint32_t n = min(st->seed_n, E.cap);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t ref = seed_list[i];
    EsdfWords* ep = reinterpret_cast<EsdfWords*>(tab.esdf) + ref;
    const float d = ep->distance;
    float out = d;
    for (int k = 0; k < 26; ++k) {
      const uint32_t nref = neighbor_ref(tab, E.L, ref, k);
      if (nref == 0xffffffffu) continue;
      const EsdfWords* np = reinterpret_cast<const EsdfWords*>(tab.esdf) + nref;
      const uint32_t nf = np->flags;
      const float nd = np->distance;
      // a neighbour that is itself waiting to be seeded still holds +-default_distance
      if (!(nf & kFlagObserved) || nd >= E.max_distance || nd <= -E.max_distance) continue;
      if (signum_d(nd) == signum_d(d) && fabsf(nd) < fabsf(d)) {
        out = fadd(nd, fmul((float)signum_d(d), nbr_dist_unscaled(E, k)));
        // (the parent the reference assigns here is zeroed again right after, cc:199-200)
        atomicOr(&ep->flags, kBitInQueue);
        push(open_list, &st->frontier_n[0], E.cap, ref, st);
        break;
      }
    }
    // published by k_esdf_seed_commit so that no thread of this kernel reads a half-seeded neighbour
    seed_val[i] = out;
  }
}

__global__ void k_esdf_seed_commit(EsdfParams E, Tables tab, const uint32_t* __restrict__ seed_list,
                                   const float* __restrict__ seed_val, const ScanState* st) {
  const uint32_t n = min(st->seed_n, E.cap);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    (reinterpret_cast<EsdfWords*>(tab.esdf) + seed_list[i])->distance = seed_val[i];
  }
}

// Step (2), processRaiseSet cc:305-369: level-synchronous BFS.  One warp per raised voxel, one
// lane per neighbour.  A neighbour whose parent points back at the raised voxel is reset and
// raised in turn; any other observed, non-fixed neighbour joins the open set.
__global__ void k_esdf_raise(EsdfParams E, Tables tab, uint32_t* raise_a, uint32_t* raise_b, uint32_t* open_list,
                             ScanState* st) {
  cg::grid_group grid = cg::this_grid();
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t level = 0;; ++level) {
    uint32_t* in = (level & 1u) ? raise_b : raise_a;
    uint32_t* out = (level & 1u) ? raise_a : raise_b;
    const uint32_t n = min(__ldcg(raise_cnt(st, level)), E.cap);
    if (n == 0) break;
    uint32_t* out_n = raise_cnt(st, level + 1);
    if (blockIdx.x == 0 && threadIdx.x == 0) *raise_cnt(st, level + 2) = 0;
    for (uint32_t q = warp; q < n; q += n_warps) {
      const uint32_t ref = __ldcg(&in[q]);
      if (lane == 0) atomicAdd(&st->esdf_counts[4], 1u);
      if (lane < 26) {
        const uint32_t nref = neighbor_ref(tab, E.L, ref, lane);
        if (nref != 0xffffffffu) {
          EsdfWords* np = reinterpret_cast<EsdfWords*>(tab.esdf) + nref;
          const uint32_t nf = np->flags;
          if ((nf & kFlagObserved) && !(nf & kFlagFixed)) {
            bool is_parent = np->px == -kOff[lane][0] && np->py == -kOff[lane][1] && np->pz == -kOff[lane][2];
            if (E.full_euclidean) {  // cc:339-347
              const F3 pd = unit3(f3((float)np->px, (float)np->py, (float)np->pz));
              is_parent = (int)roundf(pd.x) == -kOff[lane][0] && (int)roundf(pd.y) == -kOff[lane][1] &&
                          (int)roundf(pd.z) == -kOff[lane][2];
            }
            if (is_parent) {
              np->distance = (float)signum_d(np->distance) * E.default_distance;
              np->px = np->py = np->pz = 0;
              mark_mirror(tab, E.L, nref);
              push(out, out_n, E.cap, nref, st);
            } else if (!(atomicOr(&np->flags, kBitInQueue) & kFlagInQueue)) {
              push(open_list, &st->frontier_n[0], E.cap, nref, st);
            }
          }
        }
      }
    }
    grid.sync();
  }
}

// Step (3), processOpenSet cc:371-496: wavefront relaxation.  One warp per frontier voxel, one
// lane per neighbour; a lowered neighbour joins the next frontier (once: the in_queue flag).
// A voxel leaves the queue (voxel->in_queue = false, cc:384) when its warp starts on it: the flag is
// cleared BEFORE the distance is read, so a neighbour that lowers this voxel either still sees the
// flag (then its lower value is the one read here) or re-queues the voxel for the next sweep.
__global__ void k_esdf_lower(EsdfParams E, Tables tab, uint32_t* front_a, uint32_t* front_b, uint32_t* touched_list,
                             ScanState* st) {
  cg::grid_group grid = cg::this_grid();
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t sweep = 0;; ++sweep) {
    uint32_t* in = (sweep & 1u) ? front_b : front_a;
    uint32_t* out = (sweep & 1u) ? front_a : front_b;
    const uint32_t n = min(__ldcg(frontier_cnt(st, sweep)), E.cap);
    if (n == 0) break;
    uint32_t* out_n = frontier_cnt(st, sweep + 1);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      *frontier_cnt(st, sweep + 2) = 0;
      atomicAdd(&st->esdf_counts[6], 1u);
    }
    for (uint32_t q = warp; q < n; q += n_warps) {
      const uint32_t ref = __ldcg(&in[q]);
      EsdfWords* vpm = reinterpret_cast<EsdfWords*>(tab.esdf) + ref;
      if (lane == 0) {
        atomicAnd(&vpm->flags, ~kBitInQueue);
        __threadfence();
      }
      __syncwarp();
      const EsdfWords* vp = vpm;
      const float vd = *reinterpret_cast<const volatile float*>(&vp->distance);
      const uint32_t vf = *reinterpret_cast<const volatile uint32_t*>(&vp->flags);
      if (!(vf & kFlagObserved) || vd >= E.max_distance || vd <= -E.max_distance) continue;  // cc:387-390
      if (lane >= 26) continue;
      const uint32_t nref = neighbor_ref(tab, E.L, ref, lane);
      if (nref == 0xffffffffu) continue;
      EsdfWords* np = reinterpret_cast<EsdfWords*>(tab.esdf) + nref;
      const uint32_t nf = *reinterpret_cast<const volatile uint32_t*>(&np->flags);
      if (!(nf & kFlagObserved) || (nf & kFlagFixed)) continue;  // cc:407-411
      float dist = nbr_dist(E, lane);
      if (E.full_euclidean) {  // cc:414-426
        const F3 npar = f3((float)(vp->px - kOff[lane][0]), (float)(vp->py - kOff[lane][1]),
                           (float)(vp->pz - kOff[lane][2]));
        dist = fmul(E.voxel_size, fsub(norm3(npar), norm3(f3((float)vp->px, (float)vp->py, (float)vp->pz))));
        if (dist < 0.0f) continue;
      }
      const float nd = *reinterpret_cast<const volatile float*>(&np->distance);
      bool changed = false;
      int* nbits = reinterpret_cast<int*>(&np->distance);
      if (vd > 0.0f && nd > 0.0f) {  // both outside, cc:429-443
        if (fadd(fadd(vd, dist), E.min_diff) < nd) {
          const float cand = fadd(vd, dist);
          changed = atomicMin(nbits, __float_as_int(cand)) > __float_as_int(cand);
        }
      } else if (vd <= 0.0f && nd <= 0.0f) {  // both inside, cc:444-457
        if (fsub(fsub(vd, dist), E.min_diff) > nd) {
          const float cand = fsub(vd, dist);
          changed = atomicMin(nbits, __float_as_int(cand)) > __float_as_int(cand);
        }
      } else {  // signs differ, cc:458-488 (incl. the sign-vs-distance comparison of cc:464)
        const float pot = fsub(vd, fmul((float)signum_d(vd), dist));
        if (fabsf(fsub(pot, nd)) > dist) {
          // The reference ASSIGNS sign(n) * dist here, so its result depends on which source it
          // pops first.  The device keeps the candidate nearest the surface (order free): the
          // assignment is applied only when it lowers |distance|.
          const float nv = ((float)signum_d(pot) == nd) ? pot : fmul((float)signum_d(nd), dist);
          if ((nv > 0.0f) == (nd > 0.0f)) {
            changed = atomicMin(nbits, __float_as_int(nv)) > __float_as_int(nv);
          }
        }
      }
      if (changed) {
        atomicAdd(&st->esdf_counts[5], 1u);
        mark_mirror(tab, E.L, nref);
        // neighbor_voxel->parent = new_parent (cc:436,450,470,481).  Written unguarded: when two
        // sources lower the same voxel in one sweep the last writer wins; k_esdf_parents then
        // re-derives the parent from the converged distances (quasi-Euclidean mode).
        if (E.full_euclidean) {
          np->px = vp->px - kOff[lane][0];
          np->py = vp->py - kOff[lane][1];
          np->pz = vp->pz - kOff[lane][2];
        } else {
          np->px = -kOff[lane][0];
          np->py = -kOff[lane][1];
          np->pz = -kOff[lane][2];
        }
        __threadfence();  // the lowered distance is visible before the queue flag is tested
        const uint32_t old = atomicOr(&np->flags, kBitInQueue | kBitLowered);
        if (!(old & kBitLowered)) push(touched_list, &st->lowered_n, E.cap, nref, st);
        if (E.multi_queue || !(old & kFlagInQueue)) push(out, out_n, E.cap, nref, st);
      }
    }
    grid.sync();
  }
}

// Parent direction of every voxel the wavefront lowered (quasi-Euclidean mode): the first
// neighbour in table order whose converged distance reproduces this voxel's distance through
// the relaxation rule.  (The reference stores the neighbour that happened to lower it last;
// with equal candidates that is its visiting order.)
__global__ void k_esdf_parents(EsdfParams E, Tables tab, const uint32_t* __restrict__ touched_list, ScanState* st) {
  const uint32_t n = min(st->lowered_n, E.cap);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t ref = touched_list[i];
    EsdfWords* ep = reinterpret_cast<EsdfWords*>(tab.esdf) + ref;
    atomicAnd(&ep->flags, ~kBitLowered);
    if (E.full_euclidean) continue;
    const float d = ep->distance;
    for (int k = 0; k < 26; ++k) {
      const uint32_t nref = neighbor_ref(tab, E.L, ref, k);
      if (nref == 0xffffffffu) continue;
      const EsdfWords* np = reinterpret_cast<const EsdfWords*>(tab.esdf) + nref;
      if (!(np->flags & kFlagObserved)) continue;
      const float nd = np->distance;
      if (nd >= E.max_distance || nd <= -E.max_distance) continue;
      const float dist = nbr_dist(E, k);
      const bool same = (d > 0.0f && nd > 0.0f && fadd(nd, dist) == d) || (d <= 0.0f && nd <= 0.0f && fsub(nd, dist) == d);
      const bool mixed = ((d > 0.0f) != (nd > 0.0f)) && fmul((float)signum_d(d), dist) == d;
      if (same || mixed) {
        // the voxel at offset k is a source of this distance; the parent points towards it
        ep->px = kOff[k][0];
        ep->py = kOff[k][1];
        ep->pz = kOff[k][2];
        break;
      }
    }
  }
}

// blocks to propagate: every TSDF block with the kEsdf bit or queued by addNewRobotPosition
// (updated_blocks_, cc:104-110) -- incremental -- or every TSDF block (batch).  Slots that hold an
// ESDF block only (kSlotNoTsdf) are skipped like the reference skips indices without a TSDF
// block (cc:137-141).
__global__ void k_esdf_block_list(Tables tab, uint32_t n_slots, int batch, uint32_t* block_list, ScanState* st) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const uint8_t u = tab.slot_updated[s];
  const uint8_t eu = tab.slot_esdf_updated[s];
  if (eu & kEsdfPending) tab.slot_esdf_updated[s] = eu & (uint8_t)~kEsdfPending;  // updated_blocks_.clear(), cc:99,109
  if (u & kSlotNoTsdf) return;
  if (batch || (u & VBX_UPDATED_ESDF) || (eu & kEsdfPending)) {
    block_list[atomicAdd(&st->esdf_counts[0], 1u)] = s;
    tab.slot_has_esdf[s] = 1;  // allocateBlockPtrByIndex in the ESDF layer, cc:143-146
    tab.slot_esdf_updated[s] = (tab.slot_esdf_updated[s] & kEsdfPending) | 9;  // esdf_block->set_updated(true): bitset(1) = kMap only, cc:147 (+ the mirror mark)
  }
}

// updateFromTsdfBlocks with a caller-supplied block list: the listed slots get their ESDF block
__global__ void k_esdf_mark_listed(Tables tab, const uint32_t* __restrict__ block_list, uint32_t nb) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nb) return;
  const uint32_t s = block_list[i];
  tab.slot_has_esdf[s] = 1;
  tab.slot_esdf_updated[s] = (tab.slot_esdf_updated[s] & kEsdfPending) | 9;
}

// ------------------------------------------------------------------ addNewRobotPosition
// EsdfIntegrator::addNewRobotPosition (cc:25-92) with utils::getAndAllocateSphereAroundPoint
// (utils/planning_utils_inl.h:13-62).  The reference walks `for (float x = -r; x <= r; x++)` on all
// three axes and keeps the offsets whose norm is <= r; the per-axis value list (with the
// reference's accumulated float additions) comes from the host, one thread tests one (x, y, z)
// triple.  floor() of distinct list entries is distinct, so a pass visits every voxel at most
// once and needs no atomics on voxels.
struct SphereParams {
  int n;             // entries of the per-axis list
  int cx, cy, cz;    // getGridIndexFromPoint(center), planning_utils_inl.h:22-23
  float rv;          // radius / voxel_size
  float default_distance;
  int L;
  int outer;         // 0: clear sphere (cc:28-58), 1: occupied sphere (cc:60-86)
  uint32_t cap;
};

__device__ __forceinline__ bool sphere_voxel(const SphereParams& S, const float* __restrict__ xs, uint64_t gid, int* gx,
                                             int* gy, int* gz) {
  const uint64_t n = (uint64_t)S.n;
  if (gid >= n * n * n) return false;
  const float x = xs[gid / (n * n)], y = xs[(gid / n) % n], z = xs[gid % n];
  if (!(norm3(f3(x, y, z)) <= S.rv)) return false;
  *gx = (int)floorf(x) + S.cx;
  *gy = (int)floorf(y) + S.cy;
  *gz = (int)floorf(z) + S.cz;
  return true;
}

// layer->allocateBlockPtrByIndex for every block the sphere reaches (planning_utils_inl.h:57-61)
__global__ void k_esdf_sphere_blocks(SphereParams S, Tables tab, const float* __restrict__ xs, ScanState* st) {
  int gx, gy, gz;
  if (!sphere_voxel(S, xs, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, &gx, &gy, &gz)) return;
  const int bx = gx >> S.L, by = gy >> S.L, bz = gz >> S.L;
  const int lim = kCoordBias - 1;
  if (bx < -lim || bx > lim || by < -lim || by > lim || bz < -lim || bz > lim) {
    atomicOr(&st->error, kErrCoordRange);
    return;
  }
  ensure_block(tab, pack3(bx, by, bz), st);
}

// pool slots for the blocks the sphere created: they exist in the ESDF layer only
__global__ void k_esdf_sphere_assign(Tables tab, uint32_t n_blocks_before, ScanState* st) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t n_new = min(st->n_new, tab.max_blocks);
  if (j < n_new) {
    const uint32_t slot = n_blocks_before + j;
    if (slot < tab.max_blocks) {
      const uint32_t hp = tab.new_list[j];
      tab.hslot[hp] = (int32_t)slot;
      tab.slot_key[slot] = tab.hkeys[hp];
      tab.slot_updated[slot] = kSlotNoTsdf;
    } else {
      atomicOr(&st->error, kErrPoolFull);
    }
  }
  if (j == 0) st->n_blocks = min(n_blocks_before + st->n_new, tab.max_blocks);
}

__global__ void k_esdf_sphere_apply(SphereParams S, Tables tab, const float* __restrict__ xs, uint32_t* raise_list,
                                    uint32_t* open_list, ScanState* st) {
  int gx, gy, gz;
  if (!sphere_voxel(S, xs, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, &gx, &gy, &gz)) return;
  const uint32_t hp = find_block(tab, pack3(gx >> S.L, gy >> S.L, gz >> S.L));
  if (hp == 0xffffffffu) return;  // (coordinate range error raised by the allocation pass)
  const int32_t slot = tab.hslot[hp];
  if (slot < 0) return;           // (pool full, error raised by the assignment)
  const int mask = (1 << S.L) - 1;
  const uint32_t lin = (uint32_t)((gx & mask) | ((gy & mask) << S.L) | ((gz & mask) << (2 * S.L)));
  const uint32_t ref = ((uint32_t)slot << (3 * S.L)) | lin;
  if (!tab.slot_has_esdf[slot]) tab.slot_has_esdf[slot] = 1;
  EsdfWords* ep = reinterpret_cast<EsdfWords*>(tab.esdf) + ref;
  const uint32_t f = ep->flags;
  bool changed = false;
  if (!S.outer) {
    if (!(f & kFlagObserved) || (f & kFlagHallucinated)) {  // cc:44-56
      if (f & kFlagHallucinated) push(raise_list, &st->raise_n[0], S.cap, ref, st);
      ep->distance = S.default_distance;
      changed = true;
    }
  } else {
    if (!(f & kFlagObserved)) {  // cc:74-81
      ep->distance = -S.default_distance;
      changed = true;
    } else if (!(f & kFlagInQueue)) {  // cc:81-85 (in_queue stays false, as in the reference)
      push(open_list, &st->frontier_n[0], S.cap, ref, st);
    }
  }
  if (changed) {
    ep->flags = f | kBitObserved | kBitHallucinated;
    ep->px = ep->py = ep->pz = 0;
    if ((tab.slot_esdf_updated[slot] & (kEsdfPending | 8)) != (kEsdfPending | 8)) {
      tab.slot_esdf_updated[slot] |= (uint8_t)(kEsdfPending | 8);  // updated_blocks_.insert (+ the mirror mark)
    }
    atomicAdd(&st->esdf_counts[S.outer ? 2 : 1], 1u);
  }
}

__global__ void k_esdf_set_pending(ScanState* st, uint32_t n_raise, uint32_t n_open) {
  st->raise_n[0] = n_raise;
  st->frontier_n[0] = n_open;
}

__global__ void k_esdf_clear_tsdf_flag(Tables tab, const uint32_t* __restrict__ block_list, const ScanState* st) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= st->esdf_counts[0]) return;
  tab.slot_updated[block_list[i]] &= (uint8_t)~VBX_UPDATED_ESDF;  // cc:113-121
}

static inline unsigned int grid_for(uint64_t n, int block) { return (unsigned int)((n + block - 1) / block); }

int esdf_destroy(vbx_ctx* c) {
  void* ptrs[] = {c->tab.esdf, c->frontier[0], c->frontier[1], c->raise_q[0], c->raise_q[1], c->esdf_block_list,
                  c->esdf_seed_list, c->esdf_seed_val, c->esdf_touched};
  for (void* p : ptrs) {
    if (p) cudaFree(p);
  }
  c->tab.esdf = nullptr;
  c->frontier[0] = c->frontier[1] = c->raise_q[0] = c->raise_q[1] = c->esdf_block_list = nullptr;
  c->esdf_seed_list = c->esdf_touched = nullptr;
  c->esdf_seed_val = nullptr;
  c->has_esdf = false;
  return VBX_OK;
}

int esdf_create(vbx_ctx* c, const vbx_esdf_config* cfg) {
  if (c->has_esdf) esdf_destroy(c);
  c->ecfg = *cfg;
  const size_t nvox = (size_t)c->tab.max_blocks * c->vox_per_block;
  VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->tab.esdf), nvox * sizeof(EsdfVoxel)));
  // new Block<EsdfVoxel>: distance 0, all flags false, parent 0 (core/voxel.h:18-37)
  VBX_CUDA(c, cudaMemsetAsync(c->tab.esdf, 0, nvox * sizeof(EsdfVoxel), c->stream_main));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_has_esdf, 0, c->tab.max_blocks, c->stream_main));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_esdf_updated, 0, c->tab.max_blocks, c->stream_main));
  c->frontier_cap = std::min<uint64_t>(nvox, 1ull << 25);
  for (int i = 0; i < 2; ++i) {
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->frontier[i]), c->frontier_cap * sizeof(uint32_t)));
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->raise_q[i]), c->frontier_cap * sizeof(uint32_t)));
  }
  VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->esdf_block_list), c->tab.max_blocks * sizeof(uint32_t)));
  VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->esdf_seed_list), c->frontier_cap * sizeof(uint32_t)));
  VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->esdf_seed_val), c->frontier_cap * sizeof(float)));
  VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->esdf_touched), c->frontier_cap * sizeof(uint32_t)));
  int dev = c->device, sms = 0, per_sm_r = 0, per_sm_l = 0;
  VBX_CUDA(c, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  VBX_CUDA(c, cudaFuncSetAttribute(k_esdf_propagate, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)((size_t)c->vox_per_block * (sizeof(TsdfVoxel) + sizeof(EsdfVoxel)))));
  VBX_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_r, k_esdf_raise, 256, 0));
  VBX_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_l, k_esdf_lower, 256, 0));
  // persistent grids: the wavefront is a chain of grid-wide barriers over small frontiers, so the
  // barrier cost (which grows with the number of CTAs) matters more than raw parallelism
  // (measured on the 640x480 workload: 0.45 ms per update with one CTA per SM, 0.52 ms with four);
  // updates over many blocks (batch mode, LiDAR) get the wider grid, see esdf_run
  c->esdf_sms = sms;
  c->esdf_ctas_wide = std::max(1, std::min(std::min(per_sm_r, per_sm_l), 4));
  c->esdf_grid_raise = sms;
  c->esdf_grid_lower = sms;
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  c->has_esdf = true;
  return VBX_OK;
}

static int esdf_run(vbx_ctx* c, int batch, int incremental, int clear_updated_flag, const uint32_t* listed_slots,
                    uint32_t n_listed);

// EsdfIntegrator::clear(), esdf_integrator.h:135-140: forget the work addNewRobotPosition queued
int esdf_clear_state(vbx_ctx* c) {
  c->esdf_pending_raise = c->esdf_pending_open = 0;
  if (c->n_blocks == 0) return VBX_OK;
  std::vector<uint8_t> eu(c->n_blocks);
  VBX_CUDA(c, cudaMemcpyAsync(eu.data(), c->tab.slot_esdf_updated, c->n_blocks, cudaMemcpyDeviceToHost, c->stream_main));
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  for (uint8_t& u : eu) u &= (uint8_t)~kEsdfPending;
  VBX_CUDA(c, cudaMemcpyAsync(c->tab.slot_esdf_updated, eu.data(), c->n_blocks, cudaMemcpyHostToDevice, c->stream_main));
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  return VBX_OK;
}

// EsdfIntegrator::addNewRobotPosition(position), esdf_integrator.cc:25-92
int esdf_add_robot_position(vbx_ctx* c, const float p[3]) {
  cudaStream_t s = c->stream_main;
  ScanState* st = c->set[0].d_state;  // the status block of hand-off set 0
  const vbx_esdf_config& cfg = c->ecfg;
  std::memset(c->esdf_counters, 0, sizeof(c->esdf_counters));
  uint64_t launches = 0;
  const float radii[2] = {cfg.clear_sphere_radius, cfg.occupied_sphere_radius};
  SphereParams S[2];
  std::vector<float> xs[2];
  for (int k = 0; k < 2; ++k) {
    std::memset(&S[k], 0, sizeof(SphereParams));
    const float rv = radii[k] / c->voxel_size;  // radius_in_voxels, planning_utils_inl.h:24
    if (!(rv == rv) || rv > 320.0f) return fail(c, VBX_E_CAPACITY, "sphere radius above 320 voxels");
    for (float x = -rv; x <= rv; x++) xs[k].push_back(x);  // planning_utils_inl.h:26
    const I3 ci = grid_index(f3(p[0], p[1], p[2]), c->voxel_size_inv);
    S[k].n = (int)xs[k].size();
    S[k].cx = ci.x;
    S[k].cy = ci.y;
    S[k].cz = ci.z;
    S[k].rv = rv;
    S[k].default_distance = cfg.default_distance_m;
    S[k].L = c->L;
    S[k].outer = k;
    S[k].cap = (uint32_t)c->frontier_cap;
  }
  // the per-axis lists ride in the seed-value scratch (floats; frontier_cap >> 1300 entries)
  float* d_xs[2] = {c->esdf_seed_val, c->esdf_seed_val + xs[0].size()};
  VBX_CUDA(c, cudaEventRecord(c->ev0, s));
  VBX_CUDA(c, cudaMemsetAsync(st, 0, sizeof(ScanState), s));
  k_esdf_set_pending<<<1, 1, 0, s>>>(st, c->esdf_pending_raise, c->esdf_pending_open);
  for (int k = 0; k < 2; ++k) {
    if (S[k].n == 0) continue;
    VBX_CUDA(c, cudaMemcpyAsync(d_xs[k], xs[k].data(), xs[k].size() * sizeof(float), cudaMemcpyHostToDevice, s));
    const uint64_t n3 = (uint64_t)S[k].n * S[k].n * S[k].n;
    k_esdf_sphere_blocks<<<grid_for(n3, 256), 256, 0, s>>>(S[k], c->tab, d_xs[k], st);
    launches += 1;
  }
  k_esdf_sphere_assign<<<grid_for(c->tab.max_blocks, 256), 256, 0, s>>>(c->tab, c->n_blocks, st);
  launches += 2;
  for (int k = 0; k < 2; ++k) {
    if (S[k].n == 0) continue;
    const uint64_t n3 = (uint64_t)S[k].n * S[k].n * S[k].n;
    k_esdf_sphere_apply<<<grid_for(n3, 256), 256, 0, s>>>(S[k], c->tab, d_xs[k], c->raise_q[0], c->frontier[0], st);
    launches += 1;
  }
  VBX_CUDA(c, cudaEventRecord(c->ev1, s));
  VBX_CUDA(c, cudaMemcpyAsync(c->set[0].h_state, st, sizeof(ScanState), cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));  // (also keeps xs[] alive until the copies are done)
  VBX_CUDA(c, cudaGetLastError());
  VBX_CUDA(c, cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
  const ScanState& h = *c->set[0].h_state;
  if (h.error & (kErrPoolFull | kErrHashFull)) return fail(c, VBX_E_CAPACITY, "block pool / hash full in addNewRobotPosition");
  if (h.error & kErrCoordRange) return fail(c, VBX_E_INVALID, "robot position sphere outside the +-2^20 block range");
  if (h.error & kErrUpdatesFull) return fail(c, VBX_E_CAPACITY, "ESDF wavefront queue capacity exceeded");
  if (h.n_new) c->maybe_esdf_only = true;
  if (int rc = set_n_blocks(c, h.n_blocks)) return rc;
  c->esdf_pending_raise = h.raise_n[0];
  c->esdf_pending_open = h.frontier_n[0];
  c->esdf_counters[0] = h.n_new;          // ESDF blocks created
  c->esdf_counters[1] = h.esdf_counts[1]; // voxels set free
  c->esdf_counters[2] = h.esdf_counts[2]; // voxels set occupied
  c->esdf_counters[4] = h.raise_n[0];     // queued: raise_
  c->esdf_counters[5] = h.frontier_n[0];  // queued: open_
  c->esdf_counters[7] = launches;
  c->launches += launches;
  return refresh_host_mirror(c);
}

int esdf_update(vbx_ctx* c, int batch, int clear_updated_flag) {
  return esdf_run(c, batch, batch ? 0 : 1, clear_updated_flag, nullptr, 0);
}

// EsdfIntegrator::updateFromTsdfBlocks(tsdf_blocks, incremental), esdf_integrator.cc:124-302: blocks
// without a TSDF block are skipped (cc:139-141); a block listed twice is processed once.
int esdf_update_blocks(vbx_ctx* c, const int32_t* idx3, uint64_t m, int incremental) {
  if (int rc = refresh_host_mirror(c)) return rc;
  std::vector<uint32_t> slots;
  slots.reserve(m);
  std::vector<uint8_t> seen(c->n_blocks, 0), upd(c->n_blocks, 0);
  if (c->maybe_esdf_only && c->n_blocks) {
    VBX_CUDA(c, cudaMemcpyAsync(upd.data(), c->tab.slot_updated, c->n_blocks, cudaMemcpyDeviceToHost, c->stream_main));
    VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  }
  for (uint64_t i = 0; i < m; ++i) {
    auto it = c->host_key2slot.find(pack3(idx3[3 * i], idx3[3 * i + 1], idx3[3 * i + 2]));
    if (it == c->host_key2slot.end() || seen[it->second] || (upd[it->second] & kSlotNoTsdf)) continue;
    seen[it->second] = 1;
    slots.push_back((uint32_t)it->second);
  }
  return esdf_run(c, 0, incremental ? 1 : 0, 0, slots.data(), (uint32_t)slots.size());
}

static int esdf_run(vbx_ctx* c, int batch, int incremental, int clear_updated_flag, const uint32_t* listed_slots,
                    uint32_t n_listed) {
  cudaStream_t s = c->stream_main;
  ScanState* st = c->set[0].d_state;  // the status block of hand-off set 0
  const ScanState& h = *c->set[0].h_state;
  std::memset(c->esdf_counters, 0, sizeof(c->esdf_counters));
  const vbx_esdf_config& cfg = c->ecfg;
  EsdfParams E;
  std::memset(&E, 0, sizeof(E));
  E.L = c->L;
  E.voxel_size = c->voxel_size;
  E.max_distance = cfg.max_distance_m;
  E.min_distance = cfg.min_distance_m;
  E.default_distance = cfg.default_distance_m;
  E.min_diff = cfg.min_diff_m;
  E.min_weight = cfg.min_weight;
  E.full_euclidean = cfg.full_euclidean_distance;
  E.multi_queue = cfg.multi_queue;
  E.add_occupied_crust = cfg.add_occupied_crust;
  E.incremental = incremental;
  E.u1 = 1.0f;
  E.u2 = (float)std::sqrt(2.0);  // const float sqrt_2 = std::sqrt(2), neighbor_tools.cc:9
  E.u3 = (float)std::sqrt(3.0);
  E.d1 = E.u1 * c->voxel_size;
  E.d2 = E.u2 * c->voxel_size;
  E.d3 = E.u3 * c->voxel_size;
  E.cap = (uint32_t)c->frontier_cap;
  uint64_t launches = 0;
  VBX_CUDA(c, cudaEventRecord(c->ev0, s));
  if (c->profiling) cudaEventRecord(c->sev[0], s);
  VBX_CUDA(c, cudaMemsetAsync(st, 0, sizeof(ScanState), s));
  if (c->n_blocks == 0) {
    VBX_CUDA(c, cudaStreamSynchronize(s));
    return VBX_OK;
  }
  if (batch) {
    // the batch update wipes the ESDF layer (cc:95); queue entries of addNewRobotPosition would
    // point into removed blocks (the reference CHECK-fails on them), so they are dropped
    c->esdf_pending_raise = c->esdf_pending_open = 0;
  }
  // raise_ / open_ entries queued by addNewRobotPosition since the last update (they sit at the
  // head of raise_q[0] / frontier[0]; this call's own entries are appended behind them)
  const bool pending = c->esdf_pending_raise || c->esdf_pending_open;
  if (pending) {
    k_esdf_set_pending<<<1, 1, 0, s>>>(st, c->esdf_pending_raise, c->esdf_pending_open);
    launches += 1;
  }
  c->esdf_pending_raise = c->esdf_pending_open = 0;
  if (batch) {
    // esdf_layer_->removeAllBlocks() (cc:95): every ESDF block starts from scratch
    const size_t nvox = (size_t)c->n_blocks * c->vox_per_block;
    VBX_CUDA(c, cudaMemsetAsync(c->tab.esdf, 0, nvox * sizeof(EsdfVoxel), s));
    VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_has_esdf, 0, c->n_blocks, s));
    VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_esdf_updated, 0, c->n_blocks, s));
  }
  uint32_t nb = 0;
  if (listed_slots) {
    nb = n_listed;
    if (nb > 0) {
      VBX_CUDA(c, cudaMemcpyAsync(c->esdf_block_list, listed_slots, (size_t)nb * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
      VBX_CUDA(c, cudaMemcpyAsync(&st->esdf_counts[0], &nb, sizeof(uint32_t), cudaMemcpyHostToDevice, s));
      k_esdf_mark_listed<<<grid_for(nb, 256), 256, 0, s>>>(c->tab, c->esdf_block_list, nb);
      VBX_CUDA(c, cudaStreamSynchronize(s));  // the two host sources above are stack / vector memory
    }
  } else {
    // the list and its length (esdf_counts[0]) stay on the device: no host round trip in the middle of
    // the call; the launches below are sized for the upper bound (every slot) and the kernels stop at
    // the real count
    k_esdf_block_list<<<grid_for(c->n_blocks, 256), 256, 0, s>>>(c->tab, c->n_blocks, batch, c->esdf_block_list, st);
    nb = c->n_blocks;
  }
  launches += 1;
  if (nb > 0 || pending) {
    if (nb > 0) {
      // one thread block per voxel block, both slabs staged by the TMA
      const size_t slab_bytes = (size_t)c->vox_per_block * (sizeof(TsdfVoxel) + sizeof(EsdfVoxel));
      k_esdf_propagate<<<nb, (unsigned int)std::max<uint32_t>(32u, std::min<uint32_t>(1024u, c->vox_per_block)), slab_bytes, s>>>(
          E, c->tab, c->esdf_block_list, nb, c->frontier[0], c->raise_q[0], c->esdf_seed_list, st);
      launches += 1;
    }
    if (nb > 0 && incremental) {
      const unsigned int g = 148 * 8;
      k_esdf_seed<<<g, 256, 0, s>>>(E, c->tab, c->esdf_seed_list, c->frontier[0], c->esdf_seed_val, st);
      k_esdf_seed_commit<<<g, 256, 0, s>>>(E, c->tab, c->esdf_seed_list, c->esdf_seed_val, st);
      launches += 2;
    }
    if (c->profiling) cudaEventRecord(c->sev[1], s);
    {
      int per_sm = (nb <= 256 && !pending) ? c->esdf_ctas_small : c->esdf_ctas_wide;
      if (const char* e = std::getenv("VBX_ESDF_CTAS")) per_sm = std::max(1, std::min(std::atoi(e), c->esdf_ctas_wide));  // (tuning aid)
      c->esdf_grid_raise = c->esdf_grid_lower = c->esdf_sms * per_sm;
    }
    {
      void* args[] = {&E, &c->tab, &c->raise_q[0], &c->raise_q[1], &c->frontier[0], &st};
      VBX_CUDA(c, cudaLaunchCooperativeKernel((void*)k_esdf_raise, dim3(c->esdf_grid_raise), dim3(256), args, 0, s));
    }
    if (c->profiling) cudaEventRecord(c->sev[2], s);
    {
      void* args[] = {&E, &c->tab, &c->frontier[0], &c->frontier[1], &c->esdf_touched, &st};
      VBX_CUDA(c, cudaLaunchCooperativeKernel((void*)k_esdf_lower, dim3(c->esdf_grid_lower), dim3(256), args, 0, s));
    }
    k_esdf_parents<<<148 * 8, 256, 0, s>>>(E, c->tab, c->esdf_touched, st);
    if (c->profiling) cudaEventRecord(c->sev[3], s);
    launches += 3;
    if (nb > 0 && !batch && clear_updated_flag) {
      k_esdf_clear_tsdf_flag<<<grid_for(nb, 256), 256, 0, s>>>(c->tab, c->esdf_block_list, st);
      launches += 1;
    }
  }
  VBX_CUDA(c, cudaEventRecord(c->ev1, s));
  VBX_CUDA(c, cudaMemcpyAsync(c->set[0].h_state, st, sizeof(ScanState), cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  VBX_CUDA(c, cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
  if (c->profiling && (nb > 0 || pending)) {
    for (int m = 0; m < 3; ++m) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, c->sev[m], c->sev[m + 1]) == cudaSuccess) {
        c->stage_ms[9 + m] += ms;
        c->stage_calls[9 + m] += 1;
      }
    }
  }
  if (h.error & kErrUpdatesFull) return fail(c, VBX_E_CAPACITY, "ESDF wavefront queue capacity exceeded");
  for (int i = 0; i < 7; ++i) c->esdf_counters[i] = h.esdf_counts[i];
  c->esdf_counters[7] = launches;
  c->launches += launches;
  return VBX_OK;
}

}  // namespace vbx
