// Internal declarations shared by the engine's translation units (not installed;
// the public boundary is include/voxblox_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../include/voxblox_b200.h"
#include "vbx_math.cuh"
#include "vbx_order.cuh"

namespace vbx {
struct SortPlan;
}

namespace vbx {

constexpr uint64_t kEmptyKey = ~0ull;
constexpr uint64_t kInvalidPointKey = ~0ull;
constexpr int kCoordBias = 1 << 20;  // block / voxel coordinates are packed 21 bits per axis
// Internal bits of the per-slot flag bytes (never reported through the C-ABI):
//   slot_updated bit 7: the slot holds an ESDF block only -- the TSDF layer has no block at this
//     index (blocks allocated by EsdfIntegrator::addNewRobotPosition or uploaded into the ESDF layer).
//     Any TSDF touch writes the byte to 7 (Block::updated().set()), which turns the slot into a TSDF block
//     that starts from zeroed voxels, exactly like a freshly allocated one.
//   slot_esdf_updated bit 7: member of EsdfIntegrator::updated_blocks_ (esdf_integrator.h:172-175).
constexpr uint8_t kSlotNoTsdf = 0x80, kEsdfPending = 0x80;
//   bit 3 of both flag bytes (VBX_UPDATED_MIRROR): the block changed since a vbx_mirror_updated /
//     vbx_serialize_updated call last cleared this bit -- the engine's own dirty mark for the incremental
//     host mirror, independent of the three Block::updated() bits (which their consumers clear).
constexpr uint8_t kTouchedBits = 0x0F;  // what a TSDF update writes: Block::updated().set() + the mirror mark

struct EsdfVoxel {  // core/voxel.h:18-37
  float distance;
  uint8_t observed, hallucinated, in_queue, fixed;
  int32_t parent[3];
};
static_assert(sizeof(TsdfVoxel) == 12 && sizeof(EsdfVoxel) == 20, "voxel layouts");

// Error bits raised on the device (ScanState::error)
enum : uint32_t {
  kErrPoolFull = 1u,        // more blocks than max_blocks
  kErrHashFull = 2u,        // block hash probe wrapped around
  kErrCoordRange = 4u,      // |voxel coordinate| >= 2^20 * vps
  kErrUpdatesFull = 8u,     // ray-voxel updates exceed max_updates_per_pass
  kFatalErrors = 15u,       // any of the above
  kSkipped = 32u,           // not an error: the scan was queued behind a scan that must be redone (vbx_capi.cu)
};

// Device-resident per-call state; the host reads it back through pinned memory.
struct ScanState {
  uint32_t n_new;            // hash entries created by this call
  uint32_t n_touched;        // distinct blocks touched by this call
  uint32_t error;
  uint32_t n_rays;           // normal rays / bundles cast
  uint32_t n_clear_rays;     // clearing rays / bundles cast
  uint32_t n_valid_points;
  uint32_t n_voxels;         // distinct voxels updated (U)
  uint32_t n_blocks;         // pool slots in use after the call
  unsigned long long total_updates;  // K the back half runs on (0 when the call failed / is redone)
  unsigned long long total_found;    // K as counted
  // ESDF
  uint32_t esdf_counts[7];
  uint32_t raise_n2;         // third raise-level counter (see esdf_cnt: the counters rotate mod 3)
  uint32_t frontier_n[2];
  uint32_t raise_n[2];
  uint32_t seed_n;           // ESDF: new free voxels waiting for updateVoxelFromNeighbors
  uint32_t lowered_n;        // ESDF: voxels lowered by the wavefront
  uint32_t n_ray_list;       // bundle heads (Merged)
  uint32_t n_long;           // voxel runs handed to k_apply_long
  uint32_t n_verify;         // work items of k_apply_verify
  uint32_t n_refold;         // bundles folded a second time with IEEE division (diagnostic)
  uint32_t refold_members;   // ... and the points they hold
  uint32_t frontier_n2;      // third wavefront counter
  // Merged: bounding box of the valid points' voxels, both ends atomicMax'ed (so that an all-zero
  // block means "no valid point"): kb_max = v + 2^30, kb_min = 0xffffffff - (v + 2^30); the bundle
  // keys are packed relative to it (vbx_tsdf.cu, KeyLayout)
  uint32_t kb_max[3];
  uint32_t kb_min[3];
  uint32_t key_bits;         // bits a bundle key uses
  uint32_t n_big;            // Merged: bundles of at least kBigBundle members (folded first)
  uint32_t merge_ticket;     // Merged: work hand-out counter of k_merge
  uint32_t n_touch_ids;      // touched-block ids handed out (>= n_touched: ids lost to a race stay unused)
  uint32_t rec_key_bits;     // bits an update-record key uses: voxel-in-block bits + bits of the touched ids
  uint32_t esdf_ticket[6];   // ESDF queue kernels: work hand-out counters, rotating like the queue counters ([0..2] raise, [3..5] lower)
  uint32_t reserved[15];
};
static_assert(sizeof(ScanState) == 256, "the status block the host reads back is 256 bytes");

// The GPU-resident block hash + voxel pools (the device mirror of Layer<T>::block_map_,
// core/layer.h:30-32,292).
struct Tables {
  uint64_t* hkeys;        // [hcap] packed block index, kEmptyKey when free
  int32_t* hslot;         // [hcap] pool slot
  unsigned long long* htouch;  // [hcap] (call id << 32 | touched id) of the last call that touched the block
  uint32_t hmask;         // hcap - 1
  uint32_t max_blocks;
  uint32_t vox_per_block;
  uint32_t* new_list;     // [max_blocks] hash positions created by this call
  uint32_t* touched_list; // [touched_cap] touched id -> hash position (0xffffffff: unused id); null in vbx_ctx::tab,
                          // the launch code passes a copy that points at the hand-off set's own list
  uint32_t touched_cap;
  uint64_t* slot_key;     // [max_blocks] packed block index per pool slot
  uint8_t* slot_updated;  // [max_blocks] TSDF Block::updated() bits
  uint8_t* slot_esdf_updated;  // [max_blocks] ESDF Block::updated() bits
  uint8_t* slot_has_esdf;      // [max_blocks] 1 once the ESDF layer holds this block
  TsdfVoxel* tsdf;        // [max_blocks << 3L]
  EsdfVoxel* esdf;        // [max_blocks << 3L] (allocated by vbx_esdf_create)
};

__host__ __device__ inline uint64_t pack3(int x, int y, int z) {
  return ((uint64_t)(uint32_t)(z + kCoordBias) << 42) | ((uint64_t)(uint32_t)(y + kCoordBias) << 21) |
         (uint64_t)(uint32_t)(x + kCoordBias);
}
__host__ __device__ inline void unpack3(uint64_t k, int* x, int* y, int* z) {
  *x = (int)(k & 0x1fffffu) - kCoordBias;
  *y = (int)((k >> 21) & 0x1fffffu) - kCoordBias;
  *z = (int)((k >> 42) & 0x1fffffu) - kCoordBias;
}
// block-ownership sharding: the rank that owns a block (2 x 2 x 2 brick pattern for 8 ranks)
__host__ __device__ inline int block_owner(int bx, int by, int bz, int world) {
  const int a = (bx + 2 * by + 4 * bz) % world;
  return a < 0 ? a + world : a;
}
__host__ __device__ inline uint32_t hash64(uint64_t k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdULL;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ULL;
  k ^= k >> 33;
  return (uint32_t)k;
}

}  // namespace vbx

struct vbx_ctx {
  int device = 0;
  cudaStream_t stream_main = nullptr; // back halves, ESDF, block management, synchronous calls
  cudaStream_t stream_c = nullptr;    // host-to-device cloud copies of asynchronously submitted scans
  cudaStream_t stream_c2 = nullptr;   // ... alternating with this one
  cudaStream_t stream_h = nullptr;    // read-back of a queued scan's status block (keeps the copy engine out of the apply stream)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  vbx_tsdf_config cfg;
  vbx_engine_options opt;
  float voxel_size = 0, voxel_size_inv = 0;
  int vps = 16, L = 4;         // voxels per side and log2
  uint32_t vox_per_block = 4096;
  uint32_t hcap = 0;
  unsigned int grid_sms = 148;  // persistent-kernel grids are multiples of this (the SM count; VBX_GRID_SMS overrides: tuning aid)
  vbx::Tables tab;
  // scratch
  uint32_t max_points = 0;
  uint64_t max_updates = 0;
  bool timeline = false;            // VBX_ASYNC_TIMELINE: the hand-off events carry timestamps
  cudaEvent_t timeline_ref = nullptr;
  uint32_t bundle_hint = 0;         // bundles (the larger of the two maps) of the most recent Merged scan whose counters reached the host
  uint64_t record_hint = 1u << 20;  // update records of the most recent scan whose count reached the host: sizes the record sort's grid
  uint32_t* order = nullptr;               // [max_points] "sorted" integration order (synchronous calls only)
  uint32_t* order_inv = nullptr;           // [max_points] inverse of `order`
  vbx::RehashSchedule rehash{};            // libstdc++'s unordered_map growth schedule (vbx_create)
  size_t order_smem_bytes = 0;             // dynamic shared memory of k_bundle_order
  unsigned long long* long_list = nullptr; // [max_updates / 32 + 1] starts of long voxel runs
  unsigned long long* long_end = nullptr;
  uint32_t* long_state = nullptr;
  uint32_t* verify_run = nullptr;          // [max_updates / 32 + 1] work items of k_apply_verify
  unsigned long long* verify_start = nullptr;
  float* rec_sdf = nullptr;                // [max_updates] per sorted record
  float* rec_w = nullptr;
  uint32_t sort_tiles_cap[2] = {0, 0};  // tiles of the engine's radix sort (vbx_sort.cuh): [0] point keys, [1] update records
  unsigned long long* set_start = nullptr;  // Fast integrator approximate sets
  unsigned long long* set_observed = nullptr;
  uint32_t set_epoch = 1;
  int64_t fast_reset_counter = 0;
  uint32_t epoch = 0;                 // call id for touch marks
  uint32_t n_blocks = 0;              // pool slots in use (host copy, exact after a drain)
  uint32_t* d_nblocks = nullptr;      // [2] device copy, ping-pong: k_assign reads [nb_cur], writes [nb_cur ^ 1]
  int nb_cur = 0;
  // Asynchronous submission (vbx_tsdf_integrate_async): a scan passes through three stages on
  // separate streams -- front half (keys, bundle sort, bundle fold, offsets; does not touch the map)
  // on one of kLanes front streams, ray walk + block creation + record sort on stream_e, apply on
  // the main stream -- so up to kSets scans are in flight, each owning one set of hand-off
  // buffers.  Map-touching stages run in submission order.  The launch code takes the set and the
  // lane it works on as arguments.  Synchronous calls name set 0 and lane 0 and run on the main
  // stream; the other sets and lanes are allocated on the first asynchronous submission.
  static constexpr int kSets = 16, kLanes = 8, kSortStreams = 2;  // upper bounds
  int sets_in_use = 10, lanes_in_use = 6;  // (tuning aids: VBX_ASYNC_SETS, VBX_ASYNC_LANES)
  struct ScratchSet {
    float4* ray_p = nullptr;  // point_G.xyz, flags (bit 0: clearing ray)
    float4* ray_a = nullptr;  // point_G - origin, |point_G - origin|
    uint2* ray_c = nullptr;   // colour, weight bits
    uint32_t* ray_list = nullptr;    // Merged: ray slot (rank in the reference's bundle order) -> head
    uint32_t* head_list = nullptr;   // bundle id -> sorted position of its head (read again by the ray walk)
    uint32_t* touched_list = nullptr;  // [touched_cap] touched id -> hash position (written by the walk, read by the apply)
    uint32_t* cnt = nullptr;  // [max_points + 1]
    uint32_t* off = nullptr;  // [max_points + 1]
    vbx::ScanState* d_state = nullptr;
    vbx::ScanState* h_state = nullptr;  // pinned
    float* d_xyz = nullptr;
    uint8_t* d_rgba = nullptr;
    uint64_t* pkeys0 = nullptr;  // sorted bundle keys (read again by the ray walk)
    uint32_t* ckeys[2] = {nullptr, nullptr};  // [max_updates] update records (written by the walk, read by apply)
    uint32_t* cvals[2] = {nullptr, nullptr};
    vbx::SortPlan* sort_plan1 = nullptr;      // the update-record sort (vbx_sort.cuh)
    uint32_t* sort_status1 = nullptr;
    cudaEvent_t copy_done = nullptr, front_done = nullptr, walked = nullptr, sorted = nullptr, back_done = nullptr;
    cudaEvent_t applied = nullptr;      // the apply kernels are done (the status read-back follows on stream_h)
    cudaEvent_t front_start = nullptr;  // only with VBX_ASYNC_TIMELINE (vbx_debug_async_timeline)
    bool in_flight = false;
    int kind = 0;
    uint64_t launches = 0;
    // what the scan was submitted with, kept until it is known to be in the map: a scan that cannot
    // be applied asynchronously is redone from here (recover_async)
    uint64_t seq = 0;
    bool redo = false;
    float q[4] = {1, 0, 0, 0}, t[3] = {0, 0, 0};
    uint64_t n = 0;
    int freespace = 0;
    const float* in_xyz = nullptr;
    const uint8_t* in_rgba = nullptr;
  } set[kSets];
  struct FrontLane {  // scratch private to one front-half stream
    cudaStream_t stream = nullptr;
    uint64_t* pkeys1 = nullptr;
    uint32_t* pvals[2] = {nullptr, nullptr};
    vbx::SortPlan* sort_plan0 = nullptr;  // the point-key sort (vbx_sort.cuh)
    uint32_t* sort_status0 = nullptr;
    uint32_t* scan_status = nullptr;
    uint32_t* big_list = nullptr;      // [max_points / 256 + 1] ids of the big bundles
    uint32_t* first_bits = nullptr;    // [2][max_points / 32 + 1] first-occurrence bitmaps
    vbx::OrderScratch order_scratch{};  // k_bundle_order's global tables
    cudaStream_t side = nullptr;       // k_bundle_order runs here, beside k_merge
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  } lane[kLanes];
  bool async_ready = false;
  int prio_lo = 0, prio_hi = 0;  // stream priority range of the device
  cudaStream_t stream_e = nullptr;      // ray walk + block creation + record sort of asynchronously submitted scans
  cudaStream_t stream_s[kSortStreams] = {nullptr, nullptr};  // record sorts (set-private buffers: independent across scans)
  uint64_t async_seq = 0;
  uint32_t* d_hold = nullptr;           // device flag: a queued scan must be redone, later scans skip their back half
  uint64_t async_redone = 0;            // scans redone synchronously since vbx_create (reporting)
  bool hash_dirty = false;              // an asynchronous scan ran out of pool slots: rebuild the hash at the next drain
  int deferred_rc = 0;
  std::string deferred_msg;
  // incremental device -> host mirror (vbx_mirror_updated): gather staging on both sides
  void* mirror_dev = nullptr;
  void* mirror_host = nullptr;  // page-locked
  uint32_t* mirror_slots = nullptr;
  size_t mirror_cap_bytes = 0, mirror_cap_slots = 0;
  // host mirror of slot_key (refreshed lazily)
  std::vector<uint64_t> host_slot_key;
  std::unordered_map<uint64_t, int32_t> host_key2slot;
  // Block::has_data_ (core/block.h:206): never set by the integrators, carried by BlockProto; blocks loaded
  // from a .vxblx file with has_data = true are remembered per layer so that a re-save writes the flag back
  std::unordered_set<uint64_t> has_data_keys[2];
  // ESDF
  bool has_esdf = false;
  vbx_esdf_config ecfg;
  uint32_t* frontier[2] = {nullptr, nullptr};
  uint32_t* raise_q[2] = {nullptr, nullptr};
  uint64_t frontier_cap = 0;
  uint32_t* esdf_block_list = nullptr;
  uint32_t* esdf_seed_list = nullptr;
  float* esdf_seed_val = nullptr;
  uint32_t* esdf_touched = nullptr;
  int esdf_grid_raise = 0, esdf_grid_lower = 0, esdf_sms = 0, esdf_ctas_wide = 1, esdf_ctas_small = 1;
  uint32_t esdf_pending_raise = 0, esdf_pending_open = 0;  // raise_ / open_ entries queued by addNewRobotPosition
  bool maybe_esdf_only = false;                            // some slot may carry kSlotNoTsdf
  // mesher (vbx_mesh.cu): the result of the last vbx_mesh_generate stays on the device until the next one
  uint32_t* mesh_slots = nullptr;
  uint16_t* mesh_cube_off = nullptr;
  uint32_t* mesh_block_nv = nullptr;
  unsigned long long* mesh_first = nullptr;
  float* mesh_vertices = nullptr;
  float* mesh_normals = nullptr;
  uint32_t* mesh_colors = nullptr;
  uint64_t mesh_cap_blocks = 0, mesh_cap_vertices = 0, mesh_launches = 0;
  std::vector<int32_t> mesh_idx;
  std::vector<uint64_t> mesh_first_host = std::vector<uint64_t>(1, 0);
  bool mesh_use_color = false;
  // ICP (vbx_icp.cu): shuffled point order (host page-locked + device), host-cloud staging, result block
  uint32_t* icp_perm_dev = nullptr;
  uint32_t* icp_perm_host = nullptr;
  float* icp_points_dev = nullptr;
  float* icp_out_dev = nullptr;
  float* icp_out_host = nullptr;
  uint64_t icp_cap = 0;
  // reporting
  uint32_t last_passes = 1;  // passes the last synchronous integrate call needed (K > max_updates_per_pass)
  uint64_t counters[16] = {0};
  uint64_t async_wait_ns = 0, async_submit_ns = 0;  // host time of vbx_tsdf_integrate_async: waiting for a hand-off set / enqueueing
  uint64_t esdf_counters[16] = {0};
  uint64_t shard_front_counters[4] = {0};
  float last_ms = 0.f;
  uint64_t launches = 0;
  cudaEvent_t tev0 = nullptr, tev1 = nullptr;  // vbx_timer_*
  bool profiling = false;
  cudaEvent_t sev[20] = {nullptr};             // stage boundaries
  double stage_ms[16] = {0};
  uint64_t stage_calls[16] = {0};
  std::string err;
};

namespace vbx {
int fail(vbx_ctx* c, int code, const std::string& msg);
int cuda_fail(vbx_ctx* c, cudaError_t e, const char* what);
int refresh_host_mirror(vbx_ctx* c);
int mirror_updated(vbx_ctx* c, int layer, int updated_mask, int clear_mask, int32_t* idx3, void* voxels,
                   uint8_t* updated_bits, uint64_t cap, uint64_t* n, int serialized);
int esdf_destroy(vbx_ctx* c);
void mesh_destroy(vbx_ctx* c);
void icp_destroy(vbx_ctx* c);
int icp_run(vbx_ctx* c, const vbx_icp_config* cfg, const float* points, int on_device, uint64_t n, const float q[4],
            const float t[3], uint32_t seed, float out_q[4], float out_t[3], uint64_t* num_updates);
int mesh_generate(vbx_ctx* c, const vbx_mesh_config* cfg, int only_updated, int clear_flag, uint64_t* n_blocks_out,
                  uint64_t* n_vertices_out);
int mesh_download(vbx_ctx* c, int32_t* idx3, uint64_t* first_vertex, float* vertices, float* normals, uint8_t* colors);
int esdf_add_robot_position(vbx_ctx* c, const float p[3]);
int esdf_clear_state(vbx_ctx* c);
int ensure_async(vbx_ctx* c);          // allocate the extra hand-off sets / front lanes
int drain_async(vbx_ctx* c);           // wait for every asynchronously submitted scan, collect its results
int set_n_blocks(vbx_ctx* c, uint32_t n);
int init_bundle_order(vbx_ctx* c);     // rehash schedule + shared-memory opt-in of k_bundle_order
int rebuild_hash(vbx_ctx* c);          // block hash rebuilt from slot_key (after removals / a pool overflow)
void harvest_async(vbx_ctx* c, vbx_ctx::ScratchSet& S);  // collect a finished asynchronous scan's results
}  // namespace vbx

#define VBX_CUDA(c, expr)                                          \
  do {                                                             \
    cudaError_t _e = (expr);                                       \
    if (_e != cudaSuccess) return vbx::cuda_fail((c), _e, #expr);  \
  } while (0)
