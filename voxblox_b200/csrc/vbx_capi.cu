// The C-ABI of include/voxblox_b200.h: context life cycle, the host<->device block
// mirror (Layer<T> on the host side stays the reference's own container; see
// INTEGRATION.md) and the entry points that dispatch into the device pipelines.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "vbx_engine.h"
#include "vbx_sort.cuh"

namespace vbx {

int integrate_device(vbx_ctx* c, int kind, const float q[4], const float t[3], const float* d_xyz,
                     const uint8_t* d_rgba, uint64_t n, int freespace);
int debug_sort(vbx_ctx* c, const void* keys, int key_bytes, uint32_t n, int key_bits, void* keys_out,
               uint32_t* vals_out);
int debug_scan(vbx_ctx* c, const uint32_t* in, uint32_t n, uint32_t* out);
int debug_bundle_order(vbx_ctx* c, const uint32_t* hashes, uint32_t n, int force_global, uint32_t* out);
int upload_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m, const void* voxels,
                  const uint8_t* updated_bits, int serialized);
int remove_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m);
int clear_layer(vbx_ctx* c, int layer);
int integrate_async(vbx_ctx* c, int kind, const float q[4], const float t[3], const float* xyz, const uint8_t* rgba,
                    uint64_t n, int freespace, int on_device);
int esdf_create(vbx_ctx* c, const vbx_esdf_config* cfg);
int esdf_update(vbx_ctx* c, int batch, int clear_updated_flag);
int esdf_update_blocks(vbx_ctx* c, const int32_t* idx3, uint64_t m, int incremental);
int esdf_add_robot_position(vbx_ctx* c, const float p[3]);
int esdf_clear_state(vbx_ctx* c);

int fail(vbx_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg;
  return code;
}
int cuda_fail(vbx_ctx* c, cudaError_t e, const char* what) {
  if (c) c->err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
  return VBX_E_CUDA;
}

// Bring the host copy of slot -> block index up to date (new blocks are appended to
// slot_key by k_assign; removal rebuilds it).
int refresh_host_mirror(vbx_ctx* c) {
  const size_t have = c->host_slot_key.size();
  if (have < c->n_blocks) {
    c->host_slot_key.resize(c->n_blocks);
    VBX_CUDA(c, cudaMemcpyAsync(c->host_slot_key.data() + have, c->tab.slot_key + have,
                                (c->n_blocks - have) * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream_main));
    VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
    for (size_t s = have; s < c->n_blocks; ++s) c->host_key2slot[c->host_slot_key[s]] = (int32_t)s;
  }
  return VBX_OK;
}

int set_n_blocks(vbx_ctx* c, uint32_t n) {
  c->n_blocks = n;
  VBX_CUDA(c, cudaMemcpyAsync(c->d_nblocks + c->nb_cur, &c->n_blocks, sizeof(uint32_t), cudaMemcpyHostToDevice,
                              c->stream_main));
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  return VBX_OK;
}

// Collect a finished asynchronous scan: its counters, the block count, and any error it raised
// (reported by the next call that can return one).
void harvest_async(vbx_ctx* c, vbx_ctx::ScratchSet& S) {
  S.in_flight = false;
  const ScanState& h = *S.h_state;
  c->n_blocks = std::max(c->n_blocks, h.n_blocks);
  std::memset(c->counters, 0, sizeof(c->counters));
  c->counters[0] = h.n_rays;
  c->counters[1] = h.n_clear_rays;
  c->counters[2] = h.total_found;
  if (h.total_found) c->record_hint = h.total_found;
  if (S.kind == VBX_MERGED && !(h.error & kFatalErrors)) c->bundle_hint = std::max(h.n_rays, h.n_clear_rays);
  c->counters[3] = h.n_voxels;
  c->counters[4] = h.n_touched;
  c->counters[5] = h.n_new;
  c->counters[6] = S.kind == VBX_MERGED ? h.n_valid_points : (uint64_t)h.n_rays + h.n_clear_rays;
  c->counters[7] = S.launches;
  c->counters[11] = 1;
  const uint32_t fatal = h.error & kFatalErrors & ~kErrUpdatesFull;
  if (!fatal && (h.error & (kErrUpdatesFull | kSkipped))) {
    // more update records than one pass holds (or queued behind such a scan): nothing was applied;
    // recover_async redoes it synchronously, in passes, in submission order
    S.redo = true;
    return;
  }
  if (fatal & kErrPoolFull) c->hash_dirty = true;  // surplus hash entries without a pool slot
  if (fatal && !c->deferred_rc) {
    c->deferred_rc = VBX_E_CAPACITY;
    c->deferred_msg = "an asynchronously submitted scan failed on the device (error bits " + std::to_string(h.error) +
                      (fatal & kErrPoolFull ? ": block pool full, raise vbx_engine_options.max_blocks" : "") + ")";
  }
}

// Every queued scan has been waited for.  Scans that could not be applied asynchronously (and the
// scans queued behind them, which skipped their back halves) are redone synchronously from their
// retained inputs, in submission order -- no scan is lost and the update order is the callers'.
static int recover_async(vbx_ctx* c) {
  if (c->hash_dirty) {
    c->hash_dirty = false;
    if (int rc = rebuild_hash(c)) return rc;
  }
  std::vector<vbx_ctx::ScratchSet*> todo;
  for (int k = 0; k < vbx_ctx::kSets; ++k) {
    if (c->set[k].redo) todo.push_back(&c->set[k]);
  }
  if (todo.empty()) return VBX_OK;
  std::sort(todo.begin(), todo.end(), [](const vbx_ctx::ScratchSet* a, const vbx_ctx::ScratchSet* b) { return a->seq < b->seq; });
  VBX_CUDA(c, cudaMemsetAsync(c->d_hold, 0, sizeof(uint32_t), c->stream_main));
  int first_rc = VBX_OK;
  std::string first_msg;
  for (vbx_ctx::ScratchSet* S : todo) {
    S->redo = false;
    const int rc = integrate_device(c, S->kind, S->q, S->t, S->in_xyz, S->in_rgba, S->n, S->freespace);
    c->async_redone += 1;
    if (rc != VBX_OK && first_rc == VBX_OK) {
      first_rc = rc;
      first_msg = c->err;
    }
  }
  if (first_rc != VBX_OK) c->err = first_msg;
  return first_rc;
}

int drain_async(vbx_ctx* c) {
  for (int k = 0; k < c->sets_in_use; ++k) {
    vbx_ctx::ScratchSet& S = c->set[(c->async_seq + k) % c->sets_in_use];  // oldest submission first
    if (!S.in_flight) continue;
    VBX_CUDA(c, cudaEventSynchronize(S.back_done));
    harvest_async(c, S);
  }
  if (int rc = recover_async(c)) {
    if (!c->deferred_rc) return rc;
  }
  if (c->deferred_rc) {
    const int rc = c->deferred_rc;
    c->err = c->deferred_msg;
    c->deferred_rc = 0;
    return rc;
  }
  return VBX_OK;
}

template <typename T>
static cudaError_t dmalloc(T** p, size_t count) {
  return cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T));
}

// The device buffers of one hand-off set (its events are created by ensure_async).
static int alloc_set(vbx_ctx* c, vbx_ctx::ScratchSet& S) {
  const size_t np = c->max_points;
  VBX_CUDA(c, dmalloc(&S.d_xyz, 3 * np));
  VBX_CUDA(c, dmalloc(&S.d_rgba, 4 * np));
  VBX_CUDA(c, dmalloc(&S.pkeys0, np));
  for (int i = 0; i < 2; ++i) {
    VBX_CUDA(c, dmalloc(&S.ckeys[i], (size_t)c->max_updates));
    VBX_CUDA(c, dmalloc(&S.cvals[i], (size_t)c->max_updates));
  }
  VBX_CUDA(c, dmalloc(&S.ray_p, np));
  VBX_CUDA(c, dmalloc(&S.ray_a, np));
  VBX_CUDA(c, dmalloc(&S.ray_c, np));
  VBX_CUDA(c, dmalloc(&S.ray_list, np));
  VBX_CUDA(c, dmalloc(&S.head_list, np));
  VBX_CUDA(c, dmalloc(&S.touched_list, c->tab.touched_cap));
  VBX_CUDA(c, dmalloc(&S.cnt, np + 1));
  VBX_CUDA(c, dmalloc(&S.off, np + 1));
  VBX_CUDA(c, dmalloc(&S.sort_plan1, 1));
  VBX_CUDA(c, dmalloc(&S.sort_status1, (size_t)4 * c->sort_tiles_cap[1] * kRadix));
  VBX_CUDA(c, dmalloc(&S.d_state, 1));
  VBX_CUDA(c, cudaMallocHost(reinterpret_cast<void**>(&S.h_state), sizeof(ScanState)));
  return VBX_OK;
}

static void free_set(vbx_ctx::ScratchSet& S) {
  void* ptrs[] = {S.d_xyz, S.d_rgba, S.pkeys0, S.ckeys[0], S.ckeys[1], S.cvals[0], S.cvals[1], S.ray_p, S.ray_a,
                  S.ray_c, S.ray_list, S.head_list, S.touched_list, S.cnt, S.off, S.sort_plan1, S.sort_status1, S.d_state};
  for (void* p : ptrs) {
    if (p) cudaFree(p);
  }
  if (S.h_state) cudaFreeHost(S.h_state);
  cudaEvent_t evs[] = {S.copy_done, S.front_done, S.walked, S.sorted, S.back_done, S.applied, S.front_start};
  for (cudaEvent_t e : evs) {
    if (e) cudaEventDestroy(e);
  }
}

// The device buffers of one front lane, k_bundle_order's tables (vbx_order.cuh) among them (its streams
// and events are created by vbx_create / ensure_async).
static int alloc_lane(vbx_ctx* c, vbx_ctx::FrontLane& F) {
  const size_t np = c->max_points;
  VBX_CUDA(c, dmalloc(&F.pkeys1, np));
  VBX_CUDA(c, dmalloc(&F.pvals[0], np));
  VBX_CUDA(c, dmalloc(&F.pvals[1], np));
  VBX_CUDA(c, dmalloc(&F.sort_plan0, 1));
  VBX_CUDA(c, dmalloc(&F.sort_status0, (size_t)8 * c->sort_tiles_cap[0] * kRadix));
  VBX_CUDA(c, dmalloc(&F.scan_status, (np + 1) / kScanTile + 4));
  OrderScratch& g = F.order_scratch;
  g.cap = (uint32_t)np;
  // the bucket count after np insertions
  uint32_t buckets = 1;
  for (int k = 0; k < c->rehash.count && c->rehash.m[k] < np; ++k) buckets = c->rehash.n[k];
  g.bucket_cap = buckets;
  VBX_CUDA(c, dmalloc(&g.h, 2 * np));
  VBX_CUDA(c, dmalloc(&g.tau, np));
  VBX_CUDA(c, dmalloc(&g.tau2, np));
  VBX_CUDA(c, dmalloc(&g.next, np));
  VBX_CUDA(c, dmalloc(&g.bkt, np));
  VBX_CUDA(c, dmalloc(&g.A, np));
  VBX_CUDA(c, dmalloc(&g.bhead, (size_t)buckets));
  VBX_CUDA(c, dmalloc(&g.head_of, 2 * np));
  VBX_CUDA(c, dmalloc(&g.wp, 2 * (np / 32 + 2)));
  VBX_CUDA(c, dmalloc(&g.cta_tot, 64));
  VBX_CUDA(c, dmalloc(&F.big_list, np / 256 + 2));
  VBX_CUDA(c, dmalloc(&F.first_bits, 2 * (np / 32 + 2)));
  VBX_CUDA(c, cudaMemsetAsync(F.first_bits, 0, 2 * (np / 32 + 2) * sizeof(uint32_t), c->stream_main));
  return VBX_OK;
}

static void free_lane(vbx_ctx::FrontLane& F) {
  const OrderScratch& g = F.order_scratch;
  void* ptrs[] = {F.pkeys1, F.pvals[0], F.pvals[1], F.sort_plan0, F.sort_status0, F.scan_status, F.big_list, F.first_bits,
                  g.h,      g.tau,      g.tau2,     g.next,       g.bkt,          g.A,           g.bhead,    g.head_of,
                  g.wp,     g.cta_tot};
  for (void* p : ptrs) {
    if (p) cudaFree(p);
  }
  if (F.side) {
    cudaStreamSynchronize(F.side);
    cudaStreamDestroy(F.side);
  }
  if (F.ev_fork) cudaEventDestroy(F.ev_fork);
  if (F.ev_join) cudaEventDestroy(F.ev_join);
  if (F.stream) cudaStreamDestroy(F.stream);
}

}  // namespace vbx

using namespace vbx;

// every synchronous entry point first waits for asynchronously submitted scans (and reports a
// deferred error of theirs)
#define VBX_DRAIN(c)                          \
  do {                                        \
    if (int _rc = drain_async(c)) return _rc; \
  } while (0)

extern "C" {

const char* vbx_version(void) { return "voxblox_b200 0.1 (sm_100a)"; }

const char* vbx_last_error(const vbx_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int vbx_create(const vbx_tsdf_config* cfg, float voxel_size, int voxels_per_side,
               const vbx_engine_options* opt_in, vbx_ctx** out) {
  if (!cfg || !out) return VBX_E_INVALID;
  *out = nullptr;
  if (!(voxel_size > 0.0f)) return VBX_E_INVALID;  // CHECK_GT(voxel_size_, 0.0f), core/layer.h:38
  if (voxels_per_side <= 0 || voxels_per_side > 16 || (voxels_per_side & (voxels_per_side - 1))) {
    return VBX_E_INVALID;  // CHECK(isPowerOfTwo(voxels_per_side)), core/common.h:239
  }
  vbx_ctx* c = new vbx_ctx;
  c->cfg = *cfg;
  // TsdfIntegratorBase ctor, tsdf_integrator.cc:57-64
  if (c->cfg.integrator_threads == 0) c->cfg.integrator_threads = 1;
  if (c->cfg.allow_clear && !c->cfg.voxel_carving_enabled) c->cfg.allow_clear = 0;
  vbx_engine_options o;
  std::memset(&o, 0, sizeof(o));
  if (opt_in) o = *opt_in;
  int cur = 0;
  cudaError_t e = cudaGetDevice(&cur);
  if (e != cudaSuccess) {
    delete c;
    return VBX_E_CUDA;
  }
  if (!opt_in || opt_in->device < 0) o.device = cur;
  if (o.max_blocks == 0) o.max_blocks = 32768;
  if (o.max_points_per_scan == 0) o.max_points_per_scan = 1u << 20;
  if (o.max_updates_per_pass == 0) o.max_updates_per_pass = 1ull << 26;
  if (o.world_size <= 0) o.world_size = 1;
  c->opt = o;
  c->device = o.device;
  c->voxel_size = voxel_size;
  c->voxel_size_inv = (float)(1.0 / voxel_size);  // setLayer, tsdf_integrator.cc:77
  c->vps = voxels_per_side;
  c->L = 0;
  while ((1 << c->L) < voxels_per_side) ++c->L;
  c->vox_per_block = 1u << (3 * c->L);
  c->max_points = o.max_points_per_scan;
  c->max_updates = std::min<uint64_t>(o.max_updates_per_pass, 0x7fffffffull);
  int rb = 0;
  for (uint32_t v = o.max_blocks; v; v >>= 1) ++rb;
  // an update record's key = (touched id, voxel in block) in 32 bits with 0xffffffff reserved: a single
  // call may touch up to 2^(32 - 3L) - 1 blocks; the pool itself is only bounded by memory
  if (rb > 30) {
    delete c;
    return VBX_E_INVALID;
  }
  if (o.world_size > 1 && (o.rank < 0 || o.rank >= o.world_size)) {
    delete c;
    return VBX_E_INVALID;
  }
  *out = c;  // from here on the caller can read vbx_last_error and must vbx_destroy
#define CK(expr)                                   \
  do {                                             \
    cudaError_t _e = (expr);                       \
    if (_e != cudaSuccess) return cuda_fail(c, _e, #expr); \
  } while (0)
  CK(cudaSetDevice(c->device));
  {
    int sms = 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device) == cudaSuccess && sms > 0) c->grid_sms = (unsigned int)sms;
    if (const char* e = std::getenv("VBX_GRID_SMS")) c->grid_sms = (unsigned int)std::max(1, std::atoi(e));
  }
  // stream priorities for the pipelined path: the stages that run in submission order (apply, then
  // the ray walk) are the pipeline's bottleneck, so their thread blocks go first
  int prio_lo = 0, prio_hi = 0;
  CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));  // numerically lower = higher priority
  c->prio_lo = prio_lo;
  c->prio_hi = prio_hi;
  CK(cudaStreamCreateWithPriority(&c->stream_main, cudaStreamNonBlocking, prio_hi));
  CK(cudaStreamCreateWithFlags(&c->stream_c, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&c->stream_c2, cudaStreamNonBlocking));
  CK(cudaEventCreate(&c->ev0));
  CK(cudaEventCreate(&c->ev1));
  CK(cudaEventCreate(&c->tev0));
  CK(cudaEventCreate(&c->tev1));
  for (int i = 0; i < 20; ++i) CK(cudaEventCreate(&c->sev[i]));
  uint32_t hcap = 1;
  while (hcap < 2 * o.max_blocks) hcap <<= 1;
  c->hcap = hcap;
  Tables& t = c->tab;
  std::memset(&t, 0, sizeof(t));
  t.hmask = hcap - 1;
  t.max_blocks = o.max_blocks;
  CK(dmalloc(&t.hkeys, hcap));
  CK(dmalloc(&t.hslot, hcap));
  CK(dmalloc(&t.htouch, hcap));
  CK(dmalloc(&t.new_list, o.max_blocks));
  // ids lost to first-touch races stay unused (vbx_hash.cuh); (id, voxel) must fit a 32-bit record key
  t.touched_cap = (uint32_t)std::min<uint64_t>((uint64_t)o.max_blocks + 65536u, (0xffffffffull >> (3 * c->L)) - 1);
  t.vox_per_block = c->vox_per_block;
  CK(dmalloc(&t.slot_key, o.max_blocks));
  CK(dmalloc(&t.slot_updated, o.max_blocks));
  CK(dmalloc(&t.slot_esdf_updated, o.max_blocks));
  CK(dmalloc(&t.slot_has_esdf, o.max_blocks));
  CK(dmalloc(&t.tsdf, (size_t)o.max_blocks * c->vox_per_block));
  CK(cudaMemsetAsync(t.hkeys, 0xff, (size_t)hcap * sizeof(uint64_t), c->stream_main));
  CK(cudaMemsetAsync(t.hslot, 0xff, (size_t)hcap * sizeof(int32_t), c->stream_main));
  CK(cudaMemsetAsync(t.htouch, 0, (size_t)hcap * sizeof(unsigned long long), c->stream_main));
  CK(cudaMemsetAsync(t.slot_updated, 0, o.max_blocks, c->stream_main));
  CK(cudaMemsetAsync(t.slot_esdf_updated, 0, o.max_blocks, c->stream_main));
  CK(cudaMemsetAsync(t.slot_has_esdf, 0, o.max_blocks, c->stream_main));
  // new Block: voxels default-constructed = all zero bytes (core/voxel.h:12-16)
  CK(cudaMemsetAsync(t.tsdf, 0, (size_t)o.max_blocks * c->vox_per_block * sizeof(TsdfVoxel), c->stream_main));
  const size_t np = c->max_points;
  c->sort_tiles_cap[0] = (uint32_t)((np + kSortTile - 1) / kSortTile);
  c->sort_tiles_cap[1] = (uint32_t)((c->max_updates + kSortTile - 1) / kSortTile);
  if (int rc = init_bundle_order(c)) return rc;
  // hand-off set 0 and front lane 0 serve the synchronous calls; ensure_async allocates the others
  if (int rc = alloc_set(c, c->set[0])) return rc;
  if (int rc = alloc_lane(c, c->lane[0])) return rc;
  CK(cudaMemsetAsync(c->set[0].d_state, 0, sizeof(ScanState), c->stream_main));
  CK(dmalloc(&c->order, np));
  CK(dmalloc(&c->order_inv, np));
  for (int l = 0; l < vbx_ctx::kLanes; ++l) {
    CK(cudaStreamCreateWithPriority(&c->lane[l].side, cudaStreamNonBlocking, prio_lo));
    CK(cudaEventCreateWithFlags(&c->lane[l].ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->lane[l].ev_join, cudaEventDisableTiming));
  }
  CK(dmalloc(&c->long_list, (size_t)(c->max_updates / 32 + 1)));
  CK(dmalloc(&c->long_end, (size_t)(c->max_updates / 32 + 1)));
  CK(dmalloc(&c->long_state, (size_t)(c->max_updates / 32 + 1)));
  CK(dmalloc(&c->verify_run, (size_t)(c->max_updates / 32 + 1)));
  CK(dmalloc(&c->verify_start, (size_t)(c->max_updates / 32 + 1)));
  CK(dmalloc(&c->rec_sdf, (size_t)c->max_updates));
  CK(dmalloc(&c->rec_w, (size_t)c->max_updates));
  CK(dmalloc(&c->set_start, 1u << 20));
  CK(dmalloc(&c->set_observed, 1u << 20));
  CK(cudaMemsetAsync(c->set_start, 0, sizeof(unsigned long long) << 20, c->stream_main));
  CK(cudaMemsetAsync(c->set_observed, 0, sizeof(unsigned long long) << 20, c->stream_main));
  CK(dmalloc(&c->d_nblocks, 2));
  CK(cudaMemsetAsync(c->d_nblocks, 0, 2 * sizeof(uint32_t), c->stream_main));
  CK(dmalloc(&c->d_hold, 1));
  CK(cudaMemsetAsync(c->d_hold, 0, sizeof(uint32_t), c->stream_main));
  CK(cudaStreamSynchronize(c->stream_main));
#undef CK
  return VBX_OK;
}

}  // extern "C" (reopened below)

namespace vbx {
// First asynchronous submission: the remaining hand-off sets and front lanes, streams, events.
int ensure_async(vbx_ctx* c) {
  if (c->async_ready) return VBX_OK;
#define CK(expr)                                           \
  do {                                                     \
    cudaError_t _e = (expr);                               \
    if (_e != cudaSuccess) return cuda_fail(c, _e, #expr); \
  } while (0)
  if (const char* e = std::getenv("VBX_ASYNC_SETS")) c->sets_in_use = std::max(2, std::min(std::atoi(e), (int)vbx_ctx::kSets));
  if (const char* e = std::getenv("VBX_ASYNC_LANES")) c->lanes_in_use = std::max(1, std::min(std::atoi(e), (int)vbx_ctx::kLanes));
  CK(cudaStreamCreateWithFlags(&c->stream_h, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithPriority(&c->stream_e, cudaStreamNonBlocking, std::min(c->prio_lo, c->prio_hi + 1)));
  for (int i = 0; i < vbx_ctx::kSortStreams; ++i) {
    CK(cudaStreamCreateWithPriority(&c->stream_s[i], cudaStreamNonBlocking, std::min(c->prio_lo, c->prio_hi + 2)));
  }
  for (int l = 0; l < c->lanes_in_use; ++l) {
    vbx_ctx::FrontLane& F = c->lane[l];
    CK(cudaStreamCreateWithPriority(&F.stream, cudaStreamNonBlocking, c->prio_lo));
    if (l > 0) {
      if (int rc = alloc_lane(c, F)) return rc;
    }
  }
  // diagnostic: with VBX_ASYNC_TIMELINE set the hand-off events keep timestamps (vbx_debug_async_timeline)
  c->timeline = std::getenv("VBX_ASYNC_TIMELINE") != nullptr;
  const unsigned int evf = c->timeline ? cudaEventDefault : cudaEventDisableTiming;
  if (c->timeline) {
    CK(cudaEventCreate(&c->timeline_ref));
    CK(cudaEventRecord(c->timeline_ref, c->stream_main));
  }
  for (int k = 0; k < c->sets_in_use; ++k) {
    vbx_ctx::ScratchSet& S = c->set[k];
    CK(cudaEventCreateWithFlags(&S.copy_done, evf));
    CK(cudaEventCreateWithFlags(&S.front_done, evf));
    CK(cudaEventCreateWithFlags(&S.walked, evf));
    CK(cudaEventCreateWithFlags(&S.sorted, evf));
    CK(cudaEventCreateWithFlags(&S.back_done, evf));
    CK(cudaEventCreateWithFlags(&S.applied, evf));
    if (c->timeline) CK(cudaEventCreate(&S.front_start));
    if (k > 0) {
      if (int rc = alloc_set(c, S)) return rc;
    }
  }
#undef CK
  c->async_ready = true;
  return VBX_OK;
}
}  // namespace vbx

extern "C" {

void vbx_destroy(vbx_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream_main) cudaStreamSynchronize(c->stream_main);
  if (c->stream_c) cudaStreamSynchronize(c->stream_c);
  if (c->stream_c2) cudaStreamSynchronize(c->stream_c2);
  if (c->stream_h) cudaStreamSynchronize(c->stream_h);
  if (c->stream_e) cudaStreamSynchronize(c->stream_e);
  for (int i = 0; i < vbx_ctx::kSortStreams; ++i) {
    if (c->stream_s[i]) cudaStreamSynchronize(c->stream_s[i]);
  }
  for (int l = 0; l < vbx_ctx::kLanes; ++l) {
    if (c->lane[l].stream) cudaStreamSynchronize(c->lane[l].stream);
  }
  esdf_destroy(c);
  mesh_destroy(c);
  icp_destroy(c);
  Tables& t = c->tab;
  void* ptrs[] = {t.hkeys, t.hslot, t.htouch, t.new_list, t.slot_key, t.slot_updated, t.slot_esdf_updated,
                  t.slot_has_esdf, t.tsdf, c->order, c->order_inv, c->set_start, c->set_observed, c->long_list,
                  c->long_end, c->long_state, c->verify_run, c->verify_start, c->rec_sdf, c->rec_w, c->d_nblocks, c->d_hold};
  for (void* p : ptrs) {
    if (p) cudaFree(p);
  }
  if (c->mirror_dev) cudaFree(c->mirror_dev);
  if (c->mirror_host) cudaFreeHost(c->mirror_host);
  if (c->mirror_slots) cudaFree(c->mirror_slots);
  for (vbx_ctx::ScratchSet& S : c->set) free_set(S);
  for (vbx_ctx::FrontLane& F : c->lane) free_lane(F);
  if (c->timeline_ref) cudaEventDestroy(c->timeline_ref);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->tev0) cudaEventDestroy(c->tev0);
  if (c->tev1) cudaEventDestroy(c->tev1);
  for (int i = 0; i < 20; ++i) {
    if (c->sev[i]) cudaEventDestroy(c->sev[i]);
  }
  if (c->stream_main) cudaStreamDestroy(c->stream_main);
  if (c->stream_e) cudaStreamDestroy(c->stream_e);
  for (int i = 0; i < vbx_ctx::kSortStreams; ++i) {
    if (c->stream_s[i]) cudaStreamDestroy(c->stream_s[i]);
  }
  if (c->stream_c) cudaStreamDestroy(c->stream_c);
  if (c->stream_c2) cudaStreamDestroy(c->stream_c2);
  if (c->stream_h) cudaStreamDestroy(c->stream_h);
  delete c;
}

int vbx_get_tsdf_config(const vbx_ctx* c, vbx_tsdf_config* out) {
  if (!c || !out) return VBX_E_INVALID;
  *out = c->cfg;
  return VBX_OK;
}

int vbx_tsdf_integrate_device(vbx_ctx* c, int kind, const float q[4], const float t[3], const float* d_xyz,
                              const uint8_t* d_rgba, uint64_t n, int freespace) {
  if (!c || !q || !t || (n && (!d_xyz || !d_rgba))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return integrate_device(c, kind, q, t, d_xyz, d_rgba, n, freespace);
}

int vbx_tsdf_integrate(vbx_ctx* c, int kind, const float q[4], const float t[3], const float* xyz,
                       const uint8_t* rgba, uint64_t n, int freespace) {
  if (!c || !q || !t || (n && (!xyz || !rgba))) return fail(c, VBX_E_INVALID, "null argument");
  if (n > c->max_points) return fail(c, VBX_E_CAPACITY, "cloud larger than max_points_per_scan");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (n) {
    VBX_CUDA(c, cudaMemcpyAsync(c->set[0].d_xyz, xyz, n * 3 * sizeof(float), cudaMemcpyHostToDevice, c->stream_main));
    VBX_CUDA(c, cudaMemcpyAsync(c->set[0].d_rgba, rgba, n * 4, cudaMemcpyHostToDevice, c->stream_main));
  }
  return integrate_device(c, kind, q, t, c->set[0].d_xyz, c->set[0].d_rgba, n, freespace);
}

int vbx_tsdf_integrate_async(vbx_ctx* c, int kind, const float q[4], const float t[3], const float* xyz,
                             const uint8_t* rgba, uint64_t n, int freespace, int inputs_on_device) {
  if (!c || !q || !t || (n && (!xyz || !rgba))) return fail(c, VBX_E_INVALID, "null argument");
  if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, VBX_E_CUDA, "cudaSetDevice");
  return integrate_async(c, kind, q, t, xyz, rgba, n, freespace, inputs_on_device);
}

int vbx_block_owner(const vbx_ctx* c, const int32_t block_index[3], int32_t* owner) {
  if (!c || !block_index || !owner) return VBX_E_INVALID;
  *owner = c->opt.world_size > 1 ? block_owner(block_index[0], block_index[1], block_index[2], c->opt.world_size) : 0;
  return VBX_OK;
}

int vbx_debug_sort(vbx_ctx* c, const void* keys, int key_bytes, uint32_t n, int key_bits, void* keys_out,
                   uint32_t* vals_out) {
  if (!c || (n && (!keys || !keys_out || !vals_out))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return debug_sort(c, keys, key_bytes, n, key_bits, keys_out, vals_out);
}

int vbx_debug_async_timeline(vbx_ctx* c, uint64_t* seq, float* ms, int cap_sets) {
  if (!c || !seq || !ms) return VBX_E_INVALID;
  if (!c->async_ready || !c->timeline) return fail(c, VBX_E_STATE, "set VBX_ASYNC_TIMELINE before the first asynchronous submission");
  for (int k = 0; k < cap_sets; ++k) {
    if (k >= c->sets_in_use) {
      seq[k] = ~0ull;
      continue;
    }
    vbx_ctx::ScratchSet& S = c->set[k];
    seq[k] = S.seq;
    cudaEvent_t ev[5] = {S.front_start, S.front_done, S.walked, S.sorted, S.applied};
    for (int j = 0; j < 5; ++j) {
      float t = -1.f;
      if (cudaEventSynchronize(ev[j]) != cudaSuccess || cudaEventElapsedTime(&t, c->timeline_ref, ev[j]) != cudaSuccess) {
        t = -1.f;
        cudaGetLastError();
      }
      ms[5 * k + j] = t;
    }
  }
  return VBX_OK;
}

int vbx_debug_scan(vbx_ctx* c, const uint32_t* in, uint32_t n, uint32_t* out) {
  if (!c || (n && (!in || !out))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return debug_scan(c, in, n, out);
}

int vbx_debug_bundle_order(vbx_ctx* c, const uint32_t* hashes, uint32_t n, int force_global, uint32_t* out) {
  if (!c || (n && (!hashes || !out))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return debug_bundle_order(c, hashes, n, force_global, out);
}

int vbx_get_counters(const vbx_ctx* c, uint64_t out[16]) {
  if (!c || !out) return VBX_E_INVALID;
  std::memcpy(out, c->counters, sizeof(c->counters));
  out[8] = c->launches;  // kernels launched by TSDF integration since vbx_create
  out[13] = c->async_redone;  // asynchronously submitted scans that were redone synchronously (see vbx_tsdf_integrate_async)
  out[14] = c->async_wait_ns;    // host time asynchronous submissions spent waiting for a free hand-off set ...
  out[15] = c->async_submit_ns;  // ... and enqueueing (cumulative, ns)
  return VBX_OK;
}

int vbx_esdf_get_counters(const vbx_ctx* c, uint64_t out[16]) {
  if (!c || !out) return VBX_E_INVALID;
  std::memcpy(out, c->esdf_counters, sizeof(c->esdf_counters));
  return VBX_OK;
}

int vbx_last_device_ms(const vbx_ctx* c, float* ms) {
  if (!c || !ms) return VBX_E_INVALID;
  *ms = c->last_ms;
  return VBX_OK;
}

int vbx_host_alloc(vbx_ctx* c, size_t bytes, void** out) {
  if (!c || !out) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  VBX_CUDA(c, cudaHostAlloc(out, bytes, cudaHostAllocPortable));
  return VBX_OK;
}

int vbx_host_free(vbx_ctx* c, void* p) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaFreeHost(p));
  return VBX_OK;
}

int vbx_host_copy_ms(vbx_ctx* c, const void* src, size_t bytes, float* ms) {
  if (!c || !src || !ms) return VBX_E_INVALID;
  if (bytes > (size_t)c->max_points * 12) return fail(c, VBX_E_CAPACITY, "copy larger than the staging buffer");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  VBX_CUDA(c, cudaEventRecord(c->tev0, c->stream_main));
  VBX_CUDA(c, cudaMemcpyAsync(c->set[0].d_xyz, src, bytes, cudaMemcpyHostToDevice, c->stream_main));
  VBX_CUDA(c, cudaEventRecord(c->tev1, c->stream_main));
  VBX_CUDA(c, cudaEventSynchronize(c->tev1));
  VBX_CUDA(c, cudaEventElapsedTime(ms, c->tev0, c->tev1));
  return VBX_OK;
}

int vbx_timer_start(vbx_ctx* c) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  VBX_CUDA(c, cudaEventRecord(c->tev0, c->stream_main));
  return VBX_OK;
}

int vbx_timer_stop_ms(vbx_ctx* c, float* ms) {
  if (!c || !ms) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  VBX_CUDA(c, cudaEventRecord(c->tev1, c->stream_main));
  VBX_CUDA(c, cudaEventSynchronize(c->tev1));
  VBX_CUDA(c, cudaEventElapsedTime(ms, c->tev0, c->tev1));
  return VBX_OK;
}

int vbx_set_stage_profiling(vbx_ctx* c, int enabled) {
  if (!c) return VBX_E_INVALID;
  c->profiling = enabled != 0;
  std::memset(c->stage_ms, 0, sizeof(c->stage_ms));
  std::memset(c->stage_calls, 0, sizeof(c->stage_calls));
  return VBX_OK;
}

int vbx_get_stage_ms(const vbx_ctx* c, double ms[16], uint64_t calls[16]) {
  if (!c || !ms || !calls) return VBX_E_INVALID;
  std::memcpy(ms, c->stage_ms, sizeof(c->stage_ms));
  std::memcpy(calls, c->stage_calls, sizeof(c->stage_calls));
  return VBX_OK;
}

int vbx_sync(vbx_ctx* c) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));  // (the drain above already waited for every queued scan)
  return VBX_OK;
}

// Per-slot flag bytes of a layer with the engine's internal bits resolved: `has` = the layer holds a
// block in this slot, `upd` = Block::updated() bits only.
static int fetch_flags(vbx_ctx* c, int layer, std::vector<uint8_t>* upd, std::vector<uint8_t>* has) {
  upd->resize(c->n_blocks);
  has->assign(c->n_blocks, 1);
  if (c->n_blocks == 0) return VBX_OK;
  const uint8_t* src = (layer == VBX_LAYER_TSDF) ? c->tab.slot_updated : c->tab.slot_esdf_updated;
  VBX_CUDA(c, cudaMemcpyAsync(upd->data(), src, c->n_blocks, cudaMemcpyDeviceToHost, c->stream_main));
  if (layer == VBX_LAYER_ESDF) {
    VBX_CUDA(c, cudaMemcpyAsync(has->data(), c->tab.slot_has_esdf, c->n_blocks, cudaMemcpyDeviceToHost,
                                c->stream_main));
  }
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  for (uint32_t s = 0; s < c->n_blocks; ++s) {
    if (layer == VBX_LAYER_TSDF && ((*upd)[s] & kSlotNoTsdf)) (*has)[s] = 0;
    (*upd)[s] &= 0x07;  // kSlotNoTsdf / kEsdfPending / the mirror mark are internal
  }
  return VBX_OK;
}

int vbx_num_blocks(vbx_ctx* c, int layer, uint64_t* n) {
  if (!c || !n) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (layer == VBX_LAYER_TSDF && !c->maybe_esdf_only) {
    *n = c->n_blocks;
    return VBX_OK;
  }
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) {
    *n = 0;
    return VBX_OK;
  }
  std::vector<uint8_t> upd, has;
  if (int rc = fetch_flags(c, layer, &upd, &has)) return rc;
  uint64_t k = 0;
  for (uint8_t h : has) k += h ? 1 : 0;
  *n = k;
  return VBX_OK;
}

int vbx_list_blocks(vbx_ctx* c, int layer, int updated_mask, int32_t* idx3, uint64_t cap, uint64_t* n) {
  if (!c || !n) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  *n = 0;
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) return VBX_OK;
  if (int rc = refresh_host_mirror(c)) return rc;
  std::vector<uint8_t> upd, has;
  if (int rc = fetch_flags(c, layer, &upd, &has)) return rc;
  struct K3 {
    int x, y, z;
  };
  std::vector<K3> keys;
  keys.reserve(c->n_blocks);
  for (uint32_t s = 0; s < c->n_blocks; ++s) {
    if (!has[s]) continue;
    if (updated_mask && !(upd[s] & updated_mask)) continue;
    K3 k;
    unpack3(c->host_slot_key[s], &k.x, &k.y, &k.z);
    keys.push_back(k);
  }
  std::sort(keys.begin(), keys.end(), [](const K3& a, const K3& b) {
    if (a.x != b.x) return a.x < b.x;
    if (a.y != b.y) return a.y < b.y;
    return a.z < b.z;
  });
  *n = keys.size();
  if (idx3) {
    const uint64_t m = std::min<uint64_t>(cap, keys.size());
    for (uint64_t i = 0; i < m; ++i) {
      idx3[3 * i] = keys[i].x;
      idx3[3 * i + 1] = keys[i].y;
      idx3[3 * i + 2] = keys[i].z;
    }
  }
  return VBX_OK;
}

int vbx_download_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m, void* voxels,
                        uint8_t* updated_bits) {
  if (!c || (m && (!idx3 || !voxels))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) return fail(c, VBX_E_STATE, "no ESDF layer");
  if (int rc = refresh_host_mirror(c)) return rc;
  std::vector<uint8_t> upd, has;
  if (int rc = fetch_flags(c, layer, &upd, &has)) return rc;
  const size_t vbytes = (layer == VBX_LAYER_TSDF) ? sizeof(TsdfVoxel) : sizeof(EsdfVoxel);
  const size_t bbytes = vbytes * c->vox_per_block;
  const char* pool = (layer == VBX_LAYER_TSDF) ? reinterpret_cast<const char*>(c->tab.tsdf)
                                               : reinterpret_cast<const char*>(c->tab.esdf);
  for (uint64_t i = 0; i < m; ++i) {
    auto it = c->host_key2slot.find(pack3(idx3[3 * i], idx3[3 * i + 1], idx3[3 * i + 2]));
    if (it == c->host_key2slot.end() || !has[it->second]) return fail(c, VBX_E_NOT_FOUND, "block not allocated");
    VBX_CUDA(c, cudaMemcpyAsync(static_cast<char*>(voxels) + i * bbytes, pool + (size_t)it->second * bbytes,
                                bbytes, cudaMemcpyDeviceToHost, c->stream_main));
    if (updated_bits) updated_bits[i] = upd[it->second];
  }
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  return VBX_OK;
}

int vbx_mirror_updated(vbx_ctx* c, int layer, int updated_mask, int clear_mask, int32_t* idx3, void* voxels,
                       uint8_t* updated_bits, uint64_t cap, uint64_t* n) {
  if (!c || !n || (cap && (!idx3 || !voxels))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  *n = 0;
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) return VBX_OK;
  return mirror_updated(c, layer, updated_mask, clear_mask, idx3, voxels, updated_bits, cap, n, 0);
}

int vbx_serialize_updated(vbx_ctx* c, int layer, int updated_mask, int clear_mask, int32_t* idx3, uint32_t* words,
                          uint8_t* updated_bits, uint64_t cap, uint64_t* n) {
  if (!c || !n || (cap && (!idx3 || !words))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  *n = 0;
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) return VBX_OK;
  return mirror_updated(c, layer, updated_mask, clear_mask, idx3, words, updated_bits, cap, n, 1);
}

int vbx_deserialize_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m, const uint32_t* words,
                           const uint8_t* updated_bits) {
  if (!c || (m && (!idx3 || !words))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return upload_blocks(c, layer, idx3, m, words, updated_bits, 1);
}

int vbx_clear_updated(vbx_ctx* c, int layer, int updated_mask) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (c->n_blocks == 0) return VBX_OK;
  std::vector<uint8_t> upd(c->n_blocks);
  uint8_t* dst = (layer == VBX_LAYER_TSDF) ? c->tab.slot_updated : c->tab.slot_esdf_updated;
  VBX_CUDA(c, cudaMemcpyAsync(upd.data(), dst, c->n_blocks, cudaMemcpyDeviceToHost, c->stream_main));
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  for (uint8_t& u : upd) u &= (uint8_t)(~updated_mask | 0x80);  // bit 7 is the engine's own (kSlotNoTsdf / kEsdfPending)
  VBX_CUDA(c, cudaMemcpyAsync(dst, upd.data(), c->n_blocks, cudaMemcpyHostToDevice, c->stream_main));
  VBX_CUDA(c, cudaStreamSynchronize(c->stream_main));
  return VBX_OK;
}

int vbx_upload_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m, const void* voxels,
                      const uint8_t* updated_bits) {
  if (!c || (m && (!idx3 || !voxels))) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return upload_blocks(c, layer, idx3, m, voxels, updated_bits, 0);
}

int vbx_remove_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m) {
  if (!c || (m && !idx3)) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return remove_blocks(c, layer, idx3, m);
}

int vbx_clear(vbx_ctx* c, int layer) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return clear_layer(c, layer);
}

int vbx_esdf_create(vbx_ctx* c, const vbx_esdf_config* cfg) {
  if (!c || !cfg) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return esdf_create(c, cfg);
}

int vbx_esdf_update(vbx_ctx* c, int batch, int clear_updated_flag) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (!c->has_esdf) return fail(c, VBX_E_STATE, "vbx_esdf_update before vbx_esdf_create");
  return esdf_update(c, batch, clear_updated_flag);
}

int vbx_esdf_update_blocks(vbx_ctx* c, const int32_t* idx3, uint64_t m, int incremental) {
  if (!c || (m && !idx3)) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (!c->has_esdf) return fail(c, VBX_E_STATE, "vbx_esdf_update_blocks before vbx_esdf_create");
  return esdf_update_blocks(c, idx3, m, incremental);
}

int vbx_mesh_generate(vbx_ctx* c, const vbx_mesh_config* cfg, int only_mesh_updated_blocks, int clear_updated_flag,
                      uint64_t* n_blocks, uint64_t* n_vertices) {
  if (!c || !cfg) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return mesh_generate(c, cfg, only_mesh_updated_blocks, clear_updated_flag, n_blocks, n_vertices);
}

int vbx_icp_run(vbx_ctx* c, const vbx_icp_config* cfg, const float* points_C, uint64_t n, const float q_wxyz[4],
                const float t[3], uint32_t seed, float out_q_wxyz[4], float out_t[3], uint64_t* num_updates) {
  if (!c || !cfg || (n && !points_C) || !q_wxyz || !t || !out_q_wxyz || !out_t) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return icp_run(c, cfg, points_C, 0, n, q_wxyz, t, seed, out_q_wxyz, out_t, num_updates);
}

int vbx_icp_run_device(vbx_ctx* c, const vbx_icp_config* cfg, const float* d_points_C, uint64_t n, const float q_wxyz[4],
                       const float t[3], uint32_t seed, float out_q_wxyz[4], float out_t[3], uint64_t* num_updates) {
  if (!c || !cfg || (n && !d_points_C) || !q_wxyz || !t || !out_q_wxyz || !out_t) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  return icp_run(c, cfg, d_points_C, 1, n, q_wxyz, t, seed, out_q_wxyz, out_t, num_updates);
}

int vbx_mesh_download(vbx_ctx* c, int32_t* idx3, uint64_t* first_vertex, float* vertices, float* normals,
                      uint8_t* colors) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  return mesh_download(c, idx3, first_vertex, vertices, normals, colors);
}

int vbx_esdf_add_robot_position(vbx_ctx* c, const float position[3]) {
  if (!c || !position) return fail(c, VBX_E_INVALID, "null argument");
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (!c->has_esdf) return fail(c, VBX_E_STATE, "vbx_esdf_add_robot_position before vbx_esdf_create");
  return esdf_add_robot_position(c, position);
}

int vbx_esdf_clear(vbx_ctx* c) {
  if (!c) return VBX_E_INVALID;
  VBX_CUDA(c, cudaSetDevice(c->device));
  VBX_DRAIN(c);
  if (!c->has_esdf) return fail(c, VBX_E_STATE, "no ESDF integrator");
  return esdf_clear_state(c);
}

int vbx_esdf_set_max_distance(vbx_ctx* c, float max_distance_m) {
  if (!c) return VBX_E_INVALID;
  if (!c->has_esdf) return fail(c, VBX_E_STATE, "no ESDF integrator");
  // setEsdfMaxDistance, esdf_integrator.h:140-145: the default distance follows upwards
  c->ecfg.max_distance_m = max_distance_m;
  if (c->ecfg.default_distance_m < max_distance_m) c->ecfg.default_distance_m = max_distance_m;
  return VBX_OK;
}

int vbx_esdf_set_full_euclidean(vbx_ctx* c, int full_euclidean) {
  if (!c) return VBX_E_INVALID;
  if (!c->has_esdf) return fail(c, VBX_E_STATE, "no ESDF integrator");
  c->ecfg.full_euclidean_distance = full_euclidean ? 1 : 0;  // esdf_integrator.h:147-149
  return VBX_OK;
}

int vbx_esdf_get_config(const vbx_ctx* c, vbx_esdf_config* out) {
  if (!c || !out) return VBX_E_INVALID;
  if (!c->has_esdf) return VBX_E_STATE;
  *out = c->ecfg;
  return VBX_OK;
}

}  // extern "C"
