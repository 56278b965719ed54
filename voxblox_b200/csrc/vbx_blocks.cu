// Host-driven block management of the device map: the counterparts of Layer::insertBlock /
// allocateBlockPtrByIndex (+ voxel copy), removeBlock and removeAllBlocks
// (voxblox/include/voxblox/core/layer.h:103-111,152-164).  None of this is on the per-scan hot
// path; it exists so that host code which edits the Layer between scans (loading a map,
// TsdfServer's removeDistantBlocks, voxblox_ros/src/tsdf_server.cc:314-316) can keep the HBM map
// of record in step.
#include <algorithm>
#include <cstring>
#include <vector>

#include "vbx_engine.h"
#include "vbx_hash.cuh"

namespace vbx {

__global__ void k_ensure_keys(Tables tab, const uint64_t* __restrict__ keys, uint32_t m, uint32_t* __restrict__ hp_out,
                              ScanState* st) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  hp_out[i] = ensure_block(tab, keys[i], st);
}

__global__ void k_assign_uploaded(Tables tab, uint32_t n_blocks_before, uint8_t new_slot_flags, ScanState* st) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t n_new = min(st->n_new, tab.max_blocks);
  if (j < n_new) {
    const uint32_t slot = n_blocks_before + j;
    if (slot < tab.max_blocks) {
      const uint32_t hp = tab.new_list[j];
      tab.hslot[hp] = (int32_t)slot;
      tab.slot_key[slot] = tab.hkeys[hp];
      tab.slot_updated[slot] = new_slot_flags;
    } else {
      atomicOr(&st->error, kErrPoolFull);
    }
  }
  if (j == 0) st->n_blocks = min(n_blocks_before + st->n_new, tab.max_blocks);
}

__global__ void k_slots_of(Tables tab, const uint32_t* __restrict__ hp, uint32_t m, int32_t* __restrict__ slot_out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  slot_out[i] = hp[i] == 0xffffffffu ? -1 : tab.hslot[hp[i]];
}

// rebuild the hash from the per-slot keys (after blocks were removed and the pool compacted)
__global__ void k_rebuild_hash(Tables tab, uint32_t n_blocks) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_blocks) return;
  const uint64_t key = tab.slot_key[s];
  uint32_t hp = hash64(key) & tab.hmask;
  while (true) {
    const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(tab.hkeys + hp),
                                             (unsigned long long)kEmptyKey, (unsigned long long)key);
    if (old == kEmptyKey) {
      tab.hslot[hp] = (int32_t)s;
      return;
    }
    hp = (hp + 1) & tab.hmask;
  }
}

static inline unsigned int grid_for(uint64_t n, int block) { return (unsigned int)((n + block - 1) / block); }

// The block hash rebuilt from slot_key: after removals, and after a call that ran out of pool slots
// (its surplus hash entries have no slot and must not be found by later calls).
int rebuild_hash(vbx_ctx* c) {
  cudaStream_t s = c->stream_main;
  VBX_CUDA(c, cudaMemsetAsync(c->tab.hkeys, 0xff, (size_t)c->hcap * sizeof(uint64_t), s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.hslot, 0xff, (size_t)c->hcap * sizeof(int32_t), s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.htouch, 0, (size_t)c->hcap * sizeof(unsigned long long), s));
  if (c->n_blocks) k_rebuild_hash<<<grid_for(c->n_blocks, 256), 256, 0, s>>>(c->tab, c->n_blocks);
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  return VBX_OK;
}

// ---- serialised block payloads (SURVEY.md section 8f N2), voxblox/src/core/block.cc:
//   TsdfVoxel -> 3 words: distance bits, weight bits, a | b<<8 | g<<16 | r<<24      (cc:159-183, :65-90)
//   EsdfVoxel -> 2 words: distance bits, parent x,y,z as int8 in bytes 3,2,1 | flag byte
//                (observed 1, hallucinated 2, in_queue 4, fixed 8)                (cc:203-234, :110-135)
// serializeDirection (cc:8-41) ORs `int8 << shift` as a sign-extended int, so a negative y or z
// also sets every byte above it; reproduced bit for bit.
__device__ __forceinline__ uint32_t tsdf_word(uint32_t w, uint32_t k) { return k == 2u ? __byte_perm(w, 0, 0x0123) : w; }

__device__ __forceinline__ uint2 esdf_pack(const uint32_t* v) {
  auto clamp8 = [](int32_t x) { return (int)max(-128, min(127, x)); };
  uint32_t d = 0;
  d |= (uint32_t)(clamp8((int32_t)v[2]) << 24);
  d |= (uint32_t)(clamp8((int32_t)v[3]) << 16);
  d |= (uint32_t)(clamp8((int32_t)v[4]) << 8);
  const uint32_t f = v[1];  // four bool bytes: observed, hallucinated, in_queue, fixed
  uint32_t flag = 0;
  if (f & 0x000000ffu) flag |= 1u;
  if (f & 0x0000ff00u) flag |= 2u;
  if (f & 0x00ff0000u) flag |= 4u;
  if (f & 0xff000000u) flag |= 8u;
  return make_uint2(v[0], d | flag);
}

__device__ __forceinline__ void esdf_unpack(uint2 w, uint32_t* v) {
  v[0] = w.x;
  v[1] = ((w.y & 1u) ? 0x00000001u : 0u) | ((w.y & 2u) ? 0x00000100u : 0u) | ((w.y & 4u) ? 0x00010000u : 0u) |
         ((w.y & 8u) ? 0x01000000u : 0u);
  v[2] = (uint32_t)(int32_t)(int8_t)((w.y >> 24) & 0xffu);  // deserializeDirection, cc:43-63
  v[3] = (uint32_t)(int32_t)(int8_t)((w.y >> 16) & 0xffu);
  v[4] = (uint32_t)(int32_t)(int8_t)((w.y >> 8) & 0xffu);
}

// device pool -> contiguous words in block.cc's format; one thread per output word (TSDF) / voxel (ESDF)
__global__ void k_serialize_blocks(int layer, const uint32_t* __restrict__ pool, const uint32_t* __restrict__ slots,
                                   uint32_t m, uint32_t vox_per_block, uint32_t* __restrict__ out,
                                   uint8_t* __restrict__ flags, uint8_t clear_mask) {
  const uint32_t b = blockIdx.y;
  if (b >= m) return;
  const uint32_t slot = slots[b];
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (layer == VBX_LAYER_TSDF) {
    const uint32_t nw = 3u * vox_per_block;
    if (i < nw) out[(size_t)b * nw + i] = tsdf_word(__ldcs(pool + (size_t)slot * nw + i), i % 3u);
  } else if (i < vox_per_block) {
    const uint32_t* v = pool + ((size_t)slot * vox_per_block + i) * 5u;
    uint32_t w[5] = {v[0], v[1], v[2], v[3], v[4]};
    reinterpret_cast<uint2*>(out)[(size_t)b * vox_per_block + i] = esdf_pack(w);
  }
  if (i == 0 && clear_mask) flags[slot] &= (uint8_t)~clear_mask;
}

// contiguous payloads (raw voxel structs or block.cc words) -> pool slots; also the per-slot flags
__global__ void k_scatter_blocks(int layer, int serialized, const uint32_t* __restrict__ in,
                                 const int32_t* __restrict__ slots, uint32_t m, uint32_t vox_per_block,
                                 uint32_t* __restrict__ pool, const uint8_t* __restrict__ upd_in,
                                 uint8_t* __restrict__ flags, uint8_t* __restrict__ has_esdf) {
  const uint32_t b = blockIdx.y;
  if (b >= m) return;
  const int32_t slot = slots[b];
  if (slot < 0) return;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t wpv = (layer == VBX_LAYER_TSDF) ? 3u : 5u;
  if (!serialized || layer == VBX_LAYER_TSDF) {
    const uint32_t nw = wpv * vox_per_block;
    if (i < nw) {
      const uint32_t w = in[(size_t)b * nw + i];
      pool[(size_t)slot * nw + i] = (serialized ? tsdf_word(w, i % 3u) : w);  // the byte reversal is its own inverse
    }
  } else if (i < vox_per_block) {
    uint32_t v[5];
    esdf_unpack(reinterpret_cast<const uint2*>(in)[(size_t)b * vox_per_block + i], v);
    uint32_t* dst = pool + ((size_t)slot * vox_per_block + i) * 5u;
#pragma unroll
    for (int k = 0; k < 5; ++k) dst[k] = v[k];
  }
  if (i == 0) {
    flags[slot] = upd_in ? (uint8_t)(upd_in[b] & 0x07) : (uint8_t)0;  // (bit 7 is the engine's own; a TSDF upload clears kSlotNoTsdf)
    if (has_esdf) has_esdf[slot] = 1;
  }
}

static int ensure_staging(vbx_ctx* c, size_t bytes, size_t slots) {
  if (bytes <= c->mirror_cap_bytes && slots <= c->mirror_cap_slots) return VBX_OK;
  if (c->mirror_dev) cudaFree(c->mirror_dev);
  if (c->mirror_host) cudaFreeHost(c->mirror_host);
  if (c->mirror_slots) cudaFree(c->mirror_slots);
  c->mirror_dev = c->mirror_host = nullptr;
  c->mirror_slots = nullptr;
  c->mirror_cap_bytes = c->mirror_cap_slots = 0;
  const size_t want_b = std::max<size_t>(2 * bytes, 16u << 20), want_s = std::max<size_t>(2 * slots, 1024);
  VBX_CUDA(c, cudaMalloc(&c->mirror_dev, want_b));
  VBX_CUDA(c, cudaMallocHost(&c->mirror_host, want_b));
  VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mirror_slots), want_s * sizeof(uint32_t)));
  c->mirror_cap_bytes = want_b;
  c->mirror_cap_slots = want_s;
  return VBX_OK;
}

static size_t payload_bytes(const vbx_ctx* c, int layer, int serialized) {
  if (layer == VBX_LAYER_TSDF) return sizeof(TsdfVoxel) * c->vox_per_block;  // 3 words either way
  return (serialized ? 8u : sizeof(EsdfVoxel)) * c->vox_per_block;
}

// Layer::insertBlock / allocateBlockPtrByIndex + voxel copy, or Block(BlockProto) + deserializeFromIntegers
// (core/block_inl.h:73-109) when `serialized`: find-or-create the blocks, then ONE staged copy per
// chunk and a scatter kernel.
int upload_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m, const void* voxels,
                  const uint8_t* updated_bits, int serialized) {
  if (m == 0) return VBX_OK;
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) return fail(c, VBX_E_STATE, "no ESDF layer");
  if (m > c->tab.max_blocks) return fail(c, VBX_E_CAPACITY, "more blocks than the pool holds");
  cudaStream_t s = c->stream_main;
  std::vector<uint64_t> keys(m);
  for (uint64_t i = 0; i < m; ++i) {
    const int32_t* p = idx3 + 3 * i;
    const int lim = kCoordBias - 1;
    if (p[0] < -lim || p[0] > lim || p[1] < -lim || p[1] > lim || p[2] < -lim || p[2] > lim) {
      return fail(c, VBX_E_INVALID, "block index outside +-2^20");
    }
    keys[i] = pack3(p[0], p[1], p[2]);
  }
  // scratch of hand-off set 0: the point-key buffer holds the keys, the ray list the hash positions, cnt the slots
  if (m > c->max_points) return fail(c, VBX_E_CAPACITY, "upload more than max_points_per_scan blocks at once");
  vbx_ctx::ScratchSet& S = c->set[0];
  VBX_CUDA(c, cudaMemcpyAsync(S.pkeys0, keys.data(), m * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  VBX_CUDA(c, cudaMemsetAsync(S.d_state, 0, sizeof(ScanState), s));
  k_ensure_keys<<<grid_for(m, 256), 256, 0, s>>>(c->tab, S.pkeys0, (uint32_t)m, S.ray_list, S.d_state);
  // a block inserted into the ESDF layer at an index the TSDF layer does not hold occupies a slot of its own
  k_assign_uploaded<<<grid_for(c->tab.max_blocks, 256), 256, 0, s>>>(
      c->tab, c->n_blocks, layer == VBX_LAYER_ESDF ? kSlotNoTsdf : (uint8_t)0, S.d_state);
  k_slots_of<<<grid_for(m, 256), 256, 0, s>>>(c->tab, S.ray_list, (uint32_t)m, reinterpret_cast<int32_t*>(S.cnt));
  VBX_CUDA(c, cudaMemcpyAsync(S.h_state, S.d_state, sizeof(ScanState), cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  if (S.h_state->error & kFatalErrors) return fail(c, VBX_E_CAPACITY, "block pool / hash full during upload");
  if (layer == VBX_LAYER_ESDF && S.h_state->n_new) c->maybe_esdf_only = true;
  if (int rc = set_n_blocks(c, S.h_state->n_blocks)) return rc;
  const size_t bbytes = payload_bytes(c, layer, serialized);
  const uint32_t wpv = (layer == VBX_LAYER_TSDF) ? 3u : (serialized ? 1u : 5u);  // threads per voxel along x
  uint32_t* pool = layer == VBX_LAYER_TSDF ? reinterpret_cast<uint32_t*>(c->tab.tsdf) : reinterpret_cast<uint32_t*>(c->tab.esdf);
  uint8_t* flags = layer == VBX_LAYER_TSDF ? c->tab.slot_updated : c->tab.slot_esdf_updated;
  const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(m, (256ull << 20) / bbytes));
  if (int rc = ensure_staging(c, chunk * bbytes + chunk, chunk)) return rc;
  uint8_t* d_upd = static_cast<uint8_t*>(c->mirror_dev) + chunk * bbytes;
  for (uint64_t at = 0; at < m; at += chunk) {
    const uint64_t k = std::min<uint64_t>(chunk, m - at);
    VBX_CUDA(c, cudaMemcpyAsync(c->mirror_dev, static_cast<const char*>(voxels) + at * bbytes, k * bbytes,
                                cudaMemcpyHostToDevice, s));
    if (updated_bits) VBX_CUDA(c, cudaMemcpyAsync(d_upd, updated_bits + at, k, cudaMemcpyHostToDevice, s));
    const dim3 grid(grid_for((uint64_t)wpv * c->vox_per_block, 256), (unsigned int)k);
    k_scatter_blocks<<<grid, 256, 0, s>>>(layer, serialized, static_cast<const uint32_t*>(c->mirror_dev),
                                          reinterpret_cast<const int32_t*>(S.cnt) + at, (uint32_t)k,
                                          (uint32_t)c->vox_per_block, pool, updated_bits ? d_upd : nullptr, flags,
                                          layer == VBX_LAYER_ESDF ? c->tab.slot_has_esdf : nullptr);
    VBX_CUDA(c, cudaStreamSynchronize(s));  // the staging buffer is reused by the next chunk
  }
  VBX_CUDA(c, cudaGetLastError());
  return refresh_host_mirror(c);
}

int remove_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m);

// Layer::removeAllBlocks (core/layer.h:164) of ONE layer; the other layer keeps its blocks
int clear_layer(vbx_ctx* c, int layer) {
  cudaStream_t s = c->stream_main;
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) return VBX_OK;
  if (c->has_esdf && c->n_blocks) {
    // the layers share pool slots: remove this layer's block from every slot (slots that end up
    // empty are given back)
    if (int rc = refresh_host_mirror(c)) return rc;
    std::vector<int32_t> idx(3 * (size_t)c->n_blocks);
    for (uint32_t sl = 0; sl < c->n_blocks; ++sl) {
      int x, y, z;
      unpack3(c->host_slot_key[sl], &x, &y, &z);
      idx[3 * sl] = x;
      idx[3 * sl + 1] = y;
      idx[3 * sl + 2] = z;
    }
    return remove_blocks(c, layer, idx.data(), c->n_blocks);
  }
  c->has_data_keys[0].clear();
  c->has_data_keys[1].clear();
  // no ESDF layer: reset the whole map
  const size_t used = (size_t)c->n_blocks * c->vox_per_block;
  c->esdf_pending_raise = c->esdf_pending_open = 0;
  c->maybe_esdf_only = false;
  VBX_CUDA(c, cudaMemsetAsync(c->tab.tsdf, 0, used * sizeof(TsdfVoxel), s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.hkeys, 0xff, (size_t)c->hcap * sizeof(uint64_t), s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.hslot, 0xff, (size_t)c->hcap * sizeof(int32_t), s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.htouch, 0, (size_t)c->hcap * sizeof(unsigned long long), s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_updated, 0, c->tab.max_blocks, s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_esdf_updated, 0, c->tab.max_blocks, s));
  VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_has_esdf, 0, c->tab.max_blocks, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  if (int rc = set_n_blocks(c, 0)) return rc;
  c->host_slot_key.clear();
  c->host_key2slot.clear();
  return VBX_OK;
}

int remove_blocks(vbx_ctx* c, int layer, const int32_t* idx3, uint64_t m) {
  if (m == 0) return VBX_OK;
  cudaStream_t s = c->stream_main;
  if (int rc = refresh_host_mirror(c)) return rc;
  std::vector<int32_t> victims;
  for (uint64_t i = 0; i < m; ++i) {
    c->has_data_keys[layer == VBX_LAYER_ESDF ? 1 : 0].erase(pack3(idx3[3 * i], idx3[3 * i + 1], idx3[3 * i + 2]));
    auto it = c->host_key2slot.find(pack3(idx3[3 * i], idx3[3 * i + 1], idx3[3 * i + 2]));
    if (it != c->host_key2slot.end()) victims.push_back(it->second);  // erasing a missing block is a no-op
  }
  std::sort(victims.begin(), victims.end());
  victims.erase(std::unique(victims.begin(), victims.end()), victims.end());
  if (victims.empty()) return VBX_OK;
  const size_t tb = sizeof(TsdfVoxel) * c->vox_per_block, eb = sizeof(EsdfVoxel) * c->vox_per_block;
  if (layer == VBX_LAYER_ESDF && !c->has_esdf) return VBX_OK;
  // The two layers are independent in the reference (Layer::removeBlock = block_map_.erase, core/layer.h:163)
  // but share pool slots here: a slot is given back only when NEITHER layer holds a block in it.
  std::vector<uint8_t> upd(c->n_blocks), has(c->n_blocks, 0);
  VBX_CUDA(c, cudaMemcpyAsync(upd.data(), c->tab.slot_updated, c->n_blocks, cudaMemcpyDeviceToHost, s));
  if (c->has_esdf) VBX_CUDA(c, cudaMemcpyAsync(has.data(), c->tab.slot_has_esdf, c->n_blocks, cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  // queue entries of addNewRobotPosition address voxels by slot: they are dropped
  c->esdf_pending_raise = c->esdf_pending_open = 0;
  std::vector<int32_t> drop;  // slots that become free
  const uint8_t no_tsdf = kSlotNoTsdf;
  for (int32_t v : victims) {
    if (layer == VBX_LAYER_ESDF) {
      if (!has[v]) continue;  // erasing a missing block is a no-op
      VBX_CUDA(c, cudaMemsetAsync(reinterpret_cast<char*>(c->tab.esdf) + (size_t)v * eb, 0, eb, s));
      VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_has_esdf + v, 0, 1, s));
      VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_esdf_updated + v, 0, 1, s));
      if (upd[v] & kSlotNoTsdf) drop.push_back(v);
    } else {
      if (upd[v] & kSlotNoTsdf) continue;  // the TSDF layer holds no block here
      if (has[v]) {
        // the ESDF block stays; the slot's TSDF half reads as never allocated from now on
        VBX_CUDA(c, cudaMemsetAsync(reinterpret_cast<char*>(c->tab.tsdf) + (size_t)v * tb, 0, tb, s));
        VBX_CUDA(c, cudaMemcpyAsync(c->tab.slot_updated + v, &no_tsdf, 1, cudaMemcpyHostToDevice, s));
        c->maybe_esdf_only = true;
      } else {
        drop.push_back(v);
      }
    }
  }
  VBX_CUDA(c, cudaStreamSynchronize(s));  // (no_tsdf lives on this stack frame)
  if (drop.empty()) return VBX_OK;
  victims.swap(drop);
  // swap-remove in the pool (highest victim first), then rebuild the hash from slot_key
  uint32_t n = c->n_blocks;
  for (auto it = victims.rbegin(); it != victims.rend(); ++it) {
    const uint32_t v = (uint32_t)*it, last = n - 1;
    if (v != last) {
      VBX_CUDA(c, cudaMemcpyAsync(reinterpret_cast<char*>(c->tab.tsdf) + (size_t)v * tb,
                                  reinterpret_cast<char*>(c->tab.tsdf) + (size_t)last * tb, tb, cudaMemcpyDeviceToDevice, s));
      if (c->has_esdf) {
        VBX_CUDA(c, cudaMemcpyAsync(reinterpret_cast<char*>(c->tab.esdf) + (size_t)v * eb,
                                    reinterpret_cast<char*>(c->tab.esdf) + (size_t)last * eb, eb, cudaMemcpyDeviceToDevice, s));
      }
      VBX_CUDA(c, cudaMemcpyAsync(c->tab.slot_key + v, c->tab.slot_key + last, sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
      VBX_CUDA(c, cudaMemcpyAsync(c->tab.slot_updated + v, c->tab.slot_updated + last, 1, cudaMemcpyDeviceToDevice, s));
      VBX_CUDA(c, cudaMemcpyAsync(c->tab.slot_esdf_updated + v, c->tab.slot_esdf_updated + last, 1, cudaMemcpyDeviceToDevice, s));
      VBX_CUDA(c, cudaMemcpyAsync(c->tab.slot_has_esdf + v, c->tab.slot_has_esdf + last, 1, cudaMemcpyDeviceToDevice, s));
    }
    // a freed slot must read as a freshly constructed block for its next owner
    VBX_CUDA(c, cudaMemsetAsync(reinterpret_cast<char*>(c->tab.tsdf) + (size_t)last * tb, 0, tb, s));
    if (c->has_esdf) VBX_CUDA(c, cudaMemsetAsync(reinterpret_cast<char*>(c->tab.esdf) + (size_t)last * eb, 0, eb, s));
    VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_updated + last, 0, 1, s));
    VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_esdf_updated + last, 0, 1, s));
    VBX_CUDA(c, cudaMemsetAsync(c->tab.slot_has_esdf + last, 0, 1, s));
    --n;
  }
  if (int rc = set_n_blocks(c, n)) return rc;
  if (int rc = rebuild_hash(c)) return rc;
  c->host_slot_key.clear();
  c->host_key2slot.clear();
  return refresh_host_mirror(c);
}

// ------------------------------------------------------------------ incremental host mirror
// SURVEY.md section 8(f) N1: what every host consumer of the Layer does after a scan --
// getAllUpdatedBlocks(bit) (core/layer.h:194-203), read the blocks, updated().reset(bit)
// (e.g. mesh_integrator.h:168-183, esdf_integrator.cc:113-121) -- as ONE call: the dirty blocks
// are gathered into a contiguous staging buffer by a kernel, leave the device in one copy into
// page-locked memory, and their bits are cleared on the device.
__global__ void k_gather_blocks(const uint4* __restrict__ pool, const uint32_t* __restrict__ slots, uint32_t m,
                                uint32_t vec_per_block, uint4* __restrict__ out, uint8_t* __restrict__ flags,
                                uint8_t clear_mask) {
  // one CTA per (block, 1/8 of its payload): 16-byte loads, fully coalesced both ways
  const uint32_t b = blockIdx.x >> 3, part = blockIdx.x & 7u;
  if (b >= m) return;
  const uint32_t slot = slots[b];
  const uint32_t per = (vec_per_block + 7u) / 8u;
  const uint32_t lo = part * per, hi = min(vec_per_block, lo + per);
  const uint4* src = pool + (size_t)slot * vec_per_block;
  uint4* dst = out + (size_t)b * vec_per_block;
  for (uint32_t i = lo + threadIdx.x; i < hi; i += blockDim.x) dst[i] = __ldcs(src + i);
  if (part == 0 && threadIdx.x == 0 && clear_mask) flags[slot] &= (uint8_t)~clear_mask;
}

int mirror_updated(vbx_ctx* c, int layer, int updated_mask, int clear_mask, int32_t* idx3, void* voxels,
                   uint8_t* updated_bits, uint64_t cap, uint64_t* n, int serialized) {
  cudaStream_t s = c->stream_main;
  *n = 0;
  if (c->n_blocks == 0) return VBX_OK;
  if (int rc = refresh_host_mirror(c)) return rc;
  // the flags are one byte per block: a single small copy decides what is dirty
  std::vector<uint8_t> upd(c->n_blocks), has(c->n_blocks, 1);
  uint8_t* flags = (layer == VBX_LAYER_TSDF) ? c->tab.slot_updated : c->tab.slot_esdf_updated;
  VBX_CUDA(c, cudaMemcpyAsync(upd.data(), flags, c->n_blocks, cudaMemcpyDeviceToHost, s));
  if (layer == VBX_LAYER_ESDF) {
    VBX_CUDA(c, cudaMemcpyAsync(has.data(), c->tab.slot_has_esdf, c->n_blocks, cudaMemcpyDeviceToHost, s));
  }
  VBX_CUDA(c, cudaStreamSynchronize(s));
  for (uint32_t sl = 0; sl < c->n_blocks; ++sl) {
    if (layer == VBX_LAYER_TSDF && (upd[sl] & kSlotNoTsdf)) has[sl] = 0;  // an ESDF-only slot
    upd[sl] &= 0x7f;  // (bit 3, the mirror mark, may be selected by updated_mask; it is not reported)
  }
  struct Item {
    int x, y, z;
    uint32_t slot;
  };
  std::vector<Item> items;
  for (uint32_t sl = 0; sl < c->n_blocks; ++sl) {
    if (!has[sl]) continue;
    if (updated_mask && !(upd[sl] & updated_mask)) continue;
    Item it;
    unpack3(c->host_slot_key[sl], &it.x, &it.y, &it.z);
    it.slot = sl;
    items.push_back(it);
  }
  *n = items.size();
  if (items.empty() || items.size() > cap) return VBX_OK;  // (too small a buffer: the caller grows it and retries)
  std::sort(items.begin(), items.end(), [](const Item& a, const Item& b) {
    if (a.x != b.x) return a.x < b.x;
    if (a.y != b.y) return a.y < b.y;
    return a.z < b.z;
  });
  const size_t m = items.size();
  const size_t raw_bytes = ((layer == VBX_LAYER_TSDF) ? sizeof(TsdfVoxel) : sizeof(EsdfVoxel)) * c->vox_per_block;
  const size_t bbytes = payload_bytes(c, layer, serialized);
  if (raw_bytes % 16 != 0) return fail(c, VBX_E_STATE, "block payload is not a multiple of 16 bytes");
  if (int rc = ensure_staging(c, m * bbytes, m)) return rc;
  std::vector<uint32_t> slots(m);
  for (size_t i = 0; i < m; ++i) {
    slots[i] = items[i].slot;
    if (idx3) {
      idx3[3 * i] = items[i].x;
      idx3[3 * i + 1] = items[i].y;
      idx3[3 * i + 2] = items[i].z;
    }
    if (updated_bits) updated_bits[i] = upd[items[i].slot] & 0x07;
  }
  VBX_CUDA(c, cudaMemcpyAsync(c->mirror_slots, slots.data(), m * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  const char* pool = (layer == VBX_LAYER_TSDF) ? reinterpret_cast<const char*>(c->tab.tsdf)
                                               : reinterpret_cast<const char*>(c->tab.esdf);
  if (serialized) {
    const uint32_t tpv = (layer == VBX_LAYER_TSDF) ? 3u : 1u;
    const dim3 grid(grid_for((uint64_t)tpv * c->vox_per_block, 256), (unsigned int)m);
    k_serialize_blocks<<<grid, 256, 0, s>>>(layer, reinterpret_cast<const uint32_t*>(pool), c->mirror_slots, (uint32_t)m,
                                            (uint32_t)c->vox_per_block, static_cast<uint32_t*>(c->mirror_dev), flags,
                                            (uint8_t)(clear_mask & 0x7f));
  } else {
    k_gather_blocks<<<(unsigned int)(m * 8), 256, 0, s>>>(reinterpret_cast<const uint4*>(pool), c->mirror_slots,
                                                           (uint32_t)m, (uint32_t)(raw_bytes / 16),
                                                           reinterpret_cast<uint4*>(c->mirror_dev), flags,
                                                           (uint8_t)(clear_mask & 0x7f));
  }
  // straight into the caller's buffer when it is page-locked (vbx_host_alloc / cudaHostRegister),
  // otherwise through the engine's page-locked staging buffer
  cudaPointerAttributes attr;
  const bool direct = voxels && cudaPointerGetAttributes(&attr, voxels) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();  // (an unregistered pointer may leave a sticky-free error code behind)
  void* dst = direct ? voxels : c->mirror_host;
  VBX_CUDA(c, cudaMemcpyAsync(dst, c->mirror_dev, m * bbytes, cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  if (!direct && voxels) std::memcpy(voxels, c->mirror_host, m * bbytes);
  return VBX_OK;
}

}  // namespace vbx
