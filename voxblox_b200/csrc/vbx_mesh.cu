// Marching-cubes meshing of the device TSDF map: MeshIntegrator<TsdfVoxel>::generateMesh
// (voxblox/include/voxblox/mesh/mesh_integrator.h:132-160) with extractBlockMesh (:179-236),
// extractMeshInsideBlock / extractMeshOnBorder (:262-366), MarchingCubes::meshCube
// (mesh/marching_cubes.h:74-164) and updateMeshColor (mesh_integrator.h:368-388).
// SURVEY.md section 8(f) N3: the other per-scan consumer of updated TSDF blocks.
//
// The reference meshes one block per thread task and appends the triangles of its cubes in a
// fixed order (inner cubes x-major, then the max-X, max-Y and max-Z border planes).  Here one CTA
// meshes one block:
//   k_mesh_count  stages the block's (vps+1)^3 corner distances (own voxels + the seven
//                 neighbouring blocks' faces / edges / corner) in shared memory -- one coalesced read
//                 of the 48 KiB slab -- classifies every cube, and scans the per-cube vertex counts
//                 IN THE REFERENCE'S CUBE ORDER, so that every cube knows where its vertices go
//   (host)        prefix sum over the per-block totals (a few hundred numbers)
//   k_mesh_emit   stages the same corner array again and writes vertices, face normals and
//                 vertex colours at those offsets
// The output of a block is therefore the reference's Mesh for that block element for element
// (vertices, normals, colours; Mesh::indices is 0..n-1 by construction, marching_cubes.h:97-99),
// with the reference's float arithmetic spelled out operation by operation (vbx_math.cuh).
// Algorithmic bytes per meshed block: 12*vps^3 read (+ faces of the neighbours) + 28 B per vertex written.
#include <algorithm>
#include <cstring>
#include <vector>

#include "vbx_engine.h"
#include "vbx_hash.cuh"
#include "vbx_mc_tables.h"

namespace vbx {

__constant__ unsigned long long kMcTri[256] = {VBX_MC_TRIANGLE_WORDS};
__constant__ int8_t kMcPair[12][2] = {VBX_MC_EDGE_PAIRS};
// cube_index_offsets_, mesh_integrator.h:94-95 / :121-123
__constant__ int8_t kCubeOff[8][3] = {{0, 0, 0}, {1, 0, 0}, {1, 1, 0}, {0, 1, 0}, {0, 0, 1}, {1, 0, 1}, {1, 1, 1}, {0, 1, 1}};

struct MeshParams {
  int L, vps;
  float voxel_size, voxel_size_inv, block_size, block_size_inv;
  float min_weight;
  int use_color;
};

constexpr int kMeshThreads = 1024;  // 4 cubes per thread at vps 16: the per-cube work is a latency chain, so more threads per block

// position of cube (x, y, z) in the order extractBlockMesh visits the cubes (mesh_integrator.h:186-235),
// and its inverse
__device__ __forceinline__ void cube_of_order(int vps, uint32_t o, int* x, int* y, int* z) {
  const uint32_t m = (uint32_t)vps - 1u, v = (uint32_t)vps;
  const uint32_t n_in = m * m * m, n_x = v * v, n_y = v * m;
  if (o < n_in) {  // x outer, y, z inner
    *x = (int)(o / (m * m));
    *y = (int)((o / m) % m);
    *z = (int)(o % m);
  } else if (o < n_in + n_x) {  // max X plane: z outer, y inner
    const uint32_t r = o - n_in;
    *x = (int)m;
    *z = (int)(r / v);
    *y = (int)(r % v);
  } else if (o < n_in + n_x + n_y) {  // max Y plane: z outer, x inner (x < vps - 1)
    const uint32_t r = o - n_in - n_x;
    *y = (int)m;
    *z = (int)(r / m);
    *x = (int)(r % m);
  } else {  // max Z plane: y outer, x inner (both < vps - 1)
    const uint32_t r = o - n_in - n_x - n_y;
    *z = (int)m;
    *y = (int)(r / m);
    *x = (int)(r % m);
  }
}

// pool slot of the TSDF block with this index, or -1 (Layer::hasBlock, mesh_integrator.h:340)
__device__ __forceinline__ int32_t tsdf_slot_of(const Tables& tab, int bx, int by, int bz) {
  const int lim = kCoordBias - 1;
  if (bx < -lim || bx > lim || by < -lim || by > lim || bz < -lim || bz > lim) return -1;
  const uint32_t hp = find_block(tab, pack3(bx, by, bz));
  if (hp == 0xffffffffu) return -1;
  const int32_t slot = tab.hslot[hp];
  if (slot < 0 || (tab.slot_updated[slot] & kSlotNoTsdf)) return -1;
  return slot;
}

// The (vps+1)^3 corner distances of one block in shared memory; NaN marks a corner whose voxel is
// missing or not observed (utils::getSdfIfValid: weight <= min_weight, utils/meshing_utils.h:16-24).
__device__ __forceinline__ void stage_corners(const MeshParams& P, const Tables& tab, uint32_t slot, float* s_sdf,
                                              int32_t* s_nslot) {
  const int n1 = P.vps + 1, mask = P.vps - 1;
  if (threadIdx.x < 8) {
    int bx, by, bz;
    unpack3(tab.slot_key[slot], &bx, &by, &bz);
    const int k = threadIdx.x;
    s_nslot[k] = k == 0 ? (int32_t)slot : tsdf_slot_of(tab, bx + (k & 1), by + ((k >> 1) & 1), bz + ((k >> 2) & 1));
  }
  __syncthreads();
  const uint32_t total = (uint32_t)n1 * n1 * n1;
  const size_t vpb = (size_t)1 << (3 * P.L);
  for (uint32_t i = threadIdx.x; i < total; i += blockDim.x) {
    const int x = (int)(i % n1), y = (int)((i / n1) % n1), z = (int)(i / (n1 * n1));
    const int k = (x == P.vps ? 1 : 0) | (y == P.vps ? 2 : 0) | (z == P.vps ? 4 : 0);
    const int32_t ns = s_nslot[k];
    float v = __int_as_float(0x7fc00000);
    if (ns >= 0) {
      const uint32_t lin = (uint32_t)(x & mask) | ((uint32_t)(y & mask) << P.L) | ((uint32_t)(z & mask) << (2 * P.L));
      const TsdfVoxel* tv = tab.tsdf + (size_t)ns * vpb + lin;  // (12-byte records: two scalar loads)
      const float w = tv->weight;
      if (w > P.min_weight) v = tv->distance;
    }
    s_sdf[i] = v;
  }
  __syncthreads();
}

// the eight corner distances of cube (x, y, z); false if one of them is not observed
__device__ __forceinline__ bool cube_sdf(const MeshParams& P, const float* s_sdf, int x, int y, int z, float sdf[8]) {
  const int n1 = P.vps + 1;
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sdf[i] = s_sdf[((z + kCubeOff[i][2]) * n1 + (y + kCubeOff[i][1])) * n1 + (x + kCubeOff[i][0])];
    ok = ok && (sdf[i] == sdf[i]);
  }
  return ok;
}

// calculateVertexConfiguration, marching_cubes.h:115-125
__device__ __forceinline__ int cube_case(const float sdf[8]) {
  int index = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) index |= (sdf[i] < 0.0f) ? (1 << i) : 0;
  return index;
}

__device__ __forceinline__ uint32_t case_vertices(int index) {
  const unsigned long long row = kMcTri[index];
  uint32_t n = 0;
  while (n < 15u && ((row >> (4 * n)) & 0xFull) != 0xFull) n += 3u;
  return n;
}

__global__ void __launch_bounds__(kMeshThreads)
k_mesh_count(MeshParams P, Tables tab, const uint32_t* __restrict__ slots, uint16_t* __restrict__ cube_off,
             uint32_t* __restrict__ block_nv) {
  extern __shared__ float s_sdf[];
  __shared__ int32_t s_nslot[8];
  __shared__ uint32_t warp_sums[kMeshThreads / 32];
  const uint32_t b = blockIdx.x;
  const uint32_t slot = slots[b];
  stage_corners(P, tab, slot, s_sdf, s_nslot);
  const uint32_t vpb = 1u << (3 * P.L);
  const uint32_t ipt = (vpb + kMeshThreads - 1) / kMeshThreads;  // consecutive order positions per thread
  const uint32_t o0 = threadIdx.x * ipt, o1 = min(vpb, o0 + ipt);
  // pass 1: this thread's vertex count
  uint32_t mine = 0;
  for (uint32_t o = o0; o < o1; ++o) {
    int x, y, z;
    cube_of_order(P.vps, o, &x, &y, &z);
    float sdf[8];
    if (cube_sdf(P, s_sdf, x, y, z, sdf)) mine += case_vertices(cube_case(sdf));
  }
  // exclusive scan of the thread totals over the CTA
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  uint32_t base = 0, total = 0;
#pragma unroll
  for (int w = 0; w < kMeshThreads / 32; ++w) {
    if (w < warp) base += warp_sums[w];
    total += warp_sums[w];
  }
  uint32_t at = base + inc - mine;
  // pass 2: where each cube's vertices start inside the block's mesh
  for (uint32_t o = o0; o < o1; ++o) {
    int x, y, z;
    cube_of_order(P.vps, o, &x, &y, &z);
    float sdf[8];
    uint32_t nv = 0;
    if (cube_sdf(P, s_sdf, x, y, z, sdf)) nv = case_vertices(cube_case(sdf));
    cube_off[(size_t)b * vpb + o] = (uint16_t)at;
    at += nv;
  }
  if (threadIdx.x == 0) block_nv[b] = total;
}

// MarchingCubes::interpolateVertex, marching_cubes.h:150-164
__device__ __forceinline__ F3 mc_interpolate(F3 v1, F3 v2, float sdf1, float sdf2) {
  const float diff = fsub(sdf1, sdf2);
  if (fabsf(diff) >= 1e-6f) {
    const float t = fdiv(sdf1, diff);
    return f3(fadd(v1.x, fmul(t, fsub(v2.x, v1.x))), fadd(v1.y, fmul(t, fsub(v2.y, v1.y))),
              fadd(v1.z, fmul(t, fsub(v2.z, v1.z))));
  }
  return f3(fmul(0.5f, fadd(v1.x, v2.x)), fmul(0.5f, fadd(v1.y, v2.y)), fmul(0.5f, fadd(v1.z, v2.z)));
}

// updateMeshColor for one vertex, mesh_integrator.h:374-387
__device__ __forceinline__ uint32_t vertex_color(const MeshParams& P, const Tables& tab, uint32_t slot, F3 origin, F3 v) {
  const size_t vpb = (size_t)1 << (3 * P.L);
  const I3 vi = grid_index(sub3(v, origin), P.voxel_size_inv);  // computeVoxelIndexFromCoordinates, core/block.h:65-70
  const TsdfVoxel* vox;
  if (vi.x >= 0 && vi.x < P.vps && vi.y >= 0 && vi.y < P.vps && vi.z >= 0 && vi.z < P.vps) {
    vox = tab.tsdf + (size_t)slot * vpb + ((uint32_t)vi.x | ((uint32_t)vi.y << P.L) | ((uint32_t)vi.z << (2 * P.L)));
  } else {
    // getBlockPtrByCoordinates(vertex) (core/layer.h:105-108,128-131), then getVoxelByCoordinates ->
    // computeTruncatedVoxelIndexFromCoordinates (core/block_inl.h:29-40)
    const I3 nb = grid_index(v, P.block_size_inv);
    const int32_t ns = tsdf_slot_of(tab, nb.x, nb.y, nb.z);
    if (ns < 0) return 0u;  // (the reference dereferences a null block pointer here)
    const F3 no = f3(fmul((float)nb.x, P.block_size), fmul((float)nb.y, P.block_size), fmul((float)nb.z, P.block_size));
    const I3 t = grid_index(sub3(v, no), P.voxel_size_inv);
    const int mx = P.vps - 1;
    const uint32_t tx = (uint32_t)max(min(t.x, mx), 0), ty = (uint32_t)max(min(t.y, mx), 0), tz = (uint32_t)max(min(t.z, mx), 0);
    vox = tab.tsdf + (size_t)ns * vpb + (tx | (ty << P.L) | (tz << (2 * P.L)));
  }
  return vox->weight > P.min_weight ? vox->color : 0u;  // utils::getColorIfValid, meshing_utils.h:45-54; Color() = 0
}

__global__ void __launch_bounds__(kMeshThreads)
k_mesh_emit(MeshParams P, Tables tab, const uint32_t* __restrict__ slots, const uint16_t* __restrict__ cube_off,
            const unsigned long long* __restrict__ first_vertex, float* __restrict__ vertices, float* __restrict__ normals,
            uint32_t* __restrict__ colors) {
  extern __shared__ float s_sdf[];
  __shared__ int32_t s_nslot[8];
  const uint32_t b = blockIdx.x;
  const uint32_t slot = slots[b];
  const unsigned long long first = first_vertex[b];
  if (first_vertex[b + 1] == first) return;  // nothing to write for this block
  stage_corners(P, tab, slot, s_sdf, s_nslot);
  int bx, by, bz;
  unpack3(tab.slot_key[slot], &bx, &by, &bz);
  // Block::origin_ = float(block index) * block_size (core/common.h:196-201)
  const F3 origin = f3(fmul((float)bx, P.block_size), fmul((float)by, P.block_size), fmul((float)bz, P.block_size));
  const uint32_t vpb = 1u << (3 * P.L);
  const uint32_t ipt = (vpb + kMeshThreads - 1) / kMeshThreads;
  const uint32_t o0 = threadIdx.x * ipt, o1 = min(vpb, o0 + ipt);
  for (uint32_t o = o0; o < o1; ++o) {
    int x, y, z;
    cube_of_order(P.vps, o, &x, &y, &z);
    float sdf[8];
    if (!cube_sdf(P, s_sdf, x, y, z, sdf)) continue;
    const int index = cube_case(sdf);
    const unsigned long long row = kMcTri[index];
    if ((row & 0xFull) == 0xFull) continue;  // no surface in this cube (incl. index == 0, marching_cubes.h:82-84)
    // coords = block.computeCoordinatesFromVoxelIndex(voxel) (core/block.h:90-92); corners = coords + offset * voxel_size
    const F3 coords = f3(fadd(origin.x, center_coord(x, P.voxel_size)), fadd(origin.y, center_coord(y, P.voxel_size)),
                         fadd(origin.z, center_coord(z, P.voxel_size)));
    unsigned long long at = first + cube_off[(size_t)b * vpb + o];
    for (int col = 0; col < 15 && ((row >> (4 * col)) & 0xFull) != 0xFull; col += 3) {
      F3 p[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        // vertices are appended as table entries col+2, col+1, col (marching_cubes.h:91-96)
        const int e = (int)((row >> (4 * (col + 2 - k))) & 0xFull);
        const int a = kMcPair[e][0], c = kMcPair[e][1];
        const F3 ca = f3(fadd(coords.x, fmul((float)kCubeOff[a][0], P.voxel_size)), fadd(coords.y, fmul((float)kCubeOff[a][1], P.voxel_size)),
                         fadd(coords.z, fmul((float)kCubeOff[a][2], P.voxel_size)));
        const F3 cc = f3(fadd(coords.x, fmul((float)kCubeOff[c][0], P.voxel_size)), fadd(coords.y, fmul((float)kCubeOff[c][1], P.voxel_size)),
                         fadd(coords.z, fmul((float)kCubeOff[c][2], P.voxel_size)));
        p[k] = mc_interpolate(ca, cc, sdf[a], sdf[c]);
      }
      const F3 n = unit3(cross3(sub3(p[1], p[0]), sub3(p[2], p[0])));  // marching_cubes.h:100-108
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        float* vo = vertices + 3 * (at + k);
        float* no = normals + 3 * (at + k);
        vo[0] = p[k].x;
        vo[1] = p[k].y;
        vo[2] = p[k].z;
        no[0] = n.x;
        no[1] = n.y;
        no[2] = n.z;
        if (P.use_color) colors[at + k] = vertex_color(P, tab, slot, origin, p[k]);
      }
      at += 3;
    }
  }
}

__global__ void k_mesh_clear_flag(Tables tab, const uint32_t* __restrict__ slots, uint32_t nb) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nb) tab.slot_updated[slots[i]] &= (uint8_t)~VBX_UPDATED_MESH;  // block->updated().reset(Update::kMesh), :171-175
}

static inline unsigned int grid_for(uint64_t n, int block) { return (unsigned int)((n + block - 1) / block); }

static void mesh_free(vbx_ctx* c) {
  void* ptrs[] = {c->mesh_slots, c->mesh_cube_off, c->mesh_block_nv, c->mesh_first, c->mesh_vertices, c->mesh_normals,
                  c->mesh_colors};
  for (void* p : ptrs) {
    if (p) cudaFree(p);
  }
  c->mesh_slots = c->mesh_block_nv = c->mesh_colors = nullptr;
  c->mesh_cube_off = nullptr;
  c->mesh_first = nullptr;
  c->mesh_vertices = c->mesh_normals = nullptr;
  c->mesh_cap_blocks = c->mesh_cap_vertices = 0;
}

void mesh_destroy(vbx_ctx* c) { mesh_free(c); }

// MeshIntegrator::generateMesh(only_mesh_updated_blocks, clear_updated_flag), mesh_integrator.h:132-160
int mesh_generate(vbx_ctx* c, const vbx_mesh_config* cfg, int only_updated, int clear_flag, uint64_t* n_blocks_out,
                  uint64_t* n_vertices_out) {
  cudaStream_t s = c->stream_main;
  c->mesh_idx.clear();
  c->mesh_first_host.assign(1, 0);
  c->mesh_use_color = cfg->use_color != 0;
  if (n_blocks_out) *n_blocks_out = 0;
  if (n_vertices_out) *n_vertices_out = 0;
  if (c->n_blocks == 0) return VBX_OK;
  if (int rc = refresh_host_mirror(c)) return rc;
  // getAllUpdatedBlocks(Update::kMesh) / getAllAllocatedBlocks of the TSDF layer, sorted by index
  std::vector<uint8_t> upd(c->n_blocks);
  VBX_CUDA(c, cudaMemcpyAsync(upd.data(), c->tab.slot_updated, c->n_blocks, cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  struct Item {
    int x, y, z;
    uint32_t slot;
  };
  std::vector<Item> items;
  for (uint32_t sl = 0; sl < c->n_blocks; ++sl) {
    if (upd[sl] & kSlotNoTsdf) continue;
    if (only_updated && !(upd[sl] & VBX_UPDATED_MESH)) continue;
    Item it;
    unpack3(c->host_slot_key[sl], &it.x, &it.y, &it.z);
    it.slot = sl;
    items.push_back(it);
  }
  if (items.empty()) return VBX_OK;
  std::sort(items.begin(), items.end(), [](const Item& a, const Item& b) {
    if (a.x != b.x) return a.x < b.x;
    if (a.y != b.y) return a.y < b.y;
    return a.z < b.z;
  });
  const uint32_t nb = (uint32_t)items.size();
  if (nb > c->mesh_cap_blocks) {
    const uint64_t want = std::max<uint64_t>(2ull * nb, 256);
    void* old[] = {c->mesh_slots, c->mesh_cube_off, c->mesh_block_nv, c->mesh_first};
    for (void* p : old) {
      if (p) cudaFree(p);
    }
    c->mesh_slots = c->mesh_block_nv = nullptr;
    c->mesh_cube_off = nullptr;
    c->mesh_first = nullptr;
    c->mesh_cap_blocks = 0;
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mesh_slots), want * sizeof(uint32_t)));
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mesh_cube_off), want * c->vox_per_block * sizeof(uint16_t)));
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mesh_block_nv), want * sizeof(uint32_t)));
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mesh_first), (want + 1) * sizeof(unsigned long long)));
    c->mesh_cap_blocks = want;
  }
  std::vector<uint32_t> slots(nb);
  c->mesh_idx.resize(3 * (size_t)nb);
  for (uint32_t i = 0; i < nb; ++i) {
    slots[i] = items[i].slot;
    c->mesh_idx[3 * i] = items[i].x;
    c->mesh_idx[3 * i + 1] = items[i].y;
    c->mesh_idx[3 * i + 2] = items[i].z;
  }
  MeshParams P;
  P.L = c->L;
  P.vps = c->vps;
  P.voxel_size = c->voxel_size;
  P.voxel_size_inv = c->voxel_size_inv;
  P.block_size = c->voxel_size * (float)c->vps;        // Layer: block_size_ = voxel_size_ * voxels_per_side_, core/layer.h:41
  P.block_size_inv = (float)(1.0 / (double)P.block_size);  // core/layer.h:43
  P.min_weight = cfg->min_weight;
  P.use_color = cfg->use_color ? 1 : 0;
  const int n1 = c->vps + 1;
  const size_t smem = (size_t)n1 * n1 * n1 * sizeof(float);
  if (smem > 48 * 1024) {
    if (smem > 200 * 1024) return fail(c, VBX_E_CAPACITY, "voxels_per_side too large for the mesher's shared-memory tile");
    VBX_CUDA(c, cudaFuncSetAttribute(k_mesh_count, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VBX_CUDA(c, cudaFuncSetAttribute(k_mesh_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  if ((uint64_t)15 * c->vox_per_block > 0xffffull) return fail(c, VBX_E_CAPACITY, "voxels_per_side too large for 16-bit cube offsets");
  VBX_CUDA(c, cudaEventRecord(c->ev0, s));
  VBX_CUDA(c, cudaMemcpyAsync(c->mesh_slots, slots.data(), nb * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  k_mesh_count<<<nb, kMeshThreads, smem, s>>>(P, c->tab, c->mesh_slots, c->mesh_cube_off, c->mesh_block_nv);
  std::vector<uint32_t> nv(nb);
  VBX_CUDA(c, cudaMemcpyAsync(nv.data(), c->mesh_block_nv, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  c->mesh_first_host.assign((size_t)nb + 1, 0);
  for (uint32_t i = 0; i < nb; ++i) c->mesh_first_host[i + 1] = c->mesh_first_host[i] + nv[i];
  const uint64_t total = c->mesh_first_host[nb];
  if (total > c->mesh_cap_vertices) {
    const uint64_t want = std::max<uint64_t>(total + total / 2, 1u << 16);
    void* old[] = {c->mesh_vertices, c->mesh_normals, c->mesh_colors};
    for (void* p : old) {
      if (p) cudaFree(p);
    }
    c->mesh_vertices = c->mesh_normals = nullptr;
    c->mesh_colors = nullptr;
    c->mesh_cap_vertices = 0;
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mesh_vertices), want * 3 * sizeof(float)));
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mesh_normals), want * 3 * sizeof(float)));
    VBX_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->mesh_colors), want * sizeof(uint32_t)));
    c->mesh_cap_vertices = want;
  }
  uint64_t launches = 1;
  if (total > 0) {
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "first-vertex table");
    VBX_CUDA(c, cudaMemcpyAsync(c->mesh_first, c->mesh_first_host.data(), ((size_t)nb + 1) * sizeof(uint64_t),
                                cudaMemcpyHostToDevice, s));
    k_mesh_emit<<<nb, kMeshThreads, smem, s>>>(P, c->tab, c->mesh_slots, c->mesh_cube_off, c->mesh_first, c->mesh_vertices,
                                               c->mesh_normals, c->mesh_colors);
    launches += 1;
  }
  if (clear_flag) {
    k_mesh_clear_flag<<<grid_for(nb, 256), 256, 0, s>>>(c->tab, c->mesh_slots, nb);
    launches += 1;
  }
  VBX_CUDA(c, cudaEventRecord(c->ev1, s));
  VBX_CUDA(c, cudaStreamSynchronize(s));
  VBX_CUDA(c, cudaGetLastError());
  VBX_CUDA(c, cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
  c->launches += launches;
  c->mesh_launches = launches;
  if (n_blocks_out) *n_blocks_out = nb;
  if (n_vertices_out) *n_vertices_out = total;
  return VBX_OK;
}

// the result of the last mesh_generate, block by block in index order
int mesh_download(vbx_ctx* c, int32_t* idx3, uint64_t* first_vertex, float* vertices, float* normals, uint8_t* colors) {
  cudaStream_t s = c->stream_main;
  const size_t nb = c->mesh_idx.size() / 3;
  if (idx3 && nb) std::memcpy(idx3, c->mesh_idx.data(), nb * 3 * sizeof(int32_t));
  if (first_vertex) std::memcpy(first_vertex, c->mesh_first_host.data(), c->mesh_first_host.size() * sizeof(uint64_t));
  const uint64_t total = c->mesh_first_host.back();
  if (total == 0) return VBX_OK;
  if (vertices) VBX_CUDA(c, cudaMemcpyAsync(vertices, c->mesh_vertices, total * 3 * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (normals) VBX_CUDA(c, cudaMemcpyAsync(normals, c->mesh_normals, total * 3 * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (colors) {
    if (!c->mesh_use_color) return fail(c, VBX_E_STATE, "the last mesh was generated without colours");
    VBX_CUDA(c, cudaMemcpyAsync(colors, c->mesh_colors, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  }
  VBX_CUDA(c, cudaStreamSynchronize(s));
  return VBX_OK;
}

}  // namespace vbx
