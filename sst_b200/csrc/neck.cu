// Voxel2PointScatterNeck.forward (mmdet3d/models/necks/voxel2point_neck.py:28-62; SURVEY 8f next-2): voxel features back to
// the points (FSD's step between the SST/sparse backbone and the point-wise heads).
//   pts_feats = voxel_feats[voxel2point_inds];  pts_mask = ~(pts_feats == padding).all(1)      (dropped voxels are padded rows)
//   results   = [pts_feats[mask] || points[mask,:3] - ((coors[mask,[3,2,1]] + 0.5) * voxel_size + pc_min) (/ (voxel_size/2))]
// The reference materialises the [N,C] gather, the mask, three filtered copies and a concat; here: one warp-per-point mask
// pass, a look-back scan over the keep flags (order-preserving compaction) and one warp-per-point write pass.
#include <stdarg.h>
#include "common.cuh"

// TI: index type of inds / coors (int64 from the modules, int32 from the sync-free engine).  M_dev != nullptr: the voxel count is
// read from the device and an index outside [0, M) marks a point that is not kept (no voxel: rows past the last frame) instead
// of an error.
template <typename TI>
__global__ void __launch_bounds__(256) v2p_mask_kernel(const float* __restrict__ voxel_feats, int C, const TI* __restrict__ inds, int N,
                                                       int M, const int32_t* __restrict__ M_dev, float padding, uint32_t* __restrict__ keep,
                                                       uint8_t* __restrict__ mask_out, int32_t* __restrict__ err) {
  pdl_wait();
  pdl_launch();
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= N) return;
  if (M_dev) M = *M_dev;
  const long long v = (long long)inds[i];
  if (v < 0 || v >= M) {
    if (lane == 0) {
      if (!M_dev) *err = 1;
      keep[i] = 0;
      mask_out[i] = 0;
    }
    return;
  }
  const float* row = voxel_feats + (size_t)v * C;
  bool all_pad = true;
  for (int c = lane; c < C; c += 32) all_pad &= (row[c] == padding);
  all_pad = __all_sync(0xffffffffu, all_pad);
  if (lane == 0) {
    keep[i] = all_pad ? 0u : 1u;
    mask_out[i] = all_pad ? 0 : 1;
  }
}

template <typename TI>
__global__ void __launch_bounds__(256) v2p_write_kernel(const float* __restrict__ points, int Cp, const TI* __restrict__ coors,
                                                        const float* __restrict__ voxel_feats, int C, const TI* __restrict__ inds, int N,
                                                        const uint32_t* __restrict__ keep, const uint32_t* __restrict__ pos, float vx, float vy,
                                                        float vz, float x0, float y0, float z0, int with_xyz, int normalize,
                                                        float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= N || !keep[i]) return;
  const int Co = C + (with_xyz ? 3 : 0);
  const float* row = voxel_feats + (size_t)(long long)inds[i] * C;
  float* o = out + (size_t)pos[i] * Co;
  for (int c = lane; c < C; c += 32) o[c] = row[c];
  if (with_xyz && lane < 3) {
    // x y z order: coors are (b, z, y, x); two roundings for (c + 0.5) * vs + min like the torch expression
    const float vs = lane == 0 ? vx : (lane == 1 ? vy : vz);
    const float mn = lane == 0 ? x0 : (lane == 1 ? y0 : z0);
    const float cc = (float)coors[(size_t)i * 4 + (3 - lane)];
    const float center = __fadd_rn(__fmul_rn(__fadd_rn(cc, 0.5f), vs), mn);
    float l = points[(size_t)i * Cp + lane] - center;
    if (normalize) l = __fdiv_rn(l, __fdiv_rn(vs, 2.0f));
    o[C + lane] = l;
  }
}

extern "C" int sstb200_voxel2point(sstb200_ctx* c, const float* points, int Cp, const int64_t* pts_coors, const float* voxel_feats, int M,
                                   int C, const int64_t* voxel2point_inds, int N, float padding, const float voxel_size[3],
                                   const float pc_min[3], int with_xyz, int normalize_local_xyz, float* out, uint8_t* mask_out,
                                   int32_t* num_out_dev, int32_t* num_out_host) {
  CHECK_ARG(c, c && N >= 0 && M >= 0 && C >= 1 && Cp >= 3 && num_out_dev);
  if (N == 0) {
    CUDA_TRY(c, cudaMemsetAsync(num_out_dev, 0, 4, c->stream));
    if (num_out_host) *num_out_host = 0;
    return SSTB_OK;
  }
  CHECK_ARG(c, points && pts_coors && voxel_feats && voxel2point_inds && out && mask_out && voxel_size && pc_min);
  arena_reset(c);
  int rc = arena_reserve(c, 2 * al256((size_t)N * 4 + 64) + scan_temps_bytes(N) + 4096);
  if (rc) return rc;
  uint32_t* keep = arena_alloc<uint32_t>(c, (size_t)N + 2);
  uint32_t* pos = arena_alloc<uint32_t>(c, (size_t)N + 2);
  uint8_t* z = arena_alloc<uint8_t>(c, scan_temps_bytes(N));
  if (!keep || !pos || !z) return sstb_fail(c, SSTB_ERR_WORKSPACE, "voxel2point: arena");
  ScanTemps st{(uint32_t*)z, (unsigned long long*)z + 32};
  CUDA_TRY(c, cudaMemsetAsync(z, 0, scan_temps_bytes(N), c->stream));
  int32_t* err = (int32_t*)(st.ticket + 2);
  const unsigned blocks = (unsigned)(((size_t)N * 32 + 255) / 256);
  launch_pdl(v2p_mask_kernel<long long>, dim3(blocks), dim3(256), (size_t)0, c->stream, voxel_feats, C, (const long long*)voxel2point_inds, N, M,
             (const int32_t*)nullptr, padding, keep, mask_out, err);
  launch_exclusive_scan(c->stream, LoadU32{keep}, (size_t)N, nullptr, st, pos, st.ticket + 1, true);
  launch_pdl(v2p_write_kernel<long long>, dim3(blocks), dim3(256), (size_t)0, c->stream, points, Cp, (const long long*)pts_coors, voxel_feats, C,
             (const long long*)voxel2point_inds, N, (const uint32_t*)keep, (const uint32_t*)pos, voxel_size[0], voxel_size[1], voxel_size[2], pc_min[0],
             pc_min[1], pc_min[2], with_xyz, normalize_local_xyz, out);
  LAUNCH_CHECK(c);
  CUDA_TRY(c, cudaMemcpyAsync(num_out_dev, st.ticket + 1, 4, cudaMemcpyDeviceToDevice, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(c->pinned_i32, st.ticket + 1, 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(c->pinned_i32 + 1, err, 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  if (c->pinned_i32[1]) return sstb_fail(c, SSTB_ERR_ARG, "voxel2point: voxel2point_inds out of range [0, %d)", M);
  if (num_out_host) *num_out_host = c->pinned_i32[0];
  return SSTB_OK;
}

// Sync-free form (the FSD segmentation engine): int32 coordinates / indices, the voxel count on the device, the kept-row count
// written to num_out_dev by the compaction scan itself.  Nothing is read back.
extern "C" int sstb200_voxel2point_dev(sstb200_ctx* c, const float* points, int Cp, const int32_t* pts_coors, const float* voxel_feats,
                                       const int32_t* num_voxels_dev, int C, const int32_t* voxel2point_inds, int N, float padding,
                                       const float voxel_size[3], const float pc_min[3], int with_xyz, int normalize_local_xyz, float* out,
                                       uint8_t* mask_out, int32_t* num_out_dev) {
  CHECK_ARG(c, c && N >= 0 && C >= 1 && Cp >= 3 && num_out_dev);
  if (N == 0) {
    CUDA_TRY(c, cudaMemsetAsync(num_out_dev, 0, 4, c->stream));
    return SSTB_OK;
  }
  CHECK_ARG(c, points && pts_coors && voxel_feats && num_voxels_dev && voxel2point_inds && out && mask_out && voxel_size && pc_min);
  arena_reset(c);
  int rc = arena_reserve(c, 2 * al256((size_t)N * 4 + 64) + scan_temps_bytes(N) + 4096);
  if (rc) return rc;
  uint32_t* keep = arena_alloc<uint32_t>(c, (size_t)N + 2);
  uint32_t* pos = arena_alloc<uint32_t>(c, (size_t)N + 2);
  uint8_t* z = arena_alloc<uint8_t>(c, scan_temps_bytes(N));
  if (!keep || !pos || !z) return sstb_fail(c, SSTB_ERR_WORKSPACE, "voxel2point_dev: arena");
  ScanTemps st{(uint32_t*)z, (unsigned long long*)z + 32};
  CUDA_TRY(c, cudaMemsetAsync(z, 0, scan_temps_bytes(N), c->stream));
  const unsigned blocks = (unsigned)(((size_t)N * 32 + 255) / 256);
  launch_pdl(v2p_mask_kernel<int32_t>, dim3(blocks), dim3(256), (size_t)0, c->stream, voxel_feats, C, voxel2point_inds, N, 0, num_voxels_dev,
             padding, keep, mask_out, (int32_t*)nullptr);
  launch_exclusive_scan(c->stream, LoadU32{keep}, (size_t)N, nullptr, st, pos, (uint32_t*)num_out_dev, true);
  launch_pdl(v2p_write_kernel<int32_t>, dim3(blocks), dim3(256), (size_t)0, c->stream, points, Cp, pts_coors, voxel_feats, C, voxel2point_inds, N,
             (const uint32_t*)keep, (const uint32_t*)pos, voxel_size[0], voxel_size[1], voxel_size[2], pc_min[0], pc_min[1], pc_min[2], with_xyz,
             normalize_local_xyz, out);
  LAUNCH_CHECK(c);
  return SSTB_OK;
}
