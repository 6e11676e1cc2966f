// Fused dynamic voxel feature encoder (V4 DynamicVFE, V6 DynamicScatterVFE), eval-mode BatchNorm.
//
// Reference (mmdet3d/models/voxel_encoders/voxel_encoder.py:229-298 / :551-612): three DynamicScatter /
// scatter_v2 calls (each re-running unique on the same coors), a dense int64 canvas to map voxels back to
// points, [P,64] and [P,128] point-feature tensors and P*C float atomics.  Here: one bitmap-rank index, one
// CSR, then one warp per voxel computes the decorated point features, both VFE layers and the max-pool in
// registers - the per-point feature tensors are never materialised.
#include <stdarg.h>
#include "index.cuh"
#include "sra.cuh"
#include "umma.cuh"

struct VfeDev {
  int F, D0, C0, C1, nlayers;
  int with_cluster, with_center, with_distance, mode_max;
  float vx, vy, vz, x_off, y_off, z_off;
  float rel_dist_scaler;
  const float* W0;  // [C0, D0]
  const float* W1;  // [C1, 2*C0]
  const float *s0, *t0, *s1, *t1;  // folded BN: y = x*s + t
};

// fold eval BatchNorm into scale/shift
__global__ void fold_bn_kernel(const float* __restrict__ w, const float* __restrict__ b, const float* __restrict__ mean,
                               const float* __restrict__ var, float eps, int C, float* __restrict__ s, float* __restrict__ t) {
  pdl_wait();
  pdl_launch();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  // F.batch_norm: (x - mean) / sqrt(var + eps) * w + b
  float inv = 1.0f / sqrtf(var[c] + eps);
  float sc = w[c] * inv;
  s[c] = sc;
  t[c] = b[c] - mean[c] * sc;
}

// rank -> output row with the reference's "first sorted row of every sample is removed" rule
// (scatter_points_cuda.cu:207-210 applied per sample by scatter_points.py:85-99).
struct SampleQuirk {
  const uint32_t* word_prefix;
  size_t words_per_sample;
  int batch;
  int enabled;
};
__device__ __forceinline__ long long quirk_row(const SampleQuirk& q, long long rank, int b) {
  if (!q.enabled) return rank;
  long long first_b = q.word_prefix[(size_t)b * q.words_per_sample];
  if (rank == first_b) return -1;
  int shift = 0;
  for (int i = 0; i <= b; i++) {
    long long f0 = q.word_prefix[(size_t)i * q.words_per_sample], f1 = q.word_prefix[(size_t)(i + 1) * q.words_per_sample];
    shift += (f1 > f0);
  }
  return rank - shift;
}

template <typename TC, bool SM>
__global__ void __launch_bounds__(SM ? 1024 : 256) vfe_mark_kernel(const TC* __restrict__ coors, int P, int B, int Z, int Y, int X, size_t cells_pad,
                                long long* __restrict__ keys, uint32_t* __restrict__ bitmap, int32_t* __restrict__ flags,
                                uint32_t nwords) {
  pdl_wait();
  pdl_launch();
  extern __shared__ uint32_t mark_sbm[];  // SM: block-private bitmap (see mark_rows_kernel in index.cuh)
  if (SM) {
    for (uint32_t w = threadIdx.x; w < nwords; w += blockDim.x) mark_sbm[w] = 0u;
    __syncthreads();
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x) {
    long long b = (long long)coors[(size_t)i * 4], z = (long long)coors[(size_t)i * 4 + 1], y = (long long)coors[(size_t)i * 4 + 2],
              x = (long long)coors[(size_t)i * 4 + 3];
    if (b < 0 || b >= B || z < 0 || z >= Z || y < 0 || y >= Y || x < 0 || x >= X) {
      keys[i] = -1;
      flags[0] = 1;
      continue;
    }
    long long key = b * (long long)cells_pad + (z * Y + y) * X + x;
    keys[i] = key;
    if (SM) atomicOr(&mark_sbm[key >> 5], 1u << (key & 31));
    else bitmap_set(bitmap, key);
  }
  if (SM) bitmap_merge(mark_sbm, bitmap, nwords);
}

template <typename TM>
__global__ void vfe_map_kernel(const long long* __restrict__ keys, int P, const uint32_t* __restrict__ bitmap,
                               const uint32_t* __restrict__ word_prefix, size_t cells_pad, SampleQuirk q,
                               TM* __restrict__ map, int32_t* __restrict__ count) {
  pdl_wait();
  pdl_launch();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  long long key = keys[i];
  long long row = -1;
  if (key >= 0) {
    size_t w = (size_t)(key >> 5);
    long long rank = (long long)word_prefix[w] + __popc(bitmap[w] & ((1u << (key & 31)) - 1u));
    row = quirk_row(q, rank, (int)(key / (long long)cells_pad));
  }
  map[i] = (TM)row;
  if (row >= 0) atomicAdd(&count[row], 1);
}

template <typename TO>
__global__ void vfe_emit_kernel(const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ word_prefix, size_t nwords,
                                size_t cells_pad, int Y, int X, SampleQuirk q, TO* __restrict__ out_coors,
                                const uint32_t* __restrict__ total, int32_t* __restrict__ num_out) {
  pdl_wait();
  pdl_launch();
  size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w == 0) {
    long long t = *total;
    if (q.enabled) {
      int ne = 0;
      for (int i = 0; i < q.batch; i++)
        ne += q.word_prefix[(size_t)(i + 1) * q.words_per_sample] > q.word_prefix[(size_t)i * q.words_per_sample];
      t -= ne;
    }
    *num_out = (int32_t)t;
  }
  // four threads per bitmap word (one byte each): the serial decode loop is at most 8 cells long
  for (size_t t = w; t < nwords * 4; t += (size_t)gridDim.x * blockDim.x) {
    const size_t ww = t >> 2;
    const int part = (int)(t & 3);
    const uint32_t word = bitmap[ww];
    uint32_t bits = (word >> (8 * part)) & 0xFFu;
    if (!bits) continue;
    long long rank = (long long)word_prefix[ww] + __popc(word & ((1u << (8 * part)) - 1u));
    int b = (ww * 32 < cells_pad) ? 0 : (int)((ww * 32) / cells_pad);
    while (bits) {
      int bit = __ffs(bits) - 1 + 8 * part;
      bits &= bits - 1;
      long long row = quirk_row(q, rank, b);
      if (row >= 0) {
        long long local = (long long)(ww * 32 + bit) - (long long)b * (long long)cells_pad;
        long long x, y, z;
        if (cells_pad < ((size_t)1 << 31)) {  // 32-bit divisions (every real canvas)
          uint32_t lc = (uint32_t)local, q1 = lc / (uint32_t)X;
          x = lc - q1 * (uint32_t)X;
          uint32_t q2 = q1 / (uint32_t)Y;
          y = q1 - q2 * (uint32_t)Y;
          z = q2;
        } else {
          x = local % X, y = (local / X) % Y, z = local / ((long long)X * Y);
        }
        out_coors[row * 4 + 0] = (TO)b;
        out_coors[row * 4 + 1] = (TO)z;
        out_coors[row * 4 + 2] = (TO)y;
        out_coors[row * 4 + 3] = (TO)x;
      }
      rank++;
    }
  }
}

// ---- the fused per-voxel kernels ---------------------------------------------------------------------
#define VFE_MAXD 16

// decorated features of point p (all lanes get the same values)
template <typename TC>
__device__ __forceinline__ void decorate(const VfeDev& v, const float* __restrict__ pts, const TC* __restrict__ coors, int p,
                                         float mx, float my, float mz, float* f) {
  int ln = lane_id();
  float raw = (ln < v.F) ? pts[(size_t)p * v.F + ln] : 0.f;
  int k = 0;
  for (; k < v.F; k++) f[k] = __shfl_sync(0xffffffffu, raw, k);
  float x = f[0], y = f[1], z = f[2];
  if (v.with_cluster) {
    f[k++] = (x - mx) / v.rel_dist_scaler;
    f[k++] = (y - my) / v.rel_dist_scaler;
    f[k++] = (z - mz) / v.rel_dist_scaler;
  }
  if (v.with_center) {
    // voxel_encoder.py:264-272: x - (coor_x * vx + x_offset)
    float cx = (float)coors[(size_t)p * 4 + 3], cy = (float)coors[(size_t)p * 4 + 2], cz = (float)coors[(size_t)p * 4 + 1];
    f[k++] = x - __fadd_rn(__fmul_rn(cx, v.vx), v.x_off);  // two roundings like torch's mul, add
    f[k++] = y - __fadd_rn(__fmul_rn(cy, v.vy), v.y_off);
    f[k++] = z - __fadd_rn(__fmul_rn(cz, v.vz), v.z_off);
  }
  if (v.with_distance) f[k++] = sqrtf(x * x + y * y + z * z);
}

// dynamic smem layout: W0t [D0][C0] | s0 t0 [2*C0] | W1at [C0][C1] | W1bt [C0][C1] | s1 t1 [2*C1]
template <typename TC, int NC0 /*C0/32*/, int NC1 /*C1/32*/>
__global__ void __launch_bounds__(256) vfe_fused_kernel(VfeDev v, const float* __restrict__ pts, const TC* __restrict__ coors,
                                                        const uint32_t* __restrict__ offsets, const int32_t* __restrict__ order,
                                                        const int32_t* __restrict__ nvox_dev, float* __restrict__ vmean /*[M,3] scratch*/,
                                                        float* __restrict__ vf0 /*[M,C0] scratch*/, float* __restrict__ out /*[M,Cout]*/,
                                                        int phase) {
  pdl_wait();
  pdl_launch();
  extern __shared__ float sm[];
  const int C0 = NC0 * 32, C1 = NC1 * 32, D0 = v.D0;
  float* W0t = sm;
  float* s0 = W0t + D0 * C0;
  float* t0 = s0 + C0;
  float* W1at = t0 + C0;
  float* W1bt = W1at + (size_t)C0 * C1;
  float* s1 = W1bt + (size_t)C0 * C1;
  float* t1 = s1 + C1;
  for (int i = threadIdx.x; i < D0 * C0; i += blockDim.x) W0t[i] = v.W0[(i % C0) * D0 + (i / C0)];
  for (int i = threadIdx.x; i < C0; i += blockDim.x) {
    s0[i] = v.s0[i];
    t0[i] = v.t0[i];
  }
  if (phase == 1 && NC1 > 0) {
    for (int i = threadIdx.x; i < C0 * C1; i += blockDim.x) {
      int k = i / C1, c = i % C1;
      W1at[i] = v.W1[(size_t)c * 2 * C0 + k];
      W1bt[i] = v.W1[(size_t)c * 2 * C0 + C0 + k];
    }
    for (int i = threadIdx.x; i < C1; i += blockDim.x) {
      s1[i] = v.s1[i];
      t1[i] = v.t1[i];
    }
  }
  __syncthreads();
  int M = *nvox_dev;
  int ln = lane_id();
  int warps = (gridDim.x * blockDim.x) >> 5;
  for (int vox = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; vox < M; vox += warps) {
    uint32_t b = offsets[vox], e = offsets[vox + 1];
    float mx = 0.f, my = 0.f, mz = 0.f;
    if (v.with_cluster) {
      if (phase == 0) {
        double sx = 0, sy = 0, sz = 0;
        for (uint32_t k = b + ln; k < e; k += 32) {
          int p = order[k];
          sx += pts[(size_t)p * v.F];
          sy += pts[(size_t)p * v.F + 1];
          sz += pts[(size_t)p * v.F + 2];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          sx += __shfl_xor_sync(0xffffffffu, sx, o);
          sy += __shfl_xor_sync(0xffffffffu, sy, o);
          sz += __shfl_xor_sync(0xffffffffu, sz, o);
        }
        float cnt = (float)(e - b);
        mx = (float)sx / cnt;
        my = (float)sy / cnt;
        mz = (float)sz / cnt;
        if (ln == 0) {
          vmean[(size_t)vox * 3] = mx;
          vmean[(size_t)vox * 3 + 1] = my;
          vmean[(size_t)vox * 3 + 2] = mz;
        }
      } else {
        mx = vmean[(size_t)vox * 3];
        my = vmean[(size_t)vox * 3 + 1];
        mz = vmean[(size_t)vox * 3 + 2];
      }
    }
    float f[VFE_MAXD];
    if (phase == 0) {
      float best[NC0], sum[NC0];
#pragma unroll
      for (int j = 0; j < NC0; j++) {
        best[j] = -INFINITY;
        sum[j] = 0.f;
      }
      for (uint32_t k = b; k < e; k++) {
        int p = order[k];
        decorate<TC>(v, pts, coors, p, mx, my, mz, f);
#pragma unroll
        for (int j = 0; j < NC0; j++) {
          int c = ln + 32 * j;
          float a = 0.f;
          for (int d = 0; d < D0; d++) a = fmaf(W0t[d * C0 + c], f[d], a);
          float y = fmaxf(fmaf(a, s0[c], t0[c]), 0.f);
          best[j] = fmaxf(best[j], y);
          sum[j] += y;
        }
      }
      float* dst = (NC1 > 0) ? vf0 : out;
#pragma unroll
      for (int j = 0; j < NC0; j++) dst[(size_t)vox * C0 + ln + 32 * j] = v.mode_max ? best[j] : sum[j] / (float)(e - b);
    } else if (NC1 > 0) {
      // voxel term: W1[:, C0:] . vf0[vox]
      float bterm[NC1 > 0 ? NC1 : 1];
#pragma unroll
      for (int j = 0; j < NC1; j++) bterm[j] = 0.f;
      for (int k = 0; k < C0; k++) {
        float g = vf0[(size_t)vox * C0 + k];
#pragma unroll
        for (int j = 0; j < NC1; j++) bterm[j] = fmaf(W1bt[(size_t)k * C1 + ln + 32 * j], g, bterm[j]);
      }
      float best[NC1 > 0 ? NC1 : 1], sum[NC1 > 0 ? NC1 : 1];
#pragma unroll
      for (int j = 0; j < NC1; j++) {
        best[j] = -INFINITY;
        sum[j] = 0.f;
      }
      for (uint32_t k = b; k < e; k++) {
        int p = order[k];
        decorate<TC>(v, pts, coors, p, mx, my, mz, f);
        float y0[NC0];
#pragma unroll
        for (int j = 0; j < NC0; j++) {
          int c = ln + 32 * j;
          float a = 0.f;
          for (int d = 0; d < D0; d++) a = fmaf(W0t[d * C0 + c], f[d], a);
          y0[j] = fmaxf(fmaf(a, s0[c], t0[c]), 0.f);
        }
        float acc[NC1 > 0 ? NC1 : 1];
#pragma unroll
        for (int j = 0; j < NC1; j++) acc[j] = bterm[j];
#pragma unroll
        for (int jj = 0; jj < NC0; jj++) {
#pragma unroll 8
          for (int l2 = 0; l2 < 32; l2++) {
            float yk = __shfl_sync(0xffffffffu, y0[jj], l2);
            const float* wr = W1at + (size_t)(jj * 32 + l2) * C1 + ln;
#pragma unroll
            for (int j = 0; j < NC1; j++) acc[j] = fmaf(wr[32 * j], yk, acc[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < NC1; j++) {
          int c = ln + 32 * j;
          float y = fmaxf(fmaf(acc[j], s1[c], t1[c]), 0.f);
          best[j] = fmaxf(best[j], y);
          sum[j] += y;
        }
      }
#pragma unroll
      for (int j = 0; j < NC1; j++) out[(size_t)vox * C1 + ln + 32 * j] = v.mode_max ? best[j] : sum[j] / (float)(e - b);
    }
  }
}


// =====================================================================================================
// Tile path (max pooling): points are visited in CSR (voxel-sorted) order in tiles of 128.
//   vfe_mean_kernel     per-voxel xyz mean (4 lanes per voxel, fp64 accumulate)
//   vfe_l0_tile_kernel  decorate + layer 0 (FFMA, fp32 exact) + in-tile segmented max -> vf0 [M,C0]
//   vfe_l1_umma_kernel  A = bf16([y0 || vf0[voxel]]) [128 x 2*C0], B = bf16(W1) -> tcgen05.mma into TMEM,
//                       epilogue BN+ReLU, post-activation tile to smem, in-tile segmented max -> vf1 [M,C1]
// Post-ReLU values are >= 0, so the max across tile edges is an integer atomicMax on the float bits
// (exact, order independent); segments interior to a tile are written with plain stores.
// =====================================================================================================
#define VT 128  // points per tile

__global__ void vfe_mean_kernel(const float* __restrict__ pts, int F, const uint32_t* __restrict__ offsets,
                                const int32_t* __restrict__ order, const int32_t* __restrict__ nvox_dev,
                                float* __restrict__ vmean) {
  pdl_wait();
  pdl_launch();
  int M = *nvox_dev;
  int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 2, l = threadIdx.x & 3;
  int ng = (gridDim.x * blockDim.x) >> 2;
  for (int v = g; v < M; v += ng) {
    uint32_t b = offsets[v], e = offsets[v + 1];
    double sx = 0, sy = 0, sz = 0;
    for (uint32_t k = b + l; k < e; k += 4) {
      const float* p = pts + (size_t)order[k] * F;
      sx += p[0];
      sy += p[1];
      sz += p[2];
    }
#pragma unroll
    for (int o = 1; o < 4; o <<= 1) {
      sx += __shfl_xor_sync(0xffffffffu, sx, o);
      sy += __shfl_xor_sync(0xffffffffu, sy, o);
      sz += __shfl_xor_sync(0xffffffffu, sz, o);
    }
    if (l == 0) {
      float cnt = (float)(e - b);
      vmean[(size_t)v * 3] = (float)sx / cnt;
      vmean[(size_t)v * 3 + 1] = (float)sy / cnt;
      vmean[(size_t)v * 3 + 2] = (float)sz / cnt;
    }
  }
}

// decorated features of the tile's points -> sF[VT][VFE_MAXD]; voxel id per row -> sVox
template <typename TC, typename TM>
__device__ __forceinline__ void tile_decorate(const VfeDev& v, const float* __restrict__ pts, const TC* __restrict__ coors,
                                              const int32_t* __restrict__ order, const TM* __restrict__ map,
                                              const float* __restrict__ vmean, int k0, int nrow, float (*sF)[VFE_MAXD], int* sVox) {
  for (int r = threadIdx.x; r < VT; r += blockDim.x) {
    if (r < nrow) {
      int p = order[k0 + r];
      int vox = (int)map[p];
      sVox[r] = vox;
      const float* pp = pts + (size_t)p * v.F;
      float x = pp[0], y = pp[1], z = pp[2];
      int k = 0;
      for (; k < v.F; k++) sF[r][k] = pp[k];
      if (v.with_cluster) {
        sF[r][k++] = (x - vmean[(size_t)vox * 3]) / v.rel_dist_scaler;
        sF[r][k++] = (y - vmean[(size_t)vox * 3 + 1]) / v.rel_dist_scaler;
        sF[r][k++] = (z - vmean[(size_t)vox * 3 + 2]) / v.rel_dist_scaler;
      }
      if (v.with_center) {
        float cx = (float)coors[(size_t)p * 4 + 3], cy = (float)coors[(size_t)p * 4 + 2], cz = (float)coors[(size_t)p * 4 + 1];
        sF[r][k++] = x - __fadd_rn(__fmul_rn(cx, v.vx), v.x_off);
        sF[r][k++] = y - __fadd_rn(__fmul_rn(cy, v.vy), v.y_off);
        sF[r][k++] = z - __fadd_rn(__fmul_rn(cz, v.vz), v.z_off);
      }
      if (v.with_distance) sF[r][k++] = sqrtf(x * x + y * y + z * z);
      for (; k < VFE_MAXD; k++) sF[r][k] = 0.f;
    } else {
      sVox[r] = -1;
    }
  }
}

// column-wise segmented max over the tile's rows (rows sorted by voxel); tile [VT][ld] fp32 in smem.  blockDim.x / C row
// groups work in parallel, each on VT / groups consecutive rows; a segment fully inside a group's rows is written with a
// plain store, the first / last segment of a group may continue in a neighbouring group or tile -> integer atomicMax on the
// float bits (values are >= 0 after ReLU; the rows concerned are zeroed beforehand by vfe_zero_edges_kernel).
#define VSUB 32  // finest row-group granularity used by the kernels below
__device__ __forceinline__ void tile_segmax(const float* tile, int ld, const int* sVox, int nrow, int C, float* __restrict__ out) {
  const int groups = blockDim.x / C;
  const int rows_per = VT / groups;
  const int c = threadIdx.x % C, grp = threadIdx.x / C;
  if (grp >= groups) return;
  const int r0 = grp * rows_per, r1 = min(r0 + rows_per, nrow);
  if (r0 >= r1) return;
  int seg = sVox[r0];
  bool first = true;  // the segment may have started in the previous group / tile
  float m = 0.f;      // post-ReLU values are >= 0
  for (int r = r0; r < r1; r++) {
    int sg = sVox[r];
    if (sg != seg) {
      if (first) atomicMax((int*)&out[(size_t)seg * C + c], __float_as_int(m));
      else out[(size_t)seg * C + c] = m;
      first = false;
      seg = sg;
      m = 0.f;
    }
    m = fmaxf(m, tile[r * ld + c]);
  }
  atomicMax((int*)&out[(size_t)seg * C + c], __float_as_int(m));  // may continue into the next group / tile
}

template <typename TC, typename TM, int C0>
__global__ void __launch_bounds__(256) vfe_l0_tile_kernel(VfeDev v, const float* __restrict__ pts, const TC* __restrict__ coors,
                                                          const uint32_t* __restrict__ offsets, const int32_t* __restrict__ order,
                                                          const TM* __restrict__ map, const int32_t* __restrict__ nvox_dev,
                                                          const float* __restrict__ vmean, float* __restrict__ vf0,
                                                          __nv_bfloat16* __restrict__ y0buf /*[P, C0] in CSR order, or null*/) {
  pdl_wait();
  pdl_launch();
  __shared__ __align__(16) float sF[VT][VFE_MAXD];
  __shared__ int sVox[VT];
  __shared__ float sW[VFE_MAXD][C0];  // W0 transposed
  __shared__ float sS[C0], sT[C0];
  extern __shared__ float sY[];  // [VT][C0+1]
  const int D0 = v.D0;
  for (int i = threadIdx.x; i < D0 * C0; i += blockDim.x) sW[i / C0][i % C0] = v.W0[(i % C0) * D0 + (i / C0)];
  for (int i = threadIdx.x; i < C0; i += blockDim.x) {
    sS[i] = v.s0[i];
    sT[i] = v.t0[i];
  }
  const int M = *nvox_dev;
  const int nvalid = M > 0 ? (int)offsets[M] : 0;
  for (int k0 = blockIdx.x * VT; k0 < nvalid; k0 += gridDim.x * VT) {
    int nrow = min(VT, nvalid - k0);
    __syncthreads();
    tile_decorate<TC, TM>(v, pts, coors, order, map, vmean, k0, nrow, sF, sVox);
    __syncthreads();
    {
      // thread = (channel c, row group): the channel's weights live in registers, the decorated point is read as float4
      const int c = threadIdx.x % C0, grp = threadIdx.x / C0, ngrp = blockDim.x / C0;
      float wreg[VFE_MAXD];
#pragma unroll
      for (int d = 0; d < VFE_MAXD; d++) wreg[d] = d < D0 ? sW[d][c] : 0.f;
      const float sc = sS[c], sh = sT[c];
      for (int r = grp; r < VT; r += ngrp) {
        float y = 0.f;
        if (r < nrow) {
          const float4* fp = reinterpret_cast<const float4*>(sF[r]);
          float a = 0.f;
#pragma unroll
          for (int q = 0; q < VFE_MAXD / 4; q++) {
            float4 f4 = fp[q];  // broadcast: all lanes of the warp read the same row
            a = fmaf(wreg[4 * q], f4.x, a);
            a = fmaf(wreg[4 * q + 1], f4.y, a);
            a = fmaf(wreg[4 * q + 2], f4.z, a);
            a = fmaf(wreg[4 * q + 3], f4.w, a);
          }
          y = fmaxf(fmaf(a, sc, sh), 0.f);
          if (y0buf) y0buf[(size_t)(k0 + r) * C0 + c] = __float2bfloat16(y);
        }
        sY[r * (C0 + 1) + c] = y;
      }
    }
    __syncthreads();
    tile_segmax(sY, C0 + 1, sVox, nrow, C0, vf0);
  }
}

// layer 1 on tensor cores.  K = 2*C0 (== 128 for C0 = 64), N = C1 (128).
template <typename TC, typename TM, int C0, int C1>
__global__ void __launch_bounds__(256) vfe_l1_umma_kernel(VfeDev v, const float* __restrict__ pts, const TC* __restrict__ coors,
                                                          const uint32_t* __restrict__ offsets, const int32_t* __restrict__ order,
                                                          const TM* __restrict__ map, const int32_t* __restrict__ nvox_dev,
                                                          const float* __restrict__ vmean, const float* __restrict__ vf0,
                                                          float* __restrict__ vf1, const __nv_bfloat16* __restrict__ y0buf) {
  pdl_wait();
  pdl_launch();
  constexpr int K = 2 * C0;
  static_assert(K % 64 == 0 && C1 % 16 == 0 && C1 <= 256, "shape");
  extern __shared__ uint8_t l1_smem_raw[];
  uint8_t* base = (uint8_t*)(((uintptr_t)l1_smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sB = base;                       // K/64 chunks x C1 rows x 128 B - staged ONCE per CTA (persistent over tiles)
  uint8_t* sA = sB + (size_t)C1 * K * 2;    // K/64 chunks x 128 rows x 128 B
  float* sTile = reinterpret_cast<float*>(sA);  // the A operand region is re-used after the MMA: [VT][C1+1] fp32
  __shared__ float sF[VT][VFE_MAXD];
  __shared__ int sVox[VT];
  __shared__ float sW0[VFE_MAXD][C0];
  __shared__ float sS0[C0], sT0[C0], sS1[C1], sT1[C1];
  __shared__ __align__(8) uint64_t mbar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int D0 = v.D0;
  const int M = *nvox_dev;
  const int nvalid = M > 0 ? (int)offsets[M] : 0;
  if ((int)blockIdx.x * VT >= nvalid) return;
  for (int i = tid; i < D0 * C0; i += blockDim.x) sW0[i / C0][i % C0] = v.W0[(i % C0) * D0 + (i / C0)];
  for (int i = tid; i < C0; i += blockDim.x) {
    sS0[i] = v.s0[i];
    sT0[i] = v.t0[i];
  }
  for (int i = tid; i < C1; i += blockDim.x) {
    sS1[i] = v.s1[i];
    sT1[i] = v.t1[i];
  }
  if (warp == 0) tmem_alloc(&tmem_slot, C1 < 32 ? 32 : C1);
  if (tid == 0) {
    mbar_init(smem_u32(&mbar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  // B operand: W1 [C1, K] fp32 -> bf16, K-major SWIZZLE_128B, once per CTA (4 pieces in flight per thread)
  for (int i0 = tid; i0 < C1 * (K / 8); i0 += blockDim.x * 4) {
    float4 f0[4], f1[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      int idx = i0 + u * blockDim.x;
      if (idx < C1 * (K / 8)) {
        const float* wp = v.W1 + (size_t)(idx / (K / 8)) * K + (idx % (K / 8)) * 8;
        f0[u] = __ldg(reinterpret_cast<const float4*>(wp));
        f1[u] = __ldg(reinterpret_cast<const float4*>(wp + 4));
      }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      int idx = i0 + u * blockDim.x;
      if (idx < C1 * (K / 8)) {
        int r = idx / (K / 8), j = idx % (K / 8);
        int4 q;
        q.x = (int)pack_bf16(f0[u].x, f0[u].y);
        q.y = (int)pack_bf16(f0[u].z, f0[u].w);
        q.z = (int)pack_bf16(f1[u].x, f1[u].y);
        q.w = (int)pack_bf16(f1[u].z, f1[u].w);
        int c = j >> 3, jj = j & 7;
        *reinterpret_cast<int4*>(sB + (size_t)c * C1 * 128 + r * 128 + ((jj ^ (r & 7)) << 4)) = q;
      }
    }
  }
  uint32_t parity = 0;
  for (int k0 = blockIdx.x * VT; k0 < nvalid; k0 += gridDim.x * VT) {
    const int nrow = min(VT, nvalid - k0);
    __syncthreads();  // previous tile's smem (sTile aliases sA) fully consumed
    for (int r = tid; r < VT; r += blockDim.x) sVox[r] = r < nrow ? (int)map[order[k0 + r]] : -1;
    __syncthreads();
    // A operand: row r = [ y0(point) (C0) || vf0[voxel] (C0) ] in bf16.  (1) y0 was written (bf16, CSR order) by the layer-0
    // kernel: plain cp.async into the swizzled operand; (2) the voxel's layer-0 max is gathered 4 rows in flight
    for (int idx = tid; idx < VT * (C0 / 8); idx += blockDim.x) {
      int r = idx / (C0 / 8), j = idx % (C0 / 8);
      int c = j >> 3, jj = j & 7;
      uint8_t* dst = sA + (size_t)c * VT * 128 + r * 128 + ((jj ^ (r & 7)) << 4);
      if (r < nrow) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(dst)), "l"(y0buf + (size_t)(k0 + r) * C0 + j * 8) : "memory");
      } else {
        *reinterpret_cast<int4*>(dst) = make_int4(0, 0, 0, 0);
      }
    }
    for (int i0 = tid; i0 < VT * (C0 / 8); i0 += blockDim.x * 4) {
      float4 g0[4], g1[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        int idx = i0 + u * blockDim.x;
        int r = idx / (C0 / 8), j = idx % (C0 / 8);
        g0[u] = g1[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (idx < VT * (C0 / 8) && r < nrow) {
          const float* gp = vf0 + (size_t)sVox[r] * C0 + j * 8;
          g0[u] = *reinterpret_cast<const float4*>(gp);
          g1[u] = *reinterpret_cast<const float4*>(gp + 4);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        int idx = i0 + u * blockDim.x;
        if (idx < VT * (C0 / 8)) {
          int r = idx / (C0 / 8), j = idx % (C0 / 8) + C0 / 8;
          int4 q;
          q.x = (int)pack_bf16(g0[u].x, g0[u].y);
          q.y = (int)pack_bf16(g0[u].z, g0[u].w);
          q.z = (int)pack_bf16(g1[u].x, g1[u].y);
          q.w = (int)pack_bf16(g1[u].z, g1[u].w);
          int c = j >> 3, jj = j & 7;
          *reinterpret_cast<int4*>(sA + (size_t)c * VT * 128 + r * 128 + ((jj ^ (r & 7)) << 4)) = q;
        }
      }
    }
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    if (tid == 0) {
      const uint32_t idesc = umma_idesc(128, C1);
      const uint32_t a0 = smem_u32(sA), b0 = smem_u32(sB);
#pragma unroll
      for (int c = 0; c < K / 64; c++)
#pragma unroll
        for (int s = 0; s < 4; s++)
          umma_bf16(tmem, umma_desc_sw128(a0 + c * VT * 128 + s * 32), umma_desc_sw128(b0 + c * C1 * 128 + s * 32), idesc,
                    (c | s) ? 1u : 0u);
      umma_commit(smem_u32(&mbar));
    }
    __syncwarp();
    mbar_wait(smem_u32(&mbar), parity);
    parity ^= 1u;
    tc_fence_after();
    // epilogue: BN + ReLU, tile to smem (operand buffers are free now: the MMA has completed)
    const int half = warp >> 2;
    const int lrow = (warp & 3) * 32 + (tid & 31);
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    constexpr int CB = C1 / 2;
#pragma unroll 1
    for (int c0 = half * CB; c0 < half * CB + CB; c0 += 32) {
      float acc[32];
      tmem_ld32(tlane + c0, acc);
#pragma unroll
      for (int i = 0; i < 32; i++) sTile[lrow * (C1 + 1) + c0 + i] = fmaxf(fmaf(acc[i], sS1[c0 + i], sT1[c0 + i]), 0.f);
    }
    tc_fence_before();
    __syncthreads();
    tile_segmax(sTile, C1 + 1, sVox, nrow, C1, vf1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_slot, C1 < 32 ? 32 : C1);
}


// rows of `out` that may be reached by atomicMax from two tiles (first / last voxel of every tile) start at 0
template <typename TM>
__global__ void vfe_zero_edges_kernel(const uint32_t* __restrict__ offsets, const int32_t* __restrict__ order,
                                      const TM* __restrict__ map, const int32_t* __restrict__ nvox_dev, int C, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int M = *nvox_dev;
  const int nvalid = M > 0 ? (int)offsets[M] : 0;
  for (int t = blockIdx.x; t * VSUB < nvalid; t += gridDim.x) {
    int k0 = t * VSUB, k1 = min(k0 + VSUB, nvalid) - 1;
    int v0 = (int)map[order[k0]], v1 = (int)map[order[k1]];
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      out[(size_t)v0 * C + c] = 0.f;
      out[(size_t)v1 * C + c] = 0.f;
    }
  }
}

template <typename TC, typename TM, int C0, int C1>
static int launch_vfe_tiles(sstb200_ctx* c, const VfeDev& v, const float* pts, const TC* coors, const Csr& r, const TM* map,
                            const int32_t* num_dev, float* vmean, float* vf0, float* out, bool umma_l1, bool* l1_done,
                            __nv_bfloat16* y0buf) {
  cudaStream_t st = c->stream;
  int grid = c->num_sms * 3;
  launch_pdl(vfe_mean_kernel, dim3(c->num_sms * 8), dim3(256), (size_t)(0), st, pts, v.F, r.offsets, r.order, num_dev, vmean);
  float* dst0 = (C1 > 0) ? vf0 : out;
  launch_pdl(vfe_zero_edges_kernel<TM>, dim3(c->num_sms * 8), dim3(64), (size_t)(0), st, r.offsets, r.order, map, num_dev, C0, dst0);
  size_t smem0 = (size_t)VT * (C0 + 1) * 4;
  launch_pdl(vfe_l0_tile_kernel<TC, TM, C0>, dim3(grid), dim3(256), (size_t)(smem0), st, v, pts, coors, r.offsets, r.order, map, num_dev, vmean, dst0,
             (C1 > 0 && umma_l1) ? y0buf : (__nv_bfloat16*)nullptr);
  *l1_done = false;
  if (C1 > 0 && umma_l1) {
    constexpr int C1s = C1 > 0 ? C1 : 32;
    size_t opA = (size_t)VT * 2 * C0 * 2, opB = (size_t)C1s * 2 * C0 * 2, tile = (size_t)VT * (C1s + 1) * 4;
    size_t smem1 = opB + (opA > tile ? opA : tile) + 1024;
    auto kern = vfe_l1_umma_kernel<TC, TM, C0, C1s>;
    static SmemAttr sa;
    CUDA_TRY(c, ensure_smem(c, sa, kern, smem1));
    launch_pdl(vfe_zero_edges_kernel<TM>, dim3(c->num_sms * 8), dim3(64), (size_t)(0), st, r.offsets, r.order, map, num_dev, C1s, out);
    launch_pdl(kern, dim3(grid), dim3(256), (size_t)(smem1), st, v, pts, coors, r.offsets, r.order, map, num_dev, vmean, vf0, out,
               (const __nv_bfloat16*)y0buf);
    *l1_done = true;
  }
  LAUNCH_CHECK(c);
  return SSTB_OK;
}

template <typename TC, int NC0, int NC1>
static int launch_vfe(sstb200_ctx* c, const VfeDev& v, const float* pts, const TC* coors, const Csr& r, const int32_t* num_dev,
                      float* vmean, float* vf0, float* out, bool skip_phase0 = false) {
  int C0 = NC0 * 32, C1 = NC1 * 32;
  size_t smem = ((size_t)v.D0 * C0 + 2 * C0 + 2 * (size_t)C0 * C1 + 2 * C1) * 4;
  size_t smem_max = ((size_t)VFE_MAXD * C0 + 2 * C0 + 2 * (size_t)C0 * C1 + 2 * C1) * 4;
  auto kern = vfe_fused_kernel<TC, NC0, NC1>;
  static SmemAttr sa;  // not a stream op, but kept out of CUDA-graph capture after warm-up
  CUDA_TRY(c, ensure_smem(c, sa, kern, smem_max));
  int grid = c->num_sms * 2;
  if (!skip_phase0) launch_pdl(kern, dim3(grid), dim3(256), (size_t)(smem), c->stream, v, pts, coors, r.offsets, r.order, num_dev, vmean, vf0, out, 0);
  if (NC1 > 0) launch_pdl(kern, dim3(grid), dim3(256), (size_t)(smem), c->stream, v, pts, coors, r.offsets, r.order, num_dev, vmean, vf0, out, 1);
  LAUNCH_CHECK(c);
  return SSTB_OK;
}

// =====================================================================================================
// Wide-input path (fp32): point dims beyond the fused kernels' register budget, e.g. FSDv2's virtual-voxel encoder
// DynamicScatterVFE(in_channels=67, feat_channels=[64,128]) (configs/fsdv2, SURVEY config 5).  Same index / CSR as above, then the
// layers as row GEMMs:  X = decorate(points)  ->  Y0 = relu(BN(X W0^T))  ->  V0 = segmax(Y0)
//                       Y1 = relu(BN(Y0 W1a^T + (V0 W1b^T)[voxel]))      ->  V1 = segmax(Y1)      ([Y0 || V0[voxel]] never materialised)
// =====================================================================================================
template <typename TC, typename TM>
__global__ void __launch_bounds__(256) vfe_decorate_wide_kernel(VfeDev v, const float* __restrict__ pts, const TC* __restrict__ coors,
                                                                const TM* __restrict__ map, const float* __restrict__ vmean, int P,
                                                                float* __restrict__ X, long long* __restrict__ row64) {
  pdl_wait();
  pdl_launch();
  const int lane = threadIdx.x & 31;
  const int p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (p >= P) return;
  const long long vox = (long long)map[p];
  if (lane == 0) row64[p] = vox < 0 ? 0 : vox;  // dropped points (quirk Q1) are in no CSR segment: any valid row keeps the GEMM in bounds
  const float* q = pts + (size_t)p * v.F;
  float* x = X + (size_t)p * v.D0;
  for (int k = lane; k < v.F; k += 32) x[k] = q[k];
  int base = v.F;
  if (v.with_cluster) {
    if (lane < 3) x[base + lane] = vox >= 0 ? (q[lane] - vmean[(size_t)vox * 3 + lane]) / v.rel_dist_scaler : 0.f;
    base += 3;
  }
  if (v.with_center) {
    if (lane < 3) {
      const float vs = lane == 0 ? v.vx : (lane == 1 ? v.vy : v.vz);
      const float off = lane == 0 ? v.x_off : (lane == 1 ? v.y_off : v.z_off);
      const float cc = (float)coors[(size_t)p * 4 + (3 - lane)];
      x[base + lane] = q[lane] - __fadd_rn(__fmul_rn(cc, vs), off);
    }
    base += 3;
  }
}

template <typename TC, typename TM>
static int vfe_wide_path(sstb200_ctx* c, const sstb200_vfe_cfg* cfg, const VfeDev& v, const float* pts, const TC* coors, const TM* map,
                         const Csr& r, int P, const int32_t* num_dev, float* vmean, float* out_feats) {
  cudaStream_t st = c->stream;
  const int D0 = v.D0, C0 = v.C0, C1 = v.C1;
  const int Cmax = C0 > C1 ? C0 : C1;
  float* X = arena_alloc<float>(c, (size_t)P * D0);
  float* Y0 = arena_alloc<float>(c, (size_t)P * C0);
  float* T1 = C1 ? arena_alloc<float>(c, (size_t)P * Cmax) : nullptr;
  float* V0 = C1 ? arena_alloc<float>(c, (size_t)P * C0) : nullptr;
  float* G = C1 ? arena_alloc<float>(c, (size_t)P * C1) : nullptr;
  long long* row64 = arena_alloc<long long>(c, (size_t)P);
  if (!X || !Y0 || !row64 || (C1 && (!T1 || !V0 || !G))) return sstb_fail(c, SSTB_ERR_WORKSPACE, "vfe (wide): arena");
  const int mode = v.mode_max ? SSTB200_REDUCE_MAX : SSTB200_REDUCE_MEAN;
  launch_pdl(vfe_mean_kernel, dim3(c->num_sms * 8), dim3(256), (size_t)0, st, pts, v.F, (const uint32_t*)r.offsets, (const int32_t*)r.order, num_dev,
             vmean);
  launch_pdl(vfe_decorate_wide_kernel<TC, TM>, dim3((unsigned)(((size_t)P * 32 + 255) / 256)), dim3(256), (size_t)0, st, v, pts, coors, map,
             (const float*)vmean, P, X, row64);
  sstb_gemm_rows_ex(st, X, D0, cfg->weight[0], D0, nullptr, nullptr, 0, nullptr, Y0, C0, P, nullptr, C0, D0, 0, nullptr, nullptr, 0, 0, 0, 0);
  sstb_add_norm_act(st, Y0, nullptr, cfg->bn_weight[0], cfg->bn_bias[0], cfg->bn_mean[0], cfg->bn_var[0], cfg->bn_eps, Y0, P, nullptr, C0, 1);
  launch_segment_reduce(c, Y0, C0, r.offsets, r.order, P, num_dev, mode, 0.f, C1 ? V0 : out_feats, nullptr, P);
  if (C1) {
    sstb_gemm_rows_ex(st, V0, C0, cfg->weight[1] + C0, 2 * C0, nullptr, nullptr, 0, nullptr, G, C1, P, num_dev, C1, C0, 0, nullptr, nullptr, 0, 0,
                      0, 0);
    sstb_gemm_rows_ex(st, Y0, C0, cfg->weight[1], 2 * C0, nullptr, G, C1, (const long long*)row64, T1, C1, P, nullptr, C1, C0, 0, nullptr, nullptr,
                      0, 0, 0, 0);
    sstb_add_norm_act(st, T1, nullptr, cfg->bn_weight[1], cfg->bn_bias[1], cfg->bn_mean[1], cfg->bn_var[1], cfg->bn_eps, T1, P, nullptr, C1, 1);
    launch_segment_reduce(c, T1, C1, r.offsets, r.order, P, num_dev, mode, 0.f, out_feats, nullptr, P);
  }
  LAUNCH_CHECK(c);
  return SSTB_OK;
}

template <typename TC>
static int vfe_forward_impl(sstb200_ctx* c, const sstb200_vfe_cfg* cfg, const float* pts, const TC* coors, int P,
                            float* out_feats, TC* out_coors, TC* inverse, int32_t* num_dev, int32_t* num_host) {
  CHECK_ARG(c, c && cfg && P >= 0 && num_dev);
  if (P == 0) {
    CUDA_TRY(c, cudaMemsetAsync(num_dev, 0, 4, c->stream));
    if (num_host) *num_host = 0;
    return SSTB_OK;
  }
  CHECK_ARG(c, pts && coors && out_feats && out_coors);
  CHECK_ARG(c, cfg->num_layers >= 1 && cfg->num_layers <= 2 && cfg->in_channels >= 3 && cfg->batch_size >= 1);
  int F = cfg->in_channels;
  int D0 = F + 3 * (cfg->with_cluster_center != 0) + 3 * (cfg->with_voxel_center != 0) + (cfg->with_distance != 0);
  int C0 = cfg->feat_channels[0], C1 = cfg->num_layers > 1 ? cfg->feat_channels[1] : 0;
  const bool wide = D0 > VFE_MAXD || F > 32;  // beyond the fused kernels: row-GEMM path below (fp32)
  if (wide && cfg->with_distance) return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "VFE with_distance is not built");
  CHECK_ARG(c, cfg->weight[0] && cfg->bn_weight[0] && cfg->bn_bias[0] && cfg->bn_mean[0] && cfg->bn_var[0]);
  if (C1) CHECK_ARG(c, cfg->weight[1] && cfg->bn_weight[1] && cfg->bn_bias[1] && cfg->bn_mean[1] && cfg->bn_var[1]);
  int Z = cfg->grid_zyx[0], Y = cfg->grid_zyx[1], X = cfg->grid_zyx[2], B = cfg->batch_size;
  CHECK_ARG(c, Z > 0 && Y > 0 && X > 0);
  size_t cells = (size_t)Z * Y * X;
  size_t cells_pad = (cells + 31) / 32 * 32;
  long long T = (long long)cells_pad * B;
  if (T > ((long long)1 << 34)) return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "voxel grid too large for bitmap rank (%lld cells)", T);
  arena_reset(c);
  int rc = arena_reserve(c, key_index_bytes(P, T) + csr_bytes(P, P) + al256((size_t)P * 4) * 3 + al256((size_t)P * 3 * 4) +
                                al256((size_t)P * C0 * 4) + al256((size_t)P * C0 * 2 + 128) + al256((size_t)(C0 + C1) * 8) + 8192 +
                                (wide ? al256((size_t)P * D0 * 4) + 4 * al256((size_t)P * (C0 > C1 ? C0 : C1) * 4) + al256((size_t)P * 8) : 0));
  if (rc) return rc;
  KeyIndex k;
  rc = key_index_alloc(c, k, P, T);
  if (rc) return rc;
  int32_t* count = arena_alloc<int32_t>(c, (size_t)P + 2);
  int32_t* map32 = inverse ? nullptr : arena_alloc<int32_t>(c, P);
  float* vmean = arena_alloc<float>(c, (size_t)P * 3);
  float* vf0 = arena_alloc<float>(c, (size_t)P * C0);
  float* fold = arena_alloc<float>(c, 2 * (size_t)(C0 + C1) + 8);
  __nv_bfloat16* y0buf = arena_alloc<__nv_bfloat16>(c, (size_t)P * C0 + 64);  // layer-0 point features (bf16, CSR order) for the tcgen05 layer 1
  if (!count || !vmean || !vf0 || !fold || !y0buf) return sstb_fail(c, SSTB_ERR_WORKSPACE, "vfe: arena");
  CUDA_TRY(c, cudaMemsetAsync(count, 0, ((size_t)P + 2) * 4, c->stream));
  int nb = (P + 255) / 256;
  if (k.nwords <= 12 * 1024) {  // <= 48 KB: block-private bitmap
    int mg = (P + 1023) / 1024;
    if (mg > c->num_sms) mg = c->num_sms;
    launch_pdl(vfe_mark_kernel<TC, true>, dim3(mg), dim3(1024), k.nwords * 4, c->stream, coors, P, B, Z, Y, X, cells_pad, k.keys, k.bitmap, k.flags,
               (uint32_t)k.nwords);
  } else {
    launch_pdl(vfe_mark_kernel<TC, false>, dim3(nb), dim3(256), (size_t)(0), c->stream, coors, P, B, Z, Y, X, cells_pad, k.keys, k.bitmap, k.flags, 0u);
  }
  key_index_scan(c, k);
  SampleQuirk q{k.word_prefix, cells_pad / 32, B, cfg->drop_first_voxel_per_sample != 0};
  int eg = (int)((k.nwords * 4 + 63) / 64);
  if (eg > c->num_sms * 32) eg = c->num_sms * 32;
  launch_pdl(vfe_emit_kernel<TC>, dim3(eg), dim3(64), (size_t)(0), c->stream, k.bitmap, k.word_prefix, k.nwords, cells_pad, Y, X, q, out_coors, k.total, num_dev);
  CUDA_TRY(c, cudaEventRecord(c->ev_coords, c->stream));   // voxel_coors / num_dev are final from here on (sstb200_branch_fork)
  Csr r;
  if (inverse) {
    launch_pdl(vfe_map_kernel<TC>, dim3(nb), dim3(256), (size_t)(0), c->stream, k.keys, P, k.bitmap, k.word_prefix, cells_pad, q, inverse, count);
    rc = csr_build<TC>(c, r, inverse, P, count, P, num_dev);
  } else {
    launch_pdl(vfe_map_kernel<int32_t>, dim3(nb), dim3(256), (size_t)(0), c->stream, k.keys, P, k.bitmap, k.word_prefix, cells_pad, q, map32, count);
    rc = csr_build<int32_t>(c, r, map32, P, count, P, num_dev);
  }
  if (rc) return rc;
  VfeDev v;
  v.F = F;
  v.D0 = D0;
  v.C0 = C0;
  v.C1 = C1;
  v.nlayers = cfg->num_layers;
  v.with_cluster = cfg->with_cluster_center != 0;
  v.with_center = cfg->with_voxel_center != 0;
  v.with_distance = cfg->with_distance != 0;
  v.mode_max = cfg->mode_max != 0;
  v.vx = cfg->voxel_size[0];
  v.vy = cfg->voxel_size[1];
  v.vz = cfg->voxel_size[2];
  v.x_off = cfg->center_offset[0];
  v.y_off = cfg->center_offset[1];
  v.z_off = cfg->center_offset[2];
  v.rel_dist_scaler = cfg->rel_dist_scaler;
  v.W0 = cfg->weight[0];
  v.W1 = cfg->weight[1];
  v.s0 = fold;
  v.t0 = fold + C0;
  v.s1 = fold + 2 * C0;
  v.t1 = fold + 2 * C0 + C1;
  if (wide) {
    rc = inverse ? vfe_wide_path<TC, TC>(c, cfg, v, pts, coors, (const TC*)inverse, r, P, num_dev, vmean, out_feats)
                 : vfe_wide_path<TC, int32_t>(c, cfg, v, pts, coors, (const int32_t*)map32, r, P, num_dev, vmean, out_feats);
    if (rc) return rc;
    if (num_host) return read_back_i32(c, num_dev, num_host);
    return SSTB_OK;
  }
  launch_pdl(fold_bn_kernel, dim3((C0 + 127) / 128), dim3(128), (size_t)(0), c->stream, cfg->bn_weight[0], cfg->bn_bias[0], cfg->bn_mean[0], cfg->bn_var[0],
                                                           cfg->bn_eps, C0, fold, fold + C0);
  if (C1)
    launch_pdl(fold_bn_kernel, dim3((C1 + 127) / 128), dim3(128), (size_t)(0), c->stream, cfg->bn_weight[1], cfg->bn_bias[1], cfg->bn_mean[1], cfg->bn_var[1],
                                                             cfg->bn_eps, C1, fold + 2 * C0, fold + 2 * C0 + C1);
  LAUNCH_CHECK(c);
  {
    // tile path (max pooling, the configurations on the hot path): layer 0 FFMA tiles; layer 1 on tcgen05 when bf16
    bool l1_done = false, tiled = false;
    const bool umma = cfg->precision == SSTB200_PREC_BF16;
#define VFE_TILE(a, b)                                                                                                          \
  if (!tiled && v.mode_max && C0 == a && C1 == b) {                                                                             \
    if (inverse) rc = launch_vfe_tiles<TC, TC, a, b>(c, v, pts, coors, r, inverse, num_dev, vmean, vf0, out_feats, umma, &l1_done, y0buf); \
    else rc = launch_vfe_tiles<TC, int32_t, a, b>(c, v, pts, coors, r, map32, num_dev, vmean, vf0, out_feats, umma, &l1_done, y0buf);    \
    if (rc) return rc;                                                                                                          \
    tiled = true;                                                                                                               \
  }
    VFE_TILE(64, 128)
    VFE_TILE(64, 64)
    VFE_TILE(64, 0)
    VFE_TILE(32, 64)
#undef VFE_TILE
#define VFE_CASE(a, b)                                                                                     \
  if (C0 == a * 32 && C1 == b * 32) {                                                                      \
    if (!(tiled && (l1_done || C1 == 0)))                                                                  \
      rc = launch_vfe<TC, a, b>(c, v, pts, coors, r, num_dev, vmean, vf0, out_feats, /*skip_phase0=*/tiled); \
    goto done;                                                                                             \
  }
    VFE_CASE(2, 4)
    VFE_CASE(2, 2)
    VFE_CASE(1, 2)
    VFE_CASE(2, 0)
    VFE_CASE(4, 4)
    VFE_CASE(4, 0)
    VFE_CASE(1, 0)
    VFE_CASE(1, 1)
    VFE_CASE(2, 8)
#undef VFE_CASE
    return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "VFE channel combination (%d,%d) not instantiated", C0, C1);
  }
done:
  if (rc) return rc;
  if (num_host) return read_back_i32(c, num_dev, num_host);
  return SSTB_OK;
}

extern "C" int sstb200_dynamic_vfe_forward(sstb200_ctx* c, const sstb200_vfe_cfg* cfg, const float* points, const int32_t* coors,
                                           int P, float* voxel_feats, int32_t* voxel_coors, int32_t* num_dev, int32_t* num_host) {
  return vfe_forward_impl<int32_t>(c, cfg, points, coors, P, voxel_feats, voxel_coors, nullptr, num_dev, num_host);
}

extern "C" int sstb200_dynamic_scatter_vfe_forward(sstb200_ctx* c, const sstb200_vfe_cfg* cfg, const float* points,
                                                   const int64_t* coors, int P, float* voxel_feats, int64_t* voxel_coors,
                                                   int64_t* unq_inv, int32_t* num_dev, int32_t* num_host) {
  CHECK_ARG(c, unq_inv);
  return vfe_forward_impl<long long>(c, cfg, points, (const long long*)coors, P, voxel_feats, (long long*)voxel_coors,
                                     (long long*)unq_inv, num_dev, num_host);
}

// DynamicScatterVFE on the frame engine's rows: int32 (b,z,y,x) coordinates of sstb200_voxelize_frames (capacity rows; rows past the
// last frame are -1 and belong to no voxel: their unq_inv is -1), int32 voxel coordinates and inverse, the voxel count on the device
// only.  The grid (cfg->grid_zyx) comes from the voxeliser geometry.
extern "C" int sstb200_dynamic_scatter_vfe_forward_i32(sstb200_ctx* c, const sstb200_vfe_cfg* cfg, const float* points, const int32_t* coors,
                                                       int num_points, float* voxel_feats, int32_t* voxel_coors, int32_t* unq_inv,
                                                       int32_t* num_voxels_dev) {
  CHECK_ARG(c, unq_inv);
  return vfe_forward_impl<int32_t>(c, cfg, points, coors, num_points, voxel_feats, voxel_coors, unq_inv, num_voxels_dev, nullptr);
}
