// Sparse 3-D convolution (SURVEY 8f next-1): SubMConv3d / SparseConv3d / SparseInverseConv3d of the reference's sparse U-Nets
// (mmdet3d/models/middle_encoders/sparse_unet.py:15-505, mmdet3d/ops/sparse_block.py:81-289), which the reference delegates to spconv
// (vendored v1: mmdet3d/ops/spconv/include/spconv/geometry.h:25-301 builds the index pairs, spconv_ops.h:95-260 runs one gather ->
// GEMM -> scatter-add per kernel offset).
//
// B200 form: OUTPUT-STATIONARY.  The rulebook is a neighbour table nbr[o][k] = input row that feeds output row o through kernel
// offset k (or -1), built from the bitmap-rank index of the active coordinates (no hash table, no sort, no atomics on features); a
// convolution is then ONE implicit-GEMM launch: an output tile gathers its <= KV input rows per offset, accumulates all offsets
// in registers / TMEM and applies the folded BatchNorm (+ residual) (+ ReLU) epilogue before its single store.  The reference's
// form writes every output row KV times with atomics-free but serialised scatter-adds and keeps BN / ReLU / residual as separate
// passes over [N, C].
#include <stdarg.h>
#include <cuda_fp16.h>
#include "index.cuh"
#include "umma.cuh"
#include "sra.cuh"

namespace {

struct SpGeom {
  int B;
  int in_shape[3];   // z, y, x
  int out_shape[3];
  int ks[3], st[3], pd[3];
  int KV;
};

__device__ __forceinline__ int sp_rank(const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ word_prefix, long long key) {
  const size_t w = (size_t)(key >> 5);
  const uint32_t bit = 1u << (key & 31);
  const uint32_t word = bitmap[w];
  if (!(word & bit)) return -1;
  return (int)(word_prefix[w] + __popc(word & (bit - 1u)));
}

// perm[rank(row i)] = i  (rows are unique: a permutation)
__global__ void sp_perm_kernel(const long long* __restrict__ keys, int n, const int32_t* __restrict__ n_dev,
                               const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ word_prefix, int32_t* __restrict__ perm) {
  pdl_wait();
  pdl_launch();
  if (n_dev) n = min(n, *n_dev);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const long long key = keys[i];
    if (key < 0) continue;
    const int r = sp_rank(bitmap, word_prefix, key);
    if (r >= 0) perm[r] = i;
  }
}

// candidate outputs of a strided convolution: o = (i + pad - delta) / stride where divisible and inside the output grid
// (all table kernels loop grid-stride over (row, offset) pairs; n_dev != nullptr: the row count is read from the device, n is a capacity)
__global__ void sp_mark_out_kernel(const int32_t* __restrict__ coors, int n, const int32_t* __restrict__ n_dev, SpGeom g,
                                   uint32_t* __restrict__ out_bitmap, int32_t* __restrict__ flags) {
  pdl_wait();
  pdl_launch();
  if (n_dev) n = min(n, *n_dev);
  const long long work = (long long)n * g.KV;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < work; t += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(t / g.KV), k = (int)(t % g.KV);
    const int4 c = *reinterpret_cast<const int4*>(coors + (size_t)i * 4);  // b, z, y, x
    if (c.x < 0 || c.x >= g.B || c.y < 0 || c.y >= g.in_shape[0] || c.z < 0 || c.z >= g.in_shape[1] || c.w < 0 || c.w >= g.in_shape[2]) {
      if (k == 0) flags[1] = 1;
      continue;
    }
    const int dz = k / (g.ks[1] * g.ks[2]), dy = (k / g.ks[2]) % g.ks[1], dx = k % g.ks[2];
    const int tz = c.y + g.pd[0] - dz, ty = c.z + g.pd[1] - dy, tx = c.w + g.pd[2] - dx;
    if (tz < 0 || ty < 0 || tx < 0) continue;
    if (tz % g.st[0] || ty % g.st[1] || tx % g.st[2]) continue;
    const int oz = tz / g.st[0], oy = ty / g.st[1], ox = tx / g.st[2];
    if (oz >= g.out_shape[0] || oy >= g.out_shape[1] || ox >= g.out_shape[2]) continue;
    const long long key = (((long long)c.x * g.out_shape[0] + oz) * g.out_shape[1] + oy) * g.out_shape[2] + ox;
    bitmap_set(out_bitmap, key);
  }
}

// nbr[o][k] = row of the input coordinate  o * stride - pad + delta_k  (or -1)
__global__ void sp_nbr_kernel(const int32_t* __restrict__ out_coors, int n_out, const int32_t* __restrict__ n_out_dev, SpGeom g,
                              const uint32_t* __restrict__ in_bitmap, const uint32_t* __restrict__ in_prefix,
                              const int32_t* __restrict__ in_perm, int32_t* __restrict__ nbr) {
  pdl_wait();
  pdl_launch();
  if (n_out_dev) n_out = min(n_out, *n_out_dev);
  const long long work = (long long)n_out * g.KV;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < work; t += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(t / g.KV), k = (int)(t % g.KV);
    const int4 c = *reinterpret_cast<const int4*>(out_coors + (size_t)o * 4);
    int res = -1;
    if (c.x >= 0 && c.x < g.B && c.y >= 0 && c.z >= 0 && c.w >= 0) {
      const int dz = k / (g.ks[1] * g.ks[2]), dy = (k / g.ks[2]) % g.ks[1], dx = k % g.ks[2];
      const int iz = c.y * g.st[0] - g.pd[0] + dz, iy = c.z * g.st[1] - g.pd[1] + dy, ix = c.w * g.st[2] - g.pd[2] + dx;
      if (iz >= 0 && iz < g.in_shape[0] && iy >= 0 && iy < g.in_shape[1] && ix >= 0 && ix < g.in_shape[2]) {
        const long long key = (((long long)c.x * g.in_shape[0] + iz) * g.in_shape[1] + iy) * g.in_shape[2] + ix;
        const int r = sp_rank(in_bitmap, in_prefix, key);
        if (r >= 0) res = in_perm[r];
      }
    }
    nbr[t] = res;
  }
}

// nbr_inv[i][k] = output row reached from input row i through offset k (the transposed table: SparseInverseConv3d), or -1
__global__ void sp_nbr_inv_kernel(const int32_t* __restrict__ in_coors, int n_in, const int32_t* __restrict__ n_in_dev, SpGeom g,
                                  const uint32_t* __restrict__ out_bitmap, const uint32_t* __restrict__ out_prefix,
                                  const int32_t* __restrict__ out_perm, int32_t* __restrict__ nbr_inv) {
  pdl_wait();
  pdl_launch();
  if (n_in_dev) n_in = min(n_in, *n_in_dev);
  const long long work = (long long)n_in * g.KV;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < work; t += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(t / g.KV), k = (int)(t % g.KV);
    const int4 c = *reinterpret_cast<const int4*>(in_coors + (size_t)i * 4);
    int res = -1;
    if (c.x >= 0 && c.x < g.B && c.y >= 0 && c.z >= 0 && c.w >= 0) {
      const int dz = k / (g.ks[1] * g.ks[2]), dy = (k / g.ks[2]) % g.ks[1], dx = k % g.ks[2];
      const int tz = c.y + g.pd[0] - dz, ty = c.z + g.pd[1] - dy, tx = c.w + g.pd[2] - dx;
      if (tz >= 0 && ty >= 0 && tx >= 0 && tz % g.st[0] == 0 && ty % g.st[1] == 0 && tx % g.st[2] == 0) {
        const int oz = tz / g.st[0], oy = ty / g.st[1], ox = tx / g.st[2];
        if (oz < g.out_shape[0] && oy < g.out_shape[1] && ox < g.out_shape[2]) {
          const long long key = (((long long)c.x * g.out_shape[0] + oz) * g.out_shape[1] + oy) * g.out_shape[2] + ox;
          const int r = sp_rank(out_bitmap, out_prefix, key);
          if (r >= 0) res = out_perm[r];
        }
      }
    }
    nbr_inv[t] = res;
  }
}

static int sp_geom(sstb200_ctx* c, SpGeom& g, int B, const int32_t* in_shape, const int32_t* out_shape, const int32_t* ks,
                   const int32_t* st, const int32_t* pd) {
  CHECK_ARG(c, B >= 1 && in_shape && out_shape && ks && st && pd);
  g.B = B;
  g.KV = 1;
  for (int d = 0; d < 3; d++) {
    CHECK_ARG(c, in_shape[d] >= 1 && out_shape[d] >= 1 && ks[d] >= 1 && ks[d] <= 7 && st[d] >= 1 && pd[d] >= 0);
    g.in_shape[d] = in_shape[d];
    g.out_shape[d] = out_shape[d];
    g.ks[d] = ks[d];
    g.st[d] = st[d];
    g.pd[d] = pd[d];
    g.KV *= ks[d];
  }
  return SSTB_OK;
}

static int sp_extents(sstb200_ctx* c, Extents& e, long long* T, int B, const int* shape) {
  long long lo[4] = {0, 0, 0, 0}, hi[4] = {B - 1, shape[0] - 1, shape[1] - 1, shape[2] - 1};
  return make_extents(c, e, 4, lo, hi, T);
}

// ------------------------------------------------------------------------------------------------------------------------------
// fp32 implicit GEMM (the 1e-3 / "exact" path): 64 x 64 output tile per CTA, 4 x 4 micro-tile per thread, K = KV * Cin walked
// offset by offset in chunks of 16 channels; offsets no row of the tile uses are skipped.
// ------------------------------------------------------------------------------------------------------------------------------
#define SPF_BM 64
#define SPF_BN 64
#define SPF_BK 16
__global__ void __launch_bounds__(256) spconv_gemm_f32_kernel(const float* __restrict__ feats, int lda, int Cin, const int32_t* __restrict__ nbr,
                                                             int n_out, const int32_t* __restrict__ n_dev, int KV,
                                                             const float* __restrict__ W, int Cout, const float* __restrict__ scale,
                                                             const float* __restrict__ shift, const float* __restrict__ residual, int ldr,
                                                             int relu, float* __restrict__ out, int ldo) {
  pdl_wait();
  pdl_launch();
  __shared__ __align__(16) float sA[SPF_BK][SPF_BM + 4];
  __shared__ __align__(16) float sB[SPF_BK][SPF_BN];
  __shared__ int sRow[SPF_BM];
  if (n_dev) n_out = min(n_out, *n_dev);
  const int tid = threadIdx.x;
  const int n0 = blockIdx.y * SPF_BN;
  const int ty = tid >> 4, tx = tid & 15;
  // row tiles grid-stride (one tile per CTA when the grid covers n_out); every barrier below is reached by the whole CTA
  for (int row0 = blockIdx.x * SPF_BM; row0 < n_out; row0 += gridDim.x * SPF_BM) {
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
    for (int k = 0; k < KV; k++) {
      int mine = -1;
      if (tid < SPF_BM) {
        const int o = row0 + tid;
        mine = o < n_out ? nbr[(size_t)o * KV + k] : -1;
        sRow[tid] = mine;
      }
      if (!__syncthreads_or(mine >= 0)) continue;   // (barrier: sRow visible; previous chunk's reads of sA / sB are complete)
      for (int c0 = 0; c0 < Cin; c0 += SPF_BK) {
        {  // A: 64 rows x 16 channels, one float4 per thread, stored transposed
          const int r = tid >> 2, q = tid & 3;
          const int src = sRow[r];
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (src >= 0 && c0 + q * 4 < Cin) v = *reinterpret_cast<const float4*>(feats + (size_t)src * lda + c0 + q * 4);
          sA[q * 4 + 0][r] = v.x;
          sA[q * 4 + 1][r] = v.y;
          sA[q * 4 + 2][r] = v.z;
          sA[q * 4 + 3][r] = v.w;
        }
        {  // B: 16 channels x 64 outputs
          const int kk = tid >> 4, q = tid & 15;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (c0 + kk < Cin && n0 + q * 4 < Cout) v = __ldg(reinterpret_cast<const float4*>(W + ((size_t)k * Cin + c0 + kk) * Cout + n0 + q * 4));
          *reinterpret_cast<float4*>(&sB[kk][q * 4]) = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < SPF_BK; kk++) {
          const float4 a = *reinterpret_cast<const float4*>(&sA[kk][ty * 4]);
          const float4 b = *reinterpret_cast<const float4*>(&sB[kk][tx * 4]);
          const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
          for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
      }
    }
    const int col = n0 + tx * 4;
    if (col >= Cout) continue;
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (scale) sc = __ldg(reinterpret_cast<const float4*>(scale + col));
    if (shift) sh = __ldg(reinterpret_cast<const float4*>(shift + col));
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int o = row0 + ty * 4 + i;
      if (o >= n_out) continue;
      float4 y;
      y.x = fmaf(acc[i][0], sc.x, sh.x);
      y.y = fmaf(acc[i][1], sc.y, sh.y);
      y.z = fmaf(acc[i][2], sc.z, sh.z);
      y.w = fmaf(acc[i][3], sc.w, sh.w);
      if (residual) {
        const float4 r4 = *reinterpret_cast<const float4*>(residual + (size_t)o * ldr + col);
        y.x += r4.x, y.y += r4.y, y.z += r4.z, y.w += r4.w;
      }
      if (relu) y.x = fmaxf(y.x, 0.f), y.y = fmaxf(y.y, 0.f), y.z = fmaxf(y.z, 0.f), y.w = fmaxf(y.w, 0.f);
      *reinterpret_cast<float4*>(out + (size_t)o * ldo + col) = y;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------------------
// weight gradient:  dW[k] += sum over output rows o with nbr[o][k] >= 0 of  X[nbr[o][k]]^T . dY[o]      (fp32, FFMA)
// CTA = (chunk of SPW_ROWS output rows, kernel offset k, 64 x 64 tile of dW[k]).  The rows of the chunk that actually have a neighbour
// at offset k (17 % on a LiDAR sweep) are compacted into shared memory first, so the reduction only walks real pairs; the partial
// tile is added to dW with fp32 atomics (summation order across chunks is not fixed, like the reference's atomics-based backward).
// ------------------------------------------------------------------------------------------------------------------------------
#define SPW_ROWS 1024
__global__ void __launch_bounds__(256) spconv_dw_kernel(const float* __restrict__ X, int Cin, const int32_t* __restrict__ nbr, int n_out, int KV,
                                                       const float* __restrict__ dY, int Cout, float* __restrict__ dW) {
  pdl_wait();
  pdl_launch();
  __shared__ int sIn[SPW_ROWS], sOut[SPW_ROWS];
  __shared__ int sCount;
  __shared__ __align__(16) float sA[16][64];
  __shared__ __align__(16) float sB[16][64];
  const int tid = threadIdx.x;
  const int k = blockIdx.y;
  const int ncot = (Cout + 63) / 64;
  const int ci0 = ((int)blockIdx.z / ncot) * 64, co0 = ((int)blockIdx.z % ncot) * 64;
  const int r0 = blockIdx.x * SPW_ROWS;
  if (tid == 0) sCount = 0;
  __syncthreads();
  for (int j = tid; j < SPW_ROWS; j += 256) {
    const int o = r0 + j;
    if (o < n_out) {
      const int v = nbr[(size_t)o * KV + k];
      if (v >= 0) {
        const int pos = atomicAdd(&sCount, 1);
        sIn[pos] = v;
        sOut[pos] = o;
      }
    }
  }
  __syncthreads();
  const int cnt = sCount;
  if (cnt == 0) return;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
  for (int q0 = 0; q0 < cnt; q0 += 16) {
    {
      const int r = tid >> 4, c4 = (tid & 15) * 4;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q0 + r < cnt) {
        if (ci0 + c4 < Cin) a = *reinterpret_cast<const float4*>(X + (size_t)sIn[q0 + r] * Cin + ci0 + c4);
        if (co0 + c4 < Cout) b = *reinterpret_cast<const float4*>(dY + (size_t)sOut[q0 + r] * Cout + co0 + c4);
      }
      *reinterpret_cast<float4*>(&sA[r][c4]) = a;
      *reinterpret_cast<float4*>(&sB[r][c4]) = b;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 16; r++) {
      const float4 a = *reinterpret_cast<const float4*>(&sA[r][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&sB[r][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int ci = ci0 + ty * 4 + i;
    if (ci >= Cin) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int co = co0 + tx * 4 + j;
      if (co < Cout) atomicAdd(&dW[((size_t)k * Cin + ci) * Cout + co], acc[i][j]);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------------------
// tensor-core implicit GEMM (precision 'bf16' = 16-bit operands, fp32 accumulation): 128-row output tile x NT output channels per
// CTA, accumulators [128, NT] fp32 in TMEM across ALL kernel offsets, operands IEEE fp16 in the K-major SWIZZLE_128B layout (same
// staging / descriptors as umma_gemm.cuh).  K is walked in stages of (kernel offset, 64 input channels): the 256 threads gather the
// 128 neighbour rows (fp32 -> fp16 on the fly, absent neighbours = zero rows that are neither loaded nor converted) and the [NT, 64]
// weight slab into one of NS operand buffers, one thread issues 4 tcgen05.mma (K = 16 each) and commits to the buffer's mbarrier; the
// global loads run TWO stages ahead in two register sets (the deep levels of a U-Net are a few CTAs walking 100-200 stages each:
// pure load latency), and a buffer is rewritten only after its commit has fired.  Offsets no row of the tile uses are skipped.  Epilogue: thread-per-row out of TMEM, y = acc * scale + shift (+ residual) (ReLU), fp32 rows.
// ------------------------------------------------------------------------------------------------------------------------------
constexpr int SPU_TM = 128;
constexpr int SPU_A_BYTES = SPU_TM * 128;
#define SPU_MAX_KV 27

// fp32 pair -> fp16x2 with saturation to +-65504 in ONE instruction (F2FP.SATFINITE.F16.F32.PACK_AB); a = low half
__device__ __forceinline__ uint32_t sp_pack_f16(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

struct SpArgs {
  const float* feats;      // [*, lda] fp32 rows (gathered through nbr, or row o itself when nbr == nullptr)
  int lda, Cin;
  const int32_t* nbr;      // [n_out, KV] or nullptr (KV must be 1: a plain row GEMM)
  int n_out;
  const int32_t* n_dev;    // optional device-side row count (<= n_out)
  int KV;
  const __half* Whi;       // [KV][Cout][Cin] fp16
  const __half* Wlo;       // SPLIT: the fp16 residue  W - float(Whi)
  int Cout;
  const float *scale, *shift, *residual;
  int ldr, act;            // act: 0 none, 1 ReLU, 2 GELU (erf form)
  float* out;
  int ldo;
};

template <int BU, bool SPLIT>
struct SpStageRegs {
  float4 a0[4], a1[4];            // 4 pieces of 8 gathered channels each
  int4 b[BU];                     // weight pieces
  int4 blo[SPLIT ? BU : 1];       // SPLIT: residue pieces
  uint32_t valid;                 // bit u: piece u has a source row (absent neighbours are neither loaded nor converted)
};

// SPLIT = the fp32-tolerance mode on the tensor core: every fp32 operand is carried as two fp16 numbers (hi = rn(x), lo = rn(x - hi):
// 22 significant bits), and a stage issues the three products hi.hi + lo.hi + hi.lo into the same fp32 TMEM accumulator (the
// dropped lo.lo term is 2^-22 relative).  Same staging, same epilogue; 3x the MMAs, 2x the operand bytes.
// LOOP = false: one output tile per CTA (grid covers the rows); LOOP = true: CTAs loop over the row tiles of the device row count
// (the grid is sized from the SM count, not from the capacity).
template <int NT, int NS, bool SPLIT, bool LOOP>
__global__ void __launch_bounds__(256, (NT == 64 && !SPLIT) ? 2 : 1) spconv_umma_kernel(SpArgs g) {
  pdl_wait();
  pdl_launch();
  extern __shared__ uint8_t sp_smem_raw[];
  uint8_t* base = (uint8_t*)(((uintptr_t)sp_smem_raw + 1023) & ~(uintptr_t)1023);
  constexpr int B_BYTES = NT * 128;
  constexpr int ST_BYTES = (SPLIT ? 2 : 1) * (SPU_A_BYTES + B_BYTES);   // [A_hi][A_lo][B_hi][B_lo] or [A][B]
  constexpr int OFF_ALO = SPU_A_BYTES, OFF_B = (SPLIT ? 2 : 1) * SPU_A_BYTES, OFF_BLO = OFF_B + B_BYTES;
  constexpr int BU = NT / 32;  // 16-byte weight pieces per thread and stage
  __shared__ __align__(8) uint64_t mbar[NS];
  __shared__ uint32_t tmem_slot;
  __shared__ uint32_t used_mask;
  __shared__ int sNbr[SPU_TM][SPU_MAX_KV];   // odd row pitch: conflict-free column reads

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n0 = blockIdx.y * NT;
  const int n_out = g.n_dev ? min(g.n_out, *g.n_dev) : g.n_out;
  if ((int)blockIdx.x * SPU_TM >= n_out) return;   // uniform per CTA, nothing allocated yet
  const int KV = g.KV, Cin = g.Cin, Cout = g.Cout;
  if (warp == 0) tmem_alloc(&tmem_slot, NT);
  if (tid == 0) {
#pragma unroll
    for (int b = 0; b < NS; b++) mbar_init(smem_u32(&mbar[b]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  // Output tiles grid-stride (one tile per CTA when the grid covers n_out).  Stage numbers keep counting across the tiles of a CTA
  // (s_base), so operand buffer s % NS and its mbarrier phase s / NS continue where the previous tile left them.
  int s_base = 0;
#pragma unroll 1
  for (int row0 = blockIdx.x * SPU_TM; row0 < n_out; row0 = LOOP ? row0 + gridDim.x * SPU_TM : n_out) {
    if (tid == 0) used_mask = 0u;
    __syncthreads();
    {
      uint32_t m = 0u;
      for (int idx = tid; idx < SPU_TM * KV; idx += 256) {
        const int r = idx / KV, k = idx - r * KV;
        const int o = row0 + r;
        const int v = o < n_out ? (g.nbr ? g.nbr[(size_t)o * KV + k] : o) : -1;
        sNbr[r][k] = v;
        if (v >= 0) m |= 1u << k;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, o);
      if (lane == 0 && m) atomicOr(&used_mask, m);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const int nch = Cin >> 6;
    const int nst = __popc(used_mask) * nch;

    // stage iterator of the loader (stages are visited in order: used offsets ascending, 64-channel chunks inside)
    uint32_t ld_mask = used_mask;
    int ld_c = 0, loaded = 0;
    const int my_r = tid >> 3, my_jj = tid & 7;   // piece u of this thread: row my_r + 32 u, 16-byte column my_jj
    auto load_next = [&](SpStageRegs<BU, SPLIT>& R) {
      if (loaded >= nst) return;
      const int k = __ffs(ld_mask) - 1, c = ld_c;
      R.valid = 0u;
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int src = sNbr[my_r + 32 * u][k];
        if (src >= 0) {
          R.valid |= 1u << u;
          const float* ap = g.feats + (size_t)src * g.lda + c * 64 + my_jj * 8;
          R.a0[u] = *reinterpret_cast<const float4*>(ap);
          R.a1[u] = *reinterpret_cast<const float4*>(ap + 4);
        }
      }
      const size_t woff = ((size_t)k * Cout + n0 + my_r) * Cin + c * 64 + my_jj * 8;
#pragma unroll
      for (int u = 0; u < BU; u++) {
        R.b[u] = __ldg(reinterpret_cast<const int4*>(g.Whi + woff + (size_t)32 * u * Cin));
        if (SPLIT) R.blo[u] = __ldg(reinterpret_cast<const int4*>(g.Wlo + woff + (size_t)32 * u * Cin));
      }
      loaded++;
      if (++ld_c == nch) {
        ld_c = 0;
        ld_mask &= ld_mask - 1u;
      }
    };
    auto run_stage = [&](int s, SpStageRegs<BU, SPLIT>& R) {
      const int b = (s_base + s) % NS, u_ = (s_base + s) / NS;
      uint8_t* sA = base + (size_t)b * ST_BYTES;
      uint8_t* sB = sA + OFF_B;
      if (u_ >= 1) {  // the MMAs that read this buffer NS stages ago have completed
        mbar_wait(smem_u32(&mbar[b]), (uint32_t)((u_ - 1) & 1));
        tc_fence_after();
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int r = my_r + 32 * u;
        const int off = r * 128 + ((my_jj ^ (r & 7)) << 4);
        int4 v = make_int4(0, 0, 0, 0), vl = make_int4(0, 0, 0, 0);
        if ((R.valid >> u) & 1u) {
          const float f[8] = {R.a0[u].x, R.a0[u].y, R.a0[u].z, R.a0[u].w, R.a1[u].x, R.a1[u].y, R.a1[u].z, R.a1[u].w};
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; e++) {
            hi[e] = sp_pack_f16(f[2 * e], f[2 * e + 1]);
            if (SPLIT) {
              const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi[e]));
              lo[e] = sp_pack_f16(f[2 * e] - h.x, f[2 * e + 1] - h.y);
            }
          }
          v = make_int4((int)hi[0], (int)hi[1], (int)hi[2], (int)hi[3]);
          if (SPLIT) vl = make_int4((int)lo[0], (int)lo[1], (int)lo[2], (int)lo[3]);
        }
        *reinterpret_cast<int4*>(sA + off) = v;
        if (SPLIT) *reinterpret_cast<int4*>(sA + OFF_ALO + off) = vl;
      }
#pragma unroll
      for (int u = 0; u < BU; u++) {
        const int r = my_r + 32 * u;
        const int off = r * 128 + ((my_jj ^ (r & 7)) << 4);
        *reinterpret_cast<int4*>(sB + off) = R.b[u];
        if (SPLIT) *reinterpret_cast<int4*>(sA + OFF_BLO + off) = R.blo[u];
      }
      load_next(R);         // the register set is free again: fetch the stage two ahead while this one is multiplied
      fence_async_smem();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
      tc_fence_before();
      __syncthreads();
      tc_fence_after();
      if (tid == 0) {
        const uint32_t idesc = umma_idesc_f16(SPU_TM, NT);
        const uint32_t a0 = smem_u32(sA), b0 = smem_u32(sB);
#pragma unroll
        for (int q = 0; q < 4; q++)
          umma_f16(tmem, umma_desc_sw128(a0 + q * 32), umma_desc_sw128(b0 + q * 32), idesc, (s | q) ? 1u : 0u);
        if (SPLIT) {
          const uint32_t al = a0 + OFF_ALO, bl = a0 + OFF_BLO;
#pragma unroll
          for (int q = 0; q < 4; q++) umma_f16(tmem, umma_desc_sw128(al + q * 32), umma_desc_sw128(b0 + q * 32), idesc, 1u);   // lo . hi
#pragma unroll
          for (int q = 0; q < 4; q++) umma_f16(tmem, umma_desc_sw128(a0 + q * 32), umma_desc_sw128(bl + q * 32), idesc, 1u);   // hi . lo
        }
        umma_commit(smem_u32(&mbar[b]));  // implicit tcgen05.fence::before_thread_sync
      }
    };

    SpStageRegs<BU, SPLIT> R0, R1;
    R0.valid = R1.valid = 0u;
    load_next(R0);
    load_next(R1);
    for (int s = 0; s < nst; s += 2) {
      run_stage(s, R0);
      if (s + 1 < nst) run_stage(s + 1, R1);
    }
    if (nst > 0) {
      const int s = s_base + nst - 1;
      mbar_wait(smem_u32(&mbar[s % NS]), (uint32_t)((s / NS) & 1));   // commit of the last stage: every MMA of the tile is done
      tc_fence_after();
    }

    // ---- epilogue -------------------------------------------------------------------------------------------------------------
    const int half = warp >> 2;                       // warps 0-3: columns [0, NT/2), warps 4-7: [NT/2, NT)
    const int lrow = (warp & 3) * 32 + lane;          // TMEM lane == row inside the tile
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int o = row0 + lrow;
    constexpr int CB = NT / 2;
    constexpr int EC = LOOP ? 16 : 32;   // columns per TMEM load (the looping kernel keeps more state live across tiles)
#pragma unroll 1
    for (int c0 = half * CB; c0 < half * CB + CB; c0 += EC) {
      float v[EC];
      if (nst > 0) {
        if (EC == 32) tmem_ld32(tlane + c0, v);
        else tmem_ld16(tlane + c0, v);
      } else {
#pragma unroll
        for (int i = 0; i < EC; i++) v[i] = 0.f;
      }
      if (o < n_out) {
        const int col = n0 + c0;
        float* op = g.out + (size_t)o * g.ldo + col;
        const float* rp = g.residual ? g.residual + (size_t)o * g.ldr + col : nullptr;
#pragma unroll
        for (int q = 0; q < EC / 4; q++) {
          float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
          if (g.scale) sc = __ldg(reinterpret_cast<const float4*>(g.scale + col) + q);
          if (g.shift) sh = __ldg(reinterpret_cast<const float4*>(g.shift + col) + q);
          float4 y;
          y.x = fmaf(v[4 * q], sc.x, sh.x);
          y.y = fmaf(v[4 * q + 1], sc.y, sh.y);
          y.z = fmaf(v[4 * q + 2], sc.z, sh.z);
          y.w = fmaf(v[4 * q + 3], sc.w, sh.w);
          if (g.act == 2) y.x = gelu_erf(y.x), y.y = gelu_erf(y.y), y.z = gelu_erf(y.z), y.w = gelu_erf(y.w);   // Linear -> GELU (-> + residual)
          if (rp) {
            const float4 r4 = *(reinterpret_cast<const float4*>(rp) + q);
            y.x += r4.x, y.y += r4.y, y.z += r4.z, y.w += r4.w;
          }
          if (g.act == 1) y.x = fmaxf(y.x, 0.f), y.y = fmaxf(y.y, 0.f), y.z = fmaxf(y.z, 0.f), y.w = fmaxf(y.w, 0.f);  // conv + BN + res -> ReLU
          *(reinterpret_cast<float4*>(op) + q) = y;
        }
      }
    }
    s_base += nst;
    tc_fence_before();   // this tile's TMEM loads and sNbr / used_mask reads are complete before the next tile reuses them
    __syncthreads();
    tc_fence_after();
  }
  if (warp == 0) tmem_dealloc(tmem, NT);
}

// max_row_ctas > 0 (device row counts): at most that many CTAs per column block, looping over the row tiles of the real row count
template <int NT, int NS, bool SPLIT, bool LOOP>
static int launch_spconv_umma(sstb200_ctx* c, const SpArgs& g, int max_row_ctas) {
  auto kern = spconv_umma_kernel<NT, NS, SPLIT, LOOP>;
  static SmemAttr sa;
  const size_t smem = (size_t)NS * (SPLIT ? 2 : 1) * (SPU_A_BYTES + NT * 128) + 1024;
  CUDA_TRY(c, ensure_smem(c, sa, kern, smem));
  int tiles = (g.n_out + SPU_TM - 1) / SPU_TM;
  if (LOOP && tiles > max_row_ctas) tiles = max_row_ctas;
  dim3 grid(tiles, g.Cout / NT);
  launch_pdl(kern, grid, dim3(256), smem, c->stream, g);
  LAUNCH_CHECK(c);
  return SSTB_OK;
}

template <bool LOOP>
static int dispatch_spconv_umma(sstb200_ctx* c, const SpArgs& g, bool split, int max_row_ctas) {
  if (split) {
    if (g.Cout % 256 == 0) return launch_spconv_umma<256, 2, true, LOOP>(c, g, max_row_ctas);
    if (g.Cout % 128 == 0) return launch_spconv_umma<128, 2, true, LOOP>(c, g, max_row_ctas);
    return launch_spconv_umma<64, 3, true, LOOP>(c, g, max_row_ctas);
  }
  if (g.Cout % 256 == 0) return launch_spconv_umma<256, 2, false, LOOP>(c, g, max_row_ctas);
  if (g.Cout % 128 == 0) return launch_spconv_umma<128, 3, false, LOOP>(c, g, max_row_ctas);
  return launch_spconv_umma<64, 3, false, LOOP>(c, g, max_row_ctas);
}

// W fp32 -> (hi, lo) fp16, elementwise
__global__ void split_f16_kernel(const float* __restrict__ w, size_t n, __half* __restrict__ hi, __half* __restrict__ lo) {
  pdl_wait();
  pdl_launch();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = w[i];
  const __half h = __float2half_rn(fminf(fmaxf(x, -65504.f), 65504.f));
  hi[i] = h;
  lo[i] = __float2half_rn(x - __half2float(h));
}

}  // namespace

// ------------------------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------------------------
extern "C" int sstb200_spconv_out_coors(sstb200_ctx* c, const int32_t* in_coors, int n_in, int batch_size, const int32_t in_shape[3],
                                        const int32_t out_shape[3], const int32_t ksize[3], const int32_t stride[3],
                                        const int32_t padding[3], int32_t* out_coors, int out_cap, int32_t* num_out_dev,
                                        int32_t* num_out_host) {
  CHECK_ARG(c, c && n_in >= 0 && num_out_dev);
  SpGeom g;
  int rc = sp_geom(c, g, batch_size, in_shape, out_shape, ksize, stride, padding);
  if (rc) return rc;
  if (n_in == 0) {
    CUDA_TRY(c, cudaMemsetAsync(num_out_dev, 0, 4, c->stream));
    if (num_out_host) *num_out_host = 0;
    return SSTB_OK;
  }
  CHECK_ARG(c, in_coors && out_coors);
  // every input reaches at most prod(ceil(k / s)) outputs
  long long per_in = 1, cells = batch_size;
  for (int d = 0; d < 3; d++) {
    per_in *= (g.ks[d] + g.st[d] - 1) / g.st[d];
    cells *= g.out_shape[d];
  }
  long long bound = (long long)n_in * per_in;
  if (bound > cells) bound = cells;
  if ((long long)out_cap < bound)
    return sstb_fail(c, SSTB_ERR_ARG, "spconv_out_coors: out_cap %d < worst case %lld rows", out_cap, bound);
  Extents e;
  long long T;
  rc = sp_extents(c, e, &T, batch_size, g.out_shape);
  if (rc) return rc;
  arena_reset(c);
  rc = arena_reserve(c, key_index_bytes(1, T) + 4096);
  if (rc) return rc;
  KeyIndex k;
  rc = key_index_alloc(c, k, 1, T);
  if (rc) return rc;
  const long long work = (long long)n_in * g.KV;
  launch_pdl(sp_mark_out_kernel, dim3((unsigned)((work + 255) / 256)), dim3(256), (size_t)0, c->stream, in_coors, n_in, (const int32_t*)nullptr, g,
             k.bitmap, k.flags);
  key_index_scan(c, k);
  launch_emit_rows<int32_t>(c, k, e, 0, out_coors, num_out_dev);
  LAUNCH_CHECK(c);
  if (num_out_host) {
    rc = read_back_i32(c, num_out_dev, num_out_host);
    if (rc) return rc;
    int32_t bad = 0;
    rc = read_back_i32(c, k.flags + 1, &bad);
    if (rc) return rc;
    if (bad) return sstb_fail(c, SSTB_ERR_ARG, "spconv_out_coors: an input coordinate lies outside batch_size / in_shape");
  }
  return SSTB_OK;
}

extern "C" int sstb200_spconv_table(sstb200_ctx* c, const int32_t* in_coors, int n_in, const int32_t* out_coors, int n_out,
                                    int batch_size, const int32_t in_shape[3], const int32_t out_shape[3], const int32_t ksize[3],
                                    const int32_t stride[3], const int32_t padding[3], int32_t* nbr, int32_t* nbr_inv,
                                    int32_t* status_host) {
  CHECK_ARG(c, c && n_in >= 0 && n_out >= 0);
  SpGeom g;
  int rc = sp_geom(c, g, batch_size, in_shape, out_shape, ksize, stride, padding);
  if (rc) return rc;
  if (status_host) *status_host = 0;
  if (n_in == 0 || n_out == 0) {
    if (nbr && n_out) CUDA_TRY(c, cudaMemsetAsync(nbr, 0xFF, (size_t)n_out * g.KV * 4, c->stream));
    if (nbr_inv && n_in) CUDA_TRY(c, cudaMemsetAsync(nbr_inv, 0xFF, (size_t)n_in * g.KV * 4, c->stream));
    return SSTB_OK;
  }
  CHECK_ARG(c, in_coors && out_coors && (nbr || nbr_inv));
  Extents ei, eo;
  long long Ti, To;
  rc = sp_extents(c, ei, &Ti, batch_size, g.in_shape);
  if (rc) return rc;
  rc = sp_extents(c, eo, &To, batch_size, g.out_shape);
  if (rc) return rc;
  arena_reset(c);
  rc = arena_reserve(c, key_index_bytes(n_in, Ti) + key_index_bytes(n_out, To) + al256((size_t)n_in * 4) + al256((size_t)n_out * 4) + 8192);
  if (rc) return rc;
  KeyIndex ki, ko;
  int32_t *perm_i = nullptr, *perm_o = nullptr;
  if (nbr) {
    rc = key_index_alloc(c, ki, n_in, Ti);
    if (rc) return rc;
    perm_i = arena_alloc<int32_t>(c, n_in);
    if (!perm_i) return sstb_fail(c, SSTB_ERR_WORKSPACE, "spconv_table: arena too small");
    launch_mark_rows<int32_t>(c, in_coors, n_in, ei, false, ki, nullptr);
    key_index_scan(c, ki);
    launch_pdl(sp_perm_kernel, dim3((n_in + 255) / 256), dim3(256), (size_t)0, c->stream, (const long long*)ki.keys, n_in, (const int32_t*)nullptr,
               (const uint32_t*)ki.bitmap, (const uint32_t*)ki.word_prefix, perm_i);
    const long long work = (long long)n_out * g.KV;
    launch_pdl(sp_nbr_kernel, dim3((unsigned)((work + 255) / 256)), dim3(256), (size_t)0, c->stream, out_coors, n_out, (const int32_t*)nullptr, g,
               (const uint32_t*)ki.bitmap,
               (const uint32_t*)ki.word_prefix, (const int32_t*)perm_i, nbr);
  }
  if (nbr_inv) {
    rc = key_index_alloc(c, ko, n_out, To);
    if (rc) return rc;
    perm_o = arena_alloc<int32_t>(c, n_out);
    if (!perm_o) return sstb_fail(c, SSTB_ERR_WORKSPACE, "spconv_table: arena too small");
    launch_mark_rows<int32_t>(c, out_coors, n_out, eo, false, ko, nullptr);
    key_index_scan(c, ko);
    launch_pdl(sp_perm_kernel, dim3((n_out + 255) / 256), dim3(256), (size_t)0, c->stream, (const long long*)ko.keys, n_out, (const int32_t*)nullptr,
               (const uint32_t*)ko.bitmap, (const uint32_t*)ko.word_prefix, perm_o);
    const long long work = (long long)n_in * g.KV;
    launch_pdl(sp_nbr_inv_kernel, dim3((unsigned)((work + 255) / 256)), dim3(256), (size_t)0, c->stream, in_coors, n_in, (const int32_t*)nullptr, g,
               (const uint32_t*)ko.bitmap,
               (const uint32_t*)ko.word_prefix, (const int32_t*)perm_o, nbr_inv);
  }
  LAUNCH_CHECK(c);
  if (status_host) {
    int32_t bad = 0;
    if (nbr) {
      rc = read_back_i32(c, ki.flags, &bad);
      if (rc) return rc;
      *status_host |= bad ? 1 : 0;
    }
    if (nbr_inv) {
      rc = read_back_i32(c, ko.flags, &bad);
      if (rc) return rc;
      *status_host |= bad ? 2 : 0;
    }
    if (*status_host)
      return sstb_fail(c, SSTB_ERR_ARG, "spconv_table: coordinates outside batch_size / spatial shape (status %d)", *status_host);
  }
  return SSTB_OK;
}

extern "C" int sstb200_spconv_forward(sstb200_ctx* c, const float* feats, int c_in, const int32_t* nbr, int n_out, int kernel_volume,
                                      const float* weight, const void* weight_h16, int c_out, const float* scale, const float* shift,
                                      const float* residual, int relu, int precision, float* out) {
  CHECK_ARG(c, c && n_out >= 0 && c_in >= 1 && c_out >= 1 && kernel_volume >= 1);
  if (n_out == 0) return SSTB_OK;
  CHECK_ARG(c, feats && nbr && out);
  CHECK_ARG(c, ((uintptr_t)feats & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)residual & 15) == 0);
  if (precision == SSTB200_PREC_FP32) {
    CHECK_ARG(c, weight != nullptr);
    if ((c_in & 3) || (c_out & 3))
      return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "spconv_forward: channel counts must be multiples of 4 (got %d -> %d)", c_in, c_out);
    dim3 grid((n_out + SPF_BM - 1) / SPF_BM, (c_out + SPF_BN - 1) / SPF_BN);
    launch_pdl(spconv_gemm_f32_kernel, grid, dim3(256), (size_t)0, c->stream, feats, c_in, c_in, nbr, n_out, (const int32_t*)nullptr, kernel_volume,
               weight, c_out, scale, shift, residual, c_out, relu, out, c_out);
    LAUNCH_CHECK(c);
    return SSTB_OK;
  }
  CHECK_ARG(c, precision == SSTB200_PREC_BF16 || precision == SSTB200_PREC_FP32_TC);
  CHECK_ARG(c, weight_h16 != nullptr && ((uintptr_t)weight_h16 & 15) == 0);
  if ((c_in & 63) || (c_out & 63) || kernel_volume > SPU_MAX_KV)
    return sstb_fail(c, SSTB_ERR_UNSUPPORTED,
                     "spconv_forward: the tensor-core path needs c_in, c_out multiples of 64 and kernel volume <= %d (got %d -> %d, %d); "
                     "use precision fp32", SPU_MAX_KV, c_in, c_out, kernel_volume);
  SpArgs g;
  g.feats = feats, g.lda = c_in, g.Cin = c_in, g.nbr = nbr, g.n_out = n_out, g.n_dev = nullptr, g.KV = kernel_volume;
  g.Whi = (const __half*)weight_h16;
  g.Wlo = g.Whi + (size_t)kernel_volume * c_out * c_in;   // FP32_TC: the residue copy follows the hi copy
  g.Cout = c_out, g.scale = scale, g.shift = shift, g.residual = residual, g.ldr = c_out, g.act = relu ? 1 : 0, g.out = out, g.ldo = c_out;
  return dispatch_spconv_umma<false>(c, g, precision == SSTB200_PREC_FP32_TC, 0);
}

// fp32-tolerance row GEMM on the tensor core (used by the fp32 mode of the SRA encoder, csrc/sra_fp32.cu):
//   out[r, :N] = act(A[r, :K] . W[N, K]^T + bias) + res[r]      with every operand split into two fp16 numbers (see SPLIT above)
int sstb_gemm_rows_x3(sstb200_ctx* c, const float* A, int lda, const float* W, const float* bias, const float* res, int ldr, float* out,
                      int ldo, int M_cap, const int32_t* M_dev, int N, int K, int act) {
  if (M_cap <= 0) return SSTB_OK;
  if ((K & 63) || (N & 63) || (lda & 3) || (ldo & 3) || (ldr & 3) || (act == 1 && res)) return SSTB_ERR_UNSUPPORTED;
  __half* hi = arena_alloc<__half>(c, (size_t)N * K);
  __half* lo = arena_alloc<__half>(c, (size_t)N * K);
  if (!hi || !lo) return sstb_fail(c, SSTB_ERR_WORKSPACE, "gemm_rows_x3: arena too small");
  const size_t n = (size_t)N * K;
  launch_pdl(split_f16_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), (size_t)0, c->stream, W, n, hi, lo);
  SpArgs g;
  g.feats = A, g.lda = lda, g.Cin = K, g.nbr = nullptr, g.n_out = M_cap, g.n_dev = M_dev, g.KV = 1, g.Whi = hi, g.Wlo = lo, g.Cout = N;
  g.scale = nullptr, g.shift = bias, g.residual = res, g.ldr = ldr, g.act = act, g.out = out, g.ldo = ldo;
  return dispatch_spconv_umma<false>(c, g, true, 0);
}

extern "C" int sstb200_spconv_backward_weight(sstb200_ctx* c, const float* feats, int c_in, const int32_t* nbr, int n_out, int kernel_volume,
                                              const float* grad_out, int c_out, float* grad_weight) {
  CHECK_ARG(c, c && n_out >= 0 && c_in >= 1 && c_out >= 1 && kernel_volume >= 1 && grad_weight);
  CUDA_TRY(c, cudaMemsetAsync(grad_weight, 0, (size_t)kernel_volume * c_in * c_out * 4, c->stream));
  if (n_out == 0) return SSTB_OK;
  CHECK_ARG(c, feats && nbr && grad_out);
  CHECK_ARG(c, ((uintptr_t)feats & 15) == 0 && ((uintptr_t)grad_out & 15) == 0);
  if ((c_in & 3) || (c_out & 3))
    return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "spconv_backward_weight: channel counts must be multiples of 4 (got %d -> %d)", c_in, c_out);
  const int tiles = ((c_in + 63) / 64) * ((c_out + 63) / 64);
  if (kernel_volume > 65535 || tiles > 65535) return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "spconv_backward_weight: grid too large");
  dim3 grid((n_out + SPW_ROWS - 1) / SPW_ROWS, kernel_volume, tiles);
  launch_pdl(spconv_dw_kernel, grid, dim3(256), (size_t)0, c->stream, feats, c_in, nbr, n_out, kernel_volume, grad_out, c_out, grad_weight);
  LAUNCH_CHECK(c);
  return SSTB_OK;
}

// ------------------------------------------------------------------------------------------------------------------------------
// Device-count variants: row counts are read from device memory (n_*_dev), host ints are capacities only, nothing is read back,
// and every kernel loops grid-stride over the real rows with a grid sized from the SM count - so a sparse U-Net can be captured
// into one CUDA graph over capacity-sized buffers.  Same kernels, same tables, same summation order as the host-count entry points.
// ------------------------------------------------------------------------------------------------------------------------------
static unsigned sp_dev_grid(const sstb200_ctx* c, long long work, int per_sm) {
  long long g = (work + 255) / 256;
  if (g > (long long)c->num_sms * per_sm) g = (long long)c->num_sms * per_sm;
  return (unsigned)(g < 1 ? 1 : g);
}

extern "C" int sstb200_spconv_out_coors_dev(sstb200_ctx* c, const int32_t* in_coors, int n_in_cap, const int32_t* n_in_dev, int batch_size,
                                            const int32_t in_shape[3], const int32_t out_shape[3], const int32_t ksize[3],
                                            const int32_t stride[3], const int32_t padding[3], int32_t* out_coors, int out_cap,
                                            int32_t* num_out_dev) {
  CHECK_ARG(c, c && n_in_cap >= 0 && num_out_dev);
  SpGeom g;
  int rc = sp_geom(c, g, batch_size, in_shape, out_shape, ksize, stride, padding);
  if (rc) return rc;
  if (n_in_cap == 0) {
    CUDA_TRY(c, cudaMemsetAsync(num_out_dev, 0, 4, c->stream));
    return SSTB_OK;
  }
  CHECK_ARG(c, in_coors && n_in_dev && out_coors);
  long long per_in = 1, cells = batch_size;
  for (int d = 0; d < 3; d++) {
    per_in *= (g.ks[d] + g.st[d] - 1) / g.st[d];
    cells *= g.out_shape[d];
  }
  long long bound = (long long)n_in_cap * per_in;
  if (bound > cells) bound = cells;
  if ((long long)out_cap < bound)
    return sstb_fail(c, SSTB_ERR_ARG, "spconv_out_coors_dev: out_cap %d < worst case %lld rows", out_cap, bound);
  Extents e;
  long long T;
  rc = sp_extents(c, e, &T, batch_size, g.out_shape);
  if (rc) return rc;
  arena_reset(c);
  rc = arena_reserve(c, key_index_bytes(1, T) + 4096);
  if (rc) return rc;
  KeyIndex k;
  rc = key_index_alloc(c, k, 1, T);
  if (rc) return rc;
  launch_pdl(sp_mark_out_kernel, dim3(sp_dev_grid(c, (long long)n_in_cap * g.KV, 8)), dim3(256), (size_t)0, c->stream, in_coors, n_in_cap,
             n_in_dev, g, k.bitmap, k.flags);
  key_index_scan(c, k);
  launch_emit_rows<int32_t>(c, k, e, 0, out_coors, num_out_dev);
  LAUNCH_CHECK(c);
  return SSTB_OK;
}

extern "C" int sstb200_spconv_table_dev(sstb200_ctx* c, const int32_t* in_coors, int n_in_cap, const int32_t* n_in_dev,
                                        const int32_t* out_coors, int n_out_cap, const int32_t* n_out_dev, int batch_size,
                                        const int32_t in_shape[3], const int32_t out_shape[3], const int32_t ksize[3],
                                        const int32_t stride[3], const int32_t padding[3], int32_t* nbr, int32_t* nbr_inv) {
  CHECK_ARG(c, c && n_in_cap >= 0 && n_out_cap >= 0);
  SpGeom g;
  int rc = sp_geom(c, g, batch_size, in_shape, out_shape, ksize, stride, padding);
  if (rc) return rc;
  if (n_in_cap == 0 || n_out_cap == 0) return SSTB_OK;   // no row can exist: nothing to describe
  CHECK_ARG(c, in_coors && n_in_dev && out_coors && n_out_dev && (nbr || nbr_inv));
  Extents ei, eo;
  long long Ti, To;
  rc = sp_extents(c, ei, &Ti, batch_size, g.in_shape);
  if (rc) return rc;
  rc = sp_extents(c, eo, &To, batch_size, g.out_shape);
  if (rc) return rc;
  arena_reset(c);
  rc = arena_reserve(c, key_index_bytes(n_in_cap, Ti) + key_index_bytes(n_out_cap, To) + al256((size_t)n_in_cap * 4) +
                            al256((size_t)n_out_cap * 4) + 8192);
  if (rc) return rc;
  if (nbr) {
    KeyIndex ki;
    rc = key_index_alloc(c, ki, n_in_cap, Ti);
    if (rc) return rc;
    int32_t* perm_i = arena_alloc<int32_t>(c, n_in_cap);
    if (!perm_i) return sstb_fail(c, SSTB_ERR_WORKSPACE, "spconv_table_dev: arena too small");
    launch_mark_rows<int32_t>(c, in_coors, n_in_cap, ei, false, ki, n_in_dev);
    key_index_scan(c, ki);
    launch_pdl(sp_perm_kernel, dim3(sp_dev_grid(c, n_in_cap, 8)), dim3(256), (size_t)0, c->stream, (const long long*)ki.keys, n_in_cap, n_in_dev,
               (const uint32_t*)ki.bitmap, (const uint32_t*)ki.word_prefix, perm_i);
    launch_pdl(sp_nbr_kernel, dim3(sp_dev_grid(c, (long long)n_out_cap * g.KV, 8)), dim3(256), (size_t)0, c->stream, out_coors, n_out_cap,
               n_out_dev, g, (const uint32_t*)ki.bitmap, (const uint32_t*)ki.word_prefix, (const int32_t*)perm_i, nbr);
  }
  if (nbr_inv) {
    KeyIndex ko;
    rc = key_index_alloc(c, ko, n_out_cap, To);
    if (rc) return rc;
    int32_t* perm_o = arena_alloc<int32_t>(c, n_out_cap);
    if (!perm_o) return sstb_fail(c, SSTB_ERR_WORKSPACE, "spconv_table_dev: arena too small");
    launch_mark_rows<int32_t>(c, out_coors, n_out_cap, eo, false, ko, n_out_dev);
    key_index_scan(c, ko);
    launch_pdl(sp_perm_kernel, dim3(sp_dev_grid(c, n_out_cap, 8)), dim3(256), (size_t)0, c->stream, (const long long*)ko.keys, n_out_cap,
               n_out_dev, (const uint32_t*)ko.bitmap, (const uint32_t*)ko.word_prefix, perm_o);
    launch_pdl(sp_nbr_inv_kernel, dim3(sp_dev_grid(c, (long long)n_in_cap * g.KV, 8)), dim3(256), (size_t)0, c->stream, in_coors, n_in_cap,
               n_in_dev, g, (const uint32_t*)ko.bitmap, (const uint32_t*)ko.word_prefix, (const int32_t*)perm_o, nbr_inv);
  }
  LAUNCH_CHECK(c);
  return SSTB_OK;
}

extern "C" int sstb200_spconv_forward_dev(sstb200_ctx* c, const float* feats, int lda, int c_in, const int32_t* nbr, int n_out_cap,
                                          const int32_t* n_out_dev, int kernel_volume, const float* weight, const void* weight_h16, int c_out,
                                          const float* scale, const float* shift, const float* residual, int ldr, int relu, int precision,
                                          float* out, int ldo) {
  CHECK_ARG(c, c && n_out_cap >= 0 && c_in >= 1 && c_out >= 1 && kernel_volume >= 1);
  if (n_out_cap == 0) return SSTB_OK;
  CHECK_ARG(c, feats && nbr && n_out_dev && out && lda >= c_in && ldo >= c_out && (!residual || ldr >= c_out));
  CHECK_ARG(c, ((uintptr_t)feats & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)residual & 15) == 0);
  CHECK_ARG(c, (lda & 3) == 0 && (ldo & 3) == 0 && (!residual || (ldr & 3) == 0));
  if (precision == SSTB200_PREC_FP32) {
    CHECK_ARG(c, weight != nullptr);
    if ((c_in & 3) || (c_out & 3))
      return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "spconv_forward_dev: channel counts must be multiples of 4 (got %d -> %d)", c_in, c_out);
    // up to 32 CTAs per SM (~300k rows at one tile each, like the host-count launch's dynamic scheduling); beyond that CTAs loop
    int tiles = (n_out_cap + SPF_BM - 1) / SPF_BM;
    if (tiles > c->num_sms * 32) tiles = c->num_sms * 32;
    dim3 grid(tiles, (c_out + SPF_BN - 1) / SPF_BN);
    launch_pdl(spconv_gemm_f32_kernel, grid, dim3(256), (size_t)0, c->stream, feats, lda, c_in, nbr, n_out_cap, n_out_dev, kernel_volume, weight,
               c_out, scale, shift, residual, ldr, relu, out, ldo);
    LAUNCH_CHECK(c);
    return SSTB_OK;
  }
  CHECK_ARG(c, precision == SSTB200_PREC_BF16 || precision == SSTB200_PREC_FP32_TC);
  CHECK_ARG(c, weight_h16 != nullptr && ((uintptr_t)weight_h16 & 15) == 0);
  if ((c_in & 63) || (c_out & 63) || kernel_volume > SPU_MAX_KV)
    return sstb_fail(c, SSTB_ERR_UNSUPPORTED,
                     "spconv_forward_dev: the tensor-core path needs c_in, c_out multiples of 64 and kernel volume <= %d (got %d -> %d, %d); "
                     "use precision fp32", SPU_MAX_KV, c_in, c_out, kernel_volume);
  SpArgs g;
  g.feats = feats, g.lda = lda, g.Cin = c_in, g.nbr = nbr, g.n_out = n_out_cap, g.n_dev = n_out_dev, g.KV = kernel_volume;
  g.Whi = (const __half*)weight_h16;
  g.Wlo = g.Whi + (size_t)kernel_volume * c_out * c_in;
  g.Cout = c_out, g.scale = scale, g.shift = shift, g.residual = residual, g.ldr = residual ? ldr : c_out, g.act = relu ? 1 : 0;
  g.out = out, g.ldo = ldo;
  return dispatch_spconv_umma<true>(c, g, precision == SSTB200_PREC_FP32_TC, c->num_sms * 4);
}

// SparseUNet.decoder_layer_forward's glue: out[o, j] = x_merge[o, j] + sum_g cat[o, j * r + g]  (r = cat_channels / channels).
// reduce_channel's view(n, C, r).sum(2) first, then the add - the order torch evaluates it in (for r = 2, the reference's
// configurations, the group sum is one rounding and the result is bit-identical to the torch expression).
__global__ void spconv_merge_kernel(const float* __restrict__ x_merge, const float* __restrict__ cat, int C, int r, int n_cap,
                                    const int32_t* __restrict__ n_dev, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int n = min(n_cap, *n_dev);
  const long long work = (long long)n * C;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < work; t += (long long)gridDim.x * blockDim.x) {
    const float* grp = cat + (size_t)t * r;   // row o = t / C starts at o * C * r, group j = t % C at j * r: together t * r
    float s = grp[0];
    for (int q = 1; q < r; q++) s += grp[q];
    out[t] = x_merge[t] + s;
  }
}

extern "C" int sstb200_spconv_decoder_merge(sstb200_ctx* c, const float* x_merge, const float* cat, int channels, int cat_channels,
                                            int n_cap, const int32_t* n_dev, float* out) {
  CHECK_ARG(c, c && n_cap >= 0 && channels >= 1 && cat_channels >= channels && cat_channels % channels == 0);
  if (n_cap == 0) return SSTB_OK;
  CHECK_ARG(c, x_merge && cat && n_dev && out);
  launch_pdl(spconv_merge_kernel, dim3(sp_dev_grid(c, (long long)n_cap * channels, 8)), dim3(256), (size_t)0, c->stream, x_merge, cat, channels,
             cat_channels / channels, n_cap, n_dev, out);
  LAUNCH_CHECK(c);
  return SSTB_OK;
}
