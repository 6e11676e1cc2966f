// Bitmap-rank index ("unique rows, sorted" without a sort), CSR grouping and segmented reduce.
// Shared by voxel.cu / window.cu / vfe.cu / sir.cu.  See DESIGN.md "voxel index".
#pragma once
#include "common.cuh"

// ------------------------------------------------------------------------------------------------
struct Extents {
  int ndim;
  long long lo[4];
  long long ext[4];
};

struct KeyIndex {
  long long* keys;        // [P]  linear key or -1
  uint32_t* bitmap;       // [nwords]
  uint32_t* word_prefix;  // [nwords+1]
  uint32_t* total;        // distinct keys (device)
  int32_t* flags;         // [0] has_invalid
  ScanTemps st;
  size_t nwords;
  long long T;
};

static size_t key_index_bytes(size_t P, long long T) {
  size_t nwords = (size_t)((T + 31) / 32);
  return al256(P * 8) + al256(nwords * 4) + al256((nwords + 1) * 4) + scan_temps_bytes(nwords) + 1024;
}

static int key_index_alloc(sstb200_ctx* c, KeyIndex& k, size_t P, long long T) {
  k.T = T;
  k.nwords = (size_t)((T + 31) / 32);
  k.keys = arena_alloc<long long>(c, P ? P : 1);
  // bitmap and scan temporaries are adjacent: ONE memset clears both
  size_t bm_bytes = al256(k.nwords * 4), st_bytes = scan_temps_bytes(k.nwords);
  uint8_t* z = arena_alloc<uint8_t>(c, bm_bytes + st_bytes);
  k.word_prefix = arena_alloc<uint32_t>(c, k.nwords + 1);
  if (!k.keys || !z || !k.word_prefix) return sstb_fail(c, SSTB_ERR_WORKSPACE, "key index: arena too small");
  k.bitmap = (uint32_t*)z;
  k.st.ticket = (uint32_t*)(z + bm_bytes);
  k.st.state = (unsigned long long*)(k.st.ticket + 64);
  k.total = k.st.ticket + 1;
  k.flags = (int32_t*)(k.st.ticket + 2);
  CUDA_TRY(c, cudaMemsetAsync(z, 0, bm_bytes + st_bytes, c->stream));
  return SSTB_OK;
}

static void key_index_scan(sstb200_ctx* c, KeyIndex& k) {
  launch_exclusive_scan(c->stream, LoadPopc{k.bitmap}, k.nwords, nullptr, k.st, k.word_prefix, k.total, true);
}

// Set one bit; most points fall into an already-marked cell, so test (L2 read, never L1: the bitmap is written by atomics
// of other SMs) before paying for the atomic.
__device__ __forceinline__ void bitmap_set(uint32_t* __restrict__ bitmap, long long key) {
  uint32_t* w = bitmap + (key >> 5);
  uint32_t bit = 1u << (key & 31);
  if ((__ldcg(w) & bit) == 0) atomicOr(w, bit);
}

// merge a block-private bitmap into the global one (skip words that are empty or already fully present)
__device__ __forceinline__ void bitmap_merge(const uint32_t* sbm, uint32_t* __restrict__ bitmap, uint32_t nwords) {
  __syncthreads();
  for (uint32_t w = threadIdx.x; w < nwords; w += blockDim.x) {
    const uint32_t v = sbm[w];
    if (v && (__ldcg(&bitmap[w]) & v) != v) atomicOr(&bitmap[w], v);
  }
}

// ---- mark kernels --------------------------------------------------------------------------------
// SM = true: each (large) block first ORs into a private shared-memory copy of the bitmap and then merges its non-zero words into
// the global one.  Same-address global atomics serialise (~10 ns each, measured): a dense LiDAR ring puts > 1000 points into one
// bitmap word, which made the plain kernel 4x slower than its traffic; privatised, a word sees at most one atomic per block.
template <typename TI, bool SM>
__global__ void __launch_bounds__(SM ? 1024 : 256) mark_rows_kernel(const TI* __restrict__ rows, int n, Extents e, bool negative_is_invalid,
                                 long long* __restrict__ keys, uint32_t* __restrict__ bitmap,
                                 int32_t* __restrict__ flags, const int32_t* __restrict__ n_dev, uint32_t nwords) {
  pdl_wait();
  pdl_launch();
  extern __shared__ uint32_t mark_sbm[];
  if (n_dev) n = *n_dev;
  if (SM) {
    for (uint32_t w = threadIdx.x; w < nwords; w += blockDim.x) mark_sbm[w] = 0u;
    __syncthreads();
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    long long key = 0;
    bool bad = false, neg = false;
#pragma unroll 4
    for (int d = 0; d < e.ndim; d++) {
      long long v = (long long)rows[(size_t)i * e.ndim + d];
      if (negative_is_invalid && v < 0) neg = true;
      long long r = v - e.lo[d];
      if (r < 0 || r >= e.ext[d]) bad = true;
      key = key * e.ext[d] + r;
    }
    if (bad || neg) {
      keys[i] = -1;
      flags[0] = 1;
      if (!neg) flags[1] = 1;  // a row outside the caller's bounds (not a "negative = invalid" row): the bounds were wrong
      continue;
    }
    keys[i] = key;
    if (SM) atomicOr(&mark_sbm[key >> 5], 1u << (key & 31));
    else bitmap_set(bitmap, key);
  }
  if (SM) bitmap_merge(mark_sbm, bitmap, nwords);
}
#define MARK_SMEM_MAX_WORDS (24 * 1024)  // 96 KB of shared memory
template <typename TI>
static void launch_mark_rows(sstb200_ctx* c, const TI* rows, int n, const Extents& e, bool negative_is_invalid, KeyIndex& k,
                             const int32_t* n_dev) {
  if (k.nwords <= MARK_SMEM_MAX_WORDS) {
    static SmemAttr sa;
    size_t smem = k.nwords * 4;
    if (smem > 48 * 1024) ensure_smem(c, sa, mark_rows_kernel<TI, true>, (size_t)MARK_SMEM_MAX_WORDS * 4);
    int grid = (n + 1023) / 1024;
    if (grid > c->num_sms) grid = c->num_sms;
    if (grid < 1) grid = 1;
    launch_pdl(mark_rows_kernel<TI, true>, dim3(grid), dim3(1024), smem, c->stream, rows, n, e, negative_is_invalid, k.keys, k.bitmap, k.flags,
               n_dev, (uint32_t)k.nwords);
  } else {
    int grid = (n + 255) / 256;
    if (n_dev && grid > c->num_sms * 8) grid = c->num_sms * 8;   // n is a capacity: the grid-stride loop covers the real rows
    if (grid < 1) grid = 1;
    launch_pdl(mark_rows_kernel<TI, false>, dim3(grid), dim3(256), (size_t)0, c->stream, rows, n, e, negative_is_invalid, k.keys,
               k.bitmap, k.flags, n_dev, 0u);
  }
}

// ---- emit unique rows (decode keys of set bits) ----------------------------------------------------
// One thread per bitmap word; SMALL = the whole key space fits 31 bits (32-bit divisions instead of 64-bit ones).
template <typename TO, bool SMALL>
__global__ void __launch_bounds__(64) emit_rows_kernel(const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ word_prefix,
                                 size_t nwords, Extents e, int shift_if_no_invalid, const int32_t* __restrict__ flags,
                                 TO* __restrict__ out_rows, const uint32_t* __restrict__ total, int32_t* __restrict__ num_out) {
  pdl_wait();
  pdl_launch();
  int shift = (shift_if_no_invalid && flags[0] == 0) ? 1 : 0;
  // four threads per bitmap word (one byte each): the serial decode loop is at most 8 cells long
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t == 0) {
    int tot = (int)(*total) - shift;
    *num_out = tot < 0 ? 0 : tot;
  }
  for (; t < nwords * 4; t += (size_t)gridDim.x * blockDim.x) {
    const size_t w = t >> 2;
    const int part = (int)(t & 3);
    const uint32_t word = bitmap[w];
    uint32_t bits = (word >> (8 * part)) & 0xFFu;
    if (!bits) continue;
    long long v = (long long)word_prefix[w] + __popc(word & ((1u << (8 * part)) - 1u)) - shift;
    while (bits) {
      int b = __ffs(bits) - 1 + 8 * part;
      bits &= bits - 1;
      if (v >= 0) {
        TO c[4];
        if (SMALL) {
          uint32_t key = (uint32_t)w * 32u + (uint32_t)b;
#pragma unroll 4
          for (int d = e.ndim - 1; d >= 0; d--) {
            uint32_t ext = (uint32_t)e.ext[d], q = key / ext;
            c[d] = (TO)((long long)(key - q * ext) + e.lo[d]);
            key = q;
          }
        } else {
          long long key = (long long)w * 32 + b;
#pragma unroll 4
          for (int d = e.ndim - 1; d >= 0; d--) {
            long long q = key / e.ext[d];
            c[d] = (TO)(key - q * e.ext[d] + e.lo[d]);
            key = q;
          }
        }
        for (int d = 0; d < e.ndim; d++) out_rows[(size_t)v * e.ndim + d] = c[d];
      }
      v++;
    }
  }
}
template <typename TO>
static void launch_emit_rows(sstb200_ctx* c, const KeyIndex& k, const Extents& e, int shift_if_no_invalid, TO* out_rows,
                             int32_t* num_out) {
  size_t eg = (k.nwords * 4 + 63) / 64;
  if (eg > (size_t)c->num_sms * 32) eg = (size_t)c->num_sms * 32;
  if (eg == 0) eg = 1;
  if (k.T < ((long long)1 << 31))
    launch_pdl(emit_rows_kernel<TO, true>, dim3((unsigned)eg), dim3(64), (size_t)(0), c->stream, (const uint32_t*)k.bitmap, (const uint32_t*)k.word_prefix, k.nwords, e, shift_if_no_invalid, (const int32_t*)k.flags, out_rows, (const uint32_t*)k.total, num_out);
  else
    launch_pdl(emit_rows_kernel<TO, false>, dim3((unsigned)eg), dim3(64), (size_t)(0), c->stream, (const uint32_t*)k.bitmap, (const uint32_t*)k.word_prefix, k.nwords, e, shift_if_no_invalid, (const int32_t*)k.flags, out_rows, (const uint32_t*)k.total, num_out);
}

// ---- map + count -------------------------------------------------------------------------------------
template <typename TM>
__global__ void map_count_kernel(const long long* __restrict__ keys, int n, const uint32_t* __restrict__ bitmap,
                                 const uint32_t* __restrict__ word_prefix, int shift_if_no_invalid,
                                 const int32_t* __restrict__ flags, TM* __restrict__ map, int32_t* __restrict__ count,
                                 const int32_t* __restrict__ n_dev = nullptr) {
  pdl_wait();
  pdl_launch();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (n_dev) n = *n_dev;
  if (i >= n) return;
  int shift = (shift_if_no_invalid && flags[0] == 0) ? 1 : 0;
  long long key = keys[i];
  long long v = -1;
  if (key >= 0) {
    size_t w = (size_t)(key >> 5);
    v = (long long)word_prefix[w] + __popc(bitmap[w] & ((1u << (key & 31)) - 1u)) - shift;
  }
  map[i] = (TM)v;
  if (v >= 0 && count) atomicAdd(&count[v], 1);
}

// ---- CSR fill (counting sort, order inside a segment unspecified) -----------------------------------------
template <typename TM>
__global__ void csr_fill_kernel(const TM* __restrict__ map, int n, const uint32_t* __restrict__ offsets,
                                int32_t* __restrict__ cursor, int32_t* __restrict__ order,
                                const int32_t* __restrict__ n_dev = nullptr) {
  pdl_wait();
  pdl_launch();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (n_dev) n = *n_dev;
  if (i >= n) return;
  long long v = (long long)map[i];
  if (v < 0) return;
  int pos = atomicAdd(&cursor[v], 1);
  order[offsets[v] + pos] = i;
}

// ---- few-segment variants (e.g. FSD instance groups: 150k points in ~256 groups) ----------------------------------------
// Direct atomics would serialise on a handful of addresses; here every block first ranks its CSR_SMALL_ITEMS points in
// shared memory and touches each global counter once.
#define CSR_SMALL_MAX 4096
#define CSR_SMALL_ITEMS 4096
template <typename TM>
__global__ void __launch_bounds__(1024) count_small_kernel(const TM* __restrict__ map, int n, int nseg, int32_t* __restrict__ count,
                                                           int32_t* __restrict__ err) {
  pdl_wait();
  pdl_launch();
  extern __shared__ int sh_cnt[];
  for (int s = threadIdx.x; s < nseg; s += blockDim.x) sh_cnt[s] = 0;
  __syncthreads();
  const int base = blockIdx.x * CSR_SMALL_ITEMS;
  for (int i = base + threadIdx.x; i < min(base + CSR_SMALL_ITEMS, n); i += blockDim.x) {
    long long v = (long long)map[i];
    if (v < 0 || v >= nseg) *err = 1;
    else atomicAdd(&sh_cnt[v], 1);
  }
  __syncthreads();
  for (int s = threadIdx.x; s < nseg; s += blockDim.x)
    if (sh_cnt[s]) atomicAdd(&count[s], sh_cnt[s]);
}
template <typename TM>
__global__ void __launch_bounds__(1024) csr_fill_small_kernel(const TM* __restrict__ map, int n, int nseg, const uint32_t* __restrict__ offsets,
                                                              int32_t* __restrict__ cursor, int32_t* __restrict__ order) {
  pdl_wait();
  pdl_launch();
  extern __shared__ int sh_cnt[];  // [nseg] counts, then [nseg] bases
  int* sh_base = sh_cnt + nseg;
  for (int s = threadIdx.x; s < nseg; s += blockDim.x) sh_cnt[s] = 0;
  __syncthreads();
  const int base = blockIdx.x * CSR_SMALL_ITEMS;
  int rank[CSR_SMALL_ITEMS / 1024];
#pragma unroll
  for (int k = 0; k < CSR_SMALL_ITEMS / 1024; k++) {
    int i = base + k * 1024 + threadIdx.x;
    rank[k] = -1;
    if (i < n) {
      long long v = (long long)map[i];
      if (v >= 0 && v < nseg) rank[k] = atomicAdd(&sh_cnt[v], 1);
    }
  }
  __syncthreads();
  for (int s = threadIdx.x; s < nseg; s += blockDim.x) sh_base[s] = sh_cnt[s] ? (int)offsets[s] + atomicAdd(&cursor[s], sh_cnt[s]) : 0;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < CSR_SMALL_ITEMS / 1024; k++) {
    int i = base + k * 1024 + threadIdx.x;
    if (rank[k] >= 0) order[sh_base[(long long)map[i]] + rank[k]] = i;
  }
}

// ---- segmented reduce: GROUP lanes cooperate on one segment, lanes stride the channels --------------------
template <int GROUP>
__global__ void __launch_bounds__(256) segment_reduce_kernel(const float* __restrict__ src, int C,
                                                             const uint32_t* __restrict__ offsets,
                                                             const int32_t* __restrict__ order, int nseg_host,
                                                             const int32_t* __restrict__ nseg_dev, int mode,
                                                             float empty_value, float* __restrict__ out,
                                                             long long* __restrict__ argmax, int n_rows) {
  pdl_wait();
  pdl_launch();
  int nseg = nseg_dev ? *nseg_dev : nseg_host;
  int groups_per_block = blockDim.x / GROUP;
  int g = threadIdx.x / GROUP, l = threadIdx.x % GROUP;
  for (int s = blockIdx.x * groups_per_block + g; s < nseg; s += gridDim.x * groups_per_block) {
    uint32_t b = offsets[s], e = offsets[s + 1];
    for (int c = l; c < C; c += GROUP) {
      if (mode == SSTB200_REDUCE_MAX) {
        float m = -INFINITY;
        long long am = n_rows;
        for (uint32_t k = b; k < e; k++) {
          int p = order[k];
          float v = src[(size_t)p * C + c];
          if (v > m || (v == m && p < am)) {
            m = v;
            am = p;
          }
        }
        if (b == e) m = empty_value;
        out[(size_t)s * C + c] = m;
        if (argmax) argmax[(size_t)s * C + c] = am;
      } else {
        // fp64 accumulation: exact for these magnitudes, so the result does not depend on CSR order
        double acc = 0.0;
        for (uint32_t k = b; k < e; k++) acc += (double)src[(size_t)order[k] * C + c];
        float r = (float)acc;
        if (mode == SSTB200_REDUCE_MEAN && e > b) r = (float)acc / (float)(e - b);
        out[(size_t)s * C + c] = r;
      }
    }
  }
}

// Vector variant (C % 4 == 0, 16-B aligned rows): GROUP lanes own one segment, each lane owns float4 channel groups
// lane, lane+GROUP, ... (NV4 of them, C = 4*GROUP*NV4 at most), and FOUR points are in flight per lane (independent index and row
// loads) - a 128-channel row is one 512-B warp transaction.  Same arithmetic as the scalar kernel (max with lowest-index tie
// break for argmax; sum/mean in fp64, so independent of the CSR order).
template <int GROUP, int NV4, bool ARG>
__global__ void __launch_bounds__(256) segment_reduce_v4_kernel(const float* __restrict__ src, int C,
                                                                const uint32_t* __restrict__ offsets,
                                                                const int32_t* __restrict__ order, int nseg_host,
                                                                const int32_t* __restrict__ nseg_dev, int mode,
                                                                float empty_value, float* __restrict__ out,
                                                                long long* __restrict__ argmax, int n_rows) {
  pdl_wait();
  pdl_launch();
  constexpr int RIF = NV4 == 1 ? 8 : 4;  // rows in flight per lane (independent 16-byte loads)
  const int nseg = nseg_dev ? *nseg_dev : nseg_host;
  const int groups_per_block = blockDim.x / GROUP;
  const int g = threadIdx.x / GROUP, l = threadIdx.x % GROUP;
  const int C4 = C >> 2;
  const float4* __restrict__ src4 = reinterpret_cast<const float4*>(src);
  // lanes of a group always run the same trip counts, but different groups of a warp do not: shuffles are group-masked
  const unsigned gmask = GROUP == 32 ? 0xffffffffu : (((1u << GROUP) - 1u) << ((threadIdx.x & 31) / GROUP * GROUP));
  const float fill = mode == SSTB200_REDUCE_MAX ? -INFINITY : 0.f;  // value of a row slot past the end of the segment
  for (int s = blockIdx.x * groups_per_block + g; s < nseg; s += gridDim.x * groups_per_block) {
    const uint32_t b = offsets[s], e = offsets[s + 1];
    float4 m[NV4];
    int am[NV4][4];
    double acc[NV4][4];
#pragma unroll
    for (int j = 0; j < NV4; j++) {
      m[j] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      am[j][0] = am[j][1] = am[j][2] = am[j][3] = n_rows;
      acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.0;
    }
    // the point ids of GROUP rows are fetched by ONE coalesced load and handed round by shuffles, so a long segment is a
    // stream of independent row loads (RIF in flight) instead of a chain of index-load -> row-load round trips
    for (uint32_t k0 = b; k0 < e; k0 += GROUP) {
      const int mine = (k0 + l < e) ? order[k0 + l] : -1;
      const int cnt = min((int)(e - k0), GROUP);
      for (int r0 = 0; r0 < cnt; r0 += RIF) {
        int p[RIF];
        float4 v[RIF][NV4];
#pragma unroll
        for (int u = 0; u < RIF; u++) {
          p[u] = __shfl_sync(gmask, mine, (r0 + u) % GROUP, GROUP);
          if (r0 + u >= cnt) p[u] = -1;
        }
#pragma unroll
        for (int u = 0; u < RIF; u++)
#pragma unroll
          for (int j = 0; j < NV4; j++)
            v[u][j] = (p[u] >= 0 && l + j * GROUP < C4) ? __ldg(&src4[(size_t)p[u] * C4 + l + j * GROUP]) : make_float4(fill, fill, fill, fill);
        if (mode == SSTB200_REDUCE_MAX && !ARG) {
          // plain max: absent rows were loaded as -inf, one FMNMX per element
#pragma unroll
          for (int u = 0; u < RIF; u++)
#pragma unroll
            for (int j = 0; j < NV4; j++) {
              m[j].x = fmaxf(m[j].x, v[u][j].x);
              m[j].y = fmaxf(m[j].y, v[u][j].y);
              m[j].z = fmaxf(m[j].z, v[u][j].z);
              m[j].w = fmaxf(m[j].w, v[u][j].w);
            }
        } else if (mode == SSTB200_REDUCE_MAX) {
#pragma unroll
          for (int u = 0; u < RIF; u++) {
            if (p[u] < 0) continue;
#pragma unroll
            for (int j = 0; j < NV4; j++) {
              const float x[4] = {v[u][j].x, v[u][j].y, v[u][j].z, v[u][j].w};
              float* mm = &m[j].x;
#pragma unroll
              for (int q = 0; q < 4; q++)
                if (x[q] > mm[q] || (x[q] == mm[q] && p[u] < am[j][q])) {
                  mm[q] = x[q];
                  am[j][q] = p[u];
                }
            }
          }
        } else {
          // fp64 accumulation: exact for these magnitudes, so the result does not depend on the CSR order
#pragma unroll
          for (int u = 0; u < RIF; u++)
#pragma unroll
            for (int j = 0; j < NV4; j++) {
              acc[j][0] += (double)v[u][j].x;
              acc[j][1] += (double)v[u][j].y;
              acc[j][2] += (double)v[u][j].z;
              acc[j][3] += (double)v[u][j].w;
            }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < NV4; j++) {
      const int c4 = l + j * GROUP;
      if (c4 >= C4) continue;
      if (mode == SSTB200_REDUCE_MAX) {
        if (b == e) m[j] = make_float4(empty_value, empty_value, empty_value, empty_value);
        reinterpret_cast<float4*>(out)[(size_t)s * C4 + c4] = m[j];
        if (ARG) {
          longlong2* a2 = reinterpret_cast<longlong2*>(argmax + (size_t)s * C + 4 * c4);
          a2[0] = make_longlong2(am[j][0], am[j][1]);
          a2[1] = make_longlong2(am[j][2], am[j][3]);
        }
      } else {
        float r[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
          r[q] = (float)acc[j][q];
          if (mode == SSTB200_REDUCE_MEAN && e > b) r[q] = (float)acc[j][q] / (float)(e - b);
        }
        reinterpret_cast<float4*>(out)[(size_t)s * C4 + c4] = make_float4(r[0], r[1], r[2], r[3]);
      }
    }
  }
}

static void launch_segment_reduce(sstb200_ctx* c, const float* src, int C, const uint32_t* offsets,
                                  const int32_t* order, int nseg_cap, const int32_t* nseg_dev, int mode,
                                  float empty_value, float* out, long long* argmax, int n_rows) {
  int grid = c->num_sms * 8;
  const bool vec = (C % 4 == 0) && C <= 256 && (((uintptr_t)src | (uintptr_t)out | (uintptr_t)argmax) & 15) == 0;
#define SEGV4(G, NV)                                                                                                                     \
  do {                                                                                                                                  \
    if (argmax)                                                                                                                         \
      launch_pdl(segment_reduce_v4_kernel<G, NV, true>, dim3(grid), dim3(256), (size_t)(0), c->stream, src, C, offsets, order, nseg_cap, \
                 nseg_dev, mode, empty_value, out, argmax, n_rows);                                                                     \
    else                                                                                                                                \
      launch_pdl(segment_reduce_v4_kernel<G, NV, false>, dim3(grid), dim3(256), (size_t)(0), c->stream, src, C, offsets, order, nseg_cap, \
                 nseg_dev, mode, empty_value, out, argmax, n_rows);                                                                     \
  } while (0)
  if (vec) {
    int c4 = C / 4;
    if (c4 > 32) SEGV4(32, 2);
    else if (c4 > 16) SEGV4(32, 1);
    else if (c4 > 8) SEGV4(16, 1);
    else if (c4 > 4) SEGV4(8, 1);
    else if (c4 > 2) SEGV4(4, 1);
    else if (c4 > 1) SEGV4(2, 1);
    else SEGV4(1, 1);
    return;
  }
#undef SEGV4
  if (C >= 32)
    launch_pdl(segment_reduce_kernel<32>, dim3(grid), dim3(256), (size_t)(0), c->stream, src, C, offsets, order, nseg_cap, nseg_dev, mode, empty_value, out, argmax, n_rows);
  else if (C > 4)
    launch_pdl(segment_reduce_kernel<8>, dim3(grid), dim3(256), (size_t)(0), c->stream, src, C, offsets, order, nseg_cap, nseg_dev, mode, empty_value, out, argmax, n_rows);
  else
    launch_pdl(segment_reduce_kernel<4>, dim3(grid), dim3(256), (size_t)(0), c->stream, src, C, offsets, order, nseg_cap, nseg_dev, mode, empty_value, out, argmax, n_rows);
}

// CSR over a map -> (offsets[nseg+1], order[n]) ; count must already hold per-segment counts.
struct Csr {
  uint32_t* offsets = nullptr;  // preset = caller-owned
  int32_t* order = nullptr;     // preset = caller-owned
  int32_t* cursor;
  ScanTemps st;
  uint32_t* total;
};
static size_t csr_bytes(size_t n, size_t nseg_cap) {
  return al256((nseg_cap + 2) * 4) * 2 + al256(n * 4 + 4) + scan_temps_bytes(nseg_cap) + 2048;
}
template <typename TM>
static int csr_build(sstb200_ctx* c, Csr& r, const TM* map, int n, const int32_t* count, size_t nseg_cap,
                     const int32_t* nseg_dev, const int32_t* n_dev = nullptr, int small_nseg = 0) {
  if (!r.offsets) r.offsets = arena_alloc<uint32_t>(c, nseg_cap + 2);  // preset = caller-owned [nseg_cap + 1]
  // cursor and scan temporaries are adjacent: ONE memset clears both
  size_t cur_bytes = al256((nseg_cap + 2) * 4), st_bytes = scan_temps_bytes(nseg_cap);
  uint8_t* z = arena_alloc<uint8_t>(c, cur_bytes + st_bytes);
  if (!r.order) r.order = arena_alloc<int32_t>(c, n + 1);
  if (!r.offsets || !z || !r.order) return sstb_fail(c, SSTB_ERR_WORKSPACE, "csr: arena too small");
  r.cursor = (int32_t*)z;
  r.st.ticket = (uint32_t*)(z + cur_bytes);
  r.st.state = (unsigned long long*)(r.st.ticket + 64);
  r.total = r.st.ticket + 1;
  CUDA_TRY(c, cudaMemsetAsync(z, 0, cur_bytes + st_bytes, c->stream));
  launch_exclusive_scan(c->stream, LoadU32{(const uint32_t*)count}, nseg_cap, nseg_dev, r.st, r.offsets, r.total, true);
  if (n > 0 && small_nseg > 0 && small_nseg <= CSR_SMALL_MAX && !n_dev)
    launch_pdl(csr_fill_small_kernel<TM>, dim3((n + CSR_SMALL_ITEMS - 1) / CSR_SMALL_ITEMS), dim3(1024), (size_t)small_nseg * 8, c->stream, map, n, small_nseg,
               (const uint32_t*)r.offsets, r.cursor, r.order);
  else if (n > 0)
    launch_pdl(csr_fill_kernel<TM>, dim3((n + 255) / 256), dim3(256), (size_t)(0), c->stream, map, n, r.offsets, r.cursor, r.order, n_dev);
  LAUNCH_CHECK(c);
  return SSTB_OK;
}


static int read_back_i32(sstb200_ctx* c, const int32_t* dev, int32_t* host) {
  CUDA_TRY(c, cudaMemcpyAsync(c->pinned_i32, dev, 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  *host = c->pinned_i32[0];
  return SSTB_OK;
}

static int make_extents(sstb200_ctx* c, Extents& e, int ndim, const long long* lo, const long long* hi, long long* T) {
  e.ndim = ndim;
  long long t = 1;
  for (int d = 0; d < 4; d++) {
    e.lo[d] = 0;
    e.ext[d] = 1;
  }
  for (int d = 0; d < ndim; d++) {
    if (hi[d] < lo[d]) return sstb_fail(c, SSTB_ERR_ARG, "extent %d: hi < lo", d);
    e.lo[d] = lo[d];
    e.ext[d] = hi[d] - lo[d] + 1;
    if (t > ((long long)1 << 40) / e.ext[d]) return sstb_fail(c, SSTB_ERR_UNSUPPORTED, "bounding grid too large");
    t *= e.ext[d];
  }
  if (t > ((long long)1 << 34))
    return sstb_fail(c, SSTB_ERR_UNSUPPORTED,
                     "bounding grid of %lld cells exceeds the bitmap-rank limit (2^34); sort fallback not built yet", t);
  *T = t;
  return SSTB_OK;
}


// One warp per segment: rank(i) = #{j in segment : idx_j < idx_i}.  Segments on this path are windows
// (<= a few hundred tokens); cost O(n^2/32) per warp.
static __global__ void __launch_bounds__(256) stable_rank_kernel(const uint32_t* __restrict__ offsets, const int32_t* __restrict__ order,
                                                          const int32_t* __restrict__ nseg_dev, int32_t* __restrict__ sorted_order,
                                                          long long* __restrict__ rank_out_i64, int32_t* __restrict__ rank_out_i32,
                                                          int32_t* __restrict__ slot_out) {
  pdl_wait();
  pdl_launch();
  int nseg = *nseg_dev;
  int warps = (gridDim.x * blockDim.x) >> 5;
  int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  for (int s = w; s < nseg; s += warps) {
    uint32_t b = offsets[s], e = offsets[s + 1];
    uint32_t n = e - b;
    for (uint32_t i = lane_id(); i < n; i += 32) {
      int me = order[b + i];
      int r = 0;
      for (uint32_t j = 0; j < n; j++) r += (order[b + j] < me);
      if (sorted_order) sorted_order[b + r] = me;
      if (rank_out_i64) rank_out_i64[me] = r;
      if (rank_out_i32) rank_out_i32[me] = r;
      if (slot_out) slot_out[me] = (int32_t)(b + r);
    }
  }
}


static __global__ void count_index_kernel(const long long* __restrict__ idx, int n, int nseg, int32_t* __restrict__ count,
                                   int32_t* __restrict__ err) {
  pdl_wait();
  pdl_launch();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long v = idx[i];
  if (v < 0 || v >= nseg) {
    *err = 1;
    return;
  }
  atomicAdd(&count[v], 1);
}

