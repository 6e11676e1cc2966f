/* libsstb200 - C ABI of the B200-native SST/FSD hot path.
 *
 * Drop-in boundary (SURVEY.md 8b).  The reference (tusen-ai/SST @ 7c95376) reaches its native code
 * through three extension modules; each entry point below names the reference interface it replaces:
 *
 *   pybind module `voxel_layer`          mmdet3d/ops/voxel/src/voxelization.cpp:6-11, voxelization.h:51-130
 *   torch_scatter.scatter / scatter_max   call sites mmdet3d/ops/sst/sst_ops.py:173-175
 *   TorchEx ingroup_indices.forward       call site  mmdet3d/ops/sst/sst_ops.py:246-264
 *
 * plus fused entry points for the parts of the path the reference runs as chains of ATen ops
 * (window partition / bucketing, the Sparse-Regional-Attention encoder layer, DynamicVFE, SIRLayer).
 *
 * Conventions
 *   - plain C types only: device pointers, sizes, a cudaStream_t passed as void*.  No torch types.
 *   - every function returns 0 on success, <0 on error; sstb200_last_error(ctx) describes it.
 *   - all work is enqueued on the context's stream (sstb200_set_stream); no function synchronises
 *     unless it has a `*_host` out-parameter that is non-NULL (documented per function).
 *   - outputs are caller-allocated.  Data-dependent row counts (number of voxels / windows) are
 *     returned in device memory (`*_dev`); capacity of such outputs is the worst case (= #inputs).
 *   - temporaries come from a per-context arena that grows on demand.
 *   - one context per (device, stream, thread).
 */
#ifndef SSTB200_H_
#define SSTB200_H_
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct sstb200_ctx sstb200_ctx;

#define SSTB200_REDUCE_SUM 0
#define SSTB200_REDUCE_MEAN 1
#define SSTB200_REDUCE_MAX 2
#define SSTB200_PREC_FP32 0 /* fp32 FFMA everywhere */
#define SSTB200_PREC_BF16 1 /* 16-bit tensor-core GEMMs, fp32 accumulate / softmax / LayerNorm / residual.  The SRA encoder uses
                             * IEEE fp16 operands (the reference's own mixed-precision mode, `fp16 = dict(loss_scale=32.0)`), the
                             * VFE / SIR tensor paths bf16; the API name of the mode stays 'bf16'. */
#define SSTB200_PREC_F16 1
#define SSTB200_PREC_FP32_TC 2 /* sstb200_spconv_forward only: fp32 tolerance on the tensor core - every operand carried as two fp16 numbers
                                * (hi + residue, 22 significant bits), three tcgen05 products per stage, fp32 accumulation in TMEM */

int sstb200_version(void);
sstb200_ctx* sstb200_create(int device);
void sstb200_destroy(sstb200_ctx* ctx);
int sstb200_set_stream(sstb200_ctx* ctx, void* cuda_stream);
const char* sstb200_last_error(sstb200_ctx* ctx);
int sstb200_num_sms(sstb200_ctx* ctx);

/* V1  voxel_layer.dynamic_voxelize(points, coors, voxel_size, coors_range, NDim=3)
 *     (voxelization.h:72-88, kernel voxelization_cuda.cu:25-65).  points [P,F] fp32 row-major,
 *     coors [P,3] int32 (z,y,x), clamped to the grid like this fork does.  No device sync
 *     (the reference's cudaDeviceSynchronize at voxelization_cuda.cu:371 is not reproduced). */
int sstb200_dynamic_voxelize(sstb200_ctx* ctx, const float* points, int num_points, int num_features,
                             const float voxel_size[3], const float coors_range[6], int32_t* coors);

/* V1' voxel_layer.hard_voxelize(points, voxels, coors, num_points_per_voxel, voxel_size, coors_range, max_points, max_voxels)
 *     (voxelization.h:51-70 -> voxelization_cpu.cpp:43-142 / voxelization_cuda.cu:68-330; SURVEY 8f next-4).  voxels
 *     [max_voxels, max_points, F], coors [max_voxels,3] (z,y,x), num_points_per_voxel [max_voxels] are caller-allocated AND
 *     zero-initialised, as ops/voxel/voxelize.py:46-53 does.  Voxels are numbered by first appearance in the point list; every
 *     voxel keeps its first max_points points in input order.  Returns the voxel count in device memory and, if
 *     voxel_num_host != NULL, on the host (one stream sync; the reference returns an int). */
int sstb200_hard_voxelize(sstb200_ctx* ctx, const float* points, int num_points, int num_features, const float voxel_size[3],
                          const float coors_range[6], int max_points, int max_voxels, float* voxels, int32_t* coors,
                          int32_t* num_points_per_voxel, int32_t* voxel_num_dev, int32_t* voxel_num_host);

/* V2  voxel_layer.dynamic_point_to_voxel_forward(feats, coors, reduce_type)
 *     (voxelization.h:96-108 -> scatter_points_cuda.cu:183-234).
 *     feats [P,C] fp32, coors [P,3] int32.  coor_lo/hi: inclusive bounds of the non-negative
 *     coordinates per column (the reference needs none because it sorts; this build ranks through a
 *     bitmap over the bounding grid).  Outputs (capacity P rows): reduced [.,C], out_coors [.,3],
 *     coors_map [P] (-1 = dropped), reduce_count [.].  num_voxels_dev: device int32.
 *     If num_voxels_host != NULL the call synchronises the stream and stores the count there; it then also fails
 *     (SSTB200 error, no silent result) if a row with non-negative coordinates lay outside coor_lo/hi.
 *     Reproduces the reference's unconditional removal of the first sorted row (:207-210). */
int sstb200_dynamic_point_to_voxel_forward(sstb200_ctx* ctx, const float* feats, const int32_t* coors,
                                           int num_points, int num_feats, int reduce_type,
                                           const int32_t coor_lo[3], const int32_t coor_hi[3],
                                           float* reduced, int32_t* out_coors, int32_t* coors_map,
                                           int32_t* reduce_count, int32_t* num_voxels_dev,
                                           int32_t* num_voxels_host);

/* V3  voxel_layer.dynamic_point_to_voxel_backward (voxelization.h:110-130 ->
 *     scatter_points_cuda.cu:236-303).  grad_feats [P,C] is fully written (zero where no grad). */
int sstb200_dynamic_point_to_voxel_backward(sstb200_ctx* ctx, float* grad_feats, const float* grad_reduced,
                                            const float* feats, const float* reduced,
                                            const int32_t* coors_map, const int32_t* reduce_count,
                                            int num_points, int num_voxels, int num_feats, int reduce_type);

/* V5a torch.unique(coors, dim=0, return_inverse=True, return_counts=True) on int64 rows
 *     (sst_ops.py:158-160,170; voxel_encoder.py:561; sir.py:70).  coors [P,ndim] int64, ndim<=4,
 *     every value inside [coor_lo, coor_hi].  Outputs: new_coors [.,ndim] (lexicographically sorted),
 *     inverse [P] int64, counts [.] int32 (may be NULL). */
int sstb200_unique_rows_i64(sstb200_ctx* ctx, const int64_t* coors, int num_rows, int ndim,
                            const int64_t* coor_lo, const int64_t* coor_hi, int64_t* new_coors,
                            int64_t* inverse, int32_t* counts, int32_t* num_unique_dev,
                            int32_t* num_unique_host);

/* V5b torch_scatter.scatter(src, index, dim=0, reduce=sum|mean) / scatter_max (sst_ops.py:173-175).
 *     src [P,C] fp32, index [P] int64 in [0,num_segments), out [num_segments,C] (empty segments: 0).
 *     argmax (int64 [num_segments,C], may be NULL): lowest row attaining the max, P if empty. */
int sstb200_segment_reduce(sstb200_ctx* ctx, const float* src, const int64_t* index, int num_rows,
                           int num_feats, int num_segments, int reduce_type, float* out, int64_t* argmax);

/* B2  ingroup_indices.forward(group_inds, out_inds) (sst_ops.py:246-264): rank of each element among
 *     the elements carrying the same id, in stable (input) order == get_inner_win_inds_slow
 *     (sst_input_layer.py:200-208).  group ids in [0, max_group_id]. */
int sstb200_ingroup_indices(sstb200_ctx* ctx, const int64_t* group_inds, int num, int64_t max_group_id,
                            int64_t* out_inds);

/* B1+B2+B3(levels)+B4  window partition and bucketing for ONE shift (do_shift = 0 | 1), fused.
 *   get_window_coors            ops/sst/sst_ops.py:266-314
 *   get_inner_win_inds          ops/sst/sst_ops.py:244-264 (stable order, sst_input_layer.py:200-208)
 *   level assignment            models/middle_encoders/sst_input_layer_v2.py:128-150
 *   make_continuous_inds + get_flat2win_inds   ops/sst/sst_ops.py:316-331, 27-64
 * coors [n,4] (b,z,y,x).  n may also be given on the device (n_dev != NULL, n = capacity).
 * token_level (int64 [n], may be NULL): drop level carried over from a preceding drop phase; when NULL the
 * level of a window follows from its token count.  All outputs caller-allocated with capacity n
 * (win_offsets n+1); pointers marked "opt" may be NULL. */
typedef struct {
  int32_t sparse_shape[3]; /* x, y, z */
  int32_t window_shape[3]; /* x, y, z (z = sparse z for 2-D windows) */
  int32_t batch_size;      /* upper bound of batch index + 1 */
  int32_t num_levels;      /* <= 8, in the iteration order of the reference's drop_info dict */
  int32_t level_id[8];     /* dict keys */
  int32_t level_lo[8];     /* drop_range[0] */
  int32_t level_hi[8];     /* drop_range[1] */
  int32_t level_max_tokens[8];
} sstb200_window_cfg;

typedef struct {
  int64_t* batch_win_inds; /* opt [n]   == get_window_coors()[0] */
  int64_t* coors_in_win;   /* opt [n,3] == get_window_coors()[1]  (z,y,x) */
  int64_t* drop_level;     /* opt [n]   dict key of the window's level */
  int64_t* flat2win_inds;  /* opt [n]   rank_in_level * max_tokens + inner */
  int32_t* pos_code;       /* opt [n]   x | y<<8 | z<<16 of coors_in_win */
  int32_t* tok_win;        /* [n]   compact window index (rank of the window id among non-empty windows) */
  int32_t* tok_inner;      /* [n]   stable rank of the token inside its window */
  int32_t* win_offsets;    /* [n+1] CSR offsets into tok_perm, R+1 entries valid */
  int32_t* tok_perm;       /* [n]   token indices grouped by window, stable order inside */
  int32_t* win_level;      /* [n]   level slot (0..num_levels-1) per window, R valid */
  int32_t* win_rank;       /* [n]   rank of the window among the windows of its level */
  int32_t* counters;       /* [20]  R, windows per level slot [8], tokens per level slot [8], number of window batches,
                            *       [18] status bits (bit0 token outside the window grid, bit1 window count not covered), [19] spare */
  int32_t* tok_slot;       /* opt [n] position of the token inside tok_perm (inverse permutation) */
  int32_t* win_batch;      /* opt [n+16], 16-byte aligned: one record of 4 ints per batch b = the windows whose first slot lies in
                              [112b, 112b+112): {first window, end window, first slot, end slot}; at most n/32 + 2 records (fits: 4 (n/32 + 2) <= n + 16) */
} sstb200_window_shift;

/* status_host (opt, int32[18]): if non-NULL the call synchronises and returns
 * [0] = bit0: token outside the window grid, bit1: window count not covered by any drop_range;
 * [1..17] = copy of counters[0..16]. */
int sstb200_window_plan(sstb200_ctx* ctx, const int64_t* coors, int n, const int32_t* n_dev,
                        const sstb200_window_cfg* cfg, int do_shift, const int64_t* token_level,
                        const sstb200_window_shift* out, int32_t* status_host);
int sstb200_window_plan_i32(sstb200_ctx* ctx, const int32_t* coors, int n, const int32_t* n_dev,
                            const sstb200_window_cfg* cfg, int do_shift, const sstb200_window_shift* out);

/* A1+A2+A3  one Sparse-Regional-Attention encoder layer (EncoderLayer.forward,
 * mmdet3d/models/sst/sst_basic_block_v2.py:77-126 with WindowAttention :41-75, nn.MultiheadAttention or
 * CosineMultiheadAttention models/sst/cosine_msa.py:449-536), eval mode (dropout = identity).
 * All weight pointers are device pointers in the reference's nn.Module layouts (row-major [out,in]). */
typedef struct {
  int32_t d_model, nhead, dim_ff;
  int32_t act;       /* 1 relu, 2 gelu(erf) */
  int32_t post_norm; /* layer_cfg['post_norm'] (default 1) */
  float norm_eps;    /* LayerNorm 1e-5 / BatchNorm 1e-5 */
  const float *in_proj_w, *in_proj_b;   /* [3d,d], [3d] */
  const float *out_proj_w, *out_proj_b; /* [d,d], [d] */
  const float *lin1_w, *lin1_b;         /* [ff,d], [ff] */
  const float *lin2_w, *lin2_b;         /* [d,ff], [d] */
  const float *norm1_w, *norm1_b, *norm2_w, *norm2_b;
  const float *norm1_mean, *norm1_var, *norm2_mean, *norm2_var; /* non-NULL: layer_cfg['use_bn'] (eval BN) */
  const float* tau; /* non-NULL: cosine attention; tau_n = 1 or nhead */
  int32_t tau_n;
  float tau_min;
  /* optional IEEE fp16 copies of the four weight matrices (tensor-core path); NULL -> fp32 path only */
  const void *in_proj_w_f16, *out_proj_w_f16, *lin1_w_f16, *lin2_w_f16;
} sstb200_sra_layer;

/* window CSR of one shift (produced by sstb200_window_plan) + positional-embedding table
 * (SSTInputLayerV2.get_pos_embed, sst_input_layer_v2.py:238-305: pos[t, axis*L + j] =
 * table[axis][coord_in_win(axis)][j], zero beyond ndim*L). */
typedef struct {
  const int32_t* win_offsets; /* [R+1] */
  const int32_t* tok_perm;    /* [n] */
  const int32_t* tok_win;     /* [n] */
  const int32_t* pos_code;    /* [n] */
  const int32_t* num_windows_dev; /* counters[0] */
  const float* pos_table;     /* [pos_ndim][pos_maxw][pos_L] fp32 */
  int32_t pos_L, pos_maxw, pos_ndim;
  int32_t max_window_tokens;  /* upper bound on tokens per window (e.g. 144) */
  const int32_t* tok_slot;    /* [n] inverse of tok_perm (needed by the bf16 path) */
  const int32_t* win_batch;   /* opt [.] window batches (see sstb200_window_shift); counters[17] = number of batches */
} sstb200_sra_plan;


/* x, y: [n, d_model] fp32 in flat voxel order (y may alias x only if precision == FP32 is not used).
 * n may be device-resident (n_dev).  */
int sstb200_sra_layer_forward(sstb200_ctx* ctx, const sstb200_sra_layer* layer, const sstb200_sra_plan* plan,
                              const float* x, float* y, int n, const int32_t* n_dev, int precision);

/* nn.Linear forward: out[M,N] = act(A[M,K] . W[N,K]^T + bias), fp32 (act: 0 none, 1 relu, 2 gelu-erf).
 * Used for SSTv2.linear0 (models/backbones/sst_v2.py:60-61,127-128) and as a building block. */
int sstb200_linear(sstb200_ctx* ctx, const float* A, const float* W, const float* bias, float* out,
                   int M, int N, int K, int act);

/* V4 DynamicVFE.forward / V6 DynamicScatterVFE.forward, eval-mode BatchNorm, <= 2 VFE layers
 * (mmdet3d/models/voxel_encoders/voxel_encoder.py:229-298 and :551-612; layers utils.py:107-144).
 * points [P,in_channels] fp32, coors [P,4] (b,z,y,x).  Output rows are the non-empty voxels sorted by
 * (b,z,y,x); capacity P.  drop_first_voxel_per_sample = 1 reproduces DynamicVFE's DynamicScatter behaviour
 * (scatter_points_cuda.cu:207-210 through the per-sample loop scatter_points.py:85-99); DynamicScatterVFE
 * (torch.unique based) keeps every voxel. */
typedef struct {
  int32_t in_channels;       /* raw point dims F (before decoration) */
  int32_t num_layers;        /* 1 or 2 */
  int32_t feat_channels[2];
  int32_t with_cluster_center, with_voxel_center, with_distance;
  int32_t mode_max;          /* 1: max pooling, 0: average */
  int32_t drop_first_voxel_per_sample;
  int32_t batch_size;
  int32_t grid_zyx[3];       /* canvas dims (voxel_encoder.py:199-204) */
  float voxel_size[3];       /* vx, vy, vz */
  float center_offset[3];    /* v/2 + range_min (voxel_encoder.py:160-162) */
  float rel_dist_scaler;     /* DynamicScatterVFE only, else 1 */
  float bn_eps;
  int32_t precision;         /* SSTB200_PREC_FP32: FFMA everywhere; SSTB200_PREC_BF16: layer 1 on tcgen05 (bf16 operands) */
  const float* weight[2];    /* vfe_layers.i.linear.weight  [C_i, in_i] */
  const float* bn_weight[2]; /* vfe_layers.i.norm.{weight,bias,running_mean,running_var} */
  const float* bn_bias[2];
  const float* bn_mean[2];
  const float* bn_var[2];
} sstb200_vfe_cfg;

int sstb200_dynamic_vfe_forward(sstb200_ctx* ctx, const sstb200_vfe_cfg* cfg, const float* points,
                                const int32_t* coors, int num_points, float* voxel_feats, int32_t* voxel_coors,
                                int32_t* num_voxels_dev, int32_t* num_voxels_host);
int sstb200_dynamic_scatter_vfe_forward(sstb200_ctx* ctx, const sstb200_vfe_cfg* cfg, const float* points,
                                        const int64_t* coors, int num_points, float* voxel_feats,
                                        int64_t* voxel_coors, int64_t* unq_inv, int32_t* num_voxels_dev,
                                        int32_t* num_voxels_host);
/* DynamicScatterVFE over the rows of sstb200_voxelize_frames (the sync-free FSD segmentation engine): coors [num_points,4] int32
 * (b,z,y,x), rows past the last frame (-1) belong to no voxel and get unq_inv -1; voxel_coors int32, unq_inv [num_points] int32.
 * cfg->grid_zyx is the voxeliser's grid (every coordinate inside it); the voxel count is written to num_voxels_dev only. */
int sstb200_dynamic_scatter_vfe_forward_i32(sstb200_ctx* ctx, const sstb200_vfe_cfg* cfg, const float* points, const int32_t* coors,
                                            int num_points, float* voxel_feats, int32_t* voxel_coors, int32_t* unq_inv,
                                            int32_t* num_voxels_dev);

/* V1 (batched, sync-free form used by the frame engine): voxelise a batch of frames stored back to back.
 * points [capacity,F]; frame_offsets_dev: device int32 [num_frames+1] (row ranges of the frames, last entry =
 * number of valid rows).  coors4 [capacity,4] int32 = (b,z,y,x) like DynamicVoxelNet.voxelize
 * (mmdet3d/models/detectors/dynamic_voxelnet.py:49-71); rows beyond the last offset get (-1,-1,-1,-1) and are
 * ignored by every later stage. */
int sstb200_voxelize_frames(sstb200_ctx* ctx, const float* points, int capacity, int num_features,
                            const int32_t* frame_offsets_dev, int num_frames, const float voxel_size[3],
                            const float coors_range[6], int32_t* coors4);

/* C5  SingleStageFSDV2.voxelize_with_batch_idx (mmdet3d/models/detectors/single_stage_fsd_v2.py:108-123): virtual-voxel coordinates
 * of the concatenated real + virtual points.  points [n, ldp] fp32 (x,y,z first), batch_idx [n] int64 ->
 * coors [n,4] int64 (batch, z, y, x) = floor_div(p - range_lo, voxel_size) with torch.div(rounding_mode='floor') semantics, no clamp. */
int sstb200_voxelize_with_batch_idx(sstb200_ctx* ctx, const float* points, int n, int ldp, const int64_t* batch_idx,
                                    const float voxel_size[3], const float range_lo[3], int64_t* coors);

/* Fork / join of a side branch.  `side` is a second context (own stream, own workspace arena).  fork: side's stream waits for the
 * point of ctx's stream at which the last sstb200_dynamic_vfe_forward / sstb200_dynamic_scatter_vfe_forward call had produced
 * voxel_coors and num_dev (the VFE layers that follow in that call keep running on ctx's stream); join: ctx's stream waits for
 * everything enqueued on side's stream so far.  The engine runs the two sstb200_window_plan calls of a frame on the side branch,
 * next to the VFE layers.  Valid on plain streams and inside sstb200_graph_begin/end (the side stream joins the capture). */
int sstb200_branch_fork(sstb200_ctx* ctx, sstb200_ctx* side);
int sstb200_branch_join(sstb200_ctx* ctx, sstb200_ctx* side);

/* CUDA-graph helpers for callers that chain several entry points per frame (the reference has no
 * counterpart: it launches ~10^3 ATen kernels per frame with >= 8 host syncs, SURVEY.md 3.1).
 * begin: start capturing the context's stream; end: stop, instantiate, return an opaque handle and the number
 * of kernel / memset+memcpy nodes; launch: replay on the context's stream. */
int sstb200_graph_begin(sstb200_ctx* ctx);
int sstb200_graph_end(sstb200_ctx* ctx, void** graph_exec_out, int32_t* num_kernel_nodes, int32_t* num_other_nodes);
int sstb200_graph_launch(sstb200_ctx* ctx, void* graph_exec);
int sstb200_graph_destroy(sstb200_ctx* ctx, void* graph_exec);

/* S1-S3  SIRLayer.forward (mmdet3d/models/voxel_encoders/voxel_encoder.py:696-764; build_mlp ops/sst/sst_ops.py:334-361;
 * DynamicVFELayerV2 voxel_encoders/utils.py:147-189), LayerNorm norm, mode='max', with_rel_mlp=True.
 * in_feats [N,in_channels] = cat(points, feats) as SIR.forward builds it (models/backbones/sir.py:77), f_cluster [N,3]
 * (un-scaled; divided by rel_dist_scaler inside), group index inv [N] int64 in [0,G) (torch.unique inverse).
 * out_point [N, C_last]; out_group [G, C0+C1] = concatenated per-layer group max (voxel_encoder.py:751). */
typedef struct {
  int32_t in_channels;
  int32_t rel_in;          /* rel_mlp_in_channel (3) */
  int32_t num_rel;         /* number of rel-MLP layers (hidden dims + in_channels) */
  int32_t rel_dims[4];
  int32_t num_vfe;         /* 1 or 2 */
  int32_t feat_channels[2];
  int32_t act;             /* 1 relu, 2 gelu */
  int32_t mode_max;
  int32_t with_shortcut;
  float norm_eps;
  float xyz_normalizer[3];
  float rel_dist_scaler;
  const float* rel_w[4];    /* rel_mlp.i.0.weight [dims[i], in_i] */
  const float* rel_ln_w[4]; /* rel_mlp.i.1.weight */
  const float* rel_ln_b[4];
  const float* vfe_w[2];    /* vfe_layers.i.linear.weight  [C_i, in_i] (in_1 = 2*C0) */
  const float* vfe_ln_w[2];
  const float* vfe_ln_b[2];
} sstb200_sir_layer;

int sstb200_sir_layer_forward(sstb200_ctx* ctx, const sstb200_sir_layer* layer, const float* in_feats,
                              const float* f_cluster, const int64_t* inv, int num_points, int num_groups,
                              float* out_point, float* out_group);

/* S1' as above, plus: a cached group CSR (csr_offsets [G+1], csr_order [N] from sstb200_group_csr; both NULL = built inside),
 * `precision` (SSTB200_PREC_BF16: the rel-MLP's last layer and both VFE layers run as tcgen05 GEMMs with bf16 operands and fp32
 * accumulation - needs feat_channels [128,128], rel-MLP [16,32,cin], cin <= 192, else SSTB200 "unsupported" error) and a row
 * pitch for out_point (>= C_last; lets SIR.forward write block i's point features straight into block i+1's [points || feats]
 * input; bf16 path only, 0 = dense).  in_feats may likewise be a pitched matrix (in_ld floats per row, 0 = dense) whose columns
 * >= in_gap_at sit in_gap floats further right (the 16-byte aligned feature block of that hand-over buffer). */
int sstb200_sir_layer_forward_ex(sstb200_ctx* ctx, const sstb200_sir_layer* layer, const float* in_feats, int in_ld,
                                 int in_gap_at, int in_gap, const float* f_cluster, const int64_t* inv, int num_points, int num_groups,
                                 const int32_t* csr_offsets, const int32_t* csr_order, int precision, float* out_point,
                                 int out_point_ld, float* out_group);

/* Points grouped by `inv` (values in [0, num_groups)): offsets [num_groups+1] int32, order [num_points] int32 (order inside a
 * group unspecified).  What SIR.forward (models/backbones/sir.py:67-87, `unique_once`) shares between its blocks. */
int sstb200_group_csr(sstb200_ctx* ctx, const int64_t* inv, int num_points, int num_groups, int32_t* offsets, int32_t* order);

/* A4'  SSTv2.recover_bev (mmdet3d/models/backbones/sst_v2.py:161-196): voxel_feat [M,C] fp32 rows at coors [M,4] int64 (b,z,y,x)
 * -> canvas [B,C,ny,nx] fp32, empty cells 0 (the canvas need not be zeroed by the caller: every element is written once).
 * Synchronises the stream to report out-of-canvas coordinates as an error (the reference would raise an index error). */
int sstb200_recover_bev(sstb200_ctx* ctx, const float* voxel_feat, const int64_t* coors, int num_voxels, int channels,
                        int batch_size, int ny, int nx, float* canvas);

/* N1  Voxel2PointScatterNeck.forward (mmdet3d/models/necks/voxel2point_neck.py:28-62; SURVEY 8f next-2): points [N,Cp] fp32,
 * pts_coors [N,4] int64 (b,z,y,x), voxel_feats [M,C] fp32 (rows of dropped voxels hold `padding`), voxel2point_inds [N] int64.
 * out [<=N, C(+3)] receives, for every point whose voxel row is not all-padding and in input order, the voxel row followed (with_xyz)
 * by the point's offset from its voxel centre; mask_out [N] (1 = kept).  The call synchronises once to return the row count (the
 * reference's boolean indexing does the same) and to report out-of-range indices as an error. */
int sstb200_voxel2point(sstb200_ctx* ctx, const float* points, int point_dims, const int64_t* pts_coors, const float* voxel_feats,
                        int num_voxels, int channels, const int64_t* voxel2point_inds, int num_points, float padding,
                        const float voxel_size[3], const float pc_min[3], int with_xyz, int normalize_local_xyz, float* out,
                        uint8_t* mask_out, int32_t* num_out_dev, int32_t* num_out_host);
/* N1' the same without a host sync: pts_coors [N,4] and voxel2point_inds [N] int32, num_points N = the point capacity, the voxel
 * count read from num_voxels_dev; a point whose index is outside [0, voxel count) (e.g. -1: rows past the last frame) is not kept
 * (mask 0).  The kept-row count is written to num_out_dev. */
int sstb200_voxel2point_dev(sstb200_ctx* ctx, const float* points, int point_dims, const int32_t* pts_coors, const float* voxel_feats,
                            const int32_t* num_voxels_dev, int channels, const int32_t* voxel2point_inds, int num_points, float padding,
                            const float voxel_size[3], const float pc_min[3], int with_xyz, int normalize_local_xyz, float* out,
                            uint8_t* mask_out, int32_t* num_out_dev);

/* A4  the whole encoder stack (SSTv2.forward's block loop, mmdet3d/models/backbones/sst_v2.py:129-133 with
 * BasicShiftBlockV2.forward, models/sst/sst_basic_block_v2.py:144-169): layer l uses the windows of shift l % 2.
 * x [n,d] input (not modified), y [n,d] output, tmp [n,d] scratch; all fp32, distinct buffers.  With precision BF16 and the
 * SST-6 shape (d=128, h=8, ff=256, post-norm LayerNorm, GELU) this runs 2 launches per layer: ragged window attention and a
 * fused tcgen05 kernel (out-proj + LN1 + FFN + LN2 + the next layer's QKV); otherwise it loops sstb200_sra_layer_forward. */
int sstb200_sra_stack_forward(sstb200_ctx* ctx, const sstb200_sra_layer* layers, int num_layers,
                              const sstb200_sra_plan* plan_shift0, const sstb200_sra_plan* plan_shift1, const float* x,
                              float* y, float* tmp, int n, const int32_t* n_dev, int precision);

/* ---- training (BASELINE config 4): SSTv2's encoder stack with everything the backward pass needs kept in `workspace`, and the
 * backward pass (the autograd graph torch builds over sst_basic_block_v2.py:100-126 / backbones/sst_v2.py:129-133 in the reference).
 * Shape: d_model 128, 8 heads, dim_ff 256, post-norm LayerNorm, GELU, windows <= 144 tokens (all configs/sst_refactor models).
 * GEMM operands and saved activations are bf16, accumulation / softmax / LayerNorm / residual stream / gradients of the
 * parameters fp32.  For these two entry points the `*_w_f16` fields of sstb200_sra_layer hold BF16 copies of the weights. */
typedef struct {
  const void *in_proj_wt, *out_proj_wt, *lin1_wt, *lin2_wt; /* bf16 TRANSPOSED copies, [in, out] row-major */
} sstb200_sra_layer_wt;
typedef struct { /* fp32 accumulators in the layout of the parameters; the call ADDS to them */
  float *in_proj_w, *in_proj_b, *out_proj_w, *out_proj_b, *lin1_w, *lin1_b, *lin2_w, *lin2_b, *norm1_w, *norm1_b, *norm2_w, *norm2_b;
} sstb200_sra_layer_grads;

size_t sstb200_sra_train_workspace_bytes(int n, int num_layers);
/* x [n,128] fp32 (not modified) -> y_out [n,128]; workspace: device buffer of sstb200_sra_train_workspace_bytes() */
int sstb200_sra_stack_forward_train(sstb200_ctx* ctx, const sstb200_sra_layer* layers, int num_layers,
                                    const sstb200_sra_plan* plan_shift0, const sstb200_sra_plan* plan_shift1, const float* x,
                                    float* y_out, void* workspace, int n);
/* dy [n,128] = d loss / d y_out  ->  dx [n,128] = d loss / d x, parameter gradients accumulated into `grads` */
int sstb200_sra_stack_backward(sstb200_ctx* ctx, const sstb200_sra_layer* layers, const sstb200_sra_layer_wt* wt,
                               const sstb200_sra_layer_grads* grads, int num_layers, const sstb200_sra_plan* plan_shift0,
                               const sstb200_sra_plan* plan_shift1, const float* x, void* workspace, const float* dy, float* dx,
                               int n);
/* torch.optim.AdamW step over a flat fp32 buffer (decoupled weight decay, bias-corrected moments); the gradient is read as
 * grads[i] * grad_scale (1 / world_size after a summing all-reduce).  step counts from 1. */
int sstb200_adamw_step(sstb200_ctx* ctx, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                       float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale);

/* ---- next-1 (SURVEY 8f): sparse 3-D convolution of the reference's sparse U-Nets (SimpleSparseUNet / VirtualVoxelMixer,
 * mmdet3d/models/middle_encoders/sparse_unet.py:15-505; SparseBasicBlock / make_sparse_convmodule, mmdet3d/ops/sparse_block.py:81-289),
 * which the reference delegates to spconv.  The three entry points replace spconv's native interface as vendored in the tree
 * (mmdet3d/ops/spconv/src/all.cc:21-33): get_indice_pairs_3d (ops.py:47-107 -> include/spconv/spconv_ops.h:25-93, geometry.h:25-301)
 * and indice_conv_fp32 / fused_indice_conv_fp32 (ops.py:110-137 -> spconv_ops.h:95-260, fused_spconv_ops.h).
 * Coordinates are int32 rows (batch, z, y, x); spatial shapes / kernel sizes / strides / paddings are (z, y, x) triples; kernel
 * offset k = (dz * ky + dy) * kx + dx reads the input cell  out * stride - padding + (dz, dy, dx)  (geometry.h:60-67).
 * The rulebook is OUTPUT-STATIONARY: nbr[o][k] = input row feeding output row o through offset k, or -1. */

/* Active output cells of SparseConv3d (non-submanifold): every output cell with at least one active input in its receptive field,
 * emitted in lexicographic (b,z,y,x) order (spconv's order is hash-insertion order; features are compared per coordinate).
 * out_cap >= min(n_in * prod(ceil(k/s)), batch * prod(out_shape)).  num_out_host != NULL: one stream sync, and an input coordinate
 * outside batch_size / in_shape is reported as an error. */
int sstb200_spconv_out_coors(sstb200_ctx* ctx, const int32_t* in_coors, int n_in, int batch_size, const int32_t in_shape[3],
                             const int32_t out_shape[3], const int32_t ksize[3], const int32_t stride[3], const int32_t padding[3],
                             int32_t* out_coors, int out_cap, int32_t* num_out_dev, int32_t* num_out_host);

/* Neighbour tables between two coordinate sets (rows unique).  SubMConv3d: out_coors = in_coors, stride 1, out_shape = in_shape.
 * nbr [n_out, KV] (may be NULL): input row at  out * stride - padding + delta_k.  nbr_inv [n_in, KV] (may be NULL): the transposed
 * table = output row that input row i feeds through offset k - the table SparseInverseConv3d runs on (indice pairs of its couple
 * conv with in / out swapped, mmdet3d/ops/spconv/conv.py:147-153).  status_host != NULL: one stream sync, coordinates outside the
 * grids are an error. */
int sstb200_spconv_table(sstb200_ctx* ctx, const int32_t* in_coors, int n_in, const int32_t* out_coors, int n_out, int batch_size,
                         const int32_t in_shape[3], const int32_t out_shape[3], const int32_t ksize[3], const int32_t stride[3],
                         const int32_t padding[3], int32_t* nbr, int32_t* nbr_inv, int32_t* status_host);

/* out[o, :] = act( (sum_k feats[nbr[o][k], :] . W[k]) * scale + shift + residual[o, :] )   - one launch for conv + folded
 * BatchNorm1d (+ residual add) (+ ReLU).  feats [*, c_in] fp32, weight [KV, c_in, c_out] fp32 = the reference's parameter layout
 * (D,H,W,in,out; mmdet3d/ops/spconv/conv.py:97-98), scale / shift [c_out] or NULL (1 / 0), residual [n_out, c_out] or NULL.
 * precision FP32: FFMA implicit GEMM (c_in, c_out multiples of 4).  precision BF16 (16-bit operands, fp32 accumulation in TMEM):
 * tcgen05 implicit GEMM over weight_h16 = IEEE fp16 copy laid out [KV, c_out, c_in]; needs c_in, c_out multiples of 64, KV <= 27.
 * precision FP32_TC: the same kernel in split mode; weight_h16 = [2][KV, c_out, c_in]: the fp16 copy followed by the fp16 residue
 * (w - float(half(w))). */
int sstb200_spconv_forward(sstb200_ctx* ctx, const float* feats, int c_in, const int32_t* nbr, int n_out, int kernel_volume,
                           const float* weight, const void* weight_h16, int c_out, const float* scale, const float* shift,
                           const float* residual, int relu, int precision, float* out);

/* Backward of sstb200_spconv_forward without epilogue (indice_conv_backward_fp32, mmdet3d/ops/spconv/src/all.cc:34-35 ->
 * spconv_ops.h:262-420).  The input gradient needs no entry point of its own: dX = sstb200_spconv_forward(dY, nbr_T, W^T) on the
 * TRANSPOSED table (nbr_inv of sstb200_spconv_table; the table SparseInverseConv3d runs on).  This call computes the weight gradient
 * grad_weight [KV, c_in, c_out] fp32 (fully written) = sum over pairs of feats[nbr[o][k]]^T . grad_out[o]; fp32 atomics across row
 * chunks, so the last bits depend on the launch like the reference's backward. */
int sstb200_spconv_backward_weight(sstb200_ctx* ctx, const float* feats, int c_in, const int32_t* nbr, int n_out, int kernel_volume,
                                   const float* grad_out, int c_out, float* grad_weight);

/* Device-count variants of the three entry points above (capacity-sized buffers, one CUDA graph per frame): every row count is
 * read from device memory (n_*_dev <= the capacity n_*_cap), nothing is read back to the host, and the kernels loop over the real
 * rows with grids sized from the SM count.  Coordinates must lie inside batch_size / the shapes (not checked on the device).
 * Rows of the outputs past the device count are left untouched.  Same tables and the same arithmetic as the host-count calls. */
int sstb200_spconv_out_coors_dev(sstb200_ctx* ctx, const int32_t* in_coors, int n_in_cap, const int32_t* n_in_dev, int batch_size,
                                 const int32_t in_shape[3], const int32_t out_shape[3], const int32_t ksize[3], const int32_t stride[3],
                                 const int32_t padding[3], int32_t* out_coors, int out_cap, int32_t* num_out_dev);
int sstb200_spconv_table_dev(sstb200_ctx* ctx, const int32_t* in_coors, int n_in_cap, const int32_t* n_in_dev, const int32_t* out_coors,
                             int n_out_cap, const int32_t* n_out_dev, int batch_size, const int32_t in_shape[3], const int32_t out_shape[3],
                             const int32_t ksize[3], const int32_t stride[3], const int32_t padding[3], int32_t* nbr, int32_t* nbr_inv);
/* feats rows have pitch lda (floats), out rows ldo, residual rows ldr (all multiples of 4): a convolution can read one half of a
 * wider matrix and write into one half of another (the decoder's [bottom || lateral] concatenation without a copy). */
int sstb200_spconv_forward_dev(sstb200_ctx* ctx, const float* feats, int lda, int c_in, const int32_t* nbr, int n_out_cap,
                               const int32_t* n_out_dev, int kernel_volume, const float* weight, const void* weight_h16, int c_out,
                               const float* scale, const float* shift, const float* residual, int ldr, int relu, int precision, float* out,
                               int ldo);
/* SparseUNet.decoder_layer_forward's merge (mmdet3d/models/middle_encoders/sparse_unet.py reduce_channel + add):
 * out[o, j] = x_merge[o, j] + sum_g cat[o, j * r + g], r = cat_channels / channels; x_merge / out [n, channels], cat [n, cat_channels],
 * the group sum first, then the add (torch's order). */
int sstb200_spconv_decoder_merge(sstb200_ctx* ctx, const float* x_merge, const float* cat, int channels, int cat_channels, int n_cap,
                                 const int32_t* n_dev, float* out);

/* ---- next-3 (SURVEY 8f): FSD instance grouping.  find_connected_componets / _single_batch / _gpu
 * (mmdet3d/models/detectors/single_stage_fsd.py:37-81; TorchEx connected_components at :20,39-45): two centres of the same sample are
 * adjacent when sqrt(dx^2 + dy^2) < dist (xy only, fp32); labels [n] = component number, components numbered sample by sample (batch
 * index ascending) and, inside a sample, by their first centre in input order - scipy.sparse.csgraph.connected_components' numbering
 * with the reference's running `base`.  centers [n, stride >= 2] fp32 (x, y first), batch_idx [n] int32 in [0, batch_size) or NULL
 * (one sample).  xy_min / xy_max bound the binning grid (centres outside are binned into the border cells: still exact).
 * num_components_host != NULL: one stream sync; a batch index outside [0, batch_size) is then reported as an error (label -1). */
int sstb200_connected_components(sstb200_ctx* ctx, const float* centers, int stride, const int32_t* batch_idx, int n, int batch_size,
                                 float dist, const float xy_min[2], const float xy_max[2], int32_t* labels,
                                 int32_t* num_components_dev, int32_t* num_components_host);

#ifdef __cplusplus
}
#endif
#endif
