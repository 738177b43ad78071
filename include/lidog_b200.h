/*
 * lidog_b200.h -- C ABI of the B200-native LiDOG hot path (liblidog_b200.so, sm_100a).
 *
 * The reference (saltoricristiano/lidog) reaches its hot path only through the
 * Python package MinkowskiEngine 0.5.4 (reference README.md:29), whose pybind
 * module `MinkowskiEngineBackend._C` is what these entry points replace.  Each
 * function names the reference call site (file:line under /root/reference) that
 * fixes its contract; the ME-internal convention it follows is in SURVEY.md
 * Appendix C.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless it
 *     says "host"; the caller owns and allocates all memory (outputs included);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 = OK, negative = error (lg_last_error_string() explains);
 *     data-dependent errors (coordinate outside the packed-key range) are
 *     reported through the device status word documented per function;
 *   - rows of coordinate matrices are int32 (batch, x, y, z); feature matrices
 *     are row-major float32.
 */
#ifndef LIDOG_B200_H
#define LIDOG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LG_OK 0
#define LG_ERR_INVALID -1     /* bad argument (shape, alignment, unsupported size) */
#define LG_ERR_CUDA -2        /* CUDA runtime / driver error */
#define LG_ERR_RANGE -3       /* coordinate outside the 16-bit-per-axis key range (device status) */
#define LG_ERR_UNSUPPORTED -4 /* shape not supported by the tensor-core path */

#define LG_TILE_ROWS 128 /* rows per gather tile; n_slots of every plan is a multiple of it */

/* operand formats of the tensor-core kernels (kind::f16 tcgen05.mma, fp32 accumulate) */
#define LG_FMT_BF16 0
#define LG_FMT_FP16 1

/* BEV duplicate-pixel policies (SURVEY.md 8a-11) */
#define LG_BEV_LAST 0 /* highest row index wins; gradient to every row of the pixel (reference behaviour) */
#define LG_BEV_MAX 1  /* channel-wise max; gradient to the first row attaining it (north_star scatter-max) */

int lg_version(void);
const char* lg_last_error_string(void); /* host string, thread-local */
int lg_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------ hash / voxelisation */

/* Open-addressing table: 16 bytes per slot {uint64 key, int32 value, pad}. */
int64_t lg_hash_capacity(int64_t n_keys); /* power of two >= 2*n_keys */
size_t lg_hash_bytes(int64_t capacity);

/* q = int32(floor(points / size)) in float32 division, per axis; writes (batch, qx, qy, qz).
 * Replaces the quantisation half of ME.utils.sparse_quantize
 * (call sites utils/datasets/semantickitti_bev.py:232-238, synth4d_bev.py:274-280,
 * nuscenes_bev.py:244-250, mix3D.py:67-72).  batch_of_row may be NULL (batch 0). */
int lg_quantize_points(const float* points_xyz, const int32_t* batch_of_row, int64_t n, float size_x, float size_y,
                       float size_z, int32_t* coords4_out, void* stream);

/* The same for float64 points, divided in float64: what the reference's TRAINING path feeds sparse_quantize -- its
 * augmentations multiply the float32 cloud by float64 matrices (utils/common/augmentation.py:10-20, applied at
 * utils/datasets/semantickitti_bev.py:214-219), and numpy keeps `float64_array / python_float` in float64. */
int lg_quantize_points_f64(const double* points_xyz, const int32_t* batch_of_row, int64_t n, double size_x,
                           double size_y, double size_z, int32_t* coords4_out, void* stream);

size_t lg_coords_unique_workspace(int64_t n);

/* Unique coordinates in first-occurrence order + hash table build.
 * coords' = floor(coords / stride) * stride on the 3 spatial axes (stride 1 = as is).
 *   table/capacity : filled with key -> unique row id (usable by lg_kernel_map afterwards)
 *   out_coords4    : [>= n, 4] unique (strided) coordinates, first-occurrence order
 *   unique_map     : [>= n] input row of each unique voxel (ascending)
 *   inverse_map    : [n] unique id of every input row
 *   labels/colabels: optional; colabel = common label of the voxel or ignore_label
 *   count_status   : int64[2] = {n_unique, status (0 or LG_ERR_RANGE)}
 * Replaces: the unique/inverse half of sparse_quantize (same call sites), the
 * coordinate-manager insert of ME.SparseTensor (utils/pipelines/trainer_lighting_2d.py:151)
 * and the stride-2 coordinate maps implied by MinkowskiConvolution(stride=2)
 * (utils/models/minkunet_bev.py:62,69,76,83). */
int lg_coords_unique(const int32_t* coords4, int64_t n, int32_t stride, void* table, int64_t capacity,
                     int32_t* out_coords4, int64_t* unique_map, int64_t* inverse_map, const int32_t* labels,
                     int32_t ignore_label, int32_t* colabels, int64_t* count_status, void* workspace,
                     size_t workspace_bytes, void* stream);

/* Every coordinate level of a batch in ONE call: level 0 = lg_coords_unique(coords4, strides[0]) (labels / colabels
 * apply to it), level l = lg_coords_unique(level l-1 coordinates, strides[l]).  The row count of a level reaches the
 * next one on the DEVICE, so the host does not wait between levels: the caller sizes every level's arrays and table
 * for the upper bound n (capacity >= lg_hash_capacity(n)), and reads all counts with one synchronisation -- the
 * coordinate manager of ME.SparseTensor (utils/pipelines/trainer_lighting_2d.py:151) plus the four stride-2 maps of
 * MinkUNet34 (utils/models/minkunet_bev.py:62,69,76,83) used to cost five host round trips per training step.
 *   levels[l].inverse_map: row of level l for every row of the level below (level 0: for every input row);
 *   counts_dev int64[2 * n_levels] = {n_unique, status} per level; counts_host (nullable, pinned host memory)
 *   receives a copy on the stream.  Scratch: library arena. */
typedef struct lgLevelOut {
  void* table;
  int64_t capacity;
  int32_t* coords4;
  int64_t* unique_map;
  int64_t* inverse_map;
} lgLevelOut;
int lg_coords_pyramid(const int32_t* coords4, int64_t n, const int32_t* labels, int32_t ignore_label, int32_t* colabels,
                      int32_t n_levels, const int32_t* strides /* host */, const lgLevelOut* levels /* host */,
                      int64_t* counts_dev, int64_t* counts_host, void* stream);

/* ------------------------------------------------------------------ kernel maps */

/* Gather plan consumed by the convolution kernels.  For slot s of tile t = s / LG_TILE_ROWS and
 * kernel offset k with bit k set in tile_mask[t]:  the operand row is nbr[k * k_stride + s]
 * (-1 = no neighbour = zero row) and the result row is out_row[s] (NULL = s itself). */
typedef struct lgConvPlan {
  const int32_t* nbr;
  int64_t k_stride; /* n_slots, or 0 when a tile uses one k only (transposed stride-2 plans) */
  const int32_t* out_row;
  const uint32_t* tile_mask; /* [n_slots / LG_TILE_ROWS][mask_words] */
  int32_t kernel_volume;     /* K */
  int32_t mask_words;        /* ceil(K / 32) */
  int64_t n_slots;
  int64_t n_out; /* rows of the result matrix */
  int64_t n_in;  /* rows of the gathered matrix */
} lgConvPlan;

/* Neighbour table for out voxel o and offset k (x fastest; odd size centred, even size 0-based;
 * offsets scaled by offset_scale = input tensor stride):  nbr[k][o] = row of (o + off_k) in table_in.
 * Replaces ME's kernel-map generation implied by every MinkowskiConvolution
 * (utils/models/minkunet_bev.py:57-123,410-442).  n_slots = round_up(n_out, LG_TILE_ROWS).
 * in_row_offset: subtracted from every row the table returns -- the table may index a larger coordinate set of which
 *   the gathered matrix is a contiguous slice (multi-source batches sharing one hashed index,
 *   utils/pipelines/trainer_lighting_2d_multi.py:146-167); 0 otherwise.
 * same_set != 0 declares that out_coords4 IS the set the table indexes (3x3x3 / 5x5x5 same-stride maps): pair
 *   (k, o -> i) then implies (K-1-k, i -> o), and only half of the offsets are probed. */
int lg_kernel_map(const void* table_in, int64_t capacity_in, const int32_t* out_coords4, int64_t n_out,
                  int32_t kernel_size, int32_t offset_scale, int32_t in_row_offset, int32_t same_set, int32_t* nbr,
                  int64_t n_slots, uint32_t* tile_mask, void* stream);

/* Same neighbour table with the rows REORDERED so that rows with the same neighbour pattern share a
 * 128-row tile (kernel_size <= 3): slot s serves result row out_row[s] (-1 = padding) and gathers
 * nbr[k][s].  The pair SET is identical to lg_kernel_map's; only the processing order differs (sort key:
 * the row's offset bits, rarest offset most significant; stable, deterministic).  The convolution kernels
 * then issue ~2.4x fewer (tile, offset) units on LiDAR scans.  Same reference contract as lg_kernel_map. */
size_t lg_kernel_map_sorted_workspace(int64_t n_out, int32_t kernel_size);
int lg_kernel_map_sorted(const void* table_in, int64_t capacity_in, const int32_t* out_coords4, int64_t n_out,
                         int32_t kernel_size, int32_t offset_scale, int32_t in_row_offset, int32_t same_set,
                         int32_t* nbr, int32_t* out_row, int64_t n_slots, uint32_t* tile_mask, void* workspace,
                         size_t workspace_bytes, void* stream);

size_t lg_scan_workspace(int64_t n_items);

/* ME-format pair lists from a neighbour table: pairs sorted by (k, out);
 * k_offsets int64[K+1] = start of each offset's list (k_offsets[K] = total). */
int lg_kernel_map_pairs(const int32_t* nbr, int32_t K, int64_t n_slots, int32_t* in_rows, int32_t* out_rows,
                        int64_t* k_offsets, void* workspace, size_t workspace_bytes, void* stream);

/* Stride-2, kernel-2 "up" plan (transposed convolution coarse -> fine, and dgrad of the stride-2
 * convolution): fine rows grouped by child index k, each group padded to LG_TILE_ROWS.
 *   parent_of_fine : int64 [n_fine] (inverse_map of the stride-2 lg_coords_unique call)
 *   gather[n_slots], out_row[n_slots], tile_mask[n_slots/128] are outputs;
 *   n_slots must be >= round_up(n_fine, 128) + 8 * 128;  slots_used int64[1] receives the used count.
 * Replaces ME's transposed kernel map (utils/models/minkunet_bev.py:89,96,103,110). */
int lg_kernel_map_up2(const int32_t* fine_coords4, const int64_t* parent_of_fine, int64_t n_fine,
                      int32_t fine_stride, int64_t parent_offset /* subtracted from the parent ids */, int32_t* gather,
                      int32_t* out_row, uint32_t* tile_mask, int64_t n_slots, int64_t* slots_used, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ sparse convolution */

/* fp32 SIMT gather-GEMM:  Y[out_row[s], :] = sum_k A[nbr[k][s], :] @ Wk,  Wk = W[wk] (Ca x N) or its
 * transpose when w_transposed (W stored [K][N][Ca]); wk = K-1-k when flip_k.  Used for shapes the
 * tensor-core path does not take (Cin = 1 stem, Cout = 7 head) and as the on-device fp32 check.
 * bias (nullable, [N]) is added once per row.  Rows without any pair receive bias / zero. */
int lg_conv_gemm_simt(const lgConvPlan* plan, const float* A, int32_t Ca, const float* W, int32_t N,
                      int32_t w_transposed, int32_t flip_k, const float* bias, float* Y, void* stream);

size_t lg_conv_wgrad_workspace(const lgConvPlan* plan, int32_t Ca, int32_t Cb);

/* dW[k] (Cin x Cout) = sum_s X_in[nbr[k][s], :]^T dY_out[out_row[s] (or s), :] over the slots of the
 * tiles whose mask has bit k.  Deterministic two-pass reduction through `workspace`. */
int lg_conv_wgrad_simt(const lgConvPlan* plan, const float* X_in, int32_t Cin, const float* dY_out, int32_t Cout,
                       float* dW, void* workspace, size_t workspace_bytes, void* stream);

/* fp32 -> 16-bit operand rows, value * scale[0] when scale != NULL (device float). */
int lg_cast_rows(const float* src, void* dst16, int64_t n_elems, int32_t fmt, const float* scale, void* stream);
/* scale_out float[4]: [0] = power of two bringing absmax(src) into [2^11, 2^12), [1] = 1/[0],
 * [2] scratch. */
int lg_absmax_scale(const float* src, int64_t n_elems, float* scale_out, void* stream);
/* W fp32 [K][Cin][Cout] -> w16 [K][Cin][Cout] and w16t [K][Cout][Cin] (either may be NULL). */
int lg_prep_weights(const float* W, int32_t K, int32_t Cin, int32_t Cout, void* w16, void* w16t, int32_t fmt,
                    void* stream);

/* tcgen05 gather-GEMM (forward and dgrad of MinkowskiConvolution / MinkowskiConvolutionTranspose,
 * utils/models/minkunet_bev.py:57-123):  Y[out_row[s], :] = out_scale * sum_k A16[nbr[k][s], :] @ B16[wk]^T
 * A16 [n_in][Ck] and B16 [K][N][Ck] are 16-bit (fmt), Ck % 32 == 0, N % 16 == 0, N <= 512.
 * out_scale: nullable device float (undoes lg_absmax_scale).  bias nullable [N].
 * Super-tile pipeline: cp.async row gathers arriving on mbarriers, weight panels by TMA, up to 4 row tiles
 * accumulating in TMEM per weight load (csrc/conv_tc2.cu). */
int lg_conv_gemm_tc(const lgConvPlan* plan, const void* A16, int32_t Ck, const void* B16, int32_t N, int32_t flip_k,
                    int32_t fmt, const float* out_scale, const float* bias, float* Y, void* stream);

size_t lg_conv_wgrad_tc_workspace(const lgConvPlan* plan, int32_t Cin, int32_t Cout);
/* tcgen05 wgrad: dW[k] = out_scale * sum_s X16[nbr[k][s], :]^T dY16[out_row[s], :]  (fp32 [K][Cin][Cout]). */
int lg_conv_wgrad_tc(const lgConvPlan* plan, const void* X16, int32_t Cin, const void* dY16, int32_t Cout,
                     int32_t fmt, const float* out_scale, float* dW, void* workspace, size_t workspace_bytes,
                     void* stream);

/* ---- layer-level entry points: ONE host call per MinkowskiConvolution each way (same contract as lg_conv_gemm_tc /
 * lg_conv_wgrad_tc; utils/models/minkunet_bev.py:57-123).
 * Forward: optionally (prep != 0) refreshes the 16-bit weight copies w16 [K][Cin][Cout] / w16t [K][Cout][Cin] from the
 * fp32 parameter W -- the caller keeps them until the parameter changes -- then runs the gather-GEMM.
 * stat_partials (nullable, float [4 * n_slots / 128][2 * Cout]): per-(tile, epilogue warp) column sums and sums of
 * squares of Y, written by the GEMM epilogue for the batch norm that follows (lgBnBranch.stat_partials), so the
 * statistics pass over Y is never run (SURVEY.md 8f-1).  Needs Cout a multiple of 32 per column block. */
int lg_conv_layer_forward(const lgConvPlan* plan, const void* X16, int32_t Cin, const float* W, int32_t Cout, void* w16,
                          void* w16t, int32_t prep, int32_t fmt, const float* bias, float* Y, float* stat_partials,
                          void* stream);
/* Backward: dX = inv_scale * dgrad (skipped when dX is NULL), dW = inv_scale * wgrad (skipped when dW is NULL);
 * dY16 is the 16-bit gradient scaled by 1 / inv_scale[0] (inv_scale nullable).  Split-K partials: library arena. */
int lg_conv_layer_backward(const lgConvPlan* plan_dgrad, const lgConvPlan* plan_wgrad, int32_t flip_dgrad,
                           const void* X16, int32_t Cin, const void* dY16, int32_t Cout, const void* w16, int32_t fmt,
                           const float* inv_scale, float* dX, float* dW, void* stream);
/* MinkowskiConvolution -> MinkowskiBatchNorm (eval: running statistics) [-> += residual] [-> MinkowskiReLU] in one
 * launch.  bn_stats float[4C] in the lg_bn_apply layout ([mean, invstd, scale, shift]; only scale / shift are read).
 * res nullable fp32 [n_out, Cout]; Y fp32 required; Y16 nullable.  Cout column blocks must be multiples of 32.
 * W, w16, w16t, prep, fmt as lg_conv_layer_forward; no bias (no tensor-core layer before a batch norm has one).
 * Y and Y16 are bit-identical to lg_conv_layer_forward followed by lg_bn_apply(Y, bn_stats, res, relu). */
int lg_conv_layer_infer(const lgConvPlan* plan, const void* X16, int32_t Cin, const float* W, int32_t Cout, void* w16,
                        void* w16t, int32_t prep, int32_t fmt, const float* bn_stats, const float* res, int32_t relu,
                        float* Y, void* Y16, void* stream);

/* Library-owned scratch arena (one block per device and stream, outside any caching allocator): bytes currently held,
 * and release (synchronises).  The layer-level calls size it themselves. */
size_t lg_arena_bytes(void);
int lg_arena_release(void);

/* ------------------------------------------------------------------ fused batch norm (+ ReLU, residual, operand cast)
 *
 * ME.MinkowskiBatchNorm / MinkowskiSyncBatchNorm are torch BatchNorm1d on the N x C feature matrix, chained with
 * ME.MinkowskiReLU and BasicBlock's `out += residual` at utils/models/minkunet_bev.py:308-368 (SyncBN conversion:
 * train_lidog.py:228).  A layer is two HBM passes each way here; the sums between the passes are what SyncBN
 * exchanges (the caller all-reduces `sums` and `count`).  C % 4 == 0, C <= 1024.  Deterministic.
 *   stats float[4C] = [mean, invstd, scale = gamma*invstd, shift = beta - mean*scale] */
size_t lg_bn_workspace(int64_t n, int32_t C);
/* sums double[2C + 1] = [sum x, sum x^2, n] of this rank's n rows. */
int lg_bn_stats(const float* x, int64_t n, int32_t C, double* sums, void* workspace, size_t workspace_bytes,
                void* stream);
/* count = rows over all ranks (read from the device double *count_dev when that is non-NULL: the all-reduced
 * count of SyncBN never visits the host); gamma/beta/running_* / num_batches_tracked (int64) nullable; running_var
 * gets the unbiased variance, momentum as torch (new = (1-m)*old + m*batch). */
int lg_bn_finalize(const double* sums, double count, const double* count_dev, int32_t C, const float* gamma,
                   const float* beta, float eps,
                   float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                   float* stats_out, void* stream);
/* y = act(x*scale + shift [+ x2*scale2 + shift2] [+ res]), act = ReLU when relu != 0; y16 (nullable) receives the
 * 16-bit copy (fmt) the next tensor-core convolution gathers. */
int lg_bn_apply(const float* x, const float* stats, const float* x2, const float* stats2, const float* res,
                int32_t relu, int64_t n, int32_t C, float* y, void* y16, int32_t fmt, void* stream);
/* g = dy * [y > 0] (relu) or dy.  sums double[3C] = [sum g, sum g*(x-mean), sum g*(x2-mean2)],
 * maxes float[3C] = [max|g|, max|x-mean|, max|x2-mean2|] per channel. */
int lg_bn_bwd_stats(const float* dy, const float* y, const float* x, const float* stats, const float* x2,
                    const float* stats2, int32_t relu, int64_t n, int32_t C, double* sums, float* maxes,
                    void* workspace, size_t workspace_bytes, void* stream);
/* branch 0 (x) or 1 (x2): coef float[3C] = [a, b, c], dx = a*g + b*(x-mean) + c; dgamma/dbeta (nullable) from
 * sums_local (this rank), coefficients from sums_global (all ranks; = sums_local without SyncBN);
 * scale_out float[3] = {2^k with bound*2^k in [2^11, 2^12), 2^-k, bound >= max|dx|}. */
int lg_bn_bwd_finalize(const double* sums_local, const double* sums_global, const float* maxes, double count,
                       const double* count_dev, int32_t C, int32_t branch, const float* gamma, const float* stats, float* coef, float* dgamma,
                       float* dbeta, float* scale_out, void* stream);
int lg_bn_bwd_gscale(const float* maxes, int32_t C, float* scale_out, void* stream);
/* dx (+ scaled 16-bit copy), optionally dx2 for the second BN branch and dres = g for a plain residual. */
int lg_bn_bwd_apply(const float* dy, const float* y, const float* x, const float* stats, const float* coef,
                    const float* x2, const float* stats2, const float* coef2, int32_t relu, int64_t n, int32_t C,
                    float* dx, void* dx16, const float* scale, float* dx2, void* dx2_16, const float* scale2,
                    float* dres, void* dres16, const float* scale_r, int32_t fmt, void* stream);

/* ---- layer-level entry points: ONE host call per MinkowskiBatchNorm(+ReLU, +residual) each way.
 *
 * The host path of a training step was as long as its GPU time (round 1: 44 ms of Python for a 45 ms step), so the
 * reference-facing layer (lidog_b200/me/norm.py) makes one call per fused layer instead of 5-9.  Scratch comes from the
 * library's own arena (lg_arena_bytes), nothing is allocated per call; the SyncBN exchange (train_lidog.py:228) runs
 * INSIDE the tail kernel of the statistics pass over NVLink peer memory when `peer` is given (see lg_peer_sum for the
 * protocol; the call consumes 1 epoch per branch forward, 1 epoch backward).
 *   stats float[4C + 2]: [mean, invstd, scale, shift] x C, then the row count over all ranks as one double. */
typedef struct lgPeerCtx {
  void* const* bufs; /* HOST array: device address in this process of every rank's exchange buffer */
  int32_t world, rank;
  uint64_t epoch; /* first epoch this call may use (1, 2, ...; identical sequence on every rank) */
} lgPeerCtx;
typedef struct lgBnBranch {
  const float* x;             /* [n, C] input of this BN */
  const float* stat_partials; /* nullable: [n_stat_rows, 2C] per-tile (sum, sum of squares) rows written by the */
  int64_t n_stat_rows;        /*   epilogue of the convolution that produced x (lg_conv_layer_forward) */
  const float *gamma, *beta;  /* nullable */
  float *running_mean, *running_var; /* nullable; updated as torch does (momentum, unbiased variance) */
  int64_t* num_batches_tracked;      /* nullable */
  float eps, momentum;
  float* stats; /* out [4C + 2], kept by the caller for the backward */
} lgBnBranch;
/* y = act(BN_a(x_a) [+ BN_b(x_b)] [+ res]); y16 (nullable) = the 16-bit operand copy of y. */
int lg_bn_layer_forward(const lgBnBranch* a, const lgBnBranch* b /* nullable */, const float* res /* nullable */,
                        int32_t relu, int64_t n, int32_t C, float* y, void* y16, int32_t fmt,
                        const lgPeerCtx* peer /* nullable */, void* stream);
typedef struct lgBnBwdBranch {
  const float* x;
  const float* stats; /* [4C + 2] from the forward */
  const float* gamma; /* nullable */
  float* dx;          /* out [n, C]; nullable when dx16 is given (the consumer reads the 16-bit copy only) */
  void* dx16;         /* nullable out: dx * scale in the 16-bit format, for the convolution backward */
  float *dgamma, *dbeta; /* nullable out [C] (this rank's sums: DDP reduces parameter gradients) */
} lgBnBwdBranch;
/* Backward of the above.  scales float[12]: [4i .. 4i+2] = {2^k, 2^-k, bound} of branch i's dx16. dres (nullable)
 * receives g = dy * [y > 0], the gradient of the plain residual.  y (the forward output) is only read for the ReLU
 * mask; y == NULL with relu says "the forward had neither a residual nor a second branch": the mask is then
 * recomputed from x with the forward's own expression (bit-identical) and the two passes read 8 bytes per element
 * less; with a residual or a second branch y is required (LG_ERR_INVALID otherwise). */
int lg_bn_layer_backward(const float* dy, int64_t dy_ld /* row pitch of dy in floats (>= C): the gradient of one input
                         of ME.cat is a column slice of a wider matrix and is consumed in place */,
                         const float* y, int32_t relu, int64_t n, int32_t C, const lgBnBwdBranch* a,
                         const lgBnBwdBranch* b /* nullable */, float* dres, int32_t fmt, float* scales,
                         const lgPeerCtx* peer /* nullable */, void* stream);

/* ------------------------------------------------------------------ instance norm (+ ReLU, operand cast)
 *
 * ME.MinkowskiInstanceNorm, the normalisation of the IBN-Net and RobustNet baselines next to LiDOG (SURVEY.md 2):
 * instance b = the rows whose batch index coords[r][0] is b (any row order), 1 <= B <= 256 (LG_ERR_UNSUPPORTED above;
 * rows with a batch index outside [0, B) are left out of the statistics and come out NaN).  Any C >= 1.
 *   y = act(((x - mean_b) * (var_b + eps)^-1/2) * weight + bias), biased variance, act = ReLU when relu != 0;
 *   y16 (nullable) = the 16-bit copy (fmt) of y the next tensor-core convolution gathers, equal to lg_cast_rows(y);
 *   stats double [2][B][C] = mean, invstd (0, 0 for an instance without rows), kept by the caller for the backward.
 * Features 16-byte aligned when C % 4 == 0.  Scratch: library arena.  Deterministic (fixed-order reductions). */
int lg_instnorm_forward(const float* x, const int32_t* coords, int64_t n, int32_t C, int32_t B, const float* weight,
                        const float* bias, float eps, int32_t relu, float* y, void* y16, int32_t fmt, double* stats,
                        void* stream);
/* Backward: g = dy * [y > 0] (relu; y is the forward output, else unused and nullable), xhat the normalised x,
 * dx = invstd * weight * (g - mean_b(g) - xhat * mean_b(g * xhat)), dweight = sum g * xhat, dbias = sum g (all
 * required outputs, dweight / dbias [C]). */
int lg_instnorm_backward(const float* dy, const float* x, const float* y, const int32_t* coords, int64_t n, int32_t C,
                         int32_t B, const float* weight, int32_t relu, const double* stats, float* dx, float* dweight,
                         float* dbias, void* stream);

/* ------------------------------------------------------------------ per-scan feature covariance (ISW loss)
 *
 * The statistic of RobustNet's instance-selective whitening loss, one of the baselines next to LiDOG (SURVEY.md 2.2):
 * scan b = the rows whose batch index coords[r][0] is b (any row order), n_b of them, X_b their features (not centred).
 *   cov float [B][C][C] = X_b^T X_b / (n_b - 1) + eps * I, exactly symmetric; eps * I when n_b <= 1;
 *   counts int32 [B] = n_b, kept by the caller for the backward.
 * 1 <= B <= 256 and 1 <= C <= 256 (LG_ERR_UNSUPPORTED outside), n < 2^31 - 1; rows with a batch index outside [0, B)
 * are left out.  Features 16-byte aligned when C % 4 == 0.  Scratch: library arena.  Deterministic (fixed-order
 * double merges, no float atomics). */
int lg_inst_cov_forward(const float* x, const int32_t* coords, int64_t n, int32_t C, int32_t B, float eps, float* cov,
                        int32_t* counts, void* stream);
/* Backward: G float [B][C][C] = dL/dcov, counts from the forward;
 * dx_r = x_r (G_b + G_b^T) / (n_b - 1) for the rows of scan b, 0 when n_b <= 1, NaN for rows outside [0, B).
 * Every element of dx is written. */
int lg_inst_cov_backward(const float* x, const int32_t* coords, int64_t n, int32_t C, int32_t B, const float* G,
                         const int32_t* counts, float* dx, void* stream);

/* ------------------------------------------------------------------ SyncBN exchange over peer memory
 *
 * train_lidog.py:228 converts every MinkowskiBatchNorm to SyncBN: 124 latency-bound exchanges of <= 3C doubles per
 * step.  lg_peer_sum replaces the NCCL call of each: one kernel publishes this rank's vector in its exchange
 * buffer, raises an epoch flag and adds the peers' vectors read over NVLink, in rank order (bit-identical on all
 * ranks).  peer_bufs: HOST array of `world` device addresses (in this process) of every rank's exchange buffer of
 * lg_peer_exchange_bytes() bytes, zero-initialised (torch symmetric memory / cudaIpc mappings). */
size_t lg_peer_exchange_bytes(void);
int lg_peer_sum(const double* local, int32_t n, void* const* peer_bufs, int32_t world, int32_t rank, uint64_t epoch,
                double* out, void* stream);

/* ------------------------------------------------------------------ LiDOG's DICE criteria (SURVEY.md 8f-2)
 *
 * soft = 0: DICELoss(ignore_label) -- the BEV criterion (utils/losses/losses.py:56-97; trainer_lighting_2d.py:181);
 * soft = 1: SoftDICELoss(ignore_label, eps, is_kitti) -- the 3D criterion (:129-187, soft targets :100-126;
 *           trainer_lighting_2d.py:194; is_kitti when num_classes == 19, :97-98).
 * logits float [n, C] (C <= 32), target int64 [n].  Forward: loss (device float) and coef float[2C] for the backward.
 * Backward: dlogits [n, C] = grad_scale[0] (device float, nullable = 1) * dLoss/dlogits.  Two HBM passes each way
 * instead of the reference's CPU round trip; fixed-order reductions. */
int lg_dice_forward(const float* logits, const int64_t* target, int64_t n, int32_t C, int32_t ignore_label,
                    int32_t soft, float eps, int32_t is_kitti, float* loss, float* coef, void* stream);
int lg_dice_backward(const float* logits, const int64_t* target, int64_t n, int32_t C, int32_t ignore_label,
                     int32_t soft, float eps, int32_t is_kitti, const float* coef, const float* grad_scale,
                     float* dlogits, void* stream);

/* ------------------------------------------------------------------ evaluation metric
 *
 * ADDS the confusion matrix of one batch into conf int64 [(C + 1) x C]: row = target class, row C = every target
 * outside [0, C) (the ignore label included), column = argmax_c logits[i, c] (first maximal index, torch's rule).
 * logits float [n, C] (1 <= C <= 32), target int64 [n].  n = 0 does nothing.  Exact and run-to-run identical.
 * IoU as torchmetrics JaccardIndex(ignore_index): rows 0..C-1; as sklearn jaccard_score(labels=range(C)): all rows. */
int lg_confusion_matrix(const float* logits, int64_t n, int32_t C, const int64_t* target, int64_t* conf, void* stream);

/* ------------------------------------------------------------------ BEV projection */

/* Bytes of the workspace that lg_bev_forward fills and lg_bev_backward reads, for the same arguments.  It holds the
 * pixel map, the row-occupancy words and the winning cell of every pooling window (one byte per output element:
 * ~340 MB at batch 8, C = 96, 2000 x 2000 -> 666 x 666). */
size_t lg_bev_workspace(int64_t n, int32_t C, int32_t batch_size, int32_t H, int32_t W, int32_t pk, int32_t ps,
                        int32_t pp);

/* Fused point-to-BEV projection: pixel scatter + raw (H,W,C)->(C,H,W) re-view + MaxPool2d(pk,ps,pp),
 * never materialising the dense tensor.  Replaces MinkUNetBaseBEV.sparse2super + filter_bounds
 * (utils/models/minkunet_bev.py:158-230).  out: float [batch, C, h, w], h = (H + 2pp - pk)/ps + 1, stored
 * NCHW (layout 0) or NHWC / channels_last (layout 1: the same logical tensor, the memory order cuDNN's
 * tensor-op convolutions of the dense 2D head consume without staging copies).
 * workspace keeps the pixel map, the row-occupancy words and each window's winning cell for lg_bev_backward. */
int lg_bev_forward(const int32_t* coords4, const float* feats, int64_t n, int32_t C, int32_t batch_size, float bound,
                   float voxel_size, int32_t H, int32_t W, int32_t pk, int32_t ps, int32_t pp, int32_t policy,
                   int32_t layout, float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the above (autograd of index_put_ + max_pool2d at minkunet_bev.py:217-221).
 * grad_feats [n, C] is fully written (rows outside the image get 0).  Atomic-free and bit-reproducible: every occupied
 * cell sums the <= 4 windows it won in ascending (i, j) order (the order of torch's CPU max_pool2d backward).
 * workspace: as the forward left it. */
int lg_bev_backward(const int32_t* coords4, const float* feats, int64_t n, int32_t C, int32_t batch_size,
                    int32_t H, int32_t W, int32_t pk, int32_t ps, int32_t pp, int32_t policy, int32_t layout,
                    const float* grad_out, float* grad_feats, const void* workspace, size_t workspace_bytes,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LIDOG_B200_H */
