/* libctl_b200.so -- C ABI of the B200-native centroid-triplet re-ID hot path.
 *
 * The reference (mikwieczorek/centroids-reid @ a1825b7) is pure Python: the path it exposes
 * is a Python module/class API called by PyTorch-Lightning hooks, there is no FFI of its
 * own.  This header is the boundary a maintainer binds instead of the torch/numpy calls at
 * the cited reference lines (see INTEGRATION.md for the ctypes stub); the Python package
 * `centroids-reid_b200` is that binding plus drop-in classes with the reference's names.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked host;
 *     buffers are caller-owned (the Python shim allocates them with torch's caching
 *     allocator) and must be contiguous and 16-byte aligned;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing
 *     synchronises unless stated;
 *   - return value: 0 = ok, negative = CTL_ERR_* (argument / capacity error),
 *     positive = cudaError_t; ctl_last_error() returns a thread-local description;
 *   - there is NO CPU fallback: without an sm_100 device every compute entry point fails.
 */
#ifndef CTL_B200_H_
#define CTL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTL_ABI_VERSION 1

#define CTL_OK 0
#define CTL_ERR_INVALID_ARGUMENT (-1)
#define CTL_ERR_WORKSPACE (-2)   /* workspace too small; ctl_last_error() names the size */
#define CTL_ERR_UNSUPPORTED (-3)
#define CTL_ERR_CAPACITY (-4)    /* a device-side list overflowed (see the entry point) */
#define CTL_ERR_NO_DEVICE (-5)

typedef void* ctl_stream_t; /* cudaStream_t */

const char* ctl_last_error(void);
int ctl_abi_version(void);
/* 0 when the current device is sm_100 (B200); CTL_ERR_NO_DEVICE otherwise. */
int ctl_device_check(void);

/* ------------------------------------------------------------------------------------------
 * Query x gallery distances, top-k and streamed CMC / mAP ranks
 * replaces: utils/reid_metric.py:25-33 (get_euclidean), :51-59 (get_cosine), :112-136
 * (R1_mAP.compute: normalize, distmat, np.argsort), utils/eval_reid.py:25-92 (eval_func),
 * inference/get_similar.py:104-128 (dist + argsort + [:, :topk]).
 * ---------------------------------------------------------------------------------------- */
#define CTL_DIST_EUCLIDEAN 0 /* squared L2, unclamped: |q|^2 + |g|^2 - 2 q.g */
#define CTL_DIST_COSINE 1    /* clamp(|1 - cos|, 1e-12) */
#define CTL_FLAG_NORMALIZE 2 /* torch.nn.functional.normalize(x, dim=1, p=2) first */
#define CTL_DIST_SQRT 4      /* euclidean only: sqrt(clamp(d, 1e-12)) -- losses/triplet_loss.py:27-41 */
#define CTL_FLAG_EXACT_PASS 8 /* ctl_l2_topk: threshold pass over EVERY gallery tile (default: a subset of the tiles --
                                 same results from a looser threshold and longer candidate lists) */

/* Row planes: the fp32 rows split into two fp16 planes (hi + 2^-11 lo, per-row power-of-two
 * scale) plus fp32 squared norms, the operand format of the tensor-core distance kernel.
 * Opaque to the caller; ctl_planes_bytes() gives the buffer size. */
size_t ctl_planes_bytes(int64_t n, int32_t d);
int ctl_planes_build(const float* x, int64_t n, int32_t d, int32_t flags, void* planes, ctl_stream_t stream);

/* out[nq, ld_out] = dist(q, g): the full matrix (get_euclidean / get_cosine drop-in). */
int ctl_dist_matrix(const void* q_planes, int64_t nq, const void* g_planes, int64_t ng, int32_t d, int32_t flags,
                    float* out, int64_t ld_out, ctl_stream_t stream);

/* Per-query k smallest distances in ascending (distance, gallery index) order, without
 * materialising the matrix.  out_idx = local gallery row + g_index_offset.  Requires
 * k <= ng.  *overflow (device int, written asynchronously) becomes non-zero if more rows
 * than the candidate capacity tie exactly at the selection threshold; the results are then
 * invalid and the shim raises CTL_ERR_CAPACITY after its result read-back. */
size_t ctl_topk_workspace_bytes(int64_t nq, int64_t ng, int32_t k);
int ctl_l2_topk(const void* q_planes, int64_t nq, const void* g_planes, int64_t ng, int32_t d, int32_t flags,
                int32_t k, int64_t g_index_offset, int64_t* out_idx, float* out_dist, int32_t* overflow,
                void* workspace, size_t workspace_bytes, ctl_stream_t stream);

/* Streamed evaluation (eval_func semantics).  Identity / camera arrays: q_pid, g_pid int32;
 * q_cam = dense camera index in [0,64); g_cammask = bit set of the cameras a gallery row
 * (or centroid, utils/eval_reid.py:52-56 respect_camids) was built from.  A gallery row is
 * junk for a query iff same pid and bit q_cam of its mask is set; it is a positive iff
 * same pid and not junk.
 *   collect : pos_keys[nq, max_pos] <- (distance, gallery index) keys of each query's
 *             positives (unordered), pos_count[nq] (zeroed by the caller);
 *   sort    : ascending sort of every row of a key matrix (counts[i] valid entries);
 *   count   : buckets[nq, max_pos + 1] (zeroed by the caller) += for every kept gallery row,
 *             the index of the first positive that sorts after it;
 *   finalize: ranks[nq, max_pos] (1-based rank of each positive among kept rows),
 *             ap[nq] (float64, eval_reid.py:75-79), -1 / NaN for queries without positives.
 * With a gallery sharded over ranks: collect per shard, all-gather + sort the keys, count
 * per shard, all-reduce(sum) the buckets, finalize. */
int ctl_eval_collect(const void* q_planes, int64_t nq, const void* g_planes, int64_t ng, int32_t d, int32_t flags,
                     const int32_t* q_pid, const int32_t* q_cam, const int32_t* g_pid, const uint64_t* g_cammask,
                     int64_t g_index_offset, int32_t max_pos, uint64_t* pos_keys, int32_t* pos_count,
                     int32_t* overflow, ctl_stream_t stream);
int ctl_sort_key_rows(uint64_t* keys, const int32_t* counts, int64_t rows, int32_t row_stride, ctl_stream_t stream);
int ctl_eval_count(const void* q_planes, int64_t nq, const void* g_planes, int64_t ng, int32_t d, int32_t flags,
                   const int32_t* q_pid, const int32_t* q_cam, const int32_t* g_pid, const uint64_t* g_cammask,
                   int64_t g_index_offset, int32_t max_pos, const uint64_t* pos_keys_sorted,
                   const int32_t* pos_count, int32_t* buckets, ctl_stream_t stream);
int ctl_eval_finalize(const int32_t* buckets, const int32_t* pos_count, int64_t nq, int32_t max_pos, int32_t* ranks,
                      double* ap, ctl_stream_t stream);
/* ctl_eval_finalize that also fills `packed` ([nq + 1][3] doubles: per query AP, first-hit rank (-1: none), number of
 * positives; last row: {*overflow, 0, 0}) -- everything eval_func's final reductions (utils/eval_reid.py:86-92) need, so
 * the host does ONE device->host copy per evaluation. */
int ctl_eval_finalize_packed(const int32_t* buckets, const int32_t* pos_count, int64_t nq, int32_t max_pos, int32_t* ranks,
                             double* ap, double* packed, const int32_t* overflow, ctl_stream_t stream);
/* One generic pass of the distance GEMM with any combination of the streamed epilogues (the
 * entry points above are compositions of this one).  NULL pointers disable a feature.
 * With both top-k and evaluation wanted, TWO passes serve both:
 *   pass 1: gmin (+ pos_keys/pos_count)            -> ctl_select_tau, ctl_sort_key_rows
 *   pass 2: tau + cand_keys (+ thr_keys + buckets) -> ctl_sort_key_rows, ctl_topk_emit,
 *                                                     ctl_eval_finalize */
typedef struct ctl_pass_desc {
  float* dist_out;            /* [nq, ld_out] full matrix */
  int64_t ld_out;
  float* gmin;                /* [nq, n_groups] minima of 16-column groups, n_groups = ceil(ng/16) */
  const float* tau;           /* [nq] candidate threshold */
  uint64_t* cand_keys;        /* [nq, cand_cap] rows with dist <= tau */
  int32_t* cand_count;        /* [nq], zeroed by the caller */
  int32_t cand_cap;
  const int32_t* q_pid;       /* identities: see ctl_eval_collect */
  const int32_t* q_cam;
  const int32_t* g_pid;
  const uint64_t* g_cammask;
  uint64_t* pos_keys;         /* [nq, max_pos] (collect) */
  int32_t* pos_count;         /* [nq], zeroed by the caller */
  int32_t max_pos;
  const uint64_t* thr_keys;   /* [nq, max_pos] sorted positives (count) */
  const int32_t* thr_count;
  int32_t* buckets;           /* [nq, max_pos + 1], zeroed by the caller */
  int32_t* overflow;          /* device int, set non-zero when a list overflows */
  int64_t g_index_offset;
  /* Optional (NULL = off). */
  const int32_t* tile_list;    /* ctl_dist_worklist: run only these 128 x 128 tiles.  For passes whose outputs do not need
                                  every tile: pos_keys / pos_count (tiles that can hold a positive) and gmin (any subset of
                                  the groups still bounds the k-th distance from above; the caller pre-fills gmin with
                                  +inf).  Rejected with dist_out, cand_keys or buckets. */
  const int32_t* g_index_map;  /* [ng] index written into the keys for gallery row i (instead of i + g_index_offset):
                                  lets the rows be stored in another order (e.g. sorted by pid) with unchanged results */
} ctl_pass_desc;
int ctl_dist_pass(const void* q_planes, int64_t nq, const void* g_planes, int64_t ng, int32_t d, int32_t flags,
                  const ctl_pass_desc* desc, ctl_stream_t stream);
/* debug aid: per-CTA epilogue cycle counters [grid][2][8] written by the following ctl_dist_pass calls */
void ctl_debug_set_dist_profile(long long* device_buffer);
/* top-k plan for (ng, k): emit_all != 0 means "skip pass 1, tau = +inf". */
int ctl_topk_plan(int64_t ng, int32_t k, int32_t* emit_all, int32_t* n_groups, int32_t* merge, int32_t* cand_cap);
int ctl_select_tau(const float* gmin, int64_t nq, int32_t n_groups, int32_t merge, int32_t k, float* tau,
                   ctl_stream_t stream);
/* Tile list for ctl_pass_desc.tile_list: tile_list[0] = count, then the kept tile ids (ascending; id = gallery tile *
 * ceil(nq/128) + query tile).  A tile is kept if
 * the identity ranges of its 128 query rows and its 128 gallery rows intersect (q_pid / g_pid in the planes' row order;
 * both NULL = no identities) or if its gallery-tile index is a multiple of keep_stride (0 = none).  With both operands
 * stored in identity order the first set is a few per cent of the matrix.  ctl_dist_subset_stride(ng, k): the stride that
 * leaves ~2.5 k column groups for ctl_select_tau (1 = use every tile).  Limits: <= 2^20 tiles, <= 5632 row tiles
 * (CTL_ERR_UNSUPPORTED beyond: run the pass without a list). */
size_t ctl_dist_worklist_bytes(int64_t nq, int64_t ng);
int ctl_dist_subset_stride(int64_t ng, int32_t k);
int ctl_dist_worklist(const int32_t* q_pid, int64_t nq, const int32_t* g_pid, int64_t ng, int32_t keep_stride,
                      int32_t* tile_list, ctl_stream_t stream);
int ctl_fill_f32(float* p, int64_t n, float value, ctl_stream_t stream);
int ctl_topk_emit(const uint64_t* cand_keys_sorted, const int32_t* cand_count, int64_t nq, int32_t cand_cap, int32_t k,
                  int64_t* out_idx, float* out_dist, int32_t* overflow, ctl_stream_t stream);
/* key <-> (distance, index) helpers for host-side merges of per-shard results */
uint64_t ctl_key_encode(float dist, uint32_t index);
void ctl_key_decode(uint64_t key, float* dist, uint32_t* index);

/* ------------------------------------------------------------------------------------------
 * Per-identity centroid mean (segmented reduction)
 * replaces: modelling/bases.py:92-95 (_calculate_centroids), the tensor part of
 * :179-262 (validation_create_centroids), inference/inference_utils.py:147-159.
 * out[s, :] = sum_{j in [indptr[s], indptr[s+1])} x[indices[j], :] / count  (CSR groups;
 * indices == NULL means contiguous rows j).
 * ---------------------------------------------------------------------------------------- */
int ctl_segment_mean(const float* x, int64_t n, int32_t d, const int64_t* indptr, const int64_t* indices,
                     int64_t n_seg, float* out, ctl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * CTL training-step losses, forward + backward in one enqueue
 * replaces: train_ctl_model.py:54-152 (everything between the trunk and manual_backward) and
 * the gradients autograd derives from it; modelling/bases.py:359-384 (create_masks_train);
 * losses/triplet_loss.py:27-41,68-173,194-205; losses/center_loss.py:26-45.
 * Batch contract (datasets/bases.py:346-406): B = P*K rows, pid-major blocks of K, padded rows
 * (is_real = 0) at the end of a block, every pid keeps >= 2 real rows.  labels[B] = class
 * index in [0, C).  All matrices fp32 row-major.
 * out_losses[8] = total, xent, triplet, center, ctl, dist_ap, dist_an, l2_mean_centroid (each
 * already multiplied by its SOLVER weight, like the reference's logged values).
 * Gradients are those of `total`: d_feats[B,D], d_centers[C,D] (dense, NOT yet rescaled by
 * 1/center_weight -- train_ctl_model.py:157-158 does that in the step), d_bn_weight[D],
 * d_fc_weight[C,D].  bn_running_mean/var are updated in place (momentum, unbiased var).
 * ---------------------------------------------------------------------------------------- */
typedef struct ctl_loss_config {
  int32_t B, D, P, K, C;
  float margin;         /* SOLVER.MARGIN (MarginRankingLoss) */
  float center_weight;  /* SOLVER.CENTER_LOSS_WEIGHT */
  float xent_weight;    /* SOLVER.QUERY_XENT_WEIGHT */
  float triplet_weight; /* SOLVER.QUERY_CONTRASTIVE_WEIGHT */
  float ctl_weight;     /* SOLVER.CENTROID_CONTRASTIVE_WEIGHT */
  float bn_eps;         /* 1e-5 */
  float bn_momentum;    /* 0.1 */
  float label_smooth;   /* 0.1 */
} ctl_loss_config;

size_t ctl_loss_workspace_bytes(const ctl_loss_config* cfg);
int ctl_loss_step(const ctl_loss_config* cfg, const float* feats, const int32_t* labels, const uint8_t* is_real,
                  const float* centers, const float* bn_weight, const float* bn_bias, float* bn_running_mean,
                  float* bn_running_var, const float* fc_weight, float* out_losses, float* d_feats, float* d_centers,
                  float* d_bn_weight, float* d_fc_weight, void* workspace, size_t workspace_bytes,
                  ctl_stream_t stream);

/* Stand-alone drop-ins (forward value + gradient of that value in one call):
 *   TripletLoss.__call__ (losses/triplet_loss.py:139-173; euclidean, margin ranking, optional
 *   anchor mask; any label multiset), CenterLoss.forward (losses/center_loss.py:26-45),
 *   CrossEntropyLabelSmooth.forward (losses/triplet_loss.py:194-205). */
size_t ctl_triplet_workspace_bytes(int32_t n, int32_t d);
int ctl_triplet_step(const float* feats, int32_t n, int32_t d, const int32_t* labels, const uint8_t* anchor_mask,
                     float margin, float* out_loss, float* out_dist_ap, float* out_dist_an, float* d_feats,
                     void* workspace, size_t workspace_bytes, ctl_stream_t stream);
/* The two remaining variants of TripletLoss (losses/triplet_loss.py:127-137,157-158): soft_margin != 0 = SoftMarginLoss
 * on (dist_an - dist_ap) (TripletLoss(margin=None): log(1 + exp(d_ap - d_an)), `margin` ignored); cosine != 0 =
 * dist_func 'cosine' (clamp(|1 - cos(x_i, x_j)|, 1e-12) with rows divided by max(|x|, 1e-12), triplet_loss.py:44-65),
 * gradient through the normalisation included. */
int ctl_triplet_step_ex(const float* feats, int32_t n, int32_t d, const int32_t* labels, const uint8_t* anchor_mask,
                        float margin, int32_t soft_margin, int32_t cosine, float* out_loss, float* out_dist_ap,
                        float* out_dist_an, float* d_feats, void* workspace, size_t workspace_bytes, ctl_stream_t stream);
int ctl_center_loss_step(const float* x, int32_t b, int32_t d, const int32_t* labels, const float* centers, int32_t c,
                         float* out_loss, float* d_x, float* d_centers, void* workspace, size_t workspace_bytes,
                         ctl_stream_t stream);
int ctl_xent_smooth_step(const float* logits, int32_t b, int32_t c, const int32_t* targets, float epsilon,
                         float* out_loss, float* d_logits, void* workspace, size_t workspace_bytes,
                         ctl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Trunk inference forward (ResNet50 / ResNet50-IBN-A), NHWC fp16 activations
 * replaces: modelling/backbones/resnet.py:51-133, resnet_ibn_a.py:18-141,
 * modelling/baseline.py:91-96, modelling/bases.py:169-177, inference/inference_utils.py:104-113.
 *   conv2d   : out = [relu]( conv(x, weight) + bias [+ residual] ), weight [Cout][k][k][Cin] fp16
 *              (eval BatchNorm folded in), 1x1 or 3x3 (pad k/2), stride 1 or 2, Cin/Cout % 64 == 0;
 *              any H, W >= 1 (torch.nn.Conv2d's output size: stride 2 gives ceil(H/2) x ceil(W/2));
 *              ReLU (if relu != 0) is applied to output channels >= relu_from only (IBN: the
 *              InstanceNorm half of bn1 is left raw for ctl_instnorm_relu);
 *   stem     : conv 7x7/2 pad 3 (3 -> 64) + folded BN [+ ReLU] from NCHW fp32 to NHWC fp16;
 *              weight_k64 = [147][64] fp32 with k = (c*7 + r)*7 + s;
 *   maxpool  : 3x3 / 2, pad 1;
 *   gap_bn   : feat = mean over H*W (fp32), emb = feat * bn_scale + bn_shift (eval BatchNorm1d);
 *   instnorm : per-(image, channel) InstanceNorm(affine) + ReLU in place on channels [0, half).
 * ---------------------------------------------------------------------------------------- */
int ctl_conv2d_nhwc_f16(const void* x, int32_t n, int32_t h, int32_t w, int32_t cin, const void* weight,
                        const float* bias, const void* residual, void* out, int32_t cout, int32_t ksize,
                        int32_t stride, int32_t relu, int32_t relu_from, ctl_stream_t stream);
/* Two 1x1 convolutions summed in ONE GEMM over the concatenated K dimension -- the last layer of a bottleneck's
 * first block, out = act(bn3(conv3(x1)) + bn_d(downsample(x2))) (resnet.py:75-85 with a downsample branch):
 *   out[n][i][j][:] = act( W[:, :cin1] x1[n][i][j][:] + W[:, cin1:] x2[n][i*stride2][j*stride2][:] + bias )
 * x1: NHWC fp16 [n][h2/stride2][w2/stride2][cin1]; x2: NHWC fp16 [n][h2][w2][cin2]; weight_cat: [cout][cin1 + cin2]
 * fp16 (both folded weight matrices side by side), bias = sum of the two folded biases.  The shortcut tensor is
 * never written to or re-read from HBM. */
int ctl_conv1x1_dual_nhwc_f16(const void* x1, int32_t cin1, const void* x2, int32_t h2, int32_t w2, int32_t cin2,
                              int32_t stride2, int32_t n, const void* weight_cat, const float* bias, void* out,
                              int32_t cout, int32_t relu, ctl_stream_t stream);
int ctl_stem_conv7x7(const float* x_nchw, int32_t n, int32_t h, int32_t w, const float* weight_k64, const float* bias,
                     int32_t relu, void* out_nhwc_f16, ctl_stream_t stream);
/* tensor-core stem: weight_k192_f16 = [64][192] fp16, k = (c*7 + r)*8 + s (s = 7 and k >= 168 zero) */
int ctl_stem_conv7x7_tc(const float* x_nchw, int32_t n, int32_t h, int32_t w, const void* weight_k192_f16,
                        const float* bias, int32_t relu, void* out_nhwc_f16, ctl_stream_t stream);
/* Fused stem for inputs up to 128 pixels wide (h % 4 == 0, w even): conv1 7x7/2 + folded bn1 (+ReLU for IBN-a) +
 * maxpool 3x3/2 in one pass; replaces resnet.py:123-126 / resnet_ibn_a.py:127-130.  `xpad` is a caller-owned
 * workspace of ctl_stem_pad_bytes(n, h, w) bytes that must have been zero-filled ONCE before its first use with a
 * given (n, h, w) (the call rewrites only the interior: zero-bordered NHWC4 fp16 copy of x).  `weight_packed_f16`
 * is [28][64][8] fp16: element (c, o, e) = folded weight w[o][ch = e % 4][r = c / 4][s = 2 * (c % 4) + e / 4],
 * zero for ch == 3 or s == 7.  Output: pooled NHWC fp16 [n][h/4][(w/2 - 1)/2 + 1][64]. */
size_t ctl_stem_pad_bytes(int32_t n, int32_t h, int32_t w);
int ctl_stem_pool_fused(const float* x_nchw, int32_t n, int32_t h, int32_t w, void* xpad, const void* weight_packed_f16,
                        const float* bias, int32_t relu, void* out_pooled_nhwc_f16, ctl_stream_t stream);
/* ctl_stem_pool_fused from uint8 HWC crops [n][h][w][3]: ToTensor + Normalize ((u / 255 - mean) / std, IEEE fp32 -- the
 * arithmetic of ctl_augment_batch_u8 without flip / crop / erasing; datasets/transforms/build.py:29-33) folded into the
 * stem's input packing, so a validation loader that ships uint8 crops never materialises the fp32 NCHW tensor.
 * Bit-identical to ctl_augment_batch_u8 (neutral parameters) followed by ctl_stem_pool_fused. */
int ctl_stem_pool_fused_u8(const void* x_u8_nhwc, int32_t n, int32_t h, int32_t w, const float* mean3_host,
                           const float* std3_host, void* xpad, const void* weight_packed_f16, const float* bias, int32_t relu,
                           void* out_pooled_nhwc_f16, ctl_stream_t stream);
int ctl_maxpool3x3s2_nhwc_f16(const void* x, int32_t n, int32_t h, int32_t w, int32_t c, void* out,
                              ctl_stream_t stream);
int ctl_gap_bn_nhwc_f16(const void* x, int32_t n, int32_t hw, int32_t c, const float* bn_scale, const float* bn_shift,
                        float* feat, float* emb, ctl_stream_t stream);
int ctl_instnorm_relu_nhwc_f16(void* x, int32_t n, int32_t hw, int32_t c, int32_t half, const float* gamma,
                               const float* beta, float eps, ctl_stream_t stream);

/* ---- whole-trunk entry points (SURVEY 8b): the eval embedding path bn(backbone(x)) behind an opaque handle ----
 * replaces: ResNet.forward / ResNet_IBN.forward (modelling/backbones/resnet.py:122-133, resnet_ibn_a.py:126-141),
 * Baseline.forward's pooling (modelling/baseline.py:91-96), ModelBase.validation_step / inference_utils._inference
 * (modelling/bases.py:169-177, inference/inference_utils.py:104-113).
 *   ctl_trunk_create   : ResNet50 (3,4,6,3 bottlenecks) or ResNet50-IBN-a (`ibn` != 0), MODEL.LAST_STRIDE 1 or 2.
 *   ctl_weights_pack   : `tensors` = the reference's `base.*`-stripped state_dict as DEVICE fp32 pointers, by name
 *                        ("conv1.weight", "bn1.running_var", "layer3.0.downsample.1.bias", "layer1.0.bn1.IN.weight", ...),
 *                        plus optionally "bn_head.weight|bias|running_mean|running_var" (ModelBase.bn, [2048]).  Folds every
 *                        eval BatchNorm into fp16 weights + fp32 biases on the device and keeps the packed operands in the
 *                        handle.  Call again whenever the parameters change (after opt.step(), load_state_dict).
 *   ctl_embed_forward  : x NCHW fp32 [n][3][h][w] on the device -> out_feat [n][2048] (global_feat) and / or out_emb
 *                        [n][2048] (= eval BatchNorm1d(global_feat); needs the bn_head.* tensors).  Activations live in the
 *                        caller's workspace of ctl_embed_workspace_bytes(...) bytes: five buffers, each the size of the
 *                        largest activation of the walk (odd sides round up at every stride-2 layer, as in torch).  Any
 *                        h, w >= 8.  All launches go to `stream`.
 * The handle is per device and not thread-safe; a missing / mis-sized tensor is CTL_ERR_INVALID_ARGUMENT naming it. */
typedef struct ctl_trunk ctl_trunk;
typedef struct ctl_named_tensor {
  const char* name;
  const float* data; /* device pointer */
  int64_t numel;
} ctl_named_tensor;
int ctl_trunk_create(ctl_trunk** out, int32_t ibn, int32_t last_stride);
void ctl_trunk_destroy(ctl_trunk* h);
int ctl_weights_pack(ctl_trunk* h, const ctl_named_tensor* tensors, int32_t n_tensors, ctl_stream_t stream);
size_t ctl_embed_workspace_bytes(const ctl_trunk* h, int32_t n, int32_t height, int32_t width);
int ctl_embed_forward(ctl_trunk* h, const float* x_nchw, int32_t n, int32_t height, int32_t width, float* out_feat,
                      float* out_emb, void* workspace, size_t workspace_bytes, ctl_stream_t stream);

/* ---- training-side trunk kernels (autograd through modelling/backbones/resnet.py:67-87 in train mode) ---- */

/* Weight gradient of ctl_conv2d_nhwc_f16's convolution (torch.nn.Conv2d backward w.r.t. weight):
 *   dw[co][r][s][ci] = sum_{n,ho,wo} dy[n][ho][wo][co] * x[n][ho*stride + r - pad][wo*stride + s - pad][ci]
 * x: NHWC fp16 [n][h][w][cin]; dy: NHWC fp16 [n][ho][wo][cout]; dw: fp32 [cout][k][k][cin] (the layout of the
 * forward's weight operand).  fp32 accumulation, deterministic (fixed split + fixed-order reduction).
 * `workspace` holds the per-split partial tiles: ctl_conv2d_wgrad_workspace_bytes(...) bytes. */
size_t ctl_conv2d_wgrad_workspace_bytes(int32_t n, int32_t h, int32_t w, int32_t cin, int32_t cout, int32_t ksize,
                                        int32_t stride);
int ctl_conv2d_wgrad_nhwc_f16(const void* x, int32_t n, int32_t h, int32_t w, int32_t cin, const void* dy, int32_t cout,
                              int32_t ksize, int32_t stride, void* workspace, size_t workspace_bytes, float* dw,
                              ctl_stream_t stream);
/* Same, with the epilogue a training step needs folded into the split-K reduction: dw is multiplied by out_scale (the
 * 1 / loss-scale un-scaling) and, with param_layout != 0, written as [cout][cin][k][k] -- torch.nn.Conv2d.weight's own
 * layout -- so the gradient needs no permute / mul pass. */
int ctl_conv2d_wgrad_nhwc_f16_ex(const void* x, int32_t n, int32_t h, int32_t w, int32_t cin, const void* dy, int32_t cout,
                                 int32_t ksize, int32_t stride, void* workspace, size_t workspace_bytes, float* dw,
                                 float out_scale, int32_t param_layout, ctl_stream_t stream);
/* Operand packs of every convolution of a training step in ONE launch: table = device array of
 * {const float* src [cout][cin][k][k]; void* fwd fp16 [cout][k][k][cin]; void* dgrad fp16 [cin][k][k][cout] with flipped
 * taps (may be NULL); int32 cout, cin, k, pad; int64 chunk_begin} (48 bytes; chunks of 8192 source elements). */
int ctl_train_pack_weights(const void* table_device, int32_t n_tensors, int64_t n_chunks, ctl_stream_t stream);

/* BatchNorm2d with batch statistics (torch.nn.BatchNorm2d in train mode, resnet.py:72-85) over NHWC fp16
 * [rows = N*H*W] rows of `pitch` elements, normalising the c channels that start at the given pointers (pitch == c
 * for a dense tensor; pitch > c addresses a channel slice, e.g. the BatchNorm half of an IBN layer); c a power of two
 * in [32, 2048].  forward: mean / biased variance over the rows (fp32 partial
 * sums combined in double, deterministic), running statistics updated in place when given (momentum, unbiased
 * variance), out = [relu](gamma * (y - mean) * invstd + beta [+ residual]) rounded to fp16; save_mean / save_invstd
 * feed the backward.  backward: g = dz * (z > 0) when the ReLU output z is given (g is written to g_out, which may
 * alias dz) else g = dz; dgamma = sum g * xhat, dbeta = sum g (both multiplied by grad_unscale, fp32);
 * dy = gamma * invstd * (g - mean_rows(g) - xhat * mean_rows(g * xhat)) rounded to fp16.
 * Workspace: ctl_bn_workspace_bytes(rows, c). */
size_t ctl_bn_workspace_bytes(int64_t rows, int32_t c);
int ctl_bn_train_forward_nhwc_f16(const void* y, int64_t rows, int32_t c, int32_t pitch, const float* gamma, const float* beta, float eps,
                                  float momentum, float* running_mean, float* running_var, const void* residual,
                                  int32_t relu, void* workspace, size_t workspace_bytes, float* save_mean,
                                  float* save_invstd, void* out, ctl_stream_t stream);
int ctl_bn_train_backward_nhwc_f16(const void* dz, const void* z, const void* y, int64_t rows, int32_t c, int32_t pitch, const float* gamma,
                                   const float* save_mean, const float* save_invstd, float grad_unscale, void* workspace,
                                   size_t workspace_bytes, void* g_out, float* dgamma, float* dbeta, void* dy,
                                   ctl_stream_t stream);
/* InstanceNorm2d(affine) + ReLU of an IBN layer's first `half` channels in train mode (resnet_ibn_a.py:18-32): y, out,
 * dz, z, dy are NHWC fp16 with rows of `pitch` elements ([n][hw][pitch]); instance statistics (biased variance) per
 * (image, channel) are saved as [n][half] fp32.  backward: g = dz * (z > 0) is written back over dz; dgamma_part /
 * dbeta_part are per-image partials [n][half] (sum over n = the parameter gradient), multiplied by grad_unscale. */
int ctl_instnorm_train_forward_nhwc_f16(const void* y, int32_t n, int32_t hw, int32_t pitch, int32_t half, const float* gamma,
                                        const float* beta, float eps, float* save_mean, float* save_invstd, void* out,
                                        ctl_stream_t stream);
int ctl_instnorm_train_backward_nhwc_f16(void* dz, const void* z, const void* y, int32_t n, int32_t hw, int32_t pitch,
                                         int32_t half, const float* gamma, const float* save_mean, const float* save_invstd,
                                         float grad_unscale, float* dgamma_part, float* dbeta_part, void* dy,
                                         ctl_stream_t stream);
/* Backward helpers of the trunk: global average pool (out[n][p][c] = dfeat[n][c] * scale, fp16), max-pool 3x3/2 pad 1
 * (gradient routed to the first maximum of every window, like torch), zero-insertion upsampling
 * out[n][2i][2j] = x[n][i][j] (+ add) (the transpose of a stride-2 subsampling), and the stem's im2col
 * ([n*ho*wo][192] fp16, k = (c*7 + r)*8 + s) that turns the 7x7 weight gradient into ctl_conv2d_wgrad_nhwc_f16
 * with cin = 192, ksize = 1. */
int ctl_gap_backward_nhwc_f16(const float* dfeat, int32_t n, int32_t hw, int32_t c, float scale, void* out,
                              ctl_stream_t stream);
int ctl_maxpool3x3s2_backward_nhwc_f16(const void* x, const void* dy, int32_t n, int32_t h, int32_t w, int32_t c, void* dx,
                                       ctl_stream_t stream);
/* Training pair of the pool: the forward also records which window tap (r*3 + s, one byte per output element,
 * [n][ho][wo][c] uint8) held the first maximum; the backward gathers from the <= 4 windows of a pixel. */
int ctl_maxpool3x3s2_argmax_nhwc_f16(const void* x, int32_t n, int32_t h, int32_t w, int32_t c, void* out, void* arg_u8,
                                     ctl_stream_t stream);
int ctl_maxpool3x3s2_backward_argmax_nhwc_f16(const void* arg_u8, const void* dy, int32_t n, int32_t h, int32_t w, int32_t c,
                                              void* dx, ctl_stream_t stream);
int ctl_upsample2_zero_nhwc_f16(const void* x, int32_t n, int32_t h, int32_t w, int32_t c, const void* add, void* out,
                                ctl_stream_t stream);
int ctl_stem_im2col_f16(const float* x_nchw, int32_t n, int32_t h, int32_t w, void* out, ctl_stream_t stream);

/* ---- optimizer step (solver/build.py:9-47, train_ctl_model.py:155-159, modelling/bases.py:102-133) ---- */

/* ---- train-mode trunk behind an opaque handle (SURVEY 8b: the train forward / backward variants) ----
 * replaces: torch autograd through ResNet.forward / ResNet_IBN.forward in train mode (modelling/backbones/resnet.py:67-87,
 * 122-133, resnet_ibn_a.py:18-32,126-141) + Baseline.forward's pooling (modelling/baseline.py:91-96) inside
 * CTLModel.training_step (train_ctl_model.py:38-179): x -> global_feat [n][2048], then d(loss)/d(global_feat) -> every
 * parameter gradient.  Same launches, same order, same bits as modelling/backbones/engine_train.py.
 *   ctl_trainer_create      : ResNet50 or ResNet50-IBN-a (`ibn` != 0), MODEL.LAST_STRIDE 1 or 2, BatchNorm momentum.
 *   ctl_trainer_bind        : `params` = the `base.*`-stripped fp32 parameters AND BatchNorm running buffers as device
 *                             pointers, by name (running_mean / running_var optional per layer, updated in place like
 *                             torch); `grads` = one fp32 output per PARAMETER, same name, the parameter's own layout
 *                             (conv [Cout][Cin][k][k]).  The handle keeps the pointers: re-bind when storage moves.
 *   ctl_train_workspace_bytes: bytes of the caller's workspace for one (n, h, w) step: the saved activations of the
 *                             forward + the scratch of the backward (≈ 60 MB per 256x128 image).  0 when the step
 *                             cannot run: h or w < 32, or an odd map at the input of a stride-2 layer (the backward
 *                             needs even maps there; ctl_last_error() names the layer and the map size).
 *   ctl_train_forward       : x NCHW fp32 -> out_feat [n][2048] fp32 (global_feat); saved tensors stay in `workspace`.
 *   ctl_train_backward      : dfeat [n][2048] fp32 = dLoss/dglobal_feat.  Activation gradients are computed on
 *                             grad_scale * dfeat in fp16 (loss scaling, the role of PL's GradScaler, utils/misc.py:111);
 *                             the parameter gradients are written UN-scaled.  Same workspace as the forward, once per forward.
 * Not thread-safe; all launches go to `stream`; 256-byte aligned workspace. */
typedef struct ctl_trainer ctl_trainer;
typedef struct ctl_named_buffer {
  const char* name;
  float* data; /* device pointer, written */
  int64_t numel;
} ctl_named_buffer;
int ctl_trainer_create(ctl_trainer** out, int32_t ibn, int32_t last_stride, float momentum);
void ctl_trainer_destroy(ctl_trainer* t);
int ctl_trainer_bind(ctl_trainer* t, const ctl_named_tensor* params, int32_t n_params, const ctl_named_buffer* grads,
                     int32_t n_grads);
size_t ctl_train_workspace_bytes(const ctl_trainer* t, int32_t n, int32_t height, int32_t width);
int ctl_train_forward(ctl_trainer* t, const float* x_nchw, int32_t n, int32_t height, int32_t width, float* out_feat,
                      void* workspace, size_t workspace_bytes, ctl_stream_t stream);
int ctl_train_backward(ctl_trainer* t, const float* dfeat, float grad_scale, void* workspace, size_t workspace_bytes,
                       ctl_stream_t stream);

/* One table entry per parameter tensor, resident on the device; chunk_begin = running sum of
 * ceil(numel / CTL_OPT_CHUNK) over the preceding entries. */
#define CTL_OPT_CHUNK 8192
typedef struct ctl_adam_entry {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t numel;
  int64_t chunk_begin;
} ctl_adam_entry;
/* torch.optim.Adam (L2 weight decay added to the gradient, bias-corrected, no amsgrad) on every tensor of the table
 * in one launch; `step` is the 1-based step count after this update; gradients are read as grad * grad_mul. */
int ctl_adam_multi_step(const void* table_device, int32_t n_tensors, int64_t n_chunks, float lr, float beta1, float beta2,
                        float eps, float weight_decay, int64_t step, float grad_mul, const int32_t* skip_flag,
                        ctl_stream_t stream);
/* torch.optim.SGD without momentum: param -= lr * grad * grad_mul (the center parameters; grad_mul =
 * 1 / SOLVER.CENTER_LOSS_WEIGHT, train_ctl_model.py:157-158). */
int ctl_sgd_step(float* param, const float* grad, int64_t numel, float lr, float grad_mul, const int32_t* skip_flag,
                 ctl_stream_t stream);
/* `skip_flag` (device int, may be NULL) of the two optimizer entry points: when non-zero at execution time the kernel
 * returns without touching parameters or moments -- GradScaler.step's "skip the step on inf / NaN gradients" without a
 * host synchronisation.  ctl_loss_scale_update is GradScaler.update() on the device: state3 = {scale, scale / base_scale,
 * base_scale / scale}; *found_inf is copied to *last_found and cleared. */
int ctl_loss_scale_update(float* state3, int32_t* tracker, int32_t* found_inf, int32_t* last_found, float base_scale,
                          float growth_factor, float backoff_factor, int32_t growth_interval, ctl_stream_t stream);
/* Gradient overflow check of dynamic loss scaling (torch.cuda.amp.GradScaler.unscale_ in the reference's PL AMP trainer,
 * utils/misc.py:111): table = device array of {float* grad; int64 numel; int64 chunk_begin} (chunks of 8192 elements, like
 * ctl_adam_multi_step); every gradient is multiplied in place by `mul` * (*mul_device if non-NULL: a device scalar such as
 * base_scale / scale) -- skipped when that factor is exactly 1 -- and *found_inf (device int,
 * OR-accumulated, cleared by the caller) becomes 1 if any element is inf or NaN. */
int ctl_grad_check_multi(const void* table_device, int32_t n_tensors, int64_t n_chunks, float mul, const float* mul_device,
                         int32_t* found_inf, ctl_stream_t stream);

/* ---- training-time augmentation (datasets/transforms/build.py:15-27, random_erasing.py:30-55) ---- */

/* images: uint8 NHWC [n][h][w][3], already resized (T.Resize stays on the host); params_device: int32 [n][8] =
 * {flip, crop_top, crop_left (offsets inside the padded image, 0..2*pad), erase_row, erase_col, erase_h, erase_w
 * (erase_h == 0: none), is_real (0: mock image -> zeros)}; mean / std: 3 floats on the HOST.
 * out = RandomErasing(Normalize(ToTensor(RandomCrop(Pad(Flip(image)))))) as fp32 NCHW [n][3][h][w]. */
int ctl_augment_batch_u8(const void* images_u8_nhwc, int32_t n, int32_t h, int32_t w, int32_t pad, const int32_t* params_device,
                         const float* mean3_host, const float* std3_host, float* out_nchw, ctl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CTL_B200_H_ */
