/* geob200 -- C ABI of the B200-native GeoTransformer registration hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  Every entry point takes plain pointers and sizes; device
 * pointers unless the name ends in `_h`; `stream` is a cudaStream_t passed as void*.  All functions
 * return 0 on success and a negative code on failure, with a message available from geob200_last_error()
 * (the reference raises c10::Error -> RuntimeError through TORCH_CHECK, common/torch_helper.h:6-35; the
 * Python host layer turns a non-zero return into RuntimeError to keep that behaviour).
 *
 * Scratch memory is provided by the caller: each op has a *_workspace_bytes() query.
 * Index tables are int64 and sentinels equal the number of support rows, as in the reference.
 */
#ifndef GEOB200_H
#define GEOB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* geob200_last_error(void);
/* number of CUDA kernels this library has launched since it was loaded (bench.py: gpu_launches) */
uint64_t geob200_launch_count(void);

/* ---- collate -------------------------------------------------------------------------------------------- */

/* Replaces ext.grid_subsampling (reference geotransformer/extensions/pybind.cpp:13-17,
 * cpu/grid_subsampling/grid_subsampling.cpp:5-62): per-cloud voxel barycentres, bit-identical values AND order.
 * points (n_points,3) f32; lengths_h host int64[batch]; s_points must hold n_points*3 floats (upper bound);
 * s_lengths device int64[batch] receives the per-cloud counts (their sum = rows written). */
size_t geob200_grid_subsample_workspace_bytes(int64_t n_points, int64_t batch);
int geob200_grid_subsample(const float* points, int64_t n_points, const int64_t* lengths_h, int64_t batch, float voxel,
                           float* s_points, int64_t* s_lengths, void* workspace, size_t workspace_bytes, void* stream);

/* Replaces ext.radius_neighbors (reference pybind.cpp:8-12, cpu/radius_neighbors/radius_neighbors.cpp:5-68)
 * fused with the column slice of modules/ops/radius_search.py:25-26.
 * For every query row: indices (offset by the cloud start) of the support points of the same batch element with
 * d2 < r*r, ascending by d2, first `width` of them, padded with the sentinel n_support.
 * max_count (device int32) receives the global maximum neighbour count (the reference's row width); a negative
 * value signals an unsupported density (> 16384 neighbours for one query).  counts (device int32[n_query]) and
 * out may be NULL (count-only pass when width == 0). */
size_t geob200_radius_search_workspace_bytes(int64_t n_query, int64_t n_support, int64_t batch);
int geob200_radius_search(const float* q_points, int64_t n_query, const float* s_points, int64_t n_support,
                          const int64_t* q_lengths_h, const int64_t* s_lengths_h, int64_t batch, float radius,
                          int64_t width, int64_t* out, int32_t* counts, int32_t* max_count, void* workspace,
                          size_t workspace_bytes, void* stream);

/* calibrate_neighbors_stack_mode (utils/data.py:190-217): hist[c] += #rows of a neighbour table (n_rows, width) with
 * exactly c entries < n_support, for c < hist_n (int32 device histogram, accumulated across calls). */
int geob200_neighbor_histogram(const int64_t* neighbors, int64_t n_rows, int64_t width, int64_t n_support, int64_t hist_n,
                               int32_t* hist, void* stream);

/* ---- KPConv-FPN backbone --------------------------------------------------------------------------------- */

/* KPConv.forward (reference geotransformer/modules/kpconv/kpconv.py:79-122), fused gather -> kernel-point
 * influence -> contraction -> neighbour-count normalisation -> bias.  neighbors (n_query, n_neighbors) int64 with
 * sentinel n_support; kernel_points (15,3); weights (15, c_in, c_out); bias may be NULL.
 * c_in == 1, or c_in, c_out multiples of 32 with c_out <= 512. */
size_t geob200_kpconv_workspace_bytes(int64_t n_support);
int geob200_kpconv(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors,
                   int64_t n_query, int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel,
                   const float* weights, const float* bias, int64_t c_in, int64_t c_out, float sigma, float* out,
                   void* workspace, size_t workspace_bytes, void* stream);

/* nn.Linear: y[m,n] = x[m,k] . weight[n,k]^T + bias (UnaryBlock.mlp, modules.py:78; every transformer Linear).
 * ldx / ldy are row strides in floats (inputs may be column slices). */
/* Same op, two-stage tensor-core formulation: gather kernel (wf = influence-weighted neighbour features, M x 15 c_in) followed by
 * the 3xTF32 tcgen05 GEMM with the neighbour-count scale and bias in its epilogue.  weights_t is the (15*c_in, c_out) weight
 * matrix transposed to (c_out, 15*c_in). */
size_t geob200_kpconv_tc_workspace_bytes(int64_t n_query, int64_t n_support, int64_t c_in);
int geob200_kpconv_tc(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors, int64_t n_query,
                      int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel, const float* weights_t,
                      const float* bias, int64_t c_in, int64_t c_out, float sigma, float* out, void* workspace, size_t workspace_bytes,
                      void* stream);

/* 1 (default): Linears run on tcgen05 with 3xTF32 when the shape allows; 0: fp32 CUDA cores only */
void geob200_set_linear_mode(int mode);
int geob200_linear(const float* x, int64_t ldx, const float* weight, const float* bias, float* y, int64_t ldy, int64_t m,
                   int64_t n, int64_t k, int relu, void* stream);
int geob200_linear_batched(const float* x, int64_t ldx, int64_t stride_x, const float* weight, int64_t ldw, int64_t stride_w,
                           const float* bias, int64_t stride_b, float* y, int64_t ldy, int64_t stride_y, int64_t m, int64_t n,
                           int64_t k, int64_t batch, int relu, void* stream);

/* GroupNorm over all n_rows of the stacked pair (modules.py:33-50) + optional residual add + optional LeakyReLU:
 * y = leaky((x - mean_g) * rstd_g * gamma + beta + residual).
 * Every GroupNorm-bearing entry point below takes a scratch workspace of at least geob200_group_norm_workspace_bytes(n_rows,
 * channels, groups, n_pairs) bytes (n_pairs = 1 for the unbatched forms; 0 for a shape the entry points reject).  It needs no
 * initialisation.  channels <= 8192. */
size_t geob200_group_norm_workspace_bytes(int64_t n_rows, int64_t channels, int64_t groups, int64_t n_pairs);
int geob200_group_norm(const float* x, int64_t n_rows, int64_t channels, int64_t groups, const float* gamma,
                       const float* beta, float eps, const float* residual, int leaky, float slope, float* y,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Fused blocks: Linear -> GroupNorm (+ residual) (+ LeakyReLU) = UnaryBlock and the unary parts of ResidualBlock
 * (modules/kpconv/modules.py:33-104,150-225); KPConv -> GroupNorm -> LeakyReLU = ConvBlock and the conv part of
 * ResidualBlock (modules.py:107-147,205-207).  On the tcgen05 path the GroupNorm statistics are produced by the GEMM
 * epilogue, so the activations are not re-read for them.  pre_norm receives the Linear / KPConv output, y the result.
 * The GroupNorm workspace: geob200_group_norm_workspace_bytes(m or n_query, n or c_out, groups, 1); the KPConv workspace of
 * geob200_kpconv_group_norm: geob200_kpconv_tc_workspace_bytes. */
int geob200_linear_group_norm(const float* x, int64_t ldx, const float* weight, const float* bias, int64_t m, int64_t n, int64_t k,
                              int64_t groups, const float* gamma, const float* beta, float eps, const float* residual, int leaky,
                              float slope, float* pre_norm, float* y, void* workspace, size_t workspace_bytes, void* stream);
int geob200_kpconv_group_norm(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors,
                              int64_t n_query, int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel,
                              const float* weights_t, const float* bias, int64_t c_in, int64_t c_out, float sigma, int64_t groups,
                              const float* gamma, const float* beta, float eps, int leaky, float slope, float* pre_norm, float* y,
                              void* gn_workspace, size_t gn_workspace_bytes, void* workspace, size_t workspace_bytes, void* stream);

/* Batched forms (several pairs per forward, rows in stack order [ref_1..ref_B, src_1..src_B], cloud_rows_h[2 * n_pairs] host row
 * counts): the statistics are taken per PAIR (cloud c belongs to pair c % n_pairs), everything else is identical.  One pair
 * is one segment: the result equals the unbatched form's bit for bit.
 * Workspace: geob200_group_norm_workspace_bytes(n_rows or m, channels or n, groups, n_pairs). */
int geob200_group_norm_batched(const float* x, int64_t n_rows, int64_t channels, int64_t groups, const float* gamma, const float* beta,
                               float eps, const float* residual, int leaky, float slope, float* y, void* workspace, size_t workspace_bytes,
                               void* stream, int64_t n_pairs, const int64_t* cloud_rows_h);
int geob200_linear_group_norm_batched(const float* x, int64_t ldx, const float* weight, const float* bias, int64_t m, int64_t n, int64_t k,
                                      int64_t groups, const float* gamma, const float* beta, float eps, const float* residual, int leaky,
                                      float slope, float* pre_norm, float* y, void* workspace, size_t workspace_bytes, void* stream,
                                      int64_t n_pairs, const int64_t* cloud_rows_h);

/* maxpool over neighbour rows with a zero shadow row (functional.py:54-67) */
int geob200_maxpool(const float* x, const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors,
                    int64_t channels, float* y, void* stream);

/* Batched maxpool over a table that is wider than a pair's own (radius_search.py:25-26 cuts to the pair's max count):
 * columns past min(n_neighbors, max(cloud_max[p], cloud_max[B + p])) are ignored for the rows of pair p. */
int geob200_cloud_max_count(const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors, int64_t n_pairs,
                            const int64_t* cloud_rows_h, int32_t* cloud_max, void* stream);
int geob200_maxpool_batched(const float* x, const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors,
                            int64_t channels, float* y, int64_t n_pairs, const int64_t* cloud_rows_h, const int32_t* cloud_max,
                            void* stream);

/* y[m] = [ x_pad[up_indices[m*up_stride]] | skip[m] ]: nearest_upsample (functional.py:6-22) fused with the
 * torch.cat of the decoder (backbone.py:75-76).  skip may be NULL (c2 = 0). */
int geob200_upsample_concat(const float* x, const int64_t* up_indices, int64_t up_stride, int64_t n_support,
                            const float* skip, int64_t n_query, int64_t c1, int64_t c2, float* y, void* stream);

/* ---- point-to-node grouping ------------------------------------------------------------------------------ */

/* point_to_node_partition (reference geotransformer/modules/ops/pointcloud_partition.py:60-107).
 * node_masks / node_knn_masks are uint8 (torch.bool); node_sizes int32.  Exact for any number of points per node (chunked
 * selection); status (may be NULL) is kept for ABI stability and always receives 0. */
int geob200_point_to_node_partition(const float* points, int64_t n_points, const float* nodes, int64_t n_nodes,
                                    int64_t point_limit, int64_t* point_to_node, uint8_t* node_masks, int32_t* node_sizes,
                                    int64_t* node_knn_indices, uint8_t* node_knn_masks, int32_t* status, void* stream);

/* knn_partition (pointcloud_partition.py:35-57): for every node the k nearest points, ascending by the matmul-form squared
 * distance pairwise_distance(nodes, points) (ties by index).  knn_sq_distances (n_nodes, k) may be NULL.  1 <= k <= min(n_points, 2048). */
int geob200_knn_partition(const float* points, int64_t n_points, const float* nodes, int64_t n_nodes, int64_t k,
                          int64_t* knn_indices, float* knn_sq_distances, void* stream);
/* pairwise_distance (ops/pairwise_distance.py:4-31) of row-major x (n, c), y (m, c): out (n, m) = clamp(x2 - 2xy + y2, 0),
 * or 2 - 2xy when normalized != 0 */
int geob200_pairwise_distance(const float* x, int64_t n, const float* y, int64_t m, int64_t channels, int normalized, float* out,
                              void* stream);
/* get_point_to_node_indices (pointcloud_partition.py:9-32): indices[i] = argmin_j pairwise_distance(points, nodes)[i, j];
 * node_sizes (int32[n_nodes], may be NULL) = points per node */
int geob200_point_to_node_indices(const float* points, int64_t n_points, const float* nodes, int64_t n_nodes, int64_t* indices,
                                  int32_t* node_sizes, void* stream);
/* apply_transform (ops/transformation.py:7-60) for one (4,4) device transform: out = points R^T + t */
int geob200_apply_transform(const float* points, int64_t n_points, const float* transform, float* out, void* stream);

/* out[r] = indices[r] < n_rows ? table[indices[r]] : 0  (index_select on a zero-padded table, ops/index_select.py) */
int geob200_gather_rows(const float* table, int64_t n_rows, int64_t channels, const int64_t* indices, int64_t n_indices,
                        float* out, void* stream);

/* ---- geometric transformer -------------------------------------------------------------------------------- */

/* GeometricStructureEmbedding.get_embedding_indices (geotransformer.py:27-55) for one cloud:
 * d_indices (n,n) = sqrt(pairwise_distance)/sigma_d, a_indices (n,n,3) = atan2(|ref x anc|, ref.anc) * factor_a */
int geob200_gse_indices(const float* points, int64_t n, float sigma_d, float factor_a, int64_t angle_k, float* d_indices,
                        float* a_indices, void* stream);

/* The same for n_clouds stacked clouds in ONE launch (cloud_rows_h: host row counts): points (sum rows, 3); the outputs are
 * concatenated cloud after cloud: d_indices (sum n_c^2), a_indices (sum n_c^2, 3) -- the layout geob200_gse_embed_pairs takes. */
int geob200_gse_indices_batched(const float* points, int64_t n_clouds, const int64_t* cloud_rows_h, float sigma_d, float factor_a,
                                int64_t angle_k, float* d_indices, float* a_indices, void* stream);

/* GeometricStructureEmbedding.forward (geotransformer.py:57-72) given the indices: sinusoid -> proj_d / proj_a ->
 * max over k -> sum, fused.  wd/wa are the nn.Linear weights (out,in); wd_t/wa_t their transposes (in,out).
 * mode 0: fp32 CUDA cores; 1: tcgen05 3xTF32; 2: tcgen05 1xTF32; 3: tcgen05 3xFP16 split (fp32-accurate, fastest). */
size_t geob200_gse_embed_workspace_bytes(int64_t n, int64_t channels);
int geob200_gse_embed(const float* d_indices, const float* a_indices, int64_t n, int64_t channels, const float* div_term,
                      const float* wd_t, const float* wa_t, const float* wd, const float* wa, const float* bd, const float* ba,
                      float* embeddings, int mode, void* workspace, size_t workspace_bytes, void* stream);

/* Same over a flat list of n_rows (anchor, point) index rows -- the (i, j) pairs of several clouds concatenated:
 * d_indices (n_rows,), a_indices (n_rows, 3) -> embeddings (n_rows, channels).  One launch for a whole batch of clouds. */
int geob200_gse_embed_pairs(const float* d_indices, const float* a_indices, int64_t n_rows, int64_t channels, const float* div_term,
                            const float* wd_t, const float* wa_t, const float* wd, const float* wa, const float* bd, const float* ba,
                            float* embeddings, int mode, void* workspace, size_t workspace_bytes, void* stream);

/* The same embedding through TABULATED projections (csrc/gse_table.cu).  proj_d(sinusoid(x)) and proj_a(sinusoid(x)) are
 * functions of one scalar, band-limited to 1 rad per index unit: geob200_gse_table_build tabulates both once per set of weights
 * on a uniform grid of step 1/inv_step (power of two) over [0, d_max] / [0, a_max] (fp64 accumulation; node = fp32 values + fp16
 * forward differences), geob200_gse_embed_table then needs 4 lookups + 3 max + 1 add per (row, channel) instead of the
 * 2 * (1 + 3) * C^2 flop contraction.  Linear-interpolation error <= max|g''| / (8 inv_step^2) (< 1e-6 at inv_step 256 for
 * unit-scale weights).  Index values outside the tabulated range are evaluated directly (sincosf + dot products with wd / wa),
 * so results never depend on d_max / a_max -- only the speed does.  channels: 128 or 256.  The same (channels, inv_step, d_max,
 * a_max) must be passed to both calls; table: geob200_gse_table_bytes(...) bytes of device memory, 16-byte aligned. */
size_t geob200_gse_table_bytes(int64_t channels, int64_t inv_step, float d_max, float a_max);
int geob200_gse_table_build(const float* div_term, const float* wd_t, const float* wa_t, const float* bd, const float* ba,
                            int64_t channels, int64_t inv_step, float d_max, float a_max, void* table, size_t table_bytes,
                            void* stream);
int geob200_gse_embed_table(const float* d_indices, const float* a_indices, int64_t n_rows, int64_t channels, const void* table,
                            size_t table_bytes, int64_t inv_step, float d_max, float a_max, const float* div_term, const float* wd,
                            const float* wa, const float* bd, const float* ba, float* embeddings, void* stream);

/* Fused multi-head attention: softmax((q.k + qp.E + qb)/sqrt(d)) v  (rpe_transformer.py:51-70 with proj_p moved onto
 * q; vanilla_transformer.py:50-68 when qp = qb = embed = NULL).  q (n_query,C), k,v (n_key,C), qp (n_query,H,C),
 * qb (n_query,H), embed (n_query,n_key,C).  With a workspace and C = 128 or 256 the streaming path runs (one coalesced
 * pass over embed on a (query, key-chunk) grid + a softmax/P.V kernel); workspace = NULL selects the single-kernel path. */
size_t geob200_attention_workspace_bytes(int64_t n_query, int64_t n_key, int64_t heads);
int geob200_attention(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const float* qp,
                      const float* qb, const float* embed, int64_t n_query, int64_t n_key, int64_t channels, int64_t heads,
                      float* out, int64_t ldo, void* workspace, size_t workspace_bytes, void* stream);
/* A batch of independent attention problems that share channels, heads and row strides (the clouds / pairs of a batched
 * forward) in ONE launch pair; all items with embed (self-attention) or all without (cross-attention). */
typedef struct { const float* q; const float* k; const float* v; const float* qp; const float* qb; const float* embed; float* out;
                 int64_t n_query, n_key; } geob200_att_item_t;
size_t geob200_attention_batched_workspace_bytes(const geob200_att_item_t* items_h, int64_t n_items, int64_t heads);
int geob200_attention_batched(const geob200_att_item_t* items_h, int64_t n_items, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo,
                              int64_t channels, int64_t heads, void* workspace, size_t workspace_bytes, void* stream);
/* self-attention kernels: 1 (default) = TMA-staged E stream (cp.async.bulk ring, q.k and P.v as tiled passes), 0 = the
 * lanes<->channels cp.async kernels */
int geob200_set_attention_tma(int on);
int geob200_head_bias(const float* q, int64_t ldq, const float* bias_p, int64_t n, int64_t channels, int64_t heads, float* qb,
                      void* stream);
/* y = LayerNorm(a + b) (b may be NULL) */
int geob200_add_layernorm(const float* a, const float* b, const float* gamma, const float* beta, int64_t n, int64_t channels,
                          float eps, float* y, void* stream);
/* F.normalize(x, p=2, dim=1) */
int geob200_l2_normalize(const float* x, int64_t n, int64_t channels, float* y, void* stream);

/* ---- matching ---------------------------------------------------------------------------------------------- */

/* SuperPointMatching.forward (superpoint_matching.py:13-50); num_out (device int32) = number of rows written =
 * min(num_correspondences, #valid ref nodes x #valid src nodes); rows past it receive index -1 / score 0. */
size_t geob200_superpoint_matching_workspace_bytes(int64_t n_ref, int64_t n_src);
int geob200_superpoint_matching(const float* ref_feats, const float* src_feats, int64_t n_ref, int64_t n_src, int64_t channels,
                                const uint8_t* ref_masks, const uint8_t* src_masks, int64_t num_correspondences, int dual,
                                int64_t* ref_corr_indices, int64_t* src_corr_indices, float* corr_scores, int32_t* num_out,
                                void* workspace, size_t workspace_bytes, void* stream);

/* patch gathers of model.py:169-174: indices/masks/points of the k points of each selected superpoint; a negative
 * corr index (padding row of geob200_superpoint_matching) yields an empty patch (sentinel indices, masks 0) */
int geob200_gather_patches(const int64_t* corr_indices, int64_t n_corr, const int64_t* node_knn_indices,
                           const uint8_t* node_knn_masks, int64_t k, const float* points, int64_t n_points,
                           int64_t* out_indices, uint8_t* out_masks, float* out_points, void* stream);

/* matching_scores = einsum('bnd,bmd->bnm') / sqrt(C) over zero-padded feature tables (model.py:176-188) */
int geob200_patch_scores(const float* ref_feats, int64_t n_ref, const float* src_feats, int64_t n_src, int64_t channels,
                         const int64_t* ref_knn_indices, const int64_t* src_knn_indices, int64_t n_patches, int64_t k,
                         float* scores, void* stream);

/* LearnableLogOptimalTransport.forward (learnable_sinkhorn.py:20-66): out (n_patches, k+1, k+1) */
int geob200_sinkhorn(const float* scores, const uint8_t* row_masks, const uint8_t* col_masks, const float* alpha,
                     int64_t n_patches, int64_t k, int64_t num_iterations, float inf, float* out, void* stream);

/* ---- local-to-global registration -------------------------------------------------------------------------- */

/* LocalGlobalRegistration.forward (local_global_registration.py:196-235), use_dustbin=False, use_global_score=False,
 * correspondence_limit=None.  log_scores (P, score_ld, score_ld) with score_ld = k or k+1 (dustbin row/col ignored).
 * Correspondence outputs have capacity P*k*topk rows; num_corr (device int32) = rows written, in (patch,i,j) order.
 * patch_transforms (P,4,4), patch_inliers (P, -1 = patch below correspondence_threshold), best_patch may be NULL. */
size_t geob200_lgr_workspace_bytes(int64_t n_patches, int64_t k, int64_t topk);
int geob200_local_global_registration(const float* ref_knn_points, const float* src_knn_points, const uint8_t* ref_knn_masks,
                                      const uint8_t* src_knn_masks, const float* log_scores, int64_t n_patches, int64_t k,
                                      int64_t score_ld, int64_t topk, float acceptance_radius, int mutual,
                                      float confidence_threshold, int64_t correspondence_threshold, int64_t num_refinement_steps,
                                      float* ref_corr_points, float* src_corr_points, float* corr_scores, int32_t* corr_patch,
                                      int32_t* num_corr, float* estimated_transform, float* patch_transforms, int32_t* patch_inliers,
                                      int32_t* best_patch, void* workspace, size_t workspace_bytes, void* stream);

/* weighted_procrustes (modules/registration/procrustes.py:6-73): transforms (batch,4,4); weights may be NULL */
int geob200_weighted_procrustes(const float* src_points, const float* ref_points, const float* weights, int64_t batch,
                                int64_t n, float weight_thresh, float eps, float* transforms, void* stream);

/* get_node_correspondences (modules/registration/matching.py:231-315): ground-truth superpoint pairs and their overlap
 * ratios under `transform` (4x4, device).  Masks are uint8 (torch.bool) or NULL (= all valid).  corr_indices (capacity
 * n_ref*n_src rows of 2 int64) and corr_overlaps (capacity n_ref*n_src) receive the pairs with overlap > 0 in row-major
 * (ref, src) order, `count` (device int32) their number. */
size_t geob200_node_correspondences_workspace_bytes(int64_t n_ref, int64_t n_src, int64_t k);
int geob200_node_correspondences(const float* ref_nodes, const float* src_nodes, const float* ref_knn_points,
                                 const float* src_knn_points, const uint8_t* ref_masks, const uint8_t* src_masks,
                                 const uint8_t* ref_knn_masks, const uint8_t* src_knn_masks, int64_t n_ref, int64_t n_src,
                                 int64_t k, const float* transform, float pos_radius, int64_t* corr_indices,
                                 float* corr_overlaps, int32_t* count, void* workspace, size_t workspace_bytes, void* stream);

/* Evaluator.forward (experiments/<exp>/loss.py:95-159; metrics.py:47-112): metrics[8] (device) =
 * {PIR, IR, RRE [deg], RTE, RMSE, RR, #correspondences, #gt superpoint pairs}.  mode 0 = 3DMatch (RMSE of the realigned
 * source cloud, RR = RMSE < rmse_threshold), 1 = KITTI (no RMSE: NaN; RR = RRE < rre_threshold and RTE < rte_threshold),
 * 2 = ModelNet (RMSE of T_est x - T_gt x; RR as KITTI).  Means over empty sets are NaN, as torch reports them. */
int geob200_evaluate(const int64_t* gt_node_corr_indices, const float* gt_node_corr_overlaps, int64_t n_gt,
                     float acceptance_overlap, const int64_t* ref_node_corr_indices, const int64_t* src_node_corr_indices,
                     int64_t n_node_corr, const float* ref_corr_points, const float* src_corr_points, int64_t n_corr,
                     float acceptance_radius, const float* gt_transform, const float* est_transform, const float* src_points,
                     int64_t n_src_points, int mode, float rmse_threshold, float rre_threshold, float rte_threshold,
                     float* metrics, void* stream);

/* Same with the three row counts optionally taken from DEVICE memory (int32, produced by geob200_node_correspondences /
 * geob200_superpoint_matching / geob200_local_global_registration): a non-NULL *_dev pointer overrides the host value
 * (n_node_corr: the smaller of the two), so a whole forward can be enqueued without a host read-back in between. */
int geob200_evaluate_counts(const int64_t* gt_node_corr_indices, const float* gt_node_corr_overlaps, int64_t n_gt, const int32_t* n_gt_dev,
                            float acceptance_overlap, const int64_t* ref_node_corr_indices, const int64_t* src_node_corr_indices,
                            int64_t n_node_corr, const int32_t* n_node_corr_dev, const float* ref_corr_points, const float* src_corr_points,
                            int64_t n_corr, const int32_t* n_corr_dev, float acceptance_radius, const float* gt_transform,
                            const float* est_transform, const float* src_points, int64_t n_src_points, int mode, float rmse_threshold,
                            float rre_threshold, float rte_threshold, float* metrics, void* stream);

/* Profiling aid (bench.py roofline): while enabled, every tcgen05 GEMM launch (nn.Linear and the KPConv contraction) is
 * bracketed by CUDA events on its stream; _read synchronises them and returns the count, shapes[3i..] = (m, n, k), ms[i]. */
int geob200_linear_profile_enable(int on);
/* split-K for deep-K GEMMs on few tiles (default on); off = every tile runs its whole K loop in one CTA */
int geob200_set_split_k(int on);
/* persistent tile loop with two TMEM accumulator sets for GEMMs of more than one wave of tiles (default on) */
int geob200_set_linear_persistent(int on);
int64_t geob200_linear_profile_read(int64_t capacity, int64_t* shapes, float* ms);

/* ---- native stage drivers (native.cu) ------------------------------------------------------------------------
 * The whole KPConv-FPN backbone / geometric transformer as ONE call: same kernels in the same order as the per-op entry
 * points above (bitwise-identical results), driven from C++ so that the host cost per pair is a few hundred microseconds
 * instead of milliseconds.  All pointers are device pointers; the structs are plain C (built from a state_dict by
 * geotransformer_b200/native.py). */
#define GEOB200_MAX_STAGES 6
typedef struct { const float* weight; const float* bias; int64_t c_in, c_out; } geob200_linear_t;
typedef struct { const float* gamma; const float* beta; } geob200_norm_t;
typedef struct { const float* weights; const float* weights_t; const float* bias; const float* kernel_points;
                 int64_t c_in, c_out; float sigma; } geob200_kpconv_t;
/* ResidualBlock (reference geotransformer/modules/kpconv/modules.py:151-225) */
typedef struct {
    int32_t has_unary1, has_shortcut, strided, reserved;
    int64_t c_in;
    geob200_linear_t unary1; geob200_norm_t norm1;
    geob200_kpconv_t conv;   geob200_norm_t norm_conv;
    geob200_linear_t unary2; geob200_norm_t norm2;
    geob200_linear_t shortcut; geob200_norm_t norm_sc;
} geob200_resblock_t;
/* KPConvFPN (reference experiments/.../backbone.py): encoder1_1 = conv1+norm1, blocks[0] = encoder1_2, then three blocks per
 * further level; decoders[0] is the coarsest decoder, the last one (level finest_decoder) has no norm/activation. */
typedef struct {
    int32_t num_stages, finest_decoder, groups, init_dim;
    geob200_kpconv_t conv1; geob200_norm_t norm1;
    geob200_resblock_t blocks[1 + 3 * (GEOB200_MAX_STAGES - 1)];
    geob200_linear_t decoders[GEOB200_MAX_STAGES];
    geob200_norm_t decoder_norms[GEOB200_MAX_STAGES];
} geob200_backbone_t;
size_t geob200_backbone_workspace_bytes(const geob200_backbone_t* net, const int64_t* level_rows);
/* out_feats[0] = coarsest encoder output (rows level_rows[S-1]); out_feats[i>0] = decoder outputs, coarse to fine.
 * GroupNorm workspace: geob200_backbone_gn_workspace_bytes with n_pairs = 1. */
int geob200_backbone_forward(const geob200_backbone_t* net, const float* feats, const float* const* points, const int64_t* level_rows,
                             const int64_t* const* neighbors, const int64_t* neighbor_width, const int64_t* const* subsampling,
                             const int64_t* subsampling_width, const int64_t* const* upsampling, const int64_t* upsampling_width,
                             float* const* out_feats, void* gn_workspace, size_t gn_workspace_bytes, void* workspace,
                             size_t workspace_bytes, void* stream);

/* Batched form (several pairs per forward, stack order [ref_1..ref_B, src_1..src_B] at every level like the reference collate
 * with batch_size B, utils/data.py:144): identical kernels over the stacked rows; the GroupNorm statistics are taken per pair
 * (modules/kpconv/modules.py:46-50 normalises over the stacked rows of ONE pair).  cloud_rows_h[level][2 * n_pairs]: host row
 * counts per cloud.  n_pairs <= 32.  The GroupNorm workspace needs geob200_backbone_gn_workspace_bytes (the largest
 * geob200_group_norm_workspace_bytes of the network).  n_pairs = 1 is the unbatched forward: cloud_rows_h and sub_cloud_max
 * may be NULL, and are ignored.
 * sub_cloud_max[level][2 * n_pairs] (device int32, geob200_cloud_max_count of the subsampling tables): the strided blocks'
 * maxpool must see every pair's table at the width the pair's own collate would have cut it to (geob200_maxpool_batched). */
size_t geob200_backbone_gn_workspace_bytes(const geob200_backbone_t* net, const int64_t* level_rows, int64_t n_pairs);
int geob200_backbone_forward_batched(const geob200_backbone_t* net, const float* feats, const float* const* points,
                                     const int64_t* level_rows, const int64_t* const* neighbors, const int64_t* neighbor_width,
                                     const int64_t* const* subsampling, const int64_t* subsampling_width,
                                     const int64_t* const* upsampling, const int64_t* upsampling_width, float* const* out_feats,
                                     void* gn_workspace, size_t gn_workspace_bytes, void* workspace, size_t workspace_bytes, void* stream,
                                     int64_t n_pairs, const int64_t* const* cloud_rows_h, const int32_t* const* sub_cloud_max);

/* one transformer layer ('self' with the structure embedding, or 'cross'); w_qkv = [Wq;Wk;Wv] (3C,C), w_kv = [Wk;Wv], wp_t = Wp^T */
typedef struct {
    int32_t is_self, reserved;
    const float* w_qkv; const float* b_qkv; const float* w_q; const float* b_q; const float* w_kv; const float* b_kv;
    const float* wp_t; const float* bp;
    geob200_linear_t att_linear; geob200_norm_t att_norm;
    geob200_linear_t expand; geob200_linear_t squeeze; geob200_norm_t out_norm;
} geob200_tlayer_t;
size_t geob200_transformer_workspace_bytes(int64_t n0, int64_t n1, int64_t channels, int64_t heads, int64_t num_layers);
/* RPEConditionalTransformer.forward on stacked features x = [feats0; feats1] (after in_proj), sequential cross updates */
int geob200_transformer_forward(const geob200_tlayer_t* layers, int64_t num_layers, int64_t channels, int64_t heads, const float* x,
                                int64_t n0, int64_t n1, const float* emb0, const float* emb1, float* out, void* workspace,
                                size_t workspace_bytes, void* stream);

/* Batched form: x rows in stack order [ref_1..ref_B, src_1..src_B] (cloud_rows_h[2B], host); embeddings_h[c] = device pointer
 * of the structure embedding (rows_c, rows_c, C) of cloud c.  Linears / LayerNorms run once over all rows; attention is one
 * batched launch pair per phase (geob200_attention_batched).  Same arithmetic per pair as geob200_transformer_forward. */
size_t geob200_transformer_batched_workspace_bytes(int64_t n_pairs, const int64_t* cloud_rows_h, int64_t channels, int64_t heads,
                                                   int64_t num_layers);
int geob200_transformer_forward_batched(const geob200_tlayer_t* layers, int64_t num_layers, int64_t channels, int64_t heads,
                                        const float* x, int64_t n_pairs, const int64_t* cloud_rows_h, const float* const* embeddings_h,
                                        float* out, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GEOB200_H */
