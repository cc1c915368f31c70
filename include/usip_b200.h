/* usip_b200.h -- C ABI of libusip_b200.so: the B200 (sm_100a) drop-in for the USIP detector /
 * descriptor hot path.  Plain pointers and sizes only: no torch types, no C++ in the signatures.
 *
 * Conventions (all functions):
 *   - every pointer is a DEVICE pointer unless the name says `host`; tensors are dense, row-major;
 *   - the caller owns and pre-allocates every buffer; the library keeps no global state;
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous, nothing synchronises;
 *   - the return value is 0 on success, otherwise a cudaError_t (or -1 for invalid arguments);
 *   - "(B,C,N)" etc. are the REFERENCE layouts (channel-major), "[P,C]" are this library's internal
 *     row-major point-major activations (row = one point / one group sample, C contiguous).
 *
 * Each entry point cites the reference interface it replaces (paths relative to lijx10/USIP).
 */
#ifndef USIP_B200_H_
#define USIP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define USIP_B200_ABI_VERSION 1
int usip_abi_version(void);
/* name of the last failing check/launch for the calling thread ("" if none); host pointer */
const char* usip_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * 1. Reference operator modules (plugin API B-1)
 * ---------------------------------------------------------------------------------------------- */

/* index_max.forward_cuda_shared_mem / forward_cuda          models/index_max_ext/index_max.cpp:132-148,
 * kernels models/index_max_ext/index_max_cuda.cu:9-25,29-61.
 * data (B,C,N) f32, index (B,N) i32 in [0,K) -> out_idx (B,C,K) i32: smallest n attaining
 * max{data[b,c,n] : index[b,n]==k, data > -1000}, else 0.  No B*K shared-memory cap.
 * scratch: B*C*K u64 (packed running max), may not alias anything. */
int usip_index_max_f32(const float* data, const int32_t* index, int32_t* out_idx,
                       unsigned long long* scratch, int B, int C, int N, int K, void* stream);

/* ball_query.forward_cuda_shared_mem                        models/ball_query_ext/ball_query.cpp:33-39,
 * kernel models/ball_query_ext/ball_query_cuda.cu:10-49.
 * dist (B,M,N) f32 -> out_idx (B,M,K) i32: first K n (ascending) with dist<=radius; 0 hits -> 0;
 * u<K hits -> out[u+i] = out[i % u]. */
int usip_ball_query_dist_f32(const float* dist, float radius, int32_t* out_idx,
                             int B, int M, int N, int K, void* stream);

/* Fused replacement of models/networks.py:355-373 (distance matrix + ball_query + gather + decenter):
 * xyz (B,3,N), feat (B,S,N) (S may be 0), centers (B,3,M) ->
 *   out_idx (B,M,K) i32      (bit-identical to ball_query on torch.norm(centers-xyz))
 *   out_group (B,3+S,M,K) f32 = x_aug gathered, xyz channels minus the centre  (`x_features`) (or NULL)
 *   out_rows  [B*M*K, ld_rows] f32: the same group as point-major rows for the MLP stack (or NULL)
 * scratch: usip_ball_group_scratch_bytes() bytes, 256-byte aligned (per cloud: bucket fill counts, 2-D bucket grid of
 * 32-byte records, overflow list).  CONTRACT: its counter region must be all-zero when the call starts -- clear it ONCE with
 * usip_ball_group_scratch_init() -- and every call leaves it all-zero again (the last CTA of each cloud restores it), so a
 * scratch buffer that is kept between calls costs no memset launch.  One scratch per stream.  Without scratch (or for
 * S > 4) the reference's in-order scan runs as a single kernel.  Two launches (build, query) chained by programmatic
 * dependent launch; the query stages its candidate buckets with one tensor-map TMA per keypoint. */
int usip_ball_group_f32(const float* xyz, const float* feat, const float* centers, float radius,
                        int32_t* out_idx, float* out_group, float* out_rows, int ld_rows,
                        void* scratch, int64_t scratch_bytes, int B, int S, int N, int M, int K, void* stream);
int64_t usip_ball_group_scratch_bytes(int B, int S, int N, int M, int K);
int usip_ball_group_scratch_init(void* scratch, int64_t scratch_bytes, int B, void* stream);

/* k-nearest-POINT grouping of the ablation detector RPN_Detector_KNN      models/networks.py:556-565
 * (torch.norm + topk(k, largest=False, sorted=False) + gather + subtract the node), without the (B,M,N) matrix.
 * out_idx (B,M,K) i32: the K points nearest to each centre, EXACT, in ascending point index (the reference's order is
 * unspecified; ties at the K-th distance: lowest index first); out_group / out_rows as in usip_ball_group_f32.  K <= N. */
int usip_knn_group_f32(const float* xyz, const float* feat, const float* centers, int32_t* out_idx, float* out_group,
                       float* out_rows, int ld_rows, int B, int S, int N, int M, int K, void* stream);

/* Farthest point sampling of the SOM nodes          data/kitti_detector_loader.py:68-83 (FarthestSampler.sample), :144-145
 * pts (B, Ns, 3) f32 row-major (the numpy subset the reference samples from), start (B,) i32 = index of the first node
 * (the reference draws it with np.random.randint) -> out_idx (B, k) i32 in selection order, out_nodes (B, 3, k) f32 (or
 * NULL).  Bit-identical to the numpy code: float64 running distances, first arg-max.  Ns <= 8192. */
int usip_fps_f32(const float* pts, const int32_t* start, int32_t* out_idx, float* out_nodes, int B, int Ns, int k,
                 void* stream);

/* Radius non-maximum suppression of the detected keypoints     evaluation/save_keypoints.py:180-216 (nms)
 * keypoints (B,3,M) f32, sigmas (B,M) f32 -> out_idx (B,M) i32: original indices of the kept keypoints in the order the
 * reference emits them (ascending sigma, ties by index), padded with -1; out_count (B,) i32.  radius < 0.01: pass-through
 * (0..M-1, count M) like the reference. */
int usip_nms_f32(const float* keypoints, const float* sigmas, float radius, int32_t* out_idx, int32_t* out_count,
                 int B, int M, void* stream);

/* operations.knn_gather_by_indexing                         models/operations.py:271-287
 * src (B,C,N), idx (B,M,K) i32 -> out (B,C,M,K): out[b,c,m,k] = src[b,c,idx[b,m,k]]. */
int usip_knn_gather_f32(const float* src, const int32_t* idx, float* out,
                        int B, int C, int N, int M, int K, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 2. Grouping front-end of RPN_Detector.forward            models/networks.py:85-108, util/som.py:17-54
 * ---------------------------------------------------------------------------------------------- */

/* som.query_topk(k=1): nearest node per point, fp32 (dx*dx+dy*dy)+dz*dz, ties -> smallest m.
 * xyz (B,3,N), node (B,3,M) -> min_idx (B,N) i32, count (B,M) i32 (must be zeroed by the caller). */
int usip_som_assign_f32(const float* xyz, const float* node, int32_t* min_idx, int32_t* count,
                        int B, int N, int M, void* stream);

/* The same result through a cell grid over the M <= 1024 nodes of each cloud (csrc/nngrid.cu): the nodes are counting-sorted
 * into ~M/2 cells, every point searches the cell shells around it until nothing outside can be closer -- ~50 distance
 * evaluations per point instead of M.  scratch: usip_som_assign_grid_scratch_bytes(B, M) bytes, 16-byte aligned. */
size_t usip_som_assign_grid_scratch_bytes(int B, int M);
int usip_som_assign_grid_f32(const float* xyz, const float* node, int32_t* min_idx, int32_t* count, void* scratch,
                             size_t scratch_bytes, int B, int N, int M, void* stream);

/* Stable counting sort of the points of every cloud by node id.
 *   seg_off (B,M+1) i32 : rows [seg_off[m], seg_off[m+1]) of cloud b belong to node m
 *   perm    (B,N)   i32 : sorted position -> original point index n (ascending n inside a node)
 *   row_seg (B,N)   i32 : b*M + node id of each sorted row
 * scratch: B * ceil(N/256) * M i32. */
int usip_cluster_sort(const int32_t* min_idx, int32_t* seg_off, int32_t* perm, int32_t* row_seg,
                      int32_t* scratch, int B, int N, int M, void* stream);

/* networks.py:87-108: cluster mean (sum/(count+1e-5), empty -> 0), decentre, concat sn.
 *   cluster_mean (B,3,M) f32 ; x_aug [B*N, ldx] (sorted rows; cols 0..2 = x - mean[node], 3..3+S-1 = sn,
 *   remaining cols up to ldx zero). */
int usip_cluster_mean_decenter(const float* xyz, const float* feat, const int32_t* seg_off,
                               const int32_t* perm, float* cluster_mean, float* x_aug, int ldx,
                               int B, int S, int N, int M, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 3. Shared-MLP stack: conv1x1 (+bias) with fused BN/ReLU prologue and BN-stat / group-max epilogue
 *    models/layers.py:248-303 (EquivariantLayer), 172-216 (MyConv2d), 23-121 (MyBatchNorm*)
 * ---------------------------------------------------------------------------------------------- */
typedef struct usip_layer_desc {
  const float* X;  int32_t ldx;        /* [P,Cin] input (pre-activation of the previous layer)       */
  int32_t P, Cin, Cout;
  const float* W;  int32_t ldw;        /* [Cout,Cin] weight rows, row stride ldw (conv weight layout)  */
  int32_t w_transposed;                /* 1: W is stored [Cin,Cout] (row stride ldw) -- dgrad uses the
                                          forward weight as-is: G_in = G_out * W                        */
  const float* bias;                   /* [Cout] or NULL                                              */
  const float* in_scale;               /* [Cin] or NULL: a = x*in_scale+in_shift (folded BatchNorm)   */
  const float* in_shift;
  int32_t in_relu;                     /* apply ReLU after the affine                                 */
  const float* addend; int32_t ld_add; /* optional [G,Cout] term added per row group                  */
  const int32_t* add_index;            /* row -> g  (NULL: g = row / add_group)                       */
  int32_t add_group;
  float* Y; int32_t ldy;               /* [P,Cout] output (NULL: not written)                         */
  float* stat_partial;                 /* [usip_layer_stat_slots(desc),2,Cout] partial (sum, sumsq) rows, or NULL */
  float* gmax; float* gmin;            /* [P/group,Cout] per-group max / min of Y, or NULL            */
  int32_t* garg_max; int32_t* garg_min;/* [P/group,Cout] row-in-group of the max / min, or NULL       */
  int32_t group;
  int32_t precision;                   /* 0 = fp32 SIMT, 1 = 3xTF32 tcgen05 (Cin%32==0, Cout%64==0) */
  void* tc_workspace;                  /* precision 1: >= usip_layer_tc_workspace_bytes(Cin,Cout) bytes */
  int64_t tc_workspace_bytes;
  int32_t tc_weights_packed;           /* 1: tc_workspace already holds the packed weights of this W  */
  int32_t debug_flags;                 /* profiling aids of the tcgen05 kernel, 0 in production (tools/tc_microbench.py).
                                          Results become WRONG with: 1 = skip the epilogue body, 2 = producers skip the X
                                          loads, 4 = no weight TMA, 32 = no Y stores, 64 = no statistics / group pass.
                                          Results stay correct (at a different precision) with: 8 = plain single-pass TF32
                                          (hi x hi product only, ~5e-4 relative: the backward-precision option of the train
                                          step), 16 = TF32 main product + two BF16 cross terms instead of 3xTF32 (~1e-6
                                          relative error); 128 = also prefetch X tiles into L2 */
  unsigned long long* debug_clocks;    /* [grid][17 warps][8] clock64() accumulators (lane 0 of each warp): where each warp
                                          role spends its time.  Only written by a library built with -DUSIP_TC_PROF
                                          (USIP_NVCC_EXTRA); NULL = off */
} usip_layer_desc;

int usip_layer_fwd(const usip_layer_desc* d, void* stream);
/* Packs the tensor-core weight tiles of n layers (precision != 0 descriptors: W, ldw, w_transposed, Cin, Cout, P, group /
 * gmax / gmin, debug_flags and tc_workspace are read) in ONE launch, exactly as usip_layer_fwd does on a call with
 * tc_weights_packed == 0; afterwards those layers may be launched with tc_weights_packed = 1.  The train step uses it to
 * re-pack all weight matrices after the optimizer update (26 launches -> 1). */
int usip_layer_tc_pack_many(const usip_layer_desc* descs, int n, void* stream);
/* number of [2,Cout] partial rows usip_layer_fwd writes into stat_partial for this descriptor (P, Cout, precision,
   group and whether group outputs are requested must already be filled in): one per 128-row tile for the SIMT kernel,
   one per (CTA, 32-lane quarter) for the persistent tcgen05 kernel.  usip_bn_finalize sums them in a fixed order. */
int usip_layer_stat_slots(const usip_layer_desc* desc);
int usip_layer_tile_rows(void);
/* bytes of tc_workspace (hi/lo TF32 split of W, pre-swizzled into tcgen05 operand tiles) */
int64_t usip_layer_tc_workspace_bytes(int Cin, int Cout);

/* Training-mode BatchNorm finalisation (F.batch_norm, layers.py:69-71): reduce the per-tile partials,
 * produce the folded affine scale = gamma/sqrt(var+eps), shift = beta - mean*scale, update running stats
 * (momentum, unbiased var) and save mean / invstd for the backward pass. */
int usip_bn_finalize(const float* stat_partial, int ntiles, int64_t count, int C,
                     const float* gamma, const float* beta, float eps, float momentum,
                     float* running_mean, float* running_var, float* scale, float* shift,
                     float* save_mean, float* save_invstd, void* stream);
/* Eval-mode: scale/shift from the running statistics. */
int usip_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean,
                        const float* running_var, float eps, int C, float* scale, float* shift, void* stream);

/* Segmented max over the sorted rows of every node (index_max + gather of networks.py:117-120,130-133):
 * X [B*N, ldx] -> pooled [B*M, ldp] (empty node -> 0), arg [B*M, C] i32 = global sorted row (or -1). */
int usip_segmax(const float* X, int ldx, const int32_t* seg_off, const int32_t* perm,
                float* pooled, int ldp, int32_t* arg, int B, int N, int M, int C, void* stream);

/* Node kNN, layers.py:417-421: ascending sqrt-distance, ties by index.  pts (B,3,M) -> knn (B,M,K) i32. */
int usip_knn_nodes(const float* pts, int32_t* knn_idx, int B, int M, int K, void* stream);

/* First kNN-fusion layer without materialising the (B,3+C,M,K) group tensor (layers.py:422-432):
 * Y[(b,m,k),:] = Z[b*M+knn[b,m,k],:] + Wxyz * (pts[b,:,knn]-pts[b,:,m]) + bias ; + BN stat partials. */
int usip_knn_combine(const float* Z, int ldz, const float* pts, const int32_t* knn_idx,
                     const float* W, int ldw, const float* bias, float* Y, int ldy, float* stat_partial,
                     int B, int M, int K, int Cout, void* stream);

/* out[q, c] = relu(scale[c]*(scale[c]>=0 ? gmax : gmin)[q,c] + shift[c])  == max_k relu(bn(y_k)) */
int usip_group_select(const float* gmax, const float* gmin, const float* scale, const float* shift,
                      float* out, int ldo, int Q, int C, void* stream);

/* networks.py:151-154: keypoints (B,3,M) = out[:, :3] + cluster_mean ; sigmas (B,M) = softplus(out[:,3]) + lb */
int usip_head_finalize(const float* out4, int ld, const float* cluster_mean, float sigma_lower_bound,
                       float* keypoints, float* sigmas, int B, int M, void* stream);

/* networks.py:383: out (B,C,M) = X[q,:] / (||X[q,:]||_2 + 1e-5); norm_out [B*M] optional (saved for backward) */
int usip_l2norm_to_bcm(const float* X, int ldx, float* out, float* norm_out, int B, int M, int C, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 4. Losses                                                  models/losses.py:44-143
 * ---------------------------------------------------------------------------------------------- */
/* min_j ||a_i - b_j||_2 and argmin (first index on exact ties).  a (B,3,Ma), b (B,3,Nb) ->
 * min_d (B,Ma) f32, arg (B,Ma) i32.  packed: B*Ma u64 scratch. */
int usip_pairwise_min_f32(const float* a, const float* b, float* min_d, int32_t* arg,
                          unsigned long long* packed, int B, int Ma, int Nb, void* stream);

/* The same result (bit-identical min_d and arg, same tie rule) for FEW queries against a LARGE point set -- the
 * keypoint-on-point-cloud searches of keypoint_detector.py:187-197 (512 keypoints against 16384 points per cloud): the
 * cloud is counting-sorted into a cell grid (one CTA per cloud) and every query scans the cell shells around it until
 * nothing outside can be closer.  scratch: usip_pairwise_min_grid_scratch_bytes(B, Nb) bytes, 16-byte aligned, contents
 * irrelevant on entry. */
size_t usip_pairwise_min_grid_scratch_bytes(int B, int Nb);
int usip_pairwise_min_grid_f32(const float* a, const float* b, float* min_d, int32_t* arg, void* scratch,
                               size_t scratch_bytes, int B, int Ma, int Nb, void* stream);

/* ChamferLoss_Brute sigma branch (losses.py:79-97) from the two pairwise-min results:
 * out[0]=loss, out[1]=chamfer_pure, out[2]=chamfer_weighted. */
int usip_chamfer_prob_reduce(const float* d_sd, const int32_t* i_sd, const float* d_ds, const int32_t* i_ds,
                             const float* sig_src, const float* sig_dst, float* out3, int B, int M, int N,
                             void* stream);

/* keypoint_detector.py:182-184: out = R @ kp * scale + shift   (kp (B,3,M), R (B,3,3), scale (B), shift (B,3)) */
int usip_transform_points(const float* kp, const float* R, const float* scale, const float* shift,
                          float* out, int B, int M, void* stream);

/* mean over (B,M) of d times alpha -> out[0]  (keypoint_detector.py:193-197) */
int usip_mean_scale(const float* d, int64_t n, float alpha, float* out, void* stream);


/* DescPairScanLoss (models/losses.py:190-237): min_j ||a[:,i] - b[:,j]||_2 over C-dim descriptors, a (B,C,Ma), b (B,C,Nb) */
int usip_desc_pairmin_f32(const float* a, const float* b, float* min_d, int32_t* arg, int B, int C, int Ma, int Nb,
                          void* stream);
/* loss (B,M) = w * clamp(dpos - dneg + gamma, 0), w = clamp(sigma_max - sigma, 0)/mean; active (B) = mean(> 0) */
int usip_desc_triplet(const float* dpos, const float* dneg, const float* sigma, float gamma, float sigma_max,
                      float* loss, float* active, int B, int M, void* stream);

/* backward of DescPairScanLoss (losses.py:199-233) with upstream gradient g_loss (B,M): anc (B,C,M), pos (B,C,Mp),
 * neg (B,C,Mn), saved (dpos, ipos, dneg, ineg) of usip_desc_pairmin_f32; g_anc / g_pos / g_neg are ACCUMULATED into
 * (pre-zero them). */
int usip_desc_triplet_bwd(const float* anc, const float* pos, const float* neg, const float* dpos, const int32_t* ipos,
                          const float* dneg, const int32_t* ineg, const float* sigma, float gamma, float sigma_max,
                          const float* g_loss, float* g_anc, float* g_pos, float* g_neg, int B, int C, int M, int Mp,
                          int Mn, void* stream);
/* backward of usip_l2norm_to_bcm: g (B,C,M), raw rows Y [B*M, C] -> GY [B*M, C]                     networks.py:383 */
int usip_l2norm_bwd(const float* g, const float* Y, int ldy, float* GY, int ldg, int B, int M, int C, void* stream);

/* PointOnSurfaceLoss                                                                   models/losses.py:146-183
 * kp (B,3,M), pc (B,3,N), sn (B,S,N) (first 3 channels = normal), arg (B,M) = nearest point (usip_pairwise_min_f32).
 * loss != NULL: loss (B,M) = (n . (kp-p)/(||kp-p|| + 1e-7))^2;  g_kp != NULL: g_kp (B,3,M) = g (B,M) * dloss/dkp. */
int usip_point_on_surface(const float* kp, const float* pc, const float* sn, const int32_t* arg, const float* g,
                          float* loss, float* g_kp, int B, int M, int N, int S, void* stream);

/* ---- backward of the loss kernels (autograd of models/losses.py / keypoint_detector.py:182-184) ---- */
/* grad of sum_i g_i*gscale*min_d_i: grad_a (B,3,Ma) overwritten, grad_b (B,3,Nb) ACCUMULATED (pre-zero) or NULL */
int usip_pairwise_min_bwd(const float* a, const float* b, const float* min_d, const int32_t* arg,
                          const float* g, float gscale, float* grad_a, float* grad_b,
                          int B, int Ma, int Nb, void* stream);
/* all four grads ACCUMULATE into pre-zeroed buffers; gout = d loss_total / d chamfer_loss (device scalar) */
int usip_chamfer_prob_bwd(const float* src, const float* dst, const float* sig_src, const float* sig_dst,
                          const float* d_sd, const int32_t* i_sd, const float* d_ds, const int32_t* i_ds,
                          const float* gout, float* g_src, float* g_dst, float* g_sig_src, float* g_sig_dst,
                          int B, int M, int N, void* stream);
int usip_transform_points_bwd(const float* g_out, const float* R, const float* scale, float* g_kp,
                              int B, int M, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 5. Backward pass of the fused plan (autograd of models/networks.py:75-162 / layers.py re-derived)
 * ---------------------------------------------------------------------------------------------- */
/* train-mode BatchNorm(+ReLU) backward: partial sums of g_z and g_z*xhat per 128-row tile ([ntiles,2,C]) */
int usip_bn_bwd_reduce(const float* G, int ldg, const float* Y, int ldy, const float* scale, const float* shift,
                       const float* mean, const float* invstd, int relu, float* part, int P, int C, void* stream);
/* -> g_gamma, g_beta (optionally accumulated) and the per-channel constants c1 = g_beta/n, c2 = g_gamma/n */
int usip_bn_bwd_finalize(const float* part, int ntiles, int64_t count, int C, float* g_gamma, float* g_beta,
                         float* c1, float* c2, int accumulate, void* stream);
/* g_y = scale*(g*1[z>0] - c1 - xhat*c2); GY may alias G */
int usip_bn_bwd_apply(const float* G, int ldg, const float* Y, int ldy, const float* scale, const float* shift,
                      const float* mean, const float* invstd, const float* c1, const float* c2, int relu,
                      float* GY, int ldo, int P, int C, void* stream);
/* group-max layers (max_k relu(bn(y_k)), layers.py:433,438) */
int usip_groupmax_bwd_select(const float* Gout, int ldg, const float* gmax, const float* gmin, const int32_t* amax,
                             const int32_t* amin, const float* scale, const float* shift, const float* mean,
                             const float* invstd, float* gz, int32_t* argsel, float* part, int Q, int C, void* stream);
int usip_groupmax_scatter_add(float* G, int ldg, const float* gsrc, const int32_t* argsel, int K, int Q, int C,
                              void* stream);
int usip_groupmax_bwd_apply(const float* Y, int ldy, const float* gz, const int32_t* argsel, const float* scale,
                            const float* mean, const float* invstd, const float* c1, const float* c2, float* GY,
                            int ldo, int K, int P, int C, void* stream);
int usip_group_sum(const float* G, int ldg, float* out, int ldo, int K, int Q, int C, void* stream);
int usip_seg_sum(const float* G, int ldg, const int32_t* seg_off, float* out, int ldo, int B, int N, int M, int C,
                 void* stream);
/* arg-max un-pooling (backward of usip_segmax): G[arg[q,c], c] (+)= gp[q,c] */
int usip_unpool_scatter(float* G, int ldg, const float* gp, int ldp, const int32_t* arg, int Q, int C,
                        int accumulate, void* stream);
/* backward of usip_knn_combine: GZ (pre-zeroed) += scatter of GY by neighbour; gW[:,0:3] += GY^T delta_xyz */
int usip_knn_combine_bwd(const float* GY, int ldg, const float* pts, const int32_t* knn_idx, float* GZ, int ldz,
                         float* gW, int ldw, int B, int M, int K, int C, void* stream);
/* out[c] += sum_r G[r,c] */
int usip_colsum(const float* G, int ldg, float* out, int P, int C, void* stream);
int usip_head_bwd(const float* g_kp, const float* g_sig, const float* out4, int ld, float* G, int B, int M,
                  void* stream);
/* gW[Cout,Cin] += GY[P,Cout]^T * act(X)[P,Cin], act = optional folded BN affine + ReLU (same prologue as forward);
 * precision 1: tcgen05 3xTF32 (MN-major operands; precision 4: the same kernel as plain single-pass TF32) when Cout>=64, Cout%4==0, Cin%64==0, P>=4096 (a 64-wide layer fills half of the
 * 128-row UMMA tile with zero rows); Cin<=8 has an HBM-bound row-streaming kernel; otherwise the register-tiled fp32 SIMT kernel */
int usip_wgrad(const float* GY, int ldg, const float* X, int ldx, const float* in_scale, const float* in_shift,
               int in_relu, float* gW, int ldw, int P, int Cout, int Cin, int precision, void* stream);

/* ---- parameter update (replaces torch.optim.Adam at models/keypoint_detector.py:42-45,207; keypoint_descriptor.py:32-35) ----
 * Adam(betas, eps, weight_decay 0) over flat fp32 buffers of n elements (n % 4 == 0, 16-byte aligned).  `lr_dev` (1 float)
 * and `step_dev` (1 int64, steps taken so far; incremented by the kernel) live in device memory so the launch can be part
 * of a CUDA graph; `arrive` is a zero-initialised uint32 scratch word.  g is multiplied by grad_scale first (1/world for a
 * summed data-parallel gradient). */
int usip_adam_step(float* p, const float* g, float* m, float* v, const float* lr_dev, int64_t* step_dev, uint32_t* arrive,
                   float beta1, float beta2, float eps, float grad_scale, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 6. Registration evaluation       evaluation/matlab/eval_outdoor/{kitti,oxford}/evaluate_*.m, eval_outdoor/external/
 * ---------------------------------------------------------------------------------------------- */
/* pdist2(b', a', 'euclidean', 'smallest', k) (evaluate_kitti.m:53, evaluate_oxford.m:63,67): for every a column the k
 * (1..8) nearest b columns in ascending distance, ties to the smaller index.  a (B,C,Ma), b (B,C,Mb) channel-major;
 * na / nb (B) valid counts or NULL (all).  idx (B,Ma,k) i32, -1 past the valid queries or candidates; dist (B,Ma,k) f32
 * or NULL.  Same arithmetic as usip_desc_pairmin_f32: the k = 1 column equals its arg bit for bit.  C <= 426. */
int usip_desc_knn_f32(const float* a, const float* b, const int32_t* na, const int32_t* nb, int32_t* idx, float* dist,
                      int B, int C, int Ma, int Mb, int k, void* stream);

/* Correspondence list: the unique (anc, pos) rows of nn12 (B,Ma,k12) (anc i -> pos nn12[i]) and, if nn21 != NULL, of
 * nn21 (B,Mb,k21) (pos j -> anc nn21[j]), in ascending (anc, pos) order -- union(matches12, matches21, 'rows') of
 * evaluate_oxford.m:63-72; with nn21 NULL and k12 = 1, [i, nn(i)] in anc order (evaluate_kitti.m:53-54).  Entries
 * outside [0, nb) / [0, na) are ignored.  corr (B,nmax,2) i32 (rows past count[b] are -1), count (B).
 * Ma, Mb <= 1024; nmax >= min(Ma*k12 + Mb*k21, Ma*Mb). */
int usip_corr_build(const int32_t* nn12, int k12, const int32_t* nn21, int k21, const int32_t* na, const int32_t* nb,
                    int32_t* corr, int32_t* count, int B, int Ma, int Mb, int nmax, void* stream);

/* Batched RANSAC rigid fit, ransacfitRt.m + ransac.m (s = 3, no degeneracy test, p, maxTrials) with the final
 * least-squares refit of estimateRigidTransform.m.  Correspondence c of pair b: x = anc_xyz[b, corr[b,c,0]],
 * y = pos_xyz[b, corr[b,c,1]] (f64 (B,Ma,3) / (B,Mb,3)), c < ncorr[b].  Inlier iff ||x - (R y + t)|| < threshold.
 * Trial tau draws 3 distinct indices from Philox-4x32-10 keyed by (seed, b, tau), or reads samples (B,max_trials+1,3)
 * when non-NULL; samples_out (same shape, or NULL) receives the indices of every trial scored.
 * Out: Rt (B,3,4) f64 mapping pos-frame points into the anc frame (NaN when empty), n_inliers, trialcount, best_trial
 * (-1 without a loop), inlier_mask (B,nmax) u8 = the best hypothesis's inliers (not recomputed after the refit),
 * status 0 ok / 1 fewer than 3 correspondences / 2 fewer than 3 inliers.
 * scratch: usip_ransac_rt_scratch_bytes(B, max_trials) bytes, 16-byte aligned.  12 launches: init, 5 x (score, scan)
 * over a fixed chunk schedule of trials, refit; no host synchronisation. */
size_t usip_ransac_rt_scratch_bytes(int B, int max_trials);
int usip_ransac_rt(const double* anc_xyz, const double* pos_xyz, const int32_t* corr, const int32_t* ncorr,
                   const int32_t* samples, int32_t* samples_out, double threshold, int max_trials, double p,
                   unsigned long long seed, double* Rt, int32_t* n_inliers, int32_t* trialcount, int32_t* best_trial,
                   uint8_t* inlier_mask, int32_t* status, void* scratch, size_t scratch_bytes, int B, int Ma, int Mb,
                   int nmax, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* USIP_B200_H_ */
