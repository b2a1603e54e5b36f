/*
 * samplenet_b200.h -- C ABI of libsamplenet_b200.so: SampleNet's sampling-and-loss hot path as
 * hand-written sm_100a CUDA.  This is the drop-in boundary: every entry point below replaces one of the
 * reference's native launchers (cited per function, paths relative to the reference tree) and keeps that
 * launcher's calling convention -- plain sizes + raw DEVICE pointers owned by the caller -- with three
 * deliberate differences (SURVEY.md 8b):
 *   1. every call takes the CUDA stream to launch on (the reference launchers use the legacy default stream);
 *   2. every call returns 0 on success or a negative SNB200_E* code and records a message retrievable with
 *      snb200_last_error() (the reference printf()s and carries on);
 *   3. the library allocates nothing: scratch is passed in, sized by the matching *_workspace_bytes() query.
 * All entry points are re-entrant (no global state besides the thread-local error string) and asynchronous
 * (they only enqueue work on `stream`; they never synchronise, so they can be captured into CUDA graphs).
 *
 * Layout tags: SNB200_BNC = (batch, points, channels) contiguous (the TF ops and ChamferDistance);
 *              SNB200_BCN = (batch, channels, points) contiguous (registration/src SoftProjection / SampleNet).
 * dtypes: float32 and int32 only.
 */
#ifndef SAMPLENET_B200_H
#define SAMPLENET_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNB200_OK 0
#define SNB200_EINVAL (-1)   /* bad size / null pointer / unsupported argument */
#define SNB200_EWORKSPACE (-2) /* workspace too small */
#define SNB200_ECUDA (-3)    /* CUDA runtime reported an error at launch */
#define SNB200_EUNSUPPORTED (-4)

#define SNB200_BNC 0
#define SNB200_BCN 1

/* flags for the distance kernels */
#define SNB200_DIST_FMA 0      /* d = fma(dz,dz,fma(dx,dx,dy*dy)): the arithmetic nvcc gives the reference CUDA kernels (bit-identical results) */
#define SNB200_DIST_UNFUSED 1  /* d = (dx*dx+dy*dy)+dz*dz, three roundings: the arithmetic of the reference CPU code */

/* how the `sigma` device scalar of the projection entry points is interpreted (sigma_mode); `sigma_floor` is the clamp:
 *   SIGMA_VALUE       *sigma is sigma itself
 *   SIGMA_FROM_T_REG  *sigma is the temperature T, sigma = max(T*T, floor)      registration/src/soft_projection.py:97-99
 *   SIGMA_FROM_T_CLS  *sigma is T, sigma = T*T                                   classification/soft_projection.py:41
 *   SIGMA_FROM_T_REC  *sigma is T, sigma = max(T, floor)^2                       reconstruction/src/soft_projection.py:51-54
 * (evaluating sigma inside the kernel removes two elementwise launches from every forward) */
#define SNB200_SIGMA_VALUE 0
#define SNB200_SIGMA_FROM_T_REG 1
#define SNB200_SIGMA_FROM_T_CLS 2
#define SNB200_SIGMA_FROM_T_REC 3

typedef void *snb200_stream_t; /* a cudaStream_t */

const char *snb200_last_error(void);
int snb200_version(void);
/* number of kernels this library has launched from the calling thread since load (bench.py's gpu_launches) */
unsigned long long snb200_launch_count(void);

/* ---------------------------------------------------------------------------------------------------------
 * Chamfer / nn_distance.  xyz1 (b,n,3), xyz2 (b,m,3) BNC; dist1,idx1 (b,n); dist2,idx2 (b,m).
 * Replaces ChamferDistanceKernelLauncher (registration/src/chamfer_distance/chamfer_distance.cpp:4-12,
 * chamfer_distance.cu:139-155) and NmDistanceKernelLauncher (classification/structural_losses/tf_nndistance.cpp:168,
 * tf_nndistance_g.cu:128-131).  Squared L2 distance to the nearest neighbour and its index; lowest index wins ties.
 * Both directions are computed by ONE launch.
 * --------------------------------------------------------------------------------------------------------- */
int snb200_nn_distance_forward(int b, int n, const float *xyz1, int m, const float *xyz2, float *dist1, int *idx1,
                               float *dist2, int *idx2, int flags, snb200_stream_t stream);

/* Replaces ChamferDistanceGradKernelLauncher (chamfer_distance.cpp:14-24, chamfer_distance.cu:189-209) and
 * NmDistanceGradKernelLauncher (tf_nndistance.cpp:208).  grad_xyz1 (b,n,3) and grad_xyz2 (b,m,3) are overwritten
 * (the launcher zeroes them itself, like the reference's cudaMemset).  Deterministic: no float atomics. */
int snb200_nn_distance_backward(int b, int n, const float *xyz1, int m, const float *xyz2, const float *grad_dist1,
                                const int *idx1, const float *grad_dist2, const int *idx2, float *grad_xyz1,
                                float *grad_xyz2, snb200_stream_t stream);

/* Fused simplification loss (registration/src/samplenet.py:171-181, classification/models/samplenet_model.py:176-188):
 * nn_distance(samp, ref) + the three reductions (two launches on `stream`).  out4 (device, 4 floats) =
 * { mean(dist1), mean_b(max_n dist1), mean(dist2), loss = out[0] + out[1] + (gamma + delta*pc_size) * out[2] }.
 * dist/idx outputs as in snb200_nn_distance_forward (needed by the backward).  workspace: see query. */
size_t snb200_simplification_loss_workspace_bytes(int b, int n, int m);
int snb200_simplification_loss_forward(int b, int n, const float *samp, int m, const float *ref, float weight21,
                                       float *dist1, int *idx1, float *dist2, int *idx2, float *out4, void *workspace,
                                       size_t workspace_bytes, int flags, snb200_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * kNN + soft projection, fused: for every query point the k nearest points of the cloud (brute force,
 * sorted by (squared distance, index)), then -- if `proj` is given -- dist/sigma, softmax over the k
 * neighbours and the weighted average of the neighbours (and of their features).
 * Replaces, in one launch: knn_cuda.KNN + pointnet2 grouping_operation + the torch ops of
 * registration/src/soft_projection.py:75-152; and tf_grouping.py:64-91 knn_point (three (B,M,N[,3]) temporaries
 * + selectionSortLauncher, tf_grouping.cpp:108) + groupPointLauncher (:142) + classification/soft_projection.py:46-82.
 *   points (b,n,3) / query (b,m,3) in `layout`; feats (b,n,f) BNC or (b,f,n) BCN, may be NULL (f = 0).
 *   sigma: DEVICE pointer to one float, already clamped by the caller (the three sub-projects clamp differently).
 *   hard != 0: one-hot weights on the nearest neighbour (TF SoftProjection(hard=True)).
 * Outputs (each may be NULL): proj (b,m,3)/(b,3,m) in `layout`; prop like feats with n->m;
 *   knn_idx (b,m,k) int32; knn_val (b,m,k) squared distances ascending; weights (b,m,k); dist_over_sigma (b,m,k).
 * 1 <= k <= 32, k <= n.
 * --------------------------------------------------------------------------------------------------------- */
int snb200_knn_soft_project_forward(int b, int n, int m, int k, int layout, const float *points, const float *query,
                                    const float *sigma, int sigma_mode, float sigma_floor, int hard, const float *feats, int f, float *proj, float *prop,
                                    int *knn_idx, float *knn_val, float *weights, float *dist_over_sigma, int flags,
                                    snb200_stream_t stream);

/* Backward of the soft projection given the saved knn_idx and weights.  grad_proj in `layout` (may be NULL),
 * grad_prop like prop (may be NULL).  Outputs (each may be NULL): grad_points, grad_query in `layout` (overwritten),
 * grad_feats like feats (overwritten), grad_sigma: DEVICE pointer to one float (overwritten), the gradient with respect to
 * SIGMA (for the FROM_T modes the caller applies d sigma / d T).
 * Replaces the autograd graph of registration/src/soft_projection.py:92-152 and groupPointGradLauncher
 * (tf_grouping.cpp:173).  workspace: see query. */
size_t snb200_soft_project_backward_workspace_bytes(int b, int n, int m, int k, int f);
int snb200_soft_project_backward(int b, int n, int m, int k, int layout, const float *points, const float *query,
                                 const float *sigma, int sigma_mode, float sigma_floor, const float *feats, int f, const int *knn_idx,
                                 const float *weights, const float *grad_proj, const float *grad_prop,
                                 float *grad_points, float *grad_query, float *grad_feats, float *grad_sigma,
                                 void *workspace, size_t workspace_bytes, snb200_stream_t stream);

/* The tail of a SampleNet training step in ONE launch: soft projection of the generated points onto the input cloud
 * (registration/src/samplenet.py:114) + nn_distance(samp, ref) + the simplification-loss reductions (samplenet.py:175-180).
 * ref (b,n_ref,3), samp (b,n_samp,3) BNC.  Outputs: proj (b,n_samp,3), knn_idx / weights / dist_over_sigma (b,n_samp,k) (saved
 * for the projection backward), dist1/idx1 (b,n_samp), dist2/idx2 (b,n_ref), out4 as in snb200_simplification_loss_forward.
 * workspace: snb200_project_and_loss_workspace_bytes() bytes of partial sums; ticket: DEVICE unsigned that must be zero at
 * the first call and is left zero by every call (allocate once, never touch).  n_ref <= 4096 (one shared-memory tile). */
size_t snb200_project_and_loss_workspace_bytes(int b, int n_samp, int n_ref);
int snb200_project_and_loss_forward(int b, int n_ref, int n_samp, int k, const float *ref, const float *samp, const float *sigma,
                                    int sigma_mode, float sigma_floor, float *proj, int *knn_idx, float *weights,
                                    float *dist_over_sigma, float *dist1, int *idx1, float *dist2, int *idx2, float weight21,
                                    float *out4, void *workspace, size_t workspace_bytes, unsigned *ticket, int flags,
                                    snb200_stream_t stream);

/* group_point: points (b,n,c) BNC [or (b,c,n) BCN], idx (b,m,ns) -> out (b,m,ns,c) BNC [or (b,c,m,ns) BCN].
 * Replaces groupPointLauncher / groupPointGradLauncher (tf_grouping.cpp:142,173; tf_grouping_g.cu:40-78) and
 * pointnet2 grouping_operation.  The grad launcher overwrites grad_points (zeroes it first). */
int snb200_group_point(int b, int n, int c, int m, int ns, int layout, const float *points, const int *idx, float *out,
                       snb200_stream_t stream);
int snb200_group_point_grad(int b, int n, int c, int m, int ns, int layout, const float *grad_out, const int *idx,
                            float *grad_points, snb200_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * SampleNet generator (registration/src/samplenet.py:40-60,90-104; rec widths reconstruction/src/samplers.py:22-36):
 * x -> 5 x [1x1 conv + BatchNorm + ReLU] -> max over points -> 3 x [Linear + BatchNorm + ReLU] -> Linear.
 * --------------------------------------------------------------------------------------------------------- */
#define SNB200_MAX_CONV_LAYERS 8
#define SNB200_MAX_FC_LAYERS 8
typedef struct snb200_layer {
    int c_in, c_out;
    const float *weight;  /* (c_out, c_in) row-major: Conv1d.weight[:, :, 0] / Linear.weight */
    const float *bias;    /* (c_out) */
    const float *bn_weight, *bn_bias;   /* (c_out) gamma/beta, NULL => no BatchNorm after this layer */
    float *bn_running_mean, *bn_running_var; /* (c_out) updated in training mode when non-NULL */
    long long *bn_num_batches_tracked;  /* int64 device scalar, +1 per training forward when non-NULL (torch BatchNorm bookkeeping) */
    float bn_eps, bn_momentum;
    int relu;             /* apply ReLU after (BatchNorm of) this layer */
} snb200_layer;

/* Per-point MLP + global max-pool.  x (b,n,3) in `layout`; feat (b, c_last).  training != 0 uses batch statistics
 * over all b*n positions (and updates the running stats), else the running stats.  workspace: see query. */
size_t snb200_encoder_workspace_bytes(int b, int n, int num_layers, const snb200_layer *layers);
int snb200_encoder_forward(int b, int n, int layout, const float *x, int num_layers, const snb200_layer *layers,
                           int training, float *feat, void *workspace, size_t workspace_bytes, snb200_stream_t stream);

/* The whole generator in one call: conv stack -> max-pool -> FC head -> out (b, c_out_last) [+ feat (b, c_conv_last), may be
 * NULL].  Default path: ONE persistent cooperative launch -- layers 2.. of the conv stack on the tensor cores (tcgen05.mma
 * kind::tf32, 3xTF32 error-compensated, fp32 TMEM accumulators), layer 1 evaluated on the fly with its BatchNorm statistics
 * derived from the input moments, the max-pool and all FC layers on the same grid (conv widths 32/64/128, up to 16 slices of
 * 256 points per SM).  Other shapes: one tensor-core launch per layer + a thread-block-cluster FC head.  flags &
 * SNB200_GEN_EXACT_FP32 selects the exact-fp32 CUDA-core conv stack instead (also taken automatically for widths the tensor
 * path does not cover).  b <= 256.  Training-mode pre-BatchNorm activations must stay below ~3e4 in magnitude on the default
 * path (fixed-point statistics exchange); beyond that the call returns NaN rows.  A flag bit not defined below is rejected with
 * SNB200_EINVAL (64, once a kernel selector, is retired and stays unused). */
#define SNB200_GEN_EXACT_FP32 1
#define SNB200_GEN_PER_LAYER_KERNELS 8 /* tensor-core path as one launch per layer instead of the persistent conv-stack kernel */
#define SNB200_GEN_SEPARATE_HEAD 16 /* keep the pool + FC head as its own thread-block-cluster launch */
#define SNB200_GEN_WORKSPACE_PRIMED 32 /* the caller keeps `workspace` across calls and its first 256 bytes are zero (freshly zeroed or as the
                                         previous PRIMED call left them): the persistent kernel cleans the rest itself, no memset in front */
#define SNB200_GEN_PROFILE_SKIP_HEAD 2 /* profiling only: stop after the conv stack (out is not written) */
#define SNB200_GEN_PROFILE_SKIP_CONV 4 /* profiling only: run only the pool + FC head on whatever the workspace holds */
size_t snb200_generator_workspace_bytes(int b, int n, int num_conv, const snb200_layer *conv, int num_fc, const snb200_layer *fc);
int snb200_generator_forward(int b, int n, int layout, const float *x, int num_conv, const snb200_layer *conv, int num_fc,
                             const snb200_layer *fc, int training, float *out, int out_transpose_inner, float *feat, int flags,
                             void *workspace, size_t workspace_bytes, snb200_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Generator TRAINING step: forward that keeps what the backward needs, and the backward itself
 * (replaces `loss.backward()` through registration/src/samplenet.py:90-104 -- stock cuDNN / cuBLAS / ATen kernels in the reference).
 *   snb200_generator_backward_supported(...) != 0 : shapes covered (the persistent conv-stack envelope, 2 <= b <= 64, BN + ReLU layers)
 *   snb200_generator_train_forward : snb200_generator_forward + `zsave`: per conv layer l a (b*n, c_out_l) float buffer that receives
 *                                    the layer's raw output; `workspace` must stay untouched until the backward has run
 *   snb200_generator_backward      : grad_out (b, c_out_last) in the layout snb200_generator_forward stores `out` -> gradients of
 *                                    every weight / bias / BatchNorm weight / BatchNorm bias (null pointers are skipped)
 * --------------------------------------------------------------------------------------------------------- */
typedef struct snb200_layer_grad {
    float *weight, *bias, *bn_weight, *bn_bias;
} snb200_layer_grad;
int snb200_generator_backward_supported(int b, int n, int num_conv, const snb200_layer *conv, int num_fc, const snb200_layer *fc);
int snb200_generator_train_forward(int b, int n, int layout, const float *x, int num_conv, const snb200_layer *conv, int num_fc,
                                   const snb200_layer *fc, float *out, int out_transpose_inner, float *feat, float *const *zsave, int flags,
                                   void *workspace, size_t workspace_bytes, snb200_stream_t stream);
size_t snb200_generator_backward_workspace_bytes(int b, int n, int num_conv, const snb200_layer *conv, int num_fc, const snb200_layer *fc);
int snb200_generator_backward(int b, int n, int layout, const float *x, int num_conv, const snb200_layer *conv, int num_fc,
                              const snb200_layer *fc, float *const *zsave, void *forward_workspace, const float *grad_out,
                              int out_transpose_inner, const snb200_layer_grad *conv_grads, const snb200_layer_grad *fc_grads,
                              void *workspace, size_t workspace_bytes, snb200_stream_t stream);

/* Fully connected head on the pooled feature: in (b, c_in0) -> out (b, c_out_last).  BatchNorm over the batch.
 * out_transpose_inner = M > 0: each output row, logically (c_out_last/M, M) -- the reference's y.view(-1, 3, M),
 * samplenet.py:104 -- is stored transposed as (M, c_out_last/M), i.e. directly in BNC order; 0 = stored as is (BCN). */
size_t snb200_fc_head_workspace_bytes(int b, int num_layers, const snb200_layer *layers);
int snb200_fc_head_forward(int b, const float *in, int num_layers, const snb200_layer *layers, int training, float *out,
                           int out_transpose_inner, void *workspace, size_t workspace_bytes, snb200_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * SampleNetProgressive: the simplification loss summed over prefixes of an ORDERED sample set, one launch
 * (replaces the per-prefix NnDistance ops + reductions of classification/train_samplenet_progressive.py:172-230).
 *   ref (b,n,3), samp (b,m,3); sizes[num_prefix] ascending prefix lengths (<= m, <= 16 of them); weights[p] = gamma + delta * sizes[p]
 *   dist1/idx1 (b,m): sample -> nearest input point (prefix p uses the slice [:sizes[p]])
 *   dist2/idx2 (b,num_prefix,n): input point -> nearest of the first sizes[p] samples
 *   terms (3*num_prefix + 1): per prefix [mean dist1[:s], mean_b max dist1[:s], mean dist2_p], then the total loss
 *   ticket: one zero-initialised unsigned, left zero.  sizes / weights are HOST arrays.
 * --------------------------------------------------------------------------------------------------------- */
size_t snb200_progressive_loss_workspace_bytes(int b, int n, int m, int num_prefix);
int snb200_progressive_loss_forward(int b, int n, int m, const float *ref, const float *samp, int num_prefix, const int *sizes, const float *weights,
                                    float *dist1, int *idx1, float *dist2, int *idx2, float *terms, void *workspace, size_t workspace_bytes,
                                    unsigned *ticket, int flags, snb200_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * EMD.  xyz1 (b,n,3), xyz2 (b,m,3), match (b,m,n), cost (b), grad1 (b,n,3), grad2 (b,m,3).
 * Replace approxmatchLauncher / matchcostLauncher / matchcostgradLauncher
 * (classification/structural_losses/tf_approxmatch.cpp:141-143, tf_approxmatch_g.cu:181,227,293-294).
 * `temp` of the reference (tf_approxmatch.cpp:168) is the workspace here.
 * --------------------------------------------------------------------------------------------------------- */
size_t snb200_approxmatch_workspace_bytes(int b, int n, int m);
int snb200_approxmatch(int b, int n, int m, const float *xyz1, const float *xyz2, float *match, void *workspace,
                       size_t workspace_bytes, snb200_stream_t stream);
/* flags & SNB200_EMD_EXACT: the parity mode -- exact exponential (exp in double, rounded to float), one float accumulator per row summed in
 * index order, the reference's level order and per-level read-modify-write of `match`: operation-for-operation the arithmetic of the CPU
 * oracle, so match values AND arg-max assignments are bit-identical to it (workspace unused).  Without the flag: the fast kernel. */
#define SNB200_EMD_EXACT 1
int snb200_approxmatch_mode(int b, int n, int m, const float *xyz1, const float *xyz2, float *match, int flags, void *workspace,
                            size_t workspace_bytes, snb200_stream_t stream);
size_t snb200_matchcost_workspace_bytes(int b);
int snb200_matchcost(int b, int n, int m, const float *xyz1, const float *xyz2, const float *match, float *cost,
                     void *workspace, size_t workspace_bytes, snb200_stream_t stream);
int snb200_matchcostgrad(int b, int n, int m, const float *xyz1, const float *xyz2, const float *match, float *grad1,
                         float *grad2, snb200_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Inference matching on the GPU (registration/src/samplenet.py:119-141 + sputils.py:7-41): order-preserving unique
 * of the NN indices, then farthest-point-sampling completion to k points.  full_pc (b,n,3) BNC, nn_idx (b,t),
 * out (b,k,3) BNC, out_idx (b,k) (may be NULL).  complete_fps == 0 -> plain gather of the first k indices.
 * --------------------------------------------------------------------------------------------------------- */
int snb200_nn_matching(int b, int n, int t, int k, const float *full_pc, const int *nn_idx, int complete_fps, float *out,
                       int *out_idx, snb200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SAMPLENET_B200_H */
