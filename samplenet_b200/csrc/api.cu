// api.cu -- the extern "C" boundary of libsamplenet_b200.so (see include/samplenet_b200.h).
// Argument validation + dispatch only; kernels live in chamfer.cu / softproj.cu / encoder.cu / emd.cu / matching.cu.
#include "common.cuh"
#include "../../include/samplenet_b200_debug.h"
#include <string.h>

namespace snb {

static thread_local char g_err[512] = "";
static thread_local unsigned long long g_launches = 0;

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches += (unsigned long long)n; }

// kernels (defined in the other translation units)
int launch_chamfer_forward(int b, int n, const float *xyz1, int m, const float *xyz2, float *dist1, int *idx1, float *dist2, int *idx2, int flags,
                           cudaStream_t stream);
int launch_chamfer_backward(int b, int n, const float *xyz1, int m, const float *xyz2, const float *grad_dist1, const int *idx1,
                            const float *grad_dist2, const int *idx2, float *grad_xyz1, float *grad_xyz2, cudaStream_t stream);
int launch_simplification_reduce(int b, int n, int m, const float *dist1, const float *dist2, float w, float *out4, cudaStream_t stream);
int launch_knn_softproj(int b, int n, int m, int k, int layout, const float *points, const float *query, const float *sigma, int sigma_mode,
                        float sigma_floor, int hard,
                        const float *feats, int f, float *proj, float *prop, int *knn_idx, float *knn_val, float *weights,
                        float *dist_over_sigma, int flags, cudaStream_t stream);
size_t softproj_bwd_workspace(int b, int n, int m, int k, int f);
int launch_softproj_backward(int b, int n, int m, int k, int layout, const float *points, const float *query, const float *sigma,
                             int sigma_mode, float sigma_floor, const float *feats, int f, const int *knn_idx, const float *weights, const float *grad_proj,
                             const float *grad_prop, float *grad_points, float *grad_query, float *grad_feats, float *grad_sigma,
                             void *workspace, cudaStream_t stream);
int launch_group_point(int b, int n, int c, int m, int ns, int layout, const float *points, const int *idx, float *out, cudaStream_t stream);
int launch_group_point_grad(int b, int n, int c, int m, int ns, int layout, const float *grad_out, const int *idx, float *grad_points,
                            cudaStream_t stream);
size_t encoder_workspace_bytes(int b, int n, int num_layers, const snb200_layer *layers);
int launch_encoder_forward(int b, int n, int layout, const float *x, int num_layers, const snb200_layer *layers, int training, float *feat,
                           void *workspace, cudaStream_t stream);
size_t fc_head_workspace_bytes(int b, int num_layers, const snb200_layer *layers);
int launch_fc_head_forward(int b, const float *in, int num_layers, const snb200_layer *layers, int training, float *out, int out_transpose_inner,
                           void *workspace, cudaStream_t stream);
size_t approxmatch_workspace_bytes(int b, int n, int m);
int launch_approxmatch(int b, int n, int m, const float *xyz1, const float *xyz2, float *match, void *workspace, cudaStream_t stream);
int launch_approxmatch_exact(int b, int n, int m, const float *xyz1, const float *xyz2, float *match, cudaStream_t stream);
int launch_matchcost(int b, int n, int m, const float *xyz1, const float *xyz2, const float *match, float *cost, float *partial, cudaStream_t stream);
int launch_matchcostgrad(int b, int n, int m, const float *xyz1, const float *xyz2, const float *match, float *grad1, float *grad2, cudaStream_t stream);
int launch_nn_matching(int b, int n, int t, int k, const float *full_pc, const int *nn_idx, int complete_fps, float *out, int *out_idx,
                       cudaStream_t stream);

int launch_tc_gemm_debug(int rows, int c_in, int c_out, const float *A, const float *W, const float *bias, float *D, unsigned desc_hi,
                         int k_adv16, int swizzle, cudaStream_t stream);
bool tc_layer_supported(int c_in, int c_out);

size_t generator_workspace_bytes(int b, int n, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc);
int launch_generator_forward(int b, int n, int layout, const float *x, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc,
                             int training, float *out, int out_transpose_inner, float *feat_out, int flags, void *workspace, cudaStream_t stream,
                             float *const *zsave = nullptr);
bool generator_backward_supported(int b, int n, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc);
size_t generator_backward_workspace_bytes(int b, int n, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc);
int launch_generator_backward(int b, int n, int layout, const float *x, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc,
                              float *const *zsave, void *fwd_workspace, const float *grad_out, int out_transpose_inner,
                              const snb200_layer_grad *gconv, const snb200_layer_grad *gfc, void *workspace, cudaStream_t stream);

int debug_head_timestamps(long long *host_out64);
int debug_conv_stack_timestamps(long long *host_out64);

size_t tail_workspace_bytes(int b, int n_samp, int n_ref);
size_t progressive_workspace_bytes(int b, int n, int m, int np);
int launch_progressive_loss(int b, int n, int m, const float *ref, const float *samp, int np, const int *sizes, const float *w21, float *dist1, int *idx1,
                            float *dist2, int *idx2, float *terms, void *workspace, unsigned *ticket, int flags, cudaStream_t stream);
int launch_tail_fused(int b, int n_ref, int n_samp, int k, const float *ref, const float *samp, const float *sigma, int sigma_mode, float sigma_floor,
                      float *proj, int *knn_idx, float *weights, float *dist_over_sigma, float *dist1, int *idx1, float *dist2, int *idx2,
                      float w21, float *out4, float *partial, unsigned *ticket, int flags, cudaStream_t stream);

static int check_layers(const char *who, int num_layers, const snb200_layer *layers, int max_layers)
{
    SNB_REQUIRE(layers != nullptr && num_layers >= 1 && num_layers <= max_layers, "%s: num_layers=%d out of range [1,%d]", who, num_layers, max_layers);
    for (int l = 0; l < num_layers; l++) {
        SNB_REQUIRE(layers[l].c_in >= 1 && layers[l].c_out >= 1, "%s: layer %d has non-positive width", who, l);
        SNB_REQUIRE(layers[l].weight != nullptr, "%s: layer %d has no weight", who, l);
        SNB_REQUIRE(l == 0 || layers[l].c_in == layers[l - 1].c_out, "%s: layer %d c_in=%d does not match previous c_out=%d", who, l,
                    layers[l].c_in, layers[l - 1].c_out);
        SNB_REQUIRE((layers[l].bn_weight == nullptr) == (layers[l].bn_bias == nullptr), "%s: layer %d needs both BN weight and bias", who, l);
    }
    return SNB200_OK;
}

// every SNB200_GEN_* bit the header defines; any other bit is rejected rather than ignored (64 selected a kernel that no longer exists
// and is not reused, so a caller that still sets it gets an error instead of a different kernel)
constexpr int kGenFlagsDefined = SNB200_GEN_EXACT_FP32 | SNB200_GEN_PROFILE_SKIP_HEAD | SNB200_GEN_PROFILE_SKIP_CONV | SNB200_GEN_PER_LAYER_KERNELS |
                                 SNB200_GEN_SEPARATE_HEAD | SNB200_GEN_WORKSPACE_PRIMED;

}  // namespace snb

using namespace snb;

#define SNB_API extern "C" __attribute__((visibility("default")))

SNB_API const char *snb200_last_error(void) { return g_err; }
SNB_API int snb200_version(void) { return 100; }
SNB_API unsigned long long snb200_launch_count(void) { return g_launches; }

SNB_API int snb200_nn_distance_forward(int b, int n, const float *xyz1, int m, const float *xyz2, float *dist1, int *idx1, float *dist2, int *idx2,
                                       int flags, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && m >= 1, "nn_distance_forward: bad sizes b=%d n=%d m=%d", b, n, m);
    SNB_REQUIRE(b <= 65535, "nn_distance_forward: batch %d exceeds the grid limit 65535", b);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(xyz1 && xyz2 && dist1 && idx1 && dist2 && idx2, "nn_distance_forward: null pointer");
    return launch_chamfer_forward(b, n, xyz1, m, xyz2, dist1, idx1, dist2, idx2, flags, (cudaStream_t)stream);
}

SNB_API int snb200_nn_distance_backward(int b, int n, const float *xyz1, int m, const float *xyz2, const float *grad_dist1, const int *idx1,
                                        const float *grad_dist2, const int *idx2, float *grad_xyz1, float *grad_xyz2, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && m >= 1 && b <= 65535, "nn_distance_backward: bad sizes b=%d n=%d m=%d", b, n, m);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(xyz1 && xyz2 && grad_dist1 && idx1 && grad_dist2 && idx2 && grad_xyz1 && grad_xyz2, "nn_distance_backward: null pointer");
    return launch_chamfer_backward(b, n, xyz1, m, xyz2, grad_dist1, idx1, grad_dist2, idx2, grad_xyz1, grad_xyz2, (cudaStream_t)stream);
}

SNB_API size_t snb200_simplification_loss_workspace_bytes(int, int, int) { return 0; }

SNB_API int snb200_simplification_loss_forward(int b, int n, const float *samp, int m, const float *ref, float weight21, float *dist1, int *idx1,
                                               float *dist2, int *idx2, float *out4, void *, size_t, int flags, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 1 && n >= 1 && m >= 1 && b <= 65535, "simplification_loss_forward: bad sizes b=%d n=%d m=%d", b, n, m);
    SNB_REQUIRE(samp && ref && dist1 && idx1 && dist2 && idx2 && out4, "simplification_loss_forward: null pointer");
    int rc = launch_chamfer_forward(b, n, samp, m, ref, dist1, idx1, dist2, idx2, flags, (cudaStream_t)stream);
    if (rc) return rc;
    return launch_simplification_reduce(b, n, m, dist1, dist2, weight21, out4, (cudaStream_t)stream);
}

SNB_API int snb200_knn_soft_project_forward(int b, int n, int m, int k, int layout, const float *points, const float *query, const float *sigma,
                                            int sigma_mode, float sigma_floor, int hard, const float *feats, int f, float *proj, float *prop, int *knn_idx, float *knn_val,
                                            float *weights, float *dist_over_sigma, int flags, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && m >= 1 && b <= 65535, "knn_soft_project_forward: bad sizes b=%d n=%d m=%d", b, n, m);
    SNB_REQUIRE(k >= 1 && k <= 32, "knn_soft_project_forward: group size k=%d outside the supported range [1,32]", k);
    SNB_REQUIRE(k <= n, "knn_soft_project_forward: k=%d exceeds the number of points n=%d", k, n);
    SNB_REQUIRE(layout == SNB200_BNC || layout == SNB200_BCN, "knn_soft_project_forward: unknown layout %d", layout);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(points && query, "knn_soft_project_forward: null input");
    const bool needs_sigma = proj || prop || weights || dist_over_sigma;
    SNB_REQUIRE(!needs_sigma || sigma, "knn_soft_project_forward: sigma is required for projection outputs");
    SNB_REQUIRE(sigma_mode >= 0 && sigma_mode <= 3, "knn_soft_project_forward: unknown sigma_mode %d", sigma_mode);
    SNB_REQUIRE(!prop || (feats && f >= 1), "knn_soft_project_forward: prop requested without features");
    return launch_knn_softproj(b, n, m, k, layout, points, query, sigma, sigma_mode, sigma_floor, hard, feats, f, proj, prop, knn_idx, knn_val, weights, dist_over_sigma,
                               flags, (cudaStream_t)stream);
}

SNB_API size_t snb200_soft_project_backward_workspace_bytes(int b, int n, int m, int k, int f) { return softproj_bwd_workspace(b, n, m, k, f); }

SNB_API int snb200_soft_project_backward(int b, int n, int m, int k, int layout, const float *points, const float *query, const float *sigma,
                                         int sigma_mode, float sigma_floor, const float *feats, int f, const int *knn_idx, const float *weights, const float *grad_proj,
                                         const float *grad_prop, float *grad_points, float *grad_query, float *grad_feats, float *grad_sigma,
                                         void *workspace, size_t workspace_bytes, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 1 && n >= 1 && m >= 1 && k >= 1 && k <= 32 && b <= 65535, "soft_project_backward: bad sizes b=%d n=%d m=%d k=%d", b, n, m, k);
    SNB_REQUIRE(layout == SNB200_BNC || layout == SNB200_BCN, "soft_project_backward: unknown layout %d", layout);
    SNB_REQUIRE(points && query && sigma && knn_idx && weights, "soft_project_backward: null input");
    SNB_REQUIRE(grad_proj || grad_prop, "soft_project_backward: no upstream gradient");
    SNB_REQUIRE(!grad_prop || (feats && f >= 1), "soft_project_backward: grad_prop without features");
    if (workspace_bytes < softproj_bwd_workspace(b, n, m, k, f) || !workspace) {
        set_error("soft_project_backward: workspace %zu < %zu bytes", workspace_bytes, softproj_bwd_workspace(b, n, m, k, f));
        return SNB200_EWORKSPACE;
    }
    return launch_softproj_backward(b, n, m, k, layout, points, query, sigma, sigma_mode, sigma_floor, feats, f, knn_idx, weights, grad_proj, grad_prop, grad_points,
                                    grad_query, grad_feats, grad_sigma, workspace, (cudaStream_t)stream);
}

SNB_API size_t snb200_project_and_loss_workspace_bytes(int b, int n_samp, int n_ref)
{
    if (b < 1 || n_samp < 1 || n_ref < 1) return 0;
    return tail_workspace_bytes(b, n_samp, n_ref);
}

SNB_API int snb200_project_and_loss_forward(int b, int n_ref, int n_samp, int k, const float *ref, const float *samp, const float *sigma,
                                            int sigma_mode, float sigma_floor, float *proj, int *knn_idx, float *weights, float *dist_over_sigma,
                                            float *dist1, int *idx1, float *dist2, int *idx2, float weight21, float *out4, void *workspace,
                                            size_t workspace_bytes, unsigned *ticket, int flags, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 1 && b <= 65535 && n_ref >= 1 && n_samp >= 1, "project_and_loss_forward: bad sizes b=%d n_ref=%d n_samp=%d", b, n_ref, n_samp);
    SNB_REQUIRE(n_ref <= 4096 && n_samp <= 4096, "project_and_loss_forward: clouds above 4096 points need the separate entry points (n_ref=%d n_samp=%d)", n_ref, n_samp);
    SNB_REQUIRE(k >= 1 && k <= 32 && k <= n_ref, "project_and_loss_forward: group size k=%d outside [1, min(32, n_ref)]", k);
    SNB_REQUIRE(sigma_mode >= 0 && sigma_mode <= 3, "project_and_loss_forward: unknown sigma_mode %d", sigma_mode);
    SNB_REQUIRE(ref && samp && sigma && proj && knn_idx && weights && dist1 && idx1 && dist2 && idx2 && out4 && ticket, "project_and_loss_forward: null pointer");
    if (!workspace || workspace_bytes < tail_workspace_bytes(b, n_samp, n_ref)) {
        set_error("project_and_loss_forward: workspace %zu < %zu bytes", workspace_bytes, tail_workspace_bytes(b, n_samp, n_ref));
        return SNB200_EWORKSPACE;
    }
    return launch_tail_fused(b, n_ref, n_samp, k, ref, samp, sigma, sigma_mode, sigma_floor, proj, knn_idx, weights, dist_over_sigma, dist1, idx1, dist2,
                             idx2, weight21, out4, reinterpret_cast<float *>(workspace), ticket, flags, (cudaStream_t)stream);
}

SNB_API int snb200_group_point(int b, int n, int c, int m, int ns, int layout, const float *points, const int *idx, float *out, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && c >= 1 && m >= 1 && ns >= 1, "group_point: bad sizes");
    SNB_REQUIRE(layout == SNB200_BNC || layout == SNB200_BCN, "group_point: unknown layout %d", layout);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(points && idx && out, "group_point: null pointer");
    return launch_group_point(b, n, c, m, ns, layout, points, idx, out, (cudaStream_t)stream);
}

SNB_API int snb200_group_point_grad(int b, int n, int c, int m, int ns, int layout, const float *grad_out, const int *idx, float *grad_points,
                                    snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && c >= 1 && m >= 1 && ns >= 1 && b <= 65535, "group_point_grad: bad sizes");
    SNB_REQUIRE(layout == SNB200_BNC || layout == SNB200_BCN, "group_point_grad: unknown layout %d", layout);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(grad_out && idx && grad_points, "group_point_grad: null pointer");
    return launch_group_point_grad(b, n, c, m, ns, layout, grad_out, idx, grad_points, (cudaStream_t)stream);
}

SNB_API size_t snb200_encoder_workspace_bytes(int b, int n, int num_layers, const snb200_layer *layers)
{
    if (check_layers("encoder_workspace_bytes", num_layers, layers, SNB200_MAX_CONV_LAYERS) || b < 1 || n < 1) return 0;
    return encoder_workspace_bytes(b, n, num_layers, layers);
}

SNB_API int snb200_encoder_forward(int b, int n, int layout, const float *x, int num_layers, const snb200_layer *layers, int training, float *feat,
                                   void *workspace, size_t workspace_bytes, snb200_stream_t stream)
{
    int rc = check_layers("encoder_forward", num_layers, layers, SNB200_MAX_CONV_LAYERS);
    if (rc) return rc;
    SNB_REQUIRE(b >= 1 && n >= 1, "encoder_forward: bad sizes b=%d n=%d", b, n);
    SNB_REQUIRE(layout == SNB200_BNC || layout == SNB200_BCN, "encoder_forward: unknown layout %d", layout);
    SNB_REQUIRE(layers[0].c_in == 3, "encoder_forward: first layer must take 3 input channels, got %d", layers[0].c_in);
    SNB_REQUIRE(x && feat, "encoder_forward: null pointer");
    for (int l = 0; l < num_layers; l++)
        SNB_REQUIRE(training || !layers[l].bn_weight || (layers[l].bn_running_mean && layers[l].bn_running_var),
                    "encoder_forward: eval mode needs running statistics (layer %d)", l);
    const size_t need = encoder_workspace_bytes(b, n, num_layers, layers);
    if (!workspace || workspace_bytes < need) { set_error("encoder_forward: workspace %zu < %zu bytes", workspace_bytes, need); return SNB200_EWORKSPACE; }
    return launch_encoder_forward(b, n, layout, x, num_layers, layers, training, feat, workspace, (cudaStream_t)stream);
}

SNB_API size_t snb200_generator_workspace_bytes(int b, int n, int num_conv, const snb200_layer *conv, int num_fc, const snb200_layer *fc)
{
    if (check_layers("generator_workspace_bytes", num_conv, conv, SNB200_MAX_CONV_LAYERS) || check_layers("generator_workspace_bytes", num_fc, fc, SNB200_MAX_FC_LAYERS) ||
        b < 1 || n < 1)
        return 0;
    return generator_workspace_bytes(b, n, num_conv, conv, num_fc, fc);
}

SNB_API int snb200_generator_forward(int b, int n, int layout, const float *x, int num_conv, const snb200_layer *conv, int num_fc,
                                     const snb200_layer *fc, int training, float *out, int out_transpose_inner, float *feat, int flags,
                                     void *workspace, size_t workspace_bytes, snb200_stream_t stream)
{
    SNB_REQUIRE((flags & ~kGenFlagsDefined) == 0, "generator_forward: flags 0x%x set bits outside the defined set 0x%x", flags, kGenFlagsDefined);
    int rc = check_layers("generator_forward", num_conv, conv, SNB200_MAX_CONV_LAYERS);
    if (rc) return rc;
    rc = check_layers("generator_forward", num_fc, fc, SNB200_MAX_FC_LAYERS);
    if (rc) return rc;
    SNB_REQUIRE(b >= 1 && b <= 256 && n >= 1, "generator_forward: bad sizes b=%d (1..256) n=%d", b, n);
    SNB_REQUIRE(layout == SNB200_BNC || layout == SNB200_BCN, "generator_forward: unknown layout %d", layout);
    SNB_REQUIRE(conv[0].c_in == 3, "generator_forward: first layer must take 3 input channels, got %d", conv[0].c_in);
    SNB_REQUIRE(fc[0].c_in == conv[num_conv - 1].c_out, "generator_forward: FC input width %d != conv output width %d", fc[0].c_in, conv[num_conv - 1].c_out);
    SNB_REQUIRE(x && out, "generator_forward: null pointer");
    SNB_REQUIRE(out_transpose_inner >= 0 && (out_transpose_inner == 0 || fc[num_fc - 1].c_out % out_transpose_inner == 0),
                "generator_forward: out_transpose_inner=%d does not divide the output width %d", out_transpose_inner, fc[num_fc - 1].c_out);
    for (int l = 0; l < num_conv; l++)
        SNB_REQUIRE(training || !conv[l].bn_weight || (conv[l].bn_running_mean && conv[l].bn_running_var),
                    "generator_forward: eval mode needs running statistics (conv layer %d)", l);
    for (int l = 0; l < num_fc; l++) {
        SNB_REQUIRE(training || !fc[l].bn_weight || (fc[l].bn_running_mean && fc[l].bn_running_var),
                    "generator_forward: eval mode needs running statistics (fc layer %d)", l);
        SNB_REQUIRE(!(training && fc[l].bn_weight && b < 2), "generator_forward: training-mode BatchNorm needs more than 1 row (fc layer %d)", l);
    }
    const size_t need = generator_workspace_bytes(b, n, num_conv, conv, num_fc, fc);
    if (!workspace || workspace_bytes < need) { set_error("generator_forward: workspace %zu < %zu bytes", workspace_bytes, need); return SNB200_EWORKSPACE; }
    return launch_generator_forward(b, n, layout, x, num_conv, conv, num_fc, fc, training, out, out_transpose_inner, feat, flags, workspace,
                                    (cudaStream_t)stream);
}

SNB_API int snb200_generator_backward_supported(int b, int n, int num_conv, const snb200_layer *conv, int num_fc, const snb200_layer *fc)
{
    if (check_layers("generator_backward_supported", num_conv, conv, SNB200_MAX_CONV_LAYERS) || check_layers("generator_backward_supported", num_fc, fc, SNB200_MAX_FC_LAYERS) ||
        b < 1 || n < 1)
        return 0;
    return generator_backward_supported(b, n, num_conv, conv, num_fc, fc) ? 1 : 0;
}

SNB_API int snb200_generator_train_forward(int b, int n, int layout, const float *x, int num_conv, const snb200_layer *conv, int num_fc,
                                           const snb200_layer *fc, float *out, int out_transpose_inner, float *feat, float *const *zsave, int flags,
                                           void *workspace, size_t workspace_bytes, snb200_stream_t stream)
{
    SNB_REQUIRE((flags & ~kGenFlagsDefined) == 0, "generator_train_forward: flags 0x%x set bits outside the defined set 0x%x", flags, kGenFlagsDefined);
    SNB_REQUIRE(zsave != nullptr, "generator_train_forward: zsave is null");
    int rc = check_layers("generator_train_forward", num_conv, conv, SNB200_MAX_CONV_LAYERS);
    if (rc) return rc;
    rc = check_layers("generator_train_forward", num_fc, fc, SNB200_MAX_FC_LAYERS);
    if (rc) return rc;
    SNB_REQUIRE(b >= 1 && n >= 1 && x && out, "generator_train_forward: bad arguments");
    SNB_REQUIRE(layout == SNB200_BNC || layout == SNB200_BCN, "generator_train_forward: unknown layout %d", layout);
    SNB_REQUIRE(generator_backward_supported(b, n, num_conv, conv, num_fc, fc), "generator_train_forward: shape outside the CUDA backward's envelope (b=%d n=%d)", b, n);
    SNB_REQUIRE(!(flags & (SNB200_GEN_EXACT_FP32 | SNB200_GEN_PER_LAYER_KERNELS | SNB200_GEN_SEPARATE_HEAD | SNB200_GEN_PROFILE_SKIP_CONV | SNB200_GEN_PROFILE_SKIP_HEAD)),
                "generator_train_forward: flags 0x%x select a path that does not keep activations", flags);
    for (int l = 0; l < num_conv; l++) SNB_REQUIRE(zsave[l] != nullptr, "generator_train_forward: zsave[%d] is null", l);
    const size_t need = generator_workspace_bytes(b, n, num_conv, conv, num_fc, fc);
    if (!workspace || workspace_bytes < need) { set_error("generator_train_forward: workspace %zu < %zu bytes", workspace_bytes, need); return SNB200_EWORKSPACE; }
    return launch_generator_forward(b, n, layout, x, num_conv, conv, num_fc, fc, 1, out, out_transpose_inner, feat, flags, workspace, (cudaStream_t)stream, zsave);
}

SNB_API size_t snb200_generator_backward_workspace_bytes(int b, int n, int num_conv, const snb200_layer *conv, int num_fc, const snb200_layer *fc)
{
    if (check_layers("generator_backward_workspace_bytes", num_conv, conv, SNB200_MAX_CONV_LAYERS) || check_layers("generator_backward_workspace_bytes", num_fc, fc, SNB200_MAX_FC_LAYERS) ||
        b < 1 || n < 1)
        return 0;
    return generator_backward_workspace_bytes(b, n, num_conv, conv, num_fc, fc);
}

SNB_API int snb200_generator_backward(int b, int n, int layout, const float *x, int num_conv, const snb200_layer *conv, int num_fc,
                                      const snb200_layer *fc, float *const *zsave, void *forward_workspace, const float *grad_out,
                                      int out_transpose_inner, const snb200_layer_grad *conv_grads, const snb200_layer_grad *fc_grads,
                                      void *workspace, size_t workspace_bytes, snb200_stream_t stream)
{
    int rc = check_layers("generator_backward", num_conv, conv, SNB200_MAX_CONV_LAYERS);
    if (rc) return rc;
    rc = check_layers("generator_backward", num_fc, fc, SNB200_MAX_FC_LAYERS);
    if (rc) return rc;
    SNB_REQUIRE(x && zsave && forward_workspace && grad_out && conv_grads && fc_grads, "generator_backward: null pointer");
    SNB_REQUIRE(generator_backward_supported(b, n, num_conv, conv, num_fc, fc), "generator_backward: shape outside the CUDA backward's envelope (b=%d n=%d)", b, n);
    const size_t need = generator_backward_workspace_bytes(b, n, num_conv, conv, num_fc, fc);
    if (!workspace || workspace_bytes < need) { set_error("generator_backward: workspace %zu < %zu bytes", workspace_bytes, need); return SNB200_EWORKSPACE; }
    return launch_generator_backward(b, n, layout, x, num_conv, conv, num_fc, fc, zsave, forward_workspace, grad_out, out_transpose_inner, conv_grads,
                                     fc_grads, workspace, (cudaStream_t)stream);
}

SNB_API int snb200_debug_head_timestamps(long long *host_out64) { return debug_head_timestamps(host_out64); }
SNB_API int snb200_debug_conv_stack_timestamps(long long *host_out64) { return debug_conv_stack_timestamps(host_out64); }

SNB_API int snb200_debug_tc_gemm(int rows, int c_in, int c_out, const float *A, const float *W, const float *bias, float *D, unsigned desc_hi,
                                 int k_adv16, int swizzle, snb200_stream_t stream)
{
    SNB_REQUIRE(rows >= 1 && tc_layer_supported(c_in, c_out), "debug_tc_gemm: unsupported shape rows=%d c_in=%d c_out=%d", rows, c_in, c_out);
    SNB_REQUIRE(A && W && bias && D, "debug_tc_gemm: null pointer");
    return launch_tc_gemm_debug(rows, c_in, c_out, A, W, bias, D, desc_hi, k_adv16, swizzle, (cudaStream_t)stream);
}

SNB_API size_t snb200_fc_head_workspace_bytes(int b, int num_layers, const snb200_layer *layers)
{
    if (check_layers("fc_head_workspace_bytes", num_layers, layers, SNB200_MAX_FC_LAYERS) || b < 1) return 0;
    return fc_head_workspace_bytes(b, num_layers, layers);
}

SNB_API int snb200_fc_head_forward(int b, const float *in, int num_layers, const snb200_layer *layers, int training, float *out,
                                   int out_transpose_inner, void *workspace, size_t workspace_bytes, snb200_stream_t stream)
{
    int rc = check_layers("fc_head_forward", num_layers, layers, SNB200_MAX_FC_LAYERS);
    if (rc) return rc;
    SNB_REQUIRE(b >= 1 && b <= 256, "fc_head_forward: batch %d outside the supported range [1,256]", b);
    SNB_REQUIRE(in && out, "fc_head_forward: null pointer");
    SNB_REQUIRE(out_transpose_inner >= 0 && (out_transpose_inner == 0 || layers[num_layers - 1].c_out % out_transpose_inner == 0),
                "fc_head_forward: out_transpose_inner=%d does not divide the output width %d", out_transpose_inner, layers[num_layers - 1].c_out);
    for (int l = 0; l < num_layers; l++) {
        SNB_REQUIRE(training || !layers[l].bn_weight || (layers[l].bn_running_mean && layers[l].bn_running_var),
                    "fc_head_forward: eval mode needs running statistics (layer %d)", l);
        SNB_REQUIRE(!(training && layers[l].bn_weight && b < 2), "fc_head_forward: training-mode BatchNorm needs more than 1 row (layer %d)", l);
    }
    const size_t need = fc_head_workspace_bytes(b, num_layers, layers);
    if (!workspace || workspace_bytes < need) { set_error("fc_head_forward: workspace %zu < %zu bytes", workspace_bytes, need); return SNB200_EWORKSPACE; }
    return launch_fc_head_forward(b, in, num_layers, layers, training, out, out_transpose_inner, workspace, (cudaStream_t)stream);
}

SNB_API size_t snb200_progressive_loss_workspace_bytes(int b, int n, int m, int num_prefix) { return progressive_workspace_bytes(b, n, m, num_prefix); }

SNB_API int snb200_progressive_loss_forward(int b, int n, int m, const float *ref, const float *samp, int num_prefix, const int *sizes, const float *weights,
                                            float *dist1, int *idx1, float *dist2, int *idx2, float *terms, void *workspace, size_t workspace_bytes,
                                            unsigned *ticket, int flags, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 1 && n >= 1 && m >= 1, "progressive_loss: bad sizes b=%d n=%d m=%d", b, n, m);
    SNB_REQUIRE(num_prefix >= 1 && num_prefix <= 16 && sizes && weights, "progressive_loss: 1..16 prefixes expected, got %d", num_prefix);
    SNB_REQUIRE(m <= 4096, "progressive_loss: at most 4096 ordered samples (one shared-memory tile), got %d", m);
    for (int p = 0; p < num_prefix; p++)
        SNB_REQUIRE(sizes[p] >= 1 && sizes[p] <= m && (p == 0 || sizes[p] > sizes[p - 1]), "progressive_loss: prefix sizes must be ascending in [1, m]");
    SNB_REQUIRE(ref && samp && dist1 && idx1 && dist2 && idx2 && terms && ticket, "progressive_loss: null pointer");
    if (!workspace || workspace_bytes < progressive_workspace_bytes(b, n, m, num_prefix)) { set_error("progressive_loss: workspace too small"); return SNB200_EWORKSPACE; }
    return launch_progressive_loss(b, n, m, ref, samp, num_prefix, sizes, weights, dist1, idx1, dist2, idx2, terms, workspace, ticket, flags, (cudaStream_t)stream);
}

SNB_API size_t snb200_approxmatch_workspace_bytes(int b, int n, int m) { return approxmatch_workspace_bytes(b, n, m); }

SNB_API int snb200_approxmatch(int b, int n, int m, const float *xyz1, const float *xyz2, float *match, void *workspace, size_t workspace_bytes,
                               snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && m >= 1, "approxmatch: bad sizes b=%d n=%d m=%d", b, n, m);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(xyz1 && xyz2 && match, "approxmatch: null pointer");
    if (!workspace || workspace_bytes < approxmatch_workspace_bytes(b, n, m)) {
        set_error("approxmatch: workspace %zu < %zu bytes", workspace_bytes, approxmatch_workspace_bytes(b, n, m));
        return SNB200_EWORKSPACE;
    }
    return launch_approxmatch(b, n, m, xyz1, xyz2, match, workspace, (cudaStream_t)stream);
}

SNB_API int snb200_approxmatch_mode(int b, int n, int m, const float *xyz1, const float *xyz2, float *match, int flags, void *workspace,
                                    size_t workspace_bytes, snb200_stream_t stream)
{
    if (!(flags & SNB200_EMD_EXACT)) return snb200_approxmatch(b, n, m, xyz1, xyz2, match, workspace, workspace_bytes, stream);
    SNB_REQUIRE(b >= 0 && n >= 1 && m >= 1, "approxmatch: bad sizes b=%d n=%d m=%d", b, n, m);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(xyz1 && xyz2 && match, "approxmatch: null pointer");
    return launch_approxmatch_exact(b, n, m, xyz1, xyz2, match, (cudaStream_t)stream);
}

SNB_API size_t snb200_matchcost_workspace_bytes(int b) { return (size_t)b * 16 * sizeof(float); }

SNB_API int snb200_matchcost(int b, int n, int m, const float *xyz1, const float *xyz2, const float *match, float *cost, void *workspace,
                             size_t workspace_bytes, snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && m >= 1 && b <= 65535, "matchcost: bad sizes b=%d n=%d m=%d", b, n, m);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(xyz1 && xyz2 && match && cost, "matchcost: null pointer");
    if (!workspace || workspace_bytes < snb200_matchcost_workspace_bytes(b)) { set_error("matchcost: workspace too small"); return SNB200_EWORKSPACE; }
    return launch_matchcost(b, n, m, xyz1, xyz2, match, cost, reinterpret_cast<float *>(workspace), (cudaStream_t)stream);
}

SNB_API int snb200_matchcostgrad(int b, int n, int m, const float *xyz1, const float *xyz2, const float *match, float *grad1, float *grad2,
                                 snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && m >= 1 && b <= 65535, "matchcostgrad: bad sizes b=%d n=%d m=%d", b, n, m);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(xyz1 && xyz2 && match && grad1 && grad2, "matchcostgrad: null pointer");
    return launch_matchcostgrad(b, n, m, xyz1, xyz2, match, grad1, grad2, (cudaStream_t)stream);
}

SNB_API int snb200_nn_matching(int b, int n, int t, int k, const float *full_pc, const int *nn_idx, int complete_fps, float *out, int *out_idx,
                               snb200_stream_t stream)
{
    SNB_REQUIRE(b >= 0 && n >= 1 && t >= 1 && k >= 1, "nn_matching: bad sizes b=%d n=%d t=%d k=%d", b, n, t, k);
    SNB_REQUIRE(complete_fps || k <= t, "nn_matching: without FPS completion k=%d must not exceed the number of indices t=%d", k, t);
    SNB_REQUIRE(k <= n, "nn_matching: k=%d exceeds the number of points n=%d", k, n);
    if (b == 0) return SNB200_OK;
    SNB_REQUIRE(full_pc && nn_idx && out, "nn_matching: null pointer");
    return launch_nn_matching(b, n, t, k, full_pc, nn_idx, complete_fps, out, out_idx, (cudaStream_t)stream);
}
