// C-ABI entry points of libbbb_b200.so (declared in include/bbb_b200.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "common.cuh"
#include "fwd_simt.cuh"
#include "misc_kernels.cuh"
#include "bwd_simt.cuh"
#include "fwd_tc.cuh"
#include "fused_tc.cuh"
#include "conv_s4_tc.cuh"
#include "mc_head.cuh"

namespace {

thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
std::atomic<int> g_wide_tiles{0};   // bbb_set_wide_tiles
long long* g_trace = nullptr;      // debug hook (bbb_debug_set_trace)
long long* g_mcx_trace = nullptr;  // debug hook (bbb_debug_set_mcx_trace): handshake stamps of the exchange kernel
// debug hook (bbb_debug_set_timeline): launch k of the instrumented kernels writes [first CTA entry, last CTA
// exit] in %globaltimer ns to g_tl[2k], g_tl[2k+1]; the slot index is fixed at launch (= capture) time
long long* g_tl = nullptr;
int g_tl_cap = 0, g_tl_n = 0;
char g_tl_names[256][64];
long long* tl_slot(bool used, const char* kind, const bbb::Geom& g) {
    if (!g_tl || !used || g_tl_n >= g_tl_cap || g_tl_n >= 256) return nullptr;
    snprintf(g_tl_names[g_tl_n], sizeof(g_tl_names[0]), "%s M=%d N=%d K=%d", kind, g.M, g.N, g.K);
    return g_tl + 4 * (g_tl_n++);
}

int fail(int code, const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    return fail(BBB_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

constexpr size_t kCounterBytes = 64;
constexpr size_t kMaxKlSlots = 4096;
constexpr size_t kBaseWorkspace = kCounterBytes + kMaxKlSlots * sizeof(double);
constexpr size_t kTcOffset = (kBaseWorkspace + 1023) / 1024 * 1024;   // prepared-operand region (tcgen05 path)

int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0; cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}

int check_desc(const bbb_layer_desc* d, bbb::Geom& g, bool linear) {
    if (!d) return fail(BBB_E_INVALID, "desc is NULL");
    if (!bbb::make_geom(*d, g)) return fail(BBB_E_INVALID, "invalid layer geometry");
    if (linear && !g.linear_like) return fail(BBB_E_INVALID, "bbb_linear_*: desc is not the degenerate 1x1 geometry");
    if (d->variant != BBB_VARIANT_BBB && d->variant != BBB_VARIANT_LRT) return fail(BBB_E_INVALID, "bad variant %d", d->variant);
    if (d->kl_convention != BBB_KL_REFERENCE && d->kl_convention != BBB_KL_TEXTBOOK) return fail(BBB_E_INVALID, "bad kl_convention");
    if (d->epilogue_act < BBB_ACT_NONE || d->epilogue_act > BBB_ACT_RELU) return fail(BBB_E_INVALID, "bad epilogue_act");
    if (!(d->prior_sigma > 0.0f)) return fail(BBB_E_INVALID, "prior_sigma must be > 0");
    return BBB_OK;
}

int forward_impl(const bbb_layer_desc* d, bool linear, const void* x, const float* W_mu, const float* W_rho,
                 const float* bias_mu, const float* bias_rho, void* y, float* kl_out, float* act_std,
                 const float* eps_a, const float* eps_b, uint64_t seed, uint64_t stream_id, const uint64_t* stream_base, void* ws,
                 size_t ws_bytes, void* stream) {
    bbb::Geom g;
    if (int rc = check_desc(d, g, linear)) return rc;
    if (!x || !W_mu || !W_rho || !y) return fail(BBB_E_INVALID, "NULL tensor pointer");
    if (d->has_bias && (!bias_mu || !bias_rho)) return fail(BBB_E_INVALID, "has_bias set but bias pointers NULL");
    if (kl_out && (!ws || ws_bytes < bbb_workspace_bytes(d)))
        return fail(BBB_E_WORKSPACE, "workspace too small: need %zu bytes", bbb_workspace_bytes(d));
    if (d->pool_k != 0) return fail(BBB_E_UNSUPPORTED, "fused max-pool epilogue is not available on this path");
    cudaStream_t st = (cudaStream_t)stream;

    int math = d->math;
    if (math == BBB_MATH_AUTO) math = bbb::tc_supported(*d, g) ? BBB_MATH_BF16_TC : BBB_MATH_FP32;
    if (math == BBB_MATH_BF16_TC || math == BBB_MATH_TF32_TC) {
        if (!bbb::tc_supported(*d, g)) return fail(BBB_E_UNSUPPORTED, "tcgen05 math mode: shape not supported by the tcgen05 path");
        const size_t need = kTcOffset + bbb::tc_workspace_bytes(g);
        if (!ws || ws_bytes < need) return fail(BBB_E_WORKSPACE, "workspace too small for the tcgen05 path: need %zu bytes", need);
        bbb::TcArgs a;
        a.wtiles = (__nv_bfloat16*)((char*)ws + kTcOffset);
        a.tf32 = math == BBB_MATH_TF32_TC;
        // operand tiles: 2 planes x npad rows x (kpad * 2 bytes of bf16 | kpad32 * 4 bytes of tf32), then the bias rows
        a.bias_ws = (float*)((char*)ws + kTcOffset + (size_t)bbb::tc_npad(g) * bbb::tc_kpad(g, a.tf32) * (a.tf32 ? 8 : 4));
        a.skip_prep = 0; a.prep_only = 0; a.y_sq = nullptr; a.out_mode = 2; a.out_pitch = 0; a.pool = 0; a.trace = g_trace;
        a.tl_prep = tl_slot(true, "weight_prep", g); a.tl_gemm = tl_slot(true, "gemm_tc", g);
        a.g = g; a.x = x; a.w_mu = W_mu; a.w_rho = W_rho; a.b_mu = bias_mu; a.b_rho = bias_rho;
        a.y = y; a.kl_out = kl_out; a.act_std = act_std; a.eps_a = eps_a; a.eps_b = eps_b;
        a.key = bbb::make_key(seed, stream_id); a.stream_base = (const unsigned long long*)stream_base;
        a.kl_counter = (unsigned int*)ws; a.kl_partials = (double*)((char*)ws + kCounterBytes);
        a.prior_mu = d->prior_mu; a.prior_sigma = d->prior_sigma;
        a.sample = d->sample; a.kl_convention = d->kl_convention; a.has_bias = d->has_bias; a.act = d->epilogue_act;
        a.act_dtype = d->act_dtype; a.variant = d->variant;
        int nl = 0;
        cudaError_t e = bbb::launch_fwd_tc(a, st, sm_count(), &nl);
        if (e != cudaSuccess) return cuda_fail(e, "fwd_tc launch");
        g_launches += nl;
        return BBB_OK;
    }
    if (math != BBB_MATH_FP32) return fail(BBB_E_INVALID, "bad math mode %d", d->math);
    if (d->act_dtype != BBB_DTYPE_F32) return fail(BBB_E_UNSUPPORTED, "BBB_MATH_FP32 path takes fp32 activations only");
    if ((size_t)bbb::simt_kl_slots(g) > kMaxKlSlots || bbb::simt_kl_slots(g) > 65535)
        return fail(BBB_E_UNSUPPORTED, "out_channels too large for the CUDA-core path (%d column tiles)", bbb::simt_kl_slots(g));

    bbb::FwdArgs a;
    a.g = g; a.x = (const float*)x; a.w_mu = W_mu; a.w_rho = W_rho; a.b_mu = bias_mu; a.b_rho = bias_rho;
    a.y = (float*)y; a.kl_out = kl_out; a.act_std = act_std; a.eps_a = eps_a; a.eps_b = eps_b;
    a.key = bbb::make_key(seed, stream_id); a.stream_base = (const unsigned long long*)stream_base;
    a.kl_counter = (unsigned int*)ws; a.kl_partials = (double*)((char*)ws + kCounterBytes);
    a.prior_mu = d->prior_mu; a.prior_sigma = d->prior_sigma;
    a.sample = d->sample; a.kl_convention = d->kl_convention; a.has_bias = d->has_bias; a.act = d->epilogue_act;
    cudaError_t e = d->variant == BBB_VARIANT_LRT ? bbb::launch_fwd_simt<BBB_VARIANT_LRT>(a, st)
                                                  : bbb::launch_fwd_simt<BBB_VARIANT_BBB>(a, st);
    if (e != cudaSuccess) return cuda_fail(e, "fwd_simt launch");
    g_launches += 1;
    return BBB_OK;
}

int backward_impl(const bbb_layer_desc* d, bool linear, const void* x, const void* grad_y, const float* W_mu,
                  const float* W_rho, const float* bias_mu, const float* bias_rho, const float* act_std,
                  const float* eps_a, const float* eps_b, uint64_t seed, uint64_t stream_id, const uint64_t* stream_base, void* grad_x,
                  float* g_W_mu, float* g_W_rho, float* g_bias_mu, float* g_bias_rho, void* ws, size_t ws_bytes,
                  void* stream) {
    bbb::Geom g;
    if (int rc = check_desc(d, g, linear)) return rc;
    if (!x || !grad_y || !W_mu || !W_rho) return fail(BBB_E_INVALID, "NULL tensor pointer");
    if (d->act_dtype != BBB_DTYPE_F32) return fail(BBB_E_UNSUPPORTED, "backward takes fp32 activations only");
    if (d->epilogue_act != BBB_ACT_NONE || d->pool_k != 0)
        return fail(BBB_E_UNSUPPORTED, "backward through a fused activation/pool epilogue is not available");
    if (d->variant == BBB_VARIANT_LRT && d->sample && !act_std)
        return fail(BBB_E_INVALID, "LRT backward needs the act_std tensor saved by the forward");
    (void)ws; (void)ws_bytes;
    bbb::BwdArgs a;
    a.g = g; a.x = (const float*)x; a.gy = (const float*)grad_y; a.w_mu = W_mu; a.w_rho = W_rho;
    a.b_mu = bias_mu; a.b_rho = bias_rho; a.act_std = act_std; a.eps_a = eps_a; a.eps_b = eps_b;
    a.key = bbb::make_key(seed, stream_id); a.stream_base = (const unsigned long long*)stream_base;
    a.gx = (float*)grad_x; a.g_w_mu = g_W_mu; a.g_w_rho = g_W_rho; a.g_b_mu = g_bias_mu; a.g_b_rho = g_bias_rho;
    a.sample = d->sample; a.has_bias = d->has_bias; a.variant = d->variant;
    int nl = 0;
    cudaError_t e = bbb::launch_bwd_simt(a, (cudaStream_t)stream, sm_count(), &nl);
    if (e != cudaSuccess) return cuda_fail(e, "bwd_simt launch");
    g_launches += nl;
    return BBB_OK;
}

}  // namespace

extern "C" {

size_t bbb_workspace_bytes(const bbb_layer_desc* desc) {
    if (!desc || desc->math == BBB_MATH_FP32) return kBaseWorkspace;
    bbb::Geom g;
    if (!bbb::make_geom(*desc, g)) return kBaseWorkspace;
    size_t a = bbb::tc_workspace_bytes(g);
    const size_t b = bbb::fused_workspace_bytes(g), c = bbb::conv_s4_workspace_bytes(g);
    if (b > a) a = b;
    if (c > a) a = c;
    return kTcOffset + a;
}

int bbb_conv2d_forward(const bbb_layer_desc* desc, const void* x, const float* W_mu, const float* W_rho,
                       const float* bias_mu, const float* bias_rho, void* y, float* kl_out, float* act_std,
                       const float* eps_a, const float* eps_b, uint64_t seed, uint64_t stream_id, const uint64_t* stream_base,
                       void* workspace, size_t workspace_bytes, void* cuda_stream) {
    return forward_impl(desc, false, x, W_mu, W_rho, bias_mu, bias_rho, y, kl_out, act_std, eps_a, eps_b, seed,
                        stream_id, stream_base, workspace, workspace_bytes, cuda_stream);
}

int bbb_linear_forward(const bbb_layer_desc* desc, const void* x, const float* W_mu, const float* W_rho,
                       const float* bias_mu, const float* bias_rho, void* y, float* kl_out, float* act_std,
                       const float* eps_a, const float* eps_b, uint64_t seed, uint64_t stream_id, const uint64_t* stream_base,
                       void* workspace, size_t workspace_bytes, void* cuda_stream) {
    return forward_impl(desc, true, x, W_mu, W_rho, bias_mu, bias_rho, y, kl_out, act_std, eps_a, eps_b, seed,
                        stream_id, stream_base, workspace, workspace_bytes, cuda_stream);
}

int bbb_conv2d_backward(const bbb_layer_desc* desc, const void* x, const void* grad_y, const float* W_mu,
                        const float* W_rho, const float* bias_mu, const float* bias_rho, const float* act_std,
                        const float* eps_a, const float* eps_b, uint64_t seed, uint64_t stream_id, const uint64_t* stream_base, void* grad_x,
                        float* g_W_mu, float* g_W_rho, float* g_bias_mu, float* g_bias_rho, void* workspace,
                        size_t workspace_bytes, void* cuda_stream) {
    return backward_impl(desc, false, x, grad_y, W_mu, W_rho, bias_mu, bias_rho, act_std, eps_a, eps_b, seed,
                         stream_id, stream_base, grad_x, g_W_mu, g_W_rho, g_bias_mu, g_bias_rho, workspace, workspace_bytes,
                         cuda_stream);
}

int bbb_linear_backward(const bbb_layer_desc* desc, const void* x, const void* grad_y, const float* W_mu,
                        const float* W_rho, const float* bias_mu, const float* bias_rho, const float* act_std,
                        const float* eps_a, const float* eps_b, uint64_t seed, uint64_t stream_id, const uint64_t* stream_base, void* grad_x,
                        float* g_W_mu, float* g_W_rho, float* g_bias_mu, float* g_bias_rho, void* workspace,
                        size_t workspace_bytes, void* cuda_stream) {
    return backward_impl(desc, true, x, grad_y, W_mu, W_rho, bias_mu, bias_rho, act_std, eps_a, eps_b, seed,
                         stream_id, stream_base, grad_x, g_W_mu, g_W_rho, g_bias_mu, g_bias_rho, workspace, workspace_bytes,
                         cuda_stream);
}

/* shape / layout checks of bbb_layer_forward_fused, callable without a GPU (host logic only) */
static int fused_check(const bbb_layer_desc* d, bbb::Geom& g, int32_t in_layout, int32_t in_pitch, int32_t prev_hw,
                       int32_t out_layout, int32_t out_pitch) {
    if (int rc = check_desc(d, g, false)) return rc;
    if (d->math == BBB_MATH_FP32 || d->math == BBB_MATH_TF32_TC) return fail(BBB_E_UNSUPPORTED, "the fused chain exists on the tcgen05 (bf16) path only");
    const int pool = d->pool_k != 0;
    if (pool && !(d->pool_k == 2 && d->pool_s == 2)) return fail(BBB_E_UNSUPPORTED, "only a 2x2 stride-2 max-pool can be fused");
    if (pool && ((g.OH | g.OW) & 1)) return fail(BBB_E_UNSUPPORTED, "fused pool needs even output height/width");
    if (out_layout == BBB_LAYOUT_PACKED_BF16 && (g.N % 64 || out_pitch != (pool ? g.OHW / 4 : g.OHW) * g.N))
        return fail(BBB_E_INVALID, "tiled packed output needs Cout %% 64 == 0 and out_pitch == pixels*Cout (got %d)", out_pitch);
    const int out_mode = out_layout == BBB_LAYOUT_PACKED_BF16 ? 0 : (out_layout == BBB_LAYOUT_ROWMAJOR_F32 ? 1 : 2);
    if (in_layout == BBB_LAYOUT_NCHW_F32) {
        if (!bbb::tc_supported(*d, g)) return fail(BBB_E_UNSUPPORTED, "shape not supported by the tcgen05 gather path");
        if (out_mode == 1 && (pool ? g.OHW / 4 : g.OHW) != 1) return fail(BBB_E_UNSUPPORTED, "row-major fp32 output needs a 1x1 map on the gather path");
    } else if (in_layout == BBB_LAYOUT_PACKED_BF16) {
        if (!bbb::fused_supported(g, pool)) return fail(BBB_E_UNSUPPORTED, "shape not supported by the fused tap-GEMM path");
        if (in_pitch != g.HW * g.Cin) return fail(BBB_E_INVALID, "tiled packed input: in_pitch must be pixels*Cin (got %d)", in_pitch);
        if (prev_hw < 1 || g.Cin % prev_hw) return fail(BBB_E_INVALID, "bad prev_hw %d", prev_hw);
    } else {
        return fail(BBB_E_INVALID, "bad in_layout %d", in_layout);
    }
    return BBB_OK;
}

int bbb_fused_supported(const bbb_layer_desc* d, int32_t in_layout, int32_t in_pitch, int32_t prev_hw,
                        int32_t out_layout, int32_t out_pitch) {
    bbb::Geom g;
    return fused_check(d, g, in_layout, in_pitch, prev_hw, out_layout, out_pitch);
}

/* which kernel runs a checked fused step: the stride-4 first-layer kernel, the gather kernel or the tap-GEMM */
enum { FUSED_KERNEL_CONV_S4 = 0, FUSED_KERNEL_GATHER = 1, FUSED_KERNEL_TAP_GEMM = 2 };
static int fused_kernel(const bbb_layer_desc* d, const bbb::Geom& g, int32_t in_layout, int32_t out_layout) {
    if (in_layout == BBB_LAYOUT_PACKED_BF16) return FUSED_KERNEL_TAP_GEMM;
    static const bool s4_on = [] { const char* e = getenv("BBB_B200_CONV1_DIRECT"); return !(e && e[0] == '0'); }();
    if (s4_on && bbb::conv_s4_supported(*d, g, d->pool_k != 0, out_layout == BBB_LAYOUT_PACKED_BF16)) return FUSED_KERNEL_CONV_S4;
    return FUSED_KERNEL_GATHER;
}

int bbb_layer_forward_fused(const bbb_layer_desc* d, const void* x, const void* x_sq, int32_t in_layout,
                            int32_t in_pitch, int32_t prev_hw, const float* W_mu, const float* W_rho,
                            const float* bias_mu, const float* bias_rho, void* y, void* y_sq, int32_t out_layout,
                            int32_t out_pitch, float* kl_out, const float* eps_a, const float* eps_b, uint64_t seed,
                            uint64_t stream_id, const uint64_t* stream_base, void* ws, size_t ws_bytes, void* stream) {
    bbb::Geom g;
    if (int rc = fused_check(d, g, in_layout, in_pitch, prev_hw, out_layout, out_pitch)) return rc;
    const bool prep_only = (d->reserved[0] & BBB_FUSED_PREP_ONLY) != 0, skip_prep = (d->reserved[0] & BBB_FUSED_SKIP_PREP) != 0;
    if (prep_only && skip_prep) return fail(BBB_E_INVALID, "PREP_ONLY and SKIP_PREP are exclusive");
    if (!W_mu || !W_rho || (!prep_only && (!x || !y))) return fail(BBB_E_INVALID, "NULL tensor pointer");
    if (d->has_bias && (!bias_mu || !bias_rho)) return fail(BBB_E_INVALID, "has_bias set but bias pointers NULL");
    const int pool = d->pool_k != 0;
    bbb::McFold fold; fold.rows = 0; fold.stride = 0;
    if (d->reserved[1] > 0) {           // MC samples folded into the batch
        if (d->variant != BBB_VARIANT_LRT || !d->sample || eps_a)
            return fail(BBB_E_UNSUPPORTED, "MC-sample folding needs the LRT variant with in-kernel Philox noise");
        if (g.B % d->reserved[1]) return fail(BBB_E_INVALID, "batch %d is not a multiple of the rows per MC sample %d", g.B, d->reserved[1]);
        fold.rows = d->reserved[1];
        fold.stride = ((unsigned long long)(uint32_t)d->reserved[3] << 32) | (uint32_t)d->reserved[2];
    }
    const size_t need = bbb_workspace_bytes(d);
    if (!ws || ws_bytes < need) return fail(BBB_E_WORKSPACE, "workspace too small for the fused path: need %zu bytes", need);
    if (out_layout == BBB_LAYOUT_PACKED_BF16 && y_sq && y_sq != (void*)((__nv_bfloat16*)y + 128 * 64))
        return fail(BBB_E_INVALID, "tiled packed output with squares: the planes are interleaved, y_sq must be y + 8192 elements");
    cudaStream_t st = (cudaStream_t)stream;
    const int out_mode = out_layout == BBB_LAYOUT_PACKED_BF16 ? 0 : (out_layout == BBB_LAYOUT_ROWMAJOR_F32 ? 1 : 2);
    int nl = 0;
    const int kernel = fused_kernel(d, g, in_layout, out_layout);
    if (kernel == FUSED_KERNEL_CONV_S4) {
        // stride-4 first layer: the tensor core reads its A operand straight from the staged image (conv_s4_tc.cuh)
        bbb::S4Args a;
        a.g = g; a.x = (const float*)x; a.w_mu = W_mu; a.w_rho = W_rho; a.b_mu = bias_mu; a.b_rho = bias_rho;
        a.y = y; a.y_sq = y_sq; a.kl_out = kl_out; a.eps_a = eps_a; a.eps_b = eps_b;
        a.key = bbb::make_key(seed, stream_id); a.stream_base = (const unsigned long long*)stream_base;
        a.kl_counter = (unsigned int*)ws; a.kl_partials = (double*)((char*)ws + kCounterBytes);
        a.prior_mu = d->prior_mu; a.prior_sigma = d->prior_sigma;
        a.sample = d->sample; a.kl_convention = d->kl_convention; a.has_bias = d->has_bias; a.act = d->epilogue_act;
        a.variant = d->variant; a.out_pitch = out_pitch;
        a.wtiles = (__nv_bfloat16*)((char*)ws + kTcOffset);
        a.bias_ws = (float*)((char*)ws + kTcOffset + (size_t)g.KH * 2 * bbb::S4_BPLANE);
        a.trace = g_trace; a.fold = fold;
        a.tl_prep = tl_slot(!skip_prep, "conv_s4_prep", g); a.tl_gemm = tl_slot(!prep_only, "conv_s4", g);
        cudaError_t e = bbb::launch_conv_s4(a, st, !skip_prep, !prep_only, &nl);
        if (e != cudaSuccess) return cuda_fail(e, "conv_s4 launch");
    } else if (kernel == FUSED_KERNEL_GATHER) {
        if (fold.rows) return fail(BBB_E_UNSUPPORTED, "MC-sample folding is not available on the gather path");
        bbb::TcArgs a;
        a.g = g; a.x = x; a.w_mu = W_mu; a.w_rho = W_rho; a.b_mu = bias_mu; a.b_rho = bias_rho;
        a.y = y; a.kl_out = kl_out; a.act_std = nullptr; a.eps_a = eps_a; a.eps_b = eps_b;
        a.key = bbb::make_key(seed, stream_id); a.stream_base = (const unsigned long long*)stream_base;
        a.kl_counter = (unsigned int*)ws; a.kl_partials = (double*)((char*)ws + kCounterBytes);
        a.prior_mu = d->prior_mu; a.prior_sigma = d->prior_sigma;
        a.sample = d->sample; a.kl_convention = d->kl_convention; a.has_bias = d->has_bias; a.act = d->epilogue_act;
        a.act_dtype = d->act_dtype; a.variant = d->variant;
        a.wtiles = (__nv_bfloat16*)((char*)ws + kTcOffset);
        a.bias_ws = (float*)((char*)ws + kTcOffset + (size_t)bbb::tc_npad(g) * bbb::tc_kpad(g) * 4);
        a.tf32 = 0;
        a.trace = g_trace; a.skip_prep = skip_prep; a.prep_only = prep_only; a.y_sq = y_sq; a.out_mode = out_mode == 1 ? 2 : out_mode; a.out_pitch = out_pitch; a.pool = pool;
        a.tl_prep = tl_slot(!skip_prep, "weight_prep", g); a.tl_gemm = tl_slot(!prep_only, "gemm_tc", g);
        cudaError_t e = bbb::launch_fwd_tc(a, st, sm_count(), &nl);
        if (e != cudaSuccess) return cuda_fail(e, "fused gather launch");
    } else {
        bbb::FusedArgs a;
        a.g = g; a.variant = d->variant; a.sample = d->sample; a.has_bias = d->has_bias; a.act = d->epilogue_act;
        a.kl_convention = d->kl_convention; a.prior_mu = d->prior_mu; a.prior_sigma = d->prior_sigma;
        a.w_mu = W_mu; a.w_rho = W_rho; a.b_mu = bias_mu; a.b_rho = bias_rho; a.eps_a = eps_a; a.eps_b = eps_b;
        a.key = bbb::make_key(seed, stream_id); a.stream_base = (const unsigned long long*)stream_base;
        a.kl_counter = (unsigned int*)ws; a.kl_partials = (double*)((char*)ws + kCounterBytes); a.kl_out = kl_out;
        const size_t cpad = (size_t)(g.N + 63) / 64 * 64, kpad = (size_t)(g.Cin + 63) / 64 * 64;
        a.wtiles = (__nv_bfloat16*)((char*)ws + kTcOffset);
        a.bias_ws = (float*)((char*)ws + kTcOffset + cpad * kpad * g.KHW * 4 + 32768);   // behind the zero sub-tile
        a.prev_hw = prev_hw; a.y = y; a.y_sq = y_sq; a.out_mode = out_mode; a.out_pitch = out_pitch; a.pool = pool;
        a.in_pitch = in_pitch; a.trace = g_trace; a.fold = fold;
        a.tl_prep = tl_slot(!skip_prep, "tap_prep", g); a.tl_gemm = tl_slot(!prep_only, "tap_gemm", g);
        const char* why = "";
        cudaError_t e = bbb::launch_fused(a, x, x_sq, st, &nl, &why, !skip_prep, !prep_only, sm_count(), g_wide_tiles.load() != 0);
        if (e != cudaSuccess) return fail(BBB_E_CUDA, "fused tap-GEMM launch: %s %s", cudaGetErrorString(e), why);
    }
    g_launches += nl;
    return BBB_OK;
}

int bbb_kl_forward(const float* W_mu, const float* W_rho, uint64_t n_w, const float* bias_mu,
                   const float* bias_rho, uint64_t n_b, float prior_mu, float prior_sigma, int32_t kl_convention,
                   float* kl_out, void* workspace, size_t workspace_bytes, void* cuda_stream) {
    if (!W_mu || !W_rho || !kl_out) return fail(BBB_E_INVALID, "NULL tensor pointer");
    if (n_b && (!bias_mu || !bias_rho)) return fail(BBB_E_INVALID, "n_b > 0 but bias pointers NULL");
    if (!workspace || workspace_bytes < kBaseWorkspace) return fail(BBB_E_WORKSPACE, "workspace too small: need %zu bytes", kBaseWorkspace);
    if (!(prior_sigma > 0.0f)) return fail(BBB_E_INVALID, "prior_sigma must be > 0");
    const uint64_t work = (n_w + 3) / 4 + n_b;
    uint64_t blocks = (work + 255) / 256;
    const uint64_t cap = (uint64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (blocks > kMaxKlSlots) blocks = kMaxKlSlots;
    bbb::kl_forward_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(
        W_mu, W_rho, n_w, bias_mu, bias_rho, n_b, prior_mu, prior_sigma, kl_convention,
        (double*)((char*)workspace + kCounterBytes), (unsigned int*)workspace, kl_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "kl_forward launch");
    g_launches += 1;
    return BBB_OK;
}

int bbb_kl_backward(const float* mu, const float* rho, uint64_t n, float prior_mu, float prior_sigma,
                    int32_t kl_convention, const float* grad_kl, float* g_mu, float* g_rho, void* cuda_stream) {
    if (!mu || !rho || !grad_kl || !g_mu || !g_rho) return fail(BBB_E_INVALID, "NULL tensor pointer");
    if (n == 0) return BBB_OK;
    uint64_t blocks = (n + 255) / 256;
    const uint64_t cap = (uint64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    bbb::kl_backward_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(
        mu, rho, n, prior_mu, prior_sigma, kl_convention, grad_kl, g_mu, g_rho);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "kl_backward launch");
    g_launches += 1;
    return BBB_OK;
}

int bbb_philox_normal_fill(float* out, uint64_t n, uint64_t seed, uint64_t stream_id, uint64_t offset,
                           void* cuda_stream) {
    if (!out) return fail(BBB_E_INVALID, "NULL output pointer");
    if (n == 0) return BBB_OK;
    uint64_t blocks = (n + 255) / 256;
    const uint64_t cap = (uint64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    bbb::philox_fill_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(out, n, bbb::make_key(seed, stream_id), offset);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "philox_fill launch");
    g_launches += 1;
    return BBB_OK;
}

int bbb_mc_combine(const float* logits, int32_t S, int32_t B, int32_t C, float* log_outputs, float* moments,
                   void* cuda_stream) {
    if (!logits || !log_outputs) return fail(BBB_E_INVALID, "NULL tensor pointer");
    if (S <= 0 || B <= 0 || C <= 0) return fail(BBB_E_INVALID, "bad S/B/C");
    if ((size_t)S * sizeof(float) > 40000) return fail(BBB_E_UNSUPPORTED, "S too large");
    bbb::mc_combine_kernel<<<B, 128, S * sizeof(float), (cudaStream_t)cuda_stream>>>(logits, S, B, C, log_outputs, moments);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "mc_combine launch");
    g_launches += 1;
    return BBB_OK;
}

size_t bbb_mc_buffer_bytes(int32_t B, int32_t C, int32_t flags, int32_t world) {
    if (B <= 0 || C <= 0 || world <= 0 || world > bbb::MCX_MAX_RANKS) return 0;
    return bbb::mcx_buffer_bytes(B, C, flags & BBB_MC_MOMENTS, world);
}
size_t bbb_mc_state_bytes(void) { return 64 + (size_t)bbb::MCX_MAX_CTAS * 2 * sizeof(double); }

int bbb_mc_exchange(const float* logits, int32_t S_local, int32_t S_total, int32_t B, int32_t C, const float* kl,
                    int32_t n_kl, int32_t flags, const int64_t* labels, float train_size, float beta, int32_t rank, int32_t world,
                    void* const* peer_buffers, void* state, float* log_outputs, float* kl_out, float* pred,
                    float* epistemic, float* aleatoric, float* entropy, float* head, uint64_t* noise_base,
                    uint64_t noise_inc, void* cuda_stream) {
    if (!log_outputs || !peer_buffers || !state) return fail(BBB_E_INVALID, "NULL pointer");
    if (S_local < 0 || S_total <= 0 || B <= 0 || C <= 0) return fail(BBB_E_INVALID, "bad S/B/C");
    if (S_local > 0 && !logits) return fail(BBB_E_INVALID, "S_local > 0 but logits is NULL");
    if (S_local > bbb::MCX_MAX_SLOCAL) return fail(BBB_E_UNSUPPORTED, "more than %d local samples per call", bbb::MCX_MAX_SLOCAL);
    if (world < 1 || world > bbb::MCX_MAX_RANKS || rank < 0 || rank >= world) return fail(BBB_E_INVALID, "bad rank/world %d/%d", rank, world);
    if ((pred || epistemic || aleatoric || entropy) && !(flags & BBB_MC_MOMENTS))
        return fail(BBB_E_INVALID, "uncertainty outputs need BBB_MC_MOMENTS");
    bbb::McxArgs a;
    a.logits = logits; a.kl = kl; a.n_kl = kl ? (n_kl > 0 ? n_kl : 1) : 0; a.S_local = S_local; a.S_total = S_total; a.B = B; a.C = C;
    a.want_moments = (flags & BBB_MC_MOMENTS) ? 1 : 0; a.normalized = (flags & BBB_MC_NORMALIZED) ? 1 : 0;
    a.labels = (const long long*)labels; a.train_size = train_size; a.beta = beta; a.rank = rank; a.world = world;
    for (int q = 0; q < bbb::MCX_MAX_RANKS; ++q) a.peer[q] = q < world ? (unsigned char*)peer_buffers[q] : nullptr;
    for (int q = 0; q < world; ++q) if (!a.peer[q]) return fail(BBB_E_INVALID, "peer buffer %d is NULL", q);
    a.seq = (unsigned int*)state; a.done = (unsigned int*)state + 1; a.timeouts = (unsigned int*)state + 2;
    a.noise_base = nullptr; a.noise_inc = 0;
    if (noise_base) { a.noise_base = (unsigned long long*)noise_base; a.noise_inc = noise_inc; }
    a.timeout_ns = 10ull * 1000 * 1000 * 1000;
    if (const char* e = getenv("BBB_B200_MC_TIMEOUT_MS")) a.timeout_ns = (unsigned long long)atoll(e) * 1000000ull;
    a.head_partials = (double*)((char*)state + 64);
    a.log_outputs = log_outputs; a.kl_out = kl_out; a.pred = pred; a.epistemic = epistemic; a.aleatoric = aleatoric;
    a.entropy = entropy; a.head = head; a.trace = g_mcx_trace;
    { bbb::Geom tg = {}; tg.M = B; tg.N = C; tg.K = S_local; a.tl = tl_slot(true, "mc_exchange", tg); }
    // the grid depends on B only: CTA c of every rank owns the same images, so flags pair up CTA by CTA.  At most
    // MCX_MAX_CTAS CTAs: all co-resident, so a CTA spinning on a peer's flag never keeps that peer's producer off an SM.
    int grid = (B + bbb::MCX_THREADS / 32 - 1) / (bbb::MCX_THREADS / 32);
    if (grid > bbb::MCX_MAX_CTAS) grid = bbb::MCX_MAX_CTAS;
    cudaError_t e = bbb::launch_pdl(bbb::mc_exchange_kernel, dim3(grid), dim3(bbb::MCX_THREADS),
                                     (size_t)(bbb::MCX_THREADS / 32) * S_local * sizeof(float), (cudaStream_t)cuda_stream, a);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "mc_exchange launch");
    g_launches += 1;
    return BBB_OK;
}

int bbb_comm_alloc(size_t bytes, void** dev_ptr) {
    if (!dev_ptr || bytes == 0) return fail(BBB_E_INVALID, "bad arguments");
    cudaError_t e = cudaMalloc(dev_ptr, bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    e = cudaMemset(*dev_ptr, 0, bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemset");
    e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceSynchronize");
    return BBB_OK;
}
int bbb_comm_free(void* dev_ptr) {
    cudaError_t e = cudaFree(dev_ptr);
    return e == cudaSuccess ? BBB_OK : cuda_fail(e, "cudaFree");
}
int bbb_comm_export(void* dev_ptr, void* handle64_host) {
    if (!dev_ptr || !handle64_host) return fail(BBB_E_INVALID, "NULL pointer");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, dev_ptr);
    if (e != cudaSuccess) return cuda_fail(e, "cudaIpcGetMemHandle");
    memcpy(handle64_host, &h, 64);
    return BBB_OK;
}
int bbb_comm_import(const void* handle64_host, void** peer_ptr) {
    if (!handle64_host || !peer_ptr) return fail(BBB_E_INVALID, "NULL pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64_host, 64);
    cudaError_t e = cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess);
    return e == cudaSuccess ? BBB_OK : cuda_fail(e, "cudaIpcOpenMemHandle");
}
int bbb_comm_unimport(void* peer_ptr) {
    cudaError_t e = cudaIpcCloseMemHandle(peer_ptr);
    return e == cudaSuccess ? BBB_OK : cuda_fail(e, "cudaIpcCloseMemHandle");
}

int bbb_noise_advance(uint64_t* base, uint64_t inc, void* cuda_stream) {
    if (!base) return fail(BBB_E_INVALID, "NULL base pointer");
    bbb::noise_advance_kernel<<<1, 1, 0, (cudaStream_t)cuda_stream>>>((unsigned long long*)base, (unsigned long long)inc);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "noise_advance launch");
    g_launches += 1;
    return BBB_OK;
}

/* debug only (not in the public header): per-CTA clock64 checkpoints of tap_gemm_kernel */
void bbb_debug_set_trace(void* dev_ptr) { g_trace = (long long*)dev_ptr; }
void bbb_debug_set_mcx_trace(void* dev_ptr) { g_mcx_trace = (long long*)dev_ptr; }
/* debug only: timeline slots (4 x int64 per instrumented launch; caller presets [INT64_MAX, 0, INT64_MAX, 0] before a run) */
void bbb_debug_set_timeline(void* dev_ptr, int capacity) { g_tl = (long long*)dev_ptr; g_tl_cap = capacity; g_tl_n = 0; }
int bbb_debug_timeline_count(void) { return g_tl_n; }
const char* bbb_debug_timeline_name(int k) { return (k >= 0 && k < g_tl_n) ? g_tl_names[k] : ""; }
/* debug only, host logic only: what bbb_layer_forward_fused launches for this step on a device with n_sm SMs and the
   given bbb_set_wide_tiles switch.  out[0] kernel (0 conv_s4, 1 gather, 2 tap-GEMM), out[1] tile width BN, out[2] CTAs
   per SM the GEMM kernel is built for (0 for the gather kernel: its occupancy follows from its shared-memory footprint),
   out[3] prep kernel (0 weight_prep, 1 conv_s4_prep, 2 tap_prep, 3 tap_prep_conv).  Returns the bbb_fused_supported
   status; out is written only on BBB_OK. */
int bbb_debug_fused_config(const bbb_layer_desc* d, int32_t in_layout, int32_t in_pitch, int32_t prev_hw, int32_t out_layout,
                           int32_t out_pitch, int32_t n_sm, int32_t prefer_wide, int32_t* out) {
    bbb::Geom g;
    if (int rc = fused_check(d, g, in_layout, in_pitch, prev_hw, out_layout, out_pitch)) return rc;
    if (!out || n_sm < 1) return fail(BBB_E_INVALID, "bbb_debug_fused_config: bad arguments");
    const int kernel = fused_kernel(d, g, in_layout, out_layout);
    out[0] = kernel;
    if (kernel == FUSED_KERNEL_CONV_S4) {
        out[1] = 64; out[2] = 1; out[3] = 1;         // Cout == 64; ~193 KB of shared memory per CTA
    } else if (kernel == FUSED_KERNEL_GATHER) {
        out[1] = bbb::TC_BN; out[2] = 0; out[3] = 0;
    } else {
        const bbb::TapConfig c = bbb::tap_config(g, bbb::tc_planes(d->variant, d->sample), d->pool_k != 0, prev_hw, n_sm,
                                                 prefer_wide != 0);
        out[1] = c.bn; out[2] = c.two_per_sm ? 2 : 1; out[3] = c.prep_conv ? 3 : 2;
    }
    return BBB_OK;
}

const char* bbb_last_error(void) { return g_err; }
int32_t bbb_abi_version(void) { return BBB_ABI_VERSION; }
uint64_t bbb_launch_count(void) { return g_launches.load(); }
int32_t bbb_set_wide_tiles(int32_t prefer_wide) { return g_wide_tiles.exchange(prefer_wide ? 1 : 0); }

}  // extern "C"
