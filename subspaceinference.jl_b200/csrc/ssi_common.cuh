// ssi_common.cuh — context, error plumbing and small device helpers shared by all
// translation units of libssi.so.  Internal; the public surface is include/ssi.h.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/ssi.h"

#define SSI_MAX_LAYERS 16
#define SSI_MAX_M      64

struct ssi_model_t {
    int L = 0;
    int dims[SSI_MAX_LAYERS + 1] = {0};
    int act[SSI_MAX_LAYERS] = {0};
    int64_t w_off[SSI_MAX_LAYERS] = {0};   // offset of vec(W_l) in the flat vector
    int64_t b_off[SSI_MAX_LAYERS] = {0};   // offset of b_l
    int64_t n = 0;                         // n_params
    int max_width = 0;                     // max over dims[0..L]
    double flops_per_point = 0;            // 2*sum(in*out)
};

// Scratch that grows on demand and is reused between calls.
struct ssi_buf_t {
    void* p = nullptr;
    size_t cap = 0;
};

struct ssi_tc_state;   // tensor-core path private state (ssi_tc.cu)
struct ssi_b1_state;   // basis path private state (ssi_basis.cu)
struct ssi_bm_state;   // basis path on the tensor cores (ssi_basis_mma.cu)
struct ssi_train_state; // on-device training step (ssi_train.cu)
struct ssi_decoder_t;   // non-linear subspace operator (ssi_decoder.cu)

struct ssi_ctx {
    // A multi-device context (ssi_ctx_create_multi) owns one ordinary context per device and no device state of its own:
    // set_* calls are replicated, batched calls are sharded by sample / chain index (SURVEY 8(b)-1, 8(e)).
    std::vector<ssi_ctx*> children;
    bool is_multi() const { return !children.empty(); }
    int device = 0;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    size_t smem_optin = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_stage[4] = {nullptr, nullptr, nullptr, nullptr};   // boundaries of the stages of ssi_swa_finish
    bool stage_pending = false;
    std::string err;

    // options
    int opt_path = SSI_PATH_AUTO;
    int opt_group = 0;
    int opt_tc_nofuse = 0;    // debugging / A-B: compute the output layer as its own GEMM
    int opt_tc_noorder = 0;   // debugging / A-B: sample-major work order on the first layer
    int opt_grad_group_gb = 0; // scratch budget (GB) of the generic gradient path per group of samples (default 6)
    int opt_gemm_simt = 0;    // 1: keep the gradient / training GEMMs on the SIMT kernel (A-B against ssi_gemm_tc.cu)
    int opt_mala_rule = 0;    // 0 textbook MALA ratio, 1 negated-gradient proposal densities (see ssi_api.cu)
    int opt_tc_pair = 1;      // GEMM layers with per-sample activations as CTA pairs (cta_group::2); 0: one CTA per tile (A-B)
    int opt_tc_prec = 1;      // operand planes of the tensor path: 1 mixed BF16/FP16 (default), 0 BF16x3 (round 1)
    int opt_b1_simt = 0;       // A-B: BASIS path on CUDA cores (k_logpost_basis1h) instead of the tensor-core kernel (k_b1_mma)
    int opt_tc_simt_basis = 0; // A-B: first layer as the FP32 SIMT basis combination instead of the tensor-core one
    int opt_gram_fp64 = 0;    // force the FP64 SIMT Gram (default: tensor-core TF32x2 Gram for large n, K <= 128)
    int opt_tc_nobasis = 0;   // debugging / A-B: run the first layer as a GEMM instead of the affine-in-z basis combination

    // model / data / subspace
    ssi_model_t model;
    bool has_model = false, has_data = false, has_sub = false;
    float* dX = nullptr;      // in0 x N
    float* dY = nullptr;      // O x N
    int64_t N = 0;
    float* dWswa = nullptr;   // n
    float* dP = nullptr;      // n x M
    int M = 0;                // columns of P (the dimension the kernels work in)
    int Mz = 0;               // dimension of the caller's z: M, or the input width of a decoder (ssi_set_decoder)
    // non-linear subspace operator: W = W_swa + decoder(z); P / dWswa then hold the decoder's affine head
    ssi_decoder_t* dec = nullptr;
    bool dec_active = false;
    int dec_out_act = SSI_ACT_IDENTITY;   // activation of the decoder's last layer
    float* dWbase = nullptr;              // W_swa proper when that activation is not the identity (W = dWbase + act(dWswa + P z'))
    ssi_buf_t bDecZ, bDecT;
    // M-space quantities for the weight prior: G = [P | W_swa]^T [P | W_swa]  ((M+1)x(M+1), double)
    double* dSubGram = nullptr;

    // scratch
    ssi_buf_t bZ, bLp, bTerms, bPartials, bW, bH0, bH1, bGram, bEig, bMisc, bGradW, bGradP;
    ssi_buf_t bGemmAmax;      // per-batch operand magnitudes of the tensor-core GEMM in flight (ssi_gemm_tc.cu)
    ssi_buf_t bSkinny;        // contraction-slice partials of the skinny weight-gradient kernel (ssi_gemm.cu)
    ssi_buf_t bRowsum;        // per-slice partials of the bias gradients (ssi_gemm.cu)

    // MH state
    ssi_buf_t bMhZ, bMhZp, bMhLp, bMhLpP, bMhCnt, bMhG;
    int64_t mh_chains = 0;       // chains of the last run (ssi_mh_get_state)
    int mh_kind = -1;            // sampler of the last run: 0 RWMH, 1 MALA, 2 HMC (ssi_hmc_get_adapt needs 2)
    // HMC integrator (ssi_hmc.cu): momentum (M x C), start energy, step size of the transition, divergence flag (C each),
    // dual-averaging state (3 x C: log eps, log eps_bar, H_bar)
    ssi_buf_t bHmcP, bHmcH0, bHmcEps, bHmcDiv, bHmcAd;

    // SWA / construction state
    int64_t swa_n = 0, swa_Kmax = 0, swa_K = 0;
    int64_t swa_ld = 0;          // leading dimension of dDev: n rounded up to 32 (columns 128-byte aligned for float4 / TMA)
    float* dSwaMean = nullptr;   // n
    float* dDev = nullptr;       // n x K_max, column-major
    float* dSwaAmax = nullptr;   // running max |deviation| over all pushes (scale of the Gram's FP16 planes)
    ssi_buf_t bSnap;

    // tensor-core path
    ssi_tc_state* tc = nullptr;
    // basis path (one hidden layer, narrow output)
    ssi_b1_state* b1 = nullptr;
    ssi_bm_state* bm = nullptr;
    // mini-batch training state (the step before the path)
    ssi_train_state* train = nullptr;

    // stats
    ssi_stats_t stats{};

    // optional device timing of the path's dominant kernel (option "time_dominant"): event pairs recorded around
    // each launch on the launching stream, summed into stats.dominant_ms at the next ssi_sync / ssi_stats
    int opt_time_dominant = 0;
    std::vector<cudaEvent_t> kt_events;
    size_t kt_used = 0;
};

// bracket a launch of the dominant kernel (no-ops unless "time_dominant" is set)
void ssi_kt_begin(ssi_ctx* ctx);
void ssi_kt_end(ssi_ctx* ctx);
void ssi_kt_collect(ssi_ctx* ctx);

// ---- error plumbing -------------------------------------------------------------------
int ssi_fail(ssi_ctx* ctx, int code, const char* fmt, ...);

#define SSI_CUDA(ctx, call)                                                              \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess)                                                          \
            return ssi_fail((ctx), SSI_ERR_CUDA, "%s failed at %s:%d: %s", #call,        \
                            __FILE__, __LINE__, cudaGetErrorString(e__));                \
    } while (0)

// entry points a multi-device context does not take (device pointers belong to one device)
#define SSI_NO_MULTI(ctx, what)                                                          \
    do {                                                                                 \
        if ((ctx)->is_multi())                                                           \
            return ssi_fail((ctx), SSI_ERR_UNSUPPORTED, "%s are not available on a multi-device context: use the host-pointer call", what); \
    } while (0)

#define SSI_TRY(expr)                                                                    \
    do {                                                                                 \
        int rc__ = (expr);                                                               \
        if (rc__ != SSI_OK) return rc__;                                                 \
    } while (0)

#define SSI_LAUNCH_CHECK(ctx)                                                            \
    do {                                                                                 \
        (ctx)->stats.kernel_launches++;                                                  \
        SSI_CUDA((ctx), cudaGetLastError());                                             \
    } while (0)

int ssi_reserve(ssi_ctx* ctx, ssi_buf_t& b, size_t bytes);
// cuTensorMapEncodeTiled through the runtime's driver entry point lookup (thread-safe, looked up once per process)
typedef CUresult (*PFN_ssi_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int ssi_tensormap_encoder(ssi_ctx* ctx, PFN_ssi_encodeTiled* out);
int ssi_use_device(ssi_ctx* ctx);
int ssi_sync_internal(ssi_ctx* ctx);     // stream sync + timers, without the public ssi_sync's range report

// ---- multi-device dispatch (ssi_multi.cu) ------------------------------------------------
int ssi_multi_create(const int32_t* devices, int32_t n_dev, ssi_ctx** out);
int ssi_multi_destroy(ssi_ctx* ctx);
int ssi_multi_sync(ssi_ctx* ctx);
int ssi_multi_set_option(ssi_ctx* ctx, const char* key, int64_t value);
int ssi_multi_stats(const ssi_ctx* ctx, ssi_stats_t* out);
int ssi_multi_set_model(ssi_ctx* ctx, int n_layers, const int32_t* dims, const int32_t* act);
int ssi_multi_set_data(ssi_ctx* ctx, const float* X, const float* Y, int64_t N);
int ssi_multi_set_subspace(ssi_ctx* ctx, const float* W_swa, const float* P, int64_t n, int32_t M);
int ssi_multi_logpost(ssi_ctx* ctx, int grad, const float* Z, int64_t B, double sigma_m, double sigma_p, double sigma_z, uint32_t mask,
                      double* lp_out, double* second_out);
// One sampler run, as a public sampler entry point (include/ssi.h) received it and checked it.  Host pointers down to
// ssi_mh_run_host_slice, which hands ssi_mh_device its shard's descriptor with device pointers.
struct ssi_mh_run_t {
    int kind = 0;                           // 0 RWMH, 1 MALA, 2 HMC
    int64_t n_chains = 0, n_steps = 0;
    uint64_t seed = 0;
    int64_t chain_offset = 0, step_offset = 0;
    double sigma_z = 1.0, sigma_m = 1.0, sigma_p = 1.0;
    uint32_t mask = 0;
    const ssi_hmc_params_t* hp = nullptr;   // kind 2 only, as are adapt0 and step_size_trace
    const float* z0 = nullptr;
    const double* adapt0 = nullptr;
    float* z_trace = nullptr;
    double* lp_trace = nullptr;
    uint8_t* accept_trace = nullptr;
    double* step_size_trace = nullptr;
};

int ssi_multi_mh_run(ssi_ctx* ctx, const ssi_mh_run_t& run);
int ssi_multi_mh_get_state(ssi_ctx* ctx, float* z_out, double* lp_out);
int ssi_multi_hmc_get_adapt(ssi_ctx* ctx, double* adapt_out);
int ssi_multi_project(ssi_ctx* ctx, const float* Z, int64_t B, float* W_out);
int ssi_multi_swa_finish(ssi_ctx* ctx, int32_t M, float* W_swa_out, float* P_out, double* s_out, int32_t install);
// per-device halves of the host-pointer MH entry points (ssi_api.cu): chains [c0, c1) of `run`, and the state of the
// n chains of the last run on this device
int ssi_mh_run_host_slice(ssi_ctx* ctx, const ssi_mh_run_t& run, int64_t c0, int64_t c1);
int ssi_mh_get_state_slice(ssi_ctx* ctx, int64_t n, float* z_out, double* lp_out);
int ssi_hmc_get_adapt_slice(ssi_ctx* ctx, int64_t n, double* adapt_out);

// ---- samplers (ssi_mh.cu, ssi_hmc.cu) --------------------------------------------------------
// the run on this device; every pointer of `run` is a device pointer
int ssi_mh_device(ssi_ctx* ctx, const ssi_mh_run_t& run);
// the samplers' one density call: log-density (kind 0) or log-density and gradient (kinds 1, 2) of the run's n_chains
// points zp into lpp (and gp), the work added to *units / *flops; the only place the run's sigmas meet the density's order
int ssi_mh_density(ssi_ctx* ctx, const ssi_mh_run_t& run, const float* zp, double* lpp, double* gp, double* units, double* flops);
int ssi_hmc_check(ssi_ctx* ctx, const ssi_hmc_params_t* hp, int M);
int ssi_hmc_prepare(ssi_ctx* ctx, const ssi_mh_run_t& run);
int ssi_hmc_transition(ssi_ctx* ctx, const ssi_mh_run_t& run, int64_t i, double* units, double* flops);

// ---- decoder (ssi_decoder.cu) -------------------------------------------------------------
void ssi_dec_destroy(ssi_ctx* ctx);
int ssi_set_decoder_impl(ssi_ctx* ctx, const float* W_swa, int n_layers, const int32_t* dims, const int32_t* act, const float* theta);
int ssi_dec_project(ssi_ctx* ctx, const float* dZ, int64_t B, const float** dZin);      // z -> z' = h(z) (device, scratch)
int ssi_dec_logpost(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p, double sigma_z, uint32_t mask,
                    double* d_lp, double* d_terms);
int ssi_dec_logpost_grad(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p, double sigma_z, uint32_t mask,
                         double* d_lp, double* d_grad);
int ssi_multi_set_decoder(ssi_ctx* ctx, const float* W_swa, int n_layers, const int32_t* dims, const int32_t* act, const float* theta);

// ---- entry points between translation units --------------------------------------------
// log-posterior of B device-resident subspace points; d_lp (B) and optional d_terms (3 x B)
int ssi_logpost_device(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p,
                       double sigma_z, uint32_t mask, double* d_lp, double* d_terms);
int ssi_project_device(ssi_ctx* ctx, const float* dZ, int64_t B, float* dW /* ldw x B */, int64_t ldw = 0 /* 0: n */);
int ssi_logpost_finalize(ssi_ctx* ctx, const double* d_sse, const float* dZ, int64_t B, double sigma_m, double sigma_p,
                         double sigma_z, uint32_t mask, double* d_lp, double* d_terms);
// value and gradient (M x B doubles) of the log-posterior of B device-resident subspace points (ssi_grad.cu)
int ssi_logpost_grad_device(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p, double sigma_z,
                            uint32_t mask, double* d_lp, double* d_grad);
int ssi_predict_device(ssi_ctx* ctx, const float* dZ, int64_t B, const float* dXg, int64_t Ng,
                       float* d_preds, double* d_mean, double* d_std, double* d_m2);
int ssi_build_first_layer_bases(ssi_ctx* ctx, float* bases, int ld);
int ssi_subspace_gram(ssi_ctx* ctx);   // fills dSubGram after set_subspace
// Gram of an n x K column-major FP32 matrix (ld = n) into a K x K double matrix on device
// Gram of an n x K column-major FP32 matrix with leading dimension ld
int ssi_gram_device(ssi_ctx* ctx, const float* dA, int64_t n, int64_t ld, int K, double* dG, bool allow_tensor, const float* d_amax);
bool ssi_gram_tc_usable(const ssi_ctx* ctx, const float* dA, int64_t n, int64_t ld, int K);
int ssi_gram_tc_device(ssi_ctx* ctx, const float* dA, int64_t n, int64_t ld, int K, double* dG, const float* d_amax);

// tensor-core path (ssi_tc.cu)
bool ssi_tc_supported(const ssi_ctx* ctx);
bool ssi_tc_preferred(const ssi_ctx* ctx);   // AUTO picks the tensor path only when padding waste is small
int  ssi_tc_prepare(ssi_ctx* ctx);        // after model+data(+subspace) change
void ssi_tc_invalidate(ssi_ctx* ctx);
void ssi_tc_destroy(ssi_ctx* ctx);
// SSE (sum of squared errors) of B samples into d_sse (B doubles)
int  ssi_tc_sse(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse);
// FP16 planes: has an evaluation since the last check left the calibrated range?  (synchronises; switches to BF16 planes)
int  ssi_tc_range_exceeded(ssi_ctx* ctx, bool* exceeded);

// basis path (ssi_basis.cu): Chain(Dense, Dense) with O <= 2, small M
bool ssi_b1_supported(const ssi_ctx* ctx);
int  ssi_b1_prepare(ssi_ctx* ctx);
void ssi_b1_invalidate(ssi_ctx* ctx);
void ssi_b1_destroy(ssi_ctx* ctx);
int  ssi_b1_sse(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse);
// value + likelihood gradient: SSE (B doubles) and per-tile gradient partials [n_tiles][M x B] floats (returned pointer)
bool ssi_b1_grad_supported(const ssi_ctx* ctx);
int  ssi_b1_grad_sse(ssi_ctx* ctx, const float* dZ, int64_t B, double coef, double* d_sse, float** d_gpart, int* n_parts);

// basis path on the tensor cores (ssi_basis_mma.cu): O = 1, H <= 64, M + 1 <= 32
bool ssi_bm_supported(const ssi_ctx* ctx);
void ssi_bm_invalidate(ssi_ctx* ctx);
void ssi_bm_destroy(ssi_ctx* ctx);
int  ssi_bm_sse(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse);
// on-device training step (ssi_train.cu)
void ssi_train_destroy(ssi_ctx* ctx);
int  ssi_train_begin_impl(ssi_ctx* ctx, const float* W0, int kind, double eta, double b1, double b2);
int  ssi_train_step_impl(ssi_ctx* ctx, const int64_t* idx, int64_t j0, int64_t nb, double* loss_out);
const float* ssi_train_weights_device(ssi_ctx* ctx);

// ---- device helpers ---------------------------------------------------------------------
__device__ __forceinline__ float ssi_act(float v, int act) {
    switch (act) {
        case SSI_ACT_RELU:    return fmaxf(v, 0.0f);
        case SSI_ACT_TANH:    return tanhf(v);
        case SSI_ACT_SIGMOID: return 1.0f / (1.0f + expf(-v));
        default:              return v;
    }
}

// act'(pre) written in terms of the output h = act(pre)
__device__ __forceinline__ float act_deriv_from_output(float h, int act) {
    switch (act) {
        case SSI_ACT_RELU:    return h > 0.0f ? 1.0f : 0.0f;
        case SSI_ACT_TANH:    return 1.0f - h * h;
        case SSI_ACT_SIGMOID: return h * (1.0f - h);
        default:              return 1.0f;
    }
}

__device__ __forceinline__ double ssi_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float ssi_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum in double; result valid in thread 0.  `red` needs 32 doubles of shared memory.
__device__ __forceinline__ double ssi_block_sum(double v, double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = ssi_warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        v = lane < nw ? red[lane] : 0.0;
        v = ssi_warp_sum(v);
    }
    return v;
}
