// ssi_api.cu — the extern "C" surface declared in include/ssi.h: context lifecycle,
// host<->device staging and per-call timing.  All compute is in the other .cu files.
#include "ssi_common.cuh"
#include "ssi_rng.cuh"

#include <cstdarg>
#include <cmath>
#include <mutex>

#include <nvtx3/nvToolsExt.h>        // header-only: NVTX ranges cost nothing unless a profiler is attached (SURVEY 5, tracing)
struct nvtx_range {
    explicit nvtx_range(const char* name) { nvtxRangePushA(name); }
    ~nvtx_range() { nvtxRangePop(); }
};
#define SSI_NVTX(name) nvtx_range nvtx_range__(name)

int ssi_mh_fetch_accepts(ssi_ctx*);
int ssi_swa_push_device(ssi_ctx*, const float*, double);
int ssi_swa_factor_device(ssi_ctx*, int, float*, double*, int*);
int ssi_swa_gram_stage(ssi_ctx*, bool, double*, bool*);
int ssi_swa_eigen_stage(ssi_ctx*, int, const double*, bool, bool*);
int ssi_swa_p_stage(ssi_ctx*, int, float*, double*, int*);

static std::mutex g_err_mu;
static std::string g_create_err;

int ssi_fail(ssi_ctx* ctx, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) {
        ctx->err = buf;
    } else {
        std::lock_guard<std::mutex> lk(g_err_mu);
        g_create_err = buf;
    }
    return code;
}

int ssi_use_device(ssi_ctx* ctx) {
    SSI_CUDA(ctx, cudaSetDevice(ctx->device));
    return SSI_OK;
}

int ssi_reserve(ssi_ctx* ctx, ssi_buf_t& b, size_t bytes) {
    if (bytes <= b.cap && b.p) return SSI_OK;
    if (b.p) {
        SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        SSI_CUDA(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    const size_t want = bytes < 256 ? 256 : bytes;
    SSI_CUDA(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
    return SSI_OK;
}

int ssi_tensormap_encoder(ssi_ctx* ctx, PFN_ssi_encodeTiled* out) {
    static std::once_flag once;
    static PFN_ssi_encodeTiled fn = nullptr;
    std::call_once(once, []() {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PFN_ssi_encodeTiled)f;
        (void)cudaGetLastError();
    });
    if (!fn) return ssi_fail(ctx, SSI_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
    *out = fn;
    return SSI_OK;
}

static void free_buf(ssi_buf_t& b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

#define SSI_KT_MAX_PAIRS 16384
void ssi_kt_begin(ssi_ctx* ctx) {
    if (!ctx->opt_time_dominant || ctx->kt_used + 2 > 2 * SSI_KT_MAX_PAIRS) return;
    while (ctx->kt_events.size() < ctx->kt_used + 2) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) { (void)cudaGetLastError(); return; }
        ctx->kt_events.push_back(e);
    }
    cudaEventRecord(ctx->kt_events[ctx->kt_used], ctx->stream);
}
void ssi_kt_end(ssi_ctx* ctx) {
    if (!ctx->opt_time_dominant || ctx->kt_events.size() < ctx->kt_used + 2) return;
    cudaEventRecord(ctx->kt_events[ctx->kt_used + 1], ctx->stream);
    ctx->kt_used += 2;
}
// after the stream has been synchronised
void ssi_kt_collect(ssi_ctx* ctx) {
    for (size_t i = 0; i + 1 < ctx->kt_used; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ctx->kt_events[i], ctx->kt_events[i + 1]) == cudaSuccess) {
            ctx->stats.dominant_ms += ms;
            ctx->stats.dominant_launches++;
        }
    }
    ctx->kt_used = 0;
    (void)cudaGetLastError();
}

struct call_timer {
    ssi_ctx* ctx;
    explicit call_timer(ssi_ctx* c) : ctx(c) { cudaEventRecord(c->ev0, c->stream); }
    void stop(bool sync) {
        cudaEventRecord(ctx->ev1, ctx->stream);
        if (sync) {
            cudaEventSynchronize(ctx->ev1);
            float ms = 0;
            cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
            ctx->stats.last_ms = ms;
        }
    }
};

extern "C" {

int ssi_version(void) { return SSI_VERSION; }

const char* ssi_last_error(const ssi_ctx* ctx) {
    if (ctx) return ctx->err.c_str();
    std::lock_guard<std::mutex> lk(g_err_mu);
    return g_create_err.c_str();
}

int ssi_ctx_create(int device, ssi_ctx** out) {
    if (!out) return ssi_fail(nullptr, SSI_ERR_ARG, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return ssi_fail(nullptr, SSI_ERR_CUDA, "no CUDA device available (%s); libssi has no CPU fallback",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= count) return ssi_fail(nullptr, SSI_ERR_ARG, "device %d out of range [0,%d)", device, count);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
        return ssi_fail(nullptr, SSI_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return ssi_fail(nullptr, SSI_ERR_CUDA, "device %d is sm_%d%d; libssi is built for sm_100a only", device, prop.major, prop.minor);
    ssi_ctx* ctx = new ssi_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    ctx->stats.sm_count = prop.multiProcessorCount;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) {
        ssi_fail(nullptr, SSI_ERR_CUDA, "context setup failed: %s", cudaGetErrorString(e));
        delete ctx;
        return SSI_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    *out = ctx;
    return SSI_OK;
}

int ssi_ctx_create_multi(const int32_t* devices, int32_t n_dev, ssi_ctx** out) { return ssi_multi_create(devices, n_dev, out); }

int ssi_ctx_devices(const ssi_ctx* ctx) { return ctx ? (ctx->is_multi() ? (int)ctx->children.size() : 1) : 0; }

int ssi_ctx_destroy(ssi_ctx* ctx) {
    if (!ctx) return SSI_OK;
    if (ctx->is_multi()) return ssi_multi_destroy(ctx);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ssi_dec_destroy(ctx);
    ssi_tc_destroy(ctx);
    ssi_b1_destroy(ctx);
    ssi_bm_destroy(ctx);
    ssi_train_destroy(ctx);
    cudaFree(ctx->dX); cudaFree(ctx->dY); cudaFree(ctx->dP); cudaFree(ctx->dSubGram);
    cudaFree(ctx->dSwaMean); cudaFree(ctx->dDev); cudaFree(ctx->dSwaAmax);
    ssi_buf_t* bufs[] = {&ctx->bZ, &ctx->bLp, &ctx->bTerms, &ctx->bPartials, &ctx->bW, &ctx->bH0, &ctx->bH1, &ctx->bGram,
                         &ctx->bEig, &ctx->bMisc, &ctx->bDecZ, &ctx->bDecT, &ctx->bGradW, &ctx->bGradP, &ctx->bRowsum, &ctx->bSkinny, &ctx->bGemmAmax, &ctx->bMhZ, &ctx->bMhZp, &ctx->bMhLp, &ctx->bMhLpP, &ctx->bMhCnt, &ctx->bMhG, &ctx->bSnap,
                         &ctx->bHmcP, &ctx->bHmcH0, &ctx->bHmcEps, &ctx->bHmcDiv, &ctx->bHmcAd};
    for (ssi_buf_t* b : bufs) free_buf(*b);
    for (cudaEvent_t e : ctx->kt_events) cudaEventDestroy(e);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    for (cudaEvent_t ev : ctx->ev_stage)
        if (ev) cudaEventDestroy(ev);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return SSI_OK;
}

int ssi_set_stream(ssi_ctx* ctx, void* cuda_stream) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NO_MULTI(ctx, "caller-provided streams");
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return SSI_OK;
}

int ssi_sync(ssi_ctx* ctx) {
    if (!ctx) return SSI_ERR_ARG;
    if (ctx->is_multi()) return ssi_multi_sync(ctx);
    SSI_TRY(ssi_sync_internal(ctx));
    // asynchronous tensor-path evaluations cannot be repeated behind the caller's back: report them
    bool exceeded = false;
    SSI_TRY(ssi_tc_range_exceeded(ctx, &exceeded));
    if (exceeded)
        return ssi_fail(ctx, SSI_ERR_RANGE, "an activation left the calibrated FP16 range of the tensor path: results of the *_dev calls since "
                                            "the last ssi_sync are invalid; the context now uses BF16 planes, repeat those calls");
    return SSI_OK;
}

}  // extern "C"

int ssi_sync_internal(ssi_ctx* ctx) {
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    if (cudaEventQuery(ctx->ev1) == cudaSuccess && cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess)
        ctx->stats.last_ms = ms;
    if (ctx->stage_pending) {
        float g = 0, e = 0, f = 0;
        if (cudaEventElapsedTime(&g, ctx->ev_stage[0], ctx->ev_stage[1]) == cudaSuccess && cudaEventElapsedTime(&e, ctx->ev_stage[1], ctx->ev_stage[2]) == cudaSuccess &&
            cudaEventElapsedTime(&f, ctx->ev_stage[2], ctx->ev_stage[3]) == cudaSuccess) {
            ctx->stats.finish_gram_ms = g; ctx->stats.finish_eigen_ms = e; ctx->stats.finish_p_ms = f;
        }
        ctx->stage_pending = false;
    }
    (void)cudaGetLastError();
    ssi_kt_collect(ctx);
    return SSI_OK;
}

extern "C" {

int ssi_set_option(ssi_ctx* ctx, const char* key, int64_t value) {
    if (!ctx || !key) return SSI_ERR_ARG;
    if (ctx->is_multi()) return ssi_multi_set_option(ctx, key, value);
    if (!strcmp(key, "path")) {
        if (value < SSI_PATH_AUTO || value > SSI_PATH_BASIS) return ssi_fail(ctx, SSI_ERR_ARG, "path must be one of SSI_PATH_*");
        ctx->opt_path = (int)value;
        return SSI_OK;
    }
    if (!strcmp(key, "group")) {
        if (value < 0 || value > 4096) return ssi_fail(ctx, SSI_ERR_ARG, "group out of range");
        ctx->opt_group = (int)value;
        ssi_tc_invalidate(ctx); ssi_b1_invalidate(ctx); ssi_bm_invalidate(ctx);
        return SSI_OK;
    }
    if (!strcmp(key, "tc_nofuse")) { ctx->opt_tc_nofuse = value != 0; ssi_tc_invalidate(ctx); ssi_b1_invalidate(ctx); ssi_bm_invalidate(ctx); return SSI_OK; }
    // gram_fp64: 1 = always the FP64 SIMT Gram, 0 = tensor-core Gram guarded by the conditioning check (default),
    // -1 = tensor-core Gram without the check (measurement only)
    if (!strcmp(key, "gram_fp64")) { ctx->opt_gram_fp64 = (int)value; return SSI_OK; }
    if (!strcmp(key, "tc_nobasis")) { ctx->opt_tc_nobasis = value != 0; ssi_tc_invalidate(ctx); ssi_b1_invalidate(ctx); ssi_bm_invalidate(ctx); return SSI_OK; }
    if (!strcmp(key, "time_dominant")) {
        ctx->opt_time_dominant = value != 0;
        ctx->stats.dominant_ms = 0; ctx->stats.dominant_launches = 0; ctx->kt_used = 0;
        return SSI_OK;
    }
    if (!strcmp(key, "grad_group_gb")) { ctx->opt_grad_group_gb = (int)value; return SSI_OK; }
    if (!strcmp(key, "gemm_simt")) { ctx->opt_gemm_simt = value != 0; return SSI_OK; }
    // MALA acceptance rule: 0 (default) = the Metropolis-adjusted Langevin ratio as documented; 1 = both proposal densities
    // evaluated with the NEGATED gradient, q(a | b) = N(a - b; -(sigma^2/2) grad(a), sigma^2) -- how AdvancedMH's MALA step is
    // remembered to be written (`spl.proposal(-t_cond.gradient)`); the pinned 0.6.2 source is not available to decide
    if (!strcmp(key, "mala_rule")) { if (value != 0 && value != 1) return ssi_fail(ctx, SSI_ERR_ARG, "mala_rule must be 0 or 1"); ctx->opt_mala_rule = (int)value; return SSI_OK; }
    if (!strcmp(key, "tc_pair")) { ctx->opt_tc_pair = value != 0; return SSI_OK; }
    if (!strcmp(key, "tc_precision")) { ctx->opt_tc_prec = value != 0; ssi_tc_invalidate(ctx); return SSI_OK; }
    if (!strcmp(key, "b1_simt")) { ctx->opt_b1_simt = value != 0; return SSI_OK; }
    if (!strcmp(key, "tc_simt_basis")) { ctx->opt_tc_simt_basis = value != 0; ssi_tc_invalidate(ctx); return SSI_OK; }
    if (!strcmp(key, "tc_noorder")) { ctx->opt_tc_noorder = value != 0; return SSI_OK; }
    return ssi_fail(ctx, SSI_ERR_ARG, "unknown option '%s'", key);
}

int ssi_stats(const ssi_ctx* ctx, ssi_stats_t* out) {
    if (!ctx || !out) return SSI_ERR_ARG;
    if (ctx->is_multi()) return ssi_multi_stats(ctx, out);
    *out = ctx->stats;
    return SSI_OK;
}

int ssi_set_model(ssi_ctx* ctx, int n_layers, const int32_t* dims, const int32_t* act) {
    if (!ctx) return SSI_ERR_ARG;
    if (ctx->is_multi()) return ssi_multi_set_model(ctx, n_layers, dims, act);
    if (n_layers < 1 || n_layers > SSI_MAX_LAYERS || !dims || !act)
        return ssi_fail(ctx, SSI_ERR_ARG, "n_layers must be in [1,%d] and dims/act non-NULL", SSI_MAX_LAYERS);
    ssi_model_t m;
    m.L = n_layers;
    int64_t off = 0;
    double fl = 0;
    for (int l = 0; l <= n_layers; ++l) {
        if (dims[l] < 1) return ssi_fail(ctx, SSI_ERR_ARG, "dims[%d]=%d must be positive", l, dims[l]);
        m.dims[l] = dims[l];
        m.max_width = dims[l] > m.max_width ? dims[l] : m.max_width;
    }
    for (int l = 0; l < n_layers; ++l) {
        if (act[l] < SSI_ACT_IDENTITY || act[l] > SSI_ACT_SIGMOID) return ssi_fail(ctx, SSI_ERR_ARG, "act[%d]=%d is not a supported activation", l, act[l]);
        m.act[l] = act[l];
        m.w_off[l] = off;
        off += (int64_t)dims[l] * dims[l + 1];
        m.b_off[l] = off;
        off += dims[l + 1];
        fl += 2.0 * (double)dims[l] * dims[l + 1];
    }
    m.n = off;
    m.flops_per_point = fl;
    const bool shape_changed = !ctx->has_model || m.n != ctx->model.n || m.dims[0] != ctx->model.dims[0] ||
                               m.dims[n_layers] != ctx->model.dims[ctx->model.L];
    ctx->model = m;
    ctx->has_model = true;
    if (shape_changed) { ctx->has_data = false; ctx->has_sub = false; }
    ssi_tc_invalidate(ctx); ssi_b1_invalidate(ctx); ssi_bm_invalidate(ctx);
    if (ctx->train) { cudaStreamSynchronize(ctx->stream); ssi_train_destroy(ctx); }      // its weights had the old model's layout
    return SSI_OK;
}

int ssi_set_data(ssi_ctx* ctx, const float* X, const float* Y, int64_t N) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_set_data");
    if (ctx->is_multi()) return ssi_multi_set_data(ctx, X, Y, N);
    if (!ctx->has_model) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_set_model must be called before ssi_set_data");
    if (!X || !Y || N < 1) return ssi_fail(ctx, SSI_ERR_ARG, "X, Y must be non-NULL and N >= 1");
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t bx = sizeof(float) * (size_t)ctx->model.dims[0] * N;
    const size_t by = sizeof(float) * (size_t)ctx->model.dims[ctx->model.L] * N;
    cudaFree(ctx->dX); cudaFree(ctx->dY);
    ctx->dX = ctx->dY = nullptr;
    ctx->has_data = false;
    SSI_CUDA(ctx, cudaMalloc(&ctx->dX, bx));
    SSI_CUDA(ctx, cudaMalloc(&ctx->dY, by));
    SSI_CUDA(ctx, cudaMemcpyAsync(ctx->dX, X, bx, cudaMemcpyHostToDevice, ctx->stream));
    SSI_CUDA(ctx, cudaMemcpyAsync(ctx->dY, Y, by, cudaMemcpyHostToDevice, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->N = N;
    ctx->has_data = true;
    ssi_tc_invalidate(ctx); ssi_b1_invalidate(ctx); ssi_bm_invalidate(ctx);
    return SSI_OK;
}

static int install_subspace(ssi_ctx* ctx, const float* W_swa, const float* P, int64_t n, int M, cudaMemcpyKind kind, bool keep_decoder = false) {
    if (!ctx->has_model) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_set_model must be called before the subspace is set");
    if (!keep_decoder) ssi_dec_destroy(ctx);            // a linear subspace replaces a decoder
    if (n != ctx->model.n) return ssi_fail(ctx, SSI_ERR_ARG, "n=%lld does not match the model's %lld parameters", (long long)n, (long long)ctx->model.n);
    if (M < 1 || M > SSI_MAX_M) return ssi_fail(ctx, SSI_ERR_ARG, "M=%d must be in [1,%d]", M, SSI_MAX_M);
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->dP); cudaFree(ctx->dSubGram);
    ctx->dP = nullptr; ctx->dSubGram = nullptr; ctx->dWswa = nullptr;
    ctx->has_sub = false;
    // [P | W_swa] as one n x (M+1) matrix so that the prior's M-space Gram is one pass
    SSI_CUDA(ctx, cudaMalloc(&ctx->dP, sizeof(float) * (size_t)n * (M + 1)));
    SSI_CUDA(ctx, cudaMalloc(&ctx->dSubGram, sizeof(double) * (size_t)(M + 1) * (M + 1)));
    ctx->dWswa = ctx->dP + (size_t)n * M;
    SSI_CUDA(ctx, cudaMemcpyAsync(ctx->dP, P, sizeof(float) * (size_t)n * M, kind, ctx->stream));
    SSI_CUDA(ctx, cudaMemcpyAsync(ctx->dWswa, W_swa, sizeof(float) * (size_t)n, kind, ctx->stream));
    ctx->M = M;
    ctx->Mz = M;
    SSI_TRY(ssi_subspace_gram(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->has_sub = true;
    ssi_tc_invalidate(ctx); ssi_b1_invalidate(ctx); ssi_bm_invalidate(ctx);
    return SSI_OK;
}

}  // extern "C"
int ssi_install_subspace_host(ssi_ctx* ctx, const float* W_swa, const float* P, int64_t n, int M) {
    return install_subspace(ctx, W_swa, P, n, M, cudaMemcpyHostToDevice, true);
}
extern "C" {

int ssi_set_decoder(ssi_ctx* ctx, const float* W_swa, int32_t n_layers, const int32_t* dims, const int32_t* act, const float* theta) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_set_decoder");
    if (ctx->is_multi()) return ssi_multi_set_decoder(ctx, W_swa, n_layers, dims, act, theta);
    return ssi_set_decoder_impl(ctx, W_swa, n_layers, dims, act, theta);
}

int ssi_set_subspace(ssi_ctx* ctx, const float* W_swa, const float* P, int64_t n, int32_t M) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_set_subspace");
    if (!W_swa || !P) return ssi_fail(ctx, SSI_ERR_ARG, "W_swa and P must be non-NULL");
    if (ctx->is_multi()) return ssi_multi_set_subspace(ctx, W_swa, P, n, M);
    return install_subspace(ctx, W_swa, P, n, M, cudaMemcpyHostToDevice);
}

int ssi_logpost_batch_dev(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p, double sigma_z,
                          uint32_t prior_mask, double* d_lp_out, double* d_terms_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_logpost_batch_dev");
    if (B < 0 || (B > 0 && (!dZ || !d_lp_out))) return ssi_fail(ctx, SSI_ERR_ARG, "Z and lp_out must be non-NULL, B >= 0");
    SSI_NO_MULTI(ctx, "device-pointer entry points");
    SSI_TRY(ssi_use_device(ctx));
    call_timer t(ctx);
    const int rc = ssi_logpost_device(ctx, dZ, B, sigma_m, sigma_p, sigma_z, prior_mask, d_lp_out, d_terms_out);
    t.stop(false);
    return rc;
}

int ssi_logpost_grad_batch_dev(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p, double sigma_z,
                               uint32_t prior_mask, double* d_lp_out, double* d_grad_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_logpost_grad_batch_dev");
    if (B < 0 || (B > 0 && (!dZ || !d_lp_out || !d_grad_out)))
        return ssi_fail(ctx, SSI_ERR_ARG, "Z, lp_out and grad_out must be non-NULL, B >= 0");
    SSI_NO_MULTI(ctx, "device-pointer entry points");
    SSI_TRY(ssi_use_device(ctx));
    call_timer t(ctx);
    const int rc = ssi_logpost_grad_device(ctx, dZ, B, sigma_m, sigma_p, sigma_z, prior_mask, d_lp_out, d_grad_out);
    t.stop(false);
    return rc;
}

int ssi_logpost_grad_batch(ssi_ctx* ctx, const float* Z, int64_t B, double sigma_m, double sigma_p, double sigma_z,
                           uint32_t prior_mask, double* lp_out, double* grad_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_logpost_grad_batch");
    if (B < 0 || (B > 0 && (!Z || !lp_out || !grad_out)))
        return ssi_fail(ctx, SSI_ERR_ARG, "Z, lp_out and grad_out must be non-NULL, B >= 0");
    if (ctx->is_multi()) return ssi_multi_logpost(ctx, 1, Z, B, sigma_m, sigma_p, sigma_z, prior_mask, lp_out, grad_out);
    if (!ctx->has_model || !ctx->has_data || !ctx->has_sub)
        return ssi_fail(ctx, SSI_ERR_STATE, "model, data and subspace must be set before evaluating the gradient");
    if (B == 0) return SSI_OK;
    SSI_TRY(ssi_use_device(ctx));
    const size_t bz = sizeof(float) * (size_t)ctx->Mz * B;
    SSI_TRY(ssi_reserve(ctx, ctx->bZ, bz));
    SSI_TRY(ssi_reserve(ctx, ctx->bLp, sizeof(double) * (size_t)B));
    SSI_TRY(ssi_reserve(ctx, ctx->bTerms, sizeof(double) * (size_t)ctx->Mz * B));
    SSI_CUDA(ctx, cudaMemcpyAsync(ctx->bZ.p, Z, bz, cudaMemcpyHostToDevice, ctx->stream));
    call_timer t(ctx);
    const int rc = ssi_logpost_grad_device(ctx, (const float*)ctx->bZ.p, B, sigma_m, sigma_p, sigma_z, prior_mask,
                                           (double*)ctx->bLp.p, (double*)ctx->bTerms.p);
    t.stop(false);
    if (rc != SSI_OK) return rc;
    SSI_CUDA(ctx, cudaMemcpyAsync(lp_out, ctx->bLp.p, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
    SSI_CUDA(ctx, cudaMemcpyAsync(grad_out, ctx->bTerms.p, sizeof(double) * (size_t)ctx->Mz * B, cudaMemcpyDeviceToHost, ctx->stream));
    return ssi_sync_internal(ctx);
}

int ssi_logpost_batch(ssi_ctx* ctx, const float* Z, int64_t B, double sigma_m, double sigma_p, double sigma_z,
                      uint32_t prior_mask, double* lp_out, double* terms_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_logpost_batch");
    if (B < 0 || (B > 0 && (!Z || !lp_out))) return ssi_fail(ctx, SSI_ERR_ARG, "Z and lp_out must be non-NULL, B >= 0");
    if (ctx->is_multi()) return ssi_multi_logpost(ctx, 0, Z, B, sigma_m, sigma_p, sigma_z, prior_mask, lp_out, terms_out);
    if (!ctx->has_model || !ctx->has_data || !ctx->has_sub)
        return ssi_fail(ctx, SSI_ERR_STATE, "model, data and subspace must be set before evaluating the log-posterior");
    if (B == 0) return SSI_OK;
    SSI_TRY(ssi_use_device(ctx));
    const size_t bz = sizeof(float) * (size_t)ctx->Mz * B;
    SSI_TRY(ssi_reserve(ctx, ctx->bZ, bz));
    SSI_TRY(ssi_reserve(ctx, ctx->bLp, sizeof(double) * (size_t)B));
    if (terms_out) SSI_TRY(ssi_reserve(ctx, ctx->bTerms, sizeof(double) * 3 * (size_t)B));
    SSI_CUDA(ctx, cudaMemcpyAsync(ctx->bZ.p, Z, bz, cudaMemcpyHostToDevice, ctx->stream));
    // second attempt only if the tensor path's FP16 planes overflowed (it then runs on BF16 planes)
    for (int attempt = 0; attempt < 2; ++attempt) {
        call_timer t(ctx);
        const int rc = ssi_logpost_device(ctx, (const float*)ctx->bZ.p, B, sigma_m, sigma_p, sigma_z, prior_mask,
                                          (double*)ctx->bLp.p, terms_out ? (double*)ctx->bTerms.p : nullptr);
        t.stop(false);
        if (rc != SSI_OK) return rc;
        SSI_CUDA(ctx, cudaMemcpyAsync(lp_out, ctx->bLp.p, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
        if (terms_out)
            SSI_CUDA(ctx, cudaMemcpyAsync(terms_out, ctx->bTerms.p, sizeof(double) * 3 * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
        SSI_TRY(ssi_sync_internal(ctx));
        bool exceeded = false;
        SSI_TRY(ssi_tc_range_exceeded(ctx, &exceeded));
        if (!exceeded) break;
    }
    return SSI_OK;
}

static const char* mh_name(int kind, bool dev) {
    static const char* names[2][3] = {{"ssi_mh_run", "ssi_mala_run", "ssi_hmc_run"}, {"ssi_mh_run_dev", "ssi_mala_run_dev", "ssi_hmc_run_dev"}};
    return names[dev ? 1 : 0][kind];
}

}  // extern "C"

// Host-pointer run of the chains [c0, c1) of `run` on this device (c0 == 0 and c1 == run.n_chains for a single-device
// context; a multi-device context hands every device its slice of the same host arrays).
int ssi_mh_run_host_slice(ssi_ctx* ctx, const ssi_mh_run_t& run, int64_t c0, int64_t c1) {
    SSI_NVTX(mh_name(run.kind, false));
    SSI_TRY(ssi_use_device(ctx));
    ssi_mh_run_t r = run;          // this device's shard, its pointers into bSnap
    r.n_chains = c1 - c0;
    r.chain_offset = run.chain_offset + c0;
    const int M = ctx->Mz;
    const size_t cs = (size_t)r.n_chains * (size_t)r.n_steps;
    const size_t bz = sizeof(float) * M * cs, bl = sizeof(double) * cs, ba = cs;
    // one scratch allocation: [z_trace | lp_trace | acc | step sizes | adaptation state | z0]
    const size_t off_l = run.z_trace ? (bz + 255) / 256 * 256 : 0;
    const size_t off_a = off_l + (run.lp_trace ? (bl + 255) / 256 * 256 : 0);
    const size_t off_e = off_a + (run.accept_trace ? (ba + 255) / 256 * 256 : 0);
    const size_t off_ad = off_e + (run.step_size_trace ? (bl + 255) / 256 * 256 : 0);
    const size_t bad = run.adapt0 ? sizeof(double) * 3 * (size_t)r.n_chains : 0;
    const size_t off_z0 = off_ad + (bad + 255) / 256 * 256;
    const size_t bz0 = run.z0 ? sizeof(float) * (size_t)M * r.n_chains : 0;
    SSI_TRY(ssi_reserve(ctx, ctx->bSnap, off_z0 + bz0 + 256));
    char* base = (char*)ctx->bSnap.p;
    r.z_trace = run.z_trace ? (float*)base : nullptr;
    r.lp_trace = run.lp_trace ? (double*)(base + off_l) : nullptr;
    r.accept_trace = run.accept_trace ? (uint8_t*)(base + off_a) : nullptr;
    r.step_size_trace = run.step_size_trace ? (double*)(base + off_e) : nullptr;
    if (run.adapt0) {
        double* dad = (double*)(base + off_ad);
        SSI_CUDA(ctx, cudaMemcpyAsync(dad, run.adapt0 + 3 * (size_t)c0, bad, cudaMemcpyHostToDevice, ctx->stream));
        r.adapt0 = dad;
    }
    if (run.z0) {
        float* dz0 = (float*)(base + off_z0);
        SSI_CUDA(ctx, cudaMemcpyAsync(dz0, run.z0 + (size_t)c0 * M, bz0, cudaMemcpyHostToDevice, ctx->stream));
        r.z0 = dz0;
    }
    for (int attempt = 0; attempt < 2; ++attempt) {      // repeated only if the tensor path's FP16 planes overflowed
        call_timer t(ctx);
        const int rc = ssi_mh_device(ctx, r);
        t.stop(false);
        if (rc != SSI_OK) return rc;
        SSI_TRY(ssi_sync_internal(ctx));
        bool exceeded = false;
        SSI_TRY(ssi_tc_range_exceeded(ctx, &exceeded));
        if (!exceeded) break;
    }
    // a step's row of the device trace is this device's chains; in the host trace rows are run.n_chains chains apart
    const int64_t ld = run.n_chains;
    const size_t rz = sizeof(float) * (size_t)M * r.n_chains, rl = sizeof(double) * (size_t)r.n_chains, ra = (size_t)r.n_chains;
    if (run.z_trace) SSI_CUDA(ctx, cudaMemcpy2DAsync(run.z_trace + (size_t)c0 * M, sizeof(float) * (size_t)M * ld, r.z_trace, rz, rz,
                                                     (size_t)r.n_steps, cudaMemcpyDeviceToHost, ctx->stream));
    if (run.lp_trace) SSI_CUDA(ctx, cudaMemcpy2DAsync(run.lp_trace + c0, sizeof(double) * (size_t)ld, r.lp_trace, rl, rl, (size_t)r.n_steps,
                                                      cudaMemcpyDeviceToHost, ctx->stream));
    if (run.accept_trace) SSI_CUDA(ctx, cudaMemcpy2DAsync(run.accept_trace + c0, (size_t)ld, r.accept_trace, ra, ra, (size_t)r.n_steps,
                                                          cudaMemcpyDeviceToHost, ctx->stream));
    if (run.step_size_trace) SSI_CUDA(ctx, cudaMemcpy2DAsync(run.step_size_trace + c0, sizeof(double) * (size_t)ld, r.step_size_trace, rl, rl,
                                                             (size_t)r.n_steps, cudaMemcpyDeviceToHost, ctx->stream));
    SSI_TRY(ssi_sync_internal(ctx));
    return ssi_mh_fetch_accepts(ctx);
}

// Every sampler entry point: one check of the whole run, before any allocation, copy or device dispatch, then the run on
// the device (dev: `r` holds device pointers) or sharded over the devices of the context.  kind_arg: the caller chose the
// kind (ssi_mh_run_from[_dev]).
static int mh_run(ssi_ctx* ctx, const ssi_mh_run_t& r, bool dev, bool kind_arg = false) {
    if (!ctx) return SSI_ERR_ARG;
    if (dev) SSI_NO_MULTI(ctx, "device-pointer entry points");
    if (kind_arg && r.kind != 0 && r.kind != 1) return ssi_fail(ctx, SSI_ERR_ARG, "kind must be 0 (RWMH) or 1 (MALA)");
    if (r.n_chains <= 0 || r.n_steps <= 0) return ssi_fail(ctx, SSI_ERR_ARG, "n_chains and n_steps must be positive");
    if (r.chain_offset < 0 || r.step_offset < 0 || r.chain_offset > 0xffffffffll - r.n_chains || r.step_offset > 0xffffffffll - r.n_steps)
        return ssi_fail(ctx, SSI_ERR_ARG, "chain ids and steps must fit 32 bits");
    if (r.step_offset > 0 && !r.z0) return ssi_fail(ctx, SSI_ERR_ARG, "a continued run (step_offset > 0) needs the chain state z");
    if (r.kind == 2) {
        SSI_TRY(ssi_hmc_check(ctx, r.hp, ctx->Mz));
        if (r.step_offset > 0 && r.hp->n_adapts > 0 && !r.adapt0)
            return ssi_fail(ctx, SSI_ERR_ARG, "a continued HMC run with n_adapts > 0 needs the adaptation state (ssi_hmc_get_adapt)");
    }
    if (!ctx->has_model || !ctx->has_data || !ctx->has_sub)
        return ssi_fail(ctx, SSI_ERR_STATE, "model, data and subspace must be set before sampling");
    if (!dev) return ctx->is_multi() ? ssi_multi_mh_run(ctx, r) : ssi_mh_run_host_slice(ctx, r, 0, r.n_chains);
    SSI_NVTX(mh_name(r.kind, true));
    SSI_TRY(ssi_use_device(ctx));
    call_timer t(ctx);
    const int rc = ssi_mh_device(ctx, r);
    t.stop(false);
    return rc;
}

extern "C" {

int ssi_mh_run(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
               double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask, const float* z0,
               float* z_trace, double* lp_trace, uint8_t* accept_trace) {
    return mh_run(ctx, {.kind = 0, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p, .mask = prior_mask, .z0 = z0,
                        .z_trace = z_trace, .lp_trace = lp_trace, .accept_trace = accept_trace}, false);
}
int ssi_mh_run_dev(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                   double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask, const float* d_z0,
                   float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace) {
    return mh_run(ctx, {.kind = 0, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p, .mask = prior_mask, .z0 = d_z0,
                        .z_trace = d_z_trace, .lp_trace = d_lp_trace, .accept_trace = d_accept_trace}, true);
}
int ssi_mala_run(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                 double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask, const float* z0,
                 float* z_trace, double* lp_trace, uint8_t* accept_trace) {
    return mh_run(ctx, {.kind = 1, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p, .mask = prior_mask, .z0 = z0,
                        .z_trace = z_trace, .lp_trace = lp_trace, .accept_trace = accept_trace}, false);
}
int ssi_mala_run_dev(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                     double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask, const float* d_z0,
                     float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace) {
    return mh_run(ctx, {.kind = 1, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p, .mask = prior_mask, .z0 = d_z0,
                        .z_trace = d_z_trace, .lp_trace = d_lp_trace, .accept_trace = d_accept_trace}, true);
}
int ssi_mh_run_from(ssi_ctx* ctx, int32_t kind, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset, int64_t step_offset,
                    double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask, const float* z_state,
                    float* z_trace, double* lp_trace, uint8_t* accept_trace) {
    return mh_run(ctx, {.kind = kind, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .step_offset = step_offset, .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p,
                        .mask = prior_mask, .z0 = z_state, .z_trace = z_trace, .lp_trace = lp_trace,
                        .accept_trace = accept_trace}, false, true);
}
int ssi_mh_run_from_dev(ssi_ctx* ctx, int32_t kind, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                        int64_t step_offset, double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                        const float* d_z_state, float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace) {
    return mh_run(ctx, {.kind = kind, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .step_offset = step_offset, .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p,
                        .mask = prior_mask, .z0 = d_z_state, .z_trace = d_z_trace, .lp_trace = d_lp_trace,
                        .accept_trace = d_accept_trace}, true, true);
}
int ssi_hmc_run(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset, int64_t step_offset,
                const ssi_hmc_params_t* hp, double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                const float* z_state, const double* adapt_state,
                float* z_trace, double* lp_trace, uint8_t* accept_trace, double* step_size_trace) {
    return mh_run(ctx, {.kind = 2, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .step_offset = step_offset, .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p,
                        .mask = prior_mask, .hp = hp, .z0 = z_state, .adapt0 = adapt_state, .z_trace = z_trace,
                        .lp_trace = lp_trace, .accept_trace = accept_trace, .step_size_trace = step_size_trace}, false);
}
int ssi_hmc_run_dev(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset, int64_t step_offset,
                    const ssi_hmc_params_t* hp, double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                    const float* d_z_state, const double* d_adapt_state,
                    float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace, double* d_step_size_trace) {
    return mh_run(ctx, {.kind = 2, .n_chains = n_chains, .n_steps = n_steps, .seed = seed, .chain_offset = chain_offset,
                        .step_offset = step_offset, .sigma_z = sigma_z, .sigma_m = sigma_m, .sigma_p = sigma_p,
                        .mask = prior_mask, .hp = hp, .z0 = d_z_state, .adapt0 = d_adapt_state, .z_trace = d_z_trace,
                        .lp_trace = d_lp_trace, .accept_trace = d_accept_trace, .step_size_trace = d_step_size_trace}, true);
}

}  // extern "C"

// final (z, lp) of the n chains of the last run on this device: what a caller saves to continue later with ssi_mh_run_from
int ssi_mh_get_state_slice(ssi_ctx* ctx, int64_t n, float* z_out, double* lp_out) {
    if (ctx->mh_chains != n) return ssi_fail(ctx, SSI_ERR_STATE, "no chains have been run on this context");
    SSI_TRY(ssi_use_device(ctx));
    if (z_out) SSI_CUDA(ctx, cudaMemcpyAsync(z_out, ctx->bMhZ.p, sizeof(float) * (size_t)ctx->Mz * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (lp_out) SSI_CUDA(ctx, cudaMemcpyAsync(lp_out, ctx->bMhLp.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSI_OK;
}
// dual-averaging state (3 x n) of the n chains of the last HMC run on this device
int ssi_hmc_get_adapt_slice(ssi_ctx* ctx, int64_t n, double* adapt_out) {
    if (ctx->mh_chains != n || ctx->mh_kind != 2) return ssi_fail(ctx, SSI_ERR_STATE, "the last run on this context was not HMC");
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaMemcpyAsync(adapt_out, ctx->bHmcAd.p, sizeof(double) * 3 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSI_OK;
}
extern "C" {

int ssi_mh_get_state(ssi_ctx* ctx, float* z_out, double* lp_out) {
    if (!ctx) return SSI_ERR_ARG;
    if (ctx->mh_chains <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "no chains have been run on this context");
    if (ctx->is_multi()) return ssi_multi_mh_get_state(ctx, z_out, lp_out);
    return ssi_mh_get_state_slice(ctx, ctx->mh_chains, z_out, lp_out);
}

int ssi_hmc_get_adapt(ssi_ctx* ctx, double* adapt_out) {
    if (!ctx) return SSI_ERR_ARG;
    if (!adapt_out) return ssi_fail(ctx, SSI_ERR_ARG, "adapt_out is NULL");
    if (ctx->mh_chains <= 0 || ctx->mh_kind != 2) return ssi_fail(ctx, SSI_ERR_STATE, "the last run on this context was not HMC");
    if (ctx->is_multi()) return ssi_multi_hmc_get_adapt(ctx, adapt_out);
    return ssi_hmc_get_adapt_slice(ctx, ctx->mh_chains, adapt_out);
}

int ssi_rng_replay(uint64_t seed, int64_t chain, int64_t step, int32_t M, float* eps_out, double* e_out) {
    if (M < 0 || chain < 0 || step < 0 || chain > 0xffffffffll || step > 0xffffffffll) return SSI_ERR_ARG;
    if (eps_out) {
        for (int blk = 0; blk * 4 < M; ++blk) {
            float e[4];
            ssi_normal4(seed, (uint32_t)chain, (uint32_t)step, (uint32_t)blk, e);
            for (int r = 0; r < 4 && blk * 4 + r < M; ++r) eps_out[blk * 4 + r] = e[r];
        }
    }
    if (e_out) *e_out = ssi_exp1(seed, (uint32_t)chain, (uint32_t)step);
    return SSI_OK;
}

int ssi_project(ssi_ctx* ctx, const float* Z, int64_t B, float* W_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_project");
    if (ctx->is_multi()) return ssi_multi_project(ctx, Z, B, W_out);
    if (!ctx->has_model || !ctx->has_sub) return ssi_fail(ctx, SSI_ERR_STATE, "model and subspace must be set");
    if (B < 0 || (B > 0 && (!Z || !W_out))) return ssi_fail(ctx, SSI_ERR_ARG, "Z and W_out must be non-NULL");
    if (B == 0) return SSI_OK;
    SSI_TRY(ssi_use_device(ctx));
    const int64_t n = ctx->model.n;
    // stream the samples through a bounded scratch
    const int64_t gmax = std::max<int64_t>(1, std::min<int64_t>(B, (int64_t)(1ull << 30) / (sizeof(float) * n)));
    SSI_TRY(ssi_reserve(ctx, ctx->bZ, sizeof(float) * (size_t)ctx->Mz * gmax));
    SSI_TRY(ssi_reserve(ctx, ctx->bW, sizeof(float) * (size_t)n * gmax));
    call_timer t(ctx);
    for (int64_t b0 = 0; b0 < B; b0 += gmax) {
        const int64_t g = std::min(gmax, B - b0);
        SSI_CUDA(ctx, cudaMemcpyAsync(ctx->bZ.p, Z + b0 * ctx->Mz, sizeof(float) * (size_t)ctx->Mz * g, cudaMemcpyHostToDevice, ctx->stream));
        const float* zin = (const float*)ctx->bZ.p;
        if (ctx->dec_active) SSI_TRY(ssi_dec_project(ctx, zin, g, &zin));       // W = W_swa + decoder(z)
        SSI_TRY(ssi_project_device(ctx, zin, g, (float*)ctx->bW.p));
        SSI_CUDA(ctx, cudaMemcpyAsync(W_out + b0 * n, ctx->bW.p, sizeof(float) * (size_t)n * g, cudaMemcpyDeviceToHost, ctx->stream));
        SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    t.stop(true);
    return SSI_OK;
}

// The sweep reduces over the samples (mean / std per grid point) and the construction streams hold one deviation matrix:
// on a multi-device context they run on its first device.
#define SSI_FIRST_DEVICE(ctx, call)                                                      \
    do {                                                                                 \
        if ((ctx)->is_multi()) {                                                         \
            ssi_ctx* parent__ = (ctx);                                                   \
            (ctx) = parent__->children[0];                                               \
            const int rc__ = (call);                                                     \
            if (rc__ < 0) parent__->err = (ctx)->err;                                    \
            return rc__;                                                                 \
        }                                                                                \
    } while (0)

int ssi_predict_batch(ssi_ctx* ctx, const float* Z, int64_t B, const float* Xg, int64_t Ng,
                      float* preds_out, double* mean_out, double* std_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_predict_batch");
    SSI_FIRST_DEVICE(ctx, ssi_predict_batch(ctx, Z, B, Xg, Ng, preds_out, mean_out, std_out));
    if (!ctx->has_model || !ctx->has_sub) return ssi_fail(ctx, SSI_ERR_STATE, "model and subspace must be set before predicting");
    if (B < 0 || Ng < 0) return ssi_fail(ctx, SSI_ERR_ARG, "B and Ng must be non-negative");
    if (B == 0 || Ng == 0) return SSI_OK;
    if (!Z || !Xg) return ssi_fail(ctx, SSI_ERR_ARG, "Z and Xg must be non-NULL");
    SSI_TRY(ssi_use_device(ctx));
    const ssi_model_t& m = ctx->model;
    const int O = m.dims[m.L], in0 = m.dims[0];
    const size_t ON = (size_t)O * Ng;
    // staging: Z | Xg | mean, m2, std (doubles) | preds (optional)
    SSI_TRY(ssi_reserve(ctx, ctx->bZ, sizeof(float) * (size_t)ctx->Mz * B));
    SSI_TRY(ssi_reserve(ctx, ctx->bLp, sizeof(float) * (size_t)in0 * Ng));
    SSI_TRY(ssi_reserve(ctx, ctx->bTerms, sizeof(double) * 3 * ON));
    if (preds_out) SSI_TRY(ssi_reserve(ctx, ctx->bMisc, sizeof(float) * ON * (size_t)B));
    float* dZ = (float*)ctx->bZ.p;
    float* dXg = (float*)ctx->bLp.p;
    double* d_mean = (double*)ctx->bTerms.p;
    double* d_m2 = d_mean + ON;
    double* d_std = d_m2 + ON;
    float* d_preds = preds_out ? (float*)ctx->bMisc.p : nullptr;
    SSI_CUDA(ctx, cudaMemcpyAsync(dZ, Z, sizeof(float) * (size_t)ctx->Mz * B, cudaMemcpyHostToDevice, ctx->stream));
    SSI_CUDA(ctx, cudaMemcpyAsync(dXg, Xg, sizeof(float) * (size_t)in0 * Ng, cudaMemcpyHostToDevice, ctx->stream));
    call_timer t(ctx);
    const int rc = ssi_predict_device(ctx, dZ, B, dXg, Ng, d_preds, d_mean, d_std, d_m2);
    t.stop(false);
    if (rc != SSI_OK) return rc;
    if (mean_out) SSI_CUDA(ctx, cudaMemcpyAsync(mean_out, d_mean, sizeof(double) * ON, cudaMemcpyDeviceToHost, ctx->stream));
    if (std_out) SSI_CUDA(ctx, cudaMemcpyAsync(std_out, d_std, sizeof(double) * ON, cudaMemcpyDeviceToHost, ctx->stream));
    if (preds_out) SSI_CUDA(ctx, cudaMemcpyAsync(preds_out, d_preds, sizeof(float) * ON * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
    return ssi_sync_internal(ctx);
}

int ssi_swa_begin(ssi_ctx* ctx, int64_t n, int64_t K_max) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_FIRST_DEVICE(ctx, ssi_swa_begin(ctx, n, K_max));
    if (n < 1 || K_max < 1) return ssi_fail(ctx, SSI_ERR_ARG, "n and K_max must be positive");
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->dSwaMean); cudaFree(ctx->dDev); cudaFree(ctx->dSwaAmax);
    ctx->dSwaMean = ctx->dDev = ctx->dSwaAmax = nullptr;
    ctx->swa_n = 0; ctx->swa_K = 0; ctx->swa_Kmax = 0; ctx->swa_ld = 0;
    SSI_CUDA(ctx, cudaMalloc(&ctx->dSwaMean, sizeof(float) * (size_t)n));
    const int64_t ld = (n + 31) / 32 * 32;
    SSI_CUDA(ctx, cudaMalloc(&ctx->dDev, sizeof(float) * (size_t)ld * K_max));
    SSI_CUDA(ctx, cudaMemsetAsync(ctx->dSwaMean, 0, sizeof(float) * (size_t)n, ctx->stream));   // W_swa = zeros (:31)
    SSI_CUDA(ctx, cudaMalloc(&ctx->dSwaAmax, sizeof(float)));
    SSI_CUDA(ctx, cudaMemsetAsync(ctx->dSwaAmax, 0, sizeof(float), ctx->stream));
    ctx->swa_n = n;
    ctx->swa_ld = ld;
    ctx->swa_Kmax = K_max;
    return SSI_OK;
}

int ssi_swa_push_dev(ssi_ctx* ctx, const float* dW, double n_scalar) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_swa_push_dev");
    SSI_NO_MULTI(ctx, "device-pointer entry points");
    if (!dW) return ssi_fail(ctx, SSI_ERR_ARG, "W must be non-NULL");
    SSI_TRY(ssi_use_device(ctx));
    call_timer t(ctx);
    const int rc = ssi_swa_push_device(ctx, dW, n_scalar);
    t.stop(false);
    return rc;
}

int ssi_swa_push(ssi_ctx* ctx, const float* W, double n_scalar) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_swa_push");
    SSI_FIRST_DEVICE(ctx, ssi_swa_push(ctx, W, n_scalar));
    if (!W) return ssi_fail(ctx, SSI_ERR_ARG, "W must be non-NULL");
    if (ctx->swa_n <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin has not been called");
    SSI_TRY(ssi_use_device(ctx));
    SSI_TRY(ssi_reserve(ctx, ctx->bSnap, sizeof(float) * (size_t)ctx->swa_n));
    SSI_CUDA(ctx, cudaMemcpyAsync(ctx->bSnap.p, W, sizeof(float) * (size_t)ctx->swa_n, cudaMemcpyHostToDevice, ctx->stream));
    call_timer t(ctx);
    const int rc = ssi_swa_push_device(ctx, (const float*)ctx->bSnap.p, n_scalar);
    t.stop(false);
    if (rc != SSI_OK) return rc;
    return ssi_sync_internal(ctx);   // the caller may reuse W immediately
}

int ssi_swa_deviations(ssi_ctx* ctx, float* A_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_FIRST_DEVICE(ctx, ssi_swa_deviations(ctx, A_out));
    if (ctx->swa_n <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin has not been called");
    if (!A_out) return ssi_fail(ctx, SSI_ERR_ARG, "A_out must be non-NULL");
    SSI_TRY(ssi_use_device(ctx));
    if (ctx->swa_K > 0)       // device columns are swa_ld apart (padded to 128 bytes), the caller's n apart
        SSI_CUDA(ctx, cudaMemcpy2DAsync(A_out, sizeof(float) * (size_t)ctx->swa_n, ctx->dDev, sizeof(float) * (size_t)ctx->swa_ld,
                                        sizeof(float) * (size_t)ctx->swa_n, (size_t)ctx->swa_K, cudaMemcpyDeviceToHost, ctx->stream));
    return ssi_sync_internal(ctx);
}

int ssi_swa_mean(ssi_ctx* ctx, float* W_swa_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_FIRST_DEVICE(ctx, ssi_swa_mean(ctx, W_swa_out));
    if (ctx->swa_n <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin has not been called");
    if (!W_swa_out) return ssi_fail(ctx, SSI_ERR_ARG, "W_swa_out must be non-NULL");
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaMemcpyAsync(W_swa_out, ctx->dSwaMean, sizeof(float) * (size_t)ctx->swa_n, cudaMemcpyDeviceToHost, ctx->stream));
    return ssi_sync_internal(ctx);
}

int64_t ssi_swa_columns(const ssi_ctx* ctx) { return ctx ? (ctx->is_multi() ? ctx->children[0]->swa_K : ctx->swa_K) : -1; }

// ---- on-device training step (the step before the path) ---------------------------------
int ssi_train_begin(ssi_ctx* ctx, const float* W0, int32_t optimiser, double eta, double beta1, double beta2) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_FIRST_DEVICE(ctx, ssi_train_begin(ctx, W0, optimiser, eta, beta1, beta2));
    if (!W0) return ssi_fail(ctx, SSI_ERR_ARG, "W0 must be non-NULL");
    SSI_TRY(ssi_use_device(ctx));
    return ssi_train_begin_impl(ctx, W0, optimiser, eta, beta1, beta2);
}

int ssi_train_step(ssi_ctx* ctx, const int64_t* idx, int64_t j0, int64_t nb, double* loss_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_train_step");
    SSI_FIRST_DEVICE(ctx, ssi_train_step(ctx, idx, j0, nb, loss_out));
    SSI_TRY(ssi_use_device(ctx));
    call_timer t(ctx);
    const int rc = ssi_train_step_impl(ctx, idx, j0, nb, loss_out);
    t.stop(false);
    return rc;
}

int ssi_train_snapshot(ssi_ctx* ctx, double n_scalar) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_FIRST_DEVICE(ctx, ssi_train_snapshot(ctx, n_scalar));
    const float* dW = ssi_train_weights_device(ctx);
    if (!dW) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_train_begin has not been called");
    if (ctx->swa_n != ctx->model.n) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin(n = %lld parameters) must precede ssi_train_snapshot", (long long)ctx->model.n);
    SSI_TRY(ssi_use_device(ctx));
    call_timer t(ctx);
    const int rc = ssi_swa_push_device(ctx, dW, n_scalar);
    t.stop(false);
    return rc;
}

int ssi_train_get_weights(ssi_ctx* ctx, float* W_out) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_FIRST_DEVICE(ctx, ssi_train_get_weights(ctx, W_out));
    const float* dW = ssi_train_weights_device(ctx);
    if (!dW) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_train_begin has not been called");
    if (!W_out) return ssi_fail(ctx, SSI_ERR_ARG, "W_out must be non-NULL");
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaMemcpyAsync(W_out, dW, sizeof(float) * (size_t)ctx->model.n, cudaMemcpyDeviceToHost, ctx->stream));
    return ssi_sync_internal(ctx);
}

int ssi_train_end(ssi_ctx* ctx) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_FIRST_DEVICE(ctx, ssi_train_end(ctx));
    SSI_TRY(ssi_use_device(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ssi_train_destroy(ctx);
    return SSI_OK;
}

// copies the results of a factorisation to the host and optionally installs them as the context's subspace
static int swa_deliver(ssi_ctx* ctx, int M, float* dPout, double* ds, int sweeps_dummy, float* W_swa_out, float* P_out, double* s_out,
                       int* sweeps, int32_t install) {
    (void)sweeps_dummy;
    const int64_t n = ctx->swa_n;
    const int K = (int)ctx->swa_K;
    if (W_swa_out) SSI_CUDA(ctx, cudaMemcpyAsync(W_swa_out, ctx->dSwaMean, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (P_out) SSI_CUDA(ctx, cudaMemcpyAsync(P_out, dPout, sizeof(float) * (size_t)n * M, cudaMemcpyDeviceToHost, ctx->stream));
    if (s_out) SSI_CUDA(ctx, cudaMemcpyAsync(s_out, ds, sizeof(double) * (size_t)K, cudaMemcpyDeviceToHost, ctx->stream));
    SSI_TRY(ssi_sync_internal(ctx));
    ctx->stats.jacobi_sweeps = *sweeps;
    if (*sweeps > 60) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "Jacobi eigen-solver did not converge in 60 sweeps");
    if (install) {
        if (!ctx->has_model || ctx->model.n != n)
            return ssi_fail(ctx, SSI_ERR_STATE, "install requested but the model (n=%lld) does not match the snapshots (n=%lld)",
                            (long long)(ctx->has_model ? ctx->model.n : 0), (long long)n);
        return install_subspace(ctx, ctx->dSwaMean, dPout, n, M, cudaMemcpyDeviceToDevice);
    }
    return SSI_OK;
}

static int swa_scratch(ssi_ctx* ctx, int M, float** dPout, double** ds) {
    const int64_t n = ctx->swa_n;
    const int K = (int)ctx->swa_K;
    // scratch: P (n x M floats) | s (K doubles)
    const size_t off_s = (sizeof(float) * (size_t)n * M + 255) / 256 * 256;
    SSI_TRY(ssi_reserve(ctx, ctx->bW, off_s + sizeof(double) * (size_t)(K > 0 ? K : 1)));
    *dPout = (float*)ctx->bW.p;
    *ds = (double*)((char*)ctx->bW.p + off_s);
    return SSI_OK;
}

int ssi_swa_finish(ssi_ctx* ctx, int32_t M, float* W_swa_out, float* P_out, double* s_out, int32_t install) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_swa_finish");
    if (ctx->is_multi()) return ssi_multi_swa_finish(ctx, M, W_swa_out, P_out, s_out, install);
    if (ctx->swa_n <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin has not been called");
    if (M < 1) return ssi_fail(ctx, SSI_ERR_ARG, "M must be positive");
    SSI_TRY(ssi_use_device(ctx));
    float* dPout;
    double* ds;
    SSI_TRY(swa_scratch(ctx, M, &dPout, &ds));
    int sweeps = 0;
    call_timer t(ctx);
    const int rc = ssi_swa_factor_device(ctx, M, dPout, ds, &sweeps);
    t.stop(false);
    if (rc != SSI_OK) return rc;
    return swa_deliver(ctx, M, dPout, ds, 0, W_swa_out, P_out, s_out, &sweeps, install);
}

int ssi_swa_gram_dev(ssi_ctx* ctx, double* dG_out, int32_t exact) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_swa_gram_dev");
    SSI_NO_MULTI(ctx, "device-pointer entry points");
    if (ctx->swa_n <= 0 || ctx->swa_K <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "no snapshots have been pushed");
    if (!dG_out) return ssi_fail(ctx, SSI_ERR_ARG, "G_out must be a device pointer to K x K doubles");
    SSI_TRY(ssi_use_device(ctx));
    call_timer t(ctx);
    bool tensor = false;
    const int rc = ssi_swa_gram_stage(ctx, exact != 0 || ctx->opt_gram_fp64 > 0, dG_out, &tensor);
    t.stop(false);
    ctx->stats.gram_path = tensor ? 2 : 1;
    return rc;
}

int ssi_swa_finish_gram(ssi_ctx* ctx, int32_t M, const double* dG, int32_t gram_exact, float* W_swa_out, float* P_out,
                        double* s_out, int32_t install) {
    if (!ctx) return SSI_ERR_ARG;
    SSI_NVTX("ssi_swa_finish_gram");
    SSI_NO_MULTI(ctx, "device-pointer entry points");
    if (ctx->swa_n <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin has not been called");
    if (M < 1) return ssi_fail(ctx, SSI_ERR_ARG, "M must be positive");
    if (!dG) return ssi_fail(ctx, SSI_ERR_ARG, "G must be a device pointer to the (all-reduced) K x K Gram");
    if (ctx->swa_K < M) return ssi_fail(ctx, SSI_ERR_RANK, "deviation matrix has %lld columns, cannot take M=%d", (long long)ctx->swa_K, M);
    if (M > SSI_MAX_M) return ssi_fail(ctx, SSI_ERR_ARG, "M=%d exceeds the supported maximum %d", M, SSI_MAX_M);
    SSI_TRY(ssi_use_device(ctx));
    float* dPout;
    double* ds;
    SSI_TRY(swa_scratch(ctx, M, &dPout, &ds));
    int sweeps = 0;
    call_timer t(ctx);
    bool need_exact = false;
    int rc = ssi_swa_eigen_stage(ctx, M, dG, gram_exact == 0, &need_exact);
    if (rc != SSI_OK) return rc;
    if (need_exact) { t.stop(false); return SSI_RETRY_EXACT; }      // same spectrum on every rank: every rank retries
    rc = ssi_swa_p_stage(ctx, M, dPout, ds, &sweeps);
    t.stop(false);
    if (rc != SSI_OK) return rc;
    if (gram_exact) ctx->stats.gram_path = 3;
    return swa_deliver(ctx, M, dPout, ds, 0, W_swa_out, P_out, s_out, &sweeps, install);
}

}  // extern "C"
