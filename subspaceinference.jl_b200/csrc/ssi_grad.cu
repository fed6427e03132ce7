// ssi_grad.cu — value and gradient of the subspace log-posterior, batched over B subspace points.
//
// Replaces the reference's gradient closure  l_pi_grad(theta) = (density(theta), backend.gradient(density, theta))
// (src/space_inference.jl:107; backends src/libs.jl:23-34: ForwardDiff by default, i.e. M dual-number forward passes
// per gradient) that feeds the :mala, :hmc and :nuts samplers (:117-120, :139-160).  Here one reverse pass per sample:
//
//     W = W_swa + P z                      k_project                                  (K1)
//     H_l = act_l(W_l H_{l-1} + b_l)       all activations kept                       ssi_reverse_pass (ssi_gemm.cu)
//     delta_L = -(pred - y)/sigma_m^2 * act_L'(pred)        (+ the squared error for lp)
//     gW_l = delta_l H_{l-1}',  gb_l = rowsum(delta_l),  delta_{l-1} = (W_l' delta_l) * act_{l-1}'(H_{l-1})
//     grad_z = P' [gW ; gb]  (+ prior terms evaluated in M-space)
//
// Every contraction goes through ssi_launch_gemm (skinny, tensor-core or SIMT kernel by shape); reductions are two-stage
// with a fixed order, so a sample's gradient does not depend on the rest of the batch.  FP32 storage, FP64 final
// accumulation of the squared error.  Any Dense chain.
#include "ssi_common.cuh"
#include "ssi_gemm.cuh"

#include <algorithm>
#include <cmath>


// grad_z(m, g) = sum_s part[s][m + g*M]  (+ prior terms), fixed order
__global__ void k_grad_finish(const float* __restrict__ part, int S, int M, int G, long long slab, const float* __restrict__ Z,
                              const double* __restrict__ Gsub /* (M+1)x(M+1) */, double inv_sp2, double inv_sz2, uint32_t mask,
                              double* __restrict__ grad /* M x G */) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= M * G) return;
    const int m = e % M, g = e / M;
    double v = 0.0;
    if (mask & SSI_TERM_LL)
        for (int s = 0; s < S; ++s) v += (double)part[(long long)s * slab + e];
    if (mask & SSI_TERM_PRIOR_W) {          // -(P'W_swa + P'P z)/sigma_p^2
        const int ld = M + 1;
        double w = Gsub[m * ld + M];
        for (int k = 0; k < M; ++k) w += Gsub[m * ld + k] * (double)Z[k + g * M];
        v -= w * inv_sp2;
    }
    if (mask & SSI_TERM_PRIOR_Z) v -= (double)Z[m + g * M] * inv_sz2;
    grad[e] = v;
}

int ssi_reduce_partials(ssi_ctx* ctx, const double* partials, int64_t B, int parts, double* d_out);
int ssi_logpost_finalize(ssi_ctx* ctx, const double* d_sse, const float* dZ, int64_t B, double sigma_m, double sigma_p,
                         double sigma_z, uint32_t mask, double* d_lp, double* d_terms);

int ssi_logpost_grad_device(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p, double sigma_z,
                            uint32_t mask, double* d_lp, double* d_grad) {
    if (!ctx->has_model || !ctx->has_data || !ctx->has_sub)
        return ssi_fail(ctx, SSI_ERR_STATE, "model, data and subspace must be set before evaluating the gradient");
    if (B <= 0) return SSI_OK;
    if (ctx->dec_active) return ssi_dec_logpost_grad(ctx, dZ, B, sigma_m, sigma_p, sigma_z, mask, d_lp, d_grad);
    if (!(sigma_m > 0) || !(sigma_p > 0) || !(sigma_z > 0))
        return ssi_fail(ctx, SSI_ERR_ARG, "sigma_m, sigma_p, sigma_z must be positive");
    if ((mask & ~(SSI_TERM_LL | SSI_TERM_PRIOR_W | SSI_TERM_PRIOR_Z)) || mask == 0)
        return ssi_fail(ctx, SSI_ERR_ARG, "prior_mask must be a non-empty OR of SSI_TERM_*");
    const ssi_model_t& m = ctx->model;
    const int64_t N = ctx->N, n = m.n;
    const int M = ctx->M;
    if (N >= (1ll << 31) || n >= (1ll << 31)) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "gradient path: N and n must fit 31 bits");

    // one hidden layer, scalar output: forward-mode tangents in registers next to the BASIS forward pass (ssi_basis.cu)
    if (ssi_b1_grad_supported(ctx) && (ctx->opt_path == SSI_PATH_AUTO || ctx->opt_path == SSI_PATH_BASIS)) {
        SSI_TRY(ssi_reserve(ctx, ctx->bMisc, sizeof(double) * (size_t)B));
        double* d_sse1 = (double*)ctx->bMisc.p;
        float* gpart1 = nullptr;
        int S1 = 0;
        SSI_TRY(ssi_b1_grad_sse(ctx, dZ, B, (mask & SSI_TERM_LL) ? 1.0 / (sigma_m * sigma_m) : 0.0, d_sse1, &gpart1, &S1));
        const int per = 32768 / M;                      // k_grad_finish indexes M x G with ints
        for (int64_t b0 = 0; b0 < B; b0 += per) {
            const int g = (int)std::min<int64_t>(per, B - b0);
            k_grad_finish<<<(M * g + 127) / 128, 128, 0, ctx->stream>>>(gpart1 + b0 * M, S1, M, g, (long long)M * B, dZ + b0 * M,
                                                                      ctx->dSubGram, 1.0 / (sigma_p * sigma_p),
                                                                      1.0 / (sigma_z * sigma_z), mask, d_grad + b0 * M);
            SSI_LAUNCH_CHECK(ctx);
        }
        SSI_TRY(ssi_logpost_finalize(ctx, d_sse1, dZ, B, sigma_m, sigma_p, sigma_z, mask, d_lp, nullptr));
        ctx->stats.last_path = SSI_PATH_BASIS;
        ctx->stats.last_units = (double)B * (double)N;
        ctx->stats.last_flops = 3.0 * (double)B * ((double)N * m.flops_per_point) + 4.0 * (double)B * (double)n * M;
        ctx->stats.last_bytes = 0;
        return SSI_OK;
    }

    // per-sample scratch: weights n, gradient n, activations sum(out_l) x N, two delta buffers maxw x N
    int maxw = 0;
    // sample strides are padded to 16 bytes so that the tensor-core GEMM (TMA) can address every sample's slice
    const long long act_elems = (ssi_act_offsets(m, N, nullptr, &maxw) + 3) & ~3ll;
    const long long np = (n + 3) & ~3ll;
    const long long d_sb = ((long long)maxw * N + 3) & ~3ll;
    const double per_sample = 4.0 * (2.0 * np + (double)act_elems + 2.0 * maxw * (double)N);
    // samples per group: the tensor-core GEMMs want many tiles per launch (the weight gradient of a 1024 x 1024 layer is only
    // 32 tiles per sample against 148 SMs), so take what a third of the free memory holds, 64 samples at most
    double budget = 6e9;
    if (ctx->opt_grad_group_gb > 0) budget = ctx->opt_grad_group_gb * 1e9;
    else {
        size_t mem_free = 0, mem_total = 0;
        if (cudaMemGetInfo(&mem_free, &mem_total) == cudaSuccess) {
            const double held = (double)ctx->bW.cap + (double)ctx->bGradW.cap + (double)ctx->bH0.cap + (double)ctx->bH1.cap;
            budget = std::max(budget, ((double)mem_free + held) / 3.0);
        }
    }
    int G = (int)std::max(1.0, std::min(64.0, budget / per_sample));
    G = (int)std::min<int64_t>(G, B);
    const long long split = 4096;                       // rows of P per partial of the final projection
    const int S = (int)((n + split - 1) / split);
    const int n_chunks = (int)((N + 255) / 256);
    SSI_TRY(ssi_reserve(ctx, ctx->bW, sizeof(float) * (size_t)np * G));
    SSI_TRY(ssi_reserve(ctx, ctx->bGradW, sizeof(float) * (size_t)np * G));
    SSI_TRY(ssi_reserve(ctx, ctx->bH0, sizeof(float) * (size_t)act_elems * G));
    SSI_TRY(ssi_reserve(ctx, ctx->bH1, sizeof(float) * (size_t)2 * d_sb * G));
    SSI_TRY(ssi_reserve(ctx, ctx->bPartials, sizeof(double) * (size_t)B * n_chunks));
    SSI_TRY(ssi_reserve(ctx, ctx->bGradP, sizeof(float) * (size_t)S * M * G));
    SSI_TRY(ssi_reserve(ctx, ctx->bMisc, sizeof(double) * (size_t)B));
    float* dW = (float*)ctx->bW.p;
    float* gW = (float*)ctx->bGradW.p;
    float* H = (float*)ctx->bH0.p;                      // [g][act_elems]
    float* D[2] = {(float*)ctx->bH1.p, (float*)ctx->bH1.p + (size_t)d_sb * G};   // [g][d_sb] each
    double* partials = (double*)ctx->bPartials.p;
    float* gpart = (float*)ctx->bGradP.p;
    double* d_sse = (double*)ctx->bMisc.p;
    const float coef = (mask & SSI_TERM_LL) ? (float)(1.0 / (sigma_m * sigma_m)) : 0.0f;

    for (int64_t b0 = 0; b0 < B; b0 += G) {
        const int g = (int)std::min<int64_t>(G, B - b0);
        SSI_TRY(ssi_project_device(ctx, dZ + b0 * M, g, dW, np));
        SSI_TRY(ssi_reverse_pass(ctx, g, N, dW, gW, np, ctx->dX, ctx->dY, H, act_elems, D, d_sb, coef, partials + b0 * n_chunks));
        // ---- grad_z = P' gW, split over rows of P, then fixed-order sum (+ priors) ----
        {
            gemm_t q{};
            q.A = ctx->dP; q.a_so = n; q.a_sk = 1; q.a_sb = 0;
            q.B = gW; q.b_sk = 1; q.b_sj = np; q.b_sb = 0;
            q.C = gpart; q.c_so = 1; q.c_sj = M; q.c_sb = (long long)M * g;
            q.O = M; q.J = g; q.K = n; q.split = split; q.epi = 0;
            SSI_TRY(ssi_launch_gemm(ctx, q, S, true, false));
            k_grad_finish<<<(M * g + 127) / 128, 128, 0, ctx->stream>>>(gpart, S, M, g, (long long)M * g, dZ + b0 * M, ctx->dSubGram,
                                                                      1.0 / (sigma_p * sigma_p), 1.0 / (sigma_z * sigma_z), mask,
                                                                      d_grad + b0 * M);
            SSI_LAUNCH_CHECK(ctx);
        }
    }
    SSI_TRY(ssi_reduce_partials(ctx, partials, B, n_chunks, d_sse));
    SSI_TRY(ssi_logpost_finalize(ctx, d_sse, dZ, B, sigma_m, sigma_p, sigma_z, mask, d_lp, nullptr));
    ctx->stats.last_path = SSI_PATH_LAYERED;
    ctx->stats.last_units = (double)B * (double)N;
    ctx->stats.last_flops = 3.0 * (double)B * ((double)N * m.flops_per_point) + 4.0 * (double)B * (double)n * M;
    ctx->stats.last_bytes = 0;
    return SSI_OK;
}
