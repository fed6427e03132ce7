// ssi_mh.cu — random-walk Metropolis-Hastings kept on the device over many chains.
//
// Replaces `sample(DensityModel(density), RWMH(MvNormal(zeros(M), sigma_z)), itr)`
// (src/space_inference.jl:111-116; AdvancedMH 0.6.2 semantics):
//   * sample 0 is a draw from the proposal and counts as the first of n_steps;
//   * step t proposes z' = z + sigma_z * eps_t and accepts iff  -e_t < lp(z') - lp(z)
//     with e_t ~ Exp(1)  (AdvancedMH tests `-randexp(rng) < log_alpha`);
//   * the log-density of the current state is cached, one evaluation per step.
// The reference runs ONE chain sequentially; here every step evaluates all chains'
// proposals in one batched log-posterior call.  No host round-trip inside the loop.
#include "ssi_common.cuh"
#include "ssi_rng.cuh"

#include <algorithm>

// zp[m,c] = z[m,c] + sigma_z * eps(chain_off + c, step, m); with init: z = 0.
// With a gradient (MALA): zp = (z + float(sigma_z^2/2 * grad)) + sigma_z * eps.
__global__ void __launch_bounds__(256)
k_mh_propose(const float* __restrict__ z, float* __restrict__ zp, long long n_chains, int M, unsigned long long seed,
             long long chain_off, unsigned step, float sigma_z, int init, const double* __restrict__ grad, double half_s2) {
    // one thread per (chain, block of 4 normals)
    const int nblk = (M + 3) >> 2;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_chains * nblk) return;
    const long long c = t / nblk;
    const int blk = (int)(t % nblk);
    float e[4];
    ssi_normal4(seed, (uint32_t)(chain_off + c), step, (uint32_t)blk, e);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int m = blk * 4 + r;
        if (m < M) {
            float base = init ? 0.0f : z[m + c * M];
            if (grad && !init) base = __fadd_rn(base, (float)(half_s2 * grad[m + c * M]));
            zp[m + c * M] = __fmaf_rn(sigma_z, e[r], base);
        }
    }
}

// accept/reject + trace write for step `step`.
__global__ void __launch_bounds__(256)
k_mh_accept(float* __restrict__ z, const float* __restrict__ zp, double* __restrict__ lp, const double* __restrict__ lpp,
            long long n_chains, int M, unsigned long long seed, long long chain_off, unsigned step, int force,
            float* __restrict__ z_trace, double* __restrict__ lp_trace, unsigned char* __restrict__ acc_trace,
            unsigned long long* __restrict__ n_acc,
            double* __restrict__ g, const double* __restrict__ gp, double half_s2, double inv2s2, int mala_rule) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned accepted = 0;
    if (c < n_chains) {
        bool acc;
        if (force) {
            acc = true;
        } else {
            const double e = ssi_exp1(seed, (uint32_t)(chain_off + c), step);
            double log_alpha = lpp[c] - lp[c];
            if (g) {
                // MALA: + log q(z | z') - log q(z' | z),  q(a | b) = N(a; b + (sigma^2/2) grad(b), sigma^2 I)
                double fwd = 0.0, rev = 0.0;
                for (int m = 0; m < M; ++m) {
                    const double a = (double)z[m + c * M], b = (double)zp[m + c * M];
                    // rule 0: q(z'|z) = N(z'; z + (s^2/2) grad(z), s^2), q(z|z') likewise.  rule 1: the densities as AdvancedMH's
                    // step is remembered to evaluate them, logpdf(proposal(-grad(x)), x - x') -- the drift enters negated and the
                    // roles of the two gradients are swapped
                    const double df = mala_rule ? (b - a + half_s2 * g[m + c * M]) : (b - a - half_s2 * g[m + c * M]);
                    const double dr = mala_rule ? (a - b + half_s2 * gp[m + c * M]) : (a - b - half_s2 * gp[m + c * M]);
                    fwd += df * df;
                    rev += dr * dr;
                }
                log_alpha += (fwd - rev) * inv2s2;
            }
            acc = (-e < log_alpha);          // NaN proposal density -> reject
        }
        if (acc) {
            lp[c] = lpp[c];
            for (int m = 0; m < M; ++m) z[m + c * M] = zp[m + c * M];
            if (g) for (int m = 0; m < M; ++m) g[m + c * M] = gp[m + c * M];
        }
        if (z_trace) {            // the trace pointers address this step's row
            float* dst = z_trace + c * M;
            for (int m = 0; m < M; ++m) dst[m] = z[m + c * M];
        }
        if (lp_trace) lp_trace[c] = lp[c];
        if (acc_trace) acc_trace[c] = acc ? 1 : 0;
        accepted = (acc && !force) ? 1u : 0u;
    }
    const unsigned warp_cnt = __popc(__ballot_sync(0xffffffffu, accepted));
    if ((threadIdx.x & 31) == 0 && warp_cnt) atomicAdd(n_acc, (unsigned long long)warp_cnt);
}

// kind 0: RWMH (src/space_inference.jl:113-116).  kind 1: MALA (:117-120,
//   `MALA(x -> MvNormal((sigma_z^2 / 2) .* x, sigma_z))`, init_params = rand(MvNormal(zeros(M), sigma_z))): the proposal is
//   z' = z + (sigma_z^2/2) grad lp(z) + sigma_z eps, accepted iff -e < lp' - lp + log q(z|z') - log q(z'|z); value and
//   gradient of every chain's proposal come from one batched reverse pass (ssi_logpost_grad_device) per step.
// step0 > 0 continues chains (SURVEY 5, checkpoint / resume): d_z0 is then the state after step step0 - 1, its
// log-density (and gradient) is re-evaluated -- the evaluation is deterministic and batch-invariant, so the continued run
// is bit-identical to an uninterrupted one -- and steps step0 .. step0 + S - 1 draw from the Philox counters of those
// steps; trace row t - step0 receives step t.
// kind 2: fixed-length HMC with per-chain dual averaging (ssi_hmc.cu, parameters hp): sample 0 and the re-established state
//   of a continued run are MALA's (value and gradient cached per chain); every later step is one HMC transition.  d_adapt0
//   (3 x C, device) is the adaptation state after step step0 - 1 (NULL: the initial one, allowed for step0 > 0 only when
//   hp->n_adapts == 0); d_etr receives the step size of every transition (NaN for step 0).
int ssi_mh_device(ssi_ctx* ctx, int kind, int64_t C, int64_t S, uint64_t seed, int64_t chain_off, int64_t step0,
                  double sigma_z, double sigma_m, double sigma_p, uint32_t mask,
                  const float* d_z0, float* d_ztr, double* d_lptr, uint8_t* d_acctr,
                  const ssi_hmc_params_t* hp, const double* d_adapt0, double* d_etr) {
    if (!ctx->has_model || !ctx->has_data || !ctx->has_sub)
        return ssi_fail(ctx, SSI_ERR_STATE, "model, data and subspace must be set before sampling");
    if (C <= 0 || S <= 0) return ssi_fail(ctx, SSI_ERR_ARG, "n_chains and n_steps must be positive");
    if (step0 < 0 || (step0 > 0 && !d_z0)) return ssi_fail(ctx, SSI_ERR_ARG, "a continued run (step_offset > 0) needs the chain state z");
    if (chain_off < 0 || chain_off + C > 0xffffffffll || step0 + S > 0xffffffffll)
        return ssi_fail(ctx, SSI_ERR_ARG, "chain ids and steps must fit 32 bits");
    const int M = ctx->Mz;         // the sampler works in the caller's z (a decoder maps it inside the density)
    if (kind == 2) {
        SSI_TRY(ssi_hmc_check(ctx, hp, M));
        if (step0 > 0 && hp->n_adapts > 0 && !d_adapt0)
            return ssi_fail(ctx, SSI_ERR_ARG, "a continued HMC run with n_adapts > 0 needs the adaptation state (ssi_hmc_get_adapt)");
    }
    SSI_TRY(ssi_reserve(ctx, ctx->bMhZ, sizeof(float) * (size_t)M * C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhZp, sizeof(float) * (size_t)M * C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhLp, sizeof(double) * (size_t)C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhLpP, sizeof(double) * (size_t)C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhCnt, sizeof(unsigned long long)));
    double *g = nullptr, *gp = nullptr;
    if (kind != 0) {
        SSI_TRY(ssi_reserve(ctx, ctx->bMhG, sizeof(double) * 2 * (size_t)M * C));
        g = (double*)ctx->bMhG.p;
        gp = g + (size_t)M * C;
    }
    const double half_s2 = 0.5 * sigma_z * sigma_z, inv2s2 = 1.0 / (2.0 * sigma_z * sigma_z);
    float* z = (float*)ctx->bMhZ.p;
    float* zp = (float*)ctx->bMhZp.p;
    double* lp = (double*)ctx->bMhLp.p;
    double* lpp = (double*)ctx->bMhLpP.p;
    unsigned long long* cnt = (unsigned long long*)ctx->bMhCnt.p;
    SSI_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), ctx->stream));
    if (kind == 2) SSI_TRY(ssi_hmc_prepare(ctx, C, hp, d_adapt0));

    const int nblk = (M + 3) / 4;
    const unsigned g_prop = (unsigned)((C * nblk + 255) / 256);
    const unsigned g_acc = (unsigned)((C + 255) / 256);
    double units = 0, flops = 0;

    if (step0 > 0) {
        // re-establish (z, lp[, grad]) of the saved state: evaluate it as a proposal and force-accept it without a trace row
        SSI_CUDA(ctx, cudaMemcpyAsync(zp, d_z0, sizeof(float) * (size_t)M * C, cudaMemcpyDeviceToDevice, ctx->stream));
        if (kind != 0) SSI_TRY(ssi_logpost_grad_device(ctx, zp, C, sigma_m, sigma_p, sigma_z, mask, lpp, gp));
        else SSI_TRY(ssi_logpost_device(ctx, zp, C, sigma_m, sigma_p, sigma_z, mask, lpp, nullptr));
        units += ctx->stats.last_units;
        flops += ctx->stats.last_flops;
        k_mh_accept<<<g_acc, 256, 0, ctx->stream>>>(z, zp, lp, lpp, C, M, seed, chain_off, 0u, 1, nullptr, nullptr, nullptr, cnt, g, gp,
                                                  half_s2, inv2s2, ctx->opt_mala_rule);
        SSI_LAUNCH_CHECK(ctx);
    }
    for (int64_t i = 0; i < S; ++i) {
        const int64_t t = step0 + i;
        if (kind == 2 && t > 0) {
            SSI_TRY(ssi_hmc_transition(ctx, C, seed, chain_off, t, hp, sigma_z, sigma_m, sigma_p, mask,
                                       d_ztr ? d_ztr + (size_t)i * C * M : nullptr, d_lptr ? d_lptr + (size_t)i * C : nullptr,
                                       d_acctr ? d_acctr + (size_t)i * C : nullptr, d_etr ? d_etr + (size_t)i * C : nullptr, &units, &flops));
            continue;
        }
        if (t == 0 && d_z0) {
            SSI_CUDA(ctx, cudaMemcpyAsync(zp, d_z0, sizeof(float) * (size_t)M * C, cudaMemcpyDeviceToDevice, ctx->stream));
        } else {
            k_mh_propose<<<g_prop, 256, 0, ctx->stream>>>(z, zp, C, M, seed, chain_off, (unsigned)t, (float)sigma_z, t == 0, g, half_s2);
            SSI_LAUNCH_CHECK(ctx);
        }
        if (kind != 0) SSI_TRY(ssi_logpost_grad_device(ctx, zp, C, sigma_m, sigma_p, sigma_z, mask, lpp, gp));
        else SSI_TRY(ssi_logpost_device(ctx, zp, C, sigma_m, sigma_p, sigma_z, mask, lpp, nullptr));
        units += ctx->stats.last_units;
        flops += ctx->stats.last_flops;
        // trace row i of this call = step t of the chain
        k_mh_accept<<<g_acc, 256, 0, ctx->stream>>>(z, zp, lp, lpp, C, M, seed, chain_off, (unsigned)t, t == 0,
                                                  d_ztr ? d_ztr + (size_t)i * C * M : nullptr, d_lptr ? d_lptr + (size_t)i * C : nullptr,
                                                  d_acctr ? d_acctr + (size_t)i * C : nullptr, cnt, g, gp, half_s2, inv2s2, ctx->opt_mala_rule);
        SSI_LAUNCH_CHECK(ctx);
        // the initial sample has no step size: all-ones bytes are a NaN double
        if (kind == 2 && d_etr) SSI_CUDA(ctx, cudaMemsetAsync(d_etr, 0xff, sizeof(double) * (size_t)C, ctx->stream));
    }
    ctx->stats.last_units = units;
    ctx->stats.last_flops = flops;
    ctx->stats.mh_proposals = C * (S - (step0 == 0 ? 1 : 0));
    ctx->mh_chains = C;
    ctx->mh_kind = kind;
    return SSI_OK;
}

int ssi_mh_fetch_accepts(ssi_ctx* ctx) {
    unsigned long long h = 0;
    if (!ctx->bMhCnt.p) return SSI_OK;
    SSI_CUDA(ctx, cudaMemcpyAsync(&h, ctx->bMhCnt.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stats.mh_accepts = (int64_t)h;
    return SSI_OK;
}
