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
// step_offset > 0 continues chains (SURVEY 5, checkpoint / resume): z0 is then the state after step step_offset - 1, its
// log-density (and gradient) is re-evaluated -- the evaluation is deterministic and batch-invariant, so the continued run
// is bit-identical to an uninterrupted one -- and the following steps draw from the Philox counters of those steps; trace
// row i receives step step_offset + i.
// kind 2: fixed-length HMC with per-chain dual averaging (ssi_hmc.cu): sample 0 and the re-established state of a continued
//   run are MALA's (value and gradient cached per chain); every later step is one HMC transition.  adapt0 is the
//   adaptation state after step step_offset - 1 (NULL: the initial one); step_size_trace receives the step size of every
//   transition (NaN for step 0).
// The arguments have been checked by the public entry point.
int ssi_mh_device(ssi_ctx* ctx, const ssi_mh_run_t& r) {
    const int M = ctx->Mz;         // the sampler works in the caller's z (a decoder maps it inside the density)
    const int64_t C = r.n_chains;
    SSI_TRY(ssi_reserve(ctx, ctx->bMhZ, sizeof(float) * (size_t)M * C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhZp, sizeof(float) * (size_t)M * C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhLp, sizeof(double) * (size_t)C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhLpP, sizeof(double) * (size_t)C));
    SSI_TRY(ssi_reserve(ctx, ctx->bMhCnt, sizeof(unsigned long long)));
    double *g = nullptr, *gp = nullptr;
    if (r.kind != 0) {
        SSI_TRY(ssi_reserve(ctx, ctx->bMhG, sizeof(double) * 2 * (size_t)M * C));
        g = (double*)ctx->bMhG.p;
        gp = g + (size_t)M * C;
    }
    const double half_s2 = 0.5 * r.sigma_z * r.sigma_z, inv2s2 = 1.0 / (2.0 * r.sigma_z * r.sigma_z);
    float* z = (float*)ctx->bMhZ.p;
    float* zp = (float*)ctx->bMhZp.p;
    double* lp = (double*)ctx->bMhLp.p;
    double* lpp = (double*)ctx->bMhLpP.p;
    unsigned long long* cnt = (unsigned long long*)ctx->bMhCnt.p;
    SSI_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), ctx->stream));
    if (r.kind == 2) SSI_TRY(ssi_hmc_prepare(ctx, r));

    const int nblk = (M + 3) / 4;
    const unsigned g_prop = (unsigned)((C * nblk + 255) / 256);
    const unsigned g_acc = (unsigned)((C + 255) / 256);
    double units = 0, flops = 0;

    if (r.step_offset > 0) {
        // re-establish (z, lp[, grad]) of the saved state: evaluate it as a proposal and force-accept it without a trace row
        SSI_CUDA(ctx, cudaMemcpyAsync(zp, r.z0, sizeof(float) * (size_t)M * C, cudaMemcpyDeviceToDevice, ctx->stream));
        SSI_TRY(ssi_mh_density(ctx, r, zp, lpp, gp, &units, &flops));
        k_mh_accept<<<g_acc, 256, 0, ctx->stream>>>(z, zp, lp, lpp, C, M, r.seed, r.chain_offset, 0u, 1, nullptr, nullptr, nullptr, cnt,
                                                  g, gp, half_s2, inv2s2, ctx->opt_mala_rule);
        SSI_LAUNCH_CHECK(ctx);
    }
    for (int64_t i = 0; i < r.n_steps; ++i) {
        const int64_t t = r.step_offset + i;
        if (r.kind == 2 && t > 0) {
            SSI_TRY(ssi_hmc_transition(ctx, r, i, &units, &flops));
            continue;
        }
        if (t == 0 && r.z0) {
            SSI_CUDA(ctx, cudaMemcpyAsync(zp, r.z0, sizeof(float) * (size_t)M * C, cudaMemcpyDeviceToDevice, ctx->stream));
        } else {
            k_mh_propose<<<g_prop, 256, 0, ctx->stream>>>(z, zp, C, M, r.seed, r.chain_offset, (unsigned)t, (float)r.sigma_z, t == 0, g, half_s2);
            SSI_LAUNCH_CHECK(ctx);
        }
        SSI_TRY(ssi_mh_density(ctx, r, zp, lpp, gp, &units, &flops));
        // trace row i of this call = step t of the chain
        k_mh_accept<<<g_acc, 256, 0, ctx->stream>>>(z, zp, lp, lpp, C, M, r.seed, r.chain_offset, (unsigned)t, t == 0,
                                                  r.z_trace ? r.z_trace + (size_t)i * C * M : nullptr, r.lp_trace ? r.lp_trace + (size_t)i * C : nullptr,
                                                  r.accept_trace ? r.accept_trace + (size_t)i * C : nullptr, cnt, g, gp, half_s2, inv2s2, ctx->opt_mala_rule);
        SSI_LAUNCH_CHECK(ctx);
        // the initial sample has no step size: all-ones bytes are a NaN double
        if (r.kind == 2 && r.step_size_trace)
            SSI_CUDA(ctx, cudaMemsetAsync(r.step_size_trace, 0xff, sizeof(double) * (size_t)C, ctx->stream));
    }
    ctx->stats.last_units = units;
    ctx->stats.last_flops = flops;
    ctx->stats.mh_proposals = C * (r.n_steps - (r.step_offset == 0 ? 1 : 0));
    ctx->mh_chains = C;
    ctx->mh_kind = r.kind;
    return SSI_OK;
}

int ssi_mh_density(ssi_ctx* ctx, const ssi_mh_run_t& r, const float* zp, double* lpp, double* gp, double* units, double* flops) {
    if (r.kind != 0) SSI_TRY(ssi_logpost_grad_device(ctx, zp, r.n_chains, r.sigma_m, r.sigma_p, r.sigma_z, r.mask, lpp, gp));
    else SSI_TRY(ssi_logpost_device(ctx, zp, r.n_chains, r.sigma_m, r.sigma_p, r.sigma_z, r.mask, lpp, nullptr));
    *units += ctx->stats.last_units;
    *flops += ctx->stats.last_flops;
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
