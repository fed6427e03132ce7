// ssi_hmc.cu — fixed-length Hamiltonian Monte Carlo (alg = :static_hmc) over many chains, with per-chain dual averaging.
//
// One transition of AdvancedHMC's StaticTrajectory (Turing's HMC(eps, n_leapfrog)) with a diagonal inverse metric m^-1:
//   p_i = n_i / sqrt(m^-1_i) with n the FP32 normals of stream 0 at (chain, t) -- the RWMH proposal noise of step t;
//   p += eps/2 g(z); L - 1 times { z_i = float((double)z_i + eps m^-1_i p_i); g = grad lp(z); p += eps g };
//   z_i = float((double)z_i + eps m^-1_i p_i); g = grad lp(z); p += eps/2 g;
//   H = -lp + 1/2 sum m^-1_i p_i^2 (FP64); accept iff -e < -(H' - H), e the Exp(1) variate of stream 1 at (chain, t).
// A drift that produces a non-finite z, or a non-finite or > 1000 energy error, makes the transition divergent: it is
// rejected, and from that drift on its position is held at the trajectory's start so that the density kernels never see a
// NaN or Inf.  The step size adapts per chain by dual averaging (Hoffman & Gelman 2014, Alg. 5, with Stan's constants):
// pooling across chains would make a chain's trace depend on which other chains share the call.
//
// The L gradient evaluations are the batched ssi_logpost_grad_device calls of MALA; the kernels here are the integrator
// around them, one thread per chain (M <= 64): k_hmc_begin, L - 1 x k_hmc_leap, k_hmc_end.
#include "ssi_common.cuh"
#include "ssi_rng.cuh"

#include <cmath>

namespace {

constexpr double kDaGamma = 0.05, kDaT0 = 10.0, kDaKappa = 0.75;   // StepSizeAdaptor / Stan defaults
constexpr double kMaxDeltaH = 1000.0;                            // AdvancedHMC's divergence threshold

struct hmc_minv_t {
    double v[SSI_MAX_M];
};

// (double)z + (eps * m^-1) * p rounded once to float; no contraction, so the oracle can restate it exactly
__device__ __forceinline__ float hmc_drift(float z, double eps_minv, double p) {
    return (float)__dadd_rn((double)z, __dmul_rn(eps_minv, p));
}

}  // namespace

// momentum, start energy, first half kick and first drift; fixes the step size eps_t of the chain for this transition
__global__ void __launch_bounds__(128)
k_hmc_begin(long long n_chains, int M, unsigned long long seed, long long chain_off, unsigned step, hmc_minv_t minv,
            double eps0, long long n_adapts, const float* __restrict__ z, const double* __restrict__ lp,
            const double* __restrict__ g, float* __restrict__ zp, double* __restrict__ p, double* __restrict__ h0,
            double* __restrict__ eps, const double* __restrict__ ad, unsigned char* __restrict__ div) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chains) return;
    const double e = n_adapts == 0 ? eps0 : exp((long long)step <= n_adapts ? ad[3 * c] : ad[3 * c + 1]);
    eps[c] = e;
    const double half_e = 0.5 * e;
    double kin = 0.0;
    bool bad = false;
    for (int blk = 0; blk * 4 < M; ++blk) {
        float nrm[4];
        ssi_normal4(seed, (uint32_t)(chain_off + c), step, (uint32_t)blk, nrm);
        for (int r = 0; r < 4 && blk * 4 + r < M; ++r) {
            const int m = blk * 4 + r;
            const size_t i = (size_t)m + (size_t)c * M;
            double pm = __ddiv_rn((double)nrm[r], __dsqrt_rn(minv.v[m]));
            kin = __dadd_rn(kin, __dmul_rn(__dmul_rn(minv.v[m], pm), pm));
            pm = __dadd_rn(pm, __dmul_rn(half_e, g[i]));
            p[i] = pm;
            const float zn = hmc_drift(z[i], __dmul_rn(e, minv.v[m]), pm);
            zp[i] = zn;
            bad |= !isfinite(zn);
        }
    }
    h0[c] = __dadd_rn(-lp[c], 0.5 * kin);
    if (bad)
        for (int m = 0; m < M; ++m) zp[(size_t)m + (size_t)c * M] = z[(size_t)m + (size_t)c * M];
    div[c] = bad ? 1 : 0;
}

// one full kick with the gradient at zp and one drift; a divergent chain stays at the trajectory's start z
__global__ void __launch_bounds__(128)
k_hmc_leap(long long n_chains, int M, hmc_minv_t minv, const float* __restrict__ z, float* __restrict__ zp,
           double* __restrict__ p, const double* __restrict__ gp, const double* __restrict__ eps, unsigned char* __restrict__ div) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chains || div[c]) return;
    const double e = eps[c];
    bool bad = false;
    for (int m = 0; m < M; ++m) {
        const size_t i = (size_t)m + (size_t)c * M;
        const double pm = __dadd_rn(p[i], __dmul_rn(e, gp[i]));
        p[i] = pm;
        const float zn = hmc_drift(zp[i], __dmul_rn(e, minv.v[m]), pm);
        zp[i] = zn;
        bad |= !isfinite(zn);
    }
    if (bad) {
        for (int m = 0; m < M; ++m) zp[(size_t)m + (size_t)c * M] = z[(size_t)m + (size_t)c * M];
        div[c] = 1;
    }
}

// last half kick, energy error, divergence test, accept / reject, state and trace writes, dual-averaging update and the
// warp-aggregated accept count.  accept trace: 1 accepted, 0 rejected, 2 rejected as divergent.
__global__ void __launch_bounds__(128)
k_hmc_end(long long n_chains, int M, unsigned long long seed, long long chain_off, unsigned step, hmc_minv_t minv,
          double eps0, long long n_adapts, double delta, float* __restrict__ z, double* __restrict__ lp, double* __restrict__ g,
          const float* __restrict__ zp, const double* __restrict__ lpp, const double* __restrict__ gp, const double* __restrict__ p,
          const double* __restrict__ h0, const double* __restrict__ eps, double* __restrict__ ad, const unsigned char* __restrict__ div,
          float* __restrict__ z_trace, double* __restrict__ lp_trace, unsigned char* __restrict__ acc_trace,
          double* __restrict__ eps_trace, unsigned long long* __restrict__ n_acc) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned accepted = 0;
    if (c < n_chains) {
        const double e = eps[c], half_e = 0.5 * e;
        double kin = 0.0;
        for (int m = 0; m < M; ++m) {
            const size_t i = (size_t)m + (size_t)c * M;
            const double pm = __dadd_rn(p[i], __dmul_rn(half_e, gp[i]));
            kin = __dadd_rn(kin, __dmul_rn(__dmul_rn(minv.v[m], pm), pm));
        }
        const double dH = __dadd_rn(__dadd_rn(-lpp[c], 0.5 * kin), -h0[c]);
        const bool divergent = div[c] || !isfinite(dH) || dH > kMaxDeltaH;
        const double ex = ssi_exp1(seed, (uint32_t)(chain_off + c), step);
        const bool acc = !divergent && (-ex < -dH);
        const double alpha = divergent ? 0.0 : (dH <= 0.0 ? 1.0 : exp(-dH));
        if (acc) {
            lp[c] = lpp[c];
            for (int m = 0; m < M; ++m) {
                const size_t i = (size_t)m + (size_t)c * M;
                z[i] = zp[i];
                g[i] = gp[i];
            }
        }
        if (z_trace) {            // the trace pointers address this step's row
            float* dst = z_trace + c * M;
            for (int m = 0; m < M; ++m) dst[m] = z[m + c * M];
        }
        if (lp_trace) lp_trace[c] = lp[c];
        if (acc_trace) acc_trace[c] = acc ? 1 : (divergent ? 2 : 0);
        if (eps_trace) eps_trace[c] = e;
        if ((long long)step <= n_adapts) {
            // dual averaging after transition m = step (Hoffman & Gelman 2014, Alg. 5)
            const double mm = (double)step, w = 1.0 / (mm + kDaT0);
            const double mu = log(10.0 * eps0);
            const double hbar = (1.0 - w) * ad[3 * c + 2] + (delta - alpha) * w;
            const double log_eps = mu - sqrt(mm) / kDaGamma * hbar;
            const double mk = pow(mm, -kDaKappa);
            ad[3 * c] = log_eps;
            ad[3 * c + 1] = mk * log_eps + (1.0 - mk) * ad[3 * c + 1];
            ad[3 * c + 2] = hbar;
        }
        accepted = acc ? 1u : 0u;
    }
    const unsigned warp_cnt = __popc(__ballot_sync(0xffffffffu, accepted));
    if ((threadIdx.x & 31) == 0 && warp_cnt) atomicAdd(n_acc, (unsigned long long)warp_cnt);
}

// (log eps, log eps_bar, H_bar) = (log eps0, 0, 0) for every chain
__global__ void k_hmc_adapt_init(long long n_chains, double log_eps0, double* __restrict__ ad) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chains) return;
    ad[3 * c] = log_eps0;
    ad[3 * c + 1] = 0.0;
    ad[3 * c + 2] = 0.0;
}

int ssi_hmc_check(ssi_ctx* ctx, const ssi_hmc_params_t* hp, int M) {
    if (!hp) return ssi_fail(ctx, SSI_ERR_ARG, "HMC parameters are NULL");
    if (!(hp->step_size > 0.0) || !std::isfinite(hp->step_size))
        return ssi_fail(ctx, SSI_ERR_ARG, "step_size must be positive and finite (got %g)", hp->step_size);
    if (hp->n_leapfrog < 1) return ssi_fail(ctx, SSI_ERR_ARG, "n_leapfrog must be >= 1 (got %d)", hp->n_leapfrog);
    if (hp->n_adapts < 0 || hp->n_adapts > 0xffffffffll)
        return ssi_fail(ctx, SSI_ERR_ARG, "n_adapts must be in [0, 2^32) (got %lld)", (long long)hp->n_adapts);
    if (!(hp->target_accept > 0.0 && hp->target_accept < 1.0))
        return ssi_fail(ctx, SSI_ERR_ARG, "target_accept must be in (0, 1) (got %g)", hp->target_accept);
    if (M > SSI_MAX_M) return ssi_fail(ctx, SSI_ERR_ARG, "M=%d exceeds the supported maximum %d", M, SSI_MAX_M);
    if (hp->inv_metric)
        for (int m = 0; m < M; ++m)
            if (!(hp->inv_metric[m] > 0.0) || !std::isfinite(hp->inv_metric[m]))
                return ssi_fail(ctx, SSI_ERR_ARG, "inv_metric[%d] must be positive and finite (got %g)", m, hp->inv_metric[m]);
    return SSI_OK;
}

// per-run state: the integrator buffers and the adaptation state, (log eps0, 0, 0) or run.adapt0 (3 x n_chains, device)
int ssi_hmc_prepare(ssi_ctx* ctx, const ssi_mh_run_t& r) {
    const int M = ctx->Mz;
    const int64_t C = r.n_chains;
    SSI_TRY(ssi_reserve(ctx, ctx->bHmcP, sizeof(double) * (size_t)M * C));
    SSI_TRY(ssi_reserve(ctx, ctx->bHmcH0, sizeof(double) * (size_t)C));
    SSI_TRY(ssi_reserve(ctx, ctx->bHmcEps, sizeof(double) * (size_t)C));
    SSI_TRY(ssi_reserve(ctx, ctx->bHmcAd, sizeof(double) * 3 * (size_t)C));
    SSI_TRY(ssi_reserve(ctx, ctx->bHmcDiv, (size_t)C));
    double* ad = (double*)ctx->bHmcAd.p;
    if (r.adapt0) {
        SSI_CUDA(ctx, cudaMemcpyAsync(ad, r.adapt0, sizeof(double) * 3 * (size_t)C, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        k_hmc_adapt_init<<<(unsigned)((C + 127) / 128), 128, 0, ctx->stream>>>(C, std::log(r.hp->step_size), ad);
        SSI_LAUNCH_CHECK(ctx);
    }
    return SSI_OK;
}

// transition t = step_offset + i >= 1 of all chains into trace row i: (z, lp, g) = (bMhZ, bMhLp, first half of bMhG) is
// the current state, bMhZp / bMhLpP / the second half of bMhG hold the trajectory
int ssi_hmc_transition(ssi_ctx* ctx, const ssi_mh_run_t& r, int64_t i, double* units, double* flops) {
    const int M = ctx->Mz;
    const int64_t C = r.n_chains;
    const unsigned t = (unsigned)(r.step_offset + i);
    const ssi_hmc_params_t* hp = r.hp;
    hmc_minv_t minv;
    for (int m = 0; m < SSI_MAX_M; ++m) minv.v[m] = (hp->inv_metric && m < M) ? hp->inv_metric[m] : 1.0;
    float* z = (float*)ctx->bMhZ.p;
    float* zp = (float*)ctx->bMhZp.p;
    double* lp = (double*)ctx->bMhLp.p;
    double* lpp = (double*)ctx->bMhLpP.p;
    double* g = (double*)ctx->bMhG.p;
    double* gp = g + (size_t)M * C;
    double* p = (double*)ctx->bHmcP.p;
    double* h0 = (double*)ctx->bHmcH0.p;
    double* eps = (double*)ctx->bHmcEps.p;
    double* ad = (double*)ctx->bHmcAd.p;
    unsigned char* div = (unsigned char*)ctx->bHmcDiv.p;
    unsigned long long* cnt = (unsigned long long*)ctx->bMhCnt.p;
    const unsigned grid = (unsigned)((C + 127) / 128);

    k_hmc_begin<<<grid, 128, 0, ctx->stream>>>(C, M, r.seed, r.chain_offset, t, minv, hp->step_size, hp->n_adapts, z, lp, g, zp, p,
                                               h0, eps, ad, div);
    SSI_LAUNCH_CHECK(ctx);
    for (int l = 0; l < hp->n_leapfrog; ++l) {
        if (l > 0) {
            k_hmc_leap<<<grid, 128, 0, ctx->stream>>>(C, M, minv, z, zp, p, gp, eps, div);
            SSI_LAUNCH_CHECK(ctx);
        }
        SSI_TRY(ssi_mh_density(ctx, r, zp, lpp, gp, units, flops));
    }
    k_hmc_end<<<grid, 128, 0, ctx->stream>>>(C, M, r.seed, r.chain_offset, t, minv, hp->step_size, hp->n_adapts, hp->target_accept,
                                             z, lp, g, zp, lpp, gp, p, h0, eps, ad, div, r.z_trace ? r.z_trace + (size_t)i * C * M : nullptr,
                                             r.lp_trace ? r.lp_trace + (size_t)i * C : nullptr, r.accept_trace ? r.accept_trace + (size_t)i * C : nullptr,
                                             r.step_size_trace ? r.step_size_trace + (size_t)i * C : nullptr, cnt);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}
