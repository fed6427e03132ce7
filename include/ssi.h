/*
 * ssi.h — C ABI of the B200-native subspace log-posterior library (libssi.so).
 *
 * The reference (efmanu/SubspaceInference.jl) has no FFI seam: its hot path is an
 * inline Julia closure.  This header defines the seam at exactly the two cut points
 * SURVEY.md 8(b) names, so that the Julia functions above it keep their signatures
 * and reach CUDA only through `ccall` (see INTEGRATION.md for the Julia stubs):
 *
 *   - density(z) closure + the RWMH sampler loop   src/space_inference.jl:90-95, :108-116, :125
 *   - SWA moments / deviation matrix / psvd / P    src/subspace_construction.jl:31, :44-52, :61-65
 *
 * Conventions
 *   - every entry point is extern "C", takes plain pointers and sizes, returns
 *     0 on success and a negative SSI_ERR_* code on failure; the message is kept per
 *     context (ssi_last_error).  No C++ exception crosses the ABI.
 *   - all matrices are COLUMN-MAJOR (Julia-native), so the shim passes pointer(Array):
 *       X  in0 x N      Y  O x N      P  n x M      Z  M x B
 *       z_trace  M x n_chains x n_steps          lp_trace / accept_trace  n_chains x n_steps
 *   - flat parameter order is Flux.destructure's: per Dense layer vec(W_l) (out x in,
 *     column-major) followed by b_l                 src/libs.jl:55-57, :19-22
 *   - the caller owns every buffer for the duration of the call only; the context owns
 *     all device memory and its stream; set_* calls copy.
 *   - a context is not re-entrant.  ssi_ctx_create binds it to ONE device; ssi_ctx_create_multi returns a context that
 *     drives several devices from the one calling process (the reference is a single Julia process,
 *     src/space_inference.jl:82-84): set_* calls are replicated, the batched host-pointer calls shard samples / chains
 *     across the devices and every device lands its slice in the caller's host arrays.  A sampler run's arguments are
 *     checked before it is sharded, so a rejected run fails as on one device and leaves the last run's state readable.
 *     Alternatively one process (and one context) per GPU shards chains by `chain_offset`.  Either way the counter-based
 *     RNG is keyed on the GLOBAL chain id, so results do not depend on the number of GPUs.
 *   - distinct contexts are independent (no shared mutable state), also on the same device.
 *   - there is no CPU fallback: every compute entry point fails with SSI_ERR_CUDA when
 *     no sm_100 device is usable.
 */
#ifndef SSI_H
#define SSI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSI_VERSION 200            /* 0.2.0 */

/* error codes */
#define SSI_OK             0
#define SSI_ERR_ARG       -1       /* bad argument / call order */
#define SSI_ERR_CUDA      -2       /* CUDA runtime or driver failure, or no usable device */
#define SSI_ERR_STATE     -3       /* model / data / subspace not set */
#define SSI_ERR_RANK      -4       /* deviation matrix has fewer than M usable columns */
#define SSI_ERR_UNSUPPORTED -5
#define SSI_ERR_RANGE     -6       /* asynchronous (*_dev) tensor-path results since the last ssi_sync are invalid: an
                                    * activation left the calibrated FP16 range; the context has switched to BF16 planes,
                                    * repeat the calls (the host-pointer entry points repeat by themselves)             */

/* activation codes for ssi_set_model (Flux/NNlib: identity, relu, tanh, sigmoid) */
#define SSI_ACT_IDENTITY 0
#define SSI_ACT_RELU     1
#define SSI_ACT_TANH     2
#define SSI_ACT_SIGMOID  3

/* terms of the log-posterior; `prior_mask` is an OR of these.
 * The reference AS EXECUTED is SSI_TERM_LL only: its weight-prior line is dead code
 * (src/space_inference.jl:94-95, a line-leading `+` after a complete `return`).
 * SSI_TERM_LL|SSI_TERM_PRIOR_W is what the docs describe (docs/src/nn_example.md:61-68). */
#define SSI_TERM_LL       1u       /* logpdf(MvNormal(vec(pred), sigma_m), vec(Y))       :94 */
#define SSI_TERM_PRIOR_W  2u       /* logpdf(MvNormal(zeros(n), sigma_p), W_swa + P z)   :95 */
#define SSI_TERM_PRIOR_Z  4u       /* logpdf(MvNormal(zeros(M), sigma_z), z)  (north_star) */

/* execution paths for ssi_set_option("path", ...) */
#define SSI_PATH_AUTO     0
#define SSI_PATH_FUSED    1        /* one CTA keeps a sample's whole network in shared memory */
#define SSI_PATH_LAYERED  2        /* per-layer FP32 SIMT GEMMs (any shape)                  */
#define SSI_PATH_TENSOR   3        /* tcgen05/TMEM/TMA split-precision GEMMs (wide layers)   */
#define SSI_PATH_BASIS    4        /* one hidden layer, O <= 2: first layer affine in z       */

typedef struct ssi_ctx ssi_ctx;

typedef struct ssi_stats_t {
    double last_ms;            /* device time of the last compute call (CUDA events on the ctx stream) */
    double last_flops;         /* algorithmic flops of that call: 2*sum(in*out)*N*B + 2*n*M*B          */
    double last_bytes;         /* algorithmic HBM bytes of that call (construction streams), else 0     */
    double last_units;         /* (sample x datapoint) units of that call                              */
    int64_t kernel_launches;   /* kernels launched by this context since creation                      */
    int64_t mh_accepts;        /* accepted proposals in the last ssi_mh_run / ssi_mala_run / ssi_hmc_run */
    int64_t mh_proposals;      /* proposals (transitions) in that run                                  */
    int32_t last_path;         /* SSI_PATH_* actually used by the last log-posterior evaluation        */
    int32_t sm_count;
    int32_t gram_path;         /* last ssi_swa_finish: 1 FP64 SIMT Gram, 2 tensor-core Gram, 3 tensor-core Gram
                                * rejected by the conditioning check and recomputed in FP64               */
    int32_t jacobi_sweeps;     /* sweeps of the last eigen-solve                                         */
    double gram_risk;          /* conditioning estimate of the tensor-core Gram (see DESIGN.md 4.4)       */
    double dominant_ms;        /* with option "time_dominant": summed device time of the path's dominant   */
    int64_t dominant_launches; /* kernel since the option was set (CUDA events on the launching stream)    */
    double finish_gram_ms;     /* last ssi_swa_finish, CUDA events on the context stream: Gram (K6),        */
    double finish_eigen_ms;    /* eigen-solve + conditioning check (K7),                                    */
    double finish_p_ms;        /* P = A V_M (K8)                                                            */
    int64_t tc_range_fallbacks;/* tensor path: evaluations repeated on BF16 planes because an activation left the   */
                               /* calibrated range of the FP16 planes (see DESIGN.md 4.1); 0 in normal operation   */
    int64_t gemm_tc_launches;  /* gradient / training GEMMs this context ran on the tensor cores (ssi_gemm_tc.cu)     */
    int64_t gemm_skinny_launches; /* narrow-layer GEMMs of the gradient / training paths that ran on k_gemm_skinny_* */
} ssi_stats_t;

int  ssi_version(void);

/* ---- lifecycle ------------------------------------------------------------------- */
int  ssi_ctx_create(int device, ssi_ctx** out);
/* One context over n_dev devices (SURVEY 8(b)-1): W_swa, P, X, Y are replicated on every device; ssi_logpost_batch,
 * ssi_logpost_grad_batch, ssi_mh_run, ssi_mala_run, ssi_mh_run_from, ssi_hmc_run, ssi_mh_get_state, ssi_hmc_get_adapt and
 * ssi_project split their B samples /
 * n_chains chains into contiguous ranges, one per device (chains keep their global ids: traces are bit-identical to a
 * one-device run); ssi_predict_batch, ssi_swa_* and ssi_train_* run on devices[0] (an installed subspace is replicated).
 * The *_dev entry points and ssi_set_stream take pointers / streams of ONE device and return SSI_ERR_UNSUPPORTED here.
 * ssi_stats reports the maximum over devices for times and the sum for work and counters.                          */
int  ssi_ctx_create_multi(const int32_t* devices, int32_t n_dev, ssi_ctx** out);
int  ssi_ctx_devices(const ssi_ctx* ctx);       /* number of devices the context drives */
int  ssi_ctx_destroy(ssi_ctx* ctx);
/* message of the last failure on `ctx` (or of the last failed ssi_ctx_create when ctx==NULL) */
const char* ssi_last_error(const ssi_ctx* ctx);
/* run on a caller-provided cudaStream_t (e.g. torch's current stream); NULL restores the ctx stream */
int  ssi_set_stream(ssi_ctx* ctx, void* cuda_stream);
int  ssi_sync(ssi_ctx* ctx);
/* keys: "path" (SSI_PATH_*), "group" (samples per wave on the tensor path), "tc_precision" (operand planes of the tensor
 * path: 1 = FP16 planes with power-of-two scales, the default; 0 = BF16x3), "mala_rule" (0 = the documented Metropolis-adjusted
 * Langevin ratio, the default; 1 = both proposal densities evaluated with the negated gradient, see ssi_mala_run),
 * "grad_group_gb" (scratch budget of the generic gradient path per group of samples; default a third of the free memory),
 * and switches used by the tests to force a path the library also selects on its own for some shapes, or a reference
 * kernel: "tc_nobasis", "tc_nofuse", "tc_noorder", "tc_simt_basis", "tc_pair" (1 = CTA pairs with cta_group::2, the
 * default), "b1_simt", "gram_fp64" (1 = FP64 SIMT Gram; 0 = tensor-core Gram guarded by a conditioning check, the default;
 * -1 = tensor-core Gram without the check), "gemm_simt" (1 = gradient / training GEMMs on the SIMT kernel); "time_dominant"
 * (0/1) brackets every launch of the path's dominant kernel with CUDA events (ssi_stats_t.dominant_ms).  Any other key
 * returns SSI_ERR_ARG. */
int  ssi_set_option(ssi_ctx* ctx, const char* key, int64_t value);
int  ssi_stats(const ssi_ctx* ctx, ssi_stats_t* out);

/* ---- the closure's captured state (src/space_inference.jl:86-90) ------------------- */
/* Chain(Dense(dims[0],dims[1],act[0]), ..., Dense(dims[L-1],dims[L],act[L-1]))            */
int  ssi_set_model(ssi_ctx* ctx, int n_layers, const int32_t* dims, const int32_t* act);
/* full dataset, as split_data returns it (src/libs.jl:75-77); host pointers, copied      */
int  ssi_set_data(ssi_ctx* ctx, const float* X, const float* Y, int64_t N);
/* W_swa (n) and P (n x M column-major), host pointers, copied; n must match the model    */
int  ssi_set_subspace(ssi_ctx* ctx, const float* W_swa, const float* P, int64_t n, int32_t M);

/* ---- non-linear subspace operator (SURVEY 8(f)-4): the density of auto_inference, src/space_inference.jl:246-251 -----------
 *     new_W = W_swa + decoder(z)
 * with `decoder` the Flux Chain of Dense layers trained by auto_encoder_subspace (src/subspace_construction.jl:125-141):
 * Chain(Dense(dims[0], dims[1], act[0]), ..., Dense(dims[L-1], dims[L], act[L-1])), dims[0] = the subspace dimension of z,
 * dims[L] = n (the model's parameter count), theta in Flux.destructure order (host, copied), W_swa n floats.  Replaces
 * ssi_set_subspace: afterwards every entry point takes z of dims[0] rows (ssi_logpost_*, ssi_mh_*, ssi_mala_*, ssi_project,
 * ssi_predict_batch).  The widths before the last layer are limited to 64.  The last layer is affine up to its activation, so
 * with act[L-1] = identity the whole fast path applies at z' = h(z) (DESIGN.md 4.7); another activation materialises the
 * weights per sample (LAYERED path; no weight prior, no gradient).  As in the reference's Chain branch, the weight-prior
 * line of that density is dead code (src/space_inference.jl:250-251): the default prior_mask stays SSI_TERM_LL.        */
int  ssi_set_decoder(ssi_ctx* ctx, const float* W_swa, int32_t n_layers, const int32_t* dims, const int32_t* act, const float* theta);

/* ---- density(z), batched over B subspace points (src/space_inference.jl:90-95) ----- */
/* Z: M x B (host).  lp_out: B doubles.  terms_out: 3 x B doubles (ll, prior_w, prior_z) or NULL. */
int  ssi_logpost_batch(ssi_ctx* ctx, const float* Z, int64_t B,
                       double sigma_m, double sigma_p, double sigma_z, uint32_t prior_mask,
                       double* lp_out, double* terms_out);
/* same with DEVICE pointers; asynchronous on the ctx stream (ssi_sync to wait)            */
int  ssi_logpost_batch_dev(ssi_ctx* ctx, const float* dZ, int64_t B,
                           double sigma_m, double sigma_p, double sigma_z, uint32_t prior_mask,
                           double* d_lp_out, double* d_terms_out);

/* ---- l_pi_grad(theta) = (density(theta), gradient(density, theta)), batched ------------
 * src/space_inference.jl:107 (AD backends src/libs.jl:23-34): the closure the :mala, :hmc and :nuts branches
 * (:117-120, :139-160) hand to their samplers.  One reverse pass per sample instead of ForwardDiff's M forward passes.
 * Z: M x B (host); lp_out: B doubles; grad_out: M x B doubles (d lp / d z), same prior_mask semantics as above.       */
int  ssi_logpost_grad_batch(ssi_ctx* ctx, const float* Z, int64_t B,
                            double sigma_m, double sigma_p, double sigma_z, uint32_t prior_mask,
                            double* lp_out, double* grad_out);
int  ssi_logpost_grad_batch_dev(ssi_ctx* ctx, const float* dZ, int64_t B,
                                double sigma_m, double sigma_p, double sigma_z, uint32_t prior_mask,
                                double* d_lp_out, double* d_grad_out);

/* ---- sample(DensityModel(density), RWMH(MvNormal(zeros(M), sigma_z)), itr) ----------
 * src/space_inference.jl:111-116.  n_chains independent chains, global ids
 * chain_offset .. chain_offset+n_chains-1.  Sample 0 of each chain is a draw from the
 * proposal (or z0 if given, M x n_chains) and counts as the first of n_steps; step t
 * proposes z + sigma_z*eps(chain,t) and accepts iff -e(chain,t) < lp' - lp, with eps and
 * e from the Philox stream ssi_rng_replay reproduces.  Any trace pointer may be NULL.   */
int  ssi_mh_run(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                const float* z0_or_null,
                float* z_trace, double* lp_trace, uint8_t* accept_trace);
/* same, traces left on the device (pointers are device pointers or NULL); asynchronous  */
int  ssi_mh_run_dev(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                    double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                    const float* d_z0_or_null,
                    float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace);
/* ---- sample(DensityModel(density), MALA(x -> MvNormal((sigma_z^2/2) .* x, sigma_z)), itr; init_params=...) ---------
 * src/space_inference.jl:117-120.  Same arguments, streams and trace layouts as ssi_mh_run.  Sample 0 is z0 (or a draw
 * sigma_z*eps(chain,0), the reference's init_params); step t proposes z' = z + (sigma_z^2/2) grad lp(z) + sigma_z*eps(chain,t)
 * and accepts iff -e(chain,t) < lp' - lp + log q(z|z') - log q(z'|z) with q(a|b) = N(a; b + (sigma_z^2/2) grad lp(b),
 * sigma_z^2 I) (the Metropolis-adjusted Langevin step as AdvancedMH documents it; the pinned 0.6.2 source is not
 * vendored, see DESIGN.md).  Option "mala_rule" = 1 evaluates both densities with the NEGATED gradient,
 * q(a|b) = N(a - b; -(sigma_z^2/2) grad lp(b), sigma_z^2 I) -- how that release's step is remembered to be written
 * (`proposal(-gradient)`); neither can be pinned without the source, both are held to the oracle's restatement.
 * Values and gradients come from ssi_logpost_grad_batch_dev.                                                         */
int  ssi_mala_run(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                  double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                  const float* z0_or_null,
                  float* z_trace, double* lp_trace, uint8_t* accept_trace);
int  ssi_mala_run_dev(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                      double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                      const float* d_z0_or_null,
                      float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace);
/* ---- checkpoint / resume of the chains (SURVEY 5; the docs save and reload around sampling, docs/src/nn_example.md:158,168) ----
 * The RNG is counter-based, so a chain is resumable from (seed, step, z): ssi_mh_get_state returns the final state of the last
 * run's chains (z_out M x n_chains floats, lp_out n_chains doubles, host, either may be NULL); ssi_mh_run_from continues them:
 * kind 0 = RWMH, 1 = MALA; z_state (M x n_chains) is the state after step step_offset - 1, steps step_offset ..
 * step_offset + n_steps - 1 draw from the Philox counters of those steps and fill trace rows 0 .. n_steps - 1.  The state's
 * log-density (and gradient) is re-evaluated, which is deterministic: run(0..S) is bit-identical to run(0..S/2) followed by
 * run_from(S/2..S).  step_offset == 0 is ssi_mh_run / ssi_mala_run (z_state = z0 or NULL).                                */
int  ssi_mh_get_state(ssi_ctx* ctx, float* z_out, double* lp_out);
int  ssi_mh_run_from(ssi_ctx* ctx, int32_t kind, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                     int64_t step_offset, double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                     const float* z_state, float* z_trace, double* lp_trace, uint8_t* accept_trace);
int  ssi_mh_run_from_dev(ssi_ctx* ctx, int32_t kind, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset,
                         int64_t step_offset, double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                         const float* d_z_state, float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace);
/* ---- fixed-length HMC with per-chain step-size adaptation (alg = :static_hmc) -------------------------------------------
 * AdvancedHMC's StaticTrajectory / Turing's HMC(eps, n_leapfrog) with a diagonal inverse metric, on the density of ssi_mh_run
 * (values and gradients from ssi_logpost_grad_batch_dev, n_leapfrog evaluations per transition).  Same arguments, streams
 * and trace layouts as ssi_mh_run.  Sample 0 is z_state (or sigma_z*eps(chain,0)) and counts as the first of n_steps.
 * Transition t >= 1 of a chain:
 *   p_i = n_i / sqrt(inv_metric_i) (FP64), n = the FP32 normals of stream 0 at (chain, t) -- what ssi_rng_replay returns;
 *   p += eps/2 g(z); n_leapfrog - 1 times { z_i = float((double)z_i + eps inv_metric_i p_i); g = grad lp(z); p += eps g };
 *   z_i = float((double)z_i + eps inv_metric_i p_i); g = grad lp(z); p += eps/2 g;
 *   H = -lp + 1/2 sum inv_metric_i p_i^2 (FP64); accept iff -e(chain,t) < -(H' - H)  (e: the Exp(1) variate of RWMH).
 * The transition is divergent (rejected; accept_trace 2) when a drift yields a non-finite z or H' - H is non-finite or
 * > 1000; the chain's position is then held at the trajectory's start, so no NaN or Inf reaches the density.
 * Step size: dual averaging per chain (Hoffman & Gelman 2014, Alg. 5; gamma 0.05, t0 10, kappa 0.75, mu = log(10 eps0),
 * delta = target_accept) after each transition m = t <= n_adapts, from (log eps, log eps_bar, H_bar) = (log eps0, 0, 0);
 * transition t uses exp(log eps) while t <= n_adapts and exp(log eps_bar) afterwards (n_adapts == 0: eps0 throughout).
 * Adaptation never pools across chains, so traces do not depend on which chains share a call or a device.
 *   step_size_trace  n_chains x n_steps doubles (or NULL): the eps each transition used; NaN for step 0
 *   accept_trace     1 accepted, 0 rejected, 2 rejected as divergent
 *   step_offset > 0  continues chains from z_state (the state after step step_offset - 1, ssi_mh_get_state) and, unless
 *                    n_adapts == 0, adapt_state (3 x n_chains, ssi_hmc_get_adapt): run(0..S) is bit-identical to run(0..h)
 *                    followed by run(h..S) for every h, in warm-up or after it
 * The final (z, lp) is read with ssi_mh_get_state; ssi_hmc_get_adapt returns the 3 x n_chains adaptation state of the last
 * run (SSI_ERR_STATE if the last run on the context was not HMC).  inv_metric is a host pointer in both variants.       */
typedef struct ssi_hmc_params_t {
    double  step_size;        /* initial leapfrog step size eps0 > 0                                    */
    int32_t n_leapfrog;       /* leapfrog steps per transition, >= 1                                    */
    int64_t n_adapts;         /* transitions 1..n_adapts adapt eps (dual averaging); 0 = fixed eps0     */
    double  target_accept;    /* delta in (0, 1); AdvancedHMC's StepSizeAdaptor(0.8, ...)               */
    const double* inv_metric; /* M doubles (host, copied), diagonal of M^-1; NULL = identity             */
} ssi_hmc_params_t;
int  ssi_hmc_run(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset, int64_t step_offset,
                 const ssi_hmc_params_t* hp, double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                 const float* z_state, const double* adapt_state,
                 float* z_trace, double* lp_trace, uint8_t* accept_trace, double* step_size_trace);
/* same; z_state, adapt_state and the traces are device pointers (hp->inv_metric stays a host pointer); asynchronous */
int  ssi_hmc_run_dev(ssi_ctx* ctx, int64_t n_chains, int64_t n_steps, uint64_t seed, int64_t chain_offset, int64_t step_offset,
                     const ssi_hmc_params_t* hp, double sigma_z, double sigma_m, double sigma_p, uint32_t prior_mask,
                     const float* d_z_state, const double* d_adapt_state,
                     float* d_z_trace, double* d_lp_trace, uint8_t* d_accept_trace, double* d_step_size_trace);
/* 3 x n_chains doubles (host): log eps, log eps_bar, H_bar of every chain of the last HMC run */
int  ssi_hmc_get_adapt(ssi_ctx* ctx, double* adapt_out);
/* host replay of the device stream: eps_out (M floats, N(0,1)) and e_out (Exp(1)) of (chain, step) */
int  ssi_rng_replay(uint64_t seed, int64_t chain, int64_t step, int32_t M, float* eps_out, double* e_out);
/* map(z -> W_swa + P*z, chm) (src/space_inference.jl:125): W_out n x B column-major (host) */
int  ssi_project(ssi_ctx* ctx, const float* Z, int64_t B, float* W_out);

/* ---- posterior-predictive sweep: the step AFTER the path in every docs example -------
 * docs/src/nn_example.md:207-216 (for every sample: m1 = re(W); trajectories[:, i] = m1(inp)) and
 * src/plotting.jl:8-9 (mean / std of the trajectories).  Z: M x B subspace samples, Xg: in0 x Ng grid (host).
 * mean_out / std_out: O x Ng doubles = mean(trajectories, dims=2), std(trajectories, dims=2) (corrected, B-1; NaN for
 * B == 1 as in Julia); preds_out: O x Ng x B floats (the trajectories) or NULL.  The data set need not be set.    */
int  ssi_predict_batch(ssi_ctx* ctx, const float* Z, int64_t B, const float* Xg, int64_t Ng,
                       float* preds_out, double* mean_out, double* std_out);

/* ---- subspace construction streams (src/subspace_construction.jl:31,44-52,61-65) ---- */
/* W_swa <- zeros(n) (:31), deviation matrix with room for K_max columns (:33)             */
int  ssi_swa_begin(ssi_ctx* ctx, int64_t n, int64_t K_max);
/* one snapshot W (n floats, host): W_swa <- (ns*W_swa + W)/(ns+1), column <- W - W_swa     */
/* with ns = i/c passed by the host (:46-47, :51-52)                                       */
int  ssi_swa_push(ssi_ctx* ctx, const float* W, double n_scalar);
int  ssi_swa_push_dev(ssi_ctx* ctx, const float* dW, double n_scalar);
/* psvd(A) restated as Gram + symmetric eigen-solve; P = U_M S_M = A V_M (:61-65).          */
/* W_swa_out n, P_out n x M, s_out K singular values (descending); host pointers, any NULL. */
/* If `install` != 0 the result also becomes the context's subspace (ssi_set_subspace).     */
int  ssi_swa_finish(ssi_ctx* ctx, int32_t M, float* W_swa_out, float* P_out, double* s_out, int32_t install);
/* number of columns collected so far */
int64_t ssi_swa_columns(const ssi_ctx* ctx);
/* the deviation matrix collected so far, n x K column-major (host): `reshape(A, all_len, :)` of
 * src/subspace_construction.jl:61,119,201 -- what auto_encoder_subspace trains its auto-encoder on (:134-139) and
 * diffusion_subspace hands to its diffusion map (:203)                                                             */
int  ssi_swa_deviations(ssi_ctx* ctx, float* A_out);
/* the running W_swa (n floats, host) without factorising anything */
int  ssi_swa_mean(ssi_ctx* ctx, float* W_swa_out);

/* ---- the step before the path: mini-batch training on the device (SURVEY 8(f)-3) ----------------------------------
 * Replaces, for a Dense chain with cost = Flux.Losses.mse(m(x), y), the reference's training step
 *     gs = gradient(ps) do training_loss = cost(d...) end; Flux.update!(opt, ps, gs)     src/subspace_construction.jl:39-43
 * so that snapshots feed the SWA recurrence without a host round trip.  Needs ssi_set_model and ssi_set_data (the
 * DataLoader's full X, Y: src/libs.jl:75-77); weights are in the flat layout of src/libs.jl:19-22.
 *   ssi_train_begin      W0 (n floats, host) = Flux.params of the freshly built model; optimiser 0 = Descent(eta),
 *                        1 = ADAM(eta, (beta1, beta2)) with eps = 1e-8 (Flux 0.11.2 update rule)
 *   ssi_train_step       one mini-batch: columns idx[0..nb) of the data set (host indices, a shuffled DataLoader) or, with
 *                        idx == NULL, the contiguous columns [j0, j0 + nb).  loss_out (host, may be NULL) receives
 *                        training_loss, the mean squared error BEFORE the update; asking for it synchronises.
 *   ssi_train_snapshot   W_swa <- (ns W_swa + W)/(ns + 1), deviation column <- W - W_swa (:44-52) from the device weights;
 *                        ssi_swa_begin(n, K_max) must have been called with the model's n
 *   ssi_train_get_weights  copy the current weights to the host (n floats)                                            */
#define SSI_OPT_DESCENT 0
#define SSI_OPT_ADAM 1
int  ssi_train_begin(ssi_ctx* ctx, const float* W0, int32_t optimiser, double eta, double beta1, double beta2);
int  ssi_train_step(ssi_ctx* ctx, const int64_t* idx, int64_t j0, int64_t nb, double* loss_out);
int  ssi_train_snapshot(ssi_ctx* ctx, double n_scalar);
int  ssi_train_get_weights(ssi_ctx* ctx, float* W_out);
int  ssi_train_end(ssi_ctx* ctx);

/* Row-sharded construction over several GPUs (one process and one context per GPU): every rank pushes ITS ROW SHARD of
 * each snapshot (n = shard length), then
 *   ssi_swa_gram_dev    Gram of the local deviation columns into a caller-provided DEVICE buffer (K x K doubles,
 *                       column-major); exact != 0 forces the FP64 kernel.  The host all-reduces (sums) it across ranks
 *                       (ncclAllReduce / torch.distributed): the only collective of the construction path;
 *   ssi_swa_finish_gram replicated eigen-solve of the reduced Gram, then W_swa / P ROWS of the local shard (host
 *                       pointers, any NULL) and the K singular values.  Returns SSI_RETRY_EXACT (> 0) when
 *                       gram_exact == 0 and the conditioning check rejects a tensor-core Gram: every rank sees the same
 *                       spectrum, so every rank then repeats both calls with exact = gram_exact = 1.                   */
#define SSI_RETRY_EXACT 1
int  ssi_swa_gram_dev(ssi_ctx* ctx, double* dG_out, int32_t exact);
int  ssi_swa_finish_gram(ssi_ctx* ctx, int32_t M, const double* dG, int32_t gram_exact,
                         float* W_swa_out, float* P_out, double* s_out, int32_t install);

#ifdef __cplusplus
}
#endif
#endif /* SSI_H */
