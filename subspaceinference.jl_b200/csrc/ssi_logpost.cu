// ssi_logpost.cu — density(z) batched over B subspace points.
//
// Replaces the reference closure src/space_inference.jl:90-95 (new_W = W_swa + P*z;
// model_re; Chain forward on the full dataset; Gaussian log-likelihood).  Three device
// paths compute the per-sample sum of squared errors (SSE); a common finalize kernel
// turns SSE (+ the M-space prior terms) into log-probabilities:
//
//   FUSED    one CTA projects a sample's weights straight into shared memory and pushes
//            datapoints through the whole chain with activations in shared memory
//            (small networks: README 10-20-20-2, UCI 13-50-1).
//   LAYERED  weights of a group of samples are materialised, then one batched FP32 SIMT
//            GEMM per layer (ssi_launch_gemm_simt) with fused bias/activation, the last one
//            fused with the squared-error reduction (any shape; the exact FP32 cross-check
//            of the tensor path).
//   TENSOR   ssi_tc.cu (tcgen05 / TMEM / TMA).
//
// Reductions are two-stage and fixed-order (per-CTA partials -> finalize), so a
// sample's lp does not depend on how many other samples share the call.
#include "ssi_common.cuh"
#include "ssi_gemm.cuh"

#include <algorithm>
#include <cmath>

// ======================================================================================
// FUSED path
// ======================================================================================
#define FUSED_T 128   // datapoints per pass == threads per CTA

struct fused_desc_t {
    int L;
    int dims[SSI_MAX_LAYERS + 1];
    int act[SSI_MAX_LAYERS];
    int wsrc[SSI_MAX_LAYERS], bsrc[SSI_MAX_LAYERS];     // offsets in the flat parameter vector
    int wdst[SSI_MAX_LAYERS], bdst[SSI_MAX_LAYERS];     // offsets (floats) in shared memory, 16B aligned
    int out_pad[SSI_MAX_LAYERS];                        // out rounded up to 4
    int w_floats;                                       // padded weight floats in shared memory
    int max_width;
    int M;
    int n;
};

template <int OB>
__device__ __forceinline__ void fused_block(const float* __restrict__ Ws, const float* __restrict__ bs,
                                            const float* __restrict__ hin, int in, int out_pad, int o,
                                            float acc[OB]) {
    // acc[r] = b[o+r] + sum_i W[o+r, i] * h[i]; weights are [in][out_pad] so the OB outputs
    // of one input are one or two 16-byte broadcast loads.
#pragma unroll
    for (int r = 0; r < OB; r += 4) {
        const float4 b4 = *reinterpret_cast<const float4*>(bs + o + r);
        acc[r] = b4.x; acc[r + 1] = b4.y; acc[r + 2] = b4.z; acc[r + 3] = b4.w;
    }
    const float* wrow = Ws + o;
#pragma unroll 4
    for (int i = 0; i < in; ++i) {
        const float h = hin[i * FUSED_T];
#pragma unroll
        for (int r = 0; r < OB; r += 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(wrow + r);
            acc[r]     = fmaf(w4.x, h, acc[r]);
            acc[r + 1] = fmaf(w4.y, h, acc[r + 1]);
            acc[r + 2] = fmaf(w4.z, h, acc[r + 2]);
            acc[r + 3] = fmaf(w4.w, h, acc[r + 3]);
        }
        wrow += out_pad;
    }
}

__global__ void __launch_bounds__(FUSED_T)
k_logpost_fused(const fused_desc_t d, const float* __restrict__ X, const float* __restrict__ Y,
                const float* __restrict__ Wswa, const float* __restrict__ P, const float* __restrict__ Z,
                long long N, int chunk, int n_chunks, double* __restrict__ partials) {
    extern __shared__ float4 smem4[];
    float* Ws = reinterpret_cast<float*>(smem4);
    float* buf0 = Ws + d.w_floats;
    float* buf1 = buf0 + d.max_width * FUSED_T;
    __shared__ float zs[SSI_MAX_M];
    __shared__ double red[32];

    const int tid = threadIdx.x;
    const long long b = blockIdx.y;
    if (tid < d.M) zs[tid] = Z[tid + b * d.M];
    for (int e = tid; e < d.w_floats; e += FUSED_T) Ws[e] = 0.0f;
    __syncthreads();

    // K1: W = W_swa + P z, written in the padded [in][out_pad] layout  (src/space_inference.jl:91)
    for (int l = 0; l < d.L; ++l) {
        const int in = d.dims[l], out = d.dims[l + 1], op = d.out_pad[l];
        for (int e = tid; e < in * out; e += FUSED_T) {
            const int i = d.wsrc[l] + e;
            float v = Wswa[i];
            for (int m = 0; m < d.M; ++m) v = fmaf(P[i + (long long)m * d.n], zs[m], v);
            Ws[d.wdst[l] + (e / out) * op + (e % out)] = v;
        }
        for (int o = tid; o < out; o += FUSED_T) {
            const int i = d.bsrc[l] + o;
            float v = Wswa[i];
            for (int m = 0; m < d.M; ++m) v = fmaf(P[i + (long long)m * d.n], zs[m], v);
            Ws[d.bdst[l] + o] = v;
        }
    }
    __syncthreads();

    const int in0 = d.dims[0], O = d.dims[d.L];
    const long long j_begin = (long long)blockIdx.x * chunk;
    const long long j_end = min(N, j_begin + (long long)chunk);
    double sse = 0.0;

    for (long long j0 = j_begin; j0 < j_end; j0 += FUSED_T) {
        const int nvalid = (int)min((long long)FUSED_T, j_end - j0);
        // stage X[:, j0 : j0+nvalid] (contiguous in memory) into buf0[i][t]
        const float* xsrc = X + j0 * in0;
        for (int e = tid; e < nvalid * in0; e += FUSED_T) buf0[(e % in0) * FUSED_T + (e / in0)] = xsrc[e];
        __syncthreads();
        if (tid < nvalid) {
            float* hin = buf0 + tid;
            float* hout = buf1 + tid;
            for (int l = 0; l < d.L; ++l) {
                const int in = d.dims[l], out = d.dims[l + 1], op = d.out_pad[l], act = d.act[l];
                const bool last = (l == d.L - 1);
                const float* Wl = Ws + d.wdst[l];
                const float* bl = Ws + d.bdst[l];
                int o = 0;
                for (; o + 8 <= op; o += 8) {
                    float acc[8];
                    fused_block<8>(Wl, bl, hin, in, op, o, acc);
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        if (o + r < out) {
                            const float v = ssi_act(acc[r], act);
                            if (last) {
                                const float df = v - Y[(o + r) + (j0 + tid) * O];
                                sse += (double)df * (double)df;
                            } else {
                                hout[(o + r) * FUSED_T] = v;
                            }
                        }
                    }
                }
                for (; o < op; o += 4) {
                    float acc[4];
                    fused_block<4>(Wl, bl, hin, in, op, o, acc);
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        if (o + r < out) {
                            const float v = ssi_act(acc[r], act);
                            if (last) {
                                const float df = v - Y[(o + r) + (j0 + tid) * O];
                                sse += (double)df * (double)df;
                            } else {
                                hout[(o + r) * FUSED_T] = v;
                            }
                        }
                    }
                }
                float* t = hin; hin = hout; hout = t;
            }
        }
        __syncthreads();
    }
    const double tot = ssi_block_sum(sse, red);
    if (tid == 0) partials[b * n_chunks + blockIdx.x] = tot;
}

static bool fused_layout(const ssi_ctx* ctx, fused_desc_t& d, size_t& smem_bytes) {
    const ssi_model_t& m = ctx->model;
    if (m.n >= (1ll << 30)) return false;
    d.L = m.L;
    int off = 0;
    for (int l = 0; l <= m.L; ++l) d.dims[l] = m.dims[l];
    for (int l = 0; l < m.L; ++l) {
        d.act[l] = m.act[l];
        d.wsrc[l] = (int)m.w_off[l];
        d.bsrc[l] = (int)m.b_off[l];
        d.out_pad[l] = (m.dims[l + 1] + 3) & ~3;
        d.wdst[l] = off;
        off += m.dims[l] * d.out_pad[l];
        d.bdst[l] = off;
        off += d.out_pad[l];
    }
    d.w_floats = off;
    d.max_width = m.max_width;
    d.M = ctx->M;
    d.n = (int)m.n;
    smem_bytes = ((size_t)d.w_floats + 2 * (size_t)d.max_width * FUSED_T) * sizeof(float);
    return true;
}

static int fused_chunking(int64_t N, int& chunk, int& n_chunks) {
    // depends on N only, so that a sample's summation order is the same in every call
    const int64_t passes = (N + FUSED_T - 1) / FUSED_T;
    const int64_t per = (passes + 63) / 64;   // at most 64 chunks per sample
    chunk = (int)(per * FUSED_T);
    n_chunks = (int)((N + chunk - 1) / chunk);
    return SSI_OK;
}

static int run_fused(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse) {
    fused_desc_t d{};
    size_t smem = 0;
    if (!fused_layout(ctx, d, smem)) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "model too large for the fused path");
    int chunk, n_chunks;
    fused_chunking(ctx->N, chunk, n_chunks);
    SSI_TRY(ssi_reserve(ctx, ctx->bPartials, sizeof(double) * (size_t)B * n_chunks));
    SSI_CUDA(ctx, cudaFuncSetAttribute(k_logpost_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    double* partials = (double*)ctx->bPartials.p;
    // grid.y is limited to 65535: slice the batch
    for (int64_t b0 = 0; b0 < B; b0 += 65535) {
        const int64_t nb = std::min<int64_t>(65535, B - b0);
        dim3 grid(n_chunks, (unsigned)nb);
        ssi_kt_begin(ctx);
        k_logpost_fused<<<grid, FUSED_T, smem, ctx->stream>>>(d, ctx->dX, ctx->dY, ctx->dWswa, ctx->dP,
                                                             dZ + b0 * ctx->M, ctx->N, chunk, n_chunks,
                                                             partials + b0 * n_chunks);
        SSI_LAUNCH_CHECK(ctx);
        ssi_kt_end(ctx);
    }
    extern int ssi_reduce_partials(ssi_ctx*, const double*, int64_t, int, double*);
    return ssi_reduce_partials(ctx, partials, B, n_chunks, d_sse);
}

// ======================================================================================
// partial reduction + finalize
// ======================================================================================
__global__ void k_reduce_partials(const double* __restrict__ partials, long long B, int parts,
                                  double* __restrict__ out) {
    // one warp per sample, fixed order: lane-strided then butterfly
    const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const int lane = threadIdx.x & 31;
    double s = 0.0;
    for (int p = lane; p < parts; p += 32) s += partials[b * parts + p];
    s = ssi_warp_sum(s);
    if (lane == 0) out[b] = s;
}

int ssi_reduce_partials(ssi_ctx* ctx, const double* partials, int64_t B, int parts, double* d_out) {
    const int warps = 8;
    k_reduce_partials<<<(unsigned)((B + warps - 1) / warps), warps * 32, 0, ctx->stream>>>(partials, B, parts, d_out);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}

struct finalize_args_t {
    double c_ll, inv2sm2;      // ll = c_ll - sse * inv2sm2
    double c_w, inv2sp2;       // prior_w = c_w - |W|^2 * inv2sp2
    double c_z, inv2sz2;       // prior_z = c_z - |z|^2 * inv2sz2
    uint32_t mask;
    int M;
};

__global__ void k_finalize(const finalize_args_t a, const double* __restrict__ sse, const float* __restrict__ Z,
                           const double* __restrict__ G /* (M+1)x(M+1) */, long long B,
                           double* __restrict__ lp, double* __restrict__ terms) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int M = a.M, ld = M + 1;
    // |W_swa + P z|^2 = w'w + 2 (P'w)'z + z'(P'P)z, from the Gram of [P | W_swa]; skipped when only the likelihood is asked
    // for (the reference's density as executed): the M^2 FP64 loop was most of this kernel's time in the MH loop
    double w2 = 0.0, z2 = 0.0;
    if (terms || (a.mask & (SSI_TERM_PRIOR_W | SSI_TERM_PRIOR_Z))) {
        w2 = G[M * ld + M];
        for (int i = 0; i < M; ++i) {
            const double zi = (double)Z[i + b * M];
            z2 += zi * zi;
            double row = 0.0;
            for (int j = 0; j < M; ++j) row += G[i * ld + j] * (double)Z[j + b * M];
            w2 += zi * (row + 2.0 * G[i * ld + M]);
        }
    }
    const double ll = a.c_ll - sse[b] * a.inv2sm2;
    const double pw = a.c_w - w2 * a.inv2sp2;
    const double pz = a.c_z - z2 * a.inv2sz2;
    double v = 0.0;
    if (a.mask & SSI_TERM_LL) v += ll;
    if (a.mask & SSI_TERM_PRIOR_W) v += pw;
    if (a.mask & SSI_TERM_PRIOR_Z) v += pz;
    lp[b] = v;
    if (terms) { terms[3 * b] = ll; terms[3 * b + 1] = pw; terms[3 * b + 2] = pz; }
}

// ======================================================================================
// LAYERED path
// ======================================================================================
// W[g][i] = W_swa[i] + sum_m P[i,m] z[m,g]      (src/space_inference.jl:91; K1)
// With a decoder whose head is not affine (ssi_decoder.cu): W = Wbase + act(W_swa' + P z), W_swa' being the head's bias.
__global__ void __launch_bounds__(256)
k_project(const float* __restrict__ Wswa, const float* __restrict__ P, const float* __restrict__ Z,
          long long n, int M, int G, float* __restrict__ W /* G x ldw (sample-major) or ldw x G col-major: same */,
          const float* __restrict__ Wbase, int act, long long ldw) {
    extern __shared__ float zs[];   // M x G
    for (int e = threadIdx.x; e < M * G; e += blockDim.x) zs[e] = Z[e];
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float p[SSI_MAX_M];
#pragma unroll 4
    for (int m = 0; m < M; ++m) p[m] = P[i + (long long)m * n];
    const float w0 = Wswa[i];
    const float wb = Wbase ? Wbase[i] : 0.0f;
    for (int g = 0; g < G; ++g) {
        float v = w0;
        for (int m = 0; m < M; ++m) v = fmaf(p[m], zs[m + g * M], v);
        W[i + (long long)g * ldw] = Wbase ? wb + ssi_act(v, act) : v;
    }
}

int ssi_project_device(ssi_ctx* ctx, const float* dZ, int64_t B, float* dW, int64_t ldw) {
    const int64_t n = ctx->model.n;
    if (ldw <= 0) ldw = n;
    const int M = ctx->M;
    const int gmax = std::max(1, (int)(32768 / (sizeof(float) * M)));
    for (int64_t b0 = 0; b0 < B; b0 += gmax) {
        const int G = (int)std::min<int64_t>(gmax, B - b0);
        k_project<<<(unsigned)((n + 255) / 256), 256, sizeof(float) * M * G, ctx->stream>>>(
            ctx->dWswa, ctx->dP, dZ + b0 * M, n, M, G, dW + b0 * ldw, ctx->dWbase, ctx->dec_out_act, ldw);
        SSI_LAUNCH_CHECK(ctx);
    }
    return SSI_OK;
}

static int run_layered(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse) {
    const ssi_model_t& m = ctx->model;
    const int64_t N = ctx->N, n = m.n;
    if (N >= (1ll << 31)) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "LAYERED path: N must fit 31 bits");
    // group size: bounded by scratch (two activation buffers of max hidden width)
    int hid = 1;
    for (int l = 1; l < m.L; ++l) hid = std::max(hid, m.dims[l]);
    const double per_sample = 2.0 * hid * (double)N * sizeof(float) + (double)n * sizeof(float);
    int G = ctx->opt_group > 0 ? ctx->opt_group : (int)std::max(1.0, std::min(64.0, 4e9 / per_sample));
    G = (int)std::min<int64_t>(G, B);
    SSI_TRY(ssi_reserve(ctx, ctx->bW, sizeof(float) * (size_t)n * G));
    if (m.L > 1) {
        SSI_TRY(ssi_reserve(ctx, ctx->bH0, sizeof(float) * (size_t)hid * N * G));
        if (m.L > 2) SSI_TRY(ssi_reserve(ctx, ctx->bH1, sizeof(float) * (size_t)hid * N * G));
    }
    const int O = m.dims[m.L];
    const int parts = (int)((N + GT_T - 1) / GT_T) * ((O + GT_T - 1) / GT_T);      // one per tile of the last layer
    SSI_TRY(ssi_reserve(ctx, ctx->bPartials, sizeof(double) * (size_t)B * parts));
    float* dW = (float*)ctx->bW.p;
    float* hbuf[2] = {(float*)ctx->bH0.p, (float*)ctx->bH1.p};
    double* partials = (double*)ctx->bPartials.p;

    for (int64_t b0 = 0; b0 < B; b0 += G) {
        const int g = (int)std::min<int64_t>(G, B - b0);
        SSI_TRY(ssi_project_device(ctx, dZ + b0 * ctx->M, g, dW));
        const float* hin = ctx->dX;
        long long hin_bs = 0;
        for (int l = 0; l < m.L; ++l) {
            const int out = m.dims[l + 1];
            if (l == m.L - 1) {         // the squared error against Y instead of the output
                SSI_TRY(ssi_launch_gemm_simt(ctx, ssi_dense_gemm(m, l, dW, n, hin, hin_bs, nullptr, out, 0, (int)N), g, false, false,
                                             ctx->dY, partials + b0 * parts));
            } else {
                float* hout = hbuf[l & 1];
                SSI_TRY(ssi_launch_gemm_simt(ctx, ssi_dense_gemm(m, l, dW, n, hin, hin_bs, hout, out, (long long)out * N, (int)N), g,
                                             false, false));
                hin = hout;
                hin_bs = (long long)out * N;
            }
        }
    }
    return ssi_reduce_partials(ctx, partials, B, parts, d_sse);
}

// ======================================================================================
// posterior-predictive sweep (the step after the path in every docs example)
// ======================================================================================
// Replaces, for B subspace samples at once, the user loop of docs/src/nn_example.md:207-216
//     for i in 1:itr;  m1 = re(all_chain[i]);  trajectories[:, i] = m1(inp)';  end
// and the moments plot_predictive takes of it (src/plotting.jl:8-9): mean(trajectories, dims=2) and
// std(trajectories, dims=2) (Julia's corrected estimator, B-1).  The itr x n weight vectors are never materialised on
// the host; predictions are folded into running (count, mean, M2) per grid point group by group (Chan's merge).
__global__ void __launch_bounds__(256)
k_pred_moments(const float* __restrict__ preds /* [G][ON] */, int G, long long ON, long long cnt_prev,
               double* __restrict__ mean, double* __restrict__ m2) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ON) return;
    double gm = 0.0;
    for (int g = 0; g < G; ++g) gm += (double)preds[(long long)g * ON + e];
    gm /= (double)G;
    double gm2 = 0.0;
    for (int g = 0; g < G; ++g) {
        const double d = (double)preds[(long long)g * ON + e] - gm;
        gm2 += d * d;
    }
    if (cnt_prev == 0) {
        mean[e] = gm;
        m2[e] = gm2;
    } else {
        const double tot = (double)(cnt_prev + G);
        const double delta = gm - mean[e];
        mean[e] += delta * (double)G / tot;
        m2[e] += gm2 + delta * delta * (double)cnt_prev * (double)G / tot;
    }
}

__global__ void k_pred_std(const double* __restrict__ m2, long long ON, long long B, double* __restrict__ sd) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ON) return;
    sd[e] = B > 1 ? sqrt(m2[e] / (double)(B - 1)) : nan("");      // std of one trajectory is NaN in Julia (0/0)
}

// dZ (M x B), dXg (in0 x Ng) device; d_preds (O x Ng x B) optional; d_mean, d_std (O x Ng doubles); d_m2 scratch (O x Ng)
int ssi_predict_device(ssi_ctx* ctx, const float* dZ, int64_t B, const float* dXg, int64_t Ng,
                       float* d_preds, double* d_mean, double* d_std, double* d_m2) {
    if (Ng >= (1ll << 31)) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "predictive sweep: Ng must fit 31 bits");
    if (ctx->dec_active) SSI_TRY(ssi_dec_project(ctx, dZ, B, &dZ));       // W = W_swa + decoder(z): continue with z' = h(z)
    const ssi_model_t& m = ctx->model;
    const int64_t n = m.n;
    const int O = m.dims[m.L];
    const long long ON = (long long)O * Ng;
    int hid = 1;
    for (int l = 1; l < m.L; ++l) hid = std::max(hid, m.dims[l]);
    const double per_sample = (2.0 * hid + O) * (double)Ng * sizeof(float) + (double)n * sizeof(float);
    int G = (int)std::max(1.0, std::min(64.0, 2e9 / per_sample));
    G = (int)std::min<int64_t>(G, B);
    SSI_TRY(ssi_reserve(ctx, ctx->bW, sizeof(float) * (size_t)n * G));
    if (m.L > 1) {
        SSI_TRY(ssi_reserve(ctx, ctx->bH0, sizeof(float) * (size_t)hid * Ng * G));
        if (m.L > 2) SSI_TRY(ssi_reserve(ctx, ctx->bH1, sizeof(float) * (size_t)hid * Ng * G));
    }
    SSI_TRY(ssi_reserve(ctx, ctx->bPartials, sizeof(float) * (size_t)ON * G));
    float* dW = (float*)ctx->bW.p;
    float* hbuf[2] = {(float*)ctx->bH0.p, (float*)ctx->bH1.p};
    float* pg = (float*)ctx->bPartials.p;
    for (int64_t b0 = 0; b0 < B; b0 += G) {
        const int g = (int)std::min<int64_t>(G, B - b0);
        SSI_TRY(ssi_project_device(ctx, dZ + b0 * ctx->M, g, dW));
        const float* hin = dXg;
        long long hin_bs = 0;
        for (int l = 0; l < m.L; ++l) {
            const int out = m.dims[l + 1];
            float* hout = l == m.L - 1 ? pg : hbuf[l & 1];
            SSI_TRY(ssi_launch_gemm_simt(ctx, ssi_dense_gemm(m, l, dW, n, hin, hin_bs, hout, out, (long long)out * Ng, (int)Ng), g,
                                         false, false));
            hin = hout;
            hin_bs = (long long)out * Ng;
        }
        k_pred_moments<<<(unsigned)((ON + 255) / 256), 256, 0, ctx->stream>>>(pg, g, ON, b0, d_mean, d_m2);
        SSI_LAUNCH_CHECK(ctx);
        if (d_preds)
            SSI_CUDA(ctx, cudaMemcpyAsync(d_preds + b0 * ON, pg, sizeof(float) * (size_t)ON * g, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    k_pred_std<<<(unsigned)((ON + 255) / 256), 256, 0, ctx->stream>>>(d_m2, ON, B, d_std);
    SSI_LAUNCH_CHECK(ctx);
    ctx->stats.last_units = (double)B * (double)Ng;
    ctx->stats.last_flops = (double)B * ((double)Ng * m.flops_per_point + 2.0 * (double)n * ctx->M);
    ctx->stats.last_bytes = 0;
    return SSI_OK;
}

// First-layer bases for the tensor path: B_m = (column m of [P | W_swa])_layer0 applied to X, m = 0..M,
// as FP32 pre-activations [m][N][ld] (bias parts included).  Exact FP32 SIMT GEMM, run once per (data, subspace).
int ssi_build_first_layer_bases(ssi_ctx* ctx, float* bases, int ld) {
    const int64_t N = ctx->N;
    if (N >= (1ll << 31)) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "tensor path bases: N must fit 31 bits");
    gemm_t q = ssi_dense_gemm(ctx->model, 0, ctx->dP, ctx->model.n, ctx->dX, 0, bases, ld, N * ld, (int)N);
    q.act = SSI_ACT_IDENTITY;
    return ssi_launch_gemm_simt(ctx, q, ctx->M + 1, false, false);
}

// SSE (+ the M-space prior terms) -> log-probabilities: the closed form of logpdf(MvNormal(vec(pred), sigma_m), vec(Y))
int ssi_logpost_finalize(ssi_ctx* ctx, const double* d_sse, const float* dZ, int64_t B, double sigma_m, double sigma_p,
                         double sigma_z, uint32_t mask, double* d_lp, double* d_terms) {
    const ssi_model_t& m = ctx->model;
    const double LOG_2PI = 1.8378770664093454835606594728112;
    const double k = (double)m.dims[m.L] * (double)ctx->N;
    finalize_args_t a;
    a.c_ll = -0.5 * k * LOG_2PI - k * std::log(sigma_m);
    a.inv2sm2 = 1.0 / (2.0 * sigma_m * sigma_m);
    a.c_w = -0.5 * (double)m.n * LOG_2PI - (double)m.n * std::log(sigma_p);
    a.inv2sp2 = 1.0 / (2.0 * sigma_p * sigma_p);
    a.c_z = -0.5 * (double)ctx->M * LOG_2PI - (double)ctx->M * std::log(sigma_z);
    a.inv2sz2 = 1.0 / (2.0 * sigma_z * sigma_z);
    a.mask = mask;
    a.M = ctx->M;
    k_finalize<<<(unsigned)((B + 127) / 128), 128, 0, ctx->stream>>>(a, d_sse, dZ, ctx->dSubGram, B, d_lp, d_terms);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}

// ======================================================================================
// dispatch
// ======================================================================================
static int choose_path(ssi_ctx* ctx) {
    if (ctx->dWbase) return SSI_PATH_LAYERED;       // non-affine decoder head: the weights are materialised per sample
    if (ctx->opt_path != SSI_PATH_AUTO) return ctx->opt_path;
    if (ssi_tc_preferred(ctx)) return SSI_PATH_TENSOR;
    if (ssi_bm_supported(ctx) || ssi_b1_supported(ctx)) return SSI_PATH_BASIS;
    fused_desc_t d{};
    size_t smem = 0;
    if (fused_layout(ctx, d, smem) && smem <= 100 * 1024) return SSI_PATH_FUSED;
    return SSI_PATH_LAYERED;
}

int ssi_logpost_device(ssi_ctx* ctx, const float* dZ, int64_t B, double sigma_m, double sigma_p,
                       double sigma_z, uint32_t mask, double* d_lp, double* d_terms) {
    if (!ctx->has_model || !ctx->has_data || !ctx->has_sub)
        return ssi_fail(ctx, SSI_ERR_STATE, "model, data and subspace must be set before evaluating the log-posterior");
    if (B <= 0) return SSI_OK;
    if (ctx->dec_active) return ssi_dec_logpost(ctx, dZ, B, sigma_m, sigma_p, sigma_z, mask, d_lp, d_terms);
    if (!(sigma_m > 0) || !(sigma_p > 0) || !(sigma_z > 0))
        return ssi_fail(ctx, SSI_ERR_ARG, "sigma_m, sigma_p, sigma_z must be positive");
    if ((mask & ~(SSI_TERM_LL | SSI_TERM_PRIOR_W | SSI_TERM_PRIOR_Z)) || mask == 0)
        return ssi_fail(ctx, SSI_ERR_ARG, "prior_mask must be a non-empty OR of SSI_TERM_*");
    SSI_TRY(ssi_reserve(ctx, ctx->bMisc, sizeof(double) * (size_t)B));
    double* d_sse = (double*)ctx->bMisc.p;

    const int path = choose_path(ctx);
    int rc;
    if (path == SSI_PATH_TENSOR) {
        if (!ssi_tc_supported(ctx)) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "tensor path does not support this model shape");
        rc = ssi_tc_sse(ctx, dZ, B, d_sse);
    } else if (path == SSI_PATH_BASIS) {
        // scalar output, H <= 64, M + 1 <= 32: samples along the MMA M dimension (ssi_basis_mma.cu); else CUDA cores
        if (ssi_bm_supported(ctx)) rc = ssi_bm_sse(ctx, dZ, B, d_sse);
        else if (ssi_b1_supported(ctx)) rc = ssi_b1_sse(ctx, dZ, B, d_sse);
        else return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "basis path needs Chain(Dense, Dense) with O = 1, H <= 64, M <= 31 (tensor cores) or "
                                                       "O <= 2, M in {1..8, 10, 12, 16, 20} and a basis tile that fits shared memory (CUDA cores)");
    } else if (path == SSI_PATH_FUSED) {
        fused_desc_t d{};
        size_t smem = 0;
        if (!fused_layout(ctx, d, smem) || smem > ctx->smem_optin)
            return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "fused path needs %zu bytes of shared memory (limit %zu)", smem, ctx->smem_optin);
        rc = run_fused(ctx, dZ, B, d_sse);
    } else if (path == SSI_PATH_LAYERED) {
        rc = run_layered(ctx, dZ, B, d_sse);
    } else {
        return ssi_fail(ctx, SSI_ERR_ARG, "unknown path %d", path);
    }
    if (rc != SSI_OK) return rc;
    ctx->stats.last_path = path;

    SSI_TRY(ssi_logpost_finalize(ctx, d_sse, dZ, B, sigma_m, sigma_p, sigma_z, mask, d_lp, d_terms));
    const ssi_model_t& m = ctx->model;
    ctx->stats.last_units = (double)B * (double)ctx->N;
    ctx->stats.last_flops = (double)B * ((double)ctx->N * m.flops_per_point + 2.0 * (double)m.n * ctx->M);
    ctx->stats.last_bytes = 0;
    return SSI_OK;
}
