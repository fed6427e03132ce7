// ssi_grad.cu — value and gradient of the subspace log-posterior, batched over B subspace points.
//
// Replaces the reference's gradient closure  l_pi_grad(theta) = (density(theta), backend.gradient(density, theta))
// (src/space_inference.jl:107; backends src/libs.jl:23-34: ForwardDiff by default, i.e. M dual-number forward passes
// per gradient) that feeds the :mala, :hmc and :nuts samplers (:117-120, :139-160).  Here one reverse pass per sample:
//
//     W = W_swa + P z                      k_project                                  (K1)
//     H_l = act_l(W_l H_{l-1} + b_l)       k_gemm_simt, all activations kept
//     delta_L = -(pred - y)/sigma_m^2 * act_L'(pred)        (+ the squared error for lp)
//     gW_l = delta_l H_{l-1}',  gb_l = rowsum(delta_l),  delta_{l-1} = (W_l' delta_l) * act_{l-1}'(H_{l-1})
//     grad_z = P' [gW ; gb]  (+ prior terms evaluated in M-space)
//
// Every contraction is one launch of the same strided FP32 SIMT GEMM (64x64 tile, 4x4 per thread); reductions are
// two-stage with a fixed order, so a sample's gradient does not depend on the rest of the batch.  FP32 storage, FP64
// final accumulation of the squared error.  This is the correctness-first version of SURVEY 8(f)-1: any Dense chain,
// CUDA cores only.
#include "ssi_common.cuh"
#include "ssi_gemm.cuh"

#include <algorithm>
#include <cmath>

#define GT_T 64
#define GT_K 16
#define GT_LD 68          // padded tile rows: float4 aligned, transposed fills spread over the banks

template <bool A_KFAST, bool B_JFAST>
__global__ void __launch_bounds__(256)
k_gemm_simt(const gemm_t p) {
    __shared__ __align__(16) float As[GT_K][GT_LD];
    __shared__ __align__(16) float Bs[GT_K][GT_LD];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int o0 = blockIdx.y * GT_T, j0 = blockIdx.x * GT_T;
    const long long b = blockIdx.z;
    long long k_begin = 0, k_end = p.K;
    if (p.split > 0) { k_begin = b * p.split; k_end = min(p.K, k_begin + p.split); }
    const float* A = p.A + (p.split > 0 ? 0 : b * p.a_sb);
    const float* Bm = p.B + (p.split > 0 ? 0 : b * p.b_sb);

    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0.0f;

    for (long long k0 = k_begin; k0 < k_end; k0 += GT_K) {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const int idx = tid + s * 256;
            const int o = A_KFAST ? (idx >> 4) : (idx & (GT_T - 1));
            const int k = A_KFAST ? (idx & (GT_K - 1)) : (idx >> 6);
            As[k][o] = (o0 + o < p.O && k0 + k < k_end) ? A[(long long)(o0 + o) * p.a_so + (k0 + k) * p.a_sk] : 0.0f;
        }
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const int idx = tid + s * 256;
            const int j = B_JFAST ? (idx & (GT_T - 1)) : (idx >> 4);
            const int k = B_JFAST ? (idx >> 6) : (idx & (GT_K - 1));
            Bs[k][j] = (j0 + j < p.J && k0 + k < k_end) ? Bm[(k0 + k) * p.b_sk + (long long)(j0 + j) * p.b_sj] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GT_K; ++k) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[k][tx * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][ty * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w};
            const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(a[r], bb[c], acc[r][c]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int j = j0 + ty * 4 + c;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int o = o0 + tx * 4 + r;
            if (o < p.O && j < p.J) {
                float v = acc[r][c];
                const long long ci = (long long)o * p.c_so + (long long)j * p.c_sj;
                if (p.epi == 1) v = ssi_act(v + p.bias[b * p.bias_sb + o], p.act);
                else if (p.epi == 2) v *= act_deriv_from_output(p.Hprev[b * p.h_sb + ci], p.act);
                p.C[b * p.c_sb + ci] = v;
            }
        }
    }
}

// ---- skinny shapes: the output layer of a regression / classification head has O <= 16 rows, which neither the 64x64 SIMT
// tile nor the 128-row tensor-core tile fits (and a leading dimension of 10 floats is not TMA-addressable).  Three
// memory-bound kernels, one per orientation the reverse pass produces; all sums in a fixed order.
#define SK_MAXO 16
// (1) forward, O <= 16: C(o, j) = epi(sum_k A(o, k) B(k, j)), A o-fast (W_L), B k-fast (H_{L-1}).  A warp takes four datapoints j
// at a time, lanes over k (coalesced), A transposed into shared memory as [o][K]: one shared-memory read of A serves four
// datapoints (with one it was the shared-memory pipe, not HBM, that set the pace).
template <int OO>
__global__ void __launch_bounds__(256)
k_gemm_skinny_fwd(const gemm_t p, int J_per_block) {
    extern __shared__ float sk_As[];          // [OO][K]
    const long long b = blockIdx.y;
    const int K = (int)p.K;
    const float* A = p.A + b * p.a_sb;
    for (int e = threadIdx.x; e < p.O * K; e += blockDim.x) {
        const int o = e % p.O, k = e / p.O;
        sk_As[o * K + k] = A[o + (long long)k * p.a_sk];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* Bm = p.B + b * p.b_sb;
    const int j_begin = blockIdx.x * J_per_block, j_end = min(p.J, j_begin + J_per_block);
    for (int j0 = j_begin + 4 * warp; j0 < j_end; j0 += 32) {
        const float* col[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) col[c] = Bm + (long long)min(j0 + c, j_end - 1) * p.b_sj;
        float acc[4][OO];
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int o = 0; o < OO; ++o) acc[c][o] = 0.0f;
        // four k-steps (sixteen independent loads) in flight per lane: the loop is bound by DRAM latency otherwise
        for (int k = lane; k < K; k += 128) {
            float h[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int c = 0; c < 4; ++c) h[u][c] = (k + 32 * u < K) ? col[c][k + 32 * u] : 0.0f;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (k + 32 * u < K) {
#pragma unroll
                    for (int o = 0; o < OO; ++o)
                        if (o < p.O) {
                            const float w = sk_As[o * K + k + 32 * u];
#pragma unroll
                            for (int c = 0; c < 4; ++c) acc[c][o] = fmaf(w, h[u][c], acc[c][o]);
                        }
                }
            }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int o = 0; o < OO; ++o) {
                if (o < p.O) {                       // warp-uniform
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) acc[c][o] += __shfl_xor_sync(0xffffffffu, acc[c][o], d);
                }
            }
        if (lane < 4 && j0 + lane < j_end) {
            const int j = j0 + lane;
#pragma unroll
            for (int o = 0; o < OO; ++o)
                if (o < p.O) {
                    float v = lane == 0 ? acc[0][o] : lane == 1 ? acc[1][o] : lane == 2 ? acc[2][o] : acc[3][o];
                    const long long ci = o + (long long)j * p.c_sj;
                    if (p.epi == 1) v = ssi_act(v + p.bias[b * p.bias_sb + o], p.act);
                    else if (p.epi == 2) v *= act_deriv_from_output(p.Hprev[b * p.h_sb + ci], p.act);
                    p.C[b * p.c_sb + ci] = v;
                }
        }
    }
}
// (2) back-propagated delta through the head, K <= 16: C(o, j) = epi(sum_k A(o, k) B(k, j)), A k-fast (W_L read as (i, o)),
// B k-fast (delta_L).  A thread per o (coalesced along o), its row of A in registers; the block's slice of B sits in shared
// memory, padded to KK per datapoint, and is read with broadcast 16-byte loads.
template <int KK>
__global__ void __launch_bounds__(256)
k_gemm_skinny_k(const gemm_t p, int J_per_block) {
    extern __shared__ __align__(16) float sk_Bs[];     // [J_per_block][KK]
    const long long b = blockIdx.z;
    const int o = blockIdx.x * 256 + threadIdx.x;
    const int K = (int)p.K;
    const float* Bm = p.B + b * p.b_sb;
    const int j_begin = blockIdx.y * J_per_block, j_end = min(p.J, j_begin + J_per_block);
    for (int e = threadIdx.x; e < (j_end - j_begin) * KK; e += 256) {
        const int k = e % KK, jj = e / KK;
        sk_Bs[e] = k < K ? Bm[(long long)(j_begin + jj) * p.b_sj + k] : 0.0f;
    }
    float a[KK];
#pragma unroll
    for (int k = 0; k < KK; ++k) a[k] = (o < p.O && k < K) ? p.A[b * p.a_sb + (long long)o * p.a_so + k] : 0.0f;
    __syncthreads();
    if (o >= p.O) return;
    // eight datapoints per pass, the layer outputs they need requested before the first use
    for (int j0 = j_begin; j0 < j_end; j0 += 8) {
        float hp[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            hp[u] = (p.epi == 2 && j0 + u < j_end) ? p.Hprev[b * p.h_sb + o + (long long)(j0 + u) * p.c_sj] : 0.0f;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u;
            if (j < j_end) {
                const float4* col = reinterpret_cast<const float4*>(sk_Bs + (j - j_begin) * KK);
                float v = 0.0f;
#pragma unroll
                for (int k4 = 0; k4 < KK / 4; ++k4) {
                    const float4 d = col[k4];
                    v = fmaf(a[4 * k4], d.x, v); v = fmaf(a[4 * k4 + 1], d.y, v); v = fmaf(a[4 * k4 + 2], d.z, v); v = fmaf(a[4 * k4 + 3], d.w, v);
                }
                if (p.epi == 1) v = ssi_act(v + p.bias[b * p.bias_sb + o], p.act);
                else if (p.epi == 2) v *= act_deriv_from_output(hp[u], p.act);
                p.C[b * p.c_sb + o + (long long)j * p.c_sj] = v;
            }
        }
    }
}
// (3) weight gradient of the head, O <= 16 and a long contraction: C(o, j) = sum_k A(o, k) B(k, j), A o-fast (delta_L), B j-fast
// (H_{L-1}).  A thread per j (coalesced along j), O accumulators; A is staged through shared memory 64 k at a time (padded
// to OO per k, broadcast 16-byte loads); the contraction is cut into SK_SLICES slices whose partials the second kernel adds
// in order.
#define SK_SLICES 32
#define SK_KC 64
template <int OO>
__global__ void __launch_bounds__(256)
k_gemm_skinny_gw(const gemm_t p, float* __restrict__ part /* [batch][slice][O][J] */) {
    __shared__ __align__(16) float As[SK_KC * OO];
    const long long b = blockIdx.z;
    const int j = blockIdx.x * 256 + threadIdx.x;
    const int slice = blockIdx.y;
    const long long per = (p.K + SK_SLICES - 1) / SK_SLICES;
    const long long k0 = slice * per, k1 = min(p.K, k0 + per);
    const float* A = p.A + b * p.a_sb;
    const float* Bm = p.B + b * p.b_sb + min(j, p.J - 1);
    float acc[OO];
#pragma unroll
    for (int o = 0; o < OO; ++o) acc[o] = 0.0f;
    for (long long kc = k0; kc < k1; kc += SK_KC) {
        const int nk = (int)min((long long)SK_KC, k1 - kc);
        __syncthreads();
        for (int e = threadIdx.x; e < SK_KC * OO; e += 256) {
            const int o = e % OO, kk = e / OO;
            As[e] = (o < p.O && kk < nk) ? A[(kc + kk) * p.a_sk + o] : 0.0f;
        }
        __syncthreads();
        for (int kk = 0; kk < nk; kk += 8) {
            float h[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) h[u] = (kk + u < nk) ? Bm[(kc + kk + u) * p.b_sk] : 0.0f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const float4* d4 = reinterpret_cast<const float4*>(As + (kk + u) * OO);      // rows past nk are zero
#pragma unroll
                for (int o4 = 0; o4 < OO / 4; ++o4) {
                    const float4 d = d4[o4];
                    acc[4 * o4] = fmaf(d.x, h[u], acc[4 * o4]); acc[4 * o4 + 1] = fmaf(d.y, h[u], acc[4 * o4 + 1]);
                    acc[4 * o4 + 2] = fmaf(d.z, h[u], acc[4 * o4 + 2]); acc[4 * o4 + 3] = fmaf(d.w, h[u], acc[4 * o4 + 3]);
                }
            }
        }
    }
    if (j >= p.J) return;
    float* dst = part + ((b * SK_SLICES + slice) * p.O) * (long long)p.J + j;
#pragma unroll
    for (int o = 0; o < OO; ++o)
        if (o < p.O) dst[(long long)o * p.J] = acc[o];
}
__global__ void k_gemm_skinny_gw_fin(const gemm_t p, const float* __restrict__ part) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int o = blockIdx.y;
    const long long b = blockIdx.z;
    if (j >= p.J) return;
    float t = 0.0f;
    for (int s = 0; s < SK_SLICES; ++s) t += part[((b * SK_SLICES + s) * p.O + o) * (long long)p.J + j];
    p.C[b * p.c_sb + o + (long long)j * p.c_sj] = t;
}

// Takes g when it is one of the three skinny shapes (*used = true).
static int gemm_skinny_try(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast, bool* used) {
    *used = false;
    if (ctx->opt_gemm_simt || g.split > 0 || g.c_so != 1 || batches < 1 || batches > 65535) return SSI_OK;
    if (g.K >= (1ll << 31) || (double)g.O * g.J * (double)g.K < 1e6) return SSI_OK;      // per batch: the choice must not depend on the batch size
    if (!a_kfast && !b_jfast && g.a_so == 1 && g.b_sk == 1 && g.O <= SK_MAXO && g.J >= 1024 && (size_t)g.O * g.K * 4 <= 160 * 1024) {
        const int jpb = 256;
        dim3 grid((g.J + jpb - 1) / jpb, batches);
        const size_t sm = sizeof(float) * (size_t)g.O * g.K;
        if (g.O <= 4) {
            if (sm > 48 * 1024) SSI_CUDA(ctx, cudaFuncSetAttribute(k_gemm_skinny_fwd<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            k_gemm_skinny_fwd<4><<<grid, 256, sm, ctx->stream>>>(g, jpb);
        } else {
            if (sm > 48 * 1024) SSI_CUDA(ctx, cudaFuncSetAttribute(k_gemm_skinny_fwd<SK_MAXO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            k_gemm_skinny_fwd<SK_MAXO><<<grid, 256, sm, ctx->stream>>>(g, jpb);
        }
        SSI_LAUNCH_CHECK(ctx);
        *used = true;
    } else if (a_kfast && !b_jfast && g.a_sk == 1 && g.b_sk == 1 && g.K <= SK_MAXO && g.O >= 64 && g.J >= 64) {
        const int jpb = 64;
        dim3 grid((g.O + 255) / 256, (g.J + jpb - 1) / jpb, batches);
        if (grid.y > 65535) return SSI_OK;
        if (g.K <= 4) k_gemm_skinny_k<4><<<grid, 256, sizeof(float) * jpb * 4, ctx->stream>>>(g, jpb);
        else k_gemm_skinny_k<SK_MAXO><<<grid, 256, sizeof(float) * jpb * SK_MAXO, ctx->stream>>>(g, jpb);
        SSI_LAUNCH_CHECK(ctx);
        *used = true;
    } else if (!a_kfast && b_jfast && g.a_so == 1 && g.b_sj == 1 && g.O <= SK_MAXO && g.J >= 64 && g.K >= 1024) {
        SSI_TRY(ssi_reserve(ctx, ctx->bSkinny, sizeof(float) * (size_t)batches * SK_SLICES * g.O * g.J));
        float* part = (float*)ctx->bSkinny.p;
        dim3 grid((g.J + 255) / 256, SK_SLICES, batches);
        if (g.O <= 4) k_gemm_skinny_gw<4><<<grid, 256, 0, ctx->stream>>>(g, part);
        else k_gemm_skinny_gw<SK_MAXO><<<grid, 256, 0, ctx->stream>>>(g, part);
        SSI_LAUNCH_CHECK(ctx);
        dim3 g2((g.J + 255) / 256, g.O, batches);
        k_gemm_skinny_gw_fin<<<g2, 256, 0, ctx->stream>>>(g, part);
        SSI_LAUNCH_CHECK(ctx);
        *used = true;
    }
    if (*used) ++ctx->stats.gemm_skinny_launches;
    return SSI_OK;
}

int ssi_gemm_tc_try(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast, bool* used);

int ssi_launch_gemm(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast) {
    bool taken = false;
    SSI_TRY(gemm_skinny_try(ctx, g, batches, a_kfast, b_jfast, &taken));
    if (taken) return SSI_OK;
    SSI_TRY(ssi_gemm_tc_try(ctx, g, batches, a_kfast, b_jfast, &taken));
    if (taken) return SSI_OK;
    dim3 grid((g.J + GT_T - 1) / GT_T, (g.O + GT_T - 1) / GT_T, batches);
    if (grid.y > 65535 || grid.z > 65535) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "gradient path: shape too large for one launch");
    if (a_kfast && b_jfast) k_gemm_simt<true, true><<<grid, 256, 0, ctx->stream>>>(g);
    else if (a_kfast) k_gemm_simt<true, false><<<grid, 256, 0, ctx->stream>>>(g);
    else if (b_jfast) k_gemm_simt<false, true><<<grid, 256, 0, ctx->stream>>>(g);
    else k_gemm_simt<false, false><<<grid, 256, 0, ctx->stream>>>(g);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}

// delta_L(o, j) = -(pred - y) * coef * act_L'(pred), and the per-(sample, chunk) squared-error partials.
// One block per (chunk of 256 datapoints, sample); all O outputs of a datapoint by the same thread.
__global__ void __launch_bounds__(256)
k_grad_delta_out(const float* __restrict__ pred, long long pred_sb, const float* __restrict__ Y, float* __restrict__ delta,
                 long long delta_sb, long long N, int O, int act, float coef, int n_chunks,
                 double* __restrict__ partials /* [g][n_chunks] */) {
    __shared__ double red[32];
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long g = blockIdx.y;
    double sse = 0.0;
    if (j < N) {
        for (int o = 0; o < O; ++o) {
            const long long e = o + j * O;
            const float pv = pred[g * pred_sb + e];
            const float df = pv - Y[e];
            sse += (double)df * (double)df;
            delta[g * delta_sb + e] = -df * coef * act_deriv_from_output(pv, act);
        }
    }
    const double tot = ssi_block_sum(sse, red);
    if (threadIdx.x == 0) partials[g * n_chunks + blockIdx.x] = tot;
}

// gb(o) = sum_j delta(o, j), fixed order.  delta is (O x N) with o fast: a warp takes 32 consecutive o (one coalesced
// 128-byte row per datapoint), the 8 warps of a block take every 8th datapoint of the block's slice of N; the per-block
// partials are summed in order by the second kernel.  (The first version gave a warp one o and let it stride through N:
// 32 sectors per load, 1.2 ms per 1024 x 60000 layer and sample.)
#define RS_SLICES 64
__global__ void __launch_bounds__(256)
k_grad_rowsum_part(const float* __restrict__ delta, long long d_sb, int O, long long N, float* __restrict__ part /* [g][RS_SLICES][O] */) {
    __shared__ float red[8][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int o = blockIdx.x * 32 + lane;
    const int slice = blockIdx.y;
    const long long g = blockIdx.z;
    const long long per = (N + RS_SLICES - 1) / RS_SLICES;
    const long long j0 = slice * per, j1 = min(N, j0 + per);
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
    if (o < O) {
        const float* d = delta + g * d_sb + o;
        long long j = j0 + warp;
        for (; j + 24 < j1; j += 32) {
            s0 += d[j * O]; s1 += d[(j + 8) * O]; s2 += d[(j + 16) * O]; s3 += d[(j + 24) * O];
        }
        for (; j < j1; j += 8) s0 += d[j * O];
    }
    red[warp][lane] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (warp == 0 && o < O) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += red[w][lane];
        part[(g * RS_SLICES + slice) * O + o] = t;
    }
}
__global__ void k_grad_rowsum_fin(const float* __restrict__ part, int O, float* __restrict__ out, long long out_sb) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    const long long g = blockIdx.y;
    if (o >= O) return;
    float t = 0.0f;
    for (int s = 0; s < RS_SLICES; ++s) t += part[(g * RS_SLICES + s) * O + o];
    out[g * out_sb + o] = t;
}
static int launch_rowsum(ssi_ctx* ctx, const float* delta, long long d_sb, int O, long long N, int g, float* out, long long out_sb) {
    SSI_TRY(ssi_reserve(ctx, ctx->bRowsum, sizeof(float) * (size_t)g * RS_SLICES * O));
    float* part = (float*)ctx->bRowsum.p;
    dim3 grid((O + 31) / 32, RS_SLICES, g);
    k_grad_rowsum_part<<<grid, 256, 0, ctx->stream>>>(delta, d_sb, O, N, part);
    SSI_LAUNCH_CHECK(ctx);
    dim3 g2((O + 127) / 128, g);
    k_grad_rowsum_fin<<<g2, 128, 0, ctx->stream>>>(part, O, out, out_sb);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}

int ssi_launch_delta_out(ssi_ctx* ctx, const float* pred, long long pred_sb, const float* Y, float* delta, long long delta_sb,
                         long long N, int O, int act, float coef, int n_chunks, int g, double* partials) {
    dim3 grid(n_chunks, g);
    k_grad_delta_out<<<grid, 256, 0, ctx->stream>>>(pred, pred_sb, Y, delta, delta_sb, N, O, act, coef, n_chunks, partials);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}
int ssi_launch_rowsum(ssi_ctx* ctx, const float* delta, long long d_sb, int O, long long N, int g, float* out, long long out_sb) {
    return launch_rowsum(ctx, delta, d_sb, O, N, g, out, out_sb);
}

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
    const int M = ctx->M, L = m.L, O = m.dims[L];
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
    long long act_elems = 0;
    int maxw = 0;
    long long h_off[SSI_MAX_LAYERS + 1];
    h_off[0] = 0;
    for (int l = 1; l <= L; ++l) { h_off[l] = act_elems; act_elems += (long long)m.dims[l] * N; maxw = std::max(maxw, m.dims[l]); }
    // sample strides are padded to 16 bytes so that the tensor-core GEMM (TMA) can address every sample's slice
    const long long np = (n + 3) & ~3ll;
    act_elems = (act_elems + 3) & ~3ll;
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
    SSI_TRY(ssi_reserve(ctx, ctx->bH1, sizeof(float) * (size_t)2 * (((long long)maxw * N + 3) & ~3ll) * G));
    SSI_TRY(ssi_reserve(ctx, ctx->bPartials, sizeof(double) * (size_t)B * n_chunks));
    SSI_TRY(ssi_reserve(ctx, ctx->bGradP, sizeof(float) * (size_t)S * M * G));
    SSI_TRY(ssi_reserve(ctx, ctx->bMisc, sizeof(double) * (size_t)B));
    float* dW = (float*)ctx->bW.p;
    float* gW = (float*)ctx->bGradW.p;
    float* H = (float*)ctx->bH0.p;                      // [g][act_elems]
    float* D[2] = {(float*)ctx->bH1.p, (float*)ctx->bH1.p + (size_t)(((long long)maxw * N + 3) & ~3ll) * G};   // [g][maxw x N] each
    double* partials = (double*)ctx->bPartials.p;
    float* gpart = (float*)ctx->bGradP.p;
    double* d_sse = (double*)ctx->bMisc.p;
    const long long d_sb = ((long long)maxw * N + 3) & ~3ll;
    const float coef = (mask & SSI_TERM_LL) ? (float)(1.0 / (sigma_m * sigma_m)) : 0.0f;

    for (int64_t b0 = 0; b0 < B; b0 += G) {
        const int g = (int)std::min<int64_t>(G, B - b0);
        SSI_TRY(ssi_project_device(ctx, dZ + b0 * M, g, dW, np));
        // ---- forward, every activation kept ----
        for (int l = 0; l < L; ++l) {
            const int in = m.dims[l], out = m.dims[l + 1];
            gemm_t q{};
            q.A = dW + m.w_off[l]; q.a_so = 1; q.a_sk = out; q.a_sb = np;
            q.B = l == 0 ? ctx->dX : H + h_off[l]; q.b_sk = 1; q.b_sj = in; q.b_sb = l == 0 ? 0 : act_elems;
            q.C = H + h_off[l + 1]; q.c_so = 1; q.c_sj = out; q.c_sb = act_elems;
            q.O = out; q.J = (int)N; q.K = in; q.split = 0;
            q.epi = 1; q.act = m.act[l]; q.bias = dW + m.b_off[l]; q.bias_sb = np;
            SSI_TRY(ssi_launch_gemm(ctx, q, g, false, false));
        }
        // ---- output delta + squared error ----
        {
            dim3 grid(n_chunks, g);
            k_grad_delta_out<<<grid, 256, 0, ctx->stream>>>(H + h_off[L], act_elems, ctx->dY, D[L & 1], d_sb, N, O, m.act[L - 1], coef,
                                                           n_chunks, partials + b0 * n_chunks);
            SSI_LAUNCH_CHECK(ctx);
        }
        // ---- backward ----
        for (int l = L - 1; l >= 0; --l) {
            const int in = m.dims[l], out = m.dims[l + 1];
            const float* delta = D[(l + 1) & 1];
            // gW_l(o, i) = sum_j delta(o, j) H_{l-1}(i, j)
            gemm_t q{};
            q.A = delta; q.a_so = 1; q.a_sk = out; q.a_sb = d_sb;
            q.B = l == 0 ? ctx->dX : H + h_off[l]; q.b_sk = in; q.b_sj = 1; q.b_sb = l == 0 ? 0 : act_elems;
            q.C = gW + m.w_off[l]; q.c_so = 1; q.c_sj = out; q.c_sb = np;
            q.O = out; q.J = in; q.K = N; q.split = 0; q.epi = 0;
            SSI_TRY(ssi_launch_gemm(ctx, q, g, false, true));
            SSI_TRY(launch_rowsum(ctx, delta, d_sb, out, N, g, gW + m.b_off[l], np));
            if (l > 0) {
                // delta_{l-1}(i, j) = sum_o W_l(o, i) delta_l(o, j) * act_{l-1}'(H_{l-1}(i, j))
                gemm_t r{};
                r.A = dW + m.w_off[l]; r.a_so = out; r.a_sk = 1; r.a_sb = np;
                r.B = delta; r.b_sk = 1; r.b_sj = out; r.b_sb = d_sb;
                r.C = D[l & 1]; r.c_so = 1; r.c_sj = in; r.c_sb = d_sb;
                r.O = in; r.J = (int)N; r.K = out; r.split = 0;
                r.epi = 2; r.act = m.act[l - 1]; r.Hprev = H + h_off[l]; r.h_sb = act_elems;
                SSI_TRY(ssi_launch_gemm(ctx, r, g, true, false));
            }
        }
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
