// ssi_gemm.cu — the strided FP32 GEMM (ssi_gemm.cuh) and the passes over a Dense chain built on it.
//
// ssi_launch_gemm runs each contraction on the skinny kernels below when a side is at most 16 wide, on the tensor cores
// (ssi_gemm_tc.cu) when the shape qualifies, and on k_gemm_simt otherwise.  ssi_launch_gemm_simt always takes k_gemm_simt,
// which is exact FP32: the LAYERED density, the predictive sweep and the tensor path's first-layer bases (ssi_logpost.cu)
// stay on it.  The value + gradient path (ssi_grad.cu) and the training step (ssi_train.cu) share ssi_reverse_pass:
//
//     H_l = act_l(W_l H_{l-1} + b_l)       all activations kept
//     delta_L = -(pred - y) * coef * act_L'(pred)        (+ the squared error, per chunk of 256 datapoints)
//     gW_l = delta_l H_{l-1}',  gb_l = rowsum(delta_l),  delta_{l-1} = (W_l' delta_l) * act_{l-1}'(H_{l-1})
//
// Reductions are two-stage with a fixed order, so a sample's result does not depend on the rest of the batch.
#include "ssi_common.cuh"
#include "ssi_gemm.cuh"

#include <algorithm>

#define GT_K 16
#define GT_LD 68          // padded tile rows: float4 aligned, transposed fills spread over the banks

// 64x64 tile per CTA, 4x4 per thread, fmaf in ascending k, zero-padded edges.  SSE: instead of storing C, sum
// (act(v + bias) - Y)^2 over the tile in FP64 (Y indexed like C) into partials[b][blockIdx.y * gridDim.x + blockIdx.x].
template <bool A_KFAST, bool B_JFAST, bool SSE>
__global__ void __launch_bounds__(256)
k_gemm_simt(const gemm_t p, const float* __restrict__ Y, double* __restrict__ partials) {
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
    double sse = 0.0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int j = j0 + ty * 4 + c;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int o = o0 + tx * 4 + r;
            if (o < p.O && j < p.J) {
                float v = acc[r][c];
                const long long ci = (long long)o * p.c_so + (long long)j * p.c_sj;
                if constexpr (SSE) {
                    const float df = ssi_act(v + p.bias[b * p.bias_sb + o], p.act) - Y[ci];
                    sse += (double)df * (double)df;
                } else {
                    if (p.epi == 1) v = ssi_act(v + p.bias[b * p.bias_sb + o], p.act);
                    else if (p.epi == 2) v *= act_deriv_from_output(p.Hprev[b * p.h_sb + ci], p.act);
                    p.C[b * p.c_sb + ci] = v;
                }
            }
        }
    }
    if constexpr (SSE) {
        __shared__ double red[32];
        const double tot = ssi_block_sum(sse, red);
        if (tid == 0) partials[b * gridDim.x * gridDim.y + (long long)blockIdx.y * gridDim.x + blockIdx.x] = tot;
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

int ssi_launch_gemm_simt(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast, const float* Y, double* partials) {
    if ((a_kfast && b_jfast) || (partials && (a_kfast || b_jfast)))
        return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "GEMM: no kernel for this operand orientation");
    dim3 grid((g.J + GT_T - 1) / GT_T, (g.O + GT_T - 1) / GT_T, batches);
    if (grid.y > 65535 || grid.z > 65535) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "GEMM: shape too large for one launch");
    if (partials) k_gemm_simt<false, false, true><<<grid, 256, 0, ctx->stream>>>(g, Y, partials);
    else if (a_kfast) k_gemm_simt<true, false, false><<<grid, 256, 0, ctx->stream>>>(g, nullptr, nullptr);
    else if (b_jfast) k_gemm_simt<false, true, false><<<grid, 256, 0, ctx->stream>>>(g, nullptr, nullptr);
    else k_gemm_simt<false, false, false><<<grid, 256, 0, ctx->stream>>>(g, nullptr, nullptr);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}

int ssi_launch_gemm(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast) {
    if (a_kfast && b_jfast) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "GEMM: no kernel for this operand orientation");
    bool taken = false;
    SSI_TRY(gemm_skinny_try(ctx, g, batches, a_kfast, b_jfast, &taken));
    if (taken) return SSI_OK;
    SSI_TRY(ssi_gemm_tc_try(ctx, g, batches, a_kfast, b_jfast, &taken));
    if (taken) return SSI_OK;
    return ssi_launch_gemm_simt(ctx, g, batches, a_kfast, b_jfast);
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

gemm_t ssi_dense_gemm(const ssi_model_t& m, int l, const float* W, long long w_sb, const float* H, long long h_sb, float* C,
                      long long c_sj, long long c_sb, int J) {
    const int in = m.dims[l], out = m.dims[l + 1];
    gemm_t q{};
    q.A = W + m.w_off[l]; q.a_so = 1; q.a_sk = out; q.a_sb = w_sb;
    q.B = H; q.b_sk = 1; q.b_sj = in; q.b_sb = h_sb;
    q.C = C; q.c_so = 1; q.c_sj = c_sj; q.c_sb = c_sb;
    q.O = out; q.J = J; q.K = in; q.split = 0;
    q.epi = 1; q.act = m.act[l]; q.bias = W + m.b_off[l]; q.bias_sb = w_sb;
    return q;
}

long long ssi_act_offsets(const ssi_model_t& m, long long J, long long* h_off, int* maxw) {
    long long elems = 0;
    *maxw = 0;
    for (int l = 1; l <= m.L; ++l) {
        if (h_off) h_off[l] = elems;
        elems += (long long)m.dims[l] * J;
        *maxw = std::max(*maxw, m.dims[l]);
    }
    return elems;
}

int ssi_reverse_pass(ssi_ctx* ctx, int g, long long J, const float* W, float* gW, long long w_sb, const float* X, const float* Y,
                     float* H, long long h_sb, float* const D[2], long long d_sb, float coef, double* partials) {
    const ssi_model_t& m = ctx->model;
    const int L = m.L;
    long long h_off[SSI_MAX_LAYERS + 1];
    int maxw;
    ssi_act_offsets(m, J, h_off, &maxw);
    // ---- forward, every activation kept ----
    for (int l = 0; l < L; ++l)
        SSI_TRY(ssi_launch_gemm(ctx, ssi_dense_gemm(m, l, W, w_sb, l == 0 ? X : H + h_off[l], l == 0 ? 0 : h_sb, H + h_off[l + 1],
                                                    m.dims[l + 1], h_sb, (int)J),
                                g, false, false));
    // ---- output delta + squared error ----
    const int n_chunks = (int)((J + 255) / 256);
    dim3 grid(n_chunks, g);
    k_grad_delta_out<<<grid, 256, 0, ctx->stream>>>(H + h_off[L], h_sb, Y, D[L & 1], d_sb, J, m.dims[L], m.act[L - 1], coef, n_chunks,
                                                   partials);
    SSI_LAUNCH_CHECK(ctx);
    // ---- backward ----
    for (int l = L - 1; l >= 0; --l) {
        const int in = m.dims[l], out = m.dims[l + 1];
        const float* delta = D[(l + 1) & 1];
        // gW_l(o, i) = sum_j delta(o, j) H_{l-1}(i, j)
        gemm_t q{};
        q.A = delta; q.a_so = 1; q.a_sk = out; q.a_sb = d_sb;
        q.B = l == 0 ? X : H + h_off[l]; q.b_sk = in; q.b_sj = 1; q.b_sb = l == 0 ? 0 : h_sb;
        q.C = gW + m.w_off[l]; q.c_so = 1; q.c_sj = out; q.c_sb = w_sb;
        q.O = out; q.J = in; q.K = J; q.split = 0; q.epi = 0;
        SSI_TRY(ssi_launch_gemm(ctx, q, g, false, true));
        SSI_TRY(launch_rowsum(ctx, delta, d_sb, out, J, g, gW + m.b_off[l], w_sb));
        if (l > 0) {
            // delta_{l-1}(i, j) = sum_o W_l(o, i) delta_l(o, j) * act_{l-1}'(H_{l-1}(i, j))
            gemm_t r{};
            r.A = W + m.w_off[l]; r.a_so = out; r.a_sk = 1; r.a_sb = w_sb;
            r.B = delta; r.b_sk = 1; r.b_sj = out; r.b_sb = d_sb;
            r.C = D[l & 1]; r.c_so = 1; r.c_sj = in; r.c_sb = d_sb;
            r.O = in; r.J = (int)J; r.K = out; r.split = 0;
            r.epi = 2; r.act = m.act[l - 1]; r.Hprev = H + h_off[l]; r.h_sb = h_sb;
            SSI_TRY(ssi_launch_gemm(ctx, r, g, true, false));
        }
    }
    return SSI_OK;
}
