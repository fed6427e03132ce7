// ssi_construct.cu — subspace construction streams.
//
// Replaces the numeric interior of subspace_construction
// (src/subspace_construction.jl:31,44-52,61-65):
//   K5  W_swa <- (ns*W_swa + W)/(ns+1);  column <- W - W_swa      (:46-47, :51-52)
//   K6  G = A'A          tall-skinny Gram of the n x K deviation matrix   (psvd, :63)
//   K7  G = V diag(lambda) V'   cyclic Jacobi in FP64, one CTA            (psvd, :63)
//   K8  P = A V_M  ( = U_M S_M )                                          (:65)
// The reference SVDs A directly with LowRankApprox.psvd; U_M S_M = A V_M is an identity,
// so the result is the same up to column sign.
#include "ssi_common.cuh"
#include "ssi_ptx.cuh"

#include <algorithm>
#include <cmath>

// ======================================================================================
// K5: SWA mean + deviation column, one float4 stream (16 n bytes per snapshot)
// ======================================================================================
// mean' = mean + (w - mean)/(ns+1)  ( == (ns*mean + w)/(ns+1) ),  dev = w - mean' = (w - mean) * ns/(ns+1):
// FP32 throughout, no cancellation beyond (w - mean) itself.  Two float4 per thread in flight.
__global__ void __launch_bounds__(256)
k_swa_push(const float* __restrict__ W, float* __restrict__ mean, float* __restrict__ dev,
           long long n, float inv, float c, int vec, float* __restrict__ amax /* running max |deviation| (scale of the Gram's FP16 planes) */) {
    float mx = 0.0f;
    const long long n4 = vec ? (n >> 2) : 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const float4* W4 = reinterpret_cast<const float4*>(W);
    float4* m4 = reinterpret_cast<float4*>(mean);
    float4* d4 = reinterpret_cast<float4*>(dev);
    long long i = t0;
    for (; i + stride < n4; i += 2 * stride) {
        const float4 w0 = __ldcs(W4 + i), w1 = __ldcs(W4 + i + stride);
        const float4 a0 = m4[i], a1 = m4[i + stride];
        const float4 e0 = make_float4(w0.x - a0.x, w0.y - a0.y, w0.z - a0.z, w0.w - a0.w);
        const float4 e1 = make_float4(w1.x - a1.x, w1.y - a1.y, w1.z - a1.z, w1.w - a1.w);
        m4[i] = make_float4(fmaf(e0.x, inv, a0.x), fmaf(e0.y, inv, a0.y), fmaf(e0.z, inv, a0.z), fmaf(e0.w, inv, a0.w));
        m4[i + stride] = make_float4(fmaf(e1.x, inv, a1.x), fmaf(e1.y, inv, a1.y), fmaf(e1.z, inv, a1.z), fmaf(e1.w, inv, a1.w));
        __stcs(d4 + i, make_float4(e0.x * c, e0.y * c, e0.z * c, e0.w * c));
        __stcs(d4 + i + stride, make_float4(e1.x * c, e1.y * c, e1.z * c, e1.w * c));
        mx = fmaxf(mx, fmaxf(fmaxf(fmaxf(fabsf(e0.x), fabsf(e0.y)), fmaxf(fabsf(e0.z), fabsf(e0.w))),
                             fmaxf(fmaxf(fabsf(e1.x), fabsf(e1.y)), fmaxf(fabsf(e1.z), fabsf(e1.w)))));
    }
    for (; i < n4; i += stride) {
        const float4 w0 = __ldcs(W4 + i);
        const float4 a0 = m4[i];
        const float4 e0 = make_float4(w0.x - a0.x, w0.y - a0.y, w0.z - a0.z, w0.w - a0.w);
        m4[i] = make_float4(fmaf(e0.x, inv, a0.x), fmaf(e0.y, inv, a0.y), fmaf(e0.z, inv, a0.z), fmaf(e0.w, inv, a0.w));
        __stcs(d4 + i, make_float4(e0.x * c, e0.y * c, e0.z * c, e0.w * c));
        mx = fmaxf(mx, fmaxf(fmaxf(fabsf(e0.x), fabsf(e0.y)), fmaxf(fabsf(e0.z), fabsf(e0.w))));
    }
    for (long long j = (n4 << 2) + t0; j < n; j += stride) {   // tail (n % 4), or everything when !vec
        const float e = W[j] - mean[j];
        mean[j] = fmaf(e, inv, mean[j]);
        dev[j] = e * c;
        mx = fmaxf(mx, fabsf(e));
    }
    // |deviation| = |e| c with c <= 1: max |e| is a valid (and tight enough) bound
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0 && mx > 0.0f) atomicMax(reinterpret_cast<unsigned*>(amax), __float_as_uint(mx));
}

int ssi_swa_push_device(ssi_ctx* ctx, const float* dW, double n_scalar) {
    if (ctx->swa_n <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin has not been called");
    if (ctx->swa_K >= ctx->swa_Kmax) return ssi_fail(ctx, SSI_ERR_ARG, "deviation matrix is full (K_max=%lld)", (long long)ctx->swa_Kmax);
    if (!(n_scalar >= 0)) return ssi_fail(ctx, SSI_ERR_ARG, "n_scalar must be >= 0");
    const int64_t n = ctx->swa_n;
    float* col = ctx->dDev + ctx->swa_K * ctx->swa_ld;
    // float4 path needs 16-byte aligned columns: n % 4 == 0 or fall back to the scalar tail for all
    const bool aligned = ((reinterpret_cast<uintptr_t>(dW) & 15) == 0);   // mean and the deviation column are aligned by construction
    const int blocks = ctx->sm_count * 8;
    // vec = 0: everything goes through the scalar tail loop
    k_swa_push<<<blocks, 256, 0, ctx->stream>>>(dW, ctx->dSwaMean, col, n, (float)(1.0 / (n_scalar + 1.0)),
                                                (float)(n_scalar / (n_scalar + 1.0)), aligned ? 1 : 0, ctx->dSwaAmax);
    SSI_LAUNCH_CHECK(ctx);
    ctx->swa_K++;
    ctx->stats.last_bytes = 16.0 * (double)n;
    ctx->stats.last_flops = 0;
    ctx->stats.last_units = 0;
    return SSI_OK;
}

// ======================================================================================
// K6: Gram G = A'A.  FP32 inputs, products and sums in FP64 (a*b of two floats is exact in
// double), fixed-order slab reduction: the Gram route squares the condition number, so the
// accumulation must not lose the small singular directions (SURVEY H5).
// ======================================================================================
#define GR 32
template <int GT, int MT>   // GT x GT tile per CTA, MT x MT outputs per thread, (GT/MT)^2 == 256 threads
__global__ void __launch_bounds__(256)
k_gram_partial(const float* __restrict__ A, long long n, long long ld, int K, int tiles, long long rows_per_slab,
               double* __restrict__ partial /* slabs x K x K */) {
    __shared__ __align__(16) double As[GR][GT];
    __shared__ __align__(16) double Bs[GR][GT];
    // blockIdx.y enumerates tile pairs (ta <= tb)
    int ta = 0, rem = blockIdx.y;
    while (rem >= tiles - ta) { rem -= tiles - ta; ++ta; }
    const int tb = ta + rem;
    const int a0 = ta * GT, b0 = tb * GT;
    constexpr int TPR = GT / MT;                 // threads per tile row (16)
    const int tid = threadIdx.x, tx = tid % TPR, ty = tid / TPR;
    const long long r_begin = (long long)blockIdx.x * rows_per_slab;
    const long long r_end = min(n, r_begin + rows_per_slab);

    double acc[MT][MT];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < MT; ++j) acc[i][j] = 0.0;

    for (long long r0 = r_begin; r0 < r_end; r0 += GR) {
#pragma unroll
        for (int s = 0; s < (GR * GT) / 256; ++s) {
            const int idx = tid + s * 256;
            const int r = idx % GR, c = idx / GR;
            const bool rv = (r0 + r < r_end);
            As[r][c] = (rv && a0 + c < K) ? (double)A[(r0 + r) + (long long)(a0 + c) * ld] : 0.0;
            Bs[r][c] = (rv && b0 + c < K) ? (double)A[(r0 + r) + (long long)(b0 + c) * ld] : 0.0;
        }
        __syncthreads();
#pragma unroll 4
        for (int r = 0; r < GR; ++r) {
            double x[MT], y[MT];
#pragma unroll
            for (int i = 0; i < MT; i += 2) {
                const double2 xv = *reinterpret_cast<const double2*>(&As[r][ty * MT + i]);
                const double2 yv = *reinterpret_cast<const double2*>(&Bs[r][tx * MT + i]);
                x[i] = xv.x; x[i + 1] = xv.y; y[i] = yv.x; y[i + 1] = yv.y;
            }
#pragma unroll
            for (int i = 0; i < MT; ++i)
#pragma unroll
                for (int j = 0; j < MT; ++j) acc[i][j] = fma(x[i], y[j], acc[i][j]);
        }
        __syncthreads();
    }
    double* out = partial + (long long)blockIdx.x * K * K;
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < MT; ++j) {
            const int a = a0 + ty * MT + i, b = b0 + tx * MT + j;
            if (a < K && b < K) {
                out[a + (long long)b * K] = acc[i][j];
                if (ta != tb) out[b + (long long)a * K] = acc[i][j];
            }
        }
}

__global__ void k_gram_reduce(const double* __restrict__ partial, int slabs, long long KK, double* __restrict__ G) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= KK) return;
    double s = 0.0;
    for (int p = 0; p < slabs; ++p) s += partial[(long long)p * KK + e];
    G[e] = s;
}

int ssi_gram_device(ssi_ctx* ctx, const float* dA, int64_t n, int64_t ld, int K, double* dG, bool allow_tensor, const float* d_amax) {
    if (allow_tensor && d_amax && ssi_gram_tc_usable(ctx, dA, n, ld, K)) return ssi_gram_tc_device(ctx, dA, n, ld, K, dG, d_amax);
    const int GT = K <= 32 ? 32 : 64;
    const int tiles = (K + GT - 1) / GT;
    const int pairs = tiles * (tiles + 1) / 2;
    int slabs = (int)std::max<int64_t>(1, std::min<int64_t>(2 * ctx->sm_count, (n + 1023) / 1024));
    int64_t rows_per = (n + slabs - 1) / slabs;
    rows_per = (rows_per + GR - 1) / GR * GR;
    slabs = (int)((n + rows_per - 1) / rows_per);
    SSI_TRY(ssi_reserve(ctx, ctx->bGram, sizeof(double) * (size_t)slabs * K * K));
    double* partial = (double*)ctx->bGram.p;
    if (pairs > 65535) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "too many deviation columns (K=%d)", K);
    dim3 grid(slabs, pairs);
    if (GT == 32) k_gram_partial<32, 2><<<grid, 256, 0, ctx->stream>>>(dA, n, ld, K, tiles, rows_per, partial);
    else          k_gram_partial<64, 4><<<grid, 256, 0, ctx->stream>>>(dA, n, ld, K, tiles, rows_per, partial);
    SSI_LAUNCH_CHECK(ctx);
    const long long KK = (long long)K * K;
    k_gram_reduce<<<(unsigned)((KK + 255) / 256), 256, 0, ctx->stream>>>(partial, slabs, KK, dG);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}

int ssi_subspace_gram(ssi_ctx* ctx) {
    // dP holds [P | W_swa] as an n x (M+1) column-major matrix
    // the prior's Gram stays on the exact FP64 path (K = M+1 is tiny)
    return ssi_gram_device(ctx, ctx->dP, ctx->model.n, ctx->model.n, ctx->M + 1, ctx->dSubGram, false, nullptr);
}

// ======================================================================================
// K7: symmetric eigen-solve of the K x K Gram, FP64 (Veselic-Hari / Drmac: Cholesky, then one-sided Jacobi).
//
//   1. Pivoted Cholesky  Pi G Pi' = L L'  (in place, one CTA; a pivot below K eps * trace ends it: the remaining
//      columns are the numerical null space).  The columns of L come out with decreasing norms, the order in which a
//      one-sided Jacobi method converges fastest, and their singular values are sqrt(lambda): half the dynamic range
//      (in digits) of the Gram's own columns -- 7 sweeps where Jacobi on G itself took 17 for BASELINE's construction.
//   2. One-sided (Hestenes) Jacobi on the COLUMNS of L: a rotation of columns (p, q) needs their three inner products
//      and touches those two columns only, so a half warp owns a pair, the inner products are shuffle reductions and
//      ONE barrier per round-robin round is all the synchronisation there is (the two-sided solver of round 1 rotated
//      rows and columns: two block-wide barriers per round around a serial rotation-parameter phase, 3.9 us per
//      round, 4.6 ms at K = 100).  tan(theta) is computed in FP32 from exponent-aligned inputs and polished by one
//      Newton step in FP64; c = rsqrt(1 + t^2), s = t c are orthogonal to working precision by construction, so
//      accuracy does not depend on t -- only the convergence rate does.
//   3. With the columns mutually orthogonal,  L V = U S:  lambda_i = |column i|^2 and Pi' u_i is the eigenvector.
//   K <= 160: a cluster of 8 CTAs, the columns live in shared memory (k_osj_cluster2).  Larger K (README's batchsize-1
//   loader gives K = 1000, SURVEY Q3): a cooperative grid with the matrix in global memory (L2-resident) and a grid barrier
//   per round (k_osj); no pair tables, so K is limited by memory only (ssi_swa_* accept K <= 16384).
// ======================================================================================
#define OSJ_THREADS 1024
#define OSJ_SMEM_KMAX 160
#define OSJ_KMAX 16384
__device__ __forceinline__ void osj_grid_barrier(unsigned* counter, unsigned& target, unsigned nblocks) {
    __syncthreads();
    if (nblocks > 1) {
        if (threadIdx.x == 0) {
            target += nblocks;
            __threadfence();
            atomicAdd(counter, 1u);
            while (*reinterpret_cast<volatile unsigned*>(counter) < target) { }
            __threadfence();
        }
        __syncthreads();
    }
}

// Pi G Pi' = L L' in place (full symmetric storage in, lower triangle out, strict upper triangle and the columns past the
// numerical rank zeroed); perm[r] = original index of row r.  One CTA; G has leading dimension ld >= K.
// Three block barriers per pivot step and no integer division: every warp finds the pivot for itself (same data, same
// order, same answer), the symmetric swap is one pass, the trailing update writes both triangles (the two mirror entries
// are the same fused multiply-add, bit for bit) so that the matrix stays symmetric without a mirror pass.  The first
// version (block-wide argmax through shared memory, triangle update + mirror pass indexed by 64-bit division, seven
// barriers per step) cost 0.6 ms at K = 100, 29 % of the eigen-solve.
__device__ void osj_pivoted_cholesky(double* __restrict__ G, int K, int ld, int* __restrict__ perm, double thresh) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    for (int i = tid; i < K; i += nt) perm[i] = i;
    __syncthreads();
    int rank = K;
    for (int j = 0; j < K; ++j) {
        // pivot = largest remaining diagonal entry (ties: smallest index)
        double best = -1.0;
        int bi = j;
        for (int i = j + lane; i < K; i += 32) {
            const double v = G[i + (long long)i * ld];
            if (v > best) { best = v; bi = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (!(best > thresh)) { rank = j; break; }
        if (bi != j) {       // symmetric swap j <-> bi: thread k moves the four entries of row / column k it alone touches
            for (int k = tid; k < K; k += nt) {
                if (k == j) {
                    const double t = G[j + (long long)j * ld]; G[j + (long long)j * ld] = G[bi + (long long)bi * ld]; G[bi + (long long)bi * ld] = t;
                } else if (k != bi) {
                    double t = G[j + (long long)k * ld]; G[j + (long long)k * ld] = G[bi + (long long)k * ld]; G[bi + (long long)k * ld] = t;
                    t = G[k + (long long)j * ld]; G[k + (long long)j * ld] = G[k + (long long)bi * ld]; G[k + (long long)bi * ld] = t;
                }
            }
            if (tid == 0) { const int t = perm[j]; perm[j] = perm[bi]; perm[bi] = t; }
            __syncthreads();
        }
        const double ljj = sqrt(best), inv = 1.0 / ljj;
        double* cj = G + (long long)j * ld;
        for (int i = j + tid; i < K; i += nt) cj[i] = (i == j) ? ljj : cj[i] * inv;
        __syncthreads();
        // trailing update, both triangles: G[i, k] -= L[i, j] L[k, j] for i, k > j.  A lane keeps its four entries of column j
        // in registers while the warp walks its columns k: four independent load / fma / store chains per step
        for (int i0 = j + 1 + lane; i0 < K; i0 += 128) {
            double ci[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) ci[u] = (i0 + 32 * u < K) ? cj[i0 + 32 * u] : 0.0;
            for (int k = j + 1 + warp; k < K; k += nw) {
                const double lk = -cj[k];
                double* ck = G + (long long)k * ld + i0;
                double v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = (i0 + 32 * u < K) ? ck[32 * u] : 0.0;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (i0 + 32 * u < K) ck[32 * u] = fma(ci[u], lk, v[u]);
            }
        }
        __syncthreads();
    }
    for (int k = warp; k < K; k += nw)
        for (int i = lane; i < K; i += 32)
            if (i < k || k >= rank) G[i + (long long)k * ld] = 0.0;
    __syncthreads();
}

__global__ void __launch_bounds__(OSJ_THREADS)
k_osj(double* __restrict__ G /* K x K column-major Gram; on exit the orthogonalised columns of its Cholesky factor */, int K, int max_sweeps,
      unsigned* __restrict__ sync_counter /* zeroed */, unsigned* __restrict__ rot_count /* [3], zeroed */,
      int* __restrict__ perm /* K: row r of the result is original index perm[r] */, int* __restrict__ sweeps_out) {
    __shared__ double red[32];
    __shared__ double s_tr;
    const int tid = threadIdx.x, nt = blockDim.x;
    const unsigned nb = gridDim.x;
    unsigned target = 0;
    if (blockIdx.x == 0) {
        double tr = 0.0;
        for (int i = tid; i < K; i += nt) tr += fabs(G[i + (long long)i * K]);
        tr = ssi_block_sum(tr, red);
        if (tid == 0) s_tr = tr;
        __syncthreads();
        osj_pivoted_cholesky(G, K, K, perm, (double)K * 2.220446049250313e-16 * s_tr);
    }
    osj_grid_barrier(sync_counter, target, nb);          // the other CTAs of a cooperative grid wait for the factor
    const double tol = (double)K * 2.220446049250313e-16, tol2 = tol * tol;

    const int m = (K + 1) & ~1;                  // even number of players; index K (if any) is a bye
    const int np = m / 2;
    const int hw = (blockIdx.x * nt + tid) >> 4, n_hw = (nb * nt) >> 4;      // half warps: one per column pair
    const int hl = tid & 15;
    const unsigned hmask = 0xffffu << (tid & 16);
    int sweep = 0;
    bool converged = false;
    for (; sweep < max_sweeps; ++sweep) {
        unsigned* cnt = rot_count + (sweep % 3);
        if (blockIdx.x == 0 && tid == 0) rot_count[(sweep + 1) % 3] = 0;       // next sweep's counter (idle since sweep - 2)
        for (int r = 0; r < m - 1; ++r) {
            for (int i = hw; i < np; i += n_hw) {
                int p, q;
                if (i == 0) { p = m - 1; q = r; }
                else { p = (r + i) % (m - 1); q = (r - i + (m - 1)) % (m - 1); }
                if (p > q) { const int t = p; p = q; q = t; }
                if (q >= K) continue;                                       // bye
                double* gp = G + (long long)p * K;
                double* gq = G + (long long)q * K;
                double a = 0.0, b = 0.0, c = 0.0;
                for (int k = hl; k < K; k += 16) {
                    const double x = gp[k], y = gq[k];
                    a = fma(x, x, a); b = fma(y, y, b); c = fma(x, y, c);
                }
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) {
                    a += __shfl_xor_sync(hmask, a, o);
                    b += __shfl_xor_sync(hmask, b, o);
                    c += __shfl_xor_sync(hmask, c, o);
                }
                if (c * c <= tol2 * a * b) continue;              // already orthogonal (also: a null column)
                // tan(theta) of the rotation that makes the two columns orthogonal solves  h t^2 + 2 d t - h = 0,
                // d = |g_q|^2 - |g_p|^2, h = 2 g_p.g_q: the root of smaller magnitude, t = h / (d + sign(d) sqrt(d^2 + h^2)).
                // FP32 on exponent-aligned copies, then one Newton step in FP64 (the divisor again in FP32).
                const double d = b - a, h = 2.0 * c;
                const int ex = max(__double2hiint(fabs(d)), __double2hiint(fabs(h))) >> 20;      // biased exponent of the larger
                const double sc = __hiloint2double((2046 - ex) << 20, 0);                          // 2^-(exponent): both fit FP32 after scaling
                const float df = (float)(d * sc), hf = (float)(h * sc);
                const float rf = sqrtf(fmaf(df, df, hf * hf));
                double t = (double)(hf / (df + copysignf(rf, df)));
                const double f = fma(h * t, t, fma(2.0 * d, t, -h));
                t -= f * (double)(1.0f / (float)((2.0 * (h * t + d)) * sc)) * sc;
                const double cs = rsqrt(fma(t, t, 1.0)), sn = t * cs;
                for (int k = hl; k < K; k += 16) {
                    const double x = gp[k], y = gq[k];
                    gp[k] = cs * x - sn * y;
                    gq[k] = sn * x + cs * y;
                }
                if (hl == 0) atomicAdd(cnt, 1u);
            }
            osj_grid_barrier(sync_counter, target, nb);
        }
        // every rotation of this sweep has been counted before the last barrier of the sweep
        if (*reinterpret_cast<volatile unsigned*>(cnt) == 0u) { ++sweep; converged = true; break; }
    }
    // sweeps executed (the last one without a rotation), or max_sweeps + 1 when the last sweep still rotated
    if (blockIdx.x == 0 && tid == 0) *sweeps_out = converged ? sweep : max_sweeps + 1;
}

// The same solver for K <= 160 on a CLUSTER of 8 CTAs (distributed shared memory): on one SM the ~K^2 / 2 column updates of a
// round are issue-bound (2.7 us per round at K = 100, measured; one CTA took 2.8 ms for the whole solve); spread over eight
// SMs a round costs one pair's latency chain.  Every CTA starts from its own copy of the Cholesky factor (computed
// redundantly, bit-identically).  In every round a CTA orthogonalises the pairs that fall to its warps, reading its LOCAL
// shared memory, and writes each of the two columns -- rotated or not -- into the shared memory of the ONE CTA that will
// own it in the next round (the round-robin schedule is a closed formula, so the next owner is computed, not
// communicated).  A column is thus valid exactly where it is needed: 2 column transfers per pair and round (80 KB per
// round over the whole cluster at K = 100) instead of a broadcast.
#define OSJC_CTAS 8
#define OSJC_THREADS 512
#define OSJC_HW (OSJC_THREADS / 32)        // warps (pairs) per CTA and pass: one warp per pair
static_assert((OSJ_SMEM_KMAX + 1) / 2 <= OSJC_CTAS * OSJC_HW, "k_osj_cluster2 needs a warp for every column pair");
__device__ __forceinline__ uint32_t osjc_mapa(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void osjc_st_u32(uint32_t cluster_addr, unsigned v) {
    asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
// This is the second version of the cluster solver; the first one (a cluster barrier per round) took 1.62 ms at K = 100
// against 0.77 ms.  The solver's time is 891 rounds of one rotation each at K = 100, so what counts is the latency of a round.
//   * DATAFLOW instead of a cluster barrier per round.  A rotated column goes to the shared memory of its next owner with
//     st.async, which completes transaction bytes on an mbarrier of the warp that will consume it (one mbarrier per pair slot
//     and round parity); that warp posts arrive.expect_tx for its two columns and waits on its own barrier only.  The first
//     version's barrier.cluster.arrive.release compiles to MEMBAR.ALL.GPU + ERRBAR + the hardware barrier, its acquire side to
//     CCTL.IVALL: ~1000 of the 2300 cycles of a round (ncu, profiles/r02_ncu_streams.txt).  A neighbour can run at most one
//     round ahead of a slot (its next inputs need this slot's output), hence two barriers per slot; bytes that land before
//     the consumer has posted its expect_tx are legal (the phase cannot complete without the consumer's own arrival).
//   * the pair slots are dealt out in equal contiguous runs (ceil(np / 8) per CTA).  A column moves to the neighbouring slot
//     from one round to the next, so only the two columns at each run boundary cross to another SM; and the FP64 pipe -- 64
//     lanes per clock and SM, ~80 FP64 warp instructions per pair -- is shared by 7 pairs instead of 16: the first version
//     filled CTA after CTA (16, 16, 16, 2 pairs at K = 100) and its three full SMs were FP64-bound at ~2600 cycles a round.
//   * columns are padded to IT * 32 rows (zeros), IT a template parameter: no predicates, no partial loops;
//   * tan(theta) comes from the FP32 closed form alone.  c = rsqrt(1 + t^2) and s = t c are still exact in FP64 (FP32 seed,
//     one cubically convergent correction), so the rotation is orthogonal to working precision whatever t is; an error of
//     2^-22 in t leaves 2^-22 of the pair's inner product behind instead of nothing, which the next sweep removes -- the
//     FP64 Newton step on t bought nothing but latency (same 9 sweeps at K = 100);
//   * division and square root are the approximate single-instruction forms (no slow-path calls).
__device__ __forceinline__ int osjc2_slot(int x, int r, int m) {
    if (x == m - 1 || x == r) return 0;
    int i = x - r; if (i < 0) i += m - 1;                  // x = (r + i) mod (m - 1)
    if (i >= m / 2) i = (m - 1) - i;                       // else x = (r - i) mod (m - 1)
    return i;
}
__device__ __forceinline__ void osjc_st_async_f64(uint32_t cluster_addr, double v, uint32_t cluster_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                 ::"r"(cluster_addr), "l"(__double_as_longlong(v)), "r"(cluster_bar) : "memory");
}
__device__ __forceinline__ bool osjc_try_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void osjc_wait_cluster(uint32_t bar, uint32_t parity) {
    if (osjc_try_wait_cluster(bar, parity)) return;
    const long long t0 = clock64();
    while (!osjc_try_wait_cluster(bar, parity)) {
        if (clock64() - t0 > (1ll << 31)) {
            printf("ssi: eigen-solver column wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}
template <int IT>
__global__ void __cluster_dims__(OSJC_CTAS, 1, 1) __launch_bounds__(OSJC_THREADS)
k_osj_cluster2(double* __restrict__ Gg, int K, int max_sweeps, int* __restrict__ perm_out, int* __restrict__ sweeps_out) {
    constexpr int KP = IT * 32;
    constexpr uint32_t COLB = KP * 8;                          // bytes of a column
    extern __shared__ double osj_smem[];
    double* G = osj_smem;                                     // K columns of KP rows
    int* s_perm = reinterpret_cast<int*>(G + (size_t)K * KP);  // K
    __shared__ double red[32];
    __shared__ double s_tr;
    __shared__ unsigned s_cnt, s_slot[OSJC_CTAS], s_big, s_bigslot[OSJC_CTAS];
    __shared__ __align__(8) uint64_t s_bar[OSJC_HW][2];       // [pair slot of this CTA][round parity]
    const int tid = threadIdx.x, nt = blockDim.x, hl = tid & 31, wid = tid >> 5;
    const uint32_t rank = cluster_ctarank();
    {
        double tr = 0.0;
        for (int i = tid; i < K; i += nt) tr += fabs(Gg[i + (long long)i * K]);
        tr = ssi_block_sum(tr, red);
        if (tid == 0) { s_tr = tr; s_cnt = 0; s_big = 0; }
        if (tid < 2 * OSJC_HW) mbar_init(smem_u32(&s_bar[tid >> 1][tid & 1]), 1);
        for (int k = wid; k < K; k += OSJC_HW)
            for (int i = hl; i < KP; i += 32) G[i + k * KP] = i < K ? Gg[i + (long long)k * K] : 0.0;
        fence_barrier_init();
        __syncthreads();
        osj_pivoted_cholesky(G, K, KP, s_perm, (double)K * 2.220446049250313e-16 * s_tr);
    }
    cluster_sync_all();
    const double tol = (double)K * 2.220446049250313e-16, tol2 = tol * tol;
    const int m = (K + 1) & ~1, np = m / 2;
    const int spc = (np + OSJC_CTAS - 1) / OSJC_CTAS;         // pair slots per CTA (<= OSJC_HW for K <= OSJ_SMEM_KMAX)
    const int slot = (int)rank * spc + wid;                   // this warp's pair slot in every round
    const bool has_pair = wid < spc && slot < np;
    const uint32_t g_local = smem_u32(G), bar_local = smem_u32(&s_bar[0][0]);
    const uint32_t my_bar = bar_local + (uint32_t)wid * 16u;
    // Round-robin schedule, round r: slot 0 holds columns (A, B) = (m - 1, r), slot i holds (r + i, r - i) mod (m - 1).  From one
    // round to the next both column indices of a slot grow by one (slot 0's A stays), A moves to slot i - 1 (slot 1's A becomes
    // slot 0's B, slot 0's A stays put) and B to slot i + 1 (the last slot's B becomes its own A): the two destinations of a warp
    // never change, only the column offsets advance.  Column m - 1 = K is a phantom when K is odd: slot 0 then only forwards B.
    const bool phantom = slot == 0 && (K & 1);
    const uint32_t wrap = (uint32_t)(m - 1) * COLB;
    uint32_t offA = (slot == 0 ? (uint32_t)(m - 1) : (uint32_t)slot) * COLB;
    uint32_t offB = (slot == 0 ? 0u : (uint32_t)(m - 1 - slot)) * COLB;
    uint32_t dstA = 0, dstB = 0, barA = 0, barB = 0;           // shared::cluster addresses in the CTAs of the next owners
    if (has_pair) {
        const int sa = max(slot - 1, 0), sb = min(slot + 1, np - 1);
        const int ca = sa / spc, cb = sb / spc;
        dstA = osjc_mapa(g_local, (uint32_t)ca) + (uint32_t)hl * 8u;
        dstB = osjc_mapa(g_local, (uint32_t)cb) + (uint32_t)hl * 8u;
        barA = osjc_mapa(bar_local, (uint32_t)ca) + (uint32_t)(sa - ca * spc) * 16u;
        barB = osjc_mapa(bar_local, (uint32_t)cb) + (uint32_t)(sb - cb * spc) * 16u;
    }
    const uint32_t expect = (phantom ? 1u : 2u) * COLB;
    // wait for the columns of round g >= 1 (the data of round 0 is the local Cholesky factor): g counts rounds over all sweeps,
    // the columns of round g are announced on the barrier of parity g & 1, whose ((g - 1) >> 1)-th phase that is
    auto await = [&](unsigned g) {
        if (g == 0u) return;
        const uint32_t bar = my_bar + (g & 1u) * 8u;
        if (hl == 0) mbar_expect_tx(bar, expect);
        __syncwarp();
        mbar_wait(bar, ((g - 1u) >> 1) & 1u);
    };
    const char* Gb = reinterpret_cast<const char*>(G) + hl * 8;
    unsigned g = 0;
    int sweep = 0;
    bool converged = false;
    for (; sweep < max_sweeps; ++sweep) {
        unsigned cnt = 0, big = 0;
        if (has_pair) {
            for (int r = 0; r < m - 1; ++r) {
                await(g);
                ++g;
                const uint32_t par = (g & 1u) * 8u;                          // parity of the round the results are for
                // the columns keep their index: where column j lives is the same offset in every CTA
                const uint32_t nA = slot == 0 ? offA : (offA + COLB == wrap ? 0u : offA + COLB);
                const uint32_t nB = offB + COLB == wrap ? 0u : offB + COLB;
                double x[IT], y[IT];
#pragma unroll
                for (int it = 0; it < IT; ++it) y[it] = *reinterpret_cast<const double*>(Gb + offB + it * 256);
                if (phantom) {                                               // bye: the column only moves on
#pragma unroll
                    for (int it = 0; it < IT; ++it) osjc_st_async_f64(dstB + offB + (uint32_t)it * 256u, y[it], barB + par);
                } else {
#pragma unroll
                    for (int it = 0; it < IT; ++it) x[it] = *reinterpret_cast<const double*>(Gb + offA + it * 256);
                    double a = 0.0, b = 0.0, c = 0.0;
#pragma unroll
                    for (int it = 0; it < IT; ++it) { a = fma(x[it], x[it], a); b = fma(y[it], y[it], b); c = fma(x[it], y[it], c); }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        a += __shfl_xor_sync(0xffffffffu, a, o);
                        b += __shfl_xor_sync(0xffffffffu, b, o);
                        c += __shfl_xor_sync(0xffffffffu, c, o);
                    }
                    const double c2 = c * c, ab = a * b;
                    double cs = 1.0, sn = 0.0;
                    if (c2 > tol2 * ab) {
                        // t = h / (d + sign(d) sqrt(d^2 + h^2)), d = |y|^2 - |x|^2, h = 2 x.y, on exponent-aligned FP32 copies
                        const double d = b - a, h = c + c;
                        const int ex = max(__double2hiint(fabs(d)), __double2hiint(fabs(h))) >> 20;
                        const double sc = __hiloint2double((2046 - ex) << 20, 0);
                        const float df = (float)(d * sc), hf = (float)(h * sc);
                        float rf;
                        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"(fmaf(df, df, hf * hf)));
                        const double t = (double)__fdividef(hf, df + copysignf(rf, df));
                        const double w = fma(t, t, 1.0);                  // in [1, 2]
                        float r0;
                        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"((float)w));
                        const double c0 = (double)r0;
                        const double e = fma(-w * c0, c0, 1.0);           // 1 - w c0^2, ~2^-22
                        cs = fma(c0 * e, fma(0.375, e, 0.5), c0);         // c0 (1 + e/2 + 3 e^2 / 8): error ~e^3
                        sn = t * cs;
                        ++cnt;
                        big |= (c2 > 1e-10 * ab) ? 1u : 0u;               // a rotation that was not yet of second order
                    }
#pragma unroll
                    for (int it = 0; it < IT; ++it) {
                        osjc_st_async_f64(dstA + offA + (uint32_t)it * 256u, cs * x[it] - sn * y[it], barA + par);
                        osjc_st_async_f64(dstB + offB + (uint32_t)it * 256u, sn * x[it] + cs * y[it], barB + par);
                    }
                }
                offA = nA;
                offB = nB;
            }
            if (hl == 0 && cnt) { atomicAdd(&s_cnt, cnt); atomicOr(&s_big, big); }
        }
        // end of the sweep: every CTA tells every CTA how much it rotated (the one cluster barrier per sweep)
        __syncthreads();
        if (tid < OSJC_CTAS) {
            osjc_st_u32(osjc_mapa(smem_u32(&s_slot[rank]), (uint32_t)tid), s_cnt);
            osjc_st_u32(osjc_mapa(smem_u32(&s_bigslot[rank]), (uint32_t)tid), s_big);
        }
        cluster_sync_all();
        unsigned total = 0, anybig = 0;
#pragma unroll
        for (int c = 0; c < OSJC_CTAS; ++c) { total += s_slot[c]; anybig |= s_bigslot[c]; }
        __syncthreads();
        if (tid == 0) { s_cnt = 0; s_big = 0; }
        cluster_sync_all();           // nobody publishes the next sweep's counts before everybody has read these
        // converged when nothing was rotated, or when every rotation of the sweep was so small (cos < 1e-5) that what it
        // leaves behind is of second order, cos ~ 1e-10 (quadratic convergence of the Jacobi method): the eigenvectors
        // are delivered in FP32
        if (total == 0u || !anybig) { ++sweep; converged = true; break; }
    }
    // the columns of the round that would come next have been sent to their owners: wait for them, then write them out
    if (has_pair) {
        await(g);
        const int ja = (int)(offA / COLB), jb = (int)(offB / COLB);
        for (int k = hl; k < K; k += 32) {
            if (!phantom) Gg[k + (long long)ja * K] = G[k + ja * KP];
            Gg[k + (long long)jb * K] = G[k + jb * KP];
        }
    }
    cluster_sync_all();           // no CTA leaves while a peer may still write into its shared memory
    if (rank == 0) {
        for (int i = tid; i < K; i += nt) perm_out[i] = s_perm[i];
        if (tid == 0) *sweeps_out = converged ? sweep : max_sweeps + 1;
    }
}

// eigenvalues = squared norms of the orthogonalised columns, rank-sorted descending (ties by index); eigenvectors = the
// normalised columns with their rows sent back through the pivoting permutation, written to V (K x K).  One warp per column.
__global__ void __launch_bounds__(256)
k_osj_norms(const double* __restrict__ G, int K, double* __restrict__ norms2) {
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (c >= K) return;
    double a = 0.0;
    for (int k = lane; k < K; k += 32) { const double x = G[k + (long long)c * K]; a = fma(x, x, a); }
    a = ssi_warp_sum(a);
    if (lane == 0) norms2[c] = a;
}
__global__ void __launch_bounds__(256)
k_osj_sort_normalise(const double* __restrict__ G, int K, const double* __restrict__ norms2, const int* __restrict__ perm,
                     double* __restrict__ lambda, int* __restrict__ order, double* __restrict__ V) {
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (c >= K) return;
    const double li = norms2[c];
    int rank = 0;
    for (int j = lane; j < K; j += 32) { const double lj = norms2[j]; rank += (lj > li) || (lj == li && j < c); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
    if (lane == 0) { lambda[rank] = li; order[rank] = c; }
    const double inv = li > 0.0 ? rsqrt(li) : 0.0;         // signs are arbitrary, as psvd's are
    for (int k = lane; k < K; k += 32) V[perm[k] + (long long)c * K] = G[k + (long long)c * K] * inv;
}

// ======================================================================================
// K8: P = A V_M  (second pass over A; V_M staged in shared memory, zero-padded to MP columns)
// ======================================================================================
// V_M as [Kpad][MP] floats, zero padded in both directions (Kpad = K rounded up to the stage width of k_form_p_tma)
__global__ void k_pack_v(const double* __restrict__ V, const int* __restrict__ order, int K, int Kpad, int M, int MP, float* __restrict__ out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= Kpad * MP) return;
    const int k = e / MP, j = e % MP;
    out[e] = (j < M && k < K) ? (float)V[k + (long long)order[j] * K] : 0.0f;
}

// P = A V_M as a stream through shared memory.  Per row of P the kernel spends K * M multiply-adds on 4 K bytes of A
// (50 flop/B at K = 100, M = 20): on CUDA cores the FMA pipe and HBM are busy to the same degree, so the loads must not
// cost the compute warps a single stall.  A TMA producer warp therefore keeps a ring of 5 stages (8 columns x 256 rows
// of A each) in flight, and the 2 compute warps of a CTA -- 4 consecutive rows x MP outputs per thread, 80 accumulators for
// MP = 20 -- read their operands from shared memory only: one 16-byte load of A and MP / 4 broadcast loads of V per 4 MP
// FMAs.  FOUR small CTAs per SM rather than one large one: a CTA's tile-boundary epilogue and barrier waits overlap with
// the main loops of the other three (one CTA with 8 / 10 / 12 compute warps: 0.977 / 1.056 / 0.987 ms; two CTAs of 4:
// 0.958 ms; four of 2: 0.944 ms).  What bounds it is instruction issue (ncu: 70 % of the issue slots, FMA pipe 59 %, DRAM
// 60 %); packed FFMA2 with V duplicated in shared memory was measured and is slower (twice the V loads for the same
// FMA-pipe time).  (Round 1 loaded A straight from global memory into registers with V in the constant bank: 124
// registers per thread left 16 warps per SM to cover DRAM latency, 71 % of the HBM peak with the FMA pipe half idle; and the
// module-global constant bank was shared by every context of a device.)  V lives in this CTA's shared memory now.
#define FP_ROWS 256
#define FP_KC 8
#define FP_STAGES 5
#define FP_STAGE_BYTES (FP_KC * FP_ROWS * 4)
#define FP_COMPUTE 64
#define FP_THREADS (FP_COMPUTE + 32)
template <int MP>
__global__ void __launch_bounds__(FP_THREADS, 4)
k_form_p_tma(const __grid_constant__ CUtensorMap tmA /* {n, K} FP32, box {256 rows, FP_KC columns} */, const float* __restrict__ Vp /* [Kpad][MP] */,
             long long n, int Kpad, int M, float* __restrict__ P, int n_tiles) {
    extern __shared__ __align__(1024) uint8_t fp_smem[];
    float* Vs = reinterpret_cast<float*>(fp_smem + FP_STAGES * FP_STAGE_BYTES);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(fp_smem + FP_STAGES * FP_STAGE_BYTES + (size_t)Kpad * MP * 4);
    const uint32_t smem_base = smem_u32(fp_smem);
    const uint32_t bar_full = smem_u32(s_bar), bar_empty = bar_full + 8 * FP_STAGES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < FP_STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, FP_COMPUTE / 32); }
        fence_barrier_init();
        tma_prefetch_desc(&tmA);
    }
    for (int e = threadIdx.x; e < Kpad * MP; e += FP_THREADS) Vs[e] = Vp[e];
    __syncthreads();
    const int k_stages = Kpad / FP_KC;

    if (warp == FP_COMPUTE / 32) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                for (int ks = 0; ks < k_stages; ++ks) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    const uint32_t full = bar_full + 8 * stage;
                    mbar_expect_tx(full, FP_STAGE_BYTES);                   // rows / columns past the edge arrive as zeros
#pragma unroll
                    for (int b = 0; b < FP_ROWS / 256; ++b)
                        tma_load_2d_hint(smem_base + stage * FP_STAGE_BYTES + b * (FP_KC * 256 * 4), &tmA, full,
                                         (int)((long long)tile * FP_ROWS + b * 256), ks * FP_KC, TC_EVICT_FIRST);     // A is read once
                    if (++stage == FP_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else {
        // ================= compute: 4 consecutive rows x MP columns of P per thread =================
        const int t = threadIdx.x;
        const uint32_t my = (uint32_t)(t >> 6) * (FP_KC * 256 * 4) + (uint32_t)(t & 63) * 16;       // box t / 64, rows 4 (t % 64) ..
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            float acc[4][MP];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int j = 0; j < MP; ++j) acc[r][j] = 0.0f;
            for (int ks = 0; ks < k_stages; ++ks) {
                mbar_wait(bar_full + 8 * stage, phase);
                const float* sA = reinterpret_cast<const float*>(fp_smem + stage * FP_STAGE_BYTES + my);
                const float* sV = Vs + ks * FP_KC * MP;
#pragma unroll
                for (int c = 0; c < FP_KC; ++c) {
                    const float4 d = *reinterpret_cast<const float4*>(sA + c * 256);
                    float v[MP];
#pragma unroll
                    for (int j = 0; j < MP; j += 4) {
                        const float4 v4 = *reinterpret_cast<const float4*>(sV + c * MP + j);
                        v[j] = v4.x; v[j + 1] = v4.y; v[j + 2] = v4.z; v[j + 3] = v4.w;
                    }
#pragma unroll
                    for (int j = 0; j < MP; ++j) {
                        acc[0][j] = fmaf(d.x, v[j], acc[0][j]);
                        acc[1][j] = fmaf(d.y, v[j], acc[1][j]);
                        acc[2][j] = fmaf(d.z, v[j], acc[2][j]);
                        acc[3][j] = fmaf(d.w, v[j], acc[3][j]);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_empty + 8 * stage);          // this warp is done reading the stage
                if (++stage == FP_STAGES) { stage = 0; phase ^= 1; }
            }
            const long long i = (long long)tile * FP_ROWS + 4 * t;
            if (i + 3 < n && (n & 3) == 0) {          // columns of P are n apart: 16-byte stores need n % 4 == 0
#pragma unroll
                for (int j = 0; j < MP; ++j)
                    if (j < M) __stcs(reinterpret_cast<float4*>(P + i + (long long)j * n), make_float4(acc[0][j], acc[1][j], acc[2][j], acc[3][j]));
            } else {
#pragma unroll
                for (int j = 0; j < MP; ++j)
                    if (j < M) {
#pragma unroll
                        for (int r = 0; r < 4; ++r)
                            if (i + r < n) P[i + r + (long long)j * n] = acc[r][j];
                    }
            }
        }
    }
}

template <int MP>
__global__ void __launch_bounds__(256)
k_form_p(const float* __restrict__ A, long long n, long long ld, int K, const double* __restrict__ V, const int* __restrict__ order,
         int M, float* __restrict__ P, int vs_in_smem) {
    extern __shared__ float Vs[];   // K x MP
    if (vs_in_smem) {
        for (int e = threadIdx.x; e < K * MP; e += blockDim.x) {
            const int k = e / MP, j = e % MP;
            Vs[e] = j < M ? (float)V[k + (long long)order[j] * K] : 0.0f;
        }
        __syncthreads();
    }
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float acc[MP];
#pragma unroll
    for (int j = 0; j < MP; ++j) acc[j] = 0.0f;
    for (int k = 0; k < K; ++k) {
        const float d = __ldcs(A + i + (long long)k * ld);
        if (vs_in_smem) {
#pragma unroll
            for (int j = 0; j < MP; j += 4) {
                const float4 v4 = *reinterpret_cast<const float4*>(Vs + k * MP + j);
                acc[j] = fmaf(d, v4.x, acc[j]);
                acc[j + 1] = fmaf(d, v4.y, acc[j + 1]);
                acc[j + 2] = fmaf(d, v4.z, acc[j + 2]);
                acc[j + 3] = fmaf(d, v4.w, acc[j + 3]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < MP; ++j)
                if (j < M) acc[j] = fmaf(d, (float)V[k + (long long)order[j] * K], acc[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < MP; ++j)
        if (j < M) P[i + (long long)j * n] = acc[j];
}

template <int MP>
static int launch_form_p(ssi_ctx* ctx, const float* dA, int64_t n, int64_t ld, int K, const double* dV, const int* dOrder, int M, float* dP) {
    const int Kpad = (K + FP_KC - 1) / FP_KC * FP_KC;
    const size_t v_bytes = sizeof(float) * (size_t)Kpad * MP;
    const size_t smem_tma = (size_t)FP_STAGES * FP_STAGE_BYTES + v_bytes + 2 * FP_STAGES * 8;
    if (MP <= 32 && smem_tma <= ctx->smem_optin && (ld % 4) == 0 && ((reinterpret_cast<uintptr_t>(dA) & 15) == 0) && n < (1ll << 31)) {
        PFN_ssi_encodeTiled encode = nullptr;
        SSI_TRY(ssi_tensormap_encoder(ctx, &encode));
        CUtensorMap map;
        cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)K};
        cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
        cuuint32_t box[2] = {256, FP_KC};
        cuuint32_t estr[2] = {1, 1};
        const CUresult r = encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(dA), dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return ssi_fail(ctx, SSI_ERR_CUDA, "cuTensorMapEncodeTiled (form P) failed with CUresult %d", (int)r);
        SSI_TRY(ssi_reserve(ctx, ctx->bSnap, v_bytes));
        float* stage = (float*)ctx->bSnap.p;
        k_pack_v<<<(Kpad * MP + 255) / 256, 256, 0, ctx->stream>>>(dV, dOrder, K, Kpad, M, MP, stage);
        SSI_LAUNCH_CHECK(ctx);
        const int n_tiles = (int)((n + FP_ROWS - 1) / FP_ROWS);
        SSI_CUDA(ctx, cudaFuncSetAttribute(k_form_p_tma<MP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tma));
        k_form_p_tma<MP><<<std::min(4 * ctx->sm_count, n_tiles), FP_THREADS, smem_tma, ctx->stream>>>(map, stage, n, Kpad, M, dP, n_tiles);
        SSI_LAUNCH_CHECK(ctx);
        return SSI_OK;
    }
    const size_t smem = sizeof(float) * (size_t)K * MP;
    const int in_smem = smem <= 160 * 1024;
    if (in_smem && smem > 48 * 1024)
        SSI_CUDA(ctx, cudaFuncSetAttribute(k_form_p<MP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_form_p<MP><<<(unsigned)((n + 255) / 256), 256, in_smem ? smem : 0, ctx->stream>>>(dA, n, ld, K, dV, dOrder, M, dP, in_smem);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}

// Conditioning estimate for a Gram known to eps * lambda_0 (absolute).  For each wanted direction i < M:
//   rotation into the neighbour j:  theta ~ eps lambda_0 / |lambda_i - lambda_j|, i.e. an error of
//   sqrt(lambda_i / lambda_0) * theta in column i of P relative to the largest column;
//   singular value:  |d s_i| / s_0 ~ eps sqrt(lambda_0 / lambda_i) / 2.
#define GRAM_TC_EPS 1e-7
#define GRAM_TC_RISK_MAX 1e-4   // measured: actual P error <= 0.4 x this estimate (tests/test_gpu_construct.py prints both)
__global__ void k_gram_risk(const double* __restrict__ lambda, int K, int M, double eps, double* __restrict__ out) {
    if (threadIdx.x != 0) return;
    const double l0 = lambda[0];
    double worst = 0.0;
    if (l0 > 0.0) {
        for (int i = 0; i < M && i < K; ++i) {
            const double li = lambda[i];
            if (li <= eps * eps * l0) continue;        // numerically zero direction: the column of P vanishes with it
            double gap = 1e300;
            if (i > 0) gap = fmin(gap, lambda[i - 1] - li);
            if (i + 1 < K) gap = fmin(gap, li - lambda[i + 1]);
            const double rot = gap > 0.0 ? eps * sqrt(li * l0) / gap : 1e300;
            const double sv = 0.5 * eps * sqrt(l0 / li);
            worst = fmax(worst, fmax(rot, 10.0 * sv));   // singular values are held to 1e-5 s_0, P to 1e-4
        }
    }
    *out = worst;
}

__global__ void k_singular_values(const double* __restrict__ lambda, int K, double* __restrict__ s) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < K) s[i] = sqrt(fmax(lambda[i], 0.0));
}

// ---- stages of ssi_swa_finish.  Single GPU: gram -> eigen (-> exact gram -> eigen) -> P.  Row-sharded over several
// GPUs (SURVEY 8e): every rank runs the gram stage on its row shard, the host all-reduces the K x K Gram, every rank
// runs the (replicated) eigen stage and forms the P rows of its shard.
struct swa_eig_t {
    double *dG, *dV, *dLam, *dRisk, *dNorms;
    int *dOrder, *dSweeps, *dPerm;
};
static int swa_eig_layout(ssi_ctx* ctx, int K, swa_eig_t& e) {
    // layout of bEig: G (K*K) | V (K*K) | lambda (K) | norms (K) | risk | order (K ints) | sweeps (int) | 4 counters | 3 pad | perm (K ints)
    const size_t KK = (size_t)K * K;
    SSI_TRY(ssi_reserve(ctx, ctx->bEig, sizeof(double) * (2 * KK + 2 * K + 1) + sizeof(int) * (2 * K + 8)));
    e.dG = (double*)ctx->bEig.p;
    e.dV = e.dG + KK;
    e.dLam = e.dV + KK;
    e.dNorms = e.dLam + K;
    e.dRisk = e.dNorms + K;
    e.dOrder = (int*)(e.dRisk + 1);
    e.dSweeps = e.dOrder + K;
    e.dPerm = e.dSweeps + 8;
    return SSI_OK;
}
static int swa_check_shape(ssi_ctx* ctx, int M) {
    const int K = (int)ctx->swa_K;
    if (ctx->swa_n <= 0) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_swa_begin has not been called");
    if (K < M) return ssi_fail(ctx, SSI_ERR_RANK, "deviation matrix has %d columns, cannot take M=%d", K, M);
    if (M > SSI_MAX_M) return ssi_fail(ctx, SSI_ERR_ARG, "M=%d exceeds the supported maximum %d", M, SSI_MAX_M);
    if (K > OSJ_KMAX) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "K=%d exceeds the eigen-solver limit %d", K, OSJ_KMAX);
    return SSI_OK;
}

// Gram of the local deviation columns into dG_dst (K x K doubles, device).  exact = FP64 SIMT kernel.
int ssi_swa_gram_stage(ssi_ctx* ctx, bool exact, double* dG_dst, bool* used_tensor) {
    const int64_t n = ctx->swa_n;
    const int K = (int)ctx->swa_K;
    const bool tensor = !exact && ssi_gram_tc_usable(ctx, ctx->dDev, n, ctx->swa_ld, K);
    if (used_tensor) *used_tensor = tensor;
    return ssi_gram_device(ctx, ctx->dDev, n, ctx->swa_ld, K, dG_dst, tensor, ctx->dSwaAmax);
}

// Eigen-solve of the Gram in dG_src (device; copied, not destroyed).  With `check`, evaluates the conditioning estimate
// of a tensor-core Gram and reports through *need_exact whether the Gram has to be recomputed exactly (synchronises).
int ssi_swa_eigen_stage(ssi_ctx* ctx, int M, const double* dG_src, bool check, bool* need_exact) {
    const int K = (int)ctx->swa_K;
    // every caller comes through here (single-GPU finish and the row-sharded ssi_swa_finish_gram)
    if (K > OSJ_KMAX) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "K=%d exceeds the eigen-solver limit %d", K, OSJ_KMAX);
    swa_eig_t e;
    SSI_TRY(swa_eig_layout(ctx, K, e));
    if (dG_src != e.dG)
        SSI_CUDA(ctx, cudaMemcpyAsync(e.dG, dG_src, sizeof(double) * (size_t)K * K, cudaMemcpyDeviceToDevice, ctx->stream));
    // one-sided Jacobi: on a cluster of 8 CTAs with the columns in shared memory for small K, else a cooperative grid on the
    // matrix in global memory
    unsigned* d_sync = reinterpret_cast<unsigned*>(e.dSweeps + 1);       // [sync counter | 3 rotation counters]
    SSI_CUDA(ctx, cudaMemsetAsync(d_sync, 0, 4 * sizeof(unsigned), ctx->stream));
    if (K <= OSJ_SMEM_KMAX) {
        // one warp per column pair, each column in the shared memory of the CTA that needs it next
        const int it = (K + 31) / 32;
        const size_t csm = sizeof(double) * (size_t)K * it * 32 + sizeof(int) * (size_t)K;
#define OSJC2_LAUNCH(IT_)                                                                                                       \
    do {                                                                                                                        \
        SSI_CUDA(ctx, cudaFuncSetAttribute(k_osj_cluster2<IT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csm));         \
        k_osj_cluster2<IT_><<<OSJC_CTAS, OSJC_THREADS, csm, ctx->stream>>>(e.dG, K, 60, e.dPerm, e.dSweeps);                     \
    } while (0)
        switch (it) {
            case 1: OSJC2_LAUNCH(1); break;
            case 2: OSJC2_LAUNCH(2); break;
            case 3: OSJC2_LAUNCH(3); break;
            case 4: OSJC2_LAUNCH(4); break;
            default: OSJC2_LAUNCH(5); break;
        }
#undef OSJC2_LAUNCH
    } else {
        const int np = (K + 1) / 2;
        const int grid = std::max(1, std::min(ctx->sm_count, (np * 16 + OSJ_THREADS - 1) / OSJ_THREADS));
        double* Gp = e.dG;
        int Kv = K, ms = 60;
        unsigned* sc = d_sync;
        unsigned* rc = d_sync + 1;
        int* so = e.dSweeps;
        int* pm = e.dPerm;
        void* args[] = {&Gp, &Kv, &ms, &sc, &rc, &pm, &so};
        if (grid > 1) SSI_CUDA(ctx, cudaLaunchCooperativeKernel((const void*)k_osj, dim3(grid), dim3(OSJ_THREADS), args, 0, ctx->stream));
        else SSI_CUDA(ctx, cudaLaunchKernel((const void*)k_osj, dim3(1), dim3(OSJ_THREADS), args, 0, ctx->stream));
    }
    SSI_LAUNCH_CHECK(ctx);
    k_osj_norms<<<(K * 32 + 255) / 256, 256, 0, ctx->stream>>>(e.dG, K, e.dNorms);
    SSI_LAUNCH_CHECK(ctx);
    k_osj_sort_normalise<<<(K * 32 + 255) / 256, 256, 0, ctx->stream>>>(e.dG, K, e.dNorms, e.dPerm, e.dLam, e.dOrder, e.dV);
    SSI_LAUNCH_CHECK(ctx);
    if (need_exact) *need_exact = false;
    if (!check) return SSI_OK;
    // The tensor-core Gram is accurate to ~GRAM_TC_EPS of its largest entry.  That is ample when the M wanted
    // directions are separated from their neighbours, but nearly degenerate eigenvalues rotate freely under such a
    // perturbation: estimate the damage from the spectrum and ask for the exact FP64 Gram when it could exceed the 1e-4
    // parity bar (the estimate is pessimistic: measured errors are 0.03x-0.4x of it).  One double is read back.
    k_gram_risk<<<1, 32, 0, ctx->stream>>>(e.dLam, K, M, GRAM_TC_EPS, e.dRisk);
    SSI_LAUNCH_CHECK(ctx);
    double risk = 0.0;
    SSI_CUDA(ctx, cudaMemcpyAsync(&risk, e.dRisk, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stats.gram_risk = risk;
    if (need_exact) *need_exact = (risk > GRAM_TC_RISK_MAX) && ctx->opt_gram_fp64 >= 0;
    return SSI_OK;
}

// singular values (K doubles, device) and P rows of the local shard (n x M, device) from the last eigen stage
int ssi_swa_p_stage(ssi_ctx* ctx, int M, float* dP_out, double* d_s, int* sweeps_host) {
    const int64_t n = ctx->swa_n;
    const int K = (int)ctx->swa_K;
    swa_eig_t e;
    SSI_TRY(swa_eig_layout(ctx, K, e));
    k_singular_values<<<(K + 127) / 128, 128, 0, ctx->stream>>>(e.dLam, K, d_s);
    SSI_LAUNCH_CHECK(ctx);
    int rc;
    if (M <= 4) rc = launch_form_p<4>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    else if (M <= 8) rc = launch_form_p<8>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    else if (M <= 16) rc = launch_form_p<16>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    else if (M <= 20) rc = launch_form_p<20>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    else if (M <= 24) rc = launch_form_p<24>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    else if (M <= 32) rc = launch_form_p<32>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    else if (M <= 48) rc = launch_form_p<48>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    else rc = launch_form_p<64>(ctx, ctx->dDev, n, ctx->swa_ld, K, e.dV, e.dOrder, M, dP_out);
    if (rc != SSI_OK) return rc;
    if (sweeps_host) SSI_CUDA(ctx, cudaMemcpyAsync(sweeps_host, e.dSweeps, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stats.last_bytes = 4.0 * (double)n * K * 2 + 4.0 * (double)n * M;
    ctx->stats.last_flops = 2.0 * (double)n * K * K + 2.0 * (double)n * K * M;
    ctx->stats.last_units = 0;
    return SSI_OK;
}

// Gram + eigen + P for the collected deviation matrix; leaves P (n x M) in dP_out (device),
// singular values (K doubles) in d_s.
int ssi_swa_factor_device(ssi_ctx* ctx, int M, float* dP_out, double* d_s, int* sweeps_host) {
    SSI_TRY(swa_check_shape(ctx, M));
    if (ctx->swa_n < M) return ssi_fail(ctx, SSI_ERR_RANK, "deviation matrix is %lld x %d, cannot take M=%d columns", (long long)ctx->swa_n, (int)ctx->swa_K, M);
    swa_eig_t e;
    SSI_TRY(swa_eig_layout(ctx, (int)ctx->swa_K, e));
    ctx->stats.gram_risk = 0.0;
    for (cudaEvent_t& ev : ctx->ev_stage)
        if (!ev) SSI_CUDA(ctx, cudaEventCreate(&ev));
    bool tensor = false, need_exact = false;
    cudaEventRecord(ctx->ev_stage[0], ctx->stream);
    SSI_TRY(ssi_swa_gram_stage(ctx, ctx->opt_gram_fp64 > 0, e.dG, &tensor));
    cudaEventRecord(ctx->ev_stage[1], ctx->stream);
    SSI_TRY(ssi_swa_eigen_stage(ctx, M, e.dG, tensor, &need_exact));
    ctx->stats.gram_path = tensor ? 2 : 1;
    if (need_exact) {        // the stage times then describe the exact pass
        cudaEventRecord(ctx->ev_stage[0], ctx->stream);
        SSI_TRY(ssi_swa_gram_stage(ctx, true, e.dG, nullptr));
        cudaEventRecord(ctx->ev_stage[1], ctx->stream);
        SSI_TRY(ssi_swa_eigen_stage(ctx, M, e.dG, false, nullptr));
        ctx->stats.gram_path = 3;
    }
    cudaEventRecord(ctx->ev_stage[2], ctx->stream);
    const int rc = ssi_swa_p_stage(ctx, M, dP_out, d_s, sweeps_host);
    cudaEventRecord(ctx->ev_stage[3], ctx->stream);
    ctx->stage_pending = true;
    return rc;
}
