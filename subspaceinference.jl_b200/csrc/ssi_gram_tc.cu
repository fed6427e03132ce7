// ssi_gram_tc.cu — K6 on the tensor cores: G = A'A for a tall-skinny n x K FP32 matrix (K <= 128).
//
// Replaces the factorisation work inside psvd(A) (src/subspace_construction.jl:63) for the shapes the
// construction path produces (K = number of deviation columns, n ~ 1e7): one pass over A at HBM speed.
//
//   * A is column-major n x K == K rows of length n.  A TMA box {64 rows-of-A, K8 columns-of-A} (K8 = K rounded up to 8)
//     lands in a RAW ring as a plain [K8][64] FP32 tile: 256 contiguous bytes per column.  The segment length matters
//     more than anything else here: a tile gathers one segment from each of the K columns (K different DRAM pages), and
//     TMA gathers of 128-byte segments top out at 4.6 TB/s on this part whatever the depth of the ring, 256-byte ones
//     reach 7.0 TB/s (profiles/explore/tma_gather.cu, profiles/r02_explore_tma_gather.txt) -- the 32-row tiles of the
//     first tensor-core version sat at 3.7 TB/s for that reason.
//   * eight converter warps split every raw tile between them (item = one float4 = 4 rows of one column; a warp reads 512
//     contiguous bytes, conflict-free) and write the operand of tcgen05.mma kind::f16: two FP16 planes H = fp16(s x) and
//     L = fp16(s x - H), [128][64] halves each = 128-byte rows, K-major SWIZZLE_128B, H and L back to back (32 KB per
//     operand slot).  Every converter warp walks the tiles in order, so no warp can be two phases ahead of a barrier (an
//     mbarrier parity wait cannot tell phase p from phase p + 2) and the ring depths are free: 3 operand slots, up to 4
//     raw slots.  s = 2^j puts the largest |A| (tracked by k_swa_push, one atomicMax per block) at 2^14, so H cannot
//     overflow and H + L carries 22 bits of every value that matters.
//   * one thread issues, per 16 rows of A,  [HH | HL] += H [H ; L]'  (the B operand spans the H tile and the L tile
//     behind it, so H is fetched once; FP32 accumulators in TMEM).  G = HH + HL + HL' drops only L L', 2^-24 relative.
//     (BF16 planes were tried: their L L' term is 2^-18 of H H' and all-positive on the diagonal, so it must be kept,
//     and accumulated next to H H' in FP32 a third of it was truncated away -- 3e-7 of lambda_0, measured.  Loading A
//     with plain 16-byte loads straight into registers -- no raw ring, 72 KB instead of 124 KB of shared-memory traffic per
//     tile -- was tried twice: 1.5 ms with one tile in flight per warp, 1.31 ms with sixteen converter warps keeping two
//     tiles ahead in three register buffers (53 KB per SM in flight): both bound by the latency of their own loads, where
//     the TMA ring runs at 0.94 ms.)
//   * FP32 accumulation in the tensor core truncates, so accumulators are drained every `chunk` tiles (1024 rows) into
//     per-CTA FP64 partials (each thread owns its elements: plain load-add-store, no atomics) and reset; a final
//     kernel sums the per-CTA partials in fixed order, symmetrises and undoes the scale.
//   * shared-memory traffic per tile (K = 100): 26 KB TMA write + 26 KB converter reads + 26 KB plane writes + 46 KB of
//     operand fetches by the four MMAs = 124 KB per 25.6 KB of A: at 128 B/clk that is ~1000 cycles per tile and SM, about
//     the HBM time of the tile (950 cycles at 6.5 TB/s) -- the two pipes are balanced, neither has slack.
//
// Roles (448 threads): warp 0 TMA producer, warp 1 MMA issuer + TMEM allocator, warps 2-9 converters, warps 10-13 drain.
// TMEM: 2 x (HH | HL) x 128 columns = 512.
#include "ssi_common.cuh"
#include "ssi_ptx.cuh"

#include <cuda_fp16.h>
#include <algorithm>

#define GT_ROWS 64                   // rows of A per tile (256 contiguous bytes per column)
#define GT_OP_BYTES (2 * 128 * 128)  // H | L: [128 columns of A][64 rows] FP16 each, 128-byte rows
#define GT_OPS 3                     // operand slots
#define GT_RAW_MAX 4                 // raw slots (fewer when K8 * 256 bytes do not fit four times)
#define GT_CONV 8                    // converter warps
#define GT_THREADS (64 + 32 * GT_CONV + 128)
#define GT_OFF_BAR (GT_OPS * GT_OP_BYTES)                 // operand slots first (1024-byte aligned for SWIZZLE_128B)
#define GT_NBAR (2 * GT_RAW_MAX + 2 * GT_OPS + 4)
#define GT_OFF_RAW (GT_OFF_BAR + 256)                     // barriers + TMEM slot, then the raw ring
#define GT_SMEM_MAX (227 * 1024)

struct gram_tc_params {
    const float* amax;         // device: largest |A| (from k_swa_push), defines the power-of-two scale of the FP16 planes
    long long n;
    int K, NP;                 // NP = K rounded up to 16 (MMA N)
    int K8, n_raw, raw_bytes;  // K rounded up to 8 (TMA box), raw slots and their size (K8 * 256)
    long long tiles_total;     // ceil(n / 64)
    long long tiles_per_cta;
    int chunk;                 // tiles per FP32 accumulation chunk
    double* partial;           // [grid][2][NP][128]  (pass, column b, row a)
};

__global__ void __launch_bounds__(GT_THREADS, 1)
k_gram_tc(const __grid_constant__ CUtensorMap tmA, const gram_tc_params p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    // barriers: raw_full[R] raw_empty[R] op_full[O] op_empty[O] tfull[2] tempty[2]
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + GT_OFF_BAR);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + GT_NBAR);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_rfull = smem_u32(s_bar), bar_rempty = bar_rfull + 8 * GT_RAW_MAX;
    const uint32_t bar_ofull = bar_rempty + 8 * GT_RAW_MAX, bar_oempty = bar_ofull + 8 * GT_OPS;
    const uint32_t bar_tfull = bar_oempty + 8 * GT_OPS, bar_tempty = bar_tfull + 16;

    if (threadIdx.x == 0) {
        if (smem_base & 1023u) { printf("ssi_gram_tc: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
        for (int s = 0; s < p.n_raw; ++s) { mbar_init(bar_rfull + 8 * s, 1); mbar_init(bar_rempty + 8 * s, GT_CONV); }
        for (int s = 0; s < GT_OPS; ++s) { mbar_init(bar_ofull + 8 * s, GT_CONV); mbar_init(bar_oempty + 8 * s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 128); }
        fence_barrier_init();
        tma_prefetch_desc(&tmA);
    }
    // operand rows >= K8 (columns of A that do not exist) are never written by the converters: zero them once
    for (int i = threadIdx.x; i < GT_OPS * 2 * (128 - p.K8) * 8; i += GT_THREADS) {
        const int chunk = i & 7, r = (i >> 3) % (128 - p.K8), pl = (i >> 3) / (128 - p.K8);       // pl = slot * 2 + plane
        *reinterpret_cast<uint4*>(smem + (size_t)pl * (128 * 128) + (size_t)(p.K8 + r) * 128 + chunk * 16) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async();
    if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    const long long t_begin = (long long)blockIdx.x * p.tiles_per_cta;
    const long long t_end = min(p.tiles_total, t_begin + p.tiles_per_cta);
    const long long my_tiles = max(0ll, t_end - t_begin);
    const long long n_chunks = (my_tiles + p.chunk - 1) / p.chunk;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (long long t = t_begin; t < t_end; ++t) {
                mbar_wait(bar_rempty + 8 * stage, phase ^ 1);          // every converter warp is done with this raw slot
                mbar_expect_tx(bar_rfull + 8 * stage, p.raw_bytes);
                // A is streamed exactly once: do not let it evict the FP64 partials from L2
                tma_load_2d_hint(smem_base + GT_OFF_RAW + stage * p.raw_bytes, &tmA, bar_rfull + 8 * stage, (int)(t * GT_ROWS), 0, TC_EVICT_FIRST);
                if (++stage == p.n_raw) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            // one MMA per k-step: the B operand spans the H tile (128 rows; rows >= K are zero) and the first NP rows of the
            // L tile behind it, so D = H [H ; L]^T = [HH (columns 0..127) | HL (columns 128..128+NP)] and the A operand (H)
            // is fetched from shared memory once instead of twice
            const uint32_t idesc = umma_idesc_f16(128 + p.NP, UMMA_FMT_F16, UMMA_FMT_F16);
            int stage = 0;
            uint32_t phase = 0;
            long long t = 0;
            for (long long c = 0; c < n_chunks; ++c) {
                const uint32_t ab = (uint32_t)(c & 1), aphase = (uint32_t)((c >> 1) & 1);
                mbar_wait(bar_tempty + 8 * ab, aphase ^ 1);
                tc_fence_after();
                const uint32_t d_acc = tmem_base + ab * 256;
                const long long c_end = min(my_tiles, (c + 1) * (long long)p.chunk);
                for (bool first = true; t < c_end; ++t, first = false) {
                    mbar_wait(bar_ofull + 8 * stage, phase);            // H and L tiles are ready
                    tc_fence_after();
                    const uint64_t dh = umma_desc_sw128(smem_base + stage * GT_OP_BYTES);
#pragma unroll
                    for (int k = 0; k < GT_ROWS / 16; ++k) {
                        const uint64_t ko = (uint64_t)(k * 32 >> 4);    // 16 FP16 = 32 bytes per k-step inside the 128-byte row
                        umma_bf16(d_acc, dh + ko, dh + ko, idesc, !(first && k == 0));
                    }
                    umma_commit(bar_oempty + 8 * stage);
                    if (++stage == GT_OPS) { stage = 0; phase ^= 1; }
                }
                umma_commit(bar_tfull + 8 * ab);
            }
        }
    } else if (warp < 2 + GT_CONV) {
        // ================= converters: raw FP32 tile -> FP16 planes H | L in the K-major SWIZZLE_128B operand layout =================
        const int cw = warp - 2;
        const float amax = *p.amax;
        const float sc = (amax > 0.0f && amax < 3.0e38f) ? scalbnf(1.0f, max(-100, min(100, 14 - ilogbf(amax)))) : 1.0f;
        // item i = (column i / 16 of A, rows 4 (i % 16) .. + 3): a warp reads 32 consecutive float4 = two whole columns of the
        // raw tile and writes two whole 128-byte rows of each plane (8 bytes per lane), both conflict-free
        const int items = p.K8 * 16;
        int rs = 0, os = 0;
        uint32_t rphase = 0, ophase = 0;
        for (long long t = 0; t < my_tiles; ++t) {
            mbar_wait(bar_rfull + 8 * rs, rphase);
            mbar_wait(bar_oempty + 8 * os, ophase ^ 1);       // the MMAs that read this operand slot have retired
            const uint8_t* raw = smem + GT_OFF_RAW + (size_t)rs * p.raw_bytes;
            uint8_t* opH = smem + (size_t)os * GT_OP_BYTES;
            uint8_t* opL = opH + 128 * 128;
#pragma unroll 4
            for (int i = cw * 32 + lane; i < items; i += GT_CONV * 32) {
                const int c = i >> 4, q = i & 15;
                const float4 x = *reinterpret_cast<const float4*>(raw + (size_t)i * 16);
                const float v0 = x.x * sc, v1 = x.y * sc, v2 = x.z * sc, v3 = x.w * sc;
                const __half2 h01 = __floats2half2_rn(v0, v1), h23 = __floats2half2_rn(v2, v3);
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                const __half2 l01 = __floats2half2_rn(v0 - f01.x, v1 - f01.y), l23 = __floats2half2_rn(v2 - f23.x, v3 - f23.y);
                // SWIZZLE_128B: the 16-byte chunk index is XORed with the row index inside the 8-row atom
                const uint32_t off = (uint32_t)c * 128 + (uint32_t)(((q >> 1) ^ (c & 7)) << 4) + (uint32_t)((q & 1) << 3);
                *reinterpret_cast<uint2*>(opH + off) = make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
                *reinterpret_cast<uint2*>(opL + off) = make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
            }
            fence_proxy_async();                   // generic-proxy writes -> visible to the tensor core (async proxy)
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(bar_ofull + 8 * os);
                mbar_arrive(bar_rempty + 8 * rs);
            }
            if (++rs == p.n_raw) { rs = 0; rphase ^= 1; }
            if (++os == GT_OPS) { os = 0; ophase ^= 1; }
        }
    } else {
        // ================= drain: TMEM chunk sums -> FP64 per-CTA partials =================
        // The partials (grid x 2 x NP x 128 doubles, ~34 MB at K = 100) are read-modify-written once per chunk;
        // they are tagged evict_last so that they stay in the 126 MB L2 while A streams through (evict_first).
        const int q = warp & 3;                    // TMEM lane quarter
        const int a = q * 32 + lane;               // row of the accumulator = column a of A
        const uint64_t pol = l2_policy_evict_last();
        double* part = p.partial + (long long)blockIdx.x * 2 * p.NP * 128;
        for (long long c = 0; c < n_chunks; ++c) {
            const uint32_t ab = (uint32_t)(c & 1), aphase = (uint32_t)((c >> 1) & 1);
            mbar_wait(bar_tfull + 8 * ab, aphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ab * 256;
#pragma unroll 1
            for (int pass = 0; pass < 2; ++pass) {
                // HH is symmetric: this warp's rows [32q, 32q+32) only need the column blocks that reach the diagonal
#pragma unroll 1
                for (int b0 = (pass == 0 ? q * 32 : 0); b0 < p.NP; b0 += 16) {
                    uint32_t v[16];
                    tmem_ld16(taddr + pass * 128 + b0, v);
                    tmem_ld_wait();
                    double* dst = part + ((long long)pass * p.NP + b0) * 128 + a;
                    if (c == 0) {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) st_f64_hint(dst + jj * 128, (double)__uint_as_float(v[jj]), pol);
                    } else {
                        double old[16];
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) old[jj] = ld_f64_hint(dst + jj * 128, pol);
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) st_f64_hint(dst + jj * 128, old[jj] + (double)__uint_as_float(v[jj]), pol);
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(bar_tempty + 8 * ab);
        }
        if (n_chunks == 0) {                       // a CTA without rows still owns a (zero) partial
            for (int e = 0; e < 2 * p.NP; ++e) part[(long long)e * 128 + a] = 0.0;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// stage 1: S[e] = sum over CTAs of partial[c][e], fixed order, fully coalesced (e over 2 x NP x 128)
__global__ void __launch_bounds__(128)
k_gram_tc_sum(const double* __restrict__ partial, int grid, int elems, int NP, double* __restrict__ S) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= elems) return;
    // HH entries (pass 0) left of a warp's diagonal block are never written by the drain warps (and never read by stage 2)
    const int row = e & 127, col = e >> 7;
    if (col < NP && col < (row & ~31)) { S[e] = 0.0; return; }
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int c = 0;
    for (; c + 4 <= grid; c += 4) {
        s0 += partial[(long long)c * elems + e];
        s1 += partial[(long long)(c + 1) * elems + e];
        s2 += partial[(long long)(c + 2) * elems + e];
        s3 += partial[(long long)(c + 3) * elems + e];
    }
    for (; c < grid; ++c) s0 += partial[(long long)c * elems + e];
    S[e] = (s0 + s1) + (s2 + s3);
}
// stage 2: G[a,b] = HH[min,max] + HL[a][b] + HL[b][a]   (S is [pass][column][row 128])
__global__ void k_gram_tc_sym(const double* __restrict__ S, int K, int NP, const float* __restrict__ amax, double* __restrict__ G) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= K * K) return;
    const int a = e % K, b = e / K;
    const int lo = min(a, b), hi = max(a, b);
    const float am = *amax;
    const int j = (am > 0.0f && am < 3.0e38f) ? max(-100, min(100, 14 - ilogbf(am))) : 0;      // the planes carried 2^j A
    G[a + (long long)b * K] = scalbn(S[(long long)hi * 128 + lo] + S[((long long)NP + b) * 128 + a] + S[((long long)NP + a) * 128 + b], -2 * j);
}

bool ssi_gram_tc_usable(const ssi_ctx* ctx, const float* dA, int64_t n, int64_t ld, int K) {
    return K >= 1 && K <= 128 && (ld % 4) == 0 && n >= (1 << 16) && ((reinterpret_cast<uintptr_t>(dA) & 15) == 0) &&
           n < (1ll << 31) && ctx->opt_gram_fp64 <= 0;
}

int ssi_gram_tc_device(ssi_ctx* ctx, const float* dA, int64_t n, int64_t ld, int K, double* dG, const float* d_amax) {
    PFN_ssi_encodeTiled encode = nullptr;
    SSI_TRY(ssi_tensormap_encoder(ctx, &encode));
    CUtensorMap map;
    cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)K};
    cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
    const int K8 = (K + 7) / 8 * 8;
    cuuint32_t box[2] = {GT_ROWS, (cuuint32_t)K8};
    cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(dA), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return ssi_fail(ctx, SSI_ERR_CUDA, "cuTensorMapEncodeTiled (gram) failed with CUresult %d", (int)r);

    gram_tc_params p{};
    p.amax = d_amax;
    p.n = n;
    p.K = K;
    p.NP = (K + 15) / 16 * 16;
    p.K8 = K8;
    p.raw_bytes = K8 * GT_ROWS * (int)sizeof(float);
    p.n_raw = std::min(GT_RAW_MAX, (GT_SMEM_MAX - GT_OFF_RAW) / p.raw_bytes);
    const int smem_bytes = GT_OFF_RAW + p.n_raw * p.raw_bytes;
    p.tiles_total = (n + GT_ROWS - 1) / GT_ROWS;
    const int grid = (int)std::min<long long>(ctx->sm_count, p.tiles_total);
    p.tiles_per_cta = (p.tiles_total + grid - 1) / grid;
    p.chunk = 16;                                                       // 1024 rows per FP32 chunk
    const int elems = 2 * p.NP * 128;
    SSI_TRY(ssi_reserve(ctx, ctx->bGram, sizeof(double) * (size_t)(grid + 1) * elems));
    p.partial = (double*)ctx->bGram.p;
    double* dS = p.partial + (size_t)grid * elems;
    SSI_CUDA(ctx, cudaFuncSetAttribute(k_gram_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    ssi_kt_begin(ctx);
    k_gram_tc<<<grid, GT_THREADS, smem_bytes, ctx->stream>>>(map, p);
    SSI_LAUNCH_CHECK(ctx);
    ssi_kt_end(ctx);
    k_gram_tc_sum<<<(elems + 127) / 128, 128, 0, ctx->stream>>>(p.partial, grid, elems, p.NP, dS);
    SSI_LAUNCH_CHECK(ctx);
    k_gram_tc_sym<<<(K * K + 255) / 256, 256, 0, ctx->stream>>>(dS, K, p.NP, d_amax, dG);
    SSI_LAUNCH_CHECK(ctx);
    return SSI_OK;
}
