// ssi_gemm_tc.cu — the strided FP32 GEMM of the gradient and training paths on the tensor cores.
//
// C(o, j) = epi( sum_k A(o, k) B(k, j) ) for a batch of independent problems: the contraction every step of the reverse
// pass (src/space_inference.jl:107 through the AD backends of src/libs.jl:23-34) and of the mini-batch training step
// (src/subspace_construction.jl:39-43) is made of -- forward W H, weight gradient delta H', back-propagated delta W' delta --
// with FP32 operands in whatever orientation the Julia column-major layout gives them.  The SIMT kernel in ssi_gemm.cu
// (64x64 tiles, ~17 TFLOP/s) made a gradient on the wide MLP cost 100x a density evaluation.  This one keeps the
// operands FP32 in global memory and does the split on the fly, the way the Gram kernel does:
//
//   * warp 0 lands raw FP32 tiles with TMA: A 128 (o) x 32 (k), B 256 (j) x 32 (k), either orientation (k-fast tiles
//     arrive as [rows][32 k] with 128-byte swizzle, o- / j-fast tiles as [32 k][rows]); edges are zero-filled by TMA;
//   * eight converter warps split every raw tile into two 16-bit planes in the K-major SWIZZLE_64B operand layout
//     (transposing the o- / j-fast tiles on the way; both access patterns are conflict-free): FP16 planes
//     hi = fp16(s x), lo = fp16(s x - hi) with one power-of-two scale s per operand AND BATCH that puts that batch's
//     largest magnitude at 2^14 (a strided absmax pre-pass, k_gemm_absmax; per batch so that a sample's result cannot
//     depend on what else is in the launch): 11 + 11 bits for everything within 2^-17 of the largest element (BF16 planes,
//     8 + 8 bits, left 5e-5 of the gradient norm on the test shapes: DESIGN.md 4.5).  The orientation is a template parameter;
//   * one thread issues  D += Al Bh' + Ah Bl' + Ah Bh'  (tcgen05.mma kind::f16, M = 128, N = 256, FP32 accumulators in
//     TMEM, two accumulator buffers).  The forward layers (bias + activation epilogue) keep the two small terms in an
//     accumulator of their own: they are 2^-11 of the large term, and added into the same truncating accumulator they
//     lose the bits below the running sum's ulp -- most of what the lo planes carry.  That, not the length of the
//     accumulation, was the 3.7e-5 of the gradient norm the first version of this kernel showed on the wide network
//     (FP32 FMA chains: 1.8e-5; with the split: 1.35e-5).  It costs the double buffering of those launches (+7 % on the
//     whole gradient), so the backward GEMMs, whose results are sums the error averages out of, do without;
//   * four epilogue warps drain an accumulator every `chunk` k-blocks (1024 k): the tensor core's FP32 accumulation
//     truncates, so a long contraction (the weight gradient runs over all N datapoints) is summed in FP32 through the
//     output tile itself (each tile has one owner: plain read-add-write), and the last chunk applies the epilogue
//     (bias + activation, or the activation derivative taken from the layer's output).
//   * persistent grid; tiles that share the B panel (the big operand: activations or deltas) run side by side so that it
//     is read from HBM once.
//
// Shared memory per k-block: 48 KB raw + 48 KB of plane writes + 48 KB converter reads + 72 KB operand fetches: the
// kernel is bound by the shared-memory pipe, not by the tensor pipe (DESIGN.md 4.5).  Requirements (else the caller
// falls back to the SIMT kernel): 16-byte aligned bases and strides, c_so == 1, no split-K, at least 1.6e7 multiply-adds per
// batch (the choice never depends on the number of batches).
#include "ssi_common.cuh"
#include "ssi_ptx.cuh"
#include "ssi_gemm.cuh"

#include <cuda_fp16.h>
#include <algorithm>

#define GX_BM 128
#define GX_BN 256
#define GX_BK 32
#define GX_RAW_A (GX_BM * GX_BK * 4)                 // 16 KB
#define GX_RAW_B (GX_BN * GX_BK * 4)                 // 32 KB
#define GX_RAW_STAGE (GX_RAW_A + GX_RAW_B)
#define GX_OP_A (GX_BM * GX_BK * 2)                  // 8 KB per plane
#define GX_OP_B (GX_BN * GX_BK * 2)                  // 16 KB per plane
#define GX_OP_STAGE (2 * GX_OP_A + 2 * GX_OP_B)      // Ah | Al | Bh | Bl
#define GX_STAGES 2
#define GX_CONV 8
#define GX_THREADS (64 + 32 * GX_CONV + 128)
#define GX_OFF_OP (GX_STAGES * GX_RAW_STAGE)
#define GX_OFF_BAR (GX_OFF_OP + GX_STAGES * GX_OP_STAGE)
#define GX_NBAR (4 * GX_STAGES + 4)
#define GX_SMEM (GX_OFF_BAR + GX_NBAR * 8 + 16)
#define GX_EPW 16                                    // output columns per epilogue pass (= one tcgen05.ld of 16 columns)

struct gemm_tc_params {
    const float* amaxA;          // device: largest |A| per batch (one entry when A is shared).  Per batch, not per
    const float* amaxB;          // launch: a sample's result must not depend on which other samples share its launch
    float* C; long long c_sj, c_sb;
    int O, J;
    int n_to, n_tj;
    long long n_work;
    int n_kb, chunk;             // k-blocks of 32; k-blocks per accumulation chunk
    int a_kfast, b_kfast;
    int a_batched, b_batched;
    int split_acc;               // 1: small terms (Al Bh' + Ah Bl') and the large term in separate accumulators (no double buffering)
    int epi, act;
    const float* bias; long long bias_sb;
    const float* Hprev; long long h_sb;
};

// tanh / sigmoid out of line: the epilogue is unrolled 32 wide, and their inline expansions alone were several thousand
// instructions of a kernel whose other warps stall on instruction fetch
__device__ __noinline__ float gx_act_slow(float v, int act) { return ssi_act(v, act); }
__device__ __forceinline__ float gx_act(float v, int act) {
    if (act == SSI_ACT_RELU) return fmaxf(v, 0.0f);
    if (act == SSI_ACT_TANH || act == SSI_ACT_SIGMOID) return gx_act_slow(v, act);
    return v;
}
// power-of-two scale that puts mx in [2^14, 2^15)
__device__ __forceinline__ int gx_scale_exp(float mx) {
    return (mx > 0.0f && mx < 3.0e38f) ? max(-100, min(100, 14 - ilogbf(mx))) : 0;
}
// eight consecutive k of one row -> one 16-byte chunk of each plane
__device__ __forceinline__ void gx_split8(const float v[8], uint4& hi, uint4& lo, float sc) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float a = v[2 * i] * sc, b = v[2 * i + 1] * sc;
        const __half2 hh = __floats2half2_rn(a, b);
        h[i] = *reinterpret_cast<const uint32_t*>(&hh);
        const float2 f = __half22float2(hh);
        const __half2 lh = __floats2half2_rn(a - f.x, b - f.y);
        l[i] = *reinterpret_cast<const uint32_t*>(&lh);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// raw FP32 tile (ROWS x 32 k) -> planes H, L ([ROWS][32] FP16, 64-byte rows, SWIZZLE_64B); ct = converter thread 0..255
template <int ROWS, bool KFAST>
__device__ __forceinline__ void gx_convert(const uint8_t* __restrict__ raw, uint8_t* __restrict__ H, uint8_t* __restrict__ L, int ct, float sc) {
#pragma unroll 2
    for (int i = ct; i < ROWS * 4; i += GX_CONV * 32) {
        int r, q;
        float v[8];
        if (KFAST) {
            // [ROWS][32 k], 128-byte rows, TMA SWIZZLE_128B (16-byte chunk ^ row % 8): a quarter warp reads two whole rows
            r = i >> 2; q = i & 3;
            const float4 x0 = *reinterpret_cast<const float4*>(raw + r * 128 + (((2 * q) ^ (r & 7)) << 4));
            const float4 x1 = *reinterpret_cast<const float4*>(raw + r * 128 + (((2 * q + 1) ^ (r & 7)) << 4));
            v[0] = x0.x; v[1] = x0.y; v[2] = x0.z; v[3] = x0.w; v[4] = x1.x; v[5] = x1.y; v[6] = x1.z; v[7] = x1.w;
        } else {
            // [32 k][ROWS], plain: consecutive lanes take consecutive rows of the operand (columns of the raw tile)
            r = i & (ROWS - 1); q = i / ROWS;
            const float* src = reinterpret_cast<const float*>(raw) + (8 * q) * ROWS + r;
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = src[e * ROWS];
        }
        uint4 hi, lo;
        gx_split8(v, hi, lo, sc);
        const uint32_t off = (uint32_t)r * 64u + (uint32_t)((q ^ ((r >> 1) & 3)) << 4);      // SWIZZLE_64B: chunk ^ bits [7, 9) of the address
        *reinterpret_cast<uint4*>(H + off) = hi;
        *reinterpret_cast<uint4*>(L + off) = lo;
    }
}

// AK / BK: the raw tiles of A / B are k-fast
template <bool AK, bool BK>
__global__ void __launch_bounds__(GX_THREADS, 1)
k_gemm_tc(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const gemm_tc_params p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + GX_OFF_BAR);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + GX_NBAR);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_rfull = smem_u32(s_bar), bar_rempty = bar_rfull + 8 * GX_STAGES;
    const uint32_t bar_ofull = bar_rempty + 8 * GX_STAGES, bar_oempty = bar_ofull + 8 * GX_STAGES;
    const uint32_t bar_tfull = bar_oempty + 8 * GX_STAGES, bar_tempty = bar_tfull + 16;

    if (threadIdx.x == 0) {
        if (smem_base & 1023u) { printf("ssi_gemm_tc: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
        for (int s = 0; s < GX_STAGES; ++s) {
            mbar_init(bar_rfull + 8 * s, 1); mbar_init(bar_rempty + 8 * s, GX_CONV);
            mbar_init(bar_ofull + 8 * s, GX_CONV); mbar_init(bar_oempty + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 128); }
        fence_barrier_init();
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
    }
    if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    const int n_chunks = (p.n_kb + p.chunk - 1) / p.chunk;
    const long long tiles_per_batch = (long long)p.n_to * p.n_tj;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (long long w = blockIdx.x; w < p.n_work; w += gridDim.x) {
                const int b = (int)(w / tiles_per_batch);
                const int rem = (int)(w - (long long)b * tiles_per_batch);
                const int tj = rem / p.n_to, to = rem - tj * p.n_to;
                const int ab = p.a_batched ? b : 0, bb = p.b_batched ? b : 0;
                for (int kb = 0; kb < p.n_kb; ++kb) {
                    mbar_wait(bar_rempty + 8 * stage, phase ^ 1);
                    const uint32_t full = bar_rfull + 8 * stage;
                    mbar_expect_tx(full, GX_RAW_STAGE);
                    const uint32_t dA = smem_base + stage * GX_RAW_STAGE, dB = dA + GX_RAW_A;
                    if (AK) tma_load_3d(dA, &tmA, full, kb * GX_BK, to * GX_BM, ab);
                    else tma_load_3d(dA, &tmA, full, to * GX_BM, kb * GX_BK, ab);
                    if (BK) tma_load_3d(dB, &tmB, full, kb * GX_BK, tj * GX_BN, bb);
                    else tma_load_3d(dB, &tmB, full, tj * GX_BN, kb * GX_BK, bb);
                    if (++stage == GX_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_f16(GX_BN, UMMA_FMT_F16, UMMA_FMT_F16);
            int stage = 0;
            uint32_t phase = 0;
            unsigned cidx = 0;
            for (long long w = blockIdx.x; w < p.n_work; w += gridDim.x) {
                int kb = 0;
                for (int c = 0; c < n_chunks; ++c, ++cidx) {
                    // split_acc: both buffers belong to this chunk (large term in 0, small terms in 1), each used every chunk
                    const uint32_t ab = p.split_acc ? 0u : (cidx & 1u), aphase = p.split_acc ? (cidx & 1u) : ((cidx >> 1) & 1u);
                    mbar_wait(bar_tempty + 8 * ab, aphase ^ 1);
                    if (p.split_acc) mbar_wait(bar_tempty + 8, aphase ^ 1);
                    tc_fence_after();
                    const uint32_t d_acc = tmem_base + ab * 256;
                    const uint32_t d_small = p.split_acc ? tmem_base + 256 : d_acc;
                    const int kb_end = min(p.n_kb, (c + 1) * p.chunk);
                    for (bool first = true; kb < kb_end; ++kb) {
                        mbar_wait(bar_ofull + 8 * stage, phase);
                        tc_fence_after();
                        const uint32_t op = smem_base + GX_OFF_OP + stage * GX_OP_STAGE;
                        const uint64_t dAh = umma_desc_sw64(op), dAl = umma_desc_sw64(op + GX_OP_A);
                        const uint64_t dBh = umma_desc_sw64(op + 2 * GX_OP_A), dBl = umma_desc_sw64(op + 2 * GX_OP_A + GX_OP_B);
#pragma unroll
                        for (int ks = 0; ks < GX_BK / 16; ++ks) {
                            const uint64_t ko = (uint64_t)(ks * 32 >> 4);      // 16 FP16 = 32 bytes per k-step inside the 64-byte row
                            umma_bf16(d_small, dAl + ko, dBh + ko, idesc, first ? 0u : 1u);
                            umma_bf16(d_small, dAh + ko, dBl + ko, idesc, 1u);
                            umma_bf16(d_acc, dAh + ko, dBh + ko, idesc, (first && p.split_acc) ? 0u : 1u);
                            first = false;
                        }
                        umma_commit(bar_oempty + 8 * stage);
                        if (++stage == GX_STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(bar_tfull + 8 * ab);
                }
            }
        }
    } else if (warp < 2 + GX_CONV) {
        // ================= converters =================
        const int ct = threadIdx.x - 64;
        int stage = 0;
        uint32_t phase = 0;
        for (long long w = blockIdx.x; w < p.n_work; w += gridDim.x) {
            const int b = (int)(w / tiles_per_batch);
            const float scA = scalbnf(1.0f, gx_scale_exp(p.amaxA[p.a_batched ? b : 0]));
            const float scB = scalbnf(1.0f, gx_scale_exp(p.amaxB[p.b_batched ? b : 0]));
            for (int kb = 0; kb < p.n_kb; ++kb) {
                mbar_wait(bar_rfull + 8 * stage, phase);
                mbar_wait(bar_oempty + 8 * stage, phase ^ 1);          // the MMAs that read this operand slot have retired
                const uint8_t* raw = smem + stage * GX_RAW_STAGE;
                uint8_t* op = smem + GX_OFF_OP + stage * GX_OP_STAGE;
                gx_convert<GX_BM, AK>(raw, op, op + GX_OP_A, ct, scA);
                gx_convert<GX_BN, BK>(raw + GX_RAW_A, op + 2 * GX_OP_A, op + 2 * GX_OP_A + GX_OP_B, ct, scB);
                fence_proxy_async();                   // generic-proxy writes -> visible to the tensor core (async proxy)
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(bar_ofull + 8 * stage);
                    mbar_arrive(bar_rempty + 8 * stage);
                }
                if (++stage == GX_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // ================= epilogue: TMEM -> (running FP32 sum in C) -> epilogue -> C =================
        const int q = warp & 3;                    // TMEM lane quarter
        unsigned cidx = 0;
        for (long long w = blockIdx.x; w < p.n_work; w += gridDim.x) {
            const int b = (int)(w / tiles_per_batch);
            const int rem = (int)(w - (long long)b * tiles_per_batch);
            const int tj = rem / p.n_to, to = rem - tj * p.n_to;
            const int o = to * GX_BM + q * 32 + lane;
            float* crow = p.C + (long long)b * p.c_sb + o;
            const float bias = (p.epi == 1 && o < p.O) ? p.bias[(long long)b * p.bias_sb + o] : 0.0f;
            const float unscale = scalbnf(1.0f, -(gx_scale_exp(p.amaxA[p.a_batched ? b : 0]) + gx_scale_exp(p.amaxB[p.b_batched ? b : 0])));
            for (int c = 0; c < n_chunks; ++c, ++cidx) {
                const uint32_t ab = p.split_acc ? 0u : (cidx & 1u), aphase = p.split_acc ? (cidx & 1u) : ((cidx >> 1) & 1u);
                mbar_wait(bar_tfull + 8 * ab, aphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ab * 256;
                const bool first = c == 0, last = c == n_chunks - 1;
                const bool rmw = !first, deriv = last && p.epi == 2;
                const float* hrow = deriv ? p.Hprev + (long long)b * p.h_sb + o : nullptr;
                // Everything a pass reads from global memory (the running sum of a chunked contraction, or the layer output an
                // activation derivative is taken from) is requested one pass AHEAD: sixteen independent loads per thread are
                // in flight while the previous sixteen columns are processed, instead of a load -> add -> store chain per
                // element.  (One array: a pass that needs both -- a derivative after a contraction longer than one chunk --
                // takes the layer output late.)
                const float* src = rmw ? crow : hrow;
                const bool need = (rmw || deriv) && o < p.O;
                float nxt[GX_EPW];
#pragma unroll
                for (int jj = 0; jj < GX_EPW; ++jj)
                    nxt[jj] = (need && tj * GX_BN + jj < p.J) ? src[(long long)(tj * GX_BN + jj) * p.c_sj] : 0.0f;
#pragma unroll 1
                for (int j0 = 0; j0 < GX_BN; j0 += GX_EPW) {
                    const int jb = tj * GX_BN + j0;
                    if (jb >= p.J) break;                                    // warp-uniform
                    float pre[GX_EPW];
#pragma unroll
                    for (int jj = 0; jj < GX_EPW; ++jj) pre[jj] = nxt[jj];
                    if (j0 + GX_EPW < GX_BN) {
#pragma unroll
                        for (int jj = 0; jj < GX_EPW; ++jj)
                            nxt[jj] = (need && jb + GX_EPW + jj < p.J) ? src[(long long)(jb + GX_EPW + jj) * p.c_sj] : 0.0f;
                    }
                    uint32_t v[GX_EPW];
                    tmem_ld16(taddr + j0, v);
                    tmem_ld_wait();
                    if (p.split_acc) {                       // add the small-term accumulator (FP32, round to nearest)
                        uint32_t v2[16];
                        tmem_ld16(taddr + 256 + j0, v2);
                        tmem_ld_wait();
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) v[jj] = __float_as_uint(__uint_as_float(v[jj]) + __uint_as_float(v2[jj]));
                    }
                    if (o < p.O) {
#pragma unroll
                        for (int jj = 0; jj < GX_EPW; ++jj) {
                            if (jb + jj < p.J) {
                                float val = __uint_as_float(v[jj]) * unscale;
                                if (rmw) val += pre[jj];
                                if (last) {
                                    if (p.epi == 1) val = gx_act(val + bias, p.act);
                                    else if (p.epi == 2)
                                        val *= act_deriv_from_output(rmw ? hrow[(long long)(jb + jj) * p.c_sj] : pre[jj], p.act);
                                }
                                crow[(long long)(jb + jj) * p.c_sj] = val;
                            }
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(bar_tempty + 8 * ab);
                if (p.split_acc) mbar_arrive(bar_tempty + 8);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// largest magnitude of a strided operand, per batch: rows of `fast` contiguous elements, `ld` apart, `rows` per batch, batches `sb` apart
__global__ void __launch_bounds__(256)
k_gemm_absmax(const float* __restrict__ base, long long fast, long long ld, long long rows, long long sb, long long total_rows,
              float* __restrict__ out /* [batches], zeroed */) {
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    float m = 0.0f;
    long long cur = -1;
    for (long long row = (long long)blockIdx.x * 8 + ty; row < total_rows; row += (long long)gridDim.x * 8) {
        const long long b = row / rows, r = row - b * rows;
        if (b != cur) {                      // warp-uniform: flush what belongs to the previous batch
            if (cur >= 0) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
                if (tx == 0) atomicMax(reinterpret_cast<unsigned*>(out + cur), __float_as_uint(m));     // non-negative floats order like their bits
            }
            cur = b;
            m = 0.0f;
        }
        const float* src = base + b * sb + r * ld;
        long long f = tx;
        float m1 = 0.0f, m2 = 0.0f, m3 = 0.0f;
        for (; f + 96 < fast; f += 128) {
            m = fmaxf(m, fabsf(src[f])); m1 = fmaxf(m1, fabsf(src[f + 32])); m2 = fmaxf(m2, fabsf(src[f + 64])); m3 = fmaxf(m3, fabsf(src[f + 96]));
        }
        for (; f < fast; f += 32) m = fmaxf(m, fabsf(src[f]));
        m = fmaxf(fmaxf(m, m1), fmaxf(m2, m3));
    }
    if (cur >= 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (tx == 0) atomicMax(reinterpret_cast<unsigned*>(out + cur), __float_as_uint(m));
    }
}

static bool gx_aligned(const void* p, long long stride_elems) {
    return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (stride_elems % 4) == 0 && stride_elems > 0;
}

// Runs g on the tensor cores when it qualifies (*used = true); otherwise leaves it to the caller's SIMT kernel.
int ssi_gemm_tc_try(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast, bool* used) {
    *used = false;
    if (ctx->opt_gemm_simt || g.split > 0 || g.c_so != 1 || batches < 1) return SSI_OK;
    if (g.O < 1 || g.J < 64 || g.K < 8 || g.K >= (1ll << 31)) return SSI_OK;
    // small problems: launch + pipeline fill would dominate.  Per batch, NOT per launch: which kernel evaluates a sample must
    // not depend on how many other samples share the call (results are compared bitwise across batch compositions)
    if ((double)g.O * g.J * (double)g.K < 1.6e7) return SSI_OK;
    // TMA: 16-byte aligned bases and strides
    if (a_kfast ? !(g.a_sk == 1 && gx_aligned(g.A, g.a_so)) : !(g.a_so == 1 && gx_aligned(g.A, g.a_sk))) return SSI_OK;
    if (b_jfast ? !(g.b_sj == 1 && gx_aligned(g.B, g.b_sk)) : !(g.b_sk == 1 && gx_aligned(g.B, g.b_sj))) return SSI_OK;
    const bool a_b = batches > 1 && g.a_sb != 0, b_b = batches > 1 && g.b_sb != 0;
    if ((a_b && (g.a_sb % 4 || g.a_sb < 0)) || (b_b && (g.b_sb % 4 || g.b_sb < 0))) return SSI_OK;
    if (ctx->smem_optin < GX_SMEM) return SSI_OK;

    PFN_ssi_encodeTiled encode = nullptr;
    SSI_TRY(ssi_tensormap_encoder(ctx, &encode));
    CUtensorMap mapA, mapB;
    const cuuint32_t estr[3] = {1, 1, 1};
    {
        cuuint64_t dims[3] = {a_kfast ? (cuuint64_t)g.K : (cuuint64_t)g.O, a_kfast ? (cuuint64_t)g.O : (cuuint64_t)g.K, (cuuint64_t)(a_b ? batches : 1)};
        cuuint64_t strides[2] = {(cuuint64_t)(a_kfast ? g.a_so : g.a_sk) * 4, a_b ? (cuuint64_t)g.a_sb * 4 : (cuuint64_t)16};
        cuuint32_t box[3] = {a_kfast ? (cuuint32_t)GX_BK : (cuuint32_t)GX_BM, a_kfast ? (cuuint32_t)GX_BM : (cuuint32_t)GX_BK, 1};
        if (!a_b) strides[1] = dims[1] * strides[0];
        const CUresult r = encode(&mapA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(g.A), dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, a_kfast ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return SSI_OK;          // a shape TMA cannot describe: SIMT
    }
    {
        const bool kf = !b_jfast;
        cuuint64_t dims[3] = {kf ? (cuuint64_t)g.K : (cuuint64_t)g.J, kf ? (cuuint64_t)g.J : (cuuint64_t)g.K, (cuuint64_t)(b_b ? batches : 1)};
        cuuint64_t strides[2] = {(cuuint64_t)(kf ? g.b_sj : g.b_sk) * 4, b_b ? (cuuint64_t)g.b_sb * 4 : (cuuint64_t)16};
        cuuint32_t box[3] = {kf ? (cuuint32_t)GX_BK : (cuuint32_t)GX_BN, kf ? (cuuint32_t)GX_BN : (cuuint32_t)GX_BK, 1};
        if (!b_b) strides[1] = dims[1] * strides[0];
        const CUresult r = encode(&mapB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(g.B), dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, kf ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return SSI_OK;
    }
    // one scale per operand and batch: the largest magnitude over what that batch reads (stream-ordered scratch of the context)
    const int nbA = a_b ? batches : 1, nbB = b_b ? batches : 1;
    SSI_TRY(ssi_reserve(ctx, ctx->bGemmAmax, (size_t)(nbA + nbB) * sizeof(float)));
    float* am = (float*)ctx->bGemmAmax.p;
    SSI_CUDA(ctx, cudaMemsetAsync(am, 0, (size_t)(nbA + nbB) * sizeof(float), ctx->stream));
    const long long rowsA = a_kfast ? g.O : g.K, fastA = a_kfast ? g.K : g.O, ldA = a_kfast ? g.a_so : g.a_sk;
    const long long rowsB = b_jfast ? g.K : g.J, fastB = b_jfast ? g.J : g.K, ldB = b_jfast ? g.b_sk : g.b_sj;
    const int blocks = 16 * ctx->sm_count;
    k_gemm_absmax<<<(unsigned)std::min<long long>(blocks, (rowsA * nbA + 7) / 8), 256, 0, ctx->stream>>>(g.A, fastA, ldA, rowsA, g.a_sb, rowsA * nbA, am);
    SSI_LAUNCH_CHECK(ctx);
    k_gemm_absmax<<<(unsigned)std::min<long long>(blocks, (rowsB * nbB + 7) / 8), 256, 0, ctx->stream>>>(g.B, fastB, ldB, rowsB, g.b_sb, rowsB * nbB, am + nbA);
    SSI_LAUNCH_CHECK(ctx);
    gemm_tc_params p{};
    p.amaxA = am;
    p.amaxB = am + nbA;
    p.C = g.C; p.c_sj = g.c_sj; p.c_sb = g.c_sb;
    p.O = g.O; p.J = g.J;
    p.n_to = (g.O + GX_BM - 1) / GX_BM;
    p.n_tj = (g.J + GX_BN - 1) / GX_BN;
    p.n_work = (long long)p.n_to * p.n_tj * batches;
    p.n_kb = (int)((g.K + GX_BK - 1) / GX_BK);
    p.chunk = 32;
    p.a_kfast = a_kfast ? 1 : 0; p.b_kfast = b_jfast ? 0 : 1;
    p.a_batched = a_b ? 1 : 0; p.b_batched = b_b ? 1 : 0;
    p.split_acc = g.epi == 1 ? 1 : 0;
    p.epi = g.epi; p.act = g.act; p.bias = g.bias; p.bias_sb = g.bias_sb; p.Hprev = g.Hprev; p.h_sb = g.h_sb;
    typedef void (*gx_kernel_t)(const CUtensorMap, const CUtensorMap, const gemm_tc_params);
    // the three orientations ssi_launch_gemm accepts: A k-fast with B k-fast, A o-fast with B either way
    const gx_kernel_t kern = p.a_kfast ? k_gemm_tc<true, true> : p.b_kfast ? k_gemm_tc<false, true> : k_gemm_tc<false, false>;
    SSI_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GX_SMEM));
    const int grid = (int)std::min<long long>(ctx->sm_count, p.n_work);
    kern<<<grid, GX_THREADS, GX_SMEM, ctx->stream>>>(mapA, mapB, p);
    SSI_LAUNCH_CHECK(ctx);
    ++ctx->stats.gemm_tc_launches;
    *used = true;
    return SSI_OK;
}
