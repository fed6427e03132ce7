// ssi_tc.cu — tensor-core path of the batched log-posterior (wide Dense chains).
//
// Replaces, for a group of G samples at a time, the body of the reference's density(z)
// (src/space_inference.jl:90-95):
//     new_W = W_swa + P*z            -> k_tc_project_* : one pass over P for the whole group,
//                                       weights written as split BF16 (hi, lo) K-major tiles
//     Dense: sigma.(W*x .+ b)        -> k_tc_layer<HIDDEN>: TMA -> smem -> tcgen05.mma (TMEM
//                                       accumulators) -> bias/activation epilogue -> split BF16
//     last Dense + logpdf(MvNormal)  -> k_tc_layer<FINAL>: the same GEMM with N = O rounded up to
//                                       16; the epilogue adds the bias, subtracts Y, squares and
//                                       reduces to per-warp FP64 partials (nothing is stored)
// Every Dense layer is one launch of the same warp-specialised GEMM; hidden widths and the
// input width are zero-padded to multiples of 64, so any Dense chain is supported.
//
// Precision: tcgen05 has no FP32-input mode.  Every FP32 operand x is split into two 16-bit planes
// hi + lo and each product is issued as hi*hi + hi*lo + lo*hi with FP32 accumulation in TMEM: three
// kind::f16 MMAs per product, so the roofline denominator is 1/3 of the BF16 peak.  Two plane formats
// (option "tc_precision"):
//   1 (default) "FP16x3": both planes FP16 (11 + 11 mantissa bits, representation error 2^-24 and a dropped lo*lo term
//      of 2^-24 against 2^-18 for BF16 planes: FP32-grade products from the same three MMAs), every operand scaled by a
//      power of two so that it sits high in FP16's range; the scales are undone exactly in the epilogue.
//        weights      per (layer, sample) 2^jw from a rigorous bound |W_swa| + sum_m |z_m| |P_m| <= 2^14: cannot overflow;
//        bases, X     one scale from their exact maximum (known when they are built);
//        z            per sample, from its own largest component;
//        activations  range unknown until they are computed: one scale per layer from a calibration pass at z = 0
//                     (run once per (data, subspace) with BF16 planes) that maps the largest activation to [2^9, 2^10),
//                     i.e. 64x..128x of headroom; conversions saturate; every plane-writing kernel tracks the largest
//                     activation it wrote, and a call that exceeded FP16's range is REPEATED with BF16 planes
//                     (ssi_tc_range_exceeded, checked where the host entry points synchronise anyway).
//      (kind::f16 encodes the formats of A and B separately, but mixing them -- BF16 activations against FP16 weights,
//      which would need no calibration -- raises an illegal-instruction fault on sm_100a: measured.)
//   0 "BF16x3": hi = bf16(x), lo = bf16(x - hi) for both operands (round 1; the fallback, and kept for A-B runs).
//
// Orientation: D[m, n] = sum_k A[m, k] B[n, k] with m = datapoint (128 per tile, TMEM lane),
// n = output feature (BN per tile, TMEM column), k = input feature.  A = activations
// [N][K] (K contiguous), B = weights [out][K] (K contiguous), both K-major SWIZZLE_128B.
#include "ssi_common.cuh"

#include "ssi_ptx.cuh"

#include <algorithm>
#include <cstdlib>

#define TC_BM 128
#define TC_BK 64                 // bf16 elements per k-block = 128 bytes = one swizzle row
#define TC_GMAX 32               // samples per group
#define TC_SMEM_PIPE (192 * 1024)
#define TC_SMEM_STORE (32 * 1024) // HIDDEN epilogue staging: 4 warps x 2 buffers x (hi, lo) x 32 rows x 64 B
#define TC_THREADS 192           // warp 0: TMA, warp 1: MMA + TMEM alloc, warps 2-5: epilogue

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------
// the GEMM layer kernel
// ---------------------------------------------------------------------------------------
struct tc_params {
    int N, G, m_tiles, n_tiles, k_blocks, BN, width, a_shared, act;
    int k_rev;              // odd feature tiles read the k-blocks in descending order (L2 reuse of the A row block)
    int a_il;               // A operand planes interleaved per k-block: row = [kb][hi 64 | lo 64] (the basis layer's output)
    int stages, stage_bytes;
    int mt_block;           // > 0: work order (mt block, sample, mt in block) so that concurrently running CTAs share A tiles
    int mt_pairs;           // PAIR: row-block pairs per sample, ceil(m_tiles / 2); the odd one out gets a dummy partner
    int n_work;
    uint32_t idesc;         // instruction descriptor (operand format: FP16 or BF16 planes)
    float a_scale;          // 2^ja of the NEXT layer's A planes, applied to this layer's output before it is split (1 for BF16x3)
    float* amax;            // HIDDEN: running max |activation| this layer has written (range check of the FP16 planes)
    const float* winv;      // [G] 2^-(jw_g + ja_in): accumulator -> true pre-activation (nullptr: 1)
    const float* bias;      // [G][width]  (width = padded out width of this layer)
    const float* Y;         // FINAL / FUSED: O x N column-major
    int O;                  // FINAL / FUSED: true output width
    int act_out;            // FUSED: activation of the fused output layer
    const float* Wout;      // FUSED: [G][width][TC_OP] output-layer weights, W[o, c] at [c][o]
    const float* bout;      // FUSED: [G][TC_OP]
    double* partials;       // FINAL / FUSED: [G][m_tiles*4]
};

#define TC_MODE_HIDDEN 0    // store the split activations with TMA
#define TC_MODE_FINAL  1    // this GEMM is the output layer: squared error in the epilogue
#define TC_MODE_FUSED  2    // last hidden layer; the (narrow) output layer and the squared error are folded into the epilogue
#define TC_OP 12            // FUSED: padded output width
#define TC_PREC_BF16X3 0
#define TC_PREC_FP16X3 1
#define TC_F16_MAX 65504.0f
#define TC_CAL_TOP 9        // calibration maps the largest activation seen at z = 0 to [2^TC_CAL_TOP, 2^(TC_CAL_TOP + 1))
static int tc_smem_total(int mode) {
    return TC_SMEM_PIPE + 3072 + (mode == TC_MODE_HIDDEN ? TC_SMEM_STORE : (mode == TC_MODE_FUSED ? 2 * 256 * TC_OP * 4 : 0));
}

// shared-memory carve-up (offsets from the 1024-aligned dynamic base)
//   [0, TC_SMEM_PIPE)            operand ring: stage = A_hi | A_lo | B_hi | B_lo
//   bias[2][256] floats, 12 mbarriers, TMEM base address
//   staging area (last, size depends on the mode): HIDDEN per-warp TMA-store staging (32 KB);
//   FUSED output-layer weight slices [2][256][TC_OP] (24 KB); FINAL nothing.
#define TC_OFF_BIAS TC_SMEM_PIPE
#define TC_OFF_BAR (TC_OFF_BIAS + 2 * 256 * 4)
#define TC_OFF_STORE (TC_OFF_BIAS + 3072)

__device__ __forceinline__ bool tc_decode_work(const tc_params& p, int w, int& g, int& mt, uint32_t crank = 0) {
    if (p.mt_pairs > 0) {       // CTA pairs: both CTAs always take part; row block m_tiles (odd count) is a dummy (TMA zero fill, masked epilogue)
        g = w / p.mt_pairs;
        mt = 2 * (w - g * p.mt_pairs) + (int)crank;
        return true;
    }
    if (p.mt_block > 0) {
        const int per = p.G * p.mt_block;
        const int blk = w / per, rem = w - blk * per;
        g = rem / p.mt_block;
        mt = blk * p.mt_block + (rem - g * p.mt_block);
        return mt < p.m_tiles;
    }
    g = w / p.m_tiles;
    mt = w - g * p.m_tiles;
    return true;
}

// activation as a compile-time constant: the epilogue stays straight-line code (a run-time switch per
// element bloats the unrolled loops past the instruction cache)
template <int ACT>
__device__ __forceinline__ float tc_act(float v) {
    if (ACT == SSI_ACT_RELU) return fmaxf(v, 0.0f);
    if (ACT == SSI_ACT_TANH) return tanhf(v);
    if (ACT == SSI_ACT_SIGMOID) return 1.0f / (1.0f + expf(-v));
    return v;
}

__device__ __noinline__ float tc_act_rt(float v, int act) { return ssi_act(v, act); }

// ---- the two 16-bit planes of an operand ------------------------------------------------
// Two values at a time.  FP16X3: the caller has applied the power-of-two scale; hi = FP16 (saturating: a value beyond the
// calibrated range must not become Inf), lo = FP16 of the exact remainder.  BF16X3: both planes BF16.
template <int PREC>
__device__ __forceinline__ void tc_split_a2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    if (PREC == TC_PREC_FP16X3) {
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
        const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - hf.y), "f"(x0 - hf.x));
    } else {
        const __nv_bfloat162 h2 = __floats2bfloat162_rn(x0, x1);
        const float2 hf = __bfloat1622float2(h2);
        hi = *reinterpret_cast<const uint32_t*>(&h2);
        const __nv_bfloat162 l2 = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
        lo = *reinterpret_cast<const uint32_t*>(&l2);
    }
}
// one value, run-time format (the small preparation kernels): kind 0 = BF16 | BF16, 1 = FP16 | FP16 (saturating; the
// caller's scale keeps |x| below 2^15 whenever the range is known)
__device__ __forceinline__ void tc_split1(float x, int kind, unsigned short& hi, unsigned short& lo) {
    if (kind == 1) {
        const __half h = __float2half_rn(fminf(fmaxf(x, -TC_F16_MAX), TC_F16_MAX));
        const __half l = __float2half_rn(x - __half2float(h));
        hi = __half_as_ushort(h);
        lo = __half_as_ushort(l);
    } else {
        const __nv_bfloat16 h = __float2bfloat16_rn(x);
        hi = __bfloat16_as_ushort(h);
        lo = __bfloat16_as_ushort(__float2bfloat16_rn(x - __bfloat162float(h)));
    }
}
// largest |activation| a plane-writing kernel has produced (true value, before the scale): non-negative floats order like
// their bit patterns
__device__ __forceinline__ void tc_amax_commit(float* amax, float mx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0 && amax && mx > 0.0f) atomicMax(reinterpret_cast<unsigned*>(amax), __float_as_uint(mx));
}

// PAIR (option "tc_pair"): the CTAs run as pairs on the two SMs of a TPC (cta_group::2).  A pair owns two adjacent 128-row
// blocks of one sample; every CTA loads its own A tiles and HALF of each weight tile (128 of the 256 feature rows), the
// even CTA's single thread issues 256 x 256 MMAs that read both CTAs' shared memory and write both CTAs' TMEM, and both
// epilogues drain their own accumulator.  A stage is 64 KB instead of 96 KB (three stages instead of two) and every byte
// of the weights crosses the L2 -> SM crossbar once per pair instead of once per CTA.
template <int MODE, int ACT, int PREC, bool PAIR>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc_layer(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
           const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
           const __grid_constant__ CUtensorMap tmSh, const __grid_constant__ CUtensorMap tmSl, const tc_params p) {
    // SWIZZLE_128B (TMA destination, UMMA descriptor with base_offset = 0) needs a 1024-byte aligned base
    extern __shared__ __align__(1024) uint8_t smem[];
    float* s_bias = reinterpret_cast<float*>(smem + TC_OFF_BIAS);                     // [2][256]
    float* s_wout = reinterpret_cast<float*>(smem + TC_OFF_STORE);                    // FUSED: [2][256*TC_OP]
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + TC_OFF_BAR);                 // full[4] empty[4] tfull[2] tempty[2]
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 12);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar_full = smem_u32(s_bar), bar_empty = smem_u32(s_bar + 4);
    const uint32_t bar_tfull = smem_u32(s_bar + 8), bar_tempty = smem_u32(s_bar + 10);
    const uint32_t smem_base = smem_u32(smem);
    const int BN = p.BN;
    // PAIR: this CTA holds half of the rows of every weight tile
    const uint32_t a_bytes = TC_BM * TC_BK * 2, b_bytes = (uint32_t)(PAIR ? BN / 2 : BN) * TC_BK * 2;
    const uint32_t crank = PAIR ? cluster_ctarank() : 0;
    // work items of this CTA (PAIR: of this pair)
    const int w_first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, w_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

    if (threadIdx.x == 0) {
        if (smem_base & 1023u) { printf("ssi_tc: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
        for (int s = 0; s < p.stages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        // PAIR: the leader's accumulator is free when the epilogues of BOTH CTAs have drained theirs
        for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, PAIR ? 256 : 128); }
        fence_barrier_init();
        tma_prefetch_desc(&tmAh); tma_prefetch_desc(&tmAl); tma_prefetch_desc(&tmBh); tma_prefetch_desc(&tmBl);
        if (MODE == TC_MODE_HIDDEN) { tma_prefetch_desc(&tmSh); tma_prefetch_desc(&tmSl); }
    }
    if (warp == 1) { if (PAIR) tmem_alloc_pair(smem_u32(s_tmem), 512); else tmem_alloc(smem_u32(s_tmem), 512); }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();        // the peer's barriers exist before anything arrives on them
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            // weights are re-read by every CTA working on the sample: keep them in L2; a shared A (the dataset)
            // likewise; per-sample activations are read by one CTA only
            const uint64_t pol_a = p.a_shared ? TC_EVICT_LAST : TC_EVICT_NORMAL;
            for (int w = w_first; w < p.n_work; w += w_step) {
                int g, mt;
                if (!tc_decode_work(p, w, g, mt, crank)) continue;
                for (int nt = 0; nt < p.n_tiles; ++nt) {
                    for (int kb = 0; kb < p.k_blocks; ++kb) {
                        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                        // PAIR: the bytes of both CTAs are counted on the leader's barrier, which its MMA thread waits on
                        const uint32_t full = PAIR ? mapa_u32(bar_full + 8 * stage, 0) : bar_full + 8 * stage;
                        const uint32_t sA = smem_base + stage * p.stage_bytes;
                        if (!PAIR) mbar_expect_tx(full, 2 * a_bytes + 2 * b_bytes);
                        else if (crank == 0) mbar_expect_tx(bar_full + 8 * stage, 2 * (2 * a_bytes + 2 * b_bytes));
                        // odd feature tiles walk the k-blocks backwards: the A k-blocks read last for tile nt are the first ones tile
                        // nt + 1 wants, which is what an LRU-like L2 still holds when a round of A tiles slightly exceeds it
                        const int kbe = (p.k_rev && (nt & 1)) ? p.k_blocks - 1 - kb : kb;
                        const int ka = p.a_il ? 2 * kbe * TC_BK : kbe * TC_BK;
                        // the last feature tile is the last reader of this row block's activations: let them go first
                        const uint64_t pa = (!p.a_shared && nt == p.n_tiles - 1) ? TC_EVICT_FIRST : pol_a;
                        if (PAIR) {
                            const int brow = nt * BN + (int)crank * (BN / 2);          // this CTA's half of the weight tile (the maps' box is BN/2 rows)
                            tma_load_3d_pair_hint(sA, &tmAh, full, ka, mt * TC_BM, g, pa);
                            tma_load_3d_pair_hint(sA + a_bytes, &tmAl, full, p.a_il ? ka + TC_BK : ka, mt * TC_BM, g, pa);
                            tma_load_3d_pair_hint(sA + 2 * a_bytes, &tmBh, full, kbe * TC_BK, brow, g, TC_EVICT_LAST);
                            tma_load_3d_pair_hint(sA + 2 * a_bytes + b_bytes, &tmBl, full, kbe * TC_BK, brow, g, TC_EVICT_LAST);
                        } else {
                            tma_load_3d_hint(sA, &tmAh, full, ka, mt * TC_BM, p.a_shared ? 0 : g, pa);
                            tma_load_3d_hint(sA + a_bytes, &tmAl, full, p.a_il ? ka + TC_BK : ka, mt * TC_BM, p.a_shared ? 0 : g, pa);
                            tma_load_3d_hint(sA + 2 * a_bytes, &tmBh, full, kbe * TC_BK, nt * BN, g, TC_EVICT_LAST);
                            tma_load_3d_hint(sA + 2 * a_bytes + b_bytes, &tmBl, full, kbe * TC_BK, nt * BN, g, TC_EVICT_LAST);
                        }
                        if (++stage == p.stages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0 && crank == 0) {           // PAIR: the even CTA issues for both
            const uint32_t idesc = p.idesc;
            int stage = 0;
            uint32_t phase = 0;
            uint32_t tile = 0;
            for (int w = w_first; w < p.n_work; w += w_step) {
                int g, mt;
                if (!tc_decode_work(p, w, g, mt, crank)) continue;
                for (int nt = 0; nt < p.n_tiles; ++nt, ++tile) {
                    const uint32_t ab = tile & 1, aphase = (tile >> 1) & 1;
                    mbar_wait(bar_tempty + 8 * ab, aphase ^ 1);        // epilogue has drained this accumulator
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + ab * 256;
                    for (int kb = 0; kb < p.k_blocks; ++kb) {
                        mbar_wait(bar_full + 8 * stage, phase);         // TMA bytes have landed
                        tc_fence_after();
                        const uint32_t sA = smem_base + stage * p.stage_bytes;
                        const uint64_t ah = umma_desc_sw128(sA), al = umma_desc_sw128(sA + a_bytes);
                        const uint64_t bh = umma_desc_sw128(sA + 2 * a_bytes), bl = umma_desc_sw128(sA + 2 * a_bytes + b_bytes);
#pragma unroll
                        for (int k = 0; k < TC_BK / 16; ++k) {
                            const uint64_t ko = (uint64_t)(k * 32 >> 4);   // +32 bytes per K=16 step inside the swizzle row
                            if (PAIR) {
                                umma_f16_pair(d_tmem, ah + ko, bh + ko, idesc, (kb | k) != 0);
                                umma_f16_pair(d_tmem, ah + ko, bl + ko, idesc, 1);
                                umma_f16_pair(d_tmem, al + ko, bh + ko, idesc, 1);
                            } else {
                                umma_bf16(d_tmem, ah + ko, bh + ko, idesc, (kb | k) != 0);
                                umma_bf16(d_tmem, ah + ko, bl + ko, idesc, 1);
                                umma_bf16(d_tmem, al + ko, bh + ko, idesc, 1);
                            }
                        }
                        // frees the smem slot (PAIR: of both CTAs) when the MMAs retire
                        if (PAIR) umma_commit_pair(bar_empty + 8 * stage); else umma_commit(bar_empty + 8 * stage);
                        if (++stage == p.stages) { stage = 0; phase ^= 1; }
                    }
                    // accumulator complete -> epilogue (PAIR: of both CTAs)
                    if (PAIR) umma_commit_pair(bar_tfull + 8 * ab); else umma_commit(bar_tfull + 8 * ab);
                }
            }
        }
    } else {
        // ================= epilogue (4 warps = 128 TMEM lanes) =================
        const int q = warp & 3;                      // TMEM lane quarter this warp may access
        const int et = threadIdx.x - 64;             // 0..127
        // HIDDEN: this warp's TMA-store staging: [2 buffers][hi | lo][32 rows x 64 B], SWIZZLE_64B
        const uint32_t stage_w = smem_base + TC_OFF_STORE + (uint32_t)(warp - 2) * 8192;
        const uint32_t swz = (uint32_t)((lane >> 1) & 3);
        const float asc = p.a_scale;
        float amx = 0.0f;                            // HIDDEN: largest |activation| this thread has written
        uint32_t chunk_ctr = 0;
        uint32_t tile = 0;
        // PAIR: "accumulator drained" is reported to the leader's barrier
        const uint32_t tempty_remote = PAIR ? mapa_u32(bar_tempty, 0) : 0;
        for (int w = w_first; w < p.n_work; w += w_step) {
            int g, mt;
            if (!tc_decode_work(p, w, g, mt, crank)) continue;
            const float inv = p.winv ? p.winv[g] : 1.0f;     // exact power of two: undoes the operand scales
            double sse = 0.0;
            // FUSED: 4 rows per thread (see tmem_ld_16x256b_x8), partial sums over this thread's columns
            float pred[4][TC_OP];
            if (MODE == TC_MODE_FUSED) {
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int o = 0; o < TC_OP; ++o) pred[r][o] = 0.0f;
            }

            for (int nt = 0; nt < p.n_tiles; ++nt, ++tile) {
                const uint32_t ab = tile & 1, aphase = (tile >> 1) & 1;
                float* sb = s_bias + ab * 256;
                float* sw = s_wout + ab * 256 * TC_OP;
                // stage this tile's bias (and output-layer weights) while the MMAs run
                for (int c = et; c < BN; c += 128) sb[c] = p.bias[(long long)g * p.width + nt * BN + c];
                if (MODE == TC_MODE_FUSED) {
                    const float4* src = reinterpret_cast<const float4*>(p.Wout + ((long long)g * p.width + nt * BN) * TC_OP);
                    float4* dst = reinterpret_cast<float4*>(sw);
                    for (int c = et; c < BN * TC_OP / 4; c += 128) dst[c] = src[c];
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
                mbar_wait(bar_tfull + 8 * ab, aphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ab * 256;
                if (MODE == TC_MODE_FINAL) {
                    const long long m = (long long)mt * TC_BM + q * 32 + lane;
                    const bool valid = m < p.N;
#pragma unroll 1
                    for (int c0 = 0; c0 < BN; c0 += 16) {
                        uint32_t v[16];
                        tmem_ld16(taddr + c0, v);
                        tmem_ld_wait();
                        if (valid) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                const int o = nt * BN + c0 + j;
                                if (o < p.O) {
                                    const float df = tc_act<ACT>(fmaf(__uint_as_float(v[j]), inv, sb[c0 + j])) - p.Y[o + m * p.O];
                                    sse += (double)df * (double)df;
                                }
                            }
                        }
                    }
                } else if (MODE == TC_MODE_FUSED) {
                    const int cq = 2 * (lane & 3);
#pragma unroll 1
                    for (int cb = 0; cb < BN; cb += 16) {
                        uint32_t v0[8], v1[8];
                        tmem_ld_16x256b_x2(taddr + cb, v0);                                   // lanes q*32 + [0,16)
                        tmem_ld_16x256b_x2(taddr + ((uint32_t)16 << 16) + cb, v1);            // lanes q*32 + [16,32)
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 2; ++i) {
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int col = cb + 8 * i + cq + e;
                                const float b = sb[col];
                                const float4* w4 = reinterpret_cast<const float4*>(sw + col * TC_OP);
                                float wv[TC_OP];
#pragma unroll
                                for (int o4 = 0; o4 < TC_OP / 4; ++o4) {
                                    const float4 ww = w4[o4];
                                    wv[4 * o4] = ww.x; wv[4 * o4 + 1] = ww.y; wv[4 * o4 + 2] = ww.z; wv[4 * o4 + 3] = ww.w;
                                }
                                const float h0 = tc_act<ACT>(fmaf(__uint_as_float(v0[4 * i + e]), inv, b));
                                const float h1 = tc_act<ACT>(fmaf(__uint_as_float(v0[4 * i + 2 + e]), inv, b));
                                const float h2 = tc_act<ACT>(fmaf(__uint_as_float(v1[4 * i + e]), inv, b));
                                const float h3 = tc_act<ACT>(fmaf(__uint_as_float(v1[4 * i + 2 + e]), inv, b));
#pragma unroll
                                for (int o = 0; o < TC_OP; ++o) {
                                    pred[0][o] = fmaf(h0, wv[o], pred[0][o]);
                                    pred[1][o] = fmaf(h1, wv[o], pred[1][o]);
                                    pred[2][o] = fmaf(h2, wv[o], pred[2][o]);
                                    pred[3][o] = fmaf(h3, wv[o], pred[3][o]);
                                }
                            }
                        }
                    }
                } else {
#pragma unroll 1
                    for (int c0 = 0; c0 < BN; c0 += 32, ++chunk_ctr) {
                        uint32_t v[32];
                        tmem_ld32(taddr + c0, v);
                        tmem_ld_wait();
                        uint32_t hi[16], lo[16];
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            const float x0 = tc_act<ACT>(fmaf(__uint_as_float(v[j]), inv, sb[c0 + j]));
                            const float x1 = tc_act<ACT>(fmaf(__uint_as_float(v[j + 1]), inv, sb[c0 + j + 1]));
                            amx = fmaxf(amx, fmaxf(fabsf(x0), fabsf(x1)));
                            tc_split_a2<PREC>(x0 * asc, x1 * asc, hi[j >> 1], lo[j >> 1]);
                        }
                        // the TMA store that last read this staging buffer (two chunks ago) must have finished reading
                        if (chunk_ctr >= 2) {
                            if (lane == 0) tma_store_wait_read1();
                            __syncwarp();
                        }
                        const uint32_t sh = stage_w + (chunk_ctr & 1) * 4096, sl = sh + 2048;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const uint32_t off = (uint32_t)lane * 64 + (((uint32_t)c ^ swz) << 4);
                            st_shared_v4(sh + off, hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
                            st_shared_v4(sl + off, lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
                        }
                        fence_proxy_async();
                        __syncwarp();
                        if (lane == 0) {
                            // rows >= N are clipped by TMA; the activations are consumed by the next kernel, far
                            // beyond L2 residency: do not let them evict the operands
                            tma_store_3d_hint(&tmSh, sh, nt * BN + c0, mt * TC_BM + q * 32, g, TC_EVICT_FIRST);
                            tma_store_3d_hint(&tmSl, sl, nt * BN + c0, mt * TC_BM + q * 32, g, TC_EVICT_FIRST);
                            tma_store_commit();
                        }
                    }
                }
                tc_fence_before();
                if (PAIR) mbar_arrive_cluster(tempty_remote + 8 * ab); else mbar_arrive(bar_tempty + 8 * ab);
            }
            if (MODE == TC_MODE_FUSED) {
                // the 4 threads of a quad hold the same 4 rows for interleaved columns: reduce across the quad,
                // then quad member j finishes row j
                const float* bo = p.bout + (long long)g * TC_OP;
                float mine[TC_OP];
#pragma unroll
                for (int r = 0; r < 4; ++r) {
#pragma unroll
                    for (int o = 0; o < TC_OP; ++o) {
                        float v = pred[r][o];
                        v += __shfl_xor_sync(0xffffffffu, v, 1);
                        v += __shfl_xor_sync(0xffffffffu, v, 2);
                        if (r == 0 || (lane & 3) == r) mine[o] = v;
                    }
                }
                const int r = lane & 3;
                const long long m = (long long)mt * TC_BM + q * 32 + (r >> 1) * 16 + (lane >> 2) + 8 * (r & 1);
                if (m < p.N) {
#pragma unroll
                    for (int o = 0; o < TC_OP; ++o) {
                        if (o < p.O) {
                            const float df = tc_act_rt(mine[o] + bo[o], p.act_out) - p.Y[o + m * p.O];
                            sse += (double)df * (double)df;
                        }
                    }
                }
            }
            if (MODE != TC_MODE_HIDDEN) {
                sse = ssi_warp_sum(sse);
                if (lane == 0 && mt < p.m_tiles) p.partials[(long long)g * (p.m_tiles * 4) + mt * 4 + q] = sse;
            }
        }
        if (MODE == TC_MODE_HIDDEN) {
            tc_amax_commit(p.amax, amx);
            if (lane == 0) tma_store_wait_all();
        }
    }

    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();        // no CTA leaves (or frees TMEM) while its peer's MMAs or arrivals may still touch it
    if (warp == 1) {
        tc_fence_after();
        if (PAIR) tmem_dealloc_pair(tmem_base, 512); else tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------
// operand preparation
// ---------------------------------------------------------------------------------------
// X (in0 x N column-major == [N][in0]) -> Xh, Xl [N][Kp] (zero padded); kind 0 (BF16 planes) or 1 (FP16 planes, scaled by 2^ja from max |X|)
__global__ void __launch_bounds__(256)
k_tc_split_x(const float* __restrict__ X, long long N, int in0, int Kp, int kind, float scale, bf16* __restrict__ Xh, bf16* __restrict__ Xl) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N * Kp) return;
    const long long j = e / Kp;
    const int i = (int)(e % Kp);
    unsigned short hi, lo;
    tc_split1((i < in0 ? X[j * in0 + i] : 0.0f) * scale, kind, hi, lo);
    reinterpret_cast<unsigned short*>(Xh)[e] = hi;
    reinterpret_cast<unsigned short*>(Xl)[e] = lo;
}

// ---- FP16 planes: power-of-two scales of the weight operands ------------------------------------------------------
// cmax[l][m] = max |column m of [P | W_swa]| over the flat range of layer l's weight matrix (once per subspace)
__global__ void __launch_bounds__(256)
k_tc_colmax(const float* __restrict__ PW /* n x (M+1) */, long long n, long long w_off, long long count, float* __restrict__ out) {
    __shared__ float red[8];
    const float* col = PW + (long long)blockIdx.x * n + w_off;
    float mx = 0.0f;
    for (long long e = threadIdx.x; e < count; e += blockDim.x) mx = fmaxf(mx, fabsf(col[e]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
        out[blockIdx.x] = mx;
    }
}
// Per (layer, sample): bound = cmax[M] + sum_m |z_m| cmax[m] >= max |W_swa + P z| over the layer; the scale 2^jw puts the
// bound in [2^13, 2^14), so the FP16 hi plane cannot overflow and a sample's scale depends on nothing but its own z
// (bitwise batch invariance).  wscale[l][g] = 2^jw, winv[l][g] = 2^-(jw + ja).
struct tc_ja_t { int v[SSI_MAX_LAYERS + 1]; };      // exponent of the scale of the A planes layer l consumes
__global__ void k_tc_wscale(const float* __restrict__ Z, int M, int G, const float* __restrict__ cmax /* [nl][M+1] */, int nl, int gstride,
                            const tc_ja_t ja_in, float* __restrict__ wscale, float* __restrict__ winv) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nl * G) return;
    const int l = t / G, g = t % G;
    const int ja = ja_in.v[l];
    const float* cm = cmax + l * (M + 1);
    float bound = cm[M];
    for (int m = 0; m < M; ++m) bound = fmaf(fabsf(Z[m + (long long)g * M]), cm[m], bound);
    int jw = 0;
    if (bound > 0.0f && bound < 3.0e38f) jw = 13 - ilogbf(bound);
    jw = max(-100, min(100, jw));
    wscale[l * gstride + g] = scalbnf(1.0f, jw);
    winv[l * gstride + g] = scalbnf(1.0f, -(jw + ja));
}
// max |x| of a float array into *out (one atomicMax on the bit pattern; *out zeroed by the caller)
__global__ void __launch_bounds__(256)
k_tc_absmax(const float* __restrict__ x, long long count, unsigned* __restrict__ out) {
    float mx = 0.0f;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x) mx = fmaxf(mx, fabsf(x[e]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0 && mx > 0.0f) atomicMax(out, __float_as_uint(mx));
}

// One Dense weight matrix of the group: flat (out x in, column-major: o + i*out) -> split BF16 [g][o][Kp],
// zero padded to out_pad rows and Kp columns.  Each block owns a 16(i) x 16(o) tile and one element per thread:
// P is read once for all G samples (K1, src/space_inference.jl:91) with 64-byte segments along o, the M loads of a
// thread are issued four at a time, and the transposition to the K-major GEMM operand goes through shared memory
// once per block, so that every (sample, o) row leaves as one 32-byte store along i.
#define PW_T 16
__global__ void __launch_bounds__(256)
k_tc_project_w(const float* __restrict__ Wswa, const float* __restrict__ P, const float* __restrict__ Z,
               long long n, int M, int G, long long w_off, int in, int out, int out_pad, int Kp,
               const float* __restrict__ wscale /* [G] power-of-two scales (mixed planes) or nullptr */,
               bf16* __restrict__ Wh, bf16* __restrict__ Wl) {
    __shared__ __align__(16) float zs[SSI_MAX_M][TC_GMAX];                 // [m][g], zero for g >= G
    __shared__ __align__(16) unsigned short sh[TC_GMAX][PW_T][PW_T], sl[TC_GMAX][PW_T][PW_T];   // [g][o][i]
    __shared__ float sc[TC_GMAX];
    const int tx = threadIdx.x & (PW_T - 1), ty = threadIdx.x >> 4;
    for (int e = threadIdx.x; e < M * TC_GMAX; e += 256) {
        const int m = e / TC_GMAX, g = e % TC_GMAX;
        zs[m][g] = g < G ? Z[m + g * M] : 0.0f;
    }
    if (threadIdx.x < TC_GMAX) sc[threadIdx.x] = (wscale && threadIdx.x < G) ? wscale[threadIdx.x] : 1.0f;
    const int kind = wscale ? 1 : 0;
    __syncthreads();
    const int i0 = blockIdx.x * PW_T, o0 = blockIdx.y * PW_T;
    const int i = i0 + ty, o = o0 + tx;
    const bool ok = (i < in) && (o < out);
    const long long flat = w_off + o + (long long)i * out;
    float acc[TC_GMAX];
    const float w0 = ok ? Wswa[flat] : 0.0f;
#pragma unroll
    for (int g = 0; g < TC_GMAX; ++g) acc[g] = w0;
    if (ok) {
        for (int m0 = 0; m0 < M; m0 += 4) {
            float pv[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) pv[r] = (m0 + r < M) ? P[flat + (long long)(m0 + r) * n] : 0.0f;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int m = min(m0 + r, M - 1);       // pv is zero past M
#pragma unroll
                for (int g = 0; g < TC_GMAX; g += 4) {
                    const float4 z4 = *reinterpret_cast<const float4*>(&zs[m][g]);
                    acc[g] = fmaf(pv[r], z4.x, acc[g]);
                    acc[g + 1] = fmaf(pv[r], z4.y, acc[g + 1]);
                    acc[g + 2] = fmaf(pv[r], z4.z, acc[g + 2]);
                    acc[g + 3] = fmaf(pv[r], z4.w, acc[g + 3]);
                }
            }
        }
    }
#pragma unroll
    for (int g = 0; g < TC_GMAX; ++g) {
        unsigned short hi, lo;
        tc_split1(acc[g] * sc[g], kind, hi, lo);
        sh[g][tx][ty] = hi;
        sl[g][tx][ty] = lo;
    }
    __syncthreads();
    // (g, o) rows of 16 i = 32 bytes each
    for (int c = threadIdx.x; c < G * PW_T; c += 256) {
        const int g = c / PW_T, oo = c % PW_T;
        if (o0 + oo < out_pad && i0 < Kp) {
            const long long dst = ((long long)g * out_pad + o0 + oo) * Kp + i0;
            const uint4* h4 = reinterpret_cast<const uint4*>(&sh[g][oo][0]);
            const uint4* l4 = reinterpret_cast<const uint4*>(&sl[g][oo][0]);
            uint4* dh = reinterpret_cast<uint4*>(Wh + dst);
            uint4* dl = reinterpret_cast<uint4*>(Wl + dst);
            dh[0] = h4[0]; dh[1] = h4[1];
            dl[0] = l4[0]; dl[1] = l4[1];
        }
    }
}

// bias[g][o] = (W_swa + P z_g)[b_off + o] for o < out, 0 for the padded tail
__global__ void __launch_bounds__(256)
k_tc_project_b(const float* __restrict__ Wswa, const float* __restrict__ P, const float* __restrict__ Z,
               long long n, int M, int G, long long b_off, int out, int out_pad, float* __restrict__ dst) {
    __shared__ float zs[SSI_MAX_M * TC_GMAX];
    for (int e = threadIdx.x; e < M * G; e += 256) zs[e] = Z[e];
    __syncthreads();
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= out_pad) return;
    float acc[TC_GMAX];
#pragma unroll
    for (int g = 0; g < TC_GMAX; ++g) acc[g] = 0.0f;
    if (o < out) {
        const long long flat = b_off + o;
        const float w0 = Wswa[flat];
#pragma unroll
        for (int g = 0; g < TC_GMAX; ++g) acc[g] = w0;
        for (int m = 0; m < M; ++m) {
            const float pv = P[flat + (long long)m * n];
#pragma unroll
            for (int g = 0; g < TC_GMAX; ++g) acc[g] = fmaf(pv, zs[m + g * M], acc[g]);
        }
    }
#pragma unroll
    for (int g = 0; g < TC_GMAX; ++g)
        if (g < G) dst[(long long)g * out_pad + o] = acc[g];
}

// Fused output layer: W (O x width column-major, o + c*O) -> dst[g][c][TC_OP] (zero padded);
// bias: inner = count -> dst[g][o].   dst[g][(e / inner) * dst_ld + (e % inner)] = (W_swa + P z_g)[src_off + e]
__global__ void __launch_bounds__(256)
k_tc_project_v(const float* __restrict__ Wswa, const float* __restrict__ P, const float* __restrict__ Z,
               long long n, int M, int G, long long src_off, int count, int inner, int dst_ld, long long dst_gs,
               float* __restrict__ dst) {
    __shared__ float zs[SSI_MAX_M * TC_GMAX];
    for (int e = threadIdx.x; e < M * G; e += 256) zs[e] = Z[e];
    __syncthreads();
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= count) return;
    const long long flat = src_off + e;
    float acc[TC_GMAX];
    const float w0 = Wswa[flat];
#pragma unroll
    for (int g = 0; g < TC_GMAX; ++g) acc[g] = w0;
    for (int m = 0; m < M; ++m) {
        const float pv = P[flat + (long long)m * n];
#pragma unroll
        for (int g = 0; g < TC_GMAX; ++g) acc[g] = fmaf(pv, zs[m + g * M], acc[g]);
    }
    const long long d = (long long)(e / inner) * dst_ld + (e % inner);
#pragma unroll
    for (int g = 0; g < TC_GMAX; ++g)
        if (g < G) dst[(long long)g * dst_gs + d] = acc[g];
}

// First Dense layer without a GEMM.  The pre-activation is affine in z:
//   (W1_swa + sum_m z_m P1_m) x + (b1_swa + sum_m z_m pb_m) = B_M(x) + sum_m z_m B_m(x),
// with the M+1 basis pre-activations B_m = [P | W_swa]_m applied to the dataset computed once per
// (data, subspace) in exact FP32.  Per sample this is M FMAs per activation instead of in0, and an
// HBM stream instead of tensor-core work.  z of the group lives in constant memory so the FMAs take
// it as a constant operand.

// Each thread owns two adjacent activations: all M+1 basis values are fetched up front (M+1 independent
// 8-byte loads in flight per thread), then one output per sample is a chain of M FMAs whose z operand comes
// from the constant bank (uniform across the warp).
// z of the group is staged in shared memory and read with broadcast LDS.128 (the constant-bank route, one indexed
// LDC per FMA operand, saturated the address-divergence unit: ncu showed pipe_adu at 82 %); the FMAs are packed
// FFMA2 with z as the scalar operand.  Each thread walks TC_BASIS_ITERS adjacent-pair positions.
#define TC_BASIS_THREADS 256
#define TC_BASIS_ITERS 4
template <int ACT, int MP>
__global__ void __launch_bounds__(TC_BASIS_THREADS)
k_tc_basis_layer(const float* __restrict__ bases /* [M+1][NW] */, long long NW, int M, int G,
                 const float* __restrict__ zpack /* [TC_GMAX][SSI_MAX_M], zero padded */,
                 bf16* __restrict__ Hh, bf16* __restrict__ Hl /* [g][NW] */, int fp16, float a_scale, float* __restrict__ amax) {
    __shared__ __align__(16) float zs[TC_GMAX][MP];
    for (int e = threadIdx.x; e < TC_GMAX * MP; e += TC_BASIS_THREADS) zs[e / MP][e % MP] = zpack[(e / MP) * SSI_MAX_M + (e % MP)];
    __syncthreads();
    const long long base = (long long)blockIdx.x * (TC_BASIS_THREADS * TC_BASIS_ITERS * 2);
    float amx = 0.0f;
#pragma unroll 1
    for (int it = 0; it < TC_BASIS_ITERS; ++it) {
        const long long e = base + ((long long)it * TC_BASIS_THREADS + threadIdx.x) * 2;
        if (e >= NW) break;          // leaves the loop only: the whole warp meets again at tc_amax_commit
        float2 b[MP];
#pragma unroll
        for (int m = 0; m < MP; ++m)
            b[m] = m < M ? __ldcs(reinterpret_cast<const float2*>(bases + (long long)m * NW + e)) : make_float2(0.f, 0.f);
        const float2 b0 = __ldcs(reinterpret_cast<const float2*>(bases + (long long)M * NW + e));
#pragma unroll 2
        for (int g = 0; g < G; ++g) {
            float2 x = b0;
#pragma unroll
            for (int m = 0; m < MP; m += 4) {
                const float4 z4 = *reinterpret_cast<const float4*>(&zs[g][m]);     // zero for m >= M
                x = __ffma2_rn(b[m], make_float2(z4.x, z4.x), x);
                x = __ffma2_rn(b[m + 1], make_float2(z4.y, z4.y), x);
                x = __ffma2_rn(b[m + 2], make_float2(z4.z, z4.z), x);
                x = __ffma2_rn(b[m + 3], make_float2(z4.w, z4.w), x);
            }
            const float x0 = tc_act<ACT>(x.x);
            const float x1 = tc_act<ACT>(x.y);
            amx = fmaxf(amx, fmaxf(fabsf(x0), fabsf(x1)));
            uint32_t h2, l2;
            if (fp16) tc_split_a2<TC_PREC_FP16X3>(x0 * a_scale, x1 * a_scale, h2, l2);
            else tc_split_a2<TC_PREC_BF16X3>(x0, x1, h2, l2);
            // interleaved output: 64 hi then 64 lo halves per block of 64 activations (see k_tc_basis_mma)
            bf16* o = Hh + 2 * ((long long)g * NW + (e & ~63ll)) + (e & 63);
            __stcs(reinterpret_cast<unsigned int*>(o), h2);
            __stcs(reinterpret_cast<unsigned int*>(o + 64), l2);
        }
    }
    tc_amax_commit(amax, amx);
}

// ---------------------------------------------------------------------------------------
// the same first layer ON THE TENSOR CORES: with z augmented by a constant 1 it is one GEMM
//     pre[s, e] = sum_{m <= M} zaug[s, m] * basesT[e, m],      e = (datapoint, hidden unit),  K = M+1 <= 32
// whose M dimension is the SAMPLES (up to 128 per group = the 128 TMEM lanes), N = 256 activations per tile and K = 32.
// The bases are re-laid out once as K-major split-BF16 rows [e][32] (64 bytes = one SWIZZLE_64B row); z of the group
// sits in shared memory as the A operand for the whole kernel.  BF16x3 (hi*hi + hi*lo + lo*hi), FP32 accumulate in TMEM.
// The FP32 FMA work of k_tc_basis_layer disappears (6 small MMAs per 256 activations of 128 samples) and the bases are
// read once per 128 samples instead of once per 32: the layer becomes a pure HBM stream of its own output.
// Roles as in k_tc_layer: warp 0 TMA, warp 1 MMA, warps 2-5 epilogue (activation, hi/lo split, TMA store to
// H1[s][e] viewed as a [samples][N*width] matrix).
#define TB_N 256
#define TB_STAGES 2                                // the kernel writes 4x what it reads: shared memory goes to the store side
#define TB_SBUF 3                                  // TMA-store staging buffers per epilogue warp (hi | lo, 2 x 4 KB each): the output
                                                   // stream is bound by the bytes in flight, 2 buffers gave 2.7 TB/s
#define TB_STAGE_BYTES (2 * TB_N * 64)            // basesT hi | lo
#define TB_OFF_Z (TB_STAGES * TB_STAGE_BYTES)      // zaug hi (128 x 64 B) | lo
#define TB_OFF_STORE (TB_OFF_Z + 2 * 128 * 64)
#define TB_OFF_BAR (TB_OFF_STORE + 4 * TB_SBUF * 8192)
#define TB_SMEM_TOTAL (TB_OFF_BAR + 16 * 8 + 16)

// FP16 planes (PREC 1): row s of z carries its own scale 2^jz_s (from the sample's largest component), the bases one
// scale 2^jb (from max |bases|): zinv[s] = 2^-(jz_s + jb) turns lane s of an accumulator into the true pre-activation;
// a_scale is the calibrated scale of the activations that are split and stored; amax tracks the largest one written.
template <int ACT, int PREC>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc_basis_mma(const __grid_constant__ CUtensorMap tmZh, const __grid_constant__ CUtensorMap tmZl,
               const __grid_constant__ CUtensorMap tmTh, const __grid_constant__ CUtensorMap tmTl,
               const __grid_constant__ CUtensorMap tmO, const int n_tiles, const float* __restrict__ zinv, const float a_scale,
               float* __restrict__ amax) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + TB_OFF_BAR);     // full[4] empty[4] tfull[2] tempty[2] zfull
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 16);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_u32(s_bar), bar_empty = bar_full + 8 * TB_STAGES;
    const uint32_t bar_tfull = bar_empty + 8 * TB_STAGES, bar_tempty = bar_tfull + 16, bar_z = bar_tempty + 16;

    if (threadIdx.x == 0) {
        if (smem_base & 1023u) { printf("ssi_tc: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
        for (int s = 0; s < TB_STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 128); }
        mbar_init(bar_z, 1);
        fence_barrier_init();
        tma_prefetch_desc(&tmZh); tma_prefetch_desc(&tmZl); tma_prefetch_desc(&tmTh); tma_prefetch_desc(&tmTl);
        tma_prefetch_desc(&tmO);
    }
    if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        if (lane == 0) {
            mbar_expect_tx(bar_z, 2 * 128 * 64);
            tma_load_3d_hint(smem_base + TB_OFF_Z, &tmZh, bar_z, 0, 0, 0, TC_EVICT_LAST);
            tma_load_3d_hint(smem_base + TB_OFF_Z + 128 * 64, &tmZl, bar_z, 0, 0, 0, TC_EVICT_LAST);
            int stage = 0;
            uint32_t phase = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                const uint32_t full = bar_full + 8 * stage;
                const uint32_t sB = smem_base + stage * TB_STAGE_BYTES;
                mbar_expect_tx(full, TB_STAGE_BYTES);
                tma_load_3d_hint(sB, &tmTh, full, 0, t * TB_N, 0, TC_EVICT_FIRST);          // read once per group of samples
                tma_load_3d_hint(sB + TB_N * 64, &tmTl, full, 0, t * TB_N, 0, TC_EVICT_FIRST);
                if (++stage == TB_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = PREC == TC_PREC_FP16X3 ? umma_idesc_f16(TB_N, UMMA_FMT_F16, UMMA_FMT_F16) : umma_idesc_bf16(TB_N);
            mbar_wait(bar_z, 0);
            tc_fence_after();
            const uint64_t zh = umma_desc_sw64(smem_base + TB_OFF_Z), zl = umma_desc_sw64(smem_base + TB_OFF_Z + 128 * 64);
            int stage = 0;
            uint32_t phase = 0, tile = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tile) {
                const uint32_t ab = tile & 1, aphase = (tile >> 1) & 1;
                mbar_wait(bar_tempty + 8 * ab, aphase ^ 1);
                mbar_wait(bar_full + 8 * stage, phase);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + ab * 256;
                const uint32_t sB = smem_base + stage * TB_STAGE_BYTES;
                const uint64_t bh = umma_desc_sw64(sB), bl = umma_desc_sw64(sB + TB_N * 64);
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const uint64_t ko = (uint64_t)(k * 32 >> 4);       // +32 bytes per K=16 step inside the 64-byte row
                    umma_bf16(d_tmem, zh + ko, bh + ko, idesc, k != 0);
                    umma_bf16(d_tmem, zh + ko, bl + ko, idesc, 1);
                    umma_bf16(d_tmem, zl + ko, bh + ko, idesc, 1);
                }
                umma_commit(bar_empty + 8 * stage);
                umma_commit(bar_tfull + 8 * ab);
                if (++stage == TB_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;
        // staging: per warp TB_SBUF buffers of [32 samples][hi | lo][64 activations] = 8 KB, SWIZZLE_128B.  The TMA store engine is
        // bound by ROWS: lone 64-byte rows capped the kernel at 2.2 TB/s of writes, lone 128-byte rows (hi and lo planes as two
        // tensors) at 3.6 TB/s = 8.7 ms per 128 samples.  Interleaving the planes per block of 64 activations makes every
        // sample's (hi, lo) segments ADJACENT in memory, one box row pair = 256 contiguous bytes: 7.3 ms (4.3 TB/s of writes next
        // to 1.1 TB/s of basis reads, i.e. the HBM roofline; profiles/micro/tma_store_rows.cu measures 4.5 -> 5.8 TB/s for the
        // store engine alone).  The GEMM reads the same rows as before (hi tile of k-block kb at column 128 kb, lo at 128 kb + 64).
        // Also measured and dropped: one 256-byte 1-D bulk copy per lane and half tile (10.3 ms: the engine then pays per
        // instruction); the lo halves through the LSU, scattered (32 ms) or read back transposed and coalesced (8.8 ms); and
        // two output layouts that make these stores (nearly) sequential, [e/64][sample][64] and [datapoint][sample][width]:
        // the layer drops to 6.7 / 7.6 ms, but the GEMM kernel that reads the activations then loses its contiguous A tiles
        // and slows from 32.0 to 34.3 / 34.5 ms per 128 samples (DRAM reads 57 -> 75 GB), a net loss.
        const uint32_t stage_w = smem_base + TB_OFF_STORE + (uint32_t)(warp - 2) * (TB_SBUF * 8192);
        const uint32_t swz_h = (uint32_t)((2 * lane) & 7), swz_l = (uint32_t)((2 * lane + 1) & 7);     // SWIZZLE_128B: chunk ^ (row & 7)
        const float pre_inv = zinv ? zinv[q * 32 + lane] : 1.0f;      // this thread's sample (TMEM lane)
        float amx = 0.0f;
        uint32_t chunk_ctr = 0, tile = 0, sbuf = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tile) {
            const uint32_t ab = tile & 1, aphase = (tile >> 1) & 1;
            mbar_wait(bar_tfull + 8 * ab, aphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ab * 256;
#pragma unroll 1
            for (int c0 = 0; c0 < TB_N; c0 += 64, ++chunk_ctr) {
                if (chunk_ctr >= TB_SBUF) {
                    if (lane == 0) tma_store_wait_read<TB_SBUF - 1>();
                    __syncwarp();
                }
                // staging box [32 samples][hi | lo][128 B]: row 2*lane is the sample's hi segment, row 2*lane + 1 its lo segment
                const uint32_t sh = stage_w + sbuf * 8192;
                if (++sbuf == TB_SBUF) sbuf = 0;
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c0 + 32 * half, v);
                    tmem_ld_wait();
                    uint32_t hi[16], lo[16];
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        const float x0 = tc_act<ACT>(__uint_as_float(v[j]) * pre_inv);       // powers of two: exact
                        const float x1 = tc_act<ACT>(__uint_as_float(v[j + 1]) * pre_inv);
                        amx = fmaxf(amx, fmaxf(fabsf(x0), fabsf(x1)));
                        tc_split_a2<PREC>(x0 * a_scale, x1 * a_scale, hi[j >> 1], lo[j >> 1]);
                    }
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const uint32_t ch = (uint32_t)(4 * half + c);
                        st_shared_v4(sh + (uint32_t)lane * 256 + ((ch ^ swz_h) << 4), hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
                        st_shared_v4(sh + (uint32_t)lane * 256 + 128 + ((ch ^ swz_l) << 4), lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    // rows = samples (rows >= G are clipped by TMA), columns = activations e of this tile
                    // one store of 32 x 256 contiguous bytes: segment index = 2 * (64-activation block), hi and lo adjacent
                    tma_store_3d_hint(&tmO, sh, 0, 2 * ((t * TB_N + c0) >> 6), q * 32, TC_EVICT_FIRST);
                    tma_store_commit();
                }
            }
            tc_fence_before();
            mbar_arrive(bar_tempty + 8 * ab);
        }
        tc_amax_commit(amax, amx);
        if (lane == 0) tma_store_wait_all();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// zaug[s][m] = z[m, s] (m < M), 1 (m == M: the W_swa basis), 0 (padding and s >= G), split into two planes, [128][32].
// kind 0: BF16 planes.  kind 1: FP16 planes, row s scaled by 2^jz_s with max(1, max_m |z_ms|) * 2^jz_s in [2^13, 2^14) -- a
// function of the sample alone (bitwise batch invariance); zinv[s] = 2^-jz_s * bases_inv.  One warp per sample.
__global__ void k_tc_pack_zaug(const float* __restrict__ Z, int M, int G, int kind, float bases_inv, bf16* __restrict__ zh, bf16* __restrict__ zl,
                               float* __restrict__ zinv) {
    const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), m = threadIdx.x & 31;
    if (s >= 128) return;
    const float v = s < G ? (m < M ? Z[m + (long long)s * M] : (m == M ? 1.0f : 0.0f)) : 0.0f;
    float scale = 1.0f;
    if (kind == 1) {
        float mx = fabsf(v);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        int jz = 0;
        if (mx > 0.0f && mx < 3.0e38f) jz = max(-100, min(100, 13 - ilogbf(mx)));
        scale = scalbnf(1.0f, jz);
        if (m == 0) zinv[s] = scalbnf(1.0f, -jz) * bases_inv;
    }
    unsigned short hi, lo;
    tc_split1(v * scale, kind, hi, lo);
    reinterpret_cast<unsigned short*>(zh)[s * 32 + m] = hi;
    reinterpret_cast<unsigned short*>(zl)[s * 32 + m] = lo;
}

// basesT[e][m] (K-major, KT 16-bit values per activation e, two planes)  <-  bases[m][e] FP32, m <= M.  KT = 24 when M + 1 <= 24 (48-byte
// rows; the TMA box stays 32 wide and the 8 columns past the tensor's edge arrive as zeros), else 32: the kernel that reads
// this stream is HBM-bound and a quarter of a 32-wide row would be padding for M = 20.  kind 0: BF16 planes; 1: FP16 planes
// scaled by 2^jb so that max |bases| < 2^14.
__global__ void __launch_bounds__(256)
k_tc_bases_kmajor(const float* __restrict__ bases, long long NW, int M1, int KT, int kind, float scale, bf16* __restrict__ th, bf16* __restrict__ tl) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= NW) return;
    __align__(16) unsigned short hi[32], lo[32];
#pragma unroll
    for (int m = 0; m < 32; ++m) {
        const float v = m < M1 ? bases[(long long)m * NW + e] : 0.0f;
        tc_split1(v * scale, kind, hi[m], lo[m]);
    }
    uint4* dh = reinterpret_cast<uint4*>(th + e * KT);
    uint4* dl = reinterpret_cast<uint4*>(tl + e * KT);
#pragma unroll
    for (int c = 0; c < 4; ++c)
        if (c * 8 < KT) { dh[c] = reinterpret_cast<const uint4*>(hi)[c]; dl[c] = reinterpret_cast<const uint4*>(lo)[c]; }
}

// zpack[g][m] <- Z[m + g*M], zero padded  (staging for the device-to-constant copy)
__global__ void k_tc_pack_z(const float* __restrict__ Z, int M, int G, float* __restrict__ out /* [TC_GMAX][SSI_MAX_M] */) {
    const int t = threadIdx.x + blockIdx.x * blockDim.x;
    if (t >= TC_GMAX * SSI_MAX_M) return;
    const int g = t / SSI_MAX_M, m = t % SSI_MAX_M;
    out[t] = (g < G && m < M) ? Z[m + g * M] : 0.0f;
}

template <int MP>
static void tc_launch_basis(int act, unsigned blocks, cudaStream_t st, const float* bases, long long NW, int M, int G, const float* zpack,
                            bf16* Hh, bf16* Hl, int fp16, float a_scale, float* amax) {
    switch (act) {
        case SSI_ACT_RELU:    k_tc_basis_layer<SSI_ACT_RELU, MP><<<blocks, TC_BASIS_THREADS, 0, st>>>(bases, NW, M, G, zpack, Hh, Hl, fp16, a_scale, amax); break;
        case SSI_ACT_TANH:    k_tc_basis_layer<SSI_ACT_TANH, MP><<<blocks, TC_BASIS_THREADS, 0, st>>>(bases, NW, M, G, zpack, Hh, Hl, fp16, a_scale, amax); break;
        case SSI_ACT_SIGMOID: k_tc_basis_layer<SSI_ACT_SIGMOID, MP><<<blocks, TC_BASIS_THREADS, 0, st>>>(bases, NW, M, G, zpack, Hh, Hl, fp16, a_scale, amax); break;
        default:              k_tc_basis_layer<SSI_ACT_IDENTITY, MP><<<blocks, TC_BASIS_THREADS, 0, st>>>(bases, NW, M, G, zpack, Hh, Hl, fp16, a_scale, amax); break;
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct ssi_tc_state {
    bool ready = false;
    int prec = TC_PREC_FP16X3;           // plane formats in use (option "tc_precision"; BF16X3 after a range fallback)
    bool fallback = false;               // an evaluation exceeded FP16's range: this (data, subspace) stays on BF16 planes
    tc_ja_t ja_in{};                     // FP16 planes: exponent of the scale of the A planes GEMM layer l consumes
    float* amax = nullptr;               // [SSI_MAX_LAYERS + 1] largest |activation| written into the A planes of layer l
    int nl = 0;                          // GEMM launches per group: L, or L-1 when the output layer is fused
    bool fused_out = false;              // output layer folded into the last hidden layer's epilogue (O <= TC_OP)
    bool basis = false;                  // first layer = affine-in-z combination of precomputed bases (k_tc_basis_layer)
    int l0 = 0;                          // first Dense layer that runs as a GEMM (1 when basis)
    float* bases = nullptr;              // [M+1][N][width0] FP32
    float* zpack = nullptr;              // [TC_GMAX][SSI_MAX_M] z of the current group, zero padded
    float *Wout = nullptr, *bout = nullptr;
    int Kp[SSI_MAX_LAYERS] = {0};        // padded input width of layer l
    int width[SSI_MAX_LAYERS] = {0};     // padded output width of layer l
    int BN[SSI_MAX_LAYERS] = {0};
    int G = TC_GMAX;                     // samples per group (multiples of TC_GMAX are handled TC_GMAX at a time by the SIMT kernels)
    bf16 *Xh = nullptr, *Xl = nullptr;
    bf16 *Wh[SSI_MAX_LAYERS] = {nullptr}, *Wl[SSI_MAX_LAYERS] = {nullptr};
    float* bias[SSI_MAX_LAYERS] = {nullptr};
    bf16 *Hh[2] = {nullptr, nullptr}, *Hl[2] = {nullptr, nullptr};
    // FP16 planes: column maxima of [P | W_swa] per GEMM layer, per-sample weight scales and their inverses [nl][G],
    // per-sample inverse scales of the first-layer GEMM [128]
    float *cmax = nullptr, *wscale = nullptr, *winv = nullptr, *zinv = nullptr;
    float bases_scale = 1.0f;            // 2^jb of the K-major bases (FP16 planes)
    // basis-layer output [G][N][width0] (hi, lo) and its tensor maps as the A operand of the first GEMM layer
    bf16* Bh = nullptr;                      // basis layer output [G][N][width/64][hi 64 | lo 64] (planes interleaved per k-block)
    CUtensorMap tmBasisH, tmBasisL;
    // basis layer on the tensor cores (k_tc_basis_mma): K-major two-plane bases [N*width0][KT], z of the group [128][32]
    bool basis_mma = false;
    bf16 *Th = nullptr, *Tl = nullptr, *Zh = nullptr, *Zl = nullptr;
    CUtensorMap tmZh, tmZl, tmTh, tmTl, tmO;
    int KT = 32;                             // columns per row of Th / Tl (24 or 32)
    double* partials = nullptr;
    CUtensorMap tmAh[SSI_MAX_LAYERS], tmAl[SSI_MAX_LAYERS], tmBh[SSI_MAX_LAYERS], tmBl[SSI_MAX_LAYERS];
    CUtensorMap tmBh2[SSI_MAX_LAYERS], tmBl2[SSI_MAX_LAYERS];     // boxes of BN/2 rows (CTA pairs)
    CUtensorMap tmSh[SSI_MAX_LAYERS], tmSl[SSI_MAX_LAYERS];
    PFN_encodeTiled encode = nullptr;
};

static void tc_free(ssi_tc_state* s) {
    cudaFree(s->Xh); cudaFree(s->Xl); cudaFree(s->partials); cudaFree(s->Wout); cudaFree(s->bout); cudaFree(s->bases); cudaFree(s->zpack);
    cudaFree(s->cmax); cudaFree(s->wscale); cudaFree(s->winv); cudaFree(s->zinv); cudaFree(s->amax);
    for (int i = 0; i < 2; ++i) { cudaFree(s->Hh[i]); cudaFree(s->Hl[i]); }
    cudaFree(s->Bh); cudaFree(s->Th); cudaFree(s->Tl); cudaFree(s->Zh); cudaFree(s->Zl);
    for (int l = 0; l < SSI_MAX_LAYERS; ++l) { cudaFree(s->Wh[l]); cudaFree(s->Wl[l]); cudaFree(s->bias[l]); }
    PFN_encodeTiled enc = s->encode;
    *s = ssi_tc_state();
    s->encode = enc;
    (void)cudaGetLastError();
}

void ssi_tc_invalidate(ssi_ctx* ctx) {
    if (ctx->tc) ctx->tc->ready = false;
}

void ssi_tc_destroy(ssi_ctx* ctx) {
    if (!ctx->tc) return;
    tc_free(ctx->tc);
    delete ctx->tc;
    ctx->tc = nullptr;
}

// Any Dense chain runs on this path (widths are zero-padded); AUTO prefers it when the padded
// tensor-core work is not dominated by padding, i.e. the layers are wide.
bool ssi_tc_supported(const ssi_ctx* ctx) {
    if (!ctx->has_model) return false;
    const ssi_model_t& m = ctx->model;
    if (m.dims[m.L] > 256 || ctx->M > SSI_MAX_M) return false;
    return true;
}

bool ssi_tc_preferred(const ssi_ctx* ctx) {
    if (!ssi_tc_supported(ctx)) return false;
    const ssi_model_t& m = ctx->model;
    double real = 0, padded = 0;
    for (int l = 0; l < m.L; ++l) {
        const double kp = (m.dims[l] + 63) / 64 * 64;
        const double np = l == m.L - 1 ? (m.dims[l + 1] + 15) / 16 * 16 : (m.dims[l + 1] + 63) / 64 * 64;
        real += (double)m.dims[l] * m.dims[l + 1];
        padded += kp * np;
    }
    return real >= 64.0 * 64.0 && padded <= 2.0 * real;
}

typedef void (*tc_kernel_t)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap,
                            const CUtensorMap, const tc_params);
// only the HIDDEN epilogue writes operand planes: the other modes have one instantiation per activation
template <int MODE, int PREC, bool PAIR>
static tc_kernel_t tc_kernel_for_act(int act) {
    switch (act) {
        case SSI_ACT_RELU:    return k_tc_layer<MODE, SSI_ACT_RELU, PREC, PAIR>;
        case SSI_ACT_TANH:    return k_tc_layer<MODE, SSI_ACT_TANH, PREC, PAIR>;
        case SSI_ACT_SIGMOID: return k_tc_layer<MODE, SSI_ACT_SIGMOID, PREC, PAIR>;
        default:              return k_tc_layer<MODE, SSI_ACT_IDENTITY, PREC, PAIR>;
    }
}
template <bool PAIR>
static tc_kernel_t tc_kernel_p(int mode, int act, int prec) {
    if (mode == TC_MODE_FUSED) return tc_kernel_for_act<TC_MODE_FUSED, 0, PAIR>(act);
    if (mode == TC_MODE_FINAL) return tc_kernel_for_act<TC_MODE_FINAL, 0, PAIR>(act);
    return prec == TC_PREC_FP16X3 ? tc_kernel_for_act<TC_MODE_HIDDEN, TC_PREC_FP16X3, PAIR>(act) : tc_kernel_for_act<TC_MODE_HIDDEN, TC_PREC_BF16X3, PAIR>(act);
}
static tc_kernel_t tc_kernel(int mode, int act, int prec, bool pair = false) {
    return pair ? tc_kernel_p<true>(mode, act, prec) : tc_kernel_p<false>(mode, act, prec);
}

typedef void (*tb_kernel_t)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const int,
                            const float*, const float, float*);
template <int PREC>
static tb_kernel_t tb_kernel_for_act(int act) {
    switch (act) {
        case SSI_ACT_RELU:    return k_tc_basis_mma<SSI_ACT_RELU, PREC>;
        case SSI_ACT_TANH:    return k_tc_basis_mma<SSI_ACT_TANH, PREC>;
        case SSI_ACT_SIGMOID: return k_tc_basis_mma<SSI_ACT_SIGMOID, PREC>;
        default:              return k_tc_basis_mma<SSI_ACT_IDENTITY, PREC>;
    }
}
static tb_kernel_t tb_kernel(int act, int prec) {
    return prec == TC_PREC_FP16X3 ? tb_kernel_for_act<TC_PREC_FP16X3>(act) : tb_kernel_for_act<TC_PREC_BF16X3>(act);
}

static int tc_make_map(ssi_ctx* ctx, CUtensorMap* map, void* base, uint64_t inner, uint64_t rows, uint64_t batch,
                       uint32_t box_inner, uint32_t box_rows, CUtensorMapSwizzle swz) {
    cuuint64_t dims[3] = {inner, rows, batch};
    cuuint64_t strides[2] = {inner * sizeof(bf16), inner * rows * sizeof(bf16)};
    cuuint32_t box[3] = {box_inner, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    // the planes hold BF16 or FP16 bit patterns; TMA only moves 16-bit elements (out-of-bounds elements are zero filled)
    const CUresult r = ctx->tc->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, estr,
                                       CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return ssi_fail(ctx, SSI_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return SSI_OK;
}

// device memory of the tensor path for a group of G samples (bytes), given whether the first layer runs on the bases
static double tc_group_bytes(const ssi_ctx* ctx, bool basis, int G) {
    const ssi_model_t& m = ctx->model;
    const double N = (double)ctx->N;
    const int l0 = basis ? 1 : 0;
    const bool fused = (m.L - l0 >= 2 && m.dims[m.L] <= TC_OP && !ctx->opt_tc_nofuse);
    const int nl = fused ? m.L - 1 : m.L;
    double bytes = 0, maxw = 0;
    for (int l = l0; l < nl; ++l) {
        const double kp = (m.dims[l] + 63) / 64 * 64;
        const double w = (l == m.L - 1) ? (m.dims[l + 1] + 15) / 16 * 16 : (m.dims[l + 1] + 63) / 64 * 64;
        bytes += 4.0 * G * w * kp + 4.0 * G * w;                      // two weight planes + bias
        if (l < nl - 1) maxw = std::max(maxw, w);
    }
    const int stored = std::max(0, nl - 1 - l0);                      // GEMM layers whose activations are stored
    bytes += 4.0 * G * N * maxw * std::min(stored, 2);                // ping-pong buffers, two planes each
    if (basis) bytes += 4.0 * G * N * ((m.dims[1] + 63) / 64 * 64);   // the basis layer's output
    return bytes;
}

int ssi_tc_sse(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse);

static int tc_exp_for(float mx, int top) {       // 2^j with mx * 2^j in [2^top, 2^(top + 1))
    if (!(mx > 0.0f) || !(mx < 3.0e38f)) return 0;
    return std::max(-100, std::min(100, top - ilogbf(mx)));
}

// max |x| of a device array (synchronises)
static int tc_absmax_host(ssi_ctx* ctx, const float* d, long long count, float* out) {
    unsigned* d_mx = reinterpret_cast<unsigned*>(ctx->tc->amax + SSI_MAX_LAYERS);      // last slot: scratch outside calibrated layers
    SSI_CUDA(ctx, cudaMemsetAsync(d_mx, 0, sizeof(unsigned), ctx->stream));
    k_tc_absmax<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(d, count, d_mx);
    SSI_LAUNCH_CHECK(ctx);
    SSI_CUDA(ctx, cudaMemcpyAsync(out, d_mx, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SSI_CUDA(ctx, cudaMemsetAsync(d_mx, 0, sizeof(unsigned), ctx->stream));
    return SSI_OK;
}

// operands that depend on (data, subspace) only, in the plane format of s->prec: the K-major bases of the first-layer GEMM,
// or the planes of the dataset when the first layer is a GEMM on X
static int tc_build_static_operands(ssi_ctx* ctx) {
    ssi_tc_state* s = ctx->tc;
    const ssi_model_t& m = ctx->model;
    const int64_t N = ctx->N;
    const bool fp16 = s->prec == TC_PREC_FP16X3;
    if (s->basis_mma) {
        const long long NW = (long long)N * s->width[0];
        s->bases_scale = 1.0f;
        if (fp16) {
            float mx = 0.0f;
            SSI_TRY(tc_absmax_host(ctx, s->bases, (long long)(ctx->M + 1) * NW, &mx));
            s->bases_scale = scalbnf(1.0f, tc_exp_for(mx, 13));
        }
        k_tc_bases_kmajor<<<(unsigned)((NW + 255) / 256), 256, 0, ctx->stream>>>(s->bases, NW, ctx->M + 1, s->KT, fp16 ? 1 : 0, s->bases_scale, s->Th, s->Tl);
        SSI_LAUNCH_CHECK(ctx);
    }
    if (!s->basis) {
        float xs = 1.0f;
        s->ja_in.v[0] = 0;
        if (fp16) {
            float mx = 0.0f;
            SSI_TRY(tc_absmax_host(ctx, ctx->dX, (long long)N * m.dims[0], &mx));
            s->ja_in.v[0] = tc_exp_for(mx, 13);
            xs = scalbnf(1.0f, s->ja_in.v[0]);
        }
        const long long tot = (long long)N * s->Kp[0];
        k_tc_split_x<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(ctx->dX, N, m.dims[0], s->Kp[0], fp16 ? 1 : 0, xs, s->Xh, s->Xl);
        SSI_LAUNCH_CHECK(ctx);
    }
    return SSI_OK;
}

// One evaluation at z = 0 on BF16 planes records the largest activation every layer writes; the FP16 scale of layer l's A
// planes maps it to [2^TC_CAL_TOP, 2^(TC_CAL_TOP+1)): 64x..128x of headroom below FP16's maximum for the other samples.
static int tc_calibrate(ssi_ctx* ctx) {
    ssi_tc_state* s = ctx->tc;
    float* dz = nullptr;
    double* dsse = nullptr;
    SSI_CUDA(ctx, cudaMalloc(&dz, sizeof(float) * SSI_MAX_M));
    SSI_CUDA(ctx, cudaMalloc(&dsse, sizeof(double)));
    cudaMemsetAsync(dz, 0, sizeof(float) * SSI_MAX_M, ctx->stream);
    const int64_t launches = ctx->stats.kernel_launches;
    const int rc = ssi_tc_sse(ctx, dz, 1, dsse);
    float h[SSI_MAX_LAYERS + 1] = {0};
    cudaMemcpyAsync(h, s->amax, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream);
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    cudaFree(dz); cudaFree(dsse);
    ctx->stats.kernel_launches = launches;               // preparation, not part of any call's count
    if (rc != SSI_OK) return rc;
    SSI_CUDA(ctx, e);
    for (int l = s->l0; l < s->nl; ++l)
        if (l > 0) s->ja_in.v[l] = tc_exp_for(h[l], TC_CAL_TOP);     // layer 0 reads the dataset: exact scale, set with its planes
    SSI_CUDA(ctx, cudaMemsetAsync(s->amax, 0, sizeof(float) * (SSI_MAX_LAYERS + 1), ctx->stream));
    s->prec = TC_PREC_FP16X3;
    SSI_TRY(tc_build_static_operands(ctx));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSI_OK;
}

// Did an evaluation since the last check write an activation beyond the range of its FP16 planes?  (Called where the host
// entry points have synchronised anyway.)  If so this (data, subspace) moves to BF16 planes for good and the caller repeats
// its evaluation.
int ssi_tc_range_exceeded(ssi_ctx* ctx, bool* exceeded) {
    *exceeded = false;
    ssi_tc_state* s = ctx->tc;
    if (!s || !s->ready || s->prec != TC_PREC_FP16X3) return SSI_OK;
    float h[SSI_MAX_LAYERS + 1];
    SSI_CUDA(ctx, cudaMemcpyAsync(h, s->amax, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int l = std::max(1, s->l0); l < s->nl; ++l)
        if (h[l] * scalbnf(1.0f, s->ja_in.v[l]) > 0.999f * TC_F16_MAX) *exceeded = true;
    if (*exceeded) {
        s->fallback = true;
        s->prec = TC_PREC_BF16X3;
        for (int l = 0; l <= SSI_MAX_LAYERS; ++l) s->ja_in.v[l] = 0;
        SSI_CUDA(ctx, cudaMemsetAsync(s->amax, 0, sizeof(float) * (SSI_MAX_LAYERS + 1), ctx->stream));
        SSI_TRY(tc_build_static_operands(ctx));
        ctx->stats.tc_range_fallbacks++;
    }
    return SSI_OK;
}

int ssi_tc_prepare(ssi_ctx* ctx) {
    if (!ssi_tc_supported(ctx)) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "tensor path: output width > 256 is not supported");
    if (!ctx->tc) ctx->tc = new ssi_tc_state();
    ssi_tc_state* s = ctx->tc;
    if (s->ready) return SSI_OK;
    if (!s->encode) {
        PFN_ssi_encodeTiled fn = nullptr;
        SSI_TRY(ssi_tensormap_encoder(ctx, &fn));
        s->encode = (PFN_encodeTiled)fn;
    }
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    tc_free(s);
    const int rc = [&]() -> int {
    const ssi_model_t& m = ctx->model;
    const int64_t N = ctx->N;
    const bool want_fp16 = ctx->opt_tc_prec != 0;
    s->prec = TC_PREC_BF16X3;            // the calibration pass below runs on BF16 planes, which cannot overflow
    // Sizing against the memory that is actually free (the caller -- e.g. a torch process -- may hold part of the device):
    // the first layer runs on precomputed bases when they (FP32 + K-major planes) take at most a third of what is free, and
    // a group of samples gets at most 60 % of what is left after them.
    size_t mem_free = 0, mem_total = 0;
    SSI_CUDA(ctx, cudaMemGetInfo(&mem_free, &mem_total));
    const int w0pad = (m.dims[1] + 63) / 64 * 64;
    const double bases_bytes = (double)(ctx->M + 1) * (double)N * w0pad * sizeof(float);
    const double bases_all = bases_bytes + 4.0 * (double)N * w0pad * 32;
    s->basis = (m.L >= 2 && !ctx->opt_tc_nobasis && bases_all <= (double)mem_free / 3.0);
    s->l0 = s->basis ? 1 : 0;
    s->fused_out = (m.L - s->l0 >= 2 && m.dims[m.L] <= TC_OP && !ctx->opt_tc_nofuse);
    s->nl = s->fused_out ? m.L - 1 : m.L;
    // the basis layer runs on the tensor cores when z (plus the constant 1) fits one K = 32 block; its M dimension is the
    // samples, so a group is then 128 samples (the bases are read once per group)
    s->basis_mma = s->basis && ctx->M + 1 <= 32 && !ctx->opt_tc_simt_basis;
    int gmax = s->basis_mma ? 128 : TC_GMAX;
    {
        const double budget = 0.6 * ((double)mem_free - (s->basis ? bases_all : 4.0 * (double)N * ((m.dims[0] + 63) / 64 * 64)));
        while (gmax > TC_GMAX && tc_group_bytes(ctx, s->basis, gmax) > budget) gmax -= TC_GMAX;
        while (gmax > 1 && tc_group_bytes(ctx, s->basis, gmax) > budget) gmax /= 2;
        if (tc_group_bytes(ctx, s->basis, gmax) > budget)
            return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "tensor path: one sample needs %.1f GB of activations but only %.1f GB of device memory is free",
                            tc_group_bytes(ctx, s->basis, 1) / 1e9, (double)mem_free / 1e9);
    }
    s->G = ctx->opt_group > 0 ? std::min(ctx->opt_group, gmax) : gmax;
    const int G = s->G;
    int maxw = 0;
    for (int l = 0; l < s->nl; ++l) {
        const bool last = (l == m.L - 1);          // a true output layer computed as a GEMM
        s->Kp[l] = (m.dims[l] + TC_BK - 1) / TC_BK * TC_BK;
        s->width[l] = last ? (m.dims[l + 1] + 15) / 16 * 16 : (m.dims[l + 1] + 63) / 64 * 64;
        if (last) s->BN[l] = s->width[l];            // <= 256, a multiple of 16
        else s->BN[l] = s->width[l] % 256 == 0 ? 256 : (s->width[l] % 128 == 0 ? 128 : 64);
        if (l < s->nl - 1) maxw = std::max(maxw, s->width[l]);
        if (l < s->l0) continue;                 // the basis layer has no GEMM operands
        const size_t wn = (size_t)G * s->width[l] * s->Kp[l];
        SSI_CUDA(ctx, cudaMalloc(&s->Wh[l], sizeof(bf16) * wn));
        SSI_CUDA(ctx, cudaMalloc(&s->Wl[l], sizeof(bf16) * wn));
        SSI_CUDA(ctx, cudaMalloc(&s->bias[l], sizeof(float) * (size_t)G * s->width[l]));
    }
    SSI_CUDA(ctx, cudaMalloc(&s->amax, sizeof(float) * (SSI_MAX_LAYERS + 1)));
    SSI_CUDA(ctx, cudaMemsetAsync(s->amax, 0, sizeof(float) * (SSI_MAX_LAYERS + 1), ctx->stream));
    if (want_fp16) {
        SSI_CUDA(ctx, cudaMalloc(&s->zinv, sizeof(float) * 128));
        SSI_CUDA(ctx, cudaMalloc(&s->cmax, sizeof(float) * (size_t)s->nl * (ctx->M + 1)));
        SSI_CUDA(ctx, cudaMalloc(&s->wscale, sizeof(float) * (size_t)s->nl * G));
        SSI_CUDA(ctx, cudaMalloc(&s->winv, sizeof(float) * (size_t)s->nl * G));
        SSI_CUDA(ctx, cudaMemsetAsync(s->cmax, 0, sizeof(float) * (size_t)s->nl * (ctx->M + 1), ctx->stream));
        for (int l = s->l0; l < s->nl; ++l) {
            k_tc_colmax<<<ctx->M + 1, 256, 0, ctx->stream>>>(ctx->dP, m.n, m.w_off[l], (long long)m.dims[l] * m.dims[l + 1],
                                                            s->cmax + (size_t)l * (ctx->M + 1));
            SSI_LAUNCH_CHECK(ctx);
        }
    }
    if (s->fused_out) {
        const int wl = s->width[s->nl - 1];
        SSI_CUDA(ctx, cudaMalloc(&s->Wout, sizeof(float) * (size_t)G * wl * TC_OP));
        SSI_CUDA(ctx, cudaMalloc(&s->bout, sizeof(float) * (size_t)G * TC_OP));
        SSI_CUDA(ctx, cudaMemsetAsync(s->Wout, 0, sizeof(float) * (size_t)G * wl * TC_OP, ctx->stream));
        SSI_CUDA(ctx, cudaMemsetAsync(s->bout, 0, sizeof(float) * (size_t)G * TC_OP, ctx->stream));
    }
    if (s->basis) {
        SSI_CUDA(ctx, cudaMalloc(&s->bases, (size_t)bases_bytes));
        SSI_CUDA(ctx, cudaMalloc(&s->zpack, sizeof(float) * TC_GMAX * SSI_MAX_M));
        if (w0pad != m.dims[1]) SSI_CUDA(ctx, cudaMemsetAsync(s->bases, 0, (size_t)bases_bytes, ctx->stream));
        SSI_TRY(ssi_build_first_layer_bases(ctx, s->bases, w0pad));
    } else {
        SSI_CUDA(ctx, cudaMalloc(&s->Xh, sizeof(bf16) * (size_t)N * s->Kp[0]));
        SSI_CUDA(ctx, cudaMalloc(&s->Xl, sizeof(bf16) * (size_t)N * s->Kp[0]));
    }
    // GEMM layers l0..nl-2 store their activations in H[l & 1]; the basis layer has its own double buffer
    for (int l = s->l0; l <= s->nl - 2; ++l) {
        const int i = l & 1;
        if (s->Hh[i]) continue;
        SSI_CUDA(ctx, cudaMalloc(&s->Hh[i], sizeof(bf16) * (size_t)G * N * maxw));
        SSI_CUDA(ctx, cudaMalloc(&s->Hl[i], sizeof(bf16) * (size_t)G * N * maxw));
    }
    if (s->basis) {
        const size_t NW = (size_t)N * s->width[0];
        SSI_CUDA(ctx, cudaMalloc(&s->Bh, sizeof(bf16) * 2 * (size_t)G * NW));
        if (s->basis_mma) {
            s->KT = ctx->M + 1 <= 24 ? 24 : 32;
            SSI_CUDA(ctx, cudaMalloc(&s->Th, sizeof(bf16) * NW * s->KT));
            SSI_CUDA(ctx, cudaMalloc(&s->Tl, sizeof(bf16) * NW * s->KT));
            SSI_CUDA(ctx, cudaMalloc(&s->Zh, sizeof(bf16) * 128 * 32));
            SSI_CUDA(ctx, cudaMalloc(&s->Zl, sizeof(bf16) * 128 * 32));
        }
    }
    const int m_tiles = (int)((N + TC_BM - 1) / TC_BM);
    SSI_CUDA(ctx, cudaMalloc(&s->partials, sizeof(double) * (size_t)G * m_tiles * 4));
    for (int l = s->l0; l < s->nl; ++l) {
        const CUtensorMapSwizzle S128 = CU_TENSOR_MAP_SWIZZLE_128B, S64 = CU_TENSOR_MAP_SWIZZLE_64B;
        if (l == 0) {
            SSI_TRY(tc_make_map(ctx, &s->tmAh[l], s->Xh, s->Kp[0], N, 1, TC_BK, TC_BM, S128));
            SSI_TRY(tc_make_map(ctx, &s->tmAl[l], s->Xl, s->Kp[0], N, 1, TC_BK, TC_BM, S128));
        } else if (l == s->l0) {
            // activations written by the basis layer: [G][N][width_0]
            // rows of 2 * width: [kb][hi 64 | lo 64]; the hi tile of k-block kb sits at column 128 kb, the lo tile at 128 kb + 64
            SSI_TRY(tc_make_map(ctx, &s->tmBasisH, s->Bh, 2 * (uint64_t)s->width[0], N, G, TC_BK, TC_BM, S128));
            s->tmBasisL = s->tmBasisH;
            s->tmAh[l] = s->tmBasisH;
            s->tmAl[l] = s->tmBasisL;
        } else {
            // activations written by layer l-1: [G][N][width_{l-1}], K = width_{l-1} = Kp[l]
            SSI_TRY(tc_make_map(ctx, &s->tmAh[l], s->Hh[(l - 1) & 1], s->width[l - 1], N, G, TC_BK, TC_BM, S128));
            SSI_TRY(tc_make_map(ctx, &s->tmAl[l], s->Hl[(l - 1) & 1], s->width[l - 1], N, G, TC_BK, TC_BM, S128));
        }
        SSI_TRY(tc_make_map(ctx, &s->tmBh[l], s->Wh[l], s->Kp[l], s->width[l], G, TC_BK, s->BN[l], S128));
        SSI_TRY(tc_make_map(ctx, &s->tmBl[l], s->Wl[l], s->Kp[l], s->width[l], G, TC_BK, s->BN[l], S128));
        SSI_TRY(tc_make_map(ctx, &s->tmBh2[l], s->Wh[l], s->Kp[l], s->width[l], G, TC_BK, s->BN[l] / 2, S128));
        SSI_TRY(tc_make_map(ctx, &s->tmBl2[l], s->Wl[l], s->Kp[l], s->width[l], G, TC_BK, s->BN[l] / 2, S128));
        if (l < s->nl - 1) {
            // epilogue stores of this layer's activations: 32 rows x 32 columns (64 B) per warp and chunk
            SSI_TRY(tc_make_map(ctx, &s->tmSh[l], s->Hh[l & 1], s->width[l], N, G, 32, 32, S64));
            SSI_TRY(tc_make_map(ctx, &s->tmSl[l], s->Hl[l & 1], s->width[l], N, G, 32, 32, S64));
        } else {
            s->tmSh[l] = s->tmAh[l];
            s->tmSl[l] = s->tmAl[l];
        }
    }
    for (int mode = 0; mode < 3; ++mode)
        for (int act = 0; act < 4; ++act)
            for (int prec = 0; prec < 2; ++prec)
                for (int pair = 0; pair < 2; ++pair)
                    SSI_CUDA(ctx, cudaFuncSetAttribute(tc_kernel(mode, act, prec, pair != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_total(mode)));
    if (s->basis_mma) {
        const CUtensorMapSwizzle S64 = CU_TENSOR_MAP_SWIZZLE_64B;
        const uint64_t NW = (uint64_t)N * s->width[0];
        SSI_TRY(tc_make_map(ctx, &s->tmZh, s->Zh, 32, 128, 1, 32, 128, S64));
        SSI_TRY(tc_make_map(ctx, &s->tmZl, s->Zl, 32, 128, 1, 32, 128, S64));
        SSI_TRY(tc_make_map(ctx, &s->tmTh, s->Th, (uint64_t)s->KT, NW, 1, 32, TB_N, S64));
        SSI_TRY(tc_make_map(ctx, &s->tmTl, s->Tl, (uint64_t)s->KT, NW, 1, 32, TB_N, S64));
        // the group's activations as a [samples][N*width0] matrix: boxes of 32 samples x 64 activations from the epilogue
        {   // store view: [samples][128-byte segments][64]; a box takes the (hi, lo) segment pair of 32 samples = 256 contiguous
            // bytes per sample (adjacent 128-byte rows: 5.8 TB/s through the TMA store engine against 4.5 for lone rows,
            // profiles/micro/tma_store_rows.cu)
            cuuint64_t dims[3] = {64, 2 * (cuuint64_t)NW / 64, (cuuint64_t)G};
            cuuint64_t strides[2] = {128, 2 * (cuuint64_t)NW * sizeof(bf16)};
            cuuint32_t box[3] = {64, 2, 32};
            cuuint32_t estr[3] = {1, 1, 1};
            const CUresult r = s->encode(&s->tmO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, s->Bh, dims, strides, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) return ssi_fail(ctx, SSI_ERR_CUDA, "cuTensorMapEncodeTiled (basis store) failed with CUresult %d", (int)r);
        }
        for (int act = 0; act < 4; ++act)
            for (int prec = 0; prec < 2; ++prec)
                SSI_CUDA(ctx, cudaFuncSetAttribute(tb_kernel(act, prec), cudaFuncAttributeMaxDynamicSharedMemorySize, TB_SMEM_TOTAL));
    }
    SSI_TRY(tc_build_static_operands(ctx));           // BF16 planes of the bases / the dataset
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    s->ready = true;
    if (want_fp16) SSI_TRY(tc_calibrate(ctx));       // one evaluation at z = 0 -> activation scales -> FP16 planes
    return SSI_OK;
    }();
    if (rc != SSI_OK) {          // do not keep a half-built state (and its allocations) around
        (void)cudaGetLastError();
        tc_free(s);
        return rc;
    }
    return SSI_OK;
}

int ssi_reduce_partials(ssi_ctx* ctx, const double* partials, int64_t B, int parts, double* d_out);

int ssi_tc_sse(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse) {
    SSI_TRY(ssi_tc_prepare(ctx));
    ssi_tc_state* s = ctx->tc;
    const ssi_model_t& m = ctx->model;
    const int64_t N = ctx->N, n = m.n;
    const int M = ctx->M;
    const int m_tiles = (int)((N + TC_BM - 1) / TC_BM);
    const int parts = m_tiles * 4;
    const long long NW = s->basis ? (long long)N * s->width[0] : 0;
    const bool fp16 = s->prec == TC_PREC_FP16X3;

    for (int64_t b0 = 0; b0 < B; b0 += s->G) {
        const int G = (int)std::min<int64_t>(s->G, B - b0);
        // ---- first layer as a combination of the precomputed bases ----
        if (s->basis_mma) {
            k_tc_pack_zaug<<<128 / 8, 256, 0, ctx->stream>>>(dZ + b0 * M, M, G, fp16 ? 1 : 0, 1.0f / s->bases_scale, s->Zh, s->Zl, s->zinv);
            SSI_LAUNCH_CHECK(ctx);
            const int n_tiles = (int)((NW + TB_N - 1) / TB_N);
            const int grid = std::min(ctx->sm_count, n_tiles);
            tb_kernel(m.act[0], s->prec)<<<grid, TC_THREADS, TB_SMEM_TOTAL, ctx->stream>>>(s->tmZh, s->tmZl, s->tmTh, s->tmTl, s->tmO, n_tiles,
                                                                                          fp16 ? s->zinv : nullptr,
                                                                                          scalbnf(1.0f, s->ja_in.v[1]), s->amax + 1);
            SSI_LAUNCH_CHECK(ctx);
        }
        if (fp16) {
            k_tc_wscale<<<(s->nl * G + 127) / 128, 128, 0, ctx->stream>>>(dZ + b0 * M, M, G, s->cmax, s->nl, s->G, s->ja_in, s->wscale, s->winv);
            SSI_LAUNCH_CHECK(ctx);
        }
        // ---- the SIMT kernels take TC_GMAX samples at a time ----
        for (int g0 = 0; g0 < G; g0 += TC_GMAX) {
            const int gs = std::min(TC_GMAX, G - g0);
            const float* Zg = dZ + (b0 + g0) * M;
            if (s->basis && !s->basis_mma) {
                k_tc_pack_z<<<(TC_GMAX * SSI_MAX_M + 255) / 256, 256, 0, ctx->stream>>>(Zg, M, gs, s->zpack);
                SSI_LAUNCH_CHECK(ctx);
                const long long per_cta = (long long)TC_BASIS_THREADS * TC_BASIS_ITERS * 2;
                const unsigned blocks = (unsigned)((NW + per_cta - 1) / per_cta);
                bf16* oh = s->Bh + 2 * (long long)g0 * NW;
                bf16* ol = nullptr;                                 // lo halves are interleaved behind the hi halves
                const int mx = fp16 ? 1 : 0;
                const float a1 = scalbnf(1.0f, s->ja_in.v[1]);
                float* am = s->amax + 1;
                if (M <= 8) tc_launch_basis<8>(m.act[0], blocks, ctx->stream, s->bases, NW, M, gs, s->zpack, oh, ol, mx, a1, am);
                else if (M <= 12) tc_launch_basis<12>(m.act[0], blocks, ctx->stream, s->bases, NW, M, gs, s->zpack, oh, ol, mx, a1, am);
                else if (M <= 20) tc_launch_basis<20>(m.act[0], blocks, ctx->stream, s->bases, NW, M, gs, s->zpack, oh, ol, mx, a1, am);
                else if (M <= 32) tc_launch_basis<32>(m.act[0], blocks, ctx->stream, s->bases, NW, M, gs, s->zpack, oh, ol, mx, a1, am);
                else tc_launch_basis<SSI_MAX_M>(m.act[0], blocks, ctx->stream, s->bases, NW, M, gs, s->zpack, oh, ol, mx, a1, am);
                SSI_LAUNCH_CHECK(ctx);
            }
            // K1: project the samples' weights straight into the GEMM operand layouts
            for (int l = s->l0; l < s->nl; ++l) {
                const size_t wo = (size_t)g0 * s->width[l] * s->Kp[l];
                dim3 grid(s->Kp[l] / PW_T, (s->width[l] + PW_T - 1) / PW_T);
                k_tc_project_w<<<grid, 256, 0, ctx->stream>>>(ctx->dWswa, ctx->dP, Zg, n, M, gs, m.w_off[l], m.dims[l], m.dims[l + 1],
                                                             s->width[l], s->Kp[l], fp16 ? s->wscale + (size_t)l * s->G + g0 : nullptr,
                                                             s->Wh[l] + wo, s->Wl[l] + wo);
                SSI_LAUNCH_CHECK(ctx);
                k_tc_project_b<<<(s->width[l] + 255) / 256, 256, 0, ctx->stream>>>(ctx->dWswa, ctx->dP, Zg, n, M, gs, m.b_off[l],
                                                                               m.dims[l + 1], s->width[l],
                                                                               s->bias[l] + (size_t)g0 * s->width[l]);
                SSI_LAUNCH_CHECK(ctx);
            }
            if (s->fused_out) {
                const int wl = s->width[s->nl - 1];          // padded width of the last hidden layer
                const int O = m.dims[m.L], cnt = m.dims[m.L - 1] * O;
                k_tc_project_v<<<(cnt + 255) / 256, 256, 0, ctx->stream>>>(ctx->dWswa, ctx->dP, Zg, n, M, gs, m.w_off[m.L - 1], cnt, O,
                                                                         TC_OP, (long long)wl * TC_OP,
                                                                         s->Wout + (size_t)g0 * wl * TC_OP);
                SSI_LAUNCH_CHECK(ctx);
                k_tc_project_v<<<1, 256, 0, ctx->stream>>>(ctx->dWswa, ctx->dP, Zg, n, M, gs, m.b_off[m.L - 1], O, O, 0, TC_OP,
                                                         s->bout + (size_t)g0 * TC_OP);
                SSI_LAUNCH_CHECK(ctx);
            }
        }
        // ---- the remaining Dense layers as GEMMs over the whole group ----
        for (int l = s->l0; l < s->nl; ++l) {
            tc_params p{};
            p.N = (int)N; p.G = G; p.m_tiles = m_tiles;
            p.BN = s->BN[l]; p.width = s->width[l];
            p.n_tiles = s->width[l] / s->BN[l];
            p.k_blocks = s->Kp[l] / TC_BK;
            p.a_shared = (l == 0);
            p.a_il = (l == 1 && s->basis) ? 1 : 0;
            p.k_rev = !p.a_shared ? 1 : 0;
            p.act = m.act[l];
            // CTA pairs for the layers with per-sample activations (weight rows split across the pair: BN / 2 must be a whole
            // number of 8-row swizzle atoms and a legal MMA N half)
            const bool pair = !p.a_shared && ctx->opt_tc_pair && p.BN >= 32 && (p.BN % 32) == 0 && ctx->sm_count >= 2;
            p.stage_bytes = 2 * TC_BM * TC_BK * 2 + 2 * (pair ? p.BN / 2 : p.BN) * TC_BK * 2;
            p.stage_bytes = (p.stage_bytes + 1023) / 1024 * 1024;
            p.stages = std::min(4, TC_SMEM_PIPE / p.stage_bytes);
            p.bias = s->bias[l];
            const uint32_t fmt = fp16 ? UMMA_FMT_F16 : UMMA_FMT_BF16;
            p.idesc = pair ? umma_idesc_f16_pair(p.BN, fmt, fmt) : umma_idesc_f16(p.BN, fmt, fmt);
            p.winv = fp16 ? s->winv + (size_t)l * s->G : nullptr;
            p.a_scale = scalbnf(1.0f, s->ja_in.v[l + 1]);         // of the planes this layer writes (HIDDEN)
            p.amax = s->amax + (l + 1);
            int grid = std::min(ctx->sm_count, G * m_tiles);
            // a shared A operand (the dataset): run the group's samples side by side on the same m-tiles
            p.mt_block = (p.a_shared && G > 1 && !ctx->opt_tc_noorder) ? std::max(1, (grid + G - 1) / G) : 0;
            p.n_work = p.mt_block > 0 ? (m_tiles + p.mt_block - 1) / p.mt_block * p.mt_block * G : G * m_tiles;
            if (pair) {
                p.mt_pairs = (m_tiles + 1) / 2;
                p.n_work = G * p.mt_pairs;
                grid = std::min(ctx->sm_count & ~1, 2 * p.n_work);
            }
            p.Y = ctx->dY; p.O = m.dims[m.L]; p.partials = s->partials;
            const bool last = (l == s->nl - 1);
            int mode = TC_MODE_HIDDEN;
            if (last && s->fused_out) {
                mode = TC_MODE_FUSED;
                p.act_out = m.act[m.L - 1]; p.Wout = s->Wout; p.bout = s->bout;
            } else if (last) {
                mode = TC_MODE_FINAL;
            }
            if (last) ssi_kt_begin(ctx);
            if (pair) {
                cudaLaunchConfig_t cfg{};
                cfg.gridDim = dim3(grid); cfg.blockDim = dim3(TC_THREADS);
                cfg.dynamicSmemBytes = tc_smem_total(mode); cfg.stream = ctx->stream;
                cudaLaunchAttribute attr{};
                attr.id = cudaLaunchAttributeClusterDimension;
                attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
                cfg.attrs = &attr; cfg.numAttrs = 1;
                void* args[] = {&s->tmAh[l], &s->tmAl[l], &s->tmBh2[l], &s->tmBl2[l], &s->tmSh[l], &s->tmSl[l], &p};
                SSI_CUDA(ctx, cudaLaunchKernelExC(&cfg, (const void*)tc_kernel(mode, p.act, s->prec, true), args));
            } else {
                tc_kernel(mode, p.act, s->prec)<<<grid, TC_THREADS, tc_smem_total(mode), ctx->stream>>>(s->tmAh[l], s->tmAl[l], s->tmBh[l], s->tmBl[l],
                                                                                                       s->tmSh[l], s->tmSl[l], p);
            }
            SSI_LAUNCH_CHECK(ctx);
            if (last) ssi_kt_end(ctx);
        }
        SSI_TRY(ssi_reduce_partials(ctx, s->partials, G, parts, d_sse + b0));
    }
    return SSI_OK;
}
