// ssi_basis_mma.cu — the BASIS path on the tensor cores: Chain(Dense(in, H, act), Dense(H, 1)) with H <= 64 and M + 1 <= 32,
// many samples (SURVEY H3, "stack samples along the MMA M dimension").  BASELINE configs[1]: 13-50-1 with 4096 chains.
//
// The first layer is affine in z (see ssi_basis.cu): with z augmented by a constant 1,
//     pre[s, e] = sum_{m <= M} zaug[s, m] * basesT[e, m],     e = (datapoint i, hidden unit j) = i*Hp + j,   K = 16 or 32,
// is a GEMM whose M dimension is the SAMPLES.  A CTA owns 256 samples (two 128-row A operands resident in shared memory
// for the whole kernel) and walks tiles of 2 or 4 datapoints (NT = 2 Hp or 4 x 32 activations <= 128): the basis tile is
// fetched once by TMA and multiplied with both sample groups (three-way BF16 split of both operands, six products, FP32
// accumulate in TMEM, two 128-column accumulators per group so that the MMAs of tile t+1 run under the epilogue of tile t).
// The epilogue never stores the hidden layer: lane = sample, so each thread keeps ITS sample's second-layer weights in
// registers, applies the activation to its TMEM columns, folds them into Hp-long dot products (the output layer), subtracts y
// and accumulates the squared error in an error-free two-float sum.  One FP64 partial per (sample, part) leaves the kernel.
//
// Roles: warp 0 TMA producer, warps 1 and 10 MMA issuers (one per sample group; warp 1 also allocates TMEM), warps 2-9 epilogue
// (warp w: TMEM lane quarter w % 4 of sample group (w - 2) / 4).  Bound: the epilogue (register-file bandwidth of the dot products with per-sample weights).
//
// PACKED operands (M + 1 <= 8): K = 16 leaves most of the contraction index empty (6 of 16 for M = 5), so the six
// (z part, basis part) products are laid side by side ALONG K instead of being issued as six MMAs: column c = term*(M+1) + m
// of the packed operands holds (z_part[term][m], basis_part[term][m]), 6 (M+1) <= 48 columns = at most three K=16 slabs.
// Same bytes in shared memory as the three (hi, mid, lo) tiles, half the MMAs.
#include "ssi_common.cuh"
#include "ssi_ptx.cuh"

#include <algorithm>
#include <cmath>

typedef __nv_bfloat16 bf16;

#define BM_THREADS 352
// Activations per tile: NT = (datapoints per tile) x HP <= 128 (4 accumulators of 128 TMEM columns: 2 sample groups x 2 buffers).
// HP, the hidden width rounded up, is one of 32, 40, 48, 56, 64: the epilogue walks a datapoint's columns in TMEM chunks of
// 32, 16 and 8 columns, so H = 50 costs 56 columns of work, not 64.
#define BM_STAGES 4
__host__ __device__ constexpr int bm_dpt(int hp) { return hp == 32 ? 4 : 2; }                      // datapoints per tile
__host__ __device__ constexpr int bm_nt(int hp) { return bm_dpt(hp) * hp; }
__host__ __device__ constexpr int bm_nchunk(int hp) { return hp == 32 ? 1 : (hp == 56 ? 3 : 2); }   // TMEM chunks per datapoint
__host__ __device__ constexpr int bm_chunk_size(int hp, int i) { return i == 0 ? 32 : (hp == 64 ? 32 : (hp == 40 ? 8 : (i == 1 ? 16 : 8))); }
__host__ __device__ constexpr int bm_chunk_off(int hp, int i) { return i == 0 ? 0 : (i == 1 ? 32 : 48); }
#define BM_MAXHP 64

struct bm_params {
    int n_tiles;            // ceil(N * Hp / 256)
    int Hp, H, N, S;        // padded / true hidden width, datapoints, samples of this launch
    int act_out;
    int parts;              // partial sums per sample (tile t belongs to part t % parts); a CTA walks parts blockIdx.x, +gridDim.x, ..
    int ns;                 // operand slabs per tile: 3 (hi, mid, lo) or, packed, ceil(6 (M+1) / 16)
    const float* W2;        // [S][Hp]: second-layer weights of every sample (zero beyond H)
    const float* B2;        // [S]: second-layer bias of every sample
    const float* Y;         // N targets
    double* partials;       // [S][parts]
};

template <int ACT>
__device__ __forceinline__ float bm_act(float v) {
    if (ACT == SSI_ACT_RELU) return fmaxf(v, 0.0f);
    if (ACT == SSI_ACT_TANH) return tanhf(v);
    if (ACT == SSI_ACT_SIGMOID) return 1.0f / (1.0f + expf(-v));
    return v;
}

// issue the TMEM load of SZ consecutive columns of this thread's lane
template <int SZ>
__device__ __forceinline__ void bm_tmem_ld(uint32_t taddr, uint32_t* v) {
    if (SZ == 32) tmem_ld32(taddr, v);
    else if (SZ == 16) tmem_ld16(taddr, v);
    else tmem_ld8(taddr, v);
}

// fold SZ hidden units (TMEM columns in v, second-layer weights in wh) into the partial dot products.
// ReLU clamps every pair with FMNMX (ALU pipe), then one FFMA2.  Writing every pair as (w/2) x + (w/2) |x| instead (FFMA2 +
// two FFMA with the |.| operand modifier: FMA pipes only) measured 373 us against 333 us on the UCI config, and a mix of the
// two (one pair in four as |x|, which would balance the ALU and FMA pipes on paper) 377 us: what counts is register-file
// traffic, six operand reads per hidden unit for the |x| form against four.
template <int ACT, int NL, int SZ>
__device__ __forceinline__ void bm_fold(const uint32_t* v, const float2* wh, float2* lin) {
#pragma unroll
    for (int j = 0; j < SZ; j += 2) {
        float2 x = make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1]));
        const float2 w2 = wh[j >> 1];
        x.x = bm_act<ACT>(x.x);
        x.y = bm_act<ACT>(x.y);
        lin[(j >> 1) & (NL - 1)] = __ffma2_rn(x, w2, lin[(j >> 1) & (NL - 1)]);
    }
}

// KB = 16 (SWIZZLE_32B rows of 32 bytes) or 32 (SWIZZLE_64B rows of 64 bytes)
template <int KB>
__device__ __forceinline__ uint64_t bm_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8 * KB * 2) >> 4) << 32;           // stride between 8-row groups
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(KB == 16 ? 6 : 4) << 61;            // SWIZZLE_32B : SWIZZLE_64B
    return d;
}

template <int ACT, int KB, int HP, bool PACKED, bool OUT_ID>
__global__ void __launch_bounds__(BM_THREADS, 1)
k_b1_mma(const __grid_constant__ CUtensorMap tmZ, const __grid_constant__ CUtensorMap tmT, const bm_params p) {
    constexpr uint32_t ROW = KB * 2;                       // bytes per operand row
    constexpr int BM_N = bm_nt(HP);
    constexpr uint32_t B_TILE = BM_N * ROW;                // one of (hi, mid, lo)
    constexpr uint32_t STAGE = 3 * B_TILE;
    constexpr uint32_t Z_TILE = 128 * ROW;                 // one sample group, one of (hi, mid, lo)
    constexpr uint32_t OFF_Z = BM_STAGES * STAGE;          // [group][part]
    constexpr uint32_t OFF_BAR = OFF_Z + 6 * Z_TILE;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + OFF_BAR);     // full[4] empty[4] tfull[2][2] tempty[2][2] zfull
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 20);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_u32(s_bar), bar_empty = bar_full + 8 * BM_STAGES;
    const uint32_t bar_tfull = bar_empty + 8 * BM_STAGES, bar_tempty = bar_tfull + 32, bar_z = bar_tempty + 32;
    const int block = blockIdx.y;                          // block of 256 samples

    if (threadIdx.x == 0) {
        if (smem_base & 1023u) { printf("ssi_basis_mma: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
        for (int s = 0; s < BM_STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 2); }
        for (int b = 0; b < 4; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 128); }
        mbar_init(bar_z, 1);
        fence_barrier_init();
        tma_prefetch_desc(&tmZ); tma_prefetch_desc(&tmT);
    }
    if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        if (lane == 0) {
            const int ns = PACKED ? p.ns : 3;
            mbar_expect_tx(bar_z, 2 * ns * Z_TILE);
            for (int g = 0; g < 2; ++g)
                for (int part = 0; part < ns; ++part)
                    tma_load_3d_hint(smem_base + OFF_Z + (3 * g + part) * Z_TILE, &tmZ, bar_z, 0, (block * 2 + g) * 128, part, TC_EVICT_LAST);
            int stage = 0;
            uint32_t phase = 0;
            for (int pp = blockIdx.x; pp < p.parts; pp += gridDim.x)
                for (int t = pp; t < p.n_tiles; t += p.parts) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    const uint32_t full = bar_full + 8 * stage;
                    const uint32_t sB = smem_base + stage * STAGE;
                    mbar_expect_tx(full, ns * B_TILE);
                    for (int part = 0; part < ns; ++part)     // every block of samples re-reads the bases: keep them in L2
                        tma_load_3d_hint(sB + part * B_TILE, &tmT, full, 0, t * BM_N, part, TC_EVICT_LAST);
                    if (++stage == BM_STAGES) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == 1 || warp == 10) {
        // one MMA issuer per sample group (warp 1: group 0, warp 10: group 1).  The tiles are tiny (three to twelve MMAs), so a
        // single issuing thread that serves both groups is bound by its own chain of mbarrier waits, not by the tensor pipe.
        if (lane == 0) {
            const int g = warp == 1 ? 0 : 1;
            const uint32_t idesc = umma_idesc_bf16(BM_N);
            mbar_wait(bar_z, 0);
            tc_fence_after();
            int stage = 0;
            uint32_t phase = 0, it = 0;
            for (int pp = blockIdx.x; pp < p.parts; pp += gridDim.x)
                for (int t = pp; t < p.n_tiles; t += p.parts, ++it) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t sB = smem_base + stage * STAGE;
                    const uint64_t bh = bm_desc<KB>(sB), bm = bm_desc<KB>(sB + B_TILE), bl = bm_desc<KB>(sB + 2 * B_TILE);
                    const uint32_t ab = it & 1, aphase = (it >> 1) & 1;
                    {
                        mbar_wait(bar_tempty + 8 * (2 * g + ab), aphase ^ 1);   // the epilogue two tiles back has drained this accumulator
                        tc_fence_after();
                        const uint32_t d_tmem = tmem_base + (2 * g + ab) * 128;
                        const uint64_t zh = bm_desc<KB>(smem_base + OFF_Z + (3 * g) * Z_TILE);
                        const uint64_t zm = bm_desc<KB>(smem_base + OFF_Z + (3 * g + 1) * Z_TILE);
                        const uint64_t zl = bm_desc<KB>(smem_base + OFF_Z + (3 * g + 2) * Z_TILE);
                        if (PACKED) {
                            // the six products sit side by side along K (see the header): one MMA per 16-column slab
                            umma_bf16(d_tmem, zh, bh, idesc, 0);
                            if (p.ns > 1) umma_bf16(d_tmem, zm, bm, idesc, 1);
                            if (p.ns > 2) umma_bf16(d_tmem, zl, bl, idesc, 1);
                        } else {
                            // every operand is split three ways, x = hi + mid + lo (24 bits), and the six products down to 2^-16 of
                            // hi*hi are kept (smallest first): this layer's result is squared and summed straight into lp, with
                            // no wider layer behind it
#pragma unroll
                            for (int k = 0; k < KB / 16; ++k) {
                                const uint64_t ko = (uint64_t)(k * 32 >> 4);
                                umma_bf16(d_tmem, zm + ko, bm + ko, idesc, k != 0);
                                umma_bf16(d_tmem, zl + ko, bh + ko, idesc, 1);
                                umma_bf16(d_tmem, zh + ko, bl + ko, idesc, 1);
                                umma_bf16(d_tmem, zm + ko, bh + ko, idesc, 1);
                                umma_bf16(d_tmem, zh + ko, bm + ko, idesc, 1);
                                umma_bf16(d_tmem, zh + ko, bh + ko, idesc, 1);
                            }
                        }
                        umma_commit(bar_tfull + 8 * (2 * g + ab));
                    }
                    umma_commit(bar_empty + 8 * stage);
                    if (++stage == BM_STAGES) { stage = 0; phase ^= 1; }
                }
        }
    } else {
        const int q = warp & 3, g = (warp - 2) >> 2;      // warps 2-9; a warp may only touch TMEM lanes [32 (warp % 4), +32)
        const long long srow = (long long)block * 256 + g * 128 + q * 32 + lane;      // this thread's sample
        const bool valid = srow < p.S;
        // second-layer weights and bias of this sample, in registers for the whole kernel (zero for padded hidden units)
        constexpr int DPT = BM_N / HP;                     // datapoints per tile
        float2 wh[HP / 2];
        {
            const float4* wrow = reinterpret_cast<const float4*>(p.W2 + srow * HP);
#pragma unroll
            for (int j = 0; j < HP / 4; ++j) {
                const float4 w4 = valid ? __ldg(wrow + j) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                wh[2 * j] = make_float2(w4.x, w4.y);
                wh[2 * j + 1] = make_float2(w4.z, w4.w);
            }
        }
        const float b2 = valid ? __ldg(p.B2 + srow) : 0.0f;
        const int N = p.N, parts = p.parts, n_tiles = p.n_tiles, gx = (int)gridDim.x;
        const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + (2 * g) * 128;
        const uint32_t bar_f = bar_tfull + 16 * g, bar_e = bar_tempty + 16 * g;

        // Software pipeline over the tile's TMEM chunks (per datapoint 32 [+16] [+8] or 32+32 columns, consecutive chunks in
        // different registers): the load of the next chunk is in flight while this one is folded into partial dot products;
        // the accumulator is handed back to the MMA warp as soon as its last chunk sits in registers.  (Prefetching the next
        // tile's first chunk as well costs registers the kernel does not have: 168 is the ceiling with 10 warps, three of
        // them on one scheduler, and the spills made it 25 % slower.)
        int pp = blockIdx.x, t = pp;                        // parts >= gridDim.x and n_tiles >= parts: the first tile exists
        uint32_t it = 0;
        float s_hi = 0.0f, s_lo = 0.0f;                     // squared errors of the current part, two-float (error-free) sum
        constexpr int NC = bm_nchunk(HP);
        uint32_t v[HP == 32 ? 64 : (HP > 32 ? HP : 32)];    // HP = 32: two 32-column buffers alternate between datapoints
        while (true) {
            int tn = t + parts, ppn = pp;
            if (tn >= n_tiles) { ppn = pp + gx; tn = ppn; }
            const bool more = ppn < parts;
            const uint32_t ab = it & 1;
            const int i_base = t * DPT;
            float yv[DPT];                                  // targets of this tile's datapoints (needed one datapoint from now)
#pragma unroll
            for (int d = 0; d < DPT; ++d) yv[d] = (i_base + d < N) ? __ldg(p.Y + i_base + d) : 0.0f;
            float sse_t = 0.0f;
            constexpr int NL = 4;                           // independent FFMA2 chains
            float2 lin[NL];
#pragma unroll
            for (int i = 0; i < NL; ++i) lin[i] = make_float2(0.0f, 0.0f);
            mbar_wait(bar_f + 8 * ab, (it >> 1) & 1);
            tc_fence_after();
            const uint32_t ta = taddr0 + ab * 128;
            bm_tmem_ld<32>(ta, v);
#pragma unroll
            for (int d = 0; d < DPT; ++d) {
#pragma unroll
                for (int i = 0; i < NC; ++i) {
                            const int sz = bm_chunk_size(HP, i), off = bm_chunk_off(HP, i);
                    const int boff = HP == 32 ? (d & 1) * 32 : off;              // registers of this chunk
                    // next chunk: (d, i + 1) or (d + 1, 0)
                    const bool last = (d == DPT - 1) && (i == NC - 1);
                    const int dn = (i == NC - 1) ? d + 1 : d, in_ = (i == NC - 1) ? 0 : i + 1;
                    const int szn = bm_chunk_size(HP, in_), offn = bm_chunk_off(HP, in_);
                    const int boffn = HP == 32 ? (dn & 1) * 32 : offn;
                    tmem_ld_wait();
                    if (!last) {
                        const uint32_t tan = ta + dn * HP + offn;
                        if (szn == 32) bm_tmem_ld<32>(tan, v + boffn);
                        else if (szn == 16) bm_tmem_ld<16>(tan, v + boffn);
                        else bm_tmem_ld<8>(tan, v + boffn);
                    } else {
                        tc_fence_before();
                        mbar_arrive(bar_e + 8 * ab);         // the whole accumulator is in registers
                    }
                    if (sz == 32) bm_fold<ACT, NL, 32>(v + boff, wh + (off >> 1), lin);
                    else if (sz == 16) bm_fold<ACT, NL, 16>(v + boff, wh + (off >> 1), lin);
                    else bm_fold<ACT, NL, 8>(v + boff, wh + (off >> 1), lin);
                    if (i == NC - 1) {                       // a datapoint is complete
                        float pre = (lin[0].x + lin[0].y) + (lin[1].x + lin[1].y);
                        pre += (lin[2].x + lin[2].y) + (lin[3].x + lin[3].y);
                        pre += b2;
                        if (!OUT_ID) pre = ssi_act(pre, p.act_out);
                        const float df = (i_base + d < N) ? pre - yv[d] : 0.0f;
                        sse_t = fmaf(df, df, sse_t);
#pragma unroll
                        for (int k = 0; k < NL; ++k) lin[k] = make_float2(0.0f, 0.0f);
                    }
                }
            }
            {   // (s_hi, s_lo) += sse_t without rounding error (TwoSum); no FP64 in the loop (a DADD per tile throttled the FP64 pipe)
                const float s = s_hi + sse_t;
                const float bb = s - s_hi;
                s_lo += (s_hi - (s - bb)) + (sse_t - bb);
                s_hi = s;
            }
            if (ppn != pp) {
                if (valid) p.partials[srow * parts + pp] = (double)s_hi + (double)s_lo;
                s_hi = s_lo = 0.0f;
            }
            if (!more) break;
            pp = ppn;
            t = tn;
            ++it;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

__device__ __forceinline__ void bm_split3(float v, bf16& hi, bf16& mid, bf16& lo) {
    hi = __float2bfloat16_rn(v);
    const float r1 = v - __bfloat162float(hi);
    mid = __float2bfloat16_rn(r1);
    lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
}

// which of (hi, mid, lo) = (0, 1, 2) the packed operands take for product `term`, smallest product first:
// (z, basis) = (mid,mid) (lo,hi) (hi,lo) (mid,hi) (hi,mid) (hi,hi)
__device__ __forceinline__ int bm_term_zpart(int term) { return term == 0 || term == 3 ? 1 : (term == 1 ? 2 : 0); }
__device__ __forceinline__ int bm_term_bpart(int term) { return term == 0 || term == 4 ? 1 : (term == 2 ? 2 : 0); }
__device__ __forceinline__ bf16 bm_part(float v, int part) {
    bf16 hi, mid, lo;
    bm_split3(v, hi, mid, lo);
    return part == 0 ? hi : (part == 1 ? mid : lo);
}

// zaug[slab][s][k]: z[m, s] (m < M), 1 (m == M), 0 (padding, and rows s >= S up to a multiple of 256).
// classic: slab = part of the three-way split, k = m;  packed (KB = 16): column c = slab*16 + k = term*(M+1) + m
__device__ __forceinline__ void bm_pack_zaug_elem(const float* __restrict__ Z, int M, long long S, long long S_pad, int KB, int packed_ns,
                                                  bf16* __restrict__ out, long long t) {
    if (t >= S_pad * KB) return;
    const long long s = t / KB;
    const int k = (int)(t % KB);
    if (packed_ns) {
        for (int slab = 0; slab < packed_ns; ++slab) {
            const int c = slab * 16 + k, term = c / (M + 1), m = c % (M + 1);
            const float v = (s < S && term < 6) ? (m < M ? Z[m + s * M] : 1.0f) : 0.0f;
            out[(long long)slab * S_pad * KB + t] = bm_part(v, bm_term_zpart(term));
        }
        return;
    }
    const float v = s < S ? (k < M ? Z[k + s * M] : (k == M ? 1.0f : 0.0f)) : 0.0f;
    bf16 hi, mid, lo;
    bm_split3(v, hi, mid, lo);
    out[t] = hi;
    out[S_pad * KB + t] = mid;
    out[2 * S_pad * KB + t] = lo;
}

// basesT[slab][i*Hp + j][k] (K-major, KB BF16 per activation)  <-  bases[m][i][j] FP32 (ld = H), zero padding; slabs as above
__global__ void __launch_bounds__(256)
k_bm_bases_kmajor(const float* __restrict__ bases, long long N, int H, int Hp, int M1, int KB, int packed_ns, bf16* __restrict__ out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = N * Hp * KB;
    if (t >= total) return;
    const int k = (int)(t % KB);
    const long long e = t / KB;
    const int j = (int)(e % Hp);
    const long long i = e / Hp;
    if (packed_ns) {
        for (int slab = 0; slab < packed_ns; ++slab) {
            const int c = slab * 16 + k, term = c / M1, m = c % M1;
            const float v = (term < 6 && j < H) ? bases[((long long)m * N + i) * H + j] : 0.0f;
            out[(long long)slab * total + t] = bm_part(v, bm_term_bpart(term));
        }
        return;
    }
    const float v = (k < M1 && j < H) ? bases[((long long)k * N + i) * H + j] : 0.0f;
    bf16 hi, mid, lo;
    bm_split3(v, hi, mid, lo);
    out[t] = hi;
    out[total + t] = mid;
    out[2 * total + t] = lo;
}

// W2[s][j] = (W_swa + P z_s)[second layer weight j] for j < H, 0 for H <= j < Hp;  B2[s] = its bias
__device__ __forceinline__ void bm_project_w2_elem(const float* __restrict__ PW, const float* __restrict__ Z, long long n, int M, int H,
                                                   int Hp, long long w2_off, long long b2_off, long long e,
                                                   float* __restrict__ W2, float* __restrict__ B2) {
    const long long s = e / (Hp + 1);
    const int j = (int)(e % (Hp + 1));
    float v = 0.0f;
    if (j < H || j == Hp) {
        const long long k = j < H ? w2_off + j : b2_off;
        v = PW[k + (long long)M * n];
        for (int m = 0; m < M; ++m) v = fmaf(PW[k + (long long)m * n], Z[s * M + m], v);
    }
    if (j == Hp) B2[s] = v;
    else W2[s * Hp + j] = v;
}

// the per-call preparation in ONE launch (two launches cost 8 us of a 360 us MH step): blocks [0, zblocks) pack the split z
// operand, the rest project the second-layer weights
__global__ void __launch_bounds__(256)
k_bm_prepare(const float* __restrict__ Z, int M, long long S, long long S_pad, int KB, int packed_ns, bf16* __restrict__ zaug,
             unsigned zblocks, const float* __restrict__ PW, long long n, int H, int Hp, long long w2_off, long long b2_off,
             float* __restrict__ W2, float* __restrict__ B2) {
    if (blockIdx.x < zblocks) {
        bm_pack_zaug_elem(Z, M, S, S_pad, KB, packed_ns, zaug, (long long)blockIdx.x * blockDim.x + threadIdx.x);
    } else {
        const long long e = (long long)(blockIdx.x - zblocks) * blockDim.x + threadIdx.x;
        if (e < S * (Hp + 1)) bm_project_w2_elem(PW, Z, n, M, H, Hp, w2_off, b2_off, e, W2, B2);
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct ssi_bm_state {
    bool ready = false;
    int KB = 16, Hp = 64;
    int packed_ns = 0;                       // 0: three-way split as three slabs; else packed products, this many K=16 slabs
    long long n_tiles = 0;
    bf16* T = nullptr;                       // basesT [slabs][N*Hp][KB]
    CUtensorMap tmT;
    PFN_encodeTiled encode = nullptr;
};

void ssi_bm_invalidate(ssi_ctx* ctx) {
    if (ctx->bm) ctx->bm->ready = false;
}
void ssi_bm_destroy(ssi_ctx* ctx) {
    if (!ctx->bm) return;
    cudaFree(ctx->bm->T);
    delete ctx->bm;
    ctx->bm = nullptr;
}

bool ssi_bm_supported(const ssi_ctx* ctx) {
    if (!ctx->has_model || !ctx->has_sub || !ctx->has_data) return false;
    const ssi_model_t& m = ctx->model;
    if (m.L != 2 || m.dims[2] != 1 || m.dims[1] > BM_MAXHP || ctx->M + 1 > 32) return false;
    const long long Hp = 64;
    return ctx->N * Hp < (1ll << 31) && !ctx->opt_b1_simt;
}

static int bm_make_map(ssi_ctx* ctx, CUtensorMap* map, void* base, uint64_t inner, uint64_t rows, uint32_t box_rows, int slabs) {
    cuuint64_t dims[3] = {inner, rows, (cuuint64_t)slabs};          // third dimension: the operand slabs
    cuuint64_t strides[2] = {inner * sizeof(bf16), inner * rows * sizeof(bf16)};
    cuuint32_t box[3] = {(cuuint32_t)inner, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapSwizzle swz = inner == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B;
    const CUresult r = ctx->bm->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, estr,
                                       CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return ssi_fail(ctx, SSI_ERR_CUDA, "cuTensorMapEncodeTiled (basis mma) failed with CUresult %d", (int)r);
    return SSI_OK;
}

static int bm_prepare(ssi_ctx* ctx) {
    if (!ctx->bm) ctx->bm = new ssi_bm_state();
    ssi_bm_state* s = ctx->bm;
    if (s->ready) return SSI_OK;
    if (!s->encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        SSI_CUDA(ctx, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn) return ssi_fail(ctx, SSI_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
        s->encode = (PFN_encodeTiled)fn;
    }
    const ssi_model_t& m = ctx->model;
    const int H = m.dims[1], M1 = ctx->M + 1;
    const long long N = ctx->N;
    s->KB = M1 <= 16 ? 16 : 32;
    s->Hp = H <= 32 ? 32 : (H <= 40 ? 40 : (H <= 48 ? 48 : (H <= 56 ? 56 : 64)));
    s->packed_ns = M1 <= 8 ? (6 * M1 + 15) / 16 : 0;
    const int slabs = s->packed_ns ? s->packed_ns : 3;
    const long long NW = N * s->Hp;
    const int NT = bm_nt(s->Hp);
    s->n_tiles = (NW + NT - 1) / NT;
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(s->T);
    s->T = nullptr;
    SSI_CUDA(ctx, cudaMalloc(&s->T, sizeof(bf16) * slabs * (size_t)NW * s->KB));
    // bases [m][N][H] in scratch, exact FP32 (bias parts included), then the K-major split-BF16 copy
    SSI_TRY(ssi_reserve(ctx, ctx->bH0, sizeof(float) * (size_t)M1 * N * H));
    SSI_TRY(ssi_build_first_layer_bases(ctx, (float*)ctx->bH0.p, H));
    const long long total = NW * s->KB;
    k_bm_bases_kmajor<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>((const float*)ctx->bH0.p, N, H, s->Hp, M1, s->KB, s->packed_ns, s->T);
    SSI_LAUNCH_CHECK(ctx);
    SSI_TRY(bm_make_map(ctx, &s->tmT, s->T, s->KB, (uint64_t)NW, NT, slabs));
    s->ready = true;
    return SSI_OK;
}

typedef void (*bm_kernel_t)(const CUtensorMap, const CUtensorMap, const bm_params);
template <int KB, int HP, bool PACKED, bool OUT_ID>
static bm_kernel_t bm_pick_act(int act) {
    switch (act) {
        case SSI_ACT_RELU:    return k_b1_mma<SSI_ACT_RELU, KB, HP, PACKED, OUT_ID>;
        case SSI_ACT_TANH:    return k_b1_mma<SSI_ACT_TANH, KB, HP, PACKED, OUT_ID>;
        case SSI_ACT_SIGMOID: return k_b1_mma<SSI_ACT_SIGMOID, KB, HP, PACKED, OUT_ID>;
        default:              return k_b1_mma<SSI_ACT_IDENTITY, KB, HP, PACKED, OUT_ID>;
    }
}
template <int KB, int HP, bool PACKED>
static bm_kernel_t bm_pick(int act, int act_out) {
    return act_out == SSI_ACT_IDENTITY ? bm_pick_act<KB, HP, PACKED, true>(act) : bm_pick_act<KB, HP, PACKED, false>(act);
}

int ssi_reduce_partials(ssi_ctx* ctx, const double* partials, int64_t B, int parts, double* d_out);

int ssi_bm_sse(ssi_ctx* ctx, const float* dZ, int64_t B, double* d_sse) {
    SSI_TRY(bm_prepare(ctx));
    ssi_bm_state* s = ctx->bm;
    const ssi_model_t& m = ctx->model;
    const int M = ctx->M, H = m.dims[1], KB = s->KB, Hp = s->Hp;
    const int slabs = s->packed_ns ? s->packed_ns : 3;
    const int a0 = m.act[0], a1 = m.act[1];
    bm_kernel_t kern = nullptr;
#define BM_PICK_HP(HPV)                                                                                      \
    if (Hp == HPV)                                                                                           \
        kern = s->packed_ns ? bm_pick<16, HPV, true>(a0, a1)                                                 \
                            : (KB == 16 ? bm_pick<16, HPV, false>(a0, a1) : bm_pick<32, HPV, false>(a0, a1));
    BM_PICK_HP(32) BM_PICK_HP(40) BM_PICK_HP(48) BM_PICK_HP(56) BM_PICK_HP(64)
#undef BM_PICK_HP
    if (!kern) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "basis mma path: no kernel for padded hidden width %d", Hp);
    // at least 120 KB so that exactly one CTA (which allocates all 512 TMEM columns) is resident per SM
    const size_t smem = std::max<size_t>((size_t)BM_STAGES * 3 * 128 * KB * 2 + 6 * 128 * KB * 2 + 24 * 8 + 16, 120 * 1024);
    SSI_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    const int64_t n_blocks = (B + 255) / 256;
    const int64_t S_pad = n_blocks * 256;
    // Partial sums per sample: tile t belongs to part t % parts.  `parts` depends on the dataset and the device only, never
    // on B, so a sample's summation order (hence its lp, bit for bit) is the same whatever else shares the call.
    const int parts = (int)std::min<int64_t>(s->n_tiles, ctx->sm_count);
    // A CTA walks `ppc` parts of one block of samples (its z operands and second-layer weights are loaded once): with many
    // blocks, fewer and longer CTAs amortise the pipeline fill.  Keep at least three full waves of CTAs.
    int gx = parts;
    for (int ppc = 8; ppc > 1; ppc >>= 1) {
        const int g = (parts + ppc - 1) / ppc;
        const double waves = (double)g * (double)n_blocks / ctx->sm_count;
        if (waves >= 3.0 && waves / std::ceil(waves) >= 0.9) { gx = g; break; }
    }
    // scratch: zaug [slabs][S_pad][KB] bf16, W2 [B][Hp] + B2 [B] floats, partials [B][parts] doubles
    const size_t off_w2 = (slabs * sizeof(bf16) * (size_t)S_pad * KB + 255) / 256 * 256;
    SSI_TRY(ssi_reserve(ctx, ctx->bW, off_w2 + sizeof(float) * (size_t)B * (Hp + 1)));
    SSI_TRY(ssi_reserve(ctx, ctx->bPartials, sizeof(double) * (size_t)B * parts));
    bf16* zaug = (bf16*)ctx->bW.p;
    float* W2 = (float*)((char*)ctx->bW.p + off_w2);
    float* B2 = W2 + (size_t)B * Hp;
    double* partials = (double*)ctx->bPartials.p;
    {
        const unsigned zblocks = (unsigned)((S_pad * KB + 255) / 256), wblocks = (unsigned)((B * (Hp + 1) + 255) / 256);
        k_bm_prepare<<<zblocks + wblocks, 256, 0, ctx->stream>>>(dZ, M, B, S_pad, KB, s->packed_ns, zaug, zblocks, ctx->dP, m.n, H, Hp,
                                                               m.w_off[1], m.b_off[1], W2, B2);
        SSI_LAUNCH_CHECK(ctx);
    }
    CUtensorMap tmZ;
    SSI_TRY(bm_make_map(ctx, &tmZ, zaug, KB, (uint64_t)S_pad, 128, slabs));
    bm_params p{};
    p.n_tiles = (int)s->n_tiles; p.Hp = Hp; p.H = H; p.N = (int)ctx->N; p.S = (int)B; p.act_out = m.act[1]; p.parts = parts;
    p.ns = slabs;
    p.W2 = W2; p.B2 = B2; p.Y = ctx->dY; p.partials = partials;
    if (n_blocks > 65535) return ssi_fail(ctx, SSI_ERR_UNSUPPORTED, "basis mma path: more than 16.7M samples per call");
    dim3 grid(gx, (unsigned)n_blocks);
    ssi_kt_begin(ctx);
    kern<<<grid, BM_THREADS, smem, ctx->stream>>>(tmZ, s->tmT, p);
    SSI_LAUNCH_CHECK(ctx);
    ssi_kt_end(ctx);
    return ssi_reduce_partials(ctx, partials, B, parts, d_sse);
}
