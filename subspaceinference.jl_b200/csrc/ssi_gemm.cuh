// ssi_gemm.cuh -- the strided FP32 GEMM (ssi_gemm.cu, ssi_gemm_tc.cu) and the passes over a Dense chain built on it.
#pragma once
#include "ssi_common.cuh"

struct gemm_t {
    // C(o, j) = sum_k A(o, k) B(k, j) for batch b = blockIdx.z; all strides in elements
    const float* A; long long a_so, a_sk, a_sb;
    const float* B; long long b_sk, b_sj, b_sb;
    float* C;       long long c_so, c_sj, c_sb;
    int O, J;
    long long K;            // contraction length (per batch when split > 0: the last batch may be shorter)
    long long split;        // > 0: batch b covers k in [b*split, min(K, (b+1)*split))
    int epi;                // 0 plain, 1 bias + activation, 2 multiply by act'(Hprev(o, j))
    int act;
    const float* bias; long long bias_sb;
    const float* Hprev; long long h_sb;       // indexed like C
};

#define GT_T 64           // k_gemm_simt's tile edge along o and j

// a_kfast: A is contiguous along k (else along o); b_jfast: B is contiguous along j (else along k); not both.
// Skinny, tensor-core or SIMT kernel, whichever fits the shape.
int ssi_launch_gemm(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast);
// Always the exact FP32 SIMT kernel.  With partials (A o-fast, B k-fast, epi 1): C is not stored; instead
// partials[b][tile] = sum over the 64x64 tile of (C(o, j) - Y(o, j))^2 in FP64, Y indexed like C, tile = to * tiles_j + tj.
int ssi_launch_gemm_simt(ssi_ctx* ctx, const gemm_t& g, int batches, bool a_kfast, bool b_jfast, const float* Y = nullptr,
                         double* partials = nullptr);

// Dense layer l as a GEMM: C = act_l(W_l H + b_l), W_l (out x in, o fast) and b_l read from the flat Flux.destructure
// vector W.  H is in x J with datapoints in_l apart; C(o, j) is at C + o + j * c_sj.  Sample b's W, H and C are
// w_sb, h_sb and c_sb further on.
gemm_t ssi_dense_gemm(const ssi_model_t& m, int l, const float* W, long long w_sb, const float* H, long long h_sb, float* C,
                      long long c_sj, long long c_sb, int J);
// The activations a reverse pass over J datapoints keeps: H_l (dims[l] x J) at h_off[l] (if h_off), l = 1..L.  Returns
// their total; *maxw is the widest layer, which sizes each of the two delta buffers (maxw x J).
long long ssi_act_offsets(const ssi_model_t& m, long long J, long long* h_off, int* maxw);
// One reverse pass of ctx's model for g samples over J datapoints X (in0 x J), Y (O x J): the forward pass with every
// activation kept in H, delta_L = -(pred - y) * coef * act_L'(pred) with the squared-error partials [g][ceil(J / 256)],
// then per layer from the last the weight gradient, the bias row-sum and the back-propagated delta.  The gradient gW has
// W's flat layout.  Sample b's W and gW are w_sb apart, its activations h_sb, its deltas d_sb (in D[0] and D[1]).
int ssi_reverse_pass(ssi_ctx* ctx, int g, long long J, const float* W, float* gW, long long w_sb, const float* X, const float* Y,
                     float* H, long long h_sb, float* const D[2], long long d_sb, float coef, double* partials);
