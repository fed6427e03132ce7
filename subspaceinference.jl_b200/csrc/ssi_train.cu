// ssi_train.cu — the step BEFORE the path (SURVEY 8(f)-3): the mini-batch training step inside subspace_construction,
//
//     gs = gradient(ps) do  training_loss = cost(d...)  end;  Flux.update!(opt, ps, gs)      src/subspace_construction.jl:39-43
//
// for a Dense chain with cost = Flux.Losses.mse(m(x), y) and opt = Descent(eta) or ADAM(eta, (b1, b2)) (README.md:86-88,
// docs/src/nn_example.md), kept on the device so that every snapshot reaches the SWA recurrence (k_swa_push) without a
// host round trip.  The weights live in the reference's flat layout [vec(W_1); b_1; ...] (src/libs.jl:19-22).
//
//     H_l = act_l(W_l H_{l-1} + b_l)                              forward over the mini-batch, activations kept
//     loss = mean((pred - y)^2)                                    over the O x nb outputs
//     delta_L = 2/(O nb) (pred - y) act_L'(pred)
//     gW_l = delta_l H_{l-1}',  gb_l = rowsum(delta_l),  delta_{l-1} = (W_l' delta_l) * act_{l-1}'(H_{l-1})
//     Descent: W -= eta g          ADAM (Flux 0.11): m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;
//                                                    W -= eta m/(1-b1^t) / (sqrt(v/(1-b2^t)) + 1e-8)
//
// The forward and backward passes are the gradient path's ssi_reverse_pass (ssi_gemm.cu) with one sample; the optimiser
// update is one element-wise pass evaluated in FP64 like Julia's broadcast with Float64 hyper-parameters.
// Correctness-first: this is a "next" row, measured but not tuned.
#include "ssi_common.cuh"
#include "ssi_gemm.cuh"

#include <algorithm>
#include <cmath>

struct ssi_train_state {
    int kind = 0;                 // 0 Descent, 1 ADAM
    double eta = 0.1, b1 = 0.9, b2 = 0.999;
    double bp1 = 0.9, bp2 = 0.999;   // running powers beta^t (Flux keeps them per array; all arrays step together)
    long long steps = 0;
    float* W = nullptr;           // n
    float* G = nullptr;           // n
    float* m = nullptr;           // n (ADAM)
    float* v = nullptr;           // n (ADAM)
    double* loss = nullptr;       // 1
    ssi_buf_t bAct, bDelta, bXb, bYb, bIdx, bPart;
};

void ssi_train_destroy(ssi_ctx* ctx) {
    ssi_train_state* t = ctx->train;
    if (!t) return;
    cudaFree(t->W); cudaFree(t->G); cudaFree(t->m); cudaFree(t->v); cudaFree(t->loss);
    ssi_buf_t* bufs[] = {&t->bAct, &t->bDelta, &t->bXb, &t->bYb, &t->bIdx, &t->bPart};
    for (ssi_buf_t* b : bufs) { cudaFree(b->p); b->p = nullptr; b->cap = 0; }
    delete t;
    ctx->train = nullptr;
}

// mini-batch columns picked by index (a shuffled DataLoader): Xb(:, j) = X(:, idx[j]), Yb likewise
__global__ void __launch_bounds__(256)
k_train_gather(const float* __restrict__ X, const float* __restrict__ Y, const long long* __restrict__ idx, int in0, int O,
               long long nb, float* __restrict__ Xb, float* __restrict__ Yb) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long per = in0 + O;
    if (e >= nb * per) return;
    const long long j = e / per;
    const int r = (int)(e % per);
    const long long src = idx[j];
    if (r < in0) Xb[j * in0 + r] = X[src * in0 + r];
    else Yb[j * O + (r - in0)] = Y[src * O + (r - in0)];
}

// loss = sum(partials) / count, fixed order
__global__ void k_train_loss(const double* __restrict__ partials, int n_chunks, double inv_count, double* __restrict__ loss) {
    if (blockIdx.x || threadIdx.x) return;
    double s = 0.0;
    for (int c = 0; c < n_chunks; ++c) s += partials[c];
    *loss = s * inv_count;
}

__global__ void __launch_bounds__(256)
k_train_update(float* __restrict__ W, const float* __restrict__ G, float* __restrict__ m, float* __restrict__ v, long long n,
               int kind, double eta, double b1, double b2, double bp1, double bp2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double g = (double)G[i];
    if (kind == 0) {
        W[i] = (float)((double)W[i] - eta * g);
        return;
    }
    const float mt = (float)(b1 * (double)m[i] + (1.0 - b1) * g);
    const float vt = (float)(b2 * (double)v[i] + (1.0 - b2) * g * g);
    m[i] = mt;
    v[i] = vt;
    const float d = (float)((double)mt / (1.0 - bp1) / (sqrt((double)vt / (1.0 - bp2)) + 1e-8) * eta);
    W[i] = W[i] - d;
}

int ssi_train_begin_impl(ssi_ctx* ctx, const float* W0, int kind, double eta, double b1, double b2) {
    if (!ctx->has_model || !ctx->has_data)
        return ssi_fail(ctx, SSI_ERR_STATE, "ssi_set_model and ssi_set_data must be called before ssi_train_begin");
    if (kind != 0 && kind != 1) return ssi_fail(ctx, SSI_ERR_ARG, "optimiser must be 0 (Descent) or 1 (ADAM)");
    if (!(eta > 0) || !(b1 >= 0 && b1 < 1) || !(b2 >= 0 && b2 < 1)) return ssi_fail(ctx, SSI_ERR_ARG, "eta > 0 and beta in [0, 1) required");
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ssi_train_destroy(ctx);
    ssi_train_state* t = ctx->train = new ssi_train_state();
    const size_t n = (size_t)ctx->model.n;
    t->kind = kind; t->eta = eta; t->b1 = b1; t->b2 = b2; t->bp1 = b1; t->bp2 = b2;
    SSI_CUDA(ctx, cudaMalloc(&t->W, sizeof(float) * n));
    SSI_CUDA(ctx, cudaMalloc(&t->G, sizeof(float) * n));
    SSI_CUDA(ctx, cudaMalloc(&t->loss, sizeof(double)));
    if (kind == 1) {
        SSI_CUDA(ctx, cudaMalloc(&t->m, sizeof(float) * n));
        SSI_CUDA(ctx, cudaMalloc(&t->v, sizeof(float) * n));
        SSI_CUDA(ctx, cudaMemsetAsync(t->m, 0, sizeof(float) * n, ctx->stream));
        SSI_CUDA(ctx, cudaMemsetAsync(t->v, 0, sizeof(float) * n, ctx->stream));
    }
    SSI_CUDA(ctx, cudaMemcpyAsync(t->W, W0, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
    SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSI_OK;
}

int ssi_train_step_impl(ssi_ctx* ctx, const int64_t* idx, int64_t j0, int64_t nb, double* loss_out) {
    ssi_train_state* t = ctx->train;
    if (!t) return ssi_fail(ctx, SSI_ERR_STATE, "ssi_train_begin has not been called");
    if (!ctx->has_data) return ssi_fail(ctx, SSI_ERR_STATE, "the data set was replaced: call ssi_train_begin again");
    const ssi_model_t& m = ctx->model;
    const int L = m.L, in0 = m.dims[0], O = m.dims[L];
    const int64_t N = ctx->N;
    if (nb < 1 || nb >= (1ll << 31)) return ssi_fail(ctx, SSI_ERR_ARG, "mini-batch size must be in [1, 2^31)");
    if (!idx && (j0 < 0 || j0 + nb > N)) return ssi_fail(ctx, SSI_ERR_ARG, "mini-batch [%lld, %lld) outside the %lld datapoints", (long long)j0, (long long)(j0 + nb), (long long)N);

    const float* Xb = ctx->dX + j0 * in0;
    const float* Yb = ctx->dY + j0 * O;
    if (idx) {
        for (int64_t j = 0; j < nb; ++j)
            if (idx[j] < 0 || idx[j] >= N) return ssi_fail(ctx, SSI_ERR_ARG, "mini-batch index %lld outside the %lld datapoints", (long long)idx[j], (long long)N);
        SSI_TRY(ssi_reserve(ctx, t->bIdx, sizeof(long long) * (size_t)nb));
        SSI_TRY(ssi_reserve(ctx, t->bXb, sizeof(float) * (size_t)in0 * nb));
        SSI_TRY(ssi_reserve(ctx, t->bYb, sizeof(float) * (size_t)O * nb));
        SSI_CUDA(ctx, cudaMemcpyAsync(t->bIdx.p, idx, sizeof(long long) * (size_t)nb, cudaMemcpyHostToDevice, ctx->stream));
        const long long tot = nb * (long long)(in0 + O);
        k_train_gather<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(ctx->dX, ctx->dY, (const long long*)t->bIdx.p, in0, O, nb,
                                                                           (float*)t->bXb.p, (float*)t->bYb.p);
        SSI_LAUNCH_CHECK(ctx);
        SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));     // idx is the caller's buffer
        Xb = (const float*)t->bXb.p;
        Yb = (const float*)t->bYb.p;
    }

    int maxw = 0;
    const long long act_elems = ssi_act_offsets(m, nb, nullptr, &maxw);
    const int n_chunks = (int)((nb + 255) / 256);
    SSI_TRY(ssi_reserve(ctx, t->bAct, sizeof(float) * (size_t)act_elems));
    SSI_TRY(ssi_reserve(ctx, t->bDelta, sizeof(float) * (size_t)2 * maxw * nb));
    SSI_TRY(ssi_reserve(ctx, t->bPart, sizeof(double) * (size_t)n_chunks));
    float* D[2] = {(float*)t->bDelta.p, (float*)t->bDelta.p + (size_t)maxw * nb};
    // delta_L = 2/(O nb) (pred - y) act'(pred): the reverse pass computes -(pred - y) * coef * act'
    const double count = (double)O * (double)nb;
    SSI_TRY(ssi_reverse_pass(ctx, 1, nb, t->W, t->G, m.n, Xb, Yb, (float*)t->bAct.p, act_elems, D, (long long)maxw * nb,
                             (float)(-2.0 / count), (double*)t->bPart.p));
    k_train_loss<<<1, 32, 0, ctx->stream>>>((const double*)t->bPart.p, n_chunks, 1.0 / count, t->loss);
    SSI_LAUNCH_CHECK(ctx);
    k_train_update<<<(unsigned)((m.n + 255) / 256), 256, 0, ctx->stream>>>(t->W, t->G, t->m, t->v, m.n, t->kind, t->eta, t->b1, t->b2,
                                                                       t->bp1, t->bp2);
    SSI_LAUNCH_CHECK(ctx);
    t->bp1 *= t->b1;
    t->bp2 *= t->b2;
    t->steps++;
    ctx->stats.last_flops = 3.0 * (double)nb * m.flops_per_point;      // forward + two backward contractions per layer
    if (loss_out) {
        SSI_CUDA(ctx, cudaMemcpyAsync(loss_out, t->loss, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SSI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SSI_OK;
}

const float* ssi_train_weights_device(ssi_ctx* ctx) { return ctx->train ? ctx->train->W : nullptr; }
