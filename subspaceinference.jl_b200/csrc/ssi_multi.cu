// ssi_multi.cu — one context driving several devices from the single calling process (SURVEY 8(b)-1, 8(e)).
//
// The reference is ONE Julia process (src/space_inference.jl:82-84): a `ccall` shim cannot bring torchrun or MPI with it.
// ssi_ctx_create_multi(devices, n) therefore returns a context that owns one ordinary context per device; every set_* call is
// replicated (W_swa, P, X, Y live on every device), and the batched host-pointer calls are sharded by sample / chain index:
// device d evaluates a contiguous range and lands its results in its slice of the caller's host arrays.  Chains keep
// their GLOBAL ids in the Philox counters, so the traces are bit-identical to a one-device run.  No collective is needed
// (the results go to host memory), hence no NCCL inside the library.  One host thread per device issues that device's
// work; the calling thread joins them.
#include "ssi_common.cuh"

#include <algorithm>
#include <thread>

namespace {

// [begin, end) of the items device d of n_dev owns; multiples of 32 so that every device keeps whole warps / groups
void shard_range(int64_t total, int n_dev, int d, int64_t& b, int64_t& e) {
    int64_t per = (total + n_dev - 1) / n_dev;
    per = (per + 31) / 32 * 32;
    b = std::min(total, (int64_t)d * per);
    e = std::min(total, (int64_t)(d + 1) * per);
}

// run fn(child, d) on every device, one thread each; the first failure's code and message become the parent's
template <typename F>
int for_each_device(ssi_ctx* ctx, F fn) {
    const int n = (int)ctx->children.size();
    std::vector<int> rc(n, SSI_OK);
    if (n == 1) {
        rc[0] = fn(ctx->children[0], 0);
    } else {
        std::vector<std::thread> th;
        th.reserve(n);
        for (int d = 0; d < n; ++d) th.emplace_back([&, d]() { rc[d] = fn(ctx->children[d], d); });
        for (auto& t : th) t.join();
    }
    for (int d = 0; d < n; ++d)
        if (rc[d] < 0) {
            ctx->err = "device " + std::to_string(ctx->children[d]->device) + ": " + ctx->children[d]->err;
            return rc[d];
        }
    return SSI_OK;
}

// run fn(child, begin, end) on every device whose shard [begin, end) of `total` items is not empty.  A device with an empty
// shard takes no part; when the call does work (`work`), that device's per-call stats are cleared, so that ssi_stats
// reports this call and not the device's previous one.
template <typename F>
int for_each_shard(ssi_ctx* ctx, int64_t total, bool work, F fn) {
    const int n_dev = (int)ctx->children.size();
    return for_each_device(ctx, [&](ssi_ctx* c, int d) {
        int64_t b, e;
        shard_range(total, n_dev, d, b, e);
        if (e > b) return fn(c, b, e);
        if (work) {
            ssi_stats_t& s = c->stats;
            s.last_ms = s.last_flops = s.last_bytes = s.last_units = 0.0;
            s.mh_accepts = s.mh_proposals = 0;
        }
        return (int)SSI_OK;
    });
}

}  // namespace

extern "C" int ssi_ctx_create(int device, ssi_ctx** out);
extern "C" int ssi_ctx_destroy(ssi_ctx* ctx);

int ssi_multi_create(const int32_t* devices, int32_t n_dev, ssi_ctx** out) {
    if (!out) return ssi_fail(nullptr, SSI_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!devices || n_dev < 1 || n_dev > 64) return ssi_fail(nullptr, SSI_ERR_ARG, "devices must name 1..64 devices");
    for (int i = 0; i < n_dev; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return ssi_fail(nullptr, SSI_ERR_ARG, "device %d is listed twice", devices[i]);
    ssi_ctx* parent = new ssi_ctx();
    for (int i = 0; i < n_dev; ++i) {
        ssi_ctx* child = nullptr;
        const int rc = ssi_ctx_create(devices[i], &child);
        if (rc != SSI_OK) {           // the message of the failed create is already in the global slot
            for (ssi_ctx* c : parent->children) ssi_ctx_destroy(c);
            parent->children.clear();
            delete parent;
            return rc;
        }
        parent->children.push_back(child);
    }
    parent->device = devices[0];
    parent->sm_count = parent->children[0]->sm_count;
    *out = parent;
    return SSI_OK;
}

int ssi_multi_destroy(ssi_ctx* ctx) {
    for (ssi_ctx* c : ctx->children) ssi_ctx_destroy(c);
    ctx->children.clear();
    delete ctx;
    return SSI_OK;
}

extern "C" {
int ssi_sync(ssi_ctx*);
int ssi_set_option(ssi_ctx*, const char*, int64_t);
int ssi_stats(const ssi_ctx*, ssi_stats_t*);
int ssi_set_model(ssi_ctx*, int, const int32_t*, const int32_t*);
int ssi_set_data(ssi_ctx*, const float*, const float*, int64_t);
int ssi_set_subspace(ssi_ctx*, const float*, const float*, int64_t, int32_t);
int ssi_logpost_batch(ssi_ctx*, const float*, int64_t, double, double, double, uint32_t, double*, double*);
int ssi_logpost_grad_batch(ssi_ctx*, const float*, int64_t, double, double, double, uint32_t, double*, double*);
int ssi_project(ssi_ctx*, const float*, int64_t, float*);
int ssi_swa_finish(ssi_ctx*, int32_t, float*, float*, double*, int32_t);
}

int ssi_multi_sync(ssi_ctx* ctx) {
    return for_each_device(ctx, [](ssi_ctx* c, int) { return ssi_sync(c); });
}

int ssi_multi_set_option(ssi_ctx* ctx, const char* key, int64_t value) {
    for (ssi_ctx* c : ctx->children) {
        const int rc = ssi_set_option(c, key, value);
        if (rc != SSI_OK) { ctx->err = c->err; return rc; }
    }
    return SSI_OK;
}

// devices work side by side: times are the maximum over devices, work and counters are summed
int ssi_multi_stats(const ssi_ctx* ctx, ssi_stats_t* out) {
    ssi_stats_t acc{};
    for (size_t d = 0; d < ctx->children.size(); ++d) {
        ssi_stats_t s{};
        ssi_stats(ctx->children[d], &s);
        if (d == 0) acc = s;
        else {
            acc.last_ms = std::max(acc.last_ms, s.last_ms);
            acc.last_flops += s.last_flops;
            acc.last_bytes += s.last_bytes;
            acc.last_units += s.last_units;
            acc.kernel_launches += s.kernel_launches;
            acc.mh_accepts += s.mh_accepts;
            acc.mh_proposals += s.mh_proposals;
            acc.dominant_ms = std::max(acc.dominant_ms, s.dominant_ms);
            acc.dominant_launches += s.dominant_launches;
            acc.gemm_tc_launches += s.gemm_tc_launches;
            acc.gemm_skinny_launches += s.gemm_skinny_launches;
        }
    }
    *out = acc;
    return SSI_OK;
}

int ssi_multi_set_model(ssi_ctx* ctx, int n_layers, const int32_t* dims, const int32_t* act) {
    const int rc = for_each_device(ctx, [&](ssi_ctx* c, int) { return ssi_set_model(c, n_layers, dims, act); });
    if (rc == SSI_OK) { ctx->model = ctx->children[0]->model; ctx->has_model = true; }
    return rc;
}

int ssi_multi_set_data(ssi_ctx* ctx, const float* X, const float* Y, int64_t N) {
    const int rc = for_each_device(ctx, [&](ssi_ctx* c, int) { return ssi_set_data(c, X, Y, N); });
    if (rc == SSI_OK) { ctx->N = N; ctx->has_data = true; }
    return rc;
}

int ssi_multi_set_subspace(ssi_ctx* ctx, const float* W_swa, const float* P, int64_t n, int32_t M) {
    const int rc = for_each_device(ctx, [&](ssi_ctx* c, int) { return ssi_set_subspace(c, W_swa, P, n, M); });
    if (rc == SSI_OK) { ctx->M = M; ctx->Mz = M; ctx->has_sub = true; }
    return rc;
}

int ssi_multi_set_decoder(ssi_ctx* ctx, const float* W_swa, int n_layers, const int32_t* dims, const int32_t* act, const float* theta) {
    const int rc = for_each_device(ctx, [&](ssi_ctx* c, int) { return ssi_set_decoder_impl(c, W_swa, n_layers, dims, act, theta); });
    if (rc == SSI_OK) { ctx->M = ctx->children[0]->M; ctx->Mz = ctx->children[0]->Mz; ctx->has_sub = true; }
    return rc;
}

// density(z) (grad == 0: second_out = terms, 3 x B) or l_pi_grad (grad == 1: second_out = gradient, M x B) over B points:
// device d takes the samples [b0_d, b1_d) and writes its slice of the host outputs
int ssi_multi_logpost(ssi_ctx* ctx, int grad, const float* Z, int64_t B, double sigma_m, double sigma_p, double sigma_z, uint32_t mask,
                      double* lp_out, double* second_out) {
    if (!ctx->has_model || !ctx->has_data || !ctx->has_sub)
        return ssi_fail(ctx, SSI_ERR_STATE, "model, data and subspace must be set before evaluating the log-posterior");
    if (B == 0) return SSI_OK;
    const int M = ctx->Mz;
    return for_each_shard(ctx, B, true, [&](ssi_ctx* c, int64_t b0, int64_t b1) {
        double* second = second_out ? second_out + (size_t)b0 * (grad ? M : 3) : nullptr;
        return grad ? ssi_logpost_grad_batch(c, Z + (size_t)b0 * M, b1 - b0, sigma_m, sigma_p, sigma_z, mask, lp_out + b0, second)
                    : ssi_logpost_batch(c, Z + (size_t)b0 * M, b1 - b0, sigma_m, sigma_p, sigma_z, mask, lp_out + b0, second);
    });
}

// chains [c0_d, c1_d) of the run go to device d with their global ids chain_offset + c; every device writes its columns
// of each step's row of the host traces.  The arguments have been checked for the whole run before any device starts.
int ssi_multi_mh_run(ssi_ctx* ctx, const ssi_mh_run_t& run) {
    const int rc = for_each_shard(ctx, run.n_chains, true,
                                  [&](ssi_ctx* c, int64_t c0, int64_t c1) { return ssi_mh_run_host_slice(c, run, c0, c1); });
    if (rc == SSI_OK) { ctx->mh_chains = run.n_chains; ctx->mh_kind = run.kind; }
    return rc;
}

int ssi_multi_mh_get_state(ssi_ctx* ctx, float* z_out, double* lp_out) {
    const int M = ctx->Mz;
    return for_each_shard(ctx, ctx->mh_chains, false, [&](ssi_ctx* c, int64_t c0, int64_t c1) {
        return ssi_mh_get_state_slice(c, c1 - c0, z_out ? z_out + (size_t)c0 * M : nullptr, lp_out ? lp_out + c0 : nullptr);
    });
}

int ssi_multi_hmc_get_adapt(ssi_ctx* ctx, double* adapt_out) {
    return for_each_shard(ctx, ctx->mh_chains, false, [&](ssi_ctx* c, int64_t c0, int64_t c1) {
        return ssi_hmc_get_adapt_slice(c, c1 - c0, adapt_out + 3 * (size_t)c0);
    });
}

int ssi_multi_project(ssi_ctx* ctx, const float* Z, int64_t B, float* W_out) {
    if (!ctx->has_model || !ctx->has_sub) return ssi_fail(ctx, SSI_ERR_STATE, "model and subspace must be set");
    if (B == 0) return SSI_OK;
    const int M = ctx->Mz;
    const int64_t n = ctx->model.n;
    return for_each_shard(ctx, B, true, [&](ssi_ctx* c, int64_t b0, int64_t b1) {
        return ssi_project(c, Z + (size_t)b0 * M, b1 - b0, W_out + (size_t)b0 * n);
    });
}

// the construction streams run on the first device; an installed subspace is then replicated to the others
int ssi_multi_swa_finish(ssi_ctx* ctx, int32_t M, float* W_swa_out, float* P_out, double* s_out, int32_t install) {
    ssi_ctx* c0 = ctx->children[0];
    if (!install || ctx->children.size() == 1) {
        const int rc = ssi_swa_finish(c0, M, W_swa_out, P_out, s_out, install);
        if (rc < 0) ctx->err = c0->err;
        else if (install) { ctx->M = M; ctx->Mz = M; ctx->has_sub = true; }
        return rc;
    }
    const int64_t n = c0->swa_n;
    std::vector<float> w, p;
    if (!W_swa_out) { w.resize((size_t)n); W_swa_out = w.data(); }
    if (!P_out) { p.resize((size_t)n * M); P_out = p.data(); }
    const int rc = ssi_swa_finish(c0, M, W_swa_out, P_out, s_out, 0);
    if (rc != SSI_OK) { if (rc < 0) ctx->err = c0->err; return rc; }
    return ssi_multi_set_subspace(ctx, W_swa_out, P_out, n, M);
}
