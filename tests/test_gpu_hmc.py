"""Fixed-length HMC with per-chain dual averaging on the device (alg = :static_hmc, ssi_hmc_run) against the Float64
restatement in tests/hmc_oracle.py, plus the invariances the other samplers keep: chain sharding, resume, several devices."""
import math

import numpy as np
import pytest

import hmc_oracle as hmc
import ssi_oracle as orc

pytestmark = pytest.mark.gpu

LL_PZ = orc.TERM_LL | orc.TERM_PRIOR_Z


def _setup(engine, prob):
    engine.set_model(prob.dims, prob.acts)
    engine.set_data(prob.X, prob.Y)
    engine.set_subspace(prob.W_swa, prob.P)


def _tensor_problem():
    """A net wide enough that the reverse pass runs its large contractions on the tensor cores (ssi_gemm_tc.cu)."""
    dims, acts, N, M = (96, 256, 192, 8), (1, 2, 0), 3000, 12
    rng = np.random.default_rng(96256)
    n = orc.n_params(dims)
    return orc.Problem(dims, acts, rng.standard_normal((dims[0], N)).astype(np.float32),
                       rng.standard_normal((dims[-1], N)).astype(np.float32), orc.glorot_flat(rng, dims),
                       (0.3 * rng.standard_normal((n, M))).astype(np.float32))


# name, problem, sigma_z, sigma_m, step size: in the oracle's chains of this test the step sizes leave 2 to 4 of the 28
# transitions rejected, just below the stability limit of the leapfrog integrator
TEACHER_CASES = [
    ("readme", lambda: orc.make_problem("readme"), 0.45, 1.0, 0.45),                 # generic reverse pass
    ("uci", lambda: orc.make_problem("uci", N=1500), 0.02, 0.1, 0.02),               # BASIS value + gradient fast path
    ("tensor", _tensor_problem, 0.005, 0.7, 1e-3),                                    # tensor-core GEMM gradient
]


@pytest.mark.parametrize("name,make,sigma_z,sigma_m,eps", TEACHER_CASES, ids=[c[0] for c in TEACHER_CASES])
def test_trajectories_teacher_forced(ssi, engine, name, make, sigma_z, sigma_m, eps):
    """Fixed step size, L = 5: from the device's own state at t - 1 and the replayed momentum, the Float64 oracle integrates
    the same trajectory and takes the same decision outside a tie band of 1e-5 |lp|."""
    prob = make()
    _setup(engine, prob)
    C, S, L, seed = 4, 8, 5, 31337
    before = engine.stats().gemm_tc_launches
    zt, lt, at, et = engine.hmc_run(C, S, seed, eps, L, sigma_z=sigma_z, sigma_m=sigma_m)
    if name == "tensor":
        assert engine.stats().gemm_tc_launches > before
    assert np.isnan(et[:, 0]).all() and (et[:, 1:] == eps).all()
    near_ties = 0
    for c in range(C):
        z = zt[:, c, :].T
        np.testing.assert_array_equal(z[0], orc.propose_f32(np.zeros(prob.M, np.float32), sigma_z, orc.rng_normals(seed, c, 0, prob.M)))
        assert at[c, 0] == 1
        for t in range(1, S):
            lp, g = orc.density_and_grad(prob, z[t - 1], sigma_m)
            np.testing.assert_allclose(lt[c, t - 1], lp, rtol=1e-5)
            e = orc.rng_exponential(seed, c, t)
            z_next, _, g_next, dH, accepted, divergent, _ = hmc.hmc_transition(
                prob, z[t - 1], g, lp, eps, L, None, orc.rng_normals(seed, c, t, prob.M), e, sigma_m=sigma_m)
            if divergent:
                assert at[c, t] == 2, f"chain {c} step {t} diverges in the oracle"
                continue
            margin = -dH + e
            if abs(margin) <= 1e-5 * max(1.0, abs(lp)):
                near_ties += 1
                continue
            assert at[c, t] == (1 if accepted else 0), f"decision differs at chain {c} step {t}, margin {margin}"
            expect = z_next
            # The gradient is held to 1e-4 of its norm (test_gradient_vs_oracle); through L kicks of eps and L drifts that
            # moves the end point by at most eps^2 L^2 1e-4 max|g| (twice that for the curvature along the way), plus one
            # FP32 rounding of the position per drift.
            gmax = max(np.abs(g).max(), np.abs(g_next).max())
            tol = 2 * eps * eps * L * L * 1e-4 * gmax + L * 2.4e-7 * np.abs(expect).max() + 1e-12
            np.testing.assert_allclose(z[t], expect, rtol=0, atol=tol, err_msg=f"chain {c} step {t}")
    assert near_ties <= 3
    assert 0 < (at[:, 1:] == 1).mean() < 1           # both outcomes occur


def test_step_size_adaptation(ssi, engine):
    """n_adapts = 30: every step size the device uses is the dual-averaging update (Alg. 5) of its previous one with the
    oracle's teacher-forced acceptance statistic; after warm-up the step size is exp(log eps_bar) of ssi_hmc_get_adapt.
    A weak likelihood (sigma_m = 100) under the z prior keeps the device's energies equal to the oracle's to ~1e-8, so that
    the acceptance statistic, not the density's FP32 rounding, is what is compared."""
    prob = orc.make_problem("readme")
    _setup(engine, prob)
    C, S, L, seed, eps0, delta, na, sm = 6, 40, 4, 777, 0.1, 0.8, 30, 100.0
    zt, lt, at, et = engine.hmc_run(C, S, seed, eps0, L, n_adapts=na, target_accept=delta, sigma_m=sm, mask=LL_PZ)
    ad = engine.hmc_adapt()
    mu = math.log(10 * eps0)
    f = lambda zz: orc.density_and_grad(prob, zz, sm, 1.0, 1.0, LL_PZ)
    for c in range(C):
        z = zt[:, c, :].T
        assert et[c, 1] == pytest.approx(eps0, rel=1e-15)
        log_eps_bar = 0.0
        for t in range(1, na + 1):
            lp, g = f(z[t - 1])
            out = hmc.hmc_transition(prob, z[t - 1], g, lp, et[c, t], L, None, orc.rng_normals(seed, c, t, prob.M),
                                     orc.rng_exponential(seed, c, t), grad_fn=f)
            hbar_prev = 0.0 if t == 1 else (mu - math.log(et[c, t])) * hmc.DA_GAMMA / math.sqrt(t - 1)
            state = hmc.dual_averaging_update((math.log(et[c, t]), log_eps_bar, hbar_prev), t, out[6], eps0, delta)
            log_eps_bar = state[1]
            if t < na:
                assert et[c, t + 1] == pytest.approx(math.exp(state[0]), rel=1e-4), f"chain {c} transition {t}"
        assert (et[c, na + 1:] == et[c, na + 1]).all()
        assert et[c, na + 1] == pytest.approx(math.exp(ad[1, c]), rel=1e-15)
        assert ad[1, c] == pytest.approx(log_eps_bar, rel=1e-4, abs=1e-6)
    assert 0 < (at[:, 1:] == 1).mean() < 1


def _linear_head_problem(N=2000, lam=(81.0, 90.0, 100.0, 110.0, 121.0), sigma_m=0.1):
    """uci 13-50-1 relu with P's nonzero rows only in the output layer's weights and bias: pred is affine in z, so with
    mask LL | PRIOR_Z (sigma_z = 1) the posterior is exactly Gaussian.  P is chosen so that its precision has the
    eigenvalues `lam` (a mildly anisotropic target)."""
    base = orc.make_problem("uci", N=N)
    rng = np.random.default_rng(5150)
    dims, M = base.dims, len(lam)
    _, (w1, _, _, _) = orc.layer_offsets(dims)
    W1, bb1 = orc.restructure(base.W_swa.astype(np.float64), dims)[0]
    H = np.maximum(W1 @ base.X.astype(np.float64) + bb1[:, None], 0.0)
    Haug = np.vstack([H, np.ones((1, N))])                      # output-layer weights (50) then bias (1)
    ev, U = np.linalg.eigh(Haug @ Haug.T)
    keep = ev > 1e-6 * ev.max()
    Q, _ = np.linalg.qr(rng.standard_normal((int(keep.sum()), M)))
    Pout = U[:, keep] @ (Q / np.sqrt(ev[keep])[:, None]) * (sigma_m * np.sqrt(np.asarray(lam) - 1.0))[None, :]
    P = np.zeros((orc.n_params(dims), M), np.float32)
    P[w1:w1 + Haug.shape[0]] = Pout
    return orc.Problem(dims, base.acts, base.X, base.Y, base.W_swa, P), sigma_m


def test_exact_gaussian_posterior(ssi, engine):
    """4096 chains, 100 warm-up transitions then 50 more on an exactly Gaussian posterior: the final states' mean and
    covariance are the posterior's (mean and precision from M + 1 oracle gradients) and the acceptance rate after warm-up
    is near the 0.8 target."""
    prob, sm = _linear_head_problem()
    _setup(engine, prob)
    M = prob.M
    g0 = orc.density_and_grad(prob, np.zeros(M), sm, 1.0, 1.0, LL_PZ)[1]
    A = np.stack([g0 - orc.density_and_grad(prob, np.eye(M)[i], sm, 1.0, 1.0, LL_PZ)[1] for i in range(M)], axis=1)
    A = 0.5 * (A + A.T)                                           # gradient = g0 - A z
    mean = np.linalg.solve(A, g0)
    Lc = np.linalg.cholesky(A)                                    # whitened w = Lc^T (z - mean) ~ N(0, I)
    C, na, extra = 4096, 100, 50
    zt, lt, at, et = engine.hmc_run(C, na + extra + 1, 2468, 0.1, 5, n_adapts=na, sigma_m=sm, mask=LL_PZ,
                                    want_z=False, want_lp=False)
    z, _ = engine.mh_state()
    w = (z.astype(np.float64) - mean[:, None]).T @ Lc
    se = 1.0 / math.sqrt(C)
    assert np.all(np.abs(w.mean(axis=0)) < 4 * se), w.mean(axis=0) / se
    np.testing.assert_allclose(w.var(axis=0), 1.0, rtol=0.10)
    acc = (at[:, na + 1:] == 1).mean()
    assert 0.7 <= acc <= 0.9, acc
    # dual averaging probes mu = log(10 eps0) early in warm-up, where some transitions may diverge; none may after it
    assert not (at[:, na + 1:] == 2).any()


def test_chain_sharding_is_bitwise_invariant(ssi, engine):
    """Chains [0, 32) in one call == [0, 16) and [16, 32) in two calls, for all four traces (adaptation is per chain)."""
    prob = orc.make_problem("uci", N=1500)
    _setup(engine, prob)
    kw = dict(n_adapts=6, sigma_z=0.02, sigma_m=0.1)
    full = engine.hmc_run(32, 12, 7, 0.01, 4, **kw)
    a = engine.hmc_run(16, 12, 7, 0.01, 4, chain_offset=0, **kw)
    b = engine.hmc_run(16, 12, 7, 0.01, 4, chain_offset=16, **kw)
    np.testing.assert_array_equal(full[0], np.concatenate([a[0], b[0]], axis=1))
    for k in (1, 2, 3):
        np.testing.assert_array_equal(full[k], np.concatenate([a[k], b[k]], axis=0))


@pytest.mark.parametrize("h", [3, 10])
def test_resume_is_bitwise_identical(ssi, engine, h):
    """run(0..S) == run(0..h) then run(h..S) from ssi_mh_get_state + ssi_hmc_get_adapt, with h inside warm-up (3) and
    after it (10)."""
    prob = orc.make_problem("uci", N=600)
    _setup(engine, prob)
    C, S, seed = 37, 14, 909
    kw = dict(n_adapts=6, sigma_z=0.05, sigma_m=0.3, chain_offset=11)
    full = engine.hmc_run(C, S, seed, 0.02, 3, **kw)
    z_end, lp_end = engine.mh_state()
    np.testing.assert_array_equal(z_end, full[0][:, :, -1])
    np.testing.assert_array_equal(lp_end, full[1][:, -1])
    head = engine.hmc_run(C, h, seed, 0.02, 3, **kw)
    z_mid, _ = engine.mh_state()
    ad_mid = engine.hmc_adapt()
    for k in range(4):
        np.testing.assert_array_equal(head[k], full[k][..., :h])
    # ... the process may exit here: (seed, step, z, adaptation state) is the whole checkpoint ...
    tail = engine.hmc_run(C, S - h, seed, 0.02, 3, z0=z_mid, step_offset=h, adapt_state=ad_mid, **kw)
    for k in range(4):
        np.testing.assert_array_equal(tail[k], full[k][..., h:])
    assert engine.stats().mh_proposals == C * (S - h)
    with pytest.raises(ssi.SsiError) as ei:                   # warm-up state missing
        engine.hmc_run(C, 2, seed, 0.02, 3, z0=z_mid, step_offset=h, **kw)
    assert ei.value.code == -1
    fixed = dict(kw, n_adapts=0)                              # a fixed step size needs no adaptation state
    f_full = engine.hmc_run(C, S, seed, 0.02, 3, **fixed)
    engine.hmc_run(C, h, seed, 0.02, 3, **fixed)
    f_tail = engine.hmc_run(C, S - h, seed, 0.02, 3, z0=engine.mh_state()[0], step_offset=h, **fixed)
    np.testing.assert_array_equal(f_tail[0], f_full[0][:, :, h:])
    engine.mh_run(C, 2, seed, sigma_z=0.05, sigma_m=0.3)
    with pytest.raises(ssi.SsiError) as ei:                   # the last run was not HMC
        engine.hmc_adapt()
    assert ei.value.code == -3


def test_multi_device_context_matches_single(ssi, engine):
    """ssi_ctx_create_multi over every visible device (the degenerate 1-device case with one GPU): bit-identical traces and
    adaptation state; the device-pointer entry point is refused."""
    import torch
    ndev = torch.cuda.device_count()
    prob = orc.make_problem("uci", N=900)
    _setup(engine, prob)
    kw = dict(n_adapts=4, sigma_z=0.05, sigma_m=0.2, chain_offset=7)
    ref = engine.hmc_run(301, 7, 5, 0.02, 3, **kw)
    ad_ref = engine.hmc_adapt()
    for devs in ([0], list(range(ndev))):
        with ssi.Engine(devs) as multi:
            _setup(multi, prob)
            out = multi.hmc_run(301, 7, 5, 0.02, 3, **kw)
            for k in range(4):
                np.testing.assert_array_equal(out[k], ref[k])
            np.testing.assert_array_equal(multi.hmc_adapt(), ad_ref)
            st = multi.stats()
            assert st.mh_proposals == 301 * 6 and st.mh_accepts == int((ref[2][:, 1:] == 1).sum())
            z_end, _ = multi.mh_state()
            tail_m = multi.hmc_run(301, 2, 5, 0.02, 3, z0=z_end, step_offset=7, adapt_state=ad_ref, **kw)
            tail_s = engine.hmc_run(301, 2, 5, 0.02, 3, z0=z_end, step_offset=7, adapt_state=ad_ref, **kw)
            for k in range(4):
                np.testing.assert_array_equal(tail_m[k], tail_s[k])
            with pytest.raises(ssi.SsiError) as ei:
                multi.hmc_run_dev(4, 2, 5, 0.02, 3)
            assert ei.value.code == -5


def test_divergence_is_contained(ssi, engine):
    """A chain started far in the tail with a large step size diverges: its transitions are rejected as divergent (2), its
    position stays finite and unchanged, and the other chains are bitwise those of a run without it."""
    prob = orc.make_problem("uci", N=1500)
    _setup(engine, prob)
    C, S, seed = 8, 10, 4
    rng = np.random.default_rng(8)
    z0 = (0.02 * rng.standard_normal((prob.M, C))).astype(np.float32)
    z0_tail = np.concatenate([z0, np.full((prob.M, 1), 50.0, np.float32)], axis=1)
    kw = dict(n_adapts=4, sigma_z=0.02, sigma_m=0.1)
    base = engine.hmc_run(C, S, seed, 0.05, 5, z0=z0, **kw)
    out = engine.hmc_run(C + 1, S, seed, 0.05, 5, z0=z0_tail, **kw)
    np.testing.assert_array_equal(out[0][:, :C], base[0])
    for k in (1, 2, 3):
        np.testing.assert_array_equal(out[k][:C], base[k])
    acc = out[2][C]
    assert (acc[1:] == 2).any()
    for t in range(1, S):
        if acc[t] != 1:
            np.testing.assert_array_equal(out[0][:, C, t], out[0][:, C, t - 1])
    assert np.isfinite(out[0]).all() and np.isfinite(out[1]).all() and np.isfinite(out[3][:, 1:]).all()


def test_device_pointer_entry_point_equals_host(ssi, engine):
    """ssi_hmc_run_dev into torch buffers == ssi_hmc_run, bit for bit, including a continued run from device state."""
    import torch
    prob = orc.make_problem("uci", N=1200)
    _setup(engine, prob)
    C, S, seed, M = 50, 9, 13, prob.M
    kw = dict(n_adapts=5, sigma_z=0.03, sigma_m=0.2, chain_offset=3)
    ref = engine.hmc_run(C, S, seed, 0.02, 4, **kw)
    engine.hmc_run(C, 4, seed, 0.02, 4, **kw)
    z_mid, ad_mid = engine.mh_state()[0], engine.hmc_adapt()
    dev = torch.device("cuda", 0)
    zt = torch.empty((S, C, M), dtype=torch.float32, device=dev)
    lt = torch.empty((S, C), dtype=torch.float64, device=dev)
    at = torch.empty((S, C), dtype=torch.uint8, device=dev)
    et = torch.empty((S, C), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    engine.hmc_run_dev(C, S, seed, 0.02, 4, d_z_trace=zt.data_ptr(), d_lp_trace=lt.data_ptr(), d_accept=at.data_ptr(),
                       d_step_size=et.data_ptr(), **kw)
    engine.sync()
    np.testing.assert_array_equal(zt.cpu().numpy().transpose(2, 1, 0), ref[0])
    np.testing.assert_array_equal(lt.cpu().numpy().T, ref[1])
    np.testing.assert_array_equal(at.cpu().numpy().T, ref[2])
    np.testing.assert_array_equal(et.cpu().numpy().T, ref[3])
    dz = torch.from_numpy(np.ascontiguousarray(z_mid.T)).to(dev)
    dad = torch.from_numpy(np.ascontiguousarray(ad_mid.T)).to(dev)
    lt2 = torch.empty((S - 4, C), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    engine.hmc_run_dev(C, S - 4, seed, 0.02, 4, step_offset=4, d_z0=dz.data_ptr(), d_adapt=dad.data_ptr(),
                       d_lp_trace=lt2.data_ptr(), **kw)
    engine.sync()
    np.testing.assert_array_equal(lt2.cpu().numpy().T, ref[1][:, 4:])


def test_api_static_hmc(ssi):
    """sub_inference / auto_inference with alg=:static_hmc return itr weight vectors whose lp is the oracle likelihood;
    auto_inference's default :hmc (NUTS in the reference) is still not a device sampler."""
    rng = np.random.default_rng(21)
    X = rng.standard_normal((13, 300)).astype(np.float32)
    Y = rng.standard_normal((1, 300)).astype(np.float32)
    data = ssi.DataLoader(X, Y, batchsize=100)
    m = ssi.Chain(ssi.Dense(13, 50, ssi.relu, rng=rng), ssi.Dense(50, 1, rng=rng))
    w = ssi.extract_params(m)
    P = (0.05 * rng.standard_normal((w.shape[0], 4))).astype(np.float32)
    chn, lp = ssi.sub_inference(m, data, w, P, σ_z=0.1, σ_m=0.5, itr=12, M=4, alg=":static_hmc", seed=3,
                                n_leapfrog=4, step_size=0.02)
    assert len(chn) == 12 and chn[0].shape == w.shape and lp.shape == (12,)
    for wt, l in zip(chn, lp):
        np.testing.assert_allclose(l, orc.gaussian_loglik(orc.forward(wt, m.dims, m.acts, X), Y, 0.5), rtol=1e-5)
    dec = ssi.Chain(ssi.Dense(4, w.shape[0], rng=rng))       # linear head: W = W_swa + decoder(z)
    chn, lp = ssi.auto_inference(m, data, dec, w, σ_z=0.1, σ_m=0.5, itr=12, M=4, alg=":static_hmc", seed=3,
                                 n_leapfrog=4, step_size=0.02)
    assert len(chn) == 12 and lp.shape == (12,)
    for wt, l in zip(chn, lp):
        np.testing.assert_allclose(l, orc.gaussian_loglik(orc.forward(wt, m.dims, m.acts, X), Y, 0.5), rtol=1e-5)
    with pytest.raises(NotImplementedError):
        ssi.auto_inference(m, data, dec, w, M=4, itr=3)
