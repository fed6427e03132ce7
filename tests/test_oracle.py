"""Pins the CPU oracle (oracle/ssi_oracle.py) against independent closed forms.

The reference has no golden vectors (test/runtests.jl is empty, SURVEY 8c), so the oracle is
checked against scipy's multivariate normal, numpy's SVD, a second restatement of the forward
pass in torch Float64, known Philox4x32-10 answers, and the committed golden fixtures."""
import math
from pathlib import Path

import numpy as np
import pytest
import scipy.stats as st

import ssi_oracle as orc
from conftest import stable_seed

GOLD = Path(__file__).parent / "golden"


def test_param_layout_matches_flux_destructure():
    dims = (3, 4, 2)
    rng = np.random.default_rng(0)
    layers = [(rng.standard_normal((4, 3)), rng.standard_normal(4)), (rng.standard_normal((2, 4)), rng.standard_normal(2))]
    w = orc.flatten_params(layers)
    assert w.size == orc.n_params(dims) == 3 * 4 + 4 + 4 * 2 + 2
    # vec(W) is column-major: element (o, i) at o + i*out
    assert w[1 + 2 * 4] == layers[0][0][1, 2]
    assert w[12 + 3] == layers[0][1][3]
    back = orc.restructure(w, dims)
    for (W, b), (W2, b2) in zip(layers, back):
        np.testing.assert_array_equal(W, W2)
        np.testing.assert_array_equal(b, b2)


def test_forward_matches_torch_float64():
    torch = pytest.importorskip("torch")
    prob = orc.make_problem("readme")
    z = np.array([0.3, -1.2, 0.7])
    w = orc.project(prob.W_swa, prob.P, z)
    pred = orc.forward(w, prob.dims, prob.acts, prob.X)
    h = torch.tensor(prob.X, dtype=torch.float64)
    for (W, b), a in zip(orc.restructure(w, prob.dims), prob.acts):
        h = torch.tensor(W) @ h + torch.tensor(b)[:, None]
        if a == orc.ACT_RELU:
            h = torch.relu(h)
    np.testing.assert_allclose(pred, h.numpy(), rtol=1e-13, atol=1e-13)


@pytest.mark.parametrize("sigma", [1.0, 0.1, 2.5])
def test_gaussian_loglik_matches_scipy(sigma):
    rng = np.random.default_rng(1)
    pred, Y = rng.standard_normal((2, 50)), rng.standard_normal((2, 50))
    ref = st.multivariate_normal(mean=pred.T.reshape(-1), cov=sigma ** 2).logpdf(Y.T.reshape(-1))
    assert math.isclose(orc.gaussian_loglik(pred, Y, sigma), ref, rel_tol=1e-12)
    w = rng.standard_normal(30)
    ref_w = st.multivariate_normal(mean=np.zeros(30), cov=sigma ** 2).logpdf(w)
    assert math.isclose(orc.log_prior_w(w, sigma), ref_w, rel_tol=1e-12)


def test_q1_density_is_likelihood_only_by_default():
    prob = orc.make_problem("readme")
    z = np.array([0.1, 0.2, -0.3])
    ll, pw, pz = orc.density_terms(prob, z, 1.0, 1.0, 1.0)
    assert orc.density(prob, z) == ll
    assert orc.density(prob, z, mask=orc.TERM_LL | orc.TERM_PRIOR_W) == ll + pw
    # sigma_p has no effect on the reference density (dead code)
    assert orc.density(prob, z, sigma_p=7.0) == ll


def test_lp_invariant_to_datapoint_order():
    prob = orc.make_problem("readme")
    z = np.array([0.5, 0.5, 0.5])
    perm = np.random.default_rng(3).permutation(prob.N)
    prob2 = orc.Problem(prob.dims, prob.acts, prob.X[:, perm], prob.Y[:, perm], prob.W_swa, prob.P)
    assert math.isclose(orc.density(prob, z), orc.density(prob2, z), rel_tol=1e-13)


def test_philox_known_answers():
    # Random123 known-answer tests for philox4x32-10
    out = orc.philox4x32_10(np.array([0, 0, 0, 0]), np.array([0, 0]))
    assert [hex(int(v)) for v in out] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    out = orc.philox4x32_10(np.array([0xffffffff] * 4), np.array([0xffffffff] * 2))
    assert [hex(int(v)) for v in out] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    out = orc.philox4x32_10(np.array([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]), np.array([0xa4093822, 0x299f31d0]))
    assert [hex(int(v)) for v in out] == ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_rng_moments():
    eps = np.concatenate([orc.rng_normals(7, c, 0, 20) for c in range(2000)])
    assert abs(eps.mean()) < 0.02 and abs(eps.std() - 1.0) < 0.02
    e = np.array([orc.rng_exponential(7, c, 1) for c in range(4000)])
    assert abs(e.mean() - 1.0) < 0.05 and e.min() > 0


def test_q5_q6_rwmh_semantics():
    prob = orc.make_problem("readme")
    z, lp, acc, margin = orc.rwmh_chain(prob, 10, seed=11, chain=0, sigma_z=1.0)
    # Q5: sample 0 is a draw from the proposal and is kept
    np.testing.assert_array_equal(z[0], orc.propose_f32(np.zeros(3, np.float32), 1.0, orc.rng_normals(11, 0, 0, 3)))
    assert lp[0] == orc.density(prob, z[0])
    for t in range(1, 10):
        if acc[t]:
            assert margin[t] > 0 and lp[t] == orc.density(prob, z[t])
        else:                      # rejected: state repeats
            assert margin[t] <= 0 and lp[t] == lp[t - 1] and np.array_equal(z[t], z[t - 1])


def test_rwmh_all_rejected_keeps_state():
    prob = orc.make_problem("readme")
    z, lp, acc, _ = orc.rwmh_chain(prob, 6, seed=1, chain=0, density_fn=lambda zz: 0.0 if np.allclose(zz, 0.25) else -1e300,
                                   z0=np.full(3, 0.25, np.float32))
    assert acc[1:].sum() == 0 and np.all(z == 0.25)


def test_q2_q4_swa_recurrence_is_not_a_running_mean():
    rng = np.random.default_rng(5)
    snaps = [rng.standard_normal(6) for _ in range(4)]
    ns = [1.0, 1.0, 2.0, 2.0]            # two mini-batches per epoch: n = i/c repeats (Q2)
    W_swa, P, s, A = orc.construct_from_snapshots(snaps, ns, M=2)
    m = np.zeros(6)
    for w, n in zip(snaps, ns):
        m = (n * m + w) / (n + 1)
    np.testing.assert_allclose(W_swa, m)
    assert not np.allclose(W_swa, np.mean(snaps, axis=0))
    # Q4: deviation against the UPDATED mean
    m1 = (1.0 * np.zeros(6) + snaps[0]) / 2.0
    np.testing.assert_allclose(A[:, 0], snaps[0] - m1)
    # Q3: all columns kept
    assert A.shape == (6, 4)


def test_svd_and_gram_routes_agree():
    rng = np.random.default_rng(6)
    n, K, M = 200, 12, 4
    base = rng.standard_normal(n)
    snaps = [base + 0.1 * np.cumsum(rng.standard_normal((K, n)), axis=0)[k] for k in range(K)]
    ns = np.arange(1, K + 1, dtype=float)
    W1, P1, s1, A = orc.construct_from_snapshots(snaps, ns, M, route="svd")
    W2, P2, s2, _ = orc.construct_from_snapshots(snaps, ns, M, route="gram")
    np.testing.assert_allclose(s1[:M], s2[:M], rtol=1e-9)
    np.testing.assert_allclose(orc.align_signs(P2, P1), P1, rtol=1e-7, atol=1e-9)
    # P columns orthogonal with norms s_k
    G = P1.T @ P1
    np.testing.assert_allclose(G, np.diag(s1[:M] ** 2), atol=1e-9 * s1[0] ** 2)
    with pytest.raises(ValueError):
        orc.construct_from_snapshots(snaps[:2], ns[:2], M)       # fewer columns than M


def test_weight_prior_m_space_identity():
    """|W_swa + P z|^2 = w'w + 2 (P'w)'z + z'P'P z — the identity the device finalize uses."""
    prob = orc.make_problem("readme")
    z = np.array([0.3, -0.4, 1.1])
    w = orc.project(prob.W_swa, prob.P, z)
    Pd, wd = prob.P.astype(np.float64), prob.W_swa.astype(np.float64)
    rhs = wd @ wd + 2 * (Pd.T @ wd) @ z + z @ (Pd.T @ Pd) @ z
    assert math.isclose(w @ w, rhs, rel_tol=1e-12)


@pytest.mark.parametrize("name", ["readme", "uci_small", "wide_small"])
def test_golden_logpost(name):
    g = np.load(GOLD / f"logpost_{name}.npz")
    prob = orc.Problem(tuple(g["dims"]), tuple(g["acts"]), g["X"], g["Y"], g["W_swa"], g["P"])
    lp, terms = orc.logpost_batch(prob, g["Z"], float(g["sigma_m"]), float(g["sigma_p"]), float(g["sigma_z"]), mask=7)
    np.testing.assert_allclose(terms, g["terms"], rtol=1e-12)
    np.testing.assert_allclose(lp, g["terms"].sum(axis=0), rtol=1e-12)


def test_golden_mh():
    g = np.load(GOLD / "mh_readme.npz")
    prob = orc.Problem(tuple(g["dims"]), tuple(g["acts"]), g["X"], g["Y"], g["W_swa"], g["P"])
    for c in range(int(g["n_chains"])):
        z, lp, acc, _ = orc.rwmh_chain(prob, int(g["n_steps"]), int(g["seed"]), c, float(g["sigma_z"]), float(g["sigma_m"]))
        np.testing.assert_array_equal(z, g["z_trace"][c])
        np.testing.assert_allclose(lp, g["lp_trace"][c], rtol=1e-12)
        np.testing.assert_array_equal(acc, g["accept"][c])


def test_golden_construction():
    g = np.load(GOLD / "construct_small.npz")
    W_swa, P, s, _ = orc.construct_from_snapshots(list(g["snapshots"]), g["n_scalars"], int(g["M"]))
    np.testing.assert_allclose(W_swa, g["W_swa"], rtol=1e-12)
    np.testing.assert_allclose(orc.align_signs(P, g["P"]), g["P"], rtol=1e-8, atol=1e-12)
    np.testing.assert_allclose(s, g["s"], rtol=1e-10, atol=1e-12)


def test_predictive_sweep_against_torch_float64():
    """The sweep after the path (docs/src/nn_example.md:207-216, src/plotting.jl:8-9): trajectories, mean, corrected std."""
    import torch
    rng = np.random.default_rng(11)
    dims, acts, M, B, Ng = (3, 8, 5, 2), (2, 1, 0), 4, 7, 13
    n = orc.n_params(dims)
    W_swa, P = orc.glorot_flat(rng, dims), (0.2 * rng.standard_normal((n, M))).astype(np.float32)
    Z, Xg = rng.standard_normal((M, B)), rng.standard_normal((dims[0], Ng))
    traj, mu, sd = orc.predictive_sweep(dims, acts, W_swa, P, Z, Xg)
    assert traj.shape == (2, Ng, B)
    ref = []
    for b in range(B):
        w = torch.from_numpy(W_swa.astype(np.float64) + P.astype(np.float64) @ Z[:, b])
        h, off = torch.from_numpy(Xg), 0
        for l, act in enumerate(acts):
            i, o = dims[l], dims[l + 1]
            Wl = w[off:off + i * o].reshape(i, o).T          # column-major (o, i)
            off += i * o
            h = Wl @ h + w[off:off + o][:, None]
            off += o
            h = [lambda x: x, torch.relu, torch.tanh, torch.sigmoid][act](h)
        ref.append(h)
    ref = torch.stack(ref, dim=2)
    np.testing.assert_allclose(traj, ref.numpy(), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(mu, ref.mean(dim=2).numpy(), rtol=1e-12)
    np.testing.assert_allclose(sd, ref.std(dim=2, unbiased=True).numpy(), rtol=1e-11)
    assert np.isnan(orc.predictive_sweep(dims, acts, W_swa, P, Z[:, :1], Xg)[2]).all()


@pytest.mark.parametrize("dims,acts", [((3, 6, 4, 2), (2, 3, 0)), ((5, 9, 1), (1, 0)), ((4, 3), (2,))])
def test_density_gradient_against_torch_autograd_and_central_differences(dims, acts):
    """l_pi_grad (src/space_inference.jl:107): the analytic reverse-mode restatement vs torch autograd (Float64) and
    central differences, with every combination of terms."""
    import torch
    rng = np.random.default_rng(sum(dims))
    n, M, N = orc.n_params(dims), 4, 17
    prob = orc.Problem(dims, acts, rng.standard_normal((dims[0], N)).astype(np.float32),
                       rng.standard_normal((dims[-1], N)).astype(np.float32), orc.glorot_flat(rng, dims),
                       (0.3 * rng.standard_normal((n, M))).astype(np.float32))
    z = rng.standard_normal(M)
    sm, sp, sz = 0.7, 1.3, 0.9
    for mask in (1, 2, 4, 3, 7):
        lp, g = orc.density_and_grad(prob, z, sm, sp, sz, mask)
        assert lp == orc.density(prob, z, sm, sp, sz, mask)
        # central differences
        fd = np.array([(orc.density(prob, z + 1e-6 * e, sm, sp, sz, mask) - orc.density(prob, z - 1e-6 * e, sm, sp, sz, mask)) / 2e-6
                       for e in np.eye(M)])
        np.testing.assert_allclose(g, fd, rtol=2e-5, atol=1e-6 * max(1.0, np.abs(g).max()))
        # torch autograd
        zt = torch.tensor(z, dtype=torch.float64, requires_grad=True)
        w = torch.from_numpy(prob.W_swa.astype(np.float64)) + torch.from_numpy(prob.P.astype(np.float64)) @ zt
        h, off = torch.from_numpy(prob.X.astype(np.float64)), 0
        for l, act in enumerate(acts):
            i, o = dims[l], dims[l + 1]
            Wl = w[off:off + i * o].reshape(i, o).T
            off += i * o
            h = Wl @ h + w[off:off + o][:, None]
            off += o
            h = [lambda x: x, torch.relu, torch.tanh, torch.sigmoid][act](h)
        Y = torch.from_numpy(prob.Y.astype(np.float64))
        tot = 0.0
        if mask & 1:
            tot = tot - ((h - Y) ** 2).sum() / (2 * sm * sm)
        if mask & 2:
            tot = tot - (w ** 2).sum() / (2 * sp * sp)
        if mask & 4:
            tot = tot - (zt ** 2).sum() / (2 * sz * sz)
        tot.backward()
        np.testing.assert_allclose(g, zt.grad.numpy(), rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("dims,acts", [((3, 6, 4, 2), (2, 3, 0)), ((5, 9, 7, 3), (1, 0, 2)), ((4, 5, 2), (3, 1))])
def test_mse_gradient_against_torch_autograd(dims, acts):
    """The training step's cost, Flux.Losses.mse(m(x), y) (src/subspace_construction.jl:39-43): loss and dL/dw in the flat
    layout vs torch autograd in Float64, every activation in a hidden and in the output position."""
    import torch
    rng = np.random.default_rng(stable_seed(dims, acts))
    nb = 13
    w = orc.glorot_flat(rng, dims) + 0.1 * rng.standard_normal(orc.n_params(dims)).astype(np.float32)
    X = rng.standard_normal((dims[0], nb)).astype(np.float32)
    Y = rng.standard_normal((dims[-1], nb)).astype(np.float32)
    loss, gw = orc.mse_loss_and_grad(w, dims, acts, X, Y)
    wt = torch.tensor(w, dtype=torch.float64, requires_grad=True)
    h, off = torch.from_numpy(X.astype(np.float64)), 0
    for l, act in enumerate(acts):
        i, o = dims[l], dims[l + 1]
        Wl = wt[off:off + i * o].reshape(i, o).T
        off += i * o
        h = [lambda x: x, torch.relu, torch.tanh, torch.sigmoid][act](Wl @ h + wt[off:off + o][:, None])
        off += o
    tot = torch.mean((h - torch.from_numpy(Y.astype(np.float64))) ** 2)
    tot.backward()
    np.testing.assert_allclose(loss, tot.item(), rtol=1e-12)
    np.testing.assert_allclose(gw, wt.grad.numpy(), rtol=1e-10, atol=1e-12 * np.abs(gw).max())


def test_adam_step_matches_flux_adam(ssi):
    """Five steps of the Float64 ADAM restatement vs the package's Flux 0.11 ADAM (torch, Float32)."""
    import torch
    rng = np.random.default_rng(5)
    n, eta, beta = 257, 3e-3, (0.8, 0.99)
    w0 = rng.standard_normal(n).astype(np.float32)
    p = torch.tensor(w0, requires_grad=True)
    opt = ssi.ADAM(eta, beta)
    w, m, v = w0.astype(np.float64), np.zeros(n), np.zeros(n)
    for t in range(1, 6):
        g = (rng.standard_normal(n) * 10.0 ** rng.uniform(-4, 1, n)).astype(np.float32)
        p.grad = torch.from_numpy(g.copy())
        opt.update([p])
        w, m, v = orc.adam_step(w, g, m, v, t, eta, *beta)
        np.testing.assert_allclose(p.detach().numpy(), w, rtol=0, atol=4 * np.spacing(np.float32(np.abs(w).max())) + 1e-6 * eta,
                                   err_msg=f"step {t}")


def test_mala_restatement_satisfies_detailed_balance():
    """pi(z) q(z'|z) alpha(z -> z') == pi(z') q(z|z') alpha(z' -> z): the proposal-density ratio in mala_log_alpha is
    the one that makes the Langevin proposal reversible, for an arbitrary pair of points."""
    rng = np.random.default_rng(8)
    prob = orc.make_problem("readme")
    s = 0.3
    for _ in range(5):
        z, zp = rng.standard_normal(prob.M) * 0.2, rng.standard_normal(prob.M) * 0.2
        lp, g = orc.density_and_grad(prob, z)
        lpp, gp = orc.density_and_grad(prob, zp)
        h = 0.5 * s * s
        logq = lambda a, b, gb: -np.sum((a - b - h * gb) ** 2) / (2 * s * s)
        la_fwd = orc.mala_log_alpha(z, zp, lp, lpp, g, gp, s)
        la_rev = orc.mala_log_alpha(zp, z, lpp, lp, gp, g, s)
        assert abs(la_fwd + la_rev) < 1e-9 * max(1.0, abs(la_fwd))
        lhs = lp + logq(zp, z, g) + min(0.0, la_fwd)
        rhs = lpp + logq(z, zp, gp) + min(0.0, la_rev)
        assert abs(lhs - rhs) < 1e-8 * max(1.0, abs(lhs))
    zt, lt, acc, _ = orc.mala_chain(prob, 6, 3, 0, sigma_z=0.05)
    assert acc[0] == 1 and zt.shape == (6, prob.M) and np.isfinite(lt).all()


def test_next_rows_golden_fixture_is_reproduced():
    """tests/golden/next_rows.npz (gradient, MALA, predictive sweep) is what the oracle computes today."""
    g = np.load(Path(__file__).parent / "golden" / "next_rows.npz")
    for name in ("readme", "uci"):
        prob = orc.Problem(tuple(int(d) for d in g[f"{name}_dims"]), tuple(int(a) for a in g[f"{name}_acts"]), g[f"{name}_X"],
                           g[f"{name}_Y"], g[f"{name}_W_swa"], g[f"{name}_P"])
        sm, sp, sz = g[f"{name}_sig"]
        for k, mask in enumerate((1, 3, 7)):
            for b in range(g[f"{name}_Z"].shape[1]):
                lp, grad = orc.density_and_grad(prob, g[f"{name}_Z"][:, b].astype(np.float64), sm, sp, sz, mask)
                np.testing.assert_allclose(lp, g[f"{name}_lp"][k, b], rtol=1e-12)
                np.testing.assert_allclose(grad, g[f"{name}_grad"][k, :, b], rtol=1e-9, atol=1e-9)
    prob = orc.make_problem("readme")
    for c in range(3):
        z, lp, acc, _ = orc.mala_chain(prob, 8, int(g["mala_seed"]), c, sigma_z=float(g["mala_sigma_z"]))
        np.testing.assert_array_equal(acc, g["mala_accept"][c])
        np.testing.assert_array_equal(z, g["mala_z"][c])
    traj, mu, sd = orc.predictive_sweep(prob.dims, prob.acts, prob.W_swa, prob.P, g["pred_Z"], g["pred_Xg"])
    np.testing.assert_allclose(mu, g["pred_mean"], rtol=1e-12)
    np.testing.assert_allclose(sd, g["pred_std"], rtol=1e-10)


def test_bench_workloads_match_the_oracle_problems():
    """workloads.py (what bench.py times) generates exactly the problems the oracle-based tests use."""
    import sys
    sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
    import workloads
    for name, N in (("readme", None), ("uci", 300), ("wide", 40)):
        a, b = workloads.make(name, N=N), orc.make_problem(name, N=N)
        assert tuple(a.dims) == tuple(b.dims) and tuple(a.acts) == tuple(b.acts) and a.M == b.M and a.N == b.N
        for k in ("X", "Y", "W_swa", "P"):
            np.testing.assert_array_equal(getattr(a, k), getattr(b, k))
