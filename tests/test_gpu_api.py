"""The reference-facing functions (host mirror) end to end, README-style."""
import numpy as np
import pytest

import ssi_oracle as orc

pytestmark = pytest.mark.gpu


def test_readme_example(ssi, capsys):
    """README.md:46-80 with the reference's sizes: 10-20-20-2, N=100, M=3, T=10, c=1, itr=10."""
    rng = np.random.default_rng(0)
    X = rng.random((10, 100)).astype(np.float32)
    Y = rng.random((2, 100)).astype(np.float32)
    data = ssi.DataLoader(X, Y, batchsize=20, shuffle=True, rng=rng)
    m = ssi.Chain(ssi.Dense(10, 20, rng=rng), ssi.Dense(20, 20, rng=rng), ssi.Dense(20, 2, rng=rng))
    L1 = lambda mm, x, y: ssi.mse(mm(x), y)
    chn, lp, W_swa = ssi.subspace_inference(m, L1, data, ssi.ADAM(0.01), itr=10, T=10, c=1, M=3, seed=5)
    assert len(chn) == 10 and chn[0].shape == (682,) and lp.shape == (10,) and W_swa.shape == (682,)
    assert "Traing loss" in capsys.readouterr().out
    # every returned lp is the oracle density of the returned weight vector (likelihood only)
    for w, l in zip(chn, lp):
        pred = orc.forward(w, m.dims, m.acts, X)
        np.testing.assert_allclose(l, orc.gaussian_loglik(pred, Y, 1.0), rtol=1e-5)


def test_construction_then_inference_alias(ssi):
    rng = np.random.default_rng(1)
    X = rng.standard_normal((13, 400)).astype(np.float32)
    Y = rng.standard_normal((1, 400)).astype(np.float32)
    data = ssi.DataLoader(X, Y, batchsize=100)
    m = ssi.Chain(ssi.Dense(13, 50, ssi.relu, rng=rng), ssi.Dense(50, 1, rng=rng))
    L = lambda mm, x, y: ssi.mse(mm(x), y)
    W_swa, P = ssi.subspace_construction(m, L, data, ssi.Descent(0.05), T=5, c=1, M=5, print_freq=10)
    assert W_swa.shape == (751,) and P.shape == (751, 5)
    zt, lt = ssi.inference(m, data, W_swa, P, σ_z=0.1, σ_m=0.5, itr=20, M=5, alg=":mh", n_chains=8, seed=3)
    assert zt.shape == (5, 8, 20) and lt.shape == (8, 20)
    prob = orc.Problem(m.dims, m.acts, X, Y, W_swa, P)
    ref = orc.density(prob, zt[:, 3, 19], 0.5)
    np.testing.assert_allclose(lt[3, 19], ref, rtol=1e-5)
    with pytest.raises(ValueError):
        ssi.inference(m, data, W_swa, P, M=4)                # P has 5 columns


@pytest.mark.parametrize("dims,acts,M,B,Ng", [
    ((2, 200, 50, 50, 50, 1), (1, 1, 1, 1, 0), 20, 100, 100),    # the docs' network and grid (nn_example.md:112-118, 207)
    ((10, 20, 20, 2), (0, 0, 0), 3, 10, 37),                      # README network
    ((13, 50, 1), (1, 0), 5, 1, 5),                               # one trajectory: std is NaN, as in Julia
    ((4, 300, 3), (2, 3), 6, 130, 1000),                          # several groups of samples
])
def test_posterior_predictive_sweep_vs_oracle(ssi, engine, dims, acts, M, B, Ng):
    rng = np.random.default_rng(B + Ng)
    n = orc.n_params(dims)
    W_swa, P = orc.glorot_flat(rng, dims), (0.1 * rng.standard_normal((n, M))).astype(np.float32)
    Z = rng.standard_normal((M, B)).astype(np.float32)
    Xg = rng.uniform(-3, 3, (dims[0], Ng)).astype(np.float32)
    engine.set_model(dims, acts)
    engine.set_subspace(W_swa, P)                  # no data set: the sweep does not need it
    mean, std, traj = engine.predict(Z, Xg, return_trajectories=True)
    t_ref, m_ref, s_ref = orc.predictive_sweep(dims, acts, W_swa, P, Z, Xg)
    scale = np.abs(t_ref).max()
    np.testing.assert_allclose(traj, t_ref, rtol=1e-5, atol=1e-5 * scale)       # FP32 forward vs Float64 oracle
    np.testing.assert_allclose(mean, m_ref, rtol=1e-5, atol=1e-5 * scale)
    if B > 1:
        np.testing.assert_allclose(std, s_ref, rtol=1e-4, atol=1e-5 * scale)
    else:
        assert np.isnan(std).all()
    mean2, std2 = engine.predict(Z, Xg)            # without trajectories: same moments
    np.testing.assert_array_equal(mean2, mean)


def test_next_rows_golden(ssi, engine):
    """Gradient, MALA and the predictive sweep against the committed fixture tests/golden/next_rows.npz."""
    from pathlib import Path
    g = np.load(Path(__file__).parent / "golden" / "next_rows.npz")
    for name in ("readme", "uci"):
        dims, acts = tuple(int(d) for d in g[f"{name}_dims"]), tuple(int(a) for a in g[f"{name}_acts"])
        engine.set_model(dims, acts)
        engine.set_data(g[f"{name}_X"], g[f"{name}_Y"])
        engine.set_subspace(g[f"{name}_W_swa"], g[f"{name}_P"])
        sm, sp, sz = (float(v) for v in g[f"{name}_sig"])
        for k, mask in enumerate((1, 3, 7)):
            lp, grad = engine.logpost_grad(g[f"{name}_Z"], sm, sp, sz, mask=mask)
            np.testing.assert_allclose(lp, g[f"{name}_lp"][k], rtol=1e-5)
            gn = np.linalg.norm(g[f"{name}_grad"][k], axis=0)
            assert (np.abs(grad - g[f"{name}_grad"][k]).max(axis=0) <= 1e-4 * gn).all()
    prob = orc.make_problem("readme")
    engine.set_model(prob.dims, prob.acts)
    engine.set_data(prob.X, prob.Y)
    engine.set_subspace(prob.W_swa, prob.P)
    zt, lt, at = engine.mala_run(3, 8, int(g["mala_seed"]), sigma_z=float(g["mala_sigma_z"]), sigma_m=1.0)
    safe = np.abs(g["mala_margin"]) > 1e-3           # free-running comparison away from near ties
    assert safe[:, 1:].all(), "regenerate the fixture with a seed whose decisions are not near ties"
    np.testing.assert_array_equal(at, g["mala_accept"])
    np.testing.assert_allclose(np.transpose(zt, (1, 2, 0)), g["mala_z"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(lt, g["mala_lp"], rtol=1e-5)
    mean, std = engine.predict(g["pred_Z"], g["pred_Xg"])
    np.testing.assert_allclose(mean, g["pred_mean"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(std, g["pred_std"], rtol=1e-4, atol=1e-6)


# every option key with its default value; setting it leaves the context as it was
KEPT_OPTIONS = {"path": 0, "group": 0, "grad_group_gb": 0, "time_dominant": 0, "mala_rule": 0, "tc_precision": 1,
                "gram_fp64": 0, "gemm_simt": 0, "b1_simt": 0, "tc_pair": 1, "tc_nobasis": 0, "tc_nofuse": 0,
                "tc_simt_basis": 0, "tc_noorder": 0}
# A-B switches whose losing variants have been removed from the library
REMOVED_OPTIONS = ("eig_cluster", "formp_simt", "gram_chunk", "gemm_prec", "gemm_split_acc", "gemm_fwd_chunk", "gemm_chunk",
                   "gemm_tc_mask", "tc_k32", "tc_nokrev", "tc_alast", "bm_variant", "bm_nopack")


def test_option_keys(ssi, engine):
    for key, value in KEPT_OPTIONS.items():
        engine.set_option(key, value)
    for key in REMOVED_OPTIONS:
        with pytest.raises(ssi.SsiError) as e:
            engine.set_option(key, 0)
        assert e.value.code == -1 and "unknown option" in str(e.value), key
