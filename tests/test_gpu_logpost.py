"""Parity of the CUDA log-posterior path against the Float64 oracle and the golden fixtures.
Tolerance: 1e-5 relative on every per-sample log-prob (north_star), FP32 device arithmetic."""
from pathlib import Path

import numpy as np
import pytest

import ssi_oracle as orc
from conftest import stable_seed

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).parent / "golden"
RTOL = 1e-5


def _setup(engine, prob):
    engine.set_model(prob.dims, prob.acts)
    engine.set_data(prob.X, prob.Y)
    engine.set_subspace(prob.W_swa, prob.P)


def _basis_ok(prob):
    M = prob.P.shape[1]
    return len(prob.dims) == 3 and prob.dims[-1] <= 2 and (M <= 8 or M in (10, 12, 16, 20))


def _paths_for(ssi, prob):
    paths = [ssi.PATH_LAYERED]
    if orc.n_params(prob.dims) < 12000:
        paths.append(ssi.PATH_FUSED)
    if _basis_ok(prob):
        paths.append(ssi.PATH_BASIS)
    return paths


@pytest.mark.parametrize("name", ["readme", "uci_small", "wide_small"])
def test_golden_all_terms(ssi, engine, name):
    g = np.load(GOLD / f"logpost_{name}.npz")
    prob = orc.Problem(tuple(int(d) for d in g["dims"]), tuple(int(a) for a in g["acts"]), g["X"], g["Y"], g["W_swa"], g["P"])
    _setup(engine, prob)
    sm, sp, sz = float(g["sigma_m"]), float(g["sigma_p"]), float(g["sigma_z"])
    for path in _paths_for(ssi, prob) + [ssi.PATH_AUTO]:
        engine.set_option("path", path)
        lp, terms = engine.logpost(g["Z"], sm, sp, sz, mask=7, return_terms=True)
        np.testing.assert_allclose(terms, g["terms"], rtol=RTOL, err_msg=f"path {path}")
        np.testing.assert_allclose(lp, g["terms"].sum(axis=0), rtol=RTOL)
        # reference as executed: likelihood only (Q1); sigma_p must not matter
        lp_ll = engine.logpost(g["Z"], sm, 123.0, sz)
        np.testing.assert_allclose(lp_ll, g["terms"][0], rtol=RTOL)
        assert engine.stats().last_path == (path if path != ssi.PATH_AUTO else engine.stats().last_path)


@pytest.mark.parametrize("dims,acts,N,M,B", [
    ((10, 20, 20, 2), (0, 0, 0), 100, 3, 1),          # README, one z at a time like the reference
    ((13, 50, 1), (1, 0), 777, 5, 37),                # ragged N, odd B
    ((5, 7, 3), (2, 3), 130, 2, 9),                   # tanh / sigmoid, widths not multiples of 4
    ((3, 1), (0,), 1, 1, 3),                          # single layer, single datapoint
    ((33, 65, 17, 9, 4), (1, 2, 1, 0), 257, 6, 5),    # deeper chain
    ((13, 50, 1), (1, 0), 10000, 5, 130),             # C2 shape: BASIS path, samples not a multiple of the warp block
    ((4, 9, 2), (2, 1), 65, 7, 70),                   # BASIS: tanh hidden, relu output, O = 2, ST = 4
    ((6, 31, 1), (3, 0), 200, 12, 33),                # BASIS: sigmoid hidden, M = 12
    ((3, 5, 2), (0, 2), 64, 20, 3),                   # BASIS: identity hidden, M = 20 (ST = 2), tanh output
    ((8, 16, 1), (1, 0), 1, 1, 1),                    # BASIS: one datapoint, one sample, M = 1
])
def test_random_shapes_vs_oracle(ssi, engine, dims, acts, N, M, B):
    rng = np.random.default_rng(stable_seed(dims, N, M, B))
    n = orc.n_params(dims)
    prob = orc.Problem(dims, acts, rng.standard_normal((dims[0], N)).astype(np.float32),
                       rng.standard_normal((dims[-1], N)).astype(np.float32), orc.glorot_flat(rng, dims),
                       (0.3 * rng.standard_normal((n, M))).astype(np.float32))
    Z = rng.standard_normal((M, B)).astype(np.float32)
    _setup(engine, prob)
    ref, ref_terms = orc.logpost_batch(prob, Z, 0.7, 1.3, 0.9, mask=7)
    for path in (ssi.PATH_FUSED, ssi.PATH_LAYERED) + ((ssi.PATH_BASIS, ssi.PATH_AUTO) if _basis_ok(prob) else ()):
        engine.set_option("path", path)
        lp, terms = engine.logpost(Z, 0.7, 1.3, 0.9, mask=7, return_terms=True)
        if path == ssi.PATH_AUTO:
            assert engine.stats().last_path == ssi.PATH_BASIS
        np.testing.assert_allclose(terms, ref_terms, rtol=RTOL, err_msg=f"path {path}")
        np.testing.assert_allclose(lp, ref, rtol=RTOL)


def test_batch_invariance_bitwise(ssi, engine):
    """A sample's lp must not depend on which other samples share the call (fixed-order
    reductions): this is what makes chain sharding over GPUs reproduce the 1-GPU trace."""
    prob = orc.make_problem("uci", N=3000)
    _setup(engine, prob)
    Z = (0.1 * np.random.default_rng(0).standard_normal((prob.M, 64))).astype(np.float32)
    for path in (ssi.PATH_FUSED, ssi.PATH_LAYERED, ssi.PATH_BASIS):
        engine.set_option("path", path)
        full = engine.logpost(Z, 0.1)
        part = np.concatenate([engine.logpost(Z[:, :5], 0.1), engine.logpost(Z[:, 5:40], 0.1), engine.logpost(Z[:, 40:], 0.1)])
        np.testing.assert_array_equal(full, part)


def test_uci_full_size_properties(ssi, engine):
    """Full C2 size (N=10k, B=4096): oracle on a sample of columns + permutation invariance."""
    prob = orc.make_problem("uci")
    _setup(engine, prob)
    rng = np.random.default_rng(1)
    Z = (0.1 * rng.standard_normal((prob.M, 4096))).astype(np.float32)
    lp = engine.logpost(Z, 0.1)
    assert engine.stats().last_path == ssi.PATH_BASIS          # AUTO: one hidden layer, O = 1, M = 5
    idx = rng.choice(4096, 12, replace=False)
    ref, _ = orc.logpost_batch(prob, Z[:, idx], 0.1)
    np.testing.assert_allclose(lp[idx], ref, rtol=RTOL)
    perm = rng.permutation(prob.N)
    engine.set_data(prob.X[:, perm], prob.Y[:, perm])
    lp2 = engine.logpost(Z[:, :256], 0.1)
    np.testing.assert_allclose(lp2, lp[:256], rtol=2e-6)
    assert engine.stats().last_units == 256 * prob.N
    # the exact-FP32 FUSED path agrees on every sample of the big batch
    engine.set_data(prob.X, prob.Y)
    engine.set_option("path", ssi.PATH_FUSED)
    np.testing.assert_allclose(engine.logpost(Z, 0.1), lp, rtol=2e-6)


def test_project_matches_oracle(ssi, engine):
    prob = orc.make_problem("readme")
    _setup(engine, prob)
    Z = np.random.default_rng(2).standard_normal((3, 11)).astype(np.float32)
    W = engine.project(Z)
    ref = np.stack([orc.project(prob.W_swa, prob.P, Z[:, b]) for b in range(11)], axis=1)
    np.testing.assert_allclose(W, ref, rtol=1e-6, atol=1e-6)


def test_error_behaviour(ssi):
    eng = ssi.Engine(0)
    try:
        with pytest.raises(ssi.SsiError) as ei:
            eng._check(eng._lib.ssi_logpost_batch(eng._h, None, 0, 1.0, 1.0, 1.0, 1, None, None) or
                       eng._lib.ssi_set_data(eng._h, None, None, 5))
        assert ei.value.code in (-1, -3)
        eng.set_model((4, 3, 2), (1, 0))
        with pytest.raises(ssi.SsiError) as ei:
            eng.set_subspace(np.zeros(5, np.float32), np.zeros((5, 2), np.float32))   # wrong n
        assert ei.value.code == -1
        prob_n = orc.n_params((4, 3, 2))
        eng.set_subspace(np.zeros(prob_n, np.float32), np.zeros((prob_n, 2), np.float32))
        eng.M = 2
        with pytest.raises(ssi.SsiError) as ei:
            eng.logpost(np.zeros((2, 1), np.float32))                                 # data not set
        assert ei.value.code == -3
        eng.set_data(np.zeros((4, 6), np.float32), np.zeros((2, 6), np.float32))
        with pytest.raises(ssi.SsiError):
            eng.logpost(np.zeros((2, 1), np.float32), sigma_m=0.0)
        with pytest.raises(ssi.SsiError):
            eng.logpost(np.zeros((2, 1), np.float32), mask=0)
        assert eng.logpost(np.zeros((2, 0), np.float32)).shape == (0,)                # empty batch
        # all-zero weights: pred = 0, lp = closed form of |Y|^2 = 0
        lp = eng.logpost(np.zeros((2, 3), np.float32), sigma_m=2.0)
        np.testing.assert_allclose(lp, -0.5 * 12 * np.log(2 * np.pi) - 12 * np.log(2.0), rtol=1e-12)
    finally:
        eng.close()


@pytest.mark.parametrize("dims,acts,N,M,B", [
    ((10, 20, 20, 2), (0, 0, 0), 100, 3, 5),          # README network
    ((13, 50, 1), (1, 0), 3000, 5, 70),               # UCI shape, more than one group of samples (fast forward-mode path)
    ((6, 31, 1), (2, 3), 200, 8, 37),                 # fast path: tanh hidden, sigmoid output, M = 8
    ((4, 9, 1), (3, 1), 65, 1, 5),                    # fast path: sigmoid hidden, relu output, M = 1
    ((5, 7, 3), (2, 3), 130, 2, 9),                   # tanh / sigmoid, ragged widths
    ((3, 1), (0,), 1, 1, 3),                          # single layer, single datapoint
    ((33, 65, 17, 9, 4), (1, 2, 1, 0), 257, 6, 4),    # deeper chain
    ((96, 128, 128, 10), (1, 1, 0), 300, 20, 3),      # wide-ish chain: several tiles per GEMM, split projection
    ((96, 256, 192, 8), (1, 2, 0), 3000, 12, 3),      # big enough for the tensor-core GEMM: ragged tiles, 3 accumulation chunks
    ((100, 132, 68, 8), (2, 1, 0), 1500, 6, 4),       # tensor-core GEMM with ragged rows (132 = 128 + 4), columns and k tails
])
def test_gradient_vs_oracle(ssi, engine, dims, acts, N, M, B):
    """l_pi_grad (src/space_inference.jl:107) batched: value within 1e-5 relative, gradient within 1e-4 of its norm
    (FP32 reverse pass vs the Float64 oracle), for every combination of terms."""
    rng = np.random.default_rng(stable_seed(dims, N, M, B, "g"))
    n = orc.n_params(dims)
    prob = orc.Problem(dims, acts, rng.standard_normal((dims[0], N)).astype(np.float32),
                       rng.standard_normal((dims[-1], N)).astype(np.float32), orc.glorot_flat(rng, dims),
                       (0.3 * rng.standard_normal((n, M))).astype(np.float32))
    Z = (0.5 * rng.standard_normal((M, B))).astype(np.float32)
    _setup(engine, prob)
    for mask in (1, 7, 2, 4):
        lp, grad = engine.logpost_grad(Z, 0.7, 1.3, 0.9, mask=mask)
        for b in range(B):
            lp_ref, g_ref = orc.density_and_grad(prob, Z[:, b].astype(np.float64), 0.7, 1.3, 0.9, mask)
            assert abs(lp[b] - lp_ref) <= RTOL * abs(lp_ref)
            np.testing.assert_allclose(grad[:, b], g_ref, rtol=0, atol=1e-4 * max(np.linalg.norm(g_ref), 1e-12), err_msg=f"mask {mask} sample {b}")
    fast = len(dims) == 3 and dims[-1] == 1 and M <= 8
    assert engine.stats().last_path == (ssi.PATH_BASIS if fast else ssi.PATH_LAYERED)
    if fast:        # the generic reverse-mode path must agree with the forward-mode fast path
        lp_f, g_f = engine.logpost_grad(Z, 0.7, 1.3, 0.9, mask=1)
        engine.set_option("path", ssi.PATH_LAYERED)
        lp_g, g_g = engine.logpost_grad(Z, 0.7, 1.3, 0.9, mask=1)
        assert engine.stats().last_path == ssi.PATH_LAYERED
        engine.set_option("path", ssi.PATH_AUTO)
        np.testing.assert_allclose(lp_f, lp_g, rtol=2e-6)
        np.testing.assert_allclose(g_f, g_g, rtol=0, atol=2e-4 * np.abs(g_g).max())
    if dims in ((96, 256, 192, 8), (100, 132, 68, 8)):
        # the large contractions ran on the tensor cores (ssi_gemm_tc.cu) and agree with the SIMT kernel
        assert engine.stats().gemm_tc_launches > 0
        lp_t, g_t = engine.logpost_grad(Z, 0.7, 1.3, 0.9, mask=1)
        before = engine.stats().gemm_tc_launches
        engine.set_option("gemm_simt", 1)
        lp_s, g_s = engine.logpost_grad(Z, 0.7, 1.3, 0.9, mask=1)
        assert engine.stats().gemm_tc_launches == before
        engine.set_option("gemm_simt", 0)
        np.testing.assert_allclose(lp_t, lp_s, rtol=2e-6)
        np.testing.assert_allclose(g_t, g_s, rtol=0, atol=5e-5 * np.linalg.norm(g_s, axis=0).max())
    # a sample's gradient does not depend on the rest of the batch
    lp_a, g_a = engine.logpost_grad(Z[:, :2], 0.7, 1.3, 0.9, mask=7)
    lp_b, g_b = engine.logpost_grad(Z, 0.7, 1.3, 0.9, mask=7)
    np.testing.assert_array_equal(g_a, g_b[:, :2])
    np.testing.assert_array_equal(lp_a, lp_b[:2])


@pytest.mark.parametrize("dims,acts,N,M,B", [
    ((13, 50, 1), (1, 0), 10000, 5, 700),      # C2 shape: K = 16, Hp = 64, three blocks of 256 samples (ragged)
    ((13, 50, 1), (1, 0), 333, 5, 1),          # a single sample, ragged datapoint tail
    ((6, 31, 1), (3, 2), 200, 12, 33),         # Hp = 32, sigmoid hidden (padded units must cancel), tanh output
    ((4, 64, 1), (2, 0), 65, 20, 300),         # K = 32 (M + 1 = 21), H = 64 exactly
    ((5, 17, 1), (0, 1), 1, 31, 5),            # M + 1 = 32, one datapoint, identity hidden, relu output
    ((7, 40, 1), (1, 0), 4001, 1, 2500),       # M + 1 = 2: one packed K slab; 10 blocks of samples (several parts per CTA)
    ((9, 64, 1), (1, 1), 777, 7, 300),         # M + 1 = 8: three packed slabs, all 48 columns used; relu output
    ((3, 20, 1), (2, 3), 150, 4, 40),          # two packed slabs, Hp = 32, tanh hidden, sigmoid output
    ((11, 44, 1), (1, 0), 501, 9, 130),        # Hp = 48 (TMEM chunks 32 + 16), M + 1 = 10: three-way split as six MMAs, K = 16
    ((8, 37, 1), (3, 0), 77, 2, 9),            # Hp = 40 (chunks 32 + 8), odd number of datapoints: half-empty last tile
])
def test_basis_path_kernels_vs_oracle(ssi, engine, dims, acts, N, M, B):
    """BASIS path, tensor-core kernel (samples along the MMA M dimension) and CUDA-core kernel: both within 1e-5 of the
    Float64 oracle; the tensor-core result of a sample is bitwise independent of the batch it arrives in."""
    rng = np.random.default_rng(stable_seed(dims, N, M, B, "bm"))
    n = orc.n_params(dims)
    prob = orc.Problem(dims, acts, rng.standard_normal((dims[0], N)).astype(np.float32),
                       rng.standard_normal((dims[-1], N)).astype(np.float32), orc.glorot_flat(rng, dims),
                       (0.3 * rng.standard_normal((n, M))).astype(np.float32))
    Z = (0.7 * rng.standard_normal((M, B))).astype(np.float32)
    _setup(engine, prob)
    ref, _ = orc.logpost_batch(prob, Z, 0.7)
    out = {}
    for simt in (0, 1):
        engine.set_option("b1_simt", simt)
        try:
            out[simt] = engine.logpost(Z, 0.7)
        except ssi.SsiError as e:          # the CUDA-core kernel does not take every shape the tensor-core kernel takes
            assert simt == 1 and e.code == -5
            continue
        assert engine.stats().last_path == (ssi.PATH_BASIS if simt == 0 else engine.stats().last_path)
        np.testing.assert_allclose(out[simt], ref, rtol=RTOL, err_msg=f"b1_simt={simt}")
    engine.set_option("b1_simt", 0)
    k = min(B, 3)
    np.testing.assert_array_equal(engine.logpost(Z[:, B - k:], 0.7), out[0][B - k:])
