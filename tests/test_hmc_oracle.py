"""CPU checks of the HMC restatement (tests/hmc_oracle.py) that the device sampler is held to, and of the keyword checks of
alg=:static_hmc, which run before any device context exists."""
import math

import numpy as np
import pytest

import hmc_oracle as hmc
import ssi_oracle as orc


def _gaussian(mean, cov):
    prec = np.linalg.inv(cov)

    def grad_fn(z):
        d = np.asarray(z, np.float64) - mean
        return -0.5 * float(d @ prec @ d), -(prec @ d)
    return grad_fn


def test_leapfrog_is_reversible_in_float64():
    """Without the Float32 rounding of the position the integrator is exactly time-reversible: L steps, negate p, L steps
    return to the start."""
    mean, cov = np.array([0.3, -1.0, 2.0]), np.array([[1.0, 0.4, 0.1], [0.4, 0.5, 0.0], [0.1, 0.0, 2.0]])
    f = _gaussian(mean, cov)
    rng = np.random.default_rng(0)
    inv_metric = np.array([1.0, 0.5, 2.0])
    for _ in range(5):
        z0, p0 = rng.standard_normal(3), rng.standard_normal(3)
        _, g0 = f(z0)
        z1, p1, _, g1, div = hmc.leapfrog(f, z0, p0, g0, 0.1, 17, inv_metric, round_f32=False)
        assert not div
        z2, p2, _, _, div = hmc.leapfrog(f, z1, -p1, g1, 0.1, 17, inv_metric, round_f32=False)
        assert not div
        np.testing.assert_allclose(z2, z0, rtol=0, atol=1e-12)
        np.testing.assert_allclose(-p2, p0, rtol=0, atol=1e-12)


def test_chains_reproduce_a_correlated_gaussian():
    """Many independent chains of hmc_chain (adapted step size, then fixed) on a 2-D correlated Gaussian: the final states'
    mean and covariance are those of the target within 4 standard errors."""
    mean = np.array([1.0, -2.0])
    cov = np.array([[1.0, 0.8], [0.8, 1.5]])
    f = _gaussian(mean, cov)
    n, steps = 300, 40
    Z = np.empty((n, 2))
    for c in range(n):
        zt, _, acc, eps, _ = hmc.hmc_chain(None, steps, 4242, c, 0.5, 4, n_adapts=20, grad_fn=f, M=2)
        assert np.isnan(eps[0]) and np.all(eps[1:] > 0) and acc[0] == 1
        assert np.all(eps[21:] == eps[21])                # fixed after warm-up
        Z[c] = zt[-1]
    se_mean = np.sqrt(np.diag(cov) / n)
    assert np.all(np.abs(Z.mean(0) - mean) < 4 * se_mean), (Z.mean(0), mean)
    S = np.cov(Z.T)
    se_cov = np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / n)
    assert np.all(np.abs(S - cov) < 4 * se_cov), (S, cov)


def test_dual_averaging_by_hand():
    """Three updates of Alg. 5 evaluated by hand, and alpha == delta keeps log eps at mu = log(10 eps0)."""
    eps0, delta = 0.2, 0.8
    mu = math.log(2.0)
    s = hmc.dual_averaging_init(eps0)
    assert s == (math.log(0.2), 0.0, 0.0)
    s1 = hmc.dual_averaging_update(s, 1, 0.5, eps0, delta)
    hb1 = 0.3 / 11
    le1 = mu - 1.0 / 0.05 * hb1
    assert s1 == pytest.approx((le1, le1, hb1), rel=1e-14)
    s2 = hmc.dual_averaging_update(s1, 2, 1.0, eps0, delta)
    hb2 = (1 - 1 / 12) * hb1 + (0.8 - 1.0) / 12
    le2 = mu - math.sqrt(2) / 0.05 * hb2
    w2 = 2 ** -0.75
    assert s2 == pytest.approx((le2, w2 * le2 + (1 - w2) * le1, hb2), rel=1e-14)
    s3 = hmc.dual_averaging_update(s2, 3, 0.0, eps0, delta)
    hb3 = (1 - 1 / 13) * hb2 + 0.8 / 13
    le3 = mu - math.sqrt(3) / 0.05 * hb3
    w3 = 3 ** -0.75
    assert s3 == pytest.approx((le3, w3 * le3 + (1 - w3) * s2[1], hb3), rel=1e-14)
    s = hmc.dual_averaging_init(eps0)
    for m in range(1, 30):
        s = hmc.dual_averaging_update(s, m, delta, eps0, delta)
        assert s[0] == pytest.approx(mu, abs=1e-15) and s[2] == 0.0
    assert hmc.step_size(s, 5, 0, eps0) == eps0
    assert hmc.step_size(s, 5, 10, eps0) == math.exp(s[0])
    assert hmc.step_size(s, 11, 10, eps0) == math.exp(s[1])


def test_divergent_transition_is_rejected_and_held():
    """A trajectory that overflows the Float32 position is divergent: rejected, the state unchanged, alpha = 0."""
    f = _gaussian(np.zeros(2), np.eye(2) * 1e-6)
    z = np.array([1e3, -1e3], np.float32)
    lp, g = f(z)
    out = hmc.hmc_transition(None, z, g, lp, 10.0, 5, None, np.array([0.1, 0.2], np.float32), 0.5, grad_fn=f)
    zn, lpn, _, _, accepted, divergent, alpha = out
    assert divergent and not accepted and alpha == 0.0
    np.testing.assert_array_equal(zn, z)
    assert lpn == lp


def test_static_hmc_keywords_are_checked_before_a_context_exists(ssi):
    rng = np.random.default_rng(1)
    m = ssi.Chain(ssi.Dense(3, 4, ssi.relu, rng=rng), ssi.Dense(4, 1, rng=rng))
    dl = ssi.DataLoader(rng.random((3, 5)).astype(np.float32), rng.random((1, 5)).astype(np.float32), batchsize=5)
    w = ssi.extract_params(m)
    P = np.zeros((w.shape[0], 2), np.float32)
    for bad in (dict(n_leapfrog=0), dict(step_size=-1), dict(step_size=float("nan")), dict(target_accept=1.0),
                dict(n_adapts=-1), dict(inv_metric=[1.0, 0.0]), dict(inv_metric=[1.0])):
        with pytest.raises(ValueError):
            ssi.sub_inference(m, dl, w, P, M=2, alg=":static_hmc", **bad)
    dec = ssi.Chain(ssi.Dense(2, w.shape[0], rng=rng))
    with pytest.raises(ValueError):
        ssi.auto_inference(m, dl, dec, w, M=2, alg=":static_hmc", n_leapfrog=0)
    for alg in (":hmc", ":nuts", ":advi"):
        with pytest.raises(NotImplementedError):
            ssi.sub_inference(m, dl, w, P, M=2, alg=alg)
    with pytest.raises(NotImplementedError):
        ssi.auto_inference(m, dl, dec, w, M=2)               # the reference's default :hmc
