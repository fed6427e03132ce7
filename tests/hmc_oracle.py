"""Float64 restatement of the device's fixed-length HMC (alg = :static_hmc, include/ssi.h ssi_hmc_run) for the tests.

Builds on oracle/ssi_oracle.py (density, gradient, the replayed Philox streams) and restates, with the device's roundings,
  * the leapfrog integrator: Float64 momentum and gradient, the position kept in Float32 and rounded once per drift;
  * the divergence rule: a drift that yields a non-finite position holds the trajectory at its start, and a divergent
    transition (that, or an energy error that is non-finite or > 1000, AdvancedHMC's threshold) is rejected;
  * the accept rule of RWMH on stream 1: accept iff -e < -dH;
  * the per-chain dual averaging of the step size (Hoffman & Gelman 2014, Alg. 5; Stan's / AdvancedHMC's constants).
Like the rest of the oracle it is test infrastructure: nothing in the product path imports it.
"""
from __future__ import annotations

import math

import numpy as np

import ssi_oracle as orc

DA_GAMMA, DA_T0, DA_KAPPA = 0.05, 10.0, 0.75
MAX_DELTA_H = 1000.0


def _drift(z, eps, inv_metric, p, round_f32: bool):
    zn = np.asarray(z, np.float64) + (eps * inv_metric) * p
    if not round_f32:
        return zn
    with np.errstate(over="ignore", invalid="ignore"):      # an overflow is a divergence, detected by the caller
        return zn.astype(np.float32)


def _kinetic(inv_metric, p) -> float:
    kin = 0.0
    with np.errstate(over="ignore", invalid="ignore"):      # a non-finite energy marks a divergence
        for v in (inv_metric * p) * p:                        # summed in index order, as the device does
            kin += float(v)
    return kin


def leapfrog(grad_fn, z, p, g, eps: float, L: int, inv_metric, round_f32: bool = True):
    """L leapfrog steps from (z, p) with the gradient g at z: half kick, L - 1 x (drift, gradient, full kick), drift,
    gradient, half kick.  grad_fn(z) -> (lp, g).  Returns (z', p', lp', g', divergent); once a drift yields a non-finite
    position the trajectory is held at its start z (divergent = True) and the gradient is not evaluated further."""
    inv_metric = np.asarray(inv_metric, np.float64)
    z0 = np.asarray(z)
    p = np.asarray(p, np.float64) + (0.5 * eps) * np.asarray(g, np.float64)
    zc, lp_c, g_c = z0, None, None
    for l in range(L):
        if l > 0:
            p = p + eps * g_c
        zn = _drift(zc, eps, inv_metric, p, round_f32)
        if not np.all(np.isfinite(zn)):
            return z0, p, None, None, True
        zc = zn
        lp_c, g_c = grad_fn(zc)
        g_c = np.asarray(g_c, np.float64)
    p = p + (0.5 * eps) * g_c
    return zc, p, lp_c, g_c, False


def hmc_transition(prob, z, g, lp, eps: float, L: int, inv_metric, normals, e: float, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0,
                   mask=orc.TERM_LL, grad_fn=None, round_f32: bool = True):
    """One transition from the state (z, lp, g): momentum p = normals / sqrt(inv_metric), L leapfrog steps, the energy
    error dH = H' - H with H = -lp + 1/2 sum inv_metric p^2, accept iff not divergent and -e < -dH.
    grad_fn(z) -> (lp, g) replaces the density of `prob` (closed-form targets).
    Returns (z', lp', g', dH, accepted, divergent, alpha): the state after the transition (the start when rejected) and
    alpha = min(1, exp(-dH)), 0 when divergent."""
    if grad_fn is None:
        grad_fn = lambda zz: orc.density_and_grad(prob, zz, sigma_m, sigma_p, sigma_z, mask)
    inv_metric = np.ones(len(z)) if inv_metric is None else np.asarray(inv_metric, np.float64)
    p0 = np.asarray(normals, np.float32).astype(np.float64) / np.sqrt(inv_metric)
    h0 = -lp + 0.5 * _kinetic(inv_metric, p0)
    zp, p, lpp, gp, divergent = leapfrog(grad_fn, z, p0, g, eps, L, inv_metric, round_f32)
    dH = math.nan
    if not divergent:
        dH = (-lpp + 0.5 * _kinetic(inv_metric, p)) + -h0
        divergent = not math.isfinite(dH) or dH > MAX_DELTA_H
    accepted = (not divergent) and (-e < -dH)
    alpha = 0.0 if divergent else (1.0 if dH <= 0 else math.exp(-dH))
    if accepted:
        return zp, lpp, gp, dH, True, divergent, alpha
    return z, lp, g, dH, False, divergent, alpha


def dual_averaging_init(eps0: float):
    """(log eps, log eps_bar, H_bar) before the first transition."""
    return (math.log(eps0), 0.0, 0.0)


def dual_averaging_update(state, m: int, alpha: float, eps0: float, delta: float):
    """Hoffman & Gelman 2014, Alg. 5, after transition m >= 1 with acceptance statistic alpha:
    H_bar <- (1 - 1/(m + t0)) H_bar + (delta - alpha)/(m + t0); log eps = mu - sqrt(m)/gamma H_bar;
    log eps_bar <- m^-kappa log eps + (1 - m^-kappa) log eps_bar, mu = log(10 eps0)."""
    _, log_eps_bar, hbar = state
    w = 1.0 / (m + DA_T0)
    hbar = (1.0 - w) * hbar + (delta - alpha) * w
    log_eps = math.log(10.0 * eps0) - math.sqrt(m) / DA_GAMMA * hbar
    mk = m ** -DA_KAPPA
    return (log_eps, mk * log_eps + (1.0 - mk) * log_eps_bar, hbar)


def step_size(state, t: int, n_adapts: int, eps0: float) -> float:
    """The step size transition t uses: eps0 when n_adapts == 0, exp(log eps) while t <= n_adapts, exp(log eps_bar) after."""
    if n_adapts == 0:
        return eps0
    return math.exp(state[0] if t <= n_adapts else state[1])


def hmc_chain(prob, n_steps: int, seed: int, chain: int, step_size0: float, n_leapfrog: int, n_adapts: int = 0,
              target_accept: float = 0.8, inv_metric=None, sigma_z=1.0, sigma_m=1.0, sigma_p=1.0, mask=orc.TERM_LL,
              z0=None, grad_fn=None, M: int | None = None):
    """One chain of ssi_hmc_run: sample 0 is z0 or sigma_z * eps(chain, 0) (MALA's init), step t >= 1 one hmc_transition
    with the normals of stream 0 and the Exp(1) variate of stream 1 at (chain, t), the step size adapted by dual averaging
    over transitions 1..n_adapts.
    Returns (z_trace (n_steps, M) f32, lp_trace, accept (1 / 0 / 2 divergent), step_size_trace (NaN at 0), adapt state)."""
    if grad_fn is None:
        grad_fn = lambda zz: orc.density_and_grad(prob, zz, sigma_m, sigma_p, sigma_z, mask)
    M = prob.M if prob is not None else (M if M is not None else len(z0))
    z = (orc.propose_f32(np.zeros(M, np.float32), sigma_z, orc.rng_normals(seed, chain, 0, M)) if z0 is None
         else np.asarray(z0, np.float32).copy())
    lp, g = grad_fn(z)
    z_tr = np.empty((n_steps, M), np.float32)
    lp_tr = np.empty(n_steps)
    acc = np.zeros(n_steps, np.uint8)
    eps_tr = np.full(n_steps, np.nan)
    z_tr[0], lp_tr[0], acc[0] = z, lp, 1
    state = dual_averaging_init(step_size0)
    for t in range(1, n_steps):
        eps = step_size(state, t, n_adapts, step_size0)
        z, lp, g, _, accepted, divergent, alpha = hmc_transition(
            prob, z, g, lp, eps, n_leapfrog, inv_metric, orc.rng_normals(seed, chain, t, M), orc.rng_exponential(seed, chain, t),
            grad_fn=grad_fn)
        if t <= n_adapts:
            state = dual_averaging_update(state, t, alpha, step_size0, target_accept)
        z_tr[t], lp_tr[t], acc[t], eps_tr[t] = z, lp, 1 if accepted else (2 if divergent else 0), eps
    return z_tr, lp_tr, acc, eps_tr, state
