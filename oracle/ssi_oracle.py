"""CPU oracle for the subspace log-posterior path (TEST INFRASTRUCTURE, NOT PRODUCT).

This file is a NumPy Float64 restatement of the algorithm that
efmanu/SubspaceInference.jl executes on its hot path.  It exists so that the CUDA
library can be checked against something; nothing in the product path may import
it.  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs are allowed to call into ``oracle/``.

PARITY UNPINNED.  The reference ships no tests, golden vectors or fixtures
(``test/runtests.jl`` is empty) and Julia is not installed in the build image, so
this restatement could not be checked against outputs of the reference itself.
All arithmetic on the path lives in un-vendored dependencies pinned in
``Manifest.toml``: Flux 0.11.2 (Chain/Dense/destructure), NNlib 0.7.23
(activations), Distributions 0.24.18 + PDMats 0.11.1 (MvNormal/logpdf),
AdvancedMH 0.6.2 + AbstractMCMC 3.2.1 (RWMH sampler), LowRankApprox 0.5.0 (psvd).
Their published algorithms are restated here, anchored on the reference's own call
sites (cited per function as ``src/<file>:<line>`` relative to the reference
root).  Independent closed forms (scipy multivariate normal, numpy SVD) pin the
restatement in ``tests/test_oracle.py``.

Conventions: all matrices are column-major in the reference; here X is (in0, N),
Y is (O, N), P is (n, M), Z is (M, B) as C-ordered NumPy arrays with the same
index meaning.  Everything is evaluated in Float64 like the reference (SURVEY Q7);
the inputs are the *same Float32 values* the device sees, upcast.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Callable, Sequence

import numpy as np

# activation codes shared with include/ssi.h
ACT_IDENTITY, ACT_RELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3

# prior mask bits shared with include/ssi.h
TERM_LL, TERM_PRIOR_W, TERM_PRIOR_Z = 1, 2, 4

_LOG_2PI = math.log(2.0 * math.pi)


# --------------------------------------------------------------------------------------
# Parameter layout: Flux.destructure / restructure          (src/libs.jl:55-57, :19-22)
# --------------------------------------------------------------------------------------
def n_params(dims: Sequence[int]) -> int:
    """Length of the flat parameter vector of Chain(Dense(d0,d1),...,Dense(d_{L-1},d_L))."""
    return int(sum(dims[l] * dims[l + 1] + dims[l + 1] for l in range(len(dims) - 1)))


def layer_offsets(dims: Sequence[int]):
    """[(w_off, b_off, in, out)] per layer.

    Flux.destructure concatenates, per Dense layer, ``vec(W_l)`` (W_l is out x in,
    column-major: element (o, i) at ``o + i*out``) followed by ``b_l``
    (src/libs.jl:56-57; same order as extract_params, src/libs.jl:19-22).
    """
    offs, p = [], 0
    for l in range(len(dims) - 1):
        din, dout = int(dims[l]), int(dims[l + 1])
        offs.append((p, p + din * dout, din, dout))
        p += din * dout + dout
    return offs


def restructure(w: np.ndarray, dims: Sequence[int]):
    """Flat vector -> [(W_l (out,in), b_l (out,))], no dtype cast (SURVEY Q7)."""
    layers = []
    for w_off, b_off, din, dout in layer_offsets(dims):
        W = w[w_off:w_off + din * dout].reshape(din, dout).T  # column-major (out,in)
        b = w[b_off:b_off + dout]
        layers.append((W, b))
    return layers


def flatten_params(layers) -> np.ndarray:
    """[(W_l, b_l)] -> flat vector, the inverse of :func:`restructure` (src/libs.jl:19-22)."""
    parts = []
    for W, b in layers:
        parts.append(np.asarray(W).T.reshape(-1))  # vec() of column-major (out,in)
        parts.append(np.asarray(b).reshape(-1))
    return np.concatenate(parts)


def _activate(h: np.ndarray, act: int) -> np.ndarray:
    if act == ACT_IDENTITY:
        return h
    if act == ACT_RELU:
        return np.maximum(h, 0.0)
    if act == ACT_TANH:
        return np.tanh(h)
    if act == ACT_SIGMOID:
        return 1.0 / (1.0 + np.exp(-h))
    raise ValueError(f"unknown activation code {act}")


# --------------------------------------------------------------------------------------
# density(z)                                               (src/space_inference.jl:90-95)
# --------------------------------------------------------------------------------------
def project(W_swa: np.ndarray, P: np.ndarray, z: np.ndarray) -> np.ndarray:
    """``new_W = W_swa + P*z`` (src/space_inference.jl:91), Float64."""
    return np.asarray(W_swa, np.float64) + np.asarray(P, np.float64) @ np.asarray(z, np.float64)


def forward(w: np.ndarray, dims, acts, X: np.ndarray) -> np.ndarray:
    """Dense-chain forward on the full dataset: ``H_l = act_l.(W_l*H_{l-1} .+ b_l)``
    (Flux Dense, called at src/space_inference.jl:94 through src/libs.jl:55-57)."""
    h = np.asarray(X, np.float64)
    for (W, b), act in zip(restructure(np.asarray(w, np.float64), dims), acts):
        h = _activate(W @ h + b[:, None], act)
    return h


def gaussian_loglik(pred: np.ndarray, Y: np.ndarray, sigma: float) -> float:
    """``logpdf(MvNormal(vec(pred), sigma), vec(Y))`` for a scalar-std isotropic normal
    (Distributions/PDMats ScalMat; src/space_inference.jl:94):
    ``-k/2 log(2pi) - k log(sigma) - ||y - pred||^2 / (2 sigma^2)``, k = O*N."""
    r = np.asarray(Y, np.float64) - pred
    k = r.size
    return -0.5 * k * _LOG_2PI - k * math.log(sigma) - float(np.sum(r * r)) / (2.0 * sigma * sigma)


def log_prior_w(w: np.ndarray, sigma_p: float) -> float:
    """The weight-prior term written at src/space_inference.jl:95 —
    ``logpdf(MvNormal(zeros(n), sigma_p), new_W)``.  It is DEAD CODE in the
    reference (line-leading ``+`` after a complete ``return``; SURVEY Q1), so it is
    only added when TERM_PRIOR_W is set in the mask."""
    n = w.size
    return -0.5 * n * _LOG_2PI - n * math.log(sigma_p) - float(np.dot(w, w)) / (2.0 * sigma_p * sigma_p)


def log_prior_z(z: np.ndarray, sigma_z: float) -> float:
    """Optional isotropic prior on the subspace coordinates (north_star's sigma_z
    prior; not present in the reference density, where sigma_z is only the proposal
    std, src/space_inference.jl:113)."""
    z = np.asarray(z, np.float64)
    m = z.size
    return -0.5 * m * _LOG_2PI - m * math.log(sigma_z) - float(np.dot(z, z)) / (2.0 * sigma_z * sigma_z)


@dataclass
class Problem:
    """Everything ``density`` closes over (src/space_inference.jl:86-90)."""
    dims: Sequence[int]
    acts: Sequence[int]
    X: np.ndarray          # (in0, N)   split_data, src/libs.jl:75-77
    Y: np.ndarray          # (O, N)
    W_swa: np.ndarray      # (n,)
    P: np.ndarray          # (n, M)

    @property
    def M(self) -> int:
        return int(self.P.shape[1])

    @property
    def N(self) -> int:
        return int(self.X.shape[1])


def density_terms(prob: Problem, z, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0):
    """(loglik, log_prior_w, log_prior_z) for one subspace point."""
    w = project(prob.W_swa, prob.P, z)
    pred = forward(w, prob.dims, prob.acts, prob.X)
    return (gaussian_loglik(pred, prob.Y, sigma_m),
            log_prior_w(w, sigma_p),
            log_prior_z(z, sigma_z))


def density(prob: Problem, z, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0, mask=TERM_LL) -> float:
    """The reference's ``density(z)`` as executed: mask=TERM_LL (likelihood only, Q1)."""
    ll, pw, pz = density_terms(prob, z, sigma_m, sigma_p, sigma_z)
    return ((ll if mask & TERM_LL else 0.0) + (pw if mask & TERM_PRIOR_W else 0.0)
            + (pz if mask & TERM_PRIOR_Z else 0.0))


def _act_deriv_from_output(h: np.ndarray, act: int) -> np.ndarray:
    """act'(pre) written in terms of the output h = act(pre) (NNlib: identity, relu, tanh, sigmoid)."""
    if act == 1:
        return (h > 0).astype(np.float64)
    if act == 2:
        return 1.0 - h * h
    if act == 3:
        return h * (1.0 - h)
    return np.ones_like(h)


def _forward_all(w: np.ndarray, dims, acts, X: np.ndarray):
    """(layers, [H_0 = X, H_1, ..., H_L]): the forward pass with every activation kept, Float64."""
    layers = restructure(np.asarray(w, np.float64), dims)
    hs = [np.asarray(X, np.float64)]
    for (W, b), act in zip(layers, acts):
        hs.append(_activate(W @ hs[-1] + b[:, None], act))
    return layers, hs


def _reverse_gw(layers, hs, dims, acts, delta: np.ndarray) -> np.ndarray:
    """Reverse pass through the Dense chain from the output delta dL/d(pre_L) (O, N): dL/dw in the flat layout,
    ``gW_l = delta_l H_{l-1}'``, ``gb_l = rowsum(delta_l)``, ``delta_{l-1} = (W_l' delta_l) * act_{l-1}'(H_{l-1})``."""
    gw = np.zeros(n_params(dims))
    offs = layer_offsets(dims)
    for l in range(len(layers) - 1, -1, -1):
        W, _ = layers[l]
        w0, b0, _, dout = offs[l]
        gw[w0:b0] = (delta @ hs[l].T).reshape(-1, order="F")       # vec(W_l) is column-major (o + i*out)
        gw[b0:b0 + dout] = delta.sum(axis=1)
        if l > 0:
            delta = (W.T @ delta) * _act_deriv_from_output(hs[l], acts[l - 1])
    return gw


def density_and_grad(prob: Problem, z, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0, mask=TERM_LL):
    """``l_pi_grad(theta) = (density(theta), gradient(density, theta))`` (src/space_inference.jl:107), the closure of
    the :mala/:hmc/:nuts branches.  The reference differentiates ``density`` with ForwardDiff/ReverseDiff/Zygote
    (src/libs.jl:23-34); the derivative is restated analytically here (reverse mode through the Dense chain, then
    ``P' grad_W``) and pinned against torch autograd and central differences in tests/test_oracle.py."""
    z = np.asarray(z, np.float64)
    w = project(prob.W_swa, prob.P, z)
    layers, hs = _forward_all(w, prob.dims, prob.acts, prob.X)
    lp = density(prob, z, sigma_m, sigma_p, sigma_z, mask)
    gw = np.zeros_like(w)
    if mask & TERM_LL:
        delta = -(hs[-1] - np.asarray(prob.Y, np.float64)) / (sigma_m * sigma_m) * _act_deriv_from_output(hs[-1], prob.acts[-1])
        gw = _reverse_gw(layers, hs, prob.dims, prob.acts, delta)
    P = np.asarray(prob.P, np.float64)
    g = P.T @ gw
    if mask & TERM_PRIOR_W:
        g = g - P.T @ w / (sigma_p * sigma_p)
    if mask & TERM_PRIOR_Z:
        g = g - z / (sigma_z * sigma_z)
    return lp, g


def logpost_batch(prob: Problem, Z, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0, mask=TERM_LL):
    """Batched restatement: one ``density`` call per column of Z (M, B).
    Returns (lp (B,), terms (3, B))."""
    Z = np.asarray(Z, np.float64)
    B = Z.shape[1]
    terms = np.empty((3, B))
    for b in range(B):
        terms[:, b] = density_terms(prob, Z[:, b], sigma_m, sigma_p, sigma_z)
    sel = np.array([bool(mask & TERM_LL), bool(mask & TERM_PRIOR_W), bool(mask & TERM_PRIOR_Z)], float)
    return sel @ terms, terms


# --------------------------------------------------------------------------------------
# Counter-based RNG (build-defined; the reference uses Julia's unseeded GLOBAL_RNG,
# src/space_inference.jl:116, which is not reproducible even against itself)
# --------------------------------------------------------------------------------------
_PHILOX_M0, _PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
_PHILOX_W0, _PHILOX_W1 = 0x9E3779B9, 0xBB67AE85
STREAM_NORMAL, STREAM_ACCEPT = 0, 1


def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon et al. 2011).  counter: (...,4) uint32, key: (2,) uint32.
    Vectorised over leading dims; returns (...,4) uint32."""
    c = np.array(counter, dtype=np.uint64) & 0xFFFFFFFF
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    c0, c1, c2, c3 = c[..., 0], c[..., 1], c[..., 2], c[..., 3]
    for _ in range(10):
        p0 = _PHILOX_M0 * c0
        p1 = _PHILOX_M1 * c2
        hi0, lo0 = p0 >> 32, p0 & 0xFFFFFFFF
        hi1, lo1 = p1 >> 32, p1 & 0xFFFFFFFF
        c0, c1, c2, c3 = (hi1 ^ c1 ^ k0) & 0xFFFFFFFF, lo1, (hi0 ^ c3 ^ k1) & 0xFFFFFFFF, lo0
        k0 = (k0 + _PHILOX_W0) & 0xFFFFFFFF
        k1 = (k1 + _PHILOX_W1) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def _seed_key(seed: int):
    return np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)


def rng_normals(seed: int, chain: int, step: int, M: int) -> np.ndarray:
    """The M standard normals of (chain, step), Float32.

    counter = (chain, step, j, STREAM_NORMAL); block j gives 4 uint32 (x0..x3) ->
    u = (x + 0.5) * 2^-32 in Float64; Box-Muller in Float64:
    r0 = sqrt(-2 ln u0), (n0, n1) = r0 * (cos, sin)(2 pi u1); r1 = sqrt(-2 ln u2),
    (n2, n3) = r1 * (cos, sin)(2 pi u3); each rounded once to Float32.
    """
    nblk = (M + 3) // 4
    ctr = np.zeros((nblk, 4), dtype=np.uint64)
    ctr[:, 0] = chain & 0xFFFFFFFF
    ctr[:, 1] = step & 0xFFFFFFFF
    ctr[:, 2] = np.arange(nblk)
    ctr[:, 3] = STREAM_NORMAL
    x = philox4x32_10(ctr, _seed_key(seed)).astype(np.float64)
    u = (x + 0.5) * 2.0 ** -32
    out = np.empty((nblk, 4))
    for a in (0, 2):
        r = np.sqrt(-2.0 * np.log(u[:, a]))
        ang = 2.0 * np.pi * u[:, a + 1]
        out[:, a] = r * np.cos(ang)
        out[:, a + 1] = r * np.sin(ang)
    return out.reshape(-1)[:M].astype(np.float32)


def rng_exponential(seed: int, chain: int, step: int) -> float:
    """Exp(1) variate for the accept test of (chain, step): e = -ln(u),
    u = (x0 + 0.5) * 2^-32 from counter (chain, step, 0, STREAM_ACCEPT).  Float64."""
    ctr = np.array([chain & 0xFFFFFFFF, step & 0xFFFFFFFF, 0, STREAM_ACCEPT], dtype=np.uint64)
    x0 = float(philox4x32_10(ctr, _seed_key(seed))[0])
    return -math.log((x0 + 0.5) * 2.0 ** -32)


# --------------------------------------------------------------------------------------
# Random-walk Metropolis-Hastings           (src/space_inference.jl:108-116,125; AdvancedMH)
# --------------------------------------------------------------------------------------
def propose_f32(z: np.ndarray, sigma_z: float, eps: np.ndarray) -> np.ndarray:
    """z' = z + sigma_z * eps as one fused multiply-add per element, Float32 result
    (the device keeps the chain state in Float32)."""
    return (z.astype(np.float64) + np.float64(np.float32(sigma_z)) * eps.astype(np.float64)).astype(np.float32)


def rwmh_chain(prob: Problem, n_steps: int, seed: int, chain: int, sigma_z=1.0, sigma_m=1.0,
               sigma_p=1.0, mask=TERM_LL, z0=None,
               density_fn: Callable[[np.ndarray], float] | None = None):
    """One chain of AdvancedMH's RWMH as the reference drives it
    (``sample(DensityModel(density), RWMH(MvNormal(zeros(M), sigma_z)), itr)``,
    src/space_inference.jl:111-116):

    * sample 1 is a draw from the proposal, z0 = sigma_z*eps_0, and it counts (Q5);
    * step t: z' = z + sigma_z*eps_t, log_alpha = lp(z') - lp(z) (symmetric proposal),
      accept iff ``-randexp() < log_alpha`` (Q6);
    * lp of the current state is cached in the transition.

    Returns (z_trace (n_steps, M) f32, lp_trace (n_steps,) f64, accept (n_steps,) u8,
    margin (n_steps,) f64 = log_alpha + e, the distance of each decision from a tie).
    """
    M = prob.M
    if density_fn is None:
        density_fn = lambda zz: density(prob, zz, sigma_m, sigma_p, sigma_z, mask)
    z_tr = np.empty((n_steps, M), np.float32)
    lp_tr = np.empty(n_steps)
    acc = np.zeros(n_steps, np.uint8)
    margin = np.full(n_steps, np.inf)
    if z0 is None:
        z = propose_f32(np.zeros(M, np.float32), sigma_z, rng_normals(seed, chain, 0, M))
    else:
        z = np.asarray(z0, np.float32).copy()
    lp = density_fn(z)
    z_tr[0], lp_tr[0], acc[0] = z, lp, 1
    for t in range(1, n_steps):
        zp = propose_f32(z, sigma_z, rng_normals(seed, chain, t, M))
        lpp = density_fn(zp)
        e = rng_exponential(seed, chain, t)
        log_alpha = lpp - lp
        margin[t] = log_alpha + e
        if -e < log_alpha:
            z, lp, acc[t] = zp, lpp, 1
        z_tr[t], lp_tr[t] = z, lp
    return z_tr, lp_tr, acc, margin


def mala_propose_f32(z: np.ndarray, grad: np.ndarray, sigma_z: float, eps: np.ndarray) -> np.ndarray:
    """z' = (z + float32(sigma_z^2/2 * grad)) + sigma_z*eps with the device's roundings: the drift is formed in Float64
    and rounded once, added in Float32, and the noise enters through one fused multiply-add."""
    drift = (0.5 * sigma_z * sigma_z * np.asarray(grad, np.float64)).astype(np.float32)
    base = (np.asarray(z, np.float32) + drift).astype(np.float32)
    return propose_f32(base, sigma_z, eps)


def mala_log_alpha(z, zp, lp, lpp, g, gp, sigma_z: float, rule: int = 0) -> float:
    """lp' - lp + log q(z | z') - log q(z' | z),  q(a | b) = N(a; b + (sigma_z^2/2) grad lp(b), sigma_z^2 I)  (rule 0).
    rule 1 evaluates both densities with the NEGATED gradient, q(a | b) = N(a - b; -(sigma_z^2/2) grad lp(b), sigma_z^2 I):
    AdvancedMH's MALA step is remembered to build its densities from ``proposal(-gradient)``; the pinned 0.6.2 source is
    not in /root/reference to decide, so the library offers both (option ``mala_rule``) and this oracle restates both."""
    z, zp = np.asarray(z, np.float64), np.asarray(zp, np.float64)
    h = 0.5 * sigma_z * sigma_z * (-1.0 if rule else 1.0)
    fwd = float(np.sum((zp - z - h * np.asarray(g, np.float64)) ** 2))
    rev = float(np.sum((z - zp - h * np.asarray(gp, np.float64)) ** 2))
    return lpp - lp + (fwd - rev) / (2.0 * sigma_z * sigma_z)


def mala_chain(prob: Problem, n_steps: int, seed: int, chain: int, sigma_z=1.0, sigma_m=1.0, sigma_p=1.0,
               mask=TERM_LL, z0=None, rule: int = 0):
    """One chain of ``sample(DensityModel(density), MALA(x -> MvNormal((sigma_z^2 / 2) .* x, sigma_z)), itr;
    init_params=rand(MvNormal(zeros(M), sigma_z)))`` (src/space_inference.jl:117-120): sample 1 is the initial point
    z0 = sigma_z*eps_0, step t draws the increment from N((sigma_z^2/2) grad lp(z), sigma_z^2 I) and accepts iff
    ``-randexp() < log_alpha`` with the proposal-density ratio of the Metropolis-adjusted Langevin algorithm as
    AdvancedMH documents it (AdvancedMH 0.6.2 is not vendored: PARITY UNPINNED; the restatement is pinned by the
    detailed-balance test in tests/test_oracle.py).  Same stream as rwmh_chain.
    Returns (z_trace (n_steps, M) f32, lp_trace, accept, margin)."""
    M = prob.M
    f = lambda zz: density_and_grad(prob, zz, sigma_m, sigma_p, sigma_z, mask)
    z_tr = np.empty((n_steps, M), np.float32)
    lp_tr = np.empty(n_steps)
    acc = np.zeros(n_steps, np.uint8)
    margin = np.full(n_steps, np.inf)
    z = (propose_f32(np.zeros(M, np.float32), sigma_z, rng_normals(seed, chain, 0, M)) if z0 is None
         else np.asarray(z0, np.float32).copy())
    lp, g = f(z)
    z_tr[0], lp_tr[0], acc[0] = z, lp, 1
    for t in range(1, n_steps):
        zp = mala_propose_f32(z, g, sigma_z, rng_normals(seed, chain, t, M))
        lpp, gp = f(zp)
        e = rng_exponential(seed, chain, t)
        la = mala_log_alpha(z, zp, lp, lpp, g, gp, sigma_z, rule)
        margin[t] = la + e
        if -e < la:
            z, lp, g, acc[t] = zp, lpp, gp, 1
        z_tr[t], lp_tr[t] = z, lp
    return z_tr, lp_tr, acc, margin


def predictive_sweep(dims, acts, W_swa: np.ndarray, P: np.ndarray, Z: np.ndarray, Xg: np.ndarray):
    """docs/src/nn_example.md:207-216: ``for i in 1:itr; m1 = re(all_chain[i]); trajectories[:, i] = m1(inp)'``, then
    src/plotting.jl:8-9: ``mean(trajectories, dims=2)``, ``std(trajectories, dims=2)`` (Julia's std is the corrected
    estimator; one trajectory gives NaN).  Returns (trajectories (O, Ng, B), mean (O, Ng), std (O, Ng))."""
    Z = np.asarray(Z, np.float64)
    if Z.ndim == 1:
        Z = Z[:, None]
    Xg = np.asarray(Xg, np.float64)
    traj = np.stack([forward(project(W_swa, P, Z[:, b]), dims, acts, Xg) for b in range(Z.shape[1])], axis=2)
    with np.errstate(invalid="ignore", divide="ignore"):
        sd = traj.std(axis=2, ddof=1) if Z.shape[1] > 1 else np.full(traj.shape[:2], np.nan)
    return traj, traj.mean(axis=2), sd


def samples_to_weights(prob: Problem, z_trace: np.ndarray) -> np.ndarray:
    """``map(z -> W_swa + P*z.params, chm)`` (src/space_inference.jl:125): (n_steps, n)."""
    return np.stack([project(prob.W_swa, prob.P, z) for z in z_trace])


# --------------------------------------------------------------------------------------
# Mini-batch training step                                (src/subspace_construction.jl:39-43)
# --------------------------------------------------------------------------------------
def mse_loss_and_grad(w: np.ndarray, dims, acts, X: np.ndarray, Y: np.ndarray):
    """``training_loss = Flux.Losses.mse(m(x), y)`` and its gradient for the Dense chain with flat parameters ``w``:
    loss = mean((pred - Y)^2) over all O*nb entries, gw = dL/dw in the flat layout [vec(W_1); b_1; ...].  Float64."""
    layers, hs = _forward_all(w, dims, acts, X)
    r = hs[-1] - np.asarray(Y, np.float64)
    delta = (2.0 / r.size) * r * _act_deriv_from_output(hs[-1], acts[-1])
    return float(np.mean(r * r)), _reverse_gw(layers, hs, dims, acts, delta)


def adam_step(w, g, m, v, t: int, eta: float, b1: float = 0.9, b2: float = 0.999):
    """Step t (1-based) of Flux 0.11's ADAM, in Float64: ``m = b1 m + (1-b1) g``, ``v = b2 v + (1-b2) g^2``,
    ``w -= eta m/(1-b1^t) / (sqrt(v/(1-b2^t)) + 1e-8)`` (Flux keeps b^t as a running product starting at b).
    Returns (w, m, v)."""
    g = np.asarray(g, np.float64)
    m = b1 * np.asarray(m, np.float64) + (1.0 - b1) * g
    v = b2 * np.asarray(v, np.float64) + (1.0 - b2) * g * g
    w = np.asarray(w, np.float64) - m / (1.0 - b1 ** t) / (np.sqrt(v / (1.0 - b2 ** t)) + 1e-8) * eta
    return w, m, v


# --------------------------------------------------------------------------------------
# Subspace construction                       (src/subspace_construction.jl:31,44-52,61-65)
# --------------------------------------------------------------------------------------
def swa_push(W_swa: np.ndarray, W: np.ndarray, n_scalar: float):
    """One snapshot: ``W_swa = (n.*W_swa + W)./(n+1)`` then ``W_dev = W - W_swa``
    against the UPDATED mean (src/subspace_construction.jl:46-47,51; Q2, Q4).
    ``n_scalar`` is ``i/c`` with i the EPOCH index."""
    W = np.asarray(W, np.float64)
    W_swa = (n_scalar * W_swa + W) / (n_scalar + 1.0)
    return W_swa, W - W_swa


def construct_from_snapshots(snapshots, n_scalars, M: int, route: str = "svd"):
    """The moment recurrence + factorisation of ``subspace_construction`` given the
    sequence of post-update weight snapshots (the SGD step that produces them,
    src/subspace_construction.jl:39-43, is outside the path).

    W_swa starts at ZEROS (src/subspace_construction.jl:31, Q2); every deviation
    column is kept (Q3); ``P = U[:,1:M]*Diagonal(s[1:M])`` (:63-65).  ``psvd`` is
    restated by an exact SVD (route="svd") or by the Gram route the device uses
    (route="gram": eigen-decomposition of A'A, P = A V_M).  Columns are equal up to
    sign.  Returns (W_swa (n,), P (n,M), s (K,), A (n,K)).
    """
    snapshots = [np.asarray(s, np.float64) for s in snapshots]
    n = snapshots[0].size
    W_swa = np.zeros(n)
    cols = []
    for W, ns in zip(snapshots, n_scalars):
        W_swa, dev = swa_push(W_swa, W, float(ns))
        cols.append(dev)
    A = np.stack(cols, axis=1)                                 # reshape(A, all_len, :)  (:61)
    if A.shape[1] < M or min(A.shape) < M:
        raise ValueError("rank of deviation matrix smaller than M")  # U[:,1:M] BoundsError in Julia
    if route == "svd":
        U, s, _ = np.linalg.svd(A, full_matrices=False)
        P = U[:, :M] * s[:M]
    elif route == "gram":
        G = A.T @ A
        lam, V = np.linalg.eigh(G)
        order = np.argsort(lam)[::-1]
        lam, V = lam[order], V[:, order]
        s = np.sqrt(np.maximum(lam, 0.0))
        P = A @ V[:, :M]                                       # = U_M S_M
    else:
        raise ValueError(route)
    return W_swa, P, s, A


def align_signs(P: np.ndarray, P_ref: np.ndarray) -> np.ndarray:
    """Flip columns of P to match the sign convention of P_ref (SVD sign ambiguity)."""
    sgn = np.sign(np.sum(P * P_ref, axis=0))
    sgn[sgn == 0] = 1.0
    return P * sgn


# --------------------------------------------------------------------------------------
# Synthetic configurations (BASELINE.json configs; SURVEY 8d)
# --------------------------------------------------------------------------------------
def glorot_flat(rng: np.random.Generator, dims) -> np.ndarray:
    """Flux's default Dense init (glorot_uniform weights, zero bias), flattened."""
    layers = []
    for l in range(len(dims) - 1):
        din, dout = dims[l], dims[l + 1]
        lim = math.sqrt(6.0 / (din + dout))
        layers.append((rng.uniform(-lim, lim, size=(dout, din)), np.zeros(dout)))
    return flatten_params(layers).astype(np.float32)


def synthetic_subspace(rng: np.random.Generator, n: int, M: int, scales) -> np.ndarray:
    """P (n, M) = orthonormal columns times the given singular values, Float32."""
    Q, _ = np.linalg.qr(rng.standard_normal((n, M)))
    return (Q * np.asarray(scales)[None, :]).astype(np.float32)


def make_problem(name: str, seed: int | None = None, N: int | None = None) -> Problem:
    """Synthetic inputs of the BASELINE configs, Float32-valued.

    "readme": 10-20-20-2 identity, N=100, M=3            (README.md:52-79)
    "uci"   : 13-50-1 relu, N=10k, M=5
    "wide"  : 784-1024-1024-10 relu, N=60k, M=20
    """
    if name == "readme":
        dims, acts, M, n_def, seed_def = (10, 20, 20, 2), (0, 0, 0), 3, 100, 1234
    elif name == "uci":
        dims, acts, M, n_def, seed_def = (13, 50, 1), (1, 0), 5, 10000, 2024
    elif name == "wide":
        dims, acts, M, n_def, seed_def = (784, 1024, 1024, 10), (1, 1, 0), 20, 60000, 31337
    else:
        raise ValueError(name)
    N = n_def if N is None else N
    rng = np.random.default_rng(seed_def if seed is None else seed)
    n = n_params(dims)
    W_swa = glorot_flat(rng, dims)
    if name == "readme":
        X = rng.random((dims[0], N), dtype=np.float32)
        Y = rng.random((dims[-1], N), dtype=np.float32)
        scales = 10.0 ** (-np.arange(M) / M)
    elif name == "uci":
        X = rng.standard_normal((dims[0], N)).astype(np.float32)
        w_true = glorot_flat(rng, dims)
        Y = (forward(w_true, dims, acts, X) + 0.1 * rng.standard_normal((dims[-1], N))).astype(np.float32)
        W_swa = (w_true + 0.01 * rng.standard_normal(n)).astype(np.float32)
        scales = np.array([1.0, 0.5, 0.25, 0.12, 0.06])
    else:
        X = rng.random((dims[0], N), dtype=np.float32)
        lab = rng.integers(0, dims[-1], size=N)
        Y = -np.ones((dims[-1], N), np.float32)
        Y[lab, np.arange(N)] = 1.0
        scales = 0.5 ** np.arange(1, M + 1)
    P = synthetic_subspace(rng, n, M, scales)
    return Problem(dims, acts, X, Y, W_swa, P)


# --------------------------------------------------------------------------------------
# Non-linear subspace operator (auto-encoder decoder)   (src/space_inference.jl:238-251)
# --------------------------------------------------------------------------------------
def decoder_forward(theta: np.ndarray, dims, acts, z: np.ndarray) -> np.ndarray:
    """``decoder(z)`` for a Flux Chain of Dense layers dims[0] -> ... -> dims[-1] with parameters ``theta`` in
    Flux.destructure order (the decoder auto_encoder_subspace trains, src/subspace_construction.jl:125-141)."""
    return forward(np.asarray(theta, np.float64), dims, acts, np.asarray(z, np.float64).reshape(-1, 1)).reshape(-1)


def density_decoder(prob: Problem, dec_theta, dec_dims, dec_acts, z, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0, mask=TERM_LL) -> float:
    """``density(z)`` of auto_inference, Chain branch (src/space_inference.jl:246-251): ``new_W = W_swa + decoder(z)``, then
    the same likelihood as sub_inference; the weight-prior line is dead code there too (a line-leading ``+``, :250-251),
    so the default mask is the likelihood alone.  prob.P is not used."""
    z = np.asarray(z, np.float64)
    w = np.asarray(prob.W_swa, np.float64) + decoder_forward(dec_theta, dec_dims, dec_acts, z)
    pred = forward(w, prob.dims, prob.acts, np.asarray(prob.X, np.float64))
    v = 0.0
    if mask & TERM_LL:
        v += gaussian_loglik(pred, np.asarray(prob.Y, np.float64), sigma_m)
    if mask & TERM_PRIOR_W:
        v += log_prior_w(w, sigma_p)
    if mask & TERM_PRIOR_Z:
        v += log_prior_z(z, sigma_z)
    return v
