"""Host-side mirror of the reference's public functions for the accelerated path.

Same names, argument meaning, defaults and error behaviour as
  subspace_construction   src/subspace_construction.jl:26-67
  subspace_inference      src/space_inference.jl:33-54
  sub_inference           src/space_inference.jl:82-125   (alias `inference`, README.md:153-154)
Everything numeric goes through the C ABI (include/ssi.h); there is no CPU fallback.
Keyword arguments that do not exist in the reference (n_chains, seed, prior_mask, device,
return_z, engine) default to the reference's behaviour: one chain, likelihood-only density
(the weight-prior line is dead code in the reference, src/space_inference.jl:94-95).
"""
from __future__ import annotations

import numpy as np

from ._lib import TERM_LL
from .engine import Engine
from .flux import ADAM, Chain, DataLoader, Descent, extract_params, load_params, mse, split_data, train_step

_RWMH_ALIASES = ("rwmh", "mh")
_DEVICE_ALGS = (*_RWMH_ALIASES, "mala", "static_hmc")


def _sym(s) -> str:
    return str(s).lstrip(":")


def _check_alg(a: str):
    if a not in _DEVICE_ALGS:
        if a in ("advi", "hmc", "nuts"):
            # the reference's :hmc is NUTS with Stan's windowed adaptation (AdvancedHMC); the device's fixed-length sampler
            # is a different algorithm and answers to :static_hmc only
            raise NotImplementedError(f"{a} is not available on the device path (Engine.logpost_grad is its l_pi_grad; "
                                      "alg=:static_hmc is the device's fixed-length HMC)")
        raise ValueError(f"{a} is not available")                         # src/space_inference.jl:162, :316


def _hmc_options(itr: int, M: int, n_leapfrog, step_size, n_adapts, target_accept, inv_metric) -> dict:
    """Validated keywords of alg=:static_hmc (ValueError before any context exists)."""
    if isinstance(n_leapfrog, bool) or int(n_leapfrog) != n_leapfrog or n_leapfrog < 1:
        raise ValueError(f"n_leapfrog must be an integer >= 1 (got {n_leapfrog!r})")
    step_size = float(step_size)
    if not (np.isfinite(step_size) and step_size > 0):
        raise ValueError(f"step_size must be positive and finite (got {step_size!r})")
    n_adapts = itr // 2 if n_adapts is None else n_adapts
    if isinstance(n_adapts, bool) or int(n_adapts) != n_adapts or n_adapts < 0:
        raise ValueError(f"n_adapts must be an integer >= 0 (got {n_adapts!r})")
    target_accept = float(target_accept)
    if not 0.0 < target_accept < 1.0:
        raise ValueError(f"target_accept must be in (0, 1) (got {target_accept!r})")
    if inv_metric is not None:
        inv_metric = np.asarray(inv_metric, dtype=np.float64).reshape(-1)
        if inv_metric.shape[0] != M or not (np.all(np.isfinite(inv_metric)) and np.all(inv_metric > 0)):
            raise ValueError(f"inv_metric must hold M={M} positive finite values")
    return dict(n_leapfrog=int(n_leapfrog), step_size=step_size, n_adapts=int(n_adapts), target_accept=target_accept,
                inv_metric=inv_metric)


def _sample(eng: Engine, a: str, n_chains: int, itr: int, seed: int, σ_z, σ_m, σ_p, prior_mask, chain_offset, hmc):
    """(z_trace, lp_trace) of the device sampler `a`; warm-up transitions of :static_hmc stay in the trace, as AdvancedHMC's
    `sample` keeps them by default."""
    if a == "static_hmc":
        zt, lt, _, _ = eng.hmc_run(n_chains, itr, seed, sigma_z=σ_z, sigma_m=σ_m, sigma_p=σ_p, mask=prior_mask,
                                   chain_offset=chain_offset, want_accept=False, want_step_size=False, **hmc)
        return zt, lt
    zt, lt, _ = eng.mh_run(n_chains, itr, seed, sigma_z=σ_z, sigma_m=σ_m, sigma_p=σ_p, mask=prior_mask,
                           chain_offset=chain_offset, want_accept=False, kind="mala" if a == "mala" else "rwmh")
    return zt, lt


def shard_rows(n: int, rank: int, world: int):
    """[begin, end) of the flat-parameter rows rank owns in a row-sharded construction (SURVEY 8e); multiples of 32 so
    that every shard keeps the aligned fast paths."""
    per = -(-n // world)
    per = -(-per // 32) * 32
    return min(n, rank * per), min(n, (rank + 1) * per)


def subspace_construction(model, cost, data, opt, *, T: int = 10, c: int = 1, M: int = 3, print_freq: int = 1,
                          engine: Engine | None = None, device: int = 0, install: bool = False,
                          shard: tuple[int, int] | None = None, all_reduce=None, device_train: bool = False):
    """(W_swa, P) from SGD snapshots.  The per-mini-batch training step is host plumbing
    (src/subspace_construction.jl:39-43); the moment recurrence, deviation matrix, Gram,
    eigen-solve and P = U_M S_M run on the device (:44-52, :61-65).

    shard=(rank, world) with all_reduce=fn: row-sharded construction over `world` GPUs.  Every rank trains the same
    replica and pushes rows shard_rows(n, rank, world) of each snapshot; the K x K Gram is summed across ranks by
    `all_reduce` (the only collective) and the function returns the rank's ROWS of W_swa and P.

    device_train=True keeps the training step itself on the device (SURVEY 8(f)-3): forward, backward and the
    Descent/ADAM update run in the library and every snapshot goes device-to-device into the SWA recurrence.  It is
    defined for cost = mse(model(x), y) (the cost of README.md:86 and the docs' regression examples); the first
    mini-batch's device loss is checked against `cost` and any other cost raises.  `model` receives the trained
    weights at the end, as it would from the host loop."""
    if not isinstance(model, Chain):
        raise TypeError("Error: model_re function is not available for this model")   # src/libs.jl:59
    own = engine is None
    eng = engine or Engine(device)
    try:
        n = int(extract_params(model).shape[0])
        n_batches = len(data)
        K_max = max(1, (T // c) * n_batches)
        r0, r1 = shard_rows(n, *shard) if shard is not None else (0, n)
        if shard is not None and (all_reduce is None or install):
            raise ValueError("a sharded construction needs all_reduce and cannot install its (partial) subspace")
        eng.swa_begin(r1 - r0, K_max)
        training_loss = 0.0
        if device_train:
            if shard is not None:
                raise ValueError("device_train pushes whole snapshots: it cannot be combined with a row shard")
            training_loss = _train_on_device(eng, model, cost, data, opt, T, c, print_freq)
            T = 0                                              # the host loop below has nothing left to do
        for i in range(1, T + 1):
            for x, y in data:
                training_loss = train_step(model, cost, opt, x, y)
                if i % c == 0:
                    eng.swa_push(extract_params(model)[r0:r1], i / c)   # n = i/c (:46), epoch index (Q2)
            if i % print_freq == 0 or i == T:
                print("Traing loss: ", training_loss, " Epoch: ", i)    # (sic) :56-58
        if install:
            eng.set_model(model.dims, model.acts)
        if shard is not None:
            W_swa, P, _ = eng.swa_finish_sharded(M, all_reduce)
        else:
            W_swa, P, _ = eng.swa_finish(M, install=install)
        return W_swa, P
    finally:
        if own:
            eng.close()


def _train_on_device(eng: Engine, model, cost, data, opt, T: int, c: int, print_freq: int) -> float:
    """The epoch loop of src/subspace_construction.jl:37-58 with the mini-batch step and the snapshot push on the device."""
    if isinstance(opt, ADAM):
        kind, eta, beta = "adam", opt.eta, opt.beta
        if opt.state:
            raise ValueError("device_train needs a fresh optimiser (ADAM state lives on the device)")
    elif isinstance(opt, Descent):
        kind, eta, beta = "descent", opt.eta, (0.9, 0.999)
    else:
        raise TypeError("device_train supports Descent and ADAM")
    X, Y = split_data(data)
    eng.set_model(model.dims, model.acts)
    eng.set_data(X, Y)
    eng.train_begin(extract_params(model), kind, eta, beta)
    training_loss, checked = 0.0, False
    try:
        for i in range(1, T + 1):
            for sel in data.index_batches():
                if not checked:                                # the device step assumes cost = mse(model(x), y)
                    import torch
                    with torch.no_grad():
                        host = float(cost(model, torch.as_tensor(np.asarray(X[..., sel], np.float32)),
                                          torch.as_tensor(np.asarray(Y[..., sel], np.float32))))
                contiguous = len(sel) > 0 and int(sel[-1]) - int(sel[0]) == len(sel) - 1 and bool(np.all(np.diff(sel) == 1))
                training_loss = eng.train_step((int(sel[0]), len(sel)) if contiguous else sel)
                if not checked:
                    if abs(training_loss - host) > 1e-4 * max(1.0, abs(host)):
                        raise ValueError("device_train: cost(model, x, y) is not mse(model(x), y) "
                                         f"(host {host:.6g}, device {training_loss:.6g})")
                    checked = True
                if i % c == 0:
                    eng.train_snapshot(i / c)                  # n = i/c (:46), epoch index (Q2)
            if i % print_freq == 0 or i == T:
                print("Traing loss: ", training_loss, " Epoch: ", i)    # (sic) :56-58
        load_params(model, eng.train_weights())
    finally:
        eng.train_end()
    return training_loss


def sub_inference(in_model, data, W_swa, P, *, σ_z: float = 1.0, σ_m: float = 1.0, σ_p: float = 1.0, itr: int = 100,
                  M: int = 3, alg="rwmh", backend="forwarddiff",
                  n_chains: int = 1, seed: int = 0, chain_offset: int = 0, prior_mask: int = TERM_LL,
                  engine: Engine | None = None, device: int = 0, return_z: bool = False,
                  n_leapfrog: int = 10, step_size: float = 0.1, n_adapts: int | None = None, target_accept: float = 0.8,
                  inv_metric=None):
    """RWMH in the subspace.  Returns (chn, lp): with n_chains == 1 (the reference) `chn` is a
    list of `itr` weight vectors W_swa + P z and `lp` the `itr` log-probabilities
    (src/space_inference.jl:125).  With n_chains > 1 `chn` is the (M, n_chains, itr) array of
    subspace samples (materialising itr x n_chains weight vectors is what the device path
    avoids; use Engine.project on the samples you need) and lp is (n_chains, itr).

    alg=:static_hmc runs fixed-length HMC on the device (n_leapfrog leapfrog steps per transition, initial step size
    step_size adapted per chain by dual averaging over the first n_adapts transitions (default itr // 2) towards
    target_accept, diagonal inverse metric inv_metric (default ones)); the warm-up samples stay in the returned trace."""
    a = _sym(alg)
    _check_alg(a)
    hmc = _hmc_options(itr, M, n_leapfrog, step_size, n_adapts, target_accept, inv_metric) if a == "static_hmc" else None
    if not isinstance(in_model, Chain):
        raise TypeError("Error: density function is not avaliable for this model")   # :103
    P = np.asarray(P)
    if P.ndim != 2 or P.shape[1] != M:
        raise ValueError(f"DimensionMismatch: P has {P.shape[-1]} columns but M = {M}")   # P*z fails in Julia (:91)
    X, Y = split_data(data)
    own = engine is None
    eng = engine or Engine(device)
    try:
        eng.set_model(in_model.dims, in_model.acts)
        eng.set_data(X, Y)
        eng.set_subspace(W_swa, P)
        zt, lt = _sample(eng, a, n_chains, itr, seed, σ_z, σ_m, σ_p, prior_mask, chain_offset, hmc)
        if n_chains == 1 and not return_z:
            W = eng.project(zt[:, 0, :])                                  # map(z -> W_swa + P*z, chm)
            return [W[:, t].copy() for t in range(itr)], lt[0].copy()
        return zt, lt
    finally:
        if own:
            eng.close()


inference = sub_inference


def auto_encoder_subspace(model, cost, data, opt, encoder, decoder, *, T: int = 10, c: int = 1, M: int = 3, print_freq: int = 1,
                          engine: Engine | None = None, device: int = 0, rng: np.random.Generator | None = None):
    """(W_swa, decoder): the SWA moments and deviation matrix as in subspace_construction (on the device), then an
    auto-encoder Chain(encoder, decoder) trained on the deviation columns (src/subspace_construction.jl:93-143).  Like the
    SGD step, the auto-encoder training is host plumbing outside the accelerated path (`Flux.train!`, one epoch, ADAM(),
    DataLoader(re_weight, batchsize = 5, shuffle = true), :134-141) and is delegated to torch autograd; its loss is
    `Flux.mse(sae(X), X)` -- the `+ sum(sqnorm, autops)` line is a separate statement that never contributes (:130-131).
    M is accepted and unused, as in the reference (the decoder's input width is the subspace dimension)."""
    if not isinstance(model, Chain) or not isinstance(encoder, Chain) or not isinstance(decoder, Chain):
        raise TypeError("Error: model_re function is not available for this model")
    own = engine is None
    eng = engine or Engine(device)
    try:
        n = int(extract_params(model).shape[0])
        if encoder.dims[0] != n or decoder.dims[-1] != n or encoder.dims[-1] != decoder.dims[0]:
            raise ValueError("DimensionMismatch: encoder must map n -> M and decoder M -> n")
        eng.swa_begin(n, max(1, (T // c) * len(data)))
        training_loss = 0.0
        for i in range(1, T + 1):
            for x, y in data:
                training_loss = train_step(model, cost, opt, x, y)
                if i % c == 0:
                    eng.swa_push(extract_params(model), i / c)
            if i % print_freq == 0 or i == T:
                print("Traing loss: ", training_loss, " Epoch: ", i)
        W_swa = eng.swa_mean()
        re_weight = eng.swa_deviations()                                   # reshape(A, all_len, :)   (:119)
        sae = Chain(*encoder.layers, *decoder.layers)
        autoloss = lambda mm, X: mse(mm(X), X)
        aopt = ADAM()                                                       # opt = ADAM()  (:134)
        wdata = DataLoader(re_weight, re_weight, batchsize=5, shuffle=True, rng=rng)
        for X, _ in wdata:
            train_step(sae, lambda mm, a, b: autoloss(mm, a), aopt, X, X)
        return W_swa, decoder
    finally:
        if own:
            eng.close()


def auto_inference(m, data, decoder, W_swa, *, σ_z: float = 1.0, σ_m: float = 1.0, σ_p: float = 1.0, itr: int = 100, M: int = 3,
                   alg="hmc", backend="forwarddiff", n_chains: int = 1, seed: int = 0, chain_offset: int = 0,
                   prior_mask: int = TERM_LL, engine: Engine | None = None, device: int = 0, return_z: bool = False,
                   n_leapfrog: int = 10, step_size: float = 0.1, n_adapts: int | None = None, target_accept: float = 0.8,
                   inv_metric=None):
    """Sampling with a decoder in place of P: density(z) evaluates the model at W_swa + decoder(z)
    (src/space_inference.jl:238-318).  :rwmh, :mala and :static_hmc run on the device as in sub_inference; the reference's
    default here is :hmc (NUTS with windowed adaptation), whose host-side sampler is not part of the device path
    (Engine.logpost_grad is its l_pi_grad)."""
    a = _sym(alg)
    _check_alg(a)
    hmc = _hmc_options(itr, M, n_leapfrog, step_size, n_adapts, target_accept, inv_metric) if a == "static_hmc" else None
    if not isinstance(m, Chain) or not isinstance(decoder, Chain):
        raise TypeError("Error: density function is not avaliable for this model")
    if decoder.dims[0] != M:
        raise ValueError(f"DimensionMismatch: the decoder takes {decoder.dims[0]} inputs but M = {M}")
    X, Y = split_data(data)
    own = engine is None
    eng = engine or Engine(device)
    try:
        eng.set_model(m.dims, m.acts)
        eng.set_data(X, Y)
        eng.set_decoder(W_swa, decoder.dims, decoder.acts, extract_params(decoder))
        zt, lt = _sample(eng, a, n_chains, itr, seed, σ_z, σ_m, σ_p, prior_mask, chain_offset, hmc)
        if n_chains == 1 and not return_z:
            W = eng.project(zt[:, 0, :])                                  # map(z -> W_swa + decoder(z.params), chm)  (:277)
            return [W[:, t].copy() for t in range(itr)], lt[0].copy()
        return zt, lt
    finally:
        if own:
            eng.close()


def autoencoder_inference(model, cost, data, opt, encoder, decoder, *, σ_z: float = 1.0, σ_m: float = 1.0, σ_p: float = 1.0,
                          itr: int = 1000, T: int = 25, c: int = 1, M: int = 20, print_freq: int = 1, alg="hmc",
                          backend="forwarddiff", **kw):
    """construct the decoder subspace -> sample -> (chn, lp)   (src/space_inference.jl:198-210)."""
    W_swa, decoder = auto_encoder_subspace(model, cost, data, opt, encoder, decoder, T=T, c=c, M=M, print_freq=print_freq,
                                           device=kw.get("device", 0))
    return auto_inference(model, data, decoder, W_swa, σ_z=σ_z, σ_m=σ_m, σ_p=σ_p, itr=itr, M=M, alg=alg, backend=backend, **kw)


def predictive(in_model, W_swa, P, z_samples, inp, *, return_trajectories: bool = True,
               engine: Engine | None = None, device: int = 0):
    """The sweep every docs example runs on the samples (docs/src/nn_example.md:207-216, src/plotting.jl:8-9):
    trajectories[:, i] = re(W_swa + P z_i)(inp), their mean and (corrected) std over the samples.  `z_samples` is
    (M, B) — e.g. sub_inference(..., return_z=True)[0][:, 0, :]; `inp` is (in0, Ng).
    Returns (trajectories (O, Ng, B) or None, mean (O, Ng), std (O, Ng))."""
    if not isinstance(in_model, Chain):
        raise TypeError("Error: model_re function is not available for this model")   # src/libs.jl:59
    own = engine is None
    eng = engine or Engine(device)
    try:
        eng.set_model(in_model.dims, in_model.acts)
        eng.set_subspace(W_swa, P)
        out = eng.predict(z_samples, inp, return_trajectories=return_trajectories)
        return (out[2], out[0], out[1]) if return_trajectories else (None, out[0], out[1])
    finally:
        if own:
            eng.close()


def subspace_inference(model, cost, data, opt, *, σ_z: float = 1.0, σ_m: float = 1.0, σ_p: float = 1.0,
                       itr: int = 1000, T: int = 25, c: int = 1, M: int = 20, print_freq: int = 1, alg="rwmh",
                       backend="forwarddiff", method="subspace", **kw):
    """construct -> sample -> (chn, lp, W_swa)   (src/space_inference.jl:33-54).  device_train=True (not in the reference) keeps
    the training step of the construction on the device as well, see subspace_construction."""
    device_train = bool(kw.pop("device_train", False))
    if _sym(method) == "subspace":
        W_swa, P = subspace_construction(model, cost, data, opt, T=T, c=c, M=M, print_freq=print_freq,
                                         device=kw.get("device", 0), device_train=device_train)
    elif _sym(method) == "diffusion":
        raise NotImplementedError("diffusion_subspace is not available on the device path")
    else:
        raise ValueError("Error: No method found")                        # :42
    if _sym(alg) in ("turing_mh", "turing_nuts"):
        raise NotImplementedError("turing_inference is not available on the device path")
    chn, lp = sub_inference(model, data, W_swa, P, σ_z=σ_z, σ_m=σ_m, σ_p=σ_p, itr=itr, M=M, alg=alg, backend=backend, **kw)
    return chn, lp, W_swa
