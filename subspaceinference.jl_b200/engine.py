"""Thin object wrapper over the C ABI: one Engine == one ssi_ctx == one GPU."""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np

from . import _lib
from ._lib import RETRY_EXACT, SsiError, Stats, TERM_LL


def _f32(a, order="F") -> np.ndarray:
    return np.require(np.asarray(a, dtype=np.float32), requirements=["ALIGNED", "F_CONTIGUOUS" if order == "F" else "C_CONTIGUOUS"])


def _ptr(a) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(None)


class Engine:
    """Owns a device context.  Matrices are passed in the reference's (Julia) orientation:
    X (in0, N), Y (O, N), P (n, M), Z (M, B); they are handed to the library column-major."""

    def __init__(self, device=0):
        """device: one CUDA device index, or a sequence of indices for a multi-device context (ssi_ctx_create_multi: one
        process drives all of them; batched host calls are sharded by sample / chain, everything else is replicated)."""
        self._lib = _lib.load()
        h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            devs = np.asarray(device, dtype=np.int32)
            rc = self._lib.ssi_ctx_create_multi(_ptr(devs), len(devs), C.byref(h))
            self.devices = tuple(int(d) for d in devs)
        else:
            rc = self._lib.ssi_ctx_create(int(device), C.byref(h))
            self.devices = (int(device),)
        if rc != 0:
            raise SsiError(rc, self._lib.ssi_last_error(None).decode())
        self._h = h
        self.device = self.devices[0]
        self.dims: tuple[int, ...] | None = None
        self.M = 0
        self.N = 0
        self.n = 0

    # ---- plumbing -------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise SsiError(rc, self._lib.ssi_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ssi_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_option(self, key: str, value: int):
        self._check(self._lib.ssi_set_option(self._h, key.encode(), int(value)))

    def set_stream(self, cuda_stream_handle: int | None):
        self._check(self._lib.ssi_set_stream(self._h, C.c_void_p(cuda_stream_handle or None)))

    def sync(self):
        self._check(self._lib.ssi_sync(self._h))

    def stats(self) -> Stats:
        s = Stats()
        self._check(self._lib.ssi_stats(self._h, C.byref(s)))
        return s

    # ---- captured state of the density closure -----------------------------------------
    def set_model(self, dims: Sequence[int], acts: Sequence[int]):
        dims_a = np.asarray(dims, dtype=np.int32)
        acts_a = np.asarray(acts, dtype=np.int32)
        if len(acts_a) != len(dims_a) - 1:
            raise ValueError("need one activation per layer")
        self._check(self._lib.ssi_set_model(self._h, len(acts_a), _ptr(dims_a), _ptr(acts_a)))
        self.dims = tuple(int(d) for d in dims_a)
        self.n = int(sum(dims_a[l] * dims_a[l + 1] + dims_a[l + 1] for l in range(len(acts_a))))

    def set_data(self, X, Y):
        X, Y = _f32(X), _f32(Y)
        if X.ndim != 2 or Y.ndim != 2 or X.shape[1] != Y.shape[1]:
            raise ValueError("X must be (in0, N) and Y (O, N)")
        if self.dims is None or X.shape[0] != self.dims[0] or Y.shape[0] != self.dims[-1]:
            raise ValueError("data shape does not match the model")
        self._check(self._lib.ssi_set_data(self._h, _ptr(X), _ptr(Y), X.shape[1]))
        self.N = int(X.shape[1])

    def set_subspace(self, W_swa, P):
        W_swa, P = _f32(W_swa), _f32(P)
        if P.ndim != 2 or W_swa.ndim != 1 or P.shape[0] != W_swa.shape[0]:
            raise ValueError("W_swa must be (n,) and P (n, M)")
        self._check(self._lib.ssi_set_subspace(self._h, _ptr(W_swa), _ptr(P), P.shape[0], P.shape[1]))
        self.M = int(P.shape[1])

    def set_decoder(self, W_swa, dims: Sequence[int], acts: Sequence[int], theta):
        """Non-linear subspace operator: W = W_swa + decoder(z), decoder = Chain of Dense layers dims[0] (= dimension of z)
        -> ... -> dims[-1] (= n), parameters `theta` in Flux.destructure order (src/space_inference.jl:246-251)."""
        W_swa, theta = _f32(W_swa).reshape(-1), _f32(theta).reshape(-1)
        dims_a, acts_a = np.asarray(dims, dtype=np.int32), np.asarray(acts, dtype=np.int32)
        if len(acts_a) != len(dims_a) - 1:
            raise ValueError("need one activation per decoder layer")
        if theta.shape[0] != int(sum(dims_a[l] * dims_a[l + 1] + dims_a[l + 1] for l in range(len(acts_a)))):
            raise ValueError("theta does not have the decoder's number of parameters")
        self._check(self._lib.ssi_set_decoder(self._h, _ptr(W_swa), len(acts_a), _ptr(dims_a), _ptr(acts_a), _ptr(theta)))
        self.M = int(dims_a[0])

    # ---- density(z), batched -----------------------------------------------------------
    def logpost(self, Z, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0, mask=TERM_LL, return_terms=False):
        Z = _f32(Z)
        if Z.ndim == 1:
            Z = Z.reshape(-1, 1, order="F")
        if Z.shape[0] != self.M:
            raise ValueError(f"Z must have M={self.M} rows")
        B = Z.shape[1]
        lp = np.empty(B, np.float64)
        terms = np.empty((B, 3), np.float64) if return_terms else None
        self._check(self._lib.ssi_logpost_batch(self._h, _ptr(Z), B, sigma_m, sigma_p, sigma_z, mask, _ptr(lp), _ptr(terms)))
        return (lp, terms.T.copy()) if return_terms else lp

    def logpost_dev(self, dZ_ptr: int, B: int, d_lp_ptr: int, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0, mask=TERM_LL,
                    d_terms_ptr: int | None = None):
        """Device-pointer variant (asynchronous on the context stream)."""
        self._check(self._lib.ssi_logpost_batch_dev(self._h, C.c_void_p(dZ_ptr), B, sigma_m, sigma_p, sigma_z, mask,
                                                    C.c_void_p(d_lp_ptr), C.c_void_p(d_terms_ptr or None)))

    def logpost_grad(self, Z, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0, mask=TERM_LL):
        """(lp (B,), grad (M, B)) — the reference's l_pi_grad closure (src/space_inference.jl:107), batched."""
        Z = _f32(Z)
        if Z.ndim == 1:
            Z = Z.reshape(-1, 1, order="F")
        if Z.shape[0] != self.M:
            raise ValueError(f"Z must have M={self.M} rows")
        B = Z.shape[1]
        lp = np.empty(B, np.float64)
        grad = np.empty((self.M, B), np.float64, order="F")
        self._check(self._lib.ssi_logpost_grad_batch(self._h, _ptr(Z), B, sigma_m, sigma_p, sigma_z, mask, _ptr(lp), _ptr(grad)))
        return lp, grad

    def logpost_grad_dev(self, dZ_ptr: int, B: int, d_lp_ptr: int, d_grad_ptr: int, sigma_m=1.0, sigma_p=1.0, sigma_z=1.0,
                         mask=TERM_LL):
        self._check(self._lib.ssi_logpost_grad_batch_dev(self._h, C.c_void_p(dZ_ptr), B, sigma_m, sigma_p, sigma_z, mask,
                                                         C.c_void_p(d_lp_ptr), C.c_void_p(d_grad_ptr)))

    def project(self, Z) -> np.ndarray:
        """W_swa + P z for every column of Z: (n, B)."""
        Z = _f32(Z)
        if Z.ndim == 1:
            Z = Z.reshape(-1, 1, order="F")
        W = np.empty((self.n, Z.shape[1]), np.float32, order="F")
        self._check(self._lib.ssi_project(self._h, _ptr(Z), Z.shape[1], _ptr(W)))
        return W

    def predict(self, Z, Xg, return_trajectories: bool = False):
        """Posterior-predictive sweep: (mean, std[, trajectories]) of re(W_swa + P z)(Xg) over the columns of Z.
        mean/std are (O, Ng) float64 (std corrected, as Julia's), trajectories (O, Ng, B) float32."""
        Z, Xg = _f32(Z), _f32(Xg)
        if Z.ndim == 1:
            Z = Z.reshape(-1, 1, order="F")
        if Z.shape[0] != self.M:
            raise ValueError(f"Z must have M={self.M} rows")
        if Xg.ndim != 2 or self.dims is None or Xg.shape[0] != self.dims[0]:
            raise ValueError("Xg must be (in0, Ng)")
        B, Ng, O = Z.shape[1], Xg.shape[1], self.dims[-1]
        mean = np.empty((O, Ng), np.float64, order="F")
        std = np.empty((O, Ng), np.float64, order="F")
        traj = np.empty((O, Ng, B), np.float32, order="F") if return_trajectories else None
        self._check(self._lib.ssi_predict_batch(self._h, _ptr(Z), B, _ptr(Xg), Ng, _ptr(traj), _ptr(mean), _ptr(std)))
        return (mean, std, traj) if return_trajectories else (mean, std)

    # ---- RWMH ------------------------------------------------------------------------------
    def _traces(self, n_chains: int, n_steps: int, want_z, want_lp, want_accept, want_step_size=False):
        """Host traces of a sampler run (None where not wanted): z (M, n_chains, n_steps) f32, lp / accept / step size f64 / u8 / f64."""
        per_chain = lambda want, dtype: np.empty((n_chains, n_steps), dtype, order="F") if want else None
        return (np.empty((self.M, n_chains, n_steps), np.float32, order="F") if want_z else None,
                per_chain(want_lp, np.float64), per_chain(want_accept, np.uint8), per_chain(want_step_size, np.float64))

    def mh_run(self, n_chains: int, n_steps: int, seed: int, sigma_z=1.0, sigma_m=1.0, sigma_p=1.0, mask=TERM_LL,
               chain_offset: int = 0, z0=None, want_z=True, want_lp=True, want_accept=True, kind: str = "rwmh"):
        """Returns (z_trace (M, n_chains, n_steps) f32, lp_trace (n_chains, n_steps) f64,
        accept (n_chains, n_steps) u8); entries not requested are None."""
        zt, lt, at, _ = self._traces(n_chains, n_steps, want_z, want_lp, want_accept)
        z0a = _f32(z0) if z0 is not None else None
        if z0a is not None and z0a.shape != (self.M, n_chains):
            raise ValueError("z0 must be (M, n_chains)")
        fn = {"rwmh": self._lib.ssi_mh_run, "mala": self._lib.ssi_mala_run}[kind]
        self._check(fn(self._h, n_chains, n_steps, seed, chain_offset, sigma_z, sigma_m, sigma_p, mask,
                       _ptr(z0a), _ptr(zt), _ptr(lt), _ptr(at)))
        self._last_chains = n_chains
        return zt, lt, at

    def mh_state(self):
        """Final (z (M, n_chains) f32, lp (n_chains,) f64) of the last run's chains: what to save for mh_run_from."""
        n = self._last_chains
        z = np.empty((self.M, n), np.float32, order="F")
        lp = np.empty(n, np.float64)
        self._check(self._lib.ssi_mh_get_state(self._h, _ptr(z), _ptr(lp)))
        return z, lp

    def mh_run_from(self, z_state, step_offset: int, n_steps: int, seed: int, sigma_z=1.0, sigma_m=1.0, sigma_p=1.0, mask=TERM_LL,
                    chain_offset: int = 0, want_z=True, want_lp=True, want_accept=True, kind: str = "rwmh"):
        """Continue chains saved with mh_state(): steps step_offset .. step_offset + n_steps - 1 of the same Philox streams."""
        z_state = _f32(z_state)
        n_chains = z_state.shape[1]
        zt, lt, at, _ = self._traces(n_chains, n_steps, want_z, want_lp, want_accept)
        self._check(self._lib.ssi_mh_run_from(self._h, {"rwmh": 0, "mala": 1}[kind], n_chains, n_steps, seed, chain_offset, step_offset,
                                              sigma_z, sigma_m, sigma_p, mask, _ptr(z_state), _ptr(zt), _ptr(lt), _ptr(at)))
        self._last_chains = n_chains
        return zt, lt, at

    def mala_run(self, *a, **kw):
        """MALA with the same arguments as mh_run (src/space_inference.jl:117-120)."""
        return self.mh_run(*a, kind="mala", **kw)

    def mh_run_dev(self, n_chains: int, n_steps: int, seed: int, sigma_z=1.0, sigma_m=1.0, sigma_p=1.0, mask=TERM_LL,
                   chain_offset: int = 0, d_z0: int | None = None, d_z_trace: int | None = None,
                   d_lp_trace: int | None = None, d_accept: int | None = None, kind: str = "rwmh"):
        fn = {"rwmh": self._lib.ssi_mh_run_dev, "mala": self._lib.ssi_mala_run_dev}[kind]
        self._check(fn(self._h, n_chains, n_steps, seed, chain_offset, sigma_z, sigma_m, sigma_p, mask,
                                             C.c_void_p(d_z0 or None), C.c_void_p(d_z_trace or None),
                                             C.c_void_p(d_lp_trace or None), C.c_void_p(d_accept or None)))

    # ---- fixed-length HMC with per-chain dual averaging (alg = :static_hmc) -------------------------------------
    def _hmc_params(self, step_size, n_leapfrog, n_adapts, target_accept, inv_metric):
        minv = None
        if inv_metric is not None:
            minv = np.ascontiguousarray(np.asarray(inv_metric, dtype=np.float64).reshape(-1))
            if minv.shape[0] != self.M:
                raise ValueError(f"inv_metric must have M={self.M} entries")
        hp = _lib.HmcParams(float(step_size), int(n_leapfrog), int(n_adapts), float(target_accept), _ptr(minv).value)
        return hp, minv                      # minv must outlive the call that reads hp

    def hmc_run(self, n_chains: int, n_steps: int, seed: int, step_size: float, n_leapfrog: int, n_adapts: int = 0,
                target_accept: float = 0.8, inv_metric=None, sigma_z=1.0, sigma_m=1.0, sigma_p=1.0, mask=TERM_LL,
                chain_offset: int = 0, z0=None, step_offset: int = 0, adapt_state=None,
                want_z=True, want_lp=True, want_accept=True, want_step_size=True):
        """Fixed-length HMC (ssi_hmc_run): n_leapfrog leapfrog steps per transition, diagonal inverse metric inv_metric
        (M values, default ones), step size adapted per chain by dual averaging over transitions 1..n_adapts.
        Returns (z_trace (M, n_chains, n_steps) f32, lp_trace (n_chains, n_steps) f64, accept (n_chains, n_steps) u8 with
        1 accepted / 0 rejected / 2 divergent, step_size_trace (n_chains, n_steps) f64, NaN at step 0); entries not
        requested are None.  step_offset > 0 continues chains from z0 = mh_state()[0] and adapt_state = hmc_adapt()."""
        zt, lt, at, et = self._traces(n_chains, n_steps, want_z, want_lp, want_accept, want_step_size)
        z0a = _f32(z0) if z0 is not None else None
        if z0a is not None and z0a.shape != (self.M, n_chains):
            raise ValueError("z0 must be (M, n_chains)")
        ada = None
        if adapt_state is not None:
            ada = np.require(np.asarray(adapt_state, dtype=np.float64), requirements=["ALIGNED", "F_CONTIGUOUS"])
            if ada.shape != (3, n_chains):
                raise ValueError("adapt_state must be (3, n_chains)")
        hp, _minv = self._hmc_params(step_size, n_leapfrog, n_adapts, target_accept, inv_metric)
        self._check(self._lib.ssi_hmc_run(self._h, n_chains, n_steps, seed, chain_offset, step_offset, C.byref(hp),
                                          sigma_z, sigma_m, sigma_p, mask, _ptr(z0a), _ptr(ada), _ptr(zt), _ptr(lt), _ptr(at), _ptr(et)))
        self._last_chains = n_chains
        return zt, lt, at, et

    def hmc_run_dev(self, n_chains: int, n_steps: int, seed: int, step_size: float, n_leapfrog: int, n_adapts: int = 0,
                    target_accept: float = 0.8, inv_metric=None, sigma_z=1.0, sigma_m=1.0, sigma_p=1.0, mask=TERM_LL,
                    chain_offset: int = 0, step_offset: int = 0, d_z0: int | None = None, d_adapt: int | None = None,
                    d_z_trace: int | None = None, d_lp_trace: int | None = None, d_accept: int | None = None,
                    d_step_size: int | None = None):
        """Device-pointer variant of hmc_run (asynchronous on the context stream)."""
        hp, _minv = self._hmc_params(step_size, n_leapfrog, n_adapts, target_accept, inv_metric)
        self._check(self._lib.ssi_hmc_run_dev(self._h, n_chains, n_steps, seed, chain_offset, step_offset, C.byref(hp),
                                              sigma_z, sigma_m, sigma_p, mask, C.c_void_p(d_z0 or None), C.c_void_p(d_adapt or None),
                                              C.c_void_p(d_z_trace or None), C.c_void_p(d_lp_trace or None),
                                              C.c_void_p(d_accept or None), C.c_void_p(d_step_size or None)))
        self._last_chains = n_chains

    def hmc_adapt(self) -> np.ndarray:
        """(3, n_chains) f64: log eps, log eps_bar, H_bar of every chain of the last HMC run (what hmc_run's adapt_state takes)."""
        a = np.empty((3, self._last_chains), np.float64, order="F")
        self._check(self._lib.ssi_hmc_get_adapt(self._h, _ptr(a)))
        return a

    def rng_replay(self, seed: int, chain: int, step: int, M: int | None = None):
        M = self.M if M is None else M
        eps = np.empty(M, np.float32)
        e = C.c_double()
        rc = self._lib.ssi_rng_replay(seed, chain, step, M, _ptr(eps), C.byref(e))
        if rc != 0:
            raise SsiError(rc, "ssi_rng_replay: bad arguments")
        return eps, e.value

    # ---- construction streams ----------------------------------------------------------------
    def swa_begin(self, n: int, K_max: int):
        self._check(self._lib.ssi_swa_begin(self._h, n, K_max))
        self._swa_n = int(n)

    def swa_push(self, W, n_scalar: float):
        W = _f32(W).reshape(-1)
        if W.shape[0] != self._swa_n:
            raise ValueError("snapshot length does not match ssi_swa_begin")
        self._check(self._lib.ssi_swa_push(self._h, _ptr(W), float(n_scalar)))

    def swa_push_dev(self, dW_ptr: int, n_scalar: float):
        self._check(self._lib.ssi_swa_push_dev(self._h, C.c_void_p(dW_ptr), float(n_scalar)))

    # ---- the step before the path: mini-batch training on the device (include/ssi.h, ssi_train_*) ----
    def train_begin(self, W0, optimiser: str = "descent", eta: float = 0.1, beta=(0.9, 0.999)):
        """Start training from the flat weights W0 (src/libs.jl:19-22 layout).  optimiser: "descent" | "adam"."""
        kinds = {"descent": 0, "adam": 1}
        if optimiser not in kinds:
            raise ValueError("optimiser must be 'descent' or 'adam'")
        W0 = _f32(W0).reshape(-1)
        if W0.shape[0] != self.n:
            raise ValueError("W0 does not have the model's number of parameters")
        self._check(self._lib.ssi_train_begin(self._h, _ptr(W0), kinds[optimiser], float(eta), float(beta[0]), float(beta[1])))

    def train_step(self, batch, *, want_loss: bool = True):
        """One mini-batch of `gradient + update!` (src/subspace_construction.jl:39-43) with cost = mse(m(x), y).
        batch: an array of observation indices, or a (start, count) tuple for contiguous columns.  Returns
        training_loss (before the update) or None."""
        loss = C.c_double(0.0)
        lp = C.byref(loss) if want_loss else None
        if isinstance(batch, tuple):
            rc = self._lib.ssi_train_step(self._h, None, int(batch[0]), int(batch[1]), lp)
        else:
            idx = np.ascontiguousarray(np.asarray(batch, dtype=np.int64).reshape(-1))
            rc = self._lib.ssi_train_step(self._h, _ptr(idx), 0, int(idx.shape[0]), lp)
        self._check(rc)
        return float(loss.value) if want_loss else None

    def train_snapshot(self, n_scalar: float):
        """swa_push of the device-resident weights (no host round trip)."""
        self._check(self._lib.ssi_train_snapshot(self._h, float(n_scalar)))

    def train_weights(self) -> np.ndarray:
        W = np.empty(self.n, np.float32)
        self._check(self._lib.ssi_train_get_weights(self._h, _ptr(W)))
        return W

    def train_end(self):
        self._check(self._lib.ssi_train_end(self._h))

    def swa_deviations(self) -> np.ndarray:
        """The deviation matrix collected so far, (n, K) float32 (`reshape(A, all_len, :)`, src/subspace_construction.jl:61)."""
        A = np.empty((self._swa_n, self.swa_columns()), np.float32, order="F")
        self._check(self._lib.ssi_swa_deviations(self._h, _ptr(A)))
        return A

    def swa_mean(self) -> np.ndarray:
        W = np.empty(self._swa_n, np.float32)
        self._check(self._lib.ssi_swa_mean(self._h, _ptr(W)))
        return W

    def swa_columns(self) -> int:
        return int(self._lib.ssi_swa_columns(self._h))

    def swa_gram_dev(self, dG_ptr: int, exact: bool = False):
        """Gram of the local row shard's deviation columns into a device buffer of K x K doubles (to be all-reduced)."""
        self._check(self._lib.ssi_swa_gram_dev(self._h, C.c_void_p(dG_ptr), int(exact)))

    def swa_finish_gram(self, M: int, dG_ptr: int, gram_exact: bool = False, install: bool = False, want_P: bool = True):
        """Eigen-solve of the all-reduced Gram + W_swa / P rows of the local shard.  Returns None when the conditioning
        check asks for the exact Gram (SSI_RETRY_EXACT): repeat swa_gram_dev(exact=True), all-reduce, and call again
        with gram_exact=True."""
        n, K = self._swa_n, self.swa_columns()
        W_swa = np.empty(n, np.float32)
        P = np.empty((n, M), np.float32, order="F") if want_P else None
        s = np.empty(max(K, 1), np.float64)
        rc = self._lib.ssi_swa_finish_gram(self._h, M, C.c_void_p(dG_ptr), int(gram_exact), _ptr(W_swa), _ptr(P), _ptr(s), int(install))
        if rc == RETRY_EXACT:
            return None
        self._check(rc)
        if install:
            self.M = M
        return W_swa, P, s[:K]

    def swa_finish_sharded(self, M: int, all_reduce, install: bool = False):
        """Row-sharded finish: `all_reduce(tensor)` sums a CUDA float64 tensor in place across the ranks that hold the
        other row shards (e.g. torch.distributed.all_reduce).  The only collective of the construction path."""
        import torch
        K = self.swa_columns()
        G = torch.empty(K * K, dtype=torch.float64, device=f"cuda:{self.device}")
        for exact in (False, True):
            self.swa_gram_dev(G.data_ptr(), exact)
            self.sync()
            all_reduce(G)
            torch.cuda.synchronize(self.device)
            out = self.swa_finish_gram(M, G.data_ptr(), gram_exact=exact, install=install)
            if out is not None:
                return out
        raise RuntimeError("unreachable: the exact Gram is never rejected")

    def swa_finish(self, M: int, install: bool = False, want_P: bool = True):
        n, K = self._swa_n, self.swa_columns()
        W_swa = np.empty(n, np.float32)
        P = np.empty((n, M), np.float32, order="F") if want_P else None
        s = np.empty(max(K, 1), np.float64)
        self._check(self._lib.ssi_swa_finish(self._h, M, _ptr(W_swa), _ptr(P), _ptr(s), int(install)))
        if install:
            self.M = M
        return W_swa, P, s[:K]
