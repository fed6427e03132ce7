"""Argument checks of the host sampler entry points: a bad run is rejected with the same code and message on a single-device
and on a multi-device context, and the state of the previous run survives it; devices without work in a call report none."""
import ctypes as C

import numpy as np
import pytest

import ssi_oracle as orc

pytestmark = pytest.mark.gpu

SEED, SIGMA_Z, SIGMA_M = 5, 0.05, 0.2
ENTRIES = ("mh_run", "mala_run", "mh_run_from", "hmc_run")
BASE = dict(n_chains=16, n_steps=3, chain_offset=0, step_offset=0, kind=0, z=False, adapt=False,
            step_size=0.02, n_leapfrog=3, n_adapts=4, target_accept=0.8, inv_metric=None)

# name, entry points it applies to, arguments that differ from BASE, expected code
BAD = [
    ("no_chains", ENTRIES, dict(n_chains=0), -1),
    ("no_steps", ENTRIES, dict(n_steps=0), -1),
    ("negative_chain_offset", ENTRIES, dict(chain_offset=-1), -1),
    ("chain_ids_past_32_bits", ENTRIES, dict(chain_offset=2**32 - 8), -1),
    ("continued_without_z", ("mh_run_from", "hmc_run"), dict(step_offset=2), -1),
    ("hmc_kind_to_run_from", ("mh_run_from",), dict(kind=2), -1),
    ("step_size_zero", ("hmc_run",), dict(step_size=0.0), -1),
    ("step_size_inf", ("hmc_run",), dict(step_size=np.inf), -1),
    ("n_leapfrog_zero", ("hmc_run",), dict(n_leapfrog=0), -1),
    ("n_adapts_negative", ("hmc_run",), dict(n_adapts=-1), -1),
    ("n_adapts_past_32_bits", ("hmc_run",), dict(n_adapts=2**32), -1),
    ("target_accept_zero", ("hmc_run",), dict(target_accept=0.0), -1),
    ("target_accept_one", ("hmc_run",), dict(target_accept=1.0), -1),
    ("inv_metric_zero", ("hmc_run",), dict(inv_metric=[1.0, 1.0, 0.0, 1.0, 1.0]), -1),
    ("inv_metric_nan", ("hmc_run",), dict(inv_metric=[1.0, np.nan, 1.0, 1.0, 1.0]), -1),
    ("continued_hmc_without_adaptation_state", ("hmc_run",), dict(step_offset=2, z=True), -1),
]


def _call(eng, entry, **args):
    """One host call of `entry` without traces, BASE overridden by `args`: (return code, error message)."""
    a = dict(BASE, **args)
    lib, h = eng._lib, eng._h
    n, S, off = a["n_chains"], a["n_steps"], a["chain_offset"]
    z = np.zeros((eng.M, max(n, 1)), np.float32, order="F") if a["z"] else None
    zp = C.c_void_p(z.ctypes.data) if z is not None else None
    sig = (SIGMA_Z, SIGMA_M, 1.0, orc.TERM_LL)
    if entry == "mh_run":
        rc = lib.ssi_mh_run(h, n, S, SEED, off, *sig, zp, None, None, None)
    elif entry == "mala_run":
        rc = lib.ssi_mala_run(h, n, S, SEED, off, *sig, zp, None, None, None)
    elif entry == "mh_run_from":
        rc = lib.ssi_mh_run_from(h, a["kind"], n, S, SEED, off, a["step_offset"], *sig, zp, None, None, None)
    else:
        hp, _minv = eng._hmc_params(a["step_size"], a["n_leapfrog"], a["n_adapts"], a["target_accept"], a["inv_metric"])
        ad = np.zeros((3, max(n, 1)), np.float64, order="F") if a["adapt"] else None
        rc = lib.ssi_hmc_run(h, n, S, SEED, off, a["step_offset"], C.byref(hp), *sig, zp,
                             C.c_void_p(ad.ctypes.data) if ad is not None else None, None, None, None, None)
    return rc, lib.ssi_last_error(h).decode()


def _contexts(ssi):
    import torch
    ndev = torch.cuda.device_count()
    return [ssi.Engine(0), ssi.Engine([0])] + ([ssi.Engine(list(range(ndev)))] if ndev > 1 else [])


def test_rejected_runs_agree_and_keep_the_previous_state(ssi):
    """Every bad run of the table, on every host entry point it applies to: the same code and message on every context,
    and mh_state() / hmc_adapt() still return the previous HMC run's state bit for bit."""
    prob = orc.make_problem("uci", N=900)
    ctxs = _contexts(ssi)
    try:
        prev = []
        for eng in ctxs:
            eng.set_model(prob.dims, prob.acts)
            eng.set_data(prob.X, prob.Y)
            eng.set_subspace(prob.W_swa, prob.P)
            eng.hmc_run(40, 4, SEED, 0.02, 3, n_adapts=2, sigma_z=SIGMA_Z, sigma_m=SIGMA_M, want_z=False, want_lp=False)
            prev.append((*eng.mh_state(), eng.hmc_adapt()))
        for name, entries, args, code in BAD:
            for entry in entries:
                got = [_call(eng, entry, **args) for eng in ctxs]
                assert got[0][0] == code, (name, entry, got[0])
                for g in got[1:]:
                    assert g == got[0], (name, entry, got)
                for eng, (z, lp, ad) in zip(ctxs, prev):
                    z2, lp2 = eng.mh_state()
                    np.testing.assert_array_equal(z2, z, err_msg=f"{name} {entry}")
                    np.testing.assert_array_equal(lp2, lp, err_msg=f"{name} {entry}")
                    np.testing.assert_array_equal(eng.hmc_adapt(), ad, err_msg=f"{name} {entry}")
    finally:
        for eng in ctxs:
            eng.close()


def test_rejected_without_subspace(ssi):
    prob = orc.make_problem("uci", N=900)
    ctxs = _contexts(ssi)
    try:
        for eng in ctxs:
            eng.set_model(prob.dims, prob.acts)
            eng.set_data(prob.X, prob.Y)
        for entry in ENTRIES:
            got = [_call(eng, entry) for eng in ctxs]
            assert got[0][0] == -3, (entry, got[0])
            assert all(g == got[0] for g in got[1:]), (entry, got)
    finally:
        for eng in ctxs:
            eng.close()


def test_idle_devices_report_no_work(ssi):
    """64 chains then 16 on several devices: the second run leaves every device but the first idle (shards are whole warps),
    and the stats are that run's alone; likewise a log-posterior of 16 samples after one of 64."""
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs two devices")
    prob = orc.make_problem("uci", N=900)
    rng = np.random.default_rng(64)
    Z = (0.1 * rng.standard_normal((prob.M, 64))).astype(np.float32)
    with ssi.Engine(0) as single, ssi.Engine(list(range(ndev))) as multi:
        for eng in (single, multi):
            eng.set_model(prob.dims, prob.acts)
            eng.set_data(prob.X, prob.Y)
            eng.set_subspace(prob.W_swa, prob.P)
        multi.mh_run(64, 4, SEED, sigma_z=SIGMA_Z, sigma_m=SIGMA_M)
        _, _, at = multi.mh_run(16, 4, SEED, sigma_z=SIGMA_Z, sigma_m=SIGMA_M)
        st = multi.stats()
        assert st.mh_proposals == 16 * 3
        assert st.mh_accepts == int(at[:, 1:].sum())
        multi.logpost(Z, SIGMA_M)
        multi.logpost(Z[:, :16], SIGMA_M)
        single.logpost(Z[:, :16], SIGMA_M)
        assert multi.stats().last_units == single.stats().last_units
