"""Fixed-length HMC on the device (ssi_hmc_run_dev, alg = :static_hmc): time per transition, the integrator's overhead over
the L batched gradient calls it makes, and effective samples per second against MALA and RWMH.  Not the headline bench.
  python profiles/bench_hmc.py [--out profiles/r03_bench_hmc.json]

  uci   13-50-1 relu, N = 10k, M = 5, 4096 chains, L = 10, 100 transitions
  wide  784-1024-1024-10 relu, N = 60k, M = 20, 64 chains, L = 4, 3 transitions
overhead = (time of one transition) / (L x time of one ssi_logpost_grad_batch_dev call at the same B) - 1: what the
integrator kernels (k_hmc_begin, k_hmc_leap, k_hmc_end) add to the gradient evaluations.
ESS/s: every sampler starts from the same equilibrated states (the chains after HMC's warm-up), runs at its tuned step
size (HMC: dual averaging to 0.8; MALA / RWMH: the sigma_z of a grid whose acceptance is closest to 0.574 / 0.234), and the
effective sample size of the slowest z coordinate over all chains (Geyer's initial monotone sequence on the chain-averaged
autocovariance) is divided by the wall time of the host-pointer call that ran those steps (trace copies included)."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import subspaceinference_jl_b200 as ssi  # noqa: E402
import workloads  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(eng, fn, reps):
    fn()
    eng.sync()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    eng.sync()
    return (time.perf_counter() - t0) / reps


def overhead(name, N, C, L, T, sigma_m, eps):
    prob = workloads.make(name, N=N)
    eng = ssi.Engine(0)
    eng.set_model(prob.dims, prob.acts)
    eng.set_data(prob.X, prob.Y)
    eng.set_subspace(prob.W_swa, prob.P)
    dev = torch.device("cuda", 0)
    M = prob.M
    Z = (0.01 * torch.randn((C, M), generator=torch.Generator().manual_seed(1))).to(dev, torch.float32)
    lp = torch.empty(C, dtype=torch.float64, device=dev)
    g = torch.empty((C, M), dtype=torch.float64, device=dev)
    t_grad = timed(eng, lambda: eng.logpost_grad_dev(Z.data_ptr(), C, lp.data_ptr(), g.data_ptr(), sigma_m=sigma_m), 5)
    lt = torch.empty((T + 1, C), dtype=torch.float64, device=dev)
    run = lambda: eng.hmc_run_dev(C, T + 1, 7, eps, L, sigma_z=0.01, sigma_m=sigma_m, d_lp_trace=lt.data_ptr())
    t_run = timed(eng, run, 1)
    # the initial sample costs one gradient call: the T transitions are the rest
    t_trans = (t_run - t_grad) / T
    out = {"workload": f"{name} {'-'.join(map(str, prob.dims))}, N={prob.N}, M={M}", "chains": C, "n_leapfrog": L,
           "transitions": T, "step_size": eps, "ms_per_transition": t_trans * 1e3, "ms_grad_call": t_grad * 1e3,
           "overhead_vs_L_grad_calls": t_trans / (L * t_grad) - 1.0, "units_per_s": C * prob.N * L / t_trans}
    eng.close()
    return out


def ess_slowest(zt):
    """zt (M, C, T): effective sample size of the slowest coordinate over all chains."""
    M, C, T = zt.shape
    x = zt.astype(np.float64) - zt.mean(axis=(1, 2), keepdims=True)
    f = np.fft.rfft(x, n=2 * T, axis=2)
    acov = np.fft.irfft(f * np.conj(f), axis=2)[:, :, :T].mean(axis=1) / T      # (M, T), averaged over chains
    ess = []
    for m in range(M):
        rho = acov[m] / acov[m, 0]
        tau, prev = -1.0, np.inf
        for k in range(0, T - 1, 2):
            pair = rho[k] + rho[k + 1]
            if pair <= 0:
                break
            pair = min(pair, prev)                  # initial monotone sequence
            tau += 2.0 * pair
            prev = pair
        ess.append(C * T / max(tau, 1.0))
    return float(min(ess)), [float(e) for e in ess]


def ess_per_second(C=4096, L=10, sigma_m=0.1):
    prob = workloads.make("uci")
    eng = ssi.Engine(0)
    eng.set_model(prob.dims, prob.acts)
    eng.set_data(prob.X, prob.Y)
    eng.set_subspace(prob.W_swa, prob.P)
    out = {"workload": f"uci {'-'.join(map(str, prob.dims))}, N={prob.N}, M={prob.M}, sigma_m={sigma_m}, likelihood only",
           "chains": C}
    # HMC warm-up: these states start every sampler
    _, _, _, et = eng.hmc_run(C, 101, 11, 0.01, L, n_adapts=100, sigma_z=0.01, sigma_m=sigma_m, want_z=False, want_lp=False)
    z_eq, _ = eng.mh_state()
    ad = eng.hmc_adapt()
    res = {}
    T_hmc = 200
    eng.sync()
    t0 = time.perf_counter()
    zt, _, at, et = eng.hmc_run(C, T_hmc, 11, 0.01, L, n_adapts=100, sigma_m=sigma_m, z0=z_eq, step_offset=101, adapt_state=ad,
                                want_lp=False)
    t = time.perf_counter() - t0
    e_min, e_all = ess_slowest(zt)
    res["static_hmc"] = {"n_leapfrog": L, "steps": T_hmc, "median_step_size": float(np.median(et[:, 1:])),
                         "accept_rate": float((at[:, 1:] == 1).mean()), "seconds": t, "ess_slowest": e_min, "ess_per_coord": e_all,
                         "ess_per_s": e_min / t}
    for kind, target, T, grid in (("mala", 0.574, 1000, (2e-3, 4e-3, 8e-3, 1.2e-2, 1.6e-2, 2.4e-2, 3.2e-2)),
                                  ("rwmh", 0.234, 2000, (2e-3, 4e-3, 8e-3, 1.2e-2, 1.6e-2, 2.4e-2, 3.2e-2))):
        best = None
        for s in grid:
            _, _, a = eng.mh_run(1024, 40, 3, sigma_z=s, sigma_m=sigma_m, z0=z_eq[:, :1024], want_z=False, want_lp=False, kind=kind)
            r = float(a[:, 1:].mean())
            if best is None or abs(r - target) < abs(best[1] - target):
                best = (s, r)
        s = best[0]
        eng.sync()
        t0 = time.perf_counter()
        zt, _, a = eng.mh_run(C, T, 12, sigma_z=s, sigma_m=sigma_m, z0=z_eq, want_lp=False, kind=kind)
        t = time.perf_counter() - t0
        e_min, e_all = ess_slowest(zt)
        res[kind] = {"sigma_z": s, "steps": T, "accept_rate": float(a[:, 1:].mean()), "seconds": t, "ess_slowest": e_min,
                     "ess_per_coord": e_all, "ess_per_s": e_min / t}
    out["samplers"] = res
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"gpu": gpu_info(),
           "timing": "host clock around work that ends in a device synchronise; warm-up call first",
           "uci": overhead("uci", None, 4096, 10, 100, 0.1, 0.005),
           "wide": overhead("wide", None, 64, 4, 3, 1.0, 1e-4),
           "ess": ess_per_second()}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
