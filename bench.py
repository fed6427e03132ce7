#!/usr/bin/env python
"""bench.py — log-posterior evals/s in (sample x datapoint) units on N B200s of one node.

A "step" is one batched log-posterior evaluation (the hot call, ssi_logpost_batch) over B
subspace points per GPU on the full synthetic dataset:
    W = W_swa + P z  ->  Dense-chain forward over all N datapoints  ->  Gaussian log-lik -> lp[b]
Workloads (BASELINE.json configs):
    wide  784-1024-1024-10 relu, N=60000, M=20  (configs[2]/[4]; default, the config the metric's
          1/2/4/8-GPU sweep is quoted on; B per GPU fixed => weak scaling)
    uci   13-50-1 relu, N=10000, M=5, 4096 chains (configs[1])

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload wide|uci|...] [--batch B] [--dump-outputs DIR]
  python bench.py --impl reference ...      # the CPU restatement of the reference's path

--dump-outputs DIR writes what the last timed step computed, as the caller receives it, to DIR/<name>.npy: lp (samples,)
float64 for the density workloads, z_trace (M, chains, steps) float32 and lp_trace (chains, steps) float64 for the MH / MALA
workloads (every rank's chains when N > 1).  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.

Synthetic inputs come from workloads.py (NumPy); oracle/ is touched only as the checker after the timed region and by the
CPU-baseline / --impl reference legs.
  value   device-timed (CUDA events on the launching stream) with Z already resident in HBM (ssi_logpost_batch_dev);
  e2e     the same metric through the reference-facing HOST-pointer call, ssi_logpost_batch (ssi_mh_run for the MH
          workloads): host Z -> H2D -> kernels -> D2H of lp inside every timed step, then the gather the sampler needs.
Extra keys of the one JSON line (rank 0):
  streams          BASELINE configs[3] (n = 10,020,874, K = 100, M = 20): SWA push, Gram, eigen-solve, P and the whole
                   ssi_swa_finish as GB/s and fractions of the measured HBM peak, with a Float64 (torch, on the device) check of P
  mh_c5            BASELINE configs[4] per GPU: RWMH steps of 8192 chains with the NCCL gather of the z and lp traces,
                   time inside / outside the collective
  multi_device_ctx N > 1: the same step through ONE process and ONE multi-device context (ssi_ctx_create_multi), no torchrun
  timeline         N > 1: per-step device time of the compute and of the NCCL gather (max over ranks), clocks of every rank
Multi-GPU: proposals are sharded across ranks (no data-path collective); lp is all-gathered (NCCL) inside the step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (oracle problem name, default B per GPU, sigma_m, z scale)
    "wide": ("wide", 16384, 1.0, 0.1),
    "uci": ("uci", 4096, 0.1, 0.1),
    # configs[1] as the sampler runs it: a step = MH_STEPS Metropolis-Hastings steps of 4096 chains per GPU, all on the device
    "uci-mh": ("uci", 4096, 0.1, 0.01),
    # the same with the Metropolis-adjusted Langevin sampler (value + gradient per step; units are still forward evaluations)
    "uci-mala": ("uci", 4096, 0.1, 0.01),
    # configs[4] per GPU: 8192 of the 65536 chains in the M=20 subspace of the wide MLP, samples and log-probs gathered with NCCL
    "wide-mh": ("wide", 8192, 1.0, 0.02),
    # MALA on the wide MLP: value + gradient per step, the reverse pass on the tensor-core GEMM (ssi_gemm_tc.cu)
    "wide-mala": ("wide", 512, 1.0, 0.02),
}
MH_STEPS_BY_WORKLOAD = {"wide-mh": 2, "wide-mala": 2}      # a wide MH step is 8192 x 60000 units (~3 s): two per bench step
MH_STEPS = 100


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self._stop, self._t = gpu_index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        pw = [float(r[3]) for r in self.rows if r[3].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_mhz_min": sm[0] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "power_w_max": max(pw) if pw else None, "samples": len(self.rows)}


def cpu_reference(workload: str, budget_s: float, steps: int = 1, warmup: int = 0):
    """The reference's CPU path restated (oracle/ssi_oracle.py): one z per call, Float64, per-layer BLAS GEMM over the full
    dataset, EVERY host core (NumPy/OpenBLAS threads = os.cpu_count(); torchrun's OMP_NUM_THREADS=1 is overridden).
    Bounded sample.  A second opinion with torch's CPU Float64 GEMMs is timed beside it; `value` is the faster of the two."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import ssi_oracle as orc
    host_cpus = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=host_cpus)
    except Exception:
        pass
    name, _, sigma_m, zs = WORKLOADS[workload]
    prob = orc.make_problem(name)
    rng = np.random.default_rng(0)
    X64, Y64 = prob.X.astype(np.float64), prob.Y.astype(np.float64)
    prob64 = orc.Problem(prob.dims, prob.acts, X64, Y64, prob.W_swa, prob.P)
    z = zs * rng.standard_normal(prob.M)
    orc.density(prob64, z, sigma_m)                        # warm-up (BLAS threads, page faults)
    t0 = time.perf_counter()
    lp_np = orc.density(prob64, z, sigma_m)
    per_eval = time.perf_counter() - t0
    evals_per_step = max(1, int(budget_s / max(per_eval, 1e-6) / max(1, steps + warmup)))
    times = []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        for _ in range(evals_per_step):
            z = zs * rng.standard_normal(prob.M)
            orc.density(prob64, z, sigma_m)
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    units = evals_per_step * len(times) * prob.N
    try:
        from threadpoolctl import threadpool_info
        blas_threads = max([i.get("num_threads", 1) for i in threadpool_info() if i.get("user_api") == "blas"] or [1])
    except Exception:
        blas_threads = host_cpus
    value, kind_note, cores = units / total, "NumPy/OpenBLAS", int(blas_threads)
    torch_check = None
    try:        # the same evaluation with torch's CPU Float64 kernels (MKL / oneDNN), all cores
        import torch
        torch.set_num_threads(host_cpus)
        Xt, Yt = torch.from_numpy(X64), torch.from_numpy(Y64)
        W64, P64 = torch.from_numpy(prob.W_swa.astype(np.float64)), torch.from_numpy(prob.P.astype(np.float64))

        def dens_t(zv):
            w = W64 + P64 @ torch.from_numpy(zv)
            h, off = Xt, 0
            for l, act in enumerate(prob.acts):
                din, dout = prob.dims[l], prob.dims[l + 1]
                Wl = w[off:off + din * dout].reshape(din, dout).T         # column-major (out x in)
                off += din * dout
                h = Wl @ h + w[off:off + dout][:, None]
                off += dout
                h = (h, torch.relu(h), torch.tanh(h), torch.sigmoid(h))[act]
            k = Yt.numel()
            return float(-0.5 * k * np.log(2 * np.pi) - k * np.log(sigma_m) - ((Yt - h) ** 2).sum() / (2 * sigma_m ** 2))

        lp_t = dens_t(z)
        n_t = max(1, min(evals_per_step, int(5.0 / max(per_eval, 1e-6))))
        t0 = time.perf_counter()
        for _ in range(n_t):
            dens_t(zs * rng.standard_normal(prob.M))
        t_t = time.perf_counter() - t0
        lp_np = orc.density(prob64, z, sigma_m)
        torch_check = {"value": n_t * prob.N / t_t, "threads": torch.get_num_threads(), "evals": n_t,
                       "agrees_with_numpy": bool(abs(lp_t - lp_np) <= 1e-9 * abs(lp_np))}
        if torch_check["value"] > value:
            value, kind_note, cores = torch_check["value"], "torch CPU Float64", torch.get_num_threads()
    except Exception as ex:       # the cross-check is optional
        torch_check = {"error": str(ex)[:200]}
    return {"value": value, "unit": "sample*datapoint/s", "cores": cores, "host_cpus": host_cpus, "kind": "port",
            "sample": f"{evals_per_step * len(times)} sequential density(z) evaluations (one z per call, Float64 {kind_note}, "
                      f"all {host_cpus} host cores, full N={prob.N}) of workload {workload}; lower bound on the reference's time "
                      f"(no Flux.destructure/alloc overhead)",
            "numpy_openblas": {"value": units / total, "threads": int(blas_threads)}, "torch_f64": torch_check,
            "ms_per_step": 1e3 * total / len(times), "evals_per_step": evals_per_step}


def workload_config(workload, B, world):
    import workloads
    MH_STEPS = MH_STEPS_BY_WORKLOAD.get(workload, 100)
    name = WORKLOADS[workload][0]
    dims, _, M, N, _ = workloads.CONFIGS[name]
    what = (f"{MH_STEPS} on-device {'MALA' if workload.endswith('-mala') else 'RWMH'} steps of {B} chains per GPU (one batched "
            f"log-posterior{' + gradient' if workload.endswith('-mala') else ''} per step)" if workload.endswith(("-mh", "-mala"))
            else f"batched log-posterior over {B} subspace points per GPU")
    return {"workload": f"{workload}: MLP {'-'.join(map(str, dims))}, N={N}, M={M}, {what}",
            "dims": list(dims), "N": N, "M": M, "batch_per_gpu": B, "global_batch": B * world,
            "parallelism": (f"chains sharded x{world}, W_swa/P/X/Y replicated, NCCL all-gather of the z and lp traces"
                            if workload.endswith(("-mh", "-mala")) else
                            f"proposals sharded x{world}, W_swa/P/X/Y replicated, NCCL all-gather of lp"),
            "l2": "inputs larger than L2 (X + per-sample activations stream through HBM); no explicit flush"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    res = cpu_reference(args.workload, budget_s=max(10.0, 8.0 * (args.steps + args.warmup)), steps=args.steps, warmup=args.warmup)
    cfg = workload_config(args.workload, args.batch, world)
    line = {"impl": "reference", "metric": "log-posterior evals/sec (samples x datapoints)", "value": res["value"],
            "unit": "sample*datapoint/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "host_cpus", "kind", "sample", "numpy_openblas", "torch_f64")},
            "e2e": {"value": res["value"], "unit": "sample*datapoint/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------------------------
# extra sections of the JSON line
# ------------------------------------------------------------------------------------------------------------------
def streams_section(ssi, torch, dev, local_rank, peaks, n=10_020_874, K=100, M=20, reps=3):
    """BASELINE configs[3]: the construction streams on a ~10M-parameter flat vector, each against the measured HBM peak;
    P checked against a Float64 Gram-route restatement evaluated with torch on the device (a checker, outside the timing)."""
    stream = torch.cuda.current_stream(dev)
    eng = ssi.Engine(local_rank)
    eng.set_stream(stream.cuda_stream)
    try:
        g = torch.Generator(device=dev).manual_seed(4)
        w = 0.05 * torch.randn(n, device=dev, generator=g)
        snaps = []
        for _ in range(K):                         # W_t = W_0 + cumulative 1e-3 N(0,1) steps (SURVEY 8d, C4), n_t = t
            w = w + 1e-3 * torch.randn(n, device=dev, generator=g)
            snaps.append(w.clone())
        best = {"push": 1e9, "finish": 1e9, "gram": 1e9, "eigen": 1e9, "p": 1e9}
        W_swa = np.empty(n, np.float32)
        P = np.empty((n, M), np.float32, order="F")
        for rep in range(reps):
            eng.swa_begin(n, K)
            stream.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for t, s in enumerate(snaps):
                eng.swa_push_dev(s.data_ptr(), float(t + 1))
            e1.record(stream)
            stream.synchronize()
            best["push"] = min(best["push"], e0.elapsed_time(e1) / K)
            last = rep == reps - 1
            eng._check(eng._lib.ssi_swa_finish(eng._h, M, W_swa.ctypes.data if last else None, P.ctypes.data if last else None, None, 0))
            st = eng.stats()
            if not last:                           # the last repetition also copies W_swa and P to the host
                best["finish"] = min(best["finish"], st.last_ms)
            best["gram"] = min(best["gram"], st.finish_gram_ms)
            best["eigen"] = min(best["eigen"], st.finish_eigen_ms)
            best["p"] = min(best["p"], st.finish_p_ms)
        # Float64 restatement on the device: mean recurrence (src/subspace_construction.jl:46-47), deviations against the
        # updated mean (:51), Gram, eigh, P = A V_M
        mean = torch.zeros(n, dtype=torch.float64, device=dev)
        G = torch.zeros(K, K, dtype=torch.float64, device=dev)
        A = torch.empty(K, n, dtype=torch.float32, device=dev)
        for t, s in enumerate(snaps, start=1):
            s64 = s.double()
            mean = (t * mean + s64) / (t + 1.0)
            A[t - 1] = (s64 - mean).float()
        del snaps
        for c0 in range(0, n, 1 << 21):
            blk = A[:, c0:c0 + (1 << 21)].double()
            G += blk @ blk.T
        lam, V = torch.linalg.eigh(G)
        V = V.flip(1)[:, :M]
        err_p, pmax = 0.0, 0.0
        Pd = torch.from_numpy(P).to(dev)
        for c0 in range(0, n, 1 << 21):
            ref = A[:, c0:c0 + (1 << 21)].double().T @ V
            got = Pd[c0:c0 + (1 << 21)].double()
            if c0 == 0:
                sgn = torch.sign((ref * got).sum(0))
            err_p = max(err_p, float((got * sgn - ref).abs().max()))
            pmax = max(pmax, float(ref.abs().max()))
        err_w = float((torch.from_numpy(W_swa).to(dev).double() - mean).abs().max() / mean.abs().max())
        hbm = peaks["hbm_gbs"]

        def entry(ms, nbytes):
            return {"ms": ms, "gbs": nbytes / (ms * 1e-3) / 1e9, "frac": nbytes / (ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes": nbytes}

        st = eng.stats()
        traffic = {}
        tfile = ROOT / "profiles" / "traffic.json"
        if tfile.exists():
            traffic = json.loads(tfile.read_text()).get("streams", {})
        return {"config": f"BASELINE configs[3]: n={n}, K={K} snapshots, M={M}", "hbm_peak_gbs": hbm,
                "swa_push": {**entry(best["push"], 16.0 * n), "note": "per snapshot; back-to-back pushes: part of the traffic is served by "
                             "L2 (160 MB per push against 126 MB of L2), see dram_bytes_ncu for what reaches DRAM"},
                "gram": entry(best["gram"], 4.0 * n * K),
                "eigen": {"ms": best["eigen"], "sweeps": st.jacobi_sweeps},
                "form_p": entry(best["p"], 4.0 * n * K + 4.0 * n * M),
                "finish": entry(best["finish"], 2 * 4.0 * n * K + 4.0 * n * M),
                "gram_path": st.gram_path, "gram_risk": st.gram_risk,
                "parity_vs_f64": {"W_swa_rel_err": err_w, "P_rel_err_up_to_sign": err_p / pmax, "tolerance": 1e-4,
                                  "checker": "torch Float64 on the device (Gram route), outside the timed region"},
                "dram_bytes_ncu": traffic}
    finally:
        eng.close()


def mh_c5_section(ssi, torch, dist, eng, prob, dev, rank, world, stream, chains=8192, steps=2, sigma_z=0.02):
    """BASELINE configs[4] per GPU: `steps` RWMH steps of `chains` chains, then the NCCL gather of the z and lp traces."""
    M = prob.M
    d_z = torch.empty(M * chains * steps, dtype=torch.float32, device=dev)
    d_lp = torch.empty(chains * steps, dtype=torch.float64, device=dev)
    d_z_all = torch.empty(world * d_z.numel(), dtype=torch.float32, device=dev) if world > 1 else None
    d_lp_all = torch.empty(world * d_lp.numel(), dtype=torch.float64, device=dev) if world > 1 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

    def once():
        ev[0].record(stream)
        eng.mh_run_dev(chains, steps, 2024, sigma_z=sigma_z, sigma_m=1.0, chain_offset=rank * chains,
                       d_z_trace=d_z.data_ptr(), d_lp_trace=d_lp.data_ptr())
        ev[1].record(stream)
        if world > 1:
            dist.all_gather_into_tensor(d_z_all, d_z)
            dist.all_gather_into_tensor(d_lp_all, d_lp)
        ev[2].record(stream)

    once()                                       # warm-up (allocations, NCCL channels)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    once()
    torch.cuda.synchronize()
    t = torch.tensor([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[2])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sampler_ms, gather_ms, total_ms = (float(v) for v in t)
    units = float(chains) * world * prob.N * steps
    return {"config": f"BASELINE configs[4]: {chains} RWMH chains per GPU x {world} GPUs = {chains * world} chains, {steps} steps, "
                      f"M={M} subspace of {'-'.join(map(str, prob.dims))}, N={prob.N}",
            "value": units / (total_ms * 1e-3), "unit": "sample*datapoint/s", "ms_total": total_ms,
            "ms_sampler": sampler_ms, "ms_per_mh_step": sampler_ms / steps, "ms_nccl_gather": gather_ms,
            "gather_bytes_per_gpu": int(d_z.numel() * 4 + d_lp.numel() * 8),
            "timing": "CUDA events on the launching stream, max over ranks"}


def multi_ctx_section(ssi, torch, prob, world, B, sigma_m, zs, steps):
    """N > 1, rank 0 alone, after every rank has released its GPU: ONE process, ONE multi-device context
    (ssi_ctx_create_multi) over all N devices, the host-pointer call a single Julia process would make."""
    eng = ssi.Engine(list(range(world)))
    try:
        eng.set_model(prob.dims, prob.acts)
        eng.set_data(prob.X, prob.Y)
        eng.set_subspace(prob.W_swa, prob.P)
        rng = np.random.default_rng(99)
        Z = np.asfortranarray((zs * rng.standard_normal((prob.M, B * world))).astype(np.float32))
        eng.logpost(Z[:, :256 * world], sigma_m)               # warm-up: operand preparation on every device
        t0 = time.perf_counter()
        for _ in range(steps):
            lp = eng.logpost(Z, sigma_m)
        wall = (time.perf_counter() - t0) / steps
        dev_ms = eng.stats().last_ms
        return {"n_devices": world, "processes": 1, "call": "ssi_logpost_batch on a context from ssi_ctx_create_multi (host pointers)",
                "value": float(B) * world * prob.N / wall, "unit": "sample*datapoint/s", "ms_per_step_wall": wall * 1e3,
                "ms_per_step_device_max": dev_ms, "steps": steps, "finite": bool(np.isfinite(lp).all())}
    finally:
        eng.close()


DUMP_LIMIT = 64 << 20


def mh_traces(z_flat, lp_flat, world, chains, steps, M):
    """Flat device traces gathered rank after rank (each rank's block an (M, chains, steps) / (chains, steps) column-major
    buffer) in the shapes mh_run returns, over all world * chains chains: z (M, world*chains, steps), lp (world*chains, steps)."""
    z = z_flat.reshape(world, steps, chains, M).transpose(3, 0, 2, 1).reshape(M, world * chains, steps)
    lp = lp_flat.reshape(world, steps, chains).transpose(0, 2, 1).reshape(world * chains, steps)
    return z, lp


def dump_outputs(out_dir, arrays: dict):
    """Write every {name: (array, sample axis)} as out_dir/<name>.npy.  Above DUMP_LIMIT bytes in all, every array keeps the
    same fixed sample of its samples / chains (sorted ids drawn with default_rng(0)), so two dumps still compare entry for entry."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    total = sum(a.nbytes for a, _ in arrays.values())
    a0, ax0 = next(iter(arrays.values()))
    n = a0.shape[ax0]
    keep = None
    if total > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * DUMP_LIMIT // total), replace=False))
    for name, (a, axis) in arrays.items():
        np.save(out_dir / f"{name}.npy", a if keep is None else np.take(a, keep, axis=axis))


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line, on the process's real stdout."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def guard_stdout():
    """Libraries write banners to file descriptor 1 ("NCCL version ..." at the first collective): keep stdout for the JSON
    line alone by pointing fd 1 at stderr for the rest of the run."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("SSI_BENCH_WORKLOAD", "wide"), choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="subspace points per GPU per step")
    ap.add_argument("--path", default="auto", choices=["auto", "fused", "layered", "tensor", "basis"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the streams / mh_c5 / multi_device_ctx sections")
    ap.add_argument("--opt", action="append", default=[], help="library A/B switch, key=value (ssi_set_option); repeatable")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.batch <= 0:
        args.batch = int(os.environ.get("SSI_BENCH_BATCH", WORKLOADS[args.workload][1]))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import subspaceinference_jl_b200 as ssi
    import workloads              # synthetic inputs (NumPy); the oracle is only the checker after the timed region

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    # a host-side group for the waits that must not occupy a GPU: a rank parked in an NCCL barrier keeps a spinning kernel
    # on its device, and a persistent grid launched beside it (the multi-device section below) runs in two waves
    host_group = dist.new_group(backend="gloo") if world > 1 else None

    name, _, sigma_m, zs = WORKLOADS[args.workload]
    prob = workloads.make(name)
    B = args.batch
    eng = ssi.Engine(local_rank)
    eng.set_model(prob.dims, prob.acts)
    eng.set_data(prob.X, prob.Y)
    eng.set_subspace(prob.W_swa, prob.P)
    eng.set_option("path", {"auto": 0, "fused": 1, "layered": 2, "tensor": 3, "basis": 4}[args.path])
    for kv in args.opt:
        k, v = kv.split("=")
        eng.set_option(k, int(v))
    # a non-default stream: the library treats a NULL handle as "use the context's own stream",
    # and CUDA events must be recorded on the stream the kernels are launched on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)

    # this rank's shard of the global proposal batch (global ids rank*B .. rank*B+B-1)
    rng = np.random.default_rng(31337 + rank)
    Z_host = torch.from_numpy((zs * rng.standard_normal((B, prob.M))).astype(np.float32)).pin_memory()   # (B, M) row-major == M x B col-major
    Z_np = Z_host.numpy().T                                  # the M x B column-major view the host-pointer call takes (pinned memory)
    dZ = Z_host.to(dev)
    d_lp = torch.empty(B, dtype=torch.float64, device=dev)
    d_lp_all = torch.empty(B * world, dtype=torch.float64, device=dev) if world > 1 else None

    mh = args.workload.endswith(("-mh", "-mala"))
    mh_kind = "mala" if args.workload.endswith("-mala") else "rwmh"
    MH_STEPS = MH_STEPS_BY_WORKLOAD.get(args.workload, 100)
    d_tr_all = None
    units_per_eval_batch = MH_STEPS if mh else 1
    if mh:
        d_lp_tr = torch.empty(B * MH_STEPS, dtype=torch.float64, device=dev)      # lp trace (n_chains x n_steps), stays on the device
        d_z_tr = torch.empty(prob.M * B * MH_STEPS, dtype=torch.float32, device=dev)
        d_lp = d_lp_tr[B * (MH_STEPS - 1):]
        if world > 1:      # every rank ends up with all chains' samples and log-probs (SURVEY 8e: the only collectives)
            d_tr_all = (torch.empty(world * d_z_tr.numel(), dtype=torch.float32, device=dev),
                        torch.empty(world * d_lp_tr.numel(), dtype=torch.float64, device=dev))
    timeline = []                       # (before compute, after compute, after gather) event triples of the timed steps

    def gather_device():
        if world > 1:
            if mh:
                dist.all_gather_into_tensor(d_tr_all[0], d_z_tr)
                dist.all_gather_into_tensor(d_tr_all[1], d_lp_tr)
            else:
                dist.all_gather_into_tensor(d_lp_all, d_lp)

    def step_device(record=False):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if record else None
        if record:
            ev[0].record(stream)
        if mh:
            eng.mh_run_dev(B, MH_STEPS, 2024, sigma_z=zs, sigma_m=sigma_m, chain_offset=rank * B, d_z0=dZ.data_ptr(),
                           d_z_trace=d_z_tr.data_ptr(), d_lp_trace=d_lp_tr.data_ptr(), kind=mh_kind)
        else:
            eng.logpost_dev(dZ.data_ptr(), B, d_lp.data_ptr(), sigma_m=sigma_m)
        if record:
            ev[1].record(stream)
        gather_device()
        if record:
            ev[2].record(stream)
            timeline.append(ev)

    e2e_out = {}

    def step_e2e():
        """The call a user of the reference-facing API makes: HOST buffers in, HOST results out (ssi_logpost_batch / ssi_mh_run copy
        host -> device, run the kernels and copy the results back before they return), then the gather of the results."""
        if mh:
            zt, lt, _ = eng.mh_run(B, MH_STEPS, 2024, sigma_z=zs, sigma_m=sigma_m, chain_offset=rank * B, z0=Z_np, want_accept=False, kind=mh_kind)
            e2e_out["lp0"] = float(lt[0, 0])
            if world > 1:
                d_z_tr.copy_(torch.from_numpy(zt.reshape(-1, order="F")), non_blocking=True)
                d_lp_tr.copy_(torch.from_numpy(lt.reshape(-1, order="F")), non_blocking=True)
        else:
            lp = eng.logpost(Z_np, sigma_m)
            e2e_out["lp0"] = float(lp[0])
            if world > 1:
                d_lp.copy_(torch.from_numpy(lp), non_blocking=True)
        gather_device()
        stream.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        step_device()
    launches0 = eng.stats().kernel_launches
    # the library brackets every launch of the path's dominant kernel with CUDA events on the launching stream
    eng.set_option("time_dominant", 1)
    with ClockSampler(local_rank) as clk:
        ms_dev = timed(lambda: step_device(record=True), args.steps)
    eng.sync()
    if args.dump_outputs and rank == 0:
        if mh:
            z, lp = d_tr_all if world > 1 else (d_z_tr, d_lp_tr)
            z, lp = mh_traces(z.cpu().numpy(), lp.cpu().numpy(), world, B, MH_STEPS, prob.M)
            dump_outputs(args.dump_outputs, {"z_trace": (z, 1), "lp_trace": (lp, 0)})
        else:
            dump_outputs(args.dump_outputs, {"lp": ((d_lp_all if world > 1 else d_lp).cpu().numpy(), 0)})
    st = eng.stats()
    dom_ms, dom_n = st.dominant_ms, st.dominant_launches
    eng.set_option("time_dominant", 0)
    launches = st.kernel_launches - launches0
    path_used = ssi.PATH_NAMES[st.last_path]
    clocks = clk.summary()
    # per-step split of the device time: compute | NCCL gather (max over ranks), and every rank's clocks
    tl = torch.tensor([[ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])] for ev in timeline], dtype=torch.float64, device=dev)
    clocks_all = [clocks]
    if world > 1:
        dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        clocks_all = [None] * world
        dist.all_gather_object(clocks_all, clocks)
    step_e2e()
    e2e_steps = min(args.steps, 3)
    ms_e2e = timed(step_e2e, e2e_steps)

    # sanity: the timed path produced the oracle's numbers (one sample, checked after timing), through BOTH entry points
    if rank == 0:
        sys.path.insert(0, str(ROOT / "oracle"))
        import ssi_oracle as orc
        ref = orc.density(orc.Problem(prob.dims, prob.acts, prob.X, prob.Y, prob.W_swa, prob.P),
                          Z_host[0].numpy().astype(np.float64), sigma_m)
        got_dev = float((d_lp_tr if mh else d_lp)[0].item())          # MH: trace entry (chain 0, step 0) = lp(z0)
        for got in (got_dev, e2e_out["lp0"]):
            if not np.isfinite(got) or abs(got - ref) > 1e-5 * abs(ref):
                raise SystemExit(f"bench result mismatch vs oracle: {got} vs {ref}")

    line = None
    if rank == 0:
        peaks = load_peaks()
        units_step = float(B) * world * prob.N * units_per_eval_batch
        flops_unit = 2.0 * sum(a * b for a, b in zip(prob.dims[:-1], prob.dims[1:])) + 2.0 * prob.n * prob.M / prob.N
        value = units_step * args.steps / (ms_dev * 1e-3)
        e2e = units_step * e2e_steps / (ms_e2e * 1e-3)
        per_gpu_flops = flops_unit * B * prob.N * units_per_eval_batch * args.steps / (ms_dev * 1e-3)
        peak_tf = peaks["bf16_tflops_sustained"]
        sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
        # dominant kernel (rank 0): its own algorithmic flops per launch over its own average launch time
        dims = prob.dims
        if path_used == "tensor":      # k_tc_layer<FUSED>: every Dense layer after the first (the first is the basis-layer stream)
            dom_name = "k_tc_layer<FUSED>: Dense layers 2..L as tcgen05 split-precision GEMM (3 MMAs per product) + fused output layer + squared error"
            dom_flops_unit = 2.0 * sum(a * b for a, b in zip(dims[1:-1], dims[2:]))
        else:
            dom_name = {"basis": "BASIS path (first layer affine in z): k_b1_mma on the tensor cores for the density, k_logpost_basis1h_grad "
                                 "on CUDA cores for value+gradient (MALA)",
                        "fused": "k_logpost_fused: whole chain per (sample, datapoint)"}.get(path_used, path_used)
            dom_flops_unit = flops_unit
        units_launch = float(B) * prob.N * units_per_eval_batch * args.steps / max(dom_n, 1)
        dom_avg_ms = dom_ms / max(dom_n, 1)
        dom_tf = dom_flops_unit * units_launch / (dom_avg_ms * 1e-3) / 1e12 if dom_n else None
        traffic, traffic_src = None, None
        tfile = ROOT / "profiles" / "traffic.json"       # dram__bytes_read+write per launch from the committed ncu --set full capture
        if tfile.exists():
            ent = json.loads(tfile.read_text()).get(f"{args.workload}:{path_used}", {})
            traffic, traffic_src = ent.get("bytes_per_launch"), ent.get("source")
        h2d = int(Z_host.numel() * 4)
        d2h = int((B * MH_STEPS * 8 + prob.M * B * MH_STEPS * 4) if mh else B * 8)
        line = {
            "metric": "log-posterior evals/sec (samples x datapoints)", "value": value, "unit": "sample*datapoint/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, B, world),
            "path": path_used,
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "sample*datapoint/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps,
                    "call": ("ssi_mh_run" if mh_kind == "rwmh" else "ssi_mala_run") if mh else "ssi_logpost_batch",
                    "note": "host-pointer C-ABI call: Z from (pinned) host memory, results into host memory, every step; N > 1 adds the "
                            "H2D of the results and the NCCL gather the sampler needs"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": dom_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (dom_tf / peak_tf) if dom_tf else None, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": dom_name, "launches": int(dom_n), "avg_launch_ms": dom_avg_ms,
                         "share_of_step": dom_ms / ms_dev if ms_dev else None,
                         "flops_per_unit": dom_flops_unit, "units_per_launch": units_launch,
                         "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']}); kernel timed inside a long step",
                         "note": "algorithmic FP32 flops of this kernel (padding not counted). FP32-grade results need 3 16-bit MMAs "
                                 "per product (hi*hi + hi*lo + lo*hi), so the tensor pipe executes 3x this figure: "
                                 "mma_frac = 3*frac is the share of the BF16 peak the kernel keeps busy",
                         "mma_frac": (3.0 * dom_tf / peak_tf) if (dom_tf and path_used == "tensor") else None,
                         # a 13-50-1 net has no GEMM to speak of: against the FP32 CUDA-core peak (128 FMA/clk/SM at the maximum SM
                         # clock) the same figure reads as follows (> 1 is possible because the first layer runs on the tensor cores)
                         "frac_of_fp32_simt_peak": ((dom_tf / (sm_count * 128 * 2 * clocks["sm_max_mhz"] * 1e6 / 1e12))
                                                    if (dom_tf and path_used != "tensor" and clocks.get("sm_max_mhz")) else None)},
            # the whole step (all kernels of the path), full algorithmic flops per unit incl. the first layer and the projection
            "step_roofline": {"achieved": per_gpu_flops / 1e12, "peak": peak_tf, "unit": "TFLOP/s", "frac": per_gpu_flops / 1e12 / peak_tf,
                              "flops_per_unit": flops_unit, "per": "GPU",
                              # SURVEY 8(d): the fraction against every denominator, so that no choice is hidden.  Split
                              # precision issues three 16-bit MMAs per FP32-grade product, so peak/3 is the honest ceiling for
                              # the GEMM layers (the first layer and the projection are not GEMMs here, which is how the step
                              # can exceed it).
                              "frac_of": {"bf16_sustained": per_gpu_flops / 1e12 / peak_tf,
                                          "bf16_burst": per_gpu_flops / 1e12 / peaks.get("bf16_tflops", peak_tf),
                                          "bf16_sustained_div3_split_precision": 3.0 * per_gpu_flops / 1e12 / peak_tf}},
            "timeline": {"compute_ms_per_step": [float(v) for v in tl[:, 0]], "gather_ms_per_step": [float(v) for v in tl[:, 1]],
                         "note": "CUDA events on the launching stream around the compute and around the NCCL gather of every timed step, max over ranks",
                         "clocks_per_rank": clocks_all},
        }
    extras = not args.no_extras
    # ---- BASELINE configs[4] per GPU, with the collective timed on its own (all ranks take part) ----
    if extras and name == "wide":
        sec = mh_c5_section(ssi, torch, dist, eng, prob, dev, rank, world, stream)
        if rank == 0:
            line["mh_c5"] = sec
    eng.close()
    del dZ, d_lp, d_lp_all, d_tr_all
    torch.cuda.empty_cache()
    if rank == 0 and extras:
        line["streams"] = streams_section(ssi, torch, dev, local_rank, load_peaks())
        torch.cuda.empty_cache()
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=host_group)     # every rank has released its device memory (host-side wait: the GPUs stay idle)
        if rank == 0 and extras:
            try:
                line["multi_device_ctx"] = multi_ctx_section(ssi, torch, prob, world, B if not mh else B, sigma_m, zs, 1)
            except Exception as ex:        # reported, never fatal for the headline line
                line["multi_device_ctx"] = {"error": str(ex)[:300]}
        dist.barrier(group=host_group)
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_reference(args.workload, budget_s=15.0)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "host_cpus", "kind", "sample", "numpy_openblas", "torch_f64")}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
