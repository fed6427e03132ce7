"""Every kernel family ssi_launch_gemm (ssi_gemm.cu) picks for the gradient and training paths, at the shapes where it
picks it, against the Float64 oracle: narrow heads and bottleneck layers on the skinny kernels, the tensor-core GEMM right
after a bottleneck, and the thresholds between the families.

Dispatch, per GEMM and per batch (never per launch, so that a sample's result cannot depend on the rest of its batch):
  skinny   O.J.K >= 1e6 and
             forward           O <= 16, J >= 1024, O.K floats <= 160 KB   k_gemm_skinny_fwd  (bias + activation epilogue)
             back-propagation  K <= 16, O >= 64, J >= 64                  k_gemm_skinny_k    (activation-derivative epilogue)
             weight gradient   O <= 16, J >= 64, K >= 1024                k_gemm_skinny_gw + _fin (32 ordered slices)
           each as <4> (the narrow side <= 4) or <16>;
  tc       O.J.K >= 1.6e7, J >= 64, K >= 8, 16-byte aligned bases and strides       k_gemm_tc
  simt     everything else                                                          k_gemm_simt
For a layer l of width out after width in, over nb datapoints: forward (O, J, K) = (out, nb, in), weight gradient
(out, in, nb), back-propagation into layer l-1 (in, nb, out).  Per training step and per logpost_grad call (one launch for
all B samples), with "-" for the first layer, which has no back-propagation:

  case                        acts                    nb    forward            weight gradient     back-propagation
  64-1024-1024-1              relu tanh id           1025  tc tc fwd<4>       tc tc gw<4>         -  tc  k<4>  (tanh')
      head forward J = 1025 >= 1024, head weight gradient K = 1025 >= 1024, O.J.K = 1.05e6 >= 1e6: tc 5, skinny 3
  64-1024-1024-1              relu tanh id           1023  tc tc simt         tc tc simt          -  tc  k<4>
      J = K = 1023 < 1024 and 1.05e6 < 1.6e7: the head forward and weight gradient go to SIMT: tc 5, skinny 1
  64-1024-1024-O, O = 2..4    relu tanh sig/relu/tanh 1536 tc tc fwd<4>       tc tc gw<4>         -  tc  k<4>
                  O = 5, 16   relu tanh id           1536  tc tc fwd<16>      tc tc gw<16>        -  tc  k<16>
      tc 5, skinny 3.  At O = 16 the head GEMMs would qualify for k_gemm_tc too (2.5e7, aligned): skinny is tried first
                  O = 17      relu tanh id           1536  tc tc simt         tc tc simt          -  tc  simt
      17 > 16 leaves the skinny kernels, and a leading dimension of 17 floats is not 16-byte aligned: tc 5, skinny 0
  32-4096-4                   relu id                1100  tc fwd<4>          simt gw<4>          -  k<4>  (relu')
      the head forward stages 4 x 4096 floats = 64 KB of A (over the 48 KB default); the first weight gradient has
      J = 32 < 64: tc 1, skinny 3
  256-1024-12-1024-10         relu tanh relu id      1536  tc fwd<16> tc fwd<16>  tc gw<16> simt gw<16>  -  k<16> tc k<16>
      fwd<16> with tanh into the bottleneck; k_gemm_tc out of it with K = 12 (one partial k-block) and back into it with
      O = 12 (one partial row tile) + tanh'; W3's gradient has J = 12 < 64; the k<16> take relu': tc 4, skinny 6
  256-1024-4-1024-3           relu sig relu id       1536  tc fwd<4> simt fwd<4>  tc gw<4> simt gw<4>    -  k<4> simt k<4>
      out of the bottleneck K = 4 < 8; back into it O.J.K = 6.3e6 < 1.6e7: tc 2, skinny 6
(the sizes keep O.J.K above 1e6 for every skinny launch; the simt column with option gemm_simt is every launch.)
The counters ssi_stats_t.gemm_tc_launches / gemm_skinny_launches pin this table: a later change of a threshold fails here
instead of quietly moving a case off the kernel it was written for.

Training step: each block (W_l, b_l) read through `probe_grad` against `orc.mse_loss_and_grad`, on the default kernels and
with every GEMM on SIMT.  logpost_grad: B = 5 samples (batched operands, per-sample scales, blockIdx.y/z > 0 in the skinny
kernels) with masks 1 and 7.  A block's error cannot be read from grad_z = P' grad_W with a dense P: a 1025-parameter head
in a 1.1M-parameter net contributes only its share.  So P is block-isolating: every column is Gaussian on the rows of one
parameter block and zero elsewhere, the columns dealt round-robin over the blocks; rms_m(grad_dev - grad_ref) /
rms_m(grad_ref) over a block's columns then estimates that block's relative error, since E[(P_m' x)^2] ~ |x|^2 for a
Gaussian P_m.  M = 64 (8 or more columns per block) on the bottlenecks and on 32-4096-4; M = 1 (one dense column: both
ends of the split grad_z GEMM and k_grad_finish) on the scalar head.

Bars (as in test_gpu_train_scale.py): 5e-5 of the block norm on every kernel; on the default kernels at most 2.5x the SIMT
error plus TC_TRUNCATION for a block whose reverse pass runs through k_gemm_tc (its weight gradient, or a back-propagation
above it), else plus SKINNY_FLOOR.

Measured on one B200 at its 1000 W power limit, worst block error relative to the block norm, default kernels / SIMT:
  training step: blocks through k_gemm_tc 7.6e-6 / 9.1e-7; the others (skinny or SIMT reverse pass) 2.3e-6 / 8.6e-7, and
  6.5e-7 / 6.5e-7 where no tensor-core forward over K = 1024 feeds them (32-4096-4, the bottlenecks' upper layers).
  logpost_grad, per-block estimates with M = 64: 7.0e-6 / 2.7e-6 through k_gemm_tc, 3.5e-6 / 3.0e-6 otherwise; one dense
  column (scalar head): 1.95e-5 / 4.7e-6.  Loss within 1.2e-7, value within 1.8e-7.  The file runs in about 12 s.
Each of these single-line faults fails training and logpost_grad cases here: k_gemm_skinny_fwd without the activation,
or dropping each block's last datapoint; k_gemm_skinny_k skipping a block's last partial group of eight datapoints, or
without the activation derivative; k_gemm_skinny_gw_fin summing 31 of the 32 slices.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import pytest

import ssi_oracle as orc
from conftest import stable_seed
from train_probe import BLOCK_BAR, LOSS_RTOL, RELU_BAND, TC_OVER_SIMT, TC_TRUNCATION, block_errors, probe_grad, problem

pytestmark = pytest.mark.gpu

# Blocks whose reverse pass stays off k_gemm_tc (skinny or SIMT kernels: FP32, round to nearest) may exceed 2.5x the SIMT
# error by this much.  Measured: at most 1.25e-6, and only downstream of a tensor-core forward over K = 1024 -- head17, which
# runs no skinny kernel, shows the same 1.05e-6; without such a forward the skinny blocks are 0.2-1.8x the SIMT error.
SKINNY_FLOOR = 2e-6
LP_RTOL = 1e-5
B_SAMPLES = 5


@dataclass(frozen=True)
class Case:
    name: str
    dims: tuple
    acts: tuple
    nb: int
    fwd: tuple          # kernel of each layer's forward GEMM
    gw: tuple           # ... weight gradient
    bp: tuple           # ... back-propagation through the layer into the previous one's output (None for the first)

    @property
    def launches(self):
        """(k_gemm_tc, k_gemm_skinny_*) launches per step."""
        ks = [k for k in self.fwd + self.gw + self.bp if k]
        return sum(k == "tc" for k in ks), sum(k not in ("tc", "simt") for k in ks)

    def floor(self, block):
        """TC_TRUNCATION when the block's reverse pass runs through k_gemm_tc, else SKINNY_FLOOR."""
        l = int(block[1:]) - 1
        chain = list(self.bp[l + 1:]) + ([self.gw[l]] if block[0] == "W" else [])
        return TC_TRUNCATION if "tc" in chain else SKINNY_FLOOR


def _head(O, act, fam):
    return Case(f"head{O}", (64, 1024, 1024, O), (orc.ACT_RELU, orc.ACT_TANH, act), 1536,
                ("tc", "tc", f"fwd{fam}"), ("tc", "tc", f"gw{fam}"), (None, "tc", f"k{fam}"))


SCALAR = Case("scalar_head", (64, 1024, 1024, 1), (1, 2, 0), 1025, ("tc", "tc", "fwd4"), ("tc", "tc", "gw4"), (None, "tc", "k4"))
SCALAR_BELOW = Case("scalar_head_below_thresholds", (64, 1024, 1024, 1), (1, 2, 0), 1023,
                    ("tc", "tc", "simt"), ("tc", "tc", "simt"), (None, "tc", "k4"))
HEADS = [_head(2, orc.ACT_SIGMOID, 4), _head(3, orc.ACT_RELU, 4), _head(4, orc.ACT_TANH, 4), _head(5, orc.ACT_IDENTITY, 16),
         _head(16, orc.ACT_IDENTITY, 16),
         Case("head17", (64, 1024, 1024, 17), (1, 2, 0), 1536, ("tc", "tc", "simt"), ("tc", "tc", "simt"), (None, "tc", "simt"))]
WIDE4 = Case("fwd4_over_48KB", (32, 4096, 4), (1, 0), 1100, ("tc", "fwd4"), ("simt", "gw4"), (None, "k4"))
BOTTLENECK = Case("bottleneck", (256, 1024, 12, 1024, 10), (1, 2, 1, 0), 1536,
                  ("tc", "fwd16", "tc", "fwd16"), ("tc", "gw16", "simt", "gw16"), (None, "k16", "tc", "k16"))
BOTTLENECK4 = Case("bottleneck4", (256, 1024, 4, 1024, 3), (1, 3, 1, 0), 1536,
                   ("tc", "fwd4", "simt", "fwd4"), ("tc", "gw4", "simt", "gw4"), (None, "k4", "simt", "k4"))
CASES = [SCALAR, SCALAR_BELOW, *HEADS, WIDE4, BOTTLENECK, BOTTLENECK4]


def _launches(engine):
    s = engine.stats()
    return np.array([s.gemm_tc_launches, s.gemm_skinny_launches])


def _check_blocks(label, case, err_d, err_s):
    """Print every block's error per mode, then hold it to the bars."""
    for (name, ed), (_, es) in zip(err_d, err_s):
        fl = case.floor(name) if name[0] in "Wb" else (TC_TRUNCATION if case.launches[0] else SKINNY_FLOOR)
        print(f"  {name:>6}: default {ed:.2e}  SIMT {es:.2e}  ratio {ed / es:.2f}  "
              f"({'tc' if fl == TC_TRUNCATION else 'fp32'} floor)")
    for (name, ed), (_, es) in zip(err_d, err_s):
        fl = case.floor(name) if name[0] in "Wb" else (TC_TRUNCATION if case.launches[0] else SKINNY_FLOOR)
        assert es < BLOCK_BAR, (label, name, "simt", es)
        assert ed < BLOCK_BAR and ed <= TC_OVER_SIMT * es + fl, (label, name, ed, es, fl)


def _check_training(engine, case, W0, X, Y, batch, label):
    cols = np.arange(batch[0], batch[0] + batch[1]) if isinstance(batch, tuple) else np.asarray(batch)
    loss_ref, g_ref = orc.mse_loss_and_grad(W0, case.dims, case.acts, X[:, cols], Y[:, cols])
    res = {}
    for mode in ("default", "simt"):
        engine.set_option("gemm_simt", int(mode == "simt"))
        before = _launches(engine)
        loss, g, W1 = probe_grad(engine, W0, batch)
        n = (_launches(engine) - before) / 2            # probe_grad takes two steps
        res[mode] = (loss, block_errors(g, g_ref, case.dims), tuple(int(v) for v in n), W1)
    engine.set_option("gemm_simt", 0)
    (loss_d, err_d, n_d, W1_d), (loss_s, err_s, n_s, _) = res["default"], res["simt"]
    print(f"\n{label}: loss rel err default {abs(loss_d / loss_ref - 1):.1e} simt {abs(loss_s / loss_ref - 1):.1e}; "
          f"launches per step (tc, skinny) {n_d}, under gemm_simt {n_s}")
    _check_blocks(label, case, err_d, err_s)
    assert n_d == case.launches and n_s == (0, 0), (n_d, n_s, case.launches)
    for mode, loss in (("default", loss_d), ("simt", loss_s)):
        assert abs(loss / loss_ref - 1) <= LOSS_RTOL, (mode, loss, loss_ref)
    return W1_d


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c.name}-nb{c.nb}")
def test_training_step(engine, case):
    """One training step per case as a window batch (and, on the scalar head, as a shuffled index batch): every block on
    the default kernels and on SIMT against the oracle, and the launches of each kernel family per step."""
    N = case.nb + 70
    W0, X, Y = problem(case.dims, case.acts, N, stable_seed("dispatch", case.name, case.nb))
    engine.set_model(case.dims, case.acts)
    engine.set_data(X, Y)
    _check_training(engine, case, W0, X, Y, (37, case.nb), f"{case.name} nb={case.nb} window")
    if case is SCALAR:
        idx = np.random.default_rng(5).permutation(N)[:case.nb]
        _check_training(engine, case, W0, X, Y, idx, f"{case.name} nb={case.nb} index batch")


def _block_isolating_subspace(rng, W_swa, dims, M):
    """P (n, M) whose column m is Gaussian on the rows of parameter block m % (2L) and zero elsewhere, scaled so that P z
    with z ~ N(0, 0.25) moves a block by ~5 % of its rms; with M < 2L, one dense column scaled block by block.
    Returns P and [(name, columns)] (one group of all columns when P is dense)."""
    offs = orc.layer_offsets(dims)
    blocks = [(f"{k}{l + 1}", lo, hi) for l, (w, b, _, out) in enumerate(offs) for k, lo, hi in (("W", w, b), ("b", b, b + out))]
    P = np.zeros((W_swa.size, M), np.float32)
    dense = M < len(blocks)
    groups = [("P dense", np.arange(M))] if dense else [(name, np.arange(i, M, len(blocks))) for i, (name, _, _) in enumerate(blocks)]
    for i, (name, lo, hi) in enumerate(blocks):
        cols = np.arange(M) if dense else np.arange(i, M, len(blocks))
        scale = 0.1 * np.sqrt(np.mean(W_swa[lo:hi].astype(np.float64) ** 2) / len(cols))
        P[lo:hi, cols] = scale * rng.standard_normal((hi - lo, len(cols)))
    return P, groups


def _clear_relu_band(W_swa, P, Z, dims, acts, X, rng):
    """`problem`'s relu band at every sample point W_swa + P z_b at once: the bias (in W_swa) of every relu unit whose Float64
    pre-activation comes within RELU_BAND of 0 at any sample and datapoint is drawn again, layer by layer.  (Redrawing z
    instead would not end: a sample has ~1.5M relu pre-activations, and moving them all moves ~100 into the band.)"""
    D = P.astype(np.float64) @ Z.astype(np.float64)
    hs = [X.astype(np.float64)] * Z.shape[1]
    for (w_off, b_off, din, dout), act in zip(orc.layer_offsets(dims), acts):
        Ws = [(W_swa[w_off:b_off].astype(np.float64) + D[w_off:b_off, s]).reshape(din, dout).T for s in range(len(hs))]
        b = W_swa[b_off:b_off + dout]

        def pre(rows):
            return [Ws[s][rows] @ hs[s] + (b[rows].astype(np.float64) + D[b_off + rows, s])[:, None] for s in range(len(hs))]

        full = pre(np.arange(dout))
        if act == orc.ACT_RELU:
            redo = np.flatnonzero(np.min([np.abs(p).min(axis=1) for p in full], axis=0) < RELU_BAND)
            while len(redo):
                b[redo] = rng.uniform(-0.1, 0.1, len(redo))
                sub = pre(redo)
                for p, q in zip(full, sub):
                    p[redo] = q
                redo = redo[np.min([np.abs(q).min(axis=1) for q in sub], axis=0) < RELU_BAND]
        hs = [orc._activate(p, act) for p in full]


@pytest.mark.parametrize("mask", [1, 7])
@pytest.mark.parametrize("case,M", [(SCALAR, 1), (SCALAR_BELOW, 1), (WIDE4, 64), (BOTTLENECK, 64), (BOTTLENECK4, 64)],
                         ids=lambda v: f"{v.name}-nb{v.nb}" if isinstance(v, Case) else f"M{v}")
def test_logpost_grad(engine, case, M, mask):
    """logpost_grad on B = 5 samples, N = the case's nb: value within 1e-5 and every block of the gradient against the
    oracle on the default kernels and on SIMT, the launches per call, and a sample alone equal bit for bit to the same
    sample inside the batch."""
    dims, acts, N = case.dims, case.acts, case.nb
    W_swa, X, Y = problem(dims, acts, N, stable_seed("dispatch-lp", case.name, case.nb, mask))
    rng = np.random.default_rng(stable_seed("dispatch-P", case.name, case.nb, mask))
    P, groups = _block_isolating_subspace(rng, W_swa, dims, M)
    Z = (0.5 * rng.standard_normal((M, B_SAMPLES))).astype(np.float32)
    _clear_relu_band(W_swa, P, Z, dims, acts, X, rng)
    prob = orc.Problem(dims, acts, X, Y, W_swa, P)
    engine.set_model(dims, acts)
    engine.set_data(X, Y)
    engine.set_subspace(W_swa, P)
    sm, sp, sz = 0.8, 1.5, 2.0
    out = {}
    for mode in ("default", "simt"):
        engine.set_option("gemm_simt", int(mode == "simt"))
        before = _launches(engine)
        lp, g = engine.logpost_grad(Z, sm, sp, sz, mask)
        out[mode] = (lp, g, tuple(int(v) for v in _launches(engine) - before))
    engine.set_option("gemm_simt", 0)
    worst = {mode: {name: 0.0 for name, _ in groups} for mode in out}
    lp_err = {mode: 0.0 for mode in out}
    for s in range(B_SAMPLES):
        lp_ref, g_ref = orc.density_and_grad(prob, Z[:, s].astype(np.float64), sm, sp, sz, mask)
        for mode, (lp, g, _) in out.items():
            lp_err[mode] = max(lp_err[mode], abs(lp[s] / lp_ref - 1))
            for name, cols in groups:
                e = np.sqrt(np.mean((g[cols, s] - g_ref[cols]) ** 2) / np.mean(g_ref[cols] ** 2))
                worst[mode][name] = max(worst[mode][name], e)
    label = f"{case.name} nb={N} logpost_grad M={M} mask {mask}"
    print(f"\n{label}: lp rel err default {lp_err['default']:.1e} simt {lp_err['simt']:.1e}; launches per call (tc, skinny) "
          f"{out['default'][2]}, under gemm_simt {out['simt'][2]}")
    _check_blocks(label, case, list(worst["default"].items()), list(worst["simt"].items()))
    assert out["default"][2] == case.launches and out["simt"][2] == (0, 0)
    assert lp_err["default"] <= LP_RTOL and lp_err["simt"] <= LP_RTOL, lp_err
    lp1, g1 = engine.logpost_grad(Z[:, 4:5], sm, sp, sz, mask)
    np.testing.assert_array_equal(g1[:, 0], out["default"][1][:, 4])
    assert lp1[0] == out["default"][0][4]
