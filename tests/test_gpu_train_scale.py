"""The on-device training step (src/subspace_construction.jl:39-43) and the long-contraction GEMMs of the gradient path at
the sizes they run at, against the Float64 oracle.

The device's FP32 gradient is read through one Descent step (`probe_grad`, tests/train_probe.py) and compared block by
block (every W_l and b_l) with `ssi_oracle.mse_loss_and_grad`, on the tensor-core kernels and, beside them, with every
contraction forced onto the FP32 SIMT kernel (option gemm_simt).

What the shapes reach (ssi_grad.cu / ssi_gemm_tc.cu dispatch):
  * C4, 784-2048-2048-2048-10 relu, nb = 512 (the benched step): the three hidden forwards, three hidden weight gradients
    and two back-propagations on k_gemm_tc (8 launches).  Forward and back-propagated K = 2048 is two accumulation chunks of
    1024 k, so the running-sum read-modify-write and, on its last chunk, bias + relu or the relu derivative read late from
    the layer output.  The head runs k_gemm_skinny_k (back-propagation) and SIMT (forward, weight gradient).
  * C4 at nb = 1536: the head forward on k_gemm_skinny_fwd with 80 KB of shared memory (over the 48 KB default), the head
    weight gradient on k_gemm_skinny_gw, and hidden weight gradients over K = 1536 (two chunks); the loss sums six
    256-column partials.
  * 97-1300-1100-7 tanh/sigmoid/identity at nb = 1025: ragged o, j and k tiles; the hidden weight gradient's last chunk is a
    single k-block; the tanh back-propagation through K = 1100 takes the multi-chunk derivative epilogue; the layers that
    read X (row stride 97, not 16-byte aligned) fall back to SIMT in the same step.
  * logpost_grad on 96-1300-1100-8: the batched (per-sample operand) form of the same multi-chunk epilogues.

Measured on one B200 at its 1000 W power limit, worst block error relative to the block norm, tensor cores / SIMT:
  C4 nb = 512 (window and index batch): 1.10e-5 / 4.2e-7;  nb = 1536: 1.13e-5 / 5.9e-7;  97-1300-1100-7: 6.4e-6 / 4.9e-7.
  Loss within 2.9e-7 (tensor cores) and 1.2e-8 (SIMT) of the oracle.  ADAM: 0.24 of the per-element bar; SWA mean and
  deviations 0.31 of theirs.  logpost_grad on 96-1300-1100-8: 6.8e-7 / 1.3e-6 (mask 1), 4.2e-6 / 3.1e-6 (mask 7).
The tensor-core error is up to 64 times the SIMT error per block: it is the truncation bias of k_gemm_tc's accumulator
(TC_TRUNCATION in tests/train_probe.py; with 16-block chunks it halves), so the tensor-core bar is 2.5x the SIMT error
plus that budget.  The relu data sets are built without pre-activations near the kink (`problem`); before that, one flipped
relu decision put 2e-4 of the block norm on the first layers' gradient on SIMT and tensor cores alike.
"""
import numpy as np
import pytest

import ssi_oracle as orc
from conftest import stable_seed
from train_probe import BLOCK_BAR, LOSS_RTOL, TC_OVER_SIMT, TC_TRUNCATION, block_errors, probe_grad, problem

pytestmark = pytest.mark.gpu

C4_DIMS, C4_ACTS = (784, 2048, 2048, 2048, 10), (1, 1, 1, 0)
RAGGED_DIMS, RAGGED_ACTS = (97, 1300, 1100, 7), (2, 3, 0)


def _setup(engine, dims, acts, X, Y):
    engine.set_model(dims, acts)
    engine.set_data(X, Y)


def _columns(batch):
    if isinstance(batch, tuple):
        return np.arange(batch[0], batch[0] + batch[1])
    return np.asarray(batch)


def _check_step(engine, label, dims, acts, W0, X, Y, batch, tc_launches):
    """Probe the step on the tensor-core kernels and on SIMT; check loss and every block against the oracle."""
    cols = _columns(batch)
    loss_ref, g_ref = orc.mse_loss_and_grad(W0, dims, acts, X[:, cols], Y[:, cols])
    res = {}
    for mode in ("tc", "simt"):
        engine.set_option("gemm_simt", int(mode == "simt"))
        before = engine.stats().gemm_tc_launches
        loss, g, W1 = probe_grad(engine, W0, batch)
        launches = (engine.stats().gemm_tc_launches - before) / 2          # probe_grad takes two steps
        res[mode] = (loss, block_errors(g, g_ref, dims), launches, W1)
    engine.set_option("gemm_simt", 0)
    (loss_t, err_t, n_t, W1_t), (loss_s, err_s, n_s, _) = res["tc"], res["simt"]
    print(f"\n{label}: loss {loss_ref:.9g}, rel err tc {abs(loss_t / loss_ref - 1):.1e} simt {abs(loss_s / loss_ref - 1):.1e}; "
          f"k_gemm_tc launches per step {n_t} (simt {n_s})")
    for (name, et), (_, es) in zip(err_t, err_s):
        print(f"  {name:>4}: tensor cores {et:.2e}  SIMT {es:.2e}  ratio {et / es:.2f}")
    assert n_t == tc_launches and n_s == 0
    for mode, loss in (("tc", loss_t), ("simt", loss_s)):
        assert abs(loss / loss_ref - 1) <= LOSS_RTOL, (mode, loss, loss_ref)
    for (name, et), (_, es) in zip(err_t, err_s):
        assert es < BLOCK_BAR, (name, "simt", es)
        assert et < BLOCK_BAR and et <= TC_OVER_SIMT * es + TC_TRUNCATION, (name, et, es)
    return W1_t


@pytest.mark.parametrize("nb", [512, 1536])
def test_training_gradient_c4(engine, nb):
    """C4 (784-2048-2048-2048-10, relu, identity head) at the benched mini-batch and at one that puts the head on the skinny
    kernels, as a contiguous window and, at nb = 512, as an index batch over the same columns (the gather path).  Also:
    the window and the index batch give identical weights (same kernels: 784 * 4 bytes is 16-byte aligned), a repeated probe
    gives identical weights, and a step without the loss read back updates the weights identically."""
    W0, X, Y = problem(C4_DIMS, C4_ACTS, 4096, stable_seed("c4", nb))
    _setup(engine, C4_DIMS, C4_ACTS, X, Y)
    j0 = 1024 + 5
    W1_win = _check_step(engine, f"C4 nb={nb} window j0={j0}", C4_DIMS, C4_ACTS, W0, X, Y, (j0, nb), 8)
    _, _, W1_again = probe_grad(engine, W0, (j0, nb))
    np.testing.assert_array_equal(W1_again, W1_win)
    _, _, W1_noloss = probe_grad(engine, W0, (j0, nb), want_loss=False)
    np.testing.assert_array_equal(W1_noloss, W1_win)
    if nb == 512:
        W1_idx = _check_step(engine, f"C4 nb={nb} index batch", C4_DIMS, C4_ACTS, W0, X, Y, np.arange(j0, j0 + nb), 8)
        np.testing.assert_array_equal(W1_idx, W1_win)


@pytest.mark.parametrize("kind", ["index", "window"])
def test_training_gradient_ragged(engine, kind):
    """97-1300-1100-7 (tanh, sigmoid, identity) at an odd nb = 1025: ragged tiles on every axis, a weight gradient whose last
    accumulation chunk is one k-block, the tanh derivative after a two-chunk back-propagation, and SIMT layers (the ones that
    read X, whose row stride of 97 floats TMA cannot address) mixed into the same step."""
    N, nb = 3000, 1025
    W0, X, Y = problem(RAGGED_DIMS, RAGGED_ACTS, N, stable_seed("ragged", kind))
    _setup(engine, RAGGED_DIMS, RAGGED_ACTS, X, Y)
    batch = np.random.default_rng(3).permutation(N)[:nb] if kind == "index" else (3, nb)
    # k_gemm_tc: hidden forward (K = 1300), hidden weight gradient (K = 1025), back-propagation into the tanh layer (K = 1100)
    _check_step(engine, f"97-1300-1100-7 nb={nb} {kind}", RAGGED_DIMS, RAGGED_ACTS, W0, X, Y, batch, 3)


def test_adam_and_snapshots_teacher_forced(ssi):
    """Eight ADAM steps on C4 at nb = 512 (engine A), each checked against a Float64 ADAM step taken from A's own weights
    with the gradient A used (read by a Descent probe on engine B at the same weights and batch: the kernels are
    deterministic).  The optimiser's m and v live in FP32 on the device, so the allowed error is 1e-6 eta plus 2 ulp of W.
    A snapshot follows every step; the SWA mean and the deviation columns are checked against the Float64 recurrence."""
    W0, X, Y = problem(C4_DIMS, C4_ACTS, 4096, stable_seed("adam"))
    eta, beta, nb, steps = 1e-3, (0.9, 0.999), 512, 8
    n = orc.n_params(C4_DIMS)
    with ssi.Engine(0) as A, ssi.Engine(0) as B:
        for e in (A, B):
            _setup(e, C4_DIMS, C4_ACTS, X, Y)
        A.swa_begin(n, steps)
        A.train_begin(W0, "adam", eta, beta)
        m, v = np.zeros(n), np.zeros(n)
        W_t = W0
        snaps = []
        worst = 0.0
        for t in range(1, steps + 1):
            batch = ((t * 700) % (4096 - nb), nb)
            _, g, _ = probe_grad(B, W_t, batch)
            A.train_step(batch, want_loss=False)
            A.train_snapshot(float(t))
            W_next = A.train_weights()
            w_ref, m, v = orc.adam_step(W_t, g, m, v, t, eta, *beta)
            tol = 1e-6 * eta + 2 * np.spacing(np.abs(w_ref).astype(np.float32)).astype(np.float64)
            err = np.abs(W_next - w_ref)
            worst = max(worst, float((err / tol).max()))
            assert np.all(err <= tol), f"step {t}: {int((err > tol).sum())} elements off, worst {(err / tol).max():.2f} x the bar"
            W_t = W_next
            snaps.append(W_t)
        # the device runs the recurrence in FP32: a few roundings of the largest |W| an element has taken
        tol = 8 * np.spacing(np.max(np.abs(snaps), axis=0)).astype(np.float64)
        D = A.swa_deviations()
        assert D.shape == (n, steps)
        swa, err_dev = np.zeros(n), 0.0
        for k, W in enumerate(snaps):
            swa, dev = orc.swa_push(swa, W, float(k + 1))
            err_dev = max(err_dev, float((np.abs(D[:, k] - dev) / tol).max()))
        err_mean = float((np.abs(A.swa_mean() - swa) / tol).max())
        print(f"\nC4 ADAM {steps} steps: worst |W - W_ref| {worst:.2f} x (1e-6 eta + 2 ulp); SWA mean {err_mean:.2f}, "
              f"deviations {err_dev:.2f} x 8 ulp(max |W|)")
        assert err_mean <= 1 and err_dev <= 1


@pytest.mark.parametrize("mask", [1, 7])
def test_gradient_long_contractions(engine, mask):
    """logpost_grad on 96-1300-1100-8 (tanh, sigmoid, identity), N = 1500: per-sample operands on k_gemm_tc with two-chunk
    forward (bias + sigmoid), weight-gradient and back-propagation (tanh derivative) epilogues, against the Float64 oracle
    and against the same call on SIMT, with the bars of test_gradient_wide_on_tensor_cores."""
    dims, acts, N, M, B = (96, 1300, 1100, 8), (2, 3, 0), 1500, 6, 3
    W_swa, X, Y = problem(dims, acts, N, stable_seed("grad", mask))
    rng = np.random.default_rng(stable_seed("grad-P", mask))
    prob = orc.Problem(dims, acts, X, Y, W_swa, orc.synthetic_subspace(rng, orc.n_params(dims), M, 0.5 ** np.arange(1, M + 1)))
    engine.set_model(dims, acts)
    engine.set_data(X, Y)
    engine.set_subspace(prob.W_swa, prob.P)
    Z = (0.5 * rng.standard_normal((M, B))).astype(np.float32)
    sm, sp, sz = 0.8, 1.5, 2.0
    before = engine.stats().gemm_tc_launches
    lp, g = engine.logpost_grad(Z, sm, sp, sz, mask)
    # 2 forward layers, 2 weight gradients, 1 back-propagation into the tanh layer (the head is on the skinny kernels)
    assert engine.stats().gemm_tc_launches - before == 5
    engine.set_option("gemm_simt", 1)
    lp_s, g_s = engine.logpost_grad(Z, sm, sp, sz, mask)
    engine.set_option("gemm_simt", 0)
    worst = worst_s = 0.0
    for b in range(B):
        lp_ref, g_ref = orc.density_and_grad(prob, Z[:, b].astype(np.float64), sm, sp, sz, mask)
        nrm = np.linalg.norm(g_ref)
        worst = max(worst, np.linalg.norm(g[:, b] - g_ref) / nrm)
        worst_s = max(worst_s, np.linalg.norm(g_s[:, b] - g_ref) / nrm)
        assert abs(lp[b] - lp_ref) <= 1e-6 * abs(lp_ref) and abs(lp_s[b] - lp_ref) <= 1e-6 * abs(lp_ref)
    print(f"\n96-1300-1100-8 mask {mask} gradient: tensor cores {worst:.2e}, SIMT {worst_s:.2e} of the gradient norm")
    assert worst < 5e-5 and worst < 2.5 * worst_s
    lp1, g1 = engine.logpost_grad(Z[:, 2:3], sm, sp, sz, mask)
    np.testing.assert_array_equal(g1[:, 0], g[:, 2])
    assert lp1[0] == lp[2]
