"""Reading the on-device training step's FP32 gradient and holding it to the Float64 oracle, for the GPU tests.

The library has no gradient readback, and none is needed: a Descent step computes W1 = float((double)W0 - eta * (double)G)
(ssi_train.cu, k_train_update), so g = (W0 - W1) / eta in Float64 recovers the device's FP32 gradient G to about 2^-24
relative wherever eta |G| >> |W0| (`probe_grad`).  `block_errors` then compares it with `ssi_oracle.mse_loss_and_grad`
block by block (every W_l and b_l), and `problem` builds training data whose relu decisions the device cannot flip.
Like the rest of the oracle it is test infrastructure: nothing in the product path imports it.
"""
from __future__ import annotations

import numpy as np

import ssi_oracle as orc

BLOCK_BAR = 5e-5            # per-block error, relative to the block norm
TC_OVER_SIMT = 2.5          # tensor-core error no worse than this multiple of the FP32 SIMT error ...
# ... plus the truncation of k_gemm_tc's FP32 accumulator: every MMA's add rounds toward zero, six adds per 32-wide k-block,
# and the accumulator is drained every 32 k-blocks.  Measured: the error is linear in the chunk length (halved at 16), and
# systematic, so the row sums of the bias gradients keep it (SIMT rounds to nearest: 1e-7 to 5e-7 on these shapes).
TC_TRUNCATION = 32 * 6 * 2.0 ** -24
RELU_BAND = 3e-5            # no relu pre-activation of the data sets below comes closer than this to 0
LOSS_RTOL = 1e-5


def problem(dims, acts, N, seed):
    """Training data as profiles/bench_streams.py builds it for C4: X uniform in [0, 1), Y standard normal.  The weights
    are Flux's glorot init with biases drawn uniform in [-0.1, 0.1), so that every bias term of the epilogues counts.

    relu is not differentiable at 0: a pre-activation within FP32 rounding of 0 can take the other branch on the device,
    and one such flip moves a whole block's gradient by ~1e-3 of its norm (one element of delta_l against a sum of nb
    rank-one terms).  So the bias of every relu unit whose pre-activation comes within RELU_BAND of 0 on any datapoint is
    drawn again, layer by layer in Float64, until none does."""
    rng = np.random.default_rng(seed)
    W0 = orc.glorot_flat(rng, dims)
    X = rng.random((dims[0], N), dtype=np.float32)
    Y = rng.standard_normal((dims[-1], N)).astype(np.float32)
    h = X.astype(np.float64)
    for (w_off, b_off, din, dout), act in zip(orc.layer_offsets(dims), acts):
        W = W0[w_off:b_off].reshape(din, dout).T.astype(np.float64)
        b = W0[b_off:b_off + dout]
        b[:] = rng.uniform(-0.1, 0.1, dout)
        pre = W @ h + b.astype(np.float64)[:, None]
        redo = np.flatnonzero(np.abs(pre).min(axis=1) < RELU_BAND) if act == orc.ACT_RELU else []
        while len(redo):
            b[redo] = rng.uniform(-0.1, 0.1, len(redo))
            pre[redo] = W[redo] @ h + b[redo].astype(np.float64)[:, None]
            redo = redo[np.abs(pre[redo]).min(axis=1) < RELU_BAND]
        h = orc._activate(pre, act)
    return W0, X, Y


def probe_grad(engine, W0, batch, want_loss=True):
    """(loss, g, W1): the FP32 gradient the device's training step computes at W0 on `batch`, read through one Descent step.

    A first step at eta = 1 gives max |G| to FP32 precision; the probe step is then the power of two that puts
    eta max|G| near 2^40, so that (W0 - W1) / eta is exact in Float64 apart from the one FP32 rounding of W1, and nothing
    overflows.  W1 (the probe's raw output) is returned for bitwise comparisons.  The training state is left at W0 again,
    so the caller may probe once more or begin its own run."""
    W0 = np.asarray(W0, np.float32)
    engine.train_begin(W0, "descent", 1.0)
    engine.train_step(batch)
    gmax = np.abs(W0.astype(np.float64) - engine.train_weights()).max()
    eta = 2.0 ** (40 - int(np.ceil(np.log2(gmax))))
    engine.train_begin(W0, "descent", eta)
    loss = engine.train_step(batch, want_loss=want_loss)
    W1 = engine.train_weights()
    engine.train_begin(W0, "descent", eta)
    return loss, (W0.astype(np.float64) - W1.astype(np.float64)) / eta, W1


def block_errors(g, g_ref, dims):
    """[(name, |g - g_ref| / |g_ref|)] for every W_l and b_l."""
    out = []
    for l, (w_off, b_off, din, dout) in enumerate(orc.layer_offsets(dims)):
        for name, lo, hi in ((f"W{l + 1}", w_off, b_off), (f"b{l + 1}", b_off, b_off + dout)):
            out.append((name, np.linalg.norm(g[lo:hi] - g_ref[lo:hi]) / np.linalg.norm(g_ref[lo:hi])))
    return out
