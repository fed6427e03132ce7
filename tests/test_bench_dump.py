"""bench.py --dump-outputs (host logic only): the gathered MH traces come out in mh_run's shapes with the global chain
order, and a dump over the size limit keeps the same chains of every array."""
import numpy as np

import bench


def test_mh_traces_match_mh_run_layout():
    rng = np.random.default_rng(0)
    world, chains, steps, M = 3, 5, 4, 2
    z_ranks = [rng.standard_normal((M, chains, steps)).astype(np.float32) for _ in range(world)]
    lp_ranks = [rng.standard_normal((chains, steps)) for _ in range(world)]
    z_flat = np.concatenate([z.reshape(-1, order="F") for z in z_ranks])        # all_gather_into_tensor: rank blocks in order
    lp_flat = np.concatenate([lp.reshape(-1, order="F") for lp in lp_ranks])
    z, lp = bench.mh_traces(z_flat, lp_flat, world, chains, steps, M)
    np.testing.assert_array_equal(z, np.concatenate(z_ranks, axis=1))
    np.testing.assert_array_equal(lp, np.concatenate(lp_ranks, axis=0))


def test_dump_outputs_whole_and_sampled(tmp_path, monkeypatch):
    z = np.arange(2 * 100 * 3, dtype=np.float32).reshape(2, 100, 3)
    lp = np.arange(100 * 3, dtype=np.float64).reshape(100, 3)
    bench.dump_outputs(tmp_path / "all", {"z_trace": (z, 1), "lp_trace": (lp, 0)})
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "z_trace.npy"), z)
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "lp_trace.npy"), lp)
    monkeypatch.setattr(bench, "DUMP_LIMIT", (z.nbytes + lp.nbytes) // 4)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, {"z_trace": (z, 1), "lp_trace": (lp, 0)})
    zs, ls = np.load(tmp_path / "a" / "z_trace.npy"), np.load(tmp_path / "a" / "lp_trace.npy")
    assert zs.nbytes + ls.nbytes <= bench.DUMP_LIMIT and ls.shape[0] == zs.shape[1] == 25
    ids = (ls[:, 0] / 3).astype(int)                       # lp[c, 0] == 3 c: the chains kept
    np.testing.assert_array_equal(zs, z[:, ids])
    assert np.all(np.diff(ids) > 0)
    np.testing.assert_array_equal(np.load(tmp_path / "b" / "z_trace.npy"), zs)       # a fixed sample
