"""bench.py --dump-outputs: the arrays written for one trackBatch result (CPU only, no device needed)."""
import os

import numpy as np

import bench
from ground_fusion_b200._lib import OBS_DTYPE


def test_dump_outputs_pads_each_frame_to_max_cnt(tmp_path):
    rng = np.random.default_rng(0)
    batch = []
    for m, p in ((3, 0), (0, 2), (6, 6)):
        obs = np.zeros(m, OBS_DTYPE)
        obs["id"] = rng.integers(0, 1000, m)
        obs["track_cnt"] = rng.integers(1, 9, m)
        obs["v"] = rng.standard_normal((m, 8))
        status = rng.integers(0, 2, p).astype(np.uint8)
        info = {"n_prev": p, "n_tracked": m, "n_kept": 1, "n_new": 2, "n_candidates": 3, "nms_rounds": 4, "eig_fixups": 5, "lk_iterations": 6}
        batch.append((obs, status, info))
    bench.dump_outputs(str(tmp_path), batch, 6)
    out = {fn[:-4]: np.load(tmp_path / fn) for fn in os.listdir(tmp_path)}
    assert sorted(out) == ["info", "n_obs", "n_prev", "obs_id", "obs_track_cnt", "obs_v", "status"]
    assert all(a.dtype == np.float64 for a in out.values())
    assert out["obs_v"].shape == (3, 6, 8) and out["info"].shape == (3, 8)
    for f, (obs, status, info) in enumerate(batch):
        m, p = len(obs), len(status)
        assert out["n_obs"][f] == m and out["n_prev"][f] == p
        np.testing.assert_array_equal(out["obs_id"][f, :m], obs["id"])
        assert (out["obs_id"][f, m:] == -1).all()
        np.testing.assert_array_equal(out["obs_track_cnt"][f, :m], obs["track_cnt"])
        np.testing.assert_array_equal(out["obs_v"][f, :m], obs["v"])
        assert (out["obs_v"][f, m:] == 0).all()
        np.testing.assert_array_equal(out["status"][f, :p], status)
        assert (out["status"][f, p:] == 0).all()
        np.testing.assert_array_equal(out["info"][f], list(info.values()))
