"""GPU test of `bench.py --dump-outputs DIR`: after the timed steps the arrays the last one handed its caller are written as float32 /
float64 .npy files (64 MB at most in all). The inputs are seeded, so the same arguments give the same outputs; the pyramids and the
optical flow of the dump are those of the frame the last timed step processed (checked against the C oracle, bit for bit), and
--steps sets the number of frames of the timed loop."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WARMUP = 3


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(WARMUP),
                        "--step-only", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == steps and d["value"] > 0
    return d, {os.path.basename(f)[:-4]: np.load(f) for f in sorted(glob.glob(os.path.join(str(out_dir), "*.npy")))}


def _check_last_frame(out, steps, inp, oracle_lk):
    """The frame of the last timed step: bench.py's session has run the Python-harness loop (WARMUP + min(steps, 100) frames), the
    native warm-up (WARMUP frames) and the timed loop (steps frames) by then."""
    import bench
    k = 2 * WARMUP + min(steps, 100) + steps
    j, jp = bench.frame_index(k), bench.frame_index(k - 1)
    left, right, prev = (inp.frames[a, c].cpu().numpy() for a, c in ((j, 0), (j, 1), (jp, 0)))
    pl, pr, pp = (oracle_lk.pyramid(x, bench.WIN, bench.MAXLEVEL) for x in (left, right, prev))
    for side, p in (("left", pl), ("right", pr)):
        for lv in range(p.levels):
            g, d = p.download(lv, padded=False)
            assert np.array_equal(out[f"pyramid_{side}_gray_l{lv}"], g) and np.array_equal(out[f"pyramid_{side}_grad_l{lv}"], d), (steps, side, lv)
    nxt, _, _ = oracle_lk.lk(pp, pl, inp.points, inp.init_guess(jp, j), accum_mode=1)
    nxt2, st2, ts2 = oracle_lk.lk(pl, pr, nxt, None, accum_mode=1)
    assert np.array_equal(out["lk_temporal_next_xy"].view(np.uint32), nxt.view(np.uint32)), steps
    assert np.array_equal(out["lk_stereo_next_xy"].view(np.uint32), nxt2.view(np.uint32)), steps
    assert np.array_equal(out["lk_status"], st2) and np.array_equal(out["lk_track_status"], ts2), steps


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path, oracle_lk):
    import torch
    import bench
    da, a = _bench(tmp_path / "a", 100)
    assert {"lk_temporal_next_xy", "lk_stereo_next_xy", "lk_status", "lk_track_status", "ekf_mean", "ekf_covariance", "ekf_outlier_status",
            "ekf_chi2", "pyramid_left_gray_l0", "pyramid_left_grad_l0", "pyramid_right_gray_l3", "pyramid_right_grad_l3"} <= set(a)
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert all(np.isfinite(x).all() for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["ekf_covariance"].shape == (160, 160) and a["ekf_covariance"].any() and a["ekf_outlier_status"].shape == (bench.CHECKS,)
    _, b = _bench(tmp_path / "b", 100)
    assert a.keys() == b.keys()
    assert all(np.array_equal(a[k], b[k]) for k in a), [k for k in a if not np.array_equal(a[k], b[k])]
    # one more timed step (the Python-harness loop runs 100 frames in both runs): one more frame's launches, the next frame's outputs
    dc, c = _bench(tmp_path / "c", 101)
    per_frame = dc["gpu_launches"] - da["gpu_launches"]
    assert per_frame > 0 and da["gpu_launches"] == 100 * per_frame and dc["gpu_launches"] == 101 * per_frame
    assert not np.array_equal(a["ekf_mean"], c["ekf_mean"])
    inp = bench.Inputs(torch.device("cuda"))
    _check_last_frame(a, 100, inp, oracle_lk)
    _check_last_frame(c, 101, inp, oracle_lk)
