"""bench.py --dump-outputs: what the value leg returned for the last frame of each camera stream, as float32 / float64 .npy
files, equal to what the extractor returns for the same frame."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("keypoints", "descriptors", "brute_force_matches", "projection_matches", "pose", "pose_outliers",
         "local_ba_poses", "local_ba_points", "local_ba_outliers")


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_frame_of_each_stream(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--frames-per-step", "1",
                        "--streams", "2", "--ring", "12", "--no-cpu-baseline", "--no-latency", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(out)) == sorted("stream%d_%s.npy" % (s, n) for s in (0, 1) for n in NAMES)
    arrays = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert arrays["stream0_pose"].shape == (12,) and arrays["stream0_local_ba_poses"].shape == (60, 12)
    from openvslam_b200 import feature, synth
    ext = feature.orb_extractor(feature.orb_params(max_num_keypts=4000))
    # 3 warm-up frames (the floor) + 1 timed frame: stream k's last frame is ring frame (3 + 11 k) % 12, i.e. base frame 3 / 2,
    # unshifted, of rank 0's workload (seed 100 * rank + base index)
    for s, seed in ((0, 3), (1, 2)):
        kps, desc = ext.extract(synth.frame(1920, 960, seed=seed))
        want = np.stack([kps[f].astype(np.float32) for f in ("x", "y", "size", "angle", "response", "octave")], 1)
        assert np.array_equal(arrays["stream%d_keypoints" % s], want)
        assert np.array_equal(arrays["stream%d_descriptors" % s], desc.astype(np.float32))
    ext.close()
