"""The map file of a saved run (fast_lio_sam_qn.cpp:398-411, save_map_pcd): <dir>/<seq>_map.pcd, ASCII x y z intensity."""
import os

import numpy as np


def test_save_run_writes_map_pcd(tmp_path, synth):
    from b200reg import io
    seq = synth.make_sequence(3, 4, pts_per_keyframe=300, spacing=5.0)
    rng = np.random.default_rng(0)
    m = (rng.standard_normal((500, 4)) * [40.0, 40.0, 2.0, 50.0]).astype(np.float32)
    d = str(tmp_path / "run")
    io.save_run(d, seq["clouds"], seq["poses"], seq["stamps"], map_xyzi=m, seq_name="s")
    p = os.path.join(d, "s_map.pcd")
    with open(p, "rb") as f:
        head = f.read(400).decode()
    assert "FIELDS x y z intensity" in head and "DATA ascii" in head and "POINTS 500" in head
    assert np.array_equal(io.load_pcd(p), m)  # %.9g round-trips fp32 exactly
    # without a map nothing new is written
    d2 = str(tmp_path / "run2")
    io.save_run(d2, seq["clouds"], seq["poses"], seq["stamps"])
    assert sorted(os.listdir(d2)) == ["pcd", "poses_kitti.txt", "poses_tum.txt"]
