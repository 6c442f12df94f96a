"""bench.py --dump-outputs: the files two builds are compared by (host side; no GPU needed)."""
import os
import subprocess
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _extracted(kind, inpoints):
    cand = types.SimpleNamespace(type=kind, outwards=1, p=[0.25 * k for k in range(7)])
    idx = np.array(inpoints, np.int64)
    return types.SimpleNamespace(shape=types.SimpleNamespace(to_cand=lambda: cand), inpoints=idx, total=len(idx))


def test_dump_outputs_writes_counts_shapes_and_sampled_labels(tmp_path):
    import bench
    from tools.ransac_e2e import SCENES

    n = SCENES["c4"][0]
    step = n // (1 << 20)
    ex = {"c4": [_extracted(0, [0, step, 2 * step + 1, n - 1]), _extracted(3, [3 * step])], "c5": []}
    counts = np.arange(4096, dtype=np.int32)
    bench.dump_outputs(str(tmp_path), counts, ex, 1)
    files = sorted(os.listdir(tmp_path))
    assert files == ["ransac_c4_inliers.npy", "ransac_c4_sampled_point_shape.npy", "ransac_c4_shapes.npy",
                     "ransac_c5_inliers.npy", "ransac_c5_sampled_point_shape.npy", "ransac_c5_shapes.npy", "score_counts.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    for f in files:
        assert np.load(tmp_path / f).dtype in (np.float32, np.float64)
    np.testing.assert_array_equal(np.load(tmp_path / "score_counts.npy"), counts)
    shapes = np.load(tmp_path / "ransac_c4_shapes.npy")
    assert shapes.shape == (2, 9) and shapes[:, 0].tolist() == [0, 3] and shapes[1, 2:].tolist() == [0.25 * k for k in range(7)]
    np.testing.assert_array_equal(np.load(tmp_path / "ransac_c4_inliers.npy"), [4, 1])
    lab = np.load(tmp_path / "ransac_c4_sampled_point_shape.npy")
    assert len(lab) == (n + step - 1) // step
    assert lab[:4].tolist() == [0, 0, -1, 1] and lab[-1] == (0 if (n - 1) % step == 0 else -1)
    assert (lab >= 0).sum() == 3 + ((n - 1) % step == 0)
    assert np.load(tmp_path / "ransac_c5_shapes.npy").shape == (0, 9)


def test_dump_outputs_without_sample_when_sharded(tmp_path):
    import bench

    bench.dump_outputs(str(tmp_path), np.zeros(8, np.int32), {"c2": [_extracted(1, [5])]}, 2)
    assert sorted(os.listdir(tmp_path)) == ["ransac_c2_inliers.npy", "ransac_c2_shapes.npy", "score_counts.npy"]


def test_steps_below_one_is_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr
