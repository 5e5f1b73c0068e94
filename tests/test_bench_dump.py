"""bench.py --dump-outputs: the writer's dtypes and size cap (no GPU), and on the B200 that the files hold what the
last timed forward step returned, checked against the oracle on that step's seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import gvcnn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_dump_outputs_dtypes_and_limit(tmp_path, monkeypatch):
    arrays = {"S": np.arange(6, dtype=np.float32).reshape(2, 3) / 7, "bins": np.array([0, 7, -3], dtype=np.int32),
              "x64": np.array([1 / 3], dtype=np.float64), "h": np.array([0.5, -2.0], dtype=np.float16)}
    bench.dump_outputs(str(tmp_path / "d"), arrays)
    got = {n: np.load(tmp_path / "d" / (n + ".npy")) for n in arrays}
    assert [got[n].dtype for n in arrays] == [np.float32, np.float64, np.float64, np.float32]
    for n, a in arrays.items():
        np.testing.assert_array_equal(got[n], a)
    monkeypatch.setattr(bench, "DUMP_LIMIT", 24 + 24 + 8 + 8 - 1)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "e"), arrays)
    assert not (tmp_path / "e").exists()


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path, c_oracle):
    K = 5                           # steps use input sets 0, 1, 2, 0, 1: the last one is set 1
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(K), "--warmup", "1",
                          "--no-sweep", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-4000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == K
    got = {n: np.load(tmp_path / (n + ".npy")) for n in ("S", "x", "xsum", "scores", "bins")}
    B, V, D, G, Cr = (bench.CFG[k] for k in ("B", "V", "D", "G", "C_raw"))
    assert {n: (a.dtype, a.shape) for n, a in got.items()} == {
        "S": (np.float32, (B, D)), "x": (np.float32, (B, V)), "xsum": (np.float32, (V,)),
        "scores": (np.float32, (V,)), "bins": (np.float64, (V,))}
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_LIMIT

    F, R, W, _, _ = (t.numpy() for t in bench.synth_inputs(B, V, D, Cr, 10 * ((K - 1) % bench.NSETS), 0))
    b = bench.literal_bias(V).numpy()
    x64 = c_oracle.view_score_x_f64(R, W, b)
    s64 = O.score_from_x(x64.sum(axis=0) / B)                       # the batch mean's score (nets/model.py:146-147)
    np.testing.assert_allclose(got["x"], x64, rtol=0, atol=1e-4)
    np.testing.assert_allclose(got["xsum"], x64.sum(axis=0), rtol=1e-4, atol=1e-1)
    np.testing.assert_allclose(got["scores"], s64, rtol=0, atol=1e-5)
    bins = got["bins"].astype(np.int32)
    assert np.array_equal(bins, got["bins"])
    s32 = s64.astype(np.float32)
    assert np.all((bins == O.bins_from_scores(s32, G)) | O.edge_ulps_distance(s32, G, k=8))
    np.testing.assert_array_equal(got["S"], c_oracle.pool_fuse_fwd(F, bins, G, "max", 1.0))
