"""CPU test of bench.py's reference arm: it must print one JSON line with the keys tools parse,
and write its last step's outputs with --dump-outputs, without touching a GPU or the original
project's sources."""
import glob
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_json(tmp_path):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    dump = tmp_path / "out"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "0", "--dump-outputs", str(dump)], capture_output=True, text=True,
                         timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["matches_per_image"] > 100   # the planted workload really produces matches
    files = {os.path.basename(f)[:-4]: np.load(f) for f in glob.glob(str(dump / "*.npy"))}
    assert sum(os.path.getsize(f) for f in glob.glob(str(dump / "*"))) <= 64 << 20
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert not {"query_image", "keypoints3d", "descriptors3d_db", "descriptors3d_coarse_db"} & set(files)
    M = d["config"]["matches_per_image"]
    assert files["b_ids"].shape == (M,) and files["mkpts_query_f"].shape == (M, 2) and files["mconf"].dtype == np.float32
    assert np.array_equal(files["j_ids"], files["j_ids"].round()) and files["j_ids"].max() < 64 * 64
    # conf_matrix (1 x 5000 x 4096) is larger than a dump keeps: a sample at ascending flat indices
    idx = files["conf_matrix_sample_index"]
    assert files["conf_matrix"].shape == idx.shape == (1 << 20,) and (np.diff(idx) >= 0).all()
    assert idx.max() < 5000 * 4096 and 0 <= files["conf_matrix"].min() and files["conf_matrix"].max() <= 1
