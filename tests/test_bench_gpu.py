"""GPU: bench.py --dump-outputs writes what the timed path returned in its last step -- float .npy files within
the size bound, equal to what a Context returns for the same seeded scene and the dumped pairs."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_dump_outputs_equal_a_direct_call(tmp_path):
    import pycolmap_b200 as pb
    from pycolmap_b200 import synthetic as syn

    n_img, K = 40, 1024
    out_dir = tmp_path / "out"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--images", str(n_img),
           "--feats", str(K), "--no-cpu", "--no-e2e", "--dump-outputs", str(out_dir)]
    run = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert run.returncode == 0, run.stderr[-2000:]
    line = json.loads(run.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["pairs_per_step"] == n_img * (n_img - 1) // 2

    files = sorted(glob.glob(str(out_dir / "*.npy")))
    assert sum(os.path.getsize(f) for f in files) <= bench.DUMP_BYTES
    d = {os.path.basename(f)[:-4]: np.load(f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert len(d["pairs"]) == n_img * (n_img - 1) // 2 and d["has_lists"].all()   # small run: every pair, every list

    scene = syn.make_scene(n_img, K, seed=0, device="cuda")
    cam = dict(model=0, width=1600, height=1200, params=[1200.0, 800.0, 600.0], has_prior_focal_length=1)
    ctx = pb.Context(device=0)
    ctx.set_images([scene["desc"][i].cpu().numpy() for i in range(n_img)],
                   [scene["kpts"][i].cpu().numpy() for i in range(n_img)], [cam] * n_img)
    pairs = np.ascontiguousarray(d["pairs"].astype(np.int32))
    res = ctx.match_pairs(pairs, pb.SiftMatchingOptions(max_num_matches=32768), pb.TwoViewGeometryOptions())
    geoms = [res.two_view_geometry(k) for k in range(len(pairs))]
    want_matches = [res.matches(k) for k in range(len(pairs))]
    assert np.array_equal(d["num_matches"], [len(m) for m in want_matches])
    assert np.array_equal(d["matches"], np.concatenate(want_matches))
    assert np.array_equal(d["config"], [int(g.config) for g in geoms])
    assert np.array_equal(d["num_inliers"], [len(g.inlier_matches) for g in geoms])
    assert np.array_equal(d["inlier_matches"], np.concatenate([g.inlier_matches for g in geoms]))
    for m in ("E", "F", "H"):
        assert np.array_equal(d[m], np.stack([getattr(g, m) for g in geoms])), m
    assert d["num_inliers"].sum() > 0
    res.free()
    ctx.close()
