"""bench.py --dump-outputs: the files hold what the timed path computes, and a sampled array keeps the rows it names."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def design1():
    from designcsg_b200 import api, build
    build.build()
    ctx = api.Context(0)
    ctx.build(scenes.materialize("design1")["dir"])
    yield ctx
    ctx.close()


def _expected(ctx, level, gd_steps):
    box = ctx.bbox(10.0)
    mesh = ctx.extract(box, level, gd_steps=gd_steps)
    want = {"box": box.astype(np.float64), "counts": np.array([mesh.num_vertices, mesh.num_triangles, mesh.num_cells], dtype=np.float64),
            "vertices": mesh.vertices(), "vertex_keys": mesh.vertex_keys().astype(np.float64),
            "triangles": mesh.triangles().astype(np.float64), "cell_ids": mesh.cell_ids().astype(np.float64),
            "cell_masks": mesh.cell_masks().astype(np.float64)}
    mesh.free()
    return want


def test_dump_outputs_of_a_small_run(design1, tmp_path):
    """The whole command at 64^3: the JSON line reports the steps asked for, and the dump equals dcsg_extract's arrays."""
    out = tmp_path / "dump"
    proc = subprocess.run([sys.executable, os.path.join(H.REPO, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--level", "6",
                           "--gd-steps", "5", "--no-cpu-baseline", "--dump-outputs", str(out)],
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-3000:]
    line = json.loads(proc.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2
    want = _expected(design1, 6, 5)
    assert sorted(os.listdir(out)) == sorted(n + ".npy" for n in want)           # nothing sampled at this size
    for name, a in want.items():
        got = np.load(out / (name + ".npy"))
        assert got.dtype == (np.float32 if name == "vertices" else np.float64), name
        assert np.array_equal(got, a, equal_nan=True), name


def test_dump_outputs_samples_long_arrays(design1, tmp_path, monkeypatch):
    """Past DUMP_ROWS rows an array keeps the seeded, sorted rows stored beside it."""
    sys.path.insert(0, H.REPO)
    import bench
    monkeypatch.setattr(bench, "DUMP_ROWS", 1000)
    box = design1.bbox(10.0)
    mesh = design1.extract(box, 6, gd_steps=5, copy_to_host=False)
    bench.dump_outputs(str(tmp_path), box, mesh, "cuda:0")
    mesh.free()
    want = _expected(design1, 6, 5)
    for group, names in (("vertex", ("vertices", "vertex_keys")), ("triangle", ("triangles",)), ("cell", ("cell_ids", "cell_masks"))):
        rows = np.load(tmp_path / (group + "_rows.npy")).astype(np.int64)
        assert len(rows) == 1000 and np.all(np.diff(rows) > 0)
        for name in names:
            assert np.array_equal(np.load(tmp_path / (name + ".npy")), want[name][rows], equal_nan=True), name
    assert np.array_equal(np.load(tmp_path / "counts.npy"), want["counts"])
