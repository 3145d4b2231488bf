"""The indexed binary PLY (dcsg_mesh_weld, dcsg_write_ply_indexed, dcsg_export_indexed, the CLI's --ply-indexed): a re-encoding
of the reference's export with shared float vertices and optional normals.  The files are parsed with numpy here."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes

HEADER = ("ply\nformat binary_little_endian 1.0\ncomment DesignCSG export, indexed: vertices shared between faces\n"
          "element vertex {V}\nproperty float x\nproperty float y\nproperty float z\n{N}"
          "element face {T}\nproperty list uchar uint vertex_indices\nend_header\n")
NORMALS = "property float nx\nproperty float ny\nproperty float nz\n"
FACE = np.dtype([("count", "u1"), ("idx", "<u4", 3)])                  # packed: 13 bytes


def read_indexed_ply(path):
    """(xyz (V,3) float32, normals (V,3) float32 or None, faces (T,3) uint32); checks the header text and the file size."""
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode().split("\n")
    V = int(next(l for l in lines if l.startswith("element vertex")).split()[2])
    T = int(next(l for l in lines if l.startswith("element face")).split()[2])
    normals = NORMALS in data[:end].decode()
    assert data[:end].decode() == HEADER.format(V=V, T=T, N=NORMALS if normals else "")
    vdt = np.dtype([("xyz", "<f4", 3)] + ([("n", "<f4", 3)] if normals else []))
    assert len(data) == end + V * vdt.itemsize + T * FACE.itemsize
    verts = np.frombuffer(data, vdt, V, end)
    faces = np.frombuffer(data, FACE, T, end + V * vdt.itemsize)
    assert np.all(faces["count"] == 3)
    assert T == 0 or faces["idx"].max() < V
    return verts["xyz"].copy(), (verts["n"].copy() if normals else None), faces["idx"].copy()


def soup_ply_vertex_rows(path):
    """The vertex-row section of the reference's soup PLY (3 doubles per corner) and its triangle count."""
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    T = int(next(l for l in data[:end].decode().split("\n") if l.startswith("element face")).split()[2])
    return data[end:end + 72 * T], T


def numpy_weld(vertices, triangles):
    """Vertices with equal uint32 position words merged, numbered by their first occurrence."""
    rows = np.ascontiguousarray(vertices, dtype=np.float32).view(np.uint32).reshape(-1, 3)
    keys = np.ascontiguousarray(rows).view(np.dtype((np.void, 12))).ravel()
    _, first, inverse = np.unique(keys, return_index=True, return_inverse=True)
    order = np.sort(first)
    new_id = np.searchsorted(order, first)              # unique u -> rank of its first occurrence
    return vertices[order], new_id[inverse.ravel()][triangles].astype(np.uint32)


def export_levels(name):
    cfg = scenes.materialize(name)["export_config"]
    return float(cfg[0]), int(cfg[1]), int(cfg[2]), int(cfg[3]), float(cfg[4]), int(cfg[5])


# ---- CPU ----------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("level", [5, 6])
def test_lattice_vertices_are_distinct_positions(level):
    """Every vertex of a lattice mesh is one lattice edge's midpoint, and distinct edges give distinct positions: the weld of a
    keyed (uniform) mesh would merge nothing, so it is skipped."""
    from oracle.oracle import Oracle
    orc = Oracle.for_scene(scenes.materialize("design1"), "port")
    box = orc.bbox(10.0)
    got = H.emul_extract(orc.lattice_sdf(box, 1 << level), box, level)
    rows = np.ascontiguousarray(got["vertices"], dtype=np.float32).view(np.uint32).reshape(-1, 3)
    assert len(rows) > 1000
    assert len(np.unique(rows, axis=0)) == len(rows)


def _run_cli(args, env_extra):
    env = dict(os.environ, **env_extra)
    # a build or a device call would fail loudly: the checks must come first
    code = ("import sys, designcsg_b200.build as b, designcsg_b200.api as a\n"
            "def boom(*x, **k): raise RuntimeError('touched the build or the device')\n"
            "b.build = boom; a.Context = boom\n"
            "from designcsg_b200.__main__ import main\n"
            "sys.argv = ['designcsg_b200'] + %r\n"
            "main()\n" % (args,))
    return subprocess.run([sys.executable, "-c", code], cwd=H.REPO, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                          text=True, timeout=120)


@pytest.mark.parametrize("extra", [["--ply", "s.ply"], ["--stl", "s.stl"], ["--ply", "s.ply", "--stl", "s.stl"]])
def test_cli_rejects_indexed_with_soup_files(extra):
    proc = _run_cli(["export", "no_such_scene", "--ply-indexed", "i.ply"] + extra, {"WORLD_SIZE": "1"})
    assert proc.returncode != 0
    assert "--ply-indexed cannot be combined" in proc.stdout and "touched" not in proc.stdout, proc.stdout


def test_cli_rejects_sharded_indexed_without_level():
    proc = _run_cli(["export", "no_such_scene", "--ply-indexed", "i.ply"], {"WORLD_SIZE": "2", "RANK": "0", "LOCAL_RANK": "0"})
    assert proc.returncode != 0
    assert "needs --level" in proc.stdout and "touched" not in proc.stdout, proc.stdout


# ---- GPU ----------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctxs():
    from designcsg_b200 import api, build
    build.build()
    made = {}

    def get(name):
        if name not in made:
            ctx = api.Context(0)
            ctx.build(scenes.materialize(name)["dir"])
            made[name] = ctx
        return made[name]

    yield get
    for ctx in made.values():
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,level", [("design1", 6), ("design1", 7), ("stress", 6), ("stress", 7)])
def test_uniform_file_is_the_extracted_mesh(ctxs, tmp_path, name, level):
    ctx = ctxs(name)
    steps = export_levels(name)[5]
    path = str(tmp_path / "i.ply")
    rep = ctx.export_indexed(scenes.materialize(name)["dir"], level, path)
    xyz, nrm, faces = read_indexed_ply(path)
    mesh = ctx.extract(np.array(rep.box, dtype=np.float32), level, gd_steps=steps)
    assert nrm is None and len(faces) == mesh.num_triangles == rep.num_triangles > 0
    assert len(xyz) == mesh.num_vertices == rep.num_vertices
    assert np.array_equal(xyz.view(np.uint32), mesh.vertices().view(np.uint32))
    assert np.array_equal(faces, mesh.triangles())
    mesh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("name,level", [("design1", 7), ("design1", 0), ("design2", 0)])
def test_expanded_file_is_the_reference_ply(ctxs, tmp_path, name, level):
    """level 0 = the design's own adaptive levels (walk + retopologize, welded before the projection)."""
    ctx = ctxs(name)
    scene = scenes.materialize(name)["dir"]
    soup_path, idx_path = str(tmp_path / "soup.ply"), str(tmp_path / "i.ply")
    ctx.export(scene, level, ply_path=soup_path)
    rep = ctx.export_indexed(scene, level, idx_path)
    xyz, _, faces = read_indexed_ply(idx_path)
    rows, T = soup_ply_vertex_rows(soup_path)
    assert len(faces) == T == rep.num_triangles > 0
    assert xyz[faces].astype(np.float64).tobytes() == rows
    print("indexed[%s level %s]: %d triangles, %d vertices in the file (%d soup corners), %d vs %d bytes"
          % (name, level or "shipped", T, len(xyz), 3 * T, os.path.getsize(idx_path), os.path.getsize(soup_path)))


def _adaptive(ctx, name, retopologize, **kwargs):
    search, lo, hi, grid, thr, _ = export_levels(name)
    box = ctx.bbox(search)
    return ctx.extract(box, grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=retopologize,
                       defer_projection=True, **kwargs)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["design1", "design2"])
@pytest.mark.parametrize("retopologize", [False, True])
def test_weld_equals_numpy(ctxs, name, retopologize):
    ctx = ctxs(name)
    mesh = _adaptive(ctx, name, retopologize)
    v0, t0 = mesh.vertices(), mesh.triangles()
    want_v, want_t = numpy_weld(v0, t0)
    mesh.weld()
    got_v, got_t = mesh.vertices(), mesh.triangles()
    assert mesh.num_vertices == len(got_v) == len(want_v) < len(v0)
    assert np.array_equal(got_v.view(np.uint32), want_v.view(np.uint32))
    assert np.array_equal(got_t, want_t)
    assert len(np.unique(got_v.view(np.uint32), axis=0)) == len(got_v)         # no two vertices are equal
    assert np.unique(got_t).size == len(got_v)                                  # and every one is used
    if not retopologize:
        # soup: vertex 3t+i is first used by triangle t, so the ids appear in increasing order of first use
        ids = got_t.ravel()
        _, first = np.unique(ids, return_index=True)
        assert np.all(np.diff(ids[np.sort(first)].astype(np.int64)) > 0)
    print("weld[%s, retopologize=%d]: %d -> %d vertices" % (name, retopologize, len(v0), len(got_v)))
    mesh.free()


@pytest.mark.gpu
def test_weld_leaves_a_lattice_mesh_unchanged(ctxs):
    ctx = ctxs("design1")
    mesh = ctx.extract(ctx.bbox(10.0), 6, gd_steps=3)
    v, t = mesh.vertices(), mesh.triangles()
    mesh.weld()
    assert mesh.num_vertices == len(v)
    assert np.array_equal(mesh.vertices().view(np.uint32), v.view(np.uint32)) and np.array_equal(mesh.triangles(), t)
    mesh.free()


@pytest.mark.gpu
def test_weld_before_projection_is_exact(ctxs, tmp_path):
    """Equal starting positions project to equal positions and normals: weld-then-project = project-then-expand."""
    ctx = ctxs("design1")
    steps = export_levels("design1")[5]
    late = _adaptive(ctx, "design1", True)
    ctx.project(late, steps, want_normals=True)
    early = _adaptive(ctx, "design1", True)
    early.weld()
    ctx.project(early, steps, want_normals=True)
    assert np.array_equal(early.soup().view(np.uint32), late.soup().view(np.uint32))
    expanded = []
    for i, mesh in enumerate((late, early)):
        path = str(tmp_path / ("%d.ply" % i))
        mesh.write_ply_indexed(path, normals=True)
        xyz, nrm, faces = read_indexed_ply(path)
        expanded.append((xyz[faces].view(np.uint32), nrm[faces].view(np.uint32)))
    assert np.array_equal(expanded[0][0], expanded[1][0]) and np.array_equal(expanded[0][1], expanded[1][1])
    late.free()
    early.free()


@pytest.mark.gpu
@pytest.mark.parametrize("level", [6, 0])
def test_file_normals_are_eval_normal(ctxs, tmp_path, level):
    ctx = ctxs("design1")
    path = str(tmp_path / "n.ply")
    ctx.export_indexed(scenes.materialize("design1")["dir"], level, path, normals=True)
    xyz, nrm, faces = read_indexed_ply(path)
    assert nrm is not None and len(xyz) > 0
    assert np.array_equal(nrm.view(np.uint32), ctx.eval_normal(xyz).view(np.uint32))


@pytest.mark.gpu
def test_soup_writers_on_a_welded_mesh(ctxs):
    from designcsg_b200 import api
    ctx = ctxs("design1")
    mesh = _adaptive(ctx, "design1", True)
    ply, stl, soup = mesh.format_ply(), mesh.format_stl(), mesh.soup()
    mesh.weld()
    assert np.array_equal(mesh.format_ply(), ply) and np.array_equal(mesh.format_stl(), stl)
    assert np.array_equal(mesh.soup().view(np.uint32), soup.view(np.uint32))
    with pytest.raises(api.DcsgError):
        mesh.project_and_write_files(3, ply_path=None, stl_path=None)
    mesh.free()


@pytest.mark.gpu
def test_far_box_header_only_and_repeat_runs(ctxs, tmp_path):
    ctx = ctxs("design1")
    box = np.array([8.0, 8.0, 8.0, 2.0, 2.0, 2.0], dtype=np.float32)           # Design1 lives inside +-3.4
    for kwargs in ({}, {"min_level": 3, "max_level": 5, "retopologize": True}):
        mesh = ctx.extract(box, 6, gd_steps=3, want_normals=True, **kwargs)
        mesh.weld()
        for normals in (False, True):
            path = str(tmp_path / "e.ply")
            mesh.write_ply_indexed(path, normals=normals)
            assert open(path, "rb").read() == HEADER.format(V=0, T=0, N=NORMALS if normals else "").encode()
        mesh.free()
    scene = scenes.materialize("design1")["dir"]
    a, b = str(tmp_path / "a.ply"), str(tmp_path / "b.ply")
    ctx.export_indexed(scene, 0, a, normals=True)
    ctx.export_indexed(scene, 0, b, normals=True)
    assert open(a, "rb").read() == open(b, "rb").read()


@pytest.mark.gpu
def test_sharded_indexed_on_two_gpus(tmp_path):
    """tools/check_indexed_multi_gpu.py under torchrun (skipped on a one-GPU box)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = os.path.join(H.REPO, "tools", "check_indexed_multi_gpu.py")
    proc = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                           "127.0.0.1", "--master-port", "29537", script, str(tmp_path)], stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=900)
    assert proc.returncode == 0 and "INDEXED MULTI-GPU OK" in proc.stdout, proc.stdout[-3000:]
