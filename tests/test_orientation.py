"""Outward winding (dcsg_mesh_orient, the exports' DCSG_EXPORT_OUTWARD, the CLI's --outward).

The reference's lookup table does not orient its loops consistently, so its files mix both windings.  Which triangles face
inwards depends only on the cell's corner mask and the triangle's slot in the table row; kDcsgTriFlip (mc_table.inc) holds
that bit per slot, decided per loop.  The rule is restated here in numpy and checked on the CPU mesher harness and on the
device's meshes and files."""
import importlib.util
import json
import os
import re

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes
from tests.test_indexed_export import _run_cli, export_levels, numpy_weld, read_indexed_ply

CSRC = os.path.join(H.REPO, "designcsg_b200", "csrc")
LOOPS = json.load(open(os.path.join(H.HERE, "golden", "lookup_loops.json")))["loops"]
# corner c as (dx, dy, dz) (reference geometry.hpp:264-279); cell edge e as its two end corners (mesh.hpp:187-209)
CORNER = np.array([(0, 0, 1), (1, 0, 1), (1, 0, 0), (0, 0, 0), (0, 1, 1), (1, 1, 1), (1, 1, 0), (0, 1, 0)])
EDGE_ENDS = [(0, 1), (1, 2), (3, 2), (0, 3), (4, 5), (5, 6), (7, 6), (4, 7), (0, 4), (1, 5), (2, 6), (3, 7)]


def strip(loop):
    """getIndexTriangleStrip (reference geometry.hpp:228-248)."""
    q, out = list(loop), []
    if len(q) & 1:
        out.append((q[0], q[1], q[-1]))
        q.pop(0)
    lo, hi = 0, len(q) - 1
    while hi - lo >= 3:
        out += [(q[lo], q[lo + 1], q[hi - 1]), (q[hi - 1], q[hi], q[lo])]
        lo, hi = lo + 1, hi - 1
    return out


def outward_dir(mask, e):
    """Outside corner minus inside corner of cell edge e (a set mask bit is S < 0: inside)."""
    a, b = EDGE_ENDS[e]
    assert ((mask >> a) & 1) != ((mask >> b) & 1)
    return (CORNER[b] - CORNER[a]) * (1 if (mask >> a) & 1 else -1)


def midpoint(e):
    a, b = EDGE_ENDS[e]
    return (CORNER[a] + CORNER[b]) / 2.0


def loop_rule():
    """The flip bits by the loop rule: a loop faces inwards when its Newell normal points against the inside -> outside
    direction of the edges it crosses; every strip triangle of the loop takes its bit."""
    flips = np.zeros(256, dtype=np.uint8)
    for mask, cycles in enumerate(LOOPS):
        t = 0
        for loop in cycles:
            pts = np.array([midpoint(e) for e in loop])
            n = np.cross(pts, np.roll(pts, -1, axis=0)).sum(axis=0)
            s = sum(float(n @ outward_dir(mask, e)) for e in loop)
            assert s != 0.0
            for _ in strip(loop):
                flips[mask] |= (s < 0) << t
                t += 1
    return flips


def triangle_rule():
    """The rejected alternative: each triangle by its own normal against the summed inside -> outside directions of its edges."""
    flips = np.zeros(256, dtype=np.uint8)
    for mask, cycles in enumerate(LOOPS):
        tris = [t for loop in cycles for t in strip(loop)]
        for t, tri in enumerate(tris):
            p = [midpoint(e) for e in tri]
            d = sum(outward_dir(mask, e) for e in tri)
            flips[mask] |= (float(np.cross(p[1] - p[0], p[2] - p[0]) @ d) < 0) << t
    return flips


def parse_table(name, dtype):
    text = open(os.path.join(CSRC, "mc_table.inc")).read()
    body = re.search(r"%s\[[^\]]*\] = \{([^}]*)\}" % name, text).group(1)
    return np.array([int(v) for v in body.replace("\n", "").split(",") if v.strip()], dtype=dtype)


TRI_COUNT = parse_table("kDcsgTriCount", np.int64)
FLIP = loop_rule()


def triangle_flags(cell_masks, unit=1, flips=FLIP):
    """Per triangle of a mesh in canonical order (cell, table slot, `unit` strip children): does its slot face inwards?"""
    masks = np.asarray(cell_masks, dtype=np.int64)
    per_cell = TRI_COUNT[masks]
    cell = np.repeat(np.arange(len(masks)), per_cell)
    slot = np.arange(len(cell)) - np.repeat(np.cumsum(per_cell) - per_cell, per_cell)
    flagged = ((flips[masks[cell]].astype(np.int64) >> slot) & 1).astype(bool)
    return np.repeat(flagged, unit)


def oriented(triangles, flags):
    t = np.array(triangles, copy=True).reshape(-1, 3)
    t[flags, 1], t[flags, 2] = triangles[flags, 2], triangles[flags, 1]
    return t


def inconsistent_edges(triangles):
    """(edges used by exactly two non-degenerate faces, those of them both faces traverse the same way).  Non-degenerate: three
    distinct vertex ids."""
    t = np.asarray(triangles, dtype=np.int64).reshape(-1, 3)
    t = t[(t[:, 0] != t[:, 1]) & (t[:, 1] != t[:, 2]) & (t[:, 0] != t[:, 2])]
    a = t.ravel()
    b = t[:, [1, 2, 0]].ravel()
    lo, hi = np.minimum(a, b), np.maximum(a, b)
    key = lo * (int(t.max()) + 1 if len(t) else 1) + hi
    _, inverse, counts = np.unique(key, return_inverse=True, return_counts=True)
    two = counts[inverse.ravel()] == 2
    forward = (a < b)[two]
    k = inverse.ravel()[two]
    fwd = np.bincount(k, weights=forward, minlength=len(counts))
    shared = counts == 2
    return int(shared.sum()), int(((fwd != 1) & shared).sum())


def signed_volume(vertices, triangles):
    p = np.asarray(vertices, dtype=np.float64)[np.asarray(triangles).reshape(-1, 3)]
    return float(np.einsum("ij,ij->i", p[:, 0], np.cross(p[:, 1], p[:, 2])).sum() / 6.0)


# ---- CPU ----------------------------------------------------------------------------------------------------------------------

def test_flip_table_is_the_loop_rule_and_the_generator_reproduces_the_file():
    assert np.array_equal(parse_table("kDcsgTriFlip", np.uint8), FLIP)
    assert sum(bin(int(f)).count("1") for f in FLIP) == 399          # of the table's 820 triangles
    assert all(int(f) >> int(c) == 0 for f, c in zip(FLIP, TRI_COUNT))
    spec = importlib.util.spec_from_file_location("gen_mc_table", os.path.join(H.REPO, "tools", "gen_mc_table.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    assert gen.render() == open(os.path.join(CSRC, "mc_table.inc")).read()


def test_the_rules_differ_at_ten_table_entries():
    """Deciding triangle by triangle disagrees with the loop rule at 10 slots of 5 masks."""
    diff = np.unpackbits((FLIP ^ triangle_rule())[:, None], axis=1).sum()
    assert diff == 10
    assert sorted(np.nonzero(FLIP ^ triangle_rule())[0].tolist()) == [62, 95, 124, 182, 250]


@pytest.fixture(scope="module")
def lattices():
    from oracle.oracle import Oracle
    made = {}

    def get(name, level):
        if (name, level) not in made:
            orc = Oracle.for_scene(scenes.materialize(name), "port")
            box = orc.bbox(10.0)
            made[(name, level)] = (box, orc.lattice_sdf(box, 1 << level))
        return made[(name, level)]

    return get


CASES = [("design1", 5), ("design1", 6), ("design1", 7), ("design2", 6), ("design2", 7), ("stress", 6)]


@pytest.mark.parametrize("no_cull", [False, True])
@pytest.mark.parametrize("name,level", CASES)
def test_cpu_mesher_oriented_is_consistent_and_outward(lattices, name, level, no_cull):
    box, lattice = lattices(name, level)
    mesh = H.emul_extract(lattice, box, level, no_cull=no_cull)
    tris = mesh["triangles"]
    assert len(tris) == TRI_COUNT[mesh["cell_masks"]].sum() > 1000
    shared, bad_written = inconsistent_edges(tris)
    fixed = oriented(tris, triangle_flags(mesh["cell_masks"]))
    shared_o, bad = inconsistent_edges(fixed)
    assert shared_o == shared and bad == 0 and bad_written > 0
    volume = signed_volume(mesh["vertices"], fixed)
    cell = np.prod(np.asarray(box[3:], dtype=np.float64) / (1 << level))
    inside = float((np.asarray(lattice) < 0).sum()) * cell
    print("%s 2^%d cull=%d: %d shared edges, %d inconsistent as written -> 0; volume %.2f -> %.2f (inside samples %.2f)"
          % (name, level, not no_cull, shared, bad_written, signed_volume(mesh["vertices"], tris), volume, inside))
    assert volume > 0 and abs(volume - inside) < 0.1 * inside


def test_the_triangle_rule_leaves_inconsistent_edges(lattices):
    box, lattice = lattices("design2", 6)
    mesh = H.emul_extract(lattice, box, 6, no_cull=True)
    _, bad = inconsistent_edges(oriented(mesh["triangles"], triangle_flags(mesh["cell_masks"], flips=triangle_rule())))
    assert bad > 0


@pytest.mark.parametrize("out", [["--ply", "s.ply"], ["--stl", "s.stl"], ["--ply-indexed", "i.ply"]])
def test_cli_accepts_outward(out):
    """Accepted with each output: the command gets as far as the build (which the test replaces by a failure)."""
    proc = _run_cli(["export", "no_such_scene", "--outward"] + out, {"WORLD_SIZE": "1"})
    assert proc.returncode != 0 and "touched the build or the device" in proc.stdout, proc.stdout


def test_cli_refusals_fire_with_outward():
    proc = _run_cli(["export", "no_such_scene", "--outward", "--ply-indexed", "i.ply", "--stl", "s.stl"], {"WORLD_SIZE": "1"})
    assert proc.returncode != 0 and "--ply-indexed cannot be combined" in proc.stdout and "touched" not in proc.stdout, proc.stdout
    proc = _run_cli(["export", "no_such_scene", "--outward", "--ply-indexed", "i.ply"], {"WORLD_SIZE": "2", "RANK": "0", "LOCAL_RANK": "0"})
    assert proc.returncode != 0 and "needs --level" in proc.stdout and "touched" not in proc.stdout, proc.stdout


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


def _retopo_unit(name, retopologize):
    _, lo, hi, grid, _, _ = export_levels(name)
    p = 1 << (grid - min(lo, hi))
    return 3 * p - 2 if retopologize and p >= 2 else 1


def _adaptive(ctx, name, retopologize):
    search, lo, hi, grid, thr, _ = export_levels(name)
    return ctx.extract(ctx.bbox(search), grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=retopologize,
                       defer_projection=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name,level", [("design1", 6), ("design1", 7), ("design2", 6), ("design2", 7), ("stress", 6), ("stress", 7)])
def test_device_orient_is_the_rule(ctxs, name, level):
    ctx = ctxs(name)
    mesh = ctx.extract(ctx.bbox(10.0), level, gd_steps=3)
    v, t, soup = mesh.vertices(), mesh.triangles(), mesh.soup()
    want = oriented(t, triangle_flags(mesh.cell_masks()))
    mesh.orient()
    assert np.array_equal(mesh.triangles(), want)                                      # host copy refreshed
    assert np.array_equal(mesh.soup().view(np.uint32), v[want].view(np.uint32))         # device triangles, vertices untouched
    assert np.array_equal(mesh.vertices().view(np.uint32), v.view(np.uint32))
    assert np.array_equal(np.sort(mesh.soup().view(np.uint32), axis=None), np.sort(soup.view(np.uint32), axis=None))
    mesh.orient()                                                                       # a no-op
    assert np.array_equal(mesh.triangles(), want) and np.array_equal(mesh.soup().view(np.uint32), v[want].view(np.uint32))
    assert inconsistent_edges(want)[1] == 0
    mesh.free()


@pytest.mark.gpu
def test_slabs_oriented_one_by_one_are_the_oriented_whole(ctxs):
    ctx = ctxs("design2")
    box, n = ctx.bbox(10.0), 1 << 7
    whole = ctx.extract(box, 7)
    whole.orient()
    soups = []
    for r in range(4):
        slab = ctx.extract(box, 7, slab=(r * n // 4, (r + 1) * n // 4))
        slab.orient()
        soups.append(slab.soup())
        slab.free()
    assert np.array_equal(np.concatenate(soups).view(np.uint32), whole.soup().view(np.uint32))
    whole.free()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["design1", "design2"])
@pytest.mark.parametrize("retopologize", [False, True])
@pytest.mark.parametrize("weld_first", [False, True])
def test_adaptive_orient_is_the_rule(ctxs, name, retopologize, weld_first):
    ctx = ctxs(name)
    mesh = _adaptive(ctx, name, retopologize)
    v0, t0 = mesh.vertices(), mesh.triangles()
    flags = triangle_flags(mesh.cell_masks(), _retopo_unit(name, retopologize))
    assert len(flags) == len(t0)
    want_v, want_t = numpy_weld(v0, oriented(t0, flags))
    if weld_first:
        mesh.weld()
        mesh.orient()
    else:
        mesh.orient()
        assert np.array_equal(mesh.triangles(), oriented(t0, flags))
        mesh.weld()
    assert np.array_equal(mesh.vertices().view(np.uint32), want_v.view(np.uint32))
    assert np.array_equal(mesh.triangles(), want_t)
    shared, bad = inconsistent_edges(want_t)
    volume = signed_volume(want_v, want_t)
    print("%s shipped levels, retopologize=%d: %d shared edges, %d inconsistent, volume %.3f" % (name, retopologize, shared, bad, volume))
    assert shared > 0 and bad == 0 and volume > 0
    mesh.free()


@pytest.mark.gpu
def test_orient_refuses_meshes_without_cells(ctxs):
    from designcsg_b200 import api
    ctx = ctxs("design1")
    with pytest.raises(api.DcsgError) as err:
        api.Mesh(ctx).orient()
    assert err.value.code == -2


def read_stl(path):
    data = open(path, "rb").read()
    T = int(np.frombuffer(data, "<u4", 1, 80)[0])
    assert len(data) == 84 + 50 * T
    rec = np.frombuffer(data, np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]), T, 84)
    return rec


def read_soup_ply(path):
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    T = int(next(l for l in data[:end].decode().split("\n") if l.startswith("element face")).split()[2])
    return np.frombuffer(data, "<f8", 9 * T, end).reshape(T, 3, 3), data[end + 72 * T:]


@pytest.mark.gpu
@pytest.mark.parametrize("level", [7, 0])
def test_oriented_files(ctxs, tmp_path, level):
    """level 0 = Design1's shipped octree levels (adaptive walk + retopologize)."""
    ctx = ctxs("design1")
    scene = scenes.materialize("design1")["dir"]
    if level:
        mesh = ctx.extract(ctx.bbox(10.0), level)
        flags = triangle_flags(mesh.cell_masks())
    else:
        mesh = _adaptive(ctx, "design1", True)
        flags = triangle_flags(mesh.cell_masks(), _retopo_unit("design1", True))
    mesh.free()
    f = {k: str(tmp_path / k) for k in ("d.ply", "d.stl", "o.ply", "o.stl", "di.ply", "oi.ply")}
    ctx.export(scene, level, f["d.stl"], f["d.ply"])
    rep = ctx.export(scene, level, f["o.stl"], f["o.ply"], outward=True)
    assert rep.num_triangles == len(flags) > 0
    # soup PLY: corners 1 and 2 swapped on the flagged triangles, face rows unchanged
    (dv, dfaces), (ov, ofaces) = read_soup_ply(f["d.ply"]), read_soup_ply(f["o.ply"])
    assert ofaces == dfaces
    assert np.array_equal(ov, dv[np.arange(len(dv))[:, None], np.where(flags[:, None], [0, 2, 1], [0, 1, 2])])
    # STL: B and C swapped on the UNflagged triangles (the records' x z y order mirrors the mesh)
    ds, os_ = read_stl(f["d.stl"]), read_stl(f["o.stl"])
    assert np.array_equal(os_["n"], ds["n"]) and np.array_equal(os_["a"], ds["a"])
    assert np.array_equal(os_["v"], ds["v"][np.arange(len(ds))[:, None], np.where(flags[:, None], [0, 1, 2], [0, 2, 1])])
    # in its own coordinates the oriented STL is a consistently outward-wound surface
    xyz, tris = numpy_weld(os_["v"].reshape(-1, 3).copy(), np.arange(3 * len(os_)).reshape(-1, 3))
    shared, bad = inconsistent_edges(tris)
    assert shared > 0 and bad == 0 and signed_volume(xyz, tris) > 0
    assert inconsistent_edges(numpy_weld(ds["v"].reshape(-1, 3).copy(), np.arange(3 * len(ds)).reshape(-1, 3))[1])[1] > 0
    # indexed PLY: the same vertex rows, face rows swapped on the flagged triangles
    ctx.export_indexed(scene, level, f["di.ply"])
    ctx.export_indexed(scene, level, f["oi.ply"], outward=True)
    (dx, _, dt), (ox, _, ot) = read_indexed_ply(f["di.ply"]), read_indexed_ply(f["oi.ply"])
    assert np.array_equal(ox.view(np.uint32), dx.view(np.uint32))
    assert np.array_equal(ot, oriented(dt, flags))
    # the flag was restored: the default export is the reference's bytes again
    ctx.export(scene, level, f["o.stl"], None)
    assert open(f["o.stl"], "rb").read() == open(f["d.stl"], "rb").read()


@pytest.mark.gpu
def test_sharded_oriented_exports_on_one_rank(tmp_path):
    """dcsg_export_sharded and dcsg_export_sharded_indexed with DCSG_EXPORT_OUTWARD on a one-rank communicator write the files
    of the single-GPU oriented exports."""
    import torch  # noqa: F401  (before the communicator, see tests/test_sharded_export.py)
    from designcsg_b200 import api
    try:
        uid = api.comm_unique_id()
    except api.DcsgError as e:
        if e.code != -7:
            raise
        pytest.skip("NCCL is not loadable: %s" % e)
    scene = scenes.materialize("design1")["dir"]
    ctx = api.Context(0)
    comm = api.Comm(ctx, uid, 0, 1)
    try:
        for level in (7, 0):
            ctx.export(scene, level, str(tmp_path / "1.stl"), str(tmp_path / "1.ply"), outward=True)
            comm.export(scene, level, str(tmp_path / "w.stl"), str(tmp_path / "w.ply"), outward=True)
            for ext in ("stl", "ply"):
                assert (tmp_path / ("1." + ext)).read_bytes() == (tmp_path / ("w." + ext)).read_bytes(), (level, ext)
        ctx.export_indexed(scene, 7, str(tmp_path / "1i.ply"), outward=True)
        comm.export_indexed(scene, 7, str(tmp_path / "wi.ply"), outward=True)
        assert (tmp_path / "1i.ply").read_bytes() == (tmp_path / "wi.ply").read_bytes()
    finally:
        comm.close()
        ctx.close()
