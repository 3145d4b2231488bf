"""Mesh inspection (dcsg_mesh_inspect, Mesh.inspect, the CLI's `inspect`): edge topology, shells, area, volume, centroid and
extents.  The definitions are restated here operation for operation in numpy (inspect_model) and checked on hand-made meshes
with known answers, on the CPU mesher harness, and against the device on hand-made and library meshes."""
import ctypes
import json
import math
import subprocess
import sys

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes
from tests.test_indexed_export import _run_cli, export_levels, read_indexed_ply
from tests.test_orientation import inconsistent_edges, oriented, triangle_flags

COUNTS = ("num_vertices", "num_triangles", "unreferenced_vertices", "nonfinite_vertices", "degenerate_triangles",
          "zero_area_triangles", "nonfinite_triangles", "edges", "boundary_edges", "manifold_edges", "nonmanifold_edges",
          "misoriented_edges", "components")


def _min_total(x):
    """Exact float minimum with -0 below +0 (the device's rule, so that the order of its reduction cannot show)."""
    m = x.min()
    return np.float32(-0.0) if m == 0 and np.signbit(x[x == 0]).any() else m


def _max_total(x):
    m = x.max()
    return np.float32(0.0) if m == 0 and (~np.signbit(x[x == 0])).any() else m


def inspect_model(vertices, triangles):
    """dcsg_mesh_inspect in numpy.  Per-triangle terms in the same sequence of double operations as the device; sums with
    math.fsum.  Returns the report's fields, the per-component arrays, and `scale`: the sums of |term| the tolerances use."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    v = np.asarray(vertices, dtype=np.float32).reshape(-1, 3)
    t = np.asarray(triangles, dtype=np.int64).reshape(-1, 3)
    V, T = len(v), len(t)
    assert T == 0 or t.max() < V
    deg = (t[:, 0] == t[:, 1]) | (t[:, 1] == t[:, 2]) | (t[:, 0] == t[:, 2])
    g = t[~deg]
    ref = np.zeros(V, dtype=bool)
    ref[g.ravel()] = True
    finite_v = np.isfinite(v).all(axis=1)
    tri_finite = finite_v[g].all(axis=1)
    r = {"num_vertices": V, "num_triangles": T, "unreferenced_vertices": int(V - ref.sum()),
         "nonfinite_vertices": int((ref & ~finite_v).sum()), "degenerate_triangles": int(deg.sum()),
         "nonfinite_triangles": int((~tri_finite).sum())}
    # edges
    a, b = g.ravel(), g[:, [1, 2, 0]].ravel()
    key = (np.minimum(a, b) << 32) | np.maximum(a, b)
    _, inv, k = np.unique(key, return_inverse=True, return_counts=True)
    f = np.bincount(inv.ravel(), weights=(a < b), minlength=len(k))
    r.update(edges=len(k), boundary_edges=int((k == 1).sum()), manifold_edges=int((k == 2).sum()),
             nonmanifold_edges=int((k >= 3).sum()), misoriented_edges=int(((k == 2) & (f != 1)).sum()))
    # per-triangle terms (zero for non-finite triangles)
    p = v[g].astype(np.float64)
    A, B, C = p[:, 0], p[:, 1], p[:, 2]
    with np.errstate(all="ignore"):
        u, w = B - A, C - A
        n = np.stack([u[:, 1] * w[:, 2] - u[:, 2] * w[:, 1], u[:, 2] * w[:, 0] - u[:, 0] * w[:, 2],
                      u[:, 0] * w[:, 1] - u[:, 1] * w[:, 0]], axis=1)
        area = 0.5 * np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])
        vol = ((A[:, 0] * (B[:, 1] * C[:, 2] - B[:, 2] * C[:, 1]) + A[:, 1] * (B[:, 2] * C[:, 0] - B[:, 0] * C[:, 2]))
               + A[:, 2] * (B[:, 0] * C[:, 1] - B[:, 1] * C[:, 0])) / 6.0
        moment = vol[:, None] * ((A + B) + C)
    area[~tri_finite], vol[~tri_finite], moment[~tri_finite] = 0.0, 0.0, 0.0
    r["zero_area_triangles"] = int((tri_finite & (n == 0).all(axis=1)).sum())
    r["area"], r["signed_volume"] = math.fsum(area), math.fsum(vol)
    m = [math.fsum(moment[:, c]) for c in range(3)]
    r["centroid"] = [m[c] / (4.0 * r["signed_volume"]) if r["signed_volume"] != 0.0 else float("nan") for c in range(3)]
    use = v[ref & finite_v]
    r["bbox_min"] = [float(_min_total(use[:, c])) if len(use) else float("inf") for c in range(3)]
    r["bbox_max"] = [float(_max_total(use[:, c])) if len(use) else -float("inf") for c in range(3)]
    # components: labelled by their smallest vertex id, numbered in that order
    ends = np.concatenate([g[:, [0, 1]], g[:, [0, 2]]])
    graph = coo_matrix((np.ones(len(ends)), (ends[:, 0], ends[:, 1])), shape=(V, V))
    _, label = connected_components(graph, directed=False) if V else (0, np.zeros(0, np.int64))
    smallest = np.full(label.max() + 1 if V else 0, V, dtype=np.int64)
    np.minimum.at(smallest, label, np.arange(V))
    roots = np.unique(smallest[label[ref]])
    r["components"] = len(roots)
    comp = np.searchsorted(roots, smallest[label[g[:, 0]]]) if len(g) else np.zeros(0, np.int64)
    counts = np.bincount(comp, minlength=len(roots))
    order = np.argsort(comp, kind="stable")
    cuts = np.cumsum(counts)[:-1]
    r["component_triangles"] = counts.astype(np.uint64)
    r["component_area"] = np.array([math.fsum(x) for x in np.split(area[order], cuts)]) if len(roots) else np.zeros(0)
    r["component_signed_volume"] = np.array([math.fsum(x) for x in np.split(vol[order], cuts)]) if len(roots) else np.zeros(0)
    r["scale"] = {"area": np.abs(area).sum(), "signed_volume": np.abs(vol).sum(), "moment": np.abs(moment).sum(axis=0),
                  "component_area": np.bincount(comp, weights=np.abs(area), minlength=len(roots)),
                  "component_signed_volume": np.bincount(comp, weights=np.abs(vol), minlength=len(roots))}
    return r


def assert_report(got, want, components=True):
    """Every count and the box exactly; the sums within 1e-9 * sum |term| of fsum."""
    for name in COUNTS:
        assert got[name] == want[name], (name, got[name], want[name])
    for name in ("bbox_min", "bbox_max"):
        assert np.array_equal(np.array(got[name], np.float32).view(np.uint32), np.array(want[name], np.float32).view(np.uint32)), \
            (name, got[name], want[name])
    s = want["scale"]
    for name in ("area", "signed_volume"):
        assert abs(got[name] - want[name]) <= 1e-9 * s[name], (name, got[name], want[name])
    vol = want["signed_volume"]
    for c in range(3):
        if vol == 0.0:
            assert math.isnan(got["centroid"][c])
        else:
            # the error of sum moment / (4 sum vol) from the errors of the two sums
            tol = 1e-9 * (s["moment"][c] + abs(want["centroid"][c]) * 4.0 * s["signed_volume"]) / abs(4.0 * vol)
            assert abs(got["centroid"][c] - want["centroid"][c]) <= tol, (c, got["centroid"], want["centroid"])
    if components:
        assert np.array_equal(got["component_triangles"], want["component_triangles"])
        for name in ("component_area", "component_signed_volume"):
            assert np.all(np.abs(got[name] - want[name]) <= 1e-9 * s[name]), name


# ---- hand-made meshes ----------------------------------------------------------------------------------------------------------

def cube(offset=(0.0, 0.0, 0.0), first=0):
    """Unit cube: vertex i at (i & 1, i >> 1 & 1, i >> 2 & 1) + offset, ids from `first`, 12 outward-wound triangles."""
    v = np.array([(i & 1, i >> 1 & 1, i >> 2 & 1) for i in range(8)], dtype=np.float32) + np.asarray(offset, np.float32)
    tris = []
    for d in range(3):
        e1, e2 = [x for x in range(3) if x != d]
        for side in (0, 1):
            q = [(side << d) | (i << e1) | (j << e2) for i, j in ((0, 0), (1, 0), (1, 1), (0, 1))]
            for tri in ((q[0], q[1], q[2]), (q[0], q[2], q[3])):
                p = v[list(tri)].astype(np.float64)
                if np.cross(p[1] - p[0], p[2] - p[0]) @ (p.mean(axis=0) - (v.mean(axis=0))) < 0:
                    tri = (tri[0], tri[2], tri[1])
                tris.append(tri)
    return v, np.array(tris, dtype=np.uint32) + first


def hand_meshes():
    v, t = cube()
    v2, t2 = cube((3.0, 0.0, 0.0), 8)
    fin_v = np.array([(0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (0, -1, 0)], dtype=np.float32)
    nan_v = np.concatenate([v, [[np.nan, 0.5, 0.5]]]).astype(np.float32)
    return {
        "cube": (v, t),
        "cube_minus_one": (v, t[1:]),
        "cube_flipped": (v, np.concatenate([t[:1, [0, 2, 1]], t[1:]])),
        "two_cubes": (np.concatenate([v, v2]), np.concatenate([t, t2])),
        "fin": (fin_v, np.array([(0, 1, 2), (1, 0, 3), (0, 1, 4)], dtype=np.uint32)),
        "degenerate": (v, np.concatenate([t, [(0, 0, 1)]]).astype(np.uint32)),
        "zero_area": (np.concatenate([v, v[:1]]), np.concatenate([t, [(0, 8, 7)]]).astype(np.uint32)),
        "nan_vertex": (nan_v, np.concatenate([t, [(0, 1, 8)]]).astype(np.uint32)),
        "unreferenced": (np.concatenate([v, np.full((5, 3), 7.0, np.float32)]), t),
        "empty": (v[:4], np.zeros((0, 3), dtype=np.uint32)),
    }


def test_hand_made_meshes_have_the_known_answers():
    m = {name: inspect_model(v, t) for name, (v, t) in hand_meshes().items()}
    c = m["cube"]
    assert (c["edges"], c["manifold_edges"], c["boundary_edges"], c["misoriented_edges"], c["components"]) == (18, 18, 0, 0, 1)
    assert c["area"] == 6.0 and c["signed_volume"] == 1.0 and c["centroid"] == [0.5, 0.5, 0.5]
    assert c["bbox_min"] == [0.0] * 3 and c["bbox_max"] == [1.0] * 3
    assert (m["cube_minus_one"]["boundary_edges"], m["cube_minus_one"]["manifold_edges"]) == (3, 15)
    assert m["cube_flipped"]["misoriented_edges"] == 3 and m["cube_flipped"]["manifold_edges"] == 18
    two = m["two_cubes"]
    # the cube at x = 3 has terms / 6 that are not exact in double
    assert two["components"] == 2 and abs(two["signed_volume"] - 2.0) < 1e-14
    assert np.allclose(two["component_signed_volume"], [1.0, 1.0], rtol=0, atol=1e-14) and list(two["component_triangles"]) == [12, 12]
    assert np.allclose(two["centroid"], [2.0, 0.5, 0.5], rtol=0, atol=1e-14)
    fin = m["fin"]
    assert (fin["nonmanifold_edges"], fin["boundary_edges"], fin["edges"]) == (1, 6, 7)
    d = m["degenerate"]
    assert d["degenerate_triangles"] == 1 and d["edges"] == 18 and d["signed_volume"] == 1.0 and list(d["component_triangles"]) == [12]
    z = m["zero_area"]
    assert z["zero_area_triangles"] == 1 and z["boundary_edges"] == 3 and z["components"] == 1 and z["area"] == 6.0
    n = m["nan_vertex"]
    assert (n["nonfinite_vertices"], n["nonfinite_triangles"], n["components"]) == (1, 1, 1)
    assert n["area"] == 6.0 and n["bbox_max"] == [1.0] * 3 and list(n["component_triangles"]) == [13]
    u = m["unreferenced"]
    assert u["unreferenced_vertices"] == 5 and u["bbox_max"] == [1.0] * 3 and u["components"] == 1
    e = m["empty"]
    assert e["unreferenced_vertices"] == 4 and e["edges"] == e["components"] == 0 and e["area"] == 0.0
    assert all(math.isnan(x) for x in e["centroid"]) and e["bbox_min"] == [math.inf] * 3 and e["bbox_max"] == [-math.inf] * 3


_LATTICES = {}


def _lattice(name, level):
    from oracle.oracle import Oracle
    if (name, level) not in _LATTICES:
        orc = Oracle.for_scene(scenes.materialize(name), "port")
        box = orc.bbox(10.0)
        _LATTICES[(name, level)] = (box, orc.lattice_sdf(box, 1 << level))
    return _LATTICES[(name, level)]


@pytest.mark.parametrize("no_cull", [False, True])
@pytest.mark.parametrize("level", [5, 6, 7])
def test_cpu_mesher_edges_are_the_orientation_check(level, no_cull):
    box, lattice = _lattice("design1", level)
    mesh = H.emul_extract(lattice, box, level, no_cull=no_cull)
    tris = oriented(mesh["triangles"], triangle_flags(mesh["cell_masks"]))
    r = inspect_model(mesh["vertices"], tris)
    assert (r["manifold_edges"], r["misoriented_edges"]) == inconsistent_edges(tris)
    assert r["misoriented_edges"] == 0 and r["signed_volume"] > 0
    written = inspect_model(mesh["vertices"], mesh["triangles"])
    assert (written["manifold_edges"], written["misoriented_edges"]) == inconsistent_edges(mesh["triangles"])
    print("design1 2^%d cull=%d: %d edges, %d boundary, %d non-manifold, %d shells, volume %.4f"
          % (level, not no_cull, r["edges"], r["boundary_edges"], r["nonmanifold_edges"], r["components"], r["signed_volume"]))


def test_cli_refuses_inspect_on_several_ranks():
    proc = _run_cli(["inspect", "no_such_scene", "--level", "7"], {"WORLD_SIZE": "2", "RANK": "0", "LOCAL_RANK": "0"})
    assert proc.returncode != 0 and "one GPU" in proc.stdout and "touched" not in proc.stdout, proc.stdout


def test_cli_accepts_inspect():
    """On one rank the command gets as far as the build (which the test replaces by a failure)."""
    proc = _run_cli(["inspect", "no_such_scene", "--outward", "--components"], {"WORLD_SIZE": "1"})
    assert proc.returncode != 0 and "touched the build or the device" in proc.stdout, proc.stdout


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


def device_arrays(mesh):
    """The mesh's device vertices and triangles, read through torch once every queued stream is done."""
    import torch
    torch.cuda.synchronize()
    v = torch.as_tensor(mesh.device("vertices"), device="cuda").cpu().numpy() if mesh.num_vertices else np.zeros((0, 3), np.float32)
    t = torch.as_tensor(mesh.device("triangles"), device="cuda").cpu().numpy().view(np.uint32) if mesh.num_triangles \
        else np.zeros((0, 3), np.uint32)
    return v, t


def check(mesh):
    v, t = device_arrays(mesh)
    got = mesh.inspect(components=True)
    assert_report(got, inspect_model(v, t))
    return got


@pytest.mark.gpu
def test_hand_made_meshes_on_the_device(ctxs):
    """Written into a carrier mesh through its torch views; the counts set on a copy of its struct."""
    import torch
    from designcsg_b200 import api
    ctx = ctxs("design1")
    carrier = ctx.extract(ctx.bbox(10.0), 6, copy_to_host=False)
    vview = torch.as_tensor(carrier.device("vertices"), device="cuda")
    tview = torch.as_tensor(carrier.device("triangles"), device="cuda")
    part = api.Mesh(ctx)
    try:
        for name, (v, t) in hand_meshes().items():
            vview[:len(v)] = torch.from_numpy(np.ascontiguousarray(v, np.float32)).cuda()
            tview[:len(t)] = torch.from_numpy(np.ascontiguousarray(t, np.uint32).view(np.int32)).cuda()
            torch.cuda.synchronize()
            ctypes.memmove(ctypes.byref(part.c), ctypes.byref(carrier.c), ctypes.sizeof(api.MeshStruct))
            part.c.num_vertices, part.c.num_triangles = len(v), len(t)
            got = part.inspect(components=True)
            assert_report(got, inspect_model(v, t))
            print(name, {k: got[k] for k in COUNTS}, got["area"], got["signed_volume"], got["centroid"])
        v, t = hand_meshes()["cube"]
        t = t.copy()
        t[5, 1] = len(v)
        tview[:len(t)] = torch.from_numpy(t.view(np.int32)).cuda()
        torch.cuda.synchronize()
        part.c.num_vertices, part.c.num_triangles = len(v), len(t)
        with pytest.raises(api.DcsgError) as err:
            part.inspect()
        assert err.value.code == -2
    finally:
        part._ctx = None                                    # borrowed storage: the carrier frees it
        carrier.free()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["design1", "design2", "stress"])
@pytest.mark.parametrize("level", [6, 7])
@pytest.mark.parametrize("no_cull", [False, True])
@pytest.mark.parametrize("steps", [0, 50])
def test_library_meshes(ctxs, name, level, no_cull, steps):
    ctx = ctxs(name)
    mesh = ctx.extract(ctx.bbox(10.0), level, gd_steps=steps, no_cull=no_cull, copy_to_host=False)
    written = check(mesh)
    mesh.orient()
    wound = check(mesh)
    assert written["misoriented_edges"] > 0 and wound["misoriented_edges"] == 0
    assert wound["signed_volume"] > 0
    print("%s 2^%d cull=%d steps=%d: %d edges, %d boundary, %d non-manifold, %d misoriented as written, %d shells, area %.4f, "
          "volume %.4f" % (name, level, not no_cull, steps, wound["edges"], wound["boundary_edges"], wound["nonmanifold_edges"],
                           written["misoriented_edges"], wound["components"], wound["area"], wound["signed_volume"]))
    mesh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["design1", "design2"])
@pytest.mark.parametrize("retopologize", [False, True])
def test_shipped_levels(ctxs, name, retopologize):
    ctx = ctxs(name)
    search, lo, hi, grid, thr, steps = export_levels(name)
    mesh = ctx.extract(ctx.bbox(search), grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=retopologize,
                       defer_projection=True, copy_to_host=False)
    ctx.project(mesh, steps)
    soup = check(mesh)
    mesh.weld()
    welded = check(mesh)
    if not retopologize:        # a soup: every triangle has vertices of its own
        assert soup["edges"] == soup["boundary_edges"] == 3 * soup["num_triangles"] and soup["components"] == soup["num_triangles"]
    print("%s shipped levels, retopologize=%d, welded: %d triangles, %d edges, %d boundary, %d non-manifold, %d misoriented, "
          "%d degenerate, %d shells, volume %.4f" % (name, retopologize, welded["num_triangles"], welded["edges"],
                                                    welded["boundary_edges"], welded["nonmanifold_edges"], welded["misoriented_edges"],
                                                    welded["degenerate_triangles"], welded["components"], welded["signed_volume"]))
    mesh.free()


@pytest.mark.gpu
def test_full_size_design1(ctxs):
    ctx = ctxs("design1")
    mesh = ctx.extract(ctx.bbox(10.0), 10, defer_projection=True, copy_to_host=False)
    mesh.orient()
    ctx.project(mesh, 50)
    got = check(mesh)
    assert got["misoriented_edges"] == 0 and got["num_triangles"] > 8_000_000
    print("design1 1024^3:", {k: got[k] for k in COUNTS}, got["area"], got["signed_volume"], got["centroid"])
    mesh.free()


def _same_report(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.dtype == y.dtype and x.tobytes() == y.tobytes(), k


@pytest.mark.gpu
def test_deterministic_and_pure(ctxs):
    import torch
    ctx = ctxs("design2")
    box = ctx.bbox(10.0)
    mesh = ctx.extract(box, 7, gd_steps=50)
    mesh.orient()
    h = (mesh.vertices(), mesh.triangles(), mesh.cell_masks())
    d = [torch.as_tensor(mesh.device(k), device="cuda").clone() for k in ("vertices", "triangles", "cell_masks")]
    first = mesh.inspect(components=True)
    second = mesh.inspect(components=True)
    _same_report(first, second)
    assert all(torch.equal(a.view(torch.uint8), torch.as_tensor(mesh.device(k), device="cuda").view(torch.uint8))
               for a, k in zip(d, ("vertices", "triangles", "cell_masks")))
    assert all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip(h, (mesh.vertices(), mesh.triangles(), mesh.cell_masks())))
    # four z-slabs: each a mesh of its own, their terms those of the whole
    whole = mesh.inspect()
    want = inspect_model(mesh.vertices(), mesh.triangles())
    n = 1 << 7
    slabs = []
    for r in range(4):
        slab = ctx.extract(box, 7, gd_steps=50, slab=(r * n // 4, (r + 1) * n // 4))
        slab.orient()
        slabs.append(check(slab))
        slab.free()
    assert sum(s["num_triangles"] for s in slabs) == whole["num_triangles"]
    assert sum(s["boundary_edges"] for s in slabs) > whole["boundary_edges"]           # the cuts
    for name in ("area", "signed_volume"):
        assert abs(sum(s[name] for s in slabs) - whole[name]) <= 2e-9 * want["scale"][name], name
    mesh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("level,outward", [(7, False), (7, True), (0, False)])
def test_cli_reports_the_indexed_file(ctxs, tmp_path, level, outward):
    """`inspect` prints the report of the mesh `export --ply-indexed` writes with the same options (level 0 = the design's
    shipped levels)."""
    ctx = ctxs("design1")
    scene = scenes.materialize("design1")["dir"]
    path = str(tmp_path / "i.ply")
    ctx.export_indexed(scene, level, path, outward=outward)
    xyz, _, faces = read_indexed_ply(path)
    args = [sys.executable, "-m", "designcsg_b200", "inspect", scene, "--components"] + (["--level", str(level)] if level else []) \
        + (["--outward"] if outward else [])
    proc = subprocess.run(args, cwd=H.REPO, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert proc.returncode == 0, proc.stderr[-3000:]
    got = json.loads(proc.stdout.strip().split("\n")[-1])
    for k in ("component_triangles", "component_area", "component_signed_volume"):
        got[k] = np.array(got[k], dtype=np.uint64 if k == "component_triangles" else np.float64)
    assert_report(got, inspect_model(xyz, faces))


@pytest.mark.gpu
def test_gathered_whole_on_one_rank(tmp_path):
    """The borrowed `whole` of a one-rank gather inspects like the single-GPU extraction."""
    import torch  # noqa: F401  (before the communicator, see tests/test_sharded_export.py)
    from designcsg_b200 import api
    try:
        uid = api.comm_unique_id()
    except api.DcsgError as e:
        if e.code != -7:
            raise
        pytest.skip("NCCL is not loadable: %s" % e)
    ctx = api.Context(0)
    ctx.build(scenes.materialize("design1")["dir"])
    comm = api.Comm(ctx, uid, 0, 1)
    try:
        box = comm.bbox(10.0)
        local, whole, _ = comm.extract(box, 7, gd_steps=50, gather_to=0)
        gathered = whole.inspect(components=True)
        whole._ctx = None                                   # borrowed arrays: nothing to free
        single = ctx.extract(box, 7, gd_steps=50)
        _same_report(gathered, single.inspect(components=True))
        assert gathered["num_triangles"] > 0
        single.free()
        local.free()
    finally:
        comm.close()
        ctx.close()
