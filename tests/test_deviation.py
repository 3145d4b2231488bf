"""Mesh deviation (dcsg_mesh_deviation, Mesh.deviation, `inspect --deviation`): the scene's SDF sampled at the vertices and over
every triangle.  The definition (include/dcsg.h, DESIGN.md 7e) is restated in numpy operation for operation (deviation_model)
with any SDF; it is checked on hand-made meshes with known answers and on the CPU mesher harness with the oracle's SDF, and
on the device against the model with the library's own dcsg_eval_sdf."""
import ctypes
import json
import math
import subprocess
import sys

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes
from tests.test_indexed_export import _run_cli, export_levels
from tests.test_inspect import _max_total, _min_total, device_arrays, hand_meshes

FLOATS = ("vertex_max_abs", "min_sdf", "max_sdf", "max_abs")
COUNTS = ("num_vertices", "num_triangles", "measured_vertices", "measured_triangles", "samples", "nan_samples", "over_tolerance",
          "worst_triangle")
NO_TRIANGLE = 2 ** 64 - 1


def sample_ij(k):
    """The (i, j) of the S = (k+1)(k+2)/2 - 3 samples of a triangle, i ascending then j ascending, corners excluded."""
    return [(i, j) for i in range(k + 1) for j in range(k + 1 - i) if (i, j) not in ((0, 0), (k, 0), (0, k))]


def sample_points(v, t, k):
    """(T, S, 3) float32: ((a * (k-i-j) + b * i) + c * j) / k per coordinate, one IEEE float operation at a time."""
    ij = sample_ij(k)
    a, b, c = v[t[:, 0]], v[t[:, 1]], v[t[:, 2]]
    out = np.empty((len(t), len(ij), 3), np.float32)
    with np.errstate(all="ignore"):
        for s, (i, j) in enumerate(ij):
            out[:, s] = ((a * np.float32(k - i - j) + b * np.float32(i)) + c * np.float32(j)) / np.float32(k)
    return out


def triangle_area(v, t):
    """dcsg_mesh_inspect's area_t: the same double sequence as tests/test_inspect.py's inspect_model."""
    p = v[t].astype(np.float64)
    A, B, C = p[:, 0], p[:, 1], p[:, 2]
    u, w = B - A, C - A
    n = np.stack([u[:, 1] * w[:, 2] - u[:, 2] * w[:, 1], u[:, 2] * w[:, 0] - u[:, 0] * w[:, 2], u[:, 0] * w[:, 1] - u[:, 1] * w[:, 0]], axis=1)
    return 0.5 * np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])


def deviation_model(vertices, triangles, k, tolerance, sdf):
    """dcsg_mesh_deviation in numpy.  sdf: a callable on float32 (n, 3) arrays returning n float32 values.  Returns the report's
    fields, `triangle_max_abs`, the measured triangles' sample points and values, and `scale`: the sums of |term| the
    tolerances of the two double results use."""
    v = np.asarray(vertices, dtype=np.float32).reshape(-1, 3)
    t = np.asarray(triangles, dtype=np.int64).reshape(-1, 3)
    V, T, S = len(v), len(t), len(sample_ij(k))
    assert T == 0 or t.max() < V
    deg = (t[:, 0] == t[:, 1]) | (t[:, 1] == t[:, 2]) | (t[:, 0] == t[:, 2])
    ref = np.zeros(V, dtype=bool)
    ref[t[~deg].ravel()] = True
    finite_v = np.isfinite(v).all(axis=1)
    measured_v = ref & finite_v
    measured_t = ~deg & finite_v[t].all(axis=1) if T else np.zeros(0, bool)
    fv = np.asarray(sdf(v), np.float32) if V else np.zeros(0, np.float32)
    idx = np.nonzero(measured_t)[0]
    tm = t[idx]
    pts = sample_points(v, tm, k)
    fs = np.asarray(sdf(pts.reshape(-1, 3)), np.float32).reshape(len(tm), S) if len(tm) and S else np.zeros((len(tm), S), np.float32)
    vals = np.concatenate([fv[tm].reshape(len(tm), 3), fs], axis=1)
    nan = np.isnan(vals)
    with np.errstate(invalid="ignore"):
        absx = np.abs(vals)
        w = np.where(nan, np.float32(-np.inf), absx)
    best = w.max(axis=1) if len(tm) else np.zeros(0, np.float32)
    slot = w.argmax(axis=1) if len(tm) else np.zeros(0, np.int64)
    clean = ~nan.any(axis=1)
    tmax = np.full(T, np.nan, np.float32)
    tmax[idx] = np.where(clean, best, np.float32(np.nan))
    r = {"num_vertices": V, "num_triangles": T, "measured_vertices": int(measured_v.sum()), "measured_triangles": len(idx),
         "samples": int(measured_v.sum()) + S * len(idx), "nan_samples": int(np.isnan(fv[measured_v]).sum() + np.isnan(fs).sum()),
         "over_tolerance": int((~(tmax[idx] <= np.float32(tolerance))).sum()), "triangle_max_abs": tmax, "points": pts,
         "values": vals, "index": idx}
    good = vals[~nan]
    r["min_sdf"] = float(_min_total(good)) if good.size else math.inf
    r["max_sdf"] = float(_max_total(good)) if good.size else -math.inf
    r["max_abs"] = float(best.max()) if len(best) else -math.inf
    r["worst_triangle"], r["worst_point"] = NO_TRIANGLE, [math.nan] * 3
    if r["max_abs"] > -math.inf:
        row = int(np.argmax(best == np.float32(r["max_abs"])))
        r["worst_triangle"] = int(idx[row])
        s = int(slot[row])
        r["worst_point"] = [float(x) for x in (v[tm[row, s]] if s < 3 else pts[row, s - 3])]
    # area-weighted mean over the clean measured triangles: mean_t = sequential double sum of |f| / (3 + S)
    total = np.zeros(len(tm))
    for n in range(3 + S):
        total = total + absx[:, n].astype(np.float64)
    mean = total / float(3 + S)
    area = triangle_area(v, tm) if len(tm) else np.zeros(0)
    am = (area * mean)[clean]
    sum_area = math.fsum(area[clean])
    r["mean_abs"] = math.fsum(am) / sum_area if sum_area != 0.0 else math.nan
    vv = fv[measured_v]
    vv = vv[~np.isnan(vv)]
    r["vertex_max_abs"] = float(np.abs(vv).max()) if len(vv) else -math.inf
    sq = vv.astype(np.float64) * vv.astype(np.float64)
    r["vertex_rms"] = math.sqrt(math.fsum(sq) / len(vv)) if len(vv) else math.nan
    r["scale"] = {"mean_abs": (np.abs(am).sum() + abs(r["mean_abs"]) * area[clean].sum()) / sum_area if sum_area else 0.0,
                  "vertex_rms": r["vertex_rms"] if len(vv) else 0.0}
    return r


def _same_f32(a, b):
    a, b = np.float32(a), np.float32(b)
    return (np.isnan(a) and np.isnan(b)) or a.view(np.uint32) == b.view(np.uint32)


def assert_deviation(got, want):
    """Counts, extremes, worst triangle and point, triangle_max_abs: exact (NaN as NaN); the two double results within
    1e-9 * sum |term| of fsum."""
    for name in COUNTS:
        assert got[name] == want[name], (name, got[name], want[name])
    for name in FLOATS:
        assert _same_f32(got[name], want[name]), (name, got[name], want[name])
    assert all(_same_f32(x, y) for x, y in zip(got["worst_point"], want["worst_point"])), (got["worst_point"], want["worst_point"])
    if "triangle_max_abs" in got:
        g, w = got["triangle_max_abs"], want["triangle_max_abs"]
        assert np.array_equal(np.isnan(g), np.isnan(w))
        ok = ~np.isnan(w)
        assert np.array_equal(g[ok].view(np.uint32), w[ok].view(np.uint32))
    for name in ("mean_abs", "vertex_rms"):
        if math.isnan(want[name]):
            assert math.isnan(got[name]), name
        else:
            assert abs(got[name] - want[name]) <= 1e-9 * want["scale"][name], (name, got[name], want[name])


# ---- CPU ----------------------------------------------------------------------------------------------------------------------

def octahedron():
    v = np.array([(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)], np.float32)
    t = [(x, y, z) for x in (0, 1) for y in (2, 3) for z in (4, 5)]
    return v, np.array(t, np.uint32)


def unit_sphere(p):
    p = np.asarray(p, np.float32)
    return np.sqrt((p * p).sum(axis=1, dtype=np.float32)) - np.float32(1.0)


def test_octahedron_known_answers():
    v, t = octahedron()
    r = deviation_model(v, t, 3, 0.1, unit_sphere)
    centroid = np.float32(1.0) / np.float32(3.0)
    assert sample_ij(3).index((1, 1)) == 3
    assert np.all(r["values"][:, :3] == 0.0)                                   # every corner is on the sphere
    assert np.all(np.abs(r["points"][:, 3]) == centroid)
    f_centroid = unit_sphere([[centroid] * 3])[0]
    assert abs(float(f_centroid) - (1 / math.sqrt(3) - 1)) < 1e-6
    assert r["min_sdf"] == float(f_centroid) and r["max_sdf"] == 0.0 and r["max_abs"] == -float(f_centroid)
    assert r["samples"] == 6 + 7 * 8 and r["measured_triangles"] == 8 and r["measured_vertices"] == 6
    assert r["over_tolerance"] == 8 and deviation_model(v, t, 3, 0.5, unit_sphere)["over_tolerance"] == 0
    # all eight faces tie: the smallest index wins, at its first sample that reaches the maximum (the centroid)
    assert np.all(r["triangle_max_abs"] == r["max_abs"])
    assert r["worst_triangle"] == 0 and r["worst_point"] == [float(centroid)] * 3
    rolled = deviation_model(v, np.roll(t, -3, axis=0), 3, 0.1, unit_sphere)
    assert rolled["worst_triangle"] == 0
    # one face moved closer: it alone is the worst
    t2 = t.copy()
    v2 = np.concatenate([v, [[0.5, 0.0, 0.0]]]).astype(np.float32)
    t2[5, 0] = 6
    r2 = deviation_model(v2, t2, 3, 0.1, unit_sphere)
    assert r2["worst_triangle"] == 5 and r2["max_abs"] > r["max_abs"]
    assert r["vertex_max_abs"] == 0.0 and r["vertex_rms"] == 0.0 and 0.0 < r["mean_abs"] < r["max_abs"]
    print("octahedron k=3:", {k: r[k] for k in COUNTS + FLOATS}, r["mean_abs"])


@pytest.mark.parametrize("k", range(1, 17))
def test_sample_count(k):
    v, t = octahedron()
    ij = sample_ij(k)
    assert len(ij) == (k + 1) * (k + 2) // 2 - 3 and ij == sorted(ij) and len(set(ij)) == len(ij)
    r = deviation_model(v, t, k, 0.0, unit_sphere)
    assert r["samples"] == 6 + 8 * len(ij) and r["points"].shape == (8, len(ij), 3)
    assert r["over_tolerance"] == (8 if k > 1 else 0)


def test_unmeasured_and_nan_valued_triangles():
    m = hand_meshes()
    plane = lambda p: np.asarray(p, np.float32)[:, 0] - np.float32(0.25)
    d = deviation_model(*m["degenerate"], 4, 1.0, plane)
    assert math.isnan(d["triangle_max_abs"][-1]) and not np.isnan(d["triangle_max_abs"][:-1]).any()
    assert (d["measured_triangles"], d["measured_vertices"], d["nan_samples"]) == (12, 8, 0)
    n = deviation_model(*m["nan_vertex"], 4, 1.0, plane)
    assert math.isnan(n["triangle_max_abs"][-1]) and n["measured_triangles"] == 12 and n["measured_vertices"] == 8
    assert n["samples"] == 8 + 12 * 12 and n["over_tolerance"] == 0
    u = deviation_model(*m["unreferenced"], 4, 1.0, plane)
    assert u["measured_vertices"] == 8 and u["vertex_max_abs"] == 0.75
    # NaN values: the SDF is NaN on the plane x = 1, which every face but x = 0 touches
    nan_at_one = lambda p: np.where(np.asarray(p, np.float32)[:, 0] == 1.0, np.float32(np.nan), plane(p))
    c = deviation_model(*m["cube"], 4, 10.0, nan_at_one)
    bad = np.isnan(c["triangle_max_abs"])
    assert bad.sum() == 10 and c["over_tolerance"] == 10 and c["measured_triangles"] == 12
    assert c["nan_samples"] == 4 + int((c["points"][..., 0] == 1.0).sum()) and c["nan_samples"] > 4 + 2 * 12
    assert math.isnan(c["mean_abs"]) is False and c["vertex_max_abs"] == 0.25 and c["min_sdf"] == -0.25
    # the worst value (x = 0.75 in a face that touches x = 1) lies in a triangle whose triangle_max_abs is NaN
    assert c["max_abs"] == 0.5 and bad[c["worst_triangle"]] and c["worst_point"][0] == 0.75
    e = deviation_model(*m["empty"], 4, 1.0, plane)
    assert (e["samples"], e["worst_triangle"], e["max_abs"], e["min_sdf"]) == (0, NO_TRIANGLE, -math.inf, math.inf)
    assert math.isnan(e["mean_abs"]) and math.isnan(e["vertex_rms"]) and all(math.isnan(x) for x in e["worst_point"])


def test_oracle_design1_cpu_mesh():
    """The model with the oracle's CPU SDF on the CPU mesher harness's Design1 mesh at 2^5."""
    from oracle.oracle import Oracle
    orc = Oracle.for_scene(scenes.materialize("design1"), "port")
    box = orc.bbox(10.0)
    mesh = H.emul_extract(orc.lattice_sdf(box, 1 << 5), box, 5)
    cell = float(box[3]) / 32
    r = deviation_model(mesh["vertices"], mesh["triangles"], 4, cell / 10, orc.eval_sdf)
    assert r["measured_triangles"] == len(mesh["triangles"]) and r["nan_samples"] == 0
    assert r["max_abs"] < cell and r["min_sdf"] < 0 < r["max_sdf"]
    print("design1 2^5 (oracle, k=4, tol=cell/10):", {k: r[k] for k in COUNTS + FLOATS}, r["mean_abs"], r["vertex_rms"])


@pytest.mark.parametrize("extra,message", [(["--subdivision", "0"], "--subdivision"), (["--subdivision", "17"], "--subdivision"),
                                           (["--tolerance", "-1"], "--tolerance"), (["--tolerance", "nan"], "--tolerance")])
def test_cli_refuses_bad_deviation_options(extra, message):
    proc = _run_cli(["inspect", "no_such_scene", "--deviation"] + extra, {"WORLD_SIZE": "1"})
    assert proc.returncode != 0 and message in proc.stdout and "touched" not in proc.stdout, proc.stdout


def test_cli_accepts_deviation():
    proc = _run_cli(["inspect", "no_such_scene", "--deviation", "--subdivision", "9", "--tolerance", "0.01"], {"WORLD_SIZE": "1"})
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


def check(ctx, mesh, k, tolerance=0.0):
    v, t = device_arrays(mesh)
    got = mesh.deviation(k, tolerance, per_triangle=True)
    want = deviation_model(v, t, k, tolerance, ctx.eval_sdf)
    assert_deviation(got, want)
    return got, want


@pytest.mark.gpu
def test_hand_made_meshes_on_the_device(ctxs):
    """Written into a carrier mesh through its torch views (tests/test_inspect.py's technique), scaled into Design1."""
    import torch
    from designcsg_b200 import api
    ctx = ctxs("design1")
    carrier = ctx.extract(ctx.bbox(10.0), 6, copy_to_host=False)
    vview = torch.as_tensor(carrier.device("vertices"), device="cuda")
    tview = torch.as_tensor(carrier.device("triangles"), device="cuda")
    part = api.Mesh(ctx)
    try:
        meshes = dict(hand_meshes(), octahedron=octahedron())
        for name, (v, t) in meshes.items():
            v = (np.asarray(v, np.float32) * np.float32(0.7) - np.float32(0.3)).astype(np.float32)
            vview[:len(v)] = torch.from_numpy(np.ascontiguousarray(v)).cuda()
            tview[:len(t)] = torch.from_numpy(np.ascontiguousarray(t, np.uint32).view(np.int32)).cuda()
            torch.cuda.synchronize()
            ctypes.memmove(ctypes.byref(part.c), ctypes.byref(carrier.c), ctypes.sizeof(api.MeshStruct))
            part.c.num_vertices, part.c.num_triangles = len(v), len(t)
            for k in (1, 4, 9):
                got, _ = check(ctx, part, k, 0.05)
            print(name, {k: got[k] for k in COUNTS + FLOATS})
        for k, tol in ((0, 0.0), (17, 0.0), (4, -1.0), (4, float("nan"))):
            with pytest.raises(api.DcsgError) as err:
                part.deviation(k, tol)
            assert err.value.code == -2
        v, t = hand_meshes()["cube"]
        t = t.copy()
        t[5, 1] = len(v)
        tview[:len(t)] = torch.from_numpy(t.view(np.int32)).cuda()
        torch.cuda.synchronize()
        part.c.num_vertices, part.c.num_triangles = len(v), len(t)
        with pytest.raises(api.DcsgError) as err:
            part.deviation()
        assert err.value.code == -2
    finally:
        part._ctx = None                                    # borrowed storage: the carrier frees it
        carrier.free()


@pytest.mark.gpu
def test_before_build():
    from designcsg_b200 import api, build
    build.build()
    ctx = api.Context(0)
    try:
        with pytest.raises(api.DcsgError) as err:
            api.Mesh(ctx).deviation()
        assert err.value.code == -4
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["design1", "design2", "stress"])
@pytest.mark.parametrize("level", [6, 7])
@pytest.mark.parametrize("no_cull", [False, True])
def test_library_meshes(ctxs, name, level, no_cull):
    from oracle.oracle import Oracle
    ctx = ctxs(name)
    box = ctx.bbox(10.0)
    cell = float(box[3]) / (1 << level)
    rms = {}
    for steps in (0, 50):
        mesh = ctx.extract(box, level, gd_steps=steps, no_cull=no_cull, copy_to_host=False)
        for k in (1, 4, 9):
            got, want = check(ctx, mesh, k, cell / 10)
            print("%s 2^%d cull=%d steps=%d k=%d:" % (name, level, not no_cull, steps, k), {x: got[x] for x in COUNTS + FLOATS},
                  got["mean_abs"], got["vertex_rms"])
        rms[steps] = got["vertex_rms"]
        mesh.free()
    assert rms[50] < rms[0], rms
    # the values are the reference's: a few hundred of the last samples through the oracle's CPU SDF, bit for bit
    orc = Oracle.for_scene(scenes.materialize(name), "port")
    pts = want["points"].reshape(-1, 3)
    pick = np.random.default_rng(level).choice(len(pts), size=min(300, len(pts)), replace=False)
    assert np.array_equal(orc.eval_sdf(pts[pick]).view(np.uint32), want["values"][:, 3:].reshape(-1)[pick].view(np.uint32))


@pytest.mark.gpu
def test_chunks(ctxs):
    """Design1 at 2^9 with k = 4: about 25 M samples, more than one chunk of 2^24."""
    ctx = ctxs("design1")
    mesh = ctx.extract(ctx.bbox(10.0), 9, gd_steps=50, copy_to_host=False)
    assert mesh.num_triangles * 12 > 1 << 24
    got, _ = check(ctx, mesh, 4, 1e-3)
    print("design1 2^9 k=4:", {k: got[k] for k in COUNTS + FLOATS}, got["mean_abs"], got["vertex_rms"])
    mesh.free()


SPHERE = """from DesignCSG import *
import numpy as np
draw(sphere_brush, Transform.initial(position=np.array([0.0, 0.0, 0.0]), yaw=0.0, pitch=0.0, roll=0.0, scale=np.array([1.0, 1.0, 1.0])))
commit()
"""


@pytest.mark.gpu
def test_sphere_sagitta(tmp_path):
    """A sphere: chords lie inside it, so the samples reach below the surface by at most the sagitta e^2 / (8 r).  Its compiled
    SDF is g (|p| - r) with a gradient g below 1 -- an SDF value, not a distance -- so the bound is g e^2 / (8 r) in f."""
    from designcsg_b200 import api, build
    build.build()
    (tmp_path / "sphere.py").write_text(SPHERE)
    scene = api.compile_design(str(tmp_path / "sphere.py"), str(tmp_path / "scene"))
    ctx = api.Context(0)
    try:
        ctx.build(scene)
        f0, f1 = (float(x) for x in ctx.eval_sdf(np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0]], np.float32)))
        g, r = f1 - f0, -f0 / (f1 - f0)
        assert 0 < g <= 1 and abs(float(ctx.eval_sdf(np.array([[0.0, -r, 0.0]], np.float32))[0])) < 1e-6
        box = ctx.bbox(10.0)
        worst = {}
        for level in (6, 7):
            mesh = ctx.extract(box, level, gd_steps=50, copy_to_host=False)
            got, _ = check(ctx, mesh, 4, 0.0)
            v, t = device_arrays(mesh)
            p = v[t].astype(np.float64)
            e = max(np.linalg.norm(p[:, i] - p[:, (i + 1) % 3], axis=1).max() for i in range(3))
            assert got["max_sdf"] <= got["vertex_max_abs"]
            assert got["max_abs"] <= g * e * e / (8.0 * r) + got["vertex_max_abs"] + 1e-6, (got["max_abs"], g, r, e)
            worst[level] = got["max_abs"]
            print("sphere r=%.3f g=%.3f 2^%d: longest edge %.4e, bound %.4e, max_abs %.4e" % (r, g, level, e, g * e * e / (8 * r), got["max_abs"]))
            mesh.free()
        assert worst[7] < worst[6]
        print("sphere: max_abs 2^6 %.3e, 2^7 %.3e, ratio %.3f" % (worst[6], worst[7], worst[6] / worst[7]))
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["design1", "design2"])
def test_shipped_levels_welded(ctxs, name):
    ctx = ctxs(name)
    search, lo, hi, grid, thr, steps = export_levels(name)
    mesh = ctx.extract(ctx.bbox(search), grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=True,
                       defer_projection=True, copy_to_host=False)
    mesh.weld()
    ctx.project(mesh, steps)
    got, _ = check(ctx, mesh, 4, 1e-3)
    print("%s shipped levels, welded:" % name, {k: got[k] for k in COUNTS + FLOATS}, got["mean_abs"])
    mesh.free()


@pytest.mark.gpu
def test_slab(ctxs):
    ctx = ctxs("design2")
    mesh = ctx.extract(ctx.bbox(10.0), 7, gd_steps=50, slab=(32, 80), copy_to_host=False)
    got, _ = check(ctx, mesh, 4, 1e-3)
    assert got["measured_triangles"] == mesh.num_triangles > 0
    mesh.free()


@pytest.mark.gpu
def test_exact_only_build_gives_the_same_bits(ctxs, monkeypatch):
    from designcsg_b200 import api
    fast = ctxs("design1")
    box = fast.bbox(10.0)
    mesh = fast.extract(box, 6, gd_steps=50, copy_to_host=False)
    want = mesh.deviation(4, 1e-3, per_triangle=True)
    monkeypatch.setenv("DCSG_EXACT_ONLY", "1")
    exact = api.Context(0)
    try:
        exact.build(scenes.materialize("design1")["dir"])
        other = exact.extract(box, 6, gd_steps=50, copy_to_host=False)
        assert np.array_equal(device_arrays(other)[0].view(np.uint32), device_arrays(mesh)[0].view(np.uint32))
        got = other.deviation(4, 1e-3, per_triangle=True)
        _same_report(got, want)
        other.free()
    finally:
        exact.close()
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
    mesh = ctx.extract(ctx.bbox(10.0), 7, gd_steps=50)
    mesh.orient()
    h = (mesh.vertices(), mesh.triangles(), mesh.cell_masks())
    d = [torch.as_tensor(mesh.device(k), device="cuda").clone() for k in ("vertices", "triangles", "cell_masks")]
    first = mesh.deviation(9, 1e-3, per_triangle=True)
    second = mesh.deviation(9, 1e-3, per_triangle=True)
    _same_report(first, second)
    torch.cuda.synchronize()
    assert all(torch.equal(a.view(torch.uint8), torch.as_tensor(mesh.device(k), device="cuda").view(torch.uint8))
               for a, k in zip(d, ("vertices", "triangles", "cell_masks")))
    assert all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip(h, (mesh.vertices(), mesh.triangles(), mesh.cell_masks())))
    mesh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("level", [7, 0])
def test_cli_reports_the_deviation(ctxs, level):
    """`inspect --deviation` reports Mesh.deviation of the mesh it builds the way `inspect` does (level 0 = shipped levels)."""
    ctx = ctxs("design1")
    scene = scenes.materialize("design1")["dir"]
    args = [sys.executable, "-m", "designcsg_b200", "inspect", scene, "--deviation", "--subdivision", "5"] \
        + (["--level", str(level)] if level else [])
    proc = subprocess.run(args, cwd=H.REPO, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert proc.returncode == 0, proc.stderr[-3000:]
    got = json.loads(proc.stdout.strip().split("\n")[-1])["deviation"]
    search, lo, hi, grid, thr, steps = export_levels("design1")
    if level:
        lo = hi = grid = level
    box = ctx.bbox(search)
    mesh = ctx.extract(box, grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=True, defer_projection=True,
                       copy_to_host=False)
    if not (lo >= grid and hi == grid):
        mesh.weld()
    ctx.project(mesh, steps)
    cell = float(max(box[3:6])) / (1 << grid)
    want = mesh.deviation(5, cell / 10)
    assert got["cell"] == cell and got["tolerance"] == cell / 10 and got["subdivision"] == 5
    for k, x in want.items():
        assert _same_f32(got[k], x) if k in FLOATS else got[k] == x, (k, got[k], x)
    mesh.free()
