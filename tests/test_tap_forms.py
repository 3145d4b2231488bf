"""The two tap forms of the checked fast copy (DESIGN.md 3b): the rolled loop over one inlined evaluation, and the per-axis
straight-line forms (host_scene.cu, generate_primary_sdf_axis) in which the taps of a normal along one axis share the work
of the unchanged coordinates.

On the CPU: the per-axis functions and the single-evaluation fast function are cut out of dcsg_scene_source() and compiled
for the host around the same brush text (tests/cpu_emul/tap_axes.cpp).  Wherever the round's flag stays down each of the seven
values equals the single evaluation at v + offset[k] bit for bit, and a zero or NaN coordinate always raises the flag.
On the GPU: DCSG_TAP_FORM=loop and =axis give the same normals, the same projected meshes and the same projection counters."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes
from tests.test_fast_copy_host import SCENES, _function

HERE = os.path.dirname(os.path.abspath(__file__))
AXIS_FUNCTIONS = ["dcsg_primary_sdf_xc(", "dcsg_primary_sdf_x(", "dcsg_primary_sdf_y(", "dcsg_primary_sdf_z("]


def _build(scene):
    from designcsg_b200 import api
    from oracle.build import cl_to_cpp
    src = api.scene_source(scene["dir"])
    fast = src[src.index("namespace dcsg_fast {\n__device__ float sdf_bank("):]
    parts = [_function(fast, "float dcsg_primary_sdf(float3 dcsg_v, bool& dcsg_inexact_out) {")]
    parts += [_function(fast, "void " + f + "float3 dcsg_v, float dcsg_e, float (&dcsg_out)") for f in AXIS_FUNCTIONS]
    generated = "\n".join(parts)
    text = cl_to_cpp(scene["scene.cl"], scene=True)
    out = os.path.join(HERE, "cpu_emul", "_build", "axes_" + hashlib.sha256((generated + text).encode()).hexdigest()[:16])
    lib = os.path.join(out, "libtapaxes.so")
    if not os.path.exists(lib):
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "generated.inc"), "w") as f:
            f.write(generated)
        with open(os.path.join(out, "scene.inc"), "w") as f:
            f.write(text)
        cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-fpermissive",
               "-I", os.path.join(H.REPO, "oracle"), '-DGENERATED_INC="%s"' % os.path.join(out, "generated.inc"),
               '-DSCENE_INC="%s"' % os.path.join(out, "scene.inc"), os.path.join(HERE, "cpu_emul", "tap_axes.cpp"), "-o", lib + ".tmp"]
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert proc.returncode == 0, proc.stdout[-4000:]
        os.replace(lib + ".tmp", lib)
    return ctypes.CDLL(lib), generated


def _eval(lib, scene, pts):
    """-> (axis values [n, 9]: +x -x +y -y +z -z centre of the round with the centre, then +x -x of the x function without it;
    single evaluations at the seven taps [n, 7]; flag of the round; flag of the round without the centre; any single
    evaluation flagged)"""
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    table = np.zeros(131072, dtype=np.float32)
    raw = open(os.path.join(scene["dir"], "arbitrary_data.hex"), "rb").read()
    table[:len(raw) // 4] = np.frombuffer(raw, dtype="<f4")
    n = len(pts)
    axes, single = np.empty((n, 9), np.float32), np.empty((n, 7), np.float32)
    flag, flag6, single_flag = np.empty(n, np.uint8), np.empty(n, np.uint8), np.empty(n, np.uint8)
    f32p, u8p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint8)
    lib.tap_axes_eval(pts.ctypes.data_as(f32p), ctypes.c_size_t(n), table.ctypes.data_as(f32p), axes.ctypes.data_as(f32p),
                      single.ctypes.data_as(f32p), flag.ctypes.data_as(u8p), flag6.ctypes.data_as(u8p), single_flag.ctypes.data_as(u8p))
    return axes, single, flag.astype(bool), flag6.astype(bool), single_flag.astype(bool)


def _same(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.mark.parametrize("name", SCENES)
def test_axis_forms_equal_single_evaluations_wherever_unflagged(name, libdcsg):
    scene = scenes.materialize(name)
    lib, _ = _build(scene)
    rng = np.random.default_rng(13)
    random = rng.uniform(-4.5, 4.5, (100000, 3)).astype(np.float32)
    dyadic = (np.round(rng.uniform(-4.5, 4.5, (100000, 3)) * 16) / 16).astype(np.float32)      # on lattice planes, zeros
    e = np.float32(0.005)
    vals = np.array([0.0, -0.0, e, -e, 2 * e, 5.0, -5.0, 5.0 + e, 1e-30, -1e-45, 2.0 ** -61, 1e37, -3e38, np.inf, -np.inf,
                     np.nan, 1.5, -0.75, 4.9999995, 2.5], dtype=np.float32)
    special = np.stack(np.meshgrid(vals, vals, vals, indexing="ij"), axis=-1).reshape(-1, 3)
    with np.errstate(all="ignore"):
        for label, pts in (("random", random), ("dyadic", dyadic), ("special", special)):
            axes, single, flag, flag6, single_flag = _eval(lib, scene, pts)
            same = _same(axes[:, :7], single)
            assert same[~flag].all(), "%s / %s: %d unflagged rounds differ" % (name, label, int((~same.all(axis=1) & ~flag).sum()))
            same6 = _same(axes[:, [7, 8, 2, 3, 4, 5]], single[:, :6])
            assert same6[~flag6].all(), "%s / %s: rounds without the centre differ" % (name, label)
            # the per-axis tests include the single evaluations' tests: an unflagged round never rests on a flagged value
            assert not (single_flag & ~flag).any()
            zero_or_nan = ((pts == 0) | np.isnan(pts)).any(axis=1)
            assert flag[zero_or_nan].all() and flag6[zero_or_nan].all()
            if label == "random":
                assert flag.mean() < 1e-3                        # the conditions fail on a measure-zero set


def test_design1_axis_forms_share_the_unchanged_coordinates(libdcsg):
    """Design1 is axis-aligned: an x-tap pair shares every y- and z-difference and its test; the x function forms three
    x-differences per distinct x offset (0, +5, -5) and tests each once."""
    _, generated = _build(scenes.materialize("design1"))
    fx = _function(generated, "void dcsg_primary_sdf_xc(float3 dcsg_v")
    assert "__fmaf_rn" not in fx
    for c, variants in (("x", "0pm"), ("y", "0"), ("z", "0")):
        for v in variants:
            assert fx.count("DCSG_BAD_UNLESS_ABS_GE(dcsg_d%s%s," % (c, v)) == 3
    for v in "pm":
        assert "dcsg_dy%s" % v not in fx and "dcsg_dz%s" % v not in fx


def test_tap_form_gate(libdcsg, monkeypatch):
    """compile_scene keeps the per-axis form for Design1 and the rolled loop, with a note, for the Hilbert design (its
    projection kernel is too large for the instruction cache); DCSG_TAP_FORM forces either."""
    from designcsg_b200 import api
    for form, name, note in (("", "design1", False), ("", "design2", True), ("axis", "design2", False), ("loop", "design1", False)):
        monkeypatch.setenv("DCSG_TAP_FORM", form)
        log = api.compile_scene_offline(scenes.materialize(name)["dir"])
        assert ("keep the rolled tap loop" in log) == note, (form, name, log[:300])


# ---- GPU: the two forms against each other ------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def pairs():
    from designcsg_b200 import api, build
    build.build()
    made = {}

    def get(name):
        if name not in made:
            ctxs = []
            for form in ("loop", "axis"):
                os.environ["DCSG_TAP_FORM"] = form
                try:
                    c = api.Context(0)
                    c.build(scenes.materialize(name)["dir"])
                finally:
                    os.environ.pop("DCSG_TAP_FORM")
                ctxs.append(c)
            made[name] = ctxs
        return made[name]

    yield get
    for ctxs in made.values():
        for c in ctxs:
            c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["design1", "design2", "stress"])
def test_forms_give_the_same_normals(name, pairs):
    from tests.test_gpu_parity import _special_points
    loop, axis = pairs(name)
    assert "keep the rolled tap loop" not in axis.build_log and "exact-only" not in axis.build_log
    pts = np.concatenate([np.random.default_rng(17).uniform(-4.5, 4.5, (100000, 3)).astype(np.float32), _special_points()])
    with np.errstate(all="ignore"):
        a, b = loop.eval_normal(pts), axis.eval_normal(pts)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name,level", [("design1", 7), ("design1", 8), ("design2", 7), ("design2", 8), ("stress", 8)])
def test_forms_give_the_same_projection(name, level, pairs):
    loop, axis = pairs(name)
    box = loop.bbox(10.0)
    assert np.array_equal(axis.bbox(10.0), box)
    meshes, stats = [], []
    for c in (loop, axis):
        c.project_stats()
        meshes.append(c.extract(box, level, gd_steps=50, want_normals=True))
        stats.append(c.project_stats())
    a, b = meshes
    assert np.array_equal(a.triangles(), b.triangles())
    assert np.array_equal(a.vertices().view(np.uint32), b.vertices().view(np.uint32))
    assert np.array_equal(a.normals().view(np.uint32), b.normals().view(np.uint32))
    assert stats[0] == stats[1]
    for m in meshes:
        m.free()



def test_axis_form_flag_is_one_predicate_chain(libdcsg, tmp_path):
    """In the per-axis form (Design1's default) the seven evaluations' 63 square roots and their transform tests chain into
    the one predicate of the fast copy's flag, and nothing stores a flag to shared memory (DESIGN.md 3b)."""
    import re
    import shutil
    from designcsg_b200 import api
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not installed")
    cubin = tmp_path / "scene.cubin"
    api.compile_scene_offline(scenes.materialize("design1")["dir"], str(cubin))
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", "dcsg_k_project", str(cubin)], stdout=subprocess.PIPE, text=True).stdout
    ins = [m.group(1) for m in re.finditer(r"/\*[0-9a-f]{4,5}\*/\s+(.*?);", sass)]
    chain = [t for t in ins if re.match(r"FSETP\.\w+\.OR (P\d), PT, .*, \1\b", t)]
    assert sum("MUFU.RSQ" in t for t in ins) >= 63 + 9
    assert len(chain) >= 63 + 36 and len({re.match(r"FSETP\.\w+\.OR (P\d)", t).group(1) for t in chain}) == 1
    assert sum(t.startswith("@") and "STS" in t for t in ins) == 0
