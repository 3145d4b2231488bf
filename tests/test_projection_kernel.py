"""The projection kernel (dcsg_k_project, scene_kernels.cuh) from arbitrary starting points.

The kernel's loop is more than the reference's descent: persistent warps refill lanes from a cursor, vertices on which the
checked fast copy flags a tap round are handed to an exact phase through a device-wide list of (vertex, steps done), and
three early exits (a fixed point, an all-NaN position, Brent's cycle skipping) stop a vertex before its last step.  Here:

* on the CPU, a numpy restatement of dcsg_project_phase (``model``) walks the plain descent of the oracle step by step,
  with the round's flag from the host harness of the fast copy (tests/model_harness/round_flags.cpp, square roots
  included), and counts what the kernel must execute; it also shows that the pinned inputs reach every exit and every kind of deferral;
* on the GPU, points are written into a carrier mesh and projected through dcsg_project: final positions and normals equal
  the oracle's plain descent (``Oracle.gradient_descent``, no early exit) bit for bit wherever they are numbers, the
  counters of dcsg_project_stats equal the model's, the vertices past the projected count are untouched, and the file
  paths write the same bytes whichever way the rows are formatted;
* dcsg_sqrt_checked over all 2^32 inputs (tests/gpu_harness/sqrt_checked.cu).

NaN sign and payload are not compared: the GPU's arithmetic produces 0x7fffffff, the x86 oracle 0xffc00000 (DESIGN.md 3).
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes
from tests.test_fast_copy_host import _function
from tests.test_tap_forms import AXIS_FUNCTIONS

HERE = os.path.dirname(os.path.abspath(__file__))
# dcsg_sqrt_checked flags exactly the positive normal inputs below this threshold (and every input outside the normal
# positive floats); the sweep below finds it on the device
SQRT_FLAG_BELOW = 2.0 ** -100
STEPS = [0, 1, 2, 3, 7, 50, 64, 129]
MAX_STEPS = max(STEPS)
CANONICAL_NAN = np.uint32(0x7fffffff)


# ---- point sets ---------------------------------------------------------------------------------------------------------

def _special_grid():
    from tests.test_gpu_parity import _special_points
    return _special_points()


_surface_cache = {}


def _surface_points(name):
    """Unique vertices of the scene's uniform lattice mesh before projection (edge midpoints), from the oracle."""
    if name not in _surface_cache:
        orc = _oracle(name)
        box = orc.bbox(10.0)
        soup = orc.get_surface(box, 6, 6, 6).reshape(-1, 3)
        _surface_cache[name] = np.unique(soup, axis=0)
    return _surface_cache[name]


def _points(name, kind):
    """Deterministic starting points of one kind for one scene (float32, [n, 3])."""
    rng = np.random.default_rng(sum(map(ord, name + kind)))
    if kind == "special":
        return _special_grid()
    if kind == "partial":                   # one or two coordinates of the special grid replaced by ordinary values
        p = _special_grid().copy()
        keep = rng.integers(0, 3, len(p))
        for c in range(3):
            two = rng.random(len(p)) < 0.5
            replace = (c != keep) & (two | (c == (keep + 1) % 3))
            p[replace, c] = rng.uniform(-4.5, 4.5, int(replace.sum())).astype(np.float32)
        return p
    if kind == "uniform":
        return rng.uniform(-5.0, 5.0, (2048, 3)).astype(np.float32)
    if kind == "jitter":                    # lattice midpoints moved by a few ulps, and by +-e along one axis
        m = _surface_points(name)
        m = m[rng.permutation(len(m))[:2048]]
        half = len(m) // 2
        ulps = m[:half].copy()
        ulps.view(np.int32)[:] += rng.integers(-4, 5, ulps.shape).astype(np.int32)
        taps = m[half:].copy()
        axis = rng.integers(0, 3, len(taps))
        taps[np.arange(len(taps)), axis] += np.where(rng.random(len(taps)) < 0.5, np.float32(0.005), np.float32(-0.005))
        return np.concatenate([ulps, taps]).astype(np.float32)
    if kind == "outside":                   # synth64: 0.05 .. 0.5 outside the surface along the normal
        m = _surface_points(name)
        m = m[rng.permutation(len(m))[:2048]]
        with np.errstate(all="ignore"):
            n = _oracle(name).eval_normal(m)
        ok = np.isfinite(n).all(axis=1)
        d = rng.uniform(0.05, 0.5, (int(ok.sum()), 1)).astype(np.float32)
        return (m[ok] + n[ok] * d).astype(np.float32)
    raise KeyError(kind)


def _kinds(name):
    return ["special", "partial", "uniform", "jitter"] + (["outside"] if name == "synth64" else [])


# ---- CPU: oracle, flags of the fast copy, trajectories, the model ------------------------------------------------------

_oracles = {}


def _oracle(name):
    from oracle.oracle import Oracle
    if name not in _oracles:
        _oracles[name] = Oracle.for_scene(scenes.materialize(name), "port")
    return _oracles[name]


_flag_libs = {}


def _flag_lib(name):
    """tests/model_harness/round_flags.cpp for this scene: the fast copy's round flag, square roots included."""
    if name in _flag_libs:
        return _flag_libs[name]
    from designcsg_b200 import api
    from oracle.build import cl_to_cpp
    scene = scenes.materialize(name)
    src = api.scene_source(scene["dir"])
    fast = src[src.index("namespace dcsg_fast {\n__device__ float sdf_bank("):]
    parts = [_function(fast, "float dcsg_primary_sdf(float3 dcsg_v, bool& dcsg_inexact_out) {")]
    parts += [_function(fast, "void " + f + "float3 dcsg_v, float dcsg_e, float (&dcsg_out)") for f in AXIS_FUNCTIONS]
    generated = "\n".join(parts)
    text = cl_to_cpp(scene["scene.cl"], scene=True)
    define = "-DSQRT_FLAG_BELOW=%s" % float(SQRT_FLAG_BELOW).hex()
    harness = [os.path.join(HERE, "model_harness", "round_flags.cpp"), os.path.join(HERE, "cpu_emul", "tap_axes.cpp")]
    key = hashlib.sha256((generated + text + define + "".join(open(f).read() for f in harness)).encode())
    out = os.path.join(HERE, "model_harness", "_build", "flags_" + key.hexdigest()[:16])
    lib = os.path.join(out, "libroundflags.so")
    if not os.path.exists(lib):
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "generated.inc"), "w") as f:
            f.write(generated)
        with open(os.path.join(out, "scene.inc"), "w") as f:
            f.write(text)
        cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-fpermissive", define,
               "-I", os.path.join(H.REPO, "oracle"), '-DGENERATED_INC="%s"' % os.path.join(out, "generated.inc"),
               '-DSCENE_INC="%s"' % os.path.join(out, "scene.inc"), harness[0], "-o", lib + ".tmp"]
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert proc.returncode == 0, proc.stdout[-4000:]
        os.replace(lib + ".tmp", lib)
    table = np.zeros(131072, dtype=np.float32)
    raw = open(os.path.join(scene["dir"], "arbitrary_data.hex"), "rb").read()
    table[:len(raw) // 4] = np.frombuffer(raw, dtype="<f4")
    _flag_libs[name] = (ctypes.CDLL(lib), table)
    return _flag_libs[name]


def round_flags(name, pts):
    """Per point: does the fast copy flag the tap round at it (the OR over the seven taps of the single evaluation's flag)?"""
    lib, table = _flag_lib(name)
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    flag = np.empty(len(pts), np.uint8)
    f32p = ctypes.POINTER(ctypes.c_float)
    lib.round_flags(pts.ctypes.data_as(f32p), ctypes.c_size_t(len(pts)), table.ctypes.data_as(f32p),
                    flag.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
    return flag.astype(bool)


def _bits(p):
    """Position bits as the GPU sees them after arithmetic: every NaN canonical."""
    b = np.ascontiguousarray(p, dtype=np.float32).view(np.uint32).copy()
    b[np.isnan(p)] = CANONICAL_NAN
    return b


def _oracle_step(orc, p):
    pad = (-len(p)) % 3
    q = np.concatenate([p, np.zeros((pad, 3), np.float32)]) if pad else p
    return orc.gradient_descent(q.reshape(-1, 3, 3), 1).reshape(-1, 3)[:len(p)]


class Trajectory:
    """pos[k]: the plain descent after k steps (the oracle, one step at a time); bits[k] as the kernel compares them (the
    loaded input for k = 0, canonical NaNs after); flag[k]: the fast copy's round flag at pos[k] (None: exact-only)."""

    def __init__(self, name, pts, steps, flags=True):
        orc = _oracle(name)
        pts = np.ascontiguousarray(pts, dtype=np.float32)
        self.pos = np.empty((steps + 1,) + pts.shape, np.float32)
        self.bits = np.empty((steps + 1,) + pts.shape, np.uint32)
        self.pos[0], self.bits[0] = pts, pts.view(np.uint32)
        live = ~np.isnan(pts).all(axis=1)
        with np.errstate(all="ignore"):
            for k in range(steps):
                nxt = self.pos[k].copy()
                nxt[live] = _oracle_step(orc, self.pos[k][live])
                self.pos[k + 1] = nxt
                self.bits[k + 1] = _bits(nxt)
                # a position the update does not change, or an all-NaN one, stays as it is: stop evaluating it
                live &= ~((self.bits[k + 1] == _bits(self.pos[k])).all(axis=1) | np.isnan(nxt).all(axis=1))
            self.flag = None
            if flags:
                self.flag = np.empty((steps + 1, len(pts)), bool)
                self.flag[0] = round_flags(name, pts)
                for k in range(steps):
                    same = (self.bits[k + 1] == self.bits[k]).all(axis=1)
                    self.flag[k + 1] = self.flag[k]
                    if (~same).any():
                        self.flag[k + 1][~same] = round_flags(name, self.pos[k + 1][~same])


def model(tr, steps, normals, fast=True, detect_cycles=True):
    """dcsg_project_phase (scene_kernels.cuh) restated per vertex, vectorised over the vertices.  Returns (trajectory index
    of the final position per vertex, rounds of phase 1, rounds of the exact phase, events)."""
    n = tr.pos.shape[1]
    rows = np.arange(n)
    allnan = lambda k: np.isnan(tr.pos[k, rows]).all(axis=1)
    k = np.zeros(n, np.int64)
    step = np.zeros(n, np.int64)
    mark_k = np.zeros(n, np.int64)
    mark_step = np.full(n, -1, np.int64)
    exact = np.zeros(n, bool) if fast else np.ones(n, bool)
    r_fast = np.zeros(n, np.int64)
    r_exact = np.zeros(n, np.int64)
    ev = {"deferrals": 0, "deferred at step 0": 0, "deferred mid-run, then moving": 0, "deferred in the normal round": 0,
          "cycle jumps, period >= 2": 0, "fixed-point stops": 0, "all-NaN at load": 0, "all-NaN mid-run": 0,
          "partial-NaN, stepped on": 0}
    moves_after = np.full(n, -1, np.int64)      # position changes after a deferral at step >= 1 (-1: none)
    partial_moving = np.zeros(n, bool)
    at_load = allnan(k)
    ev["all-NaN at load"] = int((at_load & (steps > 0)).sum())
    step[at_load] = steps
    active = (step < steps) | normals
    while active.any():
        a = active.copy()
        r_fast += a & ~exact
        r_exact += a & exact
        flagged = np.zeros(n, bool)
        if fast:
            flagged = a & ~exact & tr.flag[k, rows]
            ev["deferrals"] += int(flagged.sum())
            ev["deferred at step 0"] += int((flagged & (step == 0)).sum())
            ev["deferred in the normal round"] += int((flagged & (step >= steps)).sum())
            moves_after[flagged & (step >= 1) & (step < steps)] = 0
            # the exact phase reloads the vertex: position as written back, step = (entry >> 40) - 1, Brent reset
            exact |= flagged
            step[flagged & allnan(k)] = steps
            mark_step[flagged] = -1
            active[flagged] = (step[flagged] < steps) | normals
        go = a & ~flagged & (step < steps)
        kn = np.minimum(k + 1, steps)
        fixed = (tr.bits[kn, rows] == tr.bits[k, rows]).all(axis=1)
        nan_all = np.isnan(tr.pos[kn, rows]).all(axis=1)
        some_nan = np.isnan(tr.pos[k, rows]).any(axis=1) & ~np.isnan(tr.pos[k, rows]).all(axis=1)
        ev["fixed-point stops"] += int((go & fixed).sum())
        ev["all-NaN mid-run"] += int((go & ~fixed & nan_all).sum())
        partial_moving |= go & ~fixed & some_nan
        moves_after[go & ~fixed & (moves_after >= 0)] += 1
        k = np.where(go, kn, k)
        step = np.where(go, np.where(fixed | nan_all, steps, step + 1), step)
        if detect_cycles:
            d = go & (step < steps)
            hit = d & (mark_step >= 0) & (tr.bits[k, rows] == tr.bits[mark_k, rows]).all(axis=1)
            period = np.where(hit, step - mark_step, 1)
            ev["cycle jumps, period >= 2"] += int((hit & (period >= 2)).sum())
            step = np.where(hit, steps - (steps - step) % period, step)
            mark_step[hit] = -1
            pow2 = d & ~hit & ((step & (step - 1)) == 0)
            mark_k[pow2] = k[pow2]
            mark_step[pow2] = step[pow2]
        done = go & (step == steps)
        active[done] = normals
        active[a & ~flagged & ~go] = False            # the normal round
    ev["deferred mid-run, then moving"] = int((moves_after >= 2).sum())
    ev["partial-NaN, stepped on"] = int(partial_moving.sum())
    return k, int(r_fast.sum()), int(r_exact.sum()), ev


def _same(a, b):
    """Bit for bit wherever a is a number, NaN in the same fields."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    m = ~np.isnan(a)
    return np.array_equal(a.view(np.uint32)[m], b.view(np.uint32)[m])


# ---- CPU tests ------------------------------------------------------------------------------------------------------------

COVERAGE = [("design1", "special"), ("design1", "partial"), ("design1", "uniform"), ("design1", "jitter"),
            ("synth64", "outside"), ("synth64", "jitter"), ("design2", "uniform")]


def test_model_reaches_every_exit_and_every_kind_of_deferral(libdcsg):
    """The model on the pinned inputs: its early exits and its restarts land on the plain descent's final positions, and
    the inputs reach every exit and every kind of deferral the GPU tests rely on (counts printed)."""
    total = {}
    with np.errstate(all="ignore"):
        for name, kind in COVERAGE:
            tr = Trajectory(name, _points(name, kind), MAX_STEPS)
            for steps in (7, 50, 64, MAX_STEPS):
                rows = np.arange(len(tr.pos[0]))
                k, r_fast, r_exact, ev = model(tr, steps, normals=True)
                assert _same(tr.pos[k, rows], tr.pos[steps]), (name, kind, steps)
                # an exact-only build: one phase, nothing deferred, the same final positions
                k, r_fast, r_exact, _ = model(tr, steps, normals=True, fast=False)
                assert r_fast == 0 and _same(tr.pos[k, rows], tr.pos[steps]), (name, kind, steps)
                for key, v in ev.items():
                    total[key] = total.get(key, 0) + v
    print("\nprojection coverage: " + ", ".join("%s %d" % kv for kv in total.items()))
    for key, v in total.items():
        assert v > 0, key


def test_model_all_nan_vertex_takes_one_deferred_normal_round(libdcsg):
    """Hand-checkable: an all-NaN vertex is final at load; with normals its one round flags (NaN taps) and runs again in
    the exact phase, without normals nothing runs."""
    tr = Trajectory("design1", np.full((1, 3), np.nan, np.float32), 7)
    k, r_fast, r_exact, ev = model(tr, 7, normals=True)
    assert (k[0], r_fast, r_exact, ev["deferred in the normal round"]) == (0, 1, 1, 1)
    assert model(tr, 7, normals=False)[1:3] == (0, 0)
    assert model(tr, 7, normals=True, fast=False)[1:3] == (0, 1)


def test_sqrt_harness_compiles_for_sm100a():
    _sqrt_harness()


# ---- dcsg_sqrt_checked, all 2^32 inputs ----------------------------------------------------------------------------------

def _sqrt_harness():
    prelude = open(os.path.join(H.REPO, "designcsg_b200", "csrc", "scene_prelude.cuh")).read()

    def cut(signature):                     # from the start of the signature's line to the matching brace (first occurrence)
        at = prelude.index(signature)
        start = prelude.rindex("\n", 0, at) + 1
        depth, i = 0, prelude.index("{", at)
        while True:
            depth += {"{": 1, "}": -1}.get(prelude[i], 0)
            i += 1
            if depth == 0:
                return prelude[start:i]
    # the predicate form comes first in the prelude (#if DCSG_FLAG_PRED)
    text = "\n".join(cut(s) for s in ("DCSG_DEV void dcsg_flag_init()", "DCSG_DEV bool dcsg_flag_take()",
                                      "DCSG_DEV float dcsg_sqrt_checked(float x)"))
    assert "dcsg_flagp" in text and "rsqrt.approx" in text
    harness = os.path.join(HERE, "gpu_harness", "sqrt_checked.cu")
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-fmad=false", "-prec-sqrt=true", "-O3", "-shared", "-Xcompiler", "-fPIC"]
    key = hashlib.sha256((text + open(harness).read() + " ".join(flags)).encode()).hexdigest()[:16]
    out = os.path.join(HERE, "gpu_harness", "_build", "sqrt_" + key)
    lib = os.path.join(out, "libsqrtchecked.so")
    if not os.path.exists(lib):
        from designcsg_b200.build import CUDA_HOME
        os.makedirs(out, exist_ok=True)
        inc = os.path.join(out, "prelude.inc")
        with open(inc, "w") as f:
            f.write(text)
        cmd = [os.path.join(CUDA_HOME, "bin", "nvcc"), *flags, '-DPRELUDE_INC="%s"' % inc, harness, "-o", lib + ".tmp"]
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert proc.returncode == 0, proc.stdout[-4000:]
        os.replace(lib + ".tmp", lib)
    so = ctypes.CDLL(lib)
    so.sqrt_checked_sweep.argtypes = [ctypes.POINTER(ctypes.c_uint64)]
    so.device_sqrtf.argtypes = [ctypes.POINTER(ctypes.c_float), ctypes.c_uint64, ctypes.POINTER(ctypes.c_float)]
    return so


@pytest.mark.gpu
def test_sqrt_checked_over_every_float():
    so = _sqrt_harness()
    out = (ctypes.c_uint64 * 6)()
    assert so.sqrt_checked_sweep(out) == 0
    wrong, missed, flagged, lo, hi, swept = (int(v) for v in out)
    assert swept == 1 << 32
    assert wrong == 0, "%d unflagged results differ from sqrtf" % wrong
    assert missed == 0, "%d NaN / Inf / zero / negative / denormal inputs not flagged" % missed
    # the flagged positive normals: one interval [2^-126, T)
    assert lo == 0x00800000 and flagged == hi - lo + 1
    t = float(np.uint32(hi + 1).view(np.float32))
    print("\ndcsg_sqrt_checked flags the positive normals below T = %r = 2^%g" % (t, np.log2(t)))
    assert 2.0 ** -101 <= t <= 2.0 ** -100
    assert t == SQRT_FLAG_BELOW                              # the host model's square-root hook uses this threshold
    # device sqrtf (-prec-sqrt=true) against numpy's float32 square root
    x = np.random.default_rng(23).integers(0, 1 << 32, 1 << 24, dtype=np.uint64).astype(np.uint32).view(np.float32)
    y = np.empty_like(x)
    f32p = ctypes.POINTER(ctypes.c_float)
    assert so.device_sqrtf(x.ctypes.data_as(f32p), len(x), y.ctypes.data_as(f32p)) == 0
    with np.errstate(all="ignore"):
        assert _same(y, np.sqrt(x))


# ---- GPU: arbitrary starting points through dcsg_project ------------------------------------------------------------------

VARIANTS = {"design1": ("design1", {}), "design1-loop": ("design1", {"DCSG_TAP_FORM": "loop"}),
            "design1-exact": ("design1", {"DCSG_EXACT_ONLY": "1"}), "design2": ("design2", {}),
            "design2-axis": ("design2", {"DCSG_TAP_FORM": "axis"}), "stress": ("stress", {}), "synth64": ("synth64", {})}
VARIANTS.update({"random%d" % i: ("random%d" % i, {}) for i in range(5)})


@pytest.fixture(scope="module")
def contexts():
    from designcsg_b200 import api, build
    build.build()
    made = {}

    def get(variant):
        if variant not in made:
            name, env = VARIANTS[variant]
            saved = {k: os.environ.get(k) for k in env}
            os.environ.update(env)          # both are read when the scene is built: one context per variant
            try:
                c = api.Context(0)
                c.build(scenes.materialize(name)["dir"])
            finally:
                for k, v in saved.items():
                    if v is None:
                        os.environ.pop(k)
                    else:
                        os.environ[k] = v
            made[variant] = c
        return made[variant]

    yield get
    for c in made.values():
        c.close()


class Carrier:
    """A mesh extracted with defer_projection whose vertex array holds the points to project (through the torch view of
    its device array, as tools/check_multi_gpu.py reads it)."""

    def __init__(self, ctx, need, level=6):
        import torch
        box = ctx.bbox(10.0)
        while True:
            self.mesh = ctx.extract(box, level, defer_projection=True, copy_to_host=False)
            if self.mesh.num_vertices > need or level >= 9:
                break
            self.mesh.free()
            level += 1
        assert self.mesh.num_vertices > need, (need, self.mesh.num_vertices)
        self.ctx = ctx
        self.view = torch.as_tensor(self.mesh.device("vertices"), device="cuda")
        torch.cuda.synchronize()
        self.original = self.view.clone()

    def project(self, pts, steps, normals):
        """dcsg_project on the first len(pts) vertices (a copy of the mesh struct with that count); -> (positions, normals,
        stats).  The vertices past them must come back untouched."""
        import torch
        from designcsg_b200 import api
        n = len(pts)
        self.view.copy_(self.original)
        self.view[:n] = torch.from_numpy(np.ascontiguousarray(pts, np.float32)).cuda()
        torch.cuda.synchronize()
        part = api.Mesh(self.ctx)
        ctypes.memmove(ctypes.byref(part.c), ctypes.byref(self.mesh.c), ctypes.sizeof(api.MeshStruct))
        part.c.num_vertices = n
        self.ctx.project_stats()
        self.ctx.project(part, steps, normals)
        stats = self.ctx.project_stats()                    # synchronises the context's stream
        torch.cuda.synchronize()
        got = self.view[:n].cpu().numpy()
        assert torch.equal(self.view[n:].view(torch.int32), self.original[n:].view(torch.int32))
        nrm = None
        if normals:
            nrm = torch.as_tensor(part.device("normals"), device="cuda")[:n].cpu().numpy()
        part._ctx = None                                    # borrowed storage: the carrier frees it
        return got, nrm, stats

    def free(self):
        self.mesh.free()


def _fast(ctx, env=None):
    """Was the checked fast copy built (DCSG_EXACT_ONLY=1 and the build's own fall-backs make an exact-only module)?"""
    return (env or {}).get("DCSG_EXACT_ONLY") != "1" and "exact-only" not in ctx.build_log


def _check_projection(variant, ctx, name, pts, tr, carrier, fast):
    rows = np.arange(len(pts))
    with np.errstate(all="ignore"):
        for steps in STEPS:
            for normals in (False, True):
                got, nrm, stats = carrier.project(pts, steps, normals)
                want = tr.pos[steps]
                assert _same(got, want), "%s: %d steps%s: %d positions differ from the plain descent" % (
                    variant, steps, " + normals" if normals else "", int((~_eq_rows(got, want)).sum()))
                if normals:
                    assert _same(nrm, _oracle(name).eval_normal(want)), "%s: %d steps: normals differ" % (variant, steps)
                k, r_fast, r_exact, _ = model(tr, steps, normals, fast=fast)
                assert _same(tr.pos[k, rows], want)
                if fast:
                    assert stats == (r_fast + r_exact, r_exact), (variant, steps, normals, stats, (r_fast + r_exact, r_exact))
                else:
                    assert stats == (r_exact, r_exact), (variant, steps, normals, stats, r_exact)


def _eq_rows(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return ((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all(axis=1)


_trajectories = {}


def _trajectory(name, kind, fast):
    key = (name, kind)
    if key not in _trajectories or (fast and _trajectories[key].flag is None):
        _trajectories[key] = Trajectory(name, _points(name, kind), MAX_STEPS, flags=fast)
    return _trajectories[key]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_projection_equals_plain_descent(variant, contexts):
    """Every point set of the scene, steps 0 .. 129 with and without normals: positions and normals bit-exact against the
    oracle's plain descent, dcsg_project_stats equal to the host model's count."""
    name = VARIANTS[variant][0]
    ctx = contexts(variant)
    fast = _fast(ctx, VARIANTS[variant][1])
    assert fast == (variant != "design1-exact")         # synth64 keeps its fast copy (its flag rate is under the limit)
    sets = {kind: _points(name, kind) for kind in _kinds(name)}
    carrier = Carrier(ctx, max(len(p) for p in sets.values()))
    try:
        for kind, pts in sets.items():
            _check_projection("%s/%s" % (variant, kind), ctx, name, pts, _trajectory(name, kind, fast), carrier, fast)
    finally:
        carrier.free()


@pytest.mark.gpu
def test_projected_counts_and_untouched_tail(contexts):
    """Counts around the warp and block sizes, and one larger than the persistent grid holds (148 SMs x 8 blocks x 256
    lanes), so that warps refill from the cursor."""
    ctx = contexts("design1")
    pool = np.concatenate([_special_grid(), _points("design1", "uniform")])
    pool = pool[np.random.default_rng(5).permutation(len(pool))]
    carrier = Carrier(ctx, 600_000, level=9)
    try:
        for n in (1, 31, 32, 33, 255, 256, 257):
            _check_projection("design1/%d" % n, ctx, "design1", pool[:n], Trajectory("design1", pool[:n], MAX_STEPS), carrier,
                              _fast(ctx))
        big = np.random.default_rng(9).uniform(-5.0, 5.0, (600_000, 3)).astype(np.float32)
        big[:len(pool)] = pool
        tr = Trajectory("design1", big, 3)
        rows = np.arange(len(big))
        with np.errstate(all="ignore"):
            for normals in (False, True):
                got, nrm, stats = carrier.project(big, 3, normals)
                assert _same(got, tr.pos[3])
                if normals:
                    assert _same(nrm, _oracle("design1").eval_normal(tr.pos[3]))
                k, r_fast, r_exact, _ = model(tr, 3, normals)
                assert _same(tr.pos[k, rows], tr.pos[3])
                assert stats == (r_fast + r_exact, r_exact)
    finally:
        carrier.free()


# ---- GPU: the file paths on positions with NaN fields ---------------------------------------------------------------------

def _ply_fields(data, ntris):
    head = data.index(b"end_header\n") + len(b"end_header\n")
    v = np.frombuffer(data, dtype="<f8", count=ntris * 9, offset=head)
    return data[:head], v, data[head + ntris * 72:]


def _stl_fields(data, ntris):
    rec = np.frombuffer(data, dtype=np.uint8, offset=84).reshape(ntris, 50)
    return data[:84], rec[:, :48].copy().view("<f4"), rec[:, 48:].tobytes()


def _same_f64(a, b):
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    m = ~np.isnan(a)
    return np.array_equal(a.view(np.uint64)[m], b.view(np.uint64)[m])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["special", "uniform"])
def test_file_paths_agree_on_nan_positions(kind, contexts, tmp_path, monkeypatch):
    """The segments of the pipelined and the plain formatting, and the pipelined and the plain file writers, give the same
    bytes with the rows formatted on the device (DCSG_HOST_EXPAND_PERMILLE=0) and on host threads (1000), on a carrier
    whose vertices are points that project to NaN fields; against the oracle's files the fields are equal where numbers."""
    import torch
    ctx = contexts("design1")
    orc = _oracle("design1")
    steps = 50
    pts = _points("design1", kind)
    carrier = Carrier(ctx, len(pts))
    mesh = carrier.mesh
    nv, nt = mesh.num_vertices, mesh.num_triangles
    fill = torch.from_numpy(np.resize(pts, (nv, 3)).astype(np.float32)).cuda()

    def load():
        carrier.view.copy_(fill)
        torch.cuda.synchronize()

    def segments():
        return [x.tobytes() for x in mesh.format_segments(0)]

    results = []
    try:
        for permille in ("0", "1000"):
            monkeypatch.setenv("DCSG_HOST_EXPAND_PERMILLE", permille)
            load()
            piped = [x.tobytes() for x in mesh.project_and_format_segments(steps, 0)]
            load()
            ctx.project(mesh, steps)
            assert segments() == piped, permille
            load()
            mesh.project_and_write_files(steps, str(tmp_path / "p.stl"), str(tmp_path / "p.ply"))
            load()
            ctx.project(mesh, steps)
            mesh.write_ply(str(tmp_path / "w.ply"))
            mesh.write_stl(str(tmp_path / "w.stl"))
            ply, stl = (tmp_path / "w.ply").read_bytes(), (tmp_path / "w.stl").read_bytes()
            assert (tmp_path / "p.ply").read_bytes() == ply and (tmp_path / "p.stl").read_bytes() == stl, permille
            results.append((piped, ply, stl))
            projected = carrier.view.cpu().numpy()
        assert results[0] == results[1], "device-formatted and host-expanded rows differ"
        # the oracle's descent on the same soup, its writers
        tris = mesh.triangles() if mesh.c.h_triangles else torch.as_tensor(mesh.device("triangles"), device="cuda").cpu().numpy()
        soup = np.resize(pts, (nv, 3)).astype(np.float32)[tris]
        with np.errstate(all="ignore"):
            want = orc.gradient_descent(soup, steps)
        orc.write_ply(str(tmp_path / "o.ply"), want)
        orc.write_stl(str(tmp_path / "o.stl"), want)
        _, ply, stl = results[0]
        oply, ostl = (tmp_path / "o.ply").read_bytes(), (tmp_path / "o.stl").read_bytes()
        gh, gv, gf = _ply_fields(ply, nt)
        oh, ov, of = _ply_fields(oply, nt)
        assert gh == oh and gf == of and _same_f64(gv, ov)
        gh, gr, ga = _stl_fields(stl, nt)
        oh, orr, oa = _stl_fields(ostl, nt)
        assert gh == oh and ga == oa and _same(gr, orr)
        # both formatters widen each float with its sign and payload kept, NaN included (the GPU's 0x7fffffff is written
        # as 0x7fffffffe0000000), and the STL records hold the float bits as they are
        got = projected[tris].reshape(-1, 9)
        assert np.array_equal(gv.view(np.uint64), got.reshape(-1).astype(np.float64).view(np.uint64))
        assert np.array_equal(gr.view(np.uint32).reshape(-1, 12)[:, 3:], got[:, [0, 2, 1, 3, 5, 4, 6, 8, 7]].view(np.uint32))
        if kind == "special":
            assert np.isnan(gv).any() and (gv.view(np.uint64) == 0x7fffffffe0000000).any()
    finally:
        carrier.free()
