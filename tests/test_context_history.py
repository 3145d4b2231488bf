"""Context-history tests: a result must not depend on which calls the context ran before it.

libdcsg keeps state between calls on purpose -- grow-only device buffers, the leaf / alive bitmaps that a sparse extraction's
clean-up pass leaves all-zero, fixed byte offsets in the small scratch buffer, the projection's cursor slots and counters, the
compiled module of the last dcsg_build, the search histogram behind dcsg_plan_slabs, a caller's stream.  A slip there does not
crash: it leaves a stale bit or table, and a result comes out wrong only after some other call came first.

So every operation of a catalogue is reduced to raw bytes and counts, and its REFERENCE is its result as the first call after
dcsg_build on a fresh context.  The references of the small uniform lattices are pinned absolutely as well: the oracle's
surface and the host emulator of the mesher, array for array.  The GPU tests then run the operations in other orders and
circumstances -- seeded sequences on one long-lived context, one mesh object reused across shapes, rebuilds of other scenes on
one context, a caller's stream held back by a spin kernel, two contexts driven from two threads -- and every result must
equal its reference bit for bit.
"""
import collections
import concurrent.futures
import os
import random
import shutil
import tempfile
import threading

import numpy as np
import pytest

from tests import helpers as H
from tests.golden import scenes

SEEDS = (11, 23, 37)
SEQUENCE_LENGTH = 150
SLEEP_CYCLES = 50_000_000           # torch.cuda._sleep: ~25 ms of one spinning thread at B200 clocks

# ---------------------------------------------------------------------------------------------------------------------------
# reduction of results to bytes
# ---------------------------------------------------------------------------------------------------------------------------


def _b(a):
    return np.ascontiguousarray(a).view(np.uint8).tobytes()


def _device(mesh, name):
    """A device array of the mesh, read through torch (on torch's current stream)."""
    import torch
    ptr = {"vertices": mesh.c.d_vertices, "normals": mesh.c.d_normals, "triangles": mesh.c.d_triangles}[name]
    rows = mesh.num_triangles if name == "triangles" else mesh.num_vertices
    if not ptr or rows == 0:
        return None
    return torch.as_tensor(mesh.device(name), device="cuda").clone()


def _mesh_result(mesh, device=False):
    """Counts, NULL-ness of the optional arrays, and every array the mesh holds (host copies, or the device arrays)."""
    c = mesh.c
    out = {"counts": (mesh.num_vertices, mesh.num_triangles, mesh.num_cells, int(c.lattice_samples), mesh.owned_vertices,
                      mesh.halo_vertices),
           "has": tuple(bool(p) for p in (c.d_normals, c.d_vertex_keys, c.h_vertices, c.h_normals, c.h_vertex_keys))}
    if device:
        for name in ("vertices", "normals", "triangles"):
            t = _device(mesh, name)
            out["d_" + name] = None if t is None else _b(t.cpu().numpy())
        return out
    if c.h_vertices:
        out["vertices"] = _b(mesh.vertices())
        out["triangles"] = _b(mesh.triangles())
        out["cell_ids"] = _b(mesh.cell_ids())
        out["cell_masks"] = _b(mesh.cell_masks())
    if c.h_normals:
        out["normals"] = _b(mesh.normals())
    if c.h_vertex_keys:
        out["vertex_keys"] = _b(mesh.vertex_keys())
    return out


def _report(rep):
    return {k: (_b(v) if isinstance(v, np.ndarray) else v) for k, v in rep.items()}


# ---------------------------------------------------------------------------------------------------------------------------
# the catalogue
# ---------------------------------------------------------------------------------------------------------------------------


class Env:
    """What an operation needs besides the context: the scene's box (from its fresh bbox(10.0)), a directory for files, a
    hook run before the library calls that care about stream order, and the meshes of operations that are still open."""

    def __init__(self, boxes, tmp):
        self.boxes, self.tmp, self.held = boxes, tmp, {}
        self.pre = lambda: None
        self.on_torch_stream = False        # the context launches on a torch stream (set_stream)

    def box(self, scene):
        return self.boxes[scene]


Op = collections.namedtuple("Op", "scene kind level slab begin end")
# kind: sparse / dense / adaptive (an extraction of that kind comes first), lattice, bbox, eval, preview, refused, other.
# begin / end: a two-part operation -- `begin` extracts and leaves the mesh open, `end` finishes it, possibly many calls later.
# An operation with end = None is one call sequence; its result is begin's.

CATALOGUE = {}


def op(key, scene, kind, level=0, slab=False, end=None):
    def deco(fn):
        CATALOGUE[key] = Op(scene, kind, level, slab, fn, end)
        return fn
    return deco


def _extract_op(key, scene, level, kind="sparse", slab=(0, 0), **kw):
    def fn(ctx, e):
        e.pre()
        m = ctx.extract(e.box(scene), level, slab=slab, dense=(kind == "dense"), **kw)
        r = _mesh_result(m)
        m.free()
        return r
    ukind = "dense" if kw.get("no_cull") else kind
    CATALOGUE[key] = Op(scene, ukind, level, slab != (0, 0), fn, None)


def _adaptive_op(key, scene, lo, hi, grid, retopologize=False, slab=(0, 0), gd_steps=0):
    def fn(ctx, e):
        m = ctx.extract(e.box(scene), grid, min_level=lo, max_level=hi, retopologize=retopologize, slab=slab, gd_steps=gd_steps)
        r = _mesh_result(m)
        m.free()
        return r
    CATALOGUE[key] = Op(scene, "adaptive", grid, slab != (0, 0), fn, None)


D1 = "design1"
for L in (3, 4, 5, 7, 9):
    _extract_op("d1/u%d" % L, D1, L)
for L in (3, 4, 5, 7):
    _extract_op("d1/u%d-dense" % L, D1, L, kind="dense")
_extract_op("d1/u5-nocull", D1, 5, no_cull=True)
_extract_op("d1/u6-gd5-normals", D1, 6, gd_steps=5, want_normals=True)
_extract_op("d1/u6-gd5", D1, 6, gd_steps=5)
_extract_op("d1/u6-normals", D1, 6, want_normals=True)
_extract_op("d1/u6-dense-gd5-normals", D1, 6, kind="dense", gd_steps=5, want_normals=True)
_extract_op("d1/u5-slab-first", D1, 5, slab=(0, 1), gd_steps=2)
_extract_op("d1/u5-slab-last", D1, 5, slab=(31, 32), gd_steps=2)
_extract_op("d1/u5-slab-3-11", D1, 5, slab=(3, 11), gd_steps=2, want_normals=True)
_extract_op("d1/u7-slab-5-67", D1, 7, slab=(5, 67))
_extract_op("d1/u7-slab-last", D1, 7, slab=(127, 128))
_extract_op("d1/u9-slab-200-301", D1, 9, slab=(200, 301))
_adaptive_op("d1/a356", D1, 3, 5, 6)
_adaptive_op("d1/a356-retopo", D1, 3, 5, 6, retopologize=True, gd_steps=3)
_adaptive_op("d1/a467", D1, 4, 6, 7)
_adaptive_op("d1/a467-retopo", D1, 4, 6, 7, retopologize=True)
_adaptive_op("d1/a356-slab", D1, 3, 5, 6, slab=(16, 48))


def _bbox_plan(scene, diameter):
    def fn(ctx, e):
        box = ctx.bbox(diameter)
        return {"box": _b(box), "plan": tuple(ctx.plan_slabs(box, 7, 4)), "plan9": tuple(ctx.plan_slabs(box, 9, 3, granularity=16))}
    return fn


def _plan_only(scene):
    def fn(ctx, e):     # before any search of this scene: equal slabs
        return {"plan": tuple(ctx.plan_slabs(e.box(scene), 7, 4))}
    return fn


def _points(n=20000, seed=5):
    rng = np.random.default_rng(seed)
    pts = rng.uniform(-4.5, 4.5, (n, 3)).astype(np.float32)
    pts[:8] = [[0, 0, 0], [-0.0, 0, 0], [np.nan, 0, 0], [np.inf, 1, 1], [1e-40, 0, 0], [1e37, 0, 0], [0.5, 0.5, 0.5], [3, -2, 1]]
    return pts


def _eval_host(ctx, e):
    pts = _points()
    with np.errstate(all="ignore"):
        return {"sdf": _b(ctx.eval_sdf(pts)), "normal": _b(ctx.eval_normal(pts[:5000]))}


def _eval_device(ctx, e):
    """dcsg_eval_*_device on points torch wrote on its current stream (the context's stream after set_stream)."""
    import torch
    pts = _points(30000, 9)
    src = torch.from_numpy(pts).cuda()
    torch.cuda.current_stream().synchronize()
    x = torch.full((len(pts), 3), float("nan"), device="cuda")
    d = torch.full((len(pts),), float("nan"), device="cuda")
    nrm = torch.full((len(pts), 3), float("nan"), device="cuda")
    e.pre()
    x.copy_(src)
    if not e.on_torch_stream:
        torch.cuda.current_stream().synchronize()        # the context's own stream does not wait for torch's
    ctx._check(ctx.lib.dcsg_eval_sdf_device(ctx.h, x.data_ptr(), len(pts), d.data_ptr()))
    e.pre()
    ctx._check(ctx.lib.dcsg_eval_normal_device(ctx.h, x.data_ptr(), len(pts), nrm.data_ptr()))
    if not e.on_torch_stream:
        torch.cuda.synchronize()                         # the calls only queue kernels on the context's own stream
    return {"sdf": _b(d.cpu().numpy()), "normal": _b(nrm.cpu().numpy())}


def _preview(ctx, e):
    return {"rgb": _b(ctx.preview(*H.PREVIEW_CAMERAS[1]))}


def _sample_lattice(scene, L, z0, z1):
    def fn(ctx, e):
        return {"values": _b(ctx.sample_lattice(e.box(scene), L, z0, z1))}
    return fn


for scene, tag in ((D1, "d1"), ("design2", "d2"), ("stress", "st"), ("synth64", "s64"), ("logo", "logo")):
    CATALOGUE[tag + "/bbox10"] = Op(scene, "bbox", 0, False, _bbox_plan(scene, 10.0), None)
    CATALOGUE[tag + "/plan-only"] = Op(scene, "other", 0, False, _plan_only(scene), None)
    CATALOGUE[tag + "/eval"] = Op(scene, "eval", 0, False, _eval_host, None)
CATALOGUE["d1/bbox8"] = Op(D1, "bbox", 0, False, _bbox_plan(D1, 8.0), None)
CATALOGUE["d1/eval-device"] = Op(D1, "eval", 0, False, _eval_device, None)
CATALOGUE["d1/preview"] = Op(D1, "preview", 0, False, _preview, None)
CATALOGUE["d1/lattice-all"] = Op(D1, "lattice", 5, False, _sample_lattice(D1, 5, 0, 0), None)
CATALOGUE["d1/lattice-3-10"] = Op(D1, "lattice", 6, False, _sample_lattice(D1, 6, 3, 10), None)
CATALOGUE["d1/lattice-top"] = Op(D1, "lattice", 5, False, _sample_lattice(D1, 5, 32, 33), None)


@op("d1/weld", D1, "adaptive", 6)
def _weld(ctx, e):
    e.pre()
    m = ctx.extract(e.box(D1), 6, min_level=3, max_level=5, gd_steps=2, want_normals=True)
    e.pre()
    m.weld()
    r = _mesh_result(m)
    m.free()
    return r


@op("d1/orient", D1, "sparse", 6)
def _orient(ctx, e):
    e.pre()
    m = ctx.extract(e.box(D1), 6, gd_steps=3)
    e.pre()
    m.orient()
    r = _mesh_result(m)
    r["stl"] = _b(m.format_stl())
    m.free()
    return r


@op("d1/inspect", D1, "sparse", 6)
def _inspect(ctx, e):
    e.pre()
    m = ctx.extract(e.box(D1), 6, gd_steps=4)
    e.pre()
    r = _report(m.inspect(components=True))
    m.free()
    return r


@op("d1/deviation", D1, "adaptive", 6)
def _deviation(ctx, e):
    m = ctx.extract(e.box(D1), 6, min_level=4, max_level=6, gd_steps=3, copy_to_host=False)
    r = _report(m.deviation(4, 0.01, per_triangle=True))
    m.free()
    return r


@op("d1/format", D1, "sparse", 5)
def _format(ctx, e):
    m = ctx.extract(e.box(D1), 5, gd_steps=3, copy_to_host=False)
    r = {"ply": _b(m.format_ply()), "stl": _b(m.format_stl())}
    m.free()
    return r


@op("d1/ply-indexed", D1, "sparse", 5)
def _ply_indexed(ctx, e):
    m = ctx.extract(e.box(D1), 5, gd_steps=2, want_normals=True, copy_to_host=False)
    path = os.path.join(e.tmp, "indexed-%d.ply" % threading.get_ident())
    m.write_ply_indexed(path, normals=True)
    m.free()
    with open(path, "rb") as f:
        return {"file": f.read()}


def _begin_deferred(key, scene, level, **kw):
    def fn(ctx, e):
        e.pre()
        e.held[key] = ctx.extract(e.box(scene), level, defer_projection=True, copy_to_host=False, **kw)
        return {}
    return fn


def _end_segments(key):
    def fn(ctx, e):
        m = e.held.pop(key)
        r = {"segments": [_b(a) for a in m.project_and_format_segments(5, 17)]}
        r.update(_mesh_result(m, device=True))
        m.free()
        return r
    return fn


def _end_project(key):
    def fn(ctx, e):
        import torch
        m = e.held.pop(key)
        e.pre()
        ctx.project(m, 5, want_normals=True)
        if e.on_torch_stream:
            r = _mesh_result(m, device=True)     # through torch on the context's stream, no device synchronise
            r["stats"] = ctx.project_stats()
        else:
            torch.cuda.synchronize()             # dcsg_project only queues the projection on the context's own stream
            stats = ctx.project_stats()
            r = _mesh_result(m, device=True)
            r["stats"] = stats
        torch.cuda.current_stream().synchronize()
        m.free()
        return r
    return fn


CATALOGUE["d1/segments-u6"] = Op(D1, "sparse", 6, False, _begin_deferred("d1/segments-u6", D1, 6), _end_segments("d1/segments-u6"))
CATALOGUE["d1/segments-u7-slab"] = Op(D1, "sparse", 7, True, _begin_deferred("d1/segments-u7-slab", D1, 7, slab=(40, 101)),
                                      _end_segments("d1/segments-u7-slab"))
CATALOGUE["d1/segments-a356"] = Op(D1, "adaptive", 6, False, _begin_deferred("d1/segments-a356", D1, 6, min_level=3, max_level=5,
                                                                             retopologize=True), _end_segments("d1/segments-a356"))
CATALOGUE["d1/project-u6"] = Op(D1, "sparse", 6, False, _begin_deferred("d1/project-u6", D1, 6), _end_project("d1/project-u6"))

FAR_BOX = np.array([8.0, 8.0, 8.0, 2.0, 2.0, 2.0], dtype=np.float32)      # Design1 lives inside +-3.4


@op("d1/project-empty", D1, "project0", 6)
def _project_empty(ctx, e):
    m = ctx.extract(FAR_BOX, 6, defer_projection=True, want_normals=True)
    ctx.project(m, 5, want_normals=True)
    r = _mesh_result(m)
    r["segments"] = [_b(a) for a in m.project_and_format_segments(5, 0)]
    m.free()
    return r


def _refused(fn):
    def run(ctx, e):
        from designcsg_b200 import api
        try:
            fn(ctx, e)
        except api.DcsgError as err:
            return {"code": err.code}
        return {"code": 0}
    return run


CATALOGUE["d1/refuse-slab"] = Op(D1, "refused", 0, False, _refused(lambda ctx, e: ctx.extract(e.box(D1), 5, slab=(20, 7))), None)
CATALOGUE["d1/refuse-lattice"] = Op(D1, "refused", 0, False, _refused(
    lambda ctx, e: ctx.extract(np.array([0.1, 0.0, 0.0, 6.7, 6.7, 6.7], dtype=np.float32), 7)), None)


def _inspect_bad_id(ctx, e):
    import torch
    m = ctx.extract(e.box(D1), 4, copy_to_host=False)
    t = torch.as_tensor(m.device("triangles"), device="cuda")
    t[len(t) // 2, 1] = m.num_vertices                 # one id >= V
    torch.cuda.synchronize()
    try:
        m.inspect(components=True)
    finally:
        m.free()


CATALOGUE["d1/refuse-inspect"] = Op(D1, "refused", 0, False, _refused(_inspect_bad_id), None)


@op("d1/chain", D1, "sparse", 6)
def _chain_d1(ctx, e):
    return _chain(ctx, e, D1)


@op("d2/chain", "design2", "sparse", 6)
def _chain_d2(ctx, e):
    return _chain(ctx, e, "design2")


def _chain(ctx, e, scene):
    """extract -> project -> inspect -> format -> preview: what one thread of a GUI does per export."""
    m = ctx.extract(e.box(scene), 6, defer_projection=True, copy_to_host=False)
    ctx.project(m, 4, want_normals=True)
    r = {"inspect": _report(m.inspect()), "stl": _b(m.format_stl()), "ply": _b(m.format_ply())}
    m.free()
    r.update(_preview(ctx, e))
    return r


def _synth_swap(ctx, e):
    """set_arbitrary_data with moved primitives, then the scene's own table again: both results, in one operation."""
    raw = open(os.path.join(scenes.materialize("synth64")["dir"], "arbitrary_data.hex"), "rb").read()
    original = np.zeros(131072, dtype=np.float32)
    original[:len(raw) // 4] = np.frombuffer(raw, dtype="<f4")
    swapped = _swapped_table(original)
    pts = _points(8000, 3)
    r = {}
    for tag, table in (("swapped", swapped), ("restored", original)):
        ctx.set_arbitrary_data(table)
        m = ctx.extract(e.box("synth64"), 5, gd_steps=2)
        r[tag] = (_b(ctx.eval_sdf(pts)), _mesh_result(m))
        m.free()
    return r


def _swapped_table(original):
    used = int(np.flatnonzero(original).max()) + 1
    out = original.copy()
    out[:used] *= np.random.default_rng(7).uniform(0.8, 1.2, used).astype(np.float32)
    return out


CATALOGUE["s64/swap"] = Op("synth64", "sparse", 5, False, _synth_swap, None)
for scene, tag in (("design2", "d2"), ("stress", "st"), ("synth64", "s64")):
    for L in (3, 4):
        _extract_op("%s/u%d" % (tag, L), scene, L)
        _extract_op("%s/u%d-dense" % (tag, L), scene, L, kind="dense")
    _extract_op(tag + "/u6-gd3-normals", scene, 6, gd_steps=3, want_normals=True)
_extract_op("st/u6-slab-odd", "stress", 6, slab=(13, 50), gd_steps=2)
_adaptive_op("d2/a356", "design2", 3, 5, 6)
_extract_op("logo/u5-gd3", "logo", 5, gd_steps=3, want_normals=True)
_adaptive_op("logo/a345", "logo", 3, 4, 5)
for scene, tag in ((D1, "d1"), ("logo", "logo"), ("synth64", "s64")):
    CATALOGUE[tag + "/preview"] = Op(scene, "preview", 0, False, _preview, None)

# after each build of the rebuild test: the plan before any search first, then these
REBUILD_OPS = {
    D1: ["d1/plan-only", "d1/bbox10", "d1/u5-slab-3-11", "d1/u6-gd5-normals", "d1/a356-retopo", "d1/eval", "d1/preview", "d1/project-u6"],
    "design2": ["d2/plan-only", "d2/bbox10", "d2/u4", "d2/u6-gd3-normals", "d2/a356", "d2/eval"],
    "logo": ["logo/plan-only", "logo/bbox10", "logo/u5-gd3", "logo/a345", "logo/eval", "logo/preview"],
    "synth64": ["s64/plan-only", "s64/bbox10", "s64/u4", "s64/u6-gd3-normals", "s64/eval", "s64/preview", "s64/swap"],
}

# ---------------------------------------------------------------------------------------------------------------------------
# seeded call sequences on Design1
# ---------------------------------------------------------------------------------------------------------------------------

# transition classes a sequence must contain, with the motif that guarantees each.  The first one opens every sequence: on a
# fresh context u4 leaves the bitmaps clean, and u9 then outgrows them (the clean bitmaps are reallocated and cleared); in the
# others the buffers of an earlier, larger extraction are reused.
GROWTH = "sparse>larger sparse (buffers grow)"
MOTIFS = {
    GROWTH: ["d1/u4", "d1/u9"],
    "sparse>sparse (buffers kept)": ["d1/u7", "d1/u5"],
    "large>small>large": ["d1/u9", "d1/u4", "d1/u9-slab-200-301"],
    "sparse>dense>sparse": ["d1/u5", "d1/u5-dense", "d1/u7"],
    "slab>whole": ["d1/u5-slab-last", "d1/u5"],
    "whole>slab": ["d1/u7", "d1/u7-slab-5-67"],
    "adaptive>uniform": ["d1/a467", "d1/u4"],
    "lattice between sparse": ["d1/u5", "d1/lattice-3-10", "d1/u5"],
    "bbox between sparse": ["d1/u7", "d1/bbox8", "d1/u3"],
    "project of 0 vertices": ["d1/project-empty"],
    "held across extraction": ["d1/segments-u6", "d1/u9", "/end d1/segments-u6", "d1/project-u6", "d1/a356", "/end d1/project-u6"],
    "refused slab>good": ["d1/refuse-slab", "d1/u5"],
    "refused lattice>good": ["d1/refuse-lattice", "d1/u7-slab-last"],
    "refused inspect>good": ["d1/refuse-inspect", "d1/inspect"],
}


def d1_keys():
    return sorted(k for k, o in CATALOGUE.items() if o.scene == D1 and k not in ("d1/plan-only", "d1/chain"))


def _weight(key):
    o = CATALOGUE[key]
    if o.level >= 9:
        return 2
    return {"sparse": 6, "dense": 3, "adaptive": 3}.get(o.kind, 2)


def make_sequence(seed, n=SEQUENCE_LENGTH):
    """Steps for one context: [(key, part)], part 'all' (the whole operation), 'begin' or 'end'.  Every motif is placed once at
    a seeded position; the rest is drawn with weights; a two-part operation ends 1 to 6 steps after it began."""
    rng = random.Random(seed)
    keys = d1_keys()
    weights = [_weight(k) for k in keys]
    blocks, first = [], None
    for name in sorted(MOTIFS):
        block = []
        for k in MOTIFS[name]:
            if k.startswith("/end "):
                block.append((k[5:], "end"))
            else:
                block.append((k, "begin" if CATALOGUE[k].end else "all"))
        if name == GROWTH:
            first = block
        else:
            blocks.append(block)
    motif_steps = len(first)
    motif_steps += sum(len(b) for b in blocks)
    filler = []
    while len(filler) + motif_steps < n:
        filler.append([(rng.choices(keys, weights)[0], None)])
    units = blocks + filler
    rng.shuffle(units)
    units.insert(0, first)
    steps, open_ends = [], []               # open_ends: [steps to go, key]
    for unit in units:
        for key, part in unit:
            if part is None:
                if not CATALOGUE[key].end:
                    part = "all"
                elif key in [k for _, k in open_ends]:
                    continue
                else:
                    part = "begin"
                    open_ends.append([rng.randint(1, 6), key])
            elif part == "begin" and any(k == key for _, k in open_ends):
                closing = [x for x in open_ends if x[1] == key][0]
                open_ends.remove(closing)
                steps.append((key, "end"))
            steps.append((key, part))
        for x in list(open_ends):
            x[0] -= 1
            if x[0] <= 0:
                open_ends.remove(x)
                steps.append((x[1], "end"))
    steps.extend((k, "end") for _, k in open_ends)
    return _balance(steps)


def _balance(steps):
    """A motif's own 'end' closes its own 'begin'; drop an 'end' whose operation is not open (and close what is left open)."""
    out, open_keys = [], set()
    for key, part in steps:
        if part == "begin":
            if key in open_keys:
                out.append((key, "end"))
            open_keys.add(key)
        elif part == "end":
            if key not in open_keys:
                continue
            open_keys.discard(key)
        out.append((key, part))
    out.extend((k, "end") for k in sorted(open_keys))
    return out


def _extraction(step):
    key, part = step
    o = CATALOGUE[key]
    if part == "end" or o.kind not in ("sparse", "dense", "adaptive"):
        return None
    return o


def transitions(steps):
    """How often each transition class occurs in a sequence."""
    found = collections.Counter()
    ext = [(i, _extraction(s)) for i, s in enumerate(steps) if _extraction(s)]
    for n, ((i, a), (j, b)) in enumerate(zip(ext, ext[1:])):
        if a.kind == "sparse" and b.kind == "sparse":
            # b's bitmaps fit in what an earlier whole-lattice extraction of at least b's level allocated
            fits = any(not o.slab and o.level >= b.level for _, o in ext[:n + 1])
            found["sparse>sparse (buffers kept)" if fits else GROWTH] += 1
        if a.slab and not b.slab and b.kind != "adaptive":
            found["slab>whole"] += 1
        if not a.slab and b.slab and a.kind != "adaptive":
            found["whole>slab"] += 1
        if a.kind == "adaptive" and b.kind != "adaptive":
            found["adaptive>uniform"] += 1
        if a.kind == "sparse" and b.kind == "sparse":
            between = {CATALOGUE[k].kind for k, _ in steps[i + 1:j]}
            if "lattice" in between:
                found["lattice between sparse"] += 1
            if "bbox" in between:
                found["bbox between sparse"] += 1
    for (_, a), (_, b), (_, c) in zip(ext, ext[1:], ext[2:]):
        if a.level >= 9 and b.kind == "sparse" and b.level <= 5 and c.level >= 9:
            found["large>small>large"] += 1
        if a.kind == "sparse" and b.kind == "dense" and c.kind == "sparse":
            found["sparse>dense>sparse"] += 1
    began = {}
    for i, (key, part) in enumerate(steps):
        if part == "begin":
            began[key] = i
        elif part == "end" and any(_extraction(s) for s in steps[began[key] + 1:i]):
            found["held across extraction"] += 1
        if CATALOGUE[key].kind == "project0":
            found["project of 0 vertices"] += 1
    for (ka, _), (kb, _) in zip(steps, steps[1:]):
        if CATALOGUE[ka].kind == "refused" and CATALOGUE[kb].kind != "refused":
            found["refused %s>good" % ka.split("-")[1]] += 1
    return found


def test_sequences_are_deterministic_and_cover_every_transition():
    for seed in SEEDS:
        steps = make_sequence(seed)
        assert steps == make_sequence(seed)
        assert abs(len(steps) - SEQUENCE_LENGTH) <= 25
        open_keys = set()
        for key, part in steps:                 # two-part operations are well nested per key
            assert key in CATALOGUE and part in ("all", "begin", "end")
            assert (part == "all") == (CATALOGUE[key].end is None)
            if part == "begin":
                assert key not in open_keys
                open_keys.add(key)
            elif part == "end":
                open_keys.remove(key)
        assert not open_keys
        found = transitions(steps)
        missing = sorted(set(MOTIFS) - set(found))
        assert not missing, "seed %d lacks %s" % (seed, missing)
        print("seed %d: %d steps, %s" % (seed, len(steps), dict(sorted(found.items()))))
    assert make_sequence(SEEDS[0]) != make_sequence(SEEDS[1])


def test_catalogue_covers_the_configurations():
    d1 = {k: CATALOGUE[k] for k in d1_keys()}
    assert {o.level for o in d1.values() if o.kind == "sparse" and not o.slab} >= {3, 4, 5, 6, 7, 9}
    assert {o.kind for o in d1.values()} >= {"sparse", "dense", "adaptive", "lattice", "bbox", "eval", "preview", "refused", "project0"}
    for name in scenes.names():
        assert any(o.scene == name for o in CATALOGUE.values())
    for ops in REBUILD_OPS.values():
        assert all(k in CATALOGUE for k in ops)


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: references on fresh contexts
# ---------------------------------------------------------------------------------------------------------------------------


def run_op(ctx, env, key):
    """Both parts of an operation back to back; the projection counters it left are part of its result."""
    o = CATALOGUE[key]
    r = o.begin(ctx, env)
    if o.end:
        r = o.end(ctx, env)
    return r, ctx.project_stats()


def run_step(ctx, env, key, part):
    o = CATALOGUE[key]
    fn = {"all": o.begin, "begin": o.begin, "end": o.end}[part]
    r = fn(ctx, env)
    return r, ctx.project_stats()


def _fresh(key, boxes, tmp):
    from designcsg_b200 import api
    ctx = api.Context(0)
    try:
        ctx.build(scenes.materialize(CATALOGUE[key].scene)["dir"])
        return run_op(ctx, Env(boxes, tmp), key)
    finally:
        ctx.close()


def _parallel(fn, items):
    workers = max(2, min(16, os.cpu_count() or 2))
    with concurrent.futures.ThreadPoolExecutor(workers) as pool:       # NVRTC compiles dominate; ctypes releases the GIL
        return dict(zip(items, pool.map(fn, items)))


@pytest.fixture(scope="module")
def refs():
    """Every catalogue operation as the first call after dcsg_build on a fresh context of its scene."""
    from designcsg_b200 import build
    build.build()
    for name in set(o.scene for o in CATALOGUE.values()):
        scenes.materialize(name)
    tmp = tempfile.mkdtemp(prefix="dcsg_history_")
    first = _parallel(lambda k: _fresh(k, {}, tmp), sorted(k for k in CATALOGUE if k.endswith("/bbox10")))
    boxes = {CATALOGUE[k].scene: np.frombuffer(r[0]["box"], dtype=np.float32).copy() for k, r in first.items()}
    rest = _parallel(lambda k: _fresh(k, boxes, tmp), sorted(k for k in CATALOGUE if k not in first))
    rest.update(first)
    yield rest, boxes, tmp
    shutil.rmtree(tmp, ignore_errors=True)


def _diff(got, want):
    """Names of the fields that differ (None when equal)."""
    if got == want:
        return None
    r, s = got[0], want[0]
    fields = sorted(set(r) | set(s))
    bad = [f for f in fields if r.get(f) != s.get(f)]
    if got[1] != want[1]:
        bad.append("project_stats %s != %s" % (got[1], want[1]))
    return bad


@pytest.mark.gpu
@pytest.mark.parametrize("name", scenes.names())
@pytest.mark.parametrize("level", [3, 4])
def test_small_lattices_are_pinned_to_the_oracle_and_the_emulator(refs, name, level):
    """Levels 3 and 4, where dcsg_k_descend_top runs the whole descent alone: the fresh references equal the oracle's surface
    as a canonical soup, the host emulator array for array, and the dense pass."""
    from oracle.oracle import Oracle
    ref, boxes, _ = refs
    tag = {"design1": "d1", "design2": "d2", "stress": "st", "synth64": "s64"}[name]
    box = boxes[name]
    orc = Oracle.for_scene(scenes.materialize(name), "port")
    sparse, dense = ref["%s/u%d" % (tag, level)][0], ref["%s/u%d-dense" % (tag, level)][0]
    for field in ("vertices", "triangles", "vertex_keys", "cell_ids", "cell_masks"):
        assert sparse[field] == dense[field], field
    assert sparse["counts"][:3] == dense["counts"][:3] and dense["counts"][3] == ((1 << level) + 1) ** 3 and sparse["counts"][3] > 0
    vertices = np.frombuffer(sparse["vertices"], np.float32).reshape(-1, 3)
    triangles = np.frombuffer(sparse["triangles"], np.uint32).reshape(-1, 3)
    want = orc.get_surface(box, level, level, level)
    assert len(triangles) == len(want) > 0
    assert np.array_equal(H.canon_soup(H.soup_from_indexed(vertices, triangles)), H.canon_soup(want))
    emu = H.emul_extract(orc.lattice_sdf(box, 1 << level), box, level)
    for field in ("cell_ids", "cell_masks", "triangles", "vertex_keys", "vertices"):
        assert sparse[field] == _b(emu[field]), field


@pytest.mark.gpu
def test_references_are_what_the_catalogue_says(refs):
    """The fresh references themselves: refusals have their codes, the empty projection is empty, the normals exist only where
    asked for, the plan before any search is the equal split."""
    ref, boxes, _ = refs
    assert ref["d1/refuse-slab"][0] == {"code": -2}
    assert ref["d1/refuse-lattice"][0] == {"code": -6}
    assert ref["d1/refuse-inspect"][0] == {"code": -2}
    assert ref["d1/project-empty"][0]["counts"][:3] == (0, 0, 0) and ref["d1/project-empty"][1] == (0, 0)
    assert ref["d1/plan-only"][0]["plan"] == (0, 32, 64, 96, 128)
    assert ref["d1/u6-gd5"][0]["has"][0] is False and ref["d1/u6-gd5-normals"][0]["has"][0] is True
    assert ref["d1/u6-gd5-normals"][1][0] > 0
    assert ref["d1/u6-dense-gd5-normals"][0]["vertices"] == ref["d1/u6-gd5-normals"][0]["vertices"]
    assert ref["d1/u6-dense-gd5-normals"][0]["normals"] == ref["d1/u6-gd5-normals"][0]["normals"]
    swap = ref["s64/swap"][0]
    assert swap["swapped"][0] != swap["restored"][0] and swap["swapped"][1] != swap["restored"][1]


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_seeded_sequence_on_one_context(refs, seed):
    from designcsg_b200 import api
    ref, boxes, tmp = refs
    steps = make_sequence(seed)
    ctx = api.Context(0)
    ctx.build(scenes.materialize(D1)["dir"])
    env = Env(boxes, tmp)
    env.on_torch_stream = False
    pending = {}
    try:
        for i, (key, part) in enumerate(steps):
            got = run_step(ctx, env, key, part)
            if part == "begin":
                pending[key] = got[1]
                continue
            if part == "end":           # the begin's counters belong to the operation too (they are zero: it only extracts)
                assert pending.pop(key) == (0, 0)
            bad = _diff(got, ref[key])
            assert bad is None, "seed %d, step %d (%s %s): %s differ; before it: %s" % (
                seed, i, key, part, bad, steps[max(0, i - 8):i])
    finally:
        for m in env.held.values():
            m.free()
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: one mesh object across shapes
# ---------------------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_mesh_reuse_across_shapes(refs):
    """extract(..., mesh=m) into one dcsg_mesh whose previous contents had another shape: every result equals a fresh mesh's,
    host copies, normals (NULL when not asked for), the oriented state and the STL winding included."""
    from designcsg_b200 import api
    _, boxes, _ = refs
    box = boxes[D1]
    ctx = api.Context(0)
    ctx.build(scenes.materialize(D1)["dir"])
    steps = [
        (dict(grid_level=9, gd_steps=2, want_normals=True), None),
        (dict(grid_level=6, min_level=3, max_level=5, retopologize=True), None),
        (dict(grid_level=7, gd_steps=3, want_normals=True), None),
        (dict(grid_level=7, gd_steps=3), None),
        (dict(grid_level=6, min_level=3, max_level=5, gd_steps=2, want_normals=True), "weld"),
        (dict(grid_level=6, gd_steps=2), "orient"),
        (dict(grid_level=6, min_level=4, max_level=6, gd_steps=2), None),
        (dict(grid_level=6, min_level=4, max_level=6, gd_steps=2), "orient"),
        (dict(grid_level=5, gd_steps=2, slab=(4, 20)), None),
        (dict(grid_level=8, dense=True, want_normals=True), None),
        (dict(grid_level=4), None),
    ]
    reused = api.Mesh(ctx)
    try:
        for i, (kw, after) in enumerate(steps):
            kw = dict(kw)
            level = kw.pop("grid_level")
            results = []
            for mesh in (None, reused):
                m = ctx.extract(box, level, mesh=mesh, **kw)
                if after == "weld":
                    m.weld()
                elif after == "orient":
                    m.orient()
                r = _mesh_result(m)
                r["stl"] = _b(m.format_stl())
                r["inspect"] = _report(m.inspect())
                results.append(r)
                if mesh is None:
                    m.free()
            fresh, got = results
            if not kw.get("want_normals"):
                assert not reused.c.d_normals and not reused.c.h_normals, "step %d: normals left over" % i
            bad = [f for f in sorted(fresh) if fresh[f] != got.get(f)]
            assert not bad, "step %d (%s, %s): %s differ" % (i, kw, after, bad)
    finally:
        reused.free()
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: rebuilds on one context
# ---------------------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_rebuilds_on_one_context(refs, tmp_path):
    """Design1 -> Design2 -> the logo -> synth64 (its side table swapped and left so) -> a scene that fails to compile ->
    Design1 -> synth64: after each build the fixed operations equal the fresh-context references -- the slab plan before any
    search of the new scene, the side table, the projection counters included."""
    from designcsg_b200 import api
    ref, boxes, tmp = refs
    broken = tmp_path / "broken"
    src = scenes.materialize(D1)["dir"]
    broken.mkdir()
    for fn in ("scene.txt", "buildprocedure.txt", "arbitrary_data.hex", "exportConfig.txt"):
        (broken / fn).write_bytes(open(os.path.join(src, fn), "rb").read())
    (broken / "scene.cu").write_text(open(os.path.join(src, "scene.cu")).read().replace("length(v)-0.5", "lenght(v)-0.5"))
    ctx = api.Context(0)
    env = Env(boxes, tmp)
    env.on_torch_stream = False
    try:
        for name in (D1, "design2", "logo", "synth64", None, D1, "synth64"):
            if name is None:
                with pytest.raises(api.DcsgError) as e:
                    ctx.build(str(broken))
                assert e.value.code == -1 and "lenght" in ctx.build_log
                with pytest.raises(api.DcsgError) as e:
                    ctx.extract(boxes[D1], 5)
                assert e.value.code == -4
                continue
            ctx.build(scenes.materialize(name)["dir"])
            for key in REBUILD_OPS[name]:
                bad = _diff(run_op(ctx, env, key), ref[key])
                assert bad is None, "after building %s: %s: %s differ" % (name, key, bad)
            if name == "synth64":
                raw = open(os.path.join(scenes.materialize(name)["dir"], "arbitrary_data.hex"), "rb").read()
                table = np.zeros(131072, dtype=np.float32)
                table[:len(raw) // 4] = np.frombuffer(raw, dtype="<f4")
                ctx.set_arbitrary_data(_swapped_table(table))        # the next build must not inherit it
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: a caller's stream
# ---------------------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_callers_stream(refs):
    """dcsg_set_stream with torch streams: a spin kernel queued on the stream before each library call holds the stream back,
    so any work the library put on another stream without an event would run first and read or leave the wrong data.  The
    results are read through torch on the same stream, without a device synchronise."""
    import torch
    from designcsg_b200 import api
    ref, boxes, tmp = refs
    ctx = api.Context(0)
    ctx.build(scenes.materialize(D1)["dir"])
    env = Env(boxes, tmp)
    env.on_torch_stream = True
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    try:
        for stream in (s1, s2, torch.cuda.default_stream(), s1):
            torch.cuda.synchronize()
            ctx.set_stream(stream.cuda_stream)
            with torch.cuda.stream(stream):
                env.pre = lambda: torch.cuda._sleep(SLEEP_CYCLES)
                for key in ("d1/eval-device", "d1/project-u6", "d1/weld", "d1/orient", "d1/inspect", "d1/u5", "d1/bbox10"):
                    bad = _diff(run_op(ctx, env, key), ref[key])
                    assert bad is None, "stream %s: %s: %s differ" % (stream, key, bad)
    finally:
        torch.cuda.synchronize()
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: two contexts at once
# ---------------------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_two_contexts_in_two_threads(refs):
    from designcsg_b200 import api
    ref, boxes, tmp = refs
    ctxs = {}
    for name in (D1, "design2"):
        ctxs[name] = api.Context(0)
        ctxs[name].build(scenes.materialize(name)["dir"])
    results = {D1: [], "design2": []}
    errors = []

    def drive(name, key):
        try:
            env = Env(boxes, tmp)
            env.on_torch_stream = False
            for _ in range(4):
                results[name].append(run_op(ctxs[name], env, key))
        except Exception as err:       # reported by the main thread
            errors.append(err)

    threads = [threading.Thread(target=drive, args=(D1, "d1/chain")), threading.Thread(target=drive, args=("design2", "d2/chain"))]
    try:
        for t in threads:
            t.start()
    finally:
        for t in threads:
            t.join()
        for c in ctxs.values():
            c.close()
    assert not errors, errors
    for name, key in ((D1, "d1/chain"), ("design2", "d2/chain")):
        assert len(results[name]) == 4
        for i, got in enumerate(results[name]):
            assert _diff(got, ref[key]) is None, "%s round %d: %s" % (name, i, _diff(got, ref[key]))
