"""Numeric golden vectors from the REFERENCE'S OWN code (oracle/_ref), committed as small fixtures.

    python tests/golden/make_vectors.py          # needs /root/reference (build container only)

For every stock scene this builds the reference-flavour oracle (the reference's k2.cl + scene.cl text and
its cms / ISV / CVector sources, compiled headless by oracle/build.py) and records in
tests/golden/<scene>/vectors.npz:

  points / sdf / normals    seeded random points in the search volume, k2's answers
  box                       result of the 256^3 bounding-box search
  lattice16                 SDF on the 17^3 lattice of grid level 4
  L, tris, soup_sha         uniform export at grid level L: triangle count, sha256 of the sorted soup
  gd_steps, gd_sha          ... after gradient descent
  ply_sha, stl_sha          sha256 of the files the reference's writers produce for that mesh
  preview_sha               sha256 of the 640x480 RGB frame the reference's kernel k1 renders for tests.helpers.PREVIEW_CAMERAS
  adaptive_*                adaptive octree levels (min < max <= grid): triangle count, sha256 of the sorted soup
                            of getSurface, and of getSurface + retopologize
The CPU port (oracle/) and the CUDA path are both tested against these.

It also records tests/golden/<scene>/pins.npz and tests/golden/lookup_table.npz (see PIN_SCENES below):

  seed5_sdf_sha             the SDF on 20000 points drawn with seed 5
  walk5_*                   uniform walk at grid level 5 in the walk's own order: count, sha256, and after 3 descent steps
  lattice_points            three lattice points of the 33^3 lattice
  special_sdf / _normals    SDF and 6-tap normals on the 20^3 grid of special coordinates
  adaptive_walk_*           the adaptive walk in its own order
  table                     (lookup_table.npz) the 256x16 triangle table read from the reference's lookupTable.txt

    python tests/golden/make_vectors.py --pins-from-port   # the same files from the port, where no reference build exists
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle.oracle import Oracle  # noqa: E402
from tests import helpers as H  # noqa: E402
from tests.golden import scenes  # noqa: E402

LEVEL = {"design1": 5, "design2": 5, "stress": 6, "synth64": 5}
ADAPTIVE = {"design1": (3, 5, 6), "design2": (4, 6, 6), "stress": (3, 6, 6), "synth64": (3, 5, 6)}     # min, max, grid
GD_STEPS = 5


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def logo_vectors():
    """The reference's Logo.py (three Bezier-outline letters, ~6 k sub-segments per SDF evaluation, a mutable
    program-scope variable): the CPU needs ~0.2 ms per evaluation, so the fixture is small and the 256^3 bounding-box
    search (9 minutes on 8 cores) is only re-run with --slow; otherwise the recorded box is kept."""
    scene = scenes.materialize("logo")
    ref = Oracle.for_scene(scene, "reference")
    out = os.path.join(HERE, "logo", "vectors.npz")
    if "--slow" in sys.argv or not os.path.exists(out):
        box = ref.bbox(10.0)
    else:
        box = np.load(out)["box"]
    rng = np.random.default_rng(2025)
    pts = rng.uniform(-3.2, 3.2, (1000, 3)).astype(np.float32)
    L = 5
    soup = ref.get_surface(box, L, L, L)
    gd = ref.gradient_descent(H.canon_soup(soup)[:300], 2)           # projection is per vertex: a subset is enough
    adaptive = ref.get_surface(box, 3, 5, 5)
    np.savez_compressed(out, points=pts, sdf=ref.eval_sdf(pts), normals=ref.eval_normal(pts[:200]), box=box,
                        lattice8=ref.lattice_sdf(box, 8), L=L, tris=len(soup), soup_sha=sha(H.canon_soup(soup)), gd_steps=2,
                        gd_sha=sha(gd), adaptive_levels=np.array([3, 5, 5]), adaptive_tris=len(adaptive),
                        adaptive_sha=sha(H.canon_soup(adaptive)))
    print("logo L", L, "tris", len(soup), "adaptive", len(adaptive), "box", box)


# tests/golden/<scene>/pins.npz: what tests/test_oracle_pinning.py's direct comparisons with the reference build compare, so
# that they also run without one.  Recorded from the reference build, or with --pins-from-port from the port, which those
# direct comparisons found bit-identical to it on these inputs; the file's `source` says which.
PIN_SCENES = {"design1": (3, 5, 6), "design2": (4, 6, 6), "stress": (3, 6, 6)}      # adaptive levels: min, max, grid
PIN_DIRECT = ("design1", "design2")
PIN_LATTICE_POINTS = ((0, 0, 0), (32, 7, 19), (13, 32, 1))
SPECIAL_VALUES = [0.0, -0.0, 5.0, -5.0, 1e-30, -1e-30, 1e-45, 2.0 ** -61, 2.0 ** -59, 1e37, -1e37, 3e38, np.inf, -np.inf, np.nan,
                  1.5, -0.75, 4.9999995, 5.0000005, 1e-18]


def special_points():
    """The 20^3 grid of special coordinates (signed zeros, denormal / tiny / huge / infinite / NaN, centres and planes)."""
    vals = np.array(SPECIAL_VALUES, dtype=np.float32)
    return np.ascontiguousarray(np.stack(np.meshgrid(vals, vals, vals, indexing="ij"), axis=-1).reshape(-1, 3))


def seed5_points():
    return np.random.default_rng(5).uniform(-5, 5, (20000, 3)).astype(np.float32)


def pins(orc, name):
    box = orc.bbox(10.0)
    out = {}
    if name in PIN_DIRECT:
        soup = orc.get_surface(box, 5, 5, 5)                 # walk order, unsorted
        with np.errstate(all="ignore"):
            sp = special_points()
            out.update(seed5_sdf_sha=sha(orc.eval_sdf(seed5_points())), walk5_tris=len(soup), walk5_sha=sha(soup),
                       walk5_gd3_sha=sha(orc.gradient_descent(soup, 3)),
                       lattice_points=np.array([orc.lattice_point(box, 32, *p) for p in PIN_LATTICE_POINTS]),
                       special_sdf=orc.eval_sdf(sp), special_normals=orc.eval_normal(sp))
    lo, hi, grid = PIN_SCENES[name]
    adaptive = orc.get_surface(box, lo, hi, grid)
    out.update(adaptive_levels=np.array([lo, hi, grid]), adaptive_walk_tris=len(adaptive), adaptive_walk_sha=sha(adaptive))
    return out


def record_pins(flavour):
    from oracle import build as obuild
    from oracle.oracle import tri_table
    for name in PIN_SCENES:
        orc = Oracle.for_scene(scenes.materialize(name), flavour)
        assert orc.flavour == flavour
        np.savez_compressed(os.path.join(HERE, name, "pins.npz"), source=flavour, **pins(orc, name))
        print(name, "pins from the", flavour)
    if flavour == "reference":
        table, n = orc.load_lookup_file(os.path.join(obuild.REFERENCE, "lookupTable.txt"))   # the reference's own reader
        assert n == 820
    else:
        table = tri_table()
    np.savez_compressed(os.path.join(HERE, "lookup_table.npz"), source=flavour, table=table)


def main():
    if "--logo" in sys.argv:
        return logo_vectors()
    if "--pins-from-port" in sys.argv:
        return record_pins("port")
    record_pins("reference")
    for name in scenes.names():
        scene = scenes.materialize(name)
        ref = Oracle.for_scene(scene, "reference")
        assert ref.flavour == "reference"
        rng = np.random.default_rng(2024)
        pts = rng.uniform(-4.5, 4.5, (2000, 3)).astype(np.float32)
        box = ref.bbox(10.0)
        L = LEVEL[name]
        soup = ref.get_surface(box, L, L, L)
        gd = ref.gradient_descent(soup, GD_STEPS)
        with tempfile.TemporaryDirectory() as tmp:
            ref.write_ply(os.path.join(tmp, "m.ply"), gd)
            ref.write_stl(os.path.join(tmp, "m.stl"), gd)
            ply_sha = hashlib.sha256(open(os.path.join(tmp, "m.ply"), "rb").read()).hexdigest()
            stl_sha = hashlib.sha256(open(os.path.join(tmp, "m.stl"), "rb").read()).hexdigest()
        order = np.lexsort(soup.reshape(-1, 9).T[::-1])
        lo, hi, grid = ADAPTIVE[name]
        adaptive = ref.get_surface(box, lo, hi, grid)
        retopo = ref.get_surface(box, lo, hi, grid, retopologize=True)
        previews = [sha(ref.preview(*cam)) for cam in H.PREVIEW_CAMERAS]
        out = os.path.join(HERE, name)
        os.makedirs(out, exist_ok=True)
        np.savez_compressed(os.path.join(out, "vectors.npz"),
                            points=pts, sdf=ref.eval_sdf(pts), normals=ref.eval_normal(pts[:500]), box=box,
                            lattice16=ref.lattice_sdf(box, 16), L=L, tris=len(soup),
                            soup_sha=sha(soup.reshape(-1, 9)[order]), gd_steps=GD_STEPS,
                            gd_sha=sha(gd.reshape(-1, 9)[order]), ply_sha=ply_sha, stl_sha=stl_sha,
                            adaptive_levels=np.array([lo, hi, grid]), adaptive_tris=len(adaptive),
                            adaptive_sha=sha(H.canon_soup(adaptive)), adaptive_retopo_sha=sha(H.canon_soup(retopo)),
                            preview_sha=np.array(previews))
        print(name, "L", L, "tris", len(soup), "box", box)


if __name__ == "__main__":
    main()
