"""Pins the CPU oracle (oracle/, our restatement) to the reference:
 * against the committed vectors recorded from the reference's own code (tests/golden/*/vectors.npz);
 * against tests/golden/*/pins.npz and tests/golden/lookup_table.npz, what the direct comparisons below compare;
 * where a build of the reference's sources exists (oracle/_ref), directly as well."""
import hashlib
import os
import re

import numpy as np
import pytest

from oracle import build as obuild
from oracle.oracle import Oracle, tri_table
from tests.golden import make_vectors as mv
from tests.golden import scenes

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module", params=scenes.names())
def pinned(request):
    name = request.param
    scene = scenes.materialize(name)
    return name, Oracle.for_scene(scene, "port"), np.load(os.path.join(HERE, "golden", name, "vectors.npz"))


def test_point_values_match_reference_vectors(pinned):
    _, orc, vec = pinned
    assert np.array_equal(orc.eval_sdf(vec["points"]), vec["sdf"])
    assert np.array_equal(orc.eval_normal(vec["points"][:500]), vec["normals"], equal_nan=True)


def test_bbox_and_lattice_match_reference_vectors(pinned):
    _, orc, vec = pinned
    assert np.array_equal(orc.bbox(10.0), vec["box"])
    assert np.array_equal(orc.lattice_sdf(vec["box"], 16), vec["lattice16"])


def test_surface_projection_and_files_match_reference_vectors(pinned, tmp_path):
    _, orc, vec = pinned
    L = int(vec["L"])
    soup = orc.get_surface(vec["box"], L, L, L)
    assert len(soup) == int(vec["tris"])
    order = np.lexsort(soup.reshape(-1, 9).T[::-1])
    assert sha(soup.reshape(-1, 9)[order]) == str(vec["soup_sha"])
    gd = orc.gradient_descent(soup, int(vec["gd_steps"]))
    assert sha(gd.reshape(-1, 9)[order]) == str(vec["gd_sha"])
    orc.write_ply(str(tmp_path / "m.ply"), gd)
    orc.write_stl(str(tmp_path / "m.stl"), gd)
    assert hashlib.sha256((tmp_path / "m.ply").read_bytes()).hexdigest() == str(vec["ply_sha"])
    assert hashlib.sha256((tmp_path / "m.stl").read_bytes()).hexdigest() == str(vec["stl_sha"])


def _ref_or_skip(name):
    if not obuild.have_reference() and not os.path.exists(obuild.ref_lib_path(name)):
        pytest.skip("no build of the reference sources available")
    return Oracle.for_scene(scenes.materialize(name), "reference")


def _ref_or_none(name):
    """The reference build for a direct comparison, where one exists; the stored pins are compared either way."""
    if not obuild.have_reference() and not os.path.exists(obuild.ref_lib_path(name)):
        return None
    return Oracle.for_scene(scenes.materialize(name), "reference")


def _pins(name):
    """tests/golden/<name>/pins.npz (make_vectors.py): what the comparisons below compare with the reference build."""
    return np.load(os.path.join(HERE, "golden", name, "pins.npz"))


def _same_bits(a, b):
    """Bit for bit (the sign of a zero included) wherever the values are numbers; NaN at the same places."""
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a.view(np.uint32)[~np.isnan(a)], b.view(np.uint32)[~np.isnan(b)])


@pytest.mark.parametrize("name", ["design1", "design2"])
def test_port_equals_reference_build_directly(name):
    orc, pin = Oracle.for_scene(scenes.materialize(name), "port"), _pins(name)
    pts = mv.seed5_points()
    box = orc.bbox(10.0)
    a = orc.get_surface(box, 5, 5, 5)
    assert sha(orc.eval_sdf(pts)) == str(pin["seed5_sdf_sha"])
    assert len(a) == int(pin["walk5_tris"]) and sha(a) == str(pin["walk5_sha"])        # same triangles in the same (walk) order
    assert sha(orc.gradient_descent(a, 3)) == str(pin["walk5_gd3_sha"])
    assert np.array_equal([orc.lattice_point(box, 32, *p) for p in mv.PIN_LATTICE_POINTS], pin["lattice_points"])
    ref = _ref_or_none(name)
    if ref is None:
        return
    assert np.array_equal(orc.eval_sdf(pts), ref.eval_sdf(pts))
    box = ref.bbox(10.0)
    a, b = orc.get_surface(box, 5, 5, 5), ref.get_surface(box, 5, 5, 5)
    assert np.array_equal(a, b)
    assert np.array_equal(orc.gradient_descent(a, 3), ref.gradient_descent(b, 3), equal_nan=True)
    for ix, iy, iz in mv.PIN_LATTICE_POINTS:
        assert np.array_equal(orc.lattice_point(box, 32, ix, iy, iz), ref.lattice_point(box, 32, ix, iy, iz))


@pytest.mark.parametrize("name", ["design1", "design2"])
def test_port_equals_reference_build_on_special_points(name):
    """Signed zeros, object centres and centre planes, denormal / tiny / huge / infinite / NaN coordinates: the points on
    which the GPU's checked fast copy must fall back to its exact copy (tests/test_gpu_parity.py compares the GPU with the
    port there).  This closes the chain on the CPU: on the same points the port returns the bits of the reference's own
    k2.cl -- values and 6-tap normals."""
    orc, pin = Oracle.for_scene(scenes.materialize(name), "port"), _pins(name)
    pts = mv.special_points()
    with np.errstate(all="ignore"):
        a, n = orc.eval_sdf(pts), orc.eval_normal(pts)
        assert _same_bits(a, pin["special_sdf"])
        assert _same_bits(n, pin["special_normals"])
        ref = _ref_or_none(name)
        if ref is not None:
            assert _same_bits(a, ref.eval_sdf(pts))
            assert np.array_equal(n, ref.eval_normal(pts), equal_nan=True)


def test_lookup_table_forms_agree():
    """golden loops --(oracle triangulation)--> table == the product's generated mc_table.inc
    == the table the reference's own reader parses from its own lookupTable.txt (stored in tests/golden/lookup_table.npz;
    read again where the reference is present)."""
    table = tri_table()
    assert (table >= 0).sum() == 820 * 3 and table[0, 0] == -1 and table[255, 0] == -1
    text = open(os.path.join(REPO, "designcsg_b200", "csrc", "mc_table.inc")).read()
    body = text.split("kDcsgTriTable[256 * 16] = {")[1].split("};")[0]
    assert np.array_equal(np.array([int(v) for v in re.findall(r"-?\d+", body)]).reshape(256, 16), table)
    counts = text.split("kDcsgTriCount[256] = {")[1].split("};")[0]
    assert np.array_equal(np.array([int(v) for v in re.findall(r"\d+", counts)]), (table >= 0).sum(axis=1) // 3)
    assert np.array_equal(np.load(os.path.join(HERE, "golden", "lookup_table.npz"))["table"], table)
    lookup = os.path.join(obuild.REFERENCE, "lookupTable.txt")
    if os.path.exists(lookup):
        ref = _ref_or_skip("design1")
        parsed, n = ref.load_lookup_file(lookup)
        assert n == 820 and np.array_equal(parsed, table)


def _reference_retopologize(name, box, lo, hi, grid):
    """getSurface + cms::retopologize of the reference build, in a process of its own: the function reads dead stack frames
    (mesh.hpp:413-430), so besides keeping other samples it can fault, and a fault must not take the test run with it.
    Returns the soup, or None when the child died."""
    import subprocess
    import sys
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        np.save(os.path.join(tmp, "box.npy"), np.asarray(box, dtype=np.float32))
        code = ("import sys, numpy as np; sys.path.insert(0, %r); from oracle.oracle import Oracle; from tests.golden import scenes; "
                "ref = Oracle.for_scene(scenes.materialize(%r), 'reference'); "
                "np.save(%r, ref.get_surface(np.load(%r), %d, %d, %d, retopologize=True))"
                % (REPO, name, os.path.join(tmp, "out.npy"), os.path.join(tmp, "box.npy"), lo, hi, grid))
        done = subprocess.run([sys.executable, "-c", code], timeout=600, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        if done.returncode != 0 or not os.path.exists(os.path.join(tmp, "out.npy")):
            return None
        return np.load(os.path.join(tmp, "out.npy"))


@pytest.mark.parametrize("name,lo,hi,grid", [("design1", 3, 5, 6), ("design2", 4, 6, 6), ("stress", 3, 6, 6)])
def test_adaptive_walk_and_retopologize_equal_reference_build(name, lo, hi, grid):
    """Adaptive octree levels (edge ambiguity + complex edges) and cms::retopologize: the port against the
    reference's own sources, same triangles in the same order (the walk: against the stored pins, and directly where a
    reference build exists; retopologize, the reference's undefined behaviour, only directly)."""
    orc, pin = Oracle.for_scene(scenes.materialize(name), "port"), _pins(name)
    assert [int(v) for v in pin["adaptive_levels"]] == [lo, hi, grid]
    box = orc.bbox(10.0)
    walk = orc.get_surface(box, lo, hi, grid)
    assert len(walk) == int(pin["adaptive_walk_tris"]) and sha(walk) == str(pin["adaptive_walk_sha"])
    a = orc.get_surface(box, lo, hi, grid, retopologize=True)
    assert len(a) == len(walk) * (3 * (1 << (grid - lo)) - 2)
    ref = _ref_or_none(name)
    if ref is None:
        return
    box = ref.bbox(10.0)
    assert np.array_equal(orc.get_surface(box, lo, hi, grid), ref.get_surface(box, lo, hi, grid))
    b = _reference_retopologize(name, box, lo, hi, grid)
    if b is None:
        pytest.xfail("reference retopologize (undefined behaviour) crashed in this run")
    if not np.array_equal(a, b):
        # cms::retopologize reads dead stack frames (mesh.hpp:413-430): which samples it keeps is whatever the garbage says.
        # Every CPU-oracle run so far kept all of them (the behaviour the port restates); a run that does not is the
        # reference's undefined behaviour showing, not a regression of the port.
        pytest.xfail("reference retopologize (undefined behaviour) kept %d triangles instead of %d in this run" % (len(b), len(a)))


def test_adaptive_vectors_recorded_from_the_reference(pinned):
    name, orc, vec = pinned
    if "adaptive_levels" not in vec:
        pytest.skip("vectors.npz predates the adaptive fixtures")
    lo, hi, grid = (int(v) for v in vec["adaptive_levels"])
    soup = orc.get_surface(vec["box"], lo, hi, grid)
    assert len(soup) == int(vec["adaptive_tris"])
    assert sha(H_canon(soup)) == str(vec["adaptive_sha"])
    retopo = orc.get_surface(vec["box"], lo, hi, grid, retopologize=True)
    assert sha(H_canon(retopo)) == str(vec["adaptive_retopo_sha"])


def H_canon(soup):
    a = np.ascontiguousarray(soup, dtype=np.float32).reshape(-1, 9)
    return a[np.lexsort(a.T[::-1])]
