"""File bytes against a numpy encoder of the formats: the soup PLY and STL (device formatters, host row expansion, the chunked
file pipeline), the indexed PLY writer and the weld -- at every tail, chunk, split and index limit, on adversarial float bits.

The encoder builds the files from the formats alone: happly's header and rows for the soup PLY, the STL layout, DESIGN.md
§7b for the indexed PLY.  It is anchored once against the oracle's writers; after that it is the reference for every path."""
import ctypes

import numpy as np
import pytest

from tests.golden import scenes
from tests.test_indexed_export import HEADER as INDEXED_HEADER, NORMALS as INDEXED_NORMALS, export_levels, numpy_weld, \
    read_indexed_ply

# the largest first + n of a soup PLY: its last index 3 (first + n) - 1 is then 2^32 - 2, and (first + n) * 3 = 2^32 - 1
INDEX_LIMIT = 0xffffffff // 3

SOUP_PLY_HEADER = ("ply\nformat binary_little_endian 1.0\ncomment Written with hapPLY (https://github.com/nmwsharp/happly)\n"
                   "element vertex {V}\nproperty double x\nproperty double y\nproperty double z\n"
                   "element face {T}\nproperty list uchar uint vertex_indices\nend_header\n")
STL_RECORD = np.dtype([("normal", "<u4", 3), ("corners", "<u4", 9), ("attribute", "<u2")])      # packed: 50 bytes
FACE_ROW = np.dtype([("count", "u1"), ("idx", "<u4", 3)])                                         # packed: 13 bytes


# ---- the encoder -------------------------------------------------------------------------------------------------------------

def is_nan_bits(b):
    b = np.asarray(b, np.uint32)
    return ((b & 0x7f800000) == 0x7f800000) & ((b & 0x007fffff) != 0)


def widen(values):
    """float32 -> the float64 bit patterns: exact for every number (denormals, zeros and infinities included); a NaN keeps its
    sign and payload and comes out quiet (bit 51 set), as IEEE 754's conversion makes a signalling NaN."""
    f = np.ascontiguousarray(values, np.float32)
    b = f.view(np.uint32).astype(np.uint64)
    with np.errstate(invalid="ignore"):
        out = f.astype(np.float64).view(np.uint64).copy()
    nan = is_nan_bits(f.view(np.uint32))
    out[nan] = ((b[nan] >> np.uint64(31)) << np.uint64(63)) | np.uint64(0x7ff8000000000000) | \
        ((b[nan] & np.uint64(0x7fffff)) << np.uint64(29))
    return out


def _corners(vertices, triangles):
    v = np.ascontiguousarray(vertices, np.float32).reshape(-1, 3)
    t = np.asarray(triangles).reshape(-1, 3).astype(np.int64)
    return v, t


def ply_vertex_rows(vertices, triangles):
    """Three doubles per corner, corners A, B, C of every triangle."""
    v, t = _corners(vertices, triangles)
    return widen(v[t]).astype("<u8").tobytes()


def ply_face_rows(first, n):
    """uchar 3, uint32 3i, 3i + 1, 3i + 2 for i = first .. first + n - 1."""
    assert (first + n) * 3 <= 0xffffffff
    rows = np.zeros(n, FACE_ROW)
    rows["count"] = 3
    rows["idx"] = np.arange(first, first + n, dtype=np.uint64)[:, None] * 3 + np.arange(3, dtype=np.uint64)
    return rows.tobytes()


def stl_records(vertices, triangles, acb=False):
    """A zero normal, the corners A, B, C (A, C, B when acb) each as (x, z, y), a zero attribute."""
    v, t = _corners(vertices, triangles)
    recs = np.zeros(len(t), STL_RECORD)
    c = v.view(np.uint32)[t[:, [0, 2, 1] if acb else [0, 1, 2]]]            # (T, corner, xyz)
    recs["corners"] = c[:, :, [0, 2, 1]].reshape(-1, 9)
    return recs.tobytes()


def encode_ply(vertices, triangles, first=0, total=None):
    n = len(np.asarray(triangles).reshape(-1, 3))
    total = n if total is None else total
    return SOUP_PLY_HEADER.format(V=3 * total, T=total).encode() + ply_vertex_rows(vertices, triangles) + ply_face_rows(first, n)


def encode_stl(vertices, triangles, acb=False, total=None):
    n = len(np.asarray(triangles).reshape(-1, 3))
    total = n if total is None else total
    return bytes(80) + np.uint32(total).astype("<u4").tobytes() + stl_records(vertices, triangles, acb)


def encode_ply_indexed(vertices, triangles, normals=None):
    v, t = _corners(vertices, triangles)
    dt = np.dtype([("xyz", "<u4", 3)] + ([("n", "<u4", 3)] if normals is not None else []))
    rows = np.zeros(len(v), dt)
    rows["xyz"] = v.view(np.uint32)
    if normals is not None:
        rows["n"] = np.ascontiguousarray(normals, np.float32).reshape(-1, 3).view(np.uint32)
    faces = np.zeros(len(t), FACE_ROW)
    faces["count"] = 3
    faces["idx"] = t
    header = INDEXED_HEADER.format(V=len(v), T=len(t), N=INDEXED_NORMALS if normals is not None else "")
    return header.encode() + rows.tobytes() + faces.tobytes()


def assert_bytes(got, want, what):
    g = np.frombuffer(got, np.uint8) if isinstance(got, (bytes, bytearray)) else np.ascontiguousarray(got).view(np.uint8).ravel()
    w = np.frombuffer(want, np.uint8) if isinstance(want, (bytes, bytearray)) else np.ascontiguousarray(want).view(np.uint8).ravel()
    if g.size == w.size and np.array_equal(g, w):
        return
    k = min(g.size, w.size)
    bad = np.flatnonzero(g[:k] != w[:k])
    at = int(bad[0]) if bad.size else k
    raise AssertionError("%s: %d bytes, want %d; first difference at byte %d: %s vs %s" % (
        what, g.size, w.size, at, g[at:at + 16].tobytes().hex(), w[at:at + 16].tobytes().hex()))


# ---- adversarial float sets ----------------------------------------------------------------------------------------------------

def _lanes():
    """Every word whose bytes are all 0x00 or 0xff, NaNs left out."""
    words = [sum(0xff << (8 * k) for k in range(4) if m >> k & 1) for m in range(16)]
    return [w for w in words if not is_nan_bits(w)]


SPECIAL = np.array(sorted(set([0x00000000, 0x80000000,                  # +-0
                               0x00000001, 0x80000001, 0x007fffff, 0x807fffff,      # smallest and largest denormals
                               0x00800000, 0x80800000, 0x7f7fffff, 0xff7fffff,      # FLT_MIN, FLT_MAX
                               0x7f800000, 0xff800000,                              # +-Inf
                               0x3f800000, 0xbf800001] + _lanes())), dtype=np.uint32)
QUIET_NANS = [0x7fc00001, 0xffc12345, 0x7fffffff]
SIGNALLING_NANS = [0x7f800001, 0xff800001, 0x7fa00000]
NANS = np.array(QUIET_NANS + SIGNALLING_NANS, dtype=np.uint32)
SETS = ("random", "special", "nan")


def float_bits(kind, shape, rng):
    """uint32 float patterns: `random` (any bits but NaN), `special`, `nan` (the NaN set mixed half and half with the special
    set), `mixed` (each word from one of the three)."""
    if kind == "random":
        b = rng.integers(0, 1 << 32, size=shape, dtype=np.uint64).astype(np.uint32)
        return np.where(is_nan_bits(b), b ^ np.uint32(0x40000000), b)      # exponent 0xff -> 0xbf
    if kind == "special":
        return rng.choice(SPECIAL, size=shape)
    if kind == "nan":
        return np.where(rng.random(shape) < 0.5, rng.choice(NANS, size=shape), rng.choice(SPECIAL, size=shape))
    pick = rng.integers(0, 3, size=shape)
    out = float_bits("random", shape, rng)
    out[pick == 1] = float_bits("special", int((pick == 1).sum()), rng)
    out[pick == 2] = float_bits("nan", int((pick == 2).sum()), rng)
    return out


def random_mesh(kind, n, rng, V=None):
    """n triangles on V vertices (default n // 2 + 1: many degenerate triangles), positions from a float set."""
    V = n // 2 + 1 if V is None else V
    return float_bits(kind, (V, 3), rng).view(np.float32), rng.integers(0, V, size=(n, 3)).astype(np.uint32)


# ---- CPU: the encoder against the oracle, the host row functions against the encoder --------------------------------------------

def test_encoder_is_the_oracle_writers(tmp_path):
    from oracle.oracle import Oracle
    orc = Oracle.for_scene(scenes.materialize("design1"), "port")
    soup = orc.get_surface(orc.bbox(10.0), 5, 5, 5)
    assert len(soup) > 1000
    v, t = soup.reshape(-1, 3), np.arange(3 * len(soup)).reshape(-1, 3)
    orc.write_ply(str(tmp_path / "o.ply"), soup)
    orc.write_stl(str(tmp_path / "o.stl"), soup)
    assert_bytes((tmp_path / "o.ply").read_bytes(), encode_ply(v, t), "PLY")
    assert_bytes((tmp_path / "o.stl").read_bytes(), encode_stl(v, t), "STL")


def test_encoder_known_bytes():
    """One record of each by hand: the x z y order, the quieted NaN, the face row."""
    v = np.array([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0], [7.0, 8.0, 9.0]], np.float32)
    v.view(np.uint32)[2, 1] = 0x7f800001
    rec = stl_records(v, [[0, 1, 2]])
    assert len(rec) == 50 and rec[:12] == bytes(12) and rec[48:] == bytes(2)
    assert np.frombuffer(rec[12:48], "<u4")[:6].tolist() == [0x3f800000, 0x40400000, 0x40000000, 0x40800000, 0x40c00000, 0x40a00000]
    assert np.frombuffer(rec[12:48], "<u4")[8] == 0x7f800001
    acb = stl_records(v, [[0, 1, 2]], acb=True)
    assert acb[:12] == rec[:12] and acb[12:24] == rec[12:24] and acb[24:36] == rec[36:48] and acb[36:48] == rec[24:36]
    assert widen(np.array([0x7f800001, 0xffc12345, 0x00000001], np.uint32).view(np.float32)).tolist() == \
        [0x7ff8000020000000, 0xfff82468a0000000, 0x36a0000000000000]
    assert ply_face_rows(2, 1) == bytes([3, 6, 0, 0, 0, 7, 0, 0, 0, 8, 0, 0, 0])


def _aligned(nbytes, offset, align=64):
    """A uint8 array of nbytes that starts `offset` bytes past an `align`-byte boundary (and the buffer that owns it)."""
    buf = np.zeros(nbytes + offset + 2 * align, np.uint8)
    skip = (-buf.ctypes.data) % align + offset
    return buf[skip:skip + nbytes]


def host_soup_rows(vertices, triangles, stl_offset=0):
    """dcsg_soup_rows with the STL records `stl_offset` bytes past a word boundary (the PLY rows must be 8-byte aligned)."""
    from designcsg_b200 import api
    lib = api.load_library()
    v, t = _corners(vertices, triangles)
    soup = np.ascontiguousarray(v[t]).reshape(-1, 9)
    ply, stl = _aligned(72 * len(t), 0), _aligned(50 * len(t), stl_offset)
    ply[:] = 0xa5
    stl[:] = 0xa5
    rc = lib.dcsg_soup_rows(soup.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), len(t), ply.ctypes.data_as(api._u8p),
                            stl.ctypes.data_as(api._u8p))
    assert rc == 0
    return ply.tobytes(), stl.tobytes()


def host_face_rows(first, n, offset=0):
    from designcsg_b200 import api
    lib = api.load_library()
    out = _aligned(13 * n, offset)
    out[:] = 0xa5
    rc = lib.dcsg_ply_face_rows(first, n, out.ctypes.data_as(api._u8p), out.size)
    if rc != 0:
        raise api.DcsgError(rc, "dcsg_ply_face_rows(%d, %d)" % (first, n))
    return out.tobytes()


@pytest.mark.parametrize("kind", SETS)
def test_host_rows_equal_the_encoder(libdcsg, kind):
    """Every count 0 .. 67 (both STL paths: two records per 25 words from a word boundary, one at a time elsewhere; the face
    rows' four-row blocks and their tails), on every float set."""
    rng = np.random.default_rng(11)
    for n in range(68):
        v, t = random_mesh(kind, n, rng)
        rows, recs = ply_vertex_rows(v, t), stl_records(v, t)
        for off in (0, 1, 2, 3):
            ply, stl = host_soup_rows(v, t, off)
            assert_bytes(ply, rows, "PLY rows, n=%d" % n)
            assert_bytes(stl, recs, "STL records, n=%d, offset %d" % (n, off))
        for first in (0, 1, 3, 1 << 30 | 1):
            for off in (0, 1, 2, 3):
                assert_bytes(host_face_rows(first, n, off), ply_face_rows(first, n), "face rows, first=%d n=%d" % (first, n))


def test_host_face_rows_at_the_index_limit(libdcsg):
    from designcsg_b200 import api
    for n in (1, 2, 3, 4, 5, 13):
        first = INDEX_LIMIT - n
        for off in (0, 1):
            assert_bytes(host_face_rows(first, n, off), ply_face_rows(first, n), "face rows, first=%d n=%d" % (first, n))
        assert np.frombuffer(ply_face_rows(first, n)[-4:], "<u4")[0] == 0xfffffffe
        with pytest.raises(api.DcsgError):
            host_face_rows(first + 1, n)
    host_face_rows(INDEX_LIMIT, 0)
    with pytest.raises(api.DcsgError):
        host_face_rows(INDEX_LIMIT + 1, 0)


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


def _tensor(mesh, name):
    import torch
    return torch.as_tensor(mesh.device(name), device="cuda")


def write_device(mesh, name, array):
    """Bits into the first rows of a device array of the mesh (an integer copy: no float operation touches them)."""
    import torch
    view = _tensor(mesh, name)
    a = np.ascontiguousarray(array)
    view.view(torch.int32)[:len(a)] = torch.from_numpy(a.view(np.int32).reshape(len(a), -1)).cuda()
    torch.cuda.synchronize()


def read_device(mesh, name, count):
    import torch
    torch.cuda.synchronize()
    view = _tensor(mesh, name)
    return view.view(torch.int32)[:count].cpu().numpy().view(np.float32 if name in ("vertices", "normals") else np.uint32)


class Part:
    """A Mesh over a carrier's device arrays with counts of its own (a copy of the carrier's struct)."""

    def __init__(self, carrier):
        from designcsg_b200 import api
        self.mesh = api.Mesh(carrier._ctx)
        ctypes.memmove(ctypes.byref(self.mesh.c), ctypes.byref(carrier.c), ctypes.sizeof(api.MeshStruct))

    def set(self, vertices, triangles):
        self.mesh.c.num_vertices, self.mesh.c.num_triangles = vertices, triangles
        return self.mesh

    def release(self):
        self.mesh._ctx = None                                # borrowed storage: the carrier frees it


def _refused(call):
    from designcsg_b200 import api
    with pytest.raises(api.DcsgError) as err:
        call()
    assert err.value.code == -2 and "32 bits" in str(err.value), err.value


PLAIN_COUNTS = list(range(68)) + list(range(4093, 4100)) + [(1 << 20) + 3]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", SETS)
def test_plain_formatters(ctxs, tmp_path, kind):
    """format_ply / format_stl, their views, write_ply / write_stl and format_segments(first) on hand-made meshes written into
    a lattice carrier: every count 0 .. 67, 4093 .. 4099 and 2^20 + 3, random in-range ids, every float set."""
    ctx = ctxs("design1")
    carrier = ctx.extract(ctx.bbox(10.0), 9, copy_to_host=False)
    assert carrier.num_triangles > max(PLAIN_COUNTS) and carrier.num_vertices > max(PLAIN_COUNTS) // 2 + 1
    part = Part(carrier)
    rng = np.random.default_rng(SETS.index(kind))
    try:
        for n in PLAIN_COUNTS:
            v, t = random_mesh(kind, n, rng)
            if n:
                write_device(carrier, "vertices", v)
                write_device(carrier, "triangles", t)
            mesh = part.set(len(v), n)
            want_ply, want_stl = encode_ply(v, t), encode_stl(v, t)
            assert_bytes(mesh.format_ply(), want_ply, "format_ply n=%d" % n)
            assert_bytes(mesh.format_stl(), want_stl, "format_stl n=%d" % n)
            assert_bytes(mesh.format_ply_view(), want_ply, "format_ply_view n=%d" % n)
            assert_bytes(mesh.format_stl_view(), want_stl, "format_stl_view n=%d" % n)
            mesh.write_ply(str(tmp_path / "w.ply"))
            mesh.write_stl(str(tmp_path / "w.stl"))
            assert_bytes((tmp_path / "w.ply").read_bytes(), want_ply, "write_ply n=%d" % n)
            assert_bytes((tmp_path / "w.stl").read_bytes(), want_stl, "write_stl n=%d" % n)
            rows, recs = ply_vertex_rows(v, t), stl_records(v, t)
            for first in (0, 1, 3, 1 << 30 | 1, INDEX_LIMIT - n):
                a, b, c = mesh.format_segments(first)
                assert_bytes(a, rows, "segment rows n=%d first=%d" % (n, first))
                assert_bytes(b, ply_face_rows(first, n), "segment faces n=%d first=%d" % (n, first))
                assert_bytes(c, recs, "segment records n=%d first=%d" % (n, first))
            _refused(lambda: mesh.format_segments(INDEX_LIMIT - n + 1))
        # one triangle past the limit in the whole-file formatters (refused before any buffer is sized)
        mesh = part.set(1, INDEX_LIMIT + 1)
        _refused(mesh.format_ply_view)
        _refused(lambda: mesh.write_ply(str(tmp_path / "x.ply")))
    finally:
        part.release()
        carrier.free()


def _host_split(n, permille):
    """The file pipeline's split of a one-chunk mesh (n < 400000): the device formats [0, split), the host expands the rest.
    Every chunk end and every host share is a multiple of four (the host share is floor4(chunk * permille / 1000), and those
    floors never add up past n * permille / 1000), so on any mesh the last chunk's host range starts at n mod 4."""
    assert n < 400000
    return n - ((n * permille // 1000) & ~3)


PERMILLES = (0, 1, 3, 250, 600, 999, 1000)


def _slab_pair(ctx, box, level, residue):
    """Two z-slabs (0, z) and (z, 2^level), z nearest the middle, whose first holds a triangle count of the given residue mod 4
    (the stress scene: Design1's symmetry makes every count of its lattices a multiple of four)."""
    N = 1 << level
    for z in sorted(range(1, N), key=lambda z: abs(z - N // 2)):
        lo = ctx.extract(box, level, slab=(0, z), defer_projection=True, copy_to_host=False)
        if lo.num_triangles % 4 == residue:
            return lo, ctx.extract(box, level, slab=(z, N), defer_projection=True, copy_to_host=False)
        lo.free()
    raise AssertionError("no slab with %d triangles mod 4" % residue)


def _adversarial_positions(mesh, rng):
    """Overwrite every vertex position with mixed adversarial bits; -> (positions, triangles) as the pipeline will read them."""
    v = float_bits("mixed", (mesh.num_vertices, 3), rng).view(np.float32)
    write_device(mesh, "vertices", v)
    return v, read_device(mesh, "triangles", mesh.num_triangles)


PIPELINE_MESHES = [("lattice", 6), ("lattice", 8), ("lattice", 9), ("lattice", 10), ("slab", 0), ("slab", 1), ("slab", 2),
                   ("slab", 3), ("adaptive", 0), ("adaptive", 1), ("oriented", 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,arg", PIPELINE_MESHES)
def test_pipeline(ctxs, tmp_path, monkeypatch, kind, arg):
    """project_and_format_segments and project_and_write_files with gd_steps = 0 (the positions as written) on real deferred
    meshes -- Design1 lattices of 1 to 12 chunks, z-slabs of every triangle count mod 4, an adaptive soup (unit 1) and a
    retopologized one (unit 3p - 2), an oriented mesh (A, C, B records) -- at every host share of the rows.  Chunks and host
    shares are multiples of four triangles, so an odd count is what starts a host range on an odd triangle."""
    ctx = ctxs("design1" if kind in ("lattice", "adaptive") else "stress")
    box = ctx.bbox(10.0)
    other = None
    if kind == "lattice":
        mesh = ctx.extract(box, arg, defer_projection=True, copy_to_host=False)
    elif kind == "slab":
        mesh, other = _slab_pair(ctx, box, 8, arg)
    elif kind == "adaptive":
        search, lo, hi, grid, thr, _ = export_levels("design1")
        mesh = ctx.extract(ctx.bbox(search), grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=bool(arg),
                           defer_projection=True, copy_to_host=False)
    else:
        mesh = ctx.extract(box, arg, defer_projection=True, copy_to_host=False)
        mesh.orient()
    if other is not None:
        other.free()
    acb = kind == "oriented"
    n = mesh.num_triangles
    try:
        v, t = _adversarial_positions(mesh, np.random.default_rng(n))
        rows, faces, recs = ply_vertex_rows(v, t), ply_face_rows(0, n), stl_records(v, t, acb)
        want_ply = SOUP_PLY_HEADER.format(V=3 * n, T=n).encode() + rows + faces
        want_stl = encode_stl(v, t, acb)[:84] + recs
        for p in PERMILLES:
            monkeypatch.setenv("DCSG_HOST_EXPAND_PERMILLE", str(p))
            a, b, c = mesh.project_and_format_segments(0, 0)
            assert_bytes(a, rows, "rows, permille %d" % p)
            assert_bytes(b, faces, "faces, permille %d" % p)
            assert_bytes(c, recs, "records, permille %d" % p)
            mesh.project_and_write_files(0, str(tmp_path / "p.stl"), str(tmp_path / "p.ply"))
            assert_bytes((tmp_path / "p.ply").read_bytes(), want_ply, "PLY file, permille %d" % p)
            assert_bytes((tmp_path / "p.stl").read_bytes(), want_stl, "STL file, permille %d" % p)
        # the soup index limit: accepted up to it, refused one past it
        first = INDEX_LIMIT - n
        a, b, c = mesh.project_and_format_segments(0, first)
        assert_bytes(a, rows, "rows at the index limit")
        assert_bytes(b, ply_face_rows(first, n), "faces at the index limit")
        assert_bytes(c, recs, "records at the index limit")
        _refused(lambda: mesh.project_and_format_segments(0, first + 1))
        for name in ("x.ply", "x.stl"):
            (tmp_path / name).write_bytes(b"")
        _refused(lambda: mesh.project_and_write_files(0, str(tmp_path / "x.stl"), str(tmp_path / "x.ply"), first_triangle=first + 1,
                                                      total_triangles=INDEX_LIMIT + 1, create_files=False))
        assert (tmp_path / "x.ply").read_bytes() == b"" and (tmp_path / "x.stl").read_bytes() == b""
        if kind == "slab":
            assert n % 4 == arg and n < 400000
            # an odd count: the host range starts on an odd triangle (FileSink::expand_rows one record at a time), and the
            # device's part ends in k_format_stl's single record
            if arg % 2:
                assert all(_host_split(n, p) % 2 == 1 for p in PERMILLES if 0 < p < 1000)
        print("%s %s: %d triangles, %d vertices, n mod 4 = %d" % (kind, arg, n, mesh.num_vertices, n % 4))
    finally:
        mesh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("permille", [0, 600, 1000])
def test_two_ranks_into_one_pair_of_files(ctxs, tmp_path, monkeypatch, permille):
    """Two z-slabs written as the ranks of a sharded export write them: into files made beforehand (create_files=False), the
    second rank first, at its first triangle (odd: its STL records start off a word boundary of the file)."""
    monkeypatch.setenv("DCSG_HOST_EXPAND_PERMILLE", str(permille))
    ctx = ctxs("stress")
    lo, hi = _slab_pair(ctx, ctx.bbox(10.0), 8, 1)
    try:
        rng = np.random.default_rng(permille)
        v0, t0 = _adversarial_positions(lo, rng)
        v1, t1 = _adversarial_positions(hi, rng)
        n0, n1 = len(t0), len(t1)
        total = n0 + n1
        v, t = np.concatenate([v0, v1]), np.concatenate([t0, t1 + np.uint32(len(v0))])
        want_ply, want_stl = encode_ply(v, t), encode_stl(v, t)
        paths = {"ply": str(tmp_path / "s.ply"), "stl": str(tmp_path / "s.stl")}
        for key, want in (("ply", want_ply), ("stl", want_stl)):
            head = len(SOUP_PLY_HEADER.format(V=3 * total, T=total)) if key == "ply" else 84
            with open(paths[key], "wb") as f:               # the headers in place, every row byte wrong
                f.write(want[:head] + b"\xa5" * (len(want) - head))
        hi.project_and_write_files(0, paths["stl"], paths["ply"], first_triangle=n0, total_triangles=total, create_files=False)
        lo.project_and_write_files(0, paths["stl"], paths["ply"], first_triangle=0, total_triangles=total, create_files=False)
        assert_bytes(open(paths["ply"], "rb").read(), want_ply, "sharded PLY")
        assert_bytes(open(paths["stl"], "rb").read(), want_stl, "sharded STL")
    finally:
        lo.free()
        hi.free()


@pytest.mark.gpu
def test_device_widening_of_nans(ctxs):
    """k_format_ply_vertices against the host's widening on every NaN of the set, field by field; prints the device's
    patterns.  Both quiet a signalling NaN and keep its sign and payload."""
    ctx = ctxs("design1")
    carrier = ctx.extract(ctx.bbox(10.0), 5, copy_to_host=False)
    part = Part(carrier)
    try:
        bits = np.concatenate([NANS, SPECIAL]).astype(np.uint32)
        k = -(-len(bits) // 3) * 3
        v = np.resize(bits, k).reshape(-1, 3).view(np.float32)
        t = np.arange(len(v), dtype=np.uint32).reshape(-1, 1).repeat(3, axis=1)
        write_device(carrier, "vertices", v)
        write_device(carrier, "triangles", t)
        mesh = part.set(len(v), len(t))
        dev = np.frombuffer(mesh.format_segments(0)[0].tobytes(), "<u8").reshape(-1, 3, 3)[:, 0].ravel()
        host = np.frombuffer(host_soup_rows(v, t)[0], "<u8").reshape(-1, 3, 3)[:, 0].ravel()
        for f, d, h in zip(v.view(np.uint32).ravel()[:len(NANS)], dev, host):
            print("float %08x -> device %016x, host %016x" % (f, d, h))
        assert np.array_equal(dev, host)
        assert np.array_equal(dev, widen(v).ravel())
    finally:
        part.release()
        carrier.free()


# indexed writer: vertex counts around the chunk rule's steps (chunks = clamp(V / 200000, 1, 12))
INDEXED_COUNTS = [(1, 0), (1, 1), (199999, 5), (200000, 4097), (200001, 2), (399999, 3), (400000, 4), (2399999, 7),
                  (2400000, 1), (2400001, 6)]


@pytest.mark.gpu
def test_indexed_writer(ctxs, tmp_path):
    """write_ply_indexed with and without normals on a Design1 lattice at 2^10 (12 vertex chunks), and on counts-only copies
    of it at the chunk rule's steps: vertex and normal rows are the float bits as they are, NaNs included."""
    ctx = ctxs("design1")
    carrier = ctx.extract(ctx.bbox(10.0), 10, want_normals=True, defer_projection=True, copy_to_host=False)
    assert carrier.num_vertices > 12 * 200000 and carrier.c.d_normals
    rng = np.random.default_rng(7)
    part = Part(carrier)
    path = str(tmp_path / "i.ply")
    try:
        V, T = carrier.num_vertices, carrier.num_triangles
        v = float_bits("mixed", (V, 3), rng).view(np.float32)
        nrm = float_bits("mixed", (V, 3), rng).view(np.float32)
        write_device(carrier, "vertices", v)
        write_device(carrier, "normals", nrm)
        t = read_device(carrier, "triangles", T)
        for normals in (False, True):
            carrier.write_ply_indexed(path, normals=normals)
            assert_bytes(open(path, "rb").read(), encode_ply_indexed(v, t, nrm if normals else None), "indexed, normals=%d" % normals)
        for nv, nt in INDEXED_COUNTS:
            tt = rng.integers(0, nv, size=(nt, 3)).astype(np.uint32)
            if nt:
                write_device(carrier, "triangles", tt)
            mesh = part.set(nv, nt)
            for normals in (False, True):
                mesh.write_ply_indexed(path, normals=normals)
                assert_bytes(open(path, "rb").read(), encode_ply_indexed(v[:nv], tt, nrm[:nv] if normals else None),
                             "indexed V=%d T=%d normals=%d" % (nv, nt, normals))
        xyz, got_n, faces = read_indexed_ply(path)          # the last file parses as the format says
        assert np.array_equal(xyz.view(np.uint32), v[:nv].view(np.uint32)) and np.array_equal(faces, tt)
        assert np.array_equal(got_n.view(np.uint32), nrm[:nv].view(np.uint32))
    finally:
        part.release()
        carrier.free()


def weld_pool(rng):
    """Position patterns (uint32 words) whose repeats the weld must merge and whose near misses it must keep apart."""
    one, two, five = 0x3f800000, 0x40000000, 0x40a00000
    rows = [
        (0x00000000, 0x00000000, 0x00000000), (0x80000000, 0x00000000, 0x00000000),       # +-0 in each coordinate
        (0x00000000, 0x80000000, 0x00000000), (0x00000000, 0x00000000, 0x80000000),
        (0x7fc00001, one, one), (0x7fc00002, one, one), (0xffc00001, one, one),             # NaNs: payload, sign
        (one, 0x7f800001, one), (one, 0x7fa00000, one), (one, one, 0x7fffffff), (one, one, 0x7fc00000),
        (one, two, five), (one ^ 1, two, five), (one, two ^ 1, five), (one, two, five ^ 1),  # one bit apart
        (one, two, five ^ 0x80000000), (one ^ 0x00400000, two, five),
        (two, one, five), (one, one, five), (two, two, five),                                # equal z, other x, y
        (one, two, 0x40400000), (one, two, 0x40800000), (one, two, 0x00000001),              # equal x, y, other z
        (0x00000001, 0x00000001, 0x00000001), (0x7f800000, 0xff800000, 0x7f7fffff),
    ]
    extra = float_bits("mixed", (8, 3), rng)
    return np.concatenate([np.array(rows, np.uint32), extra])


def _first_of_groups(bits):
    """Input index of the first occurrence of each distinct position, in increasing order (= the weld's survivors)."""
    keys = np.ascontiguousarray(bits, np.uint32).reshape(-1, 3).view(np.dtype((np.void, 12))).ravel()
    _, first = np.unique(keys, return_index=True)
    return np.sort(first)


WELD_COUNTS = [1, 2, 255, 256, 257, 4097, (1 << 20) + 3]


@pytest.mark.gpu
def test_weld_on_adversarial_positions(ctxs):
    """dcsg_mesh_weld on positions drawn from a small pool (most repeat): equal words merge, +-0 and NaNs of other payloads
    do not, the same NaN does; the smallest input index of a group keeps its normal; a second weld changes nothing."""
    ctx = ctxs("design2")
    search, lo, hi, grid, thr, _ = export_levels("design2")
    carrier = ctx.extract(ctx.bbox(search), grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=True,
                          want_normals=True, defer_projection=True, copy_to_host=False)
    assert not carrier.c.d_vertex_keys and carrier.c.d_normals
    assert carrier.num_vertices > max(WELD_COUNTS) and carrier.num_triangles > max(WELD_COUNTS)
    rng = np.random.default_rng(5)
    part = Part(carrier)
    try:
        for V in WELD_COUNTS:
            pool = weld_pool(rng)
            pos = pool[rng.integers(0, len(pool), size=V)]
            if V >= len(pool):
                pos[:len(pool)] = pool                      # every pattern at least once
            v = pos.view(np.float32)
            i = np.arange(V, dtype=np.uint32)
            nrm = np.stack([i, i | 0x40000000, ~i], axis=1).astype(np.uint32).view(np.float32)     # one of its own per vertex
            T = max(1, V // 2)
            t = rng.integers(0, V, size=(T, 3)).astype(np.uint32)
            write_device(carrier, "vertices", v)
            write_device(carrier, "normals", nrm)
            write_device(carrier, "triangles", t)
            mesh = part.set(V, T)
            want_v, want_t = numpy_weld(v, t)
            keep = _first_of_groups(pos)
            assert np.array_equal(want_v.view(np.uint32), pos[keep])
            for round_ in (1, 2):
                mesh.weld()
                m = mesh.num_vertices
                got_v, got_n, got_t = read_device(carrier, "vertices", m), read_device(carrier, "normals", m), \
                    read_device(carrier, "triangles", T)
                assert m == len(want_v), (V, round_, m, len(want_v))
                assert np.array_equal(got_v.view(np.uint32), want_v.view(np.uint32)), (V, round_)
                assert np.array_equal(got_t, want_t), (V, round_)
                assert np.array_equal(got_n.view(np.uint32), nrm[keep].view(np.uint32)), (V, round_)
            print("weld V=%d: %d distinct positions" % (V, len(want_v)))
    finally:
        part.release()
        carrier.free()
