"""Python host side of the B200 export path: ctypes binding of libdcsg.so (include/dcsg.h).

The reference's host is C++ (Evaluator, OnExportInner); the C ABI is the drop-in boundary, and this
module is the thin Python front used by the CLI, the tests and bench.py.  ``Evaluator`` mirrors the
reference class of the same name (master/Evaluator.h:20-57): ``build``, ``eval_sdf_at_points``,
``eval_normal_at_points``, ``setArbitraryData``.  There is no CPU path: if libdcsg.so is missing or no
CUDA device is present the calls raise.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdcsg.so")
PLUGIN_DIR = os.path.join(HERE, "plugin")

STAGES = ("lattice", "classify", "emit", "project", "copy")

_f32p = ctypes.POINTER(ctypes.c_float)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_u32p = ctypes.POINTER(ctypes.c_uint32)
_u64p = ctypes.POINTER(ctypes.c_uint64)


class DcsgError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("libdcsg error %d: %s" % (code, message))
        self.code = code


class ExtractCfg(ctypes.Structure):
    _fields_ = [("box", ctypes.c_float * 6), ("grid_level", ctypes.c_int), ("min_level", ctypes.c_int),
                ("max_level", ctypes.c_int), ("complex_threshold", ctypes.c_float), ("gd_steps", ctypes.c_int),
                ("want_normals", ctypes.c_int), ("slab_z0", ctypes.c_int), ("slab_z1", ctypes.c_int),
                ("copy_to_host", ctypes.c_int), ("no_cull", ctypes.c_int), ("dense", ctypes.c_int),
                ("retopologize", ctypes.c_int), ("defer_projection", ctypes.c_int)]


class MeshStruct(ctypes.Structure):
    _fields_ = [("num_vertices", ctypes.c_uint64), ("num_triangles", ctypes.c_uint64), ("num_cells", ctypes.c_uint64),
                ("d_vertices", ctypes.c_void_p), ("d_normals", ctypes.c_void_p), ("d_vertex_keys", ctypes.c_void_p),
                ("d_triangles", ctypes.c_void_p), ("d_cell_ids", ctypes.c_void_p), ("d_cell_masks", ctypes.c_void_p),
                ("h_vertices", _f32p), ("h_normals", _f32p), ("h_vertex_keys", _u64p), ("h_triangles", _u32p),
                ("h_cell_ids", _u64p), ("h_cell_masks", _u8p),
                ("lattice_samples", ctypes.c_uint64), ("stage_ms", ctypes.c_float * len(STAGES)),
                ("owned_vertices", ctypes.c_uint64), ("halo_vertices", ctypes.c_uint64), ("reserved", ctypes.c_void_p)]


class ExportReport(ctypes.Structure):
    _fields_ = [("box", ctypes.c_float * 6), ("num_vertices", ctypes.c_uint64), ("num_triangles", ctypes.c_uint64),
                ("num_cells", ctypes.c_uint64), ("bbox_ms", ctypes.c_float), ("extract_ms", ctypes.c_float * len(STAGES)),
                ("format_ms", ctypes.c_float), ("write_ms", ctypes.c_float), ("total_ms", ctypes.c_float)]


class ShardInfo(ctypes.Structure):
    _fields_ = [("rank", ctypes.c_int), ("world", ctypes.c_int), ("slab_z0", ctypes.c_int), ("slab_z1", ctypes.c_int),
                ("first_vertex", ctypes.c_uint64), ("first_triangle", ctypes.c_uint64), ("total_vertices", ctypes.c_uint64),
                ("total_triangles", ctypes.c_uint64), ("total_cells", ctypes.c_uint64)]


PROGRESS_STATES = ("IDLE", "ESTIMATING_BOUNDING_BOX", "PERFORMING_CMS", "RETOPOLOGIZING", "GRADIENT_DESCENT", "WRITING_STL",
                   "WRITING_PLY", "COMPLETE")                   # dcsg.h DCSG_PROGRESS_*, reference DesignCSG.cpp:603-614
PROGRESS_FN = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64)

PLY_NORMALS = 1                                                 # dcsg.h DCSG_PLY_NORMALS
EXPORT_OUTWARD = 1                                              # dcsg.h DCSG_EXPORT_OUTWARD

_lib = None


def load_library():
    """Load libdcsg.so from the package directory.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError("%s is missing; build it with `python -m designcsg_b200.build` "
                                "(the export path has no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, cp, sz, ci = ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int
    lib.dcsg_version.restype = cp
    lib.dcsg_create.argtypes = [ci, ctypes.POINTER(vp)]
    lib.dcsg_destroy.argtypes = [vp]
    lib.dcsg_destroy.restype = None
    lib.dcsg_last_error.argtypes = [vp]
    lib.dcsg_last_error.restype = cp
    lib.dcsg_set_stream.argtypes = [vp, vp]
    lib.dcsg_build.argtypes = [vp, cp, cp, sz]
    lib.dcsg_compile_scene.argtypes = [cp, cp, cp, sz]
    lib.dcsg_scene_source.argtypes = [cp, cp, sz, ctypes.POINTER(sz)]
    lib.dcsg_set_arbitrary_data.argtypes = [vp, _f32p, sz]
    lib.dcsg_eval_sdf.argtypes = [vp, _f32p, sz, _f32p]
    lib.dcsg_eval_normal.argtypes = [vp, _f32p, sz, _f32p]
    lib.dcsg_eval_sdf_device.argtypes = [vp, vp, sz, vp]
    lib.dcsg_eval_normal_device.argtypes = [vp, vp, sz, vp]
    lib.dcsg_bbox.argtypes = [vp, ctypes.c_float, _f32p]
    lib.dcsg_preview.argtypes = [vp, _f32p, _f32p, _f32p, _f32p, _u8p]
    lib.dcsg_sample_lattice.argtypes = [vp, _f32p, ci, ci, ci, _f32p]
    lib.dcsg_lattice_device_ptr.argtypes = [vp]
    lib.dcsg_lattice_device_ptr.restype = vp
    lib.dcsg_extract.argtypes = [vp, ctypes.POINTER(ExtractCfg), ctypes.POINTER(MeshStruct)]
    lib.dcsg_mesh_free.argtypes = [vp, ctypes.POINTER(MeshStruct)]
    lib.dcsg_mesh_free.restype = None
    lib.dcsg_mesh_soup.argtypes = [vp, ctypes.POINTER(MeshStruct), _f32p]
    lib.dcsg_write_stl.argtypes = [vp, ctypes.POINTER(MeshStruct), cp]
    lib.dcsg_write_ply.argtypes = [vp, ctypes.POINTER(MeshStruct), cp]
    lib.dcsg_format_stl.argtypes = [vp, ctypes.POINTER(MeshStruct), _u8p, sz, ctypes.POINTER(sz)]
    lib.dcsg_format_ply.argtypes = [vp, ctypes.POINTER(MeshStruct), _u8p, sz, ctypes.POINTER(sz)]
    lib.dcsg_export.argtypes = [vp, cp, ci, cp, cp, ctypes.POINTER(ExportReport)]
    lib.dcsg_fp32_peak.argtypes = [vp, ci, ctypes.POINTER(ctypes.c_double)]
    lib.dcsg_set_progress_callback.argtypes = [vp, PROGRESS_FN, vp]
    lib.dcsg_project_stats.argtypes = [vp, _u64p, _u64p]
    lib.dcsg_format_stl_view.argtypes = [vp, ctypes.POINTER(MeshStruct), ctypes.POINTER(_u8p), ctypes.POINTER(sz)]
    lib.dcsg_format_ply_view.argtypes = [vp, ctypes.POINTER(MeshStruct), ctypes.POINTER(_u8p), ctypes.POINTER(sz)]
    lib.dcsg_launch_count.restype = ctypes.c_ulonglong
    lib.dcsg_format_segments.argtypes = [vp, ctypes.POINTER(MeshStruct), ctypes.c_uint64, ctypes.POINTER(_u8p), ctypes.POINTER(_u8p),
                                         ctypes.POINTER(_u8p)]
    lib.dcsg_project_and_format_segments.argtypes = [vp, ctypes.POINTER(MeshStruct), ci, ctypes.c_uint64, ctypes.POINTER(_u8p),
                                                     ctypes.POINTER(_u8p), ctypes.POINTER(_u8p)]
    lib.dcsg_project_and_write_files.argtypes = [vp, ctypes.POINTER(MeshStruct), ci, ctypes.c_uint64, ctypes.c_uint64, ci, cp, cp]
    lib.dcsg_file_header.argtypes = [ci, ctypes.c_uint64, _u8p, sz, ctypes.POINTER(sz)]
    lib.dcsg_ply_face_rows.argtypes = [ctypes.c_uint64, ctypes.c_uint64, _u8p, sz]
    lib.dcsg_soup_rows.argtypes = [_f32p, ctypes.c_uint64, _u8p, _u8p]
    lib.dcsg_comm_unique_id.argtypes = [_u8p]
    lib.dcsg_comm_create.argtypes = [vp, _u8p, ci, ci, ctypes.POINTER(vp)]
    lib.dcsg_comm_destroy.argtypes = [vp]
    lib.dcsg_comm_destroy.restype = None
    lib.dcsg_comm_rank.argtypes = [vp]
    lib.dcsg_comm_world.argtypes = [vp]
    lib.dcsg_comm_barrier.argtypes = [vp]
    lib.dcsg_bbox_sharded.argtypes = [vp, vp, ctypes.c_float, _f32p]
    lib.dcsg_extract_sharded.argtypes = [vp, vp, ctypes.POINTER(ExtractCfg), ci, ctypes.POINTER(MeshStruct), ctypes.POINTER(MeshStruct),
                                         ctypes.POINTER(ShardInfo)]
    lib.dcsg_export_sharded.argtypes = [vp, vp, cp, ci, cp, cp, ctypes.POINTER(ExportReport)]
    lib.dcsg_project.argtypes = [vp, ctypes.POINTER(MeshStruct), ci, ci]
    lib.dcsg_plan_slabs.argtypes = [vp, _f32p, ci, ci, ci, ctypes.POINTER(ci)]
    lib.dcsg_mesh_weld.argtypes = [vp, ctypes.POINTER(MeshStruct)]
    lib.dcsg_write_ply_indexed.argtypes = [vp, ctypes.POINTER(MeshStruct), ci, cp]
    lib.dcsg_export_indexed.argtypes = [vp, cp, ci, ci, cp, ctypes.POINTER(ExportReport)]
    lib.dcsg_export_sharded_indexed.argtypes = [vp, vp, cp, ci, ci, cp, ctypes.POINTER(ExportReport)]
    lib.dcsg_mesh_orient.argtypes = [vp, ctypes.POINTER(MeshStruct)]
    lib.dcsg_set_export_flags.argtypes = [vp, ci]
    _lib = lib
    return lib


def file_header(ply, total_triangles):
    """Header bytes of the PLY (happly) or STL file for a mesh of total_triangles (dcsg_file_header)."""
    lib = load_library()
    need = ctypes.c_size_t(0)
    lib.dcsg_file_header(int(ply), total_triangles, None, 0, ctypes.byref(need))
    buf = np.empty(need.value, dtype=np.uint8)
    lib.dcsg_file_header(int(ply), total_triangles, buf.ctypes.data_as(_u8p), buf.size, ctypes.byref(need))
    return buf


def ply_face_rows(first_triangle, num_triangles):
    """The 13-byte face rows of the soup PLY for a range of triangles (dcsg_ply_face_rows; host only)."""
    lib = load_library()
    buf = np.empty(13 * num_triangles, dtype=np.uint8)
    rc = lib.dcsg_ply_face_rows(first_triangle, num_triangles, buf.ctypes.data_as(_u8p), buf.size)
    if rc != 0:
        raise DcsgError(rc, "dcsg_ply_face_rows(%d, %d)" % (first_triangle, num_triangles))
    return buf


def soup_rows(soup):
    """PLY vertex rows and STL records of a (T,3,3) float32 soup, expanded on the host (dcsg_soup_rows)."""
    lib = load_library()
    t = np.ascontiguousarray(soup, dtype=np.float32).reshape(-1, 9)
    ply, stl = np.empty(72 * len(t), dtype=np.uint8), np.empty(50 * len(t), dtype=np.uint8)
    rc = lib.dcsg_soup_rows(t.ctypes.data_as(_f32p), len(t), ply.ctypes.data_as(_u8p), stl.ctypes.data_as(_u8p))
    if rc != 0:
        raise DcsgError(rc, "dcsg_soup_rows")
    return ply, stl


def launch_count():
    """Kernels launched by libdcsg in this process so far."""
    return int(load_library().dcsg_launch_count())


def compile_design(design_path, out_dir, env=None):
    """Run a design script against the plug-in modules, as the reference's "Run" does
    (master/DesignCSG.cpp:531-568: copy to compiled.py, run python in the working directory).
    The scene files (scene.cu, scene.txt, buildprocedure.txt, arbitrary_data.hex, exportConfig.txt)
    land in out_dir, which is returned."""
    os.makedirs(out_dir, exist_ok=True)
    run_env = dict(os.environ)
    run_env["PYTHONPATH"] = PLUGIN_DIR + os.pathsep + run_env.get("PYTHONPATH", "")
    if env:
        run_env.update(env)
    with open(design_path) as src, open(os.path.join(out_dir, "compiled.py"), "w") as dst:
        dst.write(src.read())
    proc = subprocess.run([sys.executable, "compiled.py"], cwd=out_dir, env=run_env, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True)
    with open(os.path.join(out_dir, "log.txt"), "w") as f:
        f.write(proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError("design script failed:\n" + proc.stdout)
    return out_dir


def compile_scene_offline(scene_dir, cubin_path=None):
    """NVRTC-compile a scene directory for sm_100a without touching a GPU; returns the compiler log."""
    lib = load_library()
    log = ctypes.create_string_buffer(1 << 20)
    rc = lib.dcsg_compile_scene(scene_dir.encode(), cubin_path.encode() if cubin_path else None, log, len(log))
    if rc != 0:
        raise DcsgError(rc, log.value.decode(errors="replace"))
    return log.value.decode(errors="replace")


def scene_source(scene_dir):
    lib = load_library()
    need = ctypes.c_size_t(0)
    lib.dcsg_scene_source(scene_dir.encode(), None, 0, ctypes.byref(need))
    buf = ctypes.create_string_buffer(need.value + 1)
    rc = lib.dcsg_scene_source(scene_dir.encode(), buf, len(buf), ctypes.byref(need))
    if rc != 0:
        raise DcsgError(rc, "dcsg_scene_source failed")
    return buf.value.decode()


class DevicePtr:
    """Zero-copy view of a library-owned device array (``__cuda_array_interface__``), e.g. for
    ``torch.as_tensor(mesh.device('vertices'), device='cuda')``."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr or 0), False),
                                         "version": 2, "strides": None}
        self._owner = owner


class Mesh:
    """Result of Context.extract: indexed mesh in canonical order (see include/dcsg.h)."""

    def __init__(self, ctx):
        self._ctx = ctx
        self.c = MeshStruct()

    num_vertices = property(lambda self: int(self.c.num_vertices))
    num_triangles = property(lambda self: int(self.c.num_triangles))
    num_cells = property(lambda self: int(self.c.num_cells))
    owned_vertices = property(lambda self: int(self.c.owned_vertices))      # z-slabs: vertices without the halo plane's copies
    halo_vertices = property(lambda self: int(self.c.halo_vertices))

    @property
    def stage_ms(self):
        return {name: float(self.c.stage_ms[i]) for i, name in enumerate(STAGES)}

    def _host(self, ptr, count, dtype, cols=None):
        if count == 0 and self.c.h_vertices:        # an empty array of a mesh that WAS copied (e.g. a slab without vertices)
            return np.empty((0, cols) if cols else (0,), dtype=dtype)
        if not ptr:
            raise ValueError("mesh was extracted without copy_to_host")
        a = np.ctypeslib.as_array(ptr, shape=(max(count, 1),))[:count].view(dtype)
        return a.reshape(-1, cols).copy() if cols else a.copy()

    def vertices(self):
        return self._host(self.c.h_vertices, self.num_vertices * 3, np.float32, 3)

    def normals(self):
        return self._host(self.c.h_normals, self.num_vertices * 3, np.float32, 3)

    def vertex_keys(self):
        return self._host(self.c.h_vertex_keys, self.num_vertices, np.uint64)

    def triangles(self):
        return self._host(self.c.h_triangles, self.num_triangles * 3, np.uint32, 3)

    def cell_ids(self):
        return self._host(self.c.h_cell_ids, self.num_cells, np.uint64)

    def cell_masks(self):
        return self._host(self.c.h_cell_masks, self.num_cells, np.uint8)

    def device(self, name):
        spec = {"vertices": (self.c.d_vertices, (self.num_vertices, 3), "<f4"),
                "normals": (self.c.d_normals, (self.num_vertices, 3), "<f4"),
                # 64/32-bit ids are exposed as signed (torch has no arithmetic on unsigned 32/64); they fit
                "vertex_keys": (self.c.d_vertex_keys, (self.num_vertices,), "<i8"),
                "triangles": (self.c.d_triangles, (self.num_triangles, 3), "<i4"),
                "cell_ids": (self.c.d_cell_ids, (self.num_cells,), "<i8"),
                "cell_masks": (self.c.d_cell_masks, (self.num_cells,), "|u1")}[name]
        return DevicePtr(spec[0], spec[1], spec[2], self)

    def soup(self):
        """(T,3,3) float32 triangle soup -- the reference's in-memory mesh (vector<Triangle3f>)."""
        out = np.empty((self.num_triangles, 3, 3), dtype=np.float32)
        self._ctx._check(self._ctx.lib.dcsg_mesh_soup(self._ctx.h, ctypes.byref(self.c), out.ctypes.data_as(_f32p)))
        return out

    def write_stl(self, path):
        self._ctx._check(self._ctx.lib.dcsg_write_stl(self._ctx.h, ctypes.byref(self.c), path.encode()))

    def write_ply(self, path):
        self._ctx._check(self._ctx.lib.dcsg_write_ply(self._ctx.h, ctypes.byref(self.c), path.encode()))

    def weld(self):
        """dcsg_mesh_weld: merge vertices with bit-identical positions (numbered by first occurrence), renumber the triangles.
        A lattice mesh comes back unchanged.  The host arrays are refreshed when the mesh was copied to the host."""
        self._ctx._check(self._ctx.lib.dcsg_mesh_weld(self._ctx.h, ctypes.byref(self.c)))

    def orient(self):
        """dcsg_mesh_orient: swap corners 1 and 2 of the inward-facing triangles so that every triangle faces out of the solid.
        Vertices, cells and triangle order stay; the host arrays are refreshed when the mesh was copied to the host; a second
        call changes nothing.  The STL writers then list the corners A, C, B (the files are no longer the reference's bytes)."""
        self._ctx._check(self._ctx.lib.dcsg_mesh_orient(self._ctx.h, ctypes.byref(self.c)))

    def write_ply_indexed(self, path, normals=False):
        """dcsg_write_ply_indexed: binary PLY with shared float vertices (and the mesh's normals) -- not the reference's format."""
        self._ctx._check(self._ctx.lib.dcsg_write_ply_indexed(self._ctx.h, ctypes.byref(self.c), PLY_NORMALS if normals else 0,
                                                              path.encode()))

    def _format(self, fn):
        need = ctypes.c_size_t(0)
        self._ctx._check(fn(self._ctx.h, ctypes.byref(self.c), None, 0, ctypes.byref(need)))
        buf = np.empty(need.value, dtype=np.uint8)
        self._ctx._check(fn(self._ctx.h, ctypes.byref(self.c), buf.ctypes.data_as(_u8p), buf.size, ctypes.byref(need)))
        return buf

    def format_stl(self):
        return self._format(self._ctx.lib.dcsg_format_stl)

    def _view(self, fn):
        ptr, size = _u8p(), ctypes.c_size_t(0)
        self._ctx._check(fn(self._ctx.h, ctypes.byref(self.c), ctypes.byref(ptr), ctypes.byref(size)))
        return np.ctypeslib.as_array(ptr, shape=(size.value,))      # pinned, library-owned, no copy

    def format_stl_view(self):
        return self._view(self._ctx.lib.dcsg_format_stl_view)

    def format_ply_view(self):
        return self._view(self._ctx.lib.dcsg_format_ply_view)

    def format_ply(self):
        return self._format(self._ctx.lib.dcsg_format_ply)

    def project_and_format_segments(self, gd_steps, first_triangle):
        """dcsg_project_and_format_segments: projection pipelined with formatting and the device -> host copies (mesh from
        extract(..., defer_projection=True)); returns the same three views as format_segments."""
        a, b, c = _u8p(), _u8p(), _u8p()
        self._ctx._check(self._ctx.lib.dcsg_project_and_format_segments(self._ctx.h, ctypes.byref(self.c), gd_steps, first_triangle,
                                                                        ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        n = self.num_triangles
        view = lambda p, size: np.ctypeslib.as_array(p, shape=(max(size, 1),))[:size]
        return view(a, n * 72), view(b, n * 13), view(c, n * 50)

    def project_and_write_files(self, gd_steps, stl_path=None, ply_path=None, first_triangle=0, total_triangles=None, create_files=True):
        """dcsg_project_and_write_files: projection, formatting, D2H and file writes as one pipeline."""
        total = self.num_triangles if total_triangles is None else total_triangles
        self._ctx._check(self._ctx.lib.dcsg_project_and_write_files(
            self._ctx.h, ctypes.byref(self.c), gd_steps, first_triangle, total, int(create_files),
            stl_path.encode() if stl_path else None, ply_path.encode() if ply_path else None))

    def format_segments(self, first_triangle):
        """This rank's byte ranges of the files (dcsg_format_segments): PLY vertex rows, PLY face rows, STL records as
        zero-copy views of the library's pinned buffer."""
        a, b, c = _u8p(), _u8p(), _u8p()
        self._ctx._check(self._ctx.lib.dcsg_format_segments(self._ctx.h, ctypes.byref(self.c), first_triangle, ctypes.byref(a),
                                                            ctypes.byref(b), ctypes.byref(c)))
        n = self.num_triangles
        view = lambda p, size: np.ctypeslib.as_array(p, shape=(max(size, 1),))[:size]
        return view(a, n * 72), view(b, n * 13), view(c, n * 50)

    def free(self):
        if self._ctx is not None and self._ctx.h:
            self._ctx.lib.dcsg_mesh_free(self._ctx.h, ctypes.byref(self.c))
        self._ctx = None


class Context:
    """One CUDA device + one compiled scene (dcsg_ctx)."""

    def __init__(self, device=0):
        self.lib = load_library()
        self.h = ctypes.c_void_p()
        rc = self.lib.dcsg_create(device, ctypes.byref(self.h))
        if rc != 0:
            raise DcsgError(rc, "dcsg_create(%d) failed: no usable CUDA device (the export path has no CPU fallback)" % device)
        self.device = device
        self.build_log = ""
        self._export_flags = 0

    def _check(self, rc):
        if rc != 0:
            raise DcsgError(rc, self.lib.dcsg_last_error(self.h).decode(errors="replace"))

    def close(self):
        if self.h:
            self.lib.dcsg_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_progress_callback(self, fn):
        """dcsg_set_progress_callback; fn = an api.PROGRESS_FN instance (kept alive here) or None."""
        self._progress = fn                 # the C side keeps the raw pointer: keep the ctypes thunk alive
        self._check(self.lib.dcsg_set_progress_callback(self.h, fn if fn is not None else ctypes.cast(None, PROGRESS_FN), None))

    def set_stream(self, cuda_stream):
        self._check(self.lib.dcsg_set_stream(self.h, ctypes.c_void_p(cuda_stream)))

    def build(self, scene_dir):
        log = ctypes.create_string_buffer(1 << 20)
        rc = self.lib.dcsg_build(self.h, scene_dir.encode(), log, len(log))
        self.build_log = log.value.decode(errors="replace")
        if rc != 0:
            raise DcsgError(rc, self.build_log or self.lib.dcsg_last_error(self.h).decode(errors="replace"))
        return self.build_log

    def set_arbitrary_data(self, data):
        d = np.ascontiguousarray(data, dtype=np.float32)
        self._check(self.lib.dcsg_set_arbitrary_data(self.h, d.ctypes.data_as(_f32p), d.size))

    def eval_sdf(self, points):
        p = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
        out = np.empty(len(p), dtype=np.float32)
        self._check(self.lib.dcsg_eval_sdf(self.h, p.ctypes.data_as(_f32p), len(p), out.ctypes.data_as(_f32p)))
        return out

    def eval_normal(self, points):
        p = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
        out = np.empty((len(p), 3), dtype=np.float32)
        self._check(self.lib.dcsg_eval_normal(self.h, p.ctypes.data_as(_f32p), len(p), out.ctypes.data_as(_f32p)))
        return out

    def bbox(self, search_diameter):
        box = np.zeros(6, dtype=np.float32)
        self._check(self.lib.dcsg_bbox(self.h, ctypes.c_float(search_diameter), box.ctypes.data_as(_f32p)))
        return box

    def preview(self, campos, right, up, forward):
        """dcsg_preview: the reference's 640x480 ray-marched view (kernel k1) as a (480, 640, 3) uint8 image."""
        vecs = [np.ascontiguousarray(v, dtype=np.float32).reshape(3) for v in (campos, right, up, forward)]
        out = np.empty((480, 640, 3), dtype=np.uint8)
        self._check(self.lib.dcsg_preview(self.h, *[v.ctypes.data_as(_f32p) for v in vecs], out.ctypes.data_as(_u8p)))
        return out

    def sample_lattice(self, box6, grid_level, z_begin=0, z_end=0, to_host=True):
        b = np.ascontiguousarray(box6, dtype=np.float32)
        n = (1 << grid_level) + 1
        if z_begin == 0 and z_end == 0:
            z_end = n
        out = np.empty((z_end - z_begin, n, n), dtype=np.float32) if to_host else None
        self._check(self.lib.dcsg_sample_lattice(self.h, b.ctypes.data_as(_f32p), grid_level, z_begin, z_end,
                                                 out.ctypes.data_as(_f32p) if to_host else None))
        return out

    def extract(self, box6, grid_level, gd_steps=0, want_normals=False, slab=(0, 0), copy_to_host=True,
                no_cull=False, mesh=None, min_level=None, max_level=None, complex_threshold=float(np.pi / 4),
                dense=False, retopologize=False, defer_projection=False):
        """dcsg_extract.  min_level / max_level default to grid_level (the uniform lattice: indexed mesh); any other
        min <= max <= grid runs the reference's adaptive octree walk and returns a triangle soup (no vertex keys)."""
        cfg = ExtractCfg()
        for i in range(6):
            cfg.box[i] = float(box6[i])
        cfg.grid_level = grid_level
        cfg.min_level = grid_level if min_level is None else min_level
        cfg.max_level = grid_level if max_level is None else max_level
        cfg.complex_threshold = complex_threshold
        cfg.gd_steps = gd_steps
        cfg.want_normals = int(want_normals)
        cfg.slab_z0, cfg.slab_z1 = slab
        cfg.copy_to_host = int(copy_to_host)
        cfg.no_cull = int(no_cull)
        cfg.dense = int(dense)
        cfg.retopologize = int(retopologize)
        cfg.defer_projection = int(defer_projection)
        mesh = mesh or Mesh(self)
        self._check(self.lib.dcsg_extract(self.h, ctypes.byref(cfg), ctypes.byref(mesh.c)))
        return mesh

    def project(self, mesh, gd_steps, want_normals=False):
        """dcsg_project: gradient-descent projection of a mesh extracted with defer_projection; asynchronous on the
        context's stream."""
        self._check(self.lib.dcsg_project(self.h, ctypes.byref(mesh.c), gd_steps, int(want_normals)))

    def plan_slabs(self, box6, grid_level, world, granularity=8):
        """Balanced z-slab boundaries for `world` ranks from the last bbox() call's surface histogram (dcsg_plan_slabs)."""
        b = np.ascontiguousarray(box6, dtype=np.float32)
        bounds = (ctypes.c_int * (world + 1))()
        self._check(self.lib.dcsg_plan_slabs(self.h, b.ctypes.data_as(_f32p), grid_level, world, granularity, bounds))
        return [int(v) for v in bounds]

    def project_stats(self):
        """(tap rounds, rounds repeated through the exact copy) executed by the projection kernel since the last call."""
        a, b = ctypes.c_uint64(0), ctypes.c_uint64(0)
        self._check(self.lib.dcsg_project_stats(self.h, ctypes.byref(a), ctypes.byref(b)))
        return int(a.value), int(b.value)

    def fp32_peak_tflops(self, mode=0):
        """Measured non-tensor FP32 rate: mode 0 = FFMA (2 FLOP/instr), mode 1 = FMUL+FADD (1 FLOP/instr)."""
        v = ctypes.c_double(0.0)
        self._check(self.lib.dcsg_fp32_peak(self.h, mode, ctypes.byref(v)))
        return v.value

    def set_export_flags(self, flags):
        """dcsg_set_export_flags: options of the dcsg_export* calls on this context (EXPORT_OUTWARD)."""
        self._check(self.lib.dcsg_set_export_flags(self.h, flags))
        self._export_flags = flags

    def _with_export_flags(self, outward, call):
        """Run call() with DCSG_EXPORT_OUTWARD set or cleared as asked; the context's flags are restored afterwards."""
        before = self._export_flags
        wanted = (before | EXPORT_OUTWARD) if outward else (before & ~EXPORT_OUTWARD)
        if wanted == before:
            return call()
        self.set_export_flags(wanted)
        try:
            return call()
        finally:
            self.set_export_flags(before)

    def export(self, scene_dir, grid_level=0, stl_path=None, ply_path=None, outward=False):
        """dcsg_export; outward=True orients the mesh before the files are written (not the reference's bytes then)."""
        rep = ExportReport()
        self._with_export_flags(outward, lambda: self._check(self.lib.dcsg_export(
            self.h, scene_dir.encode(), grid_level, stl_path.encode() if stl_path else None, ply_path.encode() if ply_path else None,
            ctypes.byref(rep))))
        return rep

    def export_indexed(self, scene_dir, grid_level=0, ply_path=None, normals=False, outward=False):
        """dcsg_export_indexed: the export pipeline writing the indexed PLY (adaptive meshes welded before the projection);
        outward=True orients the mesh first."""
        rep = ExportReport()
        self._with_export_flags(outward, lambda: self._check(self.lib.dcsg_export_indexed(
            self.h, scene_dir.encode(), grid_level, PLY_NORMALS if normals else 0, ply_path.encode(), ctypes.byref(rep))))
        return rep


def comm_unique_id():
    """dcsg_comm_unique_id: 128 bytes rank 0 creates and hands to the other ranks (any side channel)."""
    lib = load_library()
    buf = np.zeros(128, dtype=np.uint8)
    rc = lib.dcsg_comm_unique_id(buf.ctypes.data_as(_u8p))
    if rc != 0:
        raise DcsgError(rc, "dcsg_comm_unique_id failed (NCCL not loadable?)")
    return buf


class Comm:
    """dcsg_comm: this rank's end of a multi-GPU export (one process per GPU).  Everything collective happens inside
    libdcsg -- NCCL for the small collectives, peer stores for the mesh; Python only hands over the 128-byte id."""

    def __init__(self, ctx, unique_id, rank, world):
        self.ctx, self.rank, self.world = ctx, rank, world
        self.h = ctypes.c_void_p()
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        assert uid.size == 128
        ctx._check(ctx.lib.dcsg_comm_create(ctx.h, uid.ctypes.data_as(_u8p), rank, world, ctypes.byref(self.h)))

    def close(self):
        if self.h:
            self.ctx.lib.dcsg_comm_destroy(self.h)
            self.h = ctypes.c_void_p()

    def barrier(self):
        self.ctx._check(self.ctx.lib.dcsg_comm_barrier(self.h))

    def bbox(self, search_diameter):
        box = np.zeros(6, dtype=np.float32)
        self.ctx._check(self.ctx.lib.dcsg_bbox_sharded(self.ctx.h, self.h, ctypes.c_float(search_diameter), box.ctypes.data_as(_f32p)))
        return box

    def extract(self, box6, grid_level, gd_steps=0, want_normals=False, gather_to=0, mesh=None, defer_projection=False):
        """dcsg_extract_sharded -> (this rank's slab mesh, whole mesh [borrowed device arrays on rank gather_to, counts
        everywhere], ShardInfo)."""
        cfg = ExtractCfg()
        for i in range(6):
            cfg.box[i] = float(box6[i])
        cfg.grid_level = cfg.min_level = cfg.max_level = grid_level
        cfg.gd_steps = gd_steps
        cfg.want_normals = int(want_normals)
        cfg.defer_projection = int(defer_projection)
        mesh = mesh or Mesh(self.ctx)
        whole = Mesh(self.ctx)
        info = ShardInfo()
        self.ctx._check(self.ctx.lib.dcsg_extract_sharded(self.ctx.h, self.h, ctypes.byref(cfg), gather_to, ctypes.byref(mesh.c),
                                                          ctypes.byref(whole.c), ctypes.byref(info)))
        whole._borrowed = True
        return mesh, whole, info

    def export(self, scene_dir, grid_level=0, stl_path=None, ply_path=None, outward=False):
        """dcsg_export_sharded; outward=True orients every rank's slab before the files are written."""
        rep = ExportReport()
        self.ctx._with_export_flags(outward, lambda: self.ctx._check(self.ctx.lib.dcsg_export_sharded(
            self.ctx.h, self.h, scene_dir.encode(), grid_level, stl_path.encode() if stl_path else None,
            ply_path.encode() if ply_path else None, ctypes.byref(rep))))
        return rep

    def export_indexed(self, scene_dir, grid_level, ply_path, normals=False, outward=False):
        """dcsg_export_sharded_indexed: the indexed PLY over all ranks; uniform lattice (grid_level > 0) only."""
        rep = ExportReport()
        self.ctx._with_export_flags(outward, lambda: self.ctx._check(self.ctx.lib.dcsg_export_sharded_indexed(
            self.ctx.h, self.h, scene_dir.encode(), grid_level, PLY_NORMALS if normals else 0, ply_path.encode(), ctypes.byref(rep))))
        return rep


class Evaluator:
    """Same surface as the reference's Evaluator (master/Evaluator.h:20-57), backed by libdcsg."""

    def __init__(self, device=0, scene_dir="."):
        self.ctx = Context(device)
        self.scene_dir = scene_dir

    def build(self, scene_dir=None):
        """Returns (0, "Success!") or (-1, build log), like the reference (Evaluator.cpp:45-112)."""
        try:
            log = self.ctx.build(scene_dir or self.scene_dir)
            return 0, log or "Success!"
        except DcsgError as e:
            if e.code == -1:
                return -1, self.ctx.build_log
            raise

    def eval_sdf_at_points(self, points):
        return self.ctx.eval_sdf(points)

    def eval_normal_at_points(self, points):
        return self.ctx.eval_normal(points)

    def setArbitraryData(self, data, items=None):
        self.ctx.set_arbitrary_data(data if items is None else data[:items])
