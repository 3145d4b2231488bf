/* dcsg.h -- C ABI of libdcsg.so, the B200-native (sm_100a) export path of DesignCSG.
 *
 * Drop-in boundary for the reference's C++ host side of the export path.  Every entry point names the
 * reference interface it replaces (paths relative to /root/reference):
 *
 *   dcsg_create / dcsg_destroy      Evaluator::Evaluator (master/Evaluator.cpp:14-40) + the OpenCL device /
 *                                   context / queue set-up it borrows from the preview pane
 *                                   (master/DrawPane.cpp:29-121, master/Utils.cpp:27-46)
 *   dcsg_build                      BasicDrawPane::loadScene's parsing of scene.txt / buildprocedure.txt
 *                                   (master/DrawPane.cpp:243-371) + Evaluator::build -> clBuildProgram of
 *                                   k2.cl ++ scene.cl (master/Evaluator.cpp:45-112, master/Utils.cpp:48-103)
 *                                   + updateExportArbitraryData (master/DesignCSG.cpp:507-529)
 *   dcsg_set_arbitrary_data         Evaluator::setArbitraryData (master/Evaluator.cpp:213-225)
 *   dcsg_eval_sdf / dcsg_eval_normal  Evaluator::eval_sdf_at_points / eval_normal_at_points
 *                                   (master/Evaluator.cpp:117-165, :167-211) = kernel k2 (master/k2.cl:234-280)
 *   dcsg_bbox                       the 256^3 bounding-box search of MyFrame::OnExportInner
 *                                   (master/DesignCSG.cpp:668-712)
 *   dcsg_sample_lattice             ISV3D64 (master/ISV.hpp:15-108): the lattice the mesher samples
 *   dcsg_extract                    cms::Mesh::getSurface + cms::retopologize (identity in the uniform
 *                                   configuration) + cms::performGradientDescent
 *                                   (master/cms/main/Headers/mesh.hpp:82-380, :432-529, :531-593)
 *   dcsg_write_stl / dcsg_write_ply cms::writeTrianglesToSTL / writeTrianglesToPLY
 *                                   (master/cms/main/Headers/utils.hpp:41-103, :106-154; master/happly.h)
 *   dcsg_export                     MyFrame::OnExportInner end to end (master/DesignCSG.cpp:638-790),
 *                                   driven by exportConfig.txt as parsed in MyFrame::OnExport (:815-835)
 *
 * Conventions: plain pointers and sizes, no C++ types, no exceptions across the boundary.  Functions
 * return DCSG_OK (0) or a negative dcsg_status; dcsg_last_error() gives the text.  The reference reports
 * a failed kernel build as (-1, build log) (Evaluator.cpp:64-89); dcsg_build does the same.
 * Host buffers are borrowed for the duration of a call.  Meshes are owned by the library and released
 * with dcsg_mesh_free.  A context is bound to one CUDA device; calls on one context are serialised by
 * the caller or by the library's internal lock (the reference uses a process-wide mutex,
 * Evaluator.cpp:10,120,170).  There is NO CPU fallback: without a CUDA device dcsg_create fails.
 */
#ifndef DCSG_H
#define DCSG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dcsg_ctx dcsg_ctx;

typedef enum dcsg_status {
    DCSG_OK = 0,
    DCSG_ERR_BUILD = -1,            /* scene source failed to compile; the log holds the compiler output */
    DCSG_ERR_INVALID = -2,          /* bad argument / scene file / configuration */
    DCSG_ERR_CUDA = -3,             /* CUDA runtime error */
    DCSG_ERR_NO_SCENE = -4,         /* called before a successful dcsg_build */
    DCSG_ERR_IO = -5,
    DCSG_ERR_LATTICE = -6,          /* bounding box is not exactly representable on the lattice (DESIGN.md) */
    DCSG_ERR_UNSUPPORTED = -7       /* e.g. gathering the soup of an adaptive walk, NCCL / peer access not available */
} dcsg_status;

/* limits of the scene protocol (reference DrawPane.h:14-15, Evaluator.h:16-17, Evaluator.cpp:7) */
#define DCSG_MAX_OBJECTS 512
#define DCSG_MAX_BUILD_STEPS 256
#define DCSG_STACK_SLOTS 64
#define DCSG_ARBITRARY_DATA_POINTS 131072

const char* dcsg_version(void);

int  dcsg_create(int device, dcsg_ctx** out);
void dcsg_destroy(dcsg_ctx* ctx);
const char* dcsg_last_error(const dcsg_ctx* ctx);
/* launch on the caller's stream (e.g. torch's current stream) instead of the context's own */
int  dcsg_set_stream(dcsg_ctx* ctx, void* cuda_stream);

/* Compile scene_dir/{scene.cu, scene.txt, buildprocedure.txt} for sm_100a with NVRTC, load the module and
 * upload scene_dir/arbitrary_data.hex if present.  log (may be NULL) receives the compiler log.
 * The module holds the scene twice: as written, and as a checked fast copy whose results are used only where they
 * are provably the same bits (DESIGN.md 3b).  Environment, read here: DCSG_EXACT_ONLY=1 builds without the fast
 * copy; DCSG_FAST_MATH=1 allows FMA contraction (NOT parity mode); DCSG_NVRTC_EXTRA="..." appends NVRTC options. */
int  dcsg_build(dcsg_ctx* ctx, const char* scene_dir, char* log, size_t log_capacity);
/* Same compilation without a device: writes the cubin (and, if ptx_path != NULL, nothing else) to
 * cubin_path.  Used by build checks on machines without a GPU. */
int  dcsg_compile_scene(const char* scene_dir, const char* cubin_path, char* log, size_t log_capacity);
/* The full translation unit handed to NVRTC for this scene (for inspection / offline nvcc builds). */
int  dcsg_scene_source(const char* scene_dir, char* out, size_t capacity, size_t* needed);

int  dcsg_set_arbitrary_data(dcsg_ctx* ctx, const float* data, size_t items);

/* xyz: n points as x,y,z triples (host).  out: n floats / 3n floats (host). */
int  dcsg_eval_sdf(dcsg_ctx* ctx, const float* xyz, size_t n, float* out);
int  dcsg_eval_normal(dcsg_ctx* ctx, const float* xyz, size_t n, float* out3);
/* same with device pointers, asynchronous on the context's stream */
int  dcsg_eval_sdf_device(dcsg_ctx* ctx, const float* d_xyz, size_t n, float* d_out);
int  dcsg_eval_normal_device(dcsg_ctx* ctx, const float* d_xyz, size_t n, float* d_out3);

/* box6 = center.xyz, diameters.xyz of the cube handed to the mesher (box_t, CVector.h) */
int  dcsg_bbox(dcsg_ctx* ctx, float search_diameter, float* box6);

/* The preview the reference renders every idle frame: BasicDrawPane::idled -> kernel k1 (master/DrawPane.cpp:122-240,
 * master/k1.cl:480-580).  640 x 480 sphere tracing from campos along the camera basis (right, up, forward), k1's SDF
 * (scene + the three axis-gizmo cylinders), 6-tap normals, materials.  rgb_host receives 640*480*3 bytes, rows top to
 * bottom -- the buffer the reference blits.  Off the export path; a second consumer of the compiled scene. */
int  dcsg_preview(dcsg_ctx* ctx, const float* campos3, const float* right3, const float* up3, const float* forward3,
                  uint8_t* rgb_host);

/* fp32 SDF on lattice planes [z_begin, z_end) of the (2^grid_level + 1)^3 lattice, x fastest then y then z.
 * out_host may be NULL (values stay in the context's device buffer, see dcsg_lattice_device_ptr). */
int  dcsg_sample_lattice(dcsg_ctx* ctx, const float* box6, int grid_level, int z_begin, int z_end, float* out_host);
const float* dcsg_lattice_device_ptr(const dcsg_ctx* ctx);

typedef struct dcsg_extract_cfg {
    float box[6];                   /* from dcsg_bbox */
    int   grid_level;               /* N = 2^grid_level cells per side; lattice (N+1)^3 */
    int   min_level, max_level;     /* octree levels, min <= max <= grid_level.  min = max = grid_level is the uniform
                                       lattice (indexed mesh, z-slabs); anything else is the reference's adaptive walk
                                       (mesh.hpp:212-267): triangle soup (vertex i of triangle t = vertex 3t+i, no keys);
                                       z-slabs of it must be cut on multiples of 2^(grid_level - min_level) layers */
    float complex_threshold;        /* complexSurfaceThreshold, radians (adaptive walk) */
    int   gd_steps;                 /* gradient-descent projection steps (reference: 50) */
    int   want_normals;             /* 6-tap normals at the final vertices */
    int   slab_z0, slab_z1;         /* cell layers [z0, z1) handled by this context; 0,0 = all */
    int   copy_to_host;             /* also fill the h_* arrays (pinned) */
    int   no_cull;                  /* 1 = skip the reference's centre-sample cull (NOT parity) */
    int   dense;                    /* 1 = evaluate every lattice sample (dcsg_k_lattice); 0 = octree-ordered sparse
                                       evaluation that skips what the reference's walk skips (same output) */
    int   retopologize;             /* 1 = run cms::retopologize between the walk and the projection the way the reference
                                       build behaves (mesh.hpp:432-529, see DESIGN.md): every triangle becomes
                                       3*2^(grid-min) - 2 triangles; identity when min = grid */
    int   defer_projection;         /* 1 = stop after emission; the caller runs dcsg_project (multi-GPU: the mesh gather of
                                       keys / triangles overlaps the projection) */
} dcsg_extract_cfg;

enum { DCSG_STAGE_LATTICE = 0, DCSG_STAGE_CLASSIFY, DCSG_STAGE_EMIT, DCSG_STAGE_PROJECT, DCSG_STAGE_COPY, DCSG_STAGE_COUNT };

typedef struct dcsg_mesh {
    uint64_t num_vertices, num_triangles, num_cells;
    /* device arrays (owned by the library) */
    float*    d_vertices;           /* 3 per vertex, ascending vertex key */
    float*    d_normals;            /* 3 per vertex or NULL */
    uint64_t* d_vertex_keys;        /* 3*(x + P*(y + P*z)) + axis, global lattice indices; NULL for adaptive soups */
    uint32_t* d_triangles;          /* 3 per triangle: canonical order = cell index, then table order */
    uint64_t* d_cell_ids;           /* x + N*(y + N*z), ascending; adaptive: level << 56 | nx + n*(ny + n*nz), n = 2^level */
    uint8_t*  d_cell_masks;         /* 8-bit corner sign mask per active cell */
    /* host copies (pinned) when copy_to_host was set, else NULL */
    float*    h_vertices;
    float*    h_normals;
    uint64_t* h_vertex_keys;
    uint32_t* h_triangles;
    uint64_t* h_cell_ids;
    uint8_t*  h_cell_masks;
    uint64_t  lattice_samples;      /* SDF evaluations of the lattice pass */
    float     stage_ms[DCSG_STAGE_COUNT];   /* device time per stage (CUDA events on the launch stream) */
    /* z-slabs of a uniform lattice: the first owned_vertices vertices are this slab's own (sample planes [slab_z0, slab_z1),
     * plus the lattice's closing plane in the last slab); the halo_vertices after them are copies of the NEXT slab's first
     * vertices, in its order, kept so that the slab's mesh is self-contained.  Hence owned vertices and triangles of the
     * slabs, concatenated in slab order with the vertex ids of slab r shifted by the owned vertices of the slabs before it,
     * ARE the whole mesh -- no weld.  Whole lattice / soups: owned = num_vertices, halo = 0. */
    uint64_t  owned_vertices, halo_vertices;
    void*     reserved;
} dcsg_mesh;

int  dcsg_extract(dcsg_ctx* ctx, const dcsg_extract_cfg* cfg, dcsg_mesh* out);
/* cms::performGradientDescent (mesh.hpp:531-593) on the vertices of a mesh extracted with defer_projection (or with
 * gd_steps = 0), plus the optional final normals.  ASYNCHRONOUS on the context's stream: the device arrays are
 * final once that stream reaches the point after this call. */
int  dcsg_project(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, int want_normals);
void dcsg_mesh_free(dcsg_ctx* ctx, dcsg_mesh* mesh);
/* Measurement support: what the projection kernel really executed since the last call (then cleared) -- tap_rounds = rounds
 * of seven SDF evaluations (six taps + the centre; a vertex that reaches a fixed point stops early, so this is less than
 * vertices x steps), exact_rounds = rounds evaluated a second time through the exact copy of the scene (DESIGN.md 3b). */
int  dcsg_project_stats(dcsg_ctx* ctx, uint64_t* tap_rounds, uint64_t* exact_rounds);

/* Triangle soup, 9 floats per triangle, into a host buffer (the reference's in-memory mesh). */
int  dcsg_mesh_soup(dcsg_ctx* ctx, const dcsg_mesh* mesh, float* out_host);

/* Files byte-compatible with the reference's writers.  The bodies are laid out on the device. */
int  dcsg_write_stl(dcsg_ctx* ctx, const dcsg_mesh* mesh, const char* path);
int  dcsg_write_ply(dcsg_ctx* ctx, const dcsg_mesh* mesh, const char* path);
/* The same bytes into caller memory (size query with out == NULL). */
int  dcsg_format_stl(dcsg_ctx* ctx, const dcsg_mesh* mesh, uint8_t* out, size_t capacity, size_t* needed);
int  dcsg_format_ply(dcsg_ctx* ctx, const dcsg_mesh* mesh, uint8_t* out, size_t capacity, size_t* needed);

/* The same bytes left in the library's pinned host buffer (no extra copy); valid until the next format / write
 * call on this context. */
int  dcsg_format_stl_view(dcsg_ctx* ctx, const dcsg_mesh* mesh, const uint8_t** bytes, size_t* size);
int  dcsg_format_ply_view(dcsg_ctx* ctx, const dcsg_mesh* mesh, const uint8_t** bytes, size_t* size);
/* Multi-GPU file export without a mesh gather.  The ranks' triangles are consecutive in rank order (canonical order)
 * and the reference's files are triangle soup, so rank r's PLY vertex rows (72 B / triangle), PLY face rows (13 B /
 * triangle, soup indices continuing from 3 * first_triangle) and STL records (50 B / triangle) are contiguous byte
 * ranges of the single-GPU files:   PLY = header | vertex rows of all ranks | face rows of all ranks;
 * STL = 84-byte header | records of all ranks.  The three views point into the library's pinned host buffer (valid
 * until the next format / write call on this context); first_triangle = triangles of the ranks below (count
 * all-gather).  dcsg_file_header returns the header for the TOTAL triangle count (ply = 1: happly's, ply = 0: STL's). */
int  dcsg_format_segments(dcsg_ctx* ctx, const dcsg_mesh* mesh, uint64_t first_triangle, const uint8_t** ply_vertex_rows,
                          const uint8_t** ply_face_rows, const uint8_t** stl_records);
int  dcsg_file_header(int ply, uint64_t total_triangles, uint8_t* out, size_t capacity, size_t* needed);
/* The face rows of the soup PLY for triangles [first_triangle, first_triangle + num_triangles): 13 bytes each, the byte 3
 * and the little-endian indices 3i, 3i+1, 3i+2 (reference utils.hpp:131-141 through happly.h:1640-1668).  They depend on
 * the triangle COUNT only, so they are produced on the host (no device, no context): the pipelined export writes them
 * straight into its pinned buffer instead of sending them over PCIe; sharded writers can do the same. */
int  dcsg_ply_face_rows(uint64_t first_triangle, uint64_t num_triangles, uint8_t* out, size_t capacity);
/* The other rows of the two files from a triangle soup (9 floats per triangle), on the host, no device: the PLY vertex rows
 * (9 doubles per triangle, reference utils.hpp:117-123 through happly.h:1538-1562) and the STL records (zero normal, A B C as
 * x z y, zero attribute = 50 bytes, utils.hpp:59-99).  This is what the file pipeline's host threads run on the part of the
 * triangles that crosses the link as float soup (36 B instead of 122 B of finished rows); ply_rows must be 8-byte aligned. */
int  dcsg_soup_rows(const float* soup, uint64_t num_triangles, uint8_t* ply_rows, uint8_t* stl_records);
/* dcsg_project + dcsg_format_segments as ONE pipelined pass over a mesh extracted with defer_projection: vertices are
 * projected in chunks (uniform lattice: z-ordered, cut on cell layers; adaptive walk: runs of soup triangles / of the strips
 * cms::retopologize makes of them), and as soon as a chunk's triangles have all their vertices their file rows are
 * formatted and copied to pinned host memory on a second stream while the next chunk is projected.  Same bytes as the
 * two separate calls; synchronous. */
int  dcsg_project_and_format_segments(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, uint64_t first_triangle,
                                      const uint8_t** ply_vertex_rows, const uint8_t** ply_face_rows,
                                      const uint8_t** stl_records);

/* The same pipeline writing FILES: every chunk that has reached pinned host memory is written (pwrite, a pool of
 * writer threads) while later chunks are still being projected and copied.  A single-GPU export passes
 * first_triangle = 0, total_triangles = the mesh's, create_files = 1 (files created, headers written).  In a
 * multi-GPU export every rank writes its byte ranges of the shared files (created beforehand, create_files = 0;
 * one rank writes the headers, dcsg_file_header).  Either path may be NULL.  dcsg_export uses this for every configuration. */
int  dcsg_project_and_write_files(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, uint64_t first_triangle,
                                  uint64_t total_triangles, int create_files, const char* stl_path, const char* ply_path);

/* Progress of dcsg_export, the counterpart of the reference's exportProcessState + the counters its GUI thread polls
 * every 100 ms (master/DesignCSG.cpp:603-614, :754-768, :854-1023).  The callback runs on the thread that called
 * dcsg_export, at every state change and -- while the files are written -- once per chunk with done = triangles whose
 * rows have reached the files so far, total = triangles of the mesh (the reference's numTrianglesWritten / maxTriangles);
 * for DCSG_PROGRESS_GRADIENT_DESCENT done / total are projection steps (gradientDescentStepsCompleted); otherwise 0 / 0.
 * It must not call back into the same context.  fn = NULL removes it. */
enum {
    DCSG_PROGRESS_IDLE = 0,
    DCSG_PROGRESS_ESTIMATING_BOUNDING_BOX,
    DCSG_PROGRESS_PERFORMING_CMS,
    DCSG_PROGRESS_RETOPOLOGIZING,
    DCSG_PROGRESS_GRADIENT_DESCENT,
    DCSG_PROGRESS_WRITING_STL,
    DCSG_PROGRESS_WRITING_PLY,
    DCSG_PROGRESS_COMPLETE
};
typedef void (*dcsg_progress_fn)(void* user, int state, uint64_t done, uint64_t total);
int  dcsg_set_progress_callback(dcsg_ctx* ctx, dcsg_progress_fn fn, void* user);

/* Number of CUDA kernels this library has launched in this process (measurement support). */
unsigned long long dcsg_launch_count(void);

/* ---- indexed binary PLY (no reference counterpart: the reference writes triangle soup only, utils.hpp:41-154) ----------------
 * An opt-in format beside the reference's files, which stay as they are.  Binary little-endian, header:
 *   ply / format binary_little_endian 1.0 / comment DesignCSG export, indexed: vertices shared between faces /
 *   element vertex V / property float x, y, z [/ property float nx, ny, nz  with DCSG_PLY_NORMALS] /
 *   element face T / property list uchar uint vertex_indices / end_header
 * then V vertex rows (12 B, 24 B with normals) and T face rows (the byte 3, three uint32 vertex ids: 13 B).  Face i is triangle i
 * of the reference's files, same corner order, degenerate faces kept: expanding the file, double(vertex[face]), gives the
 * vertex rows of the soup PLY byte for byte.  V < 2^32. */
#define DCSG_PLY_NORMALS 1

/* Weld (no reference counterpart): vertices whose positions are bit-identical (all three float words equal) become one, numbered
 * in the order of the smallest input index among them; triangles are renumbered, normals follow their vertices, num_vertices
 * shrinks, host copies (copy_to_host) are refreshed.  Deterministic.  Applies to the positions the mesh holds at the call.
 * A lattice mesh (vertex keys) is returned unchanged: it holds every position once already.  A slab of a sharded adaptive
 * extraction is refused (DCSG_ERR_UNSUPPORTED).  A welded adaptive mesh is no longer accepted by the soup file pipeline
 * (dcsg_project_and_*); dcsg_project, dcsg_mesh_soup and the soup writers work on it and give the same bytes as before. */
int  dcsg_mesh_weld(dcsg_ctx* ctx, dcsg_mesh* mesh);
/* The indexed PLY of a mesh as it is (no projection); flags & DCSG_PLY_NORMALS needs d_normals.  No reference counterpart. */
int  dcsg_write_ply_indexed(dcsg_ctx* ctx, const dcsg_mesh* mesh, int flags, const char* path);

/* ---- outward winding (no reference counterpart: the reference's lookup table winds 399 of its 820 triangles inwards, and its
 * STL records carry zero normals, so its files mix both windings; DESIGN.md 7c) ----------------------------------------------
 * dcsg_mesh_orient swaps corners 1 and 2 of every inward-facing triangle, in place on the device: afterwards every triangle
 * (A, B, C) has (B - A) x (C - A) pointing out of the solid.  Which triangles face inwards follows from the cell's corner mask
 * and the triangle's slot in the table row alone.  Vertices, normals, cells and the triangle order are untouched; host copies
 * (copy_to_host) are refreshed; a second call is a no-op.  Works before and after dcsg_mesh_weld and on the `local` mesh of
 * dcsg_extract_sharded; a mesh the library does not own or without cell masks (the borrowed `whole` of a gather) is refused
 * with DCSG_ERR_INVALID.  Every writer reads the corners through d_triangles; the STL writers of an oriented mesh list the
 * corners A, C, B, because the records store each corner as (x, z, y) (reference utils.hpp:59-99), which mirrors the mesh.
 * The files are then no longer the reference's bytes. */
int  dcsg_mesh_orient(dcsg_ctx* ctx, dcsg_mesh* mesh);

/* Per-context options of the four dcsg_export* calls (like the progress callback).  DCSG_EXPORT_OUTWARD: dcsg_mesh_orient on the
 * (slab's) mesh right after the extraction, so that every file the export writes is outward-wound.  0, the default, writes
 * the reference's bytes. */
#define DCSG_EXPORT_OUTWARD 1
int  dcsg_set_export_flags(dcsg_ctx* ctx, int flags);

/* ---- mesh inspection (no reference counterpart: the reference never checks the mesh it writes; DESIGN.md 7d) -------------------
 * dcsg_mesh_inspect reports whether a mesh is a closed, consistently wound solid, and its area, volume, centre of mass and
 * extents, computed on the device from d_vertices, d_triangles and the two counts alone.  It works on every mesh the library
 * hands out: uniform or adaptive, welded or not, oriented or not, the `local` slab of a sharded extraction (a mesh of its own:
 * its cut shows as boundary edges) and the borrowed `whole` of a gather.  Synchronous; the mesh, its host copies and the
 * device are left unchanged.  Deterministic: the same bits on every run.  V = num_vertices (< 2^32), T = num_triangles.
 *   degenerate triangle   two of its three ids are equal; counted, then ignored by everything below
 *   referenced vertex     used by a non-degenerate triangle; unreferenced_vertices = V - referenced
 *   non-finite            nonfinite_vertices: referenced vertices with a NaN or Inf coordinate; nonfinite_triangles: non-degenerate
 *                         triangles with such a corner -- they count for edges and components, not for area, volume, centroid, box
 *   edges                 the half-edges (a,b), (b,c), (c,a) of the non-degenerate triangles, by undirected pair; per edge k
 *                         half-edges, f of them with a < b: boundary k = 1, manifold k = 2, non-manifold k >= 3, misoriented
 *                         k = 2 and f != 1 (both faces traverse the edge the same way)
 *   per triangle          in double from the float corners: u = b - a, w = c - a, n = u x w, area_t = |n| / 2,
 *                         vol_t = a . (b x c) / 6, centroid_t = vol_t (a + b + c); zero_area_triangles: finite ones with n = 0
 *   totals                area, signed_volume = sums over the non-degenerate finite triangles; centroid = sum centroid_t /
 *                         (4 signed_volume), NaN when the volume is 0; bbox_min / bbox_max = exact float extremes over the
 *                         referenced finite vertices (+Inf / -Inf without any)
 *   components            shells: vertices connected through the ids of non-degenerate triangles, counted over referenced
 *                         vertices and numbered in the order of their smallest vertex id
 * The component arrays (host, NULL allowed with component_capacity = 0) receive the first min(capacity, components) components'
 * triangle counts, areas and signed volumes; floor(V / 3) bounds `components`.  A triangle id >= V returns DCSG_ERR_INVALID.
 * A mesh without triangles gives a zeroed report (NaN centroid, +Inf / -Inf box). */
typedef struct dcsg_mesh_report {
    uint64_t num_vertices, num_triangles;
    uint64_t unreferenced_vertices, nonfinite_vertices;
    uint64_t degenerate_triangles, zero_area_triangles, nonfinite_triangles;
    uint64_t edges, boundary_edges, manifold_edges, nonmanifold_edges, misoriented_edges;
    uint64_t components;
    double   area, signed_volume, centroid[3];
    float    bbox_min[3], bbox_max[3];
} dcsg_mesh_report;

int  dcsg_mesh_inspect(dcsg_ctx* ctx, const dcsg_mesh* mesh, dcsg_mesh_report* report, uint64_t component_capacity,
                       uint64_t* component_triangles, double* component_area, double* component_signed_volume);

/* ---- mesh deviation (no reference counterpart: DESIGN.md 7e) ------------------------------------------------------------------
 * dcsg_mesh_deviation samples the scene's SDF f over every triangle of a mesh, on the device: how far the mesh strays from the
 * design.  f is what dcsg_eval_sdf returns (the checked fast copy, the exact copy as its fallback): every value used here is
 * bit-identical to dcsg_eval_sdf at the same point.  f is the SDF VALUE, not the Euclidean distance to the surface: the two
 * agree for exact SDFs (a lone sphere) but not under CSG min / max, smooth minima or non-uniform scale -- hence the names
 * *_sdf / *_abs.  Reads d_vertices, d_triangles and the two counts, like dcsg_mesh_inspect, and works on the same meshes.
 * Synchronous; the mesh, its host copies and the device state are left unchanged.  Deterministic: min, max and argmax are
 * exact, every floating-point sum is a reduction in a fixed order (no atomics).  V = num_vertices (< 2^32), T = num_triangles.
 *   degenerate triangle   two of its ids are equal (dcsg_mesh_inspect's rule); a triangle id >= V returns DCSG_ERR_INVALID,
 *                         checked before any vertex is read through it
 *   measured triangle     not degenerate, and its nine corner floats are finite
 *   measured vertex       finite, and referenced by a non-degenerate triangle
 *   samples               k = subdivision, 1 <= k <= 16.  A measured triangle (a, b, c) has its 3 corners, whose values are the
 *                         vertices' own f(v) (evaluated once per vertex), and S = (k+1)(k+2)/2 - 3 further samples, one per (i, j)
 *                         with i, j >= 0, i + j <= k other than (0,0), (k,0), (0,k), i ascending then j ascending, at the fp32
 *                         point p = ((a * (float)(k-i-j) + b * (float)i) + c * (float)j) / (float)k per coordinate, in this
 *                         order of IEEE operations (no contraction).  A sample on an edge two triangles share is evaluated for
 *                         each of them.  k = 1: corners only; k = 4: 12 more samples per triangle.
 *   triangle_max_abs[t]   max |f| over t's 3 + S values; NaN when t is not measured or any of its values is NaN
 *   report                samples = measured_vertices + S * measured_triangles (the evaluations used), nan_samples = NaN values
 *                         among them; over_tolerance = measured triangles with triangle_max_abs > tolerance or NaN;
 *                         vertex_max_abs, vertex_rms = sqrt(sum f^2 / n) over the n non-NaN values of the measured vertices;
 *                         min_sdf / max_sdf = extremes over the non-NaN values (corners and samples) of the measured triangles,
 *                         -0 below +0; max_abs = max(max_sdf, -min_sdf); worst_triangle = the smallest t whose non-NaN values
 *                         reach max_abs (triangle_max_abs[t] == max_abs when t has no NaN value), worst_point = the first of its
 *                         values in corner-then-(i, j) order that does; mean_abs = sum area_t mean_t / sum area_t over the
 *                         measured triangles without a NaN value, mean_t = (double sum of |f| over the 3 + S values in sample
 *                         order) / (3 + S), area_t = dcsg_mesh_inspect's per-triangle area bit for bit; NaN when sum area_t = 0
 *   empty                 without a measured triangle: the triangle counts 0, min_sdf = +Inf, max_sdf = max_abs = -Inf, worst_triangle =
 *                         UINT64_MAX, worst_point NaN; without a non-NaN vertex value vertex_max_abs = -Inf, vertex_rms NaN
 * tolerance >= 0 (a negative or NaN one is DCSG_ERR_INVALID); triangle_max_abs: host array of T floats, or NULL.  Before dcsg_build:
 * DCSG_ERR_NO_SCENE. */
typedef struct dcsg_deviation_report {
    uint64_t num_vertices, num_triangles;
    uint64_t measured_vertices, measured_triangles;
    uint64_t samples, nan_samples, over_tolerance;
    uint64_t worst_triangle;
    float    vertex_max_abs, min_sdf, max_sdf, max_abs;
    float    worst_point[3];
    double   vertex_rms, mean_abs;
} dcsg_deviation_report;

int  dcsg_mesh_deviation(dcsg_ctx* ctx, const dcsg_mesh* mesh, int subdivision, float tolerance, dcsg_deviation_report* report,
                         float* triangle_max_abs);

typedef struct dcsg_export_report {
    float    box[6];
    uint64_t num_vertices, num_triangles, num_cells;
    float    bbox_ms, extract_ms[DCSG_STAGE_COUNT], format_ms, write_ms, total_ms;
} dcsg_export_report;

/* OnExportInner: reads scene_dir/exportConfig.txt (9 lines), runs bbox -> extract -> project -> write.
 * grid_level_override > 0 replaces min/max/grid level by that value (uniform lattice).  Either path may be
 * NULL. */
int  dcsg_export(dcsg_ctx* ctx, const char* scene_dir, int grid_level_override, const char* stl_path,
                 const char* ply_path, dcsg_export_report* report);

/* dcsg_export's pipeline writing the indexed PLY instead of the soup files (no reference counterpart): bbox -> extract (the
 * reference's retopologize included) -> adaptive levels: weld BEFORE the projection (equal starting positions project to equal
 * positions and normals, so each is projected once) -> projection in chunks of vertices pipelined with the copies and the
 * writes; the face rows are formatted and copied while the projection runs.  Same progress states as dcsg_export; while the
 * file is written, done / total of DCSG_PROGRESS_WRITING_PLY count vertex rows.  report->num_vertices = the file's vertices. */
int  dcsg_export_indexed(dcsg_ctx* ctx, const char* scene_dir, int grid_level_override, int flags, const char* ply_path,
                         dcsg_export_report* report);

/* ---- multi-GPU export: one process per GPU, one node (no reference counterpart: the reference's export runs on one OpenCL
 * device, DesignCSG.cpp:638-790).  The lattice is cut into z-slabs, one per rank.  NCCL carries the small collectives (the
 * all-reduce of the sharded bounding-box search, the all-gather of the slabs' counts, barriers); the mesh itself is stored by
 * the kernels straight into the gathering rank's arrays through peer mappings (CUDA IPC over NVLink), at offsets that follow
 * from the gathered counts -- slabs own their vertices exactly, so nothing is welded.  NCCL is loaded at run time
 * (libnccl.so.2, or the path in DCSG_NCCL_LIBRARY); single-GPU hosts never need it.
 *   rank 0:     dcsg_comm_unique_id(id); hand id to the other ranks (pipe, file, socket, MPI, ...)
 *   every rank: dcsg_create(local device) -> dcsg_build -> dcsg_comm_create(ctx, id, rank, world, &comm)   [collective]
 *               dcsg_export_sharded(...) or dcsg_bbox_sharded + dcsg_extract_sharded                        [collective]
 *               dcsg_comm_destroy(comm) before dcsg_destroy(ctx) */
typedef struct dcsg_comm dcsg_comm;
#define DCSG_COMM_ID_BYTES 128
int  dcsg_comm_unique_id(uint8_t id[DCSG_COMM_ID_BYTES]);
int  dcsg_comm_create(dcsg_ctx* ctx, const uint8_t id[DCSG_COMM_ID_BYTES], int rank, int world, dcsg_comm** out);
void dcsg_comm_destroy(dcsg_comm* comm);
int  dcsg_comm_rank(const dcsg_comm* comm);
int  dcsg_comm_world(const dcsg_comm* comm);
int  dcsg_comm_barrier(dcsg_comm* comm);        /* returns once every rank's queued device work, peer stores included, is complete */

/* dcsg_bbox over all ranks: every rank searches its share of the 256^3 samples, the six extreme indices and the surface
 * histogram are all-reduced (integers: the result is the single-GPU box, bit for bit, on every rank). */
int  dcsg_bbox_sharded(dcsg_ctx* ctx, dcsg_comm* comm, float search_diameter, float* box6);

typedef struct dcsg_shard_info {
    int      rank, world;
    int      slab_z0, slab_z1;              /* this rank's cell layers (dcsg_plan_slabs over the last sharded search) */
    uint64_t first_vertex, first_triangle;  /* global index of this rank's first own vertex / triangle */
    uint64_t total_vertices, total_triangles, total_cells;
} dcsg_shard_info;

/* dcsg_extract of this rank's z-slab (cfg->slab_* are ignored: the slabs are planned from the last dcsg_bbox_sharded search,
 * the same on every rank; adaptive octree levels: gather_to = -1 only, the ranks keep their slabs of the soup).  `local` receives the slab's self-contained mesh as from dcsg_extract.
 * gather_to >= 0: the projection runs here too and the WHOLE mesh -- vertices in key order, triangles in canonical order,
 * global vertex ids: the arrays of a single-GPU dcsg_extract -- is complete in the arrays of rank gather_to when the call
 * returns; `whole` (optional) then holds borrowed device pointers to them on that rank (valid until the next sharded call
 * on this communicator; dcsg_mesh_free is not needed) and the total counts on every rank.  gather_to = -1: nothing is
 * gathered (cfg->defer_projection may be set: sharded file export).  Collective. */
int  dcsg_extract_sharded(dcsg_ctx* ctx, dcsg_comm* comm, const dcsg_extract_cfg* cfg, int gather_to, dcsg_mesh* local,
                          dcsg_mesh* whole, dcsg_shard_info* info);

/* dcsg_export over all ranks: sharded search, slab plan, extraction; rank 0 creates the files and writes the headers, then
 * every rank projects its slab and writes the byte ranges of its own triangles (they are consecutive in the files: rank
 * order is the canonical triangle order).  Same files as dcsg_export on one GPU, byte for byte.  grid_level_override > 0:
 * uniform lattice; 0: the design's own exportConfig.txt -- adaptive octree levels are cut on whole level-min nodes, their
 * canonical order is (level, node), and every rank writes one byte range per octree level.  Collective. */
int  dcsg_export_sharded(dcsg_ctx* ctx, dcsg_comm* comm, const char* scene_dir, int grid_level_override, const char* stl_path,
                         const char* ply_path, dcsg_export_report* report);

/* dcsg_export_indexed over all ranks, uniform lattice only (grid_level_override > 0; no reference counterpart).  Rank r
 * projects and writes only the vertices its slab owns, at header + row bytes * first_vertex, and its face rows with ids +
 * first_vertex at header + row bytes * total_vertices + 13 * first_triangle; rank 0 creates the file.  Same file as
 * dcsg_export_indexed on one GPU, byte for byte.  Adaptive levels return DCSG_ERR_UNSUPPORTED on every rank before the first
 * collective (the weld spans slabs).  Collective. */
int  dcsg_export_sharded_indexed(dcsg_ctx* ctx, dcsg_comm* comm, const char* scene_dir, int grid_level_override, int flags,
                                 const char* ply_path, dcsg_export_report* report);

/* Multi-GPU: z-slab boundaries (cell layers, multiples of `granularity`) that give `world` ranks about the same
 * amount of surface, estimated from the per-z sign-change counts of the last dcsg_bbox search on this context.
 * Every rank computes the same plan from its own (identical) search, so nothing is communicated.  bounds has
 * world + 1 entries: rank r meshes layers [bounds[r], bounds[r+1]).  Falls back to equal slabs without an
 * estimate -- before the first search after dcsg_build (a rebuild forgets the previous scene's search).  No reference
 * counterpart. */
int  dcsg_plan_slabs(dcsg_ctx* ctx, const float* box6, int grid_level, int world, int granularity, int* bounds);

/* Measurement support (no reference counterpart): achieved non-tensor FP32 rate of this device in TFLOP/s.
 * mode 0 = FFMA chains (2 FLOP / instruction), mode 1 = FMUL + FADD without contraction (1 FLOP / instruction,
 * the ceiling of parity mode).  Used by bench.py as the roofline denominator of the SDF kernels. */
int  dcsg_fp32_peak(dcsg_ctx* ctx, int mode, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* DCSG_H */
