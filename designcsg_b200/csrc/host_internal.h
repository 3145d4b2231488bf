// host_internal.h -- declarations shared by the host-side translation units of libdcsg.so
// (host_scene.cu: scene files -> specialised CUDA source -> cubin; host_context.cu: context, point evaluation,
// bounding box, slab plan, preview; host_extract.cu: lattice passes and dcsg_extract; host_files.cu: byte-exact
// files, the projection / format / copy / write pipeline, the one driver behind dcsg_export, dcsg_export_sharded,
// dcsg_export_indexed and dcsg_export_sharded_indexed; host_indexed.cu: the weld and the indexed PLY's pipeline;
// host_inspect.cu: the mesh report; host_deviation.cu: the mesh's deviation from the design; host_comm.cu: the communicator and the sharded search and extraction).  Not part of the ABI (include/dcsg.h is).
#pragma once
#include <cuda_runtime.h>
#include <nvrtc.h>
#include <set>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <condition_variable>
#include <cerrno>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <emmintrin.h>

#include "../../include/dcsg.h"
#include "mesher.h"
#include "scene_params.h"

// x-consecutive lattice samples per thread of dcsg_k_lattice (1, 2, 4 or 8); tunable through the environment
inline int dcsg_lattice_spt() {
    static const int v = [] {
        const char* e = getenv("DCSG_LATTICE_SPT");
        const int n = e ? atoi(e) : 4;
        return (n == 1 || n == 2 || n == 4 || n == 8) ? n : 4;
    }();
    return v;
}
#define DCSG_LATTICE_SPT dcsg_lattice_spt()

double dcsg_fp32_peak_tflops(int mode, int reps, cudaStream_t stream);     // peak_kernels.cu

namespace dcsg_host {

// ---------------------------------------------------------------------------------------------
// small utilities
// ---------------------------------------------------------------------------------------------
inline std::string format(const char* fmt, ...) {
    char buf[2048];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    return std::string(buf);
}

inline bool read_file(const std::string& path, std::string& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    out.clear();
    char buf[65536];
    size_t n;
    while ((n = fread(buf, 1, sizeof(buf), f)) > 0) out.append(buf, n);
    fclose(f);
    return true;
}

inline double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// grow-only device buffer: repeated extractions of the same size allocate nothing
struct DevBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&ptr, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(ptr); }
};

struct HostBuf {        // pinned
    void* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost(&ptr, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(ptr); }
};

// ---------------------------------------------------------------------------------------------
// scene files (reference DrawPane.cpp:267-371: fgets + sscanf per field; limits DrawPane.h:14-15)
// ---------------------------------------------------------------------------------------------
struct Scene {
    int num_objects = 0;
    int shape_id[DCSG_MAX_OBJECTS];
    int material_id[DCSG_MAX_OBJECTS];
    float position[DCSG_MAX_OBJECTS][3], right[DCSG_MAX_OBJECTS][3], up[DCSG_MAX_OBJECTS][3], forward[DCSG_MAX_OBJECTS][3];
    int num_steps = 0;
    int steps[DCSG_MAX_BUILD_STEPS][4];
    std::string scene_cu;
    int private_words = 0;                  // per-thread words of the design's program-scope variables ("// DCSG_PRIVATE_WORDS n")
    std::vector<float> arbitrary_data;      // may be empty
    std::vector<std::string> export_config; // 9 lines when exportConfig.txt exists
};

// host_scene.cu
bool load_scene(const std::string& dir, Scene& sc, std::string& err);
bool scene_wants_fast_path(const Scene& sc);
// tapAxes: the fast copy's normals through the per-axis forms (generate_primary_sdf_axis) instead of the rolled tap loop
std::string assemble_source(const Scene& sc, bool fastPath, std::string& err, bool flagInShared = false, bool tapAxes = false);
bool compile_scene(const Scene& sc, std::vector<char>& cubin, std::string& log, std::string& err, bool exactOnly = false);
bool compile_source(const std::string& src, std::vector<char>& cubin, std::string& log);
// what a kernel of an sm_100a cubin occupies: registers per thread, local memory (the largest stack frame of the kernel and of the
// functions compiled into its text section), bytes of code.  Read from the ELF, no device needed.
struct KernelFootprint {
    int registers = -1;
    uint32_t frameBytes = 0;
    uint64_t textBytes = 0;
};
bool kernel_footprint(const std::vector<char>& cubin, const char* kernel, KernelFootprint& fp);
void copy_log(const std::string& log, char* out, size_t cap);

}  // namespace dcsg_host

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
struct dcsg_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    std::string error;
    std::mutex lock;

    int sm_count = 0;               // multiprocessors of `device` (persistent grids are sized from it)
    int project_blocks_per_sm = 8;  // resident blocks of dcsg_k_project per multiprocessor (dcsg_build asks the occupancy calculator)
    int node_ranks = 1;             // ranks sharing this host (set by dcsg_comm_create): they share its cores and memory bandwidth
    dcsg_progress_fn progress = nullptr;    // optional, see dcsg_set_progress_callback
    void* progress_user = nullptr;
    int export_flags = 0;           // DCSG_EXPORT_*, see dcsg_set_export_flags

    bool built = false;
    cudaStream_t copy_stream = nullptr;
    cudaStream_t aux_stream = nullptr;      // the clean-up pass of a sparse extraction runs here, under whatever follows on `stream`
    cudaEvent_t aux_ready = nullptr, aux_done = nullptr;
    bool aux_pending = false;
    cudaEvent_t chunk_event[16] = {nullptr};
    cudaEvent_t copied_event[16] = {nullptr};
    dcsg_host::Scene scene;
    cudaLibrary_t lib = nullptr;
    cudaKernel_t k_eval_sdf = nullptr, k_eval_normal = nullptr, k_bbox = nullptr, k_lattice = nullptr,
                 k_coarse_nodes = nullptr, k_project = nullptr, k_descend = nullptr, k_descend_list = nullptr, k_descend_top = nullptr, k_leaf = nullptr, k_corners = nullptr, k_adapt_level = nullptr, k_preview = nullptr, k_flag_rate = nullptr;
    float* d_arbitrary = nullptr;
    float* d_camera_axes[3] = {nullptr, nullptr, nullptr};      // rgt_g / upp_g / fwd_g of the module (k1.cl:35-37)

    uint8_t* d_tri_count = nullptr;
    int8_t* d_tri_table = nullptr;
    uint8_t* d_tri_flip = nullptr;          // kDcsgTriFlip: the inward-facing triangles of every table row

    // workspace
    dcsg_host::DevBuf pts, vals, axes, sign, leaf, cfail, coarse, levels, alive, vinfo, tiles, small, lattice_values, fmt,
           adapt_emit, adapt_snap, search_bits, project_cursor, project_list, lists, masks, soup,
           weld,                    // dcsg_mesh_weld: sort / scan scratch, then the compacted vertices and normals
           orient,                  // dcsg_mesh_orient: per-cell counts, their prefix and the scan's scratch
           inspect,                 // dcsg_mesh_inspect: sort / reduction scratch, the component runs, the totals
           deviation;               // dcsg_mesh_deviation: vertex values, per-triangle terms, one chunk's points and values
    dcsg_host::HostBuf pinned, pinned_small, pinned_soup;
    // sparse extraction: `leaf` (as leafAlive) and `alive` are all-zero between extractions -- every sparse
    // extraction zeroes the words it wrote (dcsg_launch_cleanup); anything else that writes them clears this flag
    bool sparse_clean = false;
    // multi-GPU (host_comm.cu), both optional.  exchange_pre: queued on the stream right before dcsg_extract reads its sizes
    // back -- d_counts = {cells, triangles, vertices incl. halo copies, halo copies} of this slab on the device -- so that the
    // all-gather of the ranks' counts shares the extraction's one host round trip (32 words: [0..3] as said, [16 + l] =
    // triangles of octree level l in the adaptive walk).  exchange_post: after that round trip,
    // before the emitters are launched: offsets from the gathered counts, the gathering rank's arrays (re)allocated.
    int (*exchange_pre)(dcsg_ctx* ctx, void* user, const uint32_t* d_counts, cudaStream_t stream) = nullptr;
    int (*exchange_post)(dcsg_ctx* ctx, void* user, dcsg_mesher_params& mp) = nullptr;
    void* exchange_user = nullptr;
    bool skip_final_sync = false;   // dcsg_extract returns with its last kernels still queued (stage times are read by the caller)
    uint32_t zhist[512] = {0};      // sign changes of the last bounding-box search per z index: [0,256) in-plane edges, [256,512) z-edges
    float zhist_c = 0.0f;           // its voxel size; 0 = no search of the current scene yet (dcsg_build clears it)
    cudaEvent_t ev[DCSG_STAGE_COUNT + 2] = {nullptr};
};

namespace dcsg_host {

inline int fail(dcsg_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->error = msg;
    return code;
}

#define CUDA_TRY(ctx, expr)                                                                              \
    do {                                                                                                 \
        cudaError_t e__ = (expr);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            return fail(ctx, DCSG_ERR_CUDA, format("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__))); \
    } while (0)

inline void report_progress(dcsg_ctx* ctx, int state, uint64_t done, uint64_t total) {
    if (ctx && ctx->progress) ctx->progress(ctx->progress_user, state, done, total);
}

extern std::atomic<unsigned long long> g_launches;      // kernels launched by this library (claimed as gpu_launches by bench.py); contexts on several threads count here

// every scene kernel runs 256-thread blocks; smemWords = the design's per-thread private words (Scene::private_words)
inline cudaError_t launch(cudaKernel_t k, dim3 grid, dim3 block, void** args, cudaStream_t s, int smemWords = 0) {
    ++g_launches;
    return cudaLaunchKernel((const void*)k, grid, block, args, (size_t)smemWords * 256 * 4, s);
}

// dcsg_k_project runs persistent warps that take batches of vertices from a device counter (scene_kernels.cuh); `slot`
// picks one of 16 counters so that launches queued back to back on one stream (the file pipeline's chunks) do not share.
// gather_* (multi-GPU, optional): the first gather_count vertices are also stored to these arrays (the gathering rank's, already
// offset to this slab's first vertex)
// list_offset: where this launch's part of the exact phase's list starts (launches in flight at the same time must not share)
int launch_project(dcsg_ctx* ctx, float* d_vertices, unsigned long long count, int gd_steps, float* d_normals, cudaStream_t stream, int slot = 0,
                   float* gather_vertices = nullptr, float* gather_normals = nullptr, unsigned long long gather_count = 0,
                   unsigned long long list_offset = 0);

// Lattice geometry shared by dcsg_sample_lattice and dcsg_extract.
struct LatticeSetup {
    int L, N, P, pitch, z0, nzc, nzp;
    uint32_t planeWords;
    std::vector<float> px, py, pz;      // ISV3D64::getPoint per axis (reference ISV.hpp:103-108)
    float leafThr;
    float coarseThr[16];
    uint32_t thickMask;                 // octree levels whose nodes are thicker than the slab
};

// host_extract.cu
// swaps corners 1 and 2 of the inward-facing triangles (dcsg_mesh_orient); a no-op on an oriented mesh
int orient_locked(dcsg_ctx* ctx, dcsg_mesh* mesh);
int setup_lattice(dcsg_ctx* ctx, const float* box, int grid_level, int z0, int z1, LatticeSetup& s, bool check);
int run_lattice(dcsg_ctx* ctx, const LatticeSetup& s, float* d_values, dcsg_lattice_params& lp);

// Pool of host threads behind the file pipeline.  Two kinds of jobs:
//   write   a byte range of pinned host memory -> pwrite at a file offset (in pieces of 8 MiB so that several threads share
//           one range): file chunks are written while later chunks are still on their way from the device;
//   expand  a run of triangles that came over the link as float soup (36 B per triangle) -> the PLY vertex rows (9 doubles,
//           reference utils.hpp:117-123) and STL records (zero normal, A B C as x z y, zero attribute: utils.hpp:59-99) in
//           the pinned file image, then the writes of those rows.  The device -> host link bounds the export (122 B per
//           triangle as finished rows); rows the host expands cost the link 36 B.
class FileSink {
public:
    explicit FileSink(int threads) {
        for (int i = 0; i < threads; i++) workers_.emplace_back([this] { run(); });
    }
    ~FileSink() { finish(); }
    void submit(int fd, const uint8_t* data, size_t size, uint64_t offset) {
        if (fd < 0 || !size) return;
        const size_t piece = (size_t)8 << 20;
        std::lock_guard<std::mutex> g(m_);
        for (size_t done = 0; done < size; done += piece) {
            Job job;
            job.fd = fd; job.data = data + done; job.size = std::min(piece, size - done); job.offset = offset + done;
            jobs_.push_back(job);
        }
        cv_.notify_all();
    }
    // soup: 9 floats per triangle; plyRows / stlRecords: where the rows of the run's first triangle go in the file image;
    // fdPly / fdStl (-1: none) + offsets: where they go in the files; acb: STL records list the corners A, C, B (stl_words)
    void submit_expand(const float* soup, uint64_t tris, uint8_t* plyRows, uint8_t* stlRecords, int fdPly, uint64_t offsetPly, int fdStl,
                       uint64_t offsetStl, bool acb) {
        if (!tris) return;
        const uint64_t piece = 32768;
        std::lock_guard<std::mutex> g(m_);
        for (uint64_t done = 0; done < tris; done += piece) {
            Job job;
            job.soup = soup + done * 9; job.tris = std::min(piece, tris - done);
            job.plyRows = plyRows + done * 72; job.stlRecords = stlRecords + done * 50;
            job.fd = fdPly; job.offset = offsetPly + done * 72; job.fdStl = fdStl; job.offsetStl = offsetStl + done * 50;
            job.acb = acb;
            jobs_.push_back(job);
        }
        cv_.notify_all();
    }
    bool finish() {             // waits for the queue to drain and joins the workers; false if any write failed
        {
            std::lock_guard<std::mutex> g(m_);
            closing_ = true;
            cv_.notify_all();
        }
        for (auto& t : workers_) if (t.joinable()) t.join();
        workers_.clear();
        return !failed_;
    }
    // The rows are written once and read by nobody on this core (the file writers / the caller come later): non-temporal
    // stores keep the host from first READING every destination line (a plain store to uncached memory costs a
    // read-for-ownership), which matters because host memory traffic -- DMA writes included -- is what bounds the export.
    // acb: the corners in the order A, C, B -- an outward-wound mesh, which the (x, z, y) axis order would otherwise mirror
    static void stl_words(const float* s, uint32_t rec[12], bool acb) {
        rec[0] = rec[1] = rec[2] = 0u;
        for (int v = 0; v < 3; v++) {
            const float* c = s + (acb && v ? 3 - v : v) * 3;
            memcpy(&rec[3 + v * 3 + 0], &c[0], 4);
            memcpy(&rec[3 + v * 3 + 1], &c[2], 4);
            memcpy(&rec[3 + v * 3 + 2], &c[1], 4);
        }
    }
    static void expand_rows(const float* soup, uint64_t tris, uint8_t* plyRows, uint8_t* stlRecords, bool acb) {
        long long* rows = reinterpret_cast<long long*>(plyRows);    // 72-byte rows in a 256-byte aligned image: 8-byte aligned
        for (uint64_t i = 0; i < tris; i++) {
            const float* s = soup + i * 9;
            for (int k = 0; k < 9; k++) {
                const double d = (double)s[k];
                long long bits;
                memcpy(&bits, &d, 8);
                _mm_stream_si64(rows + i * 9 + k, bits);
            }
        }
        // STL records are 50 bytes: two of them are 25 aligned words when the run starts on an even record of the file
        uint64_t i = 0;
        if ((reinterpret_cast<uintptr_t>(stlRecords) & 3u) == 0) {
            for (; i + 2 <= tris; i += 2) {
                uint32_t a[12], b[12];
                stl_words(soup + i * 9, a, acb);
                stl_words(soup + (i + 1) * 9, b, acb);
                int* out = reinterpret_cast<int*>(stlRecords + i * 50);
                for (int k = 0; k < 12; k++) _mm_stream_si32(out + k, (int)a[k]);
                _mm_stream_si32(out + 12, (int)(b[0] << 16));                   // attribute of the first (0) | low half of b[0]
                for (int k = 1; k < 12; k++) _mm_stream_si32(out + 12 + k, (int)((b[k - 1] >> 16) | (b[k] << 16)));
                _mm_stream_si32(out + 24, (int)(b[11] >> 16));                  // high half of b[11] | attribute of the second (0)
            }
        }
        for (; i < tris; i++) {
            uint32_t rec[12];
            stl_words(soup + i * 9, rec, acb);
            uint8_t* r = stlRecords + i * 50;
            memcpy(r, rec, 48);
            r[48] = r[49] = 0;
        }
        _mm_sfence();
    }
private:
    struct Job {
        int fd = -1; const uint8_t* data = nullptr; size_t size = 0; uint64_t offset = 0;
        const float* soup = nullptr; uint64_t tris = 0; uint8_t* plyRows = nullptr; uint8_t* stlRecords = nullptr; int fdStl = -1; uint64_t offsetStl = 0;
        bool acb = false;
    };
    bool write_all(int fd, const uint8_t* data, size_t size, uint64_t offset) {
        size_t done = 0;
        while (done < size) {
            const ssize_t w = pwrite(fd, data + done, size - done, (off_t)(offset + done));
            if (w <= 0) return false;
            done += (size_t)w;
        }
        return true;
    }
    void run() {
        for (;;) {
            Job job;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [this] { return closing_ || !jobs_.empty(); });
                if (jobs_.empty()) return;
                job = jobs_.front();
                jobs_.pop_front();
            }
            if (job.soup) {
                expand_rows(job.soup, job.tris, job.plyRows, job.stlRecords, job.acb);
                if (job.fd >= 0 && !write_all(job.fd, job.plyRows, job.tris * 72, job.offset)) failed_ = true;
                if (job.fdStl >= 0 && !write_all(job.fdStl, job.stlRecords, job.tris * 50, job.offsetStl)) failed_ = true;
            } else if (!write_all(job.fd, job.data, job.size, job.offset)) {
                failed_ = true;
            }
        }
    }
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<Job> jobs_;
    std::vector<std::thread> workers_;
    bool closing_ = false;
    bool failed_ = false;
};

struct MeshStorage {        // owned by a dcsg_mesh through `reserved`
    DevBuf vertices, normals, keys, triangles, cell_ids, cell_masks;
    HostBuf host;
    // Everything the chunked file pipeline (dcsg_project_and_format_segments) cuts a mesh by is kept here, in the mesh, not in
    // the context: a mesh can be projected and written after later extractions on its context.
    bool uniform = false;
    // uniform extractions: triangles before each of the slab's own cell layers and vertices before each of its sample planes
    // (own planes, then the halo plane), closed by the totals -- what the chunked file pipeline cuts the mesh by
    std::vector<uint64_t> layerTriFirst, planeVertFirst;
    // adaptive extractions: the mesh is a sequence of equal units -- a soup triangle (1 triangle, 3 vertices) or the strip
    // cms::retopologize makes of one (3p - 2 triangles on 3p vertices) -- and a unit's triangles only use its own vertices
    uint64_t unitTriangles = 0, unitVertices = 0;
    std::vector<uint64_t> levelTriangles;   // adaptive: triangles per octree level (the mesh is ordered level by level)
    // Where this mesh's triangles sit in the whole mesh of a sharded export: runs {local first, count, global first}.  Empty =
    // one run starting at the caller's first_triangle.  (Adaptive slabs: one run per octree level.)
    struct Run { uint64_t local, count, global; };
    std::vector<Run> runs;
    // Outward winding (dcsg_mesh_orient).  cellUnit: consecutive triangles per table triangle of a cell (1, or the 3p - 2 of a
    // retopologized strip); set by the extraction and, unlike unitTriangles, kept by the weld.  0 = the cells do not describe
    // the triangles.  oriented: the triangles face outwards; the STL writers then list the corners A, C, B.
    uint64_t cellUnit = 0;
    bool oriented = false;
};


// host_files.cu
std::string ply_header(uint64_t tris);
std::string stl_header(uint64_t tris);
// creates the file at its final size with the header in place; returns the descriptor or -1
int create_sized_file(const char* path, const std::string& header, uint64_t total_bytes);
// FileSink threads for the file pipelines (DCSG_HOST_THREADS)
int host_threads(const dcsg_ctx* ctx);

// host_indexed.cu
std::string indexed_ply_header(uint64_t vertices, uint64_t triangles, bool normals);
// merges the vertices of equal positions (adaptive meshes; a lattice mesh is returned unchanged)
int weld_locked(dcsg_ctx* ctx, dcsg_mesh* mesh);
// Where a mesh's rows go in the indexed file: vertex rows [0, vertices) of the mesh at vertexOffset, all its face rows (ids +
// base) at faceOffset.
struct IndexedTarget {
    int fd;
    uint64_t vertexOffset, faceOffset;
    uint32_t base;
    uint64_t vertices;
};
// gd_steps >= 0: project the vertices (and compute the normals) chunk by chunk, pipelined with the copies and the writes;
// gd_steps < 0: the mesh is final (its d_normals are written)
int indexed_pipeline_locked(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, bool normals, const IndexedTarget& t);

// host_comm.cu
dcsg_ctx* comm_ctx(const dcsg_comm* c);

// host_context.cu
// dcsg_k_eval_sdf / dcsg_k_eval_normal on n device points, asynchronous on the context's stream (the scene is built)
int eval_device_locked(dcsg_ctx* ctx, cudaKernel_t k, const float* d_xyz, size_t n, float* d_out);
int bbox_locked(dcsg_ctx* ctx, float search_diameter, float* box6, int ixBegin, int ixEnd,
                int (*reduce)(void* user, int* d_minmax, uint32_t* d_hist, cudaStream_t stream), void* reduce_user);
int plan_slabs_locked(dcsg_ctx* ctx, const float* box6, int grid_level, int world, int granularity, int* bounds);

}  // namespace dcsg_host
