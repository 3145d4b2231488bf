// host_files.cu -- byte-exact STL / PLY (reference cms/main/Headers/utils.hpp:41-154, master/happly.h), the projection /
// format / device-to-host / file-write pipeline, and the one driver behind dcsg_export, dcsg_export_sharded,
// dcsg_export_indexed and dcsg_export_sharded_indexed (MyFrame::OnExportInner end to end).
#include "host_internal.h"

using namespace dcsg_host;

// Builds the scene and reads exportConfig.txt, positional (reference DesignCSG.cpp:827-835), with the export's fixed choices:
// retopologize, the level override, the projection deferred to the file pipeline.
static int export_config(dcsg_ctx* ctx, const char* scene_dir, int grid_level_override, dcsg_extract_cfg& cfg, float& search) {
    const int rc = dcsg_build(ctx, scene_dir, nullptr, 0);
    if (rc != DCSG_OK) return rc;
    const std::vector<std::string>& ec = ctx->scene.export_config;
    if (ec.size() < 6) return fail(ctx, DCSG_ERR_INVALID, "exportConfig.txt needs at least 6 lines");
    // The reference feeds the lines to std::stof / std::stoi (which throw on garbage); nothing may be thrown across the
    // C ABI, so the same leading-number syntax is parsed with strtof / strtol and a bad line is DCSG_ERR_INVALID.
    float fv[6];
    long iv[6];
    for (int i = 0; i < 6; i++) {
        const char* text = ec[i].c_str();
        char* end = nullptr;
        errno = 0;
        if (i == 0 || i == 4) { fv[i] = strtof(text, &end); iv[i] = 0; }
        else { iv[i] = strtol(text, &end, 10); fv[i] = 0.0f; }
        if (end == text || errno == ERANGE || (i != 0 && i != 4 && (iv[i] < INT_MIN || iv[i] > INT_MAX)))
            return fail(ctx, DCSG_ERR_INVALID, format("exportConfig.txt line %d is not a number: '%.40s'", i + 1, text));
    }
    search = fv[0];
    if (!(search > 0.0f) || !std::isfinite(search)) return fail(ctx, DCSG_ERR_INVALID, "exportConfig.txt line 1: the search diameter must be positive");
    memset(&cfg, 0, sizeof(cfg));
    cfg.min_level = (int)iv[1];
    cfg.max_level = (int)iv[2];
    cfg.grid_level = (int)iv[3];
    cfg.complex_threshold = fv[4];
    cfg.gd_steps = (int)iv[5];
    cfg.retopologize = 1;           // OnExportInner always runs cms::retopologize (DesignCSG.cpp:749)
    if (grid_level_override > 0) cfg.min_level = cfg.max_level = cfg.grid_level = grid_level_override;
    cfg.defer_projection = 1;       // the projection runs in chunks, pipelined with formatting, D2H and the file writes
    return DCSG_OK;
}

std::string dcsg_host::ply_header(uint64_t tris) {
    // happly's writeHeader (master/happly.h:1998-2040) for addVertexPositions + addFaceIndices
    return format("ply\nformat binary_little_endian 1.0\n"
                  "comment Written with hapPLY (https://github.com/nmwsharp/happly)\n"
                  "element vertex %llu\nproperty double x\nproperty double y\nproperty double z\n"
                  "element face %llu\nproperty list uchar uint vertex_indices\nend_header\n",
                  (unsigned long long)(tris * 3), (unsigned long long)tris);
}

std::string dcsg_host::stl_header(uint64_t tris) {
    // 80 zero bytes and the triangle count (reference utils.hpp:59-66)
    std::string header(84, '\0');
    const uint32_t count = (uint32_t)tris;
    memcpy(&header[80], &count, 4);
    return header;
}

int dcsg_host::create_sized_file(const char* path, const std::string& header, uint64_t total_bytes) {
    const int fd = open(path, O_RDWR | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return -1;
    if (ftruncate(fd, (off_t)total_bytes) != 0 || pwrite(fd, header.data(), header.size(), 0) != (ssize_t)header.size()) {
        close(fd);
        return -1;
    }
    return fd;
}

int dcsg_host::host_threads(const dcsg_ctx* ctx) {
    const char* e = getenv("DCSG_HOST_THREADS");
    const int cores = (int)std::max(4u, std::thread::hardware_concurrency());
    const int n = e ? atoi(e) : std::min(16, std::max(2, cores / std::max(1, ctx->node_ranks)));
    return std::max(1, std::min(64, n));
}

// An outward-wound mesh (dcsg_mesh_orient) lists its STL corners A, C, B: the records store every corner as (x, z, y), and
// that swap of two axes would turn the winding inside out again.  Meshes the library does not own are written as they are.
static bool stl_acb(const dcsg_mesh* mesh) {
    const MeshStorage* st = (const MeshStorage*)mesh->reserved;
    return st && st->oriented;
}

extern "C" {
// Lay the file out in pinned host memory: header bytes by the host, body by the device kernels.
static int format_locked(dcsg_ctx* ctx, const dcsg_mesh* mesh, bool ply, uint8_t** bytes, size_t* size) {
    const uint64_t n = mesh->num_triangles;
    if (ply && n * 3 > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "PLY soup indices exceed 32 bits (happly.h:1654-1662)");
    const std::string header = ply ? ply_header(n) : stl_header(n);
    const size_t body = ply ? n * 72 + n * 13 : n * 50;
    const size_t total = header.size() + body;
    CUDA_TRY(ctx, ctx->pinned.reserve(total + 64));
    CUDA_TRY(ctx, ctx->fmt.reserve(body + 64));
    uint8_t* h = ctx->pinned.as<uint8_t>();
    memcpy(h, header.data(), header.size());
    if (n) {
        uint8_t* d = ctx->fmt.as<uint8_t>();
        if (ply) {
            dcsg_launch_format_ply_vertices(mesh->d_vertices, mesh->d_triangles, n, (double*)d, ctx->stream);
            dcsg_launch_format_ply_faces(0, n, d + n * 72, ctx->stream); g_launches += 2;
        } else {
            dcsg_launch_format_stl(mesh->d_vertices, mesh->d_triangles, n, d, stl_acb(mesh), ctx->stream); ++g_launches;
        }
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(h + header.size(), d, body, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    *bytes = h;
    *size = total;
    return DCSG_OK;
}

int dcsg_format_segments(dcsg_ctx* ctx, const dcsg_mesh* mesh, uint64_t first_triangle, const uint8_t** ply_vertex_rows,
                         const uint8_t** ply_face_rows, const uint8_t** stl_records) {
    if (!ctx || !mesh || !ply_vertex_rows || !ply_face_rows || !stl_records) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t n = mesh->num_triangles;
    if ((first_triangle + n) * 3 > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "PLY soup indices exceed 32 bits (happly.h:1654-1662)");
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t offFaces = align(n * 72), offStl = offFaces + align(n * 13), total = offStl + align(n * 50);
    CUDA_TRY(ctx, ctx->pinned.reserve(total + 64));
    CUDA_TRY(ctx, ctx->fmt.reserve(total + 64));
    uint8_t* h = ctx->pinned.as<uint8_t>();
    uint8_t* d = ctx->fmt.as<uint8_t>();
    if (n) {
        dcsg_launch_format_ply_vertices(mesh->d_vertices, mesh->d_triangles, n, (double*)d, ctx->stream);
        dcsg_launch_format_ply_faces(first_triangle, n, d + offFaces, ctx->stream);
        dcsg_launch_format_stl(mesh->d_vertices, mesh->d_triangles, n, d + offStl, stl_acb(mesh), ctx->stream);
        g_launches += 3;
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(h, d, n * 72, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(h + offFaces, d + offFaces, n * 13, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(h + offStl, d + offStl, n * 50, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    *ply_vertex_rows = h;
    *ply_face_rows = h + offFaces;
    *stl_records = h + offStl;
    return DCSG_OK;
}

// Projection pipelined with the file formatters and the device -> host copies.  Triangles are in cell order and vertices
// in key order, both z-major, so the mesh is cut into chunks of about equal triangle count on tile boundaries of the
// cell bitmap: chunk c needs the vertices of all lattice planes up to the one above its last cell layer.  Per chunk:
// project its new vertices, format its triangles (compute stream), then copy the three byte ranges (copy stream) while
// the next chunk is being projected.  The PLY face rows do not come from the device at all (FaceRowFill).
// With a sink, every chunk that has reached pinned memory is handed to the writer threads (files: fdPly / fdStl, this
// rank's rows start at triangle first_triangle of total_triangles).
// PLY face rows written by host threads (see pipeline_locked); joins on destruction, so every early return is safe.
class FaceRowFill {
    std::vector<std::thread> workers;
    static void rows(uint8_t* out, uint64_t first, uint64_t lo, uint64_t hi) {
        uint8_t* o = out + lo * 13;
        uint64_t i = lo;
        // four rows are 13 words: streamed past the cache where the run is word aligned (see FileSink::expand_rows)
        if ((reinterpret_cast<uintptr_t>(o) & 3u) == 0) {
            for (; i + 4 <= hi; i += 4, o += 52) {
                uint8_t block[52];
                for (int r = 0; r < 4; r++) {
                    const uint32_t base = (uint32_t)((first + i + r) * 3);
                    const uint32_t idx[3] = {base, base + 1u, base + 2u};
                    block[r * 13] = 3;
                    memcpy(block + r * 13 + 1, idx, 12);
                }
                int words[13];
                memcpy(words, block, 52);
                for (int k = 0; k < 13; k++) _mm_stream_si32(reinterpret_cast<int*>(o) + k, words[k]);
            }
            _mm_sfence();
        }
        for (; i < hi; i++, o += 13) {
            const uint32_t base = (uint32_t)((first + i) * 3);
            const uint32_t idx[3] = {base, base + 1u, base + 2u};
            o[0] = 3;
            memcpy(o + 1, idx, 12);         // little-endian host, like the reference's (happly writes native byte order)
        }
    }
public:
    FaceRowFill(uint8_t* out, uint64_t first, uint64_t n) {
        const uint64_t threads = std::max<uint64_t>(1, std::min<uint64_t>(4, n / 500000));
        for (uint64_t t = 0; t < threads && n; t++) {
            const uint64_t lo = n * t / threads, hi = n * (t + 1) / threads;
            try {
                workers.emplace_back(rows, out, first, lo, hi);
            } catch (...) {                 // no thread to be had: fill the range here (no exception crosses the C ABI)
                rows(out, first, lo, hi);
            }
        }
    }
    void join() {
        for (auto& w : workers) w.join();
        workers.clear();
    }
    ~FaceRowFill() { join(); }
};

// Share of the triangles whose file rows the host expands from float soup (DCSG_HOST_EXPAND_PERMILLE, 0 .. 1000) and the
// number of host threads behind the pipeline (DCSG_HOST_THREADS).  Measured on this pool's box (16 vCPU, one B200,
// tools/e2e_probe.py, 24 vCPU): finished rows for every triangle 23.8 ms, 60 % of them expanded by the host 19.3, all of
// them 25 -- the host's memory system is the limit either way (1.18 GB of file image must land in it), so the default gives
// the host 60 % on a single-GPU host and leaves everything to the device when several ranks share the host's cores.
static int host_expand_permille(const dcsg_ctx* ctx) {
    const char* e = getenv("DCSG_HOST_EXPAND_PERMILLE");        // read per call: a handful of calls per export
    return e ? atoi(e) : (ctx->node_ranks > 1 ? 0 : 600);
}

struct FileTargets { FileSink* sink; int fdPly, fdStl; uint64_t totalTriangles; size_t plyHeader; };

static int pipeline_locked(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, uint64_t first_triangle, const uint8_t** ply_vertex_rows,
                           const uint8_t** ply_face_rows, const uint8_t** stl_records, const FileTargets* files) {
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    MeshStorage* st = (MeshStorage*)mesh->reserved;
    if (st->uniform ? st->layerTriFirst.empty() : st->unitTriangles == 0)
        return fail(ctx, DCSG_ERR_INVALID, "the projection / file pipeline needs a mesh from dcsg_extract (defer_projection)");
    const uint64_t n = mesh->num_triangles, nVerts = mesh->num_vertices;
    if ((first_triangle + n) * 3 > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "PLY soup indices exceed 32 bits (happly.h:1654-1662)");
    for (const MeshStorage::Run& r : st->runs)
        if ((r.global + r.count) * 3 > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "PLY soup indices exceed 32 bits (happly.h:1654-1662)");
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t offFaces = align(n * 72), offStl = offFaces + align(n * 13), total = offStl + align(n * 50);
    CUDA_TRY(ctx, ctx->pinned.reserve(total + 64));
    CUDA_TRY(ctx, ctx->fmt.reserve(total + 64));
    uint8_t* h = ctx->pinned.as<uint8_t>();
    uint8_t* d = ctx->fmt.as<uint8_t>();
    if (ply_vertex_rows) *ply_vertex_rows = h;
    if (ply_face_rows) *ply_face_rows = h + offFaces;
    if (stl_records) *stl_records = h + offStl;
    if (!n) return DCSG_OK;
    if (!ctx->copy_stream) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (auto& ev : ctx->chunk_event) if (!ev) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    for (auto& ev : ctx->copied_event) if (!ev) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaStream_t cs = ctx->stream, ds = ctx->copy_stream;

    // The face rows of a triangle soup hold no information from the device: row i is the byte 3 followed by the indices
    // 3i, 3i+1, 3i+2 (reference utils.hpp:131-141 through happly.h:1640-1668), a function of the triangle COUNT alone.
    // The device -> host link is what bounds this pipeline (1.18 GB per 1024^3 export at ~52 GB/s), so these 13 of the
    // 135 bytes per triangle are written straight into the pinned buffer by a few host threads while the device
    // projects and the copy engine moves the rows that do come from the device.
    // where this mesh's triangles sit in the whole mesh: one run from first_triangle, or -- a slab of an adaptive walk in a
    // sharded export -- one run per octree level (MeshStorage::runs)
    std::vector<MeshStorage::Run> runs = st->runs;
    if (runs.empty()) runs.push_back(MeshStorage::Run{0, n, first_triangle});
    // pieces of the local range [t0, t1) with their global first triangle
    auto for_each_piece = [&runs](uint64_t t0, uint64_t t1, const std::function<void(uint64_t, uint64_t, uint64_t)>& f) {
        for (const MeshStorage::Run& r : runs) {
            const uint64_t a = std::max(t0, r.local), b = std::min(t1, r.local + r.count);
            if (a < b) f(a, b - a, r.global + (a - r.local));
        }
    };
    std::vector<std::unique_ptr<FaceRowFill>> faces;
    for (const MeshStorage::Run& r : runs) faces.emplace_back(new FaceRowFill(h + offFaces + r.local * 13, r.global, r.count));
    auto join_faces = [&faces] { for (auto& f : faces) f->join(); };
    // Of every chunk, the first part leaves the device as finished rows (122 B per triangle over the link), the rest as
    // float soup (36 B) that host threads expand into the same rows (FileSink::submit_expand): the link and the host's
    // cores work side by side.  host_expand_permille = the share of the triangles the host expands.
    const uint64_t hostPermille = (uint64_t)std::max(0, std::min(1000, host_expand_permille(ctx)));
    struct Range { uint64_t tri0, split, tri1; };       // [tri0, split) formatted on the device, [split, tri1) expanded on the host
    std::vector<Range> ranges;
    float* d_soup = nullptr;
    float* h_soup = nullptr;
    if (hostPermille) {
        const size_t soupBytes = (size_t)(n * hostPermille / 1000 + 64) * 36;
        CUDA_TRY(ctx, ctx->soup.reserve(soupBytes));
        CUDA_TRY(ctx, ctx->pinned_soup.reserve(soupBytes));
        d_soup = ctx->soup.as<float>();
        h_soup = ctx->pinned_soup.as<float>();
    }
    uint64_t soupDone = 0;                               // triangles in the soup staging buffers so far
    std::vector<uint64_t> soupFirst;
    FileSink* pool = files ? files->sink : nullptr;
    std::unique_ptr<FileSink> ownPool;
    if (hostPermille && !pool) { ownPool.reset(new FileSink(host_threads(ctx))); pool = ownPool.get(); }

    // chunk boundaries on cell layers: dcsg_extract counted the triangles of every layer and the vertices of every plane
    const std::vector<uint64_t>& layerFirst = st->layerTriFirst;        // [own layers + 1]
    const std::vector<uint64_t>& planeFirst = st->planeVertFirst;       // [own planes (+ halo plane) + 1]
    const int chunks = (int)std::max<uint64_t>(1, std::min<uint64_t>(12, n / 200000));
    uint64_t triDone = 0, vertDone = 0;
    float* d_normals = nullptr;
    for (int c = 0; c < chunks; c++) {
        uint64_t triEnd = n, vertEnd = nVerts;
        if (c + 1 < chunks) {
            const uint64_t target = n * (uint64_t)(c + 1) / chunks;
            if (st->uniform) {
                // layers [0, b) are complete in this chunk: the last layer boundary with at most `target` triangles before it
                const size_t b = (size_t)(std::upper_bound(layerFirst.begin(), layerFirst.end(), target) - layerFirst.begin()) - 1;
                triEnd = layerFirst[b] & ~3ull;                             // format kernels work on groups of 4 / 2 triangles
                vertEnd = planeFirst[std::min(b + 1, planeFirst.size() - 1)];   // layer i's triangles use the planes i and i + 1
            } else {
                // adaptive walk: the mesh is a sequence of units (a soup triangle, or the strip cms::retopologize makes of
                // one) whose triangles only use the unit's own vertices; cut on a multiple of four units
                const uint64_t units = (target / st->unitTriangles) & ~3ull;
                triEnd = units * st->unitTriangles;
                vertEnd = units * st->unitVertices;
            }
            if (triEnd < triDone) triEnd = triDone;
            if (vertEnd < vertDone) vertEnd = vertDone;
        }
        if (vertEnd > vertDone && gd_steps > 0) {
            if (int rc = launch_project(ctx, mesh->d_vertices + vertDone * 3, vertEnd - vertDone, gd_steps, d_normals, cs, c, nullptr, nullptr, 0, vertDone)) return rc;
        }
        vertDone = vertEnd;
        if (triEnd > triDone) {
            const uint64_t hostTris = std::min<uint64_t>(((triEnd - triDone) * hostPermille / 1000) & ~3ull, n * hostPermille / 1000 - soupDone);
            const uint64_t split = triEnd - hostTris, m = split - triDone;
            if (m) {
                dcsg_launch_format_ply_vertices(mesh->d_vertices, mesh->d_triangles + triDone * 3, m, (double*)(d + triDone * 72), cs);
                dcsg_launch_format_stl(mesh->d_vertices, mesh->d_triangles + triDone * 3, m, d + offStl + triDone * 50, st->oriented, cs);
                g_launches += 2;
            }
            if (hostTris) { dcsg_launch_expand_soup(mesh->d_vertices, mesh->d_triangles + split * 3, hostTris, d_soup + soupDone * 9, cs); ++g_launches; }
            CUDA_TRY(ctx, cudaGetLastError());
            CUDA_TRY(ctx, cudaEventRecord(ctx->chunk_event[c], cs));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ds, ctx->chunk_event[c], 0));
            if (hostTris) CUDA_TRY(ctx, cudaMemcpyAsync(h_soup + soupDone * 9, d_soup + soupDone * 9, hostTris * 36, cudaMemcpyDeviceToHost, ds));
            if (m) {
                CUDA_TRY(ctx, cudaMemcpyAsync(h + triDone * 72, d + triDone * 72, m * 72, cudaMemcpyDeviceToHost, ds));
                CUDA_TRY(ctx, cudaMemcpyAsync(h + offStl + triDone * 50, d + offStl + triDone * 50, m * 50, cudaMemcpyDeviceToHost, ds));
            }
            CUDA_TRY(ctx, cudaEventRecord(ctx->copied_event[ranges.size()], ds));
            ranges.push_back(Range{triDone, split, triEnd});
            soupFirst.push_back(soupDone);
            soupDone += hostTris;
        }
        triDone = triEnd;
    }
    // everything is queued on the device; feed the host threads as the chunks land in pinned memory
    const int fdPly = files ? files->fdPly : -1, fdStl = files ? files->fdStl : -1;
    const uint64_t plyRows = files ? files->plyHeader : 0, plyFaces = files ? files->plyHeader + 72 * files->totalTriangles : 0, stlRecords = 84;
    if (files) {
        join_faces();
        for (const MeshStorage::Run& r : runs) files->sink->submit(fdPly, h + offFaces + r.local * 13, r.count * 13, plyFaces + 13 * r.global);
    }
    if (pool) {
        for (size_t c = 0; c < ranges.size(); c++) {
            CUDA_TRY(ctx, cudaEventSynchronize(ctx->copied_event[c]));
            const uint64_t t0 = ranges[c].tri0, split = ranges[c].split;
            const float* soup = h_soup + soupFirst[c] * 9;
            for_each_piece(split, ranges[c].tri1, [&](uint64_t a, uint64_t count, uint64_t global) {
                pool->submit_expand(soup + (a - split) * 9, count, h + a * 72, h + offStl + a * 50, fdPly, plyRows + 72 * global, fdStl,
                                    stlRecords + 50 * global, st->oriented);
            });
            if (files) {
                for_each_piece(t0, split, [&](uint64_t a, uint64_t count, uint64_t global) {
                    pool->submit(fdPly, h + a * 72, count * 72, plyRows + 72 * global);
                    pool->submit(fdStl, h + offStl + a * 50, count * 50, stlRecords + 50 * global);
                });
                if (c == 0) report_progress(ctx, DCSG_PROGRESS_GRADIENT_DESCENT, (uint64_t)std::max(gd_steps, 0), (uint64_t)std::max(gd_steps, 0));
                report_progress(ctx, DCSG_PROGRESS_WRITING_STL, ranges[c].tri1, n);     // both files are written chunk by chunk
            }
        }
        if (files) report_progress(ctx, DCSG_PROGRESS_WRITING_PLY, n, n);
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ds));
    CUDA_TRY(ctx, cudaStreamSynchronize(cs));
    join_faces();
    if (ownPool && !ownPool->finish()) return fail(ctx, DCSG_ERR_IO, "host expansion failed");
    return DCSG_OK;
}

int dcsg_project_and_format_segments(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, uint64_t first_triangle,
                                     const uint8_t** ply_vertex_rows, const uint8_t** ply_face_rows, const uint8_t** stl_records) {
    if (!ctx || !mesh || !mesh->reserved || !ply_vertex_rows || !ply_face_rows || !stl_records) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    return pipeline_locked(ctx, mesh, gd_steps, first_triangle, ply_vertex_rows, ply_face_rows, stl_records, nullptr);
}

int dcsg_project_and_write_files(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, uint64_t first_triangle, uint64_t total_triangles,
                                 int create_files, const char* stl_path, const char* ply_path) {
    if (!ctx || !mesh || !mesh->reserved) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (first_triangle + mesh->num_triangles > total_triangles) return fail(ctx, DCSG_ERR_INVALID, "triangle range exceeds the total");
    const std::string plyHeader = ply_header(total_triangles);
    // create_files: the files at their final size with the headers in place (reference utils.hpp:59-66, happly.h:1998-2040)
    auto open_file = [&](const char* path, const std::string& header, uint64_t rowBytes) {
        return create_files ? create_sized_file(path, header, header.size() + rowBytes * total_triangles) : open(path, O_RDWR);
    };
    int fdPly = -1, fdStl = -1;
    if (ply_path && (fdPly = open_file(ply_path, plyHeader, 85)) < 0) return fail(ctx, DCSG_ERR_IO, std::string("cannot open ") + ply_path);
    if (stl_path && (fdStl = open_file(stl_path, stl_header(total_triangles), 50)) < 0) {
        if (fdPly >= 0) close(fdPly);
        return fail(ctx, DCSG_ERR_IO, std::string("cannot open ") + stl_path);
    }
    int rc;
    bool ok;
    {
        FileSink sink(host_threads(ctx));
        FileTargets files{&sink, fdPly, fdStl, total_triangles, plyHeader.size()};
        rc = pipeline_locked(ctx, mesh, gd_steps, first_triangle, nullptr, nullptr, nullptr, &files);
        ok = sink.finish();
    }
    if (fdPly >= 0) close(fdPly);
    if (fdStl >= 0) close(fdStl);
    if (rc != DCSG_OK) return rc;
    return ok ? DCSG_OK : fail(ctx, DCSG_ERR_IO, "short write");
}


int dcsg_ply_face_rows(uint64_t first_triangle, uint64_t num_triangles, uint8_t* out, size_t capacity) {
    if (!out || capacity < num_triangles * 13) return DCSG_ERR_INVALID;
    if ((first_triangle + num_triangles) * 3 > 0xffffffffull) return DCSG_ERR_INVALID;      // happly.h:1654-1662
    FaceRowFill fill(out, first_triangle, num_triangles);
    fill.join();
    return DCSG_OK;
}

int dcsg_soup_rows(const float* soup, uint64_t num_triangles, uint8_t* ply_rows, uint8_t* stl_records) {
    if (!soup || !ply_rows || !stl_records || (reinterpret_cast<uintptr_t>(ply_rows) & 7u)) return DCSG_ERR_INVALID;
    FileSink::expand_rows(soup, num_triangles, ply_rows, stl_records, false);
    return DCSG_OK;
}

int dcsg_file_header(int ply, uint64_t total_triangles, uint8_t* out, size_t capacity, size_t* needed) {
    const std::string header = ply ? ply_header(total_triangles) : stl_header(total_triangles);
    if (needed) *needed = header.size();
    if (!out) return DCSG_OK;
    if (capacity < header.size()) return DCSG_ERR_INVALID;
    memcpy(out, header.data(), header.size());
    return DCSG_OK;
}

static int format_api(dcsg_ctx* ctx, const dcsg_mesh* mesh, bool ply, uint8_t* out, size_t capacity, size_t* needed) {
    if (!ctx || !mesh) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t n = mesh->num_triangles;
    const size_t total = ply ? ply_header(n).size() + n * 85 : 84 + n * 50;
    if (needed) *needed = total;
    if (!out) return DCSG_OK;
    if (capacity < total) return fail(ctx, DCSG_ERR_INVALID, "output buffer too small");
    uint8_t* bytes;
    size_t size;
    int rc = format_locked(ctx, mesh, ply, &bytes, &size);
    if (rc != DCSG_OK) return rc;
    memcpy(out, bytes, size);
    return DCSG_OK;
}

static int view_api(dcsg_ctx* ctx, const dcsg_mesh* mesh, bool ply, const uint8_t** bytes, size_t* size) {
    if (!ctx || !mesh || !bytes || !size) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    uint8_t* b = nullptr;
    int rc = format_locked(ctx, mesh, ply, &b, size);
    *bytes = b;
    return rc;
}
int dcsg_format_stl_view(dcsg_ctx* ctx, const dcsg_mesh* mesh, const uint8_t** bytes, size_t* size) { return view_api(ctx, mesh, false, bytes, size); }
int dcsg_format_ply_view(dcsg_ctx* ctx, const dcsg_mesh* mesh, const uint8_t** bytes, size_t* size) { return view_api(ctx, mesh, true, bytes, size); }
unsigned long long dcsg_launch_count(void) { return g_launches.load(); }

int dcsg_format_stl(dcsg_ctx* ctx, const dcsg_mesh* mesh, uint8_t* out, size_t capacity, size_t* needed) {
    return format_api(ctx, mesh, false, out, capacity, needed);
}
int dcsg_format_ply(dcsg_ctx* ctx, const dcsg_mesh* mesh, uint8_t* out, size_t capacity, size_t* needed) {
    return format_api(ctx, mesh, true, out, capacity, needed);
}

static int write_api(dcsg_ctx* ctx, const dcsg_mesh* mesh, bool ply, const char* path) {
    if (!ctx || !mesh || !path) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    uint8_t* bytes;
    size_t size;
    int rc = format_locked(ctx, mesh, ply, &bytes, &size);
    if (rc != DCSG_OK) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ctx, DCSG_ERR_IO, std::string("cannot open ") + path);
    const size_t w = fwrite(bytes, 1, size, f);
    fclose(f);
    return w == size ? DCSG_OK : fail(ctx, DCSG_ERR_IO, std::string("short write to ") + path);
}

int dcsg_write_stl(dcsg_ctx* ctx, const dcsg_mesh* mesh, const char* path) { return write_api(ctx, mesh, false, path); }
int dcsg_write_ply(dcsg_ctx* ctx, const dcsg_mesh* mesh, const char* path) { return write_api(ctx, mesh, true, path); }

// What an export writes: the reference's soup files (a null path is skipped) or the indexed PLY.
struct ExportFiles {
    bool indexed, normals;          // normals: the indexed PLY's DCSG_PLY_NORMALS
    const char* stl_path;           // soup only
    const char* ply_path;
};

// MyFrame::OnExportInner end to end, on one GPU (comm = nullptr) or as one rank of a sharded export.  One GPU is the sharded
// export at world size 1: the slab is the whole mesh, its first vertex and triangle are 0, and nothing waits at a barrier.
// Rank 0 creates the files at their final size with the headers in place; then every rank writes its own rows at their
// offsets.  ctx->lock is never held across a barrier or a public dcsg_* call: they take it themselves.
static int run_export(dcsg_ctx* ctx, dcsg_comm* comm, const char* scene_dir, int grid_level_override, const ExportFiles& files,
                      dcsg_export_report* report) {
    if (comm && comm_ctx(comm) != ctx) return DCSG_ERR_INVALID;
    const double t0 = now_ms();
    bool outward;           // dcsg_set_export_flags, read once for the whole export
    {
        std::lock_guard<std::mutex> g(ctx->lock);
        outward = (ctx->export_flags & DCSG_EXPORT_OUTWARD) != 0;
    }
    dcsg_extract_cfg cfg;
    float search = 0.0f;
    int rc = export_config(ctx, scene_dir, grid_level_override, cfg, search);
    if (rc != DCSG_OK) return rc;
    // decided from exportConfig.txt alone, the same on every rank, before the first collective
    if (comm && files.indexed && !(cfg.min_level >= cfg.grid_level && cfg.max_level == cfg.grid_level))
        return fail(ctx, DCSG_ERR_UNSUPPORTED, "the sharded indexed export needs a uniform lattice (grid_level_override > 0): the weld of an adaptive mesh spans slabs");
    auto barrier = [&] {
        if (!comm) return;
        const int brc = dcsg_comm_barrier(comm);
        if (rc == DCSG_OK) rc = brc;
    };
    dcsg_export_report rep;
    memset(&rep, 0, sizeof(rep));
    double t = now_ms();
    report_progress(ctx, DCSG_PROGRESS_ESTIMATING_BOUNDING_BOX, 0, 0);
    rc = comm ? dcsg_bbox_sharded(ctx, comm, search, cfg.box) : dcsg_bbox(ctx, search, cfg.box);
    if (rc != DCSG_OK) return rc;
    rep.bbox_ms = (float)(now_ms() - t);
    memcpy(rep.box, cfg.box, sizeof(rep.box));
    dcsg_mesh mesh;
    memset(&mesh, 0, sizeof(mesh));
    dcsg_shard_info info;
    memset(&info, 0, sizeof(info));
    report_progress(ctx, DCSG_PROGRESS_PERFORMING_CMS, 0, 0);
    rc = comm ? dcsg_extract_sharded(ctx, comm, &cfg, -1, &mesh, nullptr, &info) : dcsg_extract(ctx, &cfg, &mesh);
    if (rc != DCSG_OK) { dcsg_mesh_free(ctx, &mesh); return rc; }
    memcpy(rep.extract_ms, mesh.stage_ms, sizeof(rep.extract_ms));
    report_progress(ctx, DCSG_PROGRESS_RETOPOLOGIZING, 0, 0);       // done inside the extraction (identity on a uniform lattice)
    t = now_ms();
    if (outward) {
        // right after the extraction, before the weld and the projection: a pure map over (cell, table slot), and every writer
        // reads the corners through the triangles
        std::lock_guard<std::mutex> g(ctx->lock);
        rc = orient_locked(ctx, &mesh);
    }
    if (!comm) {
        if (rc == DCSG_OK && files.indexed) {
            // adaptive walk: equal pre-projection positions project to equal positions and normals, so welding first projects
            // each position once and gives the same file as welding after the projection (a lattice mesh is returned unchanged)
            std::lock_guard<std::mutex> g(ctx->lock);
            rc = weld_locked(ctx, &mesh);
        }
        info.total_vertices = mesh.num_vertices;
        info.total_triangles = mesh.num_triangles;
        info.total_cells = mesh.num_cells;
    }
    const uint64_t V = info.total_vertices, T = info.total_triangles, row = files.normals ? 24 : 12;
    rep.num_vertices = V;
    rep.num_triangles = T;
    rep.num_cells = info.total_cells;
    if (rc == DCSG_OK && files.indexed && V > 0xffffffffull) rc = fail(ctx, DCSG_ERR_INVALID, "more than 2^32 vertices");
    report_progress(ctx, DCSG_PROGRESS_GRADIENT_DESCENT, 0, (uint64_t)std::max(cfg.gd_steps, 0));
    const std::string plyHeader = files.indexed ? indexed_ply_header(V, T, files.normals) : ply_header(T);
    if (rc == DCSG_OK && (!comm || dcsg_comm_rank(comm) == 0)) {
        const struct { const char* path; std::string header; uint64_t body; } made[2] = {
            {files.stl_path, stl_header(T), 50 * T}, {files.ply_path, plyHeader, files.indexed ? row * V + 13 * T : 85 * T}};
        for (const auto& f : made) {
            if (!f.path || rc != DCSG_OK) continue;
            const int fd = create_sized_file(f.path, f.header, f.header.size() + f.body);
            if (fd < 0) rc = fail(ctx, DCSG_ERR_IO, std::string("cannot create ") + f.path);
            else close(fd);
        }
    }
    barrier();
    if (rc == DCSG_OK && !files.indexed) {
        rc = dcsg_project_and_write_files(ctx, &mesh, cfg.gd_steps, info.first_triangle, T, 0, files.stl_path, files.ply_path);
    } else if (rc == DCSG_OK) {
        const int fd = open(files.ply_path, O_WRONLY);
        if (fd < 0) {
            rc = fail(ctx, DCSG_ERR_IO, std::string("cannot open ") + files.ply_path);
        } else {
            // the slab's owned vertices (the ranks' owned vertices in rank order are the whole mesh's) and its faces, ids +
            // first_vertex
            std::lock_guard<std::mutex> g(ctx->lock);
            rc = indexed_pipeline_locked(ctx, &mesh, std::max(cfg.gd_steps, 0), files.normals,
                                         IndexedTarget{fd, plyHeader.size() + row * info.first_vertex, plyHeader.size() + row * V + 13 * info.first_triangle,
                                                       (uint32_t)info.first_vertex, mesh.owned_vertices});
            close(fd);
        }
    }
    barrier();
    rep.write_ms = (float)(now_ms() - t);
    if (rc == DCSG_OK) report_progress(ctx, DCSG_PROGRESS_COMPLETE, T, T);
    dcsg_mesh_free(ctx, &mesh);
    rep.total_ms = (float)(now_ms() - t0);
    if (report) *report = rep;
    return rc;
}

int dcsg_export(dcsg_ctx* ctx, const char* scene_dir, int grid_level_override, const char* stl_path, const char* ply_path,
                dcsg_export_report* report) {
    if (!ctx || !scene_dir) return DCSG_ERR_INVALID;
    return run_export(ctx, nullptr, scene_dir, grid_level_override, ExportFiles{false, false, stl_path, ply_path}, report);
}

int dcsg_export_sharded(dcsg_ctx* ctx, dcsg_comm* comm, const char* scene_dir, int grid_level_override, const char* stl_path,
                        const char* ply_path, dcsg_export_report* report) {
    if (!ctx || !comm || !scene_dir) return DCSG_ERR_INVALID;
    return run_export(ctx, comm, scene_dir, grid_level_override, ExportFiles{false, false, stl_path, ply_path}, report);
}

int dcsg_export_indexed(dcsg_ctx* ctx, const char* scene_dir, int grid_level_override, int flags, const char* ply_path,
                        dcsg_export_report* report) {
    if (!ctx || !scene_dir || !ply_path || (flags & ~DCSG_PLY_NORMALS)) return DCSG_ERR_INVALID;
    return run_export(ctx, nullptr, scene_dir, grid_level_override, ExportFiles{true, (flags & DCSG_PLY_NORMALS) != 0, nullptr, ply_path}, report);
}

int dcsg_export_sharded_indexed(dcsg_ctx* ctx, dcsg_comm* comm, const char* scene_dir, int grid_level_override, int flags,
                                const char* ply_path, dcsg_export_report* report) {
    if (!ctx || !comm || !scene_dir || !ply_path || (flags & ~DCSG_PLY_NORMALS)) return DCSG_ERR_INVALID;
    return run_export(ctx, comm, scene_dir, grid_level_override, ExportFiles{true, (flags & DCSG_PLY_NORMALS) != 0, nullptr, ply_path}, report);
}

}  // extern "C"

