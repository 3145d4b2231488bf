// host_indexed.cu -- the indexed binary PLY (vertices shared between faces, optional normals): the weld of adaptive meshes,
// and the projection / format / copy / write pipeline of that file (the exports that write it: host_files.cu).
// An opt-in format beyond the reference's soup files (host_files.cu), which stay the default and unchanged.
#include "host_internal.h"

using namespace dcsg_host;

std::string dcsg_host::indexed_ply_header(uint64_t vertices, uint64_t triangles, bool normals) {
    return format("ply\nformat binary_little_endian 1.0\n"
                  "comment DesignCSG export, indexed: vertices shared between faces\n"
                  "element vertex %llu\nproperty float x\nproperty float y\nproperty float z\n%s"
                  "element face %llu\nproperty list uchar uint vertex_indices\nend_header\n",
                  (unsigned long long)vertices, normals ? "property float nx\nproperty float ny\nproperty float nz\n" : "",
                  (unsigned long long)triangles);
}

int dcsg_host::weld_locked(dcsg_ctx* ctx, dcsg_mesh* mesh) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    MeshStorage* st = (MeshStorage*)mesh->reserved;
    if (mesh->d_vertex_keys) return DCSG_OK;        // a lattice mesh holds every position once already (one per lattice edge)
    if (!st->runs.empty()) return fail(ctx, DCSG_ERR_UNSUPPORTED, "a slab of a sharded adaptive extraction cannot be welded: equal positions span slabs");
    const uint64_t n = mesh->num_vertices;
    if (n > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "more than 2^32 vertices");
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t scratch = align(dcsg_weld_scratch_bytes(n)), outBytes = align(n * 12);
    const bool normals = mesh->d_normals != nullptr;
    CUDA_TRY(ctx, ctx->weld.reserve(scratch + outBytes * (normals ? 2 : 1) + 256));
    uint8_t* w = ctx->weld.as<uint8_t>();
    dcsg_weld_params p;
    p.vertices = mesh->d_vertices;
    p.normals = mesh->d_normals;
    p.triangles = mesh->d_triangles;
    p.numVertices = n;
    p.numTriangles = mesh->num_triangles;
    p.scratch = w;
    p.outVertices = reinterpret_cast<float*>(w + scratch);
    p.outNormals = normals ? reinterpret_cast<float*>(w + scratch + outBytes) : nullptr;
    p.unique = reinterpret_cast<uint32_t*>(w + scratch + outBytes * (normals ? 2 : 1));
    cudaStream_t s = ctx->stream;
    CUDA_TRY(ctx, dcsg_launch_weld(p, s));
    g_launches += 6;                // the weld's own kernels; cub's sort and scan passes are not counted
    CUDA_TRY(ctx, ctx->pinned_small.reserve(64));
    uint32_t* h_unique = ctx->pinned_small.as<uint32_t>();
    CUDA_TRY(ctx, cudaMemcpyAsync(h_unique, p.unique, 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    const uint64_t m = *h_unique;
    if (m) {
        CUDA_TRY(ctx, cudaMemcpyAsync(mesh->d_vertices, p.outVertices, m * 12, cudaMemcpyDeviceToDevice, s));
        if (normals) CUDA_TRY(ctx, cudaMemcpyAsync(mesh->d_normals, p.outNormals, m * 12, cudaMemcpyDeviceToDevice, s));
    }
    // host copies (copy_to_host): same arrays, fewer vertices
    if (mesh->h_vertices && m) CUDA_TRY(ctx, cudaMemcpyAsync(mesh->h_vertices, mesh->d_vertices, m * 12, cudaMemcpyDeviceToHost, s));
    if (mesh->h_normals && normals && m) CUDA_TRY(ctx, cudaMemcpyAsync(mesh->h_normals, mesh->d_normals, m * 12, cudaMemcpyDeviceToHost, s));
    if (mesh->h_triangles && mesh->num_triangles)
        CUDA_TRY(ctx, cudaMemcpyAsync(mesh->h_triangles, mesh->d_triangles, mesh->num_triangles * 12, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    mesh->num_vertices = m;
    mesh->owned_vertices = m;
    mesh->halo_vertices = 0;
    // triangles now share vertices across source triangles: the soup file pipeline's units no longer hold (it refuses the mesh)
    st->unitTriangles = st->unitVertices = 0;
    return DCSG_OK;
}

// The face rows do not depend on the projection: they are formatted and copied on the copy stream while the first chunks
// are projected.
int dcsg_host::indexed_pipeline_locked(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, bool normals, const IndexedTarget& t) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    MeshStorage* st = (MeshStorage*)mesh->reserved;
    const bool project = gd_steps >= 0;
    if (project && !ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    if (project && normals) {
        CUDA_TRY(ctx, st->normals.reserve(std::max<uint64_t>(mesh->num_vertices, 1) * 12));
        mesh->d_normals = st->normals.as<float>();
    }
    if (normals && !mesh->d_normals) return fail(ctx, DCSG_ERR_INVALID, "DCSG_PLY_NORMALS needs a mesh with normals");
    const uint64_t n = t.vertices, nt = mesh->num_triangles;
    const size_t row = normals ? 24 : 12;
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t offFaces = align(n * row), offRows = align(nt * 13);
    CUDA_TRY(ctx, ctx->pinned.reserve(offFaces + offRows + 64));
    CUDA_TRY(ctx, ctx->fmt.reserve(offRows + (normals ? align(n * 24) : 0) + 64));
    uint8_t* h = ctx->pinned.as<uint8_t>();
    uint8_t* dFaces = ctx->fmt.as<uint8_t>();
    float* dRows = reinterpret_cast<float*>(dFaces + offRows);
    if (!ctx->copy_stream) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (auto& ev : ctx->chunk_event) if (!ev) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    for (auto& ev : ctx->copied_event) if (!ev) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaStream_t cs = ctx->stream, ds = ctx->copy_stream;
    const int kFaces = 15;          // event slots of the face rows; chunks use 0 .. 11

    CUDA_TRY(ctx, cudaEventRecord(ctx->chunk_event[kFaces], cs));       // the mesh's triangles are final here
    CUDA_TRY(ctx, cudaStreamWaitEvent(ds, ctx->chunk_event[kFaces], 0));
    if (nt) {
        dcsg_launch_format_ply_indexed_faces(mesh->d_triangles, nt, t.base, dFaces, ds); ++g_launches;
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(h + offFaces, dFaces, nt * 13, cudaMemcpyDeviceToHost, ds));
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->copied_event[kFaces], ds));

    const int chunks = (int)std::max<uint64_t>(1, std::min<uint64_t>(12, n / 200000));
    const bool runProjection = project && (gd_steps > 0 || normals);
    if (runProjection && n) CUDA_TRY(ctx, ctx->project_list.reserve((size_t)n * 8));     // no reallocation between the chunks
    std::vector<uint64_t> chunkEnd;
    for (int c = 0; c < chunks; c++) {
        const uint64_t v0 = n * (uint64_t)c / chunks, v1 = n * (uint64_t)(c + 1) / chunks;
        chunkEnd.push_back(v1);
        if (v1 == v0) continue;
        if (runProjection) {
            if (int rc = launch_project(ctx, mesh->d_vertices + v0 * 3, v1 - v0, gd_steps, normals ? mesh->d_normals + v0 * 3 : nullptr, cs, c,
                                        nullptr, nullptr, 0, v0)) return rc;
        }
        const uint8_t* src = reinterpret_cast<const uint8_t*>(mesh->d_vertices + v0 * 3);
        if (normals) {
            dcsg_launch_format_ply_indexed_vertices(mesh->d_vertices + v0 * 3, mesh->d_normals + v0 * 3, v1 - v0, dRows + v0 * 6, cs); ++g_launches;
            src = reinterpret_cast<const uint8_t*>(dRows + v0 * 6);
        }
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaEventRecord(ctx->chunk_event[c], cs));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ds, ctx->chunk_event[c], 0));
        CUDA_TRY(ctx, cudaMemcpyAsync(h + v0 * row, src, (v1 - v0) * row, cudaMemcpyDeviceToHost, ds));
        CUDA_TRY(ctx, cudaEventRecord(ctx->copied_event[c], ds));
    }
    // everything is queued on the device; hand the rows to the writer threads as they land in pinned memory
    bool ok = true;
    {
        FileSink sink(host_threads(ctx));
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->copied_event[kFaces]));
        sink.submit(t.fd, h + offFaces, nt * 13, t.faceOffset);
        uint64_t v0 = 0;
        for (int c = 0; c < chunks; c++) {
            const uint64_t v1 = chunkEnd[c];
            if (v1 > v0) {
                CUDA_TRY(ctx, cudaEventSynchronize(ctx->copied_event[c]));
                sink.submit(t.fd, h + v0 * row, (v1 - v0) * row, t.vertexOffset + v0 * row);
            }
            if (c == 0 && project) report_progress(ctx, DCSG_PROGRESS_GRADIENT_DESCENT, (uint64_t)std::max(gd_steps, 0), (uint64_t)std::max(gd_steps, 0));
            if (project) report_progress(ctx, DCSG_PROGRESS_WRITING_PLY, v1, n);
            v0 = v1;
        }
        ok = sink.finish();
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ds));
    CUDA_TRY(ctx, cudaStreamSynchronize(cs));
    return ok ? DCSG_OK : fail(ctx, DCSG_ERR_IO, "short write");
}

extern "C" {

int dcsg_mesh_weld(dcsg_ctx* ctx, dcsg_mesh* mesh) {
    if (!ctx || !mesh || !mesh->reserved) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    return weld_locked(ctx, mesh);
}

int dcsg_write_ply_indexed(dcsg_ctx* ctx, const dcsg_mesh* mesh_in, int flags, const char* path) {
    if (!ctx || !mesh_in || !mesh_in->reserved || !path || (flags & ~DCSG_PLY_NORMALS)) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    dcsg_mesh mesh = *mesh_in;          // gd_steps < 0: the pipeline reads the mesh and changes nothing in it
    const bool normals = (flags & DCSG_PLY_NORMALS) != 0;
    if (normals && !mesh.d_normals) return fail(ctx, DCSG_ERR_INVALID, "DCSG_PLY_NORMALS needs a mesh with normals");
    if (mesh.num_vertices > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "more than 2^32 vertices");
    const uint64_t V = mesh.num_vertices, T = mesh.num_triangles, row = normals ? 24 : 12;
    const std::string header = indexed_ply_header(V, T, normals);
    const int fd = create_sized_file(path, header, header.size() + row * V + 13 * T);
    if (fd < 0) return fail(ctx, DCSG_ERR_IO, std::string("cannot create ") + path);
    const int rc = indexed_pipeline_locked(ctx, &mesh, -1, normals, IndexedTarget{fd, header.size(), header.size() + row * V, 0u, V});
    close(fd);
    return rc;
}

}  // extern "C"
