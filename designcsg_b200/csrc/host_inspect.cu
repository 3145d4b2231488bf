// host_inspect.cu -- dcsg_mesh_inspect: edge topology, shells, area, volume, centroid and extents of a mesh, computed on the
// device from its vertex and triangle arrays (kernels: mesher_kernels.cu "mesh inspection").  No reference counterpart.
#include "host_internal.h"

using namespace dcsg_host;

static void empty_report(uint64_t V, dcsg_mesh_report* r) {
    memset(r, 0, sizeof(*r));
    r->num_vertices = V;
    r->unreferenced_vertices = V;
    for (int c = 0; c < 3; c++) {
        r->centroid[c] = NAN;
        r->bbox_min[c] = INFINITY;
        r->bbox_max[c] = -INFINITY;
    }
}

extern "C" {

int dcsg_mesh_inspect(dcsg_ctx* ctx, const dcsg_mesh* mesh, dcsg_mesh_report* report, uint64_t component_capacity,
                      uint64_t* component_triangles, double* component_area, double* component_signed_volume) {
    if (!ctx || !mesh || !report) return DCSG_ERR_INVALID;
    if (component_capacity && (!component_triangles || !component_area || !component_signed_volume)) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    const uint64_t V = mesh->num_vertices, T = mesh->num_triangles;
    if (V > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "dcsg_mesh_inspect: more than 2^32 vertices");
    dcsg_mesh_report r;
    empty_report(V, &r);
    r.num_triangles = T;
    if (!T) {
        *report = r;
        return DCSG_OK;
    }
    if (!mesh->d_triangles || (V && !mesh->d_vertices)) return fail(ctx, DCSG_ERR_INVALID, "dcsg_mesh_inspect: the mesh has no device arrays");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t scratch = align(dcsg_inspect_scratch_bytes(V, T)), comps = align(T * sizeof(dcsg_inspect_component));
    CUDA_TRY(ctx, ctx->inspect.reserve(scratch + comps + sizeof(dcsg_inspect_totals)));
    uint8_t* w = ctx->inspect.as<uint8_t>();
    dcsg_inspect_params p;
    p.vertices = mesh->d_vertices;
    p.triangles = mesh->d_triangles;
    p.numVertices = V;
    p.numTriangles = T;
    p.scratch = w;
    p.components = reinterpret_cast<dcsg_inspect_component*>(w + scratch);
    p.totals = reinterpret_cast<dcsg_inspect_totals*>(w + scratch + comps);
    cudaStream_t s = ctx->stream;
    CUDA_TRY(ctx, ctx->pinned_small.reserve(sizeof(dcsg_inspect_totals)));
    dcsg_inspect_totals* h = ctx->pinned_small.as<dcsg_inspect_totals>();
    // the ids are checked before any vertex is read through them
    CUDA_TRY(ctx, dcsg_launch_inspect_check(p, s));
    ++g_launches;
    CUDA_TRY(ctx, cudaMemcpyAsync(&h->badIds, &p.totals->badIds, sizeof(h->badIds), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    if (h->badIds) return fail(ctx, DCSG_ERR_INVALID, format("dcsg_mesh_inspect: a triangle refers to a vertex id >= %llu", (unsigned long long)V));
    CUDA_TRY(ctx, dcsg_launch_inspect(p, s));
    g_launches += 6;                // init, triangles, flatten, labels, the two head passes; cub's passes are not counted
    CUDA_TRY(ctx, cudaMemcpyAsync(h, p.totals, sizeof(*h), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    const dcsg_inspect_totals t = *h;
    if (t.componentRuns != t.v.roots + (t.t.degenerate ? 1 : 0))
        return fail(ctx, DCSG_ERR_CUDA, format("dcsg_mesh_inspect: %llu component runs for %llu components",
                                               (unsigned long long)t.componentRuns, (unsigned long long)t.v.roots));
    r.unreferenced_vertices = V - t.v.referenced;
    r.nonfinite_vertices = t.v.nonfinite;
    r.degenerate_triangles = t.t.degenerate;
    r.zero_area_triangles = t.t.zeroArea;
    r.nonfinite_triangles = t.t.nonfinite;
    r.edges = t.e.edges;
    r.boundary_edges = t.e.boundary;
    r.manifold_edges = t.e.manifold;
    r.nonmanifold_edges = t.e.nonmanifold;
    r.misoriented_edges = t.e.misoriented;
    r.components = t.v.roots;
    r.area = t.t.area;
    r.signed_volume = t.t.volume;
    for (int c = 0; c < 3; c++) {
        r.centroid[c] = t.t.volume == 0.0 ? NAN : t.t.moment[c] / (4.0 * t.t.volume);
        r.bbox_min[c] = t.v.lo[c];
        r.bbox_max[c] = t.v.hi[c];
    }
    const uint64_t n = std::min<uint64_t>(component_capacity, r.components);
    if (n) {
        CUDA_TRY(ctx, ctx->pinned_small.reserve(n * sizeof(dcsg_inspect_component)));
        dcsg_inspect_component* hc = ctx->pinned_small.as<dcsg_inspect_component>();
        CUDA_TRY(ctx, cudaMemcpyAsync(hc, p.components, n * sizeof(*hc), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(ctx, cudaStreamSynchronize(s));
        for (uint64_t i = 0; i < n; i++) {
            component_triangles[i] = hc[i].triangles;
            component_area[i] = hc[i].area;
            component_signed_volume[i] = hc[i].volume;
        }
    }
    *report = r;
    return DCSG_OK;
}

}  // extern "C"
