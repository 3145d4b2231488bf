// host_deviation.cu -- dcsg_mesh_deviation: the scene's SDF sampled at the vertices and over every triangle of a mesh, on the
// device (kernels: mesher_kernels.cu "mesh deviation"; the values come from the scene module's dcsg_k_eval_sdf, the kernel
// behind dcsg_eval_sdf, so that every value is that call's bits).  No reference counterpart.
#include "host_internal.h"

using namespace dcsg_host;

static void empty_report(uint64_t V, uint64_t T, dcsg_deviation_report* r) {
    memset(r, 0, sizeof(*r));
    r->num_vertices = V;
    r->num_triangles = T;
    r->worst_triangle = UINT64_MAX;
    r->vertex_max_abs = -INFINITY;
    r->min_sdf = INFINITY;
    r->max_sdf = -INFINITY;
    r->max_abs = -INFINITY;
    for (int c = 0; c < 3; c++) r->worst_point[c] = NAN;
    r->vertex_rms = NAN;
    r->mean_abs = NAN;
}

extern "C" {

int dcsg_mesh_deviation(dcsg_ctx* ctx, const dcsg_mesh* mesh, int subdivision, float tolerance, dcsg_deviation_report* report,
                        float* triangle_max_abs) {
    if (!ctx || !mesh || !report) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (subdivision < 1 || subdivision > kDeviationMaxK)
        return fail(ctx, DCSG_ERR_INVALID, format("dcsg_mesh_deviation: subdivision %d is outside [1, %d]", subdivision, kDeviationMaxK));
    if (!(tolerance >= 0.0f)) return fail(ctx, DCSG_ERR_INVALID, "dcsg_mesh_deviation: the tolerance is negative or NaN");
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "dcsg_mesh_deviation before dcsg_build");
    const uint64_t V = mesh->num_vertices, T = mesh->num_triangles;
    if (V > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "dcsg_mesh_deviation: more than 2^32 vertices");
    dcsg_deviation_report r;
    empty_report(V, T, &r);
    if (!T) {
        *report = r;
        return DCSG_OK;
    }
    if (!mesh->d_triangles || (V && !mesh->d_vertices)) return fail(ctx, DCSG_ERR_INVALID, "dcsg_mesh_deviation: the mesh has no device arrays");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int k = subdivision;
    dcsg_deviation_params p = {};
    p.vertices = mesh->d_vertices;
    p.triangles = mesh->d_triangles;
    p.numVertices = V;
    p.numTriangles = T;
    p.k = k;
    p.samples = (k + 1) * (k + 2) / 2 - 3;
    for (int i = 0, s = 0; i <= k; i++)
        for (int j = 0; i + j <= k; j++) {
            if ((i == 0 && j == 0) || (i == k && j == 0) || (i == 0 && j == k)) continue;
            p.ij[2 * s] = (uint8_t)i;
            p.ij[2 * s + 1] = (uint8_t)j;
            s++;
        }
    p.tolerance = tolerance;
    const size_t scratch = (dcsg_deviation_scratch_bytes(V, T, p.samples) + 255) & ~(size_t)255;
    CUDA_TRY(ctx, ctx->deviation.reserve(scratch + sizeof(dcsg_deviation_totals)));
    p.scratch = ctx->deviation.ptr;
    p.totals = reinterpret_cast<dcsg_deviation_totals*>(ctx->deviation.as<uint8_t>() + scratch);
    cudaStream_t s = ctx->stream;
    CUDA_TRY(ctx, ctx->pinned_small.reserve(sizeof(dcsg_deviation_totals)));
    // the ids are checked before any vertex is read through them (dcsg_mesh_inspect's check)
    dcsg_inspect_params check = {};
    check.triangles = mesh->d_triangles;
    check.numVertices = V;
    check.numTriangles = T;
    check.totals = dcsg_deviation_check_totals(p);
    CUDA_TRY(ctx, dcsg_launch_inspect_check(check, s));
    ++g_launches;
    uint32_t* badIds = ctx->pinned_small.as<uint32_t>();
    CUDA_TRY(ctx, cudaMemcpyAsync(badIds, &check.totals->badIds, sizeof(*badIds), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    if (*badIds) return fail(ctx, DCSG_ERR_INVALID, format("dcsg_mesh_deviation: a triangle refers to a vertex id >= %llu", (unsigned long long)V));
    // vertices: every one is evaluated (AoS xyz already); the marks decide which ones count
    CUDA_TRY(ctx, dcsg_launch_deviation_marks(p, s));
    ++g_launches;
    int rc = eval_device_locked(ctx, ctx->k_eval_sdf, mesh->d_vertices, V, dcsg_deviation_vertex_values(p));
    if (rc != DCSG_OK) return rc;
    // triangles, chunk by chunk: points, their values, the per-triangle terms
    const uint64_t chunk = dcsg_deviation_chunk(T, p.samples);
    for (uint64_t first = 0; first < T; first += chunk) {
        const uint64_t n = std::min(chunk, T - first);
        if (p.samples) {
            CUDA_TRY(ctx, dcsg_launch_deviation_points(p, first, n, s));
            ++g_launches;
            rc = eval_device_locked(ctx, ctx->k_eval_sdf, dcsg_deviation_points(p), n * (uint64_t)p.samples, dcsg_deviation_values(p));
            if (rc != DCSG_OK) return rc;
        }
        CUDA_TRY(ctx, dcsg_launch_deviation_triangles(p, first, n, s));
        ++g_launches;
    }
    CUDA_TRY(ctx, dcsg_launch_deviation_totals(p, s));
    ++g_launches;                   // the totals' kernel; cub's passes are not counted
    dcsg_deviation_totals* h = ctx->pinned_small.as<dcsg_deviation_totals>();
    CUDA_TRY(ctx, cudaMemcpyAsync(h, p.totals, sizeof(*h), cudaMemcpyDeviceToHost, s));
    if (triangle_max_abs)
        CUDA_TRY(ctx, cudaMemcpyAsync(triangle_max_abs, dcsg_deviation_triangle_max_abs(p), T * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    const dcsg_deviation_totals t = *h;
    r.measured_vertices = t.measuredVertices;
    r.measured_triangles = t.measuredTriangles;
    r.samples = t.measuredVertices + (uint64_t)p.samples * t.measuredTriangles;
    r.nan_samples = t.nanVertices + t.nanSamples;
    r.over_tolerance = t.overTolerance;
    r.worst_triangle = t.worstTriangle;
    r.vertex_max_abs = t.vertexMaxAbs;
    r.min_sdf = t.minSdf;
    r.max_sdf = t.maxSdf;
    r.max_abs = t.maxAbs;
    for (int c = 0; c < 3; c++) r.worst_point[c] = t.worstPoint[c];
    r.vertex_rms = t.vertexValues ? sqrt(t.vertexSumSq / (double)t.vertexValues) : NAN;
    r.mean_abs = t.sumArea == 0.0 ? NAN : t.sumAreaMean / t.sumArea;
    *report = r;
    return DCSG_OK;
}

}  // extern "C"
