// host_context.cu -- context life cycle, scene build, point evaluation, bounding-box search, slab plan, preview.
//
// Plays the role of the reference's Evaluator (master/Evaluator.{h,cpp}) and of the set-up half of the export driver
// (MyFrame::OnExportInner, master/DesignCSG.cpp:638-712).  CUDA runtime API only (static cudart; the NVRTC cubin is loaded
// with cudaLibraryLoadData), so the library loads on machines without a driver and fails loudly in dcsg_create there.
#include "host_internal.h"
#include "mc_table.inc"

using namespace dcsg_host;

namespace dcsg_host {
std::atomic<unsigned long long> g_launches{0};      // kernels launched by this library (claimed as gpu_launches by bench.py)

int eval_device_locked(dcsg_ctx* ctx, cudaKernel_t k, const float* d_xyz, size_t n, float* d_out) {
    if (n == 0) return DCSG_OK;
    unsigned long long nn = n;
    void* args[] = {(void*)&d_xyz, (void*)&d_out, &nn};
    CUDA_TRY(ctx, launch(k, dim3((unsigned)((n + 255) / 256)), dim3(256), args, ctx->stream, ctx->scene.private_words));
    return DCSG_OK;
}
}

extern "C" {

const char* dcsg_version(void) { return "designcsg_b200 0.1 (sm_100a)"; }

const char* dcsg_last_error(const dcsg_ctx* ctx) { return ctx ? ctx->error.c_str() : "null context"; }

int dcsg_create(int device, dcsg_ctx** out) {
    if (!out) return DCSG_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        fprintf(stderr, "libdcsg: no CUDA device available (%s); there is no CPU fallback\n", cudaGetErrorString(e));
        return DCSG_ERR_CUDA;
    }
    if (device < 0 || device >= count) return DCSG_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return DCSG_ERR_CUDA;
    dcsg_ctx* ctx = new dcsg_ctx();
    ctx->device = device;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return DCSG_ERR_CUDA; }
    if (cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->sm_count < 1) { delete ctx; return DCSG_ERR_CUDA; }
    for (auto& ev : ctx->ev) cudaEventCreate(&ev);
    cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&ctx->aux_ready, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->aux_done, cudaEventDisableTiming);
    cudaMalloc((void**)&ctx->d_tri_count, 256);
    cudaMalloc((void**)&ctx->d_tri_table, 256 * 16);
    cudaMalloc((void**)&ctx->d_tri_flip, 256);
    cudaMemcpy(ctx->d_tri_count, kDcsgTriCount, 256, cudaMemcpyHostToDevice);
    cudaMemcpy(ctx->d_tri_table, kDcsgTriTable, 256 * 16, cudaMemcpyHostToDevice);
    cudaMemcpy(ctx->d_tri_flip, kDcsgTriFlip, 256, cudaMemcpyHostToDevice);
    if (cudaGetLastError() != cudaSuccess) { delete ctx; return DCSG_ERR_CUDA; }
    *out = ctx;
    return DCSG_OK;
}

void dcsg_destroy(dcsg_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (DevBuf* b : {&ctx->pts, &ctx->vals, &ctx->axes, &ctx->sign, &ctx->leaf, &ctx->cfail, &ctx->coarse, &ctx->levels, &ctx->alive, &ctx->vinfo,
                      &ctx->tiles, &ctx->small, &ctx->lattice_values, &ctx->fmt, &ctx->adapt_emit, &ctx->adapt_snap, &ctx->search_bits, &ctx->project_cursor, &ctx->lists, &ctx->masks, &ctx->soup, &ctx->project_list, &ctx->weld, &ctx->orient, &ctx->inspect, &ctx->deviation})
        b->release();
    ctx->pinned.release();
    ctx->pinned_small.release();
    ctx->pinned_soup.release();
    if (ctx->lib) cudaLibraryUnload(ctx->lib);
    cudaFree(ctx->d_tri_count);
    cudaFree(ctx->d_tri_table);
    cudaFree(ctx->d_tri_flip);
    for (auto& ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) { cudaStreamSynchronize(ctx->aux_stream); cudaStreamDestroy(ctx->aux_stream); }
    if (ctx->aux_ready) cudaEventDestroy(ctx->aux_ready);
    if (ctx->aux_done) cudaEventDestroy(ctx->aux_done);
    for (auto& ev : ctx->chunk_event) if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->copied_event) if (ev) cudaEventDestroy(ev);
    delete ctx;
}

int dcsg_set_stream(dcsg_ctx* ctx, void* cuda_stream) {
    if (!ctx) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return DCSG_OK;
}

int dcsg_set_progress_callback(dcsg_ctx* ctx, dcsg_progress_fn fn, void* user) {
    if (!ctx) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    ctx->progress = fn;
    ctx->progress_user = fn ? user : nullptr;
    return DCSG_OK;
}

int dcsg_set_export_flags(dcsg_ctx* ctx, int flags) {
    if (!ctx || (flags & ~DCSG_EXPORT_OUTWARD)) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    ctx->export_flags = flags;
    return DCSG_OK;
}

int dcsg_scene_source(const char* scene_dir, char* out, size_t capacity, size_t* needed) {
    Scene sc;
    std::string err;
    if (!scene_dir || !load_scene(scene_dir, sc, err)) return DCSG_ERR_IO;
    std::string src = assemble_source(sc, scene_wants_fast_path(sc), err);
    if (src.empty()) return DCSG_ERR_INVALID;
    if (needed) *needed = src.size() + 1;
    copy_log(src, out, capacity);
    return DCSG_OK;
}

int dcsg_compile_scene(const char* scene_dir, const char* cubin_path, char* log, size_t log_capacity) {
    Scene sc;
    std::string err;
    if (!scene_dir || !load_scene(scene_dir, sc, err)) { copy_log(err, log, log_capacity); return DCSG_ERR_IO; }
    std::vector<char> cubin;
    std::string clog;
    if (!compile_scene(sc, cubin, clog, err)) {
        copy_log(err.empty() ? clog : err, log, log_capacity);
        return err.empty() ? DCSG_ERR_BUILD : DCSG_ERR_INVALID;
    }
    copy_log(clog, log, log_capacity);
    if (cubin_path) {
        FILE* f = fopen(cubin_path, "wb");
        if (!f) return DCSG_ERR_IO;
        fwrite(cubin.data(), 1, cubin.size(), f);
        fclose(f);
    }
    return DCSG_OK;
}

int dcsg_build(dcsg_ctx* ctx, const char* scene_dir, char* log, size_t log_capacity) {
    if (!ctx || !scene_dir) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    ctx->built = false;
    // the slab plan follows the last search of THIS scene: a previous scene's surface histogram must not plan the new one's slabs
    memset(ctx->zhist, 0, sizeof(ctx->zhist));
    ctx->zhist_c = 0.0f;
    std::string err;
    if (!load_scene(scene_dir, ctx->scene, err)) { copy_log(err, log, log_capacity); return fail(ctx, DCSG_ERR_IO, err); }
    std::vector<char> cubin;
    std::string clog;
    if (!compile_scene(ctx->scene, cubin, clog, err)) {
        if (!err.empty()) { copy_log(err, log, log_capacity); return fail(ctx, DCSG_ERR_INVALID, err); }
        copy_log(clog, log, log_capacity);
        return fail(ctx, DCSG_ERR_BUILD, "scene failed to compile:\n" + clog);   // reference: (-1, build log)
    }
    bool calibrated = false;
reload:
    copy_log(clog.empty() ? std::string("Success!") : clog, log, log_capacity);
    if (ctx->lib) { cudaStreamSynchronize(ctx->stream); cudaLibraryUnload(ctx->lib); ctx->lib = nullptr; }
    CUDA_TRY(ctx, cudaLibraryLoadData(&ctx->lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_flag_rate, ctx->lib, "dcsg_k_flag_rate"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_eval_sdf, ctx->lib, "dcsg_k_eval_sdf"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_eval_normal, ctx->lib, "dcsg_k_eval_normal"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_bbox, ctx->lib, "dcsg_k_bbox"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_lattice, ctx->lib, "dcsg_k_lattice"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_coarse_nodes, ctx->lib, "dcsg_k_coarse_nodes"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_project, ctx->lib, "dcsg_k_project"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_descend, ctx->lib, "dcsg_k_descend"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_descend_list, ctx->lib, "dcsg_k_descend_list"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_descend_top, ctx->lib, "dcsg_k_descend_top"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_leaf, ctx->lib, "dcsg_k_leaf"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_corners, ctx->lib, "dcsg_k_corners"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_adapt_level, ctx->lib, "dcsg_k_adapt_level"));
    CUDA_TRY(ctx, cudaLibraryGetKernel(&ctx->k_preview, ctx->lib, "dcsg_k_preview"));
    {
        // per-thread copies of the design's program-scope variables live in dynamic shared memory (launch(): private_words
        // x 1 KiB per block, on top of ~8 KiB static); beyond the default 48 KiB per block a kernel has to opt in
        const int dynBytes = ctx->scene.private_words * 256 * 4;
        if (dynBytes > 36 * 1024) {
            for (cudaKernel_t k : {ctx->k_eval_sdf, ctx->k_eval_normal, ctx->k_bbox, ctx->k_lattice, ctx->k_coarse_nodes, ctx->k_project,
                                   ctx->k_descend, ctx->k_descend_list, ctx->k_descend_top, ctx->k_leaf, ctx->k_corners, ctx->k_adapt_level, ctx->k_preview}) {
                if (cudaFuncSetAttribute((const void*)k, cudaFuncAttributeMaxDynamicSharedMemorySize, dynBytes) != cudaSuccess) {
                    cudaGetLastError();
                    const std::string msg = format("the design declares %d program-scope scalars: %d bytes of per-block shared memory exceed what a kernel can get on this device",
                                                   ctx->scene.private_words, dynBytes);
                    copy_log(msg, log, log_capacity);
                    return fail(ctx, DCSG_ERR_BUILD, msg);
                }
            }
        }
    }
    {
        // the projection's persistent grid is sized to the blocks that can be resident at once (registers per thread differ
        // between the tap forms and scenes)
        int resident = 0;
        CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, (const void*)ctx->k_project, 256, (size_t)ctx->scene.private_words * 256 * 4));
        ctx->project_blocks_per_sm = std::max(1, std::min(8, resident));
    }
    {
        size_t sz = 0;
        void* ptr = nullptr;
        ctx->d_camera_axes[0] = ctx->d_camera_axes[1] = ctx->d_camera_axes[2] = nullptr;
        const char* names[3] = {"rgt_g", "upp_g", "fwd_g"};
        for (int k = 0; k < 3; k++) {
            CUDA_TRY(ctx, cudaLibraryGetGlobal(&ptr, &sz, ctx->lib, names[k]));
            ctx->d_camera_axes[k] = (float*)ptr;
        }
    }
    size_t bytes = 0;
    void* dptr = nullptr;
    CUDA_TRY(ctx, cudaLibraryGetGlobal(&dptr, &bytes, ctx->lib, "arbitrary_data"));
    ctx->d_arbitrary = (float*)dptr;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_arbitrary, 0, bytes, ctx->stream));
    if (!ctx->scene.arbitrary_data.empty())
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_arbitrary, ctx->scene.arbitrary_data.data(), ctx->scene.arbitrary_data.size() * 4,
                                      cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    // Is the checked fast copy worth having on THIS scene?  A sample of points spread over the search volume (where the
    // export evaluates): if more than 1.5 % of the evaluations fail the fast copy's test, most warps would run both copies
    // (break-even of 172 + 283 * P(warp flagged) against 283 instructions), so the module is rebuilt exact-only.  Design1:
    // 0 %; the 4096-primitive synthetic scene, whose box brushes take sqrt(0) inside every box: ~half of them.
    if (!calibrated && scene_wants_fast_path(ctx->scene)) {
        calibrated = true;
        const size_t n = 1 << 16;
        float diameter = 10.0f;
        if (!ctx->scene.export_config.empty()) { const float d = strtof(ctx->scene.export_config[0].c_str(), nullptr); if (d > 0.0f && std::isfinite(d)) diameter = d; }
        std::vector<float> pts(n * 3);
        uint64_t state = 0x9e3779b97f4a7c15ull;
        for (float& v : pts) {          // splitmix64: the same sample for every build of every scene
            state += 0x9e3779b97f4a7c15ull;
            uint64_t z = state;
            z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
            z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
            z ^= z >> 31;
            v = ((float)(z >> 40) / 16777216.0f - 0.5f) * diameter;
        }
        CUDA_TRY(ctx, ctx->pts.reserve(n * 12 + 16));
        CUDA_TRY(ctx, ctx->small.reserve(4096));
        uint32_t* d_flagged = ctx->small.as<uint32_t>() + 200;
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->pts.ptr, pts.data(), n * 12, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaMemsetAsync(d_flagged, 0, 4, ctx->stream));
        const float* d_xyz = ctx->pts.as<float>();
        unsigned long long nn = n;
        void* args[] = {(void*)&d_xyz, &nn, &d_flagged};
        CUDA_TRY(ctx, launch(ctx->k_flag_rate, dim3((unsigned)(n / 256)), dim3(256), args, ctx->stream, ctx->scene.private_words));
        uint32_t flagged = 0;
        CUDA_TRY(ctx, cudaMemcpyAsync(&flagged, d_flagged, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        if ((double)flagged > 0.015 * (double)n) {
            std::vector<char> exactCubin;
            std::string exactLog;
            if (compile_scene(ctx->scene, exactCubin, exactLog, err, true)) {
                cubin.swap(exactCubin);
                clog = format("[dcsg] the checked fast copy failed its test on %.1f %% of a sample of evaluations: built exact-only\n", 100.0 * flagged / n) + exactLog;
                goto reload;
            }
        }
    }
    ctx->built = true;
    return DCSG_OK;
}

int dcsg_set_arbitrary_data(dcsg_ctx* ctx, const float* data, size_t items) {
    if (!ctx || !data) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "dcsg_set_arbitrary_data before dcsg_build");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    items = std::min(items, (size_t)DCSG_ARBITRARY_DATA_POINTS);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_arbitrary, data, items * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DCSG_OK;
}

int dcsg_eval_sdf_device(dcsg_ctx* ctx, const float* d_xyz, size_t n, float* d_out) {
    if (!ctx) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return eval_device_locked(ctx, ctx->k_eval_sdf, d_xyz, n, d_out);
}

int dcsg_eval_normal_device(dcsg_ctx* ctx, const float* d_xyz, size_t n, float* d_out3) {
    if (!ctx) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return eval_device_locked(ctx, ctx->k_eval_normal, d_xyz, n, d_out3);
}

// host-buffer evaluation in chunks of 2^24 points (the reference's MAX_EVAL_POINTS, Evaluator.h:16)
static int eval_host(dcsg_ctx* ctx, bool normals, const float* xyz, size_t n, float* out) {
    if (!ctx || (n && (!xyz || !out))) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t chunk = (size_t)1 << 24;
    const size_t width = normals ? 3 : 1;
    CUDA_TRY(ctx, ctx->pts.reserve(std::min(n, chunk) * 12 + 16));
    CUDA_TRY(ctx, ctx->vals.reserve(std::min(n, chunk) * 4 * width + 16));
    for (size_t done = 0; done < n; done += chunk) {
        const size_t m = std::min(chunk, n - done);
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->pts.ptr, xyz + done * 3, m * 12, cudaMemcpyHostToDevice, ctx->stream));
        int rc = eval_device_locked(ctx, normals ? ctx->k_eval_normal : ctx->k_eval_sdf, ctx->pts.as<float>(), m, ctx->vals.as<float>());
        if (rc != DCSG_OK) return rc;
        CUDA_TRY(ctx, cudaMemcpyAsync(out + done * width, ctx->vals.ptr, m * 4 * width, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return DCSG_OK;
}

int dcsg_eval_sdf(dcsg_ctx* ctx, const float* xyz, size_t n, float* out) { return eval_host(ctx, false, xyz, n, out); }
int dcsg_eval_normal(dcsg_ctx* ctx, const float* xyz, size_t n, float* out3) { return eval_host(ctx, true, xyz, n, out3); }

}  // extern "C"

// The 256^3 search, or the ix columns [ixBegin, ixEnd) of it (multi-GPU: every rank searches its columns; `reduce`, called
// with the device pointers of the six extreme indices and of the 512-bin histogram, all-reduces them over the ranks before
// they are read back -- min / max / sum of integers, so every rank ends up with the bits of the single-GPU search).
int dcsg_host::bbox_locked(dcsg_ctx* ctx, float search_diameter, float* box6, int ixBegin, int ixEnd,
                           int (*reduce)(void* user, int* d_minmax, uint32_t* d_hist, cudaStream_t stream), void* reduce_user) {
    const int R = 256;
    float c = (float)search_diameter / R;
    CUDA_TRY(ctx, ctx->small.reserve(4096));
    int init[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};
    int* d_mm = ctx->small.as<int>();
    uint32_t* d_hist = ctx->small.as<uint32_t>() + 256;        // bytes 1024 .. 3071 of `small`
    CUDA_TRY(ctx, ctx->search_bits.reserve((size_t)R * R * R / 8));
    uint32_t* d_bits = ctx->search_bits.as<uint32_t>();
    CUDA_TRY(ctx, cudaMemcpyAsync(d_mm, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(d_hist, 0, 512 * 4, ctx->stream));
    // the x-edges of the last own column end in the next column: its sign bits are needed too (its samples count for the
    // extremes as well -- they belong to the search, whichever rank evaluates them)
    const int ixSearchEnd = std::min(R, ixEnd + 1);
    uint32_t firstThread = (uint32_t)ixBegin << 16;
    void* args[] = {&c, &d_mm, &d_bits, &firstThread};
    CUDA_TRY(ctx, launch(ctx->k_bbox, dim3((unsigned)(ixSearchEnd - ixBegin) * (R * R / 256)), dim3(256), args, ctx->stream, ctx->scene.private_words));
    dcsg_launch_surface_hist(d_bits, d_hist, ixBegin, ixEnd, ctx->stream); ++g_launches;
    if (reduce) { if (int rc = reduce(reduce_user, d_mm, d_hist, ctx->stream)) return rc; }
    int mm[6];
    CUDA_TRY(ctx, cudaMemcpyAsync(mm, d_mm, sizeof(mm), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->zhist, d_hist, 512 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->zhist_c = c;
    // back to coordinates: p(i) = (-c/2) + c*i; min / max are seeded with 0 (DesignCSG.cpp:690-705)
    const float h = -c / 2;
    float lo[3] = {0.0f, 0.0f, 0.0f}, hi[3] = {0.0f, 0.0f, 0.0f};
    for (int a = 0; a < 3; a++) {
        if (mm[a] == INT_MAX) continue;                 // nothing inside
        const float pmin = h + c * (float)mm[a], pmax = h + c * (float)mm[3 + a];
        if (pmin < lo[a]) lo[a] = pmin;
        if (pmax > hi[a]) hi[a] = pmax;
    }
    float dia[3];
    for (int a = 0; a < 3; a++) {
        box6[a] = (float)((lo[a] + hi[a]) * 0.5);       // `(min + max) * 0.5` is float*double -> float
        dia[a] = hi[a] - lo[a];
    }
    const float yz = dia[1] > dia[2] ? dia[1] : dia[2];
    const float m = dia[0] > yz ? dia[0] : yz;          // T_max(x, T_max(y, z))
    box6[3] = box6[4] = box6[5] = m;
    return DCSG_OK;
}

extern "C" {

int dcsg_bbox(dcsg_ctx* ctx, float search_diameter, float* box6) {
    if (!ctx || !box6) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return bbox_locked(ctx, search_diameter, box6, 0, 256, nullptr, nullptr);
}

int dcsg_plan_slabs(dcsg_ctx* ctx, const float* box6, int grid_level, int world, int granularity, int* bounds) {
    if (!ctx || !box6 || !bounds || world < 1 || granularity < 1 || grid_level < 0 || grid_level > 11) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    return plan_slabs_locked(ctx, box6, grid_level, world, granularity, bounds);
}

}  // extern "C"

int dcsg_host::plan_slabs_locked(dcsg_ctx* ctx, const float* box6, int grid_level, int world, int granularity, int* bounds) {
    const int N = 1 << grid_level;
    if (N % granularity != 0 || N / granularity < world) return fail(ctx, DCSG_ERR_INVALID, "dcsg_plan_slabs: too many ranks for this lattice / granularity");
    const int units = N / granularity;                      // boundaries sit on multiples of `granularity` layers
    // weight of every unit: the search histogram resampled onto the mesh lattice (piecewise constant per search voxel)
    std::vector<double> weight(units, 0.0);
    const double c = ctx->zhist_c;
    const double oz = (double)box6[2] - 0.5 * (double)box6[5], pitch = (double)box6[5] / N * granularity;
    double total = 0.0;
    if (c > 0.0 && pitch > 0.0) {
        // in-plane edges of search plane b sit at z_b = -c/2 + c*(b-128) (spread over the voxel around it); z-edges
        // span [z_b, z_b + c].  Each is spread over the mesh units it overlaps.
        for (int b = 0; b < 512; b++) {
            if (!ctx->zhist[b]) continue;
            const double zb = -0.5 * c + c * ((b & 255) - 128);
            const double lo = b < 256 ? zb - 0.5 * c : zb, hi = lo + c;
            const double u0 = (lo - oz) / pitch, u1 = (hi - oz) / pitch;
            for (int u = std::max(0, (int)floor(u0)); u < units && u < u1; u++) {
                const double overlap = std::min(u1, (double)u + 1.0) - std::max(u0, (double)u);
                if (overlap > 0.0) { weight[u] += ctx->zhist[b] * overlap / (u1 - u0); total += ctx->zhist[b] * overlap / (u1 - u0); }
            }
        }
    }
    // nearly all of a slab's work scales with its surface (projection, the band of lattice samples around it, the list
    // kernels of the mesher); what scales with its thickness -- the coarse levels of the descent -- gets a small share
    // (round 1's sweeping bitmap passes made that 18 %; with them gone the end slabs of Design1 were 13 % short of surface)
    if (total > 0.0) {
        const double perUnit = 0.03 * total / units;
        for (int u = 0; u < units; u++) weight[u] += perUnit;
        total += perUnit * units;
    }
    bounds[0] = 0;
    bounds[world] = N;
    if (total <= 0.0) {                                      // no estimate (no dcsg_bbox call yet, empty scene): equal slabs
        for (int r = 1; r < world; r++) bounds[r] = (int)((int64_t)units * r / world) * granularity;
        return DCSG_OK;
    }
    double acc = 0.0;
    int u = 0;
    for (int r = 1; r < world; r++) {
        const double target = total * r / world;
        while (u < units && acc + weight[u] * 0.5 < target) acc += weight[u++];
        int cut = std::max(u, bounds[r - 1] / granularity + 1);          // at least one unit per rank ...
        cut = std::min(cut, units - (world - r));                        // ... and room for the ranks above
        bounds[r] = cut * granularity;
    }
    return DCSG_OK;
}

extern "C" {

int dcsg_preview(dcsg_ctx* ctx, const float* campos3, const float* right3, const float* up3, const float* forward3, uint8_t* rgb_host) {
    if (!ctx || !campos3 || !right3 || !up3 || !forward3 || !rgb_host) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)640 * 480 * 3;
    CUDA_TRY(ctx, ctx->fmt.reserve(bytes));
    struct { float campos[3], right[3], up[3], forward[3]; unsigned char* pixels; } params;
    memcpy(params.campos, campos3, 12);
    memcpy(params.right, right3, 12);
    memcpy(params.up, up3, 12);
    memcpy(params.forward, forward3, 12);
    params.pixels = ctx->fmt.as<unsigned char>();
    // k1 publishes the camera basis to the materials through program-scope variables (k1.cl:35-37, :516-518); k2 zeroes
    // them (k2.cl:253-255), so they are set for this launch and cleared again
    const float* axes[3] = {right3, up3, forward3};
    const float zero[3] = {0.0f, 0.0f, 0.0f};
    for (int k = 0; k < 3; k++) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_camera_axes[k], axes[k], 12, cudaMemcpyHostToDevice, ctx->stream));
    void* args[] = {&params};
    CUDA_TRY(ctx, launch(ctx->k_preview, dim3((640 * 480 + 255) / 256), dim3(256), args, ctx->stream, ctx->scene.private_words));
    for (int k = 0; k < 3; k++) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_camera_axes[k], zero, 12, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(rgb_host, params.pixels, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DCSG_OK;
}

int dcsg_fp32_peak(dcsg_ctx* ctx, int mode, double* tflops) {
    if (!ctx || !tflops) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const double v = dcsg_fp32_peak_tflops(mode, 5, ctx->stream);
    if (v < 0.0) return fail(ctx, DCSG_ERR_CUDA, "fp32 peak micro-benchmark failed");
    *tflops = v;
    return DCSG_OK;
}

}  // extern "C"

