// host_comm.cu -- the multi-GPU export behind the C ABI: one process per GPU, one node.
//
// The reference's export driver (MyFrame::OnExportInner, master/DesignCSG.cpp:638-790) runs on one OpenCL device; here the
// lattice is cut into z-slabs, one per rank, and a C / C++ host drives the whole sharded export through dcsg_comm_* and
// dcsg_*_sharded -- no Python, no torch on the path.  What crosses GPUs:
//   * NCCL (over NVLink / NVSwitch), small collectives only: all-reduce of the sharded 256^3 bounding-box search (six extreme
//     indices + the 512-bin surface histogram the slab plan is cut from), all-gather of the slabs' {vertices, triangles,
//     cells} counts, a one-word all-reduce as completion signal / barrier, a broadcast of IPC handles when arrays are (re)allocated;
//   * the mesh itself travels WITHOUT a collective: the gathering rank's arrays are mapped into every rank (CUDA IPC), a
//     slab's vertex ids plus the slab's global vertex offset ARE the whole mesh's ids (mesher.h "Ownership"), so the emit
//     kernels store keys and triangles, and the projection kernel the final positions, straight to their places in those
//     arrays (peer stores over NVLink) -- the transfer rides under the compute, tile by tile, and nothing is welded.
// NCCL is loaded at run time (dlopen): libdcsg.so itself does not depend on it, single-GPU hosts never load it, and inside a
// PyTorch process the already loaded libnccl.so.2 is the one that gets used.
#include "host_internal.h"

#include <dlfcn.h>
#include <nccl.h>

using namespace dcsg_host;

namespace {

struct NcclApi {
    void* lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    std::string error;
};

NcclApi* nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* override_path = getenv("DCSG_NCCL_LIBRARY");
        const char* names[] = {override_path, "libnccl.so.2", "libnccl.so"};
        for (const char* name : names) {
            if (!name || !*name) continue;
            api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (!api.lib) { api.error = std::string("cannot load NCCL (libnccl.so.2): ") + (dlerror() ? dlerror() : "not found"); return; }
        bool ok = true;
        auto sym = [&](const char* name) { void* p = dlsym(api.lib, name); if (!p) { ok = false; api.error = std::string("NCCL lacks ") + name; } return p; };
        api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
        api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
        api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
        api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
        api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
        api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
        api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
        api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
        if (!ok) { dlclose(api.lib); api.lib = nullptr; }
    });
    return api.lib ? &api : nullptr;
}

}  // namespace

enum { kArrKeys = 0, kArrTriangles, kArrVertices, kArrNormals, kArrCount };
static const size_t kArrItemBytes[kArrCount] = {8, 12, 12, 12};

struct dcsg_comm {
    dcsg_ctx* ctx = nullptr;
    int rank = 0, world = 1;
    ncclComm_t nccl = nullptr;
    // the whole mesh on the gathering rank; `arr` are that rank's allocations (its own pointers there, IPC mappings elsewhere)
    int dst = -1;
    uint64_t capVertices = 0, capTriangles = 0;
    void* arr[kArrCount] = {nullptr, nullptr, nullptr, nullptr};
    DevBuf dev;                 // small device buffer for the collectives
    HostBuf host;               // pinned mirror
    // this step: counts[r] = {own vertices, triangles, cells, halo copies} of rank r; prefixes
    std::vector<uint64_t> counts, voff, toff;
    int slab[17] = {0};
    bool adaptive = false;      // the current extraction is the adaptive walk: soup, one run of the whole mesh per octree level
    uint64_t unitTriangles = 1, unitVertices = 3;
    std::vector<MeshStorage::Run> runs;
    bool gather = false;        // the current extraction points its emitters at the gathering rank's arrays ...
    int wantDst = 0;            // ... which belong to this rank
    bool wantNormals = false;
};

namespace {

#define NCCL_TRY(comm, expr)                                                                                         \
    do {                                                                                                             \
        ncclResult_t r__ = (expr);                                                                                   \
        if (r__ != ncclSuccess)                                                                                      \
            return fail((comm)->ctx, DCSG_ERR_CUDA, format("%s:%d %s -> NCCL: %s", __FILE__, __LINE__, #expr, nccl_api()->GetErrorString(r__))); \
    } while (0)

// 16 x u64 scratch words per rank on the device / in pinned memory
uint64_t* dev_words(dcsg_comm* c) { return c->dev.as<uint64_t>(); }
uint64_t* host_words(dcsg_comm* c) { return c->host.as<uint64_t>(); }

// One-word all-reduce on the context's stream + wait: every rank's earlier work on its stream -- peer stores included -- is
// complete when this returns (a rank enters the collective only after that work, in stream order).
int barrier(dcsg_comm* c) {
    dcsg_ctx* ctx = c->ctx;
    NcclApi* n = nccl_api();
    uint64_t* word = dev_words(c) + 256;            // byte 2048: past the gathered counts (16 ranks x 32 words)
    NCCL_TRY(c, n->AllReduce(word, word, 1, ncclUint64, ncclSum, c->nccl, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DCSG_OK;
}

uint64_t grown(uint64_t capacity, uint64_t needed) {       // the same on every rank: a pure function of gathered counts
    return needed <= capacity ? capacity : needed + needed / 4 + 4096;
}

// (Re)allocate the gathered arrays on rank dst and map them everywhere.  Collective; every rank takes the same decision
// from the same counts.  Importers unmap before the exporter frees.
int ensure_gather_arrays(dcsg_comm* c, int dst, uint64_t vertices, uint64_t triangles) {
    dcsg_ctx* ctx = c->ctx;
    NcclApi* n = nccl_api();
    const bool same = c->dst == dst;
    const uint64_t capV = grown(same ? c->capVertices : 0, vertices), capT = grown(same ? c->capTriangles : 0, triangles);
    if (same && capV == c->capVertices && capT == c->capTriangles) return DCSG_OK;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (c->dst >= 0) {
        if (c->rank != c->dst)
            for (void*& p : c->arr) { if (p) cudaIpcCloseMemHandle(p); p = nullptr; }
        if (int rc = barrier(c)) return rc;
        if (c->rank == c->dst)
            for (void*& p : c->arr) { if (p) cudaFree(p); p = nullptr; }
        c->dst = -1;
        c->capVertices = c->capTriangles = 0;
    }
    cudaIpcMemHandle_t* h_handles = reinterpret_cast<cudaIpcMemHandle_t*>(host_words(c) + 288);
    uint8_t* d_handles = reinterpret_cast<uint8_t*>(dev_words(c) + 288);
    if (c->rank == dst) {
        for (int a = 0; a < kArrCount; a++) {
            const uint64_t items = a == kArrTriangles ? capT : capV;
            CUDA_TRY(ctx, cudaMalloc(&c->arr[a], items * kArrItemBytes[a]));        // plain cudaMalloc: pool memory cannot be exported
            CUDA_TRY(ctx, cudaIpcGetMemHandle(&h_handles[a], c->arr[a]));
        }
        CUDA_TRY(ctx, cudaMemcpyAsync(d_handles, h_handles, sizeof(cudaIpcMemHandle_t) * kArrCount, cudaMemcpyHostToDevice, ctx->stream));
    }
    NCCL_TRY(c, n->Broadcast(d_handles, d_handles, sizeof(cudaIpcMemHandle_t) * kArrCount, ncclUint8, dst, c->nccl, ctx->stream));
    if (c->rank != dst) {
        CUDA_TRY(ctx, cudaMemcpyAsync(h_handles, d_handles, sizeof(cudaIpcMemHandle_t) * kArrCount, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        for (int a = 0; a < kArrCount; a++) {
            const cudaError_t e = cudaIpcOpenMemHandle(&c->arr[a], h_handles[a], cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                cudaGetLastError();
                return fail(ctx, DCSG_ERR_UNSUPPORTED, format("cannot map the gathering rank's arrays into rank %d (%s): the mesh gather needs peer access "
                                                             "between the GPUs of the node", c->rank, cudaGetErrorString(e)));
            }
        }
    }
    c->dst = dst;
    c->capVertices = capV;
    c->capTriangles = capT;
    return barrier(c);
}

// ---- hooks called from inside dcsg_extract (host_extract.cu) -------------------------------------------------------
int exchange_pre(dcsg_ctx* ctx, void* user, const uint32_t* d_counts, cudaStream_t stream) {
    dcsg_comm* c = (dcsg_comm*)user;
    NcclApi* n = nccl_api();
    // the slab's counts block (32 words: {cells, triangles, vertices incl. halo copies, halo copies}, triangles per octree
    // level at [16 + l] in the adaptive walk) x world, gathered next to the extraction's own read-back
    uint32_t* d_all = reinterpret_cast<uint32_t*>(dev_words(c));
    NCCL_TRY(c, n->AllGather(d_counts, d_all, 32, ncclUint32, c->nccl, stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(host_words(c), d_all, (size_t)c->world * 128, cudaMemcpyDeviceToHost, stream));
    return DCSG_OK;
}

int exchange_post(dcsg_ctx* ctx, void* user, dcsg_mesher_params& mp) {
    dcsg_comm* c = (dcsg_comm*)user;
    const uint32_t* all = reinterpret_cast<const uint32_t*>(host_words(c));
    c->counts.assign((size_t)c->world * 4, 0);
    c->voff.assign(c->world + 1, 0);
    c->toff.assign(c->world + 1, 0);
    c->runs.clear();
    for (int r = 0; r < c->world; r++) {
        const uint32_t* mine = all + r * 32;
        uint64_t cells = mine[0], tris = mine[1], verts = mine[2], halo = mine[3];
        if (c->adaptive) {          // soup: the walk's triangles times what cms::retopologize makes of each, 3 fresh vertices per unit vertex
            tris *= c->unitTriangles;
            verts = mine[1] * c->unitVertices;
            halo = 0;
        }
        c->counts[r * 4 + 0] = verts - halo;
        c->counts[r * 4 + 1] = tris;
        c->counts[r * 4 + 2] = cells;
        c->counts[r * 4 + 3] = halo;
        c->voff[r + 1] = c->voff[r] + (verts - halo);
        c->toff[r + 1] = c->toff[r] + tris;
    }
    if (c->voff[c->world] >= 0xffffffffull || c->toff[c->world] * 3 >= 0xffffffffull)
        return fail(ctx, DCSG_ERR_INVALID, "the whole mesh exceeds 32-bit vertex / index counts");
    if (c->adaptive) {
        // canonical order of the adaptive walk = (octree level, node): this rank's triangles of level l follow those of
        // the ranks below on the same level and precede everybody's triangles of level l + 1
        uint64_t before = 0, local = 0;
        for (int lvl = 0; lvl < 16; lvl++) {
            uint64_t below = 0, level = 0;
            for (int r = 0; r < c->world; r++) {
                const uint64_t t = (uint64_t)all[r * 32 + 16 + lvl] * c->unitTriangles;
                if (r < c->rank) below += t;
                level += t;
            }
            const uint64_t mine = (uint64_t)all[c->rank * 32 + 16 + lvl] * c->unitTriangles;
            if (mine) c->runs.push_back(MeshStorage::Run{local, mine, before + below});
            local += mine;
            before += level;
        }
        return DCSG_OK;
    }
    if (!c->gather) return DCSG_OK;
    (void)mp;
    return ensure_gather_arrays(c, c->wantDst, c->voff[c->world], c->toff[c->world]);
}

// DCSG_TRACE=1: rank 0 prints the host-side wall time of every phase of the sharded calls (developer aid; nsys is not
// available on the boxes)
bool trace_on() {
    static const bool v = [] { const char* e = getenv("DCSG_TRACE"); return e && atoi(e) != 0; }();
    return v;
}
struct Trace {
    dcsg_comm* c;
    const char* what;
    double last;
    std::string line;
    Trace(dcsg_comm* comm, const char* name) : c(comm), what(name), last(now_ms()) {}
    void mark(const char* phase) {
        if (!trace_on() || c->rank != 0) return;
        const double t = now_ms();
        line += format(" %s %.3f", phase, t - last);
        last = t;
    }
    ~Trace() { if (trace_on() && c->rank == 0 && !line.empty()) fprintf(stderr, "[dcsg trace] %s:%s\n", what, line.c_str()); }
};

struct ReduceUser { dcsg_comm* c; };
int reduce_search(void* user, int* d_minmax, uint32_t* d_hist, cudaStream_t stream) {
    dcsg_comm* c = ((ReduceUser*)user)->c;
    NcclApi* n = nccl_api();
    NCCL_TRY(c, n->GroupStart());
    NCCL_TRY(c, n->AllReduce(d_minmax, d_minmax, 3, ncclInt32, ncclMin, c->nccl, stream));
    NCCL_TRY(c, n->AllReduce(d_minmax + 3, d_minmax + 3, 3, ncclInt32, ncclMax, c->nccl, stream));
    NCCL_TRY(c, n->AllReduce(d_hist, d_hist, 512, ncclUint32, ncclSum, c->nccl, stream));
    NCCL_TRY(c, n->GroupEnd());
    return DCSG_OK;
}

}  // namespace

dcsg_ctx* dcsg_host::comm_ctx(const dcsg_comm* c) { return c->ctx; }

extern "C" {

int dcsg_comm_unique_id(uint8_t id[DCSG_COMM_ID_BYTES]) {
    static_assert(sizeof(ncclUniqueId) == DCSG_COMM_ID_BYTES, "NCCL unique id size");
    NcclApi* n = nccl_api();
    if (!id || !n) return n ? DCSG_ERR_INVALID : DCSG_ERR_UNSUPPORTED;
    ncclUniqueId u;
    if (n->GetUniqueId(&u) != ncclSuccess) return DCSG_ERR_CUDA;
    memcpy(id, &u, sizeof(u));
    return DCSG_OK;
}

int dcsg_comm_create(dcsg_ctx* ctx, const uint8_t id[DCSG_COMM_ID_BYTES], int rank, int world, dcsg_comm** out) {
    if (!ctx || !id || !out || world < 1 || world > 16 || rank < 0 || rank >= world) return DCSG_ERR_INVALID;
    *out = nullptr;
    std::lock_guard<std::mutex> g(ctx->lock);
    NcclApi* n = nccl_api();
    if (!n) return fail(ctx, DCSG_ERR_UNSUPPORTED, "NCCL is not available: libnccl.so.2 could not be loaded (set DCSG_NCCL_LIBRARY to its path)");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    dcsg_comm* c = new dcsg_comm();
    c->ctx = ctx;
    c->rank = rank;
    c->world = world;
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    ncclResult_t r = n->CommInitRank(&c->nccl, world, u, rank);
    if (r != ncclSuccess) { delete c; return fail(ctx, DCSG_ERR_CUDA, std::string("ncclCommInitRank: ") + n->GetErrorString(r)); }
    if (c->dev.reserve(4096) != cudaSuccess || c->host.reserve(4096) != cudaSuccess || cudaMemset(c->dev.ptr, 0, 4096) != cudaSuccess) {
        n->CommDestroy(c->nccl);
        delete c;
        return fail(ctx, DCSG_ERR_CUDA, "dcsg_comm_create: out of memory");
    }
    ctx->node_ranks = world;        // one node: the ranks share the host's cores and memory bandwidth (file pipeline defaults)
    *out = c;
    return DCSG_OK;
}

void dcsg_comm_destroy(dcsg_comm* c) {
    if (!c) return;
    dcsg_ctx* ctx = c->ctx;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->exchange_user == c) { ctx->exchange_pre = nullptr; ctx->exchange_post = nullptr; ctx->exchange_user = nullptr; }
    ctx->node_ranks = 1;
    if (c->dst >= 0) {
        for (void*& p : c->arr) {
            if (!p) continue;
            if (c->rank == c->dst) cudaFree(p); else cudaIpcCloseMemHandle(p);
            p = nullptr;
        }
    }
    c->dev.release();
    c->host.release();
    if (c->nccl && nccl_api()) nccl_api()->CommDestroy(c->nccl);
    delete c;
}

int dcsg_comm_rank(const dcsg_comm* c) { return c ? c->rank : -1; }
int dcsg_comm_world(const dcsg_comm* c) { return c ? c->world : 0; }

int dcsg_comm_barrier(dcsg_comm* c) {
    if (!c) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(c->ctx->lock);
    CUDA_TRY(c->ctx, cudaSetDevice(c->ctx->device));
    return barrier(c);
}

int dcsg_bbox_sharded(dcsg_ctx* ctx, dcsg_comm* c, float search_diameter, float* box6) {
    if (!ctx || !c || c->ctx != ctx || !box6) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    // ix columns of the 256^3 search in equal shares; every rank ends up with the same box and the same histogram
    const int a = 256 * c->rank / c->world, b = 256 * (c->rank + 1) / c->world;
    ReduceUser user{c};
    Trace trace(c, "bbox_sharded");
    const int rc = bbox_locked(ctx, search_diameter, box6, a, b, c->world > 1 ? reduce_search : nullptr, &user);
    trace.mark("search+allreduce");
    return rc;
}

int dcsg_extract_sharded(dcsg_ctx* ctx, dcsg_comm* c, const dcsg_extract_cfg* cfg_in, int gather_to, dcsg_mesh* local, dcsg_mesh* whole,
                         dcsg_shard_info* info) {
    if (!ctx || !c || c->ctx != ctx || !cfg_in || !local) return DCSG_ERR_INVALID;
    if (gather_to >= c->world || (gather_to >= 0 && cfg_in->defer_projection)) return DCSG_ERR_INVALID;
    const bool uniform = cfg_in->min_level >= cfg_in->grid_level && cfg_in->max_level == cfg_in->grid_level;
    if (!uniform && gather_to >= 0)
        return fail(ctx, DCSG_ERR_UNSUPPORTED, "adaptive octree levels: the ranks keep their slabs of the soup (gather_to = -1; dcsg_export_sharded writes the files)");
    if (cfg_in->max_level > cfg_in->grid_level || cfg_in->max_level < 0 || cfg_in->min_level < 0 || cfg_in->grid_level < 3 || cfg_in->grid_level > 11)
        return fail(ctx, DCSG_ERR_INVALID, "octree levels must satisfy 0 <= min, 0 <= max <= grid level, 3 <= grid level <= 11");
    dcsg_extract_cfg cfg = *cfg_in;
    {
        std::lock_guard<std::mutex> g(ctx->lock);
        // uniform lattice: boundaries on any layer (a flat face of a design puts a tenth of a rank's triangles into ONE layer:
        // on multiples of 8 layers Design1's end slabs came out 13 % short); adaptive walk: on whole level-`min` nodes, so that
        // every node that can emit lies inside one slab
        const int minLevel = std::min(cfg.min_level, cfg.max_level);
        const int granularity = uniform ? 1 : (1 << (cfg.grid_level - minLevel));
        c->adaptive = !uniform;
        const uint64_t points = (!uniform && cfg.retopologize) ? (1ull << (cfg.grid_level - minLevel)) : 1ull;
        c->unitTriangles = points >= 2 ? 3 * points - 2 : 1;
        c->unitVertices = points >= 2 ? 3 * points : 3;
        if (int rc = plan_slabs_locked(ctx, cfg.box, cfg.grid_level, c->world, granularity, c->slab)) return rc;
        c->gather = gather_to >= 0;
        c->wantDst = gather_to >= 0 ? gather_to : 0;
        c->wantNormals = cfg.want_normals != 0;
        ctx->exchange_pre = exchange_pre;
        ctx->exchange_post = exchange_post;
        ctx->exchange_user = c;
        // the projection is queued right behind the emitters: no host round trip in between (not when the caller projects itself)
        ctx->skip_final_sync = !cfg_in->defer_projection;
    }
    cfg.slab_z0 = c->slab[c->rank];
    cfg.slab_z1 = c->slab[c->rank + 1];
    cfg.defer_projection = 1;
    cfg.copy_to_host = 0;
    const int gd_steps = cfg.gd_steps, want_normals = cfg.want_normals;
    Trace trace(c, "extract_sharded");
    trace.mark("plan");
    int rc = dcsg_extract(ctx, &cfg, local);
    trace.mark("extract");
    {
        std::lock_guard<std::mutex> g(ctx->lock);
        ctx->exchange_pre = nullptr;
        ctx->exchange_post = nullptr;
        ctx->exchange_user = nullptr;
        ctx->skip_final_sync = false;
    }
    if (rc != DCSG_OK) return rc;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    MeshStorage* st = (MeshStorage*)local->reserved;
    st->runs = c->runs;             // adaptive: where this rank's triangles sit in the whole mesh, level by level
    float* d_normals = nullptr;
    if (want_normals) {
        CUDA_TRY(ctx, st->normals.reserve(std::max<uint64_t>(local->num_vertices, 1) * 12));
        d_normals = st->normals.as<float>();
    }
    local->d_normals = d_normals;
    if (info) {
        memset(info, 0, sizeof(*info));
        info->rank = c->rank;
        info->world = c->world;
        info->slab_z0 = cfg.slab_z0;
        info->slab_z1 = cfg.slab_z1;
        info->first_vertex = c->voff[c->rank];
        info->first_triangle = c->toff[c->rank];
        info->total_vertices = c->voff[c->world];
        info->total_triangles = c->toff[c->world];
        for (int r = 0; r < c->world; r++) info->total_cells += c->counts[r * 4 + 2];
    }
    if (!cfg_in->defer_projection) {
        float* gv = c->gather ? reinterpret_cast<float*>(c->arr[kArrVertices]) + c->voff[c->rank] * 3 : nullptr;
        float* gn = c->gather && d_normals ? reinterpret_cast<float*>(c->arr[kArrNormals]) + c->voff[c->rank] * 3 : nullptr;
        if (c->gather) {
            // keys and triangles are final after the emitters: they travel on the side stream, under the projection -- the keys
            // as they are (copy engine over NVLink), the triangles with the slab's vertex offset added (global ids).  (Stored by
            // the emitters themselves, seven ranks' 140 MB arrived at the gathering rank at once and sat on everybody's
            // critical path: 0.2 ms of a 2.4 ms step at eight GPUs.)
            CUDA_TRY(ctx, cudaEventRecord(ctx->aux_ready, ctx->stream));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->aux_ready, 0));
            if (local->owned_vertices)
                CUDA_TRY(ctx, cudaMemcpyAsync(reinterpret_cast<uint64_t*>(c->arr[kArrKeys]) + c->voff[c->rank], local->d_vertex_keys,
                                              local->owned_vertices * 8, cudaMemcpyDefault, ctx->aux_stream));
            dcsg_launch_rebase_indices(local->d_triangles, local->num_triangles * 3, (uint32_t)c->voff[c->rank],
                                       reinterpret_cast<uint32_t*>(c->arr[kArrTriangles]) + c->toff[c->rank] * 3, ctx->sm_count, ctx->aux_stream);
            ++g_launches;
            CUDA_TRY(ctx, cudaGetLastError());
            CUDA_TRY(ctx, cudaEventRecord(ctx->aux_done, ctx->aux_stream));
            ctx->aux_pending = true;
        }
        if (local->num_vertices && (gd_steps > 0 || d_normals || gv)) {
            if (int prc = launch_project(ctx, local->d_vertices, local->num_vertices, gd_steps, d_normals, ctx->stream, 0, gv, gn, local->owned_vertices)) return prc;
        }
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[6], ctx->stream));
        if (c->gather) CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->aux_done, 0));      // the completion signal covers the side stream
        trace.mark("launch_project");
        // everybody's stores have landed in the gathering rank's arrays once the one-word all-reduce is through
        if (int brc = barrier(c)) return brc;
        trace.mark("project+barrier");
        for (int i = 0; i < 3; i++) cudaEventElapsedTime(&local->stage_ms[i], ctx->ev[i], ctx->ev[i + 1]);      // dcsg_extract left them unread
        cudaEventElapsedTime(&local->stage_ms[DCSG_STAGE_PROJECT], ctx->ev[5], ctx->ev[6]);
        local->stage_ms[DCSG_STAGE_COPY] = 0.0f;
    }
    if (whole) {
        memset(whole, 0, sizeof(*whole));
        whole->num_vertices = whole->owned_vertices = c->voff[c->world];
        whole->num_triangles = c->toff[c->world];
        for (int r = 0; r < c->world; r++) whole->num_cells += c->counts[r * 4 + 2];
        if (c->gather && c->rank == c->dst && !cfg_in->defer_projection) {       // borrowed views of the communicator's arrays
            whole->d_vertex_keys = reinterpret_cast<uint64_t*>(c->arr[kArrKeys]);
            whole->d_triangles = reinterpret_cast<uint32_t*>(c->arr[kArrTriangles]);
            whole->d_vertices = reinterpret_cast<float*>(c->arr[kArrVertices]);
            whole->d_normals = d_normals ? reinterpret_cast<float*>(c->arr[kArrNormals]) : nullptr;
        }
    }
    return DCSG_OK;
}

}  // extern "C"
