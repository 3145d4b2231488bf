// host_extract.cu -- lattice passes and dcsg_extract: dense / octree-ordered sparse lattice, classify, emit, adaptive
// octree mode, projection.  Replaces ISV3D64 (master/ISV.hpp), cms::Mesh::getSurface, retopologize and
// performGradientDescent (master/cms/main/Headers/mesh.hpp:82-593) as driven by MyFrame::OnExportInner
// (master/DesignCSG.cpp:638-790).  Everything between "scene compiled" and "mesh arrays" stays in HBM; one host round
// trip per extraction (the mesh size).
#include "host_internal.h"

using namespace dcsg_host;

namespace dcsg_host {

// The dense restatement is only valid when the reference's own arithmetic puts every octree corner and
// centre exactly on the lattice (SURVEY.md 8a "Geometry of the closed form"); this walks the octree's
// recursive halving per axis (octree.hpp:24-32, geometry.hpp:264-279) and the lattice snap
// (ISV.hpp:91-96) and checks that they agree bit for bit.  True for every box dcsg_bbox produces from a
// dyadic search diameter (10.0 in all shipped designs).
bool lattice_is_exact(const LatticeSetup& s, const float* box, std::string& why) {
    const std::vector<float>* tables[3] = {&s.px, &s.py, &s.pz};
    for (int a = 0; a < 3; a++) {
        const float c0 = box[a], d = box[3 + a];
        const float h0 = d / 2.0f;                      // Box3f half diameter (DesignCSG.cpp:718)
        const std::vector<float>& t = *tables[a];
        const float w = (float)(int64_t)s.N;
        for (int i = 0; i <= s.N; i++) {                // lattice point snaps onto itself
            int64_t idx = (int64_t)(w * (t[i] - c0 + d / 2.0f) / d);
            if (idx != i) { why = format("axis %d: lattice point %d snaps to %lld", a, i, (long long)idx); return false; }
        }
        // every node of every level once (2N per axis): a child's centre is its parent's plus or minus half the
        // parent's half diameter (octree.hpp:24-32 through getCorners(0.5), geometry.hpp:264-279)
        std::vector<float> centres(1, c0), next;
        float h = h0;
        for (int lvl = 0; lvl <= s.L; lvl++) {
            const int sh = s.L - lvl;                   // a node spans 2^sh cells
            for (int node = 0; node < (1 << lvl); node++) {
                const float c = centres[node];
                // getCorners(1.0): what corner masks, edge midpoints and (adaptive mode) coarse leaves are built from
                const float lo = c + 1.0f * (h * -1.0f), hi = c + 1.0f * (h * 1.0f);
                if (lo != t[node << sh] || hi != t[(node + 1) << sh]) { why = format("axis %d: level %d node corners off the lattice", a, lvl); return false; }
                if (lvl < s.L) {
                    if (c != t[(node << sh) + (1 << (sh - 1))]) { why = format("axis %d: level %d node centre off the lattice", a, lvl); return false; }
                } else {
                    const int64_t idx = (int64_t)(w * (c - c0 + d / 2.0f) / d);      // leaf centre truncates to the min corner
                    if (idx != node) { why = format("axis %d: leaf centre %d snaps to %lld", a, node, (long long)idx); return false; }
                }
            }
            if (lvl == s.L) break;
            next.resize((size_t)2 << lvl);
            for (int node = 0; node < (1 << lvl); node++) {
                next[2 * node] = centres[node] + 0.5f * (h * -1.0f);       // centre.sum(half.termProduct(sign).scaled(0.5))
                next[2 * node + 1] = centres[node] + 0.5f * (h * 1.0f);
            }
            centres.swap(next);
            h = 0.5f * h;
        }
    }
    return true;
}

int setup_lattice(dcsg_ctx* ctx, const float* box, int grid_level, int z0, int z1, LatticeSetup& s, bool check) {
    if (grid_level < 3 || grid_level > 11) return fail(ctx, DCSG_ERR_INVALID, "grid_level must be in [3, 11]");
    s.L = grid_level;
    s.N = 1 << grid_level;
    s.P = s.N + 1;
    if (z0 == 0 && z1 == 0) z1 = s.N;
    if (z0 < 0 || z1 > s.N || z0 >= z1) return fail(ctx, DCSG_ERR_INVALID, "bad slab range");
    s.z0 = z0;
    s.nzc = z1 - z0;
    s.nzp = s.nzc + 1;
    s.pitch = (s.P + 31) / 32 * 32;         // rows start on word boundaries: +pitch is a whole-word step
    const uint64_t PB = (uint64_t)s.pitch * s.P;                        // bits per plane
    s.planeWords = (uint32_t)((PB + 127) / 128) * 4;
    if ((uint64_t)s.planeWords * (uint64_t)s.nzp >= 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "slab too large for 32-bit word indices");
    const float* c = box;
    const float* d = box + 3;
    std::vector<float>* tables[3] = {&s.px, &s.py, &s.pz};
    for (int a = 0; a < 3; a++) {
        tables[a]->assign(s.pitch, 0.0f);                   // entries past P are padding
        const float origin = c[a] - 0.5f * d[a];            // v3f_sub(center, v3f_scale(diameters, 0.5))
        for (int i = 0; i < s.P; i++) (*tables[a])[i] = origin + d[a] * (float)i / (float)(int64_t)s.N;
    }
    // cull thresholds: halfDiameter.magnitude() * 1.1f per level (mesh.hpp:167-170, geometry.hpp:75-77)
    float h[3] = {d[0] / 2.0f, d[1] / 2.0f, d[2] / 2.0f};
    for (int lvl = 0; lvl <= s.L; lvl++) {
        const float mag = sqrtf(h[0] * h[0] + h[1] * h[1] + h[2] * h[2]);
        const float thr = mag * 1.1f;
        if (lvl < s.L) s.coarseThr[lvl] = thr; else s.leafThr = thr;
        for (int a = 0; a < 3; a++) h[a] = 0.5f * h[a];
    }
    s.thickMask = 0;
    for (int lvl = 0; lvl < s.L; lvl++) {
        const int size = 1 << (s.L - lvl);
        if (!(size <= s.nzc && (s.z0 % size) == 0 && (s.nzc % size) == 0)) s.thickMask |= 1u << lvl;
    }
    if (check) {
        std::string why;
        if (!lattice_is_exact(s, box, why)) return fail(ctx, DCSG_ERR_LATTICE, "bounding box is not exact on the lattice: " + why);
    }
    return DCSG_OK;
}

// device copies of the axis tables + everything dcsg_k_lattice needs; launches it
int run_lattice(dcsg_ctx* ctx, const LatticeSetup& s, float* d_values, dcsg_lattice_params& lp) {
    if (ctx->aux_pending) {         // a sparse extraction's clean-up pass may still be zeroing the bitmaps this pass writes
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->aux_done, 0));
        ctx->aux_pending = false;
    }
    ctx->sparse_clean = false;
    const size_t planeBytes = (size_t)s.planeWords * 4;
    const size_t padWords = (size_t)s.planeWords + 64;
    CUDA_TRY(ctx, ctx->axes.reserve((size_t)3 * s.pitch * 4));
    CUDA_TRY(ctx, ctx->sign.reserve(planeBytes * s.nzp + padWords * 4));
    CUDA_TRY(ctx, ctx->leaf.reserve(planeBytes * s.nzp + padWords * 4));
    CUDA_TRY(ctx, ctx->cfail.reserve(planeBytes * s.nzp + padWords * 4));
    uint64_t off = 0;
    memset(&lp, 0, sizeof(lp));
    for (int lvl = 0; lvl < s.L; lvl++) {       // node bitmaps exist for thick levels only
        lp.coarseOff[lvl] = off;
        if ((s.thickMask >> lvl) & 1u) off += ((1ull << (3 * lvl)) + 31) / 32;
    }
    CUDA_TRY(ctx, ctx->coarse.reserve((size_t)(off + 16) * 4));
    float* ax = ctx->axes.as<float>();
    CUDA_TRY(ctx, cudaMemcpyAsync(ax, s.px.data(), (size_t)s.pitch * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ax + s.pitch, s.py.data(), (size_t)s.pitch * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ax + 2 * s.pitch, s.pz.data(), (size_t)s.pitch * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->coarse.ptr, 0, (size_t)(off + 16) * 4, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->sign.as<uint8_t>() + planeBytes * s.nzp, 0, padWords * 4, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->leaf.as<uint8_t>() + planeBytes * s.nzp, 0, padWords * 4, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->cfail.as<uint8_t>() + planeBytes * s.nzp, 0, padWords * 4, ctx->stream));
    lp.px = ax;
    lp.py = ax + s.pitch;
    lp.pz = ax + 2 * s.pitch;
    lp.P = s.P;
    lp.pitch = s.pitch;
    lp.z0 = s.z0;
    lp.nzp = s.nzp;
    lp.L = s.L;
    lp.planeWords = s.planeWords;
    lp.sign = ctx->sign.as<uint32_t>();
    lp.leaf = ctx->leaf.as<uint32_t>();
    lp.cfail = ctx->cfail.as<uint32_t>();
    lp.values = d_values;
    lp.leafThr = s.leafThr;
    for (int lvl = 0; lvl < s.L; lvl++) lp.coarseThr[lvl] = s.coarseThr[lvl];
    lp.coarse = ctx->coarse.as<uint32_t>();
    void* args[] = {&lp};
    const uint32_t groups = (uint32_t)(s.pitch / DCSG_LATTICE_SPT) * (uint32_t)s.P;     // one thread per group of SPT samples
    dim3 grid((groups + 255) / 256, (unsigned)s.nzp, 1);
    CUDA_TRY(ctx, launch(ctx->k_lattice, grid, dim3(256), args, ctx->stream, ctx->scene.private_words));
    // octree levels whose nodes are thicker than the slab: their centres may lie on another rank's planes,
    // so the few nodes that touch the slab are evaluated separately into per-level node bitmaps
    if (s.thickMask) {
        std::vector<int> nodes;
        for (int lvl = 0; lvl < s.L; lvl++) {
            if (!((s.thickMask >> lvl) & 1u)) continue;
            const int sh = s.L - lvl, size = 1 << sh, n = 1 << lvl;
            for (int nz = s.z0 >> sh; nz <= (s.z0 + s.nzc - 1) >> sh; nz++)
                for (int ny = 0; ny < n; ny++)
                    for (int nx = 0; nx < n; nx++) {
                        nodes.push_back((nx << sh) + (size >> 1));
                        nodes.push_back((ny << sh) + (size >> 1));
                        nodes.push_back((nz << sh) + (size >> 1));
                        nodes.push_back(lvl);
                    }
        }
        if (!nodes.empty()) {
            const int n = (int)(nodes.size() / 4);
            CUDA_TRY(ctx, ctx->small.reserve(std::max<size_t>(nodes.size() * 4, 4096)));
            CUDA_TRY(ctx, cudaMemcpyAsync(ctx->small.ptr, nodes.data(), nodes.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));      // `nodes` is pageable stack-owned memory
            const void* dn = ctx->small.ptr;
            void* cargs[] = {&lp, &dn, (void*)&n};
            CUDA_TRY(ctx, launch(ctx->k_coarse_nodes, dim3((n + 255) / 256), dim3(256), cargs, ctx->stream, ctx->scene.private_words));
        }
    }
    return DCSG_OK;
}

// Sparse form of the lattice pass: walk the octree levels top-down on the device, evaluating only the samples
// the reference's walk evaluates (scene_kernels.cuh "descent").  Produces sign bits (valid at the corners of
// surviving cells), the surviving-leaf bitmap and the work lists of everything that follows: the words of the leaf
// bitmap that are not zero (-> classify, emit) and the sample words next to them (-> corner pass).  The leaf and the
// alive bitmap are all-zero outside the words this extraction writes; dcsg_extract zeroes those again at its end
// (dcsg_launch_cleanup), so nothing ever sweeps the whole lattice.  d_evals receives the number of SDF evaluations.
struct SparseLists {
    uint32_t* counts;           // device: [1] alive leaf words, [2] corner words, [3] vertex words, [8 + l] alive words of level l
    uint32_t* parentList;
    uint32_t* cellList;
    uint32_t* cornerList;
    uint32_t* vertList;
    uint32_t* leafMask;
    uint32_t* leafMask31;
    uint32_t* aliveMask;
    uint32_t* aliveMask31;
    uint32_t* scratch;
    uint32_t numBits, rowWords;
};

constexpr int kFirstListLevel = 4;      // grid levels are >= 3, so level L-1 >= 2; levels below this one sweep their bitmaps

int run_descent(dcsg_ctx* ctx, const LatticeSetup& s, dcsg_leaf_params& lf, uint64_t** d_evals, SparseLists& sl) {
    const size_t planeBytes = (size_t)s.planeWords * 4;
    const size_t padWords = (size_t)s.planeWords + 64;
    const size_t bitmapBytes = planeBytes * s.nzp + padWords * 4;
    CUDA_TRY(ctx, ctx->axes.reserve((size_t)3 * s.pitch * 4));
    CUDA_TRY(ctx, ctx->sign.reserve(bitmapBytes));
    // the two bitmaps that must be all-zero where this extraction does not write: fresh or foreign memory is cleared once
    {
        const void* before[2] = {ctx->leaf.ptr, ctx->alive.ptr};
        CUDA_TRY(ctx, ctx->leaf.reserve(bitmapBytes));              // reused as leafAlive
        CUDA_TRY(ctx, ctx->alive.reserve(bitmapBytes));
        if (!ctx->sparse_clean || before[0] != ctx->leaf.ptr || before[1] != ctx->alive.ptr) {
            CUDA_TRY(ctx, cudaMemsetAsync(ctx->leaf.ptr, 0, ctx->leaf.cap, ctx->stream));
            CUDA_TRY(ctx, cudaMemsetAsync(ctx->alive.ptr, 0, ctx->alive.cap, ctx->stream));
        }
        ctx->sparse_clean = false;                                  // until the clean-up pass of this extraction has been queued
    }
    // per-level node bitmaps, full size (sum over levels ~ N^3/7 bits)
    std::vector<uint64_t> off(s.L + 1, 0);
    for (int lvl = 0; lvl < s.L; lvl++) {
        const uint64_t n = 1ull << lvl, q = n < 32 ? 32 : n;
        off[lvl + 1] = off[lvl] + q * n * n / 32;
    }
    // (+ two more bitmaps of level L-1's size: the verdicts of its centre samples, reused by the leaf pass)
    const uint64_t lastLevelWords = off[s.L] - off[s.L - 1];
    CUDA_TRY(ctx, ctx->levels.reserve((size_t)(off[s.L] + 2 * lastLevelWords + 64) * 4));
    CUDA_TRY(ctx, ctx->small.reserve(4096));
    // work lists and word masks
    const uint32_t numVertWords = s.planeWords * (uint32_t)s.nzp;
    const uint32_t maskWords = (numVertWords + 31u) / 32u + 2u;
    const uint32_t maskTiles = (maskWords + 1023u) / 1024u;          // CTAs of the work-list kernels (mesher_kernels.cu kWorklistTile)
    // words of the finest coarse level that can touch the slab: capacity of the two per-level parent lists (ping-pong)
    const uint64_t lastN = 1ull << (s.L - 1), lastQ = lastN < 32 ? 32 : lastN;
    const uint64_t lastLayers = (uint64_t)(((s.z0 + s.nzc - 1) >> 1) - (s.z0 >> 1) + 1);
    const uint64_t parentCap = lastQ / 32 * lastN * lastLayers;
    CUDA_TRY(ctx, ctx->lists.reserve(((size_t)parentCap * 2 + (size_t)numVertWords * 3 + 64) * 4));
    CUDA_TRY(ctx, ctx->masks.reserve(((size_t)maskWords * 5 + (size_t)maskTiles * 2 + 64) * 4));
    uint32_t* parentLists[2] = {ctx->lists.as<uint32_t>(), ctx->lists.as<uint32_t>() + parentCap};
    sl.cellList = parentLists[1] + parentCap;
    sl.cornerList = sl.cellList + numVertWords;
    sl.vertList = sl.cornerList + numVertWords;
    sl.leafMask = ctx->masks.as<uint32_t>();
    sl.leafMask31 = sl.leafMask + maskWords;
    sl.aliveMask = sl.leafMask31 + maskWords;
    sl.aliveMask31 = sl.aliveMask + maskWords;
    uint32_t* candMask = sl.aliveMask31 + maskWords;
    sl.scratch = candMask + maskWords;
    // bytes 640 .. 767 of `small` (between the evaluation counter and the search histogram): [0] unused, [1] alive leaf
    // words, [2] corner words, [3] vertex words, [8 + l] words of level l that hold an alive node
    sl.counts = ctx->small.as<uint32_t>() + 160;
    sl.numBits = numVertWords;
    sl.rowWords = (uint32_t)s.pitch >> 5;
    CUDA_TRY(ctx, cudaMemsetAsync(sl.leafMask, 0, (size_t)maskWords * 5 * 4, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(sl.counts, 0, 128, ctx->stream));
    float* ax = ctx->axes.as<float>();
    CUDA_TRY(ctx, cudaMemcpyAsync(ax, s.px.data(), (size_t)s.pitch * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ax + s.pitch, s.py.data(), (size_t)s.pitch * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ax + 2 * s.pitch, s.pz.data(), (size_t)s.pitch * 4, cudaMemcpyHostToDevice, ctx->stream));
    uint64_t* counter = ctx->small.as<uint64_t>() + 64;         // away from the bbox slots
    CUDA_TRY(ctx, cudaMemsetAsync(counter, 0, 8, ctx->stream));
    uint32_t* levels = ctx->levels.as<uint32_t>();
    // the first levels (a few thousand nodes between them) run in one launch of one CTA: dcsg_k_descend_top
    dcsg_descend_top_params top;
    memset(&top, 0, sizeof(top));
    static const int topWanted = [] { const char* e = getenv("DCSG_TOP_LEVELS"); return e ? atoi(e) : DCSG_TOP_DEFAULT; }();
    const int topLevels = std::max(0, std::min(std::min(topWanted, DCSG_TOP_LEVELS), s.L));
    for (int lvl = 0; lvl < s.L; lvl++) {
        dcsg_descend_params dp;
        memset(&dp, 0, sizeof(dp));
        dp.px = ax; dp.py = ax + s.pitch; dp.pz = ax + 2 * s.pitch;
        dp.L = s.L;
        dp.level = lvl;
        const int sh = s.L - lvl;
        dp.nzLo = s.z0 >> sh;
        dp.nzCount = ((s.z0 + s.nzc - 1) >> sh) - dp.nzLo + 1;
        dp.parent = lvl ? levels + off[lvl - 1] : nullptr;
        dp.out = levels + off[lvl];
        dp.thr = s.coarseThr[lvl];
        dp.evalCount = (dcsg_u64*)counter;
        // levels 0 .. 3 sweep their (tiny) bitmaps; from level 4 on a level follows the list of the previous level's words
        // that hold an alive node.  Every level from 3 on produces such a list for the next one.
        const bool fromList = lvl >= kFirstListLevel;
        if (lvl >= kFirstListLevel - 1 || lvl == s.L - 1) { dp.outList = parentLists[lvl & 1]; dp.outCount = sl.counts + 8 + lvl; }
        if (fromList) { dp.parentList = parentLists[(lvl - 1) & 1]; dp.parentCount = sl.counts + 8 + lvl - 1; }
        if (fromList && lvl == s.L - 1) {
            dp.centreSign = levels + off[s.L];
            dp.centreAlive = levels + off[s.L] + lastLevelWords;
            dp.leafThr = s.leafThr;
        }
        if (lvl < topLevels) {
            top.level[top.count++] = dp;
            if (lvl == topLevels - 1) {
                void* targs[] = {&top};
                CUDA_TRY(ctx, launch(ctx->k_descend_top, dim3(1), dim3(256), targs, ctx->stream, ctx->scene.private_words));
            }
            continue;
        }
        const uint64_t n = 1ull << lvl, q = n < 32 ? 32 : n;
        const uint64_t words = q / 32 * n * (uint64_t)dp.nzCount;
        void* args[] = {&dp};
        if (fromList) {
            const uint64_t parentWords = std::max<uint64_t>(1, words / 8);          // upper bound of the list's length
            const unsigned ctas = (unsigned)std::min<uint64_t>((uint64_t)ctx->sm_count * 6, (parentWords + 3) / 4);
            CUDA_TRY(ctx, launch(ctx->k_descend_list, dim3(std::max(1u, ctas)), dim3(256), args, ctx->stream, ctx->scene.private_words));
        } else {
            CUDA_TRY(ctx, launch(ctx->k_descend, dim3((unsigned)((words + 255) / 256)), dim3(256), args, ctx->stream, ctx->scene.private_words));
        }
    }
    const int lastLevel = s.L - 1;
    sl.parentList = parentLists[lastLevel & 1];
    uint32_t* parentCount = sl.counts + 8 + lastLevel;
    memset(&lf, 0, sizeof(lf));
    lf.px = ax; lf.py = ax + s.pitch; lf.pz = ax + 2 * s.pitch;
    lf.L = s.L; lf.N = s.N; lf.P = s.P; lf.pitch = s.pitch;
    lf.z0 = s.z0; lf.nzc = s.nzc; lf.nzp = s.nzp;
    lf.planeWords = s.planeWords;
    lf.parent = levels + off[s.L - 1];
    lf.leafAlive = ctx->leaf.as<uint32_t>();
    lf.sign = ctx->sign.as<uint32_t>();
    lf.leafThr = s.leafThr;
    lf.evalCount = (dcsg_u64*)counter;
    lf.parentList = sl.parentList; lf.parentCount = parentCount;
    if (s.L - 1 >= kFirstListLevel) { lf.centreSign = levels + off[s.L]; lf.centreAlive = levels + off[s.L] + lastLevelWords; }
    lf.leafMask = sl.leafMask;
    lf.leafMask31 = sl.leafMask31;
    lf.candMask = candMask;
    lf.cornerList = sl.cornerList; lf.cornerCount = sl.counts + 2;
    void* largs[] = {&lf};
    // persistent grids: the list lengths only exist on the device
    const dim3 grid((unsigned)(ctx->sm_count * 6), 1, 1);
    CUDA_TRY(ctx, launch(ctx->k_leaf, grid, dim3(256), largs, ctx->stream, ctx->scene.private_words));
    dcsg_worklist_params wl;
    memset(&wl, 0, sizeof(wl));
    wl.mask = sl.leafMask; wl.mask31 = sl.leafMask31; wl.numBits = sl.numBits; wl.rowWords = sl.rowWords; wl.planeWords = s.planeWords;
    wl.mode = 0; wl.listA = sl.cellList; wl.listB = sl.cornerList; wl.counts = sl.counts + 1; wl.scratch = sl.scratch;
    dcsg_launch_worklists(wl, ctx->stream); g_launches += 2;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, launch(ctx->k_corners, grid, dim3(256), largs, ctx->stream, ctx->scene.private_words));
    *d_evals = counter;
    return DCSG_OK;
}

// ---------------------------------------------------------------------------------------------------------
// adaptive octree mode (reference mesh.hpp:212-267 + retopologize :432-529): dense lattice bitmaps, one
// dcsg_k_adapt_level launch per octree level, then soup emission from the per-level leaf bitmaps.
// Records ev[1] (lattice done), ev[2] (levels decided + counted), ev[3] (soup emitted / retopologized).
// ---------------------------------------------------------------------------------------------------------
int extract_adaptive(dcsg_ctx* ctx, const dcsg_extract_cfg* cfg, const LatticeSetup& s, MeshStorage* st, uint64_t& nVerts,
                     uint64_t& nTris, uint64_t& nCells, uint64_t& evals) {
    cudaStream_t stream = ctx->stream;
    const int maxLevel = cfg->max_level;
    const int minLevel = std::min(cfg->min_level, cfg->max_level);     // level == max never splits (mesh.hpp:265-267)
    // z-slabs: every node that can emit (level >= min) must lie inside one slab
    {
        const int unit = 1 << (s.L - minLevel);
        if (s.z0 % unit != 0 || (s.z0 + s.nzc) % unit != 0)
            return fail(ctx, DCSG_ERR_INVALID, format("adaptive octree levels: z-slab boundaries must be multiples of %d cell layers (the size of a level-%d node)", unit, minLevel));
    }
    dcsg_lattice_params lp;
    int rc = run_lattice(ctx, s, nullptr, lp);
    if (rc != DCSG_OK) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], stream));

    // where the reference's edge samples land on the lattice (mesh.hpp:221-238 through ISV.hpp:91-96):
    // sample i of an edge from `start` to `end` is start + (end - start) * (i / points), truncated onto the
    // lattice.  Per tested level, axis and walking direction: snapped index of the sample nominally at j.
    const int numTested = std::max(0, maxLevel - minLevel);
    std::vector<int> snap((size_t)std::max(1, numTested) * 6 * s.P, 0);
    const std::vector<float>* tables[3] = {&s.px, &s.py, &s.pz};
    for (int lvl = minLevel; lvl < maxLevel; lvl++) {
        const int sh = s.L - lvl, size = 1 << sh;
        for (int a = 0; a < 3; a++) {
            const std::vector<float>& t = *tables[a];
            const float c0 = cfg->box[a], d = cfg->box[3 + a], w = (float)(int64_t)s.N;
            for (int dir = 0; dir < 2; dir++) {
                int* row = &snap[((size_t)(lvl - minLevel) * 6 + a * 2 + dir) * s.P];
                for (int j = 0; j <= s.N; j++) {
                    const int s0 = (j >> sh) << sh;
                    if (j == s0) { row[j] = j; continue; }              // a node corner, not an interior sample
                    const int s1 = s0 + size;
                    const int i = dir == 0 ? j - s0 : s1 - j;
                    const float start = dir == 0 ? t[s0] : t[s1], end = dir == 0 ? t[s1] : t[s0];
                    const float delta = end - start;
                    const float fraction = (float)i / (float)size;
                    const float point = start + fraction * delta;
                    int64_t idx = (int64_t)(w * (point - c0 + d / 2.0f) / d);
                    if (idx < 0 || idx > s.N) return fail(ctx, DCSG_ERR_LATTICE, "edge sample snaps outside the lattice");
                    row[j] = (int)idx;
                }
            }
        }
    }
    CUDA_TRY(ctx, ctx->adapt_snap.reserve(snap.size() * 4));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->adapt_snap.ptr, snap.data(), snap.size() * 4, cudaMemcpyHostToDevice, stream));

    // per-level node bitmaps (split, emit), levels 0 .. maxLevel
    std::vector<uint64_t> off(maxLevel + 2, 0);
    for (int lvl = 0; lvl <= maxLevel; lvl++) {
        const uint64_t n = 1ull << lvl, q = n < 32 ? 32 : n;
        off[lvl + 1] = off[lvl] + q * n * n / 32;
    }
    if (off[maxLevel + 1] >= 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "octree too deep for 32-bit word indices");
    CUDA_TRY(ctx, ctx->levels.reserve((size_t)(off[maxLevel + 1] + 64) * 4));
    CUDA_TRY(ctx, ctx->adapt_emit.reserve((size_t)(off[maxLevel + 1] + 64) * 4));
    CUDA_TRY(ctx, ctx->small.reserve(4096));
    uint64_t* counter = ctx->small.as<uint64_t>() + 64;
    CUDA_TRY(ctx, cudaMemsetAsync(counter, 0, 8, stream));
    uint32_t* split = ctx->levels.as<uint32_t>();
    uint32_t* emit = ctx->adapt_emit.as<uint32_t>();
    for (int lvl = 0; lvl <= maxLevel; lvl++) {
        dcsg_adapt_params ap;
        memset(&ap, 0, sizeof(ap));
        ap.px = lp.px; ap.py = lp.py; ap.pz = lp.pz;
        ap.L = s.L; ap.level = lvl; ap.minLevel = minLevel; ap.maxLevel = maxLevel;
        ap.pitch = s.pitch; ap.planeWords = s.planeWords;
        ap.sign = lp.sign; ap.leaf = lp.leaf; ap.cfail = lp.cfail;
        ap.z0 = s.z0;
        ap.nodeZLo = s.z0 >> (s.L - lvl);
        ap.nodeZHi = ((s.z0 + s.nzc - 1) >> (s.L - lvl)) + 1;
        ap.coarse = lp.coarse;
        for (int l = 0; l < 16; l++) ap.coarseOff[l] = lp.coarseOff[l];
        ap.thickMask = s.thickMask;
        ap.parentSplit = lvl ? split + off[lvl - 1] : nullptr;
        ap.split = split + off[lvl];
        ap.emit = emit + off[lvl];
        ap.snap = ctx->adapt_snap.as<int>() + (size_t)std::max(0, std::min(lvl, maxLevel - 1) - minLevel) * 6 * s.P;
        ap.threshold = cfg->complex_threshold;
        ap.evalCount = (dcsg_u64*)counter;
        const uint64_t words = off[lvl + 1] - off[lvl];
        void* args[] = {&ap};
        CUDA_TRY(ctx, launch(ctx->k_adapt_level, dim3((unsigned)((words + 255) / 256)), dim3(256), args, stream, ctx->scene.private_words));
    }

    dcsg_adapt_emit_params ep;
    memset(&ep, 0, sizeof(ep));
    ep.g.N = s.N; ep.g.P = s.P; ep.g.L = s.L; ep.g.z0 = s.z0; ep.g.nzc = s.nzc; ep.g.nzp = s.nzp;
    ep.g.pitch = s.pitch; ep.g.planeWords = s.planeWords; ep.g.PB = (uint32_t)s.pitch * (uint32_t)s.P;
    ep.sign = lp.sign;
    ep.emit = emit;
    for (int lvl = 0; lvl <= maxLevel + 1; lvl++) ep.levelOff[lvl] = (uint32_t)off[lvl];
    ep.minLevel = minLevel; ep.maxLevel = maxLevel;
    ep.firstWord = (uint32_t)off[minLevel]; ep.endWord = (uint32_t)off[maxLevel + 1];
    ep.numTiles = (ep.endWord - ep.firstWord + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    // per-tile sums | counts block of 32 words: {cells, triangles, 0, 0} + triangles per octree level at [16 + level]
    CUDA_TRY(ctx, ctx->tiles.reserve(((size_t)ep.numTiles * 2 + 48) * 4));
    ep.tileCells = ctx->tiles.as<uint32_t>();
    ep.tileTris = ep.tileCells + ep.numTiles;
    uint32_t* d_counts = ep.tileTris + ep.numTiles;
    CUDA_TRY(ctx, cudaMemsetAsync(d_counts, 0, 32 * 4, stream));
    ep.levelTris = d_counts + 16;
    ep.px = lp.px; ep.py = lp.py; ep.pz = lp.pz;
    ep.triCount = ctx->d_tri_count; ep.triTable = ctx->d_tri_table;
    dcsg_launch_adapt_count(ep, stream); ++g_launches;
    dcsg_mesher_params sp;                      // the tile scan only reads the tile arrays and counts
    memset(&sp, 0, sizeof(sp));
    sp.tileCells = ep.tileCells; sp.tileTris = ep.tileTris; sp.tileVerts = nullptr;
    sp.numCellWords = ep.numTiles * DCSG_TILE_WORDS; sp.numVertWords = 0;       // = ep.numTiles tiles of sums
    sp.totals = d_counts;
    dcsg_launch_scan_tiles(sp, stream); ++g_launches;
    CUDA_TRY(ctx, cudaGetLastError());
    // multi-GPU: the ranks' counts (the per-level ones included) are all-gathered next to this read-back
    if (ctx->exchange_pre) { rc = ctx->exchange_pre(ctx, ctx->exchange_user, d_counts, stream); if (rc != DCSG_OK) return rc; }
    CUDA_TRY(ctx, ctx->pinned_small.reserve(32 * 4 + 64));
    uint32_t* totals = ctx->pinned_small.as<uint32_t>();
    uint64_t* normalEvals = reinterpret_cast<uint64_t*>(totals + 32);
    CUDA_TRY(ctx, cudaMemcpyAsync(totals, d_counts, 32 * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(normalEvals, counter, 8, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(stream));
    nCells = totals[0];
    const uint64_t preTris = totals[1];
    evals = (uint64_t)s.P * s.P * s.nzp + *normalEvals;
    st->levelTriangles.assign(16, 0);
    for (int lvl = 0; lvl < 16; lvl++) st->levelTriangles[lvl] = totals[16 + lvl];

    // soup with identity indices, so that the mesh keeps its indexed shape; retopologize writes a truly indexed mesh:
    // the 3*points - 2 triangles of a source triangle share its 3*points resampled points (k_retopo_points)
    const uint32_t points = cfg->retopologize ? (1u << (s.L - minLevel)) : 1u;
    nTris = points >= 2 ? preTris * (3ull * points - 2ull) : preTris;
    for (uint64_t& t : st->levelTriangles) t *= points >= 2 ? (3ull * points - 2ull) : 1ull;       // retopologize multiplies every triangle
    nVerts = points >= 2 ? preTris * 3ull * points : nTris * 3;
    if (nTris * 3 > 0xffffffffull) return fail(ctx, DCSG_ERR_INVALID, "soup exceeds 32-bit vertex indices");       // the files are soup (happly.h:1654-1662)
    CUDA_TRY(ctx, st->vertices.reserve(std::max<uint64_t>(nVerts, 1) * 12));
    CUDA_TRY(ctx, st->triangles.reserve(std::max<uint64_t>(nTris, 1) * 12));
    CUDA_TRY(ctx, st->cell_ids.reserve(std::max<uint64_t>(nCells, 1) * 8));
    CUDA_TRY(ctx, st->cell_masks.reserve(std::max<uint64_t>(nCells, 1)));
    ep.cellIds = st->cell_ids.as<uint64_t>();
    ep.cellMasks = st->cell_masks.as<uint8_t>();
    if (points >= 2) {
        CUDA_TRY(ctx, ctx->fmt.reserve(std::max<uint64_t>(preTris, 1) * 36));
        ep.soup = ctx->fmt.as<float>();
        dcsg_launch_adapt_emit(ep, stream); ++g_launches;
        dcsg_launch_retopo_expand(ep.soup, preTris, points, st->vertices.as<float>(), st->triangles.as<uint32_t>(), stream);
        g_launches += 2;
    } else {
        ep.soup = st->vertices.as<float>();
        dcsg_launch_adapt_emit(ep, stream); ++g_launches;
        dcsg_launch_iota(st->triangles.as<uint32_t>(), nVerts, stream); ++g_launches;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[3], stream));
    return DCSG_OK;
}

}  // namespace dcsg_host

namespace dcsg_host {
int launch_project(dcsg_ctx* ctx, float* d_vertices, unsigned long long count, int gd_steps, float* d_normals, cudaStream_t stream, int slot,
                   float* gather_vertices, float* gather_normals, unsigned long long gather_count, unsigned long long list_offset) {
    if (!count) return DCSG_OK;
    const int smCount = ctx->sm_count;
    // 16 slots of {vertex cursor, entries appended to the exact phase's list, entries claimed from it, -} (launches queued back
    // to back on one stream -- the file pipeline's chunks -- do not share) | 2 statistics counters (never reset here:
    // dcsg_project_stats reads and clears them)
    struct Args {               // dcsg_project_args of scene_kernels.cuh
        float* verts; unsigned long long n; int steps; float* normals; unsigned long long* cursor; float* gatherVerts; float* gatherNormals;
        unsigned long long gatherCount; unsigned long long* deferred; int detectCycles;
    } args;
    const bool fresh = ctx->project_cursor.ptr == nullptr;
    CUDA_TRY(ctx, ctx->project_cursor.reserve((16 * 4 + 2) * sizeof(unsigned long long)));
    if (fresh) CUDA_TRY(ctx, cudaMemsetAsync(ctx->project_cursor.ptr, 0, (16 * 4 + 2) * sizeof(unsigned long long), stream));
    // the list of the exact phase: one slot per vertex of the launch, zero = not written yet
    {
        const void* before = ctx->project_list.ptr;
        CUDA_TRY(ctx, ctx->project_list.reserve((size_t)(list_offset + count) * 8));
        (void)before;
    }
    unsigned long long* cursor = ctx->project_cursor.as<unsigned long long>() + (size_t)(slot & 15) * 4;
    unsigned long long* stats = ctx->project_cursor.as<unsigned long long>() + 64;
    unsigned long long* list = ctx->project_list.as<unsigned long long>() + list_offset;
    CUDA_TRY(ctx, cudaMemsetAsync(cursor, 0, 4 * sizeof(unsigned long long), stream));
    CUDA_TRY(ctx, cudaMemsetAsync(list, 0, (size_t)count * 8, stream));
    // persistent warps: no more blocks than can be resident (dcsg_build asks the occupancy calculator), no more than there
    // are batches of work
    const unsigned long long blocks = std::min<unsigned long long>((count + 255) / 256, (unsigned long long)smCount * ctx->project_blocks_per_sm);
    // cycle detection needs the update to be a pure function of the position: not with designs that keep mutable
    // program-scope state between evaluations; DCSG_PROJECT_ALL_STEPS=1 switches it off (measurement)
    static const bool allSteps = [] { const char* e = getenv("DCSG_PROJECT_ALL_STEPS"); return e && atoi(e) != 0; }();
    args.verts = d_vertices; args.n = count; args.steps = gd_steps; args.normals = d_normals; args.cursor = cursor;
    args.gatherVerts = gather_vertices; args.gatherNormals = gather_normals; args.gatherCount = gather_count;
    args.deferred = list;
    args.detectCycles = (ctx->scene.private_words == 0 && !allSteps) ? 1 : 0;
    void* kargs[] = {&args, &stats};
    CUDA_TRY(ctx, launch(ctx->k_project, dim3((unsigned)blocks), dim3(256), kargs, stream, ctx->scene.private_words));
    return DCSG_OK;
}
}  // namespace dcsg_host

extern "C" {

int dcsg_sample_lattice(dcsg_ctx* ctx, const float* box6, int grid_level, int z_begin, int z_end, float* out_host) {
    if (!ctx || !box6) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    LatticeSetup s;
    const int N = 1 << grid_level;
    if (z_begin == 0 && z_end == 0) z_end = N + 1;
    if (z_begin < 0 || z_end > N + 1 || z_begin >= z_end) return fail(ctx, DCSG_ERR_INVALID, "bad plane range");
    // planes [z_begin, z_end) = cell layers [z_begin, z_end-1) plus the closing plane
    int rc;
    if (z_end - z_begin >= 2) {
        rc = setup_lattice(ctx, box6, grid_level, z_begin, z_end - 1, s, false);
    } else {            // a single plane: run a one-layer slab and keep its first (or last) plane
        const bool top = (z_begin == N);
        rc = setup_lattice(ctx, box6, grid_level, top ? N - 1 : z_begin, top ? N : z_begin + 1, s, false);
    }
    if (rc != DCSG_OK) return rc;
    const size_t PB = (size_t)s.P * s.P;
    CUDA_TRY(ctx, ctx->lattice_values.reserve(PB * s.nzp * 4));
    dcsg_lattice_params lp;
    rc = run_lattice(ctx, s, ctx->lattice_values.as<float>(), lp);
    if (rc != DCSG_OK) return rc;
    if (out_host) {
        const size_t skip = (size_t)(z_begin - s.z0) * PB;
        CUDA_TRY(ctx, cudaMemcpyAsync(out_host, ctx->lattice_values.as<float>() + skip, PB * (size_t)(z_end - z_begin) * 4,
                                      cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DCSG_OK;
}

const float* dcsg_lattice_device_ptr(const dcsg_ctx* ctx) { return ctx ? ctx->lattice_values.as<float>() : nullptr; }

int dcsg_project(dcsg_ctx* ctx, dcsg_mesh* mesh, int gd_steps, int want_normals) {
    if (!ctx || !mesh || !mesh->reserved) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    MeshStorage* st = (MeshStorage*)mesh->reserved;
    const uint64_t nVerts = mesh->num_vertices;
    float* d_normals = nullptr;
    if (want_normals) {
        CUDA_TRY(ctx, st->normals.reserve(std::max<uint64_t>(nVerts, 1) * 12));
        d_normals = st->normals.as<float>();
    }
    mesh->d_normals = d_normals;
    if (nVerts && (gd_steps > 0 || d_normals)) {
        if (int rc = launch_project(ctx, mesh->d_vertices, nVerts, gd_steps, d_normals, ctx->stream)) return rc;
    }
    return DCSG_OK;         // asynchronous: ordered on the context's stream
}

int dcsg_project_stats(dcsg_ctx* ctx, uint64_t* tap_rounds, uint64_t* exact_rounds) {
    if (!ctx) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    unsigned long long v[2] = {0, 0};
    if (ctx->project_cursor.ptr) {
        unsigned long long* stats = ctx->project_cursor.as<unsigned long long>() + 64;
        CUDA_TRY(ctx, cudaMemcpyAsync(v, stats, sizeof(v), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaMemsetAsync(stats, 0, sizeof(v), ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (tap_rounds) *tap_rounds = v[0];
    if (exact_rounds) *exact_rounds = v[1];
    return DCSG_OK;
}

void dcsg_mesh_free(dcsg_ctx* ctx, dcsg_mesh* mesh) {
    if (!mesh) return;
    if (ctx) cudaSetDevice(ctx->device);
    MeshStorage* st = (MeshStorage*)mesh->reserved;
    if (st) {
        for (DevBuf* b : {&st->vertices, &st->normals, &st->keys, &st->triangles, &st->cell_ids, &st->cell_masks}) b->release();
        st->host.release();
        delete st;
    }
    memset(mesh, 0, sizeof(*mesh));
}

int dcsg_extract(dcsg_ctx* ctx, const dcsg_extract_cfg* cfg, dcsg_mesh* out) {
    if (!ctx || !cfg || !out) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    if (!ctx->built) return fail(ctx, DCSG_ERR_NO_SCENE, "no scene built");
    const bool uniform = cfg->min_level >= cfg->grid_level && cfg->max_level == cfg->grid_level;
    if (cfg->max_level > cfg->grid_level || cfg->max_level < 0 || cfg->min_level < 0)
        return fail(ctx, DCSG_ERR_INVALID, "octree levels must satisfy 0 <= min, 0 <= max <= grid level");
    if (!uniform && cfg->no_cull) return fail(ctx, DCSG_ERR_UNSUPPORTED, "no_cull applies to the uniform configuration only");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    // a mesh object can be reused across calls: its buffers only grow
    MeshStorage* st = (MeshStorage*)out->reserved;
    if (!st) { memset(out, 0, sizeof(*out)); st = new MeshStorage(); out->reserved = st; }
    out->owned_vertices = out->halo_vertices = 0;

    // A z-slab is processed with one extra cell layer below and above it (where the lattice goes on): the vertices on its
    // first sample plane then see all four cells around their edges, and those on the NEXT slab's first plane can be
    // numbered here exactly as that slab will number them (mesher.h "Ownership").  Cells are emitted for the slab's own
    // layers only, so slabs concatenate to the whole mesh without a weld.
    const int Ncells = 1 << cfg->grid_level;
    int ownZ0 = cfg->slab_z0, ownZ1 = cfg->slab_z1;
    if (ownZ0 == 0 && ownZ1 == 0) ownZ1 = Ncells;
    const bool slabOk = ownZ0 >= 0 && ownZ1 <= Ncells && ownZ0 < ownZ1;
    const int procZ0 = uniform && slabOk && ownZ0 > 0 ? ownZ0 - 1 : ownZ0;
    const int procZ1 = uniform && slabOk && ownZ1 < Ncells ? ownZ1 + 1 : ownZ1;
    LatticeSetup s;
    int rc = setup_lattice(ctx, cfg->box, cfg->grid_level, procZ0, procZ1, s, true);
    if (rc != DCSG_OK) return rc;
    cudaStream_t stream = ctx->stream;
    if (ctx->aux_pending) {         // the previous extraction's clean-up pass reads its work lists and zeroes its bitmaps
        CUDA_TRY(ctx, cudaStreamWaitEvent(stream, ctx->aux_done, 0));
        ctx->aux_pending = false;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], stream));
    static const bool traceOn = [] { const char* e = getenv("DCSG_TRACE"); return e && atoi(e) != 0; }();
    double traceT[6] = {now_ms(), 0, 0, 0, 0, 0};

    uint64_t nCells = 0, nTris = 0, nVerts = 0, nHalo = 0;
    uint64_t evals = 0;
    dcsg_mesher_params mp;
    memset(&mp, 0, sizeof(mp));
    st->layerTriFirst.clear();
    st->planeVertFirst.clear();
    st->levelTriangles.clear();
    st->runs.clear();
    st->cellUnit = 0;
    st->oriented = false;
    if (!uniform) {
        ctx->sparse_clean = false;              // the dense lattice pass writes the bitmaps the sparse pass keeps all-zero
        rc = extract_adaptive(ctx, cfg, s, st, nVerts, nTris, nCells, evals);
        if (rc != DCSG_OK) return rc;
        if (ctx->exchange_post) { rc = ctx->exchange_post(ctx, ctx->exchange_user, mp); if (rc != DCSG_OK) return rc; }
        mp.vertices = st->vertices.as<float>();
        mp.vertexKeys = nullptr;                // soup vertices have no lattice key
        mp.triangles = st->triangles.as<uint32_t>();
        mp.cellIds = st->cell_ids.as<uint64_t>();
        mp.cellMasks = st->cell_masks.as<uint8_t>();
    } else {
    // ---- stage 1: lattice -> sign / cull bitmaps ------------------------------------------------
    dcsg_lattice_params lp;
    dcsg_leaf_params lf;
    SparseLists sl;
    memset(&sl, 0, sizeof(sl));
    uint64_t* d_evals = nullptr;
    const bool sparse = !cfg->dense && !cfg->no_cull;
    if (!sparse) ctx->sparse_clean = false;
    rc = sparse ? run_descent(ctx, s, lf, &d_evals, sl) : run_lattice(ctx, s, nullptr, lp);
    if (rc != DCSG_OK) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], stream));

    // ---- stage 2: classify, edges, device-wide scan -----------------------------------------------
    mp.g.N = s.N; mp.g.P = s.P; mp.g.L = s.L; mp.g.z0 = s.z0; mp.g.nzc = s.nzc; mp.g.nzp = s.nzp;
    mp.g.pitch = s.pitch;
    mp.g.planeWords = s.planeWords;
    mp.g.PB = (uint32_t)s.pitch * (uint32_t)s.P;
    mp.ownCell0 = ownZ0 - s.z0; mp.ownCell1 = ownZ1 - s.z0;
    mp.ownVert0 = ownZ0 - s.z0;
    mp.haloVert = ownZ1 < Ncells ? 1 : 0;
    mp.ownVert1 = ownZ1 - s.z0 + (mp.haloVert ? 0 : 1);       // the last slab also owns the lattice's closing plane
    if (sparse) {
        mp.sign = lf.sign;
        mp.leafAlive = lf.leafAlive;
        mp.cellList = sl.cellList; mp.cellCount = sl.counts + 1;
        mp.vertList = sl.vertList; mp.vertCount = sl.counts + 3;
        mp.aliveMask = sl.aliveMask;
        mp.aliveMask31 = sl.aliveMask31;
    } else {
        mp.sign = lp.sign;
        mp.leaf = lp.leaf;
        mp.coarse.cfail = lp.cfail;
        mp.coarse.nodeBits = lp.coarse;
        for (int l = 0; l < 16; l++) mp.coarse.off[l] = lp.coarseOff[l];
        mp.coarse.thickMask = s.thickMask;
    }
    mp.noCull = cfg->no_cull ? 1u : 0u;
    mp.numCellWords = s.planeWords * (uint32_t)s.nzc;
    mp.numVertWords = s.planeWords * (uint32_t)s.nzp;
    const uint32_t cellTiles = (mp.numCellWords + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    const uint32_t vertTiles = (mp.numVertWords + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    const size_t padWords = (size_t)s.planeWords + 64;
    CUDA_TRY(ctx, ctx->alive.reserve(((size_t)mp.numVertWords + padWords) * 4));
    CUDA_TRY(ctx, ctx->vinfo.reserve((size_t)mp.numVertWords * 16 + 64));
    // per-tile sums | counts block (32 words: totals, halo count; the all-gather of a sharded export reads it whole) | triangles
    // per cell layer | vertices per sample plane
    CUDA_TRY(ctx, ctx->tiles.reserve(((size_t)cellTiles * 2 + vertTiles + 40 + (size_t)s.nzc + s.nzp) * 4));
    if (!sparse) CUDA_TRY(ctx, cudaMemsetAsync(ctx->alive.as<uint32_t>() + mp.numCellWords, 0, padWords * 4, stream));
    mp.alive = ctx->alive.as<uint32_t>();
    mp.vinfo = ctx->vinfo.as<uint4>();
    mp.tileCells = ctx->tiles.as<uint32_t>();
    mp.tileTris = mp.tileCells + cellTiles;
    mp.tileVerts = mp.tileTris + cellTiles;
    mp.totals = mp.tileVerts + vertTiles;
    mp.layerTris = mp.totals + 32;
    mp.planeVerts = mp.layerTris + s.nzc;
    mp.px = ctx->axes.as<float>(); mp.py = mp.px + s.pitch; mp.pz = mp.px + 2 * s.pitch;
    mp.triCount = ctx->d_tri_count;
    mp.triTable = ctx->d_tri_table;
    CUDA_TRY(ctx, cudaMemsetAsync(mp.totals, 0, (size_t)(32 + s.nzc + s.nzp) * 4, stream));
    const int ctas = ctx->sm_count * 8;
    dcsg_launch_classify(mp, ctas, stream); ++g_launches;
    if (sparse) {               // vertex-owner words = the words next to an alive cell word
        dcsg_worklist_params wl;
        memset(&wl, 0, sizeof(wl));
        wl.mask = sl.aliveMask; wl.mask31 = sl.aliveMask31; wl.numBits = sl.numBits; wl.rowWords = sl.rowWords; wl.planeWords = s.planeWords;
        wl.mode = 1; wl.listA = nullptr; wl.listB = sl.vertList; wl.counts = sl.counts + 2; wl.scratch = sl.scratch;   // counts[3] <- len(listB)
        dcsg_launch_worklists(wl, stream); g_launches += 2;
    }
    dcsg_launch_edges(mp, ctas, stream); ++g_launches;
    dcsg_launch_scan_tiles(mp, stream); ++g_launches;
    CUDA_TRY(ctx, cudaGetLastError());
    evals = (uint64_t)s.P * s.P * s.nzp;
    // the one host round trip: output sizes (and the per-layer counts the chunked file pipeline cuts the mesh by)
    CUDA_TRY(ctx, ctx->pinned_small.reserve((size_t)(32 + s.nzc + s.nzp) * 4 + 64));
    uint32_t* h_totals = ctx->pinned_small.as<uint32_t>();
    uint64_t* h_evals = reinterpret_cast<uint64_t*>(h_totals + ((32 + s.nzc + s.nzp + 1) & ~1));
    // totals[3] = copies of the next slab's first vertices (the halo plane's count)
    if (mp.haloVert) CUDA_TRY(ctx, cudaMemcpyAsync(mp.totals + 3, mp.planeVerts + mp.ownVert1, 4, cudaMemcpyDeviceToDevice, stream));
    if (ctx->exchange_pre) { rc = ctx->exchange_pre(ctx, ctx->exchange_user, mp.totals, stream); if (rc != DCSG_OK) return rc; }
    CUDA_TRY(ctx, cudaMemcpyAsync(h_totals, mp.totals, (size_t)(32 + s.nzc + s.nzp) * 4, cudaMemcpyDeviceToHost, stream));
    if (sparse) CUDA_TRY(ctx, cudaMemcpyAsync(h_evals, d_evals, 8, cudaMemcpyDeviceToHost, stream));
    // the lengths of the cell and vertex lists ride along: the emitters below get one CTA per tile that exists
    uint32_t* h_lists = reinterpret_cast<uint32_t*>(h_evals + 1);
    if (sparse) CUDA_TRY(ctx, cudaMemcpyAsync(h_lists, sl.counts, 16, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], stream));
    traceT[1] = now_ms();
    CUDA_TRY(ctx, cudaStreamSynchronize(stream));
    traceT[2] = now_ms();
    if (sparse) evals = *h_evals;
    nCells = h_totals[0]; nTris = h_totals[1]; nVerts = h_totals[2];
    {
        const uint32_t* layerTris = h_totals + 32;
        const uint32_t* planeVerts = layerTris + s.nzc;
        nHalo = mp.haloVert ? planeVerts[mp.ownVert1] : 0;
        // prefixes over the slab's own layers / planes (own layer i = global layer ownZ0 + i); the halo plane closes the list
        st->layerTriFirst.assign(1, 0);
        for (int zl = mp.ownCell0; zl < mp.ownCell1; zl++) st->layerTriFirst.push_back(st->layerTriFirst.back() + layerTris[zl]);
        st->planeVertFirst.assign(1, 0);
        for (int zl = mp.ownVert0; zl < mp.ownVert1 + mp.haloVert; zl++) st->planeVertFirst.push_back(st->planeVertFirst.back() + planeVerts[zl]);
        if (st->layerTriFirst.back() != nTris || st->planeVertFirst.back() != nVerts)
            return fail(ctx, DCSG_ERR_CUDA, "internal: per-layer counts disagree with the totals");
    }

    // ---- stage 3: emit vertices and triangles --------------------------------------------------------
    CUDA_TRY(ctx, st->vertices.reserve(std::max<uint64_t>(nVerts, 1) * 12));
    CUDA_TRY(ctx, st->keys.reserve(std::max<uint64_t>(nVerts, 1) * 8));
    CUDA_TRY(ctx, st->triangles.reserve(std::max<uint64_t>(nTris, 1) * 12));
    CUDA_TRY(ctx, st->cell_ids.reserve(std::max<uint64_t>(nCells, 1) * 8));
    CUDA_TRY(ctx, st->cell_masks.reserve(std::max<uint64_t>(nCells, 1)));
    mp.vertices = st->vertices.as<float>();
    mp.vertexKeys = st->keys.as<uint64_t>();
    mp.triangles = st->triangles.as<uint32_t>();
    mp.cellIds = st->cell_ids.as<uint64_t>();
    mp.cellMasks = st->cell_masks.as<uint8_t>();
    if (ctx->exchange_post) {   // multi-GPU (host_comm.cu): offsets from the gathered counts, emitters pointed at the gathering rank's arrays
        rc = ctx->exchange_post(ctx, ctx->exchange_user, mp);
        if (rc != DCSG_OK) return rc;
    }
    // A resident CTA holds about two tiles' worth of threads at 1024^3, so a persistent grid ends with the few CTAs that got
    // a third tile running alone (ncu: sm__cycles_active max 1.46 x avg).  The list lengths are known by now: one CTA per
    // tile, and the hardware hands them out as CTAs retire.
    const uint32_t cellTilesNow = sparse ? (h_lists[1] + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS : 0u;
    const uint32_t vertTilesNow = sparse ? (h_lists[3] + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS : 0u;
    dcsg_launch_emit_vertices(mp, sparse ? (int)std::max(vertTilesNow, 1u) : ctas, stream); ++g_launches;
    dcsg_launch_emit_triangles(mp, sparse ? (int)std::max(cellTilesNow, 1u) : ctas, stream); ++g_launches;
    if (sparse) {
        dcsg_cleanup_params cp;
        memset(&cp, 0, sizeof(cp));
        cp.cellList = sl.cellList; cp.cellCount = sl.counts + 1;
        cp.leafAlive = ctx->leaf.as<uint32_t>(); cp.alive = ctx->alive.as<uint32_t>();
        // on the side stream: nothing on `stream` needs it before the next extraction (which waits for it), so it runs under
        // the projection instead of in front of it
        CUDA_TRY(ctx, cudaEventRecord(ctx->aux_ready, stream));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->aux_ready, 0));
        dcsg_launch_cleanup(cp, ctx->sm_count * 2, ctx->aux_stream); ++g_launches;
        CUDA_TRY(ctx, cudaEventRecord(ctx->aux_done, ctx->aux_stream));
        ctx->aux_pending = true;
        ctx->sparse_clean = true;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[3], stream));
    }   // uniform

    // ---- stage 4: projection (gradient descent) + optional normals -------------------------------------
    if (cfg->want_normals) CUDA_TRY(ctx, st->normals.reserve(std::max<uint64_t>(nVerts, 1) * 12));
    float* d_normals = cfg->want_normals ? st->normals.as<float>() : nullptr;
    if (!cfg->defer_projection && nVerts && (cfg->gd_steps > 0 || d_normals)) {
        if (int rc = launch_project(ctx, mp.vertices, nVerts, cfg->gd_steps, d_normals, stream)) return rc;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], stream));

    out->num_vertices = nVerts;
    out->num_triangles = nTris;
    out->num_cells = nCells;
    out->d_vertices = mp.vertices;
    out->d_normals = d_normals;
    out->d_vertex_keys = mp.vertexKeys;
    out->d_triangles = mp.triangles;
    out->d_cell_ids = mp.cellIds;
    out->d_cell_masks = mp.cellMasks;
    out->lattice_samples = evals;
    st->uniform = uniform;
    if (!uniform) {
        const uint64_t points = cfg->retopologize ? (1ull << (cfg->grid_level - std::min(cfg->min_level, cfg->max_level))) : 1ull;
        st->unitTriangles = points >= 2 ? 3 * points - 2 : 1;
        st->unitVertices = points >= 2 ? 3 * points : 3;
    }
    st->cellUnit = uniform ? 1 : st->unitTriangles;
    out->owned_vertices = nVerts - nHalo;
    out->halo_vertices = nHalo;
    out->h_vertices = out->h_normals = nullptr;
    out->h_vertex_keys = nullptr; out->h_triangles = nullptr; out->h_cell_ids = nullptr; out->h_cell_masks = nullptr;

    // ---- stage 5: optional copy to pinned host memory --------------------------------------------------
    if (cfg->copy_to_host) {
        const size_t bV = nVerts * 12, bN = d_normals ? nVerts * 12 : 0, bK = mp.vertexKeys ? nVerts * 8 : 0, bT = nTris * 12, bC = nCells * 8, bM = nCells;
        auto align = [](size_t v) { return (v + 63) & ~(size_t)63; };
        const size_t total = align(bV) + align(bN) + align(bK) + align(bT) + align(bC) + align(bM) + 64;
        CUDA_TRY(ctx, st->host.reserve(total));
        uint8_t* base = st->host.as<uint8_t>();
        size_t o = 0;
        out->h_vertices = (float*)(base + o); o += align(bV);
        if (d_normals) { out->h_normals = (float*)(base + o); o += align(bN); }
        if (bK) { out->h_vertex_keys = (uint64_t*)(base + o); o += align(bK); }
        out->h_triangles = (uint32_t*)(base + o); o += align(bT);
        out->h_cell_ids = (uint64_t*)(base + o); o += align(bC);
        out->h_cell_masks = base + o;
        if (bV) CUDA_TRY(ctx, cudaMemcpyAsync(out->h_vertices, out->d_vertices, bV, cudaMemcpyDeviceToHost, stream));
        if (bN) CUDA_TRY(ctx, cudaMemcpyAsync(out->h_normals, out->d_normals, bN, cudaMemcpyDeviceToHost, stream));
        if (bK) CUDA_TRY(ctx, cudaMemcpyAsync(out->h_vertex_keys, out->d_vertex_keys, bK, cudaMemcpyDeviceToHost, stream));
        if (bT) CUDA_TRY(ctx, cudaMemcpyAsync(out->h_triangles, out->d_triangles, bT, cudaMemcpyDeviceToHost, stream));
        if (bC) CUDA_TRY(ctx, cudaMemcpyAsync(out->h_cell_ids, out->d_cell_ids, bC, cudaMemcpyDeviceToHost, stream));
        if (bM) CUDA_TRY(ctx, cudaMemcpyAsync(out->h_cell_masks, out->d_cell_masks, bM, cudaMemcpyDeviceToHost, stream));
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[5], stream));
    traceT[3] = now_ms();
    if (ctx->skip_final_sync) return DCSG_OK;       // dcsg_extract_sharded queues the projection right behind and reads the stage times later
    CUDA_TRY(ctx, cudaStreamSynchronize(stream));
    traceT[4] = now_ms();
    for (int i = 0; i < DCSG_STAGE_COUNT; i++) cudaEventElapsedTime(&out->stage_ms[i], ctx->ev[i], ctx->ev[i + 1]);
    if (traceOn && uniform && ctx->device == 0)
        fprintf(stderr, "[dcsg trace] extract: queue-to-sizes %.3f wait-sizes %.3f queue-emit %.3f wait-end %.3f | device: lattice %.3f classify %.3f emit %.3f\n",
                traceT[1] - traceT[0], traceT[2] - traceT[1], traceT[3] - traceT[2], traceT[4] - traceT[3], out->stage_ms[0], out->stage_ms[1], out->stage_ms[2]);
    return DCSG_OK;
}

int dcsg_mesh_soup(dcsg_ctx* ctx, const dcsg_mesh* mesh, float* out_host) {
    if (!ctx || !mesh || !out_host) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t n = mesh->num_triangles;
    if (!n) return DCSG_OK;
    CUDA_TRY(ctx, ctx->fmt.reserve(n * 36));
    dcsg_launch_expand_soup(mesh->d_vertices, mesh->d_triangles, n, ctx->fmt.as<float>(), ctx->stream); ++g_launches;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(out_host, ctx->fmt.ptr, n * 36, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DCSG_OK;
}

int dcsg_mesh_orient(dcsg_ctx* ctx, dcsg_mesh* mesh) {
    if (!ctx || !mesh) return DCSG_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->lock);
    return orient_locked(ctx, mesh);
}

}  // extern "C"

// The winding of a triangle is a function of its cell's corner mask and its slot in the table row (tools/gen_mc_table.py), so
// orienting a mesh is one pass over its cells: no geometry, the same on every schedule, slab and octree level.
int dcsg_host::orient_locked(dcsg_ctx* ctx, dcsg_mesh* mesh) {
    MeshStorage* st = (MeshStorage*)mesh->reserved;
    if (!st || !st->cellUnit || (mesh->num_cells && !mesh->d_cell_masks))
        return fail(ctx, DCSG_ERR_INVALID, "dcsg_mesh_orient needs a mesh from dcsg_extract: its cells' corner masks decide the winding");
    if (st->oriented) return DCSG_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t n = mesh->num_cells;
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t scratch = align(dcsg_orient_scratch_bytes(n));
    CUDA_TRY(ctx, ctx->orient.reserve(scratch + 256));
    uint8_t* w = ctx->orient.as<uint8_t>();
    dcsg_orient_params p;
    p.cellMasks = mesh->d_cell_masks;
    p.numCells = n;
    p.triCount = ctx->d_tri_count;
    p.triFlip = ctx->d_tri_flip;
    p.unit = (uint32_t)st->cellUnit;
    p.triangles = mesh->d_triangles;
    p.numTriangles = mesh->num_triangles;
    p.scratch = w;
    p.total = reinterpret_cast<uint32_t*>(w + scratch);
    cudaStream_t s = ctx->stream;
    CUDA_TRY(ctx, dcsg_launch_orient(p, s));
    g_launches += 2;                // the count and the swap; cub's scan passes are not counted
    CUDA_TRY(ctx, ctx->pinned_small.reserve(64));
    uint32_t* h_total = ctx->pinned_small.as<uint32_t>();
    CUDA_TRY(ctx, cudaMemcpyAsync(h_total, p.total, 4, cudaMemcpyDeviceToHost, s));
    if (mesh->h_triangles && mesh->num_triangles)
        CUDA_TRY(ctx, cudaMemcpyAsync(mesh->h_triangles, mesh->d_triangles, mesh->num_triangles * 12, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    if (*h_total != mesh->num_triangles)
        return fail(ctx, DCSG_ERR_INVALID, format("dcsg_mesh_orient: the cells account for %u triangles, the mesh holds %llu", *h_total,
                                                  (unsigned long long)mesh->num_triangles));
    st->oriented = true;
    return DCSG_OK;
}

