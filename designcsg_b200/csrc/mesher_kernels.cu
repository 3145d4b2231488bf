// mesher_kernels.cu -- the bit-parallel mesher: classify / compact / emit (sm_100a, ahead of time).
//
// Replaces the reference's CPU octree walk (master/cms/main/Headers/mesh.hpp:82-380): per node it
// fetched a centre sample and 8 corner samples through a mutex-guarded block cache, built the 8-bit
// corner mask, and pushed lookup-table triangles on edge midpoints into a vector under a lock.
// Here the lattice kernel has already reduced every sample to a sign bit and a cull bit, and the
// whole extraction is word-parallel integer work on those bitmaps:
//
//   classify   1 thread / 4 words (128 cells): 8 funnel-shifted sign words -> active word, minus culled cells
//              -> alive bitmap; the tile's surface cells are gathered in shared memory and counted one per
//              thread (triangle counts from the 256-entry table, ancestor culls on the dense path); per-tile sums
//   edges      1 thread / 32 lattice points : sign XOR neighbours AND any-adjacent-alive -> the three
//              owned-edge words (= mesh vertices, deduplicated by construction); per-tile sums
//   scan       one CTA: exclusive prefix over the per-tile sums (device-wide offsets) + totals
//   vertices   per tile: block scan of per-word counts -> first vertex id of every word, vertex
//              keys and edge-midpoint positions written in key order
//   triangles  per tile: surface cells gathered in shared memory (canonical order), one cell per thread ->
//              compacted active-cell records and indexed triangles (cell index, then table order)
//
// All of it is HBM/L2-bound integer traffic over bitmaps of (N+1)^3/8 bytes; see DESIGN.md for the
// algorithmic byte counts.  The word-level logic lives in mesher_bits.cuh and is unit-tested on the
// CPU against the oracle (tests/test_mesher_bits.py); this file adds the CTA-level scans and I/O.
#include "mesher.h"

#include <algorithm>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_reduce.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

namespace {

constexpr int kThreads = 256;
constexpr int kRounds = DCSG_TILE_WORDS / kThreads;     // list entries per thread and tile
constexpr uint32_t kPer = DCSG_TILE_WORDS / kThreads;
constexpr uint32_t kWorklistTile = 1024;                // mask words per CTA of the work-list kernels (4 per thread)

// exclusive scan of one value per thread across the CTA; returns the exclusive prefix, total in `total`
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T& total, T* smem /* kThreads/32 + 1 */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        T w = lane < kThreads / 32 ? smem[lane] : T(0);
        T winc = w;
#pragma unroll
        for (int d = 1; d < kThreads / 32; d <<= 1) {
            const T o = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += o;
        }
        if (lane < kThreads / 32) smem[lane] = winc - w;           // exclusive prefix of the warp sums
        if (lane == kThreads / 32 - 1) smem[kThreads / 32] = winc; // CTA total
    }
    __syncthreads();
    const T out = smem[warp] + inc - v;
    total = smem[kThreads / 32];
    __syncthreads();
    return out;
}

template <typename T>
__device__ __forceinline__ T block_sum(T v, T* smem) {
    T total;
    block_exclusive_scan(v, total, smem);
    return total;
}

__device__ __forceinline__ void word_to_plane(const dcsg_grid& g, uint32_t w, int& zl, uint32_t& wi) {
    zl = (int)(w / g.planeWords);
    wi = w - (uint32_t)zl * g.planeWords;
}

// ---------------------------------------------------------------------------------------------
// Work lists.  Every kernel below handles list entry i = bitmap word list[i] (or word i without a list); a CTA tile is
// DCSG_TILE_WORDS consecutive ENTRIES, so tiles are equally full however sparse the surface is, and a persistent grid
// loops over them (the list lengths only exist on the device).
__device__ __forceinline__ uint32_t list_count(const uint32_t* countPtr, uint32_t all) { return countPtr ? *countPtr : all; }
__device__ __forceinline__ uint32_t list_word(const uint32_t* list, uint32_t i) { return list ? list[i] : i; }

// Per-layer / per-plane counters.  The entries of a tile ascend, so a tile touches a handful of consecutive layers; all
// CTAs work on the same few layers at the same time, and adding every warp's count straight to the global counter
// serialises on a few addresses (measured: 0.2 ms of the classify kernel).  A CTA therefore collects its tile in shared
// memory -- kLayerSlots layers from the tile's first one -- and adds each slot once; layers beyond that go to global memory.
constexpr int kLayerSlots = 16;
struct LayerCounts {
    uint32_t slot[kLayerSlots];
    int first;
};
__device__ __forceinline__ void layer_counts_begin(LayerCounts& lc, int firstLayer) {
    if (threadIdx.x < kLayerSlots) lc.slot[threadIdx.x] = 0u;
    if (threadIdx.x == 0) lc.first = firstLayer;
    __syncthreads();
}
__device__ __forceinline__ void layer_counts_add(LayerCounts& lc, uint32_t* counters, int layer, uint32_t value) {
    if (!value) return;
    const int rel = layer - lc.first;
    if (rel >= 0 && rel < kLayerSlots) atomicAdd(&lc.slot[rel], value);
    else atomicAdd(&counters[layer], value);
}
__device__ __forceinline__ void layer_counts_end(LayerCounts& lc, uint32_t* counters) {
    __syncthreads();
    if (threadIdx.x < kLayerSlots && lc.slot[threadIdx.x]) atomicAdd(&counters[lc.first + (int)threadIdx.x], lc.slot[threadIdx.x]);
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// Classification.  Word-parallel part: thread t owns entries kPer*t .. kPer*t + kPer-1 of the tile and derives their surface cells
// from the eight funnel-shifted corner words (minus the leaf-level cull).  Per-cell part (triangle counts, and on the
// dense path the ancestor culls): the CTA gathers the tile's surface cells into shared memory and handles them one
// per thread, like k_emit_triangles below -- a lattice row holds too few of them to keep a warp busy.
constexpr uint32_t kCellChunk = 2048;       // cells gathered per pass; denser tiles take several passes

__device__ __forceinline__ uint32_t cell_mask_at(const dcsg_grid& g, const uint32_t* sign, int zl, uint32_t lp) {
    const uint32_t* lower = sign + (uint64_t)zl * g.planeWords;
    const uint32_t* upper = lower + g.planeWords;
    const uint32_t l0 = dcsg_plane_bits(lower, lp), l1 = dcsg_plane_bits(lower, (int64_t)lp + g.pitch);
    const uint32_t u0 = dcsg_plane_bits(upper, lp), u1 = dcsg_plane_bits(upper, (int64_t)lp + g.pitch);
    // corners 0:(0,0,1) 1:(1,0,1) 2:(1,0,0) 3:(0,0,0) 4:(0,1,1) 5:(1,1,1) 6:(1,1,0) 7:(0,1,0)
    return ((u0 & 1u) << 0) | (((u0 >> 1) & 1u) << 1) | (((l0 >> 1) & 1u) << 2) | ((l0 & 1u) << 3) |
           ((u1 & 1u) << 4) | (((u1 >> 1) & 1u) << 5) | (((l1 >> 1) & 1u) << 6) | ((l1 & 1u) << 7);
}

// cells [chunk, chunk + kCellChunk) of a tile into s_cell (entry inside the tile << 5 | bit), canonical order;
// thread t owns words[0..3] = tile entries 4t .. 4t+3, its first cell has index myFirst inside the tile
__device__ __forceinline__ void gather_cells(const uint32_t words[kPer], uint32_t myFirst, uint32_t mine, uint32_t chunk, uint16_t* s_cell,
                                             uint32_t window = kCellChunk) {
    if (myFirst < chunk + window && myFirst + mine > chunk) {
        uint32_t idx = myFirst;
#pragma unroll
        for (int k = 0; k < kPer; ++k)
            for (uint32_t bits = words[k]; bits; bits &= bits - 1, ++idx)
                if (idx >= chunk && idx < chunk + window) s_cell[idx - chunk] = (uint16_t)(((threadIdx.x * kPer + k) << 5) | (__ffs(bits) - 1));
    }
}

__global__ void __launch_bounds__(kThreads) k_classify(const dcsg_mesher_params p) {
    __shared__ unsigned long long smem64[kThreads / 32 + 1];
    __shared__ uint32_t smem32[kThreads / 32 + 1];
    __shared__ uint32_t s_alive[DCSG_TILE_WORDS];       // the tile's surface-cell words; ancestor culls clear bits here
    __shared__ uint32_t s_word[DCSG_TILE_WORDS];        // bitmap word of every entry of the tile
    __shared__ uint16_t s_cell[kCellChunk];
    __shared__ LayerCounts s_layers;
    const uint32_t count = list_count(p.cellCount, p.numCellWords);
    const uint32_t tiles = (count + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    const bool ancestors = !p.noCull && !p.leafAlive;     // dense path: the coarse levels' culls are applied here
    for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const uint32_t tileBase = tile * DCSG_TILE_WORDS;
        uint32_t words[kPer];
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const uint32_t e = tileBase + threadIdx.x * kPer + k;
            uint32_t alive = 0u, w = 0u;
            if (e < count) {
                w = list_word(p.cellList, e);
                int zl; uint32_t wi;
                word_to_plane(p.g, w, zl, wi);
                uint32_t uncut = 0xffffffffu;                 // cells the leaf-level cull leaves standing
                if (p.leafAlive) uncut = p.leafAlive[w];       // culls already applied
                else if (!p.noCull) uncut = ~p.leaf[w];
                if (uncut) {
                    uint32_t corner[8];
                    dcsg_corner_words(p.g, p.sign, zl, wi, corner);
                    alive = dcsg_active_word(p.g, wi, corner) & uncut;
                }
            }
            words[k] = alive;
            s_alive[threadIdx.x * kPer + k] = alive;
            s_word[threadIdx.x * kPer + k] = w;
            mine += dcsg_popc(alive);
        }
        uint32_t tileTotal;
        const uint32_t myFirst = block_exclusive_scan(mine, tileTotal, smem32);
        layer_counts_begin(s_layers, (int)(s_word[0] / p.g.planeWords));
        uint32_t tris = 0;
        for (uint32_t chunk = 0; chunk < tileTotal; chunk += kCellChunk) {
            gather_cells(words, myFirst, mine, chunk, s_cell);
            __syncthreads();
            const uint32_t inChunk = min(kCellChunk, tileTotal - chunk);
            for (uint32_t i = threadIdx.x; i < inChunk; i += kThreads) {
                {
                    const uint32_t code = s_cell[i];
                    int zl; uint32_t wi;
                    word_to_plane(p.g, s_word[code >> 5], zl, wi);
                    const uint32_t lp = wi * 32u + (code & 31u);
                    bool culled = false;
                    if (ancestors) {
                        const uint32_t y = lp / (uint32_t)p.g.pitch, x = lp - y * (uint32_t)p.g.pitch;
                        culled = dcsg_coarse_culled(p.g, p.coarse, x, y, (uint32_t)(p.g.z0 + zl));
                    }
                    if (culled) atomicAnd(&s_alive[code >> 5], ~(1u << (code & 31u)));
                    else if (zl >= p.ownCell0 && zl < p.ownCell1) {             // halo cells only lend their alive bit to the edges
                        const uint32_t n = __ldg(&p.triCount[cell_mask_at(p.g, p.sign, zl, lp)]);
                        tris += n;
                        layer_counts_add(s_layers, p.layerTris, zl, n);
                    }
                }
            }
            __syncthreads();
        }
        layer_counts_end(s_layers, p.layerTris);
        uint32_t cells = 0;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const uint32_t e = tileBase + threadIdx.x * kPer + k;
            if (e >= count) continue;
            const uint32_t alive = s_alive[threadIdx.x * kPer + k];
            const uint32_t w = s_word[threadIdx.x * kPer + k];
            p.alive[w] = alive;
            if (alive && p.aliveMask) {
                atomicOr(&p.aliveMask[w >> 5], 1u << (w & 31u));
                if (alive >> 31) atomicOr(&p.aliveMask31[w >> 5], 1u << (w & 31u));
            }
            const int zl = (int)(w / p.g.planeWords);
            if (zl >= p.ownCell0 && zl < p.ownCell1) cells += dcsg_popc(alive);
        }
        // low 32 bits cells, high 32 bits triangles: one reduction over the CTA
        const unsigned long long total = block_sum((unsigned long long)cells | ((unsigned long long)tris << 32), smem64);
        if (threadIdx.x == 0) {
            p.tileCells[tile] = (uint32_t)total;
            p.tileTris[tile] = (uint32_t)(total >> 32);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Owned edges = mesh vertices: one thread per entry of the vertex list (the words next to an alive cell word).  Planes
// below the slab's first own plane and above the halo plane get no vertices: their edges belong to other slabs.
__global__ void __launch_bounds__(kThreads) k_edges(const dcsg_mesher_params p) {
    __shared__ uint32_t smem[kThreads / 32 + 1];
    __shared__ LayerCounts s_planes;
    const uint32_t count = list_count(p.vertCount, p.numVertWords);
    const uint32_t tiles = (count + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    const int firstPlane = p.ownVert0, endPlane = p.ownVert1 + (p.haloVert ? 1 : 0);
    for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const uint32_t tileBase = tile * DCSG_TILE_WORDS;
        layer_counts_begin(s_planes, (int)(list_word(p.vertList, tileBase) / p.g.planeWords));
        uint32_t verts = 0;
#pragma unroll 1
        for (int r = 0; r < kRounds; ++r) {
            const uint32_t e = tileBase + r * kThreads + threadIdx.x;
            uint32_t cnt = 0;
            if (e < count) {
                const uint32_t w = list_word(p.vertList, e);
                int zl; uint32_t wi;
                word_to_plane(p.g, w, zl, wi);
                uint32_t ex = 0u, ey = 0u, ez = 0u;
                if (zl >= firstPlane && zl < endPlane) dcsg_edge_words(p.g, p.sign, p.alive, zl, wi, ex, ey, ez);
                p.vinfo[w] = make_uint4(ex, ey, ez, 0u);
                cnt = dcsg_popc(ex) + dcsg_popc(ey) + dcsg_popc(ez);
                layer_counts_add(s_planes, p.planeVerts, zl, cnt);
            }
            verts += cnt;
        }
        layer_counts_end(s_planes, p.planeVerts);
        const uint32_t total = block_sum(verts, smem);
        if (threadIdx.x == 0) p.tileVerts[tile] = total;
    }
}

// ---------------------------------------------------------------------------------------------
// device-wide offsets: exclusive prefix over the per-tile sums, in place.  One CTA of 1024 threads per array (three
// arrays, three CTAs): every thread sums a contiguous run of tiles, the 1024 partial sums are scanned once, and the run is
// written back -- two block barriers per array.
__global__ void __launch_bounds__(1024) k_scan_tiles(const dcsg_mesher_params p) {
    __shared__ uint32_t warpSums[33];
    const int a = blockIdx.x;
    uint32_t* const array = a == 0 ? p.tileCells : (a == 1 ? p.tileTris : p.tileVerts);
    const uint32_t entries = a == 2 ? list_count(p.vertCount, p.numVertWords) : list_count(p.cellCount, p.numCellWords);
    const uint32_t count = (entries + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t per = (count + 1023u) / 1024u;
    const uint32_t begin = min(count, threadIdx.x * per), end = min(count, begin + per);
    uint32_t sum = 0;
    if (array) for (uint32_t i = begin; i < end; ++i) sum += array[i];
    uint32_t inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) warpSums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t ws = warpSums[lane];
        uint32_t winc = ws;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += o;
        }
        warpSums[lane] = winc - ws;
        if (lane == 31) warpSums[32] = winc;
    }
    __syncthreads();
    uint32_t running = warpSums[warp] + inc - sum;
    if (array) for (uint32_t i = begin; i < end; ++i) {
        const uint32_t v = array[i];
        array[i] = running;
        running += v;
    }
    if (threadIdx.x == 0) p.totals[a] = warpSums[32];
}

// ---------------------------------------------------------------------------------------------
// Vertices: thread t owns entries 4t .. 4t+3 of the tile, so one block scan numbers the tile's vertices in key order
// (phase A: first id of every word into vinfo, the vertices' sources into shared memory); then one thread per VERTEX
// computes the edge midpoint and the key and stores them to consecutive addresses (phase B).
constexpr uint32_t kVertChunk = 2048;

__global__ void __launch_bounds__(kThreads) k_emit_vertices(const dcsg_mesher_params p) {
    __shared__ uint32_t smem[kThreads / 32 + 1];
    __shared__ uint32_t s_vword[DCSG_TILE_WORDS];
    __shared__ uint32_t s_src[kVertChunk];              // entry inside the tile << 7 | bit << 2 | axis
    const uint32_t count = list_count(p.vertCount, p.numVertWords);
    const uint32_t tiles = (count + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const uint32_t tileBase = tile * DCSG_TILE_WORDS;
        const uint32_t tileFirst = p.tileVerts[tile];       // exclusive prefix of this tile
        const uint32_t tileEnd = tile + 1 < tiles ? p.tileVerts[tile + 1] : p.totals[2];
        if (tileEnd == tileFirst) continue;                 // no vertex in this tile: nobody reads these words' ids
        uint4 info[kPer];
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const uint32_t e = tileBase + threadIdx.x * kPer + k;
            info[k] = make_uint4(0u, 0u, 0u, 0u);
            uint32_t w = 0u;
            if (e < count) { w = list_word(p.vertList, e); info[k] = p.vinfo[w]; }
            s_vword[threadIdx.x * kPer + k] = w;
            mine += dcsg_popc(info[k].x) + dcsg_popc(info[k].y) + dcsg_popc(info[k].z);
        }
        uint32_t total;
        const uint32_t myFirst = block_exclusive_scan(mine, total, smem);
        {
            uint32_t id = tileFirst + myFirst;
#pragma unroll
            for (int k = 0; k < kPer; ++k) {
                const uint32_t cnt = dcsg_popc(info[k].x) + dcsg_popc(info[k].y) + dcsg_popc(info[k].z);
                if (cnt) p.vinfo[s_vword[threadIdx.x * kPer + k]].w = id;
                id += cnt;
            }
        }
        for (uint32_t chunk = 0; chunk < total; chunk += kVertChunk) {
            if (myFirst < chunk + kVertChunk && myFirst + mine > chunk) {
                uint32_t idx = myFirst;
#pragma unroll
                for (int k = 0; k < kPer; ++k) {
                    for (uint32_t any = info[k].x | info[k].y | info[k].z; any; any &= any - 1) {
                        const uint32_t b = __ffs(any) - 1;
#pragma unroll
                        for (uint32_t axis = 0; axis < 3; ++axis) {
                            const uint32_t bits = axis == 0 ? info[k].x : (axis == 1 ? info[k].y : info[k].z);
                            if (!((bits >> b) & 1u)) continue;
                            if (idx >= chunk && idx < chunk + kVertChunk) s_src[idx - chunk] = ((threadIdx.x * kPer + k) << 7) | (b << 2) | axis;
                            ++idx;
                        }
                    }
                }
            }
            __syncthreads();
            const uint32_t inChunk = min(kVertChunk, total - chunk);
            for (uint32_t i = threadIdx.x; i < inChunk; i += kThreads) {
                const uint32_t src = s_src[i];
                const int axis = (int)(src & 3u);
                int zl; uint32_t wi;
                word_to_plane(p.g, s_vword[src >> 7], zl, wi);
                const uint32_t gz = (uint32_t)(p.g.z0 + zl);
                const uint32_t lp = wi * 32u + ((src >> 2) & 31u);
                const uint32_t y = lp / (uint32_t)p.g.pitch, x = lp - y * (uint32_t)p.g.pitch;
                float mid[3];
                dcsg_edge_midpoint(p.px, p.py, p.pz, x, y, gz, axis, mid);
                const uint32_t id = tileFirst + chunk + i;
                p.vertices[(uint64_t)id * 3 + 0] = mid[0];
                p.vertices[(uint64_t)id * 3 + 1] = mid[1];
                p.vertices[(uint64_t)id * 3 + 2] = mid[2];
                p.vertexKeys[id] = dcsg_vertex_key(p.g, x, y, gz, axis);
            }
            __syncthreads();
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Triangles.  The CTA gathers the surface cells of its tile of the cell list into shared memory -- thread t owns entries
// 4t .. 4t+3, so one block scan numbers the cells in canonical order (word, then bit) -- and works through them
// kEmitChunk cells at a time in two phases:
//   A  one thread per CELL: corner mask from the sign bitmap, triangle count from the table, the compacted cell record;
//      a block scan gives every cell its first triangle, and every triangle of the chunk is tagged with its cell;
//   B  one thread per TRIANGLE: three times table edge -> owner word in vinfo -> vertex id, 12 bytes stored next to the
//      neighbouring threads'.  A cell emits 1 .. 5 triangles, so a thread per cell would leave most lanes idle here and
//      scatter its stores.
constexpr uint32_t kEmitChunk = 1024;

__global__ void __launch_bounds__(kThreads) k_emit_triangles(const dcsg_mesher_params p) {
    __shared__ uint32_t smem32[kThreads / 32 + 1];
    __shared__ uint32_t s_word[DCSG_TILE_WORDS];
    __shared__ uint16_t s_cell[kEmitChunk];             // entry inside the tile (10 bits) << 5 | bit
    __shared__ uint16_t s_triOff[kEmitChunk];           // first triangle of the cell inside the chunk
    __shared__ uint16_t s_triCell[kEmitChunk * 5];      // cell of every triangle of the chunk
    __shared__ uint8_t s_mask[kEmitChunk];
    const uint32_t count = list_count(p.cellCount, p.numCellWords);
    const uint32_t tiles = (count + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const uint32_t tileBase = tile * DCSG_TILE_WORDS;
        const uint32_t cellBase = p.tileCells[tile];         // exclusive prefixes of this tile
        uint32_t triRunning = p.tileTris[tile];
        if ((tile + 1 < tiles ? p.tileCells[tile + 1] : p.totals[0]) == cellBase) continue;     // no own cell in this tile
        uint32_t words[kPer];
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const uint32_t e = tileBase + threadIdx.x * kPer + k;
            uint32_t w = 0u, alive = 0u;
            if (e < count) {
                w = list_word(p.cellList, e);
                const int zl = (int)(w / p.g.planeWords);
                if (zl >= p.ownCell0 && zl < p.ownCell1) alive = p.alive[w];
            }
            words[k] = alive;
            s_word[threadIdx.x * kPer + k] = w;
            mine += dcsg_popc(alive);
        }
        uint32_t tileTotal;
        const uint32_t myFirst = block_exclusive_scan(mine, tileTotal, smem32);     // index of my first cell inside the tile
        for (uint32_t chunk = 0; chunk < tileTotal; chunk += kEmitChunk) {
            gather_cells(words, myFirst, mine, chunk, s_cell, kEmitChunk);
            __syncthreads();
            const uint32_t inChunk = min(kEmitChunk, tileTotal - chunk);
            // ---- phase A: one cell per thread, 256 cells per pass (a tile rarely holds more)
            uint32_t chunkTris = 0;
            for (uint32_t pass = 0; pass < inChunk; pass += kThreads) {
                const uint32_t i = pass + threadIdx.x;
                uint32_t n = 0;
                if (i < inChunk) {
                    const uint32_t code = s_cell[i];
                    int zl; uint32_t wi;
                    word_to_plane(p.g, s_word[code >> 5], zl, wi);
                    const uint32_t lp = wi * 32u + (code & 31u);
                    const uint32_t mask = cell_mask_at(p.g, p.sign, zl, lp);
                    n = __ldg(&p.triCount[mask]);
                    s_mask[i] = (uint8_t)mask;
                    const uint32_t y = lp / (uint32_t)p.g.pitch, x = lp - y * (uint32_t)p.g.pitch;
                    const uint32_t cell = cellBase + chunk + i;
                    p.cellIds[cell] = (uint64_t)x + (uint64_t)p.g.N * ((uint64_t)y + (uint64_t)p.g.N * (uint32_t)(p.g.z0 + zl));
                    p.cellMasks[cell] = (uint8_t)mask;
                }
                uint32_t passTris;
                const uint32_t off = chunkTris + block_exclusive_scan(n, passTris, smem32);
                chunkTris += passTris;
                if (i < inChunk) {
                    s_triOff[i] = (uint16_t)off;
                    for (uint32_t q = 0; q < n; ++q) s_triCell[off + q] = (uint16_t)i;
                }
            }
            __syncthreads();
            // ---- phase B: one triangle per thread (12 consecutive bytes each: a warp stores 384 contiguous bytes)
            for (uint32_t tri = threadIdx.x; tri < chunkTris; tri += kThreads) {
                const uint32_t i = s_triCell[tri];
                const uint32_t t = tri - s_triOff[i];
                const uint32_t code = s_cell[i];
                const uint64_t w = s_word[code >> 5];
                const uint32_t bit = code & 31u;
                const int8_t* row = p.triTable + (uint32_t)s_mask[i] * 16u + t * 3u;
                uint32_t ids[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const uint32_t edge = dcsg_edge_code(__ldg(&row[k]));
                    // owner point of the edge: (+dx, +dy, +dz) from the cell's min corner -> bit position inside / past the cell's word
                    const uint32_t pos = bit + (edge & 1u) + ((edge >> 1) & 1u) * (uint32_t)p.g.pitch;
                    const uint4 info = p.vinfo[w + (pos >> 5) + ((edge >> 2) & 1u) * (uint64_t)p.g.planeWords];
                    ids[k] = info.w + dcsg_vertex_rank(info.x, info.y, info.z, pos & 31u, (int)(edge >> 3));
                }
                const uint64_t at = (uint64_t)(triRunning + tri) * 3u;
                p.triangles[at + 0] = ids[0]; p.triangles[at + 1] = ids[1]; p.triangles[at + 2] = ids[2];
            }
            triRunning += chunkTris;
            __syncthreads();
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Work lists from word masks (mesher.h dcsg_worklist_params).  Thread t of a tile owns mask words 4t .. 4t+3, so the bits
// it lists ascend; two launches: per-tile counts, then every CTA sums the counts of the tiles before it (a thousand values)
// and writes its entries.
__device__ __forceinline__ uint32_t wl_bits(const dcsg_worklist_params& p, uint32_t mw, bool dilated) {
    const uint32_t first = mw * 32u;
    if (first >= p.numBits) return 0u;
    uint32_t v = 0u;
    if (!dilated) v = p.mask[mw];
    else {
        const int64_t b0 = (int64_t)first;
#pragma unroll
        for (int dz = 0; dz < 2; ++dz)
#pragma unroll
            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                for (int dx = 0; dx < 2; ++dx)
                    v |= dcsg_plane_bits(dx ? p.mask31 : p.mask, b0 - (int64_t)(dz ? p.planeWords : 0u) - (int64_t)(dy ? p.rowWords : 0u) - dx);
    }
    const uint32_t rest = p.numBits - first;
    return rest < 32u ? v & ((1u << rest) - 1u) : v;
}

__global__ void __launch_bounds__(kThreads) k_worklist_count(const dcsg_worklist_params p, uint32_t tiles) {
    __shared__ unsigned long long smem64[kThreads / 32 + 1];
    uint32_t a = 0, b = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t mw = blockIdx.x * kWorklistTile + threadIdx.x * 4u + k;
        if (p.mode == 0) a += dcsg_popc(wl_bits(p, mw, false));
        b += dcsg_popc(wl_bits(p, mw, true));
    }
    const unsigned long long total = block_sum((unsigned long long)a | ((unsigned long long)b << 32), smem64);
    if (threadIdx.x == 0) {
        p.scratch[blockIdx.x] = (uint32_t)total;
        p.scratch[tiles + blockIdx.x] = (uint32_t)(total >> 32);
    }
}

__global__ void __launch_bounds__(kThreads) k_worklist_fill(const dcsg_worklist_params p, uint32_t tiles) {
    __shared__ unsigned long long smem64[kThreads / 32 + 1];
    unsigned long long before = 0;
    for (uint32_t t = threadIdx.x; t < blockIdx.x; t += kThreads) before += (unsigned long long)p.scratch[t] | ((unsigned long long)p.scratch[tiles + t] << 32);
    before = block_sum(before, smem64);
    uint32_t wa[4], wb[4];
    uint32_t a = 0, b = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t mw = blockIdx.x * kWorklistTile + threadIdx.x * 4u + k;
        wa[k] = p.mode == 0 ? wl_bits(p, mw, false) : 0u;
        wb[k] = wl_bits(p, mw, true);
        a += dcsg_popc(wa[k]);
        b += dcsg_popc(wb[k]);
    }
    unsigned long long total;
    const unsigned long long mine = block_exclusive_scan((unsigned long long)a | ((unsigned long long)b << 32), total, smem64);
    uint32_t posA = (uint32_t)before + (uint32_t)mine, posB = (uint32_t)(before >> 32) + (uint32_t)(mine >> 32);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t base = (blockIdx.x * kWorklistTile + threadIdx.x * 4u + k) * 32u;
        for (uint32_t bits = wa[k]; bits; bits &= bits - 1) p.listA[posA++] = base + (uint32_t)(__ffs(bits) - 1);
        for (uint32_t bits = wb[k]; bits; bits &= bits - 1) p.listB[posB++] = base + (uint32_t)(__ffs(bits) - 1);
    }
    if (blockIdx.x == tiles - 1 && threadIdx.x == 0) {
        p.counts[0] = (uint32_t)before + (uint32_t)total;
        p.counts[1] = (uint32_t)(before >> 32) + (uint32_t)(total >> 32);
    }
}

// ---------------------------------------------------------------------------------------------
// clean-up of a sparse extraction (mesher.h dcsg_cleanup_params): the bitmaps are all-zero again afterwards
__global__ void __launch_bounds__(kThreads) k_cleanup(const dcsg_cleanup_params p) {
    const uint32_t cells = *p.cellCount;
    const uint64_t threads = (uint64_t)gridDim.x * kThreads;
    for (uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x; t < cells; t += threads) {
        const uint32_t w = p.cellList[t];
        p.leafAlive[w] = 0u;
        p.alive[w] = 0u;
    }
}

// ---------------------------------------------------------------------------------------------
// file bodies.  STL record (reference utils.hpp:59-99): normal (0,0,0), A, B, C each as (x, z, y),
// uint16 0 = 50 bytes.  Two records = 100 bytes = 25 aligned words per thread.  kACB: A, C, B instead -- the records of an
// outward-wound mesh, whose winding the (x, z, y) axis order would otherwise mirror
template <bool kACB>
__device__ __forceinline__ void stl_record_words(const float* v, const uint32_t* tri, uint32_t f[12]) {
    f[0] = f[1] = f[2] = 0u;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float* q = v + (uint64_t)tri[kACB && k ? 3 - k : k] * 3;
        f[3 + k * 3 + 0] = __float_as_uint(q[0]);
        f[3 + k * 3 + 1] = __float_as_uint(q[2]);
        f[3 + k * 3 + 2] = __float_as_uint(q[1]);
    }
}

template <bool kACB>
__global__ void __launch_bounds__(kThreads) k_format_stl(const float* __restrict__ v, const uint32_t* __restrict__ tris,
                                                         uint64_t n, uint8_t* __restrict__ out) {
    const uint64_t pair = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t t0 = pair * 2;
    if (t0 >= n) return;
    uint32_t a[12], b[12];
    stl_record_words<kACB>(v, tris + t0 * 3, a);
    uint32_t* o = reinterpret_cast<uint32_t*>(out + t0 * 50);
#pragma unroll
    for (int i = 0; i < 12; ++i) o[i] = a[i];
    if (t0 + 1 < n) {
        stl_record_words<kACB>(v, tris + (t0 + 1) * 3, b);
        o[12] = b[0] << 16;                                    // attribute of A (0) | low half of b[0]
#pragma unroll
        for (int i = 1; i < 12; ++i) o[12 + i] = (b[i - 1] >> 16) | (b[i] << 16);
        o[24] = b[11] >> 16;                                   // high half of b[11] | attribute of B (0)
    } else {
        *reinterpret_cast<uint16_t*>(out + t0 * 50 + 48) = 0;
    }
}

// PLY vertex rows (reference utils.hpp:117-123 through happly.h:1538-1562): x, y, z as double
__global__ void __launch_bounds__(kThreads) k_format_ply_vertices(const float* __restrict__ v, const uint32_t* __restrict__ tris,
                                                                  uint64_t n, double* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;     // soup vertex
    if (i >= n * 3) return;
    const float* q = v + (uint64_t)tris[i] * 3;
    out[i * 3 + 0] = (double)q[0];
    out[i * 3 + 1] = (double)q[1];
    out[i * 3 + 2] = (double)q[2];
}

// Four PLY face rows (uchar 3, three little-endian uint32 indices = 13 bytes) from their 12 indices: 13 aligned words
// when all four rows exist, bytes for the last partial group
__device__ __forceinline__ void store_face_rows(const uint32_t idx[12], uint64_t t0, uint64_t n, uint8_t* __restrict__ out) {
    uint8_t bytes[52];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        bytes[r * 13] = 3;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
#pragma unroll
            for (int s = 0; s < 4; ++s) bytes[r * 13 + 1 + k * 4 + s] = (uint8_t)(idx[r * 3 + k] >> (8 * s));
        }
    }
    if (t0 + 4 <= n) {
        uint32_t* o = reinterpret_cast<uint32_t*>(out + t0 * 13);
#pragma unroll
        for (int i = 0; i < 13; ++i)
            o[i] = (uint32_t)bytes[i * 4] | ((uint32_t)bytes[i * 4 + 1] << 8) | ((uint32_t)bytes[i * 4 + 2] << 16) |
                   ((uint32_t)bytes[i * 4 + 3] << 24);
    } else {
        const int valid = (int)(n - t0) * 13;
        for (int i = 0; i < valid; ++i) out[t0 * 13 + i] = bytes[i];
    }
}

// face rows of the indexed PLY: the mesh's own vertex ids plus `base` (a slab's first vertex in the whole mesh)
__global__ void __launch_bounds__(kThreads) k_format_ply_indexed_faces(const uint32_t* __restrict__ tris, uint64_t n, uint32_t base,
                                                                       uint8_t* __restrict__ out) {
    const uint64_t t0 = ((uint64_t)blockIdx.x * kThreads + threadIdx.x) * 4;
    if (t0 >= n) return;
    uint32_t idx[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) idx[i] = t0 * 3 + i < n * 3 ? tris[t0 * 3 + i] + base : 0u;
    store_face_rows(idx, t0, n, out);
}

// vertex rows of the indexed PLY with normals: x y z nx ny nz as float
__global__ void __launch_bounds__(kThreads) k_format_ply_indexed_vertices(const float* __restrict__ v, const float* __restrict__ nrm,
                                                                          uint64_t n, float* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        out[i * 6 + c] = v[i * 3 + c];
        out[i * 6 + 3 + c] = nrm[i * 3 + c];
    }
}

// PLY face rows (happly.h:587-603): uchar 3, then uint32 3i, 3i+1, 3i+2 = 13 bytes; four rows = 13 words
__global__ void __launch_bounds__(kThreads) k_format_ply_faces(uint64_t first, uint64_t n, uint8_t* __restrict__ out) {
    const uint64_t quad = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t t0 = quad * 4;
    if (t0 >= n) return;
    uint32_t idx[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) idx[i] = (uint32_t)((first + t0) * 3 + i);
    store_face_rows(idx, t0, n, out);
}

__global__ void __launch_bounds__(kThreads) k_expand_soup(const float* __restrict__ v, const uint32_t* __restrict__ tris,
                                                          uint64_t n, float* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n * 3) return;
    const float* q = v + (uint64_t)tris[i] * 3;
    out[i * 3 + 0] = q[0];
    out[i * 3 + 1] = q[1];
    out[i * 3 + 2] = q[2];
}


// ---------------------------------------------------------------------------------------------
// adaptive octree mode: leaves live on several levels (dcsg_k_adapt_level decides which nodes emit), the output
// is the reference's triangle SOUP (mesh.hpp:283-305): lookupTable[mask] on the midpoints of the NODE's edges.
// Canonical order: level, then node index (x fastest), then table order.  One thread owns one word of the
// concatenated per-level emit bitmaps.
// ---------------------------------------------------------------------------------------------
struct AdaptNodeWord { int level; uint32_t xw, ny, nz; };

__device__ __forceinline__ AdaptNodeWord adapt_decode(const dcsg_adapt_emit_params& p, uint32_t w) {
    AdaptNodeWord d;
    d.level = p.minLevel;
    while (d.level < p.maxLevel && w >= p.levelOff[d.level + 1]) ++d.level;
    const uint32_t local = w - p.levelOff[d.level];
    const uint32_t n = 1u << d.level;
    const uint32_t wordsPerRow = (n < 32u ? 32u : n) >> 5;
    d.xw = local % wordsPerRow;
    const uint32_t rest = local / wordsPerRow;
    d.ny = rest % n;
    d.nz = rest / n;
    return d;
}

__device__ __forceinline__ uint32_t adapt_bit(const dcsg_adapt_emit_params& p, uint32_t x, uint32_t y, uint32_t z) {
    const uint32_t lp = x + (uint32_t)p.g.pitch * y;
    return (p.sign[(uint64_t)(z - (uint32_t)p.g.z0) * p.g.planeWords + (lp >> 5)] >> (lp & 31u)) & 1u;     // slab-local plane
}

__device__ __forceinline__ uint32_t adapt_node_mask(const dcsg_adapt_emit_params& p, uint32_t x0, uint32_t y0, uint32_t z0, uint32_t size) {
    const uint32_t x1 = x0 + size, y1 = y0 + size, z1 = z0 + size;
    return (adapt_bit(p, x0, y0, z1) << 0) | (adapt_bit(p, x1, y0, z1) << 1) | (adapt_bit(p, x1, y0, z0) << 2) |
           (adapt_bit(p, x0, y0, z0) << 3) | (adapt_bit(p, x0, y1, z1) << 4) | (adapt_bit(p, x1, y1, z1) << 5) |
           (adapt_bit(p, x1, y1, z0) << 6) | (adapt_bit(p, x0, y1, z0) << 7);
}

__global__ void __launch_bounds__(kThreads) k_adapt_count(const dcsg_adapt_emit_params p) {
    __shared__ unsigned long long smem64[kThreads / 32 + 1];
    const uint32_t tileBase = p.firstWord + blockIdx.x * DCSG_TILE_WORDS;
    uint32_t cells = 0, tris = 0;
#pragma unroll 1
    for (int r = 0; r < kRounds; ++r) {
        const uint32_t w = tileBase + r * kThreads + threadIdx.x;
        if (w >= p.endWord) continue;
        uint32_t bits = p.emit[w];
        if (!bits) continue;
        const AdaptNodeWord d = adapt_decode(p, w);
        const int sh = p.g.L - d.level;
        uint32_t wordTris = 0;
        while (bits) {
            const uint32_t b = __ffs(bits) - 1;
            bits &= bits - 1;
            const uint32_t mask = adapt_node_mask(p, (d.xw * 32u + b) << sh, d.ny << sh, d.nz << sh, 1u << sh);
            wordTris += __ldg(&p.triCount[mask]);
            ++cells;
        }
        tris += wordTris;
        // triangles per octree level: the canonical order is (level, node), so in a sharded export a rank's triangles
        // form one run per level of the whole mesh
        if (p.levelTris && wordTris) atomicAdd(&p.levelTris[d.level], wordTris);
    }
    const unsigned long long total = block_sum((unsigned long long)cells | ((unsigned long long)tris << 32), smem64);
    if (threadIdx.x == 0) {
        p.tileCells[blockIdx.x] = (uint32_t)total;
        p.tileTris[blockIdx.x] = (uint32_t)(total >> 32);
    }
}

__global__ void __launch_bounds__(kThreads) k_adapt_emit(const dcsg_adapt_emit_params p) {
    __shared__ unsigned long long smem64[kThreads / 32 + 1];
    const uint32_t tileBase = p.firstWord + blockIdx.x * DCSG_TILE_WORDS;
    uint32_t cellRunning = p.tileCells[blockIdx.x];      // exclusive prefixes of this tile
    uint32_t triRunning = p.tileTris[blockIdx.x];
#pragma unroll 1
    for (int r = 0; r < kRounds; ++r) {
        const uint32_t w = tileBase + r * kThreads + threadIdx.x;
        const uint32_t word = w < p.endWord ? p.emit[w] : 0u;
        AdaptNodeWord d = {0, 0u, 0u, 0u};
        uint32_t myTris = 0;
        if (word) {
            d = adapt_decode(p, w);
            const int sh = p.g.L - d.level;
            for (uint32_t bits = word; bits; bits &= bits - 1) {
                const uint32_t b = __ffs(bits) - 1;
                myTris += __ldg(&p.triCount[adapt_node_mask(p, (d.xw * 32u + b) << sh, d.ny << sh, d.nz << sh, 1u << sh)]);
            }
        }
        unsigned long long total;
        const unsigned long long before = block_exclusive_scan((unsigned long long)dcsg_popc(word) | ((unsigned long long)myTris << 32), total, smem64);
        uint32_t cellId = cellRunning + (uint32_t)before;
        uint32_t triId = triRunning + (uint32_t)(before >> 32);
        cellRunning += (uint32_t)total;
        triRunning += (uint32_t)(total >> 32);
        if (!word) continue;
        const int sh = p.g.L - d.level;
        const uint32_t size = 1u << sh, n = 1u << d.level;
        for (uint32_t bits = word; bits; bits &= bits - 1) {
            const uint32_t b = __ffs(bits) - 1;
            const uint32_t nx = d.xw * 32u + b;
            const uint32_t x0 = nx << sh, y0 = d.ny << sh, z0 = d.nz << sh;
            const uint32_t mask = adapt_node_mask(p, x0, y0, z0, size);
            p.cellIds[cellId] = ((uint64_t)d.level << 56) | ((uint64_t)nx + (uint64_t)n * ((uint64_t)d.ny + (uint64_t)n * d.nz));
            p.cellMasks[cellId] = (uint8_t)mask;
            ++cellId;
            const uint32_t count = __ldg(&p.triCount[mask]);
            const int8_t* row = p.triTable + mask * 16;
            for (uint32_t t = 0; t < count; ++t) {
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const uint32_t code = dcsg_edge_code(__ldg(&row[t * 3 + k]));
                    const int axis = (int)(code >> 3);
                    const uint32_t ax = x0 + (code & 1u) * size, ay = y0 + ((code >> 1) & 1u) * size, az = z0 + ((code >> 2) & 1u) * size;
                    const uint32_t bx = ax + (axis == 0 ? size : 0u), by = ay + (axis == 1 ? size : 0u), bz = az + (axis == 2 ? size : 0u);
                    float* out = p.soup + ((uint64_t)triId * 3 + k) * 3;
                    out[0] = 0.5f * p.px[ax] + 0.5f * p.px[bx];       // Vector3f::midpoint, geometry.hpp:91-93
                    out[1] = 0.5f * p.py[ay] + 0.5f * p.py[by];
                    out[2] = 0.5f * p.pz[az] + 0.5f * p.pz[bz];
                }
                ++triId;
            }
        }
    }
}

// cms::retopologize as the reference build behaves (mesh.hpp:432-529; see oracle/mesher_port.cpp
// retopologize_as_built for the provenance): every triangle edge is resampled at `points` positions
// start + (i/points)*delta and the 3*points-gon is cut into a strip (geometry.hpp:228-248) of
// 3*points - 2 triangles.  The strip's triangles share the polygon's 3*points points (each is used by up to four of
// them, 66 soup vertices from 24 points at points = 8), so the result is written INDEXED: point k of source triangle t
// is vertex t * 3*points + k, computed once -- and projected once: equal inputs give equal outputs, the soup the
// reference projects vertex by vertex holds bit-identical copies.  One thread per point, one per output triangle.
__device__ __forceinline__ void retopo_point(const float* tri, uint32_t k, uint32_t points, float out[3]) {
    const uint32_t e = k / points, i = k - e * points;
    const float* start = tri + e * 3;
    const float* end = tri + ((e + 1u) % 3u) * 3;
    const float f = (float)i / (float)(int)points;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float delta = end[c] - start[c];
        out[c] = start[c] + f * delta;
    }
}

__global__ void __launch_bounds__(kThreads) k_retopo_points(const float* __restrict__ in, uint64_t numIn, uint32_t points,
                                                            float* __restrict__ vertices) {
    const uint32_t n = 3u * points;
    const uint64_t o = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (o >= numIn * n) return;
    const uint64_t t = o / n;
    retopo_point(in + t * 9, (uint32_t)(o - t * n), points, vertices + o * 3);
}

__global__ void __launch_bounds__(kThreads) k_retopo_triangles(uint64_t numIn, uint32_t points, uint32_t* __restrict__ triangles) {
    const uint32_t n = 3u * points;                                // even for points >= 2 (points == 1 is the identity)
    const uint32_t perTri = n - 2u;
    const uint64_t o = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (o >= numIn * perTri) return;
    const uint64_t t = o / perTri;
    const uint32_t j = (uint32_t)(o - t * perTri);
    const uint32_t A = j >> 1, B = A + 1u, D = n - 1u - A, C = D - 1u;
    const uint32_t first = (uint32_t)(t * n);
    triangles[o * 3 + 0] = first + ((j & 1u) ? C : A);
    triangles[o * 3 + 1] = first + ((j & 1u) ? D : B);
    triangles[o * 3 + 2] = first + ((j & 1u) ? A : C);
}

// multi-GPU: a slab's triangles with GLOBAL vertex ids (local id + the slab's vertex offset in the whole mesh), written to the
// gathering rank's array (a peer mapping over NVLink) on a side stream while the projection runs
__global__ void __launch_bounds__(kThreads) k_rebase_indices(const uint32_t* __restrict__ in, uint64_t n, uint32_t base, uint32_t* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    for (uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) out[i] = in[i] + base;
}

__global__ void __launch_bounds__(kThreads) k_iota(uint32_t* __restrict__ out, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i < n) out[i] = (uint32_t)i;
}

// Sign changes of the 256^3 bounding-box search lattice per z index (dcsg_k_bbox wrote one sign bit per sample; word
// (ix*256 + iy)*8 + iz/32).  hist[0..255] = x- and y-edges lying in plane iz, hist[256..511] = z-edges from iz to iz+1.
__global__ void __launch_bounds__(kThreads) k_surface_hist(const uint32_t* __restrict__ bits, uint32_t* __restrict__ hist, uint32_t firstWord) {
    __shared__ uint32_t s_hist[512];
    for (int i = threadIdx.x; i < 512; i += kThreads) s_hist[i] = 0u;
    __syncthreads();
    const uint32_t w = firstWord + blockIdx.x * kThreads + threadIdx.x;        // 2^19 words; a rank takes those of its ix columns
    const uint32_t zw = w & 7u, iy = (w >> 3) & 255u, ix = w >> 11;
    const uint32_t v = bits[w];
    const uint32_t up = zw < 7u ? bits[w + 1] : 0u;
    uint32_t cz = v ^ ((v >> 1) | (up << 31));
    if (zw == 7u) cz &= 0x7fffffffu;                                   // no sample above iz = 255
    uint32_t cxy_lo = iy < 255u ? (v ^ bits[w + 8]) : 0u;
    uint32_t cxy_hi = ix < 255u ? (v ^ bits[w + 2048]) : 0u;
    for (uint32_t m = cz; m; m &= m - 1) atomicAdd(&s_hist[256 + zw * 32u + (__ffs(m) - 1)], 1u);
    for (uint32_t m = cxy_lo; m; m &= m - 1) atomicAdd(&s_hist[zw * 32u + (__ffs(m) - 1)], 1u);
    for (uint32_t m = cxy_hi; m; m &= m - 1) atomicAdd(&s_hist[zw * 32u + (__ffs(m) - 1)], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < 512; i += kThreads)
        if (s_hist[i]) atomicAdd(&hist[i], s_hist[i]);
}

// ---------------------------------------------------------------------------------------------
// weld: vertices whose positions are bit-identical become one, numbered by the smallest input index among them
// (dcsg_launch_weld).  Sorted positions j, input vertices i.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pos_bits(const float* v, uint64_t i, int c) { return __float_as_uint(v[i * 3 + c]); }

__global__ void __launch_bounds__(kThreads) k_weld_init(const float* __restrict__ v, uint64_t n, uint32_t* __restrict__ zKey,
                                                        uint32_t* __restrict__ index) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    zKey[i] = pos_bits(v, i, 2);
    index[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(kThreads) k_weld_xy(const float* __restrict__ v, uint64_t n, const uint32_t* __restrict__ index,
                                                      uint64_t* __restrict__ xyKey) {
    const uint64_t j = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (j >= n) return;
    const uint32_t i = index[j];
    xyKey[j] = ((uint64_t)pos_bits(v, i, 0) << 32) | pos_bits(v, i, 1);
}

// a run of equal keys starts at its head; headPos = j at heads (0 elsewhere, a max-scan spreads it), first[i] = i is a head
__global__ void __launch_bounds__(kThreads) k_weld_heads(const float* __restrict__ v, uint64_t n, const uint64_t* __restrict__ xyKey,
                                                         const uint32_t* __restrict__ index, uint32_t* __restrict__ headPos,
                                                         uint32_t* __restrict__ first) {
    const uint64_t j = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (j >= n) return;
    const uint32_t i = index[j];
    const bool head = j == 0 || xyKey[j] != xyKey[j - 1] || pos_bits(v, i, 2) != pos_bits(v, index[j - 1], 2);
    headPos[j] = head ? (uint32_t)j : 0u;
    first[i] = head ? 1u : 0u;
}

__global__ void __launch_bounds__(kThreads) k_weld_rep(uint64_t n, const uint32_t* __restrict__ index, const uint32_t* __restrict__ runHead,
                                                       uint32_t* __restrict__ rep) {
    const uint64_t j = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (j >= n) return;
    rep[index[j]] = index[runHead[j]];
}

__global__ void __launch_bounds__(kThreads) k_weld_compact(const float* __restrict__ v, const float* __restrict__ nrm, uint64_t n,
                                                           const uint32_t* __restrict__ first, const uint32_t* __restrict__ newId,
                                                           float* __restrict__ outV, float* __restrict__ outN, uint32_t* __restrict__ unique) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    if (i == n - 1) *unique = newId[i] + first[i];
    if (!first[i]) return;
    const uint64_t o = newId[i];
#pragma unroll
    for (int c = 0; c < 3; ++c) outV[o * 3 + c] = v[i * 3 + c];
    if (nrm) {
#pragma unroll
        for (int c = 0; c < 3; ++c) outN[o * 3 + c] = nrm[i * 3 + c];
    }
}

__global__ void __launch_bounds__(kThreads) k_weld_remap(uint32_t* __restrict__ tris, uint64_t count, const uint32_t* __restrict__ rep,
                                                         const uint32_t* __restrict__ newId) {
    const uint64_t k = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (k < count) tris[k] = newId[rep[tris[k]]];
}

// ---------------------------------------------------------------------------------------------
// outward winding (dcsg_launch_orient): per cell, its triangle count (table triangles x unit), an exclusive scan, then one
// thread per cell swaps corners 1 and 2 of the triangles of its flagged table slots
__global__ void __launch_bounds__(kThreads) k_orient_count(const uint8_t* __restrict__ masks, uint64_t n, const uint8_t* __restrict__ triCount,
                                                           uint32_t unit, uint32_t* __restrict__ count) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i < n) count[i] = (uint32_t)__ldg(&triCount[masks[i]]) * unit;
}

__global__ void __launch_bounds__(kThreads) k_orient_apply(const dcsg_orient_params p, const uint32_t* __restrict__ first) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= p.numCells) return;
    const uint32_t mask = p.cellMasks[i];
    const uint64_t f = first[i];
    const uint64_t end = f + (uint64_t)__ldg(&p.triCount[mask]) * p.unit;
    if (i == p.numCells - 1) *p.total = (uint32_t)end;
    if (end > p.numTriangles) return;                   // cells that do not match the triangles (the caller fails the call)
    for (uint32_t flip = __ldg(&p.triFlip[mask]); flip; flip &= flip - 1) {
        uint32_t* tri = p.triangles + (f + (uint64_t)(__ffs(flip) - 1) * p.unit) * 3;
        for (uint32_t c = 0; c < p.unit; ++c, tri += 3) {
            const uint32_t b = tri[1];
            tri[1] = tri[2];
            tri[2] = b;
        }
    }
}

struct WeldMax {
    __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

inline uint32_t blocks_for(uint64_t items, uint32_t per_block) { return (uint32_t)((items + per_block - 1) / per_block); }

// Scratch of the weld: n-word arrays, then cub's temporary storage (the largest any of its four calls needs)
struct WeldLayout {
    size_t xyA, xyB, idxA, idxB, headPos, runHead, first, newId, rep, temp, tempBytes, total;
    explicit WeldLayout(uint64_t n) {
        auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
        size_t o = 0;
        xyA = o; o += align(n * 8);
        xyB = o; o += align(n * 8);
        idxA = o; o += align(n * 4);
        idxB = o; o += align(n * 4);
        headPos = o; o += align(n * 4);
        runHead = o; o += align(n * 4);
        first = o; o += align(n * 4);
        newId = o; o += align(n * 4);
        rep = o; o += align(n * 4);
        size_t a = 0, b = 0, c = 0, d = 0;
        const long long items = (long long)n;
        cub::DeviceRadixSort::SortPairs(nullptr, a, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, items);
        cub::DeviceRadixSort::SortPairs(nullptr, b, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, items);
        cub::DeviceScan::InclusiveScan(nullptr, c, (uint32_t*)nullptr, (uint32_t*)nullptr, WeldMax(), items);
        cub::DeviceScan::ExclusiveSum(nullptr, d, (uint32_t*)nullptr, (uint32_t*)nullptr, items);
        tempBytes = std::max(std::max(a, b), std::max(c, d));
        temp = o; o += align(tempBytes);
        total = o;
    }
};

// Scratch of the orientation: per-cell counts and their exclusive prefix, then cub's temporary storage
struct OrientLayout {
    size_t count, first, temp, tempBytes, total;
    explicit OrientLayout(uint64_t n) {
        auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
        count = 0;
        first = align(n * 4);
        temp = first + align(n * 4);
        tempBytes = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tempBytes, (uint32_t*)nullptr, (uint32_t*)nullptr, (long long)n);
        total = temp + align(tempBytes);
    }
};

// ---------------------------------------------------------------------------------------------
// mesh inspection (dcsg_launch_inspect).  Triangles t, half-edges 3t + e, vertices v.
// ---------------------------------------------------------------------------------------------
constexpr uint64_t kNoEdge = ~0ull;                     // half-edge key of a degenerate triangle: sorts after every real key
constexpr uint32_t kNoLabel = ~0u;                      // component label of a degenerate triangle

__device__ __forceinline__ bool inspect_degenerate(uint32_t a, uint32_t b, uint32_t c) { return a == b || b == c || a == c; }

__global__ void __launch_bounds__(kThreads) k_inspect_check(const uint32_t* __restrict__ tris, uint64_t count, uint64_t numVertices,
                                                            uint32_t* __restrict__ bad) {
    const uint64_t k = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (k < count && tris[k] >= numVertices) atomicOr(bad, 1u);
}

__global__ void __launch_bounds__(kThreads) k_inspect_init(uint64_t n, uint32_t* __restrict__ parent, uint8_t* __restrict__ ref) {
    const uint64_t v = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (v >= n) return;
    parent[v] = (uint32_t)v;
    ref[v] = 0;
}

// Union-find whose parents only ever decrease (parent[v] <= v): a root is the smallest id of its tree.  Only roots are
// written by atomicCAS, only non-roots by the path halving's plain stores, and both store an ancestor, so every interleaving
// leaves the same partition, and the final roots -- the components' smallest ids -- do not depend on the schedule.
__device__ __forceinline__ uint32_t uf_find(uint32_t* p, uint32_t x) {
    volatile uint32_t* vp = p;
    uint32_t cur = vp[x];
    if (cur == x) return x;
    uint32_t prev = x, next;
    while (cur > (next = vp[cur])) {
        vp[prev] = next;
        prev = cur;
        cur = next;
    }
    return cur;
}

__device__ __forceinline__ void uf_unite(uint32_t* p, uint32_t a, uint32_t b) {
    a = uf_find(p, a);
    b = uf_find(p, b);
    while (a != b) {
        if (a > b) { const uint32_t t = a; a = b; b = t; }
        const uint32_t old = atomicCAS(&p[b], b, a);     // hook the larger root under the smaller one
        if (old == b) return;
        b = uf_find(p, old);                              // b was hooked meanwhile: go on from its new root
        a = uf_find(p, a);
    }
}

// per triangle: its half-edge keys min << 32 | max with the direction bit (a < b), the referenced marks, the unions
__global__ void __launch_bounds__(kThreads) k_inspect_triangles(const uint32_t* __restrict__ tris, uint64_t n, uint64_t* __restrict__ keys,
                                                                uint8_t* __restrict__ fwd, uint8_t* __restrict__ ref, uint32_t* parent) {
    const uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= n) return;
    const uint32_t id[3] = {tris[t * 3], tris[t * 3 + 1], tris[t * 3 + 2]};
    const bool deg = inspect_degenerate(id[0], id[1], id[2]);
#pragma unroll
    for (int e = 0; e < 3; ++e) {
        const uint32_t x = id[e], y = id[e == 2 ? 0 : e + 1];
        keys[t * 3 + e] = deg ? kNoEdge : ((uint64_t)min(x, y) << 32) | max(x, y);
        fwd[t * 3 + e] = x < y ? 1 : 0;
    }
    if (deg) return;
    ref[id[0]] = ref[id[1]] = ref[id[2]] = 1;
    uf_unite(parent, id[0], id[1]);
    uf_unite(parent, id[0], id[2]);
}

// Every vertex to its root.  No path halving here: a halving store of another thread could put an older ancestor back over a
// root this pass has already written.  Each thread writes only its own vertex, and only the root, which no longer changes.
__global__ void __launch_bounds__(kThreads) k_inspect_flatten(uint64_t n, uint32_t* parent) {
    const uint64_t v = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (v >= n) return;
    volatile uint32_t* vp = parent;
    uint32_t r = (uint32_t)v, next;
    while ((next = vp[r]) != r) r = next;
    vp[v] = r;
}

__global__ void __launch_bounds__(kThreads) k_inspect_labels(const uint32_t* __restrict__ tris, uint64_t n, const uint32_t* __restrict__ parent,
                                                             uint32_t* __restrict__ label, uint32_t* __restrict__ index) {
    const uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= n) return;
    const uint32_t a = tris[t * 3], b = tris[t * 3 + 1], c = tris[t * 3 + 2];
    label[t] = inspect_degenerate(a, b, c) ? kNoLabel : parent[a];
    index[t] = (uint32_t)t;
}

// The shells' sums (dcsg_launch_inspect): the sorted (label, triangle) sequence is cut into pieces at every label change and
// every kInspectPiece-th item; each piece, then each shell's run of piece partials, is one segment of a segmented reduction --
// one CTA per segment in a fixed order, unlike a reduction by key, whose look-back combines the partials of a run that spans
// tiles in an order that depends on the schedule.
constexpr long long kInspectPiece = 4096;
using InspectCount = thrust::counting_iterator<long long>;

__global__ void __launch_bounds__(kThreads) k_inspect_piece_heads(const uint32_t* __restrict__ label, uint64_t n, uint8_t* __restrict__ head) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i < n) head[i] = i == 0 || label[i] != label[i - 1] || i % kInspectPiece == 0;
}

// piece q starts a shell's run when its first item's label differs from the previous piece's (flags past the pieces: 0)
__global__ void __launch_bounds__(kThreads) k_inspect_run_heads(const uint32_t* __restrict__ label, uint64_t n, const long long* __restrict__ pieceBegin,
                                                                const long long* __restrict__ pieces, uint8_t* __restrict__ head) {
    const long long q = (long long)blockIdx.x * kThreads + threadIdx.x;
    if ((uint64_t)q < n) head[q] = q < *pieces && (q == 0 || label[pieceBegin[q]] != label[pieceBegin[q - 1]]);
}

// end of segment s: the next one's begin, or `total` after the last of *count
struct InspectSegmentEnd {
    const long long* begin;
    const long long* count;
    long long total;
    __device__ long long operator()(long long s) const { return s + 1 < *count ? begin[s + 1] : total; }
};
using InspectEnds = thrust::transform_iterator<InspectSegmentEnd, InspectCount>;

// exact float minimum / maximum, -0 below +0, so that the order of the reduction cannot show
__device__ __forceinline__ float min_total(float a, float b) { return (a < b || (a == b && signbit(a))) ? a : b; }
__device__ __forceinline__ float max_total(float a, float b) { return (a > b || (a == b && !signbit(b))) ? a : b; }

struct InspectVertexTerm {
    const float* v;
    const uint8_t* ref;
    const uint32_t* parent;
    __device__ dcsg_inspect_vertex_sums operator()(long long i) const {
        dcsg_inspect_vertex_sums s;
        const float x = v[i * 3], y = v[i * 3 + 1], z = v[i * 3 + 2];
        const bool r = ref[i] != 0, finite = isfinite(x) && isfinite(y) && isfinite(z), use = r && finite;
        s.referenced = r;
        s.nonfinite = r && !finite;
        s.roots = r && parent[i] == (uint32_t)i;
        s.lo[0] = use ? x : INFINITY; s.lo[1] = use ? y : INFINITY; s.lo[2] = use ? z : INFINITY;
        s.hi[0] = use ? x : -INFINITY; s.hi[1] = use ? y : -INFINITY; s.hi[2] = use ? z : -INFINITY;
        return s;
    }
};
struct InspectVertexSum {
    __device__ dcsg_inspect_vertex_sums operator()(const dcsg_inspect_vertex_sums& a, const dcsg_inspect_vertex_sums& b) const {
        dcsg_inspect_vertex_sums s;
        s.referenced = a.referenced + b.referenced;
        s.nonfinite = a.nonfinite + b.nonfinite;
        s.roots = a.roots + b.roots;
        for (int c = 0; c < 3; ++c) { s.lo[c] = min_total(a.lo[c], b.lo[c]); s.hi[c] = max_total(a.hi[c], b.hi[c]); }
        return s;
    }
};

// The per-triangle terms, one fixed sequence of double operations (the library is compiled with -fmad=false): DESIGN.md 7d.
struct InspectTriangleTerm {
    const float* v;
    const uint32_t* tris;
    __device__ dcsg_inspect_triangle_sums operator()(long long t) const {
        dcsg_inspect_triangle_sums s = {};
        const uint32_t ia = tris[t * 3], ib = tris[t * 3 + 1], ic = tris[t * 3 + 2];
        if (inspect_degenerate(ia, ib, ic)) { s.degenerate = 1; return s; }
        const float* fa = v + (uint64_t)ia * 3;
        const float* fb = v + (uint64_t)ib * 3;
        const float* fc = v + (uint64_t)ic * 3;
        bool finite = true;
        for (int c = 0; c < 3; ++c) finite = finite && isfinite(fa[c]) && isfinite(fb[c]) && isfinite(fc[c]);
        if (!finite) { s.nonfinite = 1; return s; }
        const double ax = fa[0], ay = fa[1], az = fa[2], bx = fb[0], by = fb[1], bz = fb[2], cx = fc[0], cy = fc[1], cz = fc[2];
        const double ux = bx - ax, uy = by - ay, uz = bz - az, wx = cx - ax, wy = cy - ay, wz = cz - az;
        const double nx = uy * wz - uz * wy, ny = uz * wx - ux * wz, nz = ux * wy - uy * wx;
        s.zeroArea = nx == 0.0 && ny == 0.0 && nz == 0.0;
        s.area = 0.5 * sqrt((nx * nx + ny * ny) + nz * nz);
        s.volume = ((ax * (by * cz - bz * cy) + ay * (bz * cx - bx * cz)) + az * (bx * cy - by * cx)) / 6.0;
        s.moment[0] = s.volume * ((ax + bx) + cx);
        s.moment[1] = s.volume * ((ay + by) + cy);
        s.moment[2] = s.volume * ((az + bz) + cz);
        return s;
    }
};
struct InspectTriangleSum {
    __device__ dcsg_inspect_triangle_sums operator()(const dcsg_inspect_triangle_sums& a, const dcsg_inspect_triangle_sums& b) const {
        dcsg_inspect_triangle_sums s;
        s.degenerate = a.degenerate + b.degenerate;
        s.zeroArea = a.zeroArea + b.zeroArea;
        s.nonfinite = a.nonfinite + b.nonfinite;
        s.area = a.area + b.area;
        s.volume = a.volume + b.volume;
        for (int c = 0; c < 3; ++c) s.moment[c] = a.moment[c] + b.moment[c];
        return s;
    }
};

// component runs: the triangles of a run, by index, in ascending order (the sort is stable)
struct InspectComponentTerm {
    InspectTriangleTerm term;
    __device__ dcsg_inspect_component operator()(uint32_t t) const {
        const dcsg_inspect_triangle_sums s = term((long long)t);
        return dcsg_inspect_component{1, s.area, s.volume};
    }
};
struct InspectComponentSum {
    __device__ dcsg_inspect_component operator()(const dcsg_inspect_component& a, const dcsg_inspect_component& b) const {
        return dcsg_inspect_component{a.triangles + b.triangles, a.area + b.area, a.volume + b.volume};
    }
};

// half-edge runs: (1 << 32 | direction bit) summed per key = (k half-edges) << 32 | (f of them with a < b)
struct InspectHalfEdge {
    __device__ uint64_t operator()(uint8_t forward) const { return (1ull << 32) | forward; }
};
struct InspectAdd {
    __device__ uint64_t operator()(uint64_t a, uint64_t b) const { return a + b; }
};
struct InspectEdgeTerm {
    const uint64_t* key;
    const uint64_t* packed;
    const uint64_t* runs;
    __device__ dcsg_inspect_edge_sums operator()(long long i) const {
        dcsg_inspect_edge_sums s = {};
        if ((uint64_t)i >= *runs || key[i] == kNoEdge) return s;
        const uint64_t k = packed[i] >> 32, f = packed[i] & 0xffffffffull;
        s.edges = 1;
        s.boundary = k == 1;
        s.manifold = k == 2;
        s.nonmanifold = k >= 3;
        s.misoriented = k == 2 && f != 1;
        return s;
    }
};
struct InspectEdgeSum {
    __device__ dcsg_inspect_edge_sums operator()(const dcsg_inspect_edge_sums& a, const dcsg_inspect_edge_sums& b) const {
        return dcsg_inspect_edge_sums{a.edges + b.edges, a.boundary + b.boundary, a.manifold + b.manifold, a.nonmanifold + b.nonmanifold,
                                      a.misoriented + b.misoriented};
    }
};

using InspectHalfEdges = thrust::transform_iterator<InspectHalfEdge, const uint8_t*>;
using InspectComponentTerms = thrust::transform_iterator<InspectComponentTerm, const uint32_t*>;

// bits of the sort keys: ids < n need bitsFor(n) bits, and the sentinels' low bits (all ones) still sort last
inline int bits_for(uint64_t n) {
    int b = 1;
    while (b < 32 && (n >> b)) ++b;
    return b;
}

// Scratch of the inspection: half-edge keys and direction bits (sorted copies), the runs' packed counts, union-find parents and
// referenced marks, triangle labels and indices (sorted copies), the edge run count, then cub's temporary storage
struct InspectLayout {
    size_t keysA, keysB, fwdA, fwdB, packed, parent, ref, labelA, labelB, indexA, indexB, head, pieceBegin, runBegin, partial, runs, counts,
        temp, tempBytes, total;
    InspectLayout(uint64_t nv, uint64_t nt) {
        auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const uint64_t h = nt * 3;
        size_t o = 0;
        keysA = o; o += align(h * 8);
        keysB = o; o += align(h * 8);
        fwdA = o; o += align(h);
        fwdB = o; o += align(h);
        packed = o; o += align(h * 8);
        parent = o; o += align(nv * 4);
        ref = o; o += align(nv);
        labelA = o; o += align(nt * 4);
        labelB = o; o += align(nt * 4);
        indexA = o; o += align(nt * 4);
        indexB = o; o += align(nt * 4);
        head = o; o += align(nt);
        pieceBegin = o; o += align(nt * 8);
        runBegin = o; o += align(nt * 8);
        partial = o; o += align(nt * sizeof(dcsg_inspect_component));
        runs = o; o += align(8);
        counts = o; o += align(16);
        size_t b[10] = {};
        const long long hi = (long long)h, ti = (long long)nt, vi = (long long)nv;
        cub::DeviceRadixSort::SortPairs(nullptr, b[0], (uint64_t*)nullptr, (uint64_t*)nullptr, (uint8_t*)nullptr, (uint8_t*)nullptr, hi);
        cub::DeviceReduce::ReduceByKey(nullptr, b[1], (uint64_t*)nullptr, (uint64_t*)nullptr, InspectHalfEdges(nullptr, InspectHalfEdge()),
                                       (uint64_t*)nullptr, (uint64_t*)nullptr, InspectAdd(), hi);
        cub::DeviceRadixSort::SortPairs(nullptr, b[2], (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, ti);
        cub::DeviceSelect::Flagged(nullptr, b[3], InspectCount(0), (const uint8_t*)nullptr, (long long*)nullptr, (long long*)nullptr, ti);
        const int segs = (int)std::min<uint64_t>(nt, 0x7fffffffull);
        const InspectEnds ends(InspectCount(0), InspectSegmentEnd{});
        cub::DeviceSegmentedReduce::Reduce(nullptr, b[7], InspectComponentTerms(nullptr, InspectComponentTerm{}),
                                           (dcsg_inspect_component*)nullptr, segs, (const long long*)nullptr, ends, InspectComponentSum(),
                                           dcsg_inspect_component{});
        cub::DeviceSegmentedReduce::Reduce(nullptr, b[8], (const dcsg_inspect_component*)nullptr, (dcsg_inspect_component*)nullptr, segs,
                                           (const long long*)nullptr, ends, InspectComponentSum(), dcsg_inspect_component{});
        cub::DeviceReduce::Reduce(nullptr, b[4], thrust::make_transform_iterator(InspectCount(0), InspectVertexTerm{}),
                                  (dcsg_inspect_vertex_sums*)nullptr, vi, InspectVertexSum(), dcsg_inspect_vertex_sums{});
        cub::DeviceReduce::Reduce(nullptr, b[5], thrust::make_transform_iterator(InspectCount(0), InspectTriangleTerm{}),
                                  (dcsg_inspect_triangle_sums*)nullptr, ti, InspectTriangleSum(), dcsg_inspect_triangle_sums{});
        cub::DeviceReduce::Reduce(nullptr, b[6], thrust::make_transform_iterator(InspectCount(0), InspectEdgeTerm{}),
                                  (dcsg_inspect_edge_sums*)nullptr, hi, InspectEdgeSum(), dcsg_inspect_edge_sums{});
        tempBytes = *std::max_element(b, b + 10);
        temp = o; o += align(tempBytes);
        total = o;
    }
};

// ---------------------------------------------------------------------------------------------
// mesh deviation (dcsg_launch_deviation_*).  The SDF values come from the scene module's dcsg_k_eval_sdf, which the host
// launches on the vertices and on every chunk's points: this file only makes the points and reduces the values.
// ---------------------------------------------------------------------------------------------

// sample (i, j) of triangle (a, b, c) at subdivision k, per coordinate in this order of IEEE operations (-fmad=false)
__device__ __forceinline__ void deviation_point(const float* a, const float* b, const float* c, int i, int j, int k, float* p) {
    const float w0 = (float)(k - i - j), wi = (float)i, wj = (float)j, kk = (float)k;
#pragma unroll
    for (int d = 0; d < 3; ++d) p[d] = ((a[d] * w0 + b[d] * wi) + c[d] * wj) / kk;
}

__global__ void __launch_bounds__(kThreads) k_deviation_marks(const uint32_t* __restrict__ tris, uint64_t n, uint8_t* __restrict__ ref) {
    const uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= n) return;
    const uint32_t a = tris[t * 3], b = tris[t * 3 + 1], c = tris[t * 3 + 2];
    if (!inspect_degenerate(a, b, c)) ref[a] = ref[b] = ref[c] = 1;
}

// one thread per sample point: point q of the chunk is sample q % S of triangle first + q / S
__global__ void __launch_bounds__(kThreads) k_deviation_points(const dcsg_deviation_params p, uint64_t first, uint64_t count, float* __restrict__ pts) {
    const uint64_t q = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (q >= count * (uint64_t)p.samples) return;
    const uint64_t t = first + q / (uint64_t)p.samples;
    const int s = (int)(q % (uint64_t)p.samples);
    const uint32_t* id = p.triangles + t * 3;
    float x[3];
    deviation_point(p.vertices + (uint64_t)id[0] * 3, p.vertices + (uint64_t)id[1] * 3, p.vertices + (uint64_t)id[2] * 3, p.ij[2 * s],
                    p.ij[2 * s + 1], p.k, x);
    pts[q * 3] = x[0];
    pts[q * 3 + 1] = x[1];
    pts[q * 3 + 2] = x[2];
}

// Per-triangle terms: triangle_max_abs, the largest |f| of the non-NaN values (-Inf without any) and the first slot that has
// it (0..2 corners, 3 + s sample s), the exact extremes, NaN samples, and area_t * mean_t and area_t -- zero for a triangle
// with a NaN value.  Not measured: NaN, -Inf, +Inf / -Inf extremes, zeros.
struct DeviationTerms {
    float *tmax, *best, *lo, *hi;
    double *areaMean, *area;
    uint8_t *nanSamples, *slot, *measured;
};

__global__ void __launch_bounds__(kThreads) k_deviation_triangles(const dcsg_deviation_params p, uint64_t first, uint64_t count,
                                                                  const float* __restrict__ vval, const float* __restrict__ vals,
                                                                  DeviationTerms d) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= count) return;
    const uint64_t t = first + i;
    const dcsg_inspect_triangle_sums s = InspectTriangleTerm{p.vertices, p.triangles}((long long)t);
    const bool measured = !s.degenerate && !s.nonfinite;
    float best = -INFINITY, lo = INFINITY, hi = -INFINITY;
    int slot = 0xff, nans = 0, nanSamples = 0;
    double sum = 0.0;
    if (measured) {
        const float corner[3] = {vval[p.triangles[t * 3]], vval[p.triangles[t * 3 + 1]], vval[p.triangles[t * 3 + 2]]};
        const float* v = vals + i * (uint64_t)p.samples;
        for (int n = 0; n < 3 + p.samples; ++n) {
            const float x = n < 3 ? corner[n] : v[n - 3];
            if (isnan(x)) {
                ++nans;
                nanSamples += n >= 3;
                continue;
            }
            const float ax = fabsf(x);
            if (ax > best) { best = ax; slot = n; }
            lo = min_total(lo, x);
            hi = max_total(hi, x);
            sum = sum + (double)ax;
        }
    }
    const bool clean = measured && !nans;
    d.tmax[t] = clean ? best : NAN;
    d.best[t] = best;
    d.lo[t] = lo;
    d.hi[t] = hi;
    d.areaMean[t] = clean ? s.area * (sum / (double)(3 + p.samples)) : 0.0;
    d.area[t] = clean ? s.area : 0.0;
    d.nanSamples[t] = (uint8_t)nanSamples;
    d.slot[t] = (uint8_t)slot;
    d.measured[t] = measured;
}

struct DeviationVertexSums {
    uint64_t measured, nan, values;
    float maxAbs;
    double sumSq;
};
struct DeviationVertexTerm {
    const float* v;
    const float* vval;
    const uint8_t* ref;
    __device__ DeviationVertexSums operator()(long long i) const {
        const bool m = ref[i] && isfinite(v[i * 3]) && isfinite(v[i * 3 + 1]) && isfinite(v[i * 3 + 2]);
        const float x = vval[i];
        const bool use = m && !isnan(x);
        return DeviationVertexSums{m, m && isnan(x), use, use ? fabsf(x) : -INFINITY, use ? (double)x * (double)x : 0.0};
    }
};
struct DeviationVertexSum {
    __device__ DeviationVertexSums operator()(const DeviationVertexSums& a, const DeviationVertexSums& b) const {
        return DeviationVertexSums{a.measured + b.measured, a.nan + b.nan, a.values + b.values, fmaxf(a.maxAbs, b.maxAbs), a.sumSq + b.sumSq};
    }
};

struct DeviationTriangleSums {
    uint64_t measured, nanSamples, over;
    float lo, hi, best;
    uint64_t bestTriangle;                      // the smallest t with this best; UINT64_MAX while best = -Inf
    double areaMean, area;
};
struct DeviationTriangleTerm {
    DeviationTerms d;
    float tolerance;
    __device__ DeviationTriangleSums operator()(long long t) const {
        const bool m = d.measured[t] != 0;
        const float tmax = d.tmax[t], best = d.best[t];
        return DeviationTriangleSums{m, d.nanSamples[t], m && !(tmax <= tolerance), d.lo[t], d.hi[t], best,
                                     best == -INFINITY ? ~0ull : (uint64_t)t, d.areaMean[t], d.area[t]};
    }
};
// every operation is exact or a sum; the argmax is a maximum over (best, -index), a total order: ties go to the lower index
struct DeviationTriangleSum {
    __device__ DeviationTriangleSums operator()(const DeviationTriangleSums& a, const DeviationTriangleSums& b) const {
        const bool takeB = b.best > a.best || (b.best == a.best && b.bestTriangle < a.bestTriangle);
        return DeviationTriangleSums{a.measured + b.measured, a.nanSamples + b.nanSamples, a.over + b.over, min_total(a.lo, b.lo),
                                     max_total(a.hi, b.hi), takeB ? b.best : a.best, takeB ? b.bestTriangle : a.bestTriangle,
                                     a.areaMean + b.areaMean, a.area + b.area};
    }
};

__global__ void k_deviation_finish(const dcsg_deviation_params p, const DeviationTerms d, const DeviationVertexSums* __restrict__ vs,
                                   const DeviationTriangleSums* __restrict__ ts) {
    dcsg_deviation_totals& o = *p.totals;
    o.measuredVertices = vs->measured;
    o.nanVertices = vs->nan;
    o.vertexValues = vs->values;
    o.vertexMaxAbs = vs->maxAbs;
    o.vertexSumSq = vs->sumSq;
    o.measuredTriangles = ts->measured;
    o.nanSamples = ts->nanSamples;
    o.overTolerance = ts->over;
    o.minSdf = ts->lo;
    o.maxSdf = ts->hi;
    o.maxAbs = ts->best;
    o.worstTriangle = ts->bestTriangle;
    o.sumAreaMean = ts->areaMean;
    o.sumArea = ts->area;
    float x[3] = {NAN, NAN, NAN};
    const uint64_t t = ts->bestTriangle;
    if (t != ~0ull) {
        const uint32_t* id = p.triangles + t * 3;
        const int slot = d.slot[t];
        if (slot < 3) {
            for (int c = 0; c < 3; ++c) x[c] = p.vertices[(uint64_t)id[slot] * 3 + c];
        } else {
            deviation_point(p.vertices + (uint64_t)id[0] * 3, p.vertices + (uint64_t)id[1] * 3, p.vertices + (uint64_t)id[2] * 3,
                            p.ij[2 * (slot - 3)], p.ij[2 * (slot - 3) + 1], p.k, x);
        }
    }
    for (int c = 0; c < 3; ++c) o.worstPoint[c] = x[c];
}

using DeviationVertexTerms = thrust::transform_iterator<DeviationVertexTerm, InspectCount>;
using DeviationTriangleTerms = thrust::transform_iterator<DeviationTriangleTerm, InspectCount>;

// Scratch of the deviation: the vertices' referenced marks and values, the per-triangle terms (35 B per triangle), one chunk's
// points and values, the id check's totals, the two reductions' results, then cub's temporary storage
struct DeviationLayout {
    size_t ref, vval, tmax, best, lo, hi, areaMean, area, nanSamples, slot, measured, pts, vals, check, vsum, tsum, temp, tempBytes, total;
    DeviationLayout(uint64_t nv, uint64_t nt, int samples) {
        auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const uint64_t chunk = dcsg_deviation_chunk(nt, samples) * (uint64_t)samples;
        size_t o = 0;
        ref = o; o += align(nv);
        vval = o; o += align(nv * 4);
        tmax = o; o += align(nt * 4);
        best = o; o += align(nt * 4);
        lo = o; o += align(nt * 4);
        hi = o; o += align(nt * 4);
        areaMean = o; o += align(nt * 8);
        area = o; o += align(nt * 8);
        nanSamples = o; o += align(nt);
        slot = o; o += align(nt);
        measured = o; o += align(nt);
        pts = o; o += align(chunk * 12);
        vals = o; o += align(chunk * 4);
        check = o; o += align(sizeof(dcsg_inspect_totals));
        vsum = o; o += align(sizeof(DeviationVertexSums));
        tsum = o; o += align(sizeof(DeviationTriangleSums));
        size_t a = 0, b = 0;
        cub::DeviceReduce::Reduce(nullptr, a, DeviationVertexTerms(InspectCount(0), DeviationVertexTerm{}), (DeviationVertexSums*)nullptr,
                                  (long long)nv, DeviationVertexSum(), DeviationVertexSums{});
        cub::DeviceReduce::Reduce(nullptr, b, DeviationTriangleTerms(InspectCount(0), DeviationTriangleTerm{}), (DeviationTriangleSums*)nullptr,
                                  (long long)nt, DeviationTriangleSum(), DeviationTriangleSums{});
        tempBytes = std::max(a, b);
        temp = o; o += align(tempBytes);
        total = o;
    }
    DeviationTerms terms(void* scratch) const {
        uint8_t* w = static_cast<uint8_t*>(scratch);
        return DeviationTerms{reinterpret_cast<float*>(w + tmax), reinterpret_cast<float*>(w + best), reinterpret_cast<float*>(w + lo),
                              reinterpret_cast<float*>(w + hi), reinterpret_cast<double*>(w + areaMean), reinterpret_cast<double*>(w + area),
                              w + nanSamples, w + slot, w + measured};
    }
};

}  // namespace

// persistent grids: `ctas` CTAs (the host passes a multiple of the SM count), never more than there can be tiles
static uint32_t grid_for(uint32_t maxEntries, int ctas) {
    const uint32_t tiles = (maxEntries + DCSG_TILE_WORDS - 1) / DCSG_TILE_WORDS;
    return tiles < (uint32_t)ctas ? (tiles ? tiles : 1u) : (uint32_t)ctas;
}
void dcsg_launch_classify(const dcsg_mesher_params& p, int ctas, cudaStream_t s) {
    if (p.numCellWords) k_classify<<<grid_for(p.numCellWords, ctas), kThreads, 0, s>>>(p);
}
void dcsg_launch_edges(const dcsg_mesher_params& p, int ctas, cudaStream_t s) {
    if (p.numVertWords) k_edges<<<grid_for(p.numVertWords, ctas), kThreads, 0, s>>>(p);
}
void dcsg_launch_scan_tiles(const dcsg_mesher_params& p, cudaStream_t s) { k_scan_tiles<<<3, 1024, 0, s>>>(p); }
void dcsg_launch_emit_vertices(const dcsg_mesher_params& p, int ctas, cudaStream_t s) {
    if (p.numVertWords) k_emit_vertices<<<grid_for(p.numVertWords, ctas), kThreads, 0, s>>>(p);
}
void dcsg_launch_emit_triangles(const dcsg_mesher_params& p, int ctas, cudaStream_t s) {
    if (p.numCellWords) k_emit_triangles<<<grid_for(p.numCellWords, ctas), kThreads, 0, s>>>(p);
}
void dcsg_launch_worklists(const dcsg_worklist_params& p, cudaStream_t s) {
    const uint32_t maskWords = (p.numBits + 31u) / 32u;
    const uint32_t tiles = (maskWords + kWorklistTile - 1) / kWorklistTile;
    if (!tiles) return;
    k_worklist_count<<<tiles, kThreads, 0, s>>>(p, tiles);
    k_worklist_fill<<<tiles, kThreads, 0, s>>>(p, tiles);
}
void dcsg_launch_cleanup(const dcsg_cleanup_params& p, int ctas, cudaStream_t s) { k_cleanup<<<ctas, kThreads, 0, s>>>(p); }
void dcsg_launch_format_stl(const float* v, const uint32_t* t, uint64_t n, uint8_t* out, bool acb, cudaStream_t s) {
    if (!n) return;
    if (acb) k_format_stl<true><<<blocks_for((n + 1) / 2, kThreads), kThreads, 0, s>>>(v, t, n, out);
    else k_format_stl<false><<<blocks_for((n + 1) / 2, kThreads), kThreads, 0, s>>>(v, t, n, out);
}
void dcsg_launch_format_ply_vertices(const float* v, const uint32_t* t, uint64_t n, double* out, cudaStream_t s) {
    if (n) k_format_ply_vertices<<<blocks_for(n * 3, kThreads), kThreads, 0, s>>>(v, t, n, out);
}
void dcsg_launch_format_ply_faces(uint64_t first, uint64_t n, uint8_t* out, cudaStream_t s) {
    if (n) k_format_ply_faces<<<blocks_for((n + 3) / 4, kThreads), kThreads, 0, s>>>(first, n, out);
}
void dcsg_launch_expand_soup(const float* v, const uint32_t* t, uint64_t n, float* out, cudaStream_t s) {
    if (n) k_expand_soup<<<blocks_for(n * 3, kThreads), kThreads, 0, s>>>(v, t, n, out);
}

void dcsg_launch_adapt_count(const dcsg_adapt_emit_params& p, cudaStream_t s) {
    if (p.numTiles) k_adapt_count<<<p.numTiles, kThreads, 0, s>>>(p);
}
void dcsg_launch_adapt_emit(const dcsg_adapt_emit_params& p, cudaStream_t s) {
    if (p.numTiles) k_adapt_emit<<<p.numTiles, kThreads, 0, s>>>(p);
}
void dcsg_launch_retopo_expand(const float* in, uint64_t numIn, uint32_t points, float* vertices, uint32_t* triangles, cudaStream_t s) {
    if (!numIn || points < 2) return;
    k_retopo_points<<<blocks_for(numIn * 3ull * points, kThreads), kThreads, 0, s>>>(in, numIn, points, vertices);
    k_retopo_triangles<<<blocks_for(numIn * (3ull * points - 2ull), kThreads), kThreads, 0, s>>>(numIn, points, triangles);
}
void dcsg_launch_rebase_indices(const uint32_t* in, uint64_t n, uint32_t base, uint32_t* out, int ctas, cudaStream_t s) {
    if (n) k_rebase_indices<<<ctas, kThreads, 0, s>>>(in, n, base, out);
}
void dcsg_launch_iota(uint32_t* out, uint64_t n, cudaStream_t s) {
    if (n) k_iota<<<blocks_for(n, kThreads), kThreads, 0, s>>>(out, n);
}
void dcsg_launch_surface_hist(const uint32_t* signbits, uint32_t* hist512, int ixBegin, int ixEnd, cudaStream_t s) {
    // 2048 words per ix column (256 iy x 8 words of 32 iz); the x-edges of column ix read column ix + 1
    if (ixEnd > ixBegin) k_surface_hist<<<(uint32_t)(ixEnd - ixBegin) * 2048u / kThreads, kThreads, 0, s>>>(signbits, hist512, (uint32_t)ixBegin * 2048u);
}
void dcsg_launch_format_ply_indexed_faces(const uint32_t* t, uint64_t n, uint32_t base, uint8_t* out, cudaStream_t s) {
    if (n) k_format_ply_indexed_faces<<<blocks_for((n + 3) / 4, kThreads), kThreads, 0, s>>>(t, n, base, out);
}
void dcsg_launch_format_ply_indexed_vertices(const float* v, const float* nrm, uint64_t n, float* out, cudaStream_t s) {
    if (n) k_format_ply_indexed_vertices<<<blocks_for(n, kThreads), kThreads, 0, s>>>(v, nrm, n, out);
}

size_t dcsg_weld_scratch_bytes(uint64_t n) { return WeldLayout(n).total; }

// LSD radix sort of (z, then x << 32 | y) with the input index as value: stable, so every run of equal positions is in
// ascending index order and starts with its smallest index.  Heads of runs -> the run's head for every vertex (max-scan of
// the heads' positions) -> new ids by an exclusive scan of the first occurrences in INPUT order.  Kernels and cub calls only:
// the output cannot depend on the schedule.
cudaError_t dcsg_launch_weld(const dcsg_weld_params& p, cudaStream_t s) {
    const uint64_t n = p.numVertices;
    if (!n) return cudaMemsetAsync(p.unique, 0, 4, s);
    const WeldLayout l(n);
    uint8_t* w = static_cast<uint8_t*>(p.scratch);
    uint64_t* xyA = reinterpret_cast<uint64_t*>(w + l.xyA);
    uint64_t* xyB = reinterpret_cast<uint64_t*>(w + l.xyB);
    uint32_t* zA = reinterpret_cast<uint32_t*>(xyA);            // the z pass runs before the x|y keys exist
    uint32_t* zB = reinterpret_cast<uint32_t*>(xyB);
    uint32_t* idxA = reinterpret_cast<uint32_t*>(w + l.idxA);
    uint32_t* idxB = reinterpret_cast<uint32_t*>(w + l.idxB);
    uint32_t* headPos = reinterpret_cast<uint32_t*>(w + l.headPos);
    uint32_t* runHead = reinterpret_cast<uint32_t*>(w + l.runHead);
    uint32_t* first = reinterpret_cast<uint32_t*>(w + l.first);
    uint32_t* newId = reinterpret_cast<uint32_t*>(w + l.newId);
    uint32_t* rep = reinterpret_cast<uint32_t*>(w + l.rep);
    void* temp = w + l.temp;
    size_t tempBytes = l.tempBytes;
    const long long items = (long long)n;
    const uint32_t blocks = blocks_for(n, kThreads);
    cudaError_t e;
    k_weld_init<<<blocks, kThreads, 0, s>>>(p.vertices, n, zA, idxA);
    if ((e = cub::DeviceRadixSort::SortPairs(temp, tempBytes, zA, zB, idxA, idxB, items, 0, 32, s)) != cudaSuccess) return e;
    k_weld_xy<<<blocks, kThreads, 0, s>>>(p.vertices, n, idxB, xyA);
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceRadixSort::SortPairs(temp, tempBytes, xyA, xyB, idxB, idxA, items, 0, 64, s)) != cudaSuccess) return e;
    k_weld_heads<<<blocks, kThreads, 0, s>>>(p.vertices, n, xyB, idxA, headPos, first);
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceScan::InclusiveScan(temp, tempBytes, headPos, runHead, WeldMax(), items, s)) != cudaSuccess) return e;
    k_weld_rep<<<blocks, kThreads, 0, s>>>(n, idxA, runHead, rep);
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceScan::ExclusiveSum(temp, tempBytes, first, newId, items, s)) != cudaSuccess) return e;
    k_weld_compact<<<blocks, kThreads, 0, s>>>(p.vertices, p.normals, n, first, newId, p.outVertices, p.outNormals, p.unique);
    if (p.numTriangles) k_weld_remap<<<blocks_for(p.numTriangles * 3, kThreads), kThreads, 0, s>>>(p.triangles, p.numTriangles * 3, rep, newId);
    return cudaGetLastError();
}

size_t dcsg_orient_scratch_bytes(uint64_t n) { return OrientLayout(n).total; }

cudaError_t dcsg_launch_orient(const dcsg_orient_params& p, cudaStream_t s) {
    const uint64_t n = p.numCells;
    if (!n) return cudaMemsetAsync(p.total, 0, 4, s);
    const OrientLayout l(n);
    uint8_t* w = static_cast<uint8_t*>(p.scratch);
    uint32_t* count = reinterpret_cast<uint32_t*>(w + l.count);
    uint32_t* first = reinterpret_cast<uint32_t*>(w + l.first);
    size_t tempBytes = l.tempBytes;
    const uint32_t blocks = blocks_for(n, kThreads);
    k_orient_count<<<blocks, kThreads, 0, s>>>(p.cellMasks, n, p.triCount, p.unit, count);
    cudaError_t e = cub::DeviceScan::ExclusiveSum(w + l.temp, tempBytes, count, first, (long long)n, s);
    if (e != cudaSuccess) return e;
    k_orient_apply<<<blocks, kThreads, 0, s>>>(p, first);
    return cudaGetLastError();
}

size_t dcsg_inspect_scratch_bytes(uint64_t nv, uint64_t nt) { return InspectLayout(nv, nt).total; }

cudaError_t dcsg_launch_inspect_check(const dcsg_inspect_params& p, cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(p.totals, 0, sizeof(dcsg_inspect_totals), s);
    if (e != cudaSuccess) return e;
    k_inspect_check<<<blocks_for(p.numTriangles * 3, kThreads), kThreads, 0, s>>>(p.triangles, p.numTriangles * 3, p.numVertices, &p.totals->badIds);
    return cudaGetLastError();
}

// Edges: the half-edge keys radix-sorted with their direction bits, then one reduction by key gives every edge's (k, f).
// Components: union-find over the non-degenerate triangles' ids, flattened to the smallest id, then the (label, triangle)
// pairs radix-sorted (stable: ascending triangles within a label) and summed by two segmented reductions (pieces, then the
// shells' runs of pieces).  Sums: cub reductions of the per-vertex, per-triangle and per-edge terms.  No floating-point atomics
// and no floating-point reduction by key: every result is the same bits on every run.
cudaError_t dcsg_launch_inspect(const dcsg_inspect_params& p, cudaStream_t s) {
    const uint64_t nv = p.numVertices, nt = p.numTriangles, nh = nt * 3;
    const InspectLayout l(nv, nt);
    uint8_t* w = static_cast<uint8_t*>(p.scratch);
    uint64_t* keysA = reinterpret_cast<uint64_t*>(w + l.keysA);
    uint64_t* keysB = reinterpret_cast<uint64_t*>(w + l.keysB);
    uint8_t* fwdA = w + l.fwdA;
    uint8_t* fwdB = w + l.fwdB;
    uint64_t* packed = reinterpret_cast<uint64_t*>(w + l.packed);
    uint32_t* parent = reinterpret_cast<uint32_t*>(w + l.parent);
    uint8_t* ref = w + l.ref;
    uint32_t* labelA = reinterpret_cast<uint32_t*>(w + l.labelA);
    uint32_t* labelB = reinterpret_cast<uint32_t*>(w + l.labelB);
    uint32_t* indexA = reinterpret_cast<uint32_t*>(w + l.indexA);
    uint32_t* indexB = reinterpret_cast<uint32_t*>(w + l.indexB);
    uint8_t* head = w + l.head;
    long long* pieceBegin = reinterpret_cast<long long*>(w + l.pieceBegin);
    long long* runBegin = reinterpret_cast<long long*>(w + l.runBegin);
    dcsg_inspect_component* partial = reinterpret_cast<dcsg_inspect_component*>(w + l.partial);
    uint64_t* runs = reinterpret_cast<uint64_t*>(w + l.runs);
    long long* counts = reinterpret_cast<long long*>(w + l.counts);        // {pieces, shell runs}
    void* temp = w + l.temp;
    size_t tempBytes;
    const long long hi = (long long)nh, ti = (long long)nt, vi = (long long)nv;
    const int vertexBits = bits_for(nv);
    cudaError_t e;
    k_inspect_init<<<blocks_for(nv, kThreads), kThreads, 0, s>>>(nv, parent, ref);
    k_inspect_triangles<<<blocks_for(nt, kThreads), kThreads, 0, s>>>(p.triangles, nt, keysA, fwdA, ref, parent);
    k_inspect_flatten<<<blocks_for(nv, kThreads), kThreads, 0, s>>>(nv, parent);
    k_inspect_labels<<<blocks_for(nt, kThreads), kThreads, 0, s>>>(p.triangles, nt, parent, labelA, indexA);
    // edges; the sorted keys' unique copies go to keysA, free after the sort
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceRadixSort::SortPairs(temp, tempBytes, keysA, keysB, fwdA, fwdB, hi, 0, 32 + vertexBits, s)) != cudaSuccess) return e;
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceReduce::ReduceByKey(temp, tempBytes, keysB, keysA, InspectHalfEdges(fwdB, InspectHalfEdge()), packed, runs, InspectAdd(),
                                            hi, s)) != cudaSuccess) return e;
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceReduce::Reduce(temp, tempBytes, thrust::make_transform_iterator(InspectCount(0), InspectEdgeTerm{keysA, packed, runs}),
                                       &p.totals->e, hi, InspectEdgeSum(), dcsg_inspect_edge_sums{}, s)) != cudaSuccess) return e;
    // components: pieces of the sorted sequence, then the shells' runs of pieces (the two counts are read back for the grids)
    const InspectTriangleTerm term{p.vertices, p.triangles};
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceRadixSort::SortPairs(temp, tempBytes, labelA, labelB, indexA, indexB, ti, 0, vertexBits, s)) != cudaSuccess) return e;
    k_inspect_piece_heads<<<blocks_for(nt, kThreads), kThreads, 0, s>>>(labelB, nt, head);
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceSelect::Flagged(temp, tempBytes, InspectCount(0), head, pieceBegin, counts, ti, s)) != cudaSuccess) return e;
    k_inspect_run_heads<<<blocks_for(nt, kThreads), kThreads, 0, s>>>(labelB, nt, pieceBegin, counts, head);
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceSelect::Flagged(temp, tempBytes, InspectCount(0), head, runBegin, counts + 1, ti, s)) != cudaSuccess) return e;
    long long h[2];
    if ((e = cudaMemcpyAsync(h, counts, sizeof(h), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
    if (h[0] > 0x7fffffffll) return cudaErrorInvalidValue;         // cub's segment counts are int
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceSegmentedReduce::Reduce(temp, tempBytes, InspectComponentTerms(indexB, InspectComponentTerm{term}), partial, (int)h[0],
                                                pieceBegin, InspectEnds(InspectCount(0), InspectSegmentEnd{pieceBegin, counts, ti}),
                                                InspectComponentSum(), dcsg_inspect_component{}, s)) != cudaSuccess) return e;
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceSegmentedReduce::Reduce(temp, tempBytes, (const dcsg_inspect_component*)partial, p.components, (int)h[1], runBegin,
                                                InspectEnds(InspectCount(0), InspectSegmentEnd{runBegin, counts + 1, h[0]}),
                                                InspectComponentSum(), dcsg_inspect_component{}, s)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(&p.totals->componentRuns, counts + 1, 8, cudaMemcpyDeviceToDevice, s)) != cudaSuccess) return e;
    // sums
    dcsg_inspect_vertex_sums v0 = {};
    for (int c = 0; c < 3; ++c) { v0.lo[c] = INFINITY; v0.hi[c] = -INFINITY; }
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceReduce::Reduce(temp, tempBytes, thrust::make_transform_iterator(InspectCount(0), InspectVertexTerm{p.vertices, ref, parent}),
                                       &p.totals->v, vi, InspectVertexSum(), v0, s)) != cudaSuccess) return e;
    tempBytes = l.tempBytes;
    if ((e = cub::DeviceReduce::Reduce(temp, tempBytes, thrust::make_transform_iterator(InspectCount(0), term), &p.totals->t, ti,
                                       InspectTriangleSum(), dcsg_inspect_triangle_sums{}, s)) != cudaSuccess) return e;
    return cudaGetLastError();
}

uint64_t dcsg_deviation_chunk(uint64_t nt, int samples) {
    return samples ? std::min<uint64_t>(nt, std::max<uint64_t>(1, kDeviationChunkSamples / (uint64_t)samples)) : nt;
}

size_t dcsg_deviation_scratch_bytes(uint64_t nv, uint64_t nt, int samples) { return DeviationLayout(nv, nt, samples).total; }

static uint8_t* deviation_at(const dcsg_deviation_params& p, size_t offset) { return static_cast<uint8_t*>(p.scratch) + offset; }
float* dcsg_deviation_vertex_values(const dcsg_deviation_params& p) {
    return reinterpret_cast<float*>(deviation_at(p, DeviationLayout(p.numVertices, p.numTriangles, p.samples).vval));
}
float* dcsg_deviation_points(const dcsg_deviation_params& p) {
    return reinterpret_cast<float*>(deviation_at(p, DeviationLayout(p.numVertices, p.numTriangles, p.samples).pts));
}
float* dcsg_deviation_values(const dcsg_deviation_params& p) {
    return reinterpret_cast<float*>(deviation_at(p, DeviationLayout(p.numVertices, p.numTriangles, p.samples).vals));
}
const float* dcsg_deviation_triangle_max_abs(const dcsg_deviation_params& p) {
    return reinterpret_cast<const float*>(deviation_at(p, DeviationLayout(p.numVertices, p.numTriangles, p.samples).tmax));
}

cudaError_t dcsg_launch_deviation_marks(const dcsg_deviation_params& p, cudaStream_t s) {
    uint8_t* ref = deviation_at(p, DeviationLayout(p.numVertices, p.numTriangles, p.samples).ref);
    cudaError_t e = cudaMemsetAsync(ref, 0, p.numVertices, s);
    if (e != cudaSuccess) return e;
    k_deviation_marks<<<blocks_for(p.numTriangles, kThreads), kThreads, 0, s>>>(p.triangles, p.numTriangles, ref);
    return cudaGetLastError();
}

cudaError_t dcsg_launch_deviation_points(const dcsg_deviation_params& p, uint64_t first, uint64_t count, cudaStream_t s) {
    if (!count || !p.samples) return cudaSuccess;
    k_deviation_points<<<blocks_for(count * (uint64_t)p.samples, kThreads), kThreads, 0, s>>>(p, first, count, dcsg_deviation_points(p));
    return cudaGetLastError();
}

cudaError_t dcsg_launch_deviation_triangles(const dcsg_deviation_params& p, uint64_t first, uint64_t count, cudaStream_t s) {
    if (!count) return cudaSuccess;
    const DeviationLayout l(p.numVertices, p.numTriangles, p.samples);
    k_deviation_triangles<<<blocks_for(count, kThreads), kThreads, 0, s>>>(p, first, count, reinterpret_cast<const float*>(deviation_at(p, l.vval)),
                                                                           reinterpret_cast<const float*>(deviation_at(p, l.vals)), l.terms(p.scratch));
    return cudaGetLastError();
}

// Two cub reductions in a fixed order (the vertices' terms, the triangles' terms), then one thread writes the totals and the
// worst point, recomputed from its slot by the points kernel's arithmetic.
cudaError_t dcsg_launch_deviation_totals(const dcsg_deviation_params& p, cudaStream_t s) {
    const DeviationLayout l(p.numVertices, p.numTriangles, p.samples);
    DeviationVertexSums* vs = reinterpret_cast<DeviationVertexSums*>(deviation_at(p, l.vsum));
    DeviationTriangleSums* ts = reinterpret_cast<DeviationTriangleSums*>(deviation_at(p, l.tsum));
    const DeviationTerms d = l.terms(p.scratch);
    size_t tempBytes = l.tempBytes;
    cudaError_t e;
    const DeviationVertexSums v0{0, 0, 0, -INFINITY, 0.0};
    if ((e = cub::DeviceReduce::Reduce(deviation_at(p, l.temp), tempBytes,
                                       DeviationVertexTerms(InspectCount(0), DeviationVertexTerm{p.vertices, reinterpret_cast<const float*>(deviation_at(p, l.vval)),
                                                                                                 deviation_at(p, l.ref)}),
                                       vs, (long long)p.numVertices, DeviationVertexSum(), v0, s)) != cudaSuccess) return e;
    tempBytes = l.tempBytes;
    const DeviationTriangleSums t0{0, 0, 0, INFINITY, -INFINITY, -INFINITY, ~0ull, 0.0, 0.0};
    if ((e = cub::DeviceReduce::Reduce(deviation_at(p, l.temp), tempBytes, DeviationTriangleTerms(InspectCount(0), DeviationTriangleTerm{d, p.tolerance}),
                                       ts, (long long)p.numTriangles, DeviationTriangleSum(), t0, s)) != cudaSuccess) return e;
    k_deviation_finish<<<1, 1, 0, s>>>(p, d, vs, ts);
    return cudaGetLastError();
}

// the id check of the deviation is the inspection's, on totals of its own in the deviation's scratch
dcsg_inspect_totals* dcsg_deviation_check_totals(const dcsg_deviation_params& p) {
    return reinterpret_cast<dcsg_inspect_totals*>(deviation_at(p, DeviationLayout(p.numVertices, p.numTriangles, p.samples).check));
}
