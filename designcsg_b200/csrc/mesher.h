// mesher.h -- host-callable launchers of the ahead-of-time compiled mesher kernels (mesher_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "mesher_bits.cuh"

// List entries (bitmap words) handled by one CTA tile.  A word holds up to 32 surface cells and a flat face of the design
// fills thousands of consecutive words completely, so large tiles differ in work by the factor 32 and the slowest SM of the
// emit kernels took 2.8 x the average (ncu, 1024 entries per tile); with one entry per thread the heavy tiles are short
// and spread over all CTAs.
#define DCSG_TILE_WORDS 256u

// The mesher kernels run over WORK LISTS: ascending indices of the bitmap words that can hold a surface cell (cell list) or
// own a mesh vertex (vertex list), one list entry per thread, DCSG_TILE_WORDS entries per CTA tile.  The sparse lattice pass
// produces the lists on the device (a few percent of the lattice's words); list == NULL means "every word" (dense lattice
// pass).  List lengths live in device memory, so the kernels are persistent: a fixed grid loops over the tiles.
//
// Ownership inside a z-slab: the slab is processed with one extra cell layer below and above it (where the lattice goes
// on), so that the vertices on its first and on the next slab's first sample plane are complete.  Cells of layers
// [ownCell0, ownCell1) are emitted; vertices of planes [ownVert0, ownVert1) are this slab's; those of plane ownVert1
// (haloVert = 1: the next slab's first plane) are numbered after them and stored as copies, so the slab's mesh is self
// contained AND its vertex ids plus the slab's global vertex offset are the ids of the whole mesh (no weld).
struct dcsg_mesher_params {
    dcsg_grid g;
    // inputs produced by the lattice kernel
    const uint32_t* sign;           // [nzp][planeWords]
    const uint32_t* leaf;           // [nzp][planeWords]
    dcsg_coarse coarse;
    uint32_t noCull;                // 1 = ignore the cull bits (clean, non-parity mode)
    const uint32_t* leafAlive;      // sparse path: cells surviving every cull of the walk (then leaf / coarse are unused)
    int ownCell0, ownCell1;         // local cell layers this slab emits
    int ownVert0, ownVert1;         // local sample planes whose vertices this slab owns
    int haloVert;                   // 1 = plane ownVert1 is numbered too (copies of the next slab's first vertices)
    // work lists
    const uint32_t* cellList;       // ascending cell-word indices, or NULL = all numCellWords words
    const uint32_t* cellCount;      // device: entries of cellList (NULL with cellList == NULL)
    const uint32_t* vertList;
    const uint32_t* vertCount;
    uint32_t numCellWords, numVertWords;
    uint32_t* aliveMask;            // sparse path: one bit per cell word, set where `alive` is not zero (NULL otherwise)
    uint32_t* aliveMask31;          // ... set where the word's last cell (bit 31) is alive
    // intermediates
    uint32_t* alive;                // [nzc][planeWords] surviving active cells
    uint4* vinfo;                   // [nzp][planeWords] {x-edge bits, y-edge bits, z-edge bits, first vertex id}; only list words are valid
    uint32_t* tileCells;            // per tile of the cell list: count, later exclusive prefix
    uint32_t* tileTris;
    uint32_t* tileVerts;            // per tile of the vertex list
    uint32_t* layerTris;            // [nzc] triangles per cell layer (zeroed by the host)
    uint32_t* planeVerts;           // [nzp] vertices per sample plane (zeroed by the host)
    uint32_t* totals;               // {cells, triangles, vertices incl. the halo plane's}
    // tables
    const float* px;
    const float* py;
    const float* pz;
    const uint8_t* triCount;        // [256]
    const int8_t* triTable;         // [256][16]
    // outputs (sized from totals)
    uint64_t* cellIds;              // x + N*(y + N*z), ascending
    uint8_t* cellMasks;
    uint32_t* triangles;            // 3 vertex ids per triangle, cell order then table order
    float* vertices;                // xyz per vertex, ascending key order
    uint64_t* vertexKeys;           // 3*(x + P*(y + P*z)) + axis
};

void dcsg_launch_classify(const dcsg_mesher_params& p, int ctas, cudaStream_t s);
void dcsg_launch_edges(const dcsg_mesher_params& p, int ctas, cudaStream_t s);
void dcsg_launch_scan_tiles(const dcsg_mesher_params& p, cudaStream_t s);
void dcsg_launch_emit_vertices(const dcsg_mesher_params& p, int ctas, cudaStream_t s);
void dcsg_launch_emit_triangles(const dcsg_mesher_params& p, int ctas, cudaStream_t s);

// Work lists from word masks (one bit per bitmap word, flat: bit zl * planeWords + w).  mode 0: listA = set bits of `mask`,
// listB = set bits of its dilation over the words at (x - {0,1}, y - {0,1}, z - {0,1}) -- the sample words that can hold a
// corner of an alive leaf (leaf pass -> classify, corner pass); mode 1: listB only (alive cell words -> vertex-owner words).
// Only a word's LAST cell reaches into the next word along x, hence the second mask.
// Ascending order; counts[0] / counts[1] receive the lengths.  scratch: 2 * tiles words.
struct dcsg_worklist_params {
    const uint32_t* mask;           // numBits bits, padded with one zero word
    const uint32_t* mask31;         // same layout: words whose bit 31 is set
    uint32_t numBits;               // words of the bitmaps = bits of the mask
    uint32_t rowWords, planeWords;
    int mode;
    uint32_t* listA;
    uint32_t* listB;
    uint32_t* counts;               // device: {len(listA), len(listB)}
    uint32_t* scratch;
};
void dcsg_launch_worklists(const dcsg_worklist_params& p, cudaStream_t s);

// End of a sparse extraction: zero again what it wrote into the all-zero bitmaps -- leafAlive and alive are only ever
// non-zero at the words of the cell list.
struct dcsg_cleanup_params {
    const uint32_t* cellList;
    const uint32_t* cellCount;
    uint32_t* leafAlive;
    uint32_t* alive;
};
void dcsg_launch_cleanup(const dcsg_cleanup_params& p, int ctas, cudaStream_t s);

// byte-exact file bodies built on the device (reference utils.hpp:41-154, happly.h:587-603).  acb: the records list the
// corners A, C, B (an outward-wound mesh: the STL's x z y axis order mirrors it, see dcsg_mesh_orient)
void dcsg_launch_format_stl(const float* vertices, const uint32_t* triangles, uint64_t numTriangles,
                            uint8_t* out /* 50 B per triangle */, bool acb, cudaStream_t s);
void dcsg_launch_format_ply_vertices(const float* vertices, const uint32_t* triangles, uint64_t numTriangles,
                                     double* out /* 9 doubles per triangle */, cudaStream_t s);
void dcsg_launch_format_ply_faces(uint64_t firstTriangle, uint64_t numTriangles,
                                  uint8_t* out /* 13 B per triangle */, cudaStream_t s);
// triangle soup (9 floats per triangle) from the indexed mesh
void dcsg_launch_expand_soup(const float* vertices, const uint32_t* triangles, uint64_t numTriangles,
                             float* out, cudaStream_t s);

// rows of the indexed binary PLY (dcsg_write_ply_indexed): face rows = the byte 3 and the triangle's vertex ids + base as
// little-endian uint32 (13 B); vertex rows with normals = x y z nx ny nz as float (24 B).  Without normals the vertex rows
// are the bytes of the vertex array itself.
void dcsg_launch_format_ply_indexed_faces(const uint32_t* triangles, uint64_t numTriangles, uint32_t base,
                                          uint8_t* out /* 13 B per triangle */, cudaStream_t s);
void dcsg_launch_format_ply_indexed_vertices(const float* vertices, const float* normals, uint64_t numVertices,
                                             float* out /* 6 floats per vertex */, cudaStream_t s);

// Weld: vertices whose three position words are bit-identical become one vertex, numbered in the order of the smallest input
// index among them.  The unique vertices (and normals, if any) are compacted into outVertices / outNormals, the triangles are
// renumbered in place, and *unique (device) receives the new vertex count.  Deterministic; n < 2^32.
struct dcsg_weld_params {
    const float* vertices;
    const float* normals;           // or NULL
    uint32_t* triangles;
    uint64_t numVertices, numTriangles;
    void* scratch;                  // dcsg_weld_scratch_bytes(numVertices) bytes of device memory
    float* outVertices;             // 3 floats per input vertex
    float* outNormals;              // idem, when normals != NULL
    uint32_t* unique;
};
size_t dcsg_weld_scratch_bytes(uint64_t numVertices);
cudaError_t dcsg_launch_weld(const dcsg_weld_params& p, cudaStream_t s);

// Outward winding (dcsg_mesh_orient): the triangles are cell i's table triangles in cell order, each one `unit` consecutive
// triangles (1, or the 3p - 2 of the strip cms::retopologize makes of it, which keeps its winding).  Bit t of triFlip[mask]
// marks table triangle t as inward-facing (tools/gen_mc_table.py); all `unit` triangles of a marked slot get their corners
// 1 and 2 swapped in place.  A pure map over (cell, slot, child): uniform lattices, z-slabs and the adaptive (level, node)
// order alike.  *total (device) receives the triangles the cells account for; the caller compares it with numTriangles.
struct dcsg_orient_params {
    const uint8_t* cellMasks;
    uint64_t numCells;
    const uint8_t* triCount;        // [256]
    const uint8_t* triFlip;         // [256]
    uint32_t unit;
    uint32_t* triangles;
    uint64_t numTriangles;          // triangles past this bound are never touched
    void* scratch;                  // dcsg_orient_scratch_bytes(numCells) bytes of device memory
    uint32_t* total;
};
size_t dcsg_orient_scratch_bytes(uint64_t numCells);
cudaError_t dcsg_launch_orient(const dcsg_orient_params& p, cudaStream_t s);

// ---- adaptive octree mode (mesher_kernels.cu "adaptive") ----------------------------------------------
struct dcsg_adapt_emit_params {
    dcsg_grid g;                    // the slab of sample planes the sign bitmap covers (z0 = its first plane)
    uint32_t* levelTris;            // [16] triangles per octree level (zeroed by the host), or NULL
    const uint32_t* sign;
    const uint32_t* emit;           // per-level node bitmaps, concatenated; level l starts at word levelOff[l]
    uint32_t levelOff[18];
    int minLevel, maxLevel;
    uint32_t firstWord, endWord;    // = levelOff[minLevel], levelOff[maxLevel + 1]
    uint32_t numTiles;
    uint32_t* tileCells;            // per tile: count, after dcsg_launch_scan_tiles the exclusive prefix
    uint32_t* tileTris;
    const float* px;
    const float* py;
    const float* pz;
    const uint8_t* triCount;
    const int8_t* triTable;
    float* soup;                    // 9 floats per triangle
    uint64_t* cellIds;              // level << 56 | nx + n*(ny + n*nz)
    uint8_t* cellMasks;
};
void dcsg_launch_adapt_count(const dcsg_adapt_emit_params& p, cudaStream_t s);
void dcsg_launch_adapt_emit(const dcsg_adapt_emit_params& p, cudaStream_t s);
// cms::retopologize as the reference build behaves: numIn triangles -> numIn * (3*points - 2) triangles
void dcsg_launch_retopo_expand(const float* in, uint64_t numIn, uint32_t points, float* vertices, uint32_t* triangles, cudaStream_t s);
void dcsg_launch_iota(uint32_t* out, uint64_t n, cudaStream_t s);
// out[i] = in[i] + base (multi-GPU: slab-local vertex ids -> ids of the whole mesh, stored to the gathering rank's array)
void dcsg_launch_rebase_indices(const uint32_t* in, uint64_t n, uint32_t base, uint32_t* out, int ctas, cudaStream_t s);
// per-z sign-change counts of the 256^3 search lattice (load balancing of z-slabs); hist512 must be zeroed
// (columns [ixBegin, ixEnd) of the search; needs the sign bits of column ixEnd too, unless ixEnd = 256)
void dcsg_launch_surface_hist(const uint32_t* signbits, uint32_t* hist512, int ixBegin, int ixEnd, cudaStream_t s);
