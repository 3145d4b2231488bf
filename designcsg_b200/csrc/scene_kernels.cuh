// scene_kernels.cuh -- hand-written CUDA kernels (sm_100a) that evaluate the compiled scene's SDF.
//
// Second part of the NVRTC translation unit (see scene_prelude.cuh for the layout).  Everything that
// needs the SDF inlined lives here; the bit-parallel mesher kernels that only read sign bits are
// compiled ahead of time (mesher_kernels.cu).  All kernels are compute bound on the FP32 pipe
// (DESIGN.md "Rooflines"): ~300-1100 float operations per sample against 0-4 bytes of HBM traffic.
//
// Replaces, in the reference: kernel k2 (master/k2.cl:234-280) and its per-block launches through
// Evaluator::eval_*_at_points (master/Evaluator.cpp:117-211); the 256^3 bounding-box loop
// (master/DesignCSG.cpp:668-712); the ISV3D64 block cache (master/ISV.hpp); the centre-sample cull
// of the octree walk (master/cms/main/Headers/mesh.hpp:164-170); and performGradientDescent
// (mesh.hpp:531-593).

// resident 256-thread blocks per SM the sparse lattice kernels (leaf, corners) are compiled for: they hand evaluations
// out lane by lane between stretches of bitmap work and live on occupancy (6 -> 40 registers, 5 -> 48)
#ifndef DCSG_SPARSE_MIN_BLOCKS
#define DCSG_SPARSE_MIN_BLOCKS 6
#endif

#ifndef DCSG_LATTICE_SPT
#define DCSG_LATTICE_SPT 4          // x-consecutive samples per thread in the lattice kernel (1, 2, 4, 8)
#endif


// ---------------------------------------------------------------------------------------------
// kernel entry, and the one way the kernels evaluate the scene: through the checked fast copy, again through the
// exact copy when the fast copy says its result may differ (scene_prelude.cuh "Two copies of the scene, one result").
// The exact copy sits behind a call that is not inlined: one instance per module, off the hot instruction stream.
// ---------------------------------------------------------------------------------------------
#ifndef DCSG_FAST_PATH
#define DCSG_FAST_PATH 0
#endif
DCSG_DEV void dcsg_enter() {
    dcsg_exact::dcsg_init_private();
#if DCSG_FAST_PATH
    dcsg_flag_init();
#endif
}
#if DCSG_FAST_PATH
__device__ __noinline__ float dcsg_sdf_exact_call(float x, float y, float z) { return dcsg_exact::dcsg_primary_sdf(float3(x, y, z)); }
DCSG_DEV float dcsg_sdf(float3 q) {
    bool inexact = false;
    float s = dcsg_fast::dcsg_primary_sdf(q, inexact);
    if (inexact | dcsg_flag_take()) s = dcsg_sdf_exact_call(q.x, q.y, q.z);
    return s;
}
#else
DCSG_DEV float dcsg_sdf(float3 q) { return dcsg_exact::dcsg_primary_sdf(q); }
#endif

// ---------------------------------------------------------------------------------------------
// normal + value at one point.  Reference get_normal (k2.cl:149-179): six taps at +-NORMAL_EPSILON
// (a double literal narrowed to float when the tap vectors are built), differences in float, the
// 1/(2e) scale in double (`1.0/twoE*Dx`), then normalize.  The seven evaluations (six taps and,
// optionally, the centre) run through the fast copy's per-axis straight-line forms where the scene's
// projection kernel fits their budget (compile_scene), else through ONE inlined copy of the SDF inside
// a rolled loop, which keeps the instruction footprint of heavy scenes inside the instruction cache.
// ---------------------------------------------------------------------------------------------
#ifndef DCSG_TAPS_SHARED
// 1 = dcsg_primary_sdf7: the seven evaluations as one straight-line function whose taps share the transform
// arithmetic (bit-identical, ~10 % fewer instructions on Design1); 0 = rolled loop over one inlined copy.
// Measured on B200 (round 1): 101 instead of 48 registers on Design1 (12.9 vs 12.7 ms, no gain) and 26.9 vs 21.6 ms
// on the Hilbert design (instruction footprint) -- so the loop stays the default; -DDCSG_TAPS_SHARED=1 through
// DCSG_NVRTC_EXTRA selects the other form (tests pass with either).
#define DCSG_TAPS_SHARED 0
#endif
#ifndef DCSG_TAP_AXES
// 1 = the fast copy's taps through the per-axis forms (dcsg_fast::dcsg_primary_sdf_x / _y / _z), chosen per scene by
// compile_scene; 0 = rolled loop over one inlined copy
#define DCSG_TAP_AXES 0
#endif
// Rolled tap loop without per-iteration selects: tap k is v + dcsg_tap_offset[k] and its value goes to a per-thread
// column of shared memory.  The reference builds the taps as v + (e,0,0), v - (e,0,0), ... (k2.cl:155-166); in IEEE
// arithmetic x - y == x + (-y) bit for bit, the untouched coordinates of a plus tap are v.c + 0.0f (as written there:
// -0 becomes +0) and those of a minus tap v.c - 0.0f == v.c + (-0.0f), which returns v.c unchanged (-0 included) --
// the centre row (-0,-0,-0) therefore reproduces v itself.
#define DCSG_TAP_E ((float)NORMAL_EPSILON)
__constant__ float dcsg_tap_offset[7][4] = {
    {DCSG_TAP_E, 0.0f, 0.0f, 0.0f},  {-DCSG_TAP_E, -0.0f, -0.0f, 0.0f}, {0.0f, DCSG_TAP_E, 0.0f, 0.0f}, {-0.0f, -DCSG_TAP_E, -0.0f, 0.0f},
    {0.0f, 0.0f, DCSG_TAP_E, 0.0f},  {-0.0f, -0.0f, -DCSG_TAP_E, 0.0f}, {-0.0f, -0.0f, -0.0f, 0.0f}};
__shared__ float dcsg_tap_value[7 * DCSG_BLOCK];
__shared__ unsigned dcsg_exact_rounds[DCSG_BLOCK];      // per thread: tap rounds evaluated a second time through the exact copy

// kMode 0: the checked fast copy, and where it says its result may differ, the exact copy right away (every caller but
// the projection); 1: the fast copy only -- `flagged` tells the caller that the values must not be used (the projection hands
// such a vertex to the warps of its exact phase instead of making this whole warp wait for the exact copy); 2: exact copy only.
template <bool kWithCentre, int kMode>
DCSG_DEV float3 dcsg_normal_and_sdf_mode(float3 v, float& centre, bool& flagged) {
    flagged = false;
    float f0 = 0.0f, f1 = 0.0f, f2 = 0.0f, f3 = 0.0f, f4 = 0.0f, f5 = 0.0f, f6 = 0.0f;
#if DCSG_TAPS_SHARED
    {
        float f[7];
        dcsg_exact::dcsg_primary_sdf7(v, DCSG_TAP_E, f);         // the centre's value is dead code when kWithCentre is false
        f0 = f[0]; f1 = f[1]; f2 = f[2]; f3 = f[3]; f4 = f[4]; f5 = f[5]; f6 = f[6];
    }
#elif DCSG_FAST_PATH && DCSG_TAP_AXES
    // The fast copy through the per-axis forms (host_scene.cu, generate_primary_sdf_axis): straight-line code in which the
    // taps of an axis share the unchanged coordinates' work, values in registers.  Their tests include every test of the
    // seven single evaluations, plus one the loop does not need (a coordinate of exactly +-0 or NaN).  So a flagged round
    // runs the rolled loop of the fast copy next, and only if that flags too does it go to the exact copy (mode 0) or
    // the caller (mode 1): a round is flagged exactly when the rolled loop would flag it, with the same values.
    {
        float* const mine = dcsg_tap_value + threadIdx.x;
        bool exact = kMode == 2;
        if (kMode != 2) {
            bool inexact = false;
            float tx[kWithCentre ? 3 : 2], ty[2], tz[2];
            if constexpr (kWithCentre) dcsg_fast::dcsg_primary_sdf_xc(v, DCSG_TAP_E, tx, inexact);
            else dcsg_fast::dcsg_primary_sdf_x(v, DCSG_TAP_E, tx, inexact);
            dcsg_fast::dcsg_primary_sdf_y(v, DCSG_TAP_E, ty, inexact);
            dcsg_fast::dcsg_primary_sdf_z(v, DCSG_TAP_E, tz, inexact);
            f0 = tx[0]; f1 = tx[1]; f2 = ty[0]; f3 = ty[1]; f4 = tz[0]; f5 = tz[1];
            if constexpr (kWithCentre) f6 = tx[2];
            if (inexact | dcsg_flag_take()) {                      // one test for the round
                bool again = false;
#pragma unroll 1
                for (int k = 0; k < (kWithCentre ? 7 : 6); ++k) {
                    const float3 q = float3(v.x + dcsg_tap_offset[k][0], v.y + dcsg_tap_offset[k][1], v.z + dcsg_tap_offset[k][2]);
                    mine[k * DCSG_BLOCK] = dcsg_fast::dcsg_primary_sdf(q, again);
                }
                if (again | dcsg_flag_take()) {
                    if (kMode == 1) {
                        flagged = true;
                    } else {                                       // all seven are evaluated again
                        dcsg_exact_rounds[threadIdx.x] += 1u;
                        exact = true;
                    }
                }
                if (!flagged && !exact) {
                    f0 = mine[0 * DCSG_BLOCK]; f1 = mine[1 * DCSG_BLOCK]; f2 = mine[2 * DCSG_BLOCK];
                    f3 = mine[3 * DCSG_BLOCK]; f4 = mine[4 * DCSG_BLOCK]; f5 = mine[5 * DCSG_BLOCK];
                    if (kWithCentre) f6 = mine[6 * DCSG_BLOCK];
                }
            }
        }
        if (exact) {
#pragma unroll 1
            for (int k = 0; k < (kWithCentre ? 7 : 6); ++k)
                mine[k * DCSG_BLOCK] = dcsg_sdf_exact_call(v.x + dcsg_tap_offset[k][0], v.y + dcsg_tap_offset[k][1], v.z + dcsg_tap_offset[k][2]);
            f0 = mine[0 * DCSG_BLOCK]; f1 = mine[1 * DCSG_BLOCK]; f2 = mine[2 * DCSG_BLOCK];
            f3 = mine[3 * DCSG_BLOCK]; f4 = mine[4 * DCSG_BLOCK]; f5 = mine[5 * DCSG_BLOCK];
            if (kWithCentre) f6 = mine[6 * DCSG_BLOCK];
        }
    }
#else
    {
        float* const mine = dcsg_tap_value + threadIdx.x;
#if DCSG_FAST_PATH
        if (kMode == 2) {
#pragma unroll 1
            for (int k = 0; k < (kWithCentre ? 7 : 6); ++k)
                mine[k * DCSG_BLOCK] = dcsg_sdf_exact_call(v.x + dcsg_tap_offset[k][0], v.y + dcsg_tap_offset[k][1], v.z + dcsg_tap_offset[k][2]);
        } else {
            bool inexact = false;
#pragma unroll 1
            for (int k = 0; k < (kWithCentre ? 7 : 6); ++k) {
                const float3 q = float3(v.x + dcsg_tap_offset[k][0], v.y + dcsg_tap_offset[k][1], v.z + dcsg_tap_offset[k][2]);
                mine[k * DCSG_BLOCK] = dcsg_fast::dcsg_primary_sdf(q, inexact);
            }
            if (inexact | dcsg_flag_take()) {                      // one test for the seven taps
                if (kMode == 1) {
                    flagged = true;
                } else {                                           // all seven are evaluated again
                    dcsg_exact_rounds[threadIdx.x] += 1u;
#pragma unroll 1
                    for (int k = 0; k < (kWithCentre ? 7 : 6); ++k)
                        mine[k * DCSG_BLOCK] = dcsg_sdf_exact_call(v.x + dcsg_tap_offset[k][0], v.y + dcsg_tap_offset[k][1], v.z + dcsg_tap_offset[k][2]);
                }
            }
        }
#else
#pragma unroll 1
        for (int k = 0; k < (kWithCentre ? 7 : 6); ++k) {
            const float3 q = float3(v.x + dcsg_tap_offset[k][0], v.y + dcsg_tap_offset[k][1], v.z + dcsg_tap_offset[k][2]);
            mine[k * DCSG_BLOCK] = dcsg_exact::dcsg_primary_sdf(q);
        }
#endif
        f0 = mine[0 * DCSG_BLOCK]; f1 = mine[1 * DCSG_BLOCK]; f2 = mine[2 * DCSG_BLOCK];
        f3 = mine[3 * DCSG_BLOCK]; f4 = mine[4 * DCSG_BLOCK]; f5 = mine[5 * DCSG_BLOCK];
        if (kWithCentre) f6 = mine[6 * DCSG_BLOCK];
    }
#endif
    centre = f6;
    const float Dx = f0 - f1;
    const float Dy = f2 - f3;
    const float Dz = f4 - f5;
    const float twoE = 2.0 * NORMAL_EPSILON;
    return dcsg_exact::normalize(float3(1.0 / twoE * Dx, 1.0 / twoE * Dy, 1.0 / twoE * Dz));
}

template <bool kWithCentre>
DCSG_DEV float3 dcsg_normal_and_sdf(float3 v, float& centre) {
    bool unused;
    return dcsg_normal_and_sdf_mode<kWithCentre, 0>(v, centre, unused);
}

// ---------------------------------------------------------------------------------------------
// point lists: the drop-in for Evaluator::eval_sdf_at_points / eval_normal_at_points.
// AoS (x,y,z) in, one float or AoS (nx,ny,nz) out -- the reference's buffer layout (k2.cl:263-277).
// ---------------------------------------------------------------------------------------------
extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_eval_sdf(const float* __restrict__ xyz, float* __restrict__ out, dcsg_u64 n) {
    dcsg_enter();
    const dcsg_u64 i = (dcsg_u64)blockIdx.x * DCSG_BLOCK + threadIdx.x;
    if (i >= n) return;
    out[i] = dcsg_sdf(float3(xyz[i * 3 + 0], xyz[i * 3 + 1], xyz[i * 3 + 2]));
}

extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_eval_normal(const float* __restrict__ xyz, float* __restrict__ out3, dcsg_u64 n) {
    dcsg_enter();
    const dcsg_u64 i = (dcsg_u64)blockIdx.x * DCSG_BLOCK + threadIdx.x;
    if (i >= n) return;
    float unused;
    const float3 nrm = dcsg_normal_and_sdf<false>(float3(xyz[i * 3 + 0], xyz[i * 3 + 1], xyz[i * 3 + 2]), unused);
    out3[i * 3 + 0] = nrm.x;
    out3[i * 3 + 1] = nrm.y;
    out3[i * 3 + 2] = nrm.z;
}

// How often does the checked fast copy fail its own test on this scene?  dcsg_build evaluates a sample of points with it:
// where the answer is "often" (a design whose brushes take sqrt(0) inside every box, say), every evaluation would run both
// copies, and the module is rebuilt with the exact copy alone.  Counts flagged evaluations; 0 in an exact-only module.
extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_flag_rate(const float* __restrict__ xyz, dcsg_u64 n, dcsg_u32* __restrict__ flagged) {
    dcsg_enter();
    const dcsg_u64 i = (dcsg_u64)blockIdx.x * DCSG_BLOCK + threadIdx.x;
    if (i >= n) return;
#if DCSG_FAST_PATH
    bool inexact = false;
    const float s = dcsg_fast::dcsg_primary_sdf(float3(xyz[i * 3 + 0], xyz[i * 3 + 1], xyz[i * 3 + 2]), inexact);
    (void)s;
    if (inexact | dcsg_flag_take()) atomicAdd(flagged, 1u);
#endif
}

// ---------------------------------------------------------------------------------------------
// bounding-box search (reference DesignCSG.cpp:668-712) fused with its reduction.
// 256^3 points p = (-c/2) + c*i, i in [-128,128) per axis; a point counts when sdf < c.  The
// reference then takes min / max of the coordinates of the counted points; coordinates are monotone
// in the index, so the kernel reduces the six extreme INDICES (block-level in shared memory, one
// global atomic per block and bound) and the host turns them back into coordinates.
// minmax = {minIx, minIy, minIz, maxIx, maxIy, maxIz}, pre-set to {INT_MAX.., INT_MIN..}.
// signbits (optional, 2^24 bits, one ballot word per warp = 32 consecutive iz): the sign of every search sample.
// A small follow-up kernel (k_surface_hist) counts the sign changes per z index -- the coarse analogue of the
// mesh's vertex count per layer -- to balance the z-slabs of a multi-GPU export (dcsg_plan_slabs).  It does not
// influence the result of the search.
// ---------------------------------------------------------------------------------------------
extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_bbox(float c, int* __restrict__ minmax, dcsg_u32* __restrict__ signbits, dcsg_u32 firstThread) {
    dcsg_enter();
    __shared__ int s_ext[6];
    if (threadIdx.x < 3) s_ext[threadIdx.x] = 0x7fffffff;
    else if (threadIdx.x < 6) s_ext[threadIdx.x] = (int)0x80000000;
    __syncthreads();
    // 2^24 threads for the whole search; a rank of a multi-GPU export takes the threads of its ix columns (ix = t >> 16)
    const dcsg_u32 t = firstThread + blockIdx.x * DCSG_BLOCK + threadIdx.x;
    const int iz = (int)(t & 255u) - 128;
    const int iy = (int)((t >> 8) & 255u) - 128;
    const int ix = (int)(t >> 16) - 128;
    const float h = -c / 2;
    const float s = dcsg_sdf(float3(h + c * (float)ix, h + c * (float)iy, h + c * (float)iz));
    const bool inside = s < c;
    if (signbits) {
        const unsigned negative = __ballot_sync(0xffffffffu, s < 0.0f);
        if ((threadIdx.x & 31u) == 0u) signbits[t >> 5] = negative;
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, inside);
    if (ballot) {
        // a warp covers 32 consecutive iz at fixed (ix, iy)
        const int lo = iz - (int)(threadIdx.x & 31u) + (__ffs(ballot) - 1);
        const int hi = iz - (int)(threadIdx.x & 31u) + (31 - __clz(ballot));
        if ((threadIdx.x & 31u) == 0) {
            atomicMin(&s_ext[0], ix); atomicMax(&s_ext[3], ix);
            atomicMin(&s_ext[1], iy); atomicMax(&s_ext[4], iy);
            atomicMin(&s_ext[2], lo); atomicMax(&s_ext[5], hi);
        }
    }
    __syncthreads();
    if (threadIdx.x < 3) { if (s_ext[threadIdx.x] != 0x7fffffff) atomicMin(&minmax[threadIdx.x], s_ext[threadIdx.x]); }
    else if (threadIdx.x < 6) { if (s_ext[threadIdx.x] != (int)0x80000000) atomicMax(&minmax[threadIdx.x], s_ext[threadIdx.x]); }
}

// ---------------------------------------------------------------------------------------------
// lattice kernel: the dense (N+1)^3 sample lattice of one z-slab.
//
// What the reference's mesher reads from the lattice is, per sample: the SIGN (corner masks,
// mesh.hpp:176-183) and the outcome of the centre-sample cull |s| > |halfDiameter|*1.1
// (mesh.hpp:164-170) for every octree node whose snapped centre is that sample.  The kernel
// therefore emits bitmaps and only optionally the fp32 values.  With lp = x + pitch*y the in-plane bit
// position (pitch = P rounded up to a multiple of 32, so rows start on word boundaries):
//   sign[zl][lp>>5]   bit lp&31 = s < 0
//   leaf[zl][lp>>5]   bit       = |s| > leafThr              -> leaf cell (x,y,z) culled
//   cfail[zl][lp>>5]  bit       = this sample is the centre of a coarser octree node AND that node
//                                 fails the cull.  Sample (x,y,z) is the centre of a level-(L-s) node
//                                 iff x, y and z all have the same lowest set bit 2^(s-1).
// Thread t of a plane owns the SPT x-consecutive samples lp = SPT*t .. SPT*t+SPT-1 of ONE row, so the
// y/z-dependent part of every object transform (dcsg_primary_sdf_row orders its terms x-last) is computed
// once per thread, and the index arithmetic once per SPT samples.  The 32/SPT lanes that share a bitmap
// word merge their SPT-bit fields with one warp reduction (REDUX.OR); every word is written exactly once:
// no atomics, no read-modify-write.
// ---------------------------------------------------------------------------------------------
// struct dcsg_lattice_params: see scene_params.h (shared with the host, embedded in front of this file)

extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_lattice(const dcsg_lattice_params p) {
    dcsg_enter();
    constexpr int kLanesPerWord = 32 / DCSG_LATTICE_SPT;
    const int lane = threadIdx.x & 31;
    const dcsg_u32 t = blockIdx.x * DCSG_BLOCK + threadIdx.x;          // group index inside the plane
    const dcsg_u32 groupsPerRow = (dcsg_u32)p.pitch / DCSG_LATTICE_SPT;
    const dcsg_u32 y = t / groupsPerRow;
    const dcsg_u32 x0 = (t - y * groupsPerRow) * DCSG_LATTICE_SPT;
    const int zl = blockIdx.y;
    const dcsg_u32 gz = (dcsg_u32)(p.z0 + zl);
    const bool rowValid = y < (dcsg_u32)p.P && x0 < (dcsg_u32)p.P;     // x0 >= P: padding group at the end of a row
    dcsg_u32 signBits = 0u, leafBits = 0u, failBits = 0u;
    if (rowValid) {
        const float vy = p.py[y];
        const float vz = p.pz[gz];
        // coarse node centres: x, y, z must share their lowest set bit; y and z decide it for the whole row
        const dcsg_u32 lowY = y & (0u - y), lowZ = gz & (0u - gz);
        const bool rowHasCentres = lowY == lowZ && lowY != 0u && lowY < (1u << p.L);
        const float rowThr = rowHasCentres ? p.coarseThr[p.L - __ffs(lowY)] : 0.0f;
        // straight-line on purpose (no per-sample branch): the SPT inlined evaluations then sit in one
        // basic block and the compiler shares their x-independent sub-expressions.  Padding samples
        // (x >= P, only at the end of a row; px is padded) are evaluated and masked out.
        // The dense kernel stays on the exact copy: its row form already shares the y/z part, and on a lattice centred
        // on the scene every row holds the sample x = 0 (and the padding samples), whose warps would fail the fast
        // copy's test and evaluate twice -- measured 9.9 ms against 9.6 ms at 1024^3.
        float sv[DCSG_LATTICE_SPT];
#pragma unroll
        for (int j = 0; j < DCSG_LATTICE_SPT; ++j) sv[j] = dcsg_exact::dcsg_primary_sdf_row(float3(p.px[x0 + j], vy, vz));
#pragma unroll
        for (int j = 0; j < DCSG_LATTICE_SPT; ++j) {
            const dcsg_u32 x = x0 + j;
            const bool valid = x < (dcsg_u32)p.P;
            const float s = sv[j];
            if (p.values && valid) p.values[((dcsg_u64)zl * p.P + y) * p.P + x] = s;
            const float mag = fabsf(s);
            signBits |= (valid && s < 0.0f ? 1u : 0u) << j;
            leafBits |= (valid && mag > p.leafThr ? 1u : 0u) << j;
            failBits |= (valid && rowHasCentres && (x & (0u - x)) == lowY && mag > rowThr ? 1u : 0u) << j;
        }
    }
    // the 32/SPT lanes sharing a word: field i of the word comes from lane (word_first_lane + i)
    const int field = (lane % kLanesPerWord) * DCSG_LATTICE_SPT;
    const dcsg_u32 peers = (kLanesPerWord == 32 ? 0xffffffffu : ((1u << kLanesPerWord) - 1u)) << (lane - lane % kLanesPerWord);
    const dcsg_u32 signWord = __reduce_or_sync(peers, signBits << field);
    const dcsg_u32 leafWord = __reduce_or_sync(peers, leafBits << field);
    const dcsg_u32 failWord = __reduce_or_sync(peers, failBits << field);
    const dcsg_u32 word = t / kLanesPerWord;
    if (lane % kLanesPerWord == 0 && word < p.planeWords) {
        const dcsg_u64 at = (dcsg_u64)zl * p.planeWords + word;
        p.sign[at] = signWord;
        p.leaf[at] = leafWord;
        p.cfail[at] = failWord;
    }
}

// ---------------------------------------------------------------------------------------------
// octree levels whose nodes are thicker than this rank's z-slab (multi-GPU only): their centres can lie
// on another rank's planes, so the few nodes touching the slab are evaluated here from a short
// host-built list of (x, y, z, level) lattice indices into small per-level node bitmaps.
// ---------------------------------------------------------------------------------------------
extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_coarse_nodes(const dcsg_lattice_params p, const int4* __restrict__ nodes, int n) {
    dcsg_enter();
    const int i = blockIdx.x * DCSG_BLOCK + threadIdx.x;
    if (i >= n) return;
    const int4 nd = nodes[i];
    const int lvl = nd.w;
    const int sh = p.L - lvl;
    const float s = dcsg_sdf(float3(p.px[nd.x], p.py[nd.y], p.pz[nd.z]));
    if (fabsf(s) > p.coarseThr[lvl]) {
        const dcsg_u32 node = ((dcsg_u32)nd.x >> sh) + (((dcsg_u32)nd.y >> sh) << lvl) + (((dcsg_u32)nd.z >> sh) << (2 * lvl));
        atomicOr(&p.coarse[p.coarseOff[lvl] + (node >> 5)], 1u << (node & 31u));
    }
}

// ---------------------------------------------------------------------------------------------
// descent: the octree-ordered (sparse) form of the lattice pass.
//
// The reference never samples inside a culled node: its walk (mesh.hpp:144-278) tests the centre of a
// node and drops the whole subtree when |s| > |halfDiameter|*1.1.  The dense kernel above evaluates
// every sample and lets classify apply the culls afterwards; this path applies them top-down and only
// evaluates what the walk would have touched, with the same arithmetic and therefore the same bits:
//   level l = 0 .. L-1 : candidates = children of the alive nodes of level l-1; evaluate the centre
//                        sample of each; alive_l = candidates that pass   (dcsg_k_descend: levels 0-3 sweep
//                        their whole bitmap; dcsg_k_descend_list: from level 4 on, the list of non-zero
//                        parent words the level above wrote)
//   leaves             : candidates = children of alive_(L-1); evaluate the min-corner sample (the
//                        leaf's snapped "centre"): leafAlive, its sign bit, and one mask bit per word
//                        that holds a candidate / an alive leaf                              (dcsg_k_leaf)
//   corners            : the other corners of alive leaves, over the list of sample words next to an
//                        alive leaf word (the mesher's work-list kernels build it from the masks)  (dcsg_k_corners)
// Everything stays word-parallel: one thread owns one 32-bit word of a level's bitmap (32 nodes along
// x), derives its candidate word from the parent's word by bit doubling, and the warp then hands the
// candidates out one per lane (same enumeration as the mesher's), so the SDF runs on full warps.
// Results return to the owning lane through shared memory; each bitmap word is written once, by its
// owner; the only global atomics set the mask bits.
// ---------------------------------------------------------------------------------------------
DCSG_DEV dcsg_u32 dcsg_popc32(dcsg_u32 v) { return (dcsg_u32)__popc(v); }

// 16 bits -> 32 bits, every bit doubled (parent node -> its two children along x)
DCSG_DEV dcsg_u32 dcsg_double_bits(dcsg_u32 v) {
    v &= 0xffffu;
    v = (v | (v << 8)) & 0x00ff00ffu;
    v = (v | (v << 4)) & 0x0f0f0f0fu;
    v = (v | (v << 2)) & 0x33333333u;
    v = (v | (v << 1)) & 0x55555555u;
    return v | (v << 1);
}

// hand the set bits of `bits` (one word per lane) out to the lanes of the warp, 32 per round;
// f(valid, ownerLane, bit) runs converged.  Returns the number of set bits in the warp.
// Every lane first lists its own set bits, as (lane << 5 | bit), in the warp's queue in shared memory at the position
// an exclusive scan of the counts gives it (a short divergent loop: one iteration per set bit of the fullest word);
// round r then is one load of entry 32 r + lane.  (The first form searched the scan for the owner of every entry
// and picked the bit with __fns: ~75 instructions per round against ~150 for a Design1 evaluation.)
__shared__ unsigned short dcsg_bit_queue[DCSG_BLOCK / 32][1024];
template <typename F>
DCSG_DEV dcsg_u32 dcsg_warp_for_each_bit(dcsg_u32 bits, F&& f) {
    const dcsg_u32 lane = threadIdx.x & 31u;
    const dcsg_u32 cnt = dcsg_popc32(bits);
    dcsg_u32 incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const dcsg_u32 o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= (dcsg_u32)d) incl += o;
    }
    const dcsg_u32 total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0u) return 0u;
    unsigned short* const queue = dcsg_bit_queue[threadIdx.x >> 5];
    {
        dcsg_u32 rest = bits, at = incl - cnt;
        while (rest) {
            queue[at++] = (unsigned short)((lane << 5) | (dcsg_u32)(__ffs((int)rest) - 1));
            rest &= rest - 1u;
        }
    }
    __syncwarp();
    for (dcsg_u32 base = 0; base < total; base += 32u) {
        const dcsg_u32 c = base + lane;
        const bool valid = c < total;
        const dcsg_u32 entry = valid ? (dcsg_u32)queue[c] : 0u;
        f(valid, (int)(entry >> 5), entry & 31u);
    }
    __syncwarp();                                       // the queue is free again
    return total;
}

DCSG_DEV void dcsg_count_evals(dcsg_u32 warpTotal, dcsg_u64* counter) {
    __shared__ dcsg_u32 s_total;
    if (!__syncthreads_or(warpTotal != 0u)) return;          // nothing evaluated in this CTA (the common case)
    if (threadIdx.x == 0) s_total = 0u;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && warpTotal) atomicAdd(&s_total, warpTotal);
    __syncthreads();
    if (threadIdx.x == 0 && s_total) atomicAdd(counter, (dcsg_u64)s_total);
}

// one word of the level's bitmap per thread (w: word index inside the slab's part of the level); called by whole CTAs.
// Returns the number of samples the warp evaluated.
DCSG_DEV dcsg_u32 dcsg_descend_word(const dcsg_descend_params& p, dcsg_u32 w) {
    __shared__ dcsg_u32 s_pass[DCSG_BLOCK];
    const int lvl = p.level;
    const dcsg_u32 n = 1u << lvl;
    const dcsg_u32 wordsPerRow = (n < 32u ? 32u : n) >> 5;
    const dcsg_u32 totalWords = wordsPerRow * n * (dcsg_u32)p.nzCount;
    const bool in = w < totalWords;
    dcsg_u32 xw = 0, ny = 0, nz = 0, cand = 0u;
    if (in) {
        xw = w % wordsPerRow;
        const dcsg_u32 rest = w / wordsPerRow;
        ny = rest % n;
        nz = (dcsg_u32)p.nzLo + rest / n;
        if (lvl == 0) {
            cand = 1u;                                  // the root
        } else {
            const dcsg_u32 pn = n >> 1;
            const dcsg_u32 pWordsPerRow = (pn < 32u ? 32u : pn) >> 5;
            const dcsg_u32 pw = p.parent[((dcsg_u64)(nz >> 1) * pn + (ny >> 1)) * pWordsPerRow + (xw >> 1)];
            cand = dcsg_double_bits(pw >> (16u * (xw & 1u)));
        }
    }
    s_pass[threadIdx.x] = 0u;
    __syncwarp();
    const int sh = p.L - lvl;                           // the node spans 2^sh cells; its centre is a lattice point
    const dcsg_u32 half = 1u << (sh - 1);
    const dcsg_u32 evals = dcsg_warp_for_each_bit(cand, [&](bool valid, int owner, dcsg_u32 bit) {
        const dcsg_u32 oxw = __shfl_sync(0xffffffffu, xw, owner);
        const dcsg_u32 ony = __shfl_sync(0xffffffffu, ny, owner);
        const dcsg_u32 onz = __shfl_sync(0xffffffffu, nz, owner);
        if (!valid) return;
        const dcsg_u32 nx = oxw * 32u + bit;
        const float s = dcsg_sdf(float3(p.px[(nx << sh) + half], p.py[(ony << sh) + half], p.pz[(onz << sh) + half]));
        if (!(fabsf(s) > p.thr)) atomicOr(&s_pass[(threadIdx.x & ~31) + owner], 1u << bit);
    });
    __syncwarp();
    const dcsg_u32 passed = s_pass[threadIdx.x];
    const dcsg_u32 at = (dcsg_u32)(((dcsg_u64)nz * n + ny) * wordsPerRow + xw);
    if (in) p.out[at] = passed;
    if (p.outList) {                                    // level L-1: the leaf pass works through the words with an alive node
        const unsigned has = __ballot_sync(0xffffffffu, in && passed != 0u);
        if (has) {
            const unsigned lane = threadIdx.x & 31u;
            dcsg_u32 base = 0u;
            if (lane == 0u) base = atomicAdd(p.outCount, (dcsg_u32)__popc(has));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (in && passed != 0u) p.outList[base + (dcsg_u32)__popc(has & ((1u << lane) - 1u))] = at;
        }
    }
    __syncwarp();
    return evals;
}

extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_descend(const dcsg_descend_params p) {
    dcsg_enter();
    dcsg_count_evals(dcsg_descend_word(p, blockIdx.x * DCSG_BLOCK + threadIdx.x), p.evalCount);
}

// List-driven levels.  From a few levels down, a level's bitmap is almost empty (the walk only reaches a band around the
// surface), so level l works through the LIST of level-(l-1) words that hold an alive node instead of sweeping its own
// bitmap.  A parent word is 32 nodes along x = 64 x 2 x 2 children = EIGHT child words (two along x, two rows, two
// planes), one per thread; a warp takes four parent words at a time, so nearly every lane brings candidates to the
// hand-out, and consecutive chunks go to different CTAs, which spreads short lists over the whole device.  Every child
// word has exactly one parent word: it is written once, by its owner, without atomics; words without a candidate are
// not touched at all (nobody reads them: the next level only follows the list).
struct dcsg_child_word { dcsg_u32 xw, y, z, cand; };

DCSG_DEV dcsg_child_word dcsg_child_of(const dcsg_u32* parentList, const dcsg_u32* parent, dcsg_u32 e, dcsg_u32 total, dcsg_u32 pn) {
    dcsg_child_word c;
    c.xw = c.y = c.z = c.cand = 0u;
    if (e >= total) return c;
    const dcsg_u32 child = threadIdx.x & 7u;
    const dcsg_u32 pWordsPerRow = (pn < 32u ? 32u : pn) >> 5;
    const dcsg_u32 pw = parentList[e];
    const dcsg_u32 pxw = pw % pWordsPerRow, rest = pw / pWordsPerRow;
    c.xw = 2u * pxw + (child & 1u);
    c.y = 2u * (rest % pn) + ((child >> 1) & 1u);
    c.z = 2u * (rest / pn) + (child >> 2);
    c.cand = dcsg_double_bits(parent[pw] >> (16u * (child & 1u)));
    return c;
}

// the chunks cta, cta + ctas, ... of the parent list; called by whole CTAs.  Returns the samples the warp evaluated.
DCSG_DEV dcsg_u32 dcsg_descend_chunks(const dcsg_descend_params& p, dcsg_u32 cta, dcsg_u32 ctas) {
    __shared__ dcsg_u32 s_pass[DCSG_BLOCK];
    __shared__ dcsg_u32 s_csign[DCSG_BLOCK];
    __shared__ dcsg_u32 s_calive[DCSG_BLOCK];
    const int lvl = p.level;
    const dcsg_u32 n = 1u << lvl;
    const dcsg_u32 wordsPerRow = (n < 32u ? 32u : n) >> 5;
    const dcsg_u32 total = *p.parentCount;
    const dcsg_u32 chunks = (total + 3u) >> 2;                      // four parent words per warp
    const bool record = p.centreSign != nullptr;                    // level L-1: the leaf pass reuses these samples
    const int sh = p.L - lvl;
    const dcsg_u32 half = 1u << (sh - 1);
    const dcsg_u32 lane = threadIdx.x & 31u;
    dcsg_u32 evals = 0u;
    for (dcsg_u32 chunk = cta + ctas * (threadIdx.x >> 5); chunk < chunks; chunk += ctas * (DCSG_BLOCK / 32)) {
        dcsg_child_word c = dcsg_child_of(p.parentList, p.parent, chunk * 4u + (lane >> 3), total, n >> 1);
        if (c.xw >= wordsPerRow || c.z < (dcsg_u32)p.nzLo || c.z >= (dcsg_u32)(p.nzLo + p.nzCount)) c.cand = 0u;
        s_pass[threadIdx.x] = 0u;
        if (record) { s_csign[threadIdx.x] = 0u; s_calive[threadIdx.x] = 0u; }
        __syncwarp();
        evals += dcsg_warp_for_each_bit(c.cand, [&](bool valid, int owner, dcsg_u32 bit) {
            const dcsg_u32 oxw = __shfl_sync(0xffffffffu, c.xw, owner);
            const dcsg_u32 oy = __shfl_sync(0xffffffffu, c.y, owner);
            const dcsg_u32 oz = __shfl_sync(0xffffffffu, c.z, owner);
            if (!valid) return;
            const dcsg_u32 nx = oxw * 32u + bit;
            const float s = dcsg_sdf(float3(p.px[(nx << sh) + half], p.py[(oy << sh) + half], p.pz[(oz << sh) + half]));
            const int slot = (threadIdx.x & ~31) + owner;
            if (!(fabsf(s) > p.thr)) {
                atomicOr(&s_pass[slot], 1u << bit);
                if (record) {
                    if (s < 0.0f) atomicOr(&s_csign[slot], 1u << bit);
                    if (!(fabsf(s) > p.leafThr)) atomicOr(&s_calive[slot], 1u << bit);
                }
            }
        });
        __syncwarp();
        const dcsg_u32 passed = c.cand ? s_pass[threadIdx.x] : 0u;
        const dcsg_u32 at = (dcsg_u32)(((dcsg_u64)c.z * n + c.y) * wordsPerRow + c.xw);
        if (c.cand) {
            p.out[at] = passed;
            if (record && passed) { p.centreSign[at] = s_csign[threadIdx.x]; p.centreAlive[at] = s_calive[threadIdx.x]; }
        }
        const unsigned has = __ballot_sync(0xffffffffu, passed != 0u);
        if (has) {
            dcsg_u32 base = 0u;
            if (lane == 0u) base = atomicAdd(p.outCount, (dcsg_u32)__popc(has));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (passed) p.outList[base + (dcsg_u32)__popc(has & ((1u << lane) - 1u))] = at;
        }
        __syncwarp();
    }
    return evals;
}

extern "C" __global__ void __launch_bounds__(DCSG_BLOCK, DCSG_SPARSE_MIN_BLOCKS)
dcsg_k_descend_list(const dcsg_descend_params p) {
    dcsg_enter();
    dcsg_count_evals(dcsg_descend_chunks(p, blockIdx.x, gridDim.x), p.evalCount);
}

// The top of the octree in ONE launch of ONE CTA: levels 0 .. count-1 hold a few thousand nodes between them, and as
// launches of their own each costs more latency than work (ten tiny launches are ~0.1 ms of an eight-GPU step).  The levels
// run one after the other through the same two functions -- sweeping levels first, list-driven ones after -- with a CTA
// barrier in between: a level reads its parent's bitmap, list and list length, all written by this CTA.
extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_descend_top(const dcsg_descend_top_params t) {
    dcsg_enter();
    dcsg_u32 evals = 0u;
    for (int i = 0; i < t.count; ++i) {
        const dcsg_descend_params& p = t.level[i];
        if (p.parentList) {
            evals += dcsg_descend_chunks(p, 0u, 1u);
        } else {
            const dcsg_u32 n = 1u << p.level;
            const dcsg_u32 totalWords = ((n < 32u ? 32u : n) >> 5) * n * (dcsg_u32)p.nzCount;
            for (dcsg_u32 base = 0u; base < totalWords; base += DCSG_BLOCK) evals += dcsg_descend_word(p, base + threadIdx.x);
        }
        __threadfence();
        __syncthreads();
    }
    dcsg_count_evals(evals, t.level[0].evalCount);
}


// Leaf pass: the same walk one level further down, where a node is a lattice cell and its snapped "centre" is the
// cell's min-corner sample: leafAlive, the sample's sign bit, and the mask of leaf words that are not zero.
extern "C" __global__ void __launch_bounds__(DCSG_BLOCK, DCSG_SPARSE_MIN_BLOCKS)
dcsg_k_leaf(const dcsg_leaf_params p) {
    dcsg_enter();
    __shared__ dcsg_u32 s_alive[DCSG_BLOCK];
    __shared__ dcsg_u32 s_sign[DCSG_BLOCK];
    const dcsg_u32 wordsPerRow = (dcsg_u32)p.pitch >> 5;
    const dcsg_u32 total = *p.parentCount;
    const dcsg_u32 chunks = (total + 3u) >> 2;
    const dcsg_u32 lane = threadIdx.x & 31u;
    dcsg_u32 evals = 0u;
    for (dcsg_u32 chunk = blockIdx.x + gridDim.x * (threadIdx.x >> 5); chunk < chunks; chunk += gridDim.x * (DCSG_BLOCK / 32)) {
        dcsg_child_word c = dcsg_child_of(p.parentList, p.parent, chunk * 4u + (lane >> 3), total, (dcsg_u32)p.N >> 1);
        const int zl = (int)c.z - p.z0;
        if (zl < 0 || zl >= p.nzc || c.y >= (dcsg_u32)p.N || c.xw >= wordsPerRow) c.cand = 0u;
        else {                                              // cells exist for x < N only
            const dcsg_u32 x0 = c.xw * 32u;
            if (x0 >= (dcsg_u32)p.N) c.cand = 0u;
            else if ((dcsg_u32)p.N - x0 < 32u) c.cand &= (1u << ((dcsg_u32)p.N - x0)) - 1u;
        }
        // child (1,1,1) of a node: its min corner is the node's centre, evaluated one level up -- the odd x positions of the
        // child words with odd y and z take their sign and cull verdict from there
        dcsg_u32 knownAlive = 0u, knownSign = 0u, todo = c.cand;
        if (p.centreSign && c.cand && (threadIdx.x & 6u) == 6u) {
            const dcsg_u32 pw = p.parentList[chunk * 4u + (lane >> 3)];
            const dcsg_u32 odd = c.cand & 0xaaaaaaaau;
            knownSign = dcsg_double_bits(p.centreSign[pw] >> (16u * (threadIdx.x & 1u))) & odd;
            knownAlive = dcsg_double_bits(p.centreAlive[pw] >> (16u * (threadIdx.x & 1u))) & odd;
            todo = c.cand & ~odd;
        }
        s_alive[threadIdx.x] = 0u;
        s_sign[threadIdx.x] = 0u;
        __syncwarp();
        evals += dcsg_warp_for_each_bit(todo, [&](bool valid, int owner, dcsg_u32 bit) {
            const dcsg_u32 oxw = __shfl_sync(0xffffffffu, c.xw, owner);
            const dcsg_u32 oy = __shfl_sync(0xffffffffu, c.y, owner);
            const dcsg_u32 oz = __shfl_sync(0xffffffffu, c.z, owner);
            if (!valid) return;
            const float s = dcsg_sdf(float3(p.px[oxw * 32u + bit], p.py[oy], p.pz[oz]));
            const int slot = (threadIdx.x & ~31) + owner;
            if (!(fabsf(s) > p.leafThr)) atomicOr(&s_alive[slot], 1u << bit);
            if (s < 0.0f) atomicOr(&s_sign[slot], 1u << bit);
        });
        __syncwarp();
        if (c.cand) {
            const dcsg_u64 at = (dcsg_u64)zl * p.planeWords + (dcsg_u64)c.y * wordsPerRow + c.xw;
            const dcsg_u32 alive = s_alive[threadIdx.x] | knownAlive;
            p.sign[at] = s_sign[threadIdx.x] | knownSign;
            atomicOr(&p.candMask[at >> 5], 1u << ((dcsg_u32)at & 31u));
            if (alive) {                                    // leafAlive is all-zero where nothing is alive: zero words are not written
                p.leafAlive[at] = alive;
                atomicOr(&p.leafMask[at >> 5], 1u << ((dcsg_u32)at & 31u));
                if (alive >> 31) atomicOr(&p.leafMask31[at >> 5], 1u << ((dcsg_u32)at & 31u));
            }
        }
        __syncwarp();
    }
    dcsg_count_evals(evals, p.evalCount);
}

// Corner pass: the corners of alive leaves that the leaf pass has not evaluated (it evaluated every candidate's min
// corner).  One thread per sample word of the corner list -- the words next to an alive leaf word (host: dilation of the
// leaf mask); a sample is needed when any of the cells at (x - {0,1}, y - {0,1}, z - {0,1}) is alive.  Which samples the
// leaf pass evaluated follows from the parent bitmap again (the candidates of the word).  A sign word without any
// candidate (candMask) was not written by the leaf pass of THIS extraction: its old content is stale and is replaced, not
// merged.
extern "C" __global__ void __launch_bounds__(DCSG_BLOCK, DCSG_SPARSE_MIN_BLOCKS)
dcsg_k_corners(const dcsg_leaf_params p) {
    dcsg_enter();
    __shared__ dcsg_u32 s_sign[DCSG_BLOCK];
    const dcsg_u32 wordsPerRow = (dcsg_u32)p.pitch >> 5;
    const dcsg_u32 pn = (dcsg_u32)p.N >> 1;
    const dcsg_u32 pWordsPerRow = (pn < 32u ? 32u : pn) >> 5;
    const dcsg_u32 total = *p.cornerCount;
    const dcsg_u32 tiles = (total + DCSG_BLOCK - 1u) / DCSG_BLOCK;
    dcsg_u32 evals = 0u;
    for (dcsg_u32 tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const dcsg_u32 i = tile * DCSG_BLOCK + threadIdx.x;
        dcsg_u32 xw = 0, y = 0, gz = 0, todo = 0u, seen = 0u;
        dcsg_u64 at = 0;
        if (i < total) {
            at = p.cornerList[i];
            const int zl = (int)(at / p.planeWords);
            const dcsg_u32 w = (dcsg_u32)(at - (dcsg_u64)zl * p.planeWords);
            y = w / wordsPerRow;
            xw = w - y * wordsPerRow;
            gz = (dcsg_u32)(p.z0 + zl);
            if (y < (dcsg_u32)p.P && zl < p.nzp) {
                dcsg_u32 need = 0u;
#pragma unroll
                for (int dz = 0; dz < 2; ++dz) {
                    const int pl = zl - dz;
                    if (pl < 0 || pl >= p.nzc) continue;
#pragma unroll
                    for (int dy = 0; dy < 2; ++dy) {
                        if ((int)y - dy < 0) continue;
                        const dcsg_u32* row = p.leafAlive + (dcsg_u64)pl * p.planeWords + (dcsg_u64)(y - dy) * wordsPerRow;
                        const dcsg_u32 a = row[xw];
                        const dcsg_u32 carry = xw ? (row[xw - 1] >> 31) : 0u;
                        need |= a | (a << 1) | carry;
                    }
                }
                // the leaf pass's candidates of this word (candMask says whether it had any -- only then its parent word
                // is a word the level above wrote in this extraction)
                if (need && ((p.candMask[at >> 5] >> ((dcsg_u32)at & 31u)) & 1u)) {
                    const dcsg_u32 pw = p.parent[((dcsg_u64)(gz >> 1) * pn + (y >> 1)) * pWordsPerRow + (xw >> 1)];
                    seen = dcsg_double_bits(pw >> (16u * (xw & 1u)));
                    const dcsg_u32 x0 = xw * 32u;
                    if (x0 >= (dcsg_u32)p.N) seen = 0u;
                    else if ((dcsg_u32)p.N - x0 < 32u) seen &= (1u << ((dcsg_u32)p.N - x0)) - 1u;
                }
                todo = need & ~seen;
            }
        }
        s_sign[threadIdx.x] = 0u;
        __syncwarp();
        evals += dcsg_warp_for_each_bit(todo, [&](bool valid, int owner, dcsg_u32 bit) {
            const dcsg_u32 oxw = __shfl_sync(0xffffffffu, xw, owner);
            const dcsg_u32 oy = __shfl_sync(0xffffffffu, y, owner);
            const dcsg_u32 oz = __shfl_sync(0xffffffffu, gz, owner);
            if (!valid) return;
            const float s = dcsg_sdf(float3(p.px[oxw * 32u + bit], p.py[oy], p.pz[oz]));
            if (s < 0.0f) atomicOr(&s_sign[(threadIdx.x & ~31) + owner], 1u << bit);
        });
        __syncwarp();
        if (todo) p.sign[at] = ((seen ? p.sign[at] : 0u) & ~todo) | s_sign[threadIdx.x];
        __syncwarp();
    }
    dcsg_count_evals(evals, p.evalCount);
}

// ---------------------------------------------------------------------------------------------
// projection: all gradient-descent steps of one vertex in registers (reference mesh.hpp:531-593):
//   per step  s = sdf(p), n = get_normal(p)  (both at the pre-step position),  p = p + n*(-s)
// and, when asked, the final 6-tap normal ("with normals" configs).  One UNIQUE vertex per lane at a time:
// the reference walks the triangle soup, but duplicated soup vertices are bit-identical inputs and
// therefore produce bit-identical outputs.
//
// Vertices leave the loop at different steps.  A cycle of the (deterministic) update is detected and its whole periods are
// skipped (detectCycles, see below: exact for scenes whose SDF is a pure function of the point).  A step that does not change a single bit is a fixed point of the
// (deterministic) update, all remaining steps would reproduce it, so stopping there gives the reference's result
// exactly (a third of Design1's vertices get there before step 50); and a vertex whose normal degenerated (six
// equal taps -> 0/0) sits at NaN IN ALL THREE coordinates and stays there whatever the SDF returns (NaN + x = NaN) -- it is
// final too, and not evaluating brushes at NaN also keeps user code that indexes tables by position from reading out of
// bounds (the reference has that hazard on its OpenCL device).  A position with only some NaN coordinates keeps stepping
// like the reference's: T_min / T_max are ternaries that can drop a NaN operand, so its other coordinates may still move.  With one vertex per thread for the whole kernel those lanes
// idle until the slowest vertex of their warp is through (14 % of the lane-cycles on Design1).  So the warps are
// persistent and every lane keeps its own step counter: a lane whose vertex is final takes the next one from the
// warp's batch (32 consecutive indices, handed out by `cursor`, which the host zeroes before the launch) while
// its neighbours carry on; the SDF is always evaluated by the whole warp, each lane at its own vertex and step.
// The final normal of the "with normals" configurations is one more round of the same seven taps.  Every vertex
// is read and written by exactly one lane, so the result does not depend on the schedule.
// ---------------------------------------------------------------------------------------------
// gatherVerts / gatherNormals (multi-GPU, optional): the first gatherCount vertices -- the slab's own -- are also stored to the
// gathering rank's arrays (peer memory over NVLink, already offset to this slab's first vertex), so the whole mesh is
// complete on that rank when the ranks' kernels are, without a copy afterwards.
// stats (optional): [0] += tap rounds executed (7 SDF evaluations each, 6 for a final normal), [1] += rounds evaluated through
// the exact copy -- what bench.py derives the executed-operation rate from.
//
// Two phases.  A vertex on which the checked fast copy fails its test (exactly on a centre plane of a symmetric scene: it
// fails at EVERY step) would make its whole warp run the exact copy as well, 31 lanes waiting: 0.26 % of Design1's tap
// rounds cost ~5 % of the kernel that way.  So phase 1 runs the fast copy only; a lane whose round is flagged writes its
// vertex back, appends (vertex, steps done) to a device-wide list and takes the next vertex.  A warp that finds the cursor
// drained moves on to phase 2: the same loop over the entries of that list, exact copy only, 32 flagged vertices per warp.
// Every warp passes through phase 2 after its own phase 1, so every entry is taken by its producer at the latest; the
// early finishers take most of them while the others are still draining phase 1.
struct dcsg_project_args {
    float* verts;
    dcsg_u64 n;
    int steps;
    float* normals;
    dcsg_u64* cursor;               // [0] phase-1 cursor, [1] entries appended to the list, [2] entries claimed from it
    float* gatherVerts;
    float* gatherNormals;
    dcsg_u64 gatherCount;
    dcsg_u64* deferred;             // the list: vertex | (steps done + 1) << 40; zero = not written yet (the host clears it)
    int detectCycles;
};

template <bool kExactPhase>
DCSG_DEV void dcsg_project_phase(const dcsg_project_args& a, unsigned& rounds) {
    const unsigned full = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned below = (1u << lane) - 1u;
    dcsg_u64 next = 0, end = 0;             // the warp's batch: vertex indices (phase 1) / list entries (phase 2), warp-uniform
    bool drained = false;                   // nothing left to fetch (warp-uniform)
    bool active = false;                    // this lane holds a vertex that is not final
    dcsg_u64 idx = 0;
    int step = 0;                           // steps done; == steps: only the final normal is left
    const int steps = a.steps;
    float3 pos = float3(0.0f, 0.0f, 0.0f);
    float3 mark = float3(0.0f, 0.0f, 0.0f); // Brent's cycle detection: the position after `markStep` steps (a power of two)
    int markStep = -1;
    for (;;) {
        unsigned need = __ballot_sync(full, !active);
        while (need) {
            if (next == end) {
                if (drained) break;
                dcsg_u64 first = 0, count = 0;
                if (lane == 0u) {
                    if (!kExactPhase) {
                        first = atomicAdd(&a.cursor[0], (dcsg_u64)32);
                        count = first < a.n ? (first + 32u < a.n ? 32u : a.n - first) : 0u;
                    } else {            // claim entries that exist NOW; later ones are taken by the warps that append them
                        for (;;) {
                            const dcsg_u64 taken = *(volatile dcsg_u64*)&a.cursor[2], there = *(volatile dcsg_u64*)&a.cursor[1];
                            if (taken >= there) { first = taken; count = 0; break; }
                            count = there - taken < 32u ? there - taken : 32u;
                            if (atomicCAS(&a.cursor[2], taken, taken + count) == taken) { first = taken; break; }
                        }
                    }
                }
                first = __shfl_sync(full, first, 0);
                count = __shfl_sync(full, count, 0);
                next = first;
                end = first + count;
                if (next == end) { drained = true; break; }
            }
            const unsigned left = (unsigned)(end - next);
            const unsigned wanted = (unsigned)__popc(need);
            const unsigned rank = (unsigned)__popc(need & below);
            if (!active && rank < left) {
                if (!kExactPhase) {
                    idx = next + rank;
                    step = 0;
                } else {
                    dcsg_u64 entry;
                    do { entry = *(volatile dcsg_u64*)&a.deferred[next + rank]; } while (entry == 0ull);    // reserved, about to be written
                    idx = entry & 0xffffffffffull;
                    step = (int)(entry >> 40) - 1;
                }
                // (through L2: in phase 2 the position was written by another SM, and this SM's L1 may still hold the line
                // from the time it loaded a neighbouring vertex)
                pos = float3(__ldcg(&a.verts[idx * 3 + 0]), __ldcg(&a.verts[idx * 3 + 1]), __ldcg(&a.verts[idx * 3 + 2]));
                if (pos.x != pos.x && pos.y != pos.y && pos.z != pos.z) step = steps;
                markStep = -1;
                active = step < steps || a.normals != nullptr;     // otherwise final as loaded: nothing to store
                if (!active && a.gatherVerts && idx < a.gatherCount) {
                    a.gatherVerts[idx * 3 + 0] = pos.x;
                    a.gatherVerts[idx * 3 + 1] = pos.y;
                    a.gatherVerts[idx * 3 + 2] = pos.z;
                }
            }
            next += wanted < left ? wanted : left;
            need = __ballot_sync(full, !active);
        }
        if (__ballot_sync(full, active) == 0u) break;               // nothing in flight, nothing left to fetch
        if (active) {
            float s;
            bool flagged;
            const float3 nrm = dcsg_normal_and_sdf_mode<true, kExactPhase ? 2 : 1>(pos, s, flagged);
            ++rounds;
            if (flagged) {
                // phase 1 only: this vertex goes on through the exact copy.  Its position so far returns to the array
                // (positions are only ever touched by the lane that holds the vertex), the entry is published last.
                a.verts[idx * 3 + 0] = pos.x;
                a.verts[idx * 3 + 1] = pos.y;
                a.verts[idx * 3 + 2] = pos.z;
                __threadfence();
                const dcsg_u64 at = atomicAdd(&a.cursor[1], (dcsg_u64)1);
                a.deferred[at] = idx | ((dcsg_u64)(step + 1) << 40);
                active = false;
            } else if (step < steps) {
                const float m = -s;
                const float3 moved = float3(pos.x + m * nrm.x, pos.y + m * nrm.y, pos.z + m * nrm.z);
                const bool fixed = __float_as_uint(moved.x) == __float_as_uint(pos.x) &&
                                   __float_as_uint(moved.y) == __float_as_uint(pos.y) &&
                                   __float_as_uint(moved.z) == __float_as_uint(pos.z);
                pos = moved;
                step = (fixed || (pos.x != pos.x && pos.y != pos.y && pos.z != pos.z)) ? steps : step + 1;
                if (a.detectCycles && step < steps) {
                    // The update is a pure function of the position, so a position seen before closes a cycle: if the
                    // position after `step` steps equals the one after `markStep`, the sequence has period
                    // L = step - markStep from there on, and the position after all `steps` steps is the one
                    // (steps - step) mod L steps ahead -- skip the whole periods.  (Vertices of steep SDFs end up hopping
                    // between two or a few positions one ulp apart long before step 50.)  Brent's scheme: the mark
                    // moves to every power-of-two step, which bounds the detection by about twice the longer of the
                    // transient and the period.
                    if (markStep >= 0 && __float_as_uint(pos.x) == __float_as_uint(mark.x) && __float_as_uint(pos.y) == __float_as_uint(mark.y) &&
                        __float_as_uint(pos.z) == __float_as_uint(mark.z)) {
                        const int period = step - markStep;
                        step = steps - (steps - step) % period;
                        markStep = -1;                              // fewer than `period` steps are left: no second jump
                    } else if ((step & (step - 1)) == 0) {
                        mark = pos;
                        markStep = step;
                    }
                }
                if (step == steps) {
                    a.verts[idx * 3 + 0] = pos.x;
                    a.verts[idx * 3 + 1] = pos.y;
                    a.verts[idx * 3 + 2] = pos.z;
                    if (a.gatherVerts && idx < a.gatherCount) {
                        a.gatherVerts[idx * 3 + 0] = pos.x;
                        a.gatherVerts[idx * 3 + 1] = pos.y;
                        a.gatherVerts[idx * 3 + 2] = pos.z;
                    }
                    active = a.normals != nullptr;
                }
            } else {
                a.normals[idx * 3 + 0] = nrm.x;
                a.normals[idx * 3 + 1] = nrm.y;
                a.normals[idx * 3 + 2] = nrm.z;
                if (a.gatherNormals && idx < a.gatherCount) {
                    a.gatherNormals[idx * 3 + 0] = nrm.x;
                    a.gatherNormals[idx * 3 + 1] = nrm.y;
                    a.gatherNormals[idx * 3 + 2] = nrm.z;
                }
                active = false;
            }
        }
    }
}

// the per-axis form holds a tap round's values in registers: at most 64 of them, four resident blocks per SM (compile_scene
// checks the result and keeps the rolled loop for a scene whose kernel does not fit)
#if DCSG_FAST_PATH && DCSG_TAP_AXES
#define DCSG_PROJECT_BOUNDS __launch_bounds__(DCSG_BLOCK, 4)
#else
#define DCSG_PROJECT_BOUNDS __launch_bounds__(DCSG_BLOCK)
#endif
extern "C" __global__ void DCSG_PROJECT_BOUNDS
dcsg_k_project(const dcsg_project_args a, dcsg_u64* __restrict__ stats) {
    dcsg_enter();
    const unsigned lane = threadIdx.x & 31u;
    unsigned rounds = 0u, exactRounds = 0u;
#if DCSG_FAST_PATH
    dcsg_project_phase<false>(a, rounds);
    dcsg_project_phase<true>(a, exactRounds);
#else
    dcsg_project_phase<false>(a, exactRounds);      // an exact-only module: one phase, nothing is ever flagged
#endif
    if (stats) {
        const unsigned warpRounds = __reduce_add_sync(0xffffffffu, rounds + exactRounds);
        const unsigned warpExact = __reduce_add_sync(0xffffffffu, exactRounds);
        if (lane == 0u) {
            if (warpRounds) atomicAdd(&stats[0], (dcsg_u64)warpRounds);
            if (warpExact) atomicAdd(&stats[1], (dcsg_u64)warpExact);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// adaptive octree mode: the reference's subdivision criteria (mesh.hpp:212-267), one launch per level.
//
// With min < max the walk stops early where the surface is simple.  A node of level l that survives
// the centre cull (mesh.hpp:164-170)
//   l <  min : always subdivides;
//   l == max : is a leaf;
//   otherwise subdivides when (a) any INTERIOR lattice sample of any of its 12 edges is inside
//   ("edge ambiguity", :221-238) or (b) the 6-tap normals at the two ends of any edge differ by more
//   than complexSurfaceThreshold ("complex edge", :244-258, angleBetweenVectors geometry.hpp:118-124);
//   else it is a leaf.
// Leaves emit lookupTable[mask] on the midpoints of THEIR edges (big triangles at coarse levels).
// All samples are lattice samples, so (a) and the corner masks read the dense sign bitmap of
// dcsg_k_lattice; the edge samples are start + delta*(i/points) in float, then truncated onto the
// lattice by ISV3D64::getCoords -- which lattice index that is comes from a host-built table
// (`snap`, same float arithmetic), because the rounded sample can fall just below its nominal point.
// (b) needs normals at the node corners: 8 x 6 SDF evaluations per undecided node, done here.
// One thread owns one word (32 nodes along x) of the level's bitmaps; candidates (children of the
// nodes that split one level up) are handed out one per lane, twice: first the bit logic, then the
// normal test for the nodes the bits did not decide.
// ---------------------------------------------------------------------------------------------

// glibc 2.39 acosf (sysdeps/ieee754/flt-32/e_acosf.c, the fdlibm algorithm), operation for operation: the
// reference compares acosf(...) with the threshold, so the last bit matters.  Checked against libm for
// every float in [-1, 1] (tests/test_acosf_port.py runs the same text on the host).
DCSG_DEV float dcsg_acosf(float x) {
    const float one = 1.0f, pi = 3.1415925026e+00f, pio2_hi = 1.5707962513e+00f, pio2_lo = 7.5497894159e-08f,
                pS0 = 1.6666667163e-01f, pS1 = -3.2556581497e-01f, pS2 = 2.0121252537e-01f, pS3 = -4.0055535734e-02f,
                pS4 = 7.9153501429e-04f, pS5 = 3.4793309169e-05f, qS1 = -2.4033949375e+00f, qS2 = 2.0209457874e+00f,
                qS3 = -6.8828397989e-01f, qS4 = 7.7038154006e-02f;
    const int hx = __float_as_int(x);
    const int ix = hx & 0x7fffffff;
    if (ix == 0x3f800000) return hx > 0 ? 0.0f : pi + 2.0f * pio2_lo;
    if (ix > 0x3f800000) return (x - x) / (x - x);
    if (ix < 0x3f000000) {
        if (ix <= 0x32800000) return pio2_hi + pio2_lo;
        const float z = x * x;
        const float p = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
        const float q = one + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
        const float r = p / q;
        return pio2_hi - (x - (pio2_lo - x * r));
    }
    if (hx < 0) {
        const float z = (one + x) * 0.5f;
        const float p = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
        const float q = one + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
        const float s = sqrtf(z);
        const float r = p / q;
        const float w = r * s - pio2_lo;
        return pi - 2.0f * (s + w);
    }
    const float z = (one - x) * 0.5f;
    const float s = sqrtf(z);
    const float df = __int_as_float(__float_as_int(s) & 0xfffff000);
    const float c = (z - df * df) / (s + df);
    const float p = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
    const float q = one + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
    const float r = p / q;
    const float w = r * s + c;
    return 2.0f * (df + w);
}

// Vector3f::angleBetweenVectors (geometry.hpp:118-124) with tolerance 1e-6f
DCSG_DEV float dcsg_angle_between(float3 a, float3 b) {
    const float ma = sqrtf(a.x * a.x + a.y * a.y + a.z * a.z);
    const float mb = sqrtf(b.x * b.x + b.y * b.y + b.z * b.z);
    if (ma * mb < 1e-6f) return 0.0f;
    return dcsg_acosf((a.x * b.x + a.y * b.y + a.z * b.z) / (ma * mb));
}

DCSG_DEV dcsg_u32 dcsg_lattice_bit(const dcsg_u32* bitmap, dcsg_u32 planeWords, int pitch, dcsg_u32 x, dcsg_u32 y, dcsg_u32 z) {
    const dcsg_u32 lp = x + (dcsg_u32)pitch * y;
    return (bitmap[(dcsg_u64)z * planeWords + (lp >> 5)] >> (lp & 31u)) & 1u;
}

extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_adapt_level(const dcsg_adapt_params p) {
    dcsg_enter();
    __shared__ dcsg_u32 s_split[DCSG_BLOCK];
    __shared__ dcsg_u32 s_emit[DCSG_BLOCK];
    __shared__ dcsg_u32 s_undecided[DCSG_BLOCK];
    const int lvl = p.level;
    const dcsg_u32 n = 1u << lvl;
    const dcsg_u32 wordsPerRow = (n < 32u ? 32u : n) >> 5;
    const dcsg_u32 totalWords = wordsPerRow * n * n;
    const dcsg_u32 w = blockIdx.x * DCSG_BLOCK + threadIdx.x;
    const bool in = w < totalWords;
    dcsg_u32 xw = 0, ny = 0, nz = 0, cand = 0u;
    if (in) {
        xw = w % wordsPerRow;
        const dcsg_u32 rest = w / wordsPerRow;
        ny = rest % n;
        nz = rest / n;
        if ((int)nz < p.nodeZLo || (int)nz >= p.nodeZHi) {
            cand = 0u;                                      // another slab's nodes
        } else if (lvl == 0) {
            cand = 1u;
        } else {
            const dcsg_u32 pn = n >> 1;
            const dcsg_u32 pWordsPerRow = (pn < 32u ? 32u : pn) >> 5;
            const dcsg_u32 pw = p.parentSplit[((dcsg_u64)(nz >> 1) * pn + (ny >> 1)) * pWordsPerRow + (xw >> 1)];
            cand = dcsg_double_bits(pw >> (16u * (xw & 1u)));
        }
    }
    s_split[threadIdx.x] = 0u;
    s_emit[threadIdx.x] = 0u;
    s_undecided[threadIdx.x] = 0u;
    __syncwarp();
    const int sh = p.L - lvl;                               // the node spans 2^sh lattice cells
    const dcsg_u32 size = 1u << sh;
    const dcsg_u32 P = (1u << p.L) + 1u;
    const int warpBase = threadIdx.x & ~31;

    // bit of the sample at GLOBAL lattice coordinates in a slab bitmap
    auto lbit = [&](const dcsg_u32* bitmap, dcsg_u32 x, dcsg_u32 y, dcsg_u32 z) {
        return dcsg_lattice_bit(bitmap, p.planeWords, p.pitch, x, y, z - (dcsg_u32)p.z0);
    };
    // corner mask of node (x0, y0, z0): corner order of geometry.hpp:264-279
    auto corner_mask = [&](dcsg_u32 x0, dcsg_u32 y0, dcsg_u32 z0) {
        const dcsg_u32 x1 = x0 + size, y1 = y0 + size, z1 = z0 + size;
        dcsg_u32 m = 0u;
        m |= lbit(p.sign, x0, y0, z1) << 0;
        m |= lbit(p.sign, x1, y0, z1) << 1;
        m |= lbit(p.sign, x1, y0, z0) << 2;
        m |= lbit(p.sign, x0, y0, z0) << 3;
        m |= lbit(p.sign, x0, y1, z1) << 4;
        m |= lbit(p.sign, x1, y1, z1) << 5;
        m |= lbit(p.sign, x1, y1, z0) << 6;
        m |= lbit(p.sign, x0, y1, z0) << 7;
        return m;
    };

    // ---- pass 1: cull, level rules, edge ambiguity (bits only) ---------------------------------------
    dcsg_warp_for_each_bit(cand, [&](bool valid, int owner, dcsg_u32 bit) {
        const dcsg_u32 oxw = __shfl_sync(0xffffffffu, xw, owner);
        const dcsg_u32 ony = __shfl_sync(0xffffffffu, ny, owner);
        const dcsg_u32 onz = __shfl_sync(0xffffffffu, nz, owner);
        if (!valid) return;
        const dcsg_u32 x0 = (oxw * 32u + bit) << sh, y0 = ony << sh, z0 = onz << sh;
        // centre-sample cull; the leaf of the grid level samples its min corner (ISV truncation)
        // (levels whose nodes are thicker than the slab keep their verdicts in small node bitmaps: the centre may lie on
        // another rank's planes)
        bool culled;
        if ((p.thickMask >> lvl) & 1u) {
            const dcsg_u32 node = (oxw * 32u + bit) + (ony << lvl) + (onz << (2 * lvl));
            culled = ((p.coarse[p.coarseOff[lvl] + (node >> 5)] >> (node & 31u)) & 1u) != 0u;
        } else {
            culled = sh > 0 ? lbit(p.cfail, x0 + (size >> 1), y0 + (size >> 1), z0 + (size >> 1)) != 0u : lbit(p.leaf, x0, y0, z0) != 0u;
        }
        if (culled) return;
        const int slot = warpBase + owner;
        if (lvl < p.minLevel) { atomicOr(&s_split[slot], 1u << bit); return; }
        if (lvl == p.maxLevel) {
            const dcsg_u32 m = corner_mask(x0, y0, z0);
            if (m != 0u && m != 255u) atomicOr(&s_emit[slot], 1u << bit);
            return;
        }
        // edge ambiguity: interior samples of the 12 edges.  The sample's lattice index depends on the
        // direction the reference walks the edge (start + delta * i/points): x edges run + on the z1
        // side and - on the z0 side, z edges + on the x0 side and - on the x1 side, y edges +.
        const int* snapX = p.snap;
        const int* snapY = p.snap + 2 * P;
        const int* snapZ = p.snap + 4 * P;
        bool ambiguous = false;
        for (dcsg_u32 i = 1; i < size && !ambiguous; ++i) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const dcsg_u32 a = (e & 1) ? size : 0u, b = (e & 2) ? size : 0u;
                // x edge at (y0 + a, z0 + b)
                ambiguous |= lbit(p.sign, (dcsg_u32)snapX[((e & 2) ? 0u : P) + x0 + i], y0 + a, z0 + b) != 0u;
                // y edge at (x0 + a, z0 + b)
                ambiguous |= lbit(p.sign, x0 + a, (dcsg_u32)snapY[y0 + i], z0 + b) != 0u;
                // z edge at (x0 + a, y0 + b)
                ambiguous |= lbit(p.sign, x0 + a, y0 + b, (dcsg_u32)snapZ[((e & 1) ? P : 0u) + z0 + i]) != 0u;
            }
        }
        if (ambiguous) atomicOr(&s_split[slot], 1u << bit);
        else atomicOr(&s_undecided[slot], 1u << bit);
    });
    __syncwarp();

    // ---- pass 2: complex edges (normals at the eight corners) -------------------------------------------
    const dcsg_u32 undecided = s_undecided[threadIdx.x];
    const dcsg_u32 tested = dcsg_warp_for_each_bit(undecided, [&](bool valid, int owner, dcsg_u32 bit) {
        const dcsg_u32 oxw = __shfl_sync(0xffffffffu, xw, owner);
        const dcsg_u32 ony = __shfl_sync(0xffffffffu, ny, owner);
        const dcsg_u32 onz = __shfl_sync(0xffffffffu, nz, owner);
        if (!valid) return;
        const dcsg_u32 x0 = (oxw * 32u + bit) << sh, y0 = ony << sh, z0 = onz << sh;
        float3 nrm[8];
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
            // corner order: 0(-,-,+) 1(+,-,+) 2(+,-,-) 3(-,-,-) 4(-,+,+) 5(+,+,+) 6(+,+,-) 7(-,+,-)
            const dcsg_u32 cx = x0 + (((0x66 >> c) & 1) ? size : 0u);
            const dcsg_u32 cy = y0 + ((c >> 2) ? size : 0u);
            const dcsg_u32 cz = z0 + (((0x33 >> c) & 1) ? size : 0u);
            float unused;
            const float3 v = dcsg_normal_and_sdf<false>(float3(p.px[cx], p.py[cy], p.pz[cz]), unused);
            // (a private array indexed by the rolled loop would live in local memory; select into registers)
#pragma unroll
            for (int k = 0; k < 8; ++k) if (k == c) nrm[k] = v;
        }
        bool complex = false;
#pragma unroll
        for (int e = 0; e < 12; ++e) {
            const int a = e < 8 ? e : e - 8;
            const int b = e < 4 ? (e + 1) & 3 : (e < 8 ? 4 + ((e + 1) & 3) : e - 4);
            complex |= dcsg_angle_between(nrm[a], nrm[b]) > p.threshold;
        }
        const int slot = warpBase + owner;
        if (complex) atomicOr(&s_split[slot], 1u << bit);
        else {
            const dcsg_u32 m = corner_mask(x0, y0, z0);
            if (m != 0u && m != 255u) atomicOr(&s_emit[slot], 1u << bit);
        }
    });
    __syncwarp();
    if (in) {
        p.split[w] = s_split[threadIdx.x];
        p.emit[w] = s_emit[threadIdx.x];
    }
    dcsg_count_evals(tested * 48u, p.evalCount);
}

// ---------------------------------------------------------------------------------------------
// preview: the 640x480 sphere-traced view of the scene (reference kernel k1, master/k1.cl:480-580,
// launched per frame by BasicDrawPane, master/DrawPane.cpp:122-240).  Off the export path, but a
// consumer of the same compiled scene.  Per pixel: a ray through (uv, IFOV) in the camera basis,
// up to 512 marching steps of 0.85 * sdf (march, k1.cl:420-470), then the 6-tap normal and the
// material of the LAST object whose own SDF is within 2 * SDF_EPSILON (shade, k1.cl:280-379).
// k1's SDF is the scene's bytecode result united with three axis-gizmo cylinders (k1.cl:237-270) --
// k2's is not, which is why the export never uses this function.
// ---------------------------------------------------------------------------------------------
#define DCSG_PREVIEW_WIDTH 640
#define DCSG_PREVIEW_HEIGHT 480
#define DCSG_AXES_RADIUS 0.015
#define DCSG_IFOV 1.0f

DCSG_DEV float dcsg_axes_cylinder(float r, float h, float halfLength, float radius) {
    return T_max((fabsf(h)-halfLength),r-radius);
}

DCSG_DEV float dcsg_preview_sdf(float3 v) {
    float value = dcsg_exact::dcsg_primary_sdf(v);
    v = float3(v.x / 5.0, v.y / 5.0, v.z / 5.0);                   // the gizmo lives in root-scale units (k1.cl:237-238)
    {
        const float r = sqrtf(v.y * v.y + v.z * v.z);
        const float h = v.x - 0.5;
        value = T_min(value,dcsg_axes_cylinder(r, h, 0.5, DCSG_AXES_RADIUS));
    }
    {
        const float r = sqrtf(v.x * v.x + v.z * v.z);
        const float h = v.y - 0.5;
        value = T_min(value,dcsg_axes_cylinder(r, h, 0.5, DCSG_AXES_RADIUS));
    }
    {
        const float r = sqrtf(v.x * v.x + v.y * v.y);
        const float h = v.z - 0.5;
        value = T_min(value,dcsg_axes_cylinder(r, h, 0.5, DCSG_AXES_RADIUS));
    }
    return value;
}

DCSG_DEV float3 dcsg_preview_normal(float3 v) {
    const float e = (float)NORMAL_EPSILON;
    float f[6];
#pragma unroll 1
    for (int k = 0; k < 6; ++k) {
        const int axis = k >> 1;
        const float dx = axis == 0 ? e : 0.0f, dy = axis == 1 ? e : 0.0f, dz = axis == 2 ? e : 0.0f;
        const float3 q = (k & 1) ? float3(v.x - dx, v.y - dy, v.z - dz) : float3(v.x + dx, v.y + dy, v.z + dz);
        const float val = dcsg_preview_sdf(q);
#pragma unroll
        for (int j = 0; j < 6; ++j) if (j == k) f[j] = val;
    }
    const float Dx = f[0] - f[1], Dy = f[2] - f[3], Dz = f[4] - f[5];
    const float twoE = 2.0 * NORMAL_EPSILON;
    return dcsg_exact::normalize(float3(1.0 / twoE * Dx, 1.0 / twoE * Dy, 1.0 / twoE * Dz));
}

// generated by dcsg_build from scene.txt: the object loop of shade (k1.cl:300-325) with the table as immediates
namespace dcsg_exact { __device__ float3 dcsg_shade_objects(float3 v, float3 n, bool& matched); }

DCSG_DEV float3 dcsg_preview_shade(float3 v, float3 n) {
    bool matched;
    const float3 colour = dcsg_exact::dcsg_shade_objects(v, n, matched);
    if (matched) return colour;
    v = float3(v.x / 5.0, v.y / 5.0, v.z / 5.0);
    {
        const float r = sqrtf(v.y * v.y + v.z * v.z);
        const float h = v.x - 0.5;
        if (dcsg_axes_cylinder(r, h, 0.5, 0.025) < SDF_EPSILON * TOLERANCE_FACTOR_MATERIAL) return float3(1.0, 0.0, 0.0);
    }
    {
        const float r = sqrtf(v.x * v.x + v.z * v.z);
        const float h = v.y - 0.5;
        if (dcsg_axes_cylinder(r, h, 0.5, 0.025) < SDF_EPSILON * TOLERANCE_FACTOR_MATERIAL) return float3(0.0, 1.0, 0.0);
    }
    {
        const float r = sqrtf(v.x * v.x + v.y * v.y);
        const float h = v.z - 0.5;
        if (dcsg_axes_cylinder(r, h, 0.5, 0.025) < SDF_EPSILON * TOLERANCE_FACTOR_MATERIAL) return float3(0.0, 0.0, 1.0);
    }
    return float3(239.0 / 255.0, 66.0 / 255.0, 245 / 255.0);       // nothing matched: k1.cl:377
}

DCSG_DEV unsigned char dcsg_clip_channel(int value) {
    value = (value < 0) ? 0 : ((value > 255) ? 255 : value);
    return (unsigned char)value;
}

struct dcsg_preview_params {
    float campos[3];
    float right[3];
    float up[3];
    float forward[3];
    unsigned char* pixels;          // 640 x 480 x RGB, rows top to bottom (k1's tid = iy*640 + ix)
};

extern "C" __global__ void __launch_bounds__(DCSG_BLOCK)
dcsg_k_preview(const dcsg_preview_params p) {
    dcsg_enter();
    const int tid = blockIdx.x * DCSG_BLOCK + threadIdx.x;
    if (tid >= DCSG_PREVIEW_WIDTH * DCSG_PREVIEW_HEIGHT) return;
    const int iy = tid / DCSG_PREVIEW_WIDTH, ix = tid - iy * DCSG_PREVIEW_WIDTH;
    const float3 o = float3(p.campos[0], p.campos[1], p.campos[2]);
    const float2 uv = float2((float)(ix - 640 / 2), -(float)(iy - 480 / 2)) / float2(640.0 / 2.0, 640.0 / 2.0);
    const float3 rgt = float3(p.right[0], p.right[1], p.right[2]);
    const float3 upp = float3(p.up[0], p.up[1], p.up[2]);
    const float3 fwd = float3(p.forward[0], p.forward[1], p.forward[2]);
    const float3 r = float3(uv.x, uv.y, DCSG_IFOV);
    float3 colour = float3(1.0, 1.0, 1.0);
    // march (k1.cl:420-470): origin and direction in the camera basis, at most MAX_STEPS steps of 0.85 * sdf
    float d = 0.0;
    {
        float3 v = float3(dot(o, rgt), dot(o, upp), dot(o, fwd));
        const float3 dir = float3(dot(r, rgt), dot(r, upp), dot(r, fwd));
        float hit = -1.0;
#pragma unroll 1
        for (int i = 0; i < MAX_STEPS; ++i) {
            const float s = dcsg_preview_sdf(v) * TOLERANCE_FACTOR_MARCHSTEP;
            if (s < SDF_EPSILON) { hit = d; break; }
            v = v + s * dir;
            d = d + s;
            if (d > MAX_DISTANCE) break;
        }
        d = hit;
    }
    if (d > 0.0) {
        const float3 point = float3(dot(o, rgt), dot(o, upp), dot(o, fwd)) + d * float3(dot(r, rgt), dot(r, upp), dot(r, fwd));
        colour = dcsg_preview_shade(point, dcsg_preview_normal(point));
    }
    p.pixels[tid * 3 + 0] = dcsg_clip_channel((int)(255.0 * colour.x));
    p.pixels[tid * 3 + 1] = dcsg_clip_channel((int)(255.0 * colour.y));
    p.pixels[tid * 3 + 2] = dcsg_clip_channel((int)(255.0 * colour.z));
}
