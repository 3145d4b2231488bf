// round_flags.cpp -- TEST HARNESS (host).  Does the fast copy flag the tap round of the projection at a point?
//
// The projection kernel (scene_kernels.cuh) defers a vertex to its exact phase when the round's seven evaluations through
// the checked fast copy raise the flag: a generated transform test (`inexact`) or a square root through dcsg_sqrt_checked
// (scene_prelude.cuh), which flags every input outside [T, FLT_MAX] and NaN.  This file compiles tests/cpu_emul/tap_axes.cpp
// (the fast copy's generated functions around the scene's OpenCL-C text) with every float square root of the scene text --
// sqrt, sqrtf, and through them length, normalize, distance -- replaced by one that also raises that flag.
// tests/test_projection_kernel.py passes T as SQRT_FLAG_BELOW (its sweep of dcsg_sqrt_checked on the device checks T).
//   g++ -O2 -ffp-contract=off -shared -fPIC -DSQRT_FLAG_BELOW=... -DGENERATED_INC=... -DSCENE_INC=... -I oracle
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstddef>

namespace K {
static bool sqrt_flag = false;
static inline float checked_sqrt(float x) {
    if (!(x >= (float)(SQRT_FLAG_BELOW) && x <= FLT_MAX)) sqrt_flag = true;
    return std::sqrt(x);
}
static inline double checked_sqrt(double x) { return std::sqrt(x); }
template <typename T> static inline double checked_sqrt(T x) { return std::sqrt((double)x); }      // integer arguments
}  // namespace K
// (function-like: `using std::sqrt;` in the shim is left alone; the headers above are already in)
#define sqrtf(x) K::checked_sqrt((float)(x))
#define sqrt(x) K::checked_sqrt(x)

#include "../cpu_emul/tap_axes.cpp"

// flag[i]: the OR over the seven taps v + (e,0,0), v - (e,0,0), ..., v of the single evaluation's flag, square roots included
// -- the flag of the rolled tap loop, and so of a round in either tap form
extern "C" void round_flags(const float* xyz, size_t n, float* table, unsigned char* flag) {
    K::arbitrary_data = table;
    const float e = (float)NORMAL_EPSILON;
    for (size_t i = 0; i < n; i++) {
        const K::float3 v(xyz[i * 3 + 0], xyz[i * 3 + 1], xyz[i * 3 + 2]);
        const K::float3 taps[7] = {
            K::float3(v.x + e, v.y + 0.0f, v.z + 0.0f), K::float3(v.x - e, v.y - 0.0f, v.z - 0.0f),
            K::float3(v.x + 0.0f, v.y + e, v.z + 0.0f), K::float3(v.x - 0.0f, v.y - e, v.z - 0.0f),
            K::float3(v.x + 0.0f, v.y + 0.0f, v.z + e), K::float3(v.x - 0.0f, v.y - 0.0f, v.z - e), v};
        bool inexact = false;
        K::sqrt_flag = false;
        for (int k = 0; k < 7; k++) (void)K::dcsg_primary_sdf(taps[k], inexact);
        flag[i] = (inexact || K::sqrt_flag) ? 1 : 0;
    }
}
