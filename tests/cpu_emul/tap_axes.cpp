// tap_axes.cpp -- TEST HARNESS (host).  The per-axis tap forms of the fast copy against its single-evaluation form, on the CPU.
//
// libdcsg generates, for namespace dcsg_fast, the scene's SDF as one evaluation (generate_primary_sdf, fast) and the taps of a
// normal per world axis (generate_primary_sdf_axis, designcsg_b200/csrc/host_scene.cu).  tests/test_tap_forms.py cuts those
// functions out of dcsg_scene_source(), pastes them into GENERATED_INC and compiles this file with the scene's OpenCL-C text
// behind the oracle's shim, as tests/cpu_emul/fast_copy.cpp does.  The single evaluation runs at the seven points the
// reference's get_normal and the projection's centre sample evaluate: v + (e,0,0), v - (e,0,0), ..., v.
//   g++ -O2 -ffp-contract=off -shared -fPIC -DGENERATED_INC=... -DSCENE_INC=... -I oracle
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstddef>

#define STACK_MEMORY_PER_PIXEL 64

namespace K {
#include "clshim.h"
#include "k2_port.inc"

#define __device__
#define __forceinline__ inline
#define DCSG_BAD_DECLARE() bool dcsg_bad = false
#define DCSG_BAD_UNLESS_ABS_LT(x, c) dcsg_bad |= !(fabsf(x) < (c))
#define DCSG_BAD_UNLESS_ABS_GE(x, c) dcsg_bad |= !(fabsf(x) >= (c))
#define DCSG_BAD_UNLESS_ABS_GT0(x) dcsg_bad |= !(fabsf(x) > 0.0f)
#define DCSG_BAD_COMMIT(out) out |= dcsg_bad
static inline float __uint_as_float(unsigned int u) { float f; memcpy(&f, &u, 4); return f; }
static inline float __fmaf_rn(float a, float b, float c) { return fmaf(a, b, c); }

#include SCENE_INC
#include GENERATED_INC
}  // namespace K

// axes[i*9 + k]: k = +x, -x, +y, -y, +z, -z, centre from the round with the centre (xc, y, z), then +x, -x of the x function
// without it; single[i*7 + k] at the seven points.  flag: the round with the centre; flag6: the round without it (x, y, z);
// single_flag: any of the seven single evaluations flagged.
extern "C" void tap_axes_eval(const float* xyz, size_t n, float* table, float* axes, float* single, unsigned char* flag,
                              unsigned char* flag6, unsigned char* single_flag) {
    K::arbitrary_data = table;
    const float e = (float)NORMAL_EPSILON;
    for (size_t i = 0; i < n; i++) {
        const K::float3 v(xyz[i * 3 + 0], xyz[i * 3 + 1], xyz[i * 3 + 2]);
        float* a = axes + i * 9;
        bool up = false, up6 = false;
        float xc[3], x[2], y[2], z[2];
        K::dcsg_primary_sdf_xc(v, e, xc, up);
        K::dcsg_primary_sdf_y(v, e, y, up);
        K::dcsg_primary_sdf_z(v, e, z, up);
        K::dcsg_primary_sdf_x(v, e, x, up6);
        K::dcsg_primary_sdf_y(v, e, y, up6);
        K::dcsg_primary_sdf_z(v, e, z, up6);
        a[0] = xc[0]; a[1] = xc[1]; a[2] = y[0]; a[3] = y[1]; a[4] = z[0]; a[5] = z[1]; a[6] = xc[2]; a[7] = x[0]; a[8] = x[1];
        flag[i] = up ? 1 : 0;
        flag6[i] = up6 ? 1 : 0;
        // the reference's taps: v + (e,0,0) (unchanged coordinates v.c + 0.0f), v - (e,0,0) (v.c - 0.0f), ..., and v itself
        const K::float3 taps[7] = {
            K::float3(v.x + e, v.y + 0.0f, v.z + 0.0f), K::float3(v.x - e, v.y - 0.0f, v.z - 0.0f),
            K::float3(v.x + 0.0f, v.y + e, v.z + 0.0f), K::float3(v.x - 0.0f, v.y - e, v.z - 0.0f),
            K::float3(v.x + 0.0f, v.y + 0.0f, v.z + e), K::float3(v.x - 0.0f, v.y - 0.0f, v.z - e), v};
        bool inexact = false;
        for (int k = 0; k < 7; k++) single[i * 7 + k] = K::dcsg_primary_sdf(taps[k], inexact);
        single_flag[i] = inexact ? 1 : 0;
    }
}
