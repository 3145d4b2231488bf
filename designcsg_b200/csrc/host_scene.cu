// host_scene.cu -- scene files -> specialised CUDA source -> sm_100a cubin (NVRTC).
//
// Plays the role of the reference's scene loader (BasicDrawPane::loadScene, master/DrawPane.cpp:243-371) and of
// Evaluator::build / Utils::build_program (master/Evaluator.cpp:45-112, master/Utils.cpp:48-103): the CSG bytecode and the
// object table are static per scene, so they are turned into straight-line CUDA with the (%.6f-quantised, sscanf-parsed)
// transforms as immediates instead of being interpreted per sample.
#include "host_internal.h"
#include <elf.h>
#include "scene_module_src.inc"     // generated: kScenePrelude, kSceneParams, kSceneKernels (raw strings)

using namespace dcsg_host;

namespace dcsg_host {

bool load_scene(const std::string& dir, Scene& sc, std::string& err) {
    std::string text;
    if (!read_file(dir + "/scene.cu", sc.scene_cu)) { err = "cannot read " + dir + "/scene.cu"; return false; }
    sc.private_words = 0;
    {
        const size_t at = sc.scene_cu.find("// DCSG_PRIVATE_WORDS ");
        if (at != std::string::npos) sc.private_words = atoi(sc.scene_cu.c_str() + at + 22);
        // one 4-byte slot per thread and variable in the launch's dynamic shared memory: 256 threads x 192 words = 192 KiB
        // is what fits next to the kernels' static ~8 KiB on sm_100a (227 KiB per block)
        if (sc.private_words < 0 || sc.private_words > 192) { err = "scene.cu: more than 192 program-scope scalars (per-thread state does not fit in shared memory)"; return false; }
    }
    if (!read_file(dir + "/scene.txt", text)) { err = "cannot read " + dir + "/scene.txt"; return false; }
    sc.num_objects = 0;
    size_t pos = 0;
    while (pos < text.size()) {
        size_t eol = text.find('\n', pos);
        if (eol == std::string::npos) eol = text.size();
        std::string line = text.substr(pos, eol - pos);
        pos = eol + 1;
        int b = 0, m = 0;
        float v[12];
        if (sscanf(line.c_str(), "%d %d %f %f %f %f %f %f %f %f %f %f %f %f", &b, &m, &v[0], &v[1], &v[2], &v[3], &v[4],
                   &v[5], &v[6], &v[7], &v[8], &v[9], &v[10], &v[11]) != 14)
            continue;
        if (sc.num_objects >= DCSG_MAX_OBJECTS) { err = "scene.txt: more than 512 objects"; return false; }
        const int n = sc.num_objects++;
        sc.shape_id[n] = b & 0xff;          // the bank is `unsigned char` in the reference (k2.cl:36)
        sc.material_id[n] = m;
        for (int k = 0; k < 3; k++) {
            sc.position[n][k] = v[k];
            sc.right[n][k] = v[3 + k];
            sc.up[n][k] = v[6 + k];
            sc.forward[n][k] = v[9 + k];
        }
    }
    if (!read_file(dir + "/buildprocedure.txt", text)) { err = "cannot read " + dir + "/buildprocedure.txt"; return false; }
    sc.num_steps = 0;
    pos = 0;
    while (pos < text.size()) {
        size_t eol = text.find('\n', pos);
        if (eol == std::string::npos) eol = text.size();
        std::string line = text.substr(pos, eol - pos);
        pos = eol + 1;
        int c[4];
        if (sscanf(line.c_str(), "%d %d %d %d", &c[0], &c[1], &c[2], &c[3]) != 4) continue;
        if (sc.num_steps >= DCSG_MAX_BUILD_STEPS) { err = "buildprocedure.txt: more than 256 commands"; return false; }
        memcpy(sc.steps[sc.num_steps++], c, sizeof(c));
    }
    std::string raw;
    sc.arbitrary_data.clear();
    if (read_file(dir + "/arbitrary_data.hex", raw)) {
        size_t items = std::min(raw.size() / 4, (size_t)DCSG_ARBITRARY_DATA_POINTS);
        sc.arbitrary_data.resize(items);
        memcpy(sc.arbitrary_data.data(), raw.data(), items * 4);
    }
    sc.export_config.clear();
    if (read_file(dir + "/exportConfig.txt", text)) {
        pos = 0;
        while (pos < text.size()) {
            size_t eol = text.find('\n', pos);
            if (eol == std::string::npos) eol = text.size();
            if (eol > pos) sc.export_config.push_back(text.substr(pos, eol - pos));
            pos = eol + 1;
        }
    }
    return true;
}

std::string float_literal(float f) {
    uint32_t bits;
    memcpy(&bits, &f, 4);
    return format("__uint_as_float(0x%08xu)", bits);
}

uint32_t float_bits(float f) {
    uint32_t bits;
    memcpy(&bits, &f, 4);
    return bits;
}

// dot(d, a) = (d.x*a.x + d.y*a.y) + d.z*a.z with the reference's rounding: each product and each sum
// rounded once, left to right.  Two exact rewrites, both relying on fma(p, q, r) = fl(p*q + r):
//  (1) a product by +-1 never rounds, so fl(fl(p*(+-1)) + r) == fma(p, +-1, r) (addition is commutative,
//      so the exact product may be either operand of the sum it takes part in);
//  (2) a product by +-0 is an exact signed zero.  Adding a zero to a non-zero value returns that value
//      unrounded, and a sum made only of zeros is -0 iff every addend is -0, whatever the order -- so the
//      zero-coefficient terms may be applied LAST, as fma(d, +-0, acc), without changing a bit (NaN / Inf
//      operands give NaN either way).
// Axis-aligned objects have two zero coefficients per axis vector: 3 FMUL + 2 FADD become 1 FMUL + 2 FFMA.
bool is_zero_coefficient(float c) { return (float_bits(c) & 0x7fffffffu) == 0u; }
bool is_unit_coefficient(float c) { return (float_bits(c) & 0x7fffffffu) == 0x3f800000u; }

// lastAxis = -1: fewest instructions (1 FMUL + 2 FFMA for an axis-aligned axis vector).
// lastAxis = 0/1/2: the same value with every term that does not depend on that axis grouped first, so that several
//                evaluations differing only in that coordinate (the samples of one lattice row; the +/- taps of a
//                normal) share the rest (the zero terms commute, see (2); the non-zero terms keep the reference's
//                order and association).  d[] = names of the three difference variables.
std::string dot_expression(const float a[3], int lastAxis, const std::string d[3]) {
    auto product = [&](int k) { return d[k] + " * " + float_literal(a[k]); };
    auto fused = [&](int k, const std::string& acc) { return "__fmaf_rn(" + d[k] + ", " + float_literal(a[k]) + ", " + acc + ")"; };
    std::vector<int> rest, zeros;
    for (int k = 0; k < 3; k++) (is_zero_coefficient(a[k]) ? zeros : rest).push_back(k);
    if (rest.empty()) {                      // all three coefficients are zero: start from a product that is not the last axis
        int pick = (int)zeros.size() - 1;
        while (pick > 0 && zeros[pick] == lastAxis) --pick;
        rest.push_back(zeros[pick]);
        zeros.erase(zeros.begin() + pick);
    }
    std::string core;
    if (rest.size() == 1) {
        core = product(rest[0]);
    } else {
        const int i = rest[0], j = rest[1];
        if (is_unit_coefficient(a[i])) core = fused(i, product(j));
        else if (is_unit_coefficient(a[j])) core = fused(j, product(i));
        else core = "(" + product(i) + " + " + product(j) + ")";
        if (rest.size() == 3) {
            const int k = rest[2];
            core = is_unit_coefficient(a[k]) ? fused(k, core) : "(" + core + " + " + product(k) + ")";
        }
    }
    const bool coreUsesLast = lastAxis >= 0 && std::find(rest.begin(), rest.end(), lastAxis) != rest.end();
    if (coreUsesLast && !zeros.empty()) {
        // the zero terms do not involve the last axis: fold them into one signed zero that is shared, add it last
        std::string zsum = product(zeros[0]);
        for (size_t z = 1; z < zeros.size(); z++) zsum = fused(zeros[z], zsum);
        return "(" + core + " + " + zsum + ")";
    }
    if (lastAxis >= 0)                      // the last axis' zero term goes outermost, the others keep a fixed order
        std::stable_sort(zeros.begin(), zeros.end(), [&](int l, int r) { return (l == lastAxis) < (r == lastAxis); });
    for (int k : zeros) core = fused(k, core);
    return core;
}

// Specialise reference primary_sdf (k2.cl:47-144) for one scene: the interpreter's loop over the
// bytecode becomes straight-line code, the private stack becomes registers, the object table becomes
// immediates.  The arithmetic of every command is the interpreter's, in the same order:
//   IMPORT: ABC = (dot(v-o,right), dot(v-o,up), dot(v-o,forward)); slot = sdf_bank(ABC, brush)
//   MIN / MAX: T_min / T_max ternaries; NEGATE; IDENTITY; EXPORT.
//
// fast = true emits the checked form for namespace dcsg_fast (scene_prelude.cuh "Two copies of the scene, one result"):
// an axis vector with zero coefficients loses its zero terms altogether.  By (2) those terms only matter when the rest
// of the sum is itself a zero (they then decide its sign) or when their own operand is not finite (0 * Inf = NaN), so
//      dot = core                       whenever core != +-0 and the dropped operands are finite,
// and the generated code raises `inexact` otherwise: once per evaluation !(|v.c| < 2^120) for the three coordinates
// (covers every dropped operand: they are v.c - position.c with |position.c| < 2^100), and per DISTINCT non-zero term
// !(|d| >= 2^-60) when the core is a single product d * a with 2^-40 <= |a| (it then cannot be or round to zero; objects
// that share an axis and an offset share the test), or core == 0 tested on the value itself when two terms remain.
// Design1: 66 FFMAs per evaluation become 12 compares.
// One local coordinate (axis vector k of object o) in the fast copy's form, over the differences d[]: `expr`, and what guards
// it when zero terms were dropped -- `testAxis` >= 0: |d[testAxis]| >= 2^-60 (a single product); `testCore`: |expr| > 0.
// elided = false: the exact form, dot_expression(.., lastAxis, d), no test.
struct FastCoordinate {
    std::string expr;
    bool elided = false, testCore = false;
    int testAxis = -1;
};
FastCoordinate fast_coordinate(const Scene& sc, int o, int k, int lastAxis, const std::string d[3]) {
    const float (*axes[3])[3] = {&sc.right[o], &sc.up[o], &sc.forward[o]};
    const float* a = *axes[k];
    FastCoordinate fc;
    std::vector<int> rest, zeros;
    for (int c = 0; c < 3; c++) (is_zero_coefficient(a[c]) ? zeros : rest).push_back(c);
    bool elide = !zeros.empty() && !rest.empty();
    for (int c : zeros) elide = elide && fabsf(sc.position[o][c]) < 0x1p100f;
    if (elide && rest.size() == 1) elide = fabsf(a[rest[0]]) >= 0x1p-40f;       // NaN coefficients fail this too
    if (!elide) {
        fc.expr = dot_expression(a, lastAxis, d);
        return fc;
    }
    fc.elided = true;
    auto product = [&](int c) { return d[c] + " * " + float_literal(a[c]); };
    if (rest.size() == 1) {
        fc.expr = product(rest[0]);
        fc.testAxis = rest[0];
    } else {
        // two non-zero terms: the reference's sum of the two products (dot_expression without the zero term)
        const int i = rest[0], j = rest[1];
        auto fused = [&](int c, const std::string& acc) { return "__fmaf_rn(" + d[c] + ", " + float_literal(a[c]) + ", " + acc + ")"; };
        if (is_unit_coefficient(a[i])) fc.expr = fused(i, product(j));
        else if (is_unit_coefficient(a[j])) fc.expr = fused(j, product(i));
        else fc.expr = "(" + product(i) + " + " + product(j) + ")";
        fc.testCore = true;
    }
    return fc;
}

bool generate_primary_sdf(const Scene& sc, bool rowVariant, bool fast, std::string& out, std::string& err) {
    std::set<std::pair<int, uint32_t>> tested;          // (axis, position bits) whose difference already has its magnitude test
    bool anyElided = false;
    bool used[DCSG_STACK_SLOTS] = {false};
    auto slot_ok = [&](int s) { return s >= 0 && s < DCSG_STACK_SLOTS; };
    std::string body;
    for (int i = 0; i < sc.num_steps; i++) {
        const int op = sc.steps[i][0], lhs = sc.steps[i][1], rhs = sc.steps[i][2], dst = sc.steps[i][3];
        switch (op) {
        case 0: {   // IMPORT
            if (rhs < 0 || rhs >= sc.num_objects || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad IMPORT", i); return false; }
            used[dst] = true;
            const int o = rhs;
            body += format("    {   // IMPORT brush %d, object %d -> slot %d\n", lhs, o, dst);
            // v - o: subtracting +0.0f is the identity on every float (including -0.0f), so it is dropped
            const char* comp[3] = {"x", "y", "z"};
            for (int k = 0; k < 3; k++) {
                if (float_bits(sc.position[o][k]) == 0u)
                    body += format("        const float dcsg_d%s = dcsg_v.%s;\n", comp[k], comp[k]);
                else
                    body += format("        const float dcsg_d%s = dcsg_v.%s - ", comp[k], comp[k]) + float_literal(sc.position[o][k]) + ";\n";
            }
            const float (*axes[3])[3] = {&sc.right[o], &sc.up[o], &sc.forward[o]};
            const char* names[3] = {"dcsg_la", "dcsg_lb", "dcsg_lc"};
            const std::string dnames[3] = {"dcsg_dx", "dcsg_dy", "dcsg_dz"};
            for (int k = 0; k < 3; k++) {
                if (!fast) {
                    body += "        const float " + std::string(names[k]) + " = " + dot_expression(*axes[k], rowVariant ? 0 : -1, dnames) + ";\n";
                    continue;
                }
                const FastCoordinate fc = fast_coordinate(sc, o, k, rowVariant ? 0 : -1, dnames);
                body += "        const float " + std::string(names[k]) + " = " + fc.expr + ";\n";
                anyElided = anyElided || fc.elided;
                if (fc.testAxis >= 0 && tested.insert({fc.testAxis, float_bits(sc.position[o][fc.testAxis])}).second)
                    body += "        DCSG_BAD_UNLESS_ABS_GE(" + dnames[fc.testAxis] + ", 8.6736173798840355e-19f);\n";      // 2^-60
                if (fc.testCore) body += "        DCSG_BAD_UNLESS_ABS_GT0(" + std::string(names[k]) + ");\n";
            }
            body += format("        dcsg_s%d = sdf_bank(float3(dcsg_la, dcsg_lb, dcsg_lc), (unsigned char)%d);\n    }\n", dst, lhs & 0xff);
        } break;
        case 1:     // EXPORT
            if (!slot_ok(lhs)) { err = format("buildprocedure.txt command %d: bad EXPORT", i); return false; }
            used[lhs] = true;
            body += format("    dcsg_exported = dcsg_s%d;\n", lhs);
            break;
        case 2: case 3:
            if (!slot_ok(lhs) || !slot_ok(rhs) || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad slot", i); return false; }
            used[lhs] = used[rhs] = used[dst] = true;
            body += format("    dcsg_s%d = %s(dcsg_s%d,dcsg_s%d);\n", dst, op == 2 ? "T_min" : "T_max", lhs, rhs);
            break;
        case 4: case 5:
            if (!slot_ok(lhs) || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad slot", i); return false; }
            used[lhs] = used[dst] = true;
            body += format("    dcsg_s%d = %sdcsg_s%d;\n", dst, op == 4 ? "-" : "", lhs);
            break;
        default:
            break;  // unknown opcodes fall through the reference's switch without effect
        }
    }
    out = std::string("\n// ---- generated by dcsg_build from scene.txt / buildprocedure.txt ----\n") +
          "__device__ __forceinline__ float " + (rowVariant ? "dcsg_primary_sdf_row" : "dcsg_primary_sdf") +
          (fast ? "(float3 dcsg_v, bool& dcsg_inexact_out) {\n" : "(float3 dcsg_v) {\n") +
          "    float dcsg_exported = MAX_DISTANCE;\n";
    if (fast && anyElided)
        out += "    DCSG_BAD_DECLARE();\n"
               "    DCSG_BAD_UNLESS_ABS_LT(dcsg_v.x, 1.329227995784916e+36f);\n"                                             // 2^120
               "    DCSG_BAD_UNLESS_ABS_LT(dcsg_v.y, 1.329227995784916e+36f);\n"
               "    DCSG_BAD_UNLESS_ABS_LT(dcsg_v.z, 1.329227995784916e+36f);\n";
    else if (fast)
        out += "    DCSG_BAD_DECLARE();\n";
    for (int s = 0; s < DCSG_STACK_SLOTS; s++)
        if (used[s]) out += format("    float dcsg_s%d = 0.0f;\n", s);
    out += body;
    if (fast) out += "    DCSG_BAD_COMMIT(dcsg_inexact_out);\n";
    out += "    return dcsg_exported;\n}\n";
    return true;
}

// The seven evaluations of a normal + centre value (reference get_normal k2.cl:149-179 and the centre sample of
// performGradientDescent) as ONE straight-line function, object-major: for every IMPORT the seven local-coordinate
// triples are formed next to each other with the varying coordinate's terms last, so the compiler's value numbering
// shares everything that does not depend on the tap (transform arithmetic, and inside the inlined brush whatever
// depends on unchanged coordinates only).  Every single evaluation performs the reference's operations on the
// reference's operands: the taps are v + (e,0,0) (unchanged coordinates are v.y + 0.0f: -0 becomes +0), v - (e,0,0)
// (v.y - 0.0f, bit-identical to v.y), ..., and v itself.  out[] order: +x, -x, +y, -y, +z, -z, centre.
bool generate_primary_sdf7(const Scene& sc, std::string& out, std::string& err) {
    bool used[DCSG_STACK_SLOTS] = {false};
    auto slot_ok = [&](int s) { return s >= 0 && s < DCSG_STACK_SLOTS; };
    // coordinate variants: 0 = v (centre and minus taps), 1 = v + 0.0f (plus taps), 2 = v + e, 3 = v - e
    static const int tap[7][3] = {{2, 1, 1}, {3, 0, 0}, {1, 2, 1}, {0, 3, 0}, {1, 1, 2}, {0, 0, 3}, {0, 0, 0}};
    static const int tapLast[7] = {0, 0, 1, 1, 2, 2, 2};
    const char* comp[3] = {"x", "y", "z"};
    std::string body;
    for (int i = 0; i < sc.num_steps; i++) {
        const int op = sc.steps[i][0], lhs = sc.steps[i][1], rhs = sc.steps[i][2], dst = sc.steps[i][3];
        switch (op) {
        case 0: {
            if (rhs < 0 || rhs >= sc.num_objects || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad IMPORT", i); return false; }
            used[dst] = true;
            const int o = rhs;
            body += format("    {   // IMPORT brush %d, object %d -> slot %d\n", lhs, o, dst);
            for (int k = 0; k < 3; k++)
                for (int j = 0; j < 4; j++) {
                    if (float_bits(sc.position[o][k]) == 0u)
                        body += format("        const float dcsg_d%s%d = dcsg_c%s%d;\n", comp[k], j, comp[k], j);
                    else
                        body += format("        const float dcsg_d%s%d = dcsg_c%s%d - ", comp[k], j, comp[k], j) + float_literal(sc.position[o][k]) + ";\n";
                }
            const float (*axes[3])[3] = {&sc.right[o], &sc.up[o], &sc.forward[o]};
            for (int t = 0; t < 7; t++) {
                const std::string d[3] = {format("dcsg_dx%d", tap[t][0]), format("dcsg_dy%d", tap[t][1]), format("dcsg_dz%d", tap[t][2])};
                body += format("        dcsg_s%d_%d = sdf_bank(float3(", dst, t) + dot_expression(*axes[0], tapLast[t], d) + ", " +
                        dot_expression(*axes[1], tapLast[t], d) + ", " + dot_expression(*axes[2], tapLast[t], d) +
                        format("), (unsigned char)%d);\n", lhs & 0xff);
            }
            body += "    }\n";
        } break;
        case 1:
            if (!slot_ok(lhs)) { err = format("buildprocedure.txt command %d: bad EXPORT", i); return false; }
            used[lhs] = true;
            for (int t = 0; t < 7; t++) body += format("    dcsg_out[%d] = dcsg_s%d_%d;\n", t, lhs, t);
            break;
        case 2: case 3:
            if (!slot_ok(lhs) || !slot_ok(rhs) || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad slot", i); return false; }
            used[lhs] = used[rhs] = used[dst] = true;
            for (int t = 0; t < 7; t++)
                body += format("    dcsg_s%d_%d = %s(dcsg_s%d_%d,dcsg_s%d_%d);\n", dst, t, op == 2 ? "T_min" : "T_max", lhs, t, rhs, t);
            break;
        case 4: case 5:
            if (!slot_ok(lhs) || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad slot", i); return false; }
            used[lhs] = used[dst] = true;
            for (int t = 0; t < 7; t++) body += format("    dcsg_s%d_%d = %sdcsg_s%d_%d;\n", dst, t, op == 4 ? "-" : "", lhs, t);
            break;
        default:
            break;
        }
    }
    out = "\n// ---- generated by dcsg_build: seven-tap form (normal taps + centre), see generate_primary_sdf7 ----\n"
          "__device__ __forceinline__ void dcsg_primary_sdf7(float3 dcsg_v, float dcsg_e, float (&dcsg_out)[7]) {\n";
    for (int k = 0; k < 3; k++) {
        out += format("    const float dcsg_c%s0 = dcsg_v.%s;\n", comp[k], comp[k]);
        out += format("    const float dcsg_c%s1 = dcsg_v.%s + 0.0f;\n", comp[k], comp[k]);
        out += format("    const float dcsg_c%s2 = dcsg_v.%s + dcsg_e;\n", comp[k], comp[k]);
        out += format("    const float dcsg_c%s3 = dcsg_v.%s - dcsg_e;\n", comp[k], comp[k]);
    }
    out += "    for (int dcsg_t = 0; dcsg_t < 7; ++dcsg_t) dcsg_out[dcsg_t] = MAX_DISTANCE;\n";
    for (int s = 0; s < DCSG_STACK_SLOTS; s++)
        if (used[s])
            for (int t = 0; t < 7; t++) out += format("    float dcsg_s%d_%d = 0.0f;\n", s, t);
    out += body;
    out += "}\n";
    return true;
}

// The taps of a normal along ONE world axis, for namespace dcsg_fast: the fast copy's evaluations at v + e and v - e on that
// axis (and at v itself when `centre`), as one straight-line function, object-major.  For every IMPORT the differences and
// local coordinates of its evaluations are formed next to each other, each distinct one once, the varying axis' terms last;
// then sdf_bank runs once per evaluation, and the compiler's value numbering shares inside the inlined brush whatever depends
// on the unchanged coordinates only.  For an axis-aligned object a local coordinate is one product (v.c - o.c) * a of ONE
// world coordinate, so a tap along x leaves every y- and z-dependent value of every object unchanged.
//
// Three coordinate variants are enough.  The reference's taps are v + (e,0,0) and v - (e,0,0): the unchanged coordinates of
// a plus tap are v.c + 0.0f, those of a minus tap and of the centre v.c.  They differ only where v.c is -0 (+0 then), and a
// NaN may come out of the addition with other bits.  So every function also tests its own axis' coordinate, !(|v.c| > 0):
// with the flag of a whole round (x, y and z functions) down no coordinate is +-0 or NaN, v.c + 0.0f and v.c are the same
// bits, and the seven evaluations only need v.c, v.c + e and v.c - e.  The other tests are the single-evaluation form's
// (generate_primary_sdf, fast): |coordinate| < 2^120 for every coordinate value an evaluation uses (each function tests its
// axis' three values: together they cover all of them), and the magnitude tests of the elided transform terms, each distinct
// one emitted once.  The flag is the union of all of them, so where it stays down each value is the single-evaluation fast
// form's value at that tap, which is the exact copy's.  A vertex exactly on a coordinate plane already fails the |d| >= 2^-60
// test of an object centred there, so on such scenes the zero test flags nothing new.
// out[] order: +axis, -axis, centre.
bool generate_primary_sdf_axis(const Scene& sc, int axis, bool centre, std::string& out, std::string& err) {
    const char* comp[3] = {"x", "y", "z"};
    // coordinate variables: dcsg_c<axis>0 = v.c, dcsg_c<axis>p = v.c + e, dcsg_c<axis>m = v.c - e
    auto coordinate = [&](int k, char variant) { return format("dcsg_c%s%c", comp[k], k == axis ? variant : '0'); };
    std::vector<std::array<std::string, 3>> evals;
    for (char variant : centre ? std::string("pm0") : std::string("pm")) evals.push_back({coordinate(0, variant), coordinate(1, variant), coordinate(2, variant)});
    const int n = (int)evals.size();
    std::set<std::pair<std::string, uint32_t>> tested;     // (coordinate variable, position bits) whose difference has its test
    bool anyElided = false;
    bool used[DCSG_STACK_SLOTS] = {false};
    auto slot_ok = [&](int s) { return s >= 0 && s < DCSG_STACK_SLOTS; };
    std::string body;
    for (int i = 0; i < sc.num_steps; i++) {
        const int op = sc.steps[i][0], lhs = sc.steps[i][1], rhs = sc.steps[i][2], dst = sc.steps[i][3];
        switch (op) {
        case 0: {   // IMPORT
            if (rhs < 0 || rhs >= sc.num_objects || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad IMPORT", i); return false; }
            used[dst] = true;
            const int o = rhs;
            body += format("    {   // object %d, brush %d -> slot %d, all evaluations of the function\n", o, lhs, dst);
            std::map<std::string, std::string> diff, local;     // coordinate variable -> difference; expression -> local coordinate
            auto difference = [&](const std::string& c, int k) {
                auto it = diff.find(c);
                if (it != diff.end()) return it->second;
                const std::string name = "dcsg_d" + c.substr(6);
                if (float_bits(sc.position[o][k]) == 0u) body += "        const float " + name + " = " + c + ";\n";
                else body += "        const float " + name + " = " + c + " - " + float_literal(sc.position[o][k]) + ";\n";
                return diff[c] = name;
            };
            for (int k : {(axis + 1) % 3, (axis + 2) % 3, axis})        // the varying axis last
                for (const auto& e : evals) difference(e[k], k);
            std::vector<std::array<std::string, 3>> locals(n);
            for (int k = 0; k < 3; k++)
                for (int t = 0; t < n; t++) {
                    const std::string d[3] = {diff[evals[t][0]], diff[evals[t][1]], diff[evals[t][2]]};
                    const FastCoordinate fc = fast_coordinate(sc, o, k, axis, d);
                    anyElided = anyElided || fc.elided;
                    auto it = local.find(fc.expr);
                    if (it != local.end()) { locals[t][k] = it->second; continue; }
                    const std::string name = format("dcsg_l%d_%d", k, (int)local.size());
                    local[fc.expr] = locals[t][k] = name;
                    body += "        const float " + name + " = " + fc.expr + ";\n";
                    if (fc.testAxis >= 0 && tested.insert({evals[t][fc.testAxis], float_bits(sc.position[o][fc.testAxis])}).second)
                        body += "        DCSG_BAD_UNLESS_ABS_GE(" + d[fc.testAxis] + ", 8.6736173798840355e-19f);\n";      // 2^-60
                    if (fc.testCore) body += "        DCSG_BAD_UNLESS_ABS_GT0(" + name + ");\n";
                }
            for (int t = 0; t < n; t++)
                body += format("        dcsg_s%d_%d = sdf_bank(float3(%s, %s, %s), (unsigned char)%d);\n", dst, t, locals[t][0].c_str(),
                               locals[t][1].c_str(), locals[t][2].c_str(), lhs & 0xff);
            body += "    }\n";
        } break;
        case 1:     // EXPORT
            if (!slot_ok(lhs)) { err = format("buildprocedure.txt command %d: bad EXPORT", i); return false; }
            used[lhs] = true;
            for (int t = 0; t < n; t++) body += format("    dcsg_out[%d] = dcsg_s%d_%d;\n", t, lhs, t);
            break;
        case 2: case 3:
            if (!slot_ok(lhs) || !slot_ok(rhs) || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad slot", i); return false; }
            used[lhs] = used[rhs] = used[dst] = true;
            for (int t = 0; t < n; t++)
                body += format("    dcsg_s%d_%d = %s(dcsg_s%d_%d,dcsg_s%d_%d);\n", dst, t, op == 2 ? "T_min" : "T_max", lhs, t, rhs, t);
            break;
        case 4: case 5:
            if (!slot_ok(lhs) || !slot_ok(dst)) { err = format("buildprocedure.txt command %d: bad slot", i); return false; }
            used[lhs] = used[dst] = true;
            for (int t = 0; t < n; t++) body += format("    dcsg_s%d_%d = %sdcsg_s%d_%d;\n", dst, t, op == 4 ? "-" : "", lhs, t);
            break;
        default:
            break;  // unknown opcodes fall through the reference's switch without effect
        }
    }
    const std::string c = comp[axis];
    out = format("\n// ---- generated by dcsg_build: the %s-taps of a normal%s, see generate_primary_sdf_axis ----\n", c.c_str(),
                 centre ? " and the centre" : "") +
          format("__device__ __forceinline__ void dcsg_primary_sdf_%s%s(float3 dcsg_v, float dcsg_e, float (&dcsg_out)[%d], bool& dcsg_inexact_out) {\n",
                 c.c_str(), centre ? "c" : "", n) +
          "    DCSG_BAD_DECLARE();\n";
    for (int k = 0; k < 3; k++) out += format("    const float dcsg_c%s0 = dcsg_v.%s;\n", comp[k], comp[k]);
    out += format("    const float dcsg_c%sp = dcsg_v.%s + dcsg_e;\n", c.c_str(), c.c_str());
    out += format("    const float dcsg_c%sm = dcsg_v.%s - dcsg_e;\n", c.c_str(), c.c_str());
    out += format("    DCSG_BAD_UNLESS_ABS_GT0(dcsg_c%s0);\n", c.c_str());
    if (anyElided)
        for (const char* v : {"0", "p", "m"}) out += format("    DCSG_BAD_UNLESS_ABS_LT(dcsg_c%s%s, 1.329227995784916e+36f);\n", c.c_str(), v);    // 2^120
    for (int t = 0; t < n; t++) out += format("    dcsg_out[%d] = MAX_DISTANCE;\n", t);
    for (int s = 0; s < DCSG_STACK_SLOTS; s++)
        if (used[s])
            for (int t = 0; t < n; t++) out += format("    float dcsg_s%d_%d = 0.0f;\n", s, t);
    out += body;
    out += "    DCSG_BAD_COMMIT(dcsg_inexact_out);\n}\n";
    return true;
}

// The object loop of the preview's shade (reference k1.cl:300-325) with the object table as immediates: every object's
// own SDF is evaluated at the hit point; the LAST object within SDF_EPSILON * TOLERANCE_FACTOR_MATERIAL decides the
// material (k1.cl:318-321), whose shader then receives the global point, that object's local point and the normal.
std::string generate_shade_objects(const Scene& sc) {
    std::string out = "\n// ---- generated by dcsg_build from scene.txt: preview material lookup ----\n"
                      "__device__ float3 dcsg_shade_objects(float3 dcsg_v, float3 dcsg_n, bool& dcsg_matched) {\n"
                      "    int dcsg_match = -1;\n    float3 dcsg_local = float3(0.0, 0.0, 0.0);\n";
    const std::string dnames[3] = {"dcsg_dx", "dcsg_dy", "dcsg_dz"};
    const char* comp[3] = {"x", "y", "z"};
    for (int o = 0; o < sc.num_objects; o++) {
        out += "    {\n";
        for (int k = 0; k < 3; k++) {
            if (float_bits(sc.position[o][k]) == 0u) out += format("        const float dcsg_d%s = dcsg_v.%s;\n", comp[k], comp[k]);
            else out += format("        const float dcsg_d%s = dcsg_v.%s - ", comp[k], comp[k]) + float_literal(sc.position[o][k]) + ";\n";
        }
        out += "        const float3 dcsg_abc = float3(" + dot_expression(sc.right[o], -1, dnames) + ", " + dot_expression(sc.up[o], -1, dnames) + ", " +
               dot_expression(sc.forward[o], -1, dnames) + ");\n";
        out += format("        const float dcsg_s = sdf_bank(dcsg_abc, (unsigned char)%d);\n", sc.shape_id[o]);
        out += format("        if (dcsg_s < SDF_EPSILON * TOLERANCE_FACTOR_MATERIAL) { dcsg_match = %d; dcsg_local = dcsg_abc; }\n    }\n", o);
    }
    out += "    dcsg_matched = dcsg_match != -1;\n    switch (dcsg_match) {\n";
    for (int o = 0; o < sc.num_objects; o++)
        out += format("    case %d: return shader_bank(dcsg_v, dcsg_local, dcsg_n, (unsigned char)%d);\n", o, sc.material_id[o] & 0xff);
    out += "    }\n    return float3(0.0, 0.0, 0.0);\n}\n";
    return out;
}

// fastPath: also emit namespace dcsg_fast (the checked copy the kernels evaluate through).  Designs with mutable
// program-scope variables stay exact-only: evaluating a point twice is not idempotent on their per-thread state.
bool scene_wants_fast_path(const Scene& sc) {
    const char* off = getenv("DCSG_EXACT_ONLY");
    return sc.private_words == 0 && !(off && off[0] == '1');
}

std::string assemble_source(const Scene& sc, bool fastPath, std::string& err, bool flagInShared, bool tapAxes) {
    std::string gen, genRow, gen7, genFast, genAxes;
    if (!generate_primary_sdf(sc, false, false, gen, err) || !generate_primary_sdf(sc, true, false, genRow, err) ||
        !generate_primary_sdf7(sc, gen7, err) || (fastPath && !generate_primary_sdf(sc, false, true, genFast, err)))
        return std::string();
    if (fastPath) {
        // per-axis forms: x with the centre (projection), x without it (normals alone), y, z
        for (int f = 0; f < 4; f++) {
            std::string one;
            if (!generate_primary_sdf_axis(sc, f == 0 ? 0 : f - 1, f == 0, one, err)) return std::string();
            genAxes += one;
        }
    }
    std::string src;
    src.reserve(1 << 17);
    src += format("#define DCSG_FAST_PATH %d\n", fastPath ? 1 : 0);
    if (fastPath && tapAxes) src += "#define DCSG_TAP_AXES 1\n";
    if (flagInShared) src += "#define DCSG_FLAG_PRED 0\n";
    src += kScenePrelude;
    src += "\nnamespace dcsg_exact {\n#define DCSG_SQRT_F32(x) ::sqrtf(x)\n";
    src += kSceneSqrtMath;
    src += "}  // namespace dcsg_exact\n";
    if (fastPath) {
        src += "\nnamespace dcsg_fast {\n#define DCSG_SQRT_F32(x) dcsg_sqrt_checked(x)\n";
        src += kSceneSqrtMath;
        src += "}  // namespace dcsg_fast\n";
    }
    src += kSceneParams;
    src += kSceneKernels;
    std::string user = sc.scene_cu;
    if (user.find("dcsg_init_private") == std::string::npos)        // scene.cu from an older emitter
        user += "\n__device__ __forceinline__ void dcsg_init_private() {}\n";
    src += "\nnamespace dcsg_exact {\n// ---- scene.cu (user brushes, emitted by scenecompiler.commit) ----\n";
    src += user;
    src += gen;
    src += genRow;
    src += gen7;
    src += generate_shade_objects(sc);
    src += "}  // namespace dcsg_exact\n";
    if (fastPath) {
        // The per-axis forms sit in a block of their own in front of the fast copy's scene text, so that block holds the same
        // two texts as the exact copy's.  They reach its brushes through a declaration of sdf_bank, whose signature
        // scenecompiler emits (a scene whose text does not match fails to compile here, and compile_scene keeps the loop).
        src += "\nnamespace dcsg_fast {\n__device__ float sdf_bank(float3 v, unsigned char shape_id);\n";
        src += genAxes;
        src += "}  // namespace dcsg_fast\n";
        src += "\nnamespace dcsg_fast {\n// ---- scene.cu once more, against the checked fast forms ----\n";
        src += user;
        src += genFast;
        src += "}  // namespace dcsg_fast\n";
    }
    return src;
}

// Compile the scene: with the checked fast copy when the design allows it, and -- should user text that compiles once
// not compile twice (it is pasted into two namespaces) -- exact-only, with a note in the log.
bool kernel_footprint(const std::vector<char>& cubin, const char* kernel, KernelFootprint& fp) {
    fp = KernelFootprint();
    const char* base = cubin.data();
    const size_t size = cubin.size();
    if (size < sizeof(Elf64_Ehdr) || memcmp(base, ELFMAG, SELFMAG) != 0 || base[EI_CLASS] != ELFCLASS64) return false;
    Elf64_Ehdr eh;
    memcpy(&eh, base, sizeof(eh));
    if (eh.e_shentsize != sizeof(Elf64_Shdr) || eh.e_shoff + (uint64_t)eh.e_shnum * sizeof(Elf64_Shdr) > size || eh.e_shstrndx >= eh.e_shnum) return false;
    std::vector<Elf64_Shdr> sh(eh.e_shnum);
    memcpy(sh.data(), base + eh.e_shoff, eh.e_shnum * sizeof(Elf64_Shdr));
    for (const Elf64_Shdr& s : sh)
        if (s.sh_type != SHT_NOBITS && s.sh_offset + s.sh_size > size) return false;
    auto cstr = [&](const Elf64_Shdr& table, uint32_t at) -> std::string {
        if (at >= table.sh_size) return std::string();
        const char* p = base + table.sh_offset + at;
        return std::string(p, strnlen(p, table.sh_size - at));
    };
    const std::string textName = std::string(".text.") + kernel;
    int text = -1, symtab = -1, info = -1;
    for (int i = 0; i < (int)sh.size(); i++) {
        const std::string name = cstr(sh[eh.e_shstrndx], sh[i].sh_name);
        if (name == textName) text = i;
        else if (sh[i].sh_type == SHT_SYMTAB) symtab = i;
        else if (name == ".nv.info") info = i;
    }
    if (text < 0 || symtab < 0 || info < 0 || sh[symtab].sh_link >= sh.size() || sh[symtab].sh_entsize != sizeof(Elf64_Sym)) return false;
    fp.textBytes = sh[text].sh_size;
    // the kernel's symbol, and every function whose code lies in its text section (callees that are not inlined)
    std::set<uint32_t> inText;
    uint32_t kernelSym = UINT32_MAX;
    for (uint64_t off = 0; off + sizeof(Elf64_Sym) <= sh[symtab].sh_size; off += sizeof(Elf64_Sym)) {
        Elf64_Sym sym;
        memcpy(&sym, base + sh[symtab].sh_offset + off, sizeof(sym));
        const uint32_t idx = (uint32_t)(off / sizeof(Elf64_Sym));
        if (sym.st_shndx != text || ELF64_ST_TYPE(sym.st_info) != STT_FUNC) continue;
        inText.insert(idx);
        if (cstr(sh[sh[symtab].sh_link], sym.st_name) == kernel) kernelSym = idx;
    }
    if (kernelSym == UINT32_MAX) return false;
    // .nv.info: records of {u8 format, u8 attribute, u16 value-or-size}; format 4 (EIFMT_SVAL) carries `size` bytes after
    // the header.  EIATTR_REGCOUNT (0x2f) and EIATTR_FRAME_SIZE (0x11) are SVALs of {u32 symbol, u32 value}.
    const char* p = base + sh[info].sh_offset;
    const char* end = p + sh[info].sh_size;
    while (p + 4 <= end) {
        const uint8_t format = (uint8_t)p[0], attribute = (uint8_t)p[1];
        uint16_t value;
        memcpy(&value, p + 2, 2);
        const uint32_t payload = format == 4 ? value : 0u;
        if (p + 4 + payload > end) return false;
        if (format == 4 && payload >= 8 && (attribute == 0x2f || attribute == 0x11)) {
            uint32_t sym, v;
            memcpy(&sym, p + 4, 4);
            memcpy(&v, p + 8, 4);
            if (attribute == 0x2f && sym == kernelSym) fp.registers = (int)v;
            if (attribute == 0x11 && inText.count(sym)) fp.frameBytes = std::max(fp.frameBytes, v);
        }
        p += 4 + payload;
    }
    return fp.registers >= 0;
}

// The per-axis tap form earns its place when dcsg_k_project stays within 64 registers (four resident blocks of 256 threads:
// __launch_bounds__ in scene_kernels.cuh), without local memory, and with text small enough for the instruction cache.
// The projection kernel on sm_100a, rolled loop -> per-axis form (DESIGN.md 3b): Design1 23.4 -> 36.6 KiB of code at 64
// registers, projection 7.83 -> 6.48 ms at 1024^3 on a B200; the Hilbert design (design2) 37.2 -> 108.1 KiB, 12.75 -> 15.52 ms
// (instruction cache misses); synth64 22.6 -> 38.8 KiB; the stress scene and the random* scenes spill at 64 registers.
static const uint64_t kAxisTextLimit = 64 * 1024;

// Empty when the per-axis form of this cubin fits the budget, else why not.
static std::string axis_form_misfit(const std::vector<char>& cubin) {
    KernelFootprint fp;
    if (!kernel_footprint(cubin, "dcsg_k_project", fp)) return "the footprint of dcsg_k_project could not be read from the cubin";
    if (fp.registers > 64) return format("dcsg_k_project needs %d registers (budget 64)", fp.registers);
    if (fp.frameBytes > 0) return format("dcsg_k_project has a stack frame of %u bytes (local memory)", fp.frameBytes);
    if (fp.textBytes > kAxisTextLimit)
        return format("dcsg_k_project is %.1f KiB of code (limit %.0f KiB)", fp.textBytes / 1024.0, kAxisTextLimit / 1024.0);
    return std::string();
}

// DCSG_TAP_FORM=loop / axis forces the tap form of the fast copy (to compare the two); unset, the footprint decides.
bool compile_scene(const Scene& sc, std::vector<char>& cubin, std::string& log, std::string& err, bool exactOnly) {
    if (!exactOnly && scene_wants_fast_path(sc)) {
        const char* form = getenv("DCSG_TAP_FORM");
        const bool loopForced = form && strcmp(form, "loop") == 0, axisForced = form && strcmp(form, "axis") == 0;
        std::string loopNote;
        if (!loopForced) {
            const std::string src = assemble_source(sc, true, err, false, true);
            if (src.empty()) return false;
            std::string misfit;
            if (compile_source(src, cubin, log)) {
                misfit = axis_form_misfit(cubin);
                if (misfit.empty() || axisForced) return true;
            } else {
                misfit = "the per-axis form did not compile";
            }
            loopNote = "[dcsg] the normals keep the rolled tap loop: " + misfit + "\n";
        }
        const std::string src = assemble_source(sc, true, err);
        if (src.empty()) return false;
        if (compile_source(src, cubin, log)) { log = loopNote + log; return true; }
        // The fast copy keeps its flag in a PTX predicate register of the kernel (scene_prelude.cuh), which needs every
        // function of the copy inlined into the kernels; text that does not inline still builds with the flag in shared memory.
        std::string sharedLog;
        const std::string sharedSrc = assemble_source(sc, true, err, true);
        if (!sharedSrc.empty() && compile_source(sharedSrc, cubin, sharedLog)) {
            log = "[dcsg] the fast copy's flag is kept in shared memory for this design\n" + sharedLog;
            return true;
        }
        std::string exactLog;
        const std::string exactSrc = assemble_source(sc, false, err);
        if (!exactSrc.empty() && compile_source(exactSrc, cubin, exactLog)) {
            log = "[dcsg] the checked fast copy of the scene did not compile; built exact-only\n" + exactLog;
            return true;
        }
        return false;       // log holds the first attempt's diagnostics
    }
    const std::string src = assemble_source(sc, false, err);
    return !src.empty() && compile_source(src, cubin, log);
}

// NVRTC -> cubin for sm_100a.  --fmad=false: parity mode, one IEEE op per source op (DESIGN.md).
bool compile_source(const std::string& src, std::vector<char>& cubin, std::string& log) {
    nvrtcProgram prog;
    if (nvrtcCreateProgram(&prog, src.c_str(), "dcsg_scene.cu", 0, nullptr, nullptr) != NVRTC_SUCCESS) {
        log = "nvrtcCreateProgram failed";
        return false;
    }
    std::vector<std::string> opts = {"--gpu-architecture=sm_100a", "--std=c++17", "-default-device", "-lineinfo",
                                     "--prec-sqrt=true", "--prec-div=true",
                                     format("-DDCSG_LATTICE_SPT=%d", DCSG_LATTICE_SPT)};
    if (const char* extra = getenv("DCSG_NVRTC_EXTRA")) {      // developer knob: extra NVRTC options, space separated
        std::string e(extra);
        size_t pos = 0;
        while (pos < e.size()) {
            size_t sp = e.find(' ', pos);
            if (sp == std::string::npos) sp = e.size();
            if (sp > pos) opts.push_back(e.substr(pos, sp - pos));
            pos = sp + 1;
        }
    }
    const char* fast = getenv("DCSG_FAST_MATH");
    opts.push_back((fast && fast[0] == '1') ? "--fmad=true" : "--fmad=false");
    std::vector<const char*> copts;
    for (auto& o : opts) copts.push_back(o.c_str());
    nvrtcResult rc = nvrtcCompileProgram(prog, (int)copts.size(), copts.data());
    size_t logSize = 0;
    nvrtcGetProgramLogSize(prog, &logSize);
    log.assign(logSize ? logSize - 1 : 0, '\0');
    if (logSize > 1) nvrtcGetProgramLog(prog, &log[0]);
    if (rc != NVRTC_SUCCESS) {
        log += format("\n[nvrtc] %s", nvrtcGetErrorString(rc));
        nvrtcDestroyProgram(&prog);
        return false;
    }
    size_t size = 0;
    nvrtcGetCUBINSize(prog, &size);
    cubin.resize(size);
    nvrtcGetCUBIN(prog, cubin.data());
    nvrtcDestroyProgram(&prog);
    return size > 0;
}

void copy_log(const std::string& log, char* out, size_t cap) {
    if (!out || cap == 0) return;
    size_t n = std::min(cap - 1, log.size());
    memcpy(out, log.data(), n);
    out[n] = '\0';
}

}  // namespace dcsg_host

