// sqrt_checked.cu -- TEST HARNESS (device).  dcsg_sqrt_checked against IEEE sqrtf over every float bit pattern.
//
// The checked square root of the fast copy (scene_prelude.cuh) runs MUFU.RSQ and one Newton step without the range test of
// IEEE sqrtf and raises the thread's flag when its result says the input was outside [2^-101, FLT_MAX].  tests/
// test_projection_kernel.py cuts dcsg_sqrt_checked, dcsg_flag_init and dcsg_flag_take (predicate form) out of the
// prelude, pastes them into PRELUDE_INC and compiles this file for sm_100a with -fmad=false -prec-sqrt=true, so that
// ::sqrtf is the correctly rounded square root.  The sweep counts on the device and returns:
//   [0] unflagged inputs whose result differs from ::sqrtf (bit for bit)
//   [1] NaN, +-Inf, +-0, negative and denormal inputs that were NOT flagged
//   [2] flagged positive normal inputs;  [3] the smallest and [4] the largest of their bit patterns
//   [5] inputs swept
//   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -prec-sqrt=true -shared -Xcompiler -fPIC -DPRELUDE_INC=...
#include <cstdint>
#include <cuda_runtime.h>

#define DCSG_DEV __device__ __forceinline__
#define DCSG_FLAG_PRED 1
#include PRELUDE_INC

__global__ void sweep(unsigned long long* out) {
    dcsg_flag_init();
    unsigned long long wrong = 0, missed = 0, flaggedNormal = 0, swept = 0;
    unsigned lo = 0xffffffffu, hi = 0u;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += stride) {
        const unsigned u = (unsigned)i;
        const float x = __uint_as_float(u);
        const float s = dcsg_sqrt_checked(x);
        const bool flagged = dcsg_flag_take();
        const float ref = ::sqrtf(x);
        const unsigned mag = u & 0x7fffffffu;
        const bool mustFlag = mag >= 0x7f800000u || mag < 0x00800000u || (u >> 31) != 0u;    // NaN, Inf, zero, denormal, negative
        if (!flagged && __float_as_uint(s) != __float_as_uint(ref)) ++wrong;
        if (mustFlag && !flagged) ++missed;
        if (!mustFlag && flagged) {
            ++flaggedNormal;
            lo = min(lo, u);
            hi = max(hi, u);
        }
        ++swept;
    }
    atomicAdd(&out[0], wrong);
    atomicAdd(&out[1], missed);
    atomicAdd(&out[2], flaggedNormal);
    atomicMin(&out[3], (unsigned long long)lo);
    atomicMax(&out[4], (unsigned long long)hi);
    atomicAdd(&out[5], swept);
}

__global__ void plain_sqrt(const float* x, unsigned long long n, float* y) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = ::sqrtf(x[i]);
}

// 0, or the CUDA error code
extern "C" int sqrt_checked_sweep(unsigned long long* host_out) {
    unsigned long long init[6] = {0, 0, 0, 0xffffffffull, 0, 0};
    unsigned long long* d = nullptr;
    cudaError_t e = cudaMalloc(&d, sizeof(init));
    if (e == cudaSuccess) e = cudaMemcpy(d, init, sizeof(init), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        sweep<<<148 * 16, 256>>>(d);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(host_out, d, sizeof(init), cudaMemcpyDeviceToHost);
    if (d) cudaFree(d);
    return (int)e;
}

// device ::sqrtf of n host floats
extern "C" int device_sqrtf(const float* host_x, unsigned long long n, float* host_y) {
    float *dx = nullptr, *dy = nullptr;
    cudaError_t e = cudaMalloc(&dx, n * 4);
    if (e == cudaSuccess) e = cudaMalloc(&dy, n * 4);
    if (e == cudaSuccess) e = cudaMemcpy(dx, host_x, n * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        plain_sqrt<<<(unsigned)((n + 255) / 256), 256>>>(dx, n, dy);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(host_y, dy, n * 4, cudaMemcpyDeviceToHost);
    if (dx) cudaFree(dx);
    if (dy) cudaFree(dy);
    return (int)e;
}
