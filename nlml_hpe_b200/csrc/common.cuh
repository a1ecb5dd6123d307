// Shared plumbing for the C ABI: error reporting, device guard, pinned staging; the device statement of the reference's
// IPD normalisation of raw landmarks.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../include/nlml_hpe_b200.h"

namespace nlml {

inline char* last_error_buf() {
    static thread_local char buf[512] = "";
    return buf;
}
inline int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(last_error_buf(), 512, fmt, ap);
    va_end(ap);
    return code;
}

#define NLML_CUDA(expr)                                                                          \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return nlml::set_error((int)_e, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                   __FILE__, __LINE__);                                          \
    } while (0)

// Select `device` for the scope, restore the previous one on exit.
struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = cudaSetDevice(device) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

inline int check_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_error(NLML_E_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                         e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= n) return set_error(NLML_E_INVALID, "device %d out of range [0,%d)", device, n);
    cudaDeviceProp prop;
    NLML_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return set_error(NLML_E_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                         prop.major, prop.minor);
    return 0;
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------------
// IPD normalisation of RAW MediaPipe landmarks (x,y,z of landmark i at columns 3i..3i+2), the arithmetic of
// FeatureExtractor.Read_Landmarks_and_Normalizing_using_IPD (helpers/FeatureExtractor.py:30-66, with the nose-tip
// reference point of :89-90 and the .float() of :105): subtract landmark 1, divide by the inter-pupillary distance
// ||landmark 33 - landmark 263|| (1e-6 when zero), in FLOAT64 as the reference's Python floats, then round to float32.
// Every kernel that accepts raw landmarks (the Encoder+heads operand split, the Tucker phase-A loads, the Powell fit's
// staging of x) applies it through ipd_row / ipd_map, so both halves of the library see bit-identical features.
// A row must hold columns 0..791 (landmark 263).
// ---------------------------------------------------------------------------------------------
struct IpdRow {
    double ref[3];   // landmark 1
    double ipd;      // ||landmark 33 - landmark 263||, 1e-6 when zero
};
__device__ __forceinline__ IpdRow ipd_row(const float* __restrict__ row) {
    IpdRow r;
    r.ref[0] = (double)__ldg(row + 3);
    r.ref[1] = (double)__ldg(row + 4);
    r.ref[2] = (double)__ldg(row + 5);
    const double dx = (double)__ldg(row + 99) - (double)__ldg(row + 789);
    const double dy = (double)__ldg(row + 100) - (double)__ldg(row + 790);
    const double dz = (double)__ldg(row + 101) - (double)__ldg(row + 791);
    const double ipd = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
    r.ipd = ipd == 0.0 ? 1e-6 : ipd;
    return r;
}
// value x of column f of the row, coord = f % 3
__device__ __forceinline__ float ipd_map(float x, const IpdRow& r, int coord) {
    const double ref = coord == 0 ? r.ref[0] : (coord == 1 ? r.ref[1] : r.ref[2]);   // selects: no local-memory array
    return __double2float_rn(__ddiv_rn(__dsub_rn((double)x, ref), r.ipd));
}
// four consecutive columns f..f+3 of a row; columns >= F are padding and stay as they are
__device__ __forceinline__ float4 ipd_map4(float4 v, const IpdRow& r, int f, int F) {
    if (f + 0 < F) v.x = ipd_map(v.x, r, (f + 0) % 3);
    if (f + 1 < F) v.y = ipd_map(v.y, r, (f + 1) % 3);
    if (f + 2 < F) v.z = ipd_map(v.z, r, (f + 2) % 3);
    if (f + 3 < F) v.w = ipd_map(v.w, r, (f + 3) % 3);
    return v;
}
// in place on a staged, transposed tile of X: tile[f * ld + s] = feature f0 + f of sample s (f < fc, s < nsamp), sample
// s's (ref, ipd) at c[s]; samples >= nrows and features >= F are padding and stay zero.  A separate pass, one element at a time: the float64 division stays out of the register budget
// of the accumulation loop that follows.
__device__ __forceinline__ void ipd_tile(float* tile, int ld, int fc, int nsamp, const IpdRow* c, long long nrows, int f0, int F,
                                         int tid, int nthreads) {
#pragma unroll 1
    for (int idx = tid; idx < fc * nsamp; idx += nthreads) {
        const int f = idx / nsamp, s = idx % nsamp;
        if (s < nrows && f0 + f < F) tile[f * ld + s] = ipd_map(tile[f * ld + s], c[s], (f0 + f) % 3);
    }
}

}  // namespace nlml
