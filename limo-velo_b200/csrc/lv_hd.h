/*
 * lv_hd.h — host/device portability macros and the fp32 "reference arithmetic" primitives.
 *
 * The reference is built "-std=c++14 -O3" for baseline x86-64 (CMakeLists.txt:8,16): single
 * precision products and sums are rounded separately (no FMA contraction).  The fp32 part of
 * the path (world transform, squared distances, plane fit, gates) decides discrete outcomes
 * (neighbour sets, accepted matches), so device code reproduces exactly that arithmetic:
 * every fp32 multiply/add goes through lv::fmul / lv::fadd (= __fmul_rn / __fadd_rn on the
 * device, plain operators under "-ffp-contract=off" on the host).
 *
 * The same headers compile for the host (g++) so that tests/cpu_shim can unit-test the device
 * math without a GPU.  That host build is test-only and is not reachable from the C ABI.
 */
#ifndef LV_HD_H_
#define LV_HD_H_

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define LV_HD __host__ __device__ __forceinline__
#define LV_HD_NOINLINE __host__ __device__ inline
/* out of line on the device as well: rare or single-thread code that would otherwise take registers and
 * instruction-cache space from the kernel it is called in */
#define LV_HD_COLD __host__ __device__ inline __noinline__
#else
#define LV_HD inline
#define LV_HD_NOINLINE inline
#define LV_HD_COLD inline
#endif

namespace lv {

LV_HD float fmul(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
LV_HD float fadd(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
LV_HD float fsub(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fsub_rn(a, b);
#else
    return a - b;
#endif
}
LV_HD float fdiv(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fdiv_rn(a, b);
#else
    return a / b;
#endif
}
LV_HD float fsqrt(float a) {
#if defined(__CUDA_ARCH__)
    return __fsqrt_rn(a);
#else
    return sqrtf(a);
#endif
}
LV_HD double dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
LV_HD double dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
LV_HD double dsub(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}

/* (a0*b0 + a1*b1) + a2*b2, the evaluation order of a 3-term Eigen dot product */
LV_HD float dot3f(float a0, float a1, float a2, float b0, float b1, float b2) {
    return fadd(fadd(fmul(a0, b0), fmul(a1, b1)), fmul(a2, b2));
}
LV_HD double dot3d(double a0, double a1, double a2, double b0, double b1, double b2) {
    return dadd(dadd(dmul(a0, b0), dmul(a1, b1)), dmul(a2, b2));
}

}  // namespace lv
#endif
