// Operand splits of the tcgen05 BMU kernels (sm_100a): the arithmetic that makes the error-compensated products
// exact on the lattice of DESIGN.md §2.  tests/test_exact_lattice_host.py, test_f16_input_host.py and
// test_bf16_input_host.py emulate these rules on the host; every kernel and pre-pass uses the one definition here.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include "som_tc_ptx.cuh"

namespace som {
namespace tc {

// TF32 hi/lo split: hi = RNA TF32 part, lo = TF32-rounded remainder (the dropped lo.lo term is 2^-24 relative)
__device__ __forceinline__ void tf32_split(float v, float& hi, float& lo) {
    hi = tf32_rna(v);
    lo = tf32_rna(v - hi);
}
__device__ __forceinline__ void tf32_split4(const float* v, float4& hi, float4& lo) {
    tf32_split(v[0], hi.x, lo.x);
    tf32_split(v[1], hi.y, lo.y);
    tf32_split(v[2], hi.z, lo.z);
    tf32_split(v[3], hi.w, lo.w);
}
// TF32 three-way split of a squared norm, n1 + n2 + n3 (the norm tail k-step)
__device__ __forceinline__ void tf32_norm_split3(float nrm, float& n1, float& n2, float& n3) {
    n1 = tf32_rna(nrm);
    n2 = tf32_rna(nrm - n1);
    n3 = tf32_rna(nrm - n1 - n2);
}

// FP16 hi/lo split of an already scaled value: hi = fp16(v), lo = v - hi (exact in fp32; rounded to FP16 when packed)
__device__ __forceinline__ void f16_split(float v, float& hi, float& lo) {
    hi = __half2float(__float2half_rn(v));
    lo = v - hi;
}
// FP16 three-way split of a scaled squared norm: n1, n2 in FP16, n3 the fp32 remainder (rounded to FP16 when stored)
__device__ __forceinline__ void f16_norm_split3(float nrm, float& n1, float& n2, float& n3) {
    n1 = __half2float(__float2half_rn(nrm));
    n2 = __half2float(__float2half_rn(nrm - n1));
    n3 = nrm - n1 - n2;
}
// FP16 power-of-two row scale from the row's largest magnitude mx and the exponent tc_exp of the codebook's norm scale
// t_c: max |s_p x| in [64, 128) as long as a_p = s_p / t_c is an exact FP16 power of two (2^-24 .. 2^15); an all-zero
// or non-finite row takes the ideal exponent 0.  Returns s_p = 2^es and the tail operand a_p.
__device__ __forceinline__ void f16_row_scale(float mx, int tc_exp, float& sp, float& ap, int& es) {
    const int eb = (int)((__float_as_uint(mx) >> 23) & 0xffu);
    int ep = 133 - eb;
    if (!(mx > 0.f) || eb == 0xff) ep = 0;
    int ka = ep - tc_exp;
    if (ka < -24) {
        // |x| beyond ~2^24 |c|: ||c||^2 is below fp32 resolution of rd; keep the row in range instead
        es = ep;
        ap = 0.f;
    } else {
        ka = ka > 15 ? 15 : ka;                 // 2^-24 .. 2^15: exact in FP16 (subnormal below 2^-14)
        es = ka + tc_exp;
        ap = __uint_as_float((uint32_t)(127 + ka) << 23);
    }
    es = es > 120 ? 120 : (es < -120 ? -120 : es);
    sp = __uint_as_float((uint32_t)(127 + es) << 23);
}

// eight halves (one 16-byte swizzle chunk) from eight floats, round-to-nearest-even
__device__ __forceinline__ uint4 pack_h8(const float (&v)[8]) {
    __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
    __half2 c = __floats2half2_rn(v[4], v[5]), d = __floats2half2_rn(v[6], v[7]);
    return make_uint4(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b),
                      *reinterpret_cast<uint32_t*>(&c), *reinterpret_cast<uint32_t*>(&d));
}

}  // namespace tc
}  // namespace som
