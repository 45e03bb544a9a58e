// The training step's update rules, one definition each, for every kernel that applies them: the separate-kernel step
// (som_core.cu, som_filter*.cu, som_accumulate.cu), the one-kernel step (som_step_small.cu) and the multi-GPU peer tail
// (som_peer.cu, som_peer.cuh).  The outputs of those paths are compared bit for bit, so a rule changes here or nowhere.
#pragma once
#include "som_common.cuh"

namespace som {

// ---- Adam: torch.optim.Adam's single-tensor rule (lerp form of the first moment) -----------------------------------
struct AdamScalars { float w1, b2, one_m_b2, step_size, bc2_sqrt, eps; };

// The bias corrections of step t (1-based) in double as torch/optim/adam.py computes them, then narrowed.  Host and
// device `pow` may differ in the last bit, so each caller keeps the side it evaluates this on: som_adam_f32 the host,
// the kernels that read the step count from device memory the device.
__host__ __device__ __forceinline__ AdamScalars adam_scalars(double lr, double b1, double b2, float eps, double t) {
    AdamScalars a;
    a.w1 = (float)(1.0 - b1);
    a.b2 = (float)b2;
    a.one_m_b2 = (float)(1.0 - b2);
    a.step_size = (float)(lr / (1.0 - pow(b1, t)));
    a.bc2_sqrt = (float)sqrt(1.0 - pow(b2, t));
    a.eps = eps;
    return a;
}

__device__ __forceinline__ void adam_update(const AdamScalars& a, float gi, float& mi, float& vi, float& wi) {
    const float diff = gi - mi;
    // torch lerp: weight < 0.5 ? start + w*diff : end - diff*(1-w)
    mi = (a.w1 < 0.5f) ? __fmaf_rn(a.w1, diff, mi) : __fmaf_rn(-diff, 1.0f - a.w1, gi);
    vi = __fmaf_rn(a.one_m_b2 * gi, gi, vi * a.b2);
    const float denom = __fdiv_rn(__fsqrt_rn(vi), a.bc2_sqrt) + a.eps;
    wi = __fmaf_rn(-a.step_size, __fdiv_rn(mi, denom), wi);
}

// four weights of one 16-byte access per stream.  SCALED: the gradient arrives unscaled and each element is multiplied
// by gscale first (one fp32 rounding)
template <bool SCALED>
__device__ __forceinline__ void adam_update4(const AdamScalars& a, const float4& g, float gscale, float4& m, float4& v,
                                             float4& w) {
    adam_update(a, SCALED ? g.x * gscale : g.x, m.x, v.x, w.x);
    adam_update(a, SCALED ? g.y * gscale : g.y, m.y, v.y, w.y);
    adam_update(a, SCALED ? g.z * gscale : g.z, m.z, v.z, w.z);
    adam_update(a, SCALED ? g.w * gscale : g.w, m.w, v.w, w.w);
}

// ---- Gaussian neighbourhood: w(t) = expf(-(float(t*t) / two_var)), exactly as the reference generates it -----------
// models/Codebook.py:118 -- Python double arithmetic, then one rounding to fp32 at the divide
static inline float filter_two_var(double neighbourhood_range) {
    const double variance = -(neighbourhood_range / (2.0 * log(0.1)));
    return (float)(2.0 * variance);
}

// the band half-width h: the largest t with w(t) > 0, found on the host with the same fp32 steps (SURVEY 0.7)
static inline int filter_band_half_width(float two_var, int K) {
    // expf underflows to 0 below about -103.98; search a small window around that root
    const double guess = sqrt(104.5 * (double)two_var);
    long long t = (long long)guess + 2;
    if (t > K) t = K;                      // rows further than K-1 apart never meet
    while (t > 0) {
        const float sq = (float)(t * t);
        if (expf(-(sq / two_var)) > 0.f) break;
        --t;
    }
    return (int)t;
}

// w(at) for 0 <= at <= h, zero outside the band: t^2 exact in integers, converted to fp32, divided by fp32(two_var),
// negated, expf
__device__ __forceinline__ float band_weight(int at, int h, float two_var) {
    return at <= h ? expf(-(__fdiv_rn((float)((long long)at * (long long)at), two_var))) : 0.f;
}

// ---- the packed tail [sse_hi, sse_lo, n / 4096, n % 4096] of the accumulator buffer ---------------------------------
// The fp64 squared error as a float pair and the patch count as two exactly representable floats, so that ONE fp32
// sum over the ranks of [Rbar | tail] carries them too.
__device__ __forceinline__ float4 pack_tail(double sse, int64_t n) {
    const float hi = (float)sse;
    return make_float4(hi, (float)(sse - (double)hi), (float)(n >> 12), (float)(n & 4095));
}

// the patch count of a tail, or of a sum of tails, from its two count fields
__device__ __forceinline__ double tail_count(double hi, double lo) { return hi * 4096.0 + lo; }

// What the Adam tail reads from a reduced tail: numel = D * (global patch count), the gradient scale (float)(2 / numel)
// -- the same single rounding as the filter's own `scale * acc` epilogue, so the result is bit-identical to the
// host-scaled path -- and the mean squared error.
struct TailTotals { double numel; float gscale; };
__device__ __forceinline__ TailTotals tail_totals(const float* tail, int D) {
    const double numel = tail_count((double)tail[2], (double)tail[3]) * (double)D;
    return {numel, (float)(2.0 / numel)};
}
__device__ __forceinline__ double tail_loss(const float* tail, double numel) {
    return ((double)tail[0] + (double)tail[1]) / numel;
}

}  // namespace som
