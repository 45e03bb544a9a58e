// Pieces of the peer-memory tail (som_peer.cu) that other translation units fuse into their own kernels: the in-switch
// reducing load and the exact reduction of the packed buffer's 4-float tail.
#pragma once
#include "som_common.cuh"
#include "som_step_rules.cuh"

namespace som {
namespace peer {

constexpr int MAX_WORLD = 16;
struct Pads { uint32_t* p[MAX_WORLD]; };       // one peer-mapped address per rank (flag areas: layout at counter_of())

__device__ __forceinline__ float4 mm_ld_reduce(const float* mc) {
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
    return v;
}

// The 4-float tail (pack_tail, som_step_rules.cuh) of the packed accumulator buffer is NOT reduced in the
// switch: the in-switch fp32 adder is not exact enough for the loss (measured 1.2e-6 relative over 8 ranks), and the
// patch count must be exact.  Every rank reads the R tails through the peer addresses and adds them in rank order,
// the squared error in fp64 -- the same bits on every rank.
__device__ __forceinline__ float4 exact_tail(const Pads& bufs, int64_t q_tail, int world) {
    double sse = 0.0, cnt_hi = 0.0, cnt_lo = 0.0;
    // eight peer loads in flight, then the sums in rank order: issued one by one behind the fp64 adds that consume
    // them, the loads were a chain of `world` NVLink round trips on the single thread every caller waits for
    for (int r0 = 0; r0 < world; r0 += 8) {
        float4 t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            t[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + u < world) {
                const float* p = reinterpret_cast<const float*>(bufs.p[r0 + u]) + 4 * q_tail;
                asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];"
                             : "=f"(t[u].x), "=f"(t[u].y), "=f"(t[u].z), "=f"(t[u].w) : "l"(p) : "memory");
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (r0 + u < world) {
                sse += (double)t[u].x + (double)t[u].y;
                cnt_hi += (double)t[u].z;
                cnt_lo += (double)t[u].w;
            }
        }
    }
    // the summed count is an exact integer in fp64
    return pack_tail(sse, (int64_t)tail_count(cnt_hi, cnt_lo));
}


}  // namespace peer
}  // namespace som
