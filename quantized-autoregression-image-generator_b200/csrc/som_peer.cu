// Data-parallel tail of the SOM step over NVLink / NVSwitch peer memory (sm_100a, one process per GPU).
//
// The reference has no multi-GPU code; this replaces, ACROSS ranks, what train_codebook.py:240-242 (backward + Adam
// step) and models/Codebook.py:112-130 (the Gaussian S @ W) do on one device after the per-unit accumulators of every
// rank exist (som_accumulate_packed_nchw_f32).  Instead of "NCCL all-reduce, then every rank filters and updates the
// whole codebook", every rank owns a contiguous slice of units [lo, hi):
//
//   peer_reduce_rows   in-switch reduction (multimem.ld_reduce.add.f32 on the NVSwitch multicast address) of ONLY the
//                      accumulator rows this rank needs, its slice plus the filter's halo, into local memory -- the
//                      reduce-scatter half of an all-reduce, with overlap; the 4-float tail (loss numerator, global
//                      patch count) is reduced by every rank
//   (som_filter_ws_f32 on the slice + halo: G = T @ Rbar for the owned rows)
//   adam_slice_bcast   Adam on the owned rows and multimem.st of the new rows into EVERY rank's codebook -- the
//                      all-gather half, fused into the update's store
//   peer_bcast_rows    the same broadcast for the rows of W~ = T @ W a rank computed for its slice
//   peer_allreduce     plain in-place all-reduce (ld_reduce + multimem.st of a 1/R slice per rank) for the case where
//                      slicing does not pay (halo >= slice)
//
// Synchronisation between ranks: one 32-bit flag per (channel, sender) in every rank's peer-mapped flag area --
// compare-and-swap 0 -> 1 by the sender, 1 -> 0 by the receiver, system scope, so the flags reset themselves and the
// kernels replay from a CUDA graph.  A kernel that must publish its stores lets its LAST block (local arrival
// counter) run the exchange for the whole grid; a kernel that must see the peers' earlier work is preceded by a
// one-block barrier kernel.  `world` remote atomics per barrier (a first version synchronised every block with its peer
// blocks: blocks x world NVLink atomics per kernel).  Spins are bounded (~4 s): a missing peer traps instead of hanging.
// Buffers are caller-owned symmetric (peer-mapped + multicast) allocations; the library keeps no pointers.
#include "som_common.cuh"
#include "som_peer.cuh"

namespace som {
SOM_TRACE_TU(trace_set_peer)
namespace peer {

constexpr int THREADS = 512;


__device__ __forceinline__ uint64_t gtimer() {
    uint64_t v;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v)::"memory");
    return v;
}
template <int SEM>   // 0 relaxed, 1 release, 2 acquire
__device__ __forceinline__ uint32_t cas_sys(uint32_t* addr, uint32_t cmp, uint32_t val) {
    uint32_t old;
    if (SEM == 1) asm volatile("atom.global.release.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(addr), "r"(cmp), "r"(val) : "memory");
    else if (SEM == 2) asm volatile("atom.global.acquire.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(addr), "r"(cmp), "r"(val) : "memory");
    else asm volatile("atom.global.relaxed.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(addr), "r"(cmp), "r"(val) : "memory");
    return old;
}
// The cross-rank barrier of a whole GRID: the last block to arrive (local arrival counter, wraps to zero by itself) runs
// the rank-to-rank signal exchange on behalf of all blocks, so a kernel costs `world` remote atomics instead of
// blocks x world (measured at 8 ranks: the per-block form spent most of the tail's time in NVLink atomics).
// Call after the block's global / multicast stores; `counter` is a zero-initialised word of this rank's flag area.
// Returns true in the block that ran the exchange (the last one to arrive).
template <bool PREV, bool NEXT>
__device__ __forceinline__ bool grid_sync_ranks(const Pads& pads, uint32_t* counter, int channel, int rank, int world) {
    __shared__ int is_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();                                  // this block's stores before the arrival
        is_last = atomicInc(counter, gridDim.x - 1) == gridDim.x - 1;
    }
    __syncthreads();
    if (is_last) {
        if ((int)threadIdx.x < world) {
            __threadfence_system();
            const int peer = threadIdx.x;
            const uint64_t deadline = gtimer() + 4000000000ull;
            uint32_t* put = pads.p[peer] + (size_t)channel * MAX_WORLD + rank;
            while (cas_sys<PREV ? 1 : 0>(put, 0u, 1u) != 0u)
                if (gtimer() > deadline) __trap();
            uint32_t* get = pads.p[rank] + (size_t)channel * MAX_WORLD + peer;
            while (cas_sys<NEXT ? 2 : 0>(get, 1u, 0u) != 1u)
                if (gtimer() > deadline) __trap();
        }
    }
    return is_last != 0;
}

// one-block barrier over the ranks: everything this rank enqueued before it is visible to the peers' later kernels
__global__ void __launch_bounds__(32) barrier_kernel(Pads pads, int channel, int rank, int world) {
    pdl_begin();
    trace_stamp(s_trace_buf, 13);
    if ((int)threadIdx.x < world) {
        __threadfence_system();
        const int peer = threadIdx.x;
        const uint64_t deadline = gtimer() + 4000000000ull;
        uint32_t* put = pads.p[peer] + (size_t)channel * MAX_WORLD + rank;
        while (cas_sys<1>(put, 0u, 1u) != 0u)
            if (gtimer() > deadline) __trap();
        uint32_t* get = pads.p[rank] + (size_t)channel * MAX_WORLD + peer;
        while (cas_sys<2>(get, 1u, 0u) != 1u)
            if (gtimer() > deadline) __trap();
    }
    __syncwarp();
    trace_stamp(s_trace_buf, 113);                               // every peer has arrived
}

__device__ __forceinline__ void mm_st(float* mc, const float4& v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
                 ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// in-place all-reduce of n4 float4 at the multicast address: rank r reduces and re-broadcasts quads [q0, q1);
// q_tail >= 0: that quad is the packed buffer's tail, excluded from the in-switch part and summed exactly
__global__ void __launch_bounds__(THREADS) allreduce_kernel(float* mc, int64_t q0, int64_t q1, int64_t q_tail,
                                                            float4* __restrict__ tail_out, Pads bufs, Pads pads,
                                                            uint32_t* counter, int channel, int rank, int world) {
    pdl_begin();
    trace_stamp(s_trace_buf, 17);
    // (barrier_kernel ran before this launch: every rank's input is complete)
    float4 tail = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q_tail >= 0 && blockIdx.x == 0 && threadIdx.x == 0) tail = exact_tail(bufs, q_tail, world);
    const int64_t stride = (int64_t)gridDim.x * THREADS;
    for (int64_t q = q0 + blockIdx.x * (int64_t)THREADS + threadIdx.x; q < q1; q += 4 * stride) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (q + u * stride < q1) v[u] = mm_ld_reduce(mc + 4 * (q + u * stride));
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (q + u * stride < q1) mm_st(mc + 4 * (q + u * stride), v[u]);
    }
    // (no fence per thread: grid_sync_ranks' bar.sync + thread 0's system fence is cumulative over the block's stores)
    grid_sync_ranks<true, true>(pads, counter, channel, rank, world);   // every slice has landed everywhere, every tail was read
    // (the exact tail goes to a SEPARATE local buffer: peers may still be reading this rank's in-place tail)
    if (q_tail >= 0 && blockIdx.x == 0 && threadIdx.x == 0) *tail_out = tail;
}

// rows [q0, q1) (in float4 units of the K x D accumulator matrix) and the 4-float tail at quad q_tail, reduced over
// the ranks into local memory
__global__ void __launch_bounds__(THREADS) reduce_rows_kernel(const float* mc, int64_t q0, int64_t q1, int64_t q_tail,
                                                              float4* __restrict__ out, float4* __restrict__ tail_out,
                                                              Pads bufs, int world) {
    pdl_begin();
    trace_stamp(s_trace_buf, 14);
    // (barrier_kernel ran before this launch: every rank's accumulators are complete)
    const int64_t stride = (int64_t)gridDim.x * THREADS;
    for (int64_t q = q0 + blockIdx.x * (int64_t)THREADS + threadIdx.x; q < q1; q += 4 * stride) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (q + u * stride < q1) v[u] = mm_ld_reduce(mc + 4 * (q + u * stride));
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (q + u * stride < q1) out[q + u * stride - q0] = v[u];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *tail_out = exact_tail(bufs, q_tail, world);
}

// local rows -> the same rows of every rank (multicast store), then the cross-rank barrier that makes them visible
__global__ void __launch_bounds__(THREADS) bcast_rows_kernel(const float4* __restrict__ src, float* mc_dst, int64_t n4,
                                                             Pads pads, uint32_t* counter, int channel, int rank, int world) {
    pdl_begin();
    trace_stamp(s_trace_buf, 16);
    const int64_t stride = (int64_t)gridDim.x * THREADS;
    for (int64_t q = blockIdx.x * (int64_t)THREADS + threadIdx.x; q < n4; q += stride) mm_st(mc_dst + 4 * q, src[q]);
    grid_sync_ranks<true, true>(pads, counter, channel, rank, world);
}

// Adam on the n4 float4 of this rank's rows (W, m, v, g all local pointers to the slice), new rows stored to every
// rank's codebook through the multicast address, then the barrier.  g is unscaled: scaled by the reduced tail's
// gradient scale, as som_adam_dp_f32.
__global__ void __launch_bounds__(THREADS) adam_slice_bcast_kernel(const float4* __restrict__ W, float* mc_W,
                                                                   float4* __restrict__ m, float4* __restrict__ v,
                                                                   const float4* __restrict__ g, int64_t n4, int D,
                                                                   double lr, double b1, double b2, float eps,
                                                                   int64_t* __restrict__ steps_done,
                                                                   const float* __restrict__ tail,
                                                                   double* __restrict__ loss_out, Pads pads,
                                                                   uint32_t* counter, int channel, int rank, int world) {
    pdl_begin();
    trace_stamp(s_trace_buf, 15);
    const double t = (double)(steps_done[0] + 1);
    const TailTotals tt = tail_totals(tail, D);
    const AdamScalars a = adam_scalars(lr, b1, b2, eps, t);
    if (loss_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *loss_out = tail_loss(tail, tt.numel);
    const int64_t stride = (int64_t)gridDim.x * THREADS;
    for (int64_t q = blockIdx.x * (int64_t)THREADS + threadIdx.x; q < n4; q += stride) {
        float4 gq = g[q], mq = m[q], vq = v[q], wq = W[q];
        adam_update4<true>(a, gq, tt.gscale, mq, vq, wq);
        m[q] = mq; v[q] = vq;
        mm_st(mc_W + 4 * q, wq);
    }
    // the last block to arrive (every block has read steps_done[0] by then) runs the exchange and advances the step count
    const bool last = grid_sync_ranks<true, true>(pads, counter, channel, rank, world);
    if (last && threadIdx.x == 0) steps_done[0] += 1;
}

static int make_pads(Pads* pads, void* const* signal_pads, int rank, int world) {
    SOM_REQUIRE(signal_pads != nullptr && world >= 2 && world <= MAX_WORLD && rank >= 0 && rank < world, SOM_E_BADARG,
                "peer: rank=%d world=%d (2..%d ranks)", rank, world, MAX_WORLD);
    for (int r = 0; r < MAX_WORLD; ++r) pads->p[r] = r < world ? (uint32_t*)signal_pads[r] : nullptr;
    for (int r = 0; r < world; ++r) SOM_REQUIRE(pads->p[r] != nullptr, SOM_E_BADARG, "peer: null signal pad of rank %d", r);
    return SOM_OK;
}
// flag area of a rank (som_peer_signal_bytes): words [16 c, 16 c + 16) = the rank-to-rank flags of channel c,
// words [64, 68) = the local block-arrival counters of the four channels
static uint32_t* counter_of(const Pads& pads, int rank, int channel) { return pads.p[rank] + 64 + channel; }
static int launch_barrier(const Pads& pads, int channel, int rank, int world, cudaStream_t st) {
    launch_pdl(barrier_kernel, 1, 32, 0, st, pads, channel, rank, world);
    return check_launch("peer_barrier_kernel");
}
// One quad per thread while that stays within two blocks per SM: these kernels are latency-bound (a multimem load or a
// store + fence is a round trip through the switch), so the work is spread wide instead of looped (round 2 first
// version: 4 quads per thread, <= 48 blocks -- the Adam slice of 2048 rows ran on 16 SMs, four serial round trips each).
static int grid_for(int64_t n4) {
    int64_t g = ceil_div64(n4, (int64_t)THREADS);
    return (int)(g < 1 ? 1 : (g > 296 ? 296 : g));
}

}  // namespace peer

// som_filter_tc.cu
bool filter_tc_applicable(int K, int D, int h);
int launch_filter_tc_peer(const float* mc_in, float* out, int K, int D, float two_var, int h, float scale, void* ws,
                          size_t ws_bytes, cudaStream_t st, const peer::Pads& bufs, int64_t q_tail, int world,
                          float* tail_out);
}  // namespace som

using namespace som;
using namespace som::peer;

extern "C" size_t som_peer_signal_bytes(void) { return 1024; }

extern "C" int som_peer_allreduce_f32(void* mc_buf, int64_t n, void* const* peer_bufs, float* tail_out_f, int rank,
                                      int world, void* const* signal_pads, int channel, void* stream) {
    float4* tail_out = (float4*)tail_out_f;
    SOM_REQUIRE(mc_buf != nullptr && n >= 0 && n % 4 == 0 && ((uintptr_t)mc_buf & 15) == 0, SOM_E_BADARG,
                "peer_allreduce: n=%lld must be a multiple of 4 floats, 16-byte aligned", (long long)n);
    SOM_REQUIRE(channel >= 0 && channel < 4, SOM_E_BADARG, "peer: channel=%d", channel);
    SOM_REQUIRE((peer_bufs == nullptr) == (tail_out_f == nullptr) && ((uintptr_t)tail_out_f & 15) == 0, SOM_E_BADARG,
                "peer_allreduce: peer_bufs and tail_out go together (tail_out 16-byte aligned)");
    Pads pads, bufs = {};
    int rc = make_pads(&pads, signal_pads, rank, world);
    if (rc) return rc;
    int64_t n4 = n / 4, q_tail = -1;
    if (peer_bufs != nullptr) {                      // packed accumulator buffer: the last quad is the exact tail
        SOM_REQUIRE(n4 >= 1, SOM_E_BADARG, "peer_allreduce: packed buffer without a tail");
        rc = make_pads(&bufs, peer_bufs, rank, world);
        if (rc) return rc;
        q_tail = --n4;
    }
    const int64_t per = ceil_div64(n4, world);
    const int64_t q0 = per * rank < n4 ? per * rank : n4, q1 = q0 + per < n4 ? q0 + per : n4;
    rc = launch_barrier(pads, channel, rank, world, (cudaStream_t)stream);
    if (rc) return rc;
    launch_pdl(allreduce_kernel, grid_for(per), THREADS, 0, (cudaStream_t)stream, 
        (float*)mc_buf, q0, q1, q_tail, tail_out, bufs, pads, counter_of(pads, rank, channel), channel, rank, world);
    return check_launch("peer_allreduce_kernel");
}

extern "C" int som_peer_reduce_rows_f32(const void* mc_packed, void* const* peer_packed, int K, int D, int row0,
                                        int row1, int max_rows, float* out_rows, float* out_tail, int rank, int world,
                                        void* const* signal_pads, int channel, void* stream) {
    SOM_REQUIRE(mc_packed && peer_packed && out_rows && out_tail, SOM_E_BADARG, "peer_reduce_rows: null pointer");
    SOM_REQUIRE(K > 0 && D > 0 && D % 4 == 0 && row0 >= 0 && row0 <= row1 && row1 <= K && max_rows >= row1 - row0,
                SOM_E_BADARG, "peer_reduce_rows: K=%d D=%d rows [%d, %d) max %d (D must be a multiple of 4)", K, D,
                row0, row1, max_rows);
    SOM_REQUIRE((((uintptr_t)mc_packed | (uintptr_t)out_rows | (uintptr_t)out_tail) & 15) == 0, SOM_E_BADARG,
                "peer_reduce_rows: buffers must be 16-byte aligned");
    SOM_REQUIRE(channel >= 0 && channel < 4, SOM_E_BADARG, "peer: channel=%d", channel);
    Pads pads, bufs;
    int rc = make_pads(&pads, signal_pads, rank, world);
    if (rc) return rc;
    rc = make_pads(&bufs, peer_packed, rank, world);
    if (rc) return rc;
    const int64_t d4 = D / 4;
    rc = launch_barrier(pads, channel, rank, world, (cudaStream_t)stream);
    if (rc) return rc;
    (void)max_rows;
    launch_pdl(reduce_rows_kernel, grid_for((int64_t)(row1 - row0) * d4), THREADS, 0, (cudaStream_t)stream, 
        (const float*)mc_packed, (int64_t)row0 * d4, (int64_t)row1 * d4, (int64_t)K * d4, (float4*)out_rows,
        (float4*)out_tail, bufs, world);
    return check_launch("peer_reduce_rows_kernel");
}

// Reduce-scatter fused into the consumer: G rows = scale * T @ (sum over the ranks of accumulator rows [row0, row1)), the
// sum taken by the filter's own pre-pass as it reads (multimem.ld_reduce) -- no reduced copy of the rows, one kernel and
// one pass over them less than som_peer_reduce_rows_f32 + som_filter_ws_f32.  Shapes the tensor-core filter does not
// take fall back to exactly that pair (rows_scratch: max_rows x D floats).
extern "C" int som_peer_reduce_filter_rows_f32(const void* mc_packed, void* const* peer_packed, int K, int D, int row0,
                                               int row1, int max_rows, double neighbourhood_range, float scale,
                                               float* rows_scratch, float* out_rows, float* out_tail, int rank,
                                               int world, void* const* signal_pads, int channel, void* ws,
                                               size_t ws_bytes, void* stream) {
    SOM_REQUIRE(mc_packed && peer_packed && rows_scratch && out_rows && out_tail, SOM_E_BADARG,
                "peer_reduce_filter_rows: null pointer");
    SOM_REQUIRE(K > 0 && D > 0 && D % 4 == 0 && row0 >= 0 && row0 < row1 && row1 <= K && max_rows >= row1 - row0,
                SOM_E_BADARG, "peer_reduce_filter_rows: K=%d D=%d rows [%d, %d) max %d (D must be a multiple of 4)", K,
                D, row0, row1, max_rows);
    SOM_REQUIRE(neighbourhood_range > 0.0, SOM_E_BADARG, "peer_reduce_filter_rows: neighbourhood_range=%g",
                neighbourhood_range);
    SOM_REQUIRE((((uintptr_t)mc_packed | (uintptr_t)rows_scratch | (uintptr_t)out_rows | (uintptr_t)out_tail) & 15) == 0,
                SOM_E_BADARG, "peer_reduce_filter_rows: buffers must be 16-byte aligned");
    SOM_REQUIRE(channel >= 0 && channel < 4, SOM_E_BADARG, "peer: channel=%d", channel);
    const int rows = row1 - row0;
    const float two_var = filter_two_var(neighbourhood_range);
    const int h = filter_band_half_width(two_var, rows);
    if (!(filter_tc_applicable(rows, D, h) && ws != nullptr)) {
        int rc = som_peer_reduce_rows_f32(mc_packed, peer_packed, K, D, row0, row1, max_rows, rows_scratch, out_tail, rank,
                                          world, signal_pads, channel, stream);
        if (rc) return rc;
        return som_filter_ws_f32(rows_scratch, out_rows, rows, D, neighbourhood_range, scale, ws, ws_bytes, stream);
    }
    Pads pads, bufs;
    int rc = make_pads(&pads, signal_pads, rank, world);
    if (rc) return rc;
    rc = make_pads(&bufs, peer_packed, rank, world);
    if (rc) return rc;
    rc = launch_barrier(pads, channel, rank, world, (cudaStream_t)stream);      // every rank's accumulators are complete
    if (rc) return rc;
    return launch_filter_tc_peer((const float*)mc_packed + (int64_t)row0 * D, out_rows, rows, D, two_var, h, scale, ws,
                                 ws_bytes, (cudaStream_t)stream, bufs, (int64_t)K * (D / 4), world, out_tail);
}

extern "C" int som_peer_bcast_rows_f32(const float* src_rows, void* mc_dst_rows, int64_t n, int64_t max_n, int rank,
                                       int world, void* const* signal_pads, int channel, void* stream) {
    SOM_REQUIRE(src_rows && mc_dst_rows && n >= 0 && n % 4 == 0 && max_n >= n, SOM_E_BADARG,
                "peer_bcast_rows: n=%lld (multiple of 4 floats)", (long long)n);
    SOM_REQUIRE((((uintptr_t)src_rows | (uintptr_t)mc_dst_rows) & 15) == 0, SOM_E_BADARG,
                "peer_bcast_rows: buffers must be 16-byte aligned");
    SOM_REQUIRE(channel >= 0 && channel < 4, SOM_E_BADARG, "peer: channel=%d", channel);
    Pads pads;
    int rc = make_pads(&pads, signal_pads, rank, world);
    if (rc) return rc;
    (void)max_n;
    launch_pdl(bcast_rows_kernel, grid_for(n / 4), THREADS, 0, (cudaStream_t)stream, (const float4*)src_rows, (float*)mc_dst_rows,
                                                                           n / 4, pads, counter_of(pads, rank, channel),
                                                                           channel, rank, world);
    return check_launch("peer_bcast_rows_kernel");
}

extern "C" int som_peer_adam_slice_f32(const float* W_rows, void* mc_W_rows, float* m_rows, float* v_rows,
                                       const float* g_rows, int64_t n, int64_t max_n, int D, double lr, double b1,
                                       double b2, double eps, int64_t* steps_done, const float* tail, double* loss_out,
                                       int rank, int world, void* const* signal_pads, int channel, void* stream) {
    SOM_REQUIRE(W_rows && mc_W_rows && m_rows && v_rows && g_rows && steps_done && tail, SOM_E_BADARG,
                "peer_adam_slice: null pointer");
    SOM_REQUIRE(n >= 0 && n % 4 == 0 && max_n >= n && D > 0, SOM_E_BADARG, "peer_adam_slice: n=%lld D=%d", (long long)n, D);
    SOM_REQUIRE((((uintptr_t)W_rows | (uintptr_t)mc_W_rows | (uintptr_t)m_rows | (uintptr_t)v_rows | (uintptr_t)g_rows) & 15) == 0,
                SOM_E_BADARG, "peer_adam_slice: buffers must be 16-byte aligned");
    SOM_REQUIRE(channel >= 0 && channel < 4, SOM_E_BADARG, "peer: channel=%d", channel);
    Pads pads;
    int rc = make_pads(&pads, signal_pads, rank, world);
    if (rc) return rc;
    (void)max_n;
    launch_pdl(adam_slice_bcast_kernel, grid_for(n / 4), THREADS, 0, (cudaStream_t)stream, 
        (const float4*)W_rows, (float*)mc_W_rows, (float4*)m_rows, (float4*)v_rows, (const float4*)g_rows, n / 4, D, lr, b1,
        b2, (float)eps, steps_done, tail, loss_out, pads, counter_of(pads, rank, channel), channel, rank, world);
    return check_launch("peer_adam_slice_bcast_kernel");
}
