// K2: per-unit accumulation, segmented by BMU.
//
//   Wt != NULL:  Rbar[a] = sum_{p: bmu[p]==a} (Wt[a] - x_p)     sse = sum_p ||Wt[bmu_p] - x_p||^2
//   Wt == NULL:  Rbar[a] = sum_{p: bmu[p]==a} x_p
//
// Together with the neighbourhood filter this is the S^T @ grad half of the reference's autograd
// step for models/Codebook.py:128-130 + F.mse_loss (train_codebook.py:233-240), after the exact
// factorisation S = onehot(bmu) @ T (SURVEY.md A.3).
//
// Pipeline (all on the caller's stream, fully deterministic, no floating-point atomics):
//   1. keys = (int32) bmu, vals = patch id                          [pairs_kernel]
//   2. stable LSD radix sort of (key, val) pairs over ceil(log2 K) bits   [cub::DeviceRadixSort:
//      toolkit plumbing, ~1% of the step; order inside a segment is ascending patch id]
//   3. offsets[a] = first sorted position with key >= a             [offsets_kernel]
//   4. level 1: one warp per (chunk of S sorted positions, 32*VEC-wide feature slice) walks its
//      chunk in order, gathering patch rows straight from NCHW (patchify as address arithmetic,
//      VEC-wide loads, 8 rows in flight).  Segments that live inside one chunk are stored
//      directly; the (at most two) segments crossing a chunk edge go to partial[chunk][slot].
//   5. level 2: one warp per (unit, slice) adds the partials of chunk-crossing segments in chunk
//      order, zero-fills empty units, and writes counts; a single CTA reduces the sse partials.
// Bound: HBM -- algorithmic bytes 4*D per patch (x read once) + 8 (index) + 4*K*D (Rbar).
#include "som_common.cuh"
#include "som_step_rules.cuh"

#include <cub/device/device_radix_sort.cuh>

namespace som {
SOM_TRACE_TU(trace_set_accumulate)

constexpr int ACC_WARPS = 8;

constexpr int CS_BLOCK = 2048;      // patches per block of the counting sort
constexpr int CS_THREADS = 1024;
constexpr int CS_KMAX = 16384;      // bins that fit in shared memory (64 KB)

struct AccumPlan {
    int64_t n;
    int D, K;
    int S;                 // sorted positions per chunk
    int64_t n_chunks;
    int n_slices_max;      // slices at VEC=1 (upper bound used for sizing)
    int end_bit;
    size_t off_keys_a, off_keys_b, off_vals_a, off_vals_b, off_offsets, off_partial, off_sse,
        off_cub, cub_bytes, off_hist, total;
    int cs_blocks;         // > 0: our own counting sort (K <= 16 384), else cub's radix sort
    int cs_per;            // patches per block of it: CS_BLOCK, or more once that would be over one block per SM
};

// Sorted positions per level-1 chunk: enough (chunk, feature slice) warps to fill the machine, but no shorter chunks
// than that needs -- every chunk pays the key fetch, up to two partial segments and the W~ row of its first unit.
// Long rows bring their own parallelism (one warp per 128-feature slice): C3 (4096 patches, D = 4096) gets S = 32
// instead of 8 (accumulate 70.7 -> 58.6 us).  Large batches are flat in S (C4 shape: 0.39 / 0.36 / 0.35 / 0.34 / 0.36 /
// 0.43 ms at S = 8 / 16 / 32 / 64 / 128 / 256), so 64 stays the cap.
static int pick_chunk(int64_t n, int D) {
    const int64_t target = 148 * 16;
    const int64_t slices = D >= 128 ? D / 128 : 1;
    int S = 64;
    while (S > 8 && (n / S) * slices < target) S >>= 1;
    return S;
}

static int make_plan(AccumPlan* pl, int64_t n, int D, int K, bool query_cub) {
    SOM_REQUIRE(n >= 0 && n < (int64_t)INT32_MAX && D > 0 && K > 0, SOM_E_BADARG,
                "accumulate: n=%lld D=%d K=%d out of range", (long long)n, D, K);
    pl->n = n; pl->D = D; pl->K = K;
    pl->S = pick_chunk(n, D);
    pl->n_chunks = n > 0 ? ceil_div64(n, pl->S) : 0;
    pl->n_slices_max = (D + 31) / 32;
    int bits = 1;
    while (bits < 31 && (1LL << bits) < (long long)K) ++bits;
    pl->end_bit = bits;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 256); return at; };
    pl->off_keys_a = take((size_t)n * 4);
    pl->off_keys_b = take((size_t)n * 4);
    pl->off_vals_a = take((size_t)n * 4);
    pl->off_vals_b = take((size_t)n * 4);
    pl->off_offsets = take((size_t)(K + 1) * 4);
    pl->off_partial = take((size_t)pl->n_chunks * 2 * D * 4);
    // squared-error partials: per (chunk, slice) on the sorted path, per (unit, slice) on the scan path
    {
        size_t a = (size_t)pl->n_chunks * pl->n_slices_max * 8, b = (size_t)K * pl->n_slices_max * 8;
        pl->off_sse = take(a > b ? a : b);
    }
    pl->cub_bytes = 0;
    if (query_cub && n > 0) {
        cub::DoubleBuffer<int> k(nullptr, nullptr), v(nullptr, nullptr);
        size_t bytes = 0;
        cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, bytes, k, v, (int)n, 0, pl->end_bit);
        if (e != cudaSuccess) { set_error("accumulate: cub size query: %s", cudaGetErrorString(e)); return (int)e; }
        pl->cub_bytes = bytes;
    }
    pl->off_cub = take(pl->cub_bytes + 256);
    // counting sort: per-block histograms (ints) + the totals; blocks x K x 4 bytes (4 MB at 131 072 patches, 32 MB at 2^20)
    pl->cs_per = CS_BLOCK;
    if (n > (int64_t)148 * CS_BLOCK) pl->cs_per = (int)(ceil_div64(ceil_div64(n, 148), CS_THREADS) * CS_THREADS);
    pl->cs_blocks = (K <= CS_KMAX && n > 0 && n <= ((int64_t)1 << 22)) ? (int)ceil_div64(n, pl->cs_per) : 0;
    pl->off_hist = take(pl->cs_blocks > 0 ? ((size_t)pl->cs_blocks + 1) * K * 4 : 0);
    pl->total = o;
    return SOM_OK;
}

__global__ void __launch_bounds__(256) pairs_kernel(const int64_t* __restrict__ bmu, int64_t n, int K,
                                                    int* __restrict__ keys, int* __restrict__ vals) {
    pdl_begin();
    trace_stamp(s_trace_buf, 8);
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    int64_t k = bmu[p];
    k = k < 0 ? 0 : (k >= K ? K - 1 : k);
    keys[p] = (int)k;
    vals[p] = (int)p;
}

// offsets[a] = first position whose key >= a, a in [0, K]; each boundary position p writes the
// (possibly empty) range of unit ids between its left and right neighbour keys.
__global__ void __launch_bounds__(256) offsets_kernel(const int* __restrict__ skey, int64_t n, int K,
                                                      int* __restrict__ offsets) {
    pdl_begin();
    trace_stamp(s_trace_buf, 9);
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p > n) return;
    int lo = (p == 0) ? -1 : skey[p - 1];
    int hi = (p == n) ? K : skey[p];
    for (int a = lo + 1; a <= hi; ++a) offsets[a] = (int)p;
}

// ---- stable counting sort of (unit, patch) by unit, for codebooks of up to 16 384 units --------------------------------------
// Replaces pairs_kernel + the four launches of cub::DeviceRadixSort (two 7-bit passes) + offsets_kernel by four short
// kernels of our own: a one-pass sort on the whole key is possible because K bins fit in shared memory (64 KB).
//   csort_hist      block b (CS_BLOCK patches): histogram of its keys in shared memory -> hist[b][K]
//   csort_prefix    thread per key: exclusive prefix over the blocks in place, total[k]
//   csort_offsets   one CTA: exclusive scan of the totals -> offsets[0..K] (what offsets_kernel derived from the sorted keys)
//   csort_scatter   block b: every patch goes to offsets[key] + hist[b][key] + its rank among the block's earlier
//                   patches of the same key (warps take turns, match groups inside a warp): STABLE, so the patches of a
//                   unit stay in ascending order and the segmented sums keep their fixed order

__global__ void __launch_bounds__(CS_THREADS) csort_hist_kernel(const int64_t* __restrict__ bmu, int64_t n, int K, int per,
                                                                int* __restrict__ hist) {
    pdl_begin();
    trace_stamp(s_trace_buf, 8);
    extern __shared__ int cs_bins[];
    for (int k = threadIdx.x; k < K; k += CS_THREADS) cs_bins[k] = 0;
    __syncthreads();
    const int64_t p0 = (int64_t)blockIdx.x * per;
#pragma unroll 2
    for (int u = 0; u < per; u += CS_THREADS) {
        const int64_t p = p0 + u + threadIdx.x;
        if (p < n) {
            int64_t k = bmu[p];
            k = k < 0 ? 0 : (k >= K ? K - 1 : k);
            atomicAdd(&cs_bins[(int)k], 1);
        }
    }
    __syncthreads();
    int* out = hist + (int64_t)blockIdx.x * K;
    for (int k = threadIdx.x; k < K; k += CS_THREADS) out[k] = cs_bins[k];
}

__global__ void __launch_bounds__(256) csort_prefix_kernel(int* __restrict__ hist, int nb, int K, int* __restrict__ total) {
    pdl_begin();
    trace_stamp(s_trace_buf, 20);
    const int k = blockIdx.x * 256 + threadIdx.x;
    if (k >= K) return;
    constexpr int G = 32;                                  // loads in flight per thread: the loop is a chain of L2 round trips
    int run = 0;
    for (int b0 = 0; b0 < nb; b0 += G) {
        int v[G];
#pragma unroll
        for (int u = 0; u < G; ++u) v[u] = (b0 + u < nb) ? hist[(int64_t)(b0 + u) * K + k] : 0;
#pragma unroll
        for (int u = 0; u < G; ++u) {
            if (b0 + u < nb) { hist[(int64_t)(b0 + u) * K + k] = run; run += v[u]; }
        }
    }
    total[k] = run;
}

// offsets[a] = number of patches with key < a, a in [0, K]: one CTA; thread t holds keys t, 1024 + t, ... (coalesced:
// one SM pays a wavefront per touched sector, a thread-owns-16-consecutive-keys layout cost 15 us here), all loaded up
// front; warp scans of the 16 rows run side by side, then one scan over the 512 (row, warp) sums in key order
__global__ void __launch_bounds__(1024) csort_offsets_kernel(const int* __restrict__ total, int K, int* __restrict__ offsets) {
    pdl_begin();
    trace_stamp(s_trace_buf, 21);
    constexpr int PER = CS_KMAX / 1024;
    __shared__ int row_warp_s[PER * 32];
    __shared__ int group_s[PER];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int v[PER], inc[PER];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int k = u * 1024 + (int)threadIdx.x;
        v[u] = k < K ? total[k] : 0;
    }
#pragma unroll
    for (int u = 0; u < PER; ++u) inc[u] = v[u];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            const int t = __shfl_up_sync(0xffffffffu, inc[u], o);
            if (lane >= o) inc[u] += t;
        }
    }
    if (lane == 31) {
#pragma unroll
        for (int u = 0; u < PER; ++u) row_warp_s[u * 32 + warp] = inc[u];
    }
    __syncthreads();
    int mine = 0, mine_inc = 0;
    if (threadIdx.x < PER * 32) {                            // warps 0..15: inclusive scan of 32 sums each
        mine = row_warp_s[threadIdx.x];
        mine_inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, mine_inc, o);
            if (lane >= o) mine_inc += t;
        }
        if (lane == 31) group_s[warp] = mine_inc;
    }
    __syncthreads();
    if (warp == 0) {
        const int g = lane < PER ? group_s[lane] : 0;
        int gi = g;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, gi, o);
            if (lane >= o) gi += t;
        }
        if (lane < PER) group_s[lane] = gi - g;              // exclusive over the rows
        if (lane == PER - 1) offsets[K] = gi;
    }
    __syncthreads();
    if (threadIdx.x < PER * 32) row_warp_s[threadIdx.x] = group_s[warp] + mine_inc - mine;
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int k = u * 1024 + (int)threadIdx.x;
        if (k < K) offsets[k] = row_warp_s[u * 32 + warp] + inc[u] - v[u];
    }
    trace_stamp(s_trace_buf, 121);
}

__global__ void __launch_bounds__(CS_THREADS) csort_scatter_kernel(const int64_t* __restrict__ bmu, int64_t n, int K, int per,
                                                                   const int* __restrict__ hist,
                                                                   const int* __restrict__ offsets,
                                                                   int* __restrict__ skey, int* __restrict__ sid) {
    pdl_begin();
    trace_stamp(s_trace_buf, 22);
    extern __shared__ int cs_bins[];                        // patches of the block seen so far, per key
    __shared__ uint64_t turn_bar[CS_THREADS / 32];          // warp w may take its turn (one phase per round)
    for (int k = threadIdx.x; k < K; k += CS_THREADS) cs_bins[k] = 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < CS_THREADS / 32)
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(&turn_bar[threadIdx.x])));
    const int* blk = hist + (int64_t)blockIdx.x * K;
    const int64_t p0 = (int64_t)blockIdx.x * per;
    auto key_of = [&](int64_t p) -> int {
        if (p >= n) return -1;
        const int64_t k = bmu[p];
        return (int)(k < 0 ? 0 : (k >= K ? K - 1 : k));
    };
    int key_next = key_of(p0 + threadIdx.x);
    __syncthreads();
    const uint32_t my_bar = (uint32_t)__cvta_generic_to_shared(&turn_bar[warp]);
    const uint32_t next_bar = (uint32_t)__cvta_generic_to_shared(&turn_bar[(warp + 1) & (CS_THREADS / 32 - 1)]);
    if (threadIdx.x == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(my_bar) : "memory");   // warp 0 starts
    uint32_t round = 0;
#pragma unroll 1
    for (int u = 0; u < per; u += CS_THREADS, ++round) {
        const int64_t p = p0 + u + threadIdx.x;
        const int key = key_next;
        if (u + CS_THREADS < per) key_next = key_of(p + CS_THREADS);       // next round's keys fly during the turns
        // where the block's patches of this key start: two gathers, needed only AFTER the turn (kept out of it --
        // a first version let the compiler sink them into the turn and paid an L2 round trip per warp turn)
        int base = 0;
        if (key >= 0) base = offsets[key] + blk[key];
        // lanes of the warp with the same key: rank inside the group, the group's last lane updates the bin
        const unsigned grp = __match_any_sync(0xffffffffu, key);
        const int rank_in_warp = __popc(grp & ((1u << lane) - 1u));
        const int add = ((grp >> lane) == 1u) ? __popc(grp) : 0;
        // Warps take turns in warp order (ascending patch order per key), handing the turn on through one mbarrier per
        // warp: the waiting warps sleep in try_wait instead of all 32 meeting in a block barrier per turn (a turn
        // cost ~400 cycles that way, 224 turns per block at 2^20 patches).
        {
            uint32_t done = 0;
            while (!done)
                asm volatile(
                    "{\n.reg .pred p;\n"
                    "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
                    "selp.u32 %0, 1, 0, p;\n}\n"
                    : "=r"(done) : "r"(my_bar), "r"(round & 1u) : "memory");
        }
        int local = 0;
        if (key >= 0) local = cs_bins[key];
        __syncwarp();                                        // (one full-warp sync: a sync per match group serialised them)
        if (add && key >= 0) cs_bins[key] = local + add;
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(next_bar) : "memory");
        if (key >= 0) {
            const int pos = base + local + rank_in_warp;
            skey[pos] = key;
            sid[pos] = (int)p;
        }
    }
    __syncthreads();
    trace_stamp(s_trace_buf, 122);
}

template <int VEC> struct VecT;
template <> struct VecT<1> { using T = float; };
template <> struct VecT<2> { using T = float2; };
template <> struct VecT<4> { using T = float4; };

template <int VEC>
__device__ __forceinline__ void load_vec(float (&r)[VEC], const float* p) {
    using T = typename VecT<VEC>::T;
    T t = __ldg(reinterpret_cast<const T*>(p));
    const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
    for (int i = 0; i < VEC; ++i) r[i] = f[i];
}

template <int VEC>
__device__ __forceinline__ void store_vec(float* p, const float (&r)[VEC]) {
    using T = typename VecT<VEC>::T;
    T t;
    float* f = reinterpret_cast<float*>(&t);
#pragma unroll
    for (int i = 0; i < VEC; ++i) f[i] = r[i];
    *reinterpret_cast<T*>(p) = t;
}

// positions per cp.async group of seg_level1_kernel: two groups of G rows + G W~ rows per warp in shared memory
// (8 KB per warp, 64 KB per CTA, three CTAs per SM)
template <int VEC> struct L1_GROUP { static constexpr int value = (VEC == 4) ? 4 : 8; };

template <int VEC, bool STREAM>
__device__ __forceinline__ void cp_async_vec(float* smem_dst, const float* src) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
    if (VEC == 4) {
        if (STREAM) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
        else asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
    } else if (VEC == 2) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
    } else {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
    }
}
template <int VEC>
__device__ __forceinline__ void lds_vec(float (&r)[VEC], const float* smem_src) {
    using T = typename VecT<VEC>::T;
    const T t = *reinterpret_cast<const T*>(smem_src);
    const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
    for (int i = 0; i < VEC; ++i) r[i] = f[i];
}

template <int VEC>
__global__ void __launch_bounds__(ACC_WARPS * 32, 3)
seg_level1_kernel(const float* __restrict__ x, Geom g, const int* __restrict__ skey,
                  const int* __restrict__ sid, const int* __restrict__ offsets,
                  const float* __restrict__ Wt, float* __restrict__ Rbar,
                  float* __restrict__ partial, double* __restrict__ sse_part,
                  int S, int64_t n_chunks, int n_slices) {
    pdl_begin();
    trace_stamp(s_trace_buf, 10);
    const int lane = threadIdx.x & 31;
    const int64_t wg = blockIdx.x * (int64_t)ACC_WARPS + (threadIdx.x >> 5);
    const int64_t c = wg / n_slices;
    const int s = (int)(wg - c * n_slices);
    if (c >= n_chunks) return;
    const int D = g.D;
    const int d = (s * 32 + lane) * VEC;
    const bool act = d < D;
    const int doff = act ? feat_off(g, d) : 0;
    const int64_t n = g.n_patches;
    const int64_t p0 = c * S;
    const int64_t p1 = (p0 + S < n) ? p0 + S : n;

    float acc[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
    float sse = 0.f;
    int cur = -1;
    int64_t run_start = p0;
    // keys just outside the chunk decide, without touching the offsets array, whether a segment lies inside the chunk
    // (-> stored directly) or crosses an edge (-> partial slot): the same rule seg_level2_kernel applies to the offsets
    const int prev_key = (p0 > 0) ? skey[p0 - 1] : -1;
    const int next_key = (p1 < n) ? skey[p1] : -2;

    auto flush = [&](int64_t run_end) {
        if (cur < 0 || !act) return;
        const bool starts_inside = run_start > p0 || prev_key != cur;
        const bool ends_inside = run_end < p1 || next_key != cur;
        if (starts_inside && ends_inside) {
            store_vec<VEC>(Rbar + (int64_t)cur * D + d, acc);
        } else {
            int slot = (run_start == p0) ? 0 : 1;
            store_vec<VEC>(partial + ((c * 2 + slot) * (int64_t)D) + d, acc);
        }
    };

    // Rows land in SHARED memory through cp.async, not in registers: every lane owns private words of a two-group ring
    // (its slice of G patch rows and of their units' W~ rows per group), so the rows need no synchronisation, and
    // group g + 1 is on its way while group g is consumed.
    // The kernel is bound by instruction issue, not by memory (ncu, 2^20 patches: 71, later 65 warp instructions per
    // position, long-scoreboard stalls negligible), so everything per position that can be decided per GROUP is:
    // lanes 0..G-1 fetch (key, patch base) of the group's positions, two ballots turn "position valid" and "a new unit
    // starts here" into warp-wide bit masks, and the pairs go through a small shared table that every lane reads back
    // with one broadcast load (a shuffle costs its divergence check as well).  A position then costs a table load, the
    // address and one cp.async to issue, one shared load and the arithmetic to consume; W~ rows are fetched and
    // segments flushed only at the set bits (W~ also once per group, whose ring slot is recycled).  Lanes past the
    // row's end (D not a multiple of the slice) stream the slice of lane 0 and are never stored.
    constexpr int G = L1_GROUP<VEC>::value;
    constexpr unsigned GMASK = (1u << G) - 1u;
    extern __shared__ __align__(16) float l1_ring[];     // [warp][buffer][row | W~][position][lane slice], then the tables
    const int wib = threadIdx.x >> 5;
    float (*mine)[2][G][32 * VEC] = reinterpret_cast<float (*)[2][G][32 * VEC]>(l1_ring) + wib * 2;
    int4 (*tab)[G] = reinterpret_cast<int4 (*)[G]>(l1_ring + (size_t)ACC_WARPS * 2 * 2 * G * 32 * VEC) + wib * 2;
    const float* x_lane = x + (act ? doff : 0);
    const float* wt_lane = Wt + (act ? d : 0);
    // group at p: (key, patch base) in lanes 0..G-1, masks of the valid positions and of those where the key differs
    // from the position before (last_key: the key just before the group, -1 at the chunk start = always a start)
    auto fetch = [&](int64_t p, int last_key, int& k, int64_t& b, unsigned& valid, unsigned& starts) {
        k = -1;
        b = 0;
        if (lane < G && p + lane < p1) {
            k = skey[p + lane];
            b = patch_base(g, (int64_t)sid[p + lane]);
        }
        int before = __shfl_up_sync(0xffffffffu, k, 1);
        if (lane == 0) before = last_key;
        valid = __ballot_sync(0xffffffffu, k >= 0) & GMASK;
        starts = __ballot_sync(0xffffffffu, k >= 0 && k != before) & GMASK;
    };
    auto publish = [&](int buf, int k_l, int64_t b_l) {
        __syncwarp();                                     // (the table's previous readers are done)
        if (lane < G) tab[buf][lane] = make_int4((int)(uint32_t)b_l, (int)(b_l >> 32), k_l, 0);
        __syncwarp();
    };
    auto issue = [&](int buf, unsigned valid, unsigned starts) {
#pragma unroll
        for (int u = 0; u < G; ++u) {
            if (valid != GMASK && !((valid >> u) & 1u)) break;       // (only the last group of the whole batch is short)
            const int4 e = tab[buf][u];
            const int64_t base = (int64_t)(((uint64_t)(uint32_t)e.y << 32) | (uint32_t)e.x);
            cp_async_vec<VEC, true>(&mine[buf][0][u][lane * VEC], x_lane + base);
            if (Wt != nullptr && (u == 0 || ((starts >> u) & 1u)))
                cp_async_vec<VEC, false>(&mine[buf][1][u][lane * VEC], wt_lane + (int64_t)e.z * D);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    int key_cur, key_next;
    int64_t base_cur, base_next;
    unsigned valid_cur, valid_next, starts_cur, starts_next;
    fetch(p0, -1, key_cur, base_cur, valid_cur, starts_cur);
    publish(0, key_cur, base_cur);
    issue(0, valid_cur, starts_cur);
    fetch(p0 + G, __shfl_sync(0xffffffffu, key_cur, G - 1), key_next, base_next, valid_next, starts_next);
    int buf = 0;
    float wtr[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) wtr[i] = 0.f;
    for (int64_t p = p0; p < p1; p += G) {
        publish(buf ^ 1, key_next, base_next);
        issue(buf ^ 1, valid_next, starts_next);          // (an empty group past the chunk end commits nothing)
        const unsigned valid_mine = valid_cur, starts_mine = starts_cur;
        key_cur = key_next; valid_cur = valid_next; starts_cur = starts_next;
        // keys two groups ahead: in flight while this group is consumed
        fetch(p + 2 * G, __shfl_sync(0xffffffffu, key_cur, G - 1), key_next, base_next, valid_next, starts_next);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
#pragma unroll
        for (int u = 0; u < G; ++u) {
            if (valid_mine != GMASK && !((valid_mine >> u) & 1u)) break;
            const bool st = (starts_mine >> u) & 1u;
            if (st) {
                flush(p + u);
                cur = tab[buf][u].z;
                run_start = p + u;
#pragma unroll
                for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
            }
            float row[VEC];
            lds_vec<VEC>(row, &mine[buf][0][u][lane * VEC]);
            if (Wt != nullptr) {
                if (u == 0 || st) lds_vec<VEC>(wtr, &mine[buf][1][u][lane * VEC]);
#pragma unroll
                for (int i = 0; i < VEC; ++i) {
                    float r = wtr[i] - row[i];
                    acc[i] += r;
                    sse = fmaf(r, r, sse);
                }
            } else {
#pragma unroll
                for (int i = 0; i < VEC; ++i) acc[i] += row[i];
            }
        }
        buf ^= 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    flush(p1);
    if (sse_part != nullptr) {
        float t = warp_sum(act ? sse : 0.f);
        if (lane == 0) sse_part[c * n_slices + s] = (double)t;
    }
}

template <int VEC>
__global__ void __launch_bounds__(ACC_WARPS * 32)
seg_level2_kernel(const int* __restrict__ offsets, const float* __restrict__ partial,
                  float* __restrict__ Rbar, int64_t* __restrict__ counts, int K, int D, int S,
                  int n_slices) {
    pdl_begin();
    trace_stamp(s_trace_buf, 11);
    const int lane = threadIdx.x & 31;
    const int64_t wg = blockIdx.x * (int64_t)ACC_WARPS + (threadIdx.x >> 5);
    const int64_t a = wg / n_slices;
    const int s = (int)(wg - a * n_slices);
    if (a >= K) return;
    const int lo = offsets[a], hi = offsets[a + 1];
    if (s == 0 && lane == 0 && counts != nullptr) counts[a] = (int64_t)(hi - lo);
    const int d = (s * 32 + lane) * VEC;
    if (d >= D) return;
    float acc[VEC];
    if (lo == hi) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
        store_vec<VEC>(Rbar + a * D + d, acc);
        return;
    }
    const int cf = lo / S, cl = (hi - 1) / S;
    if (cf == cl) return;                              // written directly by level 1
    const int first_slot = (lo == cf * S) ? 0 : 1;
    load_vec<VEC>(acc, partial + (((int64_t)cf * 2 + first_slot) * D) + d);
    int c = cf + 1;
    for (; c + 8 <= cl + 1; c += 8) {
        float t[8][VEC];
#pragma unroll
        for (int u = 0; u < 8; ++u) load_vec<VEC>(t[u], partial + ((int64_t)(c + u) * 2 * D) + d);
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[i] += t[u][i];
    }
    for (; c <= cl; ++c) {
        float t[VEC];
        load_vec<VEC>(t, partial + ((int64_t)c * 2 * D) + d);
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] += t[i];
    }
    store_vec<VEC>(Rbar + a * D + d, acc);
}

// Tiny batches (N <= 2048: C1): no sort.  One CTA per (unit, 256*VEC-wide feature slice); every warp
// scans the BMU indices 32 at a time with a ballot and visits the matching patches in ascending order, so the
// result is deterministic and the whole accumulation is ONE launch instead of eight.
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_CH = 4096;           // patches per scan round (match list capacity in shared memory)

template <int VEC>
__global__ void __launch_bounds__(SCAN_THREADS)
acc_scan_kernel(const float* __restrict__ x, Geom g, const int64_t* __restrict__ bmu, int K,
                const float* __restrict__ Wt, float* __restrict__ Rbar, int64_t* __restrict__ counts,
                double* __restrict__ sse_part, int n_slices) {
    pdl_begin();
    trace_stamp(s_trace_buf, 10);
    __shared__ int list[SCAN_CH];
    __shared__ int n_list;
    __shared__ float sse_w[SCAN_THREADS / 32];
    const int a = blockIdx.x;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int D = g.D;
    const int d = (blockIdx.y * SCAN_THREADS + threadIdx.x) * VEC;
    const bool act = d < D;
    const int doff = act ? feat_off(g, d) : 0;
    const int64_t n = g.n_patches;
    float acc[VEC], wt[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) { acc[i] = 0.f; wt[i] = 0.f; }
    if (Wt != nullptr && act) load_vec<VEC>(wt, Wt + (int64_t)a * D + d);
    float sse = 0.f;
    int cnt = 0;
    for (int64_t base = 0; base < n; base += SCAN_CH) {
        // phase 1: warp 0 lists the patches of this round whose BMU is `a`, ascending, 256 keys per step
        if (warp == 0) {
            int m_tot = 0;
            const int64_t end = (base + SCAN_CH < n) ? base + SCAN_CH : n;
            for (int64_t p0 = base; p0 < end; p0 += 256) {
                int key[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int64_t p = p0 + 32 * i + lane;
                    key[i] = -1;
                    if (p < end) {
                        const int64_t k = bmu[p];
                        key[i] = (int)(k < 0 ? 0 : (k >= K ? K - 1 : k));
                    }
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const unsigned m = __ballot_sync(0xffffffffu, key[i] == a);
                    if (key[i] == a) list[m_tot + __popc(m & ((1u << lane) - 1u))] = (int)(p0 + 32 * i + lane - base);
                    m_tot += __popc(m);
                }
            }
            if (lane == 0) n_list = m_tot;
        }
        __syncthreads();
        // phase 2: every thread adds its feature slice of the listed patch rows, four rows in flight
        const int nl = n_list;
        cnt += nl;
        if (act) {
            for (int q = 0; q < nl; q += 4) {
                float row[4][VEC];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (q + u < nl) load_vec<VEC>(row[u], x + patch_base(g, base + list[q + u]) + doff);
                    else {
#pragma unroll
                        for (int i = 0; i < VEC; ++i) row[u][i] = 0.f;
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (q + u < nl) {
#pragma unroll
                        for (int i = 0; i < VEC; ++i) {
                            if (Wt != nullptr) {
                                const float r = wt[i] - row[u][i];
                                acc[i] += r;
                                sse = fmaf(r, r, sse);
                            } else {
                                acc[i] += row[u][i];
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();                    // list consumed before the next round overwrites it
    }
    if (act) store_vec<VEC>(Rbar + (int64_t)a * D + d, acc);
    if (counts != nullptr && blockIdx.y == 0 && threadIdx.x == 0) counts[a] = (int64_t)cnt;
    if (sse_part != nullptr) {
        const float t = warp_sum(act ? sse : 0.f);
        if (lane == 0) sse_w[warp] = t;
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot = 0.0;
            for (int w = 0; w < SCAN_THREADS / 32; ++w) tot += (double)sse_w[w];
            sse_part[(int64_t)a * n_slices + blockIdx.y] = tot;
        }
    }
}

// fixed-order double reduction of the per-(chunk, slice) squared-error partials.  `tail` (data-parallel form, may be
// NULL) receives the packed tail of the sum and the local patch count (pack_tail; 4-byte aligned, stored as floats).
__global__ void __launch_bounds__(1024) sse_reduce_kernel(const double* __restrict__ part, int64_t m,
                                                          double* __restrict__ out, float* __restrict__ tail,
                                                          int64_t n_patches) {
    pdl_begin();
    trace_stamp(s_trace_buf, 12);
    __shared__ double sh[1024];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += 1024) s += part[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (out != nullptr) *out = sh[0];
        if (tail != nullptr) {
            const float4 t = pack_tail(sh[0], n_patches);
            tail[0] = t.x; tail[1] = t.y; tail[2] = t.z; tail[3] = t.w;
        }
    }
}

template <int VEC>
static int launch_levels(const float* x, const Geom& g, const AccumPlan& pl, const int* skey,
                         const int* sid, const int* offsets, const float* Wt, float* Rbar,
                         int64_t* counts, double* sse, float* tail, float* partial, double* sse_part,
                         cudaStream_t st) {
    const int n_slices = (int)ceil_div64(g.D, 32 * VEC);
    if (pl.n_chunks > 0) {
        int64_t warps = pl.n_chunks * n_slices;
        unsigned blocks = (unsigned)ceil_div64(warps, ACC_WARPS);
        constexpr size_t ring_bytes = (size_t)ACC_WARPS * 2 * 2 * L1_GROUP<VEC>::value * 32 * VEC * sizeof(float) +
                                      (size_t)ACC_WARPS * 2 * L1_GROUP<VEC>::value * sizeof(int4);
        static PerDeviceFlag attr_done;
        const auto kernel = seg_level1_kernel<VEC>;
        int rc = smem_opt_in(attr_done, &kernel, 1, (int)ring_bytes, "accumulate");
        if (rc) return rc;
        launch_pdl(seg_level1_kernel<VEC>, blocks, ACC_WARPS * 32, ring_bytes, st, 
            x, g, skey, sid, offsets, Wt, Rbar, partial, ((sse || tail) && Wt) ? sse_part : nullptr,
            pl.S, pl.n_chunks, n_slices);
        rc = check_launch("seg_level1_kernel");
        if (rc) return rc;
    }
    {
        int64_t warps = (int64_t)pl.K * n_slices;
        unsigned blocks = (unsigned)ceil_div64(warps, ACC_WARPS);
        launch_pdl(seg_level2_kernel<VEC>, blocks, ACC_WARPS * 32, 0, st, offsets, partial, Rbar, counts,
                                                                 pl.K, g.D, pl.S, n_slices);
        int rc = check_launch("seg_level2_kernel");
        if (rc) return rc;
    }
    if (sse != nullptr || tail != nullptr) {
        int64_t m = (Wt != nullptr) ? pl.n_chunks * n_slices : 0;
        launch_pdl(sse_reduce_kernel, 1, 1024, 0, st, sse_part, m, sse, tail, g.n_patches);
        return check_launch("sse_reduce_kernel");
    }
    return SOM_OK;
}

// Which path and vector width accumulate_impl runs, from the shape, the batch's own vector width and the alignment of
// Wt and Rbar.  Scan path (static rule on the shape): tiny batches, where the eight launches of the sorted path are the
// cost; a CTA's run time grows with its unit's hit count, so skewed large batches stay on the sorted path (measured at
// C3, 4096 patches: 71 us sorted vs 135 us scanned).  Sorted paths: the library's counting sort where the plan has sort
// blocks, cub's radix sort otherwise (n = 0 sorts nothing and takes that branch for the offsets alone).
struct AccumRoute { int path, vec, n_slices; };
static AccumRoute accumulate_route(const Geom& g, const AccumPlan& pl, const float* Wt, const float* Rbar) {
    const int64_t n = g.n_patches;
    int vec = g.vec;
    if (Wt != nullptr && ((uintptr_t)Wt & 15) != 0) vec = 1;
    if (((uintptr_t)Rbar & 15) != 0) vec = 1;
    if (n > 0 && n <= 2048 && n * (int64_t)pl.K <= (1ll << 26))
        return {ACC_SCAN, vec, (int)ceil_div64(g.D, (int64_t)SCAN_THREADS * vec)};
    // a warp covers 32 * vec features of one patch row: keep all lanes busy for short rows (C4, D = 64: vec 2)
    while (vec > 1 && 32 * vec > g.D) vec >>= 1;
    return {(n > 0 && pl.cs_blocks > 0) ? ACC_COUNTING : ACC_RADIX, vec, (int)ceil_div64(g.D, 32 * vec)};
}

}  // namespace som

using namespace som;

extern "C" size_t som_accumulate_workspace_bytes(int64_t n_patches, int D, int K) {
    AccumPlan pl;
    if (make_plan(&pl, n_patches, D, K, true) != SOM_OK) return 0;
    return pl.total;
}

static int accumulate_impl(const float* x, int64_t n_img, int C, int H, int Wd, int pH,
                           int pW, const int64_t* bmu, const float* Wt, int K,
                           float* Rbar, int64_t* counts, double* sse, float* tail,
                           void* ws, size_t ws_bytes, void* stream) {
    // an empty (ragged data-parallel) share is valid: Rbar is zero-filled, the tail carries zeros
    SOM_REQUIRE(Rbar && ((x && bmu) || n_img == 0), SOM_E_BADARG, "accumulate: null pointer");
    SOM_REQUIRE(K > 0, SOM_E_BADARG, "accumulate: K=%d", K);
    Geom g;
    int rc = make_geom(&g, x, n_img, C, H, Wd, pH, pW);
    if (rc) return rc;
    AccumPlan pl;
    rc = make_plan(&pl, g.n_patches, g.D, K, true);
    if (rc) return rc;
    SOM_REQUIRE(ws != nullptr && ws_bytes >= pl.total, SOM_E_WORKSPACE,
                "accumulate: workspace %zu < required %zu", ws_bytes, pl.total);
    SOM_REQUIRE(((uintptr_t)ws & 255) == 0, SOM_E_BADARG, "accumulate: workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char* base = (char*)ws;
    int* keys_a = (int*)(base + pl.off_keys_a);
    int* keys_b = (int*)(base + pl.off_keys_b);
    int* vals_a = (int*)(base + pl.off_vals_a);
    int* vals_b = (int*)(base + pl.off_vals_b);
    int* offsets = (int*)(base + pl.off_offsets);
    float* partial = (float*)(base + pl.off_partial);
    double* sse_part = (double*)(base + pl.off_sse);
    void* cub_tmp = base + pl.off_cub;
    const int64_t n = g.n_patches;
    const AccumRoute route = accumulate_route(g, pl, Wt, Rbar);
    const int vec = route.vec;

    if (route.path == ACC_SCAN) {
        const int n_slices = route.n_slices;
        dim3 grid((unsigned)K, (unsigned)n_slices);
        double* sp = ((sse || tail) && Wt) ? sse_part : nullptr;
        if (vec == 4) launch_pdl(acc_scan_kernel<4>, grid, SCAN_THREADS, 0, st, x, g, bmu, K, Wt, Rbar, counts, sp, n_slices);
        else if (vec == 2) launch_pdl(acc_scan_kernel<2>, grid, SCAN_THREADS, 0, st, x, g, bmu, K, Wt, Rbar, counts, sp, n_slices);
        else launch_pdl(acc_scan_kernel<1>, grid, SCAN_THREADS, 0, st, x, g, bmu, K, Wt, Rbar, counts, sp, n_slices);
        rc = check_launch("acc_scan_kernel");
        if (rc) return rc;
        if (sse != nullptr || tail != nullptr) {
            launch_pdl(sse_reduce_kernel, 1, 1024, 0, st, sse_part, (Wt != nullptr) ? (int64_t)K * n_slices : 0, sse, tail, n);
            return check_launch("sse_reduce_kernel");
        }
        return SOM_OK;
    }

    const int* skey = keys_a;
    const int* sid = vals_a;
    if (route.path == ACC_COUNTING) {
        int* hist = (int*)(base + pl.off_hist);
        int* total = hist + (size_t)pl.cs_blocks * K;
        const size_t bins = (size_t)K * sizeof(int);
        static PerDeviceFlag attr_done;
        static const void* const kernels[2] = {(const void*)csort_hist_kernel, (const void*)csort_scatter_kernel};
        rc = smem_opt_in(attr_done, kernels, 2, CS_KMAX * 4, "accumulate");
        if (rc) return rc;
        launch_pdl(csort_hist_kernel, pl.cs_blocks, CS_THREADS, bins, st, bmu, n, K, pl.cs_per, hist);
        rc = check_launch("csort_hist_kernel");
        if (rc) return rc;
        launch_pdl(csort_prefix_kernel, (unsigned)ceil_div64(K, 256), 256, 0, st, hist, pl.cs_blocks, K, total);
        rc = check_launch("csort_prefix_kernel");
        if (rc) return rc;
        launch_pdl(csort_offsets_kernel, 1, 1024, 0, st, total, K, offsets);
        rc = check_launch("csort_offsets_kernel");
        if (rc) return rc;
        launch_pdl(csort_scatter_kernel, pl.cs_blocks, CS_THREADS, bins, st, bmu, n, K, pl.cs_per, hist, offsets, keys_a, vals_a);
        rc = check_launch("csort_scatter_kernel");
        if (rc) return rc;
    } else {
    if (n > 0) {
        launch_pdl(pairs_kernel, (unsigned)ceil_div64(n, 256), 256, 0, st, bmu, n, K, keys_a, vals_a);
        rc = check_launch("pairs_kernel");
        if (rc) return rc;
        cub::DoubleBuffer<int> kb(keys_a, keys_b), vb(vals_a, vals_b);
        size_t bytes = pl.cub_bytes + 256;
        cudaError_t e = cub::DeviceRadixSort::SortPairs(cub_tmp, bytes, kb, vb, (int)n, 0, pl.end_bit, st);
        if (e != cudaSuccess) { set_error("accumulate: radix sort: %s", cudaGetErrorString(e)); return (int)e; }
        skey = kb.Current();
        sid = vb.Current();
    }
    launch_pdl(offsets_kernel, (unsigned)ceil_div64(n + 1, 256), 256, 0, st, skey, n, K, offsets);
    rc = check_launch("offsets_kernel");
    if (rc) return rc;
    }

    if (vec == 4) return launch_levels<4>(x, g, pl, skey, sid, offsets, Wt, Rbar, counts, sse, tail, partial, sse_part, st);
    if (vec == 2) return launch_levels<2>(x, g, pl, skey, sid, offsets, Wt, Rbar, counts, sse, tail, partial, sse_part, st);
    return launch_levels<1>(x, g, pl, skey, sid, offsets, Wt, Rbar, counts, sse, tail, partial, sse_part, st);
}

// debug: the plan of an accumulation, as APF_COUNT int64 fields (som_common.cuh: AccumPlanField, -1 where a field does
// not apply); the first n_out are written.  x, Wt and Rbar are the pointers a call would pass (Wt may be null); only
// their alignment is read.  The answers come from the rules accumulate_impl uses.  Not in somcb.h: a test hook.
extern "C" SOM_API int som_debug_accumulate_plan(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                                 const float* Wt, int K, const float* Rbar, int64_t* out, int n_out) {
    SOM_REQUIRE(K > 0 && out != nullptr && n_out >= 0, SOM_E_BADARG, "accumulate plan: K=%d, output", K);
    Geom g;
    int rc = make_geom(&g, x, n_img, C, H, Wd, pH, pW);
    if (rc) return rc;
    AccumPlan pl;
    rc = make_plan(&pl, g.n_patches, g.D, K, false);
    if (rc) return rc;
    const AccumRoute r = accumulate_route(g, pl, Wt, Rbar);
    int64_t f[APF_COUNT];
    for (int i = 0; i < APF_COUNT; ++i) f[i] = -1;
    f[APF_PATH] = r.path;
    f[APF_VEC] = r.vec;
    f[APF_N_SLICES] = r.n_slices;
    if (r.path != ACC_SCAN) { f[APF_S] = pl.S; f[APF_N_CHUNKS] = pl.n_chunks; }
    if (r.path == ACC_COUNTING) { f[APF_CS_PER] = pl.cs_per; f[APF_CS_BLOCKS] = pl.cs_blocks; }
    for (int i = 0; i < n_out && i < APF_COUNT; ++i) out[i] = f[i];
    return SOM_OK;
}

extern "C" int som_accumulate_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH,
                                       int pW, const int64_t* bmu, const float* Wt, int K,
                                       float* Rbar, int64_t* counts, double* sse,
                                       void* ws, size_t ws_bytes, void* stream) {
    return accumulate_impl(x, n_img, C, H, Wd, pH, pW, bmu, Wt, K, Rbar, counts, sse, nullptr, ws, ws_bytes, stream);
}

extern "C" int som_accumulate_packed_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH,
                                              int pW, const int64_t* bmu, const float* Wt, int K,
                                              float* packed, void* ws, size_t ws_bytes, void* stream) {
    SOM_REQUIRE(packed && Wt, SOM_E_BADARG, "accumulate(packed): null pointer");
    const int64_t kd = (int64_t)K * C * pH * pW;
    return accumulate_impl(x, n_img, C, H, Wd, pH, pW, bmu, Wt, K, packed, nullptr, nullptr, packed + kd, ws, ws_bytes,
                           stream);
}

extern "C" int som_backward_nchw_f32(const float* grad_out, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                     const int64_t* bmu, int K, float* Rbar, void* ws, size_t ws_bytes,
                                     void* stream) {
    return som_accumulate_nchw_f32(grad_out, n_img, C, H, Wd, pH, pW, bmu, nullptr, K, Rbar, nullptr, nullptr, ws,
                                   ws_bytes, stream);
}
