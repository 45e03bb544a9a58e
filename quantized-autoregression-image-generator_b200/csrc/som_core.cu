// libsomcb core: error plumbing, geometry, and the small HBM-bound kernels of the SOM path
// (codebook norms, candidate merge, hit histogram, quantise/gather, Adam, row compaction).
#include "som_common.cuh"
#include "som_step_rules.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <atomic>
#include <mutex>
#include <string.h>

namespace som {
SOM_TRACE_TU(trace_set_core)

static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return SOM_OK;
}

unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

int current_device() {
    int dev = -1;
    return cudaGetDevice(&dev) == cudaSuccess ? dev : -1;
}

int sm_count() {
    static int cached[64];
    static std::once_flag once;
    std::call_once(once, [] { memset(cached, 0, sizeof(cached)); });
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

int make_geom(Geom* g, const void* x, int64_t n_img, int C, int H, int W, int pH, int pW, int elem_bytes) {
    SOM_REQUIRE(n_img >= 0 && C > 0 && H > 0 && W > 0 && pH > 0 && pW > 0, SOM_E_BADARG,
                "geometry: non-positive dimension (n_img=%lld C=%d H=%d W=%d pH=%d pW=%d)",
                (long long)n_img, C, H, W, pH, pW);
    SOM_REQUIRE(H % pH == 0 && W % pW == 0, SOM_E_SHAPE,
                "geometry: image %dx%d is not divisible by patch %dx%d", H, W, pH, pW);
    g->n_img = n_img; g->C = C; g->H = H; g->W = W; g->pH = pH; g->pW = pW;
    g->gH = H / pH; g->gW = W / pW; g->seq = g->gH * g->gW;
    g->D = C * pH * pW;
    g->n_patches = n_img * g->seq;
    g->img_stride = (int64_t)C * H * W;
    uintptr_t a = (uintptr_t)x;
    if (elem_bytes == 2) {
        SOM_REQUIRE((a & 1) == 0, SOM_E_BADARG, "geometry: 16-bit buffer is not 2-byte aligned");
        g->vec = 1;
        if (pW % 4 == 0 && (a & 7) == 0) g->vec = 4;
        else if (pW % 2 == 0 && (a & 3) == 0) g->vec = 2;
        return SOM_OK;
    }
    SOM_REQUIRE((a & 3) == 0, SOM_E_BADARG, "geometry: fp32 buffer is not 4-byte aligned");
    g->vec = 1;
    if (pW % 4 == 0 && (a & 15) == 0) g->vec = 4;
    else if (pW % 2 == 0 && (a & 7) == 0) g->vec = 2;
    return SOM_OK;
}

// ---------------------------------------------------------------------------------------------
// K0: ||W_j||^2, one warp per unit, fixed summation order (lane-strided, then butterfly)
// ---------------------------------------------------------------------------------------------
// Rows of at most 16 (8) features use 16 (8) lanes per unit: the lanes a full warp would leave idle only add
// exact zeros in the butterfly, and the d-loop below is unrolled with loads hoisted but the FMAs kept in the
// original order (a masked element contributes fma(0, 0, s) = s), so the result is bit-identical to the
// one-warp-per-unit, lane-strided order.  A warp owns (32 / G) * U consecutive units and has U * J loads in flight
// per lane (short rows were latency-bound at 10-26 % of the HBM copy rate with one load in flight).
// T = __half / __nv_bfloat16 (16-bit codebooks): each element is widened exactly and summed in the same order, so the
// norms equal those of the codebook's fp32 copy bit for bit.
__device__ __forceinline__ float ld_widen(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_widen(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float ld_widen(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }

template <int G, int U, int J, typename T = float>
__global__ void __launch_bounds__(256) norm2_kernel(const T* __restrict__ W, int K, int D,
                                                    float* __restrict__ out) {
    pdl_begin();
    trace_stamp(s_trace_buf, 5);
    constexpr int RPW = (32 / G) * U;                       // units per warp per iteration
    const int lane = threadIdx.x & (G - 1);
    const int sub = (threadIdx.x & 31) / G;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warp = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t base = warp * RPW; base < K; base += n_warp * RPW) {       // warp-uniform bound
        float s[U];
        int64_t r[U];
#pragma unroll
        for (int k = 0; k < U; ++k) { s[k] = 0.f; r[k] = base + k * (32 / G) + sub; }
        for (int d0 = lane; d0 < D; d0 += 32 * J) {
            float v[U][J];
#pragma unroll
            for (int k = 0; k < U; ++k)
#pragma unroll
                for (int j = 0; j < J; ++j)
                    v[k][j] = (r[k] < K && d0 + 32 * j < D) ? ld_widen(W + r[k] * D + d0 + 32 * j) : 0.f;
#pragma unroll
            for (int k = 0; k < U; ++k)
#pragma unroll
                for (int j = 0; j < J; ++j) s[k] = fmaf(v[k][j], v[k][j], s[k]);
        }
#pragma unroll
        for (int k = 0; k < U; ++k) {
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
            if (lane == 0 && r[k] < K) out[r[k]] = s[k];
        }
    }
}

// Long rows (D >= 2048: the whole-fmap codebook, a few hundred units of 16 KB): one CTA per unit, because one warp
// per four units leaves most SMs without work (C3: 128 warps, 16 us for 8 MB).  Thread t adds d = t, t + 256, ... in
// order (four loads in flight), then a warp butterfly and the eight warp sums in warp order: fixed order, and the
// rule depends on D only, so a unit's norm does not depend on how many units the launch (or the shard) holds.
template <typename T = float>
__global__ void __launch_bounds__(256) norm2_long_kernel(const T* __restrict__ W, int D, float* __restrict__ out) {
    pdl_begin();
    trace_stamp(s_trace_buf, 5);
    __shared__ float part[8];
    const T* row = W + (int64_t)blockIdx.x * D;
    float s = 0.f;
    for (int d0 = threadIdx.x; d0 < D; d0 += 4 * 256) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (d0 + 256 * j < D) ? ld_widen(row + d0 + 256 * j) : 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) s = fmaf(v[j], v[j], s);
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = part[0];
#pragma unroll
        for (int w = 1; w < 8; ++w) t += part[w];
        out[blockIdx.x] = t;
    }
}

// ---------------------------------------------------------------------------------------------
// K1b: candidate merge
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) merge_kernel(const float* __restrict__ rd,
                                                    const int64_t* __restrict__ idx, int R,
                                                    int64_t n, int64_t* __restrict__ out_idx,
                                                    float* __restrict__ out_rd) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    float best = rd[p];
    int64_t bi = idx[p];
    for (int r = 1; r < R; ++r) {
        const float v = rd[(int64_t)r * n + p];
        const int64_t i = idx[(int64_t)r * n + p];
        argmin_merge(best, bi, v, i);
    }
    out_idx[p] = bi;
    if (out_rd) out_rd[p] = best;
}

// ---------------------------------------------------------------------------------------------
// K5: hit histogram.  Small K: shared-memory private counts per CTA, one global merge per CTA.
// Large K: direct 64-bit global atomics (integer, so the result is order-independent).
// ---------------------------------------------------------------------------------------------
// Eight indices per thread per iteration as four independent 16-byte loads: with one 8-byte load in flight per
// thread the kernel was latency-bound at ~2.7 TB/s; this keeps 64 B per thread in flight.
__global__ void __launch_bounds__(512) hist_smem_kernel(const int64_t* __restrict__ idx, int64_t n,
                                                        int K, unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned int sh[];
    for (int i = threadIdx.x; i < K; i += blockDim.x) sh[i] = 0u;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t n8 = ((reinterpret_cast<uintptr_t>(idx) & 15) == 0) ? n / 8 : 0;     // groups of 8 (aligned base)
    const longlong2* v = reinterpret_cast<const longlong2*>(idx);
    for (int64_t g = tid; g < n8; g += stride) {
        longlong2 a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] = __ldg(v + g * 4 + u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (a[u].x >= 0 && a[u].x < K) atomicAdd(&sh[a[u].x], 1u);
            if (a[u].y >= 0 && a[u].y < K) atomicAdd(&sh[a[u].y], 1u);
        }
    }
    for (int64_t p = n8 * 8 + tid; p < n; p += stride) {
        int64_t j = idx[p];
        if (j >= 0 && j < K) atomicAdd(&sh[j], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        unsigned int c = sh[i];
        if (c) atomicAdd(&counts[i], (unsigned long long)c);
    }
}

// Medium and large K: range-partitioned private counters.  The K units are cut into P ranges of at most
// HIST_RANGE_MAX (224 KB of 32-bit counters, one CTA per SM); CTA b counts range b % P over index slice b / P.
// The P CTAs of a slice are co-resident and walk the same addresses at the same pace, so the slice comes from HBM
// once and from L2 P - 1 times; only 1 / P of a CTA's indices hit a shared-memory atomic, the merge is one 64-bit
// global atomic per non-zero private counter.  Measured with direct global atomics instead: 17-20 % of the HBM copy
// rate on uniform hits and 2-3 % on skewed ones (same-address serialisation in L2).
constexpr int HIST_RANGE_MAX = 57344;
__global__ void __launch_bounds__(1024) hist_range_kernel(const int64_t* __restrict__ idx, int64_t n, int K,
                                                          int Kr, int P, unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned int sh[];
    const int r = blockIdx.x % P, sl = blockIdx.x / P, S = gridDim.x / P;
    const int64_t lo = (int64_t)r * Kr;
    const unsigned int width = (unsigned int)((lo + Kr <= K ? Kr : K - lo));
    for (int i = threadIdx.x; i < Kr; i += blockDim.x) sh[i] = 0u;
    __syncthreads();
    const int64_t stride = (int64_t)S * blockDim.x;
    const int64_t tid = sl * (int64_t)blockDim.x + threadIdx.x;
    // eight indices per thread per iteration as four independent 16-byte loads (sixteen measured slower: 82 -> 52 %
    // of the HBM copy rate at K = 32768)
    const int64_t n8 = ((reinterpret_cast<uintptr_t>(idx) & 15) == 0) ? n / 8 : 0;
    const longlong2* v = reinterpret_cast<const longlong2*>(idx);
    for (int64_t g = tid; g < n8; g += stride) {
        longlong2 a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] = __ldg(v + g * 4 + u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            // unsigned compare folds "below the range" and "negative" into one test
            const unsigned long long x = (unsigned long long)(a[u].x - lo), y = (unsigned long long)(a[u].y - lo);
            if (x < width) atomicAdd(&sh[x], 1u);
            if (y < width) atomicAdd(&sh[y], 1u);
        }
    }
    for (int64_t p = n8 * 8 + tid; p < n; p += stride) {
        const unsigned long long x = (unsigned long long)(idx[p] - lo);
        if (x < width) atomicAdd(&sh[x], 1u);
    }
    __syncthreads();
    for (unsigned int i = threadIdx.x; i < width; i += blockDim.x) {
        unsigned int c = sh[i];
        if (c) atomicAdd(&counts[lo + i], (unsigned long long)c);
    }
}

__global__ void __launch_bounds__(256) hist_global_kernel(const int64_t* __restrict__ idx, int64_t n,
                                                          int K, unsigned long long* __restrict__ counts) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t n8 = ((reinterpret_cast<uintptr_t>(idx) & 15) == 0) ? n / 8 : 0;
    const longlong2* v = reinterpret_cast<const longlong2*>(idx);
    for (int64_t g = tid; g < n8; g += stride) {
        longlong2 a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] = __ldg(v + g * 4 + u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (a[u].x >= 0 && a[u].x < K) atomicAdd(&counts[a[u].x], 1ull);
            if (a[u].y >= 0 && a[u].y < K) atomicAdd(&counts[a[u].y], 1ull);
        }
    }
    for (int64_t p = n8 * 8 + tid; p < n; p += stride) {
        int64_t j = idx[p];
        if (j >= 0 && j < K) atomicAdd(&counts[j], 1ull);
    }
}

// ---------------------------------------------------------------------------------------------
// token assembly for the Transformer trainer (train_quantized_transformer.py:411-455): one pass writes
// hr_input and hr_target from the two BMU index tensors -- replaces add / cat / repeat / cat
// one thread per output element; a row of hr_input followed by the row of hr_target
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) assemble_tokens_kernel(const int64_t* __restrict__ lr_idx,
                                                              const int64_t* __restrict__ hr_idx, int64_t n,
                                                              int lr_seq, int hr_seq, int64_t lr_K, int64_t hr_K,
                                                              int base_model, int64_t* __restrict__ hr_input,
                                                              int64_t* __restrict__ hr_target) {
    // A thread owns ONE column (blockIdx.y * 256 + tid) of the concatenated [hr_input | hr_target] row, so where its
    // value comes from (lr / hr index + shift, or a constant <start>/<end> token) is decided once; the CTA then walks
    // fmaps four at a time with the four loads in flight.  No integer division in the loop (one 64-bit division per
    // element kept the flat one-element-per-thread version at 60 % of the HBM copy rate).
    const int in_w = base_model ? lr_seq + hr_seq : 1 + hr_seq;
    const int row_w = in_w + hr_seq + 1;
    const int c = blockIdx.y * 256 + threadIdx.x;
    if (c >= row_w) return;
    const int64_t* src = nullptr;          // nullptr: constant column
    int64_t sstride = 0, add = 0, cval = hr_K;
    int64_t* dst;
    int64_t dstride;
    if (c < in_w) {
        dst = hr_input + c; dstride = in_w;
        if (base_model) {
            if (c < lr_seq) { src = lr_idx + c; sstride = lr_seq; }
            else { src = hr_idx + (c - lr_seq); sstride = hr_seq; add = lr_K; }
        } else if (c > 0) { src = hr_idx + (c - 1); sstride = hr_seq; }
    } else {
        const int kk = c - in_w;
        dst = hr_target + kk; dstride = hr_seq + 1;
        if (kk < hr_seq) { src = hr_idx + kk; sstride = hr_seq; }
    }
    constexpr int R = 4;
    for (int64_t i0 = (int64_t)blockIdx.x * R; i0 < n; i0 += (int64_t)gridDim.x * R) {
        int64_t val[R];
#pragma unroll
        for (int k = 0; k < R; ++k) {
            val[k] = cval;
            if (src != nullptr && i0 + k < n) val[k] = __ldg(src + (i0 + k) * sstride) + add;
        }
#pragma unroll
        for (int k = 0; k < R; ++k)
            if (i0 + k < n) __stcs(dst + (i0 + k) * dstride, val[k]);
    }
}

// ---------------------------------------------------------------------------------------------
// quantise: out[offset(p, d)] = table[idx[p]][d]   (gather + fused unpatchify)
// one thread per VEC-wide run; consecutive threads walk d fastest inside a patch.  T: float, or a 16-bit element
// (any format: the values are copied as bit patterns)
// ---------------------------------------------------------------------------------------------
template <int VEC, typename T = float>
__global__ void __launch_bounds__(256) quantize_kernel(const int64_t* __restrict__ idx,
                                                       const T* __restrict__ table, int K,
                                                       Geom g, T* __restrict__ out) {
    constexpr int RUN = VEC * (int)sizeof(T);             // bytes per run
    const int dv = g.D / VEC;
    int64_t total = g.n_patches * dv;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += stride) {
        int64_t p = t / dv;
        int d = (int)(t - p * dv) * VEC;
        int64_t u = idx[p];
        if (u < 0) u = 0;
        if (u >= K) u = K - 1;
        const T* src = table + u * (int64_t)g.D + d;
        T* dst = out + patch_base(g, p) + feat_off(g, d);
        if (RUN == 16) *reinterpret_cast<float4*>(dst) = *reinterpret_cast<const float4*>(src);
        else if (RUN == 8) *reinterpret_cast<float2*>(dst) = *reinterpret_cast<const float2*>(src);
        else if (RUN == 4) *reinterpret_cast<float*>(dst) = *reinterpret_cast<const float*>(src);
        else *dst = *src;
    }
}

// Output-ordered form for the common layouts (W % 4 == 0 and pW % 4 == 0 or pW == 2): a thread owns U fixed
// 16-byte runs of the image (run r = (blockIdx.y * U + k) * 256 + tid), so a warp writes 512 contiguous bytes; the
// patch slot and feature each run comes from (the inverse of patch_base / feat_off) are computed ONCE and the CTA
// then walks images, so the loop has no integer division (the first output-ordered version spent its time there:
// ~300 instructions per run).  Per image a thread loads its U (2U for pW = 2) indices, then the table rows from L2,
// then issues streaming stores.  The patch-ordered kernel above reached 21-36 % of the HBM copy rate.
// A run holds V = 16 / sizeof(T) values: 4 floats, or 8 16-bit values (then PW2 means pW == 4).
template <bool PW2, typename T = float>
__global__ void __launch_bounds__(256, 4) quantize_out_kernel(const int64_t* __restrict__ idx,
                                                           const T* __restrict__ table, int K,
                                                           Geom g, T* __restrict__ out) {
    constexpr int U = 4;
    constexpr int LV = sizeof(T) == 4 ? 2 : 3;            // log2 V
    const int wq = g.W >> LV;                             // 16-byte runs per image row
    const int quads_img = (int)(g.img_stride >> LV);
    int slot[U], d[U], r[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
        r[k] = (blockIdx.y * U + k) * 256 + threadIdx.x;
        slot[k] = -1; d[k] = 0;
        if (r[k] < quads_img) {
            const int row = r[k] / wq;                    // c * H + h
            const int w = (r[k] - row * wq) << LV;
            const int c = row / g.H;
            const int h = row - c * g.H;
            const int ph = h / g.pH;
            const int i = h - ph * g.pH;
            const int pw = w / g.pW;
            const int j = w - pw * g.pW;
            slot[k] = ph * g.gW + pw;
            d[k] = (c * g.pH + i) * g.pW + j;
        }
    }
    float4* out4 = reinterpret_cast<float4*>(out);
    // The indices of the CTA's NEXT image are requested before the current image's table rows, so an iteration costs
    // one load latency, not the index -> row chain (the kernel holds ~60 registers, 4 CTAs per SM).
    int u0[U], u1[U];
    auto fetch = [&](int64_t n, int (&a0)[U], int (&a1)[U]) {
        const int64_t* ip = idx + n * g.seq;
        int64_t t0[U], t1[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            t0[k] = 0; t1[k] = 0;
            if (slot[k] >= 0) {
                t0[k] = __ldg(ip + slot[k]);
                if (PW2) t1[k] = __ldg(ip + slot[k] + 1);
            }
        }
#pragma unroll
        for (int k = 0; k < U; ++k) {
            a0[k] = (int)(t0[k] < 0 ? 0 : (t0[k] >= K ? K - 1 : t0[k]));
            a1[k] = (int)(t1[k] < 0 ? 0 : (t1[k] >= K ? K - 1 : t1[k]));
        }
    };
    if ((int64_t)blockIdx.x < g.n_img) fetch(blockIdx.x, u0, u1);
    for (int64_t n = blockIdx.x; n < g.n_img; n += gridDim.x) {
        const int64_t nn = n + gridDim.x;
        const int64_t* ipn = idx + (nn < g.n_img ? nn : n) * g.seq;
        int64_t t0[U], t1[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {                     // next image's indices: in flight during the row loads
            t0[k] = 0; t1[k] = 0;
            if (slot[k] >= 0) {
                t0[k] = __ldg(ipn + slot[k]);
                if (PW2) t1[k] = __ldg(ipn + slot[k] + 1);
            }
        }
        float4 val[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            if (slot[k] < 0) continue;
            if (PW2) {
                const float2 lo = __ldg(reinterpret_cast<const float2*>(table + u0[k] * (int64_t)g.D + d[k]));
                const float2 hi = __ldg(reinterpret_cast<const float2*>(table + u1[k] * (int64_t)g.D + d[k]));
                val[k] = make_float4(lo.x, lo.y, hi.x, hi.y);
            } else {
                val[k] = __ldg(reinterpret_cast<const float4*>(table + u0[k] * (int64_t)g.D + d[k]));
            }
        }
#pragma unroll
        for (int k = 0; k < U; ++k)
            if (slot[k] >= 0) __stcs(out4 + n * quads_img + r[k], val[k]);
#pragma unroll
        for (int k = 0; k < U; ++k) {
            u0[k] = (int)(t0[k] < 0 ? 0 : (t0[k] >= K ? K - 1 : t0[k]));
            u1[k] = (int)(t1[k] < 0 ? 0 : (t1[k] >= K ? K - 1 : t1[k]));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K4: Adam (som_step_rules.cuh)
// ---------------------------------------------------------------------------------------------
// Four streams in, three out, 28 bytes per weight: 16-byte accesses, four weights per thread per iteration
// (the scalar one-weight loop reached 73 % of the HBM copy rate; the element-wise arithmetic is unchanged).
// SCALED: the gradient arrives unscaled (adam_update4).
template <bool SCALED>
__device__ __forceinline__ void adam_body(float* __restrict__ W, float* __restrict__ m, float* __restrict__ v,
                                          const float* __restrict__ g, int64_t n, const AdamScalars& a, float gscale) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const bool al = ((reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(m) |
                      reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(g)) & 15) == 0;
    const int64_t n4 = al ? n / 4 : 0;
    float4* W4 = reinterpret_cast<float4*>(W);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (int64_t q = tid; q < n4; q += stride) {
        float4 gq = __ldcs(g4 + q), mq = m4[q], vq = v4[q], wq = W4[q];
        adam_update4<SCALED>(a, gq, gscale, mq, vq, wq);
        W4[q] = wq; m4[q] = mq; v4[q] = vq;
    }
    for (int64_t i = n4 * 4 + tid; i < n; i += stride) {
        float mi = m[i], vi = v[i], wi = W[i];
        adam_update(a, SCALED ? g[i] * gscale : g[i], mi, vi, wi);
        W[i] = wi; m[i] = mi; v[i] = vi;
    }
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ W, float* __restrict__ m,
                                                   float* __restrict__ v, const float* __restrict__ g,
                                                   int64_t n, AdamScalars a) {
    pdl_begin();
    trace_stamp(s_trace_buf, 19);
    adam_body<false>(W, m, v, g, n, a, 0.f);
}

// Same rule with the step count read from device memory, so a captured CUDA graph of the training step can be
// replayed: t = *steps_done + 1.  step_bump_kernel advances it.
__global__ void __launch_bounds__(256) adam_dev_kernel(float* __restrict__ W, float* __restrict__ m,
                                                       float* __restrict__ v, const float* __restrict__ g,
                                                       int64_t n, double lr, double b1, double b2, float eps,
                                                       const int64_t* __restrict__ steps_done) {
    pdl_begin();
    trace_stamp(s_trace_buf, 19);
    const AdamScalars a = adam_scalars(lr, b1, b2, eps, (double)(*steps_done + 1));
    adam_body<false>(W, m, v, g, n, a, 0.f);
}
__global__ void step_bump_kernel(int64_t* steps_done) { *steps_done += 1; }

// Data-parallel tail: the gradient arrives UNSCALED (g = T @ Rbar_global) and the global batch size is only known on
// the device, from the all-reduced packed tail (som_accumulate_packed_nchw_f32); thread 0 also writes the mean squared
// error.
__global__ void __launch_bounds__(256) adam_dp_kernel(float* __restrict__ W, float* __restrict__ m,
                                                      float* __restrict__ v, const float* __restrict__ g,
                                                      int64_t n, int D, double lr, double b1, double b2, float eps,
                                                      int64_t* __restrict__ steps_done,
                                                      const float* __restrict__ tail, double* __restrict__ loss_out) {
    pdl_begin();
    trace_stamp(s_trace_buf, 18);
    const double t = (double)(steps_done[0] + 1);
    const TailTotals tt = tail_totals(tail, D);
    const AdamScalars a = adam_scalars(lr, b1, b2, eps, t);
    if (loss_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *loss_out = tail_loss(tail, tt.numel);
    adam_body<true>(W, m, v, g, n, a, tt.gscale);
    // the last block to finish advances the step count (every block read it when it started): steps_done[1] is the
    // arrival counter, left at zero again
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned long long old = atomicAdd(reinterpret_cast<unsigned long long*>(steps_done + 1), 1ull);
        if (old == (unsigned long long)gridDim.x - 1ull) { steps_done[1] = 0; steps_done[0] += 1; }
    }
}

template <typename T = float>
__global__ void __launch_bounds__(256) gather_rows_kernel(const T* __restrict__ W, int D,
                                                          const int64_t* __restrict__ keep,
                                                          int64_t n_keep, T* __restrict__ out) {
    int64_t total = n_keep * D;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += stride) {
        int64_t r = t / D;
        int d = (int)(t - r * D);
        out[t] = W[keep[r] * (int64_t)D + d];
    }
}

// 16-byte aligned rows of a multiple of 16 bytes (4 floats, 8 16-bit values): one 16-byte run per thread, four in
// flight
__global__ void __launch_bounds__(256) gather_rows4_kernel(const float4* __restrict__ W, int D4,
                                                           const int64_t* __restrict__ keep,
                                                           int64_t n_keep, float4* __restrict__ out) {
    constexpr int U = 4;
    const int64_t total = n_keep * D4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t0 < total; t0 += U * stride) {
        int64_t src[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const int64_t t = t0 + k * stride;
            src[k] = -1;
            if (t < total) {
                const int64_t r = t / D4;
                src[k] = __ldg(keep + r) * (int64_t)D4 + (t - r * D4);
            }
        }
        float4 val[U];
#pragma unroll
        for (int k = 0; k < U; ++k)
            if (src[k] >= 0) val[k] = __ldcs(W + src[k]);
#pragma unroll
        for (int k = 0; k < U; ++k)
            if (src[k] >= 0) __stcs(out + (t0 + k * stride), val[k]);
    }
}

// exact widening of 16-bit values to fp32: two packed in a 32-bit word, or one
__device__ __forceinline__ float2 widen2(uint32_t r, const __half*) {
    return __half22float2(*reinterpret_cast<const __half2*>(&r));
}
__device__ __forceinline__ float2 widen2(uint32_t r, const __nv_bfloat16*) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r));
}
__device__ __forceinline__ float widen1(__half v) { return __half2float(v); }
__device__ __forceinline__ float widen1(__nv_bfloat16 v) { return __bfloat162float(v); }

// fp16 / bf16 -> fp32 (exact), eight elements per step with 16-byte loads and stores when both buffers are 16-byte
// aligned: the fp32 kernels read a 16-bit batch through this copy (som_convert_f16_f32, som_convert_bf16_f32)
template <typename T>
__global__ void __launch_bounds__(256) convert_16_f32_kernel(const T* __restrict__ in, int64_t n,
                                                             float* __restrict__ out, int vec8) {
    pdl_begin();
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t done = 0;
    if (vec8) {
        const int64_t n8 = n >> 3;
        for (int64_t i = t; i < n8; i += stride) {
            const uint4 r = __ldcs(reinterpret_cast<const uint4*>(in) + i);
            const float2 a = widen2(r.x, in), b = widen2(r.y, in), c = widen2(r.z, in), d = widen2(r.w, in);
            float4* o = reinterpret_cast<float4*>(out) + 2 * i;
            o[0] = make_float4(a.x, a.y, b.x, b.y);
            o[1] = make_float4(c.x, c.y, d.x, d.y);
        }
        done = n8 << 3;
    }
    for (int64_t i = done + t; i < n; i += stride) out[i] = widen1(in[i]);
}

static inline int grid_for(int64_t work_items, int threads, int per_sm) {
    int64_t want = ceil_div64(work_items, threads);
    int64_t cap = (int64_t)sm_count() * per_sm;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

template <typename T>
static int convert_16_f32(const char* who, const void* in, int64_t n, float* out, void* stream) {
    SOM_REQUIRE(n >= 0, SOM_E_BADARG, "%s: n=%lld", who, (long long)n);
    if (n == 0) return SOM_OK;
    SOM_REQUIRE(in && out, SOM_E_BADARG, "%s: null pointer", who);
    SOM_REQUIRE((((uintptr_t)in) & 1) == 0 && (((uintptr_t)out) & 3) == 0, SOM_E_BADARG, "%s: misaligned buffer", who);
    const int vec8 = ((((uintptr_t)in) | ((uintptr_t)out)) & 15) == 0 ? 1 : 0;
    const int blocks = grid_for(vec8 ? ceil_div64(n, 8) : n, 256, 8);
    launch_pdl(convert_16_f32_kernel<T>, blocks, 256, 0, (cudaStream_t)stream, (const T*)in, n, out, vec8);
    return check_launch("convert_16_f32_kernel");
}

template <typename T>
static int prepare_codebook(const T* W, int K, int D, float* c_norm2, void* stream) {
    SOM_REQUIRE(W && c_norm2, SOM_E_BADARG, "prepare_codebook: null pointer");
    SOM_REQUIRE(K > 0 && D > 0, SOM_E_BADARG, "prepare_codebook: K=%d D=%d", K, D);
    cudaStream_t st = (cudaStream_t)stream;
    if (D >= 2048) {
        launch_pdl(norm2_long_kernel<T>, (unsigned)K, 256, 0, st, W, D, c_norm2);
        return check_launch("norm2_long_kernel");
    }
    if (D > 16) {            // 4 units x 4 row segments in flight per lane
        int blocks = grid_for(ceil_div64(K, 4) * 32, 256, 8);
        launch_pdl(norm2_kernel<32, 4, 4, T>, blocks, 256, 0, st, W, K, D, c_norm2);
    } else if (D > 8) {      // 2 x 8 units per warp
        int blocks = grid_for(ceil_div64(K, 16) * 32, 256, 8);
        launch_pdl(norm2_kernel<16, 8, 1, T>, blocks, 256, 0, st, W, K, D, c_norm2);
    } else {                 // 4 x 8 units per warp
        int blocks = grid_for(ceil_div64(K, 32) * 32, 256, 8);
        launch_pdl(norm2_kernel<8, 8, 1, T>, blocks, 256, 0, st, W, K, D, c_norm2);
    }
    return check_launch("norm2_kernel");
}

// V = values per 16-byte run: 4 floats or 8 16-bit values
template <typename T>
static int quantize_nchw(const int64_t* idx, const T* table, int K, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                         T* out, void* stream) {
    constexpr int ES = (int)sizeof(T), V = 16 / ES;
    SOM_REQUIRE(table && ((idx && out) || n_img == 0), SOM_E_BADARG, "quantize: null pointer");
    SOM_REQUIRE(K > 0, SOM_E_BADARG, "quantize: K=%d", K);
    Geom g;
    int rc = make_geom(&g, out, n_img, C, H, Wd, pH, pW, ES);
    if (rc) return rc;
    if (g.n_patches == 0) return SOM_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const bool pw4 = (pW % V == 0), pw2 = (pW == V / 2);
    if (Wd % V == 0 && ((uintptr_t)out & 15) == 0 && (pw4 || pw2) && g.img_stride >= 256 * V &&
        g.img_stride / (256 * V) < 65535 &&
        ((uintptr_t)table & (pw4 ? 15 : 7)) == 0) {
        const int64_t quads_img = g.img_stride / V;
        const int gy = (int)ceil_div64(quads_img, 256 * 4);
        int gx = sm_count() * 8 / gy;
        if (gx < 1) gx = 1;
        if (gx > g.n_img) gx = (int)g.n_img;
        dim3 blocks((unsigned)gx, (unsigned)gy);
        if (pw2) quantize_out_kernel<true, T><<<blocks, 256, 0, s>>>(idx, table, K, g, out);
        else quantize_out_kernel<false, T><<<blocks, 256, 0, s>>>(idx, table, K, g, out);
        return check_launch("quantize_out_kernel");
    }
    int vec = g.vec;
    if (((uintptr_t)table & (4 * ES - 1)) != 0 || g.D % 4 != 0) vec = (vec == 4) ? 1 : vec;
    if (vec == 2 && (((uintptr_t)table & (2 * ES - 1)) != 0 || g.D % 2 != 0)) vec = 1;
    int64_t items = g.n_patches * (g.D / vec);
    int blocks = grid_for(items, 256, 16);
    if (vec == 4) quantize_kernel<4, T><<<blocks, 256, 0, s>>>(idx, table, K, g, out);
    else if (vec == 2) quantize_kernel<2, T><<<blocks, 256, 0, s>>>(idx, table, K, g, out);
    else quantize_kernel<1, T><<<blocks, 256, 0, s>>>(idx, table, K, g, out);
    return check_launch("quantize_kernel");
}

template <typename T>
static int gather_rows(const T* W, int D, const int64_t* keep, int64_t n_keep, T* out, void* stream) {
    constexpr int V = 16 / (int)sizeof(T);
    SOM_REQUIRE(W && keep && out, SOM_E_BADARG, "gather_rows: null pointer");
    SOM_REQUIRE(D > 0 && n_keep >= 0, SOM_E_BADARG, "gather_rows: D=%d n_keep=%lld", D, (long long)n_keep);
    if (n_keep == 0) return SOM_OK;
    if (D % V == 0 && (((uintptr_t)W | (uintptr_t)out) & 15) == 0) {
        int blocks = grid_for(n_keep * (D / V), 256 * 4, 8);
        gather_rows4_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(W), D / V, keep,
                                                                      n_keep, reinterpret_cast<float4*>(out));
        return check_launch("gather_rows4_kernel");
    }
    int blocks = grid_for(n_keep * D, 256, 16);
    gather_rows_kernel<T><<<blocks, 256, 0, (cudaStream_t)stream>>>(W, D, keep, n_keep, out);
    return check_launch("gather_rows_kernel");
}

}  // namespace som

using namespace som;

namespace som {
void trace_set_filter_tc(unsigned long long*);
void trace_set_filter(unsigned long long*);
void trace_set_l16(unsigned long long*);
void trace_set_accumulate(unsigned long long*);
void trace_set_peer(unsigned long long*);
}  // namespace som

namespace som {
static int g_pdl = 1;
bool pdl_enabled() { return g_pdl != 0; }
}
// debug: programmatic dependent launch on the step's kernel chain (default on); 0 = plain stream order, for A/B timing
extern "C" SOM_API void som_debug_set_pdl(int on) { som::g_pdl = on; }

// debug: hand every translation unit the trace buffer (8 KB + 64 KB of device memory, zero-filled; NULL switches it off)
extern "C" SOM_API int som_debug_trace(unsigned long long* buf) {
    som::trace_set_core(buf); som::trace_set_filter_tc(buf); som::trace_set_filter(buf); som::trace_set_l16(buf);
    som::trace_set_accumulate(buf); som::trace_set_peer(buf);
    return (int)cudaGetLastError();
}

extern "C" {

int som_version(void) { return SOM_ABI_VERSION; }

const char* som_last_error(void) { return som::g_err; }

uint64_t som_launch_count(void) { return som::launch_count(); }

int som_device_info(int* sm, int* major, int* minor) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { set_error("cudaGetDevice: %s", cudaGetErrorString(e)); return (int)e; }
    cudaDeviceProp p;
    e = cudaGetDeviceProperties(&p, dev);
    if (e != cudaSuccess) { set_error("cudaGetDeviceProperties: %s", cudaGetErrorString(e)); return (int)e; }
    if (sm) *sm = p.multiProcessorCount;
    if (major) *major = p.major;
    if (minor) *minor = p.minor;
    return SOM_OK;
}


int som_merge_candidates(const float* rd, const int64_t* idx, int R, int64_t n,
                         int64_t* out_idx, float* out_rd, void* stream) {
    SOM_REQUIRE(rd && idx && out_idx, SOM_E_BADARG, "merge_candidates: null pointer");
    SOM_REQUIRE(R > 0 && n >= 0, SOM_E_BADARG, "merge_candidates: R=%d n=%lld", R, (long long)n);
    if (n == 0) return SOM_OK;
    int blocks = (int)ceil_div64(n, 256);
    merge_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rd, idx, R, n, out_idx, out_rd);
    return check_launch("merge_kernel");
}

int som_histogram_i64(const int64_t* idx, int64_t n, int K, int64_t* counts, void* stream) {
    SOM_REQUIRE(counts && (idx || n == 0), SOM_E_BADARG, "histogram: null pointer");
    SOM_REQUIRE(K > 0 && n >= 0, SOM_E_BADARG, "histogram: K=%d n=%lld", K, (long long)n);
    if (n == 0) return SOM_OK;
    auto* c = reinterpret_cast<unsigned long long*>(counts);
    if (K <= 12288) {   // 48 KB of private counters: no opt-in needed, 4 CTAs/SM
        int blocks = grid_for(n, 512 * 16, 4);
        hist_smem_kernel<<<blocks, 512, (size_t)K * sizeof(unsigned int), (cudaStream_t)stream>>>(idx, n, K, c);
        return check_launch("hist_smem_kernel");
    }
    const int sms = sm_count();
    const int P = (int)ceil_div64(K, HIST_RANGE_MAX);
    // also for few indices per unit (C5 shard, 2^20 indices against 32768 units: 12.7-14.3 us, the same as direct
    // global atomics on uniform hits) -- skewed hits would serialise on one L2 address there
    if (P <= sms) {
        static PerDeviceFlag attr_done;
        const auto kernel = hist_range_kernel;
        int rc = smem_opt_in(attr_done, &kernel, 1, HIST_RANGE_MAX * (int)sizeof(unsigned int), "histogram");
        if (rc) return rc;
        const int Kr = (int)(ceil_div64(ceil_div64(K, P), 32) * 32);
        int S = sms / P;                                     // index slices; every CTA is resident (one per SM)
        const int64_t per_cta = (int64_t)1024 * 8;
        if ((int64_t)S * per_cta > n) S = (int)(n / per_cta > 0 ? n / per_cta : 1);
        // 32-bit private counters: a CTA never sees more than 2^31 indices per launch
        const int64_t chunk = (int64_t)S << 31;
        for (int64_t at = 0; at < n; at += chunk) {
            const int64_t m = (n - at < chunk) ? n - at : chunk;
            hist_range_kernel<<<P * S, 1024, (size_t)Kr * sizeof(unsigned int), (cudaStream_t)stream>>>(
                idx + at, m, K, Kr, P, c);
            rc = check_launch("hist_range_kernel");
            if (rc) return rc;
        }
        return SOM_OK;
    }
    int blocks = grid_for(n, 256 * 16, 8);
    hist_global_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(idx, n, K, c);
    return check_launch("hist_global_kernel");
}


int som_assemble_tokens_i64(const int64_t* lr_idx, const int64_t* hr_idx, int64_t n, int lr_seq, int hr_seq,
                            int64_t lr_K, int64_t hr_K, int base_model, int64_t* hr_input, int64_t* hr_target,
                            void* stream) {
    SOM_REQUIRE((hr_idx && hr_input && hr_target) || n == 0, SOM_E_BADARG, "assemble_tokens: null pointer");
    SOM_REQUIRE(!base_model || lr_idx || n == 0, SOM_E_BADARG, "assemble_tokens: base model needs lr_idx");
    SOM_REQUIRE(n >= 0 && hr_seq > 0 && lr_seq >= 0, SOM_E_BADARG, "assemble_tokens: n=%lld lr_seq=%d hr_seq=%d",
                (long long)n, lr_seq, hr_seq);
    if (n == 0) return SOM_OK;
    const int row_w = (base_model ? lr_seq + hr_seq : 1 + hr_seq) + hr_seq + 1;
    const int gy = (row_w + 255) / 256;
    int64_t gx = ceil_div64(n, 4), cap = (int64_t)sm_count() * 16 / gy;
    if (cap < 1) cap = 1;
    dim3 blocks((unsigned)(gx < cap ? gx : cap), (unsigned)gy);
    assemble_tokens_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(lr_idx, hr_idx, n, lr_seq, hr_seq, lr_K, hr_K,
                                                                     base_model, hr_input, hr_target);
    return check_launch("assemble_tokens_kernel");
}

int som_adam_f32(float* W, float* m, float* v, const float* g, int64_t n,
                 double lr, double b1, double b2, double eps, int64_t step, void* stream) {
    SOM_REQUIRE(W && m && v && g, SOM_E_BADARG, "adam: null pointer");
    SOM_REQUIRE(n >= 0 && step >= 1, SOM_E_BADARG, "adam: n=%lld step=%lld", (long long)n, (long long)step);
    if (n == 0) return SOM_OK;
    int blocks = grid_for(n, 256 * 4, 8);
    const AdamScalars a = adam_scalars(lr, b1, b2, (float)eps, (double)step);      // on the host
    launch_pdl(adam_kernel, blocks, 256, 0, (cudaStream_t)stream, W, m, v, g, n, a);
    return check_launch("adam_kernel");
}

int som_adam_devstep_f32(float* W, float* m, float* v, const float* g, int64_t n,
                         double lr, double b1, double b2, double eps, int64_t* steps_done, void* stream) {
    SOM_REQUIRE(W && m && v && g && steps_done, SOM_E_BADARG, "adam(devstep): null pointer");
    SOM_REQUIRE(n >= 0, SOM_E_BADARG, "adam(devstep): n=%lld", (long long)n);
    if (n > 0) {
        int blocks = grid_for(n, 256 * 4, 8);
        launch_pdl(adam_dev_kernel, blocks, 256, 0, (cudaStream_t)stream, W, m, v, g, n, lr, b1, b2, (float)eps, steps_done);
        int rc = check_launch("adam_dev_kernel");
        if (rc) return rc;
    }
    step_bump_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(steps_done);
    return check_launch("step_bump_kernel");
}

int som_adam_dp_f32(float* W, float* m, float* v, const float* g, int64_t n, int D,
                    double lr, double b1, double b2, double eps, int64_t* steps_done,
                    const float* tail, double* loss_out, void* stream) {
    SOM_REQUIRE(W && m && v && g && steps_done && tail, SOM_E_BADARG, "adam(dp): null pointer");
    SOM_REQUIRE(n >= 0 && D > 0, SOM_E_BADARG, "adam(dp): n=%lld D=%d", (long long)n, D);
    if (n > 0) {
        int blocks = grid_for(n, 256 * 4, 8);
        launch_pdl(adam_dp_kernel, blocks, 256, 0, (cudaStream_t)stream, W, m, v, g, n, D, lr, b1, b2, (float)eps, steps_done,
                                                                tail, loss_out);
        return check_launch("adam_dp_kernel");
    }
    step_bump_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(steps_done);
    return check_launch("step_bump_kernel");
}

int som_convert_f16_f32(const void* in, int64_t n, float* out, void* stream) {
    return convert_16_f32<__half>("convert_f16_f32", in, n, out, stream);
}

int som_convert_bf16_f32(const void* in, int64_t n, float* out, void* stream) {
    return convert_16_f32<__nv_bfloat16>("convert_bf16_f32", in, n, out, stream);
}


int som_prepare_codebook_f32(const float* W, int K, int D, float* c_norm2, void* stream) {
    return prepare_codebook(W, K, D, c_norm2, stream);
}

int som_prepare_codebook_w16(const void* W, int w_dtype, int K, int D, float* c_norm2, void* stream) {
    SOM_REQUIRE(w_dtype == ELEM_F16 || w_dtype == ELEM_BF16, SOM_E_BADARG, "prepare_codebook: w_dtype=%d", w_dtype);
    SOM_REQUIRE(((uintptr_t)W & 1) == 0, SOM_E_BADARG, "prepare_codebook: W is not 2-byte aligned");
    if (w_dtype == ELEM_F16) return prepare_codebook((const __half*)W, K, D, c_norm2, stream);
    return prepare_codebook((const __nv_bfloat16*)W, K, D, c_norm2, stream);
}

int som_quantize_nchw_f32(const int64_t* idx, const float* table, int K, int64_t n_img, int C, int H, int Wd, int pH,
                          int pW, float* out, void* stream) {
    return quantize_nchw(idx, table, K, n_img, C, H, Wd, pH, pW, out, stream);
}

int som_quantize_nchw_b16(const int64_t* idx, const void* table, int K, int64_t n_img, int C, int H, int Wd, int pH,
                          int pW, void* out, void* stream) {
    SOM_REQUIRE((((uintptr_t)table | (uintptr_t)out) & 1) == 0, SOM_E_BADARG, "quantize: 16-bit buffer misaligned");
    return quantize_nchw(idx, (const uint16_t*)table, K, n_img, C, H, Wd, pH, pW, (uint16_t*)out, stream);
}

int som_gather_rows_f32(const float* W, int D, const int64_t* keep, int64_t n_keep, float* out, void* stream) {
    return gather_rows(W, D, keep, n_keep, out, stream);
}

int som_gather_rows_b16(const void* W, int D, const int64_t* keep, int64_t n_keep, void* out, void* stream) {
    SOM_REQUIRE((((uintptr_t)W | (uintptr_t)out) & 1) == 0, SOM_E_BADARG, "gather_rows: 16-bit buffer misaligned");
    return gather_rows((const uint16_t*)W, D, keep, n_keep, (uint16_t*)out, stream);
}

}  // extern "C"
