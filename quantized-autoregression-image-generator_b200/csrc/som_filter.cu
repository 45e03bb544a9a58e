// K3: Gaussian neighbourhood filter along the unit axis.
//
//   out[a][d] = scale * sum_{t=-h..h} w(|t|) * in[a+t][d],   w(t) = expf(-( float(t*t) / two_var ))
//
// This is T @ in with T the K x K banded symmetric Toeplitz matrix that the reference builds
// densely, one row per patch, in models/Codebook.py:112-125 and multiplies in :128-130
// (forward, in = W) and in the matmul backward (in = Rbar).  Weights are generated exactly as
// the reference does (band_weight, som_step_rules.cuh).  The band half-width h is where expf
// underflows to exactly 0 (SURVEY 0.7).
//
// Mapping: lane <-> feature d (coalesced 128-byte rows), each warp owns TA consecutive units
// and slides a TA-wide window of weights held in registers over the rows j it needs, so each
// loaded value feeds TA FFMAs and each step needs one weight from the shared table.
// Bound: FFMA (2*K*D*band flop) -- in[] is K*D*4 bytes and stays L1/L2 resident.
#include "som_common.cuh"
#include "som_step_rules.cuh"

namespace som {
SOM_TRACE_TU(trace_set_filter)

constexpr int FILT_TA = 8;          // units per warp
constexpr int FILT_WARPS = 8;       // warps per CTA  -> 64 units x 32 features per CTA
constexpr int FILT_PAD = FILT_TA + 8;

// table layout: tab[t + off] for t in [-(h+PAD), h+PAD], zero outside [-h, h]
__global__ void __launch_bounds__(FILT_WARPS * 32)
filter_kernel(const float* __restrict__ in, float* __restrict__ out, int K, int D,
              float two_var, int h, float scale) {
    pdl_begin();
    trace_stamp(s_trace_buf, 4);
    extern __shared__ float tab[];
    const int off = h + FILT_PAD;
    const int tab_n = 2 * off + 1;
    for (int i = threadIdx.x; i < tab_n; i += blockDim.x) {
        const int t = i - off;
        tab[i] = band_weight(t < 0 ? -t : t, h, two_var);
    }
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int d = blockIdx.y * 32 + lane;
    const int a0 = (blockIdx.x * FILT_WARPS + warp) * FILT_TA;
    if (a0 >= K) return;
    const bool d_ok = d < D;

    float acc[FILT_TA];
#pragma unroll
    for (int i = 0; i < FILT_TA; ++i) acc[i] = 0.f;

    // rows needed by this warp: j in [a0 - h, a0 + TA - 1 + h], clipped to [0, K)
    int j_lo = a0 - h; if (j_lo < 0) j_lo = 0;
    int j_hi = a0 + FILT_TA - 1 + h; if (j_hi > K - 1) j_hi = K - 1;

    // window: win[i] = w(|j - (a0+i)|) = tab[(j - a0 - i) + off]
    const float* col = in + d;
    int j = j_lo;
    for (; j + FILT_TA <= j_hi + 1; j += FILT_TA) {
        float v[FILT_TA];
#pragma unroll
        for (int u = 0; u < FILT_TA; ++u)
            v[u] = d_ok ? __ldg(col + (int64_t)(j + u) * D) : 0.f;
        // weights needed in this group: t = (j+u) - (a0+i), u,i in [0,TA) -> t0-(TA-1) .. t0+(TA-1)
        const int t0 = j - a0 + off;
        float wv[2 * FILT_TA - 1];
#pragma unroll
        for (int q = 0; q < 2 * FILT_TA - 1; ++q) wv[q] = tab[t0 - (FILT_TA - 1) + q];
#pragma unroll
        for (int u = 0; u < FILT_TA; ++u)
#pragma unroll
            for (int i = 0; i < FILT_TA; ++i)
                acc[i] = fmaf(wv[u - i + FILT_TA - 1], v[u], acc[i]);
    }
    for (; j <= j_hi; ++j) {
        float v = d_ok ? __ldg(col + (int64_t)j * D) : 0.f;
        const int t0 = j - a0 + off;
#pragma unroll
        for (int i = 0; i < FILT_TA; ++i) acc[i] = fmaf(tab[t0 - i], v, acc[i]);
    }

    if (d_ok) {
#pragma unroll
        for (int i = 0; i < FILT_TA; ++i)
            if (a0 + i < K) out[(int64_t)(a0 + i) * D + d] = scale * acc[i];
    }
}

// Tiled variant (D % 4 == 0, D >= 48, 16-byte aligned rows).  The scalar kernel above waits a full L2 round trip
// per group of TA rows; here a CTA owns 32 units x TD features (TD = 128, or 64 for short rows), streams the
// input rows it needs through shared memory in coalesced, double-buffered (cp.async) 64-row chunks, and every
// thread keeps an 8-unit x 4-feature register tile (8 LDS.128 + 15 table reads per 256 FFMAs; a 4 x 4 tile is
// shared-memory-port bound).  There are only K*D/32 such tiles -- 1.7 warps per scheduler at C4 -- so the rows of
// every chunk are split over JS threads per tile (JS = 4 for TD = 64, 2 for TD = 128) and the JS partial sums are
// added in fixed order through shared memory at the end: deterministic, fp32 association differs from the scalar
// kernel by the split only.
constexpr int FT_JC = 64, FT_THREADS = 256, FT_U = 8;
constexpr int FT_PAD = 128 + FT_JC + 8;          // covers the unit tile + one chunk of overshoot

template <int TD, int JS>
__global__ void __launch_bounds__(FT_THREADS)
filter_tile_kernel(const float* __restrict__ in, float* __restrict__ out, int K, int D,
                   float two_var, int h, float scale) {
    pdl_begin();
    trace_stamp(s_trace_buf, 4);
    constexpr int FG = TD / 4;                     // feature groups (threads) per row
    constexpr int UG = FT_THREADS / (FG * JS);     // unit groups per CTA
    constexpr int FT_TK = UG * FT_U;               // units per CTA (32)
    constexpr int CHUNK4 = FT_JC * FG;             // float4 per chunk buffer
    constexpr int ROWS = FT_JC / JS;               // rows of a chunk per split
    static_assert(ROWS % FT_U == 0 && (JS - 1) * UG * FG * FT_U <= 2 * CHUNK4, "tile shape");
    extern __shared__ float fsm[];
    const int off = h + FT_PAD;
    const int tab_n = 2 * off + 1;
    float* tab = fsm;
    float4* chunk = reinterpret_cast<float4*>(fsm + ((tab_n + 3) & ~3));         // [2][FT_JC][FG]
    for (int i = threadIdx.x; i < tab_n; i += FT_THREADS) {
        const int t = i - off;
        tab[i] = band_weight(t < 0 ? -t : t, h, two_var);
    }
    const int a_tile = blockIdx.x * FT_TK;
    const int d_tile = blockIdx.y * TD;
    const int js = threadIdx.x / (UG * FG);
    const int tile = threadIdx.x % (UG * FG);
    const int ug = tile / FG, fg = tile % FG;
    const int a0 = a_tile + FT_U * ug;
    int j_lo = a_tile - h; if (j_lo < 0) j_lo = 0;
    int j_hi = a_tile + FT_TK - 1 + h; if (j_hi > K - 1) j_hi = K - 1;

    float4 acc[FT_U];
#pragma unroll
    for (int i = 0; i < FT_U; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);

    // chunks are double-buffered: cp.async brings chunk c + 1 in while chunk c is being multiplied
    auto issue = [&](int jc, int buf) {
#pragma unroll
        for (int i = 0; i < CHUNK4 / FT_THREADS; ++i) {
            const int idx = threadIdx.x + FT_THREADS * i;
            const int r = idx / FG, c4 = idx % FG;
            const int j = jc + r, d = d_tile + 4 * c4;
            float4* dst = chunk + buf * CHUNK4 + idx;
            if (j <= j_hi && d < D) {
                const uint32_t sa = (uint32_t)__cvta_generic_to_shared(dst);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(in + (int64_t)j * D + d) : "memory");
            } else {
                *dst = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue(j_lo, 0);
    int it = 0;
    for (int jc = j_lo; jc <= j_hi; jc += FT_JC, ++it) {
        const int buf = it & 1;
        const bool more = jc + FT_JC <= j_hi;
        if (more) issue(jc + FT_JC, buf ^ 1);              // the other buffer was released by the sync below
        if (more) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                    // table + chunk `buf` visible to every thread
        const float4* cur = chunk + buf * CHUNK4;
#pragma unroll
        for (int rr = 0; rr < ROWS; rr += FT_U) {
            const int r = js * ROWS + rr;
            const int t0 = (jc + r) - a0 + off;             // weight index of (row jc + r, unit a0)
            float wv[2 * FT_U - 1];
#pragma unroll
            for (int q = 0; q < 2 * FT_U - 1; ++q) wv[q] = tab[t0 - (FT_U - 1) + q];
#pragma unroll
            for (int u = 0; u < FT_U; ++u) {
                const float4 v = cur[(r + u) * FG + fg];
#pragma unroll
                for (int i = 0; i < FT_U; ++i) {
                    const float w = wv[u - i + FT_U - 1];   // w(|(jc + r + u) - (a0 + i)|)
                    acc[i].x = fmaf(w, v.x, acc[i].x);
                    acc[i].y = fmaf(w, v.y, acc[i].y);
                    acc[i].z = fmaf(w, v.z, acc[i].z);
                    acc[i].w = fmaf(w, v.w, acc[i].w);
                }
            }
        }
        __syncthreads();                                    // chunk `buf` consumed before it is refilled
    }
    // fixed-order sum of the JS row-split partials (the chunk buffers are free now)
    float4* red = chunk;
    if (js > 0) {
#pragma unroll
        for (int i = 0; i < FT_U; ++i) red[((js - 1) * UG * FG + tile) * FT_U + i] = acc[i];
    }
    __syncthreads();
    const int d = d_tile + 4 * fg;
    if (js == 0 && d < D) {
#pragma unroll
        for (int i = 0; i < FT_U; ++i) {
            float4 t = acc[i];
#pragma unroll
            for (int q = 1; q < JS; ++q) {
                const float4 p = red[((q - 1) * UG * FG + tile) * FT_U + i];
                t.x += p.x; t.y += p.y; t.z += p.z; t.w += p.w;
            }
            if (a0 + i < K)
                *reinterpret_cast<float4*>(out + (int64_t)(a0 + i) * D + d) =
                    make_float4(scale * t.x, scale * t.y, scale * t.z, scale * t.w);
        }
    }
}

// som_filter_tc.cu
bool filter_tc_applicable(int K, int D, int h);
size_t filter_tc_workspace_bytes(int K, int D, int h);
void filter_tc_plan_fields(int K, int D, int h, int64_t* f);
int launch_filter_tc(const float* in, float* out, int K, int D, float two_var, int h, float scale, void* ws,
                     size_t ws_bytes, cudaStream_t st);

// The kernel som_filter_f32 runs (FilterPlanField::FPF_KERNEL) and its dynamic shared memory.  The tile kernels take
// D % 4 == 0, D >= 48 and 16-byte aligned `in` and `out` while their table and chunk ring fit in 200 KB; the scalar kernel
// takes every other shape while its table fits (h <= 25 583), also the tile kernels' shapes with a wider band than
// theirs.  False where no kernel fits.
static bool filter_ffma_route(int D, int h, bool aligned16, int* kernel, size_t* smem) {
    if ((D & 3) == 0 && D >= 48 && aligned16) {
        const int td = D >= 128 ? 128 : 64;
        const size_t tab_n = (size_t)(2 * (h + FT_PAD) + 1);
        *smem = ((tab_n + 3) & ~(size_t)3) * sizeof(float) + 2 * (size_t)FT_JC * td * sizeof(float);
        *kernel = td == 128 ? FK_TILE128 : FK_TILE64;
        if (*smem <= 200 * 1024) return true;
    }
    *smem = (size_t)(2 * (h + FILT_PAD) + 1) * sizeof(float);
    *kernel = FK_SCALAR;
    return *smem <= 200 * 1024;
}

}  // namespace som

using namespace som;

extern "C" int som_filter_half_width(int K, double neighbourhood_range) {
    if (K <= 0 || !(neighbourhood_range > 0.0)) return 0;
    return filter_band_half_width(filter_two_var(neighbourhood_range), K);
}

extern "C" size_t som_filter_workspace_bytes(int K, int D, double neighbourhood_range) {
    if (K <= 0 || D <= 0 || !(neighbourhood_range > 0.0)) return 0;
    const float two_var = filter_two_var(neighbourhood_range);
    const int h = filter_band_half_width(two_var, K);
    return filter_tc_applicable(K, D, h) ? filter_tc_workspace_bytes(K, D, h) : 0;
}

extern "C" int som_filter_ws_f32(const float* in, float* out, int K, int D, double neighbourhood_range, float scale,
                                 void* ws, size_t ws_bytes, void* stream) {
    SOM_REQUIRE(in && out, SOM_E_BADARG, "filter: null pointer");
    SOM_REQUIRE(in != out, SOM_E_BADARG, "filter: in-place operation is not supported");
    SOM_REQUIRE(K > 0 && D > 0, SOM_E_BADARG, "filter: K=%d D=%d", K, D);
    SOM_REQUIRE(neighbourhood_range > 0.0, SOM_E_BADARG, "filter: neighbourhood_range=%g", neighbourhood_range);
    const float two_var = filter_two_var(neighbourhood_range);
    const int h = filter_band_half_width(two_var, K);
    // static rule on the shape: tensor cores for K >= 256 units and rows of >= 48 features (som_filter_tc.cu)
    if (filter_tc_applicable(K, D, h) && ws != nullptr)
        return launch_filter_tc(in, out, K, D, two_var, h, scale, ws, ws_bytes, (cudaStream_t)stream);
    return som_filter_f32(in, out, K, D, neighbourhood_range, scale, stream);
}

extern "C" int som_filter_f32(const float* in, float* out, int K, int D,
                              double neighbourhood_range, float scale, void* stream) {
    SOM_REQUIRE(in && out, SOM_E_BADARG, "filter: null pointer");
    SOM_REQUIRE(in != out, SOM_E_BADARG, "filter: in-place operation is not supported");
    SOM_REQUIRE(K > 0 && D > 0, SOM_E_BADARG, "filter: K=%d D=%d", K, D);
    SOM_REQUIRE(neighbourhood_range > 0.0, SOM_E_BADARG, "filter: neighbourhood_range=%g",
                neighbourhood_range);
    const float two_var = filter_two_var(neighbourhood_range);
    const int h = filter_band_half_width(two_var, K);
    int kern;
    size_t smem;
    SOM_REQUIRE(filter_ffma_route(D, h, (((uintptr_t)in | (uintptr_t)out) & 15) == 0, &kern, &smem), SOM_E_SHAPE,
                "filter: band half-width %d too large", h);
    typedef void (*FilterFn)(const float*, float*, int, int, float, int, float);
    if (kern != FK_SCALAR) {
        const int td = kern == FK_TILE128 ? 128 : 64;
        static const FilterFn tile_kernels[2] = {filter_tile_kernel<128, 2>, filter_tile_kernel<64, 4>};
        static PerDeviceFlag attr_done;
        const int rc = smem_opt_in(attr_done, tile_kernels, 2, 200 * 1024, "filter");
        if (rc) return rc;
        dim3 gt((unsigned)ceil_div64(K, 32), (unsigned)ceil_div64(D, td));      // 32 units per CTA in both shapes
        launch_pdl(tile_kernels[td == 64], gt, FT_THREADS, smem, (cudaStream_t)stream, in, out, K, D, two_var, h, scale);
        return check_launch("filter_tile_kernel");
    }
    if (smem > 48 * 1024) {
        static PerDeviceFlag attr_done;
        const FilterFn kernel = filter_kernel;
        const int rc = smem_opt_in(attr_done, &kernel, 1, 200 * 1024, "filter");
        if (rc) return rc;
    }
    dim3 grid((unsigned)ceil_div64(K, FILT_WARPS * FILT_TA), (unsigned)ceil_div64(D, 32));
    launch_pdl(filter_kernel, grid, FILT_WARPS * 32, smem, (cudaStream_t)stream, in, out, K, D, two_var, h, scale);
    return check_launch("filter_kernel");
}

// debug: the plan of a filter call, as FPF_COUNT int64 fields (som_common.cuh: FilterPlanField, -1 where a field does
// not apply); the first n_out are written.  with_ws: som_filter_ws_f32 with a workspace (else som_filter_f32, or
// som_filter_ws_f32 without one); aligned16: `in` and `out` are both 16-byte aligned.  The answers come from the rules the
// launchers use.  Not in somcb.h: a test hook, not part of the ABI.
extern "C" SOM_API int som_debug_filter_plan(int K, int D, double neighbourhood_range, int with_ws, int aligned16,
                                             int64_t* out, int n_out) {
    SOM_REQUIRE(K > 0 && D > 0 && neighbourhood_range > 0.0, SOM_E_BADARG, "filter plan: K=%d D=%d range=%g", K, D,
                neighbourhood_range);
    SOM_REQUIRE(out != nullptr && n_out >= 0, SOM_E_BADARG, "filter plan: output");
    int64_t f[FPF_COUNT];
    for (int i = 0; i < FPF_COUNT; ++i) f[i] = -1;
    const int h = filter_band_half_width(filter_two_var(neighbourhood_range), K);
    if (with_ws && filter_tc_applicable(K, D, h)) {
        filter_tc_plan_fields(K, D, h, f);
    } else {
        int kern;
        size_t smem;
        SOM_REQUIRE(filter_ffma_route(D, h, aligned16 != 0, &kern, &smem), SOM_E_SHAPE,
                    "filter: band half-width %d too large", h);
        f[FPF_KERNEL] = kern;
        f[FPF_SMEM] = (int64_t)smem;
    }
    f[FPF_H] = h;
    for (int i = 0; i < n_out && i < FPF_COUNT; ++i) out[i] = f[i];
    return SOM_OK;
}
