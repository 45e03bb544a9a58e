// One-kernel SOM training step for small problems (BASELINE config 1: batch 8 -> 512 patches, K = 1024, D = 64).
//
// The whole iteration of /root/reference/train_codebook.py:225-249 -- forward with the Gaussian neighbourhood
// (models/Codebook.py:102-135), mse_loss, backward, Adam -- in the factorised form of SURVEY.md A.3, as ONE cooperative
// kernel with two grid-wide barriers instead of ~13 launches: at this size a launch (~4 us even from a CUDA graph) costs
// more than any of the kernels.  One CTA per SM; CTA b owns the contiguous unit rows [b R, (b+1) R):
//
//   phase 0  W~ rows of the own units = sum_t w(t) W[a+t]            (band filter, input rows streamed once per CTA)
//   (no barrier: the search reads W, not W~)
//   phase 1  BMU of the own patches (n / CTAs each) against ALL units (fp32 FFMA, unit tiles staged in shared memory,
//            score x.c - ||c||^2 / 2, lowest index on ties)
//   ---- grid barrier ----
//   phase 2  Rbar rows of the own units = sum over the patches that hit them, ascending patch order, of (W~[a] - x_p);
//            squared-error partial per CTA
//   ---- grid barrier ----
//   phase 3  G rows = (2 / numel) sum_t w(t) Rbar[a+t], Adam on the own rows of W; CTA 0 adds the squared-error
//            partials in CTA order (fp64), writes the loss and advances the step count
//
// Deterministic (fixed summation orders, no atomics).  Filter weights and Adam follow som_step_rules.cuh.  Everything
// stays in L2: the working set is K*D*4*5 bytes.
#include "som_common.cuh"
#include "som_step_rules.cuh"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace som {
namespace sstep {

constexpr int THREADS = 256;
constexpr int RMAX = 32;            // unit rows per CTA
constexpr int CU = 64;              // units per chunk in the BMU phase
constexpr int PB = 64;              // patches per block in the BMU phase
constexpr int HMAX = 2048;          // band half-width the weight table holds
constexpr int NMAX = 2048;          // patches per step
constexpr int UNION_FLOATS = 32768; // 128 KB shared region reused by the phases

struct Params {
    const float* x;
    Geom g;
    float* W; float* m; float* v;
    float* Wt; float* Rbar;         // workspace, K x D each
    float* cand_val; int* cand_idx; // workspace, UC x n x 2 each (best and runner-up of every chunk)
    double* sse_part;               // workspace, one per CTA
    int64_t* bmu_out;               // n_patches (may be null)
    double* loss_out;
    int64_t* steps_done;
    int K, h, R, UC, PG, PPG;
    float two_var, gscale;
    double inv_numel;
    double lr, b1, b2;
    float eps;
};

__device__ unsigned long long g_prof_small[8];          // CTA 0: globaltimer at the phase boundaries of the last launch
__device__ __forceinline__ void stamp(int i) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long v;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v)::"memory");
        g_prof_small[i] = v;
    }
}

// Rows [a0, a1) of T @ in for the features of this thread.  The CTA first stages the input rows it needs,
// [a0 - h, a1 + h), in shared memory (zero outside [0, K)); thread (d, g) then owns the RB consecutive output rows
// r0 = g * RB .. and walks the staged rows once, ascending, with the Gaussian weights in a register window that slides
// by one row per step: one input read + one table read per RB FMAs.  out[i] = row r0 + i (valid for r0 + i < R).
template <int D, int RBCAP>
__device__ __forceinline__ void band_rows(const float* __restrict__ in, int K, int h, const float* wtab, int a0, int a1,
                                          float* s_in, int RB, float (&out)[RBCAP]) {
    const int d = threadIdx.x % D, g = threadIdx.x / D;
    const int R = a1 - a0;
    const int rows_in = R + 2 * h;
    __syncthreads();                                     // the shared region may still be in use by the previous phase
    // (plain loads: `in` may have been written by other CTAs earlier in this launch; eight in flight per thread)
    for (int i0 = threadIdx.x; i0 < rows_in * (D / 4); i0 += 8 * THREADS) {
        float4 val[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * THREADS;
            const int jl = i / (D / 4), c = i - jl * (D / 4);
            const int j = a0 - h + jl;
            val[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < rows_in * (D / 4) && j >= 0 && j < K)
                val[u] = *(reinterpret_cast<const float4*>(in + (int64_t)j * D) + c);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * THREADS;
            if (i < rows_in * (D / 4)) reinterpret_cast<float4*>(s_in)[i] = val[u];
        }
    }
    __syncthreads();
    const int r0 = g * RB;
    float acc[RBCAP], wreg[RBCAP];
#pragma unroll
    for (int i = 0; i < RBCAP; ++i) { acc[i] = 0.f; wreg[i] = 0.f; }
    if (r0 < R) {
        // staged row jl contributes to output row r0 + i with weight w(|jl - (r0 + i) - h|)
        const int jl_end = min(rows_in, r0 + RB + 2 * h);
#pragma unroll 8
        for (int jl = r0; jl < jl_end; ++jl) {
#pragma unroll
            for (int i = RBCAP - 1; i > 0; --i) wreg[i] = wreg[i - 1];
            const int t = jl - r0 - h;
            const int at = t < 0 ? -t : t;
            wreg[0] = at <= h ? wtab[at] : 0.f;
            const float val = s_in[jl * D + d];
#pragma unroll
            for (int i = 0; i < RBCAP; ++i) acc[i] = fmaf(wreg[i], val, acc[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < RBCAP; ++i) out[i] = acc[i];
}

template <int D, int RBCAP>
__global__ void __launch_bounds__(THREADS, 1) step_small_kernel(const Params P) {
    constexpr int NQ = THREADS / D;
    constexpr int DC = D < 64 ? D : 64;                 // features per register chunk in the BMU phase
    cg::grid_group grid = cg::this_grid();
    extern __shared__ float smem[];
    float* wtab = smem;                                 // HMAX + 1 (+ pad to 16 bytes)
    float* uni = smem + HMAX + 4;                       // UNION_FLOATS, reused by the phases
    __shared__ int n_list;
    __shared__ double sse_w[THREADS / 32];
    __shared__ int foff[D];                              // feature offsets inside a patch (patchify as address arithmetic)

    const int K = P.K, h = P.h;
    const int d = threadIdx.x % D, g = threadIdx.x / D;
    const int64_t n = P.g.n_patches;
    const double t_step = (double)(P.steps_done[0] + 1);           // read before any barrier: CTA 0 bumps it at the end
    for (int t = threadIdx.x; t <= h; t += THREADS) wtab[t] = band_weight(t, h, P.two_var);
    for (int t = threadIdx.x; t < D; t += THREADS) foff[t] = feat_off(P.g, t);
    const int a0 = min(K, (int)blockIdx.x * P.R), a1 = min(K, a0 + P.R);
    const int R = a1 - a0;
    const int RB = (P.R + NQ - 1) / NQ;
    __shared__ AdamScalars adam_s;
    if (threadIdx.x == 0) adam_s = adam_scalars(P.lr, P.b1, P.b2, P.eps, t_step);     // once per CTA
    stamp(0);

    // ---- phase 0: W~ rows of the own units --------------------------------------------------------------------------
    float rows[RBCAP];
    if (R > 0) {
        band_rows<D, RBCAP>(P.W, K, h, wtab, a0, a1, uni, RB, rows);
#pragma unroll
        for (int i = 0; i < RBCAP; ++i)
            if (i < RB && g * RB + i < R) P.Wt[(int64_t)(a0 + g * RB + i) * D + d] = rows[i];
    }
    stamp(1);
    // (no grid barrier here: the search below reads W and x only; W~ is first needed in phase 2)
    stamp(2);

    // ---- phase 1: scores of (a block of patches) x (a chunk of 64 units): candidates per (chunk, patch) --------------
    {
        const int uc = (int)blockIdx.x % P.UC, pg = (int)blockIdx.x / P.UC;
        if (pg < P.PG) {
            float* xs = uni;                                // PB x D
            float* sc = uni + PB * D;                       // PB x (CU + 1)
            const int u = threadIdx.x % CU, q4 = threadIdx.x / CU;
            constexpr int NG = THREADS / CU;                // 4 patch groups
            const int unit = uc * CU + u;
            const bool unit_ok = unit < K;
            const int64_t pg0 = (int64_t)pg * P.PPG;
            const int64_t pg1 = min(n, pg0 + P.PPG);
            for (int64_t pb = pg0; pb < pg1; pb += PB) {
                const int np = (int)min((int64_t)PB, pg1 - pb);
                __syncthreads();
                {   // one warp per patch row (one base-address computation per patch, not per element)
                    const int wid = threadIdx.x >> 5, ln = threadIdx.x & 31;
                    for (int pp0 = wid; pp0 < np; pp0 += 4 * (THREADS / 32)) {
                        float val[4][(D + 31) / 32];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int pp = pp0 + u * (THREADS / 32);
                            const float* src = P.x + patch_base(P.g, pb + (pp < np ? pp : 0));
#pragma unroll
                            for (int e = 0; e < (D + 31) / 32; ++e)
                                val[u][e] = (pp < np && ln + 32 * e < D) ? __ldg(src + foff[ln + 32 * e]) : 0.f;
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int pp = pp0 + u * (THREADS / 32);
#pragma unroll
                            for (int e = 0; e < (D + 31) / 32; ++e)
                                if (pp < np && ln + 32 * e < D) xs[pp * D + ln + 32 * e] = val[u][e];
                        }
                    }
                }
                __syncthreads();
                // scores accumulate in shared memory (own element): the patch loop stays a LOOP -- this code runs once
                // per launch, and fully unrolled it is bound by cold instruction fetches, not by arithmetic
                float nrm = 0.f;
                for (int dc = 0; dc < D; dc += DC) {
                    float wr[DC];
#pragma unroll
                    for (int c = 0; c < DC; c += 4) {
                        float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (unit_ok) w4 = __ldg(reinterpret_cast<const float4*>(P.W + (int64_t)unit * D + dc + c));
                        wr[c] = w4.x; wr[c + 1] = w4.y; wr[c + 2] = w4.z; wr[c + 3] = w4.w;
                    }
#pragma unroll
                    for (int c = 0; c < DC; ++c) nrm = fmaf(wr[c], wr[c], nrm);
#pragma unroll 1
                    for (int pp = q4; pp < np; pp += NG) {
                        const float4* xr = reinterpret_cast<const float4*>(xs + pp * D + dc);
                        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
                        for (int c = 0; c < DC / 4; ++c) {
                            const float4 xv = xr[c];
                            s0 = fmaf(xv.x, wr[4 * c], s0);
                            s1 = fmaf(xv.y, wr[4 * c + 1], s1);
                            s2 = fmaf(xv.z, wr[4 * c + 2], s2);
                            s3 = fmaf(xv.w, wr[4 * c + 3], s3);
                        }
                        const float sdot = (s0 + s1) + (s2 + s3);
                        float* dst = sc + pp * (CU + 1) + u;
                        *dst = (dc == 0) ? sdot : *dst + sdot;
                    }
                }
#pragma unroll 1
                for (int pp = q4; pp < np; pp += NG) {
                    float* dst = sc + pp * (CU + 1) + u;
                    *dst = unit_ok ? *dst - 0.5f * nrm : -INFINITY;
                }
                __syncthreads();
                if ((int)threadIdx.x < np) {                // first maximum and runner-up over the chunk's units, ascending
                    const float* row = sc + threadIdx.x * (CU + 1);
                    float bv = -INFINITY, sv = -INFINITY;
                    int bi = 0, si = 0;
                    for (int k0 = 0; k0 < CU; k0 += 16) {
                        float vv[16];
#pragma unroll
                        for (int k = 0; k < 16; ++k) vv[k] = row[k0 + k];
#pragma unroll
                        for (int k = 0; k < 16; ++k) {
                            const float v = vv[k];
                            if (v > bv) { sv = bv; si = bi; bv = v; bi = k0 + k; }
                            else if (v > sv) { sv = v; si = k0 + k; }
                        }
                    }
                    const int64_t o = ((int64_t)uc * n + pb + threadIdx.x) * 2;
                    P.cand_val[o] = bv; P.cand_idx[o] = uc * CU + bi;
                    P.cand_val[o + 1] = sv; P.cand_idx[o + 1] = uc * CU + si;
                }
            }
        }
    }
    stamp(3);
    grid.sync();
    stamp(4);

    // ---- phase 2: merge the candidates (every CTA, all patches), Rbar rows of the own units, squared error -----------
    float sse = 0.f;
    {
        int* bmu_s = reinterpret_cast<int*>(uni);           // NMAX
        int* list = bmu_s + NMAX;                           // 2 * NMAX (patch, row)
        __syncthreads();
        for (int64_t p = threadIdx.x; p < n; p += THREADS) {
            float bv = -INFINITY, sv2 = -INFINITY;          // best score and the second-best over ALL candidates
            int bc = 0;
            for (int c0 = 0; c0 < P.UC; c0 += 8) {          // ascending chunks, strict '>': the lowest index wins ties
                float2 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    v[u] = (c0 + u < P.UC) ? *reinterpret_cast<const float2*>(P.cand_val + ((int64_t)(c0 + u) * n + p) * 2)
                                           : make_float2(-INFINITY, -INFINITY);
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    if (v[u].x > bv) { sv2 = fmaxf(bv, v[u].y); bv = v[u].x; bc = c0 + u; }
                    else sv2 = fmaxf(sv2, v[u].x);
                }
            }
            int bi = bv > -INFINITY ? P.cand_idx[((int64_t)bc * n + p) * 2] : 0;   // a NaN row keeps unit 0, as torch.argmin does
            // Near-ties: the fp32 scores of two units can agree to the last bit while their true distances differ
            // (and the Gaussian-filtered rows of two such units differ a lot, so the pick matters for the loss).
            // Every candidate (best and runner-up of each chunk) within 2e-6 of the best score is re-scored in fp64;
            // the larger fp64 score wins, the lower index on an exact tie.  Rare, and identical in every CTA.
            const float band = 2e-6f * fmaxf(1.0f, fabsf(bv));
            if (sv2 >= bv - band && bv > -INFINITY) {
                double best64 = -INFINITY;
                int best_u = bi;
                const float* xp = P.x + patch_base(P.g, p);
                for (int c = 0; c < 2 * P.UC; ++c) {
                    const int64_t o = (int64_t)(c >> 1) * n * 2 + p * 2 + (c & 1);
                    if (P.cand_val[o] >= bv - band) {
                        const int u = P.cand_idx[o];
                        const float* wu = P.W + (int64_t)u * D;
                        double dot = 0.0, nn = 0.0;
                        for (int dd = 0; dd < D; ++dd) {
                            const double wv = (double)wu[dd];
                            dot = fma((double)__ldg(xp + feat_off(P.g, dd)), wv, dot);
                            nn = fma(wv, wv, nn);
                        }
                        const double s64 = dot - 0.5 * nn;
                        if (s64 > best64 || (s64 == best64 && u < best_u)) { best64 = s64; best_u = u; }
                    }
                }
                bi = best_u;
            }
            bmu_s[p] = bi;
            if (P.bmu_out != nullptr && (p % gridDim.x) == blockIdx.x) P.bmu_out[p] = (int64_t)bi;
        }
        __syncthreads();
        if (R > 0) {
            if (threadIdx.x < 32) {           // warp 0 lists the patches that hit the own rows, ascending
                int tot = 0;
                for (int64_t pb = 0; pb < n; pb += 32) {
                    const int64_t p = pb + threadIdx.x;
                    const int b = (p < n) ? bmu_s[p] : -1;
                    const bool hit = b >= a0 && b < a1;
                    const unsigned mask = __ballot_sync(0xffffffffu, hit);
                    if (hit) {
                        const int pos = tot + __popc(mask & ((1u << threadIdx.x) - 1u));
                        list[2 * pos] = (int)p;
                        list[2 * pos + 1] = b - a0;
                    }
                    tot += __popc(mask);
                }
                if (threadIdx.x == 0) n_list = tot;
            }
            __syncthreads();
            const int nl = n_list;
            const int doff = foff[d];
            for (int r = g; r < R; r += NQ) {
                const float wt = P.Wt[(int64_t)(a0 + r) * D + d];
                float acc = 0.f;
                for (int e0 = 0; e0 < nl; e0 += 8) {        // eight loads in flight, added in list (= patch) order
                    float xv[8];
                    bool on[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        on[u] = e0 + u < nl && list[2 * (e0 + u) + 1] == r;
                        xv[u] = on[u] ? __ldg(P.x + patch_base(P.g, (int64_t)list[2 * (e0 + u)]) + doff) : 0.f;
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (on[u]) {
                            const float res = wt - xv[u];
                            acc += res;
                            sse = fmaf(res, res, sse);
                        }
                    }
                }
                P.Rbar[(int64_t)(a0 + r) * D + d] = acc;
            }
        }
    }
    {
        const float t = warp_sum(sse);
        if ((threadIdx.x & 31) == 0) sse_w[threadIdx.x >> 5] = (double)t;
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot = 0.0;
            for (int w = 0; w < THREADS / 32; ++w) tot += sse_w[w];
            P.sse_part[blockIdx.x] = tot;
        }
    }
    stamp(5);
    grid.sync();
    stamp(6);

    // ---- phase 3: G rows, Adam on the own rows, loss -----------------------------------------------------------------
    if (R > 0) {
        band_rows<D, RBCAP>(P.Rbar, K, h, wtab, a0, a1, uni, RB, rows);
        const AdamScalars a = adam_s;
#pragma unroll
        for (int i = 0; i < RBCAP; ++i) {
            if (i < RB && g * RB + i < R) {
                const int64_t idx = (int64_t)(a0 + g * RB + i) * D + d;
                float mi = P.m[idx], vi = P.v[idx], wi = P.W[idx];
                adam_update(a, P.gscale * rows[i], mi, vi, wi);
                P.W[idx] = wi; P.m[idx] = mi; P.v[idx] = vi;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < 32) {            // fixed order: lane-strided partial sums, then a butterfly
        double tot = 0.0;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += 32) tot += P.sse_part[b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if (threadIdx.x == 0) {
            if (P.loss_out) *P.loss_out = tot * P.inv_numel;
            P.steps_done[0] += 1;
        }
    }
    stamp(7);
}

static size_t smem_bytes() { return sizeof(float) * ((size_t)HMAX + 4 + UNION_FLOATS) + 64; }

struct Plan { int grid, R, RB, UC, PG, PPG, h; float two_var; size_t off_wt, off_rbar, off_cv, off_ci, off_sse, total; };

static bool make_plan(Plan* pl, int64_t n, int D, int K, double range) {
    if (n <= 0 || n > NMAX || K <= 0 || !(range > 0.0)) return false;
    if (D != 16 && D != 32 && D != 64 && D != 128 && D != 256) return false;
    const int sms = sm_count();
    pl->R = (K + sms - 1) / sms;
    if (pl->R > RMAX) return false;
    pl->RB = (pl->R + THREADS / D - 1) / (THREADS / D);
    pl->two_var = filter_two_var(range);
    pl->h = filter_band_half_width(pl->two_var, K);
    if (pl->h > HMAX) return false;
    if ((int64_t)(pl->R + 2 * pl->h) * D > UNION_FLOATS) return false;         // staged filter rows
    if (PB * D + PB * (CU + 1) > UNION_FLOATS) return false;                   // BMU phase: patches + scores
    pl->UC = (K + CU - 1) / CU;
    const int g_units = (K + pl->R - 1) / pl->R;
    pl->grid = g_units > pl->UC ? g_units : pl->UC;
    if (pl->grid > sms) return false;
    if (pl->grid < sms && pl->grid < 2 * pl->UC) pl->grid = sms < 2 * pl->UC ? sms : 2 * pl->UC;   // room for patch groups
    pl->PG = pl->grid / pl->UC;
    pl->PPG = (int)((n + pl->PG - 1) / pl->PG);
    size_t o = 0;
    pl->off_wt = o; o = align_up(o + (size_t)K * D * 4, 256);
    pl->off_rbar = o; o = align_up(o + (size_t)K * D * 4, 256);
    pl->off_cv = o; o = align_up(o + (size_t)pl->UC * n * 2 * 4, 256);
    pl->off_ci = o; o = align_up(o + (size_t)pl->UC * n * 2 * 4, 256);
    pl->off_sse = o; o = align_up(o + (size_t)sms * 8, 256);
    pl->total = o;
    return true;
}

// the RBCAP slot of step_small_kernel<D, RBCAP> for RB output rows per thread: RBCAP = 2, 8 or 32
static int rb_slot(int RB) { return RB <= 2 ? 0 : (RB <= 8 ? 1 : 2); }

}  // namespace sstep
}  // namespace som

using namespace som;
using namespace som::sstep;

extern "C" size_t som_step_small_workspace_bytes(int64_t n_patches, int D, int K, double neighbourhood_range) {
    Plan pl;
    return make_plan(&pl, n_patches, D, K, neighbourhood_range) ? pl.total : 0;
}

extern "C" int som_step_small_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                  float* W, float* m, float* v, int K, double neighbourhood_range,
                                  double lr, double b1, double b2, double eps, int64_t* steps_done,
                                  int64_t* bmu_out, double* loss_out, void* ws, size_t ws_bytes, void* stream) {
    SOM_REQUIRE(x && W && m && v && steps_done, SOM_E_BADARG, "step_small: null pointer");
    Geom g;
    int rc = make_geom(&g, x, n_img, C, H, Wd, pH, pW);
    if (rc) return rc;
    Plan pl;
    SOM_REQUIRE(make_plan(&pl, g.n_patches, g.D, K, neighbourhood_range), SOM_E_UNSUPPORTED,
                "step_small: shape n=%lld D=%d K=%d range=%g is not covered (ask som_step_small_workspace_bytes)",
                (long long)g.n_patches, g.D, K, neighbourhood_range);
    SOM_REQUIRE(ws != nullptr && ws_bytes >= pl.total, SOM_E_WORKSPACE, "step_small: workspace %zu < required %zu",
                ws_bytes, pl.total);
    SOM_REQUIRE((((uintptr_t)ws & 255) | ((uintptr_t)W & 15)) == 0, SOM_E_BADARG,
                "step_small: workspace must be 256-byte aligned, the codebook 16-byte aligned");
    Params P;
    P.x = x; P.g = g; P.W = W; P.m = m; P.v = v;
    P.Wt = (float*)((char*)ws + pl.off_wt);
    P.Rbar = (float*)((char*)ws + pl.off_rbar);
    P.cand_val = (float*)((char*)ws + pl.off_cv);
    P.cand_idx = (int*)((char*)ws + pl.off_ci);
    P.sse_part = (double*)((char*)ws + pl.off_sse);
    P.bmu_out = bmu_out; P.loss_out = loss_out; P.steps_done = steps_done;
    P.K = K; P.h = pl.h; P.R = pl.R; P.UC = pl.UC; P.PG = pl.PG; P.PPG = pl.PPG; P.two_var = pl.two_var;
    P.gscale = (float)(2.0 / ((double)g.n_patches * (double)g.D));
    P.inv_numel = 1.0 / ((double)g.n_patches * (double)g.D);
    P.lr = lr; P.b1 = b1; P.b2 = b2; P.eps = (float)eps;

    typedef void (*KernelFn)(const Params);
    static const KernelFn fns[5][3] = {
        {step_small_kernel<16, 2>, step_small_kernel<16, 8>, step_small_kernel<16, 32>},
        {step_small_kernel<32, 2>, step_small_kernel<32, 8>, step_small_kernel<32, 32>},
        {step_small_kernel<64, 2>, step_small_kernel<64, 8>, step_small_kernel<64, 32>},
        {step_small_kernel<128, 2>, step_small_kernel<128, 8>, step_small_kernel<128, 32>},
        {step_small_kernel<256, 2>, step_small_kernel<256, 8>, step_small_kernel<256, 32>}};
    const int dslot = g.D == 16 ? 0 : g.D == 32 ? 1 : g.D == 64 ? 2 : g.D == 128 ? 3 : 4;
    const int rslot = rb_slot(pl.RB);
    KernelFn fn = fns[dslot][rslot];
    const size_t smem = smem_bytes();
    static PerDeviceFlag attr_done[15];
    rc = smem_opt_in(attr_done[3 * dslot + rslot], &fn, 1, (int)smem, "step_small");
    if (rc) return rc;
    void* args[] = {(void*)&P};
    cudaError_t le = cudaLaunchCooperativeKernel((const void*)fn, dim3((unsigned)pl.grid), dim3(THREADS), args, smem,
                                                 (cudaStream_t)stream);
    if (le != cudaSuccess) { set_error("step_small_kernel: launch: %s", cudaGetErrorString(le)); return (int)le; }
    return check_launch("step_small_kernel");
}

// debug: the plan of som_step_small_f32 for n patches of dimension D, K units and a range, as 8 int64 fields: grid, R,
// RB, the RBCAP slot (0, 1, 2: RBCAP = 2, 8, 32), UC, PG, PPG, h; all -1 where the one-kernel step does not cover the
// shape.  The first n_out are written.  Not in somcb.h: a test hook, not part of the ABI.
extern "C" SOM_API int som_debug_step_small_plan(int64_t n_patches, int D, int K, double neighbourhood_range,
                                                 int64_t* out, int n_out) {
    SOM_REQUIRE(out != nullptr && n_out >= 0, SOM_E_BADARG, "step_small plan: output");
    int64_t f[8] = {-1, -1, -1, -1, -1, -1, -1, -1};
    Plan pl;
    if (make_plan(&pl, n_patches, D, K, neighbourhood_range)) {
        const int64_t v[8] = {pl.grid, pl.R, pl.RB, rb_slot(pl.RB), pl.UC, pl.PG, pl.PPG, pl.h};
        for (int i = 0; i < 8; ++i) f[i] = v[i];
    }
    for (int i = 0; i < n_out && i < 8; ++i) out[i] = f[i];
    return SOM_OK;
}

// debug: CTA 0's globaltimer (ns) at the eight phase boundaries of the last launch
extern "C" SOM_API int som_debug_step_small_ns(unsigned long long* out8) {
    return (int)cudaMemcpyFromSymbol(out8, som::sstep::g_prof_small, 8 * sizeof(unsigned long long));
}
