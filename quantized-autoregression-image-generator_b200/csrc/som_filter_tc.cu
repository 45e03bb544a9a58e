// K3 (tensor-core variant): neighbourhood filter  out = scale * T @ in  as a banded-Toeplitz GEMM on tcgen05.
// sm_100a only.
//
//   out[a][d] = scale * sum_{t=-h..h} w(|t|) * in[a+t][d],   w(t) = expf(-( float(t*t) / two_var ))
//
// T is the K x K Gaussian neighbourhood matrix the reference builds row by row (models/Codebook.py:112-125) and
// multiplies densely (`:128-130` forward, autograd backward); h is where expf underflows to exactly 0 (SURVEY 0.7).
// For a tile of 128 units [a0, a0+128) the product is a dense GEMM  M = 128 units, N = features,
// inner = the 128 + 2h input rows [a0-h, a0+127+h]:  A[ul][jl] = w(jl - h - ul) is the SAME Toeplitz strip for every
// tile, B[d][jl] = in[a0-h+jl][d].  fp32-faithful 3xTF32 (hi.hi + lo.hi + hi.lo, fp32 accumulation in TMEM), like the
// BMU kernels.  The FFMA kernel (som_filter.cu) reaches 26-29 TFLOP/s of 2*K*D*band useful flop (C4 96 us, C3 36-43 us).
//
//   pre-pass  split_in_t_kernel : in (K x D) -> transposed, zero-padded, hi | lo split operand  Bt[d][h + j]
//                                 (K-major for the MMA: the reduction index must be the contiguous one)
//   main      filter_tc_kernel  : one CTA per (unit tile, feature tile of TNF), 320 threads, warp-specialised:
//     warp 0     TMA producer: B_hi / B_lo blocks (TNF x 32 floats each) of k-block kb into a 3-stage ring
//     warp 1     MMA issuer  : 4 k-steps x 3 products of M128 x N(TNF) x K8 kind::tf32 per k-block
//     warps 2-9  builders    : write the Toeplitz A_hi / A_lo block of k-block kb (128 x 32, SWIZZLE_128B rows) from
//                              a shared weight table -- the strip never travels through L2 (every CTA would read the
//                              same bytes at the same time: measured 14.5 B/clk/SM for such hot tiles);
//                              afterwards warps 2-5 are the epilogue: tcgen05.ld of their TMEM lane quarter,
//                              scale, 128-byte row stores.
// Bound: tensor pipe / shared-memory operand bandwidth (A 4 KB + B TNF*32 B per MMA).
// Algorithmic work: 2*K*D*(2h+1) flop; executed: 3 * 2*128*TNF*L per tile with L = 32*ceil((128+2h)/32).
#include "som_common.cuh"
#include "som_peer.cuh"
#include "som_step_rules.cuh"
#include "som_tc_ptx.cuh"
#include "som_tc_split.cuh"

namespace som {
SOM_TRACE_TU(trace_set_filter_tc)
namespace ftc {
using namespace tc;

constexpr int TMU = 128;                     // units per tile (UMMA M)
constexpr int CK = 5;                        // k-blocks that share one Toeplitz strip of the A operand
constexpr int STRIP_ROWS = TMU + KBLK * (CK - 1);        // 256: one builder thread per row
constexpr int STRIP_BYTES = STRIP_ROWS * KBLK * 4;       // 32 KB (hi or lo)
template <int TNF> constexpr int nstage_b() { return TNF == 128 ? 2 : 4; }      // B ring: 64 KB either way
constexpr int NACC = 4;                      // TMEM accumulators, k-block kb goes to kb % NACC (see the MMA loop)
constexpr int BUILD_WARPS = 8;                // two threads per unit row, 16 inner positions each
constexpr int NUM_THREADS = (2 + BUILD_WARPS) * 32;      // 320
constexpr int TAB_PAD = 160;                 // |jl - h - ul| <= h + 158
constexpr int MAX_H = 1400;                  // table of 2 * (2h + 2*TAB_PAD + 1) floats <= 25 KB

struct Params {
    int K, D, h, nkb;
    float two_var, scale;
    float* out;
    int q, na;              // accumulation chains: chain a = k-blocks [a q, (a + 1) q), na <= NACC of them
    int ks;                 // k-split: CTA blockIdx.z runs chain z; ks is 1 or na
    float* partial;         // ks > 1: [ks][K][D] unscaled partial sums, added by filter_reduce_kernel
};

struct __align__(8) Barriers {
    uint64_t b_full[4], b_empty[4], s_full[2], s_empty[2], acc_full;
    uint32_t tmem_base, pad;
};

static inline size_t smem_bytes(int tnf, int h) {
    return 1024 + 4 * (size_t)STRIP_BYTES + (size_t)(tnf == 128 ? 2 : 4) * (2 * tnf * KBLK * 4) + sizeof(Barriers) +
           2 * (size_t)(2 * (h + TAB_PAD) + 1) * sizeof(float) + 16;
}

__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, const float4& v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Bt_hi / Bt_lo [D][Kp]: column h + j holds in[j][d] (hi / lo part), zero elsewhere.  32 x 32 tiles through shared
// memory: reads coalesced along d, writes coalesced along j.
// MC: `in` is the NVSwitch multicast address of the ranks' accumulator rows (som_peer.cu) and the load is the in-switch
// reduction multimem.ld_reduce.add -- the reduce-scatter half of the data-parallel tail happens in this pre-pass's read,
// with no reduced copy of the rows in between; block (0, 0) also reduces the packed buffer's 4-float tail exactly.
struct PeerIn {
    peer::Pads bufs;        // every rank's packed buffer (peer addresses), for the exact tail
    int64_t q_tail;         // float4 index of the tail in a packed buffer
    int world;
    float4* tail_out;
};

template <bool MC>
__global__ void __launch_bounds__(256) split_in_t_kernel(const float* __restrict__ in, int K, int D, int h, int Kp,
                                                         float* __restrict__ Bhi, float* __restrict__ Blo, PeerIn pin) {
    pdl_begin();
    trace_stamp(s_trace_buf, 1);
    __shared__ float tile[32][33];
    const int jp0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
    if (MC) {
        const int rr = threadIdx.x >> 3, c4 = (threadIdx.x & 7) * 4;         // 32 rows x 8 quads (D % 4 == 0)
        const int j = jp0 + rr - h, d = d0 + c4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j >= 0 && j < K && d < D) v = peer::mm_ld_reduce(in + (int64_t)j * D + d);
        tile[rr][c4] = v.x; tile[rr][c4 + 1] = v.y; tile[rr][c4 + 2] = v.z; tile[rr][c4 + 3] = v.w;
        if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0)
            *pin.tail_out = peer::exact_tail(pin.bufs, pin.q_tail, pin.world);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int j = jp0 + ty + 8 * i - h, d = d0 + tx;
            tile[ty + 8 * i][tx] = (j >= 0 && j < K && d < D) ? __ldg(in + (int64_t)j * D + d) : 0.f;
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int d = d0 + ty + 8 * i, jp = jp0 + tx;
        if (d < D && jp < Kp) {
            float hi, lo;
            tf32_split(tile[tx][ty + 8 * i], hi, lo);
            Bhi[(int64_t)d * Kp + jp] = hi;
            Blo[(int64_t)d * Kp + jp] = lo;
        }
    }
}

template <int TNF>
__global__ void __launch_bounds__(NUM_THREADS, 1)
filter_tc_kernel(const __grid_constant__ CUtensorMap map_bhi, const __grid_constant__ CUtensorMap map_blo,
                 const Params P) {
    pdl_launch_dependents();            // (the wait comes after the barrier / weight-table / TMEM prologue)
    // TNF = 64 (D <= 64): a stage's B_hi and B_lo blocks are adjacent 64-row K-major tiles, i.e. ONE 128-row tile
    // [B_hi ; B_lo].  An M128 x N64 tf32 MMA occupies the tensor pipe as long as an N128 one (71 against 67 cycles,
    // profiles/r01_mma_issue_microbench.log), so A_hi and A_lo are each multiplied with the concatenated tile: two N128
    // MMAs per k-step instead of three N64 ones (134 against 214 cycles).  Columns [0, 64) of the accumulator collect
    // A.B_hi, columns [64, 128) A.B_lo (now including the lo.lo term); the epilogue adds the halves.
    constexpr bool CAT = (TNF == 64);
    constexpr int ACC_COLS = CAT ? 2 * TNF : TNF;
    constexpr int NSB = nstage_b<TNF>();
    constexpr int B_BYTES = TNF * KBLK * 4;
    constexpr int B_STAGE = 2 * B_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* strips = aligned_tiles(smem_raw);
    uint8_t* b_ring = strips + 4 * STRIP_BYTES;          // [strip 0: hi | lo][strip 1: hi | lo][B stages]
    Barriers& bars = *reinterpret_cast<Barriers*>(b_ring + NSB * B_STAGE);
    float* tab_hi = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(&bars) + sizeof(Barriers));
    const int off = P.h + TAB_PAD;
    const int tab_n = 2 * off + 1;
    float* tab_lo = tab_hi + tab_n;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int ut = blockIdx.x, ct = blockIdx.y;
    // k-split (few tiles, e.g. a data-parallel rank's slice of units): the accumulation chains of the unsplit kernel
    // (chain a = k-blocks [a q, (a + 1) q), one TMEM accumulator each) become CTAs -- CTA z runs exactly chain z, and
    // filter_reduce_kernel adds the partial tiles in the same fixed order, so the result is bit-identical to the
    // unsplit kernel's
    const int ksp = (int)blockIdx.z, KS = P.ks;
    const int kb_lo = KS > 1 ? ksp * P.q : 0;
    const int kb_hi = KS > 1 ? (kb_lo + P.q < P.nkb ? kb_lo + P.q : P.nkb) : P.nkb;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSB; ++s) { mbar_init(&bars.b_full[s], 1); mbar_init(&bars.b_empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&bars.s_full[s], BUILD_WARPS); mbar_init(&bars.s_empty[s], 1); }
        mbar_init(&bars.acc_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < tab_n; i += NUM_THREADS) {
        const int t = i - off;
        tf32_split(band_weight(t < 0 ? -t : t, P.h, P.two_var), tab_hi[i], tab_lo[i]);
    }
    if (warp == 1) tmem_alloc(&bars.tmem_base, NACC * ACC_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars.tmem_base;
    pdl_wait();
    trace_stamp(s_trace_buf, 2);

    if (warp == 0) {
        // ================================ TMA producer (B blocks) ================================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int kb = kb_lo; kb < kb_hi; ++kb) {
                mbar_wait(&bars.b_empty[stage], phase ^ 1);
                uint8_t* sb = b_ring + (size_t)stage * B_STAGE;
                mbar_expect_tx(&bars.b_full[stage], 2 * B_BYTES);
                // padded inner coordinate of unit tile ut starts at ut * 128 (= a0 - h + h)
                tma_load_2d(&map_bhi, &bars.b_full[stage], sb, ut * TMU + kb * KBLK, ct * TNF);
                tma_load_2d(&map_blo, &bars.b_full[stage], sb + B_BYTES, ut * TMU + kb * KBLK, ct * TNF);
                if (++stage == NSB) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ==================================
        // The issuing thread paces this kernel (round-2 counters: 8 MMAs cost ~150 cycles of issue per k-block, the
        // scalar code around them ~540: descriptors rebuilt from pointers, an integer division for the chain, clock
        // reads), so everything per k-block is an increment: descriptors are base + offset in the 16-byte address field
        // (shared addresses < 256 KB fit its 14 bits), the chain index is a counter.
        const bool leader = elect_one();
        const uint32_t strip0 = smem_u32(strips), bring0 = smem_u32(b_ring);
        const uint64_t a_desc0 = umma_desc(strip0), b_desc0 = umma_desc(bring0);
        const uint32_t bempty0 = smem_u32(&bars.b_empty[0]), sempty0 = smem_u32(&bars.s_empty[0]);
        const uint32_t accfull = smem_u32(&bars.acc_full);
        int stage = 0, sbuf = 0;
        uint32_t phase = 0, sphase = 0;
        int in_chain = 0;                                     // k-blocks already issued into the current chain (KS == 1)
        uint32_t d_addr = tmem_base;
        bool first = true;
        for (int c0 = kb_lo; c0 < kb_hi; c0 += CK) {
            const int c1 = c0 + CK < kb_hi ? c0 + CK : kb_hi;
            mbar_wait(&bars.s_full[sbuf], sphase);
            uint64_t a_desc = a_desc0 + (uint64_t)((uint32_t)sbuf * (uint32_t)(2 * STRIP_BYTES >> 4));
            for (int kb = c0; kb < c1; ++kb) {
                mbar_wait(&bars.b_full[stage], phase);
                tc_fence_after();
                // k-block c0 + j of the strip = its rows [32 j, 32 j + 128): 4 KB further on, still 1024-byte aligned
                const uint64_t ahi = a_desc, alo = a_desc + (uint64_t)(STRIP_BYTES >> 4);
                const uint64_t bhi = b_desc0 + (uint64_t)((uint32_t)stage * (uint32_t)(B_STAGE >> 4));
                const uint64_t blo = bhi + (uint64_t)(B_BYTES >> 4);
                // The tensor core adds into its fp32 accumulator with truncation, a bias that grows with the length of
                // the accumulation chain (measured 1.7e-6 relative after 372 MMAs into one accumulator, band 851): the
                // k-blocks are dealt to NACC chains with an accumulator each and the epilogue adds those in fp32 (4e-7).
                if (leader) {
#pragma unroll
                    for (int ks = 0; ks < KBLK / 8; ++ks) {
                        const uint32_t acc0 = (!first || ks != 0) ? 1u : 0u;
                        if (CAT) {
                            tc_mma<MmaKind::TF32, 1, ACC_COLS>(d_addr, ahi + 2u * ks, bhi + 2u * ks, acc0);
                            tc_mma<MmaKind::TF32, 1, ACC_COLS>(d_addr, alo + 2u * ks, bhi + 2u * ks, 1u);
                        } else {
                            tc_mma<MmaKind::TF32, 1, TNF>(d_addr, ahi + 2u * ks, bhi + 2u * ks, acc0);
                            tc_mma<MmaKind::TF32, 1, TNF>(d_addr, alo + 2u * ks, bhi + 2u * ks, 1u);
                            tc_mma<MmaKind::TF32, 1, TNF>(d_addr, ahi + 2u * ks, blo + 2u * ks, 1u);
                        }
                    }
                    tc_commit(bempty0 + 8u * (uint32_t)stage);
                    if (kb + 1 == c1) tc_commit(sempty0 + 8u * (uint32_t)sbuf);
                    if (kb + 1 == kb_hi) tc_commit(accfull);
                }
                first = false;
                if (KS == 1 && ++in_chain == P.q) { in_chain = 0; d_addr += ACC_COLS; first = true; }
                a_desc += (uint64_t)((KBLK * 128) >> 4);
                if (++stage == NSB) { stage = 0; phase ^= 1; }
            }
            if (++sbuf == 2) { sbuf = 0; sphase ^= 1; }
        }
    } else {
        // ================================ A builders, then epilogue =====================
        {
            // The A operand of CK consecutive k-blocks is ONE Toeplitz strip: with the tile's unit rows in reverse order
            // (MMA row m = unit 127 - m) the block of k-block c0 + j is rows [32 j, 32 j + 128) of
            //     S[r][c] = w(32 c0 + r + c - h - 127),   r < 128 + 32 (CK - 1),
            // so the builders write 256 rows per CK = 5 k-blocks instead of 128 per k-block (2.5x fewer shared stores).
            // One thread per strip row, all eight 16-byte chunks of it.
            const int r = threadIdx.x - 64;                    // strip row of this thread
            const uint32_t row_off = (uint32_t)r * 128u;
            const uint32_t sw = (uint32_t)(r & 7);
            const uint32_t strips_u = smem_u32(strips), tab_hi_u = smem_u32(tab_hi), tab_lo_u = smem_u32(tab_lo);
            int sbuf = 0;
            uint32_t sphase = 0;
            for (int c0 = kb_lo; c0 < kb_hi; c0 += CK) {
                const int nk = c0 + CK < kb_hi ? CK : kb_hi - c0;
                mbar_wait_warp<false>(&bars.s_empty[sbuf], sphase ^ 1, lane);
                if (r < TMU + KBLK * (nk - 1)) {
                    const uint32_t sa = strips_u + (uint32_t)sbuf * (uint32_t)(2 * STRIP_BYTES) + row_off;
                    const uint32_t t_off = (uint32_t)(c0 * KBLK + r - P.h - (TMU - 1) + off) * 4u;
                    const uint32_t th = tab_hi_u + t_off, tl = tab_lo_u + t_off;
#pragma unroll
                    for (int q = 0; q < KBLK / 4; ++q) {
                        float4 hi, lo;
                        hi.x = lds_f32(th + 16u * q); hi.y = lds_f32(th + 16u * q + 4u);
                        hi.z = lds_f32(th + 16u * q + 8u); hi.w = lds_f32(th + 16u * q + 12u);
                        lo.x = lds_f32(tl + 16u * q); lo.y = lds_f32(tl + 16u * q + 4u);
                        lo.z = lds_f32(tl + 16u * q + 8u); lo.w = lds_f32(tl + 16u * q + 12u);
                        sts_v4(sa + ((((uint32_t)q) ^ sw) << 4), hi);
                        sts_v4(sa + (uint32_t)STRIP_BYTES + ((((uint32_t)q) ^ sw) << 4), lo);
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars.s_full[sbuf]);
                if (++sbuf == 2) { sbuf = 0; sphase ^= 1; }
            }
        }
        if (warp >= 6) goto done;                               // warps 2-5 own the four TMEM lane quarters
        // epilogue: TMEM lane quarter (warp & 3), 32 columns at a time; lane m of the accumulator is unit 127 - m
        mbar_wait_warp<true>(&bars.acc_full, 0, lane);
        tc_fence_after();
        const int lg = warp & 3;
        const int u = ut * TMU + (TMU - 1) - (lg * 32 + lane);
        const bool row_ok = u < P.K;
        const bool v4 = ((P.D & 3) == 0) && ((reinterpret_cast<uintptr_t>(P.out) & 15) == 0);
        float* orow = (KS > 1 ? P.partial + (int64_t)ksp * P.K * P.D : P.out) + (int64_t)(row_ok ? u : 0) * P.D;
        const float oscale = KS > 1 ? 1.0f : P.scale;            // split: raw partial sums, scaled after the reduction
#pragma unroll 1
        for (int c = 0; c < TNF / 32; ++c) {
            uint32_t v[32], w[32];
            const uint32_t taddr = tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(c * 32);
            tmem_ld32_issue(taddr, v);
            tmem_ld_wait(v);
            if (CAT) {                                           // chain value = (A.B_hi columns) + (A.B_lo columns)
                tmem_ld32_issue(taddr + (uint32_t)TNF, w);
                tmem_ld_wait(w);
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(w[i]));
            }
            if (KS == 1) {
#pragma unroll 1
                for (int a = 1; a < P.na; ++a) {                 // fixed order: ((a0 + a1) + a2) + a3
                    tmem_ld32_issue(taddr + (uint32_t)(a * ACC_COLS), w);
                    tmem_ld_wait(w);
                    if (CAT) {
                        uint32_t w2[32];
                        tmem_ld32_issue(taddr + (uint32_t)(a * ACC_COLS + TNF), w2);
                        tmem_ld_wait(w2);
#pragma unroll
                        for (int i = 0; i < 32; ++i) w[i] = __float_as_uint(__uint_as_float(w[i]) + __uint_as_float(w2[i]));
                    }
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(w[i]));
                }
            }
            const int d0 = ct * TNF + c * 32;
            if (row_ok && d0 < P.D) {
                if (v4 && d0 + 32 <= P.D) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<float4*>(orow + d0 + 4 * q) =
                            make_float4(oscale * __uint_as_float(v[4 * q]), oscale * __uint_as_float(v[4 * q + 1]),
                                        oscale * __uint_as_float(v[4 * q + 2]), oscale * __uint_as_float(v[4 * q + 3]));
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (d0 + i < P.D) orow[d0 + i] = oscale * __uint_as_float(v[i]);
                }
            }
        }
    }

done:
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, NACC * ACC_COLS);
    }
}

// out = scale * (((p0 + p1) + p2) + p3): the unsplit epilogue's order
__global__ void __launch_bounds__(256) filter_reduce_kernel(const float* __restrict__ partial, int64_t n, int na,
                                                            float scale, float* __restrict__ out) {
    pdl_begin();
    trace_stamp(s_trace_buf, 3);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        float v = partial[i];
        for (int a = 1; a < na; ++a) v += partial[(int64_t)a * n + i];
        out[i] = scale * v;
    }
}

struct Plan {
    int h, L, nkb, Kp, tnf, ks, q, na;
    size_t off_hi, off_lo, off_part, total;
};

static void make_plan(Plan* pl, int K, int D, int h) {
    pl->h = h;
    pl->L = (TMU + 2 * h + KBLK - 1) / KBLK * KBLK;
    pl->nkb = pl->L / KBLK;                             // >= 5 >= NACC: every accumulator is written
    const int n_ut = (K + TMU - 1) / TMU;
    pl->Kp = (n_ut - 1) * TMU + pl->L;                  // multiple of 32: 128-byte row pitch granularity for TMA
    pl->tnf = D > 64 ? 128 : 64;
    const size_t one = align_up((size_t)D * pl->Kp * sizeof(float), 1024);
    pl->off_hi = 0;
    pl->off_lo = one;
    // static rule: with fewer tiles than half the SMs, the NACC accumulation chains of a tile go to NACC CTAs
    const int64_t tiles = (int64_t)n_ut * ((D + pl->tnf - 1) / pl->tnf);
    pl->q = (pl->nkb + NACC - 1) / NACC;
    pl->na = (pl->nkb + pl->q - 1) / pl->q;
    pl->ks = (tiles * 2 <= sm_count()) ? pl->na : 1;
    pl->off_part = 2 * one;
    pl->total = 2 * one + (pl->ks > 1 ? align_up((size_t)pl->ks * K * D * sizeof(float), 1024) : 0);
}

}  // namespace ftc

// Static rule on the shape: the tensor-core filter pays a transposing pre-pass and 128-unit tiles.
bool filter_tc_applicable(int K, int D, int h) {
    // ... and one CTA per tile: with fewer than 32 tiles most SMs idle and the FFMA kernel (32-unit tiles) is faster
    // (measured at C1, K = 1024, D = 64: 8 tiles, 28 us against 21 us)
    // (fewer than 74 tiles are k-split over 4 CTAs each; below ~12 tiles the FFMA kernel wins again)
    const int64_t tiles = ceil_div64(K, ftc::TMU) * ceil_div64(D, D > 64 ? 128 : 64);
    if (K < 256 || D < 48 || h > ftc::MAX_H || tiles < 12) return false;
    static int cc_major = -1;
    if (cc_major < 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
            return false;
        cc_major = v;
    }
    return cc_major == 10 && tc::get_encode_fn() != nullptr;
}

size_t filter_tc_workspace_bytes(int K, int D, int h) {
    ftc::Plan pl;
    ftc::make_plan(&pl, K, D, h);
    return pl.total;
}

// the plan of launch_filter_tc for som_debug_filter_plan (f: FPF_COUNT fields)
void filter_tc_plan_fields(int K, int D, int h, int64_t* f) {
    ftc::Plan pl;
    ftc::make_plan(&pl, K, D, h);
    f[FPF_KERNEL] = pl.tnf == 128 ? FK_TC128 : FK_TC64;
    f[FPF_SMEM] = (int64_t)ftc::smem_bytes(pl.tnf, h);
    f[FPF_NKB] = pl.nkb;
    f[FPF_Q] = pl.q;
    f[FPF_NA] = pl.na;
    f[FPF_KS] = pl.ks;
    f[FPF_KP] = pl.Kp;
}

// pin != nullptr: `in` is a multicast address, read with the in-switch reduction (see split_in_t_kernel)
int launch_filter_tc_in(const float* in, float* out, int K, int D, float two_var, int h, float scale, void* ws,
                        size_t ws_bytes, cudaStream_t st, const ftc::PeerIn* pin) {
    using namespace ftc;
    Plan pl;
    make_plan(&pl, K, D, h);
    int rc = check_workspace(ws, ws_bytes, pl.total, "filter(tc)");
    if (rc) return rc;
    float* Bhi = (float*)((char*)ws + pl.off_hi);
    float* Blo = (float*)((char*)ws + pl.off_lo);
    {
        dim3 grid((unsigned)(pl.Kp / 32), (unsigned)ceil_div64(D, 32));
        if (pin != nullptr) launch_pdl(split_in_t_kernel<true>, grid, 256, 0, st, in, K, D, h, pl.Kp, Bhi, Blo, *pin);
        else launch_pdl(split_in_t_kernel<false>, grid, 256, 0, st, in, K, D, h, pl.Kp, Bhi, Blo, PeerIn{});
        rc = check_launch("split_in_t_kernel");
        if (rc) return rc;
    }
    CUtensorMap map_bhi, map_blo;
    rc = make_map2d(&map_bhi, Bhi, (uint64_t)D, (uint64_t)pl.Kp, (uint64_t)pl.Kp * 4, KBLK, (uint32_t)pl.tnf,
                        CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_map2d(&map_blo, Blo, (uint64_t)D, (uint64_t)pl.Kp, (uint64_t)pl.Kp * 4, KBLK, (uint32_t)pl.tnf,
                    CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    Params P;
    P.K = K; P.D = D; P.h = h; P.nkb = pl.nkb; P.two_var = two_var; P.scale = scale; P.out = out;
    P.q = pl.q; P.na = pl.na;
    P.ks = pl.ks; P.partial = (float*)((char*)ws + pl.off_part);
    const size_t smem = smem_bytes(pl.tnf, h);
    typedef void (*KernelFn)(const CUtensorMap, const CUtensorMap, const Params);
    static const KernelFn kernels[2] = {filter_tc_kernel<64>, filter_tc_kernel<128>};
    static PerDeviceFlag attr_done;
    rc = smem_opt_in(attr_done, kernels, 2, 227 * 1024, "filter(tc)");
    if (rc) return rc;
    dim3 grid((unsigned)ceil_div64(K, TMU), (unsigned)ceil_div64(D, pl.tnf), (unsigned)pl.ks);
    launch_pdl(kernels[pl.tnf == 128], grid, NUM_THREADS, smem, st, map_bhi, map_blo, P);
    rc = check_launch("filter_tc_kernel");
    if (rc || pl.ks == 1) return rc;
    const int64_t n = (int64_t)K * D;
    int blocks = (int)ceil_div64(n, 256 * 4);
    if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
    launch_pdl(filter_reduce_kernel, blocks, 256, 0, st, P.partial, n, pl.ks, scale, out);
    return check_launch("filter_reduce_kernel");
}

int launch_filter_tc(const float* in, float* out, int K, int D, float two_var, int h, float scale, void* ws,
                     size_t ws_bytes, cudaStream_t st) {
    return launch_filter_tc_in(in, out, K, D, two_var, h, scale, ws, ws_bytes, st, nullptr);
}

// som_peer.cu: out = scale * T @ (sum over the ranks of the rows at the multicast address mc_in), tail reduced exactly
int launch_filter_tc_peer(const float* mc_in, float* out, int K, int D, float two_var, int h, float scale, void* ws,
                          size_t ws_bytes, cudaStream_t st, const peer::Pads& bufs, int64_t q_tail, int world,
                          float* tail_out) {
    ftc::PeerIn pin;
    pin.bufs = bufs;
    pin.q_tail = q_tail;
    pin.world = world;
    pin.tail_out = reinterpret_cast<float4*>(tail_out);
    return launch_filter_tc_in(mc_in, out, K, D, two_var, h, scale, ws, ws_bytes, st, &pin);
}

}  // namespace som
