// K1 (tensor-core variant), small patch dimension D <= 16 ("config S"): BMU search as an
// error-compensated split GEMM on tcgen05 with the argmin fused into the TMEM epilogue.  sm_100a only.
// Two operand splits share the pipeline: FP16 hi/lo with power-of-two scaling (from 65 536 patches on: kind::f16,
// 4 MMAs per 128 x 256 tile, see the note above the kernel) and TF32 hi/lo (SOM_TC_S_F16=0: kind::tf32, 7 MMAs per tile,
// described first below).  Measured at C2: 4.1-4.3 ms vs 4.8-4.9 ms per 10 000 128 patches; in the FP16 mode the
// min-reduction of the epilogue (half-rate FMNMX on the ALU pipe, ~300 cycles per tile) and not the tensor pipe
// (512 cycles per tile) sets the pace: 850 cycles per tile, 547 with the reduction switched off.
//
// Replaces patchify + torch.cdist + torch.argmin of Codebook.get_patches_bmu
// (/root/reference/models/Codebook.py:77-99) for fine patches (BASELINE config 2: P=2, D=16, K=4096).
//
// Reduced distance rd[p][j] = ||c_j||^2 - 2 x_p . c_j (the row constant ||x_p||^2 is dropped).
// With hi = RNA-rounded TF32 part and lo = TF32-rounded remainder of a value:
//     rd = n1+n2+n3  - 2 x_hi.c_hi  - 2 x_lo.c_hi  - 2 x_hi.c_lo          (lo.lo dropped: 2^-24 relative)
// Operands are stored ONCE (hi | lo in one 128-byte swizzled row) and the three products are three
// groups of tcgen05.mma k-steps that start at different 32-byte offsets inside the same rows:
//     A row (patch)  = [ x_hi (Dp) | x_lo (Dp) ]           B row (unit) = [ -2c_hi (Dp) | -2c_lo (Dp) ]
//     tail k-step    : A = [1 1 1 0 0 0 0 0]   B = [n1 n2 n3 0 0 0 0 0]   (32-byte rows, SWIZZLE_32B)
// so a 128 x 256 tile costs 3*Dp/8 + 1 MMAs of K=8 (7 for D = 16) and a unit tile is 40 KB in shared memory.
//
// One persistent CTA per SM, 448 threads, warp-specialised:
//   warp 0      TMA producer: unit tiles (32 KB block + 8 KB tail) into a 3-stage mbarrier ring
//   warp 1      MMA issuer  : one thread, M128 x N256 x K8 kind::tf32, two TMEM accumulator stages.  The
//                             barrier checks for the NEXT tile are made before the LAST MMA of the current
//                             tile is issued: the issue queue is shallow (measured: the thread runs at most
//                             1-2 MMAs ahead of the pipe), so anything between two tiles is exposed otherwise.
//   warps 2-5   builders    : read patch rows from NCHW (patchify = address arithmetic, prefetched one
//                             super-tile ahead), split hi/lo and write the swizzled A rows of R = 4 resident
//                             patch tiles; then resolve the BMU inside the winning 8-unit chunk of the
//                             previous super-tile with exact fp32 FFMA scores (batched, latency-tolerant loads)
//   warps 6-13  epilogue    : tcgen05.ld 32x32b.x32 of their TMEM lane quarter / column half, running
//                             (min, 8-unit chunk) per patch row -- under one ALU op per distance; the N x K
//                             distance matrix never leaves TMEM
// Every streamed unit tile feeds R = 4 patch tiles.  Bound: tensor pipe (TF32 rate / 3).
#include "som_common.cuh"
#include "som_tc_ptx.cuh"
#include "som_tc_split.cuh"

#include <stdlib.h>

namespace som {
namespace tcs {
using namespace tc;

constexpr int R = 4;                         // resident patch tiles per super-tile
constexpr int NSTAGE = 3;                    // unit-tile ring stages
constexpr int BUILD_WARP0 = 2, BUILD_WARPS = 4;
constexpr int EPI_WARP0 = 6, EPI_WARPS = 8;
constexpr int NUM_THREADS = (EPI_WARP0 + EPI_WARPS) * 32;       // 448
constexpr int CHUNK = 8;                     // units per refine chunk
constexpr int DMAX = 16;
constexpr int TAIL_A_BYTES = TM * 32;        // 4 KB
constexpr int TAIL_B_BYTES = TN * 32;        // 8 KB
constexpr int STAGE_BYTES = B_BLK_BYTES + TAIL_B_BYTES;         // 40 KB
constexpr int TILES_BYTES = R * A_BLK_BYTES + TAIL_A_BYTES + NSTAGE * STAGE_BYTES;   // 188 KB

struct Params {
    int nks;                // k-steps per product group: Dp / 8
    int Rr;                 // resident patch tiles per super-tile in THIS launch (1..R): fewer for small batches
    int NT;                 // unit tiles
    int n_mtiles;           // patch tiles
    int64_t rows;           // valid patches
    int64_t unit_offset;
    int64_t* out_idx;
    float* out_rd;
    const float* x;
    Geom g;
    const float* W;
    const float* cn;
    int K;
    int dbg;                // timing-elimination switches, 0 unless built with -DSOM_TC_EXPERIMENTS
    const float* scale;     // FP16 mode: [s_c, t_c] written by cb_scale_kernel earlier on the stream
};

struct __align__(8) Barriers {
    uint64_t full[NSTAGE], empty[NSTAGE];
    uint64_t a_full[R], a_empty[R];
    uint64_t acc_full[2], acc_empty[2];
    uint64_t ref_full[2];
    uint32_t tmem_base, pad;
};
struct Aux {
    Barriers bars;
    float mrg_val[R][TM];
    int mrg_idx[R][TM];
    int cbase[2][R][TM];
    int foff[DMAX];
};
constexpr uint32_t SMEM_BYTES = 1024 + TILES_BYTES + sizeof(Aux);

__device__ long long g_prof[4];              // CTA 0: cycles of the MMA loop, tiles issued

// F16 = true: the same pipeline with a two-way FP16 split instead of the TF32 one (kind::f16 MMAs have K = 16 at the
// cycle cost of a K = 8 TF32 MMA: a tile is 4 MMAs instead of 7).  Rows are scaled by exact powers of two so that the
// halves stay in FP16's normal range -- per patch (s_p, from max |x|), per codebook (s_c, from max |c|) and, for the
// norm column, t_c (from max s_c ||c||^2; the norms are quadratic in the codebook's magnitude, the products are not) --
// and one 128-byte row carries everything:
//     A row = [ hi(s_p x) (16) | lo(s_p x) (16) | a_p a_p a_p 0.. (16) | unused ]                  a_p = s_p / t_c
//     B row = [ hi(-2 s_c c) (16) | lo(-2 s_c c) (16) | n1 n2 n3 0.. (16) of t_c s_c ||c||^2 | unused ]
// so the accumulator holds s_p s_c rd: a positive factor per row, which the argmin over units does not see.  The
// winning chunk is still resolved with exact fp32 FFMA scores of the unscaled operands.
template <bool F16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
bmu_tc_s_kernel(const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_t, const Params P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* tiles = aligned_tiles(smem_raw);
    uint8_t* a_slots = tiles;
    uint8_t* a_tail = tiles + R * A_BLK_BYTES;
    uint8_t* ring = a_tail + TAIL_A_BYTES;
    Aux& aux = *reinterpret_cast<Aux*>(ring + NSTAGE * STAGE_BYTES);
    Barriers& bars = aux.bars;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&bars.full[s], 1); mbar_init(&bars.empty[s], 1); }
        for (int r = 0; r < R; ++r) { mbar_init(&bars.a_full[r], BUILD_WARPS); mbar_init(&bars.a_empty[r], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&bars.acc_full[a], 1); mbar_init(&bars.acc_empty[a], EPI_WARPS); }
        mbar_init(&bars.ref_full[0], EPI_WARPS / 2);
        mbar_init(&bars.ref_full[1], EPI_WARPS / 2);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int d = threadIdx.x; d < P.g.D; d += NUM_THREADS) aux.foff[d] = feat_off(P.g, d);
    if (F16) {
        // chunks 5..7 of every A row are never written by the builders and chunk 5 is read by the tail k-step
        for (int i = threadIdx.x; i < R * A_BLK_BYTES / 16; i += NUM_THREADS)
            reinterpret_cast<uint4*>(a_slots)[i] = make_uint4(0u, 0u, 0u, 0u);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    } else if (threadIdx.x < TM) {
        write_tail_ones(a_tail, threadIdx.x);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&bars.tmem_base, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars.tmem_base;
    const int Rr = P.Rr;
    const int n_super = (P.n_mtiles + Rr - 1) / Rr;
    const int nks = P.nks;

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
                for (int n = 0; n < P.NT; ++n) {
                    mbar_wait(&bars.empty[stage], phase ^ 1);
                    uint8_t* sbase = ring + (size_t)stage * STAGE_BYTES;
                    mbar_expect_tx(&bars.full[stage], F16 ? B_BLK_BYTES : STAGE_BYTES);
                    tma_load_2d(&map_b, &bars.full[stage], sbase, 0, n * TN);
                    if (!F16) tma_load_2d(&map_t, &bars.full[stage], sbase + B_BLK_BYTES, 0, n * TN);
                    if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ==================================
        // The whole warp runs this loop: warp-uniform control flow keeps the operand descriptors in uniform
        // registers (a lane-0-only branch costs ~140 cycles per MMA issue in R2UR/vote sequences, this ~50);
        // one elected lane issues the tcgen05 ops.  The issue queue holds ~4 MMAs, so the barrier check,
        // fence and commit of a tile hide behind the previous tile as long as the loop stays lean.
        const bool leader = elect_one();
        const uint64_t adesc0 = umma_desc(smem_u32(a_slots));
        const uint64_t atdesc = umma_desc_sw32(smem_u32(a_tail));
        const uint64_t bdesc0 = umma_desc(smem_u32(ring));
        const uint64_t btdesc0 = umma_desc_sw32(smem_u32(ring + B_BLK_BYTES));
        constexpr uint32_t STAGE_UNITS = (uint32_t)STAGE_BYTES >> 4;
        constexpr uint32_t SLOT_UNITS = (uint32_t)A_BLK_BYTES >> 4;
        int stage = 0;
        uint32_t phase = 0, a_par = 0, j = 0;
        const long long t_begin = clock64();
        for (int st = blockIdx.x; st < n_super; st += gridDim.x) {
            const int r_eff = min(Rr, P.n_mtiles - st * Rr);
            for (int n = 0; n < P.NT; ++n) {
                mbar_wait(&bars.full[stage], phase);
                const uint64_t bd = bdesc0 + (uint32_t)stage * STAGE_UNITS;
                const uint64_t btd = btdesc0 + (uint32_t)stage * STAGE_UNITS;
                for (int r = 0; r < r_eff; ++r) {
                    if (n == 0) mbar_wait(&bars.a_full[r], a_par);
                    mbar_wait(&bars.acc_empty[j & 1u], ((j >> 1) & 1u) ^ 1u);
                    tc_fence_after();
                    const uint32_t d_addr = tmem_base + (j & 1u) * TN;
                    const uint64_t ad = adesc0 + (uint32_t)r * SLOT_UNITS;
                    if (F16) {
                        if (leader) {
                            // norm tail (k-step 2 of both rows) first, then hi.hi, lo.hi, hi.lo
                            tc_mma<MmaKind::F16>(d_addr, ad + 4u, bd + 4u, 0u);
                            tc_mma<MmaKind::F16>(d_addr, ad, bd, 1u);
                            tc_mma<MmaKind::F16>(d_addr, ad + 2u, bd, 1u);
                            tc_mma<MmaKind::F16>(d_addr, ad, bd + 2u, 1u);
                            tc_commit(&bars.acc_full[j & 1u]);
                            if (n == P.NT - 1) tc_commit(&bars.a_empty[r]);
                        }
                    } else if (leader) {
                        // norm tail first, then hi.hi, lo.hi, hi.lo
                        tc_mma<MmaKind::TF32>(d_addr, atdesc, btd, 0u);
#pragma unroll
                        for (int ks = 0; ks < DMAX / 8; ++ks)
                            if (ks < nks) tc_mma<MmaKind::TF32>(d_addr, ad + 2u * ks, bd + 2u * ks, 1u);
#pragma unroll
                        for (int ks = 0; ks < DMAX / 8; ++ks)
                            if (ks < nks) tc_mma<MmaKind::TF32>(d_addr, ad + 2u * (nks + ks), bd + 2u * ks, 1u);
#pragma unroll
                        for (int ks = 0; ks < DMAX / 8; ++ks)
                            if (ks < nks) tc_mma<MmaKind::TF32>(d_addr, ad + 2u * ks, bd + 2u * (nks + ks), 1u);
                        tc_commit(&bars.acc_full[j & 1u]);
                        if (n == P.NT - 1) tc_commit(&bars.a_empty[r]);
                    }
                    ++j;
                }
                if (leader) tc_commit(&bars.empty[stage]);
                if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
            }
            a_par ^= 1;
        }
        if (blockIdx.x == 0 && leader && j > 0) { g_prof[0] = clock64() - t_begin; g_prof[1] = (long long)j; }
    } else if (warp >= BUILD_WARP0 && warp < BUILD_WARP0 + BUILD_WARPS) {
        // ================================ A builders + chunk refine =====================
        const int t = threadIdx.x - BUILD_WARP0 * 32;       // patch row inside a tile
        const int D = P.g.D;
        const int vec = P.g.vec;
        const int Dp = nks * 8;
        const uint32_t row_off = (uint32_t)t * 128u;
        const uint32_t sw = (uint32_t)(t & 7);
        const bool v4 = ((D & 3) == 0);
        const bool w4 = v4 && ((reinterpret_cast<uintptr_t>(P.W) & 15) == 0);
        const int tc_exp = F16 ? (int)((__float_as_uint(__ldg(P.scale + 1)) >> 23) & 0xffu) - 127 : 0;
        float xv[R][DMAX];
        auto foff = [&](int d) { return aux.foff[d]; };
        auto prefetch = [&](int st_next) {
            const int r_nxt = (st_next < n_super) ? min(Rr, P.n_mtiles - st_next * Rr) : 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int64_t p = (int64_t)(st_next * Rr + r) * TM + t;
                const bool ok = (r < r_nxt) && (p < P.rows);
                load_row(xv[r], P.x + (ok ? patch_base(P.g, p) : 0), ok, 0, D, vec, foff);
            }
        };
        // exact fp32 scores of the CHUNK candidates of one row, four candidates' loads in flight at a time;
        // strict '>' in ascending unit order keeps the lowest index on ties (same arithmetic as the FFMA variant)
        auto refine_row = [&](int64_t p, int u0) {
            float xr[DMAX];
            load_row(xr, P.x + patch_base(P.g, p), true, 0, D, vec, foff);
            if (u0 < 0 || u0 >= P.K) u0 = 0;           // defensive: the epilogue only writes bases in [0, K_pad)
            float best = -INFINITY;
            int bu = u0;
#pragma unroll
            for (int h = 0; h < CHUNK; h += 4) {
                float wr[4][DMAX];
                float accv[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int u = u0 + h + c;
                    const bool ok = u < P.K;
                    const float* wp = P.W + (int64_t)(ok ? u : 0) * D;
                    accv[c] = ok ? -0.5f * __ldg(P.cn + u) : -INFINITY;
#pragma unroll
                    for (int d = 0; d < DMAX; d += 4) {
                        if (d < D) {
                            if (w4) {
                                const float4 q = __ldg(reinterpret_cast<const float4*>(wp + d));
                                wr[c][d] = q.x; wr[c][d + 1] = q.y; wr[c][d + 2] = q.z; wr[c][d + 3] = q.w;
                            } else {
#pragma unroll
                                for (int e = 0; e < 4; ++e) wr[c][d + e] = (d + e < D) ? __ldg(wp + d + e) : 0.f;
                            }
                        } else {
#pragma unroll
                            for (int e = 0; e < 4; ++e) wr[c][d + e] = 0.f;
                        }
                    }
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float a = accv[c];
#pragma unroll
                    for (int d = 0; d < DMAX; ++d)
                        if (d < D) a = fmaf(xr[d], wr[c][d], a);
                    if (a > best) { best = a; bu = u0 + h + c; }
                }
            }
            P.out_idx[p] = (int64_t)bu + P.unit_offset;
            if (P.out_rd) P.out_rd[p] = -2.0f * best;
        };
        auto refine_super = [&](int st_done, int it_done) {
            mbar_wait_warp<true>(&bars.ref_full[it_done & 1], (uint32_t)(it_done >> 1) & 1u, lane);
            const int r_done = min(Rr, P.n_mtiles - st_done * Rr);
            for (int r = 0; r < r_done; ++r) {
                const int64_t p = (int64_t)(st_done * Rr + r) * TM + t;
                if (p < P.rows) refine_row(p, aux.cbase[it_done & 1][r][t]);
            }
        };

        prefetch(blockIdx.x);
        uint32_t a_epar = 1;
        int st_prev = -1, it = 0;
        for (int st = blockIdx.x; st < n_super; st += gridDim.x, ++it) {
            const int r_eff = min(Rr, P.n_mtiles - st * Rr);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (r < r_eff) {
                    mbar_wait_warp<true>(&bars.a_empty[r], a_epar, lane);
                    uint8_t* slot = a_slots + (size_t)r * A_BLK_BYTES + row_off;
                    if (F16) {
                        float m = 0.f;
#pragma unroll
                        for (int d = 0; d < DMAX; ++d) m = fmaxf(m, fabsf(xv[r][d]));
                        float sp, ap;
                        int es;
                        f16_row_scale(m, tc_exp, sp, ap, es);
                        float hi[DMAX], lo[DMAX];
#pragma unroll
                        for (int d = 0; d < DMAX; ++d) f16_split(xv[r][d] * sp, hi[d], lo[d]);     // scaling exact
                        const float h0[8] = {hi[0], hi[1], hi[2], hi[3], hi[4], hi[5], hi[6], hi[7]};
                        const float h1[8] = {hi[8], hi[9], hi[10], hi[11], hi[12], hi[13], hi[14], hi[15]};
                        const float l0[8] = {lo[0], lo[1], lo[2], lo[3], lo[4], lo[5], lo[6], lo[7]};
                        const float l1[8] = {lo[8], lo[9], lo[10], lo[11], lo[12], lo[13], lo[14], lo[15]};
                        const float tl[8] = {ap, ap, ap, 0.f, 0.f, 0.f, 0.f, 0.f};
                        *reinterpret_cast<uint4*>(slot + ((0u ^ sw) << 4)) = pack_h8(h0);
                        *reinterpret_cast<uint4*>(slot + ((1u ^ sw) << 4)) = pack_h8(h1);
                        *reinterpret_cast<uint4*>(slot + ((2u ^ sw) << 4)) = pack_h8(l0);
                        *reinterpret_cast<uint4*>(slot + ((3u ^ sw) << 4)) = pack_h8(l1);
                        *reinterpret_cast<uint4*>(slot + ((4u ^ sw) << 4)) = pack_h8(tl);
                    } else if (v4) {
                        // 16-byte chunk q of the row lands at (q ^ (t & 7)): 8 consecutive rows fill one
                        // conflict-free shared-memory wavefront
                        const int dq = Dp >> 2;
#pragma unroll
                        for (int d4 = 0; d4 < DMAX / 4; ++d4) {
                            if (d4 < dq) {
                                float4 hi, lo;
                                tf32_split4(&xv[r][4 * d4], hi, lo);
                                *reinterpret_cast<float4*>(slot + ((((uint32_t)d4) ^ sw) << 4)) = hi;
                                *reinterpret_cast<float4*>(slot + ((((uint32_t)(dq + d4)) ^ sw) << 4)) = lo;
                            }
                        }
                    } else {
#pragma unroll
                        for (int d = 0; d < DMAX; ++d) {
                            if (d < Dp) {
                                float hi, lo;
                                tf32_split(xv[r][d], hi, lo);       // zero beyond D (load_row)
                                const uint32_t kh = (uint32_t)d, kl = (uint32_t)(Dp + d);
                                *reinterpret_cast<float*>(slot + ((((kh >> 2) ^ sw) << 4) | ((kh & 3u) << 2))) = hi;
                                *reinterpret_cast<float*>(slot + ((((kl >> 2) ^ sw) << 4) | ((kl & 3u) << 2))) = lo;
                            }
                        }
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars.a_full[r]);
                }
            }
            a_epar ^= 1;
            if (st_prev >= 0 && !(P.dbg & 1)) refine_super(st_prev, it - 1);
            prefetch(st + gridDim.x);                // rows of the next super-tile, most of a super-tile ahead
            st_prev = st;
        }
        if (st_prev >= 0 && !(P.dbg & 1)) refine_super(st_prev, it - 1);
    } else if (warp >= EPI_WARP0) {
        // ================================ epilogue ====================================
        const int ew = warp - EPI_WARP0;            // 0..7
        const int half = ew >> 2;                   // column half of the accumulator
        const int lg = warp & 3;                    // TMEM lane quarter this warp may access
        const int row = lg * 32 + lane;             // patch row inside the tile
        uint32_t j = 0;
        int it = 0;
        for (int st = blockIdx.x; st < n_super; st += gridDim.x, ++it) {
            const int r_eff = min(Rr, P.n_mtiles - st * Rr);
            float best[R];
            int bidx[R];
#pragma unroll
            for (int r = 0; r < R; ++r) { best[r] = INFINITY; bidx[r] = 0; }
            for (int n = 0; n < P.NT; ++n) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    if (r < r_eff) {
                        const uint32_t acc = j & 1u;
                        mbar_wait(&bars.acc_full[acc], (j >> 1) & 1u);
                        tc_fence_after();
                        const uint32_t taddr = tmem_base + ((uint32_t)(lg * 32) << 16) + acc * TN + (uint32_t)half * 128u;
                        const int col0 = n * TN + half * 128;
                        // minimum per CHUNK(8)-column group; only (min, chunk) is tracked
                        auto consume = [&](const uint32_t (&v)[32], int c) {
                            float q[4];
#pragma unroll
                            for (int g = 0; g < 4; ++g) {
                                // balanced tree of 3-input minima (FMNMX3 runs at half rate on the ALU pipe: depth, not
                                // only count, decides how well two epilogue warps fill it)
                                const float a = fminf(fminf(__uint_as_float(v[g * 8]), __uint_as_float(v[g * 8 + 1])),
                                                      __uint_as_float(v[g * 8 + 2]));
                                const float b = fminf(fminf(__uint_as_float(v[g * 8 + 3]), __uint_as_float(v[g * 8 + 4])),
                                                      __uint_as_float(v[g * 8 + 5]));
                                const float c = fminf(__uint_as_float(v[g * 8 + 6]), __uint_as_float(v[g * 8 + 7]));
                                q[g] = fminf(fminf(a, b), c);
                            }
                            const float m = fminf(fminf(q[0], q[1]), fminf(q[2], q[3]));
                            if (m < best[r]) {
                                best[r] = m;
                                const int sub = (q[0] == m) ? 0 : (q[1] == m) ? 1 : (q[2] == m) ? 2 : 3;
                                bidx[r] = col0 + c * 32 + sub * CHUNK;
                            }
                        };
                        if (P.dbg & 6) {
                            // timing elimination (experiment builds): 2 = loads without the reduction, 4 = no loads
                            if (P.dbg & 2) {
                                uint32_t va[32], vb[32];
                                tmem_ld32_issue(taddr, va); tmem_ld_wait(va);
                                tmem_ld32_issue(taddr + 32, vb); tmem_ld_wait(vb);
                                tmem_ld32_issue(taddr + 64, va); tmem_ld_wait(va);
                                tmem_ld32_issue(taddr + 96, vb); tmem_ld_wait(vb);
                                if (va[0] == 0x7fc12345u && vb[0] == 0x7fc12345u) best[r] = 0.f;
                            }
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&bars.acc_empty[acc]);
                            ++j;
                            continue;
                        }
                        tmem_drain<4>(taddr, consume, [&] { if (lane == 0) mbar_arrive(&bars.acc_empty[acc]); });
                        ++j;
                    }
                }
            }
            // merge the two column halves (value asc, index asc); the chunk bases go to the builders
            if (half == 1) {
#pragma unroll
                for (int r = 0; r < R; ++r) { aux.mrg_val[r][row] = best[r]; aux.mrg_idx[r][row] = bidx[r]; }
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (half == 0) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    if (r < r_eff) {
                        argmin_merge(best[r], bidx[r], aux.mrg_val[r][row], aux.mrg_idx[r][row]);
                        aux.cbase[it & 1][r][row] = bidx[r];
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars.ref_full[it & 1]);       // release: chunk bases visible
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// B rows [-2 hi(c) (Dp) | -2 lo(c) (Dp) | 0..] (32 floats) and tail rows [n1 n2 n3 0 0 0 0 0]; rows >= K are
// padding units whose norm can never be the minimum
__global__ void __launch_bounds__(256) split_w_s_kernel(const float* __restrict__ W, const float* __restrict__ cn,
                                                        int K, int D, int Dp, int K_pad, float* __restrict__ Bp,
                                                        float* __restrict__ Tp) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= (int64_t)K_pad * 40) return;
    const int row = (int)(t / 40);
    const int c = (int)(t - (int64_t)row * 40);
    if (c < 32) {
        float out = 0.f;
        if (row < K && c < 2 * Dp) {
            const int d = (c < Dp) ? c : c - Dp;
            if (d < D) {
                float hi, lo;
                tf32_split(W[(int64_t)row * D + d], hi, lo);
                out = -2.0f * (c < Dp ? hi : lo);
            }
        }
        Bp[(int64_t)row * 32 + c] = out;
    } else {
        const int k = c - 32;
        float out = 0.f;
        if (row < K) {
            float n1, n2, n3;
            tf32_norm_split3(cn[row], n1, n2, n3);
            out = (k == 0) ? n1 : (k == 1) ? n2 : (k == 2) ? n3 : 0.f;
        } else if (k == 0) {
            out = PAD_NORM;
        }
        Tp[(int64_t)row * 8 + k] = out;
    }
}

// FP16 mode, per-codebook scales (powers of two): s_c puts max |s_c c| in [64, 128), t_c puts max t_c s_c ||c||^2 in
// [2^14, 2^15) (FP16 tops out at 65504); an all-zero or non-finite codebook keeps both at 1.  One CTA: the config-S
// codebooks are K x (D <= 16) floats.
__global__ void __launch_bounds__(1024) cb_scale_kernel(const float* __restrict__ W, const float* __restrict__ cn,
                                                        int K, int D, float* __restrict__ scale_out) {
    __shared__ float sh_c[32], sh_n[32];
    float mc = 0.f, mn = 0.f;
    const int64_t total = (int64_t)K * D;
    if ((reinterpret_cast<uintptr_t>(W) & 15) == 0) {
        // four 16-byte loads in flight per thread: one CTA is latency-bound otherwise
        const float4* W4 = reinterpret_cast<const float4*>(W);
        const int64_t n4 = total >> 2;
        for (int64_t i = threadIdx.x; i < n4; i += 4096) {
            float4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                q[u] = (i + u * 1024 < n4) ? __ldg(W4 + i + u * 1024) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u)
                mc = fmaxf(fmaxf(mc, fmaxf(fabsf(q[u].x), fabsf(q[u].y))), fmaxf(fabsf(q[u].z), fabsf(q[u].w)));
        }
        for (int64_t i = (n4 << 2) + threadIdx.x; i < total; i += 1024) mc = fmaxf(mc, fabsf(W[i]));
    } else {
        for (int64_t i = threadIdx.x; i < total; i += 1024) mc = fmaxf(mc, fabsf(W[i]));
    }
    for (int i = threadIdx.x; i < K; i += 1024) mn = fmaxf(mn, fabsf(cn[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mc = fmaxf(mc, __shfl_xor_sync(0xffffffffu, mc, o));
        mn = fmaxf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    }
    if ((threadIdx.x & 31) == 0) { sh_c[threadIdx.x >> 5] = mc; sh_n[threadIdx.x >> 5] = mn; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) { mc = fmaxf(mc, sh_c[w]); mn = fmaxf(mn, sh_n[w]); }
        const int ec = (int)((__float_as_uint(mc) >> 23) & 0xffu), en = (int)((__float_as_uint(mn) >> 23) & 0xffu);
        int e = 0, g = 0;
        if (mc > 0.f && ec != 0xff && en != 0xff) {
            e = 133 - ec;                                   // max |s_c c| in [64, 128)
            e = e > 60 ? 60 : (e < -60 ? -60 : e);
            const float msn = mn * __uint_as_float((uint32_t)(127 + e) << 23);
            const int es = (int)((__float_as_uint(msn) >> 23) & 0xffu);
            if (msn > 0.f && es != 0xff) g = 141 - es;     // max t_c s_c ||c||^2 in [2^14, 2^15)
            g = g > 60 ? 60 : (g < -60 ? -60 : g);
        }
        scale_out[0] = __uint_as_float((uint32_t)(127 + e) << 23);
        scale_out[1] = __uint_as_float((uint32_t)(127 + g) << 23);
    }
}

// FP16 mode B rows: 64 halves = [ hi(-2 s_c c) (16) | lo (16) | n1 n2 n3 0.. (16) of s_c ||c||^2 | 0 (16) ].  Rows >= K
// repeat unit K - 1: a padding unit then never beats a real one (ties go to the lower chunk), whatever the patch holds.
__global__ void __launch_bounds__(256) split_w_s16_kernel(const float* __restrict__ W, const float* __restrict__ cn,
                                                          int K, int D, int K_pad, const float* __restrict__ scale,
                                                          __half* __restrict__ Bp) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= (int64_t)K_pad * 64) return;
    const int row = (int)(t >> 6);
    const int c = (int)(t & 63);
    const int src = row < K ? row : K - 1;
    const float sc = scale[0], tcs = scale[1];
    float out = 0.f;
    if (c < 32) {
        const int d = c & 15;
        if (d < D) {
            float hi, lo;
            f16_split(-2.0f * sc * W[(int64_t)src * D + d], hi, lo);          // exact scaling
            out = (c < 16) ? hi : lo;
        }
    } else if (c < 35) {
        float n1, n2, n3;
        f16_norm_split3(cn[src] * sc * tcs, n1, n2, n3);
        out = (c == 32) ? n1 : (c == 33) ? n2 : n3;
    }
    Bp[(int64_t)row * 64 + c] = __float2half_rn(out);
}

}  // namespace tcs

bool tc_s_applicable(int D) { return D >= 1 && D <= tcs::DMAX; }

size_t tc_s_workspace_bytes(int64_t n_patches, int D, int K) {
    (void)n_patches; (void)D;
    const size_t K_pad = (size_t)(K + tc::TN - 1) / tc::TN * tc::TN;
    return align_up(K_pad * 32 * 4, 1024) + align_up(K_pad * 8 * 4, 1024) + 1024;     // + the FP16 mode's scale slot
}

// Split mode of the config-S kernel.  Static rule: FP16 from 65 536 patches on (C2: 4.1-4.3 vs 4.8-4.9 ms); below that
// a launch is tens of microseconds and the extra scale pre-pass (one CTA, a few us) would eat the gain, so small batches
// keep the 3xTF32 mode.  The caller's variant (SOM_BMU_TC_TF32 / SOM_BMU_TC_F16) forces one arithmetic for every size.
bool tc_s_f16_mode(int64_t n_patches, int arith) {
    return arith == 0 ? n_patches >= 65536 : arith == 2;
}

// Resident patch tiles per CTA.  Small batches: fewer resident tiles per CTA so that every SM gets a super-tile (a unit
// tile then feeds fewer MMAs, but the sweep over the unit tiles is what bounds a small batch).
static int patch_tiles(int64_t n_patches) { return (int)ceil_div64(n_patches, tc::TM); }
static int unit_tiles(int K) { return (K + tc::TN - 1) / tc::TN; }

static int tc_s_resident_tiles(int64_t n_patches) {
    const int n_mtiles = patch_tiles(n_patches);
    const int rr = (n_mtiles + sm_count() - 1) / sm_count();
    return rr < 1 ? 1 : (rr > tcs::R ? tcs::R : rr);
}

// the plan of launch_bmu_tc_s for som_debug_bmu_plan (f: PF_COUNT fields, pre-filled with -1)
void tc_s_plan_fields(int64_t n_patches, int K, int arith, int64_t* f) {
    f[PF_ARITH] = tc_s_f16_mode(n_patches, arith) ? 1 : 0;
    f[PF_CG] = 1;
    f[PF_RR] = tc_s_resident_tiles(n_patches);
    f[PF_NT] = unit_tiles(K);
    f[PF_MTILES] = patch_tiles(n_patches);
}

int launch_bmu_tc_s(const float* x, const Geom& g, const float* W, const float* cn, int K, int64_t unit_offset,
                    int64_t* out_idx, float* out_rd, void* ws, size_t ws_bytes, int arith, cudaStream_t st) {
    using namespace tcs;
    const int64_t n = g.n_patches;
    if (n == 0) return SOM_OK;
    const int D = g.D;
    const int Dp = (D + 7) / 8 * 8;
    const int K_pad = (K + TN - 1) / TN * TN;
    int rc = check_workspace(ws, ws_bytes, tc_s_workspace_bytes(n, D, K), "bmu(tc)");
    if (rc) return rc;
    float* Bp = (float*)ws;
    float* Tp = (float*)((char*)ws + align_up((size_t)K_pad * 32 * 4, 1024));
    float* scale = (float*)((char*)Tp + align_up((size_t)K_pad * 8 * 4, 1024));
    const bool f16 = tc_s_f16_mode(n, arith);
    if (f16) {
        cb_scale_kernel<<<1, 1024, 0, st>>>(W, cn, K, D, scale);
        rc = check_launch("cb_scale_kernel");
        if (rc) return rc;
        const int64_t items = (int64_t)K_pad * 64;
        split_w_s16_kernel<<<(unsigned)ceil_div64(items, 256), 256, 0, st>>>(W, cn, K, D, K_pad, scale, (__half*)Bp);
        rc = check_launch("split_w_s16_kernel");
        if (rc) return rc;
    } else {
        const int64_t items = (int64_t)K_pad * 40;
        split_w_s_kernel<<<(unsigned)ceil_div64(items, 256), 256, 0, st>>>(W, cn, K, D, Dp, K_pad, Bp, Tp);
        rc = check_launch("split_w_s_kernel");
        if (rc) return rc;
    }
    CUtensorMap map_b, map_t;
    rc = make_map2d(&map_b, Bp, (uint64_t)K_pad, 32, 128, 32, TN, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_map2d(&map_t, Tp, (uint64_t)K_pad, 8, 32, 8, TN, CU_TENSOR_MAP_SWIZZLE_32B);
    if (rc) return rc;

    Params P;
    P.nks = Dp / 8; P.NT = unit_tiles(K); P.n_mtiles = patch_tiles(n); P.rows = n;
    P.unit_offset = unit_offset; P.out_idx = out_idx; P.out_rd = out_rd;
    P.x = x; P.g = g; P.W = W; P.cn = cn; P.K = K; P.scale = scale;
    P.dbg = 0;
#ifdef SOM_TC_EXPERIMENTS
    // timing-elimination switches (skip refine / loads / conversion): results are wrong, experiment builds only
    { static int dbg = -1; if (dbg < 0) { const char* e = getenv("SOM_TC_DEBUG"); dbg = e ? atoi(e) : 0; } P.dbg = dbg; }
#endif
    static PerDeviceFlag attr_done;
    typedef void (*KernelFn)(const CUtensorMap, const CUtensorMap, const Params);
    static const KernelFn kernels[2] = {bmu_tc_s_kernel<false>, bmu_tc_s_kernel<true>};
    rc = smem_opt_in(attr_done, kernels, 2, (int)SMEM_BYTES, "bmu(tc)");
    if (rc) return rc;
    P.Rr = tc_s_resident_tiles(n);
    const int n_super = (P.n_mtiles + P.Rr - 1) / P.Rr;
    const int grid = n_super < sm_count() ? n_super : sm_count();
    kernels[f16]<<<grid, NUM_THREADS, SMEM_BYTES, st>>>(map_b, map_t, P);
    return check_launch("bmu_tc_s_kernel");
}

}  // namespace som

// debug: cycles spent by CTA 0's MMA issue loop and the tiles it issued in the last config-S launch
extern "C" SOM_API int som_debug_tc_cycles(long long* out2) {
    return (int)cudaMemcpyFromSymbol(out2, som::tcs::g_prof, 2 * sizeof(long long));
}
