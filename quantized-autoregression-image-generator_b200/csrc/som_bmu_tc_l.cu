// K1 (tensor-core variant), patch dimension D > 16: BMU search as an error-compensated 3xTF32 GEMM on tcgen05.
// sm_100a only.
//
// Replaces patchify + torch.cdist + torch.argmin of Codebook.get_patches_bmu
// (/root/reference/models/Codebook.py:77-99): BASELINE config 1 / 4 (D = 64), config 3 (whole-fmap codebook,
// D = 4096, K = 512, 4096 patches) and config 5 (D = 256, K = 32 768 per GPU).
//
//     rd[p][j] = ||c_j||^2 - 2 x_p . c_j = n1+n2+n3 - 2 x_hi.c_hi - 2 x_lo.c_hi - 2 x_hi.c_lo
// (hi = RNA TF32 part, lo = TF32-rounded remainder; the dropped lo.lo term is 2^-24 relative).  The feature
// axis is cut into 32-feature blocks; per block the hi and lo parts are stored ONCE and feed three groups of
// K=8 MMAs:  A_hi x B_hi,  A_lo x B_hi,  A_hi x B_lo.  The norms enter through one extra K=8 step
// (A = [1 1 1 0..], B = [n1 n2 n3 0..], 32-byte rows, SWIZZLE_32B).
//
// One persistent CTA per SM (or CTA pair per two SMs), 448 threads, warp-specialised:
//   warp 0      TMA producer: B_hi / B_lo blocks of the pre-split codebook into a 128 KB ring, norm tails into a
//                             2-stage ring; in the streamed mode also the pre-split A blocks
//   warp 1      MMA issuer  : warp-uniform loop, one elected lane issues M128 (M256 for pairs) x N256 x K8
//                             kind::tf32 into two TMEM accumulator stages
//   warps 2-9   builders    : two groups of four warps: a thread reads 32 features of its patch row straight from
//                             NCHW (patchify = address arithmetic, the next block's loads in flight while the
//                             current one is converted), splits hi/lo and writes both swizzled 16 KB operand
//                             blocks of its A slot -- no operand copy in HBM
//   warps 10-13 epilogue    : tcgen05.ld of their TMEM lane quarter, all 256 columns
// Modes (static rule on the shape, see make_plan):
//   resident-A  D <= 64: the patch tile's blocks stay in the two A slots for all unit tiles (C1, C4)
//   streamed    D  > 64, at least as many patch tiles as SMs: split_x_l_kernel pre-splits patch rows into an
//               L2-sized workspace chunk and the producer streams A by TMA (C5); running exact (min, index) per
//               patch row over all unit tiles -- the N x K distance matrix never leaves TMEM
//   split-K     D  > 64, few patch tiles (C3: 32 tiles, 2 unit tiles, 128 feature blocks): the feature axis is
//               split over S CTAs per patch tile, each A-slot fill feeds both TMEM accumulators (two unit
//               tiles), partial distances (S x N x K fp32) go to a workspace and splitk_argmin_kernel adds
//               them in fixed order and takes the argmin
//   CTA pairs   CG = 2 (cta_group::2): each CTA holds its own A tile and HALF of every B block; resident-A and
//               streamed modes with at least two waves of patch tiles
// Bound: tensor pipe (TF32 rate / 3): 94.8 % active at C4, 87 % at C5, 58 % at C3 (profiles/).
#include "som_common.cuh"
#include "som_tc_ptx.cuh"
#include "som_tc_split.cuh"

#include <stdlib.h>

namespace som {
namespace tcl {
using namespace tc;

constexpr int NA = 2;                        // A ring slots (hi + lo block)
constexpr int B_RING_BYTES = 4 * B_BLK_BYTES;                   // 128 KB: 4 stages of 32 KB, or 8 of 16 KB per CTA of a pair
constexpr int BUILD_WARP0 = 2, BUILD_WARPS = 8;             // two groups of 4 warps, alternate feature blocks
constexpr int EPI_WARP0 = 10, EPI_WARPS = 4;
constexpr int NUM_THREADS = (EPI_WARP0 + EPI_WARPS) * 32;       // 448
constexpr int A_SLOT_BYTES = 2 * A_BLK_BYTES;                   // 32 KB
constexpr int TAIL_A_BYTES = TM * 32;        // 4 KB
constexpr int TAIL_B_BYTES = TN * 32;        // 8 KB
constexpr int FOFF_MAX = 1024;               // feature-offset table entries kept in shared memory
constexpr int MAX_SPLIT = 8;
constexpr int NB_MAX = 8;
constexpr int TILES_BYTES = NA * A_SLOT_BYTES + B_RING_BYTES + TAIL_A_BYTES + 2 * TAIL_B_BYTES;   // 212 KB

struct Params {
    int DB;                 // 32-feature blocks
    int nks_last;           // k-steps of the last block
    int NT;                 // unit tiles
    int n_mtiles;           // patch tiles
    int S;                  // feature splits (1: ARGMIN epilogue)
    int fb_per_split;
    int U;                  // unit-tile splits (resident-A mode, small batches): candidates merged afterwards
    int nt_per_u;
    float* cand_rd;         // [U][rows]   (U > 1)
    int64_t* cand_idx;      // [U][rows]
    int K_pad;
    int64_t rows;           // valid patches
    int64_t unit_offset;
    int64_t* out_idx;
    float* out_rd;
    float* partial;         // [S][n_mtiles * 128][K_pad]   (S > 1)
    const float* x;
    Geom g;
    int dbg;                // timing-elimination switches, 0 unless built with -DSOM_TC_EXPERIMENTS
    int a_tma;              // streamed mode: A blocks arrive by TMA from the pre-split workspace (builders idle)
    int tile0;              // first patch tile of this launch inside the workspace chunk numbering (0)
};

struct __align__(8) Barriers {
    uint64_t b_full[NB_MAX], b_empty[NB_MAX];
    uint64_t t_full[2], t_empty[2];
    uint64_t a_full[NA], a_empty[NA];
    uint64_t acc_full[2], acc_empty[2];
    uint32_t tmem_base, pad;
};
struct Aux {
    Barriers bars;
    int foff[FOFF_MAX];
};
constexpr uint32_t SMEM_BYTES = 1024 + TILES_BYTES + sizeof(Aux);

// SPLITK: partial-distance epilogue (feature axis split over CTAs).  ARES: the patch tile's operand blocks stay
// resident in the two A slots for all unit tiles (D <= 64: one slot per 32-feature block) instead of streaming.
// CG = 2: CTA pairs (cluster of two, cta_group::2).  Each CTA builds its own 128-patch A tile and loads HALF of
// every B block (128 units); the leader CTA issues M256 x N256 MMAs that read both CTAs' shared memory, so B
// costs each SM half the L2 traffic and half the shared-memory fill / operand-read bandwidth.
template <bool SPLITK, bool ARES, int CG>
__global__ void __launch_bounds__(NUM_THREADS, 1)
bmu_tc_l_kernel(const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_t,
                const __grid_constant__ CUtensorMap map_a, const Params P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* tiles = aligned_tiles(smem_raw);
    // unit tiles fed by one A-slot fill: split-K jobs use both TMEM accumulators for two unit tiles at once, which
    // halves the builders' work per MMA (they are the bottleneck there); the other modes double-buffer one tile
    constexpr int NI = SPLITK ? 2 : 1;
    constexpr int B_STAGE = B_BLK_BYTES / CG;       // this CTA's share of a 256-unit block
    constexpr int NB = B_RING_BYTES / B_STAGE;
    constexpr int T_STAGE = TAIL_B_BYTES / CG;
    uint8_t* a_ring = tiles;
    uint8_t* b_ring = a_ring + NA * A_SLOT_BYTES;
    uint8_t* a_tail = b_ring + B_RING_BYTES;
    uint8_t* t_ring = a_tail + TAIL_A_BYTES;
    const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;
    const int job0 = (CG == 2) ? (int)cluster_id_x() : (int)blockIdx.x;
    const int job_stride = (CG == 2) ? (int)cluster_count_x() : (int)gridDim.x;
    Aux& aux = *reinterpret_cast<Aux*>(t_ring + 2 * TAIL_B_BYTES);
    Barriers& bars = aux.bars;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int D = P.g.D;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NB; ++s) { mbar_init(&bars.b_full[s], 1); mbar_init(&bars.b_empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&bars.t_full[s], 1); mbar_init(&bars.t_empty[s], 1); }
        for (int s = 0; s < NA; ++s) { mbar_init(&bars.a_full[s], P.a_tma ? 1 : BUILD_WARPS / 2 * CG); mbar_init(&bars.a_empty[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&bars.acc_full[a], 1); mbar_init(&bars.acc_empty[a], EPI_WARPS * CG); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (D <= FOFF_MAX)
        for (int d = threadIdx.x; d < D; d += NUM_THREADS) aux.foff[d] = feat_off(P.g, d);
    if (threadIdx.x < TM) {
        write_tail_ones(a_tail, threadIdx.x);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (CG == 2) {                      // barriers of both CTAs initialised before anything arrives remotely
        __syncthreads();
        cluster_sync_all();
    }
    if (warp == 1) tmem_alloc<CG>(&bars.tmem_base, 512);
    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = bars.tmem_base;
    // a job = (patch tile [pair], feature split); CTA `rank` of a pair owns patch tile CG * (q / S) + rank
    const int SU = P.S * P.U;                       // jobs per patch tile [pair]: feature splits x unit splits
    const int n_jobs = ((P.n_mtiles + CG - 1) / CG) * SU;

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            int bs = 0, ts = 0;
            uint32_t b_ph = 0, t_ph = 0;
            // pair mode: both CTAs load their 128-unit half; only the leader arms its barrier, for both halves
            const int row_off = (int)rank * (TN / CG);
            int as = 0;
            uint32_t a_eph = 1;
            for (int q = job0; q < n_jobs; q += job_stride) {
                const int s = (q % SU) % P.S, u = (q % SU) / P.S;
                const int fb0 = s * P.fb_per_split;
                const int fb1 = min(P.DB, fb0 + P.fb_per_split);
                const int nt0 = u * P.nt_per_u, nt1 = min(P.NT, nt0 + P.nt_per_u);
                for (int n0 = nt0; n0 < nt1; n0 += NI) {
                    const int ni = min(NI, nt1 - n0);
                    if (s == 0) {
                        for (int a = 0; a < ni; ++a) {
                            const int n = n0 + a;
                            mbar_wait(&bars.t_empty[ts], t_ph ^ 1);
                            if (rank == 0) mbar_expect_tx(&bars.t_full[ts], TAIL_B_BYTES);
                            if (CG == 1) tma_load_2d(&map_t, &bars.t_full[ts], t_ring + ts * T_STAGE, 0, n * TN);
                            else tma_load_2d_pair(&map_t, &bars.t_full[ts], t_ring + ts * T_STAGE, 0, n * TN + row_off);
                            if (++ts == 2) { ts = 0; t_ph ^= 1; }
                        }
                    }
                    for (int fb = fb0; fb < fb1; ++fb) {
                        if (P.a_tma) {
                            // pre-split patch rows: hi and lo block of this CTA's tile into A slot `as`
                            const int m = CG * (q / SU) + (int)rank;
                            mbar_wait(&bars.a_empty[as], a_eph);
                            if (rank == 0) mbar_expect_tx(&bars.a_full[as], A_SLOT_BYTES * CG);
                            uint8_t* adst = a_ring + (size_t)as * A_SLOT_BYTES;
#pragma unroll
                            for (int part = 0; part < 2; ++part) {
                                if (CG == 1) tma_load_2d(&map_a, &bars.a_full[as], adst + part * A_BLK_BYTES,
                                                         (part * P.DB + fb) * KBLK, m * TM);
                                else tma_load_2d_pair(&map_a, &bars.a_full[as], adst + part * A_BLK_BYTES,
                                                      (part * P.DB + fb) * KBLK, m * TM);
                            }
                            if (++as == NA) { as = 0; a_eph ^= 1; }
                        }
                        for (int a = 0; a < ni; ++a) {
                            const int n = n0 + a;
#pragma unroll
                            for (int part = 0; part < 2; ++part) {      // hi block, then lo block
                                mbar_wait(&bars.b_empty[bs], b_ph ^ 1);
                                if (rank == 0) mbar_expect_tx(&bars.b_full[bs], B_BLK_BYTES);
                                uint8_t* dst = b_ring + (size_t)bs * B_STAGE;
                                if (CG == 1) tma_load_2d(&map_b, &bars.b_full[bs], dst, (part * P.DB + fb) * KBLK, n * TN);
                                else tma_load_2d_pair(&map_b, &bars.b_full[bs], dst, (part * P.DB + fb) * KBLK, n * TN + row_off);
                                if (++bs == NB) { bs = 0; b_ph ^= 1; }
                            }
                        }
                    }
                }
            }
        }
    } else if (warp == 1 && rank == 0) {
        // ================================ MMA issuer ==================================
        // warp-uniform control flow (operand descriptors stay in uniform registers); one elected lane issues.
        // Pair mode: only the leader CTA issues; its commits arrive on the barriers of both CTAs.
        const bool leader = elect_one();
        auto mma_wait = [&](uint64_t* bar, uint32_t parity) {
            if (CG == 2) mbar_wait_cluster(bar, parity); else mbar_wait(bar, parity);
        };
        const uint64_t adesc0 = umma_desc(smem_u32(a_ring));
        const uint64_t bdesc0 = umma_desc(smem_u32(b_ring));
        const uint64_t atdesc = umma_desc_sw32(smem_u32(a_tail));
        const uint64_t btdesc0 = umma_desc_sw32(smem_u32(t_ring));
        constexpr uint32_t A_SLOT_UNITS = (uint32_t)A_SLOT_BYTES >> 4;
        constexpr uint32_t A_LO_UNITS = (uint32_t)A_BLK_BYTES >> 4;
        constexpr uint32_t B_UNITS = (uint32_t)B_STAGE >> 4;
        constexpr uint32_t T_UNITS = (uint32_t)T_STAGE >> 4;
        int as = 0, bs = 0, ts = 0;
        uint32_t a_ph = 0, b_ph = 0, t_ph = 0, j = 0;
        for (int q = job0; q < n_jobs; q += job_stride) {
            if (ARES && q != job0) a_ph ^= 1;                      // resident slots: one fill per job
            const int s = (q % SU) % P.S, u = (q % SU) / P.S;
            const int fb0 = s * P.fb_per_split;
            const int fb1 = min(P.DB, fb0 + P.fb_per_split);
            const int nt0 = u * P.nt_per_u, nt1 = min(P.NT, nt0 + P.nt_per_u);
            for (int n0 = nt0; n0 < nt1; n0 += NI) {
                const int ni = min(NI, nt1 - n0);
                uint32_t accum[NI];
#pragma unroll
                for (int a = 0; a < NI; ++a) {
                    accum[a] = 0;
                    if (a < ni) mma_wait(&bars.acc_empty[(j + a) & 1u], (((j + a) >> 1) & 1u) ^ 1u);
                }
                tc_fence_after();
                if (s == 0) {
#pragma unroll
                    for (int a = 0; a < NI; ++a) {
                        if (a < ni) {
                            mma_wait(&bars.t_full[ts], t_ph);
                            tc_fence_after();
                            if (leader) {
                                tc_mma<MmaKind::TF32, CG>(tmem_base + ((j + a) & 1u) * TN, atdesc, btdesc0 + (uint32_t)ts * T_UNITS, 0u);
                                tc_commit<CG>(&bars.t_empty[ts]);
                            }
                            accum[a] = 1;
                            if (++ts == 2) { ts = 0; t_ph ^= 1; }
                        }
                    }
                }
                for (int fb = fb0; fb < fb1; ++fb) {
                    const int nks = (fb == P.DB - 1) ? P.nks_last : 4;
                    if (ARES) as = fb;
                    const uint64_t ahi = adesc0 + (uint32_t)as * A_SLOT_UNITS;
                    const uint64_t alo = ahi + A_LO_UNITS;
                    if (!ARES || n0 == nt0) mma_wait(&bars.a_full[as], a_ph);
#pragma unroll
                    for (int a = 0; a < NI; ++a) {
                        if (a < ni) {
                            const uint32_t d_addr = tmem_base + ((j + a) & 1u) * TN;
                            mma_wait(&bars.b_full[bs], b_ph);
                            tc_fence_after();
                            uint64_t bd = bdesc0 + (uint32_t)bs * B_UNITS;
                            if (leader) {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    if (k < nks) tc_mma<MmaKind::TF32, CG>(d_addr, ahi + 2u * k, bd + 2u * k, accum[a] | (uint32_t)(k > 0));
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    if (k < nks) tc_mma<MmaKind::TF32, CG>(d_addr, alo + 2u * k, bd + 2u * k, 1u);
                                tc_commit<CG>(&bars.b_empty[bs]);
                            }
                            accum[a] = 1;
                            if (++bs == NB) { bs = 0; b_ph ^= 1; }
                            mma_wait(&bars.b_full[bs], b_ph);
                            tc_fence_after();
                            bd = bdesc0 + (uint32_t)bs * B_UNITS;
                            if (leader) {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    if (k < nks) tc_mma<MmaKind::TF32, CG>(d_addr, ahi + 2u * k, bd + 2u * k, 1u);
                                tc_commit<CG>(&bars.b_empty[bs]);
                            }
                            if (++bs == NB) { bs = 0; b_ph ^= 1; }
                        }
                    }
                    if (leader && (!ARES || n0 + ni >= nt1)) tc_commit<CG>(&bars.a_empty[as]);
                    if (!ARES && ++as == NA) { as = 0; a_ph ^= 1; }
                }
                if (leader) {
#pragma unroll
                    for (int a = 0; a < NI; ++a)
                        if (a < ni) tc_commit<CG>(&bars.acc_full[(j + a) & 1u]);
                }
                j += (uint32_t)ni;
            }
        }
    } else if (warp >= BUILD_WARP0 && warp < BUILD_WARP0 + BUILD_WARPS) {
        // ================================ A builders ==================================
        // Two groups of four warps; group g converts every other feature block of this CTA's stream into
        // A-ring slot g.  A group's loads for its NEXT block are in flight while it waits for its slot and
        // converts the current one: two block times (~3000 MMA cycles) of latency tolerance per load.
        const int grp = (warp - BUILD_WARP0) >> 2;
        const int t = (threadIdx.x - BUILD_WARP0 * 32) & (TM - 1);     // patch row inside the tile
        const int vec = P.g.vec;
        const bool use_tab = D <= FOFF_MAX;
        // 32 features [32 fb, 32 fb + 32) of one patch row; zero beyond D and for padding rows
        // whole-fmap patches (Seq = 1, D % 32 == 0): a patch row is one contiguous run, so the warp reads full
        // 128-byte lines -- lane l takes chunk (l & 7) of rows wrow0 + 4 i + (l >> 3), i = 0..7 -- instead of
        // every lane walking its own row
        const bool contig = (P.g.seq == 1) && ((D & 31) == 0) && ((reinterpret_cast<uintptr_t>(P.x) & 15) == 0);
        const int wrow0 = t & ~31;                                     // first row of this warp
        int64_t m_rows0 = 0;                                           // first patch of the current job's tile
        auto load_fb = [&](float (&v)[32], const float* src, bool ok, int fb) {
            if (contig) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int64_t pr = m_rows0 + wrow0 + 4 * i + (lane >> 3);
                    float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (pr < P.rows && !(P.dbg & 1))
                        f = __ldg(reinterpret_cast<const float4*>(P.x + pr * D + fb * 32 + (lane & 7) * 4));
                    v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
                }
                return;
            }
            load_row(v, src, ok && !(P.dbg & 1), fb * 32, D, vec,
                     [&](int d) { return use_tab ? aux.foff[d] : feat_off(P.g, d); });
        };
        // position in this CTA's (job, unit tile, feature block) stream
        int q = job0, n = 0, fb = 0, fb0 = 0, fb1 = 0;
        bool ok = false, live = q < n_jobs;
        const float* src = P.x;
        auto enter_job = [&]() {
            const int s = (q % SU) % P.S, m = CG * (q / SU) + (int)rank;
            fb0 = s * P.fb_per_split;
            fb1 = min(P.DB, fb0 + P.fb_per_split);
            fb = fb0;
            n = 0;                           // (builders run in the resident and split-K modes; U > 1 excludes split-K)
            const int64_t p = (int64_t)m * TM + t;
            m_rows0 = (int64_t)m * TM;
            ok = p < P.rows;
            src = P.x + (ok ? patch_base(P.g, p) : 0);
        };
        auto advance = [&]() {
            if (!live) return;
            if (ARES) {                       // resident mode: this group's block of the next job
                q += job_stride;
                if (q >= n_jobs) { live = false; return; }
                enter_job();
                fb = grp;
                return;
            }
            if (++fb == fb1) {
                fb = fb0;
                if ((n += NI) >= P.NT) {
                    q += job_stride;
                    if (q >= n_jobs) { live = false; return; }
                    enter_job();
                }
            }
        };
        if (P.a_tma) live = false;
        if (live) enter_job();
        if (ARES) {
            fb = grp;
            if (grp >= P.DB) live = false;
        } else if (grp == 1) {
            advance();
        }
        uint32_t a_eph = 1;
        float cur[32], nxt[32];
        if (live) load_fb(cur, src, ok, fb);
        while (live) {
            advance();
            if (!ARES) advance();
            const bool more = live;
            if (more) load_fb(nxt, src, ok, fb);
            mbar_wait_warp<false>(&bars.a_empty[grp], a_eph, lane);
            uint8_t* hi_blk = a_ring + (size_t)grp * A_SLOT_BYTES;
            uint8_t* lo_blk = hi_blk + A_BLK_BYTES;
            if (!(P.dbg & 2))
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float4 hi, lo;
                tf32_split4(&cur[4 * c], hi, lo);
                // 16-byte chunk q of row r lives at r * 128 + ((q ^ (r & 7)) << 4)
                const uint32_t r = contig ? (uint32_t)(wrow0 + 4 * c + (lane >> 3)) : (uint32_t)t;
                const uint32_t qk = contig ? (uint32_t)(lane & 7) : (uint32_t)c;
                const uint32_t off = r * 128u + ((qk ^ (r & 7u)) << 4);
                *reinterpret_cast<float4*>(hi_blk + off) = hi;
                *reinterpret_cast<float4*>(lo_blk + off) = lo;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                if (CG == 2) mbar_arrive_remote(&bars.a_full[grp], 0);      // the leader's barrier counts both CTAs
                else mbar_arrive(&bars.a_full[grp]);
            }
            a_eph ^= 1;
            if (!more) break;
#pragma unroll
            for (int i = 0; i < 32; ++i) cur[i] = nxt[i];
        }
    } else if (warp >= EPI_WARP0) {
        // ================================ epilogue ====================================
        // four warps, one per TMEM lane quarter; a thread owns one patch row and walks all 256 columns
        const int lg = warp & 3;                    // TMEM lane quarter this warp may access
        const int row = lg * 32 + lane;             // patch row inside the tile
        uint32_t j = 0;
        for (int q = job0; q < n_jobs; q += job_stride) {
            const int s = (q % SU) % P.S, u = (q % SU) / P.S, m = CG * (q / SU) + (int)rank;
            const int nt0 = u * P.nt_per_u, nt1 = min(P.NT, nt0 + P.nt_per_u);
            const int64_t p = (int64_t)m * TM + row;
            float best = INFINITY;
            int bidx = nt0 * TN;
            for (int n = nt0; n < nt1; ++n) {
                const uint32_t acc = j & 1u;
                mbar_wait(&bars.acc_full[acc], (j >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(lg * 32) << 16) + acc * TN;
                const int col0 = n * TN;
                auto consume = [&](const uint32_t (&v)[32], int c) {
                    if (SPLITK) {
                        if (p < P.rows) {
                            float4* dst = reinterpret_cast<float4*>(
                                P.partial + ((int64_t)s * P.n_mtiles * TM + p) * P.K_pad + col0 + c * 32);
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                dst[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                                     __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
                        }
                    } else {
                        const float mn = min32(v);
                        if (mn < best) { best = mn; bidx = col0 + c * 32 + first_eq32(v, mn); }
                    }
                };
                tmem_drain<8>(taddr, consume, [&] {
                    if (lane == 0) {
                        if (CG == 2) mbar_arrive_remote_relaxed(&bars.acc_empty[acc], 0);
                        else mbar_arrive(&bars.acc_empty[acc]);
                    }
                });
                ++j;
            }
            if (!SPLITK && p < P.rows) {
                if (P.U > 1) {                       // unit split: candidates, merged by merge_kernel
                    P.cand_idx[(int64_t)u * P.rows + p] = (int64_t)bidx + P.unit_offset;
                    P.cand_rd[(int64_t)u * P.rows + p] = best;
                } else {
                    P.out_idx[p] = (int64_t)bidx + P.unit_offset;
                    if (P.out_rd) P.out_rd[p] = best;
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync_all();    // the peer may still multicast into / arrive on this CTA's shared memory
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<CG>(tmem_base, 512);
    }
}

// split-K tail: rd[p][j] = sum_s partial[s][p][j] in fixed order, then the argmin over the K real units
// (ascending j per lane + strict '<', ties between lanes to the lower index: lowest index wins)
__global__ void __launch_bounds__(256) splitk_argmin_kernel(const float* __restrict__ partial, int S, int64_t n_pad,
                                                            int K_pad, int K, int64_t rows, int64_t unit_offset,
                                                            int64_t* __restrict__ out_idx, float* __restrict__ out_rd) {
    const int64_t p = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= rows) return;
    float best = INFINITY;
    int bidx = 0x7fffffff;
    // 16-byte loads: lane l owns units 128 i + 4 l .. + 3 (K_pad is a multiple of 256, rows are 1 KB aligned), all S
    // partial rows of an iteration in flight; per lane the units are still visited in ascending order
    const float4* prow = reinterpret_cast<const float4*>(partial + p * K_pad);
    const int64_t sstride = n_pad * (int64_t)K_pad / 4;
    for (int j0 = 4 * lane; j0 < K; j0 += 128) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 t[MAX_SPLIT];
#pragma unroll
        for (int s = 0; s < MAX_SPLIT; ++s)
            if (s < S) t[s] = __ldcs(prow + (int64_t)s * sstride + (j0 >> 2));
#pragma unroll
        for (int s = 0; s < MAX_SPLIT; ++s)
            if (s < S) { acc.x += t[s].x; acc.y += t[s].y; acc.z += t[s].z; acc.w += t[s].w; }
        if (acc.x < best) { best = acc.x; bidx = j0; }
        if (j0 + 1 < K && acc.y < best) { best = acc.y; bidx = j0 + 1; }
        if (j0 + 2 < K && acc.z < best) { best = acc.z; bidx = j0 + 2; }
        if (j0 + 3 < K && acc.w < best) { best = acc.w; bidx = j0 + 3; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        argmin_merge(best, bidx, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bidx, o));
    }
    if (lane == 0) {
        // a non-finite patch row makes every sum NaN and no '<' fires: unit 0 of the shard, as torch.argmin over an
        // all-NaN distance row does (models/Codebook.py:91-94) and as the other modes' "best = inf, index 0" start does
        if (bidx == 0x7fffffff) bidx = 0;
        out_idx[p] = (int64_t)bidx + unit_offset;
        if (out_rd) out_rd[p] = best;
    }
}

// pre-split codebook: row j = [ -2 hi(c) for every 32-feature block | -2 lo(c) for every block ], zero beyond D;
// tail rows [n1 n2 n3 0 0 0 0 0]; rows >= K are padding units whose norm can never be the minimum
__global__ void __launch_bounds__(256) split_w_l_kernel(const float* __restrict__ W, const float* __restrict__ cn,
                                                        int K, int D, int DB, int K_pad, float* __restrict__ Bp,
                                                        float* __restrict__ Tp) {
    const int64_t cols = (int64_t)DB * 32;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= (int64_t)K_pad * cols) return;
    const int row = (int)(t / cols);
    const int d = (int)(t - (int64_t)row * cols);
    float hi = 0.f, lo = 0.f;
    if (row < K && d < D) {
        tf32_split(W[(int64_t)row * D + d], hi, lo);
        hi *= -2.0f;
        lo *= -2.0f;
    }
    Bp[(int64_t)row * 2 * cols + d] = hi;
    Bp[(int64_t)row * 2 * cols + cols + d] = lo;
    if (d < 8) {
        float out = 0.f;
        if (row < K) {
            float n1, n2, n3;
            tf32_norm_split3(cn[row], n1, n2, n3);
            out = (d == 0) ? n1 : (d == 1) ? n2 : (d == 2) ? n3 : 0.f;
        } else if (d == 0) {
            out = PAD_NORM;
        }
        Tp[(int64_t)row * 8 + d] = out;
    }
}

// CTA pairs (cta_group::2).  Static rule: pairs when there is no feature split and at least two waves of patch
// tiles (measured: C4 7.44 -> 7.23 ms, C5 64.1 -> 62.1 ms; split-K shapes are faster unpaired).
// Experiment builds (-DSOM_TC_EXPERIMENTS) read SOM_TC_PAIR=0 / 1 to force the choice for A/B runs.
static int pair_mode() {
#ifdef SOM_TC_EXPERIMENTS
    static int mode = -2;
    if (mode == -2) { const char* e = getenv("SOM_TC_PAIR"); mode = e ? atoi(e) : -1; }
    return mode;
#else
    return -1;
#endif
}

// streamed mode pre-pass: patch rows p0 .. p0+rows-1 -> [ hi(x) for every 32-feature block | lo(x) for every block ],
// zero beyond D; patchify fused as address arithmetic.  One thread per (patch, 4-feature group).
__global__ void __launch_bounds__(256) split_x_l_kernel(const float* __restrict__ x, Geom g, int64_t p0, int64_t rows,
                                                        int DB, float* __restrict__ Ap) {
    const int groups = DB * 8;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= rows * groups) return;
    const int64_t pr = t / groups;
    const int d0 = (int)(t - pr * groups) * 4;
    const float* src = x + patch_base(g, p0 + pr);
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (g.vec == 4 && d0 + 3 < g.D) {
        const float4 f = __ldg(reinterpret_cast<const float4*>(src + feat_off(g, d0)));
        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (d0 + e < g.D) v[e] = __ldg(src + feat_off(g, d0 + e));
    }
    float4 hi, lo;
    tf32_split4(v, hi, lo);
    float* dst = Ap + pr * (int64_t)DB * 64 + d0;
    *reinterpret_cast<float4*>(dst) = hi;
    *reinterpret_cast<float4*>(dst + (int64_t)DB * 32) = lo;
}

struct Plan {
    int cg;
    int D, K, DB, nks_last, K_pad, NT, n_mtiles, S, fb_per_split, U, nt_per_u;
    int64_t chunk_rows;            // streamed mode: patches per pre-split workspace chunk (multiple of 128)
    size_t off_b, off_t, off_p, off_a, off_c, total;
};

static void make_plan(Plan* pl, int64_t n, int D, int K) {
    pl->D = D; pl->K = K;
    pl->DB = (D + 31) / 32;
    pl->nks_last = (D - 32 * (pl->DB - 1) + 7) / 8;
    pl->K_pad = (K + TN - 1) / TN * TN;
    pl->NT = pl->K_pad / TN;
    pl->n_mtiles = (int)ceil_div64(n, TM);
    // static split rule: with fewer patch tiles than SMs, cut the feature axis so that every SM gets a job,
    // but keep at least 8 blocks (~12k MMA cycles) per split (finer splits lose to the partial-distance traffic:
    // D = 256 with 2-block splits measured 105 us against 71 us unsplit)
    int S = sm_count() / pl->n_mtiles;
    if (S > pl->DB / 8) S = pl->DB / 8;
    if (S > MAX_SPLIT) S = MAX_SPLIT;
    // the S x N x K partial-distance buffer is written and re-read through HBM on every call: keep it within 256 MB
    // (K = 32 768, D = 512, 9.4k patches would otherwise take 2.5 GB); beyond that the unit-split / streamed modes apply
    while (S > 1 && (size_t)S * pl->n_mtiles * TM * (size_t)pl->K_pad * 4 > ((size_t)256 << 20)) --S;
    if (S < 1) S = 1;
    pl->fb_per_split = (pl->DB + S - 1) / S;
    pl->S = (pl->DB + pl->fb_per_split - 1) / pl->fb_per_split;
    // few patch tiles and many unit tiles (no feature split): spread the unit tiles of a patch tile over U CTAs
    // (each builds / streams its own copy of the A tile) and merge the U candidates per patch afterwards
    pl->U = 1;
    pl->nt_per_u = pl->NT;
    if (pl->S == 1 && 2 * pl->n_mtiles <= sm_count() && pl->NT >= 8) {
        int U = sm_count() / pl->n_mtiles;
        if (U > pl->NT / 2) U = pl->NT / 2;
        if (U > 16) U = 16;
        if (U > 1) {
            pl->nt_per_u = (pl->NT + U - 1) / U;
            pl->U = (pl->NT + pl->nt_per_u - 1) / pl->nt_per_u;
        }
    }
    pl->cg = 1;
    if (sm_count() % 2 == 0 && pair_mode() != 0 && pl->U == 1) {
        if (pair_mode() == 1) pl->cg = 2;
        else if (pl->S == 1 && pl->n_mtiles >= 2 * sm_count()) pl->cg = 2;
    }
    size_t o = 0;
    pl->off_b = o; o = align_up(o + (size_t)pl->K_pad * pl->DB * 64 * 4, 1024);
    pl->off_t = o; o = align_up(o + (size_t)pl->K_pad * 8 * 4, 1024);
    pl->off_p = o;
    if (pl->S > 1) o = align_up(o + (size_t)pl->S * pl->n_mtiles * TM * pl->K_pad * 4, 1024);
    pl->off_a = o;
    pl->chunk_rows = 0;
    if (pl->S == 1 && pl->DB > NA) {
        // streamed mode: pre-split patch rows, chunked so that a chunk (~48 MB) stays L2 resident between the
        // pre-pass and the GEMM kernel; whole waves of patch tiles per chunk
        const int64_t row_bytes = (int64_t)pl->DB * 64 * 4;
        const int64_t wave_rows = (int64_t)TM * sm_count();
        int64_t max_rows = (48ll << 20) / row_bytes;
        int64_t chunk = max_rows / wave_rows * wave_rows;
        if (chunk < TM) chunk = (max_rows / TM > 0 ? max_rows / TM : 1) * TM;
        const int64_t need = ceil_div64(n, TM) * TM;
        if (chunk > need) chunk = need;
        if (pl->U > 1 && chunk < need) { pl->U = 1; pl->nt_per_u = pl->NT; }     // unit splits need a single chunk
        pl->chunk_rows = chunk;
        o = align_up(o + (size_t)chunk * row_bytes, 1024);
    }
    pl->off_c = o;
    if (pl->U > 1) o = align_up(o + (size_t)pl->U * n * (4 + 8), 1024);
    pl->total = o;
}

// 0 split-K, 1 resident-A, 2 streamed
static int plan_mode(const Plan& pl) { return pl.S > 1 ? 0 : (pl.DB <= NA ? 1 : 2); }

}  // namespace tcl

size_t tc_l_workspace_bytes(int64_t n_patches, int D, int K) {
    tcl::Plan pl;
    tcl::make_plan(&pl, n_patches, D, K);
    return pl.total;
}

// the plan of launch_bmu_tc_l for som_debug_bmu_plan (f: PF_COUNT fields, pre-filled with -1)
void tc_l_plan_fields(int64_t n_patches, int D, int K, int64_t* f) {
    tcl::Plan pl;
    tcl::make_plan(&pl, n_patches, D, K);
    f[PF_CG] = pl.cg;
    f[PF_MODE] = tcl::plan_mode(pl);
    f[PF_S] = pl.S;
    f[PF_FB_PER_SPLIT] = pl.fb_per_split;
    f[PF_U] = pl.U;
    f[PF_CHUNK_ROWS] = pl.chunk_rows;
    f[PF_NT] = pl.NT;
    f[PF_DB] = pl.DB;
    f[PF_MTILES] = pl.n_mtiles;
}

int launch_bmu_tc_l(const float* x, const Geom& g, const float* W, const float* cn, int K, int64_t unit_offset,
                    int64_t* out_idx, float* out_rd, void* ws, size_t ws_bytes, cudaStream_t st) {
    using namespace tcl;
    const int64_t n = g.n_patches;
    if (n == 0) return SOM_OK;
    Plan pl;
    make_plan(&pl, n, g.D, K);
    int rc = check_workspace(ws, ws_bytes, pl.total, "bmu(tc)");
    if (rc) return rc;
    float* Bp = (float*)((char*)ws + pl.off_b);
    float* Tp = (float*)((char*)ws + pl.off_t);
    float* Pp = (float*)((char*)ws + pl.off_p);
    {
        const int64_t items = (int64_t)pl.K_pad * pl.DB * 32;
        split_w_l_kernel<<<(unsigned)ceil_div64(items, 256), 256, 0, st>>>(W, cn, K, g.D, pl.DB, pl.K_pad, Bp, Tp);
        rc = check_launch("split_w_l_kernel");
        if (rc) return rc;
    }
    CUtensorMap map_b, map_t, map_a;
    const uint32_t box_rows = TN / pl.cg;
    rc = make_map2d(&map_b, Bp, (uint64_t)pl.K_pad, (uint64_t)pl.DB * 64, (uint64_t)pl.DB * 64 * 4, 32, box_rows,
                        CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_map2d(&map_t, Tp, (uint64_t)pl.K_pad, 8, 32, 8, box_rows, CU_TENSOR_MAP_SWIZZLE_32B);
    if (rc) return rc;
    const int mode = plan_mode(pl);
    float* Ap = (float*)((char*)ws + pl.off_a);
    map_a = map_b;                                                   // unused unless streamed
    if (mode == 2) {
        rc = make_map2d(&map_a, Ap, (uint64_t)pl.chunk_rows, (uint64_t)pl.DB * 64, (uint64_t)pl.DB * 64 * 4, 32, TM,
                        CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
    }

    Params P;
    P.DB = pl.DB; P.nks_last = pl.nks_last; P.NT = pl.NT; P.n_mtiles = pl.n_mtiles; P.S = pl.S;
    P.fb_per_split = pl.fb_per_split; P.K_pad = pl.K_pad; P.rows = n; P.unit_offset = unit_offset;
    P.U = pl.U; P.nt_per_u = pl.nt_per_u;
    P.cand_idx = (int64_t*)((char*)ws + pl.off_c);                      // int64 first: 8-byte aligned
    P.cand_rd = (float*)((char*)ws + pl.off_c + (size_t)pl.U * n * 8);
    P.out_idx = out_idx; P.out_rd = out_rd; P.partial = pl.S > 1 ? Pp : nullptr; P.x = x; P.g = g;
    P.a_tma = (mode == 2) ? 1 : 0; P.tile0 = 0;
    P.dbg = 0;
#ifdef SOM_TC_EXPERIMENTS
    // timing-elimination switches (skip refine / loads / conversion): results are wrong, experiment builds only
    { static int dbg = -1; if (dbg < 0) { const char* e = getenv("SOM_TC_DEBUG"); dbg = e ? atoi(e) : 0; } P.dbg = dbg; }
#endif

    typedef void (*KernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const Params);
    static const KernelFn kernels[2][3] = {
        {bmu_tc_l_kernel<true, false, 1>, bmu_tc_l_kernel<false, true, 1>, bmu_tc_l_kernel<false, false, 1>},
        {bmu_tc_l_kernel<true, false, 2>, bmu_tc_l_kernel<false, true, 2>, bmu_tc_l_kernel<false, false, 2>}};
    static const char* names[3] = {"bmu_tc_l_kernel<splitk>", "bmu_tc_l_kernel<resident>", "bmu_tc_l_kernel<streamed>"};
    static PerDeviceFlag attr_done;
    rc = smem_opt_in(attr_done, &kernels[0][0], 6, (int)SMEM_BYTES, "bmu(tc)");
    if (rc) return rc;
    auto launch = [&](const Params& Pl) -> int {
        const int n_jobs = ((Pl.n_mtiles + pl.cg - 1) / pl.cg) * pl.S * pl.U;
        const int max_groups = sm_count() / pl.cg;
        const int groups = n_jobs < max_groups ? n_jobs : max_groups;
        // a cluster of cg CTAs, no PDL
        cudaError_t le = launch_kernel(kernels[pl.cg - 1][mode], (unsigned)(groups * pl.cg), NUM_THREADS, SMEM_BYTES, st,
                                       (unsigned)pl.cg, false, map_b, map_t, map_a, Pl);
        if (le != cudaSuccess) { set_error("%s: launch: %s", names[mode], cudaGetErrorString(le)); return (int)le; }
        return check_launch(names[mode]);
    };
    if (mode == 2) {
        for (int64_t p0 = 0; p0 < n; p0 += pl.chunk_rows) {
            const int64_t rows = (n - p0 < pl.chunk_rows) ? n - p0 : pl.chunk_rows;
            const int64_t items = rows * pl.DB * 8;
            split_x_l_kernel<<<(unsigned)ceil_div64(items, 256), 256, 0, st>>>(x, g, p0, rows, pl.DB, Ap);
            rc = check_launch("split_x_l_kernel");
            if (rc) return rc;
            Params Pc = P;
            Pc.rows = rows;
            Pc.n_mtiles = (int)ceil_div64(rows, TM);
            Pc.out_idx = out_idx + p0;
            Pc.out_rd = out_rd ? out_rd + p0 : nullptr;
            rc = launch(Pc);
            if (rc) return rc;
        }
        if (pl.U > 1)       // few patch tiles: one chunk (make_plan), candidates of the unit splits merged here
            return som_merge_candidates(P.cand_rd, P.cand_idx, pl.U, n, out_idx, out_rd, st);
        return SOM_OK;
    }
    rc = launch(P);
    if (rc) return rc;
    if (pl.U > 1)
        return som_merge_candidates(P.cand_rd, P.cand_idx, pl.U, n, out_idx, out_rd, st);
    if (pl.S > 1) {
        splitk_argmin_kernel<<<(unsigned)ceil_div64(n, 8), 256, 0, st>>>(Pp, pl.S, (int64_t)pl.n_mtiles * TM, pl.K_pad, K,
                                                                       n, unit_offset, out_idx, out_rd);
        return check_launch("splitk_argmin_kernel");
    }
    return SOM_OK;
}

}  // namespace som
