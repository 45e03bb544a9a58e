// K1 (tensor-core variant), 16 < D <= 256, large batches: BMU search as an error-compensated FP16-split GEMM on
// tcgen05 (kind::f16).  sm_100a only.
//
// Replaces patchify + torch.cdist + torch.argmin of Codebook.get_patches_bmu
// (/root/reference/models/Codebook.py:77-99) at BASELINE config 4 (D = 64, K = 16 384: 93 % of a training step) and
// config 5 (D = 256, K = 32 768 per GPU).  Same mathematics as the 3xTF32 kernels of som_bmu_tc_l.cu,
//     rd[p][j] = ||c_j||^2 - 2 x_p . c_j = n1+n2+n3 - 2 x_hi.c_hi - 2 x_lo.c_hi - 2 x_hi.c_lo,
// but hi / lo are FP16 (hi = fp16(v), lo = fp16(v - hi): 11 + 11 mantissa bits, as the TF32 split) and a
// kind::f16 MMA has K = 16 at the cycle cost of a K = 8 TF32 MMA: a 128 x 256 tile of D = 64 costs 13 MMAs (1664
// tensor-pipe cycles) instead of 25.  FP16's exponent range is covered by EXACT power-of-two scales (the scheme of
// config S, som_bmu_tc_s.cu): per patch s_p (max |s_p x| in [64, 128), computed by the builder from the row it
// holds), per codebook s_c (from max ||c||, so that max |s_c c| < 256) and, for the norm column, t_c
// (max t_c s_c ||c||^2 in [2^14, 2^15)).  The accumulator then holds s_p s_c rd -- a positive factor per row that the
// argmin over units does not see -- and the returned reduced distance is un-scaled exactly.
//     A block (64 features) = [ hi(s_p x) ] 16 KB + [ lo(s_p x) ] 16 KB, 128-byte SWIZZLE_128B rows of 64 halves
//     B block (64 features) = [ hi(-2 s_c c) ] 32 KB, [ lo(-2 s_c c) ] 32 KB (two ring stages)
//     tail k-step           : A = [a_p a_p a_p 0..] (a_p = s_p / t_c), B = [n1 n2 n3 0..] of t_c s_c ||c||^2
//                             (16 halves = 32-byte rows, SWIZZLE_32B)
// The patch tile stays RESIDENT in shared memory for all unit tiles (D <= 128: two 32 KB slots used as a ring over
// jobs, so the next tile is built while the current one is searched; D <= 256: four slots, one tile).
//
// One persistent CTA per SM -- or a CTA pair (cta_group::2: each CTA holds its own patch tile and HALF of every B
// block, the leader issues M256 MMAs) -- 448 threads, warp-specialised:
//   warp 0      TMA producer: B_hi / B_lo blocks and norm tails of the pre-split codebook
//   warp 1      MMA issuer  : warp-uniform loop, one elected lane issues M128 (M256) x N256 x K16 kind::f16 into two
//                             TMEM accumulator stages
//   warps 2-5   builders    : a thread reads its patch row straight from NCHW (patchify = address arithmetic),
//                             derives the row scale, splits hi / lo and writes the swizzled operand blocks + its
//                             tail row -- no operand copy in HBM
//   warps 6-13  epilogue    : tcgen05.ld of their TMEM lane quarter / column half, exact running (min, index) per
//                             patch row; the N x K distance matrix never leaves TMEM
// Bound: tensor pipe (FP16 rate / 3).
//
// 16-bit input (T = __half, som_bmu_stage_nchw_f16; T = __nv_bfloat16, som_bmu_stage_nchw_bf16): the builders read
// the 16-bit values and widen them exactly, so everything from the row scale on sees the values x.float() would
// give.  Where s_p x is itself exact in FP16, lo(s_p x) is zero: every builder warp reports whether any lo of its rows
// in a 64-feature block is non-zero, and the issuer drops the A_lo x B_hi group of that block when none is (9 instead
// of 13 MMAs per tile at D = 64).  The dropped products are exact zeros; the fp32 instantiation never reads the flag
// and keeps its MMA sequence.
//   fp16 : s_p x is exact whenever the row scale is at least 1 (row max below 128) and no clamp lowered it: such
//          fp16 tiles never keep the third product.
//   bf16 : an 8-bit significand, but fp32's exponent range.  With max |s_p x| in [64, 128) an element is exact in
//          FP16 when its scaled exponent is at least -17 (its last significand bit then sits on FP16's 2^-24 grid),
//          i.e. when it lies within about 2^-23 of its row's largest magnitude, and no clamp lowered the row scale.
//          Tanh-range latents almost always pass.  So a bf16 tile MAY keep the third product where an fp16 tile of
//          the same row maxima never does (an element further below its row max, a bf16 subnormal); the flag keeps
//          it then, and the result stays exact.
#include "som_common.cuh"
#include "som_tc_ptx.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace som {
SOM_TRACE_TU(trace_set_l16)
namespace tcl16 {
using namespace tc;

constexpr int NA_MAX = 4;                    // A slots (hi + lo block of 64 features)
constexpr int NB_MAX = 8;
constexpr int BUILD_WARP0 = 2, BUILD_WARPS = 4;
constexpr int EPI_WARP0 = 6, EPI_WARPS = 8;
constexpr int NUM_THREADS = (EPI_WARP0 + EPI_WARPS) * 32;       // 448
constexpr int A_SLOT_BYTES = 2 * A_BLK_BYTES;                   // 32 KB
constexpr int TAIL_A_BYTES = TM * 32;        // 4 KB
constexpr int TAIL_B_BYTES = TN * 32;        // 8 KB
constexpr int DMAX = 256;
constexpr int RING_BYTES = 192 * 1024;       // A slots + B stages
constexpr int TILES_BYTES = RING_BYTES + 2 * TAIL_A_BYTES + 2 * TAIL_B_BYTES;   // 216 KB

struct Params {
    int DB;                 // 64-feature blocks (1..4)
    int nks_last;           // K = 16 steps of the last block
    int NT;                 // unit tiles
    int n_mtiles;           // patch tiles
    int NA, NB;             // A slots, B ring stages (of B_BLK_BYTES / CG)
    int K_pad;
    int64_t rows;           // valid patches
    int64_t unit_offset;
    int64_t* out_idx;
    float* out_rd;
    const void* x;          // float, __half or __nv_bfloat16, per the kernel's T
    Geom g;
    const float* scale;     // [s_c, t_c] written by cb_scale_l_kernel earlier on the stream
    float* stage;           // optional patch-major copy of the patch rows (n_patches x D), written by the builders
};

struct __align__(8) Barriers {
    uint64_t b_full[NB_MAX], b_empty[NB_MAX];
    uint64_t t_full[2], t_empty[2];
    uint64_t a_full[NA_MAX], a_empty[NA_MAX];
    uint64_t acc_full[2], acc_empty[2];
    uint64_t exp_full[2];
    uint32_t tmem_base, pad;
};
struct Aux {
    Barriers bars;
    int foff[DMAX];
    float mrg_val[2][TM];
    int mrg_idx[2][TM];
    int row_exp[2][TM];
    // 16-bit input: per A slot one byte per builder warp (CG x 4, all in the leader CTA): "a lo of my rows is non-zero"
    alignas(8) uint8_t lo_nz[NA_MAX][8];
};
constexpr uint32_t SMEM_BYTES = 1024 + TILES_BYTES + sizeof(Aux);

__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46) |
           (6ull << 61);
}

// eight halves (one 16-byte swizzle chunk) from eight floats, round-to-nearest-even
__device__ __forceinline__ uint4 pack_h8(float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7) {
    __half2 a = __floats2half2_rn(v0, v1), b = __floats2half2_rn(v2, v3);
    __half2 c = __floats2half2_rn(v4, v5), d = __floats2half2_rn(v6, v7);
    return make_uint4(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b),
                      *reinterpret_cast<uint32_t*>(&c), *reinterpret_cast<uint32_t*>(&d));
}

__device__ long long g_prof16[8];             // CTA 0's MMA loop: cycles, tiles, cycles waiting (acc_empty, B, A)

// MERGED (D <= 128): one ring stage carries everything a unit tile needs of one 64-feature block -- B_hi, B_lo and
// (block 0) the norm tail -- so the issuing thread pays ONE barrier wait and ONE commit per block instead of three.
// With 13 MMAs per tile the issuing thread, not the tensor pipe, sets the pace otherwise (~48 cycles per MMA issue,
// ~100 per barrier check, ~120 per commit).
// exact fp32 values of 4 / 2 / 1 consecutive input elements (float, __half or __nv_bfloat16)
__device__ __forceinline__ void ld4(const float* p, float* o) {
    const float4 f = __ldg(reinterpret_cast<const float4*>(p));
    o[0] = f.x; o[1] = f.y; o[2] = f.z; o[3] = f.w;
}
__device__ __forceinline__ void ld4(const __half* p, float* o) {
    const uint2 r = __ldg(reinterpret_cast<const uint2*>(p));
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
}
__device__ __forceinline__ void ld2(const float* p, float* o) {
    const float2 f = __ldg(reinterpret_cast<const float2*>(p));
    o[0] = f.x; o[1] = f.y;
}
__device__ __forceinline__ void ld2(const __half* p, float* o) {
    const float2 f = __half22float2(__ldg(reinterpret_cast<const __half2*>(p)));
    o[0] = f.x; o[1] = f.y;
}
__device__ __forceinline__ float ld1(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld1(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ void ld4(const __nv_bfloat16* p, float* o) {
    const uint2 r = __ldg(reinterpret_cast<const uint2*>(p));
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.y));
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
}
__device__ __forceinline__ void ld2(const __nv_bfloat16* p, float* o) {
    const float2 f = __bfloat1622float2(__ldg(reinterpret_cast<const __nv_bfloat162*>(p)));
    o[0] = f.x; o[1] = f.y;
}
__device__ __forceinline__ float ld1(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }

template <int CG, bool MERGED, typename T>
__global__ void __launch_bounds__(NUM_THREADS, 1)
bmu_tc_l16_kernel(const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_t, const Params P) {
    constexpr bool IN16 = sizeof(T) == 2;          // a 16-bit input type (__half or __nv_bfloat16)
    pdl_launch_dependents();            // (the wait on the operand-split kernel comes after the barrier / TMEM prologue)
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment as an OFFSET into the shared array: rounding the pointer through uintptr_t made the compiler
    // forget the address space, and every access below compiled to generic LD.E / ST.E (cuobjdump, round 2)
    uint8_t* tiles = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    constexpr int B_STAGE = B_BLK_BYTES / CG;       // this CTA's share of a 256-unit block
    constexpr int T_STAGE = TAIL_B_BYTES / CG;
    constexpr int M_STAGE = 2 * B_STAGE + T_STAGE;  // merged stage: [hi | lo | tail]
    const int NA = P.NA, NB = P.NB, DB = P.DB;
    // separate rings : [A slots | B stages ........ | A tails | B tail stages]
    // merged stages  : [A slots (2) | A tails | merged stages ....................]
    uint8_t* a_ring = tiles;
    uint8_t* a_tail = MERGED ? tiles + 2 * A_SLOT_BYTES : tiles + RING_BYTES;
    uint8_t* b_ring = MERGED ? a_tail + 2 * TAIL_A_BYTES : a_ring + (size_t)NA * A_SLOT_BYTES;
    uint8_t* t_ring = a_tail + 2 * TAIL_A_BYTES;    // (separate rings only)
    Aux& aux = *reinterpret_cast<Aux*>(tiles + TILES_BYTES);
    Barriers& bars = aux.bars;
    const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;
    const int job0 = (CG == 2) ? (int)cluster_id_x() : (int)blockIdx.x;
    const int job_stride = (CG == 2) ? (int)cluster_count_x() : (int)gridDim.x;
    const int n_jobs = (P.n_mtiles + CG - 1) / CG;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int D = P.g.D;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NB_MAX; ++s) { mbar_init(&bars.b_full[s], 1); mbar_init(&bars.b_empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&bars.t_full[s], 1); mbar_init(&bars.t_empty[s], 1); }
        for (int s = 0; s < NA_MAX; ++s) { mbar_init(&bars.a_full[s], BUILD_WARPS * CG); mbar_init(&bars.a_empty[s], 1); }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bars.acc_full[a], 1);
            mbar_init(&bars.acc_empty[a], EPI_WARPS * CG);
            mbar_init(&bars.exp_full[a], BUILD_WARPS);
        }
        if (IN16)
            for (int s = 0; s < NA_MAX; ++s) *reinterpret_cast<uint64_t*>(aux.lo_nz[s]) = 0ull;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int d = threadIdx.x; d < D; d += NUM_THREADS) aux.foff[d] = feat_off(P.g, d);
    if (CG == 2) {                      // barriers of both CTAs initialised before anything arrives remotely
        __syncthreads();
        cluster_sync_all();
    }
    if (warp == 1) {
        if (CG == 1) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars.tmem_base)),
                         "r"(512));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars.tmem_base)),
                         "r"(512));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = bars.tmem_base;
    pdl_wait();
    trace_stamp(s_trace_buf, 7);

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            int bs = 0, ts = 0;
            uint32_t b_ph = 0, t_ph = 0;
            // pair mode: both CTAs load their 128-unit half; only the leader arms its barrier, for both halves
            const int row_off = (int)rank * (TN / CG);
            for (int q = job0; q < n_jobs; q += job_stride) {
                for (int n = 0; n < P.NT; ++n) {
                    if (MERGED) {
                        for (int fb = 0; fb < DB; ++fb) {
                            mbar_wait(&bars.b_empty[bs], b_ph ^ 1);
                            if (rank == 0) mbar_expect_tx(&bars.b_full[bs], 2 * B_BLK_BYTES + (fb == 0 ? TAIL_B_BYTES : 0));
                            uint8_t* dst = b_ring + (size_t)bs * M_STAGE;
#pragma unroll
                            for (int part = 0; part < 2; ++part) {
                                if (CG == 1) tma_load_2d(&map_b, &bars.b_full[bs], dst + part * B_STAGE, (part * DB + fb) * KBLK, n * TN);
                                else tma_load_2d_pair(&map_b, &bars.b_full[bs], dst + part * B_STAGE, (part * DB + fb) * KBLK, n * TN + row_off);
                            }
                            if (fb == 0) {
                                if (CG == 1) tma_load_2d(&map_t, &bars.b_full[bs], dst + 2 * B_STAGE, 0, n * TN);
                                else tma_load_2d_pair(&map_t, &bars.b_full[bs], dst + 2 * B_STAGE, 0, n * TN + row_off);
                            }
                            if (++bs == NB) { bs = 0; b_ph ^= 1; }
                        }
                        continue;
                    }
                    mbar_wait(&bars.t_empty[ts], t_ph ^ 1);
                    if (rank == 0) mbar_expect_tx(&bars.t_full[ts], TAIL_B_BYTES);
                    if (CG == 1) tma_load_2d(&map_t, &bars.t_full[ts], t_ring + ts * T_STAGE, 0, n * TN);
                    else tma_load_2d_pair(&map_t, &bars.t_full[ts], t_ring + ts * T_STAGE, 0, n * TN + row_off);
                    if (++ts == 2) { ts = 0; t_ph ^= 1; }
                    for (int fb = 0; fb < DB; ++fb) {
#pragma unroll
                        for (int part = 0; part < 2; ++part) {      // hi block, then lo block
                            mbar_wait(&bars.b_empty[bs], b_ph ^ 1);
                            if (rank == 0) mbar_expect_tx(&bars.b_full[bs], B_BLK_BYTES);
                            uint8_t* dst = b_ring + (size_t)bs * B_STAGE;
                            if (CG == 1) tma_load_2d(&map_b, &bars.b_full[bs], dst, (part * DB + fb) * KBLK, n * TN);
                            else tma_load_2d_pair(&map_b, &bars.b_full[bs], dst, (part * DB + fb) * KBLK, n * TN + row_off);
                            if (++bs == NB) { bs = 0; b_ph ^= 1; }
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
        const uint64_t atdesc0 = umma_desc_sw32(smem_u32(a_tail));
        const uint64_t btdesc0 = umma_desc_sw32(smem_u32(t_ring));
        constexpr uint32_t A_SLOT_UNITS = (uint32_t)A_SLOT_BYTES >> 4;
        constexpr uint32_t A_LO_UNITS = (uint32_t)A_BLK_BYTES >> 4;
        constexpr uint32_t B_UNITS = (uint32_t)B_STAGE >> 4;
        constexpr uint32_t T_UNITS = (uint32_t)T_STAGE >> 4;
        constexpr uint32_t TA_UNITS = (uint32_t)TAIL_A_BYTES >> 4;
        constexpr uint32_t M_UNITS = (uint32_t)M_STAGE >> 4;
        int bs = 0, ts = 0;
        uint32_t b_ph = 0, t_ph = 0, j = 0;
        int i = 0;
        const bool prof = blockIdx.x == 0;
        long long w_acc = 0, w_b = 0, w_a = 0;
        const long long t_begin = clock64();
        // IN16: bit fb set = block fb of this job's patch tile has a non-zero lo (read once per job, at n == 0)
        auto lo_flag = [&](int as) -> uint32_t {
            return *reinterpret_cast<volatile uint64_t*>(aux.lo_nz[as]) != 0ull ? 1u : 0u;
        };
        for (int q = job0; q < n_jobs; q += job_stride, ++i) {
            uint32_t lo_mask = 0xFu;
            for (int n = 0; n < P.NT; ++n) {
                long long c0 = prof ? clock64() : 0;
                mma_wait(&bars.acc_empty[j & 1u], ((j >> 1) & 1u) ^ 1u);
                if (prof) w_acc += clock64() - c0;
                const uint32_t d_addr = tmem_base + (j & 1u) * TN;
                if (MERGED) {
                    for (int fb = 0; fb < DB; ++fb) {
                        const int nks = (fb == DB - 1) ? P.nks_last : 4;
                        const int u = i * DB + fb;
                        const int as = u % NA;
                        if (n == 0) {
                            c0 = prof ? clock64() : 0;
                            mma_wait(&bars.a_full[as], (uint32_t)(u / NA) & 1u);
                            if (prof) w_a += clock64() - c0;
                            if (IN16) lo_mask = (lo_mask & ~(1u << fb)) | (lo_flag(as) << fb);
                        }
                        const uint64_t ahi = adesc0 + (uint32_t)as * A_SLOT_UNITS;
                        const uint64_t alo = ahi + A_LO_UNITS;
                        c0 = prof ? clock64() : 0;
                        mma_wait(&bars.b_full[bs], b_ph);
                        if (prof) w_b += clock64() - c0;
                        tc_fence_after();
                        const uint64_t bhi = bdesc0 + (uint32_t)bs * M_UNITS;
                        const uint64_t blo = bhi + B_UNITS;
                        if (leader) {
                            if (fb == 0)
                                tc_mma_f16_cg<CG>(d_addr, atdesc0 + (uint32_t)(i & 1) * TA_UNITS,
                                                  umma_desc_sw32(smem_u32(b_ring + (size_t)bs * M_STAGE + 2 * B_STAGE)), 0u);
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                if (k < nks) tc_mma_f16_cg<CG>(d_addr, ahi + 2u * k, bhi + 2u * k, 1u);
                            if (!IN16 || ((lo_mask >> fb) & 1u)) {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    if (k < nks) tc_mma_f16_cg<CG>(d_addr, alo + 2u * k, bhi + 2u * k, 1u);
                            }
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                if (k < nks) tc_mma_f16_cg<CG>(d_addr, ahi + 2u * k, blo + 2u * k, 1u);
                            tc_commit_cg<CG>(&bars.b_empty[bs]);
                            if (n == P.NT - 1) tc_commit_cg<CG>(&bars.a_empty[as]);
                        }
                        if (++bs == NB) { bs = 0; b_ph ^= 1; }
                    }
                    if (leader) tc_commit_cg<CG>(&bars.acc_full[j & 1u]);
                    ++j;
                    continue;
                }
                mma_wait(&bars.t_full[ts], t_ph);
                if (n == 0) {                   // block 0 of this job (and with it the job's tail rows)
                    const int u = i * DB;
                    mma_wait(&bars.a_full[u % NA], (uint32_t)(u / NA) & 1u);
                    if (IN16) lo_mask = (lo_mask & ~1u) | lo_flag(u % NA);
                }
                tc_fence_after();
                if (leader) {
                    tc_mma_f16_cg<CG>(d_addr, atdesc0 + (uint32_t)(i & 1) * TA_UNITS, btdesc0 + (uint32_t)ts * T_UNITS, 0u);
                    tc_commit_cg<CG>(&bars.t_empty[ts]);
                }
                if (++ts == 2) { ts = 0; t_ph ^= 1; }
                for (int fb = 0; fb < DB; ++fb) {
                    const int nks = (fb == DB - 1) ? P.nks_last : 4;
                    const int u = i * DB + fb;
                    const int as = u % NA;
                    if (n == 0 && fb > 0) {
                        mma_wait(&bars.a_full[as], (uint32_t)(u / NA) & 1u);
                        if (IN16) lo_mask = (lo_mask & ~(1u << fb)) | (lo_flag(as) << fb);
                    }
                    const uint64_t ahi = adesc0 + (uint32_t)as * A_SLOT_UNITS;
                    const uint64_t alo = ahi + A_LO_UNITS;
                    mma_wait(&bars.b_full[bs], b_ph);
                    tc_fence_after();
                    uint64_t bd = bdesc0 + (uint32_t)bs * B_UNITS;
                    if (leader) {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (k < nks) tc_mma_f16_cg<CG>(d_addr, ahi + 2u * k, bd + 2u * k, 1u);
                        if (!IN16 || ((lo_mask >> fb) & 1u)) {
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                if (k < nks) tc_mma_f16_cg<CG>(d_addr, alo + 2u * k, bd + 2u * k, 1u);
                        }
                        tc_commit_cg<CG>(&bars.b_empty[bs]);
                    }
                    if (++bs == NB) { bs = 0; b_ph ^= 1; }
                    mma_wait(&bars.b_full[bs], b_ph);
                    tc_fence_after();
                    bd = bdesc0 + (uint32_t)bs * B_UNITS;
                    if (leader) {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (k < nks) tc_mma_f16_cg<CG>(d_addr, ahi + 2u * k, bd + 2u * k, 1u);
                        tc_commit_cg<CG>(&bars.b_empty[bs]);
                        if (n == P.NT - 1) tc_commit_cg<CG>(&bars.a_empty[as]);
                    }
                    if (++bs == NB) { bs = 0; b_ph ^= 1; }
                }
                if (leader) tc_commit_cg<CG>(&bars.acc_full[j & 1u]);
                ++j;
            }
        }
        if (prof && leader && j > 0) {
            g_prof16[0] = clock64() - t_begin; g_prof16[1] = (long long)j;
            g_prof16[2] = w_acc; g_prof16[3] = w_b; g_prof16[4] = w_a;
        }
    } else if (warp >= BUILD_WARP0 && warp < BUILD_WARP0 + BUILD_WARPS) {
        // ================================ A builders ==================================
        const int t = threadIdx.x - BUILD_WARP0 * 32;                  // patch row inside the tile
        const int vec = P.g.vec;
        const int tc_exp = (int)((__float_as_uint(__ldg(P.scale + 1)) >> 23) & 0xffu) - 127;
        const uint32_t sw = (uint32_t)(t & 7);
        float v[64];
        // 64 features [64 fb, 64 fb + 64) of one patch row; zero beyond D and for padding rows
        // (vec counts elements: 16- / 8-byte runs of floats, 8- / 4-byte runs of halves)
        auto load_blk = [&](const T* src, bool ok, int fb) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const int d = fb * 64 + c * 4;
                float tmp[4] = {0.f, 0.f, 0.f, 0.f};
                if (ok && d < D) {
                    if (vec == 4) {
                        ld4(src + aux.foff[d], tmp);
                    } else if (vec == 2) {
                        ld2(src + aux.foff[d], tmp);
                        if (d + 2 < D) ld2(src + aux.foff[d + 2], tmp + 2);
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (d + e < D) tmp[e] = ld1(src + aux.foff[d + e]);
                    }
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) v[c * 4 + e] = tmp[e];
            }
        };
        int i = 0;
        for (int q = job0; q < n_jobs; q += job_stride, ++i) {
            const int m = CG * q + (int)rank;
            const int64_t p = (int64_t)m * TM + t;
            const bool ok = p < P.rows;
            const T* src = static_cast<const T*>(P.x) + (ok ? patch_base(P.g, p) : 0);
            // pass 1: the row's largest magnitude (a one-block row stays in registers for pass 2)
            float mx = 0.f;
            for (int fb = 0; fb < DB; ++fb) {
                load_blk(src, ok, fb);
#pragma unroll
                for (int e = 0; e < 64; ++e) mx = fmaxf(mx, fabsf(v[e]));
            }
            // power-of-two row scale: max |s_p x| in [64, 128) as long as a_p = s_p / t_c is an exact FP16 power of
            // two (2^-24 .. 2^15); an all-zero or non-finite row takes the ideal exponent 0
            const int eb = (int)((__float_as_uint(mx) >> 23) & 0xffu);
            int ep = 133 - eb;
            if (!(mx > 0.f) || eb == 0xff) ep = 0;
            int ka = ep - tc_exp, es;
            float ap;
            if (ka < -24) {
                // |x| beyond ~2^24 |c|: ||c||^2 is below fp32 resolution of rd; keep the row in range instead
                es = ep;
                ap = 0.f;
            } else {
                ka = ka > 15 ? 15 : ka;                 // 2^-24 .. 2^15: exact in FP16 (subnormal below 2^-14)
                es = ka + tc_exp;
                ap = __uint_as_float((uint32_t)(127 + ka) << 23);
            }
            es = es > 120 ? 120 : (es < -120 ? -120 : es);
            const float sp = __uint_as_float((uint32_t)(127 + es) << 23);
            for (int fb = 0; fb < DB; ++fb) {
                if (DB > 1) load_blk(src, ok, fb);
                if (P.stage != nullptr && ok) {
                    // patch-major staging copy for the update's segmented gather: a patch is sixteen 16-byte pieces
                    // in NCHW (P = 4) but ONE contiguous row here, and the builder holds it in registers anyway
                    float* srow = P.stage + p * D + fb * 64;
                    if ((D & 3) == 0) {
#pragma unroll
                        for (int c = 0; c < 16; ++c)
                            if (fb * 64 + c * 4 < D)
                                *reinterpret_cast<float4*>(srow + c * 4) = make_float4(v[c * 4], v[c * 4 + 1], v[c * 4 + 2], v[c * 4 + 3]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 64; ++e)
                            if (fb * 64 + e < D) srow[e] = v[e];
                    }
                }
                const int u = i * DB + fb;
                const int as = u % NA;
                mbar_wait_warp<true>(&bars.a_empty[as], ((uint32_t)(u / NA) & 1u) ^ 1u, lane);
                uint8_t* hi_row = a_ring + (size_t)as * A_SLOT_BYTES + (uint32_t)t * 128u;
                uint8_t* lo_row = hi_row + A_BLK_BYTES;
                bool lo_nz = false;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    float h[8], l[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float s = v[c * 8 + e] * sp;                   // exact
                        h[e] = __half2float(__float2half_rn(s));
                        l[e] = s - h[e];                                     // exact; rounded to FP16 when packed
                        if (IN16) lo_nz |= l[e] != 0.f;                       // (NaN counts as non-zero)
                    }
                    // 16-byte chunk c of row t lives at t * 128 + ((c ^ (t & 7)) << 4)
                    const uint32_t off = (((uint32_t)c) ^ sw) << 4;
                    *reinterpret_cast<uint4*>(hi_row + off) = pack_h8(h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7]);
                    *reinterpret_cast<uint4*>(lo_row + off) = pack_h8(l[0], l[1], l[2], l[3], l[4], l[5], l[6], l[7]);
                }
                if (fb == 0) {
                    // tail row t = [a_p a_p a_p 0.. | 0..] in the 32-byte swizzle (chunk ^= bit 2 of t)
                    const uint32_t sw32 = (uint32_t)(t >> 2) & 1u;
                    uint4* rowp = reinterpret_cast<uint4*>(a_tail + (size_t)(i & 1) * TAIL_A_BYTES + t * 32);
                    rowp[sw32] = pack_h8(ap, ap, ap, 0.f, 0.f, 0.f, 0.f, 0.f);
                    rowp[sw32 ^ 1u] = make_uint4(0u, 0u, 0u, 0u);
                    aux.row_exp[i & 1][t] = es;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                const bool warp_lo_nz = IN16 && __any_sync(0xffffffffu, lo_nz);
                __syncwarp();
                if (lane == 0) {
                    if (IN16) {
                        // this warp's byte of the slot's flag, in the leader CTA; the release arrive below publishes it
                        uint8_t* fl = &aux.lo_nz[as][rank * BUILD_WARPS + (warp - BUILD_WARP0)];
                        if (CG == 2) {
                            asm volatile(
                                "{\n"
                                ".reg .b32 ra;\n"
                                "mapa.shared::cluster.u32 ra, %0, 0;\n"
                                "st.shared::cluster.u8 [ra], %1;\n"
                                "}\n" ::"r"(smem_u32(fl)), "r"((uint32_t)warp_lo_nz)
                                : "memory");
                        } else {
                            *reinterpret_cast<volatile uint8_t*>(fl) = (uint8_t)warp_lo_nz;
                        }
                    }
                    if (CG == 2) mbar_arrive_remote(&bars.a_full[as], 0);      // the leader's barrier counts both CTAs
                    else mbar_arrive(&bars.a_full[as]);
                    if (fb == 0) mbar_arrive(&bars.exp_full[i & 1]);           // release: row_exp visible
                }
            }
        }
    } else if (warp >= EPI_WARP0) {
        // ================================ epilogue ====================================
        // eight warps: TMEM lane quarter (warp & 3) x column half; a thread owns one patch row and 128 columns
        const int half = (warp - EPI_WARP0) >> 2;
        const int lg = warp & 3;
        const int row = lg * 32 + lane;
        const int sc_exp = (int)((__float_as_uint(__ldg(P.scale)) >> 23) & 0xffu) - 127;
        uint32_t j = 0;
        int i = 0;
        for (int q = job0; q < n_jobs; q += job_stride, ++i) {
            const int m = CG * q + (int)rank;
            const int64_t p = (int64_t)m * TM + row;
            mbar_wait(&bars.exp_full[i & 1], (uint32_t)(i >> 1) & 1u);
            const int es = aux.row_exp[i & 1][row];
            float best = INFINITY;
            int bidx = 0;
            for (int n = 0; n < P.NT; ++n) {
                const uint32_t acc = j & 1u;
                mbar_wait(&bars.acc_full[acc], (j >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(lg * 32) << 16) + acc * TN + (uint32_t)half * 128u;
                const int col0 = n * TN + half * 128;
                uint32_t va[32], vb[32];
                auto consume = [&](const uint32_t (&vv)[32], int c) {
                    const float mn = min32(vv);
                    if (mn < best) { best = mn; bidx = col0 + c * 32 + first_eq32(vv, mn); }
                };
                tmem_ld32_issue(taddr, va);
                tmem_ld_wait(va);
                tmem_ld32_issue(taddr + 32, vb);
                consume(va, 0);
                tmem_ld_wait(vb);
                tmem_ld32_issue(taddr + 64, va);
                consume(vb, 1);
                tmem_ld_wait(va);
                tmem_ld32_issue(taddr + 96, vb);
                consume(va, 2);
                tmem_ld_wait(vb);
                // accumulator fully read: hand it back before the last reduction
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CG == 2) mbar_arrive_remote_relaxed(&bars.acc_empty[acc], 0);
                    else mbar_arrive(&bars.acc_empty[acc]);
                }
                consume(vb, 3);
                ++j;
            }
            // merge the two column halves (value asc, index asc); buffers alternate per job
            if (half == 1) { aux.mrg_val[i & 1][row] = best; aux.mrg_idx[i & 1][row] = bidx; }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (half == 0 && p < P.rows) {
                const float ov = aux.mrg_val[i & 1][row];
                const int oi = aux.mrg_idx[i & 1][row];
                if (ov < best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
                P.out_idx[p] = (int64_t)bidx + P.unit_offset;
                // the accumulator holds s_p s_c rd: undo both powers of two (exact)
                if (P.out_rd) P.out_rd[p] = ldexpf(best, -(es + sc_exp));
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync_all();    // the peer may still multicast into / arrive on this CTA's shared memory
    if (warp == 1) {
        tc_fence_after();
        if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
        else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    }
}

// Per-codebook scales (exact powers of two) from the largest squared norm M2 = max_j ||c_j||^2:
//   s_c = 2^(7 - floor(log2 sqrt(M2)))        so that  128 <= s_c max||c|| < 256, hence max |s_c c| < 256
//   t_c = 2^(14 - floor(log2 (s_c M2)))       so that  max t_c s_c ||c||^2 in [2^14, 2^15)  (FP16 tops out at 65504)
// An all-zero or non-finite codebook keeps both at 1.  One CTA over the K norms.
__device__ __forceinline__ void scales_from_max_norm(float mn, float* out2);
__global__ void __launch_bounds__(1024) cb_scale_l_kernel(const float* __restrict__ cn, int K, float* __restrict__ scale_out) {
    pdl_begin();
    trace_stamp(s_trace_buf, 6);
    __shared__ float sh[32];
    float mn = 0.f;
    for (int i = threadIdx.x; i < K; i += 1024) mn = fmaxf(mn, fabsf(__ldg(cn + i)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mn = fmaxf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = mn;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) mn = fmaxf(mn, sh[w]);
        scales_from_max_norm(mn, scale_out);
    }
}

// Pre-split codebook, FP16: row j = [ hi(-2 s_c c) for every 64-feature block | lo(..) for every block ] (halves,
// zero beyond D); tail rows = 16 halves [n1 n2 n3 0..] of t_c s_c ||c||^2.  Rows >= K repeat unit K - 1: a padding
// unit then never beats a real one (ties go to the lower index), whatever the patch holds.
// One thread per (row, pair of features).  OWN_SCALE (codebooks of up to 32 768 units): every CTA derives the two
// scales itself from the K norms (L2-resident) instead of waiting for cb_scale_l_kernel -- one launch fewer on the
// per-step critical path; CTA 0 publishes them for the search kernel.
__device__ __forceinline__ void scales_from_max_norm(float mn, float* out2) {
    // a NaN norm is dropped by fmaxf; an infinite one shows up as exponent 0xff
    const int en = (int)((__float_as_uint(mn) >> 23) & 0xffu);
    int e = 0, g = 0;
    if (mn > 0.f && en != 0xff && en != 0) {
        const int e2 = en - 127;                                     // M2 in [2^e2, 2^(e2+1))
        const int fl = (e2 >= 0) ? (e2 >> 1) : -((1 - e2) >> 1);     // floor(e2 / 2) = floor(log2 sqrt(M2))
        e = 7 - fl;
        e = e > 60 ? 60 : (e < -60 ? -60 : e);
        g = 14 - (e2 + e);
        g = g > 60 ? 60 : (g < -60 ? -60 : g);
    }
    out2[0] = __uint_as_float((uint32_t)(127 + e) << 23);
    out2[1] = __uint_as_float((uint32_t)(127 + g) << 23);
}

template <bool OWN_SCALE>
__global__ void __launch_bounds__(256) split_w_l16_kernel(const float* __restrict__ W, const float* __restrict__ cn,
                                                          int K, int D, int DB, int K_pad,
                                                          float* __restrict__ scale, __half* __restrict__ Bp,
                                                          __half* __restrict__ Tp) {
    pdl_begin();
    trace_stamp(s_trace_buf, 6);
    __shared__ float sh_max[8];
    __shared__ float sh_scale[2];
    if (OWN_SCALE) {
        float mn = 0.f;
        for (int i = threadIdx.x; i < K; i += 256) mn = fmaxf(mn, fabsf(__ldg(cn + i)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = fmaxf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if ((threadIdx.x & 31) == 0) sh_max[threadIdx.x >> 5] = mn;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < 8; ++w) mn = fmaxf(mn, sh_max[w]);
            scales_from_max_norm(mn, sh_scale);
            if (blockIdx.x == 0) { scale[0] = sh_scale[0]; scale[1] = sh_scale[1]; }
        }
        __syncthreads();
    }
    const int pairs = DB * 32;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= (int64_t)K_pad * pairs) return;
    const int row = (int)(t / pairs);
    const int d = (int)(t - (int64_t)row * pairs) * 2;
    const int src = row < K ? row : K - 1;
    const float sc = OWN_SCALE ? sh_scale[0] : scale[0], tcs = OWN_SCALE ? sh_scale[1] : scale[1];
    float v0 = 0.f, v1 = 0.f;
    if (d < D) v0 = -2.0f * sc * W[(int64_t)src * D + d];                   // exact scaling
    if (d + 1 < D) v1 = -2.0f * sc * W[(int64_t)src * D + d + 1];
    const float h0 = __half2float(__float2half_rn(v0)), h1 = __half2float(__float2half_rn(v1));
    const int64_t cols = (int64_t)DB * 64;
    __half* rowp = Bp + (int64_t)row * 2 * cols;
    *reinterpret_cast<__half2*>(rowp + d) = __floats2half2_rn(h0, h1);
    *reinterpret_cast<__half2*>(rowp + cols + d) = __floats2half2_rn(v0 - h0, v1 - h1);
    if (d < 16) {
        float o0 = 0.f, o1 = 0.f;
        if (d < 4) {
            const float nrm = cn[src] * sc * tcs;
            const float n1 = __half2float(__float2half_rn(nrm));
            const float n2 = __half2float(__float2half_rn(nrm - n1));
            const float n3 = nrm - n1 - n2;
            if (d == 0) { o0 = n1; o1 = n2; } else { o0 = n3; o1 = 0.f; }
        }
        *reinterpret_cast<__half2*>(Tp + (int64_t)row * 16 + d) = __floats2half2_rn(o0, o1);
    }
}

struct Plan {
    int cg, merged, D, K, DB, nks_last, K_pad, NT, n_mtiles, NA, NB;
    size_t off_b, off_t, off_s, total;
};

static bool make_plan(Plan* pl, int64_t n, int D, int K, bool force) {
    if (D <= 16 || D > DMAX || n <= 0 || K <= 0) return false;
    pl->D = D; pl->K = K;
    pl->DB = (D + 63) / 64;
    pl->nks_last = (D - 64 * (pl->DB - 1) + 15) / 16;
    pl->K_pad = (K + TN - 1) / TN * TN;
    pl->NT = pl->K_pad / TN;
    pl->n_mtiles = (int)ceil_div64(n, TM);
    const int sms = sm_count();
    // static rule: large batches only (at least one full wave of patch tiles and four unit tiles); smaller problems
    // keep the 3xTF32 kernels with their unit / feature splits
    // (`force`, SOM_BMU_TC_F16: any batch size -- tests and A/B runs; three unit tiles are the protocol's minimum)
    if (pl->NT < 3 || (!force && (pl->n_mtiles < sms || pl->NT < 4))) return false;
    pl->cg = (sms % 2 == 0 && pl->n_mtiles >= 2 * sms) ? 2 : 1;
    if (force && pl->DB > 2 && pl->n_mtiles >= 2 && sms % 2 == 0) pl->cg = 2;
    pl->NA = pl->DB <= 2 ? 2 : 4;
    // four-slot tiles leave 64 KB for the B ring: only CTA pairs (16 KB half blocks) keep enough stages in flight
    // (a forced single-CTA launch runs with two 32 KB stages: correct, not fast)
    if (pl->NA == 4 && pl->cg != 2 && !force) return false;
    pl->merged = pl->NA == 2 ? 1 : 0;
    if (pl->merged) pl->NB = (TILES_BYTES - 2 * A_SLOT_BYTES - 2 * TAIL_A_BYTES) / ((2 * B_BLK_BYTES + TAIL_B_BYTES) / pl->cg);
    else pl->NB = (RING_BYTES - pl->NA * A_SLOT_BYTES) / (B_BLK_BYTES / pl->cg);
    if (pl->NB > NB_MAX) pl->NB = NB_MAX;
    size_t o = 0;
    pl->off_b = o; o = align_up(o + (size_t)pl->K_pad * pl->DB * 64 * 2 * 2, 1024);
    pl->off_t = o; o = align_up(o + (size_t)pl->K_pad * 16 * 2, 1024);
    pl->off_s = o; o += 1024;
    pl->total = o;
    return true;
}

}  // namespace tcl16

bool tc_l16_applicable(int64_t n_patches, int D, int K, bool force) {
    tcl16::Plan pl;
    return tcl16::make_plan(&pl, n_patches, D, K, force);
}

size_t tc_l16_workspace_bytes(int64_t n_patches, int D, int K, bool force) {
    tcl16::Plan pl;
    return tcl16::make_plan(&pl, n_patches, D, K, force) ? pl.total : 0;
}

// the plan of launch_bmu_tc_l16 for som_debug_bmu_plan (f: PF_COUNT fields, pre-filled with -1); false where no
// FP16-split kernel covers the shape
bool tc_l16_plan_fields(int64_t n_patches, int D, int K, bool force, int64_t* f) {
    tcl16::Plan pl;
    if (!tcl16::make_plan(&pl, n_patches, D, K, force)) return false;
    f[PF_CG] = pl.cg;
    f[PF_MERGED] = pl.merged;
    f[PF_NT] = pl.NT;
    f[PF_DB] = pl.DB;
    f[PF_MTILES] = pl.n_mtiles;
    return true;
}

int launch_bmu_tc_l16(const void* x, int elem, const Geom& g, const float* W, const float* cn, int K,
                      int64_t unit_offset, int64_t* out_idx, float* out_rd, float* stage, void* ws, size_t ws_bytes,
                      bool force, cudaStream_t st) {
    using namespace tcl16;
    SOM_REQUIRE(elem == ELEM_F32 || elem == ELEM_F16 || elem == ELEM_BF16, SOM_E_BADARG, "bmu(tc f16): element type %d",
                elem);
    const int64_t n = g.n_patches;
    if (n == 0) return SOM_OK;
    Plan pl;
    SOM_REQUIRE(make_plan(&pl, n, g.D, K, force), SOM_E_UNSUPPORTED, "bmu(tc f16): shape n=%lld D=%d K=%d not covered",
                (long long)n, g.D, K);
    SOM_REQUIRE(ws != nullptr && ws_bytes >= pl.total, SOM_E_WORKSPACE, "bmu(tc f16): workspace %zu < required %zu",
                ws_bytes, pl.total);
    SOM_REQUIRE(((uintptr_t)ws & 255) == 0, SOM_E_BADARG, "bmu(tc f16): workspace must be 256-byte aligned");
    __half* Bp = (__half*)((char*)ws + pl.off_b);
    __half* Tp = (__half*)((char*)ws + pl.off_t);
    float* scale = (float*)((char*)ws + pl.off_s);
    int rc;
    {
        const int64_t items = (int64_t)pl.K_pad * pl.DB * 32;
        const unsigned blocks = (unsigned)ceil_div64(items, 256);
        if (K <= 32768) {
            launch_pdl(split_w_l16_kernel<true>, blocks, 256, 0, st, W, cn, K, g.D, pl.DB, pl.K_pad, scale, Bp, Tp);
        } else {
            launch_pdl(cb_scale_l_kernel, 1, 1024, 0, st, cn, K, scale);
            rc = check_launch("cb_scale_l_kernel");
            if (rc) return rc;
            launch_pdl(split_w_l16_kernel<false>, blocks, 256, 0, st, W, cn, K, g.D, pl.DB, pl.K_pad, scale, Bp, Tp);
        }
        rc = check_launch("split_w_l16_kernel");
        if (rc) return rc;
    }
    // the operand rows are bytes to TMA: a 64-half block is a 32-float box
    CUtensorMap map_b, map_t;
    const uint32_t box_rows = TN / pl.cg;
    rc = make_map2d(&map_b, Bp, (uint64_t)pl.K_pad, (uint64_t)pl.DB * 64, (uint64_t)pl.DB * 64 * 4, 32, box_rows,
                    CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_map2d(&map_t, Tp, (uint64_t)pl.K_pad, 8, 32, 8, box_rows, CU_TENSOR_MAP_SWIZZLE_32B);
    if (rc) return rc;

    Params P;
    P.DB = pl.DB; P.nks_last = pl.nks_last; P.NT = pl.NT; P.n_mtiles = pl.n_mtiles; P.NA = pl.NA; P.NB = pl.NB;
    P.K_pad = pl.K_pad; P.rows = n; P.unit_offset = unit_offset; P.out_idx = out_idx; P.out_rd = out_rd;
    P.x = x; P.g = g; P.scale = scale; P.stage = stage;

    typedef void (*KernelFn)(const CUtensorMap, const CUtensorMap, const Params);
    // [elem][merged][cg - 1], elem = ELEM_F32 / ELEM_F16 / ELEM_BF16
    static const KernelFn kernels[12] = {
        bmu_tc_l16_kernel<1, false, float>, bmu_tc_l16_kernel<2, false, float>,
        bmu_tc_l16_kernel<1, true, float>, bmu_tc_l16_kernel<2, true, float>,
        bmu_tc_l16_kernel<1, false, __half>, bmu_tc_l16_kernel<2, false, __half>,
        bmu_tc_l16_kernel<1, true, __half>, bmu_tc_l16_kernel<2, true, __half>,
        bmu_tc_l16_kernel<1, false, __nv_bfloat16>, bmu_tc_l16_kernel<2, false, __nv_bfloat16>,
        bmu_tc_l16_kernel<1, true, __nv_bfloat16>, bmu_tc_l16_kernel<2, true, __nv_bfloat16>};
    static PerDeviceFlag attr_done;
    if (attr_done.pending()) {
        for (int c = 0; c < 12; ++c) {
            cudaError_t e = cudaFuncSetAttribute(kernels[c], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
            if (e != cudaSuccess) { set_error("bmu(tc f16): smem opt-in: %s", cudaGetErrorString(e)); return (int)e; }
        }
        attr_done.set();
    }
    const int n_jobs = (pl.n_mtiles + pl.cg - 1) / pl.cg;
    const int max_groups = sm_count() / pl.cg;
    const int groups = n_jobs < max_groups ? n_jobs : max_groups;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(groups * pl.cg));
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)pl.cg;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // (see som_common.cuh: pdl_begin)
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    cudaError_t le = cudaLaunchKernelEx(&cfg, kernels[4 * elem + 2 * pl.merged + pl.cg - 1], map_b, map_t, P);
    if (le != cudaSuccess) { set_error("bmu_tc_l16_kernel: launch: %s", cudaGetErrorString(le)); return (int)le; }
    return check_launch("bmu_tc_l16_kernel");
}

}  // namespace som

// debug: CTA 0's MMA issue loop in the last FP16-split launch: cycles, tiles, cycles waiting for a free accumulator
// (epilogue), for B stages (TMA) and for A tiles (builders)
extern "C" SOM_API int som_debug_tc_l16_cycles(long long* out5) {
    return (int)cudaMemcpyFromSymbol(out5, som::tcl16::g_prof16, 5 * sizeof(long long));
}
