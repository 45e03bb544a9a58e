// PTX helpers shared by the tcgen05 kernels (sm_100a): mbarrier, TMA, tcgen05 MMA / commit / TMEM, the builders' row
// loader and the epilogue drain.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "som_common.cuh"

namespace som {
namespace tc {

constexpr int TM = 128;              // patches per MMA tile (UMMA M)
constexpr int TN = 256;              // units per MMA tile (UMMA N)
constexpr int KBLK = 32;             // floats per k-block: one 128-byte swizzle row
constexpr int A_BLK_BYTES = TM * KBLK * 4;     // 16 KB
constexpr int B_BLK_BYTES = TN * KBLK * 4;     // 32 KB
constexpr float PAD_NORM = 1.0e30f;            // ||c||^2 of padding units: never the minimum

// ---- PTX helpers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU.  The non-suspending
// test_wait is the fast path (the phase has usually completed already); try_wait sleeps otherwise.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_test(bar, parity)) return;
    for (uint32_t spin = 0; !mbar_try(bar, parity); ++spin)
        if (spin > (1u << 20)) __trap();
}
// warp-level wait: ONE lane polls (with optional back-off for long waits), the rest of the warp parks at
// __syncwarp.  Hundreds of threads spinning on try_wait saturate the barrier unit and slow down the single
// MMA-issuing thread's own barrier checks (measured: ~100+ cycles per check under mass polling).
template <bool BACKOFF>
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity, int lane) {
    if (lane == 0) {
        if (!mbar_test(bar, parity)) {
            for (uint32_t spin = 0; !mbar_try(bar, parity); ++spin) {
                if (BACKOFF) __nanosleep(spin < 64 ? 64 : 256);
                if (spin > (1u << 20)) __trap();
            }
        }
    }
    __syncwarp();
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// ---- CTA-pair (cta_group::2) helpers ------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_count_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster (release at cluster scope)
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
    asm volatile(
        "{\n"
        ".reg .b32 ra;\n"
        "mapa.shared::cluster.u32 ra, %0, %1;\n"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(cta)
        : "memory");
}
// The same arrival WITHOUT release semantics: for signals that publish no memory writes (an epilogue warp handing a
// TMEM accumulator back after tcgen05.ld + tcgen05.fence::before_thread_sync).  The release form compiles to
// MEMBAR.ALL.GPU + ERRBAR in front of the arrive (ncu: 16 % of all stall samples of the FP16-split kernel, on the
// critical path of every tile).
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint64_t* bar, uint32_t cta) {
    asm volatile(
        "{\n"
        ".reg .b32 ra;\n"
        "mapa.shared::cluster.u32 ra, %0, %1;\n"
        "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(cta)
        : "memory");
}
// bounded wait with cluster-scope acquire (barriers that peer CTAs arrive on)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    for (uint32_t spin = 0; !ok; ++spin) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (spin > (1u << 20)) __trap();
    }
}
// TMA load issued by either CTA of a pair; the transaction bytes land on the LEADER's barrier (peer bit cleared)
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
        : "memory");
}
// one lane of a converged warp (elect.sync): the MMA warp keeps warp-uniform control flow, so descriptors
// live in uniform registers, and only the tcgen05 instructions themselves are predicated on the elected lane
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n"
        ".reg .b32 rx;\n"
        ".reg .pred px;\n"
        "elect.sync rx|px, %1;\n"
        "@px mov.s32 %0, 1;\n"
        "}\n"
        : "+r"(pred)
        : "r"(0xFFFFFFFFu));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- tcgen05.mma / tcgen05.commit --------------------------------------------------------------------
// kind::tf32: TF32 operands, M x N x K8.  kind::f16 with FP16 operands: M x N x K16 at the cycle cost of the K8 TF32 MMA.
enum class MmaKind { TF32, F16 };
// instruction descriptor: fp32 accumulate, a/b format (TF32 2, FP16 0), K-major operands, N >> 3, M >> 4
constexpr uint32_t make_idesc(MmaKind kind, int M, int N) {
    return (1u << 4) | ((kind == MmaKind::TF32 ? 2u : 0u) << 7) | ((kind == MmaKind::TF32 ? 2u : 0u) << 10) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
#define SOM_TC_MMA_ASM(cg, kind)                                                                 \
    asm volatile(                                                                                \
        "{\n"                                                                                    \
        ".reg .pred p;\n"                                                                        \
        "setp.ne.b32 p, %4, 0;\n"                                                                \
        "tcgen05.mma.cta_group::" #cg ".kind::" #kind " [%0], %1, %2, %3, p;\n"                  \
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)                      \
        : "memory")
// M = 128 * CG rows (one 128-row half per CTA), N columns; accum = 0 overwrites the accumulator
template <MmaKind KIND, int CG = 1, int N = TN>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accum) {
    constexpr uint32_t idesc = make_idesc(KIND, TM * CG, N);
    if constexpr (KIND == MmaKind::TF32) {
        if constexpr (CG == 1) SOM_TC_MMA_ASM(1, tf32); else SOM_TC_MMA_ASM(2, tf32);
    } else {
        if constexpr (CG == 1) SOM_TC_MMA_ASM(1, f16); else SOM_TC_MMA_ASM(2, f16);
    }
}
#undef SOM_TC_MMA_ASM
// arrive (once the issued MMAs completed) on the barrier at shared address `bar` in every CTA of the pair (CG = 2:
// multicast to both)
template <int CG = 1>
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    } else {
        asm volatile(
            "{\n"
            ".reg .b16 m;\n"
            "mov.b16 m, 3;\n"
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n"
            "}\n" ::"r"(bar)
            : "memory");
    }
}
template <int CG = 1>
__device__ __forceinline__ void tc_commit(uint64_t* bar) { tc_commit<CG>(smem_u32(bar)); }

// ---- TMEM allocation (warp-wide: one warp allocates, the same warp frees) ----------------------------------
template <int CG = 1>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst, uint32_t cols) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)), "r"(cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)), "r"(cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
}
template <int CG = 1>
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
    if constexpr (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols));
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols));
}

// the 1024-byte aligned start of the dynamic shared memory (SWIZZLE_128B tiles).  The alignment is an OFFSET into the
// shared array: rounding the pointer through uintptr_t made the compiler forget the address space, and every access
// compiled to generic LD.E / ST.E (cuobjdump, round 2)
__device__ __forceinline__ uint8_t* aligned_tiles(uint8_t* smem_raw) {
    return smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
}
// K-major, SWIZZLE_128B operand descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO=1 | SBO=1024>>4
// | version=1 | layout_type=2.  Advancing one K=8 step inside the 128-byte row adds 32 B (2 units).
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// K-major SWIZZLE_32B operand descriptor (the norm tail k-step): 32-byte rows, 8-row groups 256 B apart
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46) |
           (6ull << 61);
}
// TF32 norm tail operand A: row t = [1 1 1 0 | 0 0 0 0] in the 32-byte swizzle (chunk ^= bit 2 of t)
__device__ __forceinline__ void write_tail_ones(uint8_t* a_tail, int t) {
    const uint32_t sw = (uint32_t)(t >> 2) & 1u;
    float4* rowp = reinterpret_cast<float4*>(a_tail + t * 32);
    rowp[sw] = make_float4(1.f, 1.f, 1.f, 0.f);
    rowp[sw ^ 1u] = make_float4(0.f, 0.f, 0.f, 0.f);
}

#define SOM_R32(a) "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), \
    "=r"(a[8]), "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]),           \
    "=r"(a[16]), "=r"(a[17]), "=r"(a[18]), "=r"(a[19]), "=r"(a[20]), "=r"(a[21]), "=r"(a[22]), "=r"(a[23]),         \
    "=r"(a[24]), "=r"(a[25]), "=r"(a[26]), "=r"(a[27]), "=r"(a[28]), "=r"(a[29]), "=r"(a[30]), "=r"(a[31])
#define SOM_RW32(a) "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), \
    "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),           \
    "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]),         \
    "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31])

// asynchronous TMEM load of 32 consecutive columns of this warp's 32 lanes (no wait)
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : SOM_R32(r)
        : "r"(taddr)
        : "memory");
}
// wait for all outstanding TMEM loads; the "+r" operands pin every use of r[] after the wait
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" : SOM_RW32(r)::"memory");
}
// epilogue drain of one TMEM accumulator: NCH chunks of 32 columns from taddr, the next chunk's load in flight while
// consume(v, c) reduces chunk c.  Once the last load has landed the accumulator is handed back (fence, warp sync, then
// release(), which arrives on the accumulator's empty barrier) BEFORE the last chunk is consumed.
template <int NCH, typename Consume, typename Release>
__device__ __forceinline__ void tmem_drain(uint32_t taddr, Consume&& consume, Release&& release) {
    uint32_t va[32], vb[32];
    tmem_ld32_issue(taddr, va);
#pragma unroll
    for (int c = 0; c < NCH; c += 2) {
        tmem_ld_wait(va);
        tmem_ld32_issue(taddr + (c + 1) * 32, vb);
        consume(va, c);
        tmem_ld_wait(vb);
        if (c + 2 < NCH) {
            tmem_ld32_issue(taddr + (c + 2) * 32, va);
        } else {
            tc_fence_before();
            __syncwarp();
            release();
        }
        consume(vb, c + 1);
    }
}
__device__ __forceinline__ float min32(const uint32_t (&r)[32]) {
    float m = __uint_as_float(r[0]);
#pragma unroll
    for (int i = 1; i < 32; ++i) m = fminf(m, __uint_as_float(r[i]));
    return m;
}
__device__ __forceinline__ int first_eq32(const uint32_t (&r)[32], float m) {
    int q = 31;
#pragma unroll
    for (int i = 30; i >= 0; --i) q = (__uint_as_float(r[i]) == m) ? i : q;
    return q;
}
__device__ __forceinline__ float tf32_rna(float v) {
    uint32_t o;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(o) : "f"(v));
    return __uint_as_float(o);
}


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
__device__ __forceinline__ void ld4(const __nv_bfloat16* p, float* o) {
    const uint2 r = __ldg(reinterpret_cast<const uint2*>(p));
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.y));
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
__device__ __forceinline__ void ld2(const __nv_bfloat16* p, float* o) {
    const float2 f = __bfloat1622float2(__ldg(reinterpret_cast<const __nv_bfloat162*>(p)));
    o[0] = f.x; o[1] = f.y;
}
__device__ __forceinline__ float ld1(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld1(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float ld1(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }

// builder-side loader: features [d0, d0 + N) of the NCHW patch row `src` into registers (static indexing), zero beyond
// D and where !ok.  vec is the run width of the row in elements (4, 2 or 1: Geom::vec); foff(d) is the element offset
// of feature d from the row's base.
template <int N, typename T, typename FeatOff>
__device__ __forceinline__ void load_row(float (&v)[N], const T* src, bool ok, int d0, int D, int vec, FeatOff&& foff) {
#pragma unroll
    for (int c = 0; c < N; c += 4) {
        const int d = d0 + c;
        float tmp[4] = {0.f, 0.f, 0.f, 0.f};
        if (ok && d < D) {
            if (vec == 4) {
                ld4(src + foff(d), tmp);
            } else if (vec == 2) {
                ld2(src + foff(d), tmp);
                if (d + 2 < D) ld2(src + foff(d + 2), tmp + 2);
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (d + e < D) tmp[e] = ld1(src + foff(d + e));
            }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) v[c + e] = tmp[e];
    }
}

// ---- host side: tensor maps ------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = (EncodeTiledFn)p;
    return fn;
}

// general 2-D fp32 tensor map: `cols` floats per row (row pitch `pitch_bytes`), box = box_cols x box_rows
static inline int make_map2d(CUtensorMap* map, void* base, uint64_t rows, uint64_t cols, uint64_t pitch_bytes,
                             uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swz) {
    EncodeTiledFn fn = get_encode_fn();
    SOM_REQUIRE(fn != nullptr, SOM_E_UNSUPPORTED, "bmu(tc): cuTensorMapEncodeTiled is not available");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch_bytes};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SOM_REQUIRE(r == CUDA_SUCCESS, SOM_E_UNSUPPORTED, "bmu(tc): cuTensorMapEncodeTiled failed (%d)", (int)r);
    return SOM_OK;
}

}  // namespace tc
}  // namespace som
