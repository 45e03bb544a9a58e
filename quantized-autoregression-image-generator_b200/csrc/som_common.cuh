// Shared host/device helpers for libsomcb (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <math.h>

#include "../../include/somcb.h"

namespace som {

// ---- error plumbing (thread-local message, codes per include/somcb.h) --------------------
void set_error(const char* fmt, ...);
int  fail(int code, const char* fmt, ...);
int  check_launch(const char* what);          // cudaGetLastError -> code + message; counts launches
unsigned long long launch_count();

#define SOM_REQUIRE(cond, code, ...) \
    do { if (!(cond)) return ::som::fail((code), __VA_ARGS__); } while (0)

int sm_count();                                // cached per process (device 0..n: current device)
int current_device();                          // cudaGetDevice, -1 on error

// cudaFuncSetAttribute is per device: "done once" flags are kept per device ordinal (a process may drive several
// GPUs).  Setting an attribute twice is harmless, so the flag needs no lock.
struct PerDeviceFlag {
    bool done[64] = {};
    bool pending() const { const int d = current_device(); return d < 0 || d >= 64 || !done[d]; }
    void set() { const int d = current_device(); if (d >= 0 && d < 64) done[d] = true; }
};

// ---- patch geometry ------------------------------------------------------------------------
// offset(p, d) = patch_base(p) + feat_off(d): patchify (models/layers.py:8-34) is separable, so
// every kernel treats it as address arithmetic instead of materialising (N, Seq, D).
struct Geom {
    int64_t n_img;
    int C, H, W, pH, pW;
    int gH, gW;          // patches per column / row
    int seq;             // gH * gW
    int D;               // C * pH * pW
    int64_t n_patches;   // n_img * seq
    int64_t img_stride;  // C * H * W
    int vec;             // widest aligned vector (floats) along a patch row: 4, 2 or 1
};

// element type of a feature-map batch: the BMU entry points and the FP16-split kernel's instantiations
// (1 and 2 are also the dtype codes of the version-2 feature-map shards)
enum ElemType : int { ELEM_F32 = 0, ELEM_F16 = 1, ELEM_BF16 = 2 };

// The BMU plan of a shape as som_debug_bmu_plan reports it (som_bmu.cu): one int64 per field, -1 where a field does not
// apply to the kernel family.  The planners fill it in themselves (tc_plan_fields and below), so a test can assert
// which regime a shape reaches without restating a rule.
enum PlanFamily : int { PLAN_FFMA = 0, PLAN_S = 1, PLAN_L16 = 2, PLAN_L = 3 };
enum PlanField : int {
    PF_FAMILY,          // PlanFamily
    PF_ARITH,           // operand split: 0 3xTF32, 1 FP16
    PF_CG,              // CTAs per cluster (2: CTA pairs)
    PF_MERGED,          // L16: one ring stage per 64-feature block (D <= 128)
    PF_MODE,            // L: 0 split-K, 1 resident-A, 2 streamed
    PF_S,               // L: feature splits
    PF_FB_PER_SPLIT,    // L: feature blocks per split
    PF_U,               // L: unit-tile splits
    PF_CHUNK_ROWS,      // L streamed: patch rows per pre-split chunk
    PF_NT,              // unit tiles
    PF_DB,              // feature blocks (32 features in L, 64 in L16)
    PF_RR,              // S: resident patch tiles per CTA
    PF_MTILES,          // 128-patch tiles
    PF_COUNT
};

// elem_bytes: 4 for an fp32 batch, 2 for a 16-bit one (fp16 or bf16; vec then counts 16-bit elements)
int make_geom(Geom* g, const void* x, int64_t n_img, int C, int H, int W, int pH, int pW, int elem_bytes = 4);

__host__ __device__ __forceinline__ int64_t patch_base(const Geom& g, int64_t p) {
    if (g.seq == 1) return p * g.img_stride;      // one patch per image (e.g. pre-flattened rows): no divisions
    int64_t n = p / g.seq;
    int s = (int)(p - n * g.seq);
    int ph = s / g.gW;
    int pw = s - ph * g.gW;
    return n * g.img_stride + (int64_t)(ph * g.pH) * g.W + pw * g.pW;
}

__host__ __device__ __forceinline__ int feat_off(const Geom& g, int d) {
    if (g.seq == 1) return d;        // one patch per image: the patch row IS the image
    int pp = g.pH * g.pW;
    int c = d / pp;
    int r = d - c * pp;
    int i = r / g.pW;
    int j = r - i * g.pW;
    return (c * g.H + i) * g.W + j;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- device-timestamp tracer (debug only: off unless som_debug_trace() handed the library a buffer) -------------------
// The first thread of an instrumented kernel appends (kernel id, %globaltimer) when the kernel starts; the differences
// between consecutive entries are the kernels' durations including the gaps between them -- what CUDA events cannot
// show inside a replayed graph, and ncu cannot show for a multi-rank run.  buf[0] = number of entries.
__device__ __forceinline__ void trace_stamp(unsigned long long* buf, int id) {
    if (buf != nullptr && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)::"memory");
        const unsigned long long slot = atomicAdd(buf, 1ull);
        if (slot < 4000ull) { buf[1 + 2 * slot] = (unsigned long long)id; buf[2 + 2 * slot] = t; }
    }
}
#define SOM_TRACE_TU(setter)                                                            \
    static __device__ unsigned long long* s_trace_buf = nullptr;                        \
    void setter(unsigned long long* p) { cudaMemcpyToSymbol(s_trace_buf, &p, sizeof(p)); }

// ---- programmatic dependent launch ----------------------------------------------------------------------------------
// The training step is a chain of ~20 short dependent kernels; replayed from a CUDA graph each link still cost ~1.8 us
// between the last block of one kernel and the first block of the next (device-timestamp trace).  Kernels on that chain
// are launched with the programmatic-stream-serialization attribute and begin with pdl_begin(): they let THEIR successor
// become resident at once, then block until the predecessor has completed and flushed.  Rules that keep this safe:
// every chained kernel executes the wait before its first global access and before it exits (completion is then
// transitive along the chain), and nothing before the wait touches global memory.
#ifdef SOM_PDL_EARLY_TRIGGER
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#else
__device__ __forceinline__ void pdl_launch_dependents() {}
#endif
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_begin() { pdl_launch_dependents(); pdl_wait(); }

bool pdl_enabled();                                   // som_core.cu; som_debug_set_pdl(0) turns the attribute off (A/B timing)
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace som
