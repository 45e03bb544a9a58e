// K1 (tensor-core variant): dispatch between the tcgen05 BMU kernels.  sm_100a only.
//
// Replaces patchify + torch.cdist + torch.argmin of Codebook.get_patches_bmu
// (/root/reference/models/Codebook.py:77-99).  The reduced distance
//     rd[p][j] = ||c_j||^2 - 2 x_p . c_j          (d^2 = rd + ||x_p||^2, row-constant dropped)
// is computed as an error-compensated 3xTF32 GEMM (hi/lo split of both operands, three products, norms through
// one extra k-step) with the argmin fused into the TMEM epilogue.  Static rule on the shape, no autotuner:
//   D <= 16  -> som_bmu_tc_s.cu  (config S: R = 4 resident patch tiles, chunk-tracking epilogue + exact refine)
//   D  > 16  -> som_bmu_tc_l16.cu (FP16 hi/lo split, kind::f16: D <= 256 and at least one full wave of patch tiles)
//               som_bmu_tc_l.cu  (3xTF32: resident-A for D <= 64, TMA-streamed A for larger D, split-K when there are
//                                 fewer patch tiles than SMs; CTA pairs for large problems)
// `arith`: 0 = static rule, 1 = 3xTF32 everywhere (SOM_BMU_TC_TF32), 2 = FP16 split wherever a kernel exists
// (SOM_BMU_TC_F16).
#include "som_common.cuh"
#include "som_tc_ptx.cuh"

namespace som {

// som_bmu_tc_s.cu
bool tc_s_applicable(int D);
bool tc_s_f16_mode(int64_t n_patches, int arith);
void tc_s_plan_fields(int64_t n_patches, int K, int arith, int64_t* f);
size_t tc_s_workspace_bytes(int64_t n_patches, int D, int K);
int launch_bmu_tc_s(const float* x, const Geom& g, const float* W, const float* cn, int K, int64_t unit_offset,
                    int64_t* out_idx, float* out_rd, void* ws, size_t ws_bytes, int arith, cudaStream_t st);
// som_bmu_tc_l16.cu
bool tc_l16_applicable(int64_t n_patches, int D, int K, bool force);
size_t tc_l16_workspace_bytes(int64_t n_patches, int D, int K, bool force);
bool tc_l16_plan_fields(int64_t n_patches, int D, int K, bool force, int64_t* f);
int launch_bmu_tc_l16(const void* x, int elem, const Geom& g, const float* W, const float* cn, int K,
                      int64_t unit_offset, int64_t* out_idx, float* out_rd, float* stage, void* ws, size_t ws_bytes,
                      bool force, uint32_t* wflags, cudaStream_t st);
// som_bmu_tc_l.cu
size_t tc_l_workspace_bytes(int64_t n_patches, int D, int K);
void tc_l_plan_fields(int64_t n_patches, int D, int K, int64_t* f);
int launch_bmu_tc_l(const float* x, const Geom& g, const float* W, const float* cn, int K, int64_t unit_offset,
                    int64_t* out_idx, float* out_rd, void* ws, size_t ws_bytes, cudaStream_t st);

bool tc_supported(int64_t n_patches, int D, int K) {
    if (n_patches <= 0 || D <= 0 || K <= 0) return false;
    if (n_patches / tc::TM >= (1ll << 30)) return false;
    if ((int64_t)D > (1 << 20)) return false;
    if ((int64_t)K + tc::TN >= (1ll << 31)) return false;
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

static bool use_l16(int64_t n_patches, int D, int K, int arith) {
    return arith != 1 && tc_l16_applicable(n_patches, D, K, arith == 2);
}

// The one dispatch rule of the tensor-core variants: the kernel a shape runs on (PLAN_S, PLAN_L16 or PLAN_L), or -1 where
// SOM_BMU_TC_F16 asks for an FP16-split kernel that does not cover the shape.  Workspace, staging, the split-mode query,
// the launch and som_debug_bmu_plan all read it.
static int tc_kernel(int64_t n_patches, int D, int K, int arith) {
    if (tc_s_applicable(D)) return PLAN_S;
    if (use_l16(n_patches, D, K, arith)) return PLAN_L16;
    return arith == 2 ? -1 : PLAN_L;
}

// 1: FP16 hi/lo split (kind::f16), 0: 3xTF32
int tc_split_mode(int64_t n_patches, int D, int K, int arith) {
    const int k = tc_kernel(n_patches, D, K, arith);
    if (k == PLAN_S) return tc_s_f16_mode(n_patches, arith) ? 1 : 0;
    return k == PLAN_L16 ? 1 : 0;
}

size_t tc_workspace_bytes(int64_t n_patches, int D, int K, int arith) {
    if (!tc_supported(n_patches, D, K)) return 0;
    const int k = tc_kernel(n_patches, D, K, arith);
    if (k == PLAN_S) return tc_s_workspace_bytes(n_patches, D, K);
    if (k == PLAN_L16) return tc_l16_workspace_bytes(n_patches, D, K, arith == 2);
    return tc_l_workspace_bytes(n_patches, D, K);
}

// the kernels whose builders can also emit the patch-major staging copy (som_bmu_stage_nchw_f32)
bool tc_can_stage(int64_t n_patches, int D, int K, int arith) {
    return tc_supported(n_patches, D, K) && tc_kernel(n_patches, D, K, arith) == PLAN_L16;
}

// the kernel launch_bmu_tc / launch_bmu_tc_16 runs for this shape and its plan, for som_debug_bmu_plan (f: PF_COUNT
// fields, pre-filled with -1).  SOM_E_UNSUPPORTED where they would refuse the shape.
int tc_plan_fields(int64_t n_patches, int D, int K, int arith, int64_t* f) {
    SOM_REQUIRE(tc_supported(n_patches, D, K), SOM_E_UNSUPPORTED, "bmu plan: no tensor-core kernel for D=%d K=%d", D, K);
    const int k = tc_kernel(n_patches, D, K, arith);
    SOM_REQUIRE(k >= 0, SOM_E_UNSUPPORTED, "bmu plan: no FP16-split kernel for D=%d K=%d (SOM_BMU_TC_F16)", D, K);
    f[PF_FAMILY] = k;
    if (k == PLAN_S) {
        tc_s_plan_fields(n_patches, K, arith, f);
    } else if (k == PLAN_L16) {
        tc_l16_plan_fields(n_patches, D, K, arith == 2, f);
        f[PF_ARITH] = 1;
    } else {
        tc_l_plan_fields(n_patches, D, K, f);
        f[PF_ARITH] = 0;
    }
    return SOM_OK;
}

// the kernels that read a 16-bit batch (fp16 or bf16) themselves (som_bmu_stage_nchw_f16 / _bf16): the FP16-split
// kernel of 16 < D <= 256 (the same kernel as the one that stages)
bool tc_f16_native(int64_t n_patches, int D, int K, int arith) { return tc_can_stage(n_patches, D, K, arith); }

// wflags (launch_bmu_tc too): NULL, or the B-side flag words of a 16-bit codebook whose exact fp32 copy is W
// (som_bmu_w16_nchw); only the FP16-split kernel reads them
int launch_bmu_tc_16(const void* x, int elem, const Geom& g, const float* W, const float* cn, int K,
                     int64_t unit_offset, int64_t* out_idx, float* out_rd, float* stage, void* ws, size_t ws_bytes,
                     int arith, uint32_t* wflags, cudaStream_t st) {
    if (g.n_patches == 0) return SOM_OK;
    SOM_REQUIRE(tc_f16_native(g.n_patches, g.D, K, arith), SOM_E_UNSUPPORTED,
                "bmu(%s): no kernel reads 16-bit input at n=%lld D=%d K=%d (ask som_bmu_f16_native first)",
                elem == ELEM_BF16 ? "bf16" : "f16", (long long)g.n_patches, g.D, K);
    return launch_bmu_tc_l16(x, elem, g, W, cn, K, unit_offset, out_idx, out_rd, stage, ws, ws_bytes, arith == 2, wflags,
                             st);
}

int launch_bmu_tc(const float* x, const Geom& g, const float* W, const float* cn, int K,
                  int64_t unit_offset, int64_t* out_idx, float* out_rd, float* stage, void* ws, size_t ws_bytes,
                  int arith, uint32_t* wflags, cudaStream_t st) {
    if (g.n_patches == 0) return SOM_OK;
    SOM_REQUIRE(stage == nullptr || tc_can_stage(g.n_patches, g.D, K, arith), SOM_E_UNSUPPORTED,
                "bmu: the kernel for this shape does not emit a staging copy (ask som_bmu_can_stage first)");
    const int k = tc_kernel(g.n_patches, g.D, K, arith);
    if (k == PLAN_S)
        return launch_bmu_tc_s(x, g, W, cn, K, unit_offset, out_idx, out_rd, ws, ws_bytes, arith, st);
    if (k == PLAN_L16)
        return launch_bmu_tc_l16(x, ELEM_F32, g, W, cn, K, unit_offset, out_idx, out_rd, stage, ws, ws_bytes, arith == 2,
                                 wflags, st);
    SOM_REQUIRE(k == PLAN_L, SOM_E_UNSUPPORTED, "bmu: no FP16-split kernel for D=%d K=%d (SOM_BMU_TC_F16)", g.D, K);
    return launch_bmu_tc_l(x, g, W, cn, K, unit_offset, out_idx, out_rd, ws, ws_bytes, st);
}

}  // namespace som
