// K1 dispatch: C-ABI entry points of the BMU search and the static variant rule.
#include "som_common.cuh"

namespace som {
// som_bmu_ffma.cu
size_t ffma_workspace_bytes(int64_t n_patches, int K);
int launch_bmu_ffma(const float* x, const Geom& g, const float* W, const float* cn, int K,
                    int64_t unit_offset, int64_t* out_idx, float* out_rd, void* ws, size_t ws_bytes,
                    cudaStream_t st);
// som_bmu_tc.cu
bool tc_supported(int64_t n_patches, int D, int K);
size_t tc_workspace_bytes(int64_t n_patches, int D, int K, int arith);
int tc_split_mode(int64_t n_patches, int D, int K, int arith);
bool tc_can_stage(int64_t n_patches, int D, int K, int arith);
int launch_bmu_tc(const float* x, const Geom& g, const float* W, const float* cn, int K,
                  int64_t unit_offset, int64_t* out_idx, float* out_rd, float* stage, void* ws, size_t ws_bytes,
                  int arith, uint32_t* wflags, cudaStream_t st);
bool tc_f16_native(int64_t n_patches, int D, int K, int arith);
int tc_plan_fields(int64_t n_patches, int D, int K, int arith, int64_t* f);
int launch_bmu_tc_16(const void* x, int elem, const Geom& g, const float* W, const float* cn, int K, int64_t unit_offset,
                      int64_t* out_idx, float* out_rd, float* stage, void* ws, size_t ws_bytes, int arith,
                      uint32_t* wflags, cudaStream_t st);
}  // namespace som

using namespace som;

// tensor-core variants -> arithmetic selector of som_bmu_tc.cu (0 static rule, 1 3xTF32, 2 FP16 split)
static inline bool is_tc(int variant) { return variant >= SOM_BMU_TC3X && variant <= SOM_BMU_TC_F16; }
static inline int arith_of(int variant) { return variant == SOM_BMU_TC_TF32 ? 1 : (variant == SOM_BMU_TC_F16 ? 2 : 0); }

extern "C" int som_bmu_split_mode(int64_t n_patches, int D, int K) {
    if (n_patches <= 0 || D <= 0 || K <= 0) return -1;
    if (som_bmu_pick_variant(n_patches, D, K) != SOM_BMU_TC3X) return -1;
    return tc_split_mode(n_patches, D, K, 0);
}

extern "C" int som_bmu_pick_variant(int64_t n_patches, int D, int K) {
    // Static rule on the shape (no runtime autotuner), from the measured crossovers of tools/crossover.py:
    //  * tiny codebooks (K * D < 16 384): the tensor-core kernels pay an operand-split pre-pass and 128 x 256
    //    tiles -> FFMA
    //  * D > 16: TC at every batch size.  Few patch tiles are spread over the SMs by splitting the unit tiles
    //    (candidates merged afterwards) or, for long feature axes, the features (split-K): 21 vs 26 us at C1,
    //    33 vs 48-116 us at D = 64 / K = 16 384 / n <= 2048, 30 vs 70 us at D = 256 / K = 2048, 60-75 vs ~950 us at
    //    D = 4096 (the FFMA kernel walks D in 16-feature slabs)
    //  * D <= 16: equal to FFMA (~28 us at K = 4096) up to 4096 patches, 1.6-3.4x faster from 8192 on -> TC from 4096
    if (!tc_supported(n_patches, D, K) || (int64_t)K * D < 16384) return SOM_BMU_FFMA;
    if (D > 16) return SOM_BMU_TC3X;
    return n_patches >= 4096 ? SOM_BMU_TC3X : SOM_BMU_FFMA;
}

extern "C" size_t som_bmu_workspace_bytes(int64_t n_patches, int D, int K, int variant) {
    if (n_patches <= 0 || D <= 0 || K <= 0) return 0;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(n_patches, D, K);
    if (is_tc(variant)) return tc_workspace_bytes(n_patches, D, K, arith_of(variant));
    return ffma_workspace_bytes(n_patches, K);
}

extern "C" int som_bmu_can_stage(int64_t n_patches, int D, int K, int variant) {
    if (n_patches <= 0 || D <= 0 || K <= 0) return 0;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(n_patches, D, K);
    return is_tc(variant) && tc_can_stage(n_patches, D, K, arith_of(variant)) ? 1 : 0;
}

extern "C" int som_bmu_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                const float* W, const float* c_norm2, int K, int64_t unit_offset,
                                int64_t* out_idx, float* out_rd,
                                void* ws, size_t ws_bytes, int variant, void* stream) {
    return som_bmu_stage_nchw_f32(x, n_img, C, H, Wd, pH, pW, W, c_norm2, K, unit_offset, out_idx, out_rd, nullptr, ws,
                                  ws_bytes, variant, stream);
}

extern "C" int som_bmu_stage_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                      const float* W, const float* c_norm2, int K, int64_t unit_offset,
                                      int64_t* out_idx, float* out_rd, float* stage_rows,
                                      void* ws, size_t ws_bytes, int variant, void* stream) {
    // an empty batch (torch hands out null data pointers for zero-element tensors) is a valid no-op: the reference
    // returns an empty int64 tensor for it (models/Codebook.py:77-99 on a (0, C, H, W) input)
    SOM_REQUIRE(W && c_norm2 && ((x && out_idx) || n_img == 0), SOM_E_BADARG, "bmu: null pointer");
    SOM_REQUIRE(K > 0, SOM_E_BADARG, "bmu: K=%d", K);
    SOM_REQUIRE(variant >= SOM_BMU_AUTO && variant <= SOM_BMU_TC_F16, SOM_E_BADARG, "bmu: variant=%d", variant);
    Geom g;
    int rc = make_geom(&g, x, n_img, C, H, Wd, pH, pW);
    if (rc) return rc;
    if (g.n_patches == 0) return SOM_OK;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(g.n_patches, g.D, K);
    if (is_tc(variant)) {
        SOM_REQUIRE(tc_supported(g.n_patches, g.D, K), SOM_E_UNSUPPORTED,
                    "bmu: tensor-core variant does not support D=%d K=%d", g.D, K);
        return launch_bmu_tc(x, g, W, c_norm2, K, unit_offset, out_idx, out_rd, stage_rows, ws, ws_bytes,
                             arith_of(variant), nullptr, (cudaStream_t)stream);
    }
    SOM_REQUIRE(stage_rows == nullptr, SOM_E_UNSUPPORTED, "bmu: the FFMA variant does not emit a staging copy");
    return launch_bmu_ffma(x, g, W, c_norm2, K, unit_offset, out_idx, out_rd, ws, ws_bytes,
                           (cudaStream_t)stream);
}

// debug: the kernel family and plan that a search of n patches of dimension D against K units runs with `variant`, as
// PF_COUNT int64 fields (som_common.cuh: PlanField, -1 where a field does not apply); the first n_out are written.  Tests
// use it to pin which regime a shape reaches.  The answers come from the dispatch and the planners themselves.  The
// element type of the batch enters no plan: an fp16 / bf16 batch runs the same plan, read natively where
// som_bmu_f16_native says so.  Not in somcb.h: a test hook, not part of the ABI.
extern "C" SOM_API int som_debug_bmu_plan(int64_t n_patches, int D, int K, int variant, int64_t* out, int n_out) {
    SOM_REQUIRE(n_patches > 0 && D > 0 && K > 0, SOM_E_BADARG, "bmu plan: n=%lld D=%d K=%d", (long long)n_patches, D, K);
    SOM_REQUIRE(variant >= SOM_BMU_AUTO && variant <= SOM_BMU_TC_F16, SOM_E_BADARG, "bmu plan: variant=%d", variant);
    SOM_REQUIRE(out != nullptr && n_out >= 0, SOM_E_BADARG, "bmu plan: output");
    int64_t f[PF_COUNT];
    for (int i = 0; i < PF_COUNT; ++i) f[i] = -1;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(n_patches, D, K);
    if (is_tc(variant)) {
        const int rc = tc_plan_fields(n_patches, D, K, arith_of(variant), f);
        if (rc) return rc;
    } else {
        f[PF_FAMILY] = PLAN_FFMA;
    }
    for (int i = 0; i < n_out && i < PF_COUNT; ++i) out[i] = f[i];
    return SOM_OK;
}

extern "C" int som_bmu_f16_native(int64_t n_patches, int D, int K, int variant) {
    if (n_patches <= 0 || D <= 0 || K <= 0) return 0;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(n_patches, D, K);
    return is_tc(variant) && tc_f16_native(n_patches, D, K, arith_of(variant)) ? 1 : 0;
}

// fp16 / bf16 batches: the same checks and the same kernel, instantiated for the element type
static int bmu_stage_nchw_16(const char* who, int elem, const void* x, int64_t n_img, int C, int H, int Wd, int pH,
                             int pW, const float* W, const float* c_norm2, int K, int64_t unit_offset, int64_t* out_idx,
                             float* out_rd, float* stage_rows, void* ws, size_t ws_bytes, int variant, void* stream) {
    SOM_REQUIRE(W && c_norm2 && ((x && out_idx) || n_img == 0), SOM_E_BADARG, "%s: null pointer", who);
    SOM_REQUIRE(K > 0, SOM_E_BADARG, "%s: K=%d", who, K);
    SOM_REQUIRE(variant >= SOM_BMU_AUTO && variant <= SOM_BMU_TC_F16, SOM_E_BADARG, "%s: variant=%d", who, variant);
    Geom g;
    int rc = make_geom(&g, x, n_img, C, H, Wd, pH, pW, 2);
    if (rc) return rc;
    if (g.n_patches == 0) return SOM_OK;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(g.n_patches, g.D, K);
    SOM_REQUIRE(is_tc(variant), SOM_E_UNSUPPORTED, "%s: the FFMA variant does not read 16-bit input", who);
    return launch_bmu_tc_16(x, elem, g, W, c_norm2, K, unit_offset, out_idx, out_rd, stage_rows, ws, ws_bytes,
                            arith_of(variant), nullptr, (cudaStream_t)stream);
}

extern "C" int som_bmu_stage_nchw_f16(const void* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                      const float* W, const float* c_norm2, int K, int64_t unit_offset,
                                      int64_t* out_idx, float* out_rd, float* stage_rows,
                                      void* ws, size_t ws_bytes, int variant, void* stream) {
    return bmu_stage_nchw_16("bmu(f16)", ELEM_F16, x, n_img, C, H, Wd, pH, pW, W, c_norm2, K, unit_offset, out_idx,
                             out_rd, stage_rows, ws, ws_bytes, variant, stream);
}

extern "C" int som_bmu_stage_nchw_bf16(const void* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                       const float* W, const float* c_norm2, int K, int64_t unit_offset,
                                       int64_t* out_idx, float* out_rd, float* stage_rows,
                                       void* ws, size_t ws_bytes, int variant, void* stream) {
    return bmu_stage_nchw_16("bmu(bf16)", ELEM_BF16, x, n_img, C, H, Wd, pH, pW, W, c_norm2, K, unit_offset, out_idx,
                             out_rd, stage_rows, ws, ws_bytes, variant, stream);
}

extern "C" int som_bmu_flat_f32(const float* patches, int64_t n, int D, const float* W, const float* c_norm2, int K,
                                int64_t unit_offset, int64_t* out_idx, float* out_rd,
                                void* ws, size_t ws_bytes, int variant, void* stream) {
    SOM_REQUIRE(D > 0, SOM_E_BADARG, "bmu(flat): D=%d", D);
    return som_bmu_nchw_f32(patches, n, 1, 1, D, 1, D, W, c_norm2, K, unit_offset, out_idx, out_rd, ws, ws_bytes,
                            variant, stream);
}

// ---- 16-bit codebooks -----------------------------------------------------------------------------------------------
// Workspace: [ the fp32 search's workspace | exact fp32 copy of W (K x D) | B-side flag words of the FP16-split kernel ]
struct W16Layout { size_t w32, flags, total; };
static W16Layout w16_layout(int64_t n_patches, int D, int K, int variant) {
    W16Layout l;
    l.w32 = align_up(som_bmu_workspace_bytes(n_patches, D, K, variant), 256);
    l.flags = align_up(l.w32 + (size_t)K * D * sizeof(float), 256);
    const int64_t bits = ceil_div64(K, 256) * ceil_div64(D, 64);           // (256-unit tile, 64-feature block) pairs
    l.total = l.flags + align_up((size_t)ceil_div64(bits, 32) * 4, 256);
    return l;
}

extern "C" size_t som_bmu_w16_workspace_bytes(int64_t n_patches, int D, int K, int variant) {
    if (n_patches <= 0 || D <= 0 || K <= 0) return 0;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(n_patches, D, K);
    return w16_layout(n_patches, D, K, variant).total;
}

extern "C" int som_bmu_w16_nchw(const void* x, int x_dtype, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                const void* W, int w_dtype, const float* c_norm2, int K, int64_t unit_offset,
                                int64_t* out_idx, float* out_rd, void* ws, size_t ws_bytes, int variant, void* stream) {
    SOM_REQUIRE(x_dtype >= ELEM_F32 && x_dtype <= ELEM_BF16, SOM_E_BADARG, "bmu(w16): x_dtype=%d", x_dtype);
    SOM_REQUIRE(w_dtype == ELEM_F16 || w_dtype == ELEM_BF16, SOM_E_BADARG, "bmu(w16): w_dtype=%d", w_dtype);
    SOM_REQUIRE(W && c_norm2 && ((x && out_idx) || n_img == 0), SOM_E_BADARG, "bmu(w16): null pointer");
    SOM_REQUIRE(K > 0, SOM_E_BADARG, "bmu(w16): K=%d", K);
    SOM_REQUIRE(variant >= SOM_BMU_AUTO && variant <= SOM_BMU_TC_F16, SOM_E_BADARG, "bmu(w16): variant=%d", variant);
    SOM_REQUIRE(((uintptr_t)W & 1) == 0, SOM_E_BADARG, "bmu(w16): W is not 2-byte aligned");
    Geom g;
    int rc = make_geom(&g, x, n_img, C, H, Wd, pH, pW, x_dtype == ELEM_F32 ? 4 : 2);
    if (rc) return rc;
    if (g.n_patches == 0) return SOM_OK;
    if (variant == SOM_BMU_AUTO) variant = som_bmu_pick_variant(g.n_patches, g.D, K);
    SOM_REQUIRE(x_dtype == ELEM_F32 || som_bmu_f16_native(g.n_patches, g.D, K, variant), SOM_E_UNSUPPORTED,
                "bmu(w16): no kernel reads a 16-bit batch at n=%lld D=%d K=%d (pass its fp32 copy)",
                (long long)g.n_patches, g.D, K);
    SOM_REQUIRE(!is_tc(variant) || tc_supported(g.n_patches, g.D, K), SOM_E_UNSUPPORTED,
                "bmu(w16): tensor-core variant does not support D=%d K=%d", g.D, K);
    const W16Layout l = w16_layout(g.n_patches, g.D, K, variant);
    rc = check_workspace(ws, ws_bytes, l.total, "bmu(w16)");
    if (rc) return rc;
    float* w32 = (float*)((char*)ws + l.w32);
    uint32_t* wflags = (uint32_t*)((char*)ws + l.flags);
    cudaStream_t st = (cudaStream_t)stream;
    // the exact fp32 copy, made per call for the same reason c_norm2 is: the weights may have changed since the last one
    const int64_t nw = (int64_t)K * g.D;
    rc = w_dtype == ELEM_F16 ? som_convert_f16_f32(W, nw, w32, stream) : som_convert_bf16_f32(W, nw, w32, stream);
    if (rc) return rc;
    if (x_dtype != ELEM_F32)
        return launch_bmu_tc_16(x, x_dtype, g, w32, c_norm2, K, unit_offset, out_idx, out_rd, nullptr, ws, l.w32,
                                arith_of(variant), wflags, st);
    if (is_tc(variant))
        return launch_bmu_tc((const float*)x, g, w32, c_norm2, K, unit_offset, out_idx, out_rd, nullptr, ws, l.w32,
                             arith_of(variant), wflags, st);
    return launch_bmu_ffma((const float*)x, g, w32, c_norm2, K, unit_offset, out_idx, out_rd, ws, l.w32, st);
}
