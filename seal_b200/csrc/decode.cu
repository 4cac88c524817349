// Host orchestration + C ABI (include/sealdec.h) of the constrained beam-search decode:
// BART weights, workspace, encoder pass, per-step decoder forward, fused select step.
#include "../../include/sealdec.h"
#include "bart_kernels.cuh"
#include "common.cuh"
#include "decode_kernels.cuh"
#include "fm_handle.hpp"
#include "umma_gemm.cuh"
#include "umma_gemm_2cta.cuh"

#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <set>
#include <string>
#include <vector>

using namespace sealb200;

namespace {

struct Lin {
    float* w = nullptr; float* b = nullptr; int out = 0, in = 0;
    float* w_hi = nullptr; float* w_lo = nullptr;          // TF32 split copies (gemm_mode 2)
    __half* w_h1 = nullptr; __half* w_h2 = nullptr;        // FP16 split copies of W * 2^s (gemm_mode 3)
    float w_unscale = 1.f;                                 // 2^-s
    CUtensorMap map_hi{}, map_lo{}; bool maps_ready = false;
    CUtensorMap map2_hi{}, map2_lo{}; bool maps2_ready = false;   // 128-row boxes: one CTA's half of a pair's W tile (gemm_mode 5)
};
struct LNp { float* g = nullptr; float* b = nullptr; };
struct EncLayerW { Lin qkv, o, fc1, fc2; LNp ln_attn, ln_final; };
struct DecLayerW { Lin qkv, o, cq, ckv, co, fc1, fc2; LNp ln_self, ln_cross, ln_final; };

// Every (re)allocation of a workspace buffer bumps this; a captured CUDA graph bakes buffer addresses in, so
// graphs captured under an older epoch are discarded.
uint64_t g_ws_epoch = 0;

struct Buf {
    void* p = nullptr; size_t bytes = 0;
    void ensure(size_t need) {
        if (need <= bytes) return;
        if (p) { cudaFree(p); p = nullptr; bytes = 0; }
        CUDA_CHECK(cudaMalloc(&p, need));
        bytes = need;
        ++g_ws_epoch;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

}  // namespace

struct sealbart {
    sealbart_config_t cfg{};
    int device = 0;
    float* shared = nullptr; float* enc_pos = nullptr; float* dec_pos = nullptr;
    float* lm_head = nullptr; float* final_bias = nullptr;
    bool lm_head_given = false;
    LNp enc_ln_emb, dec_ln_emb;
    Lin head;
    std::vector<EncLayerW> enc;
    std::vector<DecLayerW> dec;
    struct Slot { float* dst; uint64_t numel; };
    std::map<std::string, Slot> slots;
    std::set<std::string> loaded;
    std::vector<void*> allocs;
    uint64_t weight_bytes = 0;
    bool finalized = false;
    // workspace
    Buf enc_tok, enc_mask, ex, eqkv, eattn, etmp, effn, ckv, src_off;
    bool enc_packed = false;          // the last encoder_forward ran on the real tokens only (src_off valid)
    Buf dx, dqkv, dattn, dtmp, dcq, dffn, logits, kc, vc;
    Buf ex_hi, ex_lo, eattn_hi, eattn_lo, effn_hi, effn_lo, dx_hi, dx_lo, dattn_hi, dattn_lo, dffn_hi, dffn_lo;   // activation splits (halves or TF32)
    Buf st_scores, st_tokens, st_lo, st_hi, st_pw, st_anc, st_mask;
    Buf st_rowmax, st_rowls, st_rule, st_cval, st_cidx, st_ccnt, st_wide;     // scratch between the kernels of a step
    Buf hy_score, hy_len, hy_tok, hy_valid, hy_lo, hy_hi, err, dbg_ids, force_syms, a_hi, a_lo, splitk;
    std::vector<void*> split_allocs;
    int64_t launches = 0;
    int* ovf = nullptr;               // where the producers raise "fp16 range exceeded" (set by every entry point)
    double phase_us[5] = {0, 0, 0, 0, 0};
    bool profile_gemm = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> gemm_events;
    double gemm_flops = 0;
    std::vector<cudaEvent_t> events;
    // host-buffer entry point: persistent device staging of the inputs (stable addresses -> CUDA graph reuse)
    Buf in_ids, in_mask, in_occ;
    // CUDA graphs of whole generate calls (small batches are launch-latency-bound: ~1 900 kernels per generate)
    struct GraphEntry { std::vector<uint8_t> key; uint64_t epoch = 0; cudaGraphExec_t exec = nullptr; int64_t launches = 0; uint64_t stamp = 0; };
    std::vector<GraphEntry> graphs;
    std::vector<std::vector<uint8_t>> seen_keys;     // shapes run once already (their buffers are sized): capture next time
    uint64_t graph_stamp = 0;
    int graph_policy = -1;            // -1 auto (small batches), 0 never, 1 whenever possible
    int last_used_graph = 0;
    bool tf32_ready = false;          // 3xTF32 weight splits exist (gemm_mode 2 fallback after an fp16 range overflow)
    int64_t overflow_fallbacks = 0;
    cudaStream_t stream = nullptr;    // the host-buffer entry point's own (non-blocking) stream
};

namespace {

float* dalloc(sealbart* m, uint64_t numel) {
    void* p = nullptr;
    CUDA_CHECK(cudaMalloc(&p, std::max<uint64_t>(numel, 1) * sizeof(float)));
    CUDA_CHECK(cudaMemset(p, 0, std::max<uint64_t>(numel, 1) * sizeof(float)));
    m->allocs.push_back(p);
    m->weight_bytes += numel * sizeof(float);
    return static_cast<float*>(p);
}

void make_lin(sealbart* m, Lin& l, int out, int in) { l.out = out; l.in = in; l.w = dalloc(m, (uint64_t)out * in); l.b = dalloc(m, out); }
void make_ln(sealbart* m, LNp& l, int d) { l.g = dalloc(m, d); l.b = dalloc(m, d); }

void reg(sealbart* m, const std::string& key, float* dst, uint64_t numel) { m->slots[key] = {dst, numel}; }
void reg_lin(sealbart* m, const std::string& prefix, Lin& l, int row0, int rows) {
    reg(m, prefix + ".weight", l.w + (uint64_t)row0 * l.in, (uint64_t)rows * l.in);
    reg(m, prefix + ".bias", l.b + row0, rows);
}
void reg_ln(sealbart* m, const std::string& prefix, LNp& l, int d) {
    reg(m, prefix + ".weight", l.g, d);
    reg(m, prefix + ".bias", l.b, d);
}

void build_slots(sealbart* m) {
    const auto& c = m->cfg;
    const int d = c.d_model, f = c.ffn_dim, V = c.vocab_size, P = c.max_positions + 2;
    m->shared = dalloc(m, (uint64_t)V * d); reg(m, "model.shared.weight", m->shared, (uint64_t)V * d);
    m->enc_pos = dalloc(m, (uint64_t)P * d); reg(m, "model.encoder.embed_positions.weight", m->enc_pos, (uint64_t)P * d);
    m->dec_pos = dalloc(m, (uint64_t)P * d); reg(m, "model.decoder.embed_positions.weight", m->dec_pos, (uint64_t)P * d);
    m->final_bias = dalloc(m, V); reg(m, "final_logits_bias", m->final_bias, V);
    make_ln(m, m->enc_ln_emb, d); reg_ln(m, "model.encoder.layernorm_embedding", m->enc_ln_emb, d);
    make_ln(m, m->dec_ln_emb, d); reg_ln(m, "model.decoder.layernorm_embedding", m->dec_ln_emb, d);
    m->enc.resize(c.encoder_layers);
    for (int i = 0; i < c.encoder_layers; ++i) {
        EncLayerW& L = m->enc[i];
        const std::string p = "model.encoder.layers." + std::to_string(i) + ".";
        make_lin(m, L.qkv, 3 * d, d);
        reg_lin(m, p + "self_attn.q_proj", L.qkv, 0, d); reg_lin(m, p + "self_attn.k_proj", L.qkv, d, d);
        reg_lin(m, p + "self_attn.v_proj", L.qkv, 2 * d, d);
        make_lin(m, L.o, d, d); reg_lin(m, p + "self_attn.out_proj", L.o, 0, d);
        make_ln(m, L.ln_attn, d); reg_ln(m, p + "self_attn_layer_norm", L.ln_attn, d);
        make_lin(m, L.fc1, f, d); reg_lin(m, p + "fc1", L.fc1, 0, f);
        make_lin(m, L.fc2, d, f); reg_lin(m, p + "fc2", L.fc2, 0, d);
        make_ln(m, L.ln_final, d); reg_ln(m, p + "final_layer_norm", L.ln_final, d);
    }
    m->dec.resize(c.decoder_layers);
    for (int i = 0; i < c.decoder_layers; ++i) {
        DecLayerW& L = m->dec[i];
        const std::string p = "model.decoder.layers." + std::to_string(i) + ".";
        make_lin(m, L.qkv, 3 * d, d);
        reg_lin(m, p + "self_attn.q_proj", L.qkv, 0, d); reg_lin(m, p + "self_attn.k_proj", L.qkv, d, d);
        reg_lin(m, p + "self_attn.v_proj", L.qkv, 2 * d, d);
        make_lin(m, L.o, d, d); reg_lin(m, p + "self_attn.out_proj", L.o, 0, d);
        make_ln(m, L.ln_self, d); reg_ln(m, p + "self_attn_layer_norm", L.ln_self, d);
        make_lin(m, L.cq, d, d); reg_lin(m, p + "encoder_attn.q_proj", L.cq, 0, d);
        make_lin(m, L.ckv, 2 * d, d);
        reg_lin(m, p + "encoder_attn.k_proj", L.ckv, 0, d); reg_lin(m, p + "encoder_attn.v_proj", L.ckv, d, d);
        make_lin(m, L.co, d, d); reg_lin(m, p + "encoder_attn.out_proj", L.co, 0, d);
        make_ln(m, L.ln_cross, d); reg_ln(m, p + "encoder_attn_layer_norm", L.ln_cross, d);
        make_lin(m, L.fc1, f, d); reg_lin(m, p + "fc1", L.fc1, 0, f);
        make_lin(m, L.fc2, d, f); reg_lin(m, p + "fc2", L.fc2, 0, d);
        make_ln(m, L.ln_final, d); reg_ln(m, p + "final_layer_norm", L.ln_final, d);
    }
}

// ---- launch helpers ----------------------------------------------------------------------------
// pending: a split-K GEMM whose slices are still unsummed -- its consumer (add+LN on small batches, the attention kernels)
// folds the finish pass in; defer_rows = how many rows that consumer accepts (0: the GEMM must finish itself)
struct Ctx { sealbart* m; cudaStream_t s; SplitSrc pending{}; int64_t defer_rows = 0; };

// ---- TMA descriptors ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (!p || q != cudaDriverEntryPointSuccess) throw ApiError(SEALFM_ECUDA, "cuTensorMapEncodeTiled unavailable");
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}
// row-major [rows][K] fp32 (or fp16), box = row_bytes (128, 64 or 32) of K x box_rows, swizzled at the box's row width,
// zero fill out of bounds
void make_map(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t K, uint64_t ld, uint32_t box_rows, bool half = false,
              int row_bytes = 128) {
    cuuint64_t dims[2] = {K, rows};
    cuuint64_t strides[1] = {ld * (half ? 2 : 4)};
    cuuint32_t box[2] = {(cuuint32_t)(row_bytes / (half ? 2 : 4)), box_rows};
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapSwizzle sw = row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    CUresult r = encode_tiled()(map, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw ApiError(SEALFM_ECUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
}

constexpr int kUmmaBN = 256;
constexpr int64_t kAddLnRowMax = 2048;      // up to this many rows add+LN runs one CTA per row

void split_into(cudaStream_t s, const float* x, float* hi, float* lo, uint64_t numel) {
    const int64_t n4 = (int64_t)(numel / 4);
    const int blocks = (int)std::min<int64_t>((n4 + 255) / 256, (int64_t)sm_count() * 8);
    split_tf32_kernel<<<std::max(blocks, 1), 256, 0, s>>>(n4, reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(hi),
                                                          reinterpret_cast<float4*>(lo));
    CUDA_CHECK(cudaGetLastError());
}

// An activation tensor as the GEMMs see it: plain fp32 and/or its TF32 split (hi, lo).
struct Act {
    float* x = nullptr; float* hi = nullptr; float* lo = nullptr;   // fp32 / TF32 split
    __half* h1 = nullptr; __half* h2 = nullptr;                     // FP16 split
};

SplitOut split_of(const Act& a, int* overflow) {
    SplitOut so;
    if (a.hi) { so.a = a.hi; so.b = a.lo; so.kind = 1; }
    else if (a.h1) { so.a = a.h1; so.b = a.h2; so.kind = 2; so.overflow = overflow; }
    return so;
}

void umma_launch(cudaStream_t s, int64_t M, int N, int K, const CUtensorMap& ahi, const CUtensorMap& alo, const CUtensorMap& whi,
                 const CUtensorMap& wlo, const float* bias, const Act& C, int ldc, bool gelu) {
    using SMm = UmmaSmem<kUmmaBN>;
    const int tiles = (int)(((N + kUmmaBN - 1) / kUmmaBN) * ((M + UM - 1) / UM));
    const int ctas = std::min(tiles, sm_count());
    const int n_fastest = ((int64_t)M >= (int64_t)N) ? 1 : 0;     // stream the larger operand once
    if (gelu) {
        CUDA_CHECK(cudaFuncSetAttribute(umma_gemm_tf32x3_persistent_kernel<kUmmaBN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMm::kTotal));
        umma_gemm_tf32x3_persistent_kernel<kUmmaBN, true><<<ctas, UTHREADS2, SMm::kTotal, s>>>(ahi, alo, whi, wlo, (int)M, N, K, bias, C.x, C.hi, C.lo, ldc, n_fastest);
    } else {
        CUDA_CHECK(cudaFuncSetAttribute(umma_gemm_tf32x3_persistent_kernel<kUmmaBN, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMm::kTotal));
        umma_gemm_tf32x3_persistent_kernel<kUmmaBN, false><<<ctas, UTHREADS2, SMm::kTotal, s>>>(ahi, alo, whi, wlo, (int)M, N, K, bias, C.x, C.hi, C.lo, ldc, n_fastest);
    }
    CUDA_CHECK(cudaGetLastError());
}

// C = A W^T + b (+GELU) on the tensor cores: gemm_mode 3 / 5 = 3xFP16 (one CTA per tile / CTA pairs), 2 = 3xTF32 (fp32
// range: the fallback when an activation leaves the fp16 range).  Operands arrive pre-split from the producing kernel
// (A.h1/A.h2 or A.hi/A.lo); they are split here only if the producer did not.
void gemm_impl(Ctx& cx, int64_t M, int N, int K, const Act& A, int lda, Lin& l, const Act& C, int ldc, bool gelu);

void gemm(Ctx& cx, int64_t M, int N, int K, const Act& A, int lda, Lin& l, const Act& C, int ldc, bool gelu) {
    sealbart* m = cx.m;
    if (!m->profile_gemm || M == 0) { gemm_impl(cx, M, N, K, A, lda, l, C, ldc, gelu); return; }
    cudaEvent_t a, b;
    CUDA_CHECK(cudaEventCreate(&a)); CUDA_CHECK(cudaEventCreate(&b));
    CUDA_CHECK(cudaEventRecord(a, cx.s));
    gemm_impl(cx, M, N, K, A, lda, l, C, ldc, gelu);
    CUDA_CHECK(cudaEventRecord(b, cx.s));
    m->gemm_events.emplace_back(a, b);
    m->gemm_flops += 2.0 * (double)M * N * K;
}

void gemm_impl(Ctx& cx, int64_t M, int N, int K, const Act& A, int lda, Lin& l, const Act& C, int ldc, bool gelu) {
    if (M == 0) return;
    sealbart* m = cx.m;
    if (m->cfg.gemm_mode >= 3 && K % UK16 == 0 && lda == K && l.w_h1) {
        constexpr int rowb = 128;                              // 128-byte shared-memory rows: 64 K-halves per k-block
        // 3xFP16 on tcgen05 (persistent); operands pre-split into halves by the producers
        const __half* a1 = A.h1; const __half* a2 = A.h2;
        if (!a1) {
            m->a_hi.ensure((size_t)M * K * 2); m->a_lo.ensure((size_t)M * K * 2);
            const int blocks = (int)std::min<int64_t>(((int64_t)M * K + 255) / 256, (int64_t)sm_count() * 8);
            split_half_kernel<<<blocks, 256, 0, cx.s>>>((int64_t)M * K, A.x, 1.0f, m->a_hi.as<__half>(), m->a_lo.as<__half>(), m->ovf);
            CUDA_CHECK(cudaGetLastError()); m->launches++;
            a1 = m->a_hi.as<__half>(); a2 = m->a_lo.as<__half>();
        }
        CUtensorMap ma1, ma2;
        make_map(&ma1, a1, M, K, K, UM, true, rowb); make_map(&ma2, a2, M, K, K, UM, true, rowb);
        if (!l.maps_ready) { make_map(&l.map_hi, l.w_h1, N, K, K, kUmmaBN, true, rowb); make_map(&l.map_lo, l.w_h2, N, K, K, kUmmaBN, true, rowb); l.maps_ready = true; }
        using SMm = UmmaSmem<kUmmaBN>;
        const int tiles = (int)(((N + kUmmaBN - 1) / kUmmaBN) * ((M + UM - 1) / UM));
        const int ctas = std::min(tiles, sm_count());
        const int n_fastest = ((int64_t)M >= (int64_t)N) ? 1 : 0;
        int* ovf = m->ovf;
        // skinny problems (a few tiles for 148 SMs): split K so that the serial K loop of a tile is spread
        // over up to 8 CTAs, then sum the partial tiles in a fixed order
        const int kblocks = K / (rowb / 2);
        int k_slices = 1;
        static const int force_slices = [] { const char* e = std::getenv("SEALB200_KSLICES"); return e ? std::atoi(e) : 0; }();
        if (tiles * 2 <= sm_count() && kblocks >= 4) {
            k_slices = std::min(8, std::min(kblocks / 2, sm_count() / tiles));
            if (force_slices > 0) k_slices = std::min(force_slices, kblocks);     // experiments only
            while (k_slices > 1 && kblocks % k_slices) --k_slices;
        }
        if (m->cfg.gemm_mode == 5 && k_slices == 1 && M > UM) {
            // CTA pairs (cluster of 2, tcgen05.mma.cta_group::2) on 256 x 256 tiles: a third less operand
            // traffic out of L2 per MMA than the one-CTA kernel (umma_gemm_2cta.cuh)
            if (!l.maps2_ready) { make_map(&l.map2_hi, l.w_h1, N, K, K, 128, true, 128); make_map(&l.map2_lo, l.w_h2, N, K, K, 128, true, 128); l.maps2_ready = true; }
            const int m_tiles = (int)((M + UM - 1) / UM), n_tiles = (N + kUmmaBN - 1) / kUmmaBN;
            const int pair_tiles = ((m_tiles + 1) / 2) * n_tiles;
            const int pairs = std::min(pair_tiles, sm_count() / 2);
            // wave quantisation: when the last round of pair-tiles would keep less than half of the pairs busy, those
            // tiles are cut into K slices (one short round instead of a full one) and summed by a finish kernel
            int full_items = pair_tiles, tail_s = 1;
            static const bool tail_split = [] { const char* e = std::getenv("SEALB200_TAIL_SPLIT"); return !e || std::atoi(e) != 0; }();
            const int rem = pair_tiles % pairs;
            if (tail_split && pair_tiles > pairs && rem > 0 && rem * 2 <= pairs) {
                int sl = std::min(8, pairs / rem);
                const int nk = K / 64;
                while (sl > 1 && (nk % sl || nk / sl < 2)) --sl;
                if (sl > 1) { tail_s = sl; full_items = pair_tiles - rem; }
            }
            float* part = nullptr;
            if (tail_s > 1) { m->splitk.ensure((size_t)(pair_tiles - full_items) * tail_s * 65536 * 4); part = m->splitk.as<float>(); }
            // the epilogue stores boxes of 16 columns x 32 rows (umma_gemm_2cta.cuh); maps are passed by value, so a
            // captured graph replays them as long as the buffers keep their addresses (g_ws_epoch)
            const bool split_out = C.h1 != nullptr;
            if (split_out == (C.x != nullptr) || (split_out && !C.h2)) throw ApiError(SEALFM_EINVAL, "internal: the CTA-pair GEMM writes either fp32 or fp16 halves");
            CUtensorMap mo1, mo2, mpart;
            if (split_out) { make_map(&mo1, C.h1, M, N, ldc, 32, true, 32); make_map(&mo2, C.h2, M, N, ldc, 32, true, 32); }
            else { make_map(&mo1, C.x, M, N, ldc, 32, false, 64); mo2 = mo1; }
            if (part) make_map(&mpart, part, (uint64_t)(pair_tiles - full_items) * tail_s * 256, 256, 256, 32, false, 64);
            else mpart = mo1;
            auto launchp = [&](auto kern) {
                CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, U2_SMEM));
                launch_k(kern, 2 * pairs, UTHREADS2, U2_SMEM, cx.s, ma1, ma2, l.map2_hi, l.map2_lo, mo1, mo2, mpart, (int)M, N, K, l.b, l.w_unscale,
                         (int)split_out, n_fastest, ovf, full_items, tail_s);
            };
            if (gelu) launchp(umma_gemm_f16x3_2cta_kernel<true>); else launchp(umma_gemm_f16x3_2cta_kernel<false>);
            CUDA_CHECK(cudaGetLastError()); m->launches++;
            if (tail_s > 1) {
                const int fb = (pair_tiles - full_items) * 64;
                const int pm_tiles = (m_tiles + 1) / 2;
                if (gelu) launch_k(umma_tail_finish_kernel<true>, fb, 256, 0, cx.s, (int)M, N, ldc, n_tiles, pm_tiles, n_fastest, full_items, tail_s, part, l.b, l.w_unscale, C.x, C.h1, C.h2, ovf);
                else launch_k(umma_tail_finish_kernel<false>, fb, 256, 0, cx.s, (int)M, N, ldc, n_tiles, pm_tiles, n_fastest, full_items, tail_s, part, l.b, l.w_unscale, C.x, C.h1, C.h2, ovf);
                CUDA_CHECK(cudaGetLastError()); m->launches++;
            }
            return;
        }
        if (k_slices > 1) {
            const int64_t slice_stride = (int64_t)M * ldc;
            m->splitk.ensure((size_t)k_slices * slice_stride * 4);
            float* part = m->splitk.as<float>();
            const int ctas2 = std::min(tiles * k_slices, sm_count());
            auto launch2 = [&](auto kern) {
                CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMm::kTotalStaged));
                launch_k(kern, ctas2, UTHREADS2, SMm::kTotalStaged, cx.s, ma1, ma2, l.map_hi, l.map_lo, (int)M, N, K, nullptr, 1.0f, part, nullptr, nullptr,
                           ldc, n_fastest, ovf, k_slices, slice_stride);
            };
            launch2(umma_gemm_f16x3_persistent_kernel<kUmmaBN, false, 128>);
            CUDA_CHECK(cudaGetLastError()); m->launches++;
            if (M <= cx.defer_rows && !gelu && !C.h1 && !C.hi && ldc == N && l.b) {     // summed by the consumer kernel
                cx.pending = SplitSrc{part, k_slices, slice_stride, l.b, l.w_unscale};
                return;
            }
            const int fblocks = (int)std::min<int64_t>((M * (ldc / 4) + 255) / 256, (int64_t)sm_count() * 8);
            if (gelu) launch_k(umma_splitk_finish_kernel<true>, fblocks, 256, 0, cx.s, M, N, ldc, k_slices, slice_stride, part, l.b, l.w_unscale, C.x, C.h1, C.h2, ovf);
            else launch_k(umma_splitk_finish_kernel<false>, fblocks, 256, 0, cx.s, M, N, ldc, k_slices, slice_stride, part, l.b, l.w_unscale, C.x, C.h1, C.h2, ovf);
            CUDA_CHECK(cudaGetLastError()); m->launches++;
            return;
        }
        auto launch = [&](auto kern) {
            CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMm::kTotalStaged));
            launch_k(kern, ctas, UTHREADS2, SMm::kTotalStaged, cx.s, ma1, ma2, l.map_hi, l.map_lo, (int)M, N, K, l.b, l.w_unscale, C.x, C.h1, C.h2, ldc, n_fastest, ovf, 1, (int64_t)0);
        };
        if (gelu) launch(umma_gemm_f16x3_persistent_kernel<kUmmaBN, true, 128>); else launch(umma_gemm_f16x3_persistent_kernel<kUmmaBN, false, 128>);
        CUDA_CHECK(cudaGetLastError()); m->launches++;
        return;
    }
    if (m->cfg.gemm_mode == 2 && K % UK == 0 && lda == K && l.w_hi) {
        const float* ahi = A.hi; const float* alo = A.lo;
        if (!ahi) {
            m->a_hi.ensure((size_t)M * K * 4); m->a_lo.ensure((size_t)M * K * 4);
            split_into(cx.s, A.x, m->a_hi.as<float>(), m->a_lo.as<float>(), (uint64_t)M * K); m->launches++;
            ahi = m->a_hi.as<float>(); alo = m->a_lo.as<float>();
        }
        CUtensorMap mah, mal;
        make_map(&mah, ahi, M, K, K, UM); make_map(&mal, alo, M, K, K, UM);
        if (!l.maps_ready) { make_map(&l.map_hi, l.w_hi, N, K, K, kUmmaBN); make_map(&l.map_lo, l.w_lo, N, K, K, kUmmaBN); l.maps_ready = true; }
        umma_launch(cx.s, M, N, K, mah, mal, l.map_hi, l.map_lo, l.b, C, ldc, gelu);
        m->launches++;
        return;
    }
    throw ApiError(SEALFM_EINVAL, "GEMM: K must be a multiple of 64 (3xFP16) / 32 (3xTF32) with contiguous operands");
}

void add_ln(Ctx& cx, int64_t rows, int d, const float* a, const float* b, const LNp& ln, const Act& out) {
    const SplitSrc ps = cx.pending;
    cx.pending = SplitSrc{};
    if (rows <= kAddLnRowMax)          // small batches: a CTA per row (and the split-K finish of the GEMM before it, if pending)
        launch_k(add_ln_row_kernel, (unsigned)rows, 128, 0, cx.s, rows, d, a, b, (const float*)ln.g, (const float*)ln.b, out.x,
                 split_of(out, cx.m->ovf), ps);
    else
        launch_k(add_ln_kernel, (unsigned)((rows + 3) / 4), 128, 0, cx.s, rows, d, a, b, (const float*)ln.g, (const float*)ln.b, out.x, split_of(out, cx.m->ovf));
    cx.m->launches++;
}

__global__ void prep_enc_kernel(int64_t n, int S, const int64_t* __restrict__ ids, const int64_t* __restrict__ mask,
                                int32_t* __restrict__ tok, int32_t* __restrict__ m32, int32_t* __restrict__ pos) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    tok[i] = (int32_t)ids[i];
    m32[i] = mask[i] != 0;
    pos[i] = (int32_t)(i % S);
}

// Source lengths, their exclusive prefix sum (src_off[Q+1]) and whether every mask row is "ones then zeros"
// (right padding) -- the precondition for running the encoder on the real tokens only.  One block.
__global__ void __launch_bounds__(1024) pack_lengths_kernel(int64_t Q, int S, const int64_t* __restrict__ mask,
                                                            int32_t* __restrict__ src_off, int64_t* __restrict__ info,
                                                            int64_t hint, int32_t* __restrict__ hint_err) {
    __shared__ int64_t part[1024];
    __shared__ int bad;
    const int t = threadIdx.x;
    if (t == 0) bad = 0;
    __syncthreads();
    const int64_t per = (Q + 1023) / 1024, q0 = t * per, q1 = q0 + per < Q ? q0 + per : Q;
    int64_t sum = 0; int notprefix = 0;
    for (int64_t q = q0; q < q1; ++q) {
        int len = 0;
        for (int s2 = 0; s2 < S; ++s2) { const int on = mask[q * S + s2] != 0; if (on && s2 != len) notprefix = 1; len += on; }
        sum += len;
    }
    part[t] = sum;
    if (notprefix) atomicExch(&bad, 1);
    __syncthreads();
    if (t == 0) {
        int64_t run = 0;
        for (int i = 0; i < 1024; ++i) { const int64_t v = part[i]; part[i] = run; run += v; }
        info[0] = run; info[1] = bad;
        if (hint >= 0 && hint_err && (run != hint || bad)) *hint_err = 1;      // the caller's token count was wrong
    }
    __syncthreads();
    int64_t run = part[t];
    for (int64_t q = q0; q < q1; ++q) {
        src_off[q] = (int32_t)run;
        int len = 0;
        for (int s2 = 0; s2 < S; ++s2) len += mask[q * S + s2] != 0;
        run += len;
    }
    if (t == 0) src_off[Q] = (int32_t)info[0];
}

__global__ void prep_enc_packed_kernel(int64_t n, int S, const int64_t* __restrict__ ids, const int32_t* __restrict__ src_off,
                                       int32_t* __restrict__ tok, int32_t* __restrict__ pos) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t q = i / S; const int s2 = (int)(i % S);
    if (s2 < src_off[q + 1] - src_off[q]) { const int64_t dst = src_off[q] + s2; tok[dst] = (int32_t)ids[i]; pos[dst] = s2; }
}

__global__ void init_state_kernel(int64_t R, int B, int T, int start_tok, int pad, uint64_t lo0, uint64_t hi0,
                                  float* __restrict__ scores, int32_t* __restrict__ tokens, uint64_t* __restrict__ lo,
                                  uint64_t* __restrict__ hi, uint64_t* __restrict__ pw, int32_t* __restrict__ anc) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= R) return;
    scores[r] = (r % B) == 0 ? 0.f : -1e9f;                 // seal/beam_search.py:214-216
    for (int t = 0; t < T; ++t) { tokens[r * T + t] = t == 0 ? start_tok : pad; anc[r * T + t] = (int32_t)r; }
    lo[r] = lo0; hi[r] = hi0; pw[r] = hi0 - lo0;
}

__global__ void ids_to_tokens_kernel(int64_t R, int t, int T, const int64_t* __restrict__ ids, int32_t* __restrict__ tokens,
                                     int32_t* __restrict__ anc) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= R) return;
    for (int i = 0; i < T; ++i) { tokens[r * T + i] = i < t ? (int32_t)ids[r * t + i] : 0; anc[r * T + i] = (int32_t)r; }
}

struct Dims {
    int64_t Q, S, R; int B, T, d, f, V, ld, W;
    int64_t G = 0; const int32_t* grp_query = nullptr; const int32_t* grp_start = nullptr;   // ragged row groups (re-scoring)
};

void ensure_workspace(sealbart* m, const Dims& D) {
    const int64_t Tk = D.Q * D.S;
    const int Ld = m->cfg.decoder_layers;
    m->enc_tok.ensure(Tk * 4 * 2); m->enc_mask.ensure(Tk * 4); m->src_off.ensure((D.Q + 1) * 4 + 16 + 16);
    m->ex.ensure(Tk * D.d * 4); m->eqkv.ensure(Tk * 3 * D.d * 4); m->eattn.ensure(Tk * D.d * 4);
    m->etmp.ensure(Tk * D.d * 4); m->effn.ensure(Tk * D.f * 4);
    m->ckv.ensure((size_t)Ld * Tk * 2 * D.d * 4);
    m->dx.ensure(D.R * D.d * 4); m->dqkv.ensure(D.R * 3 * D.d * 4); m->dattn.ensure(D.R * D.d * 4);
    m->dtmp.ensure(D.R * D.d * 4); m->dcq.ensure(D.R * D.d * 4); m->dffn.ensure(D.R * D.f * 4);
    m->logits.ensure((size_t)D.R * D.ld * 4);
    m->kc.ensure((size_t)Ld * D.T * D.R * D.d * 4); m->vc.ensure((size_t)Ld * D.T * D.R * D.d * 4);
    m->st_scores.ensure(2 * D.R * 4); m->st_tokens.ensure(2 * D.R * D.T * 4);
    m->st_lo.ensure(2 * D.R * 8); m->st_hi.ensure(2 * D.R * 8); m->st_pw.ensure(2 * D.R * 8);
    m->st_anc.ensure(2 * D.R * D.T * 4); m->st_mask.ensure((size_t)2 * D.R * D.W * 4);
    m->st_rowmax.ensure(D.R * 4); m->st_rowls.ensure(D.R * 4); m->st_rule.ensure(D.R);
    m->st_cval.ensure((size_t)D.R * 2 * D.B * 4); m->st_cidx.ensure((size_t)D.R * 2 * D.B * 4); m->st_ccnt.ensure(D.R * 4);
    {
        m->ex_hi.ensure(Tk * D.d * 4); m->ex_lo.ensure(Tk * D.d * 4);
        m->eattn_hi.ensure(Tk * D.d * 4); m->eattn_lo.ensure(Tk * D.d * 4);
        m->effn_hi.ensure(Tk * D.f * 4); m->effn_lo.ensure(Tk * D.f * 4);
        m->dx_hi.ensure(D.R * D.d * 4); m->dx_lo.ensure(D.R * D.d * 4);
        m->dattn_hi.ensure(D.R * D.d * 4); m->dattn_lo.ensure(D.R * D.d * 4);
        m->dffn_hi.ensure(D.R * D.f * 4); m->dffn_lo.ensure(D.R * D.f * 4);
    }
    m->err.ensure(16);
}

// src_tokens_hint: >= 0 the caller's count of real source tokens (right-padded masks): no host synchronisation, the
// kernel that derives the offsets checks it and raises err_d[2] on a mismatch; -1 unknown: one 16-byte read-back;
// -2 do not pack (padded rows are computed; also no synchronisation).
void encoder_forward(Ctx& cx, const Dims& D, const int64_t* ids_d, const int64_t* mask_d, int64_t src_tokens_hint = -1,
                     int32_t* hint_err = nullptr) {
    sealbart* m = cx.m;
    const int64_t Tk = D.Q * D.S;
    const int d = D.d;
    int32_t* tok = m->enc_tok.as<int32_t>(); int32_t* pos = tok + Tk; int32_t* m32 = m->enc_mask.as<int32_t>();
    // Padding is not computed: with right-padded sources (the only kind SEAL produces) the encoder and the
    // cross-attention K/V projections run on the sum of the real lengths P instead of Q * S_max rows
    // (29 % fewer at S ~ U[12, 28]); query q's states are rows src_off[q] .. src_off[q+1] everywhere downstream.
    static const bool pack_enabled = [] { const char* e = std::getenv("SEALB200_PACK_ENCODER"); return !e || std::atoi(e) != 0; }();
    int32_t* src_off = m->src_off.as<int32_t>();
    int64_t* info_d = reinterpret_cast<int64_t*>(reinterpret_cast<char*>(m->src_off.p) + ((D.Q + 1) * 4 + 15) / 16 * 16);
    int64_t rows_enc = Tk;
    m->enc_packed = false;
    if (pack_enabled && src_tokens_hint != -2) {
        pack_lengths_kernel<<<1, 1024, 0, cx.s>>>(D.Q, (int)D.S, mask_d, src_off, info_d, src_tokens_hint, hint_err);
        CUDA_CHECK(cudaGetLastError()); m->launches++;
        if (src_tokens_hint > 0) { m->enc_packed = true; rows_enc = src_tokens_hint; }
        else {
            int64_t info[2] = {0, 1};
            CUDA_CHECK(cudaMemcpyAsync(info, info_d, 16, cudaMemcpyDeviceToHost, cx.s));
            CUDA_CHECK(cudaStreamSynchronize(cx.s));
            if (info[1] == 0 && info[0] > 0) { m->enc_packed = true; rows_enc = info[0]; }
        }
    }
    const int32_t* soff = m->enc_packed ? src_off : nullptr;
    if (m->enc_packed) prep_enc_packed_kernel<<<(unsigned)((Tk + 255) / 256), 256, 0, cx.s>>>(Tk, (int)D.S, ids_d, src_off, tok, pos);
    else prep_enc_kernel<<<(unsigned)((Tk + 255) / 256), 256, 0, cx.s>>>(Tk, (int)D.S, ids_d, mask_d, tok, m32, pos);
    CUDA_CHECK(cudaGetLastError()); m->launches++;
    const int64_t Te = rows_enc;                    // encoder rows actually computed
    const int gm = m->cfg.gemm_mode;
    auto mk = [&](float* plain, Buf& bh, Buf& bl, bool keep_plain) {
        Act a;
        if (keep_plain) a.x = plain;
        if (gm == 2) { a.hi = bh.as<float>(); a.lo = bl.as<float>(); }
        if (gm >= 3) { a.h1 = bh.as<__half>(); a.h2 = bl.as<__half>(); }
        return a;
    };
    int* ovf = m->ovf;
    const Act x = mk(m->ex.as<float>(), m->ex_hi, m->ex_lo, true);
    const Act qkv{m->eqkv.as<float>()};
    const Act attn = mk(m->eattn.as<float>(), m->eattn_hi, m->eattn_lo, false);
    const Act tmp{m->etmp.as<float>()};
    const Act ffn = mk(m->effn.as<float>(), m->effn_hi, m->effn_lo, false);
    const float scale = m->cfg.scale_embedding ? sqrtf((float)d) : 1.0f;
    embed_ln_kernel<<<(unsigned)((Te + 3) / 4), 128, 0, cx.s>>>(Te, d, tok, 1, pos, 0, m->shared, scale, m->enc_pos,
                                                                m->enc_ln_emb.g, m->enc_ln_emb.b, x.x, split_of(x, ovf));
    CUDA_CHECK(cudaGetLastError()); m->launches++;
    const int heads = m->cfg.heads;
    for (auto& L : m->enc) {
        gemm(cx, Te, 3 * d, d, x, d, L.qkv, qkv, 3 * d, false);
        enc_self_attn_kernel<<<dim3((unsigned)D.Q, heads), kGAttnWarps * 32, 0, cx.s>>>(D.Q, d, heads, (int)D.S, qkv.x, m32, attn.x, split_of(attn, ovf), soff);
        CUDA_CHECK(cudaGetLastError()); m->launches++;
        cx.defer_rows = kAddLnRowMax;
        gemm(cx, Te, d, d, attn, d, L.o, tmp, d, false);
        cx.defer_rows = 0;
        add_ln(cx, Te, d, x.x, tmp.x, L.ln_attn, x);
        gemm(cx, Te, D.f, d, x, d, L.fc1, ffn, D.f, true);
        cx.defer_rows = kAddLnRowMax;
        gemm(cx, Te, d, D.f, ffn, D.f, L.fc2, tmp, d, false);
        cx.defer_rows = 0;
        add_ln(cx, Te, d, x.x, tmp.x, L.ln_final, x);
    }
    // per-query cross-attention K/V of every decoder layer, once (the reference recomputes nothing
    // either: HF caches them after the first step)
    for (int l = 0; l < m->cfg.decoder_layers; ++l)
        gemm(cx, Te, 2 * d, d, x, d, m->dec[l].ckv, Act{m->ckv.as<float>() + (size_t)l * Tk * 2 * d}, 2 * d, false);
}

// one decoder step for all R rows: token at position pos = cur_len-1 -> logits [R][ld]
// `compact` (first step of a generate only): every beam of a query is the same row there (same start token, same
// source), so the step runs on one row per query -- Q rows instead of Q*B -- and the select kernel reads that
// row's logits for all of the query's beams (StepCfg::logits_shared); the k / v of position 0 are written to the
// cache entries of all B beams.  1/T of the decoder + lm_head work disappears (~8 % of a 9-step generate).
void decoder_step(Ctx& cx, const Dims& D, const int32_t* tokens, int cur_len, const int32_t* anc, bool want_logits,
                  cudaEvent_t ev_layers_done, bool compact = false) {
    sealbart* m = cx.m;
    const int d = D.d; const int64_t Rc = D.R; const int64_t Tk = D.Q * D.S;
    if (compact && (cur_len != 1 || D.grp_start)) throw ApiError(SEALFM_EINVAL, "internal: compact step only at position 0 of a generate");
    const int64_t R = compact ? D.Q : D.R;          // rows processed
    const int row_mul = compact ? D.B : 1;
    const int pos = cur_len - 1;
    const int gm = m->cfg.gemm_mode;
    auto mk = [&](float* plain, Buf& bh, Buf& bl, bool keep_plain) {
        Act a;
        if (keep_plain) a.x = plain;
        if (gm == 2) { a.hi = bh.as<float>(); a.lo = bl.as<float>(); }
        if (gm >= 3) { a.h1 = bh.as<__half>(); a.h2 = bl.as<__half>(); }
        return a;
    };
    int* ovf = m->ovf;
    const Act x = mk(m->dx.as<float>(), m->dx_hi, m->dx_lo, true);
    const Act qkv{m->dqkv.as<float>()};
    const Act attn = mk(m->dattn.as<float>(), m->dattn_hi, m->dattn_lo, false);
    const Act tmp{m->dtmp.as<float>()};
    const Act cq{m->dcq.as<float>()};
    const Act ffn = mk(m->dffn.as<float>(), m->dffn_hi, m->dffn_lo, false);
    const float scale = m->cfg.scale_embedding ? sqrtf((float)d) : 1.0f;
    launch_k(embed_ln_kernel, (unsigned)((R + 3) / 4), 128, 0, cx.s, R, d, tokens + pos, (int64_t)(D.T * row_mul), (const int32_t*)nullptr, pos,
               (const float*)m->shared, scale, (const float*)m->dec_pos, (const float*)m->dec_ln_emb.g, (const float*)m->dec_ln_emb.b, x.x, split_of(x, ovf));
    m->launches++;
    const int heads = m->cfg.heads;
    const int32_t* m32 = m->enc_mask.as<int32_t>();
    for (int l = 0; l < m->cfg.decoder_layers; ++l) {
        DecLayerW& L = m->dec[l];
        float* kc = m->kc.as<float>() + (size_t)l * D.T * Rc * d;
        float* vc = m->vc.as<float>() + (size_t)l * D.T * Rc * d;
        // the beams of a query together, distinct ancestors staged once (not at the compact first step, where a row
        // stands for all beams, nor for ragged re-scoring groups)
        static const bool sa_query = [] { const char* e = std::getenv("SEALB200_SELF_ATTN_QUERY"); return !e || std::atoi(e) != 0; }();
        const size_t saq_smem = self_attn_query_smem(pos + 1, D.B);
        const bool use_saq = sa_query && !compact && !D.grp_start && pos >= 1 && D.B >= 2 && D.B <= 32 && pos + 1 <= 128 && saq_smem <= 112 * 1024;
        cx.defer_rows = use_saq ? INT64_MAX : 0;               // that kernel sums a split-K qkv itself
        gemm(cx, R, 3 * d, d, x, d, L.qkv, qkv, 3 * d, false);
        cx.defer_rows = 0;
        const SplitSrc qkv_src = cx.pending;
        cx.pending = SplitSrc{};
        const unsigned sa_threads = 32 * std::min(heads, 16);
        if (use_saq) {
            static size_t saq_set = 0;
            if (saq_smem > saq_set) { CUDA_CHECK(cudaFuncSetAttribute(dec_self_attn_query_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024)); saq_set = 112 * 1024; }
            launch_k(dec_self_attn_query_kernel, dim3((unsigned)D.Q, heads), 32 * D.B, saq_smem, cx.s, Rc, D.B, d, pos, D.T, (const float*)qkv.x, kc, vc, anc,
                     attn.x, split_of(attn, ovf), qkv_src);
        } else if (pos + 1 <= 12)
            launch_k(dec_self_attn_kernel<3>, (unsigned)R, sa_threads, 0, cx.s, Rc, d, heads, pos, D.T, (const float*)qkv.x, kc, vc, anc, attn.x, split_of(attn, ovf), row_mul, row_mul);
        else if (pos + 1 <= 32)
            launch_k(dec_self_attn_kernel<8>, (unsigned)R, sa_threads, 0, cx.s, Rc, d, heads, pos, D.T, (const float*)qkv.x, kc, vc, anc, attn.x, split_of(attn, ovf), row_mul, row_mul);
        else
            launch_k(dec_self_attn_long_kernel, (unsigned)R, sa_threads, 0, cx.s, Rc, d, heads, pos, D.T, (const float*)qkv.x, kc, vc, anc, attn.x, split_of(attn, ovf));
        m->launches++;
        cx.defer_rows = kAddLnRowMax;
        gemm(cx, R, d, d, attn, d, L.o, tmp, d, false);
        cx.defer_rows = 0;
        add_ln(cx, R, d, x.x, tmp.x, L.ln_self, x);
        cx.defer_rows = (D.S <= kXKeys) ? INT64_MAX : 0;      // cross_attn_small_kernel sums a split-K cq itself
        gemm(cx, R, d, d, x, d, L.cq, cq, d, false);
        cx.defer_rows = 0;
        const SplitSrc cq_src = cx.pending;
        cx.pending = SplitSrc{};
        const int64_t groups = D.grp_start ? D.G : D.Q;
        const float* ckv_l = m->ckv.as<float>() + (size_t)l * Tk * 2 * d;
        const int32_t* soff_x = m->enc_packed ? m->src_off.as<int32_t>() : nullptr;
        if (D.S <= kXKeys)
            launch_k(cross_attn_small_kernel, dim3((unsigned)groups, heads), 128, 0, cx.s, groups, d, heads, compact ? 1 : D.B, (int)D.S, (const float*)cq.x,
                       ckv_l, m32, D.grp_query, D.grp_start, attn.x, split_of(attn, ovf), soff_x, cq_src);
        else
            launch_k(cross_attn_kernel, dim3((unsigned)groups, heads), kGAttnWarps * 32, 0, cx.s, groups, d, heads, compact ? 1 : D.B, (int)D.S, (const float*)cq.x,
                       ckv_l, m32, D.grp_query, D.grp_start, attn.x, split_of(attn, ovf), soff_x);
        m->launches++;
        cx.defer_rows = kAddLnRowMax;
        gemm(cx, R, d, d, attn, d, L.co, tmp, d, false);
        cx.defer_rows = 0;
        add_ln(cx, R, d, x.x, tmp.x, L.ln_cross, x);
        gemm(cx, R, D.f, d, x, d, L.fc1, ffn, D.f, true);
        cx.defer_rows = kAddLnRowMax;
        gemm(cx, R, d, D.f, ffn, D.f, L.fc2, tmp, d, false);
        cx.defer_rows = 0;
        add_ln(cx, R, d, x.x, tmp.x, L.ln_final, x);
    }
    if (ev_layers_done) CUDA_CHECK(cudaEventRecord(ev_layers_done, cx.s));
    if (want_logits) gemm(cx, R, D.V, d, x, d, m->head, Act{m->logits.as<float>()}, D.ld, false);
}

void check_model(const sealbart* m) {
    if (!m) throw ApiError(SEALFM_EINVAL, "null model");
    if (!m->finalized) throw ApiError(SEALFM_EINVAL, "sealbart_finalize not called");
    CUDA_CHECK(cudaSetDevice(m->device));
}

Dims make_dims(const sealbart* m, int64_t Q, int64_t S, int B, int T) {
    Dims D;
    D.Q = Q; D.S = S; D.B = B; D.R = Q * B; D.T = T;
    D.d = m->cfg.d_model; D.f = m->cfg.ffn_dim; D.V = m->cfg.vocab_size;
    D.ld = (D.V + 3) / 4 * 4; D.W = (D.V + 31) / 32;
    return D;
}

cudaEvent_t new_event(sealbart* m) {
    cudaEvent_t e; CUDA_CHECK(cudaEventCreate(&e)); m->events.push_back(e); return e;
}


template <typename Fn> void for_each_lin(sealbart* m, Fn&& fn) {
    for (auto& L : m->enc) { fn(L.qkv); fn(L.o); fn(L.fc1); fn(L.fc2); }
    for (auto& L : m->dec) { fn(L.qkv); fn(L.o); fn(L.cq); fn(L.ckv); fn(L.co); fn(L.fc1); fn(L.fc2); }
    fn(m->head);
}

// 3xTF32 operand copies of every weight matrix (gemm_mode 1 / 2; also the range-safe fallback of the 3xFP16 modes)
void ensure_tf32_splits(sealbart* m) {
    if (m->tf32_ready) return;
    CUDA_CHECK(cudaSetDevice(m->device));
    for_each_lin(m, [&](Lin& l) {
        const uint64_t n = (uint64_t)l.out * l.in;
        CUDA_CHECK(cudaMalloc(&l.w_hi, n * 4)); m->split_allocs.push_back(l.w_hi);
        CUDA_CHECK(cudaMalloc(&l.w_lo, n * 4)); m->split_allocs.push_back(l.w_lo);
        split_into(nullptr, l.w, l.w_hi, l.w_lo, n);
        m->weight_bytes += 2 * n * 4;
    });
    CUDA_CHECK(cudaDeviceSynchronize());
    m->tf32_ready = true;
}

}  // namespace

extern "C" {

int sealbart_create(const sealbart_config_t* cfg, int device, sealbart_t** out) {
    return guarded([&] {
        if (!cfg || !out) throw ApiError(SEALFM_EINVAL, "null argument");
        if (cfg->d_model % 128 || cfg->d_model > 1024 || cfg->heads * kHeadDim != cfg->d_model)
            throw ApiError(SEALFM_EINVAL, "d_model must be a multiple of 128, <= 1024, with 64-wide heads");
        if (cfg->ffn_dim % 64 || cfg->vocab_size <= 0) throw ApiError(SEALFM_EINVAL, "bad ffn_dim / vocab_size");
        if (cfg->gemm_mode != 2 && cfg->gemm_mode != 3 && cfg->gemm_mode != 5)
            throw ApiError(SEALFM_EINVAL, "gemm_mode must be 5 (3xFP16 on CTA pairs, default), 3 (3xFP16, one CTA per tile) or 2 (3xTF32)");
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) { cudaGetLastError(); throw ApiError(SEALFM_ENODEVICE, "no CUDA device available"); }
        if (device < 0 || device >= count) throw ApiError(SEALFM_EINVAL, "bad device id");
        CUDA_CHECK(cudaSetDevice(device));
        std::unique_ptr<sealbart> m(new sealbart());
        m->cfg = *cfg; m->device = device;
        build_slots(m.get());
        *out = m.release();
    });
}

void sealbart_free(sealbart_t* m) {
    if (!m) return;
    cudaSetDevice(m->device);
    for (void* p : m->allocs) cudaFree(p);
    for (void* p : m->split_allocs) cudaFree(p);
    if (m->lm_head_given) cudaFree(m->lm_head);
    for (Buf* b : {&m->enc_tok, &m->enc_mask, &m->src_off, &m->ex, &m->eqkv, &m->eattn, &m->etmp, &m->effn, &m->ckv, &m->dx, &m->dqkv,
                   &m->dattn, &m->dtmp, &m->dcq, &m->dffn, &m->logits, &m->kc, &m->vc, &m->st_scores, &m->st_tokens,
                   &m->st_lo, &m->st_hi, &m->st_pw, &m->st_anc, &m->st_mask, &m->st_rowmax, &m->st_rowls, &m->st_rule, &m->st_cval,
                   &m->st_cidx, &m->st_ccnt, &m->st_wide, &m->hy_score, &m->hy_len, &m->hy_tok,
                   &m->hy_valid, &m->hy_lo, &m->hy_hi, &m->err, &m->dbg_ids, &m->force_syms, &m->a_hi, &m->a_lo, &m->ex_hi, &m->ex_lo,
                   &m->eattn_hi, &m->eattn_lo, &m->effn_hi, &m->effn_lo, &m->dx_hi, &m->dx_lo, &m->dattn_hi, &m->dattn_lo,
                   &m->dffn_hi, &m->dffn_lo, &m->splitk})
        b->release();
    for (auto e : m->events) cudaEventDestroy(e);
    for (auto& g : m->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    for (Buf* b : {&m->in_ids, &m->in_mask, &m->in_occ}) b->release();
    if (m->stream) cudaStreamDestroy(m->stream);
    delete m;
}

int sealbart_set_tensor(sealbart_t* m, const char* key, const float* host, uint64_t numel) {
    return guarded([&] {
        if (!m || !key || !host) throw ApiError(SEALFM_EINVAL, "null argument");
        CUDA_CHECK(cudaSetDevice(m->device));
        std::string k(key);
        if (k == "lm_head.weight") {
            const uint64_t want = (uint64_t)m->cfg.vocab_size * m->cfg.d_model;
            if (numel != want) throw ApiError(SEALFM_EINVAL, "lm_head.weight: wrong size");
            if (!m->lm_head_given) { CUDA_CHECK(cudaMalloc(&m->lm_head, want * 4)); m->lm_head_given = true; m->weight_bytes += want * 4; }
            CUDA_CHECK(cudaMemcpy(m->lm_head, host, want * 4, cudaMemcpyHostToDevice));
            return;
        }
        if (k == "model.encoder.embed_tokens.weight" || k == "model.decoder.embed_tokens.weight") k = "model.shared.weight";
        auto it = m->slots.find(k);
        if (it == m->slots.end()) throw ApiError(SEALFM_EINVAL, "unknown state_dict key: " + k);
        if (it->second.numel != numel) throw ApiError(SEALFM_EINVAL, "wrong element count for " + k);
        CUDA_CHECK(cudaMemcpy(it->second.dst, host, numel * 4, cudaMemcpyHostToDevice));
        m->loaded.insert(k);
        m->finalized = false;
    });
}

int sealbart_finalize(sealbart_t* m) {
    return guarded([&] {
        if (!m) throw ApiError(SEALFM_EINVAL, "null model");
        for (auto& kv : m->slots)
            if (!m->loaded.count(kv.first)) throw ApiError(SEALFM_EINVAL, "state_dict tensor missing: " + kv.first);
        if (!m->lm_head_given) m->lm_head = m->shared;          // tied (seal/utils.py:48-49)
        m->head.w = m->lm_head; m->head.b = m->final_bias; m->head.out = m->cfg.vocab_size; m->head.in = m->cfg.d_model;
        {
            CUDA_CHECK(cudaSetDevice(m->device));
            for (void* p : m->split_allocs) cudaFree(p);
            m->split_allocs.clear();
            m->tf32_ready = false;
            for_each_lin(m, [](Lin& l) { l.maps_ready = false; l.maps2_ready = false; });
            unsigned int* d_max = nullptr;
            if (m->cfg.gemm_mode >= 3) { CUDA_CHECK(cudaMalloc(&d_max, 4)); m->err.ensure(16); CUDA_CHECK(cudaMemset(m->err.p, 0, 16)); }
            auto split_lin_half = [&](Lin& l) {
                const uint64_t n = (uint64_t)l.out * l.in;
                CUDA_CHECK(cudaMemset(d_max, 0, 4));
                absmax_kernel<<<sm_count() * 4, 256>>>((int64_t)n, l.w, d_max);
                unsigned int bits = 0; CUDA_CHECK(cudaMemcpy(&bits, d_max, 4, cudaMemcpyDeviceToHost));
                float mx; std::memcpy(&mx, &bits, 4);
                int sexp = 0;
                if (mx > 0.f) { int e; std::frexp(mx, &e); sexp = 14 - e; }      // max|W| * 2^s in [2^13, 2^14)
                l.w_unscale = std::ldexp(1.0f, -sexp);
                CUDA_CHECK(cudaMalloc(&l.w_h1, n * 2)); m->split_allocs.push_back(l.w_h1);
                CUDA_CHECK(cudaMalloc(&l.w_h2, n * 2)); m->split_allocs.push_back(l.w_h2);
                split_half_kernel<<<sm_count() * 8, 256>>>((int64_t)n, l.w, std::ldexp(1.0f, sexp), l.w_h1, l.w_h2, m->err.as<int>() + 1);
                CUDA_CHECK(cudaGetLastError());
                l.maps_ready = false;
                m->weight_bytes += 2 * n * 2;
            };
            if (m->cfg.gemm_mode >= 3) {
                for (auto& L : m->enc) { split_lin_half(L.qkv); split_lin_half(L.o); split_lin_half(L.fc1); split_lin_half(L.fc2); }
                for (auto& L : m->dec) { split_lin_half(L.qkv); split_lin_half(L.o); split_lin_half(L.cq); split_lin_half(L.ckv); split_lin_half(L.co); split_lin_half(L.fc1); split_lin_half(L.fc2); }
                split_lin_half(m->head);
                CUDA_CHECK(cudaDeviceSynchronize());
                cudaFree(d_max);
                m->finalized = true;
                return;
            }
            ensure_tf32_splits(m);
        }
        m->finalized = true;
    });
}

uint64_t sealbart_device_bytes(const sealbart_t* m) { return m ? m->weight_bytes : 0; }

int64_t sealdec_hyps_per_query(const sealdec_params_t* p) {
    if (!p) return 0;
    return (int64_t)(p->max_length - 1) * 2 * p->num_beams + p->num_beams;
}


}  // extern "C"

namespace {

struct GenArgs {
    const sealfm_t* fm; const uint32_t* occ_d; const sealdec_params_t* p;
    const int64_t* ids_d; const int64_t* mask_d; int64_t Q, S;
    float* o_score; int32_t* o_len; int32_t* o_tok; uint8_t* o_valid; uint64_t* o_lo; uint64_t* o_hi; int32_t* err_d;
};

// Enqueues one whole generate (encoder, every decode step, records) on cx.s.  No host synchronisation unless
// src_hint == -1.  `timing` = bracket the phases with CUDA events (not possible while the stream is being captured).
void generate_enqueue(Ctx& cx, const Dims& D, const GenArgs& a, const FmView& view, uint64_t lo0, uint64_t hi0,
                      int64_t src_hint, bool timing) {
    sealbart* m = cx.m;
    const sealdec_params_t* p = a.p;
    const int B = D.B, K = 2 * B, T = D.T;
    const int64_t Q = D.Q, R = D.R;
    for (auto e : m->events) cudaEventDestroy(e);
    m->events.clear();
    auto mark = [&]() -> cudaEvent_t {
        if (!timing) return nullptr;
        cudaEvent_t e = new_event(m);
        CUDA_CHECK(cudaEventRecord(e, cx.s));
        return e;
    };
    CUDA_CHECK(cudaMemsetAsync(a.err_d, 0, 16, cx.s));
    mark();
    encoder_forward(cx, D, a.ids_d, a.mask_d, src_hint, a.err_d + 2);
    mark();

    float* sc[2] = {m->st_scores.as<float>(), m->st_scores.as<float>() + R};
    int32_t* tk[2] = {m->st_tokens.as<int32_t>(), m->st_tokens.as<int32_t>() + R * T};
    uint64_t* lo[2] = {m->st_lo.as<uint64_t>(), m->st_lo.as<uint64_t>() + R};
    uint64_t* hi[2] = {m->st_hi.as<uint64_t>(), m->st_hi.as<uint64_t>() + R};
    uint64_t* pw[2] = {m->st_pw.as<uint64_t>(), m->st_pw.as<uint64_t>() + R};
    int32_t* an[2] = {m->st_anc.as<int32_t>(), m->st_anc.as<int32_t>() + R * T};
    uint32_t* mk[2] = {m->st_mask.as<uint32_t>(), m->st_mask.as<uint32_t>() + (size_t)R * D.W};
    init_state_kernel<<<(unsigned)((R + 255) / 256), 256, 0, cx.s>>>(R, B, T, p->decoder_start_token_id, p->pad_token_id,
                                                                    lo0, hi0, sc[0], tk[0], lo[0], hi[0], pw[0], an[0]);
    CUDA_CHECK(cudaGetLastError()); m->launches++;

    StepCfg c{};
    c.num_beams = B; c.K = K; c.V = D.V; c.ld = D.ld;
    c.min_length = p->min_length; c.max_length = p->max_length;
    c.eos_token_id = p->eos_token_id; c.pad_token_id = p->pad_token_id; c.model_eos_token_id = p->model_eos_token_id;
    c.forced_eos_token_id = p->forced_eos_token_id; c.forced_bos_token_id = p->forced_bos_token_id;
    c.stop_at_count = p->stop_at_count; c.always_allow_eos = p->always_allow_eos; c.disable_fm_index = p->disable_fm_index;
    c.remove_invalid_values = p->remove_invalid_values; c.shift = p->shift; c.T = T; c.mask_words = D.W;
    c.hyps_per_query = sealdec_hyps_per_query(p);
    using RowsFirst = SelSharedT<8192>; using RowsLater = SelSharedT<4096>;
    CUDA_CHECK(cudaFuncSetAttribute(topk_rows_kernel<512, 8192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RowsFirst)));
    CUDA_CHECK(cudaFuncSetAttribute(topk_rows_kernel<256, 4096>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RowsLater)));
    RowScratch rs{m->st_rowmax.as<float>(), m->st_rowls.as<float>(), m->st_rule.as<uint8_t>(),
                  m->st_cval.as<float>(), m->st_cidx.as<int32_t>(), m->st_ccnt.as<int32_t>()};
    int cur = 0;
    for (int step = 0; step + 1 < T; ++step) {
        const int cur_len = step + 1;
        mark();
        static const bool compact_first = [] { const char* e = std::getenv("SEALB200_COMPACT_FIRST"); return !e || std::atoi(e) != 0; }();
        const bool compact = compact_first && cur_len == 1;
        // Dead step: when ForcedEOSTokenLogitsProcessor fires (cur_len == max_length - 1, HF semantics restated
        // in apply_processors) it overwrites EVERY processed score with a constant, so neither the recorded
        // hypotheses nor the (already final) beams depend on the model output of this step -- the reference
        // computes it and discards it.  Nothing later reads this position's k / v either.
        static const bool skip_dead = [] { const char* e = std::getenv("SEALB200_SKIP_DEAD_STEP"); return !e || std::atoi(e) != 0; }();
        const bool forced_all = p->forced_eos_token_id >= 0 && cur_len == p->max_length - 1 && cur_len + 1 == T &&
                                !(p->forced_bos_token_id >= 0 && cur_len == 1);
        const bool dead = skip_dead && forced_all;
        cudaEvent_t b = timing ? new_event(m) : nullptr;
        if (!dead) decoder_step(cx, D, tk[cur], cur_len, an[cur], true, b, compact);
        else if (b) CUDA_CHECK(cudaEventRecord(b, cx.s));
        mark();
        c.cur_len = cur_len;
        c.logits_shared = (compact && !dead) ? 1 : 0;
        c.logits_ignored = dead ? 1 : 0;
        const int eff_len = cur_len - (p->forced_bos_token_id >= 0 ? 1 : 0);
        c.first_step_shared_mask = (!p->disable_fm_index && eff_len == 1) ? 1 : 0;
        c.expand_next = (cur_len + 1 < T) ? 1 : 0;
        c.hyp_base = step * K;
        StepState st{};
        st.beam_scores_in = sc[cur]; st.beam_scores_out = sc[cur ^ 1];
        st.tokens_in = tk[cur]; st.tokens_out = tk[cur ^ 1];
        st.lo_in = lo[cur]; st.lo_out = lo[cur ^ 1]; st.hi_in = hi[cur]; st.hi_out = hi[cur ^ 1];
        st.pw_in = pw[cur]; st.pw_out = pw[cur ^ 1];
        st.anc_in = an[cur]; st.anc_out = an[cur ^ 1];
        st.mask_in = mk[cur]; st.mask_out = mk[cur ^ 1];
        st.occurring_mask = a.occ_d; st.logits = m->logits.as<float>();
        st.hyp_score = a.o_score; st.hyp_len = a.o_len; st.hyp_tokens = a.o_tok; st.hyp_valid = a.o_valid;
        st.hyp_lo = a.o_lo; st.hyp_hi = a.o_hi; st.error_flag = a.err_d;
        // first step: beams 1.. carry -1e9 and are pruned exactly inside one CTA per query; afterwards one CTA per row
        if (cur_len == 1) {
            launch_k(topk_rows_kernel<512, 8192>, (unsigned)Q, 512, sizeof(RowsFirst), cx.s, c, st, rs, 1, B);
            launch_k(select_merge_kernel, (unsigned)Q, kMergeThreads, 0, cx.s, view, c, st, rs, 1);
        } else {
            launch_k(topk_rows_kernel<256, 4096>, (unsigned)R, 256, sizeof(RowsLater), cx.s, c, st, rs, B, 1);
            launch_k(select_merge_kernel, (unsigned)Q, kMergeThreads, 0, cx.s, view, c, st, rs, B);
        }
        m->launches += 2;
        if (c.expand_next && !p->disable_fm_index) {           // successor sets of the new beams -> next step's masks (:107)
            launch_expand_masks(view, cx.s, (uint64_t)R, lo[cur ^ 1], hi[cur ^ 1], mk[cur ^ 1], (uint32_t)D.W, (uint32_t)D.V,
                                (uint32_t)p->shift, m->st_wide.as<unsigned long long>());
            m->launches += 2;
        }
        mark();
        cur ^= 1;
    }
    c.cur_len = T; c.hyp_base = (T - 1) * K;
    StepState st{};
    st.hyp_score = a.o_score; st.hyp_len = a.o_len; st.hyp_tokens = a.o_tok; st.hyp_valid = a.o_valid; st.hyp_lo = a.o_lo; st.hyp_hi = a.o_hi;
    finalize_kernel<<<(unsigned)((R + 255) / 256), 256, 0, cx.s>>>(Q, c, sc[cur], tk[cur], lo[cur], hi[cur], st);
    CUDA_CHECK(cudaGetLastError()); m->launches++;
    mark();
    // events in creation order: ev0, ev_enc, then per step a, b, c, d, then end (sealdec_last_phase_us)
}

template <typename T> void key_put(std::vector<uint8_t>& k, const T& v) {
    const uint8_t* b = reinterpret_cast<const uint8_t*>(&v);
    k.insert(k.end(), b, b + sizeof(T));
}

void drop_graphs(sealbart* m) {
    for (auto& g : m->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    m->graphs.clear();
    m->seen_keys.clear();
}

}  // namespace

extern "C" {

int sealdec_generate_dx(sealbart_t* m, const sealfm_t* fm, const uint32_t* occ_d, const sealdec_params_t* p,
                        const int64_t* ids_d, const int64_t* mask_d, int64_t Q, int64_t S, sealfm_stream_t stream,
                        float* o_score, int32_t* o_len, int32_t* o_tok, uint8_t* o_valid, uint64_t* o_lo,
                        uint64_t* o_hi, int32_t* err_d, int64_t src_tokens_hint) {
    return guarded([&] {
        check_model(m);
        if (!p || !ids_d || !mask_d || !o_score || !o_len || !o_tok || !o_valid || !err_d) throw ApiError(SEALFM_EINVAL, "null argument");
        const int B = p->num_beams, K = 2 * B, T = p->max_length;
        if (B < 1 || B > kSelMaxBeams || K > kSelMaxK) throw ApiError(SEALFM_EINVAL, "num_beams must be in [1,32]");
        if (T < 2 || T > kMaxLen) throw ApiError(SEALFM_EINVAL, "max_length must be in [2,128]");
        if (Q <= 0 || S <= 0) throw ApiError(SEALFM_EINVAL, "empty batch");
        if (S > m->cfg.max_positions) throw ApiError(SEALFM_EINVAL, "source longer than max_positions");
        if (src_tokens_hint < -2 || src_tokens_hint > Q * S) throw ApiError(SEALFM_EINVAL, "bad source-token hint");
        FmView view{};
        uint64_t lo0 = 0, hi0 = 0;
        if (!p->disable_fm_index) {
            if (!fm || sealfm_device(fm) != m->device) throw ApiError(SEALFM_ENODEVICE, "FM index not bound to the model's device");
            if (!occ_d) throw ApiError(SEALFM_EINVAL, "occurring mask missing");
            view = sealfm_view(fm);
            lo0 = 0; hi0 = view.m + 1;                               // get_range([]) = (0, size()+1)  (index.py:106-110)
            if (p->n_force_decoding_from > 0) {
                std::vector<uint64_t> q(p->n_force_decoding_from), off{0, (uint64_t)p->n_force_decoding_from};
                for (int i = 0; i < p->n_force_decoding_from; ++i) q[i] = (uint64_t)p->force_decoding_from[i] + p->shift;
                int rc = sealfm_backward_search_multi(fm, 1, q.data(), off.data(), &lo0, &hi0);
                if (rc) throw ApiError(rc, sealfm_last_error());
            }
        }
        Ctx cx{m, (cudaStream_t)stream};
        m->launches = 0;
        m->ovf = err_d + 1;
        m->last_used_graph = 0;
        const Dims D = make_dims(m, Q, S, B, T);
        ensure_workspace(m, D);
        if (!p->disable_fm_index) m->st_wide.ensure(expand_scratch_bytes(view.L, (uint64_t)D.R));   // wide-row work list + BFS frontiers
        const GenArgs a{fm, occ_d, p, ids_d, mask_d, Q, S, o_score, o_len, o_tok, o_valid, o_lo, o_hi, err_d};

        // ---- CUDA graph of the whole call: a batch-20 generate is ~1 900 short kernels, i.e. launch-latency-bound.
        // Shapes, parameters and buffer addresses are the key; the first call of a key runs eagerly (it sizes every
        // lazily grown buffer), the second is captured, later ones are one cudaGraphLaunch.
        static const int env_graph = [] { const char* e = std::getenv("SEALB200_GRAPH"); return e ? std::atoi(e) : -1; }();
        const int policy = m->graph_policy >= 0 ? m->graph_policy : env_graph;
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cx.s) CUDA_CHECK(cudaStreamIsCapturing(cx.s, &cap));
        const bool small = D.R <= 4096;
        bool want_graph = cx.s != nullptr && cap == cudaStreamCaptureStatusNone && !m->profile_gemm &&
                          (policy == 1 || (policy < 0 && small));
        // inside a graph the encoder never needs the host: small batches compute the padded rows (the key then does
        // not depend on the batch's contents), larger ones use the caller's token count
        int64_t eff_hint = src_tokens_hint;
        if (want_graph) { if (small) eff_hint = -2; else if (src_tokens_hint == -1) want_graph = false; }
        if (!want_graph) { generate_enqueue(cx, D, a, view, lo0, hi0, eff_hint, cap == cudaStreamCaptureStatusNone); m->phase_us[0] = -1; return; }

        std::vector<uint8_t> key;
        key_put(key, Q); key_put(key, S); key_put(key, eff_hint); key_put(key, lo0); key_put(key, hi0);
        key_put(key, m->cfg.gemm_mode); key_put(key, cx.s);
        sealdec_params_t pc = *p; pc.force_decoding_from = nullptr; key_put(key, pc);
        for (int i = 0; i < p->n_force_decoding_from; ++i) key_put(key, p->force_decoding_from[i]);
        key_put(key, view.blocks); key_put(key, view.csym); key_put(key, view.node_tab); key_put(key, view.m);
        key_put(key, occ_d); key_put(key, ids_d); key_put(key, mask_d); key_put(key, o_score); key_put(key, o_len);
        key_put(key, o_tok); key_put(key, o_valid); key_put(key, o_lo); key_put(key, o_hi); key_put(key, err_d);
        if (!m->graphs.empty() && m->graphs.front().epoch != g_ws_epoch) drop_graphs(m);
        for (auto& g : m->graphs)
            if (g.key == key) {
                CUDA_CHECK(cudaGraphLaunch(g.exec, cx.s));
                g.stamp = ++m->graph_stamp; m->launches = g.launches; m->last_used_graph = 1;
                return;
            }
        bool seen = false;
        for (auto& k2 : m->seen_keys) if (k2 == key) { seen = true; break; }
        if (!seen) {                                           // first time: eager (sizes split-K / staging buffers)
            if (m->seen_keys.size() >= 16) m->seen_keys.erase(m->seen_keys.begin());
            m->seen_keys.push_back(key);
            generate_enqueue(cx, D, a, view, lo0, hi0, eff_hint, true);
            m->phase_us[0] = -1;
            return;
        }
        const uint64_t epoch0 = g_ws_epoch;
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        bool captured = false;
        if (cudaStreamBeginCapture(cx.s, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
            try {
                generate_enqueue(cx, D, a, view, lo0, hi0, eff_hint, false);
                captured = cudaStreamEndCapture(cx.s, &graph) == cudaSuccess && graph != nullptr;
            } catch (...) {
                cudaStreamEndCapture(cx.s, &graph);
                captured = false;
            }
            if (captured && g_ws_epoch == epoch0) captured = cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
            else captured = false;
            if (graph) cudaGraphDestroy(graph);
        }
        if (!captured) {
            // a buffer moved while capturing, or this driver cannot capture / instantiate the call (the launches were
            // only recorded, nothing ran): run it the ordinary way, and stop trying on this model
            cudaGetLastError();
            if (g_ws_epoch == epoch0) m->graph_policy = 0;
            m->launches = 0;
            generate_enqueue(cx, D, a, view, lo0, hi0, eff_hint, true);
            return;
        }
        if (m->graphs.size() >= 8) {                           // evict the least recently used
            size_t victim = 0;
            for (size_t i = 1; i < m->graphs.size(); ++i) if (m->graphs[i].stamp < m->graphs[victim].stamp) victim = i;
            cudaGraphExecDestroy(m->graphs[victim].exec);
            m->graphs.erase(m->graphs.begin() + victim);
        }
        sealbart::GraphEntry ge; ge.key = std::move(key); ge.epoch = g_ws_epoch; ge.exec = exec; ge.launches = m->launches; ge.stamp = ++m->graph_stamp;
        m->graphs.push_back(std::move(ge));
        CUDA_CHECK(cudaGraphLaunch(exec, cx.s));
        m->last_used_graph = 1;
    });
}

int sealdec_generate_d(sealbart_t* m, const sealfm_t* fm, const uint32_t* occ_d, const sealdec_params_t* p,
                       const int64_t* ids_d, const int64_t* mask_d, int64_t Q, int64_t S, sealfm_stream_t stream,
                       float* o_score, int32_t* o_len, int32_t* o_tok, uint8_t* o_valid, uint64_t* o_lo,
                       uint64_t* o_hi, int32_t* err_d) {
    return sealdec_generate_dx(m, fm, occ_d, p, ids_d, mask_d, Q, S, stream, o_score, o_len, o_tok, o_valid, o_lo, o_hi, err_d, -1);
}

int sealbart_set_option(sealbart_t* m, const char* name, int64_t value) {
    return guarded([&] {
        if (!m || !name) throw ApiError(SEALFM_EINVAL, "null argument");
        const std::string n(name);
        if (n == "cuda_graph") { if (value < -1 || value > 1) throw ApiError(SEALFM_EINVAL, "cuda_graph: -1 auto, 0 off, 1 on"); m->graph_policy = (int)value; }
        else if (n == "gemm_mode") {
            check_model(m);
            if (value == m->cfg.gemm_mode) return;
            if (value == 2 && m->cfg.gemm_mode >= 3) { ensure_tf32_splits(m); m->cfg.gemm_mode = 2; }
            else if ((value == 3 || value == 5) && m->head.w_h1) m->cfg.gemm_mode = (int)value;
            else throw ApiError(SEALFM_EINVAL, "gemm_mode can only switch between the 3xFP16 modes (3, 5) and 2 (3xTF32)");
            for_each_lin(m, [](Lin& l) { l.maps_ready = false; l.maps2_ready = false; });
            drop_graphs(m);
        }
        else throw ApiError(SEALFM_EINVAL, "unknown option: " + n);
    });
}

int64_t sealbart_get_stat(const sealbart_t* m, const char* name) {
    if (!m || !name) return -1;
    const std::string n(name);
    if (n == "last_used_graph") return m->last_used_graph;
    if (n == "overflow_fallbacks") return m->overflow_fallbacks;
    if (n == "gemm_mode") return m->cfg.gemm_mode;
    if (n == "cached_graphs") return (int64_t)m->graphs.size();
    return -1;
}

int sealdec_last_phase_us(const sealbart_t* mc, double out5[5]) {
    return guarded([&] {
        sealbart* m = const_cast<sealbart*>(mc);
        if (!m || !out5) throw ApiError(SEALFM_EINVAL, "null argument");
        CUDA_CHECK(cudaSetDevice(m->device));
        const size_t n = m->events.size();
        if (n < 3) throw ApiError(SEALFM_EINVAL, "no generate call recorded");
        CUDA_CHECK(cudaEventSynchronize(m->events[n - 1]));
        auto ms = [&](size_t a, size_t b) { float t = 0; CUDA_CHECK(cudaEventElapsedTime(&t, m->events[a], m->events[b])); return (double)t * 1e3; };
        double enc = ms(0, 1), layers = 0, head = 0, sel = 0;
        for (size_t i = 2; i + 3 < n; i += 4) { layers += ms(i, i + 1); head += ms(i + 1, i + 2); sel += ms(i + 2, i + 3); }
        out5[0] = enc; out5[1] = layers; out5[2] = head; out5[3] = sel; out5[4] = ms(0, n - 1);
    });
}

int sealdec_debug_gemm_trace(int enable, int64_t out20[20]) {
    return guarded([&] {
        if (out20) {
            CUDA_CHECK(cudaDeviceSynchronize());
            long long h[20];
            CUDA_CHECK(cudaMemcpyFromSymbol(h, g_gemm_trace, sizeof(h)));
            for (int i = 0; i < 20; ++i) out20[i] = h[i];
        }
        const int on = enable ? 1 : 0;
        CUDA_CHECK(cudaMemcpyToSymbol(g_gemm_trace_on, &on, sizeof(int)));
    });
}

int64_t sealdec_last_launch_count(const sealbart_t* m) { return m ? m->launches : 0; }

int sealdec_profile_gemm(sealbart_t* m, int enable, double* total_us, int64_t* launches, double* flops) {
    return guarded([&] {
        if (!m) throw ApiError(SEALFM_EINVAL, "null model");
        CUDA_CHECK(cudaSetDevice(m->device));
        if (total_us && launches && flops) {
            CUDA_CHECK(cudaDeviceSynchronize());
            double us = 0;
            for (auto& e : m->gemm_events) { float ms = 0; CUDA_CHECK(cudaEventElapsedTime(&ms, e.first, e.second)); us += (double)ms * 1e3; }
            *total_us = us; *launches = (int64_t)m->gemm_events.size(); *flops = m->gemm_flops;
        }
        for (auto& e : m->gemm_events) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
        m->gemm_events.clear(); m->gemm_flops = 0;
        m->profile_gemm = enable != 0;
    });
}

int sealdec_generate(sealbart_t* m, const sealfm_t* fm, const uint32_t* occ_host, const sealdec_params_t* p,
                     const int64_t* ids, const int64_t* mask, int64_t Q, int64_t S, float* o_score, int32_t* o_len,
                     int32_t* o_tok, uint8_t* o_valid, uint64_t* o_lo, uint64_t* o_hi) {
    return guarded([&] {
        check_model(m);
        if (!p || !ids || !mask || Q <= 0 || S <= 0) throw ApiError(SEALFM_EINVAL, "null argument / empty batch");
        const int64_t H = sealdec_hyps_per_query(p), T = p->max_length;
        const int W = (m->cfg.vocab_size + 31) / 32;
        // the caller's buffers are host memory: the real-token count costs nothing to know here, so the encoder
        // never has to ask the device for it (right-padded masks only; anything else takes the padded path)
        int64_t hint = 0;
        for (int64_t q = 0; q < Q && hint >= 0; ++q) {
            int64_t len = 0;
            for (int64_t s2 = 0; s2 < S; ++s2) { const bool on = mask[q * S + s2] != 0; if (on && s2 != len) { hint = -2; break; } len += on; }
            if (hint >= 0) hint += len;
        }
        if (hint == 0) hint = -2;
        if (!m->stream) CUDA_CHECK(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
        cudaStream_t s = m->stream;
        m->in_ids.ensure(Q * S * 8); m->in_mask.ensure(Q * S * 8); m->in_occ.ensure((size_t)W * 4);
        m->hy_score.ensure(Q * H * 4); m->hy_len.ensure(Q * H * 4); m->hy_tok.ensure(Q * H * T * 4);
        m->hy_valid.ensure(Q * H); m->hy_lo.ensure(Q * H * 8); m->hy_hi.ensure(Q * H * 8); m->err.ensure(16);
        CUDA_CHECK(cudaMemcpyAsync(m->in_ids.p, ids, Q * S * 8, cudaMemcpyHostToDevice, s));
        CUDA_CHECK(cudaMemcpyAsync(m->in_mask.p, mask, Q * S * 8, cudaMemcpyHostToDevice, s));
        if (occ_host) CUDA_CHECK(cudaMemcpyAsync(m->in_occ.p, occ_host, (size_t)W * 4, cudaMemcpyHostToDevice, s));
        int32_t errs[4] = {0, 0, 0, 0};
        for (int attempt = 0; attempt < 2; ++attempt) {
            int rc = sealdec_generate_dx(m, fm, occ_host ? m->in_occ.as<uint32_t>() : nullptr, p, m->in_ids.as<int64_t>(),
                                         m->in_mask.as<int64_t>(), Q, S, s, m->hy_score.as<float>(), m->hy_len.as<int32_t>(),
                                         m->hy_tok.as<int32_t>(), m->hy_valid.as<uint8_t>(), o_lo ? m->hy_lo.as<uint64_t>() : nullptr,
                                         o_hi ? m->hy_hi.as<uint64_t>() : nullptr, m->err.as<int32_t>(), hint);
            if (rc) throw ApiError(rc, last_error());
            CUDA_CHECK(cudaMemcpyAsync(errs, m->err.p, 16, cudaMemcpyDeviceToHost, s));
            CUDA_CHECK(cudaStreamSynchronize(s));
            if (!errs[1] || m->cfg.gemm_mode < 3) break;
            // An activation left the fp16 range (|x| > 65504; the producers saturate and raise the flag): this pass is
            // redone with the 3xTF32 kernels, which have fp32's range -- the caller gets exact-range results either way.
            const int mode = m->cfg.gemm_mode;
            { const int r0 = sealbart_set_option(m, "gemm_mode", 2); if (r0) throw ApiError(r0, last_error()); }
            m->overflow_fallbacks++;
            rc = sealdec_generate_dx(m, fm, occ_host ? m->in_occ.as<uint32_t>() : nullptr, p, m->in_ids.as<int64_t>(),
                                     m->in_mask.as<int64_t>(), Q, S, s, m->hy_score.as<float>(), m->hy_len.as<int32_t>(),
                                     m->hy_tok.as<int32_t>(), m->hy_valid.as<uint8_t>(), o_lo ? m->hy_lo.as<uint64_t>() : nullptr,
                                     o_hi ? m->hy_hi.as<uint64_t>() : nullptr, m->err.as<int32_t>(), hint);
            const int rc2 = sealbart_set_option(m, "gemm_mode", mode);
            if (rc) throw ApiError(rc, last_error());
            if (rc2) throw ApiError(rc2, last_error());
            CUDA_CHECK(cudaMemcpyAsync(errs, m->err.p, 16, cudaMemcpyDeviceToHost, s));
            CUDA_CHECK(cudaStreamSynchronize(s));
            break;
        }
        CUDA_CHECK(cudaMemcpyAsync(o_score, m->hy_score.p, Q * H * 4, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaMemcpyAsync(o_len, m->hy_len.p, Q * H * 4, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaMemcpyAsync(o_tok, m->hy_tok.p, Q * H * T * 4, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaMemcpyAsync(o_valid, m->hy_valid.p, Q * H, cudaMemcpyDeviceToHost, s));
        if (o_lo) CUDA_CHECK(cudaMemcpyAsync(o_lo, m->hy_lo.p, Q * H * 8, cudaMemcpyDeviceToHost, s));
        if (o_hi) CUDA_CHECK(cudaMemcpyAsync(o_hi, m->hy_hi.p, Q * H * 8, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        if (errs[2]) throw ApiError(SEALFM_EINVAL, "internal: source-token count mismatch");
        if (errs[0]) throw ApiError(SEALFM_EINVAL, "beam: fewer than num_beams non-EOS candidates (seal/beam_search.py:687-690)");
    });
}

int sealdec_debug_step_logits(sealbart_t* m, const int64_t* ids, const int64_t* mask, int64_t Q, int64_t S, int32_t B,
                              const int64_t* dec_ids, int64_t t, float* out_logits) {
    return guarded([&] {
        check_model(m);
        if (!ids || !mask || !dec_ids || !out_logits || t < 1 || t > kMaxLen) throw ApiError(SEALFM_EINVAL, "bad argument");
        const int T = (int)t;
        const Dims D = make_dims(m, Q, S, B, T);
        ensure_workspace(m, D);
        m->ovf = m->err.as<int>() + 1;
        Buf d_ids, d_mask;
        d_ids.ensure(Q * S * 8); d_mask.ensure(Q * S * 8); m->dbg_ids.ensure(D.R * t * 8);
        struct Rel { Buf *a, *b; ~Rel() { a->release(); b->release(); } } rel{&d_ids, &d_mask};
        cudaStream_t s = nullptr;
        CUDA_CHECK(cudaMemcpyAsync(d_ids.p, ids, Q * S * 8, cudaMemcpyHostToDevice, s));
        CUDA_CHECK(cudaMemcpyAsync(d_mask.p, mask, Q * S * 8, cudaMemcpyHostToDevice, s));
        CUDA_CHECK(cudaMemcpyAsync(m->dbg_ids.p, dec_ids, D.R * t * 8, cudaMemcpyHostToDevice, s));
        Ctx cx{m, s};
        m->launches = 0;
        encoder_forward(cx, D, d_ids.as<int64_t>(), d_mask.as<int64_t>());
        int32_t* tk = m->st_tokens.as<int32_t>(); int32_t* an = m->st_anc.as<int32_t>();
        ids_to_tokens_kernel<<<(unsigned)((D.R + 255) / 256), 256, 0, s>>>(D.R, T, T, m->dbg_ids.as<int64_t>(), tk, an);
        CUDA_CHECK(cudaGetLastError());
        for (int cur_len = 1; cur_len <= T; ++cur_len) decoder_step(cx, D, tk, cur_len, an, cur_len == T, nullptr);
        CUDA_CHECK(cudaMemcpy2DAsync(out_logits, (size_t)D.V * 4, m->logits.p, (size_t)D.ld * 4, (size_t)D.V * 4, D.R,
                                     cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
    });
}

int sealdec_teacher_forced(sealbart_t* m, const int64_t* ids, const int64_t* mask, int64_t Q, int64_t S,
                           const int64_t* dec_ids, const int32_t* row_query, int64_t N, int64_t T, float temperature,
                           float* out_logprob, int64_t out_full_pos, float* out_full) {
    return guarded([&] {
        check_model(m);
        if (!ids || !mask || !dec_ids || !row_query || N <= 0 || T < 1 || T > kMaxLen || Q <= 0 || S <= 0)
            throw ApiError(SEALFM_EINVAL, "bad argument");
        if (S > m->cfg.max_positions) throw ApiError(SEALFM_EINVAL, "source longer than max_positions");
        for (int64_t r = 0; r < N; ++r) {
            if (row_query[r] < 0 || row_query[r] >= Q || (r && row_query[r] < row_query[r - 1]))
                throw ApiError(SEALFM_EINVAL, "row_query must be sorted and within [0, Q)");
        }
        const int64_t kChunk = 4096;                           // decoder rows per pass (logits: 4096 x V floats)
        Dims D = make_dims(m, Q, S, 1, (int)T);
        D.R = std::min<int64_t>(N, kChunk);
        ensure_workspace(m, D);
        m->ovf = m->err.as<int>() + 1;
        cudaStream_t s = nullptr;
        Buf d_ids, d_mask, d_dec, d_gq, d_gs, d_out, d_full;
        struct Rel { std::vector<Buf*> v; ~Rel() { for (auto b : v) b->release(); } } rel{{&d_ids, &d_mask, &d_dec, &d_gq, &d_gs, &d_out, &d_full}};
        d_ids.ensure(Q * S * 8); d_mask.ensure(Q * S * 8);
        CUDA_CHECK(cudaMemcpyAsync(d_ids.p, ids, Q * S * 8, cudaMemcpyHostToDevice, s));
        CUDA_CHECK(cudaMemcpyAsync(d_mask.p, mask, Q * S * 8, cudaMemcpyHostToDevice, s));
        Ctx cx{m, s};
        m->launches = 0;
        encoder_forward(cx, D, d_ids.as<int64_t>(), d_mask.as<int64_t>());
        d_dec.ensure(D.R * T * 8); d_gq.ensure((D.R + 1) * 4); d_gs.ensure((D.R + 2) * 4);
        if (T > 1) d_out.ensure(D.R * (T - 1) * 4);
        if (out_full) d_full.ensure((size_t)D.R * D.V * 4);
        CUDA_CHECK(cudaMemsetAsync(m->err.as<int>() + 1, 0, 4, s));
        for (int64_t r0 = 0; r0 < N; r0 += kChunk) {
            const int64_t rows = std::min(kChunk, N - r0);
            std::vector<int32_t> gq, gs;
            for (int64_t r = 0; r < rows; ++r)
                if (r == 0 || row_query[r0 + r] != row_query[r0 + r - 1]) { gq.push_back(row_query[r0 + r]); gs.push_back((int32_t)r); }
            gs.push_back((int32_t)rows);
            CUDA_CHECK(cudaMemcpyAsync(d_dec.p, dec_ids + r0 * T, rows * T * 8, cudaMemcpyHostToDevice, s));
            CUDA_CHECK(cudaMemcpyAsync(d_gq.p, gq.data(), gq.size() * 4, cudaMemcpyHostToDevice, s));
            CUDA_CHECK(cudaMemcpyAsync(d_gs.p, gs.data(), gs.size() * 4, cudaMemcpyHostToDevice, s));
            Dims C = D;
            C.R = rows; C.G = (int64_t)gq.size(); C.grp_query = d_gq.as<int32_t>(); C.grp_start = d_gs.as<int32_t>();
            int32_t* tk = m->st_tokens.as<int32_t>(); int32_t* an = m->st_anc.as<int32_t>();
            ids_to_tokens_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, s>>>(rows, (int)T, (int)T, d_dec.as<int64_t>(), tk, an);
            CUDA_CHECK(cudaGetLastError());
            for (int p = 0; p < T; ++p) {
                const bool need = (p + 1 < T) || (out_full && p == out_full_pos);
                if (!need) continue;                           // the last position only feeds the full-vector output
                decoder_step(cx, C, tk, p + 1, an, true, nullptr);
                target_logprob_kernel<<<(unsigned)rows, 256, 0, s>>>(
                    rows, C.V, C.ld, m->logits.as<float>(), d_dec.as<int64_t>() + (p + 1 < T ? p + 1 : 0), T, temperature,
                    (p + 1 < T) ? d_out.as<float>() + p : nullptr, T - 1,
                    (out_full && p == out_full_pos) ? d_full.as<float>() : nullptr, C.V);
                CUDA_CHECK(cudaGetLastError()); m->launches++;
            }
            if (T > 1 && out_logprob)
                CUDA_CHECK(cudaMemcpyAsync(out_logprob + r0 * (T - 1), d_out.p, rows * (T - 1) * 4, cudaMemcpyDeviceToHost, s));
            if (out_full)
                CUDA_CHECK(cudaMemcpyAsync(out_full + (size_t)r0 * D.V, d_full.p, (size_t)rows * D.V * 4, cudaMemcpyDeviceToHost, s));
            CUDA_CHECK(cudaStreamSynchronize(s));              // gq/gs are stack temporaries; outputs consumed per chunk
        }
        int32_t ovf = 0;
        CUDA_CHECK(cudaMemcpy(&ovf, m->err.as<int>() + 1, 4, cudaMemcpyDeviceToHost));
        if (ovf) throw ApiError(SEALFM_EINVAL, "fp16 range exceeded in the 3xFP16 GEMM path (|x| > 65504); use gemm_mode 2 (3xTF32)");
    });
}

}  // extern "C"

namespace {
// sealdec_debug_gemm / sealdec_debug_gemm_split: C is written as fp32 (C != nullptr) or as the fp16 halves the next GEMM
// consumes, returned as their sum h1 + h2 in `halves_sum` with the producer's overflow flag in `overflow`
int debug_gemm(int mode, int64_t M, int32_t N, int32_t K, const float* A, const float* W, const float* bias, float* C,
               int32_t gelu, int32_t iters, double* avg_us, float* halves_sum, int32_t* overflow) {
    return guarded([&] {
        if (!A || !W || (!C && !halves_sum) || M <= 0 || N <= 0 || K <= 0) throw ApiError(SEALFM_EINVAL, "bad argument");
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { cudaGetLastError(); throw ApiError(SEALFM_ENODEVICE, "no CUDA device available"); }
        if (mode != 2 && mode != 3 && mode != 5) throw ApiError(SEALFM_EINVAL, "gemm_mode must be 2, 3 or 5");
        if (halves_sum && mode == 2) throw ApiError(SEALFM_EINVAL, "the fp16 split output exists in gemm_mode 3 and 5 only");
        sealbart fake; fake.cfg.gemm_mode = mode;
        CUDA_CHECK(cudaGetDevice(&fake.device));
        Buf dA, dW, dB, dC, whi, wlo;
        struct Rel { std::vector<Buf*> v; sealbart* f; ~Rel() { for (auto b : v) b->release(); f->a_hi.release(); f->a_lo.release(); f->err.release(); f->splitk.release(); } } rel{{&dA, &dW, &dB, &dC, &whi, &wlo}, &fake};
        const int ldc = halves_sum ? (N + 7) / 8 * 8 : (N + 3) / 4 * 4;        // 16-byte rows
        dA.ensure((size_t)M * K * 4); dW.ensure((size_t)N * K * 4); dB.ensure((size_t)N * 4); dC.ensure((size_t)M * ldc * 4);
        CUDA_CHECK(cudaMemcpy(dA.p, A, (size_t)M * K * 4, cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaMemcpy(dW.p, W, (size_t)N * K * 4, cudaMemcpyHostToDevice));
        if (bias) CUDA_CHECK(cudaMemcpy(dB.p, bias, (size_t)N * 4, cudaMemcpyHostToDevice));
        Lin l; l.w = dW.as<float>(); l.b = bias ? dB.as<float>() : nullptr; l.out = N; l.in = K;
        fake.err.ensure(16); CUDA_CHECK(cudaMemset(fake.err.p, 0, 16)); fake.ovf = fake.err.as<int>() + 1;
        if (mode == 2) {
            whi.ensure((size_t)N * K * 4); wlo.ensure((size_t)N * K * 4);
            l.w_hi = whi.as<float>(); l.w_lo = wlo.as<float>();
            split_into(nullptr, l.w, l.w_hi, l.w_lo, (uint64_t)N * K);
        } else if (mode >= 3) {
            whi.ensure((size_t)N * K * 2); wlo.ensure((size_t)N * K * 2);
            l.w_h1 = whi.as<__half>(); l.w_h2 = wlo.as<__half>();
            float mx = 0.f;
            for (int64_t i = 0; i < (int64_t)N * K; ++i) mx = std::max(mx, std::fabs(W[i]));
            int sexp = 0;
            if (mx > 0.f) { int e; std::frexp(mx, &e); sexp = 14 - e; }
            l.w_unscale = std::ldexp(1.0f, -sexp);
            split_half_kernel<<<sm_count() * 8, 256>>>((int64_t)N * K, l.w, std::ldexp(1.0f, sexp), l.w_h1, l.w_h2, fake.err.as<int>() + 1);
            CUDA_CHECK(cudaGetLastError());
        }
        Ctx cx{&fake, nullptr};
        Act out;
        if (halves_sum) { out.h1 = dC.as<__half>(); out.h2 = dC.as<__half>() + (size_t)M * ldc; }
        else out.x = dC.as<float>();
        gemm(cx, M, N, K, Act{dA.as<float>()}, K, l, out, ldc, gelu != 0);
        CUDA_CHECK(cudaDeviceSynchronize());
        if (iters > 0 && avg_us) {
            cudaEvent_t e0, e1; CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventCreate(&e1));
            CUDA_CHECK(cudaEventRecord(e0, nullptr));
            for (int i = 0; i < iters; ++i) gemm(cx, M, N, K, Act{dA.as<float>()}, K, l, out, ldc, gelu != 0);
            CUDA_CHECK(cudaEventRecord(e1, nullptr));
            CUDA_CHECK(cudaEventSynchronize(e1));
            float ms = 0; CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
            *avg_us = (double)ms * 1e3 / iters;
            cudaEventDestroy(e0); cudaEventDestroy(e1);
        }
        if (halves_sum) {
            std::vector<__half> h((size_t)2 * M * ldc);
            CUDA_CHECK(cudaMemcpy(h.data(), dC.p, h.size() * 2, cudaMemcpyDeviceToHost));
            for (int64_t r = 0; r < M; ++r)
                for (int n = 0; n < N; ++n)
                    halves_sum[r * N + n] = __half2float(h[r * ldc + n]) + __half2float(h[(size_t)M * ldc + r * ldc + n]);
            if (overflow) CUDA_CHECK(cudaMemcpy(overflow, fake.ovf, 4, cudaMemcpyDeviceToHost));
        } else {
            CUDA_CHECK(cudaMemcpy2D(C, (size_t)N * 4, dC.p, (size_t)ldc * 4, (size_t)N * 4, M, cudaMemcpyDeviceToHost));
        }
    });
}
}  // namespace

extern "C" {

int sealdec_debug_gemm(int mode, int64_t M, int32_t N, int32_t K, const float* A, const float* W, const float* bias, float* C,
                       int32_t gelu, int32_t iters, double* avg_us) {
    return debug_gemm(mode, M, N, K, A, W, bias, C, gelu, iters, avg_us, nullptr, nullptr);
}

int sealdec_debug_gemm_split(int mode, int64_t M, int32_t N, int32_t K, const float* A, const float* W, const float* bias,
                             int32_t gelu, float* halves_sum, int32_t* overflow) {
    return debug_gemm(mode, M, N, K, A, W, bias, nullptr, gelu, 0, nullptr, halves_sum, overflow);
}

int sealdec_apply_index_mask_d(const sealfm_t* fm, sealfm_stream_t stream, const sealdec_processor_cfg_t* cfg,
                               const int64_t* input_ids_d, int64_t R, int64_t t, const uint32_t* occ_d,
                               const float* in_d, float* out_d, int64_t V, int64_t ld) {
    return guarded([&] {
        if (!fm || !cfg || !input_ids_d || !in_d || !out_d) throw ApiError(SEALFM_EINVAL, "null argument");
        const int dev = sealfm_device(fm);
        if (dev < 0) throw ApiError(SEALFM_ENODEVICE, "index not bound to a CUDA device (call sealfm_to_device)");
        CUDA_CHECK(cudaSetDevice(dev));
        if (R <= 0 || t < 1) throw ApiError(SEALFM_EINVAL, "empty input");
        cudaStream_t s = (cudaStream_t)stream;
        const FmView view = sealfm_view(fm);
        const int W = (int)((V + 31) / 32);
        dim3 grid((unsigned)R, (unsigned)std::min<int64_t>((V + 255) / 256, 64));
        const bool fb = cfg->forced_bos_token_id >= 0;
        if (fb && t == 1) {                                                     // :66-69
            apply_mask_kernel<<<grid, 256, 0, s>>>(R, (int)V, ld, in_d, out_d, nullptr, W, 1, nullptr, cfg->eos_token_id,
                                                   cfg->pad_token_id, 0, cfg->forced_bos_token_id);
            CUDA_CHECK(cudaGetLastError());
            return;
        }
        const int skip = fb ? 1 : 0;                                            // :71
        if (t - skip == 1) {                                                    // :73-77
            if (!occ_d) throw ApiError(SEALFM_EINVAL, "occurring mask missing");
            apply_mask_kernel<<<grid, 256, 0, s>>>(R, (int)V, ld, in_d, out_d, occ_d, W, 1, nullptr, cfg->eos_token_id,
                                                   cfg->pad_token_id, cfg->always_allow_eos, -1);
            CUDA_CHECK(cudaGetLastError());
            return;
        }
        // scratch: lo, hi (u64), rule (u8), masks — stream-ordered allocation, no host sync
        uint64_t* lo = nullptr; uint64_t* hi = nullptr; uint8_t* rule = nullptr; uint32_t* masks = nullptr; uint64_t* fsyms = nullptr;
        // stream-ordered frees on EVERY exit path (an ApiError / CUDA_CHECK below must not leak the scratch)
        struct Scratch { void** p[5]; cudaStream_t s; ~Scratch() { for (void** q : p) if (*q) cudaFreeAsync(*q, s); } }
            guard{{(void**)&lo, (void**)&hi, (void**)&rule, (void**)&masks, (void**)&fsyms}, s};
        CUDA_CHECK(cudaMallocAsync(&lo, R * 8, s)); CUDA_CHECK(cudaMallocAsync(&hi, R * 8, s));
        CUDA_CHECK(cudaMallocAsync(&rule, R, s)); CUDA_CHECK(cudaMallocAsync(&masks, (size_t)R * W * 4, s));
        const int nf = cfg->n_force_decoding_from;
        if (nf > 0) {
            std::vector<uint64_t> f(nf);
            for (int i = 0; i < nf; ++i) f[i] = (uint64_t)cfg->force_decoding_from[i] + cfg->shift;
            CUDA_CHECK(cudaMallocAsync(&fsyms, nf * 8, s));
            CUDA_CHECK(cudaMemcpyAsync(fsyms, f.data(), nf * 8, cudaMemcpyHostToDevice, s));
            CUDA_CHECK(cudaStreamSynchronize(s));   // f is a stack temporary
        }
        rows_fold_kernel<<<(unsigned)((R + 127) / 128), 128, 0, s>>>(view, R, (int)t, input_ids_d, skip, cfg->eos_token_id,
                                                                    cfg->pad_token_id, cfg->stop_at_count, fsyms, nf, cfg->shift,
                                                                    lo, hi, rule);
        CUDA_CHECK(cudaGetLastError());
        int rc = sealfm_expand_mask_d(fm, s, R, lo, hi, masks, W, (uint32_t)V, (uint32_t)cfg->shift);
        if (rc) throw ApiError(rc, sealfm_last_error());
        apply_mask_kernel<<<grid, 256, 0, s>>>(R, (int)V, ld, in_d, out_d, masks, W, 0, rule, cfg->eos_token_id,
                                               cfg->pad_token_id, cfg->always_allow_eos, -1);
        CUDA_CHECK(cudaGetLastError());
    });
}

}  // extern "C"
