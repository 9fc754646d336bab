// text_model.cuh -- the Qwen3 decoder stack shared by Qwen3, Qwen3-VL (text) and Qwen3-ASR (thinker):
// weights in HBM, paged KV cache, prefill orchestration and the per-token decode step (CUDA graph).
// Reference: Qwen3Model / Qwen3DecoderLayer (/root/reference/src/models/qwen3/model.rs:19-214),
// Qwen3VLTextModel (qwen3vl/model.rs:743-835), Qwen3ASRThinkerTextModel (qwen3_asr/model.rs:229-306).
#pragma once
#include <cmath>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/aha_b200.h"
#include "attention.cuh"
#include "attention_mma.cuh"
#include "attention_tc.cuh"
#include "decode_fused.cuh"
#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "gemv.cuh"
#include "json.hpp"
#include "kernels_common.cuh"
#include "nccl_shim.h"
#include "sampling.cuh"

namespace aha {

// ---------------------------------------------------------------------------------------------------
struct Counters {
    uint64_t kernels = 0, graphs = 0;
};

struct Ctx {  // per-handle launch context
    cudaStream_t stream = nullptr;
    int device = 0;
    int num_sms = 148;
    Counters cnt;
    bool capturing = false;
    std::vector<void*> allocs;
    size_t alloc_bytes = 0;
    int attn_impl = 0;            // 0 = auto (tcgen05 flash attention for head_dim 64, mma.sync for 128), 1 = fp32 SIMT flash attention, 2 = mma.sync everywhere
    int gemm_impl = 0;            // 0 = auto (tcgen05 where the shape tiles), 1 = SIMT fp32, 2 / 3 / 4 = tcgen05 required: 128 x 128 tiles / persistent 128 x 256 / CTA-pair 256 x 256
    bool gemm_wide = true;        // auto: the persistent 128 x 256 kernel where N >= 256 (15-26 % faster than 128 x 128 on every prefill shape, profiles/r02_gemm_sweep.txt; AHA_GEMM_WIDE=0 turns it off)
    bool gemm_pair = true;        // auto: the CTA-pair kernel (cta_group::2, 256 x 256 tile per cluster) for prefill-sized M (>= 1024) and N >= 256: 1-3 % over the
                                  // single-CTA persistent kernel, bit-identical results (profiles/r02_gemm_sweep_pair.txt; AHA_GEMM_PAIR=0 turns it off)
    int gemm_group_m = 8;         // row blocks per band of the persistent kernel's tile walk (AHA_GEMM_GROUP)
    __half* split_ws = nullptr;   // [2][rows*K] hi | lo halves of the activation operand
    size_t split_cap = 0;         // halfs per half-buffer
    __half* split_buf(size_t halfs) {
        if (halfs > split_cap) {
            if (split_ws) { AHA_CUDA_CHECK(cudaStreamSynchronize(stream)); cudaFree(split_ws); }
            AHA_CUDA_CHECK(cudaMalloc(&split_ws, 2 * halfs * sizeof(__half)));
            split_cap = halfs;
        }
        return split_ws;
    }

    // Pre-split activations (two ping-pong buffers): a producer -- norm kernel, attention, GEMM epilogue -- writes the fp16 hi + lo
    // halves the next tensor-core GEMM reads, instead of an fp32 tensor that linear_gemm would have to read back and split.
    bool presplit = true;         // AHA_PRESPLIT=0: every GEMM splits its own fp32 input (the round-1 data flow; results are bit-identical)
    __half* act_ws[2] = {nullptr, nullptr};
    size_t act_cap[2] = {0, 0};
    __half* act_split(int which, size_t halfs) {   // hi at the returned pointer, lo at + act_cap[which]
        if (halfs > act_cap[which]) {
            if (act_ws[which]) { AHA_CUDA_CHECK(cudaStreamSynchronize(stream)); cudaFree(act_ws[which]); }
            AHA_CUDA_CHECK(cudaMalloc(&act_ws[which], 2 * halfs * sizeof(__half)));
            act_cap[which] = halfs;
        }
        return act_ws[which];
    }

    template <typename T>
    T* alloc(size_t n) {
        void* p = nullptr;
        AHA_CUDA_CHECK(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
        allocs.push_back(p);
        alloc_bytes += n * sizeof(T);
        return reinterpret_cast<T*>(p);
    }
    void free_all() {
        for (void* p : allocs) cudaFree(p);
        allocs.clear();
        if (split_ws) { cudaFree(split_ws); split_ws = nullptr; split_cap = 0; }
        for (int i = 0; i < 2; ++i)
            if (act_ws[i]) { cudaFree(act_ws[i]); act_ws[i] = nullptr; act_cap[i] = 0; }
    }
};

// ---------------------------------------------------------------------------------------------------
// Host-side weight table (descs by name) + dtype conversion.
inline float half_bits_to_float(uint16_t h) {
    const uint32_t sign = (h >> 15) & 1, exp = (h >> 10) & 0x1f, man = h & 0x3ff;
    uint32_t f;
    if (exp == 0) {
        if (man == 0) f = sign << 31;
        else {
            int e = -1; uint32_t m = man;
            do { ++e; m <<= 1; } while (!(m & 0x400));
            f = (sign << 31) | ((uint32_t)(127 - 15 - e) << 23) | ((m & 0x3ff) << 13);
        }
    } else if (exp == 31) f = (sign << 31) | 0x7f800000u | (man << 13);
    else f = (sign << 31) | ((exp + 112) << 23) | (man << 13);
    float r; std::memcpy(&r, &f, 4); return r;
}
inline float bf16_bits_to_float(uint16_t b) { uint32_t f = (uint32_t)b << 16; float r; std::memcpy(&r, &f, 4); return r; }

struct WeightTable {
    std::map<std::string, const aha_tensor_desc*> by_name;
    explicit WeightTable(const aha_tensor_desc* w, size_t n) {
        for (size_t i = 0; i < n; ++i)
            if (w[i].name) by_name[w[i].name] = &w[i];
    }
    bool has(const std::string& n) const { return by_name.count(n) != 0; }
    const aha_tensor_desc& get(const std::string& n) const {
        auto it = by_name.find(n);
        if (it == by_name.end()) throw std::runtime_error("missing weight tensor '" + n + "'");
        return *it->second;
    }
    static size_t numel(const aha_tensor_desc& d) { size_t n = 1; for (int i = 0; i < d.rank; ++i) n *= (size_t)d.shape[i]; return n; }
    // element i as float
    static float at(const aha_tensor_desc& d, size_t i) {
        switch (d.dtype) {
            case AHA_F32: return reinterpret_cast<const float*>(d.data)[i];
            case AHA_F16: return half_bits_to_float(reinterpret_cast<const uint16_t*>(d.data)[i]);
            case AHA_BF16: return bf16_bits_to_float(reinterpret_cast<const uint16_t*>(d.data)[i]);
            default: throw std::runtime_error(std::string("weight '") + (d.name ? d.name : "?") + "': unsupported dtype");
        }
    }
    void expect(const std::string& n, std::initializer_list<int64_t> shape) const {
        const aha_tensor_desc& d = get(n);
        size_t want = 1; for (auto s : shape) want *= (size_t)s;
        if (numel(d) != want) throw std::runtime_error("weight '" + n + "' has " + std::to_string(numel(d)) + " elements, expected " + std::to_string(want));
    }
    // rows [r0, r0+nr) of a [R, C] matrix -> fp16 staging (cols [c0, c0+nc))
    void rows_to_half(const std::string& n, int64_t R, int64_t C, int64_t r0, int64_t nr, int64_t c0, int64_t nc, __half* dst, int64_t dst_ld) const {
        const aha_tensor_desc& d = get(n);
        if ((int64_t)numel(d) != R * C) throw std::runtime_error("weight '" + n + "': unexpected size");
        if (d.dtype == AHA_F16) {
            const uint16_t* s = reinterpret_cast<const uint16_t*>(d.data);
            for (int64_t r = 0; r < nr; ++r) std::memcpy(reinterpret_cast<uint16_t*>(dst) + r * dst_ld, s + (r0 + r) * C + c0, (size_t)nc * 2);
        } else {
            // bf16 / f32 checkpoints are narrowed to fp16 (8 -> 10 mantissa bits for bf16: exact inside fp16's normal range).  A value
            // outside that range would silently become inf (|w| > 65504) or lose bits (|w| < 2^-14): refuse the checkpoint loudly.
            for (int64_t r = 0; r < nr; ++r)
                for (int64_t c = 0; c < nc; ++c) {
                    const float v = at(d, (size_t)((r0 + r) * C + c0 + c));
                    const float av = std::fabs(v);
                    if (!(av <= 65504.0f)) throw std::runtime_error("weight '" + n + "' holds a value outside the fp16 range (|w| > 65504 or not finite): this build stores linear weights as fp16");
                    if (d.dtype == AHA_BF16 && av != 0.0f && av < 6.103515625e-05f) throw std::runtime_error("weight '" + n + "' holds a bf16 value below fp16's normal range (|w| < 2^-14): it would lose bits as fp16");
                    dst[r * dst_ld + c] = __float2half_rn(v);
                }
        }
    }
    std::vector<float> vec_f32(const std::string& n, size_t expect_n) const {
        const aha_tensor_desc& d = get(n);
        if (numel(d) != expect_n) throw std::runtime_error("weight '" + n + "': unexpected size");
        std::vector<float> v(expect_n);
        for (size_t i = 0; i < expect_n; ++i) v[i] = at(d, i);
        return v;
    }
};

template <typename T>
inline T* upload(Ctx& c, const std::vector<T>& h) {
    T* d = c.alloc<T>(h.size());
    AHA_CUDA_CHECK(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return d;
}
inline float* upload_vec(Ctx& c, const WeightTable& wt, const std::string& name, size_t n) { return upload(c, wt.vec_f32(name, n)); }

struct LinearW {
    __half* w = nullptr;  // [N, K]
    float* b = nullptr;   // [N] or nullptr
    int N = 0, K = 0;
    CUtensorMap tmap;     // TMA descriptor of w (128 x 64 boxes, SWIZZLE_128B) when has_tmap
    bool has_tmap = false;
    CUtensorMap tmap256;  // the same with 256-row boxes (persistent 128 x 256 GEMM)
    bool has_tmap256 = false;
};

// Prefill attention dispatch: tensor-core kernel (attention_mma.cuh) unless the exact SIMT twin is requested.
template <int HD>
inline void flash_dispatch(Ctx& c, const FlashArgs& a, int nheads, bool causal) {
    if (c.attn_impl == 1) flash_attn<HD>(c.stream, a, nheads, causal);
    else if (c.attn_impl == 0) { flash_attn_tc<HD>(c.stream, a, nheads, causal, c.split_buf((flash_tc_ws_halfs<HD>(a, nheads) + 1) / 2)); c.cnt.kernels++; }
    else { flash_attn_mma<HD>(c.stream, a, nheads, causal, c.split_buf((flash_mma_ws_halfs<HD>(a, nheads) + 1) / 2)); c.cnt.kernels++; }
    c.cnt.kernels++;
}

// y = x W^T with the fused epilogues of gemm_simt.cuh.  Dispatch: tcgen05 split-fp16 kernel (gemm_tc.cuh) when the
// shape tiles (K % 64 == 0, N % 32 == 0) and there are enough rows to fill a tile, else the exact SIMT kernel.
struct ActSplit {   // fp16 hi + lo halves of an activation tensor [rows, ld]
    __half* hi = nullptr;
    __half* lo = nullptr;
    explicit operator bool() const { return hi != nullptr; }
};
inline ActSplit act_split(Ctx& c, int which, size_t halfs) {
    ActSplit a;
    a.hi = c.act_split(which, halfs);
    a.lo = a.hi + c.act_cap[which];
    return a;
}
// true when linear_gemm runs (M, W) on a tensor-core kernel: only then may a producer hand over pre-split activations
inline bool gemm_on_tc(const Ctx& c, int M, const LinearW& W) {
    return c.gemm_impl != 1 && gemm_tc_supported(M, W.N, W.K) && !(c.gemm_impl == 0 && M < 32);
}
// the tensor-core GEMM on activations that are already split ([M, K] contiguous halves); `out`: write the result split as well
inline void linear_gemm_split(Ctx& c, int epi, const __half* hi, const __half* lo, LinearW& W, const float* resid, int ldr, float* C, int ldc, int M,
                              int act = ACT_NONE, ActSplit out = ActSplit(), int ldo = 0) {
    if (M == 0) return;
    AHA_REQUIRE(gemm_on_tc(c, M, W), "linear_gemm_split: shape does not run on the tensor-core kernels");
    AHA_REQUIRE(!out || epi != EPI_RESID, "linear_gemm_split: the residual epilogue writes fp32");
    if (!W.has_tmap) { W.tmap = make_tmap_f16(W.w, (uint64_t)W.N, (uint64_t)W.K); W.has_tmap = true; }
    GemmTcArgs g;
    g.bias = W.b; g.resid = resid; g.ldr = ldr; g.C = C; g.ldc = ldc; g.M = M; g.N = W.N; g.K = W.K; g.act = act;
    g.out_hi = out.hi; g.out_lo = out.lo; g.ldo = ldo;
    g.group_m = std::max(1, c.gemm_group_m);
    if (c.gemm_impl == 4 || (c.gemm_impl == 0 && c.gemm_pair && W.N >= 256 && M >= 1024)) {
        gemm_tc3_launch(c.stream, epi, hi, lo, W.tmap, g, c.num_sms);
    } else if (c.gemm_impl == 3 || (c.gemm_impl == 0 && c.gemm_wide && W.N >= 256)) {
        if (!W.has_tmap256) { W.tmap256 = make_tmap_f16_rows(W.w, (uint64_t)W.N, (uint64_t)W.K, 256); W.has_tmap256 = true; }
        gemm_tc2_launch(c.stream, epi, hi, lo, W.tmap256, g, c.num_sms);
    } else {
        gemm_tc_launch(c.stream, epi, hi, lo, W.tmap, g);
    }
    c.cnt.kernels++;
}
inline void linear_gemm(Ctx& c, int epi, const float* A, int lda, LinearW& W, const float* resid, int ldr, float* C, int ldc, int M, int act = ACT_NONE) {
    if (M == 0) return;
    const bool tc_ok = gemm_tc_supported(M, W.N, W.K) && lda % 4 == 0;
    AHA_REQUIRE(c.gemm_impl < 2 || tc_ok, "gemm_impl=2/3/4 (tcgen05) requested but the shape does not tile (K % 64, N % 32)");
    if (c.gemm_impl == 1 || !tc_ok || (c.gemm_impl == 0 && M < 32)) {
        GemmArgs g;
        g.A = A; g.lda = lda; g.W = W.w; g.bias = W.b; g.resid = resid; g.ldr = ldr; g.C = C; g.ldc = ldc; g.M = M; g.N = W.N; g.K = W.K; g.act = act;
        gemm_simt(c.stream, epi, g);
        c.cnt.kernels++;
        return;
    }
    const size_t halfs = (size_t)M * W.K;
    __half* hi = c.split_buf(halfs);
    __half* lo = hi + c.split_cap;
    const size_t n4 = halfs / 4;
    split_f32_to_f16x2_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, c.stream>>>(A, lda, hi, lo, M, W.K);
    c.cnt.kernels++;
    linear_gemm_split(c, epi, hi, lo, W, resid, ldr, C, ldc, M, act);
}

// Upload `names` stacked along the output dimension ([sum N_i, K]); optional row interleave of two
// equally-sized matrices (gate/up -> rows g0,u0,g1,u1,...).  Row/col slices implement tensor parallelism.
struct RowSrc { std::string name; int64_t rows_total; int64_t r0; int64_t nr; };
inline LinearW upload_linear(Ctx& c, const WeightTable& wt, const std::vector<RowSrc>& parts, int64_t K_total, int64_t c0, int64_t nc,
                             bool interleave2, const std::vector<std::string>& bias_names) {
    int64_t N = 0;
    for (auto& p : parts) N += p.nr;
    std::vector<__half> stage((size_t)N * nc);
    if (interleave2) {
        AHA_REQUIRE(parts.size() == 2 && parts[0].nr == parts[1].nr, "interleave needs two equal parts");
        for (int k = 0; k < 2; ++k)
            wt.rows_to_half(parts[k].name, parts[k].rows_total, K_total, parts[k].r0, parts[k].nr, c0, nc, stage.data() + (size_t)k * nc, 2 * nc);
    } else {
        int64_t r = 0;
        for (auto& p : parts) {
            wt.rows_to_half(p.name, p.rows_total, K_total, p.r0, p.nr, c0, nc, stage.data() + (size_t)r * nc, nc);
            r += p.nr;
        }
    }
    LinearW L;
    L.N = (int)N; L.K = (int)nc;
    L.w = upload(c, stage);
    if (!bias_names.empty()) {
        std::vector<float> b;
        for (size_t i = 0; i < bias_names.size(); ++i) {
            auto v = wt.vec_f32(bias_names[i], (size_t)parts[i].rows_total);
            b.insert(b.end(), v.begin() + parts[i].r0, v.begin() + parts[i].r0 + parts[i].nr);
        }
        if (interleave2) {
            std::vector<float> bi(b.size());
            const size_t h = b.size() / 2;
            for (size_t i = 0; i < h; ++i) { bi[2 * i] = b[i]; bi[2 * i + 1] = b[h + i]; }
            b.swap(bi);
        }
        L.b = upload(c, b);
    }
    return L;
}

// One matrix uploaded through row / column maps: destination row r is source row row_map[r] (or all zeros when -1), destination
// column k is source column col_map[k] (or zero).  Used to pad shapes the tensor-core kernels do not tile (vision head_dim 72 ->
// 128-wide head slots, intermediate 4304 -> 4352): zero rows / columns leave the product unchanged.
inline LinearW upload_linear_mapped(Ctx& c, const WeightTable& wt, const std::string& name, int64_t N_src, int64_t K_src, const std::vector<int>& row_map,
                                    const std::vector<int>& col_map, const std::string& bias_name) {
    std::vector<__half> src((size_t)N_src * K_src);
    wt.rows_to_half(name, N_src, K_src, 0, N_src, 0, K_src, src.data(), K_src);
    const size_t N = row_map.size(), K = col_map.size();
    std::vector<__half> stage(N * K, __float2half(0.f));
    for (size_t r = 0; r < N; ++r) {
        if (row_map[r] < 0) continue;
        AHA_REQUIRE(row_map[r] < N_src, "row map out of range for " + name);
        const __half* sr = src.data() + (size_t)row_map[r] * K_src;
        __half* dr = stage.data() + r * K;
        for (size_t k = 0; k < K; ++k)
            if (col_map[k] >= 0) dr[k] = sr[col_map[k]];
    }
    LinearW L;
    L.N = (int)N; L.K = (int)K;
    L.w = upload(c, stage);
    if (!bias_name.empty()) {
        auto v = wt.vec_f32(bias_name, (size_t)N_src);
        std::vector<float> b(N, 0.f);
        for (size_t r = 0; r < N; ++r)
            if (row_map[r] >= 0) b[r] = v[row_map[r]];
        L.b = upload(c, b);
    }
    return L;
}

// ---------------------------------------------------------------------------------------------------
struct TextCfg {
    int H = 0, I = 0, L = 0, nh = 0, nkv = 0, hd = 0, V = 0;
    float eps = 1e-6f, theta = 1e6f;
    bool tie = false, attn_bias = false;
    bool mrope = false, mrope_asr = false;
    int mrope_section[3] = {0, 0, 0};
    static TextCfg from_json(const Json& j) {
        TextCfg c;
        c.H = j.integer("hidden_size"); c.I = j.integer("intermediate_size"); c.L = j.integer("num_hidden_layers");
        c.nh = j.integer("num_attention_heads"); c.nkv = j.integer_or("num_key_value_heads", c.nh);
        c.hd = j.integer_or("head_dim", c.H / c.nh); c.V = j.integer("vocab_size");
        c.eps = (float)j.number_or("rms_norm_eps", 1e-6); c.theta = (float)j.number_or("rope_theta", 1e6);
        c.tie = j.boolean_or("tie_word_embeddings", false); c.attn_bias = j.boolean_or("attention_bias", false);
        const std::string act = j.string_or("hidden_act", "silu");
        AHA_REQUIRE(act == "silu", "hidden_act '" + act + "' is not supported (Qwen3 family uses silu)");
        if (j.has("rope_scaling") && j.at("rope_scaling").has("mrope_section")) {
            auto s = j.at("rope_scaling").int_array("mrope_section");
            AHA_REQUIRE(s.size() == 3, "mrope_section must have 3 entries");
            for (int i = 0; i < 3; ++i) c.mrope_section[i] = s[i];
            c.mrope = true;
        }
        return c;
    }
};

struct TextLayer {
    LinearW qkv, o, gu, down;
    float *ln1 = nullptr, *ln2 = nullptr, *qn = nullptr, *kn = nullptr;
};

constexpr int kDecodeSplits = 16;        // split-KV factor of the decode attention

struct TextModel {
    TextCfg cfg;
    Ctx* ctx = nullptr;
    int tp_rank = 0, tp_world = 1;
    NcclApi::comm_t comm = nullptr;   // tensor-parallel communicator (tp_world > 1)
    float *tp_tmp = nullptr, *tp_tmp1 = nullptr;  // partial o_proj / down_proj outputs awaiting the all-reduce
    int nh_l = 0, nkv_l = 0, I_l = 0, qkv_dim = 0;  // per-rank (tensor-parallel) sizes
    __half* embed = nullptr;
    __half* lm_head = nullptr;
    float* norm = nullptr;
    std::vector<TextLayer> layers;
    float* inv_freq = nullptr;
    uint8_t* mrope_sel = nullptr;
    uint64_t weight_bytes = 0, decode_weight_bytes = 0;

    // paged KV
    int max_ctx = 0, num_pages = 0;
    float* kv_pool = nullptr;
    size_t layer_stride = 0, page_stride = 0;
    int* d_page_table = nullptr;
    std::vector<int> h_page_table, free_pages;
    int pages_mapped = 0;

    // prefill workspaces
    int max_prefill = 0;
    float *x = nullptr, *xn = nullptr, *qkv = nullptr, *attn = nullptr, *hbuf = nullptr;
    uint32_t* d_ids = nullptr;
    int* d_pos3 = nullptr;
    // decode workspaces
    float *x1 = nullptr, *qkv1 = nullptr, *attn1 = nullptr, *h1 = nullptr, *logits = nullptr, *partial = nullptr;
    int* counters = nullptr;
    float* pmax = nullptr; int* pidx = nullptr; int n_pcand = 0;
    DecodeState* d_state = nullptr;
    uint32_t* d_history = nullptr; int hist_cap = 0;
    uint32_t* d_argmax = nullptr;
    cudaGraphExec_t step_graph = nullptr;
    uint64_t step_graph_kernels = 0;
    bool use_graph = true;
    // fused persistent decode kernel (decode_fused.cuh)
    bool fused = false;
    bool fused_ll = false;               // the fused kernel keeps the residual stream on chip and exchanges packets (modes 1 and 2)
    int fused_mode = 0;                  // decode_fused.cuh MODE: 0 grid barriers, 1 packets everywhere, 2 hybrid
    int decode_impl = 0;
    // LL packet buffers.  The blocks a tensor-parallel peer writes (partial sums, argmax candidates) live in ONE separate
    // allocation per rank so that a single CUDA IPC handle maps them into the peers.
    LLPk *ll_qkv = nullptr, *ll_pb = nullptr, *ll_att = nullptr, *ll_h = nullptr;
    LLPk* ll_sym = nullptr;                         // [2][W][H] partial sums | [W][2] candidates   (this rank's copy)
    LLPk* ll_peer_sym[kFusedMaxTp] = {};            // the same block of every rank (own entry = ll_sym)
    int* d_ll_abort = nullptr;
    uint32_t ll_launches = 0;
    uint32_t* ll_flag = nullptr;                    // [4][256] local "data is out" flags
    LLPeerTab* d_ll_peers = nullptr;                // device copy of the per-peer pointer table (built once the peers are attached)
    bool ll_peers_ready = false;
    size_t ll_sym_packets() const { return (size_t)2 * tp_world * cfg.H + (size_t)tp_world * 2 + (size_t)tp_world * 256; }   // + [2][W][256] u32 flags = W * 256 packets
    FusedLayer* d_fused_layers = nullptr;
    unsigned* d_sync = nullptr;   // [0] grid barrier, [1] final ticket, then kv tickets [nkv]
    unsigned long long* d_ftrace = nullptr;
    size_t sync_words = 0;
    int fused_stages = kFusedStages;   // ring depth: re-measured on the final kernel of round 1, 11 slots 773 tok/s vs 8 slots 762 (profiles/README.md)
    int fused_grid = 0, fused_nsplit = 0;
    size_t fused_smem = 0;

    // sampler of the device loop (sampling.cuh); inactive = plain ArgMax, which the step kernels compute themselves
    bool samp_active = false;
    SampleArgs samp{};
    float* sample_work = nullptr;
    int* d_sample_err = nullptr;

    // tracing (tests)
    bool trace = false;
    float* trace_buf = nullptr;  // [L][max_prefill][H]
    int trace_S = 0;

    // ---------------------------------------------------------------------------------------------
    void load(Ctx& c, const TextCfg& cf, const WeightTable& wt, const std::string& prefix, const std::string& lm_head_name,
              int rank, int world) {
        ctx = &c; cfg = cf; tp_rank = rank; tp_world = world;
        AHA_REQUIRE(cfg.hd == 128, "head_dim must be 128 (Qwen3 family)");
        AHA_REQUIRE(cfg.nh % cfg.nkv == 0, "num_attention_heads must be a multiple of num_key_value_heads");
        AHA_REQUIRE(cfg.nkv % world == 0 && cfg.I % world == 0, "tensor-parallel world must divide num_key_value_heads and intermediate_size");
        const int G = cfg.nh / cfg.nkv;
        AHA_REQUIRE(G == 1 || G == 2 || G == 4 || G == 6, "unsupported GQA group size");
        nkv_l = cfg.nkv / world; nh_l = nkv_l * G; I_l = cfg.I / world;
        qkv_dim = (nh_l + 2 * nkv_l) * cfg.hd;
        AHA_REQUIRE(cfg.H % 16 == 0 && I_l % 16 == 0, "hidden/intermediate sizes must be multiples of 16");
        const int H = cfg.H, hd = cfg.hd;
        const size_t before = c.alloc_bytes;
        {
            std::vector<__half> st((size_t)cfg.V * H);
            wt.rows_to_half(prefix + "embed_tokens.weight", cfg.V, H, 0, cfg.V, 0, H, st.data(), H);
            embed = upload(c, st);
            if (cfg.tie) lm_head = embed;
            else {
                wt.rows_to_half(lm_head_name, cfg.V, H, 0, cfg.V, 0, H, st.data(), H);
                lm_head = upload(c, st);
            }
        }
        norm = upload_vec(c, wt, prefix + "norm.weight", H);
        layers.resize(cfg.L);
        for (int l = 0; l < cfg.L; ++l) {
            const std::string p = prefix + "layers." + std::to_string(l) + ".";
            TextLayer& T = layers[l];
            std::vector<std::string> qb, ob;
            if (cfg.attn_bias) { qb = {p + "self_attn.q_proj.bias", p + "self_attn.k_proj.bias", p + "self_attn.v_proj.bias"}; ob = {p + "self_attn.o_proj.bias"}; }
            T.qkv = upload_linear(c, wt,
                                  {{p + "self_attn.q_proj.weight", (int64_t)cfg.nh * hd, (int64_t)rank * nh_l * hd, (int64_t)nh_l * hd},
                                   {p + "self_attn.k_proj.weight", (int64_t)cfg.nkv * hd, (int64_t)rank * nkv_l * hd, (int64_t)nkv_l * hd},
                                   {p + "self_attn.v_proj.weight", (int64_t)cfg.nkv * hd, (int64_t)rank * nkv_l * hd, (int64_t)nkv_l * hd}},
                                  H, 0, H, false, qb);
            T.o = upload_linear(c, wt, {{p + "self_attn.o_proj.weight", H, 0, H}}, (int64_t)cfg.nh * hd, (int64_t)rank * nh_l * hd, (int64_t)nh_l * hd, false,
                                (rank == 0 ? ob : std::vector<std::string>{}));
            T.gu = upload_linear(c, wt, {{p + "mlp.gate_proj.weight", cfg.I, (int64_t)rank * I_l, I_l}, {p + "mlp.up_proj.weight", cfg.I, (int64_t)rank * I_l, I_l}},
                                 H, 0, H, true, {});
            T.down = upload_linear(c, wt, {{p + "mlp.down_proj.weight", H, 0, H}}, cfg.I, (int64_t)rank * I_l, I_l, false, {});
            T.ln1 = upload_vec(c, wt, p + "input_layernorm.weight", H);
            T.ln2 = upload_vec(c, wt, p + "post_attention_layernorm.weight", H);
            T.qn = upload_vec(c, wt, p + "self_attn.q_norm.weight", hd);
            T.kn = upload_vec(c, wt, p + "self_attn.k_norm.weight", hd);
        }
        weight_bytes = c.alloc_bytes - before;
        decode_weight_bytes = 0;
        for (auto& T : layers)
            decode_weight_bytes += 2ull * ((size_t)T.qkv.N * T.qkv.K + (size_t)T.o.N * T.o.K + (size_t)T.gu.N * T.gu.K + (size_t)T.down.N * T.down.K) +
                                   4ull * (2 * H + 2 * hd);
        decode_weight_bytes += 4ull * H + 2ull * (size_t)cfg.V * H;
        // RoPE tables: inv_freq in f32 powf like rope.rs:7-13; M-RoPE row selector per frequency (rope.rs:454-476 / 478-500)
        std::vector<float> inv(hd / 2);
        for (int j = 0; j < hd / 2; ++j) inv[j] = 1.0f / powf(cfg.theta, (float)(2 * j) / (float)hd);
        inv_freq = upload(c, inv);
        std::vector<uint8_t> sel(hd / 2, 0);
        if (cfg.mrope) {
            for (int dim = 1; dim < 3; ++dim) {
                const int length = cfg.mrope_asr ? cfg.mrope_section[dim] : cfg.mrope_section[dim] * 3;
                for (int idx = dim; idx < length && idx < hd / 2; idx += 3) sel[idx] = (uint8_t)dim;
            }
        }
        mrope_sel = upload(c, sel);
    }

    int max_ctx_hint = 0;
    bool fused_supported(std::string* why) const {
        auto no = [&](const char* m) { if (why) *why = m; return false; };
        if (tp_world > kFusedMaxTp) return no("more than 8 tensor-parallel ranks");
        if (cfg.hd != 128) return no("head_dim != 128");
        if (cfg.H > kFusedMaxH) return no("hidden_size > 4096 (residual stream kept in shared memory)");
        if (cfg.H % 8 || I_l % 8) return no("K not a multiple of 8");
        if (cfg.H > kFusedMaxK || I_l > kFusedMaxK || nh_l * cfg.hd > kFusedMaxK) return no("K > 8192");
        if (rows_per_stage(cfg.H, 2 * I_l, ctx->num_sms) % 2) return no("a gate/up row pair does not fit one 16 KB stage");
        if ((cfg.H + ctx->num_sms - 1) / ctx->num_sms > kFusedMaxOwnRows) return no("more residual rows per SM than the fused kernel keeps on chip");
        if (ctx->num_sms < nkv_l) return no("fewer SMs than kv heads");
        if (cfg.attn_bias) return no("attention bias");
        if (nh_l / nkv_l > 4) return no("GQA group > 4");
        if (max_ctx_hint > kFusedMaxPages * kPage) return no("max_ctx beyond the page table staged in shared memory");
        if (ceil_div(max_ctx_hint, kPage) > 65535) return no("more than 65535 KV pages");
        return true;
    }
    template <int G>
    void (*fused_kernel() const)(FusedArgs) {
        return fused_mode == 1 ? decode_step_fused_kernel<G, 1> : (fused_mode == 2 ? decode_step_fused_kernel<G, 2> : decode_step_fused_kernel<G, 0>);
    }
    template <int G>
    void fused_prepare() {
        fused_smem = fused_smem_bytes<G>(fused_ll);
        auto prep = [&](auto kernel) {
            AHA_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fused_smem));
            int nb = 0;
            AHA_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, kFusedThreads, fused_smem));
            AHA_REQUIRE(nb >= 1, "fused decode kernel does not fit on an SM");
        };
        prep(fused_kernel<G>());
    }
    void alloc_runtime(int max_ctx_, int max_prefill_, bool graph, int decode_impl_ = 0) {
        Ctx& c = *ctx;
        max_ctx = max_ctx_; max_prefill = max_prefill_; use_graph = graph; decode_impl = decode_impl_; max_ctx_hint = max_ctx_;
        {
            std::string why;
            const bool ok = fused_supported(&why);
            AHA_REQUIRE(decode_impl >= 0 && decode_impl <= 4, "decode_impl must be 0 (auto), 1 (per-op kernels), 2 (fused, packets), 3 (fused, grid barriers) or 4 (fused, hybrid)");
            AHA_REQUIRE(decode_impl < 2 || ok, "fused decode kernel unsupported for this model: " + why);
            AHA_REQUIRE(decode_impl != 3 || tp_world == 1, "the grid-barrier twin of the fused kernel is single-GPU only");
            fused = ok && decode_impl != 1;
            // auto: one GPU -> the grid-barrier kernel (measured fastest there: 794 vs 690 (hybrid) / 637 (packets) tok/s on the Qwen3-VL-2B
            // stack, profiles/README.md); tensor parallel -> the hybrid kernel: local grid barriers inside the layer, NVLink packets for the
            // two residual-stream exchanges (no cross-GPU barrier anywhere)
            fused_mode = !fused ? 0 : (decode_impl == 2 ? 1 : (decode_impl == 4 ? 2 : (decode_impl == 3 ? 0 : (tp_world > 1 ? 2 : 0))));
            fused_ll = fused && fused_mode != 0;
        }
        num_pages = ceil_div(max_ctx, kPage);
        page_stride = (size_t)2 * nkv_l * kPage * cfg.hd;
        layer_stride = page_stride * num_pages;
        kv_pool = c.alloc<float>(layer_stride * cfg.L);
        AHA_CUDA_CHECK(cudaMemset(kv_pool, 0, layer_stride * cfg.L * sizeof(float)));   // never feed uninitialised bits to the FMA pipes
        d_page_table = c.alloc<int>(num_pages);
        h_page_table.assign(num_pages, 0);
        reset_pages();
        const size_t S = max_prefill;
        x = c.alloc<float>(S * cfg.H); xn = c.alloc<float>(S * cfg.H);
        qkv = c.alloc<float>(S * qkv_dim); attn = c.alloc<float>(S * nh_l * cfg.hd); hbuf = c.alloc<float>(S * I_l);
        d_ids = c.alloc<uint32_t>(S); d_pos3 = c.alloc<int>(3 * S);
        if (tp_world > 1) { tp_tmp = c.alloc<float>(S * cfg.H); tp_tmp1 = c.alloc<float>(cfg.H); }
        x1 = c.alloc<float>(cfg.H); qkv1 = c.alloc<float>(qkv_dim); attn1 = c.alloc<float>((size_t)nh_l * cfg.hd); h1 = c.alloc<float>(I_l);
        logits = c.alloc<float>(cfg.V);
        fused_grid = c.num_sms;
        fused_nsplit = std::max(1, std::min(32, fused_grid / std::max(1, nkv_l)));
        partial = c.alloc<float>((size_t)nh_l * std::max(kDecodeSplits, fused_nsplit) * (cfg.hd + 4));   // fused kernel: 16-byte aligned rows
        sync_words = 2 + nkv_l;
        d_sync = c.alloc<unsigned>(sync_words);
        AHA_CUDA_CHECK(cudaMemset(d_sync, 0, sync_words * sizeof(unsigned)));
        counters = reinterpret_cast<int*>(d_sync + 2);
        if (fused) {
            std::vector<FusedLayer> fl(cfg.L);
            for (int l = 0; l < cfg.L; ++l) {
                TextLayer& T = layers[l];
                fl[l] = FusedLayer{T.qkv.w, T.o.w, T.gu.w, T.down.w, T.qkv.b, T.o.b, T.ln1, T.ln2, T.qn, T.kn};
            }
            d_fused_layers = upload(c, fl);
            if (fused_ll) {
                auto zalloc = [&](size_t n) { LLPk* p = c.alloc<LLPk>(n); AHA_CUDA_CHECK(cudaMemset(p, 0, n * sizeof(LLPk))); return p; };
                ll_qkv = zalloc((size_t)qkv_dim);
                ll_pb = zalloc((size_t)nh_l * fused_nsplit * kFusedPartialStride);
                ll_att = zalloc((size_t)nh_l * cfg.hd);
                ll_h = zalloc((size_t)I_l);
                void* sym = nullptr;   // its own allocation: the IPC handle of a pointer covers the whole cudaMalloc block
                AHA_CUDA_CHECK(cudaMalloc(&sym, ll_sym_packets() * sizeof(LLPk)));
                c.allocs.push_back(sym);
                AHA_CUDA_CHECK(cudaMemset(sym, 0, ll_sym_packets() * sizeof(LLPk)));
                ll_sym = reinterpret_cast<LLPk*>(sym);
                ll_peer_sym[tp_rank] = ll_sym;
                ll_flag = c.alloc<uint32_t>(4 * 256);
                AHA_CUDA_CHECK(cudaMemset(ll_flag, 0, 4 * 256 * sizeof(uint32_t)));
                AHA_REQUIRE(c.num_sms <= 256, "more than 256 SMs");
                d_ll_peers = c.alloc<LLPeerTab>(1);
                d_ll_abort = c.alloc<int>(1);
                AHA_CUDA_CHECK(cudaMemset(d_ll_abort, 0, sizeof(int)));
            }
            d_ftrace = c.alloc<unsigned long long>(kFusedTraceWords);
            AHA_CUDA_CHECK(cudaMemset(d_ftrace, 0, kFusedTraceWords * sizeof(unsigned long long)));
            switch (nh_l / nkv_l) {
                case 1: fused_prepare<1>(); break;
                case 2: fused_prepare<2>(); break;
                default: fused_prepare<4>(); break;
            }
        }
        n_pcand = gemv_grid(cfg.V, GEPI_ARGMAX);
        pmax = c.alloc<float>(std::max(n_pcand, c.num_sms)); pidx = c.alloc<int>(std::max(n_pcand, c.num_sms));
        d_state = c.alloc<DecodeState>(1);
        AHA_CUDA_CHECK(cudaMemset(d_state, 0, sizeof(DecodeState)));
        hist_cap = max_ctx;
        d_history = c.alloc<uint32_t>(hist_cap);
        d_argmax = c.alloc<uint32_t>(1);
    }

    void set_trace(bool on) {
        if (on && !trace_buf) trace_buf = ctx->alloc<float>((size_t)cfg.L * max_prefill * cfg.H);
        trace = on;
    }

    // ---- paged KV management (host side).  Physical pages are handed out from the END of the pool so the
    // logical->physical mapping is never the identity (the indirection is always exercised).
    void reset_pages() {
        free_pages.clear();
        for (int p = 0; p < num_pages; ++p) free_pages.push_back(p);
        pages_mapped = 0;
    }
    void ensure_tokens(int n_tokens) {
        AHA_REQUIRE(n_tokens <= max_ctx, "context of " + std::to_string(n_tokens) + " tokens exceeds max_ctx " + std::to_string(max_ctx));
        const int need = ceil_div(n_tokens, kPage);
        if (need <= pages_mapped) return;
        const int first = pages_mapped;
        while (pages_mapped < need) {
            h_page_table[pages_mapped++] = free_pages.back();
            free_pages.pop_back();
        }
        AHA_CUDA_CHECK(cudaMemcpyAsync(d_page_table + first, h_page_table.data() + first, (size_t)(pages_mapped - first) * sizeof(int),
                                       cudaMemcpyHostToDevice, ctx->stream));
    }
    KVSrc kv_src(int layer) const {
        KVSrc s;
        s.k = kv_pool + (size_t)layer * layer_stride;
        s.v = s.k + (size_t)nkv_l * kPage * cfg.hd;
        s.page_table = d_page_table; s.page_shift = kPageShift; s.page_stride = page_stride;
        s.tok_stride = cfg.hd; s.head_stride = (size_t)kPage * cfg.hd;
        return s;
    }

    // ---- GEMM dispatch (SIMT exact path; the tcgen05 path plugs in here)
    void gemm(int epi, const float* A, int lda, LinearW& W, const float* resid, int ldr, float* C, int ldc, int M, int act = ACT_NONE) {
        linear_gemm(*ctx, epi, A, lda, W, resid, ldr, C, ldc, M, act);
    }

    void init_tp(const void* unique_id) {
        if (tp_world <= 1) return;
        AHA_REQUIRE(unique_id != nullptr, "tp_world > 1 needs aha_options.tp_comm (128-byte ncclUniqueId)");
        NcclApi& n = NcclApi::get();
        NcclApi::unique_id id;
        std::memcpy(&id, unique_id, sizeof(id));
        n.check(n.CommInitRank(&comm, tp_world, id, tp_rank), "ncclCommInitRank");
        if (!fused_ll) return;
        // Map every rank's packet block into this process (CUDA IPC; NVLink / NVSwitch peer access): the handles travel
        // through the communicator itself, so the C ABI needs nothing beyond the unique id it already takes.
        cudaIpcMemHandle_t mine;
        AHA_CUDA_CHECK(cudaIpcGetMemHandle(&mine, ll_sym));
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
        char* d_h = ctx->alloc<char>((size_t)64 * tp_world);
        AHA_CUDA_CHECK(cudaMemcpyAsync(d_h + (size_t)64 * tp_rank, &mine, 64, cudaMemcpyHostToDevice, ctx->stream));
        n.check(n.AllGather(d_h + (size_t)64 * tp_rank, d_h, 64, NcclApi::kInt8, comm, ctx->stream), "ncclAllGather(ipc handles)");
        std::vector<cudaIpcMemHandle_t> all(tp_world);
        AHA_CUDA_CHECK(cudaMemcpyAsync(all.data(), d_h, (size_t)64 * tp_world, cudaMemcpyDeviceToHost, ctx->stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));   // every rank zeroed its block before it entered the all-gather
        for (int w = 0; w < tp_world; ++w) {
            if (w == tp_rank) continue;
            void* p = nullptr;
            AHA_CUDA_CHECK(cudaIpcOpenMemHandle(&p, all[w], cudaIpcMemLazyEnablePeerAccess));
            ll_peer_sym[w] = reinterpret_cast<LLPk*>(p);
        }
    }
    // a wait inside the fused kernel timed out (a peer GPU / CTA died): surface it instead of returning garbage
    void check_ll_abort() {
        if (!d_ll_abort) return;
        int flag = 0;
        AHA_CUDA_CHECK(cudaMemcpy(&flag, d_ll_abort, sizeof(int), cudaMemcpyDeviceToHost));
        if (flag) {
            cudaMemset(d_ll_abort, 0, sizeof(int));
            throw std::runtime_error("fused decode step: a packet never arrived (tensor-parallel peer not running the same step?)");
        }
    }
    // all-reduce(sum) of a partial projection over the tensor-parallel ranks, then x += sum (the residual add)
    void tp_reduce_add(float* partial, float* xdst, size_t n) {
        NcclApi& api = NcclApi::get();
        api.check(api.AllReduce(partial, partial, n, NcclApi::kFloat32, NcclApi::kSum, comm, ctx->stream), "ncclAllReduce");
        add_inplace_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(xdst, partial, n);
        ctx->cnt.kernels++;
    }

    // ---- prefill: ids already on device in d_ids (or embeddings already in x when embeds_ready), pos3 in d_pos3.
    // visual_idx/deepstack: Qwen3-VL deepstack injection (qwen3vl/model.rs:815-824).
    void prefill(int S, int pos0, bool embeds_ready, const int* d_visual_idx, int n_visual, const std::vector<const float*>& deepstack) {
        Ctx& c = *ctx;
        cudaStream_t st = c.stream;
        const int H = cfg.H, hd = cfg.hd;
        AHA_REQUIRE(S <= max_prefill, "prompt of " + std::to_string(S) + " tokens exceeds max_prefill " + std::to_string(max_prefill));
        ensure_tokens(pos0 + S);
        if (!embeds_ready) { embed_gather_kernel<<<S, 256, 0, st>>>(d_ids, embed, x, S, H, cfg.V); c.cnt.kernels++; }
        RopeArgs rp{inv_freq, mrope_sel, d_pos3, S};
        const float scaling = (float)(1.0 / std::sqrt((double)hd));
        for (int l = 0; l < cfg.L; ++l) {
            TextLayer& T = layers[l];
            // pre-split data flow (Ctx::presplit): norm -> [hi|lo] -> qkv GEMM; attention -> [hi|lo] -> o_proj; norm -> [hi|lo] -> gate/up
            // GEMM, whose SwiGLU epilogue writes [hi|lo] -> down_proj.  No stand-alone split pass, no fp32 intermediates.
            const bool ps = c.presplit && gemm_on_tc(c, S, T.qkv) && gemm_on_tc(c, S, T.o) && gemm_on_tc(c, S, T.gu) && gemm_on_tc(c, S, T.down) && c.attn_impl == 0;
            if (ps) {
                ActSplit n1 = act_split(c, 0, (size_t)S * H);
                rmsnorm_split_kernel<<<S, 256, 0, st>>>(x, T.ln1, cfg.eps, n1.hi, n1.lo, H); c.cnt.kernels++;
                linear_gemm_split(c, EPI_STORE, n1.hi, n1.lo, T.qkv, nullptr, 0, qkv, qkv_dim, S);
            } else {
                rmsnorm_kernel<<<S, 256, 0, st>>>(x, T.ln1, cfg.eps, xn, H); c.cnt.kernels++;
                gemm(EPI_STORE, xn, H, T.qkv, nullptr, 0, qkv, qkv_dim, S);
            }
            KVSrc kv = kv_src(l);
            qk_norm_rope_kv_kernel<128><<<dim3(S, nh_l + 2 * nkv_l), 128, 0, st>>>(qkv, T.qn, T.kn, cfg.eps, rp, const_cast<float*>(kv.k), const_cast<float*>(kv.v), kv, nh_l, nkv_l, pos0);
            c.cnt.kernels++;
            FlashArgs fa;
            fa.q = qkv; fa.q_tok_stride = qkv_dim; fa.q_head_stride = hd; fa.kv = kv;
            fa.out = attn; fa.o_tok_stride = (size_t)nh_l * hd; fa.o_head_stride = hd;
            fa.Sq = S; fa.Skv = pos0 + S; fa.q0 = 0; fa.kv0 = 0; fa.groups = nh_l / nkv_l; fa.scaling = scaling;
            if (ps) {
                ActSplit ao = act_split(c, 1, (size_t)S * std::max(nh_l * hd, I_l));
                fa.out_hi = ao.hi; fa.out_lo = ao.lo;
                flash_dispatch<128>(c, fa, nh_l, true);
                if (tp_world > 1) { linear_gemm_split(c, EPI_STORE, ao.hi, ao.lo, T.o, nullptr, 0, tp_tmp, H, S); tp_reduce_add(tp_tmp, x, (size_t)S * H); }
                else linear_gemm_split(c, EPI_RESID, ao.hi, ao.lo, T.o, x, H, x, H, S);
                ActSplit n2 = act_split(c, 0, (size_t)S * H);
                rmsnorm_split_kernel<<<S, 256, 0, st>>>(x, T.ln2, cfg.eps, n2.hi, n2.lo, H); c.cnt.kernels++;
                linear_gemm_split(c, EPI_SWIGLU, n2.hi, n2.lo, T.gu, nullptr, 0, nullptr, 0, S, ACT_NONE, ao, I_l);
                if (tp_world > 1) { linear_gemm_split(c, EPI_STORE, ao.hi, ao.lo, T.down, nullptr, 0, tp_tmp, H, S); tp_reduce_add(tp_tmp, x, (size_t)S * H); }
                else linear_gemm_split(c, EPI_RESID, ao.hi, ao.lo, T.down, x, H, x, H, S);
            } else {
                flash_dispatch<128>(c, fa, nh_l, true);
                if (tp_world > 1) { gemm(EPI_STORE, attn, nh_l * hd, T.o, nullptr, 0, tp_tmp, H, S); tp_reduce_add(tp_tmp, x, (size_t)S * H); }
                else gemm(EPI_RESID, attn, nh_l * hd, T.o, x, H, x, H, S);
                rmsnorm_kernel<<<S, 256, 0, st>>>(x, T.ln2, cfg.eps, xn, H); c.cnt.kernels++;
                gemm(EPI_SWIGLU, xn, H, T.gu, nullptr, 0, hbuf, I_l, S);
                if (tp_world > 1) { gemm(EPI_STORE, hbuf, I_l, T.down, nullptr, 0, tp_tmp, H, S); tp_reduce_add(tp_tmp, x, (size_t)S * H); }
                else gemm(EPI_RESID, hbuf, I_l, T.down, x, H, x, H, S);
            }
            if (l < (int)deepstack.size() && n_visual > 0) {
                scatter_rows_kernel<<<n_visual, 256, 0, st>>>(d_visual_idx, deepstack[l], x, H, 1); c.cnt.kernels++;
            }
            if (trace) AHA_CUDA_CHECK(cudaMemcpyAsync(trace_buf + (size_t)l * max_prefill * H, x, (size_t)S * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
        trace_S = S;
        AHA_CUDA_CHECK(cudaGetLastError());
        // last-token logits: final RMSNorm fused into the lm_head GEMV (qwen3/model.rs:186-187,142)
        head(x + (size_t)(S - 1) * H);
    }

    void head(const float* xrow) {
        GemvArgs a{};
        a.W = lm_head; a.x = xrow; a.norm_w = norm; a.eps = cfg.eps; a.out = logits; a.pmax = pmax; a.pidx = pidx; a.N = cfg.V; a.K = cfg.H;
        gemv(ctx->stream, PRO_RMSNORM, GEPI_ARGMAX, a); ctx->cnt.kernels++;
    }
    // publish argmax; advance != 0 also feeds the token back into the decode state
    void finish_argmax(int advance) {
        argmax_final_kernel<<<1, 32, 0, ctx->stream>>>(pmax, pidx, n_pcand, d_argmax, d_state, d_history, hist_cap, advance);
        ctx->cnt.kernels++;
    }

    // ---- one decode step, all inputs taken from d_state (token, pos, rope_delta)
    template <int G>
    void launch_decode_attn(const DecodeAttnArgs& a) {
        decode_attn_kernel<128, G><<<dim3(kDecodeSplits, nkv_l), 256, 0, ctx->stream>>>(a);
    }
    void decode_step_launches() {
        Ctx& c = *ctx;
        cudaStream_t st = c.stream;
        const int H = cfg.H, hd = cfg.hd;
        embed_gather_kernel<<<1, 256, 0, st>>>(&d_state->token, embed, x1, 1, H, cfg.V); c.cnt.kernels++;
        const float scaling = (float)(1.0 / std::sqrt((double)hd));
        for (int l = 0; l < cfg.L; ++l) {
            TextLayer& T = layers[l];
            GemvArgs a{};
            a.W = T.qkv.w; a.bias = T.qkv.b; a.x = x1; a.norm_w = T.ln1; a.eps = cfg.eps; a.out = qkv1; a.N = T.qkv.N; a.K = T.qkv.K;
            gemv(st, PRO_RMSNORM, GEPI_STORE, a); c.cnt.kernels++;
            KVSrc kv = kv_src(l);
            DecodeAttnArgs d{};
            d.qkv = qkv1; d.qw = T.qn; d.kw = T.kn; d.eps = cfg.eps; d.inv_freq = inv_freq; d.st = d_state;
            d.kbase = const_cast<float*>(kv.k); d.vbase = const_cast<float*>(kv.v); d.kv = kv;
            d.partial = partial; d.counters = counters; d.out = attn1; d.nh = nh_l; d.nkv = nkv_l; d.nsplit = kDecodeSplits; d.scaling = scaling;
            switch (nh_l / nkv_l) {
                case 1: launch_decode_attn<1>(d); break;
                case 2: launch_decode_attn<2>(d); break;
                case 4: launch_decode_attn<4>(d); break;
                default: launch_decode_attn<6>(d); break;
            }
            c.cnt.kernels++;
            GemvArgs o{};
            o.W = T.o.w; o.bias = T.o.b; o.x = attn1; o.resid = x1; o.out = x1; o.N = T.o.N; o.K = T.o.K;
            if (tp_world > 1) { o.resid = nullptr; o.out = tp_tmp1; gemv(st, PRO_NONE, GEPI_STORE, o); c.cnt.kernels++; tp_reduce_add(tp_tmp1, x1, H); }
            else { gemv(st, PRO_NONE, GEPI_RESID, o); c.cnt.kernels++; }
            GemvArgs g{};
            g.W = T.gu.w; g.x = x1; g.norm_w = T.ln2; g.eps = cfg.eps; g.out = h1; g.N = T.gu.N; g.K = T.gu.K;
            gemv(st, PRO_RMSNORM, GEPI_SWIGLU, g); c.cnt.kernels++;
            GemvArgs dn{};
            dn.W = T.down.w; dn.x = h1; dn.resid = x1; dn.out = x1; dn.N = T.down.N; dn.K = T.down.K;
            if (tp_world > 1) { dn.resid = nullptr; dn.out = tp_tmp1; gemv(st, PRO_NONE, GEPI_STORE, dn); c.cnt.kernels++; tp_reduce_add(tp_tmp1, x1, H); }
            else { gemv(st, PRO_NONE, GEPI_RESID, dn); c.cnt.kernels++; }
        }
        head(x1);
        finish_argmax(1);
        AHA_CUDA_CHECK(cudaGetLastError());
    }
    template <int G>
    void launch_fused(FusedArgs& fa) {
        void* args[] = {&fa};
        AHA_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)fused_kernel<G>(), dim3(fused_grid), dim3(kFusedThreads), args, fused_smem, ctx->stream));
    }
    void decode_step_fused() {
        Ctx& c = *ctx;
        FusedArgs fa{};
        fa.layers = d_fused_layers; fa.L = cfg.L; fa.H = cfg.H; fa.I = I_l; fa.nh = nh_l; fa.nkv = nkv_l; fa.hd = cfg.hd; fa.V = cfg.V; fa.qkv_dim = qkv_dim;
        fa.eps = cfg.eps; fa.scaling = (float)(1.0 / std::sqrt((double)cfg.hd));
        fa.embed = embed; fa.lm_head = lm_head; fa.final_norm = norm; fa.inv_freq = inv_freq; fa.st = d_state;
        fa.x = x1; fa.qkv1 = qkv1; fa.h1 = h1; fa.logits = logits; fa.partial = partial;
        fa.sync = d_sync; fa.pmax = pmax; fa.pidx = pidx; fa.argmax_out = d_argmax;
        fa.history = d_history; fa.hist_cap = hist_cap; fa.kv_pool = kv_pool; fa.layer_stride = layer_stride; fa.page_stride = page_stride;
        fa.page_table = d_page_table; fa.nsplit = fused_nsplit;
        { const char* e = getenv("AHA_FUSED_DBG"); fa.dbg = e ? atoi(e) : 0; }
        fa.trace = d_ftrace;
        { const char* e = getenv("AHA_FUSED_STAGES"); fa.stages = e ? std::max(2, std::min(kFusedStages, atoi(e))) : fused_stages; }
        fa.tp_rank = tp_rank; fa.tp_world = tp_world;
        fa.v0 = (int)(((long long)cfg.V * tp_rank) / tp_world);
        fa.V_l = (int)(((long long)cfg.V * (tp_rank + 1)) / tp_world) - fa.v0;
        if (fused_ll) {
            fa.ll_qkv = ll_qkv; fa.ll_pb = ll_pb; fa.ll_att = ll_att; fa.ll_h = ll_h; fa.ll_abort = d_ll_abort;
            if (!ll_peers_ready) {
                LLPeerTab tab{};
                for (int w = 0; w < tp_world; ++w) {
                    AHA_REQUIRE(ll_peer_sym[w] != nullptr, "tensor-parallel peers are not attached");
                    tab.xp[0][w] = ll_peer_sym[w];
                    tab.xp[1][w] = ll_peer_sym[w] + (size_t)tp_world * cfg.H;
                    tab.cand[w] = ll_peer_sym[w] + (size_t)2 * tp_world * cfg.H;
                    uint32_t* fl = reinterpret_cast<uint32_t*>(ll_peer_sym[w] + (size_t)2 * tp_world * cfg.H + (size_t)tp_world * 2);
                    tab.flag_xp[0][w] = fl;
                    tab.flag_xp[1][w] = fl + (size_t)tp_world * 256;
                }
                AHA_CUDA_CHECK(cudaMemcpyAsync(d_ll_peers, &tab, sizeof(tab), cudaMemcpyHostToDevice, c.stream));
                AHA_CUDA_CHECK(cudaStreamSynchronize(c.stream));   // `tab` is a stack temporary
                ll_peers_ready = true;
            }
            fa.ll_peers = d_ll_peers;
            fa.ll_xp_local[0] = ll_sym;
            fa.ll_xp_local[1] = ll_sym + (size_t)tp_world * cfg.H;
            fa.ll_cand_local = ll_sym + (size_t)2 * tp_world * cfg.H;
            {
                uint32_t* fl = reinterpret_cast<uint32_t*>(ll_sym + (size_t)2 * tp_world * cfg.H + (size_t)tp_world * 2);
                fa.ll_flag_xp_local[0] = fl;
                fa.ll_flag_xp_local[1] = fl + (size_t)tp_world * 256;
            }
            fa.ll_flag = ll_flag;
            ll_launches += 1;
            fa.ll_tag = ll_launches * 64u;   // layer l -> tag + l (L <= 62); 0 is the "never written" tag of the zeroed buffers
            AHA_REQUIRE(cfg.L <= 62, "fused decode kernel: more than 62 layers");
        } else {
            fa.v0 = 0; fa.V_l = cfg.V;
        }
        AHA_CUDA_CHECK(cudaMemsetAsync(d_sync, 0, sync_words * sizeof(unsigned), c.stream));
        switch (nh_l / nkv_l) {
            case 1: launch_fused<1>(fa); break;
            case 2: launch_fused<2>(fa); break;
            default: launch_fused<4>(fa); break;
        }
        c.cnt.kernels++;
        step_graph_kernels = 1;
    }
    // full_logits: the caller will read the whole logits row.  Under tensor parallelism the fused kernel multiplies only this
    // rank's vocabulary shard (the winner is exchanged, not the row), so such a step takes the per-op path, whose lm_head
    // is replicated.
    void decode_step(bool full_logits = false) {
        decode_step_argmax(full_logits || samp_active);
        sample(1);
    }
    void decode_step_argmax(bool full_logits) {
        Ctx& c = *ctx;
        if (fused && !(full_logits && tp_world > 1)) { decode_step_fused(); return; }
        if (!use_graph) { decode_step_launches(); return; }
        if (!step_graph) {
            const uint64_t k0 = c.cnt.kernels;
            cudaGraph_t g = nullptr;
            AHA_CUDA_CHECK(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
            try { decode_step_launches(); } catch (...) { cudaStreamEndCapture(c.stream, &g); if (g) cudaGraphDestroy(g); throw; }
            AHA_CUDA_CHECK(cudaStreamEndCapture(c.stream, &g));
            step_graph_kernels = c.cnt.kernels - k0;
            c.cnt.kernels = k0;
            AHA_CUDA_CHECK(cudaGraphInstantiate(&step_graph, g, 0));
            AHA_CUDA_CHECK(cudaGraphDestroy(g));
        }
        AHA_CUDA_CHECK(cudaGraphLaunch(step_graph, c.stream));
        c.cnt.graphs++;
        c.cnt.kernels += step_graph_kernels;
    }
    // ---- sampler.  mode / parameters follow get_logit_processor (sample.rs:7-38); `seed` keys the ChaCha12 stream.
    void set_sampler(int mode, float temperature, float top_p, int top_k, float penalty, int last_n, uint64_t seed) {
        const bool pen = !(penalty == 1.0f || last_n == 0);
        samp_active = mode != SAMPLE_ARGMAX || pen;
        if (!samp_active) return;
        AHA_REQUIRE(cfg.V <= kSampleThreads * kSampleChunk, "vocabulary too large for the device sampler");
        AHA_REQUIRE(!(mode == SAMPLE_TOPK || mode == SAMPLE_TOPK_TOPP) || top_k >= 1, "top_k must be >= 1");
        AHA_REQUIRE(!(mode == SAMPLE_TOPK || mode == SAMPLE_TOPK_TOPP) || top_k >= cfg.V || top_k <= kSampleMaxTopK,
                    "top_k > 1024 is not supported by the device sampler");
        if (!sample_work) {
            sample_work = ctx->alloc<float>((size_t)cfg.V);
            d_sample_err = ctx->alloc<int>(1);
            AHA_CUDA_CHECK(cudaMemset(d_sample_err, 0, sizeof(int)));
        }
        samp = SampleArgs{};
        samp.logits = logits; samp.work = sample_work; samp.V = cfg.V; samp.mode = mode;
        samp.inv_temp = mode == SAMPLE_ARGMAX ? 1.0f : (float)(1.0 / (double)temperature);
        samp.top_p = top_p; samp.top_k = top_k; samp.penalty = penalty; samp.last_n = last_n;
        // rand_core::SeedableRng::seed_from_u64: eight PCG32 outputs fill the 32-byte ChaCha seed
        uint64_t stt = seed;
        for (int i = 0; i < 8; ++i) {
            stt = stt * 6364136223846793005ull + 11634580027462260723ull;
            const uint32_t xs = (uint32_t)(((stt >> 18) ^ stt) >> 27);
            const uint32_t rot = (uint32_t)(stt >> 59);
            samp.key[i] = (xs >> rot) | (xs << ((32u - rot) & 31u));
        }
        samp.st = d_state; samp.history = d_history; samp.hist_cap = hist_cap; samp.token_out = d_argmax; samp.error = d_sample_err;
    }
    void clear_sampler() { samp_active = false; }
    // overwrite = 1: the step kernel has already pushed its ArgMax token; the sampled token replaces it
    void sample(int overwrite) {
        if (!samp_active) return;
        SampleArgs a = samp;
        a.overwrite = overwrite;
        sample_kernel<<<1, kSampleThreads, 0, ctx->stream>>>(a);
        AHA_CUDA_CHECK(cudaGetLastError());
        ctx->cnt.kernels++;
    }
    void check_sample_error() {
        if (samp_active) check_sample_flag();
    }
    // the error flag whichever sampler set it: a batch step samples with each slot's own sampler, not the model's active one
    void check_sample_flag() {
        if (!d_sample_err) return;
        int e = 0;
        AHA_CUDA_CHECK(cudaMemcpy(&e, d_sample_err, sizeof(int), cudaMemcpyDeviceToHost));
        if (e) {
            cudaMemset(d_sample_err, 0, sizeof(int));
            throw std::runtime_error("sampler: the token weights are all zero or not finite (rand::distr::weighted::WeightedIndex::new fails in the reference)");
        }
    }
    void set_state(uint32_t token, int pos, int rope_delta, int n_hist, uint32_t n_draws = 0) {
        DecodeState s{token, pos, rope_delta, n_hist, n_draws, {0, 0, 0}};
        AHA_CUDA_CHECK(cudaMemcpyAsync(d_state, &s, sizeof(s), cudaMemcpyHostToDevice, ctx->stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));  // `s` is a stack temporary
    }
    void destroy() {
        for (int w = 0; w < kFusedMaxTp; ++w)
            if (ll_peer_sym[w] && w != tp_rank) { cudaIpcCloseMemHandle(ll_peer_sym[w]); ll_peer_sym[w] = nullptr; }
        if (step_graph) { cudaGraphExecDestroy(step_graph); step_graph = nullptr; }
        if (comm) { NcclApi::get().CommDestroy(comm); comm = nullptr; }
    }
};

}  // namespace aha
