// api.cu -- extern "C" entry points of libaha_b200.so (see include/aha_b200.h for the contract and the
// reference items each entry replaces).  Host side = the C++ mirror of aha's model structs:
// Qwen3Model (/root/reference/src/models/qwen3/model.rs:94-214), Qwen3VLModel (qwen3vl/model.rs:837-1324),
// Qwen3ASRModel (qwen3_asr/model.rs:308-425) and generate_generic (common/generate.rs:115-159).
#include <array>
#include <chrono>
#include <functional>
#include <mutex>
#include <system_error>
#include <thread>

#include "audio_model.cuh"
#include "preprocess.cuh"
#include "text_model.cuh"
#include "batch_decode.cuh"
#include "vision_model.cuh"

using namespace aha;

namespace {
std::mutex g_err_mu;
std::string g_create_error;
}  // namespace

struct aha_model {
    enum Kind { QWEN3, QWEN3VL, QWEN3_ASR } kind = QWEN3;
    Ctx ctx;
    TextModel text;
    VisionModel vision;
    AudioModel audio;
    std::vector<uint32_t> stop_ids;
    std::string last_error;
    // Qwen3-VL state / config
    int image_token_id = -1, video_token_id = -1, vision_start_token_id = -1;
    bool have_rope_delta = false;  // rope_deltas: Option<Tensor>, qwen3vl/model.rs:842
    int rope_delta = 0;
    int audio_token_id = -1;
    int* d_scatter_idx = nullptr;
    int max_scatter = 0;
    double last_vision_secs = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // pinned staging for the host<->device scalars of a step / the tokens of a burst
    uint32_t* h_pin = nullptr;
    static constexpr int kStreamBurst = 8;   // streaming: steps the device may run ahead of the token being delivered
    cudaEvent_t ev_tok[kStreamBurst] = {};
    // KV reuse across requests (SURVEY 8f rank 4; new design: the reference clears the cache after every request, common/generate.rs:147,
    // and serialises requests behind one lock, server/api.rs:117).  A request that carries AHA_GEN_REUSE_PREFIX leaves its K/V in the paged
    // cache; the next such request prefills only what follows the longest common prefix.
    std::vector<uint32_t> cached_ids;   // tokens whose K/V occupy positions 0 .. n-1 of the paged cache
    uint64_t cached_mm_fp = 0;          // fingerprint of the multimodal tensors those tokens were embedded with (0 = none)
    size_t last_prefix_hit = 0;         // tokens the last generate call did not have to prefill
    BatchDecoder batch;                 // several sequences decoded in lockstep (aha_b200_generate_batch); buffers allocated on first use
    // Continuous batching (aha_b200_batch_open / _add / _step / _close): requests join and leave a running batch between steps
    struct BatchSession {
        bool open = false;
        bool used[kGemvBatchMax] = {};
        size_t budget[kGemvBatchMax] = {}, produced[kGemvBatchMax] = {};
    } session;
};

namespace {

void bind(aha_model* m) { AHA_CUDA_CHECK(cudaSetDevice(m->ctx.device)); }

template <typename F>
int guarded(aha_model* m, F&& f) {
    try {
        if (!m) throw std::runtime_error("null model handle");
        bind(m);
        f();
        return 0;
    } catch (const std::exception& e) {
        if (m) m->last_error = e.what();
        else { std::lock_guard<std::mutex> lk(g_err_mu); g_create_error = e.what(); }
        // leave the stream usable: drop a dangling capture, clear sticky launch errors
        if (m && m->ctx.stream) {
            cudaStreamCaptureStatus cs;
            if (cudaStreamIsCapturing(m->ctx.stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
                cudaGraph_t g = nullptr; cudaStreamEndCapture(m->ctx.stream, &g); if (g) cudaGraphDestroy(g);
            }
        }
        cudaGetLastError();
        return 1;
    }
}

const aha_tensor_desc* mm_entry(const aha_mm* mm, size_t i) {
    if (!mm || i >= mm->n) return nullptr;
    const aha_tensor_desc* d = &mm->data_vec[i];
    return d->data ? d : nullptr;
}

std::vector<float> desc_to_f32(const aha_tensor_desc& d) {
    const size_t n = WeightTable::numel(d);
    std::vector<float> v(n);
    if (d.dtype == AHA_F32) std::memcpy(v.data(), d.data, n * sizeof(float));
    else for (size_t i = 0; i < n; ++i) v[i] = WeightTable::at(d, i);
    return v;
}
std::vector<int64_t> desc_to_i64(const aha_tensor_desc& d) {
    const size_t n = WeightTable::numel(d);
    std::vector<int64_t> v(n);
    for (size_t i = 0; i < n; ++i) {
        switch (d.dtype) {
            case AHA_U32: v[i] = reinterpret_cast<const uint32_t*>(d.data)[i]; break;
            case AHA_I64: v[i] = reinterpret_cast<const int64_t*>(d.data)[i]; break;
            case AHA_U8: v[i] = reinterpret_cast<const uint8_t*>(d.data)[i]; break;
            default: throw std::runtime_error("integer tensor expected");
        }
    }
    return v;
}

// Qwen3VLModel::get_rope_index, image branch (/root/reference/src/models/qwen3vl/model.rs:901-1071,1072-1090):
// text runs get equal t/h/w ids; an image of merged grid (t,h',w') gets t_idx = base, h_idx = base+0..h'-1,
// w_idx = base+0..w'-1; the next run starts at max+1; rope_delta = max+1-S.  pos3 is [3][S].
// video_grid: video_grid_thw with every (t, h, w) row already expanded to t rows of (1, h, w) (model.rs:907-925): each frame group has
// its own <|vision_start|><|video_pad|>... run in the prompt (timestamps sit between them).
void get_rope_index(const uint32_t* ids, int S, const std::vector<std::array<int, 3>>& grid, const std::vector<std::array<int, 3>>& video_grid, int merge,
                    int image_tok, int video_tok, int vstart_tok, std::vector<int>& pos3, int& delta) {
    pos3.assign((size_t)3 * S, 0);
    if (grid.empty() && video_grid.empty()) {
        for (int r = 0; r < 3; ++r) for (int i = 0; i < S; ++i) pos3[(size_t)r * S + i] = i;
        delta = 0;
        return;
    }
    int out = 0;            // tokens emitted so far
    int last_max = -1;      // max of the last pushed chunk
    bool any = false;
    int text_start = 0, text_end = 0;
    size_t image_index = 0, video_index = 0;
    std::array<int, 3> thw{0, 0, 0};
    bool have_thw = false;
    auto push_text = [&](int len) {
        const int start = any ? last_max + 1 : 0;
        for (int i = 0; i < len; ++i) for (int r = 0; r < 3; ++r) pos3[(size_t)r * S + out + i] = start + i;
        if (len > 0) last_max = start + len - 1;
        // an empty chunk has no max in the reference either; it only matters that `any` flips
        any = true;
        out += len;
        return start + len;
    };
    for (int j0 = 0; j0 < S; ++j0) {
        if ((int)ids[j0] != vstart_tok) continue;
        const int j = j0 + 1;
        if (j >= S) throw std::runtime_error("vision_start token at the end of the prompt");
        if ((int)ids[j] == image_tok) {
            if (image_index >= grid.size()) throw std::runtime_error("more image placeholders than image_grid_thw rows");
            thw = grid[image_index++];
            have_thw = true;
            text_end = j;
        }
        if ((int)ids[j] == video_tok && video_tok >= 0) {
            if (video_index >= video_grid.size()) throw std::runtime_error("more video placeholder runs than video_grid_thw frames");
            thw = video_grid[video_index++];
            have_thw = true;
            text_end = j;
        }
        if (!have_thw) throw std::runtime_error("vision_start not followed by an image or video token");
        const int gt = thw[0], gh = thw[1] / merge, gw = thw[2] / merge;
        const int text_len = text_end - text_start;
        if (out + text_len + gt * gh * gw > S) throw std::runtime_error("image placeholders exceed the prompt length");
        const int base = push_text(text_len);
        for (int t = 0; t < gt; ++t)
            for (int h = 0; h < gh; ++h)
                for (int w = 0; w < gw; ++w) {
                    const int i = out + (t * gh + h) * gw + w;
                    pos3[i] = base + t; pos3[(size_t)S + i] = base + h; pos3[(size_t)2 * S + i] = base + w;
                }
        last_max = base + std::max(gt, std::max(gh, gw)) - 1;
        out += gt * gh * gw;
        text_start = text_end + gt * gh * gw;
    }
    if (text_start < S) push_text(S - text_start);
    if (out != S) throw std::runtime_error("get_rope_index: placeholder layout does not cover the prompt");
    int mx = 0;
    for (int v : pos3) mx = std::max(mx, v);
    delta = mx + 1 - S;
}

void upload_ids(aha_model* m, const uint32_t* ids, size_t S) {
    TextModel& T = m->text;
    AHA_REQUIRE(S >= 1, "empty input_ids");
    AHA_REQUIRE((int)S <= T.max_prefill, "prompt of " + std::to_string(S) + " tokens exceeds max_prefill " + std::to_string(T.max_prefill));
    for (size_t i = 0; i < S; ++i) AHA_REQUIRE(ids[i] < (uint32_t)T.cfg.V, "token id out of range");
    AHA_CUDA_CHECK(cudaMemcpyAsync(T.d_ids, ids, S * sizeof(uint32_t), cudaMemcpyHostToDevice, m->ctx.stream));
}
void upload_pos(aha_model* m, const std::vector<int>& pos3) {
    AHA_CUDA_CHECK(cudaMemcpyAsync(m->text.d_pos3, pos3.data(), pos3.size() * sizeof(int), cudaMemcpyHostToDevice, m->ctx.stream));
    AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));  // pos3 may be a temporary
}
void upload_scatter_idx(aha_model* m, const std::vector<int>& idx) {
    AHA_REQUIRE((int)idx.size() <= m->max_scatter, "too many placeholder tokens");
    AHA_CUDA_CHECK(cudaMemcpyAsync(m->d_scatter_idx, idx.data(), idx.size() * sizeof(int), cudaMemcpyHostToDevice, m->ctx.stream));
    AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
}

void fetch_outputs(aha_model* m, float* logits_out, uint32_t* argmax_out) {
    TextModel& T = m->text;
    if (logits_out) AHA_CUDA_CHECK(cudaMemcpyAsync(logits_out, T.logits, (size_t)T.cfg.V * sizeof(float), cudaMemcpyDeviceToHost, m->ctx.stream));
    if (argmax_out) AHA_CUDA_CHECK(cudaMemcpyAsync(m->h_pin, T.d_argmax, sizeof(uint32_t), cudaMemcpyDeviceToHost, m->ctx.stream));
    AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
    T.check_ll_abort();
    if (argmax_out) *argmax_out = m->h_pin[0];
}


// ---- KV reuse across requests: which prefix of the new prompt is already in the cache --------------------------------------------
// Longest prefix of `ids` whose K/V can be taken from a cache holding `cached`: the common prefix, cut to n - 1 (the last prompt token is
// always run: its logits are the request's first output).  Placeholder tokens (<|image_pad|>, <|video_pad|>, <|audio_pad|>) stand for rows
// of the multimodal tensors, so they only count when those tensors are the same (`same_mm`), and every placeholder of BOTH sequences must
// lie inside the common prefix -- the suffix is then plain text whose M-RoPE positions are index + rope_delta (qwen3vl/model.rs:1250-1264).
size_t prefix_match(const uint32_t* cached, size_t n_cached, const uint32_t* ids, size_t n, const uint32_t* mm_tokens, size_t n_mm_tokens, bool same_mm) {
    if (n == 0 || n_cached == 0 || !same_mm) return 0;
    size_t lcp = 0;
    while (lcp < n && lcp < n_cached && cached[lcp] == ids[lcp]) ++lcp;
    auto is_mm = [&](uint32_t t) { for (size_t i = 0; i < n_mm_tokens; ++i) if (mm_tokens[i] == t) return true; return false; };
    for (size_t i = lcp; i < n; ++i) if (is_mm(ids[i])) return 0;
    for (size_t i = lcp; i < n_cached; ++i) if (is_mm(cached[i])) return 0;
    return std::min(lcp, n - 1);
}

// 64-bit fingerprint of a host buffer: four independent multiply-xorshift lanes over 8-byte words, folded with the length.  Buffers
// beyond 1 MiB are cut into 1 MiB blocks hashed by up to 8 threads and folded in block order (the value does not depend on the thread
// count).  Not cryptographic: it guards a cache, not a boundary.
uint64_t fingerprint_block(const unsigned char* p, size_t n, uint64_t seed) {
    uint64_t h[4] = {seed ^ 0x9e3779b97f4a7c15ull, seed ^ 0xbf58476d1ce4e5b9ull, seed ^ 0x94d049bb133111ebull, seed ^ 0x2545f4914f6cdd1dull};
    const uint64_t k = 0xff51afd7ed558ccdull;
    size_t i = 0;
    for (; i + 32 <= n; i += 32) {
        uint64_t w[4];
        std::memcpy(w, p + i, 32);
        for (int l = 0; l < 4; ++l) { h[l] = (h[l] ^ w[l]) * k; h[l] ^= h[l] >> 29; }
    }
    uint64_t tail[4] = {0, 0, 0, 0};
    if (n > i) std::memcpy(tail, p + i, n - i);
    for (int l = 0; l < 4; ++l) { h[l] = (h[l] ^ tail[l]) * k; h[l] ^= h[l] >> 29; }
    uint64_t r = (uint64_t)n * 0xc4ceb9fe1a85ec53ull;
    for (int l = 0; l < 4; ++l) { r = (r ^ h[l]) * k; r ^= r >> 32; }
    return r;
}
uint64_t fingerprint_bytes(const void* data, size_t n, uint64_t seed) {
    const unsigned char* p = static_cast<const unsigned char*>(data);
    constexpr size_t kBlock = (size_t)1 << 20;
    if (n <= kBlock) return fingerprint_block(p, n, seed);
    const size_t nb = (n + kBlock - 1) / kBlock;
    std::vector<uint64_t> hb(nb);
    const unsigned nt = (unsigned)std::min<size_t>(std::min<size_t>(8, std::max(1u, std::thread::hardware_concurrency())), nb);
    auto work = [&](unsigned t) { for (size_t b = t; b < nb; b += nt) hb[b] = fingerprint_block(p + b * kBlock, std::min(kBlock, n - b * kBlock), seed + b); };
    std::vector<std::thread> th;
    unsigned started = 1;   // lane 0 is this thread
    try {
        for (unsigned t = 1; t < nt; ++t) { th.emplace_back(work, t); ++started; }
    } catch (const std::system_error&) {}   // no more threads to be had: the lanes that did not start are hashed here (same blocks, same value)
    work(0);
    for (unsigned t = started; t < nt; ++t) work(t);
    for (auto& x : th) x.join();
    return fingerprint_block(reinterpret_cast<const unsigned char*>(hb.data()), nb * sizeof(uint64_t), seed ^ (uint64_t)n);
}
// fingerprint of a request's MultiModalData (0 when it carries no tensor): dtype, shape and bytes of every present entry
uint64_t mm_fingerprint(const aha_mm* mm) {
    uint64_t fp = 0;
    for (size_t i = 0; mm && i < mm->n; ++i) {
        const aha_tensor_desc* d = mm_entry(mm, i);
        if (!d) continue;
        size_t esz = 4;
        switch (d->dtype) { case AHA_F16: case AHA_BF16: esz = 2; break; case AHA_I64: esz = 8; break; case AHA_U8: esz = 1; break; default: break; }
        uint64_t meta[11] = {(uint64_t)i + 1, (uint64_t)d->dtype, (uint64_t)d->rank};
        for (int r = 0; r < d->rank && r < 8; ++r) meta[3 + r] = (uint64_t)d->shape[r];
        fp = fingerprint_bytes(meta, sizeof(meta), fp);
        fp = fingerprint_bytes(d->data, WeightTable::numel(*d) * esz, fp);
        if (fp == 0) fp = 1;
    }
    return fp;
}
std::vector<uint32_t> mm_token_ids(const aha_model* m) {
    std::vector<uint32_t> t;
    for (int v : {m->image_token_id, m->video_token_id, m->audio_token_id}) if (v >= 0) t.push_back((uint32_t)v);
    return t;
}
void require_no_session(aha_model* m) {
    AHA_REQUIRE(!m->session.open, "a batch session is open on this handle: call aha_b200_batch_close first");
}
bool is_stop_token(const aha_model* m, uint32_t t) {
    for (uint32_t e : m->stop_ids) if (e == t) return true;
    return false;
}
bool env_flag(const char* name, bool dflt) { const char* v = std::getenv(name); return v ? std::atoi(v) != 0 : dflt; }
int env_int(const char* name, int dflt) { const char* v = std::getenv(name); return v ? std::atoi(v) : dflt; }
// projections of the batched step: 0 = batched GEMV with the weights in registers, 1 = exact SIMT GEMM (validation twin), 2 = batched GEMV with the
// cp.async weight ring
constexpr int kBatchGemvDefault = 2;   // call 25: bit-identical to 0 on every tested shape and faster at every batch size (1.89 vs 2.19 ms per step at 1 request, 4.21 vs 4.31 at 8)

// model.clear_cache(): pages, rope_deltas, and what the prefix cache remembered
void drop_cache(aha_model* m) {
    m->text.reset_pages();
    m->have_rope_delta = false;  // qwen3vl/model.rs:1279-1282
    m->rope_delta = 0;
    m->cached_ids.clear();
    m->cached_mm_fp = 0;
}

// The multi-token forward (prefill).  Mirrors Qwen3Model::forward / Qwen3VLModel::forward / Qwen3ASRThinker::forward.
void forward_prefill(aha_model* m, const uint32_t* ids, size_t S, size_t offset, const aha_mm* mm, bool initial) {
    TextModel& T = m->text;
    Ctx& c = m->ctx;
    upload_ids(m, ids, S);
    std::vector<int> pos3((size_t)3 * S);
    std::vector<const float*> deepstack;
    int n_visual = 0;
    bool embeds_ready = false;
    m->last_vision_secs = 0;
    if (m->kind == aha_model::QWEN3VL) {
        if (initial) AHA_REQUIRE(mm && mm->n == 5, "Qwen3VL process data error, must have pixel_values, image_grid_thw, pixel_values_video, video_grid_thw, cache_position");
        const aha_tensor_desc* pv = initial ? mm_entry(mm, 0) : nullptr;
        const aha_tensor_desc* thw = initial ? mm_entry(mm, 1) : nullptr;
        const aha_tensor_desc* pvv = initial ? mm_entry(mm, 2) : nullptr;
        const aha_tensor_desc* vthw = initial ? mm_entry(mm, 3) : nullptr;
        if (!(pv && thw)) { pv = nullptr; thw = nullptr; }       // `if let Some(pixel_values) && let Some(image_grid_thw)` (model.rs:1150-1151)
        if (!(pvv && vthw)) { pvv = nullptr; vthw = nullptr; }   // the same for the video pair (model.rs:1169-1170)
        std::vector<std::array<int, 3>> grid, vgrid, vgrid_frames;
        auto read_grid = [&](const aha_tensor_desc& d, std::vector<std::array<int, 3>>& out, const char* what) {
            auto g = desc_to_i64(d);
            AHA_REQUIRE(g.size() % 3 == 0 && !g.empty(), std::string(what) + " must be (n, 3)");
            int N = 0;
            for (size_t i = 0; i < g.size(); i += 3) { out.push_back({(int)g[i], (int)g[i + 1], (int)g[i + 2]}); N += (int)(g[i] * g[i + 1] * g[i + 2]); }
            return N;
        };
        if (pv || pvv) {
            VisionModel& V = m->vision;
            const int N_img = pv ? read_grid(*thw, grid, "image_grid_thw") : 0;
            const int N_vid = pvv ? read_grid(*vthw, vgrid, "video_grid_thw") : 0;
            for (auto& g : vgrid) for (int t = 0; t < g[0]; ++t) vgrid_frames.push_back({1, g[1], g[2]});
            const int N = N_img + N_vid, m2 = V.cfg.merge * V.cfg.merge;
            if (pv) AHA_REQUIRE(pv->rank == 2 && pv->shape[0] == N_img && pv->shape[1] == V.patch_dim, "pixel_values shape does not match image_grid_thw");
            if (pvv) AHA_REQUIRE(pvv->rank == 2 && pvv->shape[0] == N_vid && pvv->shape[1] == V.patch_dim, "pixel_values_video shape does not match video_grid_thw");
            AHA_REQUIRE(N <= V.max_patches, "image needs " + std::to_string(N) + " patches, max_patches is " + std::to_string(V.max_patches));
            // placeholder positions + count checks (model.rs:1158-1164, 1176-1183: the video branch raises the same text); the scatter list is
            // the image positions followed by the video positions, matching the row order of the tower's output below
            std::vector<int> idx, vidx;
            for (size_t i = 0; i < S; ++i) {
                if (pv && (int)ids[i] == m->image_token_id) idx.push_back((int)i);
                if (pvv && (int)ids[i] == m->video_token_id) vidx.push_back((int)i);
            }
            if (pv && (int)idx.size() != N_img / m2)
                throw std::runtime_error("n_image_token num: " + std::to_string(idx.size()) + " not equal to image_embed len: " + std::to_string(N_img / m2));
            if (pvv && (int)vidx.size() != N_vid / m2)
                throw std::runtime_error("n_image_token num: " + std::to_string(vidx.size()) + " not equal to image_embed len: " + std::to_string(N_vid / m2));
            idx.insert(idx.end(), vidx.begin(), vidx.end());
            const int n_embed = N / m2;
            // pixel rows -> HBM (images, then video frames), one pass of the tower over both: every grid entry is independent through all
            // blocks and mergers, so this equals the reference's two get_vision_features calls
            auto put = [&](const aha_tensor_desc& d, size_t row0, size_t rows) {
                float* dst = V.pix + row0 * V.patch_dim;
                if (d.dtype == AHA_F32) AHA_CUDA_CHECK(cudaMemcpyAsync(dst, d.data, rows * V.patch_dim * sizeof(float), cudaMemcpyHostToDevice, c.stream));
                else { auto f = desc_to_f32(d); AHA_CUDA_CHECK(cudaMemcpyAsync(dst, f.data(), f.size() * sizeof(float), cudaMemcpyHostToDevice, c.stream)); AHA_CUDA_CHECK(cudaStreamSynchronize(c.stream)); }
            };
            if (pv) put(*pv, 0, (size_t)N_img);
            if (pvv) put(*pvv, (size_t)N_img, (size_t)N_vid);
            std::vector<std::array<int, 3>> all = grid;
            all.insert(all.end(), vgrid.begin(), vgrid.end());
            AHA_CUDA_CHECK(cudaEventRecord(m->ev0, c.stream));
            V.forward(N, all);
            AHA_CUDA_CHECK(cudaEventRecord(m->ev1, c.stream));
            upload_scatter_idx(m, idx);
            embed_gather_kernel<<<(unsigned)S, 256, 0, c.stream>>>(T.d_ids, T.embed, T.x, (int)S, T.cfg.H, T.cfg.V); c.cnt.kernels++;
            scatter_rows_kernel<<<n_embed, 256, 0, c.stream>>>(m->d_scatter_idx, V.image_embeds, T.x, T.cfg.H, 0); c.cnt.kernels++;
            embeds_ready = true;
            n_visual = n_embed;   // deepstack: x[idx[r]] += ds[r] over the same list = the joint embedding of model.rs:1189-1225
            for (float* p : V.ds_out) deepstack.push_back(p);
        }
        // positions: first call -> get_rope_index, later -> arange + offset + rope_deltas (model.rs:1226-1264)
        if (!m->have_rope_delta || (initial && offset == 0)) {   // cache_position[0] == 0 recomputes get_rope_index even when rope_deltas is set (model.rs:1228)
            int delta = 0;
            get_rope_index(ids, (int)S, grid, vgrid_frames, m->vision.cfg.merge, m->image_token_id, m->video_token_id, m->vision_start_token_id, pos3, delta);
            m->rope_delta = delta; m->have_rope_delta = true;
        } else {
            for (int r = 0; r < 3; ++r) for (size_t i = 0; i < S; ++i) pos3[(size_t)r * S + i] = (int)(i + offset) + m->rope_delta;
        }
    } else if (m->kind == aha_model::QWEN3_ASR) {
        if (initial) AHA_REQUIRE(mm && mm->n == 1, "Qwen3 asr process data error, must have input_features");
        const aha_tensor_desc* feat = initial ? mm_entry(mm, 0) : nullptr;
        if (feat) {
            AHA_REQUIRE(feat->rank == 2 && feat->shape[0] == m->audio.cfg.mel, "input_features must be (num_mel_bins, frames)");
            const int Tm = (int)feat->shape[1];
            AHA_REQUIRE(Tm <= m->audio.max_frames, "input_features longer than max_frames");
            auto f = desc_to_f32(*feat);
            AHA_CUDA_CHECK(cudaMemcpyAsync(m->audio.d_mel, f.data(), f.size() * sizeof(float), cudaMemcpyHostToDevice, c.stream));
            AHA_CUDA_CHECK(cudaStreamSynchronize(c.stream));
            AHA_CUDA_CHECK(cudaEventRecord(m->ev0, c.stream));
            const int n_tok = m->audio.forward(m->audio.d_mel, Tm);
            AHA_CUDA_CHECK(cudaEventRecord(m->ev1, c.stream));
            std::vector<int> idx;
            for (size_t i = 0; i < S; ++i) if ((int)ids[i] == m->audio_token_id) idx.push_back((int)i);
            if ((int)idx.size() != n_tok)  // qwen3_asr/model.rs:348-354
                throw std::runtime_error("n_audio_tokens num: " + std::to_string(idx.size()) + " not equal to audio_feature len: " + std::to_string(n_tok));
            upload_scatter_idx(m, idx);
            embed_gather_kernel<<<(unsigned)S, 256, 0, c.stream>>>(T.d_ids, T.embed, T.x, (int)S, T.cfg.H, T.cfg.V); c.cnt.kernels++;
            scatter_rows_kernel<<<n_tok, 256, 0, c.stream>>>(m->d_scatter_idx, m->audio.audio_embeds, T.x, T.cfg.H, 0); c.cnt.kernels++;
            embeds_ready = true;
        }
        for (int r = 0; r < 3; ++r) for (size_t i = 0; i < S; ++i) pos3[(size_t)r * S + i] = (int)(i + offset);
    } else {
        for (int r = 0; r < 3; ++r) for (size_t i = 0; i < S; ++i) pos3[(size_t)r * S + i] = (int)(i + offset);
    }
    upload_pos(m, pos3);
    T.prefill((int)S, (int)offset, embeds_ready, m->d_scatter_idx, n_visual, deepstack);
}

// `extend`: prefill continuation (new design) -- S >= 1 further tokens against a cache that already holds `offset` tokens; the causal mask is
// the (S, offset + S) one the reference never builds (its (S, S) mask makes a multi-token call with a non-empty cache fail, qwen3/model.rs:164-175).
void forward_any(aha_model* m, const uint32_t* ids, size_t S, size_t offset, const aha_mm* mm, bool initial, float* logits_out, uint32_t* argmax_out,
                 bool extend = false, bool force_prefill = false) {
    TextModel& T = m->text;
    AHA_REQUIRE(ids != nullptr && S >= 1, "input_ids must hold at least one token");
    AHA_REQUIRE(offset + S <= (size_t)T.max_ctx, "context exceeds max_ctx");
    const bool has_mm = initial && mm && ((m->kind == aha_model::QWEN3VL && (mm_entry(mm, 0) || mm_entry(mm, 2))) || (m->kind == aha_model::QWEN3_ASR && mm_entry(mm, 0)));
    if (initial && m->kind == aha_model::QWEN3VL) AHA_REQUIRE(mm && mm->n == 5, "Qwen3VL process data error, must have pixel_values, image_grid_thw, pixel_values_video, video_grid_thw, cache_position");
    if (initial && m->kind == aha_model::QWEN3_ASR) AHA_REQUIRE(mm && mm->n == 1, "Qwen3 asr process data error, must have input_features");
    if (S == 1 && !has_mm && !extend && !force_prefill && (m->kind != aha_model::QWEN3VL || m->have_rope_delta)) {
        // decode step: single token against the cache
        AHA_REQUIRE(ids[0] < (uint32_t)T.cfg.V, "token id out of range");
        T.ensure_tokens((int)offset + 1);
        T.set_state(ids[0], (int)offset, m->kind == aha_model::QWEN3VL ? m->rope_delta : 0, 0);
        T.decode_step(logits_out != nullptr);
    } else {
        // The reference builds an (S,S) causal mask with offset 0 for every multi-token call
        // (qwen3/model.rs:164-175); with a non-empty cache its broadcast_add against (S, off+S) scores fails.
        if (!extend) AHA_REQUIRE(offset == 0, "seq_len > 1 with seqlen_offset > 0 is not supported (the reference's mask shape rejects it too)");
        else AHA_REQUIRE(offset <= (size_t)T.pages_mapped * kPage, "forward_extend: seqlen_offset is beyond the tokens in the cache");
        // A prompt longer than the activation workspace (max_prefill) runs as consecutive chunks against the growing cache: the first chunk is
        // the reference's call (multimodal rows are scattered there), the others are continuations.  Same K/V, same logits for the last token.
        const size_t chunk = (size_t)T.max_prefill;
        size_t done = 0;
        while (done < S) {
            const size_t n = std::min(chunk, S - done);
            const bool first = done == 0;
            if (first && !extend) {
                if (n < S && has_mm) {   // every placeholder row must be embedded by the call that carries the tensors
                    const auto mmt = mm_token_ids(m);
                    for (size_t i = n; i < S; ++i) for (uint32_t t : mmt) AHA_REQUIRE(ids[i] != t, "prompt exceeds max_prefill before its last multimodal placeholder");
                }
                // (Qwen3-VL: get_rope_index over the first chunk yields the whole prompt's rope_delta, because only text follows the last placeholder)
                forward_prefill(m, ids, n, offset, mm, initial);
            } else forward_prefill(m, ids + done, n, offset + done, nullptr, false);
            done += n;
        }
        T.finish_argmax(0);
        T.sample(0);   // device sampler of generate(): penalty / temperature / top-k / top-p on the prefill logits (no-op for plain ArgMax)
    }
    fetch_outputs(m, logits_out, argmax_out);
    if (m->kind != aha_model::QWEN3 && has_mm) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, m->ev0, m->ev1) == cudaSuccess) m->last_vision_secs = ms * 1e-3;
    }
}

}  // namespace

extern "C" {

int aha_b200_abi_version(void) { return AHA_B200_ABI_VERSION; }

int aha_b200_create(const char* kind, const char* config_json, const aha_tensor_desc* weights, size_t n_weights, const uint32_t* eos_ids,
                    size_t n_eos, const aha_options* opts, aha_model** out) {
    if (!out) return 1;
    *out = nullptr;
    aha_model* m = nullptr;
    try {
        AHA_REQUIRE(kind && config_json && weights, "kind, config_json and weights are required");
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
            throw std::runtime_error("no CUDA device visible: libaha_b200 has no CPU fallback");
        aha_options o{};
        if (opts) o = *opts;
        o.use_graph = opts ? opts->use_graph : 1;
        AHA_REQUIRE(o.device >= 0 && o.device < ndev, "invalid device ordinal");
        cudaDeviceProp prop;
        AHA_CUDA_CHECK(cudaGetDeviceProperties(&prop, o.device));
        AHA_REQUIRE(prop.major == 10, std::string("device '") + prop.name + "' is not sm_100-class (this library is built for sm_100a only)");
        m = new aha_model();
        m->ctx.device = o.device;
        m->ctx.num_sms = prop.multiProcessorCount;
        m->ctx.gemm_impl = o.gemm_impl;
        { const char* e = getenv("AHA_GEMM_WIDE"); if (e) m->ctx.gemm_wide = atoi(e) != 0; }
        { const char* e = getenv("AHA_GEMM_GROUP"); if (e) m->ctx.gemm_group_m = atoi(e); }
        { const char* e = getenv("AHA_GEMM_PAIR"); if (e) m->ctx.gemm_pair = atoi(e) != 0; }
        { const char* e = getenv("AHA_PRESPLIT"); if (e) m->ctx.presplit = atoi(e) != 0; }
        m->ctx.attn_impl = o.reserved[0];   // 0 = tensor-core flash attention (tcgen05 for head_dim 64), 1 = fp32 SIMT twin, 2 = mma.sync kernel everywhere
        AHA_CUDA_CHECK(cudaSetDevice(o.device));
        AHA_CUDA_CHECK(cudaStreamCreateWithFlags(&m->ctx.stream, cudaStreamNonBlocking));
        AHA_CUDA_CHECK(cudaEventCreate(&m->ev0));
        AHA_CUDA_CHECK(cudaEventCreate(&m->ev1));
        AHA_CUDA_CHECK(cudaMallocHost(&m->h_pin, 64 * sizeof(uint32_t)));
        for (auto& e : m->ev_tok) AHA_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        gemv_init();
        gemm_tc_init();
        flash_attn_tc_init();
        const std::string k = kind;
        const std::string cfg_text = config_json;
        Json root = JsonParser(cfg_text).parse();
        WeightTable wt(weights, n_weights);
        const int tp_rank = o.tp_world > 1 ? o.tp_rank : 0, tp_world = o.tp_world > 1 ? o.tp_world : 1;
        const int max_ctx = o.max_ctx > 0 ? o.max_ctx : 8192;
        const int max_prefill = o.max_prefill > 0 ? o.max_prefill : max_ctx;
        TextCfg tc;
        if (k == "qwen3") {
            m->kind = aha_model::QWEN3;
            tc = TextCfg::from_json(root);
            const std::string prefix = wt.has("model.embed_tokens.weight") ? "model." : "";  // qwen3/model.rs:105-109
            m->text.load(m->ctx, tc, wt, prefix, "lm_head.weight", tp_rank, tp_world);
        } else if (k == "qwen3vl") {
            m->kind = aha_model::QWEN3VL;
            tc = TextCfg::from_json(root.at("text_config"));
            tc.tie = root.boolean_or("tie_word_embeddings", false);  // lm_head tying follows the TOP-LEVEL flag (model.rs:853-861)
            AHA_REQUIRE(tc.mrope, "text_config.rope_scaling.mrope_section is required for Qwen3-VL");
            m->image_token_id = root.integer("image_token_id"); m->video_token_id = root.integer_or("video_token_id", -1);
            m->vision_start_token_id = root.integer("vision_start_token_id");
            m->text.load(m->ctx, tc, wt, "model.language_model.", "lm_head.weight", tp_rank, tp_world);
            m->vision.load(m->ctx, VisionCfg::from_json(root.at("vision_config")), wt, "model.visual.", o.max_patches > 0 ? o.max_patches : 16384);
            AHA_REQUIRE(m->vision.cfg.out_hidden == tc.H, "vision out_hidden_size must equal the text hidden_size");
        } else if (k == "qwen3_asr") {
            m->kind = aha_model::QWEN3_ASR;
            const Json& tk = root.at("thinker_config");
            tc = TextCfg::from_json(tk.at("text_config"));
            tc.mrope_asr = true;  // apply_interleaved_mrope_asr index rule (rope.rs:478-500); rows are identical so it is numerically a no-op
            m->audio_token_id = tk.integer("audio_token_id");
            m->text.load(m->ctx, tc, wt, "thinker.model.", "thinker.lm_head.weight", tp_rank, tp_world);
            m->audio.load(m->ctx, AudioCfg::from_json(tk.at("audio_config")), wt, "thinker.audio_tower.", o.max_frames > 0 ? o.max_frames : 3000);
            AHA_REQUIRE(m->audio.cfg.out_dim == tc.H, "audio output_dim must equal the text hidden_size");
        } else {
            throw std::runtime_error("unknown model kind '" + k + "' (expected qwen3 | qwen3vl | qwen3_asr)");
        }
        m->text.alloc_runtime(max_ctx, max_prefill, o.use_graph != 0, o.decode_impl);
        m->text.init_tp(o.tp_comm);
        if (m->kind == aha_model::QWEN3VL) m->vision.set_tp(m->text.tp_rank, m->text.tp_world, m->text.comm);   // images sharded over the ranks
        m->max_scatter = max_prefill;
        m->d_scatter_idx = m->ctx.alloc<int>(max_prefill);
        for (size_t i = 0; i < n_eos; ++i) m->stop_ids.push_back(eos_ids[i]);
        AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        AHA_CUDA_CHECK(cudaDeviceSynchronize());
        *out = m;
        return 0;
    } catch (const std::exception& e) {
        {
            std::lock_guard<std::mutex> lk(g_err_mu);
            g_create_error = e.what();
        }
        cudaGetLastError();
        if (m) aha_b200_destroy(m);
        return 1;
    }
}

int aha_b200_forward_initial(aha_model* m, const uint32_t* ids, size_t seq_len, size_t seqlen_offset, const aha_mm* mm, float* logits_out,
                             uint32_t* argmax_out) {
    return guarded(m, [&] { require_no_session(m); m->cached_ids.clear(); forward_any(m, ids, seq_len, seqlen_offset, mm, true, logits_out, argmax_out); });
}

int aha_b200_forward_step(aha_model* m, const uint32_t* ids, size_t seq_len, size_t seqlen_offset, float* logits_out, uint32_t* argmax_out) {
    return guarded(m, [&] { require_no_session(m); m->cached_ids.clear(); forward_any(m, ids, seq_len, seqlen_offset, nullptr, false, logits_out, argmax_out); });
}

int aha_b200_forward_extend(aha_model* m, const uint32_t* ids, size_t seq_len, size_t seqlen_offset, float* logits_out, uint32_t* argmax_out) {
    return guarded(m, [&] { require_no_session(m); m->cached_ids.clear(); forward_any(m, ids, seq_len, seqlen_offset, nullptr, false, logits_out, argmax_out, true); });
}

size_t aha_b200_last_prefix_hit(aha_model* m) { return m ? m->last_prefix_hit : 0; }

size_t aha_b200_prefix_match(const uint32_t* cached, size_t n_cached, const uint32_t* ids, size_t n, const uint32_t* mm_token_ids, size_t n_mm_tokens,
                             int same_mm) {
    if ((!cached && n_cached) || (!ids && n) || (!mm_token_ids && n_mm_tokens)) return 0;
    return prefix_match(cached, n_cached, ids, n, mm_token_ids, n_mm_tokens, same_mm != 0);
}

uint64_t aha_b200_mm_fingerprint(const aha_mm* mm) { return mm_fingerprint(mm); }

size_t aha_b200_stop_token_ids(aha_model* m, uint32_t* out, size_t cap) {
    if (!m) return 0;
    for (size_t i = 0; i < m->stop_ids.size() && i < cap && out; ++i) out[i] = m->stop_ids[i];
    return m->stop_ids.size();
}

namespace {

// get_logit_processor (sample.rs:7-38): which Sampling the request's parameters select
int sampling_mode(const aha_gen_params& p) {
    const bool has_t = !(p.temperature < 1e-7f);
    const bool has_k = p.top_k > 0, has_p = p.top_p > 0.f;
    if (!has_t) return SAMPLE_ARGMAX;
    if (!has_k) return has_p ? SAMPLE_TOPP : SAMPLE_ALL;
    return has_p ? SAMPLE_TOPK_TOPP : SAMPLE_TOPK;
}

struct GenSink {   // receives every generated token in order; returns true to stop the request (client went away)
    std::function<bool(uint32_t token, size_t index)> push;
};

// generate_generic / generate_stream_generic (common/generate.rs:115-159, 231-368) with the loop on the device:
// forward_initial + sample, then decode steps chained through DecodeState (token, position, history, RNG draw index all
// live in HBM); the host only looks at the tokens, a burst behind the device.  `stream`: tokens are handed to the sink one
// by one as their step completes (per-step event) while the device keeps running ahead inside the burst.
void generate_impl(aha_model* m, const uint32_t* ids, size_t seq_len, const aha_mm* mm, const aha_gen_params& params, const GenSink& sink, bool stream,
                   aha_usage* usage, size_t* n_generated) {
    TextModel& T = m->text;
    require_no_session(m);
    const size_t sample_len = std::max<size_t>(params.max_tokens, 1);   // `for _ in 1..sample_len`: sample_len 0 and 1 both yield exactly one token
    AHA_REQUIRE(seq_len + sample_len <= (size_t)T.max_ctx,
                "prompt + max_tokens exceeds max_ctx (the handle's KV capacity, aha_options.max_ctx; the reference's cache is unbounded)");
    using clk = std::chrono::steady_clock;
    const auto t0 = clk::now();   // prompt_secs covers everything up to the first token, the prefix lookup (fingerprint of the tensors) included
    const bool eos_on_first = (params.flags & AHA_GEN_EOS_ON_FIRST) != 0;
    // KV reuse (AHA_GEN_REUSE_PREFIX): how much of this prompt the cache already holds.  Every path that is not a hit starts from
    // model.clear_cache(), exactly where the reference starts every request.
    const bool reuse = (params.flags & AHA_GEN_REUSE_PREFIX) != 0;
    size_t hit = 0;
    uint64_t mm_fp = 0;
    if (reuse) {
        mm_fp = mm_fingerprint(mm);
        const auto mmt = mm_token_ids(m);
        hit = prefix_match(m->cached_ids.data(), m->cached_ids.size(), ids, seq_len, mmt.data(), mmt.size(), mm_fp == m->cached_mm_fp);
    }
    if (hit == 0) drop_cache(m);
    m->cached_ids.clear();   // the cache is being written: nothing is reusable until this request has completed
    m->last_prefix_hit = hit;
    std::vector<uint32_t> produced;   // what the request generated (the K/V of all but the last token end up in the cache)
    struct Reset {   // model.clear_cache() (generate.rs:147) -- also on the error path, so that a failed request never leaves rope_delta / pages behind
        aha_model* m;
        bool keep = false;
        ~Reset() { if (!keep) drop_cache(m); m->text.clear_sampler(); }
    } reset{m};
    const int mode = sampling_mode(params);
    uint32_t draws0 = 0;
    if ((params.flags & AHA_GEN_CONTINUE_RNG) != 0) {   // one LogitsProcessor across the chunks of a request: keep its stream position
        DecodeState cur;
        AHA_CUDA_CHECK(cudaMemcpy(&cur, T.d_state, sizeof(cur), cudaMemcpyDeviceToHost));
        draws0 = cur.n_draws;
    }
    T.set_sampler(mode, params.temperature, params.top_p, params.top_k, params.repeat_penalty, params.repeat_last_n, params.seed);
    T.set_state(0, 0, 0, 0, draws0);    // empty history: the first token sees no repeat-penalty context
    uint32_t tok = 0;
    if (hit > 0) forward_any(m, ids + hit, seq_len - hit, hit, nullptr, false, nullptr, &tok, true);   // only the tokens the cache does not hold yet
    else forward_any(m, ids, seq_len, 0, mm, true, nullptr, &tok);   // forward_initial + sample_and_push
    T.check_sample_error();
    const auto t1 = clk::now();
    const double vision_secs = m->last_vision_secs;
    size_t done = 1;
    produced.push_back(tok);
    bool stop = sink.push(tok, 0) || (eos_on_first && is_stop_token(m, tok));   // generate_generic never EOS-checks the first token; the ASR loop does
    if (sample_len > 1 && !stop) {
        T.ensure_tokens((int)(seq_len + sample_len));
        DecodeState cur;
        AHA_CUDA_CHECK(cudaMemcpy(&cur, T.d_state, sizeof(cur), cudaMemcpyDeviceToHost));
        T.set_state(tok, (int)seq_len, m->kind == aha_model::QWEN3VL ? m->rope_delta : 0, 1, cur.n_draws);
        AHA_CUDA_CHECK(cudaMemcpy(T.d_history, &tok, sizeof(uint32_t), cudaMemcpyHostToDevice));   // history[0] = first token (penalty context)
        const size_t burst_max = stream ? (size_t)aha_model::kStreamBurst : 32;
        while (done < sample_len && !stop) {
            const size_t n = std::min<size_t>(burst_max, sample_len - done);
            for (size_t i = 0; i < n; ++i) {
                T.decode_step();
                if (stream) {
                    AHA_CUDA_CHECK(cudaMemcpyAsync(m->h_pin + i, T.d_history + done + i, sizeof(uint32_t), cudaMemcpyDeviceToHost, m->ctx.stream));
                    AHA_CUDA_CHECK(cudaEventRecord(m->ev_tok[i], m->ctx.stream));
                }
            }
            if (!stream) {
                AHA_CUDA_CHECK(cudaMemcpyAsync(m->h_pin, T.d_history + done, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, m->ctx.stream));
                AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
            }
            for (size_t i = 0; i < n && !stop; ++i) {
                if (stream) AHA_CUDA_CHECK(cudaEventSynchronize(m->ev_tok[i]));
                const uint32_t t = m->h_pin[i];
                ++done;
                produced.push_back(t);
                stop = sink.push(t, done - 1) || is_stop_token(m, t);   // an EOS token is pushed before the break (generate.rs:139-141)
            }
            AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
            T.check_ll_abort();
            T.check_sample_error();
        }
    }
    const auto t2 = clk::now();
    if (reuse) {
        // the cache now holds the prompt and every generated token that was fed back (all but the last one): step j wrote the K/V of token j-1.
        // Steps the device ran past an EOS inside a burst wrote positions beyond that; they are simply overwritten by the next request.
        m->cached_ids.assign(ids, ids + seq_len);
        m->cached_ids.insert(m->cached_ids.end(), produced.begin(), produced.end() - 1);
        m->cached_mm_fp = mm_fp;
        reset.keep = true;
    }
    if (n_generated) *n_generated = done;
    if (usage) {
        usage->prompt_tokens += (uint32_t)seq_len;
        usage->completion_tokens += (uint32_t)done;
        usage->prompt_secs += std::chrono::duration<double>(t1 - t0).count();
        usage->completion_secs += std::chrono::duration<double>(t2 - t1).count();
        usage->vision_secs += vision_secs;
    }
}

}  // namespace

namespace {
// ---- continuous batching: the same slots and the same step, with requests joining and leaving between steps -------------------------
// (new design; the reference's server holds ONE request behind a write lock, server/api.rs:117.)  A finished request's pages go back to the
// free list at once, so a waiting request can take its place while the others keep decoding.
void session_release(aha_model* m, int slot) {
    BatchSlot& sl = m->batch.slots[slot];
    for (int k = 0; k < sl.mapped; ++k) m->text.free_pages.push_back(sl.h_table[k]);
    sl.mapped = 0;
    sl.samp_active = false;
    m->session.used[slot] = false;
    m->batch.table_for.clear();
    m->batch.clear_graphs();       // the graphs of compositions holding this slot carry its sampler arguments by value
}
void session_close(aha_model* m) {
    m->batch.reset();
    m->session = aha_model::BatchSession{};
    drop_cache(m);
    m->text.clear_sampler();
}
void session_open(aha_model* m) {
    TextModel& T = m->text;
    require_no_session(m);
    AHA_REQUIRE(T.tp_world == 1, "batch sessions are single-GPU");
    AHA_REQUIRE(T.max_prefill >= kGemvBatchMax, "batch sessions need max_prefill >= 8");
    drop_cache(m);
    m->batch.init(T, kGemvBatchMax);
    m->batch.reset();
    m->session = aha_model::BatchSession{};
    m->session.open = true;
}
// One request into a free slot: the reference's forward_initial + sample_and_push on the slot's own page table (swapped into the TextModel
// for the duration, so tower / M-RoPE / deepstack / sampler-on-prefill are the single-request code), then its decode state, history and
// sampler move into the slot.
void session_add(aha_model* m, const aha_batch_request& r, int* slot_out, uint32_t* first_token, int* finished, aha_usage* usage) {
    TextModel& T = m->text;
    BatchDecoder& B = m->batch;
    AHA_REQUIRE(m->session.open, "no batch session is open (aha_b200_batch_open)");
    AHA_REQUIRE(r.ids && r.seq_len >= 1, "batch_add: the request needs input_ids");
    AHA_REQUIRE((r.params.flags & (AHA_GEN_CONTINUE_RNG | AHA_GEN_REUSE_PREFIX)) == 0, "batch_add: CONTINUE_RNG / REUSE_PREFIX are per-handle states of the single-request calls");
    int slot = -1;
    for (int i = 0; i < kGemvBatchMax; ++i) if (!m->session.used[i]) { slot = i; break; }
    AHA_REQUIRE(slot >= 0, "batch_add: all 8 slots are decoding (step until one finishes)");
    const size_t sample_len = std::max<size_t>(r.params.max_tokens, 1);
    const size_t need = (r.seq_len + sample_len + kPage - 1) / kPage;
    AHA_REQUIRE(need <= T.free_pages.size(), "batch_add: the request needs " + std::to_string(need * kPage) + " tokens of KV capacity, " +
                                                  std::to_string(T.free_pages.size() * kPage) + " are free (max_ctx " + std::to_string(T.max_ctx) + ")");
    using clk = std::chrono::steady_clock;
    const auto t0 = clk::now();
    m->session.used[slot] = true;
    B.swap_table(slot);
    struct Guard {   // a failed prefill leaves the session as it was: own table back in place, the slot's pages back in the pool
        aha_model* m; int slot; bool ok = false;
        ~Guard() { if (ok) return; m->batch.swap_table(slot); session_release(m, slot); m->have_rope_delta = false; m->rope_delta = 0; m->text.clear_sampler(); }
    } guard{m, slot};
    m->have_rope_delta = false; m->rope_delta = 0;
    T.set_sampler(sampling_mode(r.params), r.params.temperature, r.params.top_p, r.params.top_k, r.params.repeat_penalty, r.params.repeat_last_n, r.params.seed);
    T.set_state(0, 0, 0, 0, 0);
    uint32_t tok = 0;
    forward_any(m, r.ids, r.seq_len, 0, r.mm, true, nullptr, &tok, false, true);
    T.check_sample_error();
    T.ensure_tokens((int)(r.seq_len + sample_len));       // every page the request can touch is mapped now (the step kernels only read the table)
    DecodeState cur;
    AHA_CUDA_CHECK(cudaMemcpy(&cur, T.d_state, sizeof(cur), cudaMemcpyDeviceToHost));
    B.adopt(slot, tok, (int)r.seq_len, m->kind == aha_model::QWEN3VL ? m->rope_delta : 0, cur.n_draws);
    B.swap_table(slot);
    guard.ok = true;
    T.clear_sampler();
    B.table_for.clear();
    B.clear_graphs();
    m->session.budget[slot] = sample_len;
    m->session.produced[slot] = 1;
    const bool stop = sample_len == 1 || ((r.params.flags & AHA_GEN_EOS_ON_FIRST) != 0 && is_stop_token(m, tok));
    if (usage) {
        *usage = aha_usage{};
        usage->prompt_tokens = (uint32_t)r.seq_len; usage->completion_tokens = 1;
        usage->prompt_secs = std::chrono::duration<double>(clk::now() - t0).count();
        usage->vision_secs = m->last_vision_secs;
    }
    if (stop) session_release(m, slot);
    *slot_out = slot; *first_token = tok; *finished = stop ? 1 : 0;
}
size_t session_step(aha_model* m, uint32_t* tokens_out, int32_t* status_out) {
    AHA_REQUIRE(m->session.open, "no batch session is open (aha_b200_batch_open)");
    std::vector<int> act;
    for (int i = 0; i < kGemvBatchMax; ++i) { status_out[i] = 0; tokens_out[i] = 0; if (m->session.used[i]) act.push_back(i); }
    if (act.empty()) return 0;
    // AHA_BATCH_GRAPH=0: eager launches (A/B twin of the per-composition graphs)
    m->batch.step(act, env_int("AHA_BATCH_GEMV", kBatchGemvDefault), env_flag("AHA_BATCH_GRAPH", true));
    uint32_t h_tok[kGemvBatchMax];
    AHA_CUDA_CHECK(cudaMemcpyAsync(h_tok, m->batch.d_tok, sizeof(h_tok), cudaMemcpyDeviceToHost, m->ctx.stream));
    AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
    // a request whose sampler failed (all-zero weights) poisons only the check below; the session is closed by the caller's error path
    for (int slot : act) {
        const uint32_t t = h_tok[slot];
        tokens_out[slot] = t;
        m->session.produced[slot] += 1;
        // an EOS token is delivered, then the request ends (generate.rs:139-141)
        const bool stop = m->session.produced[slot] >= m->session.budget[slot] || is_stop_token(m, t);
        status_out[slot] = stop ? 2 : 1;
    }
    for (int slot : act) if (status_out[slot] == 2) session_release(m, slot);
    m->text.check_sample_flag();   // sampler errors surface after the bookkeeping so that the slots stay consistent
    return act.size();
}

// Static batching: a batch session whose n requests are all added before the first step, then stepped until every one has finished.
// Every request follows generate_generic's rules on its own (first token never EOS-checked, an EOS token is pushed and ends THAT request,
// its own sampler / seed / repeat-penalty history) and so yields exactly the tokens aha_b200_generate would yield for it alone.
void generate_batch_impl(aha_model* m, const aha_batch_request* reqs, size_t n, uint32_t* out_tokens, size_t cap, size_t* n_out, aha_usage* usage) {
    TextModel& T = m->text;
    require_no_session(m);
    AHA_REQUIRE(n >= 1 && n <= (size_t)kGemvBatchMax, "generate_batch: 1 to 8 requests");
    AHA_REQUIRE(T.tp_world == 1, "generate_batch is single-GPU (run one batch per tensor-parallel group member instead)");
    AHA_REQUIRE(T.max_prefill >= kGemvBatchMax, "generate_batch needs max_prefill >= 8");
    size_t pages = 0;
    for (size_t i = 0; i < n; ++i) {
        AHA_REQUIRE(reqs[i].ids && reqs[i].seq_len >= 1, "generate_batch: every request needs input_ids");
        const size_t sample_len = std::max<size_t>(reqs[i].params.max_tokens, 1);
        AHA_REQUIRE(cap >= sample_len, "out_tokens capacity (per request) is smaller than max_tokens");
        AHA_REQUIRE((reqs[i].params.flags & (AHA_GEN_CONTINUE_RNG | AHA_GEN_REUSE_PREFIX)) == 0, "generate_batch: CONTINUE_RNG / REUSE_PREFIX are per-handle states of the single-request calls");
        pages += (reqs[i].seq_len + sample_len + kPage - 1) / kPage;
        n_out[i] = 0;
        if (usage) usage[i] = aha_usage{};
    }
    // the whole batch is refused before any prefill runs, rather than by the session_add that would not fit
    AHA_REQUIRE(pages <= (size_t)T.num_pages, "the requests of the batch need " + std::to_string(pages * kPage) + " tokens of KV capacity, max_ctx is " + std::to_string(T.max_ctx));
    session_open(m);
    struct Close {   // whatever happens, the handle is left as after clear_cache(), with its own page table in place
        aha_model* m;
        ~Close() { session_close(m); }
    } close{m};
    int req_of[kGemvBatchMax];   // request held by each slot: a request finished by its prefill hands its slot to the next one
    for (size_t i = 0; i < n; ++i) {
        int slot = -1, fin = 0;
        session_add(m, reqs[i], &slot, out_tokens + i * cap, &fin, usage ? usage + i : nullptr);
        req_of[slot] = (int)i;
        n_out[i] = 1;
    }
    using clk = std::chrono::steady_clock;
    const auto t_dec = clk::now();
    uint32_t tok[kGemvBatchMax];
    int32_t status[kGemvBatchMax];
    while (session_step(m, tok, status) > 0) {
        for (int slot = 0; slot < kGemvBatchMax; ++slot) {
            if (status[slot] == 0) continue;
            const size_t i = (size_t)req_of[slot];
            out_tokens[i * cap + n_out[i]++] = tok[slot];
            if (status[slot] == 2 && usage) usage[i].completion_secs = std::chrono::duration<double>(clk::now() - t_dec).count();
        }
    }
    if (usage) for (size_t i = 0; i < n; ++i) usage[i].completion_tokens = (uint32_t)n_out[i];
}
}  // namespace

int aha_b200_clear_cache(aha_model* m) {
    return guarded(m, [&] {
        AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        if (m->session.open) session_close(m);   // clear_cache ends a batch session too: every sequence's K/V is gone
        else drop_cache(m);
    });
}

int aha_b200_batch_open(aha_model* m) { return guarded(m, [&] { session_open(m); }); }

int aha_b200_batch_add(aha_model* m, const aha_batch_request* req, int32_t* slot_out, uint32_t* first_token_out, int32_t* finished_out, aha_usage* usage) {
    return guarded(m, [&] {
        AHA_REQUIRE(req && slot_out && first_token_out && finished_out, "req, slot_out, first_token_out and finished_out are required");
        int slot = -1, fin = 0;
        session_add(m, *req, &slot, first_token_out, &fin, usage);
        *slot_out = slot; *finished_out = fin;
    });
}

int aha_b200_batch_step(aha_model* m, uint32_t* tokens_out, int32_t* status_out, size_t* n_stepped_out) {
    return guarded(m, [&] {
        AHA_REQUIRE(tokens_out && status_out, "tokens_out[8] and status_out[8] are required");
        const size_t n = session_step(m, tokens_out, status_out);
        if (n_stepped_out) *n_stepped_out = n;
    });
}

int aha_b200_batch_close(aha_model* m) {
    return guarded(m, [&] { AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream)); session_close(m); });
}

int aha_b200_generate_batch(aha_model* m, const aha_batch_request* reqs, size_t n, uint32_t* out_tokens, size_t cap, size_t* n_out, aha_usage* usage) {
    return guarded(m, [&] {
        AHA_REQUIRE(reqs && out_tokens && n_out, "reqs, out_tokens and n_out are required");
        generate_batch_impl(m, reqs, n, out_tokens, cap, n_out, usage);
    });
}

int aha_b200_generate(aha_model* m, const uint32_t* ids, size_t seq_len, const aha_mm* mm, const aha_gen_params* params, uint32_t* out_tokens,
                      size_t cap, size_t* n_out, aha_usage* usage) {
    return guarded(m, [&] {
        AHA_REQUIRE(params && out_tokens && n_out, "params, out_tokens and n_out are required");
        AHA_REQUIRE(cap >= std::max<size_t>(params->max_tokens, 1), "out_tokens capacity is smaller than max_tokens");
        if (usage) *usage = aha_usage{};
        size_t n = 0;
        GenSink sink{[&](uint32_t t, size_t i) { out_tokens[i] = t; n = i + 1; return false; }};
        generate_impl(m, ids, seq_len, mm, *params, sink, false, usage, nullptr);
        *n_out = n;
    });
}

int aha_b200_generate_stream(aha_model* m, const uint32_t* ids, size_t seq_len, const aha_mm* mm, const aha_gen_params* params,
                             aha_token_callback on_token, void* user, aha_usage* usage) {
    return guarded(m, [&] {
        AHA_REQUIRE(params && on_token, "params and on_token are required");
        if (usage) *usage = aha_usage{};
        GenSink sink{[&](uint32_t t, size_t i) { return on_token(user, t, (uint32_t)i) != 0; }};
        generate_impl(m, ids, seq_len, mm, *params, sink, true, usage, nullptr);
    });
}

int aha_b200_asr_generate(aha_model* m, const aha_asr_chunk* chunks, size_t n_chunks, const aha_gen_params* params, uint32_t* out_tokens, size_t cap,
                          size_t* n_out, aha_token_callback on_token, void* user, aha_usage* usage) {
    return guarded(m, [&] {
        AHA_REQUIRE(m->kind == aha_model::QWEN3_ASR, "asr_generate needs a qwen3_asr handle");
        AHA_REQUIRE(chunks && n_chunks >= 1 && params && out_tokens && n_out, "chunks, params, out_tokens and n_out are required");
        if (usage) *usage = aha_usage{};
        // Qwen3AsrGenerateModel::generate (qwen3_asr/generate.rs:130-186): ONE LogitsProcessor for the whole request (its RNG
        // stream runs on across the chunks), no repeat penalty, every token -- the first included -- is EOS-checked, the KV
        // cache is cleared after every chunk, the token lists of the chunks are concatenated.
        size_t total = 0;
        for (size_t c = 0; c < n_chunks; ++c) {
            aha_gen_params p = *params;
            p.repeat_penalty = 1.0f;
            p.top_k = 0;                                  // get_logit_processor(Some(temperature), top_p, None, seed)
            p.flags |= AHA_GEN_EOS_ON_FIRST;
            if (c > 0) p.flags |= AHA_GEN_CONTINUE_RNG;
            AHA_REQUIRE(total + std::max<size_t>(p.max_tokens, 1) <= cap, "out_tokens capacity is smaller than n_chunks * max_tokens");
            aha_mm mm{&chunks[c].input_features, 1};
            const size_t base = total;
            bool abort = false;
            GenSink sink{[&](uint32_t t, size_t i) {
                out_tokens[base + i] = t; total = base + i + 1;
                if (on_token && on_token(user, t, (uint32_t)(base + i)) != 0) abort = true;
                return abort;
            }};
            generate_impl(m, chunks[c].ids, chunks[c].seq_len, &mm, p, sink, on_token != nullptr, usage, nullptr);
            if (abort) break;
        }
        *n_out = total;
    });
}

int aha_b200_debug_sample(aha_model* m, const float* logits, const aha_gen_params* params, const uint32_t* context, size_t n_context,
                          uint32_t draw_index, uint32_t* token_out) {
    return guarded(m, [&] {
        AHA_REQUIRE(logits && params && token_out && (context || n_context == 0), "logits, params and token_out are required");
        TextModel& T = m->text;
        AHA_REQUIRE(n_context <= (size_t)T.hist_cap, "context longer than the history buffer");
        const int mode = sampling_mode(*params);
        T.set_sampler(mode, params->temperature, params->top_p, params->top_k, params->repeat_penalty, params->repeat_last_n, params->seed);
        AHA_REQUIRE(T.samp_active, "plain ArgMax needs no sampler (temperature < 1e-7 and no repeat penalty)");
        AHA_CUDA_CHECK(cudaMemcpyAsync(T.logits, logits, (size_t)T.cfg.V * sizeof(float), cudaMemcpyHostToDevice, m->ctx.stream));
        if (n_context) AHA_CUDA_CHECK(cudaMemcpyAsync(T.d_history, context, n_context * sizeof(uint32_t), cudaMemcpyHostToDevice, m->ctx.stream));
        T.set_state(0, 0, 0, (int)n_context, draw_index);
        T.sample(0);
        AHA_CUDA_CHECK(cudaMemcpyAsync(m->h_pin, T.d_argmax, sizeof(uint32_t), cudaMemcpyDeviceToHost, m->ctx.stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        T.check_sample_error();
        T.clear_sampler();
        *token_out = m->h_pin[0];
    });
}

int aha_b200_decode_steps(aha_model* m, uint32_t first_token, size_t seqlen_offset, size_t n_steps, uint32_t* out_tokens, double* device_ms) {
    return guarded(m, [&] {
        TextModel& T = m->text;
        AHA_REQUIRE(first_token < (uint32_t)T.cfg.V, "token id out of range");
        AHA_REQUIRE(seqlen_offset + n_steps <= (size_t)T.max_ctx, "context exceeds max_ctx");
        require_no_session(m);
        m->cached_ids.clear();
        T.ensure_tokens((int)(seqlen_offset + n_steps));
        T.set_state(first_token, (int)seqlen_offset, m->kind == aha_model::QWEN3VL ? m->rope_delta : 0, 0);
        if (n_steps > 0 && !T.step_graph && T.use_graph) {  // build the graph outside the timed region (pos is restored below)
            T.decode_step();
            T.set_state(first_token, (int)seqlen_offset, m->kind == aha_model::QWEN3VL ? m->rope_delta : 0, 0);
        }
        AHA_CUDA_CHECK(cudaEventRecord(m->ev0, m->ctx.stream));
        for (size_t i = 0; i < n_steps; ++i) T.decode_step();
        AHA_CUDA_CHECK(cudaEventRecord(m->ev1, m->ctx.stream));
        if (out_tokens) AHA_CUDA_CHECK(cudaMemcpyAsync(out_tokens, T.d_history, n_steps * sizeof(uint32_t), cudaMemcpyDeviceToHost, m->ctx.stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        T.check_ll_abort();
        if (device_ms) { float ms = 0.f; AHA_CUDA_CHECK(cudaEventElapsedTime(&ms, m->ev0, m->ev1)); *device_ms = ms; }
    });
}

int aha_b200_bench_kernel(aha_model* m, const char* which, int iters, double* avg_ms, uint64_t* bytes_per_launch) {
    return guarded(m, [&] {
        AHA_REQUIRE(which && iters > 0 && avg_ms && bytes_per_launch, "which, iters, avg_ms, bytes_per_launch are required");
        TextModel& T = m->text;
        const std::string w = which;
        cudaStream_t st = m->ctx.stream;
        const int L = T.cfg.L;
        uint64_t bytes = 0;
        auto launch = [&](int i) {
            TextLayer& Y = T.layers[i % L];
            GemvArgs a{};
            if (w == "gemv_gate_up") { a.W = Y.gu.w; a.x = T.x1; a.norm_w = Y.ln2; a.eps = T.cfg.eps; a.out = T.h1; a.N = Y.gu.N; a.K = Y.gu.K; gemv(st, PRO_RMSNORM, GEPI_SWIGLU, a); bytes = 2ull * a.N * a.K; }
            else if (w == "gemv_qkv") { a.W = Y.qkv.w; a.x = T.x1; a.norm_w = Y.ln1; a.eps = T.cfg.eps; a.out = T.qkv1; a.N = Y.qkv.N; a.K = Y.qkv.K; gemv(st, PRO_RMSNORM, GEPI_STORE, a); bytes = 2ull * a.N * a.K; }
            else if (w == "gemv_down") { a.W = Y.down.w; a.x = T.h1; a.resid = T.x1; a.out = T.x1; a.N = Y.down.N; a.K = Y.down.K; gemv(st, PRO_NONE, GEPI_RESID, a); bytes = 2ull * a.N * a.K; }
            else if (w == "gemv_o") { a.W = Y.o.w; a.x = T.attn1; a.resid = T.x1; a.out = T.x1; a.N = Y.o.N; a.K = Y.o.K; gemv(st, PRO_NONE, GEPI_RESID, a); bytes = 2ull * a.N * a.K; }
            else if (w == "gemv_lm_head") { T.head(T.x1); bytes = 2ull * T.cfg.V * T.cfg.H; }
            else throw std::runtime_error("unknown kernel '" + w + "'");
            m->ctx.cnt.kernels++;
        };
        for (int i = 0; i < 3; ++i) launch(i);
        AHA_CUDA_CHECK(cudaEventRecord(m->ev0, st));
        for (int i = 0; i < iters; ++i) launch(i + 3);
        AHA_CUDA_CHECK(cudaEventRecord(m->ev1, st));
        AHA_CUDA_CHECK(cudaStreamSynchronize(st));
        float ms = 0.f;
        AHA_CUDA_CHECK(cudaEventElapsedTime(&ms, m->ev0, m->ev1));
        *avg_ms = ms / iters;
        *bytes_per_launch = bytes;
    });
}

int aha_b200_mel_spectrogram(aha_model* m, const float* wave, size_t n_samples, float* mel_out, size_t mel_cap, size_t* n_frames) {
    return guarded(m, [&] {
        AHA_REQUIRE(m->kind == aha_model::QWEN3_ASR, "mel_spectrogram needs a qwen3_asr handle");
        AHA_REQUIRE(wave && mel_out && n_frames, "wave, mel_out and n_frames are required");
        const int frames = m->audio.mel_from_host(wave, n_samples);
        AHA_REQUIRE((size_t)frames * m->audio.cfg.mel <= mel_cap, "mel_out too small");
        AHA_CUDA_CHECK(cudaMemcpyAsync(mel_out, m->audio.d_mel, (size_t)frames * m->audio.cfg.mel * sizeof(float), cudaMemcpyDeviceToHost, m->ctx.stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        *n_frames = (size_t)frames;
    });
}

// u8 HWC -> normalised, frame-duplicated, merge-block-ordered patches.
__global__ void patchify_kernel(const uint8_t* __restrict__ img, int H, int W, int patch, int merge, int tpatch, float* __restrict__ out) {
    const int gw = W / patch, gh = H / patch;
    const int p = blockIdx.x;  // patch in merge-block order (single temporal group)
    const int mw = gw / merge;
    const int blk = p / (merge * merge), in = p % (merge * merge);
    const int row = (blk / mw) * merge + in / merge, col = (blk % mw) * merge + in % merge;
    (void)gh;
    const int feat = 3 * tpatch * patch * patch;
    for (int f = threadIdx.x; f < feat; f += blockDim.x) {
        const int c = f / (tpatch * patch * patch), rem = f % (patch * patch), py = rem / patch, px = rem % patch;
        const uint8_t v = img[((size_t)(row * patch + py) * W + (col * patch + px)) * 3 + c];
        // img_transform: f32(v) * (1/255), (x - 0.5) / 0.5   (img_utils.rs:272-294 with mean = std = 0.5).  Each step rounded on its own
        // (candle runs affine, broadcast_sub and broadcast_div as three kernels; a contracted v * (1/255) - 0.5 differs in the last bit)
        const float x = __fmul_rn((float)v, 1.0f / 255.0f);
        out[(size_t)p * feat + f] = __fdiv_rn(__fsub_rn(x, 0.5f), 0.5f);
    }
}

// process_videos for one video (qwen3vl/processor.rs:253-280 + process_vision_tensor :174-227): T frames u8 (T, H, W, 3) -> rescale, normalise,
// pad the frame count to a multiple of temporal_patch_size by repeating the last frame, merge-block patch order with features (c, frame in group, py, px)
__global__ void video_patchify_kernel(const uint8_t* __restrict__ frames, int T, int H, int W, int patch, int merge, int tpatch, float* __restrict__ out) {
    const int gw = W / patch, gh = H / patch;
    const int per = gh * gw;
    const int gt = blockIdx.x / per, p = blockIdx.x % per;   // temporal group, patch in merge-block order inside it
    const int mw = gw / merge;
    const int blk = p / (merge * merge), in = p % (merge * merge);
    const int row = (blk / mw) * merge + in / merge, col = (blk % mw) * merge + in % merge;
    const int pp = patch * patch, feat = 3 * tpatch * pp;
    for (int f = threadIdx.x; f < feat; f += blockDim.x) {
        const int c = f / (tpatch * pp), tt = (f / pp) % tpatch, rem = f % pp, py = rem / patch, px = rem % patch;
        const int frame = min(gt * tpatch + tt, T - 1);
        const uint8_t v = frames[(((size_t)frame * H + (row * patch + py)) * W + (col * patch + px)) * 3 + c];
        const float x = __fmul_rn((float)v, 1.0f / 255.0f);   // affine, broadcast_sub, broadcast_div: three separately rounded steps
        out[(size_t)blockIdx.x * feat + f] = __fdiv_rn(__fsub_rn(x, 0.5f), 0.5f);
    }
}

int aha_b200_video_preprocess(aha_model* m, const uint8_t* frames_thwc, size_t n_frames, size_t h, size_t w, float* pixel_values_out, size_t cap,
                              uint32_t grid_thw_out[3]) {
    return guarded(m, [&] {
        AHA_REQUIRE(m->kind == aha_model::QWEN3VL, "video_preprocess needs a qwen3vl handle");
        AHA_REQUIRE(frames_thwc && pixel_values_out && grid_thw_out && n_frames > 0 && h > 0 && w > 0, "frames, outputs and positive sizes are required");
        VisionModel& V = m->vision;
        const int ps = V.cfg.patch, mg = V.cfg.merge, tp = V.cfg.tpatch;
        AHA_REQUIRE(h % (ps * mg) == 0 && w % (ps * mg) == 0, "frame size must already be a multiple of patch_size*merge_size (video_smart_resize output)");
        const int gt = ((int)n_frames + tp - 1) / tp, gh = (int)h / ps, gw = (int)w / ps;
        const size_t N = (size_t)gt * gh * gw;
        AHA_REQUIRE(N <= (size_t)V.max_patches, "video needs " + std::to_string(N) + " patches, max_patches is " + std::to_string(V.max_patches));
        AHA_REQUIRE(N * V.patch_dim <= cap, "pixel_values_out too small");
        uint8_t* d_in = nullptr;
        const size_t bytes = n_frames * h * w * 3;
        AHA_CUDA_CHECK(cudaMalloc(&d_in, bytes));
        try {
            AHA_CUDA_CHECK(cudaMemcpyAsync(d_in, frames_thwc, bytes, cudaMemcpyHostToDevice, m->ctx.stream));
            video_patchify_kernel<<<(unsigned)N, 256, 0, m->ctx.stream>>>(d_in, (int)n_frames, (int)h, (int)w, ps, mg, tp, V.pix);
            m->ctx.cnt.kernels++;
            AHA_CUDA_CHECK(cudaMemcpyAsync(pixel_values_out, V.pix, N * V.patch_dim * sizeof(float), cudaMemcpyDeviceToHost, m->ctx.stream));
            AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        } catch (...) { cudaFree(d_in); throw; }
        cudaFree(d_in);
        grid_thw_out[0] = (uint32_t)gt; grid_thw_out[1] = (uint32_t)gh; grid_thw_out[2] = (uint32_t)gw;
    });
}

int aha_b200_image_patchify(aha_model* m, const uint8_t* img_hwc, size_t h, size_t w, float* pixel_values_out, size_t cap, uint32_t grid_thw_out[3]) {
    return guarded(m, [&] {
        AHA_REQUIRE(m->kind == aha_model::QWEN3VL, "image_patchify needs a qwen3vl handle");
        VisionModel& V = m->vision;
        const int ps = V.cfg.patch, mg = V.cfg.merge;
        AHA_REQUIRE(h % (ps * mg) == 0 && w % (ps * mg) == 0, "image size must already be a multiple of patch_size*merge_size (img_smart_resize output)");
        const int gh = (int)h / ps, gw = (int)w / ps, N = gh * gw;
        AHA_REQUIRE(N <= V.max_patches, "image exceeds max_patches");
        AHA_REQUIRE((size_t)N * V.patch_dim <= cap, "pixel_values_out too small");
        uint8_t* d_img = nullptr;
        AHA_CUDA_CHECK(cudaMalloc(&d_img, h * w * 3));
        try {
            AHA_CUDA_CHECK(cudaMemcpyAsync(d_img, img_hwc, h * w * 3, cudaMemcpyHostToDevice, m->ctx.stream));
            patchify_kernel<<<N, 256, 0, m->ctx.stream>>>(d_img, (int)h, (int)w, ps, mg, V.cfg.tpatch, V.pix);
            m->ctx.cnt.kernels++;
            AHA_CUDA_CHECK(cudaMemcpyAsync(pixel_values_out, V.pix, (size_t)N * V.patch_dim * sizeof(float), cudaMemcpyDeviceToHost, m->ctx.stream));
            AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        } catch (...) { cudaFree(d_img); throw; }
        cudaFree(d_img);
        grid_thw_out[0] = 1; grid_thw_out[1] = (uint32_t)gh; grid_thw_out[2] = (uint32_t)gw;
    });
}

extern "C++" {
namespace {
template <typename F>
int guarded_host(F&& f) {   // host-only entries (no handle): errors land in the create-error slot read by aha_b200_last_error(NULL)
    try { f(); return 0; }
    catch (const std::exception& e) { std::lock_guard<std::mutex> lk(g_err_mu); g_create_error = e.what(); return 1; }
}
// resize (h, w, 3) u8 on the device -> (nh, nw, 3) u8 on the device; both buffers owned by the caller
void resize_on_device(aha_model* m, const uint8_t* d_in, int h, int w, uint8_t* d_out, int nh, int nw, float* d_tmp) {
    if (nh == h && nw == w) {   // imageops::resize copies when the dimensions already match
        AHA_CUDA_CHECK(cudaMemcpyAsync(d_out, d_in, (size_t)h * w * 3, cudaMemcpyDeviceToDevice, m->ctx.stream));
        return;
    }
    AHA_REQUIRE(2.0f * std::max(1.0f, (float)h / nh) + 2 <= kResizeMaxTaps && 2.0f * std::max(1.0f, (float)w / nw) + 2 <= kResizeMaxTaps,
                "image downscale factor beyond the resize kernel's tap window (15x)");
    resize_vertical_kernel<<<nh, 256, 0, m->ctx.stream>>>(d_in, h, w, nh, d_tmp);
    resize_horizontal_kernel<<<nw, 256, 0, m->ctx.stream>>>(d_tmp, nh, w, nw, d_out);
    AHA_CUDA_CHECK(cudaGetLastError());
    m->ctx.cnt.kernels += 2;
}
}  // namespace
}  // extern "C++"

int aha_b200_img_smart_resize(uint32_t img_h, uint32_t img_w, uint32_t factor, uint32_t min_pixels, uint32_t max_pixels, uint32_t* out_h, uint32_t* out_w) {
    return guarded_host([&] {
        AHA_REQUIRE(out_h && out_w, "out_h and out_w are required");
        img_smart_resize(img_h, img_w, factor, min_pixels, max_pixels, *out_h, *out_w);
    });
}

int aha_b200_image_resize(aha_model* m, const uint8_t* img_hwc, size_t h, size_t w, size_t new_h, size_t new_w, uint8_t* out_hwc) {
    return guarded(m, [&] {
        AHA_REQUIRE(img_hwc && out_hwc && h > 0 && w > 0 && new_h > 0 && new_w > 0, "images and positive sizes are required");
        uint8_t *d_in = nullptr, *d_out = nullptr;
        float* d_tmp = nullptr;
        auto cleanup = [&] { cudaFree(d_in); cudaFree(d_out); cudaFree(d_tmp); };
        try {
            AHA_CUDA_CHECK(cudaMalloc(&d_in, h * w * 3)); AHA_CUDA_CHECK(cudaMalloc(&d_out, new_h * new_w * 3)); AHA_CUDA_CHECK(cudaMalloc(&d_tmp, new_h * w * 3 * sizeof(float)));
            AHA_CUDA_CHECK(cudaMemcpyAsync(d_in, img_hwc, h * w * 3, cudaMemcpyHostToDevice, m->ctx.stream));
            resize_on_device(m, d_in, (int)h, (int)w, d_out, (int)new_h, (int)new_w, d_tmp);
            AHA_CUDA_CHECK(cudaMemcpyAsync(out_hwc, d_out, new_h * new_w * 3, cudaMemcpyDeviceToHost, m->ctx.stream));
            AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        } catch (...) { cleanup(); throw; }
        cleanup();
    });
}

int aha_b200_image_preprocess(aha_model* m, const uint8_t* img_hwc, size_t h, size_t w, uint32_t min_pixels, uint32_t max_pixels, float* pixel_values_out,
                              size_t cap, uint32_t grid_thw_out[3]) {
    return guarded(m, [&] {
        AHA_REQUIRE(m->kind == aha_model::QWEN3VL, "image_preprocess needs a qwen3vl handle");
        AHA_REQUIRE(img_hwc && pixel_values_out && grid_thw_out && h > 0 && w > 0, "image, outputs and positive sizes are required");
        VisionModel& V = m->vision;
        const int ps = V.cfg.patch, mg = V.cfg.merge;
        uint32_t rh = 0, rw = 0;
        img_smart_resize((uint32_t)h, (uint32_t)w, (uint32_t)(ps * mg), min_pixels, max_pixels, rh, rw);   // Qwen3VLProcessor::process_img
        const int gh = (int)rh / ps, gw = (int)rw / ps, N = gh * gw;
        AHA_REQUIRE(N <= V.max_patches, "image needs " + std::to_string(N) + " patches after img_smart_resize, max_patches is " + std::to_string(V.max_patches));
        AHA_REQUIRE((size_t)N * V.patch_dim <= cap, "pixel_values_out too small");
        uint8_t *d_in = nullptr, *d_rs = nullptr;
        float* d_tmp = nullptr;
        auto cleanup = [&] { cudaFree(d_in); cudaFree(d_rs); cudaFree(d_tmp); };
        try {
            AHA_CUDA_CHECK(cudaMalloc(&d_in, h * w * 3)); AHA_CUDA_CHECK(cudaMalloc(&d_rs, (size_t)rh * rw * 3)); AHA_CUDA_CHECK(cudaMalloc(&d_tmp, (size_t)rh * w * 3 * sizeof(float)));
            AHA_CUDA_CHECK(cudaMemcpyAsync(d_in, img_hwc, h * w * 3, cudaMemcpyHostToDevice, m->ctx.stream));
            resize_on_device(m, d_in, (int)h, (int)w, d_rs, (int)rh, (int)rw, d_tmp);
            patchify_kernel<<<N, 256, 0, m->ctx.stream>>>(d_rs, (int)rh, (int)rw, ps, mg, V.cfg.tpatch, V.pix);   // img_transform + frame duplication + 9-D permute
            m->ctx.cnt.kernels++;
            AHA_CUDA_CHECK(cudaMemcpyAsync(pixel_values_out, V.pix, (size_t)N * V.patch_dim * sizeof(float), cudaMemcpyDeviceToHost, m->ctx.stream));
            AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        } catch (...) { cleanup(); throw; }
        cleanup();
        grid_thw_out[0] = 1; grid_thw_out[1] = (uint32_t)gh; grid_thw_out[2] = (uint32_t)gw;
    });
}

int aha_b200_expand_placeholders(const uint32_t* ids, size_t n, uint32_t token_id, const uint32_t* counts, size_t n_counts, uint32_t* out, size_t cap,
                                 size_t* n_out) {
    return guarded_host([&] {
        AHA_REQUIRE(ids && n_out && (counts || n_counts == 0), "ids and n_out are required");
        const std::vector<uint32_t> r = expand_placeholders(ids, n, token_id, counts, n_counts);
        *n_out = r.size();
        if (out) { AHA_REQUIRE(r.size() <= cap, "out too small"); std::memcpy(out, r.data(), r.size() * sizeof(uint32_t)); }
    });
}

int aha_b200_video_smart_resize(uint32_t num_frames, uint32_t height, uint32_t width, uint32_t temporal_factor, uint32_t factor, uint32_t min_pixels,
                                uint32_t max_pixels, uint32_t video_ratio, uint32_t* out_h, uint32_t* out_w) {
    return guarded_host([&] {
        AHA_REQUIRE(out_h && out_w, "out_h and out_w are required");
        video_smart_resize(num_frames, height, width, temporal_factor, factor, min_pixels, max_pixels, video_ratio, *out_h, *out_w);
    });
}

int aha_b200_video_sample_frames(uint32_t total_frames, uint32_t rate_num, uint32_t rate_den, uint32_t fps, uint32_t min_frames, uint32_t max_frames,
                                 uint32_t* nframes_out, uint32_t* indices_out, size_t cap, size_t* n_out) {
    return guarded_host([&] {
        AHA_REQUIRE(n_out, "n_out is required");
        uint32_t nframes = 0;
        const std::vector<uint32_t> idx = video_sample_frames(total_frames, rate_num, rate_den, fps, min_frames, max_frames, nframes);
        if (nframes_out) *nframes_out = nframes;
        *n_out = idx.size();
        if (indices_out) { AHA_REQUIRE(idx.size() <= cap, "indices_out too small"); std::memcpy(indices_out, idx.data(), idx.size() * sizeof(uint32_t)); }
    });
}

int aha_b200_video_timestamps(const uint32_t* frame_indices, size_t n, float fps, uint32_t t_merge_size, float* stamps_out, size_t cap, size_t* n_out) {
    return guarded_host([&] {
        AHA_REQUIRE(frame_indices && n_out, "frame_indices and n_out are required");
        const std::vector<float> st = video_timestamps(frame_indices, n, fps, t_merge_size);
        *n_out = st.size();
        if (stamps_out) { AHA_REQUIRE(st.size() <= cap, "stamps_out too small"); std::memcpy(stamps_out, st.data(), st.size() * sizeof(float)); }
    });
}

int aha_b200_format_timestamp(float seconds, char* out, size_t cap) {
    return guarded_host([&] {
        AHA_REQUIRE(out && cap > 0, "out is required");
        // format!("<{:.1} seconds>", t): both Rust and printf print the exactly rounded decimal (ties to even) of the f32 value
        const int n = std::snprintf(out, cap, "<%.1f seconds>", (double)seconds);
        AHA_REQUIRE(n > 0 && (size_t)n < cap, "out too small");
    });
}

int aha_b200_expand_video_placeholders(const uint32_t* ids, size_t n, uint32_t video_token_id, uint32_t vision_start_token_id, uint32_t vision_end_token_id,
                                       const uint32_t* video_grid_thw, size_t n_videos, uint32_t merge_size, const uint32_t* stamp_ids,
                                       const uint32_t* stamp_lens, size_t n_stamps, uint32_t* out, size_t cap, size_t* n_out) {
    return guarded_host([&] {
        AHA_REQUIRE(ids && n_out && (video_grid_thw || n_videos == 0) && (stamp_lens || n_stamps == 0), "ids, video_grid_thw, stamp_lens and n_out are required");
        const std::vector<uint32_t> r = expand_video_placeholders(ids, n, video_token_id, vision_start_token_id, vision_end_token_id, video_grid_thw, n_videos, merge_size,
                                                                  stamp_ids, stamp_lens, n_stamps);
        *n_out = r.size();
        if (out) { AHA_REQUIRE(r.size() <= cap, "out too small"); std::memcpy(out, r.data(), r.size() * sizeof(uint32_t)); }
    });
}

size_t aha_b200_feat_extract_output_length(size_t n_frames) { return feat_extract_output_length(n_frames); }

int aha_b200_float_range_normalize(float* wave, size_t n) {
    return guarded_host([&] { AHA_REQUIRE(wave || n == 0, "wave is required"); float_range_normalize(wave, n); });
}

int aha_b200_resample(aha_model* m, const float* wave, size_t n, int64_t orig_freq, int64_t new_freq, float* out, size_t cap, size_t* n_out) {
    return guarded(m, [&] {
        AHA_REQUIRE(n_out, "n_out is required");
        AHA_REQUIRE(wave || n == 0, "wave is required");
        if (orig_freq == new_freq) {   // resample(): the waveform itself
            AHA_REQUIRE(orig_freq > 0, "Frequencies must be positive");
            *n_out = n;
            if (!out) return;
            AHA_REQUIRE(cap >= n, "output buffer too small");
            std::memcpy(out, wave, n * sizeof(float));
            return;
        }
        const SincBank B = sinc_resample_bank(orig_freq, new_freq);
        const size_t len_out = sinc_resample_out_len(B, n);
        *n_out = len_out;
        if (!out) return;
        AHA_REQUIRE(cap >= len_out, "output buffer too small");
        if (len_out == 0) return;
        float *d_w = nullptr, *d_t = nullptr, *d_o = nullptr;
        auto cleanup = [&] { cudaFree(d_w); cudaFree(d_t); cudaFree(d_o); };
        try {
            cudaStream_t st = m->ctx.stream;
            AHA_CUDA_CHECK(cudaMalloc(&d_w, std::max<size_t>(n, 1) * sizeof(float))); AHA_CUDA_CHECK(cudaMalloc(&d_t, B.taps.size() * sizeof(float)));
            AHA_CUDA_CHECK(cudaMalloc(&d_o, len_out * sizeof(float)));
            AHA_CUDA_CHECK(cudaMemcpyAsync(d_w, wave, n * sizeof(float), cudaMemcpyHostToDevice, st));
            const size_t smem = B.taps.size() * sizeof(float);
            const unsigned blocks = (unsigned)((len_out + 255) / 256);
            if (smem <= 96 * 1024) {   // the whole bank in shared memory
                AHA_CUDA_CHECK(cudaMemcpyAsync(d_t, B.taps.data(), smem, cudaMemcpyHostToDevice, st));
                if (smem > 48 * 1024) AHA_CUDA_CHECK(cudaFuncSetAttribute(sinc_resample_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                sinc_resample_kernel<true><<<blocks, 256, smem, st>>>(d_w, (long long)n, d_t, B.orig, B.fresh, B.width, B.K, d_o, (long long)len_out);
            } else {                   // 44.1 kHz and friends: hundreds of KB of taps, read from a transposed copy through the caches
                std::vector<float> tT(B.taps.size());
                for (int j = 0; j < B.fresh; ++j) for (int k = 0; k < B.K; ++k) tT[(size_t)k * B.fresh + j] = B.taps[(size_t)j * B.K + k];
                AHA_CUDA_CHECK(cudaMemcpyAsync(d_t, tT.data(), smem, cudaMemcpyHostToDevice, st));
                AHA_CUDA_CHECK(cudaStreamSynchronize(st));   // tT is a temporary
                sinc_resample_kernel<false><<<blocks, 256, 0, st>>>(d_w, (long long)n, d_t, B.orig, B.fresh, B.width, B.K, d_o, (long long)len_out);
            }
            AHA_CUDA_CHECK(cudaGetLastError());
            m->ctx.cnt.kernels++;
            AHA_CUDA_CHECK(cudaMemcpyAsync(out, d_o, len_out * sizeof(float), cudaMemcpyDeviceToHost, st));
            AHA_CUDA_CHECK(cudaStreamSynchronize(st));
        } catch (...) { cleanup(); throw; }
        cleanup();
    });
}

int aha_b200_sinc_resample_bank(int64_t orig_freq, int64_t new_freq, float* taps_out, size_t cap, int32_t dims_out[4]) {
    return guarded_host([&] {
        AHA_REQUIRE(dims_out, "dims_out is required");
        const SincBank B = sinc_resample_bank(orig_freq, new_freq);
        dims_out[0] = B.fresh; dims_out[1] = B.K; dims_out[2] = B.width; dims_out[3] = B.orig;
        if (!taps_out) return;
        AHA_REQUIRE(cap >= B.taps.size(), "output buffer too small");
        std::memcpy(taps_out, B.taps.data(), B.taps.size() * sizeof(float));
    });
}

int aha_b200_split_audio_into_chunks(size_t total_len, uint32_t sample_rate, float max_chunk_sec, size_t* lens_out, size_t cap, size_t* n_out) {
    return guarded_host([&] {
        AHA_REQUIRE(n_out && sample_rate > 0 && max_chunk_sec > 0.f, "n_out, a positive sample rate and chunk length are required");
        const std::vector<size_t> r = split_audio_into_chunks(total_len, sample_rate, max_chunk_sec);
        *n_out = r.size();
        if (lens_out) { AHA_REQUIRE(r.size() <= cap, "lens_out too small"); for (size_t i = 0; i < r.size(); ++i) lens_out[i] = r[i]; }
    });
}

int aha_b200_debug_gemm(aha_model* m, int impl, int epi, int act, int M, int N, int K, const float* x, const uint16_t* w, const float* bias,
                        const float* resid, float* out, int iters, double* device_ms) {
    return guarded(m, [&] {
        AHA_REQUIRE(x && w && out && M > 0 && N > 0 && K > 0, "x, w, out and positive sizes are required");
        Ctx& c = m->ctx;
        float *dx = nullptr, *db = nullptr, *dr = nullptr, *dy = nullptr;
        __half* dw = nullptr;
        const int Nout = epi == EPI_SWIGLU ? N / 2 : N;
        auto cleanup = [&] { cudaFree(dx); cudaFree(db); cudaFree(dr); cudaFree(dy); cudaFree(dw); };
        try {
            AHA_CUDA_CHECK(cudaMalloc(&dx, (size_t)M * K * 4)); AHA_CUDA_CHECK(cudaMalloc(&dw, (size_t)N * K * 2)); AHA_CUDA_CHECK(cudaMalloc(&dy, (size_t)M * Nout * 4));
            AHA_CUDA_CHECK(cudaMemcpy(dx, x, (size_t)M * K * 4, cudaMemcpyHostToDevice));
            AHA_CUDA_CHECK(cudaMemcpy(dw, w, (size_t)N * K * 2, cudaMemcpyHostToDevice));
            if (bias) { AHA_CUDA_CHECK(cudaMalloc(&db, (size_t)N * 4)); AHA_CUDA_CHECK(cudaMemcpy(db, bias, (size_t)N * 4, cudaMemcpyHostToDevice)); }
            if (epi == EPI_RESID) {
                AHA_REQUIRE(resid, "resid is required for the residual epilogue");
                AHA_CUDA_CHECK(cudaMalloc(&dr, (size_t)M * N * 4)); AHA_CUDA_CHECK(cudaMemcpy(dr, resid, (size_t)M * N * 4, cudaMemcpyHostToDevice));
            }
            LinearW W; W.w = dw; W.b = db; W.N = N; W.K = K;
            if (impl == 5 || impl == 6) {   // the batched decode GEMV (gemv_batch.cuh; 6 = the cp.async ring version): M <= 8 activation rows against every weight row
                AHA_REQUIRE(M <= kGemvBatchMax && (epi == EPI_STORE || epi == EPI_RESID || epi == EPI_SWIGLU), "batched GEMV: M <= 8, epilogue store / residual / SwiGLU");
                GemvBatchArgs a{};
                a.W = dw; a.x = dx; a.ldx = K; a.bias = db; a.resid = dr; a.ldr = N; a.out = dy; a.ldo = Nout; a.N = N; a.K = K; a.nb = M; a.eps = 0.f;
                const int gepi = epi == EPI_STORE ? GEPI_STORE : (epi == EPI_RESID ? GEPI_RESID : GEPI_SWIGLU);
                const int pro = epi == EPI_SWIGLU ? PRO_RMSNORM : PRO_NONE;   // (the SwiGLU instantiation carries the RMSNorm prologue: unit gain here)
                float* ones = nullptr;
                if (pro == PRO_RMSNORM) {
                    std::vector<float> h1((size_t)K, 1.0f);
                    AHA_CUDA_CHECK(cudaMalloc(&ones, (size_t)K * 4)); AHA_CUDA_CHECK(cudaMemcpy(ones, h1.data(), (size_t)K * 4, cudaMemcpyHostToDevice));
                    a.norm_w = ones; a.eps = 1e-6f;
                }
                try {
                    gemv_batch(c.stream, pro, gepi, a, impl == 6);
                    AHA_CUDA_CHECK(cudaEventRecord(m->ev0, c.stream));
                    for (int i = 0; i < std::max(iters, 0); ++i) gemv_batch(c.stream, pro, gepi, a, impl == 6);
                    AHA_CUDA_CHECK(cudaEventRecord(m->ev1, c.stream));
                    AHA_CUDA_CHECK(cudaStreamSynchronize(c.stream));
                } catch (...) { cudaFree(ones); throw; }
                cudaFree(ones);
                if (device_ms) { float ms = 0.f; AHA_CUDA_CHECK(cudaEventElapsedTime(&ms, m->ev0, m->ev1)); *device_ms = ms; }
                AHA_CUDA_CHECK(cudaMemcpy(out, dy, (size_t)M * Nout * 4, cudaMemcpyDeviceToHost));
                cleanup();
                return;
            }
            const int saved = c.gemm_impl;
            c.gemm_impl = impl;
            try {
                linear_gemm(c, epi, dx, K, W, dr, N, dy, Nout, M, act);   // warm-up + correctness run
                AHA_CUDA_CHECK(cudaEventRecord(m->ev0, c.stream));
                for (int i = 0; i < std::max(iters, 0); ++i) linear_gemm(c, epi, dx, K, W, dr, N, dy, Nout, M, act);
                AHA_CUDA_CHECK(cudaEventRecord(m->ev1, c.stream));
                AHA_CUDA_CHECK(cudaStreamSynchronize(c.stream));
            } catch (...) { c.gemm_impl = saved; throw; }
            c.gemm_impl = saved;
            if (device_ms) { float ms = 0.f; AHA_CUDA_CHECK(cudaEventElapsedTime(&ms, m->ev0, m->ev1)); *device_ms = ms; }
            AHA_CUDA_CHECK(cudaMemcpy(out, dy, (size_t)M * Nout * 4, cudaMemcpyDeviceToHost));
        } catch (...) { cleanup(); throw; }
        cleanup();
    });
}

namespace {
// Qwen3Model::forward_hidden + l2_normalize for one text; result left in T.xn[0:H] and copied to `out`
void embed_one(aha_model* m, const uint32_t* ids, size_t S, float* out) {
    require_no_session(m);
    AHA_REQUIRE(m->kind == aha_model::QWEN3, "embeddings need a qwen3 handle (Qwen3-Embedding shares Qwen3Model)");
    AHA_REQUIRE(ids && S >= 1 && out, "ids, seq_len and out are required");
    TextModel& T = m->text;
    drop_cache(m);
    upload_ids(m, ids, S);
    std::vector<int> pos3((size_t)3 * S);
    for (int r = 0; r < 3; ++r) for (size_t i = 0; i < S; ++i) pos3[(size_t)r * S + i] = (int)i;
    upload_pos(m, pos3);
    T.prefill((int)S, 0, false, nullptr, 0, {});
    const int H = T.cfg.H;
    rmsnorm_kernel<<<1, 256, 0, m->ctx.stream>>>(T.x + (size_t)(S - 1) * H, T.norm, T.cfg.eps, T.xn, H);
    l2_normalize_kernel<<<1, 256, 0, m->ctx.stream>>>(T.xn, T.xn + H, H);
    m->ctx.cnt.kernels += 2;
    AHA_CUDA_CHECK(cudaMemcpyAsync(out, T.xn + H, (size_t)H * sizeof(float), cudaMemcpyDeviceToHost, m->ctx.stream));
    AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
    drop_cache(m);   // clear_kv_cache()
}
}  // namespace

int aha_b200_embed(aha_model* m, const uint32_t* ids, size_t seq_len, float* out) {
    return guarded(m, [&] { embed_one(m, ids, seq_len, out); });
}

int aha_b200_rerank(aha_model* m, const uint32_t* query_ids, size_t query_len, const uint32_t* doc_ids, const size_t* doc_lens, size_t n_docs,
                    float* scores_out) {
    return guarded(m, [&] {
        AHA_REQUIRE(doc_ids && doc_lens && scores_out && n_docs >= 1, "documents are required (embedding input cannot be empty)");
        const int H = m->text.cfg.H;
        std::vector<float> q(H), d(H);
        embed_one(m, query_ids, query_len, q.data());
        size_t off = 0;
        for (size_t i = 0; i < n_docs; ++i) {
            embed_one(m, doc_ids + off, doc_lens[i], d.data());
            off += doc_lens[i];
            float acc = 0.f;   // (1,H) x (H,1) in fp32, like the reference's matmul of two host-side f32 tensors
            for (int k = 0; k < H; ++k) acc += q[k] * d[k];
            scores_out[i] = acc;
        }
    });
}

int aha_b200_nccl_unique_id(uint8_t out[128]) {
    try {
        AHA_REQUIRE(out != nullptr, "out is required");
        NcclApi& n = NcclApi::get();
        NcclApi::unique_id id;
        n.check(n.GetUniqueId(&id), "ncclGetUniqueId");
        std::memcpy(out, &id, 128);
        return 0;
    } catch (const std::exception& e) {
        std::lock_guard<std::mutex> lk(g_err_mu);
        g_create_error = e.what();
        return 1;
    }
}

int aha_b200_rope_index_mm(const uint32_t* ids, size_t seq_len, const uint32_t* grid_thw, size_t n_images, const uint32_t* video_grid_thw, size_t n_videos,
                           uint32_t spatial_merge_size, uint32_t image_token_id, uint32_t video_token_id, uint32_t vision_start_token_id, int32_t* pos3_out,
                           int32_t* rope_delta_out) {
    try {
        AHA_REQUIRE(ids != nullptr && seq_len > 0 && pos3_out != nullptr && rope_delta_out != nullptr, "ids, pos3_out and rope_delta_out are required");
        AHA_REQUIRE(n_images == 0 || grid_thw != nullptr, "grid_thw is required when n_images > 0");
        AHA_REQUIRE(n_videos == 0 || video_grid_thw != nullptr, "video_grid_thw is required when n_videos > 0");
        AHA_REQUIRE(spatial_merge_size > 0 && seq_len < (size_t)1 << 30, "bad spatial_merge_size / seq_len");
        std::vector<std::array<int, 3>> grid(n_images), frames;
        for (size_t i = 0; i < n_images; ++i) grid[i] = {(int)grid_thw[3 * i], (int)grid_thw[3 * i + 1], (int)grid_thw[3 * i + 2]};
        for (size_t i = 0; i < n_videos; ++i)
            for (uint32_t t = 0; t < video_grid_thw[3 * i]; ++t) frames.push_back({1, (int)video_grid_thw[3 * i + 1], (int)video_grid_thw[3 * i + 2]});
        std::vector<int> pos3;
        int delta = 0;
        get_rope_index(ids, (int)seq_len, grid, frames, (int)spatial_merge_size, (int)image_token_id, (int)video_token_id, (int)vision_start_token_id, pos3, delta);
        for (size_t i = 0; i < pos3.size(); ++i) pos3_out[i] = pos3[i];
        *rope_delta_out = delta;
        return 0;
    } catch (const std::exception& e) {
        std::lock_guard<std::mutex> lk(g_err_mu);
        g_create_error = e.what();
        return 1;
    }
}
int aha_b200_rope_index(const uint32_t* ids, size_t seq_len, const uint32_t* grid_thw, size_t n_images, uint32_t spatial_merge_size,
                        uint32_t image_token_id, uint32_t vision_start_token_id, int32_t* pos3_out, int32_t* rope_delta_out) {
    return aha_b200_rope_index_mm(ids, seq_len, grid_thw, n_images, nullptr, 0, spatial_merge_size, image_token_id, 0xffffffffu, vision_start_token_id, pos3_out,
                                  rope_delta_out);
}

void aha_b200_destroy(aha_model* m) {
    if (!m) return;
    cudaSetDevice(m->ctx.device);
    if (m->ctx.stream) cudaStreamSynchronize(m->ctx.stream);
    m->text.destroy();
    m->batch.clear_graphs();
    m->ctx.free_all();
    if (m->h_pin) cudaFreeHost(m->h_pin);
    if (m->ev0) cudaEventDestroy(m->ev0);
    if (m->ev1) cudaEventDestroy(m->ev1);
    for (auto& e : m->ev_tok) if (e) cudaEventDestroy(e);
    if (m->ctx.stream) cudaStreamDestroy(m->ctx.stream);
    delete m;
}

const char* aha_b200_last_error(aha_model* m) {
    if (m) return m->last_error.c_str();
    std::lock_guard<std::mutex> lk(g_err_mu);
    static thread_local std::string copy;
    copy = g_create_error;
    return copy.c_str();
}

void* aha_b200_stream(aha_model* m) { return m ? (void*)m->ctx.stream : nullptr; }

int aha_b200_get_stats(aha_model* m, aha_stats* out) {
    return guarded(m, [&] {
        AHA_REQUIRE(out, "out is required");
        out->kernel_launches = m->ctx.cnt.kernels;
        out->graph_launches = m->ctx.cnt.graphs;
        out->kernels_per_decode_step = m->text.step_graph_kernels;
        out->weight_bytes = m->ctx.alloc_bytes;
        out->kv_bytes_per_token = (uint64_t)m->text.cfg.L * 2 * m->text.nkv_l * m->text.cfg.hd * sizeof(float);
        out->decode_bytes_per_step_fixed = m->text.decode_weight_bytes;
    });
}
int aha_b200_reset_stats(aha_model* m) {
    return guarded(m, [&] { m->ctx.cnt = Counters{}; });
}
int aha_b200_set_trace(aha_model* m, int on) {
    return guarded(m, [&] {
        m->text.set_trace(on != 0);
        if (m->kind == aha_model::QWEN3VL) m->vision.set_trace(on != 0);
        if (m->kind == aha_model::QWEN3_ASR) m->audio.set_trace(on != 0);
    });
}
int aha_b200_debug_read(aha_model* m, const char* what, int index, float* out, size_t cap, size_t* n) {
    return guarded(m, [&] {
        AHA_REQUIRE(what && out && n, "what, out and n are required");
        const std::string w = what;
        const float* src = nullptr;
        size_t cnt = 0;
        TextModel& T = m->text;
        if (w == "hidden") {
            AHA_REQUIRE(T.trace_buf && index >= 0 && index < T.cfg.L, "hidden trace not available");
            src = T.trace_buf + (size_t)index * T.max_prefill * T.cfg.H; cnt = (size_t)T.trace_S * T.cfg.H;
        } else if (w == "vit") {
            AHA_REQUIRE(m->kind == aha_model::QWEN3VL && m->vision.trace_buf && index >= 0 && index <= m->vision.cfg.depth, "vit trace not available");
            src = m->vision.trace_buf + (size_t)index * m->vision.max_patches * m->vision.cfg.H; cnt = (size_t)m->vision.last_N * m->vision.cfg.H;
        } else if (w == "image_embeds") {
            AHA_REQUIRE(m->kind == aha_model::QWEN3VL, "image_embeds needs a qwen3vl handle");
            const int ne = m->vision.last_N / (m->vision.cfg.merge * m->vision.cfg.merge);
            src = index <= 0 ? m->vision.image_embeds : m->vision.ds_out.at(index - 1); cnt = (size_t)ne * m->vision.cfg.out_hidden;
        } else if (w == "audio") {
            AHA_REQUIRE(m->kind == aha_model::QWEN3_ASR && m->audio.trace_buf && index >= 0 && index <= m->audio.cfg.layers, "audio trace not available");
            src = m->audio.trace_buf + (size_t)index * m->audio.max_tokens * m->audio.cfg.d_model; cnt = (size_t)m->audio.last_tokens * m->audio.cfg.d_model;
        } else if (w == "audio_embeds") {
            AHA_REQUIRE(m->kind == aha_model::QWEN3_ASR, "audio_embeds needs a qwen3_asr handle");
            src = m->audio.audio_embeds; cnt = (size_t)m->audio.last_tokens * m->audio.cfg.out_dim;
        } else if (w == "fused_trace") {  // globaltimer stamps (ns, relative to the first) of CTA 0; index 0 = consumer, 1 = producer
            AHA_REQUIRE(T.d_ftrace && (index == 0 || index == 1) && cap >= 4096, "fused trace not available");
            std::vector<unsigned long long> h(4096);
            AHA_CUDA_CHECK(cudaMemcpy(h.data(), T.d_ftrace + (size_t)index * 4096, 4096 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            size_t k = 0;
            for (; k < 4096 && h[k]; ++k) out[k] = (float)(double)(h[k] - h[0]);
            *n = k; return;
        } else if (w == "fused_cta_trace") {  // barrier arrival stamps of CTA `index` (ns relative to CTA 0's first), [255] = %smid
            AHA_REQUIRE(T.d_ftrace && index >= 0 && index < 256 && cap >= 256, "fused trace not available");
            std::vector<unsigned long long> h(256);
            unsigned long long base = 0;
            AHA_CUDA_CHECK(cudaMemcpy(&base, T.d_ftrace + 8192, sizeof(base), cudaMemcpyDeviceToHost));
            AHA_CUDA_CHECK(cudaMemcpy(h.data(), T.d_ftrace + 8192 + (size_t)index * 256, 256 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            for (size_t k = 0; k < 255; ++k) out[k] = h[k] ? (float)((double)h[k] - (double)base) : -1e30f;
            out[255] = (float)h[255];
            *n = 256; return;
        } else if (w == "fused_stage_trace") {  // AHA_STAGE_TRACE builds: 4 stamps per ring stage of the traced CTA, ns relative to the earliest stamp (0 = missing)
            AHA_REQUIRE(T.d_ftrace && cap >= 4 * 8192, "fused trace not available");
            std::vector<unsigned long long> h(4 * 8192);
            AHA_CUDA_CHECK(cudaMemcpy(h.data(), T.d_ftrace + 8192, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            unsigned long long base = ~0ull;
            for (auto v : h) if (v && v < base) base = v;
            for (size_t k = 0; k < h.size(); ++k) out[k] = h[k] ? (float)((double)(h[k] - base) + 1.0) : 0.f;
            AHA_CUDA_CHECK(cudaMemset(T.d_ftrace + 8192, 0, h.size() * sizeof(unsigned long long)));
            *n = h.size(); return;
        } else if (w == "fused_sync_trace") {  // AHA_STAGE_TRACE builds, dbg bit10: [0, 4096) = 8 words per grid barrier, [4096, 8192) = 4 per activation load
            AHA_REQUIRE(T.d_ftrace && cap >= 8192, "fused trace not available");
            std::vector<unsigned long long> h(8192);
            AHA_CUDA_CHECK(cudaMemcpy(h.data(), T.d_ftrace + 8192 + 32768, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            unsigned long long base = ~0ull;
            for (auto v : h) if (v > 1000000000000ull && v < base) base = v;
            for (size_t k = 0; k < h.size(); ++k) out[k] = h[k] > 1000000000000ull ? (float)((double)(h[k] - base) + 1.0) : (float)h[k];   // small values are counts
            AHA_CUDA_CHECK(cudaMemset(T.d_ftrace + 8192 + 32768, 0, h.size() * sizeof(unsigned long long)));
            *n = h.size(); return;
        } else if (w == "rope_delta") {
            AHA_REQUIRE(cap >= 1, "out too small");
            out[0] = (float)m->rope_delta; *n = 1; return;
        } else {
            throw std::runtime_error("unknown debug tensor '" + w + "'");
        }
        AHA_REQUIRE(cnt <= cap, "out too small");
        AHA_CUDA_CHECK(cudaMemcpyAsync(out, src, cnt * sizeof(float), cudaMemcpyDeviceToHost, m->ctx.stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(m->ctx.stream));
        *n = cnt;
    });
}

}  // extern "C"
