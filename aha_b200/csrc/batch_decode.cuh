// batch_decode.cuh -- several sequences decoded in lockstep on one handle (SURVEY 8f rank 4, second half).
//
// The reference holds one request at a time behind a lock (/root/reference/src/server/api.rs:117) and every decode step
// streams all weights for ONE token.  Here up to 8 sequences share a step: each has its own page table over the common
// paged KV pool (text_model.cuh), its own DecodeState (token, position, rope_delta, sampler draw index), history and sampler
// parameters; a step is per layer
//     [rmsnorm + qkv]  gemv_batch_kernel        all sequences, every weight row read once
//     [attention]      decode_attn_batch_kernel grid.z = sequence: q/k norm, RoPE, KV append, split-KV attention, merge
//     [o_proj + res]   gemv_batch_kernel
//     [rmsnorm + gate/up + SwiGLU], [down + res]
// then final norm + lm_head for all rows and, per sequence, the two-stage ArgMax that advances its DecodeState plus (when the
// request samples) sample_kernel on its logits row.  Each sequence therefore produces exactly the tokens it would produce alone:
// the GEMV accumulates every (row, sequence) in gemv_kernel's order and the attention / sampler kernels are the single-sequence
// ones (tests/test_batch_gpu.py compares every sequence with its own fresh oracle run).
// Finished sequences leave the step (the activation rows are rebuilt from the token embeddings every step, so compaction is free).
#pragma once
#include "gemv_batch.cuh"
#include "text_model.cuh"

namespace aha {

struct BatchSlot {                       // one sequence of the batch
    std::vector<int> h_table;            // its page table (host copy), swapped into the TextModel while the sequence prefills
    int mapped = 0;
    int* d_table = nullptr;              // device copy: row of BatchDecoder::d_tables
    bool samp_active = false;
    SampleArgs samp{};                   // sampler of the request with the pointers of this slot
};

struct BatchDecoder {
    TextModel* T = nullptr;
    int cap = 0;                         // slots allocated
    float *xb = nullptr, *qkvb = nullptr, *attnb = nullptr, *hb = nullptr, *logitsb = nullptr, *partialb = nullptr;
    int* countersb = nullptr;
    float* pmaxb = nullptr; int* pidxb = nullptr; int n_pcand = 0;
    DecodeState* d_states = nullptr;     // [cap]
    uint32_t* d_hist = nullptr;          // [cap][hist_cap]
    uint32_t* d_tok = nullptr;           // [cap] token of the last step per slot
    int* d_tables = nullptr;             // [cap][num_pages]
    DecodeAttnArgs* d_attn = nullptr;    // [L][cap] attention arguments of the current active list
    std::vector<BatchSlot> slots;
    std::vector<int> table_for;          // active list the attention table was built for
    // One CUDA graph per composition of the batch (the active list changes only when a request joins or leaves): ~170 launches per step become one.
    // The graphs hold the requests' sampler parameters by value, so they are dropped whenever a request leaves its slot.
    struct StepGraph { std::vector<int> act; int simt; cudaGraphExec_t exec; uint64_t kernels; };
    std::vector<StepGraph> graphs;
    void clear_graphs() {
        for (auto& g : graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
        graphs.clear();
    }
    // no sequence in any slot (their pages go back with the model's reset_pages), no attention table, no graphs
    void reset() {
        for (auto& s : slots) { s.mapped = 0; s.samp_active = false; }
        table_for.clear();
        clear_graphs();
    }

    void init(TextModel& t, int n) {
        T = &t;
        if (n <= cap) return;
        AHA_REQUIRE(cap == 0, "batch decoder already sized");   // one size per handle: kGemvBatchMax
        Ctx& c = *t.ctx;
        cap = n;
        const TextCfg& cf = t.cfg;
        xb = c.alloc<float>((size_t)n * cf.H); qkvb = c.alloc<float>((size_t)n * t.qkv_dim); attnb = c.alloc<float>((size_t)n * t.nh_l * cf.hd);
        hb = c.alloc<float>((size_t)n * t.I_l); logitsb = c.alloc<float>((size_t)n * cf.V);
        partialb = c.alloc<float>((size_t)n * t.nh_l * kDecodeSplits * (cf.hd + 2));
        countersb = c.alloc<int>((size_t)n * t.nkv_l);
        AHA_CUDA_CHECK(cudaMemset(countersb, 0, (size_t)n * t.nkv_l * sizeof(int)));
        n_pcand = 64;
        pmaxb = c.alloc<float>((size_t)n * n_pcand); pidxb = c.alloc<int>((size_t)n * n_pcand);
        d_states = c.alloc<DecodeState>(n);
        d_hist = c.alloc<uint32_t>((size_t)n * t.hist_cap);
        d_tok = c.alloc<uint32_t>(n);
        d_tables = c.alloc<int>((size_t)n * t.num_pages);
        d_attn = c.alloc<DecodeAttnArgs>((size_t)cf.L * n);
        slots.resize(n);
        for (int i = 0; i < n; ++i) { slots[i].h_table.assign(t.num_pages, 0); slots[i].d_table = d_tables + (size_t)i * t.num_pages; }
    }

    // While slot i prefills, the TextModel's own page-table members are this slot's (prefill / ensure_tokens / kv_src work on them unchanged)
    void swap_table(int i) {
        BatchSlot& s = slots[i];
        std::swap(T->h_page_table, s.h_table);
        std::swap(T->pages_mapped, s.mapped);
        std::swap(T->d_page_table, s.d_table);
    }

    // after the prefill of slot i (the model's d_state / d_history / samp hold the request's state): move it into the slot
    void adopt(int i, uint32_t first_token, int seq_len, int rope_delta, uint32_t n_draws) {
        Ctx& c = *T->ctx;
        BatchSlot& s = slots[i];
        DecodeState st{first_token, seq_len, rope_delta, 1, n_draws, {0, 0, 0}};
        AHA_CUDA_CHECK(cudaMemcpyAsync(d_states + i, &st, sizeof(st), cudaMemcpyHostToDevice, c.stream));
        AHA_CUDA_CHECK(cudaMemcpyAsync(d_hist + (size_t)i * T->hist_cap, &first_token, sizeof(uint32_t), cudaMemcpyHostToDevice, c.stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(c.stream));   // stack temporaries
        s.samp_active = T->samp_active;
        if (s.samp_active) {
            s.samp = T->samp;
            s.samp.logits = logitsb;                 // row set per step (the slot's position in the active list)
            s.samp.st = d_states + i;
            s.samp.history = d_hist + (size_t)i * T->hist_cap;
            s.samp.token_out = d_tok + i;
        }
    }

    void build_attn_table(const std::vector<int>& act) {
        const TextCfg& cf = T->cfg;
        const int nb = (int)act.size();
        std::vector<DecodeAttnArgs> h((size_t)cf.L * cap);
        const float scaling = (float)(1.0 / std::sqrt((double)cf.hd));
        for (int l = 0; l < cf.L; ++l) {
            TextLayer& Ly = T->layers[l];
            KVSrc kv = T->kv_src(l);
            for (int j = 0; j < nb; ++j) {
                DecodeAttnArgs d{};
                const int slot = act[j];
                d.qkv = qkvb + (size_t)j * T->qkv_dim; d.qw = Ly.qn; d.kw = Ly.kn; d.eps = cf.eps; d.inv_freq = T->inv_freq; d.st = d_states + slot;
                d.kbase = const_cast<float*>(kv.k); d.vbase = const_cast<float*>(kv.v);
                d.kv = kv; d.kv.page_table = d_tables + (size_t)slot * T->num_pages;
                d.partial = partialb + (size_t)j * T->nh_l * kDecodeSplits * (cf.hd + 2);
                d.counters = countersb + (size_t)j * T->nkv_l;
                d.out = attnb + (size_t)j * T->nh_l * cf.hd;
                d.nh = T->nh_l; d.nkv = T->nkv_l; d.nsplit = kDecodeSplits; d.scaling = scaling;
                h[(size_t)l * cap + j] = d;
            }
        }
        Ctx& c = *T->ctx;
        AHA_CUDA_CHECK(cudaMemcpyAsync(d_attn, h.data(), h.size() * sizeof(DecodeAttnArgs), cudaMemcpyHostToDevice, c.stream));
        AHA_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        table_for = act;
    }

    template <int G>
    void launch_attn(int l, int nb) {
        decode_attn_batch_kernel<128, G><<<dim3(kDecodeSplits, T->nkv_l, nb), 256, 0, T->ctx->stream>>>(d_attn + (size_t)l * cap);
    }

    void proj(int pro, int epi, const LinearW& W, const float* x, int ldx, const float* norm_w, const float* resid, int ldr, float* out, int ldo, int nb, int simt) {   // simt: 0 = batched GEMV (registers), 1 = exact SIMT GEMM twin, 2 = batched GEMV with the cp.async weight ring
        Ctx& c = *T->ctx;
        if (simt == 1) {   // validation twin: the exact fp32 SIMT GEMM over the nb rows (normalised beforehand when a prologue is asked for)
            const float* a = x; int lda = ldx;
            if (pro == PRO_RMSNORM) {
                rmsnorm_kernel<<<nb, 256, 0, c.stream>>>(x, norm_w, T->cfg.eps, T->xn, W.K); c.cnt.kernels++;   // xn: [max_prefill >= 8][H] scratch of the prefill
                a = T->xn; lda = W.K;
            }
            GemmArgs g{};
            g.A = a; g.lda = lda; g.W = W.w; g.bias = W.b; g.resid = resid; g.ldr = ldr; g.C = out; g.ldc = ldo; g.M = nb; g.N = W.N; g.K = W.K; g.act = ACT_NONE;
            gemm_simt(c.stream, epi == GEPI_STORE ? EPI_STORE : (epi == GEPI_RESID ? EPI_RESID : EPI_SWIGLU), g);
            c.cnt.kernels++;
            return;
        }
        GemvBatchArgs a{};
        a.W = W.w; a.x = x; a.ldx = ldx; a.norm_w = norm_w; a.eps = T->cfg.eps; a.bias = W.b; a.resid = resid; a.ldr = ldr; a.out = out; a.ldo = ldo;
        a.N = W.N; a.K = W.K; a.nb = nb;
        gemv_batch(c.stream, pro, epi, a, simt == 2);
        c.cnt.kernels++;
    }

    // one decode step of the sequences in `act` (slot indices, at most cap); leaves every slot's next token in d_tok[slot] and its DecodeState advanced
    void step(const std::vector<int>& act, int simt, bool use_graph) {
        Ctx& c = *T->ctx;
        AHA_REQUIRE(!act.empty() && (int)act.size() <= cap, "batch step: bad active list");
        if (act != table_for) build_attn_table(act);
        if (!use_graph) { launches(act, simt); return; }
        StepGraph* g = nullptr;
        for (auto& e : graphs) if (e.simt == simt && e.act == act) { g = &e; break; }
        if (!g) {
            const uint64_t k0 = c.cnt.kernels;
            cudaGraph_t cg = nullptr;
            AHA_CUDA_CHECK(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
            try { launches(act, simt); } catch (...) { cudaStreamEndCapture(c.stream, &cg); if (cg) cudaGraphDestroy(cg); throw; }
            AHA_CUDA_CHECK(cudaStreamEndCapture(c.stream, &cg));
            StepGraph e{act, simt, nullptr, c.cnt.kernels - k0};
            c.cnt.kernels = k0;
            const cudaError_t err = cudaGraphInstantiate(&e.exec, cg, 0);
            cudaGraphDestroy(cg);
            AHA_CUDA_CHECK(err);
            graphs.push_back(e);
            g = &graphs.back();
        }
        AHA_CUDA_CHECK(cudaGraphLaunch(g->exec, c.stream));
        c.cnt.graphs++;
        c.cnt.kernels += g->kernels;
    }
    void launches(const std::vector<int>& act, int simt) {
        Ctx& c = *T->ctx;
        cudaStream_t st = c.stream;
        const TextCfg& cf = T->cfg;
        const int nb = (int)act.size(), H = cf.H;
        for (int j = 0; j < nb; ++j) { embed_gather_kernel<<<1, 256, 0, st>>>(&d_states[act[j]].token, T->embed, xb + (size_t)j * H, 1, H, cf.V); c.cnt.kernels++; }
        for (int l = 0; l < cf.L; ++l) {
            TextLayer& Ly = T->layers[l];
            proj(PRO_RMSNORM, GEPI_STORE, Ly.qkv, xb, H, Ly.ln1, nullptr, 0, qkvb, T->qkv_dim, nb, simt);
            switch (T->nh_l / T->nkv_l) {
                case 1: launch_attn<1>(l, nb); break;
                case 2: launch_attn<2>(l, nb); break;
                case 4: launch_attn<4>(l, nb); break;
                default: launch_attn<6>(l, nb); break;
            }
            c.cnt.kernels++;
            proj(PRO_NONE, GEPI_RESID, Ly.o, attnb, T->nh_l * cf.hd, nullptr, xb, H, xb, H, nb, simt);
            proj(PRO_RMSNORM, GEPI_SWIGLU, Ly.gu, xb, H, Ly.ln2, nullptr, 0, hb, T->I_l, nb, simt);
            proj(PRO_NONE, GEPI_RESID, Ly.down, hb, T->I_l, nullptr, xb, H, xb, H, nb, simt);
        }
        LinearW head; head.w = T->lm_head; head.b = nullptr; head.N = cf.V; head.K = H;
        proj(PRO_RMSNORM, GEPI_STORE, head, xb, H, T->norm, nullptr, 0, logitsb, cf.V, nb, simt);
        for (int j = 0; j < nb; ++j) {
            const int slot = act[j];
            const float* lg = logitsb + (size_t)j * cf.V;
            argmax_partial_kernel<<<n_pcand, 256, 0, st>>>(lg, cf.V, pmaxb + (size_t)j * n_pcand, pidxb + (size_t)j * n_pcand);
            argmax_final_kernel<<<1, 32, 0, st>>>(pmaxb + (size_t)j * n_pcand, pidxb + (size_t)j * n_pcand, n_pcand, d_tok + slot, d_states + slot,
                                                  d_hist + (size_t)slot * T->hist_cap, T->hist_cap, 1);
            c.cnt.kernels += 2;
            BatchSlot& s = slots[slot];
            if (s.samp_active) {   // the sampled token replaces the ArgMax one the step just pushed (the single-sequence loop does the same)
                SampleArgs a = s.samp;
                a.logits = lg;
                a.overwrite = 1;
                sample_kernel<<<1, kSampleThreads, 0, st>>>(a);
                c.cnt.kernels++;
            }
        }
        AHA_CUDA_CHECK(cudaGetLastError());
    }
};

}  // namespace aha
