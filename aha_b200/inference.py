"""Host-side mirror of aha's model-executor seam for the B200 path.

`B200Model` has the methods of `trait InferenceModel`
(/root/reference/src/models/common/mod.rs:25-45): forward_initial, forward_step, clear_cache,
stop_token_ids -- same names, argument meaning and error behaviour (errors are raised, never
swallowed) -- and `generate` = generate_generic (/root/reference/src/models/common/generate.rs:115-159).
Everything here is plumbing around libaha_b200.so; no arithmetic happens in Python."""
import ctypes as C
import json

import numpy as np

from . import _lib as L


class B200Error(RuntimeError):
    pass


class MultiModalData:
    """common/mod.rs:14-22 -- positional list of optional tensors."""

    def __init__(self, data_vec):
        self.data_vec = list(data_vec)


def nccl_unique_id():
    """128-byte ncclUniqueId created by the calling rank (rank 0); broadcast it to the other ranks."""
    lib = L.load()
    buf = (C.c_uint8 * 128)()
    if lib.aha_b200_nccl_unique_id(buf) != 0:
        raise B200Error(lib.aha_b200_last_error(None).decode())
    return bytes(buf)


def rope_index(ids, grid_thw, config, video_grid_thw=None):
    """M-RoPE position ids (3, S) int32 and rope_delta of a Qwen3-VL prompt -- the host routine forward_initial runs
    (Qwen3VLModel::get_rope_index, /root/reference/src/models/qwen3vl/model.rs:901-1133), image and video branches.  No device work."""
    lib = L.load()
    ids = np.ascontiguousarray(np.asarray(ids).reshape(-1), dtype=np.uint32)
    grid = np.ascontiguousarray(np.asarray(grid_thw if grid_thw is not None else [], dtype=np.uint32).reshape(-1, 3))
    vgrid = np.ascontiguousarray(np.asarray(video_grid_thw if video_grid_thw is not None else [], dtype=np.uint32).reshape(-1, 3))
    pos = np.empty((3, ids.size), np.int32)
    delta = C.c_int32(0)
    u32 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint32))
    rc = lib.aha_b200_rope_index_mm(u32(ids), ids.size, u32(grid), grid.shape[0], u32(vgrid), vgrid.shape[0],
                                    int(config["vision_config"]["spatial_merge_size"]), int(config["image_token_id"]),
                                    int(config.get("video_token_id", 0xffffffff)), int(config["vision_start_token_id"]),
                                    pos.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(delta))
    if rc != 0:
        raise B200Error(lib.aha_b200_last_error(None).decode())
    return pos, int(delta.value)


def prefix_match(cached_ids, ids, mm_token_ids=(), same_mm=True):
    """The rule behind generate(reuse_prefix=True), host only: how many leading tokens of `ids` a KV cache holding `cached_ids`
    can supply (see aha_b200_prefix_match in include/aha_b200.h)."""
    lib = L.load()
    a = np.ascontiguousarray(np.asarray(cached_ids, dtype=np.uint32).reshape(-1))
    b = np.ascontiguousarray(np.asarray(ids, dtype=np.uint32).reshape(-1))
    t = np.ascontiguousarray(np.asarray(list(mm_token_ids), dtype=np.uint32).reshape(-1))
    u32 = lambda x: x.ctypes.data_as(C.POINTER(C.c_uint32))
    return int(lib.aha_b200_prefix_match(u32(a), a.size, u32(b), b.size, u32(t), t.size, 1 if same_mm else 0))


def mm_fingerprint(data):
    """64-bit fingerprint of a MultiModalData list (0 = no tensor): what decides whether two requests carry the same images / audio."""
    lib = L.load()
    mm, _keep = B200Model._mm(None, data)
    return int(lib.aha_b200_mm_fingerprint(C.byref(mm))) if mm is not None else 0


class B200Model:
    def __init__(self, kind, config, weights, eos_ids=(), device=0, max_ctx=8192, max_prefill=0, max_patches=0,
                 max_frames=0, use_graph=True, decode_impl=0, gemm_impl=0, attn_impl=0, tp_rank=0, tp_world=1, tp_unique_id=None):
        self._lib = L.load()
        self.kind = kind
        self.config = config
        cfg_json = json.dumps(config).encode()
        names = list(weights.keys())
        arrs = [weights[n] if (isinstance(weights[n], np.ndarray) and weights[n].flags["C_CONTIGUOUS"]) else np.ascontiguousarray(weights[n])
                for n in names]   # (a BF16-tagged view must keep its subclass)
        descs = (L.TensorDesc * len(names))(*[L.make_desc(a, n) for a, n in zip(arrs, names)])
        eos = np.asarray(list(eos_ids), dtype=np.uint32)
        opts = L.Options(device=device, tp_rank=tp_rank, tp_world=tp_world, max_ctx=max_ctx, max_prefill=max_prefill,
                         max_patches=max_patches, max_frames=max_frames, use_graph=1 if use_graph else 0,
                         decode_impl=decode_impl, gemm_impl=gemm_impl)
        opts.reserved[0] = attn_impl
        if tp_world > 1:
            if tp_unique_id is None or len(tp_unique_id) != 128:
                raise ValueError("tp_world > 1 needs the 128-byte NCCL unique id (nccl_unique_id() on rank 0, then broadcast)")
            self._tp_id = (C.c_uint8 * 128)(*bytes(tp_unique_id))
            opts.tp_comm = C.cast(self._tp_id, C.c_void_p)
        h = C.c_void_p()
        rc = self._lib.aha_b200_create(kind.encode(), cfg_json, descs, len(names),
                                       eos.ctypes.data_as(C.POINTER(C.c_uint32)), len(eos), C.byref(opts), C.byref(h))
        if rc != 0:
            raise B200Error(self._lib.aha_b200_last_error(None).decode())
        self._h = h
        tc = config if kind == "qwen3" else (config["text_config"] if kind == "qwen3vl" else config["thinker_config"]["text_config"])
        self.vocab_size = tc["vocab_size"]
        self.hidden_size = tc["hidden_size"]

    # ------------------------------------------------------------------ helpers
    def _check(self, rc):
        if rc != 0:
            raise B200Error(self._lib.aha_b200_last_error(self._h).decode())

    def _mm(self, data):
        if data is None:
            return None, None
        vec = data.data_vec if isinstance(data, MultiModalData) else list(data)
        keep, descs = [], []
        for t in vec:
            if t is None:
                d = L.TensorDesc()
                d.data = None
            else:
                a = np.ascontiguousarray(t)
                if a.dtype == np.int32:
                    a = a.astype(np.int64)
                keep.append(a)
                d = L.make_desc(a)
            descs.append(d)
        arr = (L.TensorDesc * len(descs))(*descs)
        mm = L.MM(arr, len(descs))
        return mm, (keep, arr)

    @staticmethod
    def _ids(input_ids):
        return np.ascontiguousarray(np.asarray(input_ids, dtype=np.uint32).reshape(-1))

    # ------------------------------------------------------------------ InferenceModel
    def forward_initial(self, input_ids, seqlen_offset, data=None, want_logits=True):
        """-> logits (1,1,V) float32 (like the reference's Tensor) and sets self.last_argmax."""
        ids = self._ids(input_ids)
        mm, _keep = self._mm(data)
        logits = np.empty(self.vocab_size, np.float32) if want_logits else None
        am = C.c_uint32(0)
        self._check(self._lib.aha_b200_forward_initial(
            self._h, ids.ctypes.data_as(C.POINTER(C.c_uint32)), ids.size, int(seqlen_offset),
            C.byref(mm) if mm is not None else None,
            logits.ctypes.data_as(C.POINTER(C.c_float)) if want_logits else None, C.byref(am)))
        self.last_argmax = int(am.value)
        return logits.reshape(1, 1, -1) if want_logits else None

    def forward_step(self, input_ids, seqlen_offset, want_logits=True):
        ids = self._ids(input_ids)
        logits = np.empty(self.vocab_size, np.float32) if want_logits else None
        am = C.c_uint32(0)
        self._check(self._lib.aha_b200_forward_step(
            self._h, ids.ctypes.data_as(C.POINTER(C.c_uint32)), ids.size, int(seqlen_offset),
            logits.ctypes.data_as(C.POINTER(C.c_float)) if want_logits else None, C.byref(am)))
        self.last_argmax = int(am.value)
        return logits.reshape(1, 1, -1) if want_logits else None

    def forward_extend(self, input_ids, seqlen_offset, want_logits=True):
        """Prefill continuation (new design; the reference's (S, S) mask rejects S > 1 with a non-empty cache): further prompt
        tokens against the `seqlen_offset` tokens already in the cache -> logits of the last one."""
        ids = self._ids(input_ids)
        logits = np.empty(self.vocab_size, np.float32) if want_logits else None
        am = C.c_uint32(0)
        self._check(self._lib.aha_b200_forward_extend(
            self._h, ids.ctypes.data_as(C.POINTER(C.c_uint32)), ids.size, int(seqlen_offset),
            logits.ctypes.data_as(C.POINTER(C.c_float)) if want_logits else None, C.byref(am)))
        self.last_argmax = int(am.value)
        return logits.reshape(1, 1, -1) if want_logits else None

    def last_prefix_hit(self):
        """Prompt tokens the last generate call took from the KV cache (reuse_prefix=True) instead of prefilling them."""
        return int(self._lib.aha_b200_last_prefix_hit(self._h))

    def clear_cache(self):
        self._check(self._lib.aha_b200_clear_cache(self._h))

    def stop_token_ids(self):
        n = self._lib.aha_b200_stop_token_ids(self._h, None, 0)
        out = (C.c_uint32 * max(n, 1))()
        self._lib.aha_b200_stop_token_ids(self._h, out, n)
        return [int(out[i]) for i in range(n)]

    # ------------------------------------------------------------------ generate_generic / generate_stream_generic
    @staticmethod
    def _gen_params(max_tokens, temperature, top_p, top_k, repeat_penalty, repeat_last_n, seed, flags=0):
        return L.GenParams(temperature=temperature or 0.0, repeat_penalty=repeat_penalty, repeat_last_n=repeat_last_n,
                           max_tokens=max_tokens, seed=seed, top_p=top_p or 0.0, top_k=top_k or 0, flags=flags)

    @staticmethod
    def _usage(u):
        return dict(prompt_tokens=u.prompt_tokens, completion_tokens=u.completion_tokens, prompt_secs=u.prompt_secs,
                    completion_secs=u.completion_secs, vision_secs=u.vision_secs)

    def generate(self, input_ids, data=None, max_tokens=1024, temperature=0.0, top_p=None, top_k=None, repeat_penalty=1.0,
                 repeat_last_n=64, seed=299792458, flags=0, reuse_prefix=False):
        """-> (generated ids, usage dict).  temperature < 1e-7: ArgMax; else the device sampler (TopK / TopKThenTopP / TopP /
        All exactly as get_logit_processor picks them from temperature, top_p, top_k).  reuse_prefix: keep this request's K/V
        and prefill only what follows the prefix shared with the cache (multi-turn chats; same tokens as without it)."""
        ids = self._ids(input_ids)
        mm, _keep = self._mm(data)
        if reuse_prefix:
            flags |= L.GEN_REUSE_PREFIX
        p = self._gen_params(max_tokens, temperature, top_p, top_k, repeat_penalty, repeat_last_n, seed, flags)
        cap = max(max_tokens, 1)
        out = (C.c_uint32 * cap)()
        n = C.c_size_t(0)
        u = L.Usage()
        self._check(self._lib.aha_b200_generate(self._h, ids.ctypes.data_as(C.POINTER(C.c_uint32)), ids.size,
                                                C.byref(mm) if mm is not None else None, C.byref(p), out, cap,
                                                C.byref(n), C.byref(u)))
        return [int(out[i]) for i in range(n.value)], self._usage(u)

    def _batch_request(self, input_ids, data, params):
        """-> (L.BatchRequest, keep): `keep` holds the buffers the request points into; it must outlive the call that reads it."""
        ids = self._ids(input_ids)
        mm, k = self._mm(data)
        req = L.BatchRequest(ids=ids.ctypes.data_as(C.POINTER(C.c_uint32)), seq_len=ids.size,
                             mm=C.pointer(mm) if mm is not None else None, params=params)
        return req, (ids, mm, k)

    def generate_batch(self, requests):
        """Static batching (aha_b200_generate_batch): requests = [dict(input_ids=..., data=None, max_tokens=..., temperature=..., top_p=...,
        top_k=..., repeat_penalty=..., repeat_last_n=..., seed=...), ...] (at most 8) decoded in lockstep on this handle.
        -> [(generated ids, usage dict), ...]: per request exactly what generate() returns for it alone."""
        n = len(requests)
        arr = (L.BatchRequest * n)()
        keep = []
        cap = 1
        for i, r in enumerate(requests):
            p = self._gen_params(r.get("max_tokens", 1024), r.get("temperature", 0.0), r.get("top_p"), r.get("top_k"),
                                 r.get("repeat_penalty", 1.0), r.get("repeat_last_n", 64), r.get("seed", 299792458), r.get("flags", 0))
            arr[i], k = self._batch_request(r["input_ids"], r.get("data"), p)
            keep.append(k)
            cap = max(cap, r.get("max_tokens", 1024))
        out = (C.c_uint32 * (n * cap))()
        n_out = (C.c_size_t * n)()
        us = (L.Usage * n)()
        self._check(self._lib.aha_b200_generate_batch(self._h, arr, n, out, cap, n_out, us))
        return [([int(out[i * cap + j]) for j in range(n_out[i])], self._usage(us[i])) for i in range(n)]

    # ---- continuous batching: requests join / leave a running batch between steps (aha_b200_batch_open / _add / _step / _close)
    def batch_open(self):
        self._check(self._lib.aha_b200_batch_open(self._h))

    def batch_add(self, input_ids, data=None, max_tokens=1024, temperature=0.0, top_p=None, top_k=None, repeat_penalty=1.0, repeat_last_n=64,
                  seed=299792458, flags=0):
        """Prefill one request into a free slot -> (slot, first token, finished)."""
        req, _keep = self._batch_request(input_ids, data,
                                         self._gen_params(max_tokens, temperature, top_p, top_k, repeat_penalty, repeat_last_n, seed, flags))
        slot, fin, tok = C.c_int32(-1), C.c_int32(0), C.c_uint32(0)
        u = L.Usage()
        self._check(self._lib.aha_b200_batch_add(self._h, C.byref(req), C.byref(slot), C.byref(tok), C.byref(fin), C.byref(u)))
        return int(slot.value), int(tok.value), bool(fin.value)

    def batch_step(self):
        """One decode step of every running request -> {slot: (token, finished)} (empty when nothing is running)."""
        toks = (C.c_uint32 * 8)()
        status = (C.c_int32 * 8)()
        n = C.c_size_t(0)
        self._check(self._lib.aha_b200_batch_step(self._h, toks, status, C.byref(n)))
        return {i: (int(toks[i]), status[i] == 2) for i in range(8) if status[i] != 0}

    def batch_close(self):
        self._check(self._lib.aha_b200_batch_close(self._h))

    def generate_stream(self, input_ids, on_token, data=None, max_tokens=1024, temperature=0.0, top_p=None, top_k=None,
                        repeat_penalty=1.0, repeat_last_n=64, seed=299792458, reuse_prefix=False):
        """generate_stream_generic: on_token(token, index) is called per generated token as its step completes; a truthy
        return value ends the request.  -> usage dict."""
        ids = self._ids(input_ids)
        mm, _keep = self._mm(data)
        p = self._gen_params(max_tokens, temperature, top_p, top_k, repeat_penalty, repeat_last_n, seed,
                             L.GEN_REUSE_PREFIX if reuse_prefix else 0)
        err = []

        def _cb(_user, token, index):
            try:
                return 1 if on_token(int(token), int(index)) else 0
            except Exception as e:  # never unwind through the C ABI
                err.append(e)
                return 1
        cb = L.TOKEN_CALLBACK(_cb)
        u = L.Usage()
        self._check(self._lib.aha_b200_generate_stream(self._h, ids.ctypes.data_as(C.POINTER(C.c_uint32)), ids.size,
                                                       C.byref(mm) if mm is not None else None, C.byref(p), cb, None, C.byref(u)))
        if err:
            raise err[0]
        return self._usage(u)

    def asr_generate(self, chunks, max_tokens=1024, temperature=0.0, top_p=None, seed=34562, on_token=None):
        """Qwen3AsrGenerateModel::generate: chunks = [(ids, mel), ...] (one AudioData each).  -> (ids of all chunks, usage)."""
        keep = []
        arr = (L.AsrChunk * len(chunks))()
        for i, (ids, mel) in enumerate(chunks):
            ids = self._ids(ids)
            mel = np.ascontiguousarray(mel, np.float32)
            keep += [ids, mel]
            arr[i].ids = ids.ctypes.data_as(C.POINTER(C.c_uint32))
            arr[i].seq_len = ids.size
            arr[i].input_features = L.make_desc(mel)
        p = self._gen_params(max_tokens, temperature, top_p, None, 1.0, 64, seed)
        cap = max(max_tokens, 1) * len(chunks)
        out = (C.c_uint32 * cap)()
        n = C.c_size_t(0)
        u = L.Usage()
        cb = L.TOKEN_CALLBACK((lambda _u, t, i: 1 if on_token(int(t), int(i)) else 0) if on_token else 0)
        self._check(self._lib.aha_b200_asr_generate(self._h, arr, len(chunks), C.byref(p), out, cap, C.byref(n), cb, None, C.byref(u)))
        return [int(out[i]) for i in range(n.value)], self._usage(u)

    def debug_sample(self, logits, context=(), draw_index=0, temperature=0.0, top_p=None, top_k=None, repeat_penalty=1.0,
                     repeat_last_n=64, seed=299792458):
        """The device sampler on a given logits row (tests)."""
        lg = np.ascontiguousarray(logits, np.float32).reshape(-1)
        ctx = np.ascontiguousarray(np.asarray(list(context), dtype=np.uint32))
        p = self._gen_params(1, temperature, top_p, top_k, repeat_penalty, repeat_last_n, seed)
        tok = C.c_uint32(0)
        self._check(self._lib.aha_b200_debug_sample(self._h, lg.ctypes.data_as(C.POINTER(C.c_float)), C.byref(p),
                                                    ctx.ctypes.data_as(C.POINTER(C.c_uint32)), ctx.size, int(draw_index), C.byref(tok)))
        return int(tok.value)

    # ------------------------------------------------------------------ Qwen3-Embedding / Qwen3-Reranker
    def embed(self, input_ids):
        """Qwen3Embedding::embed_one on token ids -> unit vector (hidden_size,) float32."""
        ids = self._ids(input_ids)
        out = np.empty(self.hidden_size, np.float32)
        self._check(self._lib.aha_b200_embed(self._h, ids.ctypes.data_as(C.POINTER(C.c_uint32)), ids.size,
                                             out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def rerank(self, query_ids, documents_ids):
        """Qwen3Reranker::rerank on token ids -> cosine scores (n_docs,) float32."""
        q = self._ids(query_ids)
        docs = [self._ids(d) for d in documents_ids]
        cat = np.ascontiguousarray(np.concatenate(docs)) if docs else np.zeros(0, np.uint32)
        lens = (C.c_size_t * max(len(docs), 1))(*[d.size for d in docs])
        out = np.empty(len(docs), np.float32)
        self._check(self._lib.aha_b200_rerank(self._h, q.ctypes.data_as(C.POINTER(C.c_uint32)), q.size,
                                              cat.ctypes.data_as(C.POINTER(C.c_uint32)), lens, len(docs),
                                              out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    # ------------------------------------------------------------------ frontends
    def mel_spectrogram(self, wave):
        wave = np.ascontiguousarray(wave, dtype=np.float32).reshape(-1)
        n_mels = self.config["thinker_config"]["audio_config"]["num_mel_bins"]
        cap = n_mels * (wave.size // 160 + 2)
        out = np.empty(cap, np.float32)
        nf = C.c_size_t(0)
        self._check(self._lib.aha_b200_mel_spectrogram(self._h, wave.ctypes.data_as(C.POINTER(C.c_float)), wave.size,
                                                       out.ctypes.data_as(C.POINTER(C.c_float)), cap, C.byref(nf)))
        return out[: n_mels * nf.value].reshape(n_mels, nf.value).copy()

    def image_patchify(self, img_u8_hwc):
        img = np.ascontiguousarray(img_u8_hwc, dtype=np.uint8)
        h, w, _ = img.shape
        vc = self.config["vision_config"]
        feat = vc["in_channels"] * vc["temporal_patch_size"] * vc["patch_size"] ** 2
        n = (h // vc["patch_size"]) * (w // vc["patch_size"])
        out = np.empty((n, feat), np.float32)
        grid = (C.c_uint32 * 3)()
        self._check(self._lib.aha_b200_image_patchify(self._h, img.ctypes.data_as(C.POINTER(C.c_uint8)), h, w,
                                                      out.ctypes.data_as(C.POINTER(C.c_float)), out.size, grid))
        return out, np.array([[grid[0], grid[1], grid[2]]], dtype=np.uint32)

    def video_preprocess(self, frames_u8_thwc):
        """Qwen3VLProcessor::process_videos for one clip: RGB24 frames (T, H, W, 3) at their video_smart_resize size ->
        (pixel_values_video, video_grid_thw)."""
        fr = np.ascontiguousarray(frames_u8_thwc, dtype=np.uint8)
        t, h, w, _ = fr.shape
        vc = self.config["vision_config"]
        tp = vc["temporal_patch_size"]
        feat = vc["in_channels"] * tp * vc["patch_size"] ** 2
        n = ((t + tp - 1) // tp) * (h // vc["patch_size"]) * (w // vc["patch_size"])
        out = np.empty((n, feat), np.float32)
        grid = (C.c_uint32 * 3)()
        self._check(self._lib.aha_b200_video_preprocess(self._h, fr.ctypes.data_as(C.POINTER(C.c_uint8)), t, h, w,
                                                        out.ctypes.data_as(C.POINTER(C.c_float)), out.size, grid))
        return out, np.array([[grid[0], grid[1], grid[2]]], dtype=np.uint32)

    def image_resize(self, img_u8_hwc, new_h, new_w):
        """DynamicImage::resize_exact(new_w, new_h, CatmullRom) on the GPU."""
        img = np.ascontiguousarray(img_u8_hwc, dtype=np.uint8)
        h, w, _ = img.shape
        out = np.empty((new_h, new_w, 3), np.uint8)
        self._check(self._lib.aha_b200_image_resize(self._h, img.ctypes.data_as(C.POINTER(C.c_uint8)), h, w, new_h, new_w,
                                                    out.ctypes.data_as(C.POINTER(C.c_uint8))))
        return out

    def resample(self, wave, orig_freq, new_freq):
        """resample_simple (audio_utils.rs:245-255) of a mono f32 waveform on the GPU: windowed-sinc polyphase filter, width 6, rolloff 0.99."""
        w = np.ascontiguousarray(wave, np.float32).reshape(-1)
        n = C.c_size_t(0)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        self._check(self._lib.aha_b200_resample(self._h, fp(w), w.size, int(orig_freq), int(new_freq), None, 0, C.byref(n)))
        out = np.empty(n.value, np.float32)
        self._check(self._lib.aha_b200_resample(self._h, fp(w), w.size, int(orig_freq), int(new_freq), fp(out), out.size, C.byref(n)))
        return out[:n.value]

    def image_preprocess(self, img_u8_hwc, min_pixels=65536, max_pixels=16777216):
        """Qwen3VLProcessor::process_img + process_vision_tensor for an image of any size -> (pixel_values, grid_thw)."""
        img = np.ascontiguousarray(img_u8_hwc, dtype=np.uint8)
        h, w, _ = img.shape
        vc = self.config["vision_config"]
        from . import processors
        rh, rw = processors.img_smart_resize(h, w, vc["patch_size"] * vc["spatial_merge_size"], min_pixels, max_pixels)
        feat = vc["in_channels"] * vc["temporal_patch_size"] * vc["patch_size"] ** 2
        out = np.empty(((rh // vc["patch_size"]) * (rw // vc["patch_size"]), feat), np.float32)
        grid = (C.c_uint32 * 3)()
        self._check(self._lib.aha_b200_image_preprocess(self._h, img.ctypes.data_as(C.POINTER(C.c_uint8)), h, w, min_pixels, max_pixels,
                                                        out.ctypes.data_as(C.POINTER(C.c_float)), out.size, grid))
        return out, np.array([[grid[0], grid[1], grid[2]]], dtype=np.uint32)

    # ------------------------------------------------------------------ introspection (tests / bench)
    def decode_steps(self, first_token, seqlen_offset, n_steps, want_tokens=True, timed=False):
        """n_steps graph replays with on-device token feedback; timed=True also returns the CUDA-event ms."""
        out = (C.c_uint32 * max(n_steps, 1))() if want_tokens else None
        ms = C.c_double(0.0)
        self._check(self._lib.aha_b200_decode_steps(self._h, int(first_token), int(seqlen_offset), int(n_steps), out,
                                                    C.byref(ms)))
        toks = [int(out[i]) for i in range(n_steps)] if want_tokens else None
        return (toks, ms.value) if timed else toks

    def bench_kernel(self, which, iters=200):
        ms = C.c_double(0.0)
        nb = C.c_uint64(0)
        self._check(self._lib.aha_b200_bench_kernel(self._h, which.encode(), int(iters), C.byref(ms), C.byref(nb)))
        return ms.value, int(nb.value)

    def debug_gemm(self, x, w16, bias=None, resid=None, impl=2, epi=0, act=0, iters=0):
        """y = epilogue(x @ w16.T + bias) through the library's GEMM (impl 1 = SIMT, 2 = tcgen05). -> (y, ms)"""
        x = np.ascontiguousarray(x, np.float32)
        w16 = np.ascontiguousarray(w16, np.float16)
        M, K = x.shape
        N = w16.shape[0]
        out = np.empty((M, N // 2 if epi == 3 else N), np.float32)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float)) if a is not None else None
        b = np.ascontiguousarray(bias, np.float32) if bias is not None else None
        r = np.ascontiguousarray(resid, np.float32) if resid is not None else None
        ms = C.c_double(0.0)
        self._check(self._lib.aha_b200_debug_gemm(self._h, impl, epi, act, M, N, K, fp(x), w16.ctypes.data_as(C.POINTER(C.c_uint16)),
                                                  fp(b), fp(r), fp(out), iters, C.byref(ms)))
        return out, ms.value

    def stream_ptr(self):
        return int(self._lib.aha_b200_stream(self._h) or 0)

    def stats(self):
        s = L.Stats()
        self._check(self._lib.aha_b200_get_stats(self._h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in L.Stats._fields_}

    def reset_stats(self):
        self._check(self._lib.aha_b200_reset_stats(self._h))

    def set_trace(self, on=True):
        self._check(self._lib.aha_b200_set_trace(self._h, 1 if on else 0))

    def debug_read(self, what, index, cap):
        out = np.empty(cap, np.float32)
        n = C.c_size_t(0)
        self._check(self._lib.aha_b200_debug_read(self._h, what.encode(), int(index),
                                                  out.ctypes.data_as(C.POINTER(C.c_float)), cap, C.byref(n)))
        return out[: n.value].copy()

    def close(self):
        if getattr(self, "_h", None):
            self._lib.aha_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
