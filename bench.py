#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: greedy decode tokens/s of Qwen3-VL-2B on a 1920x1080 image + 512-token
prompt, reported as absolute and as a fraction of the HBM roofline, with the reference's CPU path timed beside it.

A "step" is one greedy decode step (one token) of the hot path at ctx ~= prompt + i: ONE launch of the persistent
fused decode kernel, the token fed back on the device.  The ViT / audio tower + LLM prefill run before the timed
region and are reported in `config`.

  python bench.py --gpus N --steps K --warmup W        (N > 1: launched under torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                 (CPU port of the reference path on the host cores)
  python bench.py --preset q0.6 | asr0.6               (BASELINE.json configs 2 and 4; default vl2 = config 3, the metric)
  python bench.py ... --dump-outputs DIR               (also write the timed call's tokens and last-step logits as .npy)

value  = K / (CUDA-event time of K launches on the library's stream, max over ranks)   -- inputs resident in HBM, one timed window of K steps
e2e    = K / wall time of K aha_b200_forward_step calls (host token in, host argmax out every step)
N > 1:  `value` is N independent replicas (one request per GPU, no data-path collective, "scaling": "weak"); the SAME
        invocation then runs ONE request tensor-parallel over the N GPUs (heads / MLP rows sharded, partial sums exchanged
        as tagged packets over NVLink inside the fused kernel) and reports it under "tp" (strong scaling), after checking
        that its greedy tokens equal the single-GPU tokens ("tp_parity")."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "tokens/s"
METRICS = {"vl2": "decode tokens/sec Qwen3-VL-2B 1080p+512ctx", "vl8": "decode tokens/sec Qwen3-VL-8B 4x2048^2 images+512ctx", "q0.6": "decode tokens/sec Qwen3-0.6B 2k ctx",
           "asr0.6": "decode tokens/sec Qwen3-ASR-0.6B 30s audio", "tiny": "decode tokens/sec (tiny functional check)"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------- workloads
def workload(preset):
    """Synthetic inputs of BASELINE.json's configs (aha_b200.synth holds the shapes the golden fixtures use too)."""
    from aha_b200 import synth
    if preset == "vl2":    # config 3: 1088x1920 noise image (img_smart_resize(1080, 1920): the resize is the identity) + 512 text ids
        return dict(kind="qwen3vl", preset="vl2", image=synth.FULL_VL2_IMAGE, n_text=synth.FULL_VL2_TEXT, max_ctx=4096, max_patches=8192)
    if preset == "q0.6":   # config 2: Qwen3-0.6B text-only, 1920-token prompt, decode inside a 2k context
        return dict(kind="qwen3", preset="q0.6", n_text=synth.FULL_Q06_PROMPT, max_ctx=2560)
    if preset == "asr0.6":  # config 4: 30 s of synthetic 16 kHz audio -> log-mel (128, 3000) -> 390 audio tokens
        return dict(kind="qwen3_asr", preset="asr0.6", seconds=synth.FULL_ASR_SECONDS, max_ctx=1024, max_frames=3000)
    if preset == "vl8":    # config 5: Qwen3-VL-8B text stack, 4 images of 2048x2048 (4 x [1,128,128] patches = 16384 image tokens) + 512 text ids
        return dict(kind="qwen3vl", preset="vl8", image=(2048, 2048), n_images=4, n_text=512, max_ctx=18432, max_patches=65536)
    if preset == "tiny":   # functional check of this script on small shapes (not a bench line)
        return dict(kind="qwen3vl", preset="tiny", image=(256, 320), n_text=64, max_ctx=1024, max_patches=1024)
    raise SystemExit(f"unknown preset {preset}")


def text_config(kind, cfg):
    return cfg if kind == "qwen3" else (cfg["text_config"] if kind == "qwen3vl" else cfg["thinker_config"]["text_config"])


def prompt_len(wl, cfg):
    if wl["kind"] == "qwen3vl":
        h, w_ = wl["image"]
        k = wl.get("n_images", 1)
        n_img = (h // 16) * (w_ // 16) // cfg["vision_config"]["spatial_merge_size"] ** 2
        return k * (1 + n_img + 1) + wl["n_text"], k * n_img
    if wl["kind"] == "qwen3":
        return wl["n_text"], 0
    from aha_b200 import synth
    n_aud = synth.asr_audio_tokens(int(wl["seconds"] * 100))
    return 4 + 1 + n_aud + 1 + 4, n_aud


def describe(wl, cfg, S, n_mm):
    tc = text_config(wl["kind"], cfg)
    if wl["kind"] == "qwen3vl":
        h, w_ = wl["image"]
        name = "Qwen3-VL-8B shape (text H 4096 x 36 layers, 32/8 heads; vision tower 1152 / 16 heads = head_dim 72, 27 blocks)" if wl["preset"] == "vl8" else "Qwen3-VL-2B shape"
        return (f"{name} ({wl['preset']}), random-init fp16 weights (seed 0), {wl.get('n_images', 1)} synthetic {w_}x{h} image(s) "
                f"({n_mm} image tokens) + {wl['n_text']} text ids, greedy decode at ctx {S}+")
    if wl["kind"] == "qwen3":
        return f"Qwen3-0.6B shape, random-init fp16 weights (seed 0), {S} synthetic prompt ids, greedy decode at ctx {S}+ (2k context, paged KV)"
    return (f"Qwen3-ASR-0.6B shape, random-init fp16 weights (seed 0), {wl['seconds']:.0f} s synthetic 16 kHz audio -> log-mel on the GPU -> "
            f"{n_mm} audio tokens, greedy decode at ctx {S}+ (H={tc['hidden_size']})")


# ----------------------------------------------------------------------------------------------------- CPU arm
def build_cpu_decoder(kind, cfg, w, ctx, rope_delta):
    """The reference's CPU decode step (oracle port, numpy fp32 + BLAS): the text stack of the model with a synthetic KV
    cache of `ctx` tokens, so that the ViT / audio tower / prefill (minutes of CPU time) is not part of the sample."""
    tc = text_config(kind, cfg)
    lm = {"qwen3": "model.", "qwen3vl": "model.language_model.", "qwen3_asr": "thinker.model."}[kind]
    w32 = {k: (v.astype(np.float32) if k.startswith(lm) else v) for k, v in w.items()}
    if kind == "qwen3":
        from oracle.qwen3 import Qwen3Model
        m = Qwen3Model(cfg, w32)
        layers = m.layers
    elif kind == "qwen3vl":
        from oracle.qwen3vl import Qwen3VLModel
        m = Qwen3VLModel(cfg, w32)
        m.rope_deltas = rope_delta
        layers = m.text.layers
    else:
        from oracle.qwen3_asr import Qwen3ASRModel
        m = Qwen3ASRModel(cfg, w32)
        layers = m.layers
    rng = np.random.default_rng(0)
    for l in layers:
        shp = (1, tc["num_key_value_heads"], ctx, tc["head_dim"])
        l.attn.kv_cache = (rng.standard_normal(shp, dtype=np.float32), rng.standard_normal(shp, dtype=np.float32))
    return m


def cpu_decode_steps(m, ctx, n, tok=5):
    t0 = time.perf_counter()
    for i in range(n):
        logits = m.forward_step(np.array([[tok]]), ctx + i)
        tok = int(np.argmax(logits))
    return time.perf_counter() - t0


def cpu_threads_available():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_rate(kind, cfg, wts, S, rope_delta, steps, warmup, budget_s=25.0):
    """tokens/s of the CPU port with the BLAS pool size that is fastest on this box.  The pool is set EXPLICITLY with
    threadpoolctl (torchrun exports OMP_NUM_THREADS=1; a GEMV over 128 threads is slower than over 16), every candidate is
    timed on the same decode step, and the pool size that was actually in effect is read back and reported."""
    from threadpoolctl import threadpool_info, threadpool_limits
    avail = cpu_threads_available()
    m = build_cpu_decoder(kind, cfg, wts, S, rope_delta)
    cands = sorted({n for n in (1, 4, 8, 16, 32, 64, avail) if 1 <= n <= avail})
    sweep = {}
    best_n, best_dt = 1, None
    spent = 0.0
    for n in cands:
        with threadpool_limits(limits=n, user_api="blas"):
            got = max([d.get("num_threads", 0) for d in threadpool_info() if d.get("user_api") == "blas"] or [0])
            cpu_decode_steps(m, S, 1)                      # page the weights in / warm the pool
            dt = cpu_decode_steps(m, S + 1, 1)
        sweep[str(got or n)] = round(1.0 / dt, 4)
        spent += 2 * dt
        if best_dt is None or dt < best_dt:
            best_n, best_dt = (got or n), dt
        if spent > budget_s:
            break
    n_steps = steps if steps else int(min(max(budget_s / max(best_dt, 1e-3), 2), 24))
    with threadpool_limits(limits=best_n, user_api="blas"):
        actual = max([d.get("num_threads", 0) for d in threadpool_info() if d.get("user_api") == "blas"] or [best_n])
        if warmup:
            cpu_decode_steps(m, S, warmup)
        # exactly n_steps steps, timed in blocks of <= 8 so that a disturbed stretch of the (shared) host shows up as such in the record
        dt, blocks, done = 0.0, [], 0
        while done < n_steps:
            nblk = min(8, n_steps - done)
            d = cpu_decode_steps(m, S + warmup + done, nblk)
            blocks.append(round(nblk / d, 4)); dt += d; done += nblk
    return dict(value=n_steps / dt, ms_per_step=1e3 * dt / n_steps, threads=int(actual), steps=n_steps, sweep_tok_s_by_blas_threads=sweep,
                host_threads_available=avail, block_tok_s=blocks)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of this run, written to the real stdout (fd 1 is pointed at stderr for everything else so that
    library chatter such as NCCL's version banner can never pollute it)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def dump_outputs(out_dir, r):
    """The timed call's results: the greedy ids of its K steps (what decode_steps returns) and the logits of the last step
    (what forward_step returns for it), float64 / float32, under 1 MB together for every preset."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "decode_tokens.npy"), np.asarray(r["timed_tokens"], np.float64))
    np.save(os.path.join(out_dir, "last_step_logits.npy"), np.asarray(r["last_logits"], np.float32))


def ncu_traffic(preset):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE fused decode-step launch from the committed `ncu --set full`
    summary of this workload (a citation of a capture under profiles/, not a measurement of this run)."""
    for name in (f"r02_fused_decode_{preset}_ncu_summary.csv", "r02_fused_decode_ncu_summary.csv", "r01_fused_decode_final_ncu_summary.csv"):
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(p) or (preset != "vl2" and not name.startswith(f"r02_fused_decode_{preset}")):
            continue
        try:
            tot = 0.0
            for row in open(p).read().splitlines()[1:]:
                nm, unit, val = row.split(",")[:3]
                if nm in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(val) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[unit]
            if tot:
                return tot, "profiles/" + name
        except Exception:
            pass
    return None, None


# ----------------------------------------------------------------------------------------------------- GPU arm
def make_inputs(m, wl, cfg, synth):
    """-> (ids, MultiModalData list or None): the request of the workload, preprocessing on the GPU through the C ABI."""
    if wl["kind"] == "qwen3vl":
        pvs, grids = zip(*[m.image_patchify(synth.synth_image(wl["image"][0], wl["image"][1], 1 + i)) for i in range(wl.get("n_images", 1))])
        pv, grid = np.concatenate(pvs, 0), np.concatenate(grids, 0)
        return synth.vl_prompt_ids(cfg, grid, wl["n_text"]), [pv, grid, None, None, None]
    if wl["kind"] == "qwen3":
        return synth.synth_text_ids(wl["n_text"], 151000, 21), None
    mel = m.mel_spectrogram(synth.synth_audio(wl["seconds"]))
    return synth.asr_prompt_ids(cfg, synth.asr_audio_tokens(mel.shape[1])), [mel]


def measure_prefix_cache(m, synth, ids, data, n_new=32, n_gen=8):
    """The second turn of a conversation about the same inputs: turn 2 = turn 1's prompt + its answer + n_new new ids.
    cold = what the reference does (cache cleared per request: tower + full prefill again); warm = AHA_GEN_REUSE_PREFIX (only the new
    tokens are prefilled, the tower is skipped).  Time to first token = usage.prompt_secs; the greedy tokens must be identical."""
    a1, _ = m.generate(ids, data, max_tokens=n_gen, reuse_prefix=True)
    p2 = np.concatenate([ids, np.asarray(a1, np.uint32), synth.synth_text_ids(n_new, 151000, 77)]).astype(np.uint32)
    warm, uw = m.generate(p2, data, max_tokens=n_gen, reuse_prefix=True)
    hit = m.last_prefix_hit()
    m.clear_cache()
    cold, uc = m.generate(p2, data, max_tokens=n_gen)
    m.clear_cache()
    return {"turn2_prompt_tokens": int(len(p2)), "hit_tokens": int(hit), "ttft_cold_ms": 1e3 * uc["prompt_secs"], "ttft_warm_ms": 1e3 * uw["prompt_secs"],
            "tower_cold_ms": 1e3 * uc["vision_secs"], "tower_warm_ms": 1e3 * uw["vision_secs"], "tokens_equal": bool(warm == cold),
            "note": "new design (SURVEY 8f rank 4): the reference clears its KV cache after every request"}


def measure_batch(m, wl, synth, n_req=8, n_prompt=128, n_gen=64):
    """Static batching (aha_b200_generate_batch): n_req text-only requests decoded in lockstep on the same handle -- every weight is read once per
    step for all of them.  tokens/s = decode tokens of all requests / wall time of the lockstep loop (host sync per step included); the same
    requests one after the other through generate() give the single-stream rate beside it, and the ids of both must agree."""
    none = [None] * 5 if wl["kind"] == "qwen3vl" else None
    reqs = [dict(input_ids=synth.synth_text_ids(n_prompt + 3 * i, 151000, 500 + i), data=none, max_tokens=n_gen) for i in range(n_req)]
    m.generate_batch(reqs[:2])                                   # warm-up (buffers, kernel attributes)
    t0 = time.perf_counter()
    res = m.generate_batch(reqs)
    wall = time.perf_counter() - t0
    dec_tokens = sum(len(t) - 1 for t, _ in res)
    dec_secs = max(u["completion_secs"] for _, u in res)
    singles, single_secs = [], 0.0
    for r in reqs:
        t, u = m.generate(r["input_ids"], r["data"], max_tokens=n_gen)
        singles.append(t); single_secs += u["completion_secs"]
    return {"requests": n_req, "prompt_tokens": [int(len(r["input_ids"])) for r in reqs], "max_tokens": n_gen,
            "value": dec_tokens / dec_secs, "unit": UNIT, "ms_per_step": 1e3 * dec_secs / max(n_gen - 1, 1), "wall_s_incl_prefill": wall,
            "one_by_one_tokens_per_s": dec_tokens / single_secs, "speedup_vs_one_by_one": (dec_tokens / dec_secs) / (dec_tokens / single_secs),
            "tokens_equal": bool(all(a == b[0] for a, b in zip(singles, res))),
            "note": "new design (SURVEY 8f rank 4): the reference serves one request at a time; batched CUDA-core GEMV + per-sequence decode attention, one CUDA graph per batch composition"}


def measure(m, wl, cfg, synth, K, W, barrier, want_e2e=True, want_last_logits=False):
    """prefill once, then time K fused decode steps (device-resident) and K forward_step calls (e2e)."""
    ids, data = make_inputs(m, wl, cfg, synth)
    S = len(ids)
    toks, usage = m.generate(ids, data, max_tokens=4)           # request 1 through the public generate(): warms everything up
    toks2, usage = m.generate(ids, data, max_tokens=4)
    assert toks == toks2, "greedy decode is not deterministic"
    m.forward_initial(ids, 0, data, want_logits=False)
    tok = m.last_argmax
    rope_delta = int(m.debug_read("rope_delta", 0, 1)[0]) if wl["kind"] == "qwen3vl" else 0
    warm = m.decode_steps(tok, S, W)
    m.reset_stats()
    barrier()
    wall0 = time.perf_counter()
    out, ms = m.decode_steps(warm[-1], S + W, K, timed=True)
    barrier()
    wall_value = time.perf_counter() - wall0
    st = m.stats()
    res = dict(S=S, usage=usage, rope_delta=rope_delta, ms=ms, tokens=[tok] + list(warm) + list(out), timed_tokens=out, wall_value=wall_value,
               launches=st["kernel_launches"], stats=st)
    if want_last_logits:
        # the last timed step once more, on the cache it saw (before the e2e loop below overwrites those positions): the same kernel on the
        # same inputs, so these are the logits that step computed, as forward_step hands them to a caller
        prev = out[-2] if K > 1 else warm[-1]
        res["last_logits"] = m.forward_step(np.array([prev], np.uint32), S + W + K - 1)
        assert m.last_argmax == out[-1], "re-running the last timed step gave a different token"
    if want_e2e:
        t = out[-1]
        barrier()
        e0 = time.perf_counter()
        for i in range(K):
            m.forward_step(np.array([t], np.uint32), S + W + i, want_logits=False)
            t = m.last_argmax
        barrier()
        res["e2e_s"] = time.perf_counter() - e0
        n = min(K, 32)
        e0 = time.perf_counter()
        for i in range(n):   # the same with the full logits row returned to the host every step (what the reference's sampler consumes)
            m.forward_step(np.array([t], np.uint32), S + W + i, want_logits=True)
        res["e2e_logits_s"] = (time.perf_counter() - e0) / n
    res["inputs"] = (ids, data)
    return res


def extra_records(m, wl, synth, r):
    """The two records beyond the metric (KV reuse, static batching): measured last on the handle, each on its own, so that nothing they do can
    reach the numbers of the line (already taken) -- a failure becomes an `error` entry."""
    ids, data = r["inputs"]
    try:
        r["prefix_cache"] = measure_prefix_cache(m, synth, ids, data)
    except Exception as e:
        r["prefix_cache"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if wl["kind"] in ("qwen3", "qwen3vl"):
        try:
            r["batch"] = measure_batch(m, wl, synth)
        except Exception as e:
            r["batch"] = {"error": f"{type(e).__name__}: {e}"[:300]}


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--preset", default=os.environ.get("AHA_BENCH_PRESET", "vl2"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tp", action="store_true", help="N > 1: skip the tensor-parallel (strong scaling) arm")
    ap.add_argument("--decode-impl", type=int, default=int(os.environ.get("AHA_DECODE_IMPL", "0")))
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last of them computed to DIR/*.npy "
                                                              "(rank 0; seeded inputs, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm")
    K, W = args.steps, max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = workload(args.preset)
    metric = METRICS[args.preset]

    from aha_b200 import synth
    cfg = synth.get_config(wl["kind"], wl["preset"])
    tc = text_config(wl["kind"], cfg)
    S, n_mm = prompt_len(wl, cfg)
    config = {"workload": describe(wl, cfg, S, n_mm), "prompt_tokens": S, "kv_dtype": "f32", "weight_dtype": "f16", "accumulate": "f32", "batch": 1,
              "l2_policy": "inputs larger than L2 (the fp16 weights of the model are streamed once per step; 126 MB L2)",
              "parallelism": "single GPU" if world == 1 else f"{world} independent replicas (one request per GPU, no data-path collective); "
                                                                f"the tensor-parallel run of ONE request over the {world} GPUs is reported under 'tp'"}

    # --------------------------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        log("[reference] generating weights ...")
        wts = synth.make_weights(wl["kind"], cfg, 0)
        delta = 0
        if wl["kind"] == "qwen3vl":
            from oracle.qwen3vl import get_rope_index
            grid = np.array([[1, wl["image"][0] // 16, wl["image"][1] // 16]])
            _, delta = get_rope_index(synth.vl_prompt_ids(cfg, grid, wl["n_text"]), grid, cfg)
        r = cpu_reference_rate(wl["kind"], cfg, wts, S, delta, K, W)
        sample = (f"{r['steps']} greedy decode steps of the oracle port (numpy fp32 + OpenBLAS, pool set to {r['threads']} threads = the fastest of the sweep "
                  f"{r['sweep_tok_s_by_blas_threads']} tok/s by pool size; {r['host_threads_available']} host threads available) of the reference's text stack at "
                  f"ctx {S}+ with a synthetic KV cache (tok/s per block of <= 8 steps: {r['block_tok_s']}); tower + prefill not in the sample; the reference itself (Rust/Candle) cannot be built here (no cargo/rustc)")
        line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": sample},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    # --------------------------------------------------------------------------------- B200 arm
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local_rank)

    from aha_b200 import B200Model, dist_util
    t0 = time.time()
    wts = synth.make_weights(wl["kind"], cfg, 0)
    log(f"[rank {rank}] weights generated in {time.time() - t0:.1f}s")
    kw = dict(eos_ids=[], device=local_rank, max_ctx=wl["max_ctx"], max_prefill=wl["max_ctx"], decode_impl=args.decode_impl)
    if "max_patches" in wl:
        kw["max_patches"] = wl["max_patches"]
    if "max_frames" in wl:
        kw["max_frames"] = wl["max_frames"]
    t0 = time.time()
    m = B200Model(wl["kind"], cfg, wts, **kw)
    log(f"[rank {rank}] model created in {time.time() - t0:.1f}s")
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    r = measure(m, wl, cfg, synth, K, W, barrier, want_last_logits=args.dump_outputs is not None)
    clocks = sampler.stop()
    assert r["S"] == S
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, r)
    usage, st = r["usage"], r["stats"]
    log(f"[rank {rank}] prefill {usage['prompt_secs']:.3f}s (tower {usage['vision_secs']:.3f}s); decode {r['ms'] / K:.4f} ms/step")

    # ---- per-op twin kernels timed alone (where the step's bytes go), CUDA events
    peak, peak_src = measured_peaks()
    kernels = {}
    for name in ("gemv_gate_up", "gemv_down", "gemv_qkv", "gemv_o", "gemv_lm_head"):
        kms, kb = m.bench_kernel(name, 280 if name != "gemv_lm_head" else 20)
        kernels[name] = {"avg_us": kms * 1e3, "bytes": kb, "gbps": kb / (kms * 1e-3) / 1e9}
    fused = st["kernels_per_decode_step"] == 1
    dev = f"cuda:{local_rank}"
    value, max_ms = dist_util.aggregate_throughput(K, r["ms"], world, dist, dev)        # units of all ranks / slowest rank
    e2e_val, _ = dist_util.aggregate_throughput(K, r["e2e_s"] * 1e3, world, dist, dev)
    step_ms = max_ms / K
    avg_ctx = S + W + (K - 1) / 2.0 + 1
    step_bytes = st["decode_bytes_per_step_fixed"] + st["kv_bytes_per_token"] * (avg_ctx + 1)
    kv_read = st["kv_bytes_per_token"] * avg_ctx
    single_tokens = r["tokens"]
    if world == 1:
        extra_records(m, wl, synth, r)
    m.close()
    del m

    # ---- N > 1: the same request tensor-parallel over the N GPUs (strong scaling), tokens checked against the single-GPU run
    tp_rec = None
    if world > 1 and not args.no_tp:
      try:
          from aha_b200 import nccl_unique_id
          uid = [nccl_unique_id() if rank == 0 else None]
          dist.broadcast_object_list(uid, src=0)
          mt = B200Model(wl["kind"], cfg, wts, tp_rank=rank, tp_world=world, tp_unique_id=uid[0], **kw)
          rt = measure(mt, wl, cfg, synth, K, W, barrier, want_e2e=True)
          tp_ms = dist_util.reduce_max(rt["ms"], dist, dev)
          tp_e2e = dist_util.reduce_max(rt["e2e_s"], dist, dev)
          n_cmp = min(len(single_tokens), len(rt["tokens"]))
          same = [int(a == b) for a, b in zip(single_tokens[:n_cmp], rt["tokens"][:n_cmp])]
          first_diff = same.index(0) if 0 in same else None
          tl = [None] * world
          dist.all_gather_object(tl, rt["tokens"])
          ranks_agree = all(t == tl[0] for t in tl)
          stt = rt["stats"]
          tp_bytes = stt["decode_bytes_per_step_fixed"] + stt["kv_bytes_per_token"] * (avg_ctx + 1)
          tp_rec = {"value": K / (tp_ms * 1e-3), "unit": UNIT, "ms_per_step": tp_ms / K, "scaling": "strong", "n_gpus": world,
                    "e2e": K / tp_e2e, "kernels_per_step": stt["kernels_per_decode_step"],
                    "exchange": f"{2 * tc['num_hidden_layers']} one-shot all-reduces per step inside the fused kernel: every rank stores its partial sums as tagged 8-byte "
                                f"packets into every peer over NVLink ({tc['hidden_size'] * 8} B per peer per exchange) and sums the {world} vectors in rank order; no NCCL call on the decode path",
                    "bytes_per_rank_per_step": tp_bytes, "gbps_per_rank": tp_bytes / (tp_ms / K * 1e-3) / 1e9,
                    "prefill_secs": rt["usage"]["prompt_secs"],
                    "tp_parity": ("ok" if first_diff is None else f"first differing greedy token at position {first_diff} of {n_cmp} (fp32 summation order differs between TP sizes)"),
                    "ranks_agree": bool(ranks_agree), "speedup_vs_1gpu": (K / (tp_ms * 1e-3)) / (K / (r["ms"] * 1e-3))}
          assert ranks_agree, "tensor-parallel ranks produced different tokens"
          mt.close()
      except Exception as e:   # the weak-scaling line must survive a failure of the strong-scaling arm
        log(f"[rank {rank}] tensor-parallel arm failed: {type(e).__name__}: {e}")
        tp_rec = {"error": f"{type(e).__name__}: {e}"[:400]}

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log("[rank 0] timing the CPU port of the reference path ...")
        c = cpu_reference_rate(wl["kind"], cfg, wts, S, r["rope_delta"], 0, 0)
        cpu_base = {"value": c["value"], "unit": UNIT, "cores": c["threads"], "kind": "port",
                    "sample": f"{c['steps']} greedy decode steps of the oracle port (numpy fp32 + OpenBLAS, {c['threads']} threads = fastest of the sweep "
                              f"{c['sweep_tok_s_by_blas_threads']}; {c['host_threads_available']} host threads available) of the text stack at ctx {S}+ with a synthetic "
                              f"KV cache (tower + prefill excluded; tok/s per block of <= 8 steps: {c['block_tok_s']}); Rust/Candle reference not buildable here"}

    if rank == 0:
        traffic, traffic_src = ncu_traffic(args.preset)
        step_gbps = step_bytes / (step_ms * 1e-3) / 1e9
        roof = ({"bound": "hbm", "kernel": "decode_step_fused_kernel (the whole decode step: one launch per token)",
                 "achieved": step_gbps, "peak": peak, "unit": "GB/s", "frac": step_gbps / peak, "peak_source": peak_src,
                 "traffic": traffic, "traffic_source": traffic_src, "bytes_per_launch": step_bytes, "avg_launch_us": step_ms * 1e3,
                 "algorithmic_bytes": "fp16 weights of every layer + lm_head read once + fp32 KV of the context read once + the new token's KV written (DESIGN.md 4)",
                 "per_op_kernels": kernels}
                if fused else
                {"bound": "hbm", "kernel": "gemv_kernel<rmsnorm, swiglu> (gate/up projection)", "achieved": kernels["gemv_gate_up"]["gbps"],
                 "peak": peak, "unit": "GB/s", "frac": kernels["gemv_gate_up"]["gbps"] / peak, "peak_source": peak_src, "traffic": None,
                 "traffic_source": None, "bytes_per_launch": kernels["gemv_gate_up"]["bytes"], "avg_launch_us": kernels["gemv_gate_up"]["avg_us"],
                 "per_op_kernels": kernels})
        roof["step"] = {"bytes": step_bytes, "gbps": step_gbps, "frac_full": step_gbps / peak, "roofline_full_tok_s": peak * 1e9 / step_bytes,
                        "roofline_kv_tok_s": peak * 1e9 / kv_read,
                        "frac_vs_fp16_kv_bytes": (st["decode_bytes_per_step_fixed"] + 0.5 * st["kv_bytes_per_token"] * (avg_ctx + 1)) / (step_ms * 1e-3) / 1e9 / peak}
        line = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": step_ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 (fp16 weights, fp32 activations/accumulate/KV)", "data": "synthetic",
                "config": dict(config, prefill_secs=usage["prompt_secs"], tower_secs=usage["vision_secs"], kernels_per_step=st["kernels_per_decode_step"],
                               value_wall_check_s=r["wall_value"]),
                "clocks": clocks, "gpu_launches": int(r["launches"]),
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": 16, "d2h_bytes_per_step": 4,
                        "with_logits_d2h_tokens_per_s": 1.0 / r["e2e_logits_s"], "logits_bytes": 4 * tc["vocab_size"]},
                "roofline": roof,
                "decode_impl": ("fused persistent kernel, phases exchange tagged packets (no grid barrier)" if fused and args.decode_impl == 2 else
                                "fused persistent kernel, grid barriers between phases" if fused else "per-op kernels (CUDA graph)"),
                "cpu_baseline": cpu_base}
        if tp_rec is not None:
            line["tp"] = tp_rec
        if r.get("prefix_cache") is not None:
            line["prefix_cache"] = r["prefix_cache"]
        if r.get("batch") is not None:
            line["batch"] = r["batch"]
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
