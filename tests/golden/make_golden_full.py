"""Full-size golden fixtures: ONE oracle forward at each BASELINE.json shape (configs 2, 3, 4), run on the CPU of the
build container (`python tests/golden/make_golden_full.py [vl2|q0.6|asr0.6 ...]`, minutes each), outputs committed as
`tests/golden/full_<name>.<i>.npz` (one fixture is split over several files so that none reaches 1 MB; `load` joins them).  Weights and inputs are re-derived from the seeds by aha_b200.synth, so the fixtures hold
only what the GPU tests compare (tests/test_fullsize_gpu.py):

  * `prefill_logits` (V) of the last prompt token, full f32;
  * `forced` = the oracle's own greedy ids (teacher-forced on the GPU side), `step_logits_sub` = every 8th logit of each
    decode step, `step_top_ids` / `step_top_vals` = the 16 largest logits of each step, `step_last_logits` = the last step
    in full, `gaps` = top-1 - top-2 per position (ids are compared wherever gap > 10 x the measured logit error);
  * Qwen3-VL: f64 checksums (sum, sum |x|) of the four image-embed tensors (main + 3 deepstack) and a 64-row sample of each;
  * Qwen3-ASR: the same for the audio-tower output, and the oracle log-mel checksum.

The oracle is the checker, never the product (oracle/__init__.py)."""
import glob
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from aha_b200 import synth  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
N_STEPS = 8
SUB = 8
TOPK = 16
SHARD_BYTES = 900_000   # float32 logits hardly compress: a fixture file holds at most this many bytes of arrays

# the three workloads; tests/test_fullsize_gpu.py and bench.py build the same inputs from these
VL2_IMAGE, VL2_TEXT, Q06_PROMPT, ASR_SECONDS = synth.FULL_VL2_IMAGE, synth.FULL_VL2_TEXT, synth.FULL_Q06_PROMPT, synth.FULL_ASR_SECONDS


def save(name, out):
    """The arrays of `out`, in order, as name.0.npz, name.1.npz, ...: a new file whenever the next array would take the current one past
    SHARD_BYTES."""
    for f in glob.glob(os.path.join(OUT, f"{name}.*.npz")):
        os.remove(f)
    shard, size, i = {}, 0, 0
    for k, v in out.items():
        v = np.asarray(v)
        if shard and size + v.nbytes > SHARD_BYTES:
            np.savez_compressed(os.path.join(OUT, f"{name}.{i}.npz"), **shard)
            shard, size, i = {}, 0, i + 1
        shard[k] = v
        size += v.nbytes
    np.savez_compressed(os.path.join(OUT, f"{name}.{i}.npz"), **shard)


def load(name):
    """Every array of fixture `name` (all its files) in one dict."""
    paths = glob.glob(os.path.join(OUT, f"{name}.*.npz"))
    assert paths, f"tests/golden/{name}.*.npz is missing: run python tests/golden/make_golden_full.py"
    g = {}
    for p in paths:
        g.update(np.load(p))
    return g


def top2gap(l):
    p = np.partition(np.asarray(l).reshape(-1), -2)
    return float(p[-1] - p[-2])


def rows_sample(n, k=64):
    return np.unique(np.linspace(0, n - 1, k).astype(np.int64))


def tensor_summary(x, k=64):
    x = np.asarray(x, np.float32)
    r = rows_sample(x.shape[0], k)
    return dict(sum=np.float64(x.astype(np.float64).sum()), abs=np.float64(np.abs(x.astype(np.float64)).sum()), rows=r, sample=x[r].copy())


def decode_block(model, first_logits, S, out):
    """Greedy teacher chain: token_i = argmax(oracle logits_{i-1}); records per-step data into `out`."""
    forced, subs, tids, tvals, gaps = [], [], [], [], [top2gap(first_logits)]
    logits = first_logits
    last = None
    for i in range(N_STEPS):
        tok = int(np.argmax(logits))
        forced.append(tok)
        t0 = time.perf_counter()
        logits = model.forward_step(np.array([[tok]], np.uint32), S + i)[0, 0]
        print(f"    step {i}: token {tok}, {time.perf_counter() - t0:.2f} s, gap {top2gap(logits):.4f}", flush=True)
        subs.append(logits[::SUB].copy())
        idx = np.argsort(-logits, kind="stable")[:TOPK]
        tids.append(idx.astype(np.int64)); tvals.append(logits[idx].copy())
        gaps.append(top2gap(logits))
        last = logits
    out.update(forced=np.array(forced, np.uint32), step_logits_sub=np.stack(subs).astype(np.float32), step_top_ids=np.stack(tids),
               step_top_vals=np.stack(tvals).astype(np.float32), step_last_logits=last.astype(np.float32), gaps=np.array(gaps, np.float64),
               sub_stride=np.int64(SUB))


def vl2():
    from oracle.qwen3vl import Qwen3VLModel, process_image
    cfg = synth.get_config("qwen3vl", "vl2")
    t0 = time.perf_counter()
    w = synth.make_weights("qwen3vl", cfg, 0)
    print(f"  weights {time.perf_counter() - t0:.1f} s", flush=True)
    m = Qwen3VLModel(cfg, w, [cfg["text_config"]["eos_token_id"]])
    pv, grid = process_image(synth.synth_image(*VL2_IMAGE, seed=1))
    ids = synth.vl_prompt_ids(cfg, grid, VL2_TEXT)
    out = dict(grid=grid, n_ids=np.int64(len(ids)), ids_crc=np.int64(int(ids.astype(np.int64).sum())), pixel_sum=np.float64(pv.astype(np.float64).sum()))
    # run the tower once for its outputs, then the whole forward (the tower runs again inside: deterministic)
    t0 = time.perf_counter()
    emb, deep = m.visual.forward(pv, grid)
    out["vision_secs_cpu"] = np.float64(time.perf_counter() - t0)
    print(f"  vision tower {out['vision_secs_cpu']:.1f} s", flush=True)
    for i, t in enumerate([emb] + list(deep)):
        s = tensor_summary(t)
        out[f"embeds{i}_sum"], out[f"embeds{i}_abs"], out[f"embeds{i}_rows"], out[f"embeds{i}_sample"] = s["sum"], s["abs"], s["rows"], s["sample"]

    class _Cached:   # feed the tower outputs computed above instead of running the 8160-token ViT a second time
        def forward(self, *_):
            return emb, deep
    real = m.visual
    m.visual = _Cached()
    t0 = time.perf_counter()
    logits = m.forward_initial(ids.reshape(1, -1), 0, [pv, grid, None, None, None])[0, 0]
    m.visual = real
    out["prefill_secs_cpu"] = np.float64(time.perf_counter() - t0)
    print(f"  LLM prefill {out['prefill_secs_cpu']:.1f} s, rope_delta {m.rope_deltas}", flush=True)
    out["prefill_logits"] = logits.astype(np.float32)
    out["rope_delta"] = np.int64(m.rope_deltas)
    decode_block(m, logits, len(ids), out)
    save("full_vl2", out)


def q06():
    from oracle.qwen3 import Qwen3Model
    cfg = synth.get_config("qwen3", "q0.6")
    w = synth.make_weights("qwen3", cfg, 0)
    m = Qwen3Model(cfg, w, [cfg["eos_token_id"]])
    ids = synth.synth_text_ids(Q06_PROMPT, 151000, 21)
    out = dict(n_ids=np.int64(len(ids)), ids_crc=np.int64(int(ids.astype(np.int64).sum())))
    t0 = time.perf_counter()
    logits = m.forward_initial(ids.reshape(1, -1), 0)[0, 0]
    out["prefill_secs_cpu"] = np.float64(time.perf_counter() - t0)
    print(f"  prefill {out['prefill_secs_cpu']:.1f} s", flush=True)
    out["prefill_logits"] = logits.astype(np.float32)
    decode_block(m, logits, len(ids), out)
    save("full_q06", out)


def asr06():
    from oracle.audio import WhisperFeatureExtractor, get_feat_extract_output_lengths
    from oracle.qwen3_asr import Qwen3ASRModel
    cfg = synth.get_config("qwen3_asr", "asr0.6")
    w = synth.make_weights("qwen3_asr", cfg, 0)
    m = Qwen3ASRModel(cfg, w)
    wave = synth.synth_audio(ASR_SECONDS)
    t0 = time.perf_counter()
    mel = WhisperFeatureExtractor().call(wave[None], 16000)[0]
    out = dict(mel_secs_cpu=np.float64(time.perf_counter() - t0), mel_shape=np.array(mel.shape), mel_sum=np.float64(mel.astype(np.float64).sum()))
    n_tok = get_feat_extract_output_lengths(mel.shape[1])
    ids = synth.asr_prompt_ids(cfg, n_tok)
    out.update(n_ids=np.int64(len(ids)), ids_crc=np.int64(int(ids.astype(np.int64).sum())), n_audio_tokens=np.int64(n_tok))
    t0 = time.perf_counter()
    feat = m.audio.forward(mel)
    out["audio_secs_cpu"] = np.float64(time.perf_counter() - t0)
    print(f"  audio tower {out['audio_secs_cpu']:.1f} s -> {feat.shape}", flush=True)
    s = tensor_summary(feat)
    out["audio_sum"], out["audio_abs"], out["audio_rows"], out["audio_sample"] = s["sum"], s["abs"], s["rows"], s["sample"]
    t0 = time.perf_counter()
    logits = m.forward_initial(ids.reshape(1, -1), 0, [mel])[0, 0]
    out["prefill_secs_cpu"] = np.float64(time.perf_counter() - t0)
    out["prefill_logits"] = logits.astype(np.float32)
    decode_block(m, logits, len(ids), out)
    save("full_asr06", out)


if __name__ == "__main__":
    which = sys.argv[1:] or ["q0.6", "asr0.6", "vl2"]
    for name in which:
        t0 = time.perf_counter()
        print(f"[{name}]", flush=True)
        {"vl2": vl2, "q0.6": q06, "asr0.6": asr06}[name]()
        print(f"[{name}] done in {time.perf_counter() - t0:.1f} s", flush=True)
    for f in sorted(os.listdir(OUT)):
        if f.startswith("full_"):
            print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")
