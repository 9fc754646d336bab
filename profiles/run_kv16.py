"""What an fp16 KV cache would cost in accuracy at BASELINE.json's own shapes (VERDICT r1 item 9: "a decision, not a guess").

Run with the measurement build of the library in place (nvcc ... -DAHA_KV_ROUND_FP16 -> variants/kv16.so, copied over
aha_b200/libaha_b200.so for the duration of this script): every K / V value is rounded to fp16 on its way into the cache, the rest of the
path is unchanged.  Prints max |dlogit| against the full-size oracle goldens (tests/golden/full_*.npz) for prefill + 8 teacher-forced
decode steps, and how many greedy ids still match.  With the default build the same script reproduces the fp32-KV numbers of DESIGN.md."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from aha_b200 import B200Model, synth   # noqa: E402
from make_golden_full import load       # noqa: E402


def chain(m, g, S, prefill_logits):
    worst = float(np.abs(prefill_logits - g["prefill_logits"]).max())
    forced, sub = g["forced"], int(g["sub_stride"])
    ids_ok = int(int(np.argmax(prefill_logits)) == int(forced[0]))
    for i in range(len(forced)):
        l = m.forward_step(np.array([forced[i]], np.uint32), S + i)[0, 0]
        e = float(np.abs(l[::sub] - g["step_logits_sub"][i]).max())
        e = max(e, float(np.abs(l[g["step_top_ids"][i]] - g["step_top_vals"][i]).max()))
        worst = max(worst, e)
        ids_ok += int(m.last_argmax == int(g["step_top_ids"][i][0]))
    return worst, ids_ok, len(forced) + 1, float(g["gaps"].min())


def main():
    out = {}
    g = load("full_q06")
    cfg = synth.get_config("qwen3", "q0.6")
    m = B200Model("qwen3", cfg, synth.make_weights("qwen3", cfg, 0), eos_ids=[], max_ctx=2048, max_prefill=2048)
    ids = synth.synth_text_ids(synth.FULL_Q06_PROMPT, 151000, 21)
    out["q0.6 (1920-token prompt)"] = chain(m, g, len(ids), m.forward_initial(ids, 0)[0, 0])
    m.close()

    g = load("full_vl2")
    cfg = synth.get_config("qwen3vl", "vl2")
    m = B200Model("qwen3vl", cfg, synth.make_weights("qwen3vl", cfg, 0), eos_ids=[], max_ctx=4096, max_prefill=4096, max_patches=8192)
    pv, grid = m.image_patchify(synth.synth_image(*synth.FULL_VL2_IMAGE, seed=1))
    ids = synth.vl_prompt_ids(cfg, grid, synth.FULL_VL2_TEXT)
    out["vl2 (1080p image + 512 ids)"] = chain(m, g, len(ids), m.forward_initial(ids, 0, [pv, grid, None, None, None])[0, 0])
    m.close()

    g = load("full_asr06")
    cfg = synth.get_config("qwen3_asr", "asr0.6")
    m = B200Model("qwen3_asr", cfg, synth.make_weights("qwen3_asr", cfg, 0), eos_ids=[], max_ctx=1024, max_frames=3000)
    mel = m.mel_spectrogram(synth.synth_audio(synth.FULL_ASR_SECONDS))
    ids = synth.asr_prompt_ids(cfg, int(g["n_audio_tokens"]))
    out["asr0.6 (30 s audio)"] = chain(m, g, len(ids), m.forward_initial(ids, 0, [mel])[0, 0])
    m.close()

    for k, (worst, ok, n, gap) in out.items():
        print(f"{k}: max |dlogit| vs the fp32 oracle golden = {worst:.3e}; greedy ids equal {ok}/{n} (smallest top-1/top-2 gap {gap:.3f})")
    print(json.dumps({k: {"max_abs_dlogit": v[0], "ids_equal": v[1], "ids": v[2], "min_gap": v[3]} for k, v in out.items()}))


if __name__ == "__main__":
    main()
