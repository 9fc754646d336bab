"""BASELINE.json's full sizes, checked through size-independent properties (the oracle would need minutes per
forward at these shapes):
  * cache consistency: forward_initial(ids[:S]) followed by forward_step(ids[S]) must give the logits of
    forward_initial(ids[:S+1]) -- ties the prefill kernels (tcgen05 GEMM, flash attention, paged KV write) to the
    decode kernels (fused step / per-op) on the same weights;
  * the two decode implementations agree; greedy decode is deterministic across requests;
  * GPU log-mel of 30 s of audio equals the oracle's (cheap on the CPU), 3000 frames -> 390 audio tokens;
  * 1088x1920 image -> 8160 patches -> 2040 image tokens, rope_delta = -1980 (closed forms from the source)."""
import numpy as np
import pytest

from conftest import TOL
from aha_b200 import B200Model, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vl2():
    cfg = synth.get_config("qwen3vl", "vl2")
    w = synth.make_weights("qwen3vl", cfg, 0)
    m = B200Model("qwen3vl", cfg, w, eos_ids=[], max_ctx=4096, max_prefill=4096, max_patches=8192)
    m1 = B200Model("qwen3vl", cfg, w, eos_ids=[], max_ctx=4096, max_prefill=4096, max_patches=8192, decode_impl=1)
    del w
    yield cfg, m, m1
    m.close(); m1.close()


def test_vl2_1080p_cache_consistency_and_closed_forms(vl2):
    cfg, m, m1 = vl2
    img = synth.synth_image(1088, 1920, 1)
    pv, grid = m.image_patchify(img)
    assert pv.shape == (8160, 1536) and grid.tolist() == [[1, 68, 120]]
    ids = synth.vl_prompt_ids(cfg, grid, 512)
    assert int((ids == cfg["image_token_id"]).sum()) == 2040 and len(ids) == 2554
    data = [pv, grid, None, None, None]
    S = len(ids) - 1
    # request A: prefill S tokens, then one decode step with token S (fused kernel)
    m.forward_initial(ids[:S], 0, data, want_logits=False)
    assert int(m.debug_read("rope_delta", 0, 1)[0]) == -1980
    a = m.forward_step(ids[S:S + 1], S)[0, 0]
    # request B: prefill all S+1 tokens
    m.clear_cache()
    b = m.forward_initial(ids, 0, data)[0, 0]
    err = float(np.abs(a - b).max())
    assert err <= TOL, err
    # per-op decode implementation on the same request
    m1.forward_initial(ids[:S], 0, data, want_logits=False)
    c = m1.forward_step(ids[S:S + 1], S)[0, 0]
    assert float(np.abs(c - b).max()) <= TOL
    print(f"\nVL2 1080p: |prefill(S)+step - prefill(S+1)| = {err:.2e} (fused), {float(np.abs(c - b).max()):.2e} (per-op); logit std {b.std():.3f}")


def test_vl2_greedy_decode_is_deterministic_and_impls_agree(vl2):
    cfg, m, m1 = vl2
    ids = synth.synth_text_ids(600, 151000, 4)
    m.clear_cache(); m1.clear_cache()
    t0, _ = m.generate(ids, [None] * 5, max_tokens=24)
    t1, _ = m.generate(ids, [None] * 5, max_tokens=24)
    t2, _ = m1.generate(ids, [None] * 5, max_tokens=24)
    assert t0 == t1
    assert t0 == t2


def test_q06_config2_2k_context():
    """config 2: Qwen3-0.6B shape, 1920-token prompt + decode to ctx 2048 (fp32 KV, see DESIGN.md section 2)."""
    cfg = synth.get_config("qwen3", "q0.6")
    w = synth.make_weights("qwen3", cfg, 0)
    m = B200Model("qwen3", cfg, w, eos_ids=[], max_ctx=2048, max_prefill=2048)
    del w
    try:
        ids = synth.synth_text_ids(1921, 151000, 9)
        m.forward_initial(ids[:1920], 0, want_logits=False)
        a = m.forward_step(ids[1920:1921], 1920)[0, 0]
        m.clear_cache()
        b = m.forward_initial(ids, 0)[0, 0]
        assert float(np.abs(a - b).max()) <= TOL
        m.clear_cache()
        toks, usage = m.generate(ids[:1920], max_tokens=128)       # runs to ctx 2048 exactly
        assert len(toks) == 128 and usage["prompt_tokens"] == 1920
        with pytest.raises(Exception, match="max_ctx"):
            m.generate(ids[:1921], max_tokens=128)
    finally:
        m.close()


def test_asr06_config4_30s_audio():
    from oracle.audio import WhisperFeatureExtractor, get_feat_extract_output_lengths
    cfg = synth.get_config("qwen3_asr", "asr0.6")
    w = synth.make_weights("qwen3_asr", cfg, 0)
    m = B200Model("qwen3_asr", cfg, w, eos_ids=[], max_ctx=1024, max_frames=3000)
    del w
    try:
        wave = synth.synth_audio(30.0)
        mel = m.mel_spectrogram(wave)
        assert mel.shape == (128, 3000)
        want = WhisperFeatureExtractor().call(wave[None], 16000)[0]
        assert float(np.abs(mel - want).max()) <= 1e-3
        n_tok = get_feat_extract_output_lengths(3000)
        assert n_tok == 390
        ids = synth.asr_prompt_ids(cfg, n_tok, n_text=9)
        S = len(ids) - 1
        m.forward_initial(ids[:S], 0, [mel], want_logits=False)
        assert m.debug_read("audio_embeds", 0, 390 * 1024).size == 390 * 1024
        a = m.forward_step(ids[S:S + 1], S)[0, 0]
        m.clear_cache()
        b = m.forward_initial(ids, 0, [mel])[0, 0]
        assert float(np.abs(a - b).max()) <= TOL
    finally:
        m.close()


# ----------------------------------------------------------------------------------------------------------------------
# Parity at BASELINE.json's own shapes: the CUDA path against ONE oracle forward per configuration, computed on the CPU of
# the build container by tests/golden/make_golden_full.py and committed as tests/golden/full_*.npz (weights and inputs are
# re-derived from the same seeds here).  Tolerance: north_star's 1e-3 on every logit; greedy ids must equal the oracle's
# wherever the oracle's top-1/top-2 gap exceeds 10x the measured error.
import sys

from conftest import GOLDEN

sys.path.insert(0, GOLDEN)
from make_golden_full import load as _golden  # noqa: E402


def _check_chain(m, g, S, prefill_logits, label):
    """prefill logits, then the oracle's greedy ids teacher-forced for 8 steps; returns the largest |dlogit| seen."""
    worst = float(np.abs(prefill_logits - g["prefill_logits"]).max())
    assert worst <= TOL, f"{label}: prefill logits differ from the oracle by {worst}"
    gaps, forced, sub = g["gaps"], g["forced"], int(g["sub_stride"])
    ids_checked = 0
    if gaps[0] > 10 * max(worst, 1e-6):
        assert int(np.argmax(prefill_logits)) == int(forced[0]), f"{label}: first greedy id differs"
        ids_checked += 1
    n = len(forced)
    for i in range(n):
        l = m.forward_step(np.array([forced[i]], np.uint32), S + i)[0, 0]
        e = float(np.abs(l[::sub] - g["step_logits_sub"][i]).max())
        e = max(e, float(np.abs(l[g["step_top_ids"][i]] - g["step_top_vals"][i]).max()))
        if i == n - 1:
            e = max(e, float(np.abs(l - g["step_last_logits"]).max()))
        assert e <= TOL, f"{label}: decode step {i} differs from the oracle by {e}"
        worst = max(worst, e)
        if gaps[i + 1] > 10 * max(e, 1e-6):
            assert m.last_argmax == int(g["step_top_ids"][i][0]), f"{label}: greedy id at step {i} differs"
            ids_checked += 1
    print(f"\n{label}: max |dlogit| vs the full-size oracle golden = {worst:.2e} over prefill + {n} steps; {ids_checked}/{n + 1} greedy ids compared (min gap {gaps.min():.3f})")
    return worst


@pytest.mark.parametrize("impl", [0, 1])
def test_vl2_1080p_matches_the_full_size_oracle_golden(vl2, impl):
    cfg, m0, m1 = vl2
    m = m1 if impl == 1 else m0
    g = _golden("full_vl2")
    VL2_IMAGE, VL2_TEXT = synth.FULL_VL2_IMAGE, synth.FULL_VL2_TEXT
    m.clear_cache()
    pv, grid = m.image_patchify(synth.synth_image(*VL2_IMAGE, seed=1))
    assert grid.tolist() == g["grid"].tolist() and abs(float(pv.astype(np.float64).sum()) - float(g["pixel_sum"])) <= 1e-3 * abs(float(g["pixel_sum"])) + 1.0
    ids = synth.vl_prompt_ids(cfg, grid, VL2_TEXT)
    assert len(ids) == int(g["n_ids"]) and int(ids.astype(np.int64).sum()) == int(g["ids_crc"])
    logits = m.forward_initial(ids, 0, [pv, grid, None, None, None])[0, 0]
    assert int(m.debug_read("rope_delta", 0, 1)[0]) == int(g["rope_delta"])
    ne = 2040 * 2048
    for i in range(4):   # the four image-embed tensors (main merger + 3 deepstack): sampled rows + checksums
        t = m.debug_read("image_embeds", i, ne).reshape(2040, 2048)
        e = float(np.abs(t[g[f"embeds{i}_rows"]] - g[f"embeds{i}_sample"]).max())
        assert e <= TOL, f"image_embeds[{i}] differs from the oracle by {e}"
        assert abs(float(np.abs(t.astype(np.float64)).sum()) - float(g[f"embeds{i}_abs"])) <= 1e-4 * float(g[f"embeds{i}_abs"])
    _check_chain(m, g, len(ids), logits, f"VL2 1080p+512 (decode_impl={impl})")


@pytest.mark.parametrize("impl", [0, 1, 2])
def test_q06_2k_matches_the_full_size_oracle_golden(impl):
    Q06_PROMPT = synth.FULL_Q06_PROMPT
    g = _golden("full_q06")
    cfg = synth.get_config("qwen3", "q0.6")
    w = synth.make_weights("qwen3", cfg, 0)
    m = B200Model("qwen3", cfg, w, eos_ids=[], max_ctx=2048, max_prefill=2048, decode_impl=impl)
    del w
    try:
        ids = synth.synth_text_ids(Q06_PROMPT, 151000, 21)
        assert int(ids.astype(np.int64).sum()) == int(g["ids_crc"])
        logits = m.forward_initial(ids, 0)[0, 0]
        _check_chain(m, g, len(ids), logits, f"Q0.6 1920-token prompt (decode_impl={impl})")
    finally:
        m.close()


def test_asr06_30s_matches_the_full_size_oracle_golden():
    ASR_SECONDS = synth.FULL_ASR_SECONDS
    g = _golden("full_asr06")
    cfg = synth.get_config("qwen3_asr", "asr0.6")
    w = synth.make_weights("qwen3_asr", cfg, 0)
    m = B200Model("qwen3_asr", cfg, w, eos_ids=[], max_ctx=1024, max_frames=3000)
    del w
    try:
        mel = m.mel_spectrogram(synth.synth_audio(ASR_SECONDS))
        assert list(mel.shape) == g["mel_shape"].tolist()
        assert abs(float(mel.astype(np.float64).sum()) - float(g["mel_sum"])) <= 1e-4 * abs(float(g["mel_sum"])) + 1.0
        ids = synth.asr_prompt_ids(cfg, int(g["n_audio_tokens"]))
        assert int(ids.astype(np.int64).sum()) == int(g["ids_crc"])
        logits = m.forward_initial(ids, 0, [mel])[0, 0]
        n_tok = int(g["n_audio_tokens"])
        feat = m.debug_read("audio_embeds", 0, n_tok * 1024).reshape(n_tok, 1024)
        e = float(np.abs(feat[g["audio_rows"]] - g["audio_sample"]).max())
        assert e <= TOL, f"audio tower output differs from the oracle by {e}"
        assert abs(float(np.abs(feat.astype(np.float64)).sum()) - float(g["audio_abs"])) <= 1e-4 * float(g["audio_abs"])
        _check_chain(m, g, len(ids), logits, "ASR-0.6 30 s")
    finally:
        m.close()
