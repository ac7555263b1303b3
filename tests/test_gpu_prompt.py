"""-m gpu tests of text prompts (generate(prompt_ids=...)): the batched decoder prefill against the forced-step route on
the same engine, the prompted seek loop against the fp32 oracle and the transformers golden (tests/golden/
prompt_tiny.json), beam search, word timestamps, long-form, the pipeline, and the full-size shapes."""
import json
import os

import numpy as np
import pytest
import torch

import helpers
import helpers_prompt as HP

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
HEADS = [[0, 1], [1, 0], [1, 3]]
MARGIN_TOL = 0.30            # tests/test_gpu_engine.py: decisive picks must agree with the oracle
LOGIT_REL_TOL = 2e-2         # max |logit - ref| <= LOGIT_REL_TOL * max|ref| + LOGIT_ABS_FLOOR (test_gpu_engine.py)
LOGIT_ABS_FLOOR = 2e-2
# prefill vs forced steps on one engine: both are bf16 between kernels; they differ in how a LayerNorm reaches its
# projection (the step folds it into the weights and normalises in the epilogue, the prefill normalises the bf16 operand)
# and in the summation order of the attention, so K / V and logits agree to a few bf16 ulps of their scale
KV_REL_TOL = 3e-2            # max |K/V prefill - forced| <= KV_REL_TOL * max |K/V forced|, per layer
PF_LOGIT_REL_TOL = 2e-2      # max |logit prefill - forced| <= PF_LOGIT_REL_TOL * max |logit forced| + 2e-2
TS_CLOSE_S, TS_CLOSE_FRAC, TS_IDENTICAL_FRAC = 0.2, 0.9, 0.85   # word times (tests/test_gpu_zz_word_timestamps.py)


def _lang_gen(**kw):
    from transformers.models.whisper.tokenization_whisper import LANGUAGES
    from turbo_whisper_workspace_b200.config import GenerationSettings
    return GenerationSettings(lang_to_id={f"<|{l}|>": 50259 + i for i, l in enumerate(LANGUAGES)}, **kw)


def _forced_route(eng, R, row, timestamps):
    """The prompt through the existing step loop: row[0] fed at position 0, row[1:] teacher-forced, the grammar's
    begin index at the prompt length.  Returns the row state after the steps that feed positions 0 .. P-2 (the state
    the prefill path starts from); returns after the step that feeds position P-1."""
    from turbo_whisper_workspace_b200.engine import init_rows
    tok0, frc, st0, P = init_rows(torch.tensor([row] * R), eng.max_len, eng.grammar, timestamps)
    eng.grammar.begin_index = P
    eng.tokens[:R].copy_(tok0.to(eng.device))
    eng.forced[:R].copy_(frc.to(eng.device))
    eng.state[:R].copy_(st0.to(eng.device))
    for _ in range(P - 1):
        eng._decode_step(R)
    before = eng.state[:R].clone()
    eng._decode_step(R)
    torch.cuda.synchronize()
    return before


def _kv(eng, R, P):
    """K / V of positions 0 .. P-1 of rows 0 .. R-1, every layer: [L, 2, R, P, D] (identity block table)."""
    L, D = eng.dims.dec_layers, eng.dims.d_model
    pool = eng.kv_pool[:, :, :R * eng.pages_per_row].reshape(L, 2, R, eng.pages_per_row * 64, D)
    return pool[:, :, :, :P].float().clone()


def _prefill_vs_forced(eng, R, prompt_ids, lang=50259, timestamps=False):
    from oracle import whisper_ref as R_
    tail = [] if timestamps else [eng.gen.no_timestamps_token_id]
    row = list(prompt_ids) + [R_.SOT, lang, R_.TRANSCRIBE] + tail
    P = len(row)
    prompts = torch.tensor([[R_.SOT, lang, R_.TRANSCRIBE]] * R, dtype=torch.int32)
    eng.decode(R, prompts, n_steps=0, timestamps=timestamps, prompt_ids=prompt_ids)      # prefill only
    got_state = eng.state[:R].clone()
    eng.kv_pool.zero_()
    eng.decode(R, prompts, n_steps=1, timestamps=timestamps, prompt_ids=prompt_ids)
    torch.cuda.synchronize()
    assert eng.tokens[:R, :P].cpu().tolist() == [row] * R
    got_logits, got_kv = eng.logits[:R].clone(), _kv(eng, R, P)
    got_pick, got_after = eng.tokens[:R, P].clone(), eng.state[:R].clone()
    eng.kv_pool.zero_()
    want_state = _forced_route(eng, R, row, timestamps)
    want_logits, want_kv = eng.logits[:R].clone(), _kv(eng, R, P)
    want_pick, want_after = eng.tokens[:R, P].clone(), eng.state[:R].clone()
    # the row state the prefill path builds by hand (position, grammar, begin flag, mode) is the one the forced steps
    # leave behind, and rows that pick the same first token continue from the same state
    assert torch.equal(got_state, want_state), (got_state[0].tolist(), want_state[0].tolist())
    same = got_pick == want_pick
    assert torch.equal(got_after[same], want_after[same])
    lerr = float((got_logits - want_logits).abs().max())
    lbound = PF_LOGIT_REL_TOL * float(want_logits.abs().max()) + 2e-2
    kv_err = [(float((got_kv[l] - want_kv[l]).abs().max()), float(want_kv[l].abs().max())) for l in range(got_kv.shape[0])]
    print(f"\n[prefill vs forced] R={R} P={P}: logits max |diff| {lerr:.4f} (bound {lbound:.4f}); K/V per layer "
          + ", ".join(f"{e:.4f}/{m:.2f}" for e, m in kv_err))
    assert lerr < lbound
    for l, (e, m) in enumerate(kv_err):
        assert e <= KV_REL_TOL * m, f"layer {l}: K/V max |diff| {e} > {KV_REL_TOL} x {m}"
    top2 = want_logits.topk(2, dim=-1).values
    decisive = (top2[:, 0] - top2[:, 1]) > 2 * lbound
    assert torch.equal(got_logits.argmax(-1)[decisive], want_logits.argmax(-1)[decisive])
    print(f"  first generated token identical on {int(same.sum())} / {R} rows")


@pytest.fixture(scope="module")
def tiny96(cuda_device):
    from oracle import whisper_ref as R
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    sd = helpers.variant_state_dict(R.WhisperDims(**helpers.TINY), "varied")
    eng = WhisperEngine(WhisperDims(**helpers.TINY), sd, device=cuda_device, max_batch=96)
    eng.enable_taps()
    clips = [helpers.synth_clip(i % 8, kind="mod" if i % 2 else "noise", seconds=30.0 - (i % 5)) for i in range(96)]
    B = eng.load_pcm(clips)
    eng.features(B)
    eng.encode(B)
    return eng


@pytest.mark.parametrize("timestamps", [False, True])
@pytest.mark.parametrize("R", [1, 24, 96])
@pytest.mark.parametrize("n", [1, 61, 62, 200])
def test_prefill_matches_forced_steps(tiny96, R, n, timestamps):
    """Same encoder state, same prompt (n prompt ids + 3 special tokens, + <|notimestamps|> without timestamps): the
    batched prefill and the existing step loop with the prompt teacher-forced leave the same K / V in every page of
    every prompt position, the same row state before the first generated position and the same logits there."""
    ids = [HP.PREV] + list(range(1000, 1000 + n - 1))
    _prefill_vs_forced(tiny96, R, ids, timestamps=timestamps)


@pytest.fixture(scope="module")
def tiny(cuda_device):
    from oracle import logmel_ref as L
    from oracle import whisper_ref as R
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    clips = [helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"), helpers.synth_clip(2, seconds=11.3, kind="mod")]
    feats = torch.stack([torch.from_numpy(L.log_mel(c)) for c in clips]).to(torch.bfloat16).float()
    rd = R.WhisperDims(**helpers.TINY)
    sd = helpers.variant_state_dict(rd, "decisive")
    eng = WhisperEngine(WhisperDims(**helpers.TINY), sd, device=cuda_device, max_batch=15,
                        gen=_lang_gen(alignment_heads=HEADS))
    eng.enable_taps()
    return clips, feats, R.WhisperRef(rd, sd), eng, sd


@pytest.mark.parametrize("case", ["ts_detect_1", "ts_detect_16", "ts_detect_63", "ts_detect_64", "ts_detect_65",
                                  "ts_detect_200", "nots_en_16", "translate_de_16"])
def test_generate_with_prompt_matches_oracle(tiny, case):
    """Greedy with a prompt against the fp32 oracle (rule of compare_generate_traces: ids identical wherever the
    oracle's margin exceeds the tolerance); rows decoded end to end equal transformers' golden ids."""
    clips, feats, ref, eng, _ = tiny
    gold = HP.golden()
    g = gold["generate"][case]
    ids = gold["prompts"][str(g["prompt"])]
    B = eng.load_pcm(clips)
    eng.features(B)
    etrace, trace = {}, {}
    got = eng.generate(B, task=g["task"], language=g["language"], return_timestamps=g["timestamps"], trace=etrace,
                       prompt_ids=ids)
    want = HP.prompted_generate(ref, feats, ids, task=g["task"], language=HP.lang_id(g["language"]),
                                return_timestamps=g["timestamps"], trace=trace)
    agreed, same, diffs = HP.compare_prompted_traces(trace, etrace, MARGIN_TOL)
    print(f"\n[{case}] {agreed} tokens agree; identical rows {same}; low-margin divergences {diffs}")
    assert same, "no row decoded identically to the oracle"
    for b in same:
        assert got[b] == want[b] == HP.strip_hf(g["ids"][b]), f"row {b}"


def test_teacher_forced_logits_with_prompt_match_oracle(tiny):
    """The oracle's first-iteration tokens teacher-forced after a 64-id prompt: raw logits at the recorded steps."""
    from oracle import whisper_ref as R
    clips, feats, ref, eng, _ = tiny
    ids = HP.golden()["prompts"]["64"]
    trace = {}
    HP.prompted_generate(ref, feats, ids, trace=trace)
    it0 = trace["iterations"][0]
    toks, P, B = it0["tokens"], trace["P"], len(clips)
    n_gen = toks.shape[1]
    eng.load_pcm(clips)
    eng.features(B)
    eng.encode(B)
    forced = torch.full((B, eng.max_len), -1, dtype=torch.int32)
    forced[:, P:P + n_gen] = toks.to(torch.int32)
    prompts = torch.tensor([[R.SOT, l, R.TRANSCRIBE] for l in trace["langs"]], dtype=torch.int32)
    seen = {}

    def on_step(s):
        if s in R.RECORD_LOGIT_STEPS and s < n_gen:
            seen[s] = eng.logits[:B].cpu().clone()
    eng.decode(B, prompts, n_steps=n_gen, forced=forced, on_step=on_step, prompt_ids=ids)
    assert seen
    for s, lg in seen.items():
        w = it0["record"][s]["logits"]
        err, bound = float((lg - w).abs().max()), LOGIT_REL_TOL * float(w.abs().max()) + LOGIT_ABS_FLOOR
        assert err < bound, f"generated step {s}: {err} > {bound}"


def _oracle_sequence_score(ref, gc, enc_row, prompt_row, seq):
    """Sum of the processed log-probabilities the fp32 oracle assigns to `seq` (teacher-forced) after `prompt_row`
    (the rule of tests/test_gpu_engine.py)."""
    from oracle import whisper_ref as R
    logits = ref.decode(torch.tensor([list(prompt_row) + list(seq)]), enc_row)[0]
    P, tot = len(prompt_row), 0.0
    for t, tok in enumerate(seq):
        lp = torch.log_softmax(logits[P - 1 + t].float()[None], -1)
        lp = R.WhisperRef.process_logits(lp, [list(seq[:t])], gc)
        tot += float(lp[0, tok])
    return tot


def test_beam_search_with_prompt_matches_transformers(tiny):
    """num_beams=5 after a 16- and a 64-id prompt.  First seek iteration against the fp32 oracle's search (token-exact
    with transformers on CPU): every returned hypothesis is grammatical, the search's own accumulated log-probability
    agrees with the oracle's teacher-forced score within the bf16 bound of tests/test_gpu_engine.py (0.02 n + 0.5), and a
    hypothesis that differs from the oracle's best is a near tie for the oracle — its length-normalised oracle score is
    within that same bound (per token) of the best one's.  The whole seek loop then reproduces transformers' ids on
    every window whose first iteration matched the oracle."""
    from oracle import whisper_ref as R
    clips, feats, ref, eng, _ = tiny
    gold = HP.golden()
    gc = R.GenConfig()
    enc = ref.encode(feats)
    langs = ref.detect_language(enc, gc)
    B = len(clips)
    for case in ("beams5_16", "beams5_64"):
        g = gold["generate"][case]
        ids = gold["prompts"][str(g["prompt"])]
        rows = torch.tensor([ids + [gc.decoder_start_token_id, langs[b], gc.task_to_id["transcribe"]] for b in range(B)])
        want = ref.beam_search(enc, rows, gc, num_beams=5)
        assert eng.load_pcm(clips) == B
        eng.features(B)
        eng.encode(B)
        got = eng.decode_beams(B, rows[:, -3:].to(torch.int32), 5, prompt_ids=ids).cpu()
        matched = []
        for b in range(B):
            n = int(eng.last_beam["length"][b])
            seq = got[b, :n].tolist()
            score = _oracle_sequence_score(ref, gc, enc[b:b + 1], rows[b].tolist(), seq)
            own = float(eng.last_beam["sum_logprob"][b])
            assert score > -1e8, f"{case} window {b}: hypothesis violates the timestamp grammar"
            assert abs(own - score) < 0.02 * n + 0.5, (case, b, own, score, n)
            w = want[b].tolist()                    # ends with eos (= pad) unless the hypothesis hit max_length
            ended = bool(w) and w[-1] == gc.pad_token_id
            while w and w[-1] == gc.pad_token_id:
                w.pop()
            w = w + [gc.eos_token_id] if ended else w
            if seq == w:
                matched.append(b)
                continue
            best = _oracle_sequence_score(ref, gc, enc[b:b + 1], rows[b].tolist(), w)
            gap = best / len(w) - score / n
            print(f"\n[{case}] window {b} differs from the oracle's best: length-normalised oracle score gap {gap:.4f}")
            assert gap < 0.02 + 0.5 / n, f"{case} window {b}: not a near tie ({gap:.4f})"
        eng.load_pcm(clips)
        eng.features(B)
        full = eng.generate(B, num_beams=5, prompt_ids=ids)
        same = [b for b in range(B) if full[b] == HP.strip_hf(g["ids"][b])]
        print(f"\n[{case}] first iteration identical to the oracle on {matched}; seek loop identical to transformers on {same}")
        assert set(matched) <= set(same), case


def test_word_timestamps_with_prompt(tiny):
    clips, feats, ref, eng, _ = tiny
    gold = HP.golden()
    g = gold["token_timestamps_16"]
    B = eng.load_pcm(clips)
    eng.features(B)
    got = eng.generate(B, token_timestamps=True, num_frames=gold["num_frames"], prompt_ids=gold["prompts"]["16"])
    same = [b for b in range(B) if got[b] == g["segment_tokens"][b]]
    assert same, "no row decoded identically to transformers"
    diffs = np.concatenate([np.abs(np.asarray(eng.last_token_ts[b]) - np.asarray(g["segment_token_timestamps"][b]))
                            for b in same])
    identical, close = float((diffs < 1e-6).mean()), float((diffs <= TS_CLOSE_S).mean())
    print(f"\n[word] rows {same}: {identical:.3f} of the token times identical, {close:.3f} within {TS_CLOSE_S} s, "
          f"max |diff| {diffs.max():.2f} s")
    # the rule of tests/test_gpu_zz_word_timestamps.py: the DTW path of bf16 cross-attention may move a token by a frame
    # or two where the path is a near tie, nowhere else
    assert identical >= TS_IDENTICAL_FRAC and close >= TS_CLOSE_FRAC
    # beam search + word timestamps with a prompt: one time per returned id
    got = eng.generate(B, num_beams=3, token_timestamps=True, num_frames=gold["num_frames"],
                       prompt_ids=gold["prompts"]["16"])
    assert [len(t) for t in eng.last_token_ts] == [len(r) for r in got]


def test_longform_with_prompt_matches_transformers(tiny):
    clips, feats, ref, eng, _ = tiny
    gold = HP.golden()["longform_16"]
    pcm = np.concatenate([helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"),
                          helpers.synth_clip(2, seconds=15.3, kind="mod")])
    got = eng.generate_long_from_pcm(pcm, prompt_ids=HP.golden()["prompts"]["16"])
    assert got == gold["tokens"]


def test_pipeline_with_prompt_matches_transformers(tiny, tmp_path, cuda_device):
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline
    clips, feats, ref, eng, sd = tiny
    gold = HP.golden()
    path = tmp_path / "golden_71s.wav"
    helpers.write_wav16(path, np.concatenate(clips))
    pipe = B200WhisperPipeline(sd, WhisperDims(**helpers.TINY), helpers.build_tokenizer(), _lang_gen(alignment_heads=HEADS),
                               devices=[cuda_device], max_batch=4, contexts_per_device=2)
    try:
        for name, ts in (("ts", True), ("nots", None), ("word", "word")):
            kw = {"return_timestamps": ts} if ts else {}
            r = pipe(str(path), chunk_length_s=30, stride_length_s=5, batch_size=24,
                     generate_kwargs={"task": "transcribe", "prompt_ids": np.asarray(gold["prompts"]["16"])}, **kw)
            g = gold[f"pipeline_30_5_24_{name}"]
            assert sorted(r.keys()) == g["keys"] and r["text"] == g["text"], name
            if ts is True:
                assert [{"text": c["text"], "timestamp": list(c["timestamp"])} for c in r["chunks"]] == g["chunks"]
    finally:
        pipe.close()


@pytest.mark.parametrize("preset", ["large_v3_turbo", "large_v3"])
def test_fullsize_prompt_vs_fp32_reference(preset, cuda_device):
    """A 128-id prompt on 2 windows at full size: logits of the first generated position (prefill + one step) against
    the plain-PyTorch fp32 reference on the GPU running the whole prompt as one forward; plus prefill vs forced steps
    at 24 rows."""
    from oracle import whisper_ref as R
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    dims = getattr(WhisperDims, preset)()
    rd = R.WhisperDims(dec_layers=dims.dec_layers)
    sd = helpers.variant_state_dict(rd, "varied", seed=3)
    eng = WhisperEngine(dims, sd, device=cuda_device, max_batch=24)
    eng.enable_taps()
    ref = R.WhisperRef(rd, {k: v.to(cuda_device) for k, v in sd.items()})
    del sd
    clips = [helpers.synth_clip(40 + i, kind="mod" if i % 2 else "noise") for i in range(2)]
    ids = [HP.PREV] + list(range(2000, 2127))
    B = eng.load_pcm(clips)
    f32 = torch.empty(B, 128, 3000, dtype=torch.float32, device=cuda_device)
    eng.features(B, out_f32=f32)
    enc = eng.encode(B).float().view(B, 1500, -1).clone()
    row = ids + [R.SOT, 50259, R.TRANSCRIBE]
    with torch.no_grad():
        want = ref.decode(torch.tensor([row] * B, device=cuda_device), enc)[:, -1]
    eng.decode(B, torch.tensor([[R.SOT, 50259, R.TRANSCRIBE]] * B, dtype=torch.int32), n_steps=1, prompt_ids=ids)
    got = eng.logits[:B]
    err, bound = float((got - want).abs().max()), LOGIT_REL_TOL * float(want.abs().max()) + LOGIT_ABS_FLOOR
    print(f"\n[{preset}] first generated position after a {len(row)}-position prompt: max |logit diff| {err:.4f} "
          f"(bound {bound:.4f})")
    assert err < bound
    del ref
    torch.cuda.empty_cache()
    if preset == "large_v3_turbo":
        clips24 = [helpers.synth_clip(60 + i, kind="mod" if i % 2 else "noise") for i in range(24)]
        B = eng.load_pcm(clips24)
        eng.features(B)
        eng.encode(B)
        _prefill_vs_forced(eng, 24, ids[:125], timestamps=False)
