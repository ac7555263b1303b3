"""-m gpu tests of the 80-mel checkpoints (large-v2, distil-large-v2, medium, small, base): the 80-bin log-mel kernels
(short and long-form), the conv stem at K = 3 * 80 = 240 (the only GEMM launch whose K is not a multiple of 64: the TMA
box zero-fills the last k-block), the encoder, greedy / beam / word-timestamp generation with the v2 token ids on the tiny
80-mel model, the pipeline against the v2 transformers golden, full-size large-v2 and medium parity against the fp32
reference, and install() with an 80-mel loader.  Tolerances are those of the 128-mel tests (test_gpu_engine.py,
test_gpu_fullsize.py, test_gpu_zz_word_timestamps.py)."""
import json
import os

import numpy as np
import pytest
import torch

import helpers
import helpers_v2 as V

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ENC_REL_TOL, ENC_MEAN_TOL = 5e-2, 1e-2
MARGIN_TOL = 0.30
WORD_HEADS = [[0, 1], [1, 0], [1, 3]]
NUM_FRAMES = [3000, 3000, 1130]
TS_CLOSE_S, TS_CLOSE_FRAC = 0.2, 0.9


def _clips():
    return [helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"), helpers.synth_clip(2, seconds=11.3, kind="mod")]


@pytest.fixture(scope="module")
def tiny(cuda_device):
    from oracle import whisper_ref as R
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    clips = _clips()
    feats = torch.stack([torch.from_numpy(V.log_mel(c)) for c in clips])
    out = {}
    for variant in ("decisive", "varied"):
        sd = V.variant_state_dict(V.ref_dims(), variant)
        gen = V.generation_settings()
        gen.alignment_heads = WORD_HEADS
        eng = WhisperEngine(WhisperDims(**V.TINY_V2), sd, device=cuda_device, max_batch=16, gen=gen)
        out[variant] = (R.WhisperRef(V.ref_dims(), sd), eng)
    return clips, feats, out


# ------------------------------------------------------------------ K1 log-mel, 80 bins
@pytest.mark.parametrize("n_valid", [480000, 12345, 0])
def test_logmel_80_vs_reference(cuda_device, n_valid):
    from turbo_whisper_workspace_b200 import ops
    rng = np.random.default_rng(0)
    B = 3
    pcm = (0.1 * rng.standard_normal((B, 480000))).astype(np.float32)
    t = np.arange(480000) / 16000.0
    pcm[1] = (0.3 * np.sin(2 * np.pi * (200 + 100 * t) * t) * (t < 20) + 1e-4 * pcm[1]).astype(np.float32)
    nv = np.array([n_valid, 480000, n_valid // 2], dtype=np.int32)
    lm = ops.LogMel(cuda_device, 4, n_mels=80)
    out = torch.empty(B, 80, 3000, dtype=torch.float32, device=cuda_device)
    out_t = torch.zeros(B, 3002, 80, dtype=torch.bfloat16, device=cuda_device)
    lm(torch.from_numpy(pcm).to(cuda_device), torch.from_numpy(nv).to(cuda_device), out_f32=out, out_t=out_t,
       out_t_row_off=1)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    for b in range(B):
        np.testing.assert_allclose(got[b], V.log_mel(pcm[b, :nv[b]]), rtol=1e-4, atol=1e-4)
    assert torch.equal(out_t[:, 1:3001, :].float().transpose(1, 2), out.to(torch.bfloat16).float())
    assert float(out_t[:, 0].abs().max()) == 0.0 and float(out_t[:, 3001].abs().max()) == 0.0
    # the 128-bin instance still answers on the same device, and n_mels outside {80, 128} is refused
    from turbo_whisper_workspace_b200 import _lib
    with pytest.raises(_lib.TwError, match="n_mels"):
        ops.LogMel(cuda_device, 1, n_mels=64)


@pytest.mark.parametrize("seconds", [75.3, 31.0])
def test_logmel_long_80_vs_reference(cuda_device, seconds):
    from turbo_whisper_workspace_b200 import ops
    n = int(seconds * 16000)
    audio = np.concatenate([helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"),
                            helpers.synth_clip(2, seconds=20.0, kind="mod")])[:n]
    got = ops.LogMel(cuda_device, 1, n_mels=80).long(audio).float().cpu().numpy().T
    want = V.log_mel_long(audio)
    assert got.shape == want.shape == (80, n // 160)
    # the time-major output is bf16: the stated 1e-4 tolerance plus half a bf16 ulp of the value
    np.testing.assert_allclose(got, want, rtol=2 ** -8, atol=1e-4)


# ------------------------------------------------------------------ conv stem (K = 240) and encoder
@pytest.mark.parametrize("variant", ["decisive", "varied"])
def test_conv_stem_k240_and_encoder_vs_oracle(tiny, cuda_device, variant):
    clips, feats, out = tiny
    ref, eng = out[variant]
    assert tuple(eng.w["conv1_w"].shape) == (256, 240)
    B = eng.load_pcm(clips)
    f32 = torch.empty(B, 80, 3000, dtype=torch.float32, device=cuda_device)
    eng.features(B, out_f32=f32)
    np.testing.assert_allclose(f32.cpu().numpy(), feats.numpy(), rtol=1e-4, atol=1e-4)
    taps = {"layers": (0,)}
    enc = eng.encode(B, taps=taps).float().view(B, 1500, -1).cpu()
    want, layers = ref.encode(feats.to(torch.bfloat16).float(), return_layers=True)
    rms = lambda t: float(t.pow(2).mean().sqrt())
    stem = taps["stem"].view(B, 1500, -1).cpu()
    assert float((stem - layers[0]).abs().max()) / rms(layers[0]) < ENC_REL_TOL
    assert float((enc - want).abs().max()) / rms(want) < ENC_REL_TOL
    assert float((enc - want).abs().mean()) / rms(want) < ENC_MEAN_TOL


# ------------------------------------------------------------------ generation with the v2 ids
def test_generate_v2_decisive(tiny):
    clips, feats, out = tiny
    ref, eng = out["decisive"]
    trace, etrace = {}, {}
    want = ref.generate(feats.to(torch.bfloat16).float(), gc=V.gen_config(), trace=trace)
    B = eng.load_pcm(clips)
    eng.features(B)
    got = eng.generate(B, trace=etrace)
    assert all(row[0] >= V.TIMESTAMP_BEGIN for row in got if row)
    agreed, identical_rows, first_diffs = helpers.compare_generate_traces(trace, etrace, MARGIN_TOL)
    assert len(identical_rows) >= 2, f"too many rows left the decisive regime: {first_diffs}"
    for b in identical_rows:
        assert got[b] == want[b]
    assert agreed >= 0.9 * sum(len(r) for r in want), (agreed, first_diffs)


def test_teacher_forced_decode_v2_varied(tiny):
    """The low-margin model with the v2 grammar ids: its language picks are near-ties for the oracle (margins 0.01-0.2,
    below the tolerance), so the oracle's prompt is given and its tokens are forced; every un-forced pick whose oracle
    margin exceeds the tolerance must equal the oracle's (test_gpu_engine.py's teacher-forced rule)."""
    clips, feats, out = tiny
    ref, eng = out["varied"]
    eng.enable_taps()
    trace = {}
    ref.generate(feats.to(torch.bfloat16).float(), gc=V.gen_config(), trace=trace)
    it0 = trace["iterations"][0]
    toks = it0["tokens"]
    B, n_gen = len(clips), toks.shape[1]
    eng.load_pcm(clips)
    eng.features(B)
    eng.encode(B)
    forced = torch.full((B, eng.max_len), -1, dtype=torch.int32)
    forced[:, 3:3 + n_gen] = toks.to(torch.int32)
    prompts = torch.tensor([[V.SOT, lang, V.TRANSCRIBE] for lang in trace["langs"]], dtype=torch.int32)
    eng.decode(B, prompts, n_steps=2 + n_gen, forced=forced)
    picks = eng.choices[:B].cpu()
    checked = disagree = 0
    for g in range(n_gen):
        rec = it0["record"][g]
        for b in range(B):
            if float(rec["margin"][b]) > MARGIN_TOL and float(rec["rule_gap"][b]) > MARGIN_TOL:
                checked += 1
                disagree += int(picks[b, 3 + g]) != int(toks[b, g])
    assert checked > 0.3 * n_gen * B, "tolerance leaves too few decisive steps to be a meaningful check"
    assert disagree == 0, f"{disagree} of {checked} decisive picks differ from the oracle"


def test_beam_search_v2(tiny):
    """num_beams=5 with the v2 ids: every returned hypothesis is grammatical for the oracle and the search's own
    accumulated log-probability agrees with the oracle's teacher-forced score (test_gpu_engine.py's rule)."""
    from oracle import whisper_ref as R
    clips, feats, out = tiny
    ref, eng = out["decisive"]
    gc = V.gen_config()
    enc = ref.encode(feats.to(torch.bfloat16).float())
    langs = ref.detect_language(enc, gc)
    prompt = torch.tensor([[gc.decoder_start_token_id, langs[b], gc.task_to_id["transcribe"]] for b in range(3)])
    want = ref.beam_search(enc, prompt, gc, num_beams=5)
    B = eng.load_pcm(clips)
    eng.features(B)
    eng.encode(B)
    got = eng.decode_beams(3, prompt.to(torch.int32), 5).cpu()
    exact = 0
    for b in range(3):
        n = int(eng.last_beam["length"][b])
        seq = got[b, :n].tolist()
        ids = torch.tensor([prompt[b].tolist() + seq])
        logits = ref.decode(ids, enc[b:b + 1])[0]
        score = 0.0
        for t, tok in enumerate(seq):
            lp = torch.log_softmax(logits[2 + t].float()[None], -1)
            score += float(R.WhisperRef.process_logits(lp, [seq[:t]], gc)[0, tok])
        own = float(eng.last_beam["sum_logprob"][b])
        assert score > -1e8, f"window {b}: hypothesis violates the timestamp grammar"
        assert abs(own - score) < 0.02 * n + 0.5, (b, own, score, n)
        w = want[b].tolist()
        while w and w[-1] == gc.pad_token_id and len(w) > n:
            w.pop()
        exact += seq == w[:n] and n == len(w)
    assert exact >= 1
    rows = eng.generate(B, num_beams=5)
    assert len(rows) == 3 and all(r and r[0] >= V.TIMESTAMP_BEGIN for r in rows)


def test_word_timestamps_v2(tiny):
    """generate(token_timestamps=True) with the v2 ids vs the oracle: identical tokens on at least one row and token
    times within the word-timestamp tolerance of test_gpu_zz_word_timestamps.py."""
    clips, feats, out = tiny
    ref, eng = out["decisive"]
    B = eng.load_pcm(clips)
    eng.features(B)
    got = eng.generate(B, token_timestamps=True, num_frames=NUM_FRAMES)
    ts = eng.last_token_ts
    ots = {}
    want = ref.generate(feats.to(torch.bfloat16).float(), gc=V.gen_config(), alignment_heads=WORD_HEADS,
                        num_frames=NUM_FRAMES, token_ts=ots)
    same_rows = [b for b in range(B) if got[b] == want[b]]
    assert same_rows, "no row decoded identically to the oracle"
    diffs = np.concatenate([np.abs(np.asarray(ts[b], np.float64) - np.asarray(ots["segments"][b], np.float64))
                            for b in same_rows])
    assert float((diffs <= TS_CLOSE_S).mean()) >= TS_CLOSE_FRAC, np.median(diffs)


# ------------------------------------------------------------------ pipeline and install()
@pytest.fixture(scope="module")
def wav(tmp_path_factory):
    p = tmp_path_factory.mktemp("audio") / "golden_v2_71s.wav"
    helpers.write_wav16(p, np.concatenate(_clips()))
    return str(p)


def _norm(r):
    return {"text": r["text"], "chunks": [{"timestamp": list(c["timestamp"]), "text": c["text"]} for c in r["chunks"]]}


def _common_prefix(a, b):
    n = 0
    while n < min(len(a), len(b)) and a[n] == b[n]:
        n += 1
    return n


def test_pipeline_v2_vs_hf_golden(cuda_device, wav):
    """The whole GPU pipeline of the decisive 80-mel model against the transformers pipeline dict (30 / 5 / 24), with
    return_timestamps=True and omitted.  Some picks of this model have oracle margins below the bf16 tolerance
    (decisive_30_0_min_margin in the fixture), after which the fp32 and bf16 decodes may legitimately part: the dicts
    must agree up to there (first timestamp, a long common text prefix), and exactly when the model is decisive."""
    from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline
    gold = json.load(open(os.path.join(GOLD, "pipeline_v2_tiny.json")))
    model, _ = V.hf_model("decisive")
    pipe = B200WhisperPipeline.from_hf_model(model, V.build_tokenizer(), devices=(cuda_device,), max_batch=8,
                                             contexts_per_device=1)
    for ts in (True, None):
        kw = {"return_timestamps": True} if ts else {}
        r = pipe(wav, chunk_length_s=30, stride_length_s=5, batch_size=24, generate_kwargs={"task": "transcribe"}, **kw)
        g = gold[f"decisive_30_5_24_{'ts' if ts else 'nots'}"]
        assert sorted(r.keys()) == g["keys"]
        if gold["decisive_30_0_min_margin"] > MARGIN_TOL:
            assert r["text"] == g["text"]
        n = _common_prefix(r["text"], g["text"])
        print(f"\n[v2 pipeline] return_timestamps={ts}: {n} / {len(g['text'])} characters identical to transformers")
        assert n >= min(len(g["text"]), 200)
        if ts:
            assert r["chunks"][0]["timestamp"][0] == g["chunks"][0]["timestamp"][0]


def test_install_with_80_mel_loader(cuda_device, wav):
    import transformers
    from turbo_whisper_workspace_b200 import install as twb
    model, _ = V.hf_model("decisive")
    tok = V.build_tokenizer()
    twb.install(devices=[cuda_device], max_batch=4, contexts_per_device=1, loader=lambda m, t=None: (model, tok))
    try:
        pipe = transformers.pipeline("automatic-speech-recognition", model="openai/whisper-large-v2", device=cuda_device)
        assert pipe.dims.n_mels == 80 and pipe.generation.no_timestamps_token_id == V.NO_TIMESTAMPS
        r = pipe(wav, chunk_length_s=30, stride_length_s=5, batch_size=24, generate_kwargs={"task": "transcribe"},
                 return_timestamps=True)
        gold = json.load(open(os.path.join(GOLD, "pipeline_v2_tiny.json")))["decisive_30_5_24_ts"]
        assert _common_prefix(r["text"], gold["text"]) >= min(len(gold["text"]), 200)
    finally:
        twb.uninstall()


# ------------------------------------------------------------------ full size: large-v2 and medium
@pytest.mark.parametrize("preset", ["large_v2", "medium"])
def test_fullsize_80_mel_vs_fp32_reference(cuda_device, preset):
    """Encoder states and teacher-forced logits of random full-size weights against the plain-PyTorch fp32 reference
    on the GPU (TF32 off), under test_gpu_fullsize.py's tolerances.  medium is the first run at d_model 1024 with 16
    heads and 24 decoder layers."""
    from oracle import whisper_ref as R
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dims = getattr(WhisperDims, preset)()
    rd = R.WhisperDims(d_model=dims.d_model, heads=dims.heads, ffn=dims.ffn, enc_layers=dims.enc_layers,
                       dec_layers=dims.dec_layers, n_mels=80, vocab=dims.vocab)
    sd = V.variant_state_dict(rd, "varied", seed=3)
    eng = WhisperEngine(dims, sd, device=cuda_device, max_batch=2, gen=V.generation_settings())
    eng.enable_taps()
    ref = R.WhisperRef(rd, {k: v.to(cuda_device) for k, v in sd.items()})
    clips = [helpers.synth_clip(40), helpers.synth_clip(41, kind="mod", seconds=17.25)]
    B = eng.load_pcm(clips)
    f32 = torch.empty(B, 80, 3000, dtype=torch.float32, device=cuda_device)
    eng.features(B, out_f32=f32)
    enc = eng.encode(B).float().view(B, 1500, -1).clone()
    want = ref.encode(f32.to(torch.bfloat16).float())
    rms = float(want.pow(2).mean().sqrt())
    err = (enc - want).abs()
    assert float(err.max()) / rms < 8e-2, float(err.max()) / rms
    assert float(err.mean()) / rms < 1.5e-2, float(err.mean()) / rms
    toks = torch.tensor([[V.SOT, V.LANG_FIRST, V.TRANSCRIBE, V.TIMESTAMP_BEGIN + 7, 1000, 2000, V.TIMESTAMP_BEGIN + 40,
                          V.TIMESTAMP_BEGIN + 40, 3000]] * B)
    wl = ref.decode(toks.to(cuda_device), enc)
    forced = torch.full((B, eng.max_len), -1, dtype=torch.int32)
    forced[:, :toks.shape[1]] = toks.to(torch.int32)
    got = []
    eng.decode(B, torch.tensor([[V.SOT, V.LANG_FIRST, V.TRANSCRIBE]] * B, dtype=torch.int32), n_steps=toks.shape[1],
               forced=forced, on_step=lambda s: got.append(eng.logits[:B].clone()))
    for s in range(toks.shape[1]):
        w = wl[:, s]
        e = float((got[s] - w).abs().max())
        bound = 2e-2 * float(w.abs().max()) + 2e-2
        assert e < bound, f"step {s}: {e} > {bound}"
        top2 = w.topk(2, dim=-1).values
        decisive = (top2[:, 0] - top2[:, 1]) > 2 * bound
        assert torch.equal(got[s].argmax(-1)[decisive], w.argmax(-1)[decisive])
