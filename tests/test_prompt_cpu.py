"""CPU tests of text prompts (generate_kwargs={"prompt_ids": ...}):
  * the prompt-aware reference (tests/helpers_prompt.py) reproduces transformers 5.5.0's generate(prompt_ids=...) token
    for token (tests/golden/prompt_tiny.json): prompt lengths across a KV page, timestamps off, explicit language,
    translate, beam search, token timestamps and un-chunked long-form;
  * the row-major unpack of the decode weights inverts pack_skinny_weight exactly for every decoder weight shape;
  * the pipeline forwards prompt_ids to the scheduler, validates them, and reproduces the golden pipeline dicts from
    the reference's token rows."""
import numpy as np
import pytest
import torch

import helpers
import helpers_prompt as HP
from oracle import logmel_ref as L
from oracle import whisper_ref as R
from turbo_whisper_workspace_b200.config import WhisperDims
from turbo_whisper_workspace_b200.engine import pack_skinny_weight, unpack_skinny_weight
from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline


@pytest.fixture(scope="module")
def gold():
    return HP.golden()


@pytest.fixture(scope="module")
def ref():
    rd = R.WhisperDims(**helpers.TINY)
    return R.WhisperRef(rd, helpers.variant_state_dict(rd, "decisive"))


@pytest.fixture(scope="module")
def feats():
    clips = [helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"), helpers.synth_clip(2, seconds=11.3, kind="mod")]
    return torch.stack([torch.from_numpy(L.log_mel(c)) for c in clips]).to(torch.bfloat16).float()


def _gen_cases():
    return sorted(HP.golden()["generate"])


@pytest.mark.parametrize("case", _gen_cases())
def test_reference_generate_with_prompt_matches_transformers(gold, ref, feats, case):
    g = gold["generate"][case]
    got = HP.prompted_generate(ref, feats, gold["prompts"][str(g["prompt"])], task=g["task"],
                               language=HP.lang_id(g["language"]), return_timestamps=g["timestamps"],
                               num_beams=g["num_beams"])
    for b, row in enumerate(got):
        assert row == HP.strip_hf(g["ids"][b]), f"row {b}"


def test_reference_token_timestamps_with_prompt_match_transformers(gold, ref, feats):
    g = gold["token_timestamps_16"]
    ts = {}
    got = HP.prompted_generate(ref, feats, gold["prompts"]["16"], alignment_heads=gold["alignment_heads"],
                               num_frames=gold["num_frames"], token_ts=ts)
    for b, row in enumerate(got):
        assert row == g["segment_tokens"][b], f"row {b}"
        np.testing.assert_array_equal(np.asarray(ts["segments"][b], dtype=np.float32),
                                      np.asarray(g["segment_token_timestamps"][b], dtype=np.float32))


@pytest.fixture(scope="module")
def long_pcm():
    return np.concatenate([helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"),
                           helpers.synth_clip(2, seconds=15.3, kind="mod")])


def test_reference_unchunked_longform_with_prompt_matches_transformers(gold, ref, long_pcm):
    feats = torch.from_numpy(L.log_mel_long(long_pcm))[None]
    got = HP.prompted_generate(ref, feats, gold["prompts"]["16"])[0]
    assert got == gold["longform_16"]["tokens"]


@pytest.mark.parametrize("preset", ["large_v3_turbo", "large_v3", "large_v2", "medium", "small", "base"])
def test_unpack_inverts_pack_for_every_decoder_weight(preset):
    d = getattr(WhisperDims, preset)()
    g = torch.Generator().manual_seed(0)
    for n, k in {(3 * d.d_model, d.d_model), (d.d_model, d.d_model), (d.ffn, d.d_model), (d.d_model, d.ffn)}:
        w = torch.randn(n, k, generator=g).to(torch.bfloat16)
        back = unpack_skinny_weight(pack_skinny_weight(w), n)
        assert back.shape == (n, k) and torch.equal(back.view(torch.int16), w.view(torch.int16)), (preset, n, k)
    # the LM head's vocab is not a multiple of 16: padded rows are dropped again
    w = torch.randn(d.vocab, 64, generator=g).to(torch.bfloat16)
    assert torch.equal(unpack_skinny_weight(pack_skinny_weight(w), d.vocab), w)


class RecordingScheduler:
    """Engine stand-in: records the keyword arguments, returns the reference's rows for the prompt it was given."""

    def __init__(self, ref=None):
        self.ref, self.calls, self.last_stats = ref, [], {}

    def run(self, clips, task="transcribe", language=None, return_timestamps=True, num_beams=1, token_timestamps=False,
            group=None, prompt_ids=None):
        self.calls.append(("run", dict(task=task, language=language, return_timestamps=return_timestamps,
                                       num_beams=num_beams, token_timestamps=token_timestamps, prompt_ids=prompt_ids)))
        if self.ref is None:
            return [[] for _ in clips]
        feats = torch.stack([torch.from_numpy(L.log_mel(c)) for c in clips])
        if not token_timestamps:
            return HP.prompted_generate(self.ref, feats, prompt_ids, task=task, return_timestamps=return_timestamps)
        rows = []
        for g0 in range(0, len(clips), group):
            sub = clips[g0:g0 + group]
            ts = {}
            ids = HP.prompted_generate(self.ref, feats[g0:g0 + group], prompt_ids, task=task,
                                       alignment_heads=HP.golden()["alignment_heads"],
                                       num_frames=[min(3000, -(-len(c) // 160)) for c in sub], token_ts=ts)
            rows += [(ids[b], ts["segments"][b]) for b in range(len(sub))]
        return rows

    def run_long(self, audio, task="transcribe", language=None, num_beams=1, prompt_ids=None):
        self.calls.append(("run_long", dict(task=task, language=language, num_beams=num_beams, prompt_ids=prompt_ids)))
        if self.ref is None:
            return []
        return HP.prompted_generate(self.ref, torch.from_numpy(L.log_mel_long(audio))[None], prompt_ids, task=task)[0]


def _pipe(sched):
    return B200WhisperPipeline(None, WhisperDims(**helpers.TINY), helpers.build_tokenizer(), scheduler=sched)


@pytest.mark.parametrize("kind", ["list", "numpy", "torch"])
def test_pipeline_forwards_prompt_ids(kind, long_pcm):
    ids = [50361, 400, 401, 402]
    val = {"list": ids, "numpy": np.asarray(ids, dtype=np.int64), "torch": torch.tensor(ids)}[kind]
    sched = RecordingScheduler()
    pipe = _pipe(sched)
    pipe(helpers.synth_clip(0, seconds=5.0), generate_kwargs={"prompt_ids": val, "num_beams": 2}, return_timestamps=True)
    assert sched.calls[-1] == ("run", dict(task="transcribe", language=None, return_timestamps=True, num_beams=2,
                                           token_timestamps=False, prompt_ids=ids))
    pipe(long_pcm, generate_kwargs={"prompt_ids": val, "prompt_condition_type": "first-segment"}, return_timestamps=True)
    assert sched.calls[-1] == ("run_long", dict(task="transcribe", language=None, num_beams=1, prompt_ids=ids))
    # without a prompt the schedulers are called exactly as before (no prompt_ids keyword)
    calls = []

    class Plain:
        last_stats = {}

        def run(self, clips, task="transcribe", language=None, return_timestamps=True):
            calls.append((task, language, return_timestamps))
            return [[] for _ in clips]
    _pipe(Plain())(helpers.synth_clip(0, seconds=5.0), return_timestamps=True)
    assert calls == [("transcribe", None, True)]


def test_pipeline_prompt_validation():
    sched = RecordingScheduler()
    pipe = _pipe(sched)
    clip = helpers.synth_clip(0, seconds=5.0)
    bad = [[], [[50361, 1]], [50361, 51866], [-1], [0.5, 1.0], np.zeros((2, 2), dtype=np.int64)]
    for v in bad:
        with pytest.raises(ValueError):
            pipe(clip, generate_kwargs={"prompt_ids": v}, return_timestamps=True)
    # decoder input = prompt + 3 specials (4 without timestamps) must be shorter than 448
    pipe(clip, generate_kwargs={"prompt_ids": [50361] + [400] * 443}, return_timestamps=True)
    with pytest.raises(ValueError, match="shorter than 448"):
        pipe(clip, generate_kwargs={"prompt_ids": [50361] + [400] * 444}, return_timestamps=True)
    with pytest.raises(ValueError, match="shorter than 448"):
        pipe(clip, generate_kwargs={"prompt_ids": [50361] + [400] * 443})
    assert len(sched.calls) == 1          # nothing reached the engines for a rejected call


def test_pipeline_prompt_condition_type_errors_match_transformers(gold):
    pipe = _pipe(RecordingScheduler())
    clip = helpers.synth_clip(0, seconds=5.0)
    for cond in ("no-such-type", "all-segments"):
        g = gold[f"condition_{cond}"]
        with pytest.raises(ValueError) as e:
            pipe(clip, generate_kwargs={"prompt_ids": [50361, 400], "prompt_condition_type": cond}, return_timestamps=True)
        assert g["raises"] == "ValueError" and str(e.value) == g["message"]
    with pytest.raises(NotImplementedError):
        pipe(clip, generate_kwargs={"prompt_ids": [50361, 400], "prompt_condition_type": "all-segments",
                                    "condition_on_prev_tokens": True}, return_timestamps=True)


@pytest.fixture(scope="module")
def wav(tmp_path_factory):
    pcm = np.concatenate([helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"),
                          helpers.synth_clip(2, seconds=11.3, kind="mod")])
    p = tmp_path_factory.mktemp("audio") / "golden_71s.wav"
    helpers.write_wav16(p, pcm)
    return str(p)


@pytest.mark.parametrize("name,ts", [("ts", True), ("nots", None), ("word", "word")])
def test_host_pipeline_with_prompt_matches_transformers(gold, ref, wav, name, ts):
    """The host pipeline (windowing, stride plumbing, _decode_asr on rows WITHOUT the prompt) on the reference's token
    rows reproduces transformers' pipeline dicts for a prompted call."""
    pipe = _pipe(RecordingScheduler(ref))
    kw = {"return_timestamps": ts} if ts else {}
    r = pipe(wav, chunk_length_s=30, stride_length_s=5, batch_size=24,
             generate_kwargs={"task": "transcribe", "prompt_ids": gold["prompts"]["16"]}, **kw)
    g = gold[f"pipeline_30_5_24_{name}"]
    assert sorted(r.keys()) == g["keys"] and r["text"] == g["text"]
    if ts:
        assert [{"text": c["text"], "timestamp": list(c["timestamp"])} for c in r["chunks"]] == g["chunks"]


def test_host_pipeline_unchunked_longform_with_prompt_matches_transformers(gold, ref, long_pcm):
    pipe = _pipe(RecordingScheduler(ref))
    r = pipe(long_pcm.copy(), return_timestamps=True, generate_kwargs={"task": "transcribe", "prompt_ids": gold["prompts"]["16"]})
    g = gold["longform_16"]
    assert r["text"] == g["text"]
    assert [{"text": c["text"], "timestamp": list(c["timestamp"])} for c in r["chunks"]] == g["chunks"]
