"""CPU tests of the 80-mel checkpoints (large-v2 and older): the oracle with the v2 token layout and the 80-bin log-mel
reference against the fixtures of tests/golden/make_golden_v2.py (transformers 5.5.0), how B200WhisperPipeline reads
such a checkpoint, the host pipeline against the v2 pipeline dicts, and the explicit rejection of English-only
checkpoints."""
import json
import os

import numpy as np
import pytest
import torch

import helpers
import helpers_v2 as V
from oracle import whisper_ref as R
from turbo_whisper_workspace_b200.config import WhisperDims
from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DEC_IDS = [V.SOT, V.LANG_FIRST, V.TRANSCRIBE, V.TIMESTAMP_BEGIN, 400, 401, V.TIMESTAMP_BEGIN + 35,
           V.TIMESTAMP_BEGIN + 35, 402]       # tests/golden/make_golden_v2.py


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "v2_tiny.npz"))


def _clips():
    return [helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"), helpers.synth_clip(2, seconds=11.3, kind="mod")]


def _feats_bf16():
    return torch.stack([torch.from_numpy(V.log_mel(c)) for c in _clips()]).to(torch.bfloat16).float()


@pytest.mark.parametrize("name", ["noise30", "sine440", "short", "mod"])
def test_logmel_80_reference_vs_hf_golden(gold, name):
    A = (0.1 * np.random.default_rng(0).standard_normal(480000)).astype(np.float32)
    t = np.arange(480000) / 16000.0
    pcm = {"noise30": A, "sine440": (0.5 * np.sin(2 * np.pi * 440.0 * t)).astype(np.float32), "short": A[:12345],
           "mod": helpers.synth_clip(1, kind="mod")}[name]
    x = V.log_mel(pcm)
    assert x.shape == (80, 3000)
    np.testing.assert_allclose(x[::4, ::25], gold[f"logmel_{name}_sub"], atol=2e-5, rtol=0)
    np.testing.assert_allclose([x.mean(), x.min(), x.max()], gold[f"logmel_{name}_stats"], atol=2e-5)


@pytest.mark.parametrize("variant", ["decisive", "varied"])
def test_model_oracle_vs_hf_golden_v2(gold, variant):
    fb = _feats_bf16()
    ref = R.WhisperRef(V.ref_dims(), V.variant_state_dict(V.ref_dims(), variant))
    enc = ref.encode(fb)
    np.testing.assert_allclose(enc[:, ::50, ::8].numpy(), gold[f"{variant}_enc_sub"], atol=2e-4, rtol=1e-4)
    logits = ref.decode(torch.tensor([DEC_IDS] * 3), enc)
    assert logits.shape[-1] == V.VOCAB
    np.testing.assert_allclose(logits[:, :, ::97].numpy(), gold[f"{variant}_logits_sub"], atol=2e-3, rtol=1e-4)
    assert ref.detect_language(enc, V.gen_config()) == gold[f"{variant}_langs"].tolist()


@pytest.mark.parametrize("variant", ["decisive", "varied"])
def test_generate_oracle_vs_hf_golden_v2(gold, variant):
    """Token for token with WhisperGenerationMixin.generate of the 80-mel model under the v2 ids (timestamps from
    50364, no-timestamps 50363, transcribe 50359)."""
    ref = R.WhisperRef(V.ref_dims(), V.variant_state_dict(V.ref_dims(), variant))
    got = ref.generate(_feats_bf16(), gc=V.gen_config())
    g = gold[f"{variant}_generate"]
    assert any(t >= V.TIMESTAMP_BEGIN for row in got for t in row)
    for b, row in enumerate(got):
        want = g[b].tolist()
        while want and want[-1] == V.EOS:
            want.pop()
        assert row == want, f"row {b}"


class _NoEngine:
    last_stats: dict = {}

    def run(self, *a, **k):
        raise AssertionError("not called")


def test_from_hf_model_reads_80_mels_and_v2_ids():
    model, _ = V.hf_model("varied")
    pipe = B200WhisperPipeline.from_hf_model(model, V.build_tokenizer(), scheduler=_NoEngine())
    assert pipe.dims == WhisperDims(**V.TINY_V2)
    pipe.dims.validate()
    g = pipe.generation
    assert (g.no_timestamps_token_id, g.timestamp_begin) == (V.NO_TIMESTAMPS, V.TIMESTAMP_BEGIN)
    assert (g.lang_first, g.lang_last) == (V.LANG_FIRST, V.LANG_LAST)
    assert g.task_to_id == {"transcribe": V.TRANSCRIBE, "translate": V.TRANSLATE}
    assert g.suppress_tokens == V.SUPPRESS_TOKENS and g.eos_token_id == V.EOS
    s = V.generation_settings()
    assert (s.no_timestamps_token_id, s.lang_first, s.lang_last, s.task_to_id) == (
        g.no_timestamps_token_id, g.lang_first, g.lang_last, g.task_to_id)


def test_english_only_checkpoint_rejected():
    model, _ = V.hf_model("varied")
    model.generation_config = V.hf_generation_config(is_multilingual=False)
    with pytest.raises(ValueError, match="English-only"):
        B200WhisperPipeline.from_hf_model(model, V.build_tokenizer(), scheduler=_NoEngine())
    # a generation config without the field is read as before
    model.generation_config = V.hf_generation_config()
    del model.generation_config.is_multilingual
    assert getattr(model.generation_config, "is_multilingual", None) is None
    B200WhisperPipeline.from_hf_model(model, V.build_tokenizer(), scheduler=_NoEngine())


def test_dims_presets_and_validation():
    for name, d, heads, layers in (("large_v2", 1280, 20, 32), ("medium", 1024, 16, 24), ("small", 768, 12, 12),
                                   ("base", 512, 8, 6)):
        dims = getattr(WhisperDims, name)()
        assert (dims.d_model, dims.heads, dims.dec_layers, dims.n_mels, dims.vocab) == (d, heads, layers, 80, 51865)
        dims.validate()
    WhisperDims.large_v3().validate()
    with pytest.raises(ValueError, match="80 or 128 mel bins"):
        WhisperDims(n_mels=64).validate()
    with pytest.raises(ValueError, match="multiples of 256"):      # whisper-tiny (d_model 384) keeps its error
        WhisperDims(d_model=384, heads=6, ffn=1536, enc_layers=4, dec_layers=4, n_mels=80, vocab=51865).validate()


class OracleSchedulerV2:
    """Engine stand-in returning the oracle's token ids for the 80-mel model (v2 ids)."""

    def __init__(self, variant):
        self.ref = R.WhisperRef(V.ref_dims(), V.variant_state_dict(V.ref_dims(), variant))
        self.last_stats = {}

    def run(self, clips, task="transcribe", language=None, return_timestamps=True, token_timestamps=False, group=None,
            num_beams=1):
        assert not token_timestamps
        feats = torch.stack([torch.from_numpy(V.log_mel(c)) for c in clips])
        return self.ref.generate(feats, task=task, gc=V.gen_config(), return_timestamps=return_timestamps,
                                 num_beams=num_beams)


@pytest.fixture(scope="module")
def wav(tmp_path_factory):
    p = tmp_path_factory.mktemp("audio") / "golden_v2_71s.wav"
    helpers.write_wav16(p, np.concatenate(_clips()))
    return str(p)


@pytest.mark.parametrize("variant,cl,st,bs,ts", [("varied", 30, 5, 24, True), ("varied", 60, 5, 32, None),
                                                 ("decisive", 60, 5, 32, True), ("decisive", 30, 5, 24, None)])
def test_host_pipeline_matches_hf_golden_v2(wav, variant, cl, st, bs, ts):
    g = json.load(open(os.path.join(GOLD, "pipeline_v2_tiny.json")))[f"{variant}_{cl}_{st}_{bs}_{'ts' if ts else 'nots'}"]
    pipe = B200WhisperPipeline(None, WhisperDims(**V.TINY_V2), V.build_tokenizer(), generation=V.generation_settings(),
                               scheduler=OracleSchedulerV2(variant))
    kw = {"return_timestamps": True} if ts else {}
    r = pipe(wav, chunk_length_s=cl, stride_length_s=st, batch_size=bs, generate_kwargs={"task": "transcribe"}, **kw)
    assert sorted(r.keys()) == g["keys"] and r["text"] == g["text"]
    if ts:
        assert [{"timestamp": list(c["timestamp"]), "text": c["text"]} for c in r["chunks"]] == g["chunks"]
