"""CPU drop-in test at the reference's model construction (SURVEY.md §8b / §8c recipe): `install()` patches the
`transformers.pipeline` factory, and the call the reference's `load_transcription_model` makes
(`pipeline("automatic-speech-recognition", model=model_name, device=device, torch_dtype=...)`,
ref:vocalis/core/audio_pipeline.py:187-200, quoted in turbo-whisper-workspace_b200/install.py) returns a
`B200WhisperPipeline`.  Called the way the reference's `transcribe()` calls it (chunk_length_s=60, batch_size=32,
stride_length_s=5, generate_kwargs={"task": ...}, return_timestamps=True; ref:vocalis/core/audio_pipeline.py:351-358),
that object must return the text and segments the reference's own `process_audio` returned with the transformers
pipeline object (stored in tests/golden/pipeline_tiny.json, `reference_process_audio_varied`, by
tests/golden/make_golden.py).  The GPU engines are replaced by the oracle scheduler of tests/test_pipeline_host_golden.py,
so the comparison is exact."""
import json
import os

import numpy as np
import torch

import helpers
from test_pipeline_host_golden import GOLD, OracleScheduler
from turbo_whisper_workspace_b200.config import WhisperDims
from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline


def test_zero_touch_install_through_load_transcription_model(tmp_path, monkeypatch):
    """INTEGRATION.md §1 option (ii): with `install()` in place, the reference's model construction (default model name
    "openai/whisper-large-v3") yields the B200 pipeline object, other tasks / models are forwarded to the original factory,
    and `uninstall()` puts the original back."""
    # importing `pipeline` from transformers the first time replaces its lazy top-level module in sys.modules: do it
    # before binding the module object that gets patched
    from transformers import pipeline  # noqa: F401
    import transformers
    import turbo_whisper_workspace_b200.install as twb
    gold = json.load(open(os.path.join(GOLD, "pipeline_tiny.json")))["reference_process_audio_varied"]
    pcm = np.concatenate([helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"),
                          helpers.synth_clip(2, seconds=11.3, kind="mod")])
    wav = tmp_path / "golden_71s.wav"
    helpers.write_wav16(wav, pcm)
    forwarded = []
    monkeypatch.setattr(transformers, "pipeline", lambda task=None, model=None, *a, **k: forwarded.append((task, model)) or "lib")
    loaded = []

    def loader(model, tokenizer=None):
        loaded.append(model)
        return "hf-model-stand-in", helpers.build_tokenizer()

    def builder(hf_model, tokenizer):
        assert hf_model == "hf-model-stand-in"
        return B200WhisperPipeline(None, WhisperDims(**helpers.TINY), tokenizer, scheduler=OracleScheduler("varied"))
    twb.install(devices=["cuda:0"], loader=loader, builder=builder)
    try:
        assert transformers.pipeline("text-classification", model="bert") == "lib" and forwarded == [("text-classification", "bert")]
        assert transformers.pipeline("automatic-speech-recognition", model="facebook/wav2vec2-base") == "lib"
        # the reference's load_transcription_model: `from transformers import pipeline` at call time, then this call
        from transformers import pipeline
        model = pipeline("automatic-speech-recognition", model="openai/whisper-large-v3", device="cpu",
                         torch_dtype=torch.float32)
        assert isinstance(model, B200WhisperPipeline)
        assert loaded == ["openai/whisper-large-v3"]            # the reference's default model name
        # the reference's transcribe() call
        res = model(str(wav), chunk_length_s=60, batch_size=32, stride_length_s=5,
                    generate_kwargs={"task": "transcribe"}, return_timestamps=True)
        assert res["text"] == gold["text"]
        assert [{"timestamp": list(c["timestamp"]), "text": c["text"]} for c in res["chunks"]] == gold["segments"]
    finally:
        twb.uninstall()
    assert transformers.pipeline("x", model="y") == "lib"       # the original factory is back
    # install(num_beams=5): the drop-in object decodes like the reference's literal call under transformers >= 4.53
    twb.install(devices=["cuda:0"], loader=loader, builder=builder, num_beams=5)
    try:
        assert transformers.pipeline("automatic-speech-recognition", model="openai/whisper-large-v3").num_beams == 5
    finally:
        twb.uninstall()
