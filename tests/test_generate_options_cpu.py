"""CPU tests of a generate call's options: config.resolve_generate_options (every error it raises, with its exact text,
and the values the engine uses), the row-length check of engine.init_rows, the engine entries checking their options
before any device work, and the pipeline's one keyword dict reaching the engines untouched through every scheduler
shape."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import helpers
from turbo_whisper_workspace_b200 import _lib
from turbo_whisper_workspace_b200 import scheduler as S
from turbo_whisper_workspace_b200.config import GenerationSettings, WhisperDims, resolve_generate_options
from turbo_whisper_workspace_b200.engine import WhisperEngine, init_rows
from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline

DIMS = WhisperDims(**helpers.TINY)
EN, FR, SOT_PREV = 50259, 50265, 50361
LONG_FORM = "long-form generate takes one clip, needs timestamps and has no token timestamps"


def _gen():
    return GenerationSettings(lang_to_id={"<|en|>": EN, "<|fr|>": FR})


def _resolve(**kw):
    return resolve_generate_options(DIMS, _gen(), **kw)


@pytest.mark.parametrize("kw, message", [
    (dict(task="summarize"),
     "The `summarize` task is not supported. The task should be one of ['transcribe', 'translate']"),
    (dict(language="xx"), "Unsupported language: xx"),
    (dict(language="<|xx|>"), "Unsupported language: <|xx|>"),
    (dict(prompt_ids=[]), "`prompt_ids` is empty"),
    (dict(prompt_ids=[[SOT_PREV, 1]]), "`prompt_ids` must be a 1-D sequence of token ids, got shape (1, 2)"),
    (dict(prompt_ids=np.zeros((2, 2), dtype=np.int64)), "`prompt_ids` must be a 1-D sequence of token ids, got shape (2, 2)"),
    (dict(prompt_ids=[0.5, 1.0]), "`prompt_ids` must hold integer token ids, got dtype float64"),
    (dict(prompt_ids=[SOT_PREV, 51866, -1]), "`prompt_ids` holds ids outside the vocabulary [0, 51866): [51866, -1]"),
    (dict(prompt_ids=[SOT_PREV] + [400] * 444),
     "The decoder input (prompt_ids and the 3 special start tokens) has 448 positions; it must be shorter than 448 "
     "(min(max_length, max_target_positions)). Shorten the prompt."),
    (dict(prompt_ids=[SOT_PREV] + [400] * 443, return_timestamps=False),
     "The decoder input (prompt_ids and the 4 special start tokens) has 448 positions; it must be shorter than 448 "
     "(min(max_length, max_target_positions)). Shorten the prompt."),
    (dict(long_form=True, return_timestamps=False), LONG_FORM),
    (dict(long_form=True, token_timestamps=True), LONG_FORM),
])
def test_resolve_generate_options_errors(kw, message):
    with pytest.raises(ValueError) as e:
        _resolve(**kw)
    assert str(e.value) == message


def test_resolve_generate_options_values():
    o = _resolve()
    assert (o.task_id, o.lang_id, o.timestamps, o.num_beams, o.token_timestamps, o.prompt_ids, o.prompt_len) == \
        (50360, -1, True, 1, False, None, 3)                         # language detected, timestamps on
    o = _resolve(task="translate", language="fr", num_beams=3)
    assert (o.task_id, o.lang_id, o.num_beams) == (50359, FR, 3)
    assert _resolve(language="<|en|>").lang_id == EN
    # timestamps off: <|notimestamps|> joins the prompt; a numpy / torch prompt becomes a list of ints
    for ids in ([SOT_PREV, 400, 401], np.asarray([SOT_PREV, 400, 401]), torch.tensor([SOT_PREV, 400, 401])):
        o = _resolve(return_timestamps=False, prompt_ids=ids)
        assert (o.timestamps, o.prompt_ids, o.prompt_len) == (False, [SOT_PREV, 400, 401], 4 + 3)
        assert all(type(v) is int for v in o.prompt_ids)
    o = _resolve(prompt_ids=[SOT_PREV] + [400] * 443, token_timestamps=True)
    assert (o.prompt_len, o.token_timestamps) == (447, True)      # the longest prompt that leaves a position
    assert _resolve(long_form=True, prompt_ids=[SOT_PREV]).prompt_len == 4


def _grammar():
    g = _lib.Grammar()
    g.pad, g.ts_begin, g.max_initial_ts = 9, 100, 50
    return g


@pytest.mark.parametrize("timestamps, prefilled, flat", [(True, True, False), (False, False, False), (True, True, True),
                                                         (False, True, True)])
def test_init_rows_rejects_rows_that_leave_no_position(timestamps, prefilled, flat):
    """decode / decode_beams called directly with prompt_ids: the row length is checked against the token buffer."""
    specials = [1, 2, 3] + ([] if timestamps else [4])
    ok = torch.tensor([[7] * (7 - len(specials)) + specials])
    assert init_rows(ok, 8, _grammar(), timestamps, prefilled=prefilled, flat=flat)[3] == 7
    with pytest.raises(ValueError) as e:
        init_rows(torch.tensor([[7] * (8 - len(specials)) + specials]), 8, _grammar(), timestamps, prefilled=prefilled,
                  flat=flat)
    assert str(e.value) == (f"The decoder input (prompt_ids and the {len(specials)} special start tokens) has 8 positions; "
                            "it must be shorter than 8 (min(max_length, max_target_positions)). Shorten the prompt.")


def test_engine_entries_check_options_before_device_work():
    """An invalid call fails before the H2D copy and the log-mel launch of generate_from_pcm / generate_long_from_pcm,
    and before the seek loop of generate."""
    work = []
    eng = SimpleNamespace(dims=DIMS, gen=_gen(), stream=None, load_pcm=lambda clips: work.append("load_pcm"),
                          logmel=SimpleNamespace(long=lambda audio: work.append("logmel.long")),
                          _seek=lambda *a, **kw: work.append("seek"))
    clip = np.zeros(16000, np.float32)
    with pytest.raises(ValueError, match="task is not supported"):
        WhisperEngine.generate_from_pcm(eng, [clip], task="summarize")
    with pytest.raises(ValueError, match="Unsupported language: xx"):
        WhisperEngine.generate_long_from_pcm(eng, np.zeros(16000 * 40, np.float32), language="xx")
    with pytest.raises(ValueError) as e:
        WhisperEngine.generate_long_from_pcm(eng, np.zeros(16000 * 40, np.float32), token_timestamps=True)
    assert str(e.value) == LONG_FORM
    with pytest.raises(ValueError, match="`prompt_ids` is empty"):
        WhisperEngine.generate(eng, 2, prompt_ids=[])
    with pytest.raises(ValueError) as e:
        WhisperEngine.generate(eng, 2, long_mel=torch.zeros(4000, 128))
    assert str(e.value) == LONG_FORM
    assert work == []


class RecordingEngine:
    """Engine stand-in: records the keywords of every call."""

    def __init__(self, device, max_batch=8):
        self.device, self.max_batch, self.calls = device, max_batch, []

    def generate_from_pcm(self, clips, **kw):
        assert len(clips) <= self.max_batch
        self.calls.append(("generate_from_pcm", len(clips), kw))
        ids = [50365, 300, 301, 50465]
        return [(ids, [0.0, 0.5, 1.0, 1.5]) if kw.get("token_timestamps") else ids for _ in clips]

    def generate_long_from_pcm(self, audio, **kw):
        self.calls.append(("generate_long_from_pcm", 1, kw))
        return [50365, 300, 301, 50465]


def _window_scheduler():
    return S.WindowScheduler(None, None, None, devices=["d0", "d1"], engine_factory=lambda d: RecordingEngine(d),
                             contexts_per_device=2)


SHAPES = {
    "window": _window_scheduler,
    "distributed_over_window": lambda: S.DistributedWindowScheduler(_window_scheduler(), rank=0, world_size=1),
    "distributed_over_engine": lambda: S.DistributedWindowScheduler(RecordingEngine("g"), rank=0, world_size=1),
}

CHUNKED = dict(chunk_length_s=30, stride_length_s=5, batch_size=3)
PROMPT = [SOT_PREV, 400, 401]
# (pipeline call, keywords every engine call must receive, windows per engine call at most)
MODES = {
    "greedy": (dict(CHUNKED, return_timestamps=True), dict(task="transcribe", language=None), 8),
    "no_timestamps": (dict(CHUNKED, generate_kwargs={"language": "en"}),
                      dict(task="transcribe", language="en", return_timestamps=False), 8),
    "beams3": (dict(CHUNKED, return_timestamps=True, generate_kwargs={"num_beams": 3, "task": "translate"}),
               dict(task="translate", language=None, num_beams=3), 2),
    "word": (dict(CHUNKED, return_timestamps="word"), dict(task="transcribe", language=None, token_timestamps=True), 3),
    "prompt": (dict(CHUNKED, return_timestamps=True, generate_kwargs={"prompt_ids": np.asarray(PROMPT)}),
               dict(task="transcribe", language=None, prompt_ids=PROMPT), 8),
    "longform": (dict(return_timestamps=True, generate_kwargs={"prompt_ids": torch.tensor(PROMPT), "num_beams": 2}),
                 dict(task="transcribe", language=None, num_beams=2, prompt_ids=PROMPT), 1),
}


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("mode", list(MODES))
def test_engines_receive_the_pipelines_keywords(shape, mode):
    """The schedulers forward the pipeline's keywords untouched; ``num_beams`` sizes the micro-batches and ``group``
    (word timestamps) makes them the HF pipeline's batches."""
    call, want, most = MODES[mode]
    sched = SHAPES[shape]()
    pipe = B200WhisperPipeline(None, DIMS, helpers.build_tokenizer(), _gen(), scheduler=sched)
    audio = helpers.synth_clip(3, seconds=100.0)
    r = pipe(audio, **call)
    assert isinstance(r["text"], str)
    calls = [c for e in sched.flat_engines for c in e.calls]
    kind = "generate_long_from_pcm" if mode == "longform" else "generate_from_pcm"
    assert calls and all(c[0] == kind and c[2] == want for c in calls), calls
    sizes = [c[1] for c in calls]
    n_win = 1 if mode == "longform" else len(pipe.last_token_rows)
    assert sum(sizes) == n_win and max(sizes) <= most
    if mode == "word":
        assert sorted(sizes, reverse=True) == [3] * (n_win // 3) + ([n_win % 3] if n_win % 3 else [])


def test_pipeline_rejects_task_and_language_before_audio_ingest():
    calls = []

    class Sched:
        last_stats = {}

        def run(self, clips, **kw):
            calls.append(kw)
            return [[] for _ in clips]
    pipe = B200WhisperPipeline(None, DIMS, helpers.build_tokenizer(), _gen(), scheduler=Sched())
    with pytest.raises(ValueError) as e:      # 12 is no audio input: ingest would raise TypeError
        pipe(12, generate_kwargs={"task": "summarize"})
    assert str(e.value) == "The `summarize` task is not supported. The task should be one of ['transcribe', 'translate']"
    with pytest.raises(ValueError) as e:
        pipe(12, generate_kwargs={"language": "xx"})
    assert str(e.value) == "Unsupported language: xx"
    assert calls == []
