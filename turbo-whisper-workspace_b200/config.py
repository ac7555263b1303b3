"""Model dimensions and generation settings of the Whisper checkpoints the path serves.

Mirrors the fields of ``WhisperConfig`` / ``generation_config.json`` that the hot path reads
(SURVEY.md §8: large-v3-turbo = 32 encoder / 4 decoder layers, large-v3 = 32 / 32).  The 128-mel checkpoints
(large-v3, large-v3-turbo, distil-large-v3) and the multilingual 80-mel ones (large-v2, distil-large-v2, medium, small,
base) are served; ``n_mels`` carries the difference down to the log-mel kernels and the conv stem."""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional

N_SAMPLES = 480000   # 30 s at 16 kHz
MEL_BINS = (80, 128)  # filterbank sizes the log-mel kernels are built for
N_FRAMES = 3000      # mel frames per window
SAMPLING_RATE = 16000

# generation_config.json of openai/whisper-large-v3(-turbo) (SURVEY.md §8)
_SUPPRESS = [
    1, 2, 7, 8, 9, 10, 14, 25, 26, 27, 28, 29, 31, 58, 59, 60, 61, 62, 63, 90, 91, 92, 93, 359, 503, 522, 542, 873,
    893, 902, 918, 922, 931, 1350, 1853, 1982, 2460, 2627, 3246, 3253, 3268, 3536, 3846, 3961, 4183, 4667, 6585, 6647,
    7273, 9061, 9383, 10428, 10929, 11938, 12033, 12331, 12562, 13793, 14157, 14635, 15265, 15618, 16553, 16604, 18362,
    18956, 20075, 21675, 22520, 26130, 26161, 26435, 28279, 29464, 31650, 32302, 32470, 36865, 42863, 47425, 49870,
    50254, 50258, 50359, 50360, 50361, 50362, 50363,
]


# generation_config.alignment_heads of the two checkpoints (from memory of the hub files, as the suppress list above —
# verify when a checkpoint is available; GenerationSettings.from_hf copies the real field).  Used by tools/ only.
ALIGNMENT_HEADS = {
    "large-v3-turbo": [[2, 4], [2, 11], [3, 3], [3, 6], [3, 11], [3, 14]],
    "large-v3": [[7, 0], [10, 17], [12, 18], [13, 12], [16, 1], [17, 14], [19, 11], [21, 4], [24, 1], [25, 6]],
}


@dataclass
class WhisperDims:
    d_model: int = 1280
    heads: int = 20
    ffn: int = 5120
    enc_layers: int = 32
    dec_layers: int = 4
    n_mels: int = 128
    max_source_positions: int = 1500
    max_target_positions: int = 448
    vocab: int = 51866

    def validate(self) -> None:
        if self.d_model != self.heads * 64:
            raise ValueError("turbo-whisper-workspace_b200 kernels are built for head_dim 64")
        if self.d_model % 256 or self.ffn % 256:
            raise ValueError("d_model and ffn must be multiples of 256")
        if self.n_mels not in MEL_BINS:
            raise ValueError(f"the log-mel kernels are built for 80 or 128 mel bins, not {self.n_mels}")
        if self.max_source_positions != 1500:
            raise ValueError("the conv-stem kernels are built for 1500 source positions")
        if self.max_target_positions > 448:
            raise ValueError("max_target_positions > 448 is not supported")

    @classmethod
    def large_v3_turbo(cls) -> "WhisperDims":
        return cls()

    @classmethod
    def large_v3(cls) -> "WhisperDims":
        return cls(dec_layers=32)

    # the 80-mel checkpoints: openai/whisper-large-v2 (distil-whisper/distil-large-v2 is large_v2() with 2 decoder
    # layers), openai/whisper-medium, -small and -base; their vocabulary has 51865 ids (no <|yue|>)
    @classmethod
    def large_v2(cls) -> "WhisperDims":
        return cls(dec_layers=32, n_mels=80, vocab=51865)

    @classmethod
    def medium(cls) -> "WhisperDims":
        return cls(d_model=1024, heads=16, ffn=4096, enc_layers=24, dec_layers=24, n_mels=80, vocab=51865)

    @classmethod
    def small(cls) -> "WhisperDims":
        return cls(d_model=768, heads=12, ffn=3072, enc_layers=12, dec_layers=12, n_mels=80, vocab=51865)

    @classmethod
    def base(cls) -> "WhisperDims":
        return cls(d_model=512, heads=8, ffn=2048, enc_layers=6, dec_layers=6, n_mels=80, vocab=51865)

    @classmethod
    def from_hf_config(cls, cfg) -> "WhisperDims":
        return cls(d_model=cfg.d_model, heads=cfg.encoder_attention_heads, ffn=cfg.encoder_ffn_dim,
                   enc_layers=cfg.encoder_layers, dec_layers=cfg.decoder_layers, n_mels=cfg.num_mel_bins,
                   max_source_positions=cfg.max_source_positions, max_target_positions=cfg.max_target_positions,
                   vocab=cfg.vocab_size)


@dataclass
class GenerationSettings:
    eos_token_id: int = 50257
    pad_token_id: int = 50257
    decoder_start_token_id: int = 50258
    no_timestamps_token_id: int = 50364
    max_length: int = 448
    max_initial_timestamp_index: int = 50
    suppress_tokens: List[int] = field(default_factory=lambda: list(_SUPPRESS))
    begin_suppress_tokens: List[int] = field(default_factory=lambda: [220, 50257])
    lang_first: int = 50259
    lang_last: int = 50358
    task_to_id: Dict[str, int] = field(default_factory=lambda: {"transcribe": 50360, "translate": 50359})
    lang_to_id: Dict[str, int] = field(default_factory=dict)  # "<|en|>" -> id, optional (explicit language)
    # word-level timestamps: (decoder layer, head) pairs of generation_config.alignment_heads (None: not available, as
    # for a generation config without the field) and WhisperConfig.median_filter_width
    alignment_heads: Optional[List[List[int]]] = None
    median_filter_width: int = 7

    @property
    def timestamp_begin(self) -> int:
        return self.no_timestamps_token_id + 1

    @classmethod
    def from_hf(cls, gc) -> "GenerationSettings":
        """From a transformers GenerationConfig carrying the Whisper fields."""
        s = cls()
        for name in ("eos_token_id", "pad_token_id", "decoder_start_token_id", "no_timestamps_token_id", "max_length",
                     "max_initial_timestamp_index"):
            v = getattr(gc, name, None)
            if v is not None:
                setattr(s, name, int(v[0] if isinstance(v, (list, tuple)) else v))
        if getattr(gc, "suppress_tokens", None) is not None:
            s.suppress_tokens = [int(t) for t in gc.suppress_tokens]
        if getattr(gc, "begin_suppress_tokens", None) is not None:
            s.begin_suppress_tokens = [int(t) for t in gc.begin_suppress_tokens]
        if getattr(gc, "task_to_id", None):
            s.task_to_id = {k: int(v) for k, v in gc.task_to_id.items()}
        if getattr(gc, "lang_to_id", None):
            s.lang_to_id = {k: int(v) for k, v in gc.lang_to_id.items()}
            ids = sorted(s.lang_to_id.values())
            if ids != list(range(ids[0], ids[-1] + 1)):
                raise ValueError("language ids must be contiguous")
            s.lang_first, s.lang_last = ids[0], ids[-1]
        if getattr(gc, "alignment_heads", None) is not None:
            s.alignment_heads = [[int(l), int(h)] for l, h in gc.alignment_heads]
        return s


def validate_prompt_ids(prompt_ids, vocab: int) -> List[int]:
    """``prompt_ids`` of generate (list / numpy / torch, normally ``[<|startofprev|>, text ids...]``) -> list of ints.
    Raises ValueError unless it is a non-empty 1-D sequence of integer ids in [0, vocab)."""
    import numpy as np
    if hasattr(prompt_ids, "detach"):
        prompt_ids = prompt_ids.detach().cpu().numpy()
    arr = np.asarray(prompt_ids)
    if arr.ndim != 1:
        raise ValueError(f"`prompt_ids` must be a 1-D sequence of token ids, got shape {tuple(arr.shape)}")
    if arr.size == 0:
        raise ValueError("`prompt_ids` is empty")
    if not (np.issubdtype(arr.dtype, np.integer) or arr.dtype == object and all(isinstance(v, (int, np.integer)) for v in arr)):
        raise ValueError(f"`prompt_ids` must hold integer token ids, got dtype {arr.dtype}")
    ids = [int(v) for v in arr]
    bad = [v for v in ids if not 0 <= v < vocab]
    if bad:
        raise ValueError(f"`prompt_ids` holds ids outside the vocabulary [0, {vocab}): {bad[:8]}")
    return ids


def decoder_prompt_len(n_prompt_ids: int, timestamps: bool, max_len: int) -> int:
    """Positions of the decoder input prompt_ids + [<|startoftranscript|>, language, task] (+ <|notimestamps|>)
    ($TF/models/whisper/generation_whisper.py:1909-1913) for ``n_prompt_ids`` prompt ids.  ``max_len`` =
    min(max_length, max_target_positions): the prompt counts against it, so a long prompt leaves fewer positions to
    generate.  ValueError unless the input is shorter than ``max_len`` (HF indexes past its positional embedding there)."""
    n = (3 if timestamps else 4) + n_prompt_ids
    if n >= max_len:
        raise ValueError(f"The decoder input (prompt_ids and the {3 if timestamps else 4} special start tokens) has "
                         f"{n} positions; it must be shorter than {max_len} (min(max_length, max_target_positions)). "
                         "Shorten the prompt.")
    return n


@dataclass(frozen=True)
class GenerateOptions:
    """A call's decoding options as the engine uses them (:func:`resolve_generate_options`)."""
    task_id: int
    lang_id: int                        # -1: detect the language
    timestamps: bool
    num_beams: int
    token_timestamps: bool
    prompt_ids: Optional[List[int]]
    prompt_len: int                     # P: positions of the decoder prompt, special tokens included


def resolve_generate_options(dims: WhisperDims, gen: GenerationSettings, *, task: str = "transcribe",
                             language: Optional[str] = None, return_timestamps: bool = True, num_beams: int = 1,
                             token_timestamps: bool = False, prompt_ids=None, long_form: bool = False) -> GenerateOptions:
    """The one check of a generate call's options, before any device work; ValueError for an invalid call.
    ``task``: a key of ``gen.task_to_id``.  ``language``: ``"en"`` or ``"<|en|>"`` (a key of ``gen.lang_to_id``),
    None = detect it.  ``return_timestamps``: False = <|notimestamps|> joins the prompt and the timestamp grammar is
    off.  ``num_beams`` > 1: beam search.  ``token_timestamps``: per-token times from the alignment heads (word
    timestamps).  ``prompt_ids``: generate(prompt_ids=...), see :func:`validate_prompt_ids`.  ``long_form``: one
    un-chunked clip longer than 30 s, which needs timestamps and has no token timestamps."""
    if prompt_ids is not None:
        prompt_ids = validate_prompt_ids(prompt_ids, dims.vocab)
    if long_form and (token_timestamps or not return_timestamps):
        raise ValueError("long-form generate takes one clip, needs timestamps and has no token timestamps")
    if task not in gen.task_to_id:
        raise ValueError(f"The `{task}` task is not supported. The task should be one of {list(gen.task_to_id)}")
    lang_id = -1
    if language is not None:
        key = language if language.startswith("<|") else f"<|{language}|>"
        if key not in gen.lang_to_id:
            raise ValueError(f"Unsupported language: {language}")
        lang_id = gen.lang_to_id[key]
    timestamps = bool(return_timestamps)
    P = decoder_prompt_len(0 if prompt_ids is None else len(prompt_ids), timestamps,
                           min(gen.max_length, dims.max_target_positions))
    return GenerateOptions(gen.task_to_id[task], lang_id, timestamps, int(num_beams), bool(token_timestamps), prompt_ids, P)
