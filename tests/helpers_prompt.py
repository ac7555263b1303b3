"""Prompt-aware reference generate (generate(prompt_ids=...)) on top of the fp32 CPU oracle, for the prompt tests.

WhisperRef.greedy / beam_search already run any multi-token decoder prompt as one forward; what a text prompt changes
is the seek loop around them ($TF/models/whisper/generation_whisper.py:1853-1918, :1141): the language is detected on
[<|startoftranscript|>] alone, every seek iteration's decoder input is prompt_ids + [SOT, language, task]
(+ <|notimestamps|>), and the returned ids exclude it.  :func:`prompted_generate` is oracle.whisper_ref's generate with
that input; the oracle module itself is unchanged."""
from __future__ import annotations

import json
import os
from typing import List, Optional, Sequence

import torch

from oracle import whisper_ref as R

HERE = os.path.dirname(os.path.abspath(__file__))
PREV = 50361   # <|startofprev|>


def golden():
    with open(os.path.join(HERE, "golden", "prompt_tiny.json")) as f:
        return json.load(f)


def lang_id(language: Optional[str]) -> Optional[int]:
    if language is None:
        return None
    from transformers.models.whisper.tokenization_whisper import LANGUAGES
    return R.LANG_FIRST + list(LANGUAGES).index(language)


def prompted_generate(ref: "R.WhisperRef", feats: torch.Tensor, prompt_ids: Sequence[int], task: str = "transcribe",
                      language: Optional[int] = None, return_timestamps: bool = True, num_beams: int = 1,
                      gc: Optional["R.GenConfig"] = None, trace: Optional[dict] = None, alignment_heads=None,
                      num_frames: Optional[Sequence[int]] = None, token_ts: Optional[dict] = None) -> List[List[int]]:
    """WhisperRef.generate with ``prompt_ids`` prepended to the decoder input of every seek iteration (the language id
    is detected on [SOT] when ``language`` is None).  Same outputs and trace layout as WhisperRef.generate."""
    gc = gc or R.GenConfig()
    TB = gc.no_timestamps_token_id + 1
    B = feats.shape[0]
    feats = feats.to(torch.float32)
    enc0 = ref.encode(feats[..., :3000])
    langs = ref.detect_language(enc0, gc) if language is None else [int(language)] * B
    tail = [] if return_timestamps else [gc.no_timestamps_token_id]
    init = torch.tensor([list(prompt_ids) + [gc.decoder_start_token_id, langs[b], gc.task_to_id[task]] + tail
                         for b in range(B)], dtype=torch.long)
    P = init.shape[1]
    seek = [0] * B
    max_frames = [feats.shape[-1]] * B
    out: List[List[int]] = [[] for _ in range(B)]
    if trace is not None:
        trace.update({"langs": langs, "iterations": [], "P": P})
    guard = 0
    while any(s < m for s, m in zip(seek, max_frames)):
        guard += 1
        assert guard <= 64, "seek loop does not advance"
        rows = [b for b in range(B) if seek[b] < max_frames[b]]
        nfr = {b: min(max_frames[b] - seek[b], 3000) for b in rows}
        seg = torch.zeros(len(rows), feats.shape[1], 3000)
        for i, b in enumerate(rows):
            seg[i, :, :nfr[b]] = feats[b, :, seek[b]:seek[b] + nfr[b]]
        enc = enc0 if guard == 1 else ref.encode(seg)
        rec = [] if trace is not None else None
        cross = [[] for _ in range(ref.dims.dec_layers)] if alignment_heads is not None else None
        if num_beams > 1:
            toks = ref.beam_search(enc, init[rows], gc, num_beams=num_beams, timestamps=return_timestamps)
        else:
            toks = ref.greedy(enc, init[rows], gc, record=rec, timestamps=return_timestamps, cross=cross)
        if cross is not None:
            tt = ref.token_timestamps(cross, alignment_heads, len(rows), P,
                                      [int(num_frames[b]) - seek[b] for b in rows])
        if trace is not None:
            trace["iterations"].append({"rows": rows, "seek": [seek[b] for b in rows], "tokens": toks.clone(),
                                        "record": rec})
        for i, b in enumerate(rows):
            s = toks[i].tolist()
            if s[-1] == gc.pad_token_id:
                n_pad = sum(1 for t in s if t == gc.pad_token_id)
                if gc.pad_token_id == gc.eos_token_id:
                    n_pad -= 1
                if n_pad:
                    s = s[:-n_pad]
            if s[-1] == gc.eos_token_id:
                s = s[:-1]
            segs, adv = ref.retrieve_segment(s, nfr[b], TB)
            if cross is not None and token_ts is not None:
                n_kept = sum(len(sg) for sg in segs)
                off = torch.tensor(seek[b], dtype=torch.float64) * 0.02 / 2
                token_ts.setdefault("segments", [[] for _ in range(B)])[b].extend((tt[i, P:P + n_kept] + off).tolist())
            seek[b] += adv
            for sg in segs:
                out[b].extend(sg)
    return out


def strip_hf(row: Sequence[int], pad: int = R.EOS) -> List[int]:
    """A row of HF's padded short-form `sequences` -> the generated ids the seek loop keeps (no eos / padding)."""
    s = list(row)
    while s and s[-1] == pad:
        s.pop()
    return s


def compare_prompted_traces(ref_trace, eng_trace, margin_tol: float):
    """helpers.compare_generate_traces for prompted rows: the engine's rows carry the P-position decoder input."""
    P = ref_trace["P"]
    assert eng_trace["langs"] == ref_trace["langs"], "language detection differs"
    alive, agreed, first_diffs = None, 0, {}
    for k, it in enumerate(ref_trace["iterations"]):
        rows = list(it["rows"])
        if alive is None:
            alive = set(rows)
        if not any(b in alive for b in rows):
            break
        e = eng_trace["iterations"][k]
        for i, b in enumerate(rows):
            if b not in alive:
                continue
            ei = e["rows"].index(b)
            assert e["seek"][ei] == it["seek"][i], f"row {b}: seek differs at iteration {k}"
            want = [int(t) for t in it["tokens"][i].tolist()]
            got = [int(t) for t in e["tokens"][ei][P:P + len(want)]]
            for g, t in enumerate(want):
                if g >= len(it["record"]):
                    break
                if got[g] != t:
                    rec = it["record"][g]
                    decisive = float(rec["margin"][i]) > margin_tol and float(rec["rule_gap"][i]) > margin_tol
                    assert not decisive, (f"row {b} diverges at DECISIVE step {g} of iteration {k}: margin "
                                          f"{float(rec['margin'][i]):.3f}")
                    first_diffs[b] = (k, g, float(rec["margin"][i]))
                    alive.discard(b)
                    break
                agreed += 1
    return agreed, sorted(alive or []), first_diffs
