"""Per-GPU Whisper engine: weight packing, workspaces, encoder forward, CUDA-graphed greedy decode
and the short-form seek loop — all arithmetic through the C ABI (include/twb200.h).

Host logic restated from transformers 5.5.0 (`$TF/`):
  * WhisperGenerationMixin.generate seek loop      $TF/models/whisper/generation_whisper.py:785-903
  * detect_language / _retrieve_init_tokens        $TF/models/whisper/generation_whisper.py:1610-1673, 1455-1608
  * _retrieve_segment                              $TF/models/whisper/generation_whisper.py:1976-2073
  * generate_with_fallback pad / eos stripping     $TF/models/whisper/generation_whisper.py:1063-1086
PyTorch supplies device memory, streams and CUDA-graph capture; nothing here computes with torch ops
on the data path (tensor allocation, H2D / D2H copies and int bookkeeping only).
"""
from __future__ import annotations

import os

import ctypes as C
import threading
from typing import Callable, Dict, List, Optional, Sequence, Union

import numpy as np
import torch

from . import _lib, ops
from ._lib import Grammar, SkinnyArgs, check
from .config import (N_FRAMES, N_SAMPLES, GenerateOptions, GenerationSettings, WhisperDims, decoder_prompt_len,
                     resolve_generate_options)

MAX_DECODE_BATCH = 96   # decode rows per engine context (projections: up to tw_dec_max_rows(); the LM head runs per 48-row chunk)
LMHEAD_ROWS = 48
_CAPTURE_LOCK = threading.Lock()   # CUDA-graph capture is serialised across the engine contexts of a process
_PREFILL_WEIGHTS_LOCK = threading.Lock()   # the contexts of a device share (and lazily extend) one weight dict
PAGE = 64
ROW_STATE = np.dtype(_lib.RowState)   # tw_row_state of include/twb200.h as a numpy record


def _bf16(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).to(torch.bfloat16).contiguous()


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


def pack_skinny_weight(w: torch.Tensor) -> torch.Tensor:
    """[N, K] bf16 (nn.Linear layout) -> FRAGMENT-MAJOR layout of the decode GEMMs (csrc/decode.cu, frag_ptr):
    ``[slab = N/16][k-step = K/32][half: rows g | rows g+8][g = 0..7][tg = 0..3][8]`` with
    element = W[16*slab + 8*half + g][32*kstep + 8*tg + e]; N is zero-padded to a multiple of 16.  The result keeps
    the 2-D shape [N_padded, K] (same bytes, different order) so that ``shape[0]`` / ``shape[1]`` still describe it."""
    n, k = w.shape
    if k % 32:
        raise ValueError("decode GEMM weights need K % 32 == 0")
    n_pad = (n + 15) // 16 * 16
    if n_pad != n:
        w = torch.cat([w, torch.zeros(n_pad - n, k, dtype=w.dtype, device=w.device)], 0)
    return (w.view(n_pad // 16, 2, 8, k // 32, 4, 8).permute(0, 3, 1, 2, 4, 5).contiguous().view(n_pad, k))


def unpack_skinny_weight(w: torch.Tensor, n: int) -> torch.Tensor:
    """Inverse of :func:`pack_skinny_weight`: fragment-major [N_padded, K] -> row-major [n, K] (nn.Linear layout, the
    tcgen05 GEMM's B operand).  A permutation of the same bf16 values, so the result is exact; runs wherever ``w``
    lives (the engine derives the prefill's row-major weights on the device)."""
    n_pad, k = w.shape
    return w.view(n_pad // 16, k // 32, 2, 8, 4, 8).permute(0, 2, 3, 1, 4, 5).contiguous().view(n_pad, k)[:n].contiguous()


def ln_fold_enabled() -> bool:
    """The decoder's LayerNorms are folded into the projections that consume them (csrc/decode.cu, LNF) unless
    TWB200_NO_LN_FOLD is set — the round-1 form (a last-CTA LayerNorm fused into the residual projections) is kept for A/B
    measurements."""
    return not os.environ.get("TWB200_NO_LN_FOLD")


def pack_weights(sd: Dict[str, torch.Tensor], dims: WhisperDims, device) -> Dict[str, torch.Tensor]:
    """HF ``WhisperForConditionalGeneration.state_dict()`` -> packed device tensors.

    * nn.Linear weights stay [out, in] (K-major = the tcgen05 B-operand layout), rounded to bf16.
    * q/k/v are fused into one [3D, D] matrix; the head_dim**-0.5 query scale
      ($TF/models/whisper/modeling_whisper.py:310) is folded into Wq / bq (exact: 0.125 is a power
      of two); k_proj has no bias -> zeros.
    * Conv1d weights [out, in, 3] become [out, 3*in] (tap-major) for the implicit-GEMM view.
    * all decoder layers' cross-attention k/v projections are stacked into one [L*2*D, D] matrix so
      the per-window cross K/V is one GEMM.
    * biases, LayerNorm parameters and positional embeddings stay fp32.
    * the DECODER's linear weights (qkv, out, cross q / out, fc1, fc2) and a second copy of the tied embedding for
      the LM head (``tok_emb_frag``) are stored fragment-major (:func:`pack_skinny_weight`): the decode GEMMs stream
      every weight exactly once per step, and this makes each warp load 512 contiguous bytes.
    """
    D = dims.d_model
    scale = (D // dims.heads) ** -0.5
    dev = torch.device(device)
    w: Dict[str, torch.Tensor] = {}

    def put(name, t):
        w[name] = t.to(dev)

    def attn(prefix_src, prefix_dst):
        q_w, q_b = _f32(sd[prefix_src + "q_proj.weight"]) * scale, _f32(sd[prefix_src + "q_proj.bias"]) * scale
        k_w = _f32(sd[prefix_src + "k_proj.weight"])
        v_w, v_b = _f32(sd[prefix_src + "v_proj.weight"]), _f32(sd[prefix_src + "v_proj.bias"])
        put(prefix_dst + "qkv_w", _bf16(torch.cat([q_w, k_w, v_w], 0)))
        put(prefix_dst + "qkv_b", torch.cat([q_b, torch.zeros_like(q_b), v_b], 0))
        put(prefix_dst + "out_w", _bf16(sd[prefix_src + "out_proj.weight"]))
        put(prefix_dst + "out_b", _f32(sd[prefix_src + "out_proj.bias"]))

    def ln(src, dst):
        put(dst + "_w", _f32(sd[src + ".weight"]))
        put(dst + "_b", _f32(sd[src + ".bias"]))

    def mlp(src, dst):
        put(dst + "fc1_w", _bf16(sd[src + "fc1.weight"]))
        put(dst + "fc1_b", _f32(sd[src + "fc1.bias"]))
        put(dst + "fc2_w", _bf16(sd[src + "fc2.weight"]))
        put(dst + "fc2_b", _f32(sd[src + "fc2.bias"]))

    e = "model.encoder."
    put("conv1_w", _bf16(sd[e + "conv1.weight"].permute(0, 2, 1).reshape(D, -1)))
    put("conv1_b", _f32(sd[e + "conv1.bias"]))
    put("conv2_w", _bf16(sd[e + "conv2.weight"].permute(0, 2, 1).reshape(D, -1)))
    put("conv2_b", _f32(sd[e + "conv2.bias"]))
    put("enc_pos", _f32(sd[e + "embed_positions.weight"]))
    for i in range(dims.enc_layers):
        s, d = f"{e}layers.{i}.", f"enc{i}."
        ln(s + "self_attn_layer_norm", d + "ln1")
        attn(s + "self_attn.", d)
        ln(s + "final_layer_norm", d + "ln2")
        mlp(s, d)
    ln(e + "layer_norm", "enc_ln")

    dd = "model.decoder."
    put("tok_emb", _bf16(sd[dd + "embed_tokens.weight"]))
    put("dec_pos", _f32(sd[dd + "embed_positions.weight"]))
    ckv_w, ckv_b = [], []
    for i in range(dims.dec_layers):
        s, d = f"{dd}layers.{i}.", f"dec{i}."
        ln(s + "self_attn_layer_norm", d + "ln1")
        attn(s + "self_attn.", d)
        ln(s + "encoder_attn_layer_norm", d + "ln2")
        put(d + "cq_w", _bf16(_f32(sd[s + "encoder_attn.q_proj.weight"]) * scale))
        put(d + "cq_b", _f32(sd[s + "encoder_attn.q_proj.bias"]) * scale)
        put(d + "cout_w", _bf16(sd[s + "encoder_attn.out_proj.weight"]))
        put(d + "cout_b", _f32(sd[s + "encoder_attn.out_proj.bias"]))
        ckv_w += [_f32(sd[s + "encoder_attn.k_proj.weight"]), _f32(sd[s + "encoder_attn.v_proj.weight"])]
        vb = _f32(sd[s + "encoder_attn.v_proj.bias"])
        ckv_b += [torch.zeros_like(vb), vb]
        ln(s + "final_layer_norm", d + "ln3")
        mlp(s, d)
    put("ckv_w", _bf16(torch.cat(ckv_w, 0)))
    put("ckv_b", torch.cat(ckv_b, 0))
    ln(dd + "layer_norm", "dec_ln")

    def fold(dst, w_f32, b_f32, ln_src):
        """LayerNorm folded into the projection that consumes it (csrc/decode.cu, LNF):
        W LN(x) + b = rstd (W' x - mean c) + d,  W' = W diag(gamma), c = row sums of the bf16 W', d = W beta + b."""
        g, be = _f32(sd[ln_src + ".weight"]), _f32(sd[ln_src + ".bias"])
        wp = _bf16(w_f32 * g[None, :])
        put(dst + "_wf", pack_skinny_weight(wp.to(dev)))
        put(dst + "_c", wp.to(torch.float64).sum(dim=1).to(torch.float32))
        put(dst + "_d", (w_f32.to(torch.float64) @ be.to(torch.float64)).to(torch.float32) + b_f32)

    do_fold = ln_fold_enabled()
    w["ln_fold"] = torch.tensor([1 if do_fold else 0])
    for i in range(dims.dec_layers):
        s = f"{dd}layers.{i}."
        d = f"dec{i}."
        if not do_fold:
            for nm in ("qkv_w", "out_w", "cq_w", "cout_w", "fc1_w", "fc2_w"):
                w[d + nm] = pack_skinny_weight(w[d + nm])
            continue
        if i > 0:      # layer 0's first LayerNorm is computed by the embedding kernel
            a_ = s + "self_attn."
            qw = torch.cat([_f32(sd[a_ + "q_proj.weight"]) * scale, _f32(sd[a_ + "k_proj.weight"]), _f32(sd[a_ + "v_proj.weight"])], 0)
            vb_ = _f32(sd[a_ + "v_proj.bias"])
            qb = torch.cat([_f32(sd[a_ + "q_proj.bias"]) * scale, torch.zeros_like(vb_), vb_], 0)
            fold(d + "qkv", qw, qb, s + "self_attn_layer_norm")
            del w[d + "qkv_w"]
        fold(d + "cq", _f32(sd[s + "encoder_attn.q_proj.weight"]) * scale, _f32(sd[s + "encoder_attn.q_proj.bias"]) * scale,
             s + "encoder_attn_layer_norm")
        fold(d + "fc1", _f32(sd[s + "fc1.weight"]), _f32(sd[s + "fc1.bias"]), s + "final_layer_norm")
        del w[d + "cq_w"], w[d + "fc1_w"]
        for nm in ("qkv_w", "out_w", "cout_w", "fc2_w"):
            if d + nm in w:
                w[d + nm] = pack_skinny_weight(w[d + nm])
    w["tok_emb_frag"] = pack_skinny_weight(w["tok_emb"])
    return w


def _bitmap(ids: Sequence[int], vocab: int) -> np.ndarray:
    bits = np.zeros((vocab + 31) // 32, dtype=np.uint32)
    for t in ids:
        if 0 <= t < vocab:
            bits[t >> 5] |= np.uint32(1 << (t & 31))
    return bits


def retrieve_segment(seq: List[int], seek_num_frames: int, ts_begin: int):
    """_retrieve_segment ($TF/models/whisper/generation_whisper.py:1976-2073) on python ints:
    slices at consecutive timestamp pairs, returns (segments, seek advance in mel frames)."""
    is_ts = [t >= ts_begin for t in seq]
    single_ending = is_ts[-2:] == [False, True]
    cuts = [i + 1 for i in range(len(seq) - 1) if is_ts[i] and is_ts[i + 1]]
    if not cuts:
        return [list(seq)], seek_num_frames
    if single_ending:
        cuts.append(len(seq))
    else:
        cuts[-1] += 1
    segs, last = [], 0
    for c in cuts:
        segs.append(seq[last:c])
        last = c
    if single_ending:
        return segs, seek_num_frames
    return segs, (seq[last - 2] - ts_begin) * 2  # input_stride = 2 mel frames per encoder position


def init_rows(rows: torch.Tensor, max_len: int, g: Grammar, timestamps: bool, prefilled: bool = False,
              flat: bool = False):
    """Host-side start of R decode rows whose decoder prompts are ``rows`` (int [R, P], :meth:`WhisperEngine.prompt_row`;
    a language of -1 asks for language detection at position 0).  Returns (tokens int32 [R, max_len], forced int32
    [R, max_len], state int32 [R, 8] = tw_row_state [R], the grammar's begin_index = P).
    ``prefilled``: positions 0 .. P-2 run as one prefill (:meth:`WhisperEngine.prefill`) and the state is the one the
    forced steps would leave at position P-1; otherwise the steps feed row[0] and teacher-force the rest of the row.
    ``flat`` (beam search): the grammar is applied by tw_beam_step on the tapped logits, not by the LM head.
    ValueError unless P < ``max_len`` (the rows must leave a position to generate)."""
    R, P = rows.shape
    decoder_prompt_len(P - (3 if timestamps else 4), timestamps, max_len)
    rows = rows.to(torch.int32)
    tokens = torch.full((R, max_len), g.pad, dtype=torch.int32)
    forced = torch.full((R, max_len), -1, dtype=torch.int32)
    st = np.zeros(R, dtype=ROW_STATE)
    st["last_ts"] = -1
    st["mode"] = (rows < 0).any(dim=1).numpy() | (2 if flat or not timestamps else 0)
    if prefilled or flat:
        tokens[:, :P] = rows
    else:
        tokens[:, 0] = rows[:, 0]
    if flat or not prefilled:
        forced[:, 1:P] = rows[:, 1:]      # an unknown language (-1) stays free
    if prefilled:
        st["pos"] = P - 1
        st["text_lo"] = st["ts_lo"] = g.ts_begin
        st["ts_hi"] = g.ts_begin + g.max_initial_ts
        st["begin"] = 1
    return tokens, forced, torch.from_numpy(st.view(np.int32).reshape(R, -1)), P


def long_guard(frames: int) -> int:
    """Seek iterations a long-form clip of ``frames`` mel frames may take before its loop counts as stuck (degenerate
    timestamp output that never advances the seek)."""
    return 64 + 4 * (int(frames) // N_FRAMES)


class LongClip:
    """One clip of a long-form call: its index in the call, frame count, device features, seek pointer, language
    (-1 until detected on its first window), seek iterations run, generated ids (segments in order) and trace."""

    def __init__(self, index: int, frames: int, feats, lang: int):
        self.index, self.frames, self.feats, self.lang = index, int(frames), feats, lang
        self.seek, self.iters = 0, 0
        self.ids: List[int] = []
        self.trace = {"iterations": []}


class LongFormRows:
    """Host bookkeeping of the long-form seek loop over many clips (no device work, unit-tested on the CPU): up to
    ``capacity`` clips are active decode rows; a clip whose seek reaches its frame count leaves, and its row is
    refilled at the next iteration from ``source`` (a callable returning ``(index, audio)`` or None when no clip is
    pending) in the order the source hands clips out.  ``admit([(index, audio), ...]) -> [(frames, feats), ...]``
    prepares the clips that enter at one refill together.  ``record``: keep every clip's seek-loop trace."""

    def __init__(self, capacity: int, source: Callable[[], Optional[tuple]], admit: Callable[[list], list],
                 lang: int = -1, record: bool = False):
        if capacity < 1:
            raise ValueError("a long-form call needs at least one decode row")
        self.capacity, self.source, self.admit, self.lang, self.record = int(capacity), source, admit, lang, record
        self.rows: List[LongClip] = []
        self.done: Dict[int, LongClip] = {}
        self.iterations = self.windows = 0
        self._pending = True

    def refill(self) -> List[LongClip]:
        """Fill the free rows from the source; returns the active rows of the next iteration (empty: the call is over)
        after counting the iteration against every row's guard."""
        while self._pending and len(self.rows) < self.capacity:
            items = []
            while len(self.rows) + len(items) < self.capacity:
                item = self.source()
                if item is None:
                    self._pending = False
                    break
                if item[0] in self.done or any(c.index == item[0] for c in self.rows) or \
                        any(i == item[0] for i, _ in items):
                    raise RuntimeError(f"long-form clip {item[0]} was handed out twice")
                items.append(item)
            if not items:
                break
            for (index, _), (frames, feats) in zip(items, self.admit(items)):
                clip = LongClip(index, frames, feats, self.lang)
                if clip.frames > 0:
                    self.rows.append(clip)
                else:
                    clip.feats = None
                    self.done[index] = clip
        for c in self.rows:
            c.iters += 1
            if c.iters > long_guard(c.frames):
                raise RuntimeError("whisper seek loop does not advance (degenerate timestamp output)")
        if self.rows:
            self.iterations += 1
            self.windows += len(self.rows)
        return list(self.rows)

    def advance(self, clip: LongClip, segments: List[List[int]], adv: int, tokens: Optional[List[int]] = None,
                beam: Optional[tuple] = None) -> None:
        """Append one iteration's segments to ``clip`` and move its seek by ``adv`` frames; a clip whose seek reaches
        its frame count leaves the active rows.  ``tokens`` (the decoder row) and ``beam`` (beam search: the search's
        own (sum of log-probabilities, length) of the returned hypothesis) go to the trace."""
        if self.record and tokens is not None:
            entry = {"rows": [0], "seek": [clip.seek], "tokens": [list(tokens)]}
            if beam is not None:
                entry["beam"] = [beam]
            clip.trace["iterations"].append(entry)
        for sg in segments:
            clip.ids.extend(sg)
        clip.seek += adv
        if clip.seek >= clip.frames:
            self.rows.remove(clip)
            clip.feats = None
            self.done[clip.index] = clip


class WhisperEngine:
    """One engine per GPU.  ``max_batch`` bounds the number of 30 s windows processed together."""

    def __init__(self, dims: WhisperDims, state_dict: Optional[Dict[str, torch.Tensor]], device="cuda:0",
                 gen: Optional[GenerationSettings] = None, max_batch: int = 24, cross_splits: int = 4,
                 shared_weights: Optional[Dict[str, torch.Tensor]] = None, own_stream: bool = False,
                 max_enc_batch: Optional[int] = None):
        """``shared_weights``: the packed weights (``.w``) of another engine on the same device — several engine
        contexts (each with its own workspaces, KV pool and stream) then serve one GPU from one copy of the model,
        so that one context's latency-bound decode overlaps another's tensor-bound encoder.
        ``max_enc_batch``: capacity of the front-end/encoder workspaces when it should exceed the decode batch
        (BASELINE.json configs[4], the log-mel + encoder-only sweep up to 256 windows); default = max_batch."""
        dims.validate()
        _lib.load()
        if not torch.cuda.is_available():
            raise _lib.TwError("turbo-whisper-workspace_b200 needs a CUDA (sm_100a) device; there is no CPU path")
        if max_batch < 1 or max_batch > MAX_DECODE_BATCH:
            raise ValueError(f"max_batch must be in [1, {MAX_DECODE_BATCH}]")
        self.dims, self.gen = dims, gen or GenerationSettings()
        self.device = torch.device(device)
        self.max_batch = max_batch
        cross_splits = int(os.environ.get("TWB200_CROSS_SPLITS", cross_splits))    # tuning knob (tools/probe_decode_tail.py)
        self.cross_splits = cross_splits
        D, F, L, Bm = dims.d_model, dims.ffn, dims.dec_layers, max_batch
        self.max_enc_batch = Be = max(max_batch, int(max_enc_batch or 0))
        S, T = dims.max_source_positions, N_FRAMES
        dev = self.device
        with torch.cuda.device(dev):
            self.w = shared_weights if shared_weights is not None else pack_weights(state_dict, dims, dev)
            self.stream = torch.cuda.Stream(device=dev) if own_stream else None
            self._capture_stream = torch.cuda.Stream(device=dev)
            bf, f32, i32 = torch.bfloat16, torch.float32, torch.int32
            z = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=dev)
            self.logmel = ops.LogMel(dev, Be, dims.n_mels)
            # ---- encoder workspaces
            self.pcm = z(Be, N_SAMPLES, dtype=f32)
            self.n_valid = z(Be, dtype=i32)
            self.mel_t = z(Be, T + 2, dims.n_mels, dtype=bf)    # row 1+t = frame t; rows 0, T+1 = conv padding
            self.mel_s = z(Be, T + 2, dims.n_mels, dtype=bf)    # seek-shifted windows
            self.h1 = z(Be, T + 2, D, dtype=bf)                 # conv1 output, same padding convention
            self.x = z(Be * S, D, dtype=f32)                    # residual stream
            self.xn = z(Be * S, D, dtype=bf)                    # LayerNorm output / encoder output
            self.qkv = z(Be * S, 3 * D, dtype=bf)
            self.att = z(Be * S, D, dtype=bf)
            self.hid = z(Be * S, F, dtype=bf)
            self.ckv = z(Be * S, L * 2 * D, dtype=bf)           # cross-attention K/V of every decoder layer
            # ---- decoder workspaces
            self.max_len = min(self.gen.max_length, dims.max_target_positions)
            self.pages_per_row = (self.max_len + PAGE - 1) // PAGE
            self.n_pages = Bm * self.pages_per_row
            self.kv_pool = z(L, 2, self.n_pages, PAGE, D, dtype=bf)
            self.block_table = z(Bm, self.pages_per_row, dtype=i32)
            self.tokens = z(Bm, self.max_len, dtype=i32)
            self.forced = torch.full((Bm, self.max_len), -1, dtype=i32, device=dev)
            self.state = z(Bm, ROW_STATE.itemsize // 4, dtype=i32)
            self.dx = z(Bm, D, dtype=f32)
            self.dxn = z(Bm, D, dtype=bf)
            self.dxb = z(Bm, D, dtype=bf)                        # bf16 copy of the residual rows (operand of the folded-LayerNorm projections)
            ln_rows = int(_lib.load().tw_dec_max_rows())                 # row stride the kernels use for these buffers
            self.ln_part = z(D // 16, ln_rows, 2, dtype=f32)            # per-CTA (mean, M2) partials of the producer (scratch)
            self.ln_stats = z(ln_rows, 2, dtype=f32)                    # (mean, rstd) per row, left by the producer's last CTA
            self.dq = z(Bm, D, dtype=bf)
            self.datt = z(Bm, D, dtype=bf)
            self.dhid = z(Bm, F, dtype=bf)
            self.n_parts = int(_lib.load().tw_dec_lmhead_parts(dims.vocab))
            self.part_val = z(Bm, self.n_parts, 3, dtype=f32)
            self.part_idx = z(Bm, self.n_parts, 2, dtype=i32)
            self.cross_part = z(Bm, dims.heads, cross_splits, 66, dtype=f32)
            self.cross_cnt = z(Bm, dims.heads, dtype=i32)
            self.ln_cnt = z(1, dtype=i32)
            self.enc_row = z(Bm, dtype=i32)
            self._identity_rows()
            self.align = None    # word-timestamp workspaces (enable_alignment)
            self._align_on = False
            self.logits = None   # optional [Bm, vocab] fp32 raw-logit tap for parity tests
            self.choices = None  # optional [Bm, max_len] int32 tap of the un-forced picks
            self.sup_bits = torch.from_numpy(_bitmap(self.gen.suppress_tokens, dims.vocab).view(np.int32)).to(dev)
            self.bsup_bits = torch.from_numpy(_bitmap(self.gen.begin_suppress_tokens, dims.vocab).view(np.int32)).to(dev)
        g = Grammar()
        g.eos, g.pad, g.no_timestamps = self.gen.eos_token_id, self.gen.pad_token_id, self.gen.no_timestamps_token_id
        g.ts_begin, g.vocab = self.gen.timestamp_begin, dims.vocab
        g.lang_first, g.lang_last = self.gen.lang_first, self.gen.lang_last
        g.max_initial_ts = self.gen.max_initial_timestamp_index
        g.begin_index = 3
        self.grammar = g
        self.ln_fold = bool(int(self.w["ln_fold"][0])) if "ln_fold" in self.w else False
        self._graphs: Dict[tuple, torch.cuda.CUDAGraph] = {}
        self._beam_ws: Dict[tuple, dict] = {}
        self._ckv_batch = max_batch
        self.use_graphs = not os.environ.get("TWB200_NO_GRAPHS")   # debug knob: eager stepping localises device faults
        self.finish_check_every = 16
        self.stats = {"enc_windows": 0, "dec_steps": 0, "launches": 0, "h2d_bytes": 0, "d2h_bytes": 0}
        # weights were repacked and workspaces zeroed by kernels on the default stream; the engine's own (non-blocking)
        # stream does not order against it
        torch.cuda.synchronize(dev)
        self._pcm_host = torch.zeros(Be, N_SAMPLES, dtype=torch.float32).pin_memory()
        self._nv_host = torch.zeros(Be, dtype=torch.int32).pin_memory()

    # ------------------------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _identity_rows(self):
        """Decode row r reads the cross K/V of encoder window r (enc_row) and owns the KV pages r * pages_per_row ..
        (block_table).  Beam search permutes both and restores them with this."""
        dev, Bm, ppr = self.device, self.max_batch, self.pages_per_row
        self.enc_row.copy_(torch.arange(Bm, dtype=torch.int32, device=dev))
        self.block_table.copy_(torch.arange(Bm * ppr, dtype=torch.int32, device=dev).view(Bm, ppr))

    def enable_taps(self):
        """Parity-test taps: raw fp32 logits of the last step and the un-forced picks of every step."""
        if self.logits is None:
            self.logits = torch.zeros(self.max_batch, self.dims.vocab, dtype=torch.float32, device=self.device)
            self.choices = torch.zeros(self.max_batch, self.max_len, dtype=torch.int32, device=self.device)
            self._graphs.clear()

    def enable_alignment(self):
        """Workspaces of the word-timestamp path (return_timestamps="word"): the alignment-head cross-attention tap
        fp32 [max_batch][slots][max_len][1500], the column statistics and the token x frame matrix."""
        heads = self.gen.alignment_heads
        if not heads:
            raise ValueError("Model generation config has no `alignment_heads`, token-level timestamps not available. "
                             "See https://gist.github.com/hollance/42e32852f24243b748ae6bc1f985b13a on how to add this "
                             "property to the generation config.")
        if self.align is not None:
            return
        d, dev, Bm, S = self.dims, self.device, self.max_batch, self.dims.max_source_positions
        for l, h in heads:
            if not (0 <= l < d.dec_layers and 0 <= h < d.heads):
                raise ValueError(f"alignment head ({l}, {h}) is outside the decoder ({d.dec_layers} layers x {d.heads} heads)")
        # slots keep the order of generation_config.alignment_heads (the head mean is order-sensitive in fp32)
        by_layer: Dict[int, List[tuple]] = {}
        for slot, (l, h) in enumerate(heads):
            by_layer.setdefault(int(l), []).append((slot, int(h)))
        layers = {}
        with torch.cuda.device(dev):
            for l, items in by_layer.items():
                # consecutive slots of one layer share a launch
                runs, cur = [], [items[0]]
                for it in items[1:]:
                    if it[0] == cur[-1][0] + 1:
                        cur.append(it)
                    else:
                        runs.append(cur)
                        cur = [it]
                runs.append(cur)
                layers[l] = [(r[0][0], torch.tensor([h for _, h in r], dtype=torch.int32, device=dev)) for r in runs]
            n = len(heads)
            self.align = {
                "layers": layers, "n_slots": n,
                "probs": torch.zeros(Bm, n, self.max_len, S, dtype=torch.float32, device=dev),
                "stats": torch.zeros(Bm, n, S, 2, dtype=torch.float32, device=dev),
                "matrix": torch.zeros(Bm, self.max_len, S, dtype=torch.float32, device=dev),
                "n_frames": torch.zeros(Bm, dtype=torch.int32, device=dev),
                "host": torch.zeros(Bm, self.max_len, S, dtype=torch.float32).pin_memory(),
            }

    def token_frames(self, B: int, tokens: List[List[int]], n_prompt: int, n_frames: Sequence[int],
                     probs: Optional[torch.Tensor] = None, n_tok: Optional[int] = None) -> List[List[int]]:
        """_extract_token_timestamps ($TF/models/whisper/generation_whisper.py:241-381) for the B rows just decoded
        with the alignment tap on: per row the encoder frame of every token position >= n_prompt of the batch's
        sequence (HF's `sequences` of this generate call: as long as the longest row, eos included) but the last.
        ``tokens``: the rows of decode(); ``n_frames[b]``: encoder frames kept for row b (the `[..., : num_frames // 2]`
        crop, already resolved to a count).  Frame -1 where HF's path leaves the table (no frames / NaN costs).
        ``probs`` / ``n_tok``: alternative source with the layout of the tap buffer and its number of generated
        positions (beam search: rows gathered by beam index; ``tokens`` is then ignored)."""
        a, lib, S = self.align, _lib.load(), self.dims.max_source_positions
        eos = self.gen.eos_token_id
        if n_tok is None:
            total = 0
            for row in tokens:
                L = len(row)
                for i in range(n_prompt, len(row)):
                    if row[i] == eos:
                        L = i + 1
                        break
                total = max(total, L)
            n_tok = total - 1 - n_prompt      # cross-attention exists for every position but the last
        if n_tok <= 0:
            return [[] for _ in range(B)]
        nf = [max(0, min(int(f), S)) for f in n_frames]
        p = lambda t: C.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            a["n_frames"][:B].copy_(torch.tensor(nf, dtype=torch.int32), non_blocking=False)
            check(lib.tw_align_matrix(p(a["probs"] if probs is None else probs), p(a["n_frames"]), B, a["n_slots"], self.max_len, S, n_prompt, n_tok,
                                      int(self.gen.median_filter_width), p(a["stats"]), p(a["matrix"]), self._stream()),
                  "tw_align_matrix")
            self.stats["launches"] += 2
            host = a["host"]
            host[:B, :n_tok].copy_(a["matrix"][:B, :n_tok], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            self.stats["d2h_bytes"] += B * n_tok * S * 4
        frames = np.empty((B, n_tok), dtype=np.int32)
        nf_host = np.asarray(nf, dtype=np.int32)
        check(lib.tw_dtw_token_frames_batch(C.c_void_p(host.data_ptr()), self.max_len * S, S, B, n_tok,
                                            nf_host.ctypes.data_as(C.c_void_p), frames.ctypes.data_as(C.c_void_p),
                                            min(B, max(1, (os.cpu_count() or 1) // 2))), "tw_dtw_token_frames_batch")
        return frames.tolist()

    # ------------------------------------------------------------------------------------ front end
    def load_pcm(self, clips: Sequence[np.ndarray]) -> int:
        """H2D of up to max_batch clips (each <= 30 s of fp32 PCM at 16 kHz; longer clips are truncated
        like WhisperFeatureExtractor(truncation=True)).  Returns the batch size."""
        B = len(clips)
        if B > self.max_enc_batch:
            raise ValueError(f"{B} windows > max_enc_batch {self.max_enc_batch}")
        torch.cuda.current_stream(self.device).synchronize()   # the pinned staging buffer may still be in flight
        host, nv = self._pcm_host, self._nv_host
        for i, c in enumerate(clips):
            c = np.asarray(c, dtype=np.float32).reshape(-1)[:N_SAMPLES]
            host[i, :len(c)] = torch.from_numpy(c)
            if len(c) < N_SAMPLES:
                host[i, len(c):] = 0
            nv[i] = len(c)
        with torch.cuda.device(self.device):
            self.pcm[:B].copy_(host[:B], non_blocking=True)
            self.n_valid[:B].copy_(nv[:B], non_blocking=True)
        self.stats["h2d_bytes"] += B * N_SAMPLES * 4 + B * 4
        return B

    def features(self, B: int, out_f32: Optional[torch.Tensor] = None):
        """K1: PCM (self.pcm[:B]) -> time-major bf16 features in self.mel_t (and optionally fp32 [B, n_mels, 3000])."""
        self.logmel(self.pcm[:B], self.n_valid[:B], out_f32=out_f32, out_t=self.mel_t, out_t_row_off=1)
        self.stats["launches"] += 1

    # ------------------------------------------------------------------------------------ encoder
    def encode(self, B: int, mel: Optional[torch.Tensor] = None, taps: Optional[dict] = None) -> torch.Tensor:
        """WhisperEncoder.forward for B windows whose time-major features are in ``mel`` (default
        self.mel_t).  Leaves the final-LayerNorm output in self.xn[:B*1500] and the cross-attention
        K/V of all decoder layers in self.ckv.  The activation buffers (x, xn, qkv, att, hid) are the prompt prefill's
        scratch as well: the returned xn is only valid until the next :meth:`prefill`."""
        d, w = self.dims, self.w
        D, S, T, F = d.d_model, d.max_source_positions, N_FRAMES, d.ffn
        M = B * S
        mel = self.mel_t if mel is None else mel
        C1 = d.n_mels
        with torch.cuda.device(self.device):
            # conv1 (k=3, pad 1) + GELU: A row t = [x[t-1], x[t], x[t+1]] = 3*n_mels contiguous elements of the padded buffer
            # (K = 240 at 80 mels: the TMA box reads zeros past K in the last 64-wide k-block)
            ops.gemm(mel, w["conv1_w"], rows=T, batches=B, a_row_stride=C1, a_batch_stride=(T + 2) * C1, a_rows=T,
                     bias=w["conv1_b"], act=1, out=self.h1, out_ld=D, out_batch_rows=T + 2, out_row_off=1)
            # conv2 (k=3, stride 2, pad 1) + GELU + positional embedding -> fp32 residual stream
            ops.gemm(self.h1, w["conv2_w"], rows=S, batches=B, a_row_stride=2 * D, a_batch_stride=(T + 2) * D,
                     a_rows=S, bias=w["conv2_b"], act=1, resid=w["enc_pos"], resid_ld=D, resid_batch_rows=0,
                     out=self.x, out_ld=D, out_batch_rows=S)
            x, xn, qkv, att, hid = self.x[:M], self.xn[:M], self.qkv[:M], self.att[:M], self.hid[:M]
            if taps is not None:
                taps["stem"] = x.clone()
            for i in range(d.enc_layers):
                p = f"enc{i}."
                ops.layernorm(x, w[p + "ln1_w"], w[p + "ln1_b"], out=xn)
                ops.gemm(xn, w[p + "qkv_w"], rows=M, bias=w[p + "qkv_b"], out=qkv)
                ops.attention_enc(qkv, B, S, d.heads, out=att)
                ops.gemm(att, w[p + "out_w"], rows=M, bias=w[p + "out_b"], resid=x, resid_ld=D, out=x)
                ops.layernorm(x, w[p + "ln2_w"], w[p + "ln2_b"], out=xn)
                ops.gemm(xn, w[p + "fc1_w"], rows=M, bias=w[p + "fc1_b"], act=1, out=hid)
                ops.gemm(hid, w[p + "fc2_w"], rows=M, bias=w[p + "fc2_b"], resid=x, resid_ld=D, out=x)
                if taps is not None and i in taps.get("layers", ()):
                    taps[f"layer{i}"] = x.clone()
            ops.layernorm(x, w["enc_ln_w"], w["enc_ln_b"], out=xn)
            # cross-attention K/V of every decoder layer in one GEMM, stored head-major
            # [(layer, k|v, head)][window][position][64] so decode streams contiguous blocks
            ops.gemm(xn, w["ckv_w"], rows=S, batches=B, a_row_stride=D, a_batch_stride=S * D, a_rows=S,
                     bias=w["ckv_b"], out=self.ckv, out_mode=1)
            self._ckv_batch = B
        self.stats["enc_windows"] += B
        self.stats["launches"] += 2 + 7 * d.enc_layers + 2
        return xn

    # ------------------------------------------------------------------------------------ decoder
    def _skinny(self, wname, x, bias, B, k, ln=None, part_out=False, fold=None):
        """tw_skinny_args for W = self.w[wname].
        ``ln="dec_ln"`` (residual projections): the kernel's last CTA writes LayerNorm(updated x) into self.dxn.
        ``part_out`` (residual projections): the kernel stores bf16(updated x) into self.dxb and per-CTA LayerNorm
        partials into self.ln_part instead — the NEXT projection has that LayerNorm folded into its weights.
        ``fold="dec1.cq"``: such a consumer — weights ``_wf`` (= W diag(gamma)), bias ``_d``, row sums ``_c``."""
        a = SkinnyArgs()
        if fold is not None:
            wname, bias = fold + "_wf", fold + "_d"
        wt = self.w[wname]
        a.w, a.x, a.ldx = wt.data_ptr(), x.data_ptr(), x.stride(0)
        a.bias = None if bias is None else self.w[bias].data_ptr()
        # fragment-major weights are padded to 16 rows: the true N is the bias length (the LM head has N = vocab)
        a.batch, a.n, a.k = B, (self.dims.vocab if bias is None else self.w[bias].shape[0]), k
        if ln is not None:
            a.ln_gamma, a.ln_beta = self.w[ln + "_w"].data_ptr(), self.w[ln + "_b"].data_ptr()
            a.ln_out_bf16, a.ln_counter = self.dxn.data_ptr(), self.ln_cnt.data_ptr()
        if part_out:
            a.ln_part_out, a.x_bf16_out = self.ln_part.data_ptr(), self.dxb.data_ptr()
            a.ln_stats_out, a.ln_counter = self.ln_stats.data_ptr(), self.ln_cnt.data_ptr()
        if fold is not None:
            a.ln_stats_in, a.ln_c = self.ln_stats.data_ptr(), self.w[fold + "_c"].data_ptr()
        return a

    def _cross_kv(self, i: int):
        """K and V pointers of decoder layer i in the head-major cross K/V ([(layer, k|v, head)][window][position][64] of
        the encoder batch that produced self.ckv) and the elements per (layer, k|v, head) block."""
        H, S = self.dims.heads, self.dims.max_source_positions
        blk = self._ckv_batch * S * 64
        base = self.ckv.data_ptr()
        return C.c_void_p(base + ((i * 2 + 0) * H) * blk * 2), C.c_void_p(base + ((i * 2 + 1) * H) * blk * 2), blk

    def _decode_step(self, B: int, finalize: bool = True) -> None:
        """One greedy step for rows 0..B-1: fixed launch sequence, positions read from self.state.
        ``finalize=False`` (beam search): the LM head only taps the raw logits; tw_beam_step picks the tokens."""
        lib, d, w, st = _lib.load(), self.dims, self.w, self._stream()
        D, F, L, H = d.d_model, d.ffn, d.dec_layers, d.heads
        p = lambda t: C.c_void_p(t.data_ptr())
        S = d.max_source_positions
        check(lib.tw_dec_embed(p(self.tokens), self.max_len, p(self.state), p(w["tok_emb"]), p(w["dec_pos"]), p(self.dx),
                               B, D, p(w["dec0.ln1_w"]), p(w["dec0.ln1_b"]), p(self.dxn), st), "tw_dec_embed")
        fold = self.ln_fold

        def normed(q, base, folded):
            """A projection that reads a LayerNorm output: folded into its weights (operand bf16(x)) or not (dxn)."""
            if folded:
                return self._skinny(None, self.dxb, None, B, D, fold=q + base)
            return self._skinny(q + base + "_w", self.dxn, q + base + "_b", B, D)

        def resid(q, base, x, k, ln):
            """A residual projection followed by LayerNorm ``ln``.  With ln_fold it publishes bf16(x) + per-CTA partials
            for the folded consumer (no serial LayerNorm tail), except before the LM head (dec_ln); without (the round-1
            form, TWB200_NO_LN_FOLD, A/B only) its last CTA writes LayerNorm(x) into dxn."""
            if fold and ln != "dec_ln":
                return self._skinny(q + base + "_w", x, q + base + "_b", B, k, part_out=True)
            return self._skinny(q + base + "_w", x, q + base + "_b", B, k, ln=ln)

        for i in range(L):
            q = f"dec{i}."
            nxt = f"dec{i + 1}.ln1" if i + 1 < L else "dec_ln"
            pool = C.c_void_p(self.kv_pool[i].data_ptr())
            # layer 0's first LayerNorm is computed by the embedding kernel
            check(lib.tw_dec_qkv(C.byref(normed(q, "qkv", fold and i > 0)), p(self.dq), pool,
                                 p(self.block_table), self.pages_per_row, self.n_pages, p(self.state), st), "tw_dec_qkv")
            check(lib.tw_dec_self_attn(p(self.dq), p(self.datt), pool, p(self.block_table), self.pages_per_row,
                                       self.n_pages, p(self.state), B, H, st), "tw_dec_self_attn")
            check(lib.tw_dec_linear(C.byref(resid(q, "out", self.datt, D, q + "ln2")), 2, p(self.dx), D, st), "self out_proj")
            check(lib.tw_dec_linear(C.byref(normed(q, "cq", fold)), 0, p(self.dq), D, st), "cross q_proj")
            kptr, vptr, blk = self._cross_kv(i)
            if self._align_on and i in self.align["layers"]:
                al = self.align
                for slot0, heads_dev in al["layers"][i]:
                    check(lib.tw_dec_align_tap(p(self.dq), D, kptr, 64, S * 64, blk, p(self.enc_row), p(self.state),
                                               p(heads_dev), int(heads_dev.numel()), slot0, al["n_slots"], self.max_len,
                                               S, B, p(al["probs"]), st), "tw_dec_align_tap")
            check(lib.tw_dec_cross_attn(p(self.dq), p(self.datt), kptr, vptr, 64, S * 64, blk, p(self.enc_row), S, B, H,
                                        self.cross_splits, p(self.cross_part), p(self.cross_cnt), st), "tw_dec_cross_attn")
            check(lib.tw_dec_linear(C.byref(resid(q, "cout", self.datt, D, q + "ln3")), 2, p(self.dx), D, st),
                  "cross out_proj")
            check(lib.tw_dec_linear(C.byref(normed(q, "fc1", fold)), 3, p(self.dhid), F, st), "fc1")
            check(lib.tw_dec_linear(C.byref(resid(q, "fc2", self.dhid, F, nxt)), 2, p(self.dx), D, st), "fc2")
        for r0 in range(0, B, LMHEAD_ROWS):      # the LM head kernel holds its per-row partials in registers: 48 rows per launch
            rows = min(LMHEAD_ROWS, B - r0)
            check(lib.tw_dec_lmhead(C.byref(self._skinny("tok_emb_frag", self.dxn[r0:], None, rows, D)), C.byref(self.grammar),
                                    p(self.state[r0:]), p(self.sup_bits), p(self.bsup_bits), p(self.part_val[r0:]),
                                    p(self.part_idx[r0:]), None if self.logits is None else p(self.logits[r0:]), st),
                  "tw_dec_lmhead")
        if finalize:
            check(lib.tw_dec_finalize(p(self.part_val), p(self.part_idx), self.n_parts, p(self.tokens), self.max_len,
                                      p(self.forced), None if self.choices is None else p(self.choices), p(self.state),
                                      C.byref(self.grammar), B, st), "tw_dec_finalize")

    # ------------------------------------------------------------------------------------ prompt prefill
    def _prefill_table(self) -> List[Dict[str, tuple]]:
        """Per decoder layer and projection: (row-major weight [N, K], bias, LayerNorm gamma, beta) of the prefill GEMMs.
        Where the decode step folds a LayerNorm into the projection (``ln_fold``), the prefill feeds the GEMM
        x_hat = (x - mean) rstd (gamma = 1, beta = 0) and uses the folded W' = W diag(gamma) with bias d = W beta + b —
        the algebra of the step's folded epilogue; elsewhere (layer 0's q|k|v, the TWB200_NO_LN_FOLD build) it is
        LayerNorm(gamma, beta) with W and b.  gamma / beta None = no LayerNorm in front (the residual projections).
        The row-major copies are derived on the device from the fragment-major decode weights (unpack_skinny_weight)
        at the first prompted call on a device and shared by every engine context of that device through ``self.w``."""
        w, d = self.w, self.dims
        D, F = d.d_model, d.ffn
        if "prefill.ones" not in w:
            with _PREFILL_WEIGHTS_LOCK:
                if "prefill.ones" not in w:
                    with torch.cuda.device(self.device):
                        rm = {}
                        for i in range(d.dec_layers):
                            q = f"dec{i}."
                            names = {"out_w": D, "cout_w": D, "fc2_w": D}
                            names.update({"qkv_wf": 3 * D, "cq_wf": D, "fc1_wf": F} if self.ln_fold else {})
                            names.update({"qkv_w": 3 * D, "cq_w": D, "fc1_w": F})
                            for nm, n in names.items():
                                if q + nm in w:
                                    rm[f"prefill.{q}{nm}"] = unpack_skinny_weight(w[q + nm], n)
                        rm["prefill.zeros"] = torch.zeros(D, dtype=torch.float32, device=self.device)
                        # the copies are made on this context's stream; other contexts use them on theirs
                        torch.cuda.current_stream(self.device).synchronize()
                    w.update(rm)
                    w["prefill.ones"] = torch.ones(D, dtype=torch.float32, device=self.device)
        table = []
        for i in range(d.dec_layers):
            q = f"dec{i}."
            ident = ("prefill.ones", "prefill.zeros")

            def proj(base, ln):
                if self.ln_fold and f"prefill.{q}{base}_wf" in w:
                    return (f"prefill.{q}{base}_wf", q + base + "_d") + ident
                return (f"prefill.{q}{base}_w", q + base + "_b") + ((q + ln + "_w", q + ln + "_b") if ln else (None, None))
            table.append({"qkv": proj("qkv", "ln1"), "out": proj("out", None), "cq": proj("cq", "ln2"),
                          "cout": proj("cout", None), "fc1": proj("fc1", "ln3"), "fc2": proj("fc2", None)})
        return table

    def prefill(self, R: int, P: int, timing: Optional[dict] = None) -> None:
        """Decoder prefill of a text prompt: positions 0 .. P-2 of the rows self.tokens[:R] (P = prompt length with
        the special tokens) through every decoder layer as one batch of M = R (P-1) activation rows — embeddings
        (tw_prefill_embed), LayerNorms (tw_layernorm), the projections on the tcgen05 GEMM (tw_gemm_bf16 with its bias /
        GELU / residual epilogues), K / V into the paged cache (tw_prefill_kv_store), causal self-attention and
        cross-attention against the windows of self.enc_row (tw_prefill_self_attn / _cross_attn).  Position P-1 is fed
        by the first decode step, which also produces the first generated token.  The last layer stops after its K / V.
        Scratch: the encoder's activation buffers (free once encode() has written self.ckv; R (P-1) <= max_enc_batch
        x 1500 always holds).  ``timing``: receives CUDA-event milliseconds per phase ("gemm", "attn", "other")."""
        T = P - 1
        if T <= 0:
            return
        d, w, lib = self.dims, self.w, _lib.load()
        D, F, H, L, S = d.d_model, d.ffn, d.heads, d.dec_layers, d.max_source_positions
        if R > self.max_batch or P > self.max_len:
            raise ValueError(f"prefill of {R} rows x {P} positions exceeds the engine ({self.max_batch} rows, {self.max_len} positions)")
        table = self._prefill_table()
        M = R * T
        p = lambda t: C.c_void_p(t.data_ptr())
        st = self._stream()
        x, xn, qkv, att, hid = self.x[:M], self.xn[:M], self.qkv[:M], self.att[:M], self.hid[:M]
        cq = self.qkv.view(-1)[:M * D].view(M, D)
        events: List[tuple] = []

        def mark(kind):
            if timing is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                events.append((kind, ev))

        launches = 0

        def gemm(name, a, out, act=0, resid=False):
            nonlocal launches
            wt, bias, _, _ = table[i][name]
            mark("gemm")
            ops.gemm(a, w[wt], rows=M, bias=w[bias], act=act, resid=x if resid else None, resid_ld=D if resid else 0,
                     out=out)
            launches += 1

        def norm(name):
            nonlocal launches
            _, _, g, b = table[i][name]
            mark("other")
            ops.layernorm(x, w[g], w[b], out=xn)
            launches += 1

        with torch.cuda.device(self.device):
            mark("other")
            check(lib.tw_prefill_embed(p(self.tokens), self.max_len, R, T, p(w["tok_emb"]), p(w["dec_pos"]), p(x), D, st),
                  "tw_prefill_embed")
            launches += 1
            for i in range(L):
                pool = self.kv_pool[i]
                norm("qkv")
                gemm("qkv", xn, qkv)
                mark("other")
                check(lib.tw_prefill_kv_store(p(qkv), R, T, D, p(pool), p(self.block_table), self.pages_per_row,
                                              self.n_pages, st), "tw_prefill_kv_store")
                launches += 1
                if i + 1 == L:      # nothing reads the last layer's outputs at the prompt positions
                    break
                mark("attn")
                check(lib.tw_prefill_self_attn(p(qkv), p(att), R, T, H, st), "tw_prefill_self_attn")
                gemm("out", att, x, resid=True)
                norm("cq")
                gemm("cq", xn, cq)
                mark("attn")
                kptr, vptr, blk = self._cross_kv(i)
                check(lib.tw_prefill_cross_attn(p(cq), D, p(att), kptr, vptr, 64, S * 64, blk, p(self.enc_row), S, R, T,
                                                H, st), "tw_prefill_cross_attn")
                launches += 2
                gemm("cout", att, x, resid=True)
                norm("fc1")
                gemm("fc1", xn, hid, act=1)
                gemm("fc2", hid, x, resid=True)
            mark("end")
        self.stats["launches"] += launches
        self.stats["prefill_rows"] = self.stats.get("prefill_rows", 0) + M
        if timing is not None:
            torch.cuda.current_stream(self.device).synchronize()
            for (kind, a), (_, b) in zip(events[:-1], events[1:]):
                timing[kind] = timing.get(kind, 0.0) + a.elapsed_time(b)

    def prompt_row(self, prompt_ids: Optional[Sequence[int]], prompt: Sequence[int], timestamps: bool) -> List[int]:
        """The decoder prompt of one row: prompt_ids + ``prompt`` ([<|startoftranscript|>, language, task])
        (+ <|notimestamps|> without timestamps)."""
        return ([] if prompt_ids is None else [int(v) for v in prompt_ids]) + [int(v) for v in prompt] + \
            ([] if timestamps else [self.gen.no_timestamps_token_id])

    @property
    def launches_per_step(self) -> int:
        taps = sum(len(r) for r in self.align["layers"].values()) if self._align_on else 0
        return 1 + 8 * self.dims.dec_layers + 2 + taps      # (+ one more LM-head launch per 48 rows beyond the first 48)

    def _graph(self, key: tuple, step, mutated: Sequence[torch.Tensor]) -> torch.cuda.CUDAGraph:
        """The CUDA graph of ``step()`` cached under ``key``.  A new one is captured after a warm-up run outside capture
        (sets kernel attributes); ``mutated``, everything the step writes, is restored after the warm-up and the capture."""
        g = self._graphs.get(key)
        if g is None:
            saved = [t.clone() for t in mutated]

            def restore():
                for t, v in zip(mutated, saved):
                    t.copy_(v)
            step()
            torch.cuda.current_stream(self.device).synchronize()
            restore()
            g = torch.cuda.CUDAGraph()
            with _CAPTURE_LOCK:
                # explicit per-device capture stream: torch's default capture stream is a process-wide singleton
                # that lives on whichever device captured first
                with torch.cuda.graph(g, stream=self._capture_stream, capture_error_mode="thread_local"):
                    step()
            restore()
            self._graphs[key] = g
        return g

    def _graph_for(self, B: int) -> torch.cuda.CUDAGraph:
        # the K/V block stride depends on the encoder batch; begin_index (3 / 4 with <|notimestamps|>) is a kernel argument
        key = (B, self._ckv_batch, int(self.grammar.begin_index), self._align_on)
        return self._graph(key, lambda: self._decode_step(B), [self.state, self.tokens])

    def decode(self, B: int, prompts: Optional[torch.Tensor], n_steps: Optional[int] = None,
               forced: Optional[torch.Tensor] = None, on_step=None, timestamps: bool = True,
               prompt_ids: Optional[Sequence[int]] = None) -> torch.Tensor:
        """Greedy decode of B rows against the encoder state left by encode().

        prompts: int32 [B, 3] = [<|startoftranscript|>, language, task]; a language of -1 asks for
                 language detection at position 0 (detect_language, $TF/...generation_whisper.py:1610-1673).
        forced:  optional int32 [B, max_len] teacher-forcing table (-1 = free running).
        timestamps: False = generate(return_timestamps=False): <|notimestamps|> is appended to the prompt and only
                 the two suppress lists are applied (no WhisperTimeStampLogitsProcessor).
        prompt_ids: text prompt of generate(prompt_ids=...): the rows start with prompt_ids + [SOT, language, task]
                 (+ <|notimestamps|>) = P positions, of which 0 .. P-2 run as one batched prefill (:meth:`prefill`) and
                 the step loop starts at position P-1; the timestamp grammar begins at P.  The language must be known,
                 and P must be shorter than max_len.
        Returns the int32 token matrix [B, max_len] on the device (prompt included)."""
        dev = self.device
        max_len = self.max_len
        prefilled = prompt_ids is not None
        with torch.cuda.device(dev):
            pr = prompts.cpu()
            if prefilled and bool((pr[:, 1] < 0).any()):
                raise ValueError("decode with prompt_ids needs the language of every row (detect it first)")
            rows = torch.tensor([self.prompt_row(prompt_ids, pr[b, :3], timestamps) for b in range(B)], dtype=torch.int32)
            tok0, frc, st0, self.grammar.begin_index = init_rows(rows, max_len, self.grammar, timestamps, prefilled)
            if forced is not None:      # the caller's teacher forcing wherever the prompt leaves a position free
                frc = torch.where(frc >= 0, frc, forced.cpu().to(torch.int32))
            self.tokens[:B].copy_(tok0.to(dev, non_blocking=False))
            self.forced[:B].copy_(frc.to(dev))
            self.state[:B].copy_(st0.to(dev))
            self.stats["h2d_bytes"] += tok0.nbytes + frc.nbytes + st0.nbytes
            steps = (max_len - 1) if n_steps is None else min(n_steps, max_len - 1)
            if prefilled:
                P = rows.shape[1]
                self.prefill(B, P)
                steps = min(steps, max_len - P)
            _lib.load().tw_set_pdl(0 if (self.use_graphs or os.environ.get("TWB200_NO_PDL")) else 1)   # PDL only pays off for eager stepping
            graph = self._graph_for(B) if self.use_graphs else None
            for s in range(steps):
                if graph is not None:
                    graph.replay()
                else:
                    self._decode_step(B)
                if on_step is not None:
                    on_step(s)
                if self.finish_check_every and (s + 1) % self.finish_check_every == 0 and s + 1 < steps:
                    self.stats["d2h_bytes"] += B * ROW_STATE.itemsize
                    if self.state[:B].cpu().numpy().view(ROW_STATE)["finished"].all():   # every row has emitted eos
                        steps = s + 1
                        break
            self.stats["dec_steps"] += steps
            self.stats["dec_row_steps"] = self.stats.get("dec_row_steps", 0) + steps * B
            self.stats["launches"] += steps * (self.launches_per_step + (B - 1) // LMHEAD_ROWS)
            return self.tokens[:B]

    # ------------------------------------------------------------------------------------ beam search
    def _enable_beam_pool(self) -> None:
        """Beam search re-gathers the paged self-attention cache by block-table permutation; the partial current page
        of every row is copied into the row's own slot of the OTHER page bank, so the pool needs two banks."""
        need = 2 * self.max_batch * self.pages_per_row
        if self.n_pages >= need:
            return
        d, dev = self.dims, self.device
        with torch.cuda.device(dev):
            self.kv_pool = torch.zeros(d.dec_layers, 2, need, PAGE, d.d_model, dtype=torch.bfloat16, device=dev)
        self.n_pages = need
        self._graphs.clear()     # the pool pointer and n_pages are baked into the captured launches

    def _beam_workspace(self, n: int, K: int, P: int, timestamps: bool, track: bool) -> dict:
        key = (n, K, P, bool(timestamps), bool(track))
        ws = self._beam_ws.get(key)
        if ws is not None:
            return ws
        gen, dev, lib = self.gen, self.device, _lib.load()
        cfg = _lib.BeamConfig()
        cfg.num_beams, cfg.vocab, cfg.max_length, cfg.prompt_len = K, self.dims.vocab, self.max_len, P
        cfg.eos, cfg.pad, cfg.no_timestamps = gen.eos_token_id, gen.pad_token_id, gen.no_timestamps_token_id
        mi = gen.max_initial_timestamp_index
        cfg.max_initial_ts = -1 if mi is None else int(mi)
        cfg.timestamps, cfg.track_indices, cfg.length_penalty = int(bool(timestamps)), int(bool(track)), 1.0
        W, R = int(lib.tw_beam_record_width(C.byref(cfg))), n * K
        i32, f32 = torch.int32, torch.float32
        with torch.cuda.device(dev):
            z = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=dev)
            ws = {"cfg": cfg, "W": W, "hist": z(2, n, K, W, dtype=i32), "fin": z(2, n, K, W, dtype=i32),
                  "run_score": z(n, K, dtype=f32), "fin_score": z(n, K, dtype=f32), "fin_flag": z(n, K, dtype=i32),
                  "fin_len": z(n, K, dtype=i32), "gram": z(n, K, 4, dtype=i32), "improvable": z(n, dtype=i32),
                  "hits_all": z(n, dtype=i32), "ctrl": z(8, dtype=i32), "cand_val": z(R, 2 * K, dtype=f32),
                  "cand_tok": z(R, 2 * K, dtype=i32), "copy_src": z(R, dtype=i32), "copy_dst": z(R, dtype=i32),
                  "copy_len": z(1, dtype=i32), "origin": z(R, dtype=i32)}
        st = _lib.BeamState()
        for name in ("hist", "fin", "run_score", "fin_score", "fin_flag", "fin_len", "gram", "improvable", "hits_all", "ctrl"):
            setattr(st, name, ws[name].data_ptr())
        ws["state"] = st
        self._beam_ws[key] = ws
        return ws

    def _beam_step(self, R: int, n: int, ws: dict) -> None:
        """decode step (no finalize; the LM head taps the raw logits) + one tw_beam_step: everything the search needs
        per position, on the device — captured as ONE CUDA graph by decode_beams."""
        p = lambda t: C.c_void_p(t.data_ptr())
        self._decode_step(R, finalize=False)
        check(_lib.load().tw_beam_step(C.byref(ws["cfg"]), C.byref(ws["state"]), p(self.logits), p(self.state),
                                       p(self.sup_bits), p(self.bsup_bits), p(ws["cand_val"]), p(ws["cand_tok"]),
                                       p(self.tokens), self.max_len, p(self.block_table), self.pages_per_row,
                                       self.max_batch * self.pages_per_row, p(self.kv_pool), self.n_pages,
                                       self.dims.dec_layers, self.dims.d_model, p(ws["copy_src"]), p(ws["copy_dst"]),
                                       p(ws["copy_len"]), p(ws["origin"]), n, self._stream()), "tw_beam_step")

    def decode_beams(self, n: int, prompts: torch.Tensor, num_beams: int, timestamps: bool = True,
                     frames_keep: Optional[Sequence[int]] = None, prompt_ids: Optional[Sequence[int]] = None) -> torch.Tensor:
        """Beam search ($TF/generation/utils.py:3076 `_beam_search`, early_stopping=False) for n windows against the
        encoder state left by encode(): n * num_beams decode rows share the windows' cross K/V through `enc_row`; per
        position ONE CUDA-graph replay runs the decode kernels (raw fp32 logits of every row) and `tw_beam_step`
        (csrc/beam.cu: log-softmax + processors + best 2K per row, the running / finished bookkeeping per window, the
        next token of every row, the paged self-attention cache re-gathered by beam of origin as a block-table
        permutation).  The host only polls the "search over" flag every few steps.
        prompts: int [n, 3] with the language resolved.  Returns int64 [n, T]: best hypothesis per window without
        the prompt, right-padded with pad_token_id.
        ``frames_keep``: per window the encoder frames kept for the token-timestamp DTW; the alignment tap runs in
        every step, the search keeps HF's `beam_indices`, the tapped rows of every position are gathered from the beam
        that produced it ($TF/models/whisper/generation_whisper.py:265-303) and ``self.last_beam_frames`` receives
        the frames.
        ``prompt_ids``: text prompt (see :meth:`decode`): the rows start with prompt_ids + prompts (+ <|notimestamps|>),
        whose positions but the last run as one prefill over the n * num_beams rows instead of forced steps."""
        K, R = int(num_beams), n * int(num_beams)
        if R > self.max_batch:
            raise ValueError(f"{n} windows x {K} beams exceed max_batch {self.max_batch}")
        if K > 8:
            raise ValueError("num_beams > 8 is not supported")
        dev, gen, d = self.device, self.gen, self.dims
        if self.logits is None:
            self.enable_taps()
        self._enable_beam_pool()
        want_frames = frames_keep is not None
        with torch.cuda.device(dev):
            prompt = torch.tensor([self.prompt_row(prompt_ids, pr, timestamps) for pr in prompts.cpu()], dtype=torch.int32)
            tok0, frc, st0, P = init_rows(prompt.repeat_interleave(K, dim=0), self.max_len, self.grammar, timestamps,
                                          prefilled=prompt_ids is not None, flat=True)
            self.grammar.begin_index = P
            self.tokens[:R].copy_(tok0.to(dev))
            self.forced[:R].copy_(frc.to(dev))
            self.state[:R].copy_(st0.to(dev))
            self._identity_rows()
            self.enc_row[:R].copy_((torch.arange(R, dtype=torch.int32) // K).to(dev))
            _lib.load().tw_set_pdl(0)
            # ---- search state
            ws = self._beam_workspace(n, K, P, timestamps, want_frames)
            L = self.max_len
            ws["hist"].fill_(gen.pad_token_id)
            ws["fin"].fill_(gen.pad_token_id)
            if want_frames:
                ws["hist"][..., L:] = -1
                ws["fin"][..., L:] = -1
            ws["hist"][0, :, :, :P] = prompt.to(dev)[:, None, :]
            ws["run_score"].fill_(-1.0e9)
            ws["run_score"][:, 0] = 0
            ws["fin_score"].fill_(-1.0e9)
            for name in ("fin_flag", "fin_len", "hits_all", "ctrl"):
                ws[name].zero_()
            ws["gram"].copy_(torch.tensor([0, 1, -1, 0], dtype=torch.int32, device=dev).expand(n, K, 4))
            ws["improvable"].fill_(1)
            if want_frames:
                self.enable_alignment()
            self._align_on = want_frames
            try:
                if prompt_ids is not None:
                    # the prompt but its last token: one prefill over the R rows (no alignment tap: the DTW drops the
                    # prompt positions)
                    self.prefill(R, P)
                else:
                    # the prompt but its last token: plain forced steps (their logits are not needed)
                    plain = self._graph_for(R) if (self.use_graphs and P > 1) else None
                    for _ in range(P - 1):
                        if plain is not None:
                            plain.replay()
                        else:
                            self._decode_step(R)
                forced_steps = 0 if prompt_ids is not None else P - 1
                key = ("beam", R, K, self._ckv_batch, P, bool(timestamps), want_frames)
                # restored after warm-up and capture: the search state (the tw_beam_state buffers) and the rows
                mutated = [ws[name] for name, _ in _lib.BeamState._fields_] + [self.state, self.tokens, self.block_table]
                graph = self._graph(key, lambda: self._beam_step(R, n, ws), mutated) if self.use_graphs else None
                steps, max_steps, poll = 0, L - P, 8
                while steps < max_steps:
                    if graph is not None:
                        graph.replay()
                    else:
                        self._beam_step(R, n, ws)
                    steps += 1
                    if steps % poll == 0 or steps == max_steps:
                        self.stats["d2h_bytes"] += 32
                        if int(ws["ctrl"][1]):       # search over: later replays left the state untouched
                            break
                ctrl = ws["ctrl"].cpu()
                if not int(ctrl[1]):
                    raise RuntimeError("beam search did not terminate within max_length")
                taken, par = int(ctrl[4]), int(ctrl[0])
                self.stats["dec_steps"] += forced_steps + steps
                self.stats["launches"] += forced_steps * self.launches_per_step + steps * (self.launches_per_step - 1 + 3)
                fin_len = ws["fin_len"][:, 0].cpu()
                fin_score = ws["fin_score"][:, 0].cpu()
                # the search's own accounting of the returned hypotheses (sum of processed log-probabilities, length)
                self.last_beam = {"sum_logprob": fin_score * fin_len.float() ** float(ws["cfg"].length_penalty),
                                  "length": fin_len.to(torch.long), "steps": taken}
                m = int(fin_len.max())
                best = ws["fin"][par, :, 0, P:P + m].to(torch.long)
                if want_frames:
                    bi = ws["fin"][par, :, 0, L:L + m].to(torch.long)        # HF's beam_indices, -1 beyond a hypothesis
                    if P > 1:
                        bi = torch.cat([bi[:, :1].expand(-1, P - 1), bi], dim=-1)
                    bi = bi.masked_fill(bi == -1, 0)                         # [n, wl]
                    wl, al = int(bi.shape[1]), self.align
                    slots = torch.arange(al["n_slots"], device=dev)
                    pos = torch.arange(wl, device=dev)
                    gathered = torch.zeros(n, al["n_slots"], self.max_len, d.max_source_positions, dtype=torch.float32,
                                           device=dev)
                    gathered[:, :, :wl] = al["probs"][bi[:, None, :], slots[None, :, None], pos[None, None, :]]
                    self.last_beam_frames = self.token_frames(n, [], P, frames_keep, probs=gathered, n_tok=wl - P)
                return best
            finally:
                self._align_on = False
                self._identity_rows()

    # ------------------------------------------------------------------------------------ generate
    def generate_from_pcm(self, clips: Sequence[np.ndarray], **options):
        """PCM windows (<= 30 s each) -> generated token ids per window (segments concatenated), the
        output contract of ``WhisperGenerationMixin.generate(..., return_timestamps=True)`` minus padding.
        ``options``: the generate options (task, language, return_timestamps, num_beams, token_timestamps, prompt_ids;
        see :meth:`generate`), checked before any device work.  With ``token_timestamps`` every window becomes
        ``(ids, times)`` with one fp32 time per id — the per-segment `token_timestamps` of
        generate(return_token_timestamps=True, return_segments=True), which the ASR pipeline reads for
        return_timestamps="word"."""
        opts = resolve_generate_options(self.dims, self.gen, **options)

        def run():
            B = self.load_pcm(clips)
            self.features(B)
            if not opts.token_timestamps:
                return self._seek(B, opts)
            # attention_mask.sum(-1) of the feature extractor: the sample mask taken every hop (160) samples
            nf = [min(N_FRAMES, -(-min(len(np.asarray(c).reshape(-1)), N_SAMPLES) // 160)) for c in clips]
            return list(zip(self._seek(B, opts, num_frames=nf), self.last_token_ts))
        if self.stream is not None:
            with torch.cuda.stream(self.stream):
                return run()
        return run()

    def generate_long_from_pcm(self, audio: np.ndarray, trace: Optional[dict] = None, **options) -> List[int]:
        """ONE clip longer than 30 s, un-chunked (the ASR pipeline without chunk_length_s,
        $TF/pipelines/automatic_speech_recognition.py:446-454): the one-clip call of :meth:`generate_long_batch`.
        Returns the generated ids (segments concatenated; timestamp tokens restart in every 30 s segment, which
        `_decode_asr` undoes).  ``trace`` receives the clip's seek-loop trace.
        ``options``: the generate options (see :meth:`generate`), checked before any device work; ``prompt_ids`` is
        prepended in every seek iteration (HF with condition_on_prev_tokens off)."""
        # checked here as well so that an invalid call fails before anything else is touched
        resolve_generate_options(self.dims, self.gen, long_form=True, **options)
        traces = None if trace is None else {}
        out = self.generate_long_batch([audio], trace=traces, **options)[0]
        if trace is not None:
            trace.update(traces[0])
        return out

    def generate_long_batch(self, audios: Optional[Sequence[np.ndarray]] = None, *,
                            source: Optional[Callable[[], Optional[tuple]]] = None, rows: Optional[int] = None,
                            trace: Optional[dict] = None, **options) -> Union[List[List[int]], Dict[int, List[int]]]:
        """Many un-chunked long-form clips decoded together: HF's batched long-form generate (every row has its own seek
        pointer and frame count, $TF/models/whisper/generation_whisper.py:654-658, :785-870), with a clip's row refilled
        by the next pending clip as soon as its seek reaches its frame count.  Up to ``rows`` (default and cap
        max_batch // num_beams) clips are active; each iteration gathers the active rows' 30 s windows out of their
        clips' whole-clip features in one launch (tw_gather_frames), encodes them and decodes them as one batch.  The
        language of a clip is detected on its first window.
        ``audios``: the clips (fp32 16 kHz), admitted longest first; returns their ids in input order.
        ``source``: instead of ``audios``, a callable returning ``(index, audio)`` or None when no clip is pending
        (several engine contexts may share one); returns {index: ids} of the clips this call took.
        ``trace``: receives {index: seek-loop trace of that clip} (the format of :meth:`generate`'s trace).
        ``options``: the generate options (see :meth:`generate`), checked before any device work."""
        opts = resolve_generate_options(self.dims, self.gen, long_form=True, **options)
        if (audios is None) == (source is None):
            raise ValueError("generate_long_batch takes either `audios` or `source`")
        if audios is not None:
            order = sorted(range(len(audios)), key=lambda i: -int(np.asarray(audios[i]).size))
            pending = iter([(i, audios[i]) for i in order])
            source = lambda: next(pending, None)

        staging: list = []

        def admit(items):
            # the clips entering together: one H2D copy, one log-mel and one floor launch; the staging buffers live
            # until the next iteration's device-to-host copy has passed them
            feats, keep = self.logmel.long_many([a for _, a in items])
            staging.append(keep)
            self.stats["launches"] += 2
            self.stats["h2d_bytes"] += int(keep[0].numel()) * 4
            return [(int(f.shape[0]), f) for f in feats]

        cap = max(1, self.max_batch // opts.num_beams)
        book = LongFormRows(min(cap, int(rows or cap)), source, admit, opts.lang_id, record=trace is not None)
        if self.stream is not None:
            with torch.cuda.stream(self.stream):
                self._seek_long(book, opts, staging)
        else:
            self._seek_long(book, opts, staging)
        if trace is not None:
            trace.update({i: dict(c.trace, langs=[c.lang]) for i, c in book.done.items()})
        if audios is not None:
            return [book.done[i].ids for i in range(len(audios))]
        return {i: c.ids for i, c in book.done.items()}

    def _strip(self, row: List[int]) -> List[int]:
        """generate_with_fallback's pad / eos stripping ($TF/...generation_whisper.py:1063-1086)."""
        pad, eos = self.gen.pad_token_id, self.gen.eos_token_id
        s = list(row)
        if s and s[-1] == pad:
            n_pad = sum(1 for t in s if t == pad)
            if pad == eos:
                n_pad -= 1
            if n_pad:
                s = s[:-n_pad]
        if s and s[-1] == eos:
            s = s[:-1]
        return s

    def generate(self, B: int, trace: Optional[dict] = None, num_frames: Optional[Sequence[int]] = None,
                 long_mel: Optional[torch.Tensor] = None, **options) -> List[List[int]]:
        """Short-form seek loop over the features in self.mel_t[:B].  ``options`` are the generate options of
        :func:`config.resolve_generate_options`, checked before any device work:

        ``task``, ``language`` (None: detected per row), ``num_beams`` (1: greedy, else beam search) and
        ``return_timestamps`` (timestamp grammar on unless False, in which case <|notimestamps|> joins the prompt).

        ``token_timestamps`` (``num_frames[b]`` = valid mel frames of row b, the attention-mask sum): the decode steps
        also tap the alignment heads' cross-attention, and ``self.last_token_ts[b]`` receives one fp32 time per returned
        id (seek offset added, as `segments[...]["token_timestamps"]` of HF's generate; ``self.last_token_ts_raw[b]`` =
        the padded `token_timestamps` output, no offset).

        ``prompt_ids`` (generate(prompt_ids=...), $TF/models/whisper/generation_whisper.py:1909-1913): every seek
        iteration's decoder input is prompt_ids + [SOT, language, task] (+ <|notimestamps|>), run as one batched prefill
        after encode(); the returned ids exclude it.  An unknown language is detected first on [SOT] alone (one decode
        position), as detect_language does before the prompt is built.

        ``long_mel`` (bf16 [T, n_mels], T > 3000, B == 1): HF's long-form mode — the loop runs over T frames and every
        iteration's window is gathered from ``long_mel`` (zero-padded to 3000 frames, _get_input_segment :1831-1850)."""
        if long_mel is not None and B != 1:
            raise ValueError("long-form generate takes one clip, needs timestamps and has no token timestamps")
        opts = resolve_generate_options(self.dims, self.gen, long_form=long_mel is not None, **options)
        if long_mel is None:
            return self._seek(B, opts, trace=trace, num_frames=num_frames)
        clip = iter([(0, long_mel)])
        book = LongFormRows(1, lambda: next(clip, None), lambda items: [(int(m.shape[0]), m) for _, m in items],
                            opts.lang_id, record=trace is not None)
        self._seek_long(book, opts)
        if trace is not None:
            trace.update(book.done[0].trace, langs=[book.done[0].lang])
        return [book.done[0].ids]

    def _decode_windows(self, n: int, mel: torch.Tensor, langs: List[int], opts: GenerateOptions,
                        frames_keep: Optional[List[int]] = None) -> List[List[int]]:
        """One seek iteration's device work for n windows whose time-major features are in ``mel``: encode, language
        detection where ``langs[i]`` is -1 (``langs`` is updated in place), greedy decode or beam search.  Returns the
        decoder rows (prompt included).  ``frames_keep``: token timestamps on (see :meth:`decode_beams`)."""
        gen, timestamps, prompt_ids = self.gen, opts.timestamps, opts.prompt_ids
        self.encode(n, mel)

        def prompts():
            return torch.tensor([[gen.decoder_start_token_id, langs[i], opts.task_id] for i in range(n)], dtype=torch.int32)
        if (opts.num_beams > 1 or prompt_ids is not None) and any(v < 0 for v in langs):
            # language detection first (one decoder position), as detect_language does before generate
            first = self.decode(n, prompts(), n_steps=1, timestamps=timestamps)[:, 1].cpu().tolist()
            for i in range(n):
                if langs[i] < 0:
                    langs[i] = int(first[i])
        pr = prompts()
        if opts.num_beams > 1:
            best = self.decode_beams(n, pr, opts.num_beams, timestamps=timestamps, frames_keep=frames_keep,
                                     prompt_ids=prompt_ids).cpu().tolist()
            toks = [self.prompt_row(prompt_ids, pr[i], timestamps) + best[i] for i in range(n)]
        else:
            self._align_on = frames_keep is not None
            try:
                toks = self.decode(n, pr, timestamps=timestamps, prompt_ids=prompt_ids).cpu().tolist()
            finally:
                self._align_on = False
        self.stats["d2h_bytes"] += n * self.max_len * 4
        for i in range(n):
            if langs[i] < 0:
                langs[i] = toks[i][1]
        return toks

    def _seek_long(self, book: LongFormRows, opts: GenerateOptions, staging: Optional[list] = None) -> None:
        """The long-form seek loop over the clips of ``book`` with the options already resolved.  ``staging``: buffers
        of the clips' admission, released once an iteration's device-to-host copy has passed their launches."""
        ts_begin, P = self.gen.timestamp_begin, opts.prompt_len
        iters0, windows0 = book.iterations, book.windows
        with torch.cuda.device(self.device):
            while True:
                rows = book.refill()
                if not rows:
                    break
                n = len(rows)
                nfr = [min(c.frames - c.seek, N_FRAMES) for c in rows]
                # the window [seek, seek + 3000) of every row's whole-clip features, zeros past the clip's last frame
                ops.gather_frames([c.feats for c in rows], [c.frames for c in rows], [c.seek for c in rows], self.mel_s,
                                  window=N_FRAMES, row_off=1)
                self.stats["launches"] += 1
                self.stats["h2d_bytes"] += n * 16
                langs = [c.lang for c in rows]
                toks = self._decode_windows(n, self.mel_s, langs, opts)
                if staging:
                    staging.clear()      # the token copy above waited for every launch of this iteration
                beam = self.last_beam if opts.num_beams > 1 else None
                for i, c in enumerate(rows):
                    c.lang = langs[i]
                    segs, adv = retrieve_segment(self._strip(toks[i][P:]), nfr[i], ts_begin)
                    book.advance(c, segs, adv, toks[i], None if beam is None else
                                 (float(beam["sum_logprob"][i]), int(beam["length"][i])))
        self.stats["long_iterations"] = self.stats.get("long_iterations", 0) + book.iterations - iters0
        self.stats["long_windows"] = self.stats.get("long_windows", 0) + book.windows - windows0
        self.stats["long_mean_rows"] = self.stats["long_windows"] / max(1, self.stats["long_iterations"])

    def _seek(self, B: int, opts: GenerateOptions, trace: Optional[dict] = None,
              num_frames: Optional[Sequence[int]] = None) -> List[List[int]]:
        """The short-form seek loop of :meth:`generate` with the options already resolved."""
        num_beams, P = opts.num_beams, opts.prompt_len
        if opts.token_timestamps:
            if num_frames is None or len(num_frames) != B:
                raise ValueError("token_timestamps needs num_frames for every row")
            self.enable_alignment()
        ts_out: List[List[float]] = [[] for _ in range(B)]
        ts_raw: List[List[float]] = [[] for _ in range(B)]
        ts_begin = self.gen.timestamp_begin
        seek = [0] * B
        max_frames = [N_FRAMES] * B
        langs = [opts.lang_id] * B
        out: List[List[int]] = [[] for _ in range(B)]
        it = 0

        def frames_keep(rows):
            # weights[..., : (num_frames - seek) // 2] (_postprocess_outputs :1146-1151, :354): python slice rules and,
            # when every active row has the same value, cropped once more up front (:322-323) — a no-op for
            # non-negative counts, a second crop from the end for negative ones
            S = self.dims.max_source_positions
            left = [int(num_frames[b]) - seek[b] for b in rows]
            twice = len(set(left)) == 1
            return [len((range(S)[: v // 2] if twice else range(S))[: v // 2]) for v in left]
        with torch.cuda.device(self.device):
            while any(s < m for s, m in zip(seek, max_frames)):
                it += 1
                if it > 64 + 4 * (max(max_frames) // N_FRAMES):
                    raise RuntimeError("whisper seek loop does not advance (degenerate timestamp output)")
                rows = [b for b in range(B) if seek[b] < max_frames[b]]
                nfr = {b: min(max_frames[b] - seek[b], N_FRAMES) for b in rows}
                n = len(rows)
                if it == 1:
                    mel = self.mel_t       # seek = 0 for every row: the window is the clip itself
                else:
                    ops.shift_frames(self.mel_t, self.mel_s,
                                     torch.tensor([seek[b] for b in rows], dtype=torch.int32, device=self.device),
                                     src_row=torch.tensor(rows, dtype=torch.int32, device=self.device))
                    self.stats["launches"] += 1
                    mel = self.mel_s
                row_langs = [langs[b] for b in rows]
                toks = self._decode_windows(n, mel, row_langs, opts,
                                            frames_keep(rows) if opts.token_timestamps else None)
                for i, b in enumerate(rows):
                    langs[b] = row_langs[i]
                tok_frames = None
                if opts.token_timestamps and num_beams > 1:
                    tok_frames = self.last_beam_frames
                elif opts.token_timestamps:
                    tok_frames = self.token_frames(n, toks, P, frames_keep(rows))
                if trace is not None:
                    trace.setdefault("iterations", []).append({"rows": list(rows), "seek": [seek[b] for b in rows],
                                                               "tokens": [list(t) for t in toks]})
                for i, b in enumerate(rows):
                    s = self._strip(toks[i][P:])
                    segs, adv = retrieve_segment(s, nfr[b], ts_begin)
                    if tok_frames is not None:
                        # token_timestamps row = [0] * prompt + jump times + [last jump time]; the segments keep the
                        # slice of their tokens (+ the seek offset in seconds, added in fp32)
                        n_kept = sum(len(sg) for sg in segs)
                        jt = (np.asarray(tok_frames[i], dtype=np.float64) * 0.02).astype(np.float32)
                        full = np.concatenate([jt, jt[-1:]]) if jt.size else np.zeros(len(toks[i]), dtype=np.float32)
                        raw = full[:n_kept]
                        off = np.float32(np.float64(seek[b]) * 0.02 / 2)
                        ts_raw[b].extend(float(x) for x in raw)
                        ts_out[b].extend(float(x) for x in (raw + off).astype(np.float32))
                    seek[b] += adv
                    for sg in segs:
                        out[b].extend(sg)
        if trace is not None:
            trace["langs"] = langs
        self.last_token_ts, self.last_token_ts_raw = ts_out, ts_raw
        return out
