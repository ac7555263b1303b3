"""Operator-level Python wrappers over the C ABI (torch tensors in, raw pointers out).

PyTorch is used for device memory and the current stream only; every computation happens in
libtwb200.so.  These mirror the entry points of include/twb200.h one to one and are what the
`-m gpu` parity tests drive."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import GemmArgs, check

N_SAMPLES, N_FRAMES = 480000, 3000


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.TwError("turbo-whisper-workspace_b200 operators need CUDA tensors (no CPU path)")


def slaney_mel_filters(n_mels: int = 128) -> np.ndarray:
    """[201, n_mels] fp32 — the filterbank WhisperFeatureExtractor(feature_size=n_mels) builds
    ($TF/models/whisper/feature_extraction_whisper.py:95-103; $TF/audio_utils.py:453-544):
    n_mels triangular filters on the slaney mel scale over 0-8 kHz, slaney area normalisation."""
    def hz_to_mel(f):
        f = np.asarray(f, dtype=np.float64)
        return np.where(f >= 1000.0, 15.0 + np.log(np.maximum(f, 1e-300) / 1000.0) * (27.0 / np.log(6.4)),
                        3.0 * f / 200.0)

    def mel_to_hz(m):
        return np.where(m >= 15.0, 1000.0 * np.exp((np.log(6.4) / 27.0) * (m - 15.0)), 200.0 * m / 3.0)

    pts = mel_to_hz(np.linspace(hz_to_mel(0.0), hz_to_mel(8000.0), n_mels + 2))
    bins = np.linspace(0, 8000, 201)
    d = np.diff(pts)
    slopes = pts[None, :] - bins[:, None]
    fb = np.maximum(0.0, np.minimum(-slopes[:, :-2] / d[:-1], slopes[:, 2:] / d[1:]))
    fb *= (2.0 / (pts[2:] - pts[:-2]))[None, :]
    return np.ascontiguousarray(fb.astype(np.float32))


class LogMel:
    """K1 front end bound to one device and one filterbank size (``n_mels``: 128 or 80, the model's
    ``WhisperDims.n_mels``): owns the constant tables and the scratch buffer."""

    def __init__(self, device, max_batch: int, n_mels: int = 128):
        lib = _lib.load()
        self.device = torch.device(device)
        self.max_batch = max_batch
        self.n_mels = n_mels
        self.tables = torch.empty(lib.tw_logmel_tables_bytes(), dtype=torch.uint8, device=self.device)
        # zero-filled ONCE: the kernel keeps its per-clip maximum / arrival counters here and re-arms them itself
        self.scratch = torch.zeros(lib.tw_logmel_scratch_bytes(max_batch), dtype=torch.uint8, device=self.device)
        fb = slaney_mel_filters(n_mels)
        with torch.cuda.device(self.device):
            check(lib.tw_logmel_init_n(_ptr(self.tables), fb.ctypes.data_as(C.c_void_p), n_mels), "tw_logmel_init_n")

    def __call__(self, pcm, n_valid=None, out_f32=None, out_t=None, out_t_row_off: int = 0):
        """pcm: cuda fp32 [B, >=480000]; n_valid: cuda int32 [B] or None.
        out_f32: cuda fp32 [B, n_mels, 3000] or None; out_t: cuda bf16 [B, rows, n_mels] or None."""
        lib = _lib.load()
        _need_cuda(pcm, n_valid, out_f32, out_t)
        B, M = pcm.shape[0], self.n_mels
        if B > self.max_batch:
            raise _lib.TwError(f"batch {B} exceeds LogMel max_batch {self.max_batch}")
        assert pcm.dtype == torch.float32 and pcm.stride(1) == 1
        if out_f32 is not None:
            assert out_f32.dtype == torch.float32 and out_f32.is_contiguous() and tuple(out_f32.shape) == (B, M, N_FRAMES)
        tb = 0
        if out_t is not None:
            assert out_t.dtype == torch.bfloat16 and out_t.shape[0] >= B and out_t.shape[2] == M and out_t.stride(2) == 1
            assert out_t.stride(1) == M and out_t.shape[1] >= out_t_row_off + N_FRAMES
            tb = out_t.stride(0)
        with torch.cuda.device(self.device):
            check(lib.tw_logmel_n(_ptr(self.tables), _ptr(pcm), pcm.stride(0), _ptr(n_valid), B, _ptr(self.scratch),
                                  _ptr(out_f32), _ptr(out_t), tb, out_t_row_off, M, _stream()), "tw_logmel_n")


    def long(self, audio: np.ndarray) -> torch.Tensor:
        """Whole-clip features of one clip longer than 30 s (un-chunked long-form input): host fp32 PCM -> cuda bf16
        [n // 160, n_mels], time-major (tw_logmel_long_n; window plan: :func:`longform_plan`)."""
        lib = _lib.load()
        audio = np.asarray(audio, dtype=np.float32).reshape(-1)
        plan = longform_plan(audio.shape[0])
        host = torch.from_numpy(longform_buffer(audio, plan))
        with torch.cuda.device(self.device):
            pcm = host.to(self.device, non_blocking=False)
            ints = torch.tensor([plan["lo"], plan["hi"], plan["row0"]], dtype=torch.int32).to(self.device)
            mx = torch.zeros(1, dtype=torch.int32, device=self.device)
            out = torch.empty(plan["frames"], self.n_mels, dtype=torch.bfloat16, device=self.device)
            check(lib.tw_logmel_long_n(_ptr(self.tables), _ptr(pcm), plan["hop_samples"], len(plan["lo"]), _ptr(ints[0]),
                                       _ptr(ints[1]), _ptr(ints[2]), _ptr(mx), _ptr(out), plan["frames"], 0, self.n_mels,
                                       _stream()),
                  "tw_logmel_long_n")
            torch.cuda.current_stream(self.device).synchronize()      # `pcm` / `ints` are freed when this returns
        return out

    def long_many(self, audios):
        """Whole-clip features of several clips: ONE host-to-device copy of their concatenated buffers
        (:func:`longform_buffer`), one tw_logmel_long_multi launch and its floor launch, every clip with its own
        max - 8 clamp — bit-identical to :meth:`long` per clip.  Returns (features, staging): cuda bf16
        [n // 160, n_mels] per clip (views of one buffer) and the device / pinned staging tensors, which the caller
        keeps until the stream has passed the launch (no synchronisation here)."""
        lib = _lib.load()
        plans = [longform_plan(int(np.asarray(a).size)) for a in audios]
        sizes = [max(p["buffer_samples"], int(np.asarray(a).size) + 200) for a, p in zip(audios, plans)]
        starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        rows = np.concatenate([[0], np.cumsum([p["frames"] for p in plans])]).astype(np.int64)
        host = torch.empty(int(starts[-1]), dtype=torch.float32, pin_memory=True)
        hv = host.numpy()
        off, clip, lo, hi, row0 = [], [], [], [], []
        for c, (a, p) in enumerate(zip(audios, plans)):
            hv[starts[c]:starts[c + 1]] = longform_buffer(np.asarray(a, dtype=np.float32).reshape(-1), p)
            off += [int(starts[c]) + k * p["hop_samples"] for k in range(len(p["lo"]))]
            clip += [c] * len(p["lo"])
            lo += p["lo"]
            hi += p["hi"]
            row0 += [int(rows[c]) + r for r in p["row0"]]
        ints = torch.tensor([clip, lo, hi, row0], dtype=torch.int32).pin_memory()
        longs = torch.from_numpy(np.concatenate([np.asarray(off, dtype=np.int64), rows])).pin_memory()
        with torch.cuda.device(self.device):
            pcm = host.to(self.device, non_blocking=True)
            ints_d = ints.to(self.device, non_blocking=True)
            longs_d = longs.to(self.device, non_blocking=True)
            mx = torch.empty(len(audios), dtype=torch.int32, device=self.device)
            out = torch.empty(int(rows[-1]), self.n_mels, dtype=torch.bfloat16, device=self.device)
            nw = len(off)
            check(lib.tw_logmel_long_multi(_ptr(self.tables), _ptr(pcm), _ptr(longs_d), _ptr(ints_d[0]), nw,
                                           _ptr(ints_d[1]), _ptr(ints_d[2]), _ptr(ints_d[3]), len(audios),
                                           _ptr(longs_d[nw:]), _ptr(mx), _ptr(out), int(rows[-1]), self.n_mels,
                                           _stream()), "tw_logmel_long_multi")
        feats = [out[int(rows[c]):int(rows[c + 1])] for c in range(len(audios))]
        return feats, (host, ints, longs, pcm, ints_d, longs_d, mx, out)


LONG_HOP_FRAMES = 2997      # frames 2 .. 2998 of a 30 s window do not touch its reflect padding


def longform_plan(n_samples: int) -> dict:
    """Cover a clip of n_samples (> 30 s) by overlapping 30 s windows for tw_logmel_long.  The clip has n // 160 frames
    (WhisperFeatureExtractor: 1 + n // 160 STFT frames, the last one dropped); frame t depends on samples
    [160 t - 200, 160 t + 200).  Window b starts at sample 2997 * 160 * b, so its frame j is clip frame 2997 b + j, and it
    is exact for j in [2, 2998] (no reflect padding of the WINDOW involved); window 0 also owns frames 0 and 1, whose
    reflect padding is the clip's own.  -> frames, hop_samples, per window lo / hi (frame range it writes) and row0
    (clip frame of frame lo), buffer_samples (what the kernel may read)."""
    frames = n_samples // 160
    lo, hi, row0 = [], [], []
    b = 0
    while True:
        first = 0 if b == 0 else 2
        last = min(N_FRAMES - 1, frames - LONG_HOP_FRAMES * b)      # exclusive
        if last <= first:
            break
        lo.append(first)
        hi.append(last)
        row0.append(LONG_HOP_FRAMES * b + first)
        b += 1
    hop = LONG_HOP_FRAMES * 160
    return {"frames": frames, "hop_samples": hop, "lo": lo, "hi": hi, "row0": row0,
            "buffer_samples": (len(lo) - 1) * hop + 480000 if lo else 0}


def longform_buffer(audio: np.ndarray, plan: dict) -> np.ndarray:
    """The fp32 buffer the windows read: the clip, the 200 samples of numpy 'reflect' padding of its END
    (x[n + k] = x[n - 2 - k]; torch.stft(center=True, pad_mode="reflect") of the whole waveform), zeros after."""
    n = audio.shape[0]
    buf = np.zeros(max(plan["buffer_samples"], n + 200), dtype=np.float32)
    buf[:n] = audio
    buf[n:n + 200] = audio[n - 2:n - 202:-1]
    return buf


def layernorm(x, gamma, beta, out=None, eps: float = 1e-5):
    """fp32 [rows, cols] -> bf16 [rows, cols]."""
    lib = _lib.load()
    _need_cuda(x, gamma, beta)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 2
    if out is None:
        out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.tw_layernorm(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(out), x.shape[0], x.shape[1], eps, _stream()),
              "tw_layernorm")
    return out


def gemm(a, w, *, rows, batches=1, a_row_stride=None, a_batch_stride=0, a_rows=None, a_row_off=None, bias=None,
         act=0, resid=None, resid_ld=0, resid_batch_rows=0, out=None, out_ld=None, out_batch_rows=0,
         out_row_off=0, k=None, out_mode=0):
    """K5 GEMM (see include/twb200.h tw_gemm_args).  `a` is any bf16 cuda tensor used as a flat base;
    `w` is bf16 [N, K]."""
    lib = _lib.load()
    _need_cuda(a, w, out, bias, resid, a_row_off)
    N, K = w.shape if k is None else (w.shape[0], k)
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and w.is_contiguous()
    args = GemmArgs()
    args.a = a.data_ptr()
    args.a_row_stride = K if a_row_stride is None else a_row_stride
    args.a_batch_stride = a_batch_stride
    args.a_rows = rows if a_rows is None else a_rows
    args.a_row_off = None if a_row_off is None else a_row_off.data_ptr()
    args.w = w.data_ptr()
    args.batches, args.rows, args.n, args.k = batches, rows, N, K
    args.bias = None if bias is None else bias.data_ptr()
    args.act = act
    args.resid = None if resid is None else resid.data_ptr()
    args.resid_ld, args.resid_batch_rows = resid_ld, resid_batch_rows
    args.out = out.data_ptr()
    args.out_f32 = 1 if out.dtype == torch.float32 else 0
    args.out_ld = N if out_ld is None else out_ld
    args.out_batch_rows, args.out_row_off = out_batch_rows, out_row_off
    args.out_mode = out_mode
    with torch.cuda.device(a.device):
        check(lib.tw_gemm_bf16(C.byref(args), _stream()), "tw_gemm_bf16")
    return out


def attention_enc(qkv, batch: int, seq: int, heads: int, out=None):
    """K6: qkv bf16 [batch*seq, 3*heads*64] -> bf16 [batch*seq, heads*64]."""
    lib = _lib.load()
    _need_cuda(qkv, out)
    D = heads * 64
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous() and tuple(qkv.shape) == (batch * seq, 3 * D)
    if out is None:
        out = torch.empty(batch * seq, D, dtype=torch.bfloat16, device=qkv.device)
    with torch.cuda.device(qkv.device):
        check(lib.tw_attention_enc(_ptr(qkv), _ptr(out), batch, seq, heads, out.stride(0), _stream()), "tw_attention_enc")
    return out


def shift_frames(src, dst, seek, src_row=None, frames: int = N_FRAMES, row_off: int = 1):
    """dst[b, row_off+t] = src[src_row[b], row_off+seek[b]+t] (zeros past `frames`); bf16 [*, rows, cols]."""
    lib = _lib.load()
    _need_cuda(src, dst, seek, src_row)
    assert src.dtype == torch.bfloat16 and dst.dtype == torch.bfloat16 and src.stride() == dst.stride()
    assert seek.dtype == torch.int32 and (src_row is None or src_row.dtype == torch.int32)
    B = seek.shape[0]
    with torch.cuda.device(src.device):
        check(lib.tw_shift_frames(_ptr(src), _ptr(dst), _ptr(src_row), _ptr(seek), B, frames, src.shape[2],
                                  src.stride(0), row_off, _stream()), "tw_shift_frames")
    return dst


def gather_frames(feats, frames, seek, dst, window: int = N_FRAMES, row_off: int = 1):
    """dst[b, row_off+t] = feats[b][seek[b]+t] for t < min(window, frames[b] - seek[b]), zeros up to ``window``: one
    launch (tw_gather_frames) over rows that each read their own clip's time-major bf16 features [frames, cols].
    ``frames`` / ``seek``: host ints per row; ``dst``: bf16 [>= rows, >= row_off + window, cols]."""
    lib = _lib.load()
    _need_cuda(dst, *feats)
    B = len(feats)
    cols = dst.shape[2]
    assert dst.dtype == torch.bfloat16 and dst.stride(2) == 1 and dst.stride(1) == cols and dst.shape[0] >= B
    assert dst.shape[1] >= row_off + window and len(frames) == len(seek) == B
    for f, n in zip(feats, frames):
        assert f.dtype == torch.bfloat16 and f.is_contiguous() and f.device == dst.device and f.shape[-1] == cols
        assert f.shape[0] >= n and f.data_ptr() % 16 == 0
    with torch.cuda.device(dst.device):
        ptrs = torch.tensor([f.data_ptr() for f in feats], dtype=torch.int64).to(dst.device)
        ints = torch.tensor([list(frames), list(seek)], dtype=torch.int32).to(dst.device)
        check(lib.tw_gather_frames(_ptr(ptrs), _ptr(ints[0]), _ptr(ints[1]), B, window, cols, _ptr(dst), dst.stride(0),
                                   row_off, _stream()), "tw_gather_frames")
    return dst


# ------------------------------------------------------------------------------------------------
# K0: audio ingest (format conversion + down-mix + windowed-sinc resampling)
# ------------------------------------------------------------------------------------------------
def sinc_resample_filters(orig_freq: int, new_freq: int, lowpass_filter_width: int = 6, rolloff: float = 0.99):
    """Filter bank of torchaudio.functional.resample (sinc_interp_hann): fp32 [new, 2*width + orig] for the
    gcd-reduced rates, plus width.  Same arithmetic, including torchaudio's fp32 phase offset -i/new that is
    promoted to fp64 before the rest of the computation; the result is cast to fp32 at the end."""
    import math
    g = math.gcd(int(orig_freq), int(new_freq))
    orig, new = int(orig_freq) // g, int(new_freq) // g
    base = min(orig, new) * rolloff
    width = math.ceil(lowpass_filter_width * orig / base)
    idx = np.arange(-width, width + orig, dtype=np.float64)[None, :] / orig
    phase = (np.arange(0, -new, -1, dtype=np.int64).astype(np.float32) / np.float32(new)).astype(np.float64)[:, None]
    t = (phase + idx) * base
    t = np.clip(t, -lowpass_filter_width, lowpass_filter_width)
    window = np.cos(t * math.pi / lowpass_filter_width / 2) ** 2
    t = t * math.pi
    with np.errstate(invalid="ignore", divide="ignore"):
        k = np.where(t == 0, 1.0, np.sin(t) / t)
    k = k * window * (base / orig)
    return k.astype(np.float32), width, orig, new


class Resampler:
    """GPU replacement of ``torchaudio.functional.resample(x, orig_freq, new_freq)`` for mono or interleaved
    multi-channel PCM (float32 or int16): one fused pass that converts, averages the channels and resamples."""

    def __init__(self, orig_freq: int, new_freq: int, device):
        self.device = torch.device(device)
        filt, self.width, self.orig, self.new = sinc_resample_filters(orig_freq, new_freq)
        # non-zero span of every phase (the clamped tails of the window are exactly or numerically zero)
        nz = np.abs(filt) > 1e-30
        first = nz.argmax(axis=1)
        last = filt.shape[1] - 1 - nz[:, ::-1].argmax(axis=1)
        span = np.stack([first, last - first + 1], axis=1).astype(np.int32)
        self.filt = torch.from_numpy(np.ascontiguousarray(filt)).to(self.device)
        self.span = torch.from_numpy(span).to(self.device)
        self.taps = int(span[:, 1].max())

    def out_len(self, n_in: int) -> int:
        return -((-self.new * int(n_in)) // self.orig)   # ceil(new * n / orig), as torchaudio

    def __call__(self, x: torch.Tensor, out: torch.Tensor = None) -> torch.Tensor:
        """x: device tensor [n] or [n, channels], float32 or int16 -> fp32 [ceil(new*n/orig)] (channel mean)."""
        _need_cuda(x)
        if x.dtype not in (torch.float32, torch.int16):
            raise _lib.TwError(f"Resampler: unsupported sample dtype {x.dtype}")
        x = x.contiguous()
        n_in = int(x.shape[0])
        ch = 1 if x.dim() == 1 else int(x.shape[1])
        n_out = self.out_len(n_in)
        if out is None:
            out = torch.empty(n_out, dtype=torch.float32, device=x.device)
        if n_out == 0:
            return out
        with torch.cuda.device(x.device):
            check(_lib.load().tw_resample(_ptr(x), 1 if x.dtype == torch.int16 else 0, ch, n_in, _ptr(out), n_out,
                                          _ptr(self.filt), _ptr(self.span), self.orig, self.new, self.width, _stream()),
                  "tw_resample")
        return out
