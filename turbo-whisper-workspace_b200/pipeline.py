"""Drop-in replacement for the Hugging Face ASR pipeline object the reference calls.

The reference's hot path is ``self.transcription_model(audio_path, chunk_length_s=60, batch_size=...,
stride_length_s=5, generate_kwargs={"task": task}, return_timestamps=True)``
(ref:vocalis/core/audio_pipeline.py:351-358), an object made by
``transformers.pipeline("automatic-speech-recognition", ...)`` (ref:vocalis/core/audio_pipeline.py:195-200).
:class:`B200WhisperPipeline` keeps that call signature and output dict
(``{"text": str, "chunks": [{"timestamp": (start, end), "text": str}, ...]}``) and restates the host
logic of ``AutomaticSpeechRecognitionPipeline`` (transformers 5.5.0, ``$TF/``):
  * preprocess / chunk_iter     $TF/pipelines/automatic_speech_recognition.py:341-477, 61-84
  * _forward (stride plumbing)  $TF/pipelines/automatic_speech_recognition.py:479-560
  * postprocess                 $TF/pipelines/automatic_speech_recognition.py:562-656
  * batching of windows         $TF/pipelines/base.py:1298-1318, $TF/pipelines/pt_utils.py:156-298
Token -> text/chunk stitching ($TF/models/whisper/tokenization_whisper.py:901-1270) is native as well:
:class:`decode_asr.AsrDecoder` (C library ``tw_decode_asr`` + a byte table built once from the tokenizer's
vocabulary); the tokenizer object is only an input of the pipeline, exactly as in HF.  Everything between PCM and
token ids runs on the GPU engine(s).
"""
from __future__ import annotations

import io
import os
import subprocess
import wave
from typing import Any, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np

from .config import N_SAMPLES, SAMPLING_RATE, GenerationSettings, WhisperDims, resolve_generate_options


# ------------------------------------------------------------------------------------------------
# audio ingest (host)
# ------------------------------------------------------------------------------------------------
def _read_wav(payload) -> Optional[Tuple[np.ndarray, int]]:
    """RIFF/WAVE reader over any bytes-like object, zero-copy for 16-bit PCM: (samples [n, channels] int16 or float32,
    sample rate), or None when the payload is not a WAV file this reader handles (integer PCM of 8 / 16 / 24 / 32 bits
    and 32-bit IEEE float, plain or WAVE_FORMAT_EXTENSIBLE; anything else is left to ffmpeg, as in HF)."""
    buf = np.frombuffer(payload, dtype=np.uint8)
    n = buf.size
    if n < 12 or bytes(buf[:4]) != b"RIFF" or bytes(buf[8:12]) != b"WAVE":
        return None
    pos, fmt, data = 12, None, None
    while pos + 8 <= n:
        cid = bytes(buf[pos:pos + 4])
        size = int(np.frombuffer(buf[pos + 4:pos + 8], dtype="<u4")[0])
        body = pos + 8
        if cid == b"fmt " and size >= 16 and body + 16 <= n:
            tag, ch, sr, _, _, bits = np.frombuffer(buf[body:body + 16], dtype=[("t", "<u2"), ("c", "<u2"), ("r", "<u4"),
                                                                                ("b", "<u4"), ("a", "<u2"), ("s", "<u2")])[0]
            if int(tag) == 0xFFFE and size >= 26 and body + 26 <= n:      # extensible: the sub-format's first two bytes
                tag = int(np.frombuffer(buf[body + 24:body + 26], dtype="<u2")[0])
            fmt = (int(tag), int(ch), int(sr), int(bits))
        elif cid == b"data":
            if size == 0 or size == 0xFFFFFFFF or body + size > n:          # streamed / truncated files: to the end
                size = n - body
            data = (body, size)
            break
        pos = body + size + (size & 1)
    if fmt is None or data is None:
        return None
    tag, ch, sr, bits = fmt
    if ch < 1 or sr < 1:
        return None
    body, size = data
    frame = ch * (bits // 8)
    if frame == 0:
        return None
    raw = buf[body:body + size - size % frame]
    if tag == 1 and bits == 16:
        x = raw.view("<i2")                                                 # zero-copy view of the payload
    elif tag == 1 and bits == 32:
        x = raw.view("<i4").astype(np.float32) / 2147483648.0
    elif tag == 1 and bits == 24:
        b3 = raw.reshape(-1, 3).astype(np.int32)
        v = b3[:, 0] | (b3[:, 1] << 8) | (b3[:, 2] << 16)
        x = ((v ^ 0x800000) - 0x800000).astype(np.float32) / 8388608.0
    elif tag == 1 and bits == 8:
        x = (raw.astype(np.float32) - 128.0) / 128.0
    elif tag == 3 and bits == 32:
        x = raw.view("<f4")
    else:
        return None
    return x.reshape(-1, ch), sr


def _read_flac(payload: bytes, verify_md5: bool = True) -> Optional[Tuple[np.ndarray, int]]:
    """Native FLAC reader (C library ``tw_flac_decode``): (samples [n, channels] int16 or float32, sample rate), or
    None when the payload is not a FLAC stream.  Frame CRCs are checked by the decoder; the MD5 signature of
    STREAMINFO (when recorded) is checked here.  Corrupt streams raise ValueError, as HF does for undecodable files."""
    if not (payload[:4] == b"fLaC" or payload[:3] == b"ID3"):
        return None
    import ctypes as C
    import hashlib
    from . import _lib
    lib = _lib.load()
    buf = np.frombuffer(payload, dtype=np.uint8)
    ptr = buf.ctypes.data_as(C.c_void_p)
    info = _lib.FlacInfo()
    if lib.tw_flac_info_read(ptr, len(payload), C.byref(info)) != 0:
        if payload[:4] == b"fLaC":
            raise ValueError("malformed FLAC stream: " + lib.tw_last_error().decode("utf-8", "replace"))
        return None        # an ID3 tag in front of something else (e.g. mp3): not ours
    n = C.c_int64(0)
    total = int(info.total_samples)
    if total == 0:         # unknown length: count first
        _lib.check(lib.tw_flac_decode(ptr, len(payload), None, 0, C.byref(n)), "tw_flac_decode")
        total = int(n.value)
    out = np.empty((total, int(info.channels)), dtype=np.int32)
    if lib.tw_flac_decode(ptr, len(payload), out.ctypes.data_as(C.c_void_p), total, C.byref(n)) != 0:
        raise ValueError("Soundfile is either not in the correct format or is malformed: "
                         + lib.tw_last_error().decode("utf-8", "replace"))
    out = out[:int(n.value)]
    bps = int(info.bits_per_sample)
    if verify_md5 and any(info.md5):
        width = (bps + 7) // 8
        raw = (out.astype("<i2") if width == 2 else out.astype("i1") if width == 1 else out.astype("<i4")).tobytes()
        if width == 3:
            raw = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 4)[:, :3].tobytes()
        if hashlib.md5(raw).digest() != bytes(info.md5):
            raise ValueError("FLAC stream decodes to samples that do not match its MD5 signature")
    if bps == 16:
        return out.astype(np.int16), int(info.sample_rate)
    return out.astype(np.float32) / float(1 << (bps - 1)), int(info.sample_rate)


_RESAMPLERS: Dict[Tuple[int, int, str], Any] = {}


def gpu_resample(x: np.ndarray, in_sr: int, out_sr: int, device) -> np.ndarray:
    """[n] or [n, channels] int16 / float32 host samples -> mono fp32 at ``out_sr`` through the fused GPU ingest
    kernel (conversion + channel mean + torchaudio-compatible windowed-sinc resampling; ops.Resampler)."""
    import torch
    from . import ops
    key = (int(in_sr), int(out_sr), str(device))
    rs = _RESAMPLERS.get(key)
    if rs is None:
        rs = _RESAMPLERS[key] = ops.Resampler(in_sr, out_sr, device)
    t = torch.from_numpy(np.array(x if x.dtype == np.int16 else x.astype(np.float32), order="C", copy=True)).to(rs.device)
    return rs(t).cpu().numpy()


def ffmpeg_read(payload, sampling_rate: int, device=None) -> np.ndarray:
    """bytes -> mono fp32 at ``sampling_rate`` ($TF/pipelines/audio_utils.py:9-45).  WAV and FLAC files are decoded
    in-process (FLAC by the C library's native reader) — at the target rate on the host, at any other rate through the
    GPU ingest kernel when a device is given; anything else goes through the same
    ``ffmpeg -i pipe:0 -ac 1 -ar SR -f f32le`` subprocess HF uses."""
    wav = _read_wav(payload)
    if wav is None:
        wav = _read_flac(payload)
    if wav is not None:
        x, sr = wav
        if sr == sampling_rate:
            # one pass; 1/32768 is a power of two, so the product equals the quotient bit for bit
            x = np.multiply(x, np.float32(1.0 / 32768.0), dtype=np.float32) if x.dtype == np.int16 else x
            return np.ascontiguousarray(x[:, 0] if x.shape[1] == 1 else x.mean(axis=1), dtype=np.float32)
        if device is not None:
            return gpu_resample(x, sr, sampling_rate, device)
    cmd = ["ffmpeg", "-i", "pipe:0", "-ac", "1", "-ar", str(sampling_rate), "-f", "f32le", "-hide_banner",
           "-loglevel", "quiet", "pipe:1"]
    try:
        with subprocess.Popen(cmd, stdin=subprocess.PIPE, stdout=subprocess.PIPE) as proc:
            out = proc.communicate(bytes(payload))[0]
    except FileNotFoundError as e:
        raise ValueError("ffmpeg was not found but is required to load audio files from filename") from e
    audio = np.frombuffer(out, np.float32)
    if audio.shape[0] == 0:
        raise ValueError("Soundfile is either not in the correct format or is malformed. Ensure that the soundfile "
                         "has a valid audio file extension (e.g. wav, flac or mp3) and is not corrupted.")
    return audio


def load_audio(inputs: Any, sampling_rate: int = SAMPLING_RATE, device=None) -> Tuple[np.ndarray, Dict[str, Any]]:
    """The input handling of ``preprocess`` ($TF/pipelines/automatic_speech_recognition.py:341-426):
    str path | bytes | np.ndarray | torch.Tensor | {"raw"|"array", "sampling_rate"} -> fp32 mono PCM.
    ``device``: CUDA device for the ingest kernel (resampling of arrays / WAV files that are not at 16 kHz);
    without one the torchaudio call HF makes is used for arrays and ffmpeg for files."""
    extra: Dict[str, Any] = {}
    if isinstance(inputs, str):
        if inputs.startswith("http://") or inputs.startswith("https://"):
            raise ValueError("remote URLs are not supported by the offline engine; pass bytes or an array")
        import mmap
        with open(inputs, "rb") as f:
            try:
                inputs = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)    # the readers work on the page cache directly
            except (ValueError, OSError):                                      # empty file / no mmap support
                inputs = f.read()
    if isinstance(inputs, (bytes, bytearray, memoryview)) or type(inputs).__name__ == "mmap":
        inputs = ffmpeg_read(inputs, sampling_rate, device)
    if hasattr(inputs, "detach") and hasattr(inputs, "cpu"):  # torch.Tensor
        inputs = inputs.detach().cpu().numpy()
    if isinstance(inputs, dict):
        inputs = dict(inputs)
        if inputs.pop("stride", None) is not None:
            raise ValueError("Stride is only usable with CTC models, try removing it !")
        if not ("sampling_rate" in inputs and ("raw" in inputs or "array" in inputs)):
            raise ValueError(
                "When passing a dictionary to AutomaticSpeechRecognitionPipeline, the dict needs to contain a "
                '"raw" key containing the numpy array or torch tensor representing the audio and a "sampling_rate" key, '
                "containing the sampling_rate associated with that array")
        arr = inputs.pop("raw", None)
        if arr is None:
            inputs.pop("path", None)
            arr = inputs.pop("array", None)
        in_sr = inputs.pop("sampling_rate")
        extra = inputs
        if hasattr(arr, "detach"):
            arr = arr.detach().cpu().numpy()
        if in_sr != sampling_rate and device is not None:
            a = np.asarray(arr)
            arr = gpu_resample(a if a.ndim == 1 else a.mean(axis=0), in_sr, sampling_rate, device)
        elif in_sr != sampling_rate:
            try:
                import torch
                from torchaudio import functional as AF
            except ImportError as e:
                raise ImportError("torchaudio is required to resample audio samples in "
                                  "AutomaticSpeechRecognitionPipeline.") from e
            arr = AF.resample(torch.from_numpy(np.asarray(arr)), in_sr, sampling_rate).numpy()
        inputs = arr
    if not isinstance(inputs, np.ndarray):
        raise TypeError(f"We expect a numpy ndarray or torch tensor as input, got `{type(inputs)}`")
    if inputs.ndim != 1:
        inputs = inputs.mean(axis=0)
    return np.ascontiguousarray(inputs, dtype=np.float32), extra


# ------------------------------------------------------------------------------------------------
# windowing
# ------------------------------------------------------------------------------------------------
def chunk_windows(n_samples: int, chunk_len: int, stride_left: int, stride_right: int
                  ) -> List[Tuple[int, int, Tuple[int, int, int], bool]]:
    """``chunk_iter`` ($TF/pipelines/automatic_speech_recognition.py:61-84) as index arithmetic:
    returns [(start, end, (len, stride_left, stride_right), is_last)], dropping windows that are not
    longer than their left stride."""
    out = []
    step = chunk_len - stride_left - stride_right
    for start in range(0, n_samples, step):
        end = start + chunk_len
        length = min(end, n_samples) - start
        sl = 0 if start == 0 else stride_left
        is_last = end >= n_samples
        sr = 0 if is_last else stride_right
        if length > sl:
            out.append((start, start + length, (length, sl, sr), is_last))
        if is_last:
            break
    return out


class B200WhisperPipeline:
    """Callable with the HF ASR-pipeline signature, backed by one :class:`WhisperEngine` per GPU."""

    def __init__(self, state_dict, dims: WhisperDims, tokenizer, generation: Optional[GenerationSettings] = None,
                 devices: Sequence[Union[str, int]] = ("cuda:0",), max_batch: int = 24, time_precision: float = 0.02,
                 scheduler=None, contexts_per_device: int = 4):
        """``scheduler``: any object with ``run(clips, task=, language=) -> token rows`` and ``last_stats``; every other
        generate option reaches ``run`` (and ``run_long``) as a keyword only when it differs from its default, which a
        scheduler forwards to its engines untouched.  Un-chunked long-form inputs (> 30 s without chunk_length_s) go to
        ``run_long(audio, **kw) -> token row``, one call per input; a scheduler may also provide
        ``run_long_many(audios, **kw) -> token rows in input order``, which then receives all long inputs of a call
        that has two or more.  Defaults to a :class:`WindowScheduler` with one GPU engine per entry of ``devices``."""
        self.dims = dims
        self.tokenizer = tokenizer
        self.generation = generation or GenerationSettings()
        self.sampling_rate = SAMPLING_RATE
        self.time_precision = time_precision  # chunk_length 30 s / max_source_positions 1500
        if scheduler is None:
            from .scheduler import WindowScheduler
            scheduler = WindowScheduler(state_dict, dims, self.generation, devices, max_batch,
                                        contexts_per_device=contexts_per_device)
        self.scheduler = scheduler
        # default beam count of a call (generate_kwargs={"num_beams": k} overrides).  1 = greedy, the mode the north star
        # names; transformers >= 4.53 pipelines default to 5, which `num_beams=5` reproduces
        self.num_beams = 1
        # device of the audio-ingest kernel (resampling of inputs that are not at 16 kHz); none with an injected scheduler
        self.ingest_device = None if not hasattr(scheduler, "devices") else scheduler.devices[0]
        from .decode_asr import AsrDecoder
        self.asr_decoder = AsrDecoder(tokenizer, segment_size=dims.max_source_positions)
        self.last_stats: Dict[str, Any] = {}
        self.last_token_rows: List[Any] = []

    @classmethod
    def from_hf_model(cls, model, tokenizer, devices=("cuda:0",), max_batch: int = 24,
                      contexts_per_device: int = 4, scheduler=None) -> "B200WhisperPipeline":
        """Build from a ``transformers.WhisperForConditionalGeneration`` (weights, config, generation_config).
        ``scheduler``: inject an engine stand-in instead of building GPU engines (tests).
        English-only checkpoints (``*.en``) are rejected: their prompt has no language or task token."""
        if getattr(model.generation_config, "is_multilingual", None) is False:
            raise ValueError("English-only Whisper checkpoints (*.en, generation_config.is_multilingual=False) are not "
                             "supported: their decoder prompt has no language or task token, and only the multilingual "
                             "prompt is implemented")
        dims = WhisperDims.from_hf_config(model.config)
        gen = GenerationSettings.from_hf(model.generation_config)
        gen.median_filter_width = int(getattr(model.config, "median_filter_width", 7))
        sd = model.state_dict() if scheduler is None else None
        return cls(sd, dims, tokenizer, gen, devices, max_batch, scheduler=scheduler,
                   contexts_per_device=contexts_per_device)

    # -------------------------------------------------------------------------------- call
    def __call__(self, inputs, chunk_length_s: float = 0, stride_length_s=None, batch_size: Optional[int] = None,
                 generate_kwargs: Optional[dict] = None, return_timestamps=None, return_language=None,
                 **unused) -> Union[Dict[str, Any], List[Dict[str, Any]]]:
        """One input -> one dict; a list / tuple of inputs -> a list of dicts.  As in HF's chunk pipeline
        ($TF/pipelines/pt_utils.py:156-298: the windows of all inputs form ONE stream that is batched `batch_size` at
        a time and regrouped per input afterwards) the windows of all files of a list call go to the engines together,
        so many short files fill the GPUs as well as one long file does."""
        many = isinstance(inputs, (list, tuple))
        items = list(inputs) if many else [inputs]
        generate_kwargs = dict(generate_kwargs or {})
        task = generate_kwargs.pop("task", None) or "transcribe"
        language = generate_kwargs.pop("language", None)
        num_beams = int(generate_kwargs.pop("num_beams", None) or self.num_beams or 1)
        prompt_ids = self._prompt(generate_kwargs)
        # return_timestamps falsy (the HF default): <|notimestamps|> joins the prompt, no timestamp grammar, and the windows
        # are merged on their overlapping text only.  "word": the engine also taps the alignment heads' cross-attention
        opts = resolve_generate_options(self.dims, self.generation, task=task, language=language,
                                        return_timestamps=bool(return_timestamps), num_beams=num_beams,
                                        token_timestamps=return_timestamps == "word", prompt_ids=prompt_ids)
        bs = max(1, int(batch_size or 1))
        # the options reach the scheduler (and its engines) as keywords, each only when it differs from its default
        run_kw: Dict[str, Any] = {"task": task, "language": language}
        if not opts.timestamps:
            run_kw["return_timestamps"] = False
        if opts.num_beams > 1:
            run_kw["num_beams"] = opts.num_beams      # beam search: every window occupies num_beams decode rows
        if opts.token_timestamps:
            # micro-batches follow HF's batches of `batch_size` consecutive windows (capped by the engine's max_batch)
            # because a row's DTW spans the decode steps of its batch's longest row
            run_kw.update(token_timestamps=True, group=bs)
        if opts.prompt_ids is not None:
            run_kw["prompt_ids"] = opts.prompt_ids
        if return_timestamps == "char":
            raise ValueError("Whisper cannot return `char` timestamps, only word level or segment level timestamps. "
                             "Use `return_timestamps='word'` or `return_timestamps=True` respectively.")
        sr = self.sampling_rate
        import time
        t0 = time.perf_counter()
        prepared = [self._prepare(x, chunk_length_s, stride_length_s) for x in items]
        t1 = time.perf_counter()
        clips = [c for p in prepared for c in p["clips"]]
        token_times = None
        if any("longform" in p for p in prepared):
            if not return_timestamps:
                raise ValueError(
                    "You have passed more than 3000 mel input features (> 30 seconds) which automatically enables "
                    "long-form generation which requires the model to predict timestamp tokens. Please either pass "
                    "`return_timestamps=True` or make sure to pass no more than 3000 mel input features.")
            if return_timestamps == "word":
                raise NotImplementedError("word timestamps for un-chunked long-form input are not implemented; pass "
                                          "chunk_length_s as the reference does")
        token_rows = self.scheduler.run(clips, **run_kw) if clips else []
        if return_timestamps == "word":
            token_times = [np.asarray(t, dtype=np.float32) for _, t in token_rows]
            token_rows = [r for r, _ in token_rows]
        # long-form input is only reached with timestamps on and without word timestamps, so run_kw holds nothing that
        # long-form generate refuses
        long_idx = [i for i, p in enumerate(prepared) if "longform" in p]
        if len(long_idx) >= 2 and hasattr(self.scheduler, "run_long_many"):
            # one batched seek loop over all long inputs, spread over the engine contexts
            long_rows = dict(zip(long_idx, self.scheduler.run_long_many([prepared[i]["longform"] for i in long_idx],
                                                                        **run_kw)))
        else:
            long_rows = {i: self.scheduler.run_long(prepared[i]["longform"], **run_kw) for i in long_idx}
        t2 = time.perf_counter()
        self.last_token_rows = token_rows      # the engines' rows of this call, window order (bench.py's output check)
        results, w0 = [], 0
        for i, p in enumerate(prepared):
            if i in long_rows:
                results.append(self._finish(p, [long_rows[i]], None, bs, return_timestamps, return_language))
                continue
            n = len(p["windows"])
            results.append(self._finish(p, token_rows[w0:w0 + n], None if token_times is None else token_times[w0:w0 + n],
                                        bs, return_timestamps, return_language))
            w0 += n
        # host phases of the call: ingest + windowing | engines (H2D, kernels, D2H of token ids) | stitching + text
        self.last_stats = dict(self.scheduler.last_stats, windows=len(clips), files=len(items),
                               audio_seconds=sum(p["n_samples"] for p in prepared) / sr,
                               host_seconds={"prepare": t1 - t0, "engines": t2 - t1, "finish": time.perf_counter() - t2})
        return results if many else results[0]

    def _prompt(self, generate_kwargs: dict):
        """Pops ``prompt_ids`` (list, numpy or torch; normally ``processor.get_prompt_ids(text)``; validated by
        resolve_generate_options) and ``prompt_condition_type`` from generate_kwargs and validates the latter as
        WhisperGenerationMixin.generate does ($TF/models/whisper/generation_whisper.py:1731-1748).  Every window's
        decoder input then starts with prompt_ids; the returned ids, and so the text, exclude it.  ``"all-segments"``
        needs condition_on_prev_tokens, which is not implemented."""
        prompt_ids = generate_kwargs.pop("prompt_ids", None)
        cond = generate_kwargs.pop("prompt_condition_type", None) or "first-segment"
        allowed = ["first-segment", "all-segments"]
        if cond not in allowed:
            raise ValueError(f"`prompt_condition_type={cond} does not exist. Make sure to set `prompt_condition_type` "
                             f"to one of {', '.join(allowed)}")
        if cond == "all-segments":
            if generate_kwargs.get("condition_on_prev_tokens") is not True:
                raise ValueError("Make sure to set `condition_on_prev_tokens=True` when setting "
                                 "`prompt_condition_type='all-segments'`.")
            raise NotImplementedError("prompt_condition_type='all-segments' needs condition_on_prev_tokens, which the "
                                      "engine does not implement")
        return prompt_ids

    def _prepare(self, inputs, chunk_length_s, stride_length_s) -> Dict[str, Any]:
        """preprocess ($TF/pipelines/automatic_speech_recognition.py:341-477) of one input: PCM, windows, clips."""
        audio, extra = load_audio(inputs, self.sampling_rate, self.ingest_device)
        sr = self.sampling_rate
        if chunk_length_s:
            if stride_length_s is None:
                stride_length_s = chunk_length_s / 6
            if isinstance(stride_length_s, (int, float)):
                stride_length_s = [stride_length_s, stride_length_s]
            chunk_len = int(round(chunk_length_s * sr))
            stride_left = int(round(stride_length_s[0] * sr))
            stride_right = int(round(stride_length_s[1] * sr))
            if chunk_len < stride_left + stride_right:
                raise ValueError("Chunk length must be superior to stride length")
            windows = chunk_windows(audio.shape[0], chunk_len, stride_left, stride_right)
            with_stride = True
            if not windows:
                # HF's chunk_iter yields nothing for empty audio and the pipeline's iterator chain ends in a bare
                # StopIteration ($TF/pipelines/pt_utils.py); same exception here, so that the reference's
                # `transcribe` turns it into its {"error": ...} dict exactly as it does today
                raise StopIteration
        else:
            windows = [(0, audio.shape[0], (audio.shape[0], 0, 0), True)]
            with_stride = False
            if audio.shape[0] > N_SAMPLES:
                # un-chunked long-form input ($TF/pipelines/automatic_speech_recognition.py:446-454): features of the
                # WHOLE clip (truncation=False) and ONE generate call whose seek loop walks all of its frames
                # ($TF/models/whisper/generation_whisper.py:654-658).  Not the reference's path (it always passes
                # chunk_length_s); sequential by construction, so it runs on one engine context
                return {"windows": windows, "with_stride": False, "clips": [], "extra": extra,
                        "n_samples": int(audio.shape[0]), "longform": audio}
        # the feature extractor truncates every window to its first 30 s (truncation=True, max_length=480000)
        clips = [audio[s:e][:N_SAMPLES] for (s, e, _, _) in windows]
        return {"windows": windows, "with_stride": with_stride, "clips": clips, "extra": extra,
                "n_samples": int(audio.shape[0])}

    def _finish(self, prep, token_rows, token_times, bs, return_timestamps, return_language) -> Dict[str, Any]:
        """_forward's stride plumbing + postprocess (:479-656) for the windows of one input."""
        sr, windows = self.sampling_rate, prep["windows"]
        # HF batches `batch_size` consecutive windows per generate call and right-pads each batch to its
        # longest row with pad_token_id; _decode_asr ignores the padding, so the grouping only affects shapes.
        pad = self.generation.pad_token_id
        model_outputs = []
        for g0 in range(0, len(windows), bs):
            rows = token_rows[g0:g0 + bs]
            width = max(1, max(len(r) for r in rows))
            for i, r in enumerate(rows):
                arr = np.full((1, width), pad, dtype=np.int64)
                arr[0, :len(r)] = r
                item: Dict[str, Any] = {"tokens": arr}
                if token_times is not None:
                    item["token_timestamps"] = token_times[g0 + i][None, :]
                if prep["with_stride"]:
                    ln, sl, srr = windows[g0 + i][2]
                    item["stride"] = (ln / sr, sl / sr, srr / sr)
                model_outputs.append(item)
        text, optional = self.asr_decoder(model_outputs, return_timestamps=return_timestamps,
                                          return_language=return_language, time_precision=self.time_precision)
        if return_timestamps and self.asr_decoder.last_flags & 1:
            import logging
            logging.getLogger(__name__).warning(
                "Whisper did not predict an ending timestamp, which can happen if audio is cut off in the middle of a word.")
        return {"text": text, **optional, **{k: [v] for k, v in prep["extra"].items()}}

    def close(self):
        self.scheduler.close()
