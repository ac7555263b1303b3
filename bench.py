#!/usr/bin/env python
"""bench.py — RTFx of the Whisper-large-v3-turbo transcription hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

metric  : RTFx = audio seconds / wall seconds, large-v3-turbo bf16 (BASELINE.json)
workload: BASELINE.json configs[1] — 24 x 30 s synthetic windows per GPU per step (random-init weights of the
          large-v3-turbo architecture, seed 0, HF init; 0.1*N(0,1) audio, seeds per window), greedy decode with
          timestamps, HF short-form seek-loop semantics.  Weak scaling: every rank owns its own 24 windows.
value   : device-timed (CUDA events) with the PCM already resident in HBM; log-mel -> encoder -> decode -> seek loop.
e2e     : the same work through the reference-facing callable (B200WhisperPipeline.__call__, the HF ASR pipeline
          signature) with HOST PCM: H2D of the audio, D2H of the token ids and host-side stitching inside the
          timed region.  The rows of the e2e call are checked against a single-context run of the same windows.
extras  : (own arm, unless --no-extras) the other BASELINE.json configs as extra keys of the same line:
          `encoder` (whole encoder at batch 24 vs the tensor-pipe peak), `decode_step` (µs per greedy step alone vs the
          HBM floor), `config3` (ONE 1 h file through the pipeline callable, sharded over the N ranks by the chunk
          scheduler — strong scaling), `config2_beams5` (the 24 windows with num_beams = 5), `config4` (large-v3, 32 decoder layers, batch 16), `config5` (log-mel +
          encoder-only sweep, batch 1..256).
The `--impl reference` arm times the reference's own CPU implementation of the path: every step is ONE real call of the
reference's `AudioProcessingPipeline.process_audio(path, task="transcribe")` (the unmodified `vocalis` package installed
under baseline/_ref, its transformers ASR pipeline object on the CPU in fp32, greedy) on ONE 30 s window of the
workload — nothing is extrapolated: `ms_per_step` is the wall time of that call.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the tree may be read-only: no __pycache__ next to the sources it imports
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WINDOWS_PER_GPU = 24
WINDOW_S = 30.0
ENC_FLOPS_PER_WINDOW = 2.2738e12          # SURVEY.md §8d
METRIC = "RTFx (audio s / wall s), large-v3-turbo bf16"


def workload_config(world: int) -> dict:
    """The `config` object — identical for both arms (the reference arm runs a bounded sample of it, see its
    `cpu_baseline.sample`)."""
    return {"workload": "whisper-large-v3-turbo bf16, 24 x 30 s windows per GPU per step (BASELINE.json configs[1]); "
                        "random-init weights (HF init, seed 0), 0.1*N(0,1) audio; greedy, timestamps, HF short-form "
                        "seek loop",
            "windows_per_gpu": WINDOWS_PER_GPU,
            "parallelism": f"window-sharded x{world}, no data-path collective",
            "l2": "working set (1.6 GB weights + >2 GB activations per step) exceeds the 126 MB L2"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def ncu_traffic():
    """DRAM bytes per launch of the two roofline kernels from THIS round's `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep); None when absent."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p))
    except (OSError, ValueError):
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        import numpy as np
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # "under load": the upper half of the samples (the sampler also sees idle gaps at the region's edges)
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# reference arm (CPU): the reference's own process_audio call
# ----------------------------------------------------------------------------------------------------
def build_hf_turbo(seed: int = 0):
    import torch
    from transformers import GenerationConfig, WhisperConfig, WhisperForConditionalGeneration
    from transformers.models.whisper.tokenization_whisper import LANGUAGES
    from oracle import whisper_ref as R
    cfg = WhisperConfig(vocab_size=51866, num_mel_bins=128, d_model=1280, encoder_layers=32, decoder_layers=4,
                        encoder_attention_heads=20, decoder_attention_heads=20, encoder_ffn_dim=5120,
                        decoder_ffn_dim=5120, max_source_positions=1500, max_target_positions=448, pad_token_id=50257,
                        bos_token_id=50257, eos_token_id=50257, decoder_start_token_id=50258)
    torch.manual_seed(seed)
    model = WhisperForConditionalGeneration(cfg).eval()
    model.generation_config = GenerationConfig(
        begin_suppress_tokens=list(R.BEGIN_SUPPRESS_TOKENS), suppress_tokens=list(R.SUPPRESS_TOKENS),
        max_initial_timestamp_index=50, max_length=448, is_multilingual=True, no_timestamps_token_id=50364,
        lang_to_id={f"<|{l}|>": 50259 + i for i, l in enumerate(LANGUAGES)},
        task_to_id={"transcribe": 50360, "translate": 50359}, return_timestamps=False, pad_token_id=50257,
        bos_token_id=50257, eos_token_id=50257, decoder_start_token_id=50258)
    return model


def build_reference_callable():
    """-> (call(path) -> result dict, kind, description).

    The reference's entry point for this path is `vocalis.core.audio_pipeline.AudioProcessingPipeline.process_audio`
    (ref:vocalis/core/audio_pipeline.py:567-688 -> transcribe :323-369).  It is imported UNMODIFIED from
    baseline/_ref (installed with `pip install --no-deps --target baseline/_ref <copy of /root/reference>`, DESIGN.md §6;
    /root/reference itself is used when present and baseline/_ref is not).  What has to be supplied around it offline
    (SURVEY.md §8c recipe): empty stub modules for its optional imports (librosa, soundfile, sherpa_onnx, pydub), a WAV
    reader in place of the `ffmpeg` binary HF's `ffmpeg_read` shells out to, diarization / LLM post-steps off
    ("diarization off" is BASELINE.json configs[0]), and the `transcription_model` object itself — the reference would
    download openai weights; here it is the same `transformers.pipeline("automatic-speech-recognition", ...)`
    construction over the random-init large-v3-turbo model on the CPU in fp32, `num_beams = 1` (greedy, the north
    star's mode).  Without the package (neither path exists) the same pipeline object is called with the reference's
    literal keyword arguments (:351-358) and the arm says kind = "port"."""
    import io
    import types
    import wave
    import importlib.machinery
    import numpy as np
    import torch
    os.environ.setdefault("HF_HUB_OFFLINE", "1")
    from transformers import WhisperFeatureExtractor, pipeline
    import transformers.pipelines.automatic_speech_recognition as asr
    import helpers

    def wav_read(payload, sampling_rate):
        with wave.open(io.BytesIO(payload)) as w:
            assert w.getframerate() == sampling_rate and w.getnchannels() == 1 and w.getsampwidth() == 2
            return np.frombuffer(w.readframes(w.getnframes()), np.int16).astype(np.float32) / 32768.0
    asr.ffmpeg_read = wav_read
    model = build_hf_turbo(0)
    pipe = pipeline("automatic-speech-recognition", model=model, tokenizer=helpers.build_tokenizer(),
                    feature_extractor=WhisperFeatureExtractor(feature_size=128), device="cpu", dtype=torch.float32)
    pipe.generation_config.num_beams = 1
    src = None
    for cand in (os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if os.path.isdir(os.path.join(cand, "vocalis", "core")):
            src = cand
            break
    if src is None:
        def call(path):
            return pipe(path, chunk_length_s=60, batch_size=32, stride_length_s=5, generate_kwargs={"task": "transcribe"},
                        return_timestamps=True)
        return call, pipe, "port", ("transformers ASR pipeline object called with the reference's literal transcribe() "
                                    "keyword arguments (vocalis package not present)")
    for m in ("librosa", "soundfile", "sherpa_onnx", "pydub"):
        if m not in sys.modules:
            stub = types.ModuleType(m)
            stub.__spec__ = importlib.machinery.ModuleSpec(m, None)
            sys.modules[m] = stub
    if not hasattr(sys.modules["pydub"], "AudioSegment"):
        sys.modules["pydub"].AudioSegment = type("AudioSegment", (), {})
    if src not in sys.path:
        sys.path.insert(0, src)
    import vocalis.core.audio_pipeline as ap
    ap.LLM_AVAILABLE = False
    p = ap.AudioProcessingPipeline()
    p.transcription_model = pipe
    p.diarize = lambda *a, **k: []

    def call(path):
        return p.process_audio(path, task="transcribe")
    return call, pipe, "reference", (f"vocalis.core.audio_pipeline.AudioProcessingPipeline.process_audio from {src} "
                                     "(unmodified), transcription_model = transformers ASR pipeline, CPU fp32, greedy")


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    import tempfile
    import numpy as np
    import torch
    import helpers
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    call, pipe, kind, what = build_reference_callable()
    tmp = tempfile.mkdtemp(prefix="twb200_ref_")

    def wav_for(i):
        path = os.path.join(tmp, f"w{i}.wav")
        helpers.write_wav16(path, helpers.synth_clip(i))
        return path
    # warm-up: untimed SHORT calls of the same pipeline object (lazy imports, thread pool, allocator); a full call
    # costs ~20 s of CPU and warms nothing more
    for i in range(args.warmup):
        pipe(wav_for(0), chunk_length_s=60, stride_length_s=5, batch_size=32, return_timestamps=True,
             generate_kwargs={"task": "transcribe", "max_new_tokens": 4})
    times, chunks, t_begin = [], None, time.perf_counter()
    for i in range(args.steps):
        path = wav_for(i % WINDOWS_PER_GPU)
        t0 = time.perf_counter()
        res = call(path)
        times.append(time.perf_counter() - t0)
        if "error" in res:
            raise SystemExit(f"bench.py: the reference call failed: {res['error']}")
        chunks = len(res.get("segments", res.get("chunks", [])))
        if time.perf_counter() - t_begin > args.reference_budget_s:
            break
    # the reference's LITERAL decoding mode: it passes only generate_kwargs={"task": ...}, and transformers >= 4.53 ASR
    # pipelines default to num_beams = 5 (SURVEY.md §0.4).  One such call, outside the timed steps (an extra key; the
    # metric above stays greedy like the own arm), when the wall-clock budget has room for it
    literal = None
    if args.steps >= 2 and not args.no_literal_beams and \
            time.perf_counter() - t_begin + 8 * max(times) < args.reference_budget_s:
        pipe.generation_config.num_beams = 5
        t0 = time.perf_counter()
        res5 = call(wav_for(0))
        dt5 = time.perf_counter() - t0
        pipe.generation_config.num_beams = 1
        if "error" not in res5:
            literal = {"what": "one process_audio call with the pipeline's default num_beams = 5 (what the reference's "
                               "literal call decodes with under the installed transformers)", "seconds": dt5,
                       "rtfx": WINDOW_S / dt5, "chunks": len(res5.get("segments", res5.get("chunks", [])))}
    t = float(np.mean(times))
    rtfx = WINDOW_S / t
    sample = (f"{len(times)} timed call(s), each ONE full reference call on ONE 30 s window of the workload (windows "
              f"0..{len(times) - 1} of the 24); {what}; per call 3 encoder + 891 decoder forwards (language id + 2 seek "
              f"iterations to max_length; random-init weights never emit eos); wall {min(times):.1f}-{max(times):.1f} s "
              f"per call; nothing extrapolated")
    line = {"impl": "reference", "metric": METRIC, "value": rtfx, "unit": "x realtime", "n_gpus": args.gpus,
            "steps": len(times), "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "cpu_baseline": {"value": rtfx, "unit": "x realtime", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": sample},
            "e2e": {"value": rtfx, "unit": "x realtime", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "steps_requested": args.steps, "chunks_last_call": chunks, "literal_num_beams_5": literal,
            "host": {"cpu_count": cores, "torch_threads": torch.get_num_threads(), "torch": torch.__version__}}
    emit(line)
    return 0


def cpu_baseline_subprocess(budget_s: float):
    """Own arm, N = 1: the reference arm's measurement (one real call) in a child process with the GPU hidden."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        # two calls: the first full call of a process carries one-off costs (allocator, thread pool) the reference arm's
        # mean over its steps does not show
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2",
                              "--warmup", "1", "--no-literal-beams"], env=env, capture_output=True, text=True,
                             timeout=budget_s)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"value": None, "unit": "x realtime", "cores": os.cpu_count(), "kind": "reference",
                "sample": "reference child process printed no result: " + out.stderr[-300:]}
    except subprocess.TimeoutExpired:
        return {"value": None, "unit": "x realtime", "cores": os.cpu_count(), "kind": "reference",
                "sample": f"reference child process exceeded {budget_s:.0f} s"}


# ----------------------------------------------------------------------------------------------------
# own arm
# ----------------------------------------------------------------------------------------------------
def cuda_timed(fn, iters, warm=1):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def gemm_roofline_probe(eng, B, iters=5):
    """Average launch duration of the dominant encoder kernel (K5 tcgen05 GEMM) on the encoder's own four
    shapes, CUDA events on the launching stream; algorithmic FLOPs = 2*M*N*K per launch."""
    from turbo_whisper_workspace_b200 import ops
    d = eng.dims
    D, F, S = d.d_model, d.ffn, d.max_source_positions
    M = B * S
    w, p = eng.w, "enc0."
    x, xn, qkv, att, hid = eng.x[:M], eng.xn[:M], eng.qkv[:M], eng.att[:M], eng.hid[:M]
    launches = [
        (lambda: ops.gemm(xn, w[p + "qkv_w"], rows=M, bias=w[p + "qkv_b"], out=qkv), 2.0 * M * 3 * D * D),
        (lambda: ops.gemm(att, w[p + "out_w"], rows=M, bias=w[p + "out_b"], resid=x, resid_ld=D, out=x), 2.0 * M * D * D),
        (lambda: ops.gemm(xn, w[p + "fc1_w"], rows=M, bias=w[p + "fc1_b"], act=1, out=hid), 2.0 * M * F * D),
        (lambda: ops.gemm(hid, w[p + "fc2_w"], rows=M, bias=w[p + "fc2_b"], resid=x, resid_ld=D, out=x), 2.0 * M * D * F),
    ]

    def all_four():
        for fn, _ in launches:
            fn()
    ms = cuda_timed(all_four, iters) / len(launches)
    flops = sum(f for _, f in launches) / len(launches)
    return ms, flops


def cross_attn_roofline_probe(eng, B, iters=20):
    """Average launch duration of the decode cross-attention kernel (largest single kernel of a step by time) on
    the engine's own head-major K/V, CUDA events on the launching stream.  Algorithmic bytes per launch =
    B * 2 (K,V) * 1500 * 1280 * 2 B (SURVEY.md §8d: 7.68 MB per sequence-layer)."""
    import ctypes as C
    import torch
    from turbo_whisper_workspace_b200 import _lib
    lib = _lib.load()
    d = eng.dims
    D, H, S = d.d_model, d.heads, d.max_source_positions
    blk = eng._ckv_batch * S * 64
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = d.dec_layers
    it = [0]

    def launch():
        i = it[0] % L          # rotate layers: 4 x 184 MB > L2
        it[0] += 1
        kptr = C.c_void_p(eng.ckv.data_ptr() + ((i * 2 + 0) * H) * blk * 2)
        vptr = C.c_void_p(eng.ckv.data_ptr() + ((i * 2 + 1) * H) * blk * 2)
        _lib.check(lib.tw_dec_cross_attn(p(eng.dq), p(eng.datt), kptr, vptr, 64, S * 64, blk, None, S, B, H,
                                         eng.cross_splits, p(eng.cross_part), p(eng.cross_cnt), st), "cross_attn")
    return cuda_timed(launch, iters, warm=L), B * 2.0 * S * D * 2


def decode_step_probe(eng, B, steps=256):
    """µs per greedy decode step of ONE context alone (CUDA-graph replays back to back, CUDA events) and the
    algorithmic HBM bytes a step has to move (SURVEY.md §8d): decoder weights once + LM head + cross K/V of the B rows
    (+ the self-attention cache, averaged over the positions visited)."""
    import torch
    d, gen = eng.dims, eng.gen
    D, F, L, S = d.d_model, d.ffn, d.dec_layers, d.max_source_positions
    prompts = torch.tensor([[gen.decoder_start_token_id, 50259, gen.task_to_id["transcribe"]]] * B, dtype=torch.int32)
    with torch.cuda.device(eng.device):
        eng.decode(B, prompts, n_steps=1)
        graph = eng._graph_for(B)
        torch.cuda.synchronize()
        steps = min(steps, eng.max_len - 4)
        ms = cuda_timed(graph.replay, steps, warm=0)
    weights = L * (4 * D * D + 4 * D * D + 2 * D * F) * 2
    lm_head = d.vocab * D * 2
    cross = B * L * 2 * S * D * 2
    self_kv = B * L * 2 * (steps / 2.0) * D * 2
    return ms * 1e3, float(weights + lm_head + cross + self_kv)


def synth_state_dict_on_device(dims, device, seed=0):
    """HF-layout random-init weights generated ON the device (N(0, 0.02) like WhisperPreTrainedModel._init_weights,
    zero biases, unit LayerNorm): the 1.5 B parameters of large-v3 take a minute on host cores."""
    import torch
    import helpers
    g = torch.Generator(device=device).manual_seed(seed)
    D, F, V = dims.d_model, dims.ffn, dims.vocab
    sd = {}

    def lin(name, o, i, bias=True):
        sd[name + ".weight"] = torch.randn(o, i, generator=g, device=device) * 0.02
        if bias:
            sd[name + ".bias"] = torch.zeros(o, device=device)

    def ln(name):
        sd[name + ".weight"] = torch.ones(D, device=device)
        sd[name + ".bias"] = torch.zeros(D, device=device)

    def attn(p):
        lin(p + "q_proj", D, D)
        lin(p + "k_proj", D, D, bias=False)
        lin(p + "v_proj", D, D)
        lin(p + "out_proj", D, D)
    e = "model.encoder."
    sd[e + "conv1.weight"] = torch.randn(D, dims.n_mels, 3, generator=g, device=device) * 0.02
    sd[e + "conv1.bias"] = torch.zeros(D, device=device)
    sd[e + "conv2.weight"] = torch.randn(D, D, 3, generator=g, device=device) * 0.02
    sd[e + "conv2.bias"] = torch.zeros(D, device=device)
    sd[e + "embed_positions.weight"] = helpers.sinusoids(dims.max_source_positions, D).to(device)
    for i in range(dims.enc_layers):
        p = f"{e}layers.{i}."
        attn(p + "self_attn.")
        ln(p + "self_attn_layer_norm")
        lin(p + "fc1", F, D)
        lin(p + "fc2", D, F)
        ln(p + "final_layer_norm")
    ln(e + "layer_norm")
    dd = "model.decoder."
    sd[dd + "embed_tokens.weight"] = torch.randn(V, D, generator=g, device=device) * 0.02
    sd[dd + "embed_positions.weight"] = torch.randn(dims.max_target_positions, D, generator=g, device=device) * 0.02
    for i in range(dims.dec_layers):
        p = f"{dd}layers.{i}."
        attn(p + "self_attn.")
        ln(p + "self_attn_layer_norm")
        attn(p + "encoder_attn.")
        ln(p + "encoder_attn_layer_norm")
        lin(p + "fc1", F, D)
        lin(p + "fc2", D, F)
        ln(p + "final_layer_norm")
    ln(dd + "layer_norm")
    return sd


def run_own(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    import helpers
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline
    from turbo_whisper_workspace_b200.scheduler import DistributedWindowScheduler

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 engine has no CPU path (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = WINDOWS_PER_GPU
    dims = WhisperDims.large_v3_turbo()
    sd = helpers.random_state_dict(dims, 0, "hf")
    tok = helpers.build_tokenizer()
    MB = args.max_batch                     # decode rows per engine context = windows per generate call
    if MB % B:
        raise SystemExit("bench.py: --max-batch must be a multiple of 24")
    pipe = B200WhisperPipeline(sd, dims, tok, devices=[dev], max_batch=MB, contexts_per_device=args.contexts)
    del sd
    engines = pipe.scheduler.flat_engines
    K = args.steps
    clips = [helpers.synth_clip(rank * B + i) for i in range(B)]
    audio = np.concatenate(clips * K)                  # K x 720 s host PCM for the e2e call (K micro-batches)
    kw = dict(chunk_length_s=30, stride_length_s=0, batch_size=B, generate_kwargs={"task": "transcribe"},
              return_timestamps=True)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def stats_sum(key):
        return sum(e.stats.get(key, 0) for e in engines)

    from turbo_whisper_workspace_b200.scheduler import balanced_microbatch

    def run_resident(n_steps):
        """n_steps steps (24 windows each) over the PCM already resident in each context's HBM buffer.  The windows are
        cut into equally sized generate calls exactly as the chunk scheduler cuts a job (`balanced_microbatch`: as few
        calls as keep every context busy, at most MB windows each); the contexts take the calls round-robin on their
        own streams.  Returns per-context end events and the rows of every call, in call order."""
        ends, errs = [None] * len(engines), []
        n_win = n_steps * B
        mb = balanced_microbatch(n_win, len(engines), MB)
        calls = [min(mb, n_win - a) for a in range(0, n_win, mb)]
        rows = [None] * len(calls)

        def work(ci):
            try:
                eng = engines[ci]
                with torch.cuda.stream(eng.stream) if eng.stream is not None else torch.cuda.stream(torch.cuda.current_stream()):
                    for k in range(ci, len(calls), len(engines)):
                        eng.features(calls[k])
                        rows[k] = eng.generate(calls[k])
                    ev = torch.cuda.Event(enable_timing=True)
                    ev.record()
                    ends[ci] = ev
            except BaseException as ex:
                errs.append(ex)
        ths = [threading.Thread(target=work, args=(ci,)) for ci in range(len(engines))]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if errs:
            raise errs[0]
        return ends, rows

    # ---- device-resident leg ("value")
    res_clips = clips * (MB // B)
    for eng in engines:
        if eng.stream is not None:
            with torch.cuda.stream(eng.stream):
                eng.load_pcm(res_clips)
        else:
            eng.load_pcm(res_clips)
    torch.cuda.synchronize()
    for _ in range(-(-args.warmup // K)):  # >= W warm-up steps, cut into the SAME call sizes as the timed region
        run_resident(K)                    # (a CUDA graph is captured per distinct row count: none inside the timing)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0, d0, w0, r0_ = stats_sum("launches"), stats_sum("dec_steps"), stats_sum("enc_windows"), stats_sum("dec_row_steps")
    e0 = torch.cuda.Event(enable_timing=True)
    e0.record()
    torch.cuda.synchronize()      # every context stream starts after e0
    ends, rows = run_resident(K)
    barrier()
    t_dev = max(e0.elapsed_time(ev) for ev in ends if ev is not None) / 1e3
    launches = stats_sum("launches") - l0
    dec_steps = stats_sum("dec_steps") - d0
    enc_windows = stats_sum("enc_windows") - w0
    dec_row_steps = stats_sum("dec_row_steps") - r0_

    # ---- end-to-end leg through the reference-facing callable
    pipe(audio[:B * 480000 * min(K, len(engines))], **kw)      # warm-up of the call path
    barrier()
    h0, dd0 = stats_sum("h2d_bytes"), stats_sum("d2h_bytes")
    t0 = time.perf_counter()
    result = pipe(audio, **kw)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    clocks = sampler.stop()
    h2d = (stats_sum("h2d_bytes") - h0) // max(K, 1)
    d2h = (stats_sum("d2h_bytes") - dd0) // max(K, 1)
    e2e_rows = list(pipe.last_token_rows)

    # ---- output check: the e2e rows (4 contexts, host path) == ONE context decoding the same 24 windows
    single = engines[0].generate_from_pcm(clips) if engines[0].stream is None else None
    if single is None:
        with torch.cuda.stream(engines[0].stream):
            single = engines[0].generate_from_pcm(clips)
    rows_ok = len(e2e_rows) == K * B and all(e2e_rows[i] == single[i % B] for i in range(len(e2e_rows)))
    # window i of every call decodes clips[i % B] (the resident buffer holds the 24 clips repeated)
    resident_ok = all(r[i] == single[i % B] for r in rows for i in range(len(r)))

    # ---- rooflines of the dominant kernels, measured live
    pk = peaks()
    eng0 = engines[0]
    stream_ctx = torch.cuda.stream(eng0.stream) if eng0.stream is not None else torch.cuda.stream(torch.cuda.current_stream())
    with stream_ctx:
        eng0.load_pcm(clips)
        eng0.features(B)
        enc_ms = cuda_timed(lambda: eng0.encode(B), iters=3, warm=1)
        ca24_ms, ca24_bytes = cross_attn_roofline_probe(eng0, B)
        gemm_ms, gemm_flops = gemm_roofline_probe(eng0, B)
        step_us, step_bytes = decode_step_probe(eng0, B)
        # the same two probes at the row count of the timed region's generate calls (the launches the bench really makes)
        R = balanced_microbatch(K * B, len(engines), MB)
        if R != B:
            eng0.load_pcm((clips * (-(-R // B)))[:R])
            eng0.features(R)
            eng0.encode(R)
            ca_ms, ca_bytes = cross_attn_roofline_probe(eng0, R, iters=12)
            stepR_us, stepR_bytes = decode_step_probe(eng0, R, steps=128)
        else:
            ca_ms, ca_bytes, stepR_us, stepR_bytes = ca24_ms, ca24_bytes, step_us, step_bytes

    t_dev, t_e2e = max_over_ranks(t_dev, t_e2e)
    audio_s = WINDOW_S * B * world * K
    traffic = ncu_traffic()
    line = None
    if rank == 0:
        ca_gbs = ca_bytes / (ca_ms * 1e-3) / 1e9
        ca24_gbs = ca24_bytes / (ca24_ms * 1e-3) / 1e9
        gemm_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12
        enc_flops = B * (ENC_FLOPS_PER_WINDOW + dims.dec_layers * 4 * 1500 * 1280 ** 2)
        enc_tf = enc_flops / (enc_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": audio_s / t_dev, "unit": "x realtime",
            "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": t_dev / K * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(world),
            "detail": {"contexts_per_gpu": len(engines), "max_windows_per_generate_call": MB,
                       "scheduling": "a step is 24 windows (the pipeline call's batch_size); the chunk scheduler packs the "
                                     "windows of the timed region into equally sized generate calls of up to 96 windows per "
                                     "engine context — one pass over the decoder weights per decode step for all rows of a "
                                     "call; results are batch-invariant (output_check)",
                       "decoder_steps_per_step": dec_steps // K,
                       "encoder_windows_per_step": enc_windows // K},
            "e2e": {"value": audio_s / t_e2e, "unit": "x realtime", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": t_e2e / K * 1e3,
                    "api": "B200WhisperPipeline.__call__(np.ndarray[steps*720 s], chunk_length_s=30, stride_length_s=0, "
                           "batch_size=24, return_timestamps=True)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "decode_attn_kernel (cross-attention over the encoder K/V; largest "
                                                   "single kernel of a step by time)",
                         "achieved": ca_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ca_gbs / pk["hbm_gbs"],
                         "traffic": traffic.get("decode_attn_kernel" if R == B else "decode_attn_kernel_%d_rows" % R),
                         "traffic_source": traffic.get("source"),
                         "peak_source": pk["source"], "bytes_per_launch": ca_bytes, "ms_per_launch": ca_ms,
                         "rows_per_launch": R,
                         "note": "timed at the row count of the timed region's generate calls; the peak is the measured COPY "
                                 "bandwidth (read + write), a read-only stream can exceed it slightly",
                         "at_24_rows": {"achieved": ca24_gbs, "frac": ca24_gbs / pk["hbm_gbs"], "ms_per_launch": ca24_ms,
                                        "bytes_per_launch": ca24_bytes, "traffic": traffic.get("decode_attn_kernel")}},
            "roofline_encoder_gemm": {"bound": "tensor", "kernel": "gemm_bf16_2cta_kernel (tcgen05; encoder qkv/out/fc1/fc2 "
                                      "shapes, fused bias/GELU/residual)", "achieved": gemm_tf,
                                      "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": gemm_tf / pk["bf16_tflops"],
                                      "traffic": traffic.get("gemm_bf16_2cta_kernel"),
                                      "traffic_source": traffic.get("source"),
                                      "peak_source": pk["source"] + " burst",
                                      "flops_per_launch": gemm_flops, "ms_per_launch": gemm_ms},
            "encoder": {"bound": "tensor", "what": "whole encoder pass at batch 24 (conv stem, 32 layers incl. attention "
                        "and LayerNorm, final LN, cross-K/V GEMM), one context alone", "ms": enc_ms,
                        "achieved": enc_tf, "unit": "TFLOP/s", "frac_burst": enc_tf / pk["bf16_tflops"],
                        "frac_sustained": enc_tf / pk["bf16_tflops_sustained"], "flops": enc_flops},
            "decode_step": {"bound": "hbm", "what": "one greedy step at 24 rows, one context alone (graph replays)",
                            "us": step_us, "bytes": step_bytes, "floor_us": step_bytes / pk["hbm_gbs"] / 1e3,
                            "frac": step_bytes / pk["hbm_gbs"] / 1e3 / step_us,
                            "launches_per_step": eng0.launches_per_step,
                            # decode share of the timed region per 24-row step: (time - encoder passes at the alone rate)
                            # / (decode row-steps / 24)
                            "in_bench_us": max(0.0, t_dev * 1e6 - (enc_windows / B) * enc_ms * 1e3) / max(1.0, dec_row_steps / B),
                            "in_bench_note": "per 24 decode rows; calls decode up to 96 rows per step",
                            "at_call_rows": {"rows": R, "us": stepR_us, "us_per_24_rows": stepR_us * B / R,
                                             "bytes": stepR_bytes, "floor_us": stepR_bytes / pk["hbm_gbs"] / 1e3,
                                             "frac": stepR_bytes / pk["hbm_gbs"] / 1e3 / stepR_us}},
            "output_check": {"chunks": len(result["chunks"]) if isinstance(result, dict) else None,
                             "rows": len(e2e_rows), "tokens_first_row": len(single[0]) if single else None,
                             "e2e_rows_equal_single_context": bool(rows_ok),
                             "resident_rows_equal_single_context": bool(resident_ok)},
        }

    # ---- extras: the other BASELINE.json configs
    if not args.no_extras:
        extras = run_extras(args, rank, world, dev, pipe, dims, tok, barrier, max_over_ranks, pk)
        if line is not None:
            line.update(extras)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_subprocess(args.reference_budget_s)
        if args.dump_outputs:
            # the timed region's last step: its last B windows, in the order the calls cover them
            dump_outputs(args.dump_outputs, [r for call in rows for r in call][-B:])
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and not (rows_ok and resident_ok):
        sys.stderr.write("bench.py: OUTPUT CHECK FAILED — multi-context rows differ from the single-context rows\n")
        return 1
    return 0


def run_extras(args, rank, world, dev, pipe, dims, tok, barrier, max_over_ranks, pk):
    out = {}
    want = {x.strip() for x in args.extras.split(",") if x.strip()}
    if "config3" in want:
        out["config3"] = extra_config3(rank, world, pipe, dims, tok, barrier, max_over_ranks)
    if "config2_beams5" in want:
        out["config2_beams5"] = extra_beams5(rank, world, pipe, barrier, max_over_ranks)
    if "config4" in want:
        out["config4"] = extra_config4(rank, world, dev, barrier, max_over_ranks, pk)
    if "config5" in want:
        if rank == 0:       # the other ranks wait at the barrier
            out["config5"] = extra_config5(dev, pipe, dims, pk)
        barrier()
    return out


def extra_config3(rank, world, pipe, dims, tok, barrier, max_over_ranks):
    import numpy as np
    import torch
    import helpers
    from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline
    from turbo_whisper_workspace_b200.scheduler import DistributedWindowScheduler
    # ---- config 3: ONE 1 h file through the pipeline callable, windows sharded over the ranks by the chunk scheduler
    hour = np.concatenate([helpers.synth_clip(1000 + i) for i in range(120)])          # 3600 s, same on every rank
    dpipe = pipe if world == 1 else B200WhisperPipeline(
        None, dims, tok, scheduler=DistributedWindowScheduler(pipe.scheduler, rank, world))
    c3 = {"what": "one 1 h synthetic file through B200WhisperPipeline.__call__ (host PCM in, dict with chunk-level "
                  "timestamps out); the windows of the ONE job are sharded over the ranks' engine contexts by the "
                  "chunk scheduler (strong scaling), token ids gathered on the host", "n_gpus": world}
    for name, cl, st, bs in (("30_5", 30, 5, 24), ("60_5_literal", 60, 5, 512)):
        ckw = dict(chunk_length_s=cl, stride_length_s=st, batch_size=bs, generate_kwargs={"task": "transcribe"},
                   return_timestamps=True)
        dpipe(hour[:16000 * 400], **ckw)                  # warm-up (graphs of the micro-batch size, call path)
        dpipe(hour, **ckw)
        barrier()
        t0 = time.perf_counter()
        r = dpipe(hour, **ckw)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        (dt,) = max_over_ranks(dt)
        rec = {"windows": dpipe.last_stats.get("windows"), "seconds": dt, "rtfx": 3600.0 / dt,
               "chunks": len(r["chunks"]), "last_timestamp": list(r["chunks"][-1]["timestamp"]) if r["chunks"] else None,
               "microbatches": [b - a for a, b in pipe.scheduler.last_stats.get("microbatches", [])][:8]}
        if world > 1:
            barrier()
            if rank == 0:       # the same job on rank 0 alone: the gathered result must be identical
                rec["equal_to_one_gpu"] = bool(pipe(hour, **ckw) == r)
            barrier()
        c3[name] = rec
    return c3


def extra_beams5(rank, world, pipe, barrier, max_over_ranks):
    import numpy as np
    import torch
    import helpers
    # ---- config 2 with the reference's LITERAL decoding mode (transformers >= 4.53 pipelines default to num_beams = 5 and
    # the reference passes only generate_kwargs={"task": ...}): 24 windows per GPU through the callable, beam search on the device
    bclips = np.concatenate([helpers.synth_clip(rank * WINDOWS_PER_GPU + i) for i in range(WINDOWS_PER_GPU)])
    bkw = dict(chunk_length_s=30, stride_length_s=0, batch_size=WINDOWS_PER_GPU, return_timestamps=True,
               generate_kwargs={"task": "transcribe", "num_beams": 5})
    pipe(bclips, **bkw)
    barrier()
    t0 = time.perf_counter()
    rb = pipe(bclips, **bkw)
    torch.cuda.synchronize()
    (dtb,) = max_over_ranks(time.perf_counter() - t0)
    return {"what": "config 2's 24 windows per GPU with generate_kwargs={'num_beams': 5} (the reference's literal "
                                     "decoding mode under transformers >= 4.53): windows x beams decode rows, tw_beam_step on the "
                                     "device, one CUDA graph per position", "n_gpus": world, "seconds": dtb,
                             "rtfx": WINDOWS_PER_GPU * WINDOW_S * world / dtb, "chunks": len(rb["chunks"]),
                             "microbatches": [b - a for a, b in pipe.scheduler.last_stats.get("microbatches", [])]}


def extra_config4(rank, world, dev, barrier, max_over_ranks, pk):
    import torch
    import helpers
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    # ---- config 4: large-v3 (32 decoder layers), batch 16 per GPU, decoder-heavy greedy decode
    torch.cuda.empty_cache()
    d4 = WhisperDims.large_v3()
    e4 = WhisperEngine(d4, synth_state_dict_on_device(d4, dev, 0), device=dev, max_batch=16)
    c4clips = [helpers.synth_clip(2000 + rank * 16 + i) for i in range(16)]
    e4.generate_from_pcm(c4clips)
    barrier()
    s0, t0 = e4.stats["dec_steps"], time.perf_counter()
    rows4 = e4.generate_from_pcm(c4clips)
    torch.cuda.synchronize()
    dt4 = time.perf_counter() - t0
    steps4 = e4.stats["dec_steps"] - s0
    step_us4, step_bytes4 = decode_step_probe(e4, 16)
    (dt4,) = max_over_ranks(dt4)
    rec = {"what": "whisper-large-v3 dims (32 decoder layers), bf16, 16 windows per GPU in one batch, greedy "
                              "with timestamps, random-init (decodes to max_length: decoder-heavy); one engine context",
                      "n_gpus": world, "seconds": dt4, "rtfx": 16 * WINDOW_S * world / dt4, "decoder_steps": steps4,
                      "tokens_first_rows": [len(r) for r in rows4[:4]],
                      "decode_step": {"us": step_us4, "bytes": step_bytes4, "floor_us": step_bytes4 / pk["hbm_gbs"] / 1e3,
                                      "frac": step_bytes4 / pk["hbm_gbs"] / 1e3 / step_us4,
                                      "launches_per_step": e4.launches_per_step}}
    del e4
    torch.cuda.empty_cache()
    return rec


def extra_config5(dev, pipe, dims, pk):
    import torch
    import helpers
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    # ---- config 5: log-mel + encoder-only sweep
    if True:
        batches = [1, 2, 4, 8, 16, 24, 32, 64, 128, 256]
        e5 = WhisperEngine(dims, None, device=dev, max_batch=24, max_enc_batch=max(batches),
                           shared_weights=pipe.scheduler.flat_engines[0].w)
        base = [helpers.synth_clip(3000 + i) for i in range(8)]
        sweep = []
        for Bs in batches:
            e5.load_pcm([base[i % 8] for i in range(Bs)])
            torch.cuda.synchronize()
            mel_ms = cuda_timed(lambda: e5.features(Bs), iters=10 if Bs <= 32 else 4, warm=2)
            enc_ms = cuda_timed(lambda: e5.encode(Bs), iters=3 if Bs <= 32 else 1, warm=1)
            mel_bytes = Bs * (480000 * 4 + 128 * 3000 * 2)
            enc_flops = Bs * (ENC_FLOPS_PER_WINDOW + dims.dec_layers * 4 * 1500 * 1280 ** 2)
            sweep.append({"batch": Bs, "logmel_ms": round(mel_ms, 4), "logmel_GBps": round(mel_bytes / mel_ms / 1e6, 1),
                          "logmel_frac_hbm": round(mel_bytes / mel_ms / 1e6 / pk["hbm_gbs"], 3),
                          "encoder_ms": round(enc_ms, 3), "encoder_TFLOPs": round(enc_flops / enc_ms / 1e9, 1),
                          "encoder_frac_burst": round(enc_flops / enc_ms / 1e9 / pk["bf16_tflops"], 3)})
        rec = {"what": "log-mel front end (fp32 PCM in, bf16 time-major features out: 2.688 MB / window) and "
                                  "encoder-only pass (2.2738 TFLOP + cross-K/V GEMM per window), one context, CUDA events",
               "sweep": sweep}
        del e5
        torch.cuda.empty_cache()
    return rec


def dump_outputs(out_dir: str, rows) -> None:
    """What the timed path's generate calls returned for the windows of its last step, so that two builds can be compared
    output for output: token_ids.npy [windows, longest row] (-1 after the end of a row) and token_counts.npy [windows],
    float32 (every id below 2**24 is exact)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    ids = np.full((len(rows), max((len(r) for r in rows), default=0)), -1, dtype=np.float32)
    for b, r in enumerate(rows):
        ids[b, :len(r)] = r
    np.save(os.path.join(out_dir, "token_ids.npy"), ids)
    np.save(os.path.join(out_dir, "token_counts.npy"), np.array([len(r) for r in rows], dtype=np.float32))


_RESULT_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version
    banner on fd 1 under torchrun), so fd 1 is pointed at stderr for the whole run and the result line goes
    to a private duplicate of the original stdout."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config3 / config4 / config5 extra keys")
    ap.add_argument("--extras", default="config3,config2_beams5,config4,config5",
                    help="comma-separated subset of the extra keys to measure")
    ap.add_argument("--contexts", type=int, default=5, help="engine contexts (streams) per GPU sharing one weight copy")
    ap.add_argument("--max-batch", type=int, default=96,
                    help="most windows per generate call of an engine context (multiple of 24, <= 96): the decoder weights "
                         "are streamed once per decode step for all rows of a call")
    ap.add_argument("--no-literal-beams", action="store_true",
                    help="reference arm: skip the extra call in the reference's literal num_beams = 5 mode")
    ap.add_argument("--reference-budget-s", type=float, default=480.0,
                    help="reference arm: stop after the call that crosses this wall-clock budget (steps reports the calls made)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="own arm: after the timed steps, write the token ids of the last timed step's windows (rank 0) "
                         "as DIR/*.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""       # the reference arm is the CPU path; set before torch is imported
        return run_reference(args, rank, world)
    if args.warmup < 3:
        args.warmup = 3
    return run_own(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
