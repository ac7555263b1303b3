#!/usr/bin/env python
"""Throughput of every served Whisper checkpoint shape on one GPU: bench.py's device-resident workload (24 x 30 s
windows per step, 0.1*N(0,1) audio, greedy with timestamps, the library's default of 4 engine contexts) on random
HF-init weights of each preset, plus the encoder and decode-step times of one context and the log-mel time at 80 and
128 bins.  One JSON line per preset goes to stdout and to profiles/checkpoints_<card>.jsonl (or --out).

    python tools/bench_checkpoints.py [--steps 2] [--warmup 1] [--presets large_v3_turbo,medium] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402  (workload helpers: synth_state_dict_on_device, cuda_timed, decode_step_probe)

# preset -> (WhisperDims factory, decoder layers override); distil-large-v2 is large-v2 with 2 decoder layers
PRESETS = {
    "large_v3_turbo": ("large_v3_turbo", None),
    "large_v3": ("large_v3", None),
    "large_v2": ("large_v2", None),
    "distil_large_v2": ("large_v2", 2),
    "medium": ("medium", None),
    "small": ("small", None),
    "base": ("base", None),
}
B = bench.WINDOWS_PER_GPU


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, limit = [s.strip() for s in out.split(",")]
    return name, limit


def logmel_ms(dev, n_mels, iters=20):
    import numpy as np
    import torch
    import helpers
    from turbo_whisper_workspace_b200 import ops
    lm = ops.LogMel(dev, B, n_mels)
    pcm = torch.from_numpy(np.stack([helpers.synth_clip(i) for i in range(B)])).to(dev)
    out_t = torch.zeros(B, 3002, n_mels, dtype=torch.bfloat16, device=dev)
    return bench.cuda_timed(lambda: lm(pcm, None, out_t=out_t, out_t_row_off=1), iters, warm=3)


def run_preset(name, dev, steps, warmup):
    import torch
    import helpers
    import helpers_v2
    from turbo_whisper_workspace_b200.config import GenerationSettings, WhisperDims
    from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline
    factory, dec_layers = PRESETS[name]
    dims = getattr(WhisperDims, factory)()
    if dec_layers is not None:
        dims.dec_layers = dec_layers
    v2 = dims.n_mels == 80
    tok = helpers_v2.build_tokenizer() if v2 else helpers.build_tokenizer()
    gen = helpers_v2.generation_settings() if v2 else GenerationSettings()
    sd = bench.synth_state_dict_on_device(dims, dev, 0)
    pipe = B200WhisperPipeline(sd, dims, tok, gen, devices=[dev], max_batch=B)
    del sd
    engines = pipe.scheduler.flat_engines
    clips = [helpers.synth_clip(i) for i in range(B)]
    for eng in engines:
        with torch.cuda.stream(eng.stream) if eng.stream is not None else torch.cuda.stream(torch.cuda.current_stream()):
            eng.load_pcm(clips)
    torch.cuda.synchronize()

    def run_resident(n_steps):
        """n_steps generate calls of 24 windows, round-robin over the contexts, each on its own stream."""
        ends, errs = [None] * len(engines), []

        def work(ci):
            try:
                eng = engines[ci]
                with torch.cuda.stream(eng.stream) if eng.stream is not None else torch.cuda.stream(torch.cuda.current_stream()):
                    for _ in range(ci, n_steps, len(engines)):
                        eng.features(B)
                        eng.generate(B)
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
        return ends

    run_resident(max(warmup, len(engines)))
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True)
    e0.record()
    torch.cuda.synchronize()
    ends = run_resident(steps)
    torch.cuda.synchronize()
    t = max(e0.elapsed_time(ev) for ev in ends if ev is not None) / 1e3
    eng0 = engines[0]
    with torch.cuda.stream(eng0.stream) if eng0.stream is not None else torch.cuda.stream(torch.cuda.current_stream()):
        eng0.features(B)
        enc_ms = bench.cuda_timed(lambda: eng0.encode(B), iters=3, warm=1)
        step_us, _ = bench.decode_step_probe(eng0, B)
    res = {"preset": name, "d_model": dims.d_model, "enc_layers": dims.enc_layers, "dec_layers": dims.dec_layers,
           "n_mels": dims.n_mels, "vocab": dims.vocab, "contexts": len(engines), "steps": steps,
           "windows": steps * B, "rtfx": round(bench.WINDOW_S * B * steps / t, 1),
           "encoder_ms_per_window": round(enc_ms / B, 3), "decode_step_us_one_context_24_rows": round(step_us, 1)}
    del pipe, engines, eng0
    torch.cuda.empty_cache()
    return res


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2, help="timed steps of 24 windows per preset")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--presets", default=",".join(PRESETS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_checkpoints.py: needs a CUDA device (no CPU path)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, limit = card()
    lm = {n: round(logmel_ms(dev, n), 4) for n in (128, 80)}
    out = args.out or os.path.join(ROOT, "profiles", "checkpoints_" + name.replace(" ", "_") + ".jsonl")
    with open(out, "w") as f:
        for p in args.presets.split(","):
            r = run_preset(p, dev, args.steps, args.warmup)
            r.update({"logmel_ms_24_windows": lm[r["n_mels"]], "logmel_ms_24_windows_80": lm[80],
                      "logmel_ms_24_windows_128": lm[128], "card": name, "power_limit": limit})
            line = json.dumps(r)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
