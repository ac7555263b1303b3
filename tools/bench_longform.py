"""Un-chunked long-form throughput (many clips > 30 s without chunk_length_s): one JSON line per arm, alternated in one
call on the same seeded clips and the same engines.
  (a) per_clip     WindowScheduler.run_long per clip in sequence (one decode row on the first context of the first GPU)
  (b) many_1gpu    WindowScheduler.run_long_many on one GPU (its engine contexts, rows refilled from a shared queue)
  (c) many_all     WindowScheduler.run_long_many on every visible GPU
Per arm: wall seconds (host clock around calls that end with the results on the host), RTFx = audio seconds / wall
seconds, windows encoded, decode steps, seek iterations and mean active rows per iteration, the clips whose ids equal arm
(a)'s, the card name and power limit read in the same call.  Random weights (bench.synth_state_dict_on_device) seldom
emit EOS, so nearly every window decodes to max_length: the step counts are what make the arms comparable.

    python tools/bench_longform.py [--clips 48] [--min-s 60] [--max-s 600] [--contexts 4] [--max-batch 24] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001
        power = None
    return name, power


def make_clips(n, lo_s, hi_s, seed=0):
    import helpers
    rng = np.random.default_rng(seed)
    secs = rng.uniform(lo_s, hi_s, size=n)
    return [np.concatenate([helpers.synth_clip(seed * 1000 + i * 17 + k, kind="mod") for k in range(int(s // 30) + 1)])
            [:int(s * 16000)] for i, s in enumerate(secs)]


def counters(engines):
    keys = ("enc_windows", "dec_steps", "long_iterations", "long_windows")
    return {k: sum(int(e.stats.get(k, 0)) for e in engines) for k in keys}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=48)
    ap.add_argument("--min-s", type=float, default=60.0)
    ap.add_argument("--max-s", type=float, default=600.0)
    ap.add_argument("--contexts", type=int, default=4)
    ap.add_argument("--max-batch", type=int, default=24)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_longform.py needs a CUDA device")
    from bench import synth_state_dict_on_device
    from turbo_whisper_workspace_b200.config import GenerationSettings, WhisperDims
    from turbo_whisper_workspace_b200.scheduler import WindowScheduler
    name, power = gpu_info()
    n_gpu = torch.cuda.device_count()
    dims = WhisperDims.large_v3_turbo()
    gen = GenerationSettings()
    sd = synth_state_dict_on_device(dims, "cuda:0")
    one = WindowScheduler(sd, dims, gen, ["cuda:0"], args.max_batch, contexts_per_device=args.contexts)
    every = one if n_gpu == 1 else WindowScheduler(sd, dims, gen, [f"cuda:{i}" for i in range(n_gpu)], args.max_batch,
                                                   contexts_per_device=args.contexts)
    del sd
    clips = make_clips(args.clips, args.min_s, args.max_s)
    audio_s = sum(c.shape[0] for c in clips) / 16000.0
    kw = dict(task="transcribe", language=None)
    arms = {
        "per_clip": (one, lambda: [one.run_long(c, **kw) for c in clips]),
        "many_1gpu": (one, lambda: one.run_long_many(clips, **kw)),
        "many_all": (every, lambda: every.run_long_many(clips, **kw)),
    }
    # warm-up: modules, kernel attributes and the step graphs of small row counts, on two short clips
    warm = make_clips(2, 31.0, 40.0, seed=1)
    one.run_long(warm[0], **kw)
    one.run_long_many(warm, **kw)
    if every is not one:
        every.run_long_many(warm, **kw)
    out = open(args.out, "a") if args.out else None
    ids = {}
    for arm, (sched, fn) in arms.items():
        engines = sched.flat_engines
        for d in sched.devices:
            torch.cuda.synchronize(d)
        c0 = counters(engines)
        t0 = time.perf_counter()
        ids[arm] = fn()
        wall = time.perf_counter() - t0
        c1 = counters(engines)
        d = {k: c1[k] - c0[k] for k in c1}
        line = {"arm": arm, "clips": len(clips), "audio_s": round(audio_s, 1), "wall_s": round(wall, 3),
                "rtfx": round(audio_s / wall, 2), "windows": d["enc_windows"], "decode_steps": d["dec_steps"],
                "seek_iterations": d["long_iterations"],
                "mean_active_rows": round(d["long_windows"] / max(1, d["long_iterations"]), 2),
                "identical_to_per_clip": sum(a == b for a, b in zip(ids[arm], ids["per_clip"])),
                "gpus": 1 if sched is one else n_gpu, "contexts_per_device": args.contexts, "max_batch": args.max_batch,
                "model": "large-v3-turbo (random weights)", "device": name, "power_limit_w": power}
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()
    if out:
        out.close()


if __name__ == "__main__":
    main()
