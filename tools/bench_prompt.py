"""Prompted decoding (generate(prompt_ids=...)) on one GPU: the batched decoder prefill against the same prompt fed
as forced decode steps.  One JSON line per (shape, rows, prompt length):
  * call_ms          one decode call: prefill (or the 3 forced special tokens when the prompt is empty) + 64 generated
                     steps (CUDA graph replays), host clock around work that ends in a device synchronise
  * prefill_ms       the prefill alone (CUDA events), split into gemm_ms / attn_ms / other_ms (embedding, LayerNorms,
                     K / V scatter); events between every launch, so the split carries a little event overhead
  * forced_ms        the same P-1 prompt positions as forced steps: P-1 replays of the step graph (CUDA events)
  * capture_ms       capture of the step graph of a prompt length not seen before (the graph cache key holds the
                     grammar's begin index, i.e. the prompt length)
  * device, power_limit_w   read in the same run
Random weights (N(0, 0.02)) and synthetic audio; the times do not depend on the values.  Prompt length 0 = the
unprompted call (forced special tokens, the benchmarked path).

    python tools/bench_prompt.py [--out FILE] [--shapes large_v3_turbo,large_v3] [--rows 24,96] [--lengths 0,16,64,128,224]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GEN_STEPS = 64


def random_state_dict(dims, device, seed=0):
    """HF-layout weights drawn on the device (the full-size models are too slow to draw on the host)."""
    g = torch.Generator(device=device).manual_seed(seed)
    D, F, V = dims.d_model, dims.ffn, dims.vocab
    r = lambda *s: torch.randn(*s, generator=g, device=device) * 0.02
    sd = {}
    e, d = "model.encoder.", "model.decoder."
    sd[e + "conv1.weight"], sd[e + "conv1.bias"] = r(D, dims.n_mels, 3), r(D)
    sd[e + "conv2.weight"], sd[e + "conv2.bias"] = r(D, D, 3), r(D)
    sd[e + "embed_positions.weight"] = r(dims.max_source_positions, D)

    def layer(p, cross):
        for a in ("self_attn.",) + (("encoder_attn.",) if cross else ()):
            for n in ("q", "k", "v", "out"):
                sd[p + a + n + "_proj.weight"] = r(D, D)
                if n != "k":
                    sd[p + a + n + "_proj.bias"] = r(D)
        for n in ("self_attn_layer_norm", "final_layer_norm") + (("encoder_attn_layer_norm",) if cross else ()):
            sd[p + n + ".weight"], sd[p + n + ".bias"] = 1 + r(D), r(D)
        sd[p + "fc1.weight"], sd[p + "fc1.bias"] = r(F, D), r(F)
        sd[p + "fc2.weight"], sd[p + "fc2.bias"] = r(D, F), r(D)
    for i in range(dims.enc_layers):
        layer(f"{e}layers.{i}.", False)
    sd[e + "layer_norm.weight"], sd[e + "layer_norm.bias"] = 1 + r(D), r(D)
    sd[d + "embed_tokens.weight"] = r(V, D)
    sd[d + "embed_positions.weight"] = r(dims.max_target_positions, D)
    for i in range(dims.dec_layers):
        layer(f"{d}layers.{i}.", True)
    sd[d + "layer_norm.weight"], sd[d + "layer_norm.bias"] = 1 + r(D), r(D)
    return sd


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001
        power = None
    return name, power


def event_ms(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default="large_v3_turbo,large_v3")
    ap.add_argument("--rows", default="24,96")
    ap.add_argument("--lengths", default="0,16,64,128,224")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_prompt.py needs a CUDA device")
    import helpers
    from turbo_whisper_workspace_b200.config import WhisperDims, resolve_generate_options
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    rows = [int(v) for v in args.rows.split(",")]
    lengths = [int(v) for v in args.lengths.split(",")]
    out = open(args.out, "w") if args.out else None
    SOT, EN, TRANSCRIBE, PREV = 50258, 50259, 50360, 50361
    for shape in args.shapes.split(","):
        dims = getattr(WhisperDims, shape)()
        sd = random_state_dict(dims, dev)
        eng = WhisperEngine(dims, sd, device=dev, max_batch=max(rows))
        del sd
        torch.cuda.empty_cache()
        clips = [helpers.synth_clip(i % 8, kind="mod" if i % 2 else "noise") for i in range(max(rows))]
        for R in rows:
            B = eng.load_pcm(clips[:R])
            eng.features(B)
            eng.encode(B)
            prompts = torch.tensor([[SOT, EN, TRANSCRIBE]] * R, dtype=torch.int32)
            for n in lengths:
                ids = None if n == 0 else [PREV] + [1000 + (7 * i) % 40000 for i in range(n - 1)]
                P = resolve_generate_options(dims, eng.gen, prompt_ids=ids).prompt_len
                # capture of a new prompt length: drop the cached step graphs of this shape first
                eng._graphs = {k: v for k, v in eng._graphs.items() if not (k[0] == R and k[2] == P)}
                eng.decode(R, prompts, n_steps=1, prompt_ids=ids)       # warm-up: tables, kernels, prefill weights
                eng._graphs = {k: v for k, v in eng._graphs.items() if not (k[0] == R and k[2] == P)}
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                eng._graph_for(R)
                torch.cuda.synchronize()
                capture_ms = (time.perf_counter() - t0) * 1e3
                # one call: prefill + GEN_STEPS generated steps (eos checks disabled so that every call runs them all)
                keep, eng.finish_check_every = eng.finish_check_every, 0
                calls = []
                for _ in range(3):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    eng.decode(R, prompts, n_steps=GEN_STEPS + (2 if ids is None else 0), prompt_ids=ids)
                    torch.cuda.synchronize()
                    calls.append((time.perf_counter() - t0) * 1e3)
                eng.finish_check_every = keep
                line = {"shape": shape, "rows": R, "prompt_ids": n, "decoder_prompt": P, "gen_steps": GEN_STEPS,
                        "call_ms": round(min(calls), 3), "call_ms_all": [round(c, 3) for c in calls],
                        "capture_ms": round(capture_ms, 2), "device": name, "power_limit_w": power}
                if ids is not None:
                    pf = []
                    for _ in range(5):
                        ph = {}
                        total = event_ms(lambda: eng.prefill(R, P))
                        eng.prefill(R, P, timing=ph)
                        pf.append((total, ph))
                    best = min(pf, key=lambda t: t[0])
                    line.update(prefill_ms=round(best[0], 3), gemm_ms=round(best[1].get("gemm", 0.0), 3),
                                attn_ms=round(best[1].get("attn", 0.0), 3), other_ms=round(best[1].get("other", 0.0), 3))
                    # the same prompt positions through the existing route: P-1 replays of the unprompted step graph,
                    # every repetition from position 1 again (the rows must stay within max_length positions)
                    def forced():
                        eng.decode(R, prompts, n_steps=1)
                        g = eng._graph_for(R)
                        assert P < eng.max_len
                        return event_ms(g.replay, P - 1) * (P - 1)
                    line["forced_ms"] = round(min(forced() for _ in range(3)), 3)
                    line["prefill_speedup"] = round(line["forced_ms"] / line["prefill_ms"], 2)
                s = json.dumps(line)
                print(s, flush=True)
                if out:
                    out.write(s + "\n")
                    out.flush()
        del eng
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
