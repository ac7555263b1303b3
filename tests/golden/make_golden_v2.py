"""Generates the 80-mel / v2-vocabulary fixtures from the INSTALLED transformers (5.5.0), offline, like make_golden.py:
a random tiny WhisperConfig(num_mel_bins=80, vocab_size=51865) at helpers.TINY widths with the generation config and
tokenizer layout of openai/whisper-large-v2 and older multilingual checkpoints (tests/helpers_v2.py).

Run in the build container (CPU):   python tests/golden/make_golden_v2.py
Outputs (small, committed):  tests/golden/v2_tiny.npz       log-mel KATs of WhisperFeatureExtractor(feature_size=80),
                                                             encoder / teacher-forced logit samples, generate ids, langs
                             tests/golden/pipeline_v2_tiny.json   ASR-pipeline dicts, return_timestamps=True / omitted
"""
import io
import json
import os
import sys
import wave

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ["HF_HUB_OFFLINE"] = "1"

import helpers  # noqa: E402
import helpers_v2 as V  # noqa: E402
from transformers import WhisperFeatureExtractor, pipeline  # noqa: E402
import transformers.pipelines.automatic_speech_recognition as asr  # noqa: E402

from oracle import whisper_ref as R  # noqa: E402

# teacher-forced decoder input: prompt, timestamps, text, a repeated timestamp
DEC_IDS = [V.SOT, V.LANG_FIRST, V.TRANSCRIBE, V.TIMESTAMP_BEGIN, 400, 401, V.TIMESTAMP_BEGIN + 35,
           V.TIMESTAMP_BEGIN + 35, 402]


def clips():
    return [helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"), helpers.synth_clip(2, seconds=11.3, kind="mod")]


def long_pcm():
    # 71.3 s: with stride 0 the 30 s windows are exactly the three clips of the model fixtures
    return np.concatenate(clips())


def main():
    fe = WhisperFeatureExtractor(feature_size=80)
    out = {}
    # ---------------------------------------------------------------- 1. log-mel known answers (80 bins)
    A = (0.1 * np.random.default_rng(0).standard_normal(480000)).astype(np.float32)
    t = np.arange(480000) / 16000.0
    sine = (0.5 * np.sin(2 * np.pi * 440.0 * t)).astype(np.float32)
    for name, pcm in (("noise30", A), ("sine440", sine), ("short", A[:12345]), ("mod", helpers.synth_clip(1, kind="mod"))):
        x = fe(pcm, sampling_rate=16000, return_tensors="np")["input_features"][0]
        out["logmel_" + name + "_sub"] = x[::4, ::25].copy()       # [20, 120] sub-sampled grid
        out["logmel_" + name + "_stats"] = np.array([x.mean(), x.min(), x.max()], dtype=np.float64)

    # ---------------------------------------------------------------- 2. model: encoder / logits / generate
    cs = clips()
    feats = torch.from_numpy(np.stack([fe(c, sampling_rate=16000, return_tensors="np")["input_features"][0] for c in cs]))
    feats_bf = feats.to(torch.bfloat16).float()   # what a bf16 pipeline feeds the model
    for variant in ("decisive", "varied"):
        model, _ = V.hf_model(variant)
        with torch.no_grad():
            enc = model.model.encoder(feats_bf).last_hidden_state
            out[f"{variant}_enc_sub"] = enc[:, ::50, ::8].numpy().copy()
            logits = model(input_features=feats_bf, decoder_input_ids=torch.tensor([DEC_IDS] * 3)).logits
            out[f"{variant}_logits_sub"] = logits[:, :, ::97].numpy().copy()
            out[f"{variant}_logits_argmax"] = logits.argmax(-1).numpy().copy()
            gen = model.generate(input_features=feats_bf, return_timestamps=True, task="transcribe", num_beams=1,
                                 do_sample=False)
            out[f"{variant}_generate"] = gen.numpy().astype(np.int32)
            out[f"{variant}_langs"] = model.detect_language(input_features=feats_bf).numpy().astype(np.int32)
    np.savez_compressed(os.path.join(HERE, "v2_tiny.npz"), **out)

    # ---------------------------------------------------------------- 3. pipeline end to end
    tok = V.build_tokenizer()
    asr.ffmpeg_read = lambda b, sr: (np.frombuffer(wave.open(io.BytesIO(b)).readframes(10 ** 9), np.int16)
                                     .astype(np.float32) / 32768.0)
    wav_path = "/tmp/golden_v2_71s.wav"
    helpers.write_wav16(wav_path, long_pcm())
    results = {}
    # decisiveness of the stride-0 windows under PCM16 quantisation, measured with the oracle
    q = helpers.quantize_pcm16(long_pcm())
    wfeats = torch.stack([torch.from_numpy(V.log_mel(q[i * 480000:(i + 1) * 480000])) for i in range(3)])
    tr = {}
    R.WhisperRef(V.ref_dims(), V.variant_state_dict(V.ref_dims(), "decisive")).generate(
        wfeats.to(torch.bfloat16).float(), gc=V.gen_config(), trace=tr)
    results["decisive_30_0_min_margin"] = float(min(min(float(r["margin"].min()), float(r["rule_gap"].min()))
                                                    for it in tr["iterations"] for r in it["record"]))
    for variant in ("decisive", "varied"):
        model, _ = V.hf_model(variant)
        pipe = pipeline("automatic-speech-recognition", model=model, tokenizer=tok, feature_extractor=fe, device="cpu",
                        dtype=torch.float32)
        pipe.generation_config.num_beams = 1      # greedy
        for (cl, st, bs) in ((30, 5, 24), (60, 5, 32)):
            for ts in (True, None):
                kw = {"return_timestamps": True} if ts else {}
                r = pipe(wav_path, chunk_length_s=cl, stride_length_s=st, batch_size=bs,
                         generate_kwargs={"task": "transcribe"}, **kw)
                g = {"text": r["text"], "keys": sorted(r.keys())}
                if ts:
                    g["chunks"] = [{"timestamp": list(c["timestamp"]), "text": c["text"]} for c in r["chunks"]]
                results[f"{variant}_{cl}_{st}_{bs}_{'ts' if ts else 'nots'}"] = g
    with open(os.path.join(HERE, "pipeline_v2_tiny.json"), "w") as f:
        json.dump(results, f, indent=1, ensure_ascii=False)
    print("v2 golden fixtures written")


if __name__ == "__main__":
    main()
