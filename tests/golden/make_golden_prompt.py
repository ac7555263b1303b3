"""Golden fixture for text prompts (generate(prompt_ids=...)), from the installed transformers 5.5.0, offline:
tests/golden/prompt_tiny.json.  The "decisive" tiny model of make_golden.py, the three fixture clips, prompt_ids =
[<|startofprev|>] + deterministic text ids.
  * generate(prompt_ids=...) ids (returned without the prompt) for prompt lengths 1, 16, 63, 64, 65 (the decoder input
    then crosses a 64-position KV page) and 200, timestamps on, language detected;
  * timestamps off with an explicit language, task="translate", num_beams=5;
  * return_token_timestamps (segment token times, alignment heads of make_golden_word.py);
  * the un-chunked 75.3 s clip of make_golden_longform.py (the prompt is prepended in every seek iteration);
  * ASR-pipeline dicts (chunk_length_s=30, stride 5) with return_timestamps True / False / "word";
  * the errors generate raises for a bad prompt_condition_type.
Run in the build container (CPU):   python tests/golden/make_golden_prompt.py
"""
import io
import json
import os
import sys
import wave

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as G  # noqa: E402  (hf_model, paths, offline switches)
import make_golden_longform as LF  # noqa: E402
import helpers  # noqa: E402
from transformers import WhisperFeatureExtractor, pipeline  # noqa: E402
import transformers.pipelines.automatic_speech_recognition as asr  # noqa: E402

PREV = 50361                                     # <|startofprev|>
ALIGNMENT_HEADS = [[0, 1], [1, 0], [1, 3]]
LENGTHS = (1, 16, 63, 64, 65, 200)


def prompt(n: int):
    text = np.random.default_rng(7).integers(300, 50000, size=256).tolist()
    return [PREV] + text[:n - 1]


def rows(t):
    return t.numpy().astype(int).tolist()


def main():
    fe = WhisperFeatureExtractor(feature_size=128)
    clips = [helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"), helpers.synth_clip(2, seconds=11.3, kind="mod")]
    f = [fe(c, sampling_rate=16000, return_tensors="np", return_attention_mask=True) for c in clips]
    feats_bf = torch.from_numpy(np.stack([x["input_features"][0] for x in f])).to(torch.bfloat16).float()
    mask = torch.from_numpy(np.stack([x["attention_mask"][0] for x in f]))
    model, _ = G.hf_model("decisive")
    res = {"prompts": {str(n): prompt(n) for n in LENGTHS}, "alignment_heads": ALIGNMENT_HEADS,
           "num_frames": mask.sum(-1).tolist(), "generate": {}}
    gen = res["generate"]
    with torch.no_grad():
        for n in LENGTHS:
            out = model.generate(input_features=feats_bf, return_timestamps=True, task="transcribe", num_beams=1,
                                 do_sample=False, prompt_ids=torch.tensor(prompt(n)))
            gen[f"ts_detect_{n}"] = {"prompt": n, "timestamps": True, "language": None, "task": "transcribe",
                                     "num_beams": 1, "ids": rows(out)}
        for n in (1, 16, 65):
            out = model.generate(input_features=feats_bf, return_timestamps=False, task="transcribe", language="en",
                                 num_beams=1, do_sample=False, prompt_ids=torch.tensor(prompt(n)))
            gen[f"nots_en_{n}"] = {"prompt": n, "timestamps": False, "language": "en", "task": "transcribe",
                                   "num_beams": 1, "ids": rows(out)}
        out = model.generate(input_features=feats_bf, return_timestamps=True, task="translate", language="de",
                             num_beams=1, do_sample=False, prompt_ids=torch.tensor(prompt(16)))
        gen["translate_de_16"] = {"prompt": 16, "timestamps": True, "language": "de", "task": "translate",
                                  "num_beams": 1, "ids": rows(out)}
        for n in (16, 64):
            out = model.generate(input_features=feats_bf, return_timestamps=True, task="transcribe", num_beams=5,
                                 do_sample=False, prompt_ids=torch.tensor(prompt(n)))
            gen[f"beams5_{n}"] = {"prompt": n, "timestamps": True, "language": None, "task": "transcribe",
                                  "num_beams": 5, "ids": rows(out)}
        model.generation_config.alignment_heads = ALIGNMENT_HEADS
        out = model.generate(input_features=feats_bf, attention_mask=mask, return_timestamps=True, task="transcribe",
                             num_beams=1, do_sample=False, return_token_timestamps=True, return_segments=True,
                             prompt_ids=torch.tensor(prompt(16)))
        res["token_timestamps_16"] = {
            "prompt": 16, "sequences": rows(out["sequences"]),
            "segment_tokens": [torch.cat([s["tokens"] for s in segs]).numpy().astype(int).tolist() for segs in out["segments"]],
            "segment_token_timestamps": [torch.cat([s["token_timestamps"] for s in segs]).double().numpy().tolist()
                                         for segs in out["segments"]]}
        for cond in ("no-such-type", "all-segments"):
            try:
                model.generate(input_features=feats_bf[:1], prompt_ids=torch.tensor(prompt(4)), prompt_condition_type=cond)
                res[f"condition_{cond}"] = {"raises": None}
            except Exception as e:  # noqa: BLE001
                res[f"condition_{cond}"] = {"raises": type(e).__name__, "message": str(e)}

    tok = helpers.build_tokenizer()
    # un-chunked long-form: generate over all frames of the 75.3 s clip, and the pipeline dict
    x = LF.clip()
    lf = fe(x, sampling_rate=16000, truncation=False, padding="longest", return_tensors="pt", return_attention_mask=True)
    model.generation_config.alignment_heads = None
    with torch.no_grad():
        toks = model.generate(input_features=lf["input_features"], attention_mask=lf["attention_mask"],
                              return_timestamps=True, task="transcribe", num_beams=1, prompt_ids=torch.tensor(prompt(16)))
    pipe = pipeline("automatic-speech-recognition", model=model, tokenizer=tok, feature_extractor=fe, device="cpu",
                    dtype=torch.float32)
    pipe.generation_config.num_beams = 1
    r = pipe(x.copy(), return_timestamps=True, generate_kwargs={"task": "transcribe", "prompt_ids": torch.tensor(prompt(16))})
    res["longform_16"] = {"prompt": 16, "tokens": toks[0].tolist(), "text": r["text"],
                          "chunks": [{"text": c["text"], "timestamp": list(c["timestamp"])} for c in r["chunks"]]}

    # chunked pipeline over the 71.3 s file of the other fixtures
    asr.ffmpeg_read = lambda b, sr: (np.frombuffer(wave.open(io.BytesIO(b)).readframes(10 ** 9), np.int16)
                                     .astype(np.float32) / 32768.0)
    wav_path = "/tmp/golden_prompt_71s.wav"
    helpers.write_wav16(wav_path, np.concatenate(clips))
    pipe.generation_config.alignment_heads = ALIGNMENT_HEADS
    for name, ts in (("ts", True), ("nots", None), ("word", "word")):
        kw = {"return_timestamps": ts} if ts else {}
        r = pipe(wav_path, chunk_length_s=30, stride_length_s=5, batch_size=24,
                 generate_kwargs={"task": "transcribe", "prompt_ids": torch.tensor(prompt(16))}, **kw)
        g = {"text": r["text"], "keys": sorted(r.keys())}
        if ts:
            g["chunks"] = [{"text": c["text"], "timestamp": list(c["timestamp"])} for c in r["chunks"]]
        res[f"pipeline_30_5_24_{name}"] = g
    with open(os.path.join(HERE, "prompt_tiny.json"), "w") as fj:
        json.dump(res, fj, ensure_ascii=False)
    print("written", sorted(res))


if __name__ == "__main__":
    main()
