"""Golden fixture for BATCHED un-chunked long-form input (transformers 5.5.0): tests/golden/longform_batch_tiny.json.
Four clips of different lengths (one frame more than 30 s, 45 s, 61.2 s and the 75.3 s clip of longform_tiny.json) go
through ONE `model.generate` call in HF's batched long-form mode: features of every clip on its own (truncation=False,
as the ASR pipeline computes them per input), zero-padded to the longest with an attention mask whose sum is each row's
`seek_num_frames` ($TF/models/whisper/generation_whisper.py:654-658, :785-870).  Greedy on both fixture models and
num_beams=2 on "varied".  Greedy and beam search share no state across rows, so each row equals the clip's solo run.
Run in the build container (CPU):   python tests/golden/make_golden_longform_batch.py
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as G  # noqa: E402
import helpers  # noqa: E402
from transformers import WhisperFeatureExtractor  # noqa: E402


def clips():
    """The four clips (fp32 16 kHz), in input order."""
    fixture = np.concatenate([helpers.synth_clip(0), helpers.synth_clip(1, kind="mod"),
                              helpers.synth_clip(2, seconds=15.3, kind="mod")])
    one_frame_over = np.concatenate([helpers.synth_clip(3, kind="mod"), helpers.synth_clip(4, seconds=0.1)])[:480161]
    return [one_frame_over,
            np.concatenate([helpers.synth_clip(5, kind="mod"), helpers.synth_clip(6, seconds=15.0)]),
            fixture,
            np.concatenate([helpers.synth_clip(7), helpers.synth_clip(8, seconds=31.2, kind="mod")])]


CASES = (("decisive", 1), ("varied", 1), ("varied", 2))


def main():
    fe = WhisperFeatureExtractor(feature_size=128)
    xs = clips()
    per = [fe(x, sampling_rate=16000, truncation=False, padding="longest", return_tensors="pt",
              return_attention_mask=True) for x in xs]
    T = max(int(p["input_features"].shape[-1]) for p in per)
    feats = torch.zeros(len(xs), 128, T)
    mask = torch.zeros(len(xs), T, dtype=torch.long)
    for i, p in enumerate(per):
        n = int(p["input_features"].shape[-1])
        feats[i, :, :n] = p["input_features"][0]
        mask[i, :n] = p["attention_mask"][0]
    res = {"samples": [int(x.shape[0]) for x in xs], "frames": mask.sum(-1).tolist()}
    for variant, beams in CASES:
        model, _ = G.hf_model(variant)
        out = model.generate(input_features=feats, attention_mask=mask, return_timestamps=True, task="transcribe",
                             num_beams=beams)
        pad = model.generation_config.pad_token_id
        rows = []
        for r in out.tolist():
            while r and r[-1] == pad:
                r.pop()
            rows.append(r)
        res[f"{variant}_beams{beams}"] = {"tokens": rows}
    with open(os.path.join(HERE, "longform_batch_tiny.json"), "w") as f:
        json.dump(res, f)
    print({k: ([len(r) for r in v["tokens"]] if isinstance(v, dict) else v) for k, v in res.items()})


if __name__ == "__main__":
    main()
