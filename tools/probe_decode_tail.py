"""Decode-step time of one context alone (graph replays, B = 24, large-v3-turbo and large-v3 dims)."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import bench, helpers
from turbo_whisper_workspace_b200.config import WhisperDims
from turbo_whisper_workspace_b200.engine import WhisperEngine
dev = torch.device("cuda:0")
cases = [("turbo", WhisperDims.large_v3_turbo(), 24), ("large-v3", WhisperDims.large_v3(), 16)]
if os.environ.get("PROBE_B48"):
    cases = [("turbo", WhisperDims.large_v3_turbo(), 24), ("turbo", WhisperDims.large_v3_turbo(), 48)]
for name, dims, B in cases:
    eng = WhisperEngine(dims, bench.synth_state_dict_on_device(dims, dev, 0), device=dev, max_batch=B)
    eng.load_pcm([helpers.synth_clip(i) for i in range(B)])
    eng.features(B)
    eng.encode(B)
    us, nbytes = bench.decode_step_probe(eng, B)
    print(json.dumps({"model": name, "B": B, "us_per_step": round(us, 1),
                      "floor_us": round(nbytes / 6458.7e3, 1), "launches": eng.launches_per_step}), flush=True)
    del eng
    torch.cuda.empty_cache()
