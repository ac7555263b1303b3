"""-m gpu tests of batched un-chunked long-form input: the per-row window gather (tw_gather_frames) against torch
slicing, WhisperEngine.generate_long_batch with rows refilled (more clips than rows) against the oracle's solo run of
every clip under the margin rule of tests/test_gpu_longform.py, and a pipeline list call of several long inputs."""
import os
import sys

import numpy as np
import pytest
import torch

import helpers
import helpers_prompt as HP

pytestmark = pytest.mark.gpu
MARGIN_TOL = 0.30
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))


def test_gather_frames_matches_slicing(cuda_device):
    from turbo_whisper_workspace_b200 import ops
    g = torch.Generator(device="cpu").manual_seed(11)
    lengths = [7530, 3001, 4500, 3000, 12000]
    seeks = [0, 2999, 2200, 0, 11996]           # start, last frames, middle, exactly one window, last 4 frames
    for cols in (128, 80):
        feats = [torch.randn(n, cols, generator=g).to(torch.bfloat16).to(cuda_device) for n in lengths]
        dst = torch.full((len(lengths) + 1, 3002, cols), 7.0, dtype=torch.bfloat16, device=cuda_device)
        ops.gather_frames(feats, lengths, seeks, dst, window=3000, row_off=1)
        for b, (f, n, s) in enumerate(zip(feats, lengths, seeks)):
            k = min(3000, n - s)
            assert torch.equal(dst[b, 1:1 + k], f[s:s + k]), (cols, b)
            assert float(dst[b, 1 + k:3001].abs().max() if k < 3000 else 0.0) == 0.0, (cols, b)
            assert bool((dst[b, 0] == 7.0).all()) and bool((dst[b, 3001] == 7.0).all())
        assert bool((dst[len(lengths)] == 7.0).all())


@pytest.mark.parametrize("n_mels", [128, 80])
def test_logmel_long_many_matches_per_clip(cuda_device, n_mels):
    """Several clips in one launch (and one floor launch, each clip with its own max - 8 clamp) equal each clip's
    tw_logmel_long_n output bit for bit, and the oracle's whole-clip features within the tolerance of
    tests/test_gpu_longform.py.  The clips differ in length and loudness, one has a silent stretch (values at its
    floor)."""
    from oracle import logmel_ref as L
    import helpers_v2 as V
    from turbo_whisper_workspace_b200 import ops
    rng = np.random.default_rng(3)
    lens = [480161, 2997 * 160 + 480000 + 333, 16000 * 75 + 77, 16000 * 41]
    audios = []
    for k, n in enumerate(lens):
        t = np.arange(n) / 16000.0
        a = (0.3 * np.sin(2 * np.pi * (200 + 40 * k + 30 * t) * t) * (0.2 + np.abs(np.sin(0.7 * t)))
             + 0.01 * rng.standard_normal(n)) * (10.0 ** -k)
        a[n // 3: n // 3 + 40000] = 0.0
        audios.append(a.astype(np.float32))
    lm = ops.LogMel(cuda_device, 1, n_mels)
    feats, keep = lm.long_many(audios)
    torch.cuda.synchronize()
    for k, a in enumerate(audios):
        one = lm.long(a)
        assert feats[k].shape == one.shape == (a.shape[0] // 160, n_mels)
        assert torch.equal(feats[k], one), k
        got = feats[k].float().cpu().numpy().T
        want = L.log_mel_long(a) if n_mels == 128 else V.log_mel_long(a)
        err = np.abs(got - want)
        assert (err <= 1e-4 + np.abs(want) * 2.0 ** -8).all(), (k, float(err.max()))


@pytest.fixture(scope="module")
def clips():
    import make_golden_longform_batch as G
    return G.clips()


def _engine(variant, cuda_device, max_batch):
    from oracle import whisper_ref as R
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    rd = R.WhisperDims(**helpers.TINY)
    sd = helpers.variant_state_dict(rd, variant)
    return R.WhisperRef(rd, sd), WhisperEngine(WhisperDims(**helpers.TINY), sd, device=cuda_device, max_batch=max_batch)


def _feats(audio):
    from oracle import logmel_ref as L
    return torch.from_numpy(L.log_mel_long(audio))[None].to(torch.bfloat16).float()


@pytest.mark.parametrize("variant", ["decisive", "varied"])
def test_generate_long_batch_matches_oracle_per_clip(cuda_device, clips, variant):
    ref, eng = _engine(variant, cuda_device, max_batch=2)          # 4 clips on 2 rows: rows are refilled
    traces = {}
    got = eng.generate_long_batch(clips, trace=traces)
    assert eng.stats["long_windows"] > eng.stats["long_iterations"] > 0
    assert 1.0 < eng.stats["long_mean_rows"] <= 2.0
    identical = total = 0
    for i, audio in enumerate(clips):
        trace = {}
        want = ref.generate(_feats(audio), trace=trace)[0]
        # a clip may leave the comparison at a low-margin step; a decisive divergence fails inside
        agreed, rows, first_diffs = helpers.compare_generate_traces(trace, traces[i], MARGIN_TOL)
        total += agreed
        if rows == [0]:
            assert got[i] == want, f"clip {i}"
        identical += got[i] == want
    assert total >= 40, "free-running agreement is implausibly short"
    # the batched rows against the engine's own solo runs (not required bit-equal: the cross-attention split count
    # follows the row count, so reductions may be ordered differently)
    solo = sum(eng.generate_long_from_pcm(a) == got[i] for i, a in enumerate(clips))
    print(f"{variant}: {identical}/{len(clips)} clips identical to the oracle, {solo}/{len(clips)} to the solo engine run")


def test_generate_long_batch_beams_and_prompt(cuda_device, clips):
    """num_beams=2 with rows refilled, window by window against the fp32 oracle (the pattern of
    tests/test_gpu_engine.py::test_beam_search_against_oracle): beam search ranks near-equal hypotheses, so bf16 noise
    may send it down another trajectory than the oracle's search.  What must hold in every window of every clip: the
    returned hypothesis is grammatical for the oracle, and the search's own accumulated log-probability of it agrees
    with the oracle's teacher-forced score of the same tokens within the bf16 logit tolerance (this breaks if a row
    read another clip's window, cross K/V or cache line); and windows reproduce the oracle's best exactly.  Then
    prompt_ids under the margin rule."""
    from oracle import whisper_ref as R
    from test_gpu_engine import _oracle_sequence_score
    ref, eng = _engine("decisive", cuda_device, max_batch=4)
    gc = R.GenConfig()
    traces = {}
    got = eng.generate_long_batch(clips, trace=traces, num_beams=2)       # 2 clips x 2 beams per iteration
    exact = windows = 0
    for i, audio in enumerate(clips):
        feats = _feats(audio)
        T = feats.shape[-1]
        tr = traces[i]
        lang = tr["langs"][0]
        assert lang == ref.detect_language(ref.encode(feats[..., :3000]), gc)[0]
        assert got[i] and got[i][0] >= 50365
        for it in tr["iterations"]:
            seek = it["seek"][0]
            win = torch.zeros(1, feats.shape[1], 3000)
            win[..., :min(3000, T - seek)] = feats[..., seek:seek + 3000]
            enc = ref.encode(win)
            prompt = [gc.decoder_start_token_id, lang, gc.task_to_id["transcribe"]]
            best = ref.beam_search(enc, torch.tensor([prompt]), gc, num_beams=2)[0].tolist()
            own, n = it["beam"][0]
            hyp = list(it["tokens"][0][3:3 + n])
            oracle_score = _oracle_sequence_score(ref, gc, enc, prompt, hyp)
            assert oracle_score > -1e8, f"clip {i} seek {seek}: hypothesis violates the timestamp grammar"
            assert abs(own - oracle_score) < 0.02 * n + 0.5, (i, seek, own, oracle_score, n)
            while len(best) > n and best[-1] == gc.pad_token_id:
                best.pop()
            exact += hyp == best
            windows += 1
    assert exact >= 1, "no window reproduces the oracle's best hypothesis"
    print(f"beams: {exact}/{windows} windows identical to the oracle's search")
    # prompt_ids with rows refilled: every clip against the oracle's prompted solo loop
    ref, eng = _engine("varied", cuda_device, max_batch=4)
    ids = HP.golden()["prompts"]["16"]
    traces = {}
    got = eng.generate_long_batch(clips, trace=traces, rows=2, prompt_ids=ids)
    total = 0
    for i, audio in enumerate(clips):
        trace = {}
        want = HP.prompted_generate(ref, _feats(audio), ids, trace=trace)[0]
        agreed, rows, first_diffs = HP.compare_prompted_traces(trace, traces[i], MARGIN_TOL)
        total += agreed
        if rows == [0]:
            assert got[i] == want, f"clip {i}"
    assert total >= 40, "free-running agreement is implausibly short"


def test_pipeline_list_of_long_inputs(cuda_device, clips):
    from oracle import whisper_ref as R
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline
    sd = helpers.variant_state_dict(R.WhisperDims(**helpers.TINY), "decisive")
    pipe = B200WhisperPipeline(sd, WhisperDims(**helpers.TINY), helpers.build_tokenizer(), devices=[cuda_device],
                               max_batch=4, contexts_per_device=2)
    try:
        longs = [clips[0], clips[2], clips[3]]
        short = helpers.synth_clip(9, seconds=12.0, kind="mod")
        together = pipe([longs[0], short, longs[1], longs[2]], return_timestamps=True)
        alone = [pipe(a, return_timestamps=True) for a in longs]
        assert [together[0]["text"], together[2]["text"], together[3]["text"]] == [r["text"] for r in alone]
        assert together[1]["chunks"] and pipe.scheduler.last_long_stats["clips"] == 3
    finally:
        pipe.close()
