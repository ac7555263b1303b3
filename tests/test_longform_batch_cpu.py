"""CPU tests of batched un-chunked long-form input (many clips > 30 s without chunk_length_s in one seek loop):
the oracle's solo run of every clip against transformers' batched long-form generate
(tests/golden/make_golden_longform_batch.py), the host bookkeeping of the multi-row loop, the schedulers'
run_long_many with stand-in engines (one process and two gloo ranks) and the pipeline's routing of a list call."""
import json
import os
import socket
import sys
import threading

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import helpers
from oracle import logmel_ref as L
from oracle import whisper_ref as R
from turbo_whisper_workspace_b200 import scheduler as S
from turbo_whisper_workspace_b200.config import WhisperDims
from turbo_whisper_workspace_b200.engine import LongFormRows, long_guard
from turbo_whisper_workspace_b200.pipeline import B200WhisperPipeline

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLD)


# ------------------------------------------------------------------------------------------------ golden
@pytest.mark.parametrize("case", ["decisive_beams1", "varied_beams1", "varied_beams2"])
def test_oracle_solo_rows_equal_hf_batched_rows(case):
    """Greedy and beam search share no state across rows: each row of HF's batched long-form generate equals the
    clip generated alone, which is what the engine's multi-row loop reproduces per clip."""
    import make_golden_longform_batch as G
    gold = json.load(open(os.path.join(GOLD, "longform_batch_tiny.json")))
    clips = G.clips()
    assert gold["samples"] == [int(c.shape[0]) for c in clips]
    assert gold["frames"] == [int(c.shape[0]) // 160 for c in clips]
    variant, beams = case.split("_beams")
    rd = R.WhisperDims(**helpers.TINY)
    ref = R.WhisperRef(rd, helpers.variant_state_dict(rd, variant))
    for i, c in enumerate(clips):
        feats = torch.from_numpy(L.log_mel_long(c))[None]
        assert ref.generate(feats, num_beams=int(beams))[0] == gold[case]["tokens"][i], f"clip {i}"


# ------------------------------------------------------------------------------------------------ bookkeeping
def _run_book(frames, capacity, advance):
    """Drive LongFormRows like the engine does, with ``advance(index, seek) -> frames`` in place of the decoder."""
    order = S.long_order(frames)
    pending = iter([(i, None) for i in order])
    admitted, groups = [], []

    def admit(items):
        groups.append([i for i, _ in items])
        admitted.extend(i for i, _ in items)
        return [(frames[i], f"feats{i}") for i, _ in items]
    book = LongFormRows(capacity, lambda: next(pending, None), admit, record=True)
    book.groups = groups
    batches = []
    while True:
        rows = book.refill()
        if not rows:
            break
        assert len(rows) <= capacity and all(c.feats == f"feats{c.index}" for c in rows)
        batches.append([(c.index, c.seek) for c in rows])
        for c in rows:
            adv = advance(c.index, c.seek)
            book.advance(c, [[c.index, c.seek]], adv, tokens=[1, 2, 3])
    return book, admitted, batches


def test_rows_refill_longest_first_and_keep_segments_in_order():
    frames = [9000, 3001, 12000, 5000, 0]
    book, admitted, batches = _run_book(frames, 2, lambda i, seek: 3000)
    assert admitted == [2, 0, 3, 1, 4]                      # longest first, each clip once
    assert book.groups[0] == [2, 0]                          # clips entering together are admitted together
    assert sorted(book.done) == [0, 1, 2, 3, 4]
    # clip 0 (3 windows) finishes before clip 2 (4 windows): clip 3 takes its row at the very next iteration
    assert batches[:4] == [[(2, 0), (0, 0)], [(2, 3000), (0, 3000)], [(2, 6000), (0, 6000)], [(2, 9000), (3, 0)]]
    for i, f in enumerate(frames):
        c = book.done[i]
        assert c.ids == [v for s in range(0, f, 3000) for v in (i, s)] and c.seek >= f and c.feats is None
        assert [it["seek"] for it in c.trace["iterations"]] == [[s] for s in range(0, f, 3000)]
    assert book.iterations == len(batches) and book.windows == sum(len(b) for b in batches)


def test_rows_guard_trips_on_a_degenerate_clip_only():
    frames = [6000, 4000]
    # clip 1 never advances (degenerate timestamp output); clip 0 finishes normally first
    with pytest.raises(RuntimeError, match="does not advance"):
        _run_book(frames, 2, lambda i, seek: 0 if i == 1 else 3000)
    # stuck for a while, then advancing: the guard counts the iterations of each clip, not of the call
    stuck = {1: 60}

    def advance(i, seek):
        if stuck.get(i, 0) > 0:
            stuck[i] -= 1
            return 0
        return 3000
    book, _, _ = _run_book(frames, 2, advance)
    assert book.done[1].iters == 62 <= long_guard(4000) and book.done[0].iters == 2 and book.iterations == 62


def test_rows_record_traces_only_on_request():
    pending = iter([(0, None)])
    book = LongFormRows(1, lambda: next(pending, None), lambda its: [(3000, None) for _ in its])
    (c,) = book.refill()
    book.advance(c, [[1, 2]], 3000, tokens=[1, 2, 3])
    assert book.done[0].ids == [1, 2] and book.done[0].trace["iterations"] == []


def test_rows_admission_rejects_a_clip_handed_out_twice():
    items = iter([(0, None), (0, None)])
    book = LongFormRows(2, lambda: next(items, None), lambda its: [(4000, None) for _ in its])
    with pytest.raises(RuntimeError, match="handed out twice"):
        book.refill()


# ------------------------------------------------------------------------------------------------ schedulers
class LongEngine:
    """Engine stand-in of the long-form path: takes every clip the source hands out and returns [len(audio)] per clip
    (the clips of a test have distinct lengths)."""
    lock = threading.Lock()

    def __init__(self, device, max_batch=8):
        self.device, self.max_batch, self.calls = device, max_batch, []

    def generate_long_batch(self, audios=None, *, source=None, rows=None, **kw):
        if audios is not None:
            order = S.long_order([len(a) for a in audios])
            it = iter([(i, audios[i]) for i in order])
            source = lambda: next(it, None)
        assert rows is None or 1 <= rows <= self.max_batch // kw.get("num_beams", 1)
        taken = {}
        while (item := source()) is not None:
            i, a = item
            taken[i] = [len(a)]
        with self.lock:
            self.calls.append((sorted(taken), rows, kw, sorted(v[0] for v in taken.values())))
        if audios is not None:
            return [taken[i] for i in range(len(audios))]
        return taken


def _clips(n):
    return [np.zeros(16000 * 31 + 160 * (7 * i % 5) + i, np.float32) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3, 4, 11])
def test_run_long_many_spreads_and_orders(n):
    sched = S.WindowScheduler(None, None, None, devices=["d0", "d1"], engine_factory=lambda d: LongEngine(d),
                              contexts_per_device=2)
    clips = _clips(n)
    kw = dict(task="translate", language=None, num_beams=2, prompt_ids=[50361, 400])
    rows = sched.run_long_many(clips, **kw)
    assert rows == [[len(c)] for c in clips]
    calls = [(e.device, c) for e in sched.flat_engines for c in e.calls]
    taken = sorted(i for _, c in calls for i in c[0])
    assert taken == list(range(n))                          # every clip on exactly one context
    assert all(c[2] == kw for _, c in calls)                # keywords untouched
    assert all(c[1] == min(4, -(-n // min(4, n))) for _, c in calls)
    assert len(calls) == min(4, n)
    if n == 2:                                               # a small job spreads over the devices first
        assert sorted(d for d, _ in calls) == ["d0", "d1"]
    # the first clip of each context is dealt longest first, contexts of different devices first
    first = {e.device + str(k): e.calls for k, e in enumerate(sched.flat_engines)}
    assert sum(1 for v in first.values() if v) == min(4, n)


def test_run_long_many_surfaces_an_engine_error():
    class Failing(LongEngine):
        def generate_long_batch(self, audios=None, *, source=None, rows=None, **kw):
            source()
            raise RuntimeError("boom on " + self.device)
    sched = S.WindowScheduler(None, None, None, devices=["d0"], engine_factory=lambda d: Failing(d), contexts_per_device=2)
    with pytest.raises(RuntimeError, match="boom on d0"):
        sched.run_long_many(_clips(5))


def test_long_partition_is_balanced_and_deterministic():
    lengths = [700, 100, 900, 300, 300, 500]
    plan = S.long_partition(lengths, 2)
    assert plan == [[2, 3, 4], [0, 5, 1]]
    assert S.long_partition(lengths, 2) == plan and sorted(sum(plan, [])) == list(range(6))
    assert S.long_partition(lengths, 4) == [[2], [0], [5, 1], [3, 4]]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n, local_window, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from test_longform_batch_cpu import LongEngine, _clips
    from turbo_whisper_workspace_b200 import scheduler as S
    if local_window:
        local = S.WindowScheduler(None, None, None, devices=[f"r{rank}"], engine_factory=lambda d: LongEngine(d),
                                  contexts_per_device=2)
        engines = local.flat_engines
    else:
        local = LongEngine(f"r{rank}")
        engines = [local]
    sch = S.DistributedWindowScheduler(local, rank, world)
    rows = sch.run_long_many(_clips(n), task="transcribe", language="en")
    mine = sorted(n for e in engines for c in e.calls for n in c[3])
    kws = [c[2] for e in engines for c in e.calls]
    torch.save({"rows": rows, "mine": mine, "kws": kws}, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.parametrize("n,local_window", [(5, True), (1, False)])
def test_two_rank_run_long_many(tmp_path, n, local_window):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), n, local_window, str(tmp_path)), nprocs=world, join=True)
    r = [torch.load(tmp_path / f"r{k}.pt") for k in range(world)]
    clips = _clips(n)
    want = [[len(c)] for c in clips]
    assert r[0]["rows"] == want and r[1]["rows"] == want
    plan = S.long_partition([len(c) for c in clips], world)
    assert [x["mine"] for x in r] == [sorted(len(clips[i]) for i in p) for p in plan]
    assert all(kw == dict(task="transcribe", language="en") for x in r for kw in x["kws"])


# ------------------------------------------------------------------------------------------------ pipeline
class OracleLongScheduler:
    """The oracle's token ids behind the scheduler interface, with run_long_many (every clip solo, as the engine's
    rows are independent)."""

    def __init__(self, variant):
        rd = R.WhisperDims(**helpers.TINY)
        self.ref = R.WhisperRef(rd, helpers.variant_state_dict(rd, variant))
        self.last_stats, self.calls = {}, []

    def run(self, clips, task="transcribe", language=None, num_beams=1):
        self.calls.append(("run", len(clips)))
        feats = torch.stack([torch.from_numpy(L.log_mel(c)) for c in clips])
        return self.ref.generate(feats, task=task, num_beams=num_beams)

    def run_long(self, audio, task="transcribe", language=None, num_beams=1):
        self.calls.append(("run_long", 1))
        return self.ref.generate(torch.from_numpy(L.log_mel_long(audio))[None], task=task, num_beams=num_beams)[0]

    def run_long_many(self, audios, task="transcribe", language=None, num_beams=1):
        self.calls.append(("run_long_many", len(audios)))
        return [self.ref.generate(torch.from_numpy(L.log_mel_long(a))[None], task=task, num_beams=num_beams)[0]
                for a in audios]


def test_pipeline_list_of_long_inputs_equals_per_clip_calls():
    sched = OracleLongScheduler("decisive")
    pipe = B200WhisperPipeline(None, WhisperDims(**helpers.TINY), helpers.build_tokenizer(), scheduler=sched)
    a = np.concatenate([helpers.synth_clip(0), helpers.synth_clip(1, seconds=4.0, kind="mod")])
    b = np.concatenate([helpers.synth_clip(2, kind="mod"), helpers.synth_clip(3, seconds=9.0)])
    short = helpers.synth_clip(4, seconds=12.0, kind="mod")
    together = pipe([a, short, b], return_timestamps=True)
    assert sched.calls == [("run", 1), ("run_long_many", 2)]
    assert set(pipe.last_stats) >= {"windows", "files", "audio_seconds", "host_seconds"}
    sched.calls.clear()
    alone = [pipe(x, return_timestamps=True) for x in (a, short, b)]
    assert sched.calls == [("run_long", 1), ("run", 1), ("run_long", 1)]
    assert together == alone
    assert all(r["chunks"] for r in together)
