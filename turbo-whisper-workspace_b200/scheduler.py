"""Chunk scheduler: shards the 30 s windows of a job across the GPUs of one box.

The reference has no multi-GPU code at all (SURVEY.md §2 rows 19-20: single process, ``cuda:0``); HF only
batches the windows of one file on one device.  Windows are independent units (no conditioning across
windows in the chunked pipeline), so the path is embarrassingly parallel: weights are replicated, the
workers pull micro-batches of consecutive windows, and only token ids travel back — there is no collective on
the data path (SURVEY.md §8e).

Two deployment shapes share the same partitioning:
  * :class:`WindowScheduler` — one process, one engine (+ one host thread) per local device;
  * :class:`DistributedWindowScheduler` — one process per GPU (torchrun); each rank runs its range on its
    own engine and the ordered token lists are gathered on the host with ``all_gather_object``.
"""
from __future__ import annotations

import threading
import time
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np


def partition(n_items: int, n_workers: int) -> List[Tuple[int, int]]:
    """Contiguous, balanced ranges [(start, end)] — worker i gets items start..end-1.  Contiguity keeps
    each worker's micro-batches full and the gathered order trivial."""
    if n_workers < 1:
        raise ValueError("n_workers must be >= 1")
    base, rem = divmod(n_items, n_workers)
    out, s = [], 0
    for i in range(n_workers):
        e = s + base + (1 if i < rem else 0)
        out.append((s, e))
        s = e
    return out


def microbatch_size(max_batch: int, num_beams: int = 1, group: Optional[int] = None) -> int:
    """Windows per engine call: every window occupies num_beams decode rows; ``group`` (word timestamps) caps it at
    the HF pipeline's batch_size so that a micro-batch is exactly one of HF's generate batches."""
    mb = max(1, max_batch // max(1, num_beams))
    return mb if not group else max(1, min(mb, int(group)))


def group_ranges(n_items: int, n_workers: int, mb: int) -> List[Tuple[int, int]]:
    """:func:`partition` over whole micro-batches of ``mb`` consecutive items (micro-batch k = items k*mb ..), so the
    micro-batch boundaries do not depend on the number of workers."""
    n_groups = (n_items + mb - 1) // mb
    return [(min(n_items, a * mb), min(n_items, b * mb)) for a, b in partition(n_groups, n_workers)]


def run_in_microbatches(engine, clips: Sequence[np.ndarray], group: Optional[int] = None, **generate_kwargs) -> List[Any]:
    """``engine.generate_from_pcm(clips[i:i + mb], **generate_kwargs)`` over micro-batches of :func:`microbatch_size`."""
    rows: List[Any] = []
    mb = microbatch_size(engine.max_batch, generate_kwargs.get("num_beams", 1), group)
    for i in range(0, len(clips), mb):
        rows.extend(engine.generate_from_pcm(clips[i:i + mb], **generate_kwargs))
    return rows


# Floor of the micro-batch size.  Measured on one B200 (profiles/r2c_microbatch.jsonl: a rank's share of a 1 h file on 8
# GPUs = 23 windows): 4 x 6 windows 0.563 s, 3 x 8 0.529 s, 2 x 12 0.520 s, 1 x 23 0.538 s — the decode loop costs ~890
# latency-bound steps per micro-batch whatever its size, so fewer, larger micro-batches win until contexts go idle.
MIN_MICROBATCH = 12


def balanced_microbatch(n_items: int, workers: int, max_mb: int, min_mb: int = MIN_MICROBATCH) -> int:
    """Micro-batch size for a job of ``n_items`` windows over ``workers`` engine contexts.  A micro-batch costs about
    the same whatever its size (the decode loop is latency-bound: ~2 x 445 steps per micro-batch), so the job should
    use as FEW micro-batches as possible while keeping every context busy in every round:
    rounds = ceil(n / (workers * max_mb)), size = ceil(n / (workers * rounds)) clamped to [min_mb, max_mb].
    One 1 h file (180 windows): 1 GPU x 4 contexts -> 8 micro-batches of 23; 8 GPUs x 4 contexts -> 15 of 12."""
    workers, max_mb = max(1, workers), max(1, max_mb)
    min_mb = max(1, min(min_mb, max_mb))
    if n_items <= 0:
        return max_mb
    rounds = -(-n_items // (workers * max_mb))
    return max(min_mb, min(max_mb, -(-n_items // (workers * rounds))))


class WorkQueue:
    """One shared queue over the windows of a job: ``take`` hands out the next micro-batch of ``size`` consecutive
    windows to whichever engine context asks first (no static per-device ranges)."""

    def __init__(self, n_items: int, size: int):
        self.n, self.pos, self.size = n_items, 0, max(1, size)
        self.lock = threading.Lock()
        self.handed: List[Tuple[int, int]] = []

    def take(self) -> Optional[Tuple[int, int]]:
        with self.lock:
            if self.pos >= self.n:
                return None
            a, b = self.pos, min(self.n, self.pos + self.size)
            self.pos = b
            self.handed.append((a, b))
            return a, b


def long_order(lengths: Sequence[int]) -> List[int]:
    """Indices of long-form clips, longest first (ties in input order): the order in which clips are admitted, so
    the longest seek loops start first and the short ones fill the rows that free up near the end."""
    return sorted(range(len(lengths)), key=lambda i: (-int(lengths[i]), i))


def long_partition(lengths: Sequence[int], n_workers: int) -> List[List[int]]:
    """Deterministic length-balanced plan of long-form clips over workers: longest first, each clip to the worker with
    the least assigned audio so far (ties: the lowest worker).  Every rank computes the same plan from the lengths."""
    if n_workers < 1:
        raise ValueError("n_workers must be >= 1")
    load, plan = [0] * n_workers, [[] for _ in range(n_workers)]
    for i in long_order(lengths):
        w = min(range(n_workers), key=lambda k: (load[k], k))
        plan[w].append(i)
        load[w] += int(lengths[i])
    return plan


class LongQueue:
    """Pending long-form clips of one call shared by engine contexts: ``take`` hands out ``(index, audio)`` (or None
    once the queue is empty or the call has failed), each clip exactly once."""

    def __init__(self, audios: Sequence[np.ndarray], order: Sequence[int]):
        self.audios, self.order, self.pos = audios, list(order), 0
        self.lock = threading.Lock()
        self.failed = False

    def take(self) -> Optional[Tuple[int, np.ndarray]]:
        with self.lock:
            if self.failed or self.pos >= len(self.order):
                return None
            i = self.order[self.pos]
            self.pos += 1
            return i, self.audios[i]


class WindowScheduler:
    """One process; ``contexts_per_device`` engine contexts per local GPU, each driven by its own host thread and
    CUDA stream and sharing one copy of the weights.  All contexts of all devices pull micro-batches of consecutive
    windows (:func:`balanced_microbatch`) from ONE :class:`WorkQueue` (no static per-device ranges: a device that
    finishes early takes the next micro-batch), so that a context's latency-bound decode overlaps another context's tensor-bound encoder (and
    another decode) on the same GPU, and one file strong-scales over the devices."""

    def __init__(self, state_dict, dims, generation, devices: Sequence[Any] = ("cuda:0",), max_batch: int = 24,
                 engine_factory: Optional[Callable[..., Any]] = None, contexts_per_device: int = 1):
        self.devices = list(devices)
        self.contexts_per_device = max(1, int(contexts_per_device))
        self.engines: List[List[Any]] = []      # [device][context]
        for d in self.devices:
            ctxs = []
            for c in range(self.contexts_per_device):
                if engine_factory is not None:
                    ctxs.append(engine_factory(d))
                else:
                    from .engine import WhisperEngine
                    shared = ctxs[0].w if ctxs else None
                    ctxs.append(WhisperEngine(dims, state_dict if shared is None else None, device=d, gen=generation,
                                              max_batch=max_batch, shared_weights=shared,
                                              own_stream=self.contexts_per_device > 1))
            self.engines.append(ctxs)
        self.last_stats: Dict[str, Any] = {}
        self.last_long_stats: Dict[str, Any] = {}      # the last run_long_many call

    @property
    def flat_engines(self) -> List[Any]:
        return [e for ctxs in self.engines for e in ctxs]

    @property
    def max_batch(self) -> int:
        return self.engines[0][0].max_batch

    def run(self, clips: Sequence[np.ndarray], group: Optional[int] = None, **generate_kwargs) -> List[Any]:
        """Token rows per window, in order.  ``generate_kwargs``: the generate options of every window, forwarded to
        ``engine.generate_from_pcm`` untouched; ``num_beams`` (default 1) sizes the micro-batches.  ``group`` = the HF
        pipeline's batch_size (word timestamps, where every row is ``(ids, times)``): micro-batches then are HF's
        generate batches (the per-token times of a row depend on the longest row of its batch,
        $TF/models/whisper/generation_whisper.py:241-381)."""
        t0 = time.perf_counter()
        n = len(clips)
        engines = self.flat_engines
        if not engines or n == 0:
            self.last_stats = {"workers": len(self.devices), "contexts_per_device": self.contexts_per_device,
                               "microbatches": [], "seconds": time.perf_counter() - t0}
            return []
        cap = min(e.max_batch for e in engines)
        # word timestamps: exactly the HF pipeline's batches; otherwise as few, equally sized micro-batches as keep
        # every context busy
        num_beams = generate_kwargs.get("num_beams", 1)
        mb = microbatch_size(cap, num_beams, group) if group else \
            balanced_microbatch(n, len(engines), microbatch_size(cap, num_beams), min(MIN_MICROBATCH, max(1, cap // max(1, num_beams))))
        queue = WorkQueue(n, mb)
        results: List[Optional[List[int]]] = [None] * n
        errors: List[BaseException] = []

        def work(engine):
            try:
                while not errors:
                    item = queue.take()
                    if item is None:
                        return
                    a, b = item
                    results[a:b] = engine.generate_from_pcm(clips[a:b], **generate_kwargs)
            except BaseException as ex:  # surfaced on the calling thread
                errors.append(ex)

        # never more host threads than micro-batches the job can produce
        n_threads = min(len(engines), -(-n // mb))
        # contexts of different devices first, so a small job spreads over the GPUs before it stacks contexts
        order = [self.engines[d][c] for c in range(self.contexts_per_device) for d in range(len(self.devices))]
        threads = [threading.Thread(target=work, args=(eng,), daemon=True) for eng in order[:n_threads]]
        if len(threads) == 1:
            threads[0].run()
        else:
            for t in threads:
                t.start()
            for t in threads:
                t.join()
        if errors:
            raise errors[0]
        self.last_stats = {"workers": len(self.devices), "contexts_per_device": self.contexts_per_device,
                           "microbatches": list(queue.handed), "seconds": time.perf_counter() - t0}
        return [r for r in results]

    def run_long(self, audio: np.ndarray, **generate_kwargs) -> List[int]:
        """Token row of ONE un-chunked long-form clip (> 30 s): HF's long-form generate is a sequential seek loop over the
        clip's frames, so it runs on one engine context (``engine.generate_long_from_pcm(audio, **generate_kwargs)``)."""
        return self.engines[0][0].generate_long_from_pcm(audio, **generate_kwargs)

    def run_long_many(self, audios: Sequence[np.ndarray], **generate_kwargs) -> List[List[int]]:
        """Token rows of many un-chunked long-form clips, in input order.  The clips are dealt longest first over the
        engine contexts (contexts of different devices first, as :meth:`run`), one each; the rest wait in ONE shared
        queue, from which every context refills a decode row as soon as one of its clips finishes
        (``engine.generate_long_batch(source=..., rows=...)``).  A context holds about ceil(n / contexts) active rows,
        capped at max_batch // num_beams.  ``generate_kwargs`` are forwarded untouched."""
        t0 = time.perf_counter()
        n = len(audios)
        order = [self.engines[d][c] for c in range(self.contexts_per_device) for d in range(len(self.devices))]
        n_ctx = min(len(order), n)
        results: List[Optional[List[int]]] = [None] * n
        if n_ctx == 0:
            self.last_long_stats = {"clips": 0, "contexts": 0, "rows": 0, "seconds": time.perf_counter() - t0}
            return []
        cap = microbatch_size(min(e.max_batch for e in order), generate_kwargs.get("num_beams", 1))
        rows = min(cap, -(-n // n_ctx))
        clips = long_order([np.asarray(a).size for a in audios])
        queue = LongQueue(audios, clips[n_ctx:])
        errors: List[BaseException] = []

        def work(engine, first):
            seed = iter([(first, audios[first])])

            def source():
                return next(seed, None) or queue.take()
            try:
                for i, ids in engine.generate_long_batch(source=source, rows=rows, **generate_kwargs).items():
                    results[i] = ids
            except BaseException as ex:  # surfaced on the calling thread
                queue.failed = True
                errors.append(ex)

        threads = [threading.Thread(target=work, args=(order[k], clips[k]), daemon=True) for k in range(n_ctx)]
        if len(threads) == 1:
            threads[0].run()
        else:
            for t in threads:
                t.start()
            for t in threads:
                t.join()
        if errors:
            raise errors[0]
        self.last_long_stats = {"clips": n, "contexts": n_ctx, "rows": rows, "seconds": time.perf_counter() - t0}
        return results

    def close(self):
        self.engines = []


class DistributedWindowScheduler:
    """One rank per GPU.  ``run`` must be called by every rank with the same ``clips`` (or the same count):
    rank r processes ``partition(n, world)[r]`` on its local engine — or on its local :class:`WindowScheduler`
    (several engine contexts on the rank's GPU pulling from a queue over the rank's range) — and the token
    lists are gathered in rank order on the host (``all_gather_object``; no data-path collective)."""

    def __init__(self, engine, rank: int, world_size: int, group=None):
        self.engine, self.rank, self.world_size, self.group = engine, rank, world_size, group
        self.last_stats: Dict[str, Any] = {}

    @property
    def devices(self):
        return getattr(self.engine, "devices", [getattr(self.engine, "device", None)])

    @property
    def flat_engines(self) -> List[Any]:
        return getattr(self.engine, "flat_engines", [self.engine])

    def local_range(self, n: int, mb: Optional[int] = None) -> Tuple[int, int]:
        return (group_ranges(n, self.world_size, mb) if mb else partition(n, self.world_size))[self.rank]

    def _group_mb(self, group: Optional[int], generate_kwargs: Dict[str, Any]) -> Optional[int]:
        """Micro-batch size of word-timestamp jobs (:func:`group_ranges`); None otherwise."""
        return microbatch_size(self.engine.max_batch, generate_kwargs.get("num_beams", 1), group) if group else None

    def run_local(self, clips: Sequence[np.ndarray], group: Optional[int] = None, **generate_kwargs) -> List[Any]:
        """Token rows of this rank's range of ``clips``; ``generate_kwargs`` are forwarded untouched."""
        s, e = self.local_range(len(clips), self._group_mb(group, generate_kwargs))
        if e <= s:
            return []
        if hasattr(self.engine, "run"):          # a local WindowScheduler (engine contexts of this rank's GPU)
            return self.engine.run(clips[s:e], group=group, **generate_kwargs)
        return run_in_microbatches(self.engine, clips[s:e], group, **generate_kwargs)

    def gather(self, local_rows: List[List[int]]) -> List[List[int]]:
        if self.world_size == 1:
            return local_rows
        import torch.distributed as dist
        buckets: List[Any] = [None] * self.world_size
        dist.all_gather_object(buckets, local_rows, group=self.group)
        rows: List[List[int]] = []
        for b in buckets:
            rows.extend(b)
        return rows

    def run(self, clips: Sequence[np.ndarray], group: Optional[int] = None, **generate_kwargs) -> List[Any]:
        t0 = time.perf_counter()
        s, e = self.local_range(len(clips), self._group_mb(group, generate_kwargs))
        rows = self.gather(self.run_local(clips, group, **generate_kwargs))
        self.last_stats = {"workers": self.world_size, "rank": self.rank, "local_range": (s, e),
                           "seconds": time.perf_counter() - t0}
        return rows

    def run_long(self, audio: np.ndarray, **generate_kwargs) -> List[int]:
        """Un-chunked long-form input does not shard (one sequential seek loop): every rank computes the same row."""
        if hasattr(self.engine, "run_long"):
            return self.engine.run_long(audio, **generate_kwargs)
        return self.engine.generate_long_from_pcm(audio, **generate_kwargs)

    def run_long_many(self, audios: Sequence[np.ndarray], **generate_kwargs) -> List[List[int]]:
        """Token rows of many un-chunked long-form clips, in input order.  Every rank computes the same
        :func:`long_partition` of the clips by length, runs its share on its local :class:`WindowScheduler` (or
        engine), and the rows are gathered with ``all_gather_object``.  Must be called by every rank with the same
        clips; ``generate_kwargs`` are forwarded untouched."""
        mine = long_partition([np.asarray(a).size for a in audios], self.world_size)[self.rank]
        local: List[List[int]] = []
        if mine:
            clips = [audios[i] for i in mine]
            if hasattr(self.engine, "run_long_many"):
                local = self.engine.run_long_many(clips, **generate_kwargs)
            else:
                local = self.engine.generate_long_batch(clips, **generate_kwargs)
        pairs = list(zip(mine, local))
        if self.world_size > 1:
            import torch.distributed as dist
            buckets: List[Any] = [None] * self.world_size
            dist.all_gather_object(buckets, pairs, group=self.group)
            pairs = [p for b in buckets for p in b]
        rows: List[Optional[List[int]]] = [None] * len(audios)
        for i, ids in pairs:
            rows[i] = ids
        return rows

    def close(self):
        if hasattr(self.engine, "close"):
            self.engine.close()
