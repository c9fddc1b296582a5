"""Serving layer (SURVEY section 8(f)3): wire formats of the reference's example server and the continuous-batching
worker, driven by a fake scheduler (no GPU): requests join between chunks, leave when finished, slots are re-used,
every client receives exactly its own chunks in order, a failing request does not take the worker down."""
import struct
import threading
import time

import numpy as np
import pytest

from oracle import prompt_cases  # noqa: F401  (puts the package on sys.path)
from faster_qwen3_tts.serving import ContinuousBatcher, to_pcm16, to_wav_bytes, wav_header


def test_wire_formats_match_reference_layout():
    h = wav_header(24000)
    assert h[:4] == b"RIFF" and h[8:12] == b"WAVE" and h[12:16] == b"fmt " and h[36:40] == b"data" and len(h) == 44
    assert struct.unpack("<I", h[4:8])[0] == 0xFFFFFFFF and struct.unpack("<I", h[40:44])[0] == 0xFFFFFFFF
    fmt = struct.unpack("<IHHIIHH", h[16:36])
    assert fmt == (16, 1, 1, 24000, 48000, 2, 16)
    pcm = np.array([0.0, 0.5, -0.5, 1.0, -1.0, 2.0], dtype=np.float32)
    raw = to_pcm16(pcm)
    assert np.frombuffer(raw, dtype="<i2").tolist() == [0, 16384, -16384, 32767, -32768, 32767]
    w = to_wav_bytes(pcm, 24000)
    assert struct.unpack("<I", w[40:44])[0] == len(raw) and struct.unpack("<I", w[4:8])[0] == 36 + len(raw)


class _FakeReq:
    def __init__(self, tag, total):
        self.tag, self.total, self.done, self.finished = tag, total, 0, 0


class _FakeSched:
    """max_batch slots; every step emits min(n, remaining) 'frames' whose values identify (request, frame).  Admits
    nothing until `admitting` is set."""

    def __init__(self, max_batch):
        self.max_batch, self.active, self.peak, self.batch_sizes = max_batch, {}, 0, []
        self.admitting = threading.Event()

    def __len__(self):
        return len(self.active)

    def has_capacity(self):
        return self.admitting.is_set() and len(self.active) < self.max_batch

    def submit(self, tie, tam, tth, tpe, tag=None, max_new_tokens=0, **kw):
        if tie is None:
            raise ValueError("bad prompt")
        self.active[tag] = _FakeReq(tag, max_new_tokens)

    def step(self, n):
        self.batch_sizes.append(len(self.active))
        out = []
        for tag, rq in list(self.active.items()):
            k = min(n, rq.total - rq.done)
            codes = np.arange(rq.done, rq.done + k, dtype=np.int64)[:, None] + 1000 * tag
            rq.done += k
            if rq.done >= rq.total:
                rq.finished = 1
                del self.active[tag]
            out.append((rq, codes))
        time.sleep(0.001)
        return out


class _Win:
    def __init__(self, ref):
        pass

    def push(self, codes):
        return codes[:, 0].astype(np.float32), 24000


def test_continuous_batcher_join_leave_and_isolation():
    sched = _FakeSched(max_batch=3)
    b = ContinuousBatcher(sched, _Win, chunk_size=4, idle_sleep=0.0005)
    totals = [9, 4, 17, 6, 12, 1, 8]
    tickets, results = [], {}

    def client(i, n):
        t = b.submit(lambda: (0, 0, 0, 0, None), max_new_tokens=n)
        chunks = [c for c in t]
        results[i] = (t.rid, np.concatenate([c[0] for c in chunks]), [c[2]["chunk_steps"] for c in chunks], chunks[-1][2]["is_final"])

    threads = []
    for i, n in enumerate(totals):
        th = threading.Thread(target=client, args=(i, n))
        th.start()
        threads.append(th)
        if i == 2:   # the first three requests are admitted together, so all slots are busy at once whatever the timing
            deadline = time.time() + 10
            while b.pending.qsize() < 3 and time.time() < deadline:
                time.sleep(0.0005)
            sched.admitting.set()
        time.sleep(0.002 * (i % 3))   # staggered arrivals: some join while others are mid-stream
    bad = b.submit(lambda: (None, 0, 0, 0, None), max_new_tokens=5)
    with pytest.raises(ValueError):
        list(bad)
    for th in threads:
        th.join(timeout=20)
    b.close()
    assert len(results) == len(totals)
    for i, n in enumerate(totals):
        rid, audio, steps, final = results[i]
        assert audio.tolist() == [1000 * rid + k for k in range(n)], i          # own frames, in order, none missing
        assert sum(steps) == n and all(s <= 4 for s in steps) and final
    assert max(sched.batch_sizes) == 3 and b.max_concurrent == 3                 # slots were shared ...
    assert len(sched.active) == 0                                                # ... and all released
