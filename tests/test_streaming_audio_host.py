"""Audio bookkeeping of streaming.StreamSession with wave_fps (host logic, no GPU): the lag, the released ranges, the
ring sizes, and a numpy restatement of the incremental front end against the oracle's waveform_to_examples."""
import math

import numpy as np
import pytest

from feature_vs_text_compound_emotion_b200 import streaming as S
from oracle import lfan_oracle as O

FPS = [24, 25, 29.97, 30, 50, 60]


@pytest.mark.parametrize("fps", FPS)
def test_lag_is_sufficient(fps):
    """With audio in step (floor(t * sr / fps) samples after t frames), frame t - L's example is complete."""
    L = S.stream_lag(fps)
    rows, step = S.example_grid(fps)
    t = np.arange(L, 200_000)
    starts = np.rint(step * (t - L).astype(np.float64)).astype(np.int64)     # Python round is half-to-even too
    assert all(int(s) == S.example_start(int(u), fps) for s, u in zip(starts[::9973], (t - L)[::9973]))
    need = 160 * (starts + rows - 1) + 400
    have = np.floor(t * 16000 / fps).astype(np.int64)
    assert (need <= have).all()
    # the closed form is tight to within one frame
    assert L - 1 <= 15681 * fps / 16000 <= L
    assert S.stream_lag(30) == 30 and S.stream_lag(25) == 25


@pytest.mark.parametrize("fps", FPS)
def test_frames_ready_is_the_exact_count(fps):
    for a in list(range(15500, 17500, 7)) + [10 ** 6 + k for k in range(0, 2000, 13)]:
        r = S.frames_ready(a, fps)
        assert (r == 0 or S.example_samples(r - 1, fps) <= a) and S.example_samples(r, fps) > a


def _schedule(kind, T, c, fps):
    """Per push: (frames, samples delivered after it) for a T-frame video pushed c frames at a time."""
    total = S.synced_samples(T, fps) - (S.synced_samples(20, fps) if kind == "short" else 0)
    pieces = [1, 533, 534, 7919]
    out, a, t, k = [], 0, 0, 0
    while t < T:
        cc = min(c, T - t)
        t += cc
        if kind == "synced":
            want = S.synced_samples(t, fps)
        elif kind == "behind":
            want = S.synced_samples(max(0, t - 2 * c), fps)
        elif kind == "ahead":
            want = S.synced_samples(t, fps) + 8000
        elif kind == "short":
            want = S.synced_samples(t, fps)
        else:                                                        # odd pieces until the audio is in step
            want = a
            while want < S.synced_samples(t, fps):
                want += pieces[k % 4]
                k += 1
        a = max(a, min(want, total if kind != "ahead" else total + 8000))
        out.append((cc, a))
    return out, total if kind != "ahead" else total + 8000


class _Sim:
    """The session's procedure on the host: rows computed when their samples are complete (written to a ring of
    logmel_ring_rows rows), held frames in a ring of hold_rows rows, examples gathered from the ring on release."""

    def __init__(self, fps, max_chunk):
        self.fps, self.mc = fps, max_chunk
        self.L = S.stream_lag(fps)
        self.R = S.logmel_ring_rows(self.L, max_chunk, fps)
        self.H = S.hold_rows(self.L, max_chunk)
        self.rows = S.example_grid(fps)[0]
        self.wave = np.zeros(0)
        self.ring = np.full((self.R, 64), np.nan)
        self.hold = np.full(self.H, -1)
        self.T = self.E = 0
        self.examples, self.released = {}, []

    def _append(self, new):
        r0, r1 = S.logmel_rows(self.wave.shape[0]), S.logmel_rows(self.wave.shape[0] + new.shape[0])
        self.wave = np.concatenate([self.wave, new])
        for f in range(r0, r1):                                       # each row from its own 400 samples only
            self.ring[f % self.R] = O.log_mel_spectrogram(self.wave[160 * f:160 * f + 400])[0]

    def _release(self, e1, n_ex=0):
        for t in range(self.E, e1):
            assert self.hold[t % self.H] == t                         # the held frame was not overwritten
            s = S.example_start(min(t, n_ex - 1) if n_ex else t, self.fps)
            self.examples[t] = self.ring[np.arange(s, s + self.rows) % self.R].copy()
        self.released.append((self.E, e1))
        self.E = e1

    def push(self, c, new):
        T1, A1 = self.T + c, self.wave.shape[0] + new.shape[0]
        assert A1 <= S.synced_samples(T1 + self.L + self.mc, self.fps)
        e1 = S.released_upto(T1, A1, self.E, self.L, self.fps)
        assert T1 - e1 <= self.L + 2 * self.mc
        self._append(new)
        for t in range(self.T, T1):
            self.hold[t % self.H] = t
        self.T = T1
        self._release(e1)
        return e1

    def close(self):
        self._append(np.full(16000, self.wave[-1]))
        n_ex = S.n_examples_total(S.logmel_rows(self.wave.shape[0]), self.fps)
        for a, cc in S.flush_schedule(self.E, self.T, self.mc):
            self._release(a + cc, n_ex)
        return np.stack([self.examples[t] for t in range(self.T)])


@pytest.mark.parametrize("fps", [30, 25])
@pytest.mark.parametrize("kind", ["synced", "behind", "ahead", "odd", "short"])
@pytest.mark.parametrize("T,c", [(1, 1), (29, 8), (31, 30), (347, 30), (300, 7)])
def test_incremental_examples_equal_the_oracle(fps, kind, T, c):
    rng = np.random.default_rng(T * 7 + c)
    sched, total = _schedule(kind, T, c, fps)
    wave = rng.standard_normal(max(total, 1)).astype(np.float32).astype(np.float64) * 0.3
    sim, a = _Sim(fps, 30), 0
    for cc, want in sched:
        sim.push(cc, wave[a:want])
        a = want
    if a == 0:
        return                                                       # no audio at all: close refuses (GPU test)
    got = sim.close()
    padded = np.concatenate([wave[:a], np.full(16000, wave[a - 1])])
    ex = O.waveform_to_examples(padded, 0.96, 1.0 / fps)
    want = np.concatenate([ex, np.repeat(ex[-1:], max(0, T - ex.shape[0]), 0)])[:T]
    assert got.shape == want.shape
    # a row alone and the batched oracle differ by the BLAS summation order only (the kernel is bit-exact either way)
    assert np.allclose(got, want, rtol=1e-12, atol=1e-12), np.abs(got - want).max()
    # the ranges are monotone and cover [0, T) in order
    flat = [f for a0, a1 in sim.released for f in range(a0, a1)]
    assert flat == list(range(T))


@pytest.mark.parametrize("fps", FPS)
@pytest.mark.parametrize("c", [1, 8, 30])
def test_synced_audio_releases_c_frames_per_push_after_warm_up(fps, c):
    L = S.stream_lag(fps)
    T = E = 0
    counts = []
    for _ in range(400 // c + 3):
        T += c
        e1 = S.released_upto(T, S.synced_samples(T, fps), E, L, fps)
        assert e1 >= E
        counts.append(e1 - E)
        E = e1
        assert E == max(0, T - L)
    warm = [k for k in counts if k != c]
    assert all(k == 0 for k in warm[:-1]) and len([k for k in warm if k]) <= 1   # one partial group at most
    sched = S.flush_schedule(E, T, 30)
    assert sched[0][0] == E and sum(k for _, k in sched) == T - E and all(0 < k <= 30 for _, k in sched)


def test_example_count_and_ring_sizes():
    for fps in FPS:
        rows, step = S.example_grid(fps)
        assert rows == 96
        for lm in (95, 96, 97, 500, 12345):
            n = S.n_examples_total(lm, fps)
            want = 1 + int(np.floor((lm - rows) / step)) if lm >= rows else 0
            assert n == want
            if n:
                assert S.example_start(n - 1, fps) + rows <= lm
    assert S.hold_rows(30, 30) == 120
    assert S.logmel_rows(399) == 0 and S.logmel_rows(400) == 1 and S.logmel_rows(559) == 1 and S.logmel_rows(560) == 2
    assert math.ceil(S.logmel_ring_rows(30, 30, 30)) >= (2 * 30 + 4 * 30) * 100 / 30 + 100
