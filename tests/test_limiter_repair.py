"""The limiter's repair machinery: wrong start-state guesses, the repair rounds and the sequential fallback.

k_limiter (csrc/ame_kernels.cuh) cuts every limiter track into tiles of 1 << lim_shift frames.  A tile that does not
start in the initial state GUESSES its start state by running the machine from the initial state over the frames in
front of it (2 G by default); k_lim_verify compares every tile's start with its predecessor's end bit for bit, two
repair rounds re-run the open tiles whose predecessor is settled, and k_lim_fallback walks what is still open, one warp
per track.  With the default window real signals never guess wrong, so that machinery only runs when the window is
shortened (ame_plan_set_limiter_guess).

The first part is a plain-Python model of the tiled scheme - the same tiles, guesses, rounds, gate and stop rule as the
kernels - checked bit for bit against oracle.limiter.alimiter_py for several guess windows.  It also predicts how many
tiles are open after rounds 0, 1 and 2, and the GPU tests (second part) require ame_plan_limiter_stats to report exactly
those counts while the output stays equal to the oracle's."""
import math
import struct

import numpy as np
import pytest

from oracle import limiter

FLAT = dict(bass_boost=0.0, mid_cut=0.0, presence_boost=0.0, treble_boost=0.0, analog_character=0, width=1.0,
            lufs=None, multiband=False)
ALT = dict(limiter_limit=0.9, limiter_attack=2.0, limiter_release=20.0)     # non-default limiter parameters


# ------------------------------------------------------------------------------------------------
# the model
# ------------------------------------------------------------------------------------------------
class LimParams:
    """The per-track constants the kernels get (design.track_params) and the tile length build_layout picks."""

    def __init__(self, fs, limit=0.98, attack_ms=5.0, release_ms=50.0):
        buffer_size = int(fs * (attack_ms / 1000.0) * 2)
        buffer_size -= buffer_size % 2
        self.B = buffer_size // 2
        self.limit, self.level, self.fsrel = limit, 1.0 / limit, fs * (release_ms / 1000.0)
        self.release_frames = int(math.ceil(fs * (release_ms / 1000.0)))
        thr = int(math.floor(limit * 32768.0))
        while thr / 32768.0 <= limit:
            thr += 1
        self.thr = thr
        self.G = self.B + self.release_frames + 8
        shift = 13
        while (1 << shift) < self.G:
            shift += 1
        self.tile = 1 << shift

    @classmethod
    def of(cls, fs, settings):
        return cls(fs, settings.get("limiter_limit", 0.98), settings.get("limiter_attack", 5.0),
                   settings.get("limiter_release", 50.0))


INIT = (1.0, 0.0, ())          # att, delta, queue ((frame, slope), ...): the state a track starts in


def _bits(x):
    return struct.unpack("<q", struct.pack("<d", x))[0]


def _same(a, b):
    """Two machine states, field by field and bit by bit (lim_equal / lim_equal_live)."""
    return (_bits(a[0]) == _bits(b[0]) and _bits(a[1]) == _bits(b[1]) and len(a[2]) == len(b[2])
            and all(f == g and _bits(d) == _bits(e) for (f, d), (g, e) in zip(a[2], b[2])))


class Track:
    def __init__(self, x, p):
        self.x, self.p = np.ascontiguousarray(x, dtype=np.int16), p
        pk = np.abs(self.x.astype(np.int32)).max(axis=1) if len(x) else np.zeros(0, np.int32)
        self.pk = pk.tolist()
        over = np.flatnonzero(pk >= p.thr)
        # next over-limit frame at or after n (len(x) if none): lets an idle machine skip quiet stretches
        nxt = np.full(len(x) + 1, len(x), dtype=np.int64)
        nxt[over] = over
        self.next_over = np.minimum.accumulate(nxt[::-1])[::-1].tolist()
        self.tiles = [(b, min(b + p.tile, len(x))) for b in range(0, len(x), p.tile)]
        # k_apply_gain's lim_last: the last over-limit frame of each tile, or -1
        self.last = []
        for b, e in self.tiles:
            k = np.searchsorted(over, e) - 1
            self.last.append(int(over[k]) if k >= 0 and over[k] >= b else -1)

    def run(self, st, lo, hi, att_out=None):
        """lim_run: the machine over frames [lo, hi) from state st; att_out[n] gets the attenuation output frame n is
        scaled by."""
        p, pk, nxt = self.p, self.pk, self.next_over
        B, thr, limit, fsrel, bufsize = p.B, p.thr, p.limit, p.fsrel, 2 * p.B
        att, delta = st[0], st[1]
        q = [[f, d, limit / (pk[f] * (1.0 / 32768.0))] for f, d in st[2]]     # lim_ratios: limit / peak from the signal
        n = lo
        while n < hi:
            if not q and delta == 0.0 and pk[n] < thr:                       # idle until the next over-limit frame
                m = min(nxt[n], hi)
                if att_out is not None:
                    att_out[n:m] = att
                n = m
                continue
            if pk[n] >= thr:
                peak = pk[n] * (1.0 / 32768.0)
                patt = min(limit / peak, 1.0)
                rdelta = (1.0 - patt) / fsrel
                ratio = limit / peak
                d = (ratio - att) / bufsize * 2
                if d < delta:
                    delta = d
                    q = [[n, rdelta, ratio]]
                else:
                    for i, e in enumerate(q):
                        pd = (ratio - e[2]) / float(n - e[0])
                        if pd < e[1]:
                            e[1] = pd
                            del q[i + 1:]
                            q.append([n, rdelta, ratio])
                            break
            att += delta
            if att_out is not None:
                att_out[n] = att
            if n >= B - 1 and q and n - (B - 1) == q[0][0]:                   # a queued peak leaves the ring
                delta = q[0][1]
                att = limit / (pk[n - (B - 1)] * (1.0 / 32768.0))
                del q[0]
            if att > 1.0:
                att, delta, q = 1.0, 0.0, []
            if att <= 0.0:
                att = 0.0000000000001
                delta = (1.0 - att) / fsrel
            if att != 1.0 and (1.0 - att) < 0.0000000000001:
                att = 1.0
            if delta != 0.0 and abs(delta) < 0.00000000000001:
                delta = 0.0
            n += 1
        return (att, delta, tuple((f, d) for f, d, _ in q))

    def output(self, att):
        """lim_emit over the whole track: output frame n is input frame n - (B - 1) scaled, clipped, levelled, rounded."""
        p = self.p
        src = np.zeros_like(self.x)
        if len(self.x) > p.B - 1:
            src[p.B - 1:] = self.x[:len(self.x) - (p.B - 1)]
        v = (src.astype(np.float64) * (1.0 / 32768.0)) * att[:, None]
        v = np.clip(v, -p.limit, p.limit) * p.level
        return np.clip(np.rint(v * 32768.0), -32768, 32767).astype(np.int16)


def model(x, p, guess=-1):
    """The tiled limiter of k_limiter / k_lim_verify / k_lim_fallback on one track.  Returns (output, [open tiles after
    round 0, 1, 2], fallback): fallback counts the tiles the sequential walk ran and where it stopped - at an exact
    start, or where its live state met a recorded start."""
    t = Track(x, p)
    nt = len(t.tiles)
    att = np.ones(len(x))
    win = 2 * p.G if guess < 0 else guess
    IN, OUT, exact = [None] * nt, [None] * nt, [0] * nt
    for k, (b, e) in enumerate(t.tiles):                                     # round 0
        first = k == 0
        prev_last = -1 if first else t.last[k - 1]
        quiet_start = first or prev_last < 0 or b - 1 - prev_last >= p.G
        if quiet_start and t.last[k] < 0:                                    # elementwise tile
            IN[k], exact[k], OUT[k] = INIT, 1, INIT
            att[b:e] = 1.0
            continue
        st, exact[k] = INIT, 1
        if not quiet_start:
            ws = max(0, b - win)
            exact[k] = int(ws == 0)
            st = t.run(INIT, ws, b)
        IN[k] = st
        OUT[k] = t.run(st, b, e, att)

    def verify():
        return [int(k > 0 and not exact[k] and not _same(IN[k], OUT[k - 1])) for k in range(nt)]

    need = verify()
    counts = [sum(need)]
    for _ in (1, 2):                                                         # repair rounds
        run = [k for k in range(1, nt) if need[k] and not need[k - 1]]      # the predecessor is settled
        for k in run:
            IN[k], exact[k] = OUT[k - 1], 0
            OUT[k] = t.run(IN[k], *t.tiles[k], att)
        need = verify()
        counts.append(sum(need))
    fb = dict(walked=0, stop_exact=0, stop_live=0)
    walking, st = False, None                                               # the fallback: in order, one track
    for k, (b, e) in enumerate(t.tiles):
        if not walking:
            if not need[k]:
                continue
            st, walking = OUT[k - 1], True
        st = t.run(st, b, e, att)
        OUT[k] = st
        fb["walked"] += 1
        if k + 1 < nt and not need[k + 1]:
            if exact[k + 1]:
                walking = False
                fb["stop_exact"] += 1
            elif _same(st, IN[k + 1]):
                walking = False
                fb["stop_live"] += 1
    return t.output(att), counts, fb


# ------------------------------------------------------------------------------------------------
# signals
# ------------------------------------------------------------------------------------------------
def _hot(x, gain):
    return np.clip(np.rint(x.astype(np.float64) * gain), -32768, 32767).astype(np.int16)


def _just_over(n, p, seed):
    """Random peaks at and just above the limiter's threshold on every frame, alternating sign."""
    rng = np.random.default_rng(seed)
    a = rng.integers(p.thr - 200, 32768, n)
    sgn = np.where(np.arange(n) % 2 == 0, 1, -1)
    return np.stack([a * sgn, a // 2 * sgn], axis=1).astype(np.int16)


def _clicks(fs, p, window, n_tiles=12, extra=0):
    """A quiet bed with full-scale clicks placed against the tile grid so that a guess over `window` frames is wrong on
    tiles 1-3 (their last click lies just outside the window, the release is still running), right on tile 4 (a click
    inside the window leaves the ring before the tile: the state is set from it), tiles 5-6 are elementwise and tiles
    8 to the last (a short last tile too) are wrong again.  With window 0 every clicked tile but 0 and 7 is wrong."""
    from audio_mastering_engine_b200 import synth
    T = p.tile
    n = n_tiles * T + extra
    x = (synth.track(n / fs + 0.01, fs, track_id=60) // 4)[:n].copy()
    assert np.abs(x.astype(np.int32)).max() < p.thr
    frames = [T // 2, 4 * T - window + 5, 4 * T + 100] + [k * T - window - 50 for k in (1, 2, 3)]
    frames += [k * T - window - 50 for k in range(8, n_tiles)] + [n - window - 50]
    for f in frames:
        x[f] = [32767, -32767]
    return x


def _cpu_signals(fs, p):
    from audio_mastering_engine_b200 import synth
    sec = 4 * p.tile / fs + 0.05                                            # 4 to 5 tiles
    return {"hot": _hot(synth.track(sec, fs, track_id=33, am_hz=2.0), 14.0),
            "alternating": _hot(synth.track(sec, fs, track_id=35, am_hz=3.0, am_db=10.0), 5.0),
            "stress": _hot(synth.stress_track(sec, fs, track_id=36), 3.5),
            "just_over": _just_over(int(sec * fs), p, 7)}


# ------------------------------------------------------------------------------------------------
# CPU: the model against the sequential limiter
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fs,settings", [(22050, {}), (22050, ALT), (48000, {})])
def test_lim_params_are_the_kernels(fs, settings):
    """The model's constants are the ones design.track_params hands the kernels."""
    from audio_mastering_engine_b200 import design
    tp = design.track_params(dict(FLAT, limiter=True, **settings), fs, 1000)
    p = LimParams.of(fs, settings)
    assert (p.B, p.limit, p.level, p.fsrel, p.release_frames, p.thr) == \
        (tp.lim_frames, tp.lim_limit, tp.lim_level, tp.lim_fs_release, tp.lim_release_frames, tp.lim_thr_i)


def test_model_is_the_sequential_limiter():
    """Whatever the guess window, the tiled scheme with its repairs gives alimiter_py's output bit for bit; the default
    window guesses right on all of these signals, and window 0 leaves tiles open after every round."""
    fs = 22050
    p = LimParams(fs)
    for name, x in _cpu_signals(fs, p).items():
        want = limiter.alimiter_py(x, fs)
        n_tiles = -(-len(x) // p.tile)
        for guess in (0, 1, p.B, p.G, 2 * p.G, -1):
            out, counts, _ = model(x, p, guess)
            assert np.array_equal(out, want), (name, guess, int(np.argmax(np.any(out != want, axis=1))))
            if guess in (-1, 2 * p.G):
                assert counts == [0, 0, 0], (name, guess)
            if guess == 0 and name in ("hot", "just_over"):                # every tile after the first clips
                assert counts == [n_tiles - 1, n_tiles - 2, n_tiles - 3], (name, counts)


def test_model_repair_paths():
    """The click pattern takes every path: wrong and right guesses in one track, repairs gated on a settled
    predecessor, a fallback that stops where its live state meets a recorded guess, one that stops at an exact
    (elementwise) tile and resumes at the next open one, and an open last tile - at a tile-multiple length, one frame
    more and one frame less."""
    fs = 22050
    p = LimParams(fs)
    w = p.B + 20
    for extra in (0, 1, -1):
        x = _clicks(fs, p, w, extra=extra)
        want = limiter.alimiter_py(x, fs)
        tail = -(-len(x) // p.tile) - 8                                     # open tiles from tile 8 on
        out, counts, fb = model(x, p, w)
        assert np.array_equal(out, want)
        assert counts == [3 + tail, 1 + tail, tail - 1], (extra, counts)
        assert fb == dict(walked=tail - 1, stop_exact=0, stop_live=1), (extra, fb)
        out, counts, fb = model(x, p, 0)
        assert np.array_equal(out, want)
        assert counts == [4 + tail, 2 + tail, tail], (extra, counts)
        assert fb == dict(walked=tail, stop_exact=1, stop_live=0), (extra, fb)
        out, counts, fb = model(x, p, -1)
        assert np.array_equal(out, want) and counts == [0, 0, 0]


# ------------------------------------------------------------------------------------------------
# GPU: the kernels with forced guesses against the oracle and the model's counts
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _call(torch, plan, xs, path):
    h_in = plan.pack(xs)
    if path == "host":
        h_out = np.empty_like(h_in)
        plan.master_host(h_in, h_out)
        return plan.unpack(h_out)
    d_in = torch.from_numpy(h_in).cuda(plan.device)
    d_out = torch.empty_like(d_in)
    plan.master_device(d_in, d_out)
    torch.cuda.synchronize(plan.device)
    return plan.unpack(d_out.cpu().numpy())


def _run(torch, xs, fss, sets, guess, path="device", **opts):
    """One call of a fresh plan with the guess window forced: (outputs, limiter_stats())."""
    from audio_mastering_engine_b200 import MasterPlan
    plan = MasterPlan([len(x) for x in xs], fss, sets, host_io=path == "host", **opts)
    try:
        plan.set_limiter_guess(guess)
        return _call(torch, plan, xs, path), plan.limiter_stats()
    finally:
        plan.close()


class Expected:
    """What every call on (xs, fss, sets) must give: the oracle's output per track, and per guess window the model's
    open-tile counts summed over the limiter tracks."""

    def __init__(self, torch, xs, fss, sets):
        self.plains, _ = _run(torch, xs, fss, [dict(s, limiter=False) for s in sets], -1)   # the limiter's input
        self.fss, self.sets = fss, sets
        self.want = [limiter.alimiter(pl, f, s.get("limiter_limit", 0.98), s.get("limiter_attack", 5.0),
                                      s.get("limiter_release", 50.0)) if s.get("limiter") else pl
                     for pl, f, s in zip(self.plains, fss, sets)]
        self._counts = {}

    def counts(self, guess):
        if guess not in self._counts:
            total = np.zeros(3, dtype=np.int64)
            for k, (pl, f, s) in enumerate(zip(self.plains, self.fss, self.sets)):
                if s.get("limiter"):
                    out, c, _ = model(pl, LimParams.of(f, s), guess)
                    assert np.array_equal(out, self.want[k]), ("model", k, guess)
                    total += c
            self._counts[guess] = [int(v) for v in total]
        return self._counts[guess]

    def check(self, outs, stats, guess, label=""):
        for k, (o, w) in enumerate(zip(outs, self.want)):
            assert np.array_equal(o, w), (label, guess, k, int(np.argmax(np.any(o != w, axis=1))))
        assert stats == self.counts(guess), (label, guess, stats, self.counts(guess))


def _check_guesses(torch, xs, fss, sets, guesses, path="device", **opts):
    exp = Expected(torch, xs, fss, sets)
    for g in guesses:
        outs, stats = _run(torch, xs, fss, sets, g, path, **opts)
        exp.check(outs, stats, g, path)
    assert exp.counts(-1) == [0, 0, 0]                # the default window guesses right (DESIGN.md, limiter)
    return exp


@pytest.mark.gpu
def test_forced_guesses_on_the_stage_signals(torch_cuda):
    """The signals of test_limiter_stage_is_bit_exact (1-, 2-, 3- and 21-tile tracks, passages at tile boundaries),
    in one launch with tracks that have no limiter: the output is the oracle's for every window, the open-tile counts
    are the model's, and window 0 leaves tiles open after round 2 - the fallback runs."""
    from audio_mastering_engine_b200 import synth
    fs = 48000
    long = synth.track(5.0, fs, track_id=31) // 2
    long[30000:30400] = _hot(long[30000:30400], 9.0)
    long[65500:65600, 0] = 32767
    long[131071] = [-32768, 32767]
    long[200000:200003] = 32700
    lim = [synth.track(1.0, fs, track_id=30) // 2,
           _hot(synth.track(1.5, fs, track_id=32, am_hz=3.0), 4.0),
           _hot(synth.track(2.0, fs, track_id=33, am_hz=2.0), 14.0),
           long, long[:32768], long[:32769], long[:100],
           _hot(synth.track(14.0, fs, track_id=34, am_hz=1.0), 14.0),
           _hot(synth.track(14.0, fs, track_id=35, am_hz=0.7, am_db=10.0), 5.0),
           _hot(synth.stress_track(11.0, fs, track_id=36), 3.5)]
    xs, sets = [], []
    for k, x in enumerate(lim):
        xs.append(x)
        sets.append(dict(FLAT, limiter=True))
        if k % 3 == 1:                                                      # tracks without the limiter in between
            xs.append(_hot(synth.track(0.7, fs, track_id=70 + k), 6.0))
            sets.append(dict(FLAT))
    exp = _check_guesses(torch_cuda, xs, [fs] * len(xs), sets, (0, 1, LimParams(fs).B + 20, -1))
    c = exp.counts(0)
    assert c[0] > 0 and c[2] > 0, c


@pytest.mark.gpu
def test_forced_guesses_at_tile_edges(torch_cuda):
    """Tracks of a whole number of tiles, one frame more and one frame less, clipping all the way (the last tile is
    open) or clicked so that the fallback stops at an elementwise tile and resumes at the next open one, and stops
    where its live state meets a right guess."""
    from audio_mastering_engine_b200 import synth
    fs = 48000
    p = LimParams(fs)
    w = p.B + 20
    xs, sets = [], []
    for extra in (0, 1, -1):
        xs.append(_hot(synth.track(4 * p.tile / fs + 0.01, fs, track_id=80, am_hz=2.0), 14.0)[:4 * p.tile + extra])
        xs.append(_clicks(fs, p, w, extra=extra))
        sets += [dict(FLAT, limiter=True)] * 2
    xs.append(synth.track(0.5, fs, track_id=81))
    sets.append(dict(FLAT))
    for x in xs[1:6:2]:
        _, _, fb = model(x, p, w)
        assert fb["stop_live"] > 0
        _, _, fb = model(x, p, 0)
        assert fb["stop_exact"] > 0
    exp = _check_guesses(torch_cuda, xs, [fs] * len(xs), sets, (0, w, -1))
    assert exp.counts(0)[2] > 0 and exp.counts(w)[2] > 0


@pytest.mark.gpu
def test_forced_guesses_across_rates_and_parameters(torch_cuda):
    """22.05 to 192 kHz with the default and other limiter parameters in one launch; at 192 kHz the default 5 ms
    attack is 960 frames of look-ahead, near the 1024 queue entries the kernels keep in shared memory."""
    from audio_mastering_engine_b200 import synth
    xs, fss, sets = [], [], []
    for i, fs in enumerate((22050, 44100, 96000, 192000)):
        for j, extra in enumerate(({}, ALT)):
            p = LimParams.of(fs, extra)
            n = 4 * p.tile + 1000 * (i + j)
            xs.append(_hot(synth.track(n / fs + 0.01, fs, track_id=90 + 2 * i + j, am_hz=2.5), 12.0)[:n])
            fss.append(fs)
            sets.append(dict(FLAT, limiter=True, **extra))
        xs.append(_hot(synth.track(0.3, fs, track_id=99 - i), 8.0))
        fss.append(fs)
        sets.append(dict(FLAT))
    assert LimParams(192000).B == 960
    exp = _check_guesses(torch_cuda, xs, fss, sets, (0, 300, -1))
    assert exp.counts(0)[2] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["device", "host"])
def test_forced_guesses_over_waves_and_slots(torch_cuda, path):
    """Three waves over two slots: every wave runs its own rounds and fallback in its slot's buffers, and the stats add
    up over the waves."""
    from audio_mastering_engine_b200 import synth
    fs = 44100
    xs, sets = [], []
    for k in range(7):
        xs.append(_hot(synth.track(0.9 + 0.35 * k, fs, track_id=100 + k, am_hz=2.0), 10.0 if k % 3 else 3.0))
        sets.append(dict(FLAT, limiter=k != 4))
    exp = _check_guesses(torch_cuda, xs, [fs] * len(xs), sets, (0, 300, -1), path, n_waves=3, n_slots=2)
    assert exp.counts(0)[2] > 0


@pytest.mark.gpu
def test_one_plan_two_inputs(torch_cuda):
    """Calls on one plan reuse lim_need and the recorded states: nothing of one call may leak into the next.  The stats
    add up over the calls since the last query, a query resets them, and the window can be changed between calls."""
    from audio_mastering_engine_b200 import AmeError, MasterPlan, synth
    fs = 48000
    n = 5 * 8192 + 77
    a = [_hot(synth.track(n / fs + 0.01, fs, track_id=110 + k, am_hz=2.0), 14.0)[:n] for k in range(2)]
    b = [_hot(synth.track(n / fs + 0.01, fs, track_id=120 + k, am_hz=0.7, am_db=10.0), 5.0)[:n] for k in range(2)]
    sets = [dict(FLAT, limiter=True)] * 2
    ea, eb = Expected(torch_cuda, a, [fs] * 2, sets), Expected(torch_cuda, b, [fs] * 2, sets)
    plan = MasterPlan([n, n], fs, sets)
    try:
        with pytest.raises(AmeError):
            plan.set_limiter_guess(-2)
        plan.set_limiter_guess(0)
        assert plan.limiter_stats() == [0, 0, 0]
        ea.check(_call(torch_cuda, plan, a, "device"), plan.limiter_stats(), 0, "a")
        eb.check(_call(torch_cuda, plan, b, "device"), plan.limiter_stats(), 0, "b after a")
        outs_a = _call(torch_cuda, plan, a, "device")
        outs_b = _call(torch_cuda, plan, b, "device")
        stats = plan.limiter_stats()
        assert stats == [x + y for x, y in zip(ea.counts(0), eb.counts(0))]
        assert plan.limiter_stats() == [0, 0, 0]
        for o, w in zip(outs_a + outs_b, ea.want + eb.want):
            assert np.array_equal(o, w)
        plan.set_limiter_guess(-1)
        ea.check(_call(torch_cuda, plan, a, "device"), plan.limiter_stats(), -1, "a, default window")
        plan.set_limiter_guess(0)
        eb.check(_call(torch_cuda, plan, b, "device"), plan.limiter_stats(), 0, "b again")
    finally:
        plan.close()
    assert ea.counts(0)[0] > 0 and eb.counts(0)[0] > 0
