"""Host-side model of the algorithm inside k_att_chain_spec (csrc/ame_kernels.cuh): the compressor's attenuation
recurrence evaluated in S time segments from guessed starts and repaired until exact.  The model restates the
kernel's control flow in Python - pass 1 from a guessed start, repair passes that carry the old and the new start and stop
where they are equal, starts handed across silent segments - and checks the claim the kernel relies on: when no
segment's start changes any more, every stored value is the one the sequential loop (pydub's, oracle/chain.py)
produces, bit for bit; and the tau form of the update used on the GPU is the reference's update.
CPU only; the CUDA kernel itself is compared with the sequential kernel and the oracle in test_gpu_parity.py."""
import math

import numpy as np
import pytest

from oracle import chain


def _entries(fs, threshold, ratio):
    """(M, inc, dec, tau) per integer rms, as build_att_table in csrc/ame_layout.h does; flagged(r) = r > thresh_rms."""
    thr, _look, attack_frames, release_frames = chain.compressor_constants(fs, threshold, ratio)
    table = {}

    def entry(r):
        if r not in table:
            m = chain.max_attenuation_for_rms(r, thr, ratio)
            inc, dec = m / attack_frames, m / release_frames
            tau = max(m - inc, 0.0)
            while tau > 0 and tau + inc >= m:
                tau = math.nextafter(tau, -1.0)
            while tau + inc < m:
                tau = math.nextafter(tau, 1e300)
            table[r] = (m, inc, dec, tau)
        return table[r]
    return thr, entry


def _update_ref(att, m, inc, dec):
    """pydub's step for a frame above threshold (below it M = 0 and nothing moves)."""
    if att <= m:
        return min(att + inc, m)
    return max(att - dec, 0)


def _update_gpu(att, m, inc, dec, tau):
    """att_update() of the kernels: both predicates on the OLD attenuation."""
    if att > m:
        return att - dec
    return att + inc if att < tau else m


def _sequential(rms, thr, entry):
    att, out = 0.0, np.zeros(len(rms))
    for i, r in enumerate(rms):
        if r > thr:
            m, inc, dec, _ = entry(int(r))
            att = _update_ref(att, m, inc, dec)
        out[i] = att
    return out


def _walk(rms, thr, entry, b0, b1, b, out, a=None):
    """Frames [b0, b1) from attenuation b, storing into out; with `a` also the previous start's trajectory, stopping
    after the first flagged frame where the two are equal.  Returns (end value, met)."""
    for i in range(b0, b1):
        r = rms[i]
        if r > thr:
            e = entry(int(r))
            b = _update_gpu(b, *e)
            if a is not None:
                a = _update_gpu(a, *e)
        out[i] = b
        if a is not None and r > thr and a == b:
            return b, True
    return b, False


def _speculative(rms, thr, entry, n_seg):
    n = len(rms)
    seg = -(-n // n_seg)
    bounds = [(min(n, t * seg), min(n, (t + 1) * seg)) for t in range(n_seg)]
    out = np.zeros(n)
    start = [0.0] * n_seg
    end = [0.0] * n_seg
    flagged = [bool(np.any(rms[b0:b1] > thr)) for b0, b1 in bounds]
    for t, (b0, b1) in enumerate(bounds):                       # pass 1, from a guess: M of the last flagged frame in front
        if t > 0 and b0 < b1:
            for i in range(b0 - 1, max(0, b0 - 64) - 1, -1):
                if rms[i] > thr:
                    start[t] = entry(int(rms[i]))[0]
                    break
        end[t], _ = _walk(rms, thr, entry, b0, b1, start[t], out)
    prev = []
    for t in range(n_seg):                                      # last segment before t that holds a flagged frame
        u = t - 1
        while u >= 0 and not flagged[u]:
            u -= 1
        prev.append(u)
    passes = 0
    while True:
        frm = [end[prev[t]] if prev[t] >= 0 else 0.0 for t in range(n_seg)]     # all lanes read, then all write
        redo = [t for t in range(n_seg) if frm[t] != start[t]]
        if not redo:
            return out, passes
        passes += 1
        assert passes <= n_seg, "one more segment must become final in every pass"
        for t in redo:
            b0, b1 = bounds[t]
            b, met = _walk(rms, thr, entry, b0, b1, frm[t], out, a=start[t])
            if not met:
                end[t] = b
            start[t] = frm[t]


def _rms_series(rng, n, kind):
    t = np.arange(n)
    if kind == "bursts":                 # loud / quiet alternation: the attenuation clamps and parks in turn
        level = 2500 + 2200 * np.sign(np.sin(2 * np.pi * t / 1700.0)) + rng.integers(-300, 300, n)
    elif kind == "held":                 # one loud passage, then a bed just over threshold: never clamps again
        level = np.where(t < 400, 20000, 3320) + rng.integers(-15, 15, n)
    elif kind == "sparse":               # a handful of flagged frames in mostly silent segments
        level = np.where(rng.random(n) < 0.004, 9000, 100)
    else:                                # noise around the threshold
        level = 3277 + rng.integers(-1500, 1500, n)
    return np.clip(level, 0, 32768).astype(np.int64)


@pytest.mark.parametrize("kind", ["bursts", "held", "sparse", "noise"])
@pytest.mark.parametrize("n_seg", [1, 7, 32])
def test_speculate_and_repair_equals_sequential(kind, n_seg):
    rng = np.random.default_rng(11)
    fs, threshold, ratio = 48000, -20.0, 4.0
    thr, entry = _entries(fs, threshold, ratio)
    rms = _rms_series(rng, 6000, kind)
    want = _sequential(rms, thr, entry)
    got, passes = _speculative(rms, thr, entry, n_seg)
    assert np.array_equal(got, want), (kind, n_seg)
    if kind == "held" and n_seg > 1:
        assert passes >= n_seg // 2          # the strictly sequential case: about one segment settles per pass


def test_tau_form_is_the_reference_update():
    """att < tau  <=>  fl(att + inc) < M for the tau of the table, so both forms take the same branch everywhere."""
    rng = np.random.default_rng(5)
    thr, entry = _entries(44100, -25.0, 6.0)
    for r in rng.integers(int(thr) + 1, 32768, 300):
        m, inc, dec, tau = entry(int(r))
        probes = [0.0, tau, math.nextafter(tau, 0.0), math.nextafter(tau, 1e9), m, math.nextafter(m, 1e9), m - inc, 2 * m]
        probes += list(rng.uniform(0, 1.5 * m, 20))
        for att in probes:
            assert _update_gpu(att, m, inc, dec, tau) == _update_ref(att, m, inc, dec), (r, att)


# ------------------------------------------------------------------------------------------------
# Model of k_att_chain as it is now: the flagged frames compacted into a dense list, S segments of equal step count,
# and the "parked prefix" shortcut - a start moved by d ulps moves every stored value of the release-branch prefix by
# d ulps (same binade, no tie, still above every max_attenuation), and nothing behind a step that clamps.
# ------------------------------------------------------------------------------------------------
def _bits(x):
    return int(np.float64(x).view(np.int64))


def _from_bits(b):
    return float(np.int64(b).view(np.float64))


class _Sum:
    def __init__(self, start):
        self.margin, self.at_p, self.lo, self.hi, self.p = None, 0, 0, -1, 0
        self.exp0 = _bits(start) >> 52
        self.open, self.ok = True, self.exp0 > 0


def _walk_list(entries, b0, b1, b, out, a=None, u=None):
    """Steps [b0, b1) in blocks of 8 as the kernel does (the meeting test is per block)."""
    i = b0
    while i < b1:
        for k in range(i, min(i + 8, b1)):
            m, inc, dec, tau = entries[k]
            if u is not None and u.open:
                ib, im = _bits(b), _bits(m)
                if ib > im:
                    u.margin = ib - im if u.margin is None else min(u.margin, ib - im)
                    idec = _bits(dec)
                    if idec != 0:
                        ed = idec >> 52
                        mant = (idec & ((1 << 52) - 1)) | ((1 << 52) if ed else 0)
                        low = (mant & -mant).bit_length() - 1
                        if (ed if ed else 1) + low == u.exp0 - 1:
                            u.ok = False
                    u.p += 1
                else:
                    u.open = False
                    u.at_p, u.lo, u.hi = ib, _bits(tau), im
                    if (ib >> 52) != u.exp0:
                        u.ok = False
            b = _update_gpu(b, m, inc, dec, tau)
            if a is not None:
                a = _update_gpu(a, m, inc, dec, tau)
            out[k] = b
        i += 8
        if a is not None and _bits(a) == _bits(b):
            return b, True
    return b, False


def _chain_v2(rms, thr, entry, n_lanes):
    flagged = [int(r) for r in rms if r > thr]
    entries = [entry(r) for r in flagged]
    n_f = len(entries)
    seg = max(64, (-(-n_f // n_lanes) + 7) // 8 * 8) if n_f else 64
    s_used = -(-n_f // seg)
    bounds = [(min(n_f, t * seg), min(n_f, (t + 1) * seg)) for t in range(s_used)]
    out = np.zeros(n_f)
    start = [0.0] * s_used
    end = [0.0] * s_used
    sums = [None] * s_used
    pending = [0] * s_used
    for t, (b0, b1) in enumerate(bounds):
        if t > 0:
            start[t] = entries[b0 - 1][0]
        end[t], _ = _walk_list(entries, b0, b1, start[t], out)
    # forecast: segments the trajectory from lane 0's (final) end crosses parked throughout walk again from that value
    guess = [None] * s_used
    if s_used:
        lb = end[0]
        for t in range(1, s_used):
            b0, b1 = bounds[t]
            max_m = max(e[0] for e in entries[b0:b1])
            sum_dec = 0.0
            for e in entries[b0:b1]:
                sum_dec += e[2]
            lo = lb - 1.000001 * sum_dec
            if lb > 0.0 and lo > max_m:
                guess[t] = lb
                lb = lo
            else:
                lb = end[t]
    quick_used = walks = 0

    def flush(t):
        if pending[t]:
            b0 = bounds[t][0]
            for i in range(b0, b0 + sums[t].p):
                out[i] = _from_bits(_bits(out[i]) + pending[t])
            pending[t] = 0

    passes = 1
    while True:
        frm = [end[t - 1] if t > 0 else 0.0 for t in range(s_used)]
        if passes == 1:
            frm = [guess[t] if guess[t] is not None else frm[t] for t in range(s_used)]
        redo = [t for t in range(s_used) if _bits(frm[t]) != _bits(start[t])]
        if not redo:
            break
        passes += 1
        assert passes <= s_used + 2
        for t in redo:
            b0, b1 = bounds[t]
            u = sums[t]
            fb = _bits(frm[t])
            d = fb - _bits(start[t])
            quick = u is not None and u.ok and (fb >> 52) == u.exp0 and (d >= 0 or u.p == 0 or u.margin > -d)
            if quick and u.open:
                quick = ((_bits(end[t]) + d) >> 52) == u.exp0
            if quick and not u.open:
                quick = u.lo <= u.at_p <= u.hi and u.lo <= u.at_p + d <= u.hi and ((u.at_p + d) >> 52) == u.exp0
            if quick:
                quick_used += 1
                pending[t] += d
                if u.p:
                    u.margin += d
                if u.open:
                    end[t] = _from_bits(_bits(end[t]) + d)
                else:
                    u.at_p += d
            else:
                walks += 1
                flush(t)
                u = sums[t] = _Sum(frm[t])
                b, met = _walk_list(entries, b0, b1, frm[t], out, a=start[t], u=u)
                if not met:
                    end[t] = b
                if u.open and (met or (_bits(end[t]) >> 52) != u.exp0):
                    u.ok = False
            start[t] = frm[t]
    for t in range(s_used):
        flush(t)
    # scatter back to frames: attenuation after every frame
    att, k, cur = np.zeros(len(rms)), 0, 0.0
    for i, r in enumerate(rms):
        if r > thr:
            cur = out[k]
            k += 1
        att[i] = cur
    return att, passes, quick_used, walks


@pytest.mark.parametrize("kind", ["bursts", "held", "sparse", "noise"])
@pytest.mark.parametrize("n_lanes", [1, 5, 32, 128])
def test_dense_list_chain_with_parked_shortcut_equals_sequential(kind, n_lanes):
    rng = np.random.default_rng(23)
    fs, threshold, ratio = 48000, -20.0, 4.0
    thr, entry = _entries(fs, threshold, ratio)
    rms = _rms_series(rng, 24000, kind)
    want = _sequential(rms, thr, entry)
    got, passes, quick, walks = _chain_v2(rms, thr, entry, n_lanes)
    assert np.array_equal(got.view(np.int64), want.view(np.int64)), (kind, n_lanes)
    if kind == "held" and n_lanes >= 32:
        # the parked chain: after one repair walk per segment the start changes are applied as integer shifts
        assert quick > walks, (quick, walks)


def test_parked_shortcut_random_thresholds():
    """Many parked regimes (different binades, ratios, levels just over threshold) - bit-exact every time."""
    rng = np.random.default_rng(99)
    for trial in range(12):
        fs = int(rng.choice([44100, 48000, 96000]))
        threshold, ratio = float(rng.uniform(-40, -5)), float(rng.uniform(1.5, 10))
        thr, entry = _entries(fs, threshold, ratio)
        n = 12000
        t = np.arange(n)
        loud = int(min(32768, thr * rng.uniform(3, 9)))
        bed = int(thr * rng.uniform(1.002, 1.2)) + 1
        level = np.where(t < rng.integers(100, 900), loud, bed) + rng.integers(-3, 4, n)
        if trial % 3 == 0:                      # a second loud passage: the chain clamps again in the middle
            level[6000:6300] = loud
        rms = np.clip(level, 0, 32768).astype(np.int64)
        want = _sequential(rms, thr, entry)
        got, _, _, _ = _chain_v2(rms, thr, entry, 64)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), trial
