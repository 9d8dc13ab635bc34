"""Host-side filter design: the reference's settings dict -> ame_track_params (include/ame.h).

Coefficients are designed with the very scipy calls the reference makes, so the CUDA kernels run the
same transfer functions:
  shelves    butter(2, fc / (0.5 fs), btype)                    audio_mastering_engine.py:285
  peaks      butter(4, [lo, hi], 'bandpass', output='sos')      :292-296
  crossover  butter(4, 250 | 4000, 'lowpass' | 'highpass', fs)  :301-302
  K filter   ffmpeg ebur128.c ebur128_init_filter (BS.1770)     called via :229
It also sizes the warm-up each time-parallel tile needs (see DESIGN.md "time parallelism").
"""
from __future__ import annotations

import functools
import math

import numpy as np
from scipy.signal import butter, lfilter, sosfilt

from . import _lib as L

EQ_PRESETS = {  # the preset table of the reference (audio_mastering_engine.py:32-38), part of the contract
    "Vocal Clarity": {"bass_boost": -1.0, "mid_cut": 2.0, "presence_boost": 2.5, "treble_boost": 1.0},
    "Bass Punch": {"bass_boost": 2.5, "mid_cut": 1.0, "presence_boost": -1.0, "treble_boost": 0.5},
    "Vintage Warmth": {"bass_boost": 1.5, "mid_cut": 0.0, "presence_boost": -1.5, "treble_boost": -2.0},
    "Lo-Fi Haze": {"bass_boost": -2.0, "mid_cut": 3.0, "presence_boost": -2.0, "treble_boost": -4.0},
    "EDM Kick & Highs": {"bass_boost": 2.0, "mid_cut": 4.0, "presence_boost": 1.0, "treble_boost": 3.0},
}

WARM_TOL = 1e-13   # residual state error, relative to the signal level, when a tile proper starts
# What this buys (profiles/r02/tiling_sensitivity.txt): at 44.1 / 48 kHz every filter of the chain re-converges BIT FOR BIT
# to the state of the sequential run a few hundred frames after such a start, so the result does not depend on the
# tiling.  At 96 / 192 kHz the 250 Hz low-pass sections (poles at radius 0.992 / 0.996) never do: two FP64 runs that
# started from states one ulp apart stay 1e-14 of full scale apart for good (the filter's own round-off noise floor, no
# warm-up length changes it), and a truncation to int16 lands on the other side of an integer for about one sample in
# 1e9 - isolated +-1 LSB samples in an hour of 96 kHz audio, which tiling produces which is a coin toss.


def _set_bq(dst, b, a):
    dst.b0, dst.b1, dst.b2, dst.a1, dst.a2 = float(b[0]), float(b[1]), float(b[2]), float(a[1]), float(a[2])


def _set_sos(dst_arr, sos):
    for i, row in enumerate(sos):
        assert row[3] == 1.0
        _set_bq(dst_arr[i], row[0:3], row[3:6])


@functools.lru_cache(maxsize=None)
def _shelf_ba(fs, fc, kind):
    b, a = butter(2, fc / (0.5 * fs), btype=kind)
    return tuple(b), tuple(a)


@functools.lru_cache(maxsize=None)
def _peak_sos(fs, center_hz, q=1.41):
    nyq = 0.5 * fs
    c = center_hz / nyq
    bw = c / q
    lo, hi = c - (bw / 2), c + (bw / 2)
    if lo <= 0:
        lo = 1e-9
    if hi >= 1.0:
        hi = 0.999999
    return butter(4, [lo, hi], btype="bandpass", output="sos")


@functools.lru_cache(maxsize=None)
def _xover_sos(fs, low_crossover=250, high_crossover=4000):
    return (butter(4, low_crossover, btype="lowpass", fs=fs, output="sos"),
            butter(4, high_crossover, btype="highpass", fs=fs, output="sos"))


@functools.lru_cache(maxsize=None)
def k_weighting_biquads(fs):
    """BS.1770 pre-filter and RLB high-pass as two biquads (ebur128.c keeps them convolved)."""
    f0, G, Q = 1681.974450955533, 3.999843853973347, 0.7071752369554196
    K = math.tan(math.pi * f0 / float(fs))
    Vh = math.pow(10.0, G / 20.0)
    Vb = math.pow(Vh, 0.4996667741545416)
    a0 = 1.0 + K / Q + K * K
    pb = ((Vh + Vb * K / Q + K * K) / a0, 2.0 * (K * K - Vh) / a0, (Vh - Vb * K / Q + K * K) / a0)
    pa = (1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0)
    f0, Q = 38.13547087602444, 0.5003270373238773
    K = math.tan(math.pi * f0 / float(fs))
    rb = (1.0, -2.0, 1.0)
    ra = (1.0, 2.0 * (K * K - 1.0) / (1.0 + K / Q + K * K), (1.0 - K / Q + K * K) / (1.0 + K / Q + K * K))
    return (pb, pa), (rb, ra)


def _decay_frames(run, pole_radius, tol=WARM_TOL):
    """Frames after which the zero-input response of the linear system `run` (a callable on a float64
    vector) has fallen below tol * (rms of its driven output).  `pole_radius` sizes the simulation."""
    est = int(math.log(tol) / math.log(min(max(pole_radius, 0.5), 0.999999))) + 64
    n0, n1 = est, int(est * 2.5) + 256
    rng = np.random.default_rng(1234)
    x = np.concatenate([rng.standard_normal(n0), np.zeros(n1)])
    y = run(x)
    ref = math.sqrt(float(np.mean(y[:n0] ** 2))) or 1.0
    tail = np.abs(y[n0:])
    idx = np.nonzero(tail > tol * ref)[0]
    w = int(idx[-1]) + 1 if idx.size else 0
    if w >= n1 - 1:   # did not decay inside the window: fall back to a generous analytic bound
        w = int(est * 3)
    return int(math.ceil((w * 1.05 + 32) / 64.0) * 64)


def _max_radius(sections):
    r = 0.0
    for b, a in sections:
        r = max(r, float(np.max(np.abs(np.roots(a)))))
    return r


@functools.lru_cache(maxsize=None)
def eq_warm_frames(fs, bass, mid_cut, presence, treble):
    secs, stages = [], []
    if bass != 0.0:
        b, a = _shelf_ba(fs, 250, "low")
        secs.append((b, a))
    if -mid_cut != 0:
        secs += [(r[0:3], r[3:6]) for r in _peak_sos(fs, 1000)]
    if presence != 0:
        secs += [(r[0:3], r[3:6]) for r in _peak_sos(fs, 4000)]
    if treble != 0.0:
        b, a = _shelf_ba(fs, 8000, "high")
        secs.append((b, a))
    if not secs:
        return 0

    def run(x):
        v = x
        if bass != 0.0:
            b, a = _shelf_ba(fs, 250, "low")
            y = lfilter(b, a, v)
            g = 10.0 ** (bass / 20.0)
            v = v + (y - v) * (g - 1) if bass > 0 else y
        if -mid_cut != 0:
            v = v + sosfilt(_peak_sos(fs, 1000), v) * (10 ** (-mid_cut / 20.0) - 1)
        if presence != 0:
            v = v + sosfilt(_peak_sos(fs, 4000), v) * (10 ** (presence / 20.0) - 1)
        if treble != 0.0:
            b, a = _shelf_ba(fs, 8000, "high")
            y = lfilter(b, a, v)
            g = 10.0 ** (treble / 20.0)
            v = v + (y - v) * (g - 1) if treble > 0 else y
        return v

    return _decay_frames(run, _max_radius(secs))


@functools.lru_cache(maxsize=None)
def xover_warm_frames(fs):
    lo, hi = _xover_sos(fs)
    secs = [(r[0:3], r[3:6]) for r in list(lo) + list(hi)]
    return _decay_frames(lambda x: np.abs(sosfilt(lo, x)) + np.abs(sosfilt(hi, x)), _max_radius(secs))


@functools.lru_cache(maxsize=None)
def kw_warm_frames(fs):
    (pb, pa), (rb, ra) = k_weighting_biquads(fs)
    return _decay_frames(lambda x: lfilter(rb, ra, lfilter(pb, pa, x)), _max_radius([(pb, pa), (rb, ra)]))


def warm_lut(analog_character):
    """float32 tanh table over all 65536 int16 inputs - the reference's own expression
    np.tanh(samples * drive) (audio_mastering_engine.py:260-263) evaluated by numpy on this host."""
    cf = analog_character / 100.0
    drive = 1.0 + (cf * 0.5)
    x = np.arange(-32768, 32768, dtype=np.int32).astype(np.int16).astype(np.float32) / (2 ** 15)
    return np.tanh(x * drive).astype(np.float32, copy=False)


def track_params(settings, fs, n_frames, offset_frames=0, chunk_seconds=30, lut_index=None, halo_frames=0):
    """Fill one ame_track_params from a reference-style settings dict.  `lut_index` maps
    analog_character -> table index and is extended in place."""
    fs = int(fs)
    if fs < 4000:       # the BS.1770 pre-filter sits at 1682 Hz: below ~3.4 kHz sampling it is not a filter any more
        raise ValueError(f"unsupported sample rate {fs} Hz")
    p = L.TrackParams()
    p.offset_frames, p.n_frames, p.sample_rate = int(offset_frames), int(n_frames), fs
    p.halo_frames = int(halo_frames)
    p.chunk_frames = int(chunk_seconds * fs) if chunk_seconds else 0
    flags = 0
    p.warm_lut = -1
    ac = settings.get("analog_character", 0)
    if ac > 0:                                            # :192
        flags |= L.AME_F_WARMTH
        cf = ac / 100.0
        for pre, fc, gdb, kind in (("wl", 120, cf * 1.0, "low"), ("wh", 12000, cf * 1.5, "high")):
            b, a = _shelf_ba(fs, fc, kind)
            setattr(p, pre + "_b0", b[0]); setattr(p, pre + "_b1", b[1]); setattr(p, pre + "_a1", a[1])
            setattr(p, pre + "_gm1", 10.0 ** (gdb / 20.0) - 1)
        if lut_index is not None:
            p.warm_lut = lut_index.setdefault(float(ac), len(lut_index))
    bass = settings.get("bass_boost", 0.0)
    mid_cut = settings.get("mid_cut", 0.0)
    presence = settings.get("presence_boost", 0.0)
    treble = settings.get("treble_boost", 0.0)
    for i, (gdb, fc, kind) in enumerate(((bass, 250, "low"), (-mid_cut, 1000, None), (presence, 4000, None),
                                         (treble, 8000, "high"))):
        st = p.eq[i]
        if gdb == 0:
            st.kind = L.AME_EQ_BYPASS
            continue
        g = 10.0 ** (gdb / 20.0)
        st.g, st.gm1 = g, g - 1
        if kind is not None:
            b, a = _shelf_ba(fs, fc, kind)
            st.kind = L.AME_EQ_SHELF_BOOST if gdb > 0 else L.AME_EQ_SHELF_CUT
            st.n_sections = 1
            _set_bq(st.s[0], b, a)
        else:
            st.kind, st.n_sections = L.AME_EQ_PEAK, 4
            _set_sos(st.s, _peak_sos(fs, fc))
    w = settings.get("width", 1.0)
    if w != 1.0:                                          # :195
        flags |= L.AME_F_WIDTH
    p.width = float(np.float32(w))
    if settings.get("multiband"):                         # :197
        flags |= L.AME_F_MULTIBAND
        lo, hi = _xover_sos(fs)
        _set_sos(p.xlp, lo)
        _set_sos(p.xhp, hi)
        for b, name in enumerate(("low", "mid", "high")):
            thr, ratio = settings.get(name + "_thresh"), settings.get(name + "_ratio")
            if thr is None or ratio is None:
                raise TypeError(f"multiband is set but {name}_thresh / {name}_ratio is missing")  # pydub would raise too
            cb = p.comp[b]
            cb.thresh_rms = 32768.0 * (10 ** (float(thr) / 20))
            cb.coef = 1 - (1.0 / ratio)
            cb.attack_frames = 5.0 * (fs / 1000.0)
            cb.release_frames = 50.0 * (fs / 1000.0)
            cb.look_frames = int(cb.attack_frames)
            cb.table = -1
        p.warm_xover = xover_warm_frames(fs)
    if settings.get("lufs") is not None:                  # :216
        flags |= L.AME_F_NORMALIZE
        p.target_lufs = float(settings.get("lufs"))
    (pb, pa), (rb, ra) = k_weighting_biquads(fs)
    _set_bq(p.kw[0], pb, pa)
    _set_bq(p.kw[1], rb, ra)
    p.warm_kw = kw_warm_frames(fs)
    p.warm_eq = eq_warm_frames(fs, float(bass), float(mid_cut), float(presence), float(treble))
    if settings.get("limiter"):                            # ffmpeg alimiter=level_in=1:level_out=1:limit=0.98:attack=5:release=50 (:223)
        flags |= L.AME_F_LIMITER
        limit = float(settings.get("limiter_limit", 0.98))
        attack, release = float(settings.get("limiter_attack", 5.0)) / 1000.0, float(settings.get("limiter_release", 50.0)) / 1000.0
        buffer_size = int(fs * attack * 2)                 # af_alimiter.c config_input, two channels
        buffer_size -= buffer_size % 2
        p.lim_frames = buffer_size // 2
        p.lim_limit, p.lim_level, p.lim_fs_release = limit, 1.0 / limit, fs * release
        p.lim_release_frames = int(math.ceil(fs * release))
        thr = int(math.floor(limit * 32768.0))
        while thr / 32768.0 <= limit:                      # smallest |s16| with x / 32768 > limit
            thr += 1
        p.lim_thr_i = thr
    if settings.get("true_peak"):
        flags |= L.AME_F_TRUE_PEAK
    if settings.get("measure_output"):                    # EBU R128 meter of the final output (ame_loudness)
        flags |= L.AME_F_MEASURE_OUTPUT
    p.flags = flags
    return p
