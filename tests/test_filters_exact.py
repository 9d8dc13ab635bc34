"""k_eq, k_band_split and k_kweight_energy held to an extended-precision reference.

The three FP64 filter kernels start every tile from a state that a warm-up run computes (DESIGN.md sections 3 and 6).
The reference here makes the oracle's own filter calls, scipy.signal.lfilter / sosfilt with the same float64
coefficients, on np.longdouble arrays.  Every step the reference defines in float32 stays float32: the float32 input
channel, the first cut shelf's samples * g, the float32 store after the EQ, width and the x 32767 of to_pcm.

Certificate.  An output sample is certain when its quantisation chain gives the same int16 at the reference value
moved by -DELTA and by +DELTA.  For the mid band, low and high move independently, since mid = x - low - high.  A
certain sample must match exactly.  Any other sample is a knife edge, and either neighbour is accepted.  Each test
prints its knife-edge candidates and the samples that actually differ from the reference's own rounding.

DELTA = 1e-6 LSB.  On a CPU, with synth.track, scipy's float64 filters deviate from the long-double run by at most
5.5e-11 LSB (250 Hz shelf, 22.05 kHz), 2.7e-10 (same, 48 kHz), 3.0e-9 (same, 384 kHz), 1.8e-9 (1 kHz peak, 384 kHz)
and 1.1e-8 (crossover low-pass, 384 kHz).  So DELTA is about 100x the worst float64 deviation.
test_oracle_obeys_certificate re-checks this at every rate used here.  A warm-up cut in half moves samples by about
1e-3 LSB, 1000x DELTA.

K-weighted sub-block energies are compared with long-double sums to KW_REL = 1e-10 relative.  float64 against long
double is at most 4.5e-13 relative at 384 kHz and 2.4e-14 at 48 kHz.  A sub-block one frame off at a tile edge is
2.6e-5 to 2e-4 of its energy.
"""
import itertools
import json
import math
import os
import subprocess

import numpy as np
import pytest
from scipy.signal import lfilter, sosfilt

from audio_mastering_engine_b200 import _lib as L, design, synth
from oracle import chain

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LD = np.longdouble
DELTA_LSB = 1e-6
DELTA = LD(DELTA_LSB) / LD(32768)          # in full-scale units
KW_REL = 1e-10
KW_ABS = 1e-20                             # decaying silence: sub-block sums of squares far below the -70 LUFS gate
AME_E_UNSUPPORTED = -4                     # include/ame.h

HIGH_RATES = (22050, 44100, 48000, 96000, 192000, 352800, 384000)
LOW_RATES = (8000, 11025, 16000)
# gain in dB of each EQ stage in its three states: bypass, positive, negative (stage 1 is -mid_cut)
STAGE_GAINS = ((0.0, 3.5, -4.5), (0.0, 2.5, -3.0), (0.0, 2.0, -5.0), (0.0, 4.0, -3.5))
STAGE_KEYS = (("bass_boost", 250, "low"), ("mid_cut", 1000, None), ("presence_boost", 4000, None), ("treble_boost", 8000, "high"))


def eq_settings(g0=0.0, g1=0.0, g2=0.0, g3=0.0, **extra):
    s = dict(bass_boost=g0, mid_cut=-g1 if g1 else 0.0, presence_boost=g2, treble_boost=g3, analog_character=0,
             width=1.0, lufs=None, multiband=False)
    s.update(extra)
    return s


def stage_gains(s):
    return (s.get("bass_boost", 0.0), -s.get("mid_cut", 0.0), s.get("presence_boost", 0.0), s.get("treble_boost", 0.0))


# ------------------------------------------------------------------------------------------------
# the reference
# ------------------------------------------------------------------------------------------------
def _ld(c):
    return np.asarray(c, dtype=np.float64).astype(LD)


def ref_eq_channel(ch32, fs, s):
    """chain.eq_channel on a float32 channel with the filter arithmetic in long double."""
    v = ch32.astype(LD)
    first = True
    for gdb, (_, fc, kind) in zip(stage_gains(s), STAGE_KEYS):
        if gdb == 0:
            continue
        g = 10.0 ** (gdb / 20.0)
        if kind is None:
            v = v + sosfilt(_ld(design._peak_sos(fs, fc)), v) * LD(g - 1)
        else:
            b, a = design._shelf_ba(fs, fc, kind)
            y = lfilter(_ld(b), _ld(a), v)
            if gdb > 0:
                v = v + (y - v) * LD(g - 1)
            else:   # samples * g: float32 while the input is still the float32 channel (numpy keeps the array's dtype)
                t = (ch32 * np.float32(g)).astype(LD) if first else v * LD(g)
                v = t + (y - t)
        first = False
    return v


def chunk_bounds(n, fs, chunk_seconds):
    return chain.chunk_bounds(n, fs, chunk_seconds) if chunk_seconds else [(0, n)]


def ref_eq(x, fs, s, chunk_seconds):
    """(left, right) long-double EQ outputs of int16[N,2] x, filter state reset at every chunk."""
    vl, vr = np.empty(len(x), LD), np.empty(len(x), LD)
    for b, e in chunk_bounds(len(x), fs, chunk_seconds):
        pcm = x[b:e]
        if s.get("analog_character", 0) > 0:
            pcm = chain.warmth(pcm, fs, s["analog_character"])
        f = chain.to_float(pcm)
        vl[b:e] = ref_eq_channel(f[:, 0], fs, s)
        vr[b:e] = ref_eq_channel(f[:, 1], fs, s)
    return vl, vr


def q_eq(vl, vr, w):
    """Float32 store after the EQ, width, to_pcm."""
    y = np.stack([vl.astype(np.float64).astype(np.float32), vr.astype(np.float64).astype(np.float32)], axis=1)
    if w != 1.0:
        y = chain.width(y, w)
    return chain.to_pcm(y)


def q64(v):
    return chain.to_pcm(np.asarray(v, dtype=LD).astype(np.float64))


class Tally:
    """Knife-edge candidates and actual flips of one test."""

    def __init__(self, name):
        self.name, self.samples, self.edges, self.flips = name, 0, 0, 0

    def check(self, got, center, corners, label):
        got = np.asarray(got, np.int32)
        cs = [np.asarray(c, np.int32) for c in corners]
        lo, hi = np.minimum.reduce(cs), np.maximum.reduce(cs)
        edge = lo != hi
        bad = np.where(edge, (got < lo) | (got > hi), got != lo)
        if bad.any():
            i = np.unravel_index(int(np.argmax(bad)), bad.shape)
            pytest.fail(f"{self.name} {label}: {int(bad.sum())} certain samples differ; first at {i}: got {got[i]}, "
                        f"reference {int(np.asarray(center, np.int32)[i])} (corners {int(lo[i])}..{int(hi[i])})")
        self.samples += got.size
        self.edges += int(edge.sum())
        self.flips += int((got != np.asarray(center, np.int32)).sum())

    def report(self):
        print(f"{self.name}: {self.samples} samples, {self.edges} knife-edge candidates, {self.flips} flips")


def certify_eq(tally, got, x, fs, s, chunk_seconds, label):
    vl, vr = ref_eq(x, fs, s, chunk_seconds)
    w = s.get("width", 1.0)
    corners = [q_eq(vl + a * DELTA, vr + b * DELTA, w) for a, b in itertools.product((-1, 1), (-1, 1))]
    tally.check(got, q_eq(vl, vr, w), corners, label)


def ref_split(pre, fs, chunk_seconds):
    """(x, low, high) in long double for an int16[N,2] pre signal, state reset at every chunk."""
    x = np.asarray(pre, np.int16).astype(LD) / LD(32768)
    lo_sos, hi_sos = (_ld(s) for s in design._xover_sos(fs))
    lo, hi = np.empty_like(x), np.empty_like(x)
    for b, e in chunk_bounds(len(x), fs, chunk_seconds):
        lo[b:e] = sosfilt(lo_sos, x[b:e], axis=0)
        hi[b:e] = sosfilt(hi_sos, x[b:e], axis=0)
    return x, lo, hi


def certify_split(tally, bands, pre, fs, chunk_seconds, label):
    x, lo, hi = ref_split(pre, fs, chunk_seconds)
    d = (-DELTA, DELTA)
    tally.check(bands[0], q64(lo), [q64(lo + a) for a in d], label + " low")
    tally.check(bands[2], q64(hi), [q64(hi + a) for a in d], label + " high")
    tally.check(bands[1], q64(x - lo - hi), [q64(x - (lo + a) - (hi + b)) for a in d for b in d], label + " mid")


def ref_kw_energies(pre, fs, dtype=LD):
    """Per 100 ms sub-block: both channels' sums of squares of the K-weighted signal (the two biquads in series)."""
    (pb, pa), (rb, ra) = design.k_weighting_biquads(fs)
    x = np.asarray(pre, np.int16).astype(dtype) / dtype(32768)
    c = (lambda v: np.asarray(v, np.float64).astype(dtype))
    y = lfilter(c(rb), c(ra), lfilter(c(pb), c(pa), x, axis=0), axis=0)
    s100 = chain.samples_in_100ms(fs)
    n_sb = len(x) // s100
    return (y[:n_sb * s100] ** 2).sum(axis=1).reshape(n_sb, s100).sum(axis=1)


def check_energies(got, want, label):
    got = np.asarray(got, np.float64)
    assert got.shape == want.shape, label
    err = np.abs(got.astype(LD) - want)
    bad = err > np.maximum(KW_REL * np.abs(want), KW_ABS)
    assert not bad.any(), (label, int(np.argmax(bad)), float(got[np.argmax(bad)]), float(want[np.argmax(bad)]))
    nz = want > KW_ABS
    return float((err[nz] / want[nz]).max()) if nz.any() else 0.0


# ------------------------------------------------------------------------------------------------
# signals and track sets
# ------------------------------------------------------------------------------------------------
def signal(kind, n, fs, seed):
    """0: synth.track; 1: synth.track at -20 dB; 2: full-scale noise; 3: synth.stress_track; 4: synth.track whose last
    third is 12 dB hot (clipped in int16, and driven past full scale by any boost)."""
    if n == 0:
        return np.zeros((0, 2), np.int16)
    secs = n / fs
    if kind == 2:
        return np.random.default_rng(seed).integers(-32768, 32768, size=(n, 2)).astype(np.int16)
    if kind == 3:
        x = synth.stress_track(max(secs, 1.0), fs, track_id=seed)
        return np.ascontiguousarray(x[(len(x) - n) // 2:][:n])
    x = synth.track(secs + 1.0 / fs, fs, track_id=seed)[:n]
    if kind == 1:
        return (x.astype(np.int32) // 10).astype(np.int16)
    if kind == 4:
        x = x.copy()
        k = 2 * n // 3
        x[k:] = np.clip(x[k:].astype(np.int32) * 4, -32768, 32767).astype(np.int16)
    return x


def eq_frames(fs):
    """Two of the slowest k_eq warm-ups at fs (every stage libame accepts there) and an odd tail."""
    return 2 * design.eq_warm_frames(fs, 2.0, 2.0, 2.0 if fs >= 22050 else 0.0, 2.0 if fs > 16000 else 0.0) + 1001


def variant_matrix(fs):
    """One settings dict per (stage states) x warmth x width that libame accepts at fs."""
    allowed = [True, True, fs >= 22050, fs > 16000]
    states = [STAGE_GAINS[s] if allowed[s] else (0.0,) for s in range(4)]
    warm = (0, 30) if fs > 24000 else (0,)
    out = []
    for gains in itertools.product(*states):
        for ac in warm:
            for w in (1.0, 1.37):
                out.append(eq_settings(*gains, analog_character=ac, width=w))
    return out


@pytest.fixture(scope="module")
def torch_cuda():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def run_eq(torch, plan, tracks):
    """Pack, stage_eq, return (d_in, d_pre, per-track pre as numpy)."""
    dev = torch.device("cuda", plan.device)
    d_in = torch.from_numpy(plan.pack(tracks)).to(dev)
    d_pre = torch.zeros_like(d_in)
    plan.stage_eq(d_in, d_pre)
    torch.cuda.synchronize()
    return d_in, d_pre, plan.unpack(d_pre.cpu().numpy())


# ------------------------------------------------------------------------------------------------
# CPU: the reference, the certificate and the settings libame rejects
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fs", LOW_RATES + HIGH_RATES)
def test_oracle_obeys_certificate(fs):
    """The oracle's float64 chain (scipy on float64) passes the certificate against the long-double reference: DELTA
    covers float64 round-off at this rate.  Also prints the largest float64 deviation of the crossover and K filter."""
    tally = Tally(f"oracle EQ {fs}")
    n = eq_frames(fs)
    for k, s in enumerate(variant_matrix(fs)):
        if k % 7 and k != len(variant_matrix(fs)) - 1:       # a spread of the matrix is enough on the CPU
            continue
        x = signal(k % 5, n, fs, 300 + k)
        want = np.concatenate([chain.process_chunk(x[b:e], fs, s) for b, e in chunk_bounds(n, fs, 0.6 * n / fs)])
        certify_eq(tally, want, x, fs, s, 0.6 * n / fs, str(s))
    tally.report()
    if fs < 11025:                                             # the 4 kHz high-pass of the crossover needs fs > 8 kHz
        return
    split = Tally(f"oracle band split {fs}")
    pre = signal(4, 2 * design.xover_warm_frames(fs) + 333, fs, 7)
    bands = chain.band_split(pre, fs)
    certify_split(split, bands, pre, fs, None, "")
    split.report()
    _, lo, _ = ref_split(pre, fs, None)
    lo64 = sosfilt(design._xover_sos(fs)[0], pre.astype(np.float64) / 32768, axis=0)
    kpre = signal(4, 3 * chain.samples_in_100ms(fs) + 333, fs, 8)
    want = ref_kw_energies(kpre, fs)
    rel = float((np.abs(ref_kw_energies(kpre, fs, np.float64) - want) / want).max())
    print(f"{fs}: crossover low-pass float64 - long double <= {float(np.abs(lo64 - lo).max()) * 32768:.2e} LSB, "
          f"K energies <= {rel:.2e} relative")
    assert rel < KW_REL / 100


def test_delta_is_far_above_float64_round_off():
    """The float64 deviation of the 250 Hz shelf from the long-double run, measured where it is largest (384 kHz), is
    below DELTA / 100."""
    fs = 384000
    x = chain.to_float(signal(0, 60000, fs, 3))[:, 0]
    b, a = design._shelf_ba(fs, 250, "low")
    dev = np.abs(lfilter(b, a, x) - lfilter(_ld(b), _ld(a), x.astype(LD))).max() * 32768
    print(f"250 Hz shelf at 384 kHz: float64 - long double <= {float(dev):.2e} LSB")
    assert dev < DELTA_LSB / 100


@pytest.fixture(scope="module")
def layout_driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("layout") / "plan_layout_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", os.path.join(ROOT, "tests", "plan_layout_driver.cpp"),
                           "-o", exe])
    return exe


def _layout_rc(driver, tmp_path, settings, fs):
    tracks = (L.TrackParams * 1)()
    tracks[0] = design.track_params(settings, fs, 1000, 0, None, {})
    (tmp_path / "tracks.bin").write_bytes(bytes(tracks))
    (tmp_path / "options.bin").write_bytes(bytes(L.PlanOptions(0, 0, 0, 0, 1, 0, 0, 0)))
    out = subprocess.run([driver, str(tmp_path / "tracks.bin"), str(tmp_path / "options.bin"), "148", "2", "3"],
                         check=True, capture_output=True, text=True).stdout
    lay = json.loads(out)
    return lay["rc"], lay["error"]


@pytest.mark.parametrize("fs", LOW_RATES)
def test_low_rate_stages_rejected(layout_driver, tmp_path, fs):
    """Below 22.05 kHz the 4 kHz peak is not of Butterworth shape (AME_E_UNSUPPORTED); at or below 16 kHz the 8 kHz
    treble shelf, and at or below 24 kHz the 12 kHz warmth shelf, cannot be designed (ValueError).  The stages the
    GPU matrix uses at these rates are accepted."""
    rc, err = _layout_rc(layout_driver, tmp_path, eq_settings(0.0, 0.0, 2.0, 0.0), fs)
    assert rc == AME_E_UNSUPPORTED and err.startswith("track 0: a filter section is not of Butterworth shape"), (rc, err)
    with pytest.raises(ValueError, match="Digital filter critical frequencies"):
        design.track_params(eq_settings(0.0, 0.0, 0.0, 2.0), fs, 1000)
    with pytest.raises(ValueError, match="Digital filter critical frequencies"):
        design.track_params(eq_settings(analog_character=10), fs, 1000)
    for s in variant_matrix(fs):
        assert _layout_rc(layout_driver, tmp_path, s, fs) == (0, ""), s


# ------------------------------------------------------------------------------------------------
# GPU: k_eq
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fs", LOW_RATES + HIGH_RATES)
def test_eq_every_variant(torch_cuda, fs):
    """Every stage in each of its states (bypass / boost / cut, bypass / +gain / -gain), warmth off / on above 24 kHz,
    width 1 / 1.37: one track per configuration, all in one launch.  Tracks are two slowest warm-ups long, with one
    chunk join at an odd frame."""
    from audio_mastering_engine_b200 import MasterPlan
    sets = variant_matrix(fs)
    n = eq_frames(fs)
    chunk = 0.6 * n / fs
    xs = [signal(k % 5, n, fs, 1000 + k) for k in range(len(sets))]
    plan = MasterPlan([n] * len(sets), fs, sets, chunk_seconds=chunk)
    _, _, got = run_eq(torch_cuda, plan, xs)
    plan.close()
    tally = Tally(f"k_eq matrix {fs}")
    for x, s, g in zip(xs, sets, got):
        certify_eq(tally, g, x, fs, s, chunk, str(s))
    tally.report()


TILE_SETS = [eq_settings(3.5, -2.5, 2.0, 4.0, analog_character=40, width=1.2),     # every stage, warmth, width
             eq_settings(-4.5, 0.0, 0.0, -3.5),                                   # both shelves cut: the float32 product
             eq_settings(0.0, 2.5, -5.0, 0.0, width=0.63),                        # peaks only
             eq_settings(0.0, 0.0, 0.0, -3.5, analog_character=75),               # treble cut first, with warmth
             eq_settings(6.0, 0.0, 6.0, 6.0, width=1.9)]                          # boosts past full scale


@pytest.mark.gpu
@pytest.mark.parametrize("tile,halo", [(8, False), (64, False), (520, False), (0, False), (64, True)])
def test_eq_tile_starts_everywhere(torch_cuda, tile, halo):
    """44.1 kHz, 0.37 s chunks (16317 frames: chunk k starts at residue 5k mod 8, every residue over 8 chunks), tiles
    of 8 / 64 / 520 frames and auto, tracks shorter than the warm-up, of 1 to 3 frames, mono, and the same batch
    with time-shard halos in front of every track."""
    from audio_mastering_engine_b200 import MasterPlan, sharding
    fs, chunk = 44100, 0.37
    n_long = 8 * int(chunk * fs) + 1234
    tracks, sets = [], []
    for k, s in enumerate(TILE_SETS):
        tracks.append(signal((0, 4, 2, 3, 4)[k], n_long, fs, 50 + k)); sets.append(s)
    mono = signal(0, n_long, fs, 60)[:, :1]
    tracks.append(np.repeat(mono, 2, axis=1)); sets.append(TILE_SETS[0])
    for k, n in enumerate((1, 2, 3, 100, 1000, 2239, 16318)):
        tracks.append(signal(4, n, fs, 70 + k)); sets.append(TILE_SETS[k % len(TILE_SETS)])
    halos = [sharding.halo_frames(fs)] * len(tracks) if halo else None
    plan = MasterPlan([len(t) for t in tracks], fs, sets, chunk_seconds=chunk, eq_tile_frames=tile, halos=halos)
    _, _, got = run_eq(torch_cuda, plan, tracks)
    plan.close()
    tally = Tally(f"k_eq tiles {tile}{' halo' if halo else ''}")
    for k, (x, s, g) in enumerate(zip(tracks, sets, got)):
        certify_eq(tally, g, x, fs, s, chunk, f"track {k} ({len(x)} frames)")
    tally.report()


@pytest.mark.gpu
@pytest.mark.parametrize("fs", (44100, 48000, 96000))
def test_warmth_exhaustive(torch_cuda, fs):
    """Warmth alone (flat EQ, width 1) for analog_character 1..100: every left value against two permutations of every
    right value.  Exact by design, so bit for bit against oracle.chain.warmth and the lossy converter pair."""
    from audio_mastering_engine_b200 import MasterPlan
    rng = np.random.default_rng(fs)
    allv = np.arange(-32768, 32768, dtype=np.int32).astype(np.int16)
    x = np.stack([np.concatenate([allv, allv]), np.concatenate([rng.permutation(allv), rng.permutation(allv)])], axis=1)
    sets = [eq_settings(analog_character=ac) for ac in range(1, 101)]
    plan = MasterPlan([len(x)] * len(sets), fs, sets, chunk_seconds=None)
    _, _, got = run_eq(torch_cuda, plan, [x] * len(sets))
    plan.close()
    for s, g in zip(sets, got):
        want = chain.to_pcm(chain.to_float(chain.warmth(x, fs, s["analog_character"])))
        assert np.array_equal(g, want), (s["analog_character"], int((g != want).sum()))


@pytest.mark.gpu
def test_width_exhaustive(torch_cuda):
    """Width alone (flat EQ): every left value against 70 right values, among them +-32768, +-32767, +-1 and 0, for
    widths in [0, 2].  float32 by definition, so bit for bit against oracle.chain.width and to_pcm."""
    from audio_mastering_engine_b200 import MasterPlan
    fs = 48000
    rng = np.random.default_rng(11)
    rights = np.concatenate([[-32768, 32767, -32767, 1, -1, 0, 16384, -16384], rng.integers(-32768, 32768, 62)])
    allv = np.arange(-32768, 32768, dtype=np.int32)
    x = np.stack([np.tile(allv, len(rights)), np.repeat(rights, len(allv))], axis=1).astype(np.int16)
    widths = (0.0, 0.37, 0.8, 1.2, 1.93, 2.0)
    sets = [eq_settings(width=w) for w in widths]
    plan = MasterPlan([len(x)] * len(sets), fs, sets, chunk_seconds=None)
    _, _, got = run_eq(torch_cuda, plan, [x] * len(sets))
    plan.close()
    for w, g in zip(widths, got):
        want = chain.to_pcm(chain.width(chain.to_float(x), w))
        assert np.array_equal(g, want), (w, int((g != want).sum()))


# ------------------------------------------------------------------------------------------------
# GPU: k_band_split
# ------------------------------------------------------------------------------------------------
def _split_batch(rates, gaps):
    """One multiband track per rate (two slowest crossover warm-ups + an odd tail), tracks without multiband between."""
    tracks, fss, sets = [], [], []
    for k, fs in enumerate(rates):
        n = 2 * design.xover_warm_frames(fs) + 333 + 2 * k
        s = dict(eq_settings(2.0, 1.0, 1.5 if fs >= 22050 else 0.0, 1.0, analog_character=25 if fs > 24000 else 0),
                 multiband=True, **synth.DEFAULT_MULTIBAND)
        tracks.append(signal(4 if k % 2 else 0, n, fs, 200 + k)); fss.append(fs); sets.append(s)
        if gaps:
            tracks.append(signal(0, 1111 + k, fs, 250 + k)); fss.append(fs); sets.append(eq_settings(1.0))
    return tracks, fss, sets


@pytest.mark.gpu
@pytest.mark.parametrize("tile", (8, 64, 0))
@pytest.mark.parametrize("mixed", (True, False))
def test_band_split_certificate(torch_cuda, tile, mixed):
    """The GPU's own pre signal through stage_band_split: every band sample against the long-double crossover.  A batch of
    every rate from 22.05 to 384 kHz (per-track coefficients, UNI=false) or of one rate (UNI=true), tracks without
    multiband between multiband ones (mb_delta packing), odd chunk lengths."""
    from audio_mastering_engine_b200 import MasterPlan
    rates = HIGH_RATES if mixed else (48000,) * 3
    tracks, fss, sets = _split_batch(rates, gaps=True)
    chunk = 0.61 * min(len(t) / f for t, f in zip(tracks[::2], fss[::2]))
    plan = MasterPlan([len(t) for t in tracks], fss, sets, chunk_seconds=chunk, xover_tile_frames=tile)
    d_in, d_pre, pres = run_eq(torch_cuda, plan, tracks)
    d_bands = torch_cuda.zeros((3, plan.mb_frames, 2), dtype=torch_cuda.int16, device=d_pre.device)
    plan.stage_band_split(d_pre, d_bands)
    torch_cuda.cuda.synchronize()
    bands = d_bands.cpu().numpy()
    tally = Tally(f"k_band_split tile {tile} {'mixed' if mixed else 'one rate'}")
    for t, (pre, fs, s) in enumerate(zip(pres, fss, sets)):
        if not s["multiband"]:
            assert plan.mb_offset(t) == -1
            continue
        o = plan.mb_offset(t)
        certify_split(tally, bands[:, o:o + len(pre)], pre, fs, chunk, f"track {t} at {fs}")
    plan.close()
    tally.report()


# ------------------------------------------------------------------------------------------------
# GPU: K-weighted sub-block energies and the loudness numbers built on them
# ------------------------------------------------------------------------------------------------
KW_RATES = (44100, 88200, 22050, 11025, 48000, 192000, 384000)


def _kw_batch(mixed):
    """(tracks, rates, settings): per rate a 3.5 s track, lengths just under / over a multiple of the sub-block, tracks
    shorter than 100 ms / 400 ms / 3 s, silence, one track without normalisation."""
    rates = KW_RATES if mixed else (44100,) * 4
    tracks, fss, sets = [], [], []
    for k, fs in enumerate(rates):
        s100 = chain.samples_in_100ms(fs)
        lufs = None if k == 2 else -14.0 + k
        st = eq_settings(1.5, 0.0, 0.0, 0.0, lufs=lufs)
        for n, kind in ((35 * s100 + 2 * k + 1, 4), (34 * s100 - 1 - k, 0), (12 * s100 + 3, 3), (4 * s100 - 1, 1),
                        (s100 - 5, 0), (7 * s100 + 1, None)):
            x = np.zeros((n, 2), np.int16) if kind is None else signal(kind, n, fs, 400 + 10 * k + len(tracks))
            tracks.append(x); fss.append(fs); sets.append(st)
    return tracks, fss, sets


def _ulps(a, b, scale):
    return abs(a - b) / np.spacing(scale)


@pytest.mark.gpu
@pytest.mark.parametrize("kw_tile", (1, 3, 0))
@pytest.mark.parametrize("mixed", (True, False))
def test_kweight_energies_and_loudness(torch_cuda, kw_tile, mixed):
    """Sub-block energies of stage_loudness_hist against long-double sums; then, given the GPU's energies, the oracle's
    histogram, gate, loudness range and gain, and stage_apply_gain against chain.apply_static_gain with the GPU's gain."""
    from audio_mastering_engine_b200 import MasterPlan
    torch = torch_cuda
    tracks, fss, sets = _kw_batch(mixed)
    plan = MasterPlan([len(t) for t in tracks], fss, sets, chunk_seconds=0.77, kw_tile_subblocks=kw_tile)
    d_in, d_pre, pres = run_eq(torch, plan, tracks)
    d_hist = torch.zeros((len(tracks), 1000), dtype=torch.int64, device=d_pre.device)
    plan.stage_loudness_hist(d_pre, d_hist)
    n_sb = [len(p) // chain.samples_in_100ms(f) for p, f in zip(pres, fss)]
    energy = plan.read_tap("subblock_energy", max(sum(n_sb), 1), np.float64)
    d_out = torch.zeros_like(d_pre)
    res = plan.stage_apply_gain(d_pre, d_hist, d_out)
    torch.cuda.synchronize()
    hist, outs = d_hist.cpu().numpy(), plan.unpack(d_out.cpu().numpy())
    worst = 0.0
    for t, (pre, fs, s, r, out) in enumerate(zip(pres, fss, sets, res, outs)):
        label = f"track {t} at {fs}, {len(pre)} frames"
        o = plan.subblock_offset(t)
        sub = energy[o:o + n_sb[t]]
        worst = max(worst, check_energies(sub, ref_kw_energies(pre, fs), label))
        s100 = chain.samples_in_100ms(fs)
        n = len(sub)
        blocks = (sub[0:n - 3] + sub[1:n - 2] + sub[2:n - 1] + sub[3:n]) / float(4 * s100) if n >= 4 else np.zeros(0)
        h = chain.block_histogram(blocks)
        assert np.array_equal(hist[t], h), label
        assert r["n_blocks"] == int(h.sum()), label
        want_i, rel = chain.gated_loudness_from_histogram(h)
        assert r["rel_threshold_energy"] == rel, label
        assert r["input_i"] == want_i or _ulps(r["input_i"], want_i, 100.0) <= 4, (label, r["input_i"], want_i)
        thresh = 10.0 * math.log10(rel) - 0.691 if h.sum() else -70.0
        assert _ulps(r["input_thresh"], thresh, 100.0) <= 4, (label, r["input_thresh"], thresh)
        lra = chain.loudness_range_from_histogram(chain.short_term_histogram(sub, fs))
        assert _ulps(r["input_lra"], lra, 100.0) <= 4, (label, r["input_lra"], lra)
        assert r["sample_peak"] == (int(np.abs(pre.astype(np.int32)).max()) if len(pre) else 0), label
        assert r["normalized"] == (s["lufs"] is not None and want_i != -math.inf), label
        if r["normalized"]:
            gain, mi = chain.static_gain_from_measured(want_i, s["lufs"])
            if r["measured_i_2dp"] != mi:      # '%.2f' of glibc against rint(x * 100) / 100: only at a rounding tie
                tie = math.floor(want_i * 100) + 0.5
                assert abs(want_i * 100 - tie) <= 4 * np.spacing(10000.0), (label, r["measured_i_2dp"], mi)
                gain = math.pow(10.0, (s["lufs"] - r["measured_i_2dp"]) / 20.0)
            assert _ulps(r["gain"], gain, gain) <= 4, (label, r["gain"], gain)
        assert np.array_equal(out, chain.apply_static_gain(pre, r["gain"])), label
    plan.close()
    print(f"k_kweight_energy tile {kw_tile} {'mixed' if mixed else 'one rate'}: largest relative energy error {worst:.2e}")
