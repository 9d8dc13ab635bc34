"""The multiband compressor held to pydub bit for bit, on band signals built to hit its edges.

Given the same int16 bands, k_window_flag -> k_tile_prefix -> k_compact -> k_att_chain -> k_compress_apply must give
what pydub's compress_dynamic_range + overlay give (oracle.cport, tied to audioop by oracle.chain): DESIGN.md section 6
allows one exception only, a floor that flips where CUDA exp10 and glibc pow differ in the last bit of the gain, i.e.
where x * 10 ** (-att / 20) lies within 1e-9 of an integer.

audioop.mul floors, so any non-zero attenuation lowers a positive sample by at least 1 LSB: on positive plateaus the
output shows exactly which frames carry an attenuation.  A frame flagged by mistake (rms <= thresh_rms, M = 0) changes
no sample, so the number of flagged frames is checked too: ame_plan_chain_stats reports it per chain, and it must equal
the number of frames whose window rms exceeds thresh_rms.

The CPU part checks the host-built attenuation table (build_att_table, through tests/att_table_driver.cpp) and the
thr_i / look / table fields of the job tables (through tests/plan_layout_driver.cpp) without a GPU."""
import json
import math
import os
import subprocess

import numpy as np
import pytest

from audio_mastering_engine_b200 import _lib as L, design
from oracle import chain, cport

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATES = (22050, 44100, 48000, 96000, 192000, 384000)
# -6.0206... and -30.3089... give thresh_rms of exactly 16384.0 and 1000.0; +6.1 dB is past the 65535 sentinel
THRESHOLDS = (-40.0, -36.0, -20.0, -0.1, 0.0, -6.020599913279624, -30.30899869919436, 6.1)
RATIOS = (1.0, 1.5, 4.0, 10.0)
THR_NEVER = 0x7fffffff         # thr_i of a band whose thresh_rms >= 65535 (build_layout)
AME_E_UNSUPPORTED = -4         # include/ame.h


def _compile(tmp_path_factory, name):
    exe = str(tmp_path_factory.mktemp(name) / name)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", os.path.join(ROOT, "tests", name + ".cpp"), "-o", exe])
    return exe


def mb_settings(low, mid, high):
    """Multiband settings with (threshold dB, ratio) per band and nothing else."""
    s = dict(multiband=True, lufs=None)
    for name, (thr, ratio) in zip(("low", "mid", "high"), (low, mid, high)):
        s[name + "_thresh"], s[name + "_ratio"] = thr, ratio
    return s


def expected_thr_i(thresh_rms):
    return THR_NEVER if thresh_rms >= 65535.0 else math.floor(thresh_rms) + 1


# ------------------------------------------------------------------------------------------------
# CPU: the attenuation table and the job tables
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def att_driver(tmp_path_factory):
    return _compile(tmp_path_factory, "att_table_driver")


@pytest.fixture(scope="module")
def layout_driver(tmp_path_factory):
    return _compile(tmp_path_factory, "plan_layout_driver")


ATT_ENTRY = np.dtype([("m", "<f8"), ("inc", "<f8"), ("dec", "<f8"), ("tau", "<f8")])


def test_att_table_bit_for_bit(att_driver, tmp_path):
    """build_att_table against oracle.chain.max_attenuation_for_rms, m / attack_frames and m / release_frames, every
    entry, bit for bit; tau by its definition: the smallest a >= 0 with fl(a + inc) >= m."""
    grid = []
    for fs in RATES:
        for thr in THRESHOLDS:
            for ratio in RATIOS:
                cb = design.track_params(mb_settings(*[(thr, ratio)] * 3), fs, 1000).comp[0]
                grid.append((fs, thr, ratio, cb))
    args = []
    for _, _, _, cb in grid:
        args += [float(cb.thresh_rms).hex(), float(cb.coef).hex(), float(cb.attack_frames).hex(), float(cb.release_frames).hex()]
    out = tmp_path / "att.bin"
    subprocess.check_call([att_driver, str(out)] + args)
    tables = np.fromfile(out, dtype=ATT_ENTRY).reshape(len(grid), 32769)
    rms = np.arange(32769)
    m_cache = {}
    for k, (fs, thr, ratio, cb) in enumerate(grid):
        thresh_rms, look, attack_frames, release_frames = chain.compressor_constants(fs, thr, ratio)
        assert (cb.thresh_rms, cb.attack_frames, cb.release_frames, cb.look_frames) == (thresh_rms, attack_frames, release_frames, look)
        if (thr, ratio) not in m_cache:
            m_cache[thr, ratio] = np.array([chain.max_attenuation_for_rms(r, thresh_rms, ratio) for r in range(32769)])
        m = m_cache[thr, ratio]
        e = tables[k]
        label = (fs, thr, ratio)
        assert np.array_equal(e["m"].view(np.int64), m.view(np.int64)), label
        assert np.array_equal(e["inc"].view(np.int64), (m / attack_frames).view(np.int64)), label
        assert np.array_equal(e["dec"].view(np.int64), (m / release_frames).view(np.int64)), label
        tau, inc = e["tau"], e["inc"]
        assert np.all(tau >= 0) and np.all(tau + inc >= m), label
        below = np.nextafter(tau, -np.inf)
        assert np.all((tau == 0) | (below + inc < m)), label
        if thresh_rms >= 32768.0 or ratio == 1.0:
            assert not e["m"].any(), label                    # nothing above threshold, or coef = 0
        else:
            over = rms > thresh_rms
            assert np.all(e["m"][over] > 0) and not e["m"][~over].any(), label


def _layout(driver, tmp_path, tracks):
    (tmp_path / "tracks.bin").write_bytes(bytes(tracks))
    (tmp_path / "options.bin").write_bytes(bytes(L.PlanOptions(0, 0, 0, 0, 1, 0, 0, 0)))
    out = subprocess.run([driver, str(tmp_path / "tracks.bin"), str(tmp_path / "options.bin"), "148", "2", "3"],
                         check=True, capture_output=True, text=True).stdout
    lay = json.loads(out)
    assert lay["rc"] == 0, lay["error"]
    return lay


def test_job_tables_thr_i_look_and_tables(layout_driver, tmp_path):
    """Every chain row carries thr_i = the smallest integer > thresh_rms (the sentinel from 65535 up) and look =
    int(5 * fs / 1000); bands share an attenuation table exactly when (thresh_rms, coef, attack, release) agree - the
    same threshold at two rates must not."""
    specs = []
    for i, fs in enumerate(RATES + (352800,)):
        for j in range(0, len(THRESHOLDS), 3):
            th = [THRESHOLDS[(j + b) % len(THRESHOLDS)] for b in range(3)]
            specs.append((fs, mb_settings(*[(t, RATIOS[(i + j + b) % len(RATIOS)]) for b, t in enumerate(th)]), 700 + 37 * j))
        specs.append((fs, dict(lufs=None), 300))                  # a track without the compressor in between
    arr = (L.TrackParams * len(specs))()
    off = 0
    for k, (fs, s, n) in enumerate(specs):
        arr[k] = design.track_params(s, fs, n, off, 0.004)    # a few chunks per track
        off += (n + 7) // 8 * 8
    lay = _layout(layout_driver, tmp_path, arr)
    mb_off = lay["mb_offset"]
    keys = {}
    n_rows = 0
    for row in lay["chain"]:
        mb_begin, n, _, band, table, thr_i, look = row[:7]
        t = max(k for k in range(len(specs)) if 0 <= mb_off[k] <= mb_begin)
        fs, s, _ = specs[t]
        name = ("low", "mid", "high")[band]
        thresh_rms, look_ref, attack_frames, release_frames = chain.compressor_constants(fs, s[name + "_thresh"], s[name + "_ratio"])
        assert thr_i == expected_thr_i(thresh_rms), (fs, s[name + "_thresh"], thr_i)
        assert look == look_ref == int(5 * fs / 1000), (fs, look)
        key = (thresh_rms, 1 - 1.0 / s[name + "_ratio"], attack_frames, release_frames)
        assert keys.setdefault(key, table) == table
        n_rows += 1
    assert len(set(keys.values())) == len(keys) == lay["scalars"]["n_att_tables"]
    assert n_rows == 3 * sum(math.ceil(n / int(0.004 * fs)) for fs, s, n in specs if s.get("multiband"))


def test_ratio_below_one_is_rejected(layout_driver, tmp_path):
    """ratio < 1 makes max_attenuation negative (the settings dict accepts it, the GUI does not offer it): k_att_chain
    orders attenuations by their bit patterns and shifts parked segments by whole ulps, which needs non-negative
    operands, so the plan refuses such a band instead of computing something unchecked."""
    for ratio in (0.5, 0.999):
        arr = (L.TrackParams * 2)()
        arr[0] = design.track_params(dict(lufs=None), 48000, 1000, 0)
        arr[1] = design.track_params(mb_settings((-20.0, 4.0), (-30.0, ratio), (-20.0, 1.0)), 48000, 1000, 1000)
        (tmp_path / "tracks.bin").write_bytes(bytes(arr))
        (tmp_path / "options.bin").write_bytes(bytes(L.PlanOptions(0, 0, 0, 0, 1, 0, 0, 0)))
        lay = json.loads(subprocess.run([layout_driver, str(tmp_path / "tracks.bin"), str(tmp_path / "options.bin"), "148", "2", "3"],
                                        check=True, capture_output=True, text=True).stdout)
        assert lay["rc"] == AME_E_UNSUPPORTED and lay["error"].startswith("track 1: compressor band 1 has a ratio below 1"), lay
    arr[1] = design.track_params(mb_settings((-20.0, 4.0), (-30.0, 1.0), (-20.0, 1.0)), 48000, 1000, 1000)
    assert _layout(layout_driver, tmp_path, arr)["rc"] == 0     # ratio 1 (coef 0) stays valid


def test_thr_i_at_integer_thresholds():
    """The thresholds the GPU cases rely on land where they should: an integer thresh_rms gets thr_i = thresh_rms + 1."""
    assert chain.compressor_constants(48000, -6.020599913279624, 2)[0] == 16384.0
    assert chain.compressor_constants(48000, -30.30899869919436, 2)[0] == 1000.0
    assert expected_thr_i(16384.0) == 16385 and expected_thr_i(1000.0) == 1001 and expected_thr_i(327.68) == 328
    assert expected_thr_i(chain.compressor_constants(48000, -0.0001, 2)[0]) == 32768
    assert expected_thr_i(chain.compressor_constants(48000, 0.0, 2)[0]) == 32769
    assert expected_thr_i(chain.compressor_constants(48000, 6.1, 2)[0]) == THR_NEVER


# ------------------------------------------------------------------------------------------------
# GPU: crafted bands through ame_stage_compress
# ------------------------------------------------------------------------------------------------
SENTINEL = -12345      # d_pre outside the multiband tracks must keep it
JUNK = 32767           # multiband packing padding: a kernel that reads past a chain sees full scale


@pytest.fixture(scope="module")
def torch_cuda():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


class Track:
    """One track of a batch: bands (3, n, 2) int16 with settings, or a plain track of n frames (no multiband)."""

    def __init__(self, fs, settings=None, bands=None, n=None, py=False):
        self.fs, self.bands, self.py = fs, bands, py
        self.settings = settings if bands is not None else dict(lufs=None)
        self.n = bands.shape[1] if bands is not None else n


def band_track(fs, settings, *bands, py=False):
    """A track from up to three band signals ((n, 2) int16, None = silent), padded with zeros to the longest."""
    n = max(len(b) for b in bands if b is not None)
    out = np.zeros((3, n, 2), dtype=np.int16)
    for k, b in enumerate(bands):
        if b is not None:
            out[k, :len(b)] = b
    return Track(fs, settings, out, py=py)


def expected(tr, chunk_seconds):
    """(output, near-integer mask, flagged frames per chain) of one multiband track, chunk by chunk, from the oracle."""
    fs, s, n = tr.fs, tr.settings, tr.n
    cf = int(chunk_seconds * fs) if chunk_seconds else n
    out = np.empty((n, 2), dtype=np.int16)
    near = np.zeros((n, 2), dtype=bool)
    steps = []
    for c0 in range(0, n, cf):
        c1 = min(c0 + cf, n)
        comp = []
        for b, name in enumerate(("low", "mid", "high")):
            thr, ratio = s[name + "_thresh"], s[name + "_ratio"]
            x = tr.bands[b, c0:c1]
            y, att = cport.compress(x, fs, thr, ratio, return_att=True)
            if tr.py:                                       # cport is audioop's twin: check it on this one
                y2, att2 = chain.compress_dynamic_range_py(x, fs, thr, ratio, return_att=True)
                assert np.array_equal(y, y2) and np.array_equal(att, att2)
            comp.append(y)
            p = x.astype(np.float64) * (10.0 ** (-att / 20))[:, None]
            near[c0:c1] |= (att != 0)[:, None] & (x != 0) & (np.abs(p - np.round(p)) < 1e-9)
            thresh_rms, look, _, _ = chain.compressor_constants(fs, thr, ratio)
            steps.append(int(np.count_nonzero(cport.window_rms(x, look) > thresh_rms)))
        out[c0:c1] = chain.overlay(chain.overlay(comp[0], comp[1]), comp[2])
    return out, near, steps


def new_plan(tracks, chunk_seconds=None, chain_warps=0):
    from audio_mastering_engine_b200 import MasterPlan
    return MasterPlan([t.n for t in tracks], [t.fs for t in tracks], [t.settings for t in tracks],
                      chunk_seconds=chunk_seconds, chain_warps=chain_warps)


def stage(torch, plan, tracks):
    """Bands into a (3, mb_frames, 2) tensor at mb_offset(t), junk in the padding, d_pre full of the sentinel; one
    stage_compress.  Returns (d_pre as numpy, chain_stats())."""
    dev = torch.device("cuda", plan.device)
    h = np.full((3, max(plan.mb_frames, 1), 2), JUNK, dtype=np.int16)
    for k, t in enumerate(tracks):
        if t.bands is not None:
            off = plan.mb_offset(k)
            h[:, off:off + t.n] = t.bands
    d_bands = torch.from_numpy(h).to(dev)
    d_pre = torch.full((plan.total_frames, 2), SENTINEL, dtype=torch.int16, device=dev)
    plan.stage_compress(d_bands, d_pre)
    torch.cuda.synchronize(dev)
    return d_pre.cpu().numpy(), plan.chain_stats()


def check(torch, tracks, chunk_seconds=None, chain_warps=0, plan=None, label=""):
    """Runs the batch (on `plan` if given) and holds it to the oracle.  Returns chain_stats()."""
    own = plan is None
    plan = new_plan(tracks, chunk_seconds, chain_warps) if own else plan
    try:
        pre, stats = stage(torch, plan, tracks)
        offsets = plan.offsets
    finally:
        if own:
            plan.close()
    untouched = np.ones(len(pre), dtype=bool)
    steps, exceptions = [], 0
    for k, (t, off) in enumerate(zip(tracks, offsets)):
        if t.bands is None:
            continue
        want, near, st = expected(t, chunk_seconds)
        steps += st
        got = pre[off:off + t.n]
        diff = got != want
        assert not np.any(diff & ~near), (label, k, np.argwhere(diff & ~near)[:8].tolist(),
                                          got[diff.any(axis=1)][:4].tolist(), want[diff.any(axis=1)][:4].tolist())
        exceptions += int(np.count_nonzero(diff))
        untouched[off:off + t.n] = False
    assert np.all(pre[untouched] == SENTINEL), (label, np.flatnonzero(np.any(pre[untouched] != SENTINEL, axis=1))[:8])
    print(f"{label}: {len(steps)} chains, {sum(steps)} flagged frames, near-integer exceptions used: {exceptions}, "
          f"chain_stats {stats}")
    assert stats["chains"] == len(steps), (label, stats, len(steps))
    assert stats["steps"] == sum(steps) and stats["max_steps"] == max(steps), (label, stats, sum(steps), max(steps))
    return stats


def plateau(n, *spans):
    """(n, 2) int16: zeros, and (l, r) over each [begin, end)."""
    x = np.zeros((n, 2), dtype=np.int16)
    for b, e, lv, rv in spans:
        x[b:e] = (lv, rv)
    return x


def noise(n, amp, seed, positive_bias=0):
    rng = np.random.default_rng(seed)
    env = amp * (0.3 + 0.7 * np.abs(np.sin(np.linspace(0, 7.0, n))))[:, None]
    return np.clip(rng.standard_normal((n, 2)) * env + positive_bias, -32768, 32767).astype(np.int16)


def edge_bands(fs):
    """(settings of the band, signal) pairs that sit on the compressor's edges; look = 240 at 48 kHz."""
    look = int(5 * fs / 1000)
    t40, t16k, t1000 = -40.0, -6.020599913279624, -30.30899869919436     # thresh_rms 327.68, 16384.0, 1000.0
    out = [
        # window rms exactly thr_i (flagged) and thr_i - 1 (not), plateaus of both signs
        ((t40, 4.0), plateau(3300, (300, 1300, 328, 328), (1800, 2800, -328, 328), (2900, 3250, -328, -328))),
        ((t40, 4.0), plateau(3300, (300, 1300, 327, 327), (1800, 2800, 327, -327))),
        ((t16k, 2.0), plateau(3300, (300, 1300, 16385, 16385), (1800, 2800, 16384, 16384))),
        ((t16k, 10.0), plateau(3300, (300, 1300, 16384, -16384), (1800, 2800, 16385, -16385))),
        # a plateau from chunk frame 0: the first look frames see windows of 1 ... look - 1 frames
        ((t40, 4.0), plateau(1200, (0, 600, 1000, 1000))),
        ((t1000, 3.0), plateau(1200, (0, 1, 30000, 30000), (1, 1200, 100, 100))),
        ((t1000, 3.0), plateau(1200, (0, 1200, 100, 100), (1, 2, 30000, -30000))),
    ]
    for pos in (look - 1, look, look + 1):                 # single loud frames on a positive bed
        x = plateau(1200, (0, 1200, 100, 100), (pos, pos + 1, 30000, 30000))
        out.append(((t1000, 3.0), x))
    # full scale: rms 32768 (the last table entry) just below 0 dBFS (thr_i = 32768), at 0 dBFS (never flagged) and past
    # the 65535 sentinel; +32767 after the -32768 window shows the attenuation
    fsig = plateau(2000, (300, 800, -32768, -32768), (800, 1300, 32767, 32767), (1300, 1400, -32768, 32767))
    out += [((-0.0001, 4.0), fsig), ((0.0, 4.0), fsig), ((6.1, 4.0), fsig), ((10.0, 10.0), noise(2000, 20000, 3))]
    # flag density: every window flagged at -100 dB (whole 2048-frame tiles), none at all, 1 / 63 / 64 / 65 frames
    out += [((-100.0, 4.0), noise(9000, 2000, 4)), ((t40, 4.0), noise(3000, 60, 5, positive_bias=40))]
    for k in (1, 63, 64, 65):
        out.append(((t40, 4.0), plateau(1200, (500, 500 + look + k - 1, 328, 328))))
    return out


def saturation_bands(n=2000):
    """Triples (low, mid, high) where the order of the two saturating adds matters, loud enough before them to keep
    an attenuation in force."""
    lo, mi, hi = (np.zeros((n, 2), dtype=np.int16) for _ in range(3))
    lo[:1000], mi[:1000], hi[:1000] = 20000, 20000, -20000
    triples = [(32767, 32767, -32768), (-32768, -32768, 32767), (32767, 1000, -2000), (-32768, -1000, 2000),
               (32767, 32767, 32767), (-32768, -32768, -32768)]
    for i in range(1000, n):
        a, b = triples[i % len(triples)], triples[(i + 1) % len(triples)]
        lo[i], mi[i], hi[i] = (a[0], b[0]), (a[1], b[1]), (a[2], b[2])
    return lo, mi, hi


@pytest.mark.gpu
def test_edges_one_band_at_a_time_and_together(torch_cuda):
    """Threshold, partial-window, full-scale, sentinel and flag-density edges, each alone in one band (the other two
    silent) and three at a time, with tracks that have no compressor in between; the overlay's saturation order with
    and without an attenuation in force."""
    fs = 48000
    edges = edge_bands(fs)
    tracks = []
    for i, (st, x) in enumerate(edges):                    # band isolation: low, mid, high in turn
        b = i % 3
        bands = [None, None, None]
        bands[b] = x
        prm = [(-20.0, 2.0)] * 3
        prm[b] = st
        tracks.append(band_track(fs, mb_settings(*prm), *bands, py=(i == 4)))
        if i % 5 == 2:
            tracks.append(Track(fs, n=777 + i))
    for i in range(0, len(edges) - 2, 3):                  # all three bands busy
        (s0, x0), (s1, x1), (s2, x2) = edges[i:i + 3]
        tracks.append(band_track(fs, mb_settings(s0, s1, s2), x0, x1, x2))
    for ratio in (1.0, 1.05):
        tracks.append(band_track(fs, mb_settings(*[(-40.0, ratio)] * 3), *saturation_bands()))
    # the crafted counts are what the oracle counts
    look = int(5 * fs / 1000)
    for k, (st, x) in zip((1, 63, 64, 65), edges[-4:]):
        thresh_rms = chain.compressor_constants(fs, *st)[0]
        assert np.count_nonzero(cport.window_rms(x, look) > thresh_rms) == k
    check(torch_cuda, tracks, label="edges")


@pytest.mark.gpu
def test_chunk_lengths_below_look_and_around_the_granules(torch_cuda):
    """One chunk per track of 1 ... 5 * 2048 + 1 frames at 48 and 192 kHz (look 240 / 960: the short ones are all partial
    windows), and a 30 s chain of 704 window-flag tiles (k_tile_prefix loops over 256-tile rounds) flagged throughout."""
    lengths = [1, 7, 8, 31, 32, 33, 255, 256, 257, 2047, 2048, 2049, 3 * 2048 - 1, 3 * 2048 + 1, 5 * 2048 - 1, 5 * 2048 + 1]
    settings = mb_settings((-30.0, 4.0), (-20.0, 2.0), (-40.0, 8.0))
    tracks = []
    for fs in (48000, 192000):
        for k, n in enumerate(lengths):
            seed = 10 * k + fs // 48000
            tracks.append(band_track(fs, settings, noise(n, 3000, seed), noise(n, 9000, seed + 1, 500), noise(n, 800, seed + 2, 100)))
            if k % 4 == 3:
                tracks.append(Track(fs, n=100 + k))
    n = 30 * 48000
    tracks.append(band_track(48000, mb_settings((-100.0, 4.0), (-30.0, 4.0), (-36.0, 2.0)),
                             noise(n, 4000, 71), noise(n, 2000, 72, 300), noise(n, 500, 73)))
    check(torch_cuda, tracks, label="lengths")


@pytest.mark.gpu
def test_chunk_starts_on_every_alignment(torch_cuda):
    """0.5 s chunks: 11025 frames at 22.05 kHz put the chunk starts of the multiband packing on every residue mod 8
    (the scalar paths of load8, list_load and the attenuation stores), 22050 at 44.1 kHz on even ones."""
    settings = mb_settings((-30.0, 4.0), (-24.0, 2.0), (-36.0, 8.0))
    tracks = []
    for k, (fs, secs) in enumerate(((22050, 4.7), (44100, 2.3), (48000, 1.6), (22050, 0.9))):
        n = int(secs * fs)
        tracks.append(band_track(fs, settings, noise(n, 4000, 40 + k), noise(n, 6000, 50 + k, 200), noise(n, 3000, 60 + k, 50)))
        tracks.append(Track(fs, n=1003 + k))
    check(torch_cuda, tracks, chunk_seconds=0.5, label="alignment")


@pytest.mark.gpu
def test_sample_rates_to_384k(torch_cuda):
    """22.05 ... 384 kHz in one launch (look 110 ... 1920, so isqrt_ratio runs with n = 2 look up to 3840): the same
    thresholds at every rate, each rate its own tables, two tracks at 48 kHz sharing theirs."""
    settings = mb_settings((-30.0, 4.0), (-20.0, 2.0), (-40.0, 8.0))
    tracks = []
    for k, fs in enumerate((22050, 44100, 48000, 96000, 192000, 352800, 384000, 48000)):
        n = int(0.25 * fs) + 3 * k
        x = noise(n, 5000, 80 + k, 200)
        x[n // 3:n // 3 + 3000] = -32768                 # rms 32768 windows at every rate
        tracks.append(band_track(fs, settings, x, noise(n, 9000, 90 + k, 300), noise(n, 700, 100 + k, 20)))
    check(torch_cuda, tracks, label="rates")


def held_signal(fs=48000):
    """test_compressor_kernels_agree's loud burst followed by a bed just above threshold: the attenuation stays parked
    above max_attenuation and never clamps again, so every k_att_chain segment has to be repaired."""
    rng = np.random.default_rng(7)
    n = 6 * fs + 1237
    t = np.arange(n) / fs
    bed = 0.02 * np.sin(2 * np.pi * 440.0 * t) + 0.002 * rng.standard_normal(n)
    burst = np.where(t < 0.2, 0.9 * np.sin(2 * np.pi * 330.0 * t), 0.0)
    return np.clip(np.stack([bed + burst, bed - burst], axis=1) * 32767, -32767, 32767).astype(np.int16)


@pytest.mark.gpu
@pytest.mark.parametrize("chain_warps", [-1, 0, 1, 3, 8])
def test_parked_chain_every_lane_count(torch_cuda, chain_warps):
    """The parked signal in one band: equal to the oracle for every lane count, with repair passes whenever there is more
    than one lane, and one pass with the sequential loop."""
    fs = 48000
    x = held_signal(fs)
    tracks = [band_track(fs, mb_settings((-38.0, 8.0), (-20.0, 2.0), (-20.0, 2.0)), x, None, None),
              band_track(fs, mb_settings((-20.0, 2.0), (-38.0, 8.0), (-20.0, 2.0)), noise(30000, 3000, 9), x[:200000], None)]
    stats = check(torch_cuda, tracks, chain_warps=chain_warps, label=f"parked chain_warps={chain_warps}")
    if chain_warps < 0:
        assert stats["max_passes"] == 1, stats
    else:
        assert stats["max_passes"] > 1, stats


@pytest.mark.gpu
def test_second_call_on_dirty_workspace(torch_cuda):
    """A densely flagged call, then a sparse one on the same plan: the second sees the first's rms / list / att / grp /
    tile_cnt buffers and must give what a fresh plan gives, chain statistics included."""
    fs = 48000
    settings = mb_settings((-40.0, 4.0), (-30.0, 2.0), (-36.0, 8.0))
    lens = (20000, 33333, 4097)
    dense = [band_track(fs, settings, noise(n, 12000, 200 + k), noise(n, 9000, 210 + k, 500), noise(n, 6000, 220 + k))
             for k, n in enumerate(lens)]
    sparse = []
    for k, n in enumerate(lens):
        x = noise(n, 40, 230 + k, 20)
        x[n // 2:n // 2 + 300] = 9000
        sparse.append(band_track(fs, settings, x, noise(n, 30, 240 + k, 30), np.zeros((n, 2), np.int16)))
    plan = new_plan(dense)
    try:
        check(torch_cuda, dense, plan=plan, label="dense")
        again = check(torch_cuda, sparse, plan=plan, label="sparse after dense")
    finally:
        plan.close()
    assert again == check(torch_cuda, sparse, label="sparse, fresh plan")
