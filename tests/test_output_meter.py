"""The EBU R128 output meter (AME_F_MEASURE_OUTPUT, ame_loudness): loudnorm's second-pass output_* report of the mastered
output, and the stand-alone meter (ame_measure_loudness / measure_loudness) over any buffer.

CPU: the ABI mirror, the settings flag, and the meter's part of the plan layout (tests/meter_layout_driver.cpp, g++ alone).
GPU: the meter against the input side (bit for bit where the output IS the pre-normalisation signal), against the oracle,
and through every layer that carries it: MasterPlan, master(), measure_loudness(), the drop-in entry point and the
time-sharded path."""
import ctypes
import json
import math
import os
import re
import subprocess

import numpy as np
import pytest

from audio_mastering_engine_b200 import _lib as L, design, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_SM, OCC_EQ, OCC_SPLIT = 148, 2, 3             # a B200 (see test_plan_layout.py)
AME_E_INVALID, AME_E_UNSUPPORTED = -1, -4
LUFS_TOL = 0.01


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from audio_mastering_engine_b200 import build
    build.build()
    return L.load()


def test_loudness_struct_and_symbols(lib):
    assert lib.ame_sizeof_loudness() == ctypes.sizeof(L.Loudness) == 64
    for name in ("ame_sizeof_loudness", "ame_measure_loudness", "ame_plan_output_loudness"):
        assert name in L.SYMBOLS and hasattr(lib, name)
    header = open(os.path.join(ROOT, "include", "ame.h")).read()
    assert re.search(r"#define AME_F_MEASURE_OUTPUT 64u", header) and L.AME_F_MEASURE_OUTPUT == 64
    assert re.search(r"#define AME_N_KERNELS 12\b", header) and lib.ame_abi_version() == 5


def test_flag_is_set_by_measure_output_only():
    base = dict(synth.c2_settings(), limiter=True, true_peak=True)
    for s, want in ((base, False), (dict(base, measure_output=True), True), (dict(base, measure_output=1), True),
                    (dict(base, measure_output=False), False), (dict(base, measure_output=None), False),
                    ({"lufs": None, "measure_output": True}, True), ({"lufs": None}, False)):
        p = design.track_params(s, 48000, 1000, 0, 30, {})
        assert bool(p.flags & L.AME_F_MEASURE_OUTPUT) == want, s
        q = design.track_params({k: v for k, v in s.items() if k != "measure_output"}, 48000, 1000, 0, 30, {})
        assert p.flags & ~L.AME_F_MEASURE_OUTPUT == q.flags          # nothing else changes


def _compile(tmp_path_factory, name):
    exe = str(tmp_path_factory.mktemp(name) / name)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", os.path.join(ROOT, "tests", name + ".cpp"), "-o", exe])
    return exe


@pytest.fixture(scope="module")
def meter_driver(tmp_path_factory):
    return _compile(tmp_path_factory, "meter_layout_driver")


@pytest.fixture(scope="module")
def plan_driver(tmp_path_factory):
    return _compile(tmp_path_factory, "plan_layout_driver")


def make_tracks(specs, chunk_seconds=30):
    """specs: (seconds, fs, settings[, halo_frames]) per track, packed as MasterPlan packs them."""
    arr = (L.TrackParams * len(specs))()
    lut, off = {}, 0
    for i, spec in enumerate(specs):
        secs, fs, s = spec[:3]
        halo = spec[3] if len(spec) > 3 else 0
        n = int(round(secs * fs))
        arr[i] = design.track_params(s, fs, n, off, chunk_seconds, lut, halo)
        off += (n + halo + 7) // 8 * 8
    return arr


def run(driver, tmp_path, tracks, n_waves=1, n_slots=0, kw_tile=0, raw=False):
    (tmp_path / "tracks.bin").write_bytes(bytes(tracks))
    (tmp_path / "options.bin").write_bytes(bytes(L.PlanOptions(0, 0, kw_tile, 0, n_waves, 0, n_slots, 0)))
    out = subprocess.run([driver, str(tmp_path / "tracks.bin"), str(tmp_path / "options.bin"), str(N_SM), str(OCC_EQ), str(OCC_SPLIT)],
                         check=True, capture_output=True, text=True).stdout
    return out if raw else json.loads(out)


def meter_batch(flags):
    """Mixed rates, multiband and plain tracks, short ones; flags[i] says whether track i carries the meter."""
    c1, c2 = synth.c1_settings(), synth.c2_settings()
    specs = [(40.0, 44100, c2), (7.0, 48000, c1), (65.0, 96000, c2), (20.0, 192000, c1), (0.3, 44100, dict(c2, limiter=True)),
             (2.5, 48000, {"lufs": -14.0}), (12.0, 96000, dict(c1, limiter=True, true_peak=True)), (0.0004, 48000, c2)]
    return [(secs, fs, dict(s, measure_output=True) if f else s) for (secs, fs, s), f in zip(specs, flags)]


@pytest.mark.parametrize("n_waves,n_slots,kw_tile", [(1, 1, 0), (3, 2, 0), (3, 1, 5), (8, 4, 0)])
@pytest.mark.parametrize("flags", [[1] * 8, [1, 0, 0, 1, 1, 0, 1, 0], [0, 0, 0, 0, 0, 0, 0, 1]])
def test_meter_jobs_cover_flagged_tracks(meter_driver, tmp_path, n_waves, n_slots, kw_tile, flags):
    tracks = make_tracks(meter_batch(flags))
    lay = run(meter_driver, tmp_path, tracks, n_waves, n_slots, kw_tile)
    assert lay["rc"] == 0, lay["error"]
    sc, tdev, mtdev = lay["scalars"], lay["tdev"], lay["meter_tdev"]
    assert sc["any_meter"] == 1
    flagged = [t for t in range(len(tracks)) if flags[t]]
    assert lay["meter_tracks"] == flagged
    # the flagged tracks' sub-blocks, packed one after the other in the meter's own energy array
    pos = 0
    for t in range(len(tracks)):
        assert mtdev[t][1:] == tdev[t][1:]
        assert mtdev[t][0] == pos
        pos += tdev[t][1] if flags[t] else 0
    assert sc["meter_sb_total"] == pos
    pos = {"kw": 0, "peak": 0, "tracks": 0}
    for w in lay["waves"]:
        t_lo, t_hi, kw_uni, kw_n, mkw_lo, mkw_n, mpk_lo, mpk_n, mtr_lo, mtr_n = w
        assert (mkw_lo, mpk_lo, mtr_lo) == (pos["kw"], pos["peak"], pos["tracks"])
        pos["kw"] += mkw_n; pos["peak"] += mpk_n; pos["tracks"] += mtr_n
        mine = [t for t in range(t_lo, t_hi) if flags[t]]
        assert lay["meter_tracks"][mtr_lo:mtr_lo + mtr_n] == mine
        kw, peak = lay["meter_kw"][mkw_lo:mkw_lo + mkw_n], lay["meter_peak"][mpk_lo:mpk_lo + mpk_n]
        assert all(r[0] in mine for r in kw) and all(r[2] in mine for r in peak)
        assert mkw_n <= kw_n
        if kw_uni:                                   # the wave's uniform K filter holds for its flagged tracks too
            assert len({tracks[t].sample_rate for t in mine} | {tracks[t].sample_rate for t in range(t_lo, t_hi)}) == 1
        for t in mine:
            tp = tracks[t]
            # K-weighting: kw_tile_sb sub-blocks per job, exactly the track's complete sub-blocks, in order
            rows = [r[1:] for r in kw if r[0] == t]
            tile = sc["kw_tile_sb"]
            assert rows == [[b, min(b + tile, tdev[t][1])] for b in range(0, tdev[t][1], tile)]
            # peak tiles: exactly the track's frames, 32768 at a time (the k_apply_gain tiles)
            rows = [r[:2] for r in peak if r[2] == t]
            assert rows == [[tp.offset_frames + b, tp.offset_frames + min(b + 32768, tp.n_frames)] for b in range(0, tp.n_frames, 32768)]
    assert pos == {"kw": len(lay["meter_kw"]), "peak": len(lay["meter_peak"]), "tracks": len(lay["meter_tracks"])}


@pytest.mark.parametrize("n_waves,n_slots", [(1, 1), (3, 2)])
def test_batch_without_the_flag_has_no_meter_and_the_same_tables(meter_driver, plan_driver, tmp_path, n_waves, n_slots):
    plain = make_tracks(meter_batch([0] * 8))
    lay = run(meter_driver, tmp_path, plain, n_waves, n_slots)
    assert lay["rc"] == 0 and lay["scalars"]["any_meter"] == 0 and lay["scalars"]["meter_sb_total"] == 0
    assert lay["meter_kw"] == [] and lay["meter_peak"] == [] and lay["meter_tracks"] == [] and lay["meter_tdev"] == []
    assert all(w[5] == w[7] == w[9] == 0 for w in lay["waves"])
    # the flag adds the meter's tables and changes none of the others
    for flags in ([1] * 8, [1, 0, 0, 1, 1, 0, 1, 0]):
        flagged = make_tracks(meter_batch(flags))
        assert run(plan_driver, tmp_path, flagged, n_waves, n_slots, raw=True) == run(plan_driver, tmp_path, plain, n_waves, n_slots, raw=True)


def test_time_shard_with_the_flag_is_rejected(meter_driver, tmp_path):
    fs = 48000
    tracks = make_tracks([(6.0, fs, dict(synth.c2_settings(), measure_output=True), 30 * (fs // 10))])
    lay = run(meter_driver, tmp_path, tracks)
    assert lay["rc"] == AME_E_UNSUPPORTED
    assert lay["error"].startswith("track 0: the output meter measures a whole track and cannot run on a time shard"), lay
    tracks[0].halo_frames = 0
    assert run(meter_driver, tmp_path, tracks)["rc"] == 0


# ---- GPU ------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


PAIRS = (("output_i", "input_i"), ("output_thresh", "input_thresh"), ("output_lra", "input_lra"), ("output_n_blocks", "n_blocks"),
         ("output_sample_peak", "sample_peak"), ("output_true_peak", "true_peak"))


def _maxima(sub, fs):
    """Ungated maxima of the momentary (4 sub-blocks) and short-term (30 sub-blocks) energies at every sub-block, LUFS."""
    from oracle import chain
    s100 = chain.samples_in_100ms(fs)
    mom = [(((sub[k - 3] + sub[k - 2]) + sub[k - 1]) + sub[k]) / (4 * s100) for k in range(3, len(sub))]
    st = [sum(float(x) for x in sub[k - 29:k + 1]) / (30 * s100) for k in range(29, len(sub))]

    def lufs(e):
        return 10.0 * math.log10(e) - 0.691 if e > 0 else -math.inf
    return lufs(max(mom)) if mom else -math.inf, lufs(max(st)) if st else -math.inf


def oracle_meter(pcm, fs):
    """The meter's definition on the oracle: ebur128 gate and range, BS.1770 true peak, and the ungated maxima of the
    momentary and short-term loudness at every 100 ms sub-block.  The maxima come from the oracle's K-weighting biquads
    (pre-filter shelf, RLB high-pass) evaluated as two sections, as the kernel evaluates them; ebur128's literal
    4th-order direct form (chain.k_weighted) is the same transfer function but ill-conditioned near z = 1, and differs
    from the sections by up to ~5e-8 LU at 192 kHz (*_literal)."""
    from scipy.signal import sosfilt
    from oracle import chain
    blocks, sub = chain.gating_block_energies(pcm, fs)
    hist = chain.block_histogram(blocks)
    integrated, rel = chain.gated_loudness_from_histogram(hist)
    _, _, (pb, pa, rb, ra) = chain.k_weighting(fs)
    y = sosfilt(np.array([np.r_[pb, pa], np.r_[rb, ra]]), np.asarray(pcm, np.int16).astype(np.float64) * (1.0 / 32768.0), axis=0)
    s100 = chain.samples_in_100ms(fs)
    n_sub = y.shape[0] // s100
    sub_sec = (y[:n_sub * s100] ** 2).sum(axis=1).reshape(n_sub, s100).sum(axis=1)
    mm, ms = _maxima(sub_sec, fs)
    mm_lit, ms_lit = _maxima(sub, fs)
    return dict(integrated=integrated, thresh=(10.0 * math.log10(rel) - 0.691) if hist.sum() else -70.0,
                lra=chain.loudness_range_from_histogram(chain.short_term_histogram(sub, fs)), true_peak=chain.true_peak(pcm, fs),
                sample_peak=int(np.abs(pcm.astype(np.int32)).max()) if len(pcm) else 0, n_blocks=int(hist.sum()),
                max_momentary=mm, max_short_term=ms, max_momentary_literal=mm_lit, max_short_term_literal=ms_lit)


def check_vs_oracle(m, want, where):
    """m: a meter reading under the plain names (integrated, thresh, ...)."""
    if want["integrated"] == -math.inf:
        assert m["integrated"] == -math.inf, where
    else:
        assert abs(m["integrated"] - want["integrated"]) <= LUFS_TOL, where
    assert m["n_blocks"] == want["n_blocks"] and m["sample_peak"] == want["sample_peak"], where
    assert m["lra"] == pytest.approx(want["lra"], abs=1e-9), where
    assert m["thresh"] == pytest.approx(want["thresh"], abs=1e-9), where
    assert m["true_peak"] == pytest.approx(want["true_peak"], rel=2e-5), where
    for k in ("max_momentary", "max_short_term"):
        if want[k] == -math.inf:
            assert m[k] == -math.inf and want[k + "_literal"] == -math.inf, (where, k)
        else:
            assert m[k] == pytest.approx(want[k], abs=1e-9), (where, k)
            assert m[k] == pytest.approx(want[k + "_literal"], abs=1e-7), (where, k)


def plain_keys(info):
    from audio_mastering_engine_b200.engine import OUTPUT_KEYS
    return {k: info[v] for k, v in OUTPUT_KEYS.items()}


def identity_batch():
    """One batch: 44.1 / 48 / 96 / 192 kHz, multiband and plain tracks, a silent track, one shorter than 400 ms and one
    between 400 ms and 3 s."""
    c1, c2 = synth.c1_settings(), synth.c2_settings()
    items = [(synth.track(4.0, 44100, track_id=1, am_hz=2.0), 44100, c2), (synth.track(3.5, 48000, track_id=2, am_hz=3.0), 48000, c1),
             (np.zeros((48000, 2), np.int16), 48000, c2), (synth.track(2.2, 96000, track_id=3), 96000, c2),
             (synth.track(0.3, 48000, track_id=4), 48000, c1), (synth.track(1.7, 192000, track_id=5, am_hz=2.0), 192000, c2),
             (synth.track(1.1, 44100, track_id=6)[:47000], 44100, c1), (synth.track(3.2, 48000, track_id=7), 48000, c2)]
    sets = [dict(s, lufs=None, limiter=False, true_peak=True, measure_output=True) for _, _, s in items]
    return [x for x, _, _ in items], [f for _, f, _ in items], sets


@gpu
def test_output_equals_input_bit_for_bit(torch_cuda):
    """lufs=None, no limiter: the output IS the pre-normalisation signal, so every output_* equals its input counterpart
    exactly - through master_host (master()) and master_device, in three waves over two slots."""
    from audio_mastering_engine_b200 import MasterPlan, master
    tracks, fss, sets = identity_batch()
    _, infos = master(tracks, fss, sets, chunk_seconds=1, n_waves=3, n_slots=2)
    plan = MasterPlan([len(x) for x in tracks], fss, sets, chunk_seconds=1, n_waves=3, n_slots=2)
    d_in = torch_cuda.as_tensor(plan.pack(tracks)).cuda()
    d_out = torch_cuda.empty_like(d_in)
    dinfos = plan.master_device(d_in, d_out)
    for path, inf in (("host", infos), ("device", dinfos)):
        for k, i in enumerate(inf):
            for o, n in PAIRS:
                assert i[o] == i[n], (path, k, o, i[o], i[n])
    i = dinfos
    assert i[2]["output_i"] == -math.inf and i[2]["output_thresh"] == -70.0 and i[2]["output_max_momentary"] == -math.inf
    assert i[4]["output_max_momentary"] == -math.inf and i[4]["output_n_blocks"] == 0        # < 400 ms
    assert i[6]["output_max_momentary"] > -70 and i[6]["output_max_short_term"] == -math.inf  # 400 ms .. 3 s
    assert i[3]["output_max_short_term"] == i[5]["output_max_short_term"] == -math.inf                       # 2.2 s, 1.7 s
    assert all(x["output_max_short_term"] > -70 for j, x in enumerate(i) if j in (0, 1, 7))
    assert [{k: v for k, v in a.items() if k != "launches"} for a in infos] == dinfos      # same waves, same bytes
    plan.close()


@gpu
@pytest.mark.parametrize("fs", [44100, 48000, 96000, 192000])
def test_master_output_vs_oracle(torch_cuda, fs):
    """C2 at -9 LUFS with the limiter: output_* of master() against the oracle applied to the returned int16 output, and
    the stand-alone meter on that output gives the same report exactly."""
    from audio_mastering_engine_b200 import master, measure_loudness
    x = synth.track(4.5, fs, track_id=fs % 17, am_hz=2.0)
    s = dict(synth.c2_settings(), lufs=-9.0, limiter=True, true_peak=True, measure_output=True)
    out, info = master(x, fs, s, chunk_seconds=1)
    m = plain_keys(info)
    check_vs_oracle(m, oracle_meter(out, fs), fs)
    assert info["output_tp"] == 20 * math.log10(info["output_true_peak"])
    assert info["output_i"] != info["input_i"]
    again = measure_loudness(out, fs)
    assert again == {"input_i": m["integrated"], "input_tp": m["tp"], "input_lra": m["lra"], "input_thresh": m["thresh"],
                     "true_peak": m["true_peak"], "sample_peak": m["sample_peak"], "n_blocks": m["n_blocks"],
                     "max_momentary": m["max_momentary"], "max_short_term": m["max_short_term"]}


@gpu
def test_flag_on_some_tracks_changes_nothing_else(torch_cuda):
    from audio_mastering_engine_b200 import MasterPlan, master, EQ_PRESETS
    fs = 48000
    tracks = [synth.track(1.0 + 0.4 * k, fs, track_id=k, am_hz=2.0) for k in range(7)]
    base = [dict(synth.c4_settings(k, EQ_PRESETS), limiter=(k % 3 == 0), true_peak=(k == 4)) for k in range(7)]
    flagged = [dict(s, measure_output=True) if k in (1, 3, 4) else s for k, s in enumerate(base)]
    a, ia = master(tracks, fs, base, chunk_seconds=1, n_waves=3, n_slots=2)
    b, ib = master(tracks, fs, flagged, chunk_seconds=1, n_waves=3, n_slots=2)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    for k, (x, y) in enumerate(zip(ia, ib)):
        x, y = dict(x), dict(y)
        extra = {key: y.pop(key) for key in list(y) if key.startswith("output_")}
        assert y.pop("launches") > x.pop("launches")                 # the meter's launches
        assert x == y and bool(extra) == (k in (1, 3, 4)), k
    # the device path, and the meter's own entries
    outs = []
    for sets in (base, flagged):
        plan = MasterPlan([len(t) for t in tracks], fs, sets, chunk_seconds=1, n_waves=3, n_slots=2)
        assert plan.output_loudness() == [None] * 7                 # nothing measured before the first call
        d_in = torch_cuda.as_tensor(plan.pack(tracks)).cuda()
        d_out = torch_cuda.zeros_like(d_in)
        plan.master_device(d_in, d_out)
        outs.append((d_out.cpu().numpy(), plan.output_loudness()))
        plan.close()
    assert np.array_equal(outs[0][0], outs[1][0])
    rep = outs[1][1]
    assert [r is not None for r in rep] == [k in (1, 3, 4) for k in range(7)]
    for k in (1, 3, 4):
        assert rep[k]["integrated"] == ib[k]["output_i"] and rep[k]["true_peak"] == ib[k]["output_true_peak"]


@gpu
def test_stand_alone_meter_on_raw_input(torch_cuda):
    from audio_mastering_engine_b200 import measure_loudness
    items = [(synth.track(5.0, 44100, track_id=21, am_hz=1.5, am_db=9.0), 44100), (synth.stress_track(6.0, 48000, track_id=22), 48000),
             (synth.track(2.0, 96000, track_id=23), 96000), (synth.track(3.1, 192000, track_id=24), 192000),
             (np.zeros((30000, 2), np.int16), 48000), (synth.track(0.35, 48000, track_id=25)[:, 0].copy(), 48000)]
    reps = measure_loudness([x for x, _ in items], [f for _, f in items])
    for (x, fs), r in zip(items, reps):
        xs = x if x.ndim == 2 else np.stack([x, x], axis=1)
        m = {k: r[v] for k, v in (("integrated", "input_i"), ("thresh", "input_thresh"), ("lra", "input_lra"), ("true_peak", "true_peak"),
                                  ("sample_peak", "sample_peak"), ("n_blocks", "n_blocks"), ("max_momentary", "max_momentary"),
                                  ("max_short_term", "max_short_term"))}
        check_vs_oracle(m, oracle_meter(xs, fs), fs)
    # one track alone, and a CUDA tensor, give the same numbers as in the batch
    assert measure_loudness(items[1][0], 48000) == reps[1]
    assert measure_loudness(torch_cuda.as_tensor(items[2][0]).cuda(), 96000) == reps[2]


@gpu
def test_errors(torch_cuda):
    from audio_mastering_engine_b200 import AmeError, MasterPlan
    plan = MasterPlan([48000], 48000, synth.c1_settings())
    d = torch_cuda.zeros((plan.total_frames, 2), dtype=torch_cuda.int16, device="cuda")
    with pytest.raises(AmeError, match=r"libame error -1: no track carries AME_F_MEASURE_OUTPUT"):
        plan.measure_loudness(d)
    assert plan.output_loudness() == [None]
    plan.close()
    with pytest.raises(AmeError, match=r"libame error -4: track 0: the output meter measures a whole track"):
        MasterPlan([48000], 48000, dict(synth.c2_settings(), measure_output=True), halos=[4800])


@gpu
def test_entry_point_reports_final_loudness(torch_cuda, tmp_path):
    from audio_mastering_engine_b200 import process_audio_with_ffmpeg_pipeline, read_wav, write_wav
    fs = 44100
    x = synth.track(6.0, fs, track_id=9, am_hz=2.0)
    src = str(tmp_path / "in.wav")
    write_wav(src, x, fs)
    runs = {}
    for key in (False, True):
        dst = str(tmp_path / f"out_{key}.wav")
        settings = dict(synth.c2_settings(), lufs=-12.0, input_file=src, output_file=dst)
        if key:
            settings["measure_output"] = True
        status, progress = [], []
        process_audio_with_ffmpeg_pipeline(settings, status.append, lambda a, b: progress.append((a, b)))
        runs[key] = (status, progress, read_wav(dst)[0])
    (s0, p0, o0), (s1, p1, o1) = runs[False], runs[True]
    assert np.array_equal(o0, o1) and p0 == p1
    line = [s for s in s1 if s.startswith("Final loudness:")]
    assert len(line) == 1 and [s for s in s1 if s != line[0]] == s0
    assert s1.index(line[0]) == s1.index("Applying final limiting and exporting...") + 1
    m = re.fullmatch(r"Final loudness: (-?[\d.]+) LUFS integrated, (-?[\d.]+) dBTP true peak, LRA ([\d.]+) LU", line[0])
    assert m, line[0]
    want = oracle_meter(o1, fs)
    assert abs(float(m.group(1)) - want["integrated"]) <= 0.005 + LUFS_TOL
    assert abs(float(m.group(2)) - 20 * math.log10(want["true_peak"])) <= 0.006
    assert abs(float(m.group(3)) - want["lra"]) <= 0.05 + 1e-9


@gpu
@pytest.mark.parametrize("limiter", [False, True])
def test_time_sharded_output_report(torch_cuda, limiter):
    from audio_mastering_engine_b200 import master, measure_loudness, sharding
    from audio_mastering_engine_b200.engine import OUTPUT_KEYS, INPUT_KEYS
    fs = 48000
    x = synth.track(9.0, fs, track_id=6, am_hz=1.0, drift_db=8.0, drift_period=3.0)
    s = dict(synth.c2_settings(), lufs=-9.0, limiter=limiter, measure_output=True)
    assert "measure_output" not in sharding._shard_settings(s)
    many, infon = sharding.master_time_sharded_local(x, fs, s, 3, chunk_seconds=1.0)
    alone = measure_loudness(many, fs)
    assert {v: infon[v] for v in OUTPUT_KEYS.values()} == {OUTPUT_KEYS[k]: alone[v] for k, v in INPUT_KEYS.items()}
    plain, _ = sharding.master_time_sharded_local(x, fs, dict(s, measure_output=False), 3, chunk_seconds=1.0)
    assert np.array_equal(plain, many)
    one, info1 = master(x, fs, s, chunk_seconds=1.0)
    if np.array_equal(one, many):
        assert {v: info1[v] for v in OUTPUT_KEYS.values()} == {v: infon[v] for v in OUTPUT_KEYS.values()}
    else:                                            # the tilings may flip isolated LSBs (DESIGN.md section 6)
        assert abs(info1["output_i"] - infon["output_i"]) <= LUFS_TOL


@gpu
def test_host_path_copies_do_not_wait_for_the_meter(torch_cuda):
    """ame_master_host meters a wave after the event its D2H copy waits for: with the meter on every track, the first
    wave's copy-out still ends before the last wave's kernels do (as without the meter), and the bytes are the same."""
    from audio_mastering_engine_b200 import MasterPlan, EQ_PRESETS
    fs = 48000
    tracks = [synth.track(20.0, fs, track_id=k, am_hz=2.0) for k in range(9)]
    base = [synth.c4_settings(k, EQ_PRESETS) for k in range(9)]
    outs = []
    for flag in (False, True):
        plan = MasterPlan([len(t) for t in tracks], fs, [dict(s, measure_output=flag) for s in base], chunk_seconds=1,
                          host_io=True, n_waves=4, n_slots=2)
        h_in = torch_cuda.from_numpy(plan.pack(tracks)).pin_memory()
        h_out = torch_cuda.empty(h_in.shape, dtype=torch_cuda.int16, pin_memory=True)
        plan.master_host(h_in, h_out)                  # warm-up
        plan.set_timing(True)
        infos = plan.master_host(h_in, h_out)
        tl = plan.wave_timeline()                      # per wave: H2D done, kernels may start, kernels done, D2H done
        print("meter", flag, "wave timeline (ms):", [tuple(round(v, 3) for v in row) for row in tl])
        assert len(tl) == 4 and tl[0][3] < tl[-1][2], (flag, tl)
        assert all("output_i" in i for i in infos) == flag
        outs.append(h_out.numpy().copy())
        plan.close()
    assert np.array_equal(outs[0], outs[1])
