"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI
(include/ame.h via ctypes), against the committed reference fixtures and the CPU oracle.

Tolerances (BASELINE.json north_star): per-sample null residual <= -80 dBFS (|diff| <= 3 LSB of int16),
integrated LUFS within 0.01 LU.  Integer stages (window rms, band truncation given equal inputs,
saturating overlay, gain rounding) are held to bit-exact; the float paths are expected to be bit-exact
too except for isolated +-1 LSB truncation flips (FP64 filters evaluated with FMA / another order).
"""
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NULL_LSB = 3           # -80 dBFS = 3.27 LSB
LUFS_TOL = 0.01


@pytest.fixture(scope="module")
def torch_cuda():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _maxdiff(a, b):
    return int(np.abs(a.astype(np.int32) - b.astype(np.int32)).max()) if a.size else 0


def _lufs_close(a, b):
    return a == b or abs(a - b) <= LUFS_TOL


def _nz(a, b):
    return float(np.mean(a != b)) if a.size else 0.0


def _run_stages(torch, plan, x):
    """in -> stage_eq -> (band split -> compress) ; returns dict of taps as numpy."""
    dev = torch.device("cuda", plan.device)
    h = plan.pack([x])
    d_in = torch.from_numpy(h).to(dev)
    d_pre = torch.zeros_like(d_in)
    taps = {}
    plan.stage_eq(d_in, d_pre)
    torch.cuda.synchronize()
    taps["pre_multiband"] = d_pre.cpu().numpy()[: len(x)]
    mbf = plan.mb_frames
    if mbf:
        d_bands = torch.zeros((3, mbf, 2), dtype=torch.int16, device=dev)
        plan.stage_band_split(d_pre, d_bands)
        torch.cuda.synchronize()
        b = d_bands.cpu().numpy()
        taps["bands"] = b[:, : len(x)].copy()
        plan.stage_compress(d_bands, d_pre)
        torch.cuda.synchronize()
    taps["out"] = d_pre.cpu().numpy()[: len(x)]
    return taps


def test_golden_reference_cases(torch_cuda, golden):
    """Fixtures produced by the reference's own functions (tests/golden/make_golden.py)."""
    from audio_mastering_engine_b200 import MasterPlan
    from oracle import chain
    g = golden
    worst = 0
    for c in g.cases:
        key, fs, settings = c["key"], c["fs"], dict(c["settings"])
        x = g.input(c)
        # the reference's whole arrays: the oracle's, held to the stored digests bit for bit
        want = {}
        want["out"] = chain.process_chunk(x, fs, settings, taps=want, compress=chain.compress_dynamic_range_py)
        assert g.equals(c, "pre_multiband", want["pre_multiband"]) and g.equals(c, "out", want["out"]), key
        settings["lufs"] = None
        for tile in (0, 512):   # auto tiles and small tiles (exercises the warm-up path)
            plan = MasterPlan([len(x)], fs, settings, chunk_seconds=None, eq_tile_frames=tile, xover_tile_frames=tile)
            taps = _run_stages(torch_cuda, plan, x)
            plan.close()
            d1 = _maxdiff(taps["pre_multiband"], want["pre_multiband"])
            d2 = _maxdiff(taps["out"], want["out"])
            worst = max(worst, d1, d2)
            assert d1 <= 1, (key, tile, d1)
            assert _nz(taps["pre_multiband"], want["pre_multiband"]) < 1e-3, (key, tile)
            assert d2 <= NULL_LSB, (key, tile, d2)
            assert _nz(taps["out"], want["out"]) < 2e-3, (key, tile)
    print("golden worst LSB diff", worst)


def test_stage_taps_vs_oracle(torch_cuda):
    from audio_mastering_engine_b200 import MasterPlan, synth
    from oracle import chain, cport
    fs = 48000
    x = synth.track(2.0, fs, track_id=11, am_hz=3.0)
    settings = dict(synth.c2_settings(), lufs=None)
    plan = MasterPlan([len(x)], fs, settings, chunk_seconds=None, eq_tile_frames=4096, xover_tile_frames=2048)
    taps = _run_stages(torch_cuda, plan, x)
    otaps = {}
    ref = chain.process_chunk(x, fs, settings, taps=otaps)
    assert _maxdiff(taps["pre_multiband"], otaps["pre_multiband"]) <= 1
    # band split given the GPU's own pre-multiband signal: integer-exact expectation
    lo, mi, hi = chain.band_split(taps["pre_multiband"], fs)
    for b, want in enumerate((lo, mi, hi)):
        assert _maxdiff(taps["bands"][b], want) <= 1
        assert _nz(taps["bands"][b], want) < 1e-4
    # compressor + overlay given the GPU's own bands
    comp = [cport.compress(taps["bands"][b], fs, settings[n + "_thresh"], settings[n + "_ratio"])
            for b, n in enumerate(("low", "mid", "high"))]
    want = chain.overlay(chain.overlay(comp[0], comp[1]), comp[2])
    assert _maxdiff(taps["out"], want) <= 1
    assert _nz(taps["out"], want) < 1e-5
    assert _maxdiff(taps["out"], ref) <= NULL_LSB
    plan.close()


@pytest.mark.parametrize("fs,secs,chunk,settings_name", [
    (44100, 3.0, 1, "c1"), (48000, 4.0, 1, "c2"), (96000, 1.5, 0.5, "c2"), (192000, 1.0, 0.4, "c2"),
    (48000, 2.0, 30, "lofi"), (22050, 2.0, 1, "bass0")])
def test_master_vs_oracle(torch_cuda, fs, secs, chunk, settings_name):
    from audio_mastering_engine_b200 import master, synth, EQ_PRESETS
    from oracle import chain
    settings = {"c1": synth.c1_settings(), "c2": synth.c2_settings(),
                "lofi": dict(EQ_PRESETS["Lo-Fi Haze"], analog_character=0, width=0.8, lufs=-16.0, multiband=True,
                             **synth.DEFAULT_MULTIBAND),
                "bass0": dict(bass_boost=0.0, mid_cut=0.0, presence_boost=3.0, treble_boost=0.0, width=1.0,
                              analog_character=0, lufs=-9.0, multiband=False)}[settings_name]
    x = synth.track(secs, fs, track_id=fs % 13, am_hz=2.0)
    for tile in (0, 1024):
        out, info = master(x, fs, settings, chunk_seconds=chunk, eq_tile_frames=tile, xover_tile_frames=tile,
                           kw_tile_subblocks=0 if tile == 0 else 3)
        ref, rinfo = chain.master(x, fs, settings, chunk_seconds=chunk)
        assert _lufs_close(info["input_i"], rinfo["input_i"])
        assert info["measured_i_2dp"] == rinfo["measured_i_2dp"]
        assert info["n_blocks"] == rinfo["n_blocks"]
        assert info["input_lra"] == pytest.approx(rinfo["input_lra"], abs=1e-9)
        assert info["input_thresh"] == pytest.approx(rinfo["input_thresh"], abs=1e-9) or info["n_blocks"] == 0
        d = _maxdiff(out, ref)
        assert d <= NULL_LSB, (tile, d)
        assert _nz(out, ref) < 5e-3
        assert info["launches"] > 0


def test_batch_mixed_rates_and_edge_cases(torch_cuda):
    """Ragged lengths, mixed sample rates, silence (-inf => copied through), < 400 ms track, lufs None,
    mono input - in ONE packed batch."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    tracks, fss, sets = [], [], []
    tracks.append(synth.track(1.234, 44100, 1)[:54321]); fss.append(44100); sets.append(synth.c1_settings())
    tracks.append(np.zeros((30001, 2), np.int16)); fss.append(48000); sets.append(synth.c2_settings())
    tracks.append(synth.track(0.3, 48000, 2)); fss.append(48000); sets.append(synth.c1_settings())       # < 400 ms
    tracks.append(synth.track(1.0, 96000, 3)[:95999]); fss.append(96000); sets.append(dict(synth.c2_settings(), lufs=None))
    tracks.append(synth.track(0.7, 48000, 4)[:, 0].copy()); fss.append(48000); sets.append(synth.c1_settings())  # mono
    tracks.append(synth.track(0.001, 48000, 5)[:3]); fss.append(48000); sets.append(synth.c2_settings())  # 3 frames
    outs, infos = master(tracks, fss, sets, chunk_seconds=0.5)
    for x, fs, s, out, info in zip(tracks, fss, sets, outs, infos):
        xs = x if x.ndim == 2 else np.stack([x, x], axis=1)
        ref, rinfo = chain.master(xs, fs, s, chunk_seconds=0.5)
        assert out.shape == ref.shape
        assert _maxdiff(out, ref) <= NULL_LSB
        if s.get("lufs") is not None:
            assert info["normalized"] == rinfo["normalized"]
            if rinfo["normalized"]:
                assert abs(info["input_i"] - rinfo["input_i"]) <= LUFS_TOL
            else:
                assert info["input_i"] == -math.inf
    assert not infos[1]["normalized"] and np.array_equal(outs[1], tracks[1])


def test_stress_compressor_extremes(torch_cuda):
    """C5-style: bursts, beds, exact-zero gaps, clicks; thresh -40 / ratio 10 and thresh 0 / ratio 1."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    fs = 48000
    x = synth.stress_track(24.0, fs, track_id=3)
    for th, ra in ((-40.0, 10.0), (0.0, 1.0)):
        s = dict(synth.ALL_BOOST_EQ, analog_character=25, width=1.2, lufs=-14.0, multiband=True,
                 low_thresh=th, low_ratio=ra, mid_thresh=th, mid_ratio=ra, high_thresh=th, high_ratio=ra)
        out, info = master(x, fs, s, chunk_seconds=10)
        ref, rinfo = chain.master(x, fs, s, chunk_seconds=10)
        assert abs(info["input_i"] - rinfo["input_i"]) <= LUFS_TOL
        assert _maxdiff(out, ref) <= NULL_LSB


def test_tile_invariance_full_c2(torch_cuda):
    """Size-independent property at BASELINE config C2 (3 min, 48 kHz, multiband): the result must not
    depend on how the GPU tiles the time axis, and must null against the oracle."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    fs = 48000
    x = synth.track(180.0, fs, track_id=0, am_hz=2.0)
    s = synth.c2_settings()
    a, ia = master(x, fs, s)
    b, ib = master(x, fs, s, eq_tile_frames=8192, xover_tile_frames=4096, kw_tile_subblocks=7)
    assert ia["input_i"] == pytest.approx(ib["input_i"], abs=1e-9)
    assert _maxdiff(a, b) <= 1 and _nz(a, b) < 1e-5
    ref, rinfo = chain.master(x, fs, s)
    assert abs(ia["input_i"] - rinfo["input_i"]) <= LUFS_TOL
    assert _maxdiff(a, ref) <= NULL_LSB
    print("C2 null:", _maxdiff(a, ref), "LSB; differing samples", _nz(a, ref), "LUFS", ia["input_i"], rinfo["input_i"])


def test_error_paths(torch_cuda):
    from audio_mastering_engine_b200 import master, process_audio_with_ffmpeg_pipeline, AmeError
    with pytest.raises(ValueError, match="Input or output file not specified."):
        process_audio_with_ffmpeg_pipeline({}, lambda s: None, lambda a, b: None)
    with pytest.raises(TypeError):
        master(np.zeros((10, 2), np.float32), 48000, {})
    with pytest.raises((AmeError, ValueError)):
        master(np.zeros((100, 2), np.int16), 1000, {})       # unsupported rate


def test_wav_entry_point_roundtrip(torch_cuda, tmp_path):
    from audio_mastering_engine_b200 import process_audio, read_wav, write_wav, synth
    from oracle import chain
    fs = 44100
    x = synth.track(1.0, fs, 8)
    src, dst = str(tmp_path / "in.wav"), str(tmp_path / "out.wav")
    write_wav(src, x, fs)
    settings = dict(synth.c1_settings(), input_file=src, output_file=dst)
    status, progress, art, tags = [], [], [], []
    process_audio(settings, status.append, lambda a, b: progress.append((a, b)), art.append, tags.append)
    assert any(s.startswith("Success:") for s in status), status
    assert progress[0] == (0, 100) and progress[-1] == (5, 5) and art == [None]
    out, fs2 = read_wav(dst)
    ref, _ = chain.master(x, fs, dict(settings, limiter=True))        # the entry point ends with the limiter (:223)
    assert fs2 == fs and _maxdiff(out, ref) <= NULL_LSB
    # failure protocol (audio_mastering_engine.py:131-137)
    status.clear(); progress.clear(); art.clear(); tags.clear()
    process_audio(dict(settings, input_file=str(tmp_path / "missing.wav")), status.append,
                  lambda a, b: progress.append((a, b)), art.append, tags.append)
    assert status[-1].startswith("Error:") and progress[-1] == (0, 1) and tags == ["Processing failed."]


@pytest.mark.parametrize("fs,seconds,chunk,world", [(48000, 9.0, 1.0, 3), (44100, 5.0, 1.0, 2), (96000, 3.0, 0.5, 8)])
def test_time_sharded_equals_single_plan(torch_cuda, fs, seconds, chunk, world):
    """Long-track path (BASELINE config C3): shards by time with halo hand-off and a summed histogram must
    reproduce the single-plan result (bit for bit) and null against the oracle."""
    from audio_mastering_engine_b200 import master, synth, sharding
    from oracle import chain
    x = synth.track(seconds, fs, track_id=6, am_hz=1.0, drift_db=8.0, drift_period=3.0)
    s = synth.c2_settings()
    one, info1 = master(x, fs, s, chunk_seconds=chunk)
    many, infon = sharding.master_time_sharded_local(x, fs, s, world, chunk_seconds=chunk)
    assert infon["n_blocks"] == info1["n_blocks"]
    assert infon["input_i"] == pytest.approx(info1["input_i"], abs=1e-9)
    assert np.array_equal(one, many)
    ref, rinfo = chain.master(x, fs, s, chunk_seconds=chunk)
    assert _lufs_close(infon["input_i"], rinfo["input_i"]) and _maxdiff(many, ref) <= NULL_LSB


def test_host_path_waves_equal_single_wave(torch_cuda):
    """ame_master_host pipelines H2D / kernels / D2H over waves of tracks: same bytes as one wave."""
    from audio_mastering_engine_b200 import master, synth, EQ_PRESETS
    fs = 48000
    tracks = [synth.track(1.0 + 0.37 * k, fs, track_id=k, am_hz=2.0) for k in range(7)]
    sets = [synth.c4_settings(k + 1, EQ_PRESETS) for k in range(7)]
    a, ia = master(tracks, fs, sets, chunk_seconds=1)
    for waves in (2, 3, 7, 16):
        b, ib = master(tracks, fs, sets, chunk_seconds=1, n_waves=waves)
        assert all(np.array_equal(x, y) for x, y in zip(a, b)), waves
        assert [i["input_i"] for i in ia] == [i["input_i"] for i in ib]


def test_kernel_timing_exports(torch_cuda):
    """ame_plan_set_timing / kernel_times / kernel_timeline: every kernel the settings need shows up once per wave, begins
    before it ends, follows its predecessor in the wave's stream, and timing does not change the bytes that come out."""
    import torch
    from audio_mastering_engine_b200 import MasterPlan, synth, EQ_PRESETS
    fs = 48000
    tracks = [synth.track(1.0, fs, track_id=k, am_hz=2.0) for k in range(6)]
    sets = [dict(synth.c4_settings(k, EQ_PRESETS), limiter=(k == 2), true_peak=(k == 3)) for k in range(6)]
    plan = MasterPlan([len(t) for t in tracks], fs, sets, chunk_seconds=0.5, n_waves=3, n_slots=2)
    d_in = torch.as_tensor(plan.pack(tracks)).cuda()
    ref, out = torch.empty_like(d_in), torch.empty_like(d_in)
    plan.master_device(d_in, ref)
    plan.set_timing(True)
    for _ in range(2):
        plan.master_device(d_in, out)
    torch.cuda.synchronize()
    assert torch.equal(ref, out)
    times, steps = plan.kernel_times()
    assert steps == 2
    assert times["k_eq"][1] == 2 * 3 and times["k_apply_gain"][1] == 6 and times["k_eq"][0] > 0
    assert times["k_window_flag"][1] == 6 and times["k_att_chain"][1] == 6           # every wave has a multiband track
    assert times["k_limiter"][1] == 2 and times["k_true_peak"][1] == 2               # one wave each
    tl = plan.kernel_timeline(1)
    assert len(tl) == 3
    order = ["k_eq", "k_band_split", "k_window_flag", "k_att_chain", "k_compress_apply", "k_kweight_energy", "k_apply_gain"]
    for w in tl:
        assert all(b <= e for b, e in w.values())
        ends = [w[k][1] for k in order if k in w]
        begins = [w[k][0] for k in order if k in w]
        assert all(begins[i + 1] >= ends[i] - 1e-3 for i in range(len(ends) - 1)), w      # stream order inside a wave
    with pytest.raises(Exception):
        plan.kernel_timeline(5)
    plan.close()


def test_random_settings_sweep(torch_cuda):
    """Randomised settings over the GUI slider ranges (mastering_gui.py:44-55) and several sample rates, one
    batch per rate, every track against the oracle."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    rng = np.random.default_rng(2026)
    worst = 0
    for fs in (22050, 32000, 44100, 48000, 88200, 96000):
        tracks, sets = [], []
        for k in range(6):
            def pick(lo, hi, zero_p=0.25):
                return 0.0 if rng.random() < zero_p else float(np.round(rng.uniform(lo, hi), 1))
            s = dict(bass_boost=pick(-6, 6), mid_cut=pick(0, 6), presence_boost=pick(-6, 6), treble_boost=pick(-6, 6),
                     width=float(np.round(rng.uniform(0, 2), 2)) if rng.random() < 0.7 else 1.0,
                     analog_character=0 if (rng.random() < 0.4 or fs < 30000) else int(rng.integers(1, 101)),
                     lufs=None if rng.random() < 0.15 else float(np.round(rng.uniform(-20, -6), 1)),
                     multiband=bool(rng.random() < 0.6))
            for b in ("low", "mid", "high"):
                s[b + "_thresh"] = float(np.round(rng.uniform(-40, 0), 1))
                s[b + "_ratio"] = float(np.round(rng.uniform(1, 10), 1))
            secs = float(rng.uniform(0.45, 1.6))
            x = synth.track(secs, fs, track_id=100 + k, am_hz=float(rng.uniform(1, 8)), am_db=float(rng.uniform(0, 12)))
            x = np.clip(x.astype(np.float64) * 10 ** (rng.uniform(-12, 9) / 20), -32768, 32767).astype(np.int16)
            tracks.append(x); sets.append(s)
        outs, infos = master(tracks, fs, sets, chunk_seconds=0.5)
        for x, s, out, info in zip(tracks, sets, outs, infos):
            ref, rinfo = chain.master(x, fs, s, chunk_seconds=0.5)
            d = _maxdiff(out, ref)
            worst = max(worst, d)
            assert d <= NULL_LSB, (fs, s, d)
            if s["lufs"] is not None:
                assert _lufs_close(info["input_i"], rinfo["input_i"]), (fs, s)
    print("random sweep worst LSB diff", worst)


def test_bypass_identity_and_idempotent_normalisation(torch_cuda):
    """Property checks (SURVEY section 4.4): with every stage at its neutral setting the path reduces to the
    reference's lossy int16 -> float -> int16 converter pair; normalising an already normalised track is a no-op
    within one LSB; ratio 1 compressors pass the bands through; width 1.0 is a bypass, not an M/S round trip."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    fs = 48000
    x = synth.track(3.0, fs, 21, am_hz=3.0)
    flat = dict(bass_boost=0.0, mid_cut=0.0, presence_boost=0.0, treble_boost=0.0, analog_character=0, width=1.0,
                lufs=None, multiband=False)
    out, info = master(x, fs, flat)
    assert np.array_equal(out, chain.to_pcm(chain.to_float(x)))          # engine.py:250-257 only
    assert not info["normalized"] and info["gain"] == 1.0
    once, i1 = master(x, fs, dict(flat, lufs=-14.0))
    twice, i2 = master(once, fs, dict(flat, lufs=-14.0))
    assert abs(i2["input_i"] - (-14.0)) < 0.02
    assert _maxdiff(chain.to_pcm(chain.to_float(once)), twice) <= 1
    unity = dict(flat, multiband=True, low_thresh=-30.0, low_ratio=1.0, mid_thresh=-30.0, mid_ratio=1.0,
                 high_thresh=-30.0, high_ratio=1.0)
    mb, _ = master(x, fs, unity)
    lo, mi, hi = chain.band_split(chain.to_pcm(chain.to_float(x)), fs)
    assert np.array_equal(mb, chain.overlay(chain.overlay(lo, mi), hi))  # ratio 1 => M = 0 => untouched bands


def test_compressor_kernels_agree(torch_cuda):
    """The attenuation recurrence has two kernels: k_att_chain (one lane per chain, queue of flagged frames) and
    k_att_chain_spec (32..256 speculative time segments per chain, repaired until exact).  Same bytes from both, for
    every segment count, on ragged lengths and on signals built to defeat the speculation: a loud burst followed by a
    bed that stays just above threshold (the attenuation never clamps again, so every segment has to be re-walked)."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    fs = 48000
    rng = np.random.default_rng(7)
    n = 6 * fs + 1237
    t = np.arange(n) / fs
    bed = 0.02 * np.sin(2 * np.pi * 440.0 * t) + 0.002 * rng.standard_normal(n)
    burst = np.where(t < 0.2, 0.9 * np.sin(2 * np.pi * 330.0 * t), 0.0)
    held = np.stack([bed + burst, bed - burst], axis=1)
    held = np.clip(held * 32767, -32767, 32767).astype(np.int16)
    cases = [
        (synth.track(5.3, fs, track_id=11, am_hz=2.0)[:250003], synth.c2_settings(), 2.0),
        (synth.stress_track(8.0, fs, track_id=5), dict(synth.c2_settings(), low_thresh=-40.0, mid_thresh=-40.0, high_thresh=-40.0), 30),
        (held, dict(synth.c2_settings(), low_thresh=-36.0, low_ratio=8.0, mid_thresh=-36.0, mid_ratio=8.0), 30),
        (synth.track(0.02, fs, track_id=2)[:701], synth.c2_settings(), 30),           # shorter than 32 * 32 frames
    ]
    for x, s, chunk in cases:
        base, binfo = master(x, fs, s, chunk_seconds=chunk, chain_warps=-1)
        ref, _ = chain.master(x, fs, s, chunk_seconds=chunk)
        assert _maxdiff(base, ref) <= NULL_LSB
        for cw in (1, 3, 8):
            out, info = master(x, fs, s, chunk_seconds=chunk, chain_warps=cw)
            assert np.array_equal(out, base), cw
            assert info["input_i"] == binfo["input_i"]


def test_plan_memory_pool_reuse_and_release(torch_cuda):
    """Plan workspaces come from a per-device pool that keeps the memory of destroyed plans: results must not depend
    on whether a plan got fresh or recycled (dirty) memory, and the pool can be handed back at any time."""
    from audio_mastering_engine_b200 import master, release_cached_memory, synth
    fs = 48000
    x = synth.track(2.0, fs, track_id=21, am_hz=3.0)              # 96000 frames: the zero-copy single-track path
    y = synth.track(1.3, fs, track_id=22, am_hz=2.0)[:62001]      # ragged: the packed path
    first = [master(x, fs, synth.c2_settings(), chunk_seconds=1)[0], master(y, fs, synth.c1_settings())[0]]
    master([x, y, x], fs, [synth.c1_settings(), synth.c2_settings(), synth.c2_settings()], chunk_seconds=0.5)   # dirties a larger workspace
    again = [master(x, fs, synth.c2_settings(), chunk_seconds=1)[0], master(y, fs, synth.c1_settings())[0]]
    release_cached_memory(0)
    fresh = [master(x, fs, synth.c2_settings(), chunk_seconds=1)[0], master(y, fs, synth.c1_settings())[0]]
    for a, b, c in zip(first, again, fresh):
        assert np.array_equal(a, b) and np.array_equal(a, c)


# ------------------------------------------------------------------------------------------------
# round 2: limiter, true peak, full-size BASELINE configs, the shipped by-time path over torch.distributed
# ------------------------------------------------------------------------------------------------
def _hot(x, gain):
    return np.clip(np.rint(x.astype(np.float64) * gain), -32768, 32767).astype(np.int16)


def test_limiter_stage_is_bit_exact(torch_cuda):
    """ffmpeg alimiter (:223) on the GPU = the oracle's restatement, bit for bit, given the same normalised signal:
    quiet input (elementwise tiles only), sparse over-limit peaks, heavy clipping (one sequential run per track) and a
    multi-tile track whose over-limit passages start and end sequential runs at tile boundaries."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import limiter
    fs = 48000
    flat = dict(bass_boost=0.0, mid_cut=0.0, presence_boost=0.0, treble_boost=0.0, analog_character=0, width=1.0,
                lufs=None, multiband=False)
    long = synth.track(5.0, fs, track_id=31) // 2                      # 240000 frames = 8 limiter tiles, all below the limit
    long[30000:30400] = _hot(long[30000:30400], 9.0)                   # a passage inside tile 0
    long[65500:65600, 0] = 32767                                       # straddles the tile 1 / tile 2 boundary (65536)
    long[131071] = [-32768, 32767]                                     # last frame of tile 3
    long[200000:200003] = 32700                                        # tile 6
    cases = [synth.track(1.0, fs, track_id=30) // 2,                   # nothing over the limit
             _hot(synth.track(1.5, fs, track_id=32, am_hz=3.0), 4.0),  # sparse peaks
             _hot(synth.track(2.0, fs, track_id=33, am_hz=2.0), 14.0), # clipped most of the time
             long, long[:32768], long[:32769], long[:100],
             _hot(synth.track(14.0, fs, track_id=34, am_hz=1.0), 14.0),   # 21 tiles over the limit all the time: every start is a guess
             _hot(synth.track(14.0, fs, track_id=35, am_hz=0.7, am_db=10.0), 5.0),   # busy and quiet passages alternate
             _hot(synth.stress_track(11.0, fs, track_id=36), 3.5)]     # bursts, beds, zero gaps, clicks
    for k, x in enumerate(cases):
        plain, _ = master(x, fs, flat)
        got, _ = master(x, fs, dict(flat, limiter=True))
        want = limiter.alimiter(plain, fs)
        assert np.array_equal(got, want), (k, _maxdiff(got, want), int(np.argmax(np.any(got != want, axis=1))))
    # other look-ahead / release lengths and sample rates, in one batch with tracks that have no limiter
    xs = [_hot(synth.track(0.8, f, track_id=40 + i, am_hz=4.0), 6.0) for i, f in enumerate((44100, 96000, 22050, 48000))]
    fss = [44100, 96000, 22050, 48000]
    sets = [dict(flat, limiter=True), dict(flat, limiter=True, limiter_limit=0.9, limiter_attack=2.0, limiter_release=20.0),
            dict(flat), dict(synth.c2_settings(), limiter=True)]
    outs, _ = master(xs, fss, sets, chunk_seconds=0.5)
    plains, _ = master(xs, fss, [dict(s, limiter=False) for s in sets], chunk_seconds=0.5)
    for x, f, s, o, pl in zip(xs, fss, sets, outs, plains):
        want = limiter.alimiter(pl, f, s.get("limiter_limit", 0.98), s.get("limiter_attack", 5.0), s.get("limiter_release", 50.0)) \
            if s.get("limiter") else pl
        assert np.array_equal(o, want), f


def test_limiter_alone_and_after_time_sharding(torch_cuda):
    """ame_stage_limiter (the limiter as its own stage: what a time-sharded track ends with on the rank that gathers
    its spans) against the oracle's restatement, and the by-time path with the limiter on against the single plan."""
    import torch
    from audio_mastering_engine_b200 import limit_device, master, sharding, synth
    from oracle import limiter
    fs = 48000
    for k, x in enumerate([_hot(synth.track(3.0, fs, track_id=50, am_hz=2.0), 6.0), synth.track(0.7, fs, track_id=51)[:33001],
                           _hot(synth.track(2.0, 96000, track_id=52), 12.0)]):
        f = 96000 if k == 2 else fs
        got = limit_device(torch.as_tensor(x).cuda(), f).cpu().numpy()
        assert np.array_equal(got, limiter.alimiter(x, f)), k
    got = limit_device(torch.as_tensor(x).cuda(), 96000, dict(limiter_limit=0.8, limiter_attack=3.0, limiter_release=30.0)).cpu().numpy()
    assert np.array_equal(got, limiter.alimiter(x, 96000, 0.8, 3.0, 30.0))
    x = synth.track(9.0, fs, track_id=6, am_hz=1.0, drift_db=8.0, drift_period=3.0)
    s = dict(synth.c2_settings(), lufs=-9.0, limiter=True)         # hot target: the limiter works most of the time
    one, info1 = master(x, fs, s, chunk_seconds=1.0)
    many, infon = sharding.master_time_sharded_local(x, fs, s, 3, chunk_seconds=1.0)
    assert np.array_equal(one, many) and infon["input_i"] == pytest.approx(info1["input_i"], abs=1e-9)
    assert not np.array_equal(one, master(x, fs, dict(s, limiter=False), chunk_seconds=1.0)[0])


def test_master_with_limiter_vs_oracle(torch_cuda):
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    fs = 48000
    x = synth.track(4.0, fs, track_id=12, am_hz=2.0)
    s = dict(synth.c2_settings(), lufs=-9.0, limiter=True, true_peak=True)     # +10 dB of make-up gain: the limiter works
    out, info = master(x, fs, s, chunk_seconds=1)
    ref, rinfo = chain.master(x, fs, s, chunk_seconds=1)
    assert _lufs_close(info["input_i"], rinfo["input_i"])
    assert _maxdiff(out, ref) <= NULL_LSB
    assert info["true_peak"] == pytest.approx(rinfo["true_peak"], rel=2e-5)
    assert info["input_tp"] == pytest.approx(20 * math.log10(rinfo["true_peak"]), abs=1e-3)
    for f2 in (44100, 96000, 192000):                                          # 4x, 2x, none
        y = synth.track(0.5, f2, track_id=13)
        _, i2 = master(y, f2, dict(synth.c1_settings(), true_peak=True))
        _, r2 = chain.master(y, f2, dict(synth.c1_settings(), true_peak=True))
        assert i2["true_peak"] == pytest.approx(r2["true_peak"], rel=2e-5), f2


def test_quiet_track_through_the_entry_point_says_dynamic_mode(torch_cuda, tmp_path):
    """A track far below the target: ffmpeg's loudnorm would leave linear mode (measured_TP + offset > -1.5 dBTP).
    The drop-in entry point applies the static gain, limits, and SAYS so (status line + log) - never silently."""
    from audio_mastering_engine_b200 import process_audio_with_ffmpeg_pipeline, read_wav, write_wav, synth
    from oracle import chain
    fs = 44100
    x = (synth.stress_track(12.0, fs, 14).astype(np.int32) // 4).astype(np.int16)   # -24 LUFS, clicks 15 dB over the bursts
    src, dst = str(tmp_path / "quiet.wav"), str(tmp_path / "quiet_out.wav")
    write_wav(src, x, fs)
    settings = dict(synth.c1_settings(), lufs=-9.0, input_file=src, output_file=dst)
    status = []
    process_audio_with_ffmpeg_pipeline(settings, status.append, lambda a, b: None)
    assert any("dynamic mode" in s for s in status), status
    out, _ = read_wav(dst)
    ref, rinfo = chain.master(x, fs, dict(settings, limiter=True, true_peak=True))
    assert _maxdiff(out, ref) <= NULL_LSB
    assert 20 * math.log10(rinfo["true_peak"]) + (-9.0 - rinfo["measured_i_2dp"]) > -1.5


def test_c1_full_size(torch_cuda):
    """BASELINE config C1 at full size: 30 s, 44.1 kHz, EQ + warmth + width + -14 LUFS."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    fs = 44100
    x = synth.track(30.0, fs, track_id=0)
    for s in (synth.c1_settings(), dict(synth.c1_settings(), bass_boost=0.0, mid_cut=0.0, presence_boost=0.0, treble_boost=0.0)):
        out, info = master(x, fs, s)
        ref, rinfo = chain.master(x, fs, s)
        assert _lufs_close(info["input_i"], rinfo["input_i"]) and info["measured_i_2dp"] == rinfo["measured_i_2dp"]
        assert _maxdiff(out, ref) <= NULL_LSB


def test_c5_shaped_192k_both_compressor_extremes(torch_cuda):
    """BASELINE config C5 shape (bursts, beds, exact-zero gaps, clicks) at 192 kHz, 60 s, thresh -40 / ratio 10 and
    thresh 0 / ratio 1, three 30 s-chunk boundaries... (two chunks)."""
    from audio_mastering_engine_b200 import master, synth
    from oracle import chain
    fs = 192000
    x = synth.stress_track(60.0, fs, track_id=4)
    for th, ra in ((-40.0, 10.0), (0.0, 1.0)):
        s = dict(synth.ALL_BOOST_EQ, analog_character=25, width=1.2, lufs=-14.0, multiband=True,
                 low_thresh=th, low_ratio=ra, mid_thresh=th, mid_ratio=ra, high_thresh=th, high_ratio=ra)
        out, info = master(x, fs, s)
        ref, rinfo = chain.master(x, fs, s)
        assert abs(info["input_i"] - rinfo["input_i"]) <= LUFS_TOL
        assert _maxdiff(out, ref) <= NULL_LSB, (th, ra, _maxdiff(out, ref))


def test_c4_slice_one_batch(torch_cuda):
    """BASELINE config C4, track ids 0-35 (every EQ preset x width x warmth x multiband combination of the sweep and
    two loudness targets), 30 s each, ONE batch in three waves and two workspace slots, every track against the oracle."""
    from audio_mastering_engine_b200 import master, synth, EQ_PRESETS
    from oracle import chain
    fs, secs = 48000, 30.0
    ids = list(range(36))
    tracks = [synth.track(secs, fs, track_id=t, am_hz=2.0) for t in ids]
    sets = [synth.c4_settings(t, EQ_PRESETS) for t in ids]
    sets += []
    outs, infos = master(tracks, fs, sets, n_waves=3, n_slots=2)
    worst = 0
    for t, x, s, out, info in zip(ids, tracks, sets, outs, infos):
        ref, rinfo = chain.master(x, fs, s)
        d = _maxdiff(out, ref)
        worst = max(worst, d)
        assert d <= NULL_LSB, (t, d)
        assert _lufs_close(info["input_i"], rinfo["input_i"]), t
        assert info["measured_i_2dp"] == rinfo["measured_i_2dp"], t
    print("C4 slice worst LSB diff", worst)


def _dist_worker(rank, world, port, backend, fs, seconds, chunk, out_dir, extra):
    import torch
    import torch.distributed as dist
    from audio_mastering_engine_b200 import sharding, synth
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    x = synth.track(seconds, fs, track_id=6, am_hz=1.0, drift_db=8.0, drift_period=3.0)
    begin, out, info = sharding.master_time_sharded(x, fs, dict(synth.c2_settings(), **extra), device=dev, chunk_seconds=chunk)
    np.save(os.path.join(out_dir, f"out{rank}.npy"), out)
    np.save(os.path.join(out_dir, f"meta{rank}.npy"), np.array([begin, info["input_i"] if info else np.nan, info["n_blocks"] if info else -1]))
    dist.barrier()
    dist.destroy_process_group()


def _run_dist(tmp_path, backend, world, fs=48000, seconds=7.0, chunk=1.0, extra=None):
    import socket
    import torch.multiprocessing as mp
    from audio_mastering_engine_b200 import master, synth
    sock = socket.socket(); sock.bind(("127.0.0.1", 0)); port = sock.getsockname()[1]; sock.close()
    extra = extra or {}
    mp.spawn(_dist_worker, args=(world, port, backend, fs, seconds, chunk, str(tmp_path), extra), nprocs=world, join=True)
    x = synth.track(seconds, fs, track_id=6, am_hz=1.0, drift_db=8.0, drift_period=3.0)
    one, info1 = master(x, fs, dict(synth.c2_settings(), **extra), chunk_seconds=chunk)
    parts = [np.load(tmp_path / f"out{r}.npy") for r in range(world)]
    metas = [np.load(tmp_path / f"meta{r}.npy") for r in range(world)]
    if extra.get("limiter"):        # the limiter runs on rank 0 over the gathered spans: rank 0 returns the whole track
        assert int(metas[0][0]) == 0 and all(len(q) == 0 for q in parts[1:])
    else:
        assert [int(m[0]) for m in metas] == list(np.cumsum([0] + [len(p) for p in parts[:-1]]))
    assert np.array_equal(np.concatenate(parts, axis=0), one)
    for m in metas:
        if m[2] >= 0:
            assert m[1] == pytest.approx(info1["input_i"], abs=1e-9) and int(m[2]) == info1["n_blocks"]


def test_shipped_time_sharded_path_two_processes_gloo(torch_cuda, tmp_path):
    """sharding.master_time_sharded - the function bench.py and INTEGRATION.md use - run by TWO processes that share
    this GPU, the halo hand-off and the histogram all-reduce going through torch.distributed (gloo): the concatenated
    spans must equal the single-plan result bit for bit.  (No kernel waits on another process's kernel.)"""
    _run_dist(tmp_path, "gloo", 2)
    _run_dist(tmp_path, "gloo", 3, fs=44100, seconds=4.0)          # an empty-span-free ragged split
    _run_dist(tmp_path, "gloo", 2, extra=dict(lufs=-9.0, limiter=True))      # + gather and the limiter on rank 0


def test_shipped_time_sharded_path_nccl(torch_cuda, tmp_path):
    """The same over NCCL, one process per GPU (skipped on a one-GPU box; bench.py --gpus N times it as time_sharded)."""
    if torch_cuda.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _run_dist(tmp_path, "nccl", 2)
    _run_dist(tmp_path, "nccl", 2, extra=dict(lufs=-9.0, limiter=True))


def _c_abi_shard_worker(rank, world, fs, seconds, chunk, out_dir):
    """One rank of examples/time_shard_nccl.c, driven through ctypes: its own ncclComm_t (created with libnccl's C API,
    no torch.distributed), ame_shard_halo_exchange + ame_hist_allreduce from libame."""
    import ctypes as C
    import glob
    import time
    import torch
    from audio_mastering_engine_b200 import MasterPlan, sharding, synth
    from audio_mastering_engine_b200 import _lib as L
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    cands = glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "nccl", "lib", "libnccl.so.2"))
    nccl = C.CDLL(cands[0] if cands else "libnccl.so.2", mode=C.RTLD_GLOBAL)

    class UniqueId(C.Structure):
        _fields_ = [("internal", C.c_char * 128)]
    uid = UniqueId()
    path = os.path.join(out_dir, "nccl_id.bin")
    if rank == 0:
        assert nccl.ncclGetUniqueId(C.byref(uid)) == 0
        with open(path + ".tmp", "wb") as fh:
            fh.write(bytes(uid))
        os.rename(path + ".tmp", path)
    else:
        for _ in range(600):
            if os.path.exists(path):
                break
            time.sleep(0.05)
        C.memmove(C.byref(uid), open(path, "rb").read(), 128)
    comm = C.c_void_p()
    nccl.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, UniqueId, C.c_int]
    assert nccl.ncclCommInitRank(C.byref(comm), world, uid, rank) == 0

    x = synth.track(seconds, fs, track_id=6, am_hz=1.0, drift_db=8.0, drift_period=3.0)
    spans = sharding.plan_time_shards(len(x), fs, world, chunk)
    b, e = spans[rank]
    halo = sharding.halo_frames(fs) if rank > 0 else 0
    plan = MasterPlan([e - b], fs, synth.c2_settings(), device=rank, chunk_seconds=chunk, halos=[halo])
    tf = plan.total_frames
    d_in = torch.zeros((tf, 2), dtype=torch.int16, device=dev)
    d_in[halo:halo + e - b] = torch.from_numpy(np.ascontiguousarray(x[b:e])).to(dev)
    d_pre, d_out = torch.zeros_like(d_in), torch.zeros_like(d_in)
    d_bands = torch.zeros((3, max(plan.mb_frames, 1), 2), dtype=torch.int16, device=dev)
    d_hist = torch.zeros((1, 1000), dtype=torch.int64, device=dev)
    lib, h = plan.lib, plan.handle
    plan.stage_eq(d_in, d_pre); plan.stage_band_split(d_pre, d_bands); plan.stage_compress(d_bands, d_pre)
    L.check(lib.ame_shard_halo_exchange(h, C.c_void_p(d_pre.data_ptr()), comm, rank - 1 if rank > 0 else -1,
                                        rank + 1 if rank + 1 < world else -1, sharding.halo_frames(fs), None))
    plan.stage_loudness_hist(d_pre, d_hist)
    L.check(lib.ame_hist_allreduce(h, C.c_void_p(d_hist.data_ptr()), comm, None))
    info = plan.stage_apply_gain(d_pre, d_hist, d_out)[0]
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, f"out{rank}.npy"), d_out[halo:halo + e - b].cpu().numpy())
    np.save(os.path.join(out_dir, f"meta{rank}.npy"), np.array([b, info["input_i"], info["n_blocks"]]))
    plan.close()
    nccl.ncclCommDestroy.argtypes = [C.c_void_p]
    nccl.ncclCommDestroy(comm)


def test_c_abi_time_shard_entry_points_nccl(torch_cuda, tmp_path):
    """ame_shard_halo_exchange + ame_hist_allreduce (the by-time path for a host that is not Python) on two GPUs with a
    communicator made by libnccl's own C API: bit-identical to the single-plan result."""
    if torch_cuda.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from audio_mastering_engine_b200 import master, synth
    fs, seconds, chunk, world = 48000, 6.0, 1.0, 2
    mp.spawn(_c_abi_shard_worker, args=(world, fs, seconds, chunk, str(tmp_path)), nprocs=world, join=True)
    x = synth.track(seconds, fs, track_id=6, am_hz=1.0, drift_db=8.0, drift_period=3.0)
    one, info1 = master(x, fs, synth.c2_settings(), chunk_seconds=chunk)
    parts = [np.load(tmp_path / f"out{r}.npy") for r in range(world)]
    assert np.array_equal(np.concatenate(parts, axis=0), one)
    for r in range(world):
        m = np.load(tmp_path / f"meta{r}.npy")
        assert m[1] == pytest.approx(info1["input_i"], abs=1e-9) and int(m[2]) == info1["n_blocks"]
