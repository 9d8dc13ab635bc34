"""The plan layout (csrc/ame_layout.h) without a GPU: tests/plan_layout_driver.cpp is compiled with g++ alone (no nvcc, no
CUDA headers), runs build_layout on track parameters from design.track_params and prints every job table as JSON; the
tests check the invariants the kernels rely on."""
import json
import math
import os
import subprocess

import pytest

from audio_mastering_engine_b200 import _lib as L, design, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the device shape of a B200: 148 SMs; resident 128-thread CTAs per SM of k_eq and k_band_split<true>
# (cudaOccupancyMaxActiveBlocksPerMultiprocessor, CUDA 12.9, sm_100a)
N_SM, OCC_EQ, OCC_SPLIT = 148, 2, 3
AME_E_INVALID, AME_E_UNSUPPORTED = -1, -4      # include/ame.h


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("layout") / "plan_layout_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", os.path.join(ROOT, "tests", "plan_layout_driver.cpp"),
                           "-o", exe])
    return exe


def _align8(n):
    return (n + 7) // 8 * 8


def make_tracks(specs, chunk_seconds=30):
    """specs: (seconds, fs, settings[, halo_frames]) per track, packed one after the other as MasterPlan packs them."""
    arr = (L.TrackParams * len(specs))()
    lut, off = {}, 0
    for i, spec in enumerate(specs):
        secs, fs, s = spec[:3]
        halo = spec[3] if len(spec) > 3 else 0
        n = int(round(secs * fs))
        arr[i] = design.track_params(s, fs, n, off, chunk_seconds, lut, halo)
        off += _align8(n + halo)
    return arr


def run_layout(driver, tmp_path, tracks, n_waves=1, n_slots=0, host_io=False, eq_tile=0, xover_tile=0, kw_tile=0):
    (tmp_path / "tracks.bin").write_bytes(bytes(tracks))
    (tmp_path / "options.bin").write_bytes(bytes(L.PlanOptions(eq_tile, xover_tile, kw_tile, int(host_io), n_waves, 0, n_slots, 0)))
    out = subprocess.run([driver, str(tmp_path / "tracks.bin"), str(tmp_path / "options.bin"), str(N_SM), str(OCC_EQ),
                          str(OCC_SPLIT)], check=True, capture_output=True, text=True).stdout
    return json.loads(out)


RANGES = ("eq", "split", "chain", "wf", "mb_chunks", "kw", "gain", "lim")


def waves_of(lay):
    out = []
    for w in lay["waves"]:
        d = dict(zip(("track_lo", "track_hi", "frame_lo", "frame_hi", "seg_lo", "seg_hi", "slot", "limiter", "true_peak"), w[:9]))
        d.update(zip(RANGES, w[9:]))
        out.append(d)
    return out


def chunks_of(tp):
    """[begin, end) of every chunk of a track in the packed buffer."""
    cf = tp.chunk_frames if tp.chunk_frames > 0 else max(tp.n_frames, 1)
    base = tp.offset_frames + tp.halo_frames
    return [(base + c0, base + min(c0 + cf, tp.n_frames)) for c0 in range(0, tp.n_frames, cf)]


def check_layout(lay, tracks, n_waves, n_slots):
    assert lay["rc"] == 0, lay["error"]
    sc = lay["scalars"]
    n = len(tracks)
    waves = waves_of(lay)
    mb = [bool(t.flags & L.AME_F_MULTIBAND) for t in tracks]

    # waves: contiguous non-empty track ranges, frame ranges from the track offsets, every table covered in order
    assert len(waves) == min(n_waves, n) and sc["n_slots"] == n_slots
    assert waves[0]["track_lo"] == 0 and waves[-1]["track_hi"] == n
    for k, w in enumerate(waves):
        assert w["track_lo"] < w["track_hi"] and w["slot"] == k % n_slots
        assert w["frame_lo"] == tracks[w["track_lo"]].offset_frames
        assert w["frame_hi"] == (tracks[w["track_hi"]].offset_frames if w["track_hi"] < n else sc["total_frames"])
        if k:
            assert w["track_lo"] == waves[k - 1]["track_hi"] and w["seg_lo"] == waves[k - 1]["seg_hi"]
        assert w["limiter"] == any(tracks[t].flags & L.AME_F_LIMITER for t in range(w["track_lo"], w["track_hi"]))
        assert w["true_peak"] == any(tracks[t].flags & L.AME_F_TRUE_PEAK for t in range(w["track_lo"], w["track_hi"]))
    for name in RANGES:
        pos = 0
        for w in waves:
            lo, cnt = w[name]
            assert lo == pos and cnt >= 0, name
            pos += cnt
        assert pos == len(lay[name]), name
    assert sc["total_frames"] == max(8, max(_align8(t.offset_frames + t.halo_frames + t.n_frames) for t in tracks))
    assert sc["slot_frames"] == max(w["frame_hi"] - w["frame_lo"] for w in waves)

    def wave_rows(w, name):
        lo, cnt = w[name]
        return lay[name][lo:lo + cnt]

    def track_range(w):
        return range(w["track_lo"], w["track_hi"])

    # k_eq: per chunk, the non-empty tiles cover it once and in order; whole warps of one variant; empty padding jobs
    for w in waves:
        rows = wave_rows(w, "eq")
        assert len(rows) % 32 == 0
        for g in range(0, len(rows), 32):
            assert len({r[4] for r in rows[g:g + 32]}) == 1
        for t in track_range(w):
            tiles = [r for r in rows if r[3] == t and r[2] > r[1]]
            for cb, ce in chunks_of(tracks[t]):
                mine = [r for r in tiles if r[0] == cb]
                assert mine and mine[0][1] == cb and mine[-1][2] == ce
                for a, b in zip(mine, mine[1:]):
                    assert a[2] == b[1]
                assert all(r[2] == ce or r[2] % 8 == 0 for r in mine)
            assert sum(r[2] - r[1] for r in tiles) == tracks[t].n_frames
        assert all(r[1] == r[2] for r in rows if not r[2] > r[1])

    # k_band_split: multiband tracks only, each chunk exactly once, no tile longer than the split tile
    for w in waves:
        rows = wave_rows(w, "split")
        assert all(mb[r[3]] for r in rows)
        for t in track_range(w):
            mine = [r for r in rows if r[3] == t]
            if not mb[t]:
                continue
            cover = [(r[1], r[2]) for r in mine]
            exp = 0
            for cb, ce in chunks_of(tracks[t]):
                part = [c for c in cover if cb <= c[0] < ce]
                assert part[0][0] == cb and part[-1][1] == ce
                for a, b in zip(part, part[1:]):
                    assert a[1] == b[0]
                exp += len(part)
            assert exp == len(mine)
        assert all(r[2] - r[1] <= sc["split_tile"] for r in rows)

    # compressor chains: three bands per multiband chunk, longest first, disjoint group ranges, valid tables;
    # ceil(n / kWfTile) k_window_flag tiles per chain pointing back at it
    n_tables = sc["n_att_tables"]
    for w in waves:
        rows = wave_rows(w, "chain")
        n_chunks = sum(len(chunks_of(tracks[t])) for t in track_range(w) if mb[t])
        assert len(rows) == 3 * n_chunks and sorted(r[3] for r in rows) == sorted([0, 1, 2] * n_chunks)
        assert all(a[1] >= b[1] for a, b in zip(rows, rows[1:]))
        spans = sorted((r[2], r[2] + (r[1] + 31) // 32) for r in rows)
        for a, b in zip(spans, spans[1:]):
            assert a[1] <= b[0]
        assert all(0 <= s[0] and s[1] <= sc["slot_groups"] for s in spans)
        assert all(0 <= r[4] < n_tables for r in rows)
        wf = wave_rows(w, "wf")
        pos = 0
        for c, r in enumerate(rows):
            tiles = math.ceil(r[1] / 2048)
            assert r[7] == pos
            mine = wf[pos:pos + tiles]
            assert [j[0] for j in mine] == list(range(0, r[1], 2048))
            assert all(j[4] == w["chain"][0] + c and j[7] == pos and j[2] == r[1] and j[3] == r[2] for j in mine)
            assert all(j[1] == r[3] * sc["mb_frames"] + r[0] for j in mine)
            pos += tiles
        assert pos == len(wf)

    # per-track coverage: K-weighting sub-blocks, gain tiles, limiter tiles
    tdev = lay["tdev"]
    for w in waves:
        kw, gain, lim = wave_rows(w, "kw"), wave_rows(w, "gain"), wave_rows(w, "lim")
        for t in track_range(w):
            tp = tracks[t]
            base = tp.offset_frames + tp.halo_frames
            mine = [r for r in kw if r[0] == t]
            assert (mine[0][1] if mine else 0) == 0 and (mine[-1][2] if mine else 0) == tdev[t][1]
            assert all(a[2] == b[1] for a, b in zip(mine, mine[1:]))
            mine = [r[:2] for r in gain if r[2] == t]
            assert mine == [[base + b, base + min(b + 32768, tp.n_frames)] for b in range(0, tp.n_frames, 32768)]
            mine = [r[:2] for r in lim if r[2] == t]
            if tp.flags & L.AME_F_LIMITER:
                shift = tdev[t][6]
                assert shift >= 13 and 2 ** shift >= tp.lim_frames + tp.lim_release_frames + 8
                assert shift == 13 or 2 ** (shift - 1) < tp.lim_frames + tp.lim_release_frames + 8
                tile = 2 ** shift
                assert mine == [[base + b, base + min(b + tile, tp.n_frames)] for b in range(0, tp.n_frames, tile)]
                first = [i for i, r in enumerate(lim) if r[2] == t][0]
                assert tdev[t][4] == first
            else:
                assert not mine

    # multiband packing: from 0 in every wave, in track order, 8-aligned; -1 elsewhere; mb_frames = the largest wave's
    mb_off, largest = lay["mb_offset"], 0
    for w in waves:
        pos = 0
        for t in track_range(w):
            if mb[t]:
                assert mb_off[t] == pos and lay["mb_delta"][t] == pos - tracks[t].offset_frames
                pos += _align8(tracks[t].halo_frames + tracks[t].n_frames)
            else:
                assert mb_off[t] == -1 and lay["mb_delta"][t] == 0
        largest = max(largest, pos)
    assert sc["mb_frames"] == largest
    assert sc["any_limiter"] == any(bool(t.flags & L.AME_F_LIMITER) for t in tracks)
    assert all(0 <= x < n_tables for t, row in enumerate(lay["tracks"]) if mb[t] for x in row)


def mixed_batch():
    c2 = synth.c2_settings()
    return [(40.0, 44100, c2), (7.0, 48000, synth.c1_settings()), (65.0, 96000, c2), (20.0, 192000, synth.c1_settings()),
            (3.0, 44100, dict(c2, limiter=True, true_peak=True)), (31.0, 48000, {"lufs": -14.0}),
            (12.0, 96000, dict(synth.c1_settings(), limiter=True)), (9.0, 48000, dict(c2, low_thresh=-30.0))]


@pytest.mark.parametrize("n_waves,n_slots", [(1, 1), (3, 1), (3, 2)])
@pytest.mark.parametrize("chunk_seconds", [30, 1, 0.5])
def test_mixed_batch(driver, tmp_path, n_waves, n_slots, chunk_seconds):
    tracks = make_tracks(mixed_batch(), chunk_seconds)
    lay = run_layout(driver, tmp_path, tracks, n_waves=n_waves, n_slots=n_slots)
    check_layout(lay, tracks, n_waves, n_slots)


def test_host_io_plan_starts_with_a_one_track_wave(driver, tmp_path):
    specs = [(4.0 + k, [44100, 48000][k % 2], synth.c2_settings() if k % 3 else synth.c1_settings()) for k in range(10)]
    tracks = make_tracks(specs)
    lay = run_layout(driver, tmp_path, tracks, n_waves=4, host_io=True)
    check_layout(lay, tracks, 4, 4)
    waves = waves_of(lay)
    assert waves[0]["track_hi"] - waves[0]["track_lo"] == 1
    assert all(w["track_hi"] - w["track_lo"] >= 2 for w in waves[1:])
    plain = waves_of(run_layout(driver, tmp_path, tracks, n_waves=4))
    assert plain[0]["track_hi"] - plain[0]["track_lo"] > 1


def test_time_shard_with_halo(driver, tmp_path):
    fs = 48000
    halo = 30 * (fs // 10)                    # 3 s: whole 100 ms sub-blocks and a multiple of 8
    tracks = make_tracks([(60.0, fs, synth.c2_settings(), halo)])
    lay = run_layout(driver, tmp_path, tracks)
    check_layout(lay, tracks, 1, 1)
    sb_offset, n_sb, s100, first_block = lay["tdev"][0][:4]
    assert (sb_offset, s100, n_sb) == (0, 4800, (halo + 60 * fs) // 4800) and first_block == halo // 4800 - 3
    assert lay["eq"][0][0] == halo and lay["gain"][0][0] == halo


def test_requested_tiles(driver, tmp_path):
    tracks = make_tracks(mixed_batch()[:4])
    lay = run_layout(driver, tmp_path, tracks, eq_tile=1000, xover_tile=3000, kw_tile=4)
    check_layout(lay, tracks, 1, 1)
    assert lay["scalars"]["split_tile"] == 3000 and lay["scalars"]["kw_tile_sb"] == 4
    assert all(r[2] - r[1] <= 1000 for r in lay["eq"])


def _bad(field):
    tracks = make_tracks([(2.0, 48000, dict(synth.c2_settings(), limiter=True)), (2.0, 48000, synth.c1_settings())])
    field(tracks)
    return tracks


@pytest.mark.parametrize("edit,code,text", [
    (lambda t: setattr(t[1], "offset_frames", t[1].offset_frames + 4), AME_E_INVALID, "track 1: offset_frames must be a non-negative multiple of 8"),
    (lambda t: setattr(t[1], "offset_frames", 0), AME_E_INVALID, "tracks overlap in the packed buffer"),
    (lambda t: (setattr(t[0], "offset_frames", t[1].offset_frames), setattr(t[1], "offset_frames", 0)), AME_E_INVALID,
     "tracks must be ordered by offset_frames"),
    (lambda t: setattr(t[1], "halo_frames", 800), AME_E_INVALID, "track 1: halo_frames must be a multiple of 8 and of the 100 ms sub-block"),
    (lambda t: setattr(t[0], "halo_frames", 4800), AME_E_UNSUPPORTED, "track 0: the limiter is one sequential state machine"),
    (lambda t: setattr(t[1].eq[0].s[0], "b1", t[1].eq[0].s[0].b1 * 1.5), AME_E_UNSUPPORTED,
     "track 1: a filter section is not of Butterworth shape"),
    (lambda t: setattr(t[0].xhp[1], "b0", 0.5), AME_E_UNSUPPORTED, "track 0: a filter section is not of Butterworth shape"),
    (lambda t: setattr(t[0], "lim_frames", 0), AME_E_INVALID, "track 0: bad limiter parameters (look-ahead 0 frames"),
    (lambda t: setattr(t[0], "lim_release_frames", 1 << 20), AME_E_INVALID, "track 0: bad limiter parameters"),
    (lambda t: setattr(t[0].comp[2], "attack_frames", 0.0), AME_E_INVALID, "track 0: bad compressor band 2"),
    (lambda t: setattr(t[0].comp[0], "look_frames", 5000), AME_E_INVALID, "track 0: bad compressor band 0"),
    (lambda t: setattr(t[1], "sample_rate", 4000), AME_E_INVALID, "track 1: unsupported sample rate 4000"),
])
def test_rejected_inputs(driver, tmp_path, edit, code, text):
    lay = run_layout(driver, tmp_path, _bad(edit))
    assert lay["rc"] == code and lay["error"].startswith(text), lay


def test_valid_inputs_of_the_rejection_cases(driver, tmp_path):
    tracks = _bad(lambda t: None)
    check_layout(run_layout(driver, tmp_path, tracks), tracks, 1, 1)
