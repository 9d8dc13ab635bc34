"""Host mirror of the reference's mastering path on top of libame (include/ame.h).

Public surface (same names / argument meaning / error behaviour as audio_mastering_engine.py):
  EQ_PRESETS                                              :32-38
  process_audio(settings, status_cb, progress_cb, art_cb, tag_cb)              :94-137
  process_audio_with_ffmpeg_pipeline(settings, status_cb, progress_cb) -> path :171-226
plus the in-memory API used by tests and benchmarks:
  master(samples, fs, settings) -> (int16[N,2], info)
  measure_loudness(samples, fs) -> EBU R128 report of tracks that are not mastered
  MasterPlan - a reusable batch plan (packed layout, coefficients, device workspace).
There is no CPU fallback: without libame.so or without a CUDA device these raise.
"""
from __future__ import annotations

import ctypes as C
import logging
import math
import os
import traceback
import wave

import numpy as np

from . import _lib as L
from . import design
from .design import EQ_PRESETS  # noqa: F401  (re-exported: mastering_gui.py:11 imports it from the engine)

log = logging.getLogger("audio_mastering_engine_b200")


def _align8(n):
    return (int(n) + 7) // 8 * 8


def _loudness_dict(r):
    """One ame_loudness as a dict; tp is the true peak in dBTP."""
    return dict(integrated=r.integrated, thresh=r.thresh, lra=r.lra, true_peak=r.true_peak,
                tp=20.0 * math.log10(r.true_peak) if r.true_peak > 0 else -math.inf, sample_peak=int(r.sample_peak),
                n_blocks=int(r.n_blocks), max_momentary=r.max_momentary, max_short_term=r.max_short_term)


# the names a meter reading goes by in a mastering report (loudnorm's second-pass output_*) and in measure_loudness()
OUTPUT_KEYS = dict(integrated="output_i", tp="output_tp", lra="output_lra", thresh="output_thresh",
                   true_peak="output_true_peak", sample_peak="output_sample_peak", n_blocks="output_n_blocks",
                   max_momentary="output_max_momentary", max_short_term="output_max_short_term")
INPUT_KEYS = dict(integrated="input_i", tp="input_tp", lra="input_lra", thresh="input_thresh", true_peak="true_peak",
                  sample_peak="sample_peak", n_blocks="n_blocks", max_momentary="max_momentary", max_short_term="max_short_term")


def output_report(m):
    """A meter reading (MasterPlan.output_loudness / measure_loudness entry) under the output_* keys of results()."""
    return {OUTPUT_KEYS[k]: v for k, v in m.items()}


class MasterPlan:
    """Packed batch of tracks + per-track settings bound to one CUDA device.

    lengths[i] frames of track i are stored at frames [offsets[i], offsets[i] + lengths[i]) of ONE
    interleaved int16 stereo buffer of ``total_frames`` frames (offsets are multiples of 8).
    """

    def __init__(self, lengths, sample_rates, settings_list, device=0, chunk_seconds=30, host_io=False,
                 eq_tile_frames=0, xover_tile_frames=0, kw_tile_subblocks=0, halos=None, n_waves=1, chain_warps=0,
                 n_slots=0, precision="exact"):
        self.lib = L.load()
        n = len(lengths)
        if n == 0:
            raise ValueError("empty batch")
        if np.isscalar(sample_rates):
            sample_rates = [sample_rates] * n
        if isinstance(settings_list, dict):
            settings_list = [settings_list] * n
        self.lengths = [int(x) for x in lengths]
        self.sample_rates = [int(x) for x in sample_rates]
        self.settings = list(settings_list)
        # time shards carry `halo` frames of the previous shard's pre-normalisation tail in front of their span
        self.halos = [0] * n if halos is None else [int(h) for h in halos]
        self.offsets, off = [], 0
        for ln, h in zip(self.lengths, self.halos):
            self.offsets.append(off)
            off += _align8(ln + h)
        lut_index = {}
        arr = (L.TrackParams * n)()
        for i in range(n):
            arr[i] = design.track_params(self.settings[i], self.sample_rates[i], self.lengths[i], self.offsets[i],
                                         chunk_seconds, lut_index, self.halos[i])
        self.params = arr
        opt = L.PlanOptions(int(eq_tile_frames), int(xover_tile_frames), int(kw_tile_subblocks), 1 if host_io else 0,
                            int(n_waves), int(chain_warps), int(n_slots),
                            {"exact": 0, "fp32": 1}[precision])
        h = C.c_void_p()
        L.check(self.lib.ame_plan_create(int(device), arr, n, C.byref(opt), C.byref(h)))
        self.handle = h
        self.device = int(device)
        self.n_tracks = n
        self.total_frames = int(self.lib.ame_plan_total_frames(h))
        if lut_index:
            luts = np.empty((len(lut_index), 65536), dtype=np.float32)
            for ac, idx in lut_index.items():
                luts[idx] = design.warm_lut(ac)
            L.check(self.lib.ame_plan_set_warm_luts(h, luts.ctypes.data_as(C.c_void_p), len(lut_index)))
        self._results = (L.TrackResult * n)()
        # the output meter: tracks whose settings have "measure_output"
        self._loudness = (L.Loudness * n)() if any(arr[i].flags & L.AME_F_MEASURE_OUTPUT for i in range(n)) else None

    # -- lifetime -----------------------------------------------------------------------------
    def close(self):
        if getattr(self, "handle", None):
            self.lib.ame_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- packing helpers ------------------------------------------------------------------------
    def pack(self, tracks, out=None):
        """list of int16[N_i,2] -> one packed int16[total_frames,2] host array."""
        if out is None:
            out = np.zeros((self.total_frames, 2), dtype=np.int16)
        for t, off, ln, h in zip(tracks, self.offsets, self.lengths, self.halos):
            out[off + h:off + h + ln] = t
        return out

    def unpack(self, packed):
        return [np.array(packed[off + h:off + h + ln], copy=True)
                for off, ln, h in zip(self.offsets, self.lengths, self.halos)]

    def results(self):
        """Per-track loudness report: the numbers ffmpeg's loudnorm prints as JSON (audio_mastering_engine.py:229-237),
        plus whether real ffmpeg would have stayed in LINEAR mode (static gain) - this build always applies the
        static gain (DESIGN.md, deviation D3).  Tracks with settings["measure_output"] also carry loudnorm's output_*
        keys.  Both sides are those of the last call that fetched results (master_host, or master_device /
        normalize_device with fetch_results=True); after a call with fetch_results=False, output_loudness() reads that
        call's meter."""
        out = []
        for k, (r, s) in enumerate(zip(self._results, self.settings)):
            d = dict(input_i=r.input_i, measured_i_2dp=r.measured_i_2dp, gain=r.gain,
                     rel_threshold_energy=r.rel_threshold, n_blocks=int(r.n_blocks),
                     normalized=bool(r.normalized), sample_peak=int(r.sample_peak),
                     input_lra=r.input_lra, input_thresh=r.input_thresh, true_peak=r.true_peak,
                     true_peak_measured=bool(s.get("true_peak")))
            # ffmpeg reports the sample peak of the stream resampled to 192 kHz; this is the BS.1770 Annex 2 4x
            # oversampled peak when settings["true_peak"] is set, else the native-rate sample peak (deviation D4)
            d["input_tp"] = 20.0 * math.log10(r.true_peak) if r.true_peak > 0 else -math.inf
            if r.normalized:
                offset = float(s.get("lufs")) - r.measured_i_2dp
                d["target_offset"] = offset
                d["linear_mode_ok"] = bool(d["input_tp"] + offset <= -1.5 and r.input_lra <= 11.0)   # TP=-1.5:LRA=11 (:229)
            if self._loudness is not None and self._loudness[k].measured:
                d.update(output_report(_loudness_dict(self._loudness[k])))    # loudnorm's second-pass output_*
            out.append(d)
        return out

    def _fetch_loudness(self, stream=None):
        if self._loudness is not None:
            L.check(self.lib.ame_plan_output_loudness(self.handle, self._loudness, C.c_void_p(stream or 0)))

    def output_loudness(self, stream=None):
        """EBU R128 meter of the final output of the last master_device / master_host / normalize_device call: per track
        a dict (integrated, thresh, lra, true_peak, tp, sample_peak, n_blocks, max_momentary, max_short_term), or None
        for a track without settings["measure_output"] or before any call.  `stream` must be ordered after that call."""
        if self._loudness is None:
            return [None] * self.n_tracks
        self._fetch_loudness(stream)
        return [_loudness_dict(r) if r.measured else None for r in self._loudness]

    def measure_loudness(self, d_buf, stream=None):
        """The stand-alone meter: the same report for the flagged tracks of any CUDA int16 buffer in this plan's packed
        layout (synchronous).  Raises when no track has settings["measure_output"]."""
        res = (L.Loudness * self.n_tracks)()
        L.check(self.lib.ame_measure_loudness(self.handle, self._ptr(d_buf), res, C.c_void_p(stream or 0)))
        return [_loudness_dict(r) if r.measured else None for r in res]

    @property
    def launch_count(self):
        return int(self.lib.ame_plan_launch_count(self.handle))

    @property
    def workspace_bytes(self):
        return int(self.lib.ame_plan_workspace_bytes(self.handle))

    @property
    def n_waves(self):
        return int(self.lib.ame_plan_wave_count(self.handle))

    @property
    def n_slots(self):
        return int(self.lib.ame_plan_slot_count(self.handle))

    def limiter_stats(self):
        """Limiter tiles whose guessed start state was wrong after round 0 / 1 / 2, since the last query."""
        v = (C.c_int64 * 3)()
        L.check(self.lib.ame_plan_limiter_stats(self.handle, v))
        return [int(x) for x in v]

    def set_limiter_guess(self, frames=-1):
        """Test knob: frames the limiter's round-0 guess of a tile's start state runs over (-1 = the default 2 G;
        0 = no guess, a wrong start on every clipping tile).  Changes how much repair work runs, never the output."""
        L.check(self.lib.ame_plan_set_limiter_guess(self.handle, int(frames)))

    def chain_stats(self):
        """Compressor recurrence of the last call: chains, flagged steps (total, longest chain), passes (total, max)."""
        v = [C.c_int64() for _ in range(4)]
        mp = C.c_int32()
        L.check(self.lib.ame_plan_chain_stats(self.handle, *[C.byref(x) for x in v], C.byref(mp)))
        return dict(chains=v[0].value, steps=v[1].value, max_steps=v[2].value, passes=v[3].value, max_passes=mp.value)

    # -- the path -------------------------------------------------------------------------------
    @staticmethod
    def _ptr(x):
        if hasattr(x, "data_ptr"):
            return C.c_void_p(x.data_ptr())
        if isinstance(x, np.ndarray):
            return x.ctypes.data_as(C.c_void_p)
        return C.c_void_p(int(x))

    def master_device(self, d_in, d_out, stream=None, fetch_results=True):
        """d_in / d_out: CUDA int16 tensors (or raw device pointers) of total_frames*2 samples."""
        res = self._results if fetch_results else None
        L.check(self.lib.ame_master_device(self.handle, self._ptr(d_in), self._ptr(d_out), res, C.c_void_p(stream or 0)))
        if fetch_results:
            self._fetch_loudness(stream)
        return self.results() if fetch_results else None

    def master_host(self, h_in, h_out):
        """h_in / h_out: host int16 arrays (numpy, or pinned torch CPU tensors) in the packed layout."""
        L.check(self.lib.ame_master_host(self.handle, self._ptr(h_in), self._ptr(h_out), self._results))
        self._fetch_loudness()                             # master_host returns synchronised, meter included
        return self.results()

    def measure_device(self, d_in, d_hist, stream=None):
        L.check(self.lib.ame_measure_device(self.handle, self._ptr(d_in), self._ptr(d_hist), C.c_void_p(stream or 0)))

    def normalize_device(self, d_hist, d_out, stream=None, fetch_results=True):
        res = self._results if fetch_results else None
        L.check(self.lib.ame_normalize_device(self.handle, self._ptr(d_hist), self._ptr(d_out), res, C.c_void_p(stream or 0)))
        if fetch_results:
            self._fetch_loudness(stream)
        return self.results() if fetch_results else None

    def set_timing(self, enable=True):
        L.check(self.lib.ame_plan_set_timing(self.handle, 1 if enable else 0))

    def kernel_times(self):
        """{kernel name: (summed ms, launches)} and the number of recorded steps since set_timing()."""
        ms = (C.c_double * L.AME_N_KERNELS)()
        cnt = (C.c_int64 * L.AME_N_KERNELS)()
        steps = C.c_int(0)
        L.check(self.lib.ame_plan_kernel_times(self.handle, ms, cnt, C.byref(steps)))
        names = [self.lib.ame_kernel_name(i).decode() for i in range(L.AME_N_KERNELS)]
        return {n: (ms[i], int(cnt[i])) for i, n in enumerate(names)}, steps.value

    def wave_timeline(self):
        """Rows (h2d_done, kernels_may_start, kernels_done, d2h_done) in ms, one per wave, of the last master_host()
        made with timing enabled."""
        buf = (C.c_float * (4 * 256))()
        n = self.lib.ame_plan_wave_timeline(self.handle, buf, 256)
        if n < 0:
            L.check(n)
        return [tuple(buf[4 * w + k] for k in range(4)) for w in range(n)]

    def kernel_timeline(self, step=0):
        """[{kernel name: (begin ms, end ms)} per wave] of timed step `step` (see ame_plan_kernel_timeline)."""
        nk, nw = L.AME_N_KERNELS, 128
        buf = (C.c_float * (2 * nk * nw))()
        n = self.lib.ame_plan_kernel_timeline(self.handle, int(step), buf, nw)
        if n < 0:
            L.check(n)
        names = [self.lib.ame_kernel_name(i).decode() for i in range(nk)]
        return [{names[k]: (buf[(w * nk + k) * 2], buf[(w * nk + k) * 2 + 1]) for k in range(nk)
                 if buf[(w * nk + k) * 2] == buf[(w * nk + k) * 2]} for w in range(n)]      # NaN = not launched

    # stage entry points (parity taps)
    def stage_eq(self, d_in, d_pre, stream=None):
        L.check(self.lib.ame_stage_eq(self.handle, self._ptr(d_in), self._ptr(d_pre), C.c_void_p(stream or 0)))

    def stage_band_split(self, d_pre, d_bands, stream=None):
        L.check(self.lib.ame_stage_band_split(self.handle, self._ptr(d_pre), self._ptr(d_bands), C.c_void_p(stream or 0)))

    def stage_compress(self, d_bands, d_pre, stream=None):
        L.check(self.lib.ame_stage_compress(self.handle, self._ptr(d_bands), self._ptr(d_pre), C.c_void_p(stream or 0)))

    def stage_loudness_hist(self, d_pre, d_hist, stream=None):
        L.check(self.lib.ame_stage_loudness_hist(self.handle, self._ptr(d_pre), self._ptr(d_hist), C.c_void_p(stream or 0)))

    def stage_apply_gain(self, d_pre, d_hist, d_out, stream=None):
        L.check(self.lib.ame_stage_apply_gain(self.handle, self._ptr(d_pre), self._ptr(d_hist), self._ptr(d_out),
                                              self._results, C.c_void_p(stream or 0)))
        return self.results()

    def stage_limiter(self, d_norm, d_out, stream=None):
        """ffmpeg alimiter alone over an already normalised int16 signal (every track needs settings["limiter"])."""
        L.check(self.lib.ame_stage_limiter(self.handle, self._ptr(d_norm), self._ptr(d_out), C.c_void_p(stream or 0)))

    @property
    def mb_frames(self):
        return int(self.lib.ame_plan_mb_frames(self.handle))

    def mb_offset(self, track):
        return int(self.lib.ame_plan_mb_offset(self.handle, int(track)))

    def subblock_offset(self, track):
        return int(self.lib.ame_plan_subblock_offset(self.handle, int(track)))

    def read_tap(self, name, count, dtype):
        """Copy `count` elements of a workspace tap to a numpy array (tests / debugging)."""
        out = np.empty(int(count), dtype=dtype)
        L.check(self.lib.ame_plan_read_device(self.handle, out.ctypes.data_as(C.c_void_p), C.c_void_p(self.tap_ptr(name)),
                                              out.nbytes))
        return out

    def tap_ptr(self, name):
        fn = {"pre": self.lib.ame_plan_tap_pre, "bands": self.lib.ame_plan_tap_bands,
              "subblock_energy": self.lib.ame_plan_tap_subblock_energy}[name]
        return int(fn(self.handle) or 0)


def _as_stereo_pcm(x):
    x = np.asarray(x)
    if x.dtype != np.int16:
        raise TypeError("samples must be int16 (the reference forces 16-bit, audio_mastering_engine.py:191)")
    if x.ndim == 1:
        x = np.stack([x, x], axis=1)                      # set_channels(2) duplicates mono (:190)
    if x.ndim != 2 or x.shape[1] != 2:
        raise ValueError("samples must have shape [N] or [N,2]")
    return np.ascontiguousarray(x)


def master(samples, fs, settings, device=0, chunk_seconds=30, **plan_opts):
    """In-memory form of the hot path: split -> per-chunk chain -> concat -> normalise.

    samples: int16[N,2] (or [N] mono), or a list of such arrays (a batch; fs / settings may then be
    lists too).  Returns (out, info) or (list of out, list of info)."""
    single = not isinstance(samples, (list, tuple))
    tracks = [_as_stereo_pcm(samples)] if single else [_as_stereo_pcm(s) for s in samples]
    n = len(tracks)
    fs_list = [fs] * n if np.isscalar(fs) else list(fs)
    st_list = [settings] * n if isinstance(settings, dict) else list(settings)
    plan = MasterPlan([t.shape[0] for t in tracks], fs_list, st_list, device=device, chunk_seconds=chunk_seconds,
                      host_io=True, **plan_opts)
    try:
        if n == 1 and plan.total_frames == tracks[0].shape[0]:     # one track that is its own packed buffer: no copies
            h_out = np.empty_like(tracks[0])
            infos = plan.master_host(tracks[0], h_out)
            outs = [h_out]
        else:
            h_in = plan.pack(tracks)
            h_out = np.empty_like(h_in)
            infos = plan.master_host(h_in, h_out)
            outs = plan.unpack(h_out)
        for i in infos:
            i["launches"] = plan.launch_count
    finally:
        plan.close()
    return (outs[0], infos[0]) if single else (outs, infos)


def _meter(tracks, fs, device=0):
    """Stand-alone EBU R128 meter of int16 tracks (numpy arrays or torch tensors, [N,2] or mono [N]) on `device`: a plan
    whose tracks carry only the meter flag, the tracks uploaded into its packed layout.  One dict per track (see
    MasterPlan.output_loudness)."""
    import torch
    dev = torch.device("cuda", device)
    ts = []
    for x in tracks:
        x = x if isinstance(x, torch.Tensor) else torch.from_numpy(_as_stereo_pcm(x))
        if x.dtype != torch.int16:
            raise TypeError("samples must be int16")
        if x.ndim == 1:
            x = torch.stack([x, x], dim=1)
        if x.ndim != 2 or x.shape[1] != 2:
            raise ValueError("samples must have shape [N] or [N,2]")
        ts.append(x)
    n = len(ts)
    fs_list = [fs] * n if np.isscalar(fs) else list(fs)
    plan = MasterPlan([t.shape[0] for t in ts], fs_list, {"lufs": None, "measure_output": True}, device=device, chunk_seconds=None)
    try:
        buf = torch.zeros((plan.total_frames, 2), dtype=torch.int16, device=dev)
        for t, off in zip(ts, plan.offsets):
            buf[off:off + t.shape[0]] = t.to(dev)
        with torch.cuda.device(dev):
            return plan.measure_loudness(buf, stream=torch.cuda.current_stream(dev).cuda_stream)
    finally:
        plan.close()


def measure_loudness(samples, fs, device=0):
    """EBU R128 / BS.1770 meter on the GPU without mastering anything: integrated loudness (input_i, LUFS), relative gate
    (input_thresh), loudness range (input_lra), true peak (true_peak linear, input_tp dBTP; BS.1770 Annex 2 below 192 kHz),
    sample_peak, n_blocks and the maxima of the momentary and short-term loudness.  samples: int16[N,2] (or [N] mono,
    numpy or torch), or a list of such tracks (fs may then be a list too).  Returns a dict, or a list of dicts."""
    single = not isinstance(samples, (list, tuple))
    ms = _meter([samples] if single else list(samples), fs, device)
    out = [{INPUT_KEYS[k]: v for k, v in m.items()} for m in ms]
    return out[0] if single else out


LIMITER_KEYS = ("limiter", "limiter_limit", "limiter_attack", "limiter_release")


def limit_device(d_norm, fs, settings=None, device=None):
    """The reference's last stage alone (ffmpeg alimiter, audio_mastering_engine.py:223) on ONE track that is already
    normalised: int16[N,2] CUDA tensor -> new int16[N,2] CUDA tensor.  A time-sharded track ends with this call on the
    rank that gathers its spans (sharding.master_time_sharded): the limiter is one sequential state machine over the
    whole track, so its shards cannot carry it."""
    import torch
    st = {k: v for k, v in (settings or {}).items() if k in LIMITER_KEYS}
    st["limiter"] = True
    device = d_norm.device.index if device is None else device
    n = int(d_norm.shape[0])
    plan = MasterPlan([n], fs, st, device=device, chunk_seconds=None)
    try:
        src = d_norm
        if plan.total_frames != n:                        # the packed buffer is padded to whole groups of 8 frames
            src = torch.zeros((plan.total_frames, 2), dtype=torch.int16, device=d_norm.device)
            src[:n] = d_norm
        out = torch.empty_like(src)
        plan.stage_limiter(src, out)
        torch.cuda.synchronize(d_norm.device)
    finally:
        plan.close()
    return out[:n]


def release_cached_memory(device=0):
    """Plans take their workspace from a per-device pool that keeps the memory of closed plans for the next one;
    this hands it back to the driver."""
    L.check(L.load().ame_release_cached_memory(int(device)))


def bind_host_to_gpu_numa(device=0):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so that the pinned host buffers it allocates
    afterwards (and the threads that fill them) are local to the GPU's PCIe root: with one process per GPU on a
    two-socket box, buffers that all land on socket 0 send half of the H2D / D2H traffic across the socket link.
    Returns the node, or None when the topology cannot be read (then nothing is changed)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(device)
        name = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{name}/numa_node") as f:
            node = int(f.read())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except (OSError, ValueError, AttributeError, RuntimeError):
        return None


# ------------------------------------------------------------------------------------------------
# file boundary: stdlib wave instead of ffmpeg / pydub (SURVEY.md 8(f) row 2)
# ------------------------------------------------------------------------------------------------
def read_wav(path):
    with wave.open(path, "rb") as w:
        ch, sw, fs, n = w.getnchannels(), w.getsampwidth(), w.getframerate(), w.getnframes()
        raw = w.readframes(n)
    if sw == 2:
        x = np.frombuffer(raw, dtype="<i2")
    elif sw == 1:                                         # unsigned 8-bit -> 16-bit (set_sample_width(2), :191)
        x = ((np.frombuffer(raw, dtype=np.uint8).astype(np.int16) - 128) << 8).astype(np.int16)
    elif sw == 3:
        b = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 3)
        x = (b[:, 1].astype(np.int16) | (b[:, 2].astype(np.int8).astype(np.int16) << 8)).astype(np.int16)
    elif sw == 4:
        x = (np.frombuffer(raw, dtype="<i4") >> 16).astype(np.int16)
    else:
        raise ValueError(f"unsupported sample width {sw}")
    x = x.reshape(-1, ch)
    if ch == 1:
        x = np.repeat(x, 2, axis=1)                       # :190
    elif ch != 2:
        raise ValueError("only mono or stereo input is supported")
    return np.ascontiguousarray(x), fs


def write_wav(path, pcm, fs):
    with wave.open(path, "wb") as w:
        w.setnchannels(2)
        w.setsampwidth(2)
        w.setframerate(int(fs))
        w.writeframes(np.ascontiguousarray(pcm, dtype="<i2").tobytes())


def process_audio_with_ffmpeg_pipeline(settings, status_callback, progress_callback):
    """Drop-in for audio_mastering_engine.py:171-226 (same callback sequence, same ValueError): split -> per-chunk
    chain -> concat -> two-pass loudness normalisation -> alimiter -> WAV.  The whole file is mastered by ONE call,
    so the per-chunk status lines (the reference emits each when the chunk STARTS, :186-187) are emitted before it.
    ffmpeg's loudnorm leaves linear mode (static gain) when measured_TP + offset > -1.5 dBTP or LRA > 11; this build
    always applies the static gain (DESIGN.md, deviation D3) and says so through status_callback and the log."""
    input_file, output_file = settings.get("input_file"), settings.get("output_file")
    if not input_file or not output_file:
        raise ValueError("Input or output file not specified.")
    status_callback("Splitting audio into manageable chunks...")
    progress_callback(0, 100)
    pcm, fs = read_wav(input_file)
    chunk_frames = 30 * fs
    num_chunks = max(1, math.ceil(pcm.shape[0] / chunk_frames))
    total_steps = num_chunks + 4
    status_callback("Splitting complete.")
    run = dict(settings)
    run.setdefault("limiter", True)                       # the reference always ends with alimiter (:223)
    run.setdefault("true_peak", True)                     # needed to tell whether ffmpeg would have stayed in linear mode
    for i in range(num_chunks):
        status_callback(f"Processing chunk {i+1} of {num_chunks}...")
        progress_callback(i + 1, total_steps)
    try:
        out, info = master(pcm, fs, run)
    except Exception:
        logging.exception("CRITICAL: Failed during processing.")
        raise
    status_callback("Re-assembling processed chunks with concat filter...")
    progress_callback(num_chunks + 1, total_steps)
    status_callback("Concatenation complete.")
    if settings.get("lufs") is not None:
        status_callback("Normalizing final loudness...")
        progress_callback(num_chunks + 2, total_steps)
        if not info["normalized"]:
            log.warning("Measured loudness is -inf (silent audio). Skipping normalization.")
        elif not info.get("linear_mode_ok", True):
            msg = (f"Note: input true peak {info['input_tp']:.2f} dBTP + offset {info['target_offset']:.2f} dB / LRA "
                   f"{info['input_lra']:.1f} LU: ffmpeg loudnorm would switch to dynamic mode here; the static gain "
                   f"{20 * math.log10(info['gain']):+.2f} dB was applied and the limiter catches the overshoot.")
            log.warning(msg)
            status_callback(msg)
    status_callback("Applying final limiting and exporting...")
    progress_callback(num_chunks + 3, total_steps)
    write_wav(output_file, out, fs)
    if settings.get("measure_output"):
        msg = (f"Final loudness: {info['output_i']:.2f} LUFS integrated, {info['output_tp']:.2f} dBTP true peak, "
               f"LRA {info['output_lra']:.1f} LU")
        log.info(msg)
        status_callback(msg)
    progress_callback(total_steps, total_steps)
    log.info("Finished GPU pipeline, exported to %s", output_file)
    return output_file


def process_audio(settings, status_callback, progress_callback, art_callback, tag_callback):
    """Drop-in for audio_mastering_engine.py:94-137, mastering part only: never raises; failures are
    reported through the four callbacks exactly as the reference does (:131-137).  MP3 export, the AI
    tagger and cover-art generation are out of scope (DESIGN.md)."""
    try:
        process_audio_with_ffmpeg_pipeline(settings, status_callback, progress_callback)
        status_callback("Mastering complete. Preparing for AI analysis...")
        status_callback("Success: Processing complete! (No art generated)")
        art_callback(None)
    except Exception as e:
        log.error("FATAL ERROR in process_audio: %s", traceback.format_exc())
        status_callback(f"Error: {e}")
        progress_callback(0, 1)
        art_callback(None)
        tag_callback("Processing failed.")
