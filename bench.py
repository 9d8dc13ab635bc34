#!/usr/bin/env python
"""Benchmark of the mastering DSP chain (BASELINE.json metric: audio-seconds mastered per wall-second).

  python bench.py [--gpus N] [--steps K] [--warmup W]                      # this build, N GPUs of one node
  python bench.py ... --dump-outputs DIR                                    # + the last timed step's output as DIR/*.npy
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...                                      # the reference's CPU path

Workload (config.workload): BASELINE config C4 - the batch of 1024 synthetic 3 min stereo 48 kHz tracks with the
C4 settings sweep, sharded BY TRACK over the N GPUs (1024 / N tracks per GPU, no data-path collective): STRONG
scaling, the same 1024 tracks at every N.  A step = one pass of the whole chain (warmth + EQ + width + multiband
compressor + BS.1770 loudness + gain) over the rank's tracks.
  value    : device-resident (inputs already in HBM), CUDA-event timed, max over ranks.
  e2e      : the same tracks through the public host API (ame_master_host via MasterPlan.master_host) with pinned
             HOST buffers: H2D + chain + D2H inside the timed region; beside it the raw concurrent H2D + D2H rate of
             the same buffers on the same ranks (the ceiling the host path can reach on this box).
  roofline : per kernel from a SERIALISED pass (a one-slot plan: waves follow each other on one stream, so the kernel
             times add up to the step), DRAM traffic per launch from the tracked ncu export under profiles/.
  parity_check : three tracks of the timed batch mastered by the CPU oracle, outside the timed region.
  --dump-outputs : the mastered audio of the last timed step (rank 0's tracks at a fixed, seeded sample of frame
             positions, see dump_outputs), so that two builds can be compared output for output on identical inputs.
  time_sharded : (N > 1) BASELINE config C3 - one 60 min 96 kHz track split BY TIME over the N GPUs, halo hand-off
             between neighbours + ONE NCCL all-reduce of the int64[1000] loudness histogram - timed on the device and
             compared bit for bit with the single-plan result.
"""
from __future__ import annotations

import argparse
import csv
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "audio-sec mastered/sec (x realtime)"
UNIT = "x realtime"
B_ALG_CHAIN = 16       # bytes per stereo frame, whole chain with normalisation (SURVEY.md 8(d))
KERNEL_ALG_BYTES = {   # per-kernel algorithmic bytes per frame it processes (DESIGN.md section 4)
    "k_eq": 8, "k_band_split": 16, "k_window_flag": 18, "k_att_chain": 6, "k_compress_apply": 16,
    "k_kweight_energy": 4, "k_apply_gain": 8}
ALL_TRACK_KERNELS = ("k_eq", "k_kweight_energy", "k_apply_gain", "k_limiter", "k_true_peak")   # the others see multiband tracks only
NCU_CSV = os.path.join(ROOT, "profiles", "r02", "ncu_kernels.csv")
DUMP_VALUES = 8 << 20  # int16 samples --dump-outputs keeps (stored as float32: 32 MB)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tracks", type=int, default=1024, help="tracks of the whole job (BASELINE C4: 1024), split over the GPUs")
    ap.add_argument("--tracks-per-gpu", type=int, default=0, help="weak-scaling variant: this many tracks on every GPU")
    ap.add_argument("--seconds", type=float, default=180.0)
    ap.add_argument("--fs", type=int, default=48000)
    ap.add_argument("--wave-tracks", type=int, default=0, help="tracks per plan wave (0 = 32, or a sixth of the rank's tracks if fewer than 192)")
    ap.add_argument("--slots", type=int, default=8, help="workspace slots = waves in flight")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-wave-tracks", type=int, default=8)
    ap.add_argument("--e2e-slots", type=int, default=4)
    ap.add_argument("--chain-warps", type=int, default=0, help="ame_plan_options.chain_warps (0 = auto, -1 = sequential loop)")
    ap.add_argument("--cpu-sample-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-serial-pass", action="store_true")
    ap.add_argument("--serial-wave-tracks", type=int, default=128, help="tracks per launch of the serialised (roofline) pass: the "
                    "launch shape of the tracked ncu capture")
    ap.add_argument("--no-time-sharded", action="store_true")
    ap.add_argument("--time-sharded-seconds", type=float, default=3600.0)
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU's NUMA node")
    ap.add_argument("--kw-tile", type=int, default=0, help="ame_plan_options.kw_tile_subblocks (0 = auto)")
    ap.add_argument("--eq-tile", type=int, default=0, help="ame_plan_options.eq_tile_frames (0 = auto)")
    ap.add_argument("--xover-tile", type=int, default=0, help="ame_plan_options.xover_tile_frames (0 = auto)")
    ap.add_argument("--precision", default="exact", choices=["exact", "fp32"])
    ap.add_argument("--limiter", action="store_true", help="also run the final alimiter stage (:223; not part of north_star (a)-(d))")
    ap.add_argument("--true-peak", action="store_true", help="also measure the BS.1770 true peak")
    ap.add_argument("--ablate", default="", help="experiments only (profiles/r02/ablation.txt): comma list of "
                    "nomb (no track multiband), allmb, noeq (EQ preset None, no warmth, width 1), nolufs")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write the mastered audio of the last timed step "
                    "(a seeded sample of frames of every track of rank 0) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index, period=0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._halt.wait(self.period)

    def finish(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """{kernel: (dram bytes per frame the kernel processes, source)} from the tracked ncu export."""
    out = {}
    try:
        with open(NCU_CSV) as fh:
            for row in csv.DictReader(fh):
                out[row["kernel"]] = float(row["dram_bytes_per_frame"])
    except Exception:
        pass
    return out


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path (oracle port: numpy/scipy + pydub's Python loop on
    audioop), all host cores, bounded sample per step."""
    if rank != 0:
        return
    from oracle import cpu_arm
    cores = os.cpu_count() or 1
    pool = cpu_arm.make_pool(cores)
    ids = list(range(cores))
    secs, fs = args.cpu_sample_seconds, args.fs
    for _ in range(max(args.warmup, 1) if pool is not None else 0):
        cpu_arm.run_step(pool, ids[:cores], min(secs, 1.0), fs)      # warm the workers (imports, filter design)
    audio = wall = 0.0
    for _ in range(args.steps):
        a, w = cpu_arm.run_step(pool, ids, secs, fs)
        audio += a
        wall += w
    if pool is not None:
        pool.shutdown()
    value = audio / wall
    sample = (f"{cores} tracks x {secs:g} s of the C4 sweep per step, one per core, {args.steps} steps; "
              "ffmpeg split/concat/loudnorm/alimiter substituted by the oracle's restatements (binary absent)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C4: batch of 1024 synthetic 3 min stereo 48 kHz tracks, settings sweep (bounded CPU sample)",
                       "fs": fs, "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def batch_order(ids, synth, presets):
    """The rank's tracks as a host batcher would queue them: multiband and plain tracks alternate in runs of 4, so
    that every wave holds both kinds (the latency-bound compressor kernels of a wave run under FP64-bound filters)."""
    mb = [t for t in ids if synth.c4_settings(t, presets)["multiband"]]
    nb = [t for t in ids if not synth.c4_settings(t, presets)["multiband"]]
    out = []
    while mb or nb:
        out += mb[:4] + nb[:4]
        mb, nb = mb[4:], nb[4:]
    return out


def fill_batch(torch, synth, d_in, ids, n, secs, fs, dev, block=32):
    """Synthesise the tracks `ids` (C4 recipe, seed = 20260 + id) straight into the packed device buffer."""
    view = d_in.view(len(ids), -1, 2)
    for k in range(0, len(ids), block):
        for j, t in enumerate(ids[k:k + block]):
            view[k + j, :n] = synth.torch_track_batch(1, secs, fs, dev, first_track_id=t)[0]


def dump_outputs(path, torch, np, d_out, offsets, n, ids):
    """What a caller of master_device receives, the packed int16 output, sampled: every track at the same frame
    positions (all n when they fit in DUMP_VALUES, else a sorted draw of a fixed-seed generator), values as float32.
      output.npy          [tracks, frames, 2]  float32, the int16 samples
      output_frame.npy    [frames]             float64, frame position within each track
      output_track_id.npy [tracks]             float64, the synthetic track id (input seed) of each row"""
    k = min(n, DUMP_VALUES // (2 * len(offsets)))
    frames = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    dev = d_out.device
    idx = torch.tensor(offsets, dtype=torch.int64, device=dev)[:, None] + torch.from_numpy(frames).to(dev)[None, :]
    out = d_out[idx.reshape(-1)].reshape(len(offsets), k, 2).float().cpu().numpy()
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "output.npy"), out)
    np.save(os.path.join(path, "output_frame.npy"), frames.astype(np.float64))
    np.save(os.path.join(path, "output_track_id.npy"), np.asarray(ids, dtype=np.float64))


def run_time_sharded(args, torch, dist, rank, world, dev):
    """BASELINE config C3 through sharding.time_sharded_step: one long 96 kHz track split by time over the ranks."""
    from audio_mastering_engine_b200 import synth, sharding, MasterPlan
    fs, secs = 96000, args.time_sharded_seconds
    s = synth.c2_settings()
    track = synth.torch_track_batch(1, secs, fs, dev, first_track_id=7)[0]          # same seed on every rank: same track
    spans = sharding.plan_time_shards(track.shape[0], fs, world, 30)
    sh = sharding.TimeShard(spans[rank], fs, s, rank, world, dev.index, 30)
    sh.load(track[spans[rank][0]:spans[rank][1]])
    for _ in range(2):                                                              # warm-up (NCCL p2p channels, tiles)
        out, info, moved = sharding.time_sharded_step(sh, spans)
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        out, info, moved = sharding.time_sharded_step(sh, spans)
    e1.record()
    dist.barrier(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    mine = out.clone()
    sh.close()
    # the same track as ONE plan on this GPU: every rank checks its own span bit for bit
    plan = MasterPlan([track.shape[0]], fs, s, device=dev.index)
    d_out = torch.empty_like(track)
    ref_info = plan.master_device(track, d_out)[0]
    plan.close()
    ref = d_out[spans[rank][0]:spans[rank][1]]
    n_diff = torch.tensor([int((mine != ref).any(dim=1).sum().item())], device=dev)
    max_diff = torch.tensor([int((mine.int() - ref.int()).abs().max().item()) if mine.numel() else 0], device=dev)
    dist.all_reduce(n_diff, op=dist.ReduceOp.SUM)
    dist.all_reduce(max_diff, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    return {"config": f"C3: one {secs:g} s stereo {fs} Hz track split by time over {world} GPUs (30 s chunks, "
                      f"{len(sharding.plan_time_shards(track.shape[0], fs, world, 30))} spans)",
            "ms": ms, "value": secs / (ms * 1e-3), "unit": UNIT, "collective": "NCCL all_reduce(sum) int64[1000] + neighbour send/recv of the halo",
            "allreduce_bytes": 8000, "halo_bytes_per_rank": int(sh.send) * 4, "bytes_moved_rank0": int(moved),
            "bit_identical_to_single_plan": int(n_diff.item()) == 0, "frames_differing_from_single_plan": int(n_diff.item()),
            "frames": int(track.shape[0]), "max_abs_diff_lsb": int(max_diff.item()),
            "note": "shards and single plan tile the time-parallel filters differently; at 96 kHz the 250 Hz low-pass sections keep "
                    "an FP64 round-off floor of 1e-14 of full scale between any two tilings, so about one sample in 1e9 truncates "
                    "to the neighbouring int16 (x the make-up gain) - DESIGN.md section 6, profiles/r02/tiling_sensitivity.txt",
            "input_i": info["input_i"], "single_plan_input_i": ref_info["input_i"]}


def run_b200(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from audio_mastering_engine_b200 import MasterPlan, synth, EQ_PRESETS, bind_host_to_gpu_numa

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = None if args.no_numa_bind else bind_host_to_gpu_numa(local_rank)   # before any pinned allocation
    if world > 1:
        # NCCL writes its version banner to stdout when the communicator is created: send fd 1 to stderr until the
        # first collective is through, so that stdout carries nothing but the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    fs, secs = args.fs, args.seconds
    n = int(round(secs * fs))
    if args.tracks_per_gpu > 0:
        scaling, n_tr, first = "weak", args.tracks_per_gpu, rank * args.tracks_per_gpu
        total_tracks = n_tr * world
    else:
        from audio_mastering_engine_b200.sharding import shard_tracks
        scaling, total_tracks = "strong", args.tracks
        mine = shard_tracks(total_tracks, world, rank)
        n_tr, first = len(mine), mine.start
    ids = batch_order(list(range(first, first + n_tr)), synth, EQ_PRESETS)
    settings = [dict(synth.c4_settings(t, EQ_PRESETS), limiter=args.limiter, true_peak=args.true_peak) for t in ids]
    for a in filter(None, args.ablate.split(",")):
        over = {"nomb": dict(multiband=False), "allmb": dict(multiband=True), "nolufs": dict(lufs=None),
                "noeq": dict(bass_boost=0.0, mid_cut=0.0, presence_boost=0.0, treble_boost=0.0, analog_character=0, width=1.0)}[a]
        settings = [dict(s, **over) for s in settings]
    wave_tracks = args.wave_tracks if args.wave_tracks > 0 else (32 if n_tr >= 192 else max(1, -(-n_tr // 6)))
    n_waves = max(1, -(-n_tr // wave_tracks))
    plan_kw = dict(device=local_rank, chain_warps=args.chain_warps, kw_tile_subblocks=args.kw_tile,
                   eq_tile_frames=args.eq_tile, xover_tile_frames=args.xover_tile, precision=args.precision)
    plan = MasterPlan([n] * n_tr, fs, settings, n_waves=n_waves, n_slots=args.slots, **plan_kw)
    d_in = torch.zeros((plan.total_frames, 2), dtype=torch.int16, device=dev)
    fill_batch(torch, synth, d_in, ids, n, secs, fs, dev)
    d_out = torch.empty_like(d_in)
    stream = torch.cuda.current_stream().cuda_stream
    frames_rank = n_tr * n
    audio_rank = n_tr * secs

    for _ in range(max(args.warmup, 3)):
        plan.master_device(d_in, d_out, stream=stream, fetch_results=False)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        plan.master_device(d_in, d_out, stream=stream, fetch_results=False)
    e1.record()
    barrier()
    clocks = sampler.finish()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, np, d_out, plan.offsets, n, ids)
    launches = plan.launch_count * args.steps
    ms_max = allmax(ms)
    audio_total = total_tracks * secs
    value = audio_total * args.steps / (ms_max * 1e-3)
    infos = plan.master_device(d_in, d_out, stream=stream)             # one more pass, fetching the loudness results
    chain_stats = plan.chain_stats()
    if args.limiter:
        plan.limiter_stats()
        plan.master_device(d_in, d_out, stream=stream, fetch_results=False)
        chain_stats["limiter_open_tiles_after_round_0_1_2"] = plan.limiter_stats()
        chain_stats["limiter_tiles"] = n_tr * (-(-n // 8192))
    workspace_gb = round(plan.workspace_bytes / 1e9, 2)
    plan_slots, plan_waves, stride = plan.n_slots, plan.n_waves, plan.total_frames // n_tr
    plan.close()

    # ---- serialised pass: one slot => the waves follow each other on one stream and kernel times add up ----------
    peak, peak_src = measured_peak_gbs()
    mb_frames = sum(1 for s in settings if s["multiband"]) * n
    roofline = None
    if not args.no_serial_pass:
        ser_waves = max(1, -(-n_tr // max(args.serial_wave_tracks, 1)))
        splan = MasterPlan([n] * n_tr, fs, settings, n_waves=ser_waves, n_slots=1, **plan_kw)
        d_chk = torch.empty_like(d_out)
        splan.master_device(d_in, d_chk, stream=stream, fetch_results=False)
        torch.cuda.synchronize()
        splan.set_timing(True)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ser_steps = 3
        s0.record()
        for _ in range(ser_steps):
            splan.master_device(d_in, d_chk, stream=stream, fetch_results=False)
        s1.record()
        torch.cuda.synchronize()
        ser_ms = s0.elapsed_time(s1) / ser_steps
        ktimes, _ = splan.kernel_times()
        splan.set_timing(False)
        serial_equal = bool(torch.equal(d_chk, d_out))
        splan.close()
        del d_chk
        traffic = ncu_traffic()
        per_kernel = {}
        for name, (msum, cnt) in ktimes.items():
            if not cnt:
                continue
            step_ms = msum / ser_steps                                   # all launches of the kernel in one step
            fr = frames_rank if name in ALL_TRACK_KERNELS else mb_frames
            row = {"ms_per_step": round(step_ms, 4), "launches_per_step": cnt // ser_steps,
                   "share_of_step": round(step_ms / ser_ms, 4)}
            if name in KERNEL_ALG_BYTES:
                gbs = KERNEL_ALG_BYTES[name] * fr / (step_ms * 1e-3) / 1e9
                row.update(achieved=round(gbs, 1), frac=round(gbs / peak, 4),
                           algorithmic_bytes_per_launch=KERNEL_ALG_BYTES[name] * fr / max(cnt // ser_steps, 1))
                if name in traffic:
                    row["traffic_per_launch"] = traffic[name] * fr / max(cnt // ser_steps, 1)
            per_kernel[name] = row
        dom = max((k for k in per_kernel if "achieved" in per_kernel[k]), key=lambda k: per_kernel[k]["ms_per_step"])
        d = per_kernel[dom]
        chain_gbs = B_ALG_CHAIN * frames_rank * args.steps / (ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": d["achieved"], "peak": peak, "unit": "GB/s", "frac": d["frac"],
                    "traffic": d.get("traffic_per_launch"),
                    "traffic_source": ("dram__bytes_read.sum + dram__bytes_write.sum per frame from the tracked ncu export "
                                       "profiles/r02/ncu_kernels.csv (128-track capture), scaled to this launch's frames")
                                      if d.get("traffic_per_launch") else None,
                    "peak_source": peak_src, "kernel_ms": d["ms_per_step"] / max(d["launches_per_step"], 1),
                    "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"],
                    "chain": {"achieved": chain_gbs, "frac": chain_gbs / peak, "bytes_per_frame": B_ALG_CHAIN,
                              "note": "whole step of the timed (overlapped) run at 16 B per stereo frame"},
                    "serialised_pass": {"ms_per_step": round(ser_ms, 3), "sum_of_kernel_ms": round(sum(r["ms_per_step"] for r in per_kernel.values()), 3),
                                        "equals_timed_output": serial_equal,
                                        "waves": ser_waves,
                                        "note": "one-slot plan in waves of up to %d tracks (the launch shape of the ncu capture): every "
                                                "launch alone on the GPU, CUDA events on its stream" % args.serial_wave_tracks},
                    "per_kernel": per_kernel}

    # ---- parity: three tracks of the timed batch against the CPU oracle (outside every timed region) -------------
    parity = None
    if rank == 0 and not args.no_parity_check:
        from oracle import chain
        picks, seen = [], set()
        for k, s in enumerate(settings):                                 # a multiband + warmth one, a plain one, the loudest target
            key = ("mb" if s["multiband"] else "plain", s["lufs"] == -9.0)
            if key not in seen and len(picks) < 3:
                seen.add(key); picks.append(k)
        worst, lufs_err, rows = 0, 0.0, []
        for k in picks:
            x = d_in[k * stride:k * stride + n].cpu().numpy()
            got = d_out[k * stride:k * stride + n].cpu().numpy()
            ref, rinfo = chain.master(x, fs, settings[k])
            dlsb = int(np.abs(got.astype(np.int32) - ref.astype(np.int32)).max())
            worst = max(worst, dlsb)
            lufs_err = max(lufs_err, abs(infos[k]["input_i"] - rinfo["input_i"]))
            rows.append({"track_id": ids[k], "max_abs_diff_lsb": dlsb, "lufs_gpu": infos[k]["input_i"], "lufs_oracle": rinfo["input_i"]})
        parity = {"tracks": rows, "max_abs_diff_lsb": worst, "max_lufs_diff": lufs_err,
                  "tolerance": "<= 3 LSB (-80 dBFS), <= 0.01 LU", "ok": bool(worst <= 3 and lufs_err <= 0.01)}

    # ---- end to end through the host API: pinned host buffers, H2D + chain + D2H per step ------------------------
    e2e = None
    if not args.no_e2e:
        h_in = torch.empty((d_in.shape[0], 2), dtype=torch.int16, pin_memory=True)
        h_out = torch.empty_like(h_in, pin_memory=True)
        h_in.copy_(d_in)
        ref_out = d_out                                                  # the device-resident result, for the equality check
        torch.cuda.synchronize()
        # the raw ceiling first: all ranks copy their buffers in and out at the same time, nothing else running
        c_in, c_out = torch.cuda.Stream(), torch.cuda.Stream()
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            with torch.cuda.stream(c_in):
                d_in.copy_(h_in, non_blocking=True)                      # same bytes: d_in stays what it was
            with torch.cuda.stream(c_out):
                h_out.copy_(ref_out, non_blocking=True)
        torch.cuda.synchronize()
        copy_s = allmax(time.perf_counter() - t0) / 2
        d_in = None                                                      # the host plan brings its own device buffers
        torch.cuda.empty_cache()
        bytes_step = int(h_in.numel() * 2)
        ceiling_gbs = world * 2 * bytes_step / copy_s / 1e9             # aggregate, both directions
        e2e_waves = max(1, -(-n_tr // max(args.e2e_wave_tracks, 1)))
        hplan = MasterPlan([n] * n_tr, fs, settings, host_io=True, n_waves=e2e_waves, n_slots=args.e2e_slots, **plan_kw)
        hplan.master_host(h_in, h_out)                                   # warm-up
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            res = hplan.master_host(h_in, h_out)                         # synchronous: returns after D2H
        torch.cuda.synchronize()
        wall = allmax(time.perf_counter() - t0)
        same = bool(torch.equal(h_out.to(dev), ref_out))
        e2e_value = audio_total * args.e2e_steps / wall
        e2e = {"value": e2e_value, "unit": UNIT,
               "h2d_bytes_per_step": bytes_step * world, "d2h_bytes_per_step": (bytes_step + 64 * n_tr) * world,
               "steps": args.e2e_steps, "ms_per_step": 1e3 * wall / args.e2e_steps, "waves": e2e_waves, "slots": args.e2e_slots,
               "numa_node": numa_node, "matches_device_path": same, "first_track_lufs": res[0]["input_i"],
               "host_ceiling_gbs": round(ceiling_gbs, 1),
               "host_ceiling_note": "aggregate H2D + D2H rate of the same pinned buffers copied concurrently by all ranks, no kernels",
               "achieved_gbs": round(world * 2 * bytes_step * args.e2e_steps / wall / 1e9, 1),
               "frac_of_host_ceiling": round((world * 2 * bytes_step * args.e2e_steps / wall / 1e9) / ceiling_gbs, 3)}
        hplan.close()
        del h_in, h_out
        ref_out = None

    # ---- by-time path on the N GPUs (C3) --------------------------------------------------------------------------
    time_sharded = None
    if world > 1 and not args.no_time_sharded:
        d_in = d_out = ref_out = None
        torch.cuda.empty_cache()
        time_sharded = run_time_sharded(args, torch, dist, rank, world, dev)

    # ---- CPU baseline (rank 0, N=1 only): single thread, as the reference runs -----------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import cpu_arm
        a, w = cpu_arm.run_step(None, [0, 1, 2, 3], 5.0, fs)
        cpu = {"value": a / w, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "tracks 0-3 of the C4 sweep x 5 s each, sequential on one core (2 of 4 multiband); "
                         "oracle port = reference numpy/scipy stages + pydub Python loop on audioop; ffmpeg stages "
                         "substituted by the oracle's restatements (binary absent)",
               "host_cpus": os.cpu_count()}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": "f64" if args.precision == "exact" else "f32", "data": "synthetic",
                "config": {"workload": f"C4: {total_tracks} synthetic {secs:g} s stereo {fs} Hz tracks, C4 settings sweep, 30 s chunks, "
                                       f"sharded by track over {world} GPU(s) ({n_tr} tracks on rank 0)",
                           "tracks": total_tracks, "tracks_rank0": n_tr, "seconds": secs, "fs": fs, "chunk_seconds": 30,
                           "parallelism": f"by-track x{world}, no data-path collective", "plan_waves": plan_waves, "plan_slots": plan_slots,
                           "l2": f"inputs larger than L2 ({frames_rank * 4 / 1e9:.2f} GB per GPU per pass)"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "parity_check": parity, "time_sharded": time_sharded, "workspace_gb": workspace_gb,
                "workspace_over_input": round(workspace_gb / (frames_rank * 4 / 1e9), 2), "chain_stats": chain_stats}
        if args.ablate:
            line["config"]["ablation"] = args.ablate + " (an experiment on a changed workload, not a bench value)"
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
