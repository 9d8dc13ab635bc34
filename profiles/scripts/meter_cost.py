#!/usr/bin/env python
"""Cost of the EBU R128 output meter (settings["measure_output"], AME_F_MEASURE_OUTPUT) on one GPU.

  python profiles/scripts/meter_cost.py [--steps 5] [--warmup 2] [--reps 3] [--out FILE]

1. The bench's plan (bench.py defaults: the 1024 C4 tracks of 3 min at 48 kHz in bench order, 32 waves of 32 tracks,
   8 workspace slots, no limiter, no true peak) with and without measure_output on every track, alternated --reps
   times: ms per step (CUDA events around --steps ame_master_device calls, after --warmup), and the meter's overhead.
   The int16 outputs of the two plans and their input-side reports must be identical.
2. The stand-alone meter: ame_measure_loudness alone over the same 1024 tracks (the mastered output), in x realtime.
The card's name and power limit are read in the same run (nvidia-smi query) and printed with the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable ({e})"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=180.0)
    ap.add_argument("--fs", type=int, default=48000)
    ap.add_argument("--wave-tracks", type=int, default=32)
    ap.add_argument("--slots", type=int, default=8)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--meter-calls", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    import bench
    from audio_mastering_engine_b200 import EQ_PRESETS, MasterPlan, release_cached_memory, synth
    if not torch.cuda.is_available():
        raise SystemExit("meter_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f"card: {card(0)} (torch: {torch.cuda.get_device_name(0)})")
    fs, n, n_tr = args.fs, int(round(args.seconds * args.fs)), args.tracks
    ids = bench.batch_order(list(range(n_tr)), synth, EQ_PRESETS)
    base = [dict(synth.c4_settings(t, EQ_PRESETS), limiter=False, true_peak=False) for t in ids]
    modes = {"off": base, "on": [dict(s, measure_output=True) for s in base]}
    n_waves = max(1, -(-n_tr // args.wave_tracks))
    say(f"workload: {n_tr} tracks x {args.seconds:g} s stereo {fs} Hz (bench.py's C4 batch), {n_waves} waves, {args.slots} slots; "
        f"{args.steps} timed steps after {args.warmup} warm-up steps per plan, plans alternated {args.reps} times")
    t0 = time.time()
    probe = MasterPlan([n] * n_tr, fs, base, n_waves=n_waves, n_slots=args.slots)
    total_frames, ws_off = probe.total_frames, probe.workspace_bytes
    probe.close()
    release_cached_memory(0)                       # the probe's workspace back to the driver, so that mem_get_info sees it
    d_in = torch.zeros((total_frames, 2), dtype=torch.int16, device=dev)
    bench.fill_batch(torch, synth, d_in, ids, n, args.seconds, fs, dev)
    outs = {"off": torch.empty_like(d_in)}
    free = torch.cuda.mem_get_info(dev)[0]
    exact = free > d_in.numel() * 2 + ws_off * 1.05 + (4 << 30)       # room for a second output buffer next to a plan
    outs["on"] = torch.empty_like(d_in) if exact else outs["off"]
    say(f"inputs ready in {time.time() - t0:.1f} s; output comparison: {'element by element' if exact else 'checksums (no room for two outputs)'}")
    stream = torch.cuda.current_stream(dev).cuda_stream
    ms = {"off": [], "on": []}
    reports, sums, meta = {}, {}, {}

    def checksum(x):
        v = x.view(-1)
        acc = [0, 0, 0]
        step = 1 << 28
        for lo in range(0, v.numel(), step):
            c = v[lo:lo + step].to(torch.int64)
            w = torch.arange(lo, lo + c.numel(), device=dev, dtype=torch.int64) % 65521 + 1
            acc[0] += int(c.sum()); acc[1] += int((c * c).sum()); acc[2] += int((c * w).sum())
        return tuple(acc)

    meter_ms = None
    for rep in range(args.reps):
        for mode in ("off", "on"):
            plan = MasterPlan([n] * n_tr, fs, modes[mode], n_waves=n_waves, n_slots=args.slots)
            out = outs[mode]
            for _ in range(args.warmup):
                plan.master_device(d_in, out, stream=stream, fetch_results=False)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                plan.master_device(d_in, out, stream=stream, fetch_results=False)
            e1.record()
            torch.cuda.synchronize()
            ms[mode].append(e0.elapsed_time(e1) / args.steps)
            if rep == 0:
                res = plan.master_device(d_in, out, stream=stream)
                reports[mode] = [{k: v for k, v in r.items() if not k.startswith("output_")} for r in res]
                meta[mode] = dict(launches=plan.launch_count, workspace_gb=plan.workspace_bytes / 1e9, waves=plan.n_waves, slots=plan.n_slots)
                if mode == "on":
                    assert all("output_i" in r for r in res)
                    # the stand-alone meter over the mastered output of every track
                    for _ in range(2):
                        plan.lib.ame_measure_loudness(plan.handle, C.c_void_p(out.data_ptr()), None, C.c_void_p(stream))
                    torch.cuda.synchronize()
                    e0.record()
                    for _ in range(args.meter_calls):
                        rc = plan.lib.ame_measure_loudness(plan.handle, C.c_void_p(out.data_ptr()), None, C.c_void_p(stream))
                        assert rc == 0, rc
                    e1.record()
                    torch.cuda.synchronize()
                    meter_ms = e0.elapsed_time(e1) / args.meter_calls
                    meta["meter_launches"] = plan.launch_count
                    alone = plan.measure_loudness(out, stream=stream)
                    assert all(a["integrated"] == r["output_i"] and a["true_peak"] == r["output_true_peak"] for a, r in zip(alone, res))
                if not exact:
                    sums[mode] = checksum(out)
            plan.close()
            say(f"rep {rep} meter {mode:3s}: {ms[mode][-1]:8.2f} ms/step")
    if exact:
        a, b, step = outs["off"].view(-1), outs["on"].view(-1), 1 << 28
        same_out = all(torch.equal(a[lo:lo + step], b[lo:lo + step]) for lo in range(0, a.numel(), step))
    else:
        same_out = sums["off"] == sums["on"]
    same_rep = reports["off"] == reports["on"]
    audio = n_tr * args.seconds
    say("")
    for mode in ("off", "on"):
        m = ms[mode]
        say(f"meter {mode:3s}: ms/step min {min(m):.2f} mean {sum(m) / len(m):.2f} max {max(m):.2f}  "
            f"({audio / (min(m) * 1e-3) / 1e3:.1f}k x realtime at the min); launches/step {meta[mode]['launches']}, "
            f"workspace {meta[mode]['workspace_gb']:.3f} GB, {meta[mode]['waves']} waves / {meta[mode]['slots']} slots")
    on, off = sum(ms["on"]) / len(ms["on"]), sum(ms["off"]) / len(ms["off"])
    say(f"overhead of the meter in the overlapped step: {on - off:+.2f} ms/step ({100 * (on - off) / off:+.2f} % of the mean; "
        f"min vs min {min(ms['on']) - min(ms['off']):+.2f} ms)")
    say(f"int16 outputs identical: {same_out}; input-side reports identical: {same_rep}")
    say(f"stand-alone meter (ame_measure_loudness, {n_tr} tracks, {meta['meter_launches']} launches): {meter_ms:.2f} ms per call = "
        f"{audio / (meter_ms * 1e-3) / 1e6:.2f}M x realtime")
    say(f"card (again, after the run): {card(0)}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    if not (same_out and same_rep):
        raise SystemExit("meter on / off changed the output or the input reports")


if __name__ == "__main__":
    main()
