"""k_eq time per stereo frame for every template variant the C4 sweep uses (and a few more), each as a batch of
identical tracks - the data behind eq_cost_per_frame() in csrc/ame_layout.h (tiles are sized so that every thread of a launch
does the same amount of work; a wrong relative cost leaves the cheap tracks' warps idle at the end of the launch)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, torch
from audio_mastering_engine_b200 import MasterPlan, synth, EQ_PRESETS

dev = torch.device("cuda", 0)
fs, secs, n_tr = 48000, 60.0, 96
n = int(fs * secs)
base = synth.torch_track_batch(4, secs, fs, dev, first_track_id=0)
presets = [("none", {"bass_boost": 0.0, "mid_cut": 0.0, "presence_boost": 0.0, "treble_boost": 0.0})] + list(EQ_PRESETS.items()) + \
          [("shelf_only", {"bass_boost": 2.0, "mid_cut": 0.0, "presence_boost": 0.0, "treble_boost": 1.0}),
           ("one_peak", {"bass_boost": 0.0, "mid_cut": 2.0, "presence_boost": 0.0, "treble_boost": 0.0})]
print("preset warm width  ms  ns_per_frame_thread  rel")
rows = []
for name, eq in presets:
    for warm in (0, 25):
        for width in (1.0, 1.2):
            s = dict(eq, analog_character=warm, width=width, lufs=-14.0, multiband=False)
            plan = MasterPlan([n] * n_tr, fs, s, n_waves=1)
            d_in = torch.zeros((plan.total_frames, 2), dtype=torch.int16, device=dev)
            v = d_in.view(n_tr, -1, 2)
            for k in range(n_tr):
                v[k, :n] = base[k % 4]
            d_out = torch.empty_like(d_in)
            for _ in range(2):
                plan.master_device(d_in, d_out, fetch_results=False)
            torch.cuda.synchronize()
            plan.set_timing(True)
            for _ in range(4):
                plan.master_device(d_in, d_out, fetch_results=False)
            torch.cuda.synchronize()
            kt, _ = plan.kernel_times()
            ms = kt["k_eq"][0] / max(kt["k_eq"][1], 1)
            rows.append((name, warm, width, ms))
            plan.close()
ref = min(r[3] for r in rows)
for name, warm, width, ms in rows:
    print(f"{name:18s} {warm:3d} {width:4.1f} {ms:8.3f} {ms * 1e6 / (n_tr * n) * 37888:10.2f} {ms / ref:6.2f}")
