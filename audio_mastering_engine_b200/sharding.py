"""Multi-GPU partitioning of the mastering path (one process per GPU, torch.distributed for the plumbing).

* by track (batches): tracks are independent - contiguous blocks of tracks per rank, NO collective.
* by time (one long track): in reference semantics every 30 s chunk restarts all filter / compressor state
  (audio_mastering_engine.py:185-199), so contiguous runs of chunks per rank are independent up to the
  pre-normalisation signal.  Loudness is global (the reference measures the concatenated file, :216-220):
    1. each rank masters its span up to the pre-normalisation int16 signal,
    2. it hands the last `halo` frames of that signal to the next rank (the halo warms the K-weighting filter
       up and completes the 400 ms gating blocks that straddle the boundary),
    3. each rank histograms the blocks that END in its span (ebur128 1000-bin histogram),
    4. ONE all-reduce(sum) of the int64[1000] histogram makes integrated loudness global,
    5. every rank derives the same gain and applies it to its span.
"""
from __future__ import annotations

import math

import numpy as np

from . import design


def shard_tracks(n_tracks: int, world: int, rank: int):
    """Contiguous block of track indices for `rank` (sizes differ by at most one)."""
    base, rem = divmod(int(n_tracks), int(world))
    lo = rank * base + min(rank, rem)
    return range(lo, lo + base + (1 if rank < rem else 0))


def sub_block_frames(fs: int) -> int:
    return (int(fs) + 5) // 10


def halo_frames(fs: int) -> int:
    """Frames of the previous shard's tail a shard needs: K-filter warm-up + the 3 sub-blocks that complete
    straddling 400 ms blocks, rounded so that it is a multiple of the sub-block and of 8 frames."""
    s100 = sub_block_frames(fs)
    n_sb = int(math.ceil(design.kw_warm_frames(int(fs)) / s100)) + 3
    step = 8 // math.gcd(s100, 8)
    n_sb = (n_sb + step - 1) // step * step
    return n_sb * s100


def plan_time_shards(n_frames: int, fs: int, world: int, chunk_seconds=30):
    """[(begin, end)] frame spans, one per rank: contiguous runs of whole chunks, as even as possible.
    Ranks that would get no chunk get an empty span at the end."""
    cf = int(chunk_seconds * fs)
    s100 = sub_block_frames(fs)
    if cf % s100:
        raise ValueError(f"time sharding needs the chunk ({cf} frames) to be a whole number of 100 ms sub-blocks "
                         f"({s100} frames) at {fs} Hz")
    n_chunks = max(1, math.ceil(n_frames / cf))
    spans = []
    for r in range(world):
        c = shard_tracks(n_chunks, world, r)
        lo, hi = min(c.start * cf, n_frames), min(c.stop * cf, n_frames)
        spans.append((lo, hi))
    return spans


class TimeShard:
    """One rank's part of a time-sharded track: a MasterPlan over [halo | span] plus the device buffers."""

    def __init__(self, span, fs, settings, rank, world, device=0, chunk_seconds=30, **plan_opts):
        import torch
        from .engine import MasterPlan
        self.torch = torch
        self.begin, self.end = span
        self.n = self.end - self.begin
        self.rank, self.world, self.fs = rank, world, int(fs)
        self.halo = halo_frames(fs) if (rank > 0 and self.begin > 0 and self.n > 0) else 0
        self.send = halo_frames(fs)                       # what the next rank expects from us
        self.dev = torch.device("cuda", device)
        self.plan = None
        if self.n > 0:
            self.plan = MasterPlan([self.n], fs, settings, device=device, chunk_seconds=chunk_seconds, halos=[self.halo],
                                   **plan_opts)
            tf = self.plan.total_frames
            self.d_in = torch.zeros((tf, 2), dtype=torch.int16, device=self.dev)
            self.d_pre = torch.zeros((tf, 2), dtype=torch.int16, device=self.dev)
            self.d_out = torch.zeros((tf, 2), dtype=torch.int16, device=self.dev)
            self.d_bands = torch.zeros((3, max(self.plan.mb_frames, 1), 2), dtype=torch.int16, device=self.dev)
        self.d_hist = torch.zeros((1, 1000), dtype=torch.int64, device=self.dev)

    def load(self, span_pcm):
        """span_pcm: int16[n,2] (numpy or tensor) - this rank's slice of the input track."""
        if self.n:
            t = self.torch.as_tensor(span_pcm)
            self.d_in[self.halo:self.halo + self.n].copy_(t, non_blocking=True)

    def pre_normalisation(self, stream=None):
        """Steps 1: warmth / EQ / width / multiband over the span -> self.d_pre[halo:halo+n]."""
        if self.n:
            self.plan.stage_eq(self.d_in, self.d_pre, stream)
            self.plan.stage_band_split(self.d_pre, self.d_bands, stream)
            self.plan.stage_compress(self.d_bands, self.d_pre, stream)

    def tail(self):
        """Last `send` frames of this shard's pre-normalisation signal (what the next rank's halo holds).
        Shorter spans are left-padded with zeros: the reference's signal simply starts later."""
        out = self.torch.zeros((self.send, 2), dtype=self.torch.int16, device=self.dev)
        k = min(self.send, self.n + self.halo)            # may reach into our own halo when the span is short
        if k:
            out[self.send - k:] = self.d_pre[self.halo + self.n - k:self.halo + self.n]
        return out

    def set_halo(self, prev_tail):
        if self.halo:
            self.d_pre[:self.halo].copy_(prev_tail[-self.halo:])

    def histogram(self, stream=None):
        self.d_hist.zero_()
        if self.n:
            self.plan.stage_loudness_hist(self.d_pre, self.d_hist, stream)
        return self.d_hist

    def normalise(self, d_hist, stream=None):
        """Steps 5: gain from the (all-reduced) histogram; returns (int16[n,2] tensor, info)."""
        if not self.n:
            return self.torch.zeros((0, 2), dtype=self.torch.int16, device=self.dev), None
        info = self.plan.stage_apply_gain(self.d_pre, d_hist, self.d_out, stream)[0]
        if self.world > 1:                                # short-term (3 s) windows are not stitched across shards
            info["input_lra"] = None
            info.pop("linear_mode_ok", None)
        return self.d_out[self.halo:self.halo + self.n], info

    def close(self):
        if self.plan is not None:
            self.plan.close()
            self.plan = None


def _exchange_tail(sh, spans, group):
    """Halo hand-off between neighbours: every rank sends the tail of its pre-normalisation signal (a few 100 ms of
    audio) to the next rank and receives its predecessor's.  A rank without a span forwards what it received, so the
    next non-empty rank still gets the tail of the nearest non-empty rank before it.  One stereo frame travels as one
    int32 (NCCL has no int16)."""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    torch_dev = sh.dev if dist.get_backend(group) == "nccl" else torch.device("cpu")
    prev = None
    if rank > 0:
        prev = torch.empty((sh.send, 1), dtype=torch.int32, device=torch_dev)
        dist.recv(prev, src=dist.get_global_rank(group, rank - 1) if group is not None else rank - 1, group=group)
    if rank < world - 1:
        mine = sh.tail().view(torch.int32) if sh.n else prev
        if mine is None:                                  # rank 0 without a span: nothing precedes the track
            mine = torch.zeros((sh.send, 1), dtype=torch.int32, device=sh.dev)
        dist.send(mine.to(torch_dev).contiguous(), dst=dist.get_global_rank(group, rank + 1) if group is not None else rank + 1,
                  group=group)
    if sh.halo and prev is not None:
        sh.set_halo(prev.to(sh.dev).view(torch.int16))
    return int(sh.send) * 4 * ((rank > 0) + (rank < world - 1))


def time_sharded_step(sh, spans, group=None):
    """One pass of the by-time path over an already loaded TimeShard: pre-normalisation chain on the rank's span,
    neighbour halo hand-off, local 400 ms block histogram, ONE all-reduce(sum) of the int64[1000] histogram, gain.
    Returns (device int16[n,2] view, info, bytes this rank sent + received)."""
    import torch
    import torch.distributed as dist
    sh.pre_normalisation()
    moved = _exchange_tail(sh, spans, group)
    hist = sh.histogram()
    if dist.get_backend(group) == "nccl":
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=group)  # the one collective the math needs
    else:
        h = hist.cpu()
        dist.all_reduce(h, op=dist.ReduceOp.SUM, group=group)
        hist.copy_(h)
    out, info = sh.normalise(hist)
    return out, info, moved + 2 * hist.numel() * 8


def _shard_settings(settings):
    """What the shards run: everything but the limiter, which is one sequential machine over the whole track, and the
    output meter, which measures the whole track (a shard's output is not the track's output)."""
    st = dict(settings)
    st["limiter"] = False
    st.pop("measure_output", None)
    return st


def _with_output_report(info, full, fs, device):
    """info + the EBU R128 meter of the joined (and limited) track `full` under the output_* keys."""
    from .engine import _meter, output_report
    return dict(info or {}, **output_report(_meter([full], fs, device)[0]))


def _gather_spans(out, spans, group, dst=0):
    """All spans of the normalised track on rank `dst`, in order: int16[N,2] device tensor there, None elsewhere.
    (send / recv of each non-empty span; one stereo frame travels as one int32.)"""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    nccl = dist.get_backend(group) == "nccl"
    glob = (lambda r: dist.get_global_rank(group, r)) if group is not None else (lambda r: r)
    if rank != dst:
        if out.shape[0]:
            msg = out.contiguous().view(torch.int32)
            dist.send(msg if nccl else msg.cpu(), dst=glob(dst), group=group)
        return None
    total = spans[-1][1]
    full = torch.empty((total, 2), dtype=torch.int16, device=out.device)
    for r, (lo, hi) in enumerate(spans):
        if hi <= lo:
            continue
        if r == dst:
            full[lo:hi] = out
        else:
            buf = torch.empty((hi - lo, 1), dtype=torch.int32, device=out.device if nccl else "cpu")
            dist.recv(buf, src=glob(r), group=group)
            full[lo:hi] = buf.to(out.device).view(torch.int16)
    return full


def master_time_sharded(track, fs, settings, group=None, device=None, chunk_seconds=30, **plan_opts):
    """Master ONE long track across the ranks of `group` (torch.distributed; NCCL on GPUs, gloo moves the small
    messages through the host).  Every rank passes the same track (numpy or tensor; at least its own span must be
    valid); returns this rank's (span_begin, int16[n,2] numpy, info).

    With settings["limiter"] (the reference's alimiter, :223) the normalised spans are gathered on rank 0, which runs
    the limiter over the whole track (engine.limit_device - parallel in time on ONE GPU, but not across shards) and
    returns (0, the whole limited track, info); the other ranks return (span_begin, an empty array, info).

    With settings["measure_output"] the spans are gathered on rank 0 too, which meters the joined (and limited) track
    and adds the report to its info under the output_* keys of MasterPlan.results(); what each rank returns is as
    without it."""
    import torch
    import torch.distributed as dist
    from .engine import limit_device
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    device = torch.cuda.current_device() if device is None else device
    spans = plan_time_shards(len(track), fs, world, chunk_seconds)
    sh = TimeShard(spans[rank], fs, _shard_settings(settings), rank, world, device, chunk_seconds, **plan_opts)
    span = track[spans[rank][0]:spans[rank][1]]
    sh.load(span if hasattr(span, "device") else np.ascontiguousarray(span))
    out, info, _ = time_sharded_step(sh, spans, group)
    measure = bool(settings.get("measure_output"))
    if settings.get("limiter"):
        full = _gather_spans(out, spans, group)
        sh.close()
        if full is None:
            return spans[rank][0], np.zeros((0, 2), dtype=np.int16), info
        full = limit_device(full, fs, settings, device)
        if measure:
            info = _with_output_report(info, full, fs, device)
        return 0, full.cpu().numpy(), info
    full = _gather_spans(out, spans, group) if measure else None
    res = out.cpu().numpy()
    sh.close()
    if full is not None:
        info = _with_output_report(info, full, fs, device)
    return spans[rank][0], res, info


def master_time_sharded_local(track, fs, settings, world, device=0, chunk_seconds=30, **plan_opts):
    """The same algorithm with all `world` shards emulated one after another on ONE GPU (tests, debugging):
    halo hand-off by copy, histogram 'all-reduce' by summation, limiter (if set) over the joined spans.
    Returns (int16[N,2], info)."""
    import torch
    from .engine import limit_device
    spans = plan_time_shards(len(track), fs, world, chunk_seconds)
    shards = [TimeShard(spans[r], fs, _shard_settings(settings), r, world, device, chunk_seconds, **plan_opts)
              for r in range(world)]
    prev_tail = None
    hists = []
    for r, sh in enumerate(shards):
        sh.load(np.ascontiguousarray(track[spans[r][0]:spans[r][1]]))
        sh.pre_normalisation()
        if prev_tail is not None:
            sh.set_halo(prev_tail)
        if sh.n:
            prev_tail = sh.tail()
        hists.append(sh.histogram().clone())
    total = hists[0].clone()
    for h in hists[1:]:
        total += h
    outs, info = [], None
    for sh in shards:
        o, i = sh.normalise(total)
        outs.append(o.clone())
        info = info or i
        sh.close()
    full = torch.cat(outs, dim=0)
    if settings.get("limiter"):
        full = limit_device(full, fs, settings, device)
    if settings.get("measure_output"):
        info = _with_output_report(info, full, fs, device)
    return full.cpu().numpy(), info
