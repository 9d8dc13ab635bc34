"""The wave driver of libame over a batch of several waves, through the entry points that share it: the two-phase calls
(ame_measure_device, then ame_normalize_device) against ame_master_device on the same plan, and the launch count of
ame_master_host on a host_io plan over the same tracks."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _batch():
    """Six short tracks at mixed rates: multiband and plain, one with the limiter, one with the true peak, two with the
    output meter."""
    from audio_mastering_engine_b200 import synth
    c1, c2 = synth.c1_settings(), synth.c2_settings()
    spec = [(0.9, 44100, dict(c2, measure_output=True)), (1.1, 48000, dict(c1, limiter=True)),
            (0.7, 96000, dict(c2, true_peak=True)), (1.0, 32000, dict(c1, measure_output=True)),
            (0.8, 48000, c2), (0.6, 88200, c1)]
    tracks = [synth.track(secs, fs, track_id=k, am_hz=2.0) for k, (secs, fs, _) in enumerate(spec)]
    return tracks, [fs for _, fs, _ in spec], [s for _, _, s in spec]


def _plan(tracks, fss, sets, **kw):
    from audio_mastering_engine_b200 import MasterPlan
    return MasterPlan([len(t) for t in tracks], fss, sets, chunk_seconds=0.5, n_waves=3, **kw)


def test_two_phase_calls_equal_master_device(torch_cuda):
    torch = torch_cuda
    tracks, fss, sets = _batch()
    plan = _plan(tracks, fss, sets, n_slots=3)
    assert plan.n_waves == 3 and plan.n_slots == 3
    d_in = torch.as_tensor(plan.pack(tracks)).cuda()
    ref = torch.zeros_like(d_in)
    ref_res = plan.master_device(d_in, ref)
    ref_loud = plan.output_loudness()
    ref_launches = plan.launch_count
    assert sum(m is not None for m in ref_loud) == 2

    # a call over another input in between: what the two-phase calls report must be their own
    plan.master_device(torch.div(d_in, 2, rounding_mode="trunc"), torch.zeros_like(d_in))
    assert plan.results() != ref_res and plan.output_loudness() != ref_loud

    d_hist = torch.zeros((len(tracks), 1000), dtype=torch.int64, device=d_in.device)
    out = torch.zeros_like(d_in)
    plan.measure_device(d_in, d_hist)
    res = plan.normalize_device(d_hist, out)
    torch.cuda.synchronize()
    assert torch.equal(out, ref)
    assert res == ref_res
    assert plan.output_loudness() == ref_loud
    assert plan.launch_count == ref_launches
    plan.close()

    host = _plan(tracks, fss, sets, n_slots=3, host_io=True)
    h_out = np.zeros_like(host.pack(tracks))
    host_res = host.master_host(host.pack(tracks), h_out)
    assert host.launch_count == ref_launches
    assert np.array_equal(h_out, ref.cpu().numpy()) and host_res == ref_res
    host.close()


def test_two_phase_calls_need_a_slot_per_wave(torch_cuda):
    from audio_mastering_engine_b200 import AmeError
    torch = torch_cuda
    tracks, fss, sets = _batch()
    plan = _plan(tracks, fss, sets, n_slots=2)
    assert plan.n_waves == 3 and plan.n_slots == 2
    d_in = torch.as_tensor(plan.pack(tracks)).cuda()
    d_hist = torch.zeros((len(tracks), 1000), dtype=torch.int64, device=d_in.device)
    with pytest.raises(AmeError, match="n_slots == n_waves"):
        plan.measure_device(d_in, d_hist)
    plan.close()
