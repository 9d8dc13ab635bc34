"""The oracle restatement (oracle/chain.py) must reproduce, bit for bit, the fixtures produced by the
reference's own functions (tests/golden/make_golden.py, audio_mastering_engine.py:250-309)."""
import numpy as np

from oracle import chain


def test_converters(golden):
    g = golden
    assert np.array_equal(chain.to_float(g["conv_in"]), g["conv_float"])
    assert np.array_equal(chain.to_pcm(g["conv_ramp_f32"]), g["conv_ramp_pcm_f32"])
    assert np.array_equal(chain.to_pcm(g["conv_ramp_f32"].astype(np.float64) * 0.999), g["conv_ramp_pcm_f64"])
    # documented knife edges (SURVEY.md 8(a) row 3)
    assert chain.to_pcm(np.array([[-0.99999, 1 / 32768]], dtype=np.float32)).tolist() == [[-32766, 0]]


def test_chunk_cases_bit_exact(golden):
    g = golden
    assert len(g.cases) >= 30
    for c in g.cases:
        key, fs, settings = c["key"], c["fs"], c["settings"]
        taps = {}
        out = chain.process_chunk(g.input(c), fs, settings, taps=taps,
                                  compress=chain.compress_dynamic_range_py)
        assert g.equals(c, "warmth", taps["warmth"]), key
        assert taps["eq"].dtype == np.float32
        assert g.equals(c, "eq", taps["eq"]), key
        assert g.equals(c, "pre_multiband", taps["pre_multiband"]), key
        assert g.equals(c, "out", out), key


def test_warmth_closed_form_matches_axis_quirk(golden):
    """lfilter(axis=-1) on an (N,2) array == the per-frame 2x2 lower-triangular mix the kernel uses."""
    g = golden
    for c in g.cases:
        pct = c["settings"].get("analog_character", 0)
        if pct > 0:
            assert g.equals(c, "warmth", chain.warmth_closed_form(g.input(c), c["fs"], pct)), c["key"]


def test_cut_shelf_is_bare_filter():
    """engine.py:289: any negative shelf gain returns the Butterworth output itself."""
    from scipy.signal import butter, lfilter
    rng = np.random.default_rng(0)
    x = rng.standard_normal(5000).astype(np.float32) * 0.1
    b, a = butter(2, 250 / 24000.0, btype="low")
    y = chain.shelf(x, 48000, 250, -2.0, "low")
    assert np.max(np.abs(y - lfilter(b, a, x))) < 1e-15
