"""CPU checks of what the audio-tail GPU tests compare against: known answers that pin what `nonsilent_region`, `audio_resample`,
`to_decibels` and `mfcc` compute, so that the GPU parity tests compare against something whose meaning is established here.  The known
answers are checked on the reference's own kernels (oracle/_ref) where that library is built, else on the plain-C restatement
(oracle/audio_oracle.c), which is what tests/test_gpu_warp_color_audio.py compares with in that case."""
import numpy as np
import pytest

from oracle import pyoracle as po


def _impl(name):
    return getattr(po, "ref_" + name) if po.have_ref() else getattr(po, name)


def test_nonsilent_region_known_answers():
    # the example of nonsilence_op.h (LeadTrailThresh): buffer [0, 0, 0, 0, 50, 50, 0, 0], window 1 -> (4, 2)
    x = np.array([0, 0, 0, 0, 50, 50, 0, 0], np.float32)
    assert _impl("nonsilent_region")(x, cutoff_db=-3.0, window_length=1, reset_interval=-1) == (4, 2)
    # digital silence with the default reference (= the maximum = 0): the threshold is 0 and `>=` holds everywhere -- the reference
    # reports the whole buffer; with a fixed reference power it reports length 0
    assert _impl("nonsilent_region")(np.zeros(100, np.float32), window_length=4, reset_interval=-1) == (0, 100)
    assert _impl("nonsilent_region")(np.zeros(100, np.float32), window_length=4, reference_power=1.0, reset_interval=-1)[1] == 0
    # a burst in the middle: the start moves back by window_length - 1, the end is the last window that still sees the burst
    x = np.zeros(1000, np.float32)
    x[400:500] = 1.0
    b, l = _impl("nonsilent_region")(x, cutoff_db=-20.0, window_length=16, reset_interval=-1)
    assert 380 <= b <= 400                                      # first window whose mean square reaches 1 % of the maximum, minus window - 1
    assert 499 <= b + l - 1 <= 499 + 15
    # a fixed reference power instead of the maximum changes the threshold, not the mechanics
    b2, l2 = _impl("nonsilent_region")(x, cutoff_db=-20.0, window_length=16, reference_power=1.0, reset_interval=-1)
    assert (b2, l2) == (b, l)


def test_audio_resample_known_answers():
    rng = np.random.default_rng(0)
    x = rng.uniform(-1, 1, 2000).astype(np.float32)
    # equal rates: the windowed sinc is sampled at integers -> the signal itself (up to the interpolated lookup of the window)
    y = _impl("audio_resample")(x, 16000.0, 16000.0)
    assert y.shape == x.shape and np.abs(y - x).max() < 1e-5
    # length rule: ceil(n * out / in)
    assert _impl("audio_resample")(x, 16000.0, 44100.0).shape == (int(np.ceil(2000 * 44100 / 16000)),)
    assert _impl("audio_resample")(x, 44100.0, 16000.0).shape == (int(np.ceil(2000 * 16000 / 44100)),)
    # a slow sine survives 2x up-sampling
    t = np.arange(4000, dtype=np.float64)
    s = np.sin(2 * np.pi * t / 200).astype(np.float32)
    u = _impl("audio_resample")(s, 1.0, 2.0, quality=90.0)
    want = np.sin(2 * np.pi * (np.arange(u.size) / 2.0) / 200)
    assert np.abs(u[100:-100] - want[100:-100]).max() < 2e-3
    # interleaved stereo: the channels are resampled independently
    st = np.stack([s, -s], axis=1)
    v = _impl("audio_resample")(st, 1.0, 2.0, quality=90.0)
    assert v.shape == (u.size, 2) and np.abs(v[:, 0] + v[:, 1]).max() < 1e-6
    assert np.abs(v[200:-200, 0] - u[200:-200]).max() < 1e-5    # the multi-channel path sums the taps in a different order


def test_to_decibels_and_mfcc_known_answers():
    x = np.array([[1.0, 10.0, 100.0, 1e-30]], np.float32)
    d = _impl("to_decibels")(x, 10.0, 1.0, -80.0)
    assert np.allclose(d, [[0.0, 10.0, 20.0, -80.0]], atol=1e-5)
    d = _impl("to_decibels")(x, 20.0, None, -200.0)              # reference = maximum (100)
    assert np.allclose(d[0, :3], [-40.0, -20.0, 0.0], atol=1e-4)
    # DCT-II of a constant column: only coefficient 0 is non-zero (= N * c: table.h defines X_k = sum x_n cos(pi (n + 1/2) k / N), no factor 2)
    m = np.full((8, 3), 2.0, np.float32)
    c = _impl("mfcc")(m, n_mfcc=4, dct_type=2, normalize=False)
    assert c.shape == (4, 3) and np.allclose(c[0], 8 * 2.0) and np.abs(c[1:]).max() < 1e-4


@pytest.mark.skipif(not po.have_ref(), reason="needs oracle/_ref (the reference's CPU kernels)")
def test_plain_c_restatements_equal_the_compiled_reference():
    """oracle/audio_oracle.c (to_decibels, mfcc, nonsilent_region, audio_resample) against oracle/_ref, bit for bit, on random sweeps."""
    rng = np.random.default_rng(21)
    for it in range(6):
        m = (np.abs(rng.normal(0, 1, (int(rng.integers(8, 90)), int(rng.integers(1, 70))))).astype(np.float32) ** 2) + 1e-12
        for args in ((10.0, None, -200.0), (20.0, 0.5, -60.0), (10.0, 1.0, -80.0)):
            assert np.array_equal(po.to_decibels(m, *args).view(np.uint32), po.ref_to_decibels(m, *args).view(np.uint32)), (it, args)
        for n_mfcc, t, norm, lift in ((13, 2, True, 22.0), (40, 3, False, 0.0), (7, 1, False, 0.0), (20, 4, True, 5.0), (20, 2, False, 10.0)):
            if t == 1 and m.shape[0] < 3:
                continue
            assert np.array_equal(po.mfcc(m, n_mfcc, t, norm, lift).view(np.uint32), po.ref_mfcc(m, n_mfcc, t, norm, lift).view(np.uint32)), (it, n_mfcc, t)
    for n, lead, trail in ((40000, 6000, 9000), (16000, 0, 3000), (1000, 300, 200), (5000, 0, 0)):
        x = (0.4 * np.sin(np.arange(n) * 0.05) + 0.05 * rng.normal(0, 1, n)).astype(np.float32)
        x[:lead] = (1e-5 * rng.normal(0, 1, lead)).astype(np.float32)
        if trail:
            x[n - trail:] = (1e-5 * rng.normal(0, 1, trail)).astype(np.float32)
        for kw in (dict(), dict(cutoff_db=-40.0, window_length=512, reset_interval=2048), dict(cutoff_db=-45.0, window_length=3000, reference_power=0.02,
                                                                                              reset_interval=-1)):
            assert po.nonsilent_region(x, **kw) == po.ref_nonsilent_region(x, **kw), (n, kw)
    for n, ir, orr, q in ((16000, 16000.0, 44100.0, 50.0), (4001, 44100.0, 16000.0, 50.0), (700, 8000.0, 16000.0, 90.0), (25000, 22050.0, 8000.0, 10.0),
                          (3000, 1.0, 0.37, 0.0)):
        x = rng.uniform(-1, 1, n).astype(np.float32)
        assert np.array_equal(po.audio_resample(x, ir, orr, q).view(np.uint32), po.ref_audio_resample(x, ir, orr, q).view(np.uint32)), (n, ir, orr, q)
        st = rng.uniform(-1, 1, (n // 3, 2)).astype(np.float32)
        assert np.array_equal(po.audio_resample(st, ir, orr, q).view(np.uint32), po.ref_audio_resample(st, ir, orr, q).view(np.uint32)), (n, "stereo")
    x = rng.uniform(-1, 1, 5000).astype(np.float32)
    assert np.array_equal(po.audio_resample(x, 5000.0, 1234.0, 50.0, out_length=1234), po.ref_audio_resample(x, 5000.0, 1234.0, 50.0, out_length=1234))
