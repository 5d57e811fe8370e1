"""The Gaussian blur restatement (oracle/gaussian_oracle.c: oracle_gaussian_window, oracle_sepconv) that the GPU tests compare with,
pinned without a GPU: the window against a numpy restatement of FillGaussian's steps, the convolution against scipy's correlate1d with
mirror (= reflect-101) borders in float64, and known answers (impulse, constant image, sigma <-> window examples)."""
import numpy as np
import pytest

from oracle import pygaussian as pg

scipy_ndimage = pytest.importorskip("scipy.ndimage")


def _np_window(sigma, d):
    r = (d - 1) // 2
    s = 0.5 / (np.float64(np.float32(sigma)) ** 2)
    w = np.zeros(d, np.float32)
    total = 0.0
    for x in range(-r, 0):
        w[x + r] = np.float32(np.exp(-(x * x) * s))
        total += np.float64(w[x + r])
    scale = 1 / (2 * total + 1)
    w[r] = np.float32(scale)
    for x in range(r):
        w[x] = np.float32(np.float64(w[x]) * scale)
        w[2 * r - x] = w[x]
    return w


def test_sigma_window_rules():
    for sigma, d in [(0.1, 3), (0.5, 5), (1.0, 7), (2.0, 13)]:
        assert pg.gaussian_params(sigma, 0) == (pytest.approx(sigma), d)
    s, d = pg.gaussian_params(0, 23)
    assert d == 23 and s == np.float32(3.8)
    assert pg.gaussian_params(0, 1) == (pytest.approx(0.5), 1)


@pytest.mark.parametrize("sigma,d", [(0.1, 3), (0.5, 5), (1.0, 7), (2.0, 13), (3.8, 23), (0.7, 1), (12.3, 75), (1.0, 31)])
def test_window_equals_numpy_restatement(sigma, d):
    w = pg.gaussian_window(sigma, d)
    assert np.array_equal(w.view(np.uint32), _np_window(sigma, d).view(np.uint32))
    assert abs(float(np.sum(w, dtype=np.float64)) - 1) <= 1e-6
    assert np.array_equal(w, w[::-1])


def _scipy(x, wins):
    y = x.astype(np.float64)
    nd = len(wins)
    for k in range(nd):                    # innermost axis first
        a = nd - 1 - k
        y = scipy_ndimage.correlate1d(y, wins[a].astype(np.float64), axis=a, mode="mirror")
    return y


@pytest.mark.parametrize("shape,sig", [((40, 52, 3), (1.5, 0.7)), ((9, 11, 1), (2.0, 3.0)), ((6, 30, 4), (4.0, 0.3)),
                                       ((3, 2, 1), (5.0, 5.0)), ((1, 17, 3), (1.0, 2.0)), ((12, 1, 3), (2.0, 1.0)),
                                       ((7, 9, 10, 1), (1.0, 2.0, 0.5)), ((2, 5, 4, 3), (3.0, 0.4, 1.2)), ((1, 1, 1, 4), (2.0, 2.0, 2.0))])
@pytest.mark.parametrize("dtype", [np.float32, np.uint8])
def test_convolution_against_scipy_mirror(shape, sig, dtype):
    """reflect-101 repeats its reflection for windows longer than the axis; scipy's `mirror` mode does the same (extent 1: index 0)."""
    rng = np.random.default_rng(sum(shape))
    x = rng.uniform(0, 255, shape).astype(np.float32) if dtype == np.float32 else rng.integers(0, 256, shape, dtype=np.uint8)
    wins = [pg.gaussian_window(*pg.gaussian_params(s, 0)) for s in sig]
    want = _scipy(x, wins)
    got = pg.sepconv(x, wins, np.float32)
    assert np.all(np.abs(got - want) <= 1e-5 * np.maximum(np.abs(want), 1.0))
    g8 = pg.sepconv(x, wins, np.uint8)
    assert np.all(np.abs(g8.astype(np.int32) - np.clip(np.round(want), 0, 255)) <= 1)
    frac = np.abs(want - np.floor(want) - 0.5)
    far = frac > 1e-3                                   # away from the .5 rounding boundaries: exact
    assert np.array_equal(g8[far], np.clip(np.floor(want + 0.5), 0, 255).astype(np.uint8)[far])


@pytest.mark.parametrize("channels", [1, 3, 4])
def test_impulse_gives_outer_product_of_windows(channels):
    x = np.zeros((21, 25, channels), np.float32)
    x[10, 12, :] = 1.0
    wy, wx = pg.gaussian_window(1.5, 11), pg.gaussian_window(0.8, 7)
    got = pg.sepconv(x, [wy, wx])
    want = np.zeros((21, 25), np.float32)
    want[5:16, 9:16] = wy[:, None] * wx[None, :]          # one non-zero tap per pass: one rounded product each
    for c in range(channels):
        assert np.array_equal(got[..., c], want)
    vol = np.zeros((9, 9, 9, 1), np.float32)
    vol[4, 4, 4] = 1
    w = pg.gaussian_window(1.0, 7)
    got = pg.sepconv(vol, [w, w, w])[1:8, 1:8, 1:8, 0]
    want = w[:, None, None] * (w[None, :, None] * w[None, None, :])     # W pass, then H, then D
    assert np.array_equal(got, want)


def test_constant_image_stays_constant():
    """The taps of a window sum to 1 only up to float rounding, so a constant moves by a few ulps per tap at most (not within one
    ulp in general: 255 under 13 + 121 taps moves by 7 ulps); u8 output rounds back to the constant."""
    for v in (0.25, 100.0, 255.0):
        x = np.full((30, 40, 3), v, np.float32)
        for sig in ((0.5, 0.5), (2.0, 7.0), (20.0, 1.0)):
            wins = [pg.gaussian_window(*pg.gaussian_params(s, 0)) for s in sig]
            got = pg.sepconv(x, wins)
            assert np.all(np.abs(got - v) <= sum(len(w) for w in wins) * np.spacing(np.float32(v))), (v, sig, np.abs(got - v).max())
            assert np.all(pg.sepconv(x.astype(np.uint8), wins, np.uint8) == np.uint8(v)), (v, sig)
