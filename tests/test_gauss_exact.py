"""The float64 Gaussian of tests/gauss_exact.py is the reference's operation, and its bound sees what the frame-relative
tolerance the GPU tests used before did not (CPU only).

* the reference's 2-D taps are the outer product of their column sums up to a gap g of float rounding (printed);
* the compiled reference and its C restatement are within their own rounding bound of the float64 value: a sequential
  sum of (2R+1)^2 products, a float sum of as many taps and one division -- (2(2R+1)^2 + 3) u S -- plus the
  separability gap (g S inside; 2 g S at the borders, where the normaliser carries the gap too);
* the radius follows the float32 sigma across every threshold k / 2;
* one count added to one background pixel is rejected by the new bar and was accepted by the old one.
"""
import numpy as np
import pytest

from tests import gauss_exact as G
from tests.conftest import ir_frame

SIGMAS = G.SIGMAS


def old_bar_failures(got, want):
    """Pixels the former Gaussian bar rejected: 1e-5 of |want| plus 1e-6 of the frame's largest |want|."""
    rel, floor = 1e-5, 1e-6
    want = np.asarray(want, np.float64)
    tol = rel * np.abs(want) + floor * float(np.abs(want).max())
    return int((np.abs(np.asarray(got, np.float64) - want) > tol).sum())


def images(shape, seed):
    """(name, float32 image) of each kind of content: IR frame, uniform uint16, mixed-sign, wide dynamic range."""
    h, w = shape
    rng = np.random.default_rng(seed)
    wide = np.exp(rng.uniform(np.log(1e-3), np.log(1e5), shape)) * rng.choice([-1.0, 1.0], shape)
    return [("ir", ir_frame(h, w, seed).astype(np.float32)),
            ("uniform u16", rng.integers(0, 65536, shape).astype(np.float32)),
            ("mixed sign", (rng.normal(0, 1000, shape) + rng.choice([-4000.0, 4000.0], shape)).astype(np.float32)),
            ("wide range", wide.astype(np.float32))]


def shapes_for(r):
    m = 2 * r + 1
    small = [(1, 1), (1, 2), (2, 1), (1, 9), (7, 1), (2, 2), (3, 5), (m - 1, m), (m, m), (m + 1, m + 2)]
    large = [(33, 20), (70, 136)] if r <= 10 else [(40, 31)]
    return small + large


def test_separability_gap():
    print()
    for s in SIGMAS:
        r = G.radius(s)
        g = G.separability_gap(s)
        print(f"sigma {s!r:>12} R {r:2d}: g = {g:.3e} = {g / G.U:7.2f} u; device bound c(R) = {G.c_of(r)} u S, "
              f"reference bound (2(2R+1)^2 + 3) u S + 2 g S = {2 * (2 * r + 1) ** 2 + 3 + 2 * g / G.U:.0f} u S")
        # the 2-D taps are a product up to rounding: a gap this size would be a different kernel, not rounding
        assert g < 2.0 ** -12, (s, g)


@pytest.mark.parametrize("oracle", ["port", "ref"])
@pytest.mark.parametrize("sigma", SIGMAS)
def test_reference_within_its_own_bound(request, oracle, sigma):
    impl = request.getfixturevalue(oracle)
    r = G.radius(sigma)
    worst = 0.0
    for shape in shapes_for(r):
        for name, img in images(shape, seed=shape[0] * 131 + shape[1] + r):
            got = impl.gaussian_filter(img, sigma)
            worst = max(worst, G.assert_reference_exact(got, img, sigma, f"{oracle} {name} {shape}"))
    print(f"{oracle} sigma {sigma!r}: worst {worst:.2f} u S")


@pytest.mark.parametrize("k", range(2, 10))
def test_radius_thresholds(port, k):
    """r changes from k - 1 to k exactly at the float32 sigma k / 2, in the helper as in the reference's kernel."""
    s0 = np.float32(k / 2)
    for s, want in [(np.nextafter(s0, np.float32(0)), k - 1), (s0, k), (np.nextafter(s0, np.float32(np.inf)), k)]:
        assert G.radius(s) == want, (s, want)
        assert port.gaussian_kernel(float(s)).shape == (2 * want + 1, 2 * want + 1), s
        assert G.taps(float(s))[0] == want


@pytest.mark.parametrize("sigma", [1.7, 2.49])
def test_resolving_power(port, sigma):
    """The oracle's output of an IR frame passes against the frame; against the same frame with one background pixel
    one or two counts higher it fails.  The former frame-relative bar let the one-count error through."""
    h, w = 70, 136
    img = ir_frame(h, w, 9)
    y, x = 12, 20  # background, away from the hot spot
    assert 7900 < img[y, x] < 8100
    got = port.gaussian_filter(img.astype(np.float32), sigma)
    G.assert_gauss_exact(got, img, sigma, "clean frame")
    print()
    for delta in (1, 2):
        moved = img.astype(np.float32)
        moved[y, x] += delta
        bad, *_ = G.check(got, moved, sigma)
        old = old_bar_failures(got, port.gaussian_filter(moved, sigma))
        print(f"sigma {sigma}: +{delta} count at ({y}, {x}): old bar flags {old} pixels, new bar {int(bad.sum())}")
        with pytest.raises(AssertionError, match="outside the bound"):
            G.assert_gauss_exact(got, moved, sigma, f"+{delta} count")
        if delta == 1:
            assert old == 0, "the former bar saw the one-count error after all"


def test_failure_report_of_frame_stacks(port):
    """A failing [n, h, w] stack is reported like a single frame: count, worst pixel (frame, row, column), its error."""
    img = np.stack([ir_frame(40, 56, 3 + t) for t in range(3)])
    got = np.stack([port.gaussian_filter(f.astype(np.float32), 1.0) for f in img])
    G.assert_gauss_exact(got, img, 1.0, "clean stack")
    got[2, 30, 7] += 0.5
    with pytest.raises(AssertionError, match=r"worst at \(2, 30, 7\) of \(3, 40, 56\)"):
        G.assert_gauss_exact(got, img, 1.0, "one pixel off")
    with pytest.raises(AssertionError, match=r"worst at \(30, 7\) of \(40, 56\)"):
        G.assert_gauss_exact(got[2], img[2], 1.0, "one pixel off, one frame")


def test_reference_edge_cases(port):
    """All zeros give exact zeros; a 1 x 1 image is its own value; NaN / Inf follow the float64 operation."""
    for s in (0.5, 2.49, 12.3):
        assert not G.reference(np.zeros((5, 9)), s)[0].any()
        v, S, N = G.reference(np.array([[3.5]]), s)
        assert v[0, 0] == pytest.approx(3.5, rel=1e-15) and S[0, 0] == v[0, 0]
    img = np.ones((9, 11), np.float32)
    img[4, 5] = np.inf
    img[0, 0] = -np.inf
    for s in (0.05, 1.0):
        got = port.gaussian_filter(img, s)
        G.assert_gauss_exact(got, img, s, f"non-finite, sigma {s}")
    v = G.reference(img, 0.05)[0]
    assert np.isnan(v[4, 4]) and v[4, 5] == np.inf, "sigma 0.05: taps of 0 meet Inf (0 * Inf = NaN) next to the Inf"
