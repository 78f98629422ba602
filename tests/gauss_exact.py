"""The Gaussian filter as an exact operation in float64, and the rounding bound a float32 kernel of it must meet.

The operation (what ``gaussian.cu`` implements, the reference's ``gaussian_filter`` up to float rounding):

* radius ``r = max(1, (int)(2 * sigma))`` with sigma taken as a float32, as both C sides do;
* ``k2`` = the reference's (2r+1)^2 float taps (``Port.gaussian_kernel``: the same ``expf`` expression as
  ``gaussian_taps_host``), ``k1`` = their column sums in float64;
* the value is the separable correlation with ``k1`` along x, then along y, over the image padded with zeros
  (``scipy.ndimage.correlate1d`` in float64, mode ``constant``);
* interior pixels (``r <= x < w - r`` and ``r <= y < h - r``) are not renormalised; every other pixel is divided by
  the exact sum of the in-bounds taps, ``N = nx * ny`` (``nx`` the in-bounds part of ``sum(k1)`` along x, the full sum
  for a column that is not within r of the left or right edge; ``ny`` likewise), which is the reference's rule.

``reference(img, sigma)`` returns ``(value, S, N)``, where ``S`` is the same operation applied to ``|img|`` (``S >=
|value|``; the error of every float evaluation below scales with it, not with the value, which may cancel).

The bound.  With ``u = 2**-24`` and ``m = 2r + 1``, a float32 evaluation of the operation that

* rounds each of the m taps to float (one rounding per tap and pass: 2 in all),
* runs each pass as a chain of at most m roundings (a product and m - 1 FMAs, or m products and adds fused into
  FMAs): 2m in all, so that ``|o - sum K x| <= gamma_(2m+2) * sum K |x|`` for the unnormalised sum ``o``,
* forms each normaliser as a float sum of at most m rounded taps (m - 1 + 1 per factor: 2m in all), then one
  product and one division (or a product, a reciprocal and a multiplication: one more) -- 2m + 3,
* multiplies interior pixels by 1.0, which is exact,

is within ``gamma_c * S`` of the value, with ``c(R) = 4(2R + 1) + 8`` (4m + 5 roundings counted above, the rest
spare) and ``gamma_c = c u / (1 - c u)`` (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., §3.1).
That argument assumes no underflow: a product that lands among the subnormals is off by up to 2**-150 absolutely,
not relatively, and the division by N scales that up, hence the absolute term ``c * 2**-149 / N``:

    |got - value| <= gamma_c * S + c * 2**-149 / N

The bound is derived, not fitted: c is not to be widened to what some kernel happens to produce.  It is sharp
enough to see one wrong input pixel: an 8,000-count background changed by one count moves the output by
``k1[r]**2`` (0.05 counts at sigma 1.7), the bound is 36 u S = 0.017 counts there.

Non-finite input: NaN and +-Inf propagate through the float64 operation as through the float one (0 * Inf = NaN for
the taps that are 0 at tiny sigma), so the non-finite pixels of the output, and the sign of each infinity, must
equal the value's; only the finite pixels go through the bound.
"""
import functools

import numpy as np
from scipy.ndimage import correlate1d

U = 2.0 ** -24
TINY = 2.0 ** -149  # the smallest float32 subnormal

# sigma grid of the tests: the common values, one float32 ulp either side of every radius threshold k / 2
# (R -> R + 1 dispatch), and large radii up to 64
THRESHOLDS = [float(np.nextafter(np.float32(k / 2), np.float32(s))) for k in range(2, 10) for s in (0, np.inf)]
SIGMAS = [0.3, 0.5, 1.0, 1.7, 2.0, 2.49] + THRESHOLDS + [5.0, 12.3, 32.4]


@functools.lru_cache(maxsize=None)
def _port():
    from oracle import oracle as O

    return O.Port()


def radius(sigma):
    """r = max(1, (int)(sigma * 2)) in float32, gaussian_taps_host's and the reference's radius."""
    return max(1, int(np.float32(sigma) * np.float32(2)))


@functools.lru_cache(maxsize=None)
def taps(sigma):
    """(r, k2, k1): the reference's float 2-D taps as float64 [dy + r, dx + r] and their float64 column sums."""
    k2 = _port().gaussian_kernel(float(np.float32(sigma))).astype(np.float64)
    r = k2.shape[0] // 2
    assert r == radius(sigma), (sigma, r)
    k2.setflags(write=False)
    k1 = k2.sum(axis=0)
    k1.setflags(write=False)
    return r, k2, k1


def c_of(r):
    """c(R) = 4(2R + 1) + 8: the rounding count of the bound."""
    return 4 * (2 * r + 1) + 8


def gamma(c):
    return c * U / (1.0 - c * U)


def normaliser(h, w, r, k1):
    """N[h, w]: 1 on interior pixels, the exact in-bounds tap sum nx * ny elsewhere."""
    nx = correlate1d(np.ones(w), k1, mode="constant", cval=0.0)
    ny = correlate1d(np.ones(h), k1, mode="constant", cval=0.0)
    n = ny[:, None] * nx[None, :]
    n[r:h - r, r:w - r] = 1.0
    return n


def reference(img, sigma):
    """(value, S, N) of the operation for a [h, w] or [n, h, w] image (any real dtype), all float64."""
    r, _k2, k1 = taps(sigma)
    x = np.asarray(img, dtype=np.float64)
    h, w = x.shape[-2:]

    def sep(a):
        with np.errstate(invalid="ignore", over="ignore"):
            t = correlate1d(a, k1, axis=-1, mode="constant", cval=0.0)
            return correlate1d(t, k1, axis=-2, mode="constant", cval=0.0)

    n = normaliser(h, w, r, k1)
    with np.errstate(invalid="ignore"):
        return sep(x) / n, sep(np.abs(x)) / n, n


def bound(S, N, r):
    """gamma_c * S + c * 2**-149 / N, per pixel."""
    c = c_of(r)
    return gamma(c) * S + c * TINY / N


def separability_gap(sigma):
    """g = max |k2 - k1 (x) k1| / (k1 (x) k1) over the taps that are not 0, in float64: how far the reference's 2-D
    taps are from the product the separable operation uses (float rounding of the taps, a few u)."""
    _r, k2, k1 = taps(sigma)
    kk = np.outer(k1, k1)
    nz = kk > 0
    return float((np.abs(k2 - kk)[nz] / kk[nz]).max()) if nz.any() else 0.0


def assert_reference_exact(want, img, sigma, what=""):
    """The reference's own output `want` (its sequential 2-D loop over the float taps k2) within its rounding bound of
    the operation: (2m^2 + 3) u S for m^2 products summed in order, a float sum of m^2 taps and one division, plus the
    separability gap -- g S inside, 2 g S at the borders, where the normaliser sum(k2) carries the gap too."""
    value, S, N = reference(img, sigma)
    m = 2 * radius(sigma) + 1
    g = separability_gap(sigma)
    err = np.abs(np.asarray(want, np.float64) - value)
    bad = err > (2 * m * m + 3) * U * S + np.where(N == 1.0, g, 2.0 * g) * S
    assert not bad.any(), f"{what}: {int(bad.sum())} pixels of the reference outside its bound (sigma {sigma!r})"
    return float((err / (U * np.where(S > 0, S, 1.0))).max()) if err.size else 0.0


def check(got, img, sigma):
    """(bad mask, value, S, N, error in units of u*S) of a float32 output against the operation; no assertion."""
    value, S, N = reference(img, sigma)
    r = radius(sigma)
    got = np.asarray(got)
    assert got.dtype == np.float32 and got.shape == value.shape, (got.dtype, got.shape, value.shape)
    g = got.astype(np.float64)
    fin = np.isfinite(value)
    with np.errstate(invalid="ignore"):
        err = np.where(fin, np.abs(g - value), 0.0)
        bad = np.where(fin, ~np.isfinite(g) | (err > bound(S, N, r)),
                       ~((np.isnan(g) & np.isnan(value)) | (g == value)))  # same NaN, same signed infinity
        ulps = np.where(fin & (S > 0), err / (U * np.where(S > 0, S, 1.0)), 0.0)
    return bad, value, S, N, ulps


def assert_gauss_exact(got, img, sigma, what=""):
    """Every pixel of `got` (float32 [h, w] or [n, h, w], the filter of `img` at `sigma`) within the bound of the
    float64 operation; the non-finite pixels exactly the operation's.  Returns the largest error seen in units of
    u * S (0 when every finite pixel is exact)."""
    bad, value, S, N, ulps = check(got, img, sigma)
    if bad.any():
        r = radius(sigma)
        got = np.asarray(got)
        # worst pixel: a non-finite mismatch first, else the largest error relative to its bound
        fin = np.isfinite(value)
        with np.errstate(invalid="ignore", divide="ignore"):
            score = np.where(fin, np.abs(got.astype(np.float64) - value) / bound(S, N, r), np.inf)
        score = np.where(bad, np.nan_to_num(score, nan=np.inf), -1.0)
        at = np.unravel_index(int(np.argmax(score)), bad.shape)
        raise AssertionError(
            f"{what}: {int(bad.sum())} of {bad.size} pixels outside the bound (sigma {float(np.float32(sigma))!r}, R {r}, "
            f"c {c_of(r)}); worst at {tuple(int(i) for i in at)} of {bad.shape}: got {float(got[at])!r}, "
            f"value {float(value[at])!r}, S {float(S[at])!r}, error {float(ulps[at]):.3g} u*S "
            f"(bound {c_of(r)} u*S + {c_of(r)} * 2**-149 / N, N {float(N[at[-2:]])!r})")  # N is per [h, w]
    return float(ulps.max()) if ulps.size else 0.0
