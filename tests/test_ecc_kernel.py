"""The restatement of the ECC kernel's own solve (tests/ecc_kernel.py) is OpenCV's iteration, and it has teeth.

  * its fixed-point shift, warp, gradients and normalisation are bit-identical to oracle/ecc.py (and to cv2.warpAffine
    where OpenCV is importable);
  * its whole solves agree with oracle/ecc.py's find_transform_ecc_translation within 2e-5 px / 1e-7 in rho with the same
    iteration count, at several grid sizes: the summation order moves the last bits and nothing else;
  * each slip planted in it below changes the (status, rho, tx, ty) bits of the cases tests/test_gpu_registration_exact.py runs,
    so the same slip in the kernel fails that bit-exact comparison.
No device needed.
"""
import numpy as np
import pytest

from oracle import ecc as oe
from tests import ecc_cases as ec
from tests import ecc_kernel as ek

SHIFT_TOL, RHO_TOL = 2e-5, 1e-7  # the restatement of OpenCV against the kernel's arithmetic (tests/test_ecc.py)


def f32(v):
    return float(np.float32(v))


STARTS = ec.boundary_starts()


# ---- the shift and the warp --------------------------------------------------------------------------------------
def oracle_weights(fx, fy):
    """warpAffine's four weights for fractions fx / 32, fy / 32, read out of oracle/ecc.py with impulse images."""
    out = []
    for y, x in ((0, 0), (0, 1), (1, 0), (1, 1)):
        img = np.zeros((3, 3), np.float32)
        img[y, x] = 1.0
        out.append(oe.warp_affine_translation(img, fx / 32.0, fy / 32.0)[0, 0])
    return out


def test_shift_weights_equal_the_oracle_table():
    for fx in range(32):
        for fy in range(32):
            sh = ek.ecc_shift(fx / 32.0, fy / 32.0)
            assert (sh.ox, sh.oy) == (0, 0)
            got = np.array([sh.w00, sh.w01, sh.w10, sh.w11], np.float32)
            assert np.array_equal(got.view(np.uint32), np.array(oracle_weights(fx, fy), np.float32).view(np.uint32)), (fx, fy)


def test_shift_origins_equal_fixed_point_origin():
    h, w = 3, 5
    idx = np.arange(1, h * w + 1, dtype=np.int64).reshape(h, w)
    for tx in STARTS:
        for ty in (STARTS[len(STARTS) // 3], -0.75, f32(1 / 64.0), tx):
            sh = ek.ecc_shift(tx, ty)
            X, Y = oe.fixed_point_origin(tx, ty, h, w)
            assert np.array_equal(X >> 5, np.arange(w)[None, :] + sh.ox + 0 * X), (tx, ty)
            assert np.array_equal(Y >> 5, np.arange(h)[:, None] + sh.oy + 0 * Y), (tx, ty)
            nn = oe.warp_affine_translation(idx, tx, ty, nearest=True)
            assert np.array_equal(nn, ek.shifted(idx, sh.oyn, sh.oxn, 0)), (tx, ty)


def test_shift_fractions_equal_fixed_point_origin():
    for tx in STARTS:
        sh = ek.ecc_shift(tx, tx)
        X, _ = oe.fixed_point_origin(tx, tx, 1, 1)
        fx = np.float32(int(X[0, 0]) & 31) * np.float32(0.03125)
        one = np.float32(1)
        assert sh.w11 == np.float32(fx * fx) and sh.w00 == np.float32((one - fx) * (one - fx)), tx


def test_warp_equals_cv2_live():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(11)
    img = rng.uniform(-3, 3, (9, 13)).astype(np.float32)
    m8 = (rng.random((9, 13)) < 0.5).astype(np.uint8)
    for tx in STARTS:
        for ty in (tx, -tx, 0.40625):
            M = np.array([[1, 0, tx], [0, 1, ty]], np.float32)
            sh = ek.ecc_shift(tx, ty)
            lin = cv2.warpAffine(img, M, (13, 9), flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
            assert np.array_equal(ek.warp(img, sh).view(np.uint32), lin.view(np.uint32)), (tx, ty)
            nn = cv2.warpAffine(m8, M, (13, 9), flags=cv2.INTER_NEAREST | cv2.WARP_INVERSE_MAP, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
            assert np.array_equal(ek.shifted(m8, sh.oyn, sh.oxn, 0), nn), (tx, ty)


# ---- clamp, normalisation, gradients -----------------------------------------------------------------------------
@pytest.mark.parametrize("h,w", [(2, 2), (2, 9), (9, 2), (3, 3), (37, 53), (120, 160)])
def test_normalisation_and_gradients_equal_the_oracle(h, w):
    rng = np.random.default_rng(h * 1000 + w)
    for thresh in (float("inf"), float("nan"), None):
        t = (rng.uniform(0, 5000, (h, w)) + 8000).astype(np.float32)
        i = (t * np.float32(rng.uniform(0.8, 1.2)) + rng.normal(0, 30, (h, w))).astype(np.float32)
        th = float(np.quantile(t, 0.7)) if thresh is None else thresh
        mask = (rng.random((h, w)) < 0.6).astype(np.uint8)
        p = ek.prepare(t, i, mask, th)
        t1, i1 = t.copy(), i.copy()  # what MaskedRegistratorECC.compute does (oracle/ecc.py:217-226)
        if np.isfinite(th):
            m = (t1 > np.float32(th)) | (i1 > np.float32(th))
            t1[m] = np.float32(th)
            i1[m] = np.float32(th)
        with np.errstate(all="ignore"):  # a clamp may leave a 2 x 2 window flat: 0 / 0, as in the kernel
            t1 = (t1 - np.min(t1)) / (np.max(t1) - np.min(t1))
            i1 = (i1 - np.min(i1)) / (np.max(i1) - np.min(i1))
        assert p.T.dtype == p.I.dtype == np.float32
        assert np.array_equal(p.T.view(np.uint32), t1.view(np.uint32)) and np.array_equal(p.I.view(np.uint32), i1.view(np.uint32))
        gx, gy = oe.gradients(i1)  # times the mask as find_transform_ecc_translation builds it
        pre = np.rint(mask.astype(np.float32) * np.float32(0.5 / 0.95)).astype(np.uint8).astype(np.float32)
        assert np.array_equal(p.gx.view(np.uint32), (gx * pre).view(np.uint32)) and np.array_equal(p.gy.view(np.uint32), (gy * pre).view(np.uint32))


def test_min_max_keys_order_every_float():
    v = np.array([-np.inf, -3e38, -1.0, -1e-45, -0.0, 0.0, 1e-45, 1.0, 3e38, np.inf], np.float32)
    k = ek.fkey(v)
    assert np.all(np.diff(k.astype(np.int64)) >= 0)
    assert all(np.float32(ek.fkey_inv(x)).view(np.uint32) == y.view(np.uint32) for x, y in zip(k, v))


# ---- whole solves against OpenCV's iteration ---------------------------------------------------------------------
def normalised(t, i, thresh=float("inf")):
    t1, i1 = t.copy(), i.copy()
    if np.isfinite(thresh):
        m = (t1 > thresh) | (i1 > thresh)
        t1[m] = thresh
        i1[m] = thresh
    return (t1 - t1.min()) / (t1.max() - t1.min()), (i1 - i1.min()) / (i1.max() - i1.min())


def oracle_cases():
    """ecc_cases.SMALL_CASES, the masked and warm cases of tests/test_ecc.py, and a seeded set drawn like
    test_gpu_fuzz.py::test_fuzz_ecc_solver: (template, image, mask, thresh, tx0, ty0)."""
    cases = []
    for k, (dx, dy) in enumerate(ec.SMALL_CASES):
        t, i = ec.small_pair(dx, dy, k=k)
        cases.append((t, i, None, float("inf"), 0.0, 0.0))
    t, i = ec.small_pair(1.2, 0.7, k=9)
    mask = np.zeros(t.shape, np.uint8)
    mask[10:100, 20:150] = 1
    cases += [(t, i, mask, float("inf"), 0.0, 0.0), (t, i, None, float("inf"), 1.0, 0.5)]
    rng = np.random.default_rng(507)
    for _ in range(12):
        h, w = int(rng.integers(24, 140)), int(rng.integers(24, 180))
        dx, dy = float(rng.uniform(-4, 4)), float(rng.uniform(-4, 4))
        t, i = ec.small_pair(dx, dy, h=h, w=w, k=int(rng.integers(0, 1000)))
        scale, offset = float(rng.choice([1.0, 5000.0])), float(rng.choice([0.0, 8000.0]))
        t, i = (t * scale + offset).astype(np.float32), (i * np.float32(scale * rng.uniform(0.8, 1.2)) + np.float32(offset)).astype(np.float32)
        mask = None
        if rng.integers(0, 2):
            mask = np.zeros((h, w), np.uint8)
            mask[int(h * 0.1):int(h * 0.9), int(w * 0.15):w] = 1
        thresh = float("inf") if rng.integers(0, 2) else float(np.quantile(t, 0.9))
        tx0, ty0 = (0.0, 0.0) if rng.integers(0, 2) else (f32(dx + rng.uniform(-1, 1)), f32(dy + rng.uniform(-1, 1)))
        cases.append((t, i, mask, thresh, tx0, ty0))
    return cases


def test_solve_is_opencvs_iteration_at_every_grid():
    bits, compared = set(), 0
    for n_case, (t, i, mask, thresh, tx0, ty0) in enumerate(oracle_cases()):
        t1, i1 = normalised(t, i, thresh)
        try:
            want = oe.find_transform_ecc_translation(t1, i1, tx0, ty0, mask=mask)
        except oe.ECCError as e:
            want = 1 if "NaN" in str(e) else 2
        if not isinstance(want, int) and want[3] > 50:
            continue  # no convergence: hundreds of chained updates (test_fuzz_ecc_solver explains why nothing compares)
        p = ek.prepare(t, i, mask, thresh)
        n = t.size
        for G in sorted({1, 3, ek.grid(n, ek.B200_SMS, True), ek.grid(n, 8, False)}):
            st, rho, tx, ty, it = ek.solve(p, tx0, ty0, G)
            if isinstance(want, int):
                assert st == want, (n_case, G)
                continue
            assert st == 0 and it == want[3], (n_case, G, st, it, want)
            assert abs(rho - want[0]) < RHO_TOL and abs(tx - want[1]) < SHIFT_TOL and abs(ty - want[2]) < SHIFT_TOL, (n_case, G, rho, tx, ty, want)
            bits.add((n_case, rho, tx, ty))
        compared += 1
    assert compared >= 15
    assert len(bits) > compared  # the order of the sums does move bits


# ---- mutations ---------------------------------------------------------------------------------------------------
def _drop_last_pixel(orig):
    return lambda p, sh: [v[:-1] for v in orig(p, sh)]


def _drop_row0(orig):
    def f(p, sh):
        w = p.T.shape[1]
        out = [v.copy() for v in orig(p, sh)]
        for v in out:
            v[:w] = 0.0
        return out
    return f


def _count_unmasked(orig):
    def f(p, sh):
        out = orig(p, sh)
        out[ek.A_N] = np.ones_like(out[ek.A_N])
        return out
    return f


def _reverse_one_sum(orig):
    def f(p, sh):
        out = orig(p, sh)
        out[ek.A_II] = out[ek.A_II][::-1].copy()  # most sums come out exact in any order; this one does not
        return out
    return f


def _nearest_plus_16(orig):
    def f(tx, ty):
        sh = orig(tx, ty)
        SX, SY = int(np.rint(f32(tx) * 1024.0)), int(np.rint(f32(ty) * 1024.0))
        return sh._replace(oxn=(SX + 16) >> 10, oyn=(SY + 16) >> 10)
    return f


def _swap_w01_w10(orig):
    return lambda tx, ty: orig(tx, ty)._replace(w01=orig(tx, ty).w10, w10=orig(tx, ty).w01)


def _replicate_left_edge(orig):
    def f(I, m):
        gx, gy = orig(I, m)
        half = np.float32(0.5)
        gx = gx.copy()
        gx[:, 0] = ((half * I[:, 1]) - (half * I[:, 0])) * m[:, 0].astype(np.float32)
        return gx, gy
    return f


MUTATIONS = {
    "drop the window's last pixel": ("pixel_terms", _drop_last_pixel),
    "drop row 0": ("pixel_terms", _drop_row0),
    "round to nearest in >>": ("_shr", lambda orig: lambda v, b: (v + (1 << (b - 1))) >> b),
    "nearest mask rounded with +16": ("ecc_shift", _nearest_plus_16),
    "swap w01 / w10": ("ecc_shift", _swap_w01_w10),
    "replicate instead of reflect-101 at the left edge": ("gradients", _replicate_left_edge),
    "count unmasked pixels into N": ("pixel_terms", _count_unmasked),
    "reverse the order of one sum": ("pixel_terms", _reverse_one_sum),
}


def mutation_cases():
    """Cases tests/test_gpu_registration_exact.py runs: the class's 448 x 358 window of an IR movie, one step from a start whose
    nearest and bilinear origins differ and a whole solve from the identity; and the masked small pair."""
    t, i = ec.ir_window_pair(3)
    G = ek.grid(t.size, ek.B200_SMS, True)
    sm_t, sm_i = ec.small_pair(1.2, 0.7, k=9)
    mask = np.zeros(sm_t.shape, np.uint8)
    mask[10:100, 20:150] = 1
    return [("ir window, one step", t, i, None, -2.3, -1.6, 1, G), ("ir window, solve", t, i, None, 0.0, 0.0, 500, G),
            ("small masked, solve", sm_t, sm_i, mask, 0.0, 0.0, 500, ek.grid(sm_t.size, ek.B200_SMS, True))]


def run_cases():
    out = []
    for _, t, i, mask, tx0, ty0, max_it, G in mutation_cases():
        out.append(ek.solve(ek.prepare(t, i, mask), tx0, ty0, G, max_it=max_it))
    return out


@pytest.fixture(scope="module")
def clean_results():
    return run_cases()


def same_bits(a, b):
    return a[0] == b[0] and a[4] == b[4] and all(np.array(x, np.float64).view(np.uint64) == np.array(y, np.float64).view(np.uint64)
                                                  for x, y in zip(a[1:4], b[1:4]))


@pytest.mark.parametrize("name", list(MUTATIONS))
def test_planted_mutation_is_caught(name, monkeypatch, clean_results):
    attr, make = MUTATIONS[name]
    monkeypatch.setattr(ek, attr, make(getattr(ek, attr)))
    mutated = run_cases()
    changed = [c[0] for c, a, b in zip(mutation_cases(), clean_results, mutated) if not same_bits(a, b)]
    # what a 2e-5 px / 1e-7 bar with equal iteration counts would have said about the same change (recorded in DESIGN §7 f-4)
    slips = [c[0] for c, a, b in zip(mutation_cases(), clean_results, mutated)
             if a[0] != b[0] or a[4] != b[4] or abs(a[1] - b[1]) >= RHO_TOL or max(abs(a[2] - b[2]), abs(a[3] - b[3])) >= SHIFT_TOL]
    print(f"\n{name}: bits change in {changed}; a 2e-5 px bar sees it in {slips}")
    assert changed, f"{name} leaves every case's bits unchanged"
