"""tests/ecc_kernel.py -- numpy restatement of the ECC solver as csrc/ecc.cu computes it, bit for bit.

oracle/ecc.py restates OpenCV's iteration (warped images, zero-meaned copies, dot products); the kernel computes the same
iteration from 15 raw fp64 sums added in a fixed order, so the two differ in the last bits.  This module restates the
kernel's own arithmetic: the clamp, min / max and normalisation, the gradients, the fixed-point shift, the 4-tap warp,
the 15 terms of every pixel, the order in which the grid adds them (which depends on the number of CTAs, hence on the
driver and the SM count), the scalar update and the stopping rule.  tests/test_gpu_registration_exact.py holds the
library to it bit for bit; tests/test_ecc_kernel.py shows that it is OpenCV's iteration and that small slips change its
bits.

Every float32 operation is a numpy float32 operation (one IEEE rounding each, like the kernel's __f*_rn intrinsics) and
every double operation a float64 one (like the __d*_rn intrinsics of ecc_update; a product of two floats is exact).
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np

THREADS = 256      # ECC_THREADS, ecc.cu:90
MAX_SLOTS = 320    # ECC_MAX_SLOTS, ecc.cu:252
B200_SMS = 148
(A_N, A_I, A_T, A_II, A_TT, A_IT, A_H11, A_H12, A_H22, A_B1, A_B2, A_C1, A_C2, A_D1, A_D2) = range(15)  # ecc.cu:40
NACC = 15
F32, F64 = np.float32, np.float64


def grid(n: int, sms: int, fused: bool) -> int:
    """CTAs of the iteration launch for a window of n pixels on a device with `sms` SMs (ecc.cu:905-916, 663).
    The cooperative solve (ecc_fused = 1) runs min(SMs, ceil(n / 256)) CTAs; the launch-per-iteration driver runs
    min(ceil(n / 256), min(2 SMs, 320))."""
    blocks = -(-n // THREADS)
    return min(sms, blocks) if fused else min(blocks, min(2 * sms, MAX_SLOTS))


# ---- clamp, min / max, normalisation, gradients (ecc.cu:60-71, 92-150, 433-479) ------------------------------------
def fkey(a) -> np.ndarray:
    """Order-preserving uint32 key of a float (ecc.cu:60-64)."""
    b = np.ascontiguousarray(a, dtype=F32).view(np.uint32)
    return b ^ np.where((b >> np.uint32(31)) != 0, np.uint32(0xFFFFFFFF), np.uint32(0x80000000))


def fkey_inv(k) -> np.float32:
    """ecc.cu:65-68."""
    k = np.uint32(k)
    return np.array([k ^ (np.uint32(0x80000000) if k >> np.uint32(31) else np.uint32(0xFFFFFFFF))], np.uint32).view(F32)[0]


def clamp_pair(own, other, th) -> np.ndarray:
    """Where either image exceeds the threshold, both take it (ecc.cu:71)."""
    return np.where((own > th) | (other > th), th, own).astype(F32)


def normalise(v, mi, span) -> np.ndarray:
    """(v - mi) / span in float32, two roundings (ecc.cu:124)."""
    with np.errstate(all="ignore"):
        return ((v - mi).astype(F32) / span).astype(F32)


def neighbours(n: int):
    """Reflect-101 neighbours of 0..n-1 (ecc.cu:145-146, 464-465; n >= 2)."""
    i = np.arange(n)
    lo, hi = i - 1, i + 1
    lo[0], hi[-1] = 1, n - 2
    return lo, hi


def gradients(I, m):
    """The [-0.5 0 0.5] derivatives with reflect-101, times the 0/1 mask (ecc.cu:147-149, 466-468)."""
    h, w = I.shape
    xm, xp = neighbours(w)
    ym, yp = neighbours(h)
    half, mf = F32(0.5), m.astype(F32)
    with np.errstate(all="ignore"):
        gx = ((half * I[:, xp]).astype(F32) - (half * I[:, xm]).astype(F32)).astype(F32) * mf
        gy = ((half * I[yp, :]).astype(F32) - (half * I[ym, :]).astype(F32)).astype(F32) * mf
    return gx.astype(F32), gy.astype(F32)


class Prepared(NamedTuple):
    T: np.ndarray      # normalised template
    I: np.ndarray      # normalised image
    gx: np.ndarray     # its gradients times the mask
    gy: np.ndarray
    mask: np.ndarray   # bool, all True without a mask


def prepare(ref, cur, mask=None, thresh=float("inf")) -> Prepared:
    """The solve's first two phases: quantile clamp (NaN = none, ecc.cu:636), min / max by key, normalisation, gradients."""
    ref, cur = np.asarray(ref, F32), np.asarray(cur, F32)
    th = F32("inf") if np.isnan(thresh) else F32(thresh)
    t0, i0 = clamp_pair(ref, cur, th), clamp_pair(cur, ref, th)
    kt, ki = fkey(t0), fkey(i0)
    mi_t, mi_i = fkey_inv(kt.min()), fkey_inv(ki.min())
    with np.errstate(all="ignore"):
        span_t, span_i = F32(fkey_inv(kt.max()) - mi_t), F32(fkey_inv(ki.max()) - mi_i)
    T, I = normalise(t0, mi_t, span_t), normalise(i0, mi_i, span_i)
    m = np.ones(ref.shape, bool) if mask is None else np.asarray(mask) != 0
    gx, gy = gradients(I, m)
    return Prepared(T, I, gx, gy, m)


# ---- one iteration's sums (ecc.cu:169-226) ---------------------------------------------------------------------------
def _shr(v: int, b: int) -> int:
    """The kernel's arithmetic right shift of a signed int: floor(v / 2^b)."""
    return v >> b


class Shift(NamedTuple):
    ox: int
    oy: int
    oxn: int
    oyn: int
    w00: np.float32
    w01: np.float32
    w10: np.float32
    w11: np.float32


def ecc_shift(tx, ty) -> Shift:
    """EccShift (ecc.cu:169-185): warpAffine's fixed point for a translation, AB_BITS = 10, INTER_BITS = 5."""
    SX, SY = int(np.rint(float(F32(tx)) * 1024.0)), int(np.rint(float(F32(ty)) * 1024.0))  # __double2int_rn
    fx, fy = F32(_shr(SX + 16, 5) & 31) * F32(0.03125), F32(_shr(SY + 16, 5) & 31) * F32(0.03125)
    one = F32(1)
    return Shift(_shr(SX + 16, 10), _shr(SY + 16, 10), _shr(SX + 512, 10), _shr(SY + 512, 10),
                 F32((one - fy) * (one - fx)), F32((one - fy) * fx), F32(fy * (one - fx)), F32(fy * fx))


def shifted(a, dy: int, dx: int, fill=0):
    """out[y, x] = a[y + dy, x + dx] where that is inside a, else `fill` (the kernel's bounds tests)."""
    h, w = a.shape
    out = np.full((h, w), fill, a.dtype)
    y0, y1, x0, x1 = max(0, -dy), min(h, h - dy), max(0, -dx), min(w, w - dx)
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = a[y0 + dy:y1 + dy, x0 + dx:x1 + dx]
    return out


def warp(s, sh: Shift) -> np.ndarray:
    """remapBilinear with a zero border: ((s00 w00 + s01 w01) + s10 w10) + s11 w11 in float32 (ecc.cu:198-203)."""
    with np.errstate(all="ignore"):
        v = (shifted(s, sh.oy, sh.ox) * sh.w00).astype(F32) + (shifted(s, sh.oy, sh.ox + 1) * sh.w01).astype(F32)
        v = v.astype(F32) + (shifted(s, sh.oy + 1, sh.ox) * sh.w10).astype(F32)
        return (v.astype(F32) + (shifted(s, sh.oy + 1, sh.ox + 1) * sh.w11).astype(F32)).astype(F32)


def pixel_terms(p: Prepared, sh: Shift) -> list:
    """The 15 values each pixel adds, in pixel order p = y w + x (ecc.cu:204-224).  A pixel outside the warped mask adds
    nothing to the ten masked sums; adding +0.0 instead is the same, since no partial sum is ever -0.0."""
    Iw, Gx, Gy = (warp(a, sh).astype(F64).ravel() for a in (p.I, p.gx, p.gy))
    m = shifted(p.mask, sh.oyn, sh.oxn, False).ravel()  # nearest (ecc.cu:205-206)
    t = p.T.astype(F64).ravel()
    z = F64(0)
    with np.errstate(all="ignore"):
        v = [None] * NACC
        v[A_H11], v[A_H12], v[A_H22], v[A_B1], v[A_B2] = Gx * Gx, Gx * Gy, Gy * Gy, Gx * Iw, Gy * Iw
        v[A_N] = m.astype(F64)
        v[A_I], v[A_T] = np.where(m, Iw, z), np.where(m, t, z)
        v[A_II], v[A_TT], v[A_IT] = np.where(m, Iw * Iw, z), np.where(m, t * t, z), np.where(m, Iw * t, z)
        v[A_C1], v[A_C2] = np.where(m, Gx, z), np.where(m, Gy, z)
        v[A_D1], v[A_D2] = np.where(m, Gx * t, z), np.where(m, Gy * t, z)
    return v


def grid_sum(v, G: int) -> np.float64:
    """The sum of v as a grid of G CTAs of 256 threads adds it.
    Thread g (of G 256) adds pixels g, g + G 256, ... in turn (ecc.cu:193, 354, 490); each warp folds its 32 lanes
    with shfl_down 16/8/4/2/1, each CTA adds its 8 warps in turn from 0.0 (ecc.cu:230-246); then value k's 8 adding
    threads take slots j, j + 8, ... from 0.0 and fold with shfl_down 4/2/1 in groups of 8 (ecc.cu:253-282)."""
    nt = G * THREADS
    v = np.asarray(v, F64)
    k = -(-len(v) // nt)
    with np.errstate(all="ignore"):
        a = np.zeros(nt, F64)
        if k:  # +0.0 for threads past the end: a partial sum is never -0.0, so adding it changes nothing
            padded = np.zeros(k * nt, F64)
            padded[:len(v)] = v
            for row in padded.reshape(k, nt):
                a = a + row
        lanes = a.reshape(G * 8, 32)
        for o in (16, 8, 4, 2, 1):
            lanes[:, :32 - o] = lanes[:, :32 - o] + lanes[:, o:]
        warps = lanes[:, 0].reshape(G, 8)
        cta = np.zeros(G, F64)
        for q in range(8):
            cta = cta + warps[:, q]
        slots = np.zeros(-(-G // 8) * 8, F64)
        slots[:G] = cta
        j = np.zeros(8, F64)
        for row in slots.reshape(-1, 8):
            j = j + row
        j4 = j[:4] + j[4:]
        j2 = j4[:2] + j4[2:]
        return F64(j2[0] + j2[1])


def sums(p: Prepared, tx, ty, G: int) -> np.ndarray:
    sh = ecc_shift(tx, ty)
    return np.array([grid_sum(v, G) for v in pixel_terms(p, sh)], F64)


# ---- the scalar update and the stopping rule (ecc.cu:284-337) ------------------------------------------------------
class State(NamedTuple):
    tx: np.float32
    ty: np.float32
    rho: float
    last_rho: float
    it: int
    status: int
    done: bool


def start(tx0, ty0, max_it=500, eps=1e-3) -> State:
    """ecc.cu:80-85, 482-483: rho = -1, last_rho = -eps."""
    rho, last = F64(-1.0), F64(-eps)
    return State(F32(tx0), F32(ty0), rho, last, 0, 0, bool(max_it <= 0 or not (abs(rho - last) >= eps)))


def update(acc, s: State, max_it=500, eps=1e-3) -> State:
    """ecc_update: OpenCV's float / double types, every double operation rounded on its own."""
    d = F64
    n, sI, sT, sII, sTT, sIT, h11, h12, h22, b1, b2, c1, c2, d1, d2 = (d(a) for a in acc)
    it, status, tx, ty, rho, last_rho = s.it + 1, 0, s.tx, s.ty, d(s.rho), d(s.last_rho)
    with np.errstate(all="ignore"):
        if n <= 0.0:
            status = 1
        else:
            meanI, meanT = sI / n, sT / n
            varI, varT = np.fmax(sII / n - meanI * meanI, d(0)), np.fmax(sTT / n - meanT * meanT, d(0))
            img_norm, tmp_norm = np.sqrt(n * varI), np.sqrt(n * varT)
            muI, muT = d(F32(meanI)), d(F32(meanT))
            H11, H12, H22 = d(F32(h11)), d(F32(h12)), d(F32(h22))
            det = H11 * H22 - H12 * H12
            idet = d(1.0) / det if det != 0.0 else d(0)
            Hi11, Hi22, Hi12 = d(F32(H22 * idet)), d(F32(H11 * idet)), d(F32(-H12 * idet))
            corr = ((sIT - muT * sI) - muI * sT) + (muI * muT) * n
            last_rho, rho = rho, corr / (img_norm * tmp_norm)
            if np.isnan(rho) or det == 0.0:
                status = 1
            else:
                pI1, pI2 = b1 - muI * c1, b2 - muI * c2
                pT1, pT2 = d1 - muT * c1, d2 - muT * c2
                ip1, ip2, tp1, tp2 = (d(F32(x)) for x in (pI1, pI2, pT1, pT2))
                iph1, iph2 = d(F32(Hi11 * ip1 + Hi12 * ip2)), d(F32(Hi12 * ip1 + Hi22 * ip2))
                lam_n = img_norm * img_norm - (ip1 * iph1 + ip2 * iph2)
                lam_d = corr - (tp1 * iph1 + tp2 * iph2)
                if lam_d <= 0.0:
                    rho, status = d(-1.0), 2
                else:
                    lam = lam_n / lam_d
                    e1, e2 = d(F32(lam * pT1 - pI1)), d(F32(lam * pT2 - pI2))
                    tx = F32(tx + F32(Hi11 * e1 + Hi12 * e2))
                    ty = F32(ty + F32(Hi12 * e1 + Hi22 * e2))
        done = status != 0 or it >= max_it or not (abs(rho - last_rho) >= eps)
    return State(tx, ty, rho, last_rho, it, status, bool(done))


def step(p: Prepared, s: State, G: int, max_it=500, eps=1e-3) -> State:
    """One iteration from state s."""
    return update(sums(p, s.tx, s.ty, G), s, max_it, eps)


def solve(p: Prepared, tx0, ty0, G: int, max_it=500, eps=1e-3):
    """The whole solve -> (status, rho, tx, ty, iterations); tx, ty are the solver's last shift whatever the status
    (rirb_ecc_compute hands back the start instead when status != 0)."""
    s = start(tx0, ty0, max_it, eps)
    while not s.done:
        s = step(p, s, G, max_it, eps)
    return s.status, float(s.rho), float(s.tx), float(s.ty), s.it
