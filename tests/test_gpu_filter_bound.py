"""The proof inputs of the filtered projection (DESIGN.md §4a) against a float64 restatement, read from the workspace
a pass leaves behind: k_unproject's point cloud and per-point coefficient C_point, and make_homography's
recentred fp32 homography Hf, its error coefficient E_cand and the exact-only flag of every candidate.  Then the
bound itself, pair by pair, on the device's numbers.

Bit-exact:
  * the point cloud: per job the count, the packed source pixels in np.nonzero (row-major) order, X, Y, Z against
    oracle.restated.get_pcd / pcd_to_f32 (NaN triples for non-finite points), and the poisoned tail of every plane;
  * the exact-only flag against §4a's rule restated from a numpy homography (only candidates whose worst corner sits
    within 1e-6 of the 0.02 threshold of the fix_x / fix_y test are undecidable in another fp64 evaluation order;
    none of the scenarios has one, and the test says so if that changes);
  * the same job alone (its phase 2 split over 32 CTAs) and inside a batch of 300 jobs (one CTA per job).

Bounded, each with the tolerance its arithmetic allows:
  * C_point and E_cand: restated <= device <= restated * (1 + 1e-6) * (1 + 2^-23) * (1 + 2^-24) * (1 + 1e-12).
    The kernel multiplies its fp64 value by 1.000001 and rounds up to fp32 (2^-23), so the device value can be no
    smaller than the exact formula and at most that much larger.  2^-24 covers |p - a|_1 taken in fp64 by the
    kernel against the fp32 p' = fl(p - a) of §4a, 1e-12 the order of the fp64 evaluation.
    C_point is +inf exactly where the point is non-finite, its ray nearly lies in the plane, or the value overflows.
  * Hf: |Hf * scale - H| <= 2^-24 |H| + 2^-40 * shadow per entry, §4a's error model: one rounding to fp32 after an
    fp64 evaluation whose error the absolute-value shadow times 2^-40 covers (fp64 differs by ~1e-15 * shadow).

The bound, on every (point, filtered candidate) pair, with q* and W_h from the float64 homography of the
unrecentred H and q_ref the reference's fp32 u/w in the operation order of oracle.restated.project_pixels:
  1. |q_ref - q*| <= C_point |1/W_h| + 2^-24 D where q* lies in [0, D]: the value form.  §4a's side-of-boundary
     argument bounds |u_c - m w_c| for integers m <= D; the same terms bound |u_c - q* w_c| for |q*| <= D, and the
     u D term covers the rounding of the division.
  2. |q_f - q*| <= E_cand |1/W_h| + (D+1)(2^-22 + 6 * 2^-24) where q* lies in [0, D], q_f from the device's Hf by
     two fp32 FMAs per row, a reciprocal at either end of its 2^-22 relative error, and the scaled FMA of the kernel.
  3. The kernel's decision |d| <= 1/2 - eps with each point's own C_point (at least as many proofs as the kernel's
     largest C per 8-point item): every proven pixel equals the reference chain's, at both ends of the reciprocal.
The FMA emulation is exact: fp32 x fp32 and fp32 x 16-bit products are exact in float64, the sum is split into its
float64 value and error (TwoSum) and rounded to fp32 once (the error decides a float64 value that sits halfway
between two floats).  Every pair check runs as float64 torch element-wise operations, one rounding each.

The unproven share (the kernel's per-item C, the correctly rounded reciprocal) is a performance property: a bound
that is too loose keeps every pixel right and sends pairs to the ~80-instruction chain."""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, engine, geometry, workloads
from oracle import restated

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U = 2.0 ** -24
FLT_MAX = float(np.finfo(np.float32).max)
POISON = 0xABABABAB
SEQ, COMPOSED, TRANSLATE = _lib.MODE_SEQ, _lib.MODE_COMPOSED, _lib.MODE_TRANSLATE
MAGIC = np.float32(12582912.0)                 # 1.5 * 2^23, the kernel's rint constant
CHUNK = 1 << 23                                 # (candidate, point) pairs per step of the pair checks
# the kernel's factor of every coefficient it rounds up: device / restated lies in [1, TOL_HI]
TOL_HI = (1 + 1e-6) * (1 + 2.0 ** -23) * (1 + 2.0 ** -24) * (1 + 1e-12)
# ceilings of the unproven share of filtered-candidate pairs per mode on the workload passes (test_workload_pass)
UNPROVEN_CEILING = {SEQ: None, COMPOSED: None, TRANSLATE: None}


# ---------------------------------------------------------------------------------------------------------------
# exact fp32 operations in float64
# ---------------------------------------------------------------------------------------------------------------
def _inf_like(t, sign):
    return torch.full_like(t, math.inf if sign > 0 else -math.inf)


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)          # a + b == s + e exactly


def _round_once(s, e):
    """fp32 of the exact s + e (float64 s, |e| <= ulp(s)/2): s.float() unless s sits halfway between two floats."""
    r = s.float()
    rd = r.double()
    other = torch.nextafter(r, torch.where(s > rd, _inf_like(r, 1), _inf_like(r, -1)))
    tie = (s == (rd + other.double()) * 0.5) & (e != 0)
    nudged = torch.nextafter(s, torch.where(e > 0, _inf_like(s, 1), _inf_like(s, -1))).float()
    return torch.where(tie, nudged, r)


def _fma32(a, b, c):
    """fmaf(a, b, c) of fp32 tensors, rounded once."""
    s, e = _two_sum(a.double() * b.double(), c.double())
    return _round_once(s, e)


def _add_ru32(a, b):
    """__fadd_ru(a, b) of fp32 tensors."""
    s, e = _two_sum(a.double(), b.double())
    r = s.float()
    rd = r.double()
    up = (rd < s) | ((rd == s) & (e > 0))
    return torch.where(up, torch.nextafter(r, _inf_like(r, 1)), r)


def _f32_dir(t, up):
    """fp32 nearest to the float64 t in one direction (up: smallest >= t, else largest <= t)."""
    r = t.float()
    rd = r.double()
    if up:
        return torch.where(rd < t, torch.nextafter(r, _inf_like(r, 1)), r)
    return torch.where(rd > t, torch.nextafter(r, _inf_like(r, -1)), r)


def _ru32(q: Fraction) -> Fraction:
    r = np.float32(float(q))
    if Fraction(float(r)) < q:
        r = np.nextafter(r, np.float32(np.inf))
    return Fraction(float(r))


def _c0h(D: int) -> np.float32:
    """splat_job_filter's c0 - 1/2: 1.0001 ((D+1) 10u + u D) - 1/2, every operation of fp32 operands rounded up."""
    f = lambda v: Fraction(float(np.float32(v)))  # noqa: E731
    Dm = f(D)
    inner = _ru32(_ru32(_ru32(Dm + 1) * f(5.9604645e-7)) + _ru32(Dm * f(5.9604645e-8)))
    return np.float32(float(_ru32(_ru32(inner * f(1.0001)) + f(-0.5))))


# ---------------------------------------------------------------------------------------------------------------
# a pass and what its workspace holds
# ---------------------------------------------------------------------------------------------------------------
def _unpack(bits: torch.Tensor, W: int) -> np.ndarray:
    b = bits.cpu().numpy().view(np.uint32)
    u8 = b.view(np.uint8).reshape(b.shape[0], b.shape[1], -1)
    return np.unpackbits(u8, axis=-1, bitorder="little")[..., :W].astype(bool)


class Camera:
    def __init__(self, cfg, kinv=None):
        self.kinv = np.asarray(cfg.K_inv() if kinv is None else kinv, np.float64)
        self.f, self.cx, self.cy = (float(np.float32(v)) for v in (cfg.focal_length, cfg.cx, cfg.cy))
        self.H, self.W = int(cfg.height), int(cfg.width)
        self.D = max(self.H, self.W)
        self.K_inv = lambda: self.kinv            # what oracle.restated.get_pcd asks of its config


def run_filter_pass(cfg, pool, batch, monkeypatch, kinv=None):
    """One pass through k_project<filter> on a fresh poisoned workspace; returns the camera and host copies of the
    source masks, the point-cloud workspace, the counts and the homography rows."""
    monkeypatch.setenv("A3D_PROJECT_KERNEL", "filter")
    monkeypatch.setenv("A3D_WS_POISON", "1")
    if kinv is not None:
        cs = engine.camera_struct(cfg)
        for i, v in enumerate(np.asarray(kinv, np.float64).reshape(-1)):
            cs.kinv[i] = float(v)
        monkeypatch.setattr(engine, "_camera_cached", lambda c: cs)
    ws = engine.Workspace(DEV)
    engine.run_pass(cfg, pool, engine.DeviceBatch(batch, DEV), ws)
    torch.cuda.synchronize()
    nc = int(batch.xform.shape[0])
    srcs = sorted(set(int(s) for s in batch.jobs["src_mask"]))
    src = dict(zip(srcs, _unpack(pool.source_bits[srcs], cfg.width)))
    return dict(cam=Camera(cfg, kinv), batch=batch, src=src, pcd=ws._bufs["pcd_ws"].cpu().numpy(),
                count=ws._bufs["pcd_count"].cpu().numpy()[:batch.n_jobs],
                hom=ws._bufs["hom_ws"].cpu().numpy()[:nc * 12].reshape(nc, 12))


def job_slice(p, j):
    jb = p["batch"].jobs[j]
    cap, b = int(jb["pcd_cap"]), _lib.PCD_PLANES * int(jb["pcd_begin"])
    return p["pcd"][b:b + _lib.PCD_PLANES * cap].reshape(_lib.PCD_PLANES, cap)


def job_hom(p, j):
    jb = p["batch"].jobs[j]
    c0 = int(jb["cand_begin"])
    return p["hom"][c0:c0 + int(jb["n_cand"])]


# ---------------------------------------------------------------------------------------------------------------
# float64 restatement of DESIGN.md §4a
# ---------------------------------------------------------------------------------------------------------------
def _word_box(src):
    rows, cols = np.nonzero(src.any(1))[0], np.nonzero(src.any(0))[0]
    return int(rows[0]), int(rows[-1]), int(cols[0]) // 32, int(cols[-1]) // 32


def _centre(box):
    """(x0, y0) the kernel recentres on, (xm, ym) the largest |x - x0|, |y - y0| over the word box."""
    r0, r1, w0, w1 = box
    x0, y0 = 16 * (w0 + w1 + 1), (r0 + r1) // 2
    return x0, y0, max(abs(32 * w0 - x0), abs(32 * w1 + 31 - x0)), max(abs(r0 - y0), abs(r1 - y0))


def _affine(jb, xf):
    """(A, b) of s = p A + b for every candidate, and their absolute-value shadows."""
    n, mode = len(xf), int(jb["mode"])
    a = jb["pivot"].astype(np.float64)
    R = xf[:, :9].astype(np.float64).reshape(n, 3, 3)
    t = xf[:, 9:].astype(np.float64)
    if mode == TRANSLATE:
        A = np.broadcast_to(np.eye(3), (n, 3, 3))
        return A, t, A, np.abs(t)
    if mode == SEQ:
        return R, a[None] - np.einsum("k,nkj->nj", a, R), np.abs(R), np.abs(a)[None] + np.einsum("k,nkj->nj", np.abs(a), np.abs(R))
    return R, t, np.abs(R), np.abs(t)


def homography(cam, jb, xf):
    """H = K (off A + n b^T)^T K^-1 (rows u, v, w; columns x, y, 1) and its absolute-value shadow."""
    A, b, Aa, ba = _affine(jb, xf)
    n = jb["normal"].astype(np.float64)
    off = float(jb["offset"])
    K = np.array([[cam.f, 0.0, cam.cx], [0.0, cam.f, cam.cy], [0.0, 0.0, 1.0]])
    with np.errstate(all="ignore"):
        G = off * A + n[None, :, None] * b[:, None, :]
        Ga = abs(off) * Aa + np.abs(n)[None, :, None] * ba[:, None, :]
        return K @ G.transpose(0, 2, 1) @ cam.kinv, np.abs(K) @ Ga.transpose(0, 2, 1) @ np.abs(cam.kinv)


def restate_candidates(cam, jb, xf, box, hf_dev):
    """Per candidate: the unrecentred H, the recentred Hc and shadow, E_cand from the device's Hf, and the
    exact-only rule with its reasons."""
    x0, y0, xm, ym = _centre(box)
    H, Ha = homography(cam, jb, xf)
    Hc, Hca = H.copy(), Ha.copy()
    Hc[:, :, 2] = H[:, :, 0] * x0 + H[:, :, 1] * y0 + H[:, :, 2]
    Hca[:, :, 2] = Ha[:, :, 0] * x0 + Ha[:, :, 1] * y0 + Ha[:, :, 2]
    scale = np.array([cam.W - 1, cam.H - 1, 1.0])
    with np.errstate(all="ignore"):
        hf_own = (Hc / scale[None, :, None]).astype(np.float32)

        def ecand(hf):
            mag = scale[None] * (np.abs(hf[:, :, 0].astype(np.float64)) * xm + np.abs(hf[:, :, 1].astype(np.float64)) * ym
                                 + np.abs(hf[:, :, 2].astype(np.float64)))
            maga = Hca[:, :, 0] * xm + Hca[:, :, 1] * ym + Hca[:, :, 2]
            return 1.25 * (3 * U * (np.maximum(mag[:, 0], mag[:, 1]) + (cam.D + 1) * mag[:, 2])
                           + 2.0 ** -40 * (np.maximum(maga[:, 0], maga[:, 1]) + (cam.D + 1) * maga[:, 2]))

        fix = {}
        for k, c in (("x", 0), ("y", 1)):
            worst = np.zeros(len(xf))
            for xx in (-xm, xm):
                for yy in (-ym, ym):
                    w = Hc[:, 2, 0] * xx + Hc[:, 2, 1] * yy + Hc[:, 2, 2]
                    own = (xx + x0, yy + y0)[c]
                    worst = np.maximum(worst, np.abs(Hc[:, c, 0] * xx + Hc[:, c, 1] * yy + Hc[:, c, 2] - own * w) / np.abs(w))
            fix[k] = worst                     # |u - x w| / |w| at the worst corner: fixed when < 0.02
        e_own, e_dev = ecand(hf_own), ecand(hf_dev)
        reasons = dict(
            rho=(np.zeros(len(xf), bool) if int(jb["mode"]) == TRANSLATE
                 else ~(np.abs(xf[:, :9].astype(np.float64)) <= 1.001).all(1)),
            hf=~((np.abs(hf_own) <= np.float32(3.0e38)).reshape(len(xf), 9).all(1)),
            size=np.full(len(xf), cam.W < 2 or cam.H < 2),
            ecand=~(e_own * (1 + 1e-6) <= 3.0e38),
            fix_x=fix["x"] < 0.02, fix_y=fix["y"] < 0.02)
    flag = np.zeros(len(xf), bool)
    for v in reasons.values():
        flag |= v
    undecided = (np.abs(fix["x"] - 0.02) < 2e-8) | (np.abs(fix["y"] - 0.02) < 2e-8)
    return dict(H=H, Hc=Hc, Hca=Hca, scale=scale, E=e_dev, flag=flag, reasons=reasons, fix=fix,
                undecided=undecided, centre=(x0, y0, xm, ym))


def restate_points(cam, jb, xf, cols, rows, P32):
    """C_point of §4a per point, and where it must be +inf."""
    x, y = cols.astype(np.float64), rows.astype(np.float64)
    k = cam.kinv
    n = jb["normal"].astype(np.float32).astype(np.float64)
    with np.errstate(all="ignore"):
        ray = [(k[i, 0] * x + k[i, 1] * y) + k[i, 2] for i in range(3)]
        dot = (n[0] * ray[0] + n[1] * ray[1]) + n[2] * ray[2]
        dmag = (np.abs(n[0] * ray[0]) + np.abs(n[1] * ray[1])) + np.abs(n[2] * ray[2])
        finite = np.isfinite(P32).all(1)
        p1 = np.abs(P32.astype(np.float64)).sum(1)
        if int(jb["mode"]) == SEQ:
            a = jb["pivot"].astype(np.float32)
            pp1 = np.abs((P32 - a[None]).astype(np.float64)).sum(1)     # p' = fl(p - a) in fp32
            amax = float(np.abs(a.astype(np.float64)).max())
            Sig = 1.001 * (1.01 * p1 + 5 * pp1) + amax
            M = 1.001 * pp1 + amax
        else:
            t = np.abs(xf[:, 9:].astype(np.float64))
            tmax = math.inf if np.isnan(t).any() else float(t.max())
            Sig = 1.001 * 5.01 * p1 + tmax
            M = 1.001 * p1 + tmax
        K1 = cam.f + max(abs(cam.cx), abs(cam.cy))
        Cp = 1.25 * U * np.abs(dot) * (K1 * (Sig + 2 * M) + cam.D * Sig)
        inf = ~finite | ~(np.abs(dot) >= 1e-6 * dmag) | ~(Cp * (1 + 1e-6) <= FLT_MAX)
    return Cp, inf


# ---------------------------------------------------------------------------------------------------------------
# A + B: what k_unproject and make_homography wrote
# ---------------------------------------------------------------------------------------------------------------
def check_point_cloud(p, j):
    """Bit-exact point cloud of job j; returns (cols, rows, XYZ fp32, device C)."""
    cam, jb = p["cam"], p["batch"].jobs[j]
    src = p["src"][int(jb["src_mask"])]
    rows, cols = np.nonzero(src)
    P, cnt, cap = len(rows), int(p["count"][j]), int(jb["pcd_cap"])
    assert cnt == P == int(src.sum()), (j, cnt, P)
    sl = job_slice(p, j)
    assert np.array_equal(sl[3, :P].view(np.uint32), (rows.astype(np.uint32) << 16) | cols.astype(np.uint32)), j
    want = restated.pcd_to_f32(restated.get_pcd(np.stack([cols, rows], 1), jb["normal"], float(jb["offset"]), cam))
    got = np.ascontiguousarray(sl[:3, :P].T)
    nan_w, nan_g = np.isnan(want), np.isnan(got)
    assert np.array_equal(nan_w, nan_g), j
    assert np.array_equal(nan_g.all(1), nan_g.any(1)), j            # non-finite points are NaN triples
    assert np.array_equal(got[~nan_g].view(np.uint32), want[~nan_w].view(np.uint32)), j
    assert (sl[:, P:].view(np.uint32) == POISON).all(), j             # nothing written past the count
    return cols, rows, got, sl[4, :P].copy()


def check_coefficients(p, j, cols, rows, P32, Cdev):
    """C_point, Hf, E_cand and the flag of job j against the restatement; returns the candidate restatement."""
    cam, jb = p["cam"], p["batch"].jobs[j]
    c0, A = int(jb["cand_begin"]), int(jb["n_cand"])
    xf = p["batch"].xform[c0:c0 + A]
    Cp, inf = restate_points(cam, jb, xf, cols, rows, P32)
    assert np.array_equal(np.isposinf(Cdev), inf), j
    assert not np.isnan(Cdev).any()
    fin = ~inf
    c = Cdev[fin].astype(np.float64)
    assert (c >= Cp[fin]).all(), (j, float(np.min(c / Cp[fin])))
    assert (c <= Cp[fin] * TOL_HI).all(), (j, float(np.max(c / Cp[fin])))

    hom = job_hom(p, j)
    hf = hom[:, :9].reshape(A, 3, 3)
    rc = restate_candidates(cam, jb, xf, _word_box(p["src"][int(jb["src_mask"])]), hf)
    assert (hom[:, 11] == 0).all()
    dec = ~rc["undecided"]
    assert np.array_equal((hom[:, 10] != 0)[dec], rc["flag"][dec]), (j, np.nonzero((hom[:, 10] != 0) != rc["flag"])[0])
    assert set(np.unique(hom[:, 10])) <= {0.0, 1.0}
    ok = ~rc["flag"]                                                  # finite, in range
    err = np.abs(hf[ok].astype(np.float64) * rc["scale"][None, :, None] - rc["Hc"][ok])
    assert (err <= U * np.abs(rc["Hc"][ok]) + 2.0 ** -40 * rc["Hca"][ok]).all(), j
    E, Edev = rc["E"][ok], hom[ok, 9].astype(np.float64)
    assert (Edev >= E).all() and (Edev <= E * TOL_HI).all(), (j, float(np.max(Edev / E)), float(np.min(Edev / E)))
    return rc


# ---------------------------------------------------------------------------------------------------------------
# C + D: the bound on every (point, filtered candidate) pair
# ---------------------------------------------------------------------------------------------------------------
def _oracle_pixel(q, n):
    """.long() on x86 and the clamp of oracle.restated.project_pixels."""
    bad = ~(q.abs() < 9.223372036854775807e18)
    v = torch.where(bad, torch.zeros_like(q), q).trunc()
    return torch.where(bad, torch.zeros_like(v), v.clamp(0, n - 1)).double()


def _reference_q(mode, X, Y, Z, m, pivot, cam):
    """The reference chain's fp32 u/w and v/w (transform of oracle.restated, then project_pixels' order)."""
    f32 = lambda v: torch.tensor(float(np.float32(v)), dtype=torch.float32, device=X.device)  # noqa: E731
    if mode == TRANSLATE:
        s = [X + m[:, 9:10], Y + m[:, 10:11], Z + m[:, 11:12]]
    else:
        if mode == SEQ:
            a = [f32(v) for v in pivot]
            X, Y, Z = X - a[0], Y - a[1], Z - a[2]
        s = [(X * m[:, j:j + 1] + Y * m[:, 3 + j:4 + j]) + Z * m[:, 6 + j:7 + j] for j in range(3)]
        s = [s[j] + a[j] for j in range(3)] if mode == SEQ else [s[j] + m[:, 9 + j:10 + j] for j in range(3)]
    fl, cx, cy, zero, one = f32(cam.f), f32(cam.cx), f32(cam.cy), f32(0), f32(1)
    u = (fl * s[0] + zero * s[1]) + cx * s[2]
    v = (zero * s[0] + fl * s[1]) + cy * s[2]
    w = (zero * s[0] + zero * s[1]) + one * s[2]
    return u / w, v / w


def new_stats():
    return dict(pairs=0, pairs_filtered=0, r1=0.0, r2=0.0, proven=0, wrong=0, unproven=0, oracle_checked=0)


def check_pairs(p, j, cols, rows, P32, Cdev, rc, st):
    """Components 1-3 of the bound and the unproven share for every pair of job j's filtered candidates."""
    cam, jb = p["cam"], p["batch"].jobs[j]
    mode = int(jb["mode"])
    c0, A = int(jb["cand_begin"]), int(jb["n_cand"])
    P = len(cols)
    st["pairs"] += P * A
    cand = np.nonzero(~rc["flag"])[0]
    if P == 0 or len(cand) == 0:
        return
    x0, y0 = rc["centre"][:2]
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(DEV, dt)  # noqa: E731
    X, Y, Z = (d(P32[:, i], torch.float32) for i in range(3))
    xd, yd = d(cols, torch.float64), d(rows, torch.float64)
    xs, ys = d(cols - x0, torch.float32), d(rows - y0, torch.float32)   # the kernel's 16-bit source coordinates
    Cpt = d(Cdev, torch.float32)
    pad = np.zeros(-P % 8, np.float32)
    Citem = d(np.repeat(np.concatenate([Cdev, pad]).reshape(-1, 8).max(1), 8)[:P], torch.float32)
    D = cam.D
    wmax, hmax = np.float32(cam.W - 1), np.float32(cam.H - 1)
    sc = lambda v: torch.tensor(float(np.float32(v)), dtype=torch.float32, device=DEV)  # noqa: E731
    chx, chy = sc(np.float32(-0.5 / np.float64(wmax))), sc(np.float32(-0.5 / np.float64(hmax)))
    c0h, magic = sc(_c0h(D)), sc(MAGIC)
    tw, th = sc(wmax), sc(hmax)
    xf = p["batch"].xform[c0:c0 + A]
    hom = job_hom(p, j)
    step = max(1, CHUNK // P)
    for lo in range(0, len(cand), step):
        ci = cand[lo:lo + step]
        st["pairs_filtered"] += P * len(ci)
        Hs = d(rc["H"][ci], torch.float64)
        hf = d(hom[ci, :9], torch.float32)
        E = d(hom[ci, 9:10], torch.float32)
        m = d(xf[ci], torch.float32)
        h = lambda r, c: Hs[:, r, c:c + 1]  # noqa: E731
        Wh = (h(2, 0) * xd + h(2, 1) * yd) + h(2, 2)
        qs = [((h(0, 0) * xd + h(0, 1) * yd) + h(0, 2)) / Wh, ((h(1, 0) * xd + h(1, 1) * yd) + h(1, 2)) / Wh]
        inv_w = (1.0 / Wh).abs()
        inr = [(q >= 0) & (q <= D) for q in qs]
        qr = _reference_q(mode, X, Y, Z, m, jb["pivot"], cam)
        pix = [_oracle_pixel(qr[0], cam.W), _oracle_pixel(qr[1], cam.H)]
        if lo == 0:                                                   # the torch chain against the oracle's numpy one
            k = ci[:4]
            if mode == TRANSLATE:
                pts = restated.transform_translate(P32, xf[k, 9:])
            else:
                Rm = xf[k, :9].reshape(-1, 3, 3)
                pts = (restated.transform_seq(P32, jb["pivot"], Rm) if mode == SEQ
                       else restated.transform_composed(P32, Rm, xf[k, 9:]))
            ocfg = restated.OracleConfig(height=cam.H, width=cam.W, focal_length=float(cam.f))
            orow, ocol = restated.project_pixels(pts, ocfg, cam.H, cam.W)
            assert np.array_equal(pix[0][:len(k)].cpu().numpy(), ocol) and np.array_equal(pix[1][:len(k)].cpu().numpy(), orow)
            st["oracle_checked"] += orow.size
        # 1. the reference chain
        eps_ref = Cpt.double() * inv_w + U * D
        fin = torch.isfinite(Cpt)
        for q, qref, ir in zip(qs, qr, inr):
            sel = ir & fin
            if sel.any():
                st["r1"] = max(st["r1"], float(((qref.double() - q).abs() / eps_ref)[sel].max()))
        # 2. + 3. the cheap value and the decision, at both ends of the reciprocal
        hq = lambda r, c: hf[:, 3 * r + c:3 * r + c + 1]  # noqa: E731
        Uq, Vq, Wq = (_fma32(hq(r, 0), xs, _fma32(hq(r, 1), ys, hq(r, 2))) for r in range(3))
        eps_f = E.double() * inv_w + (D + 1) * (2.0 ** -22 + 6 * U)
        t = 1.0 / Wq.double()
        ftz = Wq.abs() < 2.0 ** -126                                  # rcp.approx.ftz: subnormal -> +-0 -> +-inf
        ends = [torch.where(ftz, torch.copysign(_inf_like(t, 1), Wq.double()), torch.copysign(_f32_dir(t.abs() * (1 + s * 2.0 ** -22), s < 0).double(), t)).float()
                for s in (-1, 1)]
        ends.append(torch.where(ftz, torch.copysign(_inf_like(t, 1), Wq.double()), t).float())   # nominal
        for ei, r in enumerate(ends):
            sxr, syr = _fma32(Uq, r, chx), _fma32(Vq, r, chy)
            if ei < 2:
                for sr, n1, q, ir in ((sxr, cam.W - 1, qs[0], inr[0]), (syr, cam.H - 1, qs[1], inr[1])):
                    if ir.any():
                        qf = sr.double() * n1 + 0.5
                        st["r2"] = max(st["r2"], float(((qf - q).abs() / eps_f)[ir].max()))
            sat = lambda v: torch.where(torch.isnan(v), torch.zeros_like(v), v.clamp(0, 1))  # noqa: E731
            sx, sy = sat(sxr), sat(syr)
            nx = _fma32(sx, tw, magic).double() - float(MAGIC)
            ny = _fma32(sy, th, magic).double() - float(MAGIC)
            dx, dy = _fma32(sx, tw, (-nx).float()), _fma32(sy, th, (-ny).float())
            Cuse = Cpt if ei < 2 else Citem
            neg = _fma32(_add_ru32(Cuse, E), r.abs(), c0h)
            proven = (dx.abs() <= -neg) & (dy.abs() <= -neg)
            if ei < 2:
                st["proven"] += int(proven.sum())
                st["wrong"] += int((proven & ((nx != pix[0]) | (ny != pix[1]))).sum())
            else:
                st["unproven"] += int((~proven).sum())


def check_pass(p, label, jobs=None):
    """A, B and C on every job (or the given ones) of a pass; prints and returns the statistics."""
    st = new_stats()
    for j in (range(p["batch"].n_jobs) if jobs is None else jobs):
        cols, rows, P32, Cdev = check_point_cloud(p, j)
        rc = check_coefficients(p, j, cols, rows, P32, Cdev)
        check_pairs(p, j, cols, rows, P32, Cdev, rc, st)
    share = st["unproven"] / max(st["pairs_filtered"], 1)
    print(f"{label}: pairs {st['pairs']}, filtered {st['pairs_filtered']}, max |q_ref-q*|/eps_ref {st['r1']:.4f}, "
          f"max |q_f-q*|/eps_f {st['r2']:.4f}, proven (own C, both rcp ends) {st['proven']}, wrong {st['wrong']}, "
          f"unproven share {100 * share:.3f} %")
    assert st["wrong"] == 0
    assert st["r1"] < 1.0 and st["r2"] < 1.0
    assert st["oracle_checked"] > 0 or st["pairs_filtered"] == 0
    st["share"] = share
    return st


# ---------------------------------------------------------------------------------------------------------------
# scenarios
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [SEQ, COMPOSED, TRANSLATE])
@pytest.mark.parametrize("shape", ["640x480", "1024x768"])
def test_workload_pass(mode, shape, monkeypatch):
    """The workload-shaped passes of test_filtered_projection_equals_exact_chain, every job and pair, and the
    share of filtered-candidate pairs the bound leaves unproven (kernel rule: largest C of each 8-point item)."""
    wl = workloads.Workload("probe", "4 videos x 4 tracks x 16 frames, 96 candidates", 4, 4, 16, 96) if shape == "640x480" \
        else workloads.Workload("probe", "2 videos x 2 tracks x 12 frames, 144 candidates, 1024x768", 2, 2, 12, 144, 1024, 768)
    inp = workloads.build_pass(wl, 300 + mode, DEV, mode=mode)
    p = run_filter_pass(inp.cfg, inp.pool, inp.batch, monkeypatch)
    st = check_pass(p, f"workload {shape} mode {mode}")
    assert st["pairs_filtered"] > 10 ** 7
    if UNPROVEN_CEILING[mode] is not None:
        assert st["share"] < UNPROVEN_CEILING[mode]


def _adversarial_specs(rng, n_masks, A=24):
    specs = []
    for j in range(10):
        mode = j % 3
        ax = rng.randn(A, 3)
        ax /= np.linalg.norm(ax, axis=1, keepdims=True)
        ang = rng.uniform(-np.pi, np.pi, A) * (1e-3 if j == 3 else 1.0)
        xf = np.zeros((A, 12), np.float32)
        xf[:, :9] = geometry._axis_angle_to_matrix(torch.from_numpy(ax * ang[:, None])).to(torch.float32).numpy().reshape(A, 9)
        xf[:, 9:] = (rng.randn(A, 3) * rng.choice([1e-3, 0.3, 5.0])).astype(np.float32)
        kind = j % 5
        normal = rng.randn(3)
        if kind == 0:
            normal[2] = 1e-3 * rng.randn()                         # grazing
        elif kind == 1:
            normal = np.array([0.0, 0.0, 1.0]) + 1e-4 * rng.randn(3)   # fronto-parallel
        normal = (normal / np.linalg.norm(normal)).astype(np.float32)
        offset = float(np.float32(rng.choice([0.02, 0.5, 2.0, 50.0])))
        pivot = (rng.randn(3) * rng.choice([0.1, 3.0, 100.0])).astype(np.float32)
        specs.append((int(rng.randint(n_masks)), mode, normal, offset, pivot, xf, [0]))
    return specs


@pytest.mark.parametrize("seed,focal", [(0, None), (1, 40.0), (2, 6000.0), (3, 517.97)])
def test_adversarial_geometry(seed, focal, monkeypatch):
    """The generator of test_filter_kernel_adversarial_geometry on new seeds: grazing and fronto-parallel planes,
    offsets 0.02 to 50, pivots up to 100 m away, full-circle and milliradian rotations, salt-and-pepper and ragged
    sources, focal lengths 40 / 518 / 6000."""
    rng = np.random.RandomState(7100 + seed)
    H, W = [(480, 640), (768, 1024), (120, 200), (480, 640)][seed]
    cfg = OptConfig.scaled(W, H) if focal is None else OptConfig(height=H, width=W, focal_length=focal)
    n = 5
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.zeros((n, H, W), np.float32)
    for i in range(n):
        cy, cx = rng.uniform(0.2, 0.8) * H, rng.uniform(0.2, 0.8) * W
        ry, rx = rng.uniform(0.1, 0.6) * H, rng.uniform(0.1, 0.6) * W
        masks[i] = (np.abs(yy - cy) < ry) & (np.abs(xx - cx) < rx)
    masks[1, ::2] = 0                                             # ragged rows
    masks[2] *= (rng.rand(H, W) < 0.5)                            # salt and pepper
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    batch = engine.build_batch(*zip(*_adversarial_specs(rng, n)), pool.source_points)
    p = run_filter_pass(cfg, pool, batch, monkeypatch)
    check_pass(p, f"adversarial seed {seed} ({W}x{H}, f {cfg.focal_length:.0f})")


@pytest.mark.parametrize("kind", ["skewed", "rotated", "grazing"])
def test_general_intrinsics(kind, monkeypatch):
    """Cameras whose K^-1 is not the pinhole pattern (k_unproject<false>): skew, non-square pixels, an off-centre
    principal point, a rotated camera and rays lying in the plane z = const."""
    from tests.test_gpu_envelope import _general_kinv, _rotations
    W, H = 640, 480
    cfg = OptConfig.scaled(W, H)
    kinv = _general_kinv(kind, cfg)
    rng = np.random.RandomState(len(kind) * 1000 + 17)
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.zeros((4, H, W), np.float32)
    masks[0, 2:H - 2, 2:W - 2] = 1
    for i in (1, 2):
        cy, cx = rng.uniform(0.2, 0.8) * H, rng.uniform(0.2, 0.8) * W
        masks[i] = ((yy - cy) / (rng.uniform(0.1, 0.4) * H)) ** 2 + ((xx - cx) / (rng.uniform(0.1, 0.4) * W)) ** 2 < 1
    masks[2] *= rng.rand(H, W) < 0.6
    masks[3, :H // 5] = 1                                            # the rows around the grazing rays
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    specs = []
    for j, (mode, src) in enumerate([(SEQ, 0), (COMPOSED, 1), (TRANSLATE, 2), (SEQ, 3), (COMPOSED, 2), (TRANSLATE, 3)]):
        A = 16
        xf = np.zeros((A, 12), np.float32)
        xf[:, :9] = _rotations(rng, A, 0.5) if mode != TRANSLATE else np.eye(3, dtype=np.float32).reshape(9)
        xf[:, 9:] = (rng.randn(A, 3) * 0.2).astype(np.float32)
        normal = np.array([0.0, 0.0, 1.0]) if j >= 3 else np.array([0.1, -0.2, 1.0]) + 0.05 * rng.randn(3)
        normal = (normal / np.linalg.norm(normal)).astype(np.float32)
        pivot = (rng.randn(3) * 0.3 + [0, 0, 2]).astype(np.float32)
        specs.append((src, mode, normal, 2.0, pivot, xf, [0]))
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    p = run_filter_pass(cfg, pool, batch, monkeypatch, kinv=kinv)
    check_pass(p, f"general K^-1 {kind}")


def _rot(axis, angle):
    a = np.asarray(axis, np.float64)
    return geometry._axis_angle_to_matrix(torch.from_numpy(a / np.linalg.norm(a) * angle)).numpy().reshape(3, 3)


def _xf(R, t=(0.0, 0.0, 0.0)):
    x = np.zeros(12, np.float32)
    x[:9] = np.asarray(R, np.float32).reshape(9)
    x[9:] = np.asarray(t, np.float32)
    return x


def test_edge_sources(monkeypatch):
    """A single source pixel; a box touching column W-1 at W = 1057 (the padding bits of the last word fall inside
    the word box); a box over the full frame; a non-binary fp32 source (its != 0 pixels are the points); and a
    COMPOSED job with one NaN translation, where every C_point of the job is +inf."""
    W, H = 1057, 96
    cfg = OptConfig.scaled(W, H)
    rng = np.random.RandomState(5)
    masks = np.zeros((4, H, W), np.float32)
    masks[0, 50, 700] = 1
    masks[1, 10:61, 1000:] = 1
    masks[2] = 1
    masks[3, 20:80, 100:400] = rng.choice([0.0, 0.3, 0.7, 1.0], size=(60, 300)).astype(np.float32)
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV), 0.5, with_nonzero=True)
    assert pool.bits_nz is not None                                   # the source map differs from the > 0.5 map
    rots = [_xf(_rot(rng.randn(3), a), rng.randn(3) * 0.1) for a in np.linspace(-1.2, 1.2, 12)]
    nan_t = np.stack(rots)
    nan_t[5, 10] = np.nan
    normal = (np.array([0.1, -0.2, 1.0]) / np.linalg.norm([0.1, -0.2, 1.0])).astype(np.float32)
    pivot = np.array([0.1, 0.0, 2.0], np.float32)
    trans = np.stack([_xf(np.eye(3), t) for t in rng.randn(8, 3) * 0.3])
    specs = []
    for src in range(4):
        for mode, xf in ((SEQ, np.stack(rots)), (COMPOSED, np.stack(rots)), (TRANSLATE, trans)):
            specs.append((src, mode, normal, 2.0, pivot, xf, [0]))
    specs.append((3, COMPOSED, normal, 2.0, pivot, nan_t, [0]))
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    p = run_filter_pass(cfg, pool, batch, monkeypatch)
    src = p["src"]
    assert src[0].sum() == 1 and src[1][:, W - 1].any() and src[2].all()
    assert src[3].sum() == int((masks[3] != 0).sum()) > int((masks[3] > 0.5).sum())
    check_pass(p, "edge sources")
    assert np.isposinf(job_slice(p, len(specs) - 1)[4, :int(p["count"][-1])]).all()


def test_exact_only_branches(monkeypatch):
    """One candidate for every branch of the exact-only rule — rho > 1.001, a NaN entry, an fp32 overflow of H,
    the identity, pure x and y translations of a fronto-parallel plane — and negatives (a 1e-3 rad rotation, a
    translation in x and y), each checked to hit its branch with a margin from the 0.02 threshold; then frames
    one pixel wide and one pixel high, where every candidate is exact-only."""
    W, H = 640, 480
    cfg = OptConfig.scaled(W, H)
    masks = np.zeros((1, H, W), np.float32)
    masks[0, 150:330, 200:460] = 1
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    R1 = _rot([0.3, 0.5, 0.8], 0.4)
    front = np.array([0.0, 0.0, 1.0], np.float32)
    tilted = (np.array([0.2, -0.3, 1.0]) / np.linalg.norm([0.2, -0.3, 1.0])).astype(np.float32)
    pivot = np.array([0.05, -0.02, 2.0], np.float32)
    nanR = R1.copy()
    nanR[1, 2] = np.nan
    cases = [  # (mode, normal, xf, expected reasons)
        (SEQ, tilted, _xf(1.01 * _rot([0.1, 0.2, 1.0], 0.3)), {"rho"}),
        (SEQ, tilted, _xf(nanR), {"rho", "hf", "ecand"}),
        (SEQ, tilted, _xf(np.eye(3)), {"fix_x", "fix_y"}),
        (SEQ, tilted, _xf(_rot([0.3, 0.5, 0.8], 1e-3)), set()),
        (SEQ, tilted, _xf(R1), set()),
        (COMPOSED, tilted, _xf(np.eye(3), (3e38, 3e38, 3e38)), {"hf", "ecand"}),   # 1e30 stays finite in fp32
        (TRANSLATE, front, _xf(np.eye(3), (0.3, 0.0, 0.0)), {"fix_y"}),
        (TRANSLATE, front, _xf(np.eye(3), (0.0, 0.3, 0.0)), {"fix_x"}),
        (TRANSLATE, front, _xf(np.eye(3), (0.3, 0.2, 0.0)), set()),
        (TRANSLATE, front, _xf(np.eye(3)), {"fix_x", "fix_y"}),
    ]
    specs = [(0, m, nrm, 2.0, pivot, xf[None], [0]) for m, nrm, xf, _ in cases]
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    p = run_filter_pass(cfg, pool, batch, monkeypatch)
    box = _word_box(p["src"][0])
    for j, (mode, nrm, xf, want) in enumerate(cases):
        rc = restate_candidates(p["cam"], batch.jobs[j], xf[None], box, job_hom(p, j)[:, :9].reshape(1, 3, 3))
        got = {k for k, v in rc["reasons"].items() if v[0]}
        assert got == want, (j, got, want)
        for k in ("x", "y"):                                          # far from the 0.02 threshold
            assert not 0.01 <= rc["fix"][k][0] <= 0.04, (j, k, rc["fix"][k][0])
        assert (job_hom(p, j)[0, 10] != 0) == bool(want), j
    check_pass(p, "exact-only branches")

    for W, H in ((1, 40), (40, 1)):
        cfg = OptConfig(height=H, width=W)
        m = np.ones((1, H, W), np.float32)
        pool = engine.pack_masks(torch.from_numpy(m).to(DEV))
        xf = np.stack([_xf(R1), _xf(_rot([0, 1, 0], 0.2))])
        specs = [(0, SEQ, tilted, 2.0, pivot, xf, [0]), (0, TRANSLATE, tilted, 2.0, pivot, xf, [0])]
        batch = engine.build_batch(*zip(*specs), pool.source_points)
        p = run_filter_pass(cfg, pool, batch, monkeypatch)
        assert (p["hom"][:, 10] == 1).all()
        check_pass(p, f"{W}x{H} frame")


def test_split_and_batched_unproject_agree(monkeypatch):
    """A job alone (its phase 2 split over 32 CTAs) and the same job inside a batch of 300 (one CTA per job): the
    same point-cloud slice, coefficients and homography rows, bit for bit."""
    W, H = 640, 480
    cfg = OptConfig.scaled(W, H)
    rng = np.random.RandomState(11)
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.zeros((3, H, W), np.float32)
    masks[0] = ((yy - 240) / 150.0) ** 2 + ((xx - 300) / 200.0) ** 2 < 1
    masks[1, 40:300:3, 50:600] = 1
    masks[2, 100:400, 100:500] = rng.rand(300, 400) < 0.4
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    normal = (np.array([0.1, -0.2, 1.0]) / np.linalg.norm([0.1, -0.2, 1.0])).astype(np.float32)
    pivot = np.array([0.1, 0.0, 2.0], np.float32)
    rots = np.stack([_xf(_rot(rng.randn(3), a), rng.randn(3) * 0.2) for a in np.linspace(-1.5, 1.5, 40)])
    trans = np.stack([_xf(np.eye(3), t) for t in rng.randn(20, 3) * 0.3])
    probes = [(0, SEQ, normal, 2.0, pivot, rots, [0]), (1, COMPOSED, normal, 1.5, pivot, rots, [0]),
              (2, TRANSLATE, normal, 2.5, pivot, trans, [0])]
    alone = []
    for spec in probes:
        b = engine.build_batch(*zip(spec), pool.source_points)
        p = run_filter_pass(cfg, pool, b, monkeypatch)
        check_pass(p, f"alone, mode {spec[1]}")
        alone.append((job_slice(p, 0)[:, :int(p["count"][0])].copy(), job_hom(p, 0).copy()))
    specs = [probes[i % 3] for i in range(300)]
    b = engine.build_batch(*zip(*specs), pool.source_points)
    p = run_filter_pass(cfg, pool, b, monkeypatch)
    for j in range(300):
        sl, hom = alone[j % 3]
        assert int(p["count"][j]) == sl.shape[1]
        assert np.array_equal(job_slice(p, j)[:, :sl.shape[1]].view(np.uint32), sl.view(np.uint32)), j
        assert np.array_equal(job_hom(p, j).view(np.uint32), hom.view(np.uint32)), j
    check_pass(p, "batch of 300", jobs=range(3))
