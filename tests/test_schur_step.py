"""The exact-Schur LM step on every reduced-system path, against an extended-precision reference.

A full LM solve is a weak detector of a slightly wrong reduced camera system S: the cost and the gradient
are right, so LM still reaches the same minimum.  These tests check the step itself,
(Js'Js + D^2) y = Js'r with step = -y (Jacobi-scaled tangent space, slots [6F | 3C] then [3P]), on a
catalogue of problems chosen to land on each dispatch of the exact mode: the rank-1 and block-6 band
Cholesky (one-sided, two-sided, smallest and widest window), the dense k_chol_blocked route, 256- and
512-wide fused tiles, the unfused Schur kernels, split pair units, the PCG fallback, and the inputs the
COLMAP front end produces (several cameras, extra constant poses / tvec components, constant cameras,
duplicate observations, holes, outliers under SoftL1 / Cauchy).

Reference: J and r from the oracle (pinned by tests/test_oracle_ba.py), normal equations assembled block by
block in long double, solved in float64 and refined with long-double residuals.  Each GPU step is checked by
its backward error against that system (independent of the conditioning), its forward error against the
refined solution (within c kappa eps), its distance to the oracle's step and its agreement with every other
kernel variant of the same case."""
import ctypes as C
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg
import scipy.sparse as sps

import oracle
from particlesfm_b200 import _abi, synthetic as syn

LD = np.longdouble
EPS = np.finfo(np.float64).eps

# ----------------------------------------------------------------------------- tolerances
# Measured on one B200 over the whole catalogue, every pass, radius and kernel variant; each bound is 10x or more
# above the worst figure (named in the comment).
TOL_BACKWARD = 1e-13          # Cholesky paths, reduced and full system: worst 5.9e-15 (the oracle: 1.1e-14, holes)
TOL_BACKWARD_PCG = 2e-8       # PCG with exact_r_tolerance = 1e-13 (principal point, PSFM_EXACT_PCG): worst 1.3e-9
                              # (wide_tiles), 2.2e-10 on the principal-point case.  Far above what a 1e-13 residual
                              # test implies: an open finding, bounded here so that it cannot grow unnoticed
C_FORWARD = 150.0             # forward error <= C_FORWARD kappa(S_c) eps: worst 13 (two_view, kappa 1.7)
TOL_ORACLE = 1e-10            # distance to the oracle's step, or 2 C_FORWARD kappa eps when larger: both sides are
                              # backward stable, so they differ by up to twice the forward error (worst 2.1e-8,
                              # tiny_window: tracks of 2 observations, kappa ~1e7)
TOL_VARIANTS = 1e-10          # Cholesky variants of one case, or 2 C_FORWARD kappa eps when larger (worst 7.6e-9)
TOL_ONE_ITER_COST = 1e-12     # one LM iteration, Cholesky paths: final cost, relative
TOL_ONE_ITER_PARAMS = 1e-10   # one LM iteration, Cholesky paths: parameters, relative
TOL_ONE_ITER_PCG = 1e-6       # one LM iteration through PCG: cost and parameters (worst 2.6e-8, wide_tiles)

RADII = (1e4, 1e1, 1e8)       # Ceres' initial radius, a heavily damped step, a near Gauss-Newton step
PASS_A, PASS_B, PASS_C = (False, False), (True, True), (True, False)


# ----------------------------------------------------------------------------- the catalogue

def _join(a, b):
    """Points and observations of `b` appended to `a` (same images and cameras)."""
    return _abi.BAProblem(a.qvec, a.tvec, np.concatenate([a.xyz, b.xyz]), a.cam_params,
                          np.concatenate([a.obs_image, b.obs_image]),
                          np.concatenate([a.obs_point, b.obs_point + a.num_points]),
                          np.concatenate([a.obs_xy, b.obs_xy]), a.image_camera,
                          a.pose_constant, a.tvec_constant_mask, a.camera_constant)


def _replace(p, **kw):
    f = dict(qvec=p.qvec, tvec=p.tvec, xyz=p.xyz, cam_params=p.cam_params, obs_image=p.obs_image,
             obs_point=p.obs_point, obs_xy=p.obs_xy, image_camera=p.image_camera, pose_constant=p.pose_constant,
             tvec_constant_mask=p.tvec_constant_mask, camera_constant=p.camera_constant)
    f.update(kw)
    return _abi.BAProblem(**f)


def _duplicates():
    p, _ = syn.make_ba_problem(30, 900, 10, seed=49, dynamic_fraction=0.3)
    rng = np.random.default_rng(49)
    dup = rng.choice(p.num_observations, 200, replace=False)
    return _replace(p, obs_image=np.concatenate([p.obs_image, p.obs_image[dup]]),
                    obs_point=np.concatenate([p.obs_point, p.obs_point[dup]]),
                    obs_xy=np.concatenate([p.obs_xy, p.obs_xy[dup] + rng.normal(0, 0.3, (200, 2))]))


def _holes():
    """Image 17 has no observation (inactive slots inside the band), 5 points with one observation,
    5 points with none."""
    p, _ = syn.make_ba_problem(40, 500, 6, seed=50)
    keep = p.obs_image != 17
    single = np.nonzero(keep)[0][:5]
    xyz = np.concatenate([p.xyz, p.xyz[p.obs_point[single]] + 0.01, np.full((5, 3), 123.0)])
    return _replace(p, xyz=xyz,
                    obs_image=np.concatenate([p.obs_image[keep], p.obs_image[single]]),
                    obs_point=np.concatenate([p.obs_point[keep], p.num_points + np.arange(5)]),
                    obs_xy=np.concatenate([p.obs_xy[keep], p.obs_xy[single] + 0.5]))


def _extra_constants():
    p, _ = syn.make_ba_problem(40, 500, 6, seed=51)
    pc, tm = p.pose_constant.copy(), p.tvec_constant_mask.copy()
    pc[20] = 1                  # a constant pose in the middle of the band
    tm[33] = 4                  # tvec z of image 33 constant
    return _replace(p, pose_constant=pc, tvec_constant_mask=tm)


def _two_cameras():
    """Images alternate between two SIMPLE_PINHOLE cameras, focal 900 and 1100."""
    p, _ = syn.make_ba_problem(40, 500, 6, seed=52)
    cams = (np.arange(40) % 2).astype(np.int32)
    K = np.array([[900.0, 512.0, 218.0], [1100.0, 512.0, 218.0]])
    xy = p.obs_xy.copy()
    odd = cams[p.obs_image] == 1
    xy[odd] = K[1, 1:] + (xy[odd] - K[0, 1:]) * (1100.0 / 900.0)
    return _replace(p, obs_xy=xy, cam_params=K, image_camera=cams, camera_constant=np.zeros(2, np.uint8))


def _outliers(seed):
    p, _ = syn.make_ba_problem(40, 500, 6, seed=seed)
    rng = np.random.default_rng(seed)
    bad = rng.choice(p.num_observations, p.num_observations // 20, replace=False)
    ang = rng.uniform(0, 2 * np.pi, bad.shape[0])
    xy = p.obs_xy.copy()
    xy[bad] += 30.0 * np.stack([np.cos(ang), np.sin(ang)], -1)
    return _replace(p, obs_xy=xy)


class Case:
    def __init__(self, name, make, route, passes=(PASS_A, PASS_B, PASS_C), loss=_abi.LOSS_SOFT_L1, pp=False,
                 tile=256, radii=RADII):
        self.name, self.make, self.route, self.passes, self.loss, self.pp, self.tile = name, make, route, passes, loss, pp, tile
        self.radii = radii


# route: what band_chol_plan (ba_band_chol.cuh) picks for nb = 6 F and the longest track span
CATALOGUE = [
    Case("two_view", lambda: syn.make_ba_problem(2, 300, 2, seed=40)[0], "rank1"),
    Case("tiny_window", lambda: syn.make_ba_problem(12, 400, 2, seed=41)[0], ("blk6-two", 3)),
    Case("one_sided", lambda: syn.make_ba_problem(12, 400, 6, seed=42)[0], ("blk6-one", 6)),
    Case("two_sided", lambda: syn.make_ba_problem(60, 600, 6, seed=43)[0], ("blk6-two", 6)),
    Case("widest_band", lambda: syn.make_ba_problem(100, 700, 25, seed=44)[0], ("blk6-two", 25)),
    Case("just_past", lambda: syn.make_ba_problem(100, 700, 26, seed=45)[0], "dense"),
    Case("dense_covisibility", lambda: syn.make_ba_problem(30, 600, 3, seed=46, track_len_range=(3, 30))[0], "dense"),
    Case("wide_tiles", lambda: _join(syn.make_ba_problem(320, 6, 300, seed=47)[0],
                                     syn.make_ba_problem(320, 500, 8, seed=48)[0]), "dense", tile=512),
    Case("duplicates", _duplicates, ("blk6-one", 10)),
    # no 1e8: a point with one observation has a rank-2 block, damped by diag / radius only; its float64 inverse
    # (oracle and kernels alike) is then off by ~radius eps, which puts the reduced system 1e-11 off
    Case("holes", _holes, ("blk6-two", 6), radii=RADII[:2]),
    Case("extra_constants", _extra_constants, ("blk6-two", 6)),
    Case("two_cameras", _two_cameras, ("blk6-two", 6)),
    Case("constant_camera", lambda: _replace(syn.make_ba_problem(40, 500, 6, seed=53)[0],
                                             camera_constant=np.ones(1, np.uint8)), ("blk6-two", 6), passes=(PASS_B,)),
    Case("outliers_softl1", lambda: _outliers(54), ("blk6-two", 6)),
    Case("outliers_cauchy", lambda: _outliers(55), ("blk6-two", 6), loss=_abi.LOSS_CAUCHY),
    Case("principal_point", lambda: syn.make_ba_problem(12, 400, 6, seed=56)[0], "pcg", passes=(PASS_B,), pp=True),
]
CASES = {c.name: c for c in CATALOGUE}
_PROBLEMS = {}


def _problem(name):
    if name not in _PROBLEMS:
        _PROBLEMS[name] = CASES[name].make()
    return _PROBLEMS[name]


def _opts(case, rot, focal):
    o = oracle.ba_global_options(refine_rotation=rot, refine_focal_length=focal)
    o.linear_solver = _abi.SOLVER_EXACT_SCHUR
    o.loss_function_type = case.loss
    o.refine_principal_point = int(case.pp)
    return o


def _gpu_supported(case, prob, rot, focal):
    """More than one camera with free intrinsics is refused (PSFM_ERR_UNSUPPORTED)."""
    free_cams = int(np.sum(prob.camera_constant == 0))
    return not ((focal or case.pp) and prob.num_cameras > 1 and free_cams > 0)


def _span(prob):
    lo = np.full(prob.num_points, np.iinfo(np.int32).max)
    hi = np.full(prob.num_points, -1)
    np.minimum.at(lo, prob.obs_point, prob.obs_image)
    np.maximum.at(hi, prob.obs_point, prob.obs_image)
    seen = hi >= 0
    return int((hi[seen] - lo[seen]).max())


def band_route(prob):
    """band_chol_plan(6 F, 6 span + 5, span) of ba_band_chol.cuh, restated: ("blk6-one" | "blk6-two", Wb),
    "rank1" (scalar register window) or "dense" (no band kernel: dense S + k_chol_blocked)."""
    F, span = prob.num_images, _span(prob)
    nb = 6 * F
    bw = min(6 * span + 5, nb - 1)
    Wb = max(3, min(span + 1, F))
    if F >= 3 and Wb <= 25 and 6 * Wb > bw:
        return ("blk6-two" if F >= 4 * Wb else "blk6-one", Wb)
    W = ((bw + 1 + 7) // 8) * 8
    return "rank1" if W <= 152 else "dense"


def tile_width(prob):
    return 256 if np.bincount(prob.obs_point).max() <= 256 else 512


# ----------------------------------------------------------------------------- extended-precision reference

class Linearization:
    """Jacobi-scaled blocks of the normal equations at the problem's state, in long double.
    Camera slots [6F | 3C] (pose: rotation 3, translation 3; camera: f, cx, cy), points [P, 3]."""

    def __init__(self, prob, o):
        jc, jp, jk = oracle.ba_jacobians(prob, o)
        _, r, _, _ = oracle.ba_evaluate(prob, o)
        F, P, Cn = prob.num_images, prob.num_points, prob.num_cameras
        NS = 6 * F + 3 * Cn
        self.NS, self.P = NS, P
        img, pt = prob.obs_image.astype(np.int64), prob.obs_point.astype(np.int64)
        cs = np.concatenate([6 * img[:, None] + np.arange(6), 6 * F + 3 * prob.image_camera[img][:, None] + np.arange(3)], 1)
        Jc = np.concatenate([jc, jk], 2).astype(LD)                  # [M, 2, 9]
        Jp = jp.astype(LD)                                           # [M, 2, 3]
        r = r.astype(LD)
        colc = np.zeros(NS, LD); np.add.at(colc, cs, (Jc ** 2).sum(1))
        colp = np.zeros((P, 3), LD); np.add.at(colp, pt, (Jp ** 2).sum(1))
        self.scale_c, self.scale_p = 1 / (1 + np.sqrt(colc)), 1 / (1 + np.sqrt(colp))
        Jc = Jc * self.scale_c[cs][:, None, :]
        Jp = Jp * self.scale_p[pt][:, None, :]
        self.act_c = colc > 0
        self.act_p = np.bincount(pt, minlength=P) > 0
        self.cs, self.pt = cs, pt
        self.Acc = np.zeros((NS, NS), LD)
        np.add.at(self.Acc, (cs[:, :, None], cs[:, None, :]), np.einsum("mki,mkj->mij", Jc, Jc))
        self.Bo = np.einsum("mki,mkj->mij", Jc, Jp)                  # per observation: camera slots x point
        self.App = np.zeros((P, 3, 3), LD)
        np.add.at(self.App, pt, np.einsum("mki,mkj->mij", Jp, Jp))
        self.bc = np.zeros(NS, LD); np.add.at(self.bc, cs, np.einsum("mki,mk->mi", Jc, r))
        self.bp = np.zeros((P, 3), LD); np.add.at(self.bp, pt, np.einsum("mki,mk->mi", Jp, r))
        rows = np.broadcast_to(cs[:, :, None], self.Bo.shape).ravel()
        cols = np.broadcast_to((3 * pt)[:, None, None] + np.arange(3), self.Bo.shape).ravel()
        self.B = sps.csr_matrix((self.Bo.ravel(), (rows, cols)), shape=(NS, 3 * P))
        self.diag_c = np.clip(np.diagonal(self.Acc), 1e-6, 1e32) * self.act_c
        self.diag_p = np.clip(np.einsum("pii->pi", self.App), 1e-6, 1e32)


def _inv3(A):
    """Inverse of [P, 3, 3] blocks through the adjugate (long double: np.linalg.inv stops at float64)."""
    a, b, c = A[:, 0, 0], A[:, 0, 1], A[:, 0, 2]
    d, e, f = A[:, 1, 0], A[:, 1, 1], A[:, 1, 2]
    g, h, i = A[:, 2, 0], A[:, 2, 1], A[:, 2, 2]
    adj = np.stack([np.stack([e * i - f * h, c * h - b * i, b * f - c * e], -1),
                    np.stack([f * g - d * i, a * i - c * g, c * d - a * f], -1),
                    np.stack([d * h - e * g, b * g - a * h, a * e - b * d], -1)], 1)
    det = a * adj[:, 0, 0] + b * adj[:, 1, 0] + c * adj[:, 2, 0]
    return adj / det[:, None, None]


class Reference:
    """The damped system at one radius: full system A = [[Acc, B], [B', App]] + D^2, its reduced camera system
    S_c = Acc - B App^-1 B', b_c = bc - B App^-1 bp, and the refined solution x = y (the step is -y)."""

    def __init__(self, lin, radius):
        self.lin = lin
        self.Acc = lin.Acc + np.diag(lin.diag_c / radius)
        self.App = lin.App + np.einsum("pi,ij->pij", lin.diag_p / radius, np.eye(3))
        self.Hinv = _inv3(self.App) * lin.act_p[:, None, None]       # points without observations: step 0
        idx = 3 * np.arange(lin.P)[:, None, None]
        H = sps.csr_matrix((self.Hinv.ravel(), ((idx + np.arange(3)[:, None]).repeat(3, 2).ravel(),
                                                (idx + np.arange(3)[None, :]).repeat(3, 1).ravel())),
                           shape=(3 * lin.P, 3 * lin.P))
        self.Sc = self.Acc - (lin.B @ H @ lin.B.T).toarray()
        self.ia = np.nonzero(lin.act_c)[0]
        self.bcr = lin.bc - lin.B @ self._hp(lin.bp).ravel()
        self.Sa = self.Sc[np.ix_(self.ia, self.ia)]
        ev = np.linalg.eigvalsh(self.Sa.astype(np.float64))
        self.kappa = float(ev[-1] / ev[0])          # 2-norm condition number of the (SPD) reduced system
        self._chol = scipy.linalg.cho_factor(self.Sa.astype(np.float64))
        absA_c = np.abs(self.Acc).sum(1) + np.asarray(abs(lin.B).sum(1)).ravel()
        absA_p = np.asarray(abs(lin.B).sum(0)).ravel().reshape(-1, 3) + np.abs(self.App).sum(2)
        self.normA = max(absA_c[self.ia].max(), absA_p[lin.act_p].max() if lin.act_p.any() else 0)
        self.normS = np.abs(self.Sa).sum(1).max()
        # solve in float64 (through the reduced system), refine with long-double residuals of the full system
        xc, xp = np.zeros(lin.NS, LD), np.zeros((lin.P, 3), LD)
        for _ in range(4):
            rc, rp = self.residual(xc, xp)
            dc, dp = self._inner(rc, rp)
            xc, xp = xc + dc, xp + dp
        self.xc, self.xp = xc, xp

    def _hp(self, v):
        return np.einsum("pij,pj->pi", self.Hinv, v)

    def _inner(self, rc, rp):
        rhs = rc - self.lin.B @ self._hp(rp).ravel()
        dc = np.zeros(self.lin.NS, LD)
        dc[self.ia] = scipy.linalg.cho_solve(self._chol, rhs[self.ia].astype(np.float64))
        dp = self._hp(rp - (self.lin.B.T @ dc).reshape(-1, 3))
        return dc, dp

    def residual(self, xc, xp):
        """b - A x of the full system, long double (inactive camera slots and unobserved points: 0)."""
        lin = self.lin
        rc = lin.bc - self.Acc @ xc - lin.B @ xp.ravel()
        rp = lin.bp - (lin.B.T @ xc).reshape(-1, 3) - np.einsum("pij,pj->pi", self.App, xp)
        return np.where(lin.act_c, rc, 0), rp * lin.act_p[:, None]

    def reduced_backward(self, xc):
        x = xc.astype(LD)[self.ia]
        b = self.bcr[self.ia]
        return float(np.abs(self.Sa @ x - b).max() / (self.normS * np.abs(x).max() + np.abs(b).max()))

    def full_backward(self, xc, xp, slack=0.0):
        """Backward error of the full system; `slack` absolute on the point step (the GPU's (Xc - X) / scale)."""
        xc, xp = xc.astype(LD), xp.astype(LD)
        rc, rp = self.residual(xc, xp)
        num = max(np.abs(rc).max(), np.abs(rp).max()) - self.normA * slack
        den = self.normA * max(np.abs(xc).max(), np.abs(xp).max()) + max(np.abs(self.lin.bc).max(), np.abs(self.lin.bp).max())
        return float(max(num, 0.0) / den)


_LINS = {}


def linearization(name, rot, focal):
    key = (name, rot, focal)
    if key not in _LINS:
        _LINS[key] = Linearization(_problem(name), _opts(CASES[name], rot, focal))
    return _LINS[key]


@pytest.fixture(scope="module")
def references():
    cache = {}

    def get(name, rot, focal, radius):
        key = (name, rot, focal, radius)
        if key not in cache:
            cache[key] = Reference(linearization(name, rot, focal), radius)
        return cache[key]
    return get


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-300))


def _point_slack(prob, lin):
    """|(Xc - X) / scale - y| for Xc = X + scale y rounded in float64."""
    return float((4 * EPS * np.abs(prob.xyz) / lin.scale_p.astype(np.float64))[lin.act_p].max()) if lin.act_p.any() else 0.0


def _all_keys():
    for c in CATALOGUE:
        for rot, focal in c.passes:
            for radius in c.radii:
                yield c.name, rot, focal, radius


# ----------------------------------------------------------------------------- CPU: reference vs oracle, teeth

def test_catalogue_routes():
    """Every case sits on the dispatch it is named for (band_chol_plan restated, tile width)."""
    for c in CATALOGUE:
        prob = _problem(c.name)
        if c.route != "pcg":
            assert band_route(prob) == c.route, (c.name, band_route(prob))
        assert tile_width(prob) == c.tile, c.name
        assert 3 * prob.num_points + 6 * prob.num_images + 3 * prob.num_cameras <= 3500, c.name


@pytest.mark.parametrize("name", [c.name for c in CATALOGUE])
def test_reference_matches_oracle_step(references, name):
    """The oracle's exact step (SPARSE_SCHUR restatement for one camera, dense Schur otherwise) against the
    refined long-double solution: backward error, and forward error within c kappa eps."""
    case = CASES[name]
    prob = _problem(name)
    for rot, focal in case.passes:                  # two_cameras pass B: the oracle refines two cameras' focals
        o = _opts(case, rot, focal)
        for radius in case.radii:
            ref = references(name, rot, focal, radius)
            sc, sp, _ = oracle.ba_linear_step(prob, o, radius, _abi.SOLVER_EXACT_SCHUR)
            xc, xp = -sc, -sp
            tag = (name, rot, focal, radius, ref.kappa)
            assert np.all(xc[~ref.lin.act_c] == 0), tag
            assert ref.reduced_backward(xc) <= TOL_BACKWARD, (tag, ref.reduced_backward(xc))
            assert ref.full_backward(xc, xp) <= TOL_BACKWARD, (tag, ref.full_backward(xc, xp))
            fwd = C_FORWARD * ref.kappa * EPS
            assert _rel(xc, ref.xc) <= fwd, (tag, _rel(xc, ref.xc) / (ref.kappa * EPS))
            # the reference itself: refined to far below what is asserted of the kernels
            rc, rp = ref.residual(ref.xc, ref.xp)
            assert max(np.abs(rc).max(), np.abs(rp).max()) <= 1e-3 * TOL_BACKWARD * ref.normA * np.abs(ref.xc).max()


def _teeth_system(ref, name, prob):
    """S_c with one contribution dropped: the image-pair block at the largest band offset between two images
    with free slots, or — duplicates, or no such pair — the diagonal (a, b) term of one duplicated observation /
    of one observation."""
    lin = ref.lin
    S = ref.Sc.copy()
    act_img = lin.act_c[:6 * prob.num_images].reshape(-1, 6).any(1)
    best = None
    if name != "duplicates":
        for d in range(_span(prob), 0, -1):
            for i in np.nonzero(act_img[:-d] & act_img[d:])[0]:
                blk = S[6 * i:6 * i + 6, 6 * (i + d):6 * (i + d) + 6]
                if np.abs(blk).max() > 0:
                    best = (i, i + d)
                    break
            if best:
                break
    if best:
        i, j = best
        S[6 * i:6 * i + 6, 6 * j:6 * j + 6] = 0
        S[6 * j:6 * j + 6, 6 * i:6 * i + 6] = 0
        return S
    key = prob.obs_point.astype(np.int64) * prob.num_images + prob.obs_image
    order = np.argsort(key, kind="stable")
    same = np.nonzero(key[order][1:] == key[order][:-1])[0]
    a, b = (order[same[0]], order[same[0] + 1]) if len(same) else (int(np.nonzero(lin.act_c[lin.cs].any(1))[0][0]),) * 2
    T = lin.Bo[a] @ ref.Hinv[lin.pt[a]] @ lin.Bo[b].T
    S[np.ix_(lin.cs[a], lin.cs[b])] += T                     # S = Acc - sum Z_a B_b': dropping the term adds it back
    return S


@pytest.mark.parametrize("name", [c.name for c in CATALOGUE])
def test_teeth_a_dropped_block_is_detected(references, name):
    """Without mutating a kernel: a reduced system missing one image-pair block (or one duplicate observation's
    term) gives a step whose backward error against the true system is >= 100x the tolerance."""
    case = CASES[name]
    prob = _problem(name)
    for rot, focal in case.passes:
        for radius in case.radii:
            ref = references(name, rot, focal, radius)
            Sb = _teeth_system(ref, name, prob)[np.ix_(ref.ia, ref.ia)].astype(np.float64)
            xc = np.zeros(ref.lin.NS)
            xc[ref.ia] = np.linalg.solve(Sb, ref.bcr[ref.ia].astype(np.float64))
            tol = TOL_BACKWARD_PCG if case.pp else TOL_BACKWARD
            assert ref.reduced_backward(xc) >= 100 * tol, (name, rot, focal, radius, ref.reduced_backward(xc))


# ----------------------------------------------------------------------------- GPU

# read per solver or per call: one fresh ResidentSolver per variant and case
IN_PROCESS = {
    "default": {}, "tile512": {"PSFM_TILE512": "1"}, "no_pipe": {"PSFM_NO_PIPE": "1"},
    "no_pipe_schur": {"PSFM_NO_PIPE_SCHUR": "1"}, "schur_unfused": {"PSFM_SCHUR_UNFUSED": "1"},
    "old_chol": {"PSFM_OLD_CHOL": "1"}, "task_chunk1": {"PSFM_TASK_CHUNK": "1"}, "task_chunk7": {"PSFM_TASK_CHUNK": "7"},
    "exact_pcg": {"PSFM_EXACT_PCG": "1"},
}
# read once per process: a child process per switch
CHILD = {
    "chol_one_sided": {"PSFM_CHOL_ONE_SIDED": "1"}, "chol_rank1": {"PSFM_CHOL_RANK1": "1"},
    "no_pipe_back": {"PSFM_NO_PIPE_BACK": "1"}, "fused_cost": {"PSFM_FUSED_COST": "1"},
}
VARIANTS = list(IN_PROCESS) + list(CHILD)
PCG_VARIANTS = ("exact_pcg",)


def _one_iter_opts(case, rot, focal):
    o = _opts(case, rot, focal)
    o.max_num_iterations = 1
    o.function_tolerance = o.gradient_tolerance = o.parameter_tolerance = 0.0
    return o


def gpu_results():
    """Every GPU result of the catalogue under the current environment:
    steps[(case, rot, focal, radius)] = (rc, step_cam, step_pts), runs[(case, rot, focal)] = (rc, summary dict,
    qvec, tvec, xyz, cam_params)."""
    from particlesfm_b200 import _lib, ba
    L = _lib.lib()
    steps, runs = {}, {}
    for c in CATALOGUE:
        prob = _problem(c.name)
        S = ba.ResidentSolver(prob.copy())
        try:
            for rot, focal in c.passes:
                o = _opts(c, rot, focal)
                for radius in c.radii:
                    sc = np.zeros(6 * prob.num_images + 3 * prob.num_cameras)
                    sp = np.zeros((prob.num_points, 3))
                    it = C.c_int32()
                    rc = L.psfm_ba_linear_step(S._h, C.byref(o), radius, _lib.dptr(sc), _lib.dptr(sp), C.byref(it))
                    steps[(c.name, rot, focal, radius)] = (rc, sc, sp)
            for rot, focal in {PASS_A: [PASS_A, PASS_B]}.get(c.passes[0], list(c.passes)):
                S.set_state(prob.qvec, prob.tvec, prob.xyz, prob.cam_params)
                s = _abi.BASummary()
                rc = L.psfm_ba_run(S._h, C.byref(_one_iter_opts(c, rot, focal)), C.byref(s))
                p = S.get_state()
                runs[(c.name, rot, focal)] = (rc, s.as_dict(), p.qvec.copy(), p.tvec.copy(), p.xyz.copy(), p.cam_params.copy())
        finally:
            S.close()
    return steps, runs


def _child_results(env, path):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import pickle, sys; sys.path[:0] = [%r, %r]; import test_schur_step as t;"
            "pickle.dump(t.gpu_results(), open(sys.argv[1], 'wb'))") % (root, os.path.join(root, "tests"))
    subprocess.run([sys.executable, "-c", code, path], check=True, env={**os.environ, **env}, cwd=root)
    with open(path, "rb") as f:
        return pickle.load(f)


@pytest.fixture(scope="module")
def gpu_variant(tmp_path_factory):
    cache = {}

    def get(variant):
        if variant not in cache:
            if variant in CHILD:
                cache[variant] = _child_results(CHILD[variant], str(tmp_path_factory.mktemp("schur") / f"{variant}.pkl"))
            else:
                saved = {k: os.environ.get(k) for k in IN_PROCESS[variant]}
                os.environ.update(IN_PROCESS[variant])
                try:
                    cache[variant] = gpu_results()
                finally:
                    for k, v in saved.items():
                        if v is None:
                            os.environ.pop(k)
                        else:
                            os.environ[k] = v
        return cache[variant]
    return get


MEASURED = {}


def _record(what, key, value):
    k = (what, key)
    MEASURED[k] = max(MEASURED.get(k, 0.0), value)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if MEASURED and os.environ.get("PSFM_SCHUR_REPORT"):
        for (what, key), v in sorted(MEASURED.items()):
            print(f"[schur-step] {what:16s} {key:40s} {v:.3e}")


@pytest.mark.gpu
def test_gpu_paths_and_unsupported(gpu, gpu_variant):
    """The default build lands on the named path: fused tiles, explicit solves (or PCG for the principal point);
    free intrinsics of two cameras are refused."""
    steps, runs = gpu_variant("default")
    for c in CATALOGUE:
        prob = _problem(c.name)
        for (name, rot, focal), (rc, s, *_) in runs.items():
            if name != c.name:
                continue
            if not _gpu_supported(c, prob, rot, focal):
                assert rc == _abi.PSFM_ERR_UNSUPPORTED, (name, rot, focal, rc)
                continue
            assert rc == 0 and s["num_iterations"] == 1, (name, rot, focal, rc, s)
            assert s["linear_solver_used"] == _abi.SOLVER_EXACT_SCHUR, (name, s)
            if c.route == "pcg":        # no reduced system is formed
                assert s["num_explicit_solves"] == 0 and s["num_schur_products"] > 0, (name, s)
            else:
                assert s["num_explicit_solves"] == 1 and s["num_pair_entries"] > 0 and s["explicit_fused"] == 1, (name, s)
        for (name, rot, focal, radius), (rc, _, _) in steps.items():
            if name == c.name and not _gpu_supported(c, prob, rot, focal):
                assert rc == _abi.PSFM_ERR_UNSUPPORTED, (name, rot, focal, radius, rc)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_gpu_step_matches_reference(gpu, references, gpu_variant, variant):
    """Per (case, pass, radius): backward error of the reduced and of the full system, forward error within
    c kappa eps of the refined reference, distance to the oracle's step."""
    steps, _ = gpu_variant(variant)
    bad = []
    for name, rot, focal, radius in _all_keys():
        case, prob = CASES[name], _problem(name)
        if not _gpu_supported(case, prob, rot, focal):
            continue
        rc, sc, sp = steps[(name, rot, focal, radius)]
        ref = references(name, rot, focal, radius)
        tag = f"{name} rot={rot:d} focal={focal:d} r={radius:g}"
        if rc != 0:
            bad.append((tag, "rc", rc))
            continue
        pcg = case.pp or variant in PCG_VARIANTS
        slack = _point_slack(prob, ref.lin)
        xc, xp = -sc, -sp
        be_r, be_f = ref.reduced_backward(xc), ref.full_backward(xc, xp, slack)
        fe = _rel(xc, ref.xc) / (ref.kappa * EPS)
        fe_p = max(np.abs(xp - ref.xp.astype(np.float64)).max() - slack, 0) / (np.abs(ref.xp).max() * ref.kappa * EPS)
        oc, op, _ = oracle.ba_linear_step(prob, _opts(case, rot, focal), radius, _abi.SOLVER_EXACT_SCHUR)
        d_or = max(_rel(sc, oc), max(np.abs(sp - op).max() - slack, 0) / np.abs(op).max())
        kind = "pcg" if pcg else "chol"
        _record(f"backward/{kind}", f"{name}/{variant}", max(be_r, be_f))
        _record(f"fwd/(k eps)/{kind}", f"{name}/{variant}", max(fe, fe_p))
        _record(f"oracle/{kind}", f"{name}/{variant}", d_or)
        tb = TOL_BACKWARD_PCG if pcg else TOL_BACKWARD
        if not np.all(sc[~ref.lin.act_c] == 0):
            bad.append((tag, "inactive slot moved"))
        if be_r > tb or be_f > tb:
            bad.append((tag, "backward", be_r, be_f))
        if not pcg and (fe > C_FORWARD or fe_p > C_FORWARD):
            bad.append((tag, "forward / (kappa eps)", fe, fe_p, ref.kappa))
        if not pcg and d_or > max(TOL_ORACLE, 2 * C_FORWARD * ref.kappa * EPS):
            bad.append((tag, "oracle", d_or))
    assert not bad, bad


@pytest.mark.gpu
def test_gpu_variants_agree(gpu, references, gpu_variant):
    """Every Cholesky variant of a case computes the same step."""
    base, _ = gpu_variant("default")
    bad = []
    for variant in VARIANTS[1:]:
        steps, _ = gpu_variant(variant)
        for key, (rc, sc, sp) in base.items():
            rc2, sc2, sp2 = steps[key]
            if rc != rc2:
                bad.append((key, variant, "rc", rc, rc2))
                continue
            if rc != 0:
                continue
            d = max(_rel(sc2, sc), _rel(sp2, sp))
            _record("variants", f"{key[0]}/{variant}", d)
            if CASES[key[0]].pp or variant in PCG_VARIANTS:
                continue                # a PCG step is only as close as its residual test: checked by its backward error
            if d > max(TOL_VARIANTS, 2 * C_FORWARD * references(*key).kappa * EPS):
                bad.append((key, variant, d))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_gpu_one_iteration_matches_oracle(gpu, gpu_variant, variant):
    """One LM iteration on the GPU and in the oracle: the candidate path linear_step skips (k_apply_cams, the
    back-substitution, k_cost / the fused cost, the model-cost change that feeds rho)."""
    _, runs = gpu_variant(variant)
    bad = []
    for (name, rot, focal), (rc, s, q, t, X, K) in runs.items():
        case, prob = CASES[name], _problem(name)
        if not _gpu_supported(case, prob, rot, focal):
            continue
        p0 = prob.copy()
        s0 = oracle.ba_solve(p0, _one_iter_opts(case, rot, focal))
        assert s0.num_iterations == 1
        if rc != 0 or s["num_successful_steps"] != s0.num_successful_steps:
            bad.append((name, rot, focal, rc, s["num_successful_steps"], s0.num_successful_steps))
            continue
        dc = abs(s["final_cost"] - s0.final_cost) / s0.final_cost
        dp = max(_rel(q, p0.qvec), _rel(t, p0.tvec), _rel(X, p0.xyz), _rel(K, p0.cam_params))
        _record("1-iter cost", f"{name}/{variant}", dc)
        _record("1-iter params", f"{name}/{variant}", dp)
        pcg = case.pp or variant in PCG_VARIANTS
        if dc > (TOL_ONE_ITER_PCG if pcg else TOL_ONE_ITER_COST) or dp > (TOL_ONE_ITER_PCG if pcg else TOL_ONE_ITER_PARAMS):
            bad.append((name, rot, focal, dc, dp))
    assert not bad, bad


@pytest.mark.gpu
def test_fused_cost_on_wide_tiles(gpu, tmp_path):
    """Regression: with PSFM_FUSED_COST, 512-wide tiles and a 320-image pose table asked for a dynamic shared memory
    size inside the 227 KB limit but not inside it once the kernel's static part was added; the failed
    cudaFuncSetAttribute surfaced as a CUDA error of the step (and of the next call)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]; import test_schur_step as t; from particlesfm_b200 import ba;"
            "p = t._problem('wide_tiles'); S = ba.ResidentSolver(p.copy()); o = t._opts(t.CASES['wide_tiles'], True, True);"
            "sc, sp, it = S.linear_step(o, 1e4); s = S.run(t._one_iter_opts(t.CASES['wide_tiles'], True, True));"
            "np.save(sys.argv[1], sc); assert s.num_iterations == 1") % (root, os.path.join(root, "tests"))
    path = str(tmp_path / "sc.npy")
    subprocess.run([sys.executable, "-c", code, path], check=True, env={**os.environ, "PSFM_FUSED_COST": "1"}, cwd=root)
    assert np.isfinite(np.load(path)).all()
