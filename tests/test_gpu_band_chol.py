"""The single-CTA register-window band(+arrow) Cholesky of the exact-Schur mode
(csrc/ba_band_chol.cuh) against numpy on random SPD systems, through the C ABI."""
import ctypes as C

import numpy as np
import pytest

from particlesfm_b200 import _lib

pytestmark = pytest.mark.gpu


def _system(nb, bw, seed, arrow=True):
    rng = np.random.default_rng(seed)
    n = nb + 3
    B = rng.standard_normal((n, n))
    A = B @ B.T
    i, j = np.indices((n, n))
    A[(np.abs(i - j) > bw) & (i < nb) & (j < nb)] = 0.0
    if not arrow:                       # inactive intrinsics: identity rows, as k_band_assemble writes them
        A[nb:, :] = 0.0
        A[:, nb:] = 0.0
    A += np.eye(n) * (np.abs(A).sum(axis=1).max() + 1.0)
    b = rng.standard_normal(n)
    if not arrow:
        A[nb:, nb:] = np.eye(3)
        b[nb:] = 0.0
    return A, b


def _solve(A, b, nb, bw):
    x = np.zeros_like(b)
    rc = _lib.lib().psfm_ba_band_solve(_lib.dptr(np.ascontiguousarray(A)), _lib.dptr(b), nb, bw, _lib.dptr(x))
    return rc, x


# (nb, bw): tiny window, window wider than the matrix, nb not a multiple of 4, the bench shape
# (6 * 200 images, span 11/12), the 1024-thread instantiation, the widest supported window
CASES = [(30, 9), (18, 17), (18, 40), (90, 59), (1200, 71), (1200, 77), (600, 127), (3000, 71), (700, 150), (100, 31), (1203, 95),
         (64, 6), (41, 14), (500, 38),
         # block-6 kernel (nb and bw + 1 multiples of 6): window = matrix, one-sided, two-sided, the 512-thread
         # instantiation, the widest window (25 blocks), a window of 3 blocks, identity padding past the matrix
         (36, 17), (36, 35), (900, 35), (1200, 95), (1200, 149), (150, 149), (2400, 23), (78, 17), (1200, 83)]


@pytest.mark.parametrize("nb,bw", CASES)
def test_band_solve_matches_numpy(gpu, nb, bw):
    A, b = _system(nb, bw, seed=nb + bw)
    rc, x = _solve(A, b, nb, bw)
    assert rc == 0, _lib.lib().psfm_last_error()
    ref = np.linalg.solve(A, b)
    assert np.abs(x - ref).max() <= 1e-11 * np.abs(ref).max()


def test_band_solve_inactive_arrow_and_failure(gpu):
    A, b = _system(120, 35, seed=1, arrow=False)
    rc, x = _solve(A, b, 120, 35)
    assert rc == 0
    ref = np.linalg.solve(A, b)
    assert np.abs(x - ref).max() <= 1e-11 * np.abs(ref).max()
    assert np.array_equal(x[120:], np.zeros(3))
    A[57, 57] = -1.0                    # not positive definite -> reported, no garbage accepted
    rc, _ = _solve(A, b, 120, 35)
    assert rc == -1
    rc, _ = _solve(A, b, 120, 400)      # clamped to nb - 1 = 119 <= window limit: still solvable shape
    assert rc == -1
    A2, b2 = _system(400, 300, seed=2)                # window would be 304 > 152
    rc, _ = _solve(A2, b2, 400, 300)
    assert rc == -4                     # PSFM_ERR_UNSUPPORTED: wider than the register window


@pytest.mark.parametrize("bad", [57, 199, 200, 215, 330, 399])
def test_two_sided_form_reports_a_bad_pivot_wherever_it_is(gpu, bad):
    """nb = 400, bw = 35: window 40, two CTAs (top-down 184 pivots, bottom-up 176, 40 in the middle).  A negative
    diagonal on either side or in the middle must come back as an error, never as a hang or a silent solve."""
    A, b = _system(400, 35, seed=3)
    rc, x = _solve(A, b, 400, 35)
    assert rc == 0
    ref = np.linalg.solve(A, b)
    assert np.abs(x - ref).max() <= 1e-11 * np.abs(ref).max()
    A[bad, bad] = -1.0
    rc, _ = _solve(A, b, 400, 35)
    assert rc == -1


def _conditioned_system(nb, bw, kappa, seed):
    """A = L D L' with L unit lower-triangular, banded in the first nb rows (3 dense arrow rows below) and D
    log-spaced over [1/kappa, 1] in shuffled order: conditioned like a damped reduced camera system, not
    diagonally dominant."""
    rng = np.random.default_rng(seed)
    n = nb + 3
    L = np.tril(rng.standard_normal((n, n)), -1) * (0.5 / np.sqrt(bw + 1))
    i, j = np.indices((n, n))
    L[(i - j > bw) & (i < nb)] = 0.0
    L += np.eye(n)
    d = rng.permutation(np.logspace(-np.log10(kappa), 0, n))
    return (L * d) @ L.T, rng.standard_normal(n)


def _refined_solution(A, b):
    """np.linalg.solve refined with long-double residuals: accurate to ~kappa 1e-19."""
    Al, bl = A.astype(np.longdouble), b.astype(np.longdouble)
    x = np.linalg.solve(A, b).astype(np.longdouble)
    for _ in range(3):
        x += np.linalg.solve(A, (bl - Al @ x).astype(np.float64))
    return x


def _check_band_solution(A, b, x):
    """Backward error <= 8 n eps; forward error vs the refined solution <= 4 kappa eps."""
    n, eps = A.shape[0], np.finfo(np.float64).eps
    Al, xl = A.astype(np.longdouble), x.astype(np.longdouble)
    be = float(np.abs(Al @ xl - b).max() / (np.abs(A).sum(1).max() * np.abs(x).max() + np.abs(b).max()))
    ev = np.linalg.eigvalsh(A)
    kappa = ev[-1] / ev[0]
    ref = _refined_solution(A, b)
    fe = float(np.abs(xl - ref).max() / np.abs(ref).max())
    assert be <= 8 * n * eps, (be, n)
    assert fe <= 4 * kappa * eps, (fe, kappa, fe / (kappa * eps))
    return be, fe, kappa


# block-6 two-sided, block-6 widest window (25 blocks: (143 + 5) // 6 + 1), block-6 minimum window (3 blocks), rank-1 two-sided
COND_SHAPES = [(600, 35), (1200, 143), (36, 17), (1203, 95)]


@pytest.mark.parametrize("kappa", [1e4, 1e8, 1e12])
@pytest.mark.parametrize("nb,bw", COND_SHAPES)
def test_band_solve_conditioned(gpu, nb, bw, kappa):
    A, b = _conditioned_system(nb, bw, kappa, seed=nb + bw)
    rc, x = _solve(A, b, nb, bw)
    assert rc == 0, _lib.lib().psfm_last_error()
    _check_band_solution(A, b, x)


def test_band_solve_conditioned_one_sided(gpu, tmp_path):
    """The block-6 one-sided form (PSFM_CHOL_ONE_SIDED, read once per process) on the conditioned two-sided shape."""
    import os
    import subprocess
    import sys
    code = ("import numpy as np, sys; sys.path[:0] = [%r, %r]; from test_gpu_band_chol import _conditioned_system, _solve;"
            "A, b = _conditioned_system(600, 35, float(sys.argv[2]), seed=635); rc, x = _solve(A, b, 600, 35);"
            "assert rc == 0; np.save(sys.argv[1], x)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for kappa in (1e4, 1e8, 1e12):
        path = str(tmp_path / f"one_{kappa:g}.npy")
        subprocess.run([sys.executable, "-c", code % (root, os.path.join(root, "tests")), path, repr(kappa)], check=True,
                       env={**os.environ, "PSFM_CHOL_ONE_SIDED": "1"}, cwd=root)
        A, b = _conditioned_system(600, 35, kappa, seed=635)
        _check_band_solution(A, b, np.load(path))


@pytest.mark.parametrize("name", ["one_sided", "two_sided", "widest_band"])
def test_band_solve_real_reduced_systems(gpu, name):
    """Reduced camera systems S_c of bundle-adjustment problems (pass B, radius 1e4; test_schur_step's catalogue),
    rewritten into psfm_ba_band_solve's layout: 6 F band rows, 3 arrow rows (focal active, principal point identity),
    identity on the gauge's inactive slots.  The widest one (span 24, bw 149) runs the rank-1 kernel at its widest
    window (152): given only a scalar bandwidth, the block-6 form would need 26 blocks."""
    import test_schur_step as ts
    ref = ts.Reference(ts.linearization(name, True, True), 1e4)
    prob = ts._problem(name)
    nb = 6 * prob.num_images
    A = ref.Sc.astype(np.float64)
    b = ref.bcr.astype(np.float64)
    off = ~ref.lin.act_c
    A[off, :] = 0.0
    A[:, off] = 0.0
    A[off, off] = 1.0
    b[off] = 0.0
    bw = 6 * ts._span(prob) + 5
    rc, x = _solve(A, b, nb, bw)
    assert rc == 0, _lib.lib().psfm_last_error()
    _check_band_solution(A, b, x)
    assert np.all(x[off] == 0.0)


def test_two_sided_and_one_sided_forms_agree(gpu, tmp_path):
    """PSFM_CHOL_ONE_SIDED is read once per process: run the one-sided form in a child process."""
    import os
    import subprocess
    import sys
    code = ("import numpy as np, sys; sys.path[:0] = [%r, %r]; from test_gpu_band_chol import _system, _solve;"
            "A, b = _system(1203, 95, seed=9); rc, x = _solve(A, b, 1203, 95); assert rc == 0; np.save(sys.argv[1], x)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {}
    for name, env in (("two", {}), ("one", {"PSFM_CHOL_ONE_SIDED": "1"})):
        path = str(tmp_path / f"band_{name}.npy")
        subprocess.run([sys.executable, "-c", code % (root, os.path.join(root, "tests")), path], check=True, env={**os.environ, **env}, cwd=root)
        out[name] = np.load(path)
    assert np.abs(out["two"] - out["one"]).max() <= 1e-12 * np.abs(out["one"]).max()
    assert not np.array_equal(out["two"], out["one"])      # a different elimination order: not the same bits


@pytest.mark.parametrize("bad", [0, 57, 281, 282, 299, 317, 318, 450, 599])
def test_block6_two_sided_form_reports_a_bad_pivot_wherever_it_is(gpu, bad):
    """nb = 600, bw = 35: block-6 kernel, window of 6 image blocks, two CTAs (top-down 47 blocks, bottom-up 47, 6 in
    the middle)."""
    A, b = _system(600, 35, seed=5)
    rc, x = _solve(A, b, 600, 35)
    assert rc == 0
    ref = np.linalg.solve(A, b)
    assert np.abs(x - ref).max() <= 1e-11 * np.abs(ref).max()
    A[bad, bad] = -1.0
    rc, _ = _solve(A, b, 600, 35)
    assert rc == -1


def test_block6_forms_agree(gpu, tmp_path):
    """Block-6 two-sided (default) vs block-6 one-sided vs the rank-1 kernel on the bench shape (child processes:
    the switches are read once per process)."""
    import os
    import subprocess
    import sys
    code = ("import numpy as np, sys; sys.path[:0] = [%r, %r]; from test_gpu_band_chol import _system, _solve;"
            "A, b = _system(1200, 71, seed=11); rc, x = _solve(A, b, 1200, 71); assert rc == 0; np.save(sys.argv[1], x)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {}
    for name, env in (("b6two", {}), ("b6one", {"PSFM_CHOL_ONE_SIDED": "1"}), ("rank1", {"PSFM_CHOL_RANK1": "1"})):
        path = str(tmp_path / f"band_{name}.npy")
        subprocess.run([sys.executable, "-c", code % (root, os.path.join(root, "tests")), path], check=True, env={**os.environ, **env}, cwd=root)
        out[name] = np.load(path)
    scale = np.abs(out["rank1"]).max()
    assert np.abs(out["b6two"] - out["rank1"]).max() <= 1e-12 * scale
    assert np.abs(out["b6one"] - out["rank1"]).max() <= 1e-12 * scale
