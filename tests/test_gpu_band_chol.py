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
