"""The CPU oracle of the eval-time hole filling (oracle/inpaint_oracle.py) and the facts the device solver relies on: the border-clipped
stencils, symmetry and positive definiteness of the system, equality of the per-region and global solves.  Also the host-side part of
the C ABI (the workspace size and the all-zero refusal), which needs no GPU."""
import ctypes

import numpy as np
import pytest

from oracle import inpaint_oracle as IO


def _coef(shape, idx):
    return IO.stencil(shape, idx)[1].astype(np.int64)


def test_border_clipped_stencils_exact():
    assert np.array_equal(_coef((10, 10), (5, 5)), [[0, 0, 1, 0, 0], [0, 2, -8, 2, 0], [1, -8, 20, -8, 1], [0, 2, -8, 2, 0], [0, 0, 1, 0, 0]])
    assert np.array_equal(_coef((10, 10), (1, 5)), [[0, 2, -7, 2, 0], [1, -8, 20, -8, 1], [0, 2, -8, 2, 0], [0, 0, 1, 0, 0]])
    assert np.array_equal(_coef((10, 10), (0, 5)), [[1, -6, 12, -6, 1], [0, 2, -7, 2, 0], [0, 0, 1, 0, 0]])
    assert np.array_equal(_coef((10, 10), (0, 0)), [[6, -5, 1], [-5, 2, 0], [1, 0, 0]])
    # every stencil is integer-valued and mirrors with the image
    assert np.array_equal(_coef((10, 10), (9, 9)), _coef((10, 10), (0, 0))[::-1, ::-1])
    assert np.array_equal(IO.stencil((10, 10), (3, 1))[1], IO.stencil((10, 10), (3, 1))[1].round())


def test_system_symmetric_positive_definite_with_borders():
    rng = np.random.default_rng(1)
    worst = np.inf
    for _ in range(40):
        h, w = rng.integers(3, 31, size=2)
        img = rng.random((h, w)) + 1.0
        mask = rng.random((h, w)) < rng.uniform(0.05, 0.9)
        mask[0, 0] = False
        if not mask.any():
            mask[-1, -1] = True
        _, A = IO.global_solve(img, mask)
        A = A.toarray()
        assert np.array_equal(A, A.T)
        worst = min(worst, np.linalg.eigvalsh(A).min())
    assert worst > 0.0


def test_cubic_field_reproduced_in_interior_hole():
    y, x = np.mgrid[0:24, 0:30].astype(np.float64)
    field = 3.0 + 0.05 * x ** 3 - 0.02 * y ** 3 + 0.01 * x * x * y - 0.03 * x * y * y + 0.4 * x * y + 0.2 * y
    field -= field.min() - 1.0
    mask = np.zeros(field.shape, bool)
    mask[8:15, 10:19] = True
    out = IO.inpaint_biharmonic(field, mask)
    assert np.abs(out - field).max() <= 1e-8 * np.abs(field).max()


def test_region_split_equals_global_solve():
    rng = np.random.default_rng(2)
    img = (rng.random((26, 34)) * 10 + 1).astype(np.float64)
    mask = np.zeros(img.shape, bool)
    mask[0:4, 3:9] = True          # touches the top edge
    mask[10:14, 10:13] = True
    mask[12, 15] = True            # within reach of the blob: the same region
    mask[20:26, 28:34] = True      # corner
    mask[rng.random(img.shape) < 0.03] = True
    per_region = IO.inpaint_biharmonic(img, mask)
    whole, _ = IO.global_solve(img, mask)
    assert np.abs(per_region - whole).max() <= 1e-9 * np.abs(whole).max()


def test_result_clipped_to_known_range():
    img = np.full((16, 16), 5.0)
    img[6:10, 2] = 1.0
    img[6:10, 13] = 1.0
    img[5, 3:13] = 9.0
    img[10, 3:13] = 9.0
    mask = np.zeros(img.shape, bool)
    mask[6:10, 3:13] = True
    _, A = IO.global_solve(img, mask)
    raw = IO.spsolve(A.tocsc(), _rhs(img, mask))
    assert raw.max() > 9.0 or raw.min() < 1.0          # the unclipped solution overshoots the known range
    out = IO.inpaint_biharmonic(img, mask)
    assert out[mask].min() >= 1.0 and out[mask].max() <= 9.0
    assert np.allclose(out[mask], np.clip(raw, 1.0, 9.0), rtol=0, atol=1e-12)        # argwhere and boolean indexing: both row-major


def _rhs(img, mask):
    pts = np.argwhere(mask)
    rhs = np.zeros(len(pts))
    for n, p in enumerate(pts):
        b_lo, coef = IO.stencil(mask.shape, p)
        for off, c in np.ndenumerate(coef):
            q = tuple(b_lo + np.asarray(off))
            if c != 0 and not mask[q]:
                rhs[n] -= c * img[q]
    return rhs


def test_sample_without_holes_bit_identical_and_all_zero_raises():
    rng = np.random.default_rng(3)
    d = (rng.random((3, 1, 12, 20)) + 0.5).astype(np.float32)
    d[1, 0, 4:7, 5:9] = 0.0
    out = IO.inpainting(d)
    assert np.array_equal(out[0], d[0]) and np.array_equal(out[2], d[2])
    assert (out[1] != 0).all()
    d[2] = 0.0
    with pytest.raises(ValueError):
        IO.inpainting(d)


def test_abi_workspace_size_and_all_zero_refusal():
    from tta_depth_completion_b200 import _lib
    L = _lib.lib()
    n, h, w = 2, 352, 1216
    summary = (ctypes.c_uint * (4 * n + 4))()
    summary[0] = 40 * 1216
    nbytes = ctypes.c_size_t()
    assert L.ptta_inpaint_workspace_bytes(summary, n, h, w, ctypes.byref(nbytes)) == 0, _lib.last_error()
    m = min(h, w)
    arena = 8 * 40 * 1216 * (3 + 2 * min(40 * 1216, 2 * m))
    assert arena < nbytes.value < arena + (64 << 20)
    summary[4] = h * w
    assert L.ptta_inpaint_workspace_bytes(summary, n, h, w, ctypes.byref(nbytes)) != 0
    assert 'no known pixel' in _lib.last_error()
