"""CPU oracle of the eval-time hole filling of the reference's NLSPN wrapper (src/nlspn_model_adapt.py:124-127 ->
src/data_utils.py:327-354): every pixel of the prediction that is exactly 0 is filled, sample by sample, with
`skimage.restoration.inpaint_biharmonic`.

`inpaint_biharmonic` below restates scikit-image 0.18's algorithm line by line (skimage/restoration/inpaint.py:
`_get_neighborhood`, `_inpaint_biharmonic_single_channel`, `inpaint_biharmonic`; Damelin & Hoang, "On Surface Completion and
Image Inpainting by Biharmonic Functions: Numerical Aspects", 2018): the mask is split into the 8-connected labels of its
cross-dilation, each region is built as a `lil_matrix` of laplace(laplace(delta)) coefficients (scipy.ndimage, mode 'reflect')
on the 5x5 window clipped to the image, solved with `spsolve` and clipped to the (min, max) of the known pixels.  scikit-image
0.19 solves the same system in one piece; the regions are decoupled, so the solution is the same.  scikit-image is not a
dependency of this project, so this restatement is not pinned against it; only scipy is used.

`inpainting` is the per-sample wrapper: mask = (out == 0); an empty mask returns the sample untouched; a sample without any
known pixel raises ValueError from the empty `min`, as the reference does."""
import numpy as np
from scipy import ndimage as ndi
from scipy import sparse
from scipy.ndimage import laplace
from scipy.sparse.linalg import spsolve


def _get_neighborhood(nd_idx, radius, nd_shape):
    bounds_lo = (nd_idx - radius).clip(min=0)
    bounds_hi = (nd_idx + radius + 1).clip(max=nd_shape)
    return bounds_lo, bounds_hi


def stencil(shape, idx):
    """(window origin, laplace(laplace(delta))) of pixel idx on the 5x5 window clipped to an image of `shape`"""
    b_lo, b_hi = _get_neighborhood(np.asarray(idx), 2, np.asarray(shape))
    neigh_coef = np.zeros(b_hi - b_lo)
    neigh_coef[tuple(np.asarray(idx) - b_lo)] = 1
    return b_lo, laplace(laplace(neigh_coef))


def _inpaint_biharmonic_single_channel(mask, out, limits):
    matrix_unknown = sparse.lil_matrix((np.sum(mask), out.size))
    matrix_known = sparse.lil_matrix((np.sum(mask), out.size))
    mask_i = np.ravel_multi_index(np.where(mask), mask.shape)
    mask_pts = np.stack(np.where(mask), axis=-1)
    for mask_pt_n, mask_pt_idx in enumerate(mask_pts):
        b_lo, neigh_coef = stencil(out.shape, mask_pt_idx)
        it_inner = np.nditer(neigh_coef, flags=['multi_index'])
        for coef in it_inner:
            if coef == 0:
                continue
            tmp_pt_idx = np.add(b_lo, it_inner.multi_index)
            tmp_pt_i = np.ravel_multi_index(tmp_pt_idx, mask.shape)
            if mask[tuple(tmp_pt_idx)]:
                matrix_unknown[mask_pt_n, tmp_pt_i] = coef
            else:
                matrix_known[mask_pt_n, tmp_pt_i] = coef
    flat_diag_image = sparse.dia_matrix((out.flatten(), np.array([0])), shape=(out.size, out.size))
    matrix_known = matrix_known.tocsr()
    rhs = -(matrix_known * flat_diag_image).sum(axis=1)
    matrix_unknown = matrix_unknown[:, mask_i]
    matrix_unknown = sparse.csr_matrix(matrix_unknown)
    result = spsolve(matrix_unknown, rhs)
    result = np.clip(result, *limits)
    result = result.ravel()
    for mask_pt_n, mask_pt_idx in enumerate(mask_pts):
        out[tuple(mask_pt_idx)] = result[mask_pt_n]
    return out


def inpaint_biharmonic(image, mask):
    """skimage.restoration.inpaint_biharmonic(image, mask) of a 2-D float image (0.18, multichannel=False)"""
    image = np.asarray(image)
    if image.dtype not in (np.float32, np.float64):
        image = image.astype(np.float64)                      # img_as_float keeps float32 / float64
    mask = mask.astype(bool)
    kernel = ndi.generate_binary_structure(mask.ndim, 1)
    mask_dilated = ndi.binary_dilation(mask, structure=kernel)
    mask_labeled, num_labels = ndi.label(mask_dilated, structure=np.ones((3,) * mask.ndim))   # skimage.measure.label: full connectivity
    mask_labeled *= mask
    image = image[..., np.newaxis]
    out = np.copy(image)
    for idx_channel in range(image.shape[-1]):
        known_points = image[..., idx_channel][~mask]
        limits = (np.min(known_points), np.max(known_points))
        for idx_region in range(1, num_labels + 1):
            mask_region = mask_labeled == idx_region
            _inpaint_biharmonic_single_channel(mask_region, out[..., idx_channel], limits)
    return out[..., 0]


def inpainting(depth):
    """per-sample hole filling of a [N,1,H,W] (or [N,H,W]) prediction: numpy in, numpy out (a torch tensor is converted)"""
    d = depth.detach().cpu().numpy() if hasattr(depth, 'detach') else np.asarray(depth)
    out = np.array(d, copy=True)
    for b in range(out.shape[0]):
        sample = out[b, 0] if out.ndim == 4 else out[b]
        mask = sample == 0
        if not mask.any():
            continue
        sample[...] = inpaint_biharmonic(sample, mask)
    return out


def global_solve(image, mask):
    """the whole mask as ONE system (scikit-image 0.19's default split_into_regions=False), solved with spsolve and clipped"""
    image = np.asarray(image, dtype=np.float64)
    pts = np.argwhere(mask)
    index = -np.ones(mask.shape, dtype=np.int64)
    index[mask] = np.arange(len(pts))
    rows, cols, vals = [], [], []
    rhs = np.zeros(len(pts))
    for n, p in enumerate(pts):
        b_lo, coef = stencil(mask.shape, p)
        for off, c in np.ndenumerate(coef):
            if c == 0:
                continue
            q = tuple(b_lo + np.asarray(off))
            if mask[q]:
                rows.append(n)
                cols.append(index[q])
                vals.append(c)
            else:
                rhs[n] -= c * image[q]
    A = sparse.csr_matrix((vals, (rows, cols)), shape=(len(pts), len(pts)))
    known = image[~mask]
    x = np.clip(spsolve(A, rhs), known.min(), known.max())
    out = image.copy()
    out[mask] = x
    return out, A
