"""CPU tests of the mask-refinement row (SURVEY 8f N1): the oracle restatement (oracle/mask_refine_ref.py) against closed-form
properties and hand-derived geometry, and the product's host logic (mit_b200/mask_refinement.py) against the oracle.
pydensecrf and shapely are not installed and not part of the reference tree, so the DenseCRF part is `parity unpinned` (see the oracle's header)."""
import math
import os

import cv2
import numpy as np

from mit_b200.host import geometry
from oracle import cases
from oracle import mask_refine_ref as R


def _host_module():
    """mit_b200.mask_refinement imports torch/ctypes only; its geometry helpers run anywhere."""
    from mit_b200 import mask_refinement
    return mask_refinement


def test_polygon_helpers_hand_derived():
    M = _host_module()
    sq = np.array([[0, 0], [4, 0], [4, 4], [0, 4]], float)
    diamond = np.array([[2, 0], [4, 2], [2, 4], [0, 2]], float)                  # area 8
    for area, clip, dist in ((R.poly_area, R.intersection_area_rect, R.point_poly_distance), (M._poly_area, M._overlap_area, M._point_distance)):
        assert area(sq) == 16 and area(diamond) == 8 and area(sq[::-1]) == 16
        assert clip(sq, 1, 1, 3, 3) == 4 and clip(sq, 2, 2, 10, 10) == 4 and clip(sq, 5, 5, 6, 6) == 0
        assert abs(clip(diamond, 0, 0, 2, 2) - 2.0) < 1e-12                     # one quadrant of the diamond
        assert abs(clip(diamond, 1, 1, 3, 3) - 4.0) < 1e-12                     # the inscribed square
        assert abs(clip(diamond, 0, 0, 4, 1) - 1.0) < 1e-12                     # the top cap: triangle of height 1, base 2
        assert dist(sq, 2, 2) == 0 and dist(sq, 6, 2) == 2 and abs(dist(sq, 7, 8) - 5.0) < 1e-12
        assert abs(dist(diamond, 0, 0) - math.sqrt(2)) < 1e-12


def test_permutohedral_restatement_properties():
    """Closed-form checks of the lattice restatement: (1) it is a symmetric positive filter (sum_i a_i (K b)_i == sum_i b_i (K a)_i);
    (2) normalised by its response to the constant signal it approximates the Gaussian exp(-|f_i - f_j|^2 / 2) the densecrf paper
    derives it for; (3) barycentric weights sum to one."""
    rng = np.random.default_rng(0)
    H, W, s = 24, 32, 3.0
    ys, xs = np.mgrid[0:H, 0:W]
    feat = np.stack([xs.reshape(-1) / s, ys.reshape(-1) / s]).astype(np.float32)
    lat = R.Permutohedral(feat)
    assert np.allclose(lat.bary.sum(1), 1.0, atol=1e-5) and (lat.bary > -1e-6).all()
    a, b = rng.random((1, H * W)).astype(np.float32), rng.random((1, H * W)).astype(np.float32)
    Ka, Kb = lat.compute(a), lat.compute(b)
    assert abs(float((a * Kb).sum() - (b * Ka).sum())) < 1e-3 * float((a * Kb).sum())
    norm = lat.compute(np.ones((1, H * W), np.float32))
    d2 = ((feat[:, :, None] - feat[:, None, :]) ** 2).sum(0)
    G = np.exp(-0.5 * d2)
    exact = (G @ a[0]) / G.sum(1)
    approx = (Ka / norm)[0]
    inner = (slice(4, H - 4), slice(4, W - 4))
    e, x = approx.reshape(H, W)[inner], exact.reshape(H, W)[inner]
    assert np.corrcoef(e.ravel(), x.ravel())[0, 1] > 0.97 and np.abs(e - x).max() < 0.08
    # 5-D lattice of a flat-colour image degenerates to its spatial part: same filter as the 2-D lattice with the same sxy
    rgb = np.full((H * W, 3), 77, np.float32) / 7.0
    lat5 = R.Permutohedral(np.concatenate([feat, rgb.T]))
    r5, r2 = lat5.compute(a) / lat5.compute(np.ones_like(a)), Ka / norm
    assert np.abs(r5 - r2)[0].reshape(H, W)[inner].max() < 0.1


def test_dense_crf_restatement_behaviour():
    """Mean field on a two-colour image: a noisy mask snaps to the colour edge (what refine_mask is used for)."""
    rng = np.random.default_rng(1)
    H, W = 40, 60
    img = np.full((H, W, 3), 230, np.uint8)
    img[10:30, 15:45] = 20
    truth = np.zeros((H, W), np.uint8)
    truth[10:30, 15:45] = 255
    noisy = truth.copy()
    flip = rng.random((H, W)) < 0.08
    noisy[flip] = 255 - noisy[flip]
    out = R.refine_mask(img, noisy)
    assert set(np.unique(out)) <= {0, 255}
    assert (out != truth).mean() < 0.01 < (noisy != truth).mean()


_regions = cases.refine_regions
_page = cases.refine_page


def test_assignment_product_equals_oracle():
    """The product's component -> text-line assignment (own vectorised geometry, bounding-box pre-filter) against the oracle's
    statement-order restatement of complete_mask, on the components of a synthetic page plus hand-made strays."""
    M = _host_module()
    page, boxes, raw = _page()
    scale = 2.0 / 3.0
    lines = [R._Line(geometry.Quadrilateral, b * scale) for b in boxes]
    small = cv2.resize(raw, (int(raw.shape[1] * scale), int(raw.shape[0] * scale)), interpolation=cv2.INTER_LINEAR)
    small[small > 0] = 255
    num, _, stats, _ = cv2.connectedComponentsWithStats(small)
    extra = np.array([[5, 5, 30, 4, 100], [300, 2, 3, 3, 9], [0, 0, small.shape[1], small.shape[0], 500000],
                      [int(boxes[0][0][0] * scale) - 14, int(boxes[0][0][1] * scale) + 3, 6, 6, 30]], dtype=stats.dtype)
    stats = np.concatenate([stats, extra])
    want = R.assign_components(stats, lines)
    xyxy = np.stack([stats[:, 0], stats[:, 1], stats[:, 0] + stats[:, 2] - 1, stats[:, 1] + stats[:, 3] - 1, stats[:, 4]], 1)
    got = M.assign_components(xyxy[1:], [np.asarray(l.pts, float) for l in lines], [l.font_size for l in lines])
    assert np.array_equal(got, want[1:]) and (got >= 0).sum() > 20 and (got < 0).sum() >= 2


def test_oracle_dispatch_on_synthetic_page():
    page, boxes, raw = _page()
    out = R.dispatch(_regions(boxes), page, raw.copy(), geometry.Quadrilateral, dilation_offset=0)
    assert out.shape == raw.shape and set(np.unique(out)) <= {0, 255}
    strokes = page[..., 0] < 100
    assert (out[strokes] == 255).mean() > 0.99                   # every stroke is covered ...
    box_area = np.zeros_like(raw)
    for b in boxes:
        cv2.fillPoly(box_area, [b.astype(np.int32)], 255)
    box_area = cv2.dilate(box_area, np.ones((41, 41), np.uint8))
    assert (out[box_area == 0] == 0).all()                        # ... and nothing far from the text lines is


def _reference():
    """What the reference's own code returned on these inputs (tests/golden, oracle/make_reference_golden.py)."""
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_mask_refinement.npz"))


def test_scaled_float_lines_match_reference_quadrilateral():
    """dispatch builds Quadrilateral(line * scale_factor): float corners.  Our class must read them as the reference's does."""
    g = _reference()
    _, boxes, _ = _page()
    for i, b in enumerate(boxes + [np.array([[10, 20], [200, 35], [195, 80], [5, 66]])]):
        a = R._Line(geometry.Quadrilateral, b * (2.0 / 3.0))
        assert np.array_equal(a.pts, g[f"line{i}_pts"]) and a.font_size == g[f"line{i}_font_size"] and np.array_equal(a.aabb_xywh, g[f"line{i}_aabb"])


def test_oracle_dispatch_equals_reference_code_with_restated_dependencies():
    """Pins the statement-order restatement (oracle/mask_refine_ref.py: dispatch, complete_mask, assignment, rectangle arithmetic incl. the
    int32 wrap of empty lines, dilation sizes) on the reference's OWN mask_refinement code, executed unmodified with shapely / pydensecrf
    bound to the oracle's restatements of those two libraries (which remain unpinned themselves)."""
    g = _reference()
    for seed, (h, w, n), offset in cases.REFINE_DISPATCH_CASES:
        page, regions, raw = cases.refine_dispatch_case(seed, h, w, n)
        want = g[f"dispatch_{seed}"]
        got = R.dispatch(regions, page, raw.copy(), geometry.Quadrilateral, dilation_offset=offset, kernel_size=3)
        assert want.dtype == np.uint8 and np.array_equal(got, want), int((got != want).sum())
        assert (want > 0).mean() > 0.02
