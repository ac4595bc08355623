"""The contour oracle (skimage.measure.find_contours restated, the outline step of
display_instances, serve.py:160-169) against hand-worked answers and the structural facts of
marching squares on binary masks; the cycle rule the device implements against the oracle's
literal dict/deque assembly; and host-side argument validation of the contour entry points."""
import ctypes as C

import numpy as np
import pytest
from scipy import ndimage as ndi

from oracle import contours as oracle
from oracle.contours import _assemble_contours, _get_contour_segments
from matterport_maskrcnn_with_tensorflow_serving_b200 import _native as N


def _area(c):
    """Shoelace area of a closed (x, y) polygon (y down: islands come out positive)."""
    return 0.5 * float(np.sum(c[:-1, 0] * c[1:, 1] - c[1:, 0] * c[:-1, 1]))


def _padded(mask):
    p = np.zeros((mask.shape[0] + 2, mask.shape[1] + 2), np.uint8)
    p[1:-1, 1:-1] = mask
    return p


def cycle_rule(segments):
    """What the device computes: every segment's successor is the segment leaving its `to`
    point; cycles in order of their first-emitted segment, each starting at the `to` point of
    its last-emitted segment and closed."""
    leaving = {a: i for i, (a, b) in enumerate(segments)}
    seen = [False] * len(segments)
    out = []
    for i in range(len(segments)):
        if seen[i]:
            continue
        cyc, j = [], i
        while not seen[j]:
            seen[j] = True
            cyc.append(j)
            j = leaving[segments[j][1]]
        last = max(cyc)
        pts, j = [segments[last][1]], leaving[segments[last][1]]
        while True:
            pts.append(segments[j][1])
            if j == last:
                break
            j = leaving[segments[j][1]]
        out.append(np.array(pts))
    return out


def _check(mask, want):
    got = oracle.mask_contours(np.array(mask, bool))
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.dtype == np.float64
        assert np.array_equal(g, np.array(w, np.float64)), g.tolist()
    return got


def test_single_pixel_known_answer():
    m = np.zeros((3, 3), bool)
    m[1, 1] = True
    (c,) = _check(m, [[[1, 1.5], [0.5, 1], [1, 0.5], [1.5, 1], [1, 1.5]]])
    assert _area(c) == 0.5


def test_two_by_two_block():
    (c,) = _check([[0, 0, 0, 0], [0, 1, 1, 0], [0, 1, 1, 0], [0, 0, 0, 0]],
                  [[[2, 2.5], [1, 2.5], [0.5, 2], [0.5, 1], [1, 0.5], [2, 0.5], [2.5, 1],
                    [2.5, 2], [2, 2.5]]])
    assert _area(c) == 3.5        # the 2x2 block with its corners cut by the midpoints


def test_one_pixel_hole():
    outer, hole = _check([[1, 1, 1], [1, 0, 1], [1, 1, 1]],
                         [[[2, 2.5], [1, 2.5], [0, 2.5], [-0.5, 2], [-0.5, 1], [-0.5, 0],
                           [0, -0.5], [1, -0.5], [2, -0.5], [2.5, 0], [2.5, 1], [2.5, 2],
                           [2, 2.5]],
                          [[1.5, 1], [1, 0.5], [0.5, 1], [1, 1.5], [1.5, 1]]])
    assert _area(outer) > 0 and _area(hole) == -0.5


def test_diagonal_pair_is_two_contours():
    # padded cell (1, 1) is case 9: the high diagonal is not connected
    a, b = _check([[1, 0], [0, 1]],
                  [[[0, 0.5], [-0.5, 0], [0, -0.5], [0.5, 0], [0, 0.5]],
                   [[1, 1.5], [0.5, 1], [1, 0.5], [1.5, 1], [1, 1.5]]])
    assert _area(a) == _area(b) == 0.5


def test_anti_diagonal_pair_is_two_contours():
    # padded cell (1, 1) is case 6
    _check([[0, 1], [1, 0]],
           [[[1, 0.5], [0.5, 0], [1, -0.5], [1.5, 0], [1, 0.5]],
            [[0, 1.5], [-0.5, 1], [0, 0.5], [0.5, 1], [0, 1.5]]])


def test_full_mask_reaches_the_image_border():
    (c,) = oracle.mask_contours(np.ones((5, 7), bool))
    assert c[:, 0].min() == -0.5 and c[:, 0].max() == 7 - 0.5
    assert c[:, 1].min() == -0.5 and c[:, 1].max() == 5 - 0.5
    assert _area(c) > 0
    assert oracle.mask_contours(np.zeros((4, 4), bool)) == []


def test_find_contours_interpolates_off_half_levels():
    img = np.zeros((3, 3))
    img[1, 1] = 2.0
    (c,) = oracle.find_contours(img, 0.5)         # (0.5 - 0) / (2 - 0) = 0.25 of the way from 0
    assert np.array_equal(c, [[1.75, 1], [1, 0.25], [0.25, 1], [1, 1.75], [1.75, 1]])


@pytest.mark.parametrize("seed", range(3))
def test_random_masks_structure_and_cycle_rule(seed):
    rng = np.random.default_rng(seed)
    for _ in range(100):
        h, w = rng.integers(1, 16, 2)
        m = rng.random((h, w)) < rng.random()
        p = _padded(m)
        segs = _get_contour_segments(p, 0.5)
        lit = _assemble_contours(segs)
        rule = cycle_rule(segs)
        assert len(lit) == len(rule) and all(np.array_equal(a, b) for a, b in zip(lit, rule))
        cs = oracle.mask_contours(m)
        assert len(cs) == len(lit)
        assert all(np.array_equal(c[0], c[-1]) for c in cs)
        # vertices (without the closing repeats) = midpoints of the 4-adjacent padded pixel
        # pairs that differ, in (x, y) without the padding
        verts = sorted(tuple(v) for c in cs for v in c[:-1].tolist())
        edges = sorted([(c - 1.0, r + 0.5 - 1) for r, c in zip(*np.nonzero(p[1:] != p[:-1]))] +
                       [(c + 0.5 - 1, r - 1.0) for r, c in zip(*np.nonzero(p[:, 1:] != p[:, :-1]))])
        assert verts == edges
        n4 = ndi.label(p)[1]
        holes = ndi.label(1 - p, structure=np.ones((3, 3)))[1] - 1
        assert len(cs) == n4 + holes
        assert sum(_area(c) > 0 for c in cs) == n4


def test_mask_contours_batch_is_per_instance():
    rng = np.random.default_rng(5)
    masks = rng.random((9, 11, 4)) < 0.4
    masks[:, :, 2] = False
    got = oracle.mask_contours_batch(masks)
    assert len(got) == 4 and got[2] == []
    for i in range(4):
        assert all(np.array_equal(a, b) for a, b in zip(got[i], oracle.mask_contours(masks[:, :, i])))


def test_contour_entry_points_validate_arguments():
    lib = N.load()
    p16 = C.c_void_p(16)
    ok = (p16, p16, p16, p16, p16, p16, p16)
    assert lib.mrx_contours_count(None, p16, p16, p16, p16, p16, p16, 1, 4, 64, 64, None) == -1
    assert lib.mrx_contours_count(*ok, 0, 4, 64, 64, None) == -1            # B < 1
    assert lib.mrx_contours_count(*ok, 1, 0, 64, 64, None) == -1            # R < 1
    assert lib.mrx_contours_count(*ok, 1, 4, 0, 64, None) == -1
    assert lib.mrx_contours_count(*ok, 1, 4, 64, 40000, None) == -2         # side too large
    assert b"too large" in lib.mrx_last_error()
    assert lib.mrx_contours_count(*ok, 1, 4, 32767, 64, None) == -2
    assert lib.mrx_contours_write(*ok, None, None, None, None, C.c_longlong(0), 1, 4, 64, 64,
                                  None) == -1                                # no contour counts
    assert lib.mrx_contours_write(*ok, None, p16, p16, p16, C.c_longlong(8), 1, 4, 64, 64,
                                  None) == -1                                # no scratch
    assert lib.mrx_contours_write(*ok, p16, p16, p16, p16, C.c_longlong(-1), 1, 4, 64, 64,
                                  None) == -1
    assert lib.mrx_contours_write(None, *ok[1:], p16, p16, p16, p16, C.c_longlong(8), 1, 4, 64,
                                  64, None) == -1
    assert b"mrx_contours_write" in lib.mrx_last_error()
