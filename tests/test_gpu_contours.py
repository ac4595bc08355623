"""Contour polygons of display_instances (serve.py:160-169) computed on the device: every result
must equal, array for array (same number of contours, same order, same start vertex),
`oracle.contours.mask_contours` of the mask `unmold_detections` returns for the same instance."""
import numpy as np
import pytest
import torch

from oracle import contours as oracle
from matterport_maskrcnn_with_tensorflow_serving_b200 import api_utils, synth, visualize
from matterport_maskrcnn_with_tensorflow_serving_b200.engine import UnmoldEngine, make_geom

from helpers import item_of

pytestmark = pytest.mark.gpu


def _same(got, want, what=""):
    assert len(got) == len(want), (what, len(got), len(want))
    for j, (g, w) in enumerate(zip(got, want)):
        assert g.dtype == np.float64 and g.shape == w.shape, (what, j, g.shape, w.shape)
        assert np.array_equal(g, w), (what, j)


def _check(ims, dtype=np.float32):
    items = [item_of(im, dtype) for im in ims]
    got = api_utils.unmold_detections_contours_batch(items)
    ref = api_utils.unmold_detections_batch(items)
    n_contours = 0
    for (b, c, s, polys), (rb, rc, rs, rm) in zip(got, ref):
        assert np.array_equal(b, rb) and np.array_equal(c, rc) and np.array_equal(s, rs)
        assert len(polys) == rb.shape[0]
        for i in range(rb.shape[0]):
            _same(polys[i], oracle.mask_contours(rm[:, :, i]), (i, tuple(rb[i])))
            n_contours += len(polys[i])
        # the host-mask entry point on the downloaded byte masks gives the same polygons
        if rb.shape[0]:
            for i, p in enumerate(visualize.mask_contours(rm, rb)):
                _same(p, polys[i], ("visualize", i))
    return n_contours


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("hw,n,R,kw", [
    ((96, 128), 12, 16, {}),
    ((64, 96), 40, 40, dict(min_box=60, max_box_frac=1.0)),     # full-height / full-width boxes
    ((40, 56), 30, 32, dict(min_box=20, max_box_frac=1.0)),     # boxes touching every border
    ((150, 150), 30, 32, dict(min_box=1, max_box_frac=0.1)),    # boxes smaller than the tile
    ((75, 333), 37, 40, {}),                                    # widths that are no multiple of 32
    ((33, 1000), 7, 8, {}),
    ((17, 9), 3, 4, dict(min_box=1, max_box_frac=1.0)),         # width no multiple of 8
    ((64, 80), 0, 4, {}),                                       # nothing detected
])
def test_contours_equal_oracle(cuda_device, hw, n, R, kw, dtype):
    rng = np.random.default_rng(81)
    ims = [synth.make_image(rng, hw, n, num_classes=4, max_instances=R, **kw) for _ in range(3)]
    _check(ims, dtype)


def _host_check(masks, boxes=None):
    got = visualize.mask_contours(masks, boxes)
    assert len(got) == masks.shape[-1]
    for i in range(masks.shape[-1]):
        _same(got[i], oracle.mask_contours(masks[:, :, i]), i)
    return got


def test_hand_masks(cuda_device):
    H, W = 41, 45
    m = np.zeros((H, W, 5), bool)
    yy, xx = np.mgrid[:H, :W]
    m[:, :, 0] = ((yy + xx) % 2 == 0) & (yy > 2) & (yy < 30) & (xx > 1)     # every cell a saddle
    r = np.maximum(np.abs(yy - 20), np.abs(xx - 22))
    m[:, :, 1] = (r % 4 == 0) | (r % 4 == 1)                               # nested rings
    m[5, 3:40, 2] = True                                                   # one-pixel lines
    m[8:35, 20, 2] = True
    m[30, :, 2] = True
    m[:, 44, 2] = True
    # m[:, :, 3] all zero
    m[:, :, 4] = True
    got = _host_check(m)
    assert got[3] == [] and len(got[0]) > 100 and len(got[1]) == 11


def test_masks_larger_than_the_shared_memory_path(cuda_device):
    """A 256x256 checkerboard has ~130 k segments (the walk runs on global memory); next to it,
    instances that fit shared memory."""
    H = W = 260
    m = np.zeros((H, W, 3), bool)
    yy, xx = np.mgrid[:H, :W]
    m[2:258, 2:258, 0] = ((yy + xx) % 2 == 0)[2:258, 2:258]
    m[:, :, 1] = np.random.default_rng(3).random((H, W)) < 0.5            # ~60 k segments
    m[100:140, 50:90, 2] = True
    got = _host_check(m)
    assert len(got[0]) == 256 * 256 // 2 and len(got[2]) == 1


def test_boxes_limit_the_scan(cuda_device):
    """With boxes, pixels outside a box are read as zero."""
    rng = np.random.default_rng(4)
    m = rng.random((50, 70, 3)) < 0.5
    boxes = np.array([[0, 0, 50, 70], [10, 13, 31, 60], [49, 69, 50, 70]], np.int32)
    got = visualize.mask_contours(m, boxes)
    for i, (y1, x1, y2, x2) in enumerate(boxes):
        inside = np.zeros(m.shape[:2], bool)
        inside[y1:y2, x1:x2] = m[y1:y2, x1:x2, i]
        _same(got[i], oracle.mask_contours(inside), i)
    assert visualize.mask_contours(np.zeros((8, 8, 0), bool)) == []


def test_packed_and_canvas_sources_agree(cuda_device):
    ims = synth.make_batch(82, 3, (120, 200), 20, num_classes=5, max_instances=24)
    items = [item_of(im, np.float32) for im in ims]
    eng = UnmoldEngine(3, 24, (28, 28), 5)
    d_det = torch.from_numpy(np.stack([i[0] for i in items])).cuda()
    d_msk = torch.from_numpy(np.stack([i[1] for i in items])).cuda()
    eng.plan([make_geom(*i[2:]) for i in items], canvas=True)
    eng.enqueue(d_det, d_msk)
    eng.enqueue_expand_packed()
    counts = eng.fetch_meta()[0].copy()
    direct = eng.enqueue_contours(source="packed").to_host(counts)
    packed = eng.enqueue_contours(source="canvas").to_host(counts)
    ref = api_utils.unmold_detections_batch(items)
    for b in range(3):
        assert len(direct[b]) == len(packed[b]) == counts[b] == ref[b][0].shape[0]
        for k in range(int(counts[b])):
            _same(direct[b][k], packed[b][k], (b, k))
            _same(direct[b][k], oracle.mask_contours(ref[b][3][:, :, k]), (b, k))


def test_contours_full_size_batch(cuda_device):
    """BASELINE.json configs[1] shape, ragged second image."""
    ims = synth.make_batch(83, 1, (1024, 1024), 100) + synth.make_batch(84, 1, (1024, 1024), 37)
    assert _check(ims) > 1000
