"""Mask overlay of `visualize.display_instances` (reference: /root/reference/serve.py:160-169,
`mrcnn.visualize` is un-vendored there) on the device.

The reference passes the `[H, W, N]` bool masks `unmold_detections` returned to matplotlib
code that (per instance, in order) alpha-blends a colour into the image where the mask is
set, then draws boxes, captions and contour polygons as matplotlib artists and saves a PNG.
This module does the blending part -- the only part that touches every mask byte -- with
`mrx_composite_masks`, either on masks the caller holds as NumPy arrays (`apply_masks`,
`display_instances`) or directly on the device canvas of an `UnmoldEngine`
(`composite_batch`), which avoids the 105 MB per image device -> host copy of the masks
when only the overlay is wanted.  The contour polygons are computed on the device too
(`mask_contours`, `api_utils.unmold_detections_contours_batch`), but boxes, captions and
polygons are NOT drawn (matplotlib rendering is out of scope, DESIGN.md section 7).
"""
from __future__ import annotations

import colorsys
import ctypes as C
import random as _random

import numpy as np

from . import _native as N


def random_colors(n, bright=True, rng=None):
    """`n` distinct colours as RGB float triples in [0, 1]: evenly spaced hues at full
    saturation, shuffled (the values upstream's `random_colors` produces).  Upstream shuffles
    with the process-global `random`; pass a `random.Random` to get a reproducible order."""
    value = 1.0 if bright else 0.7
    colors = [colorsys.hsv_to_rgb(i / n, 1, value) for i in range(n)]
    (rng or _random).shuffle(colors)
    return colors


def blend_table(colors, alpha, R):
    """[R, 3] float64 rows `alpha * color[c] * 255` in Python's (= NumPy's) evaluation order."""
    tab = np.zeros((R, 3), dtype=np.float64)
    for i, col in enumerate(colors[:R]):
        for c in range(3):
            tab[i, c] = alpha * float(col[c]) * 255
    return tab


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _is_triple(x):
    return len(x) == 3 and not hasattr(x[0], "__len__")


class CompositeStage:
    """Device-side inputs of the overlay for one planned batch (images, blend table, scratch),
    staged once; `run()` launches `mrx_composite_masks` on the engine's current canvas.  Lets a
    pipeline (or a benchmark) separate the upload of the images from the kernel."""

    def __init__(self, engine, images, colors, alpha=0.5):
        import torch

        N.require_cuda()
        self.lib = N.load()
        self.engine = engine
        B = engine._n_images
        if B == 0 or len(images) != B:
            raise ValueError(f"{len(images)} images for a plan of {B}")
        dev = engine.device
        geom = engine._geom_host
        self.geom = geom
        sizes = [int(geom[b][0]) * int(geom[b][1]) * 3 for b in range(B)]
        offs = np.zeros(B + 1, dtype=np.int64)
        np.cumsum(sizes, out=offs[1:])
        self.offs = offs
        self.d_in = torch.empty(int(offs[-1]), dtype=torch.uint8, device=dev)
        for b, img in enumerate(images):
            t = img if torch.is_tensor(img) else torch.from_numpy(np.ascontiguousarray(img))
            if t.dtype != torch.uint8 or t.numel() != sizes[b]:
                raise ValueError(f"image {b}: expected uint8 {geom[b][0]}x{geom[b][1]}x3")
            self.d_in[int(offs[b]):int(offs[b + 1])].copy_(t.reshape(-1), non_blocking=True)
        self.d_out = torch.empty_like(self.d_in)
        shared = len(colors) > 0 and _is_triple(colors[0])
        if not shared and len(colors) != B:
            raise ValueError("colors: one list of RGB triples, or one list per image")
        tab = np.stack([blend_table(colors if shared else colors[b], alpha, engine.R)
                        for b in range(B)])
        self.alpha = alpha
        self.d_tab = torch.from_numpy(tab).to(dev)
        self.d_off = torch.from_numpy(offs[:B].copy()).to(dev)
        self.max_px = max(int(geom[b][0]) * int(geom[b][1]) for b in range(B))

    def run(self, stream=None):
        eng = self.engine
        N.check(self.lib.mrx_composite_masks(
            _ptr(eng.d_canvas), _ptr(eng.d_canvas_off), _ptr(eng.d_counts),
            _ptr(eng.d_geom), _ptr(eng.d_boxes), _ptr(self.d_in), _ptr(self.d_off),
            _ptr(self.d_tab), C.c_double(1 - self.alpha),
            _ptr(self.d_out), eng._n_images, eng.R, C.c_longlong(self.max_px),
            N.stream_ptr(stream)), "mrx_composite_masks")
        offs, geom = self.offs, self.geom
        return [self.d_out[int(offs[b]):int(offs[b + 1])].view(int(geom[b][0]), int(geom[b][1]), 3)
                for b in range(eng._n_images)]


def composite_batch(engine, images, colors, alpha=0.5, stream=None):
    """Overlay the masks an `UnmoldEngine` holds on its device canvas (after `enqueue`).

    images: list of uint8 HxWx3 arrays (NumPy or CUDA tensors), one per planned image, each
    of the engine's canvas size for that image.  colors: a list of RGB triples shared by all
    images, or one such list per image.  Returns a list of uint8 HxWx3 CUDA tensors.
    """
    return CompositeStage(engine, images, colors, alpha).run(stream)


def apply_masks(image, boxes, masks, colors, alpha=0.5):
    """NumPy in, NumPy out: the mask loop of `display_instances` for one image.

    image uint8 [H,W,3]; boxes [N,4]; masks bool [H,W,N] (the layout `unmold_detections`
    returns, which is the device canvas layout); colors: N RGB triples.  Returns uint8 [H,W,3].
    """
    import torch

    N.require_cuda()
    lib = N.load()
    image = np.ascontiguousarray(image)
    H, W = image.shape[:2]
    n = int(boxes.shape[0])
    if masks.shape[:2] != (H, W) or masks.shape[-1] != n:
        raise ValueError("masks must be [H, W, N] for N boxes")
    if n == 0:
        return image.astype(np.uint8).copy()
    dev = torch.device("cuda", torch.cuda.current_device())
    total = H * W * n
    d_canvas = torch.zeros((total + 15) // 16 * 16, dtype=torch.uint8, device=dev)
    d_canvas[:total].copy_(torch.from_numpy(
        np.ascontiguousarray(masks).view(np.uint8).reshape(-1)))
    d_off = torch.zeros(1, dtype=torch.int64, device=dev)
    d_counts = torch.tensor([n], dtype=torch.int32, device=dev)
    d_geom = torch.tensor([[H, W, H, W, 0, 0, H, W]], dtype=torch.int32, device=dev)
    d_boxes = torch.from_numpy(np.ascontiguousarray(boxes, dtype=np.int32)).to(dev)
    d_img = torch.from_numpy(image.astype(np.uint8, copy=False)).to(dev)
    d_out = torch.empty_like(d_img)
    d_tab = torch.from_numpy(blend_table(colors, alpha, n)).to(dev)
    N.check(lib.mrx_composite_masks(
        _ptr(d_canvas), _ptr(d_off), _ptr(d_counts), _ptr(d_geom), _ptr(d_boxes), _ptr(d_img),
        _ptr(d_off), _ptr(d_tab), C.c_double(1 - alpha), _ptr(d_out), 1, n,
        C.c_longlong(H * W), N.stream_ptr(None)), "mrx_composite_masks")
    return d_out.cpu().numpy()


def mask_contours(masks, boxes=None):
    """NumPy in, NumPy out: the outline step of `display_instances` for masks the caller holds.

    masks: bool [H, W, N] (the layout `unmold_detections` returns); boxes: [N, 4] int
    (y1, x1, y2, x2) -- a mask is read as zero outside its box, and only the box plus one ring
    of pixels is scanned; None = the whole image.  The masks are bit-packed on the host (1/8 of
    the bytes go to the device) and traced by `mrx_contours_*`.  Returns a list of N lists of
    float64 [K, 2] (x, y) arrays, each closed: for instance i, what
    find_contours(mask padded by one zero pixel, 0.5) gives, as `np.fliplr(verts) - 1`."""
    import torch

    from .engine import contours_device

    N.require_cuda()
    lib = N.load()
    masks = np.asarray(masks)
    if masks.ndim != 3:
        raise ValueError(f"masks must be [H, W, N], got {masks.shape}")
    H, W, n = masks.shape
    if n == 0:
        return []
    if boxes is None:
        boxes = np.tile(np.array([[0, 0, H, W]], np.int32), (n, 1))
    boxes = np.ascontiguousarray(boxes, dtype=np.int32)
    if boxes.shape != (n, 4):
        raise ValueError(f"boxes must be [{n}, 4], got {boxes.shape}")
    dev = torch.device("cuda", torch.cuda.current_device())
    packed = np.packbits(np.ascontiguousarray(masks.transpose(2, 0, 1)).astype(np.bool_), axis=-1)
    d_packed = torch.from_numpy(packed.reshape(-1)).to(dev)
    d_off = torch.zeros(1, dtype=torch.int64, device=dev)
    d_counts = torch.tensor([n], dtype=torch.int32, device=dev)
    d_geom = torch.tensor([[H, W, H, W, 0, 0, H, W]], dtype=torch.int32, device=dev)
    d_boxes = torch.from_numpy(boxes).to(dev)
    dc = contours_device(lib, dev, d_packed, d_off, d_boxes, d_counts, d_geom, 1, n, H, W)
    return dc.to_host([n])[0]


def display_instances(image, boxes, masks, class_ids=None, class_names=None, scores=None,
                      title="", figsize=(16, 16), ax=None, show_mask=True, show_bbox=True,
                      colors=None, captions=None, save_path=None):
    """Argument-compatible with the fork's `visualize.display_instances(..., save_path=)`
    (serve.py:160-169).  Computes the masked image (the pixels matplotlib would `imshow`);
    boxes, captions and contours are not drawn.  Returns the uint8 image; writes it to
    `save_path` (PNG via OpenCV) when given."""
    n = int(boxes.shape[0])
    if n:
        assert boxes.shape[0] == masks.shape[-1]
    colors = colors or random_colors(max(n, 1))
    out = apply_masks(image, boxes, masks, colors) if (show_mask and n) else \
        np.ascontiguousarray(image).astype(np.uint8).copy()
    if save_path is not None:
        import cv2

        cv2.imwrite(save_path, out[:, :, ::-1])   # OpenCV writes BGR
    return out
