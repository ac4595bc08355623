"""Drop-in for the reference's `api.helpers.utils` (imported as `api_utils`,
/root/reference/serve.py:21): same function names, positional arguments, return tuples and
NumPy value semantics, computed by the sm_100a kernels in libmrx.so.

    get_anchors(image_shape)                                         serve.py:105
    unmold_detections(detections, mrcnn_mask, original_image_shape,
                      image_shape, window)                           serve.py:147-154
    load_img(path)                                                   serve.py:86

Plus batched entry points the reference lacks (it is hard-wired to one image per call,
serve.py:48): `unmold_detections_batch`, `unmold_detections_packed_batch`,
`unmold_detections_rle_batch`, `unmold_overlay_batch`, and `unmold_detections_contours_batch`
(the contour polygons of the reference's `display_instances`, serve.py:160-169).

Numerical contract (checked by tests/ against the float64 oracle): N, boxes, class ids and
scores are bit-exact.  The mask resize runs in float32 on exact integer source coordinates;
its pre-threshold samples are within 1e-6 of the reference's float64 values, so a mask pixel
can differ from the reference only where the reference's own value is within 1e-6 of the 0.5
threshold (none on the seeded test data).

Thread safety: these functions may be called from several threads (a threaded web server);
the cached engines are guarded by a lock held from planning a batch until its results are on
the host, so calls are serialised per (device, shape) engine, never interleaved.
"""
from __future__ import annotations

import threading
import weakref
from collections import OrderedDict

import numpy as np

from . import _native as N
from .engine import AnchorGenerator, UnmoldEngine, make_geom
from .model_configs import mconfig as _default_config

_state = {"config": _default_config, "anchors": None, "engines": OrderedDict()}
_state_lock = threading.RLock()

# at most this many cached engines (one per device / R / mask shape / dtypes); the least
# recently used one is released (its canvas and input buffers freed) when a new one is needed
MAX_CACHED_ENGINES = 4


def set_config(config):
    """Use another Matterport-style config object (attribute names of mrcnn/config.py)."""
    with _state_lock:
        _state["config"] = config
        _state["anchors"] = None


def get_config():
    return _state["config"]


def release():
    """Free every cached device buffer (engines, anchor memo, pinned result pool)."""
    with _state_lock:
        for eng in _state["engines"].values():
            eng.release()
            eng._inputs = None
        _state["engines"].clear()
        _state["anchors"] = None
        _pool.clear()


def load_img(path):
    """serve.py:85-86: file -> HxWx3 uint8 RGB ndarray (file IO; stays on the host)."""
    import cv2

    img = cv2.imread(path, cv2.IMREAD_COLOR)
    if img is None:
        raise FileNotFoundError(path)
    return cv2.cvtColor(img, cv2.COLOR_BGR2RGB)


def get_anchors(image_shape):
    """[A,4] float32 normalised (y1,x1,y2,x2) FPN anchors for a molded image shape;
    memoised by shape like upstream MaskRCNN.get_anchors."""
    with _state_lock:
        if _state["anchors"] is None:
            _state["anchors"] = AnchorGenerator(_state["config"])
        return _state["anchors"].get_anchors(image_shape)


# ----------------------------------------------------------------------------- host results
class _PinnedPool:
    """Pinned host buffers for results handed to the caller as NumPy arrays without an extra
    copy: a buffer goes back to the pool when the last array viewing it is garbage collected
    (pinning 100 MB costs far more than the copy it carries, so buffers are reused)."""

    GRANULE = 1 << 20
    MAX_BYTES = 4 << 30

    def __init__(self):
        self.free = {}
        self.bytes = 0
        self.lock = threading.Lock()

    def clear(self):
        with self.lock:
            self.free.clear()
            self.bytes = 0

    def _give_back(self, size, tensor):
        with self.lock:
            if self.bytes + size <= self.MAX_BYTES:
                self.free.setdefault(size, []).append(tensor)
                self.bytes += size

    def take(self, nbytes):
        """(tensor uint8 [nbytes] pinned, release hook to attach to the final ndarray)."""
        import torch

        size = max(self.GRANULE, (int(nbytes) + self.GRANULE - 1) // self.GRANULE * self.GRANULE)
        with self.lock:
            lst = self.free.get(size)
            t = lst.pop() if lst else None
            if t is not None:
                self.bytes -= size
        if t is None:
            t = torch.empty((size,), dtype=torch.uint8).pin_memory()
        return t, size

    def as_array(self, tensor, size, nbytes):
        """uint8 ndarray [nbytes] viewing `tensor`; the buffer returns to the pool when the
        array (and everything derived from it) is gone."""
        arr = tensor[:nbytes].numpy()
        weakref.finalize(arr.base, self._give_back, size, tensor)
        return arr


_pool = _PinnedPool()


# ----------------------------------------------------------------------------- staging
def _squeeze_inputs(detections, mrcnn_mask):
    detections = np.asarray(detections)
    mrcnn_mask = np.asarray(mrcnn_mask)
    # serve.py:131-136 reshapes to (-1, *cf.OUT_*_SHAPE): accept the leading unit dim
    if detections.ndim == 3 and detections.shape[0] == 1:
        detections = detections[0]
    if mrcnn_mask.ndim == 5 and mrcnn_mask.shape[0] == 1:
        mrcnn_mask = mrcnn_mask[0]
    if detections.ndim != 2 or detections.shape[1] != 6:
        raise ValueError(f"detections must be [R,6], got {detections.shape}")
    if mrcnn_mask.ndim != 4 or mrcnn_mask.shape[0] != detections.shape[0]:
        raise ValueError(f"mrcnn_mask must be [R,mh,mw,C] with R={detections.shape[0]}, "
                         f"got {mrcnn_mask.shape}")
    if detections.dtype not in (np.float32, np.float64):
        detections = detections.astype(np.float64)
    if mrcnn_mask.dtype not in (np.float32, np.float64):
        mrcnn_mask = mrcnn_mask.astype(np.float64)
    return np.ascontiguousarray(detections), np.ascontiguousarray(mrcnn_mask)


def _engine_for(batch, R, mh, mw, Cc, det_dtype, mask_dtype):
    import torch

    key = (torch.cuda.current_device(), R, mh, mw, Cc, np.dtype(det_dtype).str,
           np.dtype(mask_dtype).str)
    with _state_lock:
        engines = _state["engines"]
        eng = engines.get(key)
        if eng is not None and eng.B < batch:
            eng.release()
            eng._inputs = None
            eng = None
        if eng is None:
            while len(engines) >= MAX_CACHED_ENGINES:
                _, old = engines.popitem(last=False)
                old.release()
                old._inputs = None
            eng = UnmoldEngine(max(batch, 1), R, (mh, mw), Cc, det_dtype, mask_dtype)
            eng._inputs = None
        engines[key] = eng
        engines.move_to_end(key)
    return eng


class _Staged:
    """One batch on its engine: inputs uploaded, geometry planned, engine lock HELD until
    `close()` (use as a context manager)."""

    def __init__(self, items, canvas=True):
        import torch

        N.require_cuda()
        dets, masks, geoms = [], [], []
        for det, msk, osh, ish, win in items:
            d, m = _squeeze_inputs(det, msk)
            dets.append(d)
            masks.append(m)
            geoms.append(make_geom(osh, ish, win))
        d0, m0 = dets[0], masks[0]
        for d, m in zip(dets, masks):
            if d.shape != d0.shape or m.shape != m0.shape or d.dtype != d0.dtype or \
                    m.dtype != m0.dtype:
                raise ValueError("all images of a batch must share shapes and dtypes")
        self.n = n = len(items)
        self.geoms = geoms
        R, (mh, mw, Cc) = d0.shape[0], m0.shape[1:]
        self.eng = eng = _engine_for(n, R, mh, mw, Cc, d0.dtype, m0.dtype)
        eng.lock.acquire()
        try:
            eng.plan(geoms, canvas=canvas)
            # cached device inputs: no np.stack, no per-call device allocation
            if eng._inputs is None:
                from .engine import _torch_dtype
                eng._inputs = (
                    torch.empty((eng.B, R, 6), dtype=_torch_dtype(d0.dtype), device=eng.device),
                    torch.empty((eng.B, R, mh, mw, Cc), dtype=_torch_dtype(m0.dtype),
                                device=eng.device))
            d_det, d_msk = eng._inputs
            for b in range(n):
                # (a read-only ndarray -- a zero-copy view of a received message, wire.py -- is
                # fine here: it is only read)
                d_det[b].copy_(_as_tensor(dets[b]), non_blocking=True)
                d_msk[b].copy_(_as_tensor(masks[b]), non_blocking=True)
            self.d_det, self.d_msk = d_det[:n], d_msk[:n]
        except BaseException:
            eng.lock.release()
            raise

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.eng.lock.release()
        return False

    def meta(self):
        counts, boxes, class_ids, scores = self.eng.fetch_meta()
        return counts, [(boxes[b, :int(counts[b])].copy(), class_ids[b, :int(counts[b])].copy(),
                         scores[b, :int(counts[b])].copy()) for b in range(self.n)]


def _as_tensor(arr):
    import torch
    import warnings

    if arr.flags.writeable:
        return torch.from_numpy(arr)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")     # "non-writable tensors are not supported": read only here
        return torch.from_numpy(arr)


def _download(parts):
    """parts: list of (device uint8 tensor 1-D, nbytes).  One pinned buffer per part from the
    pool, async copies, one synchronisation; returns uint8 ndarrays."""
    import torch

    taken = []
    for d_t, nbytes in parts:
        if nbytes == 0:
            taken.append(None)
            continue
        t, size = _pool.take(nbytes)
        t[:nbytes].copy_(d_t[:nbytes], non_blocking=True)
        taken.append((t, size, nbytes))
    torch.cuda.current_stream().synchronize()
    return [None if x is None else _pool.as_array(*x) for x in taken]


# ----------------------------------------------------------------------------- entry points
def unmold_detections_batch(items):
    """items: sequence of (detections, mrcnn_mask, original_image_shape, image_shape,
    window) with equal R / mask shape / dtypes.  Returns a list of
    (boxes, class_ids, scores, masks) as `unmold_detections` returns them per image (see the
    module docstring for the numerical contract)."""
    if len(items) == 0:
        return []
    with _Staged(items) as st:
        eng = st.eng
        eng.enqueue(st.d_det, st.d_msk)
        counts, metas = st.meta()
        parts = []
        for b in range(st.n):
            k = int(counts[b])
            H, W = st.geoms[b][0], st.geoms[b][1]
            o = int(eng._offsets[b])
            parts.append((eng.d_canvas[o:o + H * W * k], H * W * k))
        arrays = _download(parts)
    out = []
    for b in range(st.n):
        k = int(counts[b])
        H, W = st.geoms[b][0], st.geoms[b][1]
        if k == 0:
            full = np.empty((H, W, 0))            # upstream: np.empty(shape[:2] + (0,))
        else:
            full = arrays[b].reshape(H, W, k).view(np.bool_)
        out.append(metas[b] + (full,))
    return out


def unpack_masks(packed, width):
    """Inverse of the packed transport: uint8 [N, H, ceil(W/8)] -> bool [H, W, N] (the array
    `unmold_detections` returns)."""
    if packed.shape[0] == 0:
        return np.empty((packed.shape[1], width, 0))
    return np.unpackbits(packed, axis=-1, count=width).transpose(1, 2, 0).astype(np.bool_)


def unmold_detections_packed_batch(items, direct=True):
    """EXTENSION (not the reference layout): like `unmold_detections_batch` but the masks come
    back bit-packed, uint8 [N, H, ceil(W/8)] with packed[n, y] == np.packbits(masks[y, :, n]) --
    8x less device -> host traffic; `unpack_masks(packed, W)` restores the reference array.

    direct=True: the expand kernel writes the bits itself (`mrx_mask_expand_packed`; the byte
    canvas is never materialised).  direct=False: byte canvas first, then `mrx_pack_masks`
    (also what mask tiles wider than 30 columns take).  Both give identical bytes."""
    if len(items) == 0:
        return []
    with _Staged(items, canvas=not direct) as st:
        eng = st.eng
        if direct and eng.mw <= 30:
            d_packed, off = eng.enqueue_packed(st.d_det, st.d_msk)
        else:
            eng.plan(st.geoms, canvas=True)
            eng.enqueue(st.d_det, st.d_msk)
            d_packed, off = eng.pack_masks()
        counts, metas = st.meta()
        parts = []
        for b in range(st.n):
            k = int(counts[b])
            H, W = int(st.geoms[b][0]), int(st.geoms[b][1])
            wb = (W + 7) // 8
            parts.append((d_packed[int(off[b]):int(off[b]) + k * H * wb], k * H * wb))
        arrays = _download(parts)
    out = []
    for b in range(st.n):
        k = int(counts[b])
        H, W = int(st.geoms[b][0]), int(st.geoms[b][1])
        wb = (W + 7) // 8
        pk = np.empty((0, H, wb), np.uint8) if k == 0 else arrays[b].reshape(k, H, wb)
        out.append(metas[b] + (pk,))
    return out


def unmold_detections_rle_batch(items):
    """EXTENSION (not the reference layout): like `unmold_detections_batch` but every mask comes
    back as a COCO run-length encoding -- pycocotools' "uncompressed RLE" dict
    {'size': [H, W], 'counts': uint32 array} (column-major runs starting with zeros) -- computed
    on the device straight from the 28x28 tiles; the [H,W,N] masks are never materialised and
    only the run lengths (a few KB per mask) travel to the host.  Decoding a result gives exactly
    the mask `unmold_detections` returns.  Returns a list of (boxes, class_ids, scores, rles)."""
    if len(items) == 0:
        return []
    with _Staged(items, canvas=False) as st:
        eng = st.eng
        eng.enqueue(st.d_det, st.d_msk, expand=False)
        d_runs, off = eng.enqueue_rle()
        counts, metas = st.meta()
        runs = d_runs.cpu().numpy().view(np.uint32)
    out = []
    for b in range(st.n):
        H, W = int(st.geoms[b][0]), int(st.geoms[b][1])
        rles = []
        for k in range(int(counts[b])):
            i = b * eng.R + k
            rles.append({"size": [H, W],
                         "counts": runs[int(off[i]) + i:int(off[i + 1]) + i + 1].copy()})
        out.append(metas[b] + (rles,))
    return out


def unmold_detections_contours_batch(items):
    """The mask outlines of the reference's `visualize.display_instances` (serve.py:160-169),
    not an output of `unmold_detections`: for every kept instance, the contour polygons it
    hands to matplotlib's `Polygon` -- find_contours(mask padded by one zero pixel, 0.5), as
    (x, y) vertices without the padding.  Computed on the device from the tiles (packed expand,
    no byte canvas, then `mrx_contours_*`); only the polygons travel to the host.

    items as for `unmold_detections_batch`.  Returns a list of (boxes, class_ids, scores,
    contours) with contours[k] the list of float64 [K, 2] arrays of instance k, each closed
    (first row == last row), in skimage's order and with its start vertices."""
    if len(items) == 0:
        return []
    with _Staged(items, canvas=False) as st:
        eng = st.eng
        if eng.mw > 30:
            eng.plan(st.geoms, canvas=True)
            eng.enqueue(st.d_det, st.d_msk)
            dc = eng.enqueue_contours(source="canvas")
        else:
            eng.enqueue_packed(st.d_det, st.d_msk)
            dc = eng.enqueue_contours()
        counts, metas = st.meta()
        polys = dc.to_host(counts)
    return [metas[b] + (polys[b],) for b in range(st.n)]


def unmold_overlay_batch(items, images, colors=None, alpha=0.5):
    """`unmold_detections` followed by the mask overlay of `visualize.display_instances`
    (serve.py:147-169) without moving the masks to the host: the [H,W,N] canvases stay on
    the device, only boxes, class ids, scores and the blended uint8 images come back.

    items as for `unmold_detections_batch`; images: the original uint8 HxWx3 images;
    colors: RGB triples (shared list, or one list per image; default: `random_colors(R)`).
    Returns a list of (boxes, class_ids, scores, overlay_uint8)."""
    from . import visualize

    if len(items) == 0:
        return []
    with _Staged(items) as st:
        eng = st.eng
        eng.enqueue(st.d_det, st.d_msk)
        if colors is None:
            colors = visualize.random_colors(eng.R)
        overlays = visualize.composite_batch(eng, images, colors, alpha)
        counts, metas = st.meta()
        host = [o.cpu().numpy() for o in overlays]
    return [metas[b] + (host[b],) for b in range(st.n)]


def unmold_detections(detections, mrcnn_mask, original_image_shape, image_shape, window):
    """Reformat one image's detections from the molded image back to the original image.

    detections: [R, (y1, x1, y2, x2, class_id, score)] normalised coordinates
    mrcnn_mask: [R, mh, mw, num_classes]
    original_image_shape: (H, W, 3) before resizing     image_shape: molded shape
    window: (y1, x1, y2, x2) pixel box of the real image inside the molded image

    Returns boxes [N,4] int32 pixels, class_ids [N] int32, scores [N], masks [H,W,N] bool.
    Boxes, class ids and scores equal the reference's bit for bit; a mask pixel can differ
    only where the reference's float64 resized value is within 1e-6 of the 0.5 threshold.
    """
    return unmold_detections_batch(
        [(detections, mrcnn_mask, original_image_shape, image_shape, window)])[0]
