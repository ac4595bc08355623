"""Device-resident engines over the C ABI (include/mrx.h).

PyTorch tensors are used only as owners of device / pinned-host memory and for streams;
every computation on the path is a libmrx kernel launched through ctypes.

  UnmoldEngine     batched `unmold_detections` (serve.py:147-154): prologue -> class-tile
                   gather -> fused mask expand, all stream-ordered, no host sync
  AnchorGenerator  `get_anchors` (serve.py:105)
  Molder           the body of `preprocess_input` (serve.py:83-107): cv2.resize + resize_image
                   + mold_image
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _native as N


def _torch():
    import torch
    return torch


def _dtype_code(np_dtype):
    dt = np.dtype(np_dtype)
    if dt == np.float32:
        return N.MRX_F32
    if dt == np.float64:
        return N.MRX_F64
    raise TypeError(f"unsupported floating dtype {dt}; use float32 or float64")


def _torch_dtype(np_dtype):
    torch = _torch()
    return {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}[
        np.dtype(np_dtype)]


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def make_geom(original_image_shape, image_shape, window):
    """Pack one image's geometry the way mrx_unmold_prologue expects (8 x int32)."""
    oh, ow = int(original_image_shape[0]), int(original_image_shape[1])
    ih, iw = int(image_shape[0]), int(image_shape[1])
    wy1, wx1, wy2, wx2 = [int(v) for v in window]
    return [oh, ow, ih, iw, wy1, wx1, wy2, wx2]


class UnmoldEngine:
    """Batched, device-resident `unmold_detections`.

    Work buffers for up to `max_batch` images of up to `max_instances` detection rows are
    allocated once; the canvas (bool [H,W,N] per image, N innermost) lives in one device
    buffer with a fixed-capacity slot per image (capacity H*W*R rounded up to 256 B) so
    that nothing on the path depends on a host read of the kept counts.

    Thread safety: an engine is a set of device buffers plus the plan of the last batch; a
    plan -> enqueue -> fetch sequence must not interleave with another thread's.  Callers
    that share an engine hold `engine.lock` (an RLock) across the sequence -- `api_utils`
    does.  `release()` frees the big buffers (canvas, packed output); they are re-allocated
    on the next plan.
    """

    def __init__(self, max_batch, max_instances=100, mask_hw=(28, 28), num_classes=81,
                 det_dtype=np.float32, mask_dtype=np.float32, device=None,
                 chunk_bytes=0, ctas_per_sm=0):
        N.require_cuda()
        torch = _torch()
        self.lib = N.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        self.B = int(max_batch)
        self.R = int(max_instances)
        self.mh, self.mw = int(mask_hw[0]), int(mask_hw[1])
        self.C = int(num_classes)
        self.det_dtype = np.dtype(det_dtype)
        self.mask_dtype = np.dtype(mask_dtype)
        self.chunk_bytes = int(chunk_bytes)
        self.ctas_per_sm = int(ctas_per_sm)
        if self.B < 1 or self.B > N.MRX_MAX_BATCH:
            raise ValueError(f"max_batch must be in [1, {N.MRX_MAX_BATCH}]")
        dev, i32 = self.device, torch.int32
        B, R = self.B, self.R
        self.d_boxes = torch.empty((B, R, 4), dtype=i32, device=dev)
        self.d_class_ids = torch.empty((B, R), dtype=i32, device=dev)
        self.d_scores = torch.empty((B, R), dtype=_torch_dtype(self.det_dtype), device=dev)
        self.d_src_index = torch.empty((B, R), dtype=i32, device=dev)
        self.d_counts = torch.zeros((B,), dtype=i32, device=dev)
        self.d_status = torch.zeros((B,), dtype=i32, device=dev)
        self.d_tiles = torch.empty((B, R, self.mh, self.mw), dtype=torch.float32, device=dev)
        self.d_geom = torch.zeros((B, N.MRX_GEOM_INTS), dtype=i32, device=dev)
        self.d_canvas_off = torch.zeros((B,), dtype=torch.int64, device=dev)
        # scheduler words of the expand kernels: zeroed once here, left zeroed by every launch
        self.d_sched = torch.zeros((N.MRX_SCHED_WORDS,), dtype=i32, device=dev)
        self.d_canvas = None
        self.d_packed = None
        self.d_packed_off = None
        self._packed_off_host = None
        self._geom_host = None
        self._offsets = None
        self._n_images = 0
        self.lock = threading.RLock()
        # pinned staging for fetch_meta (one D2H batch + one synchronisation per call)
        self._h_meta = None

    def release(self):
        """Free the canvas and the packed-output buffer (the work buffers stay)."""
        with self.lock:
            self.d_canvas = None
            self.d_packed = None
            self._geom_host = None
            self._offsets = None
            self._packed_off_host = None
            self._n_images = 0

    # ------------------------------------------------------------------ planning
    def plan(self, geoms, canvas=True):
        """Set the per-image geometry ([n,8] ints, see make_geom) and size the canvas
        (canvas=False: geometry only, for callers that want the packed output alone)."""
        torch = _torch()
        g = np.ascontiguousarray(np.asarray(geoms, dtype=np.int32).reshape(-1, N.MRX_GEOM_INTS))
        n = g.shape[0]
        if n < 1 or n > self.B:
            raise ValueError(f"batch of {n} images does not fit max_batch={self.B}")
        if self._geom_host is not None and self._geom_host.shape == g.shape and \
                np.array_equal(self._geom_host, g) and \
                (not canvas or (self.d_canvas is not None and
                                self.d_canvas.numel() >= int(self._offsets[-1]))):
            return      # (a plan made with canvas=False may have left a smaller canvas behind)
        if (g[:, :4] < 2).any():
            raise ValueError("image sides must be >= 2")
        if (g[:, 0].astype(np.int64) * g[:, 1] > (1 << 30)).any():
            raise ValueError("canvas larger than 2^30 pixels is not supported")
        if (g[:, 0].astype(np.int64) * g[:, 1] * self.R >= (1 << 31) - (1 << 20)).any():
            raise ValueError("a canvas of H*W*R >= 2^31 bytes is not supported (32-bit chunk math)")
        cap = (g[:, 0].astype(np.int64) * g[:, 1].astype(np.int64) * self.R + 255) // 256 * 256
        off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(cap, out=off[1:])
        total = int(off[-1])
        if canvas and (self.d_canvas is None or self.d_canvas.numel() < total):
            self.d_canvas = None
            self.d_canvas = torch.empty((total,), dtype=torch.uint8, device=self.device)
        self.d_geom[:n].copy_(torch.from_numpy(g))
        self.d_canvas_off[:n].copy_(torch.from_numpy(off[:n].copy()))
        self._geom_host = g
        self._offsets = off
        self._n_images = n
        self._packed_off_host = None

    # ------------------------------------------------------------------ launch
    def enqueue(self, d_detections, d_mrcnn_mask, stream=None, expand=True):
        """Enqueue the three kernels for the planned batch on `stream` (no host sync).
        d_detections [n,R,6] and d_mrcnn_mask [n,R,mh,mw,C] are device tensors of the
        dtypes given at construction (d_mrcnn_mask may also be PINNED HOST memory: the class
        gather then reads the wanted elements over PCIe instead of the whole tensor being
        copied first).  expand=False stops after the class-tile gather."""
        n = self._n_images
        if n == 0:
            raise RuntimeError("call plan() first")
        torch = _torch()
        if tuple(d_detections.shape) != (n, self.R, 6) or \
                d_detections.dtype != _torch_dtype(self.det_dtype):
            raise ValueError(f"detections must be {(n, self.R, 6)} {self.det_dtype}, got "
                             f"{tuple(d_detections.shape)} {d_detections.dtype}")
        if tuple(d_mrcnn_mask.shape) != (n, self.R, self.mh, self.mw, self.C) or \
                d_mrcnn_mask.dtype != _torch_dtype(self.mask_dtype):
            raise ValueError(f"mrcnn_mask must be {(n, self.R, self.mh, self.mw, self.C)} "
                             f"{self.mask_dtype}, got {tuple(d_mrcnn_mask.shape)} "
                             f"{d_mrcnn_mask.dtype}")
        if not (d_detections.is_contiguous() and d_mrcnn_mask.is_contiguous()):
            raise ValueError("inputs must be contiguous")
        st = N.stream_ptr(stream)
        # steps 1-6 and the class-tile gather in one launch; tiles are stored by detection row
        # and found through d_src_index by the expand kernels
        N.check(self.lib.mrx_unmold_prepare(
            _ptr(d_detections), _dtype_code(self.det_dtype), _ptr(d_mrcnn_mask),
            _dtype_code(self.mask_dtype), n, self.R, self.mh, self.mw, self.C,
            _ptr(self.d_geom), _ptr(self.d_boxes), _ptr(self.d_class_ids), _ptr(self.d_scores),
            _ptr(self.d_src_index), _ptr(self.d_counts),
            _ptr(self.d_status), _ptr(self.d_tiles), _ptr(self.d_sched), st),
            "mrx_unmold_prepare")
        if expand:
            self.enqueue_expand(stream)

    def enqueue_expand(self, stream=None, canvas_ptr=None, images=None):
        """Only the mask-expand kernel (boxes / tiles / counts already on the device).
        canvas_ptr: write the canvases at another base address with the planned offsets
        (an integer device address, e.g. rank 0's receive buffer mapped with mrx_peer_open).
        images=(b0, b1): only that range of the planned batch (one launch per chunk lets the
        gather of a finished chunk overlap the next one)."""
        b0, b1 = (0, self._n_images) if images is None else images
        if b1 <= b0:
            return
        base = _ptr(self.d_canvas) if canvas_ptr is None else C.c_void_p(int(canvas_ptr))
        N.check(self.lib.mrx_mask_expand(
            _ptr(self.d_tiles[b0:]), _ptr(self.d_src_index[b0:]), _ptr(self.d_boxes[b0:]),
            _ptr(self.d_counts[b0:]), _ptr(self.d_geom[b0:]),
            _ptr(self.d_canvas_off[b0:]), base, b1 - b0, self.R, self.mh, self.mw,
            self.chunk_bytes, self.ctas_per_sm, _ptr(self.d_sched),
            N.stream_ptr(stream)), "mrx_mask_expand")

    def enqueue_expand_values(self, d_values, stream=None):
        """Parity instrumentation: the same kernel (second instantiation of its template) also
        stores every pre-threshold sample into d_values (float32, indexed like the canvas)."""
        n = self._n_images
        if d_values.dtype != _torch().float32 or d_values.numel() < int(self._offsets[n]):
            raise ValueError("d_values must be float32 with one element per canvas byte")
        N.check(self.lib.mrx_mask_expand_values(
            _ptr(self.d_tiles), _ptr(self.d_src_index), _ptr(self.d_boxes), _ptr(self.d_counts),
            _ptr(self.d_geom), _ptr(self.d_canvas_off), _ptr(self.d_canvas), _ptr(d_values),
            n, self.R, self.mh, self.mw, _ptr(self.d_sched), N.stream_ptr(stream)),
            "mrx_mask_expand_values")

    # ------------------------------------------------------------------ packed output
    def packed_layout(self):
        """(offsets int64 [n+1], total bytes) of the packed output of the planned batch: image b
        occupies [off[b], off[b+1]) as uint8 [R, H_b, ceil(W_b/8)] (first N_b planes valid)."""
        n = self._n_images
        if n == 0:
            raise RuntimeError("plan() first")
        if self._packed_off_host is None:
            g = self._geom_host
            wb = (g[:, 1].astype(np.int64) + 7) // 8
            sizes = (g[:, 0].astype(np.int64) * wb * self.R + 15) // 16 * 16
            off = np.zeros(n + 1, dtype=np.int64)
            np.cumsum(sizes, out=off[1:])
            self._packed_off_host = off
            self.d_packed_off = _torch().from_numpy(off[:n].copy()).to(self.device)
        return self._packed_off_host, int(self._packed_off_host[-1])

    def _packed_buffer(self):
        torch = _torch()
        off, total = self.packed_layout()
        if self.d_packed is None or self.d_packed.numel() < total:
            self.d_packed = None
            self.d_packed = torch.empty((total,), dtype=torch.uint8, device=self.device)
        return off

    def enqueue_expand_packed(self, stream=None, packed_ptr=None, images=None):
        """EXTENSION (not the reference layout): the expand step writing bit-packed masks
        directly (mrx_mask_expand_packed): packed[n, y] == np.packbits(masks[y, :, n]).
        Returns (d_packed, offsets).  packed_ptr: another base address (peer memory);
        images=(b0, b1): only that range of the planned batch."""
        b0, b1 = (0, self._n_images) if images is None else images
        if packed_ptr is None:
            off = self._packed_buffer()
            base = _ptr(self.d_packed)
        else:
            off, _ = self.packed_layout()
            base = C.c_void_p(int(packed_ptr))
        g = self._geom_host
        if b1 > b0:
            N.check(self.lib.mrx_mask_expand_packed(
                _ptr(self.d_tiles[b0:]), _ptr(self.d_src_index[b0:]), _ptr(self.d_boxes[b0:]),
                _ptr(self.d_counts[b0:]),
                _ptr(self.d_geom[b0:]), _ptr(self.d_packed_off[b0:]), base, b1 - b0, self.R,
                self.mh, self.mw, int(g[:, 1].max()), _ptr(self.d_sched), N.stream_ptr(stream)),
                "mrx_mask_expand_packed")
        return self.d_packed, off

    def enqueue_packed(self, d_detections, d_mrcnn_mask, stream=None):
        """prologue -> class-tile gather -> packed expand (no byte canvas is written)."""
        self.enqueue(d_detections, d_mrcnn_mask, stream, expand=False)
        return self.enqueue_expand_packed(stream)

    # ------------------------------------------------------------------ results
    def canvas_bytes(self, counts):
        """Algorithmic canvas bytes for kept counts (sum H*W*N)."""
        g = self._geom_host
        return int((g[:, 0].astype(np.int64) * g[:, 1] * np.asarray(counts, np.int64)).sum())

    def canvas_view(self, b, n_kept):
        """uint8 device view [H, W, n_kept] of image b's slot (values 0/1)."""
        g = self._geom_host[b]
        H, W = int(g[0]), int(g[1])
        o = int(self._offsets[b])
        return self.d_canvas[o:o + H * W * n_kept].view(H, W, n_kept)

    def enqueue_rle(self, stream=None):
        """EXTENSION: COCO run-length encodings of the planned batch's masks, from the tiles
        (after `enqueue(..., expand=False)`; no mask is materialised).  Synchronises once to
        size the output.  Returns (d_run_lengths uint32 tensor, inst_off int64 ndarray [n*R+1]):
        instance i = b*R + k owns d_run_lengths[inst_off[i] + i : inst_off[i+1] + i + 1]."""
        torch = _torch()
        n = self._n_images
        g = self._geom_host
        max_w = int(g[:, 1].max())
        dev = self.device
        d_col = torch.empty((n * self.R * max_w,), dtype=torch.int32, device=dev)
        d_off = torch.empty((n * self.R + 1,), dtype=torch.int64, device=dev)
        st = N.stream_ptr(stream)
        args = (_ptr(self.d_tiles), _ptr(self.d_src_index), _ptr(self.d_boxes), _ptr(self.d_counts),
                _ptr(self.d_geom), _ptr(d_col), _ptr(d_off))
        N.check(self.lib.mrx_rle_count(*args, n, self.R, self.mh, self.mw, max_w, st),
                "mrx_rle_count")
        off = d_off.cpu().numpy()          # the one synchronisation: how many runs there are
        total = int(off[-1])
        d_pos = torch.empty((max(total, 1),), dtype=torch.int32, device=dev)
        d_runs = torch.empty((total + n * self.R,), dtype=torch.int32, device=dev)
        N.check(self.lib.mrx_rle_write(*args, _ptr(d_pos), _ptr(d_runs), n, self.R, self.mh,
                                       self.mw, max_w, st), "mrx_rle_write")
        return d_runs, off

    def enqueue_contours(self, stream=None, source="packed"):
        """The contour polygons `display_instances` traces for every mask of the planned batch
        (mrx_contours_count / _write), from the engine's bit-packed masks.  source="packed": the
        packed buffer is already written (`enqueue_expand_packed` / `pack_masks`);
        source="canvas": bit-pack the byte canvas first (`pack_masks`).  Synchronises once, to
        size the output.  Returns a `DeviceContours`."""
        if source not in ("packed", "canvas"):
            raise ValueError("source: 'packed' or 'canvas'")
        if source == "canvas":
            self.pack_masks(stream)
        if self.d_packed is None:
            raise RuntimeError("no packed masks: run enqueue_expand_packed or pack_masks first")
        n = self._n_images
        g = self._geom_host
        return contours_device(self.lib, self.device, self.d_packed, self.d_packed_off,
                               self.d_boxes, self.d_counts, self.d_geom, n, self.R,
                               int(g[:, 0].max()), int(g[:, 1].max()), stream)

    def pack_masks(self, stream=None):
        """EXTENSION: bit-pack the byte canvases already written for the planned batch
        (mrx_pack_masks; same output layout as `enqueue_expand_packed`).  Returns
        (d_packed, offsets)."""
        n = self._n_images
        off = self._packed_buffer()
        g = self._geom_host
        N.check(self.lib.mrx_pack_masks(
            _ptr(self.d_canvas), _ptr(self.d_canvas_off), _ptr(self.d_counts), _ptr(self.d_geom),
            _ptr(self.d_packed), _ptr(self.d_packed_off), n, self.R,
            int(g[:, 0].max()), int(g[:, 1].max()), N.stream_ptr(stream)), "mrx_pack_masks")
        return self.d_packed, off

    def fetch_meta(self, stream=None):
        """Copy counts/status/boxes/class_ids/scores of the planned batch to the host
        (one batch of async copies into cached pinned memory, one synchronisation).
        Raises like numpy would on bad inputs.  The returned arrays are views of the
        staging buffers: valid until the next fetch_meta of this engine."""
        torch = _torch()
        n = self._n_images
        if self._h_meta is None:
            B, R = self.B, self.R
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()  # noqa: E731
            self._h_meta = (pin((B,), torch.int32), pin((B,), torch.int32),
                            pin((B, R, 4), torch.int32), pin((B, R), torch.int32),
                            pin((B, R), _torch_dtype(self.det_dtype)))
        hc, hs, hb, hk, hsc = self._h_meta
        st = stream or torch.cuda.current_stream(self.device)
        with torch.cuda.stream(st):
            hc[:n].copy_(self.d_counts[:n], non_blocking=True)
            hs[:n].copy_(self.d_status[:n], non_blocking=True)
            hb[:n].copy_(self.d_boxes[:n], non_blocking=True)
            hk[:n].copy_(self.d_class_ids[:n], non_blocking=True)
            hsc[:n].copy_(self.d_scores[:n], non_blocking=True)
        st.synchronize()
        counts, status = hc[:n].numpy(), hs[:n].numpy()
        if (status & N.MRX_ST_CLASS_RANGE).any():
            b = int(np.nonzero(status & N.MRX_ST_CLASS_RANGE)[0][0])
            raise IndexError(f"image {b}: class id out of bounds for axis 3 with size {self.C}")
        if (status & N.MRX_ST_BOX_RANGE).any():
            b = int(np.nonzero(status & N.MRX_ST_BOX_RANGE)[0][0])
            raise ValueError(f"image {b}: a detection box falls outside the original image; "
                             "the reference's mask paste cannot broadcast it")
        return counts, hb[:n].numpy(), hk[:n].numpy(), hsc[:n].numpy()


class DeviceContours:
    """Output of mrx_contours_write for B images of R instance slots (layout: include/mrx.h).
    seg_off: int64 ndarray [B*R+1] (host copy of the segment offsets); vertices float32
    [T + T/4, 2], contour_len int32 [T/4], inst_contours int32 [B*R] (CUDA tensors)."""

    def __init__(self, seg_off, vertices, contour_len, inst_contours, R):
        self.seg_off = seg_off
        self.vertices = vertices
        self.contour_len = contour_len
        self.inst_contours = inst_contours
        self.R = R

    def to_host(self, counts):
        """Download (one synchronisation) and split: for image b, a list of counts[b] lists of
        float64 [K, 2] (x, y) arrays -- the polygons of each instance, each closed."""
        torch = _torch()
        st = torch.cuda.current_stream()
        h = [t.to("cpu", non_blocking=True) for t in (self.vertices, self.contour_len,
                                                       self.inst_contours)]
        st.synchronize()
        vert, lens, ncont = (t.numpy() for t in h)
        vert = vert.reshape(-1, 2)
        out = []
        for b, n in enumerate(counts):
            per_image = []
            for k in range(int(n)):
                i = b * self.R + k
                o = int(self.seg_off[i])
                ls = lens[o // 4:o // 4 + int(ncont[i])]
                ends = np.cumsum(ls)
                base = o + o // 4
                per_image.append([vert[base + e - l:base + e].astype(np.float64)
                                  for l, e in zip(ls.tolist(), ends.tolist())])
            out.append(per_image)
        return out


def contours_device(lib, device, d_packed, d_packed_off, d_boxes, d_counts, d_geom, B, R,
                    max_h, max_w, stream=None):
    """mrx_contours_count, one host read of the segment offsets, mrx_contours_write.  Inputs
    are device tensors in the layouts of include/mrx.h; returns a `DeviceContours`."""
    torch = _torch()
    st = N.stream_ptr(stream)
    d_rows = torch.empty((B * R * (max_h + 1),), dtype=torch.int32, device=device)
    d_off = torch.empty((B * R + 1,), dtype=torch.int64, device=device)
    common = (_ptr(d_packed), _ptr(d_packed_off), _ptr(d_boxes), _ptr(d_counts), _ptr(d_geom),
              _ptr(d_rows), _ptr(d_off))
    N.check(lib.mrx_contours_count(*common, B, R, max_h, max_w, st), "mrx_contours_count")
    off = d_off.cpu().numpy()              # the one synchronisation: how many segments there are
    T = int(off[-1])
    d_scratch = torch.empty((max(2 * T, 1),), dtype=torch.int32, device=device)
    d_vert = torch.empty((T + T // 4, 2), dtype=torch.float32, device=device)
    d_len = torch.empty((max(T // 4, 1),), dtype=torch.int32, device=device)
    d_ncont = torch.empty((B * R,), dtype=torch.int32, device=device)
    N.check(lib.mrx_contours_write(*common, _ptr(d_scratch), _ptr(d_vert), _ptr(d_len),
                                   _ptr(d_ncont), C.c_longlong(T), B, R, max_h, max_w, st),
            "mrx_contours_write")
    return DeviceContours(off, d_vert, d_len[:T // 4], d_ncont, R)


class AnchorGenerator:
    """`get_anchors` on the device; memoised by image shape like upstream's method."""

    def __init__(self, config, device=None):
        N.require_cuda()
        torch = _torch()
        self.lib = N.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        self.scales = [float(s) for s in config.RPN_ANCHOR_SCALES]
        self.ratios = [float(r) for r in config.RPN_ANCHOR_RATIOS]
        self.strides = [int(s) for s in config.BACKBONE_STRIDES]
        self.anchor_stride = int(config.RPN_ANCHOR_STRIDE)
        if len(self.scales) != len(self.strides):
            raise ValueError("RPN_ANCHOR_SCALES and BACKBONE_STRIDES must have equal length")
        self._cache = {}

    def count(self, image_shape):
        out = C.c_longlong(0)
        N.check(self.lib.mrx_anchor_count(
            int(image_shape[0]), int(image_shape[1]), N.int_array(self.strides),
            len(self.strides), len(self.ratios), self.anchor_stride, C.byref(out)),
            "mrx_anchor_count")
        return int(out.value)

    def generate_device(self, image_shape, out=None, stream=None):
        """[A,4] float32 device tensor (not cached)."""
        torch = _torch()
        A = self.count(image_shape)
        if out is None:
            out = torch.empty((A, 4), dtype=torch.float32, device=self.device)
        N.check(self.lib.mrx_anchors(
            _ptr(out), int(image_shape[0]), int(image_shape[1]),
            N.double_array(self.scales), N.double_array(self.ratios),
            N.int_array(self.strides), len(self.strides), len(self.ratios),
            self.anchor_stride, N.stream_ptr(stream)), "mrx_anchors")
        return out

    def get_anchors(self, image_shape):
        key = tuple(int(v) for v in image_shape)
        if key not in self._cache:
            self._cache[key] = self.generate_device(image_shape).cpu().numpy()
        return self._cache[key]


def resize_image_geometry(h, w, min_dim, max_dim, min_scale, mode):
    """Host-side scalar logic of upstream utils.resize_image (serve.py:91-97): returns
    (new_h, new_w, top, left, out_h, out_w, window, scale, padding).  `crop` mode is
    random/training-only and not part of serving."""
    scale = 1
    if mode == "none":
        return h, w, 0, 0, h, w, (0, 0, h, w), 1, [(0, 0), (0, 0), (0, 0)]
    if min_dim:
        scale = max(1, min_dim / min(h, w))
    if min_scale and scale < min_scale:
        scale = min_scale
    if max_dim and mode == "square":
        image_max = max(h, w)
        if round(image_max * scale) > max_dim:
            scale = max_dim / image_max
    nh, nw = (round(h * scale), round(w * scale)) if scale != 1 else (h, w)
    if mode == "square":
        top = (max_dim - nh) // 2
        bottom = max_dim - nh - top
        left = (max_dim - nw) // 2
        right = max_dim - nw - left
        out_h, out_w = max_dim, max_dim
    elif mode == "pad64":
        assert min_dim % 64 == 0, "Minimum dimension must be a multiple of 64"
        if nh % 64 > 0:
            max_h = nh - (nh % 64) + 64
            top = (max_h - nh) // 2
            bottom = max_h - nh - top
        else:
            top = bottom = 0
        if nw % 64 > 0:
            max_w = nw - (nw % 64) + 64
            left = (max_w - nw) // 2
            right = max_w - nw - left
        else:
            left = right = 0
        out_h, out_w = nh + top + bottom, nw + left + right
    else:
        raise Exception("Mode {} not supported".format(mode))
    if top < 0 or left < 0:
        raise ValueError("image larger than IMAGE_MAX_DIM after scaling")
    padding = [(top, bottom), (left, right), (0, 0)]
    window = (top, left, nh + top, nw + left)
    return nh, nw, top, left, out_h, out_w, window, scale, padding


class Molder:
    """cv2.resize + resize_image + mold_image on the device (serve.py:88-98)."""

    def __init__(self, config, device=None):
        N.require_cuda()
        torch = _torch()
        self.lib = N.load()
        self.config = config
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)

    def cv2_resize_device(self, d_img, size_hw, stream=None):
        torch = _torch()
        sh, sw = int(d_img.shape[0]), int(d_img.shape[1])
        dh, dw = int(size_hw[0]), int(size_hw[1])
        out = torch.empty((dh, dw, 3), dtype=torch.uint8, device=self.device)
        N.check(self.lib.mrx_cv2_resize_u8c3(_ptr(d_img), sh, sw, _ptr(out), dh, dw,
                                             N.stream_ptr(stream)), "mrx_cv2_resize_u8c3")
        return out

    def mold_device(self, d_img, out_dtype=np.float32, want_u8=False, stream=None):
        """resize_image + mold_image for a uint8 HxWx3 device image.
        Returns (molded, molded_u8|None, window, scale, padding)."""
        torch = _torch()
        cfg = self.config
        h, w = int(d_img.shape[0]), int(d_img.shape[1])
        nh, nw, top, left, oh, ow, window, scale, padding = resize_image_geometry(
            h, w, cfg.IMAGE_MIN_DIM, cfg.IMAGE_MAX_DIM, cfg.IMAGE_MIN_SCALE,
            cfg.IMAGE_RESIZE_MODE)
        out = torch.empty((oh, ow, 3), dtype=_torch_dtype(out_dtype), device=self.device)
        u8 = torch.empty((oh, ow, 3), dtype=torch.uint8, device=self.device) if want_u8 \
            else None
        mean = [float(v) for v in np.asarray(cfg.MEAN_PIXEL, dtype=np.float64)]
        N.check(self.lib.mrx_mold_image(
            _ptr(d_img), h, w, nh, nw, top, left, oh, ow, N.double_array(mean),
            _dtype_code(out_dtype), _ptr(out),
            _ptr(u8) if u8 is not None else C.c_void_p(0), N.stream_ptr(stream)),
            "mrx_mold_image")
        return out, u8, window, scale, padding


    # ------------------------------------------------------------------ batched (one launch each)
    def cv2_resize_batch_device(self, images, size_hw, stream=None):
        """`cv2.resize(img, (S, S))` for a list of uint8 HxWx3 NumPy images of ANY sizes in one
        launch: one pinned staging buffer, one H2D copy.  Returns uint8 [B, dh, dw, 3] on the
        device."""
        torch = _torch()
        B = len(images)
        dh, dw = int(size_hw[0]), int(size_hw[1])
        sizes = [int(im.shape[0]) * int(im.shape[1]) * 3 for im in images]
        off = np.zeros(B + 1, dtype=np.int64)
        np.cumsum((np.asarray(sizes, dtype=np.int64) + 15) // 16 * 16, out=off[1:])
        total = int(off[-1])
        if getattr(self, "_h_stage", None) is None or self._h_stage.numel() < total:
            self._h_stage = torch.empty((total,), dtype=torch.uint8).pin_memory()
        hs = self._h_stage.numpy()
        hw = np.empty((B, 2), dtype=np.int32)
        for b, im in enumerate(images):
            hs[int(off[b]):int(off[b]) + sizes[b]] = np.ascontiguousarray(im).reshape(-1)
            hw[b] = im.shape[:2]
        d_src = self._h_stage[:total].to(self.device, non_blocking=True)
        d_off = torch.from_numpy(off[:B].copy()).to(self.device)
        d_hw = torch.from_numpy(hw).to(self.device)
        out = torch.empty((B, dh, dw, 3), dtype=torch.uint8, device=self.device)
        N.check(self.lib.mrx_cv2_resize_u8c3_batch(
            _ptr(d_src), _ptr(d_off), _ptr(d_hw), _ptr(out), B, dh, dw, N.stream_ptr(stream)),
            "mrx_cv2_resize_u8c3_batch")
        return out

    def mold_batch_device(self, d_imgs, out_dtype=np.float32, stream=None):
        """resize_image + mold_image for uint8 [B,h,w,3] device images of one size, one launch.
        Returns (molded [B,oh,ow,3], window, scale, padding)."""
        torch = _torch()
        cfg = self.config
        B, h, w = int(d_imgs.shape[0]), int(d_imgs.shape[1]), int(d_imgs.shape[2])
        nh, nw, top, left, oh, ow, window, scale, padding = resize_image_geometry(
            h, w, cfg.IMAGE_MIN_DIM, cfg.IMAGE_MAX_DIM, cfg.IMAGE_MIN_SCALE,
            cfg.IMAGE_RESIZE_MODE)
        out = torch.empty((B, oh, ow, 3), dtype=_torch_dtype(out_dtype), device=self.device)
        mean = [float(v) for v in np.asarray(cfg.MEAN_PIXEL, dtype=np.float64)]
        N.check(self.lib.mrx_mold_image_batch(
            _ptr(d_imgs), B, h, w, nh, nw, top, left, oh, ow, N.double_array(mean),
            _dtype_code(out_dtype), _ptr(out), C.c_void_p(0), N.stream_ptr(stream)),
            "mrx_mold_image_batch")
        return out, window, scale, padding


class StreamingUnmolder:
    """Host-buffer pipeline around UnmoldEngine for a stream of equally-shaped batches:
    the H2D copy of batch k+1 (own stream, double-buffered device inputs) overlaps the D2H
    copy of batch k's masks (PCIe is full duplex); results land in double-buffered pinned
    host memory and are valid after `wait(k)`.

        sm = StreamingUnmolder(engine, geoms)
        for k, (h_det, h_msk) in enumerate(batches):      # pinned [n,R,6] / [n,R,mh,mw,C]
            sm.submit(h_det, h_msk)
            if k: counts, boxes, masks = sm.wait(k - 1)

    packed=True (EXTENSION, not the reference layout): the expand kernel writes bit-packed masks
    (`mrx_mask_expand_packed`) and only those travel back: 8x fewer D2H bytes; the host buffer
    then holds, per image, uint8 [R, H, ceil(W/8)] at `engine.packed_layout()` offsets.

    mask_upload="zero_copy": `mrcnn_mask` is not copied to the device at all -- the class-tile
    gather kernel reads the 1/C of it that is needed straight from the pinned host buffer over
    PCIe (detections are still copied: 2.4 KB per image)."""

    def __init__(self, engine, geoms, packed=False, mask_upload="copy"):
        torch = _torch()
        if mask_upload not in ("copy", "zero_copy"):
            raise ValueError("mask_upload: 'copy' or 'zero_copy'")
        self.eng = engine
        self.packed = bool(packed)
        self.zero_copy = mask_upload == "zero_copy"
        engine.plan(geoms, canvas=False)       # the outputs live here, double-buffered
        n = engine._n_images
        self.n = n
        dev = engine.device
        det_t, msk_t = _torch_dtype(engine.det_dtype), _torch_dtype(engine.mask_dtype)
        self.d_det = [torch.empty((n, engine.R, 6), dtype=det_t, device=dev) for _ in range(2)]
        self.d_msk = None if self.zero_copy else [
            torch.empty((n, engine.R, engine.mh, engine.mw, engine.C), dtype=msk_t, device=dev)
            for _ in range(2)]
        self.total = engine.packed_layout()[1] if self.packed else int(engine._offsets[n])
        self.d_out = [torch.empty((self.total,), dtype=torch.uint8, device=dev) for _ in range(2)]
        self.h_out = [torch.empty((self.total,), dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.h_counts = [torch.empty((n,), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.h_boxes = [torch.empty((n, engine.R, 4), dtype=torch.int32).pin_memory()
                        for _ in range(2)]
        # three streams: inputs up, kernels, results down -- batch k's download overlaps batch
        # k+1's kernels and batch k+2's upload (PCIe is full duplex)
        self.in_stream = torch.cuda.Stream(device=dev)
        self.out_stream = torch.cuda.Stream(device=dev)
        self.main_stream = torch.cuda.current_stream(dev)
        self.h2d_done = [torch.cuda.Event() for _ in range(2)]
        self.in_free = [torch.cuda.Event() for _ in range(2)]
        self.out_ready = [torch.cuda.Event() for _ in range(2)]
        self.out_free = [torch.cuda.Event() for _ in range(2)]
        self.out_done = {}
        self.k = 0
        msk_bytes = n * engine.R * engine.mh * engine.mw * engine.C * engine.mask_dtype.itemsize
        self.h2d_bytes = self.d_det[0].numel() * self.d_det[0].element_size() + \
            (0 if self.zero_copy else msk_bytes)
        # zero copy: the gather kernel pulls one 32-byte sector per wanted element over PCIe
        self.pcie_read_bytes = n * engine.R * engine.mh * engine.mw * 32 if self.zero_copy else 0
        self.d2h_bytes = self.total + 4 * (n + 4 * n * engine.R)

    def submit(self, h_det, h_msk):
        """Queue one batch (pinned host tensors).  The host buffers of batch k are reused by
        batch k+2: consume `wait(k)`'s result before submitting batch k+2."""
        torch = _torch()
        k, i = self.k, self.k % 2
        eng = self.eng
        if self.zero_copy and not h_msk.is_pinned():
            raise ValueError("zero_copy needs the mask tensor in pinned host memory")
        with torch.cuda.stream(self.in_stream):
            if k >= 2:
                self.in_stream.wait_event(self.in_free[i])     # kernels of batch k-2 read d_*[i]
            self.d_det[i].copy_(h_det, non_blocking=True)
            if not self.zero_copy:
                self.d_msk[i].copy_(h_msk, non_blocking=True)
            self.h2d_done[i].record(self.in_stream)
        ms = self.main_stream
        ms.wait_event(self.h2d_done[i])
        if k >= 2:
            ms.wait_event(self.out_free[i])                    # download of batch k-2 read d_out[i]
        msk = h_msk if self.zero_copy else self.d_msk[i]
        eng.enqueue(self.d_det[i], msk, ms, expand=False)
        if self.packed:
            eng.enqueue_expand_packed(ms, packed_ptr=self.d_out[i].data_ptr())
        else:
            eng.enqueue_expand(ms, canvas_ptr=self.d_out[i].data_ptr())
        self.in_free[i].record(ms)
        # counts / boxes are single-buffered in the engine: copy them (50 KB) before the next
        # batch's prologue overwrites them, on the kernel stream
        with torch.cuda.stream(ms):
            self.h_counts[i].copy_(eng.d_counts[:self.n], non_blocking=True)
            self.h_boxes[i].copy_(eng.d_boxes[:self.n], non_blocking=True)
        self.out_ready[i].record(ms)
        with torch.cuda.stream(self.out_stream):
            self.out_stream.wait_event(self.out_ready[i])
            self.h_out[i].copy_(self.d_out[i], non_blocking=True)
            self.out_free[i].record(self.out_stream)
            ev = torch.cuda.Event()
            ev.record(self.out_stream)
        self.out_done[k] = ev
        self.k += 1
        return k

    def wait(self, k):
        """Block until batch k's results are in pinned host memory; returns
        (counts [n] int32, boxes [n,R,4] int32, output bytes uint8) as torch CPU tensors."""
        self.out_done.pop(k).synchronize()
        i = k % 2
        return self.h_counts[i], self.h_boxes[i], self.h_out[i]
