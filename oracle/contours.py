"""Contour polygons of visualize.display_instances (serve.py:160-169).  TEST INFRASTRUCTURE.

[UPSTREAM skimage] measure.find_contours (scikit-image >= 0.19), PARITY UNPINNED: scikit-image
is not importable here, so this module restates its marching-squares segment generation
(`_find_contours_cy.pyx`) and its contour assembly (`_find_contours.py`) for the defaults
fully_connected='low', positive_orientation='low', and the outline step of display_instances
built on them.  Same rules as the rest of oracle/ (see oracle/__init__.py): only tests/ and the
measurement tools import it; the product package never does.
"""
from __future__ import annotations

from collections import deque

import numpy as np


# Segment table (from, to) per case code ul + 2 ur + 4 ll + 8 lr of cell (r, c) with
# ul = image[r, c], ur = image[r, c+1], ll = image[r+1, c], lr = image[r+1, c+1]:
_SEGMENTS = {
    1: (("top", "left"),), 2: (("right", "top"),), 3: (("right", "left"),),
    4: (("left", "bottom"),), 5: (("top", "bottom"),),
    6: (("right", "top"), ("left", "bottom")), 7: (("right", "bottom"),),
    8: (("bottom", "right"),), 9: (("top", "left"), ("bottom", "right")),
    10: (("bottom", "top"),), 11: (("bottom", "left"),), 12: (("left", "right"),),
    13: (("top", "right"),), 14: (("left", "top"),),
}


def _get_contour_segments(image, level):
    """[UPSTREAM skimage _get_contour_segments] Marching squares: the directed segments of every
    2x2 cell, cells in row-major order, a cell's segments in table order.  Low values lie on the
    left of each segment in (row, col); that fixes the direction of every non-saddle case, and
    fully_connected='low' (high diagonal pixels not connected) fixes the pairing of the saddles
    6 and 9.  The order of the two segments inside a saddle cell is the one detail the
    documented behaviour does not force; it can only move a contour's start point or change the
    order of contours.  Edge points interpolate linearly, (level - a) / (b - a) along the edge
    (0 when a == b).

    Vectorised over the cells, but only the bounding rectangle of the pixels above `level`,
    grown by one, is scanned: every other cell is case 0.  Returns a list of
    ((r0, c0), (r1, c1)) float tuples in skimage's emission order."""
    image = np.asarray(image, dtype=np.float64)
    high = image > level
    if image.shape[0] < 2 or image.shape[1] < 2 or not high.any():
        return []
    rows = np.flatnonzero(high.any(axis=1))
    cols = np.flatnonzero(high.any(axis=0))
    r_lo, r_hi = max(rows[0] - 1, 0), min(rows[-1] + 1, image.shape[0] - 1)
    c_lo, c_hi = max(cols[0] - 1, 0), min(cols[-1] + 1, image.shape[1] - 1)
    sub = image[r_lo:r_hi + 1, c_lo:c_hi + 1]
    hs = sub > level
    case = (hs[:-1, :-1] * 1 + hs[:-1, 1:] * 2 + hs[1:, :-1] * 4 + hs[1:, 1:] * 8)
    rr, cc = np.nonzero((case != 0) & (case != 15))      # row-major, like the scan
    cases = case[rr, cc]
    ul, ur = sub[rr, cc], sub[rr, cc + 1]
    ll, lr = sub[rr + 1, cc], sub[rr + 1, cc + 1]

    def frac(a, b):
        d = b - a
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(d == 0, 0.0, (level - a) / np.where(d == 0, 1.0, d))

    r0 = (rr + r_lo).astype(np.float64)
    c0 = (cc + c_lo).astype(np.float64)
    pts = {"top": (r0, c0 + frac(ul, ur)), "bottom": (r0 + 1, c0 + frac(ll, lr)),
           "left": (r0 + frac(ul, ll), c0), "right": (r0 + frac(ur, lr), c0 + 1)}
    pts = {k: list(zip(v[0].tolist(), v[1].tolist())) for k, v in pts.items()}
    segments = []
    for i, cs in enumerate(cases.tolist()):
        for a, b in _SEGMENTS[cs]:
            segments.append((pts[a][i], pts[b][i]))
    return segments


def _assemble_contours(segments):
    """[UPSTREAM skimage _assemble_contours] Link the segments into contours, literally: the
    `starts` / `ends` dicts map an open contour's first / last point to (deque, number); a
    segment extends, closes or joins contours, and a join keeps the lower contour number, so
    the contours come out ordered by their first segment."""
    current_index = 0
    contours = {}
    starts = {}
    ends = {}
    for from_point, to_point in segments:
        # ignore degenerate segments
        if from_point == to_point:
            continue
        tail, tail_num = starts.pop(to_point, (None, None))
        head, head_num = ends.pop(from_point, (None, None))
        if tail is not None and head is not None:
            if tail is head:
                # close a contour: add the end point
                head.append(to_point)
            else:
                # join two distinct contours, keeping the one created first
                if tail_num > head_num:
                    head.extend(tail)
                    contours.pop(tail_num, None)
                    starts[head[0]] = (head, head_num)
                    ends[head[-1]] = (head, head_num)
                else:
                    tail.extendleft(reversed(head))
                    starts.pop(head[0], None)       # head[0] can be == to_point
                    contours.pop(head_num, None)
                    starts[tail[0]] = (tail, tail_num)
                    ends[tail[-1]] = (tail, tail_num)
        elif tail is None and head is None:
            new_contour = deque((from_point, to_point))
            contours[current_index] = new_contour
            starts[from_point] = (new_contour, current_index)
            ends[to_point] = (new_contour, current_index)
            current_index += 1
        elif head is None:
            # tail's first element is to_point: prepend the new segment
            tail.appendleft(from_point)
            starts[from_point] = (tail, tail_num)
        else:
            # head's last element is from_point: append the new segment
            head.append(to_point)
            ends[to_point] = (head, head_num)
    return [np.array(contour) for _, contour in sorted(contours.items())]


def find_contours(image, level):
    """[UPSTREAM skimage measure.find_contours(image, level)] with the defaults
    fully_connected='low', positive_orientation='low': list of float64 [K, 2] (row, col)
    arrays; closed contours repeat their first point at the end."""
    image = np.asarray(image, dtype=np.float64)
    if image.ndim != 2:
        raise ValueError("Only 2D arrays are supported.")
    return _assemble_contours(_get_contour_segments(image, float(level)))


def mask_contours(mask):
    """[REF] serve.py:160-169 calls visualize.display_instances; [UPSTREAM] its outline step
    for one instance: pad the mask with a ring of zeros, find_contours(padded, 0.5), and turn
    every contour into (x, y) vertices without the padding, np.fliplr(verts) - 1 -- the arrays
    handed to matplotlib's Polygon.  mask: bool [H, W].  Returns a list of float64 [K, 2]
    arrays, each closed (first row == last row)."""
    mask = np.asarray(mask)
    padded_mask = np.zeros((mask.shape[0] + 2, mask.shape[1] + 2), dtype=np.uint8)
    padded_mask[1:-1, 1:-1] = mask
    contours = find_contours(padded_mask, 0.5)
    return [np.fliplr(verts) - 1 for verts in contours]


def mask_contours_batch(masks):
    """mask_contours for every instance of a bool [H, W, N] array: a list of N lists."""
    return [mask_contours(masks[:, :, i]) for i in range(masks.shape[-1])]
