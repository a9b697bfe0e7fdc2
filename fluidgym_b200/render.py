"""Batched rendering: the static render maps (host-side setup) and the colour maps.

The reference renders a field by a bilinear splat of the cell values onto a uniform pixel grid, weight normalisation and
hole-filling sweeps (``simulation/pict/data/resample.py:300-358`` -> ``extensions/resampling.cu:191-364``).  Geometry and
output grid never change, so every pixel is a fixed linear combination of cell values -- the same map the sensors read a few
rows of (``fluidgym_b200.sensors``).  Here the whole map of one image is built once per environment instance, stored as CSR
in output image order, and evaluated for the batch by ``fgb_render_gather``; ``fgb_render_colour`` maps the result to RGB.

Image order: row 0 is the top of the domain (largest y), x runs left to right.  The wall-parallel planes of the channel flow
are shown as stored, row = z, column = x.
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np
import scipy.sparse as sp

from .sensors import _extruded_centres, _sensor_rows_localized, normalise_and_fill, pixel_map_3d, splat_matrix

IDENTITY, NORM = 0, 1           # fgb_render_gather modes (include/fluidgym_b200.h)


class RenderMap(NamedTuple):
    """CSR map [P = H * W, N]: image pixel p (row-major, image order) = sum_k w[k] field[col[k]], k in [rowptr[p], rowptr[p+1])."""
    rowptr: np.ndarray          # int32 [P + 1]
    col: np.ndarray             # int32 [nnz]
    w: np.ndarray               # float32 [nnz]
    shape: tuple                # (H, W)

    def matrix(self, n_cells: int) -> sp.csr_matrix:
        return sp.csr_matrix((self.w.astype(np.float64), self.col, self.rowptr), shape=(self.shape[0] * self.shape[1], n_cells))


def _from_csr(R: sp.csr_matrix, shape) -> RenderMap:
    R = R.tocsr()
    R.sort_indices()
    return RenderMap(R.indptr.astype(np.int32), R.indices.astype(np.int32), R.data.astype(np.float32), (int(shape[0]), int(shape[1])))


def _image_rows(W: int, H: int) -> np.ndarray:
    """pixel-grid index (y * W + x, y upwards) of every image pixel in image order"""
    return (np.arange(H - 1, -1, -1)[:, None] * W + np.arange(W)[None, :]).ravel()


def render_map_2d(vertex_list, out_shape, fill_max_steps: int) -> RenderMap:
    """The whole rendered-pixel map of a 2-D multi-block domain on ``out_shape = (W, H)`` (the splat of ``sensors.splat_matrix``,
    then normalisation and fill sweeps with 4 neighbours)."""
    W, H = int(out_shape[0]), int(out_shape[1])
    S, wsum = splat_matrix(vertex_list, (W, H))
    R, _ = normalise_and_fill(S, wsum, (H, W), fill_max_steps)
    return _from_csr(R[_image_rows(W, H)], (H, W))


def render_map_box3d(vertex: np.ndarray, out_shape, plane: int, fill_max_steps: int) -> RenderMap:
    """Slice z = ``plane`` of the rendered-voxel map of a 3-D box (``sensors.pixel_map_3d``, incl. the reference's 6-corner
    splat) on ``out_shape = (W, H, Z)`` -> image [H, W]."""
    W, H, Z = (int(s) for s in out_shape)
    R, _ = pixel_map_3d(vertex, (W, H, Z), fill_max_steps)
    return _from_csr(R[_image_rows(W, H) + W * H * int(plane)], (H, W))


def render_map_extruded(vertex2d_list, z_vertices: np.ndarray, out_shape, plane: int, fill_max_steps: int) -> RenderMap:
    """Slice z = ``plane`` of the rendered-voxel map of a z-extruded multi-block domain (columns = z plane * N2 + g); only the
    rows of that slice are built (``sensors._sensor_rows_localized``)."""
    W, H, Z = (int(s) for s in out_shape)
    centres, lower, upper = _extruded_centres(vertex2d_list, z_vertices)
    rows = _sensor_rows_localized(centres, lower, upper, (W, H, Z), fill_max_steps, 3 << 1, _image_rows(W, H) + W * H * int(plane))
    rowptr = np.zeros(len(rows) + 1, dtype=np.int64)
    rowptr[1:] = np.cumsum([len(ci) for ci, _ in rows])
    col = np.concatenate([ci for ci, _ in rows]) if rows else np.zeros(0, np.int64)
    w = np.concatenate([cw for _, cw in rows]) if rows else np.zeros(0)
    return RenderMap(rowptr.astype(np.int32), col.astype(np.int32), w.astype(np.float32), (H, W))


def render_map_cell_plane(nx: int, ny: int, nz: int, plane: int) -> RenderMap:
    """Cell plane y = ``plane`` of a uniform-in-x/z box with cells in (z, y, x) order -> image [nz, nx], one entry per pixel."""
    z, x = np.meshgrid(np.arange(nz), np.arange(nx), indexing="ij")
    col = ((z * ny + int(plane)) * nx + x).ravel()
    return RenderMap(np.arange(nz * nx + 1, dtype=np.int32), col.astype(np.int32), np.ones(nz * nx, np.float32), (nz, nx))


# ---------------------------------------------------------------------------------------------------------------------
# Colour maps: 256-entry RGB tables, linear between the anchors.  DIVERGING for signed fields (blue - white - red, the range
# symmetric about zero), SEQUENTIAL for magnitudes and temperature (dark blue - teal - yellow).
# ---------------------------------------------------------------------------------------------------------------------
_DIVERGING_ANCHORS = ((0.0, (5, 48, 97)), (0.25, (67, 147, 195)), (0.5, (247, 247, 247)), (0.75, (214, 96, 77)), (1.0, (103, 0, 31)))
_SEQUENTIAL_ANCHORS = ((0.0, (68, 1, 84)), (0.25, (59, 82, 139)), (0.5, (33, 145, 140)), (0.75, (94, 201, 98)), (1.0, (253, 231, 37)))


def _lut(anchors) -> np.ndarray:
    pos = np.array([a[0] for a in anchors])
    rgb = np.array([a[1] for a in anchors], dtype=np.float64)
    t = (np.arange(256) + 0.5) / 256.0
    return np.stack([np.rint(np.interp(t, pos, rgb[:, c])) for c in range(3)], axis=1).astype(np.uint8)


DIVERGING = _lut(_DIVERGING_ANCHORS)
SEQUENTIAL = _lut(_SEQUENTIAL_ANCHORS)


def colour_bins(img: np.ndarray, lo, hi) -> np.ndarray:
    """LUT index of every value of ``img`` [B, ...] for the range [lo, hi] ([B] arrays or scalars), in float32 as
    ``fgb_render_colour`` computes it: floor(256 (v - lo) / (hi - lo)) clamped to [0, 255]; 128 when hi <= lo."""
    img = np.asarray(img, dtype=np.float32)
    B = img.shape[0]
    lo = np.broadcast_to(np.asarray(lo, dtype=np.float32), (B,)).reshape((B,) + (1,) * (img.ndim - 1))
    hi = np.broadcast_to(np.asarray(hi, dtype=np.float32), (B,)).reshape((B,) + (1,) * (img.ndim - 1))
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(hi > lo, (img - lo) / (hi - lo), np.float32(0.5)).astype(np.float32)
    x = (t * np.float32(256.0)).astype(np.float32)
    return np.clip(np.nan_to_num(x, nan=0.0), 0, 255).astype(np.int64)


def colour_reference(img: np.ndarray, lut: np.ndarray, vmin=None, vmax=None, symmetric: bool = False) -> np.ndarray:
    """Numpy specification of ``fgb_render_colour``: ``img`` [B, H, W] -> uint8 [B, H, W, 3].  Without ``vmin`` / ``vmax`` the
    range is each environment's own min / max; ``symmetric`` widens it to [-m, m], m = max |v|."""
    img = np.asarray(img, dtype=np.float32)
    if vmin is None:
        flat = img.reshape(img.shape[0], -1)
        lo, hi = flat.min(axis=1), flat.max(axis=1)
    else:
        lo, hi = np.float32(vmin), np.float32(vmax)
    if symmetric:
        m = np.maximum(np.abs(lo), np.abs(hi))
        lo, hi = -m, m
    return lut[colour_bins(img, lo, hi)]
