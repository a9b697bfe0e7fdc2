"""Sensor sampling as a static sparse linear map (host-side setup).

The reference renders *all* cells onto a uniform grid every observation (bilinear splat with atomics,
weight normalisation, up to ``fill_max_steps`` neighbour-mean hole-filling sweeps) and then reads a few
sensor pixels (``envs/util/obs_extraction.py:10-57`` -> ``simulation/pict/data/resample.py:300-358`` ->
``extensions/resampling.cu:191-243, 296-364, 526-609``).  Geometry and output grid never change, so the
value at every pixel is a fixed linear combination of cell values; this module computes those
combinations once for the sensor pixels and hands them to ``fgb_sample_sensors`` as ELL tables.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

f32 = np.float32


def cell_centres(vertex: np.ndarray) -> np.ndarray:
    """2x2 average pooling of the vertices (shapes.py:216-225) -> [2, ny, nx] float32."""
    v = vertex.astype(f32)
    return ((v[:, :-1, :-1] + v[:, :-1, 1:] + v[:, 1:, :-1] + v[:, 1:, 1:]) * f32(0.25)).astype(f32)


def uniform_grid_transform(vertex_list, out_shape):
    """AABB_OUTER mapping world -> pixel coordinates (resample.py:66-96): returns (scale, offset[2])
    with pixel = (world - centre) / scale + out_shape / 2 - 0.5."""
    allv = np.concatenate([v.reshape(2, -1) for v in vertex_list], axis=1).astype(f32)
    lower, upper = allv.min(axis=1), allv.max(axis=1)
    size = (upper - lower).astype(f32)
    centre = (lower + size * f32(0.5)).astype(f32)
    os_ = np.asarray(out_shape, dtype=f32)
    scale = f32(np.max(size / os_))
    return scale, centre, os_


def splat_matrix(vertex_list, out_shape):
    """Sparse [n_pixels, N] bilinear splat weights and per-pixel weight sums (resampling.cu:296-344)."""
    scale, centre, os_ = uniform_grid_transform(vertex_list, out_shape)
    W, H = int(out_shape[0]), int(out_shape[1])
    centres = np.concatenate([cell_centres(v).reshape(2, -1) for v in vertex_list], axis=1)
    N = centres.shape[1]
    sc = ((centres - centre[:, None]) / scale + (os_ * f32(0.5) - f32(0.5))[:, None]).astype(f32)
    fl, ce = np.floor(sc), np.ceil(sc)
    fr = (sc - fl).astype(f32)
    rows, cols, vals = [], [], []
    for ux in (0, 1):
        for uy in (0, 1):
            px = (ce[0] if ux else fl[0]).astype(np.int64)
            py = (ce[1] if uy else fl[1]).astype(np.int64)
            w = (fr[0] if ux else 1 - fr[0]) * (fr[1] if uy else 1 - fr[1])
            ok = (px >= 0) & (px < W) & (py >= 0) & (py < H)
            rows.append((py * W + px)[ok])
            cols.append(np.arange(N)[ok])
            vals.append(w[ok].astype(np.float64))
    S = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(W * H, N))
    return S, np.asarray(S.sum(axis=1)).ravel()


def fill_levels(valid0: np.ndarray, fill_max_steps: int) -> np.ndarray:
    """Sweep index at which every pixel becomes valid in ``_FillEmptyCells`` (resampling.cu:246-293):
    0 = has splat weight, k = filled from neighbours in sweep k, -1 = never."""
    H, W = valid0.shape
    level = np.where(valid0, 0, -1).astype(np.int32)
    valid = valid0.copy()
    for k in range(1, int(fill_max_steps) + 1):
        if valid.all():
            break
        nb = np.zeros_like(valid)
        nb[:, 1:] |= valid[:, :-1]
        nb[:, :-1] |= valid[:, 1:]
        nb[1:, :] |= valid[:-1, :]
        nb[:-1, :] |= valid[1:, :]
        newly = nb & ~valid
        level[newly] = k
        valid = valid | newly
    return level


def sensor_tables(vertex_list, out_shape, sensor_px: np.ndarray, fill_max_steps: int):
    """ELL tables (idx [K, n_s] int32, w [K, n_s] float32) of the rendered-pixel map at the sensor
    pixels ``sensor_px`` = [2, n_s] integer (x, y) pixel coordinates: normalised splat row where the
    pixel received weight, otherwise the mean of the neighbours that were valid one sweep earlier."""
    W, H = int(out_shape[0]), int(out_shape[1])
    S, wsum = splat_matrix(vertex_list, out_shape)
    level = fill_levels((wsum > 1e-8).reshape(H, W), fill_max_steps)
    memo = {}

    def row(y, x):
        key = (y, x)
        if key in memo:
            return memo[key]
        lv = level[y, x]
        if lv == 0:
            a, b = S.indptr[y * W + x], S.indptr[y * W + x + 1]
            r = dict(zip(S.indices[a:b].tolist(), (S.data[a:b] / wsum[y * W + x]).tolist()))
        elif lv < 0:
            r = {}
        else:
            nb = [(y + dy, x + dx) for dx, dy in ((-1, 0), (1, 0), (0, -1), (0, 1))
                  if 0 <= x + dx < W and 0 <= y + dy < H and 0 <= level[y + dy, x + dx] < lv]
            r = {}
            for (yy, xx) in nb:
                for c, v in row(yy, xx).items():
                    r[c] = r.get(c, 0.0) + v / len(nb)
        memo[key] = r
        return r

    rows = [row(int(y), int(x)) for x, y in zip(sensor_px[0], sensor_px[1])]
    ns = len(rows)
    K = max(1, max(len(r) for r in rows))
    idx = np.zeros((K, ns), dtype=np.int32)
    w = np.zeros((K, ns), dtype=f32)
    for s_, r in enumerate(rows):
        for k, (c, v) in enumerate(sorted(r.items())):
            idx[k, s_] = c
            w[k, s_] = v
    return idx, w


# ---------------------------------------------------------------------------------------------------------------------
# D = 3 (RBC3D): the same static map.  The reference's 3-D splat kernel loops over ``DIMS << 1`` = 6 of the 8 corner
# pixels around a cell centre (resampling.cu:320: corners (x,y,z) = 000, 100, 010, 110, 001, 101 -- 011 and 111 are never
# written); the observations are defined by that kernel, so the quirk is reproduced here.  Hole filling averages the valid
# ones of the 6 face neighbours per sweep (resampling.cu:191-243).  Everything is built with sparse matrices, one sweep
# at a time, so render grids of 10^6 pixels are fine.
# ---------------------------------------------------------------------------------------------------------------------
def cell_centres_3d(vertex: np.ndarray) -> np.ndarray:
    """2x2x2 average pooling of the vertices [3, nz+1, ny+1, nx+1] -> [3, nz, ny, nx] float32."""
    v = vertex.astype(f32)
    c = 0
    for i in (0, 1):
        for j in (0, 1):
            for k in (0, 1):
                c = c + v[:, i:v.shape[1] - 1 + i, j:v.shape[2] - 1 + j, k:v.shape[3] - 1 + k]
    return (c * f32(0.125)).astype(f32)


def pixel_map_3d(vertex: np.ndarray, out_shape, fill_max_steps: int, n_corners: int = 3 << 1):
    """Sparse [W*H*Z, N] matrix R with rendered[pixel] = R @ cells (pixel index = x + W (y + H z), cells in (z, y, x)
    order) and the per-pixel fill level (0 = splat, k = filled in sweep k, -1 = never).  ``n_corners`` = 6 is what the
    reference's CUDA kernel does (and what its environments therefore observe); 8 is the full trilinear splat of its torch
    re-implementation (resample.py:442-496), used by the tests to check everything but that quirk."""
    W, H, Z = (int(s) for s in out_shape)
    allv = vertex.reshape(3, -1).astype(f32)
    centres = cell_centres_3d(vertex).reshape(3, -1)
    return _pixel_map_from_centres(centres, allv.min(axis=1), allv.max(axis=1), (W, H, Z), fill_max_steps, n_corners)


def sensor_tables_3d(vertex: np.ndarray, out_shape, sensor_px: np.ndarray, fill_max_steps: int):
    """ELL tables (idx [K, n_s] int32, w [K, n_s] float32) of the rendered-voxel map at the sensor voxels
    ``sensor_px`` = [3, n_s] integer (x, y, z) voxel coordinates (envs/rbc/rbc_env_3d.py:183-203)."""
    R, _ = pixel_map_3d(vertex, out_shape, fill_max_steps)
    return _ell_rows_at_voxels(R, out_shape, sensor_px)


def _ell_rows_at_voxels(R, out_shape, sensor_px):
    W, H, Z = (int(s) for s in out_shape)
    flat = sensor_px[0].astype(np.int64) + W * (sensor_px[1].astype(np.int64) + H * sensor_px[2].astype(np.int64))
    Rs = R[flat]
    ns = flat.size
    nnz = np.diff(Rs.indptr)
    K = max(1, int(nnz.max()))
    idx = np.zeros((K, ns), dtype=np.int32)
    w = np.zeros((K, ns), dtype=f32)
    for s_ in range(ns):
        a, b = Rs.indptr[s_], Rs.indptr[s_ + 1]
        idx[:b - a, s_] = Rs.indices[a:b]
        w[:b - a, s_] = Rs.data[a:b]
    return idx, w


def sensor_tables_extruded(vertex2d_list, z_vertices: np.ndarray, out_shape, sensor_px: np.ndarray, fill_max_steps: int):
    """sensor_tables_3d for a z-extruded multi-block domain (columns = plane * N2 + g).  Only the rows of the sensor voxels are
    built (``_sensor_rows_localized``): the full voxel map of the registered sizes has 10^7 ... 10^8 rows."""
    centres, lower, upper = _extruded_centres(vertex2d_list, z_vertices)
    W, H, Z = (int(s) for s in out_shape)
    flat = sensor_px[0].astype(np.int64) + W * (sensor_px[1].astype(np.int64) + H * sensor_px[2].astype(np.int64))
    rows = _sensor_rows_localized(centres, lower, upper, (W, H, Z), fill_max_steps, 3 << 1, flat)
    ns = flat.size
    K = max(1, max(len(r[0]) for r in rows))
    idx = np.zeros((K, ns), dtype=np.int32)
    w = np.zeros((K, ns), dtype=f32)
    for s_, (ci, cw) in enumerate(rows):
        idx[:len(ci), s_] = ci
        w[:len(ci), s_] = cw
    return idx, w


def _sensor_rows_localized(centres, lower, upper, out_shape, fill_max_steps, n_corners, sensor_flat):
    """Rows of the rendered-voxel map (``_pixel_map_from_centres``: splat + normalise + hole-fill sweeps) for the voxels
    ``sensor_flat`` only -> list of (cell indices sorted, weights float64).  The fill level of every voxel is found with dense boolean
    sweeps; the row of a voxel filled in sweep k is the mean of the rows of its face neighbours that were valid before that sweep,
    evaluated recursively (memoised) -- identical to the matrix recurrence R <- R + A R restricted to the rows that are needed."""
    W, H, Z = out_shape
    S, wsum = _splat_matrix(centres, lower, upper, out_shape, n_corners)
    npx = W * H * Z
    valid = (wsum > 1e-8).reshape(Z, H, W)
    level = np.where(valid, 0, -1).astype(np.int32)
    for k in range(1, int(fill_max_steps) + 1):
        if valid.all():
            break
        nbv = np.zeros_like(valid)
        nbv[1:] |= valid[:-1]; nbv[:-1] |= valid[1:]
        nbv[:, 1:] |= valid[:, :-1]; nbv[:, :-1] |= valid[:, 1:]
        nbv[:, :, 1:] |= valid[:, :, :-1]; nbv[:, :, :-1] |= valid[:, :, 1:]
        newly = nbv & ~valid
        if not newly.any():
            break
        level[newly] = k
        valid = valid | newly
    level = level.reshape(-1)
    strides = (1, W, W * H)
    dims = (W, H, Z)
    memo = {}

    def neighbours(v):
        x, y, z = v % W, (v // W) % H, v // (W * H)
        pos = (x, y, z)
        for ax in range(3):
            if pos[ax] > 0:
                yield v - strides[ax]
            if pos[ax] < dims[ax] - 1:
                yield v + strides[ax]

    def row(v0):
        stack = [v0]
        while stack:
            v = stack[-1]
            if v in memo:
                stack.pop()
                continue
            lv = level[v]
            if lv < 0:                                       # never filled: zero row
                memo[v] = {}
                stack.pop()
                continue
            if lv == 0:
                a, b = S.indptr[v], S.indptr[v + 1]
                inv = 1.0 / wsum[v]
                d = {}
                for c, x in zip(S.indices[a:b], S.data[a:b]):
                    d[int(c)] = d.get(int(c), 0.0) + x * inv
                memo[v] = d
                stack.pop()
                continue
            srcs = [n for n in neighbours(v) if 0 <= level[n] < lv]
            missing = [n for n in srcs if n not in memo]
            if missing:
                stack.extend(missing)
                continue
            d = {}
            f = 1.0 / len(srcs)
            for n in srcs:
                for c, x in memo[n].items():
                    d[c] = d.get(c, 0.0) + x * f
            memo[v] = d
            stack.pop()
        return memo[v0]

    out = []
    for v in np.asarray(sensor_flat, dtype=np.int64):
        d = row(int(v))
        ci = np.array(sorted(d), dtype=np.int64)
        out.append((ci, np.array([d[c] for c in ci], dtype=np.float64)))
    return out


def pixel_map_extruded(vertex2d_list, z_vertices: np.ndarray, out_shape, fill_max_steps: int, n_corners: int = 3 << 1):
    """pixel_map_3d for a z-extruded multi-block domain (CylinderJet3D / Airfoil3D): ``vertex2d_list`` = the 2-D vertex grids of
    the blocks [2, ny+1, nx+1], ``z_vertices`` [nz+1].  Columns are the cells in plane-major order (plane * N2 + g, g = block-major
    2-D cell index), the layout of fluidgym_b200/extruded3d.py."""
    W, H, Z = (int(s) for s in out_shape)
    centres, lower, upper = _extruded_centres(vertex2d_list, z_vertices)
    return _pixel_map_from_centres(centres, lower, upper, (W, H, Z), fill_max_steps, n_corners)


def _extruded_centres(vertex2d_list, z_vertices):
    z_vertices = np.asarray(z_vertices, dtype=f32)
    allxy = np.concatenate([v.reshape(2, -1) for v in vertex2d_list], axis=1).astype(f32)
    lower = np.array([allxy[0].min(), allxy[1].min(), z_vertices.min()], dtype=f32)
    upper = np.array([allxy[0].max(), allxy[1].max(), z_vertices.max()], dtype=f32)
    c2 = np.concatenate([cell_centres(v).reshape(2, -1) for v in vertex2d_list], axis=1)            # [2, N2]
    zc = ((z_vertices[:-1] + z_vertices[1:]) * f32(0.5)).astype(f32)
    nz, N2 = zc.size, c2.shape[1]
    centres = np.stack([np.tile(c2[0], nz), np.tile(c2[1], nz), np.repeat(zc, N2)]).astype(f32)     # [3, nz * N2]
    return centres, lower, upper


def _splat_matrix(centres, lower, upper, out_shape, n_corners):
    """(S csr [voxels, cells] of the raw splat weights, row sums) -- the first stage of ``_pixel_map_from_centres``"""
    W, H, Z = out_shape
    size = (upper - lower).astype(f32)
    centre = (lower + size * f32(0.5)).astype(f32)
    os_ = np.asarray([W, H, Z], dtype=f32)
    scale = f32(np.max(size / os_))
    N = centres.shape[1]
    sc = ((centres - centre[:, None]) / scale + (os_ * f32(0.5) - f32(0.5))[:, None]).astype(f32)
    fl, ce = np.floor(sc), np.ceil(sc)
    fr = (sc - fl).astype(f32)
    dims = (W, H, Z)
    rows, cols, vals = [], [], []
    for idx in range(n_corners):
        ok = np.ones(N, dtype=bool)
        w = np.ones(N, dtype=f32)
        pos = []
        for c in range(3):
            up = (idx >> c) & 1
            pc = (ce[c] if up else fl[c]).astype(np.int64)
            ok &= (pc >= 0) & (pc < dims[c])
            w = (w * (fr[c] if up else f32(1.0) - fr[c])).astype(f32)
            pos.append(pc)
        flat = pos[0] + W * (pos[1] + H * pos[2])
        rows.append(flat[ok]); cols.append(np.arange(N)[ok]); vals.append(w[ok].astype(np.float64))
    npx = W * H * Z
    S = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(npx, N))
    wsum = np.asarray(S.sum(axis=1)).ravel()
    return S, wsum


def _pixel_map_from_centres(centres, lower, upper, out_shape, fill_max_steps, n_corners):
    W, H, Z = out_shape
    S, wsum = _splat_matrix(centres, lower, upper, out_shape, n_corners)
    return normalise_and_fill(S, wsum, (Z, H, W), fill_max_steps)


def normalise_and_fill(S, wsum, grid_shape, fill_max_steps):
    """Rendered-pixel map R [pixels, cells] from the raw splat ``S`` and its row sums: rows with weight normalised, then up to
    ``fill_max_steps`` hole-filling sweeps R <- R + A R, where A gives every still empty pixel the mean of its face neighbours
    (2 per axis of ``grid_shape``, C order = pixel order) that were valid before the sweep (resampling.cu:191-293).
    Returns (R csr, fill level per pixel: 0 = splat, k = filled in sweep k, -1 = never)."""
    npx = S.shape[0]
    nd = len(grid_shape)
    valid = wsum > 1e-8
    level = np.where(valid, 0, -1).astype(np.int32)
    inv = np.zeros(npx)
    inv[valid] = 1.0 / wsum[valid]
    R = sp.diags(inv) @ S
    grid = np.arange(npx).reshape(grid_shape)
    for k in range(1, int(fill_max_steps) + 1):
        if valid.all():
            break
        v3 = valid.reshape(grid_shape)
        src_l, dst_l = [], []
        for ax in range(nd):
            for sh in (1, -1):
                a = [slice(None)] * nd
                b = [slice(None)] * nd
                a[ax] = slice(1, None) if sh == 1 else slice(0, -1)
                b[ax] = slice(0, -1) if sh == 1 else slice(1, None)
                m = (~v3[tuple(a)]) & v3[tuple(b)]
                dst_l.append(grid[tuple(a)][m]); src_l.append(grid[tuple(b)][m])
        dst, src = np.concatenate(dst_l), np.concatenate(src_l)
        if dst.size == 0:
            break
        cnt = np.bincount(dst, minlength=npx).astype(np.float64)
        A = sp.csr_matrix((1.0 / cnt[dst], (dst, src)), shape=(npx, npx))
        R = R + A @ R
        newly = cnt > 0
        level[newly] = k
        valid = valid | newly
    return R.tocsr(), level
