"""CPU restatement of the stacked pointnet2 ops the RoI head runs on the backbone's outputs — TEST INFRASTRUCTURE
(see oracle/__init__.py).  Plain loops, small cases only; at full size the checker is the output of the reference's own
kernels (compiled into oracle/_ref by oracle/ref_build.py) stored in tests/golden/roi_pool.npz.

voxel_query  : pcdet/ops/pointnet2/pointnet2_stack/src/voxel_query_gpu.cu:10-89 + voxel_query_utils.py:36-41
group_points : .../src/group_points_gpu.cu:71-103, grad :15-45"""
from __future__ import annotations

import numpy as np


def voxel_query(max_range, radius, nsample, xyz, new_xyz, new_coords, point_indices):
    """-> (idx [M, nsample] int32 with empty rows zeroed, empty_ball_mask [M] bool)"""
    M = new_coords.shape[0]
    B, R1, R2, R3 = point_indices.shape
    zr, yr, xr = max_range
    idx = np.zeros((M, nsample), dtype=np.int32)
    f32 = np.float32
    radius2 = f32(radius) * f32(radius)
    flat = point_indices.reshape(-1)
    for pt in range(M):
        b, cz, cy, cx = (int(v) for v in new_coords[pt])
        nx, ny, nz = (f32(v) for v in new_xyz[pt])
        cnt = 0
        for dz in range(-zr, zr + 1):
            z = cz + dz
            if z < 0 or z >= R1:
                continue
            for dy in range(-yr, yr + 1):
                y = cy + dy
                if y < 0 or y >= R2:
                    continue
                for dx in range(-xr, xr + 1):
                    x = cx + dx
                    if x < 0 or x >= R3:
                        continue
                    nb = int(flat[b * R1 * R2 * R3 + z * R2 * R3 + y * R3 + x])
                    if nb < 0:
                        continue
                    d = xyz[nb].astype(np.float64) - np.array([nx, ny, nz], dtype=np.float64)
                    dist2 = f32(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])      # exact products, rounded once (tests keep
                    if dist2 > radius2:                                       # their points off the radius boundary)
                        continue
                    if cnt < nsample:
                        if cnt == 0:
                            idx[pt, :] = nb
                        idx[pt, cnt] = nb
                        cnt += 1
        if cnt == 0:
            idx[pt, 0] = -1
    empty = idx[:, 0] == -1
    idx[empty] = 0
    return idx, empty


def _starts(pt, idx_batch_cnt, features_batch_cnt):
    bs, pt_cnt = 0, int(idx_batch_cnt[0])
    for k in range(1, len(idx_batch_cnt)):
        if pt < pt_cnt:
            break
        pt_cnt += int(idx_batch_cnt[k])
        bs = k
    return int(np.sum(features_batch_cnt[:bs]))


def group_points(features, features_batch_cnt, idx, idx_batch_cnt):
    M, nsample = idx.shape
    C = features.shape[1]
    out = np.zeros((M, C, nsample), dtype=np.float32)
    for pt in range(M):
        s0 = _starts(pt, idx_batch_cnt, features_batch_cnt)
        out[pt] = features[s0 + idx[pt]].T
    return out


def group_points_grad(grad_out, idx, idx_batch_cnt, features_batch_cnt, N):
    M, C, nsample = grad_out.shape
    g = np.zeros((N, C), dtype=np.float64)
    for pt in range(M):
        s0 = _starts(pt, idx_batch_cnt, features_batch_cnt)
        for s in range(nsample):
            g[s0 + idx[pt, s]] += grad_out[pt, :, s]
    return g.astype(np.float32)


def scene(seed, n_per=(5000, 4200), shape=(21, 400, 352), n_query=(3000, 3000), stride=4, jitter=0.5):
    """Sparse voxels (batch-contiguous rows), their centres, the dense voxel->row map and query points near them."""
    rng = np.random.default_rng(seed)
    vs = np.array([0.05, 0.05, 0.05], np.float32) * stride
    lo = np.array([0, -40, -3], np.float32)
    coords, cnt = [], []
    for b, n in enumerate(n_per):
        # n distinct cells inside a window holding ~8n cells (density like a LiDAR surface patch), rows sorted by cell
        wy = int(min(shape[1], max(4, round((8 * n / shape[0]) ** 0.5))))
        wx = int(min(shape[2], max(4, -(-8 * n // (shape[0] * wy)))))
        n = min(n, shape[0] * wy * wx)
        win = np.sort(rng.choice(shape[0] * wy * wx, size=n, replace=False))
        z, y, x = win // (wy * wx), (win // wx) % wy + (shape[1] - wy) // 2, win % wx + (shape[2] - wx) // 3
        coords.append(np.stack([np.full_like(z, b), z, y, x], 1))
        cnt.append(n)
    coords = np.concatenate(coords).astype(np.int32)
    xyz = np.ascontiguousarray(((coords[:, [3, 2, 1]].astype(np.float32) + 0.5) * vs + lo).astype(np.float32))
    v2p = -np.ones((len(n_per),) + tuple(shape), dtype=np.int32)
    v2p[coords[:, 0], coords[:, 1], coords[:, 2], coords[:, 3]] = np.arange(len(coords), dtype=np.int32)
    new_xyz, new_coords = [], []
    start = 0
    for b, (n, m) in enumerate(zip(cnt, n_query)):
        pick = rng.integers(0, n, m) + start
        p = xyz[pick] + rng.normal(0, jitter, (m, 3)).astype(np.float32)
        c = np.ascontiguousarray(np.floor((p - lo) / vs).astype(np.int32)[:, [2, 1, 0]])
        new_xyz.append(p)
        new_coords.append(np.concatenate([np.full((m, 1), b, np.int32), c], 1))
        start += n
    return (xyz, np.array(cnt, np.int32), np.ascontiguousarray(np.concatenate(new_xyz).astype(np.float32)),
            np.array(n_query, np.int32), np.ascontiguousarray(np.concatenate(new_coords).astype(np.int32)), v2p)


# The full-size voxel-query / grouping cases whose outputs from the reference's own kernels are stored in
# tests/golden/roi_pool.npz (oracle/make_golden.py roi_pool): scene(1), 32 feature channels.
ROI_CASES = (((4, 4, 4), 0.8, 16), ((2, 2, 2), 0.4, 16), ((1, 3, 5), 1.6, 5))
ROI_CHANNELS = 32


def roi_case_key(max_range, radius, nsample):
    return 'r%dx%dx%d_rad%g_ns%d' % (tuple(max_range) + (radius, nsample))


def roi_case_data(max_range, radius, nsample, n_rows, n_query):
    """Seeded features [n_rows, ROI_CHANNELS] and output gradient [n_query, ROI_CHANNELS, nsample] of one case."""
    ci = ROI_CASES.index((tuple(max_range), radius, nsample))
    feats = np.random.default_rng(100 + ci).standard_normal((n_rows, ROI_CHANNELS), dtype=np.float32)
    grad_out = np.random.default_rng(200 + ci).standard_normal((n_query, ROI_CHANNELS, nsample), dtype=np.float32)
    return feats, grad_out
