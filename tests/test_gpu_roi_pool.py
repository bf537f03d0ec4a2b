"""GPU parity tests of the voxel-RoI pooling primitives (SURVEY §8f rows 2-3) against (1) the outputs of the REFERENCE's own
CUDA kernels at realistic sizes, stored in tests/golden/roi_pool.npz by oracle/make_golden.py (bit-exact), and (2) the
numpy restatement oracle/pointnet2.py (small cases, also covers empty balls / ragged batches)."""
import os

import numpy as np
import pytest
import torch

from oracle import pointnet2 as o_pn
from oracle.testing import sha256_bytes

pytestmark = pytest.mark.gpu


def _golden(max_range, radius, nsample):
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'roi_pool.npz'))
    key = o_pn.roi_case_key(max_range, radius, nsample)
    return {k.split(':', 1)[1]: g[k] for k in g.files if k.startswith(key + ':')}


@pytest.mark.parametrize('max_range,radius,nsample', o_pn.ROI_CASES)
def test_voxel_query_and_grouping_vs_compiled_reference(lib_built, max_range, radius, nsample):
    """Index and grouping outputs are exact (seeded row samples, then digests of the whole arrays); the gradient within
    float-atomic reordering on seeded rows."""
    from virconv_b200 import roi_pool
    g = _golden(max_range, radius, nsample)
    xyz, xyz_cnt, new_xyz, new_cnt, new_coords, v2p = o_pn.scene(1)
    d = lambda a: torch.from_numpy(a).cuda()
    t_xyz, t_new_xyz, t_coords, t_v2p = d(xyz), d(new_xyz), d(new_coords), d(v2p)
    idx, empty = roi_pool.voxel_query(max_range, radius, nsample, t_xyz, t_new_xyz, t_coords, t_v2p)
    M = new_coords.shape[0]
    rempty = np.unpackbits(g['empty'], count=M).astype(bool)
    assert np.array_equal(empty.cpu().numpy(), rempty)
    assert np.array_equal(idx.cpu().numpy()[g['idx_rows']], g['idx'])
    assert sha256_bytes(idx) == str(g['idx_sha256'])
    assert 0 < int(rempty.sum()) < M or max_range == (4, 4, 4)
    # grouping forward / backward through the module path of the reference (VoxelQueryAndGrouping.forward :80-99)
    feats_np, go_np = o_pn.roi_case_data(max_range, radius, nsample, xyz.shape[0], M)
    feats = d(feats_np).requires_grad_(True)
    mod = roi_pool.VoxelQueryAndGrouping(max_range, radius, nsample)
    gf, gx, em = mod(t_coords, t_xyz, d(xyz_cnt), t_new_xyz, d(new_cnt), feats, t_v2p)
    assert np.array_equal(em.cpu().numpy(), rempty)
    rows = g['group_rows']
    assert np.array_equal(gf.detach().cpu().numpy()[rows], g['features'])
    assert np.array_equal(gx.detach().cpu().numpy()[rows], g['xyz'])
    assert sha256_bytes(gf) == str(g['features_sha256']) and sha256_bytes(gx) == str(g['xyz_sha256'])
    gf.backward(d(go_np))
    # float atomics in a different order; row 0 of every sample collects the gradient of all empty balls (thousands of terms)
    err = np.abs(feats.grad.cpu().numpy()[g['grad_rows']] - g['grad']).max()
    assert float(err) <= 1e-5 * float(g['grad_absmax'])


def test_voxel_query_and_grouping_vs_numpy_restatement(lib_built):
    """Small ragged case incl. empty balls, out-of-grid neighbourhoods and an empty sample, against oracle/pointnet2.py."""
    from virconv_b200 import roi_pool
    xyz, xyz_cnt, new_xyz, new_cnt, new_coords, v2p = o_pn.scene(2, n_per=(300, 1, 260), shape=(5, 40, 36), n_query=(70, 70, 70),
                                                                 jitter=0.9)
    new_coords[::9, 1:] += 30                                           # some query cells far outside the grid
    d = lambda a: torch.from_numpy(a).cuda()
    for max_range, radius, nsample in (((2, 2, 2), 0.5, 8), ((4, 4, 4), 2.0, 16), ((0, 0, 0), 0.3, 4)):
        idx, empty = roi_pool.voxel_query(max_range, radius, nsample, d(xyz), d(new_xyz), d(new_coords), d(v2p))
        widx, wempty = o_pn.voxel_query(max_range, radius, nsample, xyz, new_xyz, new_coords, v2p)
        assert np.array_equal(empty.cpu().numpy(), wempty) and np.array_equal(idx.cpu().numpy(), widx), max_range
        assert wempty.any() and not wempty.all()
    starts = np.concatenate([[0], np.cumsum(xyz_cnt)[:-1]])
    lidx = (widx.reshape(3, -1, nsample) - starts.reshape(-1, 1, 1)).reshape(-1, nsample).astype(np.int32)
    lidx[wempty] = 0
    feats = np.random.default_rng(0).normal(size=(xyz.shape[0], 24)).astype(np.float32)
    t_f = d(feats).requires_grad_(True)
    out = roi_pool.grouping_operation(t_f, d(xyz_cnt), d(lidx), d(new_cnt))
    assert np.array_equal(out.detach().cpu().numpy(), o_pn.group_points(feats, xyz_cnt, lidx, new_cnt))
    go = np.random.default_rng(1).normal(size=out.shape).astype(np.float32)
    out.backward(d(go))
    assert np.allclose(t_f.grad.cpu().numpy(), o_pn.group_points_grad(go, lidx, new_cnt, xyz_cnt, xyz.shape[0]), rtol=1e-5,
                       atol=1e-5)


def test_roi_pool_rejects_cpu_tensors(lib_built):
    from virconv_b200 import roi_pool
    with pytest.raises(Exception):
        roi_pool.voxel_query((1, 1, 1), 1.0, 4, torch.zeros(4, 3), torch.zeros(2, 3), torch.zeros(2, 4, dtype=torch.int32),
                             torch.zeros(1, 2, 2, 2, dtype=torch.int32))
