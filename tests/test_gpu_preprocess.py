"""GPU parity tests for the model-side preprocessing (SURVEY §8f row 1): StVD input point discard against the outputs of
the reference's own `DatasetTemplate.input_point_discard` (tests/golden/stvd_input.npz) and against the oracle at larger
sizes; the split/re-fuse flow of dataset.py:270-298; `PointsToVoxels` against the first-come voxeliser + MeanVFE."""
import os

import numpy as np
import pytest
import torch

from oracle import stvd as o_stvd

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def test_stvd_input_discard_matches_reference_golden(lib_built):
    from virconv_b200 import preprocess
    for name, pts, bn, rate, seed, want in o_stvd.golden_cases(np.load(os.path.join(GOLD, 'stvd_input.npz'))):
        np.random.seed(seed)                                            # the reference draws from the global generator
        out = preprocess.input_point_discard(torch.from_numpy(pts.copy()).cuda(), bin_num=bn, rate=rate)
        assert np.array_equal(out.cpu().numpy(), want, equal_nan=True), name


@pytest.mark.parametrize('n,bins,rate', [(300000, 10, 0.8), (300000, 2, 0.8), (100001, 10, 0.5), (1023, 3, 0.9), (1, 2, 0.8)])
def test_stvd_input_discard_vs_oracle_large(lib_built, n, bins, rate):
    """BASELINE config 4 size (300k virtual points) and ragged sizes; bit-exact rows in the same order."""
    from virconv_b200 import preprocess
    rng = np.random.default_rng(n + bins)
    pts = rng.normal(25, 20, (n, 8)).astype(np.float32)
    want = o_stvd.input_point_discard(pts.copy(), bins, rate, np.random.RandomState(7))
    got = preprocess.input_point_discard(torch.from_numpy(pts).cuda(), bins, rate, np.random.RandomState(7))
    assert got.shape == want.shape and np.array_equal(got.cpu().numpy(), want)
    # size-independent properties: far -> near bin order, every kept row is an input row
    x = got[:, 0].cpu().numpy()
    b = np.minimum(np.floor(x / np.float32(60 / bins)), bins - 1)
    assert np.all(np.diff(b) <= 0)


def test_stvd_empty_cloud_raises_like_the_reference(lib_built):
    from virconv_b200 import preprocess
    with pytest.raises(ZeroDivisionError):
        preprocess.input_point_discard(torch.zeros((0, 8), device='cuda'))
    with pytest.raises(Exception):
        preprocess.input_point_discard(torch.zeros((4, 8)))            # CPU tensor: no fallback


@pytest.mark.parametrize('training,later_fusion', [(True, False), (False, False), (True, True)])
def test_split_and_discard_flow(lib_built, training, later_fusion):
    """dataset.py:270-298 on one synthetic frame: indicator split, discard with bin_num 2 (train) / 10 (test), re-fusion
    with intensity / 10 for VirConv-L, two streams for VirConv-T/S."""
    from virconv_b200 import preprocess, scenes
    pts = scenes.make_points(8, n_lidar=4096, n_virtual=20000).astype(np.float32)
    virt, lidar = pts[pts[:, -1] == 1], pts[pts[:, -1] == 2]
    kept = o_stvd.input_point_discard(virt.copy(), 2 if training else 10, 0.8, np.random.RandomState(3))
    out = preprocess.split_and_discard(torch.from_numpy(pts).cuda(), training, 0.8, later_fusion, np.random.RandomState(3))
    if later_fusion:
        assert np.array_equal(out['points'].cpu().numpy(), lidar)
        assert np.array_equal(out['points_mm'].cpu().numpy(), kept)
    else:
        want = np.concatenate([lidar, kept])
        want[:, 3] /= 10
        assert set(out) == {'points'} and np.array_equal(out['points'].cpu().numpy(), want)


def test_points_to_voxels_module(lib_built):
    """`PointsToVoxels` == the dataloader's first-come voxeliser (data_processor.py:128-187) + MeanVFE, both streams."""
    from virconv_b200 import preprocess, scenes
    parts, parts_mm, want, want_mm = [], [], [], []
    for b, sid in enumerate((31, 32)):
        pts = scenes.mask_points_by_range(scenes.make_points(sid, n_lidar=3000, n_virtual=9000)).astype(np.float32)
        for src, dst, ref in ((pts[pts[:, -1] == 2], parts, want), (pts[pts[:, -1] == 1], parts_mm, want_mm)):
            dst.append(np.concatenate([np.full((len(src), 1), b, np.float32), src], 1))
            vox, coords, num = scenes.voxelize_first_come(src, max_voxels=2000)
            ref.append((scenes.mean_vfe(vox, num, 'max'), np.concatenate([np.full((len(coords), 1), b, coords.dtype), coords], 1), num))
    bd = {'batch_size': 2, 'points': torch.from_numpy(np.concatenate(parts)).cuda(),
          'points_mm': torch.from_numpy(np.concatenate(parts_mm)).cuda()}
    mod = preprocess.PointsToVoxels(max_voxels={'train': 2000, 'test': 2000}).cuda()
    bd = mod(bd)
    for sfx, ref in (('', want), ('_mm', want_mm)):
        f = np.concatenate([r[0] for r in ref])
        c = np.concatenate([r[1] for r in ref])
        n = np.concatenate([r[2] for r in ref])
        assert bd['voxel_coords' + sfx].dtype == torch.float32
        assert np.array_equal(bd['voxel_coords' + sfx].cpu().numpy().astype(np.int64), c.astype(np.int64)), sfx
        assert np.array_equal(bd['voxel_num_points' + sfx].cpu().numpy(), n), sfx
        assert np.allclose(bd['voxel_features' + sfx].cpu().numpy(), f, rtol=1e-6, atol=1e-6), sfx
