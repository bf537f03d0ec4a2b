"""CPU tests (no GPU): the oracle against the golden vectors made from the reference's own Python, and
against brute-force dense convolution (the only ground truth for the spconv internals)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import index2uv as ouv
from oracle import rulebook as orb
from oracle import spconv_cpu as osp
from oracle.backbone import VirConvL8x as OracleL
from oracle.testing import check_sampled_rows, fill_module, golden_threads, rel_err
from virconv_b200 import scenes

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _coords(rng, n, batch, shape, unique=True):
    c = np.stack([rng.integers(0, batch, n)] + [rng.integers(0, s, n) for s in shape], 1).astype(np.int32)
    if unique:
        c = np.unique(c, axis=0)
        rng.shuffle(c)
    return c


def test_index2uv_matches_reference_golden():
    g = np.load(os.path.join(GOLD, 'index2uv.npz'))
    for ci in range(int(g['n_cases'])):
        aug = g[f'aug{ci}']
        uv = ouv.index2uv(g[f'idx{ci}'], 2, [scenes.Calib(), scenes.Calib()], int(g[f'stride{ci}']),
                          aug if aug.shape[0] else None)
        assert np.array_equal(uv, g[f'uv{ci}'])


def test_mean_vfe_matches_reference_golden():
    g = np.load(os.path.join(GOLD, 'mean_vfe.npz'))
    assert np.array_equal(scenes.mean_vfe(g['voxels'], g['num'], 'max'), g['features'])


def test_voxelizer_first_come_semantics():
    rng = np.random.default_rng(0)
    pts = rng.uniform([0, -40, -3, 0, 0, 0, 0, 1], [70.4, 40, 1, 1, 1, 1, 1, 2], size=(5000, 8)).astype(np.float32)
    pts[::7] = pts[3]                      # repeated points fill one voxel past its 5 slots
    vox, coords, num = scenes.voxelize_first_come(pts, max_voxels=1000)
    # sequential restatement
    seen, order, cnt = {}, [], []
    for p in pts:
        c = tuple(np.floor((p[:3] - scenes.POINT_CLOUD_RANGE[:3]) / np.float32(0.05)).astype(int))
        if not all(0 <= c[i] < (1408, 1600, 80)[i] for i in range(3)):
            continue
        if c not in seen:
            if len(order) >= 1000:
                continue
            seen[c] = len(order)
            order.append(c)
            cnt.append(0)
        cnt[seen[c]] += 1
    assert coords.shape[0] == len(order) == 1000
    assert np.array_equal(coords, np.array([(c[2], c[1], c[0]) for c in order], dtype=np.int32))
    assert np.array_equal(num, np.minimum(cnt, 5))
    assert vox.shape == (1000, 5, 8) and np.all(vox[num == 1][:, 1:] == 0)


@pytest.mark.parametrize('mode', ['eval', 'train'])
def test_oracle_backbone_matches_reference_flow_golden(mode):
    """The restated VirConvL8x flow == the reference's classes run over the same oracle operators."""
    g = np.load(os.path.join(GOLD, 'virconv_l_small.npz'))
    m = OracleL()
    fill_module(m, int(g['seed']))
    m.train(mode == 'train')
    with torch.no_grad(), golden_threads():
        o = m(torch.from_numpy(g['voxel_features'].copy()), torch.from_numpy(g['voxel_coords'].copy()), 2,
              [scenes.Calib(), scenes.Calib()], g['aug_param'])
    for k in ('x_conv1', 'x_conv2', 'x_conv3', 'x_conv4', 'out'):
        assert np.array_equal(o[k].indices.numpy(), g[f'{mode}_{k}_indices'])
        check_sampled_rows(o[k].features, g, f'{mode}_{k}_features')


def test_scene_generator_is_deterministic_and_kitti_shaped():
    a, b = scenes.make_batch([0]), scenes.make_batch([0])
    assert np.array_equal(a.voxel_features, b.voxel_features) and np.array_equal(a.voxel_coords, b.voxel_coords)
    assert a.voxel_features.shape == (40000, 8) and a.sparse_shape() == [81, 1600, 1408]
    c = a.voxel_coords
    assert c[:, 1].max() < 81 and c[:, 2].max() < 1600 and c[:, 3].max() < 1408 and c.min() >= 0
    assert set(np.unique(a.voxel_features[:, 7])) <= {1.0, 2.0}        # 'max' VFE keeps the indicator integral


# ------------------------------------------------------------------------------------------------
# sparse-conv semantics pinned by dense convolution
# ------------------------------------------------------------------------------------------------
GEOS = [dict(kernel_size=3, stride=2, padding=1), dict(kernel_size=3, stride=2, padding=(0, 1, 1)),
        dict(kernel_size=(3, 1, 1), stride=(2, 1, 1), padding=0), dict(kernel_size=2, stride=2, padding=0)]


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_subm_and_strided_conv_equal_dense_conv3d(seed):
    rng = np.random.default_rng(seed)
    B, shape = 2, [9, 10, 11]
    c = _coords(rng, 400, B, shape)
    feats = torch.randn(c.shape[0], 5)
    x = osp.SparseConvTensor(feats, torch.from_numpy(c), shape, B)
    dense_in = x.dense()
    m = osp.SubMConv3d(5, 7, 3, bias=False)
    ref = F.conv3d(dense_in, m.weight.detach().permute(0, 4, 1, 2, 3), padding=1)
    assert rel_err(m(x).features.detach(), ref[c[:, 0], :, c[:, 1], c[:, 2], c[:, 3]]) < 1e-5
    for geo in GEOS:
        m = osp.SparseConv3d(5, 7, bias=False, **geo)
        y = m(x)
        ref = F.conv3d(dense_in, m.weight.detach().permute(0, 4, 1, 2, 3), stride=geo['stride'], padding=geo['padding'])
        assert list(y.dense().shape) == list(ref.shape)
        assert rel_err(y.dense().detach(), ref) < 1e-5
        # output set = exactly the cells whose receptive field holds an active input
        occ = F.conv3d((dense_in.abs().sum(1, keepdim=True) > 0).float(), torch.ones(1, 1, *m.kernel_size),
                       stride=geo['stride'], padding=geo['padding'])
        assert int((occ > 0).sum()) == y.indices.shape[0]
        lin = orb.linearize(y.indices.numpy(), y.spatial_shape)
        assert np.all(np.diff(lin) > 0)


def test_subm2d_duplicates_lowest_row_wins():
    rng = np.random.default_rng(0)
    c = _coords(rng, 300, 2, [12, 9], unique=False)
    assert np.unique(c, axis=0).shape[0] < c.shape[0]
    a = orb.subm_rulebook(c, [12, 9], 3)
    assert np.array_equal(a, orb.subm_rulebook_sequential(c, [12, 9], 3))
    assert np.array_equal(a[4], np.arange(c.shape[0]))               # centre = identity
    # conv value: centre from the row itself, neighbours from the lowest row of each neighbouring pixel
    feats = torch.randn(c.shape[0], 3)
    m = osp.SubMConv2d(3, 4, 3, bias=False)
    y = m(osp.SparseConvTensor(feats, torch.from_numpy(c), [12, 9], 2)).features.detach()
    w = m.weight.detach()
    lut = {}
    for r in range(c.shape[0]):
        lut.setdefault(tuple(c[r]), r)
    for r in rng.integers(0, c.shape[0], 25):
        acc = torch.zeros(4)
        for ku in range(3):
            for kv in range(3):
                if (ku, kv) == (1, 1):
                    src = r
                else:
                    src = lut.get((c[r, 0], c[r, 1] + ku - 1, c[r, 2] + kv - 1))
                if src is not None:
                    acc += w[:, ku, kv, :] @ feats[src]
        assert torch.allclose(acc, y[r], atol=1e-5)


def test_pairs_from_nbr_canonical_order():
    rng = np.random.default_rng(1)
    c = _coords(rng, 200, 1, [6, 6, 6])
    nbr = orb.subm_rulebook(c, [6, 6, 6], 3)
    pairs, num = orb.pairs_from_nbr(nbr)
    for k in range(27):
        o = pairs[1, k, :num[k]]
        assert np.all(np.diff(o) > 0) and np.array_equal(nbr[k, o], pairs[0, k, :num[k]])
        assert np.all(pairs[:, k, num[k]:] == -1)


@pytest.mark.parametrize('mode', ['train', 'eval'])
def test_oracle_virconv8x_matches_reference_flow_golden(mode):
    """VirConv-T/S backbone: restated flow (LiDAR stream with shared rulebooks, MM stream, x-batched eval +
    decompose_tensor) == the reference's VirConv8x class run over the same oracle operators."""
    from oracle.backbone import VirConv8x
    g = np.load(os.path.join(GOLD, 'virconv_t_small.npz'))
    m = VirConv8x()
    fill_module(m, int(g['seed']))
    m.train(mode == 'train')
    arrays = {k.split(':')[2]: torch.from_numpy(g[k].copy()) for k in g.files if k.startswith(f'{mode}:in:')}
    kw = dict(aug_param=g[f'{mode}:aug']) if mode == 'train' else dict(transform_param=g[f'{mode}:aug'])
    with torch.no_grad(), golden_threads():
        o = m(arrays, 2, [scenes.Calib(), scenes.Calib()], **kw)
    n = 0
    for k in g.files:
        parts = k.split(':')
        if parts[0] != mode or parts[1] == 'in' or parts[1] == 'aug' or parts[3] != 'features':
            continue
        t = o[parts[1]] if parts[2] == 'out' else o[parts[1]][parts[2]]
        assert np.array_equal(t.indices.numpy(), g[f'{mode}:{parts[1]}:{parts[2]}:indices'])
        check_sampled_rows(t.features, g, k)
        n += 1
    assert n == (9 if mode == 'train' else 21)


# ---------------------------------------------------------------------------------------- StVD input point discard
def test_stvd_input_discard_oracle_matches_reference_golden():
    """tests/golden/stvd_input.npz holds outputs of the reference's OWN `DatasetTemplate.input_point_discard`
    (dataset.py:168-189) under seeded np.random (oracle/make_golden.py): the restatement must reproduce every row."""
    from oracle import stvd
    cases = stvd.golden_cases(np.load(os.path.join(GOLD, 'stvd_input.npz')))
    assert len(cases) >= 10
    for name, pts, bn, rate, seed, want in cases:
        out = stvd.input_point_discard(pts.copy(), bin_num=bn, rate=rate, rng=np.random.RandomState(seed))
        assert np.array_equal(out, want, equal_nan=True), name


def test_stvd_host_plan_of_the_product_matches_oracle():
    """The product's host-side half (position / per_bin arithmetic + RNG draws from the bin sizes alone) against the
    oracle's, including the python-slice corner (per_bin < 0) and empty bins."""
    from oracle import stvd
    from virconv_b200 import preprocess
    rng = np.random.default_rng(5)
    for trial in range(200):
        bn = int(rng.integers(1, 11))
        counts = rng.integers(0, 400, bn) * (rng.random(bn) > 0.2)
        n_all = int(counts.sum() + rng.integers(0, 50))        # points outside every bin still count in the total
        if n_all == 0:
            continue
        rate = float(rng.choice([0.8, 0.5, 0.95, 0.1]))
        seed = int(rng.integers(0, 1 << 30))
        far_to_near = [int(counts[bn - 1 - it]) for it in range(bn)]
        want = stvd.plan(far_to_near, n_all, bn, rate, np.random.RandomState(seed))
        segs, sel, n_out = preprocess._discard_plan(counts, n_all, bn, rate, np.random.RandomState(seed))
        assert [s[0] for s in segs] == [b for b, _ in want]
        total = 0
        for (b, base, cnt, sbase), (_, wsel) in zip(segs, want):
            assert base == total
            if wsel is None:
                assert sbase < 0 and cnt == int(counts[b])
            elif len(wsel) == 0:
                assert cnt == 0
            else:
                assert sbase >= 0 and np.array_equal(sel[sbase:sbase + cnt], wsel)
            total += cnt
        assert total == n_out


# ---------------------------------------------------------------------------------------- voxel-RoI pooling primitives
def test_pointnet2_restatement_against_a_vectorised_definition():
    """oracle/pointnet2.py walks cells like the reference kernel (voxel_query_gpu.cu:40-87); here the same answer from a
    definition that does not share its control flow: all neighbours of a query cell sorted by (dz, dy, dx), filtered by
    radius, first nsample kept, padded with the first."""
    from oracle import pointnet2 as o_pn
    rng = np.random.default_rng(4)
    B, shape = 2, (4, 12, 10)
    n = 150
    lin = np.sort(rng.choice(B * shape[0] * shape[1] * shape[2], n, replace=False))
    b, rem = lin // (shape[0] * shape[1] * shape[2]), lin % (shape[0] * shape[1] * shape[2])
    coords = np.stack([b, rem // (shape[1] * shape[2]), (rem // shape[2]) % shape[1], rem % shape[2]], 1).astype(np.int32)
    xyz = np.ascontiguousarray((coords[:, [3, 2, 1]] + 0.5).astype(np.float32) * np.float32(0.4))
    v2p = -np.ones((B,) + shape, np.int32)
    v2p[coords[:, 0], coords[:, 1], coords[:, 2], coords[:, 3]] = np.arange(n)
    m = 60
    pick = rng.integers(0, n, m)
    new_xyz = (xyz[pick] + rng.normal(0, 0.3, (m, 3))).astype(np.float32)
    new_coords = np.concatenate([coords[pick, :1], np.floor(new_xyz[:, [2, 1, 0]] / np.float32(0.4)).astype(np.int32)], 1)
    for rngs, radius, ns in (((1, 1, 1), 0.55, 4), ((2, 3, 1), 0.9, 8)):
        idx, empty = o_pn.voxel_query(rngs, radius, ns, xyz, new_xyz, new_coords, v2p)
        for q in range(m):
            d = coords[:, 1:].astype(np.int64) - new_coords[q, 1:].astype(np.int64)
            cand = np.nonzero((coords[:, 0] == new_coords[q, 0]) & (np.abs(d[:, 0]) <= rngs[0]) & (np.abs(d[:, 1]) <= rngs[1])
                              & (np.abs(d[:, 2]) <= rngs[2]))[0]
            cand = cand[np.lexsort((d[cand, 2], d[cand, 1], d[cand, 0]))]
            dist2 = ((xyz[cand].astype(np.float64) - new_xyz[q].astype(np.float64)) ** 2).sum(1)
            hits = cand[dist2 <= np.float64(np.float32(radius) * np.float32(radius))][:ns]
            if len(hits) == 0:
                assert empty[q] and not idx[q].any()
            else:
                want = np.full(ns, hits[0])
                want[:len(hits)] = hits
                assert not empty[q] and np.array_equal(idx[q], want), q
    # grouping and its gradient are transposes of each other:  <group(f), g> == <f, group_grad(g)>
    feats = rng.normal(size=(n, 6)).astype(np.float32)
    cnt_f = np.array([(coords[:, 0] == i).sum() for i in range(B)], np.int32)
    order = np.argsort(new_coords[:, 0], kind='stable')
    qb = new_coords[order, 0]
    cnt_q = np.array([(qb == i).sum() for i in range(B)], np.int32)
    starts = np.concatenate([[0], np.cumsum(cnt_f)[:-1]])
    lidx = (idx[order] - starts[qb][:, None]).astype(np.int32)
    lidx[empty[order]] = 0
    out = o_pn.group_points(feats, cnt_f, lidx, cnt_q)
    g = rng.normal(size=out.shape).astype(np.float32)
    back = o_pn.group_points_grad(g, lidx, cnt_q, cnt_f, n)
    assert abs(float((out.astype(np.float64) * g).sum()) - float((feats.astype(np.float64) * back).sum())) < 1e-3


def test_reference_pointnet2_kernels_build_into_oracle_ref():
    """oracle/ref_build.py compiles the reference's stand-alone CUDA sources where they lie; on a box without
    /root/reference the prebuilt library (if it travelled) is used as is."""
    import ctypes
    from oracle import ref_build
    lib = ref_build.build()
    if lib is None:
        pytest.skip('no /root/reference and no prebuilt oracle/_ref library')
    assert os.path.exists(lib)
    if torch.cuda.is_available() or os.path.exists('/usr/local/cuda/lib64/libcudart.so'):
        h = ctypes.CDLL(lib)
        for sym in ('ref_voxel_query', 'ref_group_points', 'ref_group_points_grad'):
            assert hasattr(h, sym)
