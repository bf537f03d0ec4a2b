"""Generate tests/golden/*.npz by importing the reference's OWN Python from /root/reference.
TEST INFRASTRUCTURE (see oracle/__init__.py).  Runs only in the build container (the GPU box has no
/root/reference); the fixtures it writes are committed.

What the reference can pin (it ships no tests and no spconv):
  * `index2uv` + `X_TRANS.backward_with_param` + `Calibration.*_cuda`      -> golden/index2uv.npz
  * `MeanVFE.forward`                                                    -> golden/mean_vfe.npz
  * the control flow of `NRConvBlock` / `VirConvL8x` (block order, RGB zeroing, channel concat,
    strides handed to index2uv, published outputs), executed by the reference's classes with the
    ORACLE's CPU sparse-conv operators standing in for the absent spconv package
                                                                         -> golden/virconv_l_small.npz
  * the StVD input point discard of `DatasetTemplate`                   -> golden/stvd_input.npz
  * the backbones' state_dict layout over spconv_compat (own process)    -> golden/reference_backbones.json
  * the stacked pointnet2 CUDA kernels, built into oracle/_ref (on a GPU) -> golden/roi_pool.npz
The sparse-conv arithmetic itself stays pinned only by the dense-conv property tests.

usage:  python -m oracle.make_golden [main | backbone_layout | roi_pool]
"""
from __future__ import annotations

import importlib
import os
import sys
import types

import numpy as np
import torch

REF = '/root/reference'
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')


class AttrDict(dict):
    __getattr__ = dict.__getitem__


def import_reference():
    """Import reference modules without running pcdet's package __init__s (they pull compiled ops)."""
    from . import spconv_cpu
    sys.modules.update(spconv_cpu.as_spconv_namespace())
    for name, rel in [('pcdet', 'pcdet'), ('pcdet.utils', 'pcdet/utils'), ('pcdet.datasets', 'pcdet/datasets'),
                      ('pcdet.datasets.augmentor', 'pcdet/datasets/augmentor'), ('pcdet.models', 'pcdet/models'),
                      ('pcdet.models.backbones_3d', 'pcdet/models/backbones_3d'),
                      ('pcdet.models.backbones_3d.vfe', 'pcdet/models/backbones_3d/vfe')]:
        pkg = types.ModuleType(name)
        pkg.__path__ = [os.path.join(REF, rel)]
        sys.modules[name] = pkg
    for stub in ('pcdet.utils.box_utils', 'pcdet.utils.box_np_ops'):
        sys.modules[stub] = types.ModuleType(stub)       # only needed by augmentor paths we never call
    bb = importlib.import_module('pcdet.models.backbones_3d.spconv_backbone')
    calib = importlib.import_module('pcdet.utils.calibration_kitti')
    importlib.import_module('pcdet.models.backbones_3d.vfe.vfe_template')
    vfe = importlib.import_module('pcdet.models.backbones_3d.vfe.mean_vfe')
    return bb, calib, vfe


def import_reference_dataset():
    """`pcdet/datasets/dataset.py` with its dataloader-side imports (augmentor, spconv voxel generator) stubbed: only the
    two pure-numpy StVD methods of DatasetTemplate are used."""
    for stub, names in (('pcdet.datasets.augmentor.data_augmentor', ['DataAugmentor']),
                        ('pcdet.datasets.processor', []),
                        ('pcdet.datasets.processor.data_processor', ['DataProcessor']),
                        ('pcdet.datasets.processor.point_feature_encoder', ['PointFeatureEncoder'])):
        m = types.ModuleType(stub)
        for n in names:
            setattr(m, n, object)
        sys.modules.setdefault(stub, m)
    return importlib.import_module('pcdet.datasets.dataset')


def stvd_cases():
    """(name, points [N, 8] float32, bin_num, rate, seed): virtual points of synthetic scenes + adversarial clouds."""
    from virconv_b200 import scenes
    cases = []
    for sid, nv in ((3, 20000), (4, 5000)):
        pts = scenes.make_points(sid, n_lidar=2048, n_virtual=nv)
        virt = np.ascontiguousarray(pts[pts[:, -1] == 1]).astype(np.float32)
        for bn, seed in ((2, 10 + sid), (10, 20 + sid)):
            cases.append((f'scene{sid}_bins{bn}', virt, bn, 0.8, seed))
    rng = np.random.default_rng(99)
    wide = rng.uniform(-10, 90, (4000, 8)).astype(np.float32)          # x < 0 (dropped) and x > 60 (last bin) present
    wide[::97, 0] = np.nan
    cases.append(('wide_bins10', wide, 10, 0.8, 31))
    cases.append(('wide_bins2_rate05', wide, 2, 0.5, 32))
    cases.append(('wide_bins7', wide, 7, 0.8, 33))                      # 60/7 is not exactly representable
    near = rng.uniform(0, 6, (1500, 8)).astype(np.float32)              # everything in the nearest bin
    cases.append(('near_bins10', near, 10, 0.8, 34))
    far = rng.uniform(55, 70, (1200, 8)).astype(np.float32)             # everything in the farthest bin
    cases.append(('far_bins10', far, 10, 0.8, 35))
    cases.append(('tiny_bins2', rng.uniform(0, 60, (7, 8)).astype(np.float32), 2, 0.8, 36))
    return cases


def stvd_golden():
    from . import stvd as o_stvd
    ds_mod = import_reference_dataset()
    ds = ds_mod.DatasetTemplate.__new__(ds_mod.DatasetTemplate)
    out, report = {}, []
    for name, pts, bn, rate, seed in stvd_cases():
        np.random.seed(seed)
        ref = ds.input_point_discard(pts.copy(), bin_num=bn, rate=rate)
        np.random.seed(seed)
        mine = o_stvd.input_point_discard(pts.copy(), bin_num=bn, rate=rate, rng=np.random)
        same = ref.shape == mine.shape and np.array_equal(ref, mine, equal_nan=True)
        report.append(f'StVD input discard {name}: N={pts.shape[0]} -> {ref.shape[0]} rows, restated == reference: {same}')
        assert same, name
        # the output rows are rows of the input cloud: stored as their row numbers, every cloud once
        cloud = name.split('_bins')[0]
        assert np.array_equal(out.setdefault(f'{cloud}:points', pts), pts, equal_nan=True), name
        row_of = {r.tobytes(): i for i, r in reversed(list(enumerate(pts)))}
        out[f'{name}:cloud'] = np.array(cloud)
        out[f'{name}:out_rows'] = np.array([row_of[r.tobytes()] for r in ref], dtype=np.int32).reshape(-1)
        assert np.array_equal(pts[out[f'{name}:out_rows']], ref, equal_nan=True), name
        out[f'{name}:meta'] = np.array([bn, seed], dtype=np.int64)
        out[f'{name}:rate'] = np.float64(rate)
    np.savez_compressed(os.path.join(OUT, 'stvd_input.npz'), **out)
    return report


def backbone_layout_golden():
    """tests/golden/reference_backbones.json: the reference's VirConvL8x / VirConv8x classes (spconv_backbone.py)
    constructed over `spconv_compat.install_as_spconv()` — state_dict entries in order as 'key (shape) dtype',
    num_point_features, sparse_shape and, per sparse convolution in module order, whether it has a bias."""
    import json
    from virconv_b200 import spconv_compat
    spconv_compat.install_as_spconv()
    for name, rel in [('pcdet', 'pcdet'), ('pcdet.utils', 'pcdet/utils'), ('pcdet.datasets', 'pcdet/datasets'),
                      ('pcdet.datasets.augmentor', 'pcdet/datasets/augmentor'), ('pcdet.models', 'pcdet/models'),
                      ('pcdet.models.backbones_3d', 'pcdet/models/backbones_3d')]:
        pkg = types.ModuleType(name)
        pkg.__path__ = [os.path.join(REF, rel)]
        sys.modules[name] = pkg
    for stub in ('pcdet.utils.box_utils', 'pcdet.utils.box_np_ops'):
        sys.modules[stub] = types.ModuleType(stub)
    bb = importlib.import_module('pcdet.models.backbones_3d.spconv_backbone')
    assert bb.spconv is spconv_compat
    cfgs = {'VirConvL8x': AttrDict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.1,
                                   NUM_FILTERS=[16, 32, 64, 64]),
            'VirConv8x': AttrDict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.15,
                                  NUM_FILTERS=[16, 32, 64, 64], MM=True)}
    out = {}
    for name, cfg in cfgs.items():
        r = getattr(bb, name)(model_cfg=cfg, input_channels=8, grid_size=np.array([1408, 1600, 80]))
        out[name] = {'state_dict': [f'{k} {tuple(v.shape)} {v.dtype}' for k, v in r.state_dict().items()],
                     'num_point_features': r.num_point_features, 'sparse_shape': [int(s) for s in r.sparse_shape],
                     'conv_has_bias': [m.bias is not None for m in r.modules()
                                       if isinstance(m, spconv_compat.SparseConvolution)]}
    path = os.path.join(OUT, 'reference_backbones.json')
    with open(path, 'w') as f:
        json.dump(out, f, indent=1)
        f.write('\n')
    return path


def roi_pool_golden():
    """tests/golden/roi_pool.npz: the reference's own stacked pointnet2 kernels (oracle/_ref, oracle/ref_build.py) on the
    full-size cases of oracle/pointnet2.py — voxel query, grouping of features and of xyz, grouping gradient.  Needs a GPU.
    Stored per case: the empty-ball mask, seeded row samples of every output, the largest gradient magnitude, and SHA-256
    digests of the complete index and grouping outputs (both are exact: integer indices and pure gathers)."""
    import ctypes
    from . import pointnet2 as o_pn
    from . import ref_build
    from .testing import sha256_bytes as sha256
    lib = ctypes.CDLL(ref_build.build())
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    d = lambda a: torch.from_numpy(a).cuda()
    xyz, xyz_cnt, new_xyz, new_cnt, new_coords, v2p = o_pn.scene(1)
    M, N, C = new_coords.shape[0], xyz.shape[0], o_pn.ROI_CHANNELS
    t_xyz, t_new_xyz, t_coords, t_v2p, cnt_f, cnt_q = d(xyz), d(new_xyz), d(new_coords), d(v2p), d(xyz_cnt), d(new_cnt)
    starts = np.concatenate([[0], np.cumsum(xyz_cnt)[:-1]]).astype(np.int32)
    out = {}
    for ci, (max_range, radius, nsample) in enumerate(o_pn.ROI_CASES):
        key = o_pn.roi_case_key(max_range, radius, nsample)
        feats, grad_out = o_pn.roi_case_data(max_range, radius, nsample, N, M)
        # the kernel + the two lines of VoxelQuery.forward around it (voxel_query_utils.py:32-39)
        ridx = torch.zeros((M, nsample), dtype=torch.int32, device='cuda')
        torch.cuda.synchronize()
        lib.ref_voxel_query(M, v2p.shape[1], v2p.shape[2], v2p.shape[3], nsample, ctypes.c_float(radius), *max_range,
                            p(t_new_xyz), p(t_xyz), p(t_coords), p(t_v2p), p(ridx))
        torch.cuda.synchronize()
        empty = ridx[:, 0] == -1
        ridx[empty] = 0
        # grouping forward / backward as VoxelQueryAndGrouping.forward (:80-99) calls it: batch-local indices
        lidx = (ridx.view(len(xyz_cnt), -1, nsample) - d(starts).view(-1, 1, 1)).view(-1, nsample)
        lidx[empty] = 0
        lidx = lidx.contiguous()
        fc, go = d(feats), d(grad_out)
        rgf = torch.empty((M, C, nsample), device='cuda')
        rgx = torch.empty((M, 3, nsample), device='cuda')
        rg = torch.zeros((N, C), device='cuda')
        torch.cuda.synchronize()
        lib.ref_group_points(len(xyz_cnt), M, C, nsample, p(fc), p(cnt_f), p(lidx), p(cnt_q), p(rgf))
        lib.ref_group_points(len(xyz_cnt), M, 3, nsample, p(t_xyz), p(cnt_f), p(lidx), p(cnt_q), p(rgx))
        lib.ref_group_points_grad(len(xyz_cnt), M, C, N, nsample, p(go), p(lidx), p(cnt_q), p(cnt_f), p(rg))
        torch.cuda.synchronize()
        ridx, empty, rgf, rgx, rg = (t.cpu().numpy() for t in (ridx, empty, rgf, rgx, rg))
        rng = np.random.default_rng(300 + ci)
        idx_rows = np.sort(rng.choice(M, 256, replace=False))
        group_rows = np.sort(rng.choice(M, 8, replace=False))
        # row 0 of every sample collects the gradient of all empty balls: always in the sample
        grad_rows = np.union1d(starts, rng.choice(N, 128, replace=False))
        out.update({f'{key}:empty': np.packbits(empty), f'{key}:idx_rows': idx_rows, f'{key}:idx': ridx[idx_rows],
                    f'{key}:idx_sha256': np.array(sha256(ridx)), f'{key}:group_rows': group_rows,
                    f'{key}:features': rgf[group_rows], f'{key}:features_sha256': np.array(sha256(rgf)),
                    f'{key}:xyz': rgx[group_rows], f'{key}:xyz_sha256': np.array(sha256(rgx)),
                    f'{key}:grad_rows': grad_rows, f'{key}:grad': rg[grad_rows],
                    f'{key}:grad_absmax': np.float32(np.abs(rg).max())})
    path = os.path.join(OUT, 'roi_pool.npz')
    np.savez_compressed(path, **out)
    return path


def main():
    from virconv_b200 import scenes
    from . import index2uv as o_uv
    from .testing import GOLDEN_THREADS, fill_module, sampled_rows
    from .backbone import VirConvL8x as OracleL

    bb, calib_mod, vfe_mod = import_reference()
    torch.set_num_threads(GOLDEN_THREADS)
    os.makedirs(OUT, exist_ok=True)
    calib_dict = {'P2': scenes.P2, 'R0': scenes.R0, 'Tr_velo2cam': scenes.TR_VELO_TO_CAM}
    report = []

    # ---- index2uv ---------------------------------------------------------------------------
    rng = np.random.default_rng(7)
    cases = {}
    n_total = n_diff = 0
    for ci, (stride, with_aug) in enumerate([(1, False), (2, True), (4, True), (8, False), (8, True)]):
        B = 2
        shape = [81 // stride + 1, 1600 // stride, 1408 // stride]
        n = 3000
        idx = np.stack([rng.integers(0, B, n), rng.integers(0, shape[0], n), rng.integers(0, shape[1], n),
                        rng.integers(0, shape[2], n)], axis=1).astype(np.int32)
        idx = idx[np.argsort(idx[:, 0], kind='stable')]
        aug = None
        if with_aug:
            aug = np.stack([rng.uniform(-0.785, 0.785, B), rng.integers(0, 2, B).astype(np.float64),
                            rng.uniform(0.95, 1.05, B)], axis=1).astype(np.float32)
        ref_calibs = [calib_mod.Calibration(dict(calib_dict)) for _ in range(B)]
        tp = None if aug is None else torch.from_numpy(aug.copy())
        uv_ref, _ = bb.index2uv(torch.from_numpy(idx.copy()), B, ref_calibs, stride, bb.X_TRANS(), tp)
        uv_ref = uv_ref.int().numpy()
        uv_or = o_uv.index2uv(idx, B, [scenes.Calib() for _ in range(B)], stride, aug)
        d = int((uv_ref != uv_or).any(axis=1).sum())
        n_total += n
        n_diff += d
        maxd = int(np.abs(uv_ref.astype(np.int64) - uv_or).max())
        report.append(f'index2uv case {ci} stride={stride} aug={with_aug}: {d}/{n} rows differ from the '
                      f'reference torch evaluation (max |delta| = {maxd} px-cell)')
        cases[f'idx{ci}'] = idx
        cases[f'uv{ci}'] = uv_ref
        cases[f'stride{ci}'] = np.int32(stride)
        cases[f'aug{ci}'] = aug if aug is not None else np.zeros((0, 3), np.float32)
    np.savez_compressed(os.path.join(OUT, 'index2uv.npz'), n_cases=np.int32(5), **cases)

    # ---- MeanVFE ----------------------------------------------------------------------------
    pts = scenes.mask_points_by_range(scenes.make_points(3, n_lidar=2048, n_virtual=6000))
    vox, coords, num = scenes.voxelize_first_come(pts, max_voxels=3000)
    vfe = vfe_mod.MeanVFE(AttrDict(MODEL='max'), 8)
    bd = {'voxels': torch.from_numpy(vox), 'voxel_num_points': torch.from_numpy(num.astype(np.float32))}
    ref_feat = vfe(bd)['voxel_features'].numpy()
    mine = scenes.mean_vfe(vox, num, 'max')
    report.append(f'MeanVFE: max |ref - restated| = {np.abs(ref_feat - mine).max():.3e} over {vox.shape[0]} voxels')
    np.savez_compressed(os.path.join(OUT, 'mean_vfe.npz'), voxels=vox, num=num, coords=coords, features=ref_feat)

    # ---- VirConvL8x control flow (reference classes over the oracle operators) ---------------
    # index2uv truncates float pixel coordinates; a voxel centre that projects within an ulp of an
    # integer can land in a different pixel cell under the reference's BLAS evaluation than under the
    # oracle's fixed left-to-right order (measured: about 1 voxel in 50 000).  The fixture uses the first
    # scene pair on which every voxel agrees, and the report records the pairs that were skipped.
    uv_log = []
    ref_index2uv = bb.index2uv

    def logged_index2uv(*a, **k):
        r = ref_index2uv(*a, **k)
        uv_log.append(r[0].int().numpy().copy())
        return r
    bb.index2uv = logged_index2uv
    cfg = AttrDict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.1,
                   NUM_FILTERS=[16, 32, 64, 64])
    ref_model = bb.VirConvL8x(cfg, 8, np.array([1408, 1600, 80]))
    fill_module(ref_model, 666)
    ora_model = OracleL()
    ora_model.load_state_dict(ref_model.state_dict())
    for first_scene in range(11, 40, 2):
        batch = scenes.make_batch([first_scene, first_scene + 1], n_lidar=512, n_virtual=600, max_voxels=350,
                                  training=True)
        out, lines, flips = {}, [], 0
        for mode in ('eval', 'train'):
            ref_model.train(mode == 'train')
            ora_model.train(mode == 'train')
            ref_calibs = [calib_mod.Calibration(dict(calib_dict)) for _ in range(batch.batch_size)]
            bd = {'voxel_features': torch.from_numpy(batch.voxel_features.copy()),
                  'voxel_coords': torch.from_numpy(batch.voxel_coords.copy()), 'batch_size': batch.batch_size,
                  'calib': ref_calibs, 'aug_param': torch.from_numpy(batch.aug_param.copy())}
            del uv_log[:]
            trace = []
            np.random.seed(0)
            with torch.no_grad():
                r = ref_model(bd)
                o = ora_model(torch.from_numpy(batch.voxel_features.copy()),
                              torch.from_numpy(batch.voxel_coords.copy()), batch.batch_size, batch.calib,
                              batch.aug_param, trace=trace)
            flips += sum(int((a != t['uv']).any(axis=1).sum()) for a, t in zip(uv_log, trace))
            named = dict(r['multi_scale_3d_features'])
            named['out'] = r['encoded_spconv_tensor']
            for k, t in named.items():
                same_idx = np.array_equal(t.indices.numpy(), o[k].indices.numpy())
                err = float((t.features - o[k].features).abs().max() / t.features.abs().max())
                lines.append(f'VirConvL8x[{mode}] {k}: N={t.features.shape[0]} C={t.features.shape[1]} '
                             f'indices identical={same_idx} rel err restated-vs-reference-flow={err:.2e}')
                out.update(sampled_rows(f'{mode}_{k}_features', t.features.numpy()))
                out[f'{mode}_{k}_indices'] = t.indices.numpy().astype(np.int32)
        if flips == 0:
            report.append(f'VirConvL8x fixture: scenes ({first_scene},{first_scene + 1}), no pixel-cell flips')
            report.extend(lines)
            break
        report.append(f'VirConvL8x: scenes ({first_scene},{first_scene + 1}) skipped, {flips} voxel(s) flip pixel cell')
    np.savez_compressed(os.path.join(OUT, 'virconv_l_small.npz'), voxel_features=batch.voxel_features,
                        voxel_coords=batch.voxel_coords, aug_param=batch.aug_param, seed=np.int32(666), **out)

    # ---- VirConv8x control flow (VirConv-T/S: LiDAR stream + MM stream, train and x-batched eval) ---------
    from .backbone import VirConv8x as OracleT
    bb.index2uv = ref_index2uv
    cfg8 = AttrDict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.15,
                    NUM_FILTERS=[16, 32, 64, 64], MM=True)
    ref8 = bb.VirConv8x(cfg8, 8, np.array([1408, 1600, 80]))
    fill_module(ref8, 667)
    ora8 = OracleT()
    ora8.load_state_dict(ref8.state_dict())
    gold8 = {}
    for mode in ('train', 'eval'):
        training = mode == 'train'
        for first_scene in range(21, 60, 2):
            bm = scenes.make_batch_mm([first_scene, first_scene + 1], n_lidar=256, n_virtual=300, max_voxels=110,
                                      training=training, rot_num=3)
            fill_module(ref8, 667)                       # train-mode passes move the BN running statistics
            ora8.load_state_dict(ref8.state_dict())
            ref8.train(training)
            ora8.train(training)
            bd = {k: torch.from_numpy(v.copy()) for k, v in bm.arrays.items()}
            bd.update(batch_size=bm.batch_size, calib=[calib_mod.Calibration(dict(calib_dict)) for _ in range(bm.batch_size)])
            if training:
                bd['aug_param'] = torch.from_numpy(bm.aug_param.copy())
            else:
                bd['transform_param'] = torch.from_numpy(bm.transform_param.copy())
            with torch.no_grad():
                r = ref8(bd)
                o = ora8({k: torch.from_numpy(v.copy()) for k, v in bm.arrays.items()}, bm.batch_size, bm.calib,
                         aug_param=bm.aug_param, transform_param=bm.transform_param)
            worst, same, tensors = 0.0, True, {}
            for key in sorted(o.keys()):
                for name, t in ([('out', o[key])] if not isinstance(o[key], dict) else o[key].items()):
                    rt = r[key] if not isinstance(o[key], dict) else r[key][name]
                    if t is None:
                        assert rt is None
                        continue
                    same &= np.array_equal(t.indices.numpy(), rt.indices.numpy())
                    if same:
                        worst = max(worst, float((t.features - rt.features).abs().max() / rt.features.abs().max().clamp_min(1e-30)))
                    tensors.update(sampled_rows(f'{mode}:{key}:{name}:features', rt.features.numpy()))
                    tensors[f'{mode}:{key}:{name}:indices'] = rt.indices.numpy().astype(np.int32)
            if same and worst == 0.0:
                report.append(f'VirConv8x[{mode}] fixture: scenes ({first_scene},{first_scene + 1}), {len(tensors) // 5} published '
                              f'tensors, indices identical, restated-vs-reference-flow rel err 0')
                gold8.update(tensors)
                for k, v in bm.arrays.items():
                    gold8[f'{mode}:in:{k}'] = v
                gold8[f'{mode}:aug'] = bm.aug_param if training else bm.transform_param
                break
            report.append(f'VirConv8x[{mode}]: scenes ({first_scene},{first_scene + 1}) skipped (pixel-cell flip or mismatch: '
                          f'same_idx={same} err={worst:.2e})')
    np.savez_compressed(os.path.join(OUT, 'virconv_t_small.npz'), seed=np.int32(667), **gold8)

    # ---- StVD input point discard (dataset.py:120-189), the reference's own methods under a seeded np.random --------
    report += stvd_golden()

    with open(os.path.join(OUT, 'REPORT.txt'), 'w') as f:
        f.write('\n'.join(report) + '\n')
    print('\n'.join(report))


if __name__ == '__main__':
    what = sys.argv[1] if len(sys.argv) > 1 else 'main'
    print({'main': main, 'backbone_layout': backbone_layout_golden, 'roi_pool': roi_pool_golden}[what]())
