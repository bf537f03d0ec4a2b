"""Drop-in boundary against the reference's OWN unmodified files: its backbone classes
(`pcdet/models/backbones_3d/spconv_backbone.py`) and the dataloader's `VoxelGeneratorWrapper`
(`pcdet/datasets/processor/data_processor.py:13-59`) construct and run over `spconv_compat.install_as_spconv()`
(SURVEY §8b items 1-3).  What the reference's classes produce over the shim is stored in
tests/golden/reference_backbones.json (oracle/make_golden.py backbone_layout); the whole-detector build needs the
reference's `pcdet` package itself and runs only where a copy of it is found."""
import ast
import json
import os
import sys
import types

import numpy as np
import pytest

REF = '/root/reference'
needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'pcdet')), reason='the reference pcdet package is not present')
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


class AttrDict(dict):
    __getattr__ = dict.__getitem__


_OURS = ('pcdet', 'spconv', 'cumm', 'easydict', 'tensorboardX', 'prefetch_generator', 'skimage')


def _restore_modules(saved):
    """Drop the reference's modules and the stand-ins registered for them (third-party packages imported along the way, e.g.
    cv2, stay: they do not support being imported twice)."""
    for k in list(sys.modules):
        if k not in saved and k.split('.')[0] in _OURS:
            del sys.modules[k]
    for k, v in saved.items():
        if k.split('.')[0] in _OURS:
            sys.modules[k] = v


@pytest.fixture()
def spconv_shims():
    """`spconv` / `cumm` resolved to this repo's shims; removed from sys.modules again afterwards."""
    saved = dict(sys.modules)
    from virconv_b200 import spconv_compat
    spconv_compat.install_as_spconv()
    try:
        yield
    finally:
        _restore_modules(saved)


def test_reference_backbones_construct_over_spconv_compat():
    """Our classes against the reference's classes built over the shim (golden): state_dict keys in order, shapes and
    dtypes, num_point_features, sparse_shape, bias-free sparse convolutions; a checkpoint of the reference's layout loads."""
    import torch
    from virconv_b200 import backbone as ours
    from virconv_b200 import spconv_compat
    gold = json.load(open(os.path.join(GOLD, 'reference_backbones.json')))
    cfg_l = dict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.1, NUM_FILTERS=[16, 32, 64, 64])
    cfg_t = dict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.15, NUM_FILTERS=[16, 32, 64, 64],
                 MM=True)
    for name, cfg in (('VirConvL8x', cfg_l), ('VirConv8x', cfg_t)):
        g = gold[name]
        o = getattr(ours, name)(cfg, 8, [1408, 1600, 80])
        os_ = o.state_dict()
        assert [f'{k} {tuple(v.shape)} {v.dtype}' for k, v in os_.items()] == g['state_dict'], name
        assert o.num_point_features == g['num_point_features'], name
        assert list(o.sparse_shape) == g['sparse_shape'], name
        # a checkpoint of the reference class's layout loads into ours (weight layout (C_out, *k, C_in))
        ckpt = {}
        for entry in g['state_dict']:
            k, rest = entry.split(' ', 1)
            shape, dtype = rest.rsplit(' ', 1)
            ckpt[k] = torch.ones(ast.literal_eval(shape), dtype=getattr(torch, dtype.split('.')[1]))
        o.load_state_dict(ckpt)
        convs = [m for m in o.modules() if isinstance(m, spconv_compat.SparseConvolution)]
        assert [m.bias is not None for m in convs] == g['conv_has_bias'], name
        assert len(convs) == (20 if name == 'VirConvL8x' else 31), (name, len(convs))


def test_reference_voxel_generator_wrapper_runs_over_the_shims(spconv_shims):
    """The wrapper's spconv-2 branch over the shims: `spconv.utils` offers neither VoxelGeneratorV2 nor VoxelGenerator, so it
    builds `Point2VoxelCPU3d(vsize_xyz=, coors_range_xyz=, num_point_features=, max_num_points_per_voxel=, max_num_voxels=)`,
    calls `point_to_voxel(tv.from_numpy(points))` and takes `.numpy()` of the three outputs."""
    from virconv_b200 import scenes
    with pytest.raises(ImportError):
        from spconv.utils import VoxelGeneratorV2  # noqa: F401
    with pytest.raises(ImportError):
        from spconv.utils import VoxelGenerator  # noqa: F401
    from spconv.utils import Point2VoxelCPU3d
    import cumm.tensorview as tv
    gen = Point2VoxelCPU3d(vsize_xyz=[0.05, 0.05, 0.05], coors_range_xyz=[0, -40, -3, 70.4, 40, 1], num_point_features=8,
                           max_num_points_per_voxel=5, max_num_voxels=4000)
    pts = scenes.make_points(3, n_lidar=2048, n_virtual=6000)
    voxels, coords, num = (t.numpy() for t in gen.point_to_voxel(tv.from_numpy(pts)))
    v0, c0, n0 = scenes.voxelize_first_come(pts, max_points=5, max_voxels=4000)
    assert voxels.shape == (4000, 5, 8) and coords.shape == (4000, 3) and num.shape == (4000,)
    assert np.array_equal(voxels, v0) and np.array_equal(coords, c0) and np.array_equal(num, n0)
    assert coords[:, 0].max() < 80 and coords[:, 2].max() > 80 and coords[:, 2].max() < 1408         # zyx order


@needs_reference
@pytest.mark.parametrize('yaml_name', ['VirConv-L.yaml', 'VirConv-T.yaml', 'VirConv-S.yaml'])
def test_reference_detector_builds_under_reference_env(yaml_name, monkeypatch):
    """SURVEY §8f-2: with `reference_env.install()` the reference's unmodified `pcdet` package imports on this stack (py3.12,
    torch 2.11, no spconv / cumm / compiled pcdet.ops) and `build_network` constructs the whole detector of the VirConv
    YAMLs (VFE, 3-D backbone — this package's fused class through the registry —, BEV backbone, dense head, TEDMHead).
    The reference calls `.cuda()` while constructing its anchor generator; this container has no GPU, so that one call is
    neutralised for the test."""
    import torch
    saved = dict(sys.modules)
    cwd = os.getcwd()
    try:
        import virconv_b200.reference_env as renv
        renv.install(reference_root=REF, use_fused_backbones=True)
        from pcdet.config import cfg, cfg_from_yaml_file
        from pcdet.models import build_network
        os.chdir(os.path.join(REF, 'tools'))              # the YAMLs use paths relative to tools/ (SURVEY App. D)
        cfg_from_yaml_file(os.path.join('cfgs', 'models', 'kitti', yaml_name), cfg)
        pcr = np.array(cfg.DATA_CONFIG.POINT_CLOUD_RANGE, dtype=np.float32)
        vs = [p.VOXEL_SIZE for p in cfg.DATA_CONFIG.DATA_PROCESSOR if p.NAME == 'transform_points_to_voxels'][0]
        grid = np.round((pcr[3:6] - pcr[0:3]) / np.array(vs)).astype(np.int64)
        ds = types.SimpleNamespace(class_names=cfg.CLASS_NAMES, point_feature_encoder=types.SimpleNamespace(num_point_features=8),
                                   grid_size=grid, voxel_size=vs, point_cloud_range=pcr, depth_downsample_factor=None,
                                   test_flip=False, rot_num=1)
        monkeypatch.setattr(torch.Tensor, 'cuda', lambda self, *a, **k: self)
        model = build_network(model_cfg=cfg.MODEL, num_class=len(cfg.CLASS_NAMES), dataset=ds)
        from virconv_b200 import backbone as ours
        want = ours.VirConvL8x if yaml_name == 'VirConv-L.yaml' else ours.VirConv8x
        assert type(model.backbone_3d) is want
        names = [type(m).__name__ for m in model.module_list]
        assert names[0] == 'MeanVFE' and 'HeightCompression' in names and names[-1] in ('TEDMHead', 'TEDSHead'), names
        keys = list(model.state_dict())
        assert any(k.startswith('backbone_3d.vir_conv1.d3_conv1.0.weight') for k in keys)
        assert sum(p.numel() for p in model.backbone_3d.parameters()) in (425856, 1114624)       # SURVEY App. A
    finally:
        os.chdir(cwd)
        _restore_modules(saved)


def test_points_in_boxes_cpu_restatement():
    """reference_env's torch restatement of roiaware_pool3d_cuda.points_in_boxes_cpu against the geometric definition
    (src/roiaware_pool3d.cpp:106-140: z within +-dz/2 of the box CENTRE, local x/y strictly inside after rotating by -heading)."""
    import torch
    from virconv_b200.reference_env import _points_in_boxes_cpu
    g = torch.Generator().manual_seed(0)
    boxes = torch.tensor([[10.0, 2.0, -1.0, 4.0, 2.0, 1.5, 0.3], [20.0, -5.0, -0.5, 3.0, 1.6, 1.4, -1.2]])
    pts = torch.rand((500, 3), generator=g) * torch.tensor([30.0, 20.0, 4.0]) + torch.tensor([0.0, -10.0, -3.0])
    out = torch.zeros((2, 500), dtype=torch.int32)
    _points_in_boxes_cpu(boxes, pts, out)
    for b in range(2):
        x, y, z, dx, dy, dz, h = [float(v) for v in boxes[b]]
        for i in range(500):
            px, py, pz = [float(v) for v in pts[i]]
            c, s = np.cos(-h), np.sin(-h)
            lx = (px - x) * c - (py - y) * s
            ly = (px - x) * s + (py - y) * c
            inside = abs(pz - z) <= dz / 2 and abs(lx) < dx / 2 and abs(ly) < dy / 2
            assert int(out[b, i]) == int(inside)
