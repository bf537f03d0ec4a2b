"""GPU parity tests, backbone level: VirConvL8x on the B200 kernels against the CPU oracle and against the
golden fixture produced by the reference's own Python (tests/golden/virconv_l_small.npz)."""
import os

import numpy as np
import pytest
import torch

from oracle.backbone import VirConvL8x as OracleL
from oracle.testing import check_sampled_rows, fill_module, rel_err
from oracle import rulebook as orb

pytestmark = pytest.mark.gpu
TOL = 1e-4
CFG = dict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.1, NUM_FILTERS=[16, 32, 64, 64])
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _models(discard_mode='spconv2_compat'):
    from virconv_b200.backbone import VirConvL8x
    m = VirConvL8x(CFG, 8, [1408, 1600, 80], discard_mode=discard_mode)
    fill_module(m, 666)
    o = OracleL(discard_mode=discard_mode)
    o.load_state_dict(m.state_dict())
    return m.to('cuda:0'), o


def _run_gpu(model, vf, vc, bs, calib, aug, keep=None):
    bd = {'voxel_features': torch.from_numpy(vf.copy()).cuda(), 'voxel_coords': torch.from_numpy(vc.copy()).cuda(),
          'batch_size': bs, 'calib': calib}
    if aug is not None:
        bd['aug_param'] = torch.from_numpy(aug.copy())
    if keep is not None:
        bd['stvd_keep_rows'] = keep
    out = model(bd)
    named = dict(out['multi_scale_3d_features'])
    named['out'] = out['encoded_spconv_tensor']
    return named, out


@pytest.mark.parametrize('mode', ['eval', 'train'])
def test_virconv_l_matches_reference_golden(lib_built, mode):
    from virconv_b200 import scenes
    g = np.load(os.path.join(GOLD, 'virconv_l_small.npz'))
    model, _ = _models()
    model.train(mode == 'train')
    calib = [scenes.Calib(), scenes.Calib()]
    with torch.no_grad():
        named, _ = _run_gpu(model, g['voxel_features'], g['voxel_coords'], 2, calib, g['aug_param'])
    for k, t in named.items():
        assert np.array_equal(t.indices.cpu().numpy(), g[f'{mode}_{k}_indices']), k
        check_sampled_rows(t.features, g, f'{mode}_{k}_features', TOL)


@pytest.mark.parametrize('training', [False, True])
def test_virconv_l_forward_backward_vs_oracle(lib_built, training):
    """BASELINE config 1 shape of check: one LiDAR-only scene + one fused scene, rulebooks + features + grads."""
    from virconv_b200 import scenes
    batch = scenes.make_batch([0, 5], n_lidar=4096, n_virtual=6000, max_voxels=6000, training=training)
    model, ref = _models()
    model.train(training)
    ref.train(training)
    named, out = _run_gpu(model, batch.voxel_features, batch.voxel_coords, 2, batch.calib, batch.aug_param)
    trace = []
    o = ref(torch.from_numpy(batch.voxel_features.copy()), torch.from_numpy(batch.voxel_coords.copy()), 2, batch.calib,
            batch.aug_param, trace=trace)
    for k, t in named.items():
        assert np.array_equal(t.indices.cpu().numpy(), o[k].indices.numpy()), k
        assert rel_err(t.features.detach().cpu(), o[k].features.detach()) < TOL, k
        assert np.all(np.diff(t.indices[:, 0].cpu().numpy()) >= 0)
    # rulebooks of every layer, bit exact in canonical form (cached in the shared indice_dict under the reference's keys)
    d = named['x_conv1'].indice_dict
    od = o['x_conv1'].indice_dict
    n_checked = 0
    for key, rb in d.items():
        if isinstance(key, str) and key in od:
            assert np.array_equal(rb.nbr.cpu().numpy(), od[key]['nbr_np']), key
            n_checked += 1
    assert n_checked >= 8
    loss = sum(t.features.mean() for t in named.values())
    loss.backward()
    rloss = sum(o[k].features.mean() for k in named)
    rloss.backward()
    assert abs(float(loss) - float(rloss)) < 1e-4 * max(1.0, abs(float(rloss)))
    gp = dict(model.named_parameters())
    worst = 0.0
    for name, p in ref.named_parameters():
        e = rel_err(gp[name].grad.cpu(), p.grad)
        worst = max(worst, e)
        assert e < 2e-3, (name, e)
    print('worst parameter-grad rel err', worst)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('training', [True, False])
def test_plan_executor_matches_module_path(lib_built, precision, training):
    """The native plan executor (csrc/executor.cu: one C-ABI call per forward / backward, index ops on a side stream)
    launches the same kernels as the per-operator module path: published tensors, rulebooks, parameter gradients and
    BatchNorm running statistics must agree (up to the order of the float64 / scatter atomics)."""
    import copy
    from virconv_b200 import scenes, executor
    from virconv_b200 import spconv_compat as spc
    batch = scenes.make_batch([11, 12], n_lidar=4096, n_virtual=9000, max_voxels=7000, training=training)
    model, _ = _models()
    spc.set_precision(model, precision)
    model.train(training)
    twin = copy.deepcopy(model)
    res = {}
    for name, m, flag in (('plan', model, True), ('module', twin, False)):
        executor.ENABLED = flag
        try:
            named, out = _run_gpu(m, batch.voxel_features, batch.voxel_coords, 2, batch.calib, batch.aug_param)
            loss = sum(t.features.mean() for t in named.values())
            loss.backward()
            torch.cuda.synchronize()
        finally:
            executor.ENABLED = True
        res[name] = (named, float(loss), m)
    assert int(ops_err_flag()) == 0
    (pn, pl, pm), (mn, ml, mm) = res['plan'], res['module']
    assert isinstance(pn['x_conv1'].indice_dict, executor.LazyIndiceDict)
    for k in pn:
        assert torch.equal(pn[k].indices, mn[k].indices), k
        assert pn[k].spatial_shape == mn[k].spatial_shape
        assert rel_err(pn[k].features.detach().cpu(), mn[k].features.detach().cpu()) < 1e-5, k
    for key, rb in mn['x_conv1'].indice_dict.items():
        if isinstance(key, str):
            prb = pn['x_conv1'].indice_dict[key]
            assert torch.equal(prb.nbr, rb.nbr), key
            assert torch.equal(prb.pair_num, rb.pair_num), key
            if rb.nbr_bwd is not None:
                assert torch.equal(prb.nbr_bwd, rb.nbr_bwd), key
    assert abs(pl - ml) < 1e-5 * max(1.0, abs(ml))
    gm = dict(mm.named_parameters())
    for name, p in pm.named_parameters():
        assert p.grad is not None, name
        if precision == 'bf16':
            # the scatter-dgrad / weight-gradient atomics' order differs run to run and a 1-ulp change can flip a bf16 rounding
            # downstream: two runs of the SAME path differ by up to 6e-3 of the largest element (profiles/diag_graph_vs_exact_r2.txt)
            a, b = p.grad.double().cpu(), gm[name].grad.double().cpu()
            assert float((a - b).norm() / b.norm().clamp_min(1e-30)) < 1e-2, name
            assert rel_err(p.grad.cpu(), gm[name].grad.cpu()) < 3e-2, name
        else:
            assert rel_err(p.grad.cpu(), gm[name].grad.cpu()) < 2e-4, name
    bm = dict(mm.named_buffers())
    for name, b in pm.named_buffers():
        assert torch.allclose(b.float().cpu(), bm[name].float().cpu(), rtol=1e-5, atol=1e-7), name


def ops_err_flag():
    from virconv_b200 import ops
    return ops.tc_error_flag(torch.device('cuda:0')).item()


def test_plan_executor_partial_loss_and_single_stream(lib_built):
    """Loss on ONE published tensor only (the others get no gradient: conv_out's parameters must come back as zeros),
    and the single-stream mode of the executor."""
    from virconv_b200 import scenes, executor
    batch = scenes.make_batch([21, 22], n_lidar=2048, n_virtual=4000, max_voxels=3000, training=True)
    model, ref = _models()
    model.train()
    ref.train()
    executor.TWO_STREAMS = False
    try:
        named, _ = _run_gpu(model, batch.voxel_features, batch.voxel_coords, 2, batch.calib, batch.aug_param)
        named['x_conv4'].features.square().mean().backward()
    finally:
        executor.TWO_STREAMS = True
    o = ref(torch.from_numpy(batch.voxel_features.copy()), torch.from_numpy(batch.voxel_coords.copy()), 2, batch.calib,
            batch.aug_param)
    o['x_conv4'].features.square().mean().backward()
    gp = dict(model.named_parameters())
    for name, p in ref.named_parameters():
        g = gp[name].grad
        if name.startswith('conv_out'):
            assert g is not None and float(g.abs().max()) == 0.0, name
        else:       # squared loss: more weight on the few pre-activations whose ReLU mask flips between CPU and GPU sums
            assert rel_err(g.cpu(), p.grad) < 5e-3, name


def test_virconv_l_paper_discard(lib_built):
    """StVD layer discard really applied (paper mode), kept rows supplied by the host RNG like the reference."""
    from virconv_b200 import scenes
    batch = scenes.make_batch([3, 4], n_lidar=2048, n_virtual=3000, max_voxels=3000, training=True)
    model, ref = _models('paper')
    model.train()
    ref.train()
    # row counts per stage come from the oracle run with the same keep lists (generated progressively)
    rng = np.random.default_rng(0)
    keep = []
    # first run the oracle stage by stage to learn N per stage
    from oracle import backbone as ob
    feats = torch.from_numpy(batch.voxel_features.copy())
    feats[:, 4:7] = 0
    x = ob.spconv.SparseConvTensor(feats, torch.from_numpy(batch.voxel_coords).int(), ref.sparse_shape, 2)
    with torch.no_grad():
        for li, (blk, stride) in enumerate([(ref.vir_conv1, 1), (ref.vir_conv2, 2), (ref.vir_conv3, 4)]):
            x = blk(x, 2, batch.calib, stride, batch.aug_param)
            n = x.features.shape[0]
            keep.append(np.sort(rng.permutation(n)[:int(n * 0.9)]))
            x = ob.discard_rows(x, keep[-1])
    fill_module(ref, 666)
    model.load_state_dict(ref.state_dict())
    named, _ = _run_gpu(model, batch.voxel_features, batch.voxel_coords, 2, batch.calib, batch.aug_param, keep)
    o = ref(torch.from_numpy(batch.voxel_features.copy()), torch.from_numpy(batch.voxel_coords.copy()), 2, batch.calib,
            batch.aug_param, keep_rows=keep)
    for k, t in named.items():
        assert np.array_equal(t.indices.cpu().numpy(), o[k].indices.numpy()), k
        assert rel_err(t.features.detach().cpu(), o[k].features.detach()) < TOL, k
    sum(t.features.mean() for t in named.values()).backward()
    assert model.vir_conv1.d3_conv1[0].weight.grad is not None


def test_full_size_properties(lib_built):
    """BASELINE-size scene (16k LiDAR + 80k virtual, cap 40k/scene, batch 2): size-independent properties —
    the oracle needs ~10 s here, so only invariants are checked: shape chain, sorted batch-contiguous strided
    outputs, submanifold tables symmetric (nbr[K-1-k][nbr[k][o]] == o), pair counts, finite outputs."""
    from virconv_b200 import scenes, ops
    batch = scenes.make_batch([0, 1])
    model, _ = _models()
    model.eval()
    with torch.no_grad():
        named, out = _run_gpu(model, batch.voxel_features, batch.voxel_coords, 2, batch.calib, None)
    assert named['x_conv1'].spatial_shape == [81, 1600, 1408]
    assert named['x_conv2'].spatial_shape == [41, 800, 704]
    assert named['x_conv3'].spatial_shape == [21, 400, 352]
    assert named['x_conv4'].spatial_shape == [10, 200, 176]
    assert named['out'].spatial_shape == [4, 200, 176]
    for k in ('x_conv2', 'x_conv3', 'x_conv4', 'out'):
        t = named[k]
        idx = t.indices.cpu().numpy().astype(np.int64)
        lin = orb.linearize(idx, t.spatial_shape)
        assert np.all(np.diff(lin) > 0), k                      # strictly ascending => unique + batch-contiguous
        assert torch.isfinite(t.features).all()
    for key, rb in named['x_conv1'].indice_dict.items():
        if isinstance(key, str) and key.startswith('subm1'):   # 3-D submanifold tables
            nbr = rb.nbr
            K, n = nbr.shape
            o = torch.arange(n, device=nbr.device)
            for k in range(K):
                i = nbr[k].long()
                ok = i >= 0
                assert torch.equal(nbr[K - 1 - k][i[ok]].long(), o[ok]), (key, k)
            assert torch.equal(rb.pair_num.long(), (nbr >= 0).sum(1))
    dense = named['out'].dense()
    assert dense.shape == (2, 64, 4, 200, 176)
    assert float(dense.abs().sum()) == pytest.approx(float(named['out'].features.abs().sum()), rel=1e-5)


def test_config1_full_size_vs_oracle(lib_built):
    """BASELINE config 1 AT ITS STATED SIZE: one synthetic KITTI scene, 16 384 LiDAR returns, no virtual points, VirConv-L
    forward in fp32 (train-mode BatchNorm): every layer's canonical rulebook bit-exact against the CPU oracle, the five
    published feature maps within 1e-4 (north_star tolerance)."""
    from virconv_b200 import scenes
    batch = scenes.make_batch([7], n_lidar=16384, n_virtual=0, max_voxels=40000, training=False)
    assert batch.voxel_features.shape[0] > 10000
    model, ref = _models()
    model.train()
    ref.train()
    with torch.no_grad():
        named, _ = _run_gpu(model, batch.voxel_features, batch.voxel_coords, 1, batch.calib, None)
        o = ref(torch.from_numpy(batch.voxel_features.copy()), torch.from_numpy(batch.voxel_coords.copy()), 1, batch.calib, None)
    for k, t in named.items():
        assert np.array_equal(t.indices.cpu().numpy(), o[k].indices.numpy()), k
        assert rel_err(t.features.cpu(), o[k].features) < TOL, k
    d, od = named['x_conv1'].indice_dict, o['x_conv1'].indice_dict
    n_checked = 0
    for key, rb in d.items():
        if isinstance(key, str) and key in od:
            assert np.array_equal(rb.nbr.cpu().numpy(), od[key]['nbr_np']), key
            n_checked += 1
    assert n_checked >= 8


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_bench_batch_forward_vs_oracle(lib_built, precision):
    """The batch bench.py times (2 scenes x (16k LiDAR + 80k virtual), 40 000-voxel cap each: 80 000 input voxels),
    forward against the CPU oracle: indices bit-exact; features 1e-4 on the fp32 kernels, 2e-2 on the bf16 tensor-core
    kernels (operands rounded to bf16, fp32 accumulation)."""
    from virconv_b200 import scenes
    from virconv_b200 import spconv_compat as spc
    batch = scenes.make_batch([0, 1], training=True)
    assert batch.voxel_features.shape[0] == 80000
    model, ref = _models()
    spc.set_precision(model, precision)
    model.train()
    ref.train()
    with torch.no_grad():
        named, _ = _run_gpu(model, batch.voxel_features, batch.voxel_coords, 2, batch.calib, batch.aug_param)
        o = ref(torch.from_numpy(batch.voxel_features.copy()), torch.from_numpy(batch.voxel_coords.copy()), 2, batch.calib,
                batch.aug_param)
    assert ops_err_flag() == 0
    for k, t in named.items():
        assert np.array_equal(t.indices.cpu().numpy(), o[k].indices.numpy()), k
        assert rel_err(t.features.cpu(), o[k].features) < (TOL if precision == 'fp32' else 2e-2), k


# ------------------------------------------------------------------------------------------------ VirConv-T / -S
CFG8 = dict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.15, NUM_FILTERS=[16, 32, 64, 64], MM=True)


def _published(out_dict, sfx_list):
    res = {}
    for s in sfx_list:
        res[f'encoded_spconv_tensor{s}:out'] = out_dict['encoded_spconv_tensor' + s]
        for grp in ('multi_scale_3d_features', 'multi_scale_3d_features_mm'):
            for name, t in out_dict[grp + s].items():
                if t is not None:
                    res[f'{grp}{s}:{name}'] = t
    return res


@pytest.mark.parametrize('mode', ['train', 'eval'])
def test_virconv8x_matches_reference_golden(lib_built, mode):
    from virconv_b200 import scenes
    from virconv_b200.backbone import VirConv8x
    g = np.load(os.path.join(GOLD, 'virconv_t_small.npz'))
    m = VirConv8x(CFG8, 8, [1408, 1600, 80])
    fill_module(m, int(g['seed']))
    m.to('cuda:0').train(mode == 'train')
    bd = {k.split(':')[2]: torch.from_numpy(g[k].copy()).cuda() for k in g.files if k.startswith(f'{mode}:in:')}
    bd.update(batch_size=2, calib=[scenes.Calib(), scenes.Calib()])
    bd['aug_param' if mode == 'train' else 'transform_param'] = torch.from_numpy(g[f'{mode}:aug'].copy())
    with torch.no_grad():
        out = m(bd)
    pub = _published(out, [''] if mode == 'train' else ['', '1', '2'])
    assert len(pub) == (9 if mode == 'train' else 21)
    for k, t in pub.items():
        assert np.array_equal(t.indices.cpu().numpy(), g[f'{mode}:{k}:indices']), k
        check_sampled_rows(t.features, g, f'{mode}:{k}:features', TOL)


def test_virconv8x_forward_backward_vs_oracle(lib_built):
    from virconv_b200 import scenes
    from virconv_b200.backbone import VirConv8x
    from oracle.backbone import VirConv8x as Oracle8
    batch = scenes.make_batch_mm([2, 7], n_lidar=4096, n_virtual=6000, max_voxels=3000, training=True)
    m = VirConv8x(CFG8, 8, [1408, 1600, 80])
    fill_module(m, 667)
    ref = Oracle8()
    ref.load_state_dict(m.state_dict())
    m.to('cuda:0').train()
    ref.train()
    bd = {k: torch.from_numpy(v.copy()).cuda() for k, v in batch.arrays.items()}
    bd.update(batch_size=2, calib=batch.calib, aug_param=torch.from_numpy(batch.aug_param))
    out = m(bd)
    o = ref({k: torch.from_numpy(v.copy()) for k, v in batch.arrays.items()}, 2, batch.calib, aug_param=batch.aug_param)
    pub = _published(out, [''])
    loss, rloss = 0, 0
    for k, t in pub.items():
        grp, name = k.split(':')
        rt = o[grp] if name == 'out' else o[grp][name]
        assert np.array_equal(t.indices.cpu().numpy(), rt.indices.numpy()), k
        assert rel_err(t.features.detach().cpu(), rt.features.detach()) < TOL, k
        loss = loss + t.features.mean()
        rloss = rloss + rt.features.mean()
    loss.backward()
    rloss.backward()
    gp = dict(m.named_parameters())
    for name, p in ref.named_parameters():
        assert rel_err(gp[name].grad.cpu(), p.grad) < 2e-3, name
    # shared rulebooks: conv_input / conv1 use one 'subm1' table
    d = pub['multi_scale_3d_features:x_conv1'].indice_dict
    assert d['subm1'] is not None and len([k for k in d if isinstance(k, str)]) == 8   # subm1-4, spconv2-4, spconv_down2


def test_wgrad_kernel_variants_agree(lib_built):
    """The plan executor's two weight-gradient kernels (vc_conv_wgrad_tc3_config: half-tile stages on half the SMs — the default —
    and the one-CTA-per-SM kernel) accumulate the same bf16 products in fp32: parameter gradients agree up to summation order."""
    from virconv_b200 import _lib, scenes
    from virconv_b200 import spconv_compat as spc
    lib = _lib.load()
    batch = scenes.make_batch([51, 52], n_lidar=4096, n_virtual=9000, max_voxels=7000, training=True)
    model, _ = _models()
    spc.set_precision(model, 'bf16')
    model.train()
    grads = []
    try:
        for variant in (0, 1):
            _lib.check(lib.vc_conv_wgrad_tc3_config(variant, 0), 'vc_conv_wgrad_tc3_config')
            for p in model.parameters():
                p.grad = None
            named, out = _run_gpu(model, batch.voxel_features, batch.voxel_coords, 2, batch.calib, batch.aug_param)
            loss = sum(t.features.mean() for t in named.values())
            loss.backward()
            torch.cuda.synchronize()
            assert int(ops_err_flag()) == 0
            grads.append({k: v.grad.detach().clone() for k, v in model.named_parameters() if k.endswith('0.weight')})
    finally:
        _lib.check(lib.vc_conv_wgrad_tc3_config(1, 0), 'vc_conv_wgrad_tc3_config')
    for k in grads[0]:
        a, b = grads[0][k].double(), grads[1][k].double()
        assert float((a - b).norm() / b.norm().clamp_min(1e-30)) < 1e-2, k      # (bf16 run-to-run noise of the chain: see test_gpu_graph._grad_close)
