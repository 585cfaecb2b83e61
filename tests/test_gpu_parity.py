"""GPU parity suite (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle on the
same seeded inputs, against the committed reference goldens, and through size-independent properties
at full size.  Tolerances (stated per test): fp32 configuration 1e-3 absolute (BASELINE.json north_star),
integer / index outputs bit-exact; the bf16 configuration has no reference counterpart (the reference
is fp32-only, SURVEY section 0 row 4) and carries its own stated tolerance."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from occnet_b200 import fixtures

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = 'cuda:0'
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))          # tests/golden/sampling.py (shared with gen_fullsize.py)


def _oracle():
    from oracle import bevformer_occ as O
    from oracle import msda as OM
    from oracle import ray_metrics as ORM
    return O, OM, ORM


def make_case(base, bs=1, with_prev=False, ang=None, **kw):
    O, _, _ = _oracle()
    cfg = fixtures.make_cfg(base, **kw)
    params = O.init_params(cfg, seed=2)
    feats = fixtures.make_feats(cfg, bs=bs, seed=1)
    metas = fixtures.make_img_metas(cfg, bs=bs, can_bus_angle=ang)
    prev = None
    if with_prev:
        g = torch.Generator().manual_seed(3)
        prev = torch.randn(bs, cfg['bev_h'] * cfg['bev_w'], cfg['embed_dims'], generator=g)
    return cfg, params, feats, metas, prev


def engine_for(cfg, params, metas, precision='fp32', tc=False):
    from occnet_b200.engine import OccEngine
    eng = OccEngine(cfg, params, precision=precision, use_tensor_cores=tc, device=DEV)
    eng.set_cameras(metas)
    return eng


def to_ref_layout(out, cfg):
    """engine outputs -> reference tensor layouts (batch dim added)."""
    C = cfg['embed_dims']
    bev = out['bev_embed'].t().reshape(1, C, cfg['bev_h'], cfg['bev_w'])
    return bev, out['occ'][None], out['flow'][None]


# ------------------------------------------------------------------------------------------ operator boundary (a8)
@pytest.mark.parametrize('shape', [
    dict(B=2, M=8, C=32, Nq=300, levels=[(12, 20), (6, 10), (3, 5), (2, 3)], P=8),      # SCA-like
    dict(B=2, M=8, C=32, Nq=625, levels=[(25, 25)], P=4),                               # TSA-like
    dict(B=1, M=4, C=12, Nq=33, levels=[(5, 7), (3, 3)], P=3),                          # C % 8 != 0 -> scalar path
    dict(B=3, M=2, C=8, Nq=0, levels=[(4, 4)], P=2),                                    # empty query set
])
def test_ms_deform_attn_forward_matches_oracle(shape):
    from occnet_b200 import ops
    _, OM, _ = _oracle()
    torch.manual_seed(0)
    shapes = torch.tensor(shape['levels'])
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    Nv = int(shapes.prod(1).sum())
    B, M, C, Nq, P, L = shape['B'], shape['M'], shape['C'], shape['Nq'], shape['P'], len(shape['levels'])
    value = torch.randn(B, Nv, M, C)
    loc = torch.rand(B, Nq, M, L, P, 2) * 1.5 - 0.25      # includes out-of-image samples
    if Nq > 4:                                            # exact borders / pixel centres
        loc[0, 0] = 0.0; loc[0, 1] = 1.0; loc[0, 2] = 0.5
        loc[0, 3, :, :, :, 0] = (torch.arange(P).float() + 0.5)[None, None] / shapes[:, 1].float()[None, :, None]
    w = torch.rand(B, Nq, M, L, P)
    got = ops.ms_deform_attn_forward(value.to(DEV), shapes.to(DEV), lsi.to(DEV), loc.to(DEV), w.to(DEV), 64).cpu()
    if Nq == 0:
        assert got.shape == (B, 0, M * C)
        return
    want = OM.msda_grid_sample(value, shapes, loc, w)
    np.testing.assert_allclose(got.numpy(), want.numpy(), atol=1e-4, rtol=0)          # bound 1e-3; observed ~1e-6
    small = OM.msda_loops(value[:1, :, :, :], shapes, lsi, loc[:1, :8], w[:1, :8])
    np.testing.assert_allclose(got[:1, :8].numpy(), small.numpy(), atol=2e-5, rtol=0)


def test_ms_deform_attn_forward_error_behaviour():
    from occnet_b200 import ops, _lib
    v = torch.zeros(3, 16, 1, 8, device=DEV)
    sh = torch.tensor([[4, 4]], device=DEV); ls = torch.tensor([0], device=DEV)
    loc = torch.zeros(3, 2, 1, 1, 1, 2, device=DEV); w = torch.zeros(3, 2, 1, 1, 1, device=DEV)
    with pytest.raises(_lib.OccB200Error):                       # mmcv: batch must divide im2col_step
        ops.ms_deform_attn_forward(v, sh, ls, loc, w, 2)
    with pytest.raises(RuntimeError):                            # non-contiguous input
        ops.ms_deform_attn_forward(v.transpose(0, 1).contiguous().transpose(0, 1), sh, ls, loc, w, 64)
    with pytest.raises(RuntimeError):                            # CPU tensor
        ops.ms_deform_attn_forward(v.cpu(), sh, ls, loc, w, 64)
    fn = ops.MultiScaleDeformableAttnFunction_fp32.apply(v, sh, ls, loc, w, 64)
    assert fn.shape == (3, 2, 8)


@pytest.mark.parametrize('shape', [
    dict(B=2, M=8, C=32, Nq=200, levels=[(12, 20), (6, 10), (3, 5), (2, 3)], P=8),
    dict(B=1, M=4, C=12, Nq=33, levels=[(5, 7), (3, 3)], P=3),
    dict(B=2, M=2, C=48, Nq=17, levels=[(6, 6)], P=4),
])
def test_ms_deform_attn_backward_matches_autograd_of_oracle(shape):
    """SURVEY 8f rank 4: gradients of the operator (value / sampling_loc / attn_weight) equal torch autograd through the
    oracle's grid_sample restatement (mmcv's CPU path), fp32, tolerance 1e-3 (observed ~1e-5)."""
    from occnet_b200 import ops
    _, OM, _ = _oracle()
    torch.manual_seed(1)
    shapes = torch.tensor(shape['levels'])
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    Nv = int(shapes.prod(1).sum())
    B, M, C, Nq, P, L = shape['B'], shape['M'], shape['C'], shape['Nq'], shape['P'], len(shape['levels'])
    value = torch.randn(B, Nv, M, C, requires_grad=True)
    loc = (torch.rand(B, Nq, M, L, P, 2) * 1.3 - 0.15).requires_grad_(True)       # some samples outside / on borders
    w = torch.rand(B, Nq, M, L, P, requires_grad=True)
    go = torch.randn(B, Nq, M * C)
    out = OM.msda_grid_sample(value, shapes, loc, w)
    out.backward(go)
    vd, ld, wd = (t.detach().to(DEV).requires_grad_(True) for t in (value, loc, w))
    got = ops.MultiScaleDeformableAttnFunction_fp32.apply(vd, shapes.to(DEV), lsi.to(DEV), ld, wd, 64)
    np.testing.assert_allclose(got.detach().cpu().numpy(), out.detach().numpy(), atol=1e-4, rtol=0)
    got.backward(go.to(DEV))
    np.testing.assert_allclose(vd.grad.cpu().numpy(), value.grad.numpy(), atol=1e-3, rtol=0)
    np.testing.assert_allclose(wd.grad.cpu().numpy(), w.grad.numpy(), atol=1e-3, rtol=0)
    # d/d(loc) is discontinuous exactly on pixel-centre lines; random locations avoid them, tolerance scaled by the map size
    np.testing.assert_allclose(ld.grad.cpu().numpy(), loc.grad.numpy(), atol=2e-3, rtol=1e-3)


# ------------------------------------------------------------------------------------------ projection (a1, a2)
@pytest.mark.parametrize('base', ['small6', 'full'])
def test_pillar_projection_matches_point_sampling(base):
    O, _, _ = _oracle()
    cfg, params, feats, metas, _ = make_case(base, num_layers=1)
    eng = engine_for(cfg, params, metas)
    ref, mask = eng.project_pillars()
    pc = cfg['pc_range']
    ref_3d = O.get_reference_points(cfg['bev_h'], cfg['bev_w'], pc[5] - pc[2], cfg['num_points_in_pillar'], '3d', 1)
    rpc, m = O.point_sampling(ref_3d, pc, metas)                 # (cam, B, Nq, D, 2), (cam, B, Nq, D)
    flips = (mask.cpu().bool() != m[:, 0]).sum().item()
    assert flips == 0, f'{flips} visibility flips'               # index-like output: exact
    vis = m[:, 0]
    d = (ref.cpu() - rpc[:, 0]).abs()[vis]
    assert d.max().item() < 1e-5                                 # normalised image coords of visible points


# ------------------------------------------------------------------------------------------ feature packing (a9)
@pytest.mark.parametrize('precision,use_cams', [('fp32', True), ('fp32', False), ('bf16', True)])
def test_pack_levels_matches_get_bev_features(precision, use_cams):
    """transformer_occ.py:207-227 on its own: NCHW levels -> (cam, Nv, C) tokens + cams_embeds (if enabled) + level_embeds.
    fp32: bit-exact (same two additions in the same order); bf16 storage: the fp32 result rounded once."""
    O, _, _ = _oracle()
    cfg, params, feats, metas, _ = make_case('small6', num_layers=1, use_cams_embeds=use_cams)
    eng = engine_for(cfg, params, metas, precision)
    eng.forward([f[0].to(DEV) for f in feats], want=('bev_embed',))
    got = eng.tap('tokens').cpu()
    want, shapes, lsi = O.pack_camera_features(params, 'transformer', cfg, feats)       # (cam, Nv, B, C)
    want = want[:, :, 0]
    assert lsi.tolist() == [0] + np.cumsum([h * w for h, w in cfg['level_shapes']])[:-1].tolist()
    if precision == 'fp32':
        assert torch.equal(got, want)
    else:
        assert torch.equal(got, want.bfloat16().float())
    if not use_cams:                                             # the embedding really is off (and on in the default case)
        with_cams, _, _ = O.pack_camera_features(params, 'transformer', dict(cfg, use_cams_embeds=True), feats)
        assert not torch.equal(got, with_cams[:, :, 0])


def test_bf16_feature_input_equals_rounded_fp32_input():
    """`occb200_engine_set_input_dtype(1)`: bf16 feature levels (on-device backbone / bf16 host pipeline) give bit-identical
    results to fp32 levels holding the same bf16-rounded numbers; level sizes here hit the 16-byte and the scalar loads."""
    cfg, params, feats, metas, _ = make_case('small6')
    eng = engine_for(cfg, params, metas, 'bf16', tc=False)
    f16 = [f[0].bfloat16().to(DEV).contiguous() for f in feats]
    a = {k: v.clone() for k, v in eng.forward([f.float() for f in f16], want=('bev_embed', 'occ', 'flow')).items()}
    eng.set_input_dtype(torch.bfloat16)
    b = eng.forward(f16, want=('bev_embed', 'occ', 'flow'))
    for k in a:
        assert torch.equal(a[k], b[k]), k
    with pytest.raises(ValueError):                              # dtype contract is checked on the host
        eng.forward([f.float() for f in f16])
    host = [f.cpu().pin_memory() for f in f16]
    occ_h, flow_h = eng.forward_host(host)
    assert torch.equal(flow_h, b['flow'].cpu())


# ------------------------------------------------------------------------------------------ full path, fp32 config
def _check_fp32(cfg, params, feats, metas, prev, per_layer=True, tc=False):
    O, _, _ = _oracle()
    taps = {}
    with torch.no_grad():
        want = O.head_forward(params, cfg, feats, metas, prev_bev=None if prev is None else prev.clone(), taps=taps)
    eng = engine_for(cfg, params, metas, 'fp32', tc=tc)
    eng.enable_taps(True)
    pb = None
    if prev is not None:
        pb = prev.clone()
        if 'can_bus' in metas[0]:                                # the plugin rotates prev_bev before the engine (a9)
            pb = O.rotate_prev_bev(pb[0], cfg['bev_h'], cfg['bev_w'], metas[0]['can_bus'][-1],
                                   cfg.get('rotate_center', [100, 100]))[None]
    out = eng.forward([f[0].to(DEV) for f in feats], prev_bev=pb,
                      want=('bev_embed', 'occ', 'flow', 'occ_cls', 'occ_cls_i64'))
    torch.cuda.synchronize()
    if per_layer:
        for l in range(cfg['num_layers']):
            for name in ('tsa', 'sca', 'layer'):
                key = f'layer{l}' + ('' if name == 'layer' else '_' + name)
                err = (eng.tap(name, l).cpu() - taps[key][0]).abs().max().item()
                assert err < 1e-3, f'layer {l} {name}: {err}'
    bev, occ, flow = to_ref_layout({k: v.cpu() for k, v in out.items()}, cfg)
    assert (bev - want['bev_embed']).abs().max().item() < 1e-3
    assert (eng.tap('voxel').cpu()[None] - taps['voxel_feats']).abs().max().item() < 1e-3
    assert (occ - want['occ']).abs().max().item() < 1e-3
    assert (flow - want['flow']).abs().max().item() < 1e-3
    cls_want = want['occ'].softmax(-1).argmax(-1)[0]
    agree = (out['occ_cls'].cpu().long() == cls_want).float().mean().item()
    assert agree > 0.9995                                        # ties within 1e-3 may flip
    assert torch.equal(out['occ_cls'].cpu().long(), out['occ_cls_i64'].cpu())
    assert torch.equal(out['occ_cls_i64'].cpu(), out['occ'].cpu().argmax(-1))          # indexing: exact vs own logits
    return eng, out, want


def test_engine_fp32_toy_cfg1():
    _check_fp32(*make_case('toy'))


def test_engine_fp32_small6_two_layers():
    _check_fp32(*make_case('small6'))


def test_engine_fp32_temporal_prev_bev():
    _check_fp32(*make_case('small6', with_prev=True, ang=3.0, rotate_center=[20, 20]))


@pytest.mark.parametrize('prev', [False, True])
def test_engine_fp32_tensor_core_split_gemm(prev):
    """fp32 storage + tcgen05: every nn.Linear as ONE 3-pass bf16-split GEMM (hi.hi + lo.hi + hi.lo, ~2^-16 relative): the
    reference-precision configuration on the tensor cores, same 1e-3 bar per layer tap and output as the CUDA-core one."""
    code = ("import sys; sys.path.insert(0, 'tests'); import test_gpu_parity as t; "
            f"t._check_fp32(*t.make_case('small6', with_prev={prev}, ang={3.0 if prev else None}, rotate_center=[20, 20]), tc=True); "
            "print('OK')")
    assert 'OK' in _run_isolated(code)


@pytest.mark.parametrize('name', ['toy', 'small6', 'small6_prev'])
def test_engine_fp32_matches_reference_golden(name, golden_dir):
    """Against fixtures produced by the UNMODIFIED reference modules (tests/golden/gen_golden.py)."""
    O, _, _ = _oracle()
    spec = {'toy': ('toy', False, None, {}), 'small6': ('small6', False, None, {}),
            'small6_prev': ('small6', True, 3.0, dict(rotate_center=[20, 20]))}[name]
    cfg, params, feats, metas, prev = make_case(spec[0], with_prev=spec[1], ang=spec[2], **spec[3])
    eng = engine_for(cfg, params, metas, 'fp32')
    pb = None
    if prev is not None:
        pb = O.rotate_prev_bev(prev[0].clone(), cfg['bev_h'], cfg['bev_w'], 3.0, cfg['rotate_center'])[None]
    out = eng.forward([f[0].to(DEV) for f in feats], prev_bev=pb)
    bev, occ, flow = to_ref_layout({k: v.cpu() for k, v in out.items()}, cfg)
    g = np.load(os.path.join(golden_dir, f'ref_model_{name}.npz'))
    for k, t in (('bev_embed', bev), ('occ', occ), ('flow', flow)):
        assert tuple(t.shape) == tuple(g[k + '_shape'])
        sub = t.reshape(-1)[torch.from_numpy(g[k + '_idx'])].numpy()
        np.testing.assert_allclose(sub, g[k + '_sub'], atol=1e-3, rtol=0)
    assert (out['occ_cls'].cpu().numpy() == g['occ_cls'][0]).mean() > 0.9995


def test_engine_fp32_full_size_one_layer():
    """BASELINE configs[1] geometry (6 x 928x1600 -> 200x200 BEV, 200x200x16 voxels), one layer against the oracle."""
    _check_fp32(*make_case('full', num_layers=1), per_layer=True)


def test_engine_missing_parameter_is_loud():
    from occnet_b200.engine import OccEngine
    from occnet_b200 import _lib
    cfg, params, *_ = make_case('toy')
    bad = dict(params)
    bad.pop('transformer.encoder.layers.0.attentions.1.output_proj.weight')
    with pytest.raises(_lib.OccB200Error, match='missing parameter'):
        OccEngine(cfg, bad, 'fp32', device=DEV)
    with pytest.raises(_lib.OccB200Error, match='unknown parameter key'):
        OccEngine(cfg, dict(params, **{'img_backbone.conv1.weight': torch.zeros(3)}), 'fp32', device=DEV)


# ------------------------------------------------------------------------------------------ bf16 configuration
def _check_bf16(tc):
    O, _, _ = _oracle()
    cfg, params, feats, metas, _ = make_case('small6')
    with torch.no_grad():
        want = O.head_forward(params, cfg, feats, metas)
    eng = engine_for(cfg, params, metas, 'bf16', tc=tc)
    out = eng.forward([f[0].to(DEV) for f in feats])
    torch.cuda.synchronize()
    bev, occ, flow = to_ref_layout({k: v.cpu() for k, v in out.items()}, cfg)
    # bf16 storage (8-bit mantissa) of values / activations, fp32 accumulation: tolerance 6e-2 abs on O(1)
    # LayerNorm outputs and logits, and >= 97 % argmax agreement with the fp32 oracle.
    assert (bev - want['bev_embed']).abs().max().item() < 6e-2
    assert (bev - want['bev_embed']).abs().mean().item() < 6e-3
    assert (occ - want['occ']).abs().max().item() < 6e-2
    assert (flow - want['flow']).abs().max().item() < 6e-2
    agree = (out['occ_cls'].cpu().long() == want['occ'].softmax(-1).argmax(-1)[0]).float().mean().item()
    assert agree > 0.97, agree


def test_engine_bf16_simt_gemm():
    _check_bf16(tc=False)


def _run_isolated(code, timeout=300):
    """tcgen05 bring-up runs in a child process: a device fault there must not poison this session's context."""
    r = subprocess.run([sys.executable, '-c', code], cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, f'child failed ({r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}'
    return r.stdout


TC_GEMM_CODE = r'''
import torch, ctypes
from occnet_b200 import _lib
lib = _lib.load()
torch.manual_seed(0)
for (M, N, K) in [(128, 256, 256), (1000, 192, 512), (40000, 256, 256), (4100, 768, 256), (333, 512, 256),
                  (2000, 256, 768), (777, 192, 1536), (1000, 192, 256)]:      # K > 512: streamed (non-resident) weight tiles
    A = (torch.randn(M, K, device='cuda') * 0.5).bfloat16()
    W = (torch.randn(N, K, device='cuda') * 0.1).bfloat16()
    b = torch.randn(N, device='cuda')
    C = torch.full((M, N), float('nan'), device='cuda')
    _lib.check(lib.occb200_gemm_bf16_tc(_lib.ptr(A), _lib.ptr(W), _lib.ptr(b), _lib.ptr(C), M, N, K, _lib.stream_ptr()))
    torch.cuda.synchronize()
    ref = A.float() @ W.float().t() + b
    err = (C - ref).abs().max().item()
    print('tcgen05 gemm', M, N, K, 'max err', err)
    assert err < 2e-3, err
print('OK')
'''


def test_tcgen05_gemm_matches_fp32_matmul():
    """bf16 x bf16 -> fp32 on the tensor cores equals an fp32 matmul of the same bf16-rounded operands (exact
    products, fp32 accumulation order aside): tolerance 2e-3 on |C| ~ 2."""
    out = _run_isolated(TC_GEMM_CODE)
    assert 'OK' in out


def test_engine_bf16_tensor_cores():
    code = ("import sys; sys.path.insert(0, 'tests'); import test_gpu_parity as t; t._check_bf16(tc=True); print('OK')")
    assert 'OK' in _run_isolated(code)


# ------------------------------------------------------------------------------------------ host-buffer entry (e2e call)
def test_forward_host_equals_device_path():
    cfg, params, feats, metas, _ = make_case('small6')
    eng = engine_for(cfg, params, metas, 'fp32')
    out = eng.forward([f[0].to(DEV) for f in feats], want=('flow', 'occ_cls_i64'))
    host = [f[0].contiguous().pin_memory() for f in feats]
    occ_h, flow_h = eng.forward_host(host)
    assert occ_h.dtype == torch.int64 and not occ_h.is_cuda
    assert torch.equal(occ_h, out['occ_cls_i64'].cpu())
    assert torch.equal(flow_h, out['flow'].cpu())


def test_pipelined_host_stream_equals_sync_calls():
    """submit/wait with two frames in flight returns exactly what the synchronous host call returns, frame by frame."""
    cfg, params, _, metas, _ = make_case('small6')
    eng = engine_for(cfg, params, metas, 'fp32')
    frames = [[f[0].contiguous().pin_memory() for f in fixtures.make_feats(cfg, bs=1, seed=50 + i)] for i in range(5)]
    want = []
    for fr in frames:
        o, f = eng.forward_host(fr)
        want.append((o.clone(), f.clone()))
    got = [(o.clone(), f.clone()) for o, f in eng.stream_host(frames)]
    assert len(got) == 5
    for (go, gf), (wo, wf) in zip(got, want):
        assert torch.equal(go, wo) and torch.equal(gf, wf)
    assert not torch.equal(want[0][1], want[1][1])               # the frames really differ


# ------------------------------------------------------------------------------------------ metric (a14, a15)
def _metric_fixture():
    sem_gt, flow_gt = fixtures.make_occ_scene(seed=4)
    rng = np.random.RandomState(5)
    sem_pred = np.roll(sem_gt, 1, axis=0).copy()
    flip = rng.rand(*sem_pred.shape) < 0.03
    sem_pred[flip] = rng.randint(0, 17, int(flip.sum())).astype(np.uint8)
    flow_pred = (np.roll(flow_gt, 1, axis=0) + rng.normal(0, 0.5, flow_gt.shape)).astype(np.float32)
    return sem_pred, flow_pred, sem_gt, flow_gt


def test_render_forward_bit_exact_vs_oracle_dda():
    from occnet_b200 import ops
    _, _, ORM = _oracle()
    sem_pred, _, _, _ = _metric_fixture()
    rays = ORM.generate_lidar_rays()
    occ = np.ascontiguousarray(np.where(sem_pred < 16, 1, 0).astype(np.float32).transpose(2, 1, 0))[None]
    for origin in ([0.98, 0.0, 1.84], [-20.0, 3.0, 1.84], [500.0, 500.0, 50.0], [39.9, -39.9, 5.3]):
        o = ((np.asarray(origin, np.float32) - np.float32([-40, -40, -1])) / np.float32(0.4)).astype(np.float32)
        p = ((rays + np.asarray(origin, np.float32) - np.float32([-40, -40, -1])) / np.float32(0.4)).astype(np.float32)
        ti = np.zeros(len(rays), np.float32); ti[::97] = -1.0     # padded points are skipped
        want = ORM.render_forward(occ, o[None], p, ti)
        got = ops.render_forward(torch.from_numpy(occ)[None].to(DEV), torch.from_numpy(o)[None, None].to(DEV),
                                 torch.from_numpy(p)[None].to(DEV), torch.from_numpy(ti)[None].to(DEV),
                                 [1, 16, 200, 200], 'test')
        np.testing.assert_array_equal(got[2][0].cpu().numpy(), want[2])          # voxel indices: bit-exact
        np.testing.assert_array_equal(got[0][0].cpu().numpy(), want[0])          # fp64 traversal -> identical fp32
        np.testing.assert_array_equal(got[1][0].cpu().numpy(), want[1])


DVR_ORIGINS = ([0.98, 0.0, 1.84], [-20.0, 3.0, 1.84], [500.0, 500.0, 50.0])
DVR_OUTPUTS = ('pred_dist', 'gt_dist', 'coord')


def dvr_inputs():
    """(occ, origin, points, tindex) on the device per origin of DVR_ORIGINS, laid out as the reference's metric hands
    them to its ray-casting kernel; also the inputs of tests/golden/gen_dvr_ref.py."""
    _, _, ORM = _oracle()
    sem_pred, _, _, _ = _metric_fixture()
    rays = ORM.generate_lidar_rays()
    occ = torch.from_numpy(np.ascontiguousarray(np.where(sem_pred < 16, 1, 0).astype(np.float32).transpose(2, 1, 0)))
    occ = occ[None, None].to(DEV)
    for origin in DVR_ORIGINS:
        o = torch.tensor(origin) - torch.tensor([-40.0, -40.0, -1.0])
        o = (o / 0.4).float()[None, None].to(DEV)
        p = ((torch.from_numpy(rays) + torch.tensor(origin) - torch.tensor([-40.0, -40.0, -1.0])) / 0.4).float()[None].to(DEV)
        ti = torch.zeros(1, rays.shape[0], device=DEV)
        yield occ, o, p, ti


def test_render_forward_vs_reference_kernel(golden_dir):
    """Against the reference's own dvr.cu: its outputs on these inputs are stored in tests/golden/ref_dvr.npz
    (tests/golden/gen_dvr_ref.py runs the kernel as oracle/build_ref.py builds it)."""
    from occnet_b200 import ops
    _, _, ORM = _oracle()
    ref = np.load(os.path.join(golden_dir, 'ref_dvr.npz'))
    for j, (occ, o, p, ti) in enumerate(dvr_inputs()):
        got = ops.render_forward(occ, o, p, ti, [1, 16, 200, 200], 'test')
        want = ORM.render_forward(occ[0].cpu().numpy(), o[0].cpu().numpy(), p[0].cpu().numpy(), ti[0].cpu().numpy())
        for i, key in enumerate(DVR_OUTPUTS):
            assert got[i].dtype == torch.float32
            np.testing.assert_array_equal(got[i][0].cpu().numpy(), ref[key][j], err_msg=f'{key} differs from the reference kernel')
        np.testing.assert_array_equal(ref['pred_dist'][j], want[0])               # pins the C oracle too
        np.testing.assert_array_equal(ref['coord'][j], want[2])


@pytest.mark.parametrize('f64', [False, True])
def test_ray_metric_counters_match_oracle(f64, golden_dir):
    from occnet_b200 import metric
    _, _, ORM = _oracle()
    sem_pred, flow_pred, sem_gt, flow_gt = _metric_fixture()
    T = 2 if not f64 else 3
    orig = fixtures.make_ray_origins(T=T)
    if f64:
        orig = orig.astype(np.float64) + 1e-9
    rm = metric.RayMetric(DEV)
    pp, pg = rm.add_frame(torch.from_numpy(sem_pred), torch.from_numpy(flow_pred), torch.from_numpy(sem_gt),
                          torch.from_numpy(flow_gt), torch.from_numpy(orig), return_pcd=True)
    rays = ORM.generate_lidar_rays()
    if f64:
        # torch promotion semantics (float32 rays + float64 origins) restated with numpy float64
        lid = rays[None].astype(np.float64) + orig[:, :, None, :].reshape(1, T, 1, 3)
        want_p, want_g = [], []
        off = np.float32([-40, -40, -1]).astype(np.float64); sc = np.float64(np.float32(0.4))
        for t in range(T):
            o = ((orig[0, t] - off) / sc).astype(np.float32)
            p = ((lid[0, t] - off) / sc).astype(np.float32)
            for sem, flow, dst in ((sem_pred, flow_pred, want_p), (sem_gt, flow_gt, want_g)):
                occ = np.ascontiguousarray(np.where(sem < 16, 1, 0).astype(np.float32).transpose(2, 1, 0))[None]
                pd, _, ci = ORM.render_forward(occ, o[None], p, np.zeros(len(rays), np.float32))
                ci = ci.astype(np.int32)
                dst.append(np.concatenate([sem[ci[:, 0], ci[:, 1], ci[:, 2]].astype(np.float32)[:, None],
                                           (pd * np.float32(0.4))[:, None], flow[ci[:, 0], ci[:, 1], ci[:, 2]]], -1))
        want_p = np.concatenate(want_p); want_g = np.concatenate(want_g)
    else:
        want_p = ORM.process_one_sample(sem_pred, rays, orig, flow_pred)
        want_g = ORM.process_one_sample(sem_gt, rays, orig, flow_gt)
    np.testing.assert_array_equal(pp.cpu().numpy(), want_p)                       # class, dist, flow rows: bit-exact
    np.testing.assert_array_equal(pg.cpu().numpy(), want_g)
    valid = want_g[:, 0].astype(np.int32) != 16
    cnt = ORM.accumulate(ORM.new_counters(), want_p[valid], want_g[valid])
    vec = ORM.counters_to_vector(cnt)
    got = rm.counters.cpu().numpy()
    n = 17
    np.testing.assert_array_equal(got[:5 * n], vec[:5 * n])                        # integer counters: exact
    np.testing.assert_array_equal(got[8 * n:], vec[8 * n:])
    np.testing.assert_allclose(got[5 * n:8 * n], vec[5 * n:8 * n], rtol=1e-5)      # fp sums: order differs
    fin = rm.finalize(); want = ORM.finalize(cnt)
    assert abs(fin['miou'] - want['miou']) < 1e-12 and abs(fin['mave'] - want['mave']) < 1e-5
    if not f64:
        g = np.load(os.path.join(golden_dir, 'ref_metric.npz'))
        np.testing.assert_array_equal(pp.cpu().numpy(), g['pcd_pred'])             # the reference's own output
        np.testing.assert_allclose(fin['iou'], g['iou'], equal_nan=True, rtol=1e-12)
    # empty: zero origins leaves the counters untouched
    before = rm.counters.clone()
    rm.add_frame(torch.from_numpy(sem_pred), torch.from_numpy(flow_pred), torch.from_numpy(sem_gt),
                 torch.from_numpy(flow_gt), torch.zeros(0, 3))
    assert torch.equal(before, rm.counters)


@pytest.mark.parametrize('tc', [False, True])
def test_full_size_properties_bf16(tc):
    """BASELINE full sizes, size-independent properties: determinism (bit-identical reruns), argmax consistent with
    the engine's own logits, finite outputs; tensor-core and CUDA-core bf16 paths agree with each other."""
    cfg, params, feats, metas, _ = make_case('full', num_layers=2)
    eng = engine_for(cfg, params, metas, 'bf16', tc=tc)
    fd = [f[0].to(DEV) for f in feats]
    a = eng.forward(fd, want=('bev_embed', 'occ', 'occ_cls', 'flow'))
    a = {k: v.clone() for k, v in a.items()}
    b = eng.forward(fd, want=('bev_embed', 'occ', 'occ_cls', 'flow'))
    for k in a:
        assert torch.equal(a[k], b[k]), f'{k} not deterministic'
    assert torch.equal(a['occ'].argmax(-1).to(torch.uint8), a['occ_cls'])
    assert torch.isfinite(a['bev_embed']).all() and torch.isfinite(a['occ']).all()
    assert eng.launches_per_frame >= 10                         # every launch of the frame is one of the library's own kernels
    if tc:
        ref = engine_for(cfg, params, metas, 'bf16', tc=False).forward(fd, want=('bev_embed', 'occ', 'occ_cls', 'flow'))
        assert (a['bev_embed'] - ref['bev_embed']).abs().max().item() < 8e-2       # bf16 weights vs fp32 weights
        assert (a['occ'] - ref['occ']).abs().max().item() < 8e-2
        assert (a['occ_cls'] == ref['occ_cls']).float().mean().item() > 0.97



# ------------------------------------------------------------------------------------------ FULL SIZE, 6 LAYERS (goldens)
def _report(name, vals):
    """Measured parity numbers of this run -> gpurun_out/parity_report.json (evidence; copied to profiles/)."""
    import json
    d = os.path.join(ROOT, 'gpurun_out')
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, 'parity_report.json')
    rep = json.load(open(path)) if os.path.exists(path) else {}
    rep[name] = {k: (float(v) if not isinstance(v, (str, list)) else v) for k, v in vals.items()}
    json.dump(rep, open(path, 'w'), indent=1)


def _full6_case(prev=False):
    cfg = fixtures.make_cfg('full', num_layers=6)
    params = fixtures.init_params(cfg, seed=2, free_bias=fixtures.FREE_BIAS)
    feats = fixtures.make_feats(cfg, bs=1, seed=100)
    metas = fixtures.make_img_metas(cfg, bs=1, can_bus_angle=3.0 if prev else None)
    pb = None
    if prev:
        O, _, _ = _oracle()
        pb = torch.randn(1, cfg['bev_h'] * cfg['bev_w'], cfg['embed_dims'], generator=torch.Generator().manual_seed(3))
        pb = O.rotate_prev_bev(pb[0], cfg['bev_h'], cfg['bev_w'], 3.0, cfg.get('rotate_center', [100, 100]))[None]
    return cfg, params, feats, metas, pb


def _sub_err(key, t, golden, n):
    from sampling import sub_idx
    flat = t.reshape(-1).cpu()
    got = flat[torch.from_numpy(sub_idx(key, flat.numel(), n))].numpy()
    d = np.abs(got - golden[key + '_sub'])
    return float(d.max()), float(d.mean())


def _ray_miou_vs(pred_cls, pred_flow, gt_cls, gt_flow):
    """Ray-mIoU / mAVE of a prediction with ANOTHER prediction standing in as ground truth (parity as the metric sees it)."""
    from occnet_b200 import metric
    rm = metric.RayMetric(DEV)
    rm.add_frame(pred_cls, pred_flow, gt_cls, gt_flow, torch.from_numpy(fixtures.make_ray_origins(T=8)))
    return rm.finalize()


def _ray_counters_vs_scene(pred_cls, pred_flow):
    from occnet_b200 import metric
    sem_gt, flow_gt = fixtures.make_occ_scene(seed=4)
    rm = metric.RayMetric(DEV)
    rm.add_frame(pred_cls, pred_flow, torch.from_numpy(sem_gt), torch.from_numpy(flow_gt),
                 torch.from_numpy(fixtures.make_ray_origins(T=8)))
    return rm.counters.cpu().numpy()


@pytest.mark.parametrize('tc', [False, True])
def test_full_size_six_layers_fp32_vs_oracle_golden(tc, golden_dir):
    if tc:                                                       # tcgen05 path in a child process (a fault must not poison this one)
        code = ("import sys; sys.path.insert(0, 'tests'); import test_gpu_parity as t; "
                f"t._full6_fp32(True, {golden_dir!r}); print('OK')")
        assert 'OK' in _run_isolated(code, timeout=600)
    else:
        _full6_fp32(False, golden_dir)


def _full6_fp32(tc, golden_dir):
    """tc=True: the split-bf16 tcgen05 GEMMs (fp32-grade), tc=False: CUDA-core GEMMs.  BASELINE configs[1]: 6 x 928x1600 -> 200x200 BEV, SIX encoder layers, voxel decoder, heads, fp32 configuration.
    Every per-layer tap and every output within 1e-3 of the oracle (golden: tests/golden/gen_fullsize.py, oracle pinned
    bit-exactly to the reference modules); class volume and Ray-mIoU counters as the reference's metric sees them."""
    from sampling import N_OUT, N_TAP
    cfg, params, feats, metas, _ = _full6_case()
    g = np.load(os.path.join(golden_dir, 'full6_fp32.npz'))
    eng = engine_for(cfg, params, metas, 'fp32', tc=tc)
    eng.enable_taps(True)
    out = eng.forward([f[0].to(DEV) for f in feats], want=('bev_embed', 'occ', 'flow', 'occ_cls'))
    torch.cuda.synchronize()
    rep = {}
    for l in range(6):
        for name in ('tsa', 'sca', 'layer'):
            key = f'layer{l}' + ('' if name == 'layer' else '_' + name)
            mx, _ = _sub_err(key, eng.tap(name, l), g, N_TAP)
            rep[key] = mx
            assert mx < 1e-3, f'{key}: {mx}'
    bev, occ, flow = to_ref_layout(out, cfg)
    for key, t in (('bev_embed', bev), ('voxel', eng.tap('voxel')), ('occ', occ), ('flow', flow)):
        mx, mean = _sub_err(key, t, g, N_OUT)
        rep[key] = mx
        assert mx < 1e-3, f'{key}: {mx}'
    cls_g = torch.from_numpy(g['occ_cls'])
    agree = (out['occ_cls'].cpu() == cls_g).float().mean().item()
    assert agree > 0.9995                                        # logits within 1e-3: only near-ties may flip
    fin = _ray_miou_vs(out['occ_cls'], out['flow'], cls_g, torch.from_numpy(g['flow_f16'].astype(np.float32)))
    rep.update(class_agreement=agree, ray_miou_vs_oracle_output=fin['miou'], ray_mave_vs_oracle_output=fin['mave'])
    assert fin['miou'] > 0.995, fin['miou']                      # Ray-mIoU of the CUDA output scored against the oracle's
    cnt = _ray_counters_vs_scene(out['occ_cls'], out['flow'])
    n = 17                                                       # integer counters vs the synthetic GT scene
    rel = np.abs(cnt[:5 * n] - g['counters'][:5 * n]).sum() / max(g['counters'][:5 * n].sum(), 1)
    rep['counter_rel_diff_vs_oracle_counters'] = rel
    assert rel < 2e-3, rel
    _report('full6_fp32' + ('_tc_split' if tc else '_cuda_cores'), rep)


def _check_full6_bf16(prev, golden_dir):
    from sampling import N_OUT
    tag = 'full6_prev' if prev else 'full6'
    cfg, params, feats, metas, pb = _full6_case(prev)
    g32 = np.load(os.path.join(golden_dir, f'{tag}_fp32.npz'))
    g16 = np.load(os.path.join(golden_dir, f'{tag}_bf16.npz'))
    eng = engine_for(cfg, params, metas, 'bf16', tc=True)        # NO taps: the fused configuration bench.py times
    out = eng.forward([f[0].to(DEV) for f in feats], prev_bev=pb, want=('bev_embed', 'occ', 'flow', 'occ_cls'))
    torch.cuda.synchronize()
    bev, occ, flow = to_ref_layout(out, cfg)
    rep = {}
    for key, t in (('bev_embed', bev), ('voxel', eng.tap('voxel')), ('occ', occ), ('flow', flow)):
        rep[key + '_max_vs_bf16_model'], rep[key + '_mean_vs_bf16_model'] = _sub_err(key, t, g16, N_OUT)
        if key != 'voxel':
            rep[key + '_max_vs_fp32_oracle'], rep[key + '_mean_vs_fp32_oracle'] = _sub_err(key, t, g32, N_OUT)
    cls32, cls16 = torch.from_numpy(g32['occ_cls']), torch.from_numpy(g16['occ_cls'])
    rep['class_agreement_vs_fp32_oracle'] = (out['occ_cls'].cpu() == cls32).float().mean().item()
    rep['class_agreement_vs_bf16_model'] = (out['occ_cls'].cpu() == cls16).float().mean().item()
    fin16 = _ray_miou_vs(out['occ_cls'], out['flow'], cls16, out['flow'])
    fin32 = _ray_miou_vs(out['occ_cls'], out['flow'], cls32, out['flow'])
    rep['ray_miou_vs_bf16_model_output'], rep['ray_miou_vs_fp32_oracle_output'] = fin16['miou'], fin32['miou']
    _report(tag + '_bf16_tc', rep)
    # (i) against the fp32 oracle: what 8-bit mantissas allow.  The storage-rounding MODEL's own distance from the fp32
    # oracle on the same subsample is the yardstick: the engine may not be further away than the model by more than 25 % in
    # the mean (a wrong constant / index / layout moves the mean; rounding noise does not) or 2x in the max.
    from sampling import sub_idx
    for key in ('bev_embed', 'occ', 'flow'):
        model_d = np.abs(g16[key + '_sub'] - g32[key + '_sub'])
        rep[key + '_model_max_vs_fp32_oracle'], rep[key + '_model_mean_vs_fp32_oracle'] = float(model_d.max()), float(model_d.mean())
        assert rep[key + '_max_vs_fp32_oracle'] < 6e-2, (key, rep)
        assert rep[key + '_mean_vs_fp32_oracle'] < 6e-3, (key, rep)
        assert rep[key + '_mean_vs_fp32_oracle'] < 1.25 * model_d.mean(), (key, rep)
        assert rep[key + '_max_vs_fp32_oracle'] < 2.0 * model_d.max(), (key, rep)
    assert rep['class_agreement_vs_fp32_oracle'] > 0.99, rep
    # (ii) against the model itself.  Over six layers the path is chaotic in the rounding sense (a 1-ulp difference in an
    # fp32 accumulation order flips a bf16 rounding and the flip propagates as bf16-sized noise), so engine-vs-model can only be
    # as tight as model-vs-fp32 (measured 2.0e-2 max / 2.9e-3 mean vs 3.3e-2 / 3.8e-3); the TIGHT model comparison is the
    # one-layer test below.
    _report(tag + '_bf16_tc', rep)
    for key in ('bev_embed', 'occ', 'flow'):
        assert rep[key + '_max_vs_bf16_model'] < BF16_MODEL_TOL_MAX, (key, rep)
        assert rep[key + '_mean_vs_bf16_model'] < BF16_MODEL_TOL_MEAN, (key, rep)
        assert rep[key + '_mean_vs_bf16_model'] < 1.1 * rep[key + '_model_mean_vs_fp32_oracle'], (key, rep)
    assert rep['voxel_mean_vs_bf16_model'] < BF16_MODEL_TOL_MEAN, rep
    assert rep['class_agreement_vs_bf16_model'] > 0.995, rep
    # Ray-mIoU of the engine's class volume scored against the model's / the oracle's (random synthetic weights: logits of
    # neighbouring classes are close, so 0.4 % flipped voxels move the metric by several points; measured 0.968 / 0.911)
    assert rep['ray_miou_vs_bf16_model_output'] > 0.93 and rep['ray_miou_vs_fp32_oracle_output'] > 0.85, rep
    return rep


# engine vs storage-rounding model after SIX layers (see (ii) above) and after ONE layer (calibrated on the first GPU run of the
# test, r2 call 4, then frozen)
BF16_MODEL_TOL_MAX, BF16_MODEL_TOL_MEAN = 4e-2, 5e-3
# one layer, measured on B200 (profiles/r2_parity_report.json): bev_embed 8.6e-3 / 3.0e-4 (no prev), 9.5e-3 / 2.8e-4 (prev) -- the
# encoder output is TIGHT against the model (mean one tenth of the model's own distance from fp32); occ / flow pass through the
# bf16 voxel tensors of the decoder (every flipped rounding there is a 2^-8 relative step): 1.7e-2 / 2.2e-3
BF16_MODEL_TOL1 = {'bev_embed': (2e-2, 6e-4), 'occ': (3e-2, 3.5e-3), 'flow': (3e-2, 3.5e-3)}


def _check_full1_bf16(prev, golden_dir):
    from sampling import sub_idx
    cfg = fixtures.make_cfg('full', num_layers=1)
    params = fixtures.init_params(cfg, seed=2, free_bias=fixtures.FREE_BIAS)
    feats = fixtures.make_feats(cfg, bs=1, seed=100)
    metas = fixtures.make_img_metas(cfg, bs=1, can_bus_angle=3.0 if prev else None)
    pb = None
    if prev:
        O, _, _ = _oracle()
        pb = torch.randn(1, cfg['bev_h'] * cfg['bev_w'], cfg['embed_dims'], generator=torch.Generator().manual_seed(3))
        pb = O.rotate_prev_bev(pb[0], cfg['bev_h'], cfg['bev_w'], 3.0, cfg.get('rotate_center', [100, 100]))[None]
    g = np.load(os.path.join(golden_dir, 'full1_prev_bf16.npz' if prev else 'full1_bf16.npz'))
    eng = engine_for(cfg, params, metas, 'bf16', tc=True)        # NO taps: the fused configuration
    out = eng.forward([f[0].to(DEV) for f in feats], prev_bev=pb, want=('bev_embed', 'occ', 'flow', 'occ_cls'))
    torch.cuda.synchronize()
    bev, occ, flow = to_ref_layout(out, cfg)
    rep = {}
    n1 = len(g['bev_embed_bf16_sub'])
    for key, t in (('bev_embed', bev), ('occ', occ), ('flow', flow)):
        flat = t.reshape(-1).cpu()
        got = flat[torch.from_numpy(sub_idx(key, flat.numel(), n1))].numpy()
        d16, d32 = np.abs(got - g[key + '_bf16_sub']), np.abs(got - g[key + '_fp32_sub'])
        dm = np.abs(g[key + '_bf16_sub'] - g[key + '_fp32_sub'])
        rep.update({key + '_max_vs_bf16_model': d16.max(), key + '_mean_vs_bf16_model': d16.mean(),
                    key + '_max_vs_fp32_oracle': d32.max(), key + '_mean_vs_fp32_oracle': d32.mean(),
                    key + '_model_max_vs_fp32_oracle': dm.max(), key + '_model_mean_vs_fp32_oracle': dm.mean()})
    rep['class_agreement_vs_bf16_model'] = (out['occ_cls'].cpu() == torch.from_numpy(g['occ_cls_bf16'])).float().mean().item()
    rep['class_agreement_vs_fp32_oracle'] = (out['occ_cls'].cpu() == torch.from_numpy(g['occ_cls_fp32'])).float().mean().item()
    _report('full1' + ('_prev' if prev else '') + '_bf16_tc', rep)
    for key in ('bev_embed', 'occ', 'flow'):
        assert rep[key + '_max_vs_bf16_model'] < BF16_MODEL_TOL1[key][0], (key, rep)
        assert rep[key + '_mean_vs_bf16_model'] < BF16_MODEL_TOL1[key][1], (key, rep)
        assert rep[key + '_mean_vs_fp32_oracle'] < 1.25 * rep[key + '_model_mean_vs_fp32_oracle'] + 1e-4, (key, rep)
    assert rep['class_agreement_vs_bf16_model'] > 0.995, rep            # measured 0.9971 (near-tie voxels under random weights)


@pytest.mark.parametrize('prev', [False, True])
def test_full_size_one_layer_bf16_tensor_cores_vs_storage_rounding_model(prev, golden_dir):
    """ONE encoder layer at full size (tests/golden/gen_onelayer.py): few roundings have happened, so the engine must sit
    close to the storage-rounding model -- the tight check that the six-layer comparison cannot be."""
    _check_full1_bf16(prev, golden_dir)


def test_full_size_six_layers_bf16_tensor_cores_vs_goldens(golden_dir):
    """The configuration bench.py times (bf16 storage, tcgen05 GEMM / conv / heads, fused LayerNorm epilogues, hoisted
    value_proj, folded TSA projection, fp16 sampling projections) at FULL size, SIX layers, against (i) the fp32 oracle
    and (ii) the storage-rounding model of the same algorithm (oracle/bf16_model.py)."""
    _check_full6_bf16(False, golden_dir)


def test_full_size_six_layers_bf16_temporal_prev_bev(golden_dir):
    """Same with a previous BEV (BASELINE configs[2]: TemporalSelfAttention over [prev_bev, current]): the has_prev branch
    of the fused path (unfolded query projection over prev_t / q+pos, q+pos written by the FFN LayerNorm epilogue)."""
    _check_full6_bf16(True, golden_dir)


def test_voxel_lift_from_t32_layout_is_bit_identical():
    """When bev_embed is not requested the voxel lift reads the T32 residual stream directly (t32_to_voxel_kernel) instead of
    untiling to row-major first: same values, same rounding -> bit-identical occupancy / flow."""
    cfg, params, feats, metas, _ = make_case('small6')
    eng = engine_for(cfg, params, metas, 'bf16', tc=True)
    fd = [f[0].to(DEV) for f in feats]
    a = {k: v.clone() for k, v in eng.forward(fd, want=('bev_embed', 'occ', 'flow', 'occ_cls')).items()}
    b = eng.forward(fd, want=('occ', 'flow', 'occ_cls'))
    for k in b:
        assert torch.equal(a[k], b[k]), k


def test_layer0_tsa_constant_fold_is_bit_identical():
    """Self mode (prev_bev None): layer 0's TemporalSelfAttention + LayerNorm depend on parameters only and are computed once
    at finalize by the frame path's own kernels; an engine built with OCC_NO_L0_FOLD=1 recomputes them every frame.
    Same kernels, same inputs -> bit-identical outputs; with a prev_bev the fold must not be used."""
    code = r"""
import os, sys, torch
sys.path.insert(0, 'tests')
import test_gpu_parity as t
cfg, params, feats, metas, prev = t.make_case('small6', with_prev=True)
fd = [f[0].to(t.DEV) for f in feats]
a = t.engine_for(cfg, params, metas, 'bf16', tc=True)
os.environ['OCC_NO_L0_FOLD'] = '1'
b = t.engine_for(cfg, params, metas, 'bf16', tc=True)
del os.environ['OCC_NO_L0_FOLD']
for pb in (None, prev):
    oa = a.forward(fd, prev_bev=pb); la = a.launches_per_frame
    ob = b.forward(fd, prev_bev=pb); lb = b.launches_per_frame
    for k in oa:
        assert torch.equal(oa[k], ob[k]), k
    assert (lb - la) == (3 if pb is None else 0), (la, lb)       # layer 0: merged input GEMMs + gather + output_proj/LN
print('OK')
"""
    assert 'OK' in _run_isolated(code)


# ------------------------------------------------------------------------------------------ drop-in module API
def _plugin_head(cfg, params, precision='fp32'):
    import projects.mmdet3d_plugin  # noqa: F401
    from occnet_b200.mmcv_shim import build_head
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from test_dropin_cpu import head_cfg
    head = build_head(dict(head_cfg(cfg), precision=precision)).to(DEV).eval()
    head.load_state_dict(params, strict=True)
    return head


@pytest.mark.parametrize('bs', [1, 2])
def test_plugin_head_forward_matches_oracle(bs):
    """`BEVFormerOccHead.forward` / `get_occ` through the registry-built drop-in class (reference signature)."""
    O, _, _ = _oracle()
    cfg, params, feats, metas, _ = make_case('small6', bs=bs, num_layers=1)
    head = _plugin_head(cfg, params)
    out = head([f.to(DEV) for f in feats], metas)
    occ_cls, flow = head.get_occ(out, metas)
    assert occ_cls.dtype == torch.int64 and tuple(occ_cls.shape) == (bs, 40, 40, 16)
    for b in range(bs):                                          # frames are independent == reference at batch 1
        with torch.no_grad():
            want = O.head_forward(params, cfg, [f[b:b + 1] for f in feats], [metas[b]])
        for k in ('bev_embed', 'occ', 'flow'):
            assert (out[k][b].cpu() - want[k][0]).abs().max().item() < 1e-3, k
    bev_only = head([f.to(DEV) for f in feats], metas, only_bev=True)
    assert tuple(bev_only.shape) == (bs, 1600, 256)


def test_plugin_attention_modules_match_oracle():
    """Stand-alone TemporalSelfAttention / SpatialCrossAttention / BEVFormerEncoder forwards (operator-level C ABI)."""
    O, _, _ = _oracle()
    cfg, params, feats, metas, _ = make_case('small6', num_layers=1)
    head = _plugin_head(cfg, params)
    enc = head.transformer.encoder
    layer = enc.layers[0]
    Nq, C = cfg['bev_h'] * cfg['bev_w'], 256
    g = torch.Generator().manual_seed(11)
    q = torch.randn(1, Nq, C, generator=g)
    pos = torch.randn(1, Nq, C, generator=g)
    pc = cfg['pc_range']
    ref_2d = O.get_reference_points(cfg['bev_h'], cfg['bev_w'], dim='2d', bs=1)
    hyb = torch.stack([ref_2d, ref_2d], 1).reshape(2, Nq, 1, 2)
    pre = 'transformer.encoder.layers.0'
    with torch.no_grad():
        want_tsa = O.temporal_self_attention(params, pre + '.attentions.0', cfg, q, None, pos, hyb,
                                             torch.tensor([[cfg['bev_h'], cfg['bev_w']]]), torch.tensor([0]))
    got_tsa = layer.attentions[0](q.to(DEV), None, None, None, query_pos=pos.to(DEV), reference_points=hyb.to(DEV),
                                  spatial_shapes=torch.tensor([[cfg['bev_h'], cfg['bev_w']]], device=DEV),
                                  level_start_index=torch.tensor([0], device=DEV))
    assert (got_tsa.cpu() - want_tsa).abs().max().item() < 1e-3
    ref_3d = O.get_reference_points(cfg['bev_h'], cfg['bev_w'], pc[5] - pc[2], cfg['num_points_in_pillar'], '3d', 1)
    rpc, mask = O.point_sampling(ref_3d, pc, metas)
    value, shapes, lsi = O.pack_camera_features(params, 'transformer', cfg, feats)
    with torch.no_grad():
        want_sca = O.spatial_cross_attention(params, pre + '.attentions.1', cfg, q, value, value, rpc, mask, shapes, lsi)
    got_sca = layer.attentions[1](q.to(DEV), value.to(DEV), value.to(DEV), reference_points_cam=rpc.to(DEV),
                                  bev_mask=mask.to(DEV), spatial_shapes=shapes.to(DEV), level_start_index=lsi.to(DEV))
    assert (got_sca.cpu() - want_sca).abs().max().item() < 1e-3
    # encoder forward (module-level path) and its point_sampling against the oracle
    rpc_g, mask_g = enc.point_sampling(ref_3d.to(DEV), pc, metas)
    assert torch.equal(mask_g.cpu(), mask)
    bq = params['bev_embedding.weight'][:, None, :].to(DEV)
    bpos = O.positional_encoding(params, 'positional_encoding', 1, cfg['bev_h'], cfg['bev_w']).flatten(2).permute(2, 0, 1)
    got_enc = enc(bq, value.to(DEV), value.to(DEV), bev_h=cfg['bev_h'], bev_w=cfg['bev_w'], bev_pos=bpos.to(DEV),
                  spatial_shapes=shapes.to(DEV), level_start_index=lsi.to(DEV), img_metas=metas)
    with torch.no_grad():
        want_enc = O.head_forward(params, cfg, feats, metas, only_bev=True)
    assert (got_enc.cpu() - want_enc).abs().max().item() < 1e-3


def test_plugin_detector_output_contract():
    """`model(return_loss=False, img_feats=..., img_metas=[[...]])` -> CPU LongTensor / FloatTensor dict (bevformer_occ.py:247-250)."""
    import projects.mmdet3d_plugin  # noqa: F401
    from occnet_b200.mmcv_shim import build_detector
    from test_dropin_cpu import head_cfg
    cfg, params, feats, metas, _ = make_case('small6', num_layers=1)
    det = build_detector(dict(type='BEVFormerOcc', use_grid_mask=True, video_test_mode=True, native_backbone=False,
                              img_backbone=dict(type='ResNet', depth=50), img_neck=dict(type='FPN'),
                              pts_bbox_head=head_cfg(cfg))).to(DEV).eval()
    det.pts_bbox_head.load_state_dict(params, strict=True)
    out = det(return_loss=False, rescale=True, img_feats=[f.to(DEV) for f in feats], img_metas=[metas])
    assert set(out) == {'occ_results', 'flow_results'}
    assert out['occ_results'].dtype == torch.int64 and not out['occ_results'].is_cuda
    assert tuple(out['occ_results'].shape) == (1, 40, 40, 16) and tuple(out['flow_results'].shape) == (1, 40, 40, 16, 2)
    with pytest.raises(RuntimeError, match='pass img_feats'):
        det(return_loss=False, img=[torch.zeros(1, 6, 3, 64, 64, device=DEV)], img_metas=[metas])


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_temporal_recurrence_four_history_frames(precision):
    """BASELINE configs[2]: 4 history BEV frames feed the current one through `obtain_history_bev` (the TSA queue itself is
    2: previous BEV + current, temporal_self_attention.py:195); every step rotates prev_bev by can_bus[-1] (in the engine,
    as a row gather through torchvision's index map).  bf16: the has_prev branch of the fused tcgen05 path, bf16 bars."""
    import projects.mmdet3d_plugin  # noqa: F401
    from occnet_b200.mmcv_shim import build_detector
    from test_dropin_cpu import head_cfg
    O, _, _ = _oracle()
    cfg = fixtures.make_cfg('small6', num_layers=1, rotate_center=[20, 20])
    params = O.init_params(cfg, seed=2)
    det = build_detector(dict(type='BEVFormerOcc', pts_bbox_head=dict(head_cfg(cfg), precision=precision))).to(DEV).eval()
    det.pts_bbox_head.load_state_dict(params, strict=True)
    angles = [0.0, 2.0, -3.0, 1.5, 4.0]
    frames = [fixtures.make_feats(cfg, bs=1, seed=70 + i) for i in range(5)]
    metas = [fixtures.make_img_metas(cfg, bs=1, can_bus_angle=a) for a in angles]
    prev = det.obtain_history_bev([[f.to(DEV) for f in fr] for fr in frames[:4]], metas[:4])
    _, occ, flow = det.simple_test(metas[4], img_feats=[f.to(DEV) for f in frames[4]], prev_bev=prev)
    want_prev = None
    with torch.no_grad():
        for fr, m in zip(frames[:4], metas[:4]):
            want_prev = O.head_forward(params, cfg, fr, m, prev_bev=want_prev, only_bev=True)
        want = O.head_forward(params, cfg, frames[4], metas[4], prev_bev=want_prev)
    tol, agree = (1e-3, 0.9995) if precision == 'fp32' else (6e-2, 0.97)
    assert (prev.cpu() - want_prev).abs().max().item() < tol
    assert (flow.cpu() - want['flow']).abs().max().item() < tol
    assert (occ.cpu() == want['occ'].argmax(-1)).float().mean().item() > agree


@pytest.mark.parametrize('precision,tc', [('fp32', False), ('bf16', True)])
def test_engine_prev_rotation_map_equals_rotated_input(precision, tc):
    """`occb200_engine_set_prev_rotation`: un-rotated prev_bev + index map == prev_bev rotated beforehand by torchvision
    (the reference's call), bit for bit; clearing the map restores the pass-through."""
    from occnet_b200.engine import rotation_index_map
    O, _, _ = _oracle()
    cfg, params, feats, metas, prev = make_case('small6', with_prev=True, ang=-7.5, rotate_center=[20, 20])
    eng = engine_for(cfg, params, metas, precision, tc=tc)
    fd = [f[0].to(DEV) for f in feats]
    rotated = O.rotate_prev_bev(prev[0].clone(), cfg['bev_h'], cfg['bev_w'], -7.5, cfg['rotate_center'])[None]
    a = {k: v.clone() for k, v in eng.forward(fd, prev_bev=rotated).items()}
    eng.set_prev_rotation(rotation_index_map(cfg['bev_h'], cfg['bev_w'], -7.5, cfg['rotate_center']))
    b = {k: v.clone() for k, v in eng.forward(fd, prev_bev=prev).items()}
    eng.set_prev_rotation(None)
    c = eng.forward(fd, prev_bev=rotated)
    for k in a:
        assert torch.equal(a[k], b[k]) and torch.equal(a[k], c[k]), k
    assert not torch.equal(a['bev_embed'], eng.forward(fd, prev_bev=prev)['bev_embed'])     # the rotation matters


def test_detector_temporal_cache_and_scene_reset():
    """SURVEY 8f rank 3: `BEVFormerOcc(temporal_test=True, video_test_mode=True).forward_test` keeps the previous frame's
    BEV per stream and resets it on a new scene_token; the default (reference behaviour) never uses it."""
    import projects.mmdet3d_plugin  # noqa: F401
    from occnet_b200.mmcv_shim import build_detector
    from test_dropin_cpu import head_cfg
    O, _, _ = _oracle()
    cfg = fixtures.make_cfg('small6', num_layers=1, rotate_center=[20, 20])
    params = O.init_params(cfg, seed=2)

    def build(**kw):
        d = build_detector(dict(type='BEVFormerOcc', video_test_mode=True, pts_bbox_head=head_cfg(cfg), **kw)).to(DEV).eval()
        d.pts_bbox_head.load_state_dict(params, strict=True)
        return d
    det, ref = build(temporal_test=True), build()
    frames = [[f.to(DEV) for f in fixtures.make_feats(cfg, bs=1, seed=80 + i)] for i in range(3)]
    metas = []
    for tok, ang in (('scene-a', 0.0), ('scene-a', 2.5), ('scene-b', -1.0)):
        m = fixtures.make_img_metas(cfg, bs=1, can_bus_angle=ang)
        m[0]['scene_token'] = tok
        metas.append(m)
    outs = [det(return_loss=False, img_feats=fr, img_metas=[m]) for fr, m in zip(frames, metas)]
    plain = [ref(return_loss=False, img_feats=fr, img_metas=[m]) for fr, m in zip(frames, metas)]
    bev0, _, _ = ref.simple_test(metas[0], img_feats=frames[0])
    _, occ1, flow1 = ref.simple_test(metas[1], img_feats=frames[1], prev_bev=bev0)
    assert torch.equal(outs[0]['flow_results'], plain[0]['flow_results'])                    # first frame of a scene: no history
    assert torch.equal(outs[1]['flow_results'], flow1.cpu()) and torch.equal(outs[1]['occ_results'], occ1.cpu())
    assert not torch.equal(outs[1]['flow_results'], plain[1]['flow_results'])                # history was used
    assert torch.equal(outs[2]['flow_results'], plain[2]['flow_results'])                    # new scene: reset


def test_plugin_ray_metrics_main_matches_oracle():
    from projects.mmdet3d_plugin.datasets import ray_metrics as rm
    _, _, ORM = _oracle()
    sem_pred, flow_pred, sem_gt, flow_gt = _metric_fixture()
    orig = fixtures.make_ray_origins(T=3).astype(np.float64)     # the dataset hands float64 origins
    fin = rm.main([sem_pred], [sem_gt], [flow_pred], [flow_gt], [torch.from_numpy(orig)], device=DEV, verbose=False)
    want, _ = ORM.main([sem_pred], [sem_gt], [flow_pred], [flow_gt], [orig.astype(np.float32)])
    # (float64 vs float32 origins differ by rounding of the ray end points only; IoU counters are robust to it here)
    assert abs(fin['miou'] - want['miou']) < 5e-3
    pcd = rm.process_one_sample(sem_pred, rm.generate_lidar_rays(), fixtures.make_ray_origins(T=2), flow_pred, device=DEV)
    np.testing.assert_array_equal(pcd, ORM.process_one_sample(sem_pred, ORM.generate_lidar_rays(),
                                                              fixtures.make_ray_origins(T=2), flow_pred))


def test_plugin_submission_writer_matches_reference_format(tmp_path):
    """`datasets/submission.format_results` = the prediction half of the reference's `NuSceneOcc.format_results`
    (nuscenes_occ.py:188-257): per token {pcd_cls int8, pcd_dist fp16, pcd_flow fp16} from `process_one_sample`, pickled into a
    deterministic `submission.gz`.  Arrays must equal the oracle's restatement bit for bit."""
    import gzip
    import pickle
    from projects.mmdet3d_plugin.datasets import submission as sub
    _, _, ORM = _oracle()
    sem_pred, flow_pred, _, _ = _metric_fixture()
    origins = [fixtures.make_ray_origins(T=2), fixtures.make_ray_origins(T=3)]
    results = [{'occ_results': torch.from_numpy(sem_pred.astype(np.int64)), 'flow_results': torch.from_numpy(flow_pred)},
               {'occ_results': torch.from_numpy(sem_pred[::-1].copy().astype(np.int64)), 'flow_results': torch.from_numpy(flow_pred[::-1].copy())}]
    out = sub.format_results(results, ['tok_a', 'tok_b'], origins, submission_prefix=str(tmp_path), device=DEV)
    blob = open(os.path.join(str(tmp_path), 'submission.gz'), 'rb').read()
    loaded = pickle.loads(gzip.decompress(blob))
    assert set(loaded) == set(sub.SUBMISSION_META) | {'results'} and list(loaded['results']) == ['tok_a', 'tok_b']
    rays = ORM.generate_lidar_rays()
    for tok, res, orig in zip(('tok_a', 'tok_b'), results, origins):
        want = ORM.process_one_sample(res['occ_results'].numpy(), rays, orig, res['flow_results'].numpy())
        got = loaded['results'][tok]
        assert got['pcd_cls'].dtype == np.int8 and got['pcd_dist'].dtype == np.float16 and got['pcd_flow'].dtype == np.float16
        np.testing.assert_array_equal(got['pcd_cls'], want[:, 0].astype(np.int8))
        np.testing.assert_array_equal(got['pcd_dist'], want[:, 1].astype(np.float16))
        np.testing.assert_array_equal(got['pcd_flow'], want[:, 2:4].astype(np.float16))
        np.testing.assert_array_equal(out['results'][tok]['pcd_dist'], got['pcd_dist'])
    again = sub.format_results(results, ['tok_a', 'tok_b'], origins, submission_prefix=str(tmp_path), device=DEV)
    assert open(os.path.join(str(tmp_path), 'submission.gz'), 'rb').read() == blob and again.keys() == out.keys()
