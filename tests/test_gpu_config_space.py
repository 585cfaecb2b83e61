"""The engine across the configurations `occb200_engine_create` accepts, not only the three fixture geometries.

Every case below is `small6` plus overrides chosen to reach an index order or a tile tail that the square, tile-aligned
fixtures cannot: a non-square BEV grid (the BEV is row-major `q % bev_w`, `q / bev_w`, the voxel volume is
[X = bev_w][Y = bev_h][Z], so swapping the two is invisible on a square grid), Nq and X*Y that are not multiples of the
GEMM / head / conv tiles, pillar anchor counts D < 8, 1 and 8 cameras, class counts on both sides of the tensor-core
head's limit and FFN widths other than 512.

Each case runs in four configurations (fp32 CUDA cores, fp32 tensor-core split, bf16 CUDA cores, bf16 tensor-core fused
without taps -- the one bench.py times) against the fp32 oracle or the storage-rounding model, and through exact checks:
argmax consistency, bit-identical reruns, the T32 voxel lift, and sentinel tails behind every output buffer.
The CPU half checks the yardsticks themselves at the same cases.  The tensor-core configurations run in a child process
so that a device fault there cannot poison the session's context."""
import ctypes
import functools
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from occnet_b200 import fixtures

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = 'cuda:0'
C = 256

# name -> (make_cfg('small6', ...) overrides, temporal: (angle deg, rotate_center) or None).  1 encoder layer unless set;
# 'free_bias' replaces fixtures.FREE_BIAS where that leaves no voxel free on the case's geometry.
_RECT_TAIL = dict(bev_h=37, bev_w=23, level_shapes=[(17, 31), (9, 16), (5, 8), (2, 2)])
CASES = {
    # Nq = 851 (% 32 = 19, % 128 = 83): row-major fallbacks of the T32 paths; conv3d y-tail of 5 rows; head tail of
    # 48 voxels; a 2x2 level (the smallest the gathers accept) and level sides that are not multiples of 8
    'rect_tail': (_RECT_TAIL, None),
    # non-square with Nq % 32 == 0: fused T32 residual stream and the t32_to_voxel lift, both orientations
    'rect_aligned': (dict(bev_h=24, bev_w=40, num_layers=2), None),
    'rect_aligned_t': (dict(bev_h=40, bev_w=24, num_layers=2), None),
    # Nq = 6 (< one 32-row block), X = 2, 96 voxels (< one 128-voxel head tile)
    'tiny': (dict(bev_h=3, bev_w=2), None),
    # M = 129: one row past a 128-row GEMM tile
    'one_past_tile': (dict(bev_h=43, bev_w=3, free_bias=4.5), None),
    # Z-anchor interleave p % D and the z < D visibility lanes
    'pillar_D1': (dict(num_points_in_pillar=1), None),
    'pillar_D2': (dict(num_points_in_pillar=2), None),
    'pillar_D4': (dict(num_points_in_pillar=4), None),
    # one camera on the bf16 paths; eight fill the second visibility ballot group (cameras 4..7)
    'cams1': (dict(num_cams=1), None),
    'cams8': (dict(num_cams=8, free_bias=3.0), None),
    # tensor-core head below 17 classes; above 17 the bf16 tensor-core configuration uses the CUDA-core head
    'classes2': (dict(num_classes=2), None),
    'classes16': (dict(num_classes=16), None),
    'classes20': (dict(num_classes=20), None),
    # FFN GEMM shapes; 1024: FFN2 with K = 1024 streams its weights through the fused LayerNorm epilogue
    'ffn256': (dict(ffn_dim=256), None),
    'ffn1024': (dict(ffn_dim=1024), None),
    # prev_bev rotated by the engine's index map on a non-square grid, centre off the middle
    'temporal_rect': (_RECT_TAIL, (-7.5, [11, 18])),
}
NON_SQUARE = ('rect_tail', 'rect_aligned', 'rect_aligned_t', 'tiny', 'one_past_tile', 'temporal_rect')
PILLAR_D = ('pillar_D1', 'pillar_D2', 'pillar_D4')

# configuration name -> (precision, use_tensor_cores)
CONFIGS = {'fp32_cuda_cores': ('fp32', False), 'fp32_tc_split': ('fp32', True),
           'bf16_cuda_cores': ('bf16', False), 'bf16_tc_fused': ('bf16', True)}
OUTPUTS = ('bev_embed', 'occ', 'flow', 'occ_cls', 'occ_cls_i64')
TAIL = 4096                                                      # sentinel bytes behind every output buffer


def _oracle():
    from oracle import bevformer_occ as O
    from oracle import bf16_model as B
    return O, B


def rig_metas(cfg, can_bus_angle=None):
    """img_metas of the fixture's rig; for more than its 6 cameras, a ring of cameras at yaw i * 360/n degrees with the
    fixture's intrinsics and matrix conventions (lidar2img = viewpad @ inv(sensor2lidar))."""
    n = cfg['num_cams']
    if n <= 6:
        return fixtures.make_img_metas(cfg, bs=1, can_bus_angle=can_bus_angle)
    h, w = cfg['img_shape'][:2]
    e2l = np.linalg.inv(fixtures.PSEUDO_LIDAR2EGO)
    R0 = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
    viewpad = np.eye(4)
    viewpad[:3, :3] = np.array([[1266.0 * w / 1600, 0.0, 816.0 * w / 1600], [0.0, 1266.0 * h / 928, 491.0 * h / 928],
                                [0.0, 0.0, 1.0]], dtype=np.float32)
    l2i = []
    for i in range(n):
        a = math.radians(360.0 * i / n)
        cam2ego = np.eye(4)
        cam2ego[:3, :3] = np.array([[math.cos(a), -math.sin(a), 0.0], [math.sin(a), math.cos(a), 0.0], [0.0, 0.0, 1.0]]) @ R0
        cam2ego[:3, 3] = (math.cos(a), math.sin(a), 1.5)
        l2i.append(viewpad @ np.linalg.inv(e2l @ cam2ego))
    m = dict(lidar2img=l2i, ego2lidar=e2l, img_shape=[tuple(cfg['img_shape'])] * n)
    if can_bus_angle is not None:
        m['can_bus'] = np.zeros(18)
        m['can_bus'][-1] = can_bus_angle
    return [m]


def make_case(name):
    """-> cfg, params, feats (list of (1, cams, C, h, w)), img_metas, prev_bev (1, Nq, C) un-rotated or None."""
    over, temporal = CASES[name]
    over = dict(over)
    free_bias = over.pop('free_bias', fixtures.FREE_BIAS)
    cfg = fixtures.make_cfg('small6', **dict(dict(num_layers=1), **over))
    if temporal:
        cfg['rotate_center'] = temporal[1]
    params = fixtures.init_params(cfg, seed=2, free_bias=free_bias)
    feats = fixtures.make_feats(cfg, bs=1, seed=1)
    metas = rig_metas(cfg, temporal[0] if temporal else None)
    prev = None
    if temporal:
        prev = torch.randn(1, cfg['bev_h'] * cfg['bev_w'], C, generator=torch.Generator().manual_seed(3))
    return cfg, params, feats, metas, prev


def _engine_layout(d, cfg):
    """oracle output dict (batch 1) -> bev_embed (Nq, C), occ (X, Y, Z, ncls), flow (X, Y, Z, 2)."""
    Nq = cfg['bev_h'] * cfg['bev_w']
    return {'bev_embed': d['bev_embed'][0].reshape(C, Nq).t().contiguous(), 'occ': d['occ'][0], 'flow': d['flow'][0]}


def compute_reference(cfg, params, feats, metas, prev, model=True):
    """fp32 oracle with its per-layer taps and voxel features and (model=True) the storage-rounding model (quant=True),
    in engine layouts."""
    O, B = _oracle()
    taps = {}
    with torch.no_grad():
        f32 = O.head_forward(params, cfg, feats, metas, prev_bev=None if prev is None else prev.clone(), taps=taps)
    ref = {'fp32': _engine_layout(f32, cfg)}
    ref['fp32']['voxel'] = taps['voxel_feats'][0]
    ref['taps'] = {k: v[0] for k, v in taps.items() if k.startswith('layer')}
    if model:
        ref['bf16_model'] = _engine_layout(B.head_forward(params, cfg, feats, metas, prev_bev=prev, quant=True), cfg)
    return ref


@functools.lru_cache(maxsize=None)
def reference(name, model=True):
    return compute_reference(*make_case(name), model=model)


def _reference_file(name, directory):
    path = os.path.join(str(directory), f'{name}.pt')
    if not os.path.exists(path):
        torch.save(reference(name), path)
    return path


def _run_isolated(code, timeout=600):
    r = subprocess.run([sys.executable, '-c', code], cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, f'child failed ({r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}'
    return r.stdout


# ------------------------------------------------------------------------------------------ engine calls
def _make_engine(cfg, params, metas, precision, tc, temporal):
    from occnet_b200.engine import OccEngine, rotation_index_map
    eng = OccEngine(cfg, params, precision=precision, use_tensor_cores=tc, device=DEV)
    eng.set_cameras(metas)
    if temporal:
        eng.set_prev_rotation(rotation_index_map(cfg['bev_h'], cfg['bev_w'], temporal[0], temporal[1]))
    return eng


def forward_with_canaries(eng, feats, prev):
    """occb200_engine_forward through ctypes with every output requested.  Each output region starts as all-0xFF bytes
    (NaN for fp32, 255 for u8, -1 for i64) and is followed by TAIL sentinel bytes; afterwards every tail must be intact
    and every output fully written with in-range values."""
    X, Y, Z = eng.vox_shape
    ncls = eng.cfg['num_classes']
    spec = {'bev_embed': ((eng.Nq, C), torch.float32), 'occ': ((X, Y, Z, ncls), torch.float32),
            'flow': ((X, Y, Z, 2), torch.float32), 'occ_cls': ((X, Y, Z), torch.uint8),
            'occ_cls_i64': ((X, Y, Z), torch.int64)}
    sentinel = ((torch.arange(TAIL) * 37 + 11) % 256).to(torch.uint8).to(DEV)
    raw, nbytes = {}, {}
    for k, (shape, dt) in spec.items():
        nbytes[k] = math.prod(shape) * torch.empty((), dtype=dt).element_size()
        raw[k] = torch.full((nbytes[k] + TAIL,), 0xFF, dtype=torch.uint8, device=DEV)
        raw[k][nbytes[k]:] = sentinel
    pb = None if prev is None else prev.to(DEV, torch.float32).reshape(eng.Nq, C).contiguous()
    from occnet_b200 import _lib
    with torch.cuda.device(eng.device):
        _lib.check(eng.lib.occb200_engine_forward(
            eng._h, eng._feat_ptrs(feats), _lib.ptr(pb), *[_lib.ptr(raw[k]) for k in OUTPUTS], _lib.stream_ptr()))
    torch.cuda.synchronize()
    out = {}
    for k, (shape, dt) in spec.items():
        assert torch.equal(raw[k][nbytes[k]:], sentinel), f'{k}: write past the end of the buffer'
        out[k] = raw[k][:nbytes[k]].view(dt).view(shape)
    for k in ('bev_embed', 'occ', 'flow'):
        assert not torch.isnan(out[k]).any(), f'{k}: elements left unwritten (NaN)'
    for k in ('occ_cls', 'occ_cls_i64'):
        v = out[k].long()
        assert ((v >= 0) & (v < ncls)).all(), f'{k}: elements left unwritten or out of range'
    return out


def _check_parity_fp32(eng, out, ref, cfg):
    f32 = ref['fp32']
    for k in ('bev_embed', 'occ', 'flow'):
        err = (out[k].cpu() - f32[k]).abs().max().item()
        assert err < 1e-3, f'{k}: max |engine - fp32 oracle| = {err}'
    if eng.taps_enabled:
        for l in range(cfg['num_layers']):
            for name in ('tsa', 'sca', 'layer'):
                key = f'layer{l}' + ('' if name == 'layer' else '_' + name)
                err = (eng.tap(name, l).cpu() - ref['taps'][key]).abs().max().item()
                assert err < 1e-3, f'tap {key}: {err}'
        err = (eng.tap('voxel').cpu() - f32['voxel']).abs().max().item()
        assert err < 1e-3, f'voxel features: {err}'
    agree = (out['occ_cls'].cpu().long() == f32['occ'].argmax(-1)).float().mean().item()
    assert agree > 0.9995, f'class agreement with the fp32 oracle {agree}'


def _check_parity_bf16(out, ref, cfg, tc):
    """tc: the storage-rounding model restates the tensor-core configuration's storage points (fp16 sampling projections,
    folded TSA weights), so it is the tight yardstick there -- with test_gpu_parity's one-layer bars, or its six-layer bars
    when more than one layer has rounded.  The bf16 CUDA-core configuration keeps the projections in fp32; it is held to
    the project's bf16 bars against the fp32 oracle (test_engine_bf16_simt_gemm).  Both may not sit further from the fp32
    oracle, in the mean, than the model does."""
    from test_gpu_parity import BF16_MODEL_TOL1, BF16_MODEL_TOL_MAX, BF16_MODEL_TOL_MEAN
    f32, model = ref['fp32'], ref['bf16_model']
    tols = {k: BF16_MODEL_TOL1[k] if cfg['num_layers'] == 1 else (BF16_MODEL_TOL_MAX, BF16_MODEL_TOL_MEAN) for k in BF16_MODEL_TOL1}
    for k in ('bev_embed', 'occ', 'flow'):
        got = out[k].cpu()
        d16, d32, dm = (got - model[k]).abs(), (got - f32[k]).abs(), (model[k] - f32[k]).abs()
        if tc:
            tol_max, tol_mean = tols[k]
            assert d16.max().item() < tol_max, f'{k}: max |engine - model| = {d16.max().item()}'
            assert d16.mean().item() < tol_mean, f'{k}: mean |engine - model| = {d16.mean().item()}'
        else:
            assert d32.max().item() < 6e-2 and d32.mean().item() < 6e-3, (k, d32.max().item(), d32.mean().item())
        assert d32.mean().item() <= 1.25 * dm.mean().item() + 1e-4, \
            f'{k}: mean |engine - fp32| = {d32.mean().item()}, model itself {dm.mean().item()}'
    cls = out['occ_cls'].cpu().long()
    if tc:
        # near-tie voxels may flip; a voxel whose model logits are decided by more than the logit bar may not
        top2 = model['occ'].topk(2, -1).values
        clear = (top2[..., 0] - top2[..., 1]) > 2 * tols['occ'][0]
        assert torch.equal(cls[clear], model['occ'].argmax(-1)[clear]), 'class differs from the model on a clear voxel'
        agree = (cls == model['occ'].argmax(-1)).float().mean().item()
        assert agree > 0.99, f'class agreement with the storage-rounding model {agree}'
    else:
        agree = (cls == f32['occ'].argmax(-1)).float().mean().item()
        assert agree > 0.97, f'class agreement with the fp32 oracle {agree}'


def check_config(name, config, ref=None):
    """One case in one configuration: parity, canaries and the exact checks."""
    O, _ = _oracle()
    precision, tc = CONFIGS[config]
    cfg, params, feats, metas, prev = make_case(name)
    ref = reference(name) if ref is None else ref
    eng = _make_engine(cfg, params, metas, precision, tc, CASES[name][1])
    eng.taps_enabled = precision == 'fp32'                       # taps do not exist on the fused path
    if eng.taps_enabled:
        eng.enable_taps(True)
    fd = [f[0].to(DEV) for f in feats]
    out = forward_with_canaries(eng, fd, prev)
    if precision == 'fp32':
        _check_parity_fp32(eng, out, ref, cfg)
    else:
        _check_parity_bf16(out, ref, cfg, tc)
    # index outputs: exact against the engine's own logits
    assert torch.equal(out['occ_cls'].long(), out['occ'].argmax(-1)), 'occ_cls != argmax(occ)'
    assert torch.equal(out['occ_cls_i64'], out['occ_cls'].long()), 'occ_cls_i64 != occ_cls'
    # determinism, and outputs without bev_embed (the voxel lift from the T32 stream) equal to outputs with it
    out = {k: v.clone() for k, v in out.items()}
    again = eng.forward(fd, prev_bev=prev, want=OUTPUTS)
    for k in OUTPUTS:
        assert torch.equal(again[k], out[k]), f'{k}: rerun not bit-identical'
    lift = eng.forward(fd, prev_bev=prev, want=('occ', 'flow', 'occ_cls'))
    for k in lift:
        assert torch.equal(lift[k], out[k]), f'{k}: differs when bev_embed is not requested'
    if config == 'fp32_cuda_cores' and (name in NON_SQUARE or name in PILLAR_D or name.startswith('cams')):
        ref_cam, mask = eng.project_pillars()
        pc = cfg['pc_range']
        ref_3d = O.get_reference_points(cfg['bev_h'], cfg['bev_w'], pc[5] - pc[2], cfg['num_points_in_pillar'], '3d', 1)
        rpc, m = O.point_sampling(ref_3d, pc, metas)
        assert torch.equal(mask.cpu().bool(), m[:, 0]), 'visibility mask differs from point_sampling'
        vis = m[:, 0]
        assert (ref_cam.cpu() - rpc[:, 0]).abs()[vis].max().item() < 1e-5


# ------------------------------------------------------------------------------------------ GPU: the case table
@pytest.fixture(scope='module')
def ref_dir(tmp_path_factory):
    return tmp_path_factory.mktemp('config_space_refs')


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('name', list(CASES))
def test_engine_cuda_cores(name, precision):
    check_config(name, f'{precision}_cuda_cores')


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(CASES))
def test_engine_tensor_cores(name, ref_dir):
    """fp32 tensor-core split and bf16 tensor-core fused, in one child process per case (both are reported)."""
    path = _reference_file(name, ref_dir)
    code = (f"import sys, torch, traceback; sys.path.insert(0, 'tests'); import test_gpu_config_space as t\n"
            f"ref = torch.load({path!r})\nbad = 0\n"
            f"for config in ('fp32_tc_split', 'bf16_tc_fused'):\n"
            f"    try:\n        t.check_config({name!r}, config, ref); print(config, 'OK')\n"
            f"    except AssertionError:\n        bad += 1; print(config, 'FAILED'); traceback.print_exc(file=sys.stdout)\n"
            f"sys.exit(bad)\n")
    out = _run_isolated(code)
    assert out.count(' OK') == 2, out


# ------------------------------------------------------------------------------------------ CPU: the yardsticks
@pytest.mark.parametrize('name', list(CASES))
def test_case_yardsticks_cpu(name):
    """The storage-rounding model without rounding reproduces the fp32 oracle at every case (the bar of
    test_bf16_model_without_rounding_equals_fp32_oracle), and no case is vacuous: every camera sees some BEV cells and
    the free class is neither all nor none of the voxels."""
    O, B = _oracle()
    cfg, params, feats, metas, prev = make_case(name)
    ref = reference(name, model=False)
    exact = B.head_forward(params, cfg, feats, metas, prev_bev=prev, quant=False)
    Nq = cfg['bev_h'] * cfg['bev_w']
    for k, t in (('bev_embed', exact['bev_embed'][0].reshape(C, Nq).t()), ('occ', exact['occ'][0]),
                 ('flow', exact['flow'][0])):
        err = (t - ref['fp32'][k]).abs().max().item()
        assert err < 2e-4, f'{k}: {err}'
    pc = cfg['pc_range']
    ref_3d = O.get_reference_points(cfg['bev_h'], cfg['bev_w'], pc[5] - pc[2], cfg['num_points_in_pillar'], '3d', 1)
    _, mask = O.point_sampling(ref_3d, pc, metas)
    seen = mask[:, 0].any(-1).sum(-1)
    assert (seen > 0).all(), f'cameras that see no BEV cell: {seen.tolist()}'
    free = (ref['fp32']['occ'].argmax(-1) == cfg['num_classes'] - 1).float().mean().item()
    assert 0.0 < free < 1.0, free
    if CASES[name][1]:                                           # the rotation moves cells on this grid
        from occnet_b200.engine import rotation_index_map
        m = rotation_index_map(cfg['bev_h'], cfg['bev_w'], *CASES[name][1])
        assert (m != np.arange(Nq)).mean() > 0.5 and (m == -1).any()


def test_engine_create_refuses_grids_the_gathers_cannot_run():
    """A BEV or feature level side below 2 has no 2x2 bilinear block: refused when the engine is created, with an
    ordinary error return, not at forward time."""
    from occnet_b200 import _lib
    from occnet_b200.engine import _cfg_struct
    lib = _lib.load()
    base = fixtures.make_cfg('small6', num_layers=1)
    bad = [dict(bev_h=1, bev_w=40), dict(bev_h=40, bev_w=1), dict(bev_h=0, bev_w=40),
           dict(level_shapes=[(29, 50), (15, 25), (8, 13), (1, 7)]), dict(level_shapes=[(29, 50), (15, 1), (8, 13), (4, 7)])]
    for over in bad:
        for precision in ('fp32', 'bf16'):
            h = ctypes.c_void_p()
            c = _cfg_struct(dict(base, **over), precision, precision == 'bf16')
            rc = lib.occb200_engine_create(ctypes.byref(c), ctypes.byref(h))
            assert rc != 0 and not h.value, over
            assert b'at least 2x2' in lib.occb200_last_error(), (over, lib.occb200_last_error())
    for over in (dict(bev_h=2, bev_w=2), dict(level_shapes=[(2, 2)] * 4)):              # the smallest accepted
        h = ctypes.c_void_p()
        rc = lib.occb200_engine_create(ctypes.byref(_cfg_struct(dict(base, **over), 'fp32', False)), ctypes.byref(h))
        if rc == 0:
            lib.occb200_engine_destroy(h)
        else:                                                    # without a GPU: refused later, for the missing device
            assert b'no CUDA device' in lib.occb200_last_error(), lib.occb200_last_error()


# ------------------------------------------------------------------------------------------ GPU: shipped configuration
def _full4_case():
    cfg = fixtures.make_cfg('full', num_layers=4)                # bevformer_base_occ.py: 200x200, 4 encoder layers
    params = fixtures.init_params(cfg, seed=2, free_bias=fixtures.FREE_BIAS)
    feats = fixtures.make_feats(cfg, bs=1, seed=100)
    metas = fixtures.make_img_metas(cfg, bs=1)
    return cfg, params, feats, metas


def check_full4(config, ref):
    from test_gpu_parity import BF16_MODEL_TOL_MAX, BF16_MODEL_TOL_MEAN
    precision, tc = CONFIGS[config]
    cfg, params, feats, metas = _full4_case()
    eng = _make_engine(cfg, params, metas, precision, tc, None)
    eng.taps_enabled = precision == 'fp32'
    if eng.taps_enabled:
        eng.enable_taps(True)
    out = eng.forward([f[0].to(DEV) for f in feats], want=('bev_embed', 'occ', 'flow', 'occ_cls'))
    torch.cuda.synchronize()
    assert torch.equal(out['occ_cls'].long(), out['occ'].argmax(-1))
    if precision == 'fp32':
        _check_parity_fp32(eng, out, ref, cfg)
        return
    # the six-layer bf16 test's bars (test_gpu_parity._check_full6_bf16), here on every element
    f32, model = ref['fp32'], ref['bf16_model']
    for k in ('bev_embed', 'occ', 'flow'):
        got = out[k].cpu()
        d16, d32, dm = (got - model[k]).abs(), (got - f32[k]).abs(), (model[k] - f32[k]).abs()
        stats = (k, d16.max().item(), d16.mean().item(), d32.max().item(), d32.mean().item(), dm.max().item(), dm.mean().item())
        assert d32.max().item() < 6e-2 and d32.mean().item() < 6e-3, stats
        assert d32.mean().item() < 1.25 * dm.mean().item() and d32.max().item() < 2.0 * dm.max().item(), stats
        assert d16.max().item() < BF16_MODEL_TOL_MAX and d16.mean().item() < BF16_MODEL_TOL_MEAN, stats
        assert d16.mean().item() < 1.1 * dm.mean().item(), stats
    cls = out['occ_cls'].cpu().long()
    assert (cls == f32['occ'].argmax(-1)).float().mean().item() > 0.99
    assert (cls == model['occ'].argmax(-1)).float().mean().item() > 0.995


@pytest.mark.gpu
@pytest.mark.parametrize('config', ['fp32_tc_split', 'bf16_tc_fused'])
def test_full_size_four_layers(config, ref_dir):
    """The shipped configuration (200x200 BEV, 6 cameras at 928x1600, four encoder layers) against the oracle computed
    here: fp32 tensor-core split at 1e-3 on every tap and output, bf16 tensor-core fused against the storage-rounding model."""
    path = os.path.join(str(ref_dir), 'full4.pt')
    if not os.path.exists(path):
        torch.save(compute_reference(*_full4_case(), None), path)
    code = (f"import sys, torch; sys.path.insert(0, 'tests'); import test_gpu_config_space as t; "
            f"t.check_full4({config!r}, torch.load({path!r})); print('OK')")
    assert 'OK' in _run_isolated(code, timeout=900)


# ------------------------------------------------------------------------------------------ GPU: operator, reference call shapes
def _sca_max_len():
    """Queries per camera after SpatialCrossAttention's rebatch (spatial_cross_attention.py: max over cameras of the
    visible pillars) for the full-size fixture's cameras."""
    O, _ = _oracle()
    cfg = fixtures.make_cfg('full')
    pc = cfg['pc_range']
    ref_3d = O.get_reference_points(cfg['bev_h'], cfg['bev_w'], pc[5] - pc[2], cfg['num_points_in_pillar'], '3d', 1)
    _, mask = O.point_sampling(ref_3d, pc, fixtures.make_img_metas(cfg))
    return int(mask[:, 0].any(-1).sum(-1).max())


@pytest.mark.gpu
@pytest.mark.parametrize('call', ['tsa', 'sca'])
def test_ms_deform_attn_forward_at_reference_call_shapes(call):
    """`ops.ms_deform_attn_forward` with the shapes the reference hands mmcv: TemporalSelfAttention (value [2, 40000, 8,
    32], one 200x200 level, 4 points) and SpatialCrossAttention (value [6, 30825, 8, 32], the four full-size levels,
    8 points, Nq = the rebatched max_len).  Locations include out-of-map samples, exact borders and pixel centres."""
    from occnet_b200 import ops
    from oracle import msda as OM
    if call == 'tsa':
        B, levels, P, Nq = 2, [(200, 200)], 4, 40000
    else:
        B, levels, P, Nq = 6, fixtures.CFG_FULL['level_shapes'], 8, _sca_max_len()
        assert 1000 < Nq < 40000, Nq
    M, Cm, L = 8, 32, len(levels)
    shapes = torch.tensor(levels)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    Nv = int(shapes.prod(1).sum())
    g = torch.Generator().manual_seed(7)
    value = torch.randn(B, Nv, M, Cm, generator=g)
    loc = torch.rand(B, Nq, M, L, P, 2, generator=g) * 1.5 - 0.25
    loc[:, 0] = 0.0; loc[:, 1] = 1.0; loc[:, 2] = 0.5                 # borders and the centre
    loc[:, 3, ..., 0] = (torch.arange(P).float() + 0.5)[None, None] / shapes[:, 1].float()[None, :, None]   # pixel centres
    loc[:, 4, ..., 1] = 1.0 - 0.5 / shapes[:, 0].float()[None, :, None]                                     # last row centre
    loc[:, 5] = -0.5 / shapes[:, 1].float()[None, :, None, None]       # exactly one pixel outside: h_im / w_im = -1
    w = torch.rand(B, Nq, M, L, P, generator=g)
    got = ops.ms_deform_attn_forward(value.to(DEV), shapes.to(DEV), lsi.to(DEV), loc.to(DEV), w.to(DEV), 64).cpu()
    assert tuple(got.shape) == (B, Nq, M * Cm)
    want = OM.msda_grid_sample(value, shapes, loc, w)
    np.testing.assert_allclose(got.numpy(), want.numpy(), atol=1e-4, rtol=0)
    sub = torch.cat((torch.arange(6), torch.randperm(Nq - 6, generator=g)[:10] + 6))
    exact = OM.msda_loops(value.double(), shapes, lsi, loc[:, sub].double(), w[:, sub].double(), dtype=np.float64)
    np.testing.assert_allclose(got[:, sub].numpy(), exact.numpy(), atol=1e-4, rtol=0)      # fp32 sums of 16-32 samples
