"""Generate tests/golden/ref_*.npz by running the UNMODIFIED reference modules in this container.

The reference's hot-path modules (`/root/reference/projects/mmdet3d_plugin/bevformer/...`) import
mmcv / mmdet at module scope; those are absent here, so `occnet_b200.mmcv_shim.install_as_mmcv()`
provides stand-ins for the third-party pieces (registries, BaseModule, FFN, ConvModule,
LearnedPositionalEncoding, `multi_scale_deformable_attn_pytorch` restated in oracle/msda.py).
Everything else -- BEVFormerEncoder.point_sampling, SpatialCrossAttention's rebatch loops,
TemporalSelfAttention, MSDeformableAttention3D, TransformerOcc, BEVFormerOccHead, and the metric's
generate_lidar_rays / process_one_sample / calc_metrics -- is the reference's own code, executed
from where it lies.  The outputs are committed as small fixtures; /root/reference does not exist
on the GPU box, so nothing else reads it at test time.

Run (CPU, ~1 min):  python tests/golden/gen_golden.py
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = '/root/reference'
OUT = os.path.join(ROOT, 'tests', 'golden')

from occnet_b200 import fixtures, mmcv_shim          # noqa: E402
from oracle import bevformer_occ as O                # noqa: E402
from oracle import msda as OM                        # noqa: E402
from oracle import ray_metrics as ORM                # noqa: E402


def _pkg(name, path):
    m = types.ModuleType(name)
    m.__path__ = [path]
    sys.modules[name] = m
    if '.' in name:
        parent, _, leaf = name.rpartition('.')
        setattr(sys.modules[parent], leaf, m)
    return m


def import_reference():
    ext = types.SimpleNamespace(ms_deform_attn_forward=None, ms_deform_attn_backward=None)
    mmcv_shim.install_as_mmcv(msda_pytorch=OM.msda_grid_sample, ext_provider=lambda name: ext)
    for stub in ('cv2', 'matplotlib', 'matplotlib.pyplot', 'prettytable'):
        m = types.ModuleType(stub)
        m.__path__ = []
        sys.modules[stub] = m
    sys.modules['matplotlib'].pyplot = sys.modules['matplotlib.pyplot']
    sys.modules['prettytable'].PrettyTable = type('PrettyTable', (), {
        '__init__': lambda self, *a, **k: None, 'add_row': lambda self, *a, **k: None,
        '__str__': lambda self: '<table>'})
    base = os.path.join(REF, 'projects')
    _pkg('projects', base)
    p = os.path.join(base, 'mmdet3d_plugin')
    _pkg('projects.mmdet3d_plugin', p)
    for sub in ('bevformer', 'bevformer/modules', 'bevformer/dense_heads', 'models', 'models/utils',
                'core', 'core/bbox', 'datasets'):
        _pkg('projects.mmdet3d_plugin.' + sub.replace('/', '.'), os.path.join(p, sub))
    mods = {}
    for name in ('encoder', 'spatial_cross_attention', 'temporal_self_attention', 'transformer_occ'):
        mods[name] = importlib.import_module('projects.mmdet3d_plugin.bevformer.modules.' + name)
    mods['head'] = importlib.import_module('projects.mmdet3d_plugin.bevformer.dense_heads.bevformer_occ_head')
    return mods


def build_reference_head(cfg):
    """Same nested config as projects/configs/bevformer/bevformer_base_occ.py:67-135 with fixture sizes."""
    C = cfg['embed_dims']
    head_cfg = dict(
        type='BEVFormerOccHead', pc_range=cfg['pc_range'], bev_h=cfg['bev_h'], bev_w=cfg['bev_w'],
        num_classes=cfg['num_classes'], in_channels=C, sync_cls_avg_factor=True, with_box_refine=True,
        as_two_stage=False, use_mask=False,
        loss_occ=dict(type='CrossEntropyLoss', use_sigmoid=False, loss_weight=1.0),
        loss_flow=dict(type='L1Loss', loss_weight=0.25),
        transformer=dict(
            type='TransformerOcc', pillar_h=cfg['pillar_h'], num_classes=cfg['num_classes'],
            norm_cfg=dict(type='BN'), norm_cfg_3d=dict(type='BN3d'), use_3d=True, use_conv=False,
            rotate_prev_bev=True, use_shift=True, use_can_bus=True, embed_dims=C, num_cams=cfg['num_cams'],
            rotate_center=cfg.get('rotate_center', [100, 100]),
            encoder=dict(
                type='BEVFormerEncoder', num_layers=cfg['num_layers'], pc_range=cfg['pc_range'],
                num_points_in_pillar=cfg['num_points_in_pillar'], return_intermediate=False,
                transformerlayers=dict(
                    type='BEVFormerLayer',
                    attn_cfgs=[
                        dict(type='TemporalSelfAttention', embed_dims=C, num_levels=1),
                        dict(type='SpatialCrossAttention', pc_range=cfg['pc_range'], num_cams=cfg['num_cams'],
                             deformable_attention=dict(type='MSDeformableAttention3D', embed_dims=C,
                                                       num_points=cfg['sca_points'], num_levels=cfg['num_levels']),
                             embed_dims=C)],
                    feedforward_channels=cfg['ffn_dim'], ffn_dropout=0.1,
                    operation_order=('self_attn', 'norm', 'cross_attn', 'norm', 'ffn', 'norm')))),
        positional_encoding=dict(type='LearnedPositionalEncoding', num_feats=C // 2,
                                 row_num_embed=cfg['bev_h'], col_num_embed=cfg['bev_w']))
    return mmcv_shim.build_head(head_cfg)


CASES = {
    # name: (cfg, batch, prev_bev?, can_bus angle)
    'toy': (fixtures.make_cfg('toy'), 1, False, None),
    'small6': (fixtures.make_cfg('small6'), 1, False, None),
    'small6_b2': (fixtures.make_cfg('small6', num_layers=1), 2, False, None),
    'small6_prev': (fixtures.make_cfg('small6', rotate_center=[20, 20]), 1, True, 3.0),
}


def subsample(t, n=4096):
    flat = t.detach().reshape(-1)
    idx = torch.linspace(0, flat.numel() - 1, min(n, flat.numel())).long()
    return flat[idx].numpy().astype(np.float32), idx.numpy().astype(np.int64)


def gen_model_goldens(mods):
    for name, (cfg, bs, with_prev, ang) in CASES.items():
        torch.manual_seed(0)
        params = O.init_params(cfg, seed=2)
        head = build_reference_head(cfg).eval()
        missing = head.load_state_dict(params, strict=True)         # proves the key contract
        if name == 'small6':
            with open(os.path.join(OUT, 'ref_state_dict_keys.txt'), 'w') as f:
                f.write('\n'.join(sorted(head.state_dict().keys())) + '\n')
        feats = fixtures.make_feats(cfg, bs=bs, seed=1)
        metas = fixtures.make_img_metas(cfg, bs=bs, can_bus_angle=ang)
        prev = None
        if with_prev:
            g = torch.Generator().manual_seed(3)
            prev = torch.randn(bs, cfg['bev_h'] * cfg['bev_w'], cfg['embed_dims'], generator=g)
        with torch.no_grad():
            ref = head(feats, metas, prev_bev=None if prev is None else prev.clone())
            occ_cls, _ = head.get_occ(ref, metas)
            ora = O.head_forward(params, cfg, feats, metas, prev_bev=None if prev is None else prev.clone())
        d = {}
        for k in ('bev_embed', 'occ', 'flow'):
            err = (ref[k] - ora[k]).abs().max().item()
            print(f'[{name}] reference-vs-oracle max|diff| {k}: {err:.3e}')
            assert err < 2e-4, (name, k, err)
            d[k + '_sub'], d[k + '_idx'] = subsample(ref[k])
            d[k + '_shape'] = np.asarray(ref[k].shape)
            d[k + '_absmean'] = np.float64(ref[k].abs().double().mean().item())
        d['occ_cls'] = occ_cls.numpy().astype(np.uint8)
        np.savez_compressed(os.path.join(OUT, f'ref_model_{name}.npz'), **d)
        print(f'[{name}] wrote ref_model_{name}.npz ({missing})')


def gen_metric_golden():
    import torch.utils.cpp_extension as cpp

    class _Dvr:
        """DDA stand-in for the JIT-compiled `dvr` extension (ray_metrics.py:12): the C restatement."""
        @staticmethod
        def render_forward(sigma, origin, points, tindex, grid, phase):
            assert phase == 'test' and sigma.shape[0] == 1
            pd, gd, ci = ORM.render_forward(sigma[0].numpy(), origin[0].numpy(), points[0].numpy(),
                                            tindex[0].numpy())
            return [torch.from_numpy(pd)[None], torch.from_numpy(gd)[None], torch.from_numpy(ci)[None]]

    real_load = cpp.load
    cpp.load = lambda *a, **k: _Dvr
    torch.Tensor.cuda = lambda self, *a, **k: self                  # no GPU here: `.cuda()` is a no-op
    torch.cuda.empty_cache = lambda: None
    try:
        rm = importlib.import_module('projects.mmdet3d_plugin.datasets.ray_metrics')
    finally:
        cpp.load = real_load
    rays = rm.generate_lidar_rays()
    assert np.array_equal(rays, ORM.generate_lidar_rays())
    sem_gt, flow_gt = fixtures.make_occ_scene(seed=4)
    rng = np.random.RandomState(5)
    sem_pred = np.roll(sem_gt, 1, axis=0).copy()
    flip = rng.rand(*sem_pred.shape) < 0.03
    sem_pred[flip] = rng.randint(0, 17, int(flip.sum())).astype(np.uint8)
    flow_pred = (np.roll(flow_gt, 1, axis=0) + rng.normal(0, 0.5, flow_gt.shape)).astype(np.float32)
    orig2 = fixtures.make_ray_origins(T=2)
    pcd_pred = rm.process_one_sample(sem_pred, torch.from_numpy(rays), torch.from_numpy(orig2), flow_pred)
    pcd_gt = rm.process_one_sample(sem_gt, torch.from_numpy(rays), torch.from_numpy(orig2), flow_gt)
    mine_pred = ORM.process_one_sample(sem_pred, rays, orig2, flow_pred)
    assert np.array_equal(pcd_pred, mine_pred), np.abs(pcd_pred - mine_pred).max()
    valid = pcd_gt[:, 0].astype(np.int32) != 16
    iou_list, ave_list = rm.calc_metrics([pcd_pred[valid]], [pcd_gt[valid]])
    cnt = ORM.accumulate(ORM.new_counters(), pcd_pred[valid], pcd_gt[valid])
    fin = ORM.finalize(cnt)
    assert np.allclose(np.stack(iou_list), fin['iou'], equal_nan=True)
    assert np.allclose(ave_list, fin['ave'], equal_nan=True)
    np.savez_compressed(os.path.join(OUT, 'ref_metric.npz'),
                        rays_first=rays[:4], rays_last=rays[-4:], rays_sum=rays.astype(np.float64).sum(0),
                        pcd_pred=pcd_pred.astype(np.float32), pcd_gt_cls=pcd_gt[:, 0].astype(np.uint8),
                        pcd_gt_dist=pcd_gt[:, 1].astype(np.float32),
                        iou=np.stack(iou_list), ave=np.asarray(ave_list),
                        counters=ORM.counters_to_vector(cnt))
    print('[metric] wrote ref_metric.npz; miou', fin['miou'], 'mave', fin['mave'])


def gen_config_golden():
    """The shipped config as `Config.fromfile` loads it (`_base_` files merged), reduced to the keys the drop-in tests
    read: plugin, plugin_dir, dist_params and the model."""
    import json
    cfg = mmcv_shim.Config.fromfile(os.path.join(REF, 'projects', 'configs', 'bevformer', 'bevformer_base_occ.py'))
    keep = {k: cfg[k] for k in ('plugin', 'plugin_dir', 'dist_params', 'model')}
    with open(os.path.join(OUT, 'ref_config_base_occ.json'), 'w') as f:
        json.dump(keep, f, indent=1)
        f.write('\n')
    print('[config] wrote ref_config_base_occ.json')


if __name__ == '__main__':
    mods = import_reference()
    gen_model_goldens(mods)
    gen_metric_golden()
    gen_config_golden()
