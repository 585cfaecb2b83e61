"""CPU suite: the drop-in surface (config loading, registries, state_dict key contract) and the data-parallel host logic."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from occnet_b200 import fixtures
from occnet_b200.mmcv_shim import Config, build_detector, build_head

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


head_cfg = fixtures.head_cfg          # registry config of the head for a fixture geometry (shared with bench.py)


def shipped_config(golden_dir, tmp_path):
    """The reference's projects/configs/bevformer/bevformer_base_occ.py, reduced to plugin, plugin_dir, dist_params and
    model (written by tests/golden/gen_golden.py), laid out again as the shipped files are -- dist_params in a
    `_base_` runtime file, the rest in the config that inherits it -- and loaded through `Config.fromfile`."""
    with open(os.path.join(golden_dir, 'ref_config_base_occ.json')) as f:
        d = json.load(f)
    (tmp_path / 'default_runtime.py').write_text(f"dist_params = {d.pop('dist_params')!r}\n")
    path = tmp_path / 'bevformer_base_occ.py'
    path.write_text("_base_ = ['default_runtime.py']\n" + ''.join(f'{k} = {v!r}\n' for k, v in d.items()))
    return Config.fromfile(str(path))


def test_plugin_state_dict_keys_equal_reference(golden_dir):
    """Key contract: the drop-in head exposes exactly the parameter / buffer names of the reference head (golden
    written by tests/golden/gen_golden.py from the unmodified reference module)."""
    import projects.mmdet3d_plugin  # noqa: F401  (registers the classes)
    cfg = fixtures.make_cfg('small6')
    head = build_head(head_cfg(cfg))
    want = open(os.path.join(golden_dir, 'ref_state_dict_keys.txt')).read().split()
    assert sorted(head.state_dict().keys()) == want
    head.load_state_dict(fixtures.init_params(cfg, seed=2), strict=True)


def test_shipped_config_loads_and_builds_unchanged(golden_dir, tmp_path):
    import projects.mmdet3d_plugin  # noqa: F401
    cfg = shipped_config(golden_dir, tmp_path)
    assert cfg.plugin and cfg.plugin_dir == 'projects/mmdet3d_plugin/'
    assert cfg.model.type == 'BEVFormerOcc' and cfg.dist_params.backend == 'nccl'          # `_base_` merge works
    assert cfg.model.pts_bbox_head.transformer.encoder.num_layers == 4
    det = build_detector(cfg.model)
    head = det.pts_bbox_head
    assert type(head).__name__ == 'BEVFormerOccHead' and head.bev_h == 200 and head.num_classes == 17
    n = sum(p.numel() for p in head.parameters())
    assert abs(n - 13.63e6) < 0.05e6                                                        # SURVEY: head ~13.6 M params
    head.load_state_dict(fixtures.init_params(fixtures.make_cfg('full'), seed=2), strict=True)
    with pytest.raises(RuntimeError):                                                       # no CPU fallback
        head([torch.zeros(1, 6, 256, h, w) for h, w in fixtures.CFG_FULL['level_shapes']], fixtures.make_img_metas(fixtures.CFG_FULL))


def test_backbone_neck_containers_have_reference_keys(golden_dir, tmp_path):
    """img_backbone / img_neck of the shipped config build as parameter containers whose keys are the reference's
    (mmdet ResNet == torchvision resnet50 minus fc; mmdet FPN lateral_convs / fpn_convs) and accept the oracle's
    parameter dict unchanged."""
    import projects.mmdet3d_plugin  # noqa: F401
    from torchvision.models import resnet50
    from oracle import backbone as OB
    det = build_detector(shipped_config(golden_dir, tmp_path).model)
    sd = det.state_dict()
    bk = {k[len('img_backbone.'):] for k in sd if k.startswith('img_backbone.')}
    assert bk == {k for k in resnet50(weights=None).state_dict() if not k.startswith('fc.')}
    nk = sorted(k for k in sd if k.startswith('img_neck.'))
    assert nk == sorted(f'img_neck.{grp}.{i}.conv.{t}' for grp, n in (('lateral_convs', 3), ('fpn_convs', 4))
                        for i in range(n) for t in ('weight', 'bias'))
    p = OB.init_params(seed=5)
    missing = det.load_state_dict(p, strict=False)
    assert not missing.unexpected_keys
    assert all(k.startswith('pts_bbox_head.') or k.endswith('num_batches_tracked') for k in missing.missing_keys)
    with pytest.raises(RuntimeError):                                                       # containers only: no torch fallback
        det.img_backbone(torch.zeros(1, 3, 64, 64))
    with pytest.raises(RuntimeError):
        det.extract_feat(torch.zeros(1, 6, 3, 64, 64))


def test_contiguous_shard_rule():
    from occnet_b200.dist import contiguous_shard
    assert contiguous_shard(10, 0, 2) == [0, 1, 2, 3, 4] and contiguous_shard(10, 1, 2) == [5, 6, 7, 8, 9]
    got = [contiguous_shard(10, r, 4) for r in range(4)]                                    # ceil(10/4)=3, wrap-around pad
    assert got == [[0, 1, 2], [3, 4, 5], [6, 7, 8], [9, 0, 1]]
    assert contiguous_shard(0, 0, 2) == []
    from occnet_b200.dist import owned_unique
    assert [owned_unique(10, r, 4) for r in range(4)] == [[0, 1, 2], [0, 1, 2], [0, 1, 2], [0]]
    assert sum(len(owned_unique(7, r, 8)) for r in range(8)) == 7 and owned_unique(8, 1, 2) == [0, 1, 2, 3]
    from projects.mmdet3d_plugin.datasets.samplers import DistributedSampler
    s = DistributedSampler(list(range(10)), num_replicas=4, rank=3, shuffle=False)
    assert list(iter(s)) == [9, 0, 1]


GLOO_WORKER = r'''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["OCC_ROOT"])
from occnet_b200 import dist as od, metric
rank, local, world = od.init_from_env("gloo")
assert world == 2 and dist.get_backend() == "gloo"
frames = od.contiguous_shard(5, rank, world)
own = od.owned_unique(5, rank, world)
# per-rank counters: a deterministic function of the frames this rank owns (stands in for the GPU metric kernel).
# 5 % 2 != 0: rank 1's shard is [3, 4, 0] -- frame 0 is wrap-around padding and must NOT be counted twice
# (the reference truncates the collected results to len(dataset), apis/test.py:130).
vec = torch.zeros(metric.NUM_COUNTERS, dtype=torch.float64)
for i in own:
    rng = np.random.RandomState(frames[i])
    vec += torch.from_numpy(rng.randint(0, 50, metric.NUM_COUNTERS).astype(np.float64))
od.all_reduce_counters(vec)
want = torch.zeros_like(vec)
for f in range(5):                                                  # single-rank counters over the 5 distinct frames
    want += torch.from_numpy(np.random.RandomState(f).randint(0, 50, metric.NUM_COUNTERS).astype(np.float64))
assert torch.equal(vec, want), (vec - want).abs().max()
fin = metric.finalize_counters(vec.numpy())
assert np.isnan(fin["ave"]).sum() == 8 or True
t = od.max_over_ranks(float(rank + 1), "cpu")
assert t == 2.0
sys.stdout.write("rank %d ok %s\n" % (rank, frames)); sys.stdout.flush()
'''


def test_two_rank_gloo_shard_and_counter_allreduce(tmp_path):
    """World-size-2 run of the multi-GPU host logic on CPU: shard rule + the path's one collective."""
    script = tmp_path / 'worker.py'
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, OCC_ROOT=ROOT, MASTER_ADDR='127.0.0.1', MASTER_PORT='29533')
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2',
                        '--master-addr', '127.0.0.1', '--master-port', '29533', str(script)],
                       env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = r.stdout.replace('\n', ' ')
    assert 'ok [0, 1, 2]' in out and 'ok [3, 4, 0]' in out, r.stdout
