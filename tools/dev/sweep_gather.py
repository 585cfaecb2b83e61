"""Dev aid (not a test): time one engine configuration (env knobs are read at first launch) and print
ms/frame + per-category ms, plus max |diff| of occ logits against a reference run saved by the first call.
  python tools/dev/sweep_gather.py TAG   (env: OCC_NO_L0_FOLD, OCC_GEMM_TIMELINE, OCC_TEST_OFFSCALE)"""
import json, os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from occnet_b200 import fixtures
from occnet_b200.engine import OccEngine

tag = sys.argv[1] if len(sys.argv) > 1 else 'run'
steps = 10
cfg = fixtures.make_cfg('full', num_layers=6) if hasattr(fixtures, 'make_cfg') else fixtures.CFG_FULL
dev = torch.device('cuda:0')
params = fixtures.init_params(cfg, seed=2)
if os.environ.get('OCC_TEST_OFFSCALE'):            # experiment: shrink / spread the SCA sampling offsets (line sharing between heads)
    sc = float(os.environ['OCC_TEST_OFFSCALE'])
    for k in list(params):
        if 'attentions.1.deformable_attention.sampling_offsets' in k:
            params[k] = params[k] * sc
eng = OccEngine(cfg, params, precision='bf16', use_tensor_cores=True, device='cuda:0')
eng.set_cameras(fixtures.make_img_metas(cfg))
frames = [[f[0].contiguous().to(dev) for f in fixtures.make_feats(cfg, bs=1, seed=100 + i)] for i in range(3)]
want = ('flow', 'occ', 'occ_cls')
out = eng.forward(frames[0], want=want)
occ = out['occ'].float().cpu().numpy()
ref_path = 'gpurun_out/_sweep_ref.npy'
diff = None
if os.path.exists(ref_path):
    ref = np.load(ref_path)
    diff = float(np.abs(ref - occ).max())
else:
    os.makedirs('gpurun_out', exist_ok=True)
    np.save(ref_path, occ)
for i in range(3):
    eng.forward(frames[i % 3], want=('flow', 'occ_cls'))
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(steps):
    eng.forward(frames[i % 3], want=('flow', 'occ_cls'))
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / steps
eng.profile(True)
for i in range(steps):
    eng.forward(frames[i % 3], want=('flow', 'occ_cls'))
prof = eng.profile_read()
eng.profile(False)
print(json.dumps({'tag': tag, 'ms_per_frame': round(ms, 4), 'occ_maxdiff_vs_first': diff,
                  'cat_ms': {k: round(v[0] / steps, 4) for k, v in prof.items()}}), flush=True)
