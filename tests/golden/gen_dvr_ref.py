"""Generate tests/golden/ref_dvr.npz: the outputs of the reference's own ray-casting kernel (tools/ray_iou/lib/dvr,
built into oracle/_ref by oracle/build_ref.py) on the inputs of
tests/test_gpu_parity.py::test_render_forward_vs_reference_kernel.  Needs a GPU and a built oracle/_ref.

Run:  python tests/golden/gen_dvr_ref.py
"""
import glob
import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from test_gpu_parity import DVR_OUTPUTS, dvr_inputs      # noqa: E402


def main():
    so = glob.glob(os.path.join(ROOT, 'oracle', '_ref', 'dvr_ref*.so'))
    assert so, 'oracle/_ref/dvr_ref.so is missing: run `python -m oracle.build_ref` where the reference tree exists'
    spec = importlib.util.spec_from_file_location('dvr_ref', so[0])
    dvr = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(dvr)
    outs = {k: [] for k in DVR_OUTPUTS}
    for occ, o, p, ti in dvr_inputs():
        ref = dvr.render_forward(occ, o, p, ti, [1, 16, 200, 200], 'test')
        for key, t in zip(DVR_OUTPUTS, ref):
            assert t.dtype == torch.float32, (key, t.dtype)
            outs[key].append(t[0].cpu().numpy())
    path = os.path.join(ROOT, 'tests', 'golden', 'ref_dvr.npz')
    np.savez_compressed(path, **{k: np.stack(v) for k, v in outs.items()})
    print('[dvr] wrote', path, {k: np.stack(v).shape for k, v in outs.items()})


if __name__ == '__main__':
    main()
