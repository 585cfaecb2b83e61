"""Image backbone + neck engine (ResNet-50 + FPN in front of the hot path; SURVEY 8f rank 1).

    reference: BEVFormerOcc.extract_img_feat, detectors/bevformer_occ.py:66-99
               (img_backbone / img_neck configured in projects/configs/bevformer/bevformer_base_occ.py:48-66)

Validated on the GPU against its oracle (tests/test_backbone_gpu.py; oracle/backbone.py is pinned bit-exactly to
torchvision's resnet50 / FeaturePyramidNetwork).  The arithmetic happens in libocc_b200 through the C ABI
(`occb200_backbone_*`); torch is only the tensor container.  There is no CPU or torch fallback.
"""
import ctypes

import numpy as np
import torch

from . import _lib


def _is_param(key):
    return (key.startswith('img_backbone.') or key.startswith('img_neck.')) and not key.endswith('num_batches_tracked')


class BackboneEngine:
    """state_dict: the detector's `state_dict()` (or any mapping holding its img_backbone.* / img_neck.* entries)."""

    def __init__(self, state_dict, num_images, img_hw, precision='fp32', use_tensor_cores=None, device='cuda:0'):
        self.device = torch.device(device)
        if not torch.cuda.is_available() or self.device.type != 'cuda':
            raise RuntimeError('libocc_b200 backbone needs a CUDA device (there is no CPU path)')
        assert precision in ('fp32', 'bf16')
        self.lib = _lib.load()
        self.precision = precision
        self.num_images, (self.H, self.W) = int(num_images), (int(img_hw[0]), int(img_hw[1]))
        tc = (precision == 'bf16') if use_tensor_cores is None else bool(use_tensor_cores)
        with torch.cuda.device(self.device):
            self._h = self.lib.occb200_backbone_create(self.num_images, self.H, self.W, 1 if precision == 'bf16' else 0, int(tc))
            if not self._h:
                raise RuntimeError(self.lib.occb200_last_error().decode())
            for k, v in state_dict.items():
                if not _is_param(k):
                    continue
                a = np.ascontiguousarray(v.detach().float().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v, np.float32))
                _lib.check(self.lib.occb200_backbone_load_param(self._h, k.encode(), a.ctypes.data_as(ctypes.c_void_p), a.size))
            _lib.check(self.lib.occb200_backbone_finalize(self._h))
        self.level_shapes = []
        for l in range(4):
            h, w = ctypes.c_int(), ctypes.c_int()
            _lib.check(self.lib.occb200_backbone_level_shape(self._h, l, ctypes.byref(h), ctypes.byref(w)))
            self.level_shapes.append((h.value, w.value))

    def forward(self, img, channels_last_bf16=False):
        """img (num_images, 3, H, W) CUDA fp32 -> list of 4 x (num_images, 256, h_l, w_l) CUDA fp32; with
        `channels_last_bf16` (bf16 engines only) the levels come back as bf16 tensors of the same SHAPE whose memory is
        channels-last (num_images, h_l, w_l, 256) -- written directly by the last convolutions, and consumed as is by
        `OccEngine` (`set_input_dtype(torch.bfloat16, channels_last=True)`): no NCHW fp32 copy, no transpose."""
        if not (isinstance(img, torch.Tensor) and img.is_cuda):
            raise RuntimeError('img must be a CUDA tensor (libocc_b200 has no CPU path)')
        assert tuple(img.shape) == (self.num_images, 3, self.H, self.W), img.shape
        img = img.float().contiguous()
        if channels_last_bf16:
            if self.precision != 'bf16':
                raise RuntimeError('channels_last_bf16 output needs a bf16 backbone engine')
            outs = [torch.empty((self.num_images, h, w, 256), dtype=torch.bfloat16, device=img.device) for h, w in self.level_shapes]
            with torch.cuda.device(img.device):
                _lib.check(self.lib.occb200_backbone_forward_nhwc_bf16(self._h, _lib.ptr(img), *[_lib.ptr(o) for o in outs],
                                                                       _lib.stream_ptr()))
            return [o.permute(0, 3, 1, 2) for o in outs]
        outs = [torch.empty((self.num_images, 256, h, w), dtype=torch.float32, device=img.device) for h, w in self.level_shapes]
        with torch.cuda.device(img.device):
            _lib.check(self.lib.occb200_backbone_forward(self._h, _lib.ptr(img), *[_lib.ptr(o) for o in outs], _lib.stream_ptr()))
        return outs

    def __del__(self):
        h = getattr(self, '_h', None)
        if h:
            self.lib.occb200_backbone_destroy(h)
            self._h = None
