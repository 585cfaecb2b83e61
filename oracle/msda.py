"""ORACLE (test infrastructure only -- never imported by the product path).

CPU restatement of the multi-scale deformable attention operator that the reference
reaches through `mmcv` (third-party, NOT vendored under /root/reference, version
unpinned by the repo; BEVFormer's install page names mmcv-full 1.4.0):

  * `mmcv.ops.multi_scale_deform_attn.multi_scale_deformable_attn_pytorch`
      call sites: spatial_cross_attention.py:395-396, temporal_self_attention.py:252-253
  * `mmcv._ext.ms_deform_attn_forward`  (CUDA; same arithmetic, one thread per channel)
      call sites: multi_scale_deformable_attn_function.py:42-48, 118-124

Published algorithm (Deformable-DETR / mmcv): for every batch b, query q, head m

    out[b,q,m*C+c] = sum_l sum_p  w[b,q,m,l,p] * bilinear(value_l[b,:,m,c]; x*W_l-0.5, y*H_l-0.5)

with zero padding outside the map.  `msda_grid_sample` follows mmcv's CPU fallback
(per level F.grid_sample(..., bilinear, zeros, align_corners=False) on 2*loc-1);
`msda_loops` follows the CUDA kernel's scalar formulation (skip unless
-1 < h_im < H and -1 < w_im < W; corner valid iff inside) and is the bit-level
statement of the corner indexing the CUDA path must reproduce.

Parity status: UNPINNED upstream (the reference ships no tests or golden vectors,
SURVEY section 4).  Cross-checked in tests/test_oracle_cpu.py against the independent
implementation in transformers/models/mask2former/modeling_mask2former.py:798-837.
"""
import numpy as np
import torch
import torch.nn.functional as F


def msda_grid_sample(value, value_spatial_shapes, sampling_locations, attention_weights):
    """value (B, Nv, M, C); shapes (L, 2) [h, w]; loc (B, Nq, M, L, P, 2) [x, y] in [0,1];
    weights (B, Nq, M, L, P)  ->  (B, Nq, M*C)."""
    bs, _, num_heads, embed_dims = value.shape
    _, num_queries, num_heads, num_levels, num_points, _ = sampling_locations.shape
    sizes = [int(h) * int(w) for h, w in value_spatial_shapes]
    value_list = value.split(sizes, dim=1)
    grids = 2 * sampling_locations - 1
    per_level = []
    for lvl, (h, w) in enumerate(value_spatial_shapes):
        h, w = int(h), int(w)
        # (B, hw, M, C) -> (B*M, C, h, w)
        v = value_list[lvl].flatten(2).transpose(1, 2).reshape(bs * num_heads, embed_dims, h, w)
        # (B, Nq, M, P, 2) -> (B*M, Nq, P, 2)
        g = grids[:, :, :, lvl].transpose(1, 2).flatten(0, 1)
        per_level.append(F.grid_sample(v, g, mode='bilinear', padding_mode='zeros', align_corners=False))
    # (B, Nq, M, L, P) -> (B*M, 1, Nq, L*P)
    w_ = attention_weights.transpose(1, 2).reshape(bs * num_heads, 1, num_queries, num_levels * num_points)
    out = (torch.stack(per_level, dim=-2).flatten(-2) * w_).sum(-1)
    return out.view(bs, num_heads * embed_dims, num_queries).transpose(1, 2).contiguous()


def msda_loops(value, value_spatial_shapes, level_start_index, sampling_locations, attention_weights, dtype=np.float32):
    """Scalar (numpy) statement of the CUDA kernel's arithmetic; small cases only.  `dtype` np.float32 restates the
    kernel's fp32 rounding, np.float64 gives the operator's value to ~1e-15."""
    v = value.detach().cpu().numpy().astype(dtype)
    loc = sampling_locations.detach().cpu().numpy().astype(dtype)
    aw = attention_weights.detach().cpu().numpy().astype(dtype)
    B, Nv, M, C = v.shape
    _, Nq, _, L, P, _ = loc.shape
    out = np.zeros((B, Nq, M, C), dtype)
    fl = np.dtype(dtype).type
    for b in range(B):
        for q in range(Nq):
            for m in range(M):
                acc = np.zeros(C, dtype)
                for l in range(L):
                    H = int(value_spatial_shapes[l][0]); W = int(value_spatial_shapes[l][1])
                    base = int(level_start_index[l])
                    for p in range(P):
                        w_im = fl(loc[b, q, m, l, p, 0] * fl(W) - fl(0.5))
                        h_im = fl(loc[b, q, m, l, p, 1] * fl(H) - fl(0.5))
                        if not (h_im > -1 and w_im > -1 and h_im < H and w_im < W):
                            continue
                        h_lo = int(np.floor(h_im)); w_lo = int(np.floor(w_im))
                        lh = fl(h_im - fl(h_lo)); lw = fl(w_im - fl(w_lo))
                        hh = fl(1) - lh; hw = fl(1) - lw
                        val = np.zeros(C, dtype)
                        if h_lo >= 0 and w_lo >= 0:
                            val += fl(hh * hw) * v[b, base + h_lo * W + w_lo, m]
                        if h_lo >= 0 and w_lo + 1 <= W - 1:
                            val += fl(hh * lw) * v[b, base + h_lo * W + w_lo + 1, m]
                        if h_lo + 1 <= H - 1 and w_lo >= 0:
                            val += fl(lh * hw) * v[b, base + (h_lo + 1) * W + w_lo, m]
                        if h_lo + 1 <= H - 1 and w_lo + 1 <= W - 1:
                            val += fl(lh * lw) * v[b, base + (h_lo + 1) * W + w_lo + 1, m]
                        acc += aw[b, q, m, l, p] * val
                out[b, q, m] = acc
    return torch.from_numpy(out.reshape(B, Nq, M * C))
