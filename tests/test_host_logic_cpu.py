"""Host-side logic added in round 2, checked without a GPU: the T32 block layout for any column count (mirror of the CUDA tiler
and of the GEMM epilogue's read), the committed profile summaries (regenerated from the committed raw ncu export), and the
submission writer's argument checks."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _t32_index(row, col, ncols):
    """elementwise.cu: t32_convert_kernel (float index of element (row, col) of a [rows, ncols] matrix in the T32 layout)."""
    return ((((row >> 5) * (ncols >> 5) + (col >> 5)) * 8 + ((col & 31) >> 2)) * 32 + (row & 31)) * 4 + (col & 3)


@pytest.mark.parametrize('ncols', [192, 256])
def test_t32_layout_is_a_permutation_and_matches_the_epilogue_read(ncols):
    rows = 96
    idx = np.array([[_t32_index(r, c, ncols) for c in range(ncols)] for r in range(rows)])
    assert sorted(idx.reshape(-1)) == list(range(rows * ncols))                    # a permutation of the padded matrix
    # gemm_tc.cu epilogue: thread `lane` of the warp that owns rows row0..row0+31 reads, for the 32-column chunk
    # starting at column col, the float4s  ((row0 >> 5) * (N >> 5) + (col >> 5)) * 256 + lane + j * 32,  j = 0..7
    for row0 in (0, 32, 64):
        for col in range(0, ncols, 32):
            for lane in (0, 5, 31):
                for j in range(8):
                    f4 = ((row0 >> 5) * (ncols >> 5) + (col >> 5)) * 256 + lane + j * 32
                    want = [_t32_index(row0 + lane, col + 4 * j + k, ncols) for k in range(4)]
                    assert want == [4 * f4 + k for k in range(4)]
    # a warp instruction (fixed j) touches 32 consecutive float4 = 512 contiguous bytes: the point of the layout
    lane_addr = [(((0 >> 5) * (ncols >> 5) + 0) * 256 + lane + 3 * 32) for lane in range(32)]
    assert lane_addr == list(range(lane_addr[0], lane_addr[0] + 32))


def test_committed_profile_summaries_regenerate_from_the_committed_raw_export(tmp_path):
    """profiles/r2_traffic.json (read by bench.py for `roofline.traffic`) is a pure function of profiles/r2_frame_ncu_raw.csv."""
    raw = os.path.join(ROOT, 'profiles', 'r2_frame_ncu_raw.csv')
    want = json.load(open(os.path.join(ROOT, 'profiles', 'r2_traffic.json')))
    work = tmp_path / 'profiles'
    work.mkdir()
    for f in ('summarize.py',):
        (work / f).write_text(open(os.path.join(ROOT, 'profiles', f)).read())
    r = subprocess.run([sys.executable, str(work / 'summarize.py'), '--frame', 'r2', raw], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    got = json.load(open(work / 'r2_traffic.json'))
    assert set(got) == set(want)
    for k in want:
        assert got[k]['captured_launches'] == want[k]['captured_launches']
        assert abs(got[k]['dram_bytes_per_frame'] - want[k]['dram_bytes_per_frame']) < 1.0
    assert sum(v['launches_per_frame'] for v in got.values()) <= 51 and got['gemm']['launches_per_frame'] == 35


def test_submission_writer_checks_its_arguments_before_touching_the_gpu():
    from projects.mmdet3d_plugin.datasets import submission as sub
    with pytest.raises(AssertionError):
        sub.format_results([{'occ_results': np.zeros((200, 200, 16)), 'flow_results': np.zeros((200, 200, 16, 2))}], ['a', 'b'],
                           [np.zeros((1, 2, 3), np.float32)])
    assert set(sub.SUBMISSION_META) == {'method', 'team', 'authors', 'e-mail', 'institution / company', 'country / region'}


def test_head_softplus_polynomial_is_within_bf16_noise_of_softplus():
    """head_tc.cu: softplus(x) = max(x, 0) + t * P5(t), t = exp(-|x|): the degree-5 minimax coefficients used by the kernel,
    evaluated here in fp32 like the kernel (Horner, fused steps not modelled), against log1p(exp(x)) in fp64."""
    C = [0.9999929070472717, -0.4994262754917145, 0.32572421431541443, -0.211494579911232, 0.10287206619977951,
         -0.024528255686163902]
    x = np.concatenate([np.linspace(-30, 30, 200001), np.random.RandomState(0).normal(0, 3, 200000)]).astype(np.float32)
    t = np.exp(-np.abs(x.astype(np.float64))).astype(np.float32)
    p = np.full_like(t, np.float32(C[5]))
    for c in C[4::-1]:
        p = (p * t + np.float32(c)).astype(np.float32)
    got = (t * p + np.maximum(x, np.float32(0))).astype(np.float64)
    want = np.logaddexp(0.0, x.astype(np.float64))
    rel = np.abs(got - want) / want
    assert rel.max() < 2e-5, rel.max()                              # the hidden activations are then rounded to bf16 (2^-9 = 2e-3)
    assert np.abs(got - want).max() < 1e-5


def test_pack_transpose_swizzle_is_conflict_free_and_consistent():
    """elementwise.cu pack_levels_kernel (bf16 features): element (pixel p, channel c) of the 64 x 64 tile lives at
    p*64 + (((c >> 3) ^ (p >> 3)) << 3 | (c & 7)).  Writer: thread (c = idx >> 3, p8 = (idx & 7) * 8) stores its 8 pixels;
    reader: thread (p = idx >> 3, c8 = (idx & 7) * 8) loads 8 channels as one 16-byte piece."""
    def addr(p, c):
        return p * 64 + ((((c >> 3) ^ (p >> 3)) << 3) | (c & 7))
    assert sorted(addr(p, c) for p in range(64) for c in range(64)) == list(range(64 * 64))
    for p in range(64):                                              # reader: 8 consecutive channels are contiguous and 16-B aligned
        for c8 in range(0, 64, 8):
            a = [addr(p, c8 + k) for k in range(8)]
            assert a == list(range(a[0], a[0] + 8)) and a[0] % 8 == 0
    # writer: for a fixed k, the 32 lanes of a warp (4 channels x 8 pixel groups) hit 16 distinct 4-byte banks, 2 lanes per word
    for i in range(2):
        for warp in range(8):
            for k in range(8):
                banks = []
                for lane in range(32):
                    idx = warp * 32 + lane + i * 256
                    c, p8 = idx >> 3, (idx & 7) * 8
                    banks.append((addr(p8 + k, c) * 2 // 4) % 32)
                assert len(set(banks)) == 16 and all(banks.count(b) == 2 for b in set(banks))
    # reader: a quarter-warp (8 lanes = one pixel, 8 pieces) covers one full 128-byte row
    for p in range(64):
        pieces = sorted(addr(p, c8) * 2 // 16 for c8 in range(0, 64, 8))
        assert pieces == list(range(p * 8, p * 8 + 8))
