#!/usr/bin/env python
"""Benchmark of the camera->occupancy hot path (BASELINE.json metric: samples/s, one sample = one 6-camera
frame's FPN features -> 200x200x16 semantic + flow volume).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA path through the C ABI)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle restatement) on host cores

Workload (config.workload): BASELINE configs[3] on top of configs[1]/[2] -- 6 x (928x1600-padded) cameras, FPN levels
116x200/58x100/29x50/15x25, 200x200 BEV, 6-layer BEVFormerEncoder (TSA + SCA + FFN), Conv3d voxel decoder
200x200x16, 17-class semantic + 2-channel flow heads, bf16 storage / fp32 accumulation.  Synthetic features,
random-init weights (fixtures.py).  One step = --frames-per-step (32) frames.  Frames are independent: N GPUs run N frame
streams (weak scaling) and the only collective is the final all-reduce of the 187 metric counters.

Timing: W >= 3 warm-up steps; K steps bracketed by barrier + cuda synchronize; device time from CUDA events on the
launch stream, max over ranks.  Each step reads a different 189 MB input frame (3 rotating frames > 126 MB L2).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from occnet_b200 import dist as occdist          # noqa: E402
from occnet_b200 import fixtures                 # noqa: E402

METRIC = 'samples/s (6-cam->200x200x16 voxel)'


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sust=d.get('bf16_tflops_sustained', d['bf16_tflops']),
                    source='measured')
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source='fallback')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def workload_cfg(args):
    return fixtures.make_cfg('full', num_layers=args.layers)


def algorithmic_work(cfg, s, tc=True, feat_bytes=4):
    """Per-frame algorithmic bytes / flops by kernel category (DESIGN.md section 4; SURVEY 8d).
    `tc`: tensor-core path (fp16 sampling projections, self-mode TSA projection folded over the constant pos)."""
    qb = 2 if (tc and s == 2) else 4                                  # bytes per sampling offset / attention logit
    Nq = cfg['bev_h'] * cfg['bev_w']
    Nv = sum(h * w for h, w in cfg['level_shapes'])
    nc, L, C, F = cfg['num_cams'], cfg['num_layers'], 256, cfg['ffn_dim']
    sca_bytes = nc * Nv * C * s + Nq * 768 * qb + Nq * C * s         # value + offsets/logits + output, per launch
    tsa_bytes = Nq * C * s + Nq * 192 * qb + Nq * C * s
    gemm_flops = L * 2 * (Nq * C * C            # TSA value_proj
                          + Nq * 192 * 2 * C    # TSA offsets + weights (K = 512)
                          + Nq * C * C          # TSA output_proj
                          + Nq * 768 * C        # SCA offsets + weights
                          + nc * Nv * C * C     # SCA value_proj over all camera tokens
                          + Nq * C * C          # SCA output_proj
                          + 2 * Nq * C * F)     # FFN
    nvox = cfg['bev_h'] * cfg['bev_w'] * cfg['pillar_h']
    conv_flops = 2 * nvox * 27 * (16 * 32 + 32 * 32)
    head_flops = 2 * nvox * (32 * 64 + 64 * cfg['num_classes'] + 32 * 64 + 64 * 2)
    # dense layers as launched on the tensor-core path (fused LayerNorm epilogues, value_proj of all layers hoisted):
    # compulsory bytes = operands read + results written (weights are KB-sized and stay in SMEM / L2)
    ntok = nc * Nv
    per_layer = (Nq * C * s + Nq * C * s                              # TSA value_proj
                 + (Nq * C * s + Nq * 192 * 4 if qb == 2 else Nq * 2 * C * s) + Nq * 192 * qb   # TSA offsets+weights (folded: q + fp32 const)
                 + 2 * (Nq * C * s + Nq * C * 4 + Nq * C * 4 + Nq * C * s)   # out_proj + LN (TSA, SCA): A, residual, y fp32, y bf16
                 + Nq * C * s + Nq * 768 * qb                          # SCA offsets+weights
                 + Nq * C * s + Nq * F * s                             # FFN1
                 + Nq * F * s + Nq * C * (4 + 4 + s)                   # FFN2 + LN: A, residual, y fp32, y bf16
                 + (0 if qb == 2 else Nq * C * (s + 4)))               # (unfolded path only: y+pos bf16 out, pos in)
    gemm_bytes = L * per_layer + ntok * C * s + L * ntok * C * s      # + hoisted SCA value_proj (tokens in, L value maps out)
    pack_bytes = ntok * C * feat_bytes + ntok * C * s
    conv_bytes = nvox * (16 * s + 32 * s) + nvox * (32 * s + 32 * s)
    head_bytes = nvox * (32 * s + 2 * 4 + 1)
    return dict(sca_bytes_per_launch=sca_bytes, tsa_bytes_per_launch=tsa_bytes, gemm_flops=gemm_flops,
                gemm_bytes=gemm_bytes, pack_bytes=pack_bytes, conv_bytes=conv_bytes, head_bytes=head_bytes,
                conv_flops=conv_flops, head_flops=head_flops, Nq=Nq, Nv=Nv)


def bind_to_gpu_numa_node(local):
    """Host plumbing for the e2e leg: run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA node
    the GPU hangs off, so that N ranks do not all stream their frames through one socket.  Best effort."""
    try:
        pr = torch.cuda.get_device_properties(local)
        dev = f'{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0'
        cpus = open(f'/sys/bus/pci/devices/{dev}/local_cpulist').read().strip()
        ids = set()
        for part in cpus.split(','):
            a, _, b = part.partition('-')
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
            return f'{dev}: cpus {cpus}'
    except Exception as e:                                            # noqa: BLE001
        return f'not bound ({type(e).__name__})'
    return 'not bound'


def golden_parity(out, tag):
    """max |engine - golden| on the committed full-size subsamples (tests/golden/gen_fullsize.py): parity evidence that
    travels with the bench line without running the oracle inside the timed job."""
    gd = os.path.join(ROOT, 'tests', 'golden')
    sys.path.insert(0, gd)
    from sampling import N_OUT, sub_idx
    res = {}
    for name, fn in (('fp32_oracle', 'full6_fp32.npz'), ('bf16_storage_model', 'full6_bf16.npz')):
        path = os.path.join(gd, fn)
        if not os.path.exists(path):
            continue
        g = np.load(path)
        r = {}
        for key, t in (('occ', out['occ']), ('flow', out['flow'])):
            flat = t.reshape(-1).float().cpu()
            d = np.abs(flat[torch.from_numpy(sub_idx(key, flat.numel(), N_OUT))].numpy() - g[key + '_sub'])
            r[key + '_max_abs'] = round(float(d.max()), 6); r[key + '_mean_abs'] = round(float(d.mean()), 7)
        r['class_agreement'] = round(float((out['occ_cls'].cpu().numpy() == g['occ_cls']).mean()), 6)
        res[name] = r
    return res


def ray_parity(out, rm_cls, dev):
    """Ray-mIoU as the reference's metric sees the CUDA output: scored against the ORACLE's output of the same frame
    (golden class / flow volumes standing in as ground truth) and, like the oracle's own output, against the synthetic
    GT scene."""
    path = os.path.join(ROOT, 'tests', 'golden', 'full6_fp32.npz')
    if not os.path.exists(path):
        return None
    g = np.load(path)
    rm = rm_cls(str(dev))
    rm.add_frame(out['occ_cls'], out['flow'], torch.from_numpy(g['occ_cls']), torch.from_numpy(g['flow_f16'].astype(np.float32)),
                 torch.from_numpy(fixtures.make_ray_origins(T=8)))
    fin = rm.finalize()
    return {'miou_vs_oracle_output': round(fin['miou'], 6), 'mave_vs_oracle_output': round(fin['mave'], 6),
            'oracle_miou_vs_gt_scene': float(g['miou']), 'frame': 'seed 100 (the golden frame)'}


DUMP_BYTES = 60 * 10**6                                             # data of all files; stays under 64 MB with the headers


def dump_outputs(outs, path):
    """The last timed step's engine outputs -> <path>/<name>.npy in float32, stacked over the step's frames:
    (frames, X, Y, Z[, 2]).  Above DUMP_BYTES in all, every frame keeps the same seeded sample of voxels (row-major
    (X, Y, Z) order): (frames, voxels[, 2])."""
    os.makedirs(path, exist_ok=True)
    names = sorted(outs[0])
    nvox = int(np.prod(outs[0][names[0]].shape[:3]))                # every output is (X, Y, Z, ...)
    per_voxel = sum(outs[0][k].numel() // nvox for k in names) * 4 * len(outs)
    idx = None
    if per_voxel * nvox > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(nvox, DUMP_BYTES // per_voxel, replace=False))
        idx = torch.from_numpy(idx).to(outs[0][names[0]].device)
    for k in names:
        a = torch.stack([o[k] if idx is None else o[k].flatten(0, 2)[idx] for o in outs]).float()
        np.save(os.path.join(path, k + '.npy'), a.cpu().numpy())


def timed_region(run_steps, steps, barrier):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    run_steps(steps)
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


def run_ours(args):
    rank, local, world = occdist.init_from_env('nccl')
    assert torch.cuda.is_available(), 'bench.py needs a GPU for the product arm (no CPU fallback)'
    dev = torch.device(f'cuda:{local}')
    torch.cuda.set_device(dev)
    numa = bind_to_gpu_numa_node(local)
    import torch.distributed as dist
    from occnet_b200.engine import OccEngine
    from occnet_b200 import metric
    cfg = workload_cfg(args)
    params = fixtures.init_params(cfg, seed=2, free_bias=fixtures.FREE_BIAS)
    metas = fixtures.make_img_metas(cfg)
    use_tc = bool(args.tc)
    eng = OccEngine(cfg, params, precision=args.precision, use_tensor_cores=use_tc, device=str(dev))
    eng.set_cameras(metas)
    _, vis_mask = eng.project_pillars()
    n_hit = int(vis_mask.any(dim=2).sum().item())                   # visible (camera, pillar) pairs = SCA work items
    NF, F, K = 3, args.frames_per_step, args.steps
    W = max(args.warmup, 3)
    feat_dtype = torch.bfloat16 if args.precision == 'bf16' else torch.float32     # features in the storage precision
    frames_f32 = [[f[0].contiguous() for f in fixtures.make_feats(cfg, bs=1, seed=100 + rank * NF + i)] for i in range(NF)]
    frames_host = [[f.to(feat_dtype).contiguous().pin_memory() for f in fr] for fr in frames_f32]
    frames_dev = [[f.to(dev) for f in fr] for fr in frames_host]
    eng.set_input_dtype(feat_dtype)
    want = ('flow', 'occ_cls')

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last_step = []                                                  # --dump-outputs: outputs of the last step run

    def run_steps(n):                                               # one step = F frames through the engine
        last_step.clear()
        for i in range(n * F):
            out = eng.forward(frames_dev[i % NF], want=want)
            if args.dump_outputs and i >= (n - 1) * F:
                last_step.append(out)

    # ---- device-resident throughput (`value`): >= 1 s of warm-up, then `repeats` regions of EXACTLY K steps, median
    run_steps(W)
    barrier()
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < 1.0:
        run_steps(1)
        torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    reps = [occdist.max_over_ranks(timed_region(run_steps, K, barrier), dev) for _ in range(args.repeats)]
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(last_step, args.dump_outputs)
    ms_med = float(np.median(reps))
    launches = eng.launches_per_frame

    # ---- per-kernel timing (CUDA events inside the engine, same stream): 2 steps
    eng.profile(True)
    prof_frames = 2 * F
    for i in range(prof_frames):
        eng.forward(frames_dev[i % NF], want=want)
    prof = eng.profile_read()
    eng.profile(False)

    # ---- end to end through the host-buffer C-ABI calls: every frame's features go host->device (pinned) and the
    #      results device->host inside the timed region; two frames in flight (submit/wait)
    def stream(n_frames, frames):
        n = 0
        for _ in eng.stream_host(frames[i % NF] for i in range(n_frames)):
            n += 1
        assert n == n_frames

    def e2e_leg(frames, k):
        stream(NF, frames)
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        stream(k * F, frames)
        e1.record()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        return occdist.max_over_ranks(max(e0.elapsed_time(e1), wall), dev)   # copies run on side streams: wall clock too

    e2e_reps = [e2e_leg(frames_host, K) for _ in range(args.repeats)]
    e2e_ms = float(np.median(e2e_reps))
    h2d = sum(f.numel() * f.element_size() for f in frames_host[0]) * F
    X, Y, Z = eng.vox_shape
    d2h = (X * Y * Z * 8 + X * Y * Z * 2 * 4) * F
    e2e_sync = None
    if world == 1:                                                  # one synchronous forward_host call per frame
        for i in range(2):
            eng.forward_host(frames_host[i % NF])
        ts = time.perf_counter()
        for i in range(2 * F):
            eng.forward_host(frames_host[i % NF])
        e2e_sync = 2 * F / (time.perf_counter() - ts)
    e2e_f32 = None
    if world == 1 and feat_dtype != torch.float32:                  # the reference's feature dtype over PCIe (189 MB/frame)
        eng.set_input_dtype(torch.float32)
        f32_host = [[f.pin_memory() for f in fr] for fr in frames_f32]
        e2e_f32 = world * 4 * F / (e2e_leg(f32_host, 4) * 1e-3)
        del f32_host
        eng.set_input_dtype(feat_dtype)

    # ---- parity of THIS configuration on the golden frame + the path's single collective (187 Ray-mIoU counters)
    chk = eng.forward(frames_dev[0], want=('occ', 'flow', 'occ_cls'))
    parity = golden_parity(chk, 'ours') if rank == 0 else None
    rayp = ray_parity(chk, metric.RayMetric, dev) if rank == 0 else None
    rm = metric.RayMetric(str(dev))
    sem_gt, flow_gt = fixtures.make_occ_scene(seed=4)
    rm.add_frame(chk['occ_cls'], chk['flow'], torch.from_numpy(sem_gt), torch.from_numpy(flow_gt),
                 torch.from_numpy(fixtures.make_ray_origins(T=8)))
    rm.all_reduce()
    fin = rm.finalize()
    numa_all = [numa]
    if world > 1:
        numa_all = [None] * world
        dist.all_gather_object(numa_all, numa)

    # ---- extra single-GPU legs (rank 0, N = 1 only): drop-in module call, fp32 configuration, stock-kernel comparator
    dropin = fp32_leg = eager = temporal = None
    if world == 1:
        temporal = run_temporal_leg(args, cfg, eng, frames_dev)
        dropin = run_dropin_leg(args, cfg, params, metas, frames_host, dev) if not args.no_dropin else None
        fp32_leg = run_fp32_leg(args, cfg, params, metas, frames_f32, dev) if args.precision != 'fp32' else None
        eager = run_gpu_eager_baseline(cfg, params, metas, frames_f32, dev) if not args.no_eager else None

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    pk = peaks()
    s = 2 if args.precision == 'bf16' else 4
    work = algorithmic_work(cfg, s, tc=use_tc, feat_bytes=frames_host[0][0].element_size())
    total_prof = sum(v[0] for v in prof.values()) or 1.0
    share = {k: round(v[0] / total_prof, 4) for k, v in prof.items()}
    traffic = {}
    for tname in ('r2_traffic.json', 'r1_traffic.json'):            # dram bytes from the committed ncu --set full captures
        tpath = os.path.join(ROOT, 'profiles', tname)
        if os.path.exists(tpath):
            traffic = json.load(open(tpath))
            traffic['_source'] = 'profiles/' + tname + ' (ncu --set full capture of this build; not measured in this run)'
            break
    L = cfg['num_layers']
    per_frame_bytes = {'sca_gather': work['sca_bytes_per_launch'] * L, 'tsa_gather': work['tsa_bytes_per_launch'] * L,
                       'gemm': work['gemm_bytes'], 'pack': work['pack_bytes'], 'conv3d': work['conv_bytes'],
                       'occ_head': work['head_bytes']}
    per_frame_flops = {'gemm': work['gemm_flops'], 'conv3d': work['conv_flops'], 'occ_head': work['head_flops']}
    rooflines = {}
    for k, nbytes in per_frame_bytes.items():
        ms_k, n_k = prof[k]
        if ms_k <= 0:
            continue
        per_frame_ms = ms_k / prof_frames
        ach = nbytes / (per_frame_ms * 1e-3) / 1e9
        rooflines[k] = dict(bound='hbm', achieved=round(ach, 1), peak=pk['hbm'], unit='GB/s', frac=round(ach / pk['hbm'], 4),
                            algorithmic_bytes_per_frame=int(nbytes), launches_per_frame=n_k // prof_frames,
                            ms_per_frame=round(per_frame_ms, 4), traffic=traffic.get(k))
        if k in per_frame_flops:                                    # SURVEY 8(d): dense contractions are tensor-class
            tf = per_frame_flops[k] / (per_frame_ms * 1e-3) / 1e12
            rooflines[k].update(tensor_tflops=round(tf, 1), tensor_frac=round(tf / pk['tf_sust'], 4),
                                tensor_peak=pk['tf_sust'], algorithmic_flops_per_frame=int(per_frame_flops[k]))
    # The two gather kernels are bound by the L1 data path, not by HBM: report the bytes the bilinear gathers pull
    # through L1 next to the HBM roofline.
    sm_clk = (clocks or {}).get('sm_mhz') or 1965.0
    nsm = torch.cuda.get_device_properties(dev).multi_processor_count
    for k, nbytes_l1 in (('sca_gather', n_hit * 32 * 8 * 4 * 32 * s * L),
                         ('tsa_gather', work['Nq'] * 8 * 8 * 4 * 32 * s * L)):
        if k in rooflines:
            sec = rooflines[k]['ms_per_frame'] * 1e-3
            rooflines[k]['l1_gather_bytes_per_frame'] = int(nbytes_l1)
            if k == 'sca_gather':
                rooflines[k]['visible_cam_pillar_pairs'] = n_hit
            rooflines[k]['l1_bytes_per_clk_per_sm'] = round(nbytes_l1 / sec / (sm_clk * 1e6) / nsm, 1)
    dom = max(rooflines, key=lambda k: rooflines[k]['ms_per_frame'])
    r = rooflines[dom]
    n_l = max(r['launches_per_frame'], 1)
    tr = traffic.get(dom) if isinstance(traffic.get(dom), dict) else None
    if dom in per_frame_flops:                                      # dense layers: tensor roofline per SURVEY 8(d)
        roof = dict(kernel={'gemm': 'gemm_tc_kernel (all dense layers of a frame)'}.get(dom, dom), bound='tensor',
                    achieved=r['tensor_tflops'], peak=pk['tf_sust'], unit='TFLOP/s', frac=r['tensor_frac'],
                    peak_source=pk['source'] + ' (cuBLAS bf16 sustained)',
                    algorithmic_flops_per_launch=int(per_frame_flops[dom] / n_l), hbm_frac_on_compulsory_bytes=r['frac'])
    else:
        roof = dict(kernel={'sca_gather': 'sca gather kernel'}.get(dom, dom), bound='hbm', achieved=r['achieved'],
                    peak=pk['hbm'], unit='GB/s', frac=r['frac'], peak_source=pk['source'] + ' (copy bandwidth)',
                    algorithmic_bytes_per_launch=int(r['algorithmic_bytes_per_frame'] / n_l),
                    l1_bytes_per_clk_per_sm=r.get('l1_bytes_per_clk_per_sm'))
    if dom == 'sca_gather':
        roof['algorithmic_bytes_note'] = ('operator boundary as launched: value maps 6*Nv*256*s + fp16 offsets/logits Nq*768*2 + output '
                                          'Nq*256*s (SURVEY 8(d) quotes 166 MB/layer for a kernel that never materialises offsets/logits); '
                                          'the kernel is bound by the L1/LSU data path (l1_bytes_per_clk_per_sm), not by HBM: DESIGN.md section 4')
    roof.update(traffic=tr.get('dram_bytes_per_launch') if tr else None, traffic_source=traffic.get('_source'),
                avg_launch_ms=round(r['ms_per_frame'] / n_l, 4), launches_per_frame=n_l)
    cpu = cpu_baseline(cfg) if (world == 1 and not args.no_cpu) else None
    backbone = run_backbone_leg(args, cfg, eng, dev, want) if (not args.no_backbone and world == 1) else None
    frames_total = world * K * F
    line = {
        'metric': METRIC, 'value': round(frames_total / (ms_med * 1e-3), 2), 'unit': 'samples/s',
        'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': round(ms_med / K, 4), 'ms_per_frame': round(ms_med / (K * F), 4), 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': args.precision, 'data': 'synthetic',
        'config': {'workload': f'6cam 928x1600 FPN feats -> 200x200 BEV, {cfg["num_layers"]}-layer BEVFormerEncoder '
                               f'(TSA+SCA+FFN) + Conv3d voxel decoder 200x200x16 + occ/flow heads, {args.precision}',
                   'frames_per_step_per_gpu': F, 'parallelism': f'dp{world} (frame-sharded, no data-path collective)',
                   'l2_policy': 'inputs larger than L2: 3 rotating frames (95 MB bf16 / 189 MB fp32 each) + 0.6-1.2 GB of '
                                'per-frame intermediates',
                   'tensor_cores': use_tc, 'num_layers': cfg['num_layers'], 'feature_dtype': str(feat_dtype).replace('torch.', ''),
                   'timing': f'median of {args.repeats} regions of exactly {K} steps x {F} frames after >= 1 s warm-up',
                   'region_ms': [round(x, 2) for x in reps]},
        'e2e': {'value': round(frames_total / (e2e_ms * 1e-3), 2), 'unit': 'samples/s',
                'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': round(e2e_ms / K, 4),
                'ms_per_frame': round(e2e_ms / (K * F), 4), 'region_ms': [round(x, 2) for x in e2e_reps],
                'api': 'occb200_engine_submit_host / _wait_host (2 frames in flight), pinned host buffers, features in the '
                       'storage precision (occb200_engine_set_input_dtype)',
                'host_numa_binding': numa_all,
                'sync_call_value': round(e2e_sync, 2) if e2e_sync else None,
                'fp32_feature_upload_value': round(e2e_f32, 2) if e2e_f32 else None,
                'dropin_module_call': dropin},
        'gpu_launches': launches * K * F,
        'launches_per_frame': launches,
        'clocks': clocks,
        'roofline': roof,
        'rooflines': rooflines,
        'kernel_share': share,
        'kernel_ms_per_frame': {k: round(v[0] / prof_frames, 4) for k, v in prof.items()},
        'parity': parity,
        'fp32_config': fp32_leg,
        'temporal_config': temporal,
        'gpu_eager_baseline': eager,
        'cpu_baseline': cpu,
        'images_to_voxels': backbone,
        'ray_metric': {**(rayp or {}), 'miou_vs_gt_scene': fin['miou'], 'mave_vs_gt_scene': fin['mave'], 'frames': world,
                       'collective': 'all_reduce(sum) of 187 fp64 counters' if world > 1 else 'none (1 rank)'},
    }
    print(json.dumps(line))


def run_dropin_leg(args, cfg, params, metas, frames_host, dev):
    """e2e through the drop-in MODULE call a user of the reference makes: BEVFormerOcc.forward(return_loss=False, ...)
    (detectors/bevformer_occ.py:231-270): features host->device inside, CPU LongTensor / FloatTensor results out."""
    try:
        import projects.mmdet3d_plugin  # noqa: F401
        from occnet_b200.mmcv_shim import build_detector
        det = build_detector(dict(type='BEVFormerOcc', video_test_mode=False,
                                  pts_bbox_head=dict(fixtures.head_cfg(cfg), precision=args.precision, test_logits=False)))
        det = det.to(dev).eval()
        det.pts_bbox_head.load_state_dict(params, strict=True)
        n = 2 * args.frames_per_step

        def call(i):
            feats = [f.to(dev, non_blocking=True)[None] for f in frames_host[i % len(frames_host)]]
            return det(return_loss=False, rescale=True, img_feats=feats, img_metas=[metas])
        for i in range(3):
            out = call(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(n):
            out = call(i)
        dt = time.perf_counter() - t0
        assert out['occ_results'].dtype == torch.int64 and not out['occ_results'].is_cuda
        return {'value': round(n / dt, 2), 'unit': 'samples/s', 'ms_per_frame': round(dt / n * 1e3, 3), 'frames': n,
                'api': 'BEVFormerOcc.forward(return_loss=False, img_feats=<pinned host feats .to(cuda)>, img_metas) -> CPU '
                       'LongTensor / FloatTensor (synchronous, one frame per call)'}
    except Exception as e:                                            # noqa: BLE001 -- a leg, not the headline
        return {'error': f'{type(e).__name__}: {e}'[:300]}


def run_temporal_leg(args, cfg, eng, frames_dev):
    """BASELINE configs[2] (+ TemporalSelfAttention over history): video mode -- every frame's TSA attends to the previous
    frame's BEV, rotated by can_bus[-1] (3 degrees here; index map applied inside the engine).  4 history frames are run
    first (the reference's queue_length), then a stream of frames is timed; each produces occupancy AND the next prev_bev."""
    try:
        from occnet_b200.engine import rotation_index_map
        eng.set_prev_rotation(rotation_index_map(cfg['bev_h'], cfg['bev_w'], 3.0, cfg.get('rotate_center', [100, 100])))
        want = ('bev_embed', 'flow', 'occ_cls')
        prev = None
        for i in range(4):                                           # history (obtain_history_bev recurrence)
            prev = eng.forward(frames_dev[i % len(frames_dev)], prev_bev=prev, want=('bev_embed',))['bev_embed']
        torch.cuda.synchronize()
        n = 2 * args.frames_per_step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            prev = eng.forward(frames_dev[i % len(frames_dev)], prev_bev=prev, want=want)['bev_embed']
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        lpf = eng.launches_per_frame
        eng.set_prev_rotation(None)
        return {'value': round(1e3 / ms, 2), 'unit': 'samples/s', 'ms_per_frame': round(ms, 4), 'frames': n,
                'launches_per_frame': lpf, 'history_frames': 4, 'tsa_queue': 2,
                'what': 'device-resident, prev_bev = previous frame BEV (rotated in-engine), same precision as the headline'}
    except Exception as e:                                            # noqa: BLE001
        return {'error': f'{type(e).__name__}: {e}'[:300]}


def run_fp32_leg(args, cfg, params, metas, frames_f32, dev):
    """BASELINE configs[1] ('fp32'): the reference-precision configuration of the same engine (fp32 storage), timed and
    checked against the fp32 oracle's golden frame.  Headline = the tcgen05 3xbf16-split GEMMs (fp32-grade, <= 1e-3 at six
    layers); the CUDA-core variant is reported beside it."""
    from occnet_b200.engine import OccEngine

    def one(tc):
        e32 = OccEngine(cfg, params, precision='fp32', use_tensor_cores=tc, device=str(dev))
        e32.set_cameras(metas)
        fd = [[f.to(dev) for f in fr] for fr in frames_f32]
        for i in range(3):
            e32.forward(fd[i % len(fd)], want=('flow', 'occ_cls'))
        torch.cuda.synchronize()
        n = 48 if tc else 24
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            e32.forward(fd[i % len(fd)], want=('flow', 'occ_cls'))
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        chk = e32.forward(fd[0], want=('occ', 'flow', 'occ_cls'))
        par = golden_parity(chk, 'fp32').get('fp32_oracle')
        lpf = e32.launches_per_frame
        del e32, fd
        torch.cuda.empty_cache()
        return {'value': round(1e3 / ms, 2), 'unit': 'samples/s', 'ms_per_frame': round(ms, 4), 'frames': n,
                'launches_per_frame': lpf, 'tensor_cores': tc,
                'gemm': 'tcgen05 3xbf16-split (fp32-grade), fp32 storage; conv3d / heads / LayerNorm on CUDA cores' if tc
                        else 'fp32 CUDA cores',
                'parity_vs_fp32_oracle': par}
    try:
        leg = one(True)
        try:
            leg['cuda_core_variant'] = one(False)
        except Exception as e:                                        # noqa: BLE001
            leg['cuda_core_variant'] = {'error': f'{type(e).__name__}: {e}'[:300]}
        return leg
    except Exception as e:                                            # noqa: BLE001
        return {'error': f'{type(e).__name__}: {e}'[:300]}


def run_gpu_eager_baseline(cfg, params, metas, frames_f32, dev):
    """BASELINE.md section 5 comparator ('stock CUDA build'): the restated reference modules (oracle/bevformer_occ.py) on
    `cuda` with stock library kernels -- torch grid_sample MSDA, cuBLAS Linear, cuDNN Conv3d + BatchNorm3d, fp32, eager,
    including the reference's Python rebatch loops and nonzero() syncs.  mmcv's own CUDA op cannot be built here (its
    source is not under /root/reference), so this is the stated stand-in for the 1.3x / 6.5x targets' denominator."""
    try:
        from oracle import bevformer_occ as O
        p = {k: v.to(dev) for k, v in params.items()}
        fr = [[f[None].to(dev) for f in fr_] for fr_ in frames_f32[:2]]
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        with torch.no_grad():
            for i in range(2):
                out = O.head_forward(p, cfg, fr[i % 2], metas)
                O.get_occ(out)
            torch.cuda.synchronize()
            n = 6
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for i in range(n):
                out = O.head_forward(p, cfg, fr[i % 2], metas)
                cls, flow = O.get_occ(out)
            e1.record()
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
        ms = max(e0.elapsed_time(e1), wall) / n
        del p, fr, out
        torch.cuda.empty_cache()
        return {'value': round(1e3 / ms, 2), 'unit': 'samples/s', 'ms_per_frame': round(ms, 3), 'frames': n, 'dtype': 'fp32',
                'what': 'restated reference modules on cuda: grid_sample MSDA + cuBLAS + cuDNN, eager (stand-in for the stock '
                        'mmcv CUDA build, BASELINE.md section 5)'}
    except Exception as e:                                            # noqa: BLE001
        return {'error': f'{type(e).__name__}: {e}'[:300]}


def run_backbone_leg(args, cfg, eng, dev, want):
    """SURVEY 8f rank 1: synthetic camera IMAGES (6 x 3 x 928 x 1600, fp32, already normalised / padded) -> native ResNet-50 +
    FPN (occb200_backbone_*) -> the hot path, all on the device.  bf16: the FPN writes channels-last bf16 levels that the
    engine packs without a transpose.  Reported next to (not inside) the headline, with its own tensor roofline."""
    try:
        from occnet_b200.backbone import BackboneEngine
        H, W = cfg['img_shape'][:2]
        nc = cfg['num_cams']
        cl = args.precision == 'bf16'
        be = BackboneEngine(fixtures.init_backbone_params(seed=5), nc, (H, W), precision=args.precision,
                            use_tensor_cores=bool(args.tc) and cl, device=str(dev))
        imgs = [torch.randn(nc, 3, H, W, device=dev, generator=torch.Generator(device=dev).manual_seed(7 + i)) for i in range(3)]
        assert be.level_shapes == [tuple(s) for s in cfg['level_shapes']], be.level_shapes
        prev_dtype, prev_cl = eng.feat_dtype, eng.feat_channels_last
        eng.set_input_dtype(torch.bfloat16 if cl else torch.float32, channels_last=cl)
        n = 2 * args.frames_per_step
        for i in range(4):
            eng.forward(be.forward(imgs[i % 3], channels_last_bf16=cl), want=want)
        torch.cuda.synchronize()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        for i in range(n):
            be.forward(imgs[i % 3], channels_last_bf16=cl)
        e1.record()
        for i in range(n):
            eng.forward(be.forward(imgs[i % 3], channels_last_bf16=cl), want=want)
        e2.record()
        torch.cuda.synchronize()
        eng.set_input_dtype(prev_dtype, channels_last=prev_cl)
        bb_ms, chain_ms = e0.elapsed_time(e1) / n, e1.elapsed_time(e2) / n
        gflop = 1460.0                                                # ResNet-50 (C3-C5) + FPN at 6 x 928 x 1600, 2*MACs
        pk = peaks()
        return {'value': round(1e3 / chain_ms, 2), 'unit': 'samples/s (6 x 3 x 928 x 1600 images -> 200x200x16 voxels)',
                'ms_per_frame': round(chain_ms, 4), 'backbone_ms_per_frame': round(bb_ms, 4), 'frames': n,
                'backbone_gflop_per_frame': gflop, 'backbone_tflops': round(gflop / bb_ms, 1),
                'backbone_tensor_frac': round(gflop / bb_ms / pk['tf_sust'], 4),
                'handover': 'bf16 channels-last levels written by the FPN convolutions, packed by the engine without a '
                            'transpose' if cl else 'fp32 NCHW levels',
                'implicit_gemm': os.environ.get('OCC_BACKBONE_IMPLICIT', '1') != '0'}
    except Exception as e:                                            # noqa: BLE001
        return {'error': f'{type(e).__name__}: {e}'[:300]}


CPU_WORKER = r"""
import json, os, sys, time
sys.path.insert(0, os.environ['OCC_ROOT'])
import torch
cores = [int(c) for c in os.environ['OCC_CORES'].split(',')]
try:
    os.sched_setaffinity(0, cores)
except Exception:
    pass
torch.set_num_threads(len(cores))
from occnet_b200 import fixtures
from oracle import bevformer_occ as O
layers, frames, seed = int(os.environ['OCC_LAYERS']), int(os.environ['OCC_FRAMES']), int(os.environ['OCC_SEED'])
cfg = fixtures.make_cfg('full', num_layers=layers)
params = fixtures.init_params(cfg, seed=2, free_bias=fixtures.FREE_BIAS)
metas = fixtures.make_img_metas(cfg)
fr = [fixtures.make_feats(cfg, bs=1, seed=seed + i) for i in range(2)]
with torch.no_grad():
    t0 = time.perf_counter()
    O.get_occ(O.head_forward(params, cfg, fr[0], metas))                  # warm-up frame (also reported)
    t_warm = time.perf_counter() - t0
    print(json.dumps({'ready': True}), flush=True)
    sys.stdin.readline()                                                   # start signal: all workers timed together
    t0 = time.perf_counter()
    for i in range(frames):
        O.get_occ(O.head_forward(params, cfg, fr[(i + 1) % 2], metas))
    dt = time.perf_counter() - t0
print(json.dumps({'frames': frames, 'seconds': dt, 'warm_seconds': t_warm, 'threads': torch.get_num_threads()}), flush=True)
"""


def cpu_reference_run(layers, frames_per_worker=1, threads_per_worker=16, max_workers=None):
    """The reference's CPU path (oracle restatement: grid_sample MSDA inside the restated modules, fp32) on ALL host
    cores: torch's intra-op pool stops scaling at 16-32 threads on this workload, so the cores are split over
    independent worker processes (frames are independent -- the same data parallelism the GPU arm uses), each pinned
    to its own core set; aggregate throughput = total frames / wall time of the slowest worker."""
    try:
        avail = sorted(os.sched_getaffinity(0))
        all_cores = list(range(os.cpu_count() or len(avail)))
        try:
            os.sched_setaffinity(0, all_cores)                     # undo the e2e leg's NUMA binding
            avail = sorted(os.sched_getaffinity(0))
        except Exception:                                          # noqa: BLE001
            pass
    except AttributeError:
        avail = list(range(os.cpu_count() or 1))
    tpw = min(threads_per_worker, len(avail))
    nw = max(1, len(avail) // tpw)
    if max_workers:
        nw = min(nw, max_workers)
    procs = []
    for w in range(nw):
        cores = avail[w * tpw:(w + 1) * tpw]
        env = dict(os.environ, OCC_ROOT=ROOT, OCC_CORES=','.join(map(str, cores)), OCC_LAYERS=str(layers),
                   OCC_FRAMES=str(frames_per_worker), OCC_SEED=str(100 + 2 * w), OMP_NUM_THREADS=str(len(cores)),
                   CUDA_VISIBLE_DEVICES='')
        procs.append(subprocess.Popen([sys.executable, '-c', CPU_WORKER], env=env, stdin=subprocess.PIPE,
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True))
    for p in procs:                                                # all warmed up ...
        line = p.stdout.readline()
        assert 'ready' in line, line
    t0 = time.perf_counter()
    for p in procs:                                                # ... then released together
        p.stdin.write('go\n'); p.stdin.flush()
    res = [json.loads(p.stdout.readline()) for p in procs]
    wall = time.perf_counter() - t0
    for p in procs:
        p.wait(timeout=60)
    frames = sum(r['frames'] for r in res)
    return dict(value=round(frames / wall, 5), unit='samples/s', cores=nw * tpw, kind='port',
                sample=f'{frames} full frames ({layers} encoder layers + decoder + heads + argmax), {nw} worker processes x '
                       f'{tpw} threads pinned to disjoint cores, timed together after one warm-up frame each',
                seconds_per_frame_per_worker=round(float(np.mean([r['seconds'] / r['frames'] for r in res])), 3),
                workers=nw, threads_per_worker=tpw, wall_seconds=round(wall, 2))


def cpu_baseline(cfg):
    return cpu_reference_run(cfg['num_layers'], frames_per_worker=1)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cfg = workload_cfg(args)
    budget = float(os.environ.get('OCC_REF_BUDGET_S', '150'))
    # size the run: one frame takes ~15-25 s per 16-thread worker; keep the whole arm within a few minutes
    fpw = max(1, min(args.steps, int(budget // 25)))
    r = cpu_reference_run(cfg['num_layers'], frames_per_worker=fpw)
    steps = fpw * r['workers']
    line = {'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': 'samples/s', 'n_gpus': args.gpus,
            'steps': steps, 'warmup': 1, 'ms_per_step': round(1e3 / r['value'], 2), 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
            'config': {'workload': f'6cam 928x1600 FPN feats -> 200x200 BEV, {cfg["num_layers"]}-layer BEVFormerEncoder '
                                   f'+ Conv3d voxel decoder 200x200x16 + occ/flow heads, reference CPU path '
                                   f'(multi_scale_deformable_attn_pytorch / grid_sample), fp32',
                       'num_layers': cfg['num_layers'],
                       'note': 'CPU arm: ONE host (all its cores) whatever --gpus says; per-N ratios against it compare N GPUs '
                               'with the same single host'},
            'host_processes': r['workers'], 'gpus_used': 0,
            'cpu_baseline': dict(r, value=r['value']),
            'e2e': {'value': r['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--layers', type=int, default=6)
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--tc', type=int, default=1, help='tcgen05 tensor-core kernels (bf16 only)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-eager', action='store_true', help='skip the gpu_eager_baseline leg (stock torch kernels)')
    ap.add_argument('--no-dropin', action='store_true', help='skip the drop-in module-call e2e leg')
    ap.add_argument('--frames-per-step', type=int, default=32, help='one step = this many frames through the engine')
    ap.add_argument('--repeats', type=int, default=3, help='timed regions (each exactly --steps steps); median reported')
    ap.add_argument('--no-backbone', action='store_true', help='skip the images -> ResNet-50+FPN -> hot path leg')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed (rank 0) as DIR/<name>.npy, float32 (see dump_outputs)')
    args = ap.parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
