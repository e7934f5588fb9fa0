#!/usr/bin/env python
"""bench.py -- clips/s of the GAST-Net lifting forward (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--clips B] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): 27-frame 17-joint inference, 4096 clips per GPU
(weak scaling, clips are independent -> no collective on the data path), fp32,
SpatioTemporalModel([3,3,3], channels=128) in eval mode, synthetic keypoints, seeded weights.
One step = one forward over the GPU's whole 4096-clip batch.

Prints ONE JSON line (rank 0).  `value` times the hot path with inputs resident in HBM;
`e2e` times the same call through the drop-in module with pinned HOST buffers (H2D of the
clips and D2H of the 3D poses inside the timed region).  `--impl reference` times the CPU
port of the reference algorithm (oracle/) on the host cores instead.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, 'gast-net-3dposeestimation_b200')
for _p in (PKG, REPO):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = '27-frame 17-joint clips/sec'
UNIT = 'clips/s'
J, FW, CH, T = 17, [3, 3, 3], 128, 27
FLOP_PER_CLIP = 0.402e9          # algorithmic (needed-only) forward FLOPs, BASELINE.md §2
IO_BYTES_PER_CLIP = 3876         # compulsory (T*J*2 + J*3)*4 bytes

# The other BASELINE.json configurations, reported in `other_configs` after the headline (configs[1]) region.
# flop = algorithmic (needed-only) FLOPs per clip, SURVEY.md §8(d); `global_clips` is split over the ranks
# (strong scaling, as BASELINE.json words them: "batch 2048 clip-sharded across 8", "batch 8192, 2/4/8 sweep").
OTHER = {
    'cfg4_81f_17j_64ch': dict(J=17, fw=[3, 3, 3, 3], ch=64, T=81, flop=0.490e9, global_clips=2048,
                              what='BASELINE configs[3]: 81-frame (-arc 3,3,3,3) 17-joint inference, 64 channels'),
    'cfg5_27f_19j_128ch': dict(J=19, fw=[3, 3, 3], ch=128, T=27, flop=0.451e9, global_clips=8192,
                               what='BASELINE configs[4]: 27-frame 19-joint body+toe inference, 128 channels'),
}
TRAIN_FLOP_PER_CLIP = 1.21e9     # fwd + bwd, SURVEY.md §8(d)


def measured_peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, 'measured'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(',')])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = set()
        for r in self.rows:
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        # the busiest half of the samples = "under load"
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {'sm_mhz': statistics.median(load) if load else None,
                'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def build_model(device, J_=J, fw=FW, ch=CH, cls='full', dropout=0.05):
    import torch
    from gast_b200 import synth
    from model.gast_net import SpatioTemporalModel, SpatioTemporalModelOptimized1f
    from common.skeleton import Skeleton
    from common.graph_utils import adj_mx_from_skeleton
    adj = adj_mx_from_skeleton(Skeleton(synth.skeleton_parents(J_), [], []))
    kls = SpatioTemporalModel if cls == 'full' else SpatioTemporalModelOptimized1f
    m = kls(adj, J_, 2, J_, fw, causal=False, dropout=dropout, channels=ch)
    synth.randomize_module(m, 1)
    return m.to(device).eval()


def kernel_share(prof):
    """share of the fused GEMM family in the device time of one step, from the per-launch event pass.  The pass
    brackets every launch with its own event pair, which adds a few microseconds per launch and removes the
    overlap between a kernel's tail and the next one's head, so its SUM is not the step time; the SHARES are what
    it measures (the ncu launch list under profiles/ is the cross-check)."""
    tot = sum(prof['per_kernel_ms'].values())
    return prof['gemm_ms_per_step'] / tot if tot > 0 else 0.0


def roofline_of(prof, ms_per_step, flop_per_clip, clips, peaks, peak_src, traffic):
    share = kernel_share(prof)
    k_ms = share * ms_per_step                  # never exceeds the step it is part of
    assert k_ms <= ms_per_step * (1 + 1e-9)
    achieved = flop_per_clip * clips / (k_ms / 1000.0) / 1e12
    peak_tf = peaks.get('bf16_tflops_sustained', peaks['bf16_tflops'])
    return {'bound': 'tensor', 'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved / peak_tf,
            'frac_whole_step': flop_per_clip * clips / (ms_per_step / 1000.0) / 1e12 / peak_tf,
            'traffic': traffic,
            'kernel': 'fused GEMM family (%d launches/step)' % prof['gemm_launches'],
            'kernel_ms_per_step': k_ms, 'kernel_share_of_step': share,
            'peak_source': 'bf16_tflops_sustained of %s MEASURED_PEAKS (cuBLAS bf16, long loop)' % peak_src,
            'per_kernel_ms_event_pass': {k: round(v, 4) for k, v in prof['per_kernel_ms'].items()}}


def traffic_record():
    """DRAM bytes of the GEMM-family launches of one step, from an `ncu --set full` capture (tools/ncu_summary.py
    -> profiles/traffic.json).  The capture names the kernel-source hash it was taken from; a capture of another
    build is reported as stale instead of being passed off as a measurement of this binary."""
    tp = os.path.join(REPO, 'profiles', 'traffic.json')
    if not os.path.exists(tp):
        return None, 'no capture'
    with open(tp) as f:
        d = json.load(f)
    cur = source_hash()
    if d.get('source_hash') and d['source_hash'] != cur:
        return d.get('dram_bytes_per_step'), 'STALE: captured from kernel sources %s, this build is %s' % (d['source_hash'], cur)
    return d.get('dram_bytes_per_step'), d.get('source', '')


def source_hash():
    import hashlib
    hsh = hashlib.sha1()
    cs = os.path.join(PKG, 'csrc')
    for fn in sorted(os.listdir(cs)):
        if fn.endswith(('.cu', '.cuh')):
            with open(os.path.join(cs, fn), 'rb') as f:
                hsh.update(f.read())
    return hsh.hexdigest()[:12]


def time_forward(model, xs, K, W, barrier, stream):
    import torch
    with torch.no_grad():
        for i in range(W):
            model(xs[i % len(xs)])
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(K):
            model(xs[i % len(xs)])
        e1.record(stream)
        barrier()
    return e0.elapsed_time(e1)


def bench_other(name, cfg, device, rank, world, K, W, barrier, stream, reduce_max, peaks, peak_src):
    """clips/s + roofline of one of the other BASELINE configurations on this rank's shard"""
    import torch
    from gast_b200 import synth, engine
    m = build_model(device, cfg['J'], cfg['fw'], cfg['ch'])
    per = cfg['global_clips'] // world
    nbuf = 4
    xs = [torch.from_numpy(synth.synth_input(per, cfg['T'], cfg['J'], 2, seed=77 + rank * 10 + i)).to(device)
          for i in range(nbuf)]
    ms = reduce_max(time_forward(m, xs, K, W, barrier, stream))
    with torch.no_grad():
        prof = engine.profile_forward(m, xs[0], reps=3)
    launches = int(m._gast_last_launches)
    del m, xs
    torch.cuda.empty_cache()
    rl = roofline_of(prof, ms / K, cfg['flop'], per, peaks, peak_src, None)
    rl.pop('per_kernel_ms_event_pass')
    return {'workload': cfg['what'], 'clips_per_gpu': per, 'global_clips': per * world, 'scaling': 'strong',
            'value': per * world * K / (ms / 1000.0), 'unit': UNIT, 'ms_per_step': ms / K, 'gpu_launches_per_step': launches,
            'gemm_core': prof['gemm_core'], 'roofline': rl}


def bench_train(device, rank, world, K, W, barrier, stream, reduce_max, peaks):
    """BASELINE configs[2]: `trainval.py -arc 3,3,3 -b 128` -- main.train()'s step (main.py:219-239) on
    SpatioTemporalModelOptimized1f, b = 128 clips PER RANK (BatchNorm statistics per rank, like the replicas of
    the reference's nn.DataParallel), dropout 0.05 (the reference default), one all-reduce of the flat gradient
    buffer over NCCL when world > 1, Adam(amsgrad)."""
    import torch
    import torch.distributed as dist
    from gast_b200 import synth
    from gast_b200.trainer import GraphedTrainer
    from gast_b200.pipeline import FusedAdam
    b = 128
    m = build_model(device, J, FW, CH, cls='1f', dropout=0.05)
    # forward + loss + backward replayed from one CUDA graph (the eager step is host-launch-bound), all-reduce and
    # the one-launch Adam(amsgrad) after it
    tr = GraphedTrainer(m, lambda ps: FusedAdam(ps, lr=1e-3, amsgrad=True), (b, T, J, 2), (b, 1, J, 3))
    xs = [torch.from_numpy(synth.synth_input(b, T, J, 2, seed=300 + rank * 10 + i)).to(device) for i in range(4)]
    ys = [torch.from_numpy(synth.synth_target(b, J, seed=400 + rank * 10 + i)).to(device) for i in range(4)]
    for i in range(W):
        loss = tr.step(xs[i % 4], ys[i % 4])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(K):
        loss = tr.step(xs[i % 4], ys[i % 4])
    e1.record(stream)
    barrier()
    ms = reduce_max(e0.elapsed_time(e1))
    ar_ms = None
    if world > 1:
        for _ in range(3):
            dist.all_reduce(tr.flat.flat)
        barrier()
        e0.record(stream)
        for _ in range(20):
            dist.all_reduce(tr.flat.flat)
        e1.record(stream)
        barrier()
        ar_ms = reduce_max(e0.elapsed_time(e1)) / 20
    fl = float(loss)
    nparam = int(tr.flat.flat.numel())
    peak_tf = peaks.get('bf16_tflops_sustained', peaks['bf16_tflops'])
    out = {'workload': 'BASELINE configs[2]: Optimized1f [3,3,3]/128ch train step (fwd + mpjpe + bwd + grad all-reduce '
                       '+ Adam amsgrad), b=128 per rank, dropout 0.05; fwd+loss+bwd replayed from one CUDA graph',
           'clips_per_gpu': b, 'global_clips': b * world, 'scaling': 'weak', 'ms_per_step': ms / K,
           'value': b * world * K / (ms / 1000.0), 'unit': 'clips/s (training)',
           'allreduce_ms': ar_ms, 'allreduce_bytes': 4 * nparam, 'last_loss': fl,
           'frac_whole_step': TRAIN_FLOP_PER_CLIP * b / (ms / K / 1000.0) / 1e12 / peak_tf,
           'gpu_launches_per_step_gemm': int(m._gast_last_launches)}
    del tr, m
    torch.cuda.empty_cache()
    return out


_CPU_STATE = {}


def cpu_port_clips_per_s(sample_clips, reps, threads=None):
    """Times the CPU port of the reference (oracle/gast_torch_ref.py: the same torch CPU kernels in
    the same order as the reference modules -- bit-identical outputs, same cost) on all host
    cores.  Needed-only (Optimized1f) schedule = the reference's fastest CPU form."""
    import torch
    from oracle import gast_oracle as O
    from oracle import gast_torch_ref as TR
    from gast_b200 import synth
    if 'p' not in _CPU_STATE:
        from model.gast_net import SpatioTemporalModelOptimized1f
        from common.skeleton import Skeleton
        from common.graph_utils import adj_mx_from_skeleton
        adj_t = adj_mx_from_skeleton(Skeleton(synth.skeleton_parents(J), [], []))
        m = SpatioTemporalModelOptimized1f(adj_t, J, 2, J, FW, channels=CH)
        synth.randomize_module(m, 1)
        _CPU_STATE['p'] = {k: v.clone() for k, v in m.state_dict().items()}
        _CPU_STATE['masks'] = tuple(torch.from_numpy(a) for a in
                                    O.local_masks(O.adj_from_parents(synth.skeleton_parents(J))))
        # give the CPU baseline its best thread count: all host threads are not always the
        # fastest for these small ATen kernels
        xw = torch.from_numpy(synth.synth_input(16, T, J, 2, seed=1))
        best = (None, 1e30)
        cands = [threads] if threads else sorted({os.cpu_count(), 32, 16, 8} & set(range(1, os.cpu_count() + 1)), reverse=True)
        with torch.no_grad():
            for nt in cands:
                torch.set_num_threads(nt)
                TR.forward(xw, _CPU_STATE['p'], _CPU_STATE['masks'], FW, strided=True)      # warm
                t0 = time.perf_counter()
                TR.forward(xw, _CPU_STATE['p'], _CPU_STATE['masks'], FW, strided=True)
                dt = time.perf_counter() - t0
                if dt < best[1]:
                    best = (nt, dt)
        _CPU_STATE['threads'] = best[0]
    torch.set_num_threads(_CPU_STATE['threads'])
    x = torch.from_numpy(synth.synth_input(sample_clips, T, J, 2, seed=1234))
    ts = []
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            TR.forward(x, _CPU_STATE['p'], _CPU_STATE['masks'], FW, strided=True)
            ts.append(time.perf_counter() - t0)
    return sample_clips / statistics.median(ts), torch.get_num_threads(), ts


def run_reference(args, rank, world):
    """`--impl reference`: the reference algorithm's CPU port on the host cores (rank 0 only)."""
    if rank != 0:
        return
    sample = args.cpu_clips
    vals = []
    total_steps = args.warmup + args.steps
    per_step = []
    for s in range(total_steps):
        v, cores, ts = cpu_port_clips_per_s(sample, 1)
        if s >= args.warmup:
            vals.append(v)
            per_step.append(ts[0])
    value = sample * len(per_step) / sum(per_step)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * sum(per_step) / len(per_step),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': '27f/17j/128ch SpatioTemporalModel forward, eval, fp32 (BASELINE configs[1])',
                   'clips_per_step': sample, 'frames': T, 'joints': J, 'channels': CH,
                   'impl': 'CPU port of the reference on the host cores',
                   'note': 'same model/metric as the GPU arm on a bounded sample: %d clips per step instead of 4096 '
                           '(clips are independent; CPU throughput is flat in the batch size beyond ~64 clips)' % sample},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '%d clips per step, needed-only (Optimized1f) schedule, torch-CPU port of the '
                                   'reference (oracle/gast_torch_ref.py, bit-identical to it)' % sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--clips', type=int, default=4096, help='clips per GPU per step')
    ap.add_argument('--cpu-clips', type=int, default=256, help='clips per CPU-baseline sample / reference-arm step')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-other-configs', action='store_true', help='headline (configs[1]) only')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the 3D poses of the last timed step as DIR/poses_3d.npy '
                         '(float32, (clips, 1, 17, 3); the seeded inputs are the same in every run)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the product path has no CPU fallback '
                         '(use --impl reference for the CPU port)')
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)
    from gast_b200 import synth

    model = build_model(device)
    B = args.clips
    K, W = args.steps, max(args.warmup, 3)
    # rotating input buffers: 10 x 15 MB > 126 MB L2, so no step re-reads a cached input;
    # the per-step intermediates (~2.6 GB) already stream far more than L2 holds.
    NBUF = 10
    xs_host = [torch.from_numpy(synth.synth_input(B, T, J, 2, seed=1234 + rank * 100 + i)).pin_memory()
               for i in range(NBUF)]
    xs_dev = [x.to(device) for x in xs_host]
    y_host = torch.empty((B, 1, J, 3), dtype=torch.float32).pin_memory()
    stream = torch.cuda.current_stream(device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---------------- device-resident throughput (`value`) -----------------------------
    with torch.no_grad():
        for i in range(W):
            model(xs_dev[i % NBUF])
        launches_per_step = int(model._gast_last_launches)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            time.sleep(0.3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(K):
            y = model(xs_dev[i % NBUF])
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs:                       # what the timed path returned to its caller in its last step
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, 'poses_3d%s.npy' % ('_rank%d' % rank if rank else '')),
                    y.cpu().numpy().astype(np.float32))

        # ---------------- end to end through the public API with host buffers ----------
        for i in range(3):
            y_host.copy_(model(xs_host[i % NBUF].to(device, non_blocking=True)), non_blocking=True)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for i in range(K):
            xd = xs_host[i % NBUF].to(device, non_blocking=True)     # H2D of this step's clips
            y_host.copy_(model(xd), non_blocking=True)                 # D2H of this step's poses
        f1.record(stream)
        barrier()
        ms_e2e_serial = f0.elapsed_time(f1)
        # the serving API for host-resident clips: upload of step i+1 and download of step i-1 overlap the
        # forward of step i (gast_b200/stream.py); every step's H2D and D2H is inside the timed region
        from gast_b200.stream import PipelinedLifter
        lifter = PipelinedLifter(model, depth=2)
        y_hosts = [torch.empty((B, 1, J, 3), dtype=torch.float32).pin_memory() for _ in range(2)]
        lifter.run([xs_host[i % NBUF] for i in range(3)], [y_hosts[i % 2] for i in range(3)])
        barrier()
        f0.record(stream)
        lifter.run([xs_host[i % NBUF] for i in range(K)], [y_hosts[i % 2] for i in range(K)])
        f1.record(stream)
        barrier()
        ms_e2e = f0.elapsed_time(f1)

        # ---------------- per-kernel timing for the roofline ----------------------------
        from gast_b200 import engine
        prof = engine.profile_forward(model, xs_dev[0], reps=max(3, min(K, 10)))

    def reduce_max(v):
        tt = torch.tensor([v], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt[0])

    ms, ms_e2e, ms_e2e_serial = reduce_max(ms), reduce_max(ms_e2e), reduce_max(ms_e2e_serial)
    peaks, peak_src = measured_peaks()

    # ---------------- the other BASELINE configurations (after the headline region) -------------
    other = {}
    if not args.no_other_configs:
        del xs_dev
        model.__dict__.pop('_gast_handles', None)
        torch.cuda.empty_cache()
        Ko, Wo = K, W
        for name, cfg in OTHER.items():
            try:
                other[name] = bench_other(name, cfg, device, rank, world, Ko, Wo, barrier, stream, reduce_max, peaks, peak_src)
            except Exception as e:                                   # a failing side config must not lose the headline
                other[name] = {'error': repr(e)[:300]}
        try:
            other['cfg3_train_27f_17j_128ch_b128'] = bench_train(device, rank, world, Ko, Wo, barrier, stream, reduce_max, peaks)
        except Exception as e:
            other['cfg3_train_27f_17j_128ch_b128'] = {'error': repr(e)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_clips = B * world * K
    value = total_clips / (ms / 1000.0)
    e2e_value = total_clips / (ms_e2e / 1000.0)
    # dominant kernel: the fused GEMM family (all launches of it in one step; >99% of the algorithmic FLOPs
    # are the channel contractions)
    traffic, traffic_src = traffic_record()
    roof = roofline_of(prof, ms / K, FLOP_PER_CLIP, B, peaks, peak_src, traffic)
    roof['traffic_source'] = traffic_src
    roof['hbm_frac_compulsory'] = IO_BYTES_PER_CLIP * value / world / 1e9 / peaks['hbm_gbs']
    from gast_b200 import _lib
    ver = _lib.load().gast_version().decode()
    # bf16-equivalent tensor passes per MAC: TF32 runs at half the bf16 rate, so 3xTF32 costs 6; one TF32 product
    # + two bf16 correction products cost 2 + 2 = 4; three fp16 products (hi.hi + lo.hi + hi.lo) cost 3 (the K < 256
    # layers of block 1, ~10 % of the FLOPs, stay on the 4-pass form: the bound is quoted for the 3-pass one)
    div = 3 if 'fp16 hi+lo' in ver else 4 if 'bf16-corr' in ver else 6
    roof['arithmetic'] = ver
    roof['frac_of_fp32_parity_bound'] = roof['frac'] * div
    roof['note'] = ('fp32-grade arithmetic (parity bar 1e-4 abs): every MAC costs %d bf16-equivalent tensor passes, so the '
                    'attainable fraction of the bf16 peak is 1/%d' % (div, div))
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': '27f/17j/128ch SpatioTemporalModel forward, eval, fp32 (BASELINE configs[1])',
                   'clips_per_gpu': B, 'global_clips': B * world, 'frames': T, 'joints': J, 'channels': CH,
                   'parallelism': 'clip-sharded x%d, no collective' % world,
                   'l2': 'rotating %d input buffers (%.0f MB > 126 MB L2); intermediates %.1f GB/step'
                         % (NBUF, NBUF * B * T * J * 2 * 4 / 1e6, prof['workspace_bytes'] / 1e9),
                   'gemm_core': prof['gemm_core']},
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': B * T * J * 2 * 4,
                'd2h_bytes_per_step': B * J * 3 * 4, 'ms_per_step': ms_e2e / K,
                'api': 'gast_b200.stream.PipelinedLifter (copy stream overlaps H2D/D2H with the forward)',
                'serial_value': total_clips / (ms_e2e_serial / 1000.0)},
        'gpu_launches': launches_per_step * K,
        'clocks': clocks,
        'roofline': roof,
        'source_hash': source_hash(),
    }
    if other:
        line['other_configs'] = other
    if not args.no_cpu_baseline:
        v, cores, ts = cpu_port_clips_per_s(args.cpu_clips, 5)
        line['cpu_baseline'] = {'value': v, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                                'sample': '%d clips x 5 reps (median), needed-only schedule, torch-CPU port of the '
                                          'reference (oracle/gast_torch_ref.py)' % args.cpu_clips}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
