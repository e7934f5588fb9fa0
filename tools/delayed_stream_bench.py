"""GPU: frames/s of delayed streaming (DelayedStream, gast_stream_push_delayed) of the non-causal 27-frame/128ch and
81-frame/64ch models, with and without test-time augmentation, for 1, 64 and 1024 concurrent streams; against
recomputing the receptive field for every frame (WindowStream on n streams, or on 2n streams + tta_merge with
augmentation: the reference's way, gen_skes.py:43-69 with its callers' augment=True), and against CausalStream of the
causal model of the same shape on 2n streams (the same rings and GEMMs at twice the rows).

Device time per pushed frame with CUDA events after a warm-up; the card's name and power limit are recorded in the
same run.  Usage: python tools/delayed_stream_bench.py [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'gast-net-3dposeestimation_b200'))
sys.path.insert(0, REPO)
from gast_b200 import synth, tta  # noqa: E402
from gast_b200.realtime import CausalStream, DelayedStream, WindowStream  # noqa: E402
from common.skeleton import Skeleton  # noqa: E402
from common.graph_utils import adj_mx_from_skeleton  # noqa: E402
from model.gast_net import SpatioTemporalModelOptimized1f  # noqa: E402

LEFT, RIGHT = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]


def card():
    rec = {'device': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        rec['power_limit'], rec['max_sm_clock'] = [v.strip() for v in q.split(',')]
    except Exception as e:                                   # the timing stands; the record says what is missing
        rec['power_limit'] = 'unavailable (%s)' % type(e).__name__
    return rec


def timed(push, frames, warm, reps):
    for t in range(warm):
        push(frames[t % len(frames)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(reps):
        push(frames[t % len(frames)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='also write the records to this JSON file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('delayed_stream_bench: no CUDA device (this measures the GPU path only)')
    J = 17
    adj = adj_mx_from_skeleton(Skeleton(synth.skeleton_parents(J), [], []))
    perm = list(range(J))
    for a, b in zip(LEFT, RIGHT):
        perm[a], perm[b] = b, a
    out = {'card': card(), 'records': []}
    print(json.dumps(out['card']), flush=True)
    for fw, ch in (([3, 3, 3], 128), ([3, 3, 3, 3], 64)):
        m = SpatioTemporalModelOptimized1f(adj, J, 2, J, fw, causal=False, channels=ch, dropout=0.25)
        synth.randomize_module(m, 2)
        m = m.cuda().eval()
        mc = SpatioTemporalModelOptimized1f(adj, J, 2, J, fw, causal=True, channels=ch, dropout=0.25)
        mc.load_state_dict(m.state_dict())
        mc = mc.cuda().eval()
        for n in (1, 64, 1024):
            frames = [torch.from_numpy(synth.synth_input(n, 1, J, 2, seed=10 + i)[:, 0]).cuda() for i in range(8)]
            big = n >= 1024
            for augment in (False, True):
                kw = dict(kps_left=LEFT, kps_right=RIGHT, joints_left=LEFT, joints_right=RIGHT) if augment else {}
                ds = DelayedStream(m, n, augment=augment, **kw)
                ms_delayed = timed(lambda f: ds.push(f), frames, 100, 50 if big else 200)
                rows = 2 * n if augment else n
                ws = WindowStream(m, rows)
                if augment:
                    def win(f):
                        t = f[:, perm].clone()
                        t[..., 0] *= -1
                        return tta.tta_merge(ws.push(torch.cat([f, t])).view(2, n, J, 3), LEFT, RIGHT)
                else:
                    win = ws.push
                ms_win = timed(win, frames, 10 if big else 20, 10 if big else 50)
                cs = CausalStream(mc, rows)
                rows_frames = [torch.cat([f, f]) for f in frames] if augment else frames
                ms_causal = timed(cs.push, rows_frames, 100, 50 if big else 200)
                rec = {'model': '%d-frame/%dch non-causal' % (m.receptive_field(), ch), 'streams': n,
                       'augment': augment, 'delay': ds.delay,
                       'delayed_ms_per_push': ms_delayed, 'delayed_frames_per_s': n / ms_delayed * 1e3,
                       'delayed_launches_per_push': ds.last_launches,
                       'window_ms_per_push': ms_win, 'window_frames_per_s': n / ms_win * 1e3,
                       'speedup_vs_window': ms_win / ms_delayed,
                       'causal_stream_rows': rows, 'causal_stream_ms_per_push': ms_causal,
                       'delayed_over_causal_stream': ms_delayed / ms_causal}
                print(json.dumps(rec), flush=True)
                out['records'].append(rec)
                del ds, ws, cs
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
