"""CPU: the ring schedule of the delayed streaming path (csrc/stream.cuh, gast_stream_push_delayed), restated in
numpy (oracle/stream_oracle.py), equals the whole-sequence forward the reference runs on the edge-padded sequence
(UnchunkedGenerator(pad, causal_shift) with and without augment=True, main.py:314-318) frame by frame; and the host
bookkeeping of gast_b200.realtime.DelayedStream (DelayIndex) labels every returned pose with its frame."""
import numpy as np
import pytest

from gast_b200 import synth
from gast_b200.realtime import DelayIndex
from oracle import gast_oracle as O
from oracle.stream_oracle import RingStream, stream_geometry

J = 17
LEFT, RIGHT = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]


def schedule(delay):
    """3 streams with staggered starts, ends and resets.  Returns the per-push `ended` lists, the resets to apply
    before each push, and per stream the list of its sequences' lengths.  Stream 0: one sequence that ends early
    and is held to the end; stream 1: a sequence, its full tail of `delay` repeats, then a second one; stream 2: reset
    in the middle of its first sequence (that sequence's last poses are never returned), then a shorter one."""
    lens = {0: [23], 1: [17, 21], 2: [30, 9]}
    cut2 = 19                                             # stream 2 restarts after 19 real frames of its first sequence
    t1 = 17 + delay + 2                                   # stream 1 restarts here
    total = max(t1 + 21, cut2 + 9, 23) + 3
    plan = []
    for t in range(total):
        resets, ended = [], []
        if t == t1:
            resets.append(1)
        if t == cut2:
            resets.append(2)
        if t >= 23:
            ended.append(0)
        if 17 <= t < t1 or t >= t1 + 21:
            ended.append(1)
        if t >= cut2 + 9:
            ended.append(2)
        plan.append((resets, ended))
    return plan, lens, cut2


@pytest.mark.parametrize('fw', [[3, 3, 3], [3, 3, 3, 3]], ids=['27f', '81f'])
@pytest.mark.parametrize('causal', [False, True], ids=['noncausal', 'causal'])
@pytest.mark.parametrize('twin', [False, True], ids=['plain', 'twin'])
def test_ring_oracle_equals_whole_sequence_forward(fw, causal, twin):
    from model.gast_net import SpatioTemporalModel
    from common.skeleton import Skeleton
    from common.graph_utils import adj_mx_from_skeleton
    parents = synth.skeleton_parents(J)
    m = SpatioTemporalModel(adj_mx_from_skeleton(Skeleton(parents, [], [])), J, 2, J, fw, causal=causal, channels=16)
    synth.randomize_module(m, 21)
    p = {k: v.numpy() for k, v in m.state_dict().items()}
    adj = O.adj_from_parents(parents)
    rf = int(np.prod(fw))
    _, delay = stream_geometry(fw, causal)
    assert delay == (0 if causal else (rf - 1) // 2)
    kw = dict(kps_left=LEFT, kps_right=RIGHT, joints_left=LEFT, joints_right=RIGHT) if twin else {}
    rs = RingStream(p, adj, fw, causal, 3, J, twin=twin, **kw)
    ix = DelayIndex(3, delay)
    plan, lens, cut2 = schedule(delay)
    seqs = {(s, q): synth.synth_input(1, L, J, 2, seed=300 + 10 * s + q)[0] for s in lens for q, L in enumerate(lens[s])}
    seq_no = [0, 0, 0]
    real = [0, 0, 0]
    got = {}
    rng = np.random.RandomState(5)
    for t, (resets, ended) in enumerate(plan + [([], [0, 1, 2])] * delay):
        for s in resets:
            ix.reset([s])
            seq_no[s] += 1
            real[s] = 0
        fresh, hold, idx = ix.step(ended)
        x = rng.standard_normal((3, J, 2)).astype(np.float32)         # rows of held streams are ignored
        for s in range(3):
            if not hold[s]:
                x[s] = seqs[(s, seq_no[s])][real[s]]
                real[s] += 1
        y = rs.push(t, x, fresh, hold)
        for s in range(3):
            if idx[s] >= 0:
                assert (s, seq_no[s], int(idx[s])) not in got
                got[(s, seq_no[s], int(idx[s]))] = y[s]
    worst = 0.0
    for (s, q), seq in seqs.items():
        L = len(seq) if (s, q) != (2, 0) else cut2
        pad = (rf - 1) // 2
        shift = pad if causal else 0
        if twin:
            want = O.tta_merge(O.forward(O.tta_prepare(seq[:L], pad, shift, LEFT, RIGHT), p, adj, fw, causal=causal),
                               LEFT, RIGHT)
        else:
            padded = np.pad(seq[:L], ((pad + shift, pad - shift), (0, 0), (0, 0)), 'edge')[None]
            want = O.forward(padded, p, adj, fw, causal=causal)[0]
        n_out = L if (s, q) != (2, 0) else max(0, L - delay)          # the cut sequence loses its last `delay` poses
        for f in range(n_out):
            worst = max(worst, float(np.abs(got.pop((s, q, f)) - want[f]).max()))
    assert not got, sorted(got)                                       # nothing returned twice or for a wrong frame
    assert worst < 1e-5, worst


def test_delay_index_bookkeeping():
    """frame indices of a hand-worked scenario, delay 2"""
    ix = DelayIndex(3, 2)
    out = []
    for t in range(9):
        ended = []
        if t == 3:
            ix.reset([2])
        if t >= 2:
            ended.append(0)                                # stream 0: frames 0, 1, then held
        if t >= 6:
            ended.append(1)                                # stream 1: frames 0..5
        fresh, hold, idx = ix.step(ended)
        out.append((fresh.tolist(), hold.tolist(), idx.tolist()))
    assert [o[0] for o in out][:4] == [[True] * 3, [False] * 3, [False] * 3, [False, False, True]]
    assert [o[1][0] for o in out] == [False, False] + [True] * 7
    idx = np.array([o[2] for o in out])
    assert idx[:, 0].tolist() == [-1, -1, 0, 1, -1, -1, -1, -1, -1]
    assert idx[:, 1].tolist() == [-1, -1, 0, 1, 2, 3, 4, 5, -1]
    assert idx[:, 2].tolist() == [-1, -1, 0, -1, -1, 0, 1, 2, 3]   # restarted at push 3: its old frame 1 is lost
    with pytest.raises(ValueError, match='before their first frame'):
        ix.reset([1])
        ix.step([1])
    ix2 = DelayIndex(2, 0)
    assert ix2.step()[2].tolist() == [0, 0]
    assert ix2.step([1])[2].tolist() == [1, -1]             # causal: a held push returns nothing new


@pytest.mark.parametrize('name', ['delayed_17_333_c32', 'delayed_17_333_c32_noaug'])
def test_delayed_goldens_match_oracle(name):
    """the reference's augmented whole-sequence outputs stored for the GPU tests agree with the numpy oracle"""
    from conftest import load_golden
    from model.gast_net import SpatioTemporalModel
    from common.skeleton import Skeleton
    from common.graph_utils import adj_mx_from_skeleton
    g = load_golden(name)
    meta = g['meta']
    parents = synth.skeleton_parents(J)
    m = SpatioTemporalModel(adj_mx_from_skeleton(Skeleton(parents, [], [])), J, 2, J, meta['filter_widths'],
                            channels=meta['channels'])
    assert [[k, list(v.shape)] for k, v in m.state_dict().items()] == meta['keys']
    synth.randomize_module(m, meta['seed'])
    p = {k: v.numpy() for k, v in m.state_dict().items()}
    adj = O.adj_from_parents(parents)
    pad = (meta['receptive_field'] - 1) // 2
    for s in range(2):
        x = g['x_%d' % s]
        if meta['augment']:
            want = O.tta_merge(O.forward(O.tta_prepare(x, pad, 0, LEFT, RIGHT), p, adj, meta['filter_widths']),
                               LEFT, RIGHT)
        else:
            want = O.forward(np.pad(x, ((pad, pad), (0, 0), (0, 0)), 'edge')[None], p, adj, meta['filter_widths'])[0]
        assert np.abs(want - g['y_%d' % s]).max() < 1e-4
