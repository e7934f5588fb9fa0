"""GPU: delayed streaming of causal and non-causal models with test-time augmentation inside the stream
(gast_b200.realtime.DelayedStream, C ABI gast_stream_push_delayed) equals what the reference's inference callers
compute on the whole sequence: UnchunkedGenerator(pad, causal_shift=0[, augment=True]) + the model (+ the un-flip and
average of main.py:314-318).  Runs last: it only composes kernels the other GPU tests have already checked."""
import ctypes as C
import numpy as np
import pytest
import torch

from conftest import load_golden
from gast_b200 import synth, tta
from gast_b200.realtime import CausalStream, DelayedStream, WindowStream
from test_gpu_parity import _adj, TOL

pytestmark = pytest.mark.gpu

J = 17
LEFT, RIGHT = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
SYM = dict(kps_left=LEFT, kps_right=RIGHT, joints_left=LEFT, joints_right=RIGHT)
PERM = list(range(J))
for _l, _r in zip(LEFT, RIGHT):
    PERM[_l], PERM[_r] = _r, _l


def make(fw, ch, causal=False, strided=False, seed=12, dense=False):
    from model.gast_net import SpatioTemporalModel, SpatioTemporalModelOptimized1f
    if strided:
        m = SpatioTemporalModelOptimized1f(_adj(J), J, 2, J, fw, causal=causal, dropout=0.05, channels=ch)
    else:
        m = SpatioTemporalModel(_adj(J), J, 2, J, fw, causal=causal, dropout=0.05, channels=ch, dense=dense)
    synth.randomize_module(m, seed)
    return m.cuda().eval()


def twin_of(frames):
    """the mirrored twin of (n, J, 2) frames, with torch indexing (generators.py:227-233)"""
    t = frames[:, PERM].clone()
    t[..., 0] *= -1
    return t


def collect(ds, out, y, idx):
    """file every returned pose under (stream, 0, frame); a frame returned twice fails"""
    for b in range(ds.n):
        if idx[b] >= 0:
            key = (b, 0, int(idx[b]))
            assert key not in out
            out[key] = y[b]


def test_noncausal_stream_equals_whole_sequence_forward():
    """dilated and Optimized1f non-causal models with the same weights, 3 streams, every frame then drain()"""
    mfull = make([3, 3, 3], 32)
    m1f = make([3, 3, 3], 32, strided=True)
    m1f.load_state_dict(mfull.state_dict())
    n, T = 3, 60
    seqs = torch.from_numpy(synth.synth_input(n, T, J, 2, seed=41)).cuda()
    pad = (mfull.receptive_field() - 1) // 2
    with torch.no_grad():
        want = mfull(torch.from_numpy(np.pad(seqs.cpu().numpy(), ((0, 0), (pad, pad), (0, 0), (0, 0)), 'edge')).cuda())
    for m in (mfull, m1f):
        ds = DelayedStream(m, n)
        assert ds.delay == pad == 13
        got = {}
        for t in range(T):
            collect(ds, got, *ds.push(seqs[:, t]))
        ys, idx = ds.drain()
        assert ys.shape == (pad, n, J, 3) and idx.shape == (pad, n)
        for k in range(pad):
            collect(ds, got, ys[k], idx[k])
        assert sorted(got) == [(b, 0, t) for b in range(n) for t in range(T)]
        err = max((got[(b, 0, t)] - want[b, t]).abs().max().item() for b in range(n) for t in range(T))
        assert err < TOL, err


@pytest.mark.parametrize('name', ['delayed_17_333_c32', 'delayed_17_333_c128', 'delayed_17_3333_c64',
                                  'delayed_17_333_c32_noaug'])
def test_delayed_stream_vs_reference_golden(name):
    """against the UNMODIFIED reference's outputs (tests/golden/make_delayed_golden.py); the shorter
    sequence ends with `ended` while the other stream runs on"""
    g = load_golden(name)
    meta = g['meta']
    m = make(meta['filter_widths'], meta['channels'], seed=meta['seed'])
    assert [[k, list(v.shape)] for k, v in m.state_dict().items()] == meta['keys']
    x0, x1 = g['x_0'], g['x_1']
    assert len(x0) != len(x1)
    long_ = 0 if len(x0) > len(x1) else 1
    xs = [torch.from_numpy(x0).cuda(), torch.from_numpy(x1).cuda()]
    kw = SYM if meta['augment'] else {}
    ds = DelayedStream(m, 2, augment=meta['augment'], **kw)
    got = {}
    for t in range(len(xs[long_])):
        frame = torch.zeros((2, J, 2), device='cuda')
        ended = None
        for b in range(2):
            if t < len(xs[b]):
                frame[b] = xs[b][t]
            else:
                ended = [b]
        collect(ds, got, *ds.push(frame, ended=ended))
    ys, idx = ds.drain()
    for k in range(ds.delay):
        collect(ds, got, ys[k], idx[k])
    assert sorted(got) == sorted([(b, 0, t) for b in range(2) for t in range(len(xs[b]))])
    for b in range(2):
        y = g['y_%d' % b]
        err = max(float(np.abs(got[(b, 0, t)].cpu().numpy() - y[t]).max()) for t in range(len(y)))
        assert err < TOL, (b, err)


def test_delayed_stream_matches_window_recompute_81f():
    """81-frame model (rings of 9, 27 and 81 slots), 5 streams, 100 pushes, resets and ends at different steps:
    the rings with the twin inside against WindowStream on 2n streams (recompute the window for every frame, the
    twin fed as streams n..2n-1, ended streams fed their last frame again) + tta_merge, matched by frame_index"""
    m = make([3, 3, 3, 3], 32, seed=13)
    n, T = 5, 100
    seqs = torch.from_numpy(synth.synth_input(n, T, J, 2, seed=51)).cuda()
    ds = DelayedStream(m, n, augment=True, **SYM)
    assert ds.delay == 40
    ws = WindowStream(m, 2 * n)
    last = seqs[:, 0].clone()
    ended = set()
    worst, compared = 0.0, 0
    for t in range(T):
        if t == 37:
            ds.reset([1, 3]); ws.reset([1, 3, n + 1, n + 3]); ended -= {1, 3}
        if t == 90:
            ds.reset([0]); ws.reset([0, n]); ended -= {0}
        if t == 30:
            ended |= {2}
        if t == 60:
            ended |= {4}
        if t == 85:
            ended |= {1}
        frame = seqs[:, t].clone()
        for b in ended:
            frame[b] = last[b]
        last = frame.clone()
        y, idx = ds.push(seqs[:, t], ended=sorted(ended) or None)
        pred = ws.push(torch.cat([frame, twin_of(frame)]))
        want = tta.tta_merge(pred.view(2, n, J, 3), LEFT, RIGHT)
        for b in range(n):
            if idx[b] >= 0:
                worst = max(worst, (y[b] - want[b]).abs().max().item())
                compared += 1
    assert compared > 150
    assert worst < 2e-5, worst


def test_causal_without_augmentation_is_bitwise_causal_stream():
    m = make([3, 3, 3], 32, causal=True, strided=True, seed=14)
    n, T = 4, 45
    seqs = torch.from_numpy(synth.synth_input(n, T, J, 2, seed=61)).cuda()
    a, b = CausalStream(m, n), DelayedStream(m, n)
    assert b.delay == 0
    for t in range(T):
        if t == 20:
            a.reset([2]); b.reset([2])
        ya = a.push(seqs[:, t])
        yb, idx = b.push(seqs[:, t])
        assert torch.equal(ya, yb), t
        assert idx[2] == (t if t < 20 else t - 20) and idx[0] == t


@pytest.mark.parametrize('causal', [False, True], ids=['noncausal', 'causal'])
def test_augmented_stream_is_bitwise_twin_streams_plus_merge(causal):
    """the twin inside the rings and the merge in the shrink epilogue are bitwise what 2n plain streams fed the
    mirrored frames and tta_merge compute; and per frame they agree with tta.evaluate_sequence"""
    m = make([3, 3, 3], 32, causal=causal, seed=15)
    n, T = 3, 40
    seqs = torch.from_numpy(synth.synth_input(n, T, J, 2, seed=71)).cuda()
    aug = DelayedStream(m, n, augment=True, **SYM)
    plain = DelayedStream(m, 2 * n)
    got = {}
    for t in range(T + aug.delay):
        if t < T:
            y, idx = aug.push(seqs[:, t])
            yp, idxp = plain.push(torch.cat([seqs[:, t], twin_of(seqs[:, t])]))
        else:
            y, idx = aug.push(None, ended=range(n))
            yp, idxp = plain.push(None, ended=range(2 * n))
        merged = tta.tta_merge(yp.view(2, n, J, 3), LEFT, RIGHT)
        assert torch.equal(y, merged), t
        assert (idxp[:n] == idx).all() and (idxp[n:] == idx).all()
        collect(aug, got, y, idx)
    for b in range(n):
        want = tta.evaluate_sequence(m, seqs[b], LEFT, RIGHT, LEFT, RIGHT, causal=causal)
        err = max((got[(b, 0, t)] - want[t]).abs().max().item() for t in range(T))
        assert err < TOL, (b, err)


def test_augmented_push_launches():
    m = make([3, 3, 3], 32, causal=True, strided=True, seed=16)
    n = 8
    frames = torch.from_numpy(synth.synth_input(n, 3, J, 2, seed=81)).cuda()
    a, b = CausalStream(m, n), DelayedStream(m, n, augment=True, **SYM)
    for t in range(3):
        a.push(frames[:, t]); b.push(frames[:, t])
        assert b.last_launches <= a.last_launches + 1, (t, b.last_launches, a.last_launches)


def test_delayed_stream_errors():
    from gast_b200 import _lib as L
    from gast_b200.engine import GastError, model_handle
    with pytest.raises(GastError, match='no streaming form'):
        DelayedStream(make([3, 3, 3], 16, dense=True), 2)
    m = make([3, 3, 3], 16)
    x = torch.zeros((2, J, 2), device='cuda')
    with pytest.raises(GastError, match='out of range'):
        DelayedStream(m, 2, augment=True, kps_left=[4, 17], kps_right=[1, 2], joints_left=[4, 5],
                      joints_right=[1, 2]).push(x)
    with pytest.raises(GastError, match='needs kps_left'):
        DelayedStream(m, 2, augment=True, kps_left=LEFT, kps_right=RIGHT)
    ds = DelayedStream(m, 2)
    with pytest.raises(GastError, match='before their first frame'):
        ds.push(x, ended=[1])
    ds.push(x)                                            # the refused push changed nothing: this one starts both
    ds.reset([0])
    with pytest.raises(GastError, match='before their first frame'):
        ds.push(x, ended=[0])
    with pytest.raises(GastError, match='every stream has ended'):
        ds.push(None, ended=[1])
    m.train()
    with pytest.raises(GastError, match='eval'):
        ds.push(x)
    m.eval()
    with pytest.raises(GastError, match='CUDA device'):
        DelayedStream(make([3, 3, 3], 16).cpu(), 2)
    # a state buffer too small for the augmented layout
    h = model_handle(m, torch.device('cuda', 0))
    lib = h.lib
    nb_plain = lib.gast_stream_delayed_state_bytes(h.h, 2, 0)
    nb_aug = lib.gast_stream_delayed_state_bytes(h.h, 2, 1)
    wb = lib.gast_stream_delayed_workspace_bytes(h.h, 2, 1)
    assert 0 < nb_plain < nb_aug and wb > 0
    assert lib.gast_stream_delay(h.h) == 13
    state = torch.empty(int(nb_aug), dtype=torch.uint8, device='cuda')
    ws = torch.empty(int(wb), dtype=torch.uint8, device='cuda')
    y = torch.empty((2, J, 3), device='cuda')
    fresh = torch.ones(2, dtype=torch.int32, device='cuda')
    il = [(C.c_int32 * 6)(*v) for v in (LEFT, RIGHT, LEFT, RIGHT)]
    with torch.cuda.device(0):
        st = torch.cuda.current_stream().cuda_stream
        h.refresh(m, st)
        rc = lib.gast_stream_push_delayed(h.h, C.c_void_p(state.data_ptr()), nb_plain, 0, C.c_void_p(x.data_ptr()),
                                          C.c_void_p(y.data_ptr()), 2, C.c_void_p(fresh.data_ptr()), None, 6, *il,
                                          C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(st))
        assert rc != 0 and 'state too small' in L.last_error()
        rc = lib.gast_stream_push_delayed(h.h, C.c_void_p(state.data_ptr()), nb_aug, 0, C.c_void_p(x.data_ptr()),
                                          C.c_void_p(y.data_ptr()), 2, C.c_void_p(fresh.data_ptr()), None, 6, *il,
                                          C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(st))
        assert rc == 0, L.last_error()
    # CausalStream keeps refusing non-causal models
    with pytest.raises(RuntimeError, match='causal'):
        CausalStream(m, 2)
