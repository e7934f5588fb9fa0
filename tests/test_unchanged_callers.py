"""The reference's own callers, UNCHANGED, over the drop-in (BASELINE north_star: "trainval.py and reconstruction.py
call it unchanged"; SURVEY.md §8b).  The caller files are not part of this repository: build() copies them from an
upstream GAST-Net checkout into the git-ignored oracle/_ref/ (oracle/ref_callers.py: the caller files only, never
model/).  Without that copy the tests that run the callers are skipped.

What runs unchanged: `reconstruction.reconstruction(args)` (reconstruction.py:173-267: json -> coco_h36m ->
normalize_screen_coordinates -> UnchunkedGenerator + TTA -> model -> camera_to_world) on the real baseball clip
with a synthesised checkpoint, `main.create_model` / `main.train` (main.py:160-243) on a synthetic
ChunkedGenerator, and the `nn.DataParallel(device_ids=[0, 1])` branch of trainval.py:56-61 (2 GPUs).
"""
import importlib
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import load_golden, REPO, PKG
from gast_b200 import synth

REF = os.path.join(REPO, 'oracle', '_ref')

LEFT, RIGHT = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]


@pytest.fixture(scope='module')
def callers():
    """import the reference's reconstruction.py and main.py with the drop-in package AHEAD of the reference root on
    sys.path (INTEGRATION.md §1) -- the only 'installation' step a user performs"""
    if not os.path.exists(os.path.join(REF, 'reconstruction.py')):
        pytest.skip('reference caller files not available (build() copies them into oracle/_ref/ from an upstream '
                    'checkout, see oracle/ref_callers.py)')
    saved_path, saved_mods = list(sys.path), dict(sys.modules)
    for name in ('matplotlib', 'matplotlib.pyplot', 'matplotlib.animation', 'mpl_toolkits', 'mpl_toolkits.mplot3d'):
        if name not in sys.modules:                       # rendering back end absent from the image; never called here
            sys.modules[name] = types.ModuleType(name)
    sys.modules['matplotlib'].use = lambda *a, **k: None
    sys.modules['matplotlib.animation'].FuncAnimation = object
    sys.modules['matplotlib.animation'].writers = {}
    sys.modules['mpl_toolkits.mplot3d'].Axes3D = object
    sys.path[:] = [PKG, REF] + [p for p in sys.path if p not in (PKG, REF)]
    for name in ('reconstruction', 'main'):
        sys.modules.pop(name, None)
    rec = importlib.import_module('reconstruction')
    mn = importlib.import_module('main')
    yield rec, mn
    sys.path[:] = saved_path
    for name in list(sys.modules):
        if name not in saved_mods and name.split('.')[0] in ('reconstruction', 'main', 'tools', 'matplotlib', 'mpl_toolkits'):
            sys.modules.pop(name, None)


def test_star_imports_resolve_to_the_drop_in(callers):
    rec, mn = callers
    import model.gast_net
    assert model.gast_net.__file__.startswith(PKG)
    assert rec.SpatioTemporalModel is model.gast_net.SpatioTemporalModel           # `from model.gast_net import *`
    assert mn.SpatioTemporalModelOptimized1f is model.gast_net.SpatioTemporalModelOptimized1f
    assert mn.nn is torch.nn and mn.torch is torch                                  # trainval.py:60 needs `nn` via main
    assert os.path.abspath(rec.normalize_screen_coordinates.__code__.co_filename).startswith(REF)   # callers' own helpers
    assert os.path.abspath(rec.UnchunkedGenerator.next_epoch.__code__.co_filename).startswith(REF)
    assert os.path.abspath(rec.adj_mx_from_skeleton.__code__.co_filename).startswith(PKG)


def test_shadowed_common_modules_keep_the_reference_contract():
    """common/graph_utils.py and common/skeleton.py of the drop-in shadow the reference's for every caller: same
    results, including adj_mx_from_edges' sparse default and Skeleton.remove_joints (h36m_dataset.py:236-247).
    The reference's results are tests/golden/shadowed_common.npz (make_golden.py:shadowed_common_cases)."""
    import common.graph_utils as G
    import common.skeleton as S
    R = load_golden('shadowed_common')
    b = R['meta']
    h36m_parents = [-1, 0, 1, 2, 3, 4, 0, 6, 7, 8, 9, 0, 11, 12, 13, 14, 12, 16, 17, 18, 19, 20, 19, 22, 12, 24, 25, 26,
                    27, 28, 27, 30]
    jl, jr = [6, 7, 8, 9, 10, 16, 17, 18, 19, 20, 21, 22, 23], [1, 2, 3, 4, 5, 24, 25, 26, 27, 28, 29, 30, 31]
    a = S.Skeleton(list(h36m_parents), list(jl), list(jr))
    remove = [4, 5, 9, 10, 11, 16, 20, 21, 22, 23, 24, 28, 29, 30, 31]                # h36m_dataset.py:241
    assert list(a.remove_joints(list(remove))) == b['kept']
    assert list(a.parents()) == b['parents'] and a.num_joints() == b['num_joints'] == 17
    assert list(a.joints_left()) == b['joints_left'] and list(a.joints_right()) == b['joints_right']
    assert np.array_equal(a.has_children(), R['has_children']) and [list(c) for c in a.children()] == b['children']
    assert torch.equal(G.adj_mx_from_skeleton(a), torch.from_numpy(R['adj_skeleton']))
    for J in (15, 16, 17, 19):
        edges = [(i, q) for i, q in enumerate(synth.skeleton_parents(J)) if q >= 0]
        assert torch.equal(G.adj_mx_from_edges(J, edges, sparse=False), torch.from_numpy(R['adj_edges_dense_J%d' % J]))
        sa = G.adj_mx_from_edges(J, edges)                                              # default: sparse
        assert sa.is_sparse and torch.equal(sa.to_dense(), torch.from_numpy(R['adj_edges_sparse_J%d' % J]))


def _reconstruction_args(tmp_path, weight='27_frame_model.bin'):
    return types.SimpleNamespace(num_joints=17, keypoints_file=os.path.join(REF, 'data/keypoints/baseball.json'),
                                 kpts_format='coco', video_path=os.path.join(REF, 'data/video/baseball.mp4'),
                                 frames=27, causal=False, weight=weight, viz_output=str(tmp_path / 'out.mp4'))


def _write_checkpoint(tmp_path, seed=1):
    """./checkpoint/gastnet/27_frame_model.bin = {'model_pos': state_dict} (reconstruction.py:238-240), weights of
    golden cfg1 (synth seed 1)"""
    from model.gast_net import SpatioTemporalModel
    from common.skeleton import Skeleton
    from common.graph_utils import adj_mx_from_skeleton
    adj = adj_mx_from_skeleton(Skeleton(synth.skeleton_parents(17), LEFT, RIGHT))
    m = SpatioTemporalModel(adj, 17, 2, 17, [3, 3, 3], channels=128, dropout=0.05)
    synth.randomize_module(m, seed)
    d = tmp_path / 'checkpoint' / 'gastnet'
    d.mkdir(parents=True)
    torch.save({'model_pos': m.state_dict()}, str(d / '27_frame_model.bin'))


def test_reconstruction_reaches_the_drop_in_forward_on_cpu(callers, tmp_path, monkeypatch):
    """build container (no GPU): the unchanged caller runs up to the first forward, which refuses the CPU tensor
    loudly -- there is no fallback path to take."""
    if torch.cuda.is_available():
        pytest.skip('CPU-only check')
    rec, _ = callers
    _write_checkpoint(tmp_path)
    monkeypatch.chdir(tmp_path)
    with pytest.raises(RuntimeError, match='no CPU path'):
        rec.reconstruction(_reconstruction_args(tmp_path))


@pytest.mark.gpu
def test_reconstruction_unchanged_on_the_gpu(callers, tmp_path, monkeypatch):
    """reconstruction.reconstruction(args) end to end on the baseball clip; result against the reference-generated
    golden of the same network (cfg1) pushed through the callers' own post-processing."""
    from oracle import gast_oracle as O
    rec, _ = callers
    _write_checkpoint(tmp_path)
    monkeypatch.chdir(tmp_path)
    got = {}
    monkeypatch.setattr(rec, 'render_animation', lambda kp, meta, poses, *a, **k: got.update(poses))
    rec.reconstruction(_reconstruction_args(tmp_path))
    out = got['Reconstruction']
    g = load_golden('cfg1_baseball_17_333_c128')
    want = rec.camera_to_world(O.tta_merge(g['y'], LEFT, RIGHT), R=rec.rot, t=0)
    want[:, :, 2] -= np.min(want[:, :, 2])
    assert out.shape[1:] == (17, 3) and out.shape[0] >= want.shape[0]
    valid = np.where(np.abs(out).reshape(out.shape[0], -1).sum(1) != 0)[0]
    assert len(valid) == want.shape[0]
    assert np.abs(out[valid] - want).max() < 1e-4


@pytest.mark.gpu
def test_main_train_unchanged_on_the_gpu(callers):
    """main.create_model + main.train (main.py:160-243) with the reference's ChunkedGenerator on synthetic data;
    the epoch loss against the torch port driven by the same batches."""
    from oracle import gast_torch_ref as TR
    from oracle import gast_oracle as O
    rec, mn = callers
    rs = np.random.RandomState(5)
    p2 = [rs.standard_normal((40, 17, 2)).astype(np.float32) * 0.5 for _ in range(2)]
    p3 = [rs.standard_normal((40, 17, 3)).astype(np.float32) * 0.5 for _ in range(2)]
    args = types.SimpleNamespace(architecture='3,3,3', disable_optimizations=False, stride=1, causal=False, dropout=0.0,
                                 channels=32)
    skel = rec.Skeleton(parents=synth.skeleton_parents(17), joints_left=LEFT, joints_right=RIGHT)
    dataset = types.SimpleNamespace(skeleton=lambda: skel)
    model_train, model_pos, pad, shift = mn.create_model(args, dataset, p2)
    assert type(model_train).__name__ == 'SpatioTemporalModelOptimized1f' and pad == 13 and shift == 0
    synth.randomize_module(model_train, 4)
    sd0 = {k: v.clone() for k, v in model_train.state_dict().items()}
    model_train = model_train.cuda()
    gen = lambda: rec.ChunkedGenerator(16, None, p3, p2, 1, pad=pad, causal_shift=shift, shuffle=False, augment=False)
    opt = torch.optim.Adam(model_train.parameters(), lr=1e-3, amsgrad=True)
    model_train.train()
    loss = mn.train(model_train, gen(), opt)
    # the same epoch through the differentiable CPU port of the reference
    p = {k: v.clone().requires_grad_(v.dtype.is_floating_point and 'running' not in k) for k, v in sd0.items()}
    masks = tuple(torch.from_numpy(a) for a in O.local_masks(O.adj_from_parents(synth.skeleton_parents(17))))
    opt_ref = torch.optim.Adam([v for v in p.values() if v.requires_grad], lr=1e-3, amsgrad=True)
    tot, n, stats = 0.0, 0, {}
    for _, b3, b2 in gen().next_epoch():
        t3 = torch.from_numpy(b3.astype('float32'))
        t3[:, :, 0] = 0
        opt_ref.zero_grad()
        y = TR.forward(torch.from_numpy(b2.astype('float32')), p, masks, [3, 3, 3], strided=True, training=True, stats=stats)
        l = TR.mpjpe(y, t3)
        l.backward()
        opt_ref.step()
        tot += t3.shape[0] * t3.shape[1] * l.item()
        n += t3.shape[0] * t3.shape[1]
    assert n == 80 and abs(loss - tot / n) < 2e-4 * (tot / n), (loss, tot / n)
    # main.eval's hand-over: the eval model takes the training model's state_dict (main.py:252)
    model_pos = model_pos.cuda()
    model_pos.load_state_dict(model_train.state_dict())
    model_pos.eval()
    with torch.no_grad():
        assert torch.isfinite(model_pos(torch.from_numpy(np.pad(p2[0], ((13, 13), (0, 0), (0, 0)), 'edge')[None]).cuda())).all()


@pytest.mark.gpu
def test_dataparallel_branch_of_trainval(callers):
    """trainval.py:56-61 wraps both models in nn.DataParallel(device_ids=[0, 1]) whenever more than one GPU is
    visible: the per-forward replicas (broadcast parameter views, no `_parameters`) bind and run, eval output equals
    the single-device forward, and a training step routes gradients to the real parameters."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs (the DataParallel branch is taken only with more than one)')
    _, mn = callers
    from model.gast_net import SpatioTemporalModelOptimized1f
    from common.skeleton import Skeleton
    from common.graph_utils import adj_mx_from_skeleton
    adj = adj_mx_from_skeleton(Skeleton(synth.skeleton_parents(17), LEFT, RIGHT))
    m = SpatioTemporalModelOptimized1f(adj, 17, 2, 17, [3, 3, 3], channels=32, dropout=0.0)
    synth.randomize_module(m, 6)
    m = m.cuda()
    dp = mn.nn.DataParallel(m, device_ids=[0, 1])
    x = torch.from_numpy(synth.synth_input(10, 27, 17, 2, seed=8)).cuda()
    m.eval()
    with torch.no_grad():
        want = m(x)
        got = dp(x)
    assert torch.equal(got.cpu(), want.cpu())
    m.train()
    opt = torch.optim.Adam(dp.parameters(), lr=1e-3, amsgrad=True)
    tgt = torch.from_numpy(synth.synth_target(10, 17, seed=9)).cuda()
    before = [p.detach().clone() for p in m.parameters()]
    opt.zero_grad()
    loss = torch.mean(torch.norm(dp(x) - tgt, dim=3))
    loss.backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())
    opt.step()
    assert sum(int((a != b.detach()).any()) for a, b in zip(before, m.parameters())) > 100
    # per-replica BatchNorm statistics like the reference's DataParallel; gradients = sum over the two replicas:
    # the same step done by hand on the two halves
    m2 = SpatioTemporalModelOptimized1f(adj, 17, 2, 17, [3, 3, 3], channels=32, dropout=0.0)
    synth.randomize_module(m2, 6)
    m2 = m2.cuda().train()
    ya, yb = m2(x[:5]), m2(x[5:])
    l2 = torch.mean(torch.norm(torch.cat([ya, yb]) - tgt, dim=3))
    assert abs(l2.item() - loss.item()) < 1e-5 * abs(loss.item())
