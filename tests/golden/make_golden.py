"""Generate golden vectors by running the UNMODIFIED reference (/root/reference) on CPU fp32.

Run in the build container only (the GPU box has no /root/reference):
    python tests/golden/make_golden.py
Writes tests/golden/*.npz.  Weights are NOT stored: they are re-created anywhere from
`gast_b200.synth` (numpy RandomState keyed on state_dict key names), the .npz holds the
state_dict key/shape list, the inputs and the reference outputs.
"""
import os
import sys
import types
import json
import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = '/root/reference'

# torchsummary is imported by the reference (model/gast_net.py:2) but absent from the image
sys.modules['torchsummary'] = types.SimpleNamespace(summary=None)
sys.path.insert(0, REF)
sys.path.insert(1, os.path.join(REPO, 'gast-net-3dposeestimation_b200'))  # only for gast_b200.synth

from model.gast_net import (SpatioTemporalModel, SpatioTemporalModelOptimized1f,   # noqa: E402
                            GraphAttentionBlock)
from model.local_attention import LocalGraph, SemCHGraphConv                         # noqa: E402
from model.global_attention import MultiGlobalGraph, GlobalGraph                     # noqa: E402
from model.sem_graph_conv import SemGraphConv                                        # noqa: E402
from common.skeleton import Skeleton                                                 # noqa: E402
from common.graph_utils import adj_mx_from_skeleton                                  # noqa: E402
import model.gast_net as _ref_mod                                                    # noqa: E402
assert _ref_mod.__file__.startswith(REF), _ref_mod.__file__
from gast_b200 import synth                                                          # noqa: E402

torch.set_grad_enabled(False)


def adj_for(J):
    p = synth.skeleton_parents(J)
    return adj_mx_from_skeleton(Skeleton(parents=p, joints_left=[], joints_right=[]))


def keys_shapes(m):
    return [[k, list(v.shape)] for k, v in m.state_dict().items()]


def save(name, **kw):
    meta = kw.pop('meta')
    np.savez_compressed(os.path.join(HERE, name + '.npz'), meta=json.dumps(meta), **kw)
    print('wrote', name, {k: getattr(v, 'shape', None) for k, v in kw.items()})


def model_case(name, J, fw, ch, B, T, strided, causal=False, dense=False, seed=1, xseed=1234, x=None):
    adj = adj_for(J)
    if strided:
        m = SpatioTemporalModelOptimized1f(adj, J, 2, J, fw, causal=causal, dropout=0.05, channels=ch)
    else:
        m = SpatioTemporalModel(adj, J, 2, J, fw, causal=causal, dropout=0.05, channels=ch, dense=dense)
    synth.randomize_module(m, seed)
    m.eval()
    if x is None:
        x = synth.synth_input(B, T, J, 2, xseed)
    y = m(torch.from_numpy(x)).contiguous().numpy()
    meta = dict(kind='model', J=J, filter_widths=fw, channels=ch, strided=strided, causal=causal,
                dense=dense, seed=seed, keys=keys_shapes(m), pad=m.pad, causal_shift=m.causal_shift,
                receptive_field=m.receptive_field(), total_causal_shift=m.total_causal_shift())
    save(name, x=x, y=y, meta=meta)


def baseball_input():
    """Config 1 input exactly as reconstruction.py builds it (:105-145,:192-218,:251-253):
    json -> person 0 -> coco_h36m -> normalize_screen_coordinates -> edge-pad 13 + flipped twin."""
    from tools.mpii_coco_h36m import coco_h36m
    from common.camera import normalize_screen_coordinates
    with open(os.path.join(REF, 'data/keypoints/baseball.json')) as f:
        info = json.load(f)
    nfr = info['data'][-1]['frame_index']
    kp = np.zeros((2, nfr, 17, 2), dtype=np.float32)
    for fi in info['data']:
        for idx, sk in enumerate(fi['skeleton']):
            if len(sk['bbox']) == 0 or idx + 1 > 2:
                continue
            kp[idx, fi['frame_index'] - 1] = np.asarray(sk['pose'], dtype=np.float32)
    kp = kp[0]
    kp, valid = coco_h36m(kp)
    kp = normalize_screen_coordinates(kp[..., :2], w=1920, h=1080)[valid]
    left, right = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
    b2 = np.expand_dims(np.pad(kp, ((13, 13), (0, 0), (0, 0)), 'edge'), axis=0)
    b2 = np.concatenate((b2, b2), axis=0)          # generators.py:222-233
    b2[1, :, :, 0] *= -1
    b2[1, :, left + right] = b2[1, :, right + left]
    return b2.astype(np.float32)


def tta_cases():
    """N1 goldens: the reference's own UnchunkedGenerator (common/generators.py:162-236) builds the
    padded + mirrored batch; the un-flip/average is main.py:314-318 executed with torch."""
    from common.generators import UnchunkedGenerator
    left, right = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
    rs = np.random.RandomState(11)
    seq = rs.standard_normal((37, 17, 2)).astype(np.float32)
    out = {'seq': seq}
    for name, pad, shift in (('sym', 13, 0), ('causal', 13, 13), ('pad40', 40, 0)):
        gen = UnchunkedGenerator(None, None, [seq], pad=pad, causal_shift=shift, augment=True,
                                 kps_left=left, kps_right=right, joints_left=left, joints_right=right)
        (_, _, batch_2d), = list(gen.next_epoch())
        out['batch_' + name] = batch_2d.astype(np.float32)
    pred = torch.from_numpy(rs.standard_normal((2, 37, 17, 3)).astype(np.float32))
    out['pred'] = pred.numpy().copy()
    pred[1, :, :, 0] *= -1                                                    # main.py:315
    pred[1, :, left + right] = pred[1, :, right + left]                       # main.py:316
    out['merged'] = torch.mean(pred, dim=0, keepdim=True).numpy()             # main.py:317
    np.savez_compressed(os.path.join(HERE, 'tta_17.npz'), **out)
    print('tta_17', {k: v.shape for k, v in out.items()})


def pipeline_cases():
    """N1-N3 goldens (SURVEY.md 8f): the reference's own ChunkedGenerator, keypoint converters, screen
    normalisation, camera_to_world, mpjpe (+ autograd), p_mpjpe and torch.optim.Adam(amsgrad=True).
    Inputs are re-created in the tests from the seeds below; only outputs (and small inputs) are stored."""
    from common.generators import ChunkedGenerator
    from common.loss import mpjpe, p_mpjpe
    from common.camera import normalize_screen_coordinates, image_coordinates, camera_to_world
    from tools.mpii_coco_h36m import coco_h36m, mpii_h36m, coco_h36m_toe_format
    import tools.mpii_coco_h36m as _kc
    assert _kc.__file__.startswith(REF)
    out = {}
    left, right = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
    # --- ChunkedGenerator: 3 videos, augment + shuffle, 27-frame receptive field; and a causal, unshuffled one
    rs = np.random.RandomState(21)
    lens = (40, 7, 25)
    p2 = [rs.standard_normal((n, 17, 2)).astype(np.float32) for n in lens]
    p3 = [rs.standard_normal((n, 17, 3)).astype(np.float32) for n in lens]
    cams = [rs.standard_normal(9).astype(np.float32) for _ in lens]
    gen = ChunkedGenerator(8, cams, p3, p2, 1, pad=13, causal_shift=0, shuffle=True, random_seed=1234, augment=True,
                           kps_left=left, kps_right=right, joints_left=left, joints_right=right)
    with torch.enable_grad():
        pass
    for bi, (cam, b3, b2) in enumerate(gen.next_epoch()):
        if bi in (0, 1, gen.num_batches - 1):
            out['cg_a%d_cam' % bi] = cam.astype(np.float32).copy()
            out['cg_a%d_3d' % bi] = b3.astype(np.float32).copy()
            out['cg_a%d_2d' % bi] = b2.astype(np.float32).copy()
    out['cg_a_num_batches'] = np.array(gen.num_batches)
    gen = ChunkedGenerator(5, None, p3, p2, 3, pad=4, causal_shift=4, shuffle=False, augment=False)
    for bi, (cam, b3, b2) in enumerate(gen.next_epoch()):
        assert cam is None
        if bi in (0, gen.num_batches - 1):
            out['cg_b%d_3d' % bi] = b3.astype(np.float32).copy()
            out['cg_b%d_2d' % bi] = b2.astype(np.float32).copy()
    out['cg_b_num_batches'] = np.array(gen.num_batches)
    # --- keypoint formats (float32 pixel coordinates; one all-zero frame -> not in valid_frames)
    rs = np.random.RandomState(22)
    k17 = (rs.uniform(0, 1000, (12, 17, 2))).astype(np.float32); k17[5] = 0
    k16 = (rs.uniform(0, 1000, (9, 16, 2))).astype(np.float32); k16[2] = 0
    k133 = (rs.uniform(0, 1000, (7, 133, 2))).astype(np.float32); k133[3] = 0
    out['k17'], out['k16'], out['k133'] = k17, k16, k133
    out['coco_h36m'], out['coco_h36m_valid'] = coco_h36m(k17.copy())
    out['mpii_h36m'], out['mpii_h36m_valid'] = mpii_h36m(k16.copy())
    out['coco_toe'], out['coco_toe_valid'] = coco_h36m_toe_format(k133.copy())
    # --- screen normalisation / camera_to_world (reconstruction.py:143,204 call forms)
    out['norm_screen'] = normalize_screen_coordinates(k17[..., :2].copy(), w=1920, h=1080).astype(np.float32)
    out['img_coords'] = image_coordinates(out['norm_screen'].copy(), w=1920, h=1080).astype(np.float32)
    rot = np.array([0.1407056450843811, -0.1500701755285263, -0.755240797996521, 0.6223280429840088], dtype=np.float32)
    x3 = rs.standard_normal((11, 17, 3)).astype(np.float32)
    out['x3'] = x3
    out['rot'] = rot
    out['cam2world'] = camera_to_world(x3.copy(), R=rot, t=0).astype(np.float32)
    # --- mpjpe + gradient, p_mpjpe
    pr = torch.from_numpy(rs.standard_normal((6, 1, 17, 3)).astype(np.float32)).requires_grad_(True)
    tg = torch.from_numpy(rs.standard_normal((6, 1, 17, 3)).astype(np.float32))
    tg.data[0, 0, 3] = pr.data[0, 0, 3]                       # a zero-distance joint (gradient 0 there)
    with torch.enable_grad():
        l = mpjpe(pr, tg)
        l.backward()
    out['mp_pred'], out['mp_tgt'] = pr.detach().numpy().copy(), tg.numpy().copy()
    out['mp_loss'], out['mp_grad'] = np.array(l.item(), np.float32), pr.grad.numpy().copy()
    pp = rs.standard_normal((7, 17, 3)).astype(np.float32)
    pt = (pp * 1.7 + 0.3 * rs.standard_normal((7, 17, 3))).astype(np.float32)
    pt[2, :, 0] *= -1                                           # a mirrored target: the det(R) = -1 branch
    pp[4, :, 2] = 0.0                                           # a planar prediction: rank-deficient H
    out['pm_pred'], out['pm_tgt'] = pp, pt
    out['pm_value'] = np.array(p_mpjpe(pp.copy(), pt.copy()), np.float64)
    out['pm_per_frame'] = np.array([p_mpjpe(pp[i:i + 1].copy(), pt[i:i + 1].copy()) for i in range(7)], np.float64)
    # --- Adam(amsgrad=True), 4 steps with a learning-rate decay in between (trainval.py:78,162-164)
    shapes = [(5000,), (33, 7), (1,)]
    ps = [torch.nn.Parameter(torch.from_numpy(rs.standard_normal(sh).astype(np.float32))) for sh in shapes]
    opt = torch.optim.Adam(ps, lr=1e-3, amsgrad=True)
    grads = []
    for step in range(4):
        gs = [rs.standard_normal(sh).astype(np.float32) * (10.0 if step == 1 else 0.1) for sh in shapes]
        grads.append(gs)
        for p_, g_ in zip(ps, gs):
            p_.grad = torch.from_numpy(g_.copy())
        opt.step()
        for g in opt.param_groups:
            g['lr'] *= 0.95
    for i, p_ in enumerate(ps):
        out['adam_p%d' % i] = p_.detach().numpy().copy()
    np.savez_compressed(os.path.join(HERE, 'pipeline_17.npz'), **out)
    print('pipeline_17', {k: getattr(v, 'shape', None) for k, v in out.items()})


def pipeline_random_cases():
    """The reference's ChunkedGenerator and keypoint converters on random configurations (short videos, long
    chunks, causal shifts, ragged last batch): every batch of every configuration.  The configurations and inputs
    are re-drawn in tests/test_pipeline_oracle.py from the same RandomState(7) stream; only outputs are stored."""
    from common.generators import ChunkedGenerator
    from tools.mpii_coco_h36m import coco_h36m, mpii_h36m
    import tools.mpii_coco_h36m as _kc
    assert _kc.__file__.startswith(REF)
    left, right = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
    out = {}
    rs = np.random.RandomState(7)
    for trial in range(6):
        nseq = int(rs.randint(1, 5))
        lens = [int(v) for v in rs.randint(1, 30, nseq)]
        chunk = int(rs.choice([1, 3, 8]))
        pad = int(rs.randint(0, 14))
        shift = int(rs.choice([0, pad]))
        augment = bool(rs.randint(0, 2))
        bs = int(rs.choice([4, 7]))
        p2 = [rs.standard_normal((n, 17, 2)).astype(np.float32) for n in lens]
        p3 = [rs.standard_normal((n, 17, 3)).astype(np.float32) for n in lens]
        cams = [rs.standard_normal(9).astype(np.float32) for _ in lens]
        gen = ChunkedGenerator(bs, cams, p3, p2, chunk, pad=pad, causal_shift=shift, shuffle=True, random_seed=99,
                               augment=augment, kps_left=left, kps_right=right, joints_left=left, joints_right=right)
        out['t%d_num_batches' % trial] = np.array(gen.num_batches)
        for bi, (cam, b3, b2) in enumerate(gen.next_epoch()):
            out['t%d_b%d_cam' % (trial, bi)] = cam.astype(np.float32)
            out['t%d_b%d_3d' % (trial, bi)] = b3.astype(np.float32)
            out['t%d_b%d_2d' % (trial, bi)] = b2.astype(np.float32)
    for T in (1, 5, 64):
        k = rs.uniform(-500, 2000, (T, 17, 2)).astype(np.float32)
        out['coco_h36m_T%d' % T], out['coco_h36m_T%d_valid' % T] = coco_h36m(k.copy())
        k16 = rs.uniform(-500, 2000, (T, 16, 2)).astype(np.float32)
        out['mpii_h36m_T%d' % T], out['mpii_h36m_T%d_valid' % T] = mpii_h36m(k16.copy())
    np.savez_compressed(os.path.join(HERE, 'pipeline_17_random.npz'), **out)
    print('pipeline_17_random', len(out), 'arrays')


def shadowed_common_cases():
    """What the reference's common/skeleton.py and common/graph_utils.py return for the calls its callers make
    (h36m_dataset.py:236-247 joint removal, adj_mx_from_skeleton, adj_mx_from_edges dense and sparse): the drop-in
    package shadows both modules, and tests/test_unchanged_callers.py holds it to these results."""
    from common.skeleton import Skeleton as RS
    from common.graph_utils import adj_mx_from_skeleton as r_adj_sk, adj_mx_from_edges as r_adj_ed
    import common.graph_utils as _gu
    assert _gu.__file__.startswith(REF)
    h36m_parents = [-1, 0, 1, 2, 3, 4, 0, 6, 7, 8, 9, 0, 11, 12, 13, 14, 12, 16, 17, 18, 19, 20, 19, 22, 12, 24, 25, 26,
                    27, 28, 27, 30]
    jl, jr = [6, 7, 8, 9, 10, 16, 17, 18, 19, 20, 21, 22, 23], [1, 2, 3, 4, 5, 24, 25, 26, 27, 28, 29, 30, 31]
    remove = [4, 5, 9, 10, 11, 16, 20, 21, 22, 23, 24, 28, 29, 30, 31]                # h36m_dataset.py:241
    b = RS(list(h36m_parents), list(jl), list(jr))
    kept = [int(v) for v in b.remove_joints(list(remove))]
    out = {'has_children': np.asarray(b.has_children()), 'adj_skeleton': r_adj_sk(b).numpy()}
    for J in (15, 16, 17, 19):
        edges = [(i, q) for i, q in enumerate(synth.skeleton_parents(J)) if q >= 0]
        out['adj_edges_dense_J%d' % J] = r_adj_ed(J, edges, sparse=False).numpy()
        sp = r_adj_ed(J, edges)
        assert sp.is_sparse
        out['adj_edges_sparse_J%d' % J] = sp.to_dense().numpy()
    meta = dict(kept=kept, parents=[int(v) for v in b.parents()], num_joints=int(b.num_joints()),
                joints_left=[int(v) for v in b.joints_left()], joints_right=[int(v) for v in b.joints_right()],
                children=[[int(c) for c in ch] for ch in b.children()])
    save('shadowed_common', meta=meta, **out)


def module_cases():
    J, C = 17, 32
    adj = adj_for(J)
    x = (0.7 * np.random.RandomState(7).standard_normal((3, 5, J, C))).astype(np.float32)
    xt = torch.from_numpy(x)
    # GraphAttentionBlock on (B,C,T,N)
    blk = GraphAttentionBlock(adj, C, C, p_dropout=0.05)
    synth.randomize_module(blk, 3)
    blk.eval()
    save('mod_block_17_32', x=x, y=blk(xt.permute(0, 3, 1, 2).contiguous()).contiguous().numpy(),
         meta=dict(kind='block', J=J, C=C, seed=3, keys=keys_shapes(blk)))
    lg = LocalGraph(adj, C, C, 0.05)
    synth.randomize_module(lg, 4)
    lg.eval()
    save('mod_local_17_32', x=x, y=lg(xt).contiguous().numpy(),
         meta=dict(kind='local', J=J, C=C, seed=4, keys=keys_shapes(lg)))
    mg = MultiGlobalGraph(adj, C, C // 4, dropout=0.05)
    synth.randomize_module(mg, 5)
    mg.eval()
    save('mod_mglobal_17_32', x=x, y=mg(xt).contiguous().numpy(),
         meta=dict(kind='mglobal', J=J, C=C, seed=5, keys=keys_shapes(mg)))
    gg = GlobalGraph(adj, C, C // 4)
    synth.randomize_module(gg, 6)
    gg.eval()
    xg = xt.reshape(-1, J, C).permute(0, 2, 1).contiguous()
    save('mod_global_17_32', x=xg.numpy(), y=gg(xg).contiguous().numpy(),
         meta=dict(kind='global', J=J, C=C, seed=6, keys=keys_shapes(gg)))
    sc = SemCHGraphConv(C, C, lg.gcn_con.adj[0] if lg.gcn_con.adj.dim() == 3 else lg.gcn_con.adj)
    synth.randomize_module(sc, 7)
    save('mod_semch_17_32', x=x, y=sc(xt).contiguous().numpy(), mask=(sc.m[0]).numpy(),
         meta=dict(kind='semch', J=J, C=C, seed=7, keys=keys_shapes(sc)))
    # the non-channel-wise SemGraphConv of model/sem_graph_conv.py (shared e, bias=True)
    sg = SemGraphConv(C, C, lg.gcn_con.adj[0], bias=True)
    synth.randomize_module(sg, 8)
    save('mod_semgc_17_32', x=x, y=sg(xt).contiguous().numpy(), mask=sg.m.numpy(),
         meta=dict(kind='semgc', J=J, C=C, seed=8, keys=keys_shapes(sg)))
    # 19-joint block
    J2 = 19
    adj2 = adj_for(J2)
    x2 = (0.7 * np.random.RandomState(9).standard_normal((2, 3, J2, 16))).astype(np.float32)
    blk2 = GraphAttentionBlock(adj2, 16, 16, p_dropout=0.05)
    synth.randomize_module(blk2, 9)
    blk2.eval()
    save('mod_block_19_16', x=x2,
         y=blk2(torch.from_numpy(x2).permute(0, 3, 1, 2).contiguous()).contiguous().numpy(),
         meta=dict(kind='block', J=J2, C=16, seed=9, keys=keys_shapes(blk2)))


def _digest(t, idx):
    """compact fingerprint of one tensor: norm, sum, and the entries at `idx` (flat indices)"""
    f = t.detach().reshape(-1).double()
    return np.array([float(f.norm()), float(f.sum())], np.float64), f[idx].numpy().astype(np.float32)


def _train_run(J, fw, ch, B, nsteps, dilated, seed, threads):
    """main.train()'s loop (main.py:219-239) on the reference model, dropout 0, Adam(amsgrad) (trainval.py:78)"""
    from common.loss import mpjpe
    torch.set_num_threads(threads)
    adj = adj_for(J)
    T = int(np.prod(fw))
    if dilated:
        m = SpatioTemporalModel(adj, J, 2, J, fw, dropout=0.0, channels=ch)
    else:
        m = SpatioTemporalModelOptimized1f(adj, J, 2, J, fw, dropout=0.0, channels=ch)
    synth.randomize_module(m, seed)
    m.train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, amsgrad=True)
    steps = []
    with torch.enable_grad():
        for step in range(nsteps):
            x = torch.from_numpy(synth.synth_input(B, T, J, 2, seed=100 + step))
            tgt = torch.from_numpy(synth.synth_target(B, J, seed=200 + step))
            tgt[:, :, 0] = 0                                     # main.py:225
            opt.zero_grad()
            y = m(x)
            loss = mpjpe(y, tgt)
            loss.backward()
            grads = {k: prm.grad.detach().clone() for k, prm in m.named_parameters()}
            opt.step()
            params = {k: prm.detach().clone() for k, prm in m.named_parameters()}
            steps.append(dict(y=y.detach().contiguous().numpy().copy(), loss=loss.item(), grads=grads, params=params))
    return m, steps, T


def train_case(name, J, fw, ch, B, nsteps, full_grads, dilated=False, seed=9):
    """a12 / BASELINE configs[2] golden: the UNMODIFIED reference model in train() mode, dropout 0, driven exactly
    as main.train() drives it with optim.Adam(lr=1e-3, amsgrad=True).  Stored per step: the prediction, the loss,
    and per parameter either the whole gradient (small cases, step 0) or its norm, sum and 48 entries at the flat
    indices where |grad of step 0| is largest; the same fingerprint of every parameter after every step; the
    BatchNorm running statistics after the last step.

    The reference's OWN reproducibility is stored next to it (`alt_*`): the identical run with 3 instead of 8 CPU
    threads (different fp32 summation order, nothing else).  Adam's first updates are lr*g/(|g|+eps): every
    parameter whose gradient is rounding noise moves by +-lr at random, so from the second step on two runs of
    the reference itself only agree to ~5e-5 (step 1) / ~1e-3 (step 2) in the loss at b=128 -- the band any fp32
    implementation can be held to."""
    m, steps, T = _train_run(J, fw, ch, B, nsteps, dilated, seed, threads=8)
    alt = _train_run(J, fw, ch, B, nsteps, dilated, seed, threads=3)[1] if nsteps > 1 else None
    torch.set_num_threads(8)
    names = [k for k, _ in m.named_parameters()]
    out, idx = {}, {}
    for k in names:
        g = steps[0]['grads'][k].reshape(-1)
        idx[k] = torch.topk(g.abs(), min(48, g.numel())).indices.sort().values
        out['idx/' + k] = idx[k].numpy().astype(np.int64)
        if full_grads:
            out['grad0/' + k] = steps[0]['grads'][k].numpy().copy()
    for s, st in enumerate(steps):
        out['y%d' % s] = st['y']
        out['loss%d' % s] = np.array(st['loss'], np.float64)
        for k in names:
            out['gsum%d/%s' % (s, k)], out['gent%d/%s' % (s, k)] = _digest(st['grads'][k], idx[k])
            out['psum%d/%s' % (s, k)], out['pent%d/%s' % (s, k)] = _digest(st['params'][k], idx[k])
        if alt is not None:
            out['alt_loss%d' % s] = np.array(alt[s]['loss'], np.float64)
            out['alt_dy%d' % s] = np.array(np.abs(alt[s]['y'] - st['y']).max(), np.float64)
            out['alt_dp%d' % s] = np.array(max(float((alt[s]['params'][k] - st['params'][k]).abs().max()) for k in names), np.float64)
            out['alt_dg%d' % s] = np.array(max(float((alt[s]['grads'][k] - st['grads'][k]).norm() / (st['grads'][k].norm() + 1e-30))
                                              for k in names if float(st['grads'][k].norm()) > 1e-5), np.float64)
    for k, v in m.state_dict().items():
        if 'running_' in k or 'num_batches' in k:
            out['stat/' + k] = v.numpy().copy()
    meta = dict(kind='train', J=J, filter_widths=fw, channels=ch, B=B, T=T, nsteps=nsteps, seed=seed, dilated=dilated,
                names=names, full_grads=full_grads, lr=1e-3, amsgrad=True, threads=8, alt_threads=3 if alt else None)
    save(name, meta=meta, **out)
    if alt is not None:
        print('   reference self-noise (8 vs 3 threads):', [(float(abs(out['alt_loss%d' % s] - out['loss%d' % s]) / out['loss%d' % s]),
                                                            float(out['alt_dy%d' % s]), float(out['alt_dp%d' % s])) for s in range(nsteps)])


def train_cases():
    train_case('train_17_333_c32_b6', 17, [3, 3, 3], 32, 6, 2, full_grads=True)
    train_case('train_19_33_c32_b5', 19, [3, 3], 32, 5, 1, full_grads=True)
    train_case('train_17_333_c16_dilated_b4', 17, [3, 3, 3], 16, 4, 1, full_grads=True, dilated=True)
    # BASELINE configs[2] at its real size: -arc 3,3,3 -ch 128 -b 128, three Adam(amsgrad) steps
    train_case('train_cfg3_17_333_c128_b128', 17, [3, 3, 3], 128, 128, 3, full_grads=False)


def tc_cases():
    """widths that are multiples of 32, so that the tcgen05 GEMM core (K % 32 == 0) sees every skeleton and
    geometry: J = 15 / 16 / 19, five stages (243 frames, reconstruction.py:226-228), the dense ablation, a
    two-stage model with a 5-wide filter, causal + long-sequence (dilated) mode"""
    model_case('tc_15_333_c32_full_T29', 15, [3, 3, 3], 32, 2, 29, strided=False)
    model_case('tc_16_333_c32_full_T27', 16, [3, 3, 3], 32, 3, 27, strided=False)
    model_case('tc_19_333_c32_1f_T27', 19, [3, 3, 3], 32, 3, 27, strided=True)
    model_case('tc_17_33333_c32_1f_T243', 17, [3, 3, 3, 3, 3], 32, 1, 243, strided=True)
    model_case('tc_17_33333_c32_full_T245', 17, [3, 3, 3, 3, 3], 32, 1, 245, strided=False)
    model_case('tc_17_333_c32_dense_T28', 17, [3, 3, 3], 32, 2, 28, strided=False, dense=True)
    model_case('tc_17_35_c32_full_T17', 17, [3, 5], 32, 2, 17, strided=False)
    model_case('tc_17_333_c32_causal_full_T40', 17, [3, 3, 3], 32, 2, 40, strided=False, causal=True)
    model_case('tc_17_3333_c64_causal_full_T90', 17, [3, 3, 3, 3], 64, 1, 90, strided=False, causal=True)


def stream_cases():
    """N4 goldens (real-time causal path, gen_skes.py:43-69): what the reference produces for EVERY frame of a
    sequence with a causal model -- its own UnchunkedGenerator(pad, causal_shift=pad) (common/generators.py:
    210-221: pad + causal_shift edge-padded frames on the left, none on the right) feeding the causal dilated
    SpatioTemporalModel, whose weights are interchangeable with the causal Optimized1f that the real-time
    model is (gast_net.py:180-251).  A frame-by-frame streaming implementation must reproduce y[t] when frame t
    is pushed."""
    from common.generators import UnchunkedGenerator
    for name, fw, ch, T, seed in (('stream_17_333_c32_causal', [3, 3, 3], 32, 45, 3),
                                  ('stream_17_333_c128_causal', [3, 3, 3], 128, 33, 4),
                                  ('stream_17_3333_c64_causal', [3, 3, 3, 3], 64, 100, 5)):
        J = 17
        m = SpatioTemporalModel(adj_for(J), J, 2, J, fw, causal=True, dropout=0.05, channels=ch)
        synth.randomize_module(m, seed)
        m.eval()
        pad = (m.receptive_field() - 1) // 2
        seqs = synth.synth_input(2, T, J, 2, 700 + seed)
        ys = []
        for sq in seqs:
            gen = UnchunkedGenerator(None, None, [sq], pad=pad, causal_shift=pad, augment=False)
            (_, _, b2), = list(gen.next_epoch())
            assert b2.shape == (1, T + 2 * pad, J, 2)
            ys.append(m(torch.from_numpy(b2.astype('float32'))).contiguous().numpy()[0])
        meta = dict(kind='stream', J=J, filter_widths=fw, channels=ch, strided=False, causal=True, dense=False, seed=seed,
                    keys=keys_shapes(m), receptive_field=m.receptive_field())
        save(name, x=seqs, y=np.stack(ys), meta=meta)


def main():
    torch.manual_seed(0)
    module_cases()
    # small-width end-to-end cases (cheap for the numpy oracle and for CPU CI)
    model_case('model_17_333_c16_full_T31', 17, [3, 3, 3], 16, 3, 31, strided=False)
    model_case('model_17_333_c16_1f_T27', 17, [3, 3, 3], 16, 3, 27, strided=True)
    model_case('model_17_333_c16_1f_T81', 17, [3, 3, 3], 16, 2, 81, strided=True)
    model_case('model_17_333_c16_causal_full_T30', 17, [3, 3, 3], 16, 2, 30, strided=False, causal=True)
    model_case('model_17_333_c16_causal_1f_T27', 17, [3, 3, 3], 16, 2, 27, strided=True, causal=True)
    model_case('model_17_333_c16_dense_T27', 17, [3, 3, 3], 16, 2, 28, strided=False, dense=True)
    model_case('model_15_333_c16_full_T29', 15, [3, 3, 3], 16, 2, 29, strided=False)
    model_case('model_16_333_c16_full_T27', 16, [3, 3, 3], 16, 2, 27, strided=False)
    model_case('model_19_333_c16_full_T29', 19, [3, 3, 3], 16, 2, 29, strided=False)
    model_case('model_17_35_c8_full_T17', 17, [3, 5], 8, 2, 17, strided=False)
    model_case('model_17_33333_c8_1f_T243', 17, [3, 3, 3, 3, 3], 8, 1, 243, strided=True)
    tc_cases()
    # BASELINE.json configs at full width, small batch
    model_case('cfg2_17_333_c128_full_T27', 17, [3, 3, 3], 128, 4, 27, strided=False)
    model_case('cfg2_17_333_c128_full_T40', 17, [3, 3, 3], 128, 1, 40, strided=False)
    model_case('cfg3_17_333_c128_1f_T27', 17, [3, 3, 3], 128, 4, 27, strided=True)
    model_case('cfg4_17_3333_c64_full_T81', 17, [3, 3, 3, 3], 64, 2, 81, strided=False)
    model_case('cfg4_17_3333_c64_1f_T81', 17, [3, 3, 3, 3], 64, 2, 81, strided=True)
    model_case('cfg5_19_333_c128_full_T27', 19, [3, 3, 3], 128, 4, 27, strided=False)
    model_case('cfg1_baseball_17_333_c128', 17, [3, 3, 3], 128, 2, 303, strided=False, x=baseball_input())


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == 'tta':
        tta_cases()
    elif len(sys.argv) > 1 and sys.argv[1] == 'pipeline':
        pipeline_cases()
    elif len(sys.argv) > 1 and sys.argv[1] == 'train':
        train_cases()
    elif len(sys.argv) > 1 and sys.argv[1] == 'tc':
        tc_cases()
    elif len(sys.argv) > 1 and sys.argv[1] == 'stream':
        stream_cases()
    elif len(sys.argv) > 1 and sys.argv[1] == 'contract':
        pipeline_random_cases()
        shadowed_common_cases()
    else:
        main()
        tta_cases()
        pipeline_cases()
        pipeline_random_cases()
        shadowed_common_cases()
        train_cases()
        stream_cases()
