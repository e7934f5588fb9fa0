"""Training path (SURVEY.md §8 row a12, BASELINE configs[2]) on the GPU against the torch-CPU port of
the reference under autograd: train-mode forward (batch-stat BN, running-stat update), every
parameter gradient, and a 3-step Adam(amsgrad) loop with loss / state_dict match (dropout 0)."""
import os
import numpy as np
import pytest
import torch

from conftest import load_golden, golden_names
from gast_b200 import synth
import train_fixture as TF

REPORT_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gpurun_out')


def _report(name, lines):
    try:
        os.makedirs(REPORT_DIR, exist_ok=True)
        with open(os.path.join(REPORT_DIR, name), 'a') as f:
            f.write('\n'.join(lines) + '\n')
    except OSError:
        pass

pytestmark = pytest.mark.gpu


def _adj(J):
    from common.skeleton import Skeleton
    from common.graph_utils import adj_mx_from_skeleton
    return adj_mx_from_skeleton(Skeleton(synth.skeleton_parents(J), [], []))


def _masks(J):
    from oracle import gast_oracle as O
    return tuple(torch.from_numpy(a) for a in O.local_masks(O.adj_from_parents(synth.skeleton_parents(J))))


def _oracle_step(p, x, target, fw, J, stats):
    from oracle import gast_torch_ref as TR
    y = TR.forward(x, p, _masks(J), fw, strided=True, training=True, stats=stats)
    return y, TR.mpjpe(y, target)


@pytest.mark.parametrize('J,fw,ch,B', [(17, [3, 3, 3], 32, 6), (17, [3, 3, 3], 128, 16), (19, [3, 3], 32, 5)])
def test_train_forward_and_gradients(J, fw, ch, B):
    from model.gast_net import SpatioTemporalModelOptimized1f
    T = int(np.prod(fw))
    m = SpatioTemporalModelOptimized1f(_adj(J), J, 2, J, fw, dropout=0.0, channels=ch)
    synth.randomize_module(m, 5)
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    x = torch.from_numpy(synth.synth_input(B, T, J, 2, seed=3))
    tgt = torch.from_numpy(synth.synth_target(B, J, seed=4))
    # oracle: autograd through the torch-CPU port, in fp32 (forward / loss / running statistics) and in
    # fp64 (gradients: fp32 gradients of this net carry ~1e-2 max-normalised noise from ReLU decisions
    # of near-zero BatchNorm outputs -- the fp32 CPU port is itself that far from fp64, see
    # profiles/r01_train_grad_report.txt -- so the gradient oracle has to be the fp64 one)
    p = {k: v.clone().requires_grad_(v.dtype.is_floating_point and 'running' not in k) for k, v in sd0.items()}
    stats = {}
    y_ref, loss_ref = _oracle_step(p, x, tgt, fw, J, stats)
    # The reference's fp32 gradients move with the CPU thread count (the CPU kernels split their sums by thread), and
    # where a (Leaky)ReLU input sits within rounding of zero they move discretely: at J=17/128ch the theta/phi biases
    # of the last attention block are 1e-6 from fp64 at 8 and 16 threads but 8e-3 at 4 threads.  So the reference's
    # noise is measured at fixed thread counts, the same on every machine, and its largest value is the bar.
    g32s = []
    nthreads = torch.get_num_threads()
    try:
        for nt in (1, 4, 8, 16):
            torch.set_num_threads(nt)
            q = {k: v.detach().clone().requires_grad_(v.requires_grad) for k, v in p.items()}
            _oracle_step(q, x, tgt, fw, J, {})[1].backward()
            g32s.append({k: v.grad.double() for k, v in q.items() if v.requires_grad})
    finally:
        torch.set_num_threads(nthreads)
    pd = {k: (v.detach().double().requires_grad_(v.requires_grad) if v.dtype.is_floating_point else v.clone())
          for k, v in p.items()}
    _, loss_d = _oracle_step(pd, x.double(), tgt.double(), fw, J, {})
    loss_d.backward()
    # CUDA path
    m = m.cuda().train()
    y = m(x.cuda())
    loss = torch.mean(torch.norm(y - tgt.cuda(), dim=3))
    loss.backward()
    scale = float(y_ref.detach().abs().max())
    loss_ref = loss_ref.detach()
    assert (y.detach().cpu() - y_ref.detach()).abs().max().item() < 5e-5 * max(scale, 1.0)
    assert abs(loss.item() - loss_ref.item()) < 1e-5 * max(1.0, abs(loss_ref.item()))
    # running statistics updated like nn.BatchNorm2d(momentum=0.1)
    sd1 = m.state_dict()
    for k, v in stats.items():
        assert (sd1[k].cpu() - v).abs().max().item() < 1e-5 * max(1.0, float(v.abs().max())), k
    assert int(sd1['init_bn.num_batches_tracked']) == 1
    # every parameter gradient.  fp32 gradients of this net are chaotic at the 1e-3..1e-2 level (a BatchNorm
    # output that lands on the other side of zero flips a ReLU and changes the gradient discretely), so the
    # bar is the reference's OWN fp32 noise against fp64 (its largest over the fixed thread counts above): in
    # aggregate (all gradients concatenated, and the median per-tensor ratio) the CUDA path must be within 2x of
    # it; per tensor, where single flips dominate, within 4x or an absolute floor.
    bad = []
    num_c = den = 0.0
    num_r = [0.0] * len(g32s)
    ratios = []
    for k, prm in m.named_parameters():
        assert prm.grad is not None, k
        g, gd = prm.grad.cpu().double(), pd[k].grad
        if gd.abs().max().item() < 1e-7:       # zero by construction (a bias in front of a batch-stat BN)
            assert g.abs().max().item() < 1e-5, k
            continue
        l2 = ((g - gd).norm() / gd.norm()).item()
        mx = ((g - gd).abs().max() / gd.abs().max()).item()
        l2_ref = mx_ref = 0.0
        for i, gs in enumerate(g32s):                 # the reference port's own fp32 gradients
            l2_ref = max(l2_ref, ((gs[k] - gd).norm() / gd.norm()).item())
            mx_ref = max(mx_ref, ((gs[k] - gd).abs().max() / gd.abs().max()).item())
            num_r[i] += float((gs[k] - gd).norm() ** 2)
        num_c += float((g - gd).norm() ** 2); den += float(gd.norm() ** 2)
        ratios.append(l2 / max(l2_ref, 1e-7))
        if not (l2 < max(5e-3, 4 * l2_ref) and mx < max(2e-2, 4 * mx_ref)):
            bad.append((k, round(l2, 5), round(l2_ref, 5), round(mx, 5), round(mx_ref, 5)))
    agg_c, agg_r = (num_c / den) ** 0.5, (max(num_r) / den) ** 0.5
    med = float(np.median(ratios))
    _report('train_grad_noise.txt', ['J=%d fw=%s ch=%d B=%d: all-gradient rel. L2 error vs fp64: cuda %.3e, reference fp32 %.3e; '
                                     'median per-tensor ratio %.2f; per-tensor outliers %d' % (J, fw, ch, B, agg_c, agg_r, med, len(bad))])
    assert agg_c <= 2.0 * agg_r + 1e-6, (agg_c, agg_r)
    assert med <= 2.0, med
    assert not bad, sorted(bad, key=lambda t: -t[1])[:12]


def _run_steps(make_opt, nsteps, B=32, seed=9):
    from model.gast_net import SpatioTemporalModelOptimized1f
    J, fw, ch = 17, [3, 3, 3], 128
    m = SpatioTemporalModelOptimized1f(_adj(J), J, 2, J, fw, dropout=0.0, channels=ch)
    synth.randomize_module(m, seed)
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    p = {k: v.clone().requires_grad_(v.dtype.is_floating_point and 'running' not in k) for k, v in sd0.items()}
    opt_ref = make_opt([v for k, v in p.items() if v.requires_grad])
    m = m.cuda().train()
    opt = make_opt(list(m.parameters()))
    stats, losses, g_ref = {}, [], None
    for step in range(nsteps):
        x = torch.from_numpy(synth.synth_input(B, 27, J, 2, seed=100 + step))
        tgt = torch.from_numpy(synth.synth_target(B, J, seed=200 + step))
        opt_ref.zero_grad()
        _, loss_ref = _oracle_step(p, x, tgt, fw, J, stats)
        loss_ref.backward()
        g_ref = {k: v.grad.clone() for k, v in p.items() if v.requires_grad}
        opt_ref.step()
        opt.zero_grad()
        y = m(x.cuda())
        loss = torch.mean(torch.norm(y - tgt.cuda(), dim=3))
        loss.backward()
        opt.step()
        losses.append((loss.item(), loss_ref.item()))
    return m, p, stats, losses, g_ref


def test_three_sgd_steps_match_reference_port():
    """BASELINE configs[2] (Optimized1f [3,3,3]/128ch, here b=32 for CI time): forward + backward +
    optimiser step, three times; the loss must track the reference port to 1e-4 relative and the
    weights / running statistics must agree afterwards.  SGD(momentum) is used for the multi-step
    check because Adam's first steps are ~lr*sign(g): parameters whose gradient is rounding noise
    move by +-lr at random in ANY two implementations (CPU vs GPU reference included)."""
    m, p, stats, losses, _ = _run_steps(lambda ps: torch.optim.SGD(ps, lr=1e-2, momentum=0.9), 3)
    for step, (a, b) in enumerate(losses):
        assert abs(a - b) < 1e-4 * abs(b), (step, a, b)
    sd = m.state_dict()
    for k, v in p.items():
        # init_bn.bias has an identically zero gradient (expand_bn removes any constant it adds), so
        # its drift is pure rounding noise in any implementation and it cannot influence the output
        if 'num_batches' in k or 'running' in k or k == 'init_bn.bias':
            continue
        d = ((sd[k].cpu() - v.detach()).norm() / (v.detach().norm() + 1e-12)).item()
        assert d < 1e-3, (k, d)
    for k, v in stats.items():
        assert (sd[k].cpu() - v).abs().max().item() < 1e-4 * max(1.0, float(v.abs().max())), k
    m.eval()                                   # eval after training sees the new weights and statistics
    with torch.no_grad():
        ye = m(torch.from_numpy(synth.synth_input(4, 27, 17, 2, seed=1)).cuda())
    assert torch.isfinite(ye).all()


def test_one_adam_amsgrad_step_matches_reference_port():
    """trainval.py:78 uses Adam(amsgrad=True): one step, parameters compared where the gradient is
    well above the fp32 gradient noise (|g| > 0.1 max|g| of the tensor:
    Adam's first step is lr*sign(g), so a noise-level entry moves by +-lr at random)."""
    m, p, stats, losses, g_ref = _run_steps(lambda ps: torch.optim.Adam(ps, lr=1e-3, amsgrad=True), 1)
    assert abs(losses[0][0] - losses[0][1]) < 1e-5 * abs(losses[0][1])
    sd = m.state_dict()
    checked = 0
    for k, g in g_ref.items():
        if k == 'init_bn.bias':               # identically zero gradient: rounding noise only
            continue
        sel = g.abs() > 0.1 * g.abs().max()      # fp32 gradients carry up to ~1e-2 max-normalised noise
        if sel.any():
            d = (sd[k].cpu() - p[k].detach())[sel].abs().max().item()
            assert d < 2e-5, (k, d)
            checked += int(sel.sum())
    assert checked > 100000


def test_dropout_and_mode_errors():
    from model.gast_net import SpatioTemporalModel, SpatioTemporalModelOptimized1f
    m = SpatioTemporalModelOptimized1f(_adj(17), 17, 2, 17, [3, 3, 3], dropout=0.25, channels=32).cuda().train()
    x = torch.from_numpy(synth.synth_input(4, 27, 17, 2)).cuda()
    torch.manual_seed(0)
    y1 = m(x)
    torch.manual_seed(0)
    y2 = m(x)
    torch.manual_seed(1)
    y3 = m(x)
    assert torch.equal(y1, y2) and not torch.equal(y1, y3)      # dropout stream follows torch's seed
    y1.sum().backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())
    # a sub-module on its own has no training path: loud error, no fallback
    from model.local_attention import LocalGraph
    lg = LocalGraph(_adj(17), 32, 32, 0.1).cuda().train()
    with pytest.raises(RuntimeError, match='eval'):
        lg(torch.zeros(2, 3, 17, 32, device='cuda'))


@pytest.mark.parametrize('name', golden_names('train_'))
def test_training_vs_reference_fixture(name):
    """a12 / BASELINE configs[2] against fixtures of the UNMODIFIED reference (tests/golden/make_golden.py:
    train_case): main.train()'s loop (main.py:219-239) with Adam(amsgrad) (trainval.py:78), dropout 0.
    `train_cfg3_17_333_c128_b128` is the configuration as specified: -arc 3,3,3, 128 channels, b = 128, three
    steps.  Step 0 (forward, loss, every gradient, the first parameter update) is held to 1e-5 relative in the
    loss; the later steps to 3x the reference's own run-to-run noise (see train_fixture.check_step: SURVEY's
    "rel 1e-5 over >= 3 steps" is not met by the reference against itself -- 8 vs 3 CPU threads differ by 4e-5 at
    step 1 and 1e-3 at step 2).  The dilated case is main.py:171-175's training model."""
    g = load_golden(name)
    meta = g['meta']
    m = TF.build_module(meta).cuda().train()
    opt = torch.optim.Adam(m.parameters(), lr=meta['lr'], amsgrad=meta['amsgrad'])
    rep = ['== ' + name]
    bad = []
    for step in range(meta['nsteps']):
        x, tgt = TF.batch(meta, step)
        opt.zero_grad()
        y = m(x.cuda())
        loss = torch.mean(torch.norm(y - tgt.cuda(), dim=3))
        loss.backward()
        bad += TF.check_step(g, step, y.detach().cpu().numpy(), loss.item(), {k: p.grad for k, p in m.named_parameters()},
                             y_tol=5e-5, loss_rtol=1e-5, ent_rtol=5e-2, norm_rtol=5e-2, report=rep)
        opt.step()
        bad += TF.check_params(g, step, dict(m.named_parameters()), report=rep)
    sd = m.state_dict()
    last = TF.self_noise(g, meta['nsteps'] - 1)
    stat_tol = 1e-4 if (last is None or meta['nsteps'] == 1) else max(1e-4, 3.0 * last[1])
    for k in sd:
        if 'running_' in k:
            ref = g['stat/' + k]
            if not np.abs(sd[k].cpu().numpy() - ref).max() < stat_tol * max(1.0, np.abs(ref).max()):
                bad.append(('running statistic', k))
        if 'num_batches' in k:
            assert int(sd[k]) == int(g['stat/' + k])
    _report('train_fixture_report.txt', rep)
    assert not bad, bad[:10]


def test_two_forwards_before_backward_and_no_grad_forward():
    """several training forwards of one module may be outstanding (micro-batches summed before .backward(), a
    logging forward under no_grad in between): each backward differentiates its own forward."""
    from model.gast_net import SpatioTemporalModelOptimized1f
    m = SpatioTemporalModelOptimized1f(_adj(17), 17, 2, 17, [3, 3, 3], dropout=0.0, channels=32)
    synth.randomize_module(m, 3)
    m = m.cuda().train()
    xa = torch.from_numpy(synth.synth_input(4, 27, 17, 2, seed=1)).cuda()
    xb = torch.from_numpy(synth.synth_input(6, 27, 17, 2, seed=2)).cuda()

    def grads(x):
        m.zero_grad()
        m(x).square().sum().backward()
        return [p.grad.clone() for p in m.parameters()]
    ga, gb = grads(xa), grads(xb)
    m.zero_grad()
    ya = m(xa)
    with torch.no_grad():
        m(xb)                                             # logging forward: replaces nothing
    yb = m(xb)
    (ya.square().sum() + yb.square().sum()).backward()
    for p, a, b in zip(m.parameters(), ga, gb):
        assert torch.allclose(p.grad, a + b, rtol=1e-4, atol=1e-6 * float((a + b).abs().max() + 1e-30))


def test_model_copies_and_fused_adam_refresh():
    """deepcopy / pickling of a module that already ran (EMA, best-model snapshots) works, and FusedAdam's raw
    pointer updates are seen by the cached eval-mode constants."""
    import copy
    import io
    from model.gast_net import SpatioTemporalModelOptimized1f
    from gast_b200.pipeline import FusedAdam
    m = SpatioTemporalModelOptimized1f(_adj(17), 17, 2, 17, [3, 3, 3], dropout=0.0, channels=32)
    synth.randomize_module(m, 3)
    m = m.cuda().eval()
    x = torch.from_numpy(synth.synth_input(4, 27, 17, 2, seed=1)).cuda()
    with torch.no_grad():
        y0 = m(x)
        m2 = copy.deepcopy(m)
        assert torch.equal(m2(x), y0)
        buf = io.BytesIO()
        torch.save(m, buf)
    opt = FusedAdam(m.parameters(), lr=1e-2, amsgrad=True)
    m.train()
    m(x).square().sum().backward()
    opt.step()
    m.eval()
    with torch.no_grad():
        y1 = m(x)
        assert (y1 - y0).abs().max().item() > 1e-4        # the step is visible
        assert torch.equal(m2(x), y0)                     # the copy kept its own weights and handle


def test_fused_adam_invalidates_bn_free_submodule_constants():
    """SemCHGraphConv has no BatchNorm whose buffers would change: only the version bump of FusedAdam.step
    tells the engine that the softmaxed adjacency / packed weights are stale."""
    from model.local_attention import SemCHGraphConv, local_adjacencies
    from gast_b200.pipeline import FusedAdam
    _, con = local_adjacencies(_adj(17))
    sc = SemCHGraphConv(32, 32, con)
    synth.randomize_module(sc, 7)
    sc = sc.cuda()
    x = torch.randn(2, 3, 17, 32, device='cuda')
    with torch.no_grad():
        y0 = sc(x)
    opt = FusedAdam(sc.parameters(), lr=1e-1)
    for p in sc.parameters():
        p.grad = torch.ones_like(p)
    opt.step()
    with torch.no_grad():
        y1 = sc(x)
    assert (y1 - y0).abs().max().item() > 1e-3


def test_graphed_trainer_matches_eager_steps():
    """the CUDA-graph replay of forward + loss + backward (gast_b200.trainer.GraphedTrainer) against the eager step:
    same kernels, same order -> same parameters after three Adam(amsgrad) steps (dropout 0); with dropout the replayed
    masks differ from step to step (device-side dropout counter)."""
    from model.gast_net import SpatioTemporalModelOptimized1f
    from gast_b200.trainer import DataParallelTrainer, GraphedTrainer
    from gast_b200.pipeline import FusedAdam

    def make(drop):
        m = SpatioTemporalModelOptimized1f(_adj(17), 17, 2, 17, [3, 3, 3], dropout=drop, channels=32)
        synth.randomize_module(m, 3)
        return m.cuda()
    opt = lambda ps: FusedAdam(ps, lr=1e-3, amsgrad=True)
    B = 16
    xs = [torch.from_numpy(synth.synth_input(B, 27, 17, 2, seed=40 + i)).cuda() for i in range(3)]
    ys = [torch.from_numpy(synth.synth_target(B, 17, seed=50 + i)).cuda() for i in range(3)]
    a = DataParallelTrainer(make(0.0), opt)
    b = GraphedTrainer(make(0.0), opt, (B, 27, 17, 2), (B, 1, 17, 3))
    b.model.load_state_dict(a.model.state_dict())          # (warm-up steps of the graph trainer touch only gradients / BN stats)
    for x, y in zip(xs, ys):
        la = a.step(x, y)
        lb = b.step(x, y)
        assert abs(float(la) - float(lb)) <= 1e-6 * abs(float(la))
    # same kernels in the same order; the only freedom is the order of the atomics in the scatter-adds, i.e. noise-level
    # gradient entries, which Adam turns into +-lr (DESIGN.md §10): all but a vanishing fraction of the entries agree
    bad = tot = 0
    for (k, p), (_, q) in zip(a.model.named_parameters(), b.model.named_parameters()):
        if k == 'init_bn.bias':                       # identically zero gradient: pure noise under Adam
            continue
        bad += int(((p - q).abs() > 1e-5).sum())
        tot += p.numel()
    assert bad <= 1e-3 * tot, (bad, tot)
    c = GraphedTrainer(make(0.25), opt, (B, 27, 17, 2), (B, 1, 17, 3))
    l1 = float(c.step(xs[0], ys[0]))
    w = [p.detach().clone() for p in c.model.parameters()]
    c.graph.replay()
    g1 = c.flat.flat.clone()
    c.graph.replay()
    assert not torch.equal(g1, c.flat.flat)               # a new dropout mask at every replay
    assert l1 > 0 and all(torch.isfinite(p).all() for p in w)
