"""Pins the numpy oracle (oracle/gast_oracle.py) against golden outputs of the unmodified
reference (tests/golden/*.npz, produced by tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
from conftest import load_golden, golden_names
from oracle import gast_oracle as O
from gast_b200 import synth

TOL = 2e-5  # fp32 vs fp32 on different op orders; the reference's own fp32-vs-fp64 noise is 2e-7


def params_from_meta(meta):
    return synth.synth_state([(k, tuple(s)) for k, s in meta['keys']], meta['seed'])


def adj_for(J):
    return O.adj_from_parents(synth.skeleton_parents(J))


SMALL_MODELS = golden_names('model_')
CFG_MODELS = golden_names('cfg')


@pytest.mark.parametrize('name', SMALL_MODELS + CFG_MODELS)
def test_model_forward(name):
    g = load_golden(name)
    m = g['meta']
    if name.startswith('cfg1') or name.startswith('cfg4_17_3333_c64_full'):
        pytest.skip('large dilated case: covered on the GPU path; numpy oracle too slow for CPU CI')
    p = params_from_meta(m)
    y = O.forward(g['x'], p, adj_for(m['J']), m['filter_widths'], causal=m['causal'],
                  strided=m['strided'], dense=m['dense'])
    assert y.shape == g['y'].shape
    err = np.abs(y - g['y']).max()
    assert err < TOL, err
    pad, shift, _ = O.model_geometry(m['filter_widths'], m['causal'], m['strided'], m['dense'])
    assert pad == m['pad'] and shift == m['causal_shift']
    assert 1 + 2 * sum(pad) == m['receptive_field']


def test_block():
    for name in ('mod_block_17_32', 'mod_block_19_16'):
        g = load_golden(name)
        m = g['meta']
        p = params_from_meta(m)
        adj = adj_for(m['J'])
        y = O.graph_attention_block(g['x'].transpose(0, 3, 1, 2), p, '', O.local_masks(adj))
        assert np.abs(y - g['y']).max() < TOL


def test_local_and_global_modules():
    g = load_golden('mod_local_17_32')
    p = params_from_meta(g['meta'])
    adj = adj_for(17)
    assert np.abs(O.local_graph(g['x'], p, '', O.local_masks(adj)) - g['y']).max() < TOL
    g = load_golden('mod_mglobal_17_32')
    p = params_from_meta(g['meta'])
    assert np.abs(O.multi_global_graph(g['x'], p, '') - g['y']).max() < TOL
    g = load_golden('mod_global_17_32')
    p = params_from_meta(g['meta'])
    assert np.abs(O.global_graph(g['x'], p, '') - g['y']).max() < TOL


def test_semch_and_shared_e_variant():
    g = load_golden('mod_semch_17_32')
    p = params_from_meta(g['meta'])
    sym, con = O.local_masks(adj_for(17))
    assert (con == g['mask']).all()
    assert np.abs(O.semch_graph_conv(g['x'], p['W'], p['e'], con) - g['y']).max() < TOL
    g = load_golden('mod_semgc_17_32')  # model/sem_graph_conv.py: shared e + bias
    p = params_from_meta(g['meta'])
    assert (con == g['mask']).all()
    assert np.abs(O.semch_graph_conv(g['x'], p['W'], p['e'], con, bias=p['bias']) - g['y']).max() < TOL


def test_adjacency_and_masks():
    a = adj_for(17)
    assert (a > 0).sum() == 49 and np.allclose(a.sum(1), 1)
    sym, con = O.local_masks(a)
    assert sym.sum() == 29 and con.sum() == 54
    a19 = adj_for(19)
    assert (a19 > 0).sum() == 55
    s19, c19 = O.local_masks(a19)
    assert s19.sum() == 33 and c19.sum() == 62
    with pytest.raises(KeyError):
        O.local_masks(np.eye(14, dtype=np.float32))


def test_full_equals_1f_and_sliding_window():
    g = load_golden('model_17_333_c16_full_T31')
    m = g['meta']
    p = params_from_meta(m)
    adj = adj_for(17)
    x = g['x']
    full = O.forward(x, p, adj, m['filter_widths'])
    for t in range(full.shape[1]):
        one = O.forward(x[:, t:t + 27], p, adj, m['filter_widths'], strided=True)
        assert np.abs(one[:, 0] - full[:, t]).max() < TOL


# ---------------------------------------------------------------------------------------------
# the torch-CPU restatement (oracle/gast_torch_ref.py): same goldens, incl. the large ones
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', SMALL_MODELS + CFG_MODELS + golden_names('tc_'))
def test_torch_ref_forward(name):
    import torch
    from oracle import gast_torch_ref as TR
    g = load_golden(name)
    m = g['meta']
    if name.startswith('cfg1') or name.startswith('cfg4_17_3333_c64_full'):
        pytest.skip('large dilated case kept for the GPU path (CPU CI time)')
    p = {k: torch.from_numpy(v) for k, v in params_from_meta(m).items()}
    masks = tuple(torch.from_numpy(a) for a in O.local_masks(adj_for(m['J'])))
    with torch.no_grad():
        y = TR.forward(torch.from_numpy(g['x']), p, masks, m['filter_widths'], causal=m['causal'],
                       strided=m['strided'], dense=m['dense']).numpy()
    assert y.shape == g['y'].shape
    assert np.abs(y - g['y']).max() < TOL


def test_torch_ref_train_mode_matches_numpy_oracle_batch_stats():
    """train-mode BN (batch statistics) agrees between the two restatements, dropout = 0."""
    import torch
    from oracle import gast_torch_ref as TR
    g = load_golden('model_17_333_c16_1f_T27')
    m = g['meta']
    pn = params_from_meta(m)
    adj = adj_for(17)
    yn = O.forward(g['x'], pn, adj, m['filter_widths'], strided=True, training=True)
    p = {k: torch.from_numpy(v) for k, v in pn.items()}
    masks = tuple(torch.from_numpy(a) for a in O.local_masks(adj))
    with torch.no_grad():
        yt = TR.forward(torch.from_numpy(g['x']), p, masks, m['filter_widths'], strided=True, training=True).numpy()
    assert np.abs(yn - yt).max() < 5e-5


def test_tta_restatement_matches_reference_generator():
    """oracle.tta_prepare / tta_merge against batches the reference's UnchunkedGenerator built and the
    un-flip/average of main.py:314-318 (tests/golden/make_golden.py:tta_cases)."""
    g = load_golden('tta_17')
    left, right = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
    for name, pad, shift in (('sym', 13, 0), ('causal', 13, 13), ('pad40', 40, 0)):
        assert np.array_equal(O.tta_prepare(g['seq'], pad, shift, left, right), g['batch_' + name])
    assert np.array_equal(O.tta_merge(g['pred'], left, right), g['merged'][0])
    b = load_golden('cfg1_baseball_17_333_c128')['x']
    assert np.array_equal(O.tta_prepare(b[0, 13:-13], 13, 0, left, right), b)


# ---------------------------------------------------------------------------------------------
# training mode: the differentiable torch port against fixtures of the UNMODIFIED reference
# (forward, mpjpe, every gradient, Adam(amsgrad) steps, running statistics)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', golden_names('train_'))
def test_torch_ref_training_matches_reference_fixture(name):
    import torch
    import train_fixture as TF
    g = load_golden(name)
    meta = g['meta']
    if meta['B'] >= 128 and meta['nsteps'] > 1:
        nsteps = 2                     # CPU CI time: the third step of the b=128 case is checked on the GPU path
    else:
        nsteps = meta['nsteps']
    m = TF.build_module(meta)
    p = {k: v.clone().requires_grad_(v.dtype.is_floating_point and 'running' not in k)
         for k, v in m.state_dict().items()}
    masks = tuple(torch.from_numpy(a) for a in O.local_masks(adj_for(meta['J'])))
    opt = torch.optim.Adam([p[k] for k in meta['names']], lr=meta['lr'], amsgrad=meta['amsgrad'])
    # the CPU kernels split their sums by thread: the port runs with the thread count the fixture was written with,
    # whatever the machine's core count
    nthreads = torch.get_num_threads()
    torch.set_num_threads(meta['threads'])
    try:
        _torch_ref_training_steps(g, meta, nsteps, p, masks, opt)
    finally:
        torch.set_num_threads(nthreads)


def _torch_ref_training_steps(g, meta, nsteps, p, masks, opt):
    from oracle import gast_torch_ref as TR
    import train_fixture as TF
    stats = {}
    for step in range(nsteps):
        x, tgt = TF.batch(meta, step)
        opt.zero_grad()
        y = TR.forward(x, p, masks, meta['filter_widths'], strided=not meta['dilated'], training=True, stats=stats)
        loss = TR.mpjpe(y, tgt)
        loss.backward()
        # same ATen kernels in the same order as the reference modules: agreement is at rounding level
        # same ATen kernels in the same order as the reference modules: step 0 agrees at rounding level; later
        # steps to the reference's own thread-count noise (train_fixture.check_step)
        bad = TF.check_step(g, step, y.detach().numpy(), loss.item(), {k: p[k].grad for k in meta['names']},
                            y_tol=2e-6, loss_rtol=1e-6, ent_rtol=2e-3, norm_rtol=2e-3)
        assert not bad, bad[:10]
        if meta['full_grads'] and step == 0:
            for k in meta['names']:
                gr = g['grad0/' + k]
                if np.abs(gr).max() > 1e-12:
                    assert np.abs(p[k].grad.numpy() - gr).max() <= 2e-3 * np.abs(gr).max(), k
        opt.step()
    if nsteps == meta['nsteps']:
        last = TF.self_noise(g, nsteps - 1)
        tol = 1e-5 if (last is None or nsteps == 1) else max(1e-5, 3.0 * last[1])
        for k, v in stats.items():
            assert np.abs(v.numpy() - g['stat/' + k]).max() < tol * max(1.0, np.abs(g['stat/' + k]).max()), k
