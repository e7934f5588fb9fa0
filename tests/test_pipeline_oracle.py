"""CPU: the numpy restatement of the caller-side steps (oracle/pipeline_oracle.py, SURVEY.md 8f N1-N3)
against outputs of the unmodified reference (tests/golden/pipeline_17.npz)."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import pipeline_oracle as PO

LEFT, RIGHT = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]


def dataset():
    rs = np.random.RandomState(21)
    lens = (40, 7, 25)
    p2 = [rs.standard_normal((n, 17, 2)).astype(np.float32) for n in lens]
    p3 = [rs.standard_normal((n, 17, 3)).astype(np.float32) for n in lens]
    cams = [rs.standard_normal(9).astype(np.float32) for _ in lens]
    return lens, p2, p3, cams


@pytest.fixture(scope='module')
def G():
    return load_golden('pipeline_17')


def test_chunked_generator_matches_reference(G):
    lens, p2, p3, cams = dataset()
    pairs = PO.chunk_pairs(lens, 1, True)
    assert (len(pairs) + 7) // 8 == int(G['cg_a_num_batches'])
    pairs = np.random.RandomState(1234).permutation(pairs)        # generators.py:86-87
    for bi in (0, 1, int(G['cg_a_num_batches']) - 1):
        cam, b3, b2 = PO.chunk_batch(p2, p3, cams, pairs[bi * 8:(bi + 1) * 8], 1, 13, 0, LEFT, RIGHT, LEFT, RIGHT)
        assert np.array_equal(cam, G['cg_a%d_cam' % bi])
        assert np.array_equal(b3, G['cg_a%d_3d' % bi])
        assert np.array_equal(b2, G['cg_a%d_2d' % bi])
    pairs = PO.chunk_pairs(lens, 3, False)
    nb = int(G['cg_b_num_batches'])
    assert (len(pairs) + 4) // 5 == nb
    for bi in (0, nb - 1):
        _, b3, b2 = PO.chunk_batch(p2, p3, None, pairs[bi * 5:(bi + 1) * 5], 3, 4, 4, [], [], [], [])
        assert np.array_equal(b3, G['cg_b%d_3d' % bi])
        assert np.array_equal(b2, G['cg_b%d_2d' % bi])


def test_keypoint_formats_bit_exact(G):
    for fn, src, key in ((PO.coco_h36m, 'k17', 'coco_h36m'), (PO.mpii_h36m, 'k16', 'mpii_h36m'),
                         (PO.coco_h36m_toe_format, 'k133', 'coco_toe')):
        out, valid = fn(G[src])
        assert np.array_equal(out, G[key]), key
        assert np.array_equal(valid, G[key + '_valid']), key


def test_camera_functions(G):
    assert np.array_equal(PO.normalize_screen_coordinates(G['k17'], 1920, 1080), G['norm_screen'])
    assert np.allclose(PO.image_coordinates(G['norm_screen'], 1920, 1080), G['img_coords'], rtol=0, atol=1e-4)
    assert np.abs(PO.camera_to_world(G['x3'], G['rot'], 0) - G['cam2world']).max() < 2e-6


def test_losses(G):
    loss, grad = PO.mpjpe(G['mp_pred'], G['mp_tgt'])
    assert abs(loss - float(G['mp_loss'])) < 1e-6
    assert np.abs(grad - G['mp_grad']).max() < 1e-7
    assert grad[0, 0, 3].tolist() == [0.0, 0.0, 0.0]
    per = PO.p_mpjpe_per_frame(G['pm_pred'], G['pm_tgt'])
    assert np.abs(per - G['pm_per_frame']).max() < 2e-5           # the reference runs this in float32
    assert abs(per.mean() - float(G['pm_value'])) < 2e-5


def adam_inputs():
    rs = np.random.RandomState(22)
    # replay make_golden.pipeline_cases' RandomState(22) stream up to the Adam part
    rs.uniform(0, 1000, (12, 17, 2)); rs.uniform(0, 1000, (9, 16, 2)); rs.uniform(0, 1000, (7, 133, 2))
    rs.standard_normal((11, 17, 3))
    rs.standard_normal((6, 1, 17, 3)); rs.standard_normal((6, 1, 17, 3))
    rs.standard_normal((7, 17, 3)); rs.standard_normal((7, 17, 3))
    shapes = [(5000,), (33, 7), (1,)]
    ps = [rs.standard_normal(sh).astype(np.float32) for sh in shapes]
    grads = [[rs.standard_normal(sh).astype(np.float32) * (10.0 if step == 1 else 0.1) for sh in shapes]
             for step in range(4)]
    return ps, grads


def test_adam_amsgrad(G):
    ps, grads = adam_inputs()
    for i, p in enumerate(ps):
        p = p.astype(np.float64)
        m, v, vm = np.zeros_like(p), np.zeros_like(p), np.zeros_like(p)
        lr = 1e-3
        for step in range(4):
            PO.adam_amsgrad_step(p, grads[step][i].astype(np.float64), m, v, vm, step + 1, lr)
            lr *= 0.95
        assert np.abs(p - G['adam_p%d' % i]).max() < 2e-6, i


def test_oracle_vs_live_reference_random_configs():
    """The reference's own ChunkedGenerator / converters on random configurations (short videos, long chunks, causal
    shifts, ragged last batch; every batch of their output in tests/golden/pipeline_17_random.npz, written by
    make_golden.py:pipeline_random_cases) against the oracle, bit for bit."""
    R = load_golden('pipeline_17_random')
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
        nb = int(R['t%d_num_batches' % trial])
        pairs = PO.chunk_pairs(lens, chunk, augment)
        assert nb == (len(pairs) + bs - 1) // bs
        pairs = np.random.RandomState(99).permutation(pairs)
        for bi in range(nb):
            oc, o3, o2 = PO.chunk_batch(p2, p3, cams, pairs[bi * bs:(bi + 1) * bs], chunk, pad, shift, LEFT, RIGHT, LEFT, RIGHT)
            assert np.array_equal(oc, R['t%d_b%d_cam' % (trial, bi)]), (trial, bi)
            assert np.array_equal(o3, R['t%d_b%d_3d' % (trial, bi)]), (trial, bi)
            assert np.array_equal(o2, R['t%d_b%d_2d' % (trial, bi)]), (trial, bi)
        assert 't%d_b%d_2d' % (trial, nb) not in R
    for T in (1, 5, 64):
        k = rs.uniform(-500, 2000, (T, 17, 2)).astype(np.float32)
        b, vb = PO.coco_h36m(k)
        assert np.array_equal(R['coco_h36m_T%d' % T], b) and np.array_equal(R['coco_h36m_T%d_valid' % T], vb)
        k16 = rs.uniform(-500, 2000, (T, 16, 2)).astype(np.float32)
        b, vb = PO.mpii_h36m(k16)
        assert np.array_equal(R['mpii_h36m_T%d' % T], b) and np.array_equal(R['mpii_h36m_T%d_valid' % T], vb)
