"""Generate the delayed-stream golden vectors (tests/golden/delayed_*.npz) by running the UNMODIFIED reference on CPU
fp32, with the helpers and the reference import set-up of make_golden.py.

Run in the build container only (the GPU box has no reference checkout):
    python tests/golden/make_delayed_golden.py [OUT_DIR]        (default: tests/golden)

What is stored: what the reference's inference callers compute for every frame of a sequence -- its own
UnchunkedGenerator(pad, causal_shift=0, augment=True, kps_left/right, joints_left/right) (common/generators.py:162-236)
feeding a non-causal dilated SpatioTemporalModel, then the un-flip and average of main.py:314-318.  Two sequences of
different lengths per file (x_0, y_0, x_1, y_1), so that a test can end one stream while the other runs on; one case
without augmentation.  Weights are not stored: gast_b200.synth re-creates them from `seed`.
"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from make_golden import HERE, REF, SpatioTemporalModel, adj_for, keys_shapes, synth  # noqa: E402  (imports the reference)

LEFT, RIGHT = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
CASES = (('delayed_17_333_c32', [3, 3, 3], 32, (41, 29), True, 6),
         ('delayed_17_333_c128', [3, 3, 3], 128, (33, 20), True, 7),
         ('delayed_17_3333_c64', [3, 3, 3, 3], 64, (90, 57), True, 8),
         ('delayed_17_333_c32_noaug', [3, 3, 3], 32, (36, 25), False, 9))


def delayed_stream_cases(out_dir=HERE):
    from common.generators import UnchunkedGenerator
    import common.generators as _gen
    assert _gen.__file__.startswith(REF), _gen.__file__                      # the reference's own generator
    torch.set_grad_enabled(False)
    for name, fw, ch, lens, aug, seed in CASES:
        J = 17
        m = SpatioTemporalModel(adj_for(J), J, 2, J, fw, causal=False, dropout=0.05, channels=ch)
        synth.randomize_module(m, seed)
        m.eval()
        pad = (m.receptive_field() - 1) // 2
        out = {}
        for s, T in enumerate(lens):
            seq = synth.synth_input(1, T, J, 2, 800 + 10 * seed + s)[0]
            kw = dict(kps_left=LEFT, kps_right=RIGHT, joints_left=LEFT, joints_right=RIGHT) if aug else {}
            gen = UnchunkedGenerator(None, None, [seq], pad=pad, causal_shift=0, augment=aug, **kw)
            (_, _, b2), = list(gen.next_epoch())
            assert b2.shape == (2 if aug else 1, T + 2 * pad, J, 2)
            pred = m(torch.from_numpy(b2.astype('float32')))
            if aug:
                pred[1, :, :, 0] *= -1                                                # main.py:315
                pred[1, :, LEFT + RIGHT] = pred[1, :, RIGHT + LEFT]                   # main.py:316
                pred = torch.mean(pred, dim=0, keepdim=True)                          # main.py:317
            out['x_%d' % s], out['y_%d' % s] = seq, pred[0].contiguous().numpy()
        meta = dict(kind='delayed', J=J, filter_widths=fw, channels=ch, strided=False, causal=False, dense=False,
                    seed=seed, keys=keys_shapes(m), receptive_field=m.receptive_field(), augment=aug,
                    kps_left=LEFT, kps_right=RIGHT, joints_left=LEFT, joints_right=RIGHT)
        np.savez_compressed(os.path.join(out_dir, name + '.npz'), meta=json.dumps(meta), **out)
        print('wrote', name, {k: v.shape for k, v in out.items()})


if __name__ == '__main__':
    delayed_stream_cases(sys.argv[1] if len(sys.argv) > 1 else HERE)
