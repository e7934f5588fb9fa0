"""ORACLE (test infrastructure, not product): numpy restatement of the ring schedule of the streaming path
(csrc/stream.cuh, gast_stream_push / gast_stream_push_delayed) as the CUDA code runs it, built from the layer
functions of oracle/gast_oracle.py.

Per temporal stage i (width w_i, dilation d_i) a ring of R_i = w_i d_i slots holds the stage's input G_{i-1}; the
push of global step `step` writes slot step mod R_i, reads the taps in SLOT order p0 + k d_i (p0 = slot mod d_i) with
the folded weights rotated by r = slot div d_i, and takes the residual from slot (step - lag_i) mod R_i, lag_i =
pad_i - causal_shift_i.  A fresh stream copies the new slot to all others before the taps are read; a held stream
repeats its newest input frame; with the twin, stream b's mirrored copy is ring row n + b and the shrink output is
un-flipped and averaged (gast_oracle.tta_merge).

Checked against gast_oracle.forward on the edge-padded whole sequence (tests/test_delayed_stream_cpu.py).
"""
import numpy as np

from oracle import gast_oracle as O


def stream_geometry(filter_widths, causal):
    """per temporal stage i >= 1: (w_i, d_i, R_i, lag_i); and the delay sum_i (pad_i - causal_shift_i)"""
    st = []
    d = filter_widths[0]
    delay = 0 if causal else filter_widths[0] // 2
    for w in filter_widths[1:]:
        lag = 0 if causal else (w - 1) * d // 2
        st.append((w, d, w * d, lag))
        delay += lag
        d *= w
    return st, delay


class RingStream(object):
    """n streams of one model (parameters `p` as gast_oracle takes them); `twin` adds the mirrored copies."""

    def __init__(self, p, adj, filter_widths, causal, n, J, F=2, twin=False, kps_left=(), kps_right=(),
                 joints_left=(), joints_right=()):
        self.p, self.fw, self.n, self.J, self.F = p, list(filter_widths), n, J, F
        self.masks = O.local_masks(adj)
        self.stages, self.delay = stream_geometry(self.fw, causal)
        self.twin = twin
        self.rows = 2 * n if twin else n
        self.kperm = np.arange(J)
        self.kperm[list(kps_left)], self.kperm[list(kps_right)] = list(kps_right), list(kps_left)
        self.jl, self.jr = list(joints_left), list(joints_right)
        C = p['expand_conv.weight'].shape[0]
        self.xhist = np.zeros((self.rows, self.fw[0], J, F), np.float32)
        # ring_i[slot] = G_{i-1} of every row in gast_oracle's (B, C, T, N) layout with T = 1 squeezed: (rows, Cw, J)
        self.rings = [np.zeros((R, self.rows, C << (i + 1), J), np.float32) for i, (_, _, R, _) in enumerate(self.stages)]

    def _xpush(self, x, fresh, hold):
        for b in range(self.n):
            fr = bool(fresh[b])
            hd = (not fr) and bool(hold[b])
            v = self.xhist[b, -1].copy() if hd else x[b]
            rows = [(b, v)]
            if self.twin:
                if hd:
                    w = self.xhist[self.n + b, -1].copy()
                else:
                    w = x[b][self.kperm].copy()               # joint j of the twin = joint perm[j] of the frame
                    w[:, 0] = -w[:, 0]                         # feature 0 negated
                rows.append((self.n + b, w))
            for r, val in rows:
                if fr:
                    self.xhist[r] = val[None]
                else:
                    self.xhist[r, :-1] = self.xhist[r, 1:].copy()
                    self.xhist[r, -1] = val

    def push(self, step, x, fresh, hold):
        """x (n, J, F), fresh / hold (n) bool -> (n, J, 3)"""
        p = self.p
        self._xpush(np.asarray(x, np.float32), fresh, hold)
        fr_rows = np.concatenate([fresh, fresh]) if self.twin else np.asarray(fresh)
        h = self.xhist.transpose(0, 3, 1, 2)                                   # (rows, F, k0, J)
        h = O.batchnorm(h, p, 'init_bn.')[0]
        h = O.relu(O.batchnorm(O.conv_t(h, p['expand_conv.weight']), p, 'expand_bn.')[0])
        h = O.graph_attention_block(h, p, 'layers_graph_conv.0.', self.masks)  # (rows, 2C, 1, J)
        for i, (w, d, R, lag) in enumerate(self.stages):
            ring = self.rings[i]
            hs = step % R
            ring[hs] = h[:, :, 0]
            ring[:, fr_rows] = ring[hs, fr_rows][None]                          # fresh fill
            p0, r = hs % d, hs // d
            taps = np.stack([ring[p0 + k * d] for k in range(w)], axis=2)        # (rows, Cw, w, J): slot order
            W = p['layers_conv.%d.weight' % (2 * i)]
            Wrot = W[:, :, [(k - r - 1) % w for k in range(w)]]                 # time order -> slot order
            t = O.relu(O.batchnorm(O.conv_t(taps, Wrot), p, 'layers_bn.%d.' % (2 * i))[0])
            t = O.batchnorm(O.conv1x1(t, p['layers_conv.%d.weight' % (2 * i + 1)]), p, 'layers_bn.%d.' % (2 * i + 1))[0]
            res = ring[(step - lag) % R][:, :, None]                              # (rows, Cw, 1, J)
            h = res + O.relu(t)
            h = O.graph_attention_block(h, p, 'layers_graph_conv.%d.' % (i + 1), self.masks)
        y = O.conv1x1(h, p['shrink.weight'])[:, :, 0].transpose(0, 2, 1)         # (rows, J, 3)
        if self.twin:
            return O.tta_merge(np.stack([y[:self.n], y[self.n:]]), self.jl, self.jr)
        return y
