"""Frame-by-frame causal lifting of many concurrent keypoint streams (SURVEY.md §8f N4).

The reference's real-time model is a causal `SpatioTemporalModelOptimized1f` fed the last `receptive_field`
frames of one stream for every new frame (`gen_skes.py:43-69`, `tools/inference.py:19-110`): O(rf) work per
frame.  `CausalStream` produces the same poses with O(1) work per frame: the library keeps, per temporal stage, a
ring of that stage's past inputs for all streams (`csrc/stream.cuh`, C ABI `gast_stream_push`), so a pushed frame
computes one new position per layer.  A stream's first frame stands for its whole (edge-padded) history exactly
like `UnchunkedGenerator(pad, causal_shift=pad)` does (`common/generators.py:210-221`).

`DelayedStream` streams any (causal or non-causal) model of the drop-in classes at a fixed delay of
(receptive_field - 1) / 2 frames for a non-causal model (0 for a causal one), optionally with the test-time
augmentation every inference caller of the reference uses (UnchunkedGenerator(augment=True) and the un-flip and
average of main.py:314-318) inside the stream (C ABI `gast_stream_push_delayed`).

`WindowStream` is the generic form for any callable network: a device ring of the last `rf` input frames and one
window forward per pushed frame (what the reference does; used for non-GAST callables and as the cross-check).
"""
import ctypes as C
import numpy as np
import torch

from . import _lib as L


class CausalStream(object):
    """O(1)-per-frame lifting of `n_streams` concurrent streams with a causal model of the drop-in classes
    (`SpatioTemporalModelOptimized1f(causal=True)` as gen_skes.load_model_realtime builds it, or the dilated
    `SpatioTemporalModel(causal=True)`: the weights are interchangeable)."""

    def __init__(self, model_pos, n_streams, device=None):
        from . import engine
        if not getattr(model_pos, '_gast_causal', False):
            raise engine.GastError('CausalStream needs a causal model (gen_skes.py:59 builds it with causal=True)')
        if device is None:
            device = next(model_pos.parameters()).device
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise engine.GastError('CausalStream: the model must be on a CUDA device (there is no CPU path)')
        self.model = model_pos
        self.engine = engine
        self.rf = int(model_pos.receptive_field())
        self.n = int(n_streams)
        self.J = int(model_pos.num_joints_in)
        self.F = int(model_pos.in_features)
        self.step = 0
        self.fresh = torch.ones(self.n, dtype=torch.int32, device=self.device)     # every stream starts anew
        self._any_fresh = True
        self._state = None
        self._ws = None

    def reset(self, streams=None):
        """Forget the history of all (or the listed) streams: their next frame starts a new sequence."""
        if streams is None:
            self.fresh.fill_(1)
        else:
            self.fresh[torch.as_tensor(streams, device=self.device, dtype=torch.long)] = 1
        self._any_fresh = True

    def push(self, frame):
        """frame (n_streams, J, in_features): the newest 2D keypoints of every stream (normalised screen
        coordinates).  Returns the 3D pose of that frame, (n_streams, J, 3)."""
        eng = self.engine
        frame = torch.as_tensor(frame, dtype=torch.float32, device=self.device).contiguous()
        assert frame.shape == (self.n, self.J, self.F), frame.shape
        if self.model.training:
            raise eng.GastError('CausalStream: call .eval() on the model (streaming is inference)')
        h = eng.model_handle(self.model, self.device)
        lib = h.lib
        y = torch.empty((self.n, self.J, 3), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            h.refresh(self.model, st)
            if self._state is None:
                nb = lib.gast_stream_state_bytes(h.h, self.n)
                wb = lib.gast_stream_workspace_bytes(h.h, self.n)
                if nb == 0 or wb == 0:
                    raise eng.GastError('gast_stream_state_bytes: %s' % L.last_error())
                self._state = torch.empty(int(nb), dtype=torch.uint8, device=self.device)
                self._ws = torch.empty(int(wb), dtype=torch.uint8, device=self.device)
            fresh = self.fresh.data_ptr() if self._any_fresh else None
            rc = lib.gast_stream_push(h.h, C.c_void_p(self._state.data_ptr()), C.c_int64(self.step),
                                      C.c_void_p(frame.data_ptr()), C.c_void_p(y.data_ptr()), self.n,
                                      C.c_void_p(fresh), C.c_void_p(self._ws.data_ptr()), self._ws.numel(),
                                      C.c_void_p(st))
            if rc != 0:
                raise eng.GastError('gast_stream_push: %s' % L.last_error())
            if self._any_fresh:
                self.fresh.zero_()                       # (stream-ordered after the push that read it)
                self._any_fresh = False
        self.step += 1
        self.last_launches = int(lib.gast_last_launch_count(h.h))
        return y


class DelayIndex(object):
    """Host bookkeeping of a DelayedStream (no device needed): per stream, whether the next push starts a sequence
    (fresh), whether its sequence is over (hold: the last frame is repeated) and which frame of the current sequence
    the returned pose belongs to.  A push at position `pos` of a sequence (real frames and repeats alike) returns the
    pose of frame pos - delay; -1 when that lies before frame 0 or after the sequence's last real frame."""

    def __init__(self, n_streams, delay):
        self.n, self.delay = int(n_streams), int(delay)
        self.fresh = np.ones(self.n, dtype=bool)           # the next push starts a new sequence
        self.ended = np.zeros(self.n, dtype=bool)          # the sequence is over: pushes repeat its last frame
        self.pushed = np.zeros(self.n, dtype=np.int64)     # pushes since the sequence started
        self.real = np.zeros(self.n, dtype=np.int64)       # real frames of the sequence

    def reset(self, streams=None):
        sel = slice(None) if streams is None else np.asarray(list(streams), dtype=np.int64)
        self.fresh[sel] = True
        self.ended[sel] = False
        self.pushed[sel] = 0
        self.real[sel] = 0

    def save(self):
        return [a.copy() for a in (self.fresh, self.ended, self.pushed, self.real)]

    def restore(self, saved):
        self.fresh, self.ended, self.pushed, self.real = saved

    def step(self, ended=None):
        """Account for one push.  `ended`: streams whose sequence is over (from this push on).  Returns the fresh
        and hold masks of the push and the frame index of every returned pose."""
        now = np.zeros(self.n, dtype=bool)
        if ended is not None:
            now[np.asarray(list(ended), dtype=np.int64)] = True
        if (now & self.fresh).any():
            raise ValueError('DelayedStream: ended on stream(s) %s before their first frame'
                             % np.nonzero(now & self.fresh)[0].tolist())
        fresh = self.fresh.copy()
        hold = self.ended | now
        real = self.real + (~hold)
        idx = self.pushed - self.delay
        idx = np.where((idx >= 0) & (idx < real), idx, -1)
        self.pushed += 1
        self.real = real
        self.ended = hold
        self.fresh[:] = False
        return fresh, hold, idx


class DelayedStream(object):
    """O(1)-per-frame lifting of `n_streams` concurrent streams with ANY model of the drop-in classes, causal or not
    (`SpatioTemporalModel` or `SpatioTemporalModelOptimized1f`; not the dense ablation), optionally with test-time
    augmentation (`augment=True` and all four index lists, as UnchunkedGenerator(augment=True) and main.py:314-318
    take them).

    The pose a push returns is that of the frame pushed `delay` pushes earlier: `delay` = (receptive_field - 1) / 2
    for a non-causal model, 0 for a causal one.  A stream's sequence starts at its first frame after construction or
    `reset()` (the left edge padding of UnchunkedGenerator) and ends when `push(..., ended=[...])` lists it: from then
    on its last frame is repeated (the right edge padding), so `delay` more pushes return the sequence's last poses.
    Every returned pose is the reference's whole-sequence output for that frame."""

    def __init__(self, model_pos, n_streams, augment=False, kps_left=None, kps_right=None, joints_left=None,
                 joints_right=None, device=None):
        from . import engine
        if device is None:
            device = next(model_pos.parameters()).device
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise engine.GastError('DelayedStream: the model must be on a CUDA device (there is no CPU path)')
        lists = (kps_left, kps_right, joints_left, joints_right)
        if augment:
            if any(v is None for v in lists):
                raise engine.GastError('DelayedStream: augment=True needs kps_left, kps_right, joints_left and joints_right')
            if len(set(len(v) for v in lists)) != 1 or len(kps_left) == 0:
                raise engine.GastError('DelayedStream: the four index lists must have the same, non-zero length')
            self._sym = [(C.c_int32 * len(v))(*[int(i) for i in v]) for v in lists]
            self.n_sym = len(kps_left)
        else:
            self._sym = [None] * 4
            self.n_sym = 0
        self.augment = bool(augment)
        self.model = model_pos
        self.engine = engine
        self.n = int(n_streams)
        if self.n <= 0:
            raise engine.GastError('DelayedStream: n_streams must be positive')
        self.J = int(model_pos.num_joints_in)
        self.F = int(model_pos.in_features)
        h = engine.model_handle(model_pos, self.device)
        self.delay = int(h.lib.gast_stream_delay(h.h))
        if self.delay < 0:
            raise engine.GastError('DelayedStream: %s' % L.last_error())
        self.index = DelayIndex(self.n, self.delay)
        self.step = 0
        self._state = None
        self._ws = None
        self._blank = None

    def reset(self, streams=None):
        """Forget the history of all (or the listed) streams: their next frame starts a new sequence.  Poses of the
        old sequence that were still `delay` pushes away are not returned."""
        self.index.reset(streams)

    def push(self, frame, ended=None):
        """frame (n_streams, J, in_features): the newest 2D keypoints of every stream (normalised screen coordinates);
        the rows of ended streams are ignored (frame may be None when every stream has ended).  ended: streams whose
        sequence is over, from this push on.  Returns (poses (n_streams, J, 3) on the device, frame_index (n_streams,)
        int64 numpy): frame_index[b] is the frame of stream b's current sequence the pose belongs to, -1 if none."""
        eng = self.engine
        if self.model.training:
            raise eng.GastError('DelayedStream: call .eval() on the model (streaming is inference)')
        saved = self.index.save()
        try:
            y, idx = self._push(frame, ended)
        except Exception:
            self.index.restore(saved)                        # a refused push changes nothing
            raise
        return y, idx

    def _push(self, frame, ended):
        eng = self.engine
        try:
            fresh, hold, idx = self.index.step(ended)
        except ValueError as e:
            raise eng.GastError(str(e))
        if frame is None:
            if not hold.all():
                raise eng.GastError('DelayedStream: frame may only be None when every stream has ended')
            if self._blank is None:
                self._blank = torch.zeros((self.n, self.J, self.F), dtype=torch.float32, device=self.device)
            frame = self._blank
        frame = torch.as_tensor(frame, dtype=torch.float32, device=self.device).contiguous()
        assert frame.shape == (self.n, self.J, self.F), frame.shape
        h = eng.model_handle(self.model, self.device)
        lib = h.lib
        y = torch.empty((self.n, self.J, 3), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            h.refresh(self.model, st)
            aug = 1 if self.augment else 0
            if self._state is None:
                nb = lib.gast_stream_delayed_state_bytes(h.h, self.n, aug)
                wb = lib.gast_stream_delayed_workspace_bytes(h.h, self.n, aug)
                if nb == 0 or wb == 0:
                    raise eng.GastError('gast_stream_delayed_state_bytes: %s' % L.last_error())
                self._state = torch.empty(int(nb), dtype=torch.uint8, device=self.device)
                self._ws = torch.empty(int(wb), dtype=torch.uint8, device=self.device)
            masks = []
            for m in (fresh, hold):
                masks.append(torch.from_numpy(m.astype(np.int32)).to(self.device) if m.any() else None)
            ptr = [C.c_void_p(t.data_ptr() if t is not None else None) for t in masks]
            rc = lib.gast_stream_push_delayed(h.h, C.c_void_p(self._state.data_ptr()), self._state.numel(),
                                              C.c_int64(self.step), C.c_void_p(frame.data_ptr()),
                                              C.c_void_p(y.data_ptr()), self.n, ptr[0], ptr[1], self.n_sym,
                                              *self._sym, C.c_void_p(self._ws.data_ptr()), self._ws.numel(),
                                              C.c_void_p(st))
            if rc != 0:
                raise eng.GastError('gast_stream_push_delayed: %s' % L.last_error())
        self.step += 1
        self.last_launches = int(lib.gast_last_launch_count(h.h))
        return y, idx

    def drain(self):
        """`delay` pushes with every stream ended: the poses still owed, (delay, n_streams, J, 3) on the device, and
        their frame indices (delay, n_streams).  What finishing one video needs."""
        ys, idx = [], []
        for _ in range(self.delay):
            y, i = self.push(None, ended=range(self.n))
            ys.append(y)
            idx.append(i)
        if not ys:
            return (torch.empty((0, self.n, self.J, 3), dtype=torch.float32, device=self.device),
                    np.zeros((0, self.n), dtype=np.int64))
        return torch.stack(ys), np.stack(idx)


class WindowStream(object):
    """Generic frame-by-frame driver for any window network `net((n, rf, J, F)) -> (n, T_out, J, 3)`: keeps the last
    `rf` frames of `n_streams` streams in one device tensor used as a ring and runs one window forward per pushed
    frame (O(rf) per frame, as the reference's real-time loop does)."""

    def __init__(self, net, n_streams, device=None):
        self.model = net
        self.rf = int(net.receptive_field())
        if device is None:
            device = next(net.parameters()).device
        self.device = torch.device(device)
        self.n = int(n_streams)
        self.J = int(net.num_joints_in)
        self.F = int(net.in_features)
        # ring[:, (head + k) % rf] is the k-th oldest frame of the window; `window` is its unrolled copy
        self.ring = torch.zeros((self.n, self.rf, self.J, self.F), dtype=torch.float32, device=self.device)
        self.window = torch.empty_like(self.ring)
        self.head = 0
        self.started = torch.zeros(self.n, dtype=torch.bool, device=self.device)

    def reset(self, streams=None):
        if streams is None:
            self.started.zero_()
        else:
            self.started[torch.as_tensor(streams, device=self.device)] = False

    def push(self, frame):
        frame = torch.as_tensor(frame, dtype=torch.float32, device=self.device)
        assert frame.shape == (self.n, self.J, self.F), frame.shape
        fresh = ~self.started
        if bool(fresh.any()):
            # a stream's first frame fills its whole window: the edge padding of generators.py:217-221
            self.ring[fresh] = frame[fresh].unsqueeze(1)
            self.started |= fresh
        self.ring[:, self.head] = frame                      # overwrite the oldest slot
        self.head = (self.head + 1) % self.rf
        k = self.rf - self.head                              # unroll: oldest frame first, newest last
        self.window[:, :k] = self.ring[:, self.head:]
        self.window[:, k:] = self.ring[:, :self.head]
        with torch.no_grad():
            return self.model(self.window)[:, -1]
