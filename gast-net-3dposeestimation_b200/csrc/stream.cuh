// O(1)-per-frame causal streaming of the lifting network (SURVEY.md §8f N4; the reference's real-time path is a
// causal SpatioTemporalModelOptimized1f re-run on the last `receptive_field` frames for every new frame,
// gen_skes.py:43-69, tools/inference.py:19-110).  Included by gast_api.cu (uses its helpers).
//
// In the causal network every temporal stage i (filter width w_i, dilation d_i = w_0 ... w_{i-1}) maps its input
// sequence G_{i-1} to   S_i[t] = G_{i-1}[t] + f(G_{i-1}[t - (w_i-1) d_i], ..., G_{i-1}[t - d_i], G_{i-1}[t])
// (gast_net.py:139-143,167-174: with causal_shift = pad the residual slice and the last tap are both the newest
// position), and the blocks are pointwise in time.  So a pushed frame needs ONE new position per layer, given the
// layer inputs of the past: per stage a ring of R_i = w_i d_i slots holding G_{i-1}, slot = frame index mod R_i.
//
// Layout: rings are SLOT-major, ring_i[slot][stream][joint][channel], so that
//   * a slot is an ordinary contiguous (n_streams*J, C) activation matrix: the producing block writes it directly;
//   * the taps of stage i sit d_i slots apart: slots p, p + d_i, ..., p + (w_i-1) d_i with p = slot mod d_i -- a
//     fixed-stride gather, i.e. exactly the tap addressing the GEMM kernels already have (tap_stride), TMA-able.
// The taps appear in slot order, which is a ROTATION of time order (by r = slot div d_i): instead of moving data the
// stage's folded weights exist in w_i tap-rotated copies and the push picks copy r.  No activation is ever shifted.
//
// A stream's first frame replaces its whole history by copies of that frame (the edge padding of
// UnchunkedGenerator(pad, causal_shift = pad), common/generators.py:210-221).  With a constant history every layer
// input is constant in time, so it is enough to copy the freshly computed slot of each ring to the ring's other
// slots for those streams (stream_fill_fresh_kernel) before the stage reads its taps.
//
// Non-causal models stream the same way, `delay` = sum_i (pad_i - causal_shift_i) = (rf-1)/2 frames late
// (gast_stream_push_delayed).  Stage i reads the same w_i taps; only its residual moves: it is G_{i-1} at the
// position lag_i = pad_i - causal_shift_i behind the newest (the middle tap; lag_i = 0 for a causal model), i.e. slot
// (step - lag_i) mod R_i, still in the ring because lag_i < R_i.  The left edge is the same fresh fill; the right
// edge (UnchunkedGenerator's edge padding by `delay` copies of the last frame) is a `hold` push that repeats the
// stream's newest input frame.  With test-time augmentation the mirrored twin of stream b is stream row n + b of the
// same rings (2n rows, written by the same input push), and the shrink merges the two (stream_shrink_merge_kernel).
#pragma once

namespace gast {

// xhist (n, k0, J, F): the last k0 input frames of every stream, oldest first.  One thread per (stream, joint, feature).
__global__ void stream_xpush_kernel(float* __restrict__ xhist, const float* __restrict__ x,
                                    const int32_t* __restrict__ fresh, int n, int k0, int JF) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * JF) return;
  const int b = idx / JF, e = idx - b * JF;
  float* hrow = xhist + (long long)b * k0 * JF + e;
  const float v = x[idx];
  if (fresh && fresh[b]) {
    for (int k = 0; k < k0; ++k) hrow[(long long)k * JF] = v;
  } else {
    for (int k = 0; k + 1 < k0; ++k) hrow[(long long)k * JF] = hrow[(long long)(k + 1) * JF];
    hrow[(long long)(k0 - 1) * JF] = v;
  }
}

__device__ __forceinline__ void stream_hist_push(float* hrow, float v, bool fresh, int k0, int JF) {
  if (fresh) {
    for (int k = 0; k < k0; ++k) hrow[(long long)k * JF] = v;
  } else {
    for (int k = 0; k + 1 < k0; ++k) hrow[(long long)k * JF] = hrow[(long long)(k + 1) * JF];
    hrow[(long long)(k0 - 1) * JF] = v;
  }
}

// stream_xpush_kernel with right-edge holds and the mirrored twin.  xhist (rows, k0, J, F), rows = n, or 2n with the
// twin of stream b in row n + b.  One thread per (stream b < n, joint, feature).
//   hold[b] != 0 (and not fresh): repeat the stream's newest history frame instead of reading x (the edge padding on
//   the right, common/generators.py:217-221); fresh takes precedence.
//   twin: row n + b receives the mirrored frame, feature 0 negated and joint j read from perm[j] (tta_prepare_kernel).
__global__ void stream_xpush_hold_kernel(float* __restrict__ xhist, const float* __restrict__ x,
                                         const int32_t* __restrict__ fresh, const int32_t* __restrict__ hold, int n,
                                         int k0, int J, int F, int twin, JointPerm perm) {
  const int JF = J * F;
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * JF) return;
  const int b = idx / JF, e = idx - b * JF, j = e / F, c = e - j * F;
  const bool fr = fresh && fresh[b];
  const bool hd = !fr && hold && hold[b];
  float* hrow = xhist + (long long)b * k0 * JF + e;
  stream_hist_push(hrow, hd ? hrow[(long long)(k0 - 1) * JF] : x[idx], fr, k0, JF);
  if (twin) {
    float* trow = xhist + (long long)(n + b) * k0 * JF + e;
    float w;
    if (hd) {
      w = trow[(long long)(k0 - 1) * JF];
    } else {
      w = x[(long long)b * JF + perm.p[j] * F + c];
      if (c == 0) w = -w;
    }
    stream_hist_push(trow, w, fr, k0, JF);
  }
}

// ring (R, rows, rowlen): for every fresh stream copy its row block of slot `src` to every other slot.
// grid = (rows, chunks of the row block); row b belongs to stream b % nf (nf = n: rows n..2n-1 are the twins).
// A block whose stream is not fresh exits at once.
__global__ void stream_fill_fresh_kernel(float* __restrict__ ring, int R, int src, int n, long long rowlen,
                                         const int32_t* __restrict__ fresh, int nf) {
  const int b = blockIdx.x;
  if (!fresh[b % nf]) return;
  const long long slot_stride = (long long)n * rowlen;
  const float4* s = reinterpret_cast<const float4*>(ring + (long long)src * slot_stride + (long long)b * rowlen);
  const long long n4 = rowlen >> 2;
  for (long long i = (long long)blockIdx.y * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.y * blockDim.x) {
    const float4 v = s[i];
    for (int r = 0; r < R; ++r)
      if (r != src) reinterpret_cast<float4*>(ring + (long long)r * slot_stride + (long long)b * rowlen)[i] = v;
  }
}

// dst[n][k*Cw + c] = src[n][j*Cw + c],  j = (k - r - 1) mod taps: slot order -> time order of the taps
__global__ void rotate_taps_kernel(float* __restrict__ dst, const float* __restrict__ src, int N, int Cw, int taps, int r) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long K = (long long)taps * Cw;
  if (idx >= (long long)N * K) return;
  const long long nrow = idx / K;
  const int kc = (int)(idx - nrow * K);
  const int k = kc / Cw, c = kc - k * Cw;
  const int j = ((k - r - 1) % taps + taps) % taps;
  dst[idx] = src[nrow * K + (long long)j * Cw + c];
}

// shrink (shrink_kernel) of stream row b at joint j and of its twin row n + b at joint perm[j], merged in the epilogue
// as tta_merge_kernel does: y[b][j] = (y0 + unflip(y1)) / 2.  One warp per output row (b, j); the per-lane FMA order
// and the warp sums are shrink_kernel's, so the result is bitwise shrink_kernel followed by tta_merge_kernel.
__global__ void stream_shrink_merge_kernel(const float* __restrict__ X, int ldx, const float* __restrict__ Ws,
                                           float* __restrict__ y, int n, int J, int K, JointPerm perm) {
  long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= (long long)n * J) return;
  const int b = (int)(row / J), j = (int)(row - (long long)b * J);
  const float* xr = X + row * ldx;
  const float* xt = X + ((long long)(n + b) * J + perm.p[j]) * ldx;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, c0 = 0.f, c1 = 0.f, c2 = 0.f;
  for (int k = lane * 4; k < K; k += 128) {
    float4 w0 = ldg4(Ws + k), w1 = ldg4(Ws + K + k), w2 = ldg4(Ws + 2 * K + k);
    float4 xv = ldg4(xr + k);
    a0 = fmaf(xv.x, w0.x, fmaf(xv.y, w0.y, fmaf(xv.z, w0.z, fmaf(xv.w, w0.w, a0))));
    a1 = fmaf(xv.x, w1.x, fmaf(xv.y, w1.y, fmaf(xv.z, w1.z, fmaf(xv.w, w1.w, a1))));
    a2 = fmaf(xv.x, w2.x, fmaf(xv.y, w2.y, fmaf(xv.z, w2.z, fmaf(xv.w, w2.w, a2))));
    float4 tv = ldg4(xt + k);
    c0 = fmaf(tv.x, w0.x, fmaf(tv.y, w0.y, fmaf(tv.z, w0.z, fmaf(tv.w, w0.w, c0))));
    c1 = fmaf(tv.x, w1.x, fmaf(tv.y, w1.y, fmaf(tv.z, w1.z, fmaf(tv.w, w1.w, c1))));
    c2 = fmaf(tv.x, w2.x, fmaf(tv.y, w2.y, fmaf(tv.z, w2.z, fmaf(tv.w, w2.w, c2))));
  }
  a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2);
  c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2);
  if (lane == 0) {
    y[row * 3 + 0] = (a0 + (-c0)) / 2.0f;
    y[row * 3 + 1] = (a1 + c1) / 2.0f;
    y[row * 3 + 2] = (a2 + c2) / 2.0f;
  }
}

}  // namespace gast

struct StreamPlan {
  int n = 0;                            // rows of the rings: n_streams, or 2 n_streams with the mirrored twins
  std::vector<int> dil, R;              // per stage (index i-1): dilation d_i, ring slots R_i = w_i d_i
  std::vector<size_t> ring_off;         // float offsets into the state
  size_t xhist_off = 0, state_floats = 0;
};

// delayed = 0: gast_stream_push (causal models only); 1: gast_stream_push_delayed (causal or not)
static int stream_check(const gast_handle* h, bool delayed = false) {
  if (h->cfg.kind != GAST_KIND_MODEL) return fail("streaming is implemented for the MODEL kind only");
  if (h->cfg.dense) return fail("the dense ablation has no streaming form");
  if (!delayed && !h->cfg.causal)
    return fail("streaming needs a causal model (gen_skes.py:59: causal=True): a non-causal network "
                "has no output for the newest frame (gast_stream_push_delayed streams it with a delay)");
  return 0;
}

static int stream_plan(const gast_handle* h, int n, StreamPlan* sp, bool delayed = false) {
  if (stream_check(h, delayed)) return 1;
  if (n <= 0) return fail("streaming: n_streams must be positive");
  const gast_cfg& c = h->cfg;
  const int J = c.num_joints, L = c.num_stages;
  sp->n = n;
  size_t off = 0;
  auto take = [&](size_t nf) { size_t o = off; off += (nf + 63) & ~(size_t)63; return o; };
  sp->xhist_off = take((size_t)n * c.filter_widths[0] * J * c.in_features);
  int d = c.filter_widths[0];
  for (int i = 1; i < L; ++i) {
    const int fw = c.filter_widths[i], Cw = c.channels << i;
    sp->dil.push_back(d);
    sp->R.push_back(fw * d);
    sp->ring_off.push_back(take((size_t)fw * d * n * J * Cw));
    d *= fw;
  }
  sp->state_floats = off;
  return 0;
}

extern "C" size_t gast_stream_state_bytes(gast_t* h, int32_t n_streams) {
  if (!h) return 0;
  StreamPlan sp;
  if (stream_plan(h, n_streams, &sp)) return 0;
  return sp.state_floats * sizeof(float) + 256;
}

struct StreamBufs { float *E, *tmp, *act, *fin; BlockBufs bb; };

static void stream_bufs(const gast_handle* h, int n, Arena& a, StreamBufs* sb) {
  const int J = h->cfg.num_joints, C = h->cfg.channels, L = h->cfg.num_stages;
  const size_t rows = (size_t)n * J;
  const int Cmax = C << (L - 1);                 // widest block input
  sb->E = a.take(rows * C);
  sb->tmp = a.take(rows * Cmax);
  sb->act = a.take(rows * Cmax);
  sb->fin = a.take(rows * 2 * Cmax);
  sb->bb.XY = a.take(rows * 2 * Cmax); sb->bb.L = a.take(rows * Cmax); sb->bb.AB = a.take(rows * 8);
  sb->bb.Y = a.take(rows * Cmax); sb->bb.Gl = a.take(rows * Cmax);
}

static size_t stream_ws_bytes(const gast_handle* h, int n) {
  Arena a{nullptr, 0, 0, true};
  StreamBufs sb;
  stream_bufs(h, n, a, &sb);
  return a.off + 256;
}

extern "C" size_t gast_stream_workspace_bytes(gast_t* h, int32_t n_streams) {
  if (!h || stream_check(h) || n_streams <= 0) return 0;
  return stream_ws_bytes(h, n_streams);
}

// tap-rotated copies of the folded temporal-conv weights (+ their tcgen05 splits); rebuilt after every gast_prepare
static int stream_prepare(gast_handle* h, cudaStream_t st) {
  for (size_t i = 0; i < h->stages.size(); ++i) {
    StageConsts& s = h->stages[i];
    const int fw = h->cfg.filter_widths[i + 1];
    if (s.taps != fw) return fail("streaming: stage %zu has %d taps, expected %d", i, s.taps, fw);
    if ((int)s.Wrot.size() != fw) {
      s.Wrot.assign(fw, nullptr);
      s.tc_rot.assign(fw, TcWeights());
      for (int r = 0; r < fw; ++r)
        if (dalloc(h, &s.Wrot[r], (size_t)s.Cw * fw * s.Cw)) return 1;
    }
    const long long tot = (long long)s.Cw * fw * s.Cw;
    for (int r = 0; r < fw; ++r) {
      rotate_taps_kernel<<<cdiv(tot, 256), 256, 0, st>>>(s.Wrot[r], s.Wt, s.Cw, s.Cw, fw, r);
      if (prep_one_tc(h, st, s.tc_rot[r], s.Wrot[r], s.Cw, fw * s.Cw, 0)) return 1;
    }
  }
  CUDA_OK(cudaGetLastError());
  h->stream_ready = true;
  return 0;
}

// What distinguishes gast_stream_push_delayed from gast_stream_push (which leaves every field at its default).
struct StreamExtras {
  bool centre_residual = false;        // residual lag_i = pad_i (non-causal model) instead of 0
  const int32_t* hold = nullptr;       // device (n): repeat the newest input frame (right edge)
  bool twin = false;                   // mirrored twin in rows n..2n-1, merged by the shrink
  JointPerm kperm, jperm;              // input keypoint / output joint partners of the twin
};

// The push of one frame of every stream (both entry points).  `sp` is planned for the ring rows (n, or 2n with the
// twin); x and y are (n, J, F) and (n, J, 3).
static int stream_push_impl(gast_handle* h, const StreamPlan& sp, void* state, int64_t step, const float* x, float* y,
                            int n, const int32_t* fresh, const StreamExtras& ex, void* workspace, size_t workspace_bytes,
                            cudaStream_t st) {
  CUDA_OK(cudaSetDevice(h->cfg.device));
  if (!h->stream_ready && stream_prepare(h, st)) return 1;
  const int N = sp.n;                  // rows of the rings
  const size_t need = stream_ws_bytes(h, N);
  if (!workspace || workspace_bytes < need)
    return fail("stream push: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
  h->launches = 0; h->tc_launches = 0; h->ev_used = 0; h->ev_kind.clear();
  const gast_cfg& c = h->cfg;
  const int J = c.num_joints, C = c.channels, L = c.num_stages, k0 = c.filter_widths[0], Fin = c.in_features;
  float* sbase = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(state) + 255) & ~(uintptr_t)255);
  uintptr_t wsb = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
  Arena a{reinterpret_cast<char*>(wsb), workspace_bytes, 0, false};
  StreamBufs sb;
  stream_bufs(h, N, a, &sb);
  const long long rows = (long long)N * J;
  if (k0 * Fin > EXP_MAXKF) return fail("expand: filter_width*in_features > %d unsupported", EXP_MAXKF);
  // input history + expand (gast_net.py:163-164) on the last k0 frames
  float* xhist = sbase + sp.xhist_off;
  if (ex.hold || ex.twin)
    stream_xpush_hold_kernel<<<cdiv((long long)n * J * Fin, 256), 256, 0, st>>>(xhist, x, fresh, ex.hold, n, k0, J, Fin,
                                                                               ex.twin ? 1 : 0, ex.kperm);
  else
    stream_xpush_kernel<<<cdiv((long long)n * J * Fin, 256), 256, 0, st>>>(xhist, x, fresh, n, k0, J * Fin);
  h->launches++;
  {
    long long thr = ((rows + EXP_ROWS - 1) / EXP_ROWS) * (C / 4);
    if (k0 * Fin <= 6)
      expand_kernel<6><<<cdiv(thr, 256), 256, 0, st>>>(xhist, h->We, h->be, sb.E, rows, J, k0, 1, 1, k0, Fin, C);
    else
      expand_kernel<EXP_MAXKF><<<cdiv(thr, 256), 256, 0, st>>>(xhist, h->We, h->be, sb.E, rows, J, k0, 1, 1, k0, Fin, C);
    h->launches++;
  }
  auto slot_ptr = [&](int i /*stage 1..L-1*/) {
    const int R = sp.R[i - 1], Cw = C << i;
    return sbase + sp.ring_off[i - 1] + (size_t)(step % R) * N * J * Cw;
  };
  float* bout = (L > 1) ? slot_ptr(1) : sb.fin;
  if (run_block(h, st, h->blocks[0], sb.E, N, sb.bb, bout)) return 1;
  for (int i = 1; i < L; ++i) {
    StageConsts& s = h->stages[i - 1];
    const int Cw = s.Cw, fw = c.filter_widths[i], d = sp.dil[i - 1], R = sp.R[i - 1];
    float* ring = sbase + sp.ring_off[i - 1];
    const int hs = (int)(step % R);
    const long long slot_floats = (long long)N * J * Cw;
    if (fresh) {
      dim3 g((unsigned)N, (unsigned)std::max<long long>(1, std::min<long long>(8, (long long)J * Cw / 4 / 256)));
      stream_fill_fresh_kernel<<<g, 256, 0, st>>>(ring, R, hs, N, (long long)J * Cw, fresh, n);
      h->launches++;
    }
    const int p0 = hs % d, r = hs / d;
    // temporal conv + BN + ReLU: taps = slots p0 + k d, weights rotated to slot order (gast_net.py:173)
    GemmP p;
    gemm_defaults(p, h, N);
    p.nseg = 1;
    p.seg[0].base = ring + (long long)p0 * slot_floats; p.seg[0].ld = Cw; p.seg[0].K = fw * Cw; p.seg[0].Kc = Cw;
    p.seg[0].tap_stride = (long long)d * slot_floats;
    p.seg[0].map = RowMap{N, N, 1, 0};
    p.W = s.Wrot[r]; p.ldw = fw * Cw; p.N = Cw; p.out = sb.tmp; p.ld_out = Cw; p.bias = s.bt; p.relu = 1;
    if (launch_gemm(h, st, EPI_PLAIN, p, &s.tc_rot[r])) return 1;
    // 1x1 conv + BN + ReLU + residual (gast_net.py:170,174): G_{i-1} lag_i = pad_i - causal_shift_i positions behind
    // the newest, slot (step - lag_i) mod R_i: the newest slot for a causal model, the middle tap otherwise
    const int lag = ex.centre_residual ? (fw - 1) * d / 2 : 0;
    const int rs = (int)(((step - lag) % R + R) % R);
    gemm_defaults(p, h, N);
    p.nseg = 1; p.seg[0] = seg_flat(sb.tmp, Cw, Cw);
    p.W = s.W1; p.ldw = Cw; p.N = Cw; p.out = sb.act; p.ld_out = Cw; p.bias = s.b1; p.relu = 1;
    p.res = ring + (long long)rs * slot_floats; p.res_ld = Cw; p.res_map = RowMap{N, N, 1, 0};
    if (launch_gemm(h, st, EPI_PLAIN, p, &s.tc_1)) return 1;
    bout = (i < L - 1) ? slot_ptr(i + 1) : sb.fin;
    if (run_block(h, st, h->blocks[i], sb.act, N, sb.bb, bout)) return 1;
  }
  {
    Lookup Lk{h};
    const int Cl = C << L;
    const float* ws = Lk.get("shrink.weight", (int64_t)3 * Cl);
    if (!Lk.ok) return 1;
    if (ex.twin)
      stream_shrink_merge_kernel<<<cdiv((long long)n * J * 32, 256), 256, 0, st>>>(bout, Cl, ws, y, n, J, Cl, ex.jperm);
    else
      shrink_kernel<<<cdiv(rows * 32, 256), 256, 0, st>>>(bout, Cl, ws, y, rows, Cl);
    h->launches++;
  }
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" int gast_stream_push(gast_t* h, void* state, int64_t step, const float* x, float* y, int32_t n_streams,
                                const int32_t* fresh, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return fail("gast_stream_push: null handle");
  if (!h->prepared) return fail("gast_stream_push: gast_prepare() has not run since the last gast_bind()");
  if (step < 0 || !state || !x || !y) return fail("gast_stream_push: bad arguments");
  StreamPlan sp;
  if (stream_plan(h, n_streams, &sp)) return 1;
  return stream_push_impl(h, sp, state, step, x, y, n_streams, fresh, StreamExtras(), workspace, workspace_bytes,
                          reinterpret_cast<cudaStream_t>(stream));
}

// ---- delayed streaming (causal and non-causal models, optional test-time augmentation) ----
extern "C" int32_t gast_stream_delay(gast_t* h) {
  if (!h || stream_check(h, true)) return -1;
  if (h->cfg.causal) return 0;
  int rf = 1;
  for (int i = 0; i < h->cfg.num_stages; ++i) rf *= h->cfg.filter_widths[i];
  return (rf - 1) / 2;                 // sum_i pad_i, causal_shift_i = 0
}

extern "C" size_t gast_stream_delayed_state_bytes(gast_t* h, int32_t n_streams, int32_t augment) {
  if (!h || n_streams <= 0) return 0;
  StreamPlan sp;
  if (stream_plan(h, augment ? 2 * n_streams : n_streams, &sp, true)) return 0;
  return sp.state_floats * sizeof(float) + 256;
}

extern "C" size_t gast_stream_delayed_workspace_bytes(gast_t* h, int32_t n_streams, int32_t augment) {
  if (!h || stream_check(h, true) || n_streams <= 0) return 0;
  return stream_ws_bytes(h, augment ? 2 * n_streams : n_streams);
}

extern "C" int gast_stream_push_delayed(gast_t* h, void* state, size_t state_bytes, int64_t step, const float* x,
                                        float* y, int32_t n_streams, const int32_t* fresh, const int32_t* hold,
                                        int32_t n_sym, const int32_t* kps_left, const int32_t* kps_right,
                                        const int32_t* joints_left, const int32_t* joints_right, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  if (!h) return fail("gast_stream_push_delayed: null handle");
  if (!h->prepared) return fail("gast_stream_push_delayed: gast_prepare() has not run since the last gast_bind()");
  if (step < 0 || !state || !x || !y || n_sym < 0) return fail("gast_stream_push_delayed: bad arguments");
  if (n_sym > 0 && (!kps_left || !kps_right || !joints_left || !joints_right))
    return fail("gast_stream_push_delayed: augmentation needs kps_left, kps_right, joints_left and joints_right");
  StreamExtras ex;
  ex.twin = n_sym > 0;
  if (ex.twin) {
    if (make_perm(h->cfg.num_joints, n_sym, kps_left, kps_right, &ex.kperm)) return 1;
    if (make_perm(h->cfg.num_joints, n_sym, joints_left, joints_right, &ex.jperm)) return 1;
  }
  StreamPlan sp;
  if (stream_plan(h, ex.twin ? 2 * n_streams : n_streams, &sp, true)) return 1;
  const size_t need = sp.state_floats * sizeof(float) + 256;
  if (state_bytes < need)
    return fail("gast_stream_push_delayed: state too small (%zu < %zu bytes for %d streams%s)", state_bytes, need,
                n_streams, ex.twin ? " with augmentation" : "");
  ex.centre_residual = !h->cfg.causal;
  ex.hold = hold;
  return stream_push_impl(h, sp, state, step, x, y, n_streams, fresh, ex, workspace, workspace_bytes,
                          reinterpret_cast<cudaStream_t>(stream));
}
