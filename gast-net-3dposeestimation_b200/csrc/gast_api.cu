// libgast_b200: C ABI (include/gast_b200.h) + launch planning of the GAST-Net lifting path.
//
// Layout: every activation is channels-last, rows = (clip, frame, joint), fp32.  The
// reference's (B,C,T,N) <-> (B,T,N,C) permutes (gast_net.py:24,31,162; local_attention.py:136,149;
// global_attention.py:109,114,121,128) therefore vanish.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/gast_b200.h"
#include "gast_common.cuh"
#include "gemm_ffma.cuh"
#include "kernels_misc.cuh"
#include "gemm_tc.cuh"
#include "kernels_hbm.cuh"
#include "train_kernels.cuh"
#include "train_state.cuh"

using namespace gast;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";

static int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}

#define CUDA_OK(expr)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

extern "C" const char* gast_last_error(void) { return g_err; }
extern "C" const char* gast_version(void) {
  static const bool f16 = !(getenv("GAST_TC_F16") && atoi(getenv("GAST_TC_F16")) == 0);
  return f16 ? "gast_b200 0.3 (sm_100a; tcgen05 fp16 hi+lo for K >= 256, tf32 + bf16-corr below)"
             : "gast_b200 0.3 (sm_100a; tcgen05 tf32 + bf16-corr)";
}

// ------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------
struct Binding {
  void* ptr;
  int64_t numel;
};

struct BlockConsts {   // derived, eval mode; all device pointers owned by the handle
  int C = 0;           // input width
  int Cout = 0;        // SemCH out width (== C inside a block)
  int heads = 0, Cg = 0;
  int tpm = 0;         // 64-channel tiles per mask
  float *Wloc = nullptr, *coef[2] = {nullptr, nullptr}, *shift_loc = nullptr;
  float *Wlc = nullptr, *blc = nullptr;
  float *Wg = nullptr, *bg = nullptr, *U = nullptr, *cab = nullptr, *Ck = nullptr;
  float *Wgc = nullptr, *bgc = nullptr;
  float *Wbc = nullptr, *bbc = nullptr;
  TcWeights tc_loc, tc_lc, tc_g, tc_gc, tc_bc;   // hi/lo split copies for the tcgen05 core
};

struct StageConsts {
  int Cw = 0, taps = 0, stride = 1, dil = 1;
  float *Wt = nullptr, *bt = nullptr, *W1 = nullptr, *b1 = nullptr;
  TcWeights tc_t, tc_1;
  std::vector<float*> Wrot;          // streaming (stream.cuh): tap-rotated copies of Wt, one per rotation
  std::vector<TcWeights> tc_rot;
};

struct gast_handle {
  gast_cfg cfg;
  std::vector<int32_t> sym_r, sym_c, con_r, con_c;
  NbrTable nbr[2];
  int nnz[2] = {0, 0};
  std::unordered_map<std::string, Binding> bound;
  std::unordered_map<std::string, Binding> grads;   // gradient outputs by state_dict key (training)
  // saved-for-backward state of the training forwards still waiting for their backward, keyed by the
  // caller's workspace (which holds the saved activations): several forwards may be outstanding
  // (micro-batches summed before .backward(), a logging forward under no_grad in between)
  std::vector<std::pair<void*, TrainState>> trains;
  std::vector<void*> owned;          // cudaMalloc'ed derived buffers
  std::vector<BlockConsts> blocks;
  std::vector<StageConsts> stages;
  std::vector<int> pad, shift;       // gast_net.py:57,136-143
  float *We = nullptr, *be = nullptr;
  bool prepared = false;
  bool stream_ready = false;         // tap-rotated stage weights match the current parameters
  unsigned long long* dropout_state = nullptr;   // caller-owned device counter added to the dropout seed (graph replays)
  int launches = 0;
  int tc_launches = 0;
  int gemm_core = 0;                 // 0 auto (tcgen05 where possible), 1 force FFMA
  // training: per-GEMM tcgen05 operand copies (3xTF32), indexed by the GEMM's position in the step (train.cuh)
  std::vector<TcWeights> train_tc;
  bool train_tc_on = true;
  int block1_slabs = 1;              // clip slabs of the expand stage + first block (GAST_BLOCK1_SLABS)
  // optional per-launch device timing (bench.py roofline): event pairs around every launch
  bool timing = false;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<int> ev_kind;          // kind per recorded launch
  size_t ev_used = 0;
  int fpt = 0;
  int sm_count = 148;
  float* loss_scratch = nullptr;   // shrink+mpjpe: SHL_MAXBLOCKS double partials | ticket (zero-initialised, reset by the kernel)
};

constexpr int GAST_MAX_PENDING_TRAIN = 16;   // training forwards that may wait for their backward per handle

enum { LK_EXPAND = 0, LK_GEMM_PLAIN = 1, LK_GEMM_SEMCH = 2, LK_GEMM_GLOBAL = 3, LK_ROWDOT = 4, LK_SHRINK = 5,
       LK_TC_PLAIN = 6, LK_TC_SEMCH = 7, LK_TC_GLOBAL = 8, LK_GLOBAL_MIX = 9 };

struct TimedLaunch {   // RAII: event pair around one launch when timing is on
  gast_handle* h; cudaStream_t st; bool on;
  TimedLaunch(gast_handle* h_, cudaStream_t st_, int kind) : h(h_), st(st_), on(h_->timing) {
    if (!on) return;
    while (h->ev_pool.size() < h->ev_used + 2) {
      cudaEvent_t e; cudaEventCreate(&e); h->ev_pool.push_back(e);
    }
    h->ev_kind.push_back(kind);
    cudaEventRecord(h->ev_pool[h->ev_used], st);
  }
  ~TimedLaunch() {
    if (!on) return;
    cudaEventRecord(h->ev_pool[h->ev_used + 1], st);
    h->ev_used += 2;
  }
};

static int dalloc(gast_handle* h, float** p, size_t nfloats) {
  void* q = nullptr;
  CUDA_OK(cudaMalloc(&q, (nfloats ? nfloats : 1) * sizeof(float)));
  CUDA_OK(cudaMemset(q, 0, (nfloats ? nfloats : 1) * sizeof(float)));
  h->owned.push_back(q);
  *p = reinterpret_cast<float*>(q);
  return 0;
}

static int build_nbr(const std::vector<int32_t>& r, const std::vector<int32_t>& c, int J, NbrTable* t) {
  if (J > 32 || r.size() > 160) return fail("mask too large (J=%d nnz=%zu)", J, r.size());
  memset(t, 0, sizeof(*t));
  int z = 0;
  for (int i = 0; i < J; ++i) {
    t->row_ptr[i] = (unsigned char)z;
    while (z < (int)r.size() && r[z] == i) {
      if (z > 0 && r[z - 1] == i && c[z - 1] >= c[z]) return fail("mask nonzeros not in row-major order");
      t->col[z] = (unsigned char)c[z];
      ++z;
    }
    if (z == t->row_ptr[i]) return fail("mask row %d is empty (softmax over nothing)", i);
  }
  if (z != (int)r.size()) return fail("mask nonzeros not in row-major order");
  t->row_ptr[J] = (unsigned char)z;
  return 0;
}

static int alloc_block(gast_handle* h, BlockConsts* b, int C, int Cout, int heads, int Cg, int kind) {
  b->C = C; b->Cout = Cout; b->heads = heads; b->Cg = Cg;
  b->tpm = (Cout + 63) / 64;
  const bool has_local = (kind == GAST_KIND_MODEL || kind == GAST_KIND_BLOCK || kind == GAST_KIND_LOCAL ||
                          kind == GAST_KIND_SEMCH);
  const bool has_global = (kind == GAST_KIND_MODEL || kind == GAST_KIND_BLOCK || kind == GAST_KIND_MGLOBAL ||
                           kind == GAST_KIND_GLOBAL_HEAD);
  const int nmask = (kind == GAST_KIND_SEMCH) ? 1 : 2;
  if (has_local) {
    if (dalloc(h, &b->Wloc, (size_t)nmask * b->tpm * 128 * C)) return 1;
    for (int m = 0; m < nmask; ++m)
      if (dalloc(h, &b->coef[m], (size_t)h->nnz[m] * Cout)) return 1;
    if (dalloc(h, &b->shift_loc, (size_t)nmask * Cout)) return 1;
    if (kind != GAST_KIND_SEMCH) {
      if (dalloc(h, &b->Wlc, (size_t)C * 2 * C) || dalloc(h, &b->blc, C)) return 1;
    }
  }
  if (has_global) {
    const int Ng = heads * Cg;
    if (dalloc(h, &b->Wg, (size_t)Ng * C) || dalloc(h, &b->bg, Ng) || dalloc(h, &b->U, (size_t)2 * heads * C) ||
        dalloc(h, &b->cab, 2 * heads) || dalloc(h, &b->Ck, (size_t)heads * h->cfg.num_joints * h->cfg.num_joints))
      return 1;
    if (kind != GAST_KIND_GLOBAL_HEAD) {
      if (dalloc(h, &b->Wgc, (size_t)C * C) || dalloc(h, &b->bgc, C)) return 1;
    }
  }
  if (kind == GAST_KIND_MODEL || kind == GAST_KIND_BLOCK) {
    if (dalloc(h, &b->Wbc, (size_t)2 * C * 3 * C) || dalloc(h, &b->bbc, 2 * C)) return 1;
  }
  return 0;
}

extern "C" int gast_create(gast_t** out, const gast_cfg* cfg) {
  if (!out || !cfg) return fail("gast_create: null argument");
  *out = nullptr;
  const int J = cfg->num_joints;
  if (J < 2 || J > 32) return fail("gast_create: num_joints %d out of range", J);
  if (cfg->channels <= 0 || cfg->channels % 4) return fail("gast_create: channels must be a positive multiple of 4");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("gast_create: no CUDA device (this library has no CPU path)");
  CUDA_OK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail("gast_create: built for sm_100a, device is sm_%d%d", prop.major, prop.minor);

  gast_handle* h = new gast_handle();
  h->cfg = *cfg;
  h->sm_count = prop.multiProcessorCount;
  h->fpt = 128 / J;
  if (const char* e = getenv("GAST_BLOCK1_SLABS")) h->block1_slabs = std::max(1, atoi(e));
  if (const char* e = getenv("GAST_TRAIN_TC")) h->train_tc_on = atoi(e) != 0;   // 0: training GEMMs on the FFMA core (A/B runs)
  h->sym_r.assign(cfg->sym_rows, cfg->sym_rows + cfg->sym_nnz);
  h->sym_c.assign(cfg->sym_cols, cfg->sym_cols + cfg->sym_nnz);
  h->nnz[0] = cfg->sym_nnz;
  const int kind = cfg->kind;
  const bool need_sym = (kind != GAST_KIND_MGLOBAL && kind != GAST_KIND_GLOBAL_HEAD);
  const bool need_con = (kind == GAST_KIND_MODEL || kind == GAST_KIND_BLOCK || kind == GAST_KIND_LOCAL);
  if (need_con) {
    h->con_r.assign(cfg->con_rows, cfg->con_rows + cfg->con_nnz);
    h->con_c.assign(cfg->con_cols, cfg->con_cols + cfg->con_nnz);
    h->nnz[1] = cfg->con_nnz;
  }
  h->cfg.sym_rows = h->cfg.sym_cols = h->cfg.con_rows = h->cfg.con_cols = nullptr;
  int rc = 0;
  if (need_sym) rc |= build_nbr(h->sym_r, h->sym_c, J, &h->nbr[0]);
  if (need_con) rc |= build_nbr(h->con_r, h->con_c, J, &h->nbr[1]);
  if (rc) { delete h; return 1; }

  if (kind == GAST_KIND_MODEL) {
    const int L = cfg->num_stages;
    if (L < 1 || L > GAST_MAX_STAGES) { delete h; return fail("gast_create: num_stages %d", L); }
    for (int i = 0; i < L; ++i)
      if (cfg->filter_widths[i] % 2 == 0) { delete h; return fail("Only odd filter widths are supported"); }
    const int C = cfg->channels;
    // geometry, gast_net.py:57,136-143 / 213-220
    h->pad.push_back(cfg->filter_widths[0] / 2);
    h->shift.push_back(cfg->causal ? cfg->filter_widths[0] / 2 : 0);
    int nd = cfg->filter_widths[0];
    h->blocks.resize(L);
    h->stages.resize(L - 1);
    rc |= alloc_block(h, &h->blocks[0], C, C, 4, C / 4, kind);
    for (int i = 1; i < L; ++i) {
      const int fw = cfg->filter_widths[i];
      const int Cw = C << i;
      h->pad.push_back((fw - 1) * nd / 2);
      StageConsts& s = h->stages[i - 1];
      s.Cw = Cw;
      if (cfg->strided) {
        h->shift.push_back(cfg->causal ? fw / 2 : 0);
        s.taps = fw; s.stride = fw; s.dil = 1;
      } else {
        h->shift.push_back(cfg->causal ? (fw / 2) * nd : 0);
        if (cfg->dense) { s.taps = 2 * h->pad.back() + 1; s.stride = 1; s.dil = 1; }
        else { s.taps = fw; s.stride = 1; s.dil = nd; }
      }
      rc |= dalloc(h, &s.Wt, (size_t)Cw * s.taps * Cw) | dalloc(h, &s.bt, Cw) |
            dalloc(h, &s.W1, (size_t)Cw * Cw) | dalloc(h, &s.b1, Cw);
      rc |= alloc_block(h, &h->blocks[i], Cw, Cw, 4, Cw / 4, kind);
      nd *= fw;
    }
    rc |= dalloc(h, &h->We, (size_t)C * cfg->filter_widths[0] * cfg->in_features) | dalloc(h, &h->be, C);
    rc |= dalloc(h, &h->loss_scratch, 2 * 1024 + 4);   // shrink+mpjpe partials and ticket (SHL_MAXBLOCKS doubles + 1 word)
  } else {
    h->blocks.resize(1);
    const int C = cfg->channels;
    int Cout = C, heads = 4, Cg = C / 4;
    if (kind == GAST_KIND_SEMCH) Cout = cfg->channels_out > 0 ? cfg->channels_out : C;
    if (kind == GAST_KIND_MGLOBAL) { heads = cfg->heads; Cg = C / heads; }
    if (kind == GAST_KIND_GLOBAL_HEAD) { heads = 1; Cg = cfg->channels_out; }
    if (heads < 1 || heads > 4) { delete h; return fail("gast_create: heads=%d unsupported (1..4)", heads); }
    if (Cout % 4 || (heads * Cg) % 4) { delete h; return fail("gast_create: widths must be multiples of 4"); }
    rc |= alloc_block(h, &h->blocks[0], C, Cout, heads, Cg, kind);
  }
  if (rc) { gast_destroy(h); return 1; }
  *out = h;
  return 0;
}

extern "C" void gast_destroy(gast_t* h) {
  if (!h) return;
  for (void* p : h->owned) cudaFree(p);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  delete h;
}

extern "C" int gast_bind(gast_t* h, int32_t n, const char* const* keys, void* const* ptrs, const int64_t* numel) {
  if (!h) return fail("gast_bind: null handle");
  for (int i = 0; i < n; ++i) h->bound[keys[i]] = Binding{ptrs[i], numel[i]};
  h->prepared = false;
  return 0;
}

extern "C" int gast_set_gemm_core(gast_t* h, int32_t core) {
  if (!h) return fail("null handle");
  if (core != 0 && core != 1) return fail("gast_set_gemm_core: core must be 0 (auto) or 1 (ffma)");
  h->gemm_core = core;
  return 0;
}

extern "C" int32_t gast_last_launch_count(const gast_t* h) { return h ? h->launches : -1; }
extern "C" int32_t gast_last_tc_launch_count(const gast_t* h) { return h ? h->tc_launches : -1; }

extern "C" int gast_set_timing(gast_t* h, int32_t on) {
  if (!h) return fail("null handle");
  h->timing = on != 0;
  return 0;
}

extern "C" int32_t gast_get_timings(gast_t* h, int32_t max_n, float* ms, int32_t* kinds) {
  if (!h) return -1;
  int n = (int)(h->ev_used / 2);
  if (n > max_n) n = max_n;
  for (int i = 0; i < n; ++i) {
    if (cudaEventSynchronize(h->ev_pool[2 * i + 1]) != cudaSuccess) return -1;
    float t = 0.f;
    cudaEventElapsedTime(&t, h->ev_pool[2 * i], h->ev_pool[2 * i + 1]);
    ms[i] = t;
    kinds[i] = h->ev_kind[i];
  }
  return n;
}

// ------------------------------------------------------------------------------------------
// prepare
// ------------------------------------------------------------------------------------------
struct Lookup {
  gast_handle* h;
  bool ok = true;
  const float* get(const std::string& key, int64_t numel) {
    auto it = h->bound.find(key);
    if (it == h->bound.end()) { if (ok) fail("parameter '%s' is not bound", key.c_str()); ok = false; return nullptr; }
    if (numel >= 0 && it->second.numel != numel) {
      if (ok) fail("parameter '%s' has %lld elements, expected %lld", key.c_str(), (long long)it->second.numel, (long long)numel);
      ok = false; return nullptr;
    }
    return reinterpret_cast<const float*>(it->second.ptr);
  }
  bool has(const std::string& key) { return h->bound.count(key) != 0; }
  BnP bn(const std::string& prefix, int C) {
    BnP b;
    b.w = get(prefix + "weight", C); b.b = get(prefix + "bias", C);
    b.rm = get(prefix + "running_mean", C); b.rv = get(prefix + "running_var", C);
    return b;
  }
};

static inline unsigned cdiv(long long a, long long b) { return (unsigned)((a + b - 1) / b); }

static int prep_conv(cudaStream_t st, float* out, float* bias, const float* w, int N, int Cin, int taps, BnP bn) {
  long long total = (long long)N * Cin * taps;
  fold_conv_kernel<<<cdiv(total, 256), 256, 0, st>>>(out, bias, w, N, Cin, taps, bn);
  return 0;
}

static int prepare_local(gast_handle* h, Lookup& L, cudaStream_t st, BlockConsts& b, const std::string& lp, int kind) {
  const int C = b.C, Co = b.Cout, J = h->cfg.num_joints;
  const int nmask = (kind == GAST_KIND_SEMCH) ? 1 : 2;
  for (int m = 0; m < nmask; ++m) {
    std::string gp = (kind == GAST_KIND_SEMCH) ? lp : lp + (m == 0 ? "gcn_sym." : "gcn_con.");
    const float* W = L.get(gp + "W", (int64_t)2 * C * Co);
    const bool shared = (kind == GAST_KIND_SEMCH) && h->cfg.semch_shared_e;
    const float* e = L.get(gp + "e", shared ? h->nnz[m] : (int64_t)Co * h->nnz[m]);
    BnP bn = {nullptr, nullptr, nullptr, nullptr};
    const float* bias = nullptr;
    if (kind != GAST_KIND_SEMCH) bn = L.bn(lp + (m == 0 ? "bn_1." : "bn_2."), Co);
    else if (h->cfg.semch_bias) bias = L.get(gp + "bias", Co);
    if (!L.ok) return 1;
    long long tot = (long long)b.tpm * 128 * C;
    semch_pack_kernel<<<cdiv(tot, 256), 256, 0, st>>>(b.Wloc + (size_t)m * b.tpm * 128 * C, W, b.tpm, C, Co);
    semch_coef_kernel<<<cdiv((long long)Co * J, 128), 128, 0, st>>>(
        b.coef[m], b.shift_loc + (size_t)m * Co, e, shared ? 0 : h->nnz[m], h->nbr[m], h->nnz[m], Co, J, bn, bias);
  }
  if (kind != GAST_KIND_SEMCH) {
    const float* w = L.get(lp + "cat_conv.weight", (int64_t)C * 2 * C);
    BnP bn = L.bn(lp + "cat_bn.", C);
    if (!L.ok) return 1;
    prep_conv(st, b.Wlc, b.blc, w, C, 2 * C, 1, bn);
  }
  return 0;
}

static int prepare_global(gast_handle* h, Lookup& L, cudaStream_t st, BlockConsts& b, const std::string& gp, int kind) {
  const int C = b.C, J = h->cfg.num_joints, Cg = b.Cg;
  for (int hd = 0; hd < b.heads; ++hd) {
    std::string hp = (kind == GAST_KIND_GLOBAL_HEAD) ? gp : gp + "attentions." + std::to_string(hd) + ".";
    // inter_channels: theta/phi width.  In a block inter == Cg (global_attention.py:21-24).
    const int Ci = Cg;
    const float* gw = L.get(hp + "g.weight", (int64_t)Cg * C);
    const float* gb = L.get(hp + "g.bias", Cg);
    const float* tw = L.get(hp + "theta.weight", (int64_t)Ci * C);
    const float* tb = L.get(hp + "theta.bias", Ci);
    const float* pw = L.get(hp + "phi.weight", (int64_t)Ci * C);
    const float* pb = L.get(hp + "phi.bias", Ci);
    const float* wc = L.get(hp + "concat_project.0.weight", 2 * Ci);
    const float* ck = L.get(hp + "C_k", (int64_t)J * J);
    if (!L.ok) return 1;
    CUDA_OK(cudaMemcpyAsync(b.Wg + (size_t)hd * Cg * C, gw, sizeof(float) * Cg * C, cudaMemcpyDeviceToDevice, st));
    CUDA_OK(cudaMemcpyAsync(b.bg + (size_t)hd * Cg, gb, sizeof(float) * Cg, cudaMemcpyDeviceToDevice, st));
    CUDA_OK(cudaMemcpyAsync(b.Ck + (size_t)hd * J * J, ck, sizeof(float) * J * J, cudaMemcpyDeviceToDevice, st));
    global_collapse_kernel<<<cdiv(C, 32), 256, 0, st>>>(b.U, b.cab, tw, tb, pw, pb, wc, hd, C, Ci);
  }
  if (kind != GAST_KIND_GLOBAL_HEAD) {
    const float* w = L.get(gp + "cat_conv.weight", (int64_t)C * C);
    BnP bn = L.bn(gp + "cat_bn.", C);
    if (!L.ok) return 1;
    prep_conv(st, b.Wgc, b.bgc, w, C, C, 1, bn);
  }
  return 0;
}

static int prepare_block(gast_handle* h, Lookup& L, cudaStream_t st, BlockConsts& b, const std::string& P) {
  if (prepare_local(h, L, st, b, P + "local_graph_layer.", GAST_KIND_BLOCK)) return 1;
  if (prepare_global(h, L, st, b, P + "global_graph_layer.", GAST_KIND_BLOCK)) return 1;
  const int C = b.C;
  const float* w = L.get(P + "cat_conv.weight", (int64_t)2 * C * 3 * C);
  BnP bn = L.bn(P + "cat_bn.", 2 * C);
  if (!L.ok) return 1;
  prep_conv(st, b.Wbc, b.bbc, w, 2 * C, 3 * C, 1, bn);
  return 0;
}

static int prepare_tc(gast_handle* h, cudaStream_t st);

extern "C" int gast_prepare(gast_t* h, void* stream) {
  if (!h) return fail("gast_prepare: null handle");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->cfg.device));
  Lookup L{h};
  const int kind = h->cfg.kind;
  if (kind == GAST_KIND_MODEL) {
    const int C = h->cfg.channels, Fin = h->cfg.in_features, k0 = h->cfg.filter_widths[0];
    const float* we = L.get("expand_conv.weight", (int64_t)C * Fin * k0);
    BnP bin = L.bn("init_bn.", Fin), bex = L.bn("expand_bn.", C);
    if (!L.ok) return 1;
    expand_fold_kernel<<<cdiv(C, 128), 128, 0, st>>>(h->We, h->be, we, C, Fin, k0, bin, bex);
    for (size_t i = 0; i < h->blocks.size(); ++i)
      if (prepare_block(h, L, st, h->blocks[i], "layers_graph_conv." + std::to_string(i) + ".")) return 1;
    for (size_t i = 0; i < h->stages.size(); ++i) {
      StageConsts& s = h->stages[i];
      const float* w0 = L.get("layers_conv." + std::to_string(2 * i) + ".weight", (int64_t)s.Cw * s.Cw * s.taps);
      const float* w1 = L.get("layers_conv." + std::to_string(2 * i + 1) + ".weight", (int64_t)s.Cw * s.Cw);
      BnP b0 = L.bn("layers_bn." + std::to_string(2 * i) + ".", s.Cw);
      BnP b1 = L.bn("layers_bn." + std::to_string(2 * i + 1) + ".", s.Cw);
      if (!L.ok) return 1;
      prep_conv(st, s.Wt, s.bt, w0, s.Cw, s.Cw, s.taps, b0);
      prep_conv(st, s.W1, s.b1, w1, s.Cw, s.Cw, 1, b1);
    }
    L.get("shrink.weight", (int64_t)3 * (C << (h->cfg.num_stages)));
    if (!L.ok) return 1;
  } else if (kind == GAST_KIND_BLOCK) {
    if (prepare_block(h, L, st, h->blocks[0], "")) return 1;
  } else if (kind == GAST_KIND_LOCAL || kind == GAST_KIND_SEMCH) {
    if (prepare_local(h, L, st, h->blocks[0], "", kind)) return 1;
  } else if (kind == GAST_KIND_MGLOBAL || kind == GAST_KIND_GLOBAL_HEAD) {
    if (prepare_global(h, L, st, h->blocks[0], "", kind)) return 1;
  } else {
    return fail("gast_prepare: unknown kind %d", kind);
  }
  if (prepare_tc(h, st)) return 1;
  CUDA_OK(cudaGetLastError());
  h->prepared = true;
  h->stream_ready = false;
  return 0;
}

// ------------------------------------------------------------------------------------------
// forward planning
// ------------------------------------------------------------------------------------------
struct Geometry {          // frames per clip after each layer
  int T0 = 0;              // after expand
  std::vector<int> Ts;     // after stage i (index i-1)
  int s0 = 1;
  int T_out = 0;
};

// schedule actually run: the handle's own (cfg.strided) or, for a dilated model on a
// receptive-field-long clip, the equivalent strided one (same arithmetic per output, see
// SURVEY.md §7 "dense vs needed-only work").
struct Sched {
  int taps, stride, dil, res_mul, res_off;
};

static int stage_sched(const gast_handle* h, int i /*1-based*/, int strided_now, Sched* s) {
  const gast_cfg& c = h->cfg;
  const int fw = c.filter_widths[i];
  if (strided_now) {
    // gast_net.py:222-224,243 ; causal shift of the strided form is fw//2 (:220)
    s->taps = fw; s->stride = fw; s->dil = 1;
    s->res_mul = fw;
    s->res_off = (c.causal ? fw / 2 : 0) + fw / 2;
  } else {
    const StageConsts& sc = h->stages[i - 1];
    s->taps = sc.taps; s->stride = 1; s->dil = sc.dil;
    s->res_mul = 1;
    s->res_off = h->pad[i] + h->shift[i];   // gast_net.py:170
  }
  return 0;
}

static int geometry(const gast_handle* h, int T, int strided_now, Geometry* g) {
  const gast_cfg& c = h->cfg;
  if (strided_now && !c.strided && c.dense) return fail("dense model has no strided schedule");
  if (!strided_now && c.strided) return fail("Optimized1f handle only runs the strided schedule");
  const int k0 = c.filter_widths[0];
  g->s0 = strided_now ? k0 : 1;
  if (T < k0) return fail("input has %d frames, fewer than the first filter width %d", T, k0);
  g->T0 = (T - k0) / g->s0 + 1;
  int Tp = g->T0;
  g->Ts.clear();
  for (int i = 1; i < c.num_stages; ++i) {
    Sched s;
    stage_sched(h, i, strided_now, &s);
    const int span = (s.taps - 1) * s.dil + 1;
    if (Tp < span) return fail("input of %d frames is shorter than the receptive field", T);
    int Tn = (Tp - span) / s.stride + 1;
    // residual slice must cover the conv output (the reference would raise on the add otherwise)
    if (s.res_off + (long long)(Tn - 1) * s.res_mul >= Tp) return fail("residual slice out of range for T=%d", T);
    g->Ts.push_back(Tn);
    Tp = Tn;
  }
  g->T_out = Tp;
  return 0;
}

extern "C" int32_t gast_receptive_field(const gast_t* h) {
  if (!h || h->cfg.kind != GAST_KIND_MODEL) return -1;
  int rf = 1;
  for (int p : h->pad) rf += 2 * p;
  return rf;
}

extern "C" int32_t gast_out_frames(const gast_t* h, int32_t T, int32_t strided_now) {
  if (!h) return -1;
  if (h->cfg.kind != GAST_KIND_MODEL) return T;
  Geometry g;
  if (geometry(h, T, strided_now, &g)) return -1;
  return g.T_out;
}

// workspace carve-up ------------------------------------------------------------------
struct Arena {
  char* base; size_t size; size_t off = 0; bool dry;
  float* take(size_t nfloats) {
    size_t bytes = (nfloats * sizeof(float) + 255) & ~(size_t)255;
    float* p = dry ? nullptr : reinterpret_cast<float*>(base + off);
    off += bytes;
    return p;
  }
};

struct BlockBufs { float *XY, *L, *AB, *Y, *Gl; };

static void block_bufs(Arena& a, long long rows, int C, int Cout, int heads, int Cg, BlockBufs* b) {
  b->XY = a.take((size_t)rows * 2 * Cout);
  b->L = a.take((size_t)rows * C);
  b->AB = a.take((size_t)rows * 2 * heads);
  b->Y = a.take((size_t)rows * heads * Cg);
  b->Gl = a.take((size_t)rows * C);
}

// ------------------------------------------------------------------------------------------
// launches
// ------------------------------------------------------------------------------------------
static ASeg seg_flat(const float* base, int ld, int K) {
  ASeg s; s.base = base; s.ld = ld; s.K = K; s.Kc = K; s.tap_stride = 0; s.map = RowMap{1, 1, 1, 0};
  return s;
}

static void gemm_defaults(GemmP& p, const gast_handle* h, long long F) {
  memset(&p, 0, sizeof(p));
  p.F = (int)F; p.J = h->cfg.num_joints; p.fpt = h->fpt;
  p.res_map = RowMap{1, 1, 1, 0};
}

// A 1x1 layer with flat operands and no joint mixing does not need frame-aligned tiles: run it as
// F*J "frames" of one joint, so that every tile carries 128 rows instead of floor(128/J)*J (119 for J=17).
static void gemm_defaults_flat(GemmP& p, const gast_handle* h, long long F) {
  gemm_defaults(p, h, F);
  p.F = (int)(F * h->cfg.num_joints); p.J = 1; p.fpt = 128;
}

static int launch_gemm(gast_handle* h, cudaStream_t st, int epi, const GemmP& p, const TcWeights* tcw) {
  if (p.F <= 0) return 0;
  int Ktot = 0;
  for (int s = 0; s < p.nseg; ++s) Ktot += p.seg[s].K;
  if (Ktot != p.ldw) return fail("internal: K mismatch %d vs %d", Ktot, p.ldw);
  if (p.N % 4 || p.ld_out % 4) return fail("internal: N/ld_out must be multiples of 4");
  if (h->gemm_core == 0 && tcw && tc_supported(p, epi, *tcw)) {
    TimedLaunch tl(h, st, LK_TC_PLAIN + epi);
    int rc = tc_launch(h->sm_count, st, epi, p, *tcw);
    if (rc) return fail("tcgen05 gemm launch failed: %s", cudaGetErrorString((cudaError_t)rc));
    h->launches++;
    h->tc_launches++;
    return 0;
  }
  TimedLaunch tl(h, st, LK_GEMM_PLAIN + epi);
  dim3 grid(cdiv(p.F, p.fpt), cdiv(p.N, FF_BN));
  int hpt = 1;
  if (epi == EPI_GLOBAL) hpt = p.heads < 4 ? p.heads : 4;
  size_t smem = ffma_smem_bytes(epi, p.J, p.fpt, hpt);
  static bool attr_set_dev[64][3];          // the opt-in is per device (one handle per device in one process)
  bool& attr_done = attr_set_dev[h->cfg.device & 63][epi];
  if (!attr_done) {
    const void* fn = epi == EPI_PLAIN ? (const void*)gemm_ffma_kernel<EPI_PLAIN>
                   : epi == EPI_SEMCH ? (const void*)gemm_ffma_kernel<EPI_SEMCH>
                                      : (const void*)gemm_ffma_kernel<EPI_GLOBAL>;
    CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_done = true;
  }
  if (epi == EPI_PLAIN) gemm_ffma_kernel<EPI_PLAIN><<<grid, FF_THREADS, smem, st>>>(p);
  else if (epi == EPI_SEMCH) gemm_ffma_kernel<EPI_SEMCH><<<grid, FF_THREADS, smem, st>>>(p);
  else gemm_ffma_kernel<EPI_GLOBAL><<<grid, FF_THREADS, smem, st>>>(p);
  h->launches++;
  return 0;
}

static int launch_rowdot(gast_handle* h, cudaStream_t st, const float* X, int ldx, const BlockConsts& b,
                         float* ab, long long rows) {
  if (rows <= 0) return 0;
  const int Q = 2 * b.heads;
  unsigned blocks = cdiv(rows * 32, 256);
  TimedLaunch tl(h, st, LK_ROWDOT);
  if (Q == 8 && b.C % 4 == 0 && (size_t)8 * b.C * sizeof(float) <= 48 * 1024) {
    unsigned g = (unsigned)std::min<long long>((rows * 32 + 255) / 256, (long long)h->sm_count * 8);
    rowdot8_kernel<<<g, 256, sizeof(float) * 8 * b.C, st>>>(X, ldx, b.U, b.cab, ab, rows, b.C);
  } else if (Q == 8) rowdot_kernel<8><<<blocks, 256, 0, st>>>(X, ldx, b.U, b.cab, ab, rows, b.C);
  else if (Q == 6) rowdot_kernel<6><<<blocks, 256, 0, st>>>(X, ldx, b.U, b.cab, ab, rows, b.C);
  else if (Q == 4) rowdot_kernel<4><<<blocks, 256, 0, st>>>(X, ldx, b.U, b.cab, ab, rows, b.C);
  else if (Q == 2) rowdot_kernel<2><<<blocks, 256, 0, st>>>(X, ldx, b.U, b.cab, ab, rows, b.C);
  else return fail("internal: heads=%d", b.heads);
  h->launches++;
  return 0;
}

// SemCH (both masks) -> XY ; then local cat conv -> L          (local_attention.py:130-151)
static int run_local(gast_handle* h, cudaStream_t st, BlockConsts& b, const float* X, long long F,
                     const BlockBufs& w, float* out_L, int kind) {
  const int C = b.C, Co = b.Cout;
  const int nmask = (kind == GAST_KIND_SEMCH) ? 1 : 2;
  GemmP p;
  gemm_defaults(p, h, F);
  p.nseg = 1; p.seg[0] = seg_flat(X, C, C);
  p.W = b.Wloc; p.ldw = C; p.N = nmask * b.tpm * 128;
  p.out = (kind == GAST_KIND_SEMCH) ? out_L : w.XY;
  p.ld_out = nmask * Co;
  p.relu = (kind == GAST_KIND_SEMCH) ? 0 : 1;
  p.coef[0] = b.coef[0]; p.coef[1] = b.coef[1];
  p.shift = b.shift_loc; p.C = Co; p.tiles_per_mask = b.tpm;
  p.nbr[0] = h->nbr[0]; p.nbr[1] = h->nbr[1];
  if (launch_gemm(h, st, EPI_SEMCH, p, &b.tc_loc)) return 1;
  if (kind == GAST_KIND_SEMCH) return 0;
  gemm_defaults_flat(p, h, F);
  p.nseg = 1; p.seg[0] = seg_flat(w.XY, 2 * C, 2 * C);
  p.W = b.Wlc; p.ldw = 2 * C; p.N = C; p.out = out_L; p.ld_out = C; p.bias = b.blc; p.relu = 1;
  return launch_gemm(h, st, EPI_PLAIN, p, &b.tc_lc);
}

// collapsed theta/phi -> attention-mixed g -> Y ; then global cat conv -> Gl   (global_attention.py:52-130)
static int run_global(gast_handle* h, cudaStream_t st, BlockConsts& b, const float* X, long long F,
                      const BlockBufs& w, float* out_G, int kind) {
  const int C = b.C, J = h->cfg.num_joints, Ng = b.heads * b.Cg;
  if (launch_rowdot(h, st, X, C, b, w.AB, F * J)) return 1;
  GemmP p;
  // tcgen05 core, block / MultiGlobalGraph: plain `g` GEMM (flat 128-row tiles) into out_G as scratch, then the
  // attention mix as its own full-occupancy kernel into Y.  Measured faster than the mix fused into the GEMM
  // epilogue (the fused form stays for the FFMA core and the single-head kind, and as GAST_GLOBAL_FUSED=1).
  static const bool fused_env = getenv("GAST_GLOBAL_FUSED") && atoi(getenv("GAST_GLOBAL_FUSED")) != 0;
  if (!fused_env && h->gemm_core == 0 && kind != GAST_KIND_GLOBAL_HEAD && b.tc_g.ready && Ng % 4 == 0 &&
      b.Cg % 4 == 0 && J <= MIX_JMAX) {
    gemm_defaults_flat(p, h, F);
    p.nseg = 1; p.seg[0] = seg_flat(X, C, C);
    p.W = b.Wg; p.ldw = C; p.N = Ng; p.out = out_G; p.ld_out = Ng; p.bias = b.bg; p.relu = 0;
    if (launch_gemm(h, st, EPI_PLAIN, p, &b.tc_g)) return 1;
    static const int mix_v = getenv("GAST_MIX_V") ? atoi(getenv("GAST_MIX_V")) : 4;   // channels per thread (4 or 2)
    const int vn = (mix_v == 2 && b.Cg % 2 == 0) ? 2 : 4;
    const int GV = Ng / vn;
    const int nthr = (vn == 2) ? 2 * MIX_THREADS : MIX_THREADS;
    int fpb = GV >= nthr ? 1 : nthr / GV;
    fpb = std::max(1, std::min(fpb, (int)(40 * 1024 / (sizeof(float) * b.heads * J * MIX_JP))));   // attention rows fit 40 KB
    const size_t smem = sizeof(float) * (size_t)fpb * b.heads * J * MIX_JP;
    {
      TimedLaunch tl(h, st, LK_GLOBAL_MIX);
      if (vn == 2)
        global_mix_kernel<float2, 2 * MIX_THREADS><<<cdiv(F, fpb), 2 * MIX_THREADS, smem, st>>>(out_G, Ng, w.AB, b.Ck, w.Y, Ng, F, J, b.heads, b.Cg, fpb);
      else
        global_mix_kernel<float4, MIX_THREADS><<<cdiv(F, fpb), MIX_THREADS, smem, st>>>(out_G, Ng, w.AB, b.Ck, w.Y, Ng, F, J, b.heads, b.Cg, fpb);
      h->launches++;
    }
    CUDA_OK(cudaGetLastError());
    gemm_defaults_flat(p, h, F);
    p.nseg = 1; p.seg[0] = seg_flat(w.Y, C, C);
    p.W = b.Wgc; p.ldw = C; p.N = C; p.out = out_G; p.ld_out = C; p.bias = b.bgc; p.relu = 1;
    return launch_gemm(h, st, EPI_PLAIN, p, &b.tc_gc);
  }
  gemm_defaults(p, h, F);
  p.nseg = 1; p.seg[0] = seg_flat(X, C, C);
  p.W = b.Wg; p.ldw = C; p.N = Ng;
  p.out = (kind == GAST_KIND_GLOBAL_HEAD) ? out_G : w.Y;
  p.ld_out = Ng;
  p.ab = w.AB; p.ck = b.Ck; p.bg = b.bg; p.heads = b.heads; p.Cg = b.Cg;
  if (launch_gemm(h, st, EPI_GLOBAL, p, &b.tc_g)) return 1;
  if (kind == GAST_KIND_GLOBAL_HEAD) return 0;
  gemm_defaults_flat(p, h, F);
  p.nseg = 1; p.seg[0] = seg_flat(w.Y, C, C);
  p.W = b.Wgc; p.ldw = C; p.N = C; p.out = out_G; p.ld_out = C; p.bias = b.bgc; p.relu = 1;
  return launch_gemm(h, st, EPI_PLAIN, p, &b.tc_gc);
}

// GraphAttentionBlock (gast_net.py:22-33): X (F*J, C) -> out (F*J, 2C)
static int run_block(gast_handle* h, cudaStream_t st, BlockConsts& b, const float* X, long long F,
                     const BlockBufs& w, float* out) {
  const int C = b.C;
  static const bool global_first = getenv("GAST_BLOCK_ORDER") && atoi(getenv("GAST_BLOCK_ORDER")) != 0;   // experiment
  if (global_first) {
    if (run_global(h, st, b, X, F, w, w.Gl, GAST_KIND_BLOCK)) return 1;
    if (run_local(h, st, b, X, F, w, w.L, GAST_KIND_BLOCK)) return 1;
  } else {
    if (run_local(h, st, b, X, F, w, w.L, GAST_KIND_BLOCK)) return 1;
    if (run_global(h, st, b, X, F, w, w.Gl, GAST_KIND_BLOCK)) return 1;
  }
  GemmP p;
  gemm_defaults_flat(p, h, F);
  p.nseg = 3;
  p.seg[0] = seg_flat(X, C, C); p.seg[1] = seg_flat(w.L, C, C); p.seg[2] = seg_flat(w.Gl, C, C);
  p.W = b.Wbc; p.ldw = 3 * C; p.N = 2 * C; p.out = out; p.ld_out = 2 * C; p.bias = b.bbc; p.relu = 1;
  return launch_gemm(h, st, EPI_PLAIN, p, &b.tc_bc);
}

struct ModelBufs {
  float* act[2];
  float* tmp;
  BlockBufs bb;
};

static int plan_model(const gast_handle* h, int B, int T, int strided_now, Arena& a, ModelBufs* mb, Geometry* g) {
  if (geometry(h, T, strided_now, g)) return 1;
  const int J = h->cfg.num_joints, C = h->cfg.channels, L = h->cfg.num_stages;
  // max over layers
  size_t act = 0, tmp = 0, xy = 0, l = 0, ab = 0;
  long long rows = (long long)B * g->T0 * J;
  for (int i = 0; i < L; ++i) {
    const int Cw = C << i;
    if (i > 0) {
      rows = (long long)B * g->Ts[i - 1] * J;
      tmp = std::max(tmp, (size_t)rows * Cw);
    }
    act = std::max(act, (size_t)rows * 2 * Cw);
    xy = std::max(xy, (size_t)rows * 2 * Cw);
    l = std::max(l, (size_t)rows * Cw);
    ab = std::max(ab, (size_t)rows * 8);
  }
  mb->act[0] = a.take(act); mb->act[1] = a.take(act);
  mb->tmp = a.take(tmp);
  mb->bb.XY = a.take(xy); mb->bb.L = a.take(l); mb->bb.AB = a.take(ab); mb->bb.Y = a.take(l); mb->bb.Gl = a.take(l);
  return 0;
}

extern "C" size_t gast_workspace_bytes(const gast_t* h, int32_t B, int32_t T, int32_t strided_now) {
  if (!h) return 0;
  Arena a{nullptr, 0, 0, true};
  if (h->cfg.kind == GAST_KIND_MODEL) {
    ModelBufs mb; Geometry g;
    if (plan_model(h, B, T, strided_now, a, &mb, &g)) return 0;
  } else {
    BlockBufs bb;
    const BlockConsts& b = h->blocks[0];
    block_bufs(a, (long long)B * h->cfg.num_joints, b.C, b.Cout, b.heads ? b.heads : 4, b.Cg ? b.Cg : b.C / 4, &bb);
  }
  return a.off + 256;
}

static int forward_impl(gast_t* h, const float* x, float* y, int32_t B, int32_t T, int32_t strided_now,
                        void* workspace, size_t workspace_bytes, void* stream, const float* target, float* loss);

extern "C" int gast_forward(gast_t* h, const float* x, float* y, int32_t B, int32_t T, int32_t strided_now,
                            void* workspace, size_t workspace_bytes, void* stream) {
  return forward_impl(h, x, y, B, T, strided_now, workspace, workspace_bytes, stream, nullptr, nullptr);
}

// forward + mpjpe of the prediction against `target` (B, T_out, J, 3) in one call: the caller-side pair
// `predicted = model(x); error = mpjpe(predicted, target)` of main.py:evaluate / train with the loss taken in the shrink
// kernel's epilogue (SURVEY §8f N2)
extern "C" int gast_forward_mpjpe(gast_t* h, const float* x, const float* target, float* y, float* loss, int32_t B, int32_t T,
                                  int32_t strided_now, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return fail("gast_forward_mpjpe: null handle");
  if (h->cfg.kind != GAST_KIND_MODEL) return fail("gast_forward_mpjpe: only the MODEL kind has a shrink layer");
  if (!target || !loss) return fail("gast_forward_mpjpe: target and loss must be device pointers");
  return forward_impl(h, x, y, B, T, strided_now, workspace, workspace_bytes, stream, target, loss);
}

static int forward_impl(gast_t* h, const float* x, float* y, int32_t B, int32_t T, int32_t strided_now,
                        void* workspace, size_t workspace_bytes, void* stream, const float* target, float* loss) {
  if (!h) return fail("gast_forward: null handle");
  if (!h->prepared) return fail("gast_forward: gast_prepare() has not run since the last gast_bind()");
  if (B <= 0 || T <= 0) return fail("gast_forward: empty batch (B=%d T=%d)", B, T);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->cfg.device));
  h->launches = 0;
  h->tc_launches = 0;
  h->ev_used = 0;
  h->ev_kind.clear();
  const size_t need = gast_workspace_bytes(h, B, T, strided_now);
  if (need == 0) return 1;
  if (workspace_bytes < need || !workspace)
    return fail("gast_forward: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
  uintptr_t wsb = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
  Arena a{reinterpret_cast<char*>(wsb), workspace_bytes, 0, false};
  const int J = h->cfg.num_joints;
  const int kind = h->cfg.kind;

  if (kind != GAST_KIND_MODEL) {
    if (T != 1) return fail("gast_forward: module kinds take T == 1 (frames in B)");
    BlockConsts& b = h->blocks[0];
    BlockBufs bb;
    block_bufs(a, (long long)B * J, b.C, b.Cout, b.heads ? b.heads : 4, b.Cg ? b.Cg : b.C / 4, &bb);
    int rc = 0;
    if (kind == GAST_KIND_BLOCK) rc = run_block(h, st, b, x, B, bb, y);
    else if (kind == GAST_KIND_LOCAL || kind == GAST_KIND_SEMCH) rc = run_local(h, st, b, x, B, bb, y, kind);
    else rc = run_global(h, st, b, x, B, bb, y, kind);
    if (rc) return 1;
    CUDA_OK(cudaGetLastError());
    return 0;
  }

  ModelBufs mb; Geometry g;
  if (plan_model(h, B, T, strided_now, a, &mb, &g)) return 1;
  const gast_cfg& c = h->cfg;
  const int C = c.channels, L = c.num_stages;
  // expand (gast_net.py:163-164) + first GraphAttentionBlock, optionally in SLABS of clips: the layers of block 1 are
  // the HBM-bound ones (K = C GEMMs, row dots, attention mix, expand), and a slab whose intermediates fit the 126 MB L2
  // hands them from producer to consumer on chip; the block temporaries are reused by every slab.
  long long F = (long long)B * g.T0;
  if (F * J >= 0x7fffffffLL) return fail("expand: more than 2^31 positions in one call");
  if (c.filter_widths[0] * c.in_features > EXP_MAXKF) return fail("expand: filter_width*in_features > %d unsupported", EXP_MAXKF);
  const int nslab = std::max(1, std::min(h->block1_slabs, B));
  const int Bs = (B + nslab - 1) / nslab;
  for (int b0 = 0; b0 < B; b0 += Bs) {
    const int nb = std::min(Bs, B - b0);
    const long long Fs = (long long)nb * g.T0, rows = Fs * J;
    const float* xs = x + (long long)b0 * T * J * c.in_features;
    float* a0 = mb.act[0] + (long long)b0 * g.T0 * J * C;
    float* a1 = mb.act[1] + (long long)b0 * g.T0 * J * 2 * C;
    static const bool expand_staged = !(getenv("GAST_EXPAND_STAGED") && atoi(getenv("GAST_EXPAND_STAGED")) == 0);
    if (expand_staged && expand_rows_ok(C)) {
      // staged form (kernels_hbm.cuh): inputs of 128 rows gathered once into shared memory, weights in registers
      TimedLaunch tl(h, st, LK_EXPAND);
      const unsigned nblk = (unsigned)cdiv(rows, EXS_ROWS);
      if (c.filter_widths[0] * c.in_features <= 6)
        expand_rows_kernel<6><<<nblk, EXS_THREADS, 0, st>>>(xs, h->We, h->be, a0, rows, J, T, g.T0, g.s0,
                                                            c.filter_widths[0], c.in_features, C);
      else
        expand_rows_kernel<EXP_MAXKF><<<nblk, EXS_THREADS, 0, st>>>(xs, h->We, h->be, a0, rows, J, T, g.T0, g.s0,
                                                                    c.filter_widths[0], c.in_features, C);
      h->launches++;
    } else {
      long long thr = ((rows + EXP_ROWS - 1) / EXP_ROWS) * (C / 4);
      TimedLaunch tl(h, st, LK_EXPAND);
      if (c.filter_widths[0] * c.in_features <= 6)
        expand_kernel<6><<<cdiv(thr, 256), 256, 0, st>>>(xs, h->We, h->be, a0, rows, J, T, g.T0, g.s0,
                                                        c.filter_widths[0], c.in_features, C);
      else
        expand_kernel<EXP_MAXKF><<<cdiv(thr, 256), 256, 0, st>>>(xs, h->We, h->be, a0, rows, J, T, g.T0, g.s0,
                                                                c.filter_widths[0], c.in_features, C);
      h->launches++;
    }
    if (run_block(h, st, h->blocks[0], a0, Fs, mb.bb, a1)) return 1;
  }
  int cur = 1;
  int Tp = g.T0;
  for (int i = 1; i < L; ++i) {
    StageConsts& s = h->stages[i - 1];
    Sched sc;
    stage_sched(h, i, strided_now, &sc);
    const int Cw = s.Cw, Tn = g.Ts[i - 1];
    const long long Fn = (long long)B * Tn;
    const float* xin = mb.act[cur];
    // temporal conv + BN + ReLU (gast_net.py:173)
    GemmP p;
    gemm_defaults(p, h, Fn);
    p.nseg = 1;
    p.seg[0].base = xin; p.seg[0].ld = Cw; p.seg[0].K = sc.taps * Cw; p.seg[0].Kc = Cw;
    p.seg[0].tap_stride = (long long)sc.dil * J * Cw;
    p.seg[0].map = RowMap{Tn, Tp, sc.stride, 0};
    p.W = s.Wt; p.ldw = sc.taps * Cw; p.N = Cw; p.out = mb.tmp; p.ld_out = Cw; p.bias = s.bt; p.relu = 1;
    if (launch_gemm(h, st, EPI_PLAIN, p, &s.tc_t)) return 1;
    // 1x1 conv + BN + ReLU (+Dropout = identity in eval) + residual slice (gast_net.py:170,174 / :243,247)
    gemm_defaults(p, h, Fn);
    p.nseg = 1; p.seg[0] = seg_flat(mb.tmp, Cw, Cw);
    p.W = s.W1; p.ldw = Cw; p.N = Cw; p.out = mb.act[cur ^ 1]; p.ld_out = Cw; p.bias = s.b1; p.relu = 1;
    p.res = xin; p.res_ld = Cw; p.res_map = RowMap{Tn, Tp, sc.res_mul, sc.res_off};
    if (launch_gemm(h, st, EPI_PLAIN, p, &s.tc_1)) return 1;
    cur ^= 1;
    if (run_block(h, st, h->blocks[i], mb.act[cur], Fn, mb.bb, mb.act[cur ^ 1])) return 1;
    cur ^= 1;
    Tp = Tn;
    F = Fn;
  }
  // shrink (gast_net.py:99) ; output is already (B, T_out, J, 3)
  {
    Lookup Lk{h};
    const int Cl = C << L;
    const float* ws = Lk.get("shrink.weight", (int64_t)3 * Cl);
    if (!Lk.ok) return 1;
    long long rows = F * J;
    if (target) {
      static_assert(SHL_MAXBLOCKS == 1024, "loss_scratch is sized for 1024 block partials");
      if (!h->loss_scratch) return fail("gast_forward_mpjpe: handle has no loss scratch");
      double* partial = reinterpret_cast<double*>(h->loss_scratch);
      unsigned* ticket = reinterpret_cast<unsigned*>(h->loss_scratch + 2 * SHL_MAXBLOCKS);
      const unsigned nb = (unsigned)std::min<long long>(SHL_MAXBLOCKS, (rows + 7) / 8);
      TimedLaunch tl(h, st, LK_SHRINK);
      shrink_mpjpe_kernel<<<nb, 256, 0, st>>>(mb.act[cur], Cl, ws, y, rows, Cl, target, partial, ticket, loss);
      h->launches++;
    } else {
    TimedLaunch tl(h, st, LK_SHRINK);
    shrink_kernel<<<cdiv(rows * 32, 256), 256, 0, st>>>(mb.act[cur], Cl, ws, y, rows, Cl);
    h->launches++;
    }
  }
  CUDA_OK(cudaGetLastError());
  return 0;
}

static int prep_one_tc(gast_handle* h, cudaStream_t st, TcWeights& t, const float* W, int N, int K, int semch);
static int make_perm(int J, int n, const int32_t* left, const int32_t* right, JointPerm* p);
#include "stream.cuh"

// ------------------------------------------------------------------------------------------
// tcgen05 weight copies
// ------------------------------------------------------------------------------------------
static int prep_one_tc(gast_handle* h, cudaStream_t st, TcWeights& t, const float* W, int N, int K, int semch) {
  if (!W) return 0;
  // inference arithmetic of the tcgen05 core: 2 = every operand fp16 (hi and remainder: 22 significant bits, 3 bf16-rate
  // products per MAC; GEMMs with K >= 256 whose weights fit fp16's range, see tc_prepare_weights), 0 = tf32 + bf16
  // corrections (4 bf16-equivalent products per MAC, fp32's range).  GAST_TC_F16=0 selects the latter everywhere.
  static const int inf_prec = (getenv("GAST_TC_F16") && atoi(getenv("GAST_TC_F16")) == 0) ? 0 : 2;
  int rc = tc_prepare_weights(t, W, N, K, st, &h->owned, semch, inf_prec);
  if (rc) return fail("tcgen05 weight preparation failed (%d): %s", rc,
                      rc > 0 ? cudaGetErrorString((cudaError_t)rc) : "cuTensorMapEncodeTiled unavailable/failed");
  return 0;
}

static int prepare_tc(gast_handle* h, cudaStream_t st) {
  const int kind = h->cfg.kind;
  for (BlockConsts& b : h->blocks) {
    const int C = b.C;
    const int nmask = (kind == GAST_KIND_SEMCH) ? 1 : 2;
    if (prep_one_tc(h, st, b.tc_loc, b.Wloc, nmask * b.tpm * 128, C, 1)) return 1;
    if (prep_one_tc(h, st, b.tc_lc, b.Wlc, C, 2 * C, 0)) return 1;
    if (prep_one_tc(h, st, b.tc_g, b.Wg, b.heads * b.Cg, C, 0)) return 1;
    if (prep_one_tc(h, st, b.tc_gc, b.Wgc, C, C, 0)) return 1;
    if (prep_one_tc(h, st, b.tc_bc, b.Wbc, 2 * C, 3 * C, 0)) return 1;
  }
  for (StageConsts& s : h->stages) {
    if (prep_one_tc(h, st, s.tc_t, s.Wt, s.Cw, s.taps * s.Cw, 0)) return 1;
    if (prep_one_tc(h, st, s.tc_1, s.W1, s.Cw, s.Cw, 0)) return 1;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// test-time augmentation around the forward (SURVEY.md §8f N1)
// ------------------------------------------------------------------------------------------
static int make_perm(int J, int n, const int32_t* left, const int32_t* right, JointPerm* p) {
  if (J < 1 || J > 32) return fail("tta: J out of range");
  for (int j = 0; j < 32; ++j) p->p[j] = (unsigned char)j;
  for (int k = 0; k < n; ++k) {
    if (left[k] < 0 || left[k] >= J || right[k] < 0 || right[k] >= J) return fail("tta: joint index out of range");
    p->p[left[k]] = (unsigned char)right[k];
    p->p[right[k]] = (unsigned char)left[k];
  }
  return 0;
}

extern "C" int gast_tta_prepare(const float* seq, float* out, int32_t T, int32_t J, int32_t F, int32_t pad,
                                int32_t causal_shift, int32_t n_sym, const int32_t* kps_left, const int32_t* kps_right,
                                void* stream) {
  if (T <= 0 || F <= 0 || pad < 0 || causal_shift < 0 || causal_shift > pad) return fail("gast_tta_prepare: bad arguments");
  JointPerm perm;
  if (make_perm(J, n_sym, kps_left, kps_right, &perm)) return 1;
  const long long n = (long long)(T + 2 * pad) * J * F;
  tta_prepare_kernel<<<cdiv(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      seq, out, T, J, F, pad + causal_shift, pad - causal_shift, perm);
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" int gast_tta_merge(const float* pred, float* out, int32_t T, int32_t J, int32_t n_sym,
                              const int32_t* joints_left, const int32_t* joints_right, void* stream) {
  if (T <= 0) return fail("gast_tta_merge: bad arguments");
  JointPerm perm;
  if (make_perm(J, n_sym, joints_left, joints_right, &perm)) return 1;
  const long long n = (long long)T * J * 3;
  tta_merge_kernel<<<cdiv(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(pred, out, T, J, perm);
  CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------
// training (SURVEY.md §8 row a12)
// ------------------------------------------------------------------------------------------
#include "train.cuh"

extern "C" int gast_bind_grads(gast_t* h, int32_t n, const char* const* keys, void* const* ptrs, const int64_t* numel) {
  if (!h) return fail("gast_bind_grads: null handle");
  for (int i = 0; i < n; ++i) h->grads[keys[i]] = Binding{ptrs[i], numel[i]};
  return 0;
}

static int train_check(gast_handle* h) {
  if (h->cfg.kind != GAST_KIND_MODEL) return fail("training is implemented for the MODEL kind only");
  return 0;
}

extern "C" size_t gast_train_workspace_bytes(gast_t* h, int32_t B, int32_t T, float dropout_p) {
  if (!h || train_check(h)) return 0;
  Arena a{nullptr, 0, 0, true};
  Lookup L{h};
  TCtx c{h, nullptr, &a, &L, h->cfg.num_joints, true};
  TrainState ts;
  ts.drop_p = dropout_p;
  if (train_forward(h, c, ts, nullptr, nullptr, B, T)) return 0;
  if (train_backward(h, c, ts, nullptr)) return 0;
  return a.off + 512;
}

extern "C" int gast_forward_train(gast_t* h, const float* x, float* y, int32_t B, int32_t T, float dropout_p,
                                  uint64_t seed, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return fail("gast_forward_train: null handle");
  if (train_check(h)) return 1;
  if (dropout_p < 0.f || dropout_p >= 1.f) return fail("gast_forward_train: dropout_p out of range");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->cfg.device));
  uintptr_t wsb = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
  Arena a{reinterpret_cast<char*>(wsb), workspace_bytes, 0, false};
  Lookup L{h};
  TCtx c{h, st, &a, &L, h->cfg.num_joints, false};
  const size_t need = gast_train_workspace_bytes(h, B, T, dropout_p);
  if (need == 0) return 1;
  if (!workspace || workspace_bytes < need) return fail("gast_forward_train: workspace too small (%zu < %zu)", workspace_bytes, need);
  h->launches = 0;
  for (size_t i = 0; i < h->trains.size(); ++i)      // a workspace reused by the caller: its old state is dead
    if (h->trains[i].first == workspace) { h->trains.erase(h->trains.begin() + i); break; }
  if (h->trains.size() >= GAST_MAX_PENDING_TRAIN) h->trains.erase(h->trains.begin());   // forwards never differentiated
  h->trains.emplace_back(workspace, TrainState());
  TrainState& ts = h->trains.back().second;
  ts.drop_p = dropout_p;
  ts.seed = seed;
  if (train_forward(h, c, ts, x, y, B, T)) { h->trains.pop_back(); return 1; }
  ts.arena_off = a.off;
  ts.valid = true;
  if (h->dropout_state && dropout_p > 0.f) dropout_bump_kernel<<<1, 1, 0, st>>>(h->dropout_state);
  h->prepared = false;      // running statistics changed: eval constants are stale
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" int gast_set_dropout_state(gast_t* h, void* dev_u64) {
  if (!h) return fail("gast_set_dropout_state: null handle");
  h->dropout_state = reinterpret_cast<unsigned long long*>(dev_u64);
  return 0;
}

extern "C" int gast_backward(gast_t* h, const float* dy, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return fail("gast_backward: null handle");
  size_t ti = h->trains.size();
  for (size_t i = 0; i < h->trains.size(); ++i)
    if (h->trains[i].first == workspace) ti = i;
  if (ti == h->trains.size() || !h->trains[ti].second.valid)
    return fail("gast_backward: no training forward is saved in this workspace (already differentiated, "
                "or more than %d forwards were outstanding)", GAST_MAX_PENDING_TRAIN);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->cfg.device));
  uintptr_t wsb = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
  TrainState ts = h->trains[ti].second;
  h->trains.erase(h->trains.begin() + ti);
  Arena a{reinterpret_cast<char*>(wsb), workspace_bytes, ts.arena_off, false};
  Lookup L{h};
  TCtx c{h, st, &a, &L, h->cfg.num_joints, false};
  c.tc_slot = 1024;                         // the backward's GEMMs follow the forward's in the operand-copy table
  if (train_backward(h, c, ts, dy)) return 1;
  if (a.off > workspace_bytes) return fail("gast_backward: workspace overrun");
  CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------
// debug / probe entry: out[M,N] = A[M,K] . W[N,K]^T on a chosen GEMM core (test infrastructure
// for the numerics of the tensor-core path; not used by the forward).
// ------------------------------------------------------------------------------------------
extern "C" int gast_debug_gemm(const float* A, const float* W, float* out, int32_t M, int32_t N, int32_t K,
                               int32_t core, int32_t tc_mode, int32_t reps, float* ms_out, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (M <= 0 || N <= 0 || K <= 0 || N % 4 || K % 4) return fail("gast_debug_gemm: bad shape");
  GemmP p;
  memset(&p, 0, sizeof(p));
  p.F = M; p.J = 1; p.fpt = 128;
  p.res_map = RowMap{1, 1, 1, 0};
  p.nseg = 1;
  p.seg[0].base = A; p.seg[0].ld = K; p.seg[0].K = K; p.seg[0].Kc = K; p.seg[0].tap_stride = 0;
  p.seg[0].map = RowMap{1, 1, 1, 0};
  p.W = W; p.ldw = K; p.N = N; p.out = out; p.ld_out = N;
  cudaEvent_t e0, e1;
  CUDA_OK(cudaEventCreate(&e0));
  CUDA_OK(cudaEventCreate(&e1));
  int rc = 0;
  std::vector<void*> owned;
  TcWeights t;
  int sms = 148;
  const int prec = (core == 2) ? 1 : (core == 3) ? 2 : 0;     // core 2 = the tcgen05 core in 3xTF32 arithmetic (training); 3 = fp16 hi
  if (core == 2 || core == 3) core = 0;
  if (core == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    rc = tc_prepare_weights(t, W, N, K, st, &owned, 0, prec);
    if (rc || !t.ready || !tc_supported(p, EPI_PLAIN, t)) {
      for (void* q : owned) cudaFree(q);
      return fail("gast_debug_gemm: shape not supported by the tcgen05 core (rc=%d)", rc);
    }
  } else {
    cudaFuncSetAttribute((const void*)gemm_ffma_kernel<EPI_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
  }
  auto launch = [&]() -> int {
    if (core == 0) return tc_launch(sms, st, EPI_PLAIN, p, t, tc_mode);
    dim3 grid(cdiv(M, 128), cdiv(N, FF_BN));
    gemm_ffma_kernel<EPI_PLAIN><<<grid, FF_THREADS, ffma_smem_bytes(EPI_PLAIN, 1, 128, 1), st>>>(p);
    return (int)cudaGetLastError();
  };
  unsigned long long* dbg = nullptr;
  if (core == 0 && tc_mode == 6) {
    // timing-attribution variant: counters land in `out` (M*N floats >= 148*32*2 required)
    if ((size_t)M * N * sizeof(float) < 160 * 32 * sizeof(unsigned long long)) return fail("gast_debug_gemm: out too small for dbg");
    dbg = reinterpret_cast<unsigned long long*>(out);
    cudaMemsetAsync(dbg, 0, 160 * 32 * sizeof(unsigned long long), st);
    p.dbg = dbg;
    p.out = out + 160 * 32 * 2;      // results are garbage-tolerant in this mode; keep clear of the counters
    p.F = M - 128;                   // stay inside the buffer
  }
  rc = launch();
  if (dbg) reps = 0;
  if (!rc && reps > 0) {
    cudaEventRecord(e0, st);
    for (int i = 0; i < reps && !rc; ++i) rc = launch();
    cudaEventRecord(e1, st);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (!rc && e == cudaSuccess && reps > 0 && ms_out) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    *ms_out = ms / reps;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  for (void* q : owned) cudaFree(q);
  if (rc || e != cudaSuccess) return fail("gast_debug_gemm: %s", cudaGetErrorString(rc ? (cudaError_t)rc : e));
  return 0;
}

// ------------------------------------------------------------------------------------------
// callers / data formats either side of the forward (SURVEY.md §8f N1-N3)
// ------------------------------------------------------------------------------------------
#include "pipeline.cuh"
