/*
 * gast_b200.h -- C ABI of the B200-native GAST-Net 2D->3D lifting path (libgast_b200.so).
 *
 * The reference (fabro66/GAST-Net-3DPoseEstimation) is pure Python and has no FFI for this
 * path; its "plugin boundary" is the Python class API of model/gast_net.py.  This header is
 * the C boundary underneath our drop-in classes: plain pointers and sizes, no torch types.
 * Each entry point cites the reference interface it stands in for.
 *
 * Ownership: the caller owns ALL device memory that crosses this boundary (parameters,
 * buffers, gradients, inputs, outputs, workspace).  A handle owns only small derived
 * constants (folded/packed weights) that gast_prepare() recomputes.  Nothing here
 * synchronises the device or allocates on the forward path; all work is enqueued on the
 * caller's stream.  Every call returns 0 on success, non-zero on error with a message in
 * gast_last_error() (thread-local).  Nothing throws or aborts.
 */
#ifndef GAST_B200_H
#define GAST_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gast_handle gast_t;

/* What a handle computes.  MODEL is the product; the others are the reference's
 * sub-modules, exposed so that parity can be tested module by module. */
enum gast_kind {
  GAST_KIND_MODEL = 0,       /* SpatioTemporalModel / ...Optimized1f   model/gast_net.py:107,180 */
  GAST_KIND_BLOCK = 1,       /* GraphAttentionBlock                    model/gast_net.py:8-33    */
  GAST_KIND_LOCAL = 2,       /* LocalGraph                             model/local_attention.py:59-151 */
  GAST_KIND_MGLOBAL = 3,     /* MultiGlobalGraph                       model/global_attention.py:85-130 */
  GAST_KIND_SEMCH = 4,       /* SemCHGraphConv / SemGraphConv          model/local_attention.py:10-56, model/sem_graph_conv.py:10-55 */
  GAST_KIND_GLOBAL_HEAD = 5  /* GlobalGraph                            model/global_attention.py:7-82 */
};

#define GAST_MAX_STAGES 8

/* Mirrors the constructor arguments of SpatioTemporalModel(adj, num_joints_in, in_features,
 * num_joints_out, filter_widths, causal, dropout, channels, dense) (model/gast_net.py:113-114)
 * and SpatioTemporalModelOptimized1f(...) (:191-192).  The adjacency enters as the two
 * LocalGraph masks (model/local_attention.py:92-114) in row-major nonzero order, which is the
 * order the learnable `e` is scattered in (:25,:41). */
typedef struct gast_cfg {
  int32_t kind;                          /* enum gast_kind */
  int32_t num_joints;                    /* J: 15, 16, 17 or 19 */
  int32_t in_features;                   /* 2 (MODEL only) */
  int32_t channels;                      /* MODEL: `channels`; other kinds: input width C */
  int32_t channels_out;                  /* SEMCH: out_features; GLOBAL_HEAD: inter_channels; else 0 */
  int32_t num_stages;                    /* len(filter_widths) (MODEL only) */
  int32_t filter_widths[GAST_MAX_STAGES];
  int32_t causal;
  int32_t dense;                         /* SpatioTemporalModel(dense=True) ablation */
  int32_t strided;                       /* 1 = Optimized1f schedule, 0 = dilated */
  int32_t heads;                         /* MGLOBAL/GLOBAL_HEAD: number of heads (BLOCK/MODEL: 4) */
  int32_t semch_shared_e;                /* SEMCH: 1 = one `e` row shared by all channels (sem_graph_conv.py) */
  int32_t semch_bias;                    /* SEMCH: 1 = has bias */
  int32_t sym_nnz, con_nnz;              /* nonzeros of the two masks (SEMCH uses `sym` only) */
  const int32_t* sym_rows; const int32_t* sym_cols;   /* host arrays, row-major nonzero order */
  const int32_t* con_rows; const int32_t* con_cols;
  int32_t device;                        /* CUDA device ordinal */
} gast_cfg;

/* nn.Module construction (gast_net.py:113-157).  Copies cfg (incl. the mask arrays). */
int gast_create(gast_t** out, const gast_cfg* cfg);
void gast_destroy(gast_t* h);

/* Borrow the caller's parameter / buffer storage by state_dict key (SURVEY.md 8b lists the
 * keys; they are exactly `module.state_dict().keys()` of the reference classes).  Pointers
 * are device pointers to contiguous fp32 (int64 for num_batches_tracked, ignored).  No copy:
 * optimiser updates are seen after the next gast_prepare().  Stands in for
 * nn.Module.load_state_dict / .parameters() (main.py:193,207-208). */
int gast_bind(gast_t* h, int32_t n, const char* const* keys, void* const* dev_ptrs,
              const int64_t* numel);

/* Recompute the eval-mode derived constants from the bound parameters: BN folded into the
 * adjacent conv, softmaxed per-channel adjacencies, packed SemCH weights, collapsed
 * theta/phi vectors.  Call after binding and after every parameter change (the Python shim
 * tracks tensor versions).  Enqueued on `stream` (a cudaStream_t). */
int gast_prepare(gast_t* h, void* stream);

/* Output frames for an input of T frames: T - rf + 1 (dilated) or the strided count
 * (gast_net.py:62-69,159-177,236-251).  `strided_now` = schedule actually used. Returns <0 on error. */
int32_t gast_out_frames(const gast_t* h, int32_t T, int32_t strided_now);
int32_t gast_receptive_field(const gast_t* h);

/* Bytes of caller-provided scratch gast_forward needs for a (B,T) batch. */
size_t gast_workspace_bytes(const gast_t* h, int32_t B, int32_t T, int32_t strided_now);

/* forward(x) (gast_net.py:84-104), eval mode.
 *   MODEL:  x (B,T,J,in_features) fp32 -> y (B,T_out,J,3) fp32, both contiguous.
 *           strided_now: 0 = dilated schedule (any T >= rf), 1 = strided schedule
 *           (T a multiple of the receptive field pattern, as Optimized1f requires).
 *   other kinds: x is (B frames, J, C) with T == 1; y is (B, J, C_out)
 *           (BLOCK: C_out = 2C, channels-last).
 * All work is enqueued on `stream`. */
int gast_forward(gast_t* h, const float* x, float* y, int32_t B, int32_t T,
                 int32_t strided_now, void* workspace, size_t workspace_bytes, void* stream);

/* forward + mpjpe in one call: the caller-side pair `predicted = model(x); error = mpjpe(predicted, target)` of
 * main.py:evaluate (main.py:270-300) and of the training loop's validation pass, with the loss of common/loss.py:5-11
 * taken in the shrink kernel's epilogue (no second pass over the prediction).  MODEL kind only.
 *   target (B,T_out,J,3) fp32 device; y as gast_forward; *loss (device float) = mean over B*T_out*J joints of
 *   ||y - target||_2.  Block partial sums are double and are added in a fixed order: the loss is reproducible run to run. */
int gast_forward_mpjpe(gast_t* h, const float* x, const float* target, float* y, float* loss, int32_t B, int32_t T,
                       int32_t strided_now, void* workspace, size_t workspace_bytes, void* stream);

/* Number of kernels the last gast_forward enqueued (for bench.py's gpu_launches). */
int32_t gast_last_launch_count(const gast_t* h);

/* Number of those that ran on the tcgen05 (tensor-core) GEMM core. */
int32_t gast_last_tc_launch_count(const gast_t* h);

/* Per-launch device timing for the roofline report: when on, gast_forward brackets every
 * kernel launch with a CUDA event pair on the caller's stream; gast_get_timings waits for
 * them and returns up to max_n (milliseconds, kind) pairs of the last forward.  kinds:
 * 0 expand, 1-3 FFMA GEMM (plain/SemCH/global epilogue), 4 theta/phi row-dot, 5 shrink,
 * 6-8 tcgen05 GEMM (plain/SemCH/global), 9 attention mix of MultiGlobalGraph as its own kernel. */
int gast_set_timing(gast_t* h, int32_t on);
int32_t gast_get_timings(gast_t* h, int32_t max_n, float* ms, int32_t* kinds);

/* GEMM core selection for A/B checks on the GPU: 0 = auto (tcgen05 where the shape
 * allows), 1 = force the FP32 FFMA core.  Not a fallback switch: both are CUDA paths. */
int gast_set_gemm_core(gast_t* h, int32_t core);

/* ---- test-time augmentation around the forward (the caller-side steps of reconstruction.evaluate /
 * main.evaluate, kept on the device) -----------------------------------------------------------------
 * gast_tta_prepare: UnchunkedGenerator.next_epoch(augment=True) (common/generators.py:210-233):
 *   seq (T,J,F) -> out (2, T+2*pad, J, F): edge padding (pad+causal_shift left, pad-causal_shift right)
 *   and the mirrored twin (feature 0 negated, kps_left[k] <-> kps_right[k] swapped).
 * gast_tta_merge: main.py:314-318: pred (2,T,J,3) -> out (T,J,3) = mean(pred[0], un-flipped pred[1]).
 * Index lists are host arrays of n_sym entries. */
int gast_tta_prepare(const float* seq, float* out, int32_t T, int32_t J, int32_t F, int32_t pad, int32_t causal_shift,
                     int32_t n_sym, const int32_t* kps_left, const int32_t* kps_right, void* stream);
int gast_tta_merge(const float* pred, float* out, int32_t T, int32_t J, int32_t n_sym, const int32_t* joints_left,
                   const int32_t* joints_right, void* stream);

/* ---- training (SpatioTemporalModelOptimized1f in train() mode, main.py:213-243) -------------------
 * gast_forward_train: forward with batch-statistics BatchNorm (running stats of the bound buffers
 *   are updated in place, momentum 0.1) and Dropout(p) driven by `seed`; keeps what the backward
 *   needs in `workspace` (must stay untouched until gast_backward).  x (B,T,J,F) -> y (B,T_out,J,3).
 * gast_backward: dy (B,T_out,J,3) -> gradient of every parameter, WRITTEN (not accumulated) into the
 *   buffers bound with gast_bind_grads (same keys as gast_bind; buffers/running stats have none).
 * Only the strided schedule trains, like the reference (main.py:166-171). */
int gast_bind_grads(gast_t* h, int32_t n, const char* const* keys, void* const* dev_ptrs, const int64_t* numel);
size_t gast_train_workspace_bytes(gast_t* h, int32_t B, int32_t T, float dropout_p);
int gast_forward_train(gast_t* h, const float* x, float* y, int32_t B, int32_t T, float dropout_p, uint64_t seed,
                       void* workspace, size_t workspace_bytes, void* stream);
int gast_backward(gast_t* h, const float* dy, void* workspace, size_t workspace_bytes, void* stream);
/* Optional device-side dropout state: one uint64 on the device (caller-owned, may be null to unset) that is added to
 * `seed` by every dropout kernel and advanced once per gast_forward_train.  With it a CUDA graph that captured a
 * training step (frozen kernel arguments) draws a fresh mask at every replay. */
int gast_set_dropout_state(gast_t* h, void* dev_u64);

/* ---- real-time causal streams (SURVEY.md 8f N4; gen_skes.py:43-69, tools/inference.py:19-110) -------------
 * The reference's real-time model is a causal SpatioTemporalModelOptimized1f re-run on the last
 * receptive_field frames for every new frame.  Here a pushed frame costs ONE new position per layer: `state`
 * (caller-owned device memory, gast_stream_state_bytes, contents irrelevant before the first push) holds per
 * temporal stage a ring of that stage's past inputs for n_streams concurrent streams.
 * gast_stream_push: x (n_streams, J, in_features) = the newest frame of every stream -> y (n_streams, J, 3) =
 *   its 3D pose, identical to the whole-sequence causal forward on the sequence so far, left-padded by
 *   replicating the stream's first frame (UnchunkedGenerator(pad, causal_shift=pad), common/generators.py:210-221).
 *   step = number of frames pushed into `state` before this one (0, 1, 2, ...; the caller counts).
 *   fresh (n_streams) int32 on the device, or null: non-zero = this frame starts a new sequence on that stream
 *   (must be non-zero for every stream at step 0).  MODEL handles with causal = 1 only; all work on `stream`. */
size_t gast_stream_state_bytes(gast_t* h, int32_t n_streams);
size_t gast_stream_workspace_bytes(gast_t* h, int32_t n_streams);
int gast_stream_push(gast_t* h, void* state, int64_t step, const float* x, float* y, int32_t n_streams,
                     const int32_t* fresh, void* workspace, size_t workspace_bytes, void* stream);

/* ---- delayed streams: non-causal models and test-time augmentation, O(1) per frame --------------------------
 * A non-causal model (the accurate 27/81-frame checkpoints reconstruction.py and gen_skes.generate_skeletons run)
 * streams with the same rings when its output comes `delay` frames late: the pose a push returns is that of the
 * frame pushed `delay` pushes earlier.  gast_stream_delay = sum_i (pad_i - causal_shift_i): 0 for a causal model,
 * (receptive_field - 1) / 2 otherwise (13 for 27 frames, 40 for 81); -1 on error.
 * gast_stream_push_delayed: as gast_stream_push, for causal and non-causal MODEL handles (dilated or Optimized1f;
 *   not the dense ablation), plus
 *   hold (n_streams) int32 on the device, or null: non-zero = the stream's sequence is over; its row of x is ignored
 *     and its newest frame is repeated.  `delay` such pushes after the last real frame return the last `delay` poses,
 *     exactly the reference's edge padding on the right (UnchunkedGenerator(pad, causal_shift=0)).  fresh wins over
 *     hold.  The left edge is the fresh fill of gast_stream_push.
 *   n_sym > 0: test-time augmentation (UnchunkedGenerator(augment=True) + main.py:314-318) inside the stream: the
 *     mirrored twin of every stream (feature 0 negated, kps_left[k] <-> kps_right[k]) runs as n_streams more rows of
 *     the same rings, and y = mean(pose, un-flipped twin pose) with joints_left[k] <-> joints_right[k].  Index lists
 *     are host arrays of n_sym entries; n_sym = 0 = no augmentation.
 *   state_bytes: size of `state`, at least gast_stream_delayed_state_bytes(h, n_streams, n_sym > 0).
 * Bitwise guarantees: with a causal model, no hold and no augmentation y equals gast_stream_push's; with augmentation
 * y equals the un-augmented push of 2 n_streams streams fed the twins, followed by gast_tta_merge. */
int32_t gast_stream_delay(gast_t* h);
size_t gast_stream_delayed_state_bytes(gast_t* h, int32_t n_streams, int32_t augment);
size_t gast_stream_delayed_workspace_bytes(gast_t* h, int32_t n_streams, int32_t augment);
int gast_stream_push_delayed(gast_t* h, void* state, size_t state_bytes, int64_t step, const float* x, float* y,
                             int32_t n_streams, const int32_t* fresh, const int32_t* hold, int32_t n_sym,
                             const int32_t* kps_left, const int32_t* kps_right, const int32_t* joints_left,
                             const int32_t* joints_right, void* workspace, size_t workspace_bytes, void* stream);

/* ---- either side of the forward, on the device (SURVEY.md 8f N1-N3) --------------------------------
 * All pointers are device pointers unless marked (host).  Work is enqueued on `stream`.
 *
 * gast_chunk_gather: one training batch of ChunkedGenerator.next_epoch (common/generators.py:93-154).
 *   poses_2d (total_frames,J2,F2) / poses_3d (total_frames,J3,3) = every sequence concatenated along
 *   time; seq_start[n_seq+1] = first frame of each sequence; cameras (n_seq,ncam); pairs (B,4) int32 =
 *   the reference's (seq_i, start_3d, end_3d, flip) tuples.  Writes batch_2d (B,chunk+2*pad,J2,F2)
 *   with edge padding and the horizontal flip (:107-121), batch_3d (B,chunk,J3,3) (:123-135, may be
 *   null) and batch_cam (B,ncam) (:137-144, may be null).  kps_/joints_ lists: (host). */
int gast_chunk_gather(const float* poses_2d, const float* poses_3d, const float* cameras, const int64_t* seq_start,
                      int32_t n_seq, const int32_t* pairs, int32_t B, int32_t chunk, int32_t pad, int32_t causal_shift,
                      int32_t J2, int32_t F2, int32_t J3, int32_t ncam, int32_t n_sym2, const int32_t* kps_left,
                      const int32_t* kps_right, int32_t n_sym3, const int32_t* joints_left, const int32_t* joints_right,
                      float* batch_2d, float* batch_3d, float* batch_cam, void* stream);

/* tools/mpii_coco_h36m.py: mode 0 = coco_h36m (T,17,2)->(T,17,2) (:20-48), 1 = mpii_h36m (T,16,2)->(T,17,2)
 * (:51-59), 2 = coco_h36m_toe_format (T,J_in>=22,2)->(T,19,2) (:62-78).  valid (T) int32, may be null:
 * 1 where the frame's coordinate sum is non-zero (the mask the reference takes np.where of). */
int gast_keypoints_convert(const float* kpts, float* out, int32_t* valid, int32_t T, int32_t J_in, int32_t mode,
                           void* stream);

/* common/camera.py:8-19: normalize_screen_coordinates (inverse = 0) / image_coordinates (inverse = 1) on
 * n_points (x,y) pairs. */
int gast_normalize_screen(const float* x, float* out, int64_t n_points, float w, float h, int32_t inverse, void* stream);

/* common/camera.py:27-28 camera_to_world with one rotation for all points: qort(q, x) + t
 * (common/quaternion.py:4-18).  q[4], t[3] (host; t may be null = 0). */
int gast_camera_to_world(const float* x, float* out, int64_t n_points, const float* q, const float* t, void* stream);

/* common/loss.py:5-11 mpjpe: *loss = mean_i ||pred_i - target_i|| over n_points rows of D (<= 4) coordinates;
 * when dpred is not null it receives grad_scale * d loss / d pred (the backward of the same pass).
 * workspace: gast_mpjpe_workspace_bytes() bytes of scratch. */
size_t gast_mpjpe_workspace_bytes(void);
int gast_mpjpe(const float* pred, const float* target, int64_t n_points, int32_t D, float* loss, float* dpred,
               float grad_scale, void* workspace, void* stream);

/* common/loss.py:14-53 p_mpjpe: per_frame[n] = mean joint distance of frame n after the similarity
 * (Procrustes) alignment of pred[n] (J,3) to target[n]; the reference's scalar is the mean of per_frame. */
int gast_p_mpjpe(const float* pred, const float* target, int32_t N, int32_t J, float* per_frame, void* stream);

/* optim.Adam(amsgrad=True) (trainval.py:78,162-164) for every parameter in one launch.  table (n_chunks,4)
 * int64 on the device: {param pointer, grad pointer, offset into the flat state buffers, count <=
 * gast_adam_chunk()}.  max_exp_avg_sq null = plain Adam.  step = 1 for the first update. */
int32_t gast_adam_chunk(void);
int gast_adam_step(const int64_t* table, int32_t n_chunks, float* exp_avg, float* exp_avg_sq, float* max_exp_avg_sq,
                   double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step, void* stream);

/* Test/probe entry (not on the forward path): out[M,N] = A[M,K] . W[N,K]^T on one GEMM core
 * (core 0 = tcgen05 TF32 + bf16 corrections, 1 = FFMA, 2 = tcgen05 3xTF32 [training], 3 = tcgen05 fp16 hi + remainder [inference, K >= 256]).  tc_mode != 0 selects a timing-experiment variant of the
 * tcgen05 kernel (parts disabled; results invalid).  Runs once, then `reps` timed launches
 * (CUDA events) whose mean duration is written to *ms_out (host).  Synchronises the stream. */
int gast_debug_gemm(const float* A, const float* W, float* out, int32_t M, int32_t N, int32_t K,
                    int32_t core, int32_t tc_mode, int32_t reps, float* ms_out, void* stream);

const char* gast_last_error(void);
const char* gast_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GAST_B200_H */
