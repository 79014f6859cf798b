/* bc_b200.h -- C ABI of the B200-native behaviour-cloning hot path.
 *
 * The reference (HemuManju/carla-imitation-learning) has no FFI: its hot path is
 * Python calling torch ATen. This header is the boundary a maintainer binds with
 * ctypes (INTEGRATION.md); every entry point names the reference lines it replaces
 * (paths relative to /root/reference).
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*
 *   - the caller owns and allocates every buffer, including workspaces
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises,
 *     nothing allocates, so every call is CUDA-graph capturable
 *   - return 0 on success, negative bc_status on failure; bc_last_error_string() gives
 *     the thread-local message. There is NO CPU fallback: a missing device is an error.
 */
#ifndef BC_B200_H
#define BC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    BC_OK = 0,
    BC_ERR_ARG = -1,      /* bad shape / null pointer / misalignment */
    BC_ERR_DEVICE = -2,   /* no sm_100 device, or a CUDA runtime error */
    BC_ERR_UNSUPPORTED = -3
} bc_status;

/* BC_BF16_TP: bf16 gray planes in the "Toeplitz-ready" layout conv1's tcgen05 kernels consume without a repack:
 * plane[c = R%3][h][q = R/3][g = 0..20][8 px] holds pixels [12g + 8h, 12g + 8h + 8) of image row R (zero for R >= 256);
 * BC_TP_PLANE_ELEMS bf16 per 256x256 plane (1.32x the plain plane: the 16-pixel segments overlap by 4). */
typedef enum { BC_F32 = 0, BC_BF16 = 1, BC_BF16_TP = 2 } bc_dtype;
#define BC_TP_PLANE_ELEMS 86688   /* 3 classes x 2 halves x 86 rows x 21 groups x 8 px */

/* Geometry of ConvNet1 (src/architectures/nets.py:17-33) for 256x256 inputs. */
#define BC_H 256
#define BC_W 256
#define BC_NCONV 4
#define BC_MAX_ACTIONS 16

/* Flat parameter arena: tensors in reverse order of gradient completion
 * [fc.4 fc.2 fc.0 conv4 conv3 conv2 | conv1], weight then bias, each padded to 32 floats.
 * bc_arena_layout fills offsets (in floats) for the 14 tensors in state_dict order
 * cnn_base.{0,3,6,9}.{weight,bias}, fc.{0,2,4}.{weight,bias}; returns the arena length. */
int64_t bc_arena_layout(int obs_size, int n_actions, int64_t offsets[14], int64_t sizes[14]);

/* All device buffers of one training/inference context. The caller fills this once. */
typedef struct {
    int32_t obs_size;        /* input channels (nets.py:11)            */
    int32_t n_actions;       /* logits (nets.py:12)                    */
    int32_t batch;           /* frames in this call                    */
    int32_t x_dtype;         /* bc_dtype of x                          */
    int64_t x_stride_n;      /* element stride between samples of x    */
    int64_t x_stride_c;      /* element stride between channels of x   */
    const void* x;           /* (batch, obs, 256, 256) planar, rows contiguous; may be NULL in bf16 mode (x_tp only) */
    const int64_t* y;        /* (batch,) labels, may be NULL for forward-only  */
    const float* params;     /* parameter arena                        */
    float* grads;            /* gradient arena (same layout)           */
    float* act[4];           /* pooled activations (B,16,28,28) (B,32,12,12) (B,64,4,4) (B,128) */
    uint8_t* amax[4];        /* window-local argmax of each pool, same shapes  */
    float* gact[3];          /* gradients w.r.t. act[0..2] (act[3]'s lives in ghead) */
    float* ghead;            /* (B,128) gradient w.r.t. act[3]          */
    float* hid1;             /* (B,64)  post-ReLU fc.0                  */
    float* hid2;             /* (B,32)  post-ReLU fc.2                  */
    float* logits;           /* (B,n_actions)                           */
    float* dlogits;          /* (B,n_actions) in/out                    */
    float* loss;             /* [1] mean CE                             */
    float* partials;         /* workspace, bc_partials_floats() floats  */
    float loss_scale;        /* dlogits = (softmax-onehot)*loss_scale; 1/batch for the mean */
    int32_t conv_mode;       /* bit mask of tcgen05 (bf16) kernels: 1 forward, 2 dgrad, 4 wgrad conv2-4, 8 wgrad conv1, 16 compact conv1 gradient path (gact0_p8 / amax0_p8, needs 1|2|8); 0 = exact f32 */
    void* w_packed;          /* bc_packed_weight_bytes() bytes: bf16 MMA operand images (bc_pack_weights) */
    int32_t* err_flag;       /* device int: 1 = a bounded mbarrier wait expired, 3 = a label outside [0, n_actions) */
    void* act_bf16[3];       /* bf16 mode: bf16 copies of act[0..2] in the layouts the shifted-window kernels read
                                (csrc/conv_sw.cu, conv4_sw.cu): act1 P8 (B,2,784,8), act2 P8 (B,4,144,8),
                                act3 P8B (8,B,16,8) = [c/8][b][pixel][8]; written by the conv epilogues     */
    void* c1_acc;            /* obs_size 12 in bf16 mode only (else NULL): batch*14*126*64 f32, the raw conv1 accumulators the three
                                camera launches of the tcgen05 conv1 hand to each other (csrc/conv1_tc.cu)                       */
    const void* x_tp;        /* bf16 mode: the input as BC_BF16_TP planes (bc_stage_gray / bc_planes_to_tp); sample n,
                                channel c is the plane at x_tp + n*x_tp_stride_n + c*x_tp_stride_c (elements).
                                stride_n == stride_c is the sliding window: consecutive samples share 3 of 4 planes
                                and conv1 then loads every plane once for 4 samples                              */
    int64_t x_tp_stride_n, x_tp_stride_c;
    const uint32_t* grads_epoch; /* data-parallel peer exchange only (else NULL): device word counting COMPLETED exchanges. The gradient
                                arena is then double-buffered, bc_reduce_partials writes arena ((*grads_epoch + 1) & 1) at
                                grads + that * grads_stride -- the one bc_adam_step_exchange reads next (see bc_peer)           */
    int64_t grads_stride;    /* floats between the two arenas                                                                 */
    void* gact0_p8;          /* conv_mode bit 16: the ReLU-masked gradient w.r.t. act[0] as bf16 in the P8 layout (B,2,784,8), written by
                                conv2's tcgen05 dgrad INSTEAD of gact[0]; conv1's tcgen05 wgrad builds its dY operand from it       */
    uint8_t* amax0_p8;       /* conv_mode bit 16: amax[0] again in the P8 layout (B,2,784,8) u8, written by conv1's tcgen05 forward */
} bc_ctx;

size_t bc_partials_floats(int obs_size, int n_actions);

/* ---- a1: SequentialTorchDataset._load_file/__getitem__ (src/dataset/imitation_dataset.py:115-133)
 * rgb (n,H,W,3) u8 -> gray planes (n,H,W): (0.299R+0.587G+0.114B)/255 evaluated in f64 like
 * numpy, rounded to f32 (or bf16). A sample is 4 consecutive planes, so the sliding window
 * of the reference's shuffle=False loader is the strided view x_stride_n = H*W, x_stride_c = H*W. */
int bc_stage_gray(const uint8_t* rgb, void* gray, int64_t n_pixels, int out_dtype, void* stream);

/* The staging kernel of bf16 mode: rgb (n,256,256,3) u8 -> BC_BF16_TP planes (n * BC_TP_PLANE_ELEMS bf16), and, when
 * plain_bf16 is not NULL, the same gray values also as plain (n,256,256) bf16 planes, in one pass over the frames. */
int bc_stage_gray_tp(const uint8_t* rgb, void* tp, void* plain_bf16, int64_t n_frames, void* stream);

/* EXTENSION (no counterpart in the reference; oracle/ext_oracle.py::stage_augmented): crop + colour jitter + normalise inside the
 * staging pass. rgb (n, src_h, src_w, 3) u8 with src >= 256; table (n, 8) f32 on the device, one row per frame:
 * {crop_y, crop_x, brightness, contrast, saturation, mean, 1/std, -} (host side: data.augment_table(seed, ...)). Output
 * BC_F32 = plain (n,256,256) planes, BC_BF16_TP = Toeplitz-ready bf16 planes. Identity parameters reproduce bc_stage_gray to
 * f32 rounding; the un-augmented kernels stay the bit-exact ones. */
int bc_stage_augment(const uint8_t* rgb, int64_t n_frames, int src_h, int src_w, const float* table, void* out, int out_dtype, void* stream);

/* plain planes (f32 or bf16; 256x256, rows contiguous, `plane_stride` elements apart) -> BC_BF16_TP planes:
 * how a reference-style (B,4,256,256) batch enters the tcgen05 conv1 (bf16 mode) */
int bc_planes_to_tp(const void* planes, int in_dtype, int64_t n_planes, int64_t plane_stride, void* out_tp, void* stream);

/* bf16 tensor-core mode: re-pack the f32 master weights into the smem images the tcgen05 kernels
 * read (conv1: Toeplitz-expanded [64 x 448] bf16). Call after the parameters changed from outside (load_state_dict, a foreign
 * optimiser); bc_adam_tick_step / bc_adam_step_exchange with w_packed keep the images current themselves. */
int bc_pack_weights(const bc_ctx* c, void* stream);
size_t bc_packed_weight_bytes(void);

/* ---- a4-a8: ConvNet1.forward (src/architectures/nets.py:35-39): conv+ReLU+pool x4, MLP.
 * Writes act[], amax[], hid1, hid2, logits. */
int bc_forward(const bc_ctx* c, void* stream);
/* single stages, for unit tests: layer in 0..3 */
int bc_conv_relu_pool_fwd(const bc_ctx* c, int layer, void* stream);
/* head_mode bit0: compute CE loss + dlogits from y (imitation.py:43-44); bit1: backward through the
 * MLP from dlogits (grad partials + ghead). 0 = logits only. */
int bc_head(const bc_ctx* c, int head_mode, void* stream);

/* ---- a9-a10: training_step loss + autograd backward (src/models/imitation.py:38-45).
 * bc_backward assumes bc_forward ran on the same ctx; fills grads (and loss when with_loss). */
int bc_backward(const bc_ctx* c, int with_loss, void* stream);
/* bc_backward with work moved to `side_stream`. ev = 4 caller-owned cudaEvent_t (timing disabled) for the fork/join; capturable.
 * flags bit 1 clear: the weight-gradient kernels of conv4..conv2 run on the side stream under the dgrad chain (wgrad(l) and
 *   dgrad(l) are independent); set: they stay on `stream` (measured on B200: the persistent 148-CTA kernels leave no room, the
 *   overlap gains nothing at N = 1).
 * flags bit 0 clear: everything is joined and reduced on `stream` (like bc_backward). Set (data-parallel overlap): segments
 *   [fc..conv2] are reduced on the SIDE stream, conv1's wgrad is left running on `stream`, nothing is joined -- the caller
 *   launches the bucket-0 exchange on the side stream, then bc_reduce_partials_range(c, 4, 5, ..) + the join itself. */
int bc_backward_overlap(const bc_ctx* c, int with_loss, void* stream, void* side_stream, void* const* ev, int flags);
int bc_conv_bwd_dgrad(const bc_ctx* c, int layer, void* stream);   /* layer 1..3 -> gact[layer-1] */
int bc_conv_bwd_wgrad(const bc_ctx* c, int layer, void* stream);   /* layer 0..3 -> partials      */
int bc_reduce_partials(const bc_ctx* c, int with_loss, void* stream); /* partials -> grads (, loss) */
/* gradient segments in arena order: 0 = fc head, 1 = conv4, 2 = conv3, 3 = conv2, 4 = conv1; the
 * data-parallel exchange reduces [0,4) first so its all-reduce overlaps conv1's wgrad (SURVEY 8e) */
int bc_reduce_partials_range(const bc_ctx* c, int seg_lo, int seg_hi, int with_loss, void* stream);
int bc_loss_reduce(const bc_ctx* c, void* stream);                 /* head CTAs' CE partials -> loss (forward-only / validation_step) */

/* ---- Launch ordering contract (programmatic dependent launch). Every kernel of this library is launched with programmatic
 * stream serialisation. Kernels that READ parameters -- the conv / dgrad kernels (their bf16 operand images in w_packed), the
 * head (fc weights), the branched heads (bc_head_branched: the commanded branch's weights in the branch arena) and the
 * optimiser kernels (params, moments, state) -- fetch them BEFORE griddepcontrol.wait, under the previous kernel's tail. That is sound because the kernels that WRITE parameters, moments, state or w_packed (bc_adam_step,
 * bc_adam_tick_step, bc_adam_step_exchange, bc_pack_weights) release their dependents only after their last write. A caller
 * that writes these buffers itself must do so with ordinary (fully serialising) launches or copies -- torch ops are --
 * and never from a kernel of its own that calls griddepcontrol.launch_dependents before its last write. The same holds for
 * the command vector of the branched serving tail (bc_policy_tail_branched), which reads command[b] before its wait: no
 * kernel of this library writes it. */

/* ---- a11: Adam.step (src/models/imitation.py:82-87; torch.optim.Adam defaults).
 * state = 8 DOUBLES {lr, beta1, beta2, eps, step, grad_scale, step_size(out), bc2_sqrt(out)} on the
 * device; bc_adam_tick increments step and derives the bias corrections in f64 like torch's Python
 * scalars do (graph-replayable: nothing about the step number lives on the host). */
int bc_adam_tick(double* state, void* stream);
int bc_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                 const double* state, int64_t n, void* stream);
/* tick + step in ONE launch (what the training step uses): state9 = the 8 doubles above + one more word used as a CTA counter.
 * w_packed != NULL (bf16 mode, obs_size 4; n must be the arena of (obs_size, n_actions)): the kernel also rewrites the bf16
 * MMA operand images of the conv weights it has just updated, so the step needs no bc_pack_weights launch. */
int bc_adam_tick_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, double* state9, int64_t n,
                      void* w_packed, int obs_size, int n_actions, void* stream);

/* ---- a12 folded into a11: the DDP gradient mean (train.py:125 `pl.Trainer(gpus=[...])`, utils.py:60-64) inside the Adam step.
 * bc_peer: peer_grads_dev / peer_signals_dev are DEVICE arrays of `world` pointers -- rank r's gradient arenas (TWO arenas of n
 * floats back to back: step e uses arena e & 1) and signal pad mapped into this process (peer memory over NVLink; torch
 * symmetric memory provides both). sync_state: 4 device u32 {completed epochs, CTA counter, -, -}, zero-initialised, private to
 * the rank; bc_ctx.grads_epoch points at its first word. *err_flag = 2 if a peer never arrived (parameters are then left alone).
 * Each rank launches the exchange once per bucket and step after that bucket's gradients are complete: flag exchange, sum of the
 * `world` arenas in rank order read straight from peer memory, Adam update of floats [lo, hi) with state[5] = grad_scale =
 * 1/world. bucket 0 = [fc..conv2] (launched on a side stream under conv1's wgrad, publish = 0), bucket 1 = conv1 or the whole
 * arena (publish = 1: the tick -- do NOT call bc_adam_tick -- and the epoch are published by its last CTA; launch it after
 * bucket 0 has completed). */
typedef struct {
    const void* peer_grads_dev;
    const void* peer_signals_dev;
    uint32_t* sync_state;
    int32_t* err_flag;
    int32_t rank, world;
} bc_peer;
int bc_adam_step_exchange(float* params, float* exp_avg, float* exp_avg_sq, double* state9, int64_t n, const bc_peer* peer,
                          int64_t lo, int64_t hi, int bucket, int publish, void* w_packed, int obs_size, int n_actions, void* stream);

/* ---- K12: Imitation.forward + argmax (imitation.py:34-36, src/data/stat.py:41). Every greedy action of this library
 * (bc_argmax, bc_forward_act on both paths) follows torch.argmax: the index of the first NaN of the row if it has one (NaN
 * counts as the maximum), else the index of the first maximum (ties go to the lowest index; a row of -inf gives 0). */
int bc_argmax(const float* logits, int64_t* actions, int batch, int n_actions, void* stream);

/* ---- K13: the policy forward for closed-loop serving (BASELINE configs[4]; imitation.py:34-36 + the argmax of
 * src/data/stat.py:41), greedy actions (batch) int64 out, no separate argmax launch.
 * bc_forward_act, tail = 0: bc_forward with the action taken inside the head kernel (torch.argmax's rule, K12 above: the
 *   first NaN, else the first maximum; the same on both paths).
 * tail = 1 (batch <= BC_POLICY_TAIL_MAX_BATCH; faster up to batch 8 on B200, where the forward is a chain of launch latencies):
 *   conv1, conv2 as in bc_forward, then bc_policy_tail = conv3 + ReLU + pool, conv4 + ReLU + pool, the three Linear layers and the
 *   argmax in ONE launch (an 8-CTA thread-block cluster per sample, exact f32 FFMA on the f32 master weights in both modes,
 *   layers handed over through distributed shared memory). bc_policy_tail reads act[1] ((batch,32,12,12) f32, written by
 *   bc_conv_relu_pool_fwd(layer 1) in both modes) and params; writes logits and actions, and act[2], act[3], hid1, hid2 when
 *   those pointers are not NULL (amax[2], amax[3] are NOT written: inference only). */
#define BC_POLICY_TAIL_MAX_BATCH 64
int bc_forward_act(const bc_ctx* c, int64_t* actions, int tail, void* stream);
int bc_policy_tail(const bc_ctx* c, int64_t* actions, void* stream);

/* v[0..n) *= *scale_dev (a device scalar), nothing is touched when it is exactly 1: how `loss.backward(gradient=g)` reaches
 * gradients that the fused step has already computed for d loss (imitation.py:38-45 returns the loss, Lightning calls backward) */
int bc_scale_inplace(float* v, int64_t n, const float* scale_dev, void* stream);

/* ---- EXTENSION (no counterpart in the reference; oracle/ext_oracle.py): command-conditioned branched heads.
 * G branches of the reference's MLP shape 128 -> 64 -> 32 -> n_out (nets.py:31-33 has ONE such head); sample b is evaluated by
 * branch command[b] only (branch-select mask). loss_kind 0 = CrossEntropy on labels (imitation.py:43-44), 1 = L1, 2 = MSE on
 * (B, n_out) regression targets (steer, throttle, brake), mean reduction: pass loss_scale = 1/B (CE) or 1/(B*n_out).
 * params / grads: G x head_len floats, per branch in the order of the arena's head segment [fc.4 w,b | fc.2 w,b | fc.0 w,b]
 * (bc_head_branched_layout gives the per-branch offsets in state_dict order 0.weight 0.bias 2.weight 2.bias 4.weight 4.bias).
 * feat = bc_ctx.act[3] of the conv trunk, gfeat = bc_ctx.ghead for the trunk's backward. mode bit0: loss + dout from
 * labels/targets; bit1: backward from dout (grads, gfeat); 0 = outputs only. A command outside [0, n_branches) sets
 * *err_flag = 4 and leaves zeros in that sample's rows: out, dout (bit0) and gfeat (bit1), so the sample adds nothing to the
 * trunk's backward and no stale gradient row reaches it. */
typedef struct {
    int32_t n_branches, n_out, batch, loss_kind;
    const float* feat;        /* (B,128)                               */
    const int64_t* command;   /* (B,) in [0, n_branches)               */
    const int64_t* labels;    /* (B,) class ids (CE) or NULL           */
    const float* targets;     /* (B,n_out) (L1/MSE) or NULL            */
    const float* params;
    float* grads;
    float* out;               /* (B,n_out) outputs of the commanded branch */
    float* dout;              /* (B,n_out) d loss / d out, in/out      */
    float* gfeat;             /* (B,128)                               */
    float* loss;              /* [1]                                   */
    float* partials;          /* bc_head_branched_partials_floats() floats */
    int32_t* err_flag;        /* 3 = label out of range, 4 = command out of range */
    float loss_scale;
} bc_branched;
int bc_head_branched(const bc_branched* h, int mode, void* stream);
size_t bc_head_branched_partials_floats(int n_branches, int n_out);
int64_t bc_head_branched_layout(int n_out, int64_t offsets[6], int64_t sizes[6]);

/* ---- K13 for the branched heads: the serving forward of ConvNet1Branched (conditional imitation: the route planner's
 * command picks the branch per sample, per simulator tick). c = the trunk's context (params, act[], x as for bc_forward_act;
 * act[2], act[3], hid1, hid2 are written when not NULL), h = the branch arena (params, 16 B aligned), command, out ((batch,
 * n_out) f32: the commanded branch's outputs) and err_flag; h->feat, labels, targets, grads, dout, gfeat, loss and partials
 * are not used. h->batch must equal c->batch. actions (batch,) int64 or NULL: the greedy action over out (CE-trained
 * branches; torch.argmax's rule, K12). A command outside [0, n_branches) sets *err_flag = 4 and leaves a zero out row and
 * action 0; no branch outside the arena is read.
 * tail = 0: conv1..conv4, then the branched head kernel (bc_head_branched mode 0) with the action taken inside it.
 * tail = 1 (batch <= BC_POLICY_TAIL_MAX_BATCH): conv1, conv2, then bc_policy_tail_branched = bc_policy_tail with CTA 0 of
 *   sample b's cluster loading branch command[b]'s fc.0, fc.2, fc.4 instead of the trunk's fc; same shared memory, same
 *   arithmetic. The tail reads command[b] BEFORE griddepcontrol.wait, with the weights (launch ordering contract above: no
 *   kernel of this library writes the command vector; the caller writes it with ordinary stream-ordered work -- a host
 *   copy, a torch op -- which has completed when the tail starts, because every kernel of this library waits for its
 *   predecessor before it releases its dependents). */
int bc_forward_branched_act(const bc_ctx* c, const bc_branched* h, int64_t* actions, int tail, void* stream);
int bc_policy_tail_branched(const bc_ctx* c, const bc_branched* h, int64_t* actions, void* stream);

/* ---- self-test of the tcgen05/TMEM primitives the bf16 conv kernels are built from:
 * D[M,N] f32 = A[M,K] bf16 * B[N,K]^T bf16 (K contiguous). *err_flag is set to 1 if an mbarrier
 * wait timed out (bounded waits: a protocol bug is an error code, not a hung GPU). */
int bc_tc_gemm_selftest(const void* A, const void* B, float* D, int M, int N, int K, int* err_flag, void* stream);

/* cycles for `reps` back-to-back tcgen05.mma (M=128,K=16,bf16) of width N: cycles2[0] = issue, [1] = completion */
int bc_tc_mma_bench(int N, int reps, int mode, int grid, long long* cycles2, int* err_flag, void* stream);

const char* bc_last_error_string(void);
int bc_device_check(void);  /* BC_OK iff the current device is sm_100 */
int bc_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BC_B200_H */
