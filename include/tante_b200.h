/*
 * tante_b200.h -- C ABI of the B200-native TANTE hot path (libtante_b200.so).
 *
 * Plain C: opaque handle, raw device pointers, sizes, CUDA stream as void*.
 * No torch / C++ types cross this boundary.  Every entry point returns an int
 * status (0 = TANTE_OK); tante_last_error() gives the thread-local message.
 * The library allocates only in tante_create / tante_reserve (workspace,
 * packed-weight arena, rollout state, CUDA graphs); it never owns parameters,
 * gradients, inputs or outputs -- the caller (PyTorch) does.  All work is
 * enqueued on the caller's stream; the only host syncs are the documented
 * ones (tante_forward with n_host != NULL, tante_rollout with sync != 0).
 * A handle is single-threaded: one per process per GPU.
 *
 * The reference (zwu88/TANTE) is pure Python; nothing native exists to mirror,
 * so each entry point cites the Python call it replaces (paths under the
 * reference root).
 */
#ifndef TANTE_B200_H_
#define TANTE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define TANTE_API __attribute__((visibility("default")))
#else
#define TANTE_API
#endif

#define TANTE_OK 0
#define TANTE_ERR_INVALID 1   /* bad argument / unsupported configuration        */
#define TANTE_ERR_CUDA 2      /* a CUDA runtime call failed                      */
#define TANTE_ERR_STATE 3     /* call order violated (e.g. params not bound)     */
#define TANTE_ERR_NOMEM 4

#define TANTE_MAX_ORDER 8
#define TANTE_MAX_LAYERS 32

#define TANTE_PREC_FP32 0  /* FP32 FFMA everywhere: the <=1e-5 parity mode                    */
#define TANTE_PREC_BF16 1  /* bf16 operands on tcgen05 tensor cores, fp32 accumulate/residual */

/* Mirror of the TANTE constructor (models/tante.py:38-60) + dataset metadata
 * (n_fields, spatial_resolution: models/tante.py:64-66). */
typedef struct tante_config {
    int32_t in_T;
    int32_t n_fields;
    int32_t H, W;
    int32_t taylor_order;
    int32_t n_head;
    int32_t embed_dim;
    int32_t patch_scale;
    int32_t deg;            /* 1: fixed step (output_length frames), 0: adaptive   */
    int32_t output_length;
    float frame_interval;
    int32_t precision;      /* TANTE_PREC_*                                         */
    int32_t n_layers[TANTE_MAX_ORDER];                 /* len(segment k) of attn_axes */
    char axes[TANTE_MAX_ORDER][TANTE_MAX_LAYERS];      /* axis letter per layer: T / H / W / L / Y / A / C          */
    int32_t enc_dec_fno;    /* 0: enc_dec_type='cnn' (enc_dec_cnn.py), 1: 'fno' (enc_dec_fno.py; inference / rollout) */
    int32_t modes1, modes2; /* SpectralLayer modes of the fno encoder / decoder (models/tante.py:56-57)            */
    int32_t mlp_hidden;     /* int(embed_dim * mlp_ratio) of the block MLP (attn_backbone.py:52); 0 = embed_dim; multiple of 64, <= 1024 */
    int32_t expanded_channel; /* width E of the axis-'C' blocks (models/tante.py:47, attn_backbone.py:124-130); 0 = 128; multiple of 64, <= 256 */
    int32_t mlp_hidden_c;   /* int(expanded_channel * mlp_ratio): MLP width of the axis-'C' blocks; 0 = expanded_channel */
    int32_t stride[3];      /* overlap_ratio != 0 (enc_dec_cnn.py:64-66): stride of the three patch stages, max(1, round(k * (1 - r))); 0 = k (no overlap) */
} tante_config_t;

typedef struct tante_handle_s* tante_handle_t;

/* ---- lifecycle ------------------------------------------------------------------ */
TANTE_API const char* tante_last_error(void);
TANTE_API int tante_version(void);

/* models.TANTE(...) construction (models/tante.py:37-123).  Validates the config
 * (ValueError/KeyError cases of tante.py:76-83, enc_dec_cnn.py:199 map to
 * TANTE_ERR_INVALID). */
TANTE_API int tante_create(const tante_config_t* cfg, int device, tante_handle_t* out);
TANTE_API int tante_destroy(tante_handle_t h);

/* (Re)size the library-owned workspace for batches up to max_batch and rollouts up
 * to max_roll frames.  Called by the host module before the first forward/rollout
 * of a new size; the only allocating call besides tante_create. */
TANTE_API int tante_reserve(tante_handle_t h, int32_t max_batch, int32_t max_roll, int32_t training);
TANTE_API int64_t tante_workspace_bytes(tante_handle_t h);

/* ---- parameters: state_dict ABI (SURVEY.md §8(b)) -------------------------------- */
TANTE_API int32_t tante_param_count(tante_handle_t h);
TANTE_API const char* tante_param_name(tante_handle_t h, int32_t i);
TANTE_API int64_t tante_param_numel(tante_handle_t h, int32_t i);
/* model.parameters()/load_state_dict (trainer/r_trainer.py:102, r_evaler.py:82): the
 * fp32 master tensor stays owned by the caller; `grad` may be NULL (inference). */
TANTE_API int tante_bind_param(tante_handle_t h, const char* name, const float* data, float* grad, int64_t numel);
/* Re-derive the packed device weights (GEMM-ready layouts, bf16 copies) from the bound
 * masters.  Call after binding and after every optimizer step. */
TANTE_API int tante_pack_params(tante_handle_t h, void* stream);

/* ---- one model step: TANTE.forward (models/tante.py:125-176) ---------------------- */
/* input  : f32[B, T, D, H, W] (already cropped to the last in_T frames)
 * frames : f32[B, n_cap, D, H, W]; sample b gets n_b frames written, the rest untouched
 * R_t    : f32[B] (adaptive only, may be NULL when deg)
 * n_dev  : i32[B] device array of emitted frame counts (may be NULL)
 * n_host : if non-NULL the call synchronises the stream and stores n for sample 0 --
 *          the reference's own `math.floor(R_t[0])` host sync (tante.py:163).
 * per_sample = 0 reproduces the reference (sample 0 governs the batch);
 * per_sample = 1 gives every sample its own n = floor(R_t[b]). */
TANTE_API int tante_forward(tante_handle_t h, const float* input, int32_t B, float out_T, int32_t n_cap,
                  int32_t per_sample, float* frames, float* R_t, int32_t* n_dev, int32_t* n_host,
                  void* stream);

/* ---- adaptive rollout: R_Evaler.rollout_model (trainer/r_evaler.py:87-105),
 *      R_Trainer.rollout_model in eval mode (trainer/r_trainer.py:112-133),
 *      Evaler/Trainer.rollout_model for deg (trainer/evaler.py:121-138) ------------- */
/* window   : f32[B, T, D, H, W] channels-first initial frames (read only)
 * y_out    : f32[B, n_roll, H, W, D] channels-last (DefaultChannelsFirstFormatter.process_output)
 * rts_out  : f32[max_steps, B] R_t per model call (row s valid for samples with steps_out[b] > s)
 * ns_out   : i32[max_steps, B] frames emitted per model call
 * steps_out: i32[B] number of model calls each sample took
 * max_steps = n_roll (every call emits >= 1 frame).
 * The whole loop runs on the device (ring-buffer window, per-sample counters, one CUDA
 * graph per step); `sync` != 0 makes the call return after the rollout finished. */
TANTE_API int tante_rollout(tante_handle_t h, const float* window, int32_t B, int32_t n_roll, float out_T,
                  int32_t per_sample, float* y_out, float* rts_out, int32_t* ns_out,
                  int32_t* steps_out, int32_t sync, void* stream);

/* ---- training: taped forward + backward ---------------------------------------------
 * The reference trains through torch autograd over the same module (trainer/r_trainer.py:145-155:
 * rollout_model -> loss -> loss.backward(); fixed-step twin trainer/trainer.py:178-193).  Here one
 * model call in grad mode = tante_train_forward (keeps the activations in tape slot `slot`), and
 * its autograd node's backward = tante_backward on the same slot.  Slots are reserved with
 * tante_reserve(.., training = number of slots); a chained rollout with BPTT through the window
 * (r_trainer.py:126) holds one slot per model call until its backward ran.
 *
 * tante_train_forward: same contract as tante_forward with per_sample = 0 (sample 0's R_t governs
 *   n, tante.py:163); n_host (nullable) = the reference's host sync for floor(R_t[0]).
 * tante_backward:
 *   input       : the f32[B,T,D,H,W] tensor the forward saw (the first conv's weight gradient reads it)
 *   grad_frames : f32[B, n_frames, D, H, W] gradient of the emitted frames (n_frames <= the forward's n)
 *   grad_Rt     : f32[B] gradient of R_t (adaptive models; NULL = zero)
 *   grad_input  : f32[B,T,D,H,W], written (may be NULL when the input needs no gradient)
 *   grad_params : f32[tante_grad_numel()], written: parameter i's gradient in its state_dict layout
 *                 at tante_param_grad_offset(i) (the caller hands these views to autograd, which
 *                 accumulates into .grad -- so gradient accumulation and BPTT just work). */
/* Dropout of the NEXT taped forwards (nn.Dropout / nn.MultiheadAttention(dropout=p) inside TransformerBlock,
 * models/attn_backbone.py:47-57,81-83; p = 0.1 in configs/tante.yaml:29): p = 0 disables it.  `seed` keys the counter-based
 * mask generator for the call; the host draws a fresh one per model call (torch's generator), the tape remembers it and
 * tante_backward regenerates the same masks.  tante_forward / tante_rollout never drop (model.eval() semantics). */
TANTE_API int tante_set_dropout(tante_handle_t h, float p, uint64_t seed);
TANTE_API int64_t tante_grad_numel(tante_handle_t h);
TANTE_API int64_t tante_param_grad_offset(tante_handle_t h, int32_t i);
TANTE_API int tante_train_forward(tante_handle_t h, int32_t slot, const float* input, int32_t B, float out_T,
                        int32_t n_cap, float* frames, float* R_t, int32_t* n_host, void* stream);
TANTE_API int tante_backward(tante_handle_t h, int32_t slot, const float* input, const float* grad_frames,
                   int32_t n_frames, const float* grad_Rt, float* grad_input, float* grad_params, void* stream);

/* Frame-table variants of the two calls above for the chained BPTT rollout of the training drivers (trainer/trainer.py:144-159,
 * trainer/r_trainer.py:122-126: window = cat(window[:, n:], y), NOT detached): the window of a call is given as in_T separate
 * frames -- frame_ptrs[t] = device pointer of frame t of sample 0 (a contiguous (D, H, W) plane set, 16-byte aligned),
 * sample b at + b * frame_bstride[t] elements -- so that consecutive calls slide over ONE history buffer and no window is ever
 * concatenated; the emitted frames go to frames + b * frames_bstride (+ i * D * H * W).  tante_backward_win reads the frame
 * gradients with batch stride gf_bstride and ACCUMULATES (+=) the window gradient into grad_frame_ptrs[t] + b * grad_bstride[t]
 * (NULL entry: that frame needs no gradient; grad_frame_ptrs == NULL: none does), which is how BPTT sums the contributions of
 * later calls into the gradient of an earlier prediction in place. */
TANTE_API int tante_train_forward_win(tante_handle_t h, int32_t slot, const float* const* frame_ptrs,
                                      const int64_t* frame_bstride, int32_t B, float out_T, int32_t n_cap, float* frames,
                                      int64_t frames_bstride, float* R_t, int32_t* n_host, void* stream);
TANTE_API int tante_backward_win(tante_handle_t h, int32_t slot, const float* grad_frames, int64_t gf_bstride, int32_t n_frames,
                                 const float* grad_Rt, float* const* grad_frame_ptrs, const int64_t* grad_bstride,
                                 float* grad_params, void* stream);

/* Per-sample cursor variants of the pair above for the adaptive BPTT rollout of R_Trainer (trainer/r_trainer.py:117-133, each
 * sample its own step sequence, the window NOT detached), the whole batch in one call.  Sample b's history is its input window
 * input = f32 (B, in_T, D, H, W) (contiguous, 16-byte aligned) followed by its predictions pred + b * pred_bstride (+ j * D * H * W
 * for prediction j).  cursor = device i32[B], the frames each sample has emitted (zero before the first call): window frame t of
 * sample b is history frame cursor[b] + t.  The call emits n_b = min(floor(R_t), n_cap) frames of sample b (n_cap = floor(out_T +
 * 0.001) as in tante_forward) to pred[b, cursor[b] ..], or none once cursor[b] >= n_steps; pred must hold n_steps + n_cap - 1
 * frames per sample so that an overshooting last call stays inside it.  Then it advances the cursor by n_b and, all on the
 * device: R_t = f32[B] the call's R_t (0 where n_b = 0), ns = i32[B] n_b, steps = i32[B] += (n_b > 0), n_active (nullable, device
 * i32[1]) = samples still short of n_steps.  Nothing is synchronised.  The tape keeps the cursor the call saw.
 * tante_backward_hist reads the gradient of this call's frames from grad_pred (batch stride gp_bstride, same frame positions as
 * pred; positions past n_steps must hold zeros), takes grad_Rt = f32[B] (nullable; entries with n_b = 0 must be zero), and
 * ACCUMULATES (+=) the window gradient into grad_pred (predictions) and grad_input (input window, f32 (B, in_T, D, H, W);
 * NULL: not wanted).  Coverage as the _win pair. */
TANTE_API int tante_train_forward_hist(tante_handle_t h, int32_t slot, const float* input, float* pred, int64_t pred_bstride,
                                       int32_t* cursor, int32_t B, float out_T, int32_t n_cap, int32_t n_steps, float* R_t,
                                       int32_t* ns, int32_t* steps, int32_t* n_active, void* stream);
TANTE_API int tante_backward_hist(tante_handle_t h, int32_t slot, float* grad_pred, int64_t gp_bstride, const float* grad_Rt,
                                  float* grad_input, float* grad_params, void* stream);

/* ---- introspection for tests / profiling ------------------------------------------ */
/* Copy an internal stage tensor of the last tante_forward into `dst` (f32, device).
 * stage: "latent_in" (after embed), "latent" (after the last backbone), "deriv<k>"
 * ([B,D,H,W] decoded k-th derivative field), "rt<k>".  Returns the element count in *numel. */
TANTE_API int tante_debug_stage(tante_handle_t h, const char* stage, float* dst, int64_t cap, int64_t* numel,
                      void* stream);
/* Number of kernel launches enqueued by this handle since creation (bench.py's gpu_launches). */
TANTE_API int64_t tante_launch_count(tante_handle_t h);

/* Stand-alone launches of the fused Taylor head (K stage-1 activation matrices -> n_frames frames per
 * sample) for the K x patch-size microbenchmark (BASELINE.json configs[4]).  Uses the handle's own
 * stage-1 buffers (whatever they hold), `u` = f32[B,T,D,H,W] window, `frames` = f32[B,n_frames,D,H,W].
 * Runs `iters` launches between two CUDA events and returns the average in *ms_out (synchronises). */
TANTE_API int tante_bench_head(tante_handle_t h, const float* u, float* frames, int32_t B, int32_t n_frames,
                     int32_t iters, float* ms_out, void* stream);

/* Live per-kernel-class timing for bench.py's roofline: while enabled, every GEMM launch of this handle
 * is bracketed by CUDA events on the launching stream (un-graphed launches).  tante_profile_read
 * synchronises, returns the summed GEMM device time, the algorithmic FLOPs (2*M*N*K per launch) and the
 * launch count since enabling, and clears the counters. */
TANTE_API int tante_profile(tante_handle_t h, int32_t enable);
TANTE_API int tante_profile_read(tante_handle_t h, double* gemm_ms, double* gemm_flops, int64_t* gemm_launches);
/* Same tally split by roofline class (call BEFORE tante_profile_read, which resets it): cls 0 = GEMMs with a plain
 * bf16 / activation epilogue (tensor-bound), 1 = GEMMs with an fp32 residual / LayerNorm / embedding epilogue
 * (HBM-bound), 2 = weight-gradient GEMMs (HBM-bound).  bytes = algorithmic HBM bytes (operands + outputs once). */
TANTE_API int tante_profile_read_class(tante_handle_t h, int32_t cls, double* ms, double* flops, double* bytes,
                                       int64_t* launches);

/* Training loss of the rollout drivers (reference trainer/metrics.py:53-80, MSE.eval(...).mean(), as called from
 * trainer/trainer.py:188-190 and trainer/r_trainer.py:150-152) between the module's channels-first predictions
 * y = f32[B,nf,D,H*W] and the channels-last targets ref = f32[B,n_ref,H*W,D], frames f0 .. f0+n_use-1 (n_use <= nf: the
 * rollout drivers truncate an overshooting last call).  loss_sum (nullable, f32[1]) += sum of squared differences;
 * grad_y (nullable, f32 like y) = scale * (*gout, or 1 when gout is null) * (y - ref), zero for frames >= n_use.
 * No handle: a pure function of its arguments, launched on `stream`. */
TANTE_API int tante_mse_cl(const float* y, const float* ref, int32_t B, int32_t nf, int32_t n_use, int32_t D, int64_t HW,
                 int32_t n_ref, int32_t f0, float scale, const float* gout, float* loss_sum, float* grad_y, void* stream);

/* Evaluation metrics of the rollout drivers (reference trainer/metrics.py:53-164: MSE, NMSE, L2RE, NNMSE, RMSE, NRMSE,
 * VMSE, VRMSE as called from trainer/r_evaler.py:134-137, trainer/evaler.py:203-206): ONE pass over the channels-last
 * prediction x and target y = f32[BT, HW, C] producing the three spatial moments every one of those metrics is built from,
 * out = f64[BT, C, 3] = { sum (x-y)^2, sum y^2, sum y } over HW (written, not accumulated).  No handle: a pure function of
 * its arguments, launched on `stream` on the device that owns x. */
TANTE_API int tante_metric_moments(const float* x, const float* y, int64_t BT, int64_t HW, int32_t C, double* out,
                                   void* stream);

/* ---- optimizer tail of a training step (SURVEY.md 8(b) `allreduce_grads`; reference trainer/trainer.py:192-198,
 *      trainer/r_trainer.py:155-157: clip_grad_norm_ / clip_grad_value_ + torch.optim.AdamW.step) ------------------------
 * All three work on the FLAT gradient of tante_backward (f32[tante_grad_numel()], parameter i at tante_param_grad_offset(i)).
 *
 * tante_comm_unique_id : rank 0 fills id128 (128 bytes, ncclGetUniqueId); the host side broadcasts it.
 * tante_comm_init      : every rank, collectively: ncclCommInitRank on the handle's device; the communicator lives in the handle.
 * tante_allreduce_grads: in-place SUM all-reduce of the flat gradient on `stream` over `comm` (an ncclComm_t; NULL = the
 *                        handle's own).  NCCL is the copy already loaded in the process (dlopen, no link-time dependency).
 * tante_optimizer_step : g = grad * grad_scale (1 / world size after the sum); clip_mode 1: g *= min(1, clip / (||g||_2 + 1e-6))
 *                        over ALL parameters (clip_grad_norm_), 2: clamp to [-clip, clip] (clip_grad_value_), 0: none; then
 *                        AdamW (decoupled weight decay, bias correction with `step` counted from 1) on every parameter
 *                        through its bound master pointer, moments in the caller-owned flat buffers exp_avg / exp_avg_sq
 *                        (laid out like the gradient).  The clipped gradient is written back to `grad`; grad_sumsq (nullable,
 *                        f64[1], device) receives sum g^2 before clipping.  Follow with tante_pack_params. */
TANTE_API int tante_comm_unique_id(void* id128);
TANTE_API int tante_comm_init(tante_handle_t h, const void* id128, int32_t nranks, int32_t rank);
TANTE_API int tante_allreduce_grads(tante_handle_t h, float* grad, void* comm, void* stream);
TANTE_API int tante_optimizer_step(tante_handle_t h, float* grad, float* exp_avg, float* exp_avg_sq, float lr, float beta1,
                                   float beta2, float eps, float weight_decay, int64_t step, int32_t clip_mode, float clip,
                                   float grad_scale, double* grad_sumsq, void* stream);

/* Test hook: run one GEMM of the library stand-alone, C[M,N] = epi(A[M,K] * W[N,K]^T + bias).
 * use_tc = 1: tcgen05 bf16 kernel (A, W bf16; C bf16 when out_bf16 else f32);
 * use_tc = 0: FFMA fp32 kernel (A, W, C f32).  epi: 0 bias, 1 +relu, 2 +gelu(erf), 3 +gelu(tanh),
 * 4 + resid (f32 [M,N], may alias C), 6 = 4 plus LayerNorm(gamma, beta, eps 1e-5) of the updated row into
 * ln_out (bf16 [M,N]; tcgen05 kernel only, N == 256).  iters > 1 repeats the launch. */
TANTE_API int tante_test_gemm(int32_t use_tc, int32_t epi, const void* A, const void* W, const float* bias,
                    const float* resid, void* C, int32_t out_bf16, int32_t M, int32_t N, int32_t K,
                    int32_t iters, const float* ln_gamma, const float* ln_beta, void* ln_out, void* stream);

/* Test hook: the fused block tail (block_tail_tc.cuh; reference attn_backbone.py:81-83 + the next layer's LayerNorm) stand-alone:
 *   x_mid = x_in + att Wo^T + bo;  h = gelu_tanh(LN(x_mid; g2, be2) W1^T + b1);  x_out = x_mid + h W2^T + b2;
 *   ln_out = LN(x_out; gn, ben)   (skipped when ln_out is NULL).
 * att bf16[M,256]; Wo, W1, W2 bf16[256,256] (nn.Linear layout); vec7 = f32[7][256] = bo, g2, be2, b1, b2, gn, ben; x_in / x_out
 * f32[M,256] (may alias).  x_mid (f32) / ln2 / hpre / hact (bf16) all non-NULL select the training variant, which stores them. */
TANTE_API int tante_test_block_tail(const void* att, const void* Wo, const void* W1, const void* W2, const float* vec7,
                                    const float* x_in, float* x_out, void* ln_out, float* x_mid, void* ln2, void* hpre,
                                    void* hact, int32_t M, int32_t iters, void* stream);

/* Test hook: weight-gradient GEMM stand-alone, C[N,K] += A[M,N]^T * B[M,K] (C is accumulated into).
 * use_tc = 1: tcgen05 kernel (bf16 MN-major operands, TMA reduce-add), 2: SIMT kernel on bf16 operands,
 * 0: SIMT kernel on f32 operands.  `bias` (nullable, tcgen05 kernel only): f32[N] += column sums of A. */
TANTE_API int tante_test_wgrad(int32_t use_tc, const void* A, const void* B, float* C, float* bias, int64_t M, int32_t N,
                     int32_t K, int32_t iters, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TANTE_B200_H_ */
