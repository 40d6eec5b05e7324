/* b200mdm.h -- C ABI of libb200mdm.so: the B200 (sm_100a) sampling engine that replaces the per-step hot path of
 * GuyTevet/motion-diffusion-model (paths below are relative to the reference repository root).
 *
 * The reference is pure Python, so there is no existing FFI to mirror; each entry point states which
 * reference function(s) it replaces.  The Python host mirror (motion-diffusion-model_b200/) binds these with
 * ctypes (see INTEGRATION.md) and passes torch tensors as raw pointers (`tensor.data_ptr()`), the CUDA stream
 * as `torch.cuda.current_stream().cuda_stream`.
 *
 * Conventions
 *   - every function returns 0 on success, a negative B200MDM_E* code on failure; b200mdm_last_error() returns a
 *     thread-local description of the most recent failure;
 *   - pointers named *_dev are device pointers, *_host host pointers; no ownership is transferred;
 *   - tensors use the reference's layouts: motion x [B, njoints, nfeats, T] fp32 (T contiguous),
 *     text embedding [B, cond_dim] fp32 (the reference's [1, B, C] with the leading 1 dropped);
 *   - nothing allocates on the per-step path: b200mdm_set_cond selects the workspace of a (B, T, CFG) triple -- built
 *     on first use, then kept (with its captured step graph) in a small pool;
 *   - kernels are specialised for latent_dim 512, 4 heads of 128 and sequences of at most 256 tokens (every released
 *     MDM / DiP model; 196 frames + 1 token); other shapes -> B200MDM_ENOTIMPL;
 *   - no call synchronises the stream except where stated.
 */
#ifndef B200MDM_H_
#define B200MDM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200MDM_OK 0
#define B200MDM_EINVAL (-1)   /* contract violation (the reference raises AssertionError / ValueError) */
#define B200MDM_ECUDA (-2)    /* CUDA runtime / driver error */
#define B200MDM_ESTATE (-3)   /* call order violated (weights not finalised, schedule / cond missing ...) */
#define B200MDM_ENOTIMPL (-4) /* configuration the engine does not implement (reference: NotImplementedError) */

#define B200MDM_ARCH_TRANS_ENC 0
#define B200MDM_ARCH_TRANS_DEC 1

#define B200MDM_COND_NONE 0
#define B200MDM_COND_TEXT 1
#define B200MDM_COND_ACTION 2

#define B200MDM_MODE_X0 0   /* model output only */
#define B200MDM_MODE_DDPM 1 /* p_sample */
#define B200MDM_MODE_DDIM 2 /* ddim_sample */

#define B200MDM_FLAG_CONST_NOISE 1   /* p_sample(const_noise=True): eps row 0 repeated (gaussian_diffusion.py:527-528) */
#define B200MDM_FLAG_CLIP_DENOISED 2 /* clip_denoised=True: clamp x0 to [-1,1] (gaussian_diffusion.py:348-352) */
#define B200MDM_FLAG_PHILOX_NOISE 4  /* loops only: eps comes from the engine's counter-based stream (b200mdm_set_noise_stream)
                                        instead of a caller-provided tape -- replaces th.randn_like, gaussian_diffusion.py:525 */

#define B200MDM_TARGET_NONE 0
#define B200MDM_TARGET_SINGLE 1 /* EmbedTargetLocSingle (model/mdm.py:399-419) */
#define B200MDM_TARGET_MULTI 2  /* EmbedTargetLocMulti  (model/mdm.py:449-480) */
#define B200MDM_TARGET_SPLIT 3  /* EmbedTargetLocSplit  (model/mdm.py:422-447) */

#define B200MDM_SCHED_STRIDE 8 /* floats per schedule row, see b200mdm_set_schedule */

typedef struct b200mdm_engine b200mdm_engine;

/* Mirrors the keyword arguments utils/model_util.py:24-71 (get_model_args) passes to MDM.__init__
 * (model/mdm.py:12-135) that matter to the forward pass. */
typedef struct b200mdm_config {
  int32_t arch;              /* B200MDM_ARCH_*            (args.arch) */
  int32_t latent_dim;        /* 512                       (args.latent_dim) */
  int32_t ff_size;           /* 1024                      (hard-wired model_util.py:63) */
  int32_t num_layers;        /* 8                         (args.layers) */
  int32_t num_heads;         /* 4                         (hard-wired model_util.py:63) */
  int32_t njoints;           /* 263 humanml / 25 a2m */
  int32_t nfeats;            /* 1 humanml / 6 a2m */
  int32_t cond_mode;         /* B200MDM_COND_*            (utils/parser_util.py:269-276) */
  int32_t cond_dim;          /* 512 CLIP / 768 DistilBERT (model/mdm.py:121) */
  int32_t num_actions;       /* rows of embed_action.action_embedding */
  int32_t mask_frames;       /* args.mask_frames (model/mdm.py:241-247) */
  int32_t pos_embed_max_len; /* args.pos_embed_max_len: rows of the positional table */
  int32_t temb_rows;         /* model timesteps to pre-embed (>= original_num_steps of the diffusion) */
  int32_t context_len;       /* trans_dec (DiP) prefix completion: args.context_len frames precede x (model/mdm.py:58-61) */
  /* target-location conditioning (args.multi_target_cond, model/mdm.py:64-73): B200MDM_TARGET_*; 0 = the model has no
   * embed_target_cond.  n_goal_rows = len(all_goal_joint_names) + 2 ('traj', 'heading'; 8 for humanml), and
   * target_enc_layers = args.target_enc_layers (single / split encoders; the multi encoder has a fixed depth). */
  int32_t target_encoder;
  int32_t n_goal_rows;
  int32_t target_enc_layers;
  int32_t reserved[3];
} b200mdm_config;

const char* b200mdm_last_error(void);
int b200mdm_version(void);

/* MDM.__init__ (model/mdm.py:12-135): allocates the weight store for `cfg` on the current CUDA device. */
int b200mdm_create(const b200mdm_config* cfg, b200mdm_engine** out);
int b200mdm_destroy(b200mdm_engine* e);

/* load_model_wo_clip / load_state_dict(strict=False) (utils/model_util.py:8-15): one call per state_dict entry,
 * `name` is the reference key (SURVEY.md A.4), data fp32, host or device memory.  The target encoder's keys are the
 * reference's embed_target_cond.* names, except that the multi encoder's per-joint MLPs are addressed by row index:
 * embed_target_cond.target_loc_emb.<row>.{0,2}.{weight,bias} (row = position in all_goal_joint_names + ['traj',
 * 'heading']; the reference keys them by joint name).  "sequence_pos_encoder.pe"
 * ([max_len, d]; the buffer the reference recomputes in PositionalEncoding.__init__, model/mdm.py:301-308) is
 * accepted here as well.  Unknown names -> B200MDM_EINVAL (the reference asserts no unexpected keys). */
int b200mdm_load_weight(b200mdm_engine* e, const char* name, const float* data, const int64_t* shape, int32_t ndim);

/* Repack for the tensor cores (fp16 K-major copies, hi/lo split of the in/out projections), precompute the
 * timestep-embedding MLP (TimestepEmbedder.forward, model/mdm.py:329-330) for every model timestep and the normalised
 * row weights of the multi target encoder (WeightedSum, utils/misc.py:12).
 * Fails with B200MDM_ESTATE listing the first missing tensor. */
int b200mdm_finalize_weights(b200mdm_engine* e, void* stream);

/* SpacedDiffusion / GaussianDiffusion tables (diffusion/respace.py:74-88, gaussian_diffusion.py:166-205) after the
 * fp64->fp32 cast of _extract_into_tensor (gaussian_diffusion.py:1612).  rows_host: n_steps rows of
 *   [0] posterior_mean_coef1  [1] posterior_mean_coef2  [2] (t!=0) * exp(0.5*posterior_log_variance_clipped)
 *   [3] sqrt_recip_alphas_cumprod  [4] sqrt_recipm1_alphas_cumprod  [5] sqrt(alphas_cumprod_prev)
 *   [6] sqrt(1 - alphas_cumprod_prev - sigma_ddim^2)  [7] (t!=0) * sigma_ddim(eta)
 * timestep_map_host: _WrappedModel's map (respace.py:125-127), n_steps int32.  Synchronous copy. */
int b200mdm_set_schedule(b200mdm_engine* e, int32_t n_steps, const float* rows_host, const int32_t* timestep_map_host);

/* Canonicalises model_kwargs['y'] (data_loaders/tensors.py:22-64 + callers) once per loop and (re)builds the
 * workspace for (batch, nframes):
 *   cond_embed_dev : y['text_embed'][0]  [batch, cond_dim] fp32 device, or NULL (cond_mode none / action)
 *   lengths_host   : y['lengths'] int64 [batch] or NULL => no key mask (also ignored unless cfg.mask_frames)
 *   scale_dev      : y['scale'] fp32 [batch] device => ClassifierFreeSampleModel semantics (cond/uncond pair
 *                    packed into one batch of 2*batch, utils/sampler_util.py:27-34); NULL => single forward
 *   force_uncond   : y.get('uncond', False) for the single-forward case (model/mdm.py:208)
 *   action_host    : y['action'][:,0] int64 [batch] or NULL
 * The text projection embed_text(mask_cond(.)) (model/mdm.py:218) is evaluated here, once. */
int b200mdm_set_cond(b200mdm_engine* e, int32_t batch, int32_t nframes, const float* cond_embed_dev,
                     const int64_t* lengths_host, const float* scale_dev, int32_t force_uncond,
                     const int64_t* action_host, void* stream);

/* trans_dec (DiP, model/mdm.py:203-206,255-270): conditioning for arch = B200MDM_ARCH_TRANS_DEC.
 *   enc_text_dev   : y['text_embed'][0], BERT token features [n_tokens, batch, cond_dim] fp32 device (reference layout)
 *   text_mask_host : y['text_embed'][1], uint8 [batch, n_tokens], 1 = padding (memory_key_padding_mask)
 *   nframes        : frames of x (pred_len); the sequence is context_len + nframes tokens, no conditioning token
 * lengths / scale / force_uncond as in b200mdm_set_cond.  Must be followed by b200mdm_set_prefix when context_len > 0. */
int b200mdm_set_cond_dec(b200mdm_engine* e, int32_t batch, int32_t nframes, const float* enc_text_dev,
                         const uint8_t* text_mask_host, int32_t n_tokens, const int64_t* lengths_host,
                         const float* scale_dev, int32_t force_uncond, void* stream);
/* Target-location conditioning (model/mdm.py:197-199): embed_target_cond(y['target_cond'], y['target_joint_names'],
 * y['is_heading']) for an engine created with target_encoder != 0.  The embedding does not depend on the timestep, so it is
 * computed here, once per loop, into an engine-owned buffer, and the NEXT b200mdm_set_cond / b200mdm_set_cond_dec adds it
 * to every conditioning row it builds (trans_enc: the conditioning token; DiP: every row of the cross-attention memory),
 * in both halves of a CFG pair and after the text masking of `uncond` (the reference adds it to time_emb, which both
 * halves share).  The step graph and its launches are unchanged.
 *   target_cond_dev : y['target_cond'] fp32 [batch, n_goal_rows, 3] device; NULL clears the target (no 'target_cond' key,
 *                     or y['target_uncond']: mask_cond zeros the embedding), giving exactly the computation without targets
 *   valid_host      : uint8 [batch, n_goal_rows], 1 where the row's name is in target_joint_names[b] (row
 *                     n_goal_rows - 1, 'heading', when is_heading[b])
 * The target is consumed by the next set_cond*, which fails with B200MDM_EINVAL if its batch differs from `batch`. */
int b200mdm_set_target(b200mdm_engine* e, int32_t batch, const float* target_cond_dev, const uint8_t* valid_host, void* stream);
/* y['prefix'] [batch, njoints, nfeats, context_len] fp32 device: the frames x is a continuation of. */
int b200mdm_set_prefix(b200mdm_engine* e, const float* prefix_dev, void* stream);

/* y['inpainting_mask'] (bool as uint8) / y['inpainted_motion'] [B,J,F,T] device pointers
 * (gaussian_diffusion.py:300-304); NULL, NULL clears. */
int b200mdm_set_inpaint(b200mdm_engine* e, const uint8_t* mask_dev, const float* motion_dev);

/* MDM.forward / ClassifierFreeSampleModel.forward (model/mdm.py:189-283, utils/sampler_util.py:27-34):
 * out = model(x, timesteps, y).  timesteps_host: int32 [batch] MODEL timesteps (already mapped). */
int b200mdm_denoise(b200mdm_engine* e, const float* x_dev, const int32_t* timesteps_host, float* out_dev, void* stream);

/* One p_sample / ddim_sample (gaussian_diffusion.py:489-541 / 729-779) at schedule index `index`:
 * x_out = step(x_t, eps).  pred_xstart_dev may be NULL.  x_out_dev may alias x_t_dev. */
int b200mdm_sample_step(b200mdm_engine* e, int32_t mode, int32_t index, const float* x_t_dev, const float* noise_dev,
                        int32_t flags, float* x_out_dev, float* pred_xstart_dev, void* stream);

/* p_sample_loop / ddim_sample_loop (gaussian_diffusion.py:591-727 / 876-990) without returning to the host:
 * steps index = n_steps-1-skip_timesteps ... 0 are enqueued (one CUDA graph of a single step, replayed, when
 * use_graph != 0; the graph runs on an engine-owned stream ordered against `stream` with events).
 * x_T_dev: the initial sample (after any q_sample of init_image), not modified; x_0_dev: result (may alias x_T_dev).
 * noise_tape_dev: eps for the k-th executed step at noise_tape_dev + k*noise_step_stride elements.
 * flags: B200MDM_FLAG_*.  The tape must stay alive until the work enqueued here has completed. */
int b200mdm_sample_loop(b200mdm_engine* e, int32_t mode, int32_t skip_timesteps, const float* x_T_dev, float* x_0_dev,
                        const float* noise_tape_dev, int64_t noise_step_stride, int32_t flags, int32_t use_graph,
                        void* stream);

/* The same loop body for a sub-range of the schedule: indices first_index, first_index-1, ... (n_run of them).  This is
 * what lets the host draw the reference's per-step th.randn_like (gaussian_diffusion.py:525) in bounded chunks instead
 * of materialising an O(n_steps) tape.  x_in_dev NULL: continue from the state the previous call left in the engine;
 * x_out_dev NULL: leave the result there.  noise_tape_dev: eps of the k-th step OF THIS CALL at + k*noise_step_stride
 * (ignored with B200MDM_FLAG_PHILOX_NOISE). */
int b200mdm_sample_loop_range(b200mdm_engine* e, int32_t mode, int32_t first_index, int32_t n_run, const float* x_in_dev,
                              float* x_out_dev, const float* noise_tape_dev, int64_t noise_step_stride, int32_t flags,
                              int32_t use_graph, void* stream);

/* The engine's own noise stream (no reference counterpart: the reference draws from torch's global generator).
 * Philox4x32-10 keyed by `seed`, counter = (element/4, schedule index of the consuming step, global sample index);
 * Box-Muller on the 4 output words (exact recipe: csrc/kernels.cuh, restated in oracle/philox_oracle.py).  A sample's
 * noise depends only on (seed, its global index, step, element): sharding the batch over GPUs, or drawing the steps in
 * chunks, cannot change it.  sample_index_base = global index of this engine's sample 0. */
int b200mdm_set_noise_stream(b200mdm_engine* e, uint64_t seed, int64_t sample_index_base);
/* out[b, :] = that stream for step_id (x_T uses step_id = -1), b = 0..batch-1, n_per_sample fp32 each. */
int b200mdm_philox_normal(float* out_dev, int32_t batch, int64_t n_per_sample, uint64_t seed, int64_t sample_index_base,
                          int32_t step_id, void* stream);

/* q_sample (gaussian_diffusion.py:226-244) at schedule index `index`: out = sqrt_ac*x_start + sqrt_1mac*noise;
 * x_start_dev NULL => zeros (gaussian_diffusion.py:693-694).  sqrt_ac / sqrt_1mac are the fp32 table values. */
int b200mdm_q_sample(b200mdm_engine* e, float sqrt_ac, float sqrt_1mac, const float* x_start_dev,
                     const float* noise_dev, float* out_dev, int64_t n, void* stream);

/* Kernels launched by this engine since creation / since the last reset (bench.py's gpu_launches). */
int64_t b200mdm_launch_count(b200mdm_engine* e, int32_t reset);

/* ---- post-loop step (SURVEY.md 8f rank 2): sample/generate.py:161-166 for data_rep 'hml_vec' -- inv_transform
 * (data * std + mean, data_loaders/humanml/data/dataset.py:309-310) + recover_from_ric (data_loaders/humanml/scripts/
 * motion_process.py:366-385,437-452) in one kernel, any input / output layout through element strides:
 *   data element (b, feature f, frame t)       at data_dev[b*stride_b + f*stride_f + t*stride_t]
 *   out  element (b, frame t, joint j, axis c) at out_dev[b*ostride_b + t*ostride_t + (3j + c)*ostride_c]
 * mean_dev / std_dev: fp32 [features] or both NULL (input already de-normalised).  njoints 22 (263 features) / 21 (251). */
int b200mdm_recover_from_ric(const float* data_dev, int64_t stride_b, int64_t stride_f, int64_t stride_t,
                             const float* mean_dev, const float* std_dev, float* out_dev, int64_t ostride_b,
                             int64_t ostride_t, int64_t ostride_c, int32_t batch, int32_t nframes, int32_t njoints,
                             void* stream);

/* ---- kernel-level entry points (used by tests/ to check each kernel against a torch fp32 restatement) ---- */
/* out16[M,N] = fp16(act(A16[M,K] @ W16[N,K]^T + bias)); act: 0 none, 1 exact GELU.  K % 8 == 0, N % 8 == 0,
 * block_n: 512 = CTA-pair kernel (256 x 256 tiles, operands streamed), 513 = CTA-pair kernel with its half of a W tile
 * resident in shared memory (K <= 512 and N <= 256 x the number of clusters, B200MDM_ENOTIMPL otherwise; the kernel the
 * step dispatches for the FFN up-projection), 128 = single-CTA kernel (the mainloop the embedding / output projections use). */
int b200mdm_test_gemm_f16(const void* a16_dev, const void* w16_dev, const float* bias_dev, void* out16_dev, int32_t M,
                          int32_t N, int32_t K, int32_t act, int32_t block_n, void* stream);
/* out16[n*S, d] = softmax(q k^T / sqrt(128) + mask) v per (sample, head); qkv16 [n*S, 3d]; kvlen int32 [n] device.
 * impl must be 0 (tcgen05 kernel, S <= 256). */
int b200mdm_test_attention(const void* qkv16_dev, void* out16_dev, const int32_t* kvlen_dev, int32_t n_samples,
                           int32_t S, int32_t d, int32_t impl, void* stream);
/* Cross-attention core of the trans_dec (DiP) layers, nn.MultiheadAttention(query = sequence, key = value = text memory)
 * between its in- and out-projections (model/mdm.py:219-224 via nn.TransformerDecoderLayer): d = 512, 4 heads.
 * q16 fp16 [n*S, 512]; kv16 fp16 rows (sample, token) of pitch ld_kv >= 1024 holding k | v; mask uint8 [n, n_tokens]
 * (1 = padding token); out16 fp16 [n*S, 1024]: columns [0, 512) are written.  n_tokens <= 64. */
int b200mdm_test_cross_attention(const void* q16_dev, const void* kv16_dev, const unsigned char* mask_dev, void* out16_dev,
                                 int32_t n_samples, int32_t S, int32_t n_tokens, int32_t ld_kv, void* stream);
/* The fused QKV-projection + attention kernel of the encoder layers (nn.MultiheadAttention up to its output projection,
 * model/mdm.py:77-84): out16[n*S, 512] = concat_h softmax((h Wq_h^T + bq)(h Wk_h^T + bk)^T / sqrt(128) + mask)(h Wv_h^T + bv).
 * h16: fp16 [n*S, ld] (first 512 columns used), wqkv16: in_proj_weight fp16 [1536, 512], bqkv fp32 [1536],
 * kvlen int32 [n] device (valid keys per sample), S <= 256. */
int b200mdm_test_qkv_attention(const void* h16_dev, int32_t ld, const void* wqkv16_dev, const float* bqkv_dev,
                               void* out16_dev, const int32_t* kvlen_dev, int32_t n_samples, int32_t S, void* stream);
/* h[M,512] <- LayerNorm(h + A16[M,K] @ W16[512,K]^T + bias; gamma, beta, 1e-5) in place (the fused out-projection /
 * FFN-down kernel of the transformer layer).  h is the engine's residual-stream format: fp16 [M, 1024] = [hi | lo],
 * value = hi + lo.  K % 8 == 0. */
int b200mdm_test_gemm_resid_ln(const void* a16_dev, const void* w16_dev, const float* bias_dev, const float* gamma_dev,
                               const float* beta_dev, void* hres16_dev, int32_t M, int32_t K, void* stream);

/* Host-only (no CUDA call): which CTA-pair GEMM the step would dispatch for out16[M,N] = act(A[M,K] W[N,K]^T + bias) on a
 * device with num_sms SMs, and the tile order it implies.  plan_out[0] = 1 if the W-resident kernel is chosen (0: streaming),
 * plan_out[1] = clusters launched, plan_out[2] = rounds of tiles on the busiest cluster with the strided order of the
 * streaming kernel, plan_out[3] = the same with the W-resident order (-1 if that kernel cannot run the shape).  If
 * tile_owner is not NULL it receives, for the W-resident order, the cluster that owns tile (m_blk, n_blk) at
 * tile_owner[m_blk * tiles_n + n_blk] (tiles_m = ceil(M / 256), tiles_n = ceil(N / 256)), -1 for a tile nobody owns. */
int b200mdm_test_gemm2_plan(int32_t M, int32_t N, int32_t K, int32_t num_sms, int32_t* plan_out, int32_t* tile_owner);

#ifdef __cplusplus
}
#endif
#endif /* B200MDM_H_ */
