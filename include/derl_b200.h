/*
 * derl_b200 — C ABI of the B200 (sm_100a) PPO rollout-processing / update data path.
 *
 * The reference (mknbv/derl) is pure Python and has no FFI of its own; its boundary for
 * this path is three duck-typed Python protocols (SURVEY.md §8b).  This header is the
 * native boundary *underneath* those protocols: each entry point replaces the arithmetic
 * of one reference function and is what a binding in the reference's own tree would call
 * (ctypes stub in INTEGRATION.md).  Citations are relative to the reference root.
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; every `*_dev` pointer is DEVICE memory of the
 *     current CUDA device, every `*_host` pointer is HOST memory;
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream);
 *     device entry points only enqueue work, they never synchronise;
 *   - inputs are borrowed and never written; outputs must not alias inputs;
 *   - return value: 0 on success, a DERL_E_* code otherwise; `derl_b200_last_error()`
 *     then returns a thread-local human-readable message;
 *   - there is NO CPU fallback: without an sm_100 device every compute call fails with
 *     DERL_E_NO_DEVICE.
 */
#ifndef DERL_B200_H_
#define DERL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: derl_b200_stem_conv_relu / derl_b200_stem_backward gained `rows_dev` (fused minibatch gather).
 * 3: derl_b200_ppo_mlp_update (whole PPO update of the MuJoCo-shaped actor-critic in one launch),
 *    derl_b200_stem_conv_relu_mask / derl_b200_stem_backward_masked (tcgen05 stem pair).
 * 5: derl_b200_gather_frame_stacks (minibatch gather out of a frame-plane rollout).
 * 6: derl_b200_stem_backward (the stem backward from the float32 activation) removed:
 *    derl_b200_stem_backward_masked is the stem backward.
 * 7: derl_b200_pack_frame_stacks / derl_b200_pack_frame_stacks_workspace_bytes (frame-plane
 *    packing of one env step on the device). */
#define DERL_B200_ABI_VERSION 7

enum {
  DERL_OK = 0,
  DERL_E_INVALID = 1,   /* bad argument (null pointer, negative size, unsupported width) */
  DERL_E_NO_DEVICE = 2, /* no CUDA device, or device is not compute capability 10.x     */
  DERL_E_CUDA = 3,      /* a CUDA runtime call failed; message carries cudaGetErrorString */
  DERL_E_WORKSPACE = 4  /* caller-provided workspace too small                           */
};

/* GAE kernel variants (derl_b200_gae `variant`). AUTO picks TMA when shapes allow it. */
enum {
  DERL_GAE_AUTO = 0,
  DERL_GAE_DIRECT = 1, /* one lane per env, register-prefetched coalesced loads          */
  DERL_GAE_TMA = 2     /* one lane per env, [T_tile x 32 env] tiles staged through smem   */
                       /* by TMA (cp.async.bulk.tensor) with an mbarrier pipeline         */
};

/* ------------------------------------------------------------------ library / device */

int derl_b200_abi_version(void);
const char* derl_b200_last_error(void);
/* 0 when the current device is an sm_100 part this library has code for. */
int derl_b200_device_ok(void);
/* Number of kernels this library has launched in this process (bench.py `gpu_launches`). */
uint64_t derl_b200_launch_count(void);

/* ------------------------------------------------------------------ K1: GAE / returns
 * Replaces the arithmetic of GAE.__call__, derl/runners/trajectory_transforms.py:45-65
 * (reverse scan :56-62, two-step last row :46,:53, value_targets :63), bit-exactly:
 * float64 register arithmetic in NumPy's evaluation order, no FMA contraction, float32
 * stores.  Layout is time-major [T, N] (flat index t*N + n), N = number of envs.
 *
 *   rewards_dev     [T,N] float32 (rewards_f64 = 0) or float64 (rewards_f64 = 1)
 *   values_dev      [T,N] float32     (trailing size-1 axis already squeezed, :42-43)
 *   resets_dev      [T,N] uint8/bool  (nonzero = episode ended at this step)
 *   last_value_dev  [N]   float32     (policy.act(latest_observations)["values"], :47-52)
 *   advantages_dev  [T,N] float32 out (pre-normalisation GAE)
 *   value_targets_dev [T,N] float32 out (= advantages + values in float32, :63)
 *   stats_dev       NULL, or [DERL_GAE_STATS] float64 out: {sum(adv), sum(adv^2), count}
 *                   accumulated in float64, deterministic order (no float atomics);
 *                   feeds derl_b200_normalize for the `normalize` branch (:67-68)
 *   workspace_dev   NULL iff stats_dev is NULL; else >= derl_b200_gae_workspace_bytes(T,N)
 */
#define DERL_GAE_STATS 3
size_t derl_b200_gae_workspace_bytes(int64_t T, int64_t N);
int derl_b200_gae(const void* rewards_dev, int rewards_f64, const float* values_dev,
                  const uint8_t* resets_dev, const float* last_value_dev, int64_t T,
                  int64_t N, double gamma, double lambda, float* advantages_dev,
                  float* value_targets_dev, double* stats_dev, void* workspace_dev,
                  size_t workspace_bytes, int variant, void* stream);

/* Whole-array normalisation x <- (x - mean) / (std_pop + eps) in float32 from float64
 * {sum, sumsq, count} held in DEVICE memory (no host sync).  Replaces
 * trajectory_transforms.py:67-68 (whole rollout) and NormalizeAdvantages.__call__
 * :89-92 (per minibatch).  In-place allowed (out_dev == x_dev). */
int derl_b200_normalize(const float* x_dev, float* out_dev, int64_t count,
                        const double* stats_dev, double epsilon, void* stream);

/* {sum, sumsq, count} of a float32 vector, float64 accumulation, deterministic.
 * workspace_dev >= derl_b200_moments_workspace_bytes(count). */
size_t derl_b200_moments_workspace_bytes(int64_t count);
int derl_b200_moments(const float* x_dev, int64_t count, double* stats_dev,
                      void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ K2: minibatch gather
 * Replaces the two NumPy fancy-index copies of IterateWithMinibatches
 * (derl/runners/onpolicy.py:44-49 epoch shuffle, :57-62 minibatch slice) with ONE
 * permutation-indexed copy out of the resident, never-shuffled rollout:
 *     dst[j, :] = src[perm[start + j], :]      for j in [0, count)
 * `perm` is the epoch's composed permutation (int64, device).  Bit-exact by construction.
 *
 * derl_b200_gather_rows: one wide column (frame stacks: row_bytes = 84*84*4 = 28224).
 *   When row_bytes % 16 == 0 and src/dst are 16-byte aligned the rows move through shared
 *   memory with TMA bulk copies (cp.async.bulk, mbarrier-pipelined, persistent CTAs);
 *   otherwise a vectorised LDG/STG kernel is used.  Indices must lie in [0, n_src_rows): the
 *   kernels do not check (the Python binding can: DERL_B200_CHECK_INDICES=1).
 */
int derl_b200_gather_rows(const void* src_dev, int64_t n_src_rows, int64_t row_bytes,
                          const int64_t* perm_dev, int64_t start, int64_t count,
                          void* dst_dev, void* stream);

/* First-epoch upload: `src_host` is PINNED HOST memory (device-accessible under UVA, e.g.
 * cudaHostAlloc / torch pin_memory) holding the whole column; every gathered row is written
 * twice — to dst[j] (the minibatch) and to resident_dev[perm[start+j]] (the device copy of the
 * column, at its original position).  Because the minibatches of one epoch partition the
 * permutation, running this for every minibatch of the first epoch uploads the rollout exactly
 * once, overlapped with the update of the previous minibatch when issued on a side stream,
 * instead of a blocking 14.8 GB cudaMemcpy up front (reference: `torch.from_numpy(...).to(device)`
 * per minibatch, derl/models.py:79-88).  max_ctas > 0 limits the grid (the copy is PCIe-bound;
 * a few CTAs saturate it and leave the other SMs to the concurrent update).  Rows must be
 * 16-byte multiples of at least 2048 bytes. */
int derl_b200_gather_rows_upload(const void* src_host, int64_t n_src_rows, int64_t row_bytes,
                                 const int64_t* perm_dev, int64_t start, int64_t count,
                                 void* dst_dev, void* resident_dev, int max_ctas, void* stream);

/* derl_b200_gather_columns: up to DERL_MAX_COLUMNS narrow columns (actions, log_prob,
 * advantages, value_targets, values, rewards, resets ...) in one launch.  Column c has
 * row_bytes[c] bytes per sample.  If moments_col >= 0 that column must be float32 with
 * row_bytes 4 and its {sum, sumsq, count} over the gathered minibatch is written to
 * stats_dev (float64[3]) — the fused statistics pass of NormalizeAdvantages
 * (trajectory_transforms.py:89-92).  workspace_dev >= derl_b200_moments_workspace_bytes(count).
 */
#define DERL_MAX_COLUMNS 16
int derl_b200_gather_columns(int n_columns, const void* const* src_dev,
                             const int64_t* row_bytes, void* const* dst_dev,
                             const int64_t* perm_dev, int64_t start, int64_t count,
                             int moments_col, double* stats_dev, void* workspace_dev,
                             size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ K10: frame-stack gather
 * The minibatch gather of K2 for a rollout whose `observations` are stored as unique frame
 * planes (derl_b200/runners/frame_stacks.py): the same two NumPy fancy-index copies of
 * IterateWithMinibatches (derl/runners/onpolicy.py:44-49, :57-62), now rebuilding each
 * stacked row from the planes it shares with its neighbours:
 *     dst[j, y, x, c] = frames[index[perm[start + j] * k + c], y, x]      for j in [0, count)
 *   frames_dev  uint8 [n_frames, height, width]   unique planes
 *   index_dev   int32 [n_samples, k]              plane id of every channel of every sample
 *   dst_dev     uint8 [count, height, width, k]   bit-identical to derl_b200_gather_rows on the
 *                                                 stacked [n_samples, height, width, k] column
 * k == 4 with height*width % 16 == 0 and 16-byte aligned frames / index / dst takes the TMA path
 * (bulk plane copies into shared memory, PRMT interleave, one bulk row store); any other shape a
 * plain kernel.  Neither checks indices: perm entries must lie in [0, n_samples) and plane ids in
 * [0, n_frames) (the Python FrameStacks validates caller-supplied ids once, on the host). */
int derl_b200_gather_frame_stacks(const void* frames_dev, int64_t n_frames, int64_t height,
                                  int64_t width, const int32_t* index_dev, int64_t n_samples,
                                  int64_t k, const int64_t* perm_dev, int64_t start, int64_t count,
                                  void* dst_dev, void* stream);

/* ------------------------------------------------------------------ K11: frame-stack packing
 * Packs one env step of stacked observations into the frame-plane format K10 reads, on the
 * device: FrameStackPacker.pack (derl_b200/runners/frame_stacks.py) is the specification, and for
 * the same sequence of steps this entry point hands out the same plane ids and writes the same
 * plane bytes, bit for bit.  Channel k-1 of every stack is a new plane; for c = k-2 ... 0 channel
 * c of env n reuses the id of channel c+1 of the same stack if their bytes are equal, else the id
 * of channel c+1 of env n's previous step if those bytes are equal, else it is a new plane.  New
 * ids are handed out from the running count: channel k-1 of env 0..n-1, then the new planes of
 * channel k-2 in env order, and so on down to channel 0.
 *   stacks_dev      uint8 [n, height, width, k]   this step (NHWC stacks)
 *   prev_stacks_dev uint8 [n, height, width, k]   the previous step, or NULL on a rollout's first
 *   prev_ids_dev    int32 [n, k]                  the previous step's ids; NULL iff prev_stacks_dev is
 *   pool_dev        uint8 [capacity, height, width]  the planes; new ones are appended in place
 *   state_dev       int64 [2]                     {plane count, overflow flag}, read and updated in
 *                                                 place; zero both to start a rollout
 *   ids_dev         int32 [n, k] out              this step's plane ids (e.g. one index row)
 * Nothing is read back to the host and nothing synchronises.  A step whose planes would not fit
 * in `capacity` writes no plane at or beyond it and no ids: it sets the overflow flag, which is
 * sticky (every later step does nothing) and must be checked by the caller at the end.
 * k == 4 with height*width % 16 == 0 and 16-byte aligned stacks / prev_stacks / pool takes the
 * vectorised path; any 1 <= k <= 32 and any height x width the plain one.  capacity and n*k must
 * fit int32.  workspace_dev >= derl_b200_pack_frame_stacks_workspace_bytes(n, k) (scratch; contents
 * undefined before and after; 0 for a k outside 1..32). */
size_t derl_b200_pack_frame_stacks_workspace_bytes(int64_t n, int64_t k);
int derl_b200_pack_frame_stacks(const void* stacks_dev, const void* prev_stacks_dev,
                                const int32_t* prev_ids_dev, int64_t n, int64_t height,
                                int64_t width, int64_t k, void* pool_dev, int64_t capacity,
                                int64_t* state_dev, int32_t* ids_dev, void* workspace_dev,
                                size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ K3: fused PPO loss
 * Replaces PPOLoss.__call__ (derl/alg/ppo.py:100-108) = policy_loss (:31-64) +
 * value_loss_coef * value_loss (:73-98) together with the torch.distributions calls it
 * makes (Categorical / Independent(Normal) log_prob + entropy, derl/policies.py:42,64-66)
 * and with its autograd backward: one launch yields the scalar loss AND d loss/d inputs.
 *
 *   loss = mean_i max(-r_i*adv_i, -clamp(r_i, 1-clip, 1+clip)*adv_i) - ecoef * mean_i H_i
 *        + vcoef * mean_i max((v_i-vt_i)^2, (vold_i + clamp(v_i-vold_i, -clip, clip) - vt_i)^2)
 *   r_i = exp(logp_i(action_i) - old_logp_i);  has_clip = 0 drops both clipped branches
 *   (cliprange=None, ppo.py:47,83).  torch.max tie semantics (gradient split 1/2 : 1/2) kept.
 *
 * All vectors are float32 device arrays of length B unless noted; values/value_targets/
 * old_values may be the reference's [B,1] arrays (same memory).  Gradients already include
 * the 1/B of the means.  Reductions are float64, two-stage, deterministic.
 *
 *   stats_dev [DERL_LOSS_STATS] float32 out — the scalars the reference logs
 *   (ppo.py:57-59, 91-94, 106):
 *     [0] loss  [1] mean max(s1,s2) ("policy_loss")  [2] mean entropy  [3] value_loss
 *     [4] mean(advantages)  [5] mean(value_targets)  [6] mean(values)
 *     [7] r_squared = 1 - mean((v-vt)^2)/var_unbiased(v)   (derl/alg/common.py:9-12)
 *     [8] fraction of samples with ratio outside [1-clip, 1+clip]
 *     [9] mean(old_logp - logp)  (approximate KL)
 *   loss_dev [1] float32 out.   Either head may be skipped: pass logits_dev (or loc_dev) NULL
 *   for a value-only loss (PPOLoss.value_loss) or values_dev NULL for a policy-only loss
 *   (PPOLoss.policy_loss); the corresponding gradient pointers must then be NULL as well.
 *   workspace_dev >= derl_b200_ppo_loss_workspace_bytes(B).
 */
#define DERL_LOSS_STATS 16
size_t derl_b200_ppo_loss_workspace_bytes(int64_t B);

/* Categorical head: logits [B,A] float32 row-major, actions [B] int64, 1 <= A <= 1024. */
int derl_b200_ppo_loss_categorical(const float* logits_dev, int64_t B, int64_t A,
                                   const int64_t* actions_dev, const float* old_logp_dev,
                                   const float* advantages_dev, const float* values_dev,
                                   const float* value_targets_dev, const float* old_values_dev,
                                   int has_clip, double cliprange, double value_loss_coef,
                                   double entropy_coef, float* loss_dev, float* dlogits_dev,
                                   float* dvalues_dev, float* stats_dev, void* workspace_dev,
                                   size_t workspace_bytes, void* stream);

/* Diagonal-Gaussian head: loc, scale, actions [B,D] float32 row-major, 1 <= D <= 256. */
int derl_b200_ppo_loss_gaussian(const float* loc_dev, const float* scale_dev, int64_t B,
                                int64_t D, const float* actions_dev, const float* old_logp_dev,
                                const float* advantages_dev, const float* values_dev,
                                const float* value_targets_dev, const float* old_values_dev,
                                int has_clip, double cliprange, double value_loss_coef,
                                double entropy_coef, float* loss_dev, float* dloc_dev,
                                float* dscale_dev, float* dvalues_dev, float* stats_dev,
                                void* workspace_dev, size_t workspace_bytes, void* stream);

/* Advantage actor-critic loss on the same kernels (SURVEY.md §8f rank 4): replaces
 * A2CLoss.__call__ (derl/alg/a2c.py:19-79): policy term -mean(log_prob * adv) (:31), unclipped
 * value loss mean((v - vt)^2) (:56), entropy (:32); stats as for PPO except [7] =
 * r_squared(values, value_targets) with the reference's argument order (:62), [8] = [9] = 0. */
int derl_b200_a2c_loss_categorical(const float* logits_dev, int64_t B, int64_t A,
                                   const int64_t* actions_dev, const float* advantages_dev,
                                   const float* values_dev, const float* value_targets_dev,
                                   double value_loss_coef, double entropy_coef, float* loss_dev,
                                   float* dlogits_dev, float* dvalues_dev, float* stats_dev,
                                   void* workspace_dev, size_t workspace_bytes, void* stream);
int derl_b200_a2c_loss_gaussian(const float* loc_dev, const float* scale_dev, int64_t B,
                                int64_t D, const float* actions_dev, const float* advantages_dev,
                                const float* values_dev, const float* value_targets_dev,
                                double value_loss_coef, double entropy_coef, float* loss_dev,
                                float* dloc_dev, float* dscale_dev, float* dvalues_dev,
                                float* stats_dev, void* workspace_dev, size_t workspace_bytes,
                                void* stream);

/* ------------------------------------------------------------------ K4: frame preparation
 * Replaces the input pipeline of NatureCNNBase.forward (derl/models.py:117-123: NHWC->NCHW
 * permute, `.float() / 255`, `.contiguous()`) with one pass that also applies the
 * space-to-depth re-indexing under which the 8x8/stride-4 stem is a 2x2/stride-1 convolution:
 *     dst[b, Y, X, (i*block + j)*C + c] = dtype(float(src[b, block*Y + i, block*X + j, c]) / divisor)
 * src: uint8 [batch, height, width, channels] (NHWC), block*channels == 16, height and width
 * multiples of block; dst: [batch, height/block, width/block, block*block*channels] of
 * dst_dtype.  The division is IEEE float32 (bit-identical to `.float() / 255`); divisor 1 skips it.
 */
enum { DERL_DTYPE_F32 = 0, DERL_DTYPE_BF16 = 1, DERL_DTYPE_F16 = 2 };
int derl_b200_frames_to_s2d(const uint8_t* src_dev, int64_t batch, int64_t height,
                            int64_t width, int64_t channels, int64_t block, void* dst_dev,
                            int dst_dtype, double divisor, void* stream);

/* Space-to-depth (inverse != 0: depth-to-space) of a channels-last activation
 * [batch, height, width, C] with channel_bytes = C * sizeof(element), a multiple of 16:
 *     s2d[b, Y, X, (i*block + j)*C + c] = x[b, block*Y + i, block*X + j, c]
 * Lets a strided conv with kernel = 2 x stride (the reference's nn.Conv2d(32, 64, 4, 2),
 * derl/models.py:104) run as a 2x2 / stride-1 conv; the inverse is its backward. */
int derl_b200_space_to_depth(const void* src_dev, int64_t batch, int64_t height, int64_t width,
                             int64_t channel_bytes, int64_t block, int inverse, void* dst_dev,
                             void* stream);

/* ------------------------------------------------------------------ K6t: stem conv on uint8 frames
 * The reference's first layer (derl/models.py:102-103,117-123): permute, `.float()/255`,
 * nn.Conv2d(4, 32, 8, 4), nn.ReLU — evaluated straight from the uint8 frames on the INT8
 * tensor cores of sm_100a (tcgen05.mma with the accumulators in tensor memory: raw frame bytes x
 * two signed 8-bit digit planes of the weights, exact int32 accumulation, fp32 recombination),
 * without materialising a floating-point copy of the frames.  One kernel writes float32 or bf16;
 * the bf16 output is the float32 one rounded to nearest even.  Fixed to the Atari stem geometry:
 *   frames [batch, 84, 84, 4] uint8 NHWC; weight [32, 4, 8, 8] float32 (conv layout); bias [32];
 *   out_block 1: out [batch, 20, 20, 32] channels-last;
 *   out_block 2: out [batch, 10, 10, 128], the space-to-depth(2) arrangement of the same
 *                activation (what derl_b200_space_to_depth would produce from it);
 *   out_dtype DERL_DTYPE_F32 or DERL_DTYPE_BF16; frames and out 16-byte aligned;
 *   batch * 400 < 2^31;
 *   rows_dev  NULL, or `batch` int64 row indices into frames_dev: frame i of the batch is
 *             frames_dev[rows_dev[i]].  This fuses the minibatch gather of
 *             IterateWithMinibatches (derl/runners/onpolicy.py:44-49,57-62) into the layer
 *             (SURVEY §8f rank 2): the kernel pulls each 28 224-byte row straight out of the
 *             resident rollout and the minibatch's observations are never materialised.
 *             Indices are trusted (validate the permutation once, when it is uploaded).
 * Needs cuTensorMapEncodeTiled from the driver (DERL_E_INVALID without it).
 */
int derl_b200_stem_conv_relu(const uint8_t* frames_dev, const int64_t* rows_dev, int64_t batch,
                             const float* weight_dev, const float* bias_dev, void* out_dev,
                             int out_dtype, int out_block, void* stream);

/* ------------------------------------------------------------------ K5: ReLU backward + bias grad
 * One pass over a channels-last activation gradient [rows, channels] (rows = B*H*W):
 *     grad_pre = out > 0 ? grad_out : 0;   bias_grad[c] = sum over rows of grad_pre[:, c]
 * Replaces, per conv layer of the reference's NatureCNNBase (derl/models.py:102-109), ATen's
 * threshold_backward plus the extra read cuDNN's convolution_backward spends on the bias
 * gradient.  dtype as DERL_DTYPE_*; bias_grad is float32; channels % 4 == 0 and channels/4
 * must divide 256; deterministic.  workspace >= derl_b200_relu_bwd_bias_workspace_bytes(C).
 * unblock > 1: grad_out / out are the space-to-depth(unblock) arrangement
 * [B, blocked_height, blocked_width, unblock^2 * c] of an activation (rows = B * blocked_height
 * * blocked_width, channels = unblock^2 * c); grad_pre is then written in the PLAIN
 * [B, blocked_height*unblock, blocked_width*unblock, c] layout (depth-to-space folded into the
 * stores) and bias_grad still has `channels` entries ((i, j, c) order: fold over (i, j)). */
size_t derl_b200_relu_bwd_bias_workspace_bytes(int64_t channels);
int derl_b200_relu_bwd_bias(const void* grad_out_dev, const void* out_dev, void* grad_pre_dev,
                            float* bias_grad_dev, int64_t rows, int64_t channels, int dtype,
                            int unblock, int64_t blocked_height, int64_t blocked_width,
                            void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ K9: linear output heads
 * The heads of the actor-critic network, stacked into one weight [units, 512] (units = sum of
 * the output widths, <= 32; rows in head order), applied to the trunk's 512 features in one pass:
 *     out[r, u] = (hidden[r, :] + hidden_bias) . weight[u, :] + bias[u]
 * Replaces `outputs = [layer(base_outputs) for layer in self.output_layers]`
 * (derl/models.py:201-202: one nn.Linear(512, n) per output, derl/models.py:189-192) and, in
 * backward, their input-gradient GEMMs + add, weight-gradient GEMMs and bias reductions:
 *     grad_hidden[r, :] = sum_u grad_out[r, u] weight[u, :]
 *     grad_weight[u, :] = sum_r grad_out[r, u] (hidden[r, :] + hidden_bias)
 *     grad_bias[u]      = sum_r grad_out[r, u]
 *     grad_hidden_bias  = sum_u grad_bias[u] weight[u, :]
 * hidden_bias (nullable, [512]) is the bias of the trunk's last nn.Linear(3136, 512)
 * (derl/models.py:112-114) when the caller passes the bias-free product as `hidden`: its gradient
 * then costs 512 x units flops instead of a reduction over [batch, 512].  float32 FMA arithmetic,
 * deterministic (per-CTA partials summed in a fixed order).  features must be 512; all float
 * tensors dense row-major and 16-byte aligned.
 * workspace >= derl_b200_linear_heads_workspace_bytes(units). */
size_t derl_b200_linear_heads_workspace_bytes(int units);
int derl_b200_linear_heads_forward(const float* hidden_dev, const float* hidden_bias_dev,
                                   const float* weight_dev, const float* bias_dev, float* out_dev,
                                   int64_t batch, int features, int units, void* stream);
int derl_b200_linear_heads_backward(const float* hidden_dev, const float* hidden_bias_dev,
                                    const float* weight_dev, const float* grad_out_dev,
                                    float* grad_hidden_dev, float* grad_weight_dev,
                                    float* grad_bias_dev, float* grad_hidden_bias_dev,
                                    int64_t batch, int features, int units, void* workspace_dev,
                                    size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ host-buffer entry points
 * Same operations on HOST arrays (what a NumPy caller such as the reference's
 * TransformInteractions hook holds): the library allocates device scratch, copies in on
 * `stream`, runs the kernel, copies out and synchronises the stream before returning.
 * `normalize` != 0 additionally applies the whole-rollout normalisation (:67-68).
 */
int derl_b200_gae_host(const void* rewards_host, int rewards_f64, const float* values_host,
                       const uint8_t* resets_host, const float* last_value_host, int64_t T,
                       int64_t N, double gamma, double lambda, int normalize, double epsilon,
                       float* advantages_host, float* value_targets_host, void* stream);

/* ------------------------------------------------------------------ K6t / K7t: the stem pair of a training step
 * The entry points below are the pair a training step uses: the forward additionally emits the
 * ReLU mask as one bit per activation, and the backward consumes that mask instead of re-reading
 * the float32 activation (51 200 B per frame).
 *   relu_mask [batch, 14, 32] uint32: bit l of word (tile t, channel c) = (activation of channel c
 *     at padded pixel m = 32 t + l is > 0), m = 21 oy + ox (ox = 20 and m >= 420 are padding,
 *     bits 0), whatever out_block / blocked says.
 * Forward: out must be 128-byte aligned (TMA store); everything else as in
 *   derl_b200_stem_conv_relu (derl/models.py:102-103,117-123).
 * Backward of the same layer (ReLU mask, bias gradient and weight gradient of
 * nn.Conv2d(4, 32, 8, 4); its autograd backward) in one pass over the raw frames, the incoming
 * gradient and the mask, on the INT8 tensor cores: the gradient is quantised per (frame, channel)
 * into two signed 8-bit digit planes (block floating point, residual <= 1/508 of the channel's
 * largest element in that frame), frames are exact.
 *   frames [batch, 84, 84, 4] uint8; grad_out float32 [batch, 400, 32] tiles of the activation
 *   gradient, pixels in plain (oy*20 + ox) order (blocked = 0) or in the space-to-depth(2) order
 *   the forward emits with out_block = 2 (blocked = 1); frames, grad_out and relu_mask 16-byte
 *   aligned; grad_weight [32, 4, 8, 8] float32, grad_bias [32] float32 (overwritten);
 *   rows_dev as in derl_b200_stem_conv_relu (NULL, or the fused gather's row indices).
 *   workspace >= derl_b200_stem_backward_workspace_bytes().  Deterministic. */
int derl_b200_stem_conv_relu_mask(const uint8_t* frames_dev, const int64_t* rows_dev, int64_t batch,
                                  const float* weight_dev, const float* bias_dev, float* out_dev,
                                  uint32_t* relu_mask_dev, int out_block, void* stream);
size_t derl_b200_stem_backward_workspace_bytes(void);
int derl_b200_stem_backward_masked(const uint8_t* frames_dev, const int64_t* rows_dev,
                                   int64_t batch, const float* grad_out_dev,
                                   const uint32_t* relu_mask_dev, int blocked,
                                   float* grad_weight_dev, float* grad_bias_dev,
                                   void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ K8: whole PPO update, MLP actor-critic
 * One launch = every epoch and minibatch of one rollout's PPO update for the reference's
 * MuJoCo model (derl/models.py:224-271: two tanh MLPs obs -> 64 -> 64 -> {act_dim, 1} plus a
 * state-independent logstd): permutation gather (derl/runners/onpolicy.py:43-62), minibatch
 * advantage normalisation (trajectory_transforms.py:89-92), forward, PPOLoss with the diagonal
 * Gaussian head (derl/alg/ppo.py:24-108), backward, clip_grad_norm_ and the Adam step
 * (derl/alg/common.py:56-78; torch.optim.Adam single-tensor formulas, amsgrad / weight decay off).
 * A persistent single-CTA kernel with parameters and gradients in shared memory: at 64-row
 * minibatches the reference's 320 optimiser steps per update are launch-latency work.
 *
 *   params_dev / exp_avg_dev / exp_avg_sq_dev: 13 device pointers each, float32, dense, in the
 *     order  policy {W1 [64,obs], b1 [64], W2 [64,64], b2 [64], W3 [act,64], b3 [act]},
 *            value  {W1, b1, W2, b2, W3 [1,64], b3 [1]},  logstd [act];  updated IN PLACE
 *   observations [nsamples, obs_dim] float64 (obs_f64 = 1; cast to float32 like the reference's
 *     collocate_inputs, derl/models.py:83-87) or float32; actions [nsamples, act_dim] float32;
 *     old_logp, advantages (NOT yet normalised), value_targets, old_values [nsamples] float32
 *   perm_dev [nepochs * nsamples] int64: epoch e's minibatch j is rows
 *     perm[e * nsamples + j * minibatch ...] (a trailing short minibatch when nsamples is not a
 *     multiple, like range(0, S, mbsize) in onpolicy.py:56); indices are trusted
 *   max_grad_norm < 0: no clipping;  adam_step: optimiser steps already taken (state["step"])
 *   losses_dev [nsteps] float32, stats_dev [nsteps * DERL_LOSS_STATS] float32 out
 *     (nsteps = nepochs * ceil(nsamples / minibatch); stats as in K3, [10] = gradient norm
 *     before clipping).
 *   workspace_dev >= derl_b200_ppo_mlp_update_workspace_bytes(obs_dim, act_dim) (the Adam moments
 *     in the kernel's padded layout while it runs; contents undefined before and after).
 * derl_b200_ppo_mlp_update_smem_bytes: dynamic shared memory the shape needs, 0 = unsupported. */
size_t derl_b200_ppo_mlp_update_smem_bytes(int obs_dim, int act_dim);
size_t derl_b200_ppo_mlp_update_workspace_bytes(int obs_dim, int act_dim);
int derl_b200_ppo_mlp_update(
    float* const* params_dev, float* const* exp_avg_dev, float* const* exp_avg_sq_dev, int obs_dim,
    int act_dim, const void* observations_dev, int obs_f64, const float* actions_dev,
    const float* old_logp_dev, const float* advantages_dev, const float* value_targets_dev,
    const float* old_values_dev, int64_t nsamples, const int64_t* perm_dev, int64_t nepochs,
    int64_t minibatch, int normalize_advantages, double adv_epsilon, int has_clip, double cliprange,
    double value_loss_coef, double entropy_coef, double max_grad_norm, double lr, double beta1,
    double beta2, double adam_eps, int64_t adam_step, float* losses_dev, float* stats_dev,
    void* workspace_dev, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DERL_B200_H_ */
