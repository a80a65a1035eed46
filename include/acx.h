/* acx.h - C ABI of libacx.so, the B200 (sm_100a) implementation of the ACKTR learner hot path
 * of jrobine/actor-critic.
 *
 * The reference has no FFI layer: its boundary is the Python API (SURVEY 8(b)).  These entry points
 * are what a ctypes binding inside the reference's Python modules would call; each one cites the
 * reference code whose work it replaces.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer owned by the caller; h_* is a HOST pointer.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - no hidden device allocation, no host synchronisation unless the function says so.
 *   - return value: 0 on success, non-zero on error; acx_last_error() gives the message
 *     (thread-local).  Nothing here falls back to the CPU.
 *   - "planes": a real matrix held as 1..3 bf16 matrices hi, mid, lo with x ~= hi + mid + lo
 *     (bf16 split of fp32; 1 plane = bf16, 2 planes ~ 2^-17, 3 planes = fp32-exact).
 */
#ifndef ACX_H_
#define ACX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACX_MAX_PLANES 3

/* ---- library ------------------------------------------------------------------------------ */
const char* acx_last_error(void);
int acx_version(void);
/* number of kernels this library has launched in this process since load / last reset
 * (bench.py's "gpu_launches"). */
uint64_t acx_launch_count(void);
void acx_reset_launch_count(void);

/* ---- K-PRE: batched Atari preprocessing + frame stack (uint8, bit-exact) ------------------- */
/* Replaces, for E environments at once:
 *   AtariFrameskipWrapper.step max        wrappers.py:64-65
 *   AtariPreprocessFrameWrapper.observation wrappers.py:30-33  (cv2 RGB2GRAY + INTER_AREA 84x84)
 *   FrameStackWrapper.step / reset        wrappers.py:224-235
 *   _AutoResetWrapper.step ordering       multi_env.py:127-132
 * d_raw_a, d_raw_b : uint8 [E,210,160,3] the last two raw frames of the frameskip window
 *                    (pass the same pointer twice for a single-frame window, wrappers.py:66-67)
 * d_terminal       : uint8 [E] terminal flag of THIS step (may be NULL = all zero)
 * d_reset_mask     : uint8 [E] 1 if the previous step was terminal, i.e. the env is reset first
 *                    (may be NULL); d_reset_raw: uint8 [E,210,160,3] first frame after that reset
 * d_stack_in       : uint8 [E,84,84,4] previous stacks;  d_stack_out: uint8 [E, out_env_stride]
 *                    new stacks (out_env_stride in bytes, >= 28224; lets the caller write straight
 *                    into step t of a batch-major rollout buffer [E,T,84,84,4]).
 *                    d_stack_in == d_stack_out (in place) is allowed when out_env_stride == 28224. */
int acx_preprocess_stack_u8(const uint8_t* d_raw_a, const uint8_t* d_raw_b, const uint8_t* d_terminal,
                            const uint8_t* d_reset_mask, const uint8_t* d_reset_raw,
                            const uint8_t* d_stack_in, uint8_t* d_stack_out, size_t out_env_stride,
                            int num_envs, void* stream);
/* MultiEnv.reset (multi_env.py:49-57) + FrameStackWrapper.reset (wrappers.py:232-235):
 * stack = 4 copies of preprocess(raw). */
int acx_preprocess_reset_u8(const uint8_t* d_raw, uint8_t* d_stack_out, size_t out_env_stride,
                            int num_envs, void* stream);

/* The stages of K-PRE on their own, for the per-environment wrapper classes of the reference's API:
 * acx_frame_max_u8        byte-wise max of two frames of nbytes each (AtariFrameskipWrapper.step, wrappers.py:64-65);
 * acx_framestack_push_u8  FrameStackWrapper.step / reset on preprocessed frames (wrappers.py:224-235): d_frames uint8
 *                         [E,84,84], d_mode uint8 [E] (NULL = all 0): 0 push, 1 push after a terminal step (older frames
 *                         zeroed), 2 reset (4 copies); stacks uint8 [E,84,84,4], in place allowed. */
int acx_frame_max_u8(const uint8_t* d_a, const uint8_t* d_b, uint8_t* d_out, size_t nbytes, void* stream);
int acx_framestack_push_u8(const uint8_t* d_frames, const uint8_t* d_mode, const uint8_t* d_stack_in, uint8_t* d_stack_out,
                           int num_envs, void* stream);

/* K-PRE at any square output size and stack depth: the three calls above for stacks uint8 [E,size,size,num_frames]
 * (the num_frames frames of a pixel contiguous), size in [4, 128], num_frames in [1, 16]; anything else returns an
 * error.  The resize is cv2 INTER_AREA 210x160 -> size x size with OpenCV's tap tables (built once per size and
 * device; the first call for a size uploads them synchronously, so make it outside stream capture).
 * acx_preprocess_stack_sq_u8  as acx_preprocess_stack_u8; out_env_stride >= size*size*num_frames bytes, in place
 *                             allowed when it equals size*size*num_frames.
 * acx_preprocess_reset_sq_u8  stack = num_frames copies of preprocess(raw).
 * acx_framestack_push_sq_u8   as acx_framestack_push_u8 on frames uint8 [E,size,size]; mode 2 = num_frames copies. */
int acx_preprocess_stack_sq_u8(const uint8_t* d_raw_a, const uint8_t* d_raw_b, const uint8_t* d_terminal,
                               const uint8_t* d_reset_mask, const uint8_t* d_reset_raw,
                               const uint8_t* d_stack_in, uint8_t* d_stack_out, size_t out_env_stride,
                               int num_envs, int size, int num_frames, void* stream);
int acx_preprocess_reset_sq_u8(const uint8_t* d_raw, uint8_t* d_stack_out, size_t out_env_stride,
                               int num_envs, int size, int num_frames, void* stream);
int acx_framestack_push_sq_u8(const uint8_t* d_frames, const uint8_t* d_mode, const uint8_t* d_stack_in,
                              uint8_t* d_stack_out, int num_envs, int size, int num_frames, void* stream);

/* ---- K-RET: n-step returns and advantages --------------------------------------------------- */
/* Replaces objectives._discount/_discount_bootstrap + targets/advantage (objectives.py:123-130,
 * 178-214).  rewards f32 [E,T], terminals u8 [E,T], values f32 [E,T], bootstrap f32 [E]
 * -> targets f32 [E,T], advantages f32 [E,T] (either output may be NULL). */
int acx_returns_adv(const float* d_rewards, const uint8_t* d_terminals, const float* d_values,
                    const float* d_bootstrap_values, float gamma, int num_envs, int num_steps,
                    float* d_targets, float* d_advantages, void* stream);

/* ---- GEMM on bf16 planes (tcgen05 / TMEM / TMA) --------------------------------------------- */
typedef struct {
  const void* planes[ACX_MAX_PLANES]; /* bf16 matrices, row-major, same shape/ld */
  int num_planes;
  int rows, cols;                      /* as stored */
  int ld;                              /* elements; multiple of 8 */
} acx_planes_t;

/* A GEMM operand that is never materialised: the patch matrix of an NHWC tensor - what the im2col of nn.conv2d
 * (nn.py:88-110) or kfac's extract_image_patches (envs/atari/model.py:227-237) would build - read by TMA box loads straight
 * from the tensor.  The rows of the operand are the locations (sample, y, x) of a gx x gy output grid (any order: the
 * products that use it sum over rows); its columns come in chunks of 64 bf16 that are contiguous in memory.  `dim` /
 * `stride_bytes` describe a 5-D view of each plane (innermost first, dim[0] elements contiguous, strides multiples of
 * 16 bytes, overlapping allowed) in which chunk q of location (sample, y, x) starts at the coordinates
 * (c0[q], x + c1[q], c2[q], y + c3[q], sample).  Out-of-range coordinates read as zero. */
typedef struct {
  const void* planes[ACX_MAX_PLANES]; int num_planes;
  long long dim[5]; long long stride_bytes[4];
  int gx, gy, samples;                 /* operand rows = samples * gy * gx */
  int num_chunks;                      /* operand columns = 64 * num_chunks (<= 16 chunks) */
  signed char c0[16], c1[16], c2[16], c3[16];
} acx_gather_t;

typedef struct {
  /* C[M,N] = alpha * sum_{(i,j) in pairs} opA(A_i) * opB(B_j)  (+ bias[n]) ; fp32 accumulate.
   * trans_a == 0: A stored [M,K] (K-major);  trans_a == 1: A stored [K,M] (MN-major).
   * trans_b == 0: B stored [N,K] (K-major);  trans_b == 1: B stored [K,N] (MN-major).
   * Only (0,0) and (1,1) are implemented on the tensor-core path. */
  acx_planes_t a, b;
  int trans_a, trans_b;
  int m, n, k;
  int num_pairs;                       /* 1..6 */
  int pair_a[6], pair_b[6];            /* plane indices */
  float alpha;
  const float* bias;                   /* [n] or NULL */
  int relu;                            /* max(0, .) after bias */
  int symmetric;                       /* C = C^T known (SYRK): only tiles with tile_n >= tile_m are
                                          computed; the reduction step mirrors them */
  /* outputs (any subset): */
  float* c; int ldc;                   /* fp32 */
  void* c_planes[ACX_MAX_PLANES]; int c_num_planes; int ldc_planes; /* bf16 split of the result */
  const void* mask_plane; int mask_ld; int mask_rows; /* optional: result *= (mask[m % mask_rows][n] > 0) (bf16) */
  /* split-K: splits > 1 (0 = automatic) writes partial sums [splits][m_pad][n_pad] fp32 to the workspace; the CTA that
   * completes a tile sums them in a fixed order inside the same kernel (deterministic, no finalize launch) and produces
   * the outputs above.  The first 16 KB of the workspace are arrival counters: they must be ZERO when a workspace is first
   * used and every call leaves them zero, so a workspace can be reused by consecutive calls without clearing; two GEMMs
   * that may run concurrently need separate workspaces. */
  int splits;
  float* workspace; size_t workspace_bytes;
  /* optional (MN-major products only, trans_a == trans_b == 1): A and / or B are patch matrices read in place from NHWC
   * tensors (see acx_gather_t; `a.planes` / `b.planes` are then ignored and k = samples * gy * gx).  Both operands must
   * enumerate the same locations: either both are gathered over the same grid, or the product is `symmetric` and B = A.
   * perm_m / perm_n != 0: row / column i of the result is stored at index (i & ~63) | perm(i & 63) with
   * perm(kw*8 + p*4 + c) = p*32 + kw*4 + c - the column order of conv1's patches when they are read from the row-pair
   * interleaved observation copy (acx_obs_pairs_bf16) back to the (kh, kw, c) order of the reference. */
  const acx_gather_t* a_gather; const acx_gather_t* b_gather;
  int perm_m, perm_n;
} acx_gemm_t;

/* Row-pair interleaved bf16 copy of uint8 observations [samples, 84, 84, 4] (envs/atari/model.py:92-93; raw byte values, exact):
 * out[n][p][x][q][c] = obs[n][2p + q][x][c], bf16 [samples, 42, 84, 2, 4].  The two kernel rows 2j, 2j + 1 of conv1's 8x8 / stride-4
 * patch at (oy, ox) are then 64 contiguous elements at pair-row 2 oy + j, pixel 4 ox, in the column order (kw, q, c): the patch
 * matrix the reference's conv1 and kfac's conv1 input factor are built on never has to be stored (acx_gather_t, perm_m / perm_n). */
int acx_obs_pairs_bf16(const uint8_t* d_obs, void* d_out, int samples, void* stream);
/* conv1 of the Nature-CNN (8x8 / stride 4, 32 filters, envs/atari/model.py:173-179) as an implicit GEMM on that copy:
 * out = relu(alpha * conv(obs, W) + bias) as bf16 planes [samples * 400, 32].  w_perm: W^T planes [32, 256] whose columns are in
 * the copy's order - column (kh / 2) * 64 + kw * 8 + (kh % 2) * 4 + c holds W[kh, kw, c, :]. */
int acx_conv1_pairs_forward(const void* d_obs_pairs, const acx_planes_t* w_perm, int samples, const float* d_bias, float alpha,
                            const acx_planes_t* out, int num_pairs, const int* pair_a, const int* pair_b, void* stream);
/* impl: 0 = tcgen05 tensor-core kernel (the product path), 1 = SIMT fp32 reference kernel on the
 * same planes (debug/validation only, never selected automatically). */
int acx_gemm(const acx_gemm_t* g, int impl, void* stream);
size_t acx_gemm_workspace_bytes(const acx_gemm_t* g);
/* fp32 [rows, cols] (ld_in) -> num_planes bf16 planes (ld_out multiple of 8); scale applied first. */
int acx_split_planes(const float* d_in, int ld_in, int rows, int cols, float scale,
                     void* const* d_planes, int num_planes, int ld_out, void* stream);
/* timing probe for bench.py's live roofline: when enabled, each tensor-core kernel launch (the kernel alone, without the
 * split-K finalize step) is bracketed by two library-owned CUDA events recorded on the launching stream;
 * acx_gemm_last_ms synchronises on them and returns the duration of the most recent launch. */
int acx_gemm_enable_timing(int enable);
int acx_gemm_last_ms(float* h_ms);
int acx_debug_tc_error(void);
/* triage: with ACX_GEMM_TRACE=1 in the environment, CTA 0 of the last acx_gemm launch records cycle counts of its MMA warp:
 * [0] total, [1] waiting for operands, [2] waiting for a drained accumulator, [3] k-blocks processed. */
int acx_debug_gemm_trace(long long* h_out4);
/* triage: with ACX_INV_TRACE=1 the resident inverse-refresh kernel records, per pivot step (8 slots each), clock64 stamps
 * of the last owner CTA ([0] step start [1] panels done [2] barrier passed [3] update done [4] barrier passed) and of
 * look-ahead CTA 0 ([5] step start [6] pivot inversion done [7] barrier passed); a refresh that falls back to the fp64
 * chain records nothing.  Copies `count` (<= 1024) values. */
int acx_debug_inv_trace(long long* h_out, int count);
/* test hook: one K-FAC inverse refresh, as the learners run it, on caller-given running sums.  Builds num_blocks K-FAC blocks
 * (input factor K[i] + 1, output factor C[i], T~ tnorm[i]; shared_heads != 0: the last two blocks read one input factor, as
 * the policy and value heads do; at most 5 input factors), lays out and zeroes their state in a device arena of its own,
 * copies the sums in, sets the zero-debias factor and runs
 *   path 0  the learners' refresh: the resident fp32 kernel, or the fp64 chain when its tiles do not fit;
 *   path 1  the resident kernel only; returns -1 (and writes nothing) when the tiles do not fit;
 *   path 2  the dampings and the fp64 chain only.
 * side_stream != 0: the chain inverts its pivot blocks on a second stream, as the Atari learner does.
 * h_sums: the input factors [d, d] in factor order, then the output factors [C, C] in block order, packed.  Outputs, packed
 * in job order (the input-factor inverse of each block, then the output-factor inverse of each block): h_inv fp32 [n, n];
 * h_planes the bf16 bits of the three operand planes of each inverse [3][n][ld], ld = n rounded up to 8; h_damp the
 * dampings [2 * num_blocks] (A, G per block); *h_path_ran 0 = resident kernel, 1 = fp64 chain.  Synchronous; frees
 * everything it allocated before it returns. */
int acx_debug_kfac_invert(int num_blocks, const int* h_k, const int* h_c, const int* h_tnorm, int shared_heads, float damping,
                          float debias, const float* h_sums, int path, int side_stream, float* h_inv, uint16_t* h_planes,
                          float* h_damp, int* h_path_ran);
/* debug hook: override the UMMA shared-memory descriptor strides (bytes) used for MN-major operands;
 * 0 restores the built-in values. */
void acx_debug_set_mn_desc(uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t kstep_bytes);
/* where the split-K partials are summed: 0 = a finalize launch (default), 1 = inside the GEMM kernel where one SM can sum a
 * tile's partials in a few microseconds, else a finalize launch, 2 = always inside the kernel (two levels beyond 8 splits).
 * Every mode is deterministic.  Also ACX_GEMM_FUSE_REDUCE. */
void acx_debug_set_fuse_reduce(int mode);

/* ---- implicit-GEMM convolution on bf16 planes (tcgen05 / TMEM / N-d TMA boxes) ---------------- */
/* nn.conv2d (nn.py:88-110: NHWC, VALID, HWIO weights) without a patch matrix, for kernels whose size is a multiple of the
 * stride (the 4x4/2 and 3x3/1 layers of envs/atari/model.py:180-199):
 *   dgrad == 0:  out[samples, hw_out, hw_out, c_out] = relu?(conv(x, W) + bias);
 *                x planes [samples, hw_in, hw_in, c_in] (stride * c_in == 64), w planes = W^T [c_out, k*k*c_in] (K-major)
 *   dgrad == 1:  out[samples, hw_in, hw_in, c_in] = (mask > 0) * conv_transpose(x, W)   (what tf.gradients computes for
 *                objectives.py:79); x planes = the output gradient [samples, hw_out, hw_out, c_out], w planes = the
 *                rearranged weights written by acx_conv_dgrad_weights, mask_plane = hi plane of the forward activation
 *                below ([mask_samples, hw_in, hw_in, c_in]; sample r uses r % mask_samples) or NULL.
 * The result is written as out.num_planes bf16 planes (ld = channels).  acx_conv_supported tells whether a geometry is
 * implemented; anything else must use the im2col + acx_gemm route. */
typedef struct {
  int dgrad;
  int samples;
  int hw_in, c_in, k, stride, hw_out, c_out;
  acx_planes_t x, w, out;
  const float* bias;                   /* [c_out] or NULL (forward only) */
  int relu;                            /* forward only */
  const void* mask_plane; int mask_samples;   /* dgrad only */
  int num_pairs; int pair_a[6], pair_b[6];    /* plane pairs (x plane, w plane) accumulated in fp32 */
} acx_conv_t;
int acx_conv_supported(const acx_conv_t* c);
int acx_conv(const acx_conv_t* c, void* stream);
/* fp32 HWIO weights [k*k*c_in, c_out] -> 3 bf16 planes [stride^2 * c_in, ld] (ld >= (k/stride)^2 * c_out, multiple of 8):
 * row (py, px, ci), column (i, j, co) holds W[stride*i + py, stride*j + px, ci, co]. */
int acx_conv_dgrad_weights(const float* d_w, int hw_in, int c_in, int k, int stride, int hw_out, int c_out,
                           void* const* d_planes, int ld, void* stream);

/* triage: with ACX_CONV_DEBUG bit 32 set, CTA 0 of the last acx_conv launch records cycle counts: [0] MMA warp total,
 * [1] waiting for operands, [2] waiting for a drained accumulator, [3] tiles, [5] epilogue warp waiting for an accumulator,
 * [7] epilogue warp first wait -> last wake. */
int acx_debug_conv_trace(long long* h_out8);

/* ---- learner (one process per GPU) ----------------------------------------------------------- */
typedef struct {
  int num_envs, num_steps, num_actions, conv3_filters;
  int acktr;                   /* 1 = K-FAC (ColdStartPeriodicInvUpdateKfacOpt), 0 = A2C RMSProp */
  float gamma, entropy_beta, value_loss_weight;
  /* schedule / optimiser (a2c_acktr.py:64-71,240-251) */
  float lr_start, lr_end; double lr_decay_steps;
  float cov_ema_decay, damping, momentum, norm_constraint;
  int invert_every, num_cold_updates;
  float cold_lr, cold_momentum, clip_norm;
  float rms_decay, rms_epsilon;
  int num_locations_mode;      /* 0 = true VALID output count, 1 = kfac-0.1 input//stride */
  int world_size;              /* data-parallel ranks (factor/gradient means are divided by it) */
  int gemm_impl;               /* 0 tensor core, 1 SIMT (debug) */
  int precision;               /* activations / gradients are held as bf16 planes (x = hi + mid + lo); a GEMM of level L
                                  accumulates the plane pairs (i,j) with i+j <= L (1 pair, 3 pairs ~2^-17, 6 pairs fp32 class):
                                  0 = parity grade: forward and backward on 3 planes / 6 pairs (fp32 class: ReLU masks hinge on the
                                      sign of cancelling sums), factor SYRKs 3 pairs, preconditioning 6
                                  4 = as 0 but gradients on 2 planes / 3 pairs (conv gradients ~6e-4 on iid-uniform inputs)
                                  1 = 2 planes, forward/backward/factors 3 pairs, preconditioning 6
                                  2 = as 1 with the factor SYRKs on the hi plane only (bf16 inputs)
                                  3 = single-plane bf16 everywhere (fastest; not parity grade) */
  int use_graphs;              /* 1 = capture each (phase, schedule variant) into a CUDA graph on its second use and replay
                                  it afterwards (needs a non-NULL stream); 0 = launch kernel by kernel */
  int conv_impl;               /* 0 = gather-form input gradient of conv2 / conv3 on the tensor cores (acx_conv, dgrad) when the
                                  geometry is supported (conv3_filters 32 or 64), 1 = GEMM to an fp32 patch-gradient matrix +
                                  col2im everywhere */
  int num_lanes;               /* concurrent lanes inside one update: 0 = default (3: forward/dgrad chain | input factors |
                                  wgrad + output factors, forked and joined with events on library-owned streams, so the
                                  caller still orders everything through `stream`); 1 = strictly serial on `stream` */
  uint64_t seed;               /* Philox seed for on-device Fisher sampling */
  /* SURVEY A.7-U3: initialisation conventions of kfac that the reference does not pin (all 0 = kfac 0.1.x as SURVEY A.5
   * records it: zero-initialised running covariances with zero-debias, zero-initialised inverses) */
  int cov_init_identity;       /* 1 = running covariance sums start as identity matrices (older tf.contrib.kfac); implies
                                  no zero-debias */
  int no_zero_debias;          /* 1 = the running sums are used as they are (no 1 / (1 - decay^n) factor) */
  int inv_init_identity;       /* 1 = stored inverses start as identity: the always-run K-FAC apply (kfac_utils.py:52-53)
                                  takes real steps U = V / T~ before the first refresh instead of being a no-op */
} acx_learner_config_t;

typedef struct acx_learner acx_learner_t;

size_t acx_learner_arena_bytes(const acx_learner_config_t* cfg);
/* d_arena: caller-allocated device memory of at least acx_learner_arena_bytes (256-byte aligned). */
acx_learner_t* acx_learner_create(const acx_learner_config_t* cfg, void* d_arena, size_t arena_bytes);
void acx_learner_destroy(acx_learner_t* l);

/* flat fp32 parameter vector, per layer [K_l+1, C_l] (weights rows in (kh,kw,cin) order = the
 * reference's HWIO variable flattened, nn.py:81-83 / 31-32; then the bias row), layers in the order
 * conv1, conv2, conv3, fc4, fc_policy, fc_baseline. */
size_t acx_learner_num_params(const acx_learner_t* l);
int acx_learner_set_params(acx_learner_t* l, const float* h_params, void* stream);
int acx_learner_get_params(acx_learner_t* l, float* h_params, void* stream);
/* call after writing the "params" / "inverses" buffers directly on the device (checkpoint restore):
 * re-derives the bf16 operand planes of the weights and of the stored inverses */
int acx_learner_refresh_weights(acx_learner_t* l, void* stream);
/* named device views into the arena (for torch views, the all-reduce and checkpoints); NULL + error if unknown.
 * inputs:  "observations" u8 [N+E,84,84,4] (train rows batch-major [E,T], then the E bootstrap rows),
 *          "actions" u8 [N], "rewards" f32 [N], "terminals" u8 [N]
 * state:   "params" "velocity" "accum" (cold momentum / RMSProp ms) "factor_sums" "inverses" "sched"
 * per update: "grads" "precon" "factor_stats" "reduce_bucket" (= factor_stats [A | G] | grads | 4 scalars)
 *          "logits" f32 [N+E,A] "values" f32 [N+E] "targets" "advantages" f32 [N] "dampings" f32 [12]
 *          "input_factor_stats" (the A prefix of "reduce_bucket")
 *          "scalars" f32 [16]: 0 policy_loss 1 baseline_loss 2 mean_entropy 3 loss 4 KL-clip coeff 5 <V,U>
 *                              6 gradient global norm (cold / A2C step) 7 learning rate used
 * per block views: "params/<layer>" "grads/<layer>" "precon/<layer>" "velocity/<layer>" "accum/<layer>" ([K+1, C]), "stats/A/<factor>"
 *          "sums/A/<factor>" (conv1 conv2 conv3 fc4 heads), "stats/G/<layer>" "sums/G/<layer>",
 *          "inv/A/<layer>" "inv/G/<layer>" */
void* acx_learner_buffer(acx_learner_t* l, const char* name, size_t* num_bytes);

/* One learner update = the reference's session.run(optimize_op, feed_dict) (a2c_acktr.py:117-126).
 * phase 1: forward (train + bootstrap rows), returns, loss, backward, Fisher backward, batch factor
 *          statistics -> everything that must be all-reduced lands in buffer "reduce_bucket".
 * phase 2: (after the caller's all-reduce, if world_size > 1) EMA, scheduled inverse refresh,
 *          precondition, KL clip, momentum, apply (or cold / RMSProp step); global_step advances.
 * Inputs are read from the arena's input buffers (obs buffer + "actions","rewards","terminals");
 * d_fisher_labels (int32 [N]) / d_fisher_eps (f32 [N]) inject the Fisher samples (NULL = Philox). */
int acx_learner_phase1(acx_learner_t* l, const int32_t* d_fisher_labels, const float* d_fisher_eps, void* stream);
int acx_learner_phase2(acx_learner_t* l, void* stream);
/* Data-parallel overlap: the reduce bucket is laid out [input factors A | output factors G | gradients | 4 scalars] and the
 * A prefix (buffer "input_factor_stats", ~3/4 of the bucket) is complete long before phase 1 ends.  After
 * acx_learner_phase1 has been called (i.e. enqueued) this makes `stream` wait for that prefix only, so the caller can
 * all-reduce it on `stream` while the backward pass still runs; returns -1 (and makes nobody wait) when the last phase 1
 * computed no factor statistics or ran serially - then the prefix is complete when phase 1 is. */
/* phase 1 + phase 2 back to back as ONE captured CUDA graph per schedule variant (one graph launch per update): for callers
 * that run nothing between the phases - a single GPU, or peers set with acx_learner_set_peers and no external EMA. */
int acx_learner_update(acx_learner_t* l, const int32_t* d_fisher_labels, const float* d_fisher_eps, void* stream);
int acx_learner_wait_input_factors(acx_learner_t* l, void* stream);
/* Split exchange for data-parallel learners.  Phase 2 reads only [grads | scalars] of the reduce bucket (and the stored
 * inverses); the factor statistics [A | G] are read by the EMA alone, whose result nothing needs before the next inverse
 * refresh.  A caller may therefore reduce the statistics on a second stream / communicator while phase 2 runs:
 *   acx_learner_update_plan        what the next phase 2 will do: has_factors (a covariance update: the statistics of this
 *                                  phase 1 are live), will_invert (it refreshes the inverses: the EMA must be complete first)
 *   acx_learner_set_external_ema   on: the next phase 2 calls scale only [grads | scalars] by 1 / world_size and skip the EMA
 *   acx_learner_ema                scales the statistics by 1 / world_size and applies the EMA on `stream` (the caller orders
 *                                  it after its all-reduce of the statistics and before the next phase 1 / a refreshing phase 2)
 * (actorcritic_b200.Engine.allreduce does this for NCCL groups; bit-identical to the single all-reduce.) */
int acx_learner_update_plan(const acx_learner_t* l, int* has_factors, int* will_invert);
int acx_learner_set_external_ema(acx_learner_t* l, int on);
/* The exchange over NVLink peer memory instead of a caller-side collective (csrc/peer.cu): every rank maps every other rank's
 * arena (acx_peer_export / acx_peer_import: CUDA IPC) and hands the mapped bases to acx_learner_set_peers (entry `rank` is ignored;
 * world <= 8, one node).  From then on phase 2 starts with ONE kernel that sums the ranks' buckets in rank order - two-shot
 * reduce-scatter + all-gather on peer pointers, flag barriers between equally numbered CTAs of the GPUs - fused with the
 * 1 / world_size scaling: the whole `reduce_bucket`, or, with acx_learner_set_external_ema, only [G | grads | scalars] (the caller
 * still sums the `input_factor_stats` prefix on its own stream, waits with acx_learner_wait_reduced for this update's kernel and
 * runs acx_learner_ema).  The kernel is part of phase 2's CUDA graph, so a data-parallel update is two graph launches with no
 * collective call in between.  Every rank must run the same sequence of updates.  acx_peer_error: non-zero after a barrier
 * timed out (~2 s). */
int acx_peer_export(const void* d_ptr, unsigned char* out_handle64, unsigned long long* out_offset);
void* acx_peer_import(const unsigned char* handle64, unsigned long long offset);
int acx_learner_set_peers(acx_learner_t* l, int rank, int world, void* const* peer_arena_bases);
int acx_learner_wait_reduced(acx_learner_t* l, void* stream);
/* the same kernel for the `input_factor_stats` prefix on the caller's side stream (its own flag channel; unscaled) */
int acx_learner_peer_reduce_prefix(acx_learner_t* l, void* stream);
int acx_peer_error(void);
int acx_learner_ema(acx_learner_t* l, void* stream);
/* optional stage timing with CUDA events on the launching stream (bench.py's live roofline numbers).
 * stages: 0 forward, 1 returns+loss+heads backward, 2 backward (dgrad+wgrad), 3 factor statistics,
 *         4 cold step / factor EMA, 5 inverse refresh, 6 preconditioning, 7 KL clip+momentum+apply+operand refresh.
 * acx_learner_stage_ms synchronises on the recorded events and writes ACX_NUM_STAGES floats (last update). */
#define ACX_NUM_STAGES 8
int acx_learner_set_profiling(acx_learner_t* l, int enable);
int acx_learner_stage_ms(acx_learner_t* l, float* h_ms);
int64_t acx_learner_global_step(const acx_learner_t* l);
/* schedule counters (checkpoint / resume): global_step, number of covariance updates, whether the stored
 * inverses have been computed at least once (kfac initialises them to zero). */
int acx_learner_set_state(acx_learner_t* l, int64_t global_step, int64_t num_cov_updates, int inverses_valid, void* stream);
int acx_learner_get_state(const acx_learner_t* l, int64_t* global_step, int64_t* num_cov_updates, int* inverses_valid);
/* objectives.py:31-54 `optimize_separate` (two optimizers, two backward passes): the next acx_learner_phase1 calls
 * differentiate  policy_weight * policy_loss + value_weight * baseline_loss  instead of the configured
 * policy_loss + value_loss_weight * baseline_loss  ((1, 0) = the policy loss on its own, (0, 1) = the baseline loss). */
int acx_learner_set_loss_weights(acx_learner_t* l, float policy_weight, float value_weight);
/* the optimizer steps of nn.py:185-189 on caller-owned device vectors (count floats each): the global-norm clip
 * g * clip / max(|g|, clip), then RMSProp (TF-1: ms <- decay ms + (1 - decay) g^2; theta -= lr g / sqrt(ms + eps), ms starts
 * at one) or momentum (acc <- momentum acc + g; theta -= lr acc).  d_scratch: 296 floats; d_out_norm (may be NULL)
 * receives |g|. */
int acx_clip_rmsprop_step(float* d_params, float* d_ms, const float* d_grads, size_t count, float lr, float decay,
                          float epsilon, float clip_norm, float* d_scratch, float* d_out_norm, void* stream);
int acx_clip_momentum_step(float* d_params, float* d_accum, const float* d_grads, size_t count, float lr, float momentum,
                           float clip_norm, float* d_scratch, float* d_out_norm, void* stream);
/* DistributionPolicy.sample / mode (policies.py:86-87) on device logits [rows, num_actions]: inverse-CDF categorical draw
 * from softmax(logits) with the given uniforms d_uniform [rows] (NULL = Philox(seed, step, row)), or argmax (greedy). */
int acx_sample_actions(const float* d_logits, const float* d_uniform, uint64_t seed, uint64_t step, int rows,
                       int num_actions, int greedy, int32_t* d_actions, void* stream);
/* forward only on `rows` observations already in d_obs (uint8 [rows,84,84,4]) -> logits [rows,A],
 * values [rows]; then categorical sample (u in [0,1) given, or Philox) / argmax.  Replaces
 * ActorCriticModel.sample_actions / select_max_actions (model.py:135-169). */
int acx_learner_act(acx_learner_t* l, const uint8_t* d_obs, int rows, const float* d_uniform,
                    int greedy, int32_t* d_actions, float* d_logits, float* d_values, void* stream);

/* ---- fully connected learner (one process per GPU) ------------------------------------------- */
/* The same ACKTR / A2C update as acx_learner_*, for a stack of fully connected ReLU layers on flat fp32 observations:
 * hidden layers fc1 .. fcL (x @ W + b, ReLU; nn.py:37-52) and the heads fc_policy [H_L, A], fc_baseline [H_L, 1] reading the
 * last hidden layer, with one K-FAC fully connected block per layer (register_fully_connected, model.py:107-119; the two heads
 * share one input factor as in envs/atari/model.py:243,246).  The hyper-parameter fields mean what they mean in
 * acx_learner_config_t; precision is that config's default preset. */
typedef struct {
  int num_envs, num_steps;
  int obs_dim;                 /* D: observation features (the Box flattened row-major), 1..2048 */
  int num_hidden;              /* L: 1..4 hidden layers */
  int hidden[4];               /* their widths, multiples of 8 in [8, 1024] */
  int num_actions;             /* 1..31 */
  int acktr;
  float gamma, entropy_beta, value_loss_weight;
  float lr_start, lr_end; double lr_decay_steps;
  float cov_ema_decay, damping, momentum, norm_constraint;
  int invert_every, num_cold_updates;
  float cold_lr, cold_momentum, clip_norm;
  float rms_decay, rms_epsilon;
  int use_graphs;
  uint64_t seed;
} acx_mlp_config_t;

typedef struct acx_mlp acx_mlp_t;

size_t acx_mlp_arena_bytes(const acx_mlp_config_t* cfg);
acx_mlp_t* acx_mlp_create(const acx_mlp_config_t* cfg, void* d_arena, size_t arena_bytes);
void acx_mlp_destroy(acx_mlp_t* l);
/* flat fp32 parameter vector, per layer [K_l+1, C_l] (the [in, out] weights of nn.fully_connected_params, nn.py:8-33, then
 * the bias row), layers in the order fc1 .. fcL, fc_policy, fc_baseline. */
size_t acx_mlp_num_params(const acx_mlp_t* l);
int acx_mlp_set_params(acx_mlp_t* l, const float* h_params, void* stream);
int acx_mlp_get_params(acx_mlp_t* l, float* h_params, void* stream);
int acx_mlp_refresh_weights(acx_mlp_t* l, void* stream);
/* named device views, as acx_learner_buffer: "observations" f32 [N+E, D] (train rows batch-major [E,T], then the E bootstrap
 * rows), "actions" "rewards" "terminals", "params" "velocity" "accum" "grads" "precon" "factor_stats" "factor_sums"
 * "inverses" "reduce_bucket" "scalars" "sched" "logits" "values" "targets" "advantages" "dheads", per block
 * "params/<layer>" "grads/<layer>" "precon/<layer>" "velocity/<layer>" "accum/<layer>", "stats/A/<factor>" "sums/A/<factor>"
 * (fc1 .. fcL, heads), "stats/G/<layer>" "sums/G/<layer>" "inv/A/<layer>" "inv/G/<layer>", and "act_hi/fc<i>": the hi plane
 * of each hidden activation, whose sign is the ReLU mask of the backward pass. */
void* acx_mlp_buffer(acx_mlp_t* l, const char* name, size_t* num_bytes);
/* One update = session.run(optimize_op, feed_dict) (a2c_acktr.py:117-126) for this model: forward, returns, A2C loss and
 * gradients, Fisher backward and factor statistics, then ColdStartPeriodicInvUpdateKfacOpt.apply_gradients (kfac_utils.py:38-53)
 * or ClipGlobalNorm(RMSProp) (a2c_acktr.py:250-251); one captured CUDA graph per schedule variant.  Fisher samples as in
 * acx_learner_phase1 (NULL = Philox). */
int acx_mlp_update(acx_mlp_t* l, const int32_t* d_fisher_labels, const float* d_fisher_eps, void* stream);
int acx_mlp_set_state(acx_mlp_t* l, int64_t global_step, int64_t num_cov_updates, int inverses_valid, void* stream);
int acx_mlp_get_state(const acx_mlp_t* l, int64_t* global_step, int64_t* num_cov_updates, int* inverses_valid);
int64_t acx_mlp_global_step(const acx_mlp_t* l);
/* ActorCriticModel.sample_actions / select_max_actions (model.py:135-169): forward on `rows` <= N+E observations
 * d_obs f32 [rows, D] -> logits, values; then the categorical draw / argmax of acx_sample_actions. */
int acx_mlp_act(acx_mlp_t* l, const float* d_obs, int rows, const float* d_uniform, int greedy, int32_t* d_actions,
                float* d_logits, float* d_values, void* stream);

/* ---- convolutional learner (one process per GPU) ---------------------------------------------- */
/* The fully connected learner above with a trunk of 1..3 conv layers in front of its fully connected layers, for square
 * NHWC image observations [H, H, C]: conv1 .. convK (VALID, stride s, ReLU; HWIO weights, nn.py:55-110), the (h, w, c) flatten
 * of nn.flatten, then fc(K+1) .. fc(K+L) and the heads as acx_mlp_*.  One K-FAC conv block per conv layer
 * (register_conv2d: factors over every output location, damping lambda / T and the preconditioned block / T with T = oh * ow
 * true locations, as the Atari learner).  uint8 observations are scaled by 1/255 (envs/atari/model.py:93), fp32 ones are used
 * as given.  The handle is an acx_mlp_t: every acx_mlp_* call other than acx_mlp_act accepts it; acting goes through
 * acx_cnn_act.  Its buffers are those of acx_mlp_buffer ("observations": uint8 or f32 [N+E, H, H, C]) and per conv layer
 * "act_hi/conv<i>" [(N+E) * oh * ow, filters] (the ReLU masks). */
typedef struct {
  acx_mlp_config_t mlp;        /* num_hidden / hidden[]: the fully connected layers after the trunk; obs_dim is derived */
  int obs_hw, obs_channels;    /* H in [4, 128], C in [1, 16] */
  int obs_u8;                  /* 1: uint8 observations, 0: fp32 */
  int num_conv;                /* 1..3, and num_conv + mlp.num_hidden <= 4 */
  int filters[3];              /* multiples of 8 in [8, 128] */
  int kernel[3];               /* in [1, 8]; kernel^2 * input channels + 1 <= 3137 */
  int stride[3];               /* in [1, min(kernel, 4)]; every output at least 1 x 1, flattened output + 1 <= 3137 */
} acx_cnn_config_t;

size_t acx_cnn_arena_bytes(const acx_cnn_config_t* cfg);
acx_mlp_t* acx_cnn_create(const acx_cnn_config_t* cfg, void* d_arena, size_t arena_bytes);
/* acx_mlp_act for this learner: d_obs uint8 or f32 (as configured) [rows, H, H, C] */
int acx_cnn_act(acx_mlp_t* l, const void* d_obs, int rows, const float* d_uniform, int greedy, int32_t* d_actions,
                float* d_logits, float* d_values, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ACX_H_ */
