// layers.cuh - internal launchers shared between layers.cu, kfac.cu, gemm.cu and learner.cu
#pragma once
#include "common.cuh"

namespace acx {

// device-resident schedule state: every kernel that needs the learning rate, the zero-debias factor or the
// RNG step reads it from here, so a captured CUDA graph of an update stays valid from step to step.
struct Sched {
  unsigned long long gs;    // global_step (kfac_utils.py:38-53 semantics: cold step and K-FAC apply both count)
  unsigned long long ncov;  // number of covariance (EMA) updates so far
  float lr;                 // linear_decay(gs at the start of the update)  nn.py:154-156
  float debias;             // 1 / (1 - decay^ncov)   (1 when ncov == 0)
};

// a real matrix held as n bf16 planes p[0] + p[1] + p[2] (hi, mid, lo), row-major with leading dimension ld
struct Planes {
  bf16* p[3] = {nullptr, nullptr, nullptr};
  int n = 0;
  int ld = 0;
};

int gemm_dispatch(const acx_gemm_t* g, int impl, cudaStream_t st);
extern int g_cta_cap;
void set_cta_cap(int cap);
int returns_launch(const float* rewards, const uint8_t* terminals, const float* values, const float* bootstrap, float gamma,
                   int num_envs, int num_steps, float* targets, float* adv, cudaStream_t st);

int im2col_conv1(const uint8_t* obs, bf16* out, int rows_total, cudaStream_t st);
int im2col_bf16(const Planes& in, const Planes& out, int rows_total, int hw_in, int c, int k, int s, int hw_out, cudaStream_t st);
int col2im_mask_split(const float* dp, const bf16* act_hi, const Planes& out, int n_begin, int n_total, int mask_n, int hw_in, int c,
                      int k, int s, int hw_out, cudaStream_t st);
// im2col of uint8 (obs_u8) or fp32 NHWC observations of any geometry -> bf16 patch planes [rows, out.ld] (see layers.cu)
int im2col_obs(const void* obs, int obs_u8, const Planes& out, long long rows, int hw_in, int c, int k, int s, int hw_out,
               cudaStream_t st);
int heads_fwd(const Planes& act4, const float* vpol, const float* vval, int rows, int num_actions, float* logits, float* values,
              cudaStream_t st);
int loss_grad(const float* logits, const float* values, const uint8_t* actions, const float* targets, const int32_t* fl,
              const float* fe, uint64_t seed, const Sched* sched, int n_rows, int num_actions, float beta, float vw, float* dheads,
              float* scalars, int want_fisher, cudaStream_t st, float pw = 1.0f);
int returns_loss_grad(const float* rewards, const uint8_t* terminals, const float* bootstrap, float gamma, int num_envs, int num_steps,
                      float* targets, float* adv, const float* logits, const float* values, const uint8_t* actions, const int32_t* fl,
                      const float* fe, uint64_t seed, const Sched* sched, int num_actions, float beta, float vw, float* dheads,
                      float* scalars, int want_fisher, cudaStream_t st, float pw = 1.0f);
int heads_bwd(const float* dheads, const float* vpol, const float* vval, const Planes& act4, int n_rows, int rows_bwd,
              int num_actions, const Planes& dpre4, float* gpol, float* gval, cudaStream_t st);
int heads_gfactor(const float* dheads_fisher, int n_rows, int num_actions, float* g_pol, float* g_val, cudaStream_t st);
int colsum(const Planes& x, int rows, int cols, float scale, float* partial, int max_chunks, float* out, int out_stride,
           cudaStream_t st, float* out2 = nullptr, int out2_stride = 0, float* corner = nullptr);
int conv_border(const uint8_t* obs_u8, const Planes* act, int n_rows, int hw_in, int c, int k, int s, int hw_out, float scale,
                float* partial, int max_chunks, float* sum_tmp, float* a, int d, cudaStream_t st);
int transpose_split(const float* in, int k_rows, int c_cols, bf16* p0, bf16* p1, bf16* p2, int num_planes, int ld_out,
                    cudaStream_t st);
int weight_planes(const float* const* w, const int* k_rows, const int* c_cols, bf16* const (*t)[3], const int* ld_t,
                  bf16* const (*n)[3], const int* ld_n, int num_layers, cudaStream_t st, int perm_first = 0);
int obs_pairs_bf16(const uint8_t* obs, bf16* out, int samples, cudaStream_t st);
int conv1_pairs_forward(const bf16* obs_pairs, const Planes& wT_perm, int samples, const float* bias, float alpha, const Planes& y,
                        int num_pairs, const int* pair_a, const int* pair_b, cudaStream_t st);
int sample_actions(const float* logits, const float* uniform, uint64_t seed, uint64_t step, int rows, int num_actions, int greedy,
                   int32_t* actions, cudaStream_t st, unsigned long long* step_counter = nullptr);
int split_planes(const float* in, int ld_in, int rows, int cols, float scale, bf16* p0, bf16* p1, bf16* p2, int num_planes,
                 int ld_out, cudaStream_t st);

// conv.cu: implicit-GEMM convolution (forward) and gather-form input gradient on the tensor cores; NHWC, VALID
struct ConvGeom {
  int hw_in, c_in, k, s, hw_out, c_out;
};
bool conv_tc_supported(const ConvGeom& g, int dgrad);
int conv_tc_forward(const Planes& x, const Planes& wT, const ConvGeom& g, int samples, const float* bias, int relu, const Planes& y,
                    int num_pairs, const int* pair_a, const int* pair_b, cudaStream_t st);
int conv_tc_dgrad(const Planes& gout, const Planes& wD, const ConvGeom& g, int samples, const bf16* mask_hi, int mask_samples,
                  const Planes& dx, int num_pairs, const int* pair_a, const int* pair_b, cudaStream_t st, int lo_from_sample = -1,
                  int num_pairs_lo = 0);
int conv_dgrad_weight_planes(const float* w, const ConvGeom& g, const Planes& out, cudaStream_t st);
int conv_error_flag();

// kfac.cu
struct InvJob {          // one SPD inverse: M = debias * S + damp * I  (fp64) -> inverse fp32 + 3 bf16 planes
  const float* s;        // [n, n] running covariance sum
  int n;
  int damp_index;        // index into the device damping array
  double* work_m;        // [n, n] fp64 scratch (inverted in place)
  double* work_x;        // R [32, n] | old column panel [n, 32] | new column panel [n, 32] | pivot-block inverse [32, 32]
  float* inv;            // [n, n] fp32 result
  bf16* planes[3];       // [n, ld_planes]
  int ld_planes;
};
struct PreconJob {       // one small block: U = A^-1 (V G^-1) * scale, all fp32, C <= 64
  const float* v;        // [d, c] gradient block (weight rows + bias row)
  const float* ginv;     // [c, c]
  const float* ainv;     // [d, d]
  float* w;              // [d, c] scratch
  float* u;              // [d, c] preconditioned block
  int d, c;
  float scale;           // 1 / T~_l
};
int precondition_small(const PreconJob* d_jobs, int num_jobs, int max_d, cudaStream_t st);
int homog_border(float* a, int d, const float* colsum_scaled, cudaStream_t st);
int ema_update(float* s, const float* c, size_t count, float decay, float scale_c, cudaStream_t st);
int compute_dampings(const float* const* d_a_ptrs, const float* const* d_g_ptrs, const int* d_a_dims, const int* d_g_dims,
                     const float* d_lambda, int num_layers, float* d_damp, cudaStream_t st);
int spd_inverse_batched(const InvJob* h_jobs, const InvJob* d_jobs, int num_jobs, const Sched* sched, const float* d_damp,
                        cudaStream_t st, cudaStream_t side = nullptr);
// kfac_inv.cu: fp32 refresh with the factor tiles resident in shared memory; -1 = does not fit (use the chain above)
int spd_inverse_resident(const InvJob* h_jobs, int num_jobs, const Sched* sched, float* d_damp, const float* const* d_a_ptrs,
                         const float* const* d_g_ptrs, const int* d_a_dims, const int* d_g_dims, const float* d_lambda,
                         int num_layers, unsigned int* d_bar, cudaStream_t st);
int inv_resident_error_flag();
int inv_resident_trace_read(long long* h_out, int count);
int sched_step(Sched* s, float lr_start, float lr_end, double decay_steps, float* out_lr, int gs_inc, int ncov_inc,
               float ema_decay, int zero_debias, cudaStream_t st);
int sched_begin(Sched* s, float lr_start, float lr_end, double decay_steps, float* out_lr, cudaStream_t st);
int sched_advance(Sched* s, int gs_inc, int ncov_inc, float ema_decay, int zero_debias, cudaStream_t st);
int dot_partial(const float* a, const float* b, size_t count, float* partial, int num_partials, cudaStream_t st);
int kfac_step(float* params, float* velocity, const float* precon, size_t count, const float* dot_partials, int num_partials,
              const Sched* sched, float momentum, float norm_constraint, float* out_scalars, cudaStream_t st);
int momentum_clip_step(float* params, float* accum, const float* grads, size_t count, const float* sq_partials, int num_partials,
                       float lr, float momentum, float clip_norm, float* out_scalars, cudaStream_t st);
int rmsprop_clip_step(float* params, float* ms, const float* grads, size_t count, const float* sq_partials, int num_partials,
                      const Sched* sched, float decay, float epsilon, float clip_norm, float* out_scalars, cudaStream_t st,
                      float lr_value = 0.0f);
int fill_f32(float* p, size_t count, float v, cudaStream_t st);
int scale_f32(float* p, size_t count, float v, cudaStream_t st);

}  // namespace acx
