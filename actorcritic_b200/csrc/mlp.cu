// mlp.cu - the ACKTR / A2C learner for fully connected actor-critic models (include/acx.h `acx_mlp_*`).
//
// The update of learner.cu for a stack of fully connected ReLU layers on flat fp32 observations, built from the same
// kernels: every matrix product on the tcgen05 GEMM (gemm.cu), the loss / column sums / sampling of layers.cu, the EMA,
// inverse refresh, preconditioning and optimizer steps of kfac.cu / kfac_inv.cu.  Only the two heads (any width, any
// action count) have kernels of their own here.  Everything runs in order on the caller's stream; acx_mlp_update is one
// captured CUDA graph per schedule variant.  The host code it shares with learner.cu (arena, K-FAC blocks and their state,
// schedule, inverse refresh, graph cache) lives in learner_core.cuh / learner_core.cu.
//   forward   obs -> bf16 planes; fc_i: GEMM with bias + ReLU + plane split in the epilogue; heads (one warp per row)
//   loss      K-RET + A2C loss + output gradients + Fisher-sample output gradients (loss_grad_kernel), rows [0,N) true
//             loss, rows [N,2N) Fisher samples
//   backward  heads: input gradient (masked, split), weight gradients, output factors; fc_i: weight gradient (MN-major
//             GEMM) + bias column sums over the true-loss rows, output factor SYRK over the Fisher rows, input gradient
//             (K-major GEMM with the ReLU mask of the layer below) over both
//   factors   input factors: SYRK over the layer's input + homogeneous border from its column sums
//   phase 2   as learner.cu issue_phase2: schedule step, cold momentum / EMA, scheduled inverse refresh, preconditioning,
//             KL clip + momentum + apply, or the A2C RMSProp step; then the weight operand planes
#include <algorithm>
#include <string>

#include "learner_core.cuh"

namespace acx {
namespace {

constexpr int kActPlanes = 2;        // default preset: activations and gradients on 2 planes, 3 plane pairs ...
constexpr int kLvl = 1;
constexpr int kLvlPrecon = 2;        // ... weights, inverses and preconditioning operands on 3 planes, 6 pairs

// ------------------------------------------------------------------------------------------------
// heads of any width H and 1..31 actions (the Atari head kernels of layers.cu are fixed at 512 inputs)
// ------------------------------------------------------------------------------------------------
// logits [R, A] = x W_pol + b_pol, values [R] = x W_val + b_val  (x = the planes of the last hidden layer); one warp per row
__global__ void mlp_heads_fwd_kernel(const Planes x, int H, const float* __restrict__ vpol, const float* __restrict__ vval, int rows,
                                     int num_actions, float* __restrict__ logits, float* __restrict__ values) {
  pdl_enter();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float acc[32];
#pragma unroll
  for (int a = 0; a < 32; ++a) acc[a] = 0.0f;
  for (int j = lane; j < H; j += 32) {
    const size_t idx = (size_t)row * x.ld + j;
    float v = __bfloat162float(x.p[0][idx]);
    if (x.n > 1) v += __bfloat162float(x.p[1][idx]);
#pragma unroll
    for (int a = 0; a < 32; ++a) {
      if (a < num_actions) acc[a] = fmaf(v, __ldg(vpol + (size_t)j * num_actions + a), acc[a]);
      else if (a == num_actions) acc[a] = fmaf(v, __ldg(vval + j), acc[a]);
    }
  }
#pragma unroll
  for (int a = 0; a < 32; ++a) {
    if (a > num_actions) break;
    const float s = warp_sum(acc[a]);
    if (lane == 0) {
      if (a < num_actions)
        logits[(size_t)row * num_actions + a] = s + vpol[(size_t)H * num_actions + a];
      else
        values[row] = s + vval[H];
    }
  }
}

// dpre[r, j] = (sum_a dH[r,a] W_pol[j,a] + dH[r,A] W_val[j]) * 1[x_hi[r % mask_rows, j] > 0] -> planes [rows, ld]
__global__ void mlp_heads_bwd_data_kernel(const float* __restrict__ dheads, const float* __restrict__ vpol,
                                          const float* __restrict__ vval, const bf16* __restrict__ x_hi, int H, int rows,
                                          int mask_rows, int num_actions, const Planes out) {
  pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)rows * H) return;
  const int j = (int)(i % H), r = (int)(i / H);
  const float* d = dheads + (size_t)r * (num_actions + 1);
  float acc = d[num_actions] * __ldg(vval + j);
  for (int a = 0; a < num_actions; ++a) acc = fmaf(d[a], __ldg(vpol + (size_t)j * num_actions + a), acc);
  const float m = __bfloat162float(x_hi[(size_t)(r % mask_rows) * out.ld + j]);
  if (!(m > 0.0f)) acc = 0.0f;
  bf16 hi, mid, lo;
  split3(acc, hi, mid, lo);
  const size_t o = (size_t)r * out.ld + j;
  out.p[0][o] = hi;
  if (out.n > 1) out.p[1][o] = mid;
  if (out.n > 2) out.p[2][o] = lo;
}

// weight gradients of the heads over the true-loss rows: g_pol[j,a] = sum_n x[n,j] dH[n,a], row j = H the bias row
// (sum_n dH[n,a]); the same for the value head.  One CTA per j, 128 threads over the rows, fixed-order reduction.
__global__ void __launch_bounds__(128) mlp_heads_wgrad_kernel(const float* __restrict__ dheads, const Planes x, int H, int n_rows,
                                                              int num_actions, float* __restrict__ gpol, float* __restrict__ gval) {
  pdl_enter();
  __shared__ float red[4][32];
  const int j = blockIdx.x;
  const int ld = num_actions + 1;
  float acc[32];
#pragma unroll
  for (int a = 0; a < 32; ++a) acc[a] = 0.f;
  for (int n = threadIdx.x; n < n_rows; n += blockDim.x) {
    float v = 1.0f;
    if (j < H) {
      const size_t idx = (size_t)n * x.ld + j;
      v = __bfloat162float(x.p[0][idx]);
      if (x.n > 1) v += __bfloat162float(x.p[1][idx]);
    }
    const float* d = dheads + (size_t)n * ld;
#pragma unroll
    for (int a = 0; a < 32; ++a)
      if (a < ld) acc[a] = fmaf(v, d[a], acc[a]);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int a = 0; a < 32; ++a) {
    if (a < ld) {
      const float s = warp_sum(acc[a]);
      if (lane == 0) red[warp][a] = s;
    }
  }
  __syncthreads();
  if (threadIdx.x < ld) {
    const int a = threadIdx.x;
    const float s = red[0][a] + red[1][a] + red[2][a] + red[3][a];
    if (a < num_actions)
      gpol[(size_t)j * num_actions + a] = s;
    else
      gval[j] = s;
  }
}

}  // namespace
}  // namespace acx

using namespace acx;

// the K-FAC blocks fc1 .. fcL, fc_policy, fc_baseline and their state (KfacBlocks), plus this model's activations
struct acx_mlp : KfacBlocks {
  acx_mlp_config_t cfg;
  int E, T, N, R, A, D, L;
  // inputs
  float* obs;
  uint8_t *actions, *terminals;
  float* rewards;
  // activations and gradients
  Planes x0;                 // observations [R, pad8(D)]
  Planes act[4];             // hidden activations [R, H_i]
  Planes dpre[4];            // pre-activation gradients [2N, H_i]
  Planes wT[4], wN[4];       // W^T [C, pad8(K)] (forward), W [K, C] (input gradient)
  float *logits, *values, *targets, *adv, *dheads;
  Planes Vp, Wt;             // preconditioning operands of blocks with C > 64
  float *dot_partials, *colsum_partial, *colsum_tmp, *ws;
  size_t ws_bytes;
  Schedule sch;
  GraphCache graphs;
};

namespace acx {
namespace {

void init_dims(acx_mlp* l, const acx_mlp_config_t* c) {
  l->cfg = *c;
  l->E = c->num_envs;
  l->T = c->num_steps;
  l->N = l->E * l->T;
  l->R = l->N + l->E;
  l->A = c->num_actions;
  l->D = c->obs_dim;
  l->L = c->num_hidden;
  int in = l->D;
  for (int i = 0; i < l->L + 2; ++i) {
    Block& b = l->blk[i];
    if (i < l->L) {
      b.name = "fc" + std::to_string(i + 1);
      b.K = in;
      b.C = c->hidden[i];
      b.afac = i;
      in = b.C;
    } else {
      b.name = i == l->L ? "fc_policy" : "fc_baseline";
      b.K = in;
      b.C = i == l->L ? l->A : 1;
      b.afac = l->L;
    }
  }
  l->set_blocks(l->L + 2);
  l->sch.acktr = c->acktr != 0;
  l->sch.num_cold_updates = c->num_cold_updates;
  l->sch.invert_every = c->invert_every;
}

// lay the arena out (base == nullptr: size pass only)
size_t layout(acx_mlp* l, uint8_t* base) {
  Arena ar;
  ar.base = base;
  const int N = l->N, R = l->R, A = l->A;
  l->take_state(ar);
  l->take_tables(ar);
  // inputs
  l->obs = ar.f32((size_t)R * l->D);
  l->actions = reinterpret_cast<uint8_t*>(ar.take(N));
  l->terminals = reinterpret_cast<uint8_t*>(ar.take(N));
  l->rewards = ar.f32(N);
  // weights as GEMM operands
  for (int i = 0; i < l->L; ++i) {
    l->wT[i] = take_planes(ar, 3, l->blk[i].C, pad8(l->blk[i].K));
    l->wN[i] = take_planes(ar, 3, l->blk[i].K, l->blk[i].C);
  }
  // activations (forward rows R = N + E) and gradients (backward rows 2N: true-loss rows, then Fisher-sample rows)
  l->x0 = take_planes(ar, kActPlanes, R, pad8(l->D));
  for (int i = 0; i < l->L; ++i) {
    l->act[i] = take_planes(ar, kActPlanes, R, l->blk[i].C);
    l->dpre[i] = take_planes(ar, kActPlanes, 2 * (size_t)N, l->blk[i].C);
  }
  l->logits = ar.f32((size_t)R * A);
  l->values = ar.f32(R);
  l->targets = ar.f32(N);
  l->adv = ar.f32(N);
  l->dheads = ar.f32(2 * (size_t)N * (A + 1));
  int dmax = 0, cmax = 0;
  for (int i = 0; i < l->nb; ++i) {
    dmax = std::max(dmax, l->blk[i].K + 1);
    cmax = std::max(cmax, l->blk[i].C);
  }
  l->Vp = take_planes(ar, 3, dmax, pad8(cmax));
  l->Wt = take_planes(ar, 3, cmax, pad8(dmax));
  l->dot_partials = ar.f32(kDotPartials);
  l->colsum_partial = ar.f32((size_t)kColsumChunks * pad8(dmax));
  l->colsum_tmp = ar.f32(pad8(dmax) + 8);
  const size_t kpad = align_up((size_t)dmax, 128);
  l->ws_bytes = std::max<size_t>((size_t)48 << 20, kpad * kpad * sizeof(float) + (1 << 20));
  l->ws = reinterpret_cast<float*>(ar.take(l->ws_bytes));   // split-K partials; its arrival counters start zero
  return align_up(ar.used, 256);
}

void register_buffers(acx_mlp* l) {
  l->register_buffers();
  l->reg("observations", l->obs, (size_t)l->R * l->D * 4);
  l->reg("actions", l->actions, l->N);
  l->reg("terminals", l->terminals, l->N);
  l->reg("rewards", l->rewards, (size_t)l->N * 4);
  l->reg("logits", l->logits, (size_t)l->R * l->A * 4);
  l->reg("values", l->values, (size_t)l->R * 4);
  l->reg("targets", l->targets, (size_t)l->N * 4);
  l->reg("advantages", l->adv, (size_t)l->N * 4);
  l->reg("dheads", l->dheads, (size_t)2 * l->N * (l->A + 1) * 4);
  for (int i = 0; i < l->L; ++i) l->reg("act_hi/" + l->blk[i].name, l->act[i].p[0], (size_t)l->R * l->act[i].ld * 2);
}

int run_gemm(acx_mlp* l, const Planes& a, const Planes& b, int trans, int m, int n, int k, int level, float alpha, int symmetric,
             const GemmOut& o, cudaStream_t st) {
  acx_gemm_t g;
  fill_gemm(&g, a, b, trans, m, n, k, level, alpha, symmetric, o, l->ws, l->ws_bytes);
  return gemm_dispatch(&g, 0, st);
}

int refresh_weight_planes(acx_mlp* l, cudaStream_t st) {
  const float* w[4];
  int kr[4], cc[4], ldt[4], ldn[4];
  bf16* t[4][3];
  bf16* n[4][3];
  for (int i = 0; i < l->L; ++i) {
    const Block& B = l->blk[i];
    w[i] = l->params + B.off;
    kr[i] = B.K;
    cc[i] = B.C;
    ldt[i] = l->wT[i].ld;
    ldn[i] = l->wN[i].ld;
    for (int q = 0; q < 3; ++q) {
      t[i][q] = l->wT[i].p[q];
      n[i][q] = i > 0 ? l->wN[i].p[q] : nullptr;   // fc1 has no input gradient: observations are constants
    }
  }
  return weight_planes(w, kr, cc, t, ldt, n, ldn, l->L, st);
}

// forward of `rows` observation rows: logits, values and the hidden activations (planes) stay in the arena
int forward(acx_mlp* l, const float* obs, int rows, cudaStream_t st) {
  ACX_TRY(split_planes(obs, l->D, rows, l->D, 1.0f, l->x0.p[0], l->x0.p[1], nullptr, l->x0.n, l->x0.ld, st));
  for (int i = 0; i < l->L; ++i) {
    const Block& B = l->blk[i];
    GemmOut o;
    o.bias = l->params + B.off + (size_t)B.K * B.C;
    o.relu = 1;
    o.planes = &l->act[i];
    ACX_TRY(run_gemm(l, i == 0 ? l->x0 : l->act[i - 1], l->wT[i], 0, rows, B.C, B.K, kLvl, 1.0f, 0, o, st));
  }
  const Block& P = l->blk[l->L];
  const Block& V = l->blk[l->L + 1];
  ACX_PDL_LAUNCH(mlp_heads_fwd_kernel, ceil_div(rows, 8), 256, 0, st, l->act[l->L - 1], P.K, l->params + P.off,
                 l->params + V.off, rows, l->A, l->logits, l->values);
  return 0;
}

int issue_update_phase1(acx_mlp* l, const int32_t* fl, const float* fe, bool fisher, cudaStream_t st) {
  const int N = l->N, E = l->E, T = l->T, A = l->A, L = l->L;
  const int RB = fisher ? 2 * N : N;
  const float inv_n = 1.0f / (float)N;
  ACX_TRY(forward(l, l->obs, l->R, st));
  // targets use the bootstrap rows' values = rows [N, N+E)
  ACX_TRY(returns_loss_grad(l->rewards, l->terminals, l->values + N, l->cfg.gamma, E, T, l->targets, l->adv, l->logits, l->values,
                            l->actions, fl, fe, l->cfg.seed, l->sched, A, l->cfg.entropy_beta, l->cfg.value_loss_weight, l->dheads,
                            l->bscalars, fisher ? 1 : 0, st));
  // heads
  const Block& P = l->blk[L];
  const Block& V = l->blk[L + 1];
  const Planes& xh = l->act[L - 1];
  {
    const long long total = (long long)RB * P.K;
    ACX_PDL_LAUNCH(mlp_heads_bwd_data_kernel, (unsigned)((total + 255) / 256), 256, 0, st, l->dheads, l->params + P.off,
                   l->params + V.off, xh.p[0], P.K, RB, N, A, l->dpre[L - 1]);
    ACX_PDL_LAUNCH(mlp_heads_wgrad_kernel, P.K + 1, 128, 0, st, l->dheads, xh, P.K, N, A, l->grads + P.off, l->grads + V.off);
  }
  if (fisher) ACX_TRY(heads_gfactor(l->dheads + (size_t)N * (A + 1), N, A, l->stats + l->goff[L], l->stats + l->goff[L + 1], st));
  // hidden layers, last to first
  for (int i = L - 1; i >= 0; --i) {
    const Block& B = l->blk[i];
    const Planes& g = l->dpre[i];
    const Planes& x = i == 0 ? l->x0 : l->act[i - 1];
    GemmOut ow;   // V[:K] = x^T g over the true-loss rows
    ow.c = l->grads + B.off;
    ow.ldc = B.C;
    ACX_TRY(run_gemm(l, x, g, 1, B.K, B.C, N, kLvl, 1.0f, 0, ow, st));
    ACX_TRY(colsum(g, N, B.C, 1.0f, l->colsum_partial, kColsumChunks, l->grads + B.off + (size_t)B.K * B.C, 1, st));
    if (fisher) {   // G = g^T g / N over the Fisher rows
      GemmOut og;
      og.c = l->stats + l->goff[i];
      og.ldc = B.C;
      ACX_TRY(run_gemm(l, offset_rows(g, N), offset_rows(g, N), 1, B.C, B.C, N, kLvl, inv_n, 1, og, st));
    }
    if (i > 0) {   // input gradient of both halves, masked by the ReLU of the layer below (the Fisher half reuses the masks)
      GemmOut od;
      od.planes = &l->dpre[i - 1];
      od.mask = l->act[i - 1].p[0];
      od.mask_ld = l->act[i - 1].ld;
      od.mask_rows = N;
      ACX_TRY(run_gemm(l, g, l->wN[i], 0, RB, B.K, B.C, kLvl, 1.0f, 0, od, st));
    }
  }
  if (fisher) {   // A = [x 1]^T [x 1] / N over the train rows: SYRK, then the border from the column sums (pad columns are zero)
    for (int f = 0; f <= L; ++f) {
      const Planes& x = f == 0 ? l->x0 : l->act[f - 1];
      const int d = l->adim[f];
      float* dst = l->stats + l->aoff[f];
      GemmOut o;
      o.c = dst;
      o.ldc = d;
      ACX_TRY(run_gemm(l, x, x, 1, d - 1, d - 1, N, kLvl, inv_n, 1, o, st));
      ACX_TRY(colsum(x, N, x.ld, inv_n, l->colsum_partial, kColsumChunks, l->colsum_tmp, 1, st));
      ACX_TRY(homog_border(dst, d, l->colsum_tmp, st));
    }
  }
  return 0;
}

int precondition(acx_mlp* l, cudaStream_t st) {
  ACX_TRY(precondition_small(l->d_pjobs, l->num_pjobs, l->pjobs_max_d, st));
  for (int i = 0; i < l->nb; ++i) {
    const Block& B = l->blk[i];
    const int d = B.K + 1, C = B.C;
    if (C <= 64) continue;
    Planes vp = l->Vp;
    vp.ld = pad8(C);
    Planes wt = l->Wt;
    wt.ld = pad8(d);
    ACX_TRY(split_planes(l->grads + B.off, C, d, C, 1.0f, vp.p[0], vp.p[1], vp.p[2], 3, vp.ld, st));
    GemmOut o1;   // Wt [C, d] = G^-1 V^T
    o1.planes = &wt;
    ACX_TRY(run_gemm(l, l->ginv_pl[i], vp, 0, C, d, C, kLvlPrecon, 1.0f, 0, o1, st));
    GemmOut o2;   // U [d, C] = A^-1 W
    o2.c = l->precon + B.off;
    o2.ldc = C;
    ACX_TRY(run_gemm(l, l->ainv_pl[i], wt, 0, d, C, d, kLvlPrecon, 1.0f, 0, o2, st));
  }
  return 0;
}

int issue_update_phase2(acx_mlp* l, const Plan& p, cudaStream_t st) {
  const acx_mlp_config_t& c = l->cfg;
  const size_t P = l->num_params;
  ACX_CUDA(cudaMemcpyAsync(l->scalars, l->bscalars, 4 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // lr from the step the update starts with, then global_step += (cold ? 2 : 1) [A2C: 1], covariance counter += (cold ? 0 : 1)
  ACX_TRY(sched_step(l->sched, c.lr_start, c.lr_end, c.lr_decay_steps, l->scalars + 7, p.a2c ? 1 : (p.cold ? 2 : 1),
                     (p.a2c || p.cold) ? 0 : 1, c.cov_ema_decay, 1, st));
  if (p.a2c) {   // ClipGlobalNorm(RMSProp)   a2c_acktr.py:250-251
    ACX_TRY(dot_partial(l->grads, l->grads, P, l->dot_partials, kDotPartials, st));
    ACX_TRY(rmsprop_clip_step(l->params, l->accum, l->grads, P, l->dot_partials, kDotPartials, l->sched, c.rms_decay, c.rms_epsilon,
                              c.clip_norm, l->scalars + 6, st));
    return refresh_weight_planes(l, st);
  }
  if (p.cold) {   // kfac_utils.py:42-43: ClipGlobalNorm(Momentum)
    ACX_TRY(dot_partial(l->grads, l->grads, P, l->dot_partials, kDotPartials, st));
    ACX_TRY(momentum_clip_step(l->params, l->accum, l->grads, P, l->dot_partials, kDotPartials, c.cold_lr, c.cold_momentum,
                               c.clip_norm, l->scalars + 6, st));
  } else {        // :44 covariance updates
    ACX_TRY(ema_update(l->sums, l->stats, l->factor_floats, c.cov_ema_decay, 1.0f, st));
  }
  if (p.invert) ACX_TRY(l->invert(st));   // as the Atari learner: factor tiles resident in shared memory, else the fp64 chain
  if (p.kfac_apply) {
    ACX_TRY(precondition(l, st));
    ACX_TRY(dot_partial(l->grads, l->precon, P, l->dot_partials, kDotPartials, st));
    ACX_TRY(kfac_step(l->params, l->velocity, l->precon, P, l->dot_partials, kDotPartials, l->sched, c.momentum, c.norm_constraint,
                      l->scalars + 4, st));
  }
  if (p.refresh) ACX_TRY(refresh_weight_planes(l, st));
  return 0;
}

int check_cfg(const acx_mlp_config_t* c) {
  ACX_CHECK(c != nullptr, "null config");
  ACX_CHECK(c->num_envs > 0 && c->num_steps > 0, "num_envs and num_steps must be positive");
  ACX_CHECK((long long)c->num_envs * c->num_steps <= (1 << 20), "rollout too large");
  ACX_CHECK(c->obs_dim >= 1 && c->obs_dim <= 2048, "obs_dim must be in [1, 2048]");
  ACX_CHECK(c->num_hidden >= 1 && c->num_hidden <= 4, "num_hidden must be in [1, 4]");
  for (int i = 0; i < c->num_hidden; ++i)
    ACX_CHECK(c->hidden[i] >= 8 && c->hidden[i] <= 1024 && c->hidden[i] % 8 == 0, "hidden sizes must be multiples of 8 in [8, 1024]");
  ACX_CHECK(c->num_actions >= 1 && c->num_actions <= 31, "num_actions must be in [1, 31]");
  if (c->acktr) ACX_CHECK(c->invert_every >= 1, "invert_every");
  return 0;
}

}  // namespace
}  // namespace acx

extern "C" {

size_t acx_mlp_arena_bytes(const acx_mlp_config_t* cfg) {
  if (check_cfg(cfg)) return 0;
  acx_mlp tmp;
  init_dims(&tmp, cfg);
  return layout(&tmp, nullptr);
}

acx_mlp_t* acx_mlp_create(const acx_mlp_config_t* cfg, void* d_arena, size_t arena_bytes) {
  if (check_cfg(cfg)) return nullptr;
  acx_mlp* l = new acx_mlp();
  init_dims(l, cfg);
  const size_t need = layout(l, nullptr);
  if (d_arena == nullptr || arena_bytes < need || (reinterpret_cast<uintptr_t>(d_arena) & 255) != 0) {
    set_error("acx_mlp_create: arena must be a 256-byte aligned device buffer of at least acx_mlp_arena_bytes()");
    delete l;
    return nullptr;
  }
  layout(l, reinterpret_cast<uint8_t*>(d_arena));
  register_buffers(l);
  // zero everything persistent (pad columns of the operand planes included)
  if (l->upload(d_arena, need, !cfg->acktr, cfg->lr_start, cfg->damping) != 0) {
    delete l;
    return nullptr;
  }
  return l;
}

void acx_mlp_destroy(acx_mlp_t* l) { delete l; }

size_t acx_mlp_num_params(const acx_mlp_t* l) { return l ? l->num_params : 0; }

int acx_mlp_set_params(acx_mlp_t* l, const float* h_params, void* stream) {
  ACX_CHECK(l && h_params, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ACX_TRY(l->set_params(h_params, st));
  ACX_TRY(refresh_weight_planes(l, st));
  ACX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int acx_mlp_get_params(acx_mlp_t* l, float* h_params, void* stream) {
  ACX_CHECK(l && h_params, "null argument");
  return l->get_params(h_params, reinterpret_cast<cudaStream_t>(stream));
}

int acx_mlp_refresh_weights(acx_mlp_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ACX_TRY(refresh_weight_planes(l, st));
  return l->split_inverses(st);
}

void* acx_mlp_buffer(acx_mlp_t* l, const char* name, size_t* num_bytes) {
  return l ? l->buffer("acx_mlp_buffer", name, num_bytes) : nullptr;
}

int acx_mlp_update(acx_mlp_t* l, const int32_t* d_fisher_labels, const float* d_fisher_eps, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK((d_fisher_labels == nullptr) == (d_fisher_eps == nullptr), "inject both Fisher labels and eps, or neither");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool fisher = l->sch.fisher();
  const Plan p = l->sch.plan();
  const GraphKey key = {0, p.key() | (fisher ? 32 : 0), d_fisher_labels, d_fisher_eps};
  ACX_TRY(l->graphs.run(key, st, !l->cfg.use_graphs, [&]() {
    const int r1 = issue_update_phase1(l, d_fisher_labels, d_fisher_eps, fisher, st);
    return r1 ? r1 : issue_update_phase2(l, p, st);
  }));
  l->sch.advance(p);
  return 0;
}

int64_t acx_mlp_global_step(const acx_mlp_t* l) { return l ? l->sch.gs : -1; }

int acx_mlp_set_state(acx_mlp_t* l, int64_t global_step, int64_t num_cov_updates, int inverses_valid, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK(global_step >= 0 && num_cov_updates >= 0, "negative counters");
  return l->sch.set(global_step, num_cov_updates, inverses_valid, l->cfg.lr_start, l->cfg.cov_ema_decay, true, l->sched,
                    reinterpret_cast<cudaStream_t>(stream));
}

int acx_mlp_get_state(const acx_mlp_t* l, int64_t* global_step, int64_t* num_cov_updates, int* inverses_valid) {
  ACX_CHECK(l, "null learner");
  l->sch.get(global_step, num_cov_updates, inverses_valid);
  return 0;
}

int acx_mlp_act(acx_mlp_t* l, const float* d_obs, int rows, const float* d_uniform, int greedy, int32_t* d_actions,
                float* d_logits, float* d_values, void* stream) {
  ACX_CHECK(l && d_obs && d_actions, "null argument");
  ACX_CHECK(rows > 0 && rows <= l->R, "rows must be in [1, num_envs * num_steps + num_envs]");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  auto issue = [&]() -> int {
    ACX_TRY(forward(l, d_obs, rows, st));
    ACX_TRY(sample_actions(l->logits, d_uniform, l->cfg.seed, 0, rows, l->A, greedy, d_actions, st, l->act_counter));
    if (d_logits) ACX_CUDA(cudaMemcpyAsync(d_logits, l->logits, (size_t)rows * l->A * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (d_values) ACX_CUDA(cudaMemcpyAsync(d_values, l->values, (size_t)rows * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  };
  const GraphKey key = {1, (greedy ? 1 : 0) | (rows << 1), d_obs, d_actions, d_uniform, d_logits, d_values};
  return l->graphs.run_bounded(key, st, !l->cfg.use_graphs, issue);
}

}  // extern "C"
