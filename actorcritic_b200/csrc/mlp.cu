// mlp.cu - the ACKTR / A2C learner for fully connected actor-critic models (include/acx.h `acx_mlp_*`).
//
// The update of learner.cu for a stack of fully connected ReLU layers on flat fp32 observations, built from the same
// kernels: every matrix product on the tcgen05 GEMM (gemm.cu), the loss / column sums / sampling of layers.cu, the EMA,
// inverse refresh, preconditioning and optimizer steps of kfac.cu / kfac_inv.cu.  Only the two heads (any width, any
// action count) have kernels of their own here.  Everything runs in order on the caller's stream; acx_mlp_update is one
// captured CUDA graph per schedule variant.
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
#include <cmath>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "layers.cuh"

namespace acx {
namespace {

constexpr int kMaxLayers = 6;        // 4 hidden layers + the two heads
constexpr int kColsumChunks = 592;
constexpr int kDotPartials = 296;
constexpr int kActPlanes = 2;        // default preset: activations and gradients on 2 planes, 3 plane pairs ...
constexpr int kLvl = 1;
constexpr int kLvlPrecon = 2;        // ... weights, inverses and preconditioning operands on 3 planes, 6 pairs

struct Block {
  std::string name;
  int K, C;          // V_l = [K+1, C]
  size_t off;        // offset in the flat parameter vector
  int afac;          // input factor (the two heads share one)
};

struct Buf {
  void* ptr;
  size_t bytes;
};

struct Arena {
  uint8_t* base = nullptr;
  size_t used = 0;
  void* take(size_t bytes) {
    used = align_up(used, 256);
    void* p = base ? base + used : nullptr;
    used += bytes;
    return p;
  }
};

struct GraphEntry {
  int uses = 0;
  cudaGraphExec_t exec = nullptr;
  uint64_t launches = 0;
};
typedef std::tuple<int, const void*, const void*, const void*, const void*, const void*> GraphKey;

int pad8(int x) { return (x + 7) / 8 * 8; }

Planes take_planes(Arena& ar, int nplanes, size_t rows, int ld) {
  Planes pl;
  pl.n = nplanes;
  pl.ld = ld;
  for (int i = 0; i < nplanes; ++i) pl.p[i] = reinterpret_cast<bf16*>(ar.take(rows * (size_t)ld * sizeof(bf16)));
  return pl;
}

Planes offset_rows(const Planes& p, size_t rows) {
  Planes q = p;
  for (int i = 0; i < p.n; ++i) q.p[i] = p.p[i] + rows * (size_t)p.ld;
  return q;
}

// plane pairs (i, j) with i + j <= level, low orders first
int level_pairs(int level, int a_planes, int b_planes, int* pa, int* pb) {
  int np = 0;
  for (int s = 0; s <= level && np < 6; ++s)
    for (int i = 0; i <= s && np < 6; ++i) {
      const int j = s - i;
      if (i < a_planes && j < b_planes) {
        pa[np] = i;
        pb[np] = j;
        ++np;
      }
    }
  return np;
}

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

struct acx_mlp {
  acx_mlp_config_t cfg;
  int E, T, N, R, A, D, L, NL;
  Block blk[kMaxLayers];
  size_t num_params, params_pad;
  int adim[kMaxLayers - 1];
  size_t aoff[kMaxLayers - 1], goff[kMaxLayers], factor_floats;
  size_t ainv_off[kMaxLayers], ginv_off[kMaxLayers], inv_floats;
  // fp32 state
  float *params, *velocity, *accum, *precon, *precon_w;
  float *bucket, *stats, *grads, *bscalars;
  size_t bucket_floats;
  float *sums, *inv, *damp, *lambdas, *scalars;
  Planes ainv_pl[kMaxLayers], ginv_pl[kMaxLayers];
  Sched* sched;
  const float** d_a_ptrs;
  const float** d_g_ptrs;
  int *d_a_dims, *d_g_dims;
  InvJob h_jobs[2 * kMaxLayers];
  InvJob* d_jobs;
  unsigned int* inv_bar;
  unsigned long long* act_counter;
  PreconJob h_pjobs[kMaxLayers];
  PreconJob* d_pjobs;
  int num_pjobs, pjobs_max_d;
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
  // host mirror of the schedule
  int64_t gs, ncov;
  bool inverses_valid;
  std::map<std::string, Buf> named;
  std::map<GraphKey, GraphEntry> graphs;
};

namespace acx {
namespace {

#define ACX_TRY(expr)        \
  do {                       \
    int _r = (expr);         \
    if (_r) return _r;       \
  } while (0)

void init_dims(acx_mlp* l, const acx_mlp_config_t* c) {
  l->cfg = *c;
  l->E = c->num_envs;
  l->T = c->num_steps;
  l->N = l->E * l->T;
  l->R = l->N + l->E;
  l->A = c->num_actions;
  l->D = c->obs_dim;
  l->L = c->num_hidden;
  l->NL = l->L + 2;
  size_t off = 0;
  int in = l->D;
  for (int i = 0; i < l->NL; ++i) {
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
    b.off = off;
    off += (size_t)(b.K + 1) * b.C;
  }
  l->num_params = off;
  l->params_pad = align_up(off, 4);
  size_t f = 0;
  for (int i = 0; i <= l->L; ++i) {
    l->adim[i] = (i < l->L ? l->blk[i].K : l->blk[l->L].K) + 1;
    l->aoff[i] = f;
    f += align_up((size_t)l->adim[i] * l->adim[i], 4);
  }
  for (int i = 0; i < l->NL; ++i) {
    l->goff[i] = f;
    f += align_up((size_t)l->blk[i].C * l->blk[i].C, 4);
  }
  l->factor_floats = f;
  size_t v = 0;
  for (int i = 0; i < l->NL; ++i) {
    l->ainv_off[i] = v;
    v += align_up((size_t)(l->blk[i].K + 1) * (l->blk[i].K + 1), 4);
  }
  for (int i = 0; i < l->NL; ++i) {
    l->ginv_off[i] = v;
    v += align_up((size_t)l->blk[i].C * l->blk[i].C, 4);
  }
  l->inv_floats = v;
}

// lay the arena out (base == nullptr: size pass only)
size_t layout(acx_mlp* l, uint8_t* base) {
  Arena ar;
  ar.base = base;
  const int N = l->N, R = l->R, A = l->A, NL = l->NL;
  const size_t P = l->params_pad, F = l->factor_floats;
  auto f32 = [&](size_t n) { return reinterpret_cast<float*>(ar.take(n * sizeof(float))); };
  l->params = f32(P);
  l->velocity = f32(P);
  l->accum = f32(P);
  l->precon = f32(P);
  l->bucket_floats = P + F + 4;
  l->bucket = f32(l->bucket_floats);   // [A | G | grads | 4 loss scalars], as acx_learner's reduce bucket
  l->stats = l->bucket;
  l->grads = l->bucket + F;
  l->bscalars = l->bucket + F + P;
  l->sums = f32(F);
  l->inv = f32(l->inv_floats);
  l->damp = f32(16);
  l->lambdas = f32(8);
  l->scalars = f32(16);
  l->sched = reinterpret_cast<Sched*>(ar.take(sizeof(Sched)));
  l->d_a_ptrs = reinterpret_cast<const float**>(ar.take(kMaxLayers * sizeof(float*)));
  l->d_g_ptrs = reinterpret_cast<const float**>(ar.take(kMaxLayers * sizeof(float*)));
  l->d_a_dims = reinterpret_cast<int*>(ar.take(kMaxLayers * sizeof(int)));
  l->d_g_dims = reinterpret_cast<int*>(ar.take(kMaxLayers * sizeof(int)));
  l->d_jobs = reinterpret_cast<InvJob*>(ar.take(2 * kMaxLayers * sizeof(InvJob)));
  l->d_pjobs = reinterpret_cast<PreconJob*>(ar.take(kMaxLayers * sizeof(PreconJob)));
  l->inv_bar = reinterpret_cast<unsigned int*>(ar.take(256));
  l->act_counter = reinterpret_cast<unsigned long long*>(ar.take(256));
  l->precon_w = f32(P);
  for (int i = 0; i < NL; ++i) {
    const int d = l->blk[i].K + 1, c = l->blk[i].C;
    l->ainv_pl[i] = take_planes(ar, 3, d, pad8(d));
    l->ginv_pl[i] = take_planes(ar, 3, c, pad8(c));
  }
  for (int i = 0; i < NL; ++i) {   // inverse jobs (sorted by decreasing n at create)
    const int d = l->blk[i].K + 1, c = l->blk[i].C;
    InvJob& ja = l->h_jobs[i];
    ja.s = l->sums + l->aoff[l->blk[i].afac];
    ja.n = d;
    ja.damp_index = 2 * i;
    ja.work_m = reinterpret_cast<double*>(ar.take((size_t)d * d * sizeof(double)));
    ja.work_x = reinterpret_cast<double*>(ar.take(((size_t)3 * 32 * d + 2 * 32 * 32 + 2048) * sizeof(double)));
    ja.inv = l->inv + l->ainv_off[i];
    for (int q = 0; q < 3; ++q) ja.planes[q] = l->ainv_pl[i].p[q];
    ja.ld_planes = l->ainv_pl[i].ld;
    InvJob& jg = l->h_jobs[NL + i];
    jg.s = l->sums + l->goff[i];
    jg.n = c;
    jg.damp_index = 2 * i + 1;
    jg.work_m = reinterpret_cast<double*>(ar.take((size_t)c * c * sizeof(double)));
    jg.work_x = reinterpret_cast<double*>(ar.take(((size_t)3 * 32 * c + 2 * 32 * 32 + 2048) * sizeof(double)));
    jg.inv = l->inv + l->ginv_off[i];
    for (int q = 0; q < 3; ++q) jg.planes[q] = l->ginv_pl[i].p[q];
    jg.ld_planes = l->ginv_pl[i].ld;
  }
  l->num_pjobs = 0;
  l->pjobs_max_d = 0;
  for (int i = 0; i < NL; ++i) {   // blocks with C <= 64: batched fp32 SIMT preconditioning
    if (l->blk[i].C > 64) continue;
    PreconJob& pj = l->h_pjobs[l->num_pjobs++];
    pj.v = l->grads + l->blk[i].off;
    pj.ginv = l->inv + l->ginv_off[i];
    pj.ainv = l->inv + l->ainv_off[i];
    pj.w = l->precon_w + l->blk[i].off;
    pj.u = l->precon + l->blk[i].off;
    pj.d = l->blk[i].K + 1;
    pj.c = l->blk[i].C;
    pj.scale = 1.0f;   // fully connected: T~ = 1
    l->pjobs_max_d = std::max(l->pjobs_max_d, pj.d);
  }
  // inputs
  l->obs = f32((size_t)R * l->D);
  l->actions = reinterpret_cast<uint8_t*>(ar.take(N));
  l->terminals = reinterpret_cast<uint8_t*>(ar.take(N));
  l->rewards = f32(N);
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
  l->logits = f32((size_t)R * A);
  l->values = f32(R);
  l->targets = f32(N);
  l->adv = f32(N);
  l->dheads = f32(2 * (size_t)N * (A + 1));
  int dmax = 0, cmax = 0;
  for (int i = 0; i < NL; ++i) {
    dmax = std::max(dmax, l->blk[i].K + 1);
    cmax = std::max(cmax, l->blk[i].C);
  }
  l->Vp = take_planes(ar, 3, dmax, pad8(cmax));
  l->Wt = take_planes(ar, 3, cmax, pad8(dmax));
  l->dot_partials = f32(kDotPartials);
  l->colsum_partial = f32((size_t)kColsumChunks * pad8(dmax));
  l->colsum_tmp = f32(pad8(dmax) + 8);
  const size_t kpad = align_up((size_t)dmax, 128);
  l->ws_bytes = std::max<size_t>((size_t)48 << 20, kpad * kpad * sizeof(float) + (1 << 20));
  l->ws = reinterpret_cast<float*>(ar.take(l->ws_bytes));   // split-K partials; its arrival counters start zero
  return align_up(ar.used, 256);
}

void reg(acx_mlp* l, const std::string& name, void* p, size_t bytes) { l->named[name] = Buf{p, bytes}; }

void register_buffers(acx_mlp* l) {
  const size_t P = l->num_params;
  reg(l, "params", l->params, P * 4);
  reg(l, "velocity", l->velocity, P * 4);
  reg(l, "accum", l->accum, P * 4);
  reg(l, "precon", l->precon, P * 4);
  reg(l, "grads", l->grads, P * 4);
  reg(l, "reduce_bucket", l->bucket, l->bucket_floats * 4);
  reg(l, "factor_stats", l->stats, l->factor_floats * 4);
  reg(l, "factor_sums", l->sums, l->factor_floats * 4);
  reg(l, "inverses", l->inv, l->inv_floats * 4);
  reg(l, "dampings", l->damp, 2 * l->NL * 4);
  reg(l, "scalars", l->scalars, 16 * 4);
  reg(l, "sched", l->sched, sizeof(Sched));
  reg(l, "observations", l->obs, (size_t)l->R * l->D * 4);
  reg(l, "actions", l->actions, l->N);
  reg(l, "terminals", l->terminals, l->N);
  reg(l, "rewards", l->rewards, (size_t)l->N * 4);
  reg(l, "logits", l->logits, (size_t)l->R * l->A * 4);
  reg(l, "values", l->values, (size_t)l->R * 4);
  reg(l, "targets", l->targets, (size_t)l->N * 4);
  reg(l, "advantages", l->adv, (size_t)l->N * 4);
  reg(l, "dheads", l->dheads, (size_t)2 * l->N * (l->A + 1) * 4);
  for (int i = 0; i < l->L; ++i)
    reg(l, "act_hi/" + l->blk[i].name, l->act[i].p[0], (size_t)l->R * l->act[i].ld * 2);
  for (int f = 0; f <= l->L; ++f) {
    const std::string fn = f < l->L ? l->blk[f].name : "heads";
    const size_t b = (size_t)l->adim[f] * l->adim[f] * 4;
    reg(l, "stats/A/" + fn, l->stats + l->aoff[f], b);
    reg(l, "sums/A/" + fn, l->sums + l->aoff[f], b);
  }
  for (int i = 0; i < l->NL; ++i) {
    const Block& B = l->blk[i];
    const size_t gb = (size_t)B.C * B.C * 4, vb = (size_t)(B.K + 1) * B.C * 4;
    reg(l, "stats/G/" + B.name, l->stats + l->goff[i], gb);
    reg(l, "sums/G/" + B.name, l->sums + l->goff[i], gb);
    reg(l, "inv/A/" + B.name, l->inv + l->ainv_off[i], (size_t)(B.K + 1) * (B.K + 1) * 4);
    reg(l, "inv/G/" + B.name, l->inv + l->ginv_off[i], gb);
    reg(l, "params/" + B.name, l->params + B.off, vb);
    reg(l, "grads/" + B.name, l->grads + B.off, vb);
    reg(l, "precon/" + B.name, l->precon + B.off, vb);
    reg(l, "velocity/" + B.name, l->velocity + B.off, vb);
    reg(l, "accum/" + B.name, l->accum + B.off, vb);
  }
}

struct GemmOut {
  float* c = nullptr;
  int ldc = 0;
  const Planes* planes = nullptr;
  const float* bias = nullptr;
  int relu = 0;
  const bf16* mask = nullptr;
  int mask_ld = 0, mask_rows = 0;
};

int run_gemm(acx_mlp* l, const Planes& a, const Planes& b, int trans, int m, int n, int k, int level, float alpha, int symmetric,
             const GemmOut& o, cudaStream_t st) {
  acx_gemm_t g;
  memset(&g, 0, sizeof(g));
  for (int i = 0; i < a.n; ++i) g.a.planes[i] = a.p[i];
  for (int i = 0; i < b.n; ++i) g.b.planes[i] = b.p[i];
  g.a.num_planes = a.n;
  g.b.num_planes = b.n;
  g.a.ld = a.ld;
  g.b.ld = b.ld;
  if (trans) {
    g.a.rows = k; g.a.cols = m; g.b.rows = k; g.b.cols = n;
  } else {
    g.a.rows = m; g.a.cols = k; g.b.rows = n; g.b.cols = k;
  }
  g.trans_a = g.trans_b = trans;
  g.m = m; g.n = n; g.k = k;
  g.num_pairs = level_pairs(level, a.n, b.n, g.pair_a, g.pair_b);
  g.alpha = alpha;
  g.bias = o.bias;
  g.relu = o.relu;
  g.symmetric = symmetric;
  g.c = o.c;
  g.ldc = o.ldc;
  if (o.planes) {
    for (int i = 0; i < o.planes->n; ++i) g.c_planes[i] = o.planes->p[i];
    g.c_num_planes = o.planes->n;
    g.ldc_planes = o.planes->ld;
  }
  g.mask_plane = o.mask;
  g.mask_ld = o.mask_ld;
  g.mask_rows = o.mask_rows;
  g.workspace = l->ws;
  g.workspace_bytes = l->ws_bytes;
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

// what one update's optimizer step does, decided on the host from the schedule counters (kfac_utils.py:38-53)
struct Plan {
  bool a2c, cold, invert, kfac_apply, refresh;
  int key() const { return (a2c ? 1 : 0) | (cold ? 2 : 0) | (invert ? 4 : 0) | (kfac_apply ? 8 : 0) | (refresh ? 16 : 0); }
};

Plan plan_update(const acx_mlp* l) {
  const acx_mlp_config_t& c = l->cfg;
  Plan p = {false, false, false, false, false};
  if (!c.acktr) {
    p.a2c = true;
    p.refresh = true;
    return p;
  }
  p.cold = l->gs < c.num_cold_updates;
  const int64_t gs1 = l->gs + (p.cold ? 1 : 0);   // the cold optimizer increments global_step itself (kfac_utils.py:43)
  p.invert = gs1 > c.num_cold_updates && (gs1 - c.num_cold_updates) % c.invert_every == 0;
  // the always-run K-FAC apply (kfac_utils.py:52-53) is a no-op with zero inverses until the first refresh
  p.kfac_apply = l->inverses_valid || p.invert;
  p.refresh = p.cold || p.kfac_apply;
  return p;
}

void advance(acx_mlp* l, const Plan& p) {
  if (p.a2c) {
    l->gs += 1;
    return;
  }
  if (p.cold) l->gs += 1; else l->ncov += 1;
  if (p.invert) l->inverses_valid = true;
  l->gs += 1;
}

int precondition(acx_mlp* l, cudaStream_t st) {
  ACX_TRY(precondition_small(l->d_pjobs, l->num_pjobs, l->pjobs_max_d, st));
  for (int i = 0; i < l->NL; ++i) {
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
  if (p.invert) {   // the Atari learner's selection: factor tiles resident in shared memory, else the fp64 chain
    const int jobs = 2 * l->NL;
    const int r = spd_inverse_resident(l->h_jobs, jobs, l->sched, l->damp, l->d_a_ptrs, l->d_g_ptrs, l->d_a_dims, l->d_g_dims,
                                       l->lambdas, l->NL, l->inv_bar, st);
    if (r > 0) return r;
    if (r < 0) {
      ACX_TRY(compute_dampings(l->d_a_ptrs, l->d_g_ptrs, l->d_a_dims, l->d_g_dims, l->lambdas, l->NL, l->damp, st));
      ACX_TRY(spd_inverse_batched(l->h_jobs, l->d_jobs, jobs, l->sched, l->damp, st));
    }
  }
  if (p.kfac_apply) {
    ACX_TRY(precondition(l, st));
    ACX_TRY(dot_partial(l->grads, l->precon, P, l->dot_partials, kDotPartials, st));
    ACX_TRY(kfac_step(l->params, l->velocity, l->precon, P, l->dot_partials, kDotPartials, l->sched, c.momentum, c.norm_constraint,
                      l->scalars + 4, st));
  }
  if (p.refresh) ACX_TRY(refresh_weight_planes(l, st));
  return 0;
}

// CUDA-graph cache as learner.cu's run_cached: the first use of a variant runs eagerly (one-time host work such as tensor-map
// encoding), the second is captured and instantiated, later uses replay it.  Valid because no kernel takes a step-dependent
// scalar by value (Sched).
template <typename F>
int run_cached(acx_mlp* l, const GraphKey& key, cudaStream_t st, F&& issue) {
  if (!l->cfg.use_graphs || st == nullptr) return issue();
  {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive) return issue();
  }
  GraphEntry& ge = l->graphs[key];
  if (ge.uses == 0) {
    ge.uses = 1;
    return issue();
  }
  if (ge.exec == nullptr) {
    const uint64_t before = g_launch_count;
    ACX_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    const int r = issue();
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (r != 0 || e != cudaSuccess || graph == nullptr) {
      if (graph) cudaGraphDestroy(graph);
      if (r == 0) set_error(std::string("graph capture failed: ") + cudaGetErrorString(e));
      return r ? r : 4;
    }
    ge.launches = g_launch_count - before;
    g_launch_count = before;
    const cudaError_t e2 = cudaGraphInstantiate(&ge.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e2 != cudaSuccess) {
      ge.exec = nullptr;
      set_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e2));
      return 4;
    }
  }
  ACX_CUDA(cudaGraphLaunch(ge.exec, st));
  count_launch((int)ge.launches);
  ge.uses += 1;
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
  l->gs = 0;
  l->ncov = 0;
  l->inverses_valid = false;
  // zero everything persistent (pad columns of the operand planes included); RMSProp's ms starts at one (TF-1 default)
  cudaError_t e = cudaMemset(d_arena, 0, need);
  std::vector<float> ones;
  if (e == cudaSuccess && !cfg->acktr) {
    ones.assign(l->params_pad, 1.0f);
    e = cudaMemcpy(l->accum, ones.data(), l->params_pad * 4, cudaMemcpyHostToDevice);
  }
  Sched s0 = {0ull, 0ull, cfg->lr_start, 1.0f};
  if (e == cudaSuccess) e = cudaMemcpy(l->sched, &s0, sizeof(s0), cudaMemcpyHostToDevice);
  const float* ap[kMaxLayers];
  const float* gp[kMaxLayers];
  int ad[kMaxLayers], gd[kMaxLayers];
  float lam[8] = {0};
  for (int i = 0; i < l->NL; ++i) {
    ap[i] = l->sums + l->aoff[l->blk[i].afac];
    gp[i] = l->sums + l->goff[i];
    ad[i] = l->adim[l->blk[i].afac];
    gd[i] = l->blk[i].C;
    lam[i] = cfg->damping;   // lambda / T~ with T~ = 1
  }
  const int NL = l->NL;
  std::stable_sort(l->h_jobs, l->h_jobs + 2 * NL, [](const InvJob& a, const InvJob& b) { return a.n > b.n; });
  if (e == cudaSuccess) e = cudaMemcpy(l->d_a_ptrs, ap, NL * sizeof(float*), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(l->d_g_ptrs, gp, NL * sizeof(float*), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(l->d_a_dims, ad, NL * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(l->d_g_dims, gd, NL * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(l->lambdas, lam, sizeof(lam), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(l->d_pjobs, l->h_pjobs, sizeof(l->h_pjobs), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(l->d_jobs, l->h_jobs, sizeof(l->h_jobs), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    set_error(std::string("acx_mlp_create: ") + cudaGetErrorString(e));
    delete l;
    return nullptr;
  }
  return l;
}

void acx_mlp_destroy(acx_mlp_t* l) {
  if (l)
    for (auto& kv : l->graphs)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  delete l;
}

size_t acx_mlp_num_params(const acx_mlp_t* l) { return l ? l->num_params : 0; }

int acx_mlp_set_params(acx_mlp_t* l, const float* h_params, void* stream) {
  ACX_CHECK(l && h_params, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ACX_CUDA(cudaMemcpyAsync(l->params, h_params, l->num_params * sizeof(float), cudaMemcpyHostToDevice, st));
  ACX_TRY(refresh_weight_planes(l, st));
  ACX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int acx_mlp_get_params(acx_mlp_t* l, float* h_params, void* stream) {
  ACX_CHECK(l && h_params, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ACX_CUDA(cudaMemcpyAsync(h_params, l->params, l->num_params * sizeof(float), cudaMemcpyDeviceToHost, st));
  ACX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int acx_mlp_refresh_weights(acx_mlp_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ACX_TRY(refresh_weight_planes(l, st));
  for (int i = 0; i < l->NL; ++i) {   // the bf16 planes of the stored inverses are derived state too
    const int d = l->blk[i].K + 1, c = l->blk[i].C;
    ACX_TRY(split_planes(l->inv + l->ainv_off[i], d, d, d, 1.0f, l->ainv_pl[i].p[0], l->ainv_pl[i].p[1], l->ainv_pl[i].p[2], 3,
                         l->ainv_pl[i].ld, st));
    ACX_TRY(split_planes(l->inv + l->ginv_off[i], c, c, c, 1.0f, l->ginv_pl[i].p[0], l->ginv_pl[i].p[1], l->ginv_pl[i].p[2], 3,
                         l->ginv_pl[i].ld, st));
  }
  return 0;
}

void* acx_mlp_buffer(acx_mlp_t* l, const char* name, size_t* num_bytes) {
  if (!l || !name) return nullptr;
  auto it = l->named.find(name);
  if (it == l->named.end()) {
    set_error(std::string("acx_mlp_buffer: unknown buffer '") + name + "'");
    return nullptr;
  }
  if (num_bytes) *num_bytes = it->second.bytes;
  return it->second.ptr;
}

int acx_mlp_update(acx_mlp_t* l, const int32_t* d_fisher_labels, const float* d_fisher_eps, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK((d_fisher_labels == nullptr) == (d_fisher_eps == nullptr), "inject both Fisher labels and eps, or neither");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool fisher = l->cfg.acktr != 0 && l->gs >= l->cfg.num_cold_updates;   // kfac_utils.py:42-44
  const Plan p = plan_update(l);
  const GraphKey key(p.key() | (fisher ? 32 : 0), d_fisher_labels, d_fisher_eps, nullptr, nullptr, nullptr);
  ACX_TRY(run_cached(l, key, st, [&]() {
    const int r1 = issue_update_phase1(l, d_fisher_labels, d_fisher_eps, fisher, st);
    return r1 ? r1 : issue_update_phase2(l, p, st);
  }));
  advance(l, p);
  return 0;
}

int64_t acx_mlp_global_step(const acx_mlp_t* l) { return l ? l->gs : -1; }

int acx_mlp_set_state(acx_mlp_t* l, int64_t global_step, int64_t num_cov_updates, int inverses_valid, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK(global_step >= 0 && num_cov_updates >= 0, "negative counters");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  l->gs = global_step;
  l->ncov = num_cov_updates;
  l->inverses_valid = inverses_valid != 0;
  Sched s;
  s.gs = (unsigned long long)global_step;
  s.ncov = (unsigned long long)num_cov_updates;
  s.lr = l->cfg.lr_start;
  s.debias = num_cov_updates > 0 ? (float)(1.0 / (1.0 - pow((double)l->cfg.cov_ema_decay, (double)num_cov_updates))) : 1.0f;
  ACX_CUDA(cudaMemcpyAsync(l->sched, &s, sizeof(s), cudaMemcpyHostToDevice, st));
  ACX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int acx_mlp_get_state(const acx_mlp_t* l, int64_t* global_step, int64_t* num_cov_updates, int* inverses_valid) {
  ACX_CHECK(l, "null learner");
  if (global_step) *global_step = l->gs;
  if (num_cov_updates) *num_cov_updates = l->ncov;
  if (inverses_valid) *inverses_valid = l->inverses_valid ? 1 : 0;
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
  const GraphKey key(64 | (greedy ? 1 : 0) | (rows << 7), d_obs, d_actions, d_uniform, d_logits, d_values);
  if (l->graphs.size() > 512 && l->graphs.find(key) == l->graphs.end()) return issue();   // ever-changing buffers
  return run_cached(l, key, st, issue);
}

}  // extern "C"
