// learner.cu - the ACKTR / A2C learner engine: one device arena, every matrix product on the tcgen05 GEMM
// (gemm.cu), everything else on the streaming / reduction kernels of layers.cu and kfac.cu.
//
// One update = the reference's session.run(optimize_op, feed_dict) (a2c_acktr.py:117-126):
//   phase 1  forward of the N train rows and the E bootstrap rows in one batch (envs/atari/model.py:113,116),
//            returns/advantages (objectives.py:123-130), A2C loss and output gradients (objectives.py:132-154,78),
//            backward for the true loss and - stacked as a second batch sharing weights and ReLU masks - for
//            the Fisher-sample loss (SURVEY A.5), weight gradients, and the 11 batch factor statistics.
//            Everything a data-parallel job must sum lands in one flat fp32 bucket [A | G | grads | scalars]; the input
//            factors A come first and are complete (event `a_ready`) long before the backward pass ends, so a caller may
//            all-reduce that prefix on another stream while the rest of phase 1 still runs.
//   phase 2  schedule of ColdStartPeriodicInvUpdateKfacOpt.apply_gradients as coded (kfac_utils.py:38-53):
//            cold momentum-SGD step or factor EMA, scheduled inverse refresh, precondition, KL clip, momentum,
//            apply; or the A2C RMSProp step (a2c_acktr.py:250-251).
// The host code it shares with the fully connected learner (mlp.cu) - arena, K-FAC blocks and their state, schedule, inverse
// refresh, graph cache - lives in learner_core.cuh / learner_core.cu.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "learner_core.cuh"

namespace acx {

// peer.cu: the data-parallel exchange as one kernel over NVLink peer memory
struct PeerState {
  int rank = 0, world = 0;
  uint8_t* base[8] = {};   // arena base of every rank as mapped into this process
};
int peer_allreduce(const PeerState& ps, size_t region_offset_bytes, size_t flags_offset_bytes, size_t epochs_offset_bytes,
                   long long count, long long scale_from, float scale, int channel, cudaStream_t st);
size_t peer_flag_bytes();
size_t peer_epoch_bytes();

struct Layer {       // geometry of layer l; its K-FAC block (K, C, parameter offset, T~) is acx_learner::blk[l]
  int T;            // output locations (1 for fc)
  int k, s, cin, hw_in, hw_out;
};

// Per-lane scratch: kernels of different lanes run concurrently (streams forked from the caller's stream, also inside a
// captured graph), so each lane owns its split-K workspace and reduction partials.
struct Scratch {
  float* ws = nullptr;
  size_t ws_bytes = 0;
  float* colsum_partial = nullptr;
  float* colsum_tmp = nullptr;
};
// lane 0 = the caller's stream (forward, loss, dgrad chain); 1 = input-factor SYRKs; 2 = weight gradients; 3 = output-factor
// SYRKs; 4 = the column-sum kernels (homogeneous borders, bias gradients).  With fewer configured lanes the higher ones fold
// onto the last one (3 lanes: wgrad + output factors + column sums share lane 2 - round 1's arrangement).
constexpr int kMaxLanes = 5;

}  // namespace acx

using namespace acx;

// the K-FAC blocks conv1, conv2, conv3, fc4, fc_policy, fc_baseline and their state (KfacBlocks), plus the Nature-CNN's
// activations, lanes and data-parallel exchange
struct acx_learner : KfacBlocks {
  acx_learner_config_t cfg;
  int E, T, N, R, A, c3;
  Layer L[6];
  // inputs
  uint8_t *obs, *actions, *terminals;
  float* rewards;
  // activations
  Planes P1, act1, P2, act2, P3, act3, act4;
  Planes dpre4, dpre3, dpre2, dpre1;
  float *dP, *logits, *values, *targets, *adv, *dheads;
  Planes wT[4], wN[4];
  Planes wD[4];              // gather-form dgrad operand of conv2 / conv3 (conv.cu), unused otherwise
  bool conv_tc[4];           // layer computes its input gradient with the gather-form tensor-core kernel (conv.cu)
  bool conv_fwd_tc[4];       // layer runs its forward on the implicit-GEMM kernel (conv.cu)
  PeerState peer;            // world > 1: phase 2 sums the ranks' buckets itself (peer.cu) - the caller issues no collective for them
  uint8_t* arena_base = nullptr;
  unsigned int* peer_flags = nullptr;
  unsigned int* peer_epochs = nullptr;
  cudaEvent_t reduced = nullptr;   // [G | grads | scalars] of this update are summed over the ranks (external event, split exchange)
  bool gather;               // no patch matrix is ever stored: the conv GEMMs read their patch operands in place (TMA box loads from
                             // the activations; conv1 from the row-pair interleaved bf16 copy `obs_pairs` of the observations)
  bf16* obs_pairs;           // [R, 42, 84, 2, 4] (layers.cu: obs_pairs_bf16)
  acx_gather_t gat_x[3];     // patch operand of conv layer l over the N train samples (input factor, weight gradient)
  acx_gather_t gat_g[3];     // pre-activation gradient of conv layer l as rows (sample, y, x) over the same locations
  Planes Vp, Wt;
  float* dot_partials;
  Scratch scr[kMaxLanes];
  int lanes = 1;                          // active lanes (1 = everything on the caller's stream)
  cudaStream_t side[kMaxLanes - 1] = {nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> lane_events;   // fork / join events (timing disabled), reused every update
  size_t ev_next = 0;
  bool lane_forked[kMaxLanes] = {false, false, false, false, false};
  cudaEvent_t a_ready = nullptr;     // all input-factor statistics of the current phase 1 are complete (external event)
  bool a_ready_valid = false;        // the last phase 1 recorded it
  Schedule sch;
  uint64_t act_calls;
  int lvl_fwd, lvl_bwd, lvl_fisher, lvl_factor, lvl_precon, act_planes, grad_planes;
  // optional stage timing (CUDA events on the launching stream)
  bool profiling = false;
  float policy_weight = 1.0f, value_weight = 0.0f;   // acx_learner_set_loss_weights (value_weight is set from cfg at create)
  int loss_variant = 0;                   // 0 = the configured weights; other values key separate CUDA graphs
  bool external_ema = false;              // acx_learner_set_external_ema: phase 2 leaves statistics scaling + EMA to acx_learner_ema
  cudaEvent_t ev[ACX_NUM_STAGES + 2];
  bool ev_set[ACX_NUM_STAGES + 2];
  GraphCache graphs;
};

namespace acx {

static const int kBorderChunks = 160;   // row chunks of the batch-sum pass over a conv input (4 samples per CTA at 32 x 20)

static Planes with_ld(const Planes& p, int ld) {
  Planes q = p;
  q.ld = ld;
  return q;
}

static void setup_layers(acx_learner* l) {
  const int c3 = l->c3, A = l->A;
  const int mode = l->cfg.num_locations_mode;
  static const char* names[6] = {"conv1", "conv2", "conv3", "fc4", "fc_policy", "fc_baseline"};
  const int K[6] = {256, 512, 576, 49 * c3, 512, 512}, C[6] = {32, 64, c3, 512, A, 1};
  const int Tnorm[6] = {mode ? 84 * 84 / 16 : 400, mode ? 20 * 20 / 4 : 81, mode ? 81 : 49, 1, 1, 1};
  const Layer geo[6] = {{400, 8, 4, 4, 84, 20}, {81, 4, 2, 32, 20, 9}, {49, 3, 1, 64, 9, 7}, {1}, {1}, {1}};
  for (int i = 0; i < 6; ++i) {
    Block& b = l->blk[i];
    b.name = names[i];
    b.K = K[i];
    b.C = C[i];
    b.afac = i < 5 ? i : 4;
    b.Tnorm = Tnorm[i];
    l->L[i] = geo[i];
  }
  l->set_blocks(6);
}

static ConvGeom geom_of(const acx_learner* l, int i) {
  const Layer& L = l->L[i];
  return ConvGeom{L.hw_in, L.cin, L.k, L.s, L.hw_out, l->blk[i].C};
}

// lay the arena out (base == nullptr: size pass only)
static size_t layout(acx_learner* l, uint8_t* base) {
  Arena ar;
  ar.base = base;
  const int N = l->N, R = l->R, A = l->A, c3 = l->c3;
  const size_t B2 = 2 * (size_t)N;
  l->take_state(ar);
  l->peer_flags = reinterpret_cast<unsigned int*>(ar.take(peer_flag_bytes()));
  l->peer_epochs = reinterpret_cast<unsigned int*>(ar.take(peer_epoch_bytes()));
  l->take_tables(ar);
  // ---- inputs
  l->obs = reinterpret_cast<uint8_t*>(ar.take((size_t)R * 28224));
  l->actions = reinterpret_cast<uint8_t*>(ar.take(N));
  l->terminals = reinterpret_cast<uint8_t*>(ar.take(N));
  l->rewards = ar.f32(N);
  // ---- weights as GEMM operands
  for (int i = 0; i < 4; ++i) {
    l->wT[i] = take_planes(ar, 3, l->blk[i].C, pad8(l->blk[i].K));   // W^T [C, K]   (forward: B operand, K-major)
    l->wN[i] = take_planes(ar, 3, l->blk[i].K, pad8(l->blk[i].C));   // W   [K, C]   (dgrad:   B operand, K-major)
  }
  for (int i = 1; i <= 2; ++i) {
    const Layer& L = l->L[i];
    l->conv_tc[i] = l->cfg.conv_impl == 0 && l->cfg.gemm_impl == 0 && conv_tc_supported(geom_of(l, i), 1);
    if (l->conv_tc[i]) {
      const int m = L.k / L.s;
      l->wD[i] = take_planes(ar, 3, (size_t)L.s * L.s * L.cin, pad8(m * m * l->blk[i].C));   // rows (py,px,ci), K = (i,j,co)
    }
  }
  l->conv_tc[0] = l->conv_tc[3] = false;

  // ---- activations (forward rows R = N + E; backward rows 2N = true-loss rows then Fisher-sample rows)
  const int np = l->act_planes;
  l->obs_pairs = reinterpret_cast<bf16*>(ar.take((size_t)R * 28224 * sizeof(bf16)));
  l->P1 = take_planes(ar, 1, (size_t)R * 400, 256);
  l->act1 = take_planes(ar, np, (size_t)R * 400, 32);
  l->P2 = take_planes(ar, np, (size_t)R * 81, 512);
  l->act2 = take_planes(ar, np, (size_t)R * 81, 64);
  l->P3 = take_planes(ar, np, (size_t)R * 49, 576);
  l->act3 = take_planes(ar, np, (size_t)R * 49, c3);
  l->act4 = take_planes(ar, np, (size_t)R, 512);
  l->logits = ar.f32((size_t)R * A);
  l->values = ar.f32(R);
  l->targets = ar.f32(N);
  l->adv = ar.f32(N);
  l->dheads = ar.f32(B2 * (A + 1));
  const int ng = l->grad_planes;
  l->dpre4 = take_planes(ar, ng, B2, 512);
  l->dpre3 = take_planes(ar, ng, B2 * 49, c3);
  l->dpre2 = take_planes(ar, ng, B2 * 81, 64);
  l->dpre1 = take_planes(ar, ng, B2 * 400, 32);
  l->dP = ar.f32(std::max(B2 * 49 * 576, B2 * 81 * 512) + 81 * 512);   // patch gradients of the conv3 / conv2 input gradient
  // ---- preconditioning scratch
  int dmax = 0, cmax = 0;
  for (int i = 0; i < 6; ++i) {
    dmax = std::max(dmax, l->blk[i].K + 1);
    cmax = std::max(cmax, l->blk[i].C);
  }
  l->Vp = take_planes(ar, 3, dmax, pad8(cmax));
  l->Wt = take_planes(ar, 3, cmax, pad8(dmax));
  l->dot_partials = ar.f32(kDotPartials);
  const size_t kpad = align_up((size_t)49 * c3, 128);
  for (int i = 0; i < kMaxLanes; ++i) {
    Scratch& sc = l->scr[i];
    sc.colsum_partial = ar.f32(std::max((size_t)kColsumChunks * (size_t)std::max(49 * c3, 576), (size_t)kBorderChunks * 28224));
    sc.colsum_tmp = ar.f32(4096 + 28224 + 8);   // [0,4096): border / column-sum vectors, then the batch-summed conv input
    sc.ws_bytes = std::max<size_t>((size_t)48 << 20, kpad * kpad * sizeof(float) + (1 << 20));
    sc.ws = reinterpret_cast<float*>(ar.take(sc.ws_bytes));
  }
  return align_up(ar.used, 256);
}

// The patch operands of the three conv layers as in-place views (acx_gather_t, include/acx.h): chunk q of location
// (sample, y, x) = 64 contiguous bf16 of the layer's input tensor.
//   conv1  8x8/4 on the row-pair copy [n][42][84][2][4]: chunk j = kernel rows 2j, 2j+1 -> pair-row 2 oy + j, pixel 4 ox
//   conv2  4x4/2 on act1 [n][20][20][32]: chunk (kh, h) = kernel row kh, kernel columns 2h, 2h+1 -> row 2 oy + kh, pixel 2 (ox + h)
//   conv3  3x3/1 on act2 [n][9][9][64]:   chunk (kh, kw) -> pixel (oy + kh, ox + kw)
// and the pre-activation gradients [sample][y][x][C] as operands over the same locations.
static void setup_gather(acx_learner* l) {
  const int N = l->N;
  auto fill = [](acx_gather_t& g, const Planes& pl, int nplanes) {
    memset(&g, 0, sizeof(g));
    for (int i = 0; i < nplanes; ++i) g.planes[i] = pl.p[i];
    g.num_planes = nplanes;
  };
  {
    acx_gather_t& g = l->gat_x[0];
    Planes one;
    one.p[0] = l->obs_pairs;
    fill(g, one, 1);
    const long long prow = 84 * 8 * 2;   // bytes of one pair-row
    const long long dim[5] = {64, 20, 4, 20, N}, st[4] = {64, prow, 2 * prow, 42 * prow};
    for (int i = 0; i < 5; ++i) g.dim[i] = dim[i];
    for (int i = 0; i < 4; ++i) g.stride_bytes[i] = st[i];
    g.gx = g.gy = 20;
    g.samples = N;
    g.num_chunks = 4;
    for (int j = 0; j < 4; ++j) g.c2[j] = (signed char)j;
  }
  {
    acx_gather_t& g = l->gat_x[1];
    fill(g, l->act1, l->act1.n);
    const long long px = 32 * 2;
    const long long dim[5] = {64, 10, 4, 9, N}, st[4] = {2 * px, 20 * px, 40 * px, 400 * px};
    for (int i = 0; i < 5; ++i) g.dim[i] = dim[i];
    for (int i = 0; i < 4; ++i) g.stride_bytes[i] = st[i];
    g.gx = g.gy = 9;
    g.samples = N;
    g.num_chunks = 8;
    for (int kh = 0; kh < 4; ++kh)
      for (int h = 0; h < 2; ++h) {
        g.c1[kh * 2 + h] = (signed char)h;
        g.c2[kh * 2 + h] = (signed char)kh;
      }
  }
  {
    acx_gather_t& g = l->gat_x[2];
    fill(g, l->act2, l->act2.n);
    const long long px = 64 * 2;
    const long long dim[5] = {64, 9, 1, 9, N}, st[4] = {px, px, 9 * px, 81 * px};
    for (int i = 0; i < 5; ++i) g.dim[i] = dim[i];
    for (int i = 0; i < 4; ++i) g.stride_bytes[i] = st[i];
    g.gx = g.gy = 7;
    g.samples = N;
    g.num_chunks = 9;
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) {
        g.c1[kh * 3 + kw] = (signed char)kw;
        g.c3[kh * 3 + kw] = (signed char)kh;
      }
  }
  const Planes* dp[3] = {&l->dpre1, &l->dpre2, &l->dpre3};
  for (int li = 0; li < 3; ++li) {
    acx_gather_t& g = l->gat_g[li];
    const Layer& L = l->L[li];
    const int C = l->blk[li].C;
    fill(g, *dp[li], dp[li]->n);
    const long long px = (long long)C * 2;
    const long long dim[5] = {C, L.hw_out, 1, L.hw_out, N}, st[4] = {px, px, L.hw_out * px, (long long)L.hw_out * L.hw_out * px};
    for (int i = 0; i < 5; ++i) g.dim[i] = dim[i];
    for (int i = 0; i < 4; ++i) g.stride_bytes[i] = st[i];
    g.gx = g.gy = L.hw_out;
    g.samples = N;
    g.num_chunks = (C + 63) / 64;
    for (int j = 0; j < g.num_chunks; ++j) g.c0[j] = (signed char)(64 * j);
  }
}

static void register_buffers(acx_learner* l) {
  l->register_buffers();
  l->reg("input_factor_stats", l->stats, l->goff[0] * 4);   // the A part = the prefix of the reduce bucket
  l->reg("observations", l->obs, (size_t)l->R * 28224);
  l->reg("actions", l->actions, l->N);
  l->reg("terminals", l->terminals, l->N);
  l->reg("rewards", l->rewards, (size_t)l->N * 4);
  l->reg("logits", l->logits, (size_t)l->R * l->A * 4);
  l->reg("values", l->values, (size_t)l->R * 4);
  l->reg("targets", l->targets, (size_t)l->N * 4);
  l->reg("advantages", l->adv, (size_t)l->N * 4);
  l->reg("patches/conv1", l->P1.p[0], (size_t)l->R * 400 * 256 * 2);   // bf16 [R*400, 256], raw byte values (conv_impl / gemm_impl = 1 only)
  l->reg("obs_pairs", l->obs_pairs, (size_t)l->R * 28224 * 2);         // bf16 [R, 42, 84, 2, 4]: the row-pair copy of the observations
  // hi planes of the forward activations = the ReLU masks the backward pass applies (act > 0); exposed so that the parity
  // tests can tell arithmetic error from units whose pre-activation is within rounding of zero
  l->reg("act_hi/conv1", l->act1.p[0], (size_t)l->R * 400 * 32 * 2);
  l->reg("act_hi/conv2", l->act2.p[0], (size_t)l->R * 81 * 64 * 2);
  l->reg("act_hi/conv3", l->act3.p[0], (size_t)l->R * 49 * l->c3 * 2);
  l->reg("act_hi/fc4", l->act4.p[0], (size_t)l->R * 512 * 2);
  l->reg("dheads", l->dheads, (size_t)2 * l->N * (l->A + 1) * 4);
}

// ------------------------------------------------------------------------------------------------
// lanes: a lane = a stream + its scratch.  Lane 0 is the caller's stream; side lanes are forked from it with events and
// joined back before a phase returns, so the caller still sees one stream (and a stream capture records the fork /
// join structure as parallel graph branches).
// ------------------------------------------------------------------------------------------------
struct Lane {
  cudaStream_t st;
  const Scratch* sc;
  int index;
};

static Lane lane_of(acx_learner* l, int i, cudaStream_t main_st) {
  if (l->profiling) i = 0;                    // stage timing brackets serial work on the caller's stream
  if (i >= l->lanes) i = l->lanes - 1;        // fewer lanes configured: the higher ones fold onto the last one
  return Lane{i == 0 ? main_st : l->side[i - 1], &l->scr[i], i};
}

// an event from the per-update pool, recorded at the current tail of `from`
static int record_tail(acx_learner* l, cudaStream_t from, cudaEvent_t* out) {
  if (l->ev_next == l->lane_events.size()) {
    cudaEvent_t e;
    ACX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    l->lane_events.push_back(e);
  }
  cudaEvent_t e = l->lane_events[l->ev_next++];
  ACX_CUDA(cudaEventRecord(e, from));
  *out = e;
  return 0;
}
// everything enqueued on `from` so far happens before whatever is enqueued on `to` from now on
static int order_after(acx_learner* l, cudaStream_t from, cudaStream_t to) {
  if (from == to) return 0;
  cudaEvent_t e;
  int r = record_tail(l, from, &e);
  if (r) return r;
  ACX_CUDA(cudaStreamWaitEvent(to, e, 0));
  return 0;
}
// fork: `ln` continues after everything issued on `main_st` so far; join: `main_st` waits for the lane (a lane that was
// never forked in this phase has nothing to wait for - and inside a stream capture it is not part of the graph)
static int fork_lane(acx_learner* l, cudaStream_t main_st, const Lane& ln) {
  if (ln.index == 0) return 0;
  l->lane_forked[ln.index] = true;
  return order_after(l, main_st, ln.st);
}
static int join_lane(acx_learner* l, const Lane& ln, cudaStream_t main_st) {
  if (ln.index == 0 || !l->lane_forked[ln.index]) return 0;
  l->lane_forked[ln.index] = false;
  return order_after(l, ln.st, main_st);
}

// cap on the persistent grids of the tensor-core kernels of a lane (0 = all SMs)
static int lane_cta_cap(const acx_learner* l, int lane_index) {
  if (lane_index != 0) return 0;
  // K-FAC learners: the persistent grids of the caller's lane (forward, input gradients, conv1 weight gradient,
  // preconditioning) leave 16 SMs to the factor / weight-gradient lanes, so that their kernels start beside the critical chain
  // instead of queueing behind it: 0.674 -> 0.656 ms/update at 32 x 20 (measured 96 / 112 / 120 / 132 / 140 CTAs: 0.671 / 0.660 /
  // 0.656 / 0.656 / 0.657; capping the side lanes instead is slower).  Learners without K-FAC side work keep every SM.
  return (l->cfg.acktr && l->lanes > 1 && !l->profiling) ? 132 : 0;
}

static int run_gemm(acx_learner* l, const Planes& a, const Planes& b, int trans, int m, int n, int k, int level, float alpha,
                    int symmetric, const GemmOut& o, const Lane& ln) {
  acx_gemm_t g;
  fill_gemm(&g, a, b, trans, m, n, k, level, alpha, symmetric, o, ln.sc->ws, ln.sc->ws_bytes);
  set_cta_cap(lane_cta_cap(l, ln.index));
  const int r = gemm_dispatch(&g, l->cfg.gemm_impl, ln.st);
  set_cta_cap(0);
  return r;
}

// stage boundaries: mark k closes stage k-1 (phase 1: marks 0..4, phase 2: marks 5..9)
static void mark(acx_learner* l, int k, cudaStream_t st) {
  if (!l->profiling) return;
  cudaEventRecord(l->ev[k], st);
  l->ev_set[k] = true;
}

static int refresh_weight_planes(acx_learner* l, cudaStream_t st, bool on_lanes = false) {
  const float* w[4];
  int kr[4], cc[4], ldt[4], ldn[4];
  bf16* t[4][3];
  bf16* n[4][3];
  for (int i = 0; i < 4; ++i) {
    const Block& L = l->blk[i];
    w[i] = l->params + L.off;
    kr[i] = L.K;
    cc[i] = L.C;
    ldt[i] = l->wT[i].ld;
    ldn[i] = l->wN[i].ld;
    for (int q = 0; q < 3; ++q) {
      t[i][q] = l->wT[i].p[q];
      n[i][q] = i > 0 ? l->wN[i].p[q] : nullptr;   // conv1 has no input gradient
    }
  }
  // the three launches read the parameters and write disjoint planes: at the end of phase 2 (the tail of the update's critical
  // path) the two input-gradient operands go to side lanes next to the main one
  const Lane side[2] = {lane_of(l, 1, st), lane_of(l, 3, st)};
  const bool fork = on_lanes && l->lanes > 1 && !l->profiling && st != nullptr;
  for (int i = 1; i <= 2; ++i)
    if (l->conv_tc[i]) {
      const float* w = l->params + l->blk[i].off;
      const Lane& ln = side[i - 1];
      if (fork && ln.index != 0) {
        ACX_TRY(fork_lane(l, st, ln));
        ACX_TRY(conv_dgrad_weight_planes(w, geom_of(l, i), l->wD[i], ln.st));
      } else {
        ACX_TRY(conv_dgrad_weight_planes(w, geom_of(l, i), l->wD[i], st));
      }
    }
  ACX_TRY(weight_planes(w, kr, cc, t, ldt, n, ldn, 4, st, l->gather ? 1 : 0));   // gather: conv1's W^T columns in the row-pair copy's order
  if (fork)
    for (int i = 0; i < 2; ++i) ACX_TRY(join_lane(l, side[i], st));
  return 0;
}

// input factor of layer `li` from the patch/input planes `x` (first `rows` rows, K columns): SYRK on lane `ln`, homogeneous
// border (column sums) on lane `lb`
static int input_factor(acx_learner* l, int fac, const Planes& x, int rows, int K, float scale_sq, float scale_lin,
                        const Lane& ln, const Lane& lb) {
  const int d = K + 1;
  float* dst = l->stats + l->aoff[fac];
  GemmOut o;
  o.c = dst;
  o.ldc = d;
  ACX_TRY(run_gemm(l, x, x, 1, K, K, rows, l->lvl_factor, scale_sq, 1, o, ln));
  // homogeneous border straight from the column sums: column d-1 (stride d), row d-1 (stride 1), corner 1
  ACX_TRY(colsum(x, rows, K, scale_lin, lb.sc->colsum_partial, kColsumChunks, dst + (d - 1), d, lb.st, dst + (size_t)(d - 1) * d, 1,
                 dst + (size_t)d * d - 1));
  return 0;
}

// input factor of a conv layer: SYRK over the patch matrix; the homogeneous border P^T 1 / rows comes from the batch-summed
// layer input through window sums (one pass over the un-im2col'd input instead of a pass over the k^2/s^2 times larger P)
static int conv_input_factor(acx_learner* l, int li, const Planes& patches, const uint8_t* obs_u8, const Planes* act_in,
                             float scale_sq, float border_scale, const Lane& ln, const Lane& lb) {
  const Layer& L = l->L[li];
  const Block& B = l->blk[li];
  const int d = B.K + 1, rows = l->N * L.T;
  float* dst = l->stats + l->aoff[li];
  GemmOut o;
  o.c = dst;
  o.ldc = d;
  if (l->gather) {                   // P^T P read in place from the layer's input (conv1: columns in the row-pair copy's order)
    o.a_gather = &l->gat_x[li];
    o.perm_m = o.perm_n = li == 0 ? 1 : 0;
    Planes x;   // only the plane count matters
    x.n = l->gat_x[li].num_planes;
    x.ld = 8;
    for (int i = 0; i < x.n; ++i) x.p[i] = reinterpret_cast<bf16*>(const_cast<void*>(l->gat_x[li].planes[i]));
    ACX_TRY(run_gemm(l, x, x, 1, B.K, B.K, rows, l->lvl_factor, scale_sq, 1, o, ln));
  } else {
    ACX_TRY(run_gemm(l, patches, patches, 1, B.K, B.K, rows, l->lvl_factor, scale_sq, 1, o, ln));
  }
  ACX_TRY(conv_border(obs_u8, act_in, l->N, L.hw_in, L.cin, L.k, L.s, L.hw_out, border_scale, lb.sc->colsum_partial, kBorderChunks,
                      lb.sc->colsum_tmp + 4096, dst, d, lb.st));
  return 0;
}

// the five input factors (SURVEY A.5), each as soon as its operand exists: `stage` = 0 P1, 1 P2, 2 P3, 3 act3, 4 act4.
// The SYRK writes the K x K block of the factor, the border kernels its last row / column / corner: disjoint elements,
// so the two may run on different lanes.
static int input_factor_stage(acx_learner* l, int stage, const Lane& ln, const Lane& lb) {
  const int N = l->N, c3 = l->c3;
  const float r1 = 1.0f / (float)(N * 400), r2 = 1.0f / (float)(N * 81), r3 = 1.0f / (float)(N * 49), r4 = 1.0f / (float)N;
  switch (stage) {
    case 0: return conv_input_factor(l, 0, l->P1, l->obs, nullptr, r1 / (255.0f * 255.0f), r1 / 255.0f, ln, lb);
    case 1: return conv_input_factor(l, 1, l->P2, nullptr, &l->act1, r2, r2, ln, lb);
    case 2: return conv_input_factor(l, 2, l->P3, nullptr, &l->act2, r3, r3, ln, lb);
    case 3: return input_factor(l, 3, with_ld(l->act3, 49 * c3), N, 49 * c3, r4, r4, ln, lb);
    default: return input_factor(l, 4, l->act4, N, 512, r4, r4, ln, lb);
  }
}

// Nature-CNN forward on `rows` observations (envs/atari/model.py:173-217).  conv1 and fc4: im2col / flatten + GEMM with
// bias/ReLU epilogues (conv1 with `gather`: implicit GEMM on the row-pair copy of the observations).  conv2 / conv3
// (`conv_fwd_tc`): implicit-GEMM kernel straight from the activation planes (conv.cu); their input factors and weight
// gradients read the same activations in place, so no patch matrix is built.  Otherwise im2col + GEMM on the caller's stream.
// With `factors` every input factor is issued on the aux lane the moment its operand is complete, so the factor SYRKs
// overlap the rest of the forward and the whole backward.
static int forward(acx_learner* l, const uint8_t* obs, int rows, const Lane& ln, const Lane* aux, const Lane* aux2, bool factors) {
  const int c3 = l->c3;
  cudaStream_t st = ln.st;
  auto factor = [&](int stage) -> int {   // SYRK on aux, its border on aux2 (idle until the backward pass starts)
    if (!aux || !factors) return 0;
    ACX_TRY(fork_lane(l, st, *aux));
    ACX_TRY(fork_lane(l, st, *aux2));
    return input_factor_stage(l, stage, *aux, *aux2);
  };
  auto conv_layer = [&](int li, const Planes& in, const Planes& patches, const Planes& out) -> int {
    const Layer& L = l->L[li];
    const Block& B = l->blk[li];
    GemmOut o;
    o.relu = 1;
    o.bias = l->params + B.off + (size_t)B.K * B.C;
    o.planes = &out;
    if (!l->conv_fwd_tc[li]) {
      ACX_TRY(im2col_bf16(in, patches, rows * L.T, L.hw_in, L.cin, L.k, L.s, L.hw_out, st));
      ACX_TRY(factor(li));
      return run_gemm(l, patches, l->wT[li], 0, rows * L.T, B.C, B.K, l->lvl_fwd, 1.0f, 0, o, ln);
    }
    ACX_TRY(factor(li));   // the input factor reads the layer's input in place: nothing to build
    int pa[6], pb[6];
    const int np = level_pairs(l->lvl_fwd, in.n, l->wT[li].n, pa, pb);
    set_cta_cap(lane_cta_cap(l, 0));
    const int rc = conv_tc_forward(in, l->wT[li], geom_of(l, li), rows, o.bias, 1, out, np, pa, pb, st);
    set_cta_cap(0);
    return rc;
  };
  GemmOut o;
  o.relu = 1;
  // conv1: raw bytes are exact in bf16; the /255 of envs/atari/model.py:93 is the GEMM alpha
  o.bias = l->params + l->blk[0].off + (size_t)l->blk[0].K * l->blk[0].C;
  o.planes = &l->act1;
  if (l->gather) {
    // the row-pair interleaved bf16 copy of the observations replaces P1 (2x instead of 7.2x the observations, L2 resident);
    // conv1 forward is an implicit GEMM on it (conv.cu), its input factor and weight gradient read it in place
    ACX_TRY(obs_pairs_bf16(obs, l->obs_pairs, rows, st));
    ACX_TRY(factor(0));
    int pa[6], pb[6];
    const int np = level_pairs(l->lvl_fwd, 1, l->wT[0].n, pa, pb);
    set_cta_cap(lane_cta_cap(l, 0));
    const int rc = conv1_pairs_forward(l->obs_pairs, l->wT[0], rows, o.bias, 1.0f / 255.0f, l->act1, np, pa, pb, st);
    set_cta_cap(0);
    ACX_TRY(rc);
  } else {
    ACX_TRY(im2col_conv1(obs, l->P1.p[0], rows * 400, st));
    ACX_TRY(factor(0));
    ACX_TRY(run_gemm(l, l->P1, l->wT[0], 0, rows * 400, 32, 256, l->lvl_fwd, 1.0f / 255.0f, 0, o, ln));
  }
  ACX_TRY(conv_layer(1, l->act1, l->P2, l->act2));
  ACX_TRY(conv_layer(2, l->act2, l->P3, l->act3));
  ACX_TRY(factor(3));
  // fc4 on the (h, w, c)-flattened conv3 output (nn.py:125-126)
  o.bias = l->params + l->blk[3].off + (size_t)l->blk[3].K * l->blk[3].C;
  o.planes = &l->act4;
  ACX_TRY(run_gemm(l, with_ld(l->act3, 49 * c3), l->wT[3], 0, rows, 512, 49 * c3, l->lvl_fwd, 1.0f, 0, o, ln));
  ACX_TRY(factor(4));
  ACX_TRY(heads_fwd(l->act4, l->params + l->blk[4].off, l->params + l->blk[5].off, rows, l->A, l->logits, l->values, st));
  return 0;
}

// weight gradient V_l[:K] = X^T g over the true-loss rows, bias row = column sums of g
static int bias_grad(acx_learner* l, int li, const Planes& g, int rows, const Lane& ln) {
  const Block& L = l->blk[li];
  return colsum(g, rows, L.C, 1.0f, ln.sc->colsum_partial, kColsumChunks, l->grads + L.off + (size_t)L.K * L.C, 1, ln.st);
}
static int weight_grad(acx_learner* l, int li, const Planes& x, const Planes& g, int rows, float alpha, const Lane& ln,
                       bool with_bias = true) {
  const Block& L = l->blk[li];
  GemmOut o;
  o.c = l->grads + L.off;
  o.ldc = L.C;
  if (li < 3 && l->gather) {   // X^T g with both operands read in place over the same locations
    o.a_gather = &l->gat_x[li];
    o.b_gather = &l->gat_g[li];
    o.perm_m = li == 0 ? 1 : 0;
    Planes xa;   // only the plane counts matter
    xa.n = l->gat_x[li].num_planes;
    xa.ld = 8;
    for (int i = 0; i < xa.n; ++i) xa.p[i] = reinterpret_cast<bf16*>(const_cast<void*>(l->gat_x[li].planes[i]));
    ACX_TRY(run_gemm(l, xa, g, 1, L.K, L.C, rows, l->lvl_bwd, alpha, 0, o, ln));
    if (with_bias) ACX_TRY(bias_grad(l, li, g, rows, ln));
    return 0;
  }
  ACX_TRY(run_gemm(l, x, g, 1, L.K, L.C, rows, l->lvl_bwd, alpha, 0, o, ln));
  if (with_bias) ACX_TRY(bias_grad(l, li, g, rows, ln));
  return 0;
}

// input gradient of conv layer li: dP = g W^T (fp32) then col2im + ReLU mask of the layer below + bf16 split, over the whole
// batch at once.  Chunks of samples small enough to keep dP in L2 measured slower on B200 at 32x20 (whole 1.510 ms/update,
// 128 MB 1.533, 64 MB 1.551, 32 MB 1.599, 16 MB 1.681): the extra launches and wave tails cost more than the HBM round trip.
static int conv_dgrad(acx_learner* l, int li, const Planes& g, const bf16* act_below_hi, const Planes& g_below, int samples,
                      const Lane& ln) {
  const Layer& L = l->L[li];
  const Block& B = l->blk[li];
  if (l->conv_tc[li]) {   // gather form on the tensor cores: no dP matrix, no col2im pass (conv.cu)
    int pa[6], pb[6];
    const int np = level_pairs(l->lvl_bwd, g.n, l->wD[li].n, pa, pb);
    // samples beyond N are the Fisher-sample rows of the stacked backward batch: they only feed the output factors
    // G_l (accumulated at lvl_factor), so their input gradients are taken at lvl_fisher (level_pairs orders the pairs
    // by level: a lower level is a prefix)
    int pa2[6], pb2[6];
    const int np_lo = level_pairs(l->lvl_fisher, g.n, l->wD[li].n, pa2, pb2);
    const bool lo = samples > l->N && np_lo < np;
    set_cta_cap(lane_cta_cap(l, ln.index));
    const int rc = conv_tc_dgrad(g, l->wD[li], geom_of(l, li), samples, act_below_hi, l->N, g_below, np, pa, pb, ln.st, lo ? l->N : -1,
                                 np_lo);
    set_cta_cap(0);
    return rc;
  }
  GemmOut o;
  o.c = l->dP;
  o.ldc = B.K;
  ACX_TRY(run_gemm(l, g, l->wN[li], 0, samples * L.T, B.K, B.C, l->lvl_bwd, 1.0f, 0, o, ln));
  return col2im_mask_split(l->dP, act_below_hi, g_below, 0, samples, l->N, L.hw_in, L.cin, L.k, L.s, L.hw_out, ln.st);
}

// output factor G_l = g^T g / rows over the Fisher-sample rows
static int output_factor(acx_learner* l, int li, const Planes& g_fisher, int rows, const Lane& ln) {
  const Block& L = l->blk[li];
  // Narrow output factors (C = 32 / 64 fill a 128 x 64 MMA tile to 1/8 .. 1/2) still run faster as a split-K SYRK on the
  // tensor cores than on an fp32 SIMT Gram kernel (measured: 1.067 -> 1.043 ms/update; the MMAs are nearly free next to
  // the one pass over g).
  GemmOut o;
  o.c = l->stats + l->goff[li];
  o.ldc = L.C;
  return run_gemm(l, g_fisher, g_fisher, 1, L.C, L.C, rows, l->lvl_factor, 1.0f / (float)rows, 1, o, ln);
}

// Phase 1 as three lanes (each a chain; arrows = events):
//   lane 0  forward -> returns, loss, heads backward -> fc4 dgrad -> conv3 dgrad -> conv2 dgrad -> conv1 wgrad
//   lane 1  input factors A_l, each forked from the forward as soon as its operand exists
//   lane 2  wgrad + output factor G_l of a layer, forked as soon as that layer's pre-activation gradient exists
// With one lane (profiling, ACX lanes = 1) the same calls run back to back on the caller's stream.
static int issue_phase1(acx_learner* l, const int32_t* fisher_labels, const float* fisher_eps, cudaStream_t st) {
  const int N = l->N, E = l->E, T = l->T, A = l->A, c3 = l->c3;
  const bool fisher = l->sch.fisher();
  const int RB = fisher ? 2 * N : N;
  l->ev_next = 0;
  const Lane main_ln = lane_of(l, 0, st), fac_ln = lane_of(l, 1, st), wg_ln = lane_of(l, 2, st), gf_ln = lane_of(l, 3, st),
             cs_ln = lane_of(l, 4, st);
  mark(l, 0, st);
  ACX_TRY(forward(l, l->obs, l->R, main_ln, &fac_ln, &cs_ln, fisher));
  if (fisher && fac_ln.index != 0) {
    // every input factor has been issued: SYRKs on the factor lane, borders on the column-sum lane.
    // Raise `a_ready` behind both; inside a stream capture it becomes an external event-record node of the graph.
    ACX_TRY(order_after(l, cs_ln.st, fac_ln.st));
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    ACX_CUDA(cudaStreamIsCapturing(fac_ln.st, &cs));
    ACX_CUDA(cudaEventRecordWithFlags(l->a_ready, fac_ln.st,
                                      cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault));
  }
  mark(l, 1, st);
  // targets use the bootstrap tower's values = rows [N, N+E) (envs/atari/model.py:116,126-127)
  // (K-RET runs inside the loss kernel: one launch)
  ACX_TRY(returns_loss_grad(l->rewards, l->terminals, l->values + N, l->cfg.gamma, E, T, l->targets, l->adv, l->logits, l->values,
                            l->actions, fisher_labels, fisher_eps, l->cfg.seed, l->sched, A, l->cfg.entropy_beta, l->value_weight,
                            l->dheads, l->bscalars, fisher ? 1 : 0, st, l->policy_weight));
  ACX_TRY(heads_bwd(l->dheads, l->params + l->blk[4].off, l->params + l->blk[5].off, l->act4, N, RB, A, l->dpre4,
                    l->grads + l->blk[4].off, l->grads + l->blk[5].off, st));
  const Planes flat3 = with_ld(l->act3, 49 * c3);
  mark(l, 2, st);
  // ---- fc4
  // (each pre-activation gradient fans out to three side lanes: weight gradient | output factor | bias column sum)
  auto fan_out = [&](int li, const Planes& x, const Planes& g, int rows) -> int {
    ACX_TRY(fork_lane(l, st, wg_ln));
    ACX_TRY(fork_lane(l, st, gf_ln));
    ACX_TRY(fork_lane(l, st, cs_ln));
    const bool split_bias = cs_ln.st != wg_ln.st;
    ACX_TRY(weight_grad(l, li, x, g, rows, 1.0f, wg_ln, !split_bias));
    if (split_bias) ACX_TRY(bias_grad(l, li, g, rows, cs_ln));
    if (fisher) ACX_TRY(output_factor(l, li, offset_rows(g, (size_t)rows), rows, gf_ln));
    return 0;
  };
  ACX_TRY(fork_lane(l, st, gf_ln));
  if (fisher)
    ACX_TRY(heads_gfactor(l->dheads + (size_t)N * (A + 1), N, A, l->stats + l->goff[4], l->stats + l->goff[5], gf_ln.st));
  ACX_TRY(fan_out(3, flat3, l->dpre4, N));
  {
    GemmOut o;   // d(act3) = dpre4 W4^T, masked by ReLU(conv3) -> dpre3  (rows of the Fisher half reuse the mask)
    const Planes out = with_ld(l->dpre3, 49 * c3);
    o.planes = &out;
    o.mask = l->act3.p[0];
    o.mask_ld = 49 * c3;
    o.mask_rows = N;
    ACX_TRY(run_gemm(l, l->dpre4, l->wN[3], 0, RB, 49 * c3, 512, l->lvl_bwd, 1.0f, 0, o, main_ln));
  }
  // ---- conv3
  ACX_TRY(fan_out(2, l->P3, l->dpre3, N * 49));
  ACX_TRY(conv_dgrad(l, 2, l->dpre3, l->act2.p[0], l->dpre2, RB, main_ln));
  // ---- conv2
  ACX_TRY(fan_out(1, l->P2, l->dpre2, N * 81));
  ACX_TRY(conv_dgrad(l, 1, l->dpre2, l->act1.p[0], l->dpre1, RB, main_ln));
  // ---- conv1 (no input gradient: observations are constants, envs/atari/model.py:101-104)
  if (fisher) {
    ACX_TRY(fork_lane(l, st, gf_ln));
    ACX_TRY(output_factor(l, 0, offset_rows(l->dpre1, (size_t)N * 400), N * 400, gf_ln));
  }
  // last link of the chain: the weight GEMM stays on the caller's stream, its bias row goes to the column-sum lane
  ACX_TRY(fork_lane(l, st, cs_ln));
  ACX_TRY(bias_grad(l, 0, l->dpre1, N * 400, cs_ln));
  ACX_TRY(weight_grad(l, 0, l->P1, l->dpre1, N * 400, 1.0f / 255.0f, main_ln, false));
  mark(l, 3, st);
  // ---- join: the caller's stream now also covers the 11 batch factor statistics and every weight gradient
  ACX_TRY(join_lane(l, fac_ln, st));
  ACX_TRY(join_lane(l, wg_ln, st));
  ACX_TRY(join_lane(l, gf_ln, st));
  ACX_TRY(join_lane(l, cs_ln, st));
  mark(l, 4, st);
  return 0;
}

static int precondition(acx_learner* l, cudaStream_t st) {
  // blocks with <= 64 output channels: batched fp32 SIMT kernels on a side lane, next to fc4's two GEMMs
  const Lane main_ln = lane_of(l, 0, st), small_ln = lane_of(l, 1, st);
  ACX_TRY(fork_lane(l, st, small_ln));
  ACX_TRY(precondition_small(l->d_pjobs, l->num_pjobs, l->pjobs_max_d, small_ln.st));
  for (int i = 0; i < 6; ++i) {
    const Block& L = l->blk[i];
    const int d = L.K + 1, C = L.C;
    if (C <= 64) continue;   // done above
    Planes vp = l->Vp;
    vp.ld = pad8(C);
    Planes wt = l->Wt;
    wt.ld = pad8(d);
    ACX_TRY(split_planes(l->grads + L.off, C, d, C, 1.0f, vp.p[0], vp.p[1], vp.p[2], 3, vp.ld, st));
    GemmOut o1;   // Wt [C, d] = G^-1 V^T
    o1.planes = &wt;
    ACX_TRY(run_gemm(l, l->ginv_pl[i], vp, 0, C, d, C, l->lvl_precon, 1.0f, 0, o1, main_ln));
    GemmOut o2;   // U [d, C] = A^-1 W / T~
    o2.c = l->precon + L.off;
    o2.ldc = C;
    ACX_TRY(run_gemm(l, l->ainv_pl[i], wt, 0, d, C, d, l->lvl_precon, 1.0f / (float)L.Tnorm, 0, o2, main_ln));
  }
  ACX_TRY(join_lane(l, small_ln, st));
  return 0;
}

// SURVEY A.7-U3: the 1 / (1 - decay^n) factor belongs to zero-initialised running sums
static bool zero_debias_on(const acx_learner_config_t& c) { return !c.no_zero_debias && !c.cov_init_identity; }

static int issue_phase2(acx_learner* l, const Plan& p, cudaStream_t st) {
  const acx_learner_config_t& c = l->cfg;
  const size_t P = l->num_params;
  l->ev_next = 0;
  Lane ema_ln = lane_of(l, 0, st);
  mark(l, 5, st);
  const bool ext_ema = l->external_ema && !p.a2c && !p.cold;   // the caller runs acx_learner_ema on its own stream
  if (c.world_size > 1 && l->peer.world > 1) {
    // the exchange itself, over NVLink peer memory, fused with the 1 / world_size scaling (peer.cu): with an external EMA only
    // what this phase reads travels here - [G | grads | scalars], G left unscaled for acx_learner_ema - and `reduced` tells
    // the caller's EMA stream when it is complete; otherwise the whole bucket
    const size_t flags_off = reinterpret_cast<uint8_t*>(l->peer_flags) - l->arena_base;
    const size_t epochs_off = reinterpret_cast<uint8_t*>(l->peer_epochs) - l->arena_base;
    const float inv_world = 1.0f / (float)c.world_size;
    if (ext_ema) {
      float* region = l->bucket + l->goff[0];
      ACX_TRY(peer_allreduce(l->peer, reinterpret_cast<uint8_t*>(region) - l->arena_base, flags_off, epochs_off,
                             (long long)(l->bucket_floats - l->goff[0]), (long long)(l->factor_floats - l->goff[0]), inv_world, 0, st));
      cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
      ACX_CUDA(cudaStreamIsCapturing(st, &cs));
      ACX_CUDA(cudaEventRecordWithFlags(l->reduced, st, cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault));
    } else {
      ACX_TRY(peer_allreduce(l->peer, reinterpret_cast<uint8_t*>(l->bucket) - l->arena_base, flags_off, epochs_off,
                             (long long)l->bucket_floats, 0, inv_world, 0, st));
    }
  } else if (c.world_size > 1) {
    if (ext_ema)   // only what this phase reads: [grads | scalars]; the statistics are scaled by acx_learner_ema
      ACX_TRY(scale_f32(l->grads, l->bucket_floats - l->factor_floats, 1.0f / (float)c.world_size, st));
    else
      ACX_TRY(scale_f32(l->bucket, l->bucket_floats, 1.0f / (float)c.world_size, st));
  }
  // K-FAC updates: the loss scalars' copy and the schedule transition are needed only by the inverse refresh (debias factor) and
  // by the parameter step (learning rate) - they run on a side lane next to the preconditioning instead of ahead of it
  Lane sched_ln = lane_of(l, (p.a2c || p.cold) ? 0 : 3, st);
  ACX_TRY(fork_lane(l, st, sched_ln));
  ACX_CUDA(cudaMemcpyAsync(l->scalars, l->bscalars, 4 * sizeof(float), cudaMemcpyDeviceToDevice, sched_ln.st));
  // one launch for the whole schedule transition (kfac_utils.py:38-53): lr from the step the update starts with, then
  // global_step += (cold ? 2 : 1) [A2C: 1], covariance counter += (cold ? 0 : 1)
  ACX_TRY(sched_step(l->sched, c.lr_start, c.lr_end, c.lr_decay_steps, l->scalars + 7, p.a2c ? 1 : (p.cold ? 2 : 1),
                     (p.a2c || p.cold) ? 0 : 1, c.cov_ema_decay, zero_debias_on(c) ? 1 : 0, sched_ln.st));
  if (p.a2c) {   // ClipGlobalNorm(RMSProp)   a2c_acktr.py:250-251
    ACX_TRY(dot_partial(l->grads, l->grads, P, l->dot_partials, kDotPartials, st));
    ACX_TRY(rmsprop_clip_step(l->params, l->accum, l->grads, P, l->dot_partials, kDotPartials, l->sched, c.rms_decay,
                              c.rms_epsilon, c.clip_norm, l->scalars + 6, st));
    ACX_TRY(refresh_weight_planes(l, st));
    for (int k = 6; k <= 9; ++k) mark(l, k, st);
    return 0;
  }
  if (p.cold) {     // kfac_utils.py:42-43: ClipGlobalNorm(Momentum(3e-4, 0.9)) - this also increments global_step
    ACX_TRY(dot_partial(l->grads, l->grads, P, l->dot_partials, kDotPartials, st));
    ACX_TRY(momentum_clip_step(l->params, l->accum, l->grads, P, l->dot_partials, kDotPartials, c.cold_lr, c.cold_momentum,
                               c.clip_norm, l->scalars + 6, st));
  } else if (!ext_ema) {          // kfac_utils.py:44: all covariance updates
    // nothing else in this phase reads the running sums unless the inverses are refreshed: the HBM-bound EMA pass then
    // runs on a side lane next to the preconditioning (joined at the end of the phase, before the next update's
    // statistics overwrite its input)
    if (!p.invert) {
      ema_ln = lane_of(l, 2, st);
      ACX_TRY(fork_lane(l, st, ema_ln));
    }
    ACX_TRY(ema_update(l->sums, l->stats, l->factor_floats, c.cov_ema_decay, 1.0f, ema_ln.st));
  }
  mark(l, 6, st);
  if (p.invert) ACX_TRY(join_lane(l, sched_ln, st));   // the refresh reads the zero-debias factor of the new covariance count
  if (p.invert) {
    // ACX_INV_IMPL: 2 (default) = fp32, all factor tiles resident in shared memory, one persistent kernel (kfac_inv.cu);
    // 1 = the fp64 Gauss-Jordan as one persistent kernel; 0 = the round-1 fp64 chain of ~150 launches (also the fallback when
    // the tiles do not fit the SMs' shared memory)
    static int inv_impl = -1;
    if (inv_impl < 0) {
      const char* e = getenv("ACX_INV_IMPL");
      inv_impl = e ? atoi(e) : 2;
    }
    // (the serial pivot-block inversions of the chain run on a side lane next to the trailing updates, joined inside, step by step)
    const cudaStream_t side = lane_of(l, 1, st).st;
    if (inv_impl == 2)
      ACX_TRY(l->invert(st, side));
    else if (inv_impl == 1)
      ACX_TRY(spd_inverse_persistent(l->h_jobs, l->d_jobs, 12, l->sched, l->damp, l->d_a_ptrs, l->d_g_ptrs, l->d_a_dims,
                                     l->d_g_dims, l->lambdas, 6, l->inv_bar, st));
    else
      ACX_TRY(l->invert_chain(st, side));
  }
  mark(l, 7, st);
  if (p.kfac_apply) {
    ACX_TRY(precondition(l, st));
    mark(l, 8, st);
    ACX_TRY(join_lane(l, sched_ln, st));             // the step reads the learning rate
    ACX_TRY(dot_partial(l->grads, l->precon, P, l->dot_partials, kDotPartials, st));
    ACX_TRY(kfac_step(l->params, l->velocity, l->precon, P, l->dot_partials, kDotPartials, l->sched, c.momentum,
                      c.norm_constraint, l->scalars + 4, st));
  }
  if (p.refresh) ACX_TRY(refresh_weight_planes(l, st, true));
  ACX_TRY(join_lane(l, sched_ln, st));
  ACX_TRY(join_lane(l, ema_ln, st));
  if (!p.kfac_apply) mark(l, 8, st);
  mark(l, 9, st);
  return 0;
}

// graphs are off, or stage timing brackets the work with events on the caller's stream
static bool eager_graphs(const acx_learner* l) { return !l->cfg.use_graphs || l->profiling; }

static int phase2(acx_learner* l, cudaStream_t st) {
  const Plan p = l->sch.plan();
  GraphKey key = {2, p.key() | (l->external_ema ? 1 << 10 : 0) | (l->peer.world > 1 ? 1 << 11 : 0), nullptr, nullptr};
  const int r = l->graphs.run(key, st, eager_graphs(l), [&]() { return issue_phase2(l, p, st); });
  if (r) return r;
  l->sch.advance(p);
  return 0;
}

}  // namespace acx

extern "C" {

static int check_cfg(const acx_learner_config_t* c) {
  ACX_CHECK(c != nullptr, "null config");
  ACX_CHECK(c->num_envs > 0 && c->num_steps > 0, "num_envs and num_steps must be positive");
  ACX_CHECK(c->num_actions >= 1 && c->num_actions <= 31, "num_actions must be in [1, 31]");
  ACX_CHECK(c->conv3_filters >= 8 && c->conv3_filters <= 256 && c->conv3_filters % 8 == 0,
            "conv3_filters must be a multiple of 8 in [8, 256]");
  ACX_CHECK(c->world_size >= 1, "world_size");
  ACX_CHECK((long long)(c->num_envs) * c->num_steps <= (1 << 20), "rollout too large");
  if (c->acktr) ACX_CHECK(c->invert_every >= 1, "invert_every");
  return 0;
}

static void init_dims(acx_learner* l, const acx_learner_config_t* cfg) {
  l->cfg = *cfg;
  l->gather = cfg->conv_impl == 0 && cfg->gemm_impl == 0;
  // precision: activations / gradients are kept as act_planes bf16 planes; a GEMM of level L accumulates the plane
  // pairs (i, j) with i + j <= L  (1 pair = bf16 inputs, 3 pairs ~ 2^-17, 6 pairs = fp32 class)
  switch (cfg->precision) {
    case 1: l->act_planes = 2; l->grad_planes = 2; l->lvl_fwd = 1; l->lvl_bwd = 1; l->lvl_factor = 1; l->lvl_precon = 2; break;
    case 2: l->act_planes = 2; l->grad_planes = 2; l->lvl_fwd = 1; l->lvl_bwd = 1; l->lvl_factor = 0; l->lvl_precon = 2; break;
    case 3: l->act_planes = 1; l->grad_planes = 1; l->lvl_fwd = 0; l->lvl_bwd = 0; l->lvl_factor = 0; l->lvl_precon = 1; break;
    // 4: forward fp32 class (the ReLU masks are decided by the sign of pre-activations that suffer cancellation), gradients
    // on 2 planes / 3 pairs: 2^-17 relative to sum|terms| per GEMM, which compounds to ~6e-4 on the conv1/conv2 gradients
    // for iid-uniform observations (measured, profiles/r1_precision.md) - inside the contract but without margin
    case 4: l->act_planes = 3; l->grad_planes = 2; l->lvl_fwd = 2; l->lvl_bwd = 1; l->lvl_factor = 1; l->lvl_precon = 2; break;
    // 5: forward and backward with 6 pairs on 3 planes (the round-1 default until the mask-synchronised measurement
    // showed that the third plane is below the accumulator's own rounding: no quantity improves, profiles/r1_precision.md)
    case 5: l->act_planes = 3; l->grad_planes = 3; l->lvl_fwd = 2; l->lvl_bwd = 2; l->lvl_factor = 1; l->lvl_precon = 2; break;
    // default (parity grade): activations and gradients on 2 bf16 planes, 3 plane pairs (hi*hi + hi*lo + lo*hi: ~2^-17,
    // at the level of the fp32 tensor-core accumulation itself) for forward, backward and factor SYRKs; the
    // preconditioning products 6 pairs on 3 planes (inverses and gradient blocks have a wide dynamic range)
    default: l->act_planes = 2; l->grad_planes = 2; l->lvl_fwd = 1; l->lvl_bwd = 1; l->lvl_factor = 1; l->lvl_precon = 2; break;
  }
  // Fisher-sample rows of the backward pass (conv input gradients): they only feed the output factors G_l, which are
  // themselves accumulated at lvl_factor = 3 pairs and held to 1e-3, so 3 pairs are enough there (measured G-factor error
  // in profiles/r1_precision.md); the true-gradient rows keep lvl_bwd.  ACX_FISHER_LEVEL=2 restores 6 pairs everywhere.
  l->lvl_fisher = l->lvl_bwd < 1 ? l->lvl_bwd : 1;
  if (const char* e = getenv("ACX_PRECON_LEVEL")) {   // triage: plane-pair level of the fc4 preconditioning GEMMs
    const int v = atoi(e);
    if (v >= 0 && v <= 2) l->lvl_precon = v;
  }
  if (const char* e = getenv("ACX_FISHER_LEVEL")) {
    const int v = atoi(e);
    if (v >= 0 && v <= l->lvl_bwd) l->lvl_fisher = v;
  }
  l->E = cfg->num_envs;
  l->T = cfg->num_steps;
  l->N = l->E * l->T;
  l->R = l->N + l->E;
  l->A = cfg->num_actions;
  l->c3 = cfg->conv3_filters;
  setup_layers(l);
  l->sch.acktr = cfg->acktr != 0;
  l->sch.num_cold_updates = cfg->num_cold_updates;
  l->sch.invert_every = cfg->invert_every;
}

size_t acx_learner_arena_bytes(const acx_learner_config_t* cfg) {
  if (check_cfg(cfg)) return 0;
  acx_learner tmp;
  init_dims(&tmp, cfg);
  return layout(&tmp, nullptr);
}

acx_learner_t* acx_learner_create(const acx_learner_config_t* cfg, void* d_arena, size_t arena_bytes) {
  if (check_cfg(cfg)) return nullptr;
  acx_learner* l = new acx_learner();
  init_dims(l, cfg);
  const size_t need = layout(l, nullptr);
  if (d_arena == nullptr || arena_bytes < need || (reinterpret_cast<uintptr_t>(d_arena) & 255) != 0) {
    acx::set_error("acx_learner_create: arena must be a 256-byte aligned device buffer of at least acx_learner_arena_bytes()");
    delete l;
    return nullptr;
  }
  layout(l, reinterpret_cast<uint8_t*>(d_arena));
  l->arena_base = reinterpret_cast<uint8_t*>(d_arena);
  setup_gather(l);
  register_buffers(l);
  l->value_weight = cfg->value_loss_weight;
  l->act_calls = 0;
  l->lanes = cfg->num_lanes <= 0 ? kMaxLanes : std::min(cfg->num_lanes, kMaxLanes);
  if (cudaEventCreateWithFlags(&l->a_ready, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&l->reduced, cudaEventDisableTiming) != cudaSuccess) {
    acx::set_error("acx_learner_create: cudaEventCreateWithFlags failed");
    acx_learner_destroy(l);
    return nullptr;
  }
  for (int i = 0; i < 4; ++i)
    l->conv_fwd_tc[i] = (i == 1 || i == 2) && l->gather && conv_tc_supported(geom_of(l, i), 0);
  for (int i = 0; i + 1 < l->lanes; ++i)
    if (cudaStreamCreateWithFlags(&l->side[i], cudaStreamNonBlocking) != cudaSuccess) {
      acx::set_error("acx_learner_create: cudaStreamCreateWithFlags failed");
      acx_learner_destroy(l);
      return nullptr;
    }
  // zero everything persistent, then the initial schedule, optimizer slots and K-FAC tables
  if (l->upload(d_arena, need, !cfg->acktr, cfg->lr_start, cfg->damping) != 0) {
    acx_learner_destroy(l);
    return nullptr;
  }
  if (cfg->acktr && (cfg->cov_init_identity || cfg->inv_init_identity)) {   // SURVEY A.7-U3 (the arena is zero so far)
    std::vector<float> eye;
    cudaError_t e = cudaSuccess;
    auto put_eye = [&](float* dst, int d) {
      eye.assign((size_t)d * d, 0.0f);
      for (int i = 0; i < d; ++i) eye[(size_t)i * d + i] = 1.0f;
      if (e == cudaSuccess) e = cudaMemcpy(dst, eye.data(), eye.size() * sizeof(float), cudaMemcpyHostToDevice);
    };
    if (cfg->cov_init_identity) {
      for (int i = 0; i < 5; ++i) put_eye(l->sums + l->aoff[i], l->adim[i]);
      for (int i = 0; i < 6; ++i) put_eye(l->sums + l->goff[i], l->blk[i].C);
    }
    if (cfg->inv_init_identity) {
      for (int i = 0; i < 6; ++i) {
        put_eye(l->inv + l->ainv_off[i], l->blk[i].K + 1);
        put_eye(l->inv + l->ginv_off[i], l->blk[i].C);
      }
      l->sch.inverses_valid = true;   // the K-FAC apply is a real step from the first update on
    }
    if (e != cudaSuccess) {
      acx::set_error(std::string("acx_learner_create: cudaMemcpy: ") + cudaGetErrorString(e));
      acx_learner_destroy(l);
      return nullptr;
    }
  }
  if (cfg->acktr && cfg->inv_init_identity) {   // bf16 operand planes of the identity inverses
    if (acx_learner_refresh_weights(l, nullptr) != 0 || cudaDeviceSynchronize() != cudaSuccess) {
      acx_learner_destroy(l);
      return nullptr;
    }
  }
  return l;
}

void acx_learner_destroy(acx_learner_t* l) {
  if (!l) return;
  if (l->profiling)
    for (int k = 0; k < ACX_NUM_STAGES + 2; ++k) cudaEventDestroy(l->ev[k]);
  for (cudaEvent_t e : l->lane_events) cudaEventDestroy(e);
  if (l->a_ready) cudaEventDestroy(l->a_ready);
  if (l->reduced) cudaEventDestroy(l->reduced);
  for (cudaStream_t s : l->side)
    if (s) cudaStreamDestroy(s);
  delete l;   // the graph cache destroys its executable graphs
}

int acx_learner_set_profiling(acx_learner_t* l, int enable) {
  ACX_CHECK(l, "null learner");
  if (enable && !l->profiling) {
    for (int k = 0; k < ACX_NUM_STAGES + 2; ++k) {
      ACX_CUDA(cudaEventCreate(&l->ev[k]));
      l->ev_set[k] = false;
    }
    l->profiling = true;
  } else if (!enable && l->profiling) {
    for (int k = 0; k < ACX_NUM_STAGES + 2; ++k) cudaEventDestroy(l->ev[k]);
    l->profiling = false;
  }
  return 0;
}

int acx_learner_stage_ms(acx_learner_t* l, float* h_ms) {
  ACX_CHECK(l && h_ms, "null argument");
  ACX_CHECK(l->profiling, "profiling is off (acx_learner_set_profiling)");
  // stages 0..3 = marks 0..4 (phase 1), stages 4..7 = marks 5..9 (phase 2)
  for (int s = 0; s < ACX_NUM_STAGES; ++s) {
    const int a = s < 4 ? s : s + 1, b = a + 1;
    h_ms[s] = 0.0f;
    if (l->ev_set[a] && l->ev_set[b]) {
      ACX_CUDA(cudaEventSynchronize(l->ev[b]));
      float ms = 0.0f;
      ACX_CUDA(cudaEventElapsedTime(&ms, l->ev[a], l->ev[b]));
      h_ms[s] = ms;
    }
  }
  return 0;
}

size_t acx_learner_num_params(const acx_learner_t* l) { return l ? l->num_params : 0; }

int acx_learner_set_params(acx_learner_t* l, const float* h_params, void* stream) {
  ACX_CHECK(l && h_params, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ACX_TRY(l->set_params(h_params, st));
  ACX_TRY(refresh_weight_planes(l, st));
  ACX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int acx_learner_get_params(acx_learner_t* l, float* h_params, void* stream) {
  ACX_CHECK(l && h_params, "null argument");
  return l->get_params(h_params, reinterpret_cast<cudaStream_t>(stream));
}

int acx_learner_refresh_weights(acx_learner_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ACX_TRY(refresh_weight_planes(l, st));
  return l->split_inverses(st);
}

void* acx_learner_buffer(acx_learner_t* l, const char* name, size_t* num_bytes) {
  return l ? l->buffer("acx_learner_buffer", name, num_bytes) : nullptr;
}

int acx_learner_phase1(acx_learner_t* l, const int32_t* d_fisher_labels, const float* d_fisher_eps, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK((d_fisher_labels == nullptr) == (d_fisher_eps == nullptr), "inject both Fisher labels and eps, or neither");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool fisher = l->sch.fisher();
  GraphKey key = {1, (fisher ? 1 : 0) | (l->loss_variant << 8), d_fisher_labels, d_fisher_eps};
  const int r = l->graphs.run(key, st, eager_graphs(l), [&]() { return issue_phase1(l, d_fisher_labels, d_fisher_eps, st); });
  l->a_ready_valid = r == 0 && fisher && l->lanes > 1 && !l->profiling;
  return r;
}

int acx_learner_set_loss_weights(acx_learner_t* l, float policy_weight, float value_weight) {
  ACX_CHECK(l, "null learner");
  l->policy_weight = policy_weight;
  l->value_weight = value_weight;
  // every distinct pair replays its own captured graphs (kernel arguments are baked into a graph)
  static std::vector<std::pair<float, float>> seen;
  int id = -1;
  for (size_t i = 0; i < seen.size(); ++i)
    if (seen[i].first == policy_weight && seen[i].second == value_weight) id = (int)i;
  if (id < 0) {
    seen.push_back(std::make_pair(policy_weight, value_weight));
    id = (int)seen.size() - 1;
  }
  l->loss_variant = (policy_weight == 1.0f && value_weight == l->cfg.value_loss_weight) ? 0 : 1 + id;
  return 0;
}

int acx_learner_update(acx_learner_t* l, const int32_t* d_fisher_labels, const float* d_fisher_eps, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK((d_fisher_labels == nullptr) == (d_fisher_eps == nullptr), "inject both Fisher labels and eps, or neither");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // both phases as ONE captured graph per schedule variant (nothing has to happen between them unless the caller runs a
  // collective there): one graph launch per update
  const bool fisher = l->sch.fisher();
  const Plan p = l->sch.plan();
  const int k1 = (fisher ? 1 : 0) | (l->loss_variant << 8);
  const int k2 = p.key() | (l->external_ema ? 1 << 10 : 0) | (l->peer.world > 1 ? 1 << 11 : 0);
  GraphKey key = {4, k1 | (k2 << 16), d_fisher_labels, d_fisher_eps};
  const int r = l->graphs.run(key, st, eager_graphs(l), [&]() {
    const int r1 = issue_phase1(l, d_fisher_labels, d_fisher_eps, st);
    return r1 ? r1 : issue_phase2(l, p, st);
  });
  l->a_ready_valid = false;
  if (r) return r;
  l->sch.advance(p);
  return 0;
}

int acx_learner_update_plan(const acx_learner_t* l, int* has_factors, int* will_invert) {
  ACX_CHECK(l, "null learner");
  const Plan p = l->sch.plan();
  if (has_factors) *has_factors = (!p.a2c && !p.cold) ? 1 : 0;
  if (will_invert) *will_invert = p.invert ? 1 : 0;
  return 0;
}

int acx_learner_set_external_ema(acx_learner_t* l, int on) {
  ACX_CHECK(l, "null learner");
  l->external_ema = on != 0;
  return 0;
}

int acx_learner_ema(acx_learner_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK(l->cfg.acktr, "acx_learner_ema: not a K-FAC learner");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const acx_learner_config_t& c = l->cfg;
  if (c.world_size > 1) ACX_TRY(scale_f32(l->stats, l->factor_floats, 1.0f / (float)c.world_size, st));
  ACX_TRY(ema_update(l->sums, l->stats, l->factor_floats, c.cov_ema_decay, 1.0f, st));
  return 0;
}

int acx_learner_set_peers(acx_learner_t* l, int rank, int world, void* const* peer_arena_bases) {
  ACX_CHECK(l, "null learner");
  if (world <= 1 || peer_arena_bases == nullptr) {   // back to caller-side collectives
    l->peer = acx::PeerState();
    return 0;
  }
  ACX_CHECK(world == l->cfg.world_size && world <= 8 && rank >= 0 && rank < world, "acx_learner_set_peers: rank / world");
  acx::PeerState ps;
  ps.rank = rank;
  ps.world = world;
  for (int k = 0; k < world; ++k) {
    ps.base[k] = k == rank ? l->arena_base : reinterpret_cast<uint8_t*>(peer_arena_bases[k]);
    ACX_CHECK(ps.base[k] != nullptr, "acx_learner_set_peers: null peer arena");
  }
  l->peer = ps;
  return 0;
}

int acx_learner_peer_reduce_prefix(acx_learner_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK(l->peer.world > 1, "acx_learner_peer_reduce_prefix: no peers (acx_learner_set_peers)");
  // the input-factor statistics A (the prefix of the bucket), summed over the ranks on the caller's side stream while phase 2
  // runs; unscaled (acx_learner_ema scales all statistics)
  return acx::peer_allreduce(l->peer, reinterpret_cast<uint8_t*>(l->bucket) - l->arena_base,
                             reinterpret_cast<uint8_t*>(l->peer_flags) - l->arena_base,
                             reinterpret_cast<uint8_t*>(l->peer_epochs) - l->arena_base, (long long)l->goff[0],
                             (long long)l->goff[0], 1.0f, 1, reinterpret_cast<cudaStream_t>(stream));
}

int acx_learner_wait_reduced(acx_learner_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CUDA(cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), l->reduced, 0));
  return 0;
}

int acx_learner_wait_input_factors(acx_learner_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  if (!l->a_ready_valid) return -1;   // nothing was raised by the last phase 1: the prefix is complete only when phase 1 is
  ACX_CUDA(cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), l->a_ready, 0));
  return 0;
}

int acx_learner_phase2(acx_learner_t* l, void* stream) {
  ACX_CHECK(l, "null learner");
  return phase2(l, reinterpret_cast<cudaStream_t>(stream));
}

int64_t acx_learner_global_step(const acx_learner_t* l) { return l ? l->sch.gs : -1; }

int acx_learner_set_state(acx_learner_t* l, int64_t global_step, int64_t num_cov_updates, int inverses_valid, void* stream) {
  ACX_CHECK(l, "null learner");
  ACX_CHECK(global_step >= 0 && num_cov_updates >= 0, "negative counters");
  return l->sch.set(global_step, num_cov_updates, inverses_valid, l->cfg.lr_start, l->cfg.cov_ema_decay, zero_debias_on(l->cfg),
                    l->sched, reinterpret_cast<cudaStream_t>(stream));
}

int acx_learner_get_state(const acx_learner_t* l, int64_t* global_step, int64_t* num_cov_updates, int* inverses_valid) {
  ACX_CHECK(l, "null learner");
  l->sch.get(global_step, num_cov_updates, inverses_valid);
  return 0;
}

int acx_learner_act(acx_learner_t* l, const uint8_t* d_obs, int rows, const float* d_uniform, int greedy, int32_t* d_actions,
                    float* d_logits, float* d_values, void* stream) {
  ACX_CHECK(l && d_obs && d_actions, "null argument");
  ACX_CHECK(rows > 0 && rows <= l->R, "rows must be in [1, num_envs * num_steps + num_envs]");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // One acting step = ~8 small launches (32 rows: every kernel sits on the launch-latency floor).  With stable buffers
  // (the usual rollout loop: the environment's stack buffer in, the agent's action buffer out) the step is captured once
  // per pointer set and replayed as ONE graph launch; the call counter that seeds Philox lives on the device.
  auto issue = [&]() -> int {
    // the acting step is ONE serial chain of small launches on one stream: every kernel lets its successor be scheduled at
    // once (programmatic dependent launch, level 2) - inside an update the same setting gains nothing because the early
    // blocks compete with the other lanes
    set_pdl_override(2);
    int r = forward(l, d_obs, rows, lane_of(l, 0, st), nullptr, nullptr, false);
    if (r == 0) r = sample_actions(l->logits, d_uniform, l->cfg.seed, 0, rows, l->A, greedy, d_actions, st, l->act_counter);
    set_pdl_override(-1);
    if (r) return r;
    if (d_logits)
      ACX_CUDA(cudaMemcpyAsync(d_logits, l->logits, (size_t)rows * l->A * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (d_values) ACX_CUDA(cudaMemcpyAsync(d_values, l->values, (size_t)rows * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  };
  l->act_calls++;
  GraphKey key = {3, (greedy ? 1 : 0) | (rows << 1), d_obs, d_actions, d_uniform, d_logits, d_values};
  return l->graphs.run_bounded(key, st, eager_graphs(l), issue);
}

}  // extern "C"
