// learner_core.cu - the host code shared by learner.cu and mlp.cu (learner_core.cuh)
#include <algorithm>
#include <cmath>
#include <vector>

#include "learner_core.cuh"

namespace acx {

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

void fill_gemm(acx_gemm_t* g, const Planes& a, const Planes& b, int trans, int m, int n, int k, int level, float alpha, int symmetric,
               const GemmOut& o, float* workspace, size_t workspace_bytes) {
  memset(g, 0, sizeof(*g));
  for (int i = 0; i < a.n; ++i) g->a.planes[i] = a.p[i];
  for (int i = 0; i < b.n; ++i) g->b.planes[i] = b.p[i];
  g->a.num_planes = a.n;
  g->b.num_planes = b.n;
  g->a.ld = a.ld;
  g->b.ld = b.ld;
  if (trans) {
    g->a.rows = k; g->a.cols = m; g->b.rows = k; g->b.cols = n;
  } else {
    g->a.rows = m; g->a.cols = k; g->b.rows = n; g->b.cols = k;
  }
  g->trans_a = g->trans_b = trans;
  g->m = m; g->n = n; g->k = k;
  g->num_pairs = level_pairs(level, a.n, b.n, g->pair_a, g->pair_b);
  g->alpha = alpha;
  g->bias = o.bias;
  g->relu = o.relu;
  g->symmetric = symmetric;
  g->c = o.c;
  g->ldc = o.ldc;
  if (o.planes) {
    for (int i = 0; i < o.planes->n; ++i) g->c_planes[i] = o.planes->p[i];
    g->c_num_planes = o.planes->n;
    g->ldc_planes = o.planes->ld;
  }
  g->mask_plane = o.mask;
  g->mask_ld = o.mask_ld;
  g->mask_rows = o.mask_rows;
  g->a_gather = o.a_gather;
  g->b_gather = o.b_gather;
  g->perm_m = o.perm_m;
  g->perm_n = o.perm_n;
  g->workspace = workspace;
  g->workspace_bytes = workspace_bytes;
}

// ------------------------------------------------------------------------------------------------
// KfacBlocks
// ------------------------------------------------------------------------------------------------
void KfacBlocks::set_blocks(int n) {
  nb = n;
  size_t off = 0;
  for (int i = 0; i < nb; ++i) {
    blk[i].off = off;
    off += (size_t)(blk[i].K + 1) * blk[i].C;
  }
  num_params = off;
  params_pad = align_up(off, 4);
  const int nfac = blk[nb - 1].afac + 1;
  for (int i = 0; i < nb; ++i) adim[blk[i].afac] = blk[i].K + 1;
  size_t f = 0;
  for (int i = 0; i < nfac; ++i) {
    aoff[i] = f;
    f += align_up((size_t)adim[i] * adim[i], 4);
  }
  for (int i = 0; i < nb; ++i) {
    goff[i] = f;
    f += align_up((size_t)blk[i].C * blk[i].C, 4);
  }
  factor_floats = f;
  size_t v = 0;
  for (int i = 0; i < nb; ++i) {
    ainv_off[i] = v;
    v += align_up((size_t)(blk[i].K + 1) * (blk[i].K + 1), 4);
  }
  for (int i = 0; i < nb; ++i) {
    ginv_off[i] = v;
    v += align_up((size_t)blk[i].C * blk[i].C, 4);
  }
  inv_floats = v;
}

void KfacBlocks::take_state(Arena& ar) {
  const size_t P = params_pad, F = factor_floats;
  params = ar.f32(P);
  velocity = ar.f32(P);
  accum = ar.f32(P);
  precon = ar.f32(P);
  bucket_floats = P + F + 4;
  bucket = ar.f32(bucket_floats);
  stats = bucket;   // [A | G]: one contiguous block for the EMA, A first (the early all-reduce prefix)
  grads = bucket + F;
  bscalars = bucket + F + P;
  sums = ar.f32(F);
  inv = ar.f32(inv_floats);
  damp = ar.f32(16);
  lambdas = ar.f32(8);
  scalars = ar.f32(16);
  sched = reinterpret_cast<Sched*>(ar.take(sizeof(Sched)));
}

void KfacBlocks::take_tables(Arena& ar) {
  d_a_ptrs = reinterpret_cast<const float**>(ar.take(kMaxBlocks * sizeof(float*)));
  d_g_ptrs = reinterpret_cast<const float**>(ar.take(kMaxBlocks * sizeof(float*)));
  d_a_dims = reinterpret_cast<int*>(ar.take(kMaxBlocks * sizeof(int)));
  d_g_dims = reinterpret_cast<int*>(ar.take(kMaxBlocks * sizeof(int)));
  d_jobs = reinterpret_cast<InvJob*>(ar.take(2 * kMaxBlocks * sizeof(InvJob)));
  d_pjobs = reinterpret_cast<PreconJob*>(ar.take(kMaxBlocks * sizeof(PreconJob)));
  inv_bar = reinterpret_cast<unsigned int*>(ar.take(256));
  act_counter = reinterpret_cast<unsigned long long*>(ar.take(256));
  precon_w = ar.f32(params_pad);
  for (int i = 0; i < nb; ++i) {
    const int d = blk[i].K + 1, c = blk[i].C;
    ainv_pl[i] = take_planes(ar, 3, d, pad8(d));
    ginv_pl[i] = take_planes(ar, 3, c, pad8(c));
  }
  // inverse jobs (sorted by decreasing n at upload)
  auto job = [&](InvJob& j, const float* s, int n, int damp_index, float* out, const Planes& pl) {
    j.s = s;
    j.n = n;
    j.damp_index = damp_index;
    j.work_m = reinterpret_cast<double*>(ar.take((size_t)n * n * sizeof(double)));
    j.work_x = reinterpret_cast<double*>(ar.take(((size_t)3 * 32 * n + 2 * 32 * 32 + 2048) * sizeof(double)));
    j.inv = out;
    for (int q = 0; q < 3; ++q) j.planes[q] = pl.p[q];
    j.ld_planes = pl.ld;
  };
  for (int i = 0; i < nb; ++i) {
    job(h_jobs[i], sums + aoff[blk[i].afac], blk[i].K + 1, 2 * i, inv + ainv_off[i], ainv_pl[i]);
    job(h_jobs[nb + i], sums + goff[i], blk[i].C, 2 * i + 1, inv + ginv_off[i], ginv_pl[i]);
  }
  // small blocks (C <= 64) are preconditioned by the batched fp32 SIMT kernels
  num_pjobs = 0;
  pjobs_max_d = 0;
  for (int i = 0; i < nb; ++i) {
    if (blk[i].C > 64) continue;
    PreconJob& pj = h_pjobs[num_pjobs++];
    pj.v = grads + blk[i].off;
    pj.ginv = inv + ginv_off[i];
    pj.ainv = inv + ainv_off[i];
    pj.w = precon_w + blk[i].off;
    pj.u = precon + blk[i].off;
    pj.d = blk[i].K + 1;
    pj.c = blk[i].C;
    pj.scale = 1.0f / (float)blk[i].Tnorm;
    pjobs_max_d = std::max(pjobs_max_d, pj.d);
  }
}

void KfacBlocks::register_buffers() {
  const size_t P = num_params;
  reg("params", params, P * 4);
  reg("velocity", velocity, P * 4);
  reg("accum", accum, P * 4);
  reg("precon", precon, P * 4);
  reg("grads", grads, P * 4);
  reg("reduce_bucket", bucket, bucket_floats * 4);
  reg("factor_stats", stats, factor_floats * 4);
  reg("factor_sums", sums, factor_floats * 4);
  reg("inverses", inv, inv_floats * 4);
  reg("dampings", damp, 2 * nb * 4);
  reg("scalars", scalars, 16 * 4);
  reg("sched", sched, sizeof(Sched));
  const int heads = blk[nb - 1].afac;   // the last input factor is the one the two heads share
  for (int f = 0; f <= heads; ++f) {
    const std::string fn = f < heads ? blk[f].name : "heads";
    const size_t b = (size_t)adim[f] * adim[f] * 4;
    reg("stats/A/" + fn, stats + aoff[f], b);
    reg("sums/A/" + fn, sums + aoff[f], b);
  }
  for (int i = 0; i < nb; ++i) {
    const Block& B = blk[i];
    const size_t gb = (size_t)B.C * B.C * 4, vb = (size_t)(B.K + 1) * B.C * 4;
    reg("stats/G/" + B.name, stats + goff[i], gb);
    reg("sums/G/" + B.name, sums + goff[i], gb);
    reg("inv/A/" + B.name, inv + ainv_off[i], (size_t)(B.K + 1) * (B.K + 1) * 4);
    reg("inv/G/" + B.name, inv + ginv_off[i], gb);
    reg("params/" + B.name, params + B.off, vb);
    reg("grads/" + B.name, grads + B.off, vb);
    reg("precon/" + B.name, precon + B.off, vb);
    reg("velocity/" + B.name, velocity + B.off, vb);
    reg("accum/" + B.name, accum + B.off, vb);
  }
}

void* KfacBlocks::buffer(const char* caller, const char* name, size_t* num_bytes) {
  if (!name) return nullptr;
  auto it = named.find(name);
  if (it == named.end()) {
    set_error(std::string(caller) + ": unknown buffer '" + name + "'");
    return nullptr;
  }
  if (num_bytes) *num_bytes = it->second.bytes;
  return it->second.ptr;
}

int KfacBlocks::upload(void* arena, size_t arena_bytes, bool rmsprop, float lr_start, float damping) {
  ACX_CUDA(cudaMemset(arena, 0, arena_bytes));
  if (rmsprop) {
    const std::vector<float> ones(params_pad, 1.0f);
    ACX_CUDA(cudaMemcpy(accum, ones.data(), params_pad * 4, cudaMemcpyHostToDevice));
  }
  const Sched s0 = {0ull, 0ull, lr_start, 1.0f};
  ACX_CUDA(cudaMemcpy(sched, &s0, sizeof(s0), cudaMemcpyHostToDevice));
  const float* ap[kMaxBlocks];
  const float* gp[kMaxBlocks];
  int ad[kMaxBlocks], gd[kMaxBlocks];
  float lam[8] = {0};
  for (int i = 0; i < nb; ++i) {
    ap[i] = sums + aoff[blk[i].afac];
    gp[i] = sums + goff[i];
    ad[i] = adim[blk[i].afac];
    gd[i] = blk[i].C;
    lam[i] = damping / (float)blk[i].Tnorm;
  }
  ACX_CUDA(cudaMemcpy(d_a_ptrs, ap, nb * sizeof(float*), cudaMemcpyHostToDevice));
  ACX_CUDA(cudaMemcpy(d_g_ptrs, gp, nb * sizeof(float*), cudaMemcpyHostToDevice));
  ACX_CUDA(cudaMemcpy(d_a_dims, ad, nb * sizeof(int), cudaMemcpyHostToDevice));
  ACX_CUDA(cudaMemcpy(d_g_dims, gd, nb * sizeof(int), cudaMemcpyHostToDevice));
  ACX_CUDA(cudaMemcpy(lambdas, lam, sizeof(lam), cudaMemcpyHostToDevice));
  std::stable_sort(h_jobs, h_jobs + 2 * nb, [](const InvJob& a, const InvJob& b) { return a.n > b.n; });
  ACX_CUDA(cudaMemcpy(d_pjobs, h_pjobs, sizeof(h_pjobs), cudaMemcpyHostToDevice));
  ACX_CUDA(cudaMemcpy(d_jobs, h_jobs, sizeof(h_jobs), cudaMemcpyHostToDevice));
  return 0;
}

int KfacBlocks::set_params(const float* h_params, cudaStream_t st) {
  ACX_CUDA(cudaMemcpyAsync(params, h_params, num_params * sizeof(float), cudaMemcpyHostToDevice, st));
  return 0;
}

int KfacBlocks::get_params(float* h_params, cudaStream_t st) {
  ACX_CUDA(cudaMemcpyAsync(h_params, params, num_params * sizeof(float), cudaMemcpyDeviceToHost, st));
  ACX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int KfacBlocks::split_inverses(cudaStream_t st) {
  for (int i = 0; i < nb; ++i) {
    const int d = blk[i].K + 1, c = blk[i].C;
    ACX_TRY(split_planes(inv + ainv_off[i], d, d, d, 1.0f, ainv_pl[i].p[0], ainv_pl[i].p[1], ainv_pl[i].p[2], 3, ainv_pl[i].ld, st));
    ACX_TRY(split_planes(inv + ginv_off[i], c, c, c, 1.0f, ginv_pl[i].p[0], ginv_pl[i].p[1], ginv_pl[i].p[2], 3, ginv_pl[i].ld, st));
  }
  return 0;
}

int KfacBlocks::invert(cudaStream_t st, cudaStream_t side) {
  const int r = spd_inverse_resident(h_jobs, 2 * nb, sched, damp, d_a_ptrs, d_g_ptrs, d_a_dims, d_g_dims, lambdas, nb, inv_bar, st);
  if (r >= 0) return r;
  ACX_TRY(compute_dampings(d_a_ptrs, d_g_ptrs, d_a_dims, d_g_dims, lambdas, nb, damp, st));
  return spd_inverse_batched(h_jobs, d_jobs, 2 * nb, sched, damp, st, side);
}

// ------------------------------------------------------------------------------------------------
// Schedule
// ------------------------------------------------------------------------------------------------
Plan Schedule::plan() const {
  Plan p = {false, false, false, false, false};
  if (!acktr) {
    p.a2c = true;
    p.refresh = true;
    return p;
  }
  p.cold = gs < num_cold_updates;
  const int64_t gs1 = gs + (p.cold ? 1 : 0);   // the cold optimizer increments global_step itself (kfac_utils.py:43)
  p.invert = gs1 > num_cold_updates && (gs1 - num_cold_updates) % invert_every == 0;   // kfac_utils.py:47-50
  // kfac_utils.py:52-53 runs always; with kfac's zero-initialised inverses it is exactly a no-op (U = 0, v stays 0)
  // until the first refresh, so only the step counter moves.
  p.kfac_apply = inverses_valid || p.invert;
  p.refresh = p.cold || p.kfac_apply;
  return p;
}

void Schedule::advance(const Plan& p) {
  if (p.a2c) {
    gs += 1;
    return;
  }
  if (p.cold) gs += 1; else ncov += 1;
  if (p.invert) inverses_valid = true;
  gs += 1;
}

int Schedule::set(int64_t global_step, int64_t num_cov_updates, int valid, float lr_start, float ema_decay, bool zero_debias,
                  Sched* d_sched, cudaStream_t st) {
  gs = global_step;
  ncov = num_cov_updates;
  inverses_valid = valid != 0;
  Sched s;
  s.gs = (unsigned long long)global_step;
  s.ncov = (unsigned long long)num_cov_updates;
  s.lr = lr_start;
  s.debias = (num_cov_updates > 0 && zero_debias) ? (float)(1.0 / (1.0 - pow((double)ema_decay, (double)num_cov_updates))) : 1.0f;
  ACX_CUDA(cudaMemcpyAsync(d_sched, &s, sizeof(s), cudaMemcpyHostToDevice, st));
  ACX_CUDA(cudaStreamSynchronize(st));
  return 0;
}

void Schedule::get(int64_t* global_step, int64_t* num_cov_updates, int* valid) const {
  if (global_step) *global_step = gs;
  if (num_cov_updates) *num_cov_updates = ncov;
  if (valid) *valid = inverses_valid ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
// GraphCache
// ------------------------------------------------------------------------------------------------
bool GraphKey::operator<(const GraphKey& o) const {
  if (phase != o.phase) return phase < o.phase;
  if (variant != o.variant) return variant < o.variant;
  if (p0 != o.p0) return p0 < o.p0;
  if (p1 != o.p1) return p1 < o.p1;
  if (p2 != o.p2) return p2 < o.p2;
  if (p3 != o.p3) return p3 < o.p3;
  return p4 < o.p4;
}

GraphCache::~GraphCache() {
  for (auto& kv : graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
}

int GraphCache::end_capture(Entry& ge, cudaStream_t st, int issue_result, uint64_t launches_before) {
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(st, &graph);
  if (issue_result != 0 || e != cudaSuccess || graph == nullptr) {
    if (graph) cudaGraphDestroy(graph);
    if (issue_result == 0) set_error(std::string("graph capture failed: ") + cudaGetErrorString(e));
    return issue_result ? issue_result : 4;
  }
  ge.launches = g_launch_count - launches_before;
  g_launch_count = launches_before;
  const cudaError_t e2 = cudaGraphInstantiate(&ge.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e2 != cudaSuccess) {
    ge.exec = nullptr;
    set_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e2));
    return 4;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// test hook: one inverse refresh of a block set built as the learners build it (include/acx.h)
// ------------------------------------------------------------------------------------------------
namespace {

struct DebugRefresh {
  KfacBlocks kb;
  void* arena = nullptr;
  cudaStream_t st = nullptr, side = nullptr;
  ~DebugRefresh() {
    if (st) cudaStreamSynchronize(st);
    if (side) cudaStreamSynchronize(side);
    if (arena) cudaFree(arena);
    if (st) cudaStreamDestroy(st);
    if (side) cudaStreamDestroy(side);
  }
};

int debug_kfac_invert(int num_blocks, const int* h_k, const int* h_c, const int* h_tnorm, int shared_heads, float damping,
                      float debias, const float* h_sums, int path, int side_stream, float* h_inv, uint16_t* h_planes,
                      float* h_damp, int* h_path_ran) {
  ACX_CHECK(num_blocks >= 1 && num_blocks <= kMaxBlocks && h_k && h_c && h_tnorm && h_sums && h_inv && h_planes && h_damp &&
                h_path_ran, "bad argument");
  ACX_CHECK(path >= 0 && path <= 2, "path must be 0, 1 or 2");
  ACX_CHECK(!shared_heads || (num_blocks >= 2 && h_k[num_blocks - 1] == h_k[num_blocks - 2]),
            "shared heads need two blocks with the same input dimension");
  const int nfac = shared_heads ? num_blocks - 1 : num_blocks;
  ACX_CHECK(nfac <= kMaxBlocks - 1, "at most 5 input factors");
  DebugRefresh d;
  KfacBlocks& kb = d.kb;
  for (int i = 0; i < num_blocks; ++i) {
    ACX_CHECK(h_k[i] >= 0 && h_c[i] >= 1 && h_tnorm[i] >= 1, "bad block dimensions");
    kb.blk[i].name = "b" + std::to_string(i);
    kb.blk[i].K = h_k[i];
    kb.blk[i].C = h_c[i];
    kb.blk[i].Tnorm = h_tnorm[i];
    kb.blk[i].afac = i < nfac ? i : nfac - 1;
  }
  kb.set_blocks(num_blocks);
  Arena sizing;
  kb.take_state(sizing);
  kb.take_tables(sizing);
  const size_t bytes = align_up(sizing.used, 256);
  ACX_CUDA(cudaMalloc(&d.arena, bytes));
  Arena ar;
  ar.base = reinterpret_cast<uint8_t*>(d.arena);
  kb.take_state(ar);
  kb.take_tables(ar);
  ACX_TRY(kb.upload(d.arena, bytes, false, 0.0f, damping));
  ACX_CUDA(cudaStreamCreateWithFlags(&d.st, cudaStreamNonBlocking));
  if (side_stream) ACX_CUDA(cudaStreamCreateWithFlags(&d.side, cudaStreamNonBlocking));
  size_t off = 0;
  for (int f = 0; f < nfac; ++f) {
    const size_t n2 = (size_t)kb.adim[f] * kb.adim[f];
    ACX_CUDA(cudaMemcpy(kb.sums + kb.aoff[f], h_sums + off, n2 * sizeof(float), cudaMemcpyHostToDevice));
    off += n2;
  }
  for (int i = 0; i < num_blocks; ++i) {
    const size_t n2 = (size_t)kb.blk[i].C * kb.blk[i].C;
    ACX_CUDA(cudaMemcpy(kb.sums + kb.goff[i], h_sums + off, n2 * sizeof(float), cudaMemcpyHostToDevice));
    off += n2;
  }
  const Sched s = {0ull, 0ull, 0.0f, debias};
  ACX_CUDA(cudaMemcpy(kb.sched, &s, sizeof(s), cudaMemcpyHostToDevice));
  ACX_CUDA(cudaDeviceSynchronize());   // the set-up above ran on the legacy stream, the refresh runs on a non-blocking one
  const uint64_t launches = g_launch_count;
  if (path == 0) {
    ACX_TRY(kb.invert(d.st, d.side));
    *h_path_ran = g_launch_count - launches == 1 ? 0 : 1;   // the resident refresh is one launch, the chain several
  } else if (path == 1) {
    const int r = spd_inverse_resident(kb.h_jobs, 2 * num_blocks, kb.sched, kb.damp, kb.d_a_ptrs, kb.d_g_ptrs, kb.d_a_dims,
                                       kb.d_g_dims, kb.lambdas, num_blocks, kb.inv_bar, d.st);
    if (r < 0) return -1;
    ACX_TRY(r);
    *h_path_ran = 0;
  } else {
    ACX_TRY(compute_dampings(kb.d_a_ptrs, kb.d_g_ptrs, kb.d_a_dims, kb.d_g_dims, kb.lambdas, num_blocks, kb.damp, d.st));
    ACX_TRY(spd_inverse_batched(kb.h_jobs, kb.d_jobs, 2 * num_blocks, kb.sched, kb.damp, d.st, d.side));
    *h_path_ran = 1;
  }
  ACX_CUDA(cudaStreamSynchronize(d.st));
  size_t io = 0, po = 0;
  for (int j = 0; j < 2 * num_blocks; ++j) {
    const int i = j % num_blocks;
    const int n = j < num_blocks ? kb.blk[i].K + 1 : kb.blk[i].C;
    const float* inv = kb.inv + (j < num_blocks ? kb.ainv_off[i] : kb.ginv_off[i]);
    const Planes& pl = j < num_blocks ? kb.ainv_pl[i] : kb.ginv_pl[i];
    ACX_CUDA(cudaMemcpy(h_inv + io, inv, (size_t)n * n * sizeof(float), cudaMemcpyDeviceToHost));
    io += (size_t)n * n;
    for (int q = 0; q < 3; ++q) {
      ACX_CUDA(cudaMemcpy(h_planes + po, pl.p[q], (size_t)n * pl.ld * sizeof(bf16), cudaMemcpyDeviceToHost));
      po += (size_t)n * pl.ld;
    }
  }
  ACX_CUDA(cudaMemcpy(h_damp, kb.damp, 2 * num_blocks * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace

}  // namespace acx

extern "C" int acx_debug_kfac_invert(int num_blocks, const int* h_k, const int* h_c, const int* h_tnorm, int shared_heads,
                                     float damping, float debias, const float* h_sums, int path, int side_stream, float* h_inv,
                                     uint16_t* h_planes, float* h_damp, int* h_path_ran) {
  return acx::debug_kfac_invert(num_blocks, h_k, h_c, h_tnorm, shared_heads, damping, debias, h_sums, path, side_stream, h_inv,
                                h_planes, h_damp, h_path_ran);
}
