// learner_core.cuh - the host code that the Atari learner (learner.cu) and the fully connected learner (mlp.cu) share:
// arena and plane helpers, the GEMM descriptor, the K-FAC blocks with their state in the arena, the schedule of
// ColdStartPeriodicInvUpdateKfacOpt on the host, and the CUDA-graph cache.  Each learner keeps its own forward, backward,
// phase 1 / phase 2 and preconditioning GEMMs.
#pragma once
#include <map>
#include <string>

#include "layers.cuh"

namespace acx {

constexpr int kColsumChunks = 592;
constexpr int kDotPartials = 296;   // two chunks per SM: ~11 elements per thread at 865 k parameters
constexpr int kMaxBlocks = 6;       // K-FAC blocks of a learner: Nature-CNN 6, fully connected up to 4 hidden layers + 2 heads

#define ACX_TRY(expr)        \
  do {                       \
    int _r = (expr);         \
    if (_r) return _r;       \
  } while (0)

struct Buf {
  void* ptr;
  size_t bytes;
};

// bump allocator over the device arena (base == nullptr: size pass only)
struct Arena {
  uint8_t* base = nullptr;
  size_t used = 0;
  void* take(size_t bytes) {
    used = align_up(used, 256);
    void* p = base ? base + used : nullptr;
    used += bytes;
    return p;
  }
  float* f32(size_t n) { return reinterpret_cast<float*>(take(n * sizeof(float))); }
};

inline int pad8(int x) { return (x + 7) / 8 * 8; }
Planes take_planes(Arena& ar, int nplanes, size_t rows, int ld);
Planes offset_rows(const Planes& p, size_t rows);
// plane pairs (i, j) with i + j <= level, low orders first
int level_pairs(int level, int a_planes, int b_planes, int* pa, int* pb);

// where a GEMM writes and what its epilogue does; the gather and perm fields are the Atari learner's conv operands
struct GemmOut {
  float* c = nullptr;
  int ldc = 0;
  const Planes* planes = nullptr;
  const float* bias = nullptr;
  int relu = 0;
  const bf16* mask = nullptr;
  int mask_ld = 0, mask_rows = 0;
  const acx_gather_t* a_gather = nullptr;   // operands read in place from NHWC tensors (acx.h)
  const acx_gather_t* b_gather = nullptr;
  int perm_m = 0, perm_n = 0;
};

// C = alpha op(A) op(B) over the plane pairs of `level` (trans: A [k, m], B [k, n]; else A [m, k], B [n, k])
void fill_gemm(acx_gemm_t* g, const Planes& a, const Planes& b, int trans, int m, int n, int k, int level, float alpha, int symmetric,
               const GemmOut& o, float* workspace, size_t workspace_bytes);

// one K-FAC block: V = [K+1, C] (weights, then the bias row)
struct Block {
  std::string name;
  int K = 0, C = 0;
  size_t off = 0;   // offset of V in the flat parameter vector
  int afac = 0;     // index of its input factor (the two heads share one)
  int Tnorm = 1;    // T~ used for lambda / T~ and the 1 / T~ rescale (SURVEY A.7-U1)
};

// The K-FAC blocks of a learner and the fp32 state that goes with them in the arena: parameters, optimizer slots, the reduce
// bucket [A | G | grads | 4 loss scalars], running factor sums, inverses (fp32 and bf16 planes), dampings, the device
// schedule, and the tables of the inverse refresh and of the small-block preconditioning.
struct KfacBlocks {
  int nb = 0;                  // blocks
  Block blk[kMaxBlocks];
  size_t num_params = 0, params_pad = 0;
  int adim[kMaxBlocks - 1];    // input factor f is [adim, adim]
  size_t aoff[kMaxBlocks - 1], goff[kMaxBlocks], factor_floats = 0;
  size_t ainv_off[kMaxBlocks], ginv_off[kMaxBlocks], inv_floats = 0;
  // fp32 state
  float *params, *velocity, *accum, *precon, *precon_w;
  float *bucket, *stats, *grads, *bscalars;
  size_t bucket_floats;
  float *sums;                 // running factor sums, same layout as stats
  float *inv;                  // fp32 inverses: A^-1 per block, then G^-1 per block
  float *damp, *lambdas, *scalars;
  Planes ainv_pl[kMaxBlocks], ginv_pl[kMaxBlocks];
  Sched* sched;
  const float** d_a_ptrs;
  const float** d_g_ptrs;
  int *d_a_dims, *d_g_dims;
  InvJob h_jobs[2 * kMaxBlocks];
  InvJob* d_jobs;
  unsigned int* inv_bar;             // grid-barrier counter of the persistent inverse kernel
  unsigned long long* act_counter;   // device-resident number of acting calls (Philox step of sample_actions)
  PreconJob h_pjobs[kMaxBlocks];
  PreconJob* d_pjobs;
  int num_pjobs, pjobs_max_d;
  std::map<std::string, Buf> named;

  // offsets of the parameters, factors and inverses of blk[0, n) (names, K, C, afac and Tnorm set)
  void set_blocks(int n);
  // arena layout in two calls, state block first (one contiguous block so that it can be zeroed / checkpointed as a whole)
  void take_state(Arena& ar);
  void take_tables(Arena& ar);
  void reg(const std::string& name, void* p, size_t bytes) { named[name] = Buf{p, bytes}; }
  void register_buffers();
  void* buffer(const char* caller, const char* name, size_t* num_bytes);
  // zero the arena, then the initial device state: Sched, RMSProp's ms = 1 (TF-1 default), the pointer / dim / lambda
  // tables and the job tables (inverse jobs sorted by decreasing n)
  int upload(void* arena, size_t arena_bytes, bool rmsprop, float lr_start, float damping);
  int set_params(const float* h_params, cudaStream_t st);   // asynchronous: the caller refreshes its weight planes
  int get_params(float* h_params, cudaStream_t st);
  // the bf16 planes of the stored inverses (derived state, after the inverses were written from outside)
  int split_inverses(cudaStream_t st);
  // inverse refresh: factor tiles resident in shared memory (kfac_inv.cu); when they do not fit, dampings and then the
  // fp64 chain (kfac.cu), with its serial pivot-block inversions on `side` when given
  int invert(cudaStream_t st, cudaStream_t side = nullptr);
};

// what one update's optimizer step does, decided on the host from the schedule counters (kfac_utils.py:38-53)
struct Plan {
  bool a2c, cold, invert, kfac_apply, refresh;
  int key() const { return (a2c ? 1 : 0) | (cold ? 2 : 0) | (invert ? 4 : 0) | (kfac_apply ? 8 : 0) | (refresh ? 16 : 0); }
};

// host mirror of the schedule counters
struct Schedule {
  bool acktr = false;
  int num_cold_updates = 0, invert_every = 1;
  int64_t gs = 0, ncov = 0;
  bool inverses_valid = false;

  // kfac_utils.py:42-44: covariances (Fisher samples) only after the cold phase
  bool fisher() const { return acktr && gs >= num_cold_updates; }
  Plan plan() const;
  void advance(const Plan& p);
  // counters and the matching device Sched (lr restarts from lr_start; debias from the covariance count when zero_debias)
  int set(int64_t global_step, int64_t num_cov_updates, int valid, float lr_start, float ema_decay, bool zero_debias, Sched* d_sched,
          cudaStream_t st);
  void get(int64_t* global_step, int64_t* num_cov_updates, int* valid) const;
};

struct GraphKey {
  int phase, variant;
  const void* p0;
  const void* p1;
  const void* p2 = nullptr;
  const void* p3 = nullptr;
  const void* p4 = nullptr;
  bool operator<(const GraphKey& o) const;
};

// CUDA-graph cache: the first use of a key runs eagerly (it also performs one-time host work such as tensor-map encoding and
// function attributes), the second is captured and instantiated, later uses replay the graph.  Valid because no kernel takes
// a step-dependent scalar by value (see Sched).
struct GraphCache {
  struct Entry {
    int uses = 0;
    cudaGraphExec_t exec = nullptr;
    uint64_t launches = 0;
  };
  std::map<GraphKey, Entry> graphs;

  GraphCache() = default;
  GraphCache(const GraphCache&) = delete;
  GraphCache& operator=(const GraphCache&) = delete;
  ~GraphCache();

  template <typename F>
  int run(const GraphKey& key, cudaStream_t st, bool eager, F&& issue) {
    if (eager || st == nullptr) return issue();
    {
      // the caller is capturing this stream itself (e.g. a whole rollout as one graph): the launches simply become nodes
      // of the caller's graph
      cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
      if (cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive) return issue();
    }
    Entry& ge = graphs[key];
    if (ge.uses == 0) {
      ge.uses = 1;
      return issue();
    }
    if (ge.exec == nullptr) {
      const uint64_t before = g_launch_count;
      ACX_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      const int r = issue();
      ACX_TRY(end_capture(ge, st, r, before));
    }
    ACX_CUDA(cudaGraphLaunch(ge.exec, st));
    count_launch((int)ge.launches);
    ge.uses += 1;
    return 0;
  }
  // acting calls key their graphs by the caller's buffers: once 512 graphs exist, a new key runs eagerly (ever-changing
  // buffers must not hoard graphs)
  template <typename F>
  int run_bounded(const GraphKey& key, cudaStream_t st, bool eager, F&& issue) {
    if (graphs.size() > 512 && graphs.find(key) == graphs.end()) return issue();
    return run(key, st, eager, issue);
  }

 private:
  int end_capture(Entry& ge, cudaStream_t st, int issue_result, uint64_t launches_before);
};

}  // namespace acx
