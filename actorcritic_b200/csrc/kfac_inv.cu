// kfac_inv.cu - the K-FAC inverse refresh (kfac `posdef_inv`, driven by kfac_utils.py:47-50) with all factor matrices
// RESIDENT IN SHARED MEMORY: one persistent kernel, fp32 like the reference's Cholesky inverses.
//
// The twelve damped factors of an update (A^-1 and G^-1 per layer; 1569^2 ... 1^2 at conv3 = 32, 3137^2 at conv3 = 64) are
// cut into 64 x 64 tiles; only the upper tiles are kept (the Gauss-Jordan iterates of an SPD matrix keep a signed symmetry,
// see kfac.cu), 571 tiles = 9.4 MB at conv3 = 32 and ~1520 tiles = 25 MB at conv3 = 64: they fit the shared memory of the
// 148 SMs (33 MB), so every tile is loaded ONCE, stays in the shared memory of its owner CTA for all 49 (99) pivot steps and
// is written once at the end.  Per pivot step only the two 32 x n row panels (Rold = pivot rows, R = D^-1 Rold) travel
// through L2.  Blocked Gauss-Jordan without pivoting, 32-wide pivot blocks, per step p:
//   owners      panels:  every owner of a tile that intersects the pivot rows extracts its 32 x 64 piece of Rold, multiplies
//                        it by D_p^-1 and publishes both pieces                                               | barrier 1
//               update:  every owned tile  M_ij -= sigma_i Rold_i^T R_j  (+ pivot rows / columns / block); the owners of
//                        the blocks (p+1, p+2) and (p+2, p+2) publish them for the look-ahead of the NEXT step  | barrier 2
//   look-ahead  one dedicated CTA per job (it owns no tiles) computes D_{p+1}^-1 = (M_qq - M_pq^T D_p^-1 M_pq)^-1 from the two
//               blocks published during step p-1 - the serial 32-step inversion - while the owners run step p
// Work and ownership are static (tile g -> CTA g mod W): no atomics besides the barrier counter; a CTA that waits at a
// barrier for more than ~2 s records an error and leaves.  The fp64 kernel chain of kfac.cu is the fallback when the tiles do
// not fit (conv3 widths beyond 64, wide fully connected layers).
// The update phase was also built as four 64-thread groups with 8 x 8 register tiles: bit-identical, but measured slower on a
// B200 at 32 x 20 (0.98 vs 0.85 ms per refresh: late pivot steps have only 2-3 active tiles per CTA, and a 2-warp group
// cannot hide its own shared-memory latency), so it was removed.
#include <cstdlib>

#include "layers.cuh"

namespace acx {

namespace {

constexpr int RB = 32;        // pivot block
constexpr int TS = 64;        // tile edge
constexpr int OPLD = 68;      // row stride (floats) of the staged operand pieces: 16-byte aligned rows, spreads the banks
constexpr int RES_JOBS = 12;
constexpr int RES_THREADS = 256;
constexpr int TILE_FLOATS = TS * TS;
constexpr int STAGE_FLOATS = 3 * RB * OPLD + RB * (RB + 1) + 64;   // A piece | B piece | C piece | D^-1 [32][33 (34)] | slack
constexpr int RES_SMEM_TOTAL = 232448;   // 227 KB per CTA on sm_100 (static + dynamic)

struct ResJob {
  const float* s;   // [n, n] running covariance sum
  int n;
  int damp_index;
  float* x;         // scratch: Rold [32][ldp] | R [32][ldp] | D^-1 [2][1024] | PQ [2][1024] | QQ [2][1024]
  float* inv;       // [n, n] fp32 result
  bf16* planes[3];  // [n, ld_planes]
  int ld_planes;
  int tile_base;    // first global tile id of this job
  int nt;           // tile rows
  int ldp;          // row stride of the panels (n rounded up to 4)
};

struct ResArgs {
  ResJob jobs[RES_JOBS];
  int num_jobs;
  int steps;         // ceil(n_max / RB)
  int slots;         // tiles per owner CTA (upper bound)
  int total_tiles;
  const Sched* sched;
  float* damp;
  const float* const* a_ptrs;
  const float* const* g_ptrs;
  const int* a_dims;
  const int* g_dims;
  const float* lambdas;
  int num_layers;
  unsigned int* bar;
  int trace;
};

__device__ int g_res_error = 0;
// triage (ACX_INV_TRACE=1), per pivot step 8 slots of clock64 stamps: last owner CTA [0] step start [1] panels done
// [2] barrier 1 passed [3] update done [4] barrier 2 passed; look-ahead CTA 0: [5] start [6] inversion done [7] barrier 2 passed
__device__ long long g_res_trace[128 * 8];

__device__ __forceinline__ float* sc_rold(const ResJob& jb) { return jb.x; }
__device__ __forceinline__ float* sc_r(const ResJob& jb) { return jb.x + (size_t)RB * jb.ldp; }
__device__ __forceinline__ float* sc_dinv(const ResJob& jb, int p) { return jb.x + (size_t)2 * RB * jb.ldp + (p & 1) * 1024; }
__device__ __forceinline__ float* sc_pq(const ResJob& jb, int s) { return jb.x + (size_t)2 * RB * jb.ldp + 2048 + (s & 1) * 1024; }
__device__ __forceinline__ float* sc_qq(const ResJob& jb, int s) { return jb.x + (size_t)2 * RB * jb.ldp + 4096 + (s & 1) * 1024; }

__device__ __forceinline__ unsigned int ld_relaxed(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// grid barrier on a monotonically increasing counter.  arrive: this CTA's writes are published and counted (one release
// reduction: no separate full fence); wait: relaxed polling until all CTAs have arrived `epoch` times, then one acquire
// fence.  An early arrival for barrier k + 1 is only legal after this CTA has PASSED barrier k.
__device__ __forceinline__ void grid_arrive(unsigned int* bar, unsigned int& epoch) {
  ++epoch;
  __syncthreads();
  if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
}
__device__ __forceinline__ bool grid_wait(unsigned int* bar, unsigned int epoch) {
  int ok = 1;
  if (threadIdx.x == 0) {
    const unsigned int target = epoch * gridDim.x;
    if (ld_relaxed(bar) < target) {
      const long long t0 = clock64();
      while (ld_relaxed(bar) < target) {
        if (clock64() - t0 > 4000000000ll) {   // ~2 s: some CTA of the grid is not running
          atomicExch(&g_res_error, 31);
          ok = 0;
          break;
        }
      }
    }
    asm volatile("fence.acq_rel.gpu;" ::: "memory");
  }
  return __syncthreads_and(ok) != 0;
}

// inverse of a 32 x 32 SPD block in shared memory (row stride 33), all 256 threads; unblocked Gauss-Jordan without
// pivoting; rows / columns beyond the matrix are identity padding.  The 32 elimination steps are a serial chain (the
// critical path of the look-ahead CTA): every thread keeps its four elements (rows w, w+8, w+16, w+24 of column tx) in
// registers for all steps; per step only the pivot row and the pivot column are exchanged through a small double-buffered
// shared array, with ONE barrier:  barrier -> read row k / column k -> reciprocal -> 4 FMAs -> publish row / column k+1.
__device__ __forceinline__ void invert32(float (*d)[RB + 1], float* xbuf /* [2][64] */) {
  const int tx = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  float v[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) v[c] = d[w + 8 * c][tx];
  if (w == 0) xbuf[tx] = v[0];                     // row 0
  if (tx == 0) {
#pragma unroll
    for (int c = 0; c < 4; ++c) xbuf[32 + w + 8 * c] = v[c];   // column 0
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RB; ++k) {
    const float* rb = xbuf + (k & 1) * 64;
    const float* cb = rb + 32;
    const float inv_p = __frcp_rn(rb[k]);
    const float scaled = rb[tx] * inv_p;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int ty = w + 8 * c;
      const float col_k = cb[ty];
      float r = fmaf(-col_k, scaled, v[c]);
      if (ty == k) r = scaled;
      if (tx == k) r = -col_k * inv_p;
      if (ty == k && tx == k) r = inv_p;
      v[c] = r;
    }
    if (k + 1 < RB) {
      float* nb = xbuf + ((k + 1) & 1) * 64;
      if (w == ((k + 1) & 7)) nb[tx] = v[(k + 1) >> 3];          // row k + 1 lives in warp (k + 1) % 8, register (k + 1) / 8
      if (tx == k + 1) {
#pragma unroll
        for (int c = 0; c < 4; ++c) nb[32 + w + 8 * c] = v[c];     // column k + 1
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) d[w + 8 * c][tx] = v[c];
  __syncthreads();
}

__device__ __forceinline__ float prep_value(const ResJob& jb, int gi, int gj, float debias, float dv) {
  // the statistics are symmetric up to the rounding of the border writes: symmetrise while loading
  float v = 0.5f * (__ldcg(jb.s + (size_t)gi * jb.n + gj) + __ldcg(jb.s + (size_t)gj * jb.n + gi)) * debias;
  if (gi == gj) v += dv;
  return v;
}

// blocks (s, s+1) and (s+1, s+1) of the CURRENT matrix, if this tile holds them, for the look-ahead of step s
__device__ __forceinline__ void publish_pair(const ResJob& jb, int s, int ti, int tj, const float* T) {
  const int n = jb.n;
  const int nblk = (n + RB - 1) / RB;
  const int q = s + 1;
  if (q >= nblk) return;
  if (ti == (s >> 1) && tj == (q >> 1)) {
    const int r0 = (s & 1) * RB, c0 = (q & 1) * RB;
    float* dst = sc_pq(jb, s);
    for (int e = threadIdx.x; e < RB * RB; e += RES_THREADS) {
      const int y = e >> 5, x = e & 31;
      __stcg(dst + e, (q * RB + x < n) ? T[(r0 + y) * TS + c0 + x] : 0.0f);
    }
  }
  if (ti == (q >> 1) && tj == (q >> 1)) {
    const int r0 = (q & 1) * RB;
    float* dst = sc_qq(jb, s);
    for (int e = threadIdx.x; e < RB * RB; e += RES_THREADS) {
      const int y = e >> 5, x = e & 31;
      const bool in = q * RB + y < n && q * RB + x < n;
      __stcg(dst + e, in ? T[(r0 + y) * TS + r0 + x] : (y == x ? 1.0f : 0.0f));
    }
  }
}

// panels of step p from an owned tile that intersects the pivot rows: its 32 x 64 piece of Rold and R = D_p^-1 Rold
template <int DBG = 0>   // triage (tools/micro/inv_micro.cu): 1 = no D^-1 load, 2 = no stores, 4 = no product, 8 = no Rold extraction
__device__ __forceinline__ void panel_piece(const ResJob& jb, int p, int ti, int tj, const float* T, float* As, float* Bs,
                                            float (*Ds)[RB + 1]) {
  const int n = jb.n, tp = p >> 1, pr0 = (p & 1) * RB, p0 = p * RB;
  const bool row_stored = ti == tp;             // tile (tp, j), j >= tp (the diagonal tile is stored in full)
  if (!row_stored && tj != tp) return;          // (mirror: tile (i, tp), i < tp)
  const int nb = min(RB, n - p0);
  const int col0 = (row_stored ? tj : ti) * TS;
  __syncthreads();   // staging may still be in use
  const float* dinv = sc_dinv(jb, p);
  float* Dt = &Ds[0][0];   // D_p^-1 transposed, row stride 34: Dt[m * 34 + k] = D^-1[k][m] (8-byte aligned row pairs)
  if (!(DBG & 1)) {
    float dreg[4];   // all four loads in flight before the first shared-memory store
#pragma unroll
    for (int c = 0; c < 4; ++c) dreg[c] = __ldcg(dinv + threadIdx.x + c * RES_THREADS);
#pragma unroll
    for (int c = 0; c < 4; ++c) Dt[(threadIdx.x & 31) * 34 + (threadIdx.x >> 5) + 8 * c] = dreg[c];
  }
  if (DBG & 8) {
  } else if (row_stored) {
    for (int e = threadIdx.x; e < RB * TS; e += RES_THREADS) {
      const int k = e >> 6, c = e & 63;
      As[k * OPLD + c] = (k < nb && col0 + c < n) ? T[(pr0 + k) * TS + c] : 0.0f;
    }
  } else {          // only the mirror M_bp is stored (b processed, p not): M_pb = -M_bp^T
    for (int e = threadIdx.x; e < RB * TS; e += RES_THREADS) {
      const int c = e >> 5, k = e & 31;
      As[k * OPLD + c] = (k < nb && col0 + c < n) ? -T[c * TS + pr0 + k] : 0.0f;
    }
  }
  __syncthreads();
  // R piece = D^-1 Rold as 32 outer products: thread -> rows 2 ty, 2 ty + 1, columns 4 tx .. 4 tx + 3.  Per m and warp
  // one 8-byte broadcast load of the D^-1 column pair and one conflict-free 16-byte load of the Rold row: 6 shared-memory
  // wavefronts for 8 FMAs (the row-per-thread mapping this replaces needed 17 and was bound by shared-memory bandwidth)
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  float acc[2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
#pragma unroll 8
  for (int m = 0; m < ((DBG & 4) ? 0 : RB); ++m) {
    const float2 d2 = *reinterpret_cast<const float2*>(Dt + m * 34 + 2 * ty);
    const float4 x = *reinterpret_cast<const float4*>(As + m * OPLD + 4 * tx);
    acc[0][0] = fmaf(d2.x, x.x, acc[0][0]);
    acc[0][1] = fmaf(d2.x, x.y, acc[0][1]);
    acc[0][2] = fmaf(d2.x, x.z, acc[0][2]);
    acc[0][3] = fmaf(d2.x, x.w, acc[0][3]);
    acc[1][0] = fmaf(d2.y, x.x, acc[1][0]);
    acc[1][1] = fmaf(d2.y, x.y, acc[1][1]);
    acc[1][2] = fmaf(d2.y, x.z, acc[1][2]);
    acc[1][3] = fmaf(d2.y, x.w, acc[1][3]);
  }
  if (DBG & 2) {
    if (acc[0][0] + acc[1][3] + acc[0][1] + acc[0][2] + acc[0][3] + acc[1][0] + acc[1][1] + acc[1][2] == 12345.0f) sc_rold(jb)[0] = acc[0][3];
    return;
  }
  if (col0 + 4 * tx < jb.ldp) {   // ldp is a multiple of 4 and >= n: whole float4s, columns in [n, ldp) receive zeros
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int k2 = 2 * ty + i;
      const float4 o = *reinterpret_cast<const float4*>(As + k2 * OPLD + 4 * tx);
      __stcg(reinterpret_cast<float4*>(sc_rold(jb) + (size_t)k2 * jb.ldp + col0 + 4 * tx), o);
      __stcg(reinterpret_cast<float4*>(sc_r(jb) + (size_t)k2 * jb.ldp + col0 + 4 * tx),
             make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
    }
  }
  (void)Bs;
}

// operand pieces of one tile update, fetched into registers (issued before the previous tile is computed)
struct OpRegs {
  float4 a[2], b[2], c[2];   // c: R for the tile's ROW range (pivot-column tiles only: M_ip = -sigma_i R_i^T)
};
__device__ __forceinline__ void fetch_ops(const ResJob& jb, int p, int ti, int tj, OpRegs& o) {
  const int n = jb.n, p0 = p * RB;
  const float* rold = sc_rold(jb);
  const float* rr = sc_r(jb);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int e = threadIdx.x + h * RES_THREADS;   // 32 rows x 16 float4
    const int k = e >> 4, c = (e & 15) * 4;
    const int gi = ti * TS + c, gj = tj * TS + c;
    float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
    if (gi < n && !(gi >= p0 && gi < p0 + RB)) {     // ldp >= gi + 4: the whole float4 is inside the (zero padded) panel
      va = __ldcg(reinterpret_cast<const float4*>(rold + (size_t)k * jb.ldp + gi));
      if (gi < p0) {   // sigma_i = -1 for processed rows
        va.x = -va.x; va.y = -va.y; va.z = -va.z; va.w = -va.w;
      }
    }
    if (gj < n && !(gj >= p0 && gj < p0 + RB)) vb = __ldcg(reinterpret_cast<const float4*>(rr + (size_t)k * jb.ldp + gj));
    o.a[h] = va;
    o.b[h] = vb;
    if (tj == (p >> 1) && ti != tj)   // off-diagonal tile of the pivot's tile column (its rows are never pivot rows)
      o.c[h] = gi < n ? __ldcg(reinterpret_cast<const float4*>(rr + (size_t)k * jb.ldp + gi)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
__device__ __forceinline__ void stage_ops(const OpRegs& o, float* As, float* Bs, float* Cs, bool with_c) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int e = threadIdx.x + h * RES_THREADS;
    const int k = e >> 4, c = (e & 15) * 4;
    *reinterpret_cast<float4*>(As + k * OPLD + c) = o.a[h];
    *reinterpret_cast<float4*>(Bs + k * OPLD + c) = o.b[h];
    if (with_c) *reinterpret_cast<float4*>(Cs + k * OPLD + c) = o.c[h];
  }
}

// M_ij -= sigma_i Rold_i^T R_j on the resident tile; pivot rows / columns / block replaced (kfac.cu "Symmetry")
__device__ __forceinline__ void update_tile(const ResJob& jb, int p, int ti, int tj, float* T, const float* As, const float* Bs,
                                            const float* Cs) {
  const int n = jb.n, p0 = p * RB, tp = p >> 1;
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  float acc[4][4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 t4 = *reinterpret_cast<const float4*>(T + (4 * ty + q) * TS + 4 * tx);
    acc[q][0] = t4.x; acc[q][1] = t4.y; acc[q][2] = t4.z; acc[q][3] = t4.w;
  }
  float4 a_nxt = *reinterpret_cast<const float4*>(As + 4 * ty);
  float4 b_nxt = *reinterpret_cast<const float4*>(Bs + 4 * tx);
#pragma unroll
  for (int k = 0; k < RB; ++k) {
    const float4 a4 = a_nxt, b4 = b_nxt;
    if (k + 1 < RB) {   // the next k's operands are in flight while this k's 16 FMAs issue
      a_nxt = *reinterpret_cast<const float4*>(As + (k + 1) * OPLD + 4 * ty);
      b_nxt = *reinterpret_cast<const float4*>(Bs + (k + 1) * OPLD + 4 * tx);
    }
    const float a[4] = {a4.x, a4.y, a4.z, a4.w};
    const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[q][r] = fmaf(-a[q], b[r], acc[q][r]);
  }
  if (ti == tp || tj == tp) {
    const float* dinv = sc_dinv(jb, p);
    const float* Ri = ti == tj ? Bs : Cs;   // R for this tile's row range (diagonal tile: its own column piece)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int gi = ti * TS + 4 * ty + q;
      const bool ip = gi >= p0 && gi < p0 + RB;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int gj = tj * TS + 4 * tx + r;
        const bool jp = gj >= p0 && gj < p0 + RB;
        if (gi >= n || gj >= n || !(ip || jp)) continue;
        float v;
        if (ip && jp)
          v = __ldcg(dinv + (gi - p0) * RB + (gj - p0));
        else if (ip)
          v = Bs[(gi - p0) * OPLD + 4 * tx + r];                       // M_pj = R_j (its column is not a pivot column)
        else {
          const float x = Ri[(gj - p0) * OPLD + 4 * ty + q];              // M_ip = -sigma_i R_i^T
          v = gi < p0 ? x : -x;
        }
        acc[q][r] = v;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q)
    *reinterpret_cast<float4*>(T + (4 * ty + q) * TS + 4 * tx) = make_float4(acc[q][0], acc[q][1], acc[q][2], acc[q][3]);
}

// fp32 inverse + its bf16 operand planes from a resident tile (and its mirror)
__device__ __forceinline__ void finish_tile(const ResJob& jb, int ti, int tj, const float* T, float* stage) {
  const int n = jb.n;
  auto put = [&](int gi, int gj, float v) {
    jb.inv[(size_t)gi * n + gj] = v;
    bf16 p0, p1, p2;
    split3(v, p0, p1, p2);
    const size_t i = (size_t)gi * jb.ld_planes + gj;
    jb.planes[0][i] = p0;
    jb.planes[1][i] = p1;
    jb.planes[2][i] = p2;
  };
  // transposed copy with a padded stride (conflict-free column reads)
  __syncthreads();
  for (int e = threadIdx.x; e < TILE_FLOATS; e += RES_THREADS) stage[(e & 63) * (TS + 1) + (e >> 6)] = T[e];
  __syncthreads();
  for (int e = threadIdx.x; e < TILE_FLOATS; e += RES_THREADS) {
    const int r = e >> 6, c = e & 63;
    const int gi = ti * TS + r, gj = tj * TS + c;
    if (gi >= n || gj >= n) continue;
    if (ti == tj) {
      put(gi, gj, 0.5f * (T[e] + stage[r * (TS + 1) + c]));     // diagonal tiles hold both halves: average them
    } else {
      put(gi, gj, T[e]);
    }
  }
  if (ti != tj) {
    for (int e = threadIdx.x; e < TILE_FLOATS; e += RES_THREADS) {
      const int r = e >> 6, c = e & 63;                          // mirrored element (tj*64 + r, ti*64 + c) = T[c][r]
      const int gi = tj * TS + r, gj = ti * TS + c;
      if (gi >= n || gj >= n) continue;
      put(gi, gj, stage[r * (TS + 1) + c]);
    }
  }
}

__global__ void __launch_bounds__(RES_THREADS, 1) inv_resident_kernel(const __grid_constant__ ResArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ int s_job[16], s_ti[16], s_tj[16];
  __shared__ ResJob s_jobs[RES_JOBS];      // the job table out of the parameter bank (dynamic indexing)
  if (threadIdx.x < RES_JOBS) s_jobs[threadIdx.x] = a.jobs[threadIdx.x];
  __syncthreads();
  const int G = gridDim.x, cta = blockIdx.x;
  const int ND = a.num_jobs;            // look-ahead CTAs [0, ND), owners [ND, G)
  const int W = G - ND;
  float* stage = smem;                  // operand pieces / D^-1 / transposition buffer
  float* As = stage;
  float* Bs = stage + RB * OPLD;
  float* Cs = stage + 2 * RB * OPLD;
  float (*Ds)[RB + 1] = reinterpret_cast<float (*)[RB + 1]>(stage + 3 * RB * OPLD);
  float* tiles = smem + STAGE_FLOATS;
  unsigned int epoch = 0;
  const bool owner = cta >= ND;
  const int wid = cta - ND;
  // ---- static ownership: slot s of owner w holds global tile g = s * W + w
  if (owner && threadIdx.x < a.slots) {
    const int g = threadIdx.x * W + wid;
    int job = -1, ti = 0, tj = 0;
    if (g < a.total_tiles) {
      job = 0;
      while (job + 1 < a.num_jobs && s_jobs[job + 1].tile_base <= g) ++job;
      const int it = g - s_jobs[job].tile_base;          // column-major upper triangle: it = tj (tj + 1) / 2 + ti
      tj = (int)((sqrtf(8.0f * (float)it + 1.0f) - 1.0f) * 0.5f);
      while (tj * (tj + 1) / 2 > it) --tj;
      while ((tj + 1) * (tj + 2) / 2 <= it) ++tj;
      ti = it - tj * (tj + 1) / 2;
    }
    s_job[threadIdx.x] = job;
    s_ti[threadIdx.x] = ti;
    s_tj[threadIdx.x] = tj;
  }
  // ---- phase D: pi-adjusted dampings (kfac.cu dampings_kernel), one warp per layer
  for (int l = cta; l < a.num_layers && threadIdx.x < 32; l += G) {
    const int lane = threadIdx.x;
    const float* pa = a.a_ptrs[l];
    const float* pg = a.g_ptrs[l];
    const int da = a.a_dims[l], dg = a.g_dims[l];
    double ta = 0.0, tg = 0.0;
    for (int i = lane; i < da; i += 32) ta += (double)__ldcg(pa + (size_t)i * da + i);
    for (int i = lane; i < dg; i += 32) tg += (double)__ldcg(pg + (size_t)i * dg + i);
    ta = warp_sum_d(ta);
    tg = warp_sum_d(tg);
    if (lane == 0) {
      ta /= (double)da;
      tg /= (double)dg;
      const double pi = (ta > 0.0 && tg > 0.0) ? sqrt(ta / tg) : 1.0;
      const double root = sqrt((double)a.lambdas[l]);
      a.damp[2 * l] = (float)(pi * root);
      a.damp[2 * l + 1] = (float)(root / pi);
    }
  }
  grid_arrive(a.bar, epoch);
  if (!grid_wait(a.bar, epoch)) return;
  // ---- phase P: owners load their tiles (M = debias * sym(S) + damp * I); look-ahead CTA j: D_0^-1 of job j
  const float debias = a.sched->debias;
  if (owner) {
    for (int s = 0; s < a.slots; ++s) {
      const int job = s_job[s];
      if (job < 0) continue;
      const ResJob& jb = s_jobs[job];
      const int ti = s_ti[s], tj = s_tj[s];
      const float dv = __ldcg(a.damp + jb.damp_index);
      float* T = tiles + (size_t)s * TILE_FLOATS;
      for (int e0 = threadIdx.x; e0 < TILE_FLOATS; e0 += 4 * RES_THREADS) {
        float pv[4];   // four pairs of loads in flight before the first shared-memory store
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int e = e0 + c * RES_THREADS;
          const int gi = ti * TS + (e >> 6), gj = tj * TS + (e & 63);
          pv[c] = (gi < jb.n && gj < jb.n) ? prep_value(jb, gi, gj, debias, dv) : 0.0f;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) T[e0 + c * RES_THREADS] = pv[c];
      }
      __syncthreads();
      publish_pair(jb, 0, ti, tj, T);     // blocks (0, 1) and (1, 1) for the look-ahead of step 0
    }
  } else {
    const ResJob& jb = s_jobs[cta];
    const int nb = min(RB, jb.n);
    const float dv = __ldcg(a.damp + jb.damp_index);
    for (int e = threadIdx.x; e < RB * RB; e += RES_THREADS) {
      const int y = e >> 5, x = e & 31;
      Ds[y][x] = (y < nb && x < nb) ? prep_value(jb, y, x, debias, dv) : (y == x ? 1.0f : 0.0f);
    }
    invert32(Ds, tiles + 3 * RB * (RB + 1));
    float* dinv = sc_dinv(jb, 0);
    for (int e = threadIdx.x; e < RB * RB; e += RES_THREADS) __stcg(dinv + e, Ds[e >> 5][e & 31]);
  }
  grid_arrive(a.bar, epoch);
  if (!grid_wait(a.bar, epoch)) return;
  // ---- pivot steps
  for (int p = 0; p < a.steps; ++p) {
    const int p0 = p * RB;
    if (!owner) {
      // look-ahead CTA of job `cta`: D_{p+1}^-1 from D_p^-1 (still in Ds) and the blocks published during step p - 1
      const ResJob& jb = s_jobs[cta];
      const bool tr = a.trace == 1 && p < 128 && cta == 0 && threadIdx.x == 0;
      if (tr) g_res_trace[p * 8 + 5] = clock64();
      // barrier 1 of this step: nothing here depends on the panels, so arrive at once - but the counter is cumulative, so
      // this CTA must not arrive at barrier 2 before barrier 1 has completed (its arrival would be counted for barrier 1)
      grid_arrive(a.bar, epoch);
      const unsigned int epoch_b1 = epoch;
      const int nblk = (jb.n + RB - 1) / RB;
      if (jb.n > p0 && p + 1 < nblk) {
        float (*Ps)[RB + 1] = reinterpret_cast<float (*)[RB + 1]>(tiles);
        float (*Qs)[RB + 1] = Ps + RB;
        float (*Rs)[RB + 1] = Qs + RB;
        const float* pq = sc_pq(jb, p);
        const float* qq = sc_qq(jb, p);
        const int x = threadIdx.x & 31, w = threadIdx.x >> 5;
        {
          float pr[4], qr[4];   // eight loads in flight
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            pr[c] = __ldcg(pq + threadIdx.x + c * RES_THREADS);
            qr[c] = __ldcg(qq + threadIdx.x + c * RES_THREADS);
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            Ps[w + 8 * c][x] = pr[c];
            Qs[w + 8 * c][x] = qr[c];
          }
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 4; ++c) {   // R_q = D_p^-1 M_pq
          const int y = w + 8 * c;
          float acc = 0.0f;
#pragma unroll 8
          for (int m = 0; m < RB; ++m) acc = fmaf(Ds[y][m], Ps[m][x], acc);
          Rs[y][x] = acc;
        }
        __syncthreads();
        float v[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {   // D' = M_qq - M_pq^T R_q  (padding: M_pq columns are zero, M_qq is identity)
          const int y = w + 8 * c;
          float acc = Qs[y][x];
#pragma unroll 8
          for (int k = 0; k < RB; ++k) acc = fmaf(-Ps[k][y], Rs[k][x], acc);
          v[c] = acc;
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 4; ++c) Ds[w + 8 * c][x] = v[c];
        invert32(Ds, tiles + 3 * RB * (RB + 1));
        float* dinv = sc_dinv(jb, p + 1);
        for (int e = threadIdx.x; e < RB * RB; e += RES_THREADS) __stcg(dinv + e, Ds[e >> 5][e & 31]);
      }
      if (tr) g_res_trace[p * 8 + 6] = clock64();
      if (!grid_wait(a.bar, epoch_b1)) return;
      grid_arrive(a.bar, epoch);          // barrier 2
      if (!grid_wait(a.bar, epoch)) return;
      if (tr) g_res_trace[p * 8 + 7] = clock64();
      continue;
    }
    const bool tr = a.trace && p < 128 && cta == (a.trace == 2 ? ND : G - 1) && threadIdx.x == 0;
    const bool tr2 = tr && a.trace == 2;   // first tile of the step: [5] operands staged [6] tile updated [7] published
    if (tr) g_res_trace[p * 8 + 0] = clock64();
    // panels
    for (int s = 0; s < a.slots; ++s) {
      const int job = s_job[s];
      if (job < 0 || s_jobs[job].n <= p0) continue;
      const int nblk = (s_jobs[job].n + RB - 1) / RB;
      if (nblk < 2) continue;
      panel_piece(s_jobs[job], p, s_ti[s], s_tj[s], tiles + (size_t)s * TILE_FLOATS, As, Bs, Ds);
    }
    if (tr) g_res_trace[p * 8 + 1] = clock64();
    grid_arrive(a.bar, epoch);
    if (!grid_wait(a.bar, epoch)) return;
    if (tr) g_res_trace[p * 8 + 2] = clock64();
    // update (operands of the next tile are fetched while the current one is computed)
    auto next_active = [&](int from) {
      while (from < a.slots && (s_job[from] < 0 || s_jobs[s_job[from]].n <= p0)) ++from;
      return from;
    };
    int s = next_active(0);
    const int first = s;
    OpRegs regs;
    if (s < a.slots) fetch_ops(s_jobs[s_job[s]], p, s_ti[s], s_tj[s], regs);
    while (s < a.slots) {
      const ResJob& jb = s_jobs[s_job[s]];
      const int ti = s_ti[s], tj = s_tj[s];
      float* T = tiles + (size_t)s * TILE_FLOATS;
      __syncthreads();                 // the previous tile is done with the staging buffers
      stage_ops(regs, As, Bs, Cs, tj == (p >> 1) && ti != tj);
      __syncthreads();
      if (tr2 && s == first) g_res_trace[p * 8 + 5] = clock64();
      const int sn = next_active(s + 1);
      if (sn < a.slots) fetch_ops(s_jobs[s_job[sn]], p, s_ti[sn], s_tj[sn], regs);
      update_tile(jb, p, ti, tj, T, As, Bs, Cs);
      if (tr2 && s == first) g_res_trace[p * 8 + 6] = clock64();
      __syncthreads();
      publish_pair(jb, p + 1, ti, tj, T);    // for the look-ahead of step p + 1
      if (tr2 && s == first) g_res_trace[p * 8 + 7] = clock64();
      s = sn;
    }
    if (tr) g_res_trace[p * 8 + 3] = clock64();
    grid_arrive(a.bar, epoch);
    if (!grid_wait(a.bar, epoch)) return;
    if (tr) g_res_trace[p * 8 + 4] = clock64();
  }
  // ---- phase F
  if (owner) {
    for (int s = 0; s < a.slots; ++s) {
      const int job = s_job[s];
      if (job < 0) continue;
      finish_tile(s_jobs[job], s_ti[s], s_tj[s], tiles + (size_t)s * TILE_FLOATS, stage);
    }
  }
}

}  // namespace

int inv_resident_error_flag() {
  int v = 0;
  cudaMemcpyFromSymbol(&v, g_res_error, sizeof(int));
  return v;
}
int inv_resident_trace_read(long long* h_out, int count) {
  if (count > 128 * 8) count = 128 * 8;
  return cudaMemcpyFromSymbol(h_out, g_res_trace, (size_t)count * sizeof(long long)) == cudaSuccess ? 0 : 1;
}

// returns 0 on success, -1 if the problem does not fit this kernel (the caller then uses the fp64 kernel chain), > 0 on error
int spd_inverse_resident(const InvJob* h_jobs, int num_jobs, const Sched* sched, float* d_damp, const float* const* d_a_ptrs,
                         const float* const* d_g_ptrs, const int* d_a_dims, const int* d_g_dims, const float* d_lambda,
                         int num_layers, unsigned int* d_bar, cudaStream_t st) {
  if (num_jobs > RES_JOBS || num_jobs < 1 || num_layers > 6) return -1;
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    ACX_CUDA(cudaGetDevice(&dev));
    ACX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int grid = sms;
  if (grid < num_jobs + 8) return -1;
  ResArgs a;
  int nmax = 0, total = 0;
  for (int i = 0; i < num_jobs; ++i) {
    ResJob& jb = a.jobs[i];
    const InvJob& hj = h_jobs[i];
    jb.s = hj.s;
    jb.n = hj.n;
    jb.damp_index = hj.damp_index;
    jb.x = reinterpret_cast<float*>(hj.work_x);
    jb.inv = hj.inv;
    for (int q = 0; q < 3; ++q) jb.planes[q] = hj.planes[q];
    jb.ld_planes = hj.ld_planes;
    jb.nt = ceil_div(hj.n, TS);
    jb.ldp = (hj.n + 3) & ~3;
    jb.tile_base = total;
    total += jb.nt * (jb.nt + 1) / 2;
    nmax = hj.n > nmax ? hj.n : nmax;
  }
  for (int i = num_jobs; i < RES_JOBS; ++i) a.jobs[i] = a.jobs[0];
  const int owners = grid - num_jobs;
  int slots = ceil_div(total, owners);
  if (slots < 2) slots = 2;   // the look-ahead CTAs use the tile area for five 32 x 33 blocks
  const size_t smem = ((size_t)STAGE_FLOATS + (size_t)slots * TILE_FLOATS) * sizeof(float);
  static int dyn_limit = -1;
  if (dyn_limit < 0) {
    cudaFuncAttributes fa;
    ACX_CUDA(cudaFuncGetAttributes(&fa, inv_resident_kernel));
    dyn_limit = RES_SMEM_TOTAL - (int)fa.sharedSizeBytes;   // the ownership / job tables are static shared memory
    ACX_CUDA(cudaFuncSetAttribute(inv_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit));
  }
  if (slots > 16 || smem > (size_t)dyn_limit) return -1;
  a.num_jobs = num_jobs;
  a.steps = ceil_div(nmax, RB);
  a.slots = slots;
  a.total_tiles = total;
  a.sched = sched;
  a.damp = d_damp;
  a.a_ptrs = d_a_ptrs;
  a.g_ptrs = d_g_ptrs;
  a.a_dims = d_a_dims;
  a.g_dims = d_g_dims;
  a.lambdas = d_lambda;
  a.num_layers = num_layers;
  a.bar = d_bar;
  {
    static int tr = -1;
    if (tr < 0) {
      const char* e = getenv("ACX_INV_TRACE");
      tr = e ? atoi(e) : 0;
    }
    a.trace = tr;
  }
  ACX_CUDA(cudaMemsetAsync(d_bar, 0, sizeof(unsigned int), st));
  inv_resident_kernel<<<grid, RES_THREADS, smem, st>>>(a);
  ACX_LAUNCH_CHECK();
  return 0;
}

}  // namespace acx
