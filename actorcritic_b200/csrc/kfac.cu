// kfac.cu - the K-FAC side of the ACKTR update that is not a GEMM: homogeneous border of the input
// factors, the moving average of the factor statistics, pi-adjusted damping from traces, the fp64 chain of
// damped SPD inverses, the <V,U> reduction for the KL clip and the fused clip + momentum + apply steps (K-FAC,
// cold momentum-SGD, RMSProp).  Semantics: SURVEY A.5 (tensorflow/kfac 0.1.x as driven by
// kfac_utils.py:38-53 with the hyper-parameters of a2c_acktr.py:240-251) and nn.py:185-189.
#include "layers.cuh"

namespace acx {

// ------------------------------------------------------------------------------------------------
// A = [[P^T P, P^T 1], [1^T P, rows]] / rows : the tensor-core SYRK fills the K x K block, this writes
// the border (column / row d-1) from the scaled column sums and the corner 1.
// ------------------------------------------------------------------------------------------------
__global__ void homog_border_kernel(float* __restrict__ a, int d, const float* __restrict__ cs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= d) return;
  const float v = i < d - 1 ? cs[i] : 1.0f;
  a[(size_t)i * d + (d - 1)] = v;
  a[(size_t)(d - 1) * d + i] = v;
}

// S <- decay * S + (1 - decay) * scale_c * C      (kfac MovingAverageVariable, cov_ema_decay)
__global__ void ema_kernel(float* __restrict__ s, const float* __restrict__ c, size_t count, float decay, float wc) {
  pdl_enter();
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t n4 = count / 4;
  float4* s4 = reinterpret_cast<float4*>(s);
  const float4* c4 = reinterpret_cast<const float4*>(c);
  for (size_t j = i; j < n4; j += stride) {
    float4 a = s4[j];
    const float4 b = c4[j];
    a.x = decay * a.x + wc * b.x;
    a.y = decay * a.y + wc * b.y;
    a.z = decay * a.z + wc * b.z;
    a.w = decay * a.w + wc * b.w;
    s4[j] = a;
  }
  for (size_t j = n4 * 4 + i; j < count; j += stride) s[j] = decay * s[j] + wc * c[j];
}

__global__ void fill_kernel(float* __restrict__ p, size_t count, float v) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) p[i] = v;
}
__global__ void scale_kernel(float* __restrict__ p, size_t count, float v) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) p[i] *= v;
}

// ------------------------------------------------------------------------------------------------
// pi-adjusted damping (SURVEY A.5 "Damping"): per block, from the traces of the running sums (the
// zero-debias factor is common to A and G and cancels in pi):
//   pi = sqrt((tr A / dim A) / (tr G / dim G)),  damp_A = pi * sqrt(lambda_l),  damp_G = sqrt(lambda_l) / pi
// One warp per block (layer); out[2*l] = damp_A, out[2*l+1] = damp_G.
// ------------------------------------------------------------------------------------------------
__global__ void dampings_kernel(const float* const* __restrict__ a_ptrs, const float* const* __restrict__ g_ptrs,
                                const int* __restrict__ a_dims, const int* __restrict__ g_dims,
                                const float* __restrict__ lambdas, int num_layers, float* __restrict__ out) {
  const int l = blockIdx.x;
  if (l >= num_layers) return;
  const int lane = threadIdx.x;
  const float* a = a_ptrs[l];
  const float* g = g_ptrs[l];
  const int da = a_dims[l], dg = g_dims[l];
  double ta = 0.0, tg = 0.0;
  for (int i = lane; i < da; i += 32) ta += (double)a[(size_t)i * da + i];
  for (int i = lane; i < dg; i += 32) tg += (double)g[(size_t)i * dg + i];
  ta = warp_sum_d(ta);
  tg = warp_sum_d(tg);
  if (lane == 0) {
    ta /= (double)da;
    tg /= (double)dg;
    const double pi = (ta > 0.0 && tg > 0.0) ? sqrt(ta / tg) : 1.0;
    const double root = sqrt((double)lambdas[l]);
    out[2 * l] = (float)(pi * root);
    out[2 * l + 1] = (float)(root / pi);
  }
}

// ------------------------------------------------------------------------------------------------
// Damped SPD inverse, batched over jobs (grid.z = job), fp64, blocked in-place Gauss-Jordan without
// pivoting (safe for SPD): for each 32-wide pivot block p
//   D^-1 = inv(M_pp);  R_j = D^-1 M_pj (j != p);  M_ij -= M_ip R_j (i, j != p);
//   M_ip = -M_ip D^-1 (i != p);  M_pj = R_j;  M_pp = D^-1.
// After the last block M holds the inverse.  2 n^3 flops; runs only every `invert_every` updates.
// This chain is the fallback of the fp32 refresh with the tiles resident in shared memory (kfac_inv.cu): it runs when
// those tiles do not fit the SMs (Atari conv3 > 64, wide fully connected layers).  The same fp64 arithmetic as one
// persistent kernel with grid barriers between the steps was measured at 1.84 ms per refresh on a B200 at 32 x 20, no
// faster than this chain, and was dropped (DESIGN.md section 4).
// ------------------------------------------------------------------------------------------------
constexpr int IB = 32;  // pivot block

struct InvDev {
  const float* s;
  int n;
  int damp_index;
  double* m;     // [n, n]
  double* rbuf;  // [IB, n] row panel R, then [IB, IB] D^-1 at rbuf + IB * n
  float* inv;
  bf16* planes[3];
  int ld_planes;
};

__global__ void inv_prepare_kernel(const InvDev* __restrict__ jobs, const Sched* __restrict__ sched,
                                   const float* __restrict__ damp) {
  const InvDev jb = jobs[blockIdx.z];
  const float debias = sched->debias;
  const size_t total = (size_t)jb.n * jb.n;
  const double dv = (double)damp[jb.damp_index];
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int r = (int)(i / jb.n), c = (int)(i % jb.n);
    // symmetrise while loading: the statistics are symmetric up to the rounding of the border writes
    const double v = 0.5 * ((double)jb.s[i] + (double)jb.s[(size_t)c * jb.n + r]) * (double)debias;
    jb.m[i] = r == c ? v + dv : v;
  }
}

// fp64 reciprocal from an fp32 seed and two Newton steps (relative error 2^-23 -> 2^-46 -> 2^-92, i.e. the fp64 rounding
// floor): a short dependent chain instead of the IEEE division sequence; pivots of the damped SPD factors are far inside
// the fp32 exponent range.  r (2 - x r) is written as r + r (1 - x r): one FMA each, residual computed exactly enough.
__device__ __forceinline__ double fast_rcp(double x) {
  double r = (double)__frcp_rn((float)x);
  r = fma(r, fma(-x, r, 1.0), r);
  r = fma(r, fma(-x, r, 1.0), r);
  return r;
}

// invert an IB x IB block held in shared memory, in place (unblocked Gauss-Jordan without pivoting; rows/columns >= nb
// are identity padding).  NT = threads of the CTA (all must call it); each owns IB*IB/NT elements, fully unrolled so
// the per-thread values stay in registers.
template <int NT>
__device__ __forceinline__ void invert_block_smem(double (*d)[IB + 1]) {
  constexpr int PER = IB * IB / NT;
  for (int k = 0; k < IB; ++k) {
    __syncthreads();
    const double inv_p = fast_rcp(d[k][k]);
    double v[PER];
#pragma unroll
    for (int c = 0; c < PER; ++c) {
      const int e = threadIdx.x + c * NT;
      const int ty = e >> 5, tx = e & 31;
      const double row_k = d[k][tx], col_k = d[ty][k];
      const double scaled = row_k * inv_p;
      double r = d[ty][tx] - col_k * scaled;
      if (ty == k) r = scaled;
      if (tx == k) r = -col_k * inv_p;
      if (ty == k && tx == k) r = inv_p;
      v[c] = r;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < PER; ++c) {
      const int e = threadIdx.x + c * NT;
      d[e >> 5][e & 31] = v[c];
    }
  }
  __syncthreads();
}

// per-job scratch inside InvDev::rbuf:  R [IB][n] | Rold [IB][n] | next pivot block before inversion ([IB][IB] of an
// [IB][n] slot; only jobs with n > IB have a next pivot) | Dinv [2][IB][IB] (by pivot parity: the update kernel of step p
// reads D_p^-1 while inv_pivot_kernel already writes D_{p+1}^-1)
__device__ __forceinline__ double* scratch_r(const InvDev& jb) { return jb.rbuf; }
__device__ __forceinline__ double* scratch_rold(const InvDev& jb) { return jb.rbuf + (size_t)IB * jb.n; }
__device__ __forceinline__ double* scratch_next(const InvDev& jb) { return jb.rbuf + (size_t)2 * IB * jb.n; }   // IB x IB
__device__ __forceinline__ double* scratch_dinv(const InvDev& jb, int p) {
  return jb.rbuf + (size_t)3 * IB * jb.n + (size_t)(p & 1) * IB * IB;
}

// D_0^-1 of every job (one CTA of 256 threads per job) - later pivot inverses come from inv_pivot_kernel
__global__ void __launch_bounds__(256) inv_diag0_kernel(const InvDev* __restrict__ jobs) {
  const InvDev jb = jobs[blockIdx.z];
  const int n = jb.n;
  __shared__ double d[IB][IB + 1];
  const int nb = min(IB, n);
  for (int e = threadIdx.x; e < IB * IB; e += 256) {
    const int ty = e >> 5, tx = e & 31;
    d[ty][tx] = (ty < nb && tx < nb) ? jb.m[(size_t)ty * n + tx] : (ty == tx ? 1.0 : 0.0);
  }
  invert_block_smem<256>(d);
  double* dinv = scratch_dinv(jb, 0);
  for (int e = threadIdx.x; e < IB * IB; e += 256) dinv[e] = d[e >> 5][e & 31];
}

// Symmetry.  For an SPD input the Gauss-Jordan iterates keep a signed symmetry: with S = the pivot blocks already
// processed (blocks < p, pivots go in order), M_ij = M_ji^T when i and j are both in S or both outside, and
// M_ij = -M_ji^T otherwise.  So only the upper 64 x 64 TILES (tile_i <= tile_j; diagonal tiles in full) are stored and
// updated - half the flops and half the CTAs of the full update - and everything a step needs follows from the true
// row panel  Rold_i = M_pi  (stored for tile(i) >= tile(p), else -M_ip^T)  and  R = D^-1 Rold:
//   M_ij -= sigma_i Rold_i^T R_j   (sigma_i = -1 for processed i, +1 otherwise; i, j != p)
//   M_pj  = R_j,   M_ip = -sigma_i R_i^T,   M_pp = D^-1.
//
// step kernel A (panels): one CTA (1024 threads = one 32 x 32 block) per block b != p: Rold_b and R_b = D^-1 Rold_b.
__global__ void __launch_bounds__(1024) inv_panels_kernel(const InvDev* __restrict__ jobs, int p, int nblk) {
  const InvDev jb = jobs[blockIdx.z];
  const int n = jb.n;
  const int p0 = p * IB;
  if (p0 >= n) return;
  const int blk = blockIdx.x;
  const int b0 = blk * IB;
  if (b0 >= n || blk == p) return;
  __shared__ double d[IB][IB + 1];
  __shared__ double t[IB][IB + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int nb = min(IB, n - p0);
  d[ty][tx] = scratch_dinv(jb, p)[ty * IB + tx];
  if ((b0 >> 6) >= (p0 >> 6)) {   // stored as a row of the pivot
    const int cj = b0 + tx;
    t[ty][tx] = (ty < nb && cj < n) ? jb.m[(size_t)(p0 + ty) * n + cj] : 0.0;
  } else {                        // only its mirror M_bp is stored (b processed, p not): M_pb = -M_bp^T
    const int gi = b0 + ty;
    t[tx][ty] = (gi < n && tx < nb) ? -jb.m[(size_t)gi * n + p0 + tx] : 0.0;
  }
  __syncthreads();
  const int cj = b0 + tx;
  double acc = 0.0;
#pragma unroll 8
  for (int k = 0; k < IB; ++k) acc += d[ty][k] * t[k][tx];
  if (cj < n) {
    scratch_rold(jb)[(size_t)ty * n + cj] = t[ty][tx];
    scratch_r(jb)[(size_t)ty * n + cj] = acc;
  }
  if (blk == p + 1) {
    // look-ahead: the next pivot block as this step's update will leave it, D' = M_qq - Rold_q^T R_q (q = p + 1 is not
    // processed yet: sigma = +1; same k order as the update kernel).  inv_pivot_kernel inverts it on a side stream
    // WHILE the update kernel runs, which takes the serial 32-step Gauss-Jordan off the critical path.
    __syncthreads();          // everyone is done reading d
    d[ty][tx] = acc;          // R_q
    __syncthreads();
    const int nbq = min(IB, n - b0);
    double v = (ty < nbq && tx < nbq) ? jb.m[(size_t)(b0 + ty) * n + b0 + tx] : (ty == tx ? 1.0 : 0.0);
    if (ty < nbq && tx < nbq) {
#pragma unroll 8
      for (int k = 0; k < IB; ++k) v -= t[k][ty] * d[k][tx];
    }
    scratch_next(jb)[ty * IB + tx] = v;
  }
}

// D_{p+1}^-1 from the block the panels kernel of step p left in scratch_next (one CTA of 256 threads per job)
__global__ void __launch_bounds__(256) inv_pivot_kernel(const InvDev* __restrict__ jobs, int q) {
  const InvDev jb = jobs[blockIdx.z];
  if (q * IB >= jb.n) return;
  __shared__ double d[IB][IB + 1];
  const double* src = scratch_next(jb);
  for (int e = threadIdx.x; e < IB * IB; e += 256) d[e >> 5][e & 31] = src[e];
  invert_block_smem<256>(d);
  double* out = scratch_dinv(jb, q);
  for (int e = threadIdx.x; e < IB * IB; e += 256) out[e] = d[e >> 5][e & 31];
}

// step kernel B (update) over the upper tiles, CTA tile 64 x 64, 256 threads, 4 x 4 per thread.  (The next pivot block
// is inverted concurrently by inv_pivot_kernel from the look-ahead copy the panels kernel made.)
__global__ void __launch_bounds__(256) inv_update_kernel(const InvDev* __restrict__ jobs, int p) {
  if (blockIdx.y > blockIdx.x) return;   // lower tiles are never read
  const InvDev jb = jobs[blockIdx.z];
  const int n = jb.n;
  const int p0 = p * IB;
  if (p0 >= n) return;
  const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
  if (i0 >= n || j0 >= n) return;
  __shared__ double cs[64][IB + 1];  // sigma_i Rold^T tile [64 rows][32]
  __shared__ double rs[IB][64 + 1];  // R tile [32][64 cols]
  const int nb = min(IB, n - p0);
  const double* rold = scratch_rold(jb);
  const double* rb = scratch_r(jb);
  {
    // issue every global load before the first shared-memory store
    double rc[8], rr[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int idx = threadIdx.x + 256 * q;
      const int k = idx / 64, c = idx % 64;
      const int gi = i0 + c, gj = j0 + c;
      const double v = (gi < n && k < nb && !(gi >= p0 && gi < p0 + IB)) ? rold[(size_t)k * n + gi] : 0.0;
      rc[q] = gi < p0 ? -v : v;
      rr[q] = (gj < n && k < nb && !(gj >= p0 && gj < p0 + IB)) ? rb[(size_t)k * n + gj] : 0.0;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int idx = threadIdx.x + 256 * q;
      cs[idx % 64][idx / 64] = rc[q];
      rs[idx / 64][idx % 64] = rr[q];
    }
  }
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  // the 16 matrix elements this thread updates are fetched up front (independent loads, overlapped with the math)
  double acc[4][4];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int gi = i0 + ty + 16 * q, gj = j0 + tx + 16 * r;
      acc[q][r] = (gi < n && gj < n) ? jb.m[(size_t)gi * n + gj] : 0.0;
    }
#pragma unroll 4
  for (int k = 0; k < IB; ++k) {
    double a[4], b[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      a[q] = cs[ty + 16 * q][k];
      b[q] = rs[k][tx + 16 * q];
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[q][r] -= a[q] * b[r];
  }
  const double* dinv = scratch_dinv(jb, p);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int gi = i0 + ty + 16 * q;
    if (gi >= n) continue;
    const bool ip = gi >= p0 && gi < p0 + IB;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int gj = j0 + tx + 16 * r;
      if (gj >= n) continue;
      const bool jp = gj >= p0 && gj < p0 + IB;
      double* dst = jb.m + (size_t)gi * n + gj;
      if (ip && jp)
        *dst = dinv[(gi - p0) * IB + (gj - p0)];
      else if (ip)
        *dst = rb[(size_t)(gi - p0) * n + gj];                 // M_pj = R_j
      else if (jp) {
        const double v = rb[(size_t)(gj - p0) * n + gi];       // M_ip = -sigma_i R_i^T
        *dst = gi < p0 ? v : -v;
      } else
        *dst = acc[q][r];
    }
  }
}

__global__ void inv_finish_kernel(const InvDev* __restrict__ jobs) {
  const InvDev jb = jobs[blockIdx.z];
  const int n = jb.n;
  const size_t total = (size_t)n * jb.ld_planes;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int r = (int)(i / jb.ld_planes), c = (int)(i % jb.ld_planes);
    float v = 0.0f;
    if (c < n) {
      // only the upper 64-tiles hold the inverse (diagonal tiles in full: average their two halves)
      const int tr = r >> 6, tc = c >> 6;
      const double up = tr <= tc ? jb.m[(size_t)r * n + c] : jb.m[(size_t)c * n + r];
      v = (float)(tr == tc ? 0.5 * (up + jb.m[(size_t)c * n + r]) : up);
      jb.inv[(size_t)r * n + c] = v;
    }
    bf16 p0, p1, p2;
    split3(v, p0, p1, p2);
    jb.planes[0][i] = p0;
    jb.planes[1][i] = p1;
    jb.planes[2][i] = p2;
  }
}

// ------------------------------------------------------------------------------------------------
// reductions and the fused optimiser steps
// ------------------------------------------------------------------------------------------------
// partial[b] = sum over the b-th contiguous chunk of a[i] * b[i]   (deterministic two-stage reduction)
__global__ void __launch_bounds__(256) dot_partial_kernel(const float* __restrict__ a, const float* __restrict__ b, size_t count,
                                                          float* __restrict__ partial) {
  pdl_enter();
  __shared__ double red[8];
  const size_t per = (count + gridDim.x - 1) / gridDim.x;
  const size_t i0 = (size_t)blockIdx.x * per;
  const size_t i1 = i0 + per < count ? i0 + per : count;
  // four independent accumulators: the loads of one thread do not wait for each other's DFMA
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  size_t i = i0 + threadIdx.x;
  for (; i + 768 < i1; i += 1024) {
    a0 += (double)a[i] * (double)b[i];
    a1 += (double)a[i + 256] * (double)b[i + 256];
    a2 += (double)a[i + 512] * (double)b[i + 512];
    a3 += (double)a[i + 768] * (double)b[i + 768];
  }
  for (; i < i1; i += 256) a0 += (double)a[i] * (double)b[i];
  double acc = (a0 + a1) + (a2 + a3);
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int w = 0; w < 8; ++w) v += red[w];
    partial[blockIdx.x] = (float)v;
  }
}

__device__ __forceinline__ float sum_partials(const float* partial, int num) {
  // every thread of the block needs the same scalar: warp 0 reduces in a fixed order, broadcast via smem
  __shared__ float total;
  if (threadIdx.x < 32) {
    double v = 0.0;
    for (int i = threadIdx.x; i < num; i += 32) v += (double)partial[i];
    v = warp_sum_d(v);
    if (threadIdx.x == 0) total = (float)v;
  }
  __syncthreads();
  return total;
}

// K-FAC: s = sum <V, U>; c = min(1, sqrt(kappa / (lr^2 s))); v <- mu v + c U; theta <- theta - lr v
// (kfac _clip_updates / _update_velocities / GradientDescentOptimizer, SURVEY A.5; a2c_acktr.py:245-246)
__global__ void __launch_bounds__(256) kfac_step_kernel(float* __restrict__ params, float* __restrict__ vel,
                                                        const float* __restrict__ precon, size_t count,
                                                        const float* __restrict__ partial, int num_partials,
                                                        const Sched* __restrict__ sched, float mu, float kappa,
                                                        float* __restrict__ out_scalars) {
  pdl_enter();
  const float lr = sched->lr;
  const float s = sum_partials(partial, num_partials);
  float c = 1.0f;
  if (s > 0.0f) c = fminf(1.0f, sqrtf(kappa / (lr * lr * s)));
  if (blockIdx.x == 0 && threadIdx.x == 0 && out_scalars) {
    out_scalars[0] = c;
    out_scalars[1] = s;
    out_scalars[3] = lr;
  }
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t tid0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t done = 0;
  if ((((uintptr_t)params | (uintptr_t)vel | (uintptr_t)precon) & 15) == 0) {   // 16-byte accesses for the bulk
    const size_t quads = count >> 2;
    float4* p4 = reinterpret_cast<float4*>(params);
    float4* v4 = reinterpret_cast<float4*>(vel);
    const float4* u4 = reinterpret_cast<const float4*>(precon);
    for (size_t i = tid0; i < quads; i += stride) {
      float4 v = v4[i], th = p4[i];
      const float4 u = u4[i];
      v.x = mu * v.x + c * u.x;
      v.y = mu * v.y + c * u.y;
      v.z = mu * v.z + c * u.z;
      v.w = mu * v.w + c * u.w;
      th.x -= lr * v.x;
      th.y -= lr * v.y;
      th.z -= lr * v.z;
      th.w -= lr * v.w;
      v4[i] = v;
      p4[i] = th;
    }
    done = quads << 2;
  }
  for (size_t i = done + tid0; i < count; i += stride) {
    const float v = mu * vel[i] + c * precon[i];
    vel[i] = v;
    params[i] -= lr * v;
  }
}

// ClipGlobalNormOptimizer(MomentumOptimizer): g <- g * clip / max(||g||, clip); acc <- mu acc + g; theta -= lr acc
// (nn.py:185-189, a2c_acktr.py:240-241)
__global__ void __launch_bounds__(256) momentum_clip_kernel(float* __restrict__ params, float* __restrict__ accum,
                                                            const float* __restrict__ grads, size_t count,
                                                            const float* __restrict__ partial, int num_partials, float lr,
                                                            float mu, float clip, float* __restrict__ out_scalars) {
  pdl_enter();
  const float sq = sum_partials(partial, num_partials);
  const float norm = sqrtf(sq);
  const float scale = clip / fmaxf(norm, clip);
  if (blockIdx.x == 0 && threadIdx.x == 0 && out_scalars) out_scalars[0] = norm;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    const float a = mu * accum[i] + grads[i] * scale;
    accum[i] = a;
    params[i] -= lr * a;
  }
}

// ClipGlobalNormOptimizer(RMSPropOptimizer) with the TF-1 defaults (decay 0.9, momentum 0, eps 1e-10, ms = 1 at start):
// ms <- d ms + (1-d) g^2; theta -= lr g / sqrt(ms + eps)     (a2c_acktr.py:250-251)
__global__ void __launch_bounds__(256) rmsprop_clip_kernel(float* __restrict__ params, float* __restrict__ ms,
                                                           const float* __restrict__ grads, size_t count,
                                                           const float* __restrict__ partial, int num_partials,
                                                           const Sched* __restrict__ sched, float decay, float eps, float clip,
                                                           float* __restrict__ out_scalars, float lr_value) {
  pdl_enter();
  const float lr = sched ? sched->lr : lr_value;
  const float sq = sum_partials(partial, num_partials);
  const float norm = sqrtf(sq);
  const float scale = clip / fmaxf(norm, clip);
  if (blockIdx.x == 0 && threadIdx.x == 0 && out_scalars) {
    out_scalars[0] = norm;
    out_scalars[1] = lr;
  }
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    const float g = grads[i] * scale;
    const float m = decay * ms[i] + (1.0f - decay) * g * g;
    ms[i] = m;
    params[i] -= lr * g / sqrtf(m + eps);
  }
}

// ------------------------------------------------------------------------------------------------
// Preconditioning of the small blocks (C <= 64 output channels: conv1..3 and the two heads) in fp32 SIMT, batched over
// blocks: U = A^-1 (V G^-1) / T~.  Two launches for all of them; only fc4 (1569 x 512) is worth the tensor cores.
// ------------------------------------------------------------------------------------------------
// W[r, c] = sum_k V[r, k] Ginv[k, c];  grid (ceil(d / 64), 1, jobs), 256 threads
__global__ void __launch_bounds__(256) precon_vg_kernel(const PreconJob* __restrict__ jobs) {
  pdl_enter();
  const PreconJob jb = jobs[blockIdx.z];
  const int d = jb.d, c = jb.c;
  const int r0 = blockIdx.x * 64;
  if (r0 >= d) return;
  __shared__ float gs[64][65];
  __shared__ float vs[64][65];
  {
    float rg[16], rv[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int i = threadIdx.x + 256 * q, k = i >> 6, j = i & 63;
      rg[q] = (k < c && j < c) ? __ldg(jb.ginv + (size_t)k * c + j) : 0.0f;
      rv[q] = (r0 + k < d && j < c) ? jb.v[(size_t)(r0 + k) * c + j] : 0.0f;
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int i = threadIdx.x + 256 * q;
      gs[i >> 6][i & 63] = rg[q];
      vs[i >> 6][i & 63] = rv[q];
    }
  }
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  for (int k = 0; k < c; ++k) {
    float a[4], b[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      a[q] = vs[ty + 16 * q][k];
      b[q] = gs[k][tx + 16 * q];
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[q][r] = fmaf(a[q], b[r], acc[q][r]);
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int r = r0 + ty + 16 * q;
    if (r >= d) continue;
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int col = tx + 16 * rr;
      if (col < c) jb.w[(size_t)r * c + col] = acc[q][rr];
    }
  }
}

// U[r, c] = scale * sum_k Ainv[r, k] W[k, c];  grid (ceil(d / 16), 1, jobs), 256 threads = 16 rows x 16 column lanes
// (4 columns each), k in chunks of 64
__global__ void __launch_bounds__(256) precon_aw_kernel(const PreconJob* __restrict__ jobs) {
  pdl_enter();
  const PreconJob jb = jobs[blockIdx.z];
  const int d = jb.d, c = jb.c;
  const int r0 = blockIdx.x * 16;
  if (r0 >= d) return;
  __shared__ float as[16][65];
  __shared__ float ws[64][65];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k0 = 0; k0 < d; k0 += 64) {
    // all global loads are issued before the first shared-memory store (otherwise each load -> store pair serialises)
    float ra[4], rw[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = threadIdx.x + 256 * q, r = i >> 6, k = i & 63;
      ra[q] = (r0 + r < d && k0 + k < d) ? __ldg(jb.ainv + (size_t)(r0 + r) * d + k0 + k) : 0.0f;
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int i = threadIdx.x + 256 * q, k = i >> 6, j = i & 63;
      rw[q] = (k0 + k < d && j < c) ? jb.w[(size_t)(k0 + k) * c + j] : 0.0f;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = threadIdx.x + 256 * q;
      as[i >> 6][i & 63] = ra[q];
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int i = threadIdx.x + 256 * q;
      ws[i >> 6][i & 63] = rw[q];
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < 64; ++k) {
      const float a = as[ty][k];
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q] = fmaf(a, ws[k][tx + 16 * q], acc[q]);
    }
    __syncthreads();
  }
  const int r = r0 + ty;
  if (r < d) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int col = tx + 16 * q;
      if (col < c) jb.u[(size_t)r * c + col] = acc[q] * jb.scale;
    }
  }
}

// schedule state (one thread)
__global__ void sched_begin_kernel(Sched* s, float lr_start, float lr_end, double decay_steps, float* out_lr) {
  pdl_enter();
  // nn.py:154-156 linear_decay = polynomial_decay(power 1, cycle False), evaluated at the step the update starts with
  double g = (double)s->gs;
  if (g > decay_steps) g = decay_steps;
  s->lr = (float)(((double)lr_start - (double)lr_end) * (1.0 - g / decay_steps) + (double)lr_end);
  if (out_lr) *out_lr = s->lr;
}
__global__ void sched_advance_kernel(Sched* s, int gs_inc, int ncov_inc, float ema_decay, int zero_debias) {
  pdl_enter();
  s->gs += (unsigned long long)gs_inc;
  s->ncov += (unsigned long long)ncov_inc;
  if (ncov_inc) {
    double d = 1.0;
    if (zero_debias && s->ncov > 0) d = 1.0 / (1.0 - pow((double)ema_decay, (double)s->ncov));
    s->debias = (float)d;
  }
}

// whole schedule transition of one phase-2 call in one launch: learning rate from the step the update starts with, then
// the counters (nothing later in the phase reads global_step; the inverse refresh reads the new debias factor)
__global__ void sched_step_kernel(Sched* s, float lr_start, float lr_end, double decay_steps, float* out_lr, int gs_inc,
                                  int ncov_inc, float ema_decay, int zero_debias) {
  pdl_enter();
  double g = (double)s->gs;
  if (g > decay_steps) g = decay_steps;
  s->lr = (float)(((double)lr_start - (double)lr_end) * (1.0 - g / decay_steps) + (double)lr_end);
  if (out_lr) *out_lr = s->lr;
  s->gs += (unsigned long long)gs_inc;
  s->ncov += (unsigned long long)ncov_inc;
  if (ncov_inc) {
    double d = 1.0;
    if (zero_debias && s->ncov > 0) d = 1.0 / (1.0 - pow((double)ema_decay, (double)s->ncov));
    s->debias = (float)d;
  }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
int sched_step(Sched* s, float lr_start, float lr_end, double decay_steps, float* out_lr, int gs_inc, int ncov_inc,
               float ema_decay, int zero_debias, cudaStream_t st) {
  ACX_PDL_LAUNCH(sched_step_kernel, 1, 1, 0, st, s, lr_start, lr_end, decay_steps, out_lr, gs_inc, ncov_inc, ema_decay, zero_debias);
  return 0;
}
int sched_begin(Sched* s, float lr_start, float lr_end, double decay_steps, float* out_lr, cudaStream_t st) {
  ACX_PDL_LAUNCH(sched_begin_kernel, 1, 1, 0, st, s, lr_start, lr_end, decay_steps, out_lr);
  return 0;
}
int sched_advance(Sched* s, int gs_inc, int ncov_inc, float ema_decay, int zero_debias, cudaStream_t st) {
  ACX_PDL_LAUNCH(sched_advance_kernel, 1, 1, 0, st, s, gs_inc, ncov_inc, ema_decay, zero_debias);
  return 0;
}

static int grid_for(size_t count, int threads, int max_blocks) {
  size_t b = (count + threads - 1) / threads;
  if (b > (size_t)max_blocks) b = max_blocks;
  if (b < 1) b = 1;
  return (int)b;
}

int homog_border(float* a, int d, const float* colsum_scaled, cudaStream_t st) {
  homog_border_kernel<<<ceil_div(d, 128), 128, 0, st>>>(a, d, colsum_scaled);
  ACX_LAUNCH_CHECK();
  return 0;
}
int ema_update(float* s, const float* c, size_t count, float decay, float scale_c, cudaStream_t st) {
  ACX_CHECK(((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(c)) & 15) == 0, "unaligned factor region");
  ACX_PDL_LAUNCH(ema_kernel, grid_for(count / 4 + 1, 256, 148 * 8), 256, 0, st, s, c, count, decay, (1.0f - decay) * scale_c);
  return 0;
}
int fill_f32(float* p, size_t count, float v, cudaStream_t st) {
  if (count == 0) return 0;
  fill_kernel<<<grid_for(count, 256, 148 * 8), 256, 0, st>>>(p, count, v);
  ACX_LAUNCH_CHECK();
  return 0;
}
int scale_f32(float* p, size_t count, float v, cudaStream_t st) {
  if (count == 0) return 0;
  scale_kernel<<<grid_for(count, 256, 148 * 8), 256, 0, st>>>(p, count, v);
  ACX_LAUNCH_CHECK();
  return 0;
}
int compute_dampings(const float* const* d_a_ptrs, const float* const* d_g_ptrs, const int* d_a_dims, const int* d_g_dims,
                     const float* d_lambda, int num_layers, float* d_damp, cudaStream_t st) {
  dampings_kernel<<<num_layers, 32, 0, st>>>(d_a_ptrs, d_g_ptrs, d_a_dims, d_g_dims, d_lambda, num_layers, d_damp);
  ACX_LAUNCH_CHECK();
  return 0;
}

int spd_inverse_batched(const InvJob* h_jobs, const InvJob* d_jobs, int num_jobs, const Sched* sched, const float* d_damp,
                        cudaStream_t st, cudaStream_t side) {
  // `side`: a second stream for the pivot-block inversions (forked after each panels kernel, joined before the next one;
  // inside a stream capture these become parallel graph branches).  nullptr or == st: everything in order on `st`.
  static cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  const bool forked = side != nullptr && side != st;
  if (forked && ev_fork == nullptr) {
    ACX_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    ACX_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
  }
  static_assert(sizeof(InvJob) == sizeof(InvDev), "InvJob and InvDev must have the same layout");
  const InvDev* dj = reinterpret_cast<const InvDev*>(d_jobs);
  int nmax = 0;
  for (int i = 0; i < num_jobs; ++i) nmax = h_jobs[i].n > nmax ? h_jobs[i].n : nmax;
  ACX_CHECK(nmax > 0, "no inverse jobs");
  {
    dim3 grid(grid_for((size_t)nmax * nmax, 256, 148 * 4), 1, num_jobs);
    inv_prepare_kernel<<<grid, 256, 0, st>>>(dj, sched, d_damp);
    ACX_LAUNCH_CHECK();
  }
  inv_diag0_kernel<<<dim3(1, 1, num_jobs), 256, 0, st>>>(dj);
  ACX_LAUNCH_CHECK();
  const int steps = ceil_div(nmax, IB);
  for (int p = 0; p < steps; ++p) {
    // jobs are sorted by decreasing n by the caller, so the jobs still active at step p are a prefix
    int active = 0;
    int nact = 0;
    for (int i = 0; i < num_jobs; ++i)
      if (h_jobs[i].n > p * IB) {
        active = i + 1;
        nact = h_jobs[i].n > nact ? h_jobs[i].n : nact;
      }
    if (active == 0) break;
    const int nblk = ceil_div(nact, IB);
    const bool has_next = nblk > p + 1;
    if (nblk > 1) {
      inv_panels_kernel<<<dim3(nblk, 1, active), 1024, 0, st>>>(dj, p, nblk);
      ACX_LAUNCH_CHECK();
    }
    if (has_next) {
      cudaStream_t ps = forked ? side : st;
      if (forked) {
        ACX_CUDA(cudaEventRecord(ev_fork, st));
        ACX_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
      }
      inv_pivot_kernel<<<dim3(1, 1, active), 256, 0, ps>>>(dj, p + 1);
      ACX_LAUNCH_CHECK();
      if (forked) ACX_CUDA(cudaEventRecord(ev_join, side));
    }
    inv_update_kernel<<<dim3(ceil_div(nact, 64), ceil_div(nact, 64), active), 256, 0, st>>>(dj, p);
    ACX_LAUNCH_CHECK();
    if (has_next && forked) ACX_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
  }
  {
    dim3 grid(grid_for((size_t)nmax * (nmax + 8), 256, 148 * 4), 1, num_jobs);
    inv_finish_kernel<<<grid, 256, 0, st>>>(dj);
    ACX_LAUNCH_CHECK();
  }
  return 0;
}

int precondition_small(const PreconJob* d_jobs, int num_jobs, int max_d, cudaStream_t st) {
  if (num_jobs == 0) return 0;
  dim3 grid(ceil_div(max_d, 64), 1, num_jobs);
  ACX_PDL_LAUNCH(precon_vg_kernel, grid, 256, 0, st, d_jobs);
  ACX_PDL_LAUNCH(precon_aw_kernel, dim3(ceil_div(max_d, 16), 1, num_jobs), 256, 0, st, d_jobs);
  return 0;
}

int dot_partial(const float* a, const float* b, size_t count, float* partial, int num_partials, cudaStream_t st) {
  ACX_PDL_LAUNCH(dot_partial_kernel, num_partials, 256, 0, st, a, b, count, partial);
  return 0;
}
int kfac_step(float* params, float* velocity, const float* precon, size_t count, const float* dot_partials, int num_partials,
              const Sched* sched, float momentum, float norm_constraint, float* out_scalars, cudaStream_t st) {
  ACX_PDL_LAUNCH(kfac_step_kernel, grid_for(count, 256, 148 * 4), 256, 0, st, params, velocity, precon, count, dot_partials, num_partials, sched, momentum, norm_constraint, out_scalars);
  return 0;
}
int momentum_clip_step(float* params, float* accum, const float* grads, size_t count, const float* sq_partials, int num_partials,
                       float lr, float momentum, float clip_norm, float* out_scalars, cudaStream_t st) {
  ACX_PDL_LAUNCH(momentum_clip_kernel, grid_for(count, 256, 148 * 4), 256, 0, st, params, accum, grads, count, sq_partials, num_partials, lr, momentum, clip_norm, out_scalars);
  return 0;
}
int rmsprop_clip_step(float* params, float* ms, const float* grads, size_t count, const float* sq_partials, int num_partials,
                      const Sched* sched, float decay, float epsilon, float clip_norm, float* out_scalars, cudaStream_t st,
                      float lr_value) {
  ACX_PDL_LAUNCH(rmsprop_clip_kernel, grid_for(count, 256, 148 * 4), 256, 0, st, params, ms, grads, count, sq_partials, num_partials, sched, decay, epsilon, clip_norm, out_scalars, lr_value);
  return 0;
}

}  // namespace acx

// ---- stand-alone optimizer steps (C ABI): what objectives.py:31-54 `optimize_separate` applies per loss -----------------
extern "C" {

static const int kStepPartials = 296;

// ClipGlobalNormOptimizer(RMSPropOptimizer(lr, decay, momentum 0, eps)).apply_gradients (nn.py:185-189, a2c_acktr.py:250-251)
int acx_clip_rmsprop_step(float* d_params, float* d_ms, const float* d_grads, size_t count, float lr, float decay, float epsilon,
                          float clip_norm, float* d_scratch, float* d_out_norm, void* stream) {
  ACX_CHECK(d_params && d_ms && d_grads && d_scratch && count > 0, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int r = acx::dot_partial(d_grads, d_grads, count, d_scratch, kStepPartials, st);
  if (r) return r;
  return acx::rmsprop_clip_step(d_params, d_ms, d_grads, count, d_scratch, kStepPartials, nullptr, decay, epsilon, clip_norm,
                                d_out_norm, st, lr);
}

// ClipGlobalNormOptimizer(MomentumOptimizer(lr, momentum)).apply_gradients (nn.py:185-189, a2c_acktr.py:240-241)
int acx_clip_momentum_step(float* d_params, float* d_accum, const float* d_grads, size_t count, float lr, float momentum,
                           float clip_norm, float* d_scratch, float* d_out_norm, void* stream) {
  ACX_CHECK(d_params && d_accum && d_grads && d_scratch && count > 0, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int r = acx::dot_partial(d_grads, d_grads, count, d_scratch, kStepPartials, st);
  if (r) return r;
  return acx::momentum_clip_step(d_params, d_accum, d_grads, count, d_scratch, kStepPartials, lr, momentum, clip_norm, d_out_norm,
                                 st);
}

}  // extern "C"

