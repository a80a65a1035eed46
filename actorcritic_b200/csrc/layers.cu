// layers.cu - the non-GEMM kernels of the Nature-CNN forward/backward and the A2C objective:
// im2col (uint8 -> bf16 and bf16 -> bf16), col2im + ReLU mask + bf16 split, policy/value heads
// forward, categorical log-prob / entropy / value loss + output gradients (true loss and Fisher sample),
// heads backward, column sums, weight preparation.  Reference semantics: envs/atari/model.py:92-127,
// 173-217, nn.py:37-52,88-110, policies.py:86-89,144, objectives.py:128-154,78 (SURVEY A.4/A.5).
#include "layers.cuh"

namespace acx {

// ------------------------------------------------------------------------------------------------
// im2col for conv1: obs uint8 [R,84,84,4] -> P1 bf16 [R*400, 256] holding the RAW byte values
// (exact in bf16; the 1/255 of envs/atari/model.py:93 is folded into the GEMM alpha).
// One thread per 16 output bytes: (patch row, ky, quarter q) reads 8 contiguous input bytes and writes 8 bf16, so a
// warp writes 512 contiguous bytes per store instruction (whole sectors) and reads 32-byte runs.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) im2col_conv1_kernel(const uint8_t* __restrict__ obs, bf16* __restrict__ out,
                                                           int rows_total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)rows_total * 32) return;
  const int q = (int)(i & 3);
  const int ky = (int)(i >> 2) & 7;
  const int row = (int)(i >> 5);
  const int n = row / 400, loc = row - n * 400, oy = loc / 20, ox = loc - oy * 20;
  const uint8_t* src = obs + ((size_t)(n * 84 + oy * 4 + ky) * 84 + ox * 4) * 4 + q * 8;
  const uint2 a = __ldg(reinterpret_cast<const uint2*>(src));
  const uint32_t w[2] = {a.x, a.y};
  // byte -> bf16 without the conversion unit: PRMT builds the float 2^23 + y (0x4B000000 | y), one FADD removes the
  // 2^23, and the upper halves of two such floats (exact: y has 8 significant bits) are the packed bf16 pair
  uint32_t t[4];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const float f0 = __uint_as_float(__byte_perm(w[j], 0x4B000000u, 0x7540)) - 8388608.0f;
    const float f1 = __uint_as_float(__byte_perm(w[j], 0x4B000000u, 0x7541)) - 8388608.0f;
    const float f2 = __uint_as_float(__byte_perm(w[j], 0x4B000000u, 0x7542)) - 8388608.0f;
    const float f3 = __uint_as_float(__byte_perm(w[j], 0x4B000000u, 0x7543)) - 8388608.0f;
    t[2 * j] = __byte_perm(__float_as_uint(f0), __float_as_uint(f1), 0x7632);
    t[2 * j + 1] = __byte_perm(__float_as_uint(f2), __float_as_uint(f3), 0x7632);
  }
  *reinterpret_cast<uint4*>(out + (size_t)row * 256 + ky * 32 + q * 8) = make_uint4(t[0], t[1], t[2], t[3]);
}

// Row-pair interleaved bf16 copy of the observations: uint8 [R, 84, 84, 4] -> bf16 [R, 42, 84, 2, 4] with
// out[r][p][x][q][c] = obs[r][2p + q][x][c] (raw byte values, exact).  In this layout the two kernel rows kh = 2j, 2j + 1 of
// conv1's 8x8 / stride-4 patch at output location (oy, ox) are ONE contiguous run of 64 elements (128 bytes) starting at
// pair-row 2 oy + j, pixel 4 ox - so the patch matrix P1 (envs/atari/model.py:173-179, 227-229) never has to exist: every
// GEMM that consumed it reads 64-column chunks with TMA box loads from this copy, which is 2x the observations instead of
// 7.2x and stays in L2.  The columns of a chunk arrive in the order (kw, q, c) instead of (kh, kw, c): see perm64 (gemm.cu).
// One thread per (sample, pair-row, 4 pixels): two 16-byte loads, four 16-byte stores (64 contiguous bytes).
__global__ void __launch_bounds__(256) obs_pairs_bf16_kernel(const uint8_t* __restrict__ obs, bf16* __restrict__ out, int samples) {
  pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)samples * 42 * 21) return;
  const int xq = (int)(i % 21);
  const long long rp = i / 21;   // sample * 42 + pair-row
  const int pr = (int)(rp % 42);
  const long long r = rp / 42;
  const uint8_t* src = obs + ((size_t)(r * 84 + 2 * pr) * 84 + 4 * xq) * 4;
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(src));             // row 2p:     4 pixels x 4 channels
  const uint4 b = __ldg(reinterpret_cast<const uint4*>(src + 84 * 4));    // row 2p + 1
  const uint32_t wa[4] = {a.x, a.y, a.z, a.w}, wb[4] = {b.x, b.y, b.z, b.w};
  uint4* dst = reinterpret_cast<uint4*>(out + ((size_t)rp * 84 + 4 * xq) * 8);
#pragma unroll
  for (int px = 0; px < 4; ++px) {
    uint32_t t[4];
    const uint32_t w2[2] = {wa[px], wb[px]};
#pragma unroll
    for (int q = 0; q < 2; ++q) {   // byte -> bf16 as in im2col_conv1_kernel
      const float f0 = __uint_as_float(__byte_perm(w2[q], 0x4B000000u, 0x7540)) - 8388608.0f;
      const float f1 = __uint_as_float(__byte_perm(w2[q], 0x4B000000u, 0x7541)) - 8388608.0f;
      const float f2 = __uint_as_float(__byte_perm(w2[q], 0x4B000000u, 0x7542)) - 8388608.0f;
      const float f3 = __uint_as_float(__byte_perm(w2[q], 0x4B000000u, 0x7543)) - 8388608.0f;
      t[2 * q] = __byte_perm(__float_as_uint(f0), __float_as_uint(f1), 0x7632);
      t[2 * q + 1] = __byte_perm(__float_as_uint(f2), __float_as_uint(f3), 0x7632);
    }
    dst[px] = make_uint4(t[0], t[1], t[2], t[3]);
  }
}

// generic NHWC bf16 im2col, patch order (ky, kx, c): each (row, ky) segment is k*C contiguous elements.
// One warp per patch row (grid-stride): the row decode is warp-uniform, lanes own 16-byte vectors, every plane is
// copied by the same thread (the index math is shared), reads are k*C*2-byte runs, writes are whole contiguous rows.
__global__ void __launch_bounds__(256) im2col_bf16_kernel(const Planes pin, const Planes pout, int rows_total, int hw_in, int c,
                                                          int k, int s, int hw_out) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int seg_vec = k * c / 8;        // uint4 per (row, ky) segment
  const int row_vec = k * seg_vec;      // uint4 per patch row
  const int per = hw_out * hw_out;
  const int np = pin.n < pout.n ? pin.n : pout.n;
  for (int row = warp; row < rows_total; row += nwarps) {
    const int n = row / per, loc = row - n * per, oy = loc / hw_out, ox = loc - oy * hw_out;
    const size_t src_base = ((size_t)(n * hw_in + oy * s) * hw_in + ox * s) * c;
    const size_t dst_base = (size_t)row * (k * k * c);
    for (int v = lane; v < row_vec; v += 32) {
      const int ky = v / seg_vec, off = v - ky * seg_vec;
      const size_t src = src_base + (size_t)ky * hw_in * c + (size_t)off * 8;
      const size_t dst = dst_base + (size_t)v * 8;
      const uint4 q0 = __ldg(reinterpret_cast<const uint4*>(pin.p[0] + src));
      uint4 q1, q2;
      if (np > 1) q1 = __ldg(reinterpret_cast<const uint4*>(pin.p[1] + src));
      if (np > 2) q2 = __ldg(reinterpret_cast<const uint4*>(pin.p[2] + src));
      *reinterpret_cast<uint4*>(pout.p[0] + dst) = q0;
      if (np > 1) *reinterpret_cast<uint4*>(pout.p[1] + dst) = q1;
      if (np > 2) *reinterpret_cast<uint4*>(pout.p[2] + dst) = q2;
    }
  }
}

// observation im2col for any NHWC geometry: obs [rows / (hw_out^2), hw_in, hw_in, c] (uint8 or fp32) -> patch planes
// [rows, ld] in the order (ky, kx, c), columns k*k*c .. ld-1 zero.  uint8 observations are written as their raw byte
// values on one plane (exact in bf16; the caller folds the 1/255 into its GEMM alpha and factor scales), fp32 observations
// as the hi / mid (/ lo) split over the output's planes.  One thread per output element (grid-stride).
template <typename T>
__global__ void __launch_bounds__(256) im2col_obs_kernel(const T* __restrict__ obs, const Planes out, long long rows, int hw_in,
                                                         int c, int k, int s, int hw_out) {
  pdl_enter();
  const int kc = k * c, kkc = k * kc, per = hw_out * hw_out;
  const long long total = rows * out.ld;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / out.ld;
    const int col = (int)(i - row * out.ld);
    float v = 0.0f;
    if (col < kkc) {
      const long long n = row / per;
      const int loc = (int)(row - n * per), oy = loc / hw_out, ox = loc - oy * hw_out;
      const int ky = col / kc, rem = col - ky * kc, kx = rem / c, ci = rem - kx * c;
      v = (float)__ldg(obs + ((size_t)(n * hw_in + oy * s + ky) * hw_in + ox * s + kx) * c + ci);
    }
    bf16 hi, mid, lo;
    split3(v, hi, mid, lo);
    out.p[0][i] = hi;
    if (out.n > 1) out.p[1][i] = mid;
    if (out.n > 2) out.p[2][i] = lo;
  }
}

// col2im (adjoint of im2col) as a gather + ReLU mask + bf16 split:
//   dX[n,y,x,c] = sum_{ky,kx : (y-ky)%s==0, (x-kx)%s==0, in range} dP[(n,oy,ox), (ky,kx,c)]
//   dPre[n,y,x,c] = dX * 1[act(n % mask_n, y, x, c) > 0]       (true rows and Fisher rows share the mask)
// blockIdx.x = (sample, input row y); a thread owns (x, 4 channels), so the only integer division is per CTA.  A row of more
// than 256 such threads is spread over gridDim.y CTAs; every element is summed in the same order either way.
__global__ void __launch_bounds__(256) col2im_mask_split_kernel(const float* __restrict__ dp, const bf16* __restrict__ act_hi,
                                                                const Planes out, int n_begin, int mask_n, int hw_in, int c, int k,
                                                                int s, int hw_out) {
  // dp holds the patch gradients of samples [n_begin, n_begin + gridDim.x / hw_in) only; outputs and masks are indexed by
  // the global sample number
  const int cv = c >> 2;
  const int n = blockIdx.x / hw_in, y = blockIdx.x - n * hw_in;
  const int t = blockIdx.y * blockDim.x + threadIdx.x;
  const int x = t / cv, c4 = (t - x * cv) << 2;
  if (x >= hw_in) return;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const int kkc = k * k * c;
  const float* base = dp + (size_t)n * hw_out * hw_out * kkc + c4;
  for (int ky = y % s; ky < k && ky <= y; ky += s) {
    const int oy = (y - ky) / s;
    if (oy >= hw_out) continue;
    for (int kx = x % s; kx < k && kx <= x; kx += s) {
      const int ox = (x - kx) / s;
      if (ox >= hw_out) continue;
      const float4 v = __ldg(reinterpret_cast<const float4*>(base + (size_t)(oy * hw_out + ox) * kkc + (ky * k + kx) * c));
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
  }
  const int ng = n + n_begin;
  const size_t pix = ((size_t)((ng % mask_n) * hw_in + y) * hw_in + x) * c + c4;
  const size_t opix = ((size_t)(ng * hw_in + y) * hw_in + x) * c + c4;
  const uint2 mw = *reinterpret_cast<const uint2*>(act_hi + pix);   // 4 bf16 of the forward activation (ReLU mask)
  const float vals[4] = {__uint_as_float(mw.x << 16) > 0.0f ? acc.x : 0.0f, __uint_as_float(mw.x & 0xffff0000u) > 0.0f ? acc.y : 0.0f,
                         __uint_as_float(mw.y << 16) > 0.0f ? acc.z : 0.0f, __uint_as_float(mw.y & 0xffff0000u) > 0.0f ? acc.w : 0.0f};
  __align__(8) bf16 hi[4], mid[4], lo[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) split3(vals[j], hi[j], mid[j], lo[j]);
  *reinterpret_cast<uint2*>(out.p[0] + opix) = *reinterpret_cast<const uint2*>(hi);
  if (out.n > 1) *reinterpret_cast<uint2*>(out.p[1] + opix) = *reinterpret_cast<const uint2*>(mid);
  if (out.n > 2) *reinterpret_cast<uint2*>(out.p[2] + opix) = *reinterpret_cast<const uint2*>(lo);
}

// ------------------------------------------------------------------------------------------------
// heads forward: act4 planes [R,512] x W_pol [512,A], W_val [512,1] (+ biases) -> logits [R,A], values [R]
// (envs/atari/model.py:207-216).  One warp per row.
// ------------------------------------------------------------------------------------------------
__global__ void heads_fwd_kernel(const Planes act4, const float* __restrict__ vpol, const float* __restrict__ vval, int rows,
                                 int num_actions, float* __restrict__ logits, float* __restrict__ values) {
  pdl_enter();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float x[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const size_t idx = (size_t)row * 512 + lane + 32 * j;
    float v = __bfloat162float(act4.p[0][idx]);
    if (act4.n > 1) v += __bfloat162float(act4.p[1][idx]);
    if (act4.n > 2) v += __bfloat162float(act4.p[2][idx]);
    x[j] = v;
  }
  if (num_actions == 4 && ((uintptr_t)vpol & 15) == 0) {
    // 4 actions (Breakout, a2c_acktr.py): the policy weights of one input are one 16-byte vector, and the five dot
    // products / butterfly reductions run as independent chains (per output the summation order is that of the loop below)
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int k = lane + 32 * j;
      const float4 w = __ldg(reinterpret_cast<const float4*>(vpol) + k);
      const float wv = __ldg(vval + k);
      acc[0] = fmaf(x[j], w.x, acc[0]);
      acc[1] = fmaf(x[j], w.y, acc[1]);
      acc[2] = fmaf(x[j], w.z, acc[2]);
      acc[3] = fmaf(x[j], w.w, acc[3]);
      acc[4] = fmaf(x[j], wv, acc[4]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int u = 0; u < 5; ++u) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], o);
    if (lane == 0) {
#pragma unroll
      for (int u = 0; u < 4; ++u) logits[(size_t)row * 4 + u] = acc[u] + vpol[(size_t)512 * 4 + u];
      values[row] = acc[4] + vval[512];
    }
    return;
  }
  for (int a = 0; a <= num_actions; ++a) {
    const float* w = a < num_actions ? vpol + a : vval;
    const int ld = a < num_actions ? num_actions : 1;
    float acc = 0.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) acc = fmaf(x[j], __ldg(w + (size_t)(lane + 32 * j) * ld), acc);
    acc = warp_sum(acc);
    if (lane == 0) {
      if (a < num_actions)
        logits[(size_t)row * num_actions + a] = acc + vpol[(size_t)512 * num_actions + a];
      else
        values[row] = acc + vval[512];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (counter-based RNG) for on-device Fisher sampling / action sampling
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// ------------------------------------------------------------------------------------------------
// A2C objective + output gradients (objectives.py:128-154,78; closed forms of SURVEY A.4) and the
// Fisher-sample output gradients (SURVEY A.5).  dheads is [2N, A+1]: rows [0,N) = d(shared loss)/d(logits|value),
// rows [N,2N) = d(L_sample)/d(logits|value).  One CTA; each thread strides over rows; deterministic
// block reduction for the three scalars.  inv_count = 1/N_global_rows_per_rank (the means are per rank;
// data-parallel ranks average them afterwards).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) loss_grad_kernel(const float* __restrict__ logits, const float* __restrict__ values,
                                                        const uint8_t* __restrict__ actions, const float* __restrict__ targets,
                                                        const int32_t* __restrict__ fisher_labels,
                                                        const float* __restrict__ fisher_eps, uint64_t seed,
                                                        const Sched* __restrict__ sched, int n_rows, int num_actions, float beta, float value_weight,
                                                        float policy_weight, float* __restrict__ dheads, float* __restrict__ scalars,
                                                        int want_fisher, const float* __restrict__ rewards,
                                                        const uint8_t* __restrict__ terminals, const float* __restrict__ bootstrap,
                                                        float gamma, int num_envs, int num_steps, float* __restrict__ targets_out,
                                                        float* __restrict__ adv_out) {
  pdl_enter();
  __shared__ float red[3][32];
  if (rewards) {
    // K-RET inside this (single-CTA) kernel: the n-step returns of objectives.py:178-214 - the same fp32 recursion as
    // returns_kernel, one thread per environment - are written to `targets` before anybody reads them (one launch less on
    // the critical path between the forward and the backward pass)
    for (int e = threadIdx.x; e < num_envs; e += blockDim.x) {
      float run = bootstrap[e];
      const size_t base = (size_t)e * num_steps;
      for (int t = num_steps - 1; t >= 0; --t) {
        if (terminals[base + t]) run = 0.0f;
        run = __fadd_rn(rewards[base + t], __fmul_rn(gamma, run));
        targets_out[base + t] = run;
        if (adv_out) adv_out[base + t] = run - values[base + t];
      }
    }
    __syncthreads();
  }
  const uint64_t step = sched ? sched->gs : 0ull;
  float s_obj = 0.f, s_ent = 0.f, s_val = 0.f;
  const float inv_n = 1.0f / (float)n_rows;
  const int ld = num_actions + 1;
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) {
    const float* z = logits + (size_t)r * num_actions;
    float mx = z[0];
    for (int a = 1; a < num_actions; ++a) mx = fmaxf(mx, z[a]);
    float se = 0.f;
    for (int a = 0; a < num_actions; ++a) se += expf(z[a] - mx);
    const float lse = logf(se) + mx;
    float ent = 0.f;
    for (int a = 0; a < num_actions; ++a) {
      const float lp = z[a] - lse;
      ent -= expf(lp) * lp;
    }
    const int act = actions[r];
    const float v = values[r], tg = rewards ? targets_out[r] : targets[r];
    const float adv = tg - v;
    const float logp_a = z[act] - lse;
    s_obj += adv * logp_a;
    s_ent += ent;
    s_val += 0.5f * (tg - v) * (tg - v);
    // Fisher sample
    int yhat = 0;
    float eps = 0.f;
    if (want_fisher) {
      if (fisher_labels) {
        yhat = fisher_labels[r];
        eps = fisher_eps[r];
      } else {
        const uint4 rnd = philox4x32(make_uint4((uint32_t)r, (uint32_t)step, (uint32_t)(step >> 32), 0x46495348u),
                                     make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const float u = u01(rnd.x);
        float cum = 0.f;
        yhat = num_actions - 1;
        for (int a = 0; a < num_actions; ++a) {
          cum += expf(z[a] - lse);
          if (u < cum) {
            yhat = a;
            break;
          }
        }
        eps = sqrtf(-2.0f * logf(u01(rnd.y))) * cospif(2.0f * u01(rnd.z));
      }
    }
    float* d_true = dheads + (size_t)r * ld;
    float* d_fish = dheads + (size_t)(n_rows + r) * ld;
    for (int a = 0; a < num_actions; ++a) {
      const float lp = z[a] - lse;
      const float p = expf(lp);
      const float dz = -(adv * inv_n) * ((a == act ? 1.0f : 0.0f) - p) + (beta * inv_n) * p * (lp + ent);
      d_true[a] = policy_weight == 1.0f ? dz : policy_weight * dz;   // objectives.py:31-54: the policy loss on its own / switched off
      if (want_fisher) d_fish[a] = p - (a == yhat ? 1.0f : 0.0f);
    }
    d_true[num_actions] = -value_weight * (tg - v) * inv_n;
    if (want_fisher) d_fish[num_actions] = -eps;
  }
  s_obj = warp_sum(s_obj);
  s_ent = warp_sum(s_ent);
  s_val = warp_sum(s_val);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    red[0][warp] = s_obj;
    red[1][warp] = s_ent;
    red[2][warp] = s_val;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float o = 0.f, e = 0.f, vl = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      o += red[0][w];
      e += red[1][w];
      vl += red[2][w];
    }
    const float mean_ent = e * inv_n;
    scalars[0] = -(o * inv_n + beta * mean_ent);  // policy_loss   objectives.py:145-149
    scalars[1] = vl * inv_n;                       // baseline_loss objectives.py:154
    scalars[2] = mean_ent;                         // mean_entropy  objectives.py:138-139
    scalars[3] = scalars[0] + value_weight * scalars[1];
  }
}

// ------------------------------------------------------------------------------------------------
// heads backward.  (a) dPre4[r, j] = (sum_a dH[r,a] W_pol[j,a] + dH[r,A] W_val[j]) * 1[act4[r % N, j] > 0] -> planes
// ------------------------------------------------------------------------------------------------
__global__ void heads_bwd_data_kernel(const float* __restrict__ dheads, const float* __restrict__ vpol,
                                      const float* __restrict__ vval, const bf16* __restrict__ act4_hi, int rows, int mask_rows,
                                      int num_actions, const Planes out) {
  pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)rows * 512) return;
  const int j = (int)(i & 511), r = (int)(i >> 9);
  const float* d = dheads + (size_t)r * (num_actions + 1);
  float acc = d[num_actions] * __ldg(vval + j);
  for (int a = 0; a < num_actions; ++a) acc = fmaf(d[a], __ldg(vpol + (size_t)j * num_actions + a), acc);
  const float m = __bfloat162float(act4_hi[(size_t)(r % mask_rows) * 512 + j]);
  if (!(m > 0.0f)) acc = 0.0f;
  bf16 hi, mid, lo;
  split3(acc, hi, mid, lo);
  out.p[0][i] = hi;
  if (out.n > 1) out.p[1][i] = mid;
  if (out.n > 2) out.p[2][i] = lo;
}

// (b) weight gradients of the two heads from the TRUE-loss rows: g_pol[j,a] = sum_n act4[n,j] dH[n,a]
// (j = 512 is the bias row: sum_n dH[n,a]); same for the value head.  One CTA per j, 128 threads over n.
__global__ void __launch_bounds__(128) heads_wgrad_kernel(const float* __restrict__ dheads, const Planes act4, int n_rows,
                                                          int num_actions, float* __restrict__ gpol, float* __restrict__ gval) {
  pdl_enter();
  __shared__ float red[4][32];
  const int j = blockIdx.x;  // 0..512
  const int ld = num_actions + 1;
  float acc[32];
#pragma unroll
  for (int a = 0; a < 32; ++a) acc[a] = 0.f;
  for (int n = threadIdx.x; n < n_rows; n += blockDim.x) {
    float x = 1.0f;
    if (j < 512) {
      const size_t idx = (size_t)n * 512 + j;
      x = __bfloat162float(act4.p[0][idx]);
      if (act4.n > 1) x += __bfloat162float(act4.p[1][idx]);
      if (act4.n > 2) x += __bfloat162float(act4.p[2][idx]);
    }
    const float* d = dheads + (size_t)n * ld;
#pragma unroll
    for (int a = 0; a < 32; ++a)
      if (a < ld) acc[a] = fmaf(x, d[a], acc[a]);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int a = 0; a < 32; ++a) {
    if (a < ld) {
      const float v = warp_sum(acc[a]);
      if (lane == 0) red[warp][a] = v;
    }
  }
  __syncthreads();
  if (threadIdx.x < ld) {
    const int a = threadIdx.x;
    const float v = red[0][a] + red[1][a] + red[2][a] + red[3][a];
    if (a < num_actions)
      gpol[(size_t)j * num_actions + a] = v;
    else
      gval[j] = v;
  }
}

// (c) output factors of the heads from the FISHER rows: G_pol = dz^T dz / N [A,A], G_val = dv^T dv / N [1,1]
__global__ void __launch_bounds__(256) heads_gfactor_kernel(const float* __restrict__ dheads_fisher, int n_rows, int num_actions,
                                                            float* __restrict__ g_pol, float* __restrict__ g_val) {
  pdl_enter();
  __shared__ float red[8];
  const int ld = num_actions + 1;
  const int pair = blockIdx.x;  // 0 .. A*A (last = value)
  const int a = pair < num_actions * num_actions ? pair / num_actions : num_actions;
  const int b = pair < num_actions * num_actions ? pair % num_actions : num_actions;
  float acc = 0.f;
  for (int n = threadIdx.x; n < n_rows; n += blockDim.x) acc = fmaf(dheads_fisher[(size_t)n * ld + a], dheads_fisher[(size_t)n * ld + b], acc);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float v = 0.f;
    for (int w = 0; w < 8; ++w) v += red[w];
    v /= (float)n_rows;
    if (pair < num_actions * num_actions)
      g_pol[pair] = v;
    else
      g_val[0] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// column sums of a planes matrix over rows [0, rows): two deterministic stages.
// stage 1: each CTA owns a contiguous chunk of rows; a thread owns one 8-column vector (one 16-byte load per plane
//          and row) and a row lane, so a warp reads whole 512-byte row segments; row lanes are combined through
//          shared memory in a fixed order.  partial[chunk][cols].
// stage 2: sums the chunks (8 chunk lanes per column) and scales.
// ------------------------------------------------------------------------------------------------
constexpr int CS_THREADS = 256;
constexpr int CS_COLBLOCK = CS_THREADS * 8;   // columns per CTA (one 8-column vector per thread)

__device__ __forceinline__ void add8(float* acc, const uint4 q) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    acc[2 * i] += __uint_as_float(w[i] << 16);            // low half = even element (bf16 -> fp32 is a 16-bit shift)
    acc[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
  }
}

// grid (row chunks, column blocks of 2048)
__global__ void __launch_bounds__(CS_THREADS) colsum_stage1_kernel(const Planes x, int rows, int cols, int rows_per_chunk,
                                                                   float* __restrict__ partial) {
  pdl_enter();
  extern __shared__ float cs_smem[];   // [lanes_r][cb]
  const int col0 = blockIdx.y * CS_COLBLOCK;
  const int cb = min(CS_COLBLOCK, cols - col0);
  const int nv = cb >> 3;
  const int lanes_r = nv >= CS_THREADS ? 1 : CS_THREADS / nv;
  const int row_lane = nv >= CS_THREADS ? 0 : threadIdx.x / nv;
  const int v = nv >= CS_THREADS ? threadIdx.x : threadIdx.x % nv;
  const bool active = row_lane < lanes_r && v < nv;
  const int r0 = blockIdx.x * rows_per_chunk;
  const int r1 = min(rows, r0 + rows_per_chunk);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  if (active) {
    // two rows (up to six 16-byte loads) in flight per thread: the loads are independent, the adds are not
    int r = r0 + row_lane;
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    for (; r + lanes_r < r1; r += 2 * lanes_r) {
      const size_t i0 = (size_t)r * x.ld + col0 + (size_t)v * 8;
      const size_t i1 = i0 + (size_t)lanes_r * x.ld;
      const uint4 q00 = __ldg(reinterpret_cast<const uint4*>(x.p[0] + i0));
      const uint4 q10 = __ldg(reinterpret_cast<const uint4*>(x.p[0] + i1));
      const uint4 q01 = x.n > 1 ? __ldg(reinterpret_cast<const uint4*>(x.p[1] + i0)) : z;
      const uint4 q11 = x.n > 1 ? __ldg(reinterpret_cast<const uint4*>(x.p[1] + i1)) : z;
      const uint4 q02 = x.n > 2 ? __ldg(reinterpret_cast<const uint4*>(x.p[2] + i0)) : z;
      const uint4 q12 = x.n > 2 ? __ldg(reinterpret_cast<const uint4*>(x.p[2] + i1)) : z;
      add8(acc, q00);
      add8(acc, q01);
      add8(acc, q02);
      add8(acc, q10);
      add8(acc, q11);
      add8(acc, q12);
    }
    for (; r < r1; r += lanes_r) {
      const size_t idx = (size_t)r * x.ld + col0 + (size_t)v * 8;
      add8(acc, __ldg(reinterpret_cast<const uint4*>(x.p[0] + idx)));
      if (x.n > 1) add8(acc, __ldg(reinterpret_cast<const uint4*>(x.p[1] + idx)));
      if (x.n > 2) add8(acc, __ldg(reinterpret_cast<const uint4*>(x.p[2] + idx)));
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) cs_smem[(size_t)row_lane * cb + v * 8 + i] = acc[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < cb; c += CS_THREADS) {
    float t = 0.f;
    for (int l = 0; l < lanes_r; ++l) t += cs_smem[(size_t)l * cb + c];
    partial[(size_t)blockIdx.x * cols + col0 + c] = t;
  }
}

// uint8 [rows, cols] -> per-chunk column sums (exact in uint32, stored as fp32: sums stay below 2^24 for <= 65793 rows
// per chunk); one 16-byte vector per thread.  grid (row chunks, ceil(cols / 4096))
__global__ void __launch_bounds__(256) colsum_u8_kernel(const uint8_t* __restrict__ x, int rows, int cols, int rows_per_chunk,
                                                        float* __restrict__ partial) {
  pdl_enter();
  const int c0 = (blockIdx.y * 256 + threadIdx.x) * 16;
  if (c0 >= cols) return;
  const int r0 = blockIdx.x * rows_per_chunk;
  const int r1 = min(rows, r0 + rows_per_chunk);
  uint32_t acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0u;
  for (int r = r0; r < r1; ++r) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(x + (size_t)r * cols + c0));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[4 * i + b] += (w[i] >> (8 * b)) & 0xffu;
  }
  float* dst = partial + (size_t)blockIdx.x * cols + c0;
#pragma unroll
  for (int i = 0; i < 16; ++i) dst[i] = (float)acc[i];
}

// border of a conv input factor from the batch-summed input S [hw_in, hw_in, c]:
//   out[(ky*k + kx)*c + ch] = scale * sum_{oy,ox} S[(oy*s + ky), (ox*s + kx), ch]      (= P^T 1 without touching P)
// one warp per output element, lanes over the output locations
__global__ void __launch_bounds__(256) window_sum_kernel(const float* __restrict__ sum_in, int hw_in, int c, int k, int s,
                                                         int hw_out, float scale, float* __restrict__ a, int d) {
  pdl_enter();
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= k * k * c) return;
  const int ch = i % c, kx = (i / c) % k, ky = i / (c * k);
  float acc = 0.f;
  for (int loc = lane; loc < hw_out * hw_out; loc += 32) {
    const int oy = loc / hw_out, ox = loc - oy * hw_out;
    acc += sum_in[((size_t)(oy * s + ky) * hw_in + ox * s + kx) * c + ch];
  }
  acc = warp_sum(acc);
  if (lane == 0) {   // straight into the factor: column d-1, row d-1, and the corner (the constant 1 of [P 1]^T [P 1] / rows)
    a[(size_t)i * d + (d - 1)] = acc * scale;
    a[(size_t)(d - 1) * d + i] = acc * scale;
    if (i == 0) a[(size_t)d * d - 1] = 1.0f;
  }
}

// block (32 columns, LANES chunk lanes): every lane sums its chunks with four independent accumulators (the loads of a
// lane are independent - without them one launch-latency-sized L2 round trip per chunk bounds this kernel), then the
// lanes are combined through shared memory in a fixed order.  LANES = 8 for wide vectors, 32 for the narrow ones (bias
// gradients: 32..64 columns over up to 592 chunks, where the grid is only 1-2 CTAs).
template <int LANES>
__global__ void __launch_bounds__(32 * LANES) colsum_stage2_kernel(const float* __restrict__ partial, int chunks, int cols, float scale,
                                                                   float* __restrict__ out, int out_stride, float* __restrict__ out2,
                                                                   int out2_stride, float* __restrict__ corner) {
  pdl_enter();
  __shared__ float red[LANES][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (c < cols) {
    const float* src = partial + c;
    int k = threadIdx.y;
    for (; k + 3 * LANES < chunks; k += 4 * LANES) {
      a0 += src[(size_t)k * cols];
      a1 += src[(size_t)(k + LANES) * cols];
      a2 += src[(size_t)(k + 2 * LANES) * cols];
      a3 += src[(size_t)(k + 3 * LANES) * cols];
    }
    for (; k < chunks; k += LANES) a0 += src[(size_t)k * cols];
  }
  red[threadIdx.y][threadIdx.x] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < LANES; ++k) t += red[k][threadIdx.x];
    out[(size_t)c * out_stride] = t * scale;
    if (out2) out2[(size_t)c * out2_stride] = t * scale;   // homogeneous border: the same vector as a row and as a column
    if (corner && c == 0) *corner = 1.0f;
  }
}

static int launch_colsum_stage2(const float* partial, int chunks, int cols, float scale, float* out, int out_stride, float* out2,
                                int out2_stride, float* corner, cudaStream_t st) {
  if (cols <= 128 && chunks >= 64) {
    ACX_PDL_LAUNCH((colsum_stage2_kernel<32>), ceil_div(cols, 32), dim3(32, 32), 0, st, partial, chunks, cols, scale, out, out_stride, out2,
                   out2_stride, corner);
  } else {
    ACX_PDL_LAUNCH((colsum_stage2_kernel<8>), ceil_div(cols, 32), dim3(32, 8), 0, st, partial, chunks, cols, scale, out, out_stride, out2,
                   out2_stride, corner);
  }
  return 0;
}

// fp32 [K, C] (row-major, the V-layout weight rows) -> transposed bf16 planes [C, ld_out]
__global__ void transpose_split_kernel(const float* __restrict__ in, int k_rows, int c_cols, bf16* __restrict__ p0,
                                       bf16* __restrict__ p1, bf16* __restrict__ p2, int num_planes, int ld_out) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int k = k0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (k < k_rows && c < c_cols) ? in[(size_t)k * c_cols + c] : 0.0f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, k = k0 + threadIdx.x;
    if (c < c_cols && k < ld_out) {
      bf16 a, b, d;
      split3(k < k_rows ? tile[threadIdx.x][i] : 0.0f, a, b, d);
      const size_t idx = (size_t)c * ld_out + k;
      p0[idx] = a;
      if (num_planes > 1) p1[idx] = b;
      if (num_planes > 2) p2[idx] = d;
    }
  }
}

// all GEMM operand planes of the trunk weights in ONE launch: for layer l (grid.z) a 32 x 32 tile of W_l [K, C] is read
// once and written as W^T planes [C, ldT] (forward B operand) and, if requested, as W planes [K, ldN] (dgrad B operand)
struct WeightPlanesJob {
  const float* w;          // [K, C] fp32 (the weight rows of V_l)
  int k_rows, c_cols;
  bf16* t[3];              // W^T planes [C, ld_t]
  int ld_t;
  bf16* n[3];              // W planes [K, ld_n] or null
  int ld_n;
  int perm_t;              // W^T columns in the (kw, row parity, c) order of the row-pair observation copy (conv1)
};
struct WeightPlanesArgs {
  WeightPlanesJob job[4];
};
__global__ void weight_planes_kernel(const WeightPlanesArgs a) {
  pdl_enter();
  const WeightPlanesJob& jb = a.job[blockIdx.z];
  const int k0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  if (k0 >= jb.ld_t || c0 >= jb.c_cols) return;
  __shared__ float tile[32][33];
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int k = k0 + i, c = c0 + threadIdx.x;
    const float v = (k < jb.k_rows && c < jb.c_cols) ? jb.w[(size_t)k * jb.c_cols + c] : 0.0f;
    tile[i][threadIdx.x] = v;
    if (jb.n[0] != nullptr && k < jb.k_rows && c < jb.ld_n) {
      bf16 x, y, z;
      split3(v, x, y, z);
      const size_t idx = (size_t)k * jb.ld_n + c;
      jb.n[0][idx] = x;
      jb.n[1][idx] = y;
      jb.n[2][idx] = z;
    }
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, k = k0 + threadIdx.x;
    if (c < jb.c_cols && k < jb.ld_t) {
      bf16 x, y, z;
      split3(k < jb.k_rows ? tile[threadIdx.x][i] : 0.0f, x, y, z);
      // perm_t: weight row f = p*32 + kw*4 + ch of a 64-row chunk goes to column kw*8 + p*4 + ch (the inverse of perm64)
      const int kd = jb.perm_t ? ((k & ~63) | (((k >> 2) & 7) << 3) | (((k >> 5) & 1) << 2) | (k & 3)) : k;
      const size_t idx = (size_t)c * jb.ld_t + kd;
      jb.t[0][idx] = x;
      jb.t[1][idx] = y;
      jb.t[2][idx] = z;
    }
  }
}

// categorical sample (inverse CDF on softmax(logits)) or argmax  (policies.py:86-87)
__global__ void __launch_bounds__(1024) sample_actions_kernel(const float* __restrict__ logits, const float* __restrict__ uniform,
                                                             uint64_t seed, uint64_t step, unsigned long long* step_counter,
                                                             int rows, int num_actions, int greedy,
                                                             int32_t* __restrict__ actions) {
  pdl_enter();
  // one CTA (rows are looped): with a device-resident call counter the Philox step is read from it and advanced here, so
  // a captured CUDA graph of an acting step stays valid from call to call
  if (step_counter) step = *step_counter;
  for (int r = threadIdx.x; r < rows; r += blockDim.x) {
    const float* z = logits + (size_t)r * num_actions;
    float mx = z[0];
    int arg = 0;
    for (int a = 1; a < num_actions; ++a)
      if (z[a] > mx) {
        mx = z[a];
        arg = a;
      }
    if (greedy) {
      actions[r] = arg;
      continue;
    }
    float se = 0.f;
    for (int a = 0; a < num_actions; ++a) se += expf(z[a] - mx);
    float u;
    if (uniform)
      u = uniform[r];
    else
      u = u01(philox4x32(make_uint4((uint32_t)r, (uint32_t)step, (uint32_t)(step >> 32), 0x41435421u),
                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)))
                  .x);
    float cum = 0.f;
    int pick = num_actions - 1;
    for (int a = 0; a < num_actions; ++a) {
      cum += expf(z[a] - mx) / se;
      if (u < cum) {
        pick = a;
        break;
      }
    }
    actions[r] = pick;
  }
  if (step_counter) {
    __syncthreads();
    if (threadIdx.x == 0) *step_counter = step + 1;
  }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
int im2col_conv1(const uint8_t* obs, bf16* out, int rows_total, cudaStream_t st) {
  const long long total = (long long)rows_total * 32;
  im2col_conv1_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(obs, out, rows_total);
  ACX_LAUNCH_CHECK();
  return 0;
}
int obs_pairs_bf16(const uint8_t* obs, bf16* out, int samples, cudaStream_t st) {
  const long long total = (long long)samples * 42 * 21;
  ACX_PDL_LAUNCH(obs_pairs_bf16_kernel, (unsigned)((total + 255) / 256), 256, 0, st, obs, out, samples);
  return 0;
}
int im2col_bf16(const Planes& in, const Planes& out, int rows_total, int hw_in, int c, int k, int s, int hw_out, cudaStream_t st) {
  int blocks = ceil_div(rows_total, 8);
  if (blocks > 148 * 8) blocks = 148 * 8;
  im2col_bf16_kernel<<<blocks, 256, 0, st>>>(in, out, rows_total, hw_in, c, k, s, hw_out);
  ACX_LAUNCH_CHECK();
  return 0;
}
int col2im_mask_split(const float* dp, const bf16* act_hi, const Planes& out, int n_begin, int n_total, int mask_n, int hw_in, int c,
                      int k, int s, int hw_out, cudaStream_t st) {
  ACX_CHECK((c & 3) == 0, "col2im: channels must be a multiple of 4");
  const int row_threads = hw_in * (c / 4);
  const int threads = row_threads <= 256 ? (row_threads + 31) / 32 * 32 : 256;
  const dim3 grid(n_total * hw_in, ceil_div(row_threads, threads));
  col2im_mask_split_kernel<<<grid, threads, 0, st>>>(dp, act_hi, out, n_begin, mask_n, hw_in, c, k, s, hw_out);
  ACX_LAUNCH_CHECK();
  return 0;
}
int im2col_obs(const void* obs, int obs_u8, const Planes& out, long long rows, int hw_in, int c, int k, int s, int hw_out,
               cudaStream_t st) {
  ACX_CHECK(out.ld >= k * k * c && (out.ld & 7) == 0, "im2col_obs: ld must be a multiple of 8 covering k*k*c");
  long long blocks = (rows * out.ld + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (obs_u8)
    ACX_PDL_LAUNCH(im2col_obs_kernel<uint8_t>, (unsigned)blocks, 256, 0, st, static_cast<const uint8_t*>(obs), out, rows, hw_in, c,
                   k, s, hw_out);
  else
    ACX_PDL_LAUNCH(im2col_obs_kernel<float>, (unsigned)blocks, 256, 0, st, static_cast<const float*>(obs), out, rows, hw_in, c, k,
                   s, hw_out);
  return 0;
}
int heads_fwd(const Planes& act4, const float* vpol, const float* vval, int rows, int num_actions, float* logits, float* values,
              cudaStream_t st) {
  ACX_PDL_LAUNCH(heads_fwd_kernel, ceil_div(rows, 8), 256, 0, st, act4, vpol, vval, rows, num_actions, logits, values);
  return 0;
}
// K-RET + K-LOSS in one launch: returns / advantages of the rollout (rewards, terminals [E, T]; bootstrap [E]) into
// targets_out / adv_out, then the A2C loss and its gradient with respect to the heads
struct ReturnsIn {
  const float* rewards = nullptr;
  const uint8_t* terminals = nullptr;
  const float* bootstrap = nullptr;
  float gamma = 0.0f;
  int num_envs = 0, num_steps = 0;
  float* targets_out = nullptr;
  float* adv_out = nullptr;
};
static int loss_grad_impl(const float* logits, const float* values, const uint8_t* actions, const float* targets, const int32_t* fl,
                          const float* fe, uint64_t seed, const Sched* sched, int n_rows, int num_actions, float beta, float vw,
                          float* dheads, float* scalars, int want_fisher, cudaStream_t st, float pw, const ReturnsIn& rt) {
  // one row per thread up to 1024 rows (the serial exp / log chains of a row are the kernel's latency)
  const int threads = n_rows >= 1024 ? 1024 : (n_rows + 31) / 32 * 32;
  ACX_PDL_LAUNCH(loss_grad_kernel, 1, threads, 0, st, logits, values, actions, targets, fl, fe, seed, sched, n_rows, num_actions, beta, vw, pw,
                 dheads, scalars, want_fisher, rt.rewards, rt.terminals, rt.bootstrap, rt.gamma, rt.num_envs, rt.num_steps, rt.targets_out,
                 rt.adv_out);
  return 0;
}
int loss_grad(const float* logits, const float* values, const uint8_t* actions, const float* targets, const int32_t* fl,
              const float* fe, uint64_t seed, const Sched* sched, int n_rows, int num_actions, float beta, float vw, float* dheads,
              float* scalars, int want_fisher, cudaStream_t st, float pw) {
  return loss_grad_impl(logits, values, actions, targets, fl, fe, seed, sched, n_rows, num_actions, beta, vw, dheads, scalars, want_fisher,
                        st, pw, ReturnsIn());
}
int returns_loss_grad(const float* rewards, const uint8_t* terminals, const float* bootstrap, float gamma, int num_envs, int num_steps,
                      float* targets, float* adv, const float* logits, const float* values, const uint8_t* actions, const int32_t* fl,
                      const float* fe, uint64_t seed, const Sched* sched, int num_actions, float beta, float vw, float* dheads,
                      float* scalars, int want_fisher, cudaStream_t st, float pw) {
  ReturnsIn rt;
  rt.rewards = rewards;
  rt.terminals = terminals;
  rt.bootstrap = bootstrap;
  rt.gamma = gamma;
  rt.num_envs = num_envs;
  rt.num_steps = num_steps;
  rt.targets_out = targets;
  rt.adv_out = adv;
  return loss_grad_impl(logits, values, actions, targets, fl, fe, seed, sched, num_envs * num_steps, num_actions, beta, vw, dheads, scalars,
                        want_fisher, st, pw, rt);
}
int heads_bwd(const float* dheads, const float* vpol, const float* vval, const Planes& act4, int n_rows, int rows_bwd,
              int num_actions, const Planes& dpre4, float* gpol, float* gval, cudaStream_t st) {
  const long long total = (long long)rows_bwd * 512;
  ACX_PDL_LAUNCH(heads_bwd_data_kernel, (unsigned)((total + 255) / 256), 256, 0, st, dheads, vpol, vval, act4.p[0], rows_bwd, n_rows, num_actions, dpre4);
  ACX_PDL_LAUNCH(heads_wgrad_kernel, 513, 128, 0, st, dheads, act4, n_rows, num_actions, gpol, gval);
  return 0;
}
int heads_gfactor(const float* dheads_fisher, int n_rows, int num_actions, float* g_pol, float* g_val, cudaStream_t st) {
  ACX_PDL_LAUNCH(heads_gfactor_kernel, num_actions * num_actions + 1, 256, 0, st, dheads_fisher, n_rows, num_actions, g_pol, g_val);
  return 0;
}
int colsum(const Planes& x, int rows, int cols, float scale, float* partial, int max_chunks, float* out, int out_stride,
           cudaStream_t st, float* out2, int out2_stride, float* corner) {
  ACX_CHECK((cols & 7) == 0 && (x.ld & 7) == 0, "colsum: cols and ld must be multiples of 8");
  const int cb = cols < CS_COLBLOCK ? cols : CS_COLBLOCK;
  const int nv = cb >> 3;
  const int lanes_r = nv >= CS_THREADS ? 1 : CS_THREADS / nv;
  int chunks = ceil_div(rows, lanes_r * 4);          // at least ~4 rows per lane
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  const int rpc = ceil_div(rows, chunks);
  chunks = ceil_div(rows, rpc);
  const size_t smem = (size_t)lanes_r * cb * sizeof(float);
  static bool configured = false;
  if (!configured) {
    ACX_CUDA(cudaFuncSetAttribute(colsum_stage1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    configured = true;
  }
  ACX_PDL_LAUNCH(colsum_stage1_kernel, dim3(chunks, ceil_div(cols, CS_COLBLOCK)), CS_THREADS, smem, st, x, rows, cols, rpc, partial);
  if (int r2 = launch_colsum_stage2(partial, chunks, cols, scale, out, out_stride, out2, out2_stride, corner, st)) return r2;
  return 0;
}

// batch sum of the conv input (uint8 observations or bf16-plane activations), then the window sums = border of A_l
int conv_border(const uint8_t* obs_u8, const Planes* act, int n_rows, int hw_in, int c, int k, int s, int hw_out, float scale,
                float* partial, int max_chunks, float* sum_tmp, float* a, int d, cudaStream_t st) {
  const int cols = hw_in * hw_in * c;
  if (obs_u8) {
    ACX_CHECK((cols & 15) == 0, "conv_border: cols must be a multiple of 16");
    int chunks = ceil_div(n_rows, 16);
    if (chunks > max_chunks) chunks = max_chunks;
    const int rpc = ceil_div(n_rows, chunks);
    chunks = ceil_div(n_rows, rpc);
    ACX_PDL_LAUNCH(colsum_u8_kernel, dim3(chunks, ceil_div(cols, 4096)), 256, 0, st, obs_u8, n_rows, cols, rpc, partial);
    if (int r2 = launch_colsum_stage2(partial, chunks, cols, 1.0f, sum_tmp, 1, nullptr, 0, nullptr, st)) return r2;
  } else {
    Planes v = *act;
    v.ld = cols;
    int r = colsum(v, n_rows, cols, 1.0f, partial, max_chunks, sum_tmp, 1, st, nullptr, 0, nullptr);
    if (r) return r;
  }
  ACX_PDL_LAUNCH(window_sum_kernel, ceil_div(k * k * c, 8), 256, 0, st, sum_tmp, hw_in, c, k, s, hw_out, scale, a, d);
  return 0;
}

int transpose_split(const float* in, int k_rows, int c_cols, bf16* p0, bf16* p1, bf16* p2, int num_planes, int ld_out,
                    cudaStream_t st) {
  dim3 grid(ceil_div(ld_out, 32), ceil_div(c_cols, 32));
  transpose_split_kernel<<<grid, dim3(32, 8), 0, st>>>(in, k_rows, c_cols, p0, p1, p2, num_planes, ld_out);
  ACX_LAUNCH_CHECK();
  return 0;
}
int weight_planes(const float* const* w, const int* k_rows, const int* c_cols, bf16* const (*t)[3], const int* ld_t,
                  bf16* const (*n)[3], const int* ld_n, int num_layers, cudaStream_t st, int perm_first) {
  ACX_CHECK(num_layers >= 1 && num_layers <= 4, "weight_planes: 1..4 layers");
  WeightPlanesArgs a;
  int max_k = 0, max_c = 0;
  for (int i = 0; i < 4; ++i) {
    const int s = i < num_layers ? i : 0;
    a.job[i].w = w[s];
    a.job[i].k_rows = k_rows[s];
    a.job[i].c_cols = c_cols[s];
    a.job[i].ld_t = ld_t[s];
    a.job[i].ld_n = ld_n[s];
    a.job[i].perm_t = (s == 0 && perm_first) ? 1 : 0;
    for (int q = 0; q < 3; ++q) {
      a.job[i].t[q] = t[s][q];
      a.job[i].n[q] = n[s][q];
    }
    if (i < num_layers) {
      max_k = ld_t[s] > max_k ? ld_t[s] : max_k;
      max_c = ld_n[s] > c_cols[s] ? (ld_n[s] > max_c ? ld_n[s] : max_c) : (c_cols[s] > max_c ? c_cols[s] : max_c);
    }
  }
  dim3 grid(ceil_div(max_k, 32), ceil_div(max_c, 32), num_layers);
  ACX_PDL_LAUNCH(weight_planes_kernel, grid, dim3(32, 8), 0, st, a);
  return 0;
}
int sample_actions(const float* logits, const float* uniform, uint64_t seed, uint64_t step, int rows, int num_actions, int greedy,
                   int32_t* actions, cudaStream_t st, unsigned long long* step_counter) {
  const int threads = rows >= 1024 ? 1024 : (rows + 31) / 32 * 32;
  ACX_PDL_LAUNCH(sample_actions_kernel, 1, threads, 0, st, logits, uniform, seed, step, step_counter, rows, num_actions, greedy, actions);
  return 0;
}

}  // namespace acx

extern "C" int acx_sample_actions(const float* d_logits, const float* d_uniform, uint64_t seed, uint64_t step, int rows,
                                  int num_actions, int greedy, int32_t* d_actions, void* stream) {
  ACX_CHECK(d_logits && d_actions, "null argument");
  ACX_CHECK(rows > 0 && num_actions >= 1 && num_actions <= 1024, "rows / num_actions out of range");
  return acx::sample_actions(d_logits, d_uniform, seed, step, rows, num_actions, greedy, d_actions,
                             reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int acx_obs_pairs_bf16(const uint8_t* d_obs, void* d_out, int samples, void* stream) {
  ACX_CHECK(d_obs && d_out && samples > 0, "null argument");
  ACX_CHECK((reinterpret_cast<uintptr_t>(d_obs) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_out) & 15) == 0, "16-byte alignment");
  return acx::obs_pairs_bf16(d_obs, reinterpret_cast<acx::bf16*>(d_out), samples, reinterpret_cast<cudaStream_t>(stream));
}
