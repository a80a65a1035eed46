// preprocess.cu - K-PRE: batched Atari frame preprocessing + frame stack, uint8, bit-exact with the
// reference's cv2 path.  One kernel fuses, per environment:
//   max of the last two raw frames      (wrappers.py:64-65)
//   RGB -> gray, 15-bit fixed point      (cv2.cvtColor, wrappers.py:31)
//   210x160 -> 84x84 INTER_AREA          (cv2.resize,  wrappers.py:32): separable fp32 taps, the
//                                        multiply and the add are separate roundings (no FMA), the
//                                        horizontal pass first, taps in table order, then
//                                        round-half-even + saturate
//   frame-stack push / zero-on-terminal / reset-to-4-copies (wrappers.py:224-235, multi_env.py:127-132)
//
// HBM traffic per env-step (the roofline numerator): 2*100800 B raw + 28224 B old stack + 28224 B new
// stack = 258048 B.  The stack is NHWC with 4 uint8 channels = one 32-bit word per pixel, so the push is
// (word >> 8) | (new << 24).
//
// Mapping: one CTA per (environment, band of 12 output rows); 7 bands -> grid = 7*E.  A band needs raw
// rows [30*band, 30*band+30) (y scale is exactly 2.5: output row d uses rows floor(2.5d)..+2, and 12
// output rows use exactly 30 source rows).  Phase 1: the CTA streams its 30 raw rows of both frames with
// 16-byte loads (a 480-byte row = 30 uint4), takes the max, converts to gray, and leaves the gray band
// in shared memory as bytes.  Phase 2: a thread owns an output column and 10 source rows: horizontal taps into
// registers, vertical taps of its 4 output rows, round + stack push with coalesced 32-bit stores.
//
// The end of the file holds the same work at any square output size S in [4, 128] and stack depth k in [1, 16]
// (preprocess_sq_kernel, framestack_sq_kernel; acx_*_sq_u8) for observations other than 84x84x4: tap tables of any
// length (CSR arrays, built once per size and device), a band of output rows per CTA whose raw rows are read once, the
// horizontal pass in shared memory, stacks [E,S,S,k] written with coalesced stores over the k bytes of each pixel.  At S
// = 5 and 10, where both scales are integers, cv2 averages blocks in integers instead (resizeAreaFast_); the kernel does
// the same.  84x84x4 keeps running through the K-PRE kernels above.
#include <algorithm>
#include <cfloat>
#include <map>
#include <mutex>
#include <vector>

#include "tc.cuh"

namespace acx {

constexpr int RAW_H = 210, RAW_W = 160, OUT = 84;
constexpr int BAND_OUT = 12, BAND_SRC = 30, NUM_BANDS = 7;
constexpr int RAW_ROW_BYTES = RAW_W * 3;        // 480
constexpr int RAW_FRAME_BYTES = RAW_H * RAW_ROW_BYTES;
constexpr int STACK_BYTES = OUT * OUT * 4;

struct Taps {
  int xsrc[OUT][3];
  float xw[OUT][3];
  int xn[OUT];
  int ysrc[OUT][3];
  float yw[OUT][3];
  int yn[OUT];
};
// the tap tables live in global memory and are read through the read-only path: constant memory serialises the
// per-lane indexed reads (measured: MIO-bound), the L1/texture path does not
__device__ Taps c_taps;
static bool g_taps_ready = false;

// OpenCV computeResizeAreaTab (resize.cpp), cn = 1; weights are computed in double and stored as float.
static void build_axis(int ssize, int dsize, int (*src)[3], float (*w)[3], int* cnt) {
  const double scale = (double)ssize / dsize;
  for (int d = 0; d < dsize; ++d) {
    cnt[d] = 0;
    for (int j = 0; j < 3; ++j) {
      src[d][j] = 0;
      w[d][j] = 0.0f;
    }
    const double fsx1 = d * scale, fsx2 = fsx1 + scale;
    const double cell = scale < (ssize - fsx1) ? scale : (ssize - fsx1);
    int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
    if (sx2 > ssize - 1) sx2 = ssize - 1;
    if (sx1 > sx2) sx1 = sx2;
    if (sx1 - fsx1 > 1e-3) {
      src[d][cnt[d]] = sx1 - 1;
      w[d][cnt[d]++] = (float)((sx1 - fsx1) / cell);
    }
    for (int sx = sx1; sx < sx2; ++sx) {
      src[d][cnt[d]] = sx;
      w[d][cnt[d]++] = (float)(1.0 / cell);
    }
    if (fsx2 - sx2 > 1e-3) {
      double a = fsx2 - sx2;
      if (a > 1.0) a = 1.0;
      if (a > cell) a = cell;
      src[d][cnt[d]] = sx2;
      w[d][cnt[d]++] = (float)(a / cell);
    }
  }
}

static int ensure_taps() {
  if (g_taps_ready) return 0;
  static Taps h;
  build_axis(RAW_W, OUT, h.xsrc, h.xw, h.xn);
  build_axis(RAW_H, OUT, h.ysrc, h.yw, h.yn);
  // the kernel keeps a thread's 10 horizontal results in registers and indexes them statically: output row d must
  // use exactly the source rows 10 (d / 4) + {0,1,2 | 2,3,4 | 5,6,7 | 7,8,9}[d % 4]
  static const int first[4] = {0, 2, 5, 7};
  for (int d = 0; d < OUT; ++d) {
    ACX_CHECK(h.yn[d] == 3, "vertical tap count");
    for (int t = 0; t < 3; ++t) ACX_CHECK(h.ysrc[d][t] == 10 * (d / 4) + first[d % 4] + t, "vertical tap pattern");
  }
  ACX_CUDA(cudaMemcpyToSymbol(c_taps, &h, sizeof(Taps)));
  g_taps_ready = true;
  return 0;
}

// byte-wise unsigned max of two words in 5 instructions: the high byte of each 16-bit lane of max.u16x2(a, b) is the
// max of the odd bytes whatever the even bytes hold; the even bytes are compared with the odd ones masked off
// (`__vmaxu4` is emulated in ~8)
__device__ __forceinline__ uint32_t max_u16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("max.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t max_u8x4(uint32_t a, uint32_t b) {
  const uint32_t odd = max_u16x2(a, b);
  const uint32_t even = max_u16x2(a & 0x00ff00ffu, b & 0x00ff00ffu);
  return (odd & 0xff00ff00u) | even;
}

// 16 RGB pixels held in 12 little-endian words -> 16 gray bytes (cv2 RGB2GRAY, 15-bit fixed point:
// y = (9798 r + 19235 g + 3735 b + 16384) >> 15).  Per pixel: one PRMT gathers [r,g,b,x] into a word, two IDP.2A
// (16-bit coefficient x 8-bit sample dot products) accumulate 2*(9798 r + 19235 g + 3735 b) + 32768 < 2^24, whose
// byte 2 is y (the doubled coefficients 19596 / 38470 / 7470 still fit 16 bits, so the >> 15 becomes a byte select
// folded into the PRMTs that pack four pixels into a word): 3.5 instructions per pixel instead of 20.
__device__ __forceinline__ uint32_t dp2a_lo(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t dp2a_hi(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint4 gray16(const uint32_t* w) {
  constexpr uint32_t C_RG = 19596u | (38470u << 16);   // 2 * 9798, 2 * 19235: bytes 0, 1 of the pixel word
  constexpr uint32_t C_B = 7470u;                      // 2 * 3735: byte 2; byte 3 (the next pixel's r) gets 0
  uint32_t y2[16];
#pragma unroll
  for (int px = 0; px < 16; ++px) {
    const int b0 = px * 3, wi = b0 >> 2, sh = b0 & 3;
    const uint32_t p = sh == 0 ? w[wi] : __byte_perm(w[wi], w[wi < 11 ? wi + 1 : wi], 0x3210 + 0x1111 * sh);
    y2[px] = dp2a_hi(C_B, p, dp2a_lo(C_RG, p, 32768u));
  }
  uint32_t g[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint32_t lo = __byte_perm(y2[4 * q], y2[4 * q + 1], 0x0062);
    const uint32_t hi = __byte_perm(y2[4 * q + 2], y2[4 * q + 3], 0x0062);
    g[q] = __byte_perm(lo, hi, 0x5410);
  }
  return make_uint4(g[0], g[1], g[2], g[3]);
}

// ---- shared pieces of the two K-PRE kernels -------------------------------------------------------------------------
// phase 1 of one thread: 48 bytes (16 pixels) of frame a (and b) -> byte-wise max -> 16 gray bytes
__device__ __forceinline__ uint4 gray_group(const uint4 a0, const uint4 a1, const uint4 a2, const uint4 b0, const uint4 b1,
                                            const uint4 b2, bool single) {
  uint32_t w[12] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y, a2.z, a2.w};
  if (!single) {
    w[0] = max_u8x4(w[0], b0.x); w[1] = max_u8x4(w[1], b0.y); w[2] = max_u8x4(w[2], b0.z); w[3] = max_u8x4(w[3], b0.w);
    w[4] = max_u8x4(w[4], b1.x); w[5] = max_u8x4(w[5], b1.y); w[6] = max_u8x4(w[6], b1.z); w[7] = max_u8x4(w[7], b1.w);
    w[8] = max_u8x4(w[8], b2.x); w[9] = max_u8x4(w[9], b2.y); w[10] = max_u8x4(w[10], b2.z); w[11] = max_u8x4(w[11], b2.w);
  }
  return gray16(w);
}

// per-thread horizontal taps of output column dx (phase-2 ownership)
struct XTaps {
  int xs[3];
  float xw[3], xc[3];
  int xn;
  __device__ __forceinline__ void load(int dx) {
    xn = __ldg(&c_taps.xn[dx]);
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      xs[t] = __ldg(&c_taps.xsrc[dx][t]);
      xw[t] = __ldg(&c_taps.xw[dx][t]);
      xc[t] = -8388608.0f * xw[t];   // exact (power-of-two scaling)
    }
  }
};

// phase 2 of one worker thread (dx, rg): horizontal taps of source rows [10 rg, 10 rg + 10) of the gray band into
// registers (table order, separate roundings), then the vertical taps of output rows dy0 .. dy0 + 3 (output row
// 4 rg + j uses local source rows {0,1,2 | 2,3,4 | 5,6,7 | 7,8,9}[j]), round half to even, saturate -> q[4]
__device__ __forceinline__ void resize_column(const uint8_t* gray /* [30][160] */, int rg, int dy0, const XTaps& x,
                                              uint32_t q[4]) {
  float h[10];
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint8_t* row = gray + (10 * rg + r) * RAW_W;
    float acc = 0.0f;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      if (t < x.xn) {
        const float m = __fmaf_rn(__uint_as_float(0x4B000000u | (uint32_t)row[x.xs[t]]), x.xw[t], x.xc[t]);
        acc = t == 0 ? m : __fadd_rn(acc, m);
      }
    }
    h[r] = acc;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int l0 = j == 0 ? 0 : (j == 1 ? 2 : (j == 2 ? 5 : 7));
    const float* yw = c_taps.yw[dy0 + j];
    float sum = __fmul_rn(__ldg(yw), h[l0]);
    sum = __fadd_rn(sum, __fmul_rn(__ldg(yw + 1), h[l0 + 1]));
    sum = __fadd_rn(sum, __fmul_rn(__ldg(yw + 2), h[l0 + 2]));
    int v = __float2int_rn(sum);  // cvRound
    v = v < 0 ? 0 : (v > 255 ? 255 : v);
    q[j] = (uint32_t)v;
  }
}

// One CTA per (environment, band of 12 output rows = 30 source rows), 320 threads.
//   phase 1: 300 threads each stream 48 contiguous bytes (16 pixels) of both frames with 16-byte loads, take the
//            byte-wise max and leave 16 gray bytes in shared memory (the raw bytes never touch shared memory)
//   phase 2: 252 threads = 84 output columns x 3 row groups.  The vertical scale is exactly 2.5, so 4 output rows use
//            exactly 10 source rows: thread (dx, rg) runs the horizontal taps of column dx for source rows
//            [10 rg, 10 rg + 10) into registers, then the vertical taps of output rows [4 rg, 4 rg + 4) from those
//            registers, rounds half to even, saturates and pushes the frame stack with coalesced 32-bit accesses -
//            no intermediate row buffer, one barrier per pass.
// Environments whose previous step was terminal run both phases twice: first on the reset frame (whose observation only
// seeds the stack: 4 copies, kept in registers), then on the step frames.  Every fp32 multiply and add is a separate
// rounding (no FMA contraction of an add), in OpenCV's order, which is what makes the result bit-exact.  The one FFMA
// is exact-equivalent to I2F + FMUL: a gray byte y is read as the float 2^23 + y (0x4B000000 | y) and
// fma(2^23 + y, w, -(2^23 w)) rounds the exact product y * w once, like the multiply would; it keeps the
// byte -> float conversion off the quarter-rate conversion pipe.
// This kernel serves small batches (one band per CTA, 4 CTAs per SM); large batches use the persistent kernel below.
constexpr int KPRE_THREADS = 320;
constexpr int GROUPS = BAND_SRC * RAW_ROW_BYTES / 48;   // 300 groups of 48 bytes per band
template <bool RESET>
__global__ void __launch_bounds__(KPRE_THREADS, 4) preprocess_kernel(const uint8_t* __restrict__ raw_a,
                                                                     const uint8_t* __restrict__ raw_b,
                                                                     const uint8_t* __restrict__ terminal,
                                                                     const uint8_t* __restrict__ reset_mask,
                                                                     const uint8_t* __restrict__ reset_raw,
                                                                     const uint8_t* stack_in, uint8_t* stack_out,
                                                                     size_t out_env_stride, int num_envs) {
  pdl_enter();   // in a rollout graph this kernel follows the previous step's sampling kernel on the same stream
  __shared__ __align__(16) uint8_t s_gray[BAND_SRC * RAW_W];   // 4800 B

  const int env = blockIdx.x / NUM_BANDS;
  const int band = blockIdx.x % NUM_BANDS;
  if (env >= num_envs) return;
  const int tid = threadIdx.x;
  const size_t band_off = (size_t)env * RAW_FRAME_BYTES + (size_t)band * BAND_SRC * RAW_ROW_BYTES;
  const bool do_reset = (!RESET) && (reset_mask != nullptr) && reset_mask[env] != 0;
  const bool term = (!RESET) && (terminal != nullptr) && terminal[env] != 0;
  const uint32_t* sin = reinterpret_cast<const uint32_t*>(stack_in + (size_t)env * STACK_BYTES);
  uint32_t* sout = reinterpret_cast<uint32_t*>(stack_out + (size_t)env * out_env_stride);

  const int dx = tid % OUT, rg = tid / OUT;   // rg in 0..3 (only 0..2 work: 252 threads)
  const bool worker = rg < 3;
  const int dy0 = band * BAND_OUT + 4 * (worker ? rg : 0);
  XTaps xt;
  xt.load(dx);
  uint32_t prev[4], q2[4] = {0u, 0u, 0u, 0u};

  for (int pass = do_reset ? 0 : 1; pass < 2; ++pass) {
    const bool reset_pass = pass == 0;
    const uint8_t* fa = reset_pass ? reset_raw : raw_a;
    const uint8_t* fb = reset_pass ? reset_raw : raw_b;
    const bool single = RESET || reset_pass;
    if (tid < GROUPS) {
      const uint4* pa = reinterpret_cast<const uint4*>(fa + band_off) + tid * 3;
      const uint4 a0 = __ldg(pa), a1 = __ldg(pa + 1), a2 = __ldg(pa + 2);
      uint4 b0 = a0, b1 = a1, b2 = a2;
      if (!single) {
        const uint4* pb = reinterpret_cast<const uint4*>(fb + band_off) + tid * 3;
        b0 = __ldg(pb), b1 = __ldg(pb + 1), b2 = __ldg(pb + 2);
      }
      // group g covers pixels [16 g, 16 g + 16) of the band's 30 x 160 pixel raster (rows are 10 groups)
      *reinterpret_cast<uint4*>(s_gray + tid * 16) = gray_group(a0, a1, a2, b0, b1, b2, single);
    }
    __syncthreads();
    if (worker) {
      // the old stack words are requested first so that their latency hides behind the horizontal taps
#pragma unroll
      for (int j = 0; j < 4; ++j)
        prev[j] = (!RESET && !reset_pass && !do_reset && !term) ? sin[(dy0 + j) * OUT + dx] : 0u;
      uint32_t q[4];
      resize_column(s_gray, rg, dy0, xt, q);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (reset_pass) {
          q2[j] = q[j];
          continue;
        }
        uint32_t word;
        if (RESET) {
          word = q[j] * 0x01010101u;  // wrappers.py:234: 4 copies
        } else {
          // multi_env.py:127-132: an env that was terminal is reset first (its observation is discarded), then stepped
          const uint32_t old = do_reset ? q2[j] * 0x01010101u : prev[j];
          word = term ? 0u : (old >> 8);           // roll -1 along channels (little endian), zero on terminal
          word |= q[j] << 24;                      // newest frame in channel 3
        }
        sout[(dy0 + j) * OUT + dx] = word;
      }
    }
    if (pass == 0) __syncthreads();   // the step pass overwrites s_gray
  }
}

// Persistent variant for large batches: grid = 3 CTAs per SM, each walks bands blockIdx.x, + gridDim.x, ...  The raw
// bytes of the NEXT band (2 x 14 400 contiguous bytes) are fetched by the TMA unit (cp.async.bulk global -> shared,
// mbarrier complete_tx) into the other half of a double buffer while the CTA converts and resizes the current one, so
// every CTA keeps 28.8 KB of HBM reads in flight all the time instead of only during its load phase (ncu of the kernel
// above: long-scoreboard stalls, 5.2 TB/s).  The gray band is double buffered too: one __syncthreads per band.
constexpr int KPRE_STAGE_BYTES = 2 * BAND_SRC * RAW_ROW_BYTES;                  // 28 800
constexpr int KPRE_P_SMEM = 2 * KPRE_STAGE_BYTES + 2 * BAND_SRC * RAW_W + 16;   // 67 216
constexpr int KPRE_P_CTAS_PER_SM = 3;

__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

template <bool RESET>
__global__ void __launch_bounds__(KPRE_THREADS, KPRE_P_CTAS_PER_SM)
    preprocess_persistent_kernel(const uint8_t* __restrict__ raw_a, const uint8_t* __restrict__ raw_b,
                                 const uint8_t* __restrict__ terminal, const uint8_t* __restrict__ reset_mask,
                                 const uint8_t* __restrict__ reset_raw, const uint8_t* stack_in, uint8_t* stack_out,
                                 size_t out_env_stride, int num_items) {
  extern __shared__ __align__(128) uint8_t kpre_smem[];
  uint8_t* s_raw = kpre_smem;                                    // [2 stages][frame a | frame b][14400]
  uint8_t* s_gray = kpre_smem + 2 * KPRE_STAGE_BYTES;            // [2][4800]
  uint64_t* bars = reinterpret_cast<uint64_t*>(kpre_smem + 2 * KPRE_STAGE_BYTES + 2 * BAND_SRC * RAW_W);
  constexpr uint32_t FRAME_BAND = BAND_SRC * RAW_ROW_BYTES;      // 14400

  const int tid = threadIdx.x;
  const int stride = gridDim.x;
  auto issue = [&](int item, int stage) {   // one thread
    const int e = item / NUM_BANDS, bnd = item - e * NUM_BANDS;
    const size_t off = (size_t)e * RAW_FRAME_BYTES + (size_t)bnd * FRAME_BAND;
    uint8_t* dst = s_raw + stage * KPRE_STAGE_BYTES;
    mbar_expect_tx(&bars[stage], RESET ? FRAME_BAND : 2 * FRAME_BAND);
    bulk_load_1d(dst, raw_a + off, FRAME_BAND, &bars[stage]);
    if (!RESET) bulk_load_1d(dst + FRAME_BAND, raw_b + off, FRAME_BAND, &bars[stage]);
  };
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0 && (int)blockIdx.x < num_items) issue(blockIdx.x, 0);

  const int dx = tid % OUT, rg = tid / OUT;
  const bool worker = rg < 3;
  XTaps xt;
  xt.load(dx);

  int k = 0;
  for (int item = blockIdx.x; item < num_items; item += stride, ++k) {
    const int stage = k & 1;
    const uint32_t parity = (uint32_t)(k >> 1) & 1u;
    // the other stage was last read in phase 1 of the previous band, which every thread left through that band's
    // __syncthreads: it is free for the next band's bytes
    if (tid == 0 && item + stride < num_items) issue(item + stride, stage ^ 1);

    const int env = item / NUM_BANDS, band = item - env * NUM_BANDS;
    const bool do_reset = (!RESET) && (reset_mask != nullptr) && reset_mask[env] != 0;
    const bool term = (!RESET) && (terminal != nullptr) && terminal[env] != 0;
    const uint32_t* sin = reinterpret_cast<const uint32_t*>(stack_in + (size_t)env * STACK_BYTES);
    uint32_t* sout = reinterpret_cast<uint32_t*>(stack_out + (size_t)env * out_env_stride);
    const int dy0 = band * BAND_OUT + 4 * (worker ? rg : 0);
    uint8_t* gray = s_gray + stage * (BAND_SRC * RAW_W);
    uint32_t prev[4], q2[4] = {0u, 0u, 0u, 0u};

    if (do_reset) {   // rare (an episode ended at the previous step): the reset frame goes through plain loads
      if (tid < GROUPS) {
        const uint4* pa =
            reinterpret_cast<const uint4*>(reset_raw + (size_t)env * RAW_FRAME_BYTES + (size_t)band * FRAME_BAND) + tid * 3;
        const uint4 a0 = __ldg(pa), a1 = __ldg(pa + 1), a2 = __ldg(pa + 2);
        *reinterpret_cast<uint4*>(gray + tid * 16) = gray_group(a0, a1, a2, a0, a1, a2, true);
      }
      __syncthreads();
      if (worker) resize_column(gray, rg, dy0, xt, q2);
      __syncthreads();
    }
    if (worker) {
#pragma unroll
      for (int j = 0; j < 4; ++j) prev[j] = (!RESET && !do_reset && !term) ? sin[(dy0 + j) * OUT + dx] : 0u;
    }
    mbar_wait(&bars[stage], parity, 900 + stage);
    if (tid < GROUPS) {
      const uint4* pa = reinterpret_cast<const uint4*>(s_raw + stage * KPRE_STAGE_BYTES) + tid * 3;
      const uint4 a0 = pa[0], a1 = pa[1], a2 = pa[2];
      uint4 b0 = a0, b1 = a1, b2 = a2;
      if (!RESET) {
        const uint4* pb = pa + FRAME_BAND / 16;
        b0 = pb[0], b1 = pb[1], b2 = pb[2];
      }
      *reinterpret_cast<uint4*>(gray + tid * 16) = gray_group(a0, a1, a2, b0, b1, b2, RESET);
    }
    __syncthreads();
    if (worker) {
      uint32_t q[4];
      resize_column(gray, rg, dy0, xt, q);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t word;
        if (RESET) {
          word = q[j] * 0x01010101u;
        } else {
          const uint32_t old = do_reset ? q2[j] * 0x01010101u : prev[j];
          word = term ? 0u : (old >> 8);
          word |= q[j] << 24;
        }
        sout[(dy0 + j) * OUT + dx] = word;
      }
    }
  }
}

// 0 = one band per CTA, 1 = persistent TMA pipeline, -1 = by size (ACX_KPRE_PERSISTENT overrides, for the tests)
static int kpre_mode() {
  static int mode = -2;
  if (mode == -2) {
    const char* e = getenv("ACX_KPRE_PERSISTENT");
    mode = e ? atoi(e) : -1;
  }
  return mode;
}
static int kpre_sm_count() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}
template <bool RESET>
static int launch_kpre(const uint8_t* raw_a, const uint8_t* raw_b, const uint8_t* terminal, const uint8_t* reset_mask,
                       const uint8_t* reset_raw, const uint8_t* stack_in, uint8_t* stack_out, size_t out_env_stride,
                       int num_envs, cudaStream_t st) {
  const int items = num_envs * NUM_BANDS;
  const int slots = kpre_sm_count() * KPRE_P_CTAS_PER_SM;
  const int mode = kpre_mode();
  // the pipeline pays off once every CTA walks many bands (measured: 256 envs 4.4 vs 4.1 TB/s for the band kernel,
  // 1024 envs 4.7 vs 5.7, 4096 envs 5.3 vs 6.7 for the pipeline)
  const bool persistent = mode == 1 || (mode == -1 && items >= 8 * slots);
  if (persistent) {
    static bool configured = false;
    if (!configured) {
      ACX_CUDA(cudaFuncSetAttribute(preprocess_persistent_kernel<RESET>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    KPRE_P_SMEM));
      configured = true;
    }
    const int grid = items < slots ? items : slots;
    preprocess_persistent_kernel<RESET><<<grid, KPRE_THREADS, KPRE_P_SMEM, st>>>(
        raw_a, raw_b, terminal, reset_mask, reset_raw, stack_in, stack_out, out_env_stride, items);
  } else {
    ACX_CUDA(launch_pdl(preprocess_kernel<RESET>, dim3(items), dim3(KPRE_THREADS), 0, st, raw_a, raw_b, terminal, reset_mask, reset_raw,
                        stack_in, stack_out, out_env_stride, num_envs));
  }
  ACX_LAUNCH_CHECK();
  return 0;
}

// ---- the stages of K-PRE on their own (the per-environment wrapper classes of the reference's API) ----------------------
// byte-wise max of two frames (AtariFrameskipWrapper.step, wrappers.py:64-65); 16 bytes per thread, scalar tail
__global__ void __launch_bounds__(256) frame_max_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b,
                                                        uint8_t* __restrict__ out, size_t nbytes) {
  const size_t quads = nbytes >> 4;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (size_t i = t0; i < quads; i += stride) {
    const uint4 x = __ldg(reinterpret_cast<const uint4*>(a) + i), y = __ldg(reinterpret_cast<const uint4*>(b) + i);
    reinterpret_cast<uint4*>(out)[i] = make_uint4(max_u8x4(x.x, y.x), max_u8x4(x.y, y.y), max_u8x4(x.z, y.z), max_u8x4(x.w, y.w));
  }
  for (size_t i = (quads << 4) + t0; i < nbytes; i += stride) out[i] = a[i] > b[i] ? a[i] : b[i];
}

// FrameStackWrapper.step / reset on already preprocessed frames (wrappers.py:224-235): frames uint8 [E,84,84] (one gray
// byte per pixel), stacks one 32-bit word per pixel.  mode per environment: 0 = push, 1 = push after a terminal step
// (all older frames zero), 2 = reset (4 copies)
__global__ void __launch_bounds__(256) framestack_kernel(const uint8_t* __restrict__ frames, const uint8_t* __restrict__ mode,
                                                         const uint32_t* stack_in, uint32_t* stack_out, int num_envs) {
  const int per = OUT * OUT;
  const size_t total = (size_t)num_envs * per;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int env = (int)(i / per);
    const uint32_t q = frames[i];
    const int m = mode ? mode[env] : 0;
    uint32_t word;
    if (m == 2)
      word = q * 0x01010101u;
    else
      word = (m == 1 ? 0u : (stack_in[i] >> 8)) | (q << 24);
    stack_out[i] = word;
  }
}

// ---- K-PRE at any square size S in [4, 128] and stack depth k in [1, 16] ----------------------------------------------
// The same per-environment work as K-PRE (max, gray, INTER_AREA to S x S, stack push / zero / reset) with variable-length
// tap tables: the tap counts reach 16 (x) and 20 (y) at S = 11, so K-PRE's fixed 3-tap tables and its 2.5 row pattern do
// not carry over.  Stacks are uint8 [E, S, S, k], the k frames of a pixel contiguous.
constexpr int SQ_MIN_SIZE = 4, SQ_MAX_SIZE = 128, SQ_MAX_FRAMES = 16;
constexpr int SQ_THREADS = 256;
constexpr int SQ_BAND_SRC = 32;   // a band of output rows spans about this many source rows (K-PRE: 30)

// OpenCV's computeResizeAreaTab (resize.cpp) for one axis, cn = 1, packed CSR-style: the taps of output d are
// [off[d], off[d + 1]), in table order (build_axis above without the 3-tap bound)
static void area_axis(int ssize, int dsize, std::vector<int>& off, std::vector<int>& src, std::vector<float>& w) {
  const double scale = (double)ssize / dsize;
  off.assign(1, 0);
  src.clear();
  w.clear();
  for (int d = 0; d < dsize; ++d) {
    const double fsx1 = d * scale, fsx2 = fsx1 + scale;
    const double cell = scale < (ssize - fsx1) ? scale : (ssize - fsx1);
    int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
    if (sx2 > ssize - 1) sx2 = ssize - 1;
    if (sx1 > sx2) sx1 = sx2;
    if (sx1 - fsx1 > 1e-3) {
      src.push_back(sx1 - 1);
      w.push_back((float)((sx1 - fsx1) / cell));
    }
    for (int sx = sx1; sx < sx2; ++sx) {
      src.push_back(sx);
      w.push_back((float)(1.0 / cell));
    }
    if (fsx2 - sx2 > 1e-3) {
      double a = fsx2 - sx2;
      if (a > 1.0) a = 1.0;
      if (a > cell) a = cell;
      src.push_back(sx2);
      w.push_back((float)(a / cell));
    }
    off.push_back((int)src.size());
  }
}

// the device tables of one output size (one allocation: xoff, xsrc, yoff, ysrc as int32, then xw, yw as fp32)
struct SqTables {
  const int* xoff;
  const int* xsrc;
  const int* yoff;
  const int* ysrc;
  const float* xw;
  const float* yw;
  float scale;        // 0, or 1 / block area at the sizes where cv2 takes its integer-scale path (see sq_tables)
  int band_rows;      // output rows per CTA
  int num_bands;
  int max_src_rows;   // the most source rows one band spans
};

// shared memory of one CTA: gray rows [R][160] u8 | horizontal results [R][S] f32 | old stack bytes of the band
// [rows][S][k] | the band's new plane [rows][S] | its reset plane [rows][S]
static size_t sq_smem_bytes(const SqTables& t, int size, int frames) {
  return (size_t)t.max_src_rows * RAW_W + (size_t)t.max_src_rows * size * 4 + (size_t)t.band_rows * size * (frames + 2);
}

// max + gray + INTER_AREA of one band of one frame (pair) into `plane` [rows][S]; every thread of the CTA calls it
//   phase 1: 48 raw bytes (16 pixels) of each frame per thread with 16-byte loads -> byte-wise max -> 16 gray bytes in
//            shared memory (each raw row is read once per CTA)
//   phase 2: the horizontal taps of every (source row, output column) into shared fp32: buf = 0, buf = buf + src * w
//   phase 3: the vertical taps of every output pixel of the band: first term assigned, the rest added; round half to
//            even, saturate
// Every multiply and add is a separate fp32 rounding (__fmul_rn / __fadd_rn are never contracted into an FMA), in
// OpenCV's order, which is what makes the result bit-exact.
__device__ __forceinline__ void sq_band_plane(const uint8_t* fa, const uint8_t* fb, bool single, int R, int y0, int d0,
                                              int rows, int size, const SqTables& t, uint8_t* s_gray, float* s_h,
                                              uint8_t* plane) {
  const int tid = threadIdx.x;
  const uint4* pa = reinterpret_cast<const uint4*>(fa + (size_t)y0 * RAW_ROW_BYTES);
  const uint4* pb = reinterpret_cast<const uint4*>(fb + (size_t)y0 * RAW_ROW_BYTES);
  for (int g = tid; g < R * (RAW_ROW_BYTES / 48); g += SQ_THREADS) {
    const uint4 a0 = __ldg(pa + 3 * g), a1 = __ldg(pa + 3 * g + 1), a2 = __ldg(pa + 3 * g + 2);
    uint4 b0 = a0, b1 = a1, b2 = a2;
    if (!single) b0 = __ldg(pb + 3 * g), b1 = __ldg(pb + 3 * g + 1), b2 = __ldg(pb + 3 * g + 2);
    *reinterpret_cast<uint4*>(s_gray + 16 * g) = gray_group(a0, a1, a2, b0, b1, b2, single);
  }
  __syncthreads();
  for (int i = tid; i < R * size; i += SQ_THREADS) {
    const int r = i / size, dx = i - r * size;
    const uint8_t* row = s_gray + r * RAW_W;
    const int t0 = __ldg(t.xoff + dx), t1 = __ldg(t.xoff + dx + 1);
    float acc = __fmul_rn((float)row[__ldg(t.xsrc + t0)], __ldg(t.xw + t0));
    for (int k = t0 + 1; k < t1; ++k) acc = __fadd_rn(acc, __fmul_rn((float)row[__ldg(t.xsrc + k)], __ldg(t.xw + k)));
    s_h[i] = acc;
  }
  __syncthreads();
  for (int i = tid; i < rows * size; i += SQ_THREADS) {
    const int dl = i / size, dx = i - dl * size;
    const int t0 = __ldg(t.yoff + d0 + dl), t1 = __ldg(t.yoff + d0 + dl + 1);
    float sum = __fmul_rn(__ldg(t.yw + t0), s_h[(__ldg(t.ysrc + t0) - y0) * size + dx]);
    for (int k = t0 + 1; k < t1; ++k) sum = __fadd_rn(sum, __fmul_rn(__ldg(t.yw + k), s_h[(__ldg(t.ysrc + k) - y0) * size + dx]));
    if (t.scale != 0.0f) sum = __fmul_rn(sum, t.scale);   // integer-scale path: the exact block sum times 1 / area
    int v = __float2int_rn(sum);  // cvRound
    plane[i] = (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
  }
}

// One CTA per (environment, band of t.band_rows output rows), 256 threads.  The old stack bytes of the band are fetched
// into shared memory first (cp.async, so the fetch overlaps the frame work; every byte of the band is read before any is
// written, which makes the in-place update safe), then the frame pipeline runs - twice for an environment whose previous
// step was terminal: first on the reset frame, whose plane only seeds the stack (k copies), then on the step frames.  The
// new band [rows][S][k] is contiguous in the output and is written with coalesced 32-bit stores where it is aligned.
template <bool RESET>
__global__ void __launch_bounds__(SQ_THREADS, 4) preprocess_sq_kernel(const uint8_t* __restrict__ raw_a,
                                                                   const uint8_t* __restrict__ raw_b,
                                                                   const uint8_t* __restrict__ terminal,
                                                                   const uint8_t* __restrict__ reset_mask,
                                                                   const uint8_t* __restrict__ reset_raw,
                                                                   const uint8_t* stack_in, uint8_t* stack_out,
                                                                   size_t out_env_stride, int size, int frames,
                                                                   SqTables t) {
  extern __shared__ __align__(16) uint8_t sq_smem[];
  const int env = blockIdx.x / t.num_bands, band = blockIdx.x - env * t.num_bands;
  const int tid = threadIdx.x;
  const int d0 = band * t.band_rows;
  const int rows = min(size - d0, t.band_rows);
  const int y0 = __ldg(t.ysrc + __ldg(t.yoff + d0));
  const int R = __ldg(t.ysrc + __ldg(t.yoff + d0 + rows) - 1) + 1 - y0;
  uint8_t* s_gray = sq_smem;
  float* s_h = reinterpret_cast<float*>(sq_smem + t.max_src_rows * RAW_W);
  uint8_t* s_old = sq_smem + t.max_src_rows * RAW_W + t.max_src_rows * size * 4;
  uint8_t* s_plane = s_old + t.band_rows * size * frames;
  uint8_t* s_rplane = s_plane + t.band_rows * size;

  const bool do_reset = (!RESET) && (reset_mask != nullptr) && reset_mask[env] != 0;
  const bool term = (!RESET) && (terminal != nullptr) && terminal[env] != 0;
  const int band_bytes = rows * size * frames;
  const size_t stack_bytes = (size_t)size * size * frames;
  if (!RESET && !do_reset && !term && frames > 1) {
    const uint8_t* sin = stack_in + (size_t)env * stack_bytes + (size_t)d0 * size * frames;
    if ((((uintptr_t)sin | (uintptr_t)band_bytes) & 3) == 0) {
      for (int i = 4 * tid; i < band_bytes; i += 4 * SQ_THREADS)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(s_old + i)), "l"(sin + i) : "memory");
    } else {
      for (int i = tid; i < band_bytes; i += SQ_THREADS) s_old[i] = sin[i];
    }
  }
  const size_t frame_off = (size_t)env * RAW_FRAME_BYTES;
  if (do_reset) {
    sq_band_plane(reset_raw + frame_off, reset_raw + frame_off, true, R, y0, d0, rows, size, t, s_gray, s_h, s_rplane);
    __syncthreads();   // the step pass overwrites s_gray and s_h
  }
  sq_band_plane(raw_a + frame_off, raw_b + frame_off, RESET, R, y0, d0, rows, size, t, s_gray, s_h, s_plane);
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();

  // byte j of the band = frame c of pixel p: roll by -1 along the frames, zero on terminal, the new frame last
  auto byte_at = [&](int j) -> uint32_t {
    const int p = j / frames, c = j - p * frames;
    if (RESET || c == frames - 1) return s_plane[p];
    if (term) return 0u;
    return do_reset ? s_rplane[p] : s_old[j + 1];
  };
  uint8_t* sout = stack_out + (size_t)env * out_env_stride + (size_t)d0 * size * frames;
  int j0 = 0;
  if (((uintptr_t)sout & 3) == 0) {
    const int words = band_bytes >> 2;
    for (int w = tid; w < words; w += SQ_THREADS)
      reinterpret_cast<uint32_t*>(sout)[w] =
          byte_at(4 * w) | (byte_at(4 * w + 1) << 8) | (byte_at(4 * w + 2) << 16) | (byte_at(4 * w + 3) << 24);
    j0 = words << 2;
  }
  for (int j = j0 + tid; j < band_bytes; j += SQ_THREADS) sout[j] = (uint8_t)byte_at(j);
}

// FrameStackWrapper.step / reset on already preprocessed frames uint8 [E, S, S] for stacks uint8 [E, S, S, k]: one thread
// per pixel, frames in ascending order (frame c + 1 is read before frame c is written, so in place is safe)
__global__ void __launch_bounds__(256) framestack_sq_kernel(const uint8_t* __restrict__ frames, const uint8_t* __restrict__ mode,
                                                            const uint8_t* stack_in, uint8_t* stack_out, int num_envs,
                                                            int size, int k) {
  const int per = size * size;
  const size_t total = (size_t)num_envs * per;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int env = (int)(i / per);
    const uint8_t q = frames[i];
    const int m = mode ? mode[env] : 0;
    const uint8_t* in = stack_in + i * k;
    uint8_t* out = stack_out + i * k;
    for (int c = 0; c < k - 1; ++c) out[c] = m == 2 ? q : (m == 1 ? 0 : in[c + 1]);
    out[k - 1] = q;
  }
}

// The tap tables of one output size, built on the host once per (device, size) and kept for the life of the process.
// The first call for a size uploads them (a synchronous copy): make it outside stream capture, as for K-PRE's tables.
static int sq_tables(int size, SqTables* out) {
  static std::mutex mu;
  static std::map<std::pair<int, int>, SqTables> cache;
  static std::map<int, size_t> smem_configured;   // per device: the dynamic shared memory both kernels are allowed
  int dev = 0;
  ACX_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find({dev, size});
  if (it == cache.end()) {
    std::vector<int> xoff, xsrc, yoff, ysrc;
    std::vector<float> xw, yw;
    area_axis(RAW_W, size, xoff, xsrc, xw);
    area_axis(RAW_H, size, yoff, ysrc, yw);
    // cv2.resize takes resizeAreaFast_ instead when both scales are integers to DBL_EPSILON (sizes 5 and 10 here):
    // round(float(integer block sum) * (1.f / area)).  With unit weights the two passes add the block's bytes exactly in
    // fp32 (at most 255 * 1344 < 2^24), and one multiply by 1 / area follows.
    const double fx = 1.0 / ((double)size / RAW_W), fy = 1.0 / ((double)size / RAW_H);
    const int ix = (int)lrint(fx), iy = (int)lrint(fy);
    const bool fast = fabs(fx - ix) < DBL_EPSILON && fabs(fy - iy) < DBL_EPSILON;
    if (fast) {
      std::fill(xw.begin(), xw.end(), 1.0f);
      std::fill(yw.begin(), yw.end(), 1.0f);
    }
    std::vector<int> ints;
    ints.insert(ints.end(), xoff.begin(), xoff.end());
    ints.insert(ints.end(), xsrc.begin(), xsrc.end());
    ints.insert(ints.end(), yoff.begin(), yoff.end());
    ints.insert(ints.end(), ysrc.begin(), ysrc.end());
    std::vector<float> floats(xw);
    floats.insert(floats.end(), yw.begin(), yw.end());
    void* d = nullptr;
    const size_t ibytes = ints.size() * sizeof(int), fbytes = floats.size() * sizeof(float);
    ACX_CUDA(cudaMalloc(&d, ibytes + fbytes));
    ACX_CUDA(cudaMemcpy(d, ints.data(), ibytes, cudaMemcpyHostToDevice));
    ACX_CUDA(cudaMemcpy((char*)d + ibytes, floats.data(), fbytes, cudaMemcpyHostToDevice));
    SqTables t;
    const int* di = static_cast<const int*>(d);
    t.xoff = di;
    t.xsrc = t.xoff + xoff.size();
    t.yoff = t.xsrc + xsrc.size();
    t.ysrc = t.yoff + yoff.size();
    t.xw = reinterpret_cast<const float*>((const char*)d + ibytes);
    t.yw = t.xw + xw.size();
    t.scale = fast ? 1.0f / (float)(ix * iy) : 0.0f;
    int band_rows = SQ_BAND_SRC * size / RAW_H;
    t.band_rows = band_rows < 1 ? 1 : band_rows;
    t.num_bands = (size + t.band_rows - 1) / t.band_rows;
    t.max_src_rows = 0;
    for (int b = 0; b < t.num_bands; ++b) {
      const int d0 = b * t.band_rows, d1 = std::min(size, d0 + t.band_rows);
      t.max_src_rows = std::max(t.max_src_rows, ysrc[yoff[d1] - 1] + 1 - ysrc[yoff[d0]]);
    }
    it = cache.emplace(std::make_pair(dev, size), t).first;
  }
  // the attribute is raised once to the largest stack depth of each size met so far, outside any capture
  const size_t need = sq_smem_bytes(it->second, size, SQ_MAX_FRAMES);
  if (need > smem_configured[dev]) {
    ACX_CUDA(cudaFuncSetAttribute(preprocess_sq_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    ACX_CUDA(cudaFuncSetAttribute(preprocess_sq_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    smem_configured[dev] = need;
  }
  *out = it->second;
  return 0;
}

static int check_sq_shape(int size, int frames) {
  ACX_CHECK(size >= SQ_MIN_SIZE && size <= SQ_MAX_SIZE, "size must be in [4, 128], got " + std::to_string(size));
  ACX_CHECK(frames >= 1 && frames <= SQ_MAX_FRAMES, "num_frames must be in [1, 16], got " + std::to_string(frames));
  return 0;
}

template <bool RESET>
static int launch_kpre_sq(const uint8_t* raw_a, const uint8_t* raw_b, const uint8_t* terminal, const uint8_t* reset_mask,
                          const uint8_t* reset_raw, const uint8_t* stack_in, uint8_t* stack_out, size_t out_env_stride,
                          int num_envs, int size, int frames, cudaStream_t st) {
  SqTables t;
  int r = sq_tables(size, &t);
  if (r) return r;
  const size_t grid = (size_t)num_envs * t.num_bands;
  ACX_CHECK(grid < (1u << 31), "too many environments");
  preprocess_sq_kernel<RESET><<<(unsigned)grid, SQ_THREADS, sq_smem_bytes(t, size, frames), st>>>(
      raw_a, raw_b, terminal, reset_mask, reset_raw, stack_in, stack_out, out_env_stride, size, frames, t);
  ACX_LAUNCH_CHECK();
  return 0;
}

}  // namespace acx

extern "C" {

int acx_frame_max_u8(const uint8_t* d_a, const uint8_t* d_b, uint8_t* d_out, size_t nbytes, void* stream) {
  using namespace acx;
  if (nbytes == 0) return 0;
  ACX_CHECK(d_a && d_b && d_out, "null pointer");
  ACX_CHECK((((uintptr_t)d_a | (uintptr_t)d_b | (uintptr_t)d_out) & 15) == 0, "misaligned buffer");
  size_t blocks = ((nbytes >> 4) + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  frame_max_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(d_a, d_b, d_out, nbytes);
  ACX_LAUNCH_CHECK();
  return 0;
}

int acx_framestack_push_u8(const uint8_t* d_frames, const uint8_t* d_mode, const uint8_t* d_stack_in, uint8_t* d_stack_out,
                           int num_envs, void* stream) {
  using namespace acx;
  ACX_CHECK(num_envs >= 0, "num_envs < 0");
  if (num_envs == 0) return 0;
  ACX_CHECK(d_frames && d_stack_in && d_stack_out, "null pointer");
  ACX_CHECK((((uintptr_t)d_stack_in | (uintptr_t)d_stack_out) & 3) == 0, "misaligned stack");
  size_t blocks = ((size_t)num_envs * OUT * OUT + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  framestack_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      d_frames, d_mode, reinterpret_cast<const uint32_t*>(d_stack_in), reinterpret_cast<uint32_t*>(d_stack_out), num_envs);
  ACX_LAUNCH_CHECK();
  return 0;
}

int acx_preprocess_stack_u8(const uint8_t* d_raw_a, const uint8_t* d_raw_b, const uint8_t* d_terminal,
                            const uint8_t* d_reset_mask, const uint8_t* d_reset_raw, const uint8_t* d_stack_in,
                            uint8_t* d_stack_out, size_t out_env_stride, int num_envs, void* stream) {
  using namespace acx;
  ACX_CHECK(num_envs >= 0, "num_envs < 0");
  if (num_envs == 0) return 0;
  ACX_CHECK(d_raw_a && d_raw_b && d_stack_in && d_stack_out, "null pointer");
  ACX_CHECK(out_env_stride >= (size_t)STACK_BYTES && (out_env_stride % 4) == 0, "out_env_stride");
  ACX_CHECK(d_reset_mask == nullptr || d_reset_raw != nullptr, "reset_mask without reset_raw");
  ACX_CHECK(((uintptr_t)d_raw_a % 16) == 0 && ((uintptr_t)d_raw_b % 16) == 0 && ((uintptr_t)d_stack_in % 4) == 0 &&
                ((uintptr_t)d_stack_out % 4) == 0 && (d_reset_raw == nullptr || ((uintptr_t)d_reset_raw % 16) == 0),
            "misaligned buffer");
  int r = ensure_taps();
  if (r) return r;
  return launch_kpre<false>(d_raw_a, d_raw_b, d_terminal, d_reset_mask, d_reset_raw, d_stack_in, d_stack_out, out_env_stride,
                            num_envs, reinterpret_cast<cudaStream_t>(stream));
}

int acx_preprocess_reset_u8(const uint8_t* d_raw, uint8_t* d_stack_out, size_t out_env_stride, int num_envs, void* stream) {
  using namespace acx;
  ACX_CHECK(num_envs >= 0, "num_envs < 0");
  if (num_envs == 0) return 0;
  ACX_CHECK(d_raw && d_stack_out, "null pointer");
  ACX_CHECK(out_env_stride >= (size_t)STACK_BYTES && (out_env_stride % 4) == 0, "out_env_stride");
  ACX_CHECK(((uintptr_t)d_raw % 16) == 0 && ((uintptr_t)d_stack_out % 4) == 0, "misaligned buffer");
  int r = ensure_taps();
  if (r) return r;
  return launch_kpre<true>(d_raw, d_raw, nullptr, nullptr, nullptr, d_stack_out, d_stack_out, out_env_stride, num_envs,
                           reinterpret_cast<cudaStream_t>(stream));
}
}

extern "C" {

int acx_preprocess_stack_sq_u8(const uint8_t* d_raw_a, const uint8_t* d_raw_b, const uint8_t* d_terminal,
                               const uint8_t* d_reset_mask, const uint8_t* d_reset_raw, const uint8_t* d_stack_in,
                               uint8_t* d_stack_out, size_t out_env_stride, int num_envs, int size, int num_frames,
                               void* stream) {
  using namespace acx;
  int r = check_sq_shape(size, num_frames);
  if (r) return r;
  ACX_CHECK(num_envs >= 0, "num_envs < 0");
  if (num_envs == 0) return 0;
  const size_t stack_bytes = (size_t)size * size * num_frames;
  ACX_CHECK(d_raw_a && d_raw_b && d_stack_in && d_stack_out, "null pointer");
  ACX_CHECK(out_env_stride >= stack_bytes, "out_env_stride below size * size * num_frames");
  ACX_CHECK(d_stack_in != d_stack_out || out_env_stride == stack_bytes, "in place needs out_env_stride == size * size * num_frames");
  ACX_CHECK(d_reset_mask == nullptr || d_reset_raw != nullptr, "reset_mask without reset_raw");
  ACX_CHECK(((uintptr_t)d_raw_a % 16) == 0 && ((uintptr_t)d_raw_b % 16) == 0 &&
                (d_reset_raw == nullptr || ((uintptr_t)d_reset_raw % 16) == 0),
            "misaligned raw frames");
  return launch_kpre_sq<false>(d_raw_a, d_raw_b, d_terminal, d_reset_mask, d_reset_raw, d_stack_in, d_stack_out,
                               out_env_stride, num_envs, size, num_frames, reinterpret_cast<cudaStream_t>(stream));
}

int acx_preprocess_reset_sq_u8(const uint8_t* d_raw, uint8_t* d_stack_out, size_t out_env_stride, int num_envs, int size,
                               int num_frames, void* stream) {
  using namespace acx;
  int r = check_sq_shape(size, num_frames);
  if (r) return r;
  ACX_CHECK(num_envs >= 0, "num_envs < 0");
  if (num_envs == 0) return 0;
  ACX_CHECK(d_raw && d_stack_out, "null pointer");
  ACX_CHECK(out_env_stride >= (size_t)size * size * num_frames, "out_env_stride below size * size * num_frames");
  ACX_CHECK(((uintptr_t)d_raw % 16) == 0, "misaligned raw frames");
  return launch_kpre_sq<true>(d_raw, d_raw, nullptr, nullptr, nullptr, nullptr, d_stack_out, out_env_stride, num_envs, size,
                              num_frames, reinterpret_cast<cudaStream_t>(stream));
}

int acx_framestack_push_sq_u8(const uint8_t* d_frames, const uint8_t* d_mode, const uint8_t* d_stack_in, uint8_t* d_stack_out,
                              int num_envs, int size, int num_frames, void* stream) {
  using namespace acx;
  int r = check_sq_shape(size, num_frames);
  if (r) return r;
  ACX_CHECK(num_envs >= 0, "num_envs < 0");
  if (num_envs == 0) return 0;
  ACX_CHECK(d_frames && d_stack_in && d_stack_out, "null pointer");
  size_t blocks = ((size_t)num_envs * size * size + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  framestack_sq_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      d_frames, d_mode, d_stack_in, d_stack_out, num_envs, size, num_frames);
  ACX_LAUNCH_CHECK();
  return 0;
}
}
