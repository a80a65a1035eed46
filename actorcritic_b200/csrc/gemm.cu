// gemm.cu - GEMM on bf16 planes for sm_100a: TMA -> shared memory (128B swizzle) -> tcgen05.mma with
// the fp32 accumulator in TMEM -> tcgen05.ld epilogue.  One kernel serves every matrix product of the
// learner (conv/fc forward as im2col GEMMs, dgrad, wgrad, K-FAC factor SYRKs, preconditioning); the
// precision is chosen per call by how many bf16 plane pairs are accumulated (1 = bf16, 3 ~ 2^-17,
// 6 = fp32-class) - see DESIGN.md "precision by plane pairs".
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer,
// warps 2..5 = epilogue (one TMEM lane quarter each).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>

#include "layers.cuh"
#include "tc.cuh"

namespace acx {

constexpr int BM = 128;
constexpr int BK = 64;  // bf16 elements per k-block: one 128-byte swizzle row (TcParams.bk = 32: half rows, 64-byte swizzle - tuning knob)

struct OutParams {
  int m, n;
  float alpha;
  const float* bias;
  int relu;
  float* c;
  int ldc;
  bf16* cp[ACX_MAX_PLANES];
  int c_num_planes;
  int ldcp;
  const bf16* mask;
  int mask_ld, mask_rows;
  int perm_m, perm_n;   // result row / column i is stored at perm64(i) (acx.h: conv1 patches read from the row-pair copy)
};

// column order (kw, row parity, c) of a 64-wide conv1 patch chunk -> the reference's (kh, kw, c): 4-groups stay 4-groups
__device__ __host__ __forceinline__ int perm64(int i) {
  return (i & ~63) | (((i >> 2) & 1) << 5) | (((i >> 3) & 7) << 2) | (i & 3);
}

struct TcParams {
  OutParams out;
  int k;
  int kb_total, kb_per_split;
  int num_pairs;
  int pair_a[6], pair_b[6];
  int npa, npb;          // planes of A / B that the pairs reference (each is loaded once per k-block)
  int bn;                // tile width (32, 64, 128)
  int bk;                // k-block depth (64 or 32)
  int trace;             // triage: record where CTA 0's MMA warp spends its cycles (ACX_GEMM_TRACE=1)
  int stages;            // shared-memory ring depth
  int tiles_m, tiles_n, num_tiles, splits, total_work;
  int symmetric;
  int panel;             // SYRK panel mode: one work item = one k-split of the whole (<= 256 wide) symmetric product
  int to_workspace;
  float* ws;
  int ws_ld;
  long long ws_split_stride;  // floats
  uint32_t mn_lbo, mn_sbo, mn_kstep;
  // split-K reduction inside the kernel (no finalize launch): the CTA that completes a group of RED_GROUP consecutive
  // splits of a tile sums them in split order; with more than one group the group sums go to `ws2` and the CTA that
  // completes the last group sums those in group order - every association is fixed, so the result does not depend on
  // which CTA arrives last.  Counters: per tile `groups` group counters + 1 tile counter, zero on entry, left zero.
  // gathered MN-major operands (acx_gather_t): k-block kb = the 64 locations of box (bx x by cells, ts samples) number
  // kb % g_cells of sample group kb / g_cells; chunk q of a location comes from coordinates (c0, x + c1, c2, y + c3, sample)
  int same_operand;      // symmetric product of one operand with itself: diagonal tiles load their operand once (B = the A tiles)
  int gather_a, gather_b;
  int g_cells, g_nx, g_bx, g_by, g_ts;
  signed char ga[4][16], gb[4][16];
  int fuse, groups;
  float* ws2;
  long long ws2_stride;   // floats between group sums
  int* counters;
};
constexpr int RED_GROUP = 8;
constexpr size_t kFusedReduceBytes = 256 << 10;   // partial sums one CTA may have to read back for one tile
constexpr int RED_COUNTER_BYTES = 16384;   // head of the workspace: 4096 counters

// ------------------------------------------------------------------------------------------------
// shared epilogue math: one result element -> alpha, bias, ReLU, mask
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float finish_value(const OutParams& o, int m, int n, float acc) {
  float v = o.alpha * acc;
  if (o.bias) v += __ldg(o.bias + n);
  if (o.relu) v = fmaxf(v, 0.0f);
  if (o.mask) {
    float mk = __bfloat162float(o.mask[(size_t)(m % o.mask_rows) * o.mask_ld + n]);
    if (!(mk > 0.0f)) v = 0.0f;
  }
  return v;
}
__device__ __forceinline__ void store_value(const OutParams& o, int m, int n, float v) {
  if (o.perm_m) m = perm64(m);
  if (o.perm_n) n = perm64(n);
  if (o.c) o.c[(size_t)m * o.ldc + n] = v;
  if (o.c_num_planes > 0) {
    bf16 p0, p1, p2;
    split3(v, p0, p1, p2);
    size_t idx = (size_t)m * o.ldcp + n;
    o.cp[0][idx] = p0;
    if (o.c_num_planes > 1) o.cp[1][idx] = p1;
    if (o.c_num_planes > 2) o.cp[2][idx] = p2;
  }
}

// a lane owns columns (n, n+1) of row m (n even): 8-byte fp32 and 4-byte bf16x2 stores, so a warp writes 256 / 128
// contiguous bytes of one row per instruction
__device__ __forceinline__ void store_pair(const OutParams& o, int m, int n, float v0, float v1, bool c_vec_ok) {
  const bool two = n + 1 < o.n;
  if (o.c) {
    float* dst = o.c + (size_t)m * o.ldc + n;
    if (two && c_vec_ok) {
      *reinterpret_cast<float2*>(dst) = make_float2(v0, v1);
    } else {
      dst[0] = v0;
      if (two) dst[1] = v1;
    }
  }
  if (o.c_num_planes > 0) {
    uint32_t q0, q1, q2;
    split3x2(v0, v1, q0, q1, q2);
    const size_t idx = (size_t)m * o.ldcp + n;   // ldcp % 8 == 0 and n even: 4-byte aligned
    if (two) {
      *reinterpret_cast<uint32_t*>(o.cp[0] + idx) = q0;
      if (o.c_num_planes > 1) *reinterpret_cast<uint32_t*>(o.cp[1] + idx) = q1;
      if (o.c_num_planes > 2) *reinterpret_cast<uint32_t*>(o.cp[2] + idx) = q2;
    } else {
      o.cp[0][idx] = __ushort_as_bfloat16((unsigned short)(q0 & 0xffffu));
      if (o.c_num_planes > 1) o.cp[1][idx] = __ushort_as_bfloat16((unsigned short)(q1 & 0xffffu));
      if (o.c_num_planes > 2) o.cp[2][idx] = __ushort_as_bfloat16((unsigned short)(q2 & 0xffffu));
    }
  }
}

// four consecutive result columns (n % 4 == 0) of row m: epilogue math + stores, ragged edges handled element-wise
__device__ __forceinline__ void emit4(const OutParams& o, int m, int n, float4 acc) {
  if (m >= o.m || n >= o.n) return;
  const bool c_vec = o.c == nullptr || ((o.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(o.c) & 15) == 0);
  if (n + 3 < o.n && c_vec && (o.ldcp & 3) == 0) {
    float v[4] = {o.alpha * acc.x, o.alpha * acc.y, o.alpha * acc.z, o.alpha * acc.w};
    if (o.bias) {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] += __ldg(o.bias + n + j);
    }
    if (o.relu) {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.0f);
    }
    if (o.mask) {
      const bf16* mk = o.mask + (size_t)(m % o.mask_rows) * o.mask_ld + n;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (!(__bfloat162float(mk[j]) > 0.0f)) v[j] = 0.0f;
    }
    const int ms = o.perm_m ? perm64(m) : m, ns = o.perm_n ? perm64(n) : n;   // (a 4-group stays a 4-group)
    if (o.c) *reinterpret_cast<float4*>(o.c + (size_t)ms * o.ldc + ns) = make_float4(v[0], v[1], v[2], v[3]);
    if (o.c_num_planes > 0) {
      uint2 ph, pm, pl;
      split3x4(v[0], v[1], v[2], v[3], ph, pm, pl);
      const size_t idx = (size_t)ms * o.ldcp + ns;
      *reinterpret_cast<uint2*>(o.cp[0] + idx) = ph;
      if (o.c_num_planes > 1) *reinterpret_cast<uint2*>(o.cp[1] + idx) = pm;
      if (o.c_num_planes > 2) *reinterpret_cast<uint2*>(o.cp[2] + idx) = pl;
    }
    return;
  }
  const float a[4] = {acc.x, acc.y, acc.z, acc.w};
  for (int j = 0; j < 4; ++j) {
    if (n + j < o.n) {
      store_value(o, m, n + j, finish_value(o, m, n + j, a[j]));
    } else if (o.c_num_planes > 0 && n + j < o.ldcp) {   // the padding columns of plane outputs stay zero
      const size_t idx = (size_t)m * o.ldcp + n + j;
      o.cp[0][idx] = __float2bfloat16(0.0f);
      if (o.c_num_planes > 1) o.cp[1][idx] = __float2bfloat16(0.0f);
      if (o.c_num_planes > 2) o.cp[2][idx] = __float2bfloat16(0.0f);
    }
  }
}

// One warp sums `count` partial planes (`pstride` floats apart, row stride `ld`) of the 32 x 32 block at (m0, n0) in plane
// order.  Lane layout: 8 lanes x float4 per row, 4 rows per pass, 8 passes: acc[t] = row m0 + (lane >> 3) + 4 t, columns
// n0 + 4 (lane & 7) .. + 3.  Partials were written by other SMs: read through L2.
__device__ __forceinline__ void reduce_block(const float* __restrict__ src, long long pstride, int count, int ld, int m0, int n0,
                                             int lane, float4 (&acc)[8]) {
  const float* base = src + (size_t)(m0 + (lane >> 3)) * ld + n0 + 4 * (lane & 7);
#pragma unroll
  for (int t = 0; t < 8; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  int sidx = 0;
  for (; sidx + 1 < count; sidx += 2, base += 2 * pstride) {   // two partials (16 loads per thread) in flight; summed in plane order
    float4 x[8], y[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) x[t] = __ldcg(reinterpret_cast<const float4*>(base + (size_t)(4 * t) * ld));
#pragma unroll
    for (int t = 0; t < 8; ++t) y[t] = __ldcg(reinterpret_cast<const float4*>(base + pstride + (size_t)(4 * t) * ld));
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      acc[t].x = (acc[t].x + x[t].x) + y[t].x;
      acc[t].y = (acc[t].y + x[t].y) + y[t].y;
      acc[t].z = (acc[t].z + x[t].z) + y[t].z;
      acc[t].w = (acc[t].w + x[t].w) + y[t].w;
    }
  }
  if (sidx < count) {
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const float4 x = __ldcg(reinterpret_cast<const float4*>(base + (size_t)(4 * t) * ld));
      acc[t].x += x.x;
      acc[t].y += x.y;
      acc[t].z += x.z;
      acc[t].w += x.w;
    }
  }
}

constexpr int MAX_STAGES = 8;
constexpr int GEMM_THREADS = 320;                       // warp 0 TMA producer, warp 1 MMA, warps 2..9 epilogue
constexpr int EPI_BYTES = 8 * 32 * 32 * 4;              // one XOR-swizzled 32 x 32 fp32 staging tile per epilogue warp

// ------------------------------------------------------------------------------------------------
// the tcgen05 kernel: persistent, warp specialised.
//   warp 0      TMA producer: per k-block loads every referenced A plane and B plane ONCE into one ring stage
//   warp 1      TMEM allocator + MMA issuer (one elected lane): all plane pairs of the stage accumulate into one
//               fp32 accumulator; two accumulators in TMEM so that the epilogue of tile t overlaps the MMAs of t+1
//   warps 2..5  epilogue: tcgen05.ld -> per-warp shared-memory transpose -> row-contiguous global stores
// MAJOR 0: A stored [M,K], B stored [N,K] (both K-major).  MAJOR 1: A stored [K,M], B stored [K,N] (both MN-major).
// Work items (tile, split) are taken round-robin: w = blockIdx.x, + gridDim.x, ...
// ------------------------------------------------------------------------------------------------
__device__ long long g_gemm_trace[12];   // triage: total / waiting for operands / waiting for an accumulator / k-blocks

template <int MAJOR>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap ta0, const __grid_constant__ CUtensorMap ta1,
               const __grid_constant__ CUtensorMap ta2, const __grid_constant__ CUtensorMap tb0,
               const __grid_constant__ CUtensorMap tb1, const __grid_constant__ CUtensorMap tb2,
               const __grid_constant__ TcParams p) {
  // (p is __grid_constant__: the reduction path hands `p.out` to helper functions by reference; without it, taking the
  // address of a parameter makes every later field read a generic-address load that is re-issued after each global store -
  // measured ~700 cycles per store instruction)
  extern __shared__ __align__(1024) uint8_t smem_raw[];   // 128B-swizzled TMA tiles need 1024-byte alignment
  uint8_t* smem = smem_raw;
  if ((smem_u32(smem_raw) & 1023u) != 0) {                 // never expected; fail loudly instead of corrupting tiles
    if (threadIdx.x == 0) atomicExch(&g_tc_error, 9);
    return;
  }
  const int BN = p.bn;
  const int bk = p.bk;
  const int a_tile_bytes = BM * bk * 2;
  const int b_tile_bytes = BN * bk * 2;
  const int panel_tile_bytes = 4 * bk * 128;   // panel mode: bk k-rows x 256 columns of one plane
  // panel mode: a stage holds, per plane, the 64 k-rows x (up to) 256 columns of X once; the same shared memory feeds
  // the A side and the B side of the three upper 128 x 128 sub-tiles of X^T X
  const int stage_bytes = p.panel ? p.npa * panel_tile_bytes : p.npa * a_tile_bytes + p.npb * b_tile_bytes;
  float* epi = reinterpret_cast<float*>(smem + p.stages * stage_bytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(epi) + EPI_BYTES);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* acc_full = empty_bar + MAX_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  volatile int* red_flag = reinterpret_cast<volatile int*>(tmem_slot + 1);   // split-K reduction: the arrival order of this CTA

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem_cols = p.panel ? 512u : (uint32_t)(2 * BN);   // 64, 128 or 256 (two accumulators); panel: three + pad

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);   // the TMA thread's expect_tx arrival
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], BN > 32 ? 8 : 4);   // epilogue warps that drain an accumulator
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above overlapped the predecessor's tail; its results are visible from here on

  // work item -> (tile_m, tile_n, split)
  auto decode = [&](int w, int& tm, int& tn, int& split) {
    if (p.panel) {
      split = w;
      tm = tn = 0;
      return;
    }
    split = w / p.num_tiles;
    int t = w - split * p.num_tiles;
    if (p.symmetric) {
      tm = 0;
      int cnt = p.tiles_n;
      while (t >= cnt) {
        t -= cnt;
        ++tm;
        --cnt;
      }
      tn = tm + t;
    } else {
      tm = t / p.tiles_n;
      tn = t - tm * p.tiles_n;
    }
  };

  if (warp == 0) {
    {
      // ===== TMA producer (whole warp waits, one elected lane issues) =====
      int it = 0;
      int ring_s = 0;
      uint32_t ring_ph = 0u;
      for (int w = blockIdx.x; w < p.total_work; w += gridDim.x) {
        int tm, tn, split;
        decode(w, tm, tn, split);
        const int m0 = tm * BM, n0 = tn * BN;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        // MN-major tiles are loaded as 64-column chunks; chunks that start beyond the matrix are skipped (their
        // shared memory only feeds accumulator rows/columns that are never stored)
        const int na = MAJOR == 0 ? 0 : min(BM / 64, (p.out.m - m0 + 63) / 64);
        const int nb = MAJOR == 0 ? 0 : min(BN / 64, (p.out.n - n0 + 63) / 64);
        const int nch = (p.out.n + 63) / 64;   // panel mode: 64-column chunks of X
        const bool diag = MAJOR == 1 && p.same_operand && tm == tn;   // B tile = A tile: loaded once
        const uint32_t tx = p.panel ? (uint32_t)(p.npa * nch * bk * 128)
                                    : (MAJOR == 0 ? (uint32_t)stage_bytes
                                                  : (uint32_t)((p.npa * na + (diag ? 0 : p.npb * nb)) * bk * 128));
        // gathered operands: the chunk coordinates of this work item's (up to 4) A and (up to 2) B chunks are fixed - read them
        // from the parameters once, not per load (the issuing thread is alone: dependent parameter loads with run-time indices
        // cost it hundreds of cycles per k-block)
        int ac[4][4] = {}, bc[4][2] = {};
        if (MAJOR == 1 && p.gather_a) {
          const int qa = p.panel ? 0 : (m0 >> 6), qb = n0 >> 6;
#pragma unroll
          for (int d = 0; d < 4; ++d) {
#pragma unroll
            for (int j = 0; j < 4; ++j) ac[d][j] = p.ga[d][min(qa + j, 15)];
#pragma unroll
            for (int j = 0; j < 2; ++j) bc[d][j] = p.gb[d][min(qb + j, 15)];
          }
        }
        // ... and the box position advances incrementally (cell inside the sample group, then the next group)
        int g_cell = 0, g_grp = 0, g_cx = 0, g_cy = 0;
        if (MAJOR == 1 && p.gather_a) {
          g_grp = kb0 / p.g_cells;
          g_cell = kb0 - g_grp * p.g_cells;
          g_cy = g_cell / p.g_nx;
          g_cx = g_cell - g_cy * p.g_nx;
        }
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = ring_s;   // ring position and phase advance without a division (this thread is the bottleneck)
          const uint32_t ph = ring_ph;
          if (++ring_s == p.stages) {
            ring_s = 0;
            ring_ph ^= 1u;
          }
          // gathered operands: where the 64 locations of this k-block sit in the (x, y, sample) space
          const int gx0 = g_cx * p.g_bx, gy0 = g_cy * p.g_by, gn0 = g_grp * p.g_ts;
          if (MAJOR == 1 && p.gather_a) {
            if (++g_cx == p.g_nx) {
              g_cx = 0;
              ++g_cy;
            }
            if (++g_cell == p.g_cells) {
              g_cell = g_cx = g_cy = 0;
              ++g_grp;
            }
          }
          mbar_wait(&empty_bar[s], ph ^ 1u, 1);
          __syncwarp();
          if (!elect_one()) continue;
          mbar_expect_tx(&full_bar[s], tx);
          uint8_t* a_s = smem + s * stage_bytes;
          if (p.panel) {
            for (int i = 0; i < p.npa; ++i) {
              const CUtensorMap* ma = i == 0 ? &ta0 : (i == 1 ? &ta1 : &ta2);
#pragma unroll
              for (int j = 0; j < 4; ++j) {   // (a panel is at most 256 columns = 4 chunks)
                if (j >= nch) break;
                uint8_t* dst = a_s + i * panel_tile_bytes + j * (bk * 128);
                if (MAJOR == 1 && p.gather_a)
                  tma_load_5d(dst, ma, &full_bar[s], ac[0][j], gx0 + ac[1][j], ac[2][j], gy0 + ac[3][j], gn0);
                else
                  tma_load_2d(dst, ma, &full_bar[s], 64 * j, kb * bk);
              }
            }
            continue;
          }
          uint8_t* b_s = a_s + p.npa * a_tile_bytes;
          for (int i = 0; i < p.npa; ++i) {
            const CUtensorMap* ma = i == 0 ? &ta0 : (i == 1 ? &ta1 : &ta2);
            uint8_t* dst = a_s + i * a_tile_bytes;
            if (MAJOR == 0) {
              tma_load_2d(dst, ma, &full_bar[s], kb * bk, m0);
            } else if (p.gather_a) {
#pragma unroll
              for (int j = 0; j < 2; ++j)
                if (j < na) tma_load_5d(dst + j * (bk * 128), ma, &full_bar[s], ac[0][j], gx0 + ac[1][j], ac[2][j], gy0 + ac[3][j], gn0);
            } else {
              for (int j = 0; j < na; ++j) tma_load_2d(dst + j * (bk * 128), ma, &full_bar[s], m0 + 64 * j, kb * bk);
            }
          }
          for (int i = 0; i < p.npb && !diag; ++i) {
            const CUtensorMap* mb = i == 0 ? &tb0 : (i == 1 ? &tb1 : &tb2);
            uint8_t* dst = b_s + i * b_tile_bytes;
            if (MAJOR == 0) {
              tma_load_2d(dst, mb, &full_bar[s], kb * bk, n0);
            } else if (p.gather_b) {
#pragma unroll
              for (int j = 0; j < 2; ++j)
                if (j < nb) tma_load_5d(dst + j * (bk * 128), mb, &full_bar[s], bc[0][j], gx0 + bc[1][j], bc[2][j], gy0 + bc[3][j], gn0);
            } else {
              for (int j = 0; j < nb; ++j) tma_load_2d(dst + j * (bk * 128), mb, &full_bar[s], n0 + 64 * j, kb * bk);
            }
          }
        }
      }
      // every load of this CTA's last work item is issued: the successor's blocks may be scheduled onto SMs as they free up
      __syncwarp();
      if (elect_one()) pdl_trigger();
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one elected lane) =====
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)MAJOR << 15) | ((uint32_t)MAJOR << 16) |
                           ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    // K-major tiles: rows of bk elements = one 128-byte (bk = 64) or 64-byte (bk = 32) swizzle row, 8-row atoms
    const uint32_t lbo = MAJOR == 0 ? 16u : p.mn_lbo;
    const uint32_t sbo = MAJOR == 0 ? (bk == 64 ? 1024u : 512u) : p.mn_sbo;
    const uint32_t layout = (MAJOR == 0 && bk == 32) ? 4u : 2u;   // SWIZZLE_64B : SWIZZLE_128B
    const uint32_t kstep = MAJOR == 0 ? 32u : p.mn_kstep;
    const uint64_t kstep16 = (uint64_t)(kstep >> 4);
    // descriptor offsets (16-byte units) of every plane pair's A / B tile inside a stage
    uint32_t a_off[6], b_off[6], b_off_d[6];   // b_off_d: the B plane inside the A tiles (diagonal tiles of a one-operand SYRK)
#pragma unroll
    for (int pr = 0; pr < 6; ++pr) {
      a_off[pr] = (uint32_t)(p.pair_a[pr] * a_tile_bytes) >> 4;
      b_off[pr] = (uint32_t)(p.pair_b[pr] * b_tile_bytes) >> 4;
      b_off_d[pr] = (uint32_t)(p.pair_b[pr] * a_tile_bytes) >> 4;
    }
    const int npairs = p.num_pairs;
    const bool trace = p.trace != 0 && blockIdx.x == 0;   // ACX_GEMM_TRACE=1: where CTA 0's MMA warp spends its cycles
    long long w_full = 0, w_acc = 0, tw = 0;
    const long long t_begin = trace ? clock64() : 0;
    int it = 0, lt = 0;
    int ring_s = 0;
    uint32_t ring_ph = 0u;
    // the descriptor of stage 0 and its step from stage to stage: built once, advanced by an addition (this thread is the
    // bottleneck of the kernel: every instruction it does not execute per k-block is time the tensor pipe gets)
    const uint64_t a_desc_s0 = make_smem_desc_sw(smem_u32(smem), lbo, sbo, layout);
    const uint64_t desc_step = (uint64_t)((uint32_t)stage_bytes >> 4);
    const uint64_t b_desc_off = (uint64_t)((uint32_t)(p.npa * a_tile_bytes) >> 4);
    uint64_t a_desc_cur = a_desc_s0;
    for (int w = blockIdx.x; w < p.total_work; w += gridDim.x, ++lt) {
      int tm, tn, split;
      decode(w, tm, tn, split);
      const int kb0 = split * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      int krem = p.k - kb0 * bk;   // K elements left from this k-block on
      const int buf = p.panel ? 0 : (lt & 1);
      const uint32_t aph = p.panel ? ((uint32_t)lt & 1u) : ((uint32_t)(lt >> 1) & 1u);
      const bool diag = MAJOR == 1 && p.same_operand && !p.panel && tm == tn;
      if (trace) tw = clock64();
      mbar_wait(&acc_empty[buf], aph ^ 1u, 4);
      if (trace) w_acc += clock64() - tw;
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(p.panel ? 0 : buf * BN);
      for (int kb = kb0; kb < kb1; ++kb, ++it) {
        const int s = ring_s;   // ring position and phase advance without a division (this thread is the bottleneck)
        const uint32_t ph = ring_ph;
        // the descriptor of a tile advanced by `off` bytes is base + (off >> 4): only the 14-bit address field moves
        // (tiles are 1024-byte aligned inside the < 256 KB shared window, so the add never carries out of the field)
        const uint64_t a_desc0 = a_desc_cur;
        const uint64_t b_desc0 = diag ? a_desc_cur : a_desc_cur + b_desc_off;
        if (++ring_s == p.stages) {
          ring_s = 0;
          ring_ph ^= 1u;
          a_desc_cur = a_desc_s0;
        } else {
          a_desc_cur += desc_step;
        }
        const int kvalid = min(bk, krem);
        krem -= bk;
        if (trace) tw = clock64();
        mbar_wait(&full_bar[s], ph, 2);
        if (trace) w_full += clock64() - tw;
        tc_fence_after();
        if (elect_one()) {
          const int ksteps = (kvalid + 15) >> 4;
          uint32_t acc_flag = kb > kb0 ? 1u : 0u;
          if (p.panel) {
            // three upper sub-tiles (0,0) (0,1) (1,1): accumulators at TMEM columns 0, 128, 256
            for (int pr = 0; pr < p.num_pairs; ++pr) {
              for (int sub = 0; sub < 3; ++sub) {
                const int ti = sub == 2 ? 1 : 0, tj = sub >= 1 ? 1 : 0;
                uint64_t ad = a_desc0 + (uint64_t)((uint32_t)(p.pair_a[pr] * panel_tile_bytes + ti * a_tile_bytes) >> 4);
                uint64_t bd = a_desc0 + (uint64_t)((uint32_t)(p.pair_b[pr] * panel_tile_bytes + tj * a_tile_bytes) >> 4);
                uint32_t flag = (kb > kb0 || pr > 0) ? 1u : 0u;
                if (ksteps == 4 || ksteps == 8) {
                  umma_bf16_x4(d_tmem + (uint32_t)(sub * 128), ad, bd, (uint32_t)kstep16, (uint32_t)kstep16, idesc, flag);
                  if (ksteps == 8)
                    umma_bf16_x4(d_tmem + (uint32_t)(sub * 128), ad + 4 * kstep16, bd + 4 * kstep16, (uint32_t)kstep16, (uint32_t)kstep16, idesc, 1u);
                  continue;
                }
                for (int kk = 0; kk < ksteps; ++kk) {
                  umma_bf16(d_tmem + (uint32_t)(sub * 128), ad, bd, idesc, flag);
                  flag = 1u;
                  ad += kstep16;
                  bd += kstep16;
                }
              }
            }
          } else if (ksteps == 4) {
            // full 64-deep k-block: straight-line code (pair offsets hoisted out of the tile loop, both loops unrolled).
            // The issuing thread is alone on its scheduler: with run-time loop bounds and per-pair parameter loads the
            // issue loop itself cost ~110 cycles per MMA (measured, conv.cu trace) against 48-64 in the tensor pipe.
            if (npairs == 3) {
              umma_bf16_x4_pairs3(d_tmem, a_desc0, b_desc0, (uint32_t)kstep16, (uint32_t)kstep16, idesc, acc_flag, a_off[0],
                                  diag ? b_off_d[0] : b_off[0], a_off[1], diag ? b_off_d[1] : b_off[1], a_off[2], diag ? b_off_d[2] : b_off[2]);
            } else if (npairs == 2) {
              umma_bf16_x4_pairs2(d_tmem, a_desc0, b_desc0, (uint32_t)kstep16, (uint32_t)kstep16, idesc, acc_flag, a_off[0],
                                  diag ? b_off_d[0] : b_off[0], a_off[1], diag ? b_off_d[1] : b_off[1]);
            } else {
#pragma unroll
              for (int pr = 0; pr < 6; ++pr)
                if (pr < npairs)
                  umma_bf16_x4(d_tmem, a_desc0 + (uint64_t)a_off[pr], b_desc0 + (uint64_t)(diag ? b_off_d[pr] : b_off[pr]), (uint32_t)kstep16,
                               (uint32_t)kstep16, idesc, pr ? 1u : acc_flag);
            }
          } else if (ksteps == 8) {
            // 128-deep k-block: two groups of four steps per plane pair
#pragma unroll
            for (int pr = 0; pr < 6; ++pr)
              if (pr < npairs) {
                const uint64_t ad = a_desc0 + (uint64_t)a_off[pr], bd = b_desc0 + (uint64_t)(diag ? b_off_d[pr] : b_off[pr]);
                umma_bf16_x4(d_tmem, ad, bd, (uint32_t)kstep16, (uint32_t)kstep16, idesc, pr ? 1u : acc_flag);
                umma_bf16_x4(d_tmem, ad + 4 * kstep16, bd + 4 * kstep16, (uint32_t)kstep16, (uint32_t)kstep16, idesc, 1u);
              }
          } else {
            for (int pr = 0; pr < p.num_pairs; ++pr) {
              uint64_t ad = a_desc0 + (uint64_t)((uint32_t)(p.pair_a[pr] * a_tile_bytes) >> 4);
              uint64_t bd = b_desc0 + (uint64_t)((uint32_t)(p.pair_b[pr] * (diag ? a_tile_bytes : b_tile_bytes)) >> 4);
              for (int kk = 0; kk < ksteps; ++kk) {
                umma_bf16(d_tmem, ad, bd, idesc, acc_flag);
                acc_flag = 1u;
                ad += kstep16;
                bd += kstep16;
              }
            }
          }
          umma_commit(&empty_bar[s]);  // frees the stage once these MMAs have read it
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&acc_full[buf]);
      __syncwarp();
    }
    if (trace && lane == 0) {
      g_gemm_trace[0] = clock64() - t_begin;
      g_gemm_trace[1] = w_full;
      g_gemm_trace[2] = w_acc;
      g_gemm_trace[3] = it;
    }
  } else {
    // ===== epilogue: TMEM -> registers -> shared-memory transpose -> global =====
    // Eight warps: warp w may read the TMEM lane quarter w % 4 (32 tile rows); the two warps of a quarter take alternate
    // 32-column chunks.  After the transpose a lane owns 4 consecutive columns and 8 lanes cover one row of the chunk, so
    // every global store instruction writes whole contiguous row segments (fp32: 16 B per lane, bf16 planes: 8 B per
    // lane).  The staging tile is 32 x 32 fp32 without padding; its 16-byte groups are XOR-swizzled by the row, which
    // keeps the 128-bit row writes and the 128-bit transposed reads conflict free.
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int grp = (warp - 2) >> 2;
    float* st = epi + (size_t)(warp - 2) * (32 * 32);
    constexpr int CH = 32;
    constexpr int lpr = CH >> 2;          // lanes per row
    constexpr int rpi = 32 / lpr;         // rows per iteration
    const int rsub = lane / lpr;
    const int cl = (lane - rsub * lpr) * 4;
    auto staged = [&](int r) -> const float* { return st + r * 32 + (((cl >> 2) ^ (r & 7)) << 2); };
    const OutParams& o = p.out;
    float* const oc = o.c;
    bf16* const cp0 = o.cp[0];
    bf16* const cp1 = o.cp[1];
    bf16* const cp2 = o.cp[2];
    const int npl = o.c_num_planes;
    const bool c_vec = oc != nullptr && (o.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(oc) & 15) == 0;
    const float alpha = o.alpha;
    const float* const bias = o.bias;
    const bf16* const mask = o.mask;
    const int mask_ld = o.mask_ld, mask_rows = o.mask_rows;
    const bool relu = o.relu != 0;
    const int om = o.m, on = o.n, ldc = o.ldc, ldcp = o.ldcp;
    const bool to_ws = p.to_workspace != 0;
    float* const ws = p.ws;
    const int ws_ld = p.ws_ld;
    const long long ws_split_stride = p.ws_split_stride;
    int lt = 0;
    for (int w = blockIdx.x; w < p.total_work; w += gridDim.x, ++lt) {
      int tm, tn, split;
      decode(w, tm, tn, split);
      const int buf = p.panel ? 0 : (lt & 1);
      const uint32_t aph = p.panel ? ((uint32_t)lt & 1u) : ((uint32_t)(lt >> 1) & 1u);
      mbar_wait(&acc_full[buf], aph, 3);
      tc_fence_after();
      const int nsub = p.panel ? 3 : 1;
      for (int sub = 0; sub < nsub; ++sub) {
      const int m0 = (p.panel ? (sub == 2 ? BM : 0) : tm * BM) + q * 32;
      const int n0 = p.panel ? (sub >= 1 ? BN : 0) : tn * BN;
      const int col_base = p.panel ? sub * 128 : buf * BN;
      for (int c0 = grp * CH; c0 < BN; c0 += 2 * CH) {
        uint32_t raw[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(col_base + c0);
        tmem_ld32(taddr, raw);
        float4* strow = reinterpret_cast<float4*>(st + lane * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          strow[j ^ (lane & 7)] = make_float4(__uint_as_float(raw[4 * j]), __uint_as_float(raw[4 * j + 1]),
                                              __uint_as_float(raw[4 * j + 2]), __uint_as_float(raw[4 * j + 3]));
        if (c0 + 2 * CH >= BN && sub == nsub - 1) {   // this warp's share of the accumulator is drained: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
        __syncwarp();
        const int n = n0 + c0 + cl;
        if (to_ws) {
          float* dst = ws + (size_t)split * ws_split_stride + (size_t)(m0 + rsub) * ws_ld + n;
#pragma unroll
          for (int r = rsub; r < 32; r += rpi, dst += (size_t)rpi * ws_ld)
            *reinterpret_cast<float4*>(dst) = *reinterpret_cast<const float4*>(staged(r));
        } else if (n < on) {
          const int rows_valid = min(32, om - m0);
          float b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
          if (bias) {
            b0 = __ldg(bias + n);
            if (n + 1 < on) b1 = __ldg(bias + n + 1);
            if (n + 2 < on) b2 = __ldg(bias + n + 2);
            if (n + 3 < on) b3 = __ldg(bias + n + 3);
          }
          if (n + 3 < on && mask == nullptr) {
            // fast path: whole 4-column groups, no mask
            float* dc = oc ? oc + (size_t)(m0 + rsub) * ldc + n : nullptr;
            size_t idx = (size_t)(m0 + rsub) * ldcp + n;   // ldcp % 8 == 0 and n % 4 == 0: 8-byte aligned plane stores
#pragma unroll 4
            for (int r = rsub; r < rows_valid; r += rpi, idx += (size_t)rpi * ldcp) {
              const float4 a4 = *reinterpret_cast<const float4*>(staged(r));
              float v0 = fmaf(alpha, a4.x, b0), v1 = fmaf(alpha, a4.y, b1), v2 = fmaf(alpha, a4.z, b2), v3 = fmaf(alpha, a4.w, b3);
              if (relu) {
                v0 = fmaxf(v0, 0.0f);
                v1 = fmaxf(v1, 0.0f);
                v2 = fmaxf(v2, 0.0f);
                v3 = fmaxf(v3, 0.0f);
              }
              if (dc) {
                if (c_vec) {
                  *reinterpret_cast<float4*>(dc) = make_float4(v0, v1, v2, v3);
                } else {
                  dc[0] = v0;
                  dc[1] = v1;
                  dc[2] = v2;
                  dc[3] = v3;
                }
                dc += (size_t)rpi * ldc;
              }
              if (npl > 0) {
                uint2 ph, pm, pl;
                split3x4(v0, v1, v2, v3, ph, pm, pl);
                *reinterpret_cast<uint2*>(cp0 + idx) = ph;
                if (npl > 1) *reinterpret_cast<uint2*>(cp1 + idx) = pm;
                if (npl > 2) *reinterpret_cast<uint2*>(cp2 + idx) = pl;
              }
            }
          } else {
            // general path: ragged right edge and / or ReLU mask of the forward activation
            int mrow = mask ? (m0 + rsub) % mask_rows : 0;
            const int mstep = mask ? rpi % mask_rows : 0;
            // every mask word of this chunk is requested before the first one is used: one L2 round trip per chunk
            // instead of one per row (whole 4-column groups; the ragged edge loads element-wise below)
            uint2 mwp[16];
            if (mask && n + 3 < on) {
              int mr = mrow;
#pragma unroll
              for (int t = 0; t < 16; ++t) {
                mwp[t] = make_uint2(0u, 0u);
                if (rsub + t * rpi < rows_valid) {
                  mwp[t] = __ldg(reinterpret_cast<const uint2*>(mask + (size_t)mr * mask_ld + n));   // mask_ld % 8 == 0, n % 4 == 0
                  mr += mstep;
                  if (mr >= mask_rows) mr -= mask_rows;
                }
              }
            }
            int t_it = 0;
            for (int r = rsub; r < rows_valid; r += rpi, ++t_it) {
              const int m = m0 + r;
              const float4 a4 = *reinterpret_cast<const float4*>(staged(r));
              float v[4] = {fmaf(alpha, a4.x, b0), fmaf(alpha, a4.y, b1), fmaf(alpha, a4.z, b2), fmaf(alpha, a4.w, b3)};
              if (relu) {
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.0f);
              }
              if (mask) {
                const bf16* mk = mask + (size_t)mrow * mask_ld + n;
                if (n + 3 < on) {
                  uint2 mw = mwp[0];
#pragma unroll
                  for (int t = 1; t < 16; ++t)
                    if (t == t_it) mw = mwp[t];
                  if (!(__uint_as_float(mw.x << 16) > 0.0f)) v[0] = 0.0f;
                  if (!(__uint_as_float(mw.x & 0xffff0000u) > 0.0f)) v[1] = 0.0f;
                  if (!(__uint_as_float(mw.y << 16) > 0.0f)) v[2] = 0.0f;
                  if (!(__uint_as_float(mw.y & 0xffff0000u) > 0.0f)) v[3] = 0.0f;
                } else {
#pragma unroll
                  for (int j = 0; j < 4; ++j)
                    if (n + j < on && !(__bfloat162float(mk[j]) > 0.0f)) v[j] = 0.0f;
                }
                mrow += mstep;
                if (mrow >= mask_rows) mrow -= mask_rows;
              }
              if (n + 3 < on) {
                if (oc) {
                  float* dc = oc + (size_t)m * ldc + n;
                  if (c_vec) {
                    *reinterpret_cast<float4*>(dc) = make_float4(v[0], v[1], v[2], v[3]);
                  } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) dc[j] = v[j];
                  }
                }
                if (npl > 0) {
                  uint2 ph, pm, pl;
                  split3x4(v[0], v[1], v[2], v[3], ph, pm, pl);
                  const size_t idx = (size_t)m * ldcp + n;
                  *reinterpret_cast<uint2*>(cp0 + idx) = ph;
                  if (npl > 1) *reinterpret_cast<uint2*>(cp1 + idx) = pm;
                  if (npl > 2) *reinterpret_cast<uint2*>(cp2 + idx) = pl;
                }
              } else {
                for (int j = 0; j < 4; ++j)
                  if (n + j < on) store_value(o, m, n + j, v[j]);
              }
            }
          }
        }
        __syncwarp();
      }
      }
      if (to_ws && p.fuse) {
        // ===== split-K reduction by whichever CTA completes a group / the tile (see TcParams) =====
        auto epi_bar = [] { asm volatile("bar.sync 1, 256;" ::: "memory"); };   // the 8 epilogue warps
        const int ew = warp - 2;
        const int tile_id = p.panel ? 0 : w - split * p.num_tiles;
        int* cnt = p.counters + tile_id * (p.groups + 1);
        const int g = split / RED_GROUP;
        const int gsize = min(RED_GROUP, p.splits - g * RED_GROUP);
        const bool rtrace = p.trace != 0 && blockIdx.x == 0 && threadIdx.x == 64;
        if (rtrace) g_gemm_trace[4] = clock64();
        __threadfence();   // this thread's partial sums are visible device-wide before the CTA is counted
        if (rtrace) g_gemm_trace[5] = clock64();
        epi_bar();
        if (threadIdx.x == 64) *red_flag = atomicAdd(&cnt[g], 1);
        epi_bar();
        if (rtrace) g_gemm_trace[6] = clock64();
        if (*red_flag == gsize - 1) {
          __threadfence();
          if (rtrace) g_gemm_trace[7] = clock64();
          const int tm0 = p.panel ? 0 : tm * BM, tn0 = p.panel ? 0 : tn * BN;
          const int bw = (p.panel ? 2 * BN : BN) >> 5, bh = (p.panel ? 2 * BM : BM) >> 5;   // 32 x 32 blocks of the work item
          // lower blocks of a symmetric result are written as mirrors of the upper ones; blocks outside the result do not exist
          auto skip = [&](int m0, int n0) { return m0 >= om || n0 >= on || (p.symmetric && m0 > n0); };
          bool final_pass = p.groups == 1;
          if (!final_pass) {
            for (int b = ew; b < bw * bh; b += 8) {
              const int bi = b / bw, bj = b - bi * bw;
              const int m0 = tm0 + bi * 32, n0 = tn0 + bj * 32;
              if (skip(m0, n0)) continue;
              float4 acc[8];
              reduce_block(ws + (size_t)g * RED_GROUP * ws_split_stride, ws_split_stride, gsize, ws_ld, m0, n0, lane, acc);
              float* dst = p.ws2 + (size_t)g * p.ws2_stride + (size_t)(m0 + (lane >> 3)) * ws_ld + n0 + 4 * (lane & 7);
#pragma unroll
              for (int t = 0; t < 8; ++t) *reinterpret_cast<float4*>(dst + (size_t)(4 * t) * ws_ld) = acc[t];
            }
            __threadfence();
            epi_bar();
            if (threadIdx.x == 64) *red_flag = atomicAdd(&cnt[p.groups], 1);
            epi_bar();
            final_pass = *red_flag == p.groups - 1;
            if (final_pass) __threadfence();
          }
          if (final_pass) {
            const float* src = p.groups == 1 ? ws : p.ws2;
            const long long pst = p.groups == 1 ? ws_split_stride : p.ws2_stride;
            const int cntp = p.groups == 1 ? p.splits : p.groups;
            for (int b = ew; b < bw * bh; b += 8) {
              const int bi = b / bw, bj = b - bi * bw;
              const int m0 = tm0 + bi * 32, n0 = tn0 + bj * 32;
              if (skip(m0, n0)) continue;
              float4 acc[8];
              if (rtrace && b == ew) g_gemm_trace[8] = clock64();
              reduce_block(src, pst, cntp, ws_ld, m0, n0, lane, acc);
              if (rtrace && b == ew) g_gemm_trace[9] = clock64();
              // The sums go through the warp's staging tile (16-byte groups XOR-swizzled by the row) and ONE copy of the
              // epilogue code walks them - first the block itself, then (symmetric, off-diagonal) its mirror image read
              // transposed.  With the 16 calls unrolled this section was ~200 KB of straight-line code executed once per
              // block: every instruction fetch missed (measured ~700 cycles per store instruction).
              __syncwarp();
#pragma unroll
              for (int t = 0; t < 8; ++t) {
                const int r = (lane >> 3) + 4 * t;
                *reinterpret_cast<float4*>(st + r * 32 + (((lane & 7) ^ (r & 7)) << 2)) = acc[t];
              }
              __syncwarp();
              const int passes = (p.symmetric && m0 < n0) ? 16 : 8;
#pragma unroll 1
              for (int it = 0; it < passes; ++it) {
                const int r = (lane >> 3) + 4 * (it & 7), c4 = lane & 7;
                float4 v;
                int mm, nn;
                if (it < 8) {
                  v = *reinterpret_cast<const float4*>(st + r * 32 + ((c4 ^ (r & 7)) << 2));
                  mm = m0 + r;
                  nn = n0 + 4 * c4;
                } else {   // row r of the mirrored block = column r of the upper one; its columns 4 c4 .. + 3 = rows of the upper one
                  const int r0 = 4 * c4;
                  v.x = st[(r0 + 0) * 32 + ((((r >> 2) ^ ((r0 + 0) & 7)) << 2) + (r & 3))];
                  v.y = st[(r0 + 1) * 32 + ((((r >> 2) ^ ((r0 + 1) & 7)) << 2) + (r & 3))];
                  v.z = st[(r0 + 2) * 32 + ((((r >> 2) ^ ((r0 + 2) & 7)) << 2) + (r & 3))];
                  v.w = st[(r0 + 3) * 32 + ((((r >> 2) ^ ((r0 + 3) & 7)) << 2) + (r & 3))];
                  mm = n0 + r;
                  nn = m0 + r0;
                }
                emit4(o, mm, nn, v);
              }
              __syncwarp();
              if (rtrace && b == ew) g_gemm_trace[10] = clock64();
            }
            if (threadIdx.x == 64 && p.groups > 1) cnt[p.groups] = 0;
            if (rtrace) g_gemm_trace[11] = clock64();
          }
          if (threadIdx.x == 64) cnt[g] = 0;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// reduce split-K partials (and mirror symmetric results), then the shared epilogue.  Block (256 / L columns, L split
// lanes), L in {1, 2, 4, 8}: the split lanes are combined through shared memory in a fixed order (deterministic).
__global__ void __launch_bounds__(256) gemm_finalize_kernel(OutParams o, const float* __restrict__ ws, int ws_ld,
                                                            long long ws_split_stride, int splits, int symmetric, int bm,
                                                            int bn) {
  __shared__ float red[256];
  pdl_wait();
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int m = blockIdx.y;
  float acc = 0.0f;
  if (n < o.n) {
    int mm = m, nn = n;
    if (symmetric && (m / bm) > (n / bn)) {
      mm = n;
      nn = m;
    }
    const float* src = ws + (size_t)mm * ws_ld + nn;
    // four independent partial sums per thread: the loads of a thread do not depend on each other, and without them one
    // L2 round trip per split bounds this (tiny-grid) kernel
    const int L = blockDim.y;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int s = threadIdx.y;
    for (; s + 3 * L < splits; s += 4 * L) {
      a0 += src[(size_t)s * ws_split_stride];
      a1 += src[(size_t)(s + L) * ws_split_stride];
      a2 += src[(size_t)(s + 2 * L) * ws_split_stride];
      a3 += src[(size_t)(s + 3 * L) * ws_split_stride];
    }
    for (; s < splits; s += L) a0 += src[(size_t)s * ws_split_stride];
    acc = (a0 + a1) + (a2 + a3);
  }
  if (blockDim.y > 1) {
    red[threadIdx.y * blockDim.x + threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0) {
      acc = 0.f;
      for (int k = 0; k < (int)blockDim.y; ++k) acc += red[k * blockDim.x + threadIdx.x];
    }
  }
  if (threadIdx.y == 0 && n < o.n) store_value(o, m, n, finish_value(o, m, n, acc));
}

// the same reduction for the common aligned case (n, every leading dimension a multiple of 4, no mirroring): a thread
// owns 4 consecutive columns of one row - 16-byte loads of the partials with four splits in flight, one 16-byte fp32
// store and one 8-byte store per bf16 plane instead of scalar accesses (the scalar kernel above spent 11-12 us on a
// 672 x 512 result; this one is bound by the launch and one L2 round trip).  Fixed association order: deterministic.
__global__ void __launch_bounds__(256) gemm_finalize_vec4_kernel(OutParams o, const float* __restrict__ ws, int ws_ld,
                                                                 long long ws_split_stride, int splits) {
  pdl_wait();
  const int nq = (o.n + 3) >> 2;   // a ragged last quad is allowed for plane-only outputs whose rows are padded (see below)
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= (long long)o.m * nq) return;
  const int m = (int)(i / nq), n = (int)(i - (long long)m * nq) << 2;
  const float4* src = reinterpret_cast<const float4*>(ws + (size_t)m * ws_ld + n);
  const size_t st4 = (size_t)(ws_split_stride >> 2);
  float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
  int s = 0;
  for (; s + 3 < splits; s += 4) {
    const float4 x0 = src[(size_t)s * st4], x1 = src[(size_t)(s + 1) * st4], x2 = src[(size_t)(s + 2) * st4],
                 x3 = src[(size_t)(s + 3) * st4];
    a0.x += x0.x; a0.y += x0.y; a0.z += x0.z; a0.w += x0.w;
    a1.x += x1.x; a1.y += x1.y; a1.z += x1.z; a1.w += x1.w;
    a2.x += x2.x; a2.y += x2.y; a2.z += x2.z; a2.w += x2.w;
    a3.x += x3.x; a3.y += x3.y; a3.z += x3.z; a3.w += x3.w;
  }
  for (; s < splits; ++s) {
    const float4 x0 = src[(size_t)s * st4];
    a0.x += x0.x; a0.y += x0.y; a0.z += x0.z; a0.w += x0.w;
  }
  float v[4] = {(a0.x + a1.x) + (a2.x + a3.x), (a0.y + a1.y) + (a2.y + a3.y), (a0.z + a1.z) + (a2.z + a3.z),
                (a0.w + a1.w) + (a2.w + a3.w)};
  float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (o.bias) b4 = __ldg(reinterpret_cast<const float4*>(o.bias + n));
  v[0] = o.alpha * v[0];
  v[1] = o.alpha * v[1];
  v[2] = o.alpha * v[2];
  v[3] = o.alpha * v[3];
  if (o.bias) {
    v[0] += b4.x;
    v[1] += b4.y;
    v[2] += b4.z;
    v[3] += b4.w;
  }
  if (o.relu) {
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.0f);
  }
  if (o.mask) {
    const uint2 mw = __ldg(reinterpret_cast<const uint2*>(o.mask + (size_t)(m % o.mask_rows) * o.mask_ld + n));
    if (!(__uint_as_float(mw.x << 16) > 0.0f)) v[0] = 0.0f;
    if (!(__uint_as_float(mw.x & 0xffff0000u) > 0.0f)) v[1] = 0.0f;
    if (!(__uint_as_float(mw.y << 16) > 0.0f)) v[2] = 0.0f;
    if (!(__uint_as_float(mw.y & 0xffff0000u) > 0.0f)) v[3] = 0.0f;
  }
  const int ms = o.perm_m ? perm64(m) : m, ns = o.perm_n ? perm64(n) : n;
  if (o.c) *reinterpret_cast<float4*>(o.c + (size_t)ms * o.ldc + ns) = make_float4(v[0], v[1], v[2], v[3]);
  if (o.c_num_planes > 0) {
    if (n + 3 >= o.n) {   // ragged last quad: the padding columns of the planes are kept zero
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (n + j >= o.n) v[j] = 0.0f;
    }
    uint2 ph, pm, pl;
    split3x4(v[0], v[1], v[2], v[3], ph, pm, pl);
    const size_t idx = (size_t)ms * o.ldcp + ns;
    *reinterpret_cast<uint2*>(o.cp[0] + idx) = ph;
    if (o.c_num_planes > 1) *reinterpret_cast<uint2*>(o.cp[1] + idx) = pm;
    if (o.c_num_planes > 2) *reinterpret_cast<uint2*>(o.cp[2] + idx) = pl;
  }
}
static bool finalize_vec4_ok(const OutParams& o, int ws_ld, long long ws_split_stride) {
  auto al = [](const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; };
  if ((ws_ld & 3) || (ws_split_stride & 3)) return false;
  if (o.n & 3) {   // ragged width: only plane outputs whose padded rows hold the whole last quad, nothing read per column
    if (o.c || o.bias || o.mask || o.c_num_planes == 0 || o.ldcp < ((o.n + 3) & ~3) || ws_ld < ((o.n + 3) & ~3)) return false;
  }
  if (o.c && ((o.ldc & 3) || !al(o.c, 16))) return false;
  if (o.bias && !al(o.bias, 16)) return false;
  if (o.mask && ((o.mask_ld & 3) || !al(o.mask, 8))) return false;
  if (o.c_num_planes > 0) {
    if (o.ldcp & 3) return false;
    for (int i = 0; i < o.c_num_planes; ++i)
      if (!al(o.cp[i], 8)) return false;
  }
  return true;
}

// symmetric results: only upper 128-tiles were computed.  Four CTAs (32 x 8 threads, one row quarter each) per 32 x 32 block
// pair (bi <= bj): every thread reduces 1 element of the upper block over the splits (row-contiguous, independent loads),
// stores it, and the 8 x 32 strip is transposed through shared memory and stored again as part of the mirrored block.
__global__ void __launch_bounds__(1024) gemm_finalize_sym_kernel(OutParams o, const float* __restrict__ ws, int ws_ld,
                                                                 long long ws_split_stride, int splits, int nblk) {
  // blockDim = (256, L): L split lanes per element (deep splits - the conv1 panel SYRK has 143 - need more loads in flight
  // than one thread per element provides); lane z sums splits z, z + L, ... and the lanes are combined in lane order
  __shared__ float tile[8][33];
  __shared__ float red[3][256];
  pdl_wait();
  int t = blockIdx.x, bi = 0, cnt = nblk;
  while (t >= cnt) {
    t -= cnt;
    ++bi;
    --cnt;
  }
  const int bj = bi + t;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int L = blockDim.y, tz = threadIdx.y;
  const int r0 = blockIdx.y * 8;   // row quarter of the block
  {
    const int m = bi * 32 + r0 + ty, n = bj * 32 + tx;
    float acc = 0.0f;
    const bool in = m < o.m && n < o.n;
    if (in) {
      const float* src = ws + (size_t)m * ws_ld + n;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f, a5 = 0.f, a6 = 0.f, a7 = 0.f;
      int s = tz;
      for (; s + 7 * L < splits; s += 8 * L) {   // fixed association order: deterministic; 8 loads in flight per thread
        a0 += src[(size_t)s * ws_split_stride];
        a1 += src[(size_t)(s + L) * ws_split_stride];
        a2 += src[(size_t)(s + 2 * L) * ws_split_stride];
        a3 += src[(size_t)(s + 3 * L) * ws_split_stride];
        a4 += src[(size_t)(s + 4 * L) * ws_split_stride];
        a5 += src[(size_t)(s + 5 * L) * ws_split_stride];
        a6 += src[(size_t)(s + 6 * L) * ws_split_stride];
        a7 += src[(size_t)(s + 7 * L) * ws_split_stride];
      }
      for (; s < splits; s += L) a0 += src[(size_t)s * ws_split_stride];
      acc = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    }
    if (L > 1) {
      if (tz > 0) red[tz - 1][threadIdx.x] = acc;
      __syncthreads();
      if (tz == 0)
        for (int z = 1; z < L; ++z) acc += red[z - 1][threadIdx.x];
    }
    if (tz == 0) {
      if (in) store_value(o, m, n, finish_value(o, m, n, acc));
      tile[ty][tx] = acc;
    }
  }
  if (bi == bj) return;
  __syncthreads();
  if (tz != 0) return;
  // mirrored strip: rows bj*32 + (0..31), columns bi*32 + r0 + (0..7)
  {
    const int e = threadIdx.x;
    const int rr = e >> 3, cc = e & 7;
    const int m = bj * 32 + rr, n = bi * 32 + r0 + cc;
    if (m < o.m && n < o.n) store_value(o, m, n, finish_value(o, m, n, tile[cc][rr]));
  }
}

// ------------------------------------------------------------------------------------------------
// SIMT fp32 reference on the same planes (validation / debug only)
// ------------------------------------------------------------------------------------------------
struct SimtParams {
  OutParams out;
  const bf16* a[ACX_MAX_PLANES];
  const bf16* b[ACX_MAX_PLANES];
  int lda, ldb, trans_a, trans_b, k;
  int num_pairs;
  int pair_a[6], pair_b[6];
};

__global__ void __launch_bounds__(256) gemm_simt_kernel(SimtParams p) {
  __shared__ float as[16][65];
  __shared__ float bs[16][65];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int pr = 0; pr < p.num_pairs; ++pr) {
    const bf16* A = p.a[p.pair_a[pr]];
    const bf16* B = p.b[p.pair_b[pr]];
    for (int k0 = 0; k0 < p.k; k0 += 16) {
      for (int i = threadIdx.x; i < 16 * 64; i += 256) {
        const int kk = i / 64, r = i % 64;  // generic gather; speed is irrelevant here
        const int k = k0 + kk;
        float av = 0.f, bv = 0.f;
        if (k < p.k) {
          const int m = m0 + r, n = n0 + r;
          if (m < p.out.m) av = __bfloat162float(p.trans_a ? A[(size_t)k * p.lda + m] : A[(size_t)m * p.lda + k]);
          if (n < p.out.n) bv = __bfloat162float(p.trans_b ? B[(size_t)k * p.ldb + n] : B[(size_t)n * p.ldb + k]);
        }
        as[kk][r] = av;
        bs[kk][r] = bv;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < 16; ++kk) {
        float a4[4], b4[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          a4[i] = as[kk][ty + 16 * i];
          b4[i] = bs[kk][tx + 16 * i];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty + 16 * i, n = n0 + tx + 16 * j;
      if (m < p.out.m && n < p.out.n) store_value(p.out, m, n, finish_value(p.out, m, n, acc[i][j]));
    }
}

__global__ void split_planes_kernel(const float* __restrict__ in, int ld_in, int rows, int cols, float scale, bf16* p0,
                                    bf16* p1, bf16* p2, int num_planes, int ld_out) {
  pdl_enter();
  const size_t total = (size_t)rows * ld_out;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / ld_out), c = (int)(i % ld_out);
    float x = c < cols ? in[(size_t)r * ld_in + c] * scale : 0.0f;
    bf16 a, b, d;
    split3(x, a, b, d);
    p0[i] = a;
    if (num_planes > 1) p1[i] = b;
    if (num_planes > 2) p2[i] = d;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  });
  return fn;
}

struct MapKey {
  const void* ptr;
  int rows, cols, ld, box0, box1;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box0 == o.box0 && box1 == o.box1;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h = h * 1000003u ^ (size_t)k.rows;
    h = h * 1000003u ^ (size_t)k.cols;
    h = h * 1000003u ^ (size_t)k.ld;
    h = h * 1000003u ^ (size_t)(k.box0 * 4096 + k.box1);
    return h;
  }
};
static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;
static std::mutex g_maps_mu;

// row-major bf16 [rows, cols] with leading dimension ld; box = box0 columns x box1 rows; the swizzle span is the box row
// (64 columns: 128B, 32 columns: 64B)
static int get_tensor_map(const void* ptr, int rows, int cols, int ld, int box0, int box1, CUtensorMap* out) {
  MapKey key{ptr, rows, cols, ld, box0, box1};
  std::lock_guard<std::mutex> lock(g_maps_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) {
    *out = it->second;
    return 0;
  }
  EncodeTiledFn fn = get_encode_fn();
  ACX_CHECK(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  ACX_CHECK((ld % 8) == 0, "plane leading dimension must be a multiple of 8 bf16 elements");
  ACX_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "plane pointer must be 16-byte aligned");
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box0, (cuuint32_t)box1};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, box0 == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  ACX_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
  if (g_maps.size() > 4096) g_maps.clear();
  g_maps[key] = m;
  *out = m;
  return 0;
}

static uint32_t g_mn_lbo = 0, g_mn_sbo = 0, g_mn_kstep = 0;

static void fill_out(const acx_gemm_t* g, OutParams* o) {
  o->m = g->m;
  o->n = g->n;
  o->alpha = g->alpha;
  o->bias = g->bias;
  o->relu = g->relu;
  o->c = g->c;
  o->ldc = g->ldc;
  for (int i = 0; i < ACX_MAX_PLANES; ++i) o->cp[i] = reinterpret_cast<bf16*>(g->c_planes[i]);
  o->c_num_planes = g->c_num_planes;
  o->ldcp = g->ldc_planes;
  o->mask = reinterpret_cast<const bf16*>(g->mask_plane);
  o->mask_ld = g->mask_ld;
  o->mask_rows = g->mask_rows > 0 ? g->mask_rows : (g->m > 0 ? g->m : 1);
  o->perm_m = g->perm_m;
  o->perm_n = g->perm_n;
}

struct TcPlan {
  int bn, bk, npa, npb, stages, tiles_m, tiles_n, splits, kb_total, kb_per_split, to_ws, panel;
  int g_bx, g_by, g_ts, g_nx, g_cells;   // gathered operands: the box of 64 locations that makes one k-block
  int fuse, groups;            // split-K reduction inside the kernel
  size_t part_bytes;           // the split partials
  size_t ws_bytes;
};
static int g_fuse_mode = -1;
static int fuse_reduce_enabled() {   // ACX_GEMM_FUSE_REDUCE / acx_debug_set_fuse_reduce: 0 = finalize launches, 1 = where cheap, 2 = always
  if (g_fuse_mode < 0) {
    const char* e = getenv("ACX_GEMM_FUSE_REDUCE");
    g_fuse_mode = e ? atoi(e) : 0;
  }
  return g_fuse_mode;
}

constexpr int SMEM_LIMIT = 232448;                       // 227 KB per CTA on sm_100
constexpr int SMEM_FIXED = EPI_BYTES + 256;              // epilogue staging + barriers (the base is 1024-aligned)
static int bk128_min_stages() {   // ACX_GEMM_BK128_STAGES: ring depth from which 128-deep k-blocks are chosen automatically (0 = never)
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("ACX_GEMM_BK128_STAGES");
    v = e ? atoi(e) : 2;   // measured at 32 x 20: never 0.689, >= 3 stages 0.682, >= 2 stages 0.674 ms/update
    if (v <= 0) v = 1000;
  }
  return v;
}
static int force_bk() {                                  // tuning knob: ACX_GEMM_BK=32 / 64 overrides the automatic k-block depth
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("ACX_GEMM_BK");
    v = e ? atoi(e) : 0;
  }
  return v;
}

static int pick_bn(const acx_gemm_t* g) {
  if (g->symmetric) return g->n <= 64 ? 64 : 128;   // one tile (0,0) when n <= 64; otherwise square 128-tiles
  if (g->trans_a) return g->n <= 64 ? 64 : 128;
  if (g->n <= 32) return 32;
  if (g->n <= 64) return 64;
  return 128;
}

static void plan_tc(const acx_gemm_t* g, TcPlan* pl) {
  pl->bn = pick_bn(g);
  pl->tiles_m = ceil_div(g->m, BM);
  pl->tiles_n = ceil_div(g->n, pl->bn);
  int tiles = pl->tiles_m * pl->tiles_n;
  if (g->symmetric) tiles = pl->tiles_n * (pl->tiles_n + 1) / 2;
  // SYRK panel mode: X^T X with 128 < n <= 256 (MN-major): every CTA streams its k-range of X once and feeds all three
  // upper sub-tiles from the same shared memory
  const bool same_operand = g->a_gather ? (g->b_gather == nullptr || g->b_gather == g->a_gather) : g->a.planes[0] == g->b.planes[0];
  pl->panel = (g->symmetric && g->trans_a && pl->bn == 128 && pl->tiles_n == 2 && same_operand) ? 1 : 0;
  if (pl->panel) tiles = 1;
  // planes each side loads per k-block, and the ring depth they leave
  pl->npa = pl->npb = 1;
  for (int i = 0; i < g->num_pairs && i < 6; ++i) {
    pl->npa = g->pair_a[i] + 1 > pl->npa ? g->pair_a[i] + 1 : pl->npa;
    pl->npb = g->pair_b[i] + 1 > pl->npb ? g->pair_b[i] + 1 : pl->npb;
  }
  if (pl->panel && pl->npb > pl->npa) pl->npa = pl->npb;   // one plane set serves both operand sides
  auto stages_for = [&](int bk) {
    const int stage_bytes = pl->panel ? pl->npa * 4 * bk * 128 : (pl->npa * BM + pl->npb * pl->bn) * bk * 2;
    const int st = (SMEM_LIMIT - SMEM_FIXED) / stage_bytes;
    return st > MAX_STAGES ? MAX_STAGES : st;
  };
  // Measured at 32 x 20 (ACX_GEMM_BK=32): halving the k-block to get 4-5 ring stages instead of 2 for the 3 + 3 plane GEMMs
  // is SLOWER (1.26 vs 1.16 ms/update): twice the stage hand-offs, and 64-byte swizzle rows; so 64 unless asked.
  pl->bk = (force_bk() == 32 && !g->a_gather) ? 32 : BK;
  // 128-deep k-blocks for MN-major products whose stages are small (the deep-split conv weight gradients and output-factor
  // SYRKs: 8 MMAs per 64-deep k-block): the hand-off between producer, issuing thread and tensor pipe costs ~250 cycles per
  // k-block whatever its depth (tools/micro/mma_rate3.cu).  ACX_GEMM_BK=128 forces it wherever two stages fit, =64 forbids it.
  if (g->trans_a && force_bk() != 64 && force_bk() != 32) {
    const int st128 = stages_for(128);
    if (force_bk() == 128 ? st128 >= 2 : st128 >= bk128_min_stages()) pl->bk = 128;
  }
  pl->stages = stages_for(pl->bk);
  pl->kb_total = ceil_div(g->k, pl->bk);
  pl->g_bx = pl->g_by = pl->g_ts = pl->g_nx = pl->g_cells = 0;
  if (g->a_gather) {
    // one k-block = 64 locations = a box of bx x by grid cells (powers of two that divide the grid) of ts samples;
    // sample groups beyond the batch read as zero rows
    const acx_gather_t* ga = g->a_gather;
    int bx = 1, by = 1;
    while (bx < 8 && ga->gx % (2 * bx) == 0) bx *= 2;
    while (bx * by < pl->bk && ga->gy % (2 * by) == 0) by *= 2;
    if (const char* e = getenv("ACX_GATHER_CUT")) {   // triage: "bx,by" (powers of two; boxes that overhang the grid read zero rows)
      int a = 0, b = 0;
      if (sscanf(e, "%d,%d", &a, &b) == 2 && a >= 1 && b >= 1 && a * b <= pl->bk && (a & (a - 1)) == 0 && (b & (b - 1)) == 0) {
        bx = a;
        by = b;
      }
    }
    pl->g_bx = bx;
    pl->g_by = by;
    pl->g_ts = pl->bk / (bx * by);
    pl->g_nx = ceil_div(ga->gx, bx);
    pl->g_cells = pl->g_nx * ceil_div(ga->gy, by);
    pl->kb_total = pl->g_cells * ceil_div(ga->samples, pl->g_ts);
  }
  int splits = g->splits;
  if (splits <= 0) {  // auto: about one work item per SM, at least 256 elements of K per split
    splits = 148 / (tiles > 0 ? tiles : 1);
    int cap = (int)((long long)pl->kb_total * pl->bk / 256);   // at least 256 elements of K per split
    if (splits > cap) splits = cap;
    if (splits < 1) splits = 1;
  }
  if (splits > pl->kb_total) splits = pl->kb_total;
  if (g->splits <= 0 && fuse_reduce_enabled() == 1 && !pl->panel) {
    // shallow products (a handful of k-blocks per split: fc4 forward, the preconditioning GEMMs) are bound by pipeline
    // fill, not by the number of CTAs: fewer splits, so that the reduction stays inside the kernel
    const int max_fused = (int)(kFusedReduceBytes / ((size_t)BM * pl->bn * sizeof(float)));
    if (splits > max_fused && pl->kb_total <= 8 * max_fused) splits = max_fused;
  }
  pl->kb_per_split = ceil_div(pl->kb_total, splits);
  pl->splits = ceil_div(pl->kb_total, pl->kb_per_split);
  pl->to_ws = (pl->splits > 1 || g->symmetric) ? 1 : 0;
  const size_t plane_bytes = (size_t)pl->tiles_m * BM * pl->tiles_n * pl->bn * sizeof(float);
  pl->part_bytes = pl->to_ws ? (size_t)pl->splits * plane_bytes : 0;
  pl->groups = ceil_div(pl->splits, RED_GROUP);
  const int num_tiles = pl->panel ? 1 : tiles;
  // The reduction runs inside the kernel where ONE SM can sum a tile's partials in a few microseconds (measured: a single
  // SM reads its peers' partials at some tens of GB/s, so deep splits of large tiles - the conv factor SYRKs and weight
  // gradients - reduce faster in a finalize launch that spreads the sums over all SMs: 0.80 vs 1.32 ms/update with
  // everything fused).  ACX_GEMM_FUSE_REDUCE: 0 = never (default), 1 = where cheap, 2 = always (two-level for > 8 splits).
  const size_t tile_bytes = (size_t)(pl->panel ? 4 : 1) * BM * pl->bn * sizeof(float);
  const bool cheap = pl->groups == 1 && (size_t)pl->splits * tile_bytes <= kFusedReduceBytes;
  const int mode = fuse_reduce_enabled();
  pl->fuse = (pl->to_ws && (mode >= 2 || (mode == 1 && cheap)) &&
              (long long)num_tiles * (pl->groups + 1) * (long long)sizeof(int) <= RED_COUNTER_BYTES) ? 1 : 0;
  // workspace: [counters (zero on entry, left zero) | split partials | group sums (two-level fused reduction only)]
  pl->ws_bytes = pl->to_ws ? RED_COUNTER_BYTES + pl->part_bytes + (pl->fuse && pl->groups > 1 ? (size_t)pl->groups * plane_bytes : 0) : 0;
}

// optional timing probe: when enabled, every tensor-core kernel launch (the kernel alone, not the finalize step) is
// bracketed by two library-owned events on the launching stream; acx_gemm_last_ms() reads the last pair
static bool g_probe_on = false;
static cudaEvent_t g_probe_ev[2] = {nullptr, nullptr};

template <int MAJOR>
static int launch_tc(const CUtensorMap* ta, const CUtensorMap* tb, const TcParams& p, int grid, int smem, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    ACX_CUDA((cudaFuncSetAttribute(gemm_tc_kernel<MAJOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT)));
    configured = true;
  }
  if (g_probe_on) ACX_CUDA(cudaEventRecord(g_probe_ev[0], st));
  ACX_CUDA(launch_pdl(gemm_tc_kernel<MAJOR>, dim3(grid), dim3(GEMM_THREADS), (size_t)smem, st, ta[0], ta[1], ta[2], tb[0], tb[1],
                      tb[2], p));
    acx::count_launch();
  if (g_probe_on) ACX_CUDA(cudaEventRecord(g_probe_ev[1], st));
  return 0;
}

static int g_pdl_override = -1;
void set_pdl_override(int level) { g_pdl_override = level; }
int pdl_level() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("ACX_PDL");
    v = e ? atoi(e) : 1;
  }
  return (v > 0 && g_pdl_override >= 0) ? g_pdl_override : v;
}

// cap on the persistent grid of the next tensor-core launches (learner.cu: lane 0 of K-FAC learners), so that kernels of
// different lanes can share the SMs instead of queueing behind each other (0 = all SMs)
int g_cta_cap = 0;
void set_cta_cap(int cap) { g_cta_cap = cap; }

static int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

static int validate(const acx_gemm_t* g) {
  ACX_CHECK(g != nullptr, "null gemm");
  ACX_CHECK(g->m > 0 && g->n > 0 && g->k > 0, "empty problem");
  ACX_CHECK(g->num_pairs >= 1 && g->num_pairs <= 6, "num_pairs out of range");
  const acx_gather_t* gb_eff = g->b_gather ? g->b_gather : ((g->a_gather && g->symmetric) ? g->a_gather : nullptr);
  const int a_np = g->a_gather ? g->a_gather->num_planes : g->a.num_planes;
  const int b_np = gb_eff ? gb_eff->num_planes : g->b.num_planes;
  ACX_CHECK(a_np >= 1 && a_np <= ACX_MAX_PLANES, "a.num_planes");
  ACX_CHECK(b_np >= 1 && b_np <= ACX_MAX_PLANES, "b.num_planes");
  for (int i = 0; i < g->num_pairs; ++i) {
    ACX_CHECK(g->pair_a[i] >= 0 && g->pair_a[i] < a_np, "pair_a index");
    ACX_CHECK(g->pair_b[i] >= 0 && g->pair_b[i] < b_np, "pair_b index");
  }
  if (g->a_gather || g->b_gather) {
    const acx_gather_t* ga = g->a_gather;
    ACX_CHECK(ga != nullptr && gb_eff != nullptr, "gathered operands: both sides must be gathered (or the product symmetric with B = A)");
    ACX_CHECK(g->trans_a == 1 && g->trans_b == 1, "gathered operands are MN-major (trans_a = trans_b = 1)");
    ACX_CHECK(ga->gx >= 1 && ga->gy >= 1 && ga->samples >= 1 && (long long)ga->samples * ga->gx * ga->gy == (long long)g->k,
              "gathered operands: k must be samples * gy * gx");
    ACX_CHECK(gb_eff->gx == ga->gx && gb_eff->gy == ga->gy && gb_eff->samples == ga->samples, "gathered operands: A and B enumerate different locations");
    ACX_CHECK(ga->num_chunks >= 1 && ga->num_chunks <= 16 && g->m <= 64 * ga->num_chunks, "a_gather: m exceeds 64 * num_chunks");
    ACX_CHECK(gb_eff->num_chunks >= 1 && gb_eff->num_chunks <= 16 && g->n <= 64 * gb_eff->num_chunks, "b_gather: n exceeds 64 * num_chunks");
  }
  if (g->perm_m || g->perm_n) ACX_CHECK(g->bias == nullptr && g->mask_plane == nullptr, "perm_m / perm_n: no bias or mask");
  ACX_CHECK(g->trans_a == g->trans_b, "only (K-major,K-major) and (MN-major,MN-major) operand pairs are supported");
  ACX_CHECK(g->c != nullptr || g->c_num_planes > 0, "no output requested");
  ACX_CHECK(g->c_num_planes >= 0 && g->c_num_planes <= ACX_MAX_PLANES, "c_num_planes");
  if (g->symmetric) ACX_CHECK(g->m == g->n, "symmetric needs m == n");
  return 0;
}

static int gemm_tc(const acx_gemm_t* g, cudaStream_t st) {
  TcPlan pl;
  plan_tc(g, &pl);
  if (pl.to_ws) {
    ACX_CHECK(g->workspace != nullptr && g->workspace_bytes >= pl.ws_bytes, "split-K / symmetric GEMM needs workspace");
  }
  CUtensorMap ta[3], tb[3];
  const int major = g->trans_a ? 1 : 0;
  const acx_gather_t* ga = g->a_gather;
  const acx_gather_t* gb = ga ? (g->b_gather ? g->b_gather : ga) : nullptr;
  for (int i = 0; i < 3 && ga; ++i) {   // gathered operands: 5-D views, one box = the 64 locations of a k-block x one 64-column chunk
    const int box[5] = {64, pl.g_bx, 1, pl.g_by, pl.g_ts};
    int r = get_view_map(ga->planes[i < ga->num_planes ? i : 0], 5, ga->dim, ga->stride_bytes, box, 128, &ta[i]);
    if (r) return r;
    r = get_view_map(gb->planes[i < gb->num_planes ? i : 0], 5, gb->dim, gb->stride_bytes, box, 128, &tb[i]);
    if (r) return r;
  }
  for (int i = 0; i < 3 && !ga; ++i) {
    const int ia = i < g->a.num_planes ? i : 0, ib = i < g->b.num_planes ? i : 0;
    int r = major == 0 ? get_tensor_map(g->b.planes[ib], g->n, g->k, g->b.ld, pl.bk, pl.bn, &tb[i])
                       : get_tensor_map(g->b.planes[ib], g->k, g->n, g->b.ld, 64, pl.bk, &tb[i]);
    if (r) return r;
    r = major == 0 ? get_tensor_map(g->a.planes[ia], g->m, g->k, g->a.ld, pl.bk, BM, &ta[i])
                   : get_tensor_map(g->a.planes[ia], g->k, g->m, g->a.ld, 64, pl.bk, &ta[i]);
    if (r) return r;
  }
  TcParams p;
  fill_out(g, &p.out);
  p.k = ga ? pl.kb_total * pl.bk : g->k;   // gathered: every k-block is whole (locations beyond the batch read as zero rows)
  p.kb_total = pl.kb_total;
  p.kb_per_split = pl.kb_per_split;
  {
    const bool one = ga ? (g->b_gather == nullptr || g->b_gather == g->a_gather) : (g->a.planes[0] == g->b.planes[0] && g->a.ld == g->b.ld);
    static int dg = -1;
    if (dg < 0) {
      const char* e = getenv("ACX_SYRK_DIAG");   // 0: diagonal tiles load both operand sides (round 1)
      dg = e ? atoi(e) : 1;
    }
    p.same_operand = (dg && g->symmetric && major == 1 && one && pl.npa >= pl.npb) ? 1 : 0;
  }
  p.gather_a = p.gather_b = ga ? 1 : 0;
  p.g_cells = pl.g_cells;
  p.g_nx = pl.g_nx;
  p.g_bx = pl.g_bx;
  p.g_by = pl.g_by;
  p.g_ts = pl.g_ts;
  memset(p.ga, 0, sizeof(p.ga));
  memset(p.gb, 0, sizeof(p.gb));
  if (ga) {
    for (int q = 0; q < 16; ++q) {
      p.ga[0][q] = ga->c0[q]; p.ga[1][q] = ga->c1[q]; p.ga[2][q] = ga->c2[q]; p.ga[3][q] = ga->c3[q];
      p.gb[0][q] = gb->c0[q]; p.gb[1][q] = gb->c1[q]; p.gb[2][q] = gb->c2[q]; p.gb[3][q] = gb->c3[q];
    }
  }
  p.num_pairs = g->num_pairs;
  for (int i = 0; i < 6; ++i) {
    p.pair_a[i] = g->pair_a[i];
    p.pair_b[i] = g->pair_b[i];
  }
  p.npa = pl.npa;
  p.npb = pl.npb;
  p.bn = pl.bn;
  p.bk = pl.bk;
  p.panel = pl.panel;
  const int stage_bytes = pl.panel ? p.npa * 4 * pl.bk * 128 : (p.npa * BM + p.npb * pl.bn) * pl.bk * 2;
  p.stages = pl.stages;
  ACX_CHECK(p.stages >= 2, "tile does not fit the shared-memory ring");
  p.tiles_m = pl.tiles_m;
  p.tiles_n = pl.tiles_n;
  p.num_tiles = pl.panel ? 1 : (g->symmetric ? pl.tiles_n * (pl.tiles_n + 1) / 2 : pl.tiles_m * pl.tiles_n);
  p.splits = pl.splits;
  p.total_work = p.num_tiles * pl.splits;
  p.symmetric = g->symmetric;
  p.to_workspace = pl.to_ws;
  p.ws_ld = pl.tiles_n * pl.bn;
  p.ws_split_stride = (long long)pl.tiles_m * BM * p.ws_ld;
  p.fuse = pl.fuse;
  p.groups = pl.groups;
  p.counters = reinterpret_cast<int*>(g->workspace);
  p.ws = g->workspace + RED_COUNTER_BYTES / sizeof(float);   // partials always start behind the counter head
  p.ws2 = p.ws + (size_t)pl.splits * p.ws_split_stride;
  p.ws2_stride = p.ws_split_stride;
  {
    static int tr = -1;
    if (tr < 0) {
      const char* e = getenv("ACX_GEMM_TRACE");
      tr = e ? atoi(e) : 0;
    }
    p.trace = tr;
  }
  p.mn_lbo = g_mn_lbo ? g_mn_lbo : (uint32_t)(pl.bk * 128);
  p.mn_sbo = g_mn_sbo ? g_mn_sbo : 1024u;
  p.mn_kstep = g_mn_kstep ? g_mn_kstep : 2048u;
  int grid = p.total_work < num_sms() ? p.total_work : num_sms();
  if (g_cta_cap > 0 && grid > g_cta_cap) grid = g_cta_cap;
  grid = ceil_div(p.total_work, ceil_div(p.total_work, grid));   // the smallest grid with the same number of rounds
  const int smem = SMEM_FIXED + p.stages * stage_bytes;
  const int r = major == 0 ? launch_tc<0>(ta, tb, p, grid, smem, st) : launch_tc<1>(ta, tb, p, grid, smem, st);
  if (r) return r;
  if (pl.fuse) return 0;   // the kernel reduced and finished its own split-K partials
  if (pl.to_ws && g->symmetric && g->n > 64) {
    const int nblk = ceil_div(g->n, 32);
    const int zl = pl.splits >= 64 ? 4 : (pl.splits >= 24 ? 2 : 1);   // split lanes per element
    ACX_CUDA(launch_pdl(gemm_finalize_sym_kernel, dim3(nblk * (nblk + 1) / 2, 4), dim3(256, zl), 0, st, p.out, (const float*)p.ws, p.ws_ld,
                        p.ws_split_stride, pl.splits, nblk));
    acx::count_launch();
  } else if (pl.to_ws && !g->symmetric && pl.splits <= 16 && finalize_vec4_ok(p.out, p.ws_ld, p.ws_split_stride)) {
    // (deep split-K of a small result - the conv wgrads - keeps the kernel whose thread lanes share the splits: measured
    // 5.4 vs 14.1 us at 146 splits of a 256 x 32 result)
    const long long quads = (long long)g->m * ((g->n + 3) >> 2);
    ACX_CUDA(launch_pdl(gemm_finalize_vec4_kernel, dim3((unsigned)((quads + 255) / 256)), dim3(256), 0, st, p.out, (const float*)p.ws, p.ws_ld,
                        p.ws_split_stride, pl.splits));
    acx::count_launch();
  } else if (pl.to_ws) {
    const int lanes = pl.splits >= 8 ? 8 : (pl.splits >= 4 ? 4 : (pl.splits >= 2 ? 2 : 1));
    dim3 fg(ceil_div(g->n, 256 / lanes), g->m);
    ACX_CUDA(launch_pdl(gemm_finalize_kernel, fg, dim3(256 / lanes, lanes), 0, st, p.out, (const float*)p.ws, p.ws_ld, p.ws_split_stride,
                        pl.splits, g->symmetric, BM, pl.bn));
    acx::count_launch();
  }
  return 0;
}

static int gemm_simt(const acx_gemm_t* g, cudaStream_t st) {
  SimtParams p;
  fill_out(g, &p.out);
  for (int i = 0; i < ACX_MAX_PLANES; ++i) {
    p.a[i] = reinterpret_cast<const bf16*>(g->a.planes[i < g->a.num_planes ? i : 0]);
    p.b[i] = reinterpret_cast<const bf16*>(g->b.planes[i < g->b.num_planes ? i : 0]);
  }
  p.lda = g->a.ld;
  p.ldb = g->b.ld;
  p.trans_a = g->trans_a;
  p.trans_b = g->trans_b;
  p.k = g->k;
  p.num_pairs = g->num_pairs;
  for (int i = 0; i < 6; ++i) {
    p.pair_a[i] = g->pair_a[i];
    p.pair_b[i] = g->pair_b[i];
  }
  dim3 grid(ceil_div(g->n, 64), ceil_div(g->m, 64));
  gemm_simt_kernel<<<grid, 256, 0, st>>>(p);
  ACX_LAUNCH_CHECK();
  return 0;
}

int gemm_dispatch(const acx_gemm_t* g, int impl, cudaStream_t st) {
  int r = validate(g);
  if (r) return r;
  return impl == 1 ? gemm_simt(g, st) : gemm_tc(g, st);
}

int split_planes(const float* in, int ld_in, int rows, int cols, float scale, bf16* p0, bf16* p1, bf16* p2, int num_planes,
                 int ld_out, cudaStream_t st) {
  ACX_CHECK(num_planes >= 1 && num_planes <= ACX_MAX_PLANES, "num_planes");
  ACX_CHECK(rows > 0 && cols > 0 && ld_out >= cols, "shape");
  const size_t total = (size_t)rows * ld_out;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  ACX_PDL_LAUNCH(split_planes_kernel, blocks, 256, 0, st, in, ld_in, rows, cols, scale, p0, p1, p2, num_planes, ld_out);
  return 0;
}

int tc_error_flag() {
  int v = 0;
  cudaMemcpyFromSymbol(&v, g_tc_error, sizeof(int));
  return v;
}

}  // namespace acx

extern "C" {

int acx_gemm(const acx_gemm_t* g, int impl, void* stream) {
  return acx::gemm_dispatch(g, impl, reinterpret_cast<cudaStream_t>(stream));
}

size_t acx_gemm_workspace_bytes(const acx_gemm_t* g) {
  acx::TcPlan pl;
  acx::plan_tc(g, &pl);
  return pl.ws_bytes;
}

int acx_split_planes(const float* d_in, int ld_in, int rows, int cols, float scale, void* const* d_planes, int num_planes,
                     int ld_out, void* stream) {
  ACX_CHECK(num_planes >= 1 && num_planes <= ACX_MAX_PLANES && d_planes != nullptr, "num_planes");
  return acx::split_planes(d_in, ld_in, rows, cols, scale, reinterpret_cast<acx::bf16*>(d_planes[0]),
                           reinterpret_cast<acx::bf16*>(num_planes > 1 ? d_planes[1] : nullptr),
                           reinterpret_cast<acx::bf16*>(num_planes > 2 ? d_planes[2] : nullptr), num_planes, ld_out,
                           reinterpret_cast<cudaStream_t>(stream));
}

void acx_debug_set_mn_desc(uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t kstep_bytes) {
  acx::g_mn_lbo = lbo_bytes;
  acx::g_mn_sbo = sbo_bytes;
  acx::g_mn_kstep = kstep_bytes;
}

void acx_debug_set_fuse_reduce(int mode) { acx::g_fuse_mode = mode; }

int acx_debug_tc_error(void) {
  int e = acx::tc_error_flag();
  if (!e) e = acx::conv_error_flag();
  return e ? e : acx::inv_resident_error_flag();
}

int acx_debug_inv_trace(long long* h_out, int count) { return acx::inv_resident_trace_read(h_out, count); }

int acx_debug_gemm_trace(long long* h_out4) {
  return cudaMemcpyFromSymbol(h_out4, acx::g_gemm_trace, 12 * sizeof(long long)) == cudaSuccess ? 0 : 1;
}

int acx_gemm_enable_timing(int enable) {
  if (enable && !acx::g_probe_on) {
    for (int i = 0; i < 2; ++i) ACX_CUDA(cudaEventCreate(&acx::g_probe_ev[i]));
    acx::g_probe_on = true;
  } else if (!enable && acx::g_probe_on) {
    for (int i = 0; i < 2; ++i) cudaEventDestroy(acx::g_probe_ev[i]);
    acx::g_probe_on = false;
  }
  return 0;
}

int acx_gemm_last_ms(float* h_ms) {
  ACX_CHECK(h_ms != nullptr, "null argument");
  ACX_CHECK(acx::g_probe_on, "timing probe is off (acx_gemm_enable_timing)");
  ACX_CUDA(cudaEventSynchronize(acx::g_probe_ev[1]));
  ACX_CUDA(cudaEventElapsedTime(h_ms, acx::g_probe_ev[0], acx::g_probe_ev[1]));
  return 0;
}

}  // extern "C"
