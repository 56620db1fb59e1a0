// Weighted gradient sums S_k = sum_b w_kb d z_b / d params of the periodic
// convolutional ansaetze (conv_1d / conv_2d, wavefunctions.py:454-615; the two
// tf.gradients of training.py:545-548 and the SWO loss gradient of 169-175) on
// the 5th-generation tensor cores.  Layers l = 0 .. L-1, h_0 = sigma,
// h_{l+1} = act(conv_l(h_l) + b_l) for l <= L-2, z = sum_{pos, c} conv_{L-1}(h_{L-1}) + b_{L-1}.
// A CTA takes G configurations at a time, laid side by side as one wrap-padded
// image (row R = xx * G * PW + g * PW + yy, conv_tc.cu), all activations in
// shared memory as two fp16 planes per value (v = v1 + v2 / S, 22 mantissa
// bits; the gradient tolerance of the suite is 1e-4 of the largest entry):
//
//   forward        D[rows, 3C] += h_l[rows + tap shift, C] x W_l[tap]       (conv_tc.cu's implicit GEMM;
//                                                                            every h_l is kept)
//   backward data  D[rows, 3C] += delta_l[rows + tap shift, C] x W_l[mirrored tap]^T
//                  the transposed convolution is the SAME implicit GEMM on the
//                  delta planes padded with (k - 1 - pad) and a weight image with
//                  mirrored taps and transposed channel matrices (tc_prep_kernel);
//                  delta_{l-1} = raw . act'(h_l)
//   weight grad    D[(split, ci), (split, co)] += h_l[rows + tap shift]^T x (w_k . delta_l)[rows]
//                  one accumulator per tap; A and B are the K-major operand planes
//                  read MN-major (the reduction runs over the rows = sites x
//                  configurations); the two splits of h are stacked along M and
//                  the two splits of w . delta along N, so ONE MMA per tap and 16
//                  rows forms all four partial products.  w . delta holds the
//                  home cells only (halo and junk rows are zero), so every site
//                  is counted once.
//   layer 0        the spin plane of conv_tc.cu (row R = the 8 sites yy .. yy + 7)
//                  read MN-major with the kernel rows as M chunks: all taps in
//                  one accumulator
//   layer L-1      delta = 1: d z / d W[tap][ci][co] = sum_pos h_{L-1}[pos][ci] for every
//                  (tap, co), backward data = the column sums `wsum` of conv_tc.cu
//
// Weight-gradient accumulators are drained per batch into the CTA's slice of
// `partials` (L2 resident); bias gradients and the last layer's sums are kept in
// per-warp shared-memory slots (one writer per slot: deterministic); a
// deterministic reduction over the CTA slices follows (launch_reduce_partials).
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include <cuda_fp16.h>

#include "common.cuh"
#include "internal.h"
#include "tc_common.cuh"

namespace cgsvmc {
namespace {

using namespace tc;

constexpr int kThreads = 256;
constexpr int kWarps = 8;
constexpr int kC = 16;                 // filters (the BASELINE networks); other widths use net.cu
constexpr int kMaxL = 12;
constexpr int kTmemCols = 512;
constexpr int kSlotCols = 2 * kC;      // one weight-gradient accumulator: columns (split, co)

struct GDesc {
  int N, X, Y, kx, ky, pad_x, pad_y, bpad_x, bpad_y, L, act, NW;
  int PH, PW, G, GW;
  int rows_out, n_tiles, rows_total, kblocks;
  int n_tensor, wbuf_bytes, n_pairs;
  const __half *w1img, *wimg, *wimg_b;
  const float *bias, *wsum;
  int64_t w_off[kMaxL], b_off[kMaxL];
  int64_t P;
};

struct GPlan {
  size_t spin, sets, set_bytes, wslot, w1, consts, wk, slots, cfg, bars, total;
  int n_sets, slot_floats;
};

__host__ __device__ inline GPlan gplan(const GDesc& d, int KW) {
  GPlan p;
  size_t off = 0;
  p.spin = off; off += (size_t)d.rows_total * 16;
  p.set_bytes = (size_t)4 * d.rows_total * 16;       // [chunk][split][row][8 halfs]
  p.n_sets = d.L;                                    // h_1 .. h_{L-2}, delta, w . delta
  p.sets = off; off += (size_t)p.n_sets * p.set_bytes;
  p.wslot = off; off += (size_t)d.wbuf_bytes;
  p.w1 = off; off += (size_t)d.n_pairs * 2 * 3 * kC * 16;
  p.consts = off; off += ((size_t)(d.L - 1) * kC + kC + 4) * 4;
  p.wk = off; off += (size_t)KW * d.G * 4;
  off = (off + 15) / 16 * 16;
  p.slot_floats = d.L * kC;                          // bias gradients of layers 0 .. L-2, then the sums of h_{L-1}
  p.slots = off; off += (size_t)kWarps * KW * p.slot_floats * 4;
  off = (off + 15) / 16 * 16;
  p.cfg = off; off += (size_t)d.G * d.NW * 8;
  p.bars = off; off += 64;
  // MN-major A operands of the weight gradient (layers >= 1) are read as M = 64
  // rows = 8 chunks from their start: the rows past the real ones are junk
  // accumulator rows nobody reads, but the reads must stay inside the allocation
  const size_t last_a = p.sets + (size_t)(d.L - 3) * p.set_bytes;
  const size_t span = (size_t)8 * d.rows_total * 16 + (size_t)d.rows_total * 16;
  if (last_a + span > off) off = last_a + span;
  const size_t spin_span = (size_t)16 * d.GW * 16 + (size_t)d.rows_total * 16;
  if (p.spin + spin_span > off) off = p.spin + spin_span;
  p.total = off;
  return p;
}

__device__ __forceinline__ int word_bit(const uint64_t* words, int site) {
  return (int)((words[site >> 6] >> (site & 63)) & 1ull);
}

// d act / d x through the OUTPUT h = act(x) (cos is rejected on the host)
__device__ __noinline__ float act_grad_slow(int act, float h) {
  switch (act) {
    case CGSVMC_ACT_TANH: return 1.f - h * h;
    case CGSVMC_ACT_SIGMOID: return h * (1.f - h);
    case CGSVMC_ACT_IDENTITY: return 1.f;
    case CGSVMC_ACT_EXP: return h;
    default: return 1.f + h * h;   // tan
  }
}
__device__ __noinline__ float activate_slow(int act, float x) { return tc_activate(act, x); }

// v = h1 + h2 / S for two values at once (packed conversions)
__device__ __forceinline__ void split2_pair(float a, float b, uint32_t& h1, uint32_t& h2) {
  const __half2 p1 = __floats2half2_rn(a, b);
  const float2 f1 = __half22float2(p1);
  const __half2 p2 = __floats2half2_rn((a - f1.x) * kSplitScale, (b - f1.y) * kSplitScale);
  h1 = *reinterpret_cast<const uint32_t*>(&p1);
  h2 = *reinterpret_cast<const uint32_t*>(&p2);
}

// 16 channel values -> the four 16-byte plane entries [chunk][split] of a row
struct Row16 { uint4 q[2][2]; };
__device__ __forceinline__ Row16 split_row(const float (&v)[kC]) {
  Row16 r;
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    uint32_t a[4], b[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) split2_pair(v[8 * ch + 2 * e], v[8 * ch + 2 * e + 1], a[e], b[e]);
    r.q[ch][0] = make_uint4(a[0], a[1], a[2], a[3]);
    r.q[ch][1] = make_uint4(b[0], b[1], b[2], b[3]);
  }
  return r;
}
__device__ __forceinline__ void store_row(char* set, int rows_total, int R, const Row16& r) {
#pragma unroll
  for (int ch = 0; ch < 2; ++ch)
#pragma unroll
    for (int sp = 0; sp < 2; ++sp)
      *reinterpret_cast<uint4*>(set + ((size_t)(ch * 2 + sp) * rows_total + R) * 16) = r.q[ch][sp];
}
__device__ __forceinline__ void load_row(const char* set, int rows_total, int R, float (&v)[kC]) {
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const uint4 a = *reinterpret_cast<const uint4*>(set + ((size_t)(ch * 2) * rows_total + R) * 16);
    const uint4 b = *reinterpret_cast<const uint4*>(set + ((size_t)(ch * 2 + 1) * rows_total + R) * 16);
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 fa = __half22float2(*reinterpret_cast<const __half2*>(&aw[e]));
      const float2 fb = __half22float2(*reinterpret_cast<const __half2*>(&bw[e]));
      v[8 * ch + 2 * e] = fmaf(fb.x, 1.f / kSplitScale, fa.x);
      v[8 * ch + 2 * e + 1] = fmaf(fb.y, 1.f / kSplitScale, fa.y);
    }
  }
}

// Column sums over the 32 lanes of a warp for 8 values per lane: lane l returns
// the total of column (l >> 2) & 7 (9 shuffles instead of 40).
__device__ __forceinline__ float colsum8(const float* v, int lane) {
  float a[4], b[2];
  const bool u16 = (lane & 16) != 0, u8 = (lane & 8) != 0, u4 = (lane & 4) != 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float send = u16 ? v[i] : v[i + 4], keep = u16 ? v[i + 4] : v[i];
    a[i] = keep + __shfl_xor_sync(CGSVMC_FULL_MASK, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float send = u8 ? a[i] : a[i + 2], keep = u8 ? a[i + 2] : a[i];
    b[i] = keep + __shfl_xor_sync(CGSVMC_FULL_MASK, send, 8);
  }
  float c = (u4 ? b[1] : b[0]) + __shfl_xor_sync(CGSVMC_FULL_MASK, u4 ? b[0] : b[1], 4);
  c += __shfl_xor_sync(CGSVMC_FULL_MASK, c, 2);
  c += __shfl_xor_sync(CGSVMC_FULL_MASK, c, 1);
  return c;
}
// ... and for 16 values per lane into slot[0 .. 15] (one writer per entry)
__device__ __forceinline__ void colsum16_add(const float (&v)[kC], int lane, float* slot) {
  const float c0 = colsum8(v, lane), c1 = colsum8(v + 8, lane);
  if ((lane & 3) == 0) {
    slot[(lane >> 2) & 7] += c0;
    slot[8 + ((lane >> 2) & 7)] += c1;
  }
}

__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

template <int KW>
__global__ void __launch_bounds__(kThreads, 1)
conv_grad_tc_kernel(GDesc d, const uint64_t* __restrict__ packed, const float* __restrict__ weights, int64_t B,
                    int64_t per_cta, float* __restrict__ partials) {
  extern __shared__ __align__(1024) char smem[];
  const GPlan pl = gplan(d, KW);
  char* spin = smem + pl.spin;
  char* sets = smem + pl.sets;
  const size_t set_bytes = pl.set_bytes;
  auto hset = [&](int l) { return sets + (size_t)(l - 1) * set_bytes; };   // h_l, l = 1 .. L-2
  char* dset = sets + (size_t)(d.L - 2) * set_bytes;                       // delta, padded with (k - 1 - pad)
  char* wdset = dset + set_bytes;                                          // w_k . delta, home cells only
  char* wslot = smem + pl.wslot;
  __half* w1s = reinterpret_cast<__half*>(smem + pl.w1);
  float* bias_s = reinterpret_cast<float*>(smem + pl.consts);
  float* wsum_s = bias_s + (d.L - 1) * kC;
  float* wk_s = reinterpret_cast<float*>(smem + pl.wk);
  float* slots = reinterpret_cast<float*>(smem + pl.slots);
  uint64_t* cfg = reinterpret_cast<uint64_t*>(smem + pl.cfg);
  uint64_t* mma_bar = reinterpret_cast<uint64_t*>(smem + pl.bars);
  uint64_t* wbar = mma_bar + 1;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(mma_bar + 2);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = warp & 3;
  const int act = d.act;
  const bool relu = act == CGSVMC_ACT_RELU;
  const int RT = d.rows_total;
  const int taps = d.kx * d.ky;
  float* my_slot = slots + (size_t)warp * KW * pl.slot_floats;            // [k][slot_floats]

  // ---- one-time setup ----
  {
    const size_t n16 = (pl.sets + (size_t)pl.n_sets * set_bytes - pl.spin) / 16;
    uint4* z = reinterpret_cast<uint4*>(spin);
    for (size_t e = threadIdx.x; e < n16; e += kThreads) z[e] = make_uint4(0u, 0u, 0u, 0u);
  }
  for (int e = threadIdx.x; e < d.n_pairs * 2 * 3 * kC * 4; e += kThreads)
    reinterpret_cast<uint32_t*>(w1s)[e] = reinterpret_cast<const uint32_t*>(d.w1img)[e];
  for (int e = threadIdx.x; e < (d.L - 1) * kC; e += kThreads) bias_s[e] = d.bias[e];
  for (int e = threadIdx.x; e < kC + 1; e += kThreads) wsum_s[e] = d.wsum[e];
  for (int e = threadIdx.x; e < kWarps * KW * pl.slot_floats; e += kThreads) slots[e] = 0.f;
  float* part = partials + (size_t)blockIdx.x * KW * d.P;
  for (int64_t e = threadIdx.x; e < (int64_t)KW * d.P; e += kThreads) part[e] = 0.f;
  if (threadIdx.x == 0) {
    mbar_init(mma_bar, kWarps);      // every warp commits every round (an empty commit arrives at once)
    mbar_init(wbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)),
                 "r"((uint32_t)kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_holder;
  uint32_t mma_ph = 0, w_ph = 0;
  float wtot[KW];                    // thread 0: sum of the weights of this CTA's walkers (d z / d b_{L-1} = N)
#pragma unroll
  for (int k = 0; k < KW; ++k) wtot[k] = 0.f;

  // weight images stream through one slot: forward images j = 0 .. n_tensor - 1,
  // then the backward-data images j = n_tensor - 1 .. 0
  auto load_w = [&](bool backward, int j) {
    if (threadIdx.x == 0)
      bulk_load_async(wslot, reinterpret_cast<const char*>(backward ? d.wimg_b : d.wimg) + (size_t)j * d.wbuf_bytes,
                      (uint32_t)d.wbuf_bytes, wbar);
  };
  auto wait_w = [&]() { mbar_wait(wbar, w_ph); w_ph ^= 1u; };
  auto commit_and_wait = [&]() {
    if (elect_one())
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(mma_bar))
                   : "memory");
    __syncwarp();
    mbar_wait(mma_bar, mma_ph);
    mma_ph ^= 1u;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  };
  auto sync_async = [&]() {          // generic-proxy writes -> visible to the MMAs; TMEM reads done
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  };

  const uint32_t idesc0 = (1u << 4) | (8u << 24);                 // D = F32, A = B = F16, M = 128
  const uint32_t hi_k = 8u | (1u << 14);                          // K-major: SBO = 8 units (8 rows of 16 B)
  const uint32_t plane_units = (uint32_t)RT;

  // The implicit GEMM of one convolution over every tile: A = the operand set at
  // `set` (K-major, [chunk][split] planes), B = the weight image in the slot.
  auto conv_mmas = [&](const char* set) {
    const uint32_t idesc3 = idesc0 | ((uint32_t)(3 * kC >> 3) << 17);
    const uint32_t idesc2 = idesc0 | ((uint32_t)(2 * kC >> 3) << 17);
    const uint32_t a_units = smem_u32(set) >> 4, b_units = smem_u32(wslot) >> 4;
    const uint32_t a_lbo = (2u * plane_units) << 16, b_lbo = (uint32_t)(3 * kC) << 16;
    const uint32_t b_tap_units = (uint32_t)(kC / 8) * 3 * kC;
    for (int t = warp; t < d.n_tiles; t += kWarps) {
      const uint32_t d_tmem = tmem + (uint32_t)(t * 3 * kC);
      for (int dx = 0; dx < d.kx; ++dx)
        for (int dy = 0; dy < d.ky; ++dy) {
          const int tap = dx * d.ky + dy;
          const uint32_t a_lo = (a_units + (uint32_t)(t * 128 + dx * d.GW + dy)) | a_lbo;
          const uint32_t b_lo = (b_units + (uint32_t)tap * b_tap_units) | b_lbo;
          const uint64_t a1 = ((uint64_t)hi_k << 32) | a_lo;
          const uint64_t a2 = ((uint64_t)hi_k << 32) | (a_lo + plane_units);
          const uint64_t b = ((uint64_t)hi_k << 32) | b_lo;
          if (elect_one()) {
            mma_f16(d_tmem, a1, b, idesc3, tap ? 1u : 0u);          // [P0 P1 P2] += A1 [b1 b2 b3]
            mma_f16(d_tmem + kC, a2, b, idesc2, 1u);                 // [P1 P2]    += A2 [b1 b2]
          }
        }
    }
  };

  // accumulator row of a tile -> 16 pre-activation values
  auto load_acc = [&](int t, float (&v)[kC]) {
    const uint32_t trow = tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(t * 3 * kC);
    uint32_t p0[16], p1[16], p2[16];
    tmem_ld16_nowait(trow, p0);
    tmem_ld16_nowait(trow + kC, p1);
    tmem_ld16_nowait(trow + 2 * kC, p2);
    tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < kC; ++c)
      v[c] = fmaf(fmaf(__uint_as_float(p2[c]), 1.f / kSplitScale, __uint_as_float(p1[c])), 1.f / kSplitScale,
                  __uint_as_float(p0[c]));
  };

  // the value row of site (x, y) of configuration g into a padded operand set, wrap copies included
  auto store_site = [&](char* set, int px, int py, int g, int x, int y, const Row16& r) {
    const int x0 = x + px, y0 = y + py;
#pragma unroll
    for (int sx = -1; sx <= 1; ++sx) {
      const int xx = x0 + sx * d.X;
      if (xx < 0 || xx >= d.PH) continue;
#pragma unroll
      for (int sy = -1; sy <= 1; ++sy) {
        const int yy = y0 + sy * d.Y;
        if (yy < 0 || yy >= d.PW) continue;
        store_row(set, RT, xx * d.GW + g * d.PW + yy, r);
      }
    }
  };

  const int64_t b_begin = (int64_t)blockIdx.x * per_cta, b_end = min(B, b_begin + per_cta);
  for (int64_t b0 = b_begin; b0 < b_end; b0 += d.G) {
    const int n_cfg = (int)min((int64_t)d.G, b_end - b0);
    load_w(false, 0);
    for (int e = threadIdx.x; e < d.G * d.NW; e += kThreads)
      cfg[e] = e < n_cfg * d.NW ? packed[b0 * d.NW + e] : 0ull;
    for (int e = threadIdx.x; e < KW * d.G; e += kThreads) {
      const int k = e / d.G, g = e - k * d.G;
      wk_s[e] = g < n_cfg ? weights[(int64_t)k * B + b0 + g] : 0.f;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
      for (int k = 0; k < KW; ++k)
        for (int g = 0; g < n_cfg; ++g) wtot[k] += wk_s[k * d.G + g];
    }
    // spin plane: row R = xx * GW + g * PW + yy holds the spins of the padded sites (xx, yy .. yy + 7)
    for (int R = threadIdx.x; R < d.PH * d.GW; R += kThreads) {
      const int xx = R / d.GW, rem = R - xx * d.GW;
      const int g = rem / d.PW, yy = rem - g * d.PW;
      uint32_t w[4] = {0u, 0u, 0u, 0u};
      if (g < n_cfg) {
        int sx = xx - d.pad_x; sx += sx < 0 ? d.X : 0; sx -= sx >= d.X ? d.X : 0;
        const uint64_t* words = cfg + g * d.NW;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          uint32_t hbits = 0u;
          if (yy + e < d.PW) {
            int sy = yy + e - d.pad_y; sy += sy < 0 ? d.Y : 0; sy -= sy >= d.Y ? d.Y : 0;
            hbits = word_bit(words, sx * d.Y + sy) ? 0x3c00u : 0xbc00u;
          }
          w[e >> 1] |= hbits << (16 * (e & 1));
        }
      }
      *reinterpret_cast<uint4*>(spin + (size_t)R * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
    sync_async();

    // ================= forward: layers 0 .. L-2 =================
    for (int l = 0; l <= d.L - 2; ++l) {
      if (l == 0) {
        const uint32_t idesc3 = idesc0 | ((uint32_t)(3 * kC >> 3) << 17);
        const uint32_t a_units = smem_u32(spin) >> 4, b_units = smem_u32(w1s) >> 4;
        const uint32_t a_lbo = (uint32_t)d.GW << 16, b_lbo = (uint32_t)(3 * kC) << 16;
        for (int t = warp; t < d.n_tiles; t += kWarps) {
          const uint32_t d_tmem = tmem + (uint32_t)(t * 3 * kC);
          for (int pr = 0; pr < d.n_pairs; ++pr) {
            const uint64_t a = ((uint64_t)hi_k << 32) | ((a_units + (uint32_t)(t * 128 + 2 * pr * d.GW)) | a_lbo);
            const uint64_t b = ((uint64_t)hi_k << 32) | ((b_units + (uint32_t)(pr * 2 * 3 * kC)) | b_lbo);
            if (elect_one()) mma_f16(d_tmem, a, b, idesc3, pr > 0 ? 1u : 0u);
          }
        }
      } else {
        wait_w();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        conv_mmas(hset(l));
      }
      commit_and_wait();
      if (l >= 1) {                                 // the slot is free: next image under the epilogue
        if (l < d.n_tensor) load_w(false, l);
        else load_w(true, d.n_tensor - 1);
      }
      const bool last = l == d.L - 2;
      const float* bj = bias_s + l * kC;
      for (int t = warp >> 2; t < d.n_tiles; t += kWarps / 4) {
        float v[kC];
        load_acc(t, v);
        const int R = t * 128 + 32 * q + lane;
        const int x = R / d.GW, rem = R - x * d.GW;
        const int g = rem / d.PW, y = rem - g * d.PW;
        const bool valid = x < d.X && y < d.Y && g < n_cfg;
        if (relu) {
#pragma unroll
          for (int c = 0; c < kC; ++c) v[c] = fmaxf(v[c] + bj[c], 0.f);
        } else {
#pragma unroll
          for (int c = 0; c < kC; ++c) v[c] = activate_slow(act, v[c] + bj[c]);
        }
        if (!last) {
          if (valid) store_site(hset(l + 1), d.pad_x, d.pad_y, g, x, y, split_row(v));
        } else {
          // d z / d W_{L-1}[tap][ci][co] = sum_pos h_{L-1}[pos][ci]; delta_{L-2} = wsum . act'(h_{L-1})
#pragma unroll
          for (int k = 0; k < KW; ++k) {
            const float wkg = valid ? wk_s[k * d.G + g] : 0.f;
            float wv[kC];
#pragma unroll
            for (int c = 0; c < kC; ++c) wv[c] = valid ? wkg * v[c] : 0.f;   // junk rows may hold anything
            colsum16_add(wv, lane, my_slot + k * pl.slot_floats + (d.L - 1) * kC);
          }
          float dl[kC];
#pragma unroll
          for (int c = 0; c < kC; ++c)
            dl[c] = wsum_s[c] * (relu ? (v[c] > 0.f ? 1.f : 0.f) : act_grad_slow(act, v[c]));
          if (valid) store_site(dset, d.bpad_x, d.bpad_y, g, x, y, split_row(dl));
        }
      }
      sync_async();
    }

    // ================= backward: l = L-2 .. 0 =================
    // dset holds delta_l = d z / d (pre-activation output of conv_l), home cells + wrap copies
    const int home_off = d.bpad_x * d.GW + d.bpad_y;         // home cell of output row R in dset / wdset: R + home_off
    for (int l = d.L - 2; l >= 0; --l) {
      for (int k = 0; k < KW; ++k) {
        // w_k . delta_l at the home cells (B operand of the weight-gradient GEMMs) + bias gradient
        for (int i0 = 0; i0 < d.G * d.N; i0 += kThreads) {
          const int item = i0 + threadIdx.x;
          float v[kC];
#pragma unroll
          for (int c = 0; c < kC; ++c) v[c] = 0.f;
          if (item < d.G * d.N) {
            const int g = item / d.N, pos = item - g * d.N;
            const int x = pos / d.Y, y = pos - x * d.Y;
            const int R = x * d.GW + g * d.PW + y + home_off;
            load_row(dset, RT, R, v);
            const float wkg = wk_s[k * d.G + g];
#pragma unroll
            for (int c = 0; c < kC; ++c) v[c] *= wkg;
            store_row(wdset, RT, R, split_row(v));
          }
          colsum16_add(v, lane, my_slot + k * pl.slot_floats + l * kC);
        }
        sync_async();
        // weight-gradient GEMMs, one accumulator of 32 columns per tap; M = 64 on the
        // activation planes (half the A-operand fetch of M = 128), M = 128 on the spin plane
        const uint32_t hi_mn = plane_units | (1u << 14);          // MN-major: SBO = plane stride, LBO = 8 units
        const uint32_t idesc_mn = (1u << 4) | ((uint32_t)(l > 0 ? 4u : 8u) << 24) | (1u << 15) |
                                  (1u << 16) | ((uint32_t)(kSlotCols >> 3) << 17);
        const uint32_t b_units = (smem_u32(wdset) >> 4) + (uint32_t)home_off;
        if (l == 0) {
          // A = spin plane: M chunk = kernel row dx (stride GW rows), 8 kernel columns per chunk
          const uint32_t hi_sp = (uint32_t)d.GW | (1u << 14);
          const uint32_t a_units = smem_u32(spin) >> 4;
          if (warp == 0) {
            for (int kb = 0; kb < d.kblocks; ++kb) {
              const uint64_t a = ((uint64_t)hi_sp << 32) | ((a_units + (uint32_t)(16 * kb)) | (8u << 16));
              const uint64_t b = ((uint64_t)hi_mn << 32) | ((b_units + (uint32_t)(16 * kb)) | (8u << 16));
              if (elect_one()) mma_f16(tmem, a, b, idesc_mn, kb > 0 ? 1u : 0u);
            }
          }
          commit_and_wait();
          // accumulator row m = dx * 8 + dy, columns (chunk, split, 8 co)
          if (warp < 4) {
            const int m = 32 * warp + lane, dx = m >> 3, dy = m & 7;
            uint32_t c0[16], c1[16];
            tmem_ld16_nowait(tmem + ((uint32_t)(32 * warp) << 16), c0);
            tmem_ld16_nowait(tmem + ((uint32_t)(32 * warp) << 16) + 16u, c1);
            tmem_ld_wait();
            if (dx < d.kx && dy < d.ky) {
              float* dst = part + (size_t)k * d.P + d.w_off[0] + (size_t)(dx * d.ky + dy) * kC;
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                dst[e] += fmaf(__uint_as_float(c0[8 + e]), 1.f / kSplitScale, __uint_as_float(c0[e]));
                dst[8 + e] += fmaf(__uint_as_float(c1[8 + e]), 1.f / kSplitScale, __uint_as_float(c1[e]));
              }
            }
          }
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncthreads();
        } else {
          const uint32_t a_units = smem_u32(hset(l)) >> 4;
          const int per_pass = kTmemCols / kSlotCols;
          for (int t0 = 0; t0 < taps; t0 += per_pass) {
            const int t1 = min(taps, t0 + per_pass);
            for (int tap = t0 + warp; tap < t1; tap += kWarps) {
              const int dx = tap / d.ky, dy = tap - dx * d.ky;
              const uint32_t d_tmem = tmem + (uint32_t)((tap - t0) * kSlotCols);
              const uint32_t a_row = a_units + (uint32_t)(dx * d.GW + dy);
              for (int kb = 0; kb < d.kblocks; ++kb) {
                const uint64_t a = ((uint64_t)hi_mn << 32) | ((a_row + (uint32_t)(16 * kb)) | (8u << 16));
                const uint64_t b = ((uint64_t)hi_mn << 32) | ((b_units + (uint32_t)(16 * kb)) | (8u << 16));
                if (elect_one()) mma_f16(d_tmem, a, b, idesc_mn, kb > 0 ? 1u : 0u);
              }
            }
            commit_and_wait();
            // drain: accumulator row = (chunk_h, split_h, 8 ci), columns = (chunk_d, split_d, 8 co);
            // d W[tap][ci][co] = D11 + (D12 + D21) / S + D22 / S^2.  M = 64: rows 16 i + r in
            // lane 32 i + r (lane quarters q = 0, 1).
            if (q < 2) {
              const int sh = (lane >> 3) & 1;
              const int ci = q * 8 + (lane & 7);
              const bool active = lane < 16;
              for (int tap = t0 + (warp >> 2); tap < t1; tap += 2) {   // two warps share a lane quarter
                const uint32_t trow = tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)((tap - t0) * kSlotCols);
                uint32_t c0[16], c1[16];
                tmem_ld16_nowait(trow, c0);
                tmem_ld16_nowait(trow + 16u, c1);
                tmem_ld_wait();
                float tv[kC];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  tv[e] = fmaf(__uint_as_float(c0[8 + e]), 1.f / kSplitScale, __uint_as_float(c0[e]));
                  tv[8 + e] = fmaf(__uint_as_float(c1[8 + e]), 1.f / kSplitScale, __uint_as_float(c1[e]));
                }
                float fin[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  const float send = sh ? tv[e] : tv[8 + e];
                  const float recv = __shfl_xor_sync(CGSVMC_FULL_MASK, send, 8);
                  fin[e] = sh ? fmaf(tv[8 + e], 1.f / kSplitScale, recv) : fmaf(recv, 1.f / kSplitScale, tv[e]);
                }
                if (active) {
                  float4* dst = reinterpret_cast<float4*>(part + (size_t)k * d.P + d.w_off[l] +
                                                          ((size_t)tap * kC + ci) * kC + sh * 8);
                  float4 o0 = __ldcg(dst), o1 = __ldcg(dst + 1);
                  o0.x += fin[0]; o0.y += fin[1]; o0.z += fin[2]; o0.w += fin[3];
                  o1.x += fin[4]; o1.y += fin[5]; o1.z += fin[6]; o1.w += fin[7];
                  __stcg(dst, o0);
                  __stcg(dst + 1, o1);
                }
              }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
        }
      }
      if (l >= 1) {
        // backward data through conv_l: raw = conv^T(delta_l); delta_{l-1} = raw . act'(h_l)
        wait_w();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        conv_mmas(dset);
        commit_and_wait();
        if (l >= 2) load_w(true, l - 2);
        const char* hl = hset(l);
        for (int t = warp >> 2; t < d.n_tiles; t += kWarps / 4) {
          float v[kC];
          load_acc(t, v);
          const int R = t * 128 + 32 * q + lane;
          const int x = R / d.GW, rem = R - x * d.GW;
          const int g = rem / d.PW, y = rem - g * d.PW;
          const bool valid = x < d.X && y < d.Y && g < n_cfg;
          if (valid) {
            float hv[kC];
            load_row(hl, RT, (x + d.pad_x) * d.GW + g * d.PW + y + d.pad_y, hv);
#pragma unroll
            for (int c = 0; c < kC; ++c)
              v[c] *= relu ? (hv[c] > 0.f ? 1.f : 0.f) : act_grad_slow(act, hv[c]);
            store_site(dset, d.bpad_x, d.bpad_y, g, x, y, split_row(v));
          }
        }
        sync_async();
      }
    }
  }

  // ---- per-warp slots -> the CTA's slice: bias gradients, last layer ----
  __syncthreads();
  for (int e = threadIdx.x; e < KW * pl.slot_floats; e += kThreads) {
    const int k = e / pl.slot_floats, r = e - k * pl.slot_floats;
    float total = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) total += slots[((size_t)w * KW + k) * pl.slot_floats + r];
    const int l = r / kC, c = r - l * kC;
    if (l <= d.L - 2) {
      part[(size_t)k * d.P + d.b_off[l] + c] = total;
    } else {
      // every (tap, co) entry of the last layer's weights gets the sum over sites of input channel c
      float* dst = part + (size_t)k * d.P + d.w_off[d.L - 1];
      for (int tap = 0; tap < taps; ++tap)
        for (int co = 0; co < kC; ++co) dst[((size_t)tap * kC + c) * kC + co] = total;
    }
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < KW; ++k)
      for (int co = 0; co < kC; ++co) part[(size_t)k * d.P + d.b_off[d.L - 1] + co] = (float)d.N * wtot[k];
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 32)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)kTmemCols)
                 : "memory");
}

bool grad_enabled() {
  const char* e = getenv("CGSVMC_CONV_TC_GRAD");
  if (e != nullptr && atoi(e) == 0) return false;
  const char* f = getenv("CGSVMC_CONV_TC");
  return f == nullptr || atoi(f) != 0;
}

void size_plan(GDesc* t, int G) {
  t->G = G; t->GW = G * t->PW;
  t->rows_out = t->X * t->GW;
  t->n_tiles = (t->rows_out + 127) / 128;
  t->kblocks = (t->rows_out + 15) / 16;
  t->rows_total = (t->n_tiles * 128 + (t->kx - 1) * t->GW + (t->ky - 1) + 1 + 7) / 8 * 8;
  t->rows_total = std::max(t->rows_total, (t->PH * t->GW + 8 + 7) / 8 * 8);
}

bool make_gdesc(const cgsvmc_ansatz* a, int64_t B, GDesc* out) {
  const cgsvmc_ansatz_desc& s = a->desc;
  if (s.kind != CGSVMC_ANSATZ_CONV_1D && s.kind != CGSVMC_ANSATZ_CONV_2D) return false;
  if (s.num_layers < 3 || s.num_layers > kMaxL || s.num_filters != kC) return false;
  if (s.nonlinearity == CGSVMC_ACT_COS) return false;          // no gradient through the output value
  if (!conv_tc_supported(a, nullptr)) return false;            // shares conv_tc.cu's parameter image
  GDesc d;
  memset(&d, 0, sizeof(d));
  d.N = s.n_sites; d.L = s.num_layers; d.act = s.nonlinearity;
  d.NW = n_words(s.n_sites);
  if (s.kind == CGSVMC_ANSATZ_CONV_1D) {
    d.X = s.n_sites; d.Y = 1; d.kx = s.kernel_size; d.ky = 1;
    d.pad_x = s.kernel_size % 2 ? (s.kernel_size - 1) / 2 : s.kernel_size / 2;       // layers.py:64-73
    d.pad_y = 0;
  } else {
    d.X = s.size_x; d.Y = s.size_y; d.kx = d.ky = s.kernel_size;
    d.pad_x = d.pad_y = s.kernel_size % 2 ? (s.kernel_size - 1) / 2 : s.kernel_size / 2 - 1;   // layers.py:132-141
  }
  if (d.kx > d.X || d.ky > d.Y || d.ky > 8 || d.kx > 8) return false;
  d.bpad_x = d.kx - 1 - d.pad_x; d.bpad_y = d.ky - 1 - d.pad_y;
  d.PH = d.X + d.kx - 1; d.PW = d.Y + d.ky - 1;
  d.n_tensor = d.L - 2;
  d.n_pairs = (d.kx + 1) / 2;
  d.wbuf_bytes = d.kx * d.ky * 3 * kC * kC * 2;
  d.P = a->n_params;
  for (int l = 0; l < d.L; ++l) { d.w_off[l] = a->offsets[2 * l]; d.b_off[l] = a->offsets[2 * l + 1]; }
  // the largest batch that fits, but do not starve the grid
  bool found = false;
  for (int G = 16; G >= 1; --G) {
    GDesc t = d;
    size_plan(&t, G);
    if (t.rows_total > 8191 || t.n_tiles * 3 * kC > kTmemCols) continue;   // 2 x plane stride is a 14-bit field
    if (gplan(t, 2).total + 1024 > (size_t)a->max_smem_optin) continue;
    if (G > 1 && B > 0 && (B + G - 1) / G < (int64_t)a->num_sms) continue;
    d = t;
    found = true;
    break;
  }
  if (!found) return false;
  *out = d;
  return true;
}

template <typename F>
int opt_in(F kernel, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(smem)");
  return CGSVMC_OK;
}

}  // namespace

bool conv_tc_grad_supported(const cgsvmc_ansatz* a) {
  if (!grad_enabled()) return false;
  GDesc d;
  return make_gdesc(a, 0, &d);
}

int conv_tc_grad(cgsvmc_ansatz* a, const uint64_t* packed, const float* weights, int64_t B, int K,
                 float* out, cudaStream_t st) {
  GDesc d;
  if (!make_gdesc(a, B, &d)) { set_error("conv_tc grad: unsupported network"); return CGSVMC_ERR_UNSUPPORTED; }
  ConvTcImage img;
  if (int rc = conv_tc_image(a, &img, st)) return rc;
  d.w1img = reinterpret_cast<const __half*>(img.w1img);
  d.wimg = reinterpret_cast<const __half*>(img.wimg);
  d.wimg_b = reinterpret_cast<const __half*>(img.wimg_b);
  d.bias = img.bias;
  d.wsum = img.wsum;
  const int64_t batches = (B + d.G - 1) / d.G;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(batches, a->num_sms));
  const int64_t per_cta = ((batches + grid - 1) / grid) * d.G;
  const int used = (int)((B + per_cta - 1) / per_cta);
  const int64_t P = d.P;
  if (int rc = ensure_scratch(a, (size_t)grid * 2 * P * sizeof(float))) return rc;
  float* partials = a->scratch;
  for (int k0 = 0; k0 < K; k0 += 2) {
    const int kk = std::min(2, K - k0);
    const float* w = weights + (int64_t)k0 * B;
    const size_t smem = gplan(d, kk).total;
    if (kk == 2) {
      if (int rc = opt_in(conv_grad_tc_kernel<2>, smem)) return rc;
      conv_grad_tc_kernel<2><<<used, kThreads, smem, st>>>(d, packed, w, B, per_cta, partials);
    } else {
      if (int rc = opt_in(conv_grad_tc_kernel<1>, smem)) return rc;
      conv_grad_tc_kernel<1><<<used, kThreads, smem, st>>>(d, packed, w, B, per_cta, partials);
    }
    if (int rc = cuda_fail(cudaGetLastError(), "conv_tc grad launch")) return rc;
    if (int rc = launch_reduce_partials(partials, used, (int64_t)kk * P, out + (int64_t)k0 * P, st)) return rc;
  }
  return CGSVMC_OK;
}

}  // namespace cgsvmc
