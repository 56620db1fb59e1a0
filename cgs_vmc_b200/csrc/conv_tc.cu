// Periodic convolutional ansaetze (conv_1d / conv_2d, wavefunctions.py:454-615,
// layers.py:24-160) on the 5th-generation tensor cores: tcgen05.mma with TMEM
// accumulators, implicit GEMM, three-way fp16 operand split (33 mantissa bits:
// every product is exact to float32) with fp32 accumulation.
//
// Forward pass of a batch of G configurations, all activations in shared memory:
//
//   layer 1 (C_in = 1)    : tensor cores as well.  The spins (+-1, exact in
//       fp16) are written as a plane whose row R holds the 8 consecutive sites
//       yy .. yy + 7 of the padded image, so one K = 16 MMA covers two kernel
//       rows (dx, dx + 1) x 8 kernel columns: ceil(kx / 2) MMAs per tile.
//   layers 2 .. L-1       : tensor cores.  The G configurations are laid side by
//       side as one periodic-padded image, rows R = xx * (G * PW) + g * PW + yy
//       (PH x PW = padded lattice, wrap halo materialised like the concat
//       padding of layers.py:64-74 / 143-148).  A float32 value v is split as
//       v = a1 + a2 / S + a3 / S^2 (fp16 each, S = 2^11) and stored in K-major,
//       no-swizzle UMMA operand planes [split][8-channel chunk][row][16 B], so
//       that row r of ANY tap-shifted window is `start + 16 r`: the A operand of
//       tap (dx, dy) is the same descriptor with the start address advanced by
//       (dx * G * PW + dy) rows -- no im2col, no copies.  When eight or more
//       configurations fit, they are INTERLEAVED instead (row = xx * G * PW +
//       yy * G + g, G a multiple of 8): every tap shift is then a multiple of 8
//       rows = 128 bytes, so the 8-row x 16-byte core matrices the tensor core
//       fetches stay aligned to shared-memory lines (a misaligned core matrix
//       costs two wavefronts: measured 181 against 96 cycles per tap).  The
//       weights of a tap
//       are the B operand [b1 | b2 | b3] concatenated along N, so per tap and
//       16 input channels three MMAs cover the six significant products while
//       each activation plane is fetched from shared memory once:
//         A1 x [b1 b2 b3] -> columns [P0 P1 P2],  A2 x [b1 b2] -> [P1 P2],
//         A3 x [b1] -> [P2];   D = P0 + P1 / S + P2 / S^2   (TMEM, fp32).
//       The kernel is bound by the shared-memory reads of the A operand
//       (N = C is small), not by the tensor pipe.  Rows whose yy falls in the
//       halo are junk and are dropped by the epilogue (tcgen05.ld -> bias ->
//       nonlinearity -> split -> operand planes of the next layer, halo copies
//       included).
//   layer L (no nonlinearity, then the sum over sites and channels,
//       wavefunctions.py:583-590): with stride 1 and periodic padding every tap
//       is a bijection of the sites, so
//         z = N sum_c b_c + sum_ci (sum_pos h[pos][ci]) (sum_{tap,c} W[tap][ci][c])
//       -- a C-term dot product per site instead of a convolution.
//
// Used by log_amp, the sampler (one forward per proposal) and the local energy
// (one forward per antiparallel bond).  The gradient stays on the SIMT path.
#include <algorithm>
#include <cstdlib>

#include <cuda_fp16.h>

#include "common.cuh"
#include "internal.h"
#include "tc_common.cuh"

namespace cgsvmc {
namespace {

using namespace tc;

// Development aid (-DCGSVMC_RBM2_TIMING build, profiles/run_conv_tc_phases.py):
// thread 0 of every CTA accumulates the cycles its tensor layers spend in the
// MMA phase (issue until the commit barrier flips) and in the epilogue.
#ifdef CGSVMC_RBM2_TIMING
__device__ unsigned long long g_tc_phase[4];   // MMA cycles, epilogue cycles, layers, forwards
#define TC_PHASE_T0() const long long tc_t0_ = clock64()
#define TC_PHASE_ADD(IDX, T0) do { if (threadIdx.x == 0) atomicAdd(&g_tc_phase[IDX], (unsigned long long)(clock64() - (T0))); } while (0)
#define TC_PHASE_COUNT(IDX) do { if (threadIdx.x == 0) atomicAdd(&g_tc_phase[IDX], 1ull); } while (0)
#else
#define TC_PHASE_T0() do {} while (0)
#define TC_PHASE_ADD(IDX, T0) do {} while (0)
#define TC_PHASE_COUNT(IDX) do {} while (0)
#endif

// Activation split planes held in shared memory.  Every MMA reads a 128 x 16
// fp16 A tile (4 KB) from shared memory, which takes ~64 cycles whatever N is
// (measured: 181 cycles per tap for three MMAs with N = 48 / 32 / 16, aligned
// or not), so with C = 16 filters the MMA phase is bound by the NUMBER of
// activation planes, not by the tensor pipe.  Two planes: v = a1 + a2 / S with
// 22 mantissa bits (|error| <= 2^-23 |v|, below the rounding of a float32
// accumulation over the 25 C products of an output) against the full three-way
// split of the weights: products a1 b1, a1 b2, a1 b3, a2 b1, a2 b2.
// Three planes restore the exact float32 activations (CGSVMC_TC_ACT_SPLITS=3 at
// compile time) at 1.5x the MMA time.
#ifndef CGSVMC_TC_ACT_SPLITS
#define CGSVMC_TC_ACT_SPLITS 2
#endif
constexpr int kActSplits = CGSVMC_TC_ACT_SPLITS;
static_assert(kActSplits == 2 || kActSplits == 3, "two or three activation planes");

constexpr int kThreads = 256;
constexpr int kWarps = 8;
constexpr int kMaxTaps = 64;

struct TcDesc {
  int N, X, Y, kx, ky, pad_x, pad_y, C, L, act, NW;
  int PH, PW, G, GW;        // padded lattice, configurations per batch, G * PW
  int rows_out;             // X * GW output rows (incl. junk halo columns)
  int n_tiles;              // ceil(rows_out / 128)
  int rows_total;           // rows of one operand plane
  int n_tensor;             // L - 2
  int wbuf_bytes;           // taps * 3 * C * C * 2
  int n_wbuf;               // weight buffers in shared memory (1 or 2)
  int tmem_cols;
  int n_pairs;              // ceil(kx / 2): MMAs per tile of layer 1
  int ctas;                 // CTAs per SM the plan was sized for (1 or 2)
  int il;                   // 1: configurations interleaved, row = xx * GW + yy * G + g (G % 8 == 0);
                            // 0: side by side, row = xx * GW + g * PW + yy
  int ystep;                // rows per step in y: G (interleaved) or 1
  const __half* w1img;      // [n_pairs][2][3C][8]   layer 1 B operand
  const __half* wimg;       // [n_tensor][taps][C/8][3C][8]
  const __half* wimg_b;     // the same layers for backward-data: taps mirrored, [co chunk][3C: split, ci][8 co]
  const float* bias;        // [L - 1][C]  layers 1 .. L-1
  const float* wsum;        // [C] last-layer column sums, then z0 = N sum_c b_L[c]
};

struct SmemPlan {
  size_t act, wbuf, w1, consts, rowsum, bars, total;
};

__host__ __device__ inline SmemPlan smem_plan(const TcDesc& d) {
  SmemPlan p;
  size_t off = 0;
  p.act = off; off += (size_t)kActSplits * (d.C / 8) * d.rows_total * 16;
  p.wbuf = off; off += (size_t)d.n_wbuf * d.wbuf_bytes;
  p.w1 = off; off += (size_t)d.n_pairs * 2 * 3 * d.C * 16;
  p.consts = off; off += ((size_t)(d.L - 1) * d.C + d.C + 4 + (size_t)d.kx * d.ky) * 4;
  off = (off + 15) / 16 * 16;
  p.rowsum = off; off += (size_t)d.n_tiles * 128 * 4;
  p.bars = off; off += 64;
  p.total = off;
  return p;
}

__device__ __forceinline__ int word_bit(const uint64_t* words, int site) {
  return (int)((words[site >> 6] >> (site & 63)) & 1ull);
}

// ---------------------------------------------------------------------------
// The forward engine.  All 256 threads of the CTA call every method.
// ---------------------------------------------------------------------------
struct Engine {
  const TcDesc& d;
  __device__ explicit Engine(const TcDesc& desc) : d(desc) {}
  __half* act;       // operand planes [3 splits][C/8 chunks][rows_total][8]; the spin plane aliases plane 0
  char* wbuf;        // weight buffers of the layers 2 .. L-1
  __half* w1s;       // layer 1 B operand
  float *bias_s, *wsum_s, *rowsum;
  int* tap_shift;    // row shift dx * GW + dy of every tap
  uint64_t *mma_bar, *wbar;   // wbar[2]
  uint32_t* tmem_holder;
  uint32_t tmem;
  uint32_t mma_phase, wphase0, wphase1;
  uint32_t use_count;   // layers 2.. executed so far (selects the weight buffer)
  int CH, plane_halfs;  // 8-channel chunks per split, fp16 elements per plane

  __device__ void setup(char* smem) {
    const SmemPlan p = smem_plan(d);
    CH = d.C / 8;
    plane_halfs = d.rows_total * 8;
    act = reinterpret_cast<__half*>(smem + p.act);
    wbuf = smem + p.wbuf;
    w1s = reinterpret_cast<__half*>(smem + p.w1);
    bias_s = reinterpret_cast<float*>(smem + p.consts);
    wsum_s = bias_s + (d.L - 1) * d.C;
    tap_shift = reinterpret_cast<int*>(wsum_s + d.C + 4);
    rowsum = reinterpret_cast<float*>(smem + p.rowsum);
    mma_bar = reinterpret_cast<uint64_t*>(smem + p.bars);
    wbar = mma_bar + 1;
    tmem_holder = reinterpret_cast<uint32_t*>(mma_bar + 3);
    mma_phase = wphase0 = wphase1 = 0;
    use_count = 0;
    const int taps = d.kx * d.ky;
    for (int e = threadIdx.x; e < d.n_pairs * 2 * 3 * d.C * 4; e += kThreads)
      reinterpret_cast<uint32_t*>(w1s)[e] = reinterpret_cast<const uint32_t*>(d.w1img)[e];
    for (int e = threadIdx.x; e < (d.L - 1) * d.C; e += kThreads) bias_s[e] = d.bias[e];
    for (int e = threadIdx.x; e < d.C + 1; e += kThreads) wsum_s[e] = d.wsum[e];
    for (int e = threadIdx.x; e < taps; e += kThreads) tap_shift[e] = (e / d.ky) * d.GW + (e % d.ky) * d.ystep;
    // the planes are read beyond the written rows by junk output rows: keep
    // the bit patterns finite
    for (int e = threadIdx.x; e < kActSplits * CH * plane_halfs / 2; e += kThreads)
      reinterpret_cast<uint32_t*>(act)[e] = 0u;
    if (threadIdx.x == 0) {
      mbar_init(mma_bar, (uint32_t)min(kWarps, d.n_tiles));   // one commit per issuing warp
      mbar_init(wbar, 1);
      mbar_init(wbar + 1, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < 32) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(tmem_holder)),
                   "r"((uint32_t)d.tmem_cols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    tmem = *tmem_holder;
    // weights of the first tensor layer
    if (threadIdx.x == 0 && d.n_tensor > 0)
      bulk_load_async(wbuf, d.wimg, (uint32_t)d.wbuf_bytes, wbar);
  }

  __device__ void teardown() {
    // a prefetch issued by the last forward may still be in flight
    if (d.n_tensor > 0) {
      if (d.n_wbuf == 1 || (use_count & 1u) == 0) mbar_wait(wbar, wphase0); else mbar_wait(wbar + 1, wphase1);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem),
                   "r"((uint32_t)d.tmem_cols)
                   : "memory");
  }

  // three-way fp16 split of the C channel values of site (x, y) of
  // configuration g into the operand planes, halo copies included
  // (layers.py:64-74, 143-148).
  template <int CC>
  __device__ __forceinline__ void store_site(int g, int x, int y, const float (&v)[CC]) {
    __half2 q[3][CC / 2];
#pragma unroll
    for (int c = 0; c < CC; c += 2) {
      __half h[3][2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float val = v[c + e];
        h[0][e] = __float2half_rn(val);
        const float r1 = (val - __half2float(h[0][e])) * kSplitScale;
        h[1][e] = __float2half_rn(r1);
        const float r2 = (r1 - __half2float(h[1][e])) * kSplitScale;
        h[2][e] = __float2half_rn(r2);
      }
#pragma unroll
      for (int sp = 0; sp < kActSplits; ++sp) q[sp][c / 2] = __halves2half2(h[sp][0], h[sp][1]);
    }
    const int x0 = x + d.pad_x, y0 = y + d.pad_y;
#pragma unroll
    for (int sx = -1; sx <= 1; ++sx) {
      const int xx = x0 + sx * d.X;
      if (xx < 0 || xx >= d.PH) continue;
#pragma unroll
      for (int sy = -1; sy <= 1; ++sy) {
        const int yy = y0 + sy * d.Y;
        if (yy < 0 || yy >= d.PW) continue;
        const int R = xx * d.GW + (d.il ? yy * d.G + g : g * d.PW + yy);
        __half* base = act + R * 8;
#pragma unroll
        for (int sp = 0; sp < kActSplits; ++sp)
#pragma unroll
          for (int ch = 0; ch < CC / 8; ++ch) {
            uint4 pk;
            pk.x = *reinterpret_cast<const uint32_t*>(&q[sp][4 * ch]);
            pk.y = *reinterpret_cast<const uint32_t*>(&q[sp][4 * ch + 1]);
            pk.z = *reinterpret_cast<const uint32_t*>(&q[sp][4 * ch + 2]);
            pk.w = *reinterpret_cast<const uint32_t*>(&q[sp][4 * ch + 3]);
            *reinterpret_cast<uint4*>(base + (sp * CH + ch) * plane_halfs) = pk;
          }
      }
    }
  }

  // Spin plane of layer 1 (aliases operand plane 0, dead once the layer-1
  // MMAs have completed): row R = xx * GW + g * PW + yy holds the spins of the
  // padded sites (xx, yy .. yy + 7) of configuration g as fp16 +-1.
  __device__ void write_spin_plane(const uint64_t* cfg, int n_cfg) {
    const int rows = d.PH * d.GW;
    for (int R = threadIdx.x; R < rows; R += kThreads) {
      const int xx = R / d.GW, rem = R - xx * d.GW;
      const int g = d.il ? rem % d.G : rem / d.PW, yy = d.il ? rem / d.G : rem - g * d.PW;
      uint32_t w[4] = {0u, 0u, 0u, 0u};
      if (g < n_cfg) {
        int sx = xx - d.pad_x; sx += sx < 0 ? d.X : 0; sx -= sx >= d.X ? d.X : 0;
        const uint64_t* words = cfg + g * d.NW;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          uint32_t hbits = 0u;   // beyond the padded row: weight slots are zero there
          if (yy + e < d.PW) {
            int sy = yy + e - d.pad_y; sy += sy < 0 ? d.Y : 0; sy -= sy >= d.Y ? d.Y : 0;
            hbits = word_bit(words, sx * d.Y + sy) ? 0x3c00u : 0xbc00u;   // +1 / -1
          }
          w[e >> 1] |= hbits << (16 * (e & 1));
        }
      }
      *reinterpret_cast<uint4*>(act + R * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }

  // One layer on the tensor cores.  layer = 0: spins -> layer 1; layer >= 1:
  // network layer layer + 1 with the weights streamed through wbuf.  All MMAs
  // are issued by one elected lane of warp 0 (descriptor arithmetic stays
  // warp-uniform), then every warp runs the epilogue.
  template <int CC>
  __device__ void tensor_layer(int layer, int n_cfg) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool first = layer == 0;
    TC_PHASE_T0();
    const uint32_t buf = (!first && d.n_wbuf == 2) ? (use_count & 1u) : 0u;
    // MMA issue: tile t is issued by warp t mod n_iss (one elected lane each).
    // A single issuing thread needs ~30 uniform-datapath instructions per tap
    // (descriptors, UMOV / R2UR, elect) and was the bottleneck of the MMA phase
    // (181 cycles per tap of three MMAs whose tensor-pipe floor is 48); up to
    // eight warps issue in parallel, each into its own tiles' accumulators.
    const int n_iss = min(kWarps, d.n_tiles);
    if (warp < n_iss) {
      char* wb = wbuf + (size_t)buf * d.wbuf_bytes;
      if (!first) {
        uint64_t* bar = wbar + buf;
        const uint32_t ph = buf ? wphase1 : wphase0;
        const int j = layer - 1;
        mbar_wait(bar, ph);
        if (d.n_wbuf == 2 && warp == 0 && lane == 0) {   // prefetch the next layer's weights (wraps to the next forward)
          const int jn = (j + 1) % d.n_tensor;
          bulk_load_async(wbuf + (size_t)(buf ^ 1u) * d.wbuf_bytes,
                          reinterpret_cast<const char*>(d.wimg) + (size_t)jn * d.wbuf_bytes,
                          (uint32_t)d.wbuf_bytes, wbar + (buf ^ 1u));
        }
      }
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // instruction descriptor: D = F32, A = B = F16, K-major, M = 128; N set per MMA
      const uint32_t idesc0 = (1u << 4) | (8u << 24);
      const uint32_t idesc3 = idesc0 | ((uint32_t)(3 * CC >> 3) << 17);
      const uint32_t idesc2 = idesc0 | ((uint32_t)(2 * CC >> 3) << 17);
      const uint32_t idesc1 = idesc0 | ((uint32_t)(CC >> 3) << 17);
      const uint32_t a_units = smem_u32(act) >> 4;
      const uint32_t plane_units = (uint32_t)d.rows_total;            // 16-byte units per plane
      const uint32_t split_units = (uint32_t)(CC / 8) * plane_units;  // split s -> s + 1
      const uint32_t desc_hi = 8u | (1u << 14);                       // SBO = 8 units, version 1
      if (first) {
        // A: spin plane, second K chunk = the same plane one kernel row (GW rows) further
        const uint32_t b_units = smem_u32(w1s) >> 4;
        const uint32_t a_lbo = (uint32_t)d.GW << 16, b_lbo = (uint32_t)(3 * CC) << 16;
        for (int t = warp; t < d.n_tiles; t += n_iss) {
          const uint32_t d_tmem = tmem + (uint32_t)(t * 3 * CC);
          for (int pr = 0; pr < d.n_pairs; ++pr) {
            const uint32_t a_lo = (a_units + (uint32_t)(t * 128 + 2 * pr * d.GW)) | a_lbo;
            const uint32_t b_lo = (b_units + (uint32_t)(pr * 2 * 3 * CC)) | b_lbo;
            const uint64_t a = ((uint64_t)desc_hi << 32) | a_lo;
            const uint64_t b = ((uint64_t)desc_hi << 32) | b_lo;
            if (elect_one()) mma_f16(d_tmem, a, b, idesc3, pr > 0 ? 1u : 0u);
          }
        }
      } else {
        const uint32_t b_units = smem_u32(wb) >> 4;
        const uint32_t a_lbo = plane_units << 16, b_lbo = (uint32_t)(3 * CC) << 16;
        const uint32_t b_tap_units = (uint32_t)(CC / 8) * 3 * CC;     // per tap: [CH][3C] rows of 16 B
        for (int t = warp; t < d.n_tiles; t += n_iss) {
          const uint32_t d_tmem = tmem + (uint32_t)(t * 3 * CC);
          const uint32_t a_tile = a_units + (uint32_t)(t * 128);
          for (int dx = 0; dx < d.kx; ++dx)
          for (int dy = 0; dy < d.ky; ++dy) {
            const int tap = dx * d.ky + dy;
            const uint32_t a_row = a_tile + (uint32_t)(dx * d.GW + dy * d.ystep);
            const uint32_t b_row = b_units + (uint32_t)tap * b_tap_units;
#pragma unroll
            for (int ks = 0; ks < CC / 16; ++ks) {
              const uint32_t a_lo = (a_row + (uint32_t)(2 * ks) * plane_units) | a_lbo;
              const uint32_t b_lo = (b_row + (uint32_t)(2 * ks) * (3 * CC)) | b_lbo;
              const uint64_t a1 = ((uint64_t)desc_hi << 32) | a_lo;
              const uint64_t a2 = ((uint64_t)desc_hi << 32) | (a_lo + split_units);
              const uint64_t a3 = ((uint64_t)desc_hi << 32) | (a_lo + 2 * split_units);
              const uint64_t b = ((uint64_t)desc_hi << 32) | b_lo;
              if (elect_one()) {
                mma_f16(d_tmem, a1, b, idesc3, (tap | ks) ? 1u : 0u);   // [P0 P1 P2] += A1 [b1 b2 b3]
                mma_f16(d_tmem + CC, a2, b, idesc2, 1u);                 // [P1 P2]    += A2 [b1 b2]
                if (kActSplits == 3) mma_f16(d_tmem + 2 * CC, a3, b, idesc1, 1u);   // [P2] += A3 [b1]
              }
            }
          }
        }
      }
      if (elect_one())
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                         smem_u32(mma_bar))
                     : "memory");
      __syncwarp();
    }
    // bookkeeping replicated in every thread
    if (!first) {
      if (buf) wphase1 ^= 1u; else wphase0 ^= 1u;
      ++use_count;
    }
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1u;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    TC_PHASE_ADD(0, tc_t0_);
#ifdef CGSVMC_RBM2_TIMING
    const long long tc_t1_ = clock64();
#endif
    // one weight buffer: the MMAs that read it have completed, so the next
    // layer's weights (wrapping to the next forward) stream in under the epilogue
    if (!first && d.n_wbuf == 1 && threadIdx.x == 0) {
      const int jn = layer % d.n_tensor;          // (j + 1) % n_tensor with j = layer - 1
      bulk_load_async(wbuf, reinterpret_cast<const char*>(d.wimg) + (size_t)jn * d.wbuf_bytes,
                      (uint32_t)d.wbuf_bytes, wbar);
    }

    // ---- epilogue: TMEM -> bias -> nonlinearity -> next operand planes / row sums ----
    const int q = warp & 3;
    const bool last = layer == d.L - 2;
    const float* bj = bias_s + layer * CC;
    const bool relu = d.act == CGSVMC_ACT_RELU;
    for (int t = warp >> 2; t < d.n_tiles; t += kWarps / 4) {
      float v[CC];
      const uint32_t trow = tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(t * 3 * CC);
#pragma unroll
      for (int c0 = 0; c0 < CC; c0 += 16) {
        float p0[16], p1[16], p2[16];
        tmem_ld16(trow + (uint32_t)c0, p0);
        tmem_ld16(trow + (uint32_t)(CC + c0), p1);
        tmem_ld16(trow + (uint32_t)(2 * CC + c0), p2);
#pragma unroll
        for (int c = 0; c < 16; ++c)
          v[c0 + c] = fmaf(fmaf(p2[c], 1.f / kSplitScale, p1[c]), 1.f / kSplitScale, p0[c]);
      }
      const int R = t * 128 + 32 * q + lane;
      const int x = R / d.GW, rem = R - x * d.GW;
      const int g = d.il ? rem % d.G : rem / d.PW, y = d.il ? rem / d.G : rem - g * d.PW;
      const bool valid = x < d.X && y < d.Y && g < n_cfg;
      if (relu) {
#pragma unroll
        for (int c = 0; c < CC; ++c) v[c] = fmaxf(v[c] + bj[c], 0.f);
      } else {
#pragma unroll
        for (int c = 0; c < CC; ++c) v[c] = tc_activate(d.act, v[c] + bj[c]);
      }
      if (last) {
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < CC; ++c) s = fmaf(v[c], wsum_s[c], s);
        rowsum[R] = valid ? s : 0.f;
      } else if (valid) {
        store_site<CC>(g, x, y, v);
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    TC_PHASE_ADD(1, tc_t1_);
    TC_PHASE_COUNT(2);
  }

  // z[g] for g < n_cfg; cfg: [G][NW] packed spins in shared memory.
  template <int CC>
  __device__ void forward(const uint64_t* cfg, int n_cfg, float* z) {
    TC_PHASE_COUNT(3);
    write_spin_plane(cfg, n_cfg);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    for (int layer = 0; layer <= d.L - 2; ++layer) tensor_layer<CC>(layer, n_cfg);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int g = warp; g < n_cfg; g += kWarps) {
      float s = 0.f;
      for (int pos = lane; pos < d.N; pos += 32) {
        const int x = pos / d.Y, y = pos - x * d.Y;
        s += rowsum[x * d.GW + (d.il ? y * d.G + g : g * d.PW + y)];
      }
      s = warp_sum(s);
      if (lane == 0) z[g] = s + wsum_s[d.C];
    }
    __syncthreads();
  }
};

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
struct Extras {   // shared memory behind the engine's plan
  uint64_t* cfg;      // [G][NW]
  uint64_t* cur;      // [G][NW]
  float *z, *z_cur, *u_acc;   // [G]
};

__device__ __forceinline__ Extras carve_extras(const TcDesc& d, char* smem) {
  Extras e;
  char* p = smem + smem_plan(d).total;
  e.cfg = reinterpret_cast<uint64_t*>(p); p += (size_t)d.G * d.NW * 8;
  e.cur = reinterpret_cast<uint64_t*>(p); p += (size_t)d.G * d.NW * 8;
  e.z = reinterpret_cast<float*>(p); p += (size_t)d.G * 4;
  e.z_cur = reinterpret_cast<float*>(p); p += (size_t)d.G * 4;
  e.u_acc = reinterpret_cast<float*>(p);
  return e;
}
__host__ __device__ inline size_t extras_bytes(const TcDesc& d) { return (size_t)d.G * d.NW * 16 + (size_t)d.G * 12 + 16; }

template <int CC, int CTAS>
__global__ void __launch_bounds__(kThreads, CTAS)
tc_log_amp_kernel(TcDesc d, const uint64_t* __restrict__ packed, int64_t B, float* __restrict__ out) {
  extern __shared__ __align__(1024) char smem[];
  Engine eng(d);
  eng.setup(smem);
  const Extras ex = carve_extras(d, smem);
  const int64_t n_batches = (B + d.G - 1) / d.G;
  for (int64_t batch = blockIdx.x; batch < n_batches; batch += gridDim.x) {
    const int64_t b0 = batch * d.G;
    const int n_cfg = (int)min((int64_t)d.G, B - b0);
    for (int e = threadIdx.x; e < n_cfg * d.NW; e += kThreads) ex.cfg[e] = packed[b0 * d.NW + e];
    __syncthreads();
    eng.forward<CC>(ex.cfg, n_cfg, ex.z);
    for (int g = threadIdx.x; g < n_cfg; g += kThreads) out[b0 + g] = ex.z[g];
    __syncthreads();
  }
  eng.teardown();
}

__device__ __forceinline__ int kth_set_bit(const uint64_t* words, int nw, int k) {
  for (int w = 0; w < nw; ++w) {
    uint64_t m = words[w];
    const int c = __popcll(m);
    if (k >= c) { k -= c; continue; }
    for (int qd = 0; qd < k; ++qd) m &= m - 1;
    return w * 64 + __ffsll((long long)m) - 1;
  }
  return 0;
}

// graph_builders.py:54-89 x n_steps; a CTA owns G walkers for all steps, one
// forward pass per proposal (the reference runs two), z of the current
// configuration cached.  Same Philox stream as every other sampler kernel.
template <int CC, int CTAS>
__global__ void __launch_bounds__(kThreads, CTAS)
tc_mc_kernel(TcDesc d, uint64_t* __restrict__ packed, int64_t B, int n_steps, uint64_t seed,
             uint64_t walker0, uint64_t step0, const uint64_t* __restrict__ step0_dev,
             unsigned long long* accept_count, float* __restrict__ log_amp_out) {
  if (step0_dev != nullptr) step0 += *step0_dev;
  extern __shared__ __align__(1024) char smem[];
  Engine eng(d);
  eng.setup(smem);
  const Extras ex = carve_extras(d, smem);
  __shared__ unsigned int n_acc_s;
  if (threadIdx.x == 0) n_acc_s = 0;
  const int64_t n_batches = (B + d.G - 1) / d.G;
  for (int64_t batch = blockIdx.x; batch < n_batches; batch += gridDim.x) {
    const int64_t b0 = batch * d.G;
    const int n_cfg = (int)min((int64_t)d.G, B - b0);
    for (int e = threadIdx.x; e < n_cfg * d.NW; e += kThreads) {
      const uint64_t w = packed[b0 * d.NW + e];
      ex.cur[e] = w;
      ex.cfg[e] = w;
    }
    __syncthreads();
    eng.forward<CC>(ex.cfg, n_cfg, ex.z);
    for (int g = threadIdx.x; g < n_cfg; g += kThreads) ex.z_cur[g] = ex.z[g];
    __syncthreads();
    for (int step = 0; step < n_steps; ++step) {
      for (int g = threadIdx.x; g < n_cfg; g += kThreads) {
        uint64_t s[CGSVMC_MAX_WORDS], dn[CGSVMC_MAX_WORDS];
        int n_up = 0;
        for (int w = 0; w < d.NW; ++w) {
          s[w] = ex.cur[g * d.NW + w];
          dn[w] = ~s[w] & valid_mask_word(d.N, w);
          n_up += __popcll(s[w]);
        }
        const int n_dn = d.N - n_up;
        float u = 2.f;     // > any probability: never accepted
        if (n_up > 0 && n_dn > 0) {
          const Philox4 r = walker_step_random(seed, walker0 + (uint64_t)(b0 + g), step0 + (uint64_t)step);
          const int up = kth_set_bit(s, d.NW, (int)__umulhi(r.x, (uint32_t)n_up));
          const int dns = kth_set_bit(dn, d.NW, (int)__umulhi(r.y, (uint32_t)n_dn));
          s[up >> 6] ^= 1ull << (up & 63);
          s[dns >> 6] ^= 1ull << (dns & 63);
          u = u32_to_unit(r.z);
        }
        for (int w = 0; w < d.NW; ++w) ex.cfg[g * d.NW + w] = s[w];
        ex.u_acc[g] = u;
      }
      __syncthreads();
      eng.forward<CC>(ex.cfg, n_cfg, ex.z);
      for (int g = threadIdx.x; g < n_cfg; g += kThreads) {
        const float prob = fast_exp(2.f * (ex.z[g] - ex.z_cur[g]));
        if (prob > ex.u_acc[g]) {   // strict; NaN rejects (graph_builders.py:75-79)
          for (int w = 0; w < d.NW; ++w) ex.cur[g * d.NW + w] = ex.cfg[g * d.NW + w];
          ex.z_cur[g] = ex.z[g];
          atomicAdd(&n_acc_s, 1u);
        }
      }
      __syncthreads();
    }
    for (int e = threadIdx.x; e < n_cfg * d.NW; e += kThreads) packed[b0 * d.NW + e] = ex.cur[e];
    if (log_amp_out != nullptr)
      for (int g = threadIdx.x; g < n_cfg; g += kThreads) log_amp_out[b0 + g] = ex.z_cur[g];
    __syncthreads();
  }
  if (threadIdx.x == 0 && accept_count != nullptr && n_acc_s)
    atomicAdd(accept_count, (unsigned long long)n_acc_s);
  eng.teardown();
}

// operators.py:227-259: a CTA takes one walker at a time, lists its antiparallel
// bonds and evaluates the base configuration and every flipped one G at a time.
template <int CC, int CTAS>
__global__ void __launch_bounds__(kThreads, CTAS)
tc_eloc_kernel(TcDesc d, const int2* __restrict__ bonds_ij, const float* __restrict__ bonds_jx,
               const float* __restrict__ bonds_jz, int n_bonds, const uint64_t* __restrict__ packed,
               int64_t B, float* __restrict__ e_loc, float* __restrict__ log_amp_out,
               float* __restrict__ diag_out, float* __restrict__ off_out) {
  extern __shared__ __align__(1024) char smem[];
  Engine eng(d);
  eng.setup(smem);
  const Extras ex = carve_extras(d, smem);
  // item list and amplitudes behind the extras
  char* p = smem + smem_plan(d).total + extras_bytes(d);
  float* z_item = reinterpret_cast<float*>(p); p += (size_t)(n_bonds + 1) * 4;
  uint16_t* item_bond = reinterpret_cast<uint16_t*>(p);   // [n_bonds + 1], entry 0 unused
  __shared__ int n_items_s;
  __shared__ float diag_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
    for (int w = threadIdx.x; w < d.NW; w += kThreads) ex.cur[w] = packed[b * d.NW + w];
    __syncthreads();
    if (warp == 0) {   // ordered compaction of the active bonds + diagonal term
      float diag = 0.f;
      int count = 1;
      for (int k0 = 0; k0 < n_bonds; k0 += 32) {
        const int k = k0 + lane;
        bool anti = false;
        if (k < n_bonds) {
          const int2 bd = bonds_ij[k];
          anti = word_bit(ex.cur, bd.x) != word_bit(ex.cur, bd.y);
          diag += (anti ? -0.25f : 0.25f) * bonds_jz[k];            // operators.py:165,169
        }
        const uint32_t vote = __ballot_sync(CGSVMC_FULL_MASK, anti);
        if (anti) item_bond[count + __popc(vote & ((1u << lane) - 1u))] = (uint16_t)k;
        count += __popc(vote);
      }
      diag = warp_sum(diag);
      if (lane == 0) { n_items_s = count; diag_s = diag; }
    }
    __syncthreads();
    const int n_items = n_items_s;
    for (int i0 = 0; i0 < n_items; i0 += d.G) {
      const int n_cfg = min(d.G, n_items - i0);
      for (int e = threadIdx.x; e < n_cfg * d.NW; e += kThreads) {
        const int g = e / d.NW, w = e - g * d.NW;
        const int it = i0 + g;
        uint64_t word = ex.cur[w];
        if (it > 0) {                                                // operators.py:158-164
          const int2 bd = bonds_ij[item_bond[it]];
          if ((bd.x >> 6) == w) word ^= 1ull << (bd.x & 63);
          if ((bd.y >> 6) == w) word ^= 1ull << (bd.y & 63);
        }
        ex.cfg[e] = word;
      }
      __syncthreads();
      eng.forward<CC>(ex.cfg, n_cfg, ex.z);
      for (int g = threadIdx.x; g < n_cfg; g += kThreads) z_item[i0 + g] = ex.z[g];
      __syncthreads();
    }
    if (warp == 0) {   // E_loc = diag + sum_active jx/2 exp(z' - z)   (operators.py:168-169, 259)
      const float z0 = z_item[0];
      float off = 0.f;
      for (int it = 1 + lane; it < n_items; it += 32)
        off = fmaf(0.5f * bonds_jx[item_bond[it]], fast_exp(z_item[it] - z0), off);
      off = warp_sum(off);
      if (lane == 0) {
        e_loc[b] = diag_s + off;
        if (log_amp_out) log_amp_out[b] = z0;
        if (diag_out) diag_out[b] = diag_s;
        if (off_out) off_out[b] = off;
      }
    }
    __syncthreads();
  }
  eng.teardown();
}

// ---------------------------------------------------------------------------
// parameter image: tcgen05 B-operand planes of the tensor layers (hi / lo TF32
// split), biases, last-layer column sums.
// ---------------------------------------------------------------------------
__device__ __forceinline__ __half split_part(float w, int split) {
  const __half h1 = __float2half_rn(w);
  const float r1 = (w - __half2float(h1)) * kSplitScale;
  const __half h2 = __float2half_rn(r1);
  const float r2 = (r1 - __half2float(h2)) * kSplitScale;
  return split == 0 ? h1 : split == 1 ? h2 : __float2half_rn(r2);
}

__global__ void tc_prep_kernel(int kx, int ky, int C, int L, int N, int n_pairs,
                               const float* __restrict__ params, const int64_t* __restrict__ w_off,
                               const int64_t* __restrict__ b_off, __half* __restrict__ w1img,
                               __half* __restrict__ wimg, __half* __restrict__ wimg_b, int64_t wimg_halfs,
                               float* __restrict__ bias, float* __restrict__ wsum, int n_tensor) {
  const int taps = kx * ky;
  const int64_t per_layer = (int64_t)taps * 3 * C * C;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < wimg_halfs;
       e += (int64_t)gridDim.x * blockDim.x) {
    // [layer j][tap][chunk][n = split * C + co][8 input channels]
    const int j = (int)(e / per_layer);
    int64_t r = e - (int64_t)j * per_layer;
    const int tap = (int)(r / (3 * C * C)); r -= (int64_t)tap * 3 * C * C;
    const int chunk = (int)(r / (3 * C * 8)); r -= (int64_t)chunk * 3 * C * 8;
    const int n = (int)(r / 8), el = (int)(r - 8 * n);
    const int split = n / C, co = n - split * C;
    const int ci = chunk * 8 + el;
    const float w = params[w_off[j + 1] + ((int64_t)tap * C + ci) * C + co];   // layer j + 2, [tap][ci][co]
    wimg[e] = split_part(w, split);
    // backward-data image (conv_tc_grad.cu): the transposed convolution is the
    // same implicit GEMM with the taps mirrored and the channel matrices
    // transposed; in this element's indices: K chunk / el = output channel, n = input channel
    const int tap_m = (kx - 1 - tap / ky) * ky + (ky - 1 - tap % ky);
    const float wb = params[w_off[j + 1] + ((int64_t)tap_m * C + co) * C + ci];
    wimg_b[e] = split_part(wb, split);
  }
  if (blockIdx.x == 0) {
    // layer 1: [pair][dx_local][n = split * C + co][slot e = dy]; zero beyond the kernel
    for (int e = threadIdx.x; e < n_pairs * 2 * 3 * C * 8; e += blockDim.x) {
      int r = e;
      const int pr = r / (2 * 3 * C * 8); r -= pr * 2 * 3 * C * 8;
      const int dl = r / (3 * C * 8); r -= dl * 3 * C * 8;
      const int n = r / 8, dy = r - 8 * n;
      const int split = n / C, co = n - split * C;
      const int dx = 2 * pr + dl;
      float w = 0.f;
      if (dx < kx && dy < ky) w = params[w_off[0] + (int64_t)(dx * ky + dy) * C + co];   // [tap][0][co]
      w1img[e] = split_part(w, split);
    }
    for (int e = threadIdx.x; e < (L - 1) * C; e += blockDim.x)
      bias[e] = params[b_off[e / C] + e % C];
    for (int ci = threadIdx.x; ci < C; ci += blockDim.x) {
      float s = 0.f;
      for (int tap = 0; tap < taps; ++tap)
        for (int co = 0; co < C; ++co) s += params[w_off[L - 1] + ((int64_t)tap * C + ci) * C + co];
      wsum[ci] = s;
    }
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int co = 0; co < C; ++co) s += params[b_off[L - 1] + co];
      wsum[C] = (float)N * s;
    }
  }
}

// CGSVMC_CONV_TC=0 routes the convolutional ansaetze to the SIMT tile kernels
// (read at every call so that tests can compare the two paths).
bool tc_enabled() {
  const char* e = getenv("CGSVMC_CONV_TC");
  return e == nullptr || atoi(e) != 0;
}

// rows / tiles / TMEM columns of a plan with G configurations
void size_plan(TcDesc* t, int G) {
  t->G = G; t->GW = G * t->PW;
  t->ystep = t->il ? G : 1;
  t->rows_out = t->X * t->GW;
  t->n_tiles = (t->rows_out + 127) / 128;
  // the junk output rows of the last tile read up to the largest tap shift further
  t->rows_total = (t->n_tiles * 128 + (t->kx - 1) * t->GW + (t->ky - 1) * t->ystep + 1 + 7) / 8 * 8;
  t->rows_total = std::max(t->rows_total, (t->PH * t->GW + 8 + 7) / 8 * 8);
  int cols = 32;
  while (cols < t->n_tiles * 3 * t->C) cols *= 2;
  t->tmem_cols = cols;
}

bool make_desc_plan(const cgsvmc_ansatz* a, size_t extra_bytes_per_cfg, size_t extra_fixed, int ctas, int il,
                    TcDesc* out);

// Geometry and shared-memory plan; false when the network is outside the
// tensor-core path (the SIMT tile kernels of net.cu take over).  Plans in order
// of measured throughput (C3 / C4 / 16x16, profiles/r02g_*): two CTAs per SM
// before one, and within that the interleaved layout before the side-by-side
// one.  With two CTAs each runs its layers as [MMAs of all tiles] -> [epilogue
// of all tiles]: the tensor pipe works for one while the other runs its
// epilogue, and the single weight buffer is refilled under the epilogue.  The
// one-CTA plan (larger batches, double-buffered weights) takes what two do not fit.
bool make_desc_host(const cgsvmc_ansatz* a, size_t extra_bytes_per_cfg, size_t extra_fixed, TcDesc* out) {
  for (int ctas = 2; ctas >= 1; --ctas)
    for (int il = 1; il >= 0; --il)
      if (make_desc_plan(a, extra_bytes_per_cfg, extra_fixed, ctas, il, out)) return true;
  return false;
}

bool make_desc_plan(const cgsvmc_ansatz* a, size_t extra_bytes_per_cfg, size_t extra_fixed, int ctas, int il,
                    TcDesc* out) {
  const cgsvmc_ansatz_desc& s = a->desc;
  if (s.kind != CGSVMC_ANSATZ_CONV_1D && s.kind != CGSVMC_ANSATZ_CONV_2D) return false;
  if (s.num_layers < 3 || (s.num_filters != 16 && s.num_filters != 32)) return false;
  TcDesc d;
  memset(&d, 0, sizeof(d));
  d.N = s.n_sites; d.C = s.num_filters; d.L = s.num_layers; d.act = s.nonlinearity;
  d.NW = n_words(s.n_sites);
  if (s.kind == CGSVMC_ANSATZ_CONV_1D) {
    d.X = s.n_sites; d.Y = 1; d.kx = s.kernel_size; d.ky = 1;
    d.pad_x = s.kernel_size % 2 ? (s.kernel_size - 1) / 2 : s.kernel_size / 2;       // layers.py:64-73
    d.pad_y = 0;
  } else {
    d.X = s.size_x; d.Y = s.size_y; d.kx = d.ky = s.kernel_size;
    d.pad_x = d.pad_y = s.kernel_size % 2 ? (s.kernel_size - 1) / 2 : s.kernel_size / 2 - 1;   // layers.py:132-141
  }
  if (d.kx > d.X || d.ky > d.Y || d.kx * d.ky > kMaxTaps || d.ky > 8) return false;
  d.PH = d.X + d.kx - 1; d.PW = d.Y + d.ky - 1;
  d.n_tensor = d.L - 2;
  d.n_pairs = (d.kx + 1) / 2;
  d.wbuf_bytes = d.kx * d.ky * 3 * d.C * d.C * 2;
  // two CTAs share the SM's 228 KB, 1 KB of each CTA's share is reserved by the
  // driver; a little is kept for the kernels' static __shared__ variables
  const size_t limit = ctas == 1 ? (size_t)a->max_smem_optin : (size_t)(233472 / 2 - 1024 - 256);
  const int tmem_limit = 512 / ctas;
  d.ctas = ctas;
  d.il = il;
  bool found = false;
  // side by side, one CTA per SM: double-buffered weights (the next layer's load
  // overlaps the MMAs) when at least two configurations still fit; otherwise one
  // buffer, refilled under the epilogue
  for (int n_wbuf = (ctas == 1 && !il) ? 2 : 1; n_wbuf >= 1 && !found; --n_wbuf) {
    const int g_min = il ? 8 : ((n_wbuf == 2 || ctas == 2) ? 2 : 1);
    const int g_step = il ? 8 : 1;
    for (int G = 16; G >= g_min; G -= g_step) {
      TcDesc t = d;
      t.n_wbuf = n_wbuf;
      size_plan(&t, G);
      if (t.rows_total > 16383 || t.n_tiles * 3 * t.C > tmem_limit) continue;
      const size_t need = smem_plan(t).total + (size_t)G * t.NW * 16 + (size_t)G * 12 + 16 +
                          extra_bytes_per_cfg * G + extra_fixed + 1024;
      if (need <= limit) { d = t; found = true; break; }
    }
  }
  if (!found) return false;
  *out = d;
  return true;
}

int build_tc_image(cgsvmc_ansatz* a, TcDesc* d, cudaStream_t st) {
  const int taps = d->kx * d->ky;
  (void)taps;
  const int64_t wimg_halfs = (int64_t)d->n_tensor * taps * 3 * d->C * d->C;
  const size_t off_bytes = (size_t)2 * d->L * sizeof(int64_t);
  const size_t off_pad = (off_bytes + 255) / 256 * 256;
  const size_t small_bytes = (((size_t)(d->L - 1) * d->C + d->C + 4) * 4 + 255) / 256 * 256;
  const size_t w1_bytes = ((size_t)d->n_pairs * 2 * 3 * d->C * 16 + 255) / 256 * 256;
  const size_t wimg_bytes = ((size_t)wimg_halfs * 2 + 255) / 256 * 256;
  const size_t bytes = off_pad + small_bytes + w1_bytes + 2 * wimg_bytes;
  if (a->tables_bytes < bytes) {
    if (a->tables != nullptr) {
      if (int rc = cuda_fail(cudaDeviceSynchronize(), "tables sync")) return rc;
      cudaFree(a->tables);
      a->tables = nullptr;
      a->tables_bytes = 0;
    }
    if (int rc = cuda_fail(cudaMalloc(&a->tables, bytes), "tables alloc")) return rc;
    a->tables_bytes = bytes;
    a->tables_valid = false;
    // flat offsets of every layer's weights and biases
    std::vector<int64_t> offs(2 * d->L);
    for (int l = 0; l < d->L; ++l) { offs[l] = a->offsets[2 * l]; offs[d->L + l] = a->offsets[2 * l + 1]; }
    if (int rc = cuda_fail(cudaMemcpy(a->tables, offs.data(), off_bytes, cudaMemcpyHostToDevice),
                           "tables offsets"))
      return rc;
  }
  char* base = reinterpret_cast<char*>(a->tables);
  const int64_t* w_off = reinterpret_cast<const int64_t*>(base);
  const int64_t* b_off = w_off + d->L;
  float* bias = reinterpret_cast<float*>(base + off_pad);
  float* wsum = bias + (int64_t)(d->L - 1) * d->C;
  __half* w1img = reinterpret_cast<__half*>(base + off_pad + small_bytes);
  __half* wimg = reinterpret_cast<__half*>(base + off_pad + small_bytes + w1_bytes);
  __half* wimg_b = reinterpret_cast<__half*>(base + off_pad + small_bytes + w1_bytes + wimg_bytes);
  d->w1img = w1img;
  d->wimg = wimg;
  d->wimg_b = wimg_b;
  d->bias = bias;
  d->wsum = wsum;
  if (a->track_params && a->tables_valid) return CGSVMC_OK;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((wimg_halfs + 255) / 256, 592));
  tc_prep_kernel<<<blocks, 256, 0, st>>>(d->kx, d->ky, d->C, d->L, d->N, d->n_pairs, a->params, w_off, b_off,
                                         w1img, wimg, wimg_b, wimg_halfs, bias, wsum, d->n_tensor);
  a->tables_valid = true;
  return cuda_fail(cudaGetLastError(), "conv_tc prep launch");
}

template <typename F>
int opt_in(F kernel, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(smem)");
  return CGSVMC_OK;
}

}  // namespace

bool conv_tc_supported(const cgsvmc_ansatz* a, const cgsvmc_ham* h) {
  if (!tc_enabled()) return false;
  TcDesc d;
  const size_t fixed = h != nullptr ? (size_t)(h->n_bonds + 1) * 6 + 16 : 0;
  if (h != nullptr && h->n_bonds >= 65535) return false;
  return make_desc_host(a, 0, fixed, &d);
}

// Launches KERNEL<C, CTAS> for the plan `d` (C in {16, 32}, one or two CTAs per SM).
#define CGSVMC_TC_LAUNCH(KERNEL, grid, smem, st, ...)                                           \
  do {                                                                                          \
    if (d.C == 16 && d.ctas == 2) {                                                             \
      if (int rc = opt_in(KERNEL<16, 2>, smem)) return rc;                                      \
      KERNEL<16, 2><<<grid, kThreads, smem, st>>>(__VA_ARGS__);                                 \
    } else if (d.C == 16) {                                                                     \
      if (int rc = opt_in(KERNEL<16, 1>, smem)) return rc;                                      \
      KERNEL<16, 1><<<grid, kThreads, smem, st>>>(__VA_ARGS__);                                 \
    } else if (d.ctas == 2) {                                                                   \
      if (int rc = opt_in(KERNEL<32, 2>, smem)) return rc;                                      \
      KERNEL<32, 2><<<grid, kThreads, smem, st>>>(__VA_ARGS__);                                 \
    } else {                                                                                    \
      if (int rc = opt_in(KERNEL<32, 1>, smem)) return rc;                                      \
      KERNEL<32, 1><<<grid, kThreads, smem, st>>>(__VA_ARGS__);                                 \
    }                                                                                           \
  } while (0)

// The parameter image for conv_tc_grad.cu (same buffers the forward kernels read).
int conv_tc_image(cgsvmc_ansatz* a, ConvTcImage* img, cudaStream_t st) {
  TcDesc d;
  if (!make_desc_host(a, 0, 0, &d)) { set_error("conv_tc: unsupported network"); return CGSVMC_ERR_UNSUPPORTED; }
  if (int rc = build_tc_image(a, &d, st)) return rc;
  img->w1img = d.w1img; img->wimg = d.wimg; img->wimg_b = d.wimg_b; img->bias = d.bias; img->wsum = d.wsum;
  return CGSVMC_OK;
}

int conv_tc_log_amp(cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, float* out, cudaStream_t st) {
  TcDesc d;
  if (!make_desc_host(a, 0, 0, &d)) { set_error("conv_tc: unsupported network"); return CGSVMC_ERR_UNSUPPORTED; }
  if (int rc = build_tc_image(a, &d, st)) return rc;
  const size_t smem = smem_plan(d).total + extras_bytes(d);
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((B + d.G - 1) / d.G, (int64_t)a->num_sms * d.ctas));
  CGSVMC_TC_LAUNCH(tc_log_amp_kernel, grid, smem, st, d, packed, B, out);
  return cuda_fail(cudaGetLastError(), "conv_tc log_amp launch");
}

int conv_tc_mc_steps(cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int n_steps, uint64_t seed,
                     uint64_t walker0, uint64_t step0, unsigned long long* accept_count,
                     float* log_amp_out, cudaStream_t st) {
  TcDesc d;
  if (!make_desc_host(a, 0, 0, &d)) { set_error("conv_tc: unsupported network"); return CGSVMC_ERR_UNSUPPORTED; }
  // do not starve the grid: fewer walkers per CTA when there are few walkers
  // (interleaved plans keep G a multiple of 8)
  const int g_step = d.il ? 8 : 1;
  while (d.G > g_step && (B + d.G - 1) / d.G < (int64_t)a->num_sms * d.ctas) size_plan(&d, d.G - g_step);
  if (int rc = build_tc_image(a, &d, st)) return rc;
  const size_t smem = smem_plan(d).total + extras_bytes(d);
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((B + d.G - 1) / d.G, (int64_t)a->num_sms * d.ctas));
  CGSVMC_TC_LAUNCH(tc_mc_kernel, grid, smem, st, d, packed, B, n_steps, seed, walker0, step0,
                   a->step_counter_dev, accept_count, log_amp_out);
  return cuda_fail(cudaGetLastError(), "conv_tc mc launch");
}

int conv_tc_local_energy(cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                         float* e_loc, float* log_amp_out, float* diag_out, float* off_out,
                         cudaStream_t st) {
  TcDesc d;
  const size_t fixed = (size_t)(h->n_bonds + 1) * 6 + 16;
  if (!make_desc_host(a, 0, fixed, &d)) { set_error("conv_tc: unsupported network"); return CGSVMC_ERR_UNSUPPORTED; }
  if (int rc = build_tc_image(a, &d, st)) return rc;
  const size_t smem = smem_plan(d).total + extras_bytes(d) + fixed;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(B, (int64_t)a->num_sms * d.ctas));
  CGSVMC_TC_LAUNCH(tc_eloc_kernel, grid, smem, st, d, h->ij, h->jx, h->jz, h->n_bonds, packed, B, e_loc,
                   log_amp_out, diag_out, off_out);
  return cuda_fail(cudaGetLastError(), "conv_tc local_energy launch");
}

}  // namespace cgsvmc

#ifdef CGSVMC_RBM2_TIMING
// Development build only: reads (and clears) the conv_tc phase counters
// [MMA cycles, epilogue cycles, tensor layers, forwards], summed over CTAs.
extern "C" int cgsvmc_debug_conv_tc_phases(unsigned long long* host_out) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpyFromSymbol(host_out, cgsvmc::g_tc_phase, 4 * sizeof(unsigned long long));
  unsigned long long zero[4] = {0, 0, 0, 0};
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(cgsvmc::g_tc_phase, zero, sizeof(zero));
  return e == cudaSuccess ? 0 : -2;
}
#endif
