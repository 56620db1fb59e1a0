// Pure RBM ansatz (rbm with num_fc_layers == 0), second-generation kernels.
//
//   z(sigma) = a . sigma + a0 + sum_j log cosh(theta_j),  theta = W^T sigma + c
//                                                   (wavefunctions.py:410-436)
//
// Amplitude RATIOS are all the sampler (graph_builders.py:74-79) and the local
// energy (operators.py:168-169, 259) need.  For the exchange "raise site d,
// lower site u" theta'_j = theta_j + delta_j, delta_j = 2 W[d][j] - 2 W[u][j], and
//
//   cosh(theta + delta) / cosh(theta) = e^{-delta} (p e^{2 delta} + m),
//   p = (1 + tanh theta) / 2,  m = (1 - tanh theta) / 2          (p + m = 1)
//
// so with the per-site tables F = e^{4W}, G = e^{-4W} (e^{2 delta_j} =
// F[d][j] G[u][j]) and the per-site scalar A2[i] = 2 log2(e) (a_i - sum_j W[i][j])
//
//   log2 psi'/psi = A2[d] - A2[u] + sum_j log2(p_j F[d][j] G[u][j] + m_j).
//
// The inner loop is 2 table loads + 4 FP32 ops per hidden unit and NO
// transcendental (one lg2 per 4 hidden units, on a product); the walker state
// is (p_j, m_j) in registers, updated multiplicatively on acceptance
// (p' = p y / n, m' = m / n, n = p y + m).  All tables live in shared memory
// (copied once per CTA with a TMA bulk copy) when they fit.
//
// Mapping: LPW lanes own one walker (LPW = 8: four walkers per warp, 16: two);
// with VW = 32 / LPW lane `sub` holds hidden units j = VW (sub + LPW q) + c,
// q < KJV = HP / 32, c < VW, so a table row is read with LDS.128 / LDS.64 in
// phases of one walker (128 contiguous bytes) each -- conflict-free.
// One persistent CTA per SM (the sampler kernel: 1024 threads when the state
// fits 64 registers; the walker kernel: always 512 threads / 128 registers).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "internal.h"
#include "rbm2.h"

namespace cgsvmc {
namespace rbm2 {

// Development aid (-DCGSVMC_RBM2_TIMING, profiles/run_rbm2_phases.py): thread 0
// of every CTA stamps %globaltimer / clock64 at the phase boundaries.
#ifdef CGSVMC_RBM2_TIMING
#define RBM2_TIMING_MARKS 12
static __device__ unsigned long long g_phase_marks[2][160][RBM2_TIMING_MARKS][2];
#define RBM2_MARK(KERN, K)                                                            \
  do {                                                                                \
    if (threadIdx.x == 0 && blockIdx.x < 160) {                                       \
      unsigned long long gt_;                                                         \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                         \
      g_phase_marks[KERN][blockIdx.x][K][0] = gt_;                                    \
      g_phase_marks[KERN][blockIdx.x][K][1] = (unsigned long long)clock64();          \
    }                                                                                 \
  } while (0)
#else
#define RBM2_MARK(KERN, K) do {} while (0)
#endif

// ---------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ float lg2_approx(float x) {
  float l;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(x));
  return l;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
  return e;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Packed FP32 (sm_100 FMUL2 / FFMA2 / FADD2): two IEEE operations per issue
// slot -- the ratio loops are issue-bound, not FMA-pipe bound
// (profiles/microbench/fp32_pipes.cu).
__device__ __forceinline__ void mul2(float& o0, float& o1, float a0, float a1, float b0, float b1) {
  asm("{ .reg .b64 ra, rb; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5};\n"
      "  mul.rn.f32x2 ra, ra, rb; mov.b64 {%0, %1}, ra; }"
      : "=f"(o0), "=f"(o1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
__device__ __forceinline__ void fma2(float& o0, float& o1, float a0, float a1, float b0, float b1,
                                     float c0, float c1) {
  asm("{ .reg .b64 ra, rb, rc; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; mov.b64 rc, {%6, %7};\n"
      "  fma.rn.f32x2 ra, ra, rb, rc; mov.b64 {%0, %1}, ra; }"
      : "=f"(o0), "=f"(o1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1), "f"(c0), "f"(c1));
}
__device__ __forceinline__ void add2(float& o0, float& o1, float a0, float a1, float b0, float b1) {
  asm("{ .reg .b64 ra, rb; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5};\n"
      "  add.rn.f32x2 ra, ra, rb; mov.b64 {%0, %1}, ra; }"
      : "=f"(o0), "=f"(o1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}

// VW consecutive floats (VW = 4: LDS.128, 2: LDS.64)
template <int VW, bool WS>
__device__ __forceinline__ void ldv(const float* p, float (&v)[VW]) {
  if (VW == 4) {
    const float4 x = WS ? *reinterpret_cast<const float4*>(p) : __ldg(reinterpret_cast<const float4*>(p));
    v[0] = x.x; v[1] = x.y; v[2 % VW] = x.z; v[3 % VW] = x.w;
  } else {
    const float2 x = WS ? *reinterpret_cast<const float2*>(p) : __ldg(reinterpret_cast<const float2*>(p));
    v[0] = x.x; v[1] = x.y;
  }
}
template <int VW>
__device__ __forceinline__ void stv(float* p, const float (&v)[VW]) {
  if (VW == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2 % VW], v[3 % VW]);
  else *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
}
template <bool WS>
__device__ __forceinline__ float ld1(const float* p) {
  if (WS) return *p;
  return __ldg(p);
}

template <int LPW>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LPW / 2; o > 0; o >>= 1) v += __shfl_xor_sync(CGSVMC_FULL_MASK, v, o);
  return v;
}

// TMA bulk copies global -> shared of `bytes` (a multiple of 16) completing on
// the mbarrier at shared address bar_a (issued by one thread; the caller has
// armed the barrier with the expected byte count)
__device__ __forceinline__ void bulk_copy(void* dst, const void* src, uint32_t bytes, uint32_t bar_a) {
  char* d = reinterpret_cast<char*>(dst);
  const char* g = reinterpret_cast<const char*>(src);
  for (uint32_t done = 0; done < bytes;) {
    const uint32_t chunk = min(bytes - done, 32768u);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(d + done)),
                 "l"(g + done), "r"(chunk), "r"(bar_a)
                 : "memory");
    done += chunk;
  }
}

__device__ __forceinline__ void mbar_wait(uint32_t bar_a, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok)
                 : "r"(bar_a), "r"(parity)
                 : "memory");
}

// TMA bulk copy global -> shared of the parameter image; every thread returns
// after the bytes have landed.  `bar` is an 8-byte shared mbarrier.
// (a second region -- the bond-pair table -- may ride on the same barrier)
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar,
                                          void* dst2 = nullptr, const void* src2 = nullptr,
                                          uint32_t bytes2 = 0, void* dst3 = nullptr,
                                          const void* src3 = nullptr, uint32_t bytes3 = 0) {
  const uint32_t bar_a = smem_u32(bar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a),
                 "r"(bytes + bytes2 + bytes3)
                 : "memory");
    bulk_copy(dst, src, bytes, bar_a);
    bulk_copy(dst2, src2, bytes2, bar_a);
    bulk_copy(dst3, src3, bytes3, bar_a);
  }
  mbar_wait(bar_a, 0u);
}

// select-in-byte table: lut[v * 8 + r] = index of the r-th set bit of v
__device__ __forceinline__ uint8_t lut_entry(int e) {
  const int v = e >> 3, r = e & 7;
  int pos = 0, seen = 0;
  for (int b = 0; b < 8; ++b)
    if ((v >> b) & 1) { if (seen == r) pos = b; ++seen; }
  return (uint8_t)(r < seen ? pos : 0);
}
// The table travels inside the parameter image (prep_kernel) when the image
// is copied to shared memory; otherwise the CTA builds its own copy.
__device__ __forceinline__ void build_lut(uint8_t* lut) {
  for (int e = threadIdx.x; e < 2048; e += blockDim.x) lut[e] = lut_entry(e);
}

constexpr float kTcgPrescale = 9.5367431640625e-07f;   // 2^-20: E_loc prescale of the tensor-core gradient operands

struct Tables {
  const float* w2;    // [N][HP]  2 W
  const float* f;     // [N][HP]  exp(4 W)
  const float* g;     // [N][HP]  exp(-4 W)
  const float* a2;    // [NP]     2 log2(e) (a_i - sum_j W_ij)
  const float* base;  // [HP]     c_j - sum_i W_ij
  const float* a;     // [NP]
  const float* a0;    // [4]: a0, max |W|, 0, 0
};

__device__ __forceinline__ Tables tables_at(const float* img, const Image& im) {
  Tables t;
  t.w2 = img + im.off_w2; t.f = img + im.off_f; t.g = img + im.off_g;
  t.a2 = img + im.off_a2; t.base = img + im.off_base; t.a = img + im.off_a; t.a0 = img + im.off_a0;
  return t;
}

template <int NW>
__device__ __forceinline__ int spin_bit(const uint64_t (&s)[NW], int site) {
  uint64_t w = s[0];
#pragma unroll
  for (int i = 1; i < NW; ++i) if ((site >> 6) == i) w = s[i];
  return (int)((w >> (site & 63)) & 1ull);
}

// ---------------------------------------------------------------------------
// walker state
// ---------------------------------------------------------------------------
// theta_j = base_j + sum_{i up} 2 W[i][j];  p = 1 / (1 + e^{-2 theta}),
// m = 1 / (1 + e^{2 theta}).  Optionally returns this lane's share of
// sum_j log cosh theta_j + a . sigma (group_sum + a0 gives z).
// W2S: the 2W rows are in shared memory (default: wherever the image is).
template <int NW, int LPW, int KJV, bool WS, bool W2S = WS>
__device__ __forceinline__ float init_state(const Tables& t, const Image& im, const uint64_t (&s)[NW],
                                            int sub, float (&p)[32 / LPW * KJV],
                                            float (&m)[32 / LPW * KJV], bool want_z) {
  constexpr int VW = 32 / LPW, KJ = VW * KJV, HP = 32 * KJV;
  float th[KJ];
#pragma unroll
  for (int q = 0; q < KJV; ++q) {
    float v[VW];
    ldv<VW, WS>(t.base + VW * sub + 32 * q, v);
#pragma unroll
    for (int c = 0; c < VW; ++c) th[VW * q + c] = v[c];
  }
#pragma unroll
  for (int w = 0; w < NW; ++w) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t bits = (uint32_t)(s[w] >> (32 * h));
      const float* rows = t.w2 + (64 * w + 32 * h) * HP + VW * sub;
      while (bits) {
        const int i = __ffs((int)bits) - 1;
        bits &= bits - 1;
        const float* row = rows + i * HP;
#pragma unroll
        for (int q = 0; q < KJV; ++q) {
          float v[VW];
          ldv<VW, W2S>(row + 32 * q, v);
#pragma unroll
          for (int c = 0; c < VW; c += 2)
            add2(th[VW * q + c], th[VW * q + c + 1], th[VW * q + c], th[VW * q + c + 1], v[c], v[c + 1]);
        }
      }
    }
  }
  float zpart = 0.f;
#pragma unroll
  for (int k = 0; k < KJ; ++k) {
    // e = exp(-2|theta|) in (0, 1]; the MUFU approximations are good to ~2^-22
    // relative (ex2, rcp) / absolute (lg2 on [1, 2]) -- float32 rounding level
    const float ax = fabsf(th[k]);
    const float e = ex2_approx(-2.885390081777927f * ax);
    const float r = rcp_approx(1.f + e);
    const float big = r, small = e * r;
    p[k] = th[k] >= 0.f ? big : small;
    m[k] = th[k] >= 0.f ? small : big;
    if (want_z) zpart += fmaf(lg2_approx(1.f + e), 0.6931471805599453f, ax - 0.6931471805599453f);
  }
  if (want_z) {
    for (int i = sub; i < im.N; i += LPW) {
      const float ai = ld1<WS>(t.a + i);
      zpart += spin_bit<NW>(s, i) ? ai : -ai;
    }
  }
  return zpart;
}

// This lane's share of sum_j log2(p_j F[d][j] G[u][j] + m_j) for "raise site d,
// lower site u" (uniform within the lane group).  KEEP: also return tq[k] =
// F[d][j] G[u][j] for the acceptance update.  The fast form takes one lg2 per
// FOUR hidden units, on the product of their terms; with very large weights
// (or a far-from-normalised sampler state) that product can leave the float32
// range, so callers re-evaluate with SAFE = true (one lg2 per term) whenever a
// group total comes out non-finite.
template <int LPW, int KJV, bool WS, bool KEEP, bool SAFE = false>
__device__ __forceinline__ float exchange_log2_partial(const Tables& t, int d, int u, int sub,
                                                       const float (&p)[32 / LPW * KJV],
                                                       const float (&m)[32 / LPW * KJV],
                                                       float (&tq)[32 / LPW * KJV]) {
  constexpr int VW = 32 / LPW, KJ = VW * KJV, HP = 32 * KJV;
  const float* fr = t.f + d * HP + VW * sub;
  const float* gr = t.g + u * HP + VW * sub;
  float n[KJ];
#pragma unroll
  for (int q = 0; q < KJV; ++q) {
    float f[VW], g[VW];
    ldv<VW, WS>(fr + 32 * q, f);
    ldv<VW, WS>(gr + 32 * q, g);
#pragma unroll
    for (int c = 0; c < VW; c += 2) {
      const int k = VW * q + c;
      float fg0, fg1;
      mul2(fg0, fg1, f[c], f[c + 1], g[c], g[c + 1]);
      if (KEEP) { tq[k] = fg0; tq[k + 1] = fg1; }
      fma2(n[k], n[k + 1], p[k], p[k + 1], fg0, fg1, m[k], m[k + 1]);
    }
  }
  float lsum = 0.f;
  if (SAFE) {
#pragma unroll
    for (int k = 0; k < KJ; ++k) lsum += lg2_approx(n[k]);
  } else {
    // products of four terms, one lg2 each
#pragma unroll
    for (int k = 0; k < KJ; k += 4) {
      float pr;
      if (k + 3 < KJ) {
        float q0, q1;
        mul2(q0, q1, n[k], n[k + 1], n[k + 2], n[k + 3]);
        pr = q0 * q1;
      } else {
        pr = n[k] * n[k + 1];
      }
      lsum += lg2_approx(pr);
    }
  }
  return lsum;
}

// log2(psi'/psi) of the exchange, reduced over the lane group.
template <int LPW, int KJV, bool WS, bool KEEP>
__device__ __forceinline__ float exchange_log2_ratio(const Tables& t, int d, int u, int sub,
                                                     const float (&p)[32 / LPW * KJV],
                                                     const float (&m)[32 / LPW * KJV],
                                                     float (&tq)[32 / LPW * KJV]) {
  const float lsum = group_sum<LPW>(exchange_log2_partial<LPW, KJV, WS, KEEP>(t, d, u, sub, p, m, tq));
  return lsum + (ld1<WS>(t.a2 + d) - ld1<WS>(t.a2 + u));
}

// Butterfly transpose-reduce over a lane group: on entry part[i] is this
// lane's share of quantity i (i < LPW); on exit part[0] of lane `sub` is the
// group total of quantity `sub`.  LPW - 1 shuffles for LPW sums (a plain
// all-reduce of each would take LPW log2 LPW).
template <int LPW>
__device__ __forceinline__ void transpose_reduce(float (&part)[LPW], int sub) {
#pragma unroll
  for (int o = LPW / 2; o > 0; o >>= 1) {
    const bool upper = (sub & o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = upper ? part[i] : part[i + o];
      const float keep = upper ? part[i + o] : part[i];
      part[i] = keep + __shfl_xor_sync(CGSVMC_FULL_MASK, send, o);
    }
  }
}

// This lane's share of sum_j log2(p_j T_j + m_j) with T = one row of the
// bond-pair table (T_j = F[d][j] G[u][j], formed by pair_prep_kernel with the
// same multiply as exchange_log2_partial: identical values, half the
// shared-memory traffic and no FMUL2 per pair of hidden units).
template <int LPW, int KJV, bool WS = true>
__device__ __forceinline__ float pair_log2_partial(const float* __restrict__ row, int sub,
                                                   const float (&p)[32 / LPW * KJV],
                                                   const float (&m)[32 / LPW * KJV]) {
  constexpr int VW = 32 / LPW, KJ = VW * KJV;
  float n[KJ];
#pragma unroll
  for (int q = 0; q < KJV; ++q) {
    float tv[VW];
    ldv<VW, WS>(row + VW * sub + 32 * q, tv);
#pragma unroll
    for (int c = 0; c < VW; c += 2) {
      const int k = VW * q + c;
      fma2(n[k], n[k + 1], p[k], p[k + 1], tv[c], tv[c + 1], m[k], m[k + 1]);
    }
  }
  float lsum = 0.f;
#pragma unroll
  for (int k = 0; k < KJ; k += 4) {
    float pr;
    if (k + 3 < KJ) {
      float q0, q1;
      mul2(q0, q1, n[k], n[k + 1], n[k + 2], n[k + 3]);
      pr = q0 * q1;
    } else {
      pr = n[k] * n[k + 1];
    }
    lsum += lg2_approx(pr);
  }
  return lsum;
}

// One round of the local-energy off-diagonal sum: R (= LPW or LPW / 2) listed
// bonds of this walker starting at it0.  list entry = site to raise | site to
// lower << 8 | bond index << 16; bond_s[k].z = j_x bits.  Returns this lane's
// share of sum_k 0.5 j_x psi(flip_k) / psi (operators.py:168-169).
// pair_s != nullptr: rows of the bond-pair table (row 2 k + o, o = bit 31 of
// the entry: which end of bond k is raised) instead of two site rows.
template <int R, int LPW, int KJV, bool WS>
__device__ __forceinline__ float ratio_round(const Tables& t, const uint32_t* list, const int4* bond_s,
                                             int it0, int cnt, int sub,
                                             const float (&p)[32 / LPW * KJV],
                                             const float (&m)[32 / LPW * KJV],
                                             const float* pair_s = nullptr) {
  constexpr int HP = 32 * KJV;
  float part[R], tdummy[32 / LPW * KJV];
  if (pair_s != nullptr) {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const uint32_t ent = it0 + i < cnt ? list[it0 + i] : 0u;
      const int row = (int)(((ent >> 16) & 0x7fffu) * 2u + (ent >> 31));
      part[i] = pair_log2_partial<LPW, KJV, WS>(pair_s + (size_t)row * HP, sub, p, m);
    }
  } else {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const uint32_t ent = it0 + i < cnt ? list[it0 + i] : 0u;
      part[i] = exchange_log2_partial<LPW, KJV, WS, false>(t, (int)(ent & 0xffu), (int)((ent >> 8) & 0xffu),
                                                           sub, p, m, tdummy);
    }
  }
  // partial round (R < LPW): fold the sub-groups of R lanes first
#pragma unroll
  for (int o = LPW / 2; o >= R; o >>= 1) {
#pragma unroll
    for (int i = 0; i < R; ++i) part[i] += __shfl_xor_sync(CGSVMC_FULL_MASK, part[i], o);
  }
  transpose_reduce<R>(part, sub & (R - 1));
  const int it = it0 + (sub & (R - 1));
  const bool mine = it < cnt && sub < R;
  const uint32_t ent = mine ? list[it] : 0u;
  const int dn = (int)(ent & 0xffu), up = (int)((ent >> 8) & 0xffu);
  float total = part[0];
  // rare: a four-term product left the float32 range -- redo this lane's bond term by term
  const uint32_t bad = __ballot_sync(CGSVMC_FULL_MASK, mine && !(fabsf(total) <= 3.0e38f));
  if (bad != 0u) {
    constexpr uint32_t REP = LPW == 4 ? 0x11111111u : LPW == 8 ? 0x01010101u : LPW == 16 ? 0x00010001u : 1u;
    for (int l = 0; l < LPW; ++l) {
      if ((bad & (REP << l)) == 0u) continue;                       // warp-uniform
      const uint32_t e2 = __shfl_sync(CGSVMC_FULL_MASK, ent, l, LPW);
      const float v = group_sum<LPW>(exchange_log2_partial<LPW, KJV, WS, false, true>(
          t, (int)(e2 & 0xffu), (int)((e2 >> 8) & 0xffu), sub, p, m, tdummy));
      if (sub == l && ((bad >> (threadIdx.x & 31)) & 1u)) total = v;
    }
  }
  float term = 0.f;
  if (mine) {
    // (explicit roundings: no FMA contraction, so the fused, split and
    // gradient-less instantiations give bit-identical local energies)
    const float l2 = __fadd_rn(total, __fsub_rn(ld1<WS>(t.a2 + dn), ld1<WS>(t.a2 + up)));
    term = __fmul_rn(0.5f * __int_as_float(bond_s[(ent >> 16) & 0x7fffu].z), ex2_approx(l2));
  }
  return term;
}

// ---------------------------------------------------------------------------
// uniformly random up site and down site: the k_up-th set bit and the k_dn-th
// clear (valid) bit in site order, resolved by the LPW lanes of the group
// (each owns CB = 64 NW / LPW bits) with a packed prefix scan and the
// select-in-byte table.
// ---------------------------------------------------------------------------
template <int CB>
__device__ __forceinline__ int select_in_chunk(uint32_t c, int r, const uint8_t* lut) {
  int base = 0;
  if (CB > 16) {
    const int pc = __popc(c & 0xffffu);
    if (r >= pc) { r -= pc; c >>= 16; base += 16; }
    c &= 0xffffu;
  }
  if (CB > 8) {
    const int pc = __popc(c & 0xffu);
    if (r >= pc) { r -= pc; c >>= 8; base += 8; }
    c &= 0xffu;
  }
  return base + lut[c * 8 + r];
}

template <int NW, int LPW>
struct SitePicker {
  static constexpr int CB = 64 * NW / LPW;
  int word, shift, sub;
  uint32_t vchunk;
  uint64_t vword;
  static __device__ __forceinline__ int select_in_word(uint64_t w, int r, const uint8_t* lut) {
    uint32_t c = (uint32_t)w;
    int base = 0;
    const int pl = __popc(c);
    if (r >= pl) { r -= pl; c = (uint32_t)(w >> 32); base = 32; }
    return base + select_in_chunk<32>(c, r, lut);
  }
  __device__ __forceinline__ void setup(int n_sites, int sub_) {
    sub = sub_;
    vword = valid_mask_word(n_sites, 0);
    word = (CB * sub) >> 6;
    shift = (CB * sub) & 63;
    const uint64_t vm = valid_mask_word(n_sites, word);
    vchunk = (uint32_t)(vm >> shift) & (CB == 32 ? 0xffffffffu : ((1u << CB) - 1u));
  }
  __device__ __forceinline__ void pick(const uint64_t (&s)[NW], int k_up, int k_dn,
                                       const uint8_t* lut, int& up, int& dn) const {
    if (NW == 1) {
      // one word: popcount bisection + the select-in-byte table, no prefix scan
      // (the lower half of the lane group resolves the up site, the upper
      // half the down site: one select per lane, two broadcasts)
      const bool lower = sub < LPW / 2;
      const int r = select_in_word((lower ? s[0] : ~s[0]) & vword, lower ? k_up : k_dn, lut);
      up = __shfl_sync(CGSVMC_FULL_MASK, r, 0, LPW);
      dn = __shfl_sync(CGSVMC_FULL_MASK, r, LPW / 2, LPW);
      return;
    }
    uint64_t wv = s[0];
#pragma unroll
    for (int i = 1; i < NW; ++i) if (word == i) wv = s[i];
    const uint32_t chunk = (uint32_t)(wv >> shift);
    const uint32_t cu = chunk & vchunk, cd = ~chunk & vchunk;
    const int nu = __popc(cu), nd = __popc(cd);
    const uint32_t cnt = (uint32_t)nu | ((uint32_t)nd << 16);
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < LPW; o <<= 1) {
      const uint32_t tv = __shfl_up_sync(CGSVMC_FULL_MASK, inc, o, LPW);
      if (sub >= o) inc += tv;
    }
    const uint32_t exc = inc - cnt;
    const int ru = k_up - (int)(exc & 0xffffu), rd = k_dn - (int)(exc >> 16);
    const bool own_u = ru >= 0 && ru < nu, own_d = rd >= 0 && rd < nd;
    uint32_t res = 0;
    if (own_u) res = (uint32_t)(CB * sub + select_in_chunk<CB>(cu, ru, lut));
    if (own_d) res |= (uint32_t)(CB * sub + select_in_chunk<CB>(cd, rd, lut)) << 16;
#pragma unroll
    for (int o = LPW / 2; o > 0; o >>= 1) res |= __shfl_xor_sync(CGSVMC_FULL_MASK, res, o);
    up = (int)(res & 0xffffu);
    dn = (int)(res >> 16);
  }
};

// ---------------------------------------------------------------------------
// K2: Metropolis sampler, graph_builders.py:54-89 x n_steps
// ---------------------------------------------------------------------------
// CTA size.  The sampler kernel (mc_kernel) takes 1024 threads when the per-lane
// state fits a 64-register budget (at most 10 hidden units per lane): more
// walkers in flight per SM.  The walker kernel (estimators + sweep) always takes
// 512 threads = 128 registers: at 64 registers its small-H variants spilled
// 200-1000 B and ran 1.3-1.8x slower (6x6, H = 64, 8,192 walkers: 54.4 -> 29.8 us
// per batch iteration; H = 32: 36.1 -> 25.9 us; profiles/r02Y_rbm2_small_h.jsonl).
template <int LPW, int KJV, bool WALKER = false>
struct Geometry {
  static constexpr int VW = 32 / LPW, KJ = VW * KJV, HP = 32 * KJV, WPW = 32 / LPW;
  static constexpr int THREADS = (!WALKER && KJ <= 10) ? 1024 : 512;
  static constexpr int WARPS = THREADS / 32, SLOTS = WARPS * WPW;
};

// n_steps Metropolis exchange steps of one walker (graph_builders.py:54-89),
// run by its lane group.  On entry (p, m) is the normalised state of `s`; on
// exit `s` holds the new configuration and (p, m) an unnormalised state.
// Returns the number of accepted moves.
template <int NW, int LPW, int KJV, bool WS>
__device__ __forceinline__ unsigned int mc_sweep(const Tables& t, const Image& im,
                                                 const SitePicker<NW, LPW>& picker, const uint8_t* lut,
                                                 uint64_t (&s)[NW], float (&p)[32 / LPW * KJV],
                                                 float (&m)[32 / LPW * KJV], int sub, bool valid,
                                                 int n_steps, uint64_t seed, uint64_t walker,
                                                 uint64_t step0) {
  constexpr int KJ = 32 / LPW * KJV;
  float tq[KJ];
  // an accepted move scales p_j by at most 2^(8 log2(e) max|W|) = 2^wbits; the
  // window keeps the worst-case growth between renormalisations below 2^96
  // (p_j itself cannot overflow).  The four-term products of the ratio loop
  // could still leave the float32 range in that worst case -- every hidden
  // unit pushed the same way by every move -- which the non-finite check below
  // catches and repairs; typical growth is a bounded random walk far below it.
  const float wbits = 11.541560327111707f * ld1<WS>(t.a0 + 1);
  const int renorm_window = max(1, min(32, (int)((96.f - wbits) / (wbits + 1e-6f))));
  unsigned int n_acc = 0;
  int n_up = 0;
#pragma unroll
  for (int w = 0; w < NW; ++w) n_up += __popcll(s[w]);
  const int n_dn = im.N - n_up;
  const bool can_move = valid && n_up > 0 && n_dn > 0;
  // Between renormalisations the state is kept UNNORMALISED: an accepted
  // move only scales p_j by F[d][j] G[u][j] (m_j is untouched), and
  // lnorm = sum_j log2(p_j + m_j) -- which is exactly the log-sum of the move
  // just accepted -- is subtracted from the next proposals' sums.  One FMUL
  // per hidden unit per accepted move instead of {FMUL, FADD, RCP, 2 FMUL}.
  float lnorm = 0.f;
  int since_norm = 0;
  // lane `sub` draws the Philox block of step (LPW q + sub); the block of the
  // NEXT step is broadcast while the current ratio is in flight, so the
  // shuffles stay off the accept -> propose dependency chain
  Philox4 rnd = walker_step_random(seed, walker, step0 + (uint64_t)sub);
  uint32_t r0 = __shfl_sync(CGSVMC_FULL_MASK, rnd.x, 0, LPW);
  uint32_t r1 = __shfl_sync(CGSVMC_FULL_MASK, rnd.y, 0, LPW);
  uint32_t r2 = __shfl_sync(CGSVMC_FULL_MASK, rnd.z, 0, LPW);
  for (int step = 0; step < n_steps; ++step) {
    // uniformly random up site and uniformly random down site
    // (argmax / argmin of sigma * u, graph_builders.py:59-65)
    const int k_up = (int)__umulhi(r0, (uint32_t)n_up);
    const int k_dn = (int)__umulhi(r1, (uint32_t)n_dn);
    const float u_acc = u32_to_unit(r2);
    int up, dn;
    picker.pick(s, k_up, k_dn, lut, up, dn);
    if (!can_move) { up = 0; dn = 0; }
    const float lpart = exchange_log2_partial<LPW, KJV, WS, true>(t, dn, up, sub, p, m, tq);
    const float da2 = ld1<WS>(t.a2 + dn) - ld1<WS>(t.a2 + up);
    {
      const int nxt = step + 1;
      if ((nxt & (LPW - 1)) == 0) rnd = walker_step_random(seed, walker, step0 + (uint64_t)(nxt + sub));
      const int src = nxt & (LPW - 1);
      r0 = __shfl_sync(CGSVMC_FULL_MASK, rnd.x, src, LPW);
      r1 = __shfl_sync(CGSVMC_FULL_MASK, rnd.y, src, LPW);
      r2 = __shfl_sync(CGSVMC_FULL_MASK, rnd.z, src, LPW);
    }
    float lfull = group_sum<LPW>(lpart);
    // rare: a four-term product (or the unnormalised state) left the float32
    // range -- rebuild the normalised state from the spins and evaluate this
    // proposal term by term; warp-uniform
    if (__any_sync(CGSVMC_FULL_MASK, !(fabsf(lfull) <= 3.0e38f))) {
      init_state<NW, LPW, KJV, WS>(t, im, s, sub, p, m, false);
      lnorm = 0.f;
      since_norm = 0;
      lfull = group_sum<LPW>(exchange_log2_partial<LPW, KJV, WS, true, true>(t, dn, up, sub, p, m, tq));
    }
    const float l2 = (lfull - lnorm) + da2;
    // accept iff |psi'/psi| > sqrt(u)  <=>  (psi'/psi)^2 > u   (strict; NaN rejects)
    const float prob = ex2_approx(2.f * l2);
    if (can_move && prob > u_acc) {
#pragma unroll
      for (int k = 0; k < KJ; k += 2) mul2(p[k], p[k + 1], p[k], p[k + 1], tq[k], tq[k + 1]);
      lnorm = lfull;
      flip_bit<NW>(s, up);
      flip_bit<NW>(s, dn);
      ++n_acc;
    }
    // renormalise (p + m = 1, lnorm = 0) before the scale can overflow
    // (every `renorm_window` steps, from max |W|) or cost precision in
    // lfull - lnorm (|lnorm| large); warp-uniform
    if (++since_norm >= renorm_window || __any_sync(CGSVMC_FULL_MASK, fabsf(lnorm) > 48.f)) {
      since_norm = 0;
      lnorm = 0.f;
#pragma unroll
      for (int k = 0; k < KJ; k += 2) {
        float s0, s1;
        add2(s0, s1, p[k], p[k + 1], m[k], m[k + 1]);
        const float r0 = rcp_approx(s0), r1 = rcp_approx(s1);
        mul2(p[k], p[k + 1], p[k], p[k + 1], r0, r1);
        mul2(m[k], m[k + 1], m[k], m[k + 1], r0, r1);
      }
    }
  }
  return n_acc;
}

template <int NW, int LPW, int KJV, bool WS>
__global__ void __launch_bounds__((Geometry<LPW, KJV>::THREADS), 1)
mc_kernel(Image im, const float* __restrict__ img_g, uint64_t* __restrict__ packed, int64_t B,
          int wpc, int64_t n_batches, int n_steps, uint64_t seed, uint64_t walker0, uint64_t step0,
          const uint64_t* __restrict__ step0_dev, unsigned long long* accept_count,
          float* __restrict__ log_amp_out) {
  using Geo = Geometry<LPW, KJV>;
  RBM2_MARK(0, 0);
  if (step0_dev != nullptr) step0 += *step0_dev;
  constexpr int WPW = Geo::WPW, KJ = Geo::KJ;
  extern __shared__ __align__(16) float smem[];
  float* img_s = smem;
  uint8_t* lut = reinterpret_cast<uint8_t*>(smem + (WS ? im.off_lut : 0));
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + (WS ? im.total : 512));
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & (LPW - 1), grp = lane / LPW;
  // configurations of the first batch: requested before the table copy
  uint64_t s_first[NW];
  {
    const int64_t b = min((int64_t)blockIdx.x * wpc + min(warp * WPW + grp, wpc - 1), B - 1);
#pragma unroll
    for (int w = 0; w < NW; ++w) s_first[w] = w < im.words ? packed[b * im.words + w] : 0ull;
  }
  if (WS) bulk_load(img_s, img_g, (uint32_t)im.total * 4u, bar);
  else build_lut(lut);
  __syncthreads();
  RBM2_MARK(0, 1);
  const Tables t = tables_at(WS ? img_s : img_g, im);
  SitePicker<NW, LPW> picker;
  picker.setup(im.N, sub);
  unsigned int n_acc = 0;
  for (int64_t batch = blockIdx.x; batch < n_batches; batch += gridDim.x) {
    const int slot = warp * WPW + grp;
    const int64_t b = batch * wpc + slot;
    if (warp * WPW >= wpc || batch * wpc + warp * WPW >= B) continue;   // warp-uniform
    const bool valid = slot < wpc && b < B;
    const int64_t bb = valid ? b : B - 1;
    uint64_t s[NW];
    if (batch == blockIdx.x && valid) {
#pragma unroll
      for (int w = 0; w < NW; ++w) s[w] = s_first[w];
    } else {
#pragma unroll
      for (int w = 0; w < NW; ++w) s[w] = w < im.words ? packed[bb * im.words + w] : 0ull;
    }
    float p[KJ], m[KJ];
    init_state<NW, LPW, KJV, WS>(t, im, s, sub, p, m, false);
    RBM2_MARK(0, 2);
    n_acc += mc_sweep<NW, LPW, KJV, WS>(t, im, picker, lut, s, p, m, sub, valid, n_steps, seed,
                                        walker0 + (uint64_t)bb, step0);
    RBM2_MARK(0, 3);
    if (valid && sub == 0) {
#pragma unroll
      for (int w = 0; w < NW; ++w) if (w < im.words) packed[b * im.words + w] = s[w];
    }
    if (log_amp_out != nullptr) {
      float z = init_state<NW, LPW, KJV, WS>(t, im, s, sub, p, m, true);
      z = group_sum<LPW>(z) + ld1<WS>(t.a0);
      if (valid && sub == 0) log_amp_out[b] = z;
    }
  }
  if (accept_count != nullptr) {
    unsigned int mine = sub == 0 ? n_acc : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(CGSVMC_FULL_MASK, mine, o);
    if (lane == 0 && mine) atomicAdd(accept_count, (unsigned long long)mine);
  }
  RBM2_MARK(0, 4);
}

// ---------------------------------------------------------------------------
// K1 + K3 + K4 + K5 in one pass over the walkers ("walker kernel"):
//   amplitudes z, local energies (operators.py:227-259), weighted sums of
//   O_b = dz_b/dparams (training.py:545-558, 169-175) and energy statistics.
// do_eloc / do_grad select the phases; with both, the gradient weights are
// (1, E_loc) -- one session.run(accumulate_gradients).
// ---------------------------------------------------------------------------
// Drain of the tensor-core gradient accumulators (walker_kernel, A.tc_grad)
// into the CTA's slice of `partials`, through a shared-memory staging buffer
// [128 + 8 NC rows][17].  P0 / P1 / P2 at TMEM columns 0 / NCOL / 2 NCOL; rows
// [0, NPC): sigma (k = 0), [NPC, 2 NPC) / [2 NPC, 3 NPC): pieces 1 / 2 of the
// weights, P2 rows [0, NPC): piece 3.  The first drain of a launch stores, later
// ones add with fire-and-forget reductions (one writer per address: the order
// of the additions is the program order, the sums stay deterministic).
// Deliberately compact and out of line: it runs a few times per launch and
// would otherwise be paid in instruction fetches.
template <int THREADS, int NCOL>
__device__ __noinline__ void tcg_drain(uint32_t tmem, float* stg, int n_groups, float* part, int64_t P, int N, int H,
                                       int NC, bool add) {
  constexpr int LD = 20;                     // staging row stride (floats): 16-byte aligned rows
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int NPC = 8 * NC;
  const int grp_floats = (128 + NPC) * LD;   // one staging buffer: rows of P0 / P1 (128) + piece-3 rows (NPC)
  const int wq = warp & 3, g = warp >> 2;    // TMEM lane quarter of this warp, column-chunk group
  const int per = 2 * NPC * 4;               // (k, row, 4-column group) items of one chunk
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  __syncthreads();
  // n_groups chunks of 16 columns per round: warp (wq, g) reads lane quarter wq of chunk g
#pragma unroll 1
  for (int cbase = 0; cbase < NCOL; cbase += 16 * n_groups) {
    const int c0 = cbase + 16 * g;
    if (g < n_groups && c0 < NCOL) {
      float* sg = stg + (size_t)g * grp_floats;
      const int mrow = 32 * wq + lane;
      const uint32_t tbase = tmem + ((uint32_t)(32 * wq) << 16) + (uint32_t)c0;
      uint32_t q0[16], q1[16], q2[16];
#define RBM2_TMEM_LD16(ADDR, R)                                                                                  \
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];" \
                   : "=r"(R[0]), "=r"(R[1]), "=r"(R[2]), "=r"(R[3]), "=r"(R[4]), "=r"(R[5]), "=r"(R[6]), "=r"(R[7]), \
                     "=r"(R[8]), "=r"(R[9]), "=r"(R[10]), "=r"(R[11]), "=r"(R[12]), "=r"(R[13]), "=r"(R[14]), "=r"(R[15]) \
                   : "r"(ADDR) : "memory")
      RBM2_TMEM_LD16(tbase, q0);
      RBM2_TMEM_LD16(tbase + (uint32_t)NCOL, q1);
      if (wq < 2) RBM2_TMEM_LD16(tbase + (uint32_t)(2 * NCOL), q2);      // piece 3: rows [0, NPC) only
#undef RBM2_TMEM_LD16
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int c = 0; c < 16; c += 4) {
        float4 v;
        v.x = fmaf(__uint_as_float(q1[c]), 1.f / 2048.f, __uint_as_float(q0[c]));
        v.y = fmaf(__uint_as_float(q1[c + 1]), 1.f / 2048.f, __uint_as_float(q0[c + 1]));
        v.z = fmaf(__uint_as_float(q1[c + 2]), 1.f / 2048.f, __uint_as_float(q0[c + 2]));
        v.w = fmaf(__uint_as_float(q1[c + 3]), 1.f / 2048.f, __uint_as_float(q0[c + 3]));
        *reinterpret_cast<float4*>(sg + mrow * LD + c) = v;
        if (wq < 2 && mrow < NPC)
          *reinterpret_cast<float4*>(sg + (128 + mrow) * LD + c) =
              make_float4(__uint_as_float(q2[c]), __uint_as_float(q2[c + 1]), __uint_as_float(q2[c + 2]),
                          __uint_as_float(q2[c + 3]));
      }
    }
    __syncthreads();
    // one (chunk group, weight column k, row i, 4 columns) item per thread
#pragma unroll 1
    for (int e = threadIdx.x; e < n_groups * per; e += THREADS) {
      const int gg = e / per, e1 = e - gg * per;
      const int cc0 = cbase + 16 * gg;
      if (cc0 >= NCOL) continue;
      const float* sg = stg + (size_t)gg * grp_floats;
      const int k = e1 >= NPC * 4 ? 1 : 0, r = e1 - k * NPC * 4;
      const int i = r >> 2, c = (r & 3) * 4;
      if (i > N) continue;
      const float4 s0 = *reinterpret_cast<const float4*>(sg + i * LD + c);
      float v[4] = {s0.x, s0.y, s0.z, s0.w};
      if (k == 1) {
        const float4 p1 = *reinterpret_cast<const float4*>(sg + (NPC + i) * LD + c);
        const float4 p2 = *reinterpret_cast<const float4*>(sg + (2 * NPC + i) * LD + c);
        const float4 p3 = *reinterpret_cast<const float4*>(sg + (128 + i) * LD + c);
        const float a1[4] = {p1.x, p1.y, p1.z, p1.w}, a2[4] = {p2.x, p2.y, p2.z, p2.w},
                    a3[4] = {p3.x, p3.y, p3.z, p3.w};
#pragma unroll
        for (int u = 0; u < 4; ++u)
          v[u] = fmaf(fmaf(a3[u], 1.f / 2048.f, a2[u]), 1.f / 2048.f, a1[u]) * (1.f / kTcgPrescale);
      }
      float* row_w = part + (size_t)k * P + (size_t)(N + 1) + (size_t)i * H;    // W[i][.] (i < N), c[.] (i == N)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = cc0 + c + u;
        if (j > H) continue;
        float* dst = j < H ? row_w + j : part + (size_t)k * P + i;              // column H: a_i (i < N), a0 (i == N)
        if (add) atomicAdd(dst, v[u]);
        else *dst = v[u];
      }
    }
    __syncthreads();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

struct WalkerArgs {
  const uint64_t* packed;
  int64_t B;
  int wpc;
  int64_t n_batches;
  // local energy
  int do_eloc;
  const int2* bonds_ij; const float* bonds_jx; const float* bonds_jz; int n_bonds;
  float* e_loc; float* log_amp; float* diag; float* off;
  // gradient
  int do_grad;
  const float* weights;   // [K][B] or NULL (then weights = (1, E_loc))
  int K;
  float* partials;        // [grid][2][P]
  double* stat_partials;  // [grid][2] or NULL
  int64_t P;
  // fused Metropolis sweep after the estimators (MC kernels only): one batch
  // iteration of run_optimization_epoch (training.py:614-617) in one launch
  uint64_t* packed_rw;
  int n_steps;
  // n_iters > 1: that many consecutive batch iterations in ONE launch (the loop
  // of training.py:614-617 moved into the kernel): tables and bonds are loaded
  // once, a CTA keeps adding to its slice of `partials`, the cross-CTA
  // reduction runs once at the end.  Iteration i uses Philox steps
  // step0 + i n_steps ..., exactly like i separate launches; e_loc / log_amp
  // rows of iteration i start at i * out_stride.
  int n_iters;
  int64_t out_stride;
  uint64_t seed, walker0, step0;
  const uint64_t* step0_dev;
  unsigned long long* accept_count;
  // bond-pair table (PT kernels): [2 n_bonds][HP], row 2 k + o = F[d] * G[u]
  // for bond k with d = (o ? j_k : i_k) raised and the other end lowered
  const float* pair_table;
  // PT kernels: gradient sums on the tensor cores (tcgen05, accumulators in
  // TMEM for the whole launch) instead of the FP32 register tiles; planned by
  // the host when the shapes fit (N <= 39, H <= 159: the C2 class)
  int tc_grad;
  // walkers given as the reference's float32 [B][N] of +-1 instead of packed
  // words (the packed configurations are still written to packed_rw)
  const float* configs_f32;
  // cross-CTA reduction inside this kernel (cooperative launch: every CTA is
  // resident, so a CTA may wait for the others): out[f] += sum_cta partials,
  // stats += the energy sums, *counter += advance, stats copied to
  // stats_snapshot (may be mapped host memory)
  int fuse_reduce;
  unsigned int* sync;       // [2] arrive / depart counters, zero between launches
  float* out;
  int64_t n_out;
  double* stats;
  uint64_t* counter;
  uint64_t advance;
  double* stats_snapshot;
};

// Configuration of walker bb as packed words: from the packed array or, when
// the caller feeds float32 [B][N] of +-1 (graph_builders.py:92-125 layout),
// bit-packed here by the walker's lane group (LPW sites per ballot; LPW divides
// 64, so a ballot never straddles a word).  Warp-collective.
template <int NW, int LPW>
__device__ __forceinline__ void load_walker(const WalkerArgs& A, const Image& im, int64_t bb, int sub,
                                            int grp, uint64_t (&s)[NW]) {
  if (A.configs_f32 == nullptr) {
#pragma unroll
    for (int w = 0; w < NW; ++w) s[w] = w < im.words ? A.packed[bb * im.words + w] : 0ull;
    return;
  }
#pragma unroll
  for (int w = 0; w < NW; ++w) s[w] = 0ull;
  const float* row = A.configs_f32 + bb * im.N;
  for (int i0 = 0; i0 < im.N; i0 += LPW) {
    const int i = i0 + sub;
    const bool up = i < im.N && row[i] > 0.f;
    const uint32_t vote = __ballot_sync(CGSVMC_FULL_MASK, up);
    const uint64_t gbits = (uint64_t)((vote >> (grp * LPW)) & ((1u << LPW) - 1u));
#pragma unroll
    for (int w = 0; w < NW; ++w)
      if ((i0 >> 6) == w) s[w] |= gbits << (i0 & 63);
  }
}

// Cross-CTA reduction at the end of the walker kernel (replaces a separate
// reduction launch: ~7.5 us of kernel + launch gap per C2 step).  Requires a
// cooperative launch.  Every CTA publishes its partial sums, waits until all
// CTAs of the grid have done so, and reduces its share of the output columns
// over the CTA slices in a fixed order (deterministic): 32 columns x RG row
// groups per pass, all of a thread's loads in flight before its first add.
// CTA 0 also folds the energy statistics, advances the device-side Philox
// step counter of a captured step and publishes the statistics snapshot.
template <int THREADS>
__device__ __forceinline__ void grid_reduce(const WalkerArgs& A, float* red) {
  constexpr int RG = THREADS / 32;     // row groups (warps)
  constexpr int RU = 10;               // partial rows per thread and pass: RG * RU >= 148 CTAs in one pass
  constexpr int CU = 3;                // column chunks of 32 per pass
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_cta = (int)gridDim.x;
  __syncthreads();                     // this CTA's partial stores are issued
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(&A.sync[0], 1u);
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(A.sync) : "memory");
    } while (seen < (unsigned int)n_cta);
  }
  __syncthreads();
  const int64_t stride = 2 * A.P;
  const int64_t per = (A.n_out + n_cta - 1) / n_cta;
  const int64_t c0 = (int64_t)blockIdx.x * per, c1 = min(A.n_out, c0 + per);
  for (int64_t cbase = c0; cbase < c1; cbase += 32 * CU) {
    float acc[CU];
#pragma unroll
    for (int u = 0; u < CU; ++u) acc[u] = 0.f;
    for (int r0 = warp; r0 < n_cta; r0 += RG * RU) {
      float v[CU][RU];
#pragma unroll
      for (int u = 0; u < CU; ++u) {
        const int64_t col = cbase + 32 * u + lane;
#pragma unroll
        for (int k = 0; k < RU; ++k) {
          const int r = r0 + RG * k;
          v[u][k] = (col < c1 && r < n_cta) ? __ldcg(A.partials + (size_t)r * stride + col) : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < CU; ++u)
#pragma unroll
        for (int k = 0; k < RU; ++k) acc[u] += v[u][k];
    }
#pragma unroll
    for (int u = 0; u < CU; ++u) red[warp * (32 * CU) + 32 * u + lane] = acc[u];
    __syncthreads();
    if (threadIdx.x < 32 * CU) {
      const int64_t col = cbase + threadIdx.x;
      if (col < c1) {
        float total = 0.f;
#pragma unroll
        for (int w = 0; w < RG; ++w) total += red[w * (32 * CU) + threadIdx.x];
        A.out[col] += total;
      }
    }
    __syncthreads();
  }
  if (blockIdx.x == 0 && warp == 0 && A.stats != nullptr) {
    double e = 0.0, e2 = 0.0;
    if (A.stat_partials != nullptr)
      for (int c = lane; c < n_cta; c += 32) { e += __ldcg(A.stat_partials + 2 * c); e2 += __ldcg(A.stat_partials + 2 * c + 1); }
    e = warp_sum(e);
    e2 = warp_sum(e2);
    if (lane == 0) {
      const double s0 = A.stats[0] + e, s1 = A.stats[1] + e2,
                   s2 = A.stats[2] + (double)A.B * (double)(A.n_iters > 1 ? A.n_iters : 1);
      A.stats[0] = s0; A.stats[1] = s1; A.stats[2] = s2;
      if (A.stats_snapshot != nullptr) {
        volatile double* snap = A.stats_snapshot;
        snap[0] = s0; snap[1] = s1; snap[2] = s2; snap[3] = A.stats[3];
        __threadfence_system();
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 32 && A.counter != nullptr) *A.counter += A.advance;
  // depart: the last CTA to leave re-arms the counters for the next launch
  // (every CTA has left the wait loop before it departs)
  if (threadIdx.x == 0) {
    const unsigned int gone = atomicAdd(&A.sync[1], 1u);
    if (gone == (unsigned int)n_cta - 1u) {
      A.sync[0] = 0u;
      A.sync[1] = 0u;
      __threadfence();
    }
  }
}

// MC: after the estimators of a walker are done (and its gradient inputs are
// staged in shared memory) its lane group continues with n_steps Metropolis
// steps from the state (p, m) it already holds, and writes the configuration
// back; the CTA-wide gradient tiles follow.  Saves a launch, a second table
// load and a second state build per batch iteration.
// PT (needs WS): the local energy reads ONE row of the bond-pair table per
// amplitude ratio instead of two site rows (the binding resource of this
// kernel is shared-memory bandwidth); to make room the shared-memory image
// starts at the F table and the 2W rows of the state build are parked in the
// buffer that later stages tanh(theta) for the gradient tiles (a CTA barrier
// separates the two uses).  With the gradient on the tensor cores the rows are
// copied back during every pass's sweep, once the MMAs have read the staged
// operands; otherwise later batches of the same CTA read 2W from global memory.
template <int NW, int LPW, int KJV, bool WS, bool MC, bool PT = false>
__global__ void __launch_bounds__((Geometry<LPW, KJV, true>::THREADS), 1)
walker_kernel(Image im, const float* __restrict__ img_g, WalkerArgs A) {
  using Geo = Geometry<LPW, KJV, true>;
  constexpr int WPW = Geo::WPW, KJ = Geo::KJ, VW = Geo::VW, HP = Geo::HP;
  constexpr int SLOTS = Geo::SLOTS, THREADS = Geo::THREADS;
  static_assert(!PT || WS, "the pair-table kernel keeps its tables in shared memory");
  extern __shared__ __align__(16) float smem[];
  // ---- shared-memory carve-up (mirrors walker_smem_bytes) ----
  const int img_skip = PT ? im.off_f : 0;          // floats of the image left in global memory
  float* img_s = smem - img_skip;                  // so that img_s + off_x addresses table x
  char* cur = reinterpret_cast<char*>(smem + (WS ? im.total - img_skip : 0));
  uint64_t* bar = reinterpret_cast<uint64_t*>(cur); cur += 32;   // table mbarrier, tile counter, TMEM address, MMA mbarrier, 2W mbarrier
  int4* bond_s = reinterpret_cast<int4*>(cur); cur += (size_t)(A.do_eloc ? A.n_bonds : 0) * 16;
  const int list_ld = (A.n_bonds + 7) / 8 * 8;
  uint32_t* list_s = reinterpret_cast<uint32_t*>(cur); cur += (size_t)(A.do_eloc ? SLOTS * list_ld : 0) * 4;
  const int NP4 = (im.N + 1 + 3) / 4 * 4;
  // (PT: at least N rows, the 2W table lives here during the state build)
  float* T_s = reinterpret_cast<float*>(cur);
  cur += (size_t)max(A.do_grad ? SLOTS * HP : 0, PT ? im.N * HP : 0) * 4;
  float* ws_s = reinterpret_cast<float*>(cur); cur += (size_t)(A.do_grad ? SLOTS * 2 * NP4 : 0) * 4;
  float* e_s = reinterpret_cast<float*>(cur); cur += (size_t)SLOTS * 4;
  // select table: inside the image when it is in shared memory, else 2048 bytes here (MC only)
  uint8_t* lut = WS ? reinterpret_cast<uint8_t*>(img_s + im.off_lut) : reinterpret_cast<uint8_t*>(cur);
  // [2 n_bonds][HP]: in shared memory (PT), or -- tables too large for shared
  // memory (16x16, H = 256) -- read through L1 / L2 like the site tables: still
  // one row per amplitude ratio instead of two and no multiply per hidden unit
  const float* pair_s = PT ? reinterpret_cast<const float*>(cur) : (!WS ? A.pair_table : nullptr);
  int* tile_next_s = reinterpret_cast<int*>(bar) + 2;                // behind the 8-byte mbarrier
  uint64_t* mma_bar = bar + 2;
  uint64_t* w2_bar = bar + 3;                                        // 2W rows parked in T_s again (tcg)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bar) + 3;
  // ---- gradient sums on the tensor cores (PT kernels, A.tc_grad) ----
  // S_k[i][j] = sum_b (w_kb sigma_bi) tanh(theta_bj) is a GEMM over the walkers
  // of the CTA: A[m][b] (MN-major, K = walker slot) x B[b][j] (MN-major).
  //   B planes (in T_s): tanh theta as two fp16 planes t = t1 + t2 / S, [split][8-column chunk][slot][8];
  //       column H is the constant 1 (the a / a0 gradients ride along).
  //   A planes (in ws_s), fp16:
  //       chunks [0, NC): sigma_i (+-1; row N: 1 = the c / a0 gradients), w_0 = 1;
  //       chunks [NC, 4 NC): the three fp16 pieces of x = w_1 sigma_i 2^-20 (w_1 = E_loc;
  //       x = x1 + x2 / S + x3 / S^2; the prescale covers |E_loc| < 6.8e10).
  //   P0 += A[chunks 0 ..] x t1, P1 += A[chunks 0 ..] x t2 (M = 128: sigma and the pieces 1, 2),
  //   P2 += A[chunks 3 NC ..] x t1 (piece 3);   S_0 = P0 + P1 / S on the sigma rows,
  //   S_1 = 2^20 (rows of piece 1 + rows of piece 2 / S + rows of piece 3 / S^2).
  //   12 MMAs per batch iteration; the accumulators
  //   stay in TMEM for the whole launch (all iterations of an epoch) and are
  //   drained once.
  constexpr int NCOL = HP;                       // B columns: H real ones + the constant 1 (needs H < HP)
  constexpr int NB = NCOL / 8;                   // B chunks per split
  // (planned only for N <= 39: one spin word, so the wider kernels carry no tensor-core code)
  const bool tcg = PT && NW == 1 && A.do_grad && A.tc_grad;
  const int NC = (im.N + 1 + 7) / 8;             // A chunks per group
  uint32_t tmem = 0;
  // The tensor cores accumulate in fp32 with truncation: over the 200 MMA steps
  // of a 50-iteration launch the coherent sum E sum_b O_b drifted by 1.3e-5 of
  // its value.  The accumulators are therefore drained every kTcgSegment
  // passes (1.7e-6 against the FP32 register tiles after 50 iterations,
  // profiles/r02u_precision.txt).
  constexpr int kTcgSegment = 8;
  // drain: T_s and ws_s (contiguous, free between two passes) stage up to four
  // 16-column chunks at a time, one per group of four warps
  const int drain_groups = max(1, min(min(THREADS / 128, 4),
                                      (SLOTS * HP + SLOTS * 2 * NP4) / ((128 + 8 * NC) * 20)));

  RBM2_MARK(1, 0);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & (LPW - 1), grp = lane / LPW;
  const int slot = warp * WPW + grp;
  // configurations of the first batch: requested before the table copy so that
  // the global-memory latency overlaps it (grid <= n_batches, so b0 < B)
  uint64_t s_first[NW];
  {
    const int64_t b0 = (int64_t)blockIdx.x * A.wpc;
    const int n_valid = (int)min((int64_t)A.wpc, A.B - b0);
    const int64_t bb = b0 + min(slot, n_valid - 1);
    load_walker<NW, LPW>(A, im, bb, sub, grp, s_first);
  }
  if (PT) bulk_load(smem, img_g + img_skip, (uint32_t)(im.total - img_skip) * 4u, bar,
                    const_cast<float*>(pair_s), A.pair_table, (uint32_t)(2 * A.n_bonds * HP) * 4u,
                    T_s, img_g + im.off_w2, (uint32_t)(im.N * HP) * 4u);
  else if (WS) bulk_load(img_s, img_g, (uint32_t)im.total * 4u, bar);
  else if (MC) build_lut(lut);
  if (A.do_eloc) {
    for (int k = threadIdx.x; k < A.n_bonds; k += THREADS) {
      const int2 ij = A.bonds_ij[k];
      bond_s[k] = make_int4(ij.x, ij.y, __float_as_int(A.bonds_jx[k]), __float_as_int(A.bonds_jz[k]));
    }
  }
  if (tcg) {
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mma_bar)) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(w2_bar)) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)),
                   "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // A planes: slots without a walker must read as zero
    for (int e = threadIdx.x; e < SLOTS * 2 * NP4 / 4; e += THREADS)
      reinterpret_cast<uint4*>(ws_s)[e] = make_uint4(0u, 0u, 0u, 0u);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (tcg) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    tmem = *tmem_holder;
  }
  RBM2_MARK(1, 1);
  // t.w2: the 2W rows outside the state build at the top of a pass (the
  // sampler's rare state rebuild); with the gradient T_s holds staged operands then
  Tables t = tables_at(WS ? img_s : img_g, im);
  if (PT) t.w2 = A.do_grad ? img_g + im.off_w2 : T_s;
  SitePicker<NW, LPW> picker;
  if (MC) picker.setup(im.N, sub);
  unsigned int n_acc = 0;
  const uint64_t mc_step0 = MC ? A.step0 + (A.step0_dev != nullptr ? *A.step0_dev : 0ull) : 0ull;

  // gradient tiles: 4 rows (sites, row N = the "ones" row of c) x 4 hidden units
  constexpr int CT = HP / 4;
  const int RT = NP4 / 4;
  const int n_tiles = RT * CT;
  // The a-gradient (entries rev (+ THREADS) of [2][NP4]) and the energy
  // statistics are taken from the END of the CTA: with fewer tiles than
  // threads those warps have no tile work.
  const int rev = THREADS - 1 - (int)threadIdx.x;
  float acc_a[2] = {0.f, 0.f};
  double sum_e = 0.0, sum_e2 = 0.0;   // lane 0 of the last warp only
  float* part = A.partials + (size_t)blockIdx.x * 2 * A.P;
  // pass = one walker batch of one iteration; with one batch per CTA the swept
  // walker of an iteration stays in registers for the next one, otherwise it is
  // read back from packed_rw
  const int n_iters = MC ? max(A.n_iters, 1) : 1;
  const bool keep_s = A.n_batches <= (int64_t)gridDim.x;
  int batch_no = 0;
  uint64_t s[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) s[w] = 0ull;

  int n_drained = 0;
  for (int iter = 0; iter < n_iters; ++iter)
  for (int64_t batch = blockIdx.x; batch < A.n_batches; batch += gridDim.x, ++batch_no) {
    const int64_t b0 = batch * A.wpc;
    const int n_valid = (int)min((int64_t)A.wpc, A.B - b0);
    const bool warp_on = warp * WPW < n_valid;
    const bool valid = slot < n_valid;
    const int64_t b = b0 + slot;
    const int64_t bb = valid ? b : b0 + n_valid - 1;
    const int64_t ob = (int64_t)iter * A.out_stride + b;      // row of this pass in e_loc / log_amp / diag / off
    RBM2_MARK(1, 10);
    float p[KJ], m[KJ];
    // PT: the state build reads the 2W rows parked in T_s -- without the
    // gradient T_s holds nothing else, the first pass finds them there from the
    // table copy, and with the gradient on the tensor cores the previous pass
    // has copied them back (w2_bar)
    const bool w2_parked = PT && (!A.do_grad || batch_no == 0 || tcg);
    if (warp_on) {
      if (batch_no == 0) {
#pragma unroll
        for (int w = 0; w < NW; ++w) s[w] = s_first[w];
      } else if (iter == 0) {
        load_walker<NW, LPW>(A, im, bb, sub, grp, s);
      } else if (!keep_s) {
        // written by this lane group in the previous iteration (behind a CTA barrier)
#pragma unroll
        for (int w = 0; w < NW; ++w) s[w] = w < im.words ? __ldcg(A.packed_rw + bb * im.words + w) : 0ull;
      }
      const bool want_z = A.log_amp != nullptr;
      if (tcg && batch_no > 0) mbar_wait(smem_u32(w2_bar), (uint32_t)(batch_no - 1) & 1u);
      Tables tb = t;
      if (w2_parked) tb.w2 = T_s;
      float z = init_state<NW, LPW, KJV, WS>(tb, im, s, sub, p, m, want_z);
      if (want_z) {
        z = group_sum<LPW>(z) + ld1<WS>(t.a0);
        if (valid && sub == 0) A.log_amp[ob] = z;
      }
      RBM2_MARK(1, 2);
    }
    // every warp is done with the parked 2W rows before T_s is written for the gradient
    if (A.do_grad && w2_parked) __syncthreads();
    // the MMAs of the previous pass have read the operand planes; a full
    // segment of kTcgSegment passes is drained before the next one starts
    // (bounds the truncating accumulation in TMEM)
    const bool seg_start = tcg && (batch_no % kTcgSegment) == 0;
    if (tcg && batch_no > 0) {
      mbar_wait(smem_u32(mma_bar), (uint32_t)(batch_no - 1) & 1u);
      if (seg_start) {
        tcg_drain<THREADS, NCOL>(tmem, T_s, drain_groups, part, A.P, im.N, im.H, NC, n_drained > 0);
        ++n_drained;
        // the staging went through the operand planes: rows of empty slots must read as zero again
        for (int e = threadIdx.x; e < SLOTS * 2 * NP4 / 4; e += THREADS)
          reinterpret_cast<uint4*>(ws_s)[e] = make_uint4(0u, 0u, 0u, 0u);
        __syncthreads();
      }
    }
    if (tcg) {
      // B planes: rows of slots without a walker must read as zero (finite); the
      // 2W rows or the drain staging were there
      const int n_empty = SLOTS - n_valid;
      for (int e = threadIdx.x; e < n_empty * 2 * NB; e += THREADS) {
        const int ch = e / n_empty, sl = n_valid + e % n_empty;
        *reinterpret_cast<uint4*>(reinterpret_cast<char*>(T_s) + ((size_t)ch * SLOTS + sl) * 16) =
            make_uint4(0u, 0u, 0u, 0u);
      }
    }
    float e_val = 0.f;
    if (warp_on) {
      if (A.do_eloc) {
        // ---- enumerate antiparallel bonds (operators.py:154-167) ----
        // list entry = site to raise | site to lower << 8 | bond index << 16
        uint32_t* list = list_s + slot * list_ld;
        float diag = 0.f;
        int cnt = 0;
        for (int k0 = 0; k0 < A.n_bonds; k0 += LPW) {
          const int k = k0 + sub;
          bool anti = false;
          uint32_t ent = 0;
          if (k < A.n_bonds) {
            const int4 bd = bond_s[k];
            const int bi = spin_bit<NW>(s, bd.x);
            anti = bi != spin_bit<NW>(s, bd.y);
            diag = __fmaf_rn(anti ? -0.25f : 0.25f, __int_as_float(bd.w), diag);   // operators.py:165,169
            const int up = bi ? bd.x : bd.y, dn = bi ? bd.y : bd.x;
            // bit 31: the raised site is the bond's second end (pair-table row 2 k + 1)
            ent = (uint32_t)dn | ((uint32_t)up << 8) | ((uint32_t)k << 16) | (bi ? 0x80000000u : 0u);
          }
          const uint32_t vote = __ballot_sync(CGSVMC_FULL_MASK, anti);
          const uint32_t gbits = (vote >> (grp * LPW)) & ((1u << LPW) - 1u);
          if (anti) list[cnt + __popc(gbits & ((1u << sub) - 1u))] = ent;
          cnt += __popc(gbits);
        }
        diag = group_sum<LPW>(diag);
        __syncwarp();
        int n_max = cnt;
#pragma unroll
        for (int o = LPW; o < 32; o <<= 1) n_max = max(n_max, __shfl_xor_sync(CGSVMC_FULL_MASK, n_max, o));
        // ---- off-diagonal terms: jx/2 psi(flip)/psi on active bonds only ----
        // LPW bonds per round: the lanes' partial sums of the LPW log-ratios are
        // transpose-reduced so that lane `sub` ends up with the total of bond
        // it0 + sub and finishes it (a2 terms, ex2, coupling) alone; the LPW
        // ratio evaluations of a round are independent instruction streams.
        // Rounds are branch-free (list slots past cnt evaluate the dummy move
        // 0 -> 0) so that the compiler interleaves the evaluations; a remainder
        // of at most LPW / 2 bonds takes a half round.
        // (tables in global memory: rounds of LPW / 4 keep the rows in flight
        // within L1 -- measured at 16x16, H = 256: 6.6 ms / 5.0 / 4.9 for LPW, / 2, / 4)
        constexpr int RND = WS ? LPW : LPW / 4;
        float off_lane = 0.f;
        int it0 = 0;
        for (; n_max - it0 > RND / 2; it0 += RND)
          off_lane = __fadd_rn(off_lane, ratio_round<RND, LPW, KJV, WS>(t, list, bond_s, it0, cnt, sub, p, m, pair_s));
        if (it0 < n_max)
          off_lane = __fadd_rn(off_lane, ratio_round<RND / 2, LPW, KJV, WS>(t, list, bond_s, it0, cnt, sub, p, m, pair_s));
        const float off = group_sum<LPW>(off_lane);
        e_val = __fadd_rn(diag, off);
        RBM2_MARK(1, 3);
        if (valid && sub == 0) {
          if (A.e_loc) A.e_loc[ob] = e_val;
          if (A.diag) A.diag[ob] = diag;
          if (A.off) A.off[ob] = off;
        }
      }
      if (A.do_grad && valid) {
        // stage tanh(theta) = p - m, the signed weights w_k sigma_i and E_loc
        float w0, w1;
        if (A.weights != nullptr) {
          w0 = A.weights[b];
          w1 = A.K > 1 ? A.weights[A.B + b] : 0.f;
        } else {
          w0 = 1.f; w1 = e_val;
        }
        if (tcg) {
          // B planes: this lane's hidden units j = VW (sub + LPW q) + c -> chunk j / 8, halves (j % 8) ..
          char* bp = reinterpret_cast<char*>(T_s);
#pragma unroll
          for (int q = 0; q < KJV; ++q) {
            const int j0 = VW * sub + 32 * q;
            uint32_t h1[VW / 2], h2[VW / 2];
#pragma unroll
            for (int c = 0; c < VW; c += 2) {
              float v0 = p[VW * q + c] - m[VW * q + c], v1 = p[VW * q + c + 1] - m[VW * q + c + 1];
              if (j0 + c == im.H) v0 = 1.f;          // column H: the constant 1 (a / a0 gradients)
              if (j0 + c + 1 == im.H) v1 = 1.f;
              const __half2 a1 = __floats2half2_rn(v0, v1);
              const float2 f1 = __half22float2(a1);
              const __half2 a2 = __floats2half2_rn((v0 - f1.x) * 2048.f, (v1 - f1.y) * 2048.f);
              h1[c / 2] = *reinterpret_cast<const uint32_t*>(&a1);
              h2[c / 2] = *reinterpret_cast<const uint32_t*>(&a2);
            }
            char* dst = bp + ((size_t)(j0 >> 3) * SLOTS + slot) * 16 + (j0 & 7) * 2;
            if (VW == 4) {
              *reinterpret_cast<uint2*>(dst) = make_uint2(h1[0], h1[(VW / 2) - 1]);
              *reinterpret_cast<uint2*>(dst + (size_t)NB * SLOTS * 16) = make_uint2(h2[0], h2[(VW / 2) - 1]);
            } else {
              *reinterpret_cast<uint32_t*>(dst) = h1[0];
              *reinterpret_cast<uint32_t*>(dst + (size_t)NB * SLOTS * 16) = h2[0];
            }
          }
          // A planes: sigma, then the three fp16 pieces of w1 sigma 2^-20 (w0 = 1 on this path):
          // x = x1 + x2 / S + x3 / S^2, 33 mantissa bits; the prescale keeps |E_loc| < 6.8e10
          // inside the fp16 range, small values stay exact through the scaled residuals
          float rem = w1 * kTcgPrescale;
          uint32_t piece[3];
#pragma unroll
          for (int g = 0; g < 3; ++g) {
            const __half b = __float2half_rn(rem);
            piece[g] = (uint32_t)__half_as_ushort(b);
            rem = (rem - __half2float(b)) * 2048.f;
          }
          char* ap = reinterpret_cast<char*>(ws_s);
          for (int ch = sub; ch < 4 * NC; ch += LPW) {
            const int g = ch / NC, c = ch - g * NC;
            const uint32_t mag = g == 0 ? 0x3c00u : g == 1 ? piece[0] : g == 2 ? piece[1] : piece[2];
            uint32_t wds[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int i = 8 * c + e;
              uint32_t hb = 0u;
              if (i < im.N) hb = spin_bit<NW>(s, i) ? mag : (mag ^ 0x8000u);
              else if (i == im.N) hb = mag;
              wds[e >> 1] |= hb << (16 * (e & 1));
            }
            *reinterpret_cast<uint4*>(ap + ((size_t)ch * SLOTS + slot) * 16) = make_uint4(wds[0], wds[1], wds[2], wds[3]);
          }
        } else {
        float* Trow = T_s + slot * HP + VW * sub;
#pragma unroll
        for (int q = 0; q < KJV; ++q) {
          float v[VW];
#pragma unroll
          for (int c = 0; c < VW; ++c) v[c] = p[VW * q + c] - m[VW * q + c];
          stv<VW>(Trow + 32 * q, v);
        }
        float* wrow = ws_s + (size_t)slot * 2 * NP4;
        for (int i = sub; i < NP4; i += LPW) {
          float sg = 0.f;
          if (i < im.N) sg = spin_bit<NW>(s, i) ? 1.f : -1.f;
          else if (i == im.N) sg = 1.f;
          wrow[i] = w0 * sg;
          wrow[NP4 + i] = w1 * sg;
        }
        }
        if (sub == 0) e_s[slot] = e_val;
      }
      RBM2_MARK(1, 4);
    }
    // The gradient tiles need every walker's staged rows but not the sweep:
    // after this barrier the warps that own walkers run their Metropolis steps
    // while the warps without walkers (wpc < SLOTS) already work through the
    // tiles, 32 at a time from a shared counter; the sweeping warps join when
    // they are done.  (FMA-pipe tile work under the sampler's issue gaps.)
    if (A.do_grad) {
      if (threadIdx.x == 0) *tile_next_s = 0;
      if (tcg) {
        // slots beyond this batch's walkers: zero A rows (a shorter last batch of a launch)
        for (int e = threadIdx.x; e < (SLOTS - n_valid) * 4 * NC; e += THREADS) {
          const int ch = e / (SLOTS - n_valid), sl = n_valid + e % (SLOTS - n_valid);
          *reinterpret_cast<uint4*>(reinterpret_cast<char*>(ws_s) + ((size_t)ch * SLOTS + sl) * 16) =
              make_uint4(0u, 0u, 0u, 0u);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      }
      __syncthreads();
      if (tcg && warp == THREADS / 32 - 1) {
        // the last warp (no walkers when wpc < SLOTS) issues the 3 x SLOTS / 16 MMAs of this pass
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_units = smem_u32(ws_s) >> 4, b_units = smem_u32(T_s) >> 4;
        const uint32_t hi = (uint32_t)SLOTS | (1u << 14);               // MN-major: SBO = chunk stride, LBO = 8 rows
        // D = F32, A = B = F16, both MN-major, N = NCOL, M = 128
        const uint32_t idesc = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(NCOL >> 3) << 17) | (8u << 24);
        uint32_t elected = 0;
        asm volatile("{ .reg .pred p; elect.sync _|p, 0xffffffff; selp.u32 %0, 1, 0, p; }" : "=r"(elected));
        if (elected) {
          for (int ks = 0; ks < SLOTS / 16; ++ks) {
            const uint32_t accf = ((batch_no % kTcgSegment) > 0 || ks > 0) ? 1u : 0u;
            const uint64_t a0d = ((uint64_t)hi << 32) | ((a_units + (uint32_t)(16 * ks)) | (8u << 16));
            const uint64_t a3d = ((uint64_t)hi << 32) | ((a_units + (uint32_t)(3 * NC * SLOTS + 16 * ks)) | (8u << 16));
            const uint64_t b1d = ((uint64_t)hi << 32) | ((b_units + (uint32_t)(16 * ks)) | (8u << 16));
            const uint64_t b2d = ((uint64_t)hi << 32) | ((b_units + (uint32_t)(NB * SLOTS + 16 * ks)) | (8u << 16));
            const uint64_t ad[3] = {a0d, a0d, a3d}, bd[3] = {b1d, b2d, b1d};
#pragma unroll
            for (int u = 0; u < 3; ++u)
              asm volatile(
                  "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                  "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
                  :
                  : "r"(tmem + (uint32_t)(u * NCOL)), "l"(ad[u]), "l"(bd[u]), "r"(idesc), "r"(accf), "r"(0u)
                  : "memory");
          }
          asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                           smem_u32(mma_bar))
                       : "memory");
        }
        __syncwarp();
      }
    }
    if (MC && warp_on) {
      n_acc += mc_sweep<NW, LPW, KJV, WS>(t, im, picker, lut, s, p, m, sub, valid, A.n_steps, A.seed,
                                          A.walker0 + (uint64_t)bb, mc_step0 + (uint64_t)iter * (uint64_t)A.n_steps);
      if (valid && sub == 0) {
#pragma unroll
        for (int w = 0; w < NW; ++w) if (w < im.words) A.packed_rw[b * im.words + w] = s[w];
      }
      __syncwarp();        // a later iteration of this lane group may read the words back
      RBM2_MARK(1, 5);
    }
    // once the MMAs of this pass have read the operand planes, the MMA warp parks
    // the 2W rows in T_s again for the next pass's state build (during the sweep:
    // at C2 the last warp owns no walker)
    if (tcg && warp == THREADS / 32 - 1 && (batch + gridDim.x < A.n_batches || iter + 1 < n_iters)) {
      mbar_wait(smem_u32(mma_bar), (uint32_t)batch_no & 1u);
      if (lane == 0) {
        const uint32_t bytes = (uint32_t)(im.N * HP) * 4u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(w2_bar)), "r"(bytes)
                     : "memory");
        bulk_copy(T_s, img_g + im.off_w2, bytes, smem_u32(w2_bar));
      }
      __syncwarp();
    }
    if (A.do_grad) {
      RBM2_MARK(1, 6);
      // side sums first (the warps at the END of the CTA get here early)
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {
        const int e = rev + h2 * THREADS;
        if (!tcg && e < 2 * NP4) {
#pragma unroll 4
          for (int sb = 0; sb < n_valid; ++sb) acc_a[h2] += ws_s[(size_t)sb * 2 * NP4 + e];
        }
      }
      if (warp == THREADS / 32 - 1 && A.stat_partials != nullptr) {
        double e1 = 0.0, e2 = 0.0;
        for (int sb = lane; sb < n_valid; sb += 32) {
          const double e = (double)e_s[sb];
          e1 += e;
          e2 += e * e;
        }
        sum_e += warp_sum(e1);
        sum_e2 += warp_sum(e2);
      }
      // A grab = TG tiles x all walkers of the batch, the walkers split over the
      // 32 / TG lane groups of the warp (group wg takes walkers wg, wg + TQ, ...)
      // and the partial tiles reduce-scattered with 24 shuffles: lane (tl, wg)
      // ends up with row wg of tile tl for both weight columns.  Small grabs
      // keep the tail after the sweep short (a 32-tile grab runs ~4.5 us; the
      // warps without walkers work through the grabs during the sweep and the
      // last few used to keep 3 of 16 warps busy for ~8 us).
      constexpr int TG = 8, TQ = 32 / TG;
      const int tl = lane & (TG - 1), wg = lane / TG;
      for (;;) {
        if (tcg) break;                                      // the tensor cores do the tiles
        int tile_base = 0;
        if (lane == 0) tile_base = atomicAdd(tile_next_s, TG);
        tile_base = __shfl_sync(CGSVMC_FULL_MASK, tile_base, 0);
        if (tile_base >= n_tiles) break;
        const bool tile_ok = tile_base + tl < n_tiles;
        const int tile = min(tile_base + tl, n_tiles - 1);
        const int rt = tile / CT, ct = tile - rt * CT;
        const int i_own = 4 * rt + wg;                       // the row this lane stores: i < N: W[i][j]; i == N: c[j]
        // When the CTA's slice already holds sums (later passes of a launch)
        // the old values are requested before the accumulation loop, so the
        // L2 round trip hides behind it.
        float old[2][4];
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            old[k][c] = 0.f;
            if (batch_no != 0)
              old[k][c] = __ldcg(part + (size_t)k * A.P + im.N + 1 + (size_t)min(i_own, im.N) * im.H +
                                 min(4 * ct + c, im.H - 1));
          }
        float acc[2][4][4];
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
          for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[k][r][c] = 0.f;
#pragma unroll 2
        for (int sb = wg; sb < n_valid; sb += TQ) {
          const float4 T = *reinterpret_cast<const float4*>(T_s + sb * HP + 4 * ct);
          const float4 s0 = *reinterpret_cast<const float4*>(ws_s + (size_t)sb * 2 * NP4 + 4 * rt);
          const float4 s1 = *reinterpret_cast<const float4*>(ws_s + (size_t)sb * 2 * NP4 + NP4 + 4 * rt);
          const float tv[4] = {T.x, T.y, T.z, T.w};
          const float a0v[4] = {s0.x, s0.y, s0.z, s0.w};
          const float a1v[4] = {s1.x, s1.y, s1.z, s1.w};
#pragma unroll
          for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              acc[0][r][c] = fmaf(a0v[r], tv[c], acc[0][r][c]);
              acc[1][r][c] = fmaf(a1v[r], tv[c], acc[1][r][c]);
            }
        }
        // reduce-scatter over the walker groups (lane bits 4 and 3): fixed order, deterministic
        const bool up1 = (wg & 2) != 0, up0 = (wg & 1) != 0;
        float mine[2][4];
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float h[2];
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
              const float send = up1 ? acc[k][rr][c] : acc[k][rr + 2][c];
              const float keep = up1 ? acc[k][rr + 2][c] : acc[k][rr][c];
              h[rr] = keep + __shfl_xor_sync(CGSVMC_FULL_MASK, send, 2 * TG);
            }
            const float send = up0 ? h[0] : h[1];
            const float keep = up0 ? h[1] : h[0];
            mine[k][c] = keep + __shfl_xor_sync(CGSVMC_FULL_MASK, send, TG);
          }
        if (tile_ok && i_own <= im.N) {
#pragma unroll
          for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int j = 4 * ct + c;
              if (j >= im.H) continue;
              part[(size_t)k * A.P + im.N + 1 + (size_t)i_own * im.H + j] = mine[k][c] + old[k][c];
            }
        }
      }
      RBM2_MARK(1, 7);
      __syncthreads();
    }
  }
  if (MC && A.accept_count != nullptr) {
    unsigned int mine = sub == 0 ? n_acc : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(CGSVMC_FULL_MASK, mine, o);
    if (lane == 0 && mine) atomicAdd(A.accept_count, (unsigned long long)mine);
  }
  if (tcg && batch_no > 0) {
    // the passes since the last drain are still in TMEM
    mbar_wait(smem_u32(mma_bar), (uint32_t)(batch_no - 1) & 1u);
    tcg_drain<THREADS, NCOL>(tmem, T_s, drain_groups, part, A.P, im.N, im.H, NC, n_drained > 0);
  }
  if (A.do_grad) {
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {
      const int e = rev + h2 * THREADS;
      if (!tcg && e < 2 * NP4) {
        const int k = e / NP4, i = e - k * NP4;
        if (i <= im.N) part[(size_t)k * A.P + i] = acc_a[h2];   // a_i (i < N) and a0 (i == N)
      }
    }
    if (threadIdx.x == THREADS - 32 && A.stat_partials != nullptr) {
      A.stat_partials[2 * blockIdx.x] = sum_e;
      A.stat_partials[2 * blockIdx.x + 1] = sum_e2;
    }
  }
  RBM2_MARK(1, 8);
  if (A.do_grad && A.fuse_reduce)
    grid_reduce<THREADS>(A, T_s);      // the staging buffer is free: every tile pass ended with a CTA barrier
  if (tcg) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
  }
  RBM2_MARK(1, 9);
}

// ---------------------------------------------------------------------------
// host-side launchers of one (NW, LPW, KJV) variant
// ---------------------------------------------------------------------------
template <typename F>
inline int opt_in_smem(F kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(smem)");
  }
  return CGSVMC_OK;
}

template <int NW, int LPW, int KJV>
int launch_mc_variant(const Plan& pl, const float* img, uint64_t* packed, int64_t B, int n_steps,
                      uint64_t seed, uint64_t walker0, uint64_t step0,
                      unsigned long long* accept_count, float* log_amp_out, cudaStream_t st) {
  constexpr int THREADS = Geometry<LPW, KJV>::THREADS;
  if (pl.ws) {
    auto kern = mc_kernel<NW, LPW, KJV, true>;
    if (int rc = opt_in_smem(kern, pl.mc_smem)) return rc;
    kern<<<pl.grid, THREADS, pl.mc_smem, st>>>(pl.im, img, packed, B, pl.wpc, pl.n_batches, n_steps,
                                              seed, walker0, step0, pl.step0_dev, accept_count, log_amp_out);
  } else {
    auto kern = mc_kernel<NW, LPW, KJV, false>;
    if (int rc = opt_in_smem(kern, pl.mc_smem)) return rc;
    kern<<<pl.grid, THREADS, pl.mc_smem, st>>>(pl.im, img, packed, B, pl.wpc, pl.n_batches, n_steps,
                                              seed, walker0, step0, pl.step0_dev, accept_count, log_amp_out);
  }
  return cuda_fail(cudaGetLastError(), "rbm2 mc launch");
}

template <int NW, int LPW, int KJV>
int launch_walker_variant(const Plan& pl, const float* img, const WalkerArgs& A, cudaStream_t st) {
  constexpr int THREADS = Geometry<LPW, KJV, true>::THREADS;
  const bool mc = A.packed_rw != nullptr;
#define RBM2_LAUNCH_WALKER(WSV, MCV, PTV)                                         \
  do {                                                                            \
    auto kern = walker_kernel<NW, LPW, KJV, WSV, MCV, PTV>;                       \
    if (int rc = opt_in_smem(kern, pl.walker_smem)) return rc;                    \
    if (A.fuse_reduce) {                                                          \
      cudaLaunchConfig_t cfg = {};                                                \
      cfg.gridDim = dim3(pl.grid); cfg.blockDim = dim3(THREADS);                  \
      cfg.dynamicSmemBytes = pl.walker_smem; cfg.stream = st;                     \
      cudaLaunchAttribute attr[1];                                                \
      attr[0].id = cudaLaunchAttributeCooperative; attr[0].val.cooperative = 1;   \
      cfg.attrs = attr; cfg.numAttrs = 1;                                         \
      cudaError_t le = cudaLaunchKernelEx(&cfg, kern, pl.im, img, A);             \
      if (le != cudaSuccess) return cuda_fail(le, "rbm2 cooperative walker launch"); \
    } else {                                                                      \
      kern<<<pl.grid, THREADS, pl.walker_smem, st>>>(pl.im, img, A);              \
    }                                                                             \
  } while (0)
  if (pl.pt) {                       // planned only for LPW == 8 with the image in shared memory
    if (LPW == 8) { if (mc) RBM2_LAUNCH_WALKER(true, true, (LPW == 8)); else RBM2_LAUNCH_WALKER(true, false, (LPW == 8)); }
  } else if (pl.ws) { if (mc) RBM2_LAUNCH_WALKER(true, true, false); else RBM2_LAUNCH_WALKER(true, false, false); }
  else { if (mc) RBM2_LAUNCH_WALKER(false, true, false); else RBM2_LAUNCH_WALKER(false, false, false); }
#undef RBM2_LAUNCH_WALKER
  return cuda_fail(cudaGetLastError(), "rbm2 walker launch");
}

// walkers per CTA batch of a variant (host-side planning)
inline int variant_slots(int lpw, int kjv, bool walker) {
  const int kj = (32 / lpw) * kjv;
  return (((!walker && kj <= 10) ? 1024 : 512) / 32) * (32 / lpw);
}

#define RBM2_VARIANT_SWITCH(NWV, CALL)                       \
  switch (pl.lpw * 16 + pl.kjv) {                            \
    case 8 * 16 + 1: return CALL(NWV, 8, 1);                 \
    case 8 * 16 + 2: return CALL(NWV, 8, 2);                 \
    case 8 * 16 + 3: return CALL(NWV, 8, 3);                 \
    case 8 * 16 + 4: return CALL(NWV, 8, 4);                 \
    case 8 * 16 + 5: return CALL(NWV, 8, 5);                 \
    case 16 * 16 + 6: return CALL(NWV, 16, 6);               \
    case 16 * 16 + 7: return CALL(NWV, 16, 7);               \
    case 16 * 16 + 8: return CALL(NWV, 16, 8);               \
    default: break;                                          \
  }                                                          \
  set_error("rbm2: unsupported variant");                    \
  return CGSVMC_ERR_UNSUPPORTED;

}  // namespace rbm2
}  // namespace cgsvmc
