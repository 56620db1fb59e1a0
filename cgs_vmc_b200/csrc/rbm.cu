// Pure RBM ansatz (rbm with num_fc_layers == 0), wavefunctions.py:391-452:
//   z(sigma) = a . sigma + a0 + sum_j log cosh(theta_j),  theta = W^T sigma + c.
//
// One warp owns one walker.  theta_j and log cosh(theta_j) live in registers
// (lane l holds j = l, l + 32, ...), the spin words are replicated in every
// lane, W and a are staged in shared memory once per CTA.  A spin exchange
// (p: -1 -> +1, q: +1 -> -1) is the rank-2 update theta' = theta + 2 W[p] - 2 W[q]
// (SURVEY.md appendix A.2), so a Metropolis step or an off-diagonal matrix
// element costs O(H) instead of the O(N H) forward pass the reference runs
// twice per step (graph_builders.py:54-55, 74) / once per bond (operators.py:168).
//
// The sampler and the gradient sums of this ansatz run in rbm2 (rbm2.cu), which
// plans every shape accepted here.  This file keeps what rbm2 does not cover:
// the amplitudes (log_amp) and their directional derivative (log_amp_jvp, the
// forward half of the matrix-free S v of stochastic reconfiguration), the one-step replay of the reference's Metropolis
// step (parity hook), the local energy of Hamiltonians whose bond staging
// does not fit rbm2's shared memory (N = 256, H = 144: rbm2 takes at most 200 bonds),
// the per-bond terms of the local energy (bond values: spin-spin correlations),
// and the replica-swap values of the second Renyi entropy.
#include "common.cuh"
#include "internal.h"

namespace cgsvmc {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

struct RbmParams {
  const float* a;    // [N]
  const float* a0;   // [1]
  const float* W;    // [N, H]
  const float* c;    // [H]
  int N, H;
};

__host__ __device__ inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Shared-memory image: a[Npad] then (if WS) W[N][32 * KJ] zero padded.
template <int KJ, bool WS>
__device__ __forceinline__ void stage_params(const RbmParams& p, float* smem, const float*& a_s,
                                             const float*& Wp, int& ldw) {
  const int Npad = round_up(p.N, 32);
  float* a_sm = smem;
  for (int i = threadIdx.x; i < Npad; i += blockDim.x) a_sm[i] = i < p.N ? p.a[i] : 0.f;
  a_s = a_sm;
  if (WS) {
    constexpr int HS = 32 * KJ;
    float* W_sm = smem + Npad;
    for (int e = threadIdx.x; e < p.N * HS; e += blockDim.x) {
      const int i = e / HS, j = e - i * HS;
      W_sm[e] = j < p.H ? p.W[(size_t)i * p.H + j] : 0.f;
    }
    Wp = W_sm;
    ldw = HS;
  } else {
    Wp = p.W;
    ldw = p.H;
  }
  __syncthreads();
}

template <int NW>
__device__ __forceinline__ void load_spins(const uint64_t* packed, int64_t b, uint64_t (&s)[NW]) {
#pragma unroll
  for (int w = 0; w < NW; ++w) s[w] = packed[b * NW + w];
}

// theta_j = c_j + sum_i sigma_i W[i, j];  lc_j = log cosh theta_j.
template <int NW, int KJ, bool WS>
__device__ __forceinline__ void init_theta(const RbmParams& p, const float* Wp, int ldw,
                                           const uint64_t (&s)[NW], int lane, float (&th)[KJ],
                                           float (&lc)[KJ]) {
#pragma unroll
  for (int k = 0; k < KJ; ++k) {
    const int j = lane + 32 * k;
    th[k] = j < p.H ? p.c[j] : 0.f;
  }
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    const int n_here = min(64, p.N - 64 * w);
    const uint64_t word = s[w];
    for (int bpos = 0; bpos < n_here; ++bpos) {
      const uint32_t flip = (uint32_t)(((word >> bpos) & 1ull) ^ 1ull) << 31;
      const float* row = Wp + (size_t)(64 * w + bpos) * ldw;
#pragma unroll
      for (int k = 0; k < KJ; ++k) {
        const int j = lane + 32 * k;
        if (WS || j < p.H) th[k] += __uint_as_float(__float_as_uint(row[j]) ^ flip);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < KJ; ++k) lc[k] = log_cosh(th[k]);
}

// a . sigma + a0 + sum_j lc_j  (warp-uniform result)
template <int NW, int KJ>
__device__ __forceinline__ float full_log_amp(const RbmParams& p, const float* a_s,
                                              const uint64_t (&s)[NW], int lane,
                                              const float (&lc)[KJ]) {
  float part = 0.f;
#pragma unroll
  for (int k = 0; k < KJ; ++k) part += lc[k];
  for (int i = lane; i < p.N; i += 32) part += get_bit<NW>(s, i) ? a_s[i] : -a_s[i];
  return warp_sum(part) + p.a0[0];
}

// log(psi(sigma') / psi(sigma)) for sigma' = sigma with `dn` raised and `up`
// lowered; also returns the updated theta / log-cosh rows.
template <int KJ, bool WS>
__device__ __forceinline__ float exchange_log_ratio(const RbmParams& p, const float* a_s,
                                                    const float* Wp, int ldw, int up, int dn,
                                                    int lane, const float (&th)[KJ],
                                                    const float (&lc)[KJ], float (&tn)[KJ],
                                                    float (&ln)[KJ]) {
  const float* wu = Wp + (size_t)up * ldw;
  const float* wd = Wp + (size_t)dn * ldw;
  float part = 0.f;
#pragma unroll
  for (int k = 0; k < KJ; ++k) {
    const int j = lane + 32 * k;
    float d = 0.f;
    if (WS || j < p.H) d = wd[j] - wu[j];
    tn[k] = fmaf(2.f, d, th[k]);
    ln[k] = log_cosh(tn[k]);
    part += ln[k] - lc[k];
  }
  return warp_sum(part) + 2.f * (a_s[dn] - a_s[up]);
}

// ---------------------------------------------------------------------------
// K1: z for a batch
// ---------------------------------------------------------------------------
template <int NW, int KJ, bool WS>
__global__ void __launch_bounds__(kThreads)
rbm_log_amp_kernel(RbmParams p, const uint64_t* __restrict__ packed, int64_t B,
                   float* __restrict__ out) {
  extern __shared__ float smem[];
  const float *a_s, *Wp; int ldw;
  stage_params<KJ, WS>(p, smem, a_s, Wp, ldw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    uint64_t s[NW]; float th[KJ], lc[KJ];
    load_spins<NW>(packed, b, s);
    init_theta<NW, KJ, WS>(p, Wp, ldw, s, lane, th, lc);
    const float z = full_log_amp<NW, KJ>(p, a_s, s, lane, lc);
    if (lane == 0) out[b] = z;
  }
}

// ---------------------------------------------------------------------------
// K1 tangent: y_b = sum_p (d z_b / d params_p) v_p for a tangent v in the flat
// layout (v_a, v_a0, V, v_c), seen through `t` like the parameters through `p`:
//   y = sum_j tanh(theta_j) u_j + v_a . sigma + v_a0,  u = V^T sigma + v_c.
// theta and u are built in the same pass over the spin bits; W and V are
// staged side by side when both fit (rbm_log_amp_jvp decides).  FP32 with a
// fixed summation order: the result does not change from run to run.
// ---------------------------------------------------------------------------
template <int NW, int KJ, bool WS>
__global__ void __launch_bounds__(kThreads)
rbm_log_amp_jvp_kernel(RbmParams p, RbmParams t, const uint64_t* __restrict__ packed, int64_t B,
                       float* __restrict__ out) {
  extern __shared__ float smem[];
  const float *a_s, *Wp, *va_s, *Vp; int ldw;
  const int param_floats = round_up(p.N, 32) + (WS ? p.N * 32 * KJ : 0);
  stage_params<KJ, WS>(p, smem, a_s, Wp, ldw);
  stage_params<KJ, WS>(t, smem + param_floats, va_s, Vp, ldw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    uint64_t s[NW]; float th[KJ], u[KJ];
    load_spins<NW>(packed, b, s);
#pragma unroll
    for (int k = 0; k < KJ; ++k) {
      const int j = lane + 32 * k;
      th[k] = j < p.H ? p.c[j] : 0.f;
      u[k] = j < p.H ? t.c[j] : 0.f;
    }
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      const int n_here = min(64, p.N - 64 * w);
      const uint64_t word = s[w];
      for (int bpos = 0; bpos < n_here; ++bpos) {
        const uint32_t flip = (uint32_t)(((word >> bpos) & 1ull) ^ 1ull) << 31;
        const float* wrow = Wp + (size_t)(64 * w + bpos) * ldw;
        const float* vrow = Vp + (size_t)(64 * w + bpos) * ldw;
#pragma unroll
        for (int k = 0; k < KJ; ++k) {
          const int j = lane + 32 * k;
          if (WS || j < p.H) {
            th[k] += __uint_as_float(__float_as_uint(wrow[j]) ^ flip);
            u[k] += __uint_as_float(__float_as_uint(vrow[j]) ^ flip);
          }
        }
      }
    }
    float part = 0.f;
#pragma unroll
    for (int k = 0; k < KJ; ++k) part = fmaf(tanhf(th[k]), u[k], part);
    for (int i = lane; i < p.N; i += 32) part += get_bit<NW>(s, i) ? va_s[i] : -va_s[i];
    const float y = warp_sum(part) + t.a0[0];
    if (lane == 0) out[b] = y;
  }
}

// ---------------------------------------------------------------------------
// K2 replay: one Metropolis step consuming caller-supplied uniforms
// (graph_builders.py:59-79 verbatim)
// ---------------------------------------------------------------------------
template <int NW, int KJ, bool WS>
__global__ void __launch_bounds__(kThreads)
rbm_mc_replay_kernel(RbmParams p, uint64_t* __restrict__ packed, int64_t B,
                     const float* __restrict__ u_sites, const float* __restrict__ u_acc,
                     int32_t* down_out, int32_t* up_out, float* log_ratio_out,
                     uint8_t* accept_out) {
  extern __shared__ float smem[];
  const float *a_s, *Wp; int ldw;
  stage_params<KJ, WS>(p, smem, a_s, Wp, ldw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    uint64_t s[NW]; float th[KJ], lc[KJ];
    load_spins<NW>(packed, b, s);
    init_theta<NW, KJ, WS>(p, Wp, ldw, s, lane, th, lc);
    // argmin / argmax of sigma_i * u_i, first occurrence on ties
    float vmin = INFINITY, vmax = -INFINITY;
    int imin = p.N, imax = p.N;
    for (int i = lane; i < p.N; i += 32) {
      const float u = u_sites[b * p.N + i];
      const float v = get_bit<NW>(s, i) ? u : -u;
      if (v < vmin) { vmin = v; imin = i; }
      if (v > vmax) { vmax = v; imax = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(CGSVMC_FULL_MASK, vmin, o);
      const int oi = __shfl_xor_sync(CGSVMC_FULL_MASK, imin, o);
      if (ov < vmin || (ov == vmin && oi < imin)) { vmin = ov; imin = oi; }
      const float ow = __shfl_xor_sync(CGSVMC_FULL_MASK, vmax, o);
      const int oj = __shfl_xor_sync(CGSVMC_FULL_MASK, imax, o);
      if (ow > vmax || (ow == vmax && oj < imax)) { vmax = ow; imax = oj; }
    }
    const int dn = imin, up = imax;   // +2 at `dn`, -2 at `up` (graph_builders.py:67-73)
    float tn[KJ], ln[KJ];
    const float dl = exchange_log_ratio<KJ, WS>(p, a_s, Wp, ldw, up, dn, lane, th, lc, tn, ln);
    const bool acc = expf(dl) > sqrtf(u_acc[b]);   // graph_builders.py:75-79
    if (lane == 0) {
      if (down_out) down_out[b] = dn;
      if (up_out) up_out[b] = up;
      if (log_ratio_out) log_ratio_out[b] = dl;
      if (accept_out) accept_out[b] = acc ? 1 : 0;
      if (acc) {
        flip_bit<NW>(s, up);
        flip_bit<NW>(s, dn);
#pragma unroll
        for (int w = 0; w < NW; ++w) packed[b * NW + w] = s[w];
      }
    }
  }
}

// ---------------------------------------------------------------------------
// K3: fused local energy, operators.py:227-259
// ---------------------------------------------------------------------------
template <int NW, int KJ, bool WS>
__global__ void __launch_bounds__(kThreads)
rbm_local_energy_kernel(RbmParams p, const int2* __restrict__ bonds_ij,
                        const float* __restrict__ bonds_jx, const float* __restrict__ bonds_jz,
                        int n_bonds, const uint64_t* __restrict__ packed, int64_t B,
                        float* __restrict__ e_loc, float* __restrict__ log_amp_out,
                        float* __restrict__ diag_out, float* __restrict__ off_out) {
  extern __shared__ float smem[];
  const float *a_s, *Wp; int ldw;
  // bond table behind the parameter image
  const int param_floats = round_up(p.N, 32) + (WS ? p.N * 32 * KJ : 0);
  int4* bond_s = reinterpret_cast<int4*>(smem + round_up(param_floats, 4));
  for (int k = threadIdx.x; k < n_bonds; k += blockDim.x) {
    const int2 ij = bonds_ij[k];
    bond_s[k] = make_int4(ij.x, ij.y, __float_as_int(bonds_jx[k]), __float_as_int(bonds_jz[k]));
  }
  stage_params<KJ, WS>(p, smem, a_s, Wp, ldw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    uint64_t s[NW]; float th[KJ], lc[KJ];
    load_spins<NW>(packed, b, s);
    init_theta<NW, KJ, WS>(p, Wp, ldw, s, lane, th, lc);
    float diag = 0.f, off = 0.f;
    for (int k = 0; k < n_bonds; ++k) {
      const int4 bd = bond_s[k];
      const int bi = get_bit<NW>(s, bd.x), bj = get_bit<NW>(s, bd.y);
      const float jz = __int_as_float(bd.w);
      if (bi == bj) {
        diag = fmaf(0.25f, jz, diag);                      // operators.py:165,169
      } else {
        diag = fmaf(-0.25f, jz, diag);
        const int up = bi ? bd.x : bd.y, dn = bi ? bd.y : bd.x;
        float tn[KJ], ln[KJ];
        const float dl = exchange_log_ratio<KJ, WS>(p, a_s, Wp, ldw, up, dn, lane, th, lc, tn, ln);
        off = fmaf(0.5f * __int_as_float(bd.z), fast_exp(dl), off);   // operators.py:168-169
      }
    }
    float z = 0.f;
    if (log_amp_out != nullptr) z = full_log_amp<NW, KJ>(p, a_s, s, lane, lc);
    if (lane == 0) {
      e_loc[b] = diag + off;
      if (log_amp_out) log_amp_out[b] = z;
      if (diag_out) diag_out[b] = diag;
      if (off_out) off_out[b] = off;
    }
  }
}

// ---------------------------------------------------------------------------
// K3 per bond: values[b, k] = jz_k/4 s_i s_j + jx_k/2 [s_i != s_j] psi(flip_k)/psi,
// the summands of rbm_local_energy_kernel kept instead of reduced.  Any number
// of bonds: the first n_staged go to shared memory behind the parameter image,
// the rest are read through the read-only path (every lane reads the same bond:
// one broadcast transaction).  Lane k & 31 keeps bond k's value and the warp
// stores 32 consecutive values at a time.
// ---------------------------------------------------------------------------
template <int NW, int KJ, bool WS>
__global__ void __launch_bounds__(kThreads)
rbm_bond_values_kernel(RbmParams p, const int2* __restrict__ bonds_ij,
                       const float* __restrict__ bonds_jx, const float* __restrict__ bonds_jz,
                       int n_bonds, int n_staged, const uint64_t* __restrict__ packed, int64_t B,
                       float* __restrict__ values) {
  extern __shared__ float smem[];
  const float *a_s, *Wp; int ldw;
  const int param_floats = round_up(p.N, 32) + (WS ? p.N * 32 * KJ : 0);
  int4* bond_s = reinterpret_cast<int4*>(smem + round_up(param_floats, 4));
  for (int k = threadIdx.x; k < n_staged; k += blockDim.x) {
    const int2 ij = bonds_ij[k];
    bond_s[k] = make_int4(ij.x, ij.y, __float_as_int(bonds_jx[k]), __float_as_int(bonds_jz[k]));
  }
  stage_params<KJ, WS>(p, smem, a_s, Wp, ldw);   // ends with the CTA barrier
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    uint64_t s[NW]; float th[KJ], lc[KJ];
    load_spins<NW>(packed, b, s);
    init_theta<NW, KJ, WS>(p, Wp, ldw, s, lane, th, lc);
    float* row = values + b * (int64_t)n_bonds;
    float keep = 0.f;
    for (int k = 0; k < n_bonds; ++k) {
      int4 bd;
      if (k < n_staged) {
        bd = bond_s[k];
      } else {
        const int2 ij = __ldg(bonds_ij + k);
        bd = make_int4(ij.x, ij.y, __float_as_int(__ldg(bonds_jx + k)), __float_as_int(__ldg(bonds_jz + k)));
      }
      const int bi = get_bit<NW>(s, bd.x), bj = get_bit<NW>(s, bd.y);
      const float jx = __int_as_float(bd.z), jz = __int_as_float(bd.w);
      float v = (bi == bj ? 0.25f : -0.25f) * jz;
      if (bi != bj && jx != 0.f) {   // warp-uniform: the spins are replicated in every lane
        const int up = bi ? bd.x : bd.y, dn = bi ? bd.y : bd.x;
        float tn[KJ], ln[KJ];
        const float dl = exchange_log_ratio<KJ, WS>(p, a_s, Wp, ldw, up, dn, lane, th, lc, tn, ln);
        v += (0.5f * jx) * fast_exp(dl);
      }
      if (lane == (k & 31)) keep = v;
      if ((k & 31) == 31 || k == n_bonds - 1) {
        if (lane <= (k & 31)) row[(k & ~31) + lane] = keep;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Replica swap (second Renyi entropy): pair p = (sigma1 = row p, sigma2 = row
// P + p); for region A (mask & valid sites) and D = (sigma1 ^ sigma2) & A,
//   values[p, r] = psi(sigma1 ^ D) psi(sigma2 ^ D) / (psi(sigma1) psi(sigma2))
// with 0 when the replicas hold different numbers of up spins in A (the
// swapped pair leaves the sampled S^z sector) and exactly 1 when D is empty
// or holds every differing site (the swapped pair is the pair itself).  The
// visible bias cancels; with Delta_j = sum_{i in D} s2_i W_ij
//   log r = sum_j lc(th1_j + 2 Delta_j) - lc1_j + lc(th2_j - 2 Delta_j) - lc2_j.
// Delta is summed over D in increasing site order: it extends the last
// computed region's Delta when that D is a prefix of this one (nested
// prefixes: O(N H) per pair for the whole list) and restarts from 0
// otherwise, the same float32 additions either way, so a region's value does
// not depend on the list around it.  Lane r & 31 keeps region r's value and
// the warp stores 32 consecutive values at a time.
// ---------------------------------------------------------------------------
template <int NW, int KJ, bool WS>
__global__ void __launch_bounds__(kThreads)
rbm_swap_values_kernel(RbmParams p, const uint64_t* __restrict__ packed, int64_t P,
                       const uint64_t* __restrict__ regions, int n_regions, float* __restrict__ values) {
  extern __shared__ float smem[];
  const float *a_s, *Wp; int ldw;
  stage_params<KJ, WS>(p, smem, a_s, Wp, ldw);   // ends with the CTA barrier
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < P; b += (int64_t)gridDim.x * kWarps) {
    uint64_t s1[NW], s2[NW], dprev[NW];
    float th1[KJ], lc1[KJ], th2[KJ], lc2[KJ], dl[KJ];
    load_spins<NW>(packed, b, s1);
    load_spins<NW>(packed, P + b, s2);
    init_theta<NW, KJ, WS>(p, Wp, ldw, s1, lane, th1, lc1);
    init_theta<NW, KJ, WS>(p, Wp, ldw, s2, lane, th2, lc2);
#pragma unroll
    for (int w = 0; w < NW; ++w) dprev[w] = 0ull;
#pragma unroll
    for (int k = 0; k < KJ; ++k) dl[k] = 0.f;
    float* row = values + b * (int64_t)n_regions;
    float keep = 0.f;
    for (int r = 0; r < n_regions; ++r) {
      uint64_t d[NW];
      int up1 = 0, up2 = 0;
      bool empty = true, whole = true;
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const uint64_t valid = valid_mask_word(p.N, w);
        const uint64_t m = __ldg(regions + (int64_t)r * NW + w) & valid;
        const uint64_t diff = s1[w] ^ s2[w];
        d[w] = diff & m;
        up1 += __popcll(s1[w] & m);
        up2 += __popcll(s2[w] & m);
        empty = empty && d[w] == 0ull;
        whole = whole && d[w] == (diff & valid);
      }
      float v;
      if (up1 != up2) {
        v = 0.f;
      } else if (empty || whole) {
        v = 1.f;
      } else {
        // extend iff D restricted to the sites up to dprev's highest one is dprev
        bool extend = true;
        bool below = false;   // word w lies below dprev's highest non-zero word
#pragma unroll
        for (int w = NW - 1; w >= 0; --w) {
          uint64_t upto;
          if (below) {
            upto = ~0ull;
          } else if (dprev[w] != 0ull) {
            const int hb = 63 - __clzll(dprev[w]);
            upto = hb == 63 ? ~0ull : (2ull << hb) - 1ull;
            below = true;
          } else {
            upto = 0ull;
          }
          extend = extend && (d[w] & upto) == dprev[w];
        }
        if (!extend) {
#pragma unroll
          for (int k = 0; k < KJ; ++k) dl[k] = 0.f;
#pragma unroll
          for (int w = 0; w < NW; ++w) dprev[w] = 0ull;
        }
#pragma unroll
        for (int w = 0; w < NW; ++w) {
          uint64_t add = d[w] & ~dprev[w];   // new sites of this word, in increasing order
          while (add != 0ull) {
            const int bpos = __ffsll((long long)add) - 1;
            add &= add - 1ull;
            const uint32_t flip = (uint32_t)(((s2[w] >> bpos) & 1ull) ^ 1ull) << 31;
            const float* wrow = Wp + (size_t)(64 * w + bpos) * ldw;
#pragma unroll
            for (int k = 0; k < KJ; ++k) {
              const int j = lane + 32 * k;
              if (WS || j < p.H) dl[k] += __uint_as_float(__float_as_uint(wrow[j]) ^ flip);
            }
          }
          dprev[w] = d[w];
        }
        float part = 0.f;
#pragma unroll
        for (int k = 0; k < KJ; ++k) {
          part += log_cosh(fmaf(2.f, dl[k], th1[k])) - lc1[k];
          part += log_cosh(fmaf(-2.f, dl[k], th2[k])) - lc2[k];
        }
        v = fast_exp(warp_sum(part));
      }
      if (lane == (r & 31)) keep = v;
      if ((r & 31) == 31 || r == n_regions - 1) {
        if (lane <= (r & 31)) row[(r & ~31) + lane] = keep;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// host-side dispatch
// ---------------------------------------------------------------------------
// `flat` is a vector in the flat parameter layout: the parameters or a tangent.
RbmParams make_params(const cgsvmc_ansatz* a, const float* flat) {
  RbmParams p;
  p.N = a->desc.n_sites;
  p.H = a->desc.layer_size;
  p.a = flat + a->offsets[0];
  p.a0 = flat + a->offsets[1];
  p.W = flat + a->offsets[2];
  p.c = flat + a->offsets[3];
  return p;
}

RbmParams make_params(const cgsvmc_ansatz* a) { return make_params(a, a->params); }

int pick_kj(int H) { return H <= 64 ? 2 : H <= 128 ? 4 : H <= 160 ? 5 : 8; }
int pick_nw(int N) { return n_words(N); }

struct Geometry {
  int kj;
  bool ws;
  size_t param_bytes;
};

Geometry geometry(const cgsvmc_ansatz* a) {
  Geometry g;
  g.kj = pick_kj(a->desc.layer_size);
  const size_t base = (size_t)round_up(a->desc.n_sites, 32) * 4;
  const size_t wbytes = (size_t)a->desc.n_sites * 32 * g.kj * 4;
  g.ws = base + wbytes <= 96 * 1024;   // keep >= 2 CTAs per SM
  g.param_bytes = base + (g.ws ? wbytes : 0);
  return g;
}

int grid_for(const cgsvmc_ansatz* a, int64_t B) {
  const int64_t need = (B + kWarps - 1) / kWarps;
  const int64_t cap = (int64_t)a->num_sms * 8;
  return (int)std::max<int64_t>(1, std::min(need, cap));
}

template <typename F>
int set_smem(F kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(smem)");
  }
  return CGSVMC_OK;
}

#define RBM_DISPATCH_KJ_WS(NWV, BODY)                                   \
  switch (g.kj) {                                                       \
    case 2: if (g.ws) { BODY(NWV, 2, true) } else { BODY(NWV, 2, false) } break; \
    case 4: if (g.ws) { BODY(NWV, 4, true) } else { BODY(NWV, 4, false) } break; \
    case 5: if (g.ws) { BODY(NWV, 5, true) } else { BODY(NWV, 5, false) } break; \
    default: if (g.ws) { BODY(NWV, 8, true) } else { BODY(NWV, 8, false) } break; \
  }
#define RBM_DISPATCH(BODY)                                              \
  switch (pick_nw(a->desc.n_sites)) {                                   \
    case 1: RBM_DISPATCH_KJ_WS(1, BODY) break;                          \
    case 2: RBM_DISPATCH_KJ_WS(2, BODY) break;                          \
    default: RBM_DISPATCH_KJ_WS(4, BODY) break;                         \
  }

}  // namespace

bool rbm_fast_supported(const cgsvmc_ansatz* a) {
  return a->desc.kind == CGSVMC_ANSATZ_RBM && a->desc.num_layers == 0 &&
         a->desc.layer_size <= 256 && a->desc.n_sites <= CGSVMC_MAX_SITES &&
         n_words(a->desc.n_sites) != 3;   // kernels are instantiated for 1, 2 and 4 words
}

int rbm_log_amp(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, float* out,
                cudaStream_t st) {
  const RbmParams p = make_params(a);
  const Geometry g = geometry(a);
  const int grid = grid_for(a, B);
  const size_t smem = g.param_bytes;
#define BODY(NWV, KJV, WSV)                                                        \
  { auto kern = rbm_log_amp_kernel<NWV, KJV, WSV>;                                \
    if (int rc = set_smem(kern, smem)) return rc;                                 \
    kern<<<grid, kThreads, smem, st>>>(p, packed, B, out); }
  RBM_DISPATCH(BODY)
#undef BODY
  return cuda_fail(cudaGetLastError(), "rbm_log_amp launch");
}

int rbm_log_amp_jvp(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, const float* tangent,
                    float* out, cudaStream_t st) {
  const RbmParams p = make_params(a);
  const RbmParams t = make_params(a, tangent);
  // two parameter images (params, tangent) under the budget one has in geometry()
  Geometry g = geometry(a);
  const size_t base = (size_t)round_up(a->desc.n_sites, 32) * 4;
  const size_t wbytes = (size_t)a->desc.n_sites * 32 * g.kj * 4;
  g.ws = 2 * (base + wbytes) <= 96 * 1024;
  const size_t smem = 2 * (base + (g.ws ? wbytes : 0));
  const int grid = grid_for(a, B);
#define BODY(NWV, KJV, WSV)                                                        \
  { auto kern = rbm_log_amp_jvp_kernel<NWV, KJV, WSV>;                            \
    if (int rc = set_smem(kern, smem)) return rc;                                 \
    kern<<<grid, kThreads, smem, st>>>(p, t, packed, B, out); }
  RBM_DISPATCH(BODY)
#undef BODY
  return cuda_fail(cudaGetLastError(), "rbm_log_amp_jvp launch");
}

int rbm_mc_replay(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, const float* u_sites,
                  const float* u_acc, int32_t* down, int32_t* up, float* log_ratio,
                  uint8_t* accept, cudaStream_t st) {
  const RbmParams p = make_params(a);
  const Geometry g = geometry(a);
  const int grid = grid_for(a, B);
  const size_t smem = g.param_bytes;
#define BODY(NWV, KJV, WSV)                                                        \
  { auto kern = rbm_mc_replay_kernel<NWV, KJV, WSV>;                              \
    if (int rc = set_smem(kern, smem)) return rc;                                 \
    kern<<<grid, kThreads, smem, st>>>(p, packed, B, u_sites, u_acc, down, up,    \
                                       log_ratio, accept); }
  RBM_DISPATCH(BODY)
#undef BODY
  return cuda_fail(cudaGetLastError(), "rbm_mc_replay launch");
}

int rbm_local_energy(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed,
                     int64_t B, float* e_loc, float* log_amp_out, float* diag_out, float* off_out,
                     cudaStream_t st) {
  const RbmParams p = make_params(a);
  const Geometry g = geometry(a);
  const int grid = grid_for(a, B);
  const size_t smem = round_up((int)g.param_bytes, 16) + (size_t)h->n_bonds * sizeof(int4);
#define BODY(NWV, KJV, WSV)                                                        \
  { auto kern = rbm_local_energy_kernel<NWV, KJV, WSV>;                           \
    if (int rc = set_smem(kern, smem)) return rc;                                 \
    kern<<<grid, kThreads, smem, st>>>(p, h->ij, h->jx, h->jz, h->n_bonds, packed, B, e_loc, \
                                       log_amp_out, diag_out, off_out); }
  RBM_DISPATCH(BODY)
#undef BODY
  return cuda_fail(cudaGetLastError(), "rbm_local_energy launch");
}

int rbm_bond_values(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                    float* values, cudaStream_t st) {
  const RbmParams p = make_params(a);
  const Geometry g = geometry(a);
  const int grid = grid_for(a, B);
  // bonds fill the shared memory beside the parameter image up to 112 KB, which
  // keeps two CTAs per SM (geometry() caps the image at 96 KB)
  constexpr size_t kSmemBudget = 112 * 1024;
  const size_t param_bytes = round_up((int)g.param_bytes, 16);
  const int n_staged = (int)std::min<size_t>((size_t)h->n_bonds, (kSmemBudget - param_bytes) / sizeof(int4));
  const size_t smem = param_bytes + (size_t)n_staged * sizeof(int4);
#define BODY(NWV, KJV, WSV)                                                        \
  { auto kern = rbm_bond_values_kernel<NWV, KJV, WSV>;                            \
    if (int rc = set_smem(kern, smem)) return rc;                                 \
    kern<<<grid, kThreads, smem, st>>>(p, h->ij, h->jx, h->jz, h->n_bonds, n_staged, packed, B, \
                                       values); }
  RBM_DISPATCH(BODY)
#undef BODY
  return cuda_fail(cudaGetLastError(), "rbm_bond_values launch");
}

int rbm_swap_values(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t P, const uint64_t* regions,
                    int n_regions, float* values, cudaStream_t st) {
  const RbmParams p = make_params(a);
  const Geometry g = geometry(a);
  const int grid = grid_for(a, P);
  const size_t smem = g.param_bytes;
#define BODY(NWV, KJV, WSV)                                                        \
  { auto kern = rbm_swap_values_kernel<NWV, KJV, WSV>;                            \
    if (int rc = set_smem(kern, smem)) return rc;                                 \
    kern<<<grid, kThreads, smem, st>>>(p, packed, P, regions, n_regions, values); }
  RBM_DISPATCH(BODY)
#undef BODY
  return cuda_fail(cudaGetLastError(), "rbm_swap_values launch");
}

}  // namespace cgsvmc
