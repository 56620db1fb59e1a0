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
// the amplitudes (log_amp), the one-step replay of the reference's Metropolis
// step (parity hook), and the local energy of Hamiltonians whose bond staging
// does not fit rbm2's shared memory (N = 256, H = 144: rbm2 takes at most 200 bonds).
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
// host-side dispatch
// ---------------------------------------------------------------------------
RbmParams make_params(const cgsvmc_ansatz* a) {
  RbmParams p;
  p.N = a->desc.n_sites;
  p.H = a->desc.layer_size;
  p.a = a->params + a->offsets[0];
  p.a0 = a->params + a->offsets[1];
  p.W = a->params + a->offsets[2];
  p.c = a->params + a->offsets[3];
  return p;
}

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

}  // namespace cgsvmc
