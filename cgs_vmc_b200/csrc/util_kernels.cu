// Layout conversion, initial walker state, bond enumeration and small
// reductions.  All of these are HBM-bound integer / byte work: coalesced,
// one pass, no staging.
#include "common.cuh"
#include "internal.h"

namespace cgsvmc {
namespace {

constexpr int kThreads = 256;

// float32 [B, N] of +-1  ->  uint64 [B, W].  One warp per (walker, word):
// lanes read 32 consecutive floats, a ballot forms half a word.
__global__ void pack_kernel(const float* __restrict__ configs, int64_t B, int N, int W,
                            uint64_t* __restrict__ packed) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t item = warp; item < B * W; item += n_warps) {
    const int64_t b = item / W;
    const int w = (int)(item - b * W);
    const int i0 = w * 64 + lane, i1 = i0 + 32;
    const float v0 = i0 < N ? configs[b * N + i0] : -1.f;
    const float v1 = i1 < N ? configs[b * N + i1] : -1.f;
    const uint32_t lo = __ballot_sync(CGSVMC_FULL_MASK, v0 > 0.f);
    const uint32_t hi = __ballot_sync(CGSVMC_FULL_MASK, v1 > 0.f);
    if (lane == 0) packed[item] = ((uint64_t)hi << 32) | lo;
  }
}

__global__ void unpack_kernel(const uint64_t* __restrict__ packed, int64_t B, int N, int W,
                              float* __restrict__ configs) {
  const int64_t total = B * N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = e / N;
    const int i = (int)(e - b * N);
    const uint64_t word = packed[b * W + (i >> 6)];
    configs[e] = ((word >> (i & 63)) & 1ull) ? 1.f : -1.f;
  }
}

// utils.random_configurations (utils.py:169-192): N/2 distinct uniformly
// chosen sites are set to -1.  Selection sampling (Knuth 3.4.2 S) draws the
// subset in one ordered pass; Philox counter = (draw index, walker).
__global__ void random_configs_kernel(uint64_t* __restrict__ packed, int64_t B, int N, int W,
                                      uint64_t seed, uint64_t walker0) {
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B;
       b += (int64_t)gridDim.x * blockDim.x) {
    uint64_t words[CGSVMC_MAX_WORDS];
#pragma unroll
    for (int w = 0; w < CGSVMC_MAX_WORDS; ++w) words[w] = valid_mask_word(N, w);
    int need = N / 2;
    Philox4 r = {0, 0, 0, 0};
    for (int i = 0; i < N && need > 0; ++i) {
      if ((i & 3) == 0)
        r = walker_step_random(seed ^ 0x5DEECE66Dull, walker0 + (uint64_t)b, (uint64_t)(i >> 2));
      const uint32_t x = (i & 3) == 0 ? r.x : (i & 3) == 1 ? r.y : (i & 3) == 2 ? r.z : r.w;
      if ((int)__umulhi(x, (uint32_t)(N - i)) < need) {
#pragma unroll
        for (int w = 0; w < CGSVMC_MAX_WORDS; ++w)
          if ((i >> 6) == w) words[w] &= ~(1ull << (i & 63));
        --need;
      }
    }
    for (int w = 0; w < W; ++w) packed[b * W + w] = words[w];
  }
}

// operators.py:154-167 on bits: one thread per (walker, bond).
__global__ void flip_enum_kernel(const int2* __restrict__ ij, int n_bonds,
                                 const uint64_t* __restrict__ packed, int64_t B, int W,
                                 uint64_t* __restrict__ flipped, uint32_t* __restrict__ mask) {
  const int mask_words = (n_bonds + 31) / 32;
  const int lane = threadIdx.x & 31;
  // items are (walker, bond-group-of-32) so that a ballot builds one mask word
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t item = warp; item < B * mask_words; item += n_warps) {
    const int64_t b = item / mask_words;
    const int g = (int)(item - b * mask_words);
    const int k = g * 32 + lane;
    bool anti = false;
    if (k < n_bonds) {
      const int2 bd = ij[k];
      const uint64_t wi = packed[b * W + (bd.x >> 6)], wj = packed[b * W + (bd.y >> 6)];
      anti = (((wi >> (bd.x & 63)) ^ (wj >> (bd.y & 63))) & 1ull) != 0;
      if (flipped != nullptr) {
        for (int w = 0; w < W; ++w) {
          uint64_t word = packed[b * W + w];
          if (anti && (bd.x >> 6) == w) word ^= 1ull << (bd.x & 63);
          if (anti && (bd.y >> 6) == w) word ^= 1ull << (bd.y & 63);
          flipped[(b * n_bonds + k) * W + w] = word;
        }
      }
    }
    const uint32_t vote = __ballot_sync(CGSVMC_FULL_MASK, anti);
    if (lane == 0 && mask != nullptr) mask[item] = vote;
  }
}

__global__ void energy_stats_kernel(const float* __restrict__ e, int64_t B, double* stats) {
  double s1 = 0.0, s2 = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < B;
       i += (int64_t)gridDim.x * blockDim.x) {
    const double v = (double)e[i];
    s1 += v;
    s2 += v * v;
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  __shared__ double sh[2][kThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sh[0][warp] = s1; sh[1][warp] = s2; }
  __syncthreads();
  if (warp == 0) {
    s1 = lane < kThreads / 32 ? sh[0][lane] : 0.0;
    s2 = lane < kThreads / 32 ? sh[1][lane] : 0.0;
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) {
      atomicAdd(&stats[0], s1);
      atomicAdd(&stats[1], s2);
      if (blockIdx.x == 0) atomicAdd(&stats[2], (double)B);
    }
  }
}

// out[n] += sum_p partials[p][n]   (fixed order => deterministic).  A block
// reduces 32 consecutive outputs; its 8 warps each take every 8th partial
// (coalesced 128-byte reads), then the 8 slices are added in a fixed order.
__global__ void reduce_partials_kernel(const float* __restrict__ partials, int n_parts, int64_t n,
                                       float* __restrict__ out) {
  __shared__ float sh[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t i0 = (int64_t)blockIdx.x * 32; i0 < n; i0 += (int64_t)gridDim.x * 32) {
    const int64_t i = i0 + lane;
    float acc = 0.f;
    if (i < n)
      for (int p = warp; p < n_parts; p += 8) acc += partials[(int64_t)p * n + i];
    sh[warp][lane] = acc;
    __syncthreads();
    if (warp == 0 && i < n) {
      float total = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) total += sh[w][lane];
      out[i] += total;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// Amplitude-agnostic forms of the sampler and of the local energy, for
// wavefunctions whose amplitude is not one fused kernel: signed output
// activations (layers.py:13-21) and the sum / difference / product composites
// (wavefunctions.py:61-165).  The caller evaluates (log|psi|, sign psi) of the
// proposed / bond-flipped configurations with cgsvmc_log_amp of the parts.
// ---------------------------------------------------------------------------
// graph_builders.py:59-73: a uniformly random up site and a uniformly random
// down site are exchanged.  Same Philox convention as the fused samplers
// (k_up = mulhi(r.x, n_up), k_dn = mulhi(r.y, n_dn), u = (r.z >> 8) 2^-24), so a
// walker sees the same proposals on either path.  One warp per walker.
template <int NW>
__global__ void propose_exchange_kernel(const uint64_t* __restrict__ packed, int64_t B, int N, int W,
                                        uint64_t seed, uint64_t walker0, uint64_t step,
                                        uint64_t* __restrict__ proposed, float* __restrict__ u_acc) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp; b < B; b += n_warps) {
    uint64_t s[NW], up_mask[NW], dn_mask[NW];
    int n_up = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      s[w] = w < W ? packed[b * W + w] : 0ull;
      up_mask[w] = s[w] & valid_mask_word(N, w);
      dn_mask[w] = ~s[w] & valid_mask_word(N, w);
      n_up += __popcll(up_mask[w]);
    }
    const int n_dn = N - n_up;
    const Philox4 r = walker_step_random(seed, walker0 + (uint64_t)b, step);
    if (n_up > 0 && n_dn > 0) {
      const int up = select_kth_bit<NW>(up_mask, (int)__umulhi(r.x, (uint32_t)n_up), lane);
      const int dn = select_kth_bit<NW>(dn_mask, (int)__umulhi(r.y, (uint32_t)n_dn), lane);
      flip_bit<NW>(s, up);
      flip_bit<NW>(s, dn);
    }
    if (lane == 0) {
      for (int w = 0; w < W; ++w) proposed[b * W + w] = s[w];
      u_acc[b] = u32_to_unit(r.z);
    }
  }
}

// graph_builders.py:74-89: accept iff (psi'/psi)^2 > u (strict; NaN rejects),
// in the log domain; accepted walkers take the proposed configuration and
// amplitude.
__global__ void accept_exchange_kernel(uint64_t* __restrict__ packed, const uint64_t* __restrict__ proposed,
                                       int64_t B, int W, float* __restrict__ logabs,
                                       float* __restrict__ sign, const float* __restrict__ logabs_new,
                                       const float* __restrict__ sign_new, const float* __restrict__ u_acc,
                                       unsigned long long* accept_count) {
  unsigned int mine = 0;
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B;
       b += (int64_t)gridDim.x * blockDim.x) {
    const float prob = expf(2.f * (logabs_new[b] - logabs[b]));
    bool changed = false;
    for (int w = 0; w < W; ++w) changed |= packed[b * W + w] != proposed[b * W + w];
    if (changed && prob > u_acc[b]) {
      for (int w = 0; w < W; ++w) packed[b * W + w] = proposed[b * W + w];
      logabs[b] = logabs_new[b];
      if (sign != nullptr) sign[b] = sign_new[b];
      ++mine;
    }
  }
  mine = (unsigned int)warp_sum((float)mine);
  if ((threadIdx.x & 31) == 0 && mine && accept_count != nullptr)
    atomicAdd(accept_count, (unsigned long long)mine);
}

// operators.py:165-169, 241-259 from amplitudes: one warp per walker, lanes
// stride over the bonds.  flipped_* are [B, n_bonds]; entries of parallel
// bonds are ignored (their mask is zero in the reference).
__global__ void eloc_from_amps_kernel(const int2* __restrict__ ij, const float* __restrict__ jx,
                                      const float* __restrict__ jz, int n_bonds,
                                      const uint64_t* __restrict__ packed, int64_t B, int W,
                                      const float* __restrict__ logabs, const float* __restrict__ sign,
                                      const float* __restrict__ flipped_logabs,
                                      const float* __restrict__ flipped_sign, float* __restrict__ e_loc,
                                      float* __restrict__ diag_out, float* __restrict__ off_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp; b < B; b += n_warps) {
    const float la = logabs[b], sg = sign != nullptr ? sign[b] : 1.f;
    float diag = 0.f, off = 0.f;
    for (int k = lane; k < n_bonds; k += 32) {
      const int2 bd = ij[k];
      const uint64_t wi = packed[b * W + (bd.x >> 6)], wj = packed[b * W + (bd.y >> 6)];
      const bool anti = (((wi >> (bd.x & 63)) ^ (wj >> (bd.y & 63))) & 1ull) != 0;
      diag += (anti ? -0.25f : 0.25f) * jz[k];
      if (anti) {
        const int64_t e = b * n_bonds + k;
        const float sf = flipped_sign != nullptr ? flipped_sign[e] : 1.f;
        off += 0.5f * jx[k] * sf * sg * expf(flipped_logabs[e] - la);
      }
    }
    diag = warp_sum(diag);
    off = warp_sum(off);
    if (lane == 0) {
      if (e_loc != nullptr) e_loc[b] = diag + off;
      if (diag_out != nullptr) diag_out[b] = diag;
      if (off_out != nullptr) off_out[b] = off;
    }
  }
}

// The summands of eloc_from_amps_kernel kept per bond: values[b, k] (same
// layout as flipped_*); the ratio is not read where jx_k == 0.
__global__ void bond_values_from_amps_kernel(const int2* __restrict__ ij, const float* __restrict__ jx,
                                             const float* __restrict__ jz, int n_bonds,
                                             const uint64_t* __restrict__ packed, int64_t B, int W,
                                             const float* __restrict__ logabs, const float* __restrict__ sign,
                                             const float* __restrict__ flipped_logabs,
                                             const float* __restrict__ flipped_sign, float* __restrict__ values) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp; b < B; b += n_warps) {
    const float la = logabs[b], sg = sign != nullptr ? sign[b] : 1.f;
    for (int k = lane; k < n_bonds; k += 32) {
      const int2 bd = ij[k];
      const uint64_t wi = packed[b * W + (bd.x >> 6)], wj = packed[b * W + (bd.y >> 6)];
      const bool anti = (((wi >> (bd.x & 63)) ^ (wj >> (bd.y & 63))) & 1ull) != 0;
      const int64_t e = b * n_bonds + k;
      float v = (anti ? -0.25f : 0.25f) * jz[k];
      if (anti && jx[k] != 0.f) {
        const float sf = flipped_sign != nullptr ? flipped_sign[e] : 1.f;
        v += 0.5f * jx[k] * sf * sg * expf(flipped_logabs[e] - la);
      }
      values[e] = v;
    }
  }
}

// Replica swap, one thread per (pair, region): sigma1 = row p, sigma2 = row
// P + p, D = (sigma1 ^ sigma2) & region & valid sites.  swapped[p, r] =
// (sigma1 ^ D, sigma2 ^ D), uint64 [P, R, 2, W].
__global__ void swap_configs_kernel(const uint64_t* __restrict__ packed, int64_t P, int N, int W,
                                    const uint64_t* __restrict__ regions, int n_regions,
                                    uint64_t* __restrict__ swapped) {
  const int64_t total = P * n_regions;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = e / n_regions;
    const int r = (int)(e - p * n_regions);
    for (int w = 0; w < W; ++w) {
      const uint64_t s1 = packed[p * W + w], s2 = packed[(P + p) * W + w];
      const uint64_t d = (s1 ^ s2) & regions[(int64_t)r * W + w] & valid_mask_word(N, w);
      swapped[(e * 2) * W + w] = s1 ^ d;
      swapped[(e * 2 + 1) * W + w] = s2 ^ d;
    }
  }
}

// values[p, r] from the amplitudes of the pair (logabs / sign [2P]) and of the
// swapped pair of swap_configs_kernel (swapped_* [P, R, 2]): 0 when the
// replicas hold different numbers of up spins in the region, exactly 1 when D
// is empty or holds every differing site, else
// sign products * exp((l1' - l1) + (l2' - l2)).  Sign arrays may be NULL (+1).
__global__ void swap_values_from_amps_kernel(const uint64_t* __restrict__ packed, int64_t P, int N, int W,
                                             const uint64_t* __restrict__ regions, int n_regions,
                                             const float* __restrict__ logabs, const float* __restrict__ sign,
                                             const float* __restrict__ swapped_logabs,
                                             const float* __restrict__ swapped_sign, float* __restrict__ values) {
  const int64_t total = P * n_regions;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = e / n_regions;
    const int r = (int)(e - p * n_regions);
    int up1 = 0, up2 = 0;
    bool empty = true, whole = true;
    for (int w = 0; w < W; ++w) {
      const uint64_t valid = valid_mask_word(N, w);
      const uint64_t s1 = packed[p * W + w], s2 = packed[(P + p) * W + w];
      const uint64_t m = regions[(int64_t)r * W + w] & valid;
      const uint64_t diff = s1 ^ s2, d = diff & m;
      up1 += __popcll(s1 & m);
      up2 += __popcll(s2 & m);
      empty = empty && d == 0ull;
      whole = whole && d == (diff & valid);
    }
    float v;
    if (up1 != up2) {
      v = 0.f;
    } else if (empty || whole) {
      v = 1.f;
    } else {
      float sg = 1.f;
      if (sign != nullptr) sg = sign[p] * sign[P + p];
      if (swapped_sign != nullptr) sg *= swapped_sign[2 * e] * swapped_sign[2 * e + 1];
      v = sg * expf((swapped_logabs[2 * e] - logabs[p]) + (swapped_logabs[2 * e + 1] - logabs[P + p]));
    }
    values[e] = v;
  }
}

// SupervisedWavefunctionOptimizer (training.py:166-175): per walker
//   r_b = sign sign_t exp(z_t + log_norm - z)   (= psi_target sqrt(2^N) / psi)
//   loss  += sum_b (1 - r_b)^2                  (mean_b (psi - t)^2 / sg(psi)^2 times the batch size)
//   w_b    = 2 (1 - r_b) / total                (d loss / d log psi_b)
// acc (double [2]) += { sum (1 - r)^2, B }.
__global__ void swo_weights_kernel(const float* __restrict__ z, const float* __restrict__ sign,
                                   const float* __restrict__ zt, const float* __restrict__ sign_t,
                                   int64_t B, float log_norm, float inv_total,
                                   float* __restrict__ weights, double* acc) {
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < B;
       i += (int64_t)gridDim.x * blockDim.x) {
    float r = expf(zt[i] + log_norm - z[i]);
    if (sign != nullptr) r *= sign[i];
    if (sign_t != nullptr) r *= sign_t[i];
    const float d = 1.0f - r;
    weights[i] = 2.0f * d * inv_total;
    s += (double)d * (double)d;
  }
  s = warp_sum(s);
  __shared__ double sh[kThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) sh[warp] = s;
  __syncthreads();
  if (warp == 0) {
    s = lane < kThreads / 32 ? sh[lane] : 0.0;
    s = warp_sum(s);
    if (lane == 0 && acc != nullptr) {
      atomicAdd(&acc[0], s);
      if (blockIdx.x == 0) atomicAdd(&acc[1], (double)B);
    }
  }
}

// tf.train.AdamOptimizer step (training.py:76-91, beta1 = 0.9, eps = 1e-8):
//   m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2
//   theta -= lr sqrt(1 - b2^t) / (1 - b1^t) m / (sqrt(v) + eps)
// The gradient is either `grad[i]` or formed on the fly from the estimator
// sums of EnergyGradientOptimizer (training.py:562-564):
//   g = (S[1][i] - (stats[0] / stats[2]) S[0][i]) * inv_nb.
// lr / t come from device scalars when given (CUDA-graph replays).
__device__ __forceinline__ float adam_lr_t(float lr, float b1, float b2, uint64_t t) {
  const double td = (double)t;
  return (float)((double)lr * sqrt(1.0 - pow((double)b2, td)) / (1.0 - pow((double)b1, td)));
}

// g = (S[1][i] - mean_e S[0][i]) * inv_nb in the rounding order both kernels share
__device__ __forceinline__ float energy_gradient(float so, float seo, float mean_e, float inv_nb) {
  return __fsub_rn(__fmul_rn(seo, inv_nb), __fmul_rn(mean_e, __fmul_rn(so, inv_nb)));
}

__device__ __forceinline__ void adam_update(float* __restrict__ params, float* __restrict__ m,
                                            float* __restrict__ v, int64_t i, float g, float lr_t, float b1,
                                            float b2, float eps) {
  const float mi = __fadd_rn(__fmul_rn(b1, m[i]), __fmul_rn(1.0f - b1, g));
  const float vi = __fadd_rn(__fmul_rn(b2, v[i]), __fmul_rn(__fmul_rn(1.0f - b2, g), g));
  m[i] = mi;
  v[i] = vi;
  params[i] = __fsub_rn(params[i], __fdiv_rn(__fmul_rn(lr_t, mi), __fadd_rn(sqrtf(vi), eps)));
}

__global__ void adam_kernel(float* __restrict__ params, float* __restrict__ m, float* __restrict__ v,
                            int64_t n, const float* __restrict__ grad, const float* __restrict__ sums,
                            const double* __restrict__ stats, float inv_nb, float lr,
                            const float* __restrict__ lr_dev, float b1, float b2, float eps,
                            uint64_t t, const uint64_t* __restrict__ t_dev) {
  if (lr_dev != nullptr) lr = *lr_dev;
  if (t_dev != nullptr) t = *t_dev + 1;
  const float lr_t = adam_lr_t(lr, b1, b2, t);
  const float mean_e = stats != nullptr ? (float)(stats[0] / stats[2]) : 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float g = sums != nullptr ? energy_gradient(sums[i], sums[n + i], mean_e, inv_nb) : grad[i];
    adam_update(params, m, v, i, g, lr_t, b1, b2, eps);
  }
}

// End of an EnergyGradientOptimizer epoch (training.py:618-622) in one kernel:
// apply_gradients (the Adam step above on the energy gradient of the TOTALS --
// float32 sums [2][n] + double stats [4], or the all-reduced float64 payload
// [2 n + 4] itself), metrics (the totals' statistics written to stats_out,
// which may be mapped host memory) and reset_gradients (the local
// accumulators, and the float32 totals when they are separate buffers, are
// zeroed by the thread that consumed the entry; the statistics by the last
// block to finish -- every block has read them by then).
template <typename TS>
__global__ void epoch_end_kernel(float* __restrict__ params, float* __restrict__ m, float* __restrict__ v,
                                 int64_t n, const TS* __restrict__ tot_sums, const double* __restrict__ tot_stats,
                                 float* __restrict__ zero_a, float* __restrict__ zero_b,
                                 double* __restrict__ zero_stats_a, double* __restrict__ zero_stats_b,
                                 float inv_nb, float lr, float b1, float b2, float eps, uint64_t t,
                                 double* stats_out, unsigned int* ticket) {
  const float lr_t = adam_lr_t(lr, b1, b2, t);
  const double s0 = tot_stats[0], s1 = tot_stats[1], s2 = tot_stats[2], s3 = tot_stats[3];
  const float mean_e = (float)(s0 / s2);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float g = energy_gradient((float)tot_sums[i], (float)tot_sums[n + i], mean_e, inv_nb);
    adam_update(params, m, v, i, g, lr_t, b1, b2, eps);
    if (zero_a != nullptr) { zero_a[i] = 0.f; zero_a[n + i] = 0.f; }
    if (zero_b != nullptr) { zero_b[i] = 0.f; zero_b[n + i] = 0.f; }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(ticket, 1u);
    if (done == gridDim.x - 1) {
      if (stats_out != nullptr) {
        volatile double* o = stats_out;
        o[0] = s0; o[1] = s1; o[2] = s2; o[3] = s3;
        __threadfence_system();
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (zero_stats_a != nullptr) zero_stats_a[k] = 0.0;
        if (zero_stats_b != nullptr) zero_stats_b[k] = 0.0;
      }
      *ticket = 0u;
    }
  }
}

// One periodic convolution layer on its own (layers.py:24-160: Conv1dPeriodic /
// Conv2dPeriodic = wrap padding + snt.Conv with padding VALID, stride 1):
//   out[b, x, y, co] = bias[co] + sum_{dx, dy, ci} in[b, (x + dx - pad_x) mod X, (y + dy - pad_y) mod Y, ci]
//                                                  * w[dx, dy, ci, co]
// NHWC, w as [kx, ky, C_in, C_out] (Sonnet's layout).  One thread per output
// element with the output channel fastest: coalesced stores and weight reads,
// the input value of a (position, tap, ci) is a broadcast within the channel
// group.  The ansatz kernels fuse this into whole networks; this entry exists
// so that the layer is callable by itself like the reference's module.
__global__ void conv_periodic_kernel(const float* __restrict__ in, int64_t B, int X, int Y, int Cin, int Cout,
                                     int kx, int ky, int pad_x, int pad_y, const float* __restrict__ w,
                                     const float* __restrict__ bias, float* __restrict__ out) {
  const int64_t total = B * X * Y * Cout;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(e % Cout);
    int64_t r = e / Cout;
    const int y = (int)(r % Y); r /= Y;
    const int x = (int)(r % X);
    const int64_t b = r / X;
    float acc = bias != nullptr ? bias[co] : 0.f;
    for (int dx = 0; dx < kx; ++dx) {
      int sx = (x + dx - pad_x) % X;
      if (sx < 0) sx += X;
      for (int dy = 0; dy < ky; ++dy) {
        int sy = (y + dy - pad_y) % Y;
        if (sy < 0) sy += Y;
        const float* src = in + ((b * X + sx) * Y + sy) * Cin;
        const float* wt = w + ((size_t)(dx * ky + dy) * Cin) * Cout + co;
        for (int ci = 0; ci < Cin; ++ci) acc = fmaf(src[ci], wt[(size_t)ci * Cout], acc);
      }
    }
    out[e] = acc;
  }
}

int blocks_for(int64_t work_items, int per_block) {
  const int64_t need = (work_items + per_block - 1) / per_block;
  return (int)std::max<int64_t>(1, std::min<int64_t>(need, 148 * 16));
}

}  // namespace

int launch_pack(const float* configs, int64_t B, int N, uint64_t* packed, cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  const int W = n_words(N);
  pack_kernel<<<blocks_for(B * W, kThreads / 32), kThreads, 0, s>>>(configs, B, N, W, packed);
  return cuda_fail(cudaGetLastError(), "pack launch");
}

int launch_unpack(const uint64_t* packed, int64_t B, int N, float* configs, cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  unpack_kernel<<<blocks_for(B * N, kThreads), kThreads, 0, s>>>(packed, B, N, n_words(N), configs);
  return cuda_fail(cudaGetLastError(), "unpack launch");
}

int launch_random_configs(uint64_t* packed, int64_t B, int N, uint64_t seed, uint64_t walker0,
                          cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  random_configs_kernel<<<blocks_for(B, kThreads), kThreads, 0, s>>>(packed, B, N, n_words(N), seed,
                                                                     walker0);
  return cuda_fail(cudaGetLastError(), "random_configs launch");
}

int launch_flip_enum(const cgsvmc_ham* h, const uint64_t* packed, int64_t B, uint64_t* flipped,
                     uint32_t* mask, cudaStream_t s) {
  if (B == 0 || h->n_bonds == 0) return CGSVMC_OK;
  const int mask_words = (h->n_bonds + 31) / 32;
  flip_enum_kernel<<<blocks_for(B * mask_words, kThreads / 32), kThreads, 0, s>>>(
      h->ij, h->n_bonds, packed, B, n_words(h->n_sites), flipped, mask);
  return cuda_fail(cudaGetLastError(), "flip_enum launch");
}

__global__ void fill_kernel(float* __restrict__ dst, int64_t n, float value) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n;
       e += (int64_t)gridDim.x * blockDim.x) dst[e] = value;
}

__global__ void advance_counter_kernel(uint64_t* counter, uint64_t by) { *counter += by; }

int launch_advance_counter(uint64_t* counter, uint64_t by, cudaStream_t s) {
  advance_counter_kernel<<<1, 1, 0, s>>>(counter, by);
  return cuda_fail(cudaGetLastError(), "advance_counter launch");
}

int launch_fill(float* dst, int64_t n, float value, cudaStream_t s) {
  if (n <= 0) return CGSVMC_OK;
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 1024);
  fill_kernel<<<blocks, 256, 0, s>>>(dst, n, value);
  return cuda_fail(cudaGetLastError(), "fill launch");
}

int launch_energy_stats(const float* e, int64_t B, double* stats, cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  energy_stats_kernel<<<blocks_for(B, kThreads * 8), kThreads, 0, s>>>(e, B, stats);
  return cuda_fail(cudaGetLastError(), "energy_stats launch");
}

int launch_swo_weights(const float* z, const float* sign, const float* zt, const float* sign_t, int64_t B,
                       float log_norm, float inv_total, float* weights, double* acc, cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  swo_weights_kernel<<<blocks_for(B, kThreads * 4), kThreads, 0, s>>>(z, sign, zt, sign_t, B, log_norm,
                                                                     inv_total, weights, acc);
  return cuda_fail(cudaGetLastError(), "swo_weights launch");
}

int launch_adam(float* params, float* m, float* v, int64_t n, const float* grad, const float* sums,
                const double* stats, float inv_nb, float lr, const float* lr_dev, float b1, float b2,
                float eps, uint64_t t, const uint64_t* t_dev, cudaStream_t s) {
  if (n == 0) return CGSVMC_OK;
  adam_kernel<<<blocks_for(n, kThreads), kThreads, 0, s>>>(params, m, v, n, grad, sums, stats, inv_nb, lr,
                                                          lr_dev, b1, b2, eps, t, t_dev);
  return cuda_fail(cudaGetLastError(), "adam launch");
}

int launch_epoch_end(float* params, float* m, float* v, int64_t n, const float* tot_sums,
                     const double* tot_payload, const double* tot_stats, float* zero_a, float* zero_b,
                     double* zero_stats_a, double* zero_stats_b, float inv_nb, float lr, float b1, float b2,
                     float eps, uint64_t t, double* stats_out, unsigned int* ticket, cudaStream_t s) {
  if (n == 0) return CGSVMC_OK;
  const int blocks = blocks_for(n, kThreads);
  if (tot_payload != nullptr)
    epoch_end_kernel<double><<<blocks, kThreads, 0, s>>>(params, m, v, n, tot_payload, tot_payload + 2 * n,
                                                         zero_a, zero_b, zero_stats_a, zero_stats_b, inv_nb, lr,
                                                         b1, b2, eps, t, stats_out, ticket);
  else
    epoch_end_kernel<float><<<blocks, kThreads, 0, s>>>(params, m, v, n, tot_sums, tot_stats, zero_a, zero_b,
                                                        zero_stats_a, zero_stats_b, inv_nb, lr, b1, b2, eps, t,
                                                        stats_out, ticket);
  return cuda_fail(cudaGetLastError(), "epoch_end launch");
}

int launch_conv_periodic(const float* in, int64_t B, int X, int Y, int Cin, int Cout, int kx, int ky, int pad_x,
                         int pad_y, const float* w, const float* bias, float* out, cudaStream_t s) {
  const int64_t total = B * X * Y * Cout;
  if (total == 0) return CGSVMC_OK;
  conv_periodic_kernel<<<blocks_for(total, kThreads), kThreads, 0, s>>>(in, B, X, Y, Cin, Cout, kx, ky, pad_x, pad_y,
                                                                        w, bias, out);
  return cuda_fail(cudaGetLastError(), "conv_periodic launch");
}

int launch_reduce_partials(const float* partials, int n_parts, int64_t n, float* out,
                           cudaStream_t s) {
  reduce_partials_kernel<<<blocks_for(n, 32), kThreads, 0, s>>>(partials, n_parts, n, out);
  return cuda_fail(cudaGetLastError(), "reduce_partials launch");
}

int launch_propose_exchange(const uint64_t* packed, int64_t B, int N, uint64_t seed, uint64_t walker0,
                            uint64_t step, uint64_t* proposed, float* u_acc, cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  const int W = n_words(N);
  const int blocks = blocks_for(B, kThreads / 32);
  if (W == 1) propose_exchange_kernel<1><<<blocks, kThreads, 0, s>>>(packed, B, N, W, seed, walker0, step, proposed, u_acc);
  else if (W == 2) propose_exchange_kernel<2><<<blocks, kThreads, 0, s>>>(packed, B, N, W, seed, walker0, step, proposed, u_acc);
  else propose_exchange_kernel<4><<<blocks, kThreads, 0, s>>>(packed, B, N, W, seed, walker0, step, proposed, u_acc);
  return cuda_fail(cudaGetLastError(), "propose_exchange launch");
}

int launch_accept_exchange(uint64_t* packed, const uint64_t* proposed, int64_t B, int N, float* logabs,
                           float* sign, const float* logabs_new, const float* sign_new,
                           const float* u_acc, unsigned long long* accept_count, cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  accept_exchange_kernel<<<blocks_for(B, kThreads), kThreads, 0, s>>>(
      packed, proposed, B, n_words(N), logabs, sign, logabs_new, sign_new, u_acc, accept_count);
  return cuda_fail(cudaGetLastError(), "accept_exchange launch");
}

int launch_eloc_from_amps(const cgsvmc_ham* h, const uint64_t* packed, int64_t B, const float* logabs,
                          const float* sign, const float* flipped_logabs, const float* flipped_sign,
                          float* e_loc, float* diag, float* off, cudaStream_t s) {
  if (B == 0) return CGSVMC_OK;
  eloc_from_amps_kernel<<<blocks_for(B, kThreads / 32), kThreads, 0, s>>>(
      h->ij, h->jx, h->jz, h->n_bonds, packed, B, n_words(h->n_sites), logabs, sign, flipped_logabs,
      flipped_sign, e_loc, diag, off);
  return cuda_fail(cudaGetLastError(), "eloc_from_amps launch");
}

int launch_bond_values_from_amps(const cgsvmc_ham* h, const uint64_t* packed, int64_t B, const float* logabs,
                                 const float* sign, const float* flipped_logabs, const float* flipped_sign,
                                 float* values, cudaStream_t s) {
  if (B == 0 || h->n_bonds == 0) return CGSVMC_OK;
  bond_values_from_amps_kernel<<<blocks_for(B, kThreads / 32), kThreads, 0, s>>>(
      h->ij, h->jx, h->jz, h->n_bonds, packed, B, n_words(h->n_sites), logabs, sign, flipped_logabs,
      flipped_sign, values);
  return cuda_fail(cudaGetLastError(), "bond_values_from_amps launch");
}

int launch_swap_configs(const uint64_t* packed, int64_t P, int N, const uint64_t* regions, int n_regions,
                        uint64_t* swapped, cudaStream_t s) {
  if (P == 0 || n_regions == 0) return CGSVMC_OK;
  swap_configs_kernel<<<blocks_for(P * n_regions, kThreads), kThreads, 0, s>>>(
      packed, P, N, n_words(N), regions, n_regions, swapped);
  return cuda_fail(cudaGetLastError(), "swap_configs launch");
}

int launch_swap_values_from_amps(const uint64_t* packed, int64_t P, int N, const uint64_t* regions,
                                 int n_regions, const float* logabs, const float* sign,
                                 const float* swapped_logabs, const float* swapped_sign, float* values,
                                 cudaStream_t s) {
  if (P == 0 || n_regions == 0) return CGSVMC_OK;
  swap_values_from_amps_kernel<<<blocks_for(P * n_regions, kThreads), kThreads, 0, s>>>(
      packed, P, N, n_words(N), regions, n_regions, logabs, sign, swapped_logabs, swapped_sign, values);
  return cuda_fail(cudaGetLastError(), "swap_values_from_amps launch");
}

}  // namespace cgsvmc
