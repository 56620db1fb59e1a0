// Pure-RBM fast path, host side: parameter-image build, launch planning,
// deterministic cross-CTA reduction.  Kernels: rbm2_impl.cuh.
#include <algorithm>
#include <cstdlib>

#include "rbm2_impl.cuh"

namespace cgsvmc {
namespace rbm2 {
namespace {

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// One block per site (rows of the tables + row sums), then one block per 128
// hidden units (column sums), one block for the select table and one for max |W|.
__global__ void __launch_bounds__(128)
prep_kernel(Image im, const float* __restrict__ a, const float* __restrict__ a0,
            const float* __restrict__ W, const float* __restrict__ c, float* __restrict__ img) {
  __shared__ float red[4];
  const int tid = threadIdx.x;
  if ((int)blockIdx.x < im.N) {
    const int i = blockIdx.x;
    float rs = 0.f;
    for (int j = tid; j < im.HP; j += 128) {
      const float w = j < im.H ? W[(size_t)i * im.H + j] : 0.f;
      img[im.off_w2 + (size_t)i * im.HP + j] = 2.f * w;
      img[im.off_f + (size_t)i * im.HP + j] = expf(4.f * w);
      img[im.off_g + (size_t)i * im.HP + j] = expf(-4.f * w);
      rs += w;
    }
    rs = warp_sum(rs);
    if ((tid & 31) == 0) red[tid >> 5] = rs;
    __syncthreads();
    if (tid == 0) {
      const float total = (red[0] + red[1]) + (red[2] + red[3]);
      img[im.off_a2 + i] = 2.885390081777927f * (a[i] - total);
      img[im.off_a + i] = a[i];
    }
  } else if (blockIdx.x == gridDim.x - 2) {
    uint8_t* lut = reinterpret_cast<uint8_t*>(img + im.off_lut);
    for (int e = tid; e < 2048; e += 128) lut[e] = lut_entry(e);
  } else if (blockIdx.x == gridDim.x - 1) {
    // max |W|: bounds the growth of the sampler's unnormalised state
    float mx = 0.f;
    for (int e = tid; e < im.N * im.H; e += 128) mx = fmaxf(mx, fabsf(W[e]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(CGSVMC_FULL_MASK, mx, o));
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    if (tid == 0) {
      img[im.off_a0 + 1] = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
      img[im.off_a0 + 2] = 0.f;
      img[im.off_a0 + 3] = 0.f;
    }
  } else {
    const int j = ((int)blockIdx.x - im.N) * 128 + tid;
    if (j < im.HP) {
      float cs = 0.f;
      if (j < im.H)
        for (int i = 0; i < im.N; ++i) cs += W[(size_t)i * im.H + j];
      img[im.off_base + j] = (j < im.H ? c[j] : 0.f) - cs;
    }
    if ((int)blockIdx.x == im.N) {
      if (tid == 0) img[im.off_a0] = a0[0];
      for (int i = im.N + tid; i < im.NP; i += 128) { img[im.off_a2 + i] = 0.f; img[im.off_a + i] = 0.f; }
    }
  }
}

// out[f] += sum_c partials[c][f] in a fixed order: 32 outputs x 8 CTA slices
// per block (the partials were just written and sit in L2); every thread has
// all of its loads in flight before the first add.  Also folds the per-CTA
// energy sums into stats and, when asked, advances the device-side Philox
// step counter of a captured batch step (the producer kernel has read it).
__global__ void __launch_bounds__(256)
reduce_kernel(const float* __restrict__ partials, int n_cta, int64_t stride, int64_t n_out,
              float* __restrict__ out, const double* __restrict__ stat_partials, int64_t B,
              double* __restrict__ stats, uint64_t* counter, uint64_t advance, double* stats_snapshot) {
  __shared__ float sm[8][32];
  constexpr int U = 19;                       // 8 x 19 = 152 >= 148 CTAs in one sweep
  const int col = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int64_t f = (int64_t)blockIdx.x * 32 + col;
  float s = 0.f;
  if (f < n_out) {
    const float* src = partials + f;
    for (int c0 = slice; c0 < n_cta; c0 += 8 * U) {
      float v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = c0 + 8 * u;
        v[u] = c < n_cta ? __ldcg(src + (size_t)c * stride) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) s += v[u];
    }
  }
  sm[slice][col] = s;
  __syncthreads();
  if (slice == 0 && f < n_out)
    out[f] += ((sm[0][col] + sm[1][col]) + (sm[2][col] + sm[3][col])) +
              ((sm[4][col] + sm[5][col]) + (sm[6][col] + sm[7][col]));
  if (blockIdx.x == 0 && threadIdx.x < 32 && stat_partials != nullptr) {
    double e = 0.0, e2 = 0.0;
    for (int c = threadIdx.x; c < n_cta; c += 32) { e += stat_partials[2 * c]; e2 += stat_partials[2 * c + 1]; }
    e = warp_sum(e);
    e2 = warp_sum(e2);
    if (threadIdx.x == 0) {
      const double s0 = stats[0] + e, s1 = stats[1] + e2, s2 = stats[2] + (double)B;
      stats[0] = s0; stats[1] = s1; stats[2] = s2;
      if (stats_snapshot != nullptr) {      // may be mapped host memory
        volatile double* snap = stats_snapshot;
        snap[0] = s0; snap[1] = s1; snap[2] = s2; snap[3] = stats[3];
        __threadfence_system();
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 32 && counter != nullptr) *counter += advance;
}

// Bond-pair table for the local energy: row 2 k + o holds F[d][j] * G[u][j] with
// d the raised and u the lowered site of bond k in orientation o (o = 0: the
// bond's first site is raised).  The same single-rounding product the two-row
// ratio loop forms on the fly.
__global__ void __launch_bounds__(128)
pair_prep_kernel(Image im, const float* __restrict__ img, const int2* __restrict__ bonds, int n_bonds,
                 float* __restrict__ pair) {
  const int r = blockIdx.x, k = r >> 1, o = r & 1;
  if (k >= n_bonds) return;
  const int2 b = bonds[k];
  const int d = o ? b.y : b.x, u = o ? b.x : b.y;
  for (int j = threadIdx.x; j < im.HP; j += 128)
    pair[(size_t)r * im.HP + j] = img[im.off_f + (size_t)d * im.HP + j] * img[im.off_g + (size_t)u * im.HP + j];
}

Image make_image(int N, int H, int HP) {
  Image im;
  im.N = N; im.H = H; im.HP = HP; im.NP = round_up(N, 4);
  im.words = n_words(N);
  im.off_w2 = 0;
  im.off_f = N * HP;
  im.off_g = 2 * N * HP;
  im.off_a2 = 3 * N * HP;
  im.off_base = im.off_a2 + im.NP;
  im.off_a = im.off_base + HP;
  im.off_a0 = im.off_a + im.NP;
  im.off_lut = im.off_a0 + 4;          // 2048 bytes: select-in-byte table
  im.total = im.off_lut + 512;
  return im;
}

size_t walker_smem_bytes(const Image& im, int slots, bool ws, bool do_eloc, int n_bonds, bool do_grad,
                         bool mc = false, bool pt = false) {
  const int NP4 = round_up(im.N + 1, 4);
  size_t b = ws ? (size_t)(im.total - (pt ? im.off_f : 0)) * 4 : 0;
  if (pt) b += (size_t)2 * n_bonds * im.HP * 4;
  b += 32;
  if (do_eloc) b += (size_t)n_bonds * 16 + (size_t)slots * round_up(n_bonds, 8) * 4;
  // T_s (tanh staging; with the pair table at least N rows: the parked 2W table) and ws_s
  b += (size_t)std::max(do_grad ? slots * im.HP : 0, pt ? im.N * im.HP : 0) * 4;
  if (do_grad) b += (size_t)slots * 2 * NP4 * 4;
  b += (size_t)slots * 4;
  if (mc && !ws) b += 2048;
  return b;
}

// Fills everything but the shared-memory decisions.
bool base_plan(const cgsvmc_ansatz* a, int64_t B, Plan* pl, bool walker) {
  const cgsvmc_ansatz_desc& d = a->desc;
  if (d.kind != CGSVMC_ANSATZ_RBM || d.num_layers != 0) return false;
  if (d.layer_size < 1 || d.layer_size > 256 || d.n_sites > CGSVMC_MAX_SITES) return false;
  const int H = d.layer_size;
  const int HP = round_up(H, 32);
  pl->kjv = HP / 32;
  // 8 lanes per walker (four walkers per warp) while the state fits 128
  // registers, else 16; measured on B200 at C2: 8 lanes 100 us / step, 16 lanes
  // 110 us (profiles/r01e_*).
  pl->lpw = pl->kjv <= 5 ? 8 : 16;
  pl->im = make_image(d.n_sites, H, HP);
  pl->nw = n_words(d.n_sites) == 3 ? 4 : n_words(d.n_sites);
  const int wpw = 32 / pl->lpw, slots = variant_slots(pl->lpw, pl->kjv, walker);
  pl->slots = slots;
  const int64_t per_sm = std::max<int64_t>(1, (B + a->num_sms - 1) / a->num_sms);
  const int64_t rounds = (per_sm + slots - 1) / slots;
  int64_t wpc = (per_sm + rounds - 1) / rounds;
  wpc = std::min<int64_t>(slots, (wpc + wpw - 1) / wpw * wpw);
  pl->wpc = (int)wpc;
  pl->n_batches = (B + wpc - 1) / wpc;
  pl->grid = (int)std::min<int64_t>(pl->n_batches, a->num_sms);
  return true;
}

int build_image(cgsvmc_ansatz* a, const Plan& pl, cudaStream_t st) {
  const size_t bytes = (size_t)pl.im.total * 4;
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
  }
  if (a->track_params && a->tables_valid) return CGSVMC_OK;
  const float* p = a->params;
  const int blocks = pl.im.N + (pl.im.HP + 127) / 128 + 2;
  prep_kernel<<<blocks, 128, 0, st>>>(pl.im, p + a->offsets[0], p + a->offsets[1], p + a->offsets[2],
                                      p + a->offsets[3], a->tables);
  a->tables_valid = true;
  for (auto& pt : a->pair_tables) pt.valid = false;
  return cuda_fail(cudaGetLastError(), "rbm2 prep launch");
}

// Whether pair_slot can give (ansatz, Hamiltonian) a slot of `bytes`: the
// Hamiltonian has one that large, or there is room for another.  Allocates nothing.
bool pair_slot_possible(const cgsvmc_ansatz* a, const cgsvmc_ham* h, size_t bytes) {
  for (const auto& pt : a->pair_tables)
    if (pt.ham_uid == h->uid) return pt.bytes >= bytes;
  return (int)a->pair_tables.size() < cgsvmc_ansatz::kMaxPairTables;
}

// The pair-table slot of (ansatz, Hamiltonian); nullptr when the ansatz has
// already been used with kMaxPairTables other Hamiltonians.
cgsvmc_ansatz::PairTable* pair_slot(cgsvmc_ansatz* a, const cgsvmc_ham* h, size_t bytes) {
  if (!pair_slot_possible(a, h, bytes)) return nullptr;
  for (auto& pt : a->pair_tables)
    if (pt.ham_uid == h->uid) return &pt;
  cgsvmc_ansatz::PairTable pt;
  pt.ham_uid = h->uid;
  if (cudaMalloc(&pt.buf, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  pt.bytes = bytes;
  a->pair_tables.push_back(pt);
  return &a->pair_tables.back();
}

// (Re)builds the bond-pair table of this Hamiltonian when the tables changed.
int build_pair_table(cgsvmc_ansatz* a, const cgsvmc_ham* h, const Plan& pl,
                     cgsvmc_ansatz::PairTable* slot, cudaStream_t st) {
  if (slot->valid) return CGSVMC_OK;
  pair_prep_kernel<<<2 * h->n_bonds, 128, 0, st>>>(pl.im, a->tables, h->ij, h->n_bonds, slot->buf);
  slot->valid = true;
  return cuda_fail(cudaGetLastError(), "rbm2 pair prep launch");
}

// Launch plan of the sampler kernel (rbm2_mc_steps).
int plan_mc(const cgsvmc_ansatz* a, int64_t B, Plan* pl) {
  if (!base_plan(a, B, pl, false)) { set_error("rbm2: unsupported ansatz"); return CGSVMC_ERR_UNSUPPORTED; }
  const size_t img_bytes = (size_t)pl->im.total * 4;
  pl->ws = img_bytes + 16 <= (size_t)a->max_smem_optin;
  pl->pt = pl->pt_global = pl->tc_grad = pl->fuse = false;
  pl->mc_smem = (pl->ws ? img_bytes : 2048) + 16;
  pl->walker_smem = 0;
  pl->step0_dev = nullptr;
  return CGSVMC_OK;
}

// Launch plan of the walker kernel (rbm2_walker): table placement, bond-pair
// table, tensor-core gradient and in-kernel reduction.  Depends only on the
// shape, the device, the pair-table slots the ansatz already holds and the
// environment switches; allocates and launches nothing, so that
// cgsvmc_rbm2_plan reports what a call would run.  `no_pair_table` plans the
// two-row path (the pair-table allocation failed).
int plan_walker(const cgsvmc_ansatz* a, const cgsvmc_ham* h, int64_t B, bool do_grad, bool weighted, bool mc,
                bool no_pair_table, Plan* pl) {
  if (!base_plan(a, B, pl, true)) { set_error("rbm2: unsupported ansatz"); return CGSVMC_ERR_UNSUPPORTED; }
  const bool do_eloc = h != nullptr;
  const int slots = pl->slots;
  const int nb = do_eloc ? h->n_bonds : 0;
  pl->ws = walker_smem_bytes(pl->im, slots, true, do_eloc, nb, do_grad, mc) <= (size_t)a->max_smem_optin;
  const bool pair_ok = !no_pair_table && do_eloc && nb >= 1 && nb < 16384 &&
                       pair_slot_possible(a, h, (size_t)2 * nb * pl->im.HP * 4);
  // bond-pair table: 8 lanes per walker, at least one bond, pair index below 2^15,
  // and everything (image from F on + pair table + staging) in shared memory
  pl->pt = pair_ok && pl->ws && pl->lpw == 8 &&
           walker_smem_bytes(pl->im, slots, true, do_eloc, nb, do_grad, mc, true) <= (size_t)a->max_smem_optin;
  // tables in global memory: the pair table too (read through L1 / L2)
  pl->pt_global = pair_ok && !pl->ws;
  pl->walker_smem = walker_smem_bytes(pl->im, slots, pl->ws, do_eloc, nb, do_grad, mc, pl->pt);
  pl->mc_smem = 0;
  pl->step0_dev = nullptr;
  if (pl->walker_smem > (size_t)a->max_smem_optin) {
    set_error("rbm2: problem does not fit in shared memory");
    return CGSVMC_ERR_UNSUPPORTED;
  }
  // gradient sums on the tensor cores: pair-table kernels with weights (1, E_loc),
  // sigma + three weight pieces within M = 128 rows (N <= 39), a spare column for
  // the constant 1 (H < HP), operand planes no larger than the float staging
  // buffers they replace.  CGSVMC_RBM2_TC_GRAD=0 keeps the FP32 register tiles.
  // (read at every call so that tests can compare the two paths)
  {
    const char* e = getenv("CGSVMC_RBM2_TC_GRAD");
    const bool off = e != nullptr && atoi(e) == 0;
    const int np4 = round_up(pl->im.N + 1, 4), np8 = round_up(pl->im.N + 1, 8);
    pl->tc_grad = !off && pl->pt && do_grad && !weighted && np8 == np4 && 3 * np8 <= 128 &&
                  pl->im.H < pl->im.HP && 3 * pl->im.HP <= 512 && (slots == 64 || slots == 128);
  }
  // The cross-CTA reduction runs inside the walker kernel when the device can
  // launch it cooperatively (all CTAs co-resident: grid <= number of SMs, one
  // CTA per SM) and the staging buffer is large enough for its scratch.
  // CGSVMC_RBM2_FUSED_REDUCE=0 keeps the separate reduction kernel.
  const char* fuse_env = getenv("CGSVMC_RBM2_FUSED_REDUCE");
  const bool fuse_off = fuse_env != nullptr && atoi(fuse_env) == 0;
  pl->fuse = false;
  if (do_grad && !fuse_off && pl->grid <= a->num_sms) {
    int coop = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, a->device);
    const int threads = variant_slots(pl->lpw, pl->kjv, true) / (32 / pl->lpw) * 32;
    pl->fuse = coop != 0 && (size_t)slots * pl->im.HP >= (size_t)(threads / 32) * 96;
  }
  return CGSVMC_OK;
}

}  // namespace
}  // namespace rbm2

using namespace rbm2;

bool rbm2_supported(const cgsvmc_ansatz* a, const cgsvmc_ham* h) {
  Plan pl;
  if (!base_plan(a, 1, &pl, true)) return false;
  const int slots = pl.slots;
  const int nb = h != nullptr ? h->n_bonds : 0;
  if (nb >= 32768) return false;      // list entries keep 15 bits of bond index
  // the largest launch (accumulate) must fit with the image left in global memory
  return walker_smem_bytes(pl.im, slots, false, h != nullptr, nb, true, true) <= (size_t)a->max_smem_optin;
}

int rbm2_mc_steps(cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int n_steps, uint64_t seed,
                  uint64_t walker0, uint64_t step0, unsigned long long* accept_count,
                  float* log_amp_out, cudaStream_t st) {
  Plan pl;
  if (int rc = plan_mc(a, B, &pl)) return rc;
  pl.step0_dev = a->step_counter_dev;
  if (int rc = build_image(a, pl, st)) return rc;
  switch (pl.nw) {
    case 1: return launch_mc_nw1(pl, a->tables, packed, B, n_steps, seed, walker0, step0, accept_count, log_amp_out, st);
    case 2: return launch_mc_nw2(pl, a->tables, packed, B, n_steps, seed, walker0, step0, accept_count, log_amp_out, st);
    default: return launch_mc_nw4(pl, a->tables, packed, B, n_steps, seed, walker0, step0, accept_count, log_amp_out, st);
  }
}

int rbm2_walker(cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                float* e_loc, float* log_amp, float* diag, float* off, bool do_grad,
                const float* weights, int K, float* out, double* stats, cudaStream_t st,
                const Rbm2Sweep* sweep) {
  const bool do_eloc = h != nullptr;
  const bool mc = sweep != nullptr;
  Plan pl;
  if (int rc = plan_walker(a, h, B, do_grad, weights != nullptr, mc, false, &pl)) return rc;
  const int nb = do_eloc ? h->n_bonds : 0;
  cgsvmc_ansatz::PairTable* slot =
      (pl.pt || pl.pt_global) ? pair_slot(a, h, (size_t)2 * nb * pl.im.HP * 4) : nullptr;
  if ((pl.pt || pl.pt_global) && slot == nullptr)      // the allocation failed: the two-row path
    if (int rc = plan_walker(a, h, B, do_grad, weights != nullptr, mc, true, &pl)) return rc;
  if (int rc = build_image(a, pl, st)) return rc;
  if (slot != nullptr)
    if (int rc = build_pair_table(a, h, pl, slot, st)) return rc;
  const int64_t P = a->n_params;
  WalkerArgs A;
  memset(&A, 0, sizeof(A));
  A.pair_table = slot != nullptr ? slot->buf : nullptr;
  A.packed = packed; A.B = B; A.wpc = pl.wpc; A.n_batches = pl.n_batches;
  A.do_eloc = do_eloc ? 1 : 0;
  if (do_eloc) { A.bonds_ij = h->ij; A.bonds_jx = h->jx; A.bonds_jz = h->jz; A.n_bonds = h->n_bonds; }
  A.e_loc = e_loc; A.log_amp = log_amp; A.diag = diag; A.off = off;
  A.do_grad = do_grad ? 1 : 0;
  A.weights = weights; A.K = K; A.P = P;
  if (mc) {
    A.packed_rw = const_cast<uint64_t*>(packed);
    A.n_steps = sweep->n_steps; A.seed = sweep->seed; A.walker0 = sweep->walker0;
    A.step0 = sweep->step0; A.step0_dev = a->step_counter_dev; A.accept_count = sweep->accept_count;
  }
  A.tc_grad = pl.tc_grad ? 1 : 0;
  if (mc) A.configs_f32 = sweep->configs_f32;
  const int n_iters = mc && sweep->n_iters > 1 ? sweep->n_iters : 1;
  A.n_iters = n_iters;
  A.out_stride = n_iters > 1 ? B : 0;
  const bool fuse = pl.fuse;
  if (fuse && a->grid_sync == nullptr) {
    if (int rc = cuda_fail(cudaMalloc(&a->grid_sync, 128), "grid_sync alloc")) return rc;
    if (int rc = cuda_fail(cudaMemset(a->grid_sync, 0, 128), "grid_sync clear")) return rc;
  }
  if (do_grad) {
    const size_t part_bytes = (size_t)pl.grid * 2 * P * sizeof(float);
    const size_t part_pad = (part_bytes + 15) / 16 * 16;
    if (int rc = ensure_scratch(a, part_pad + (size_t)pl.grid * 2 * sizeof(double))) return rc;
    A.partials = a->scratch;
    A.stat_partials = stats != nullptr
        ? reinterpret_cast<double*>(reinterpret_cast<char*>(a->scratch) + part_pad) : nullptr;
  }
  uint64_t* const step_counter = mc ? sweep->advance_counter : nullptr;
  double* const snapshot = mc ? sweep->stats_snapshot : nullptr;
  if (fuse) {
    A.fuse_reduce = 1;
    A.sync = a->grid_sync;
    A.out = out; A.n_out = (int64_t)K * P; A.stats = stats;
    A.counter = step_counter; A.advance = mc ? (uint64_t)sweep->n_steps * (uint64_t)n_iters : 0ull;
    A.stats_snapshot = snapshot;
  }
  int rc;
  switch (pl.nw) {
    case 1: rc = launch_walker_nw1(pl, a->tables, A, st); break;
    case 2: rc = launch_walker_nw2(pl, a->tables, A, st); break;
    default: rc = launch_walker_nw4(pl, a->tables, A, st); break;
  }
  if (rc) return rc;
  if (do_grad && !fuse) {
    const int64_t n_out = (int64_t)K * P;
    const int blocks = (int)((n_out + 31) / 32);
    reduce_kernel<<<blocks, 256, 0, st>>>(A.partials, pl.grid, 2 * P, n_out, out, A.stat_partials, B * n_iters, stats,
                                          step_counter, mc ? (uint64_t)sweep->n_steps * (uint64_t)n_iters : 0ull,
                                          snapshot);
    return cuda_fail(cudaGetLastError(), "rbm2 reduce launch");
  }
  return CGSVMC_OK;
}

int rbm2_plan(const cgsvmc_ansatz* a, const cgsvmc_ham* h, int64_t B, int mode, int32_t (&out)[kRbm2PlanFields]) {
  for (int32_t& v : out) v = 0;
  const bool sampler = mode == CGSVMC_RBM2_PLAN_MC_STEPS;
  const bool grad_only = mode == CGSVMC_RBM2_PLAN_WEIGHTED_GRAD_SUM;
  const cgsvmc_ham* hw = sampler || grad_only ? nullptr : h;
  if (!rbm2_supported(a, hw)) {
    set_error("rbm2: the call takes another path");
    return CGSVMC_ERR_UNSUPPORTED;
  }
  const bool mc = mode == CGSVMC_RBM2_PLAN_BATCH_STEPS;
  const bool do_grad = mc || grad_only || mode == CGSVMC_RBM2_PLAN_ACCUMULATE;
  Plan pl;
  const int rc = sampler ? plan_mc(a, B, &pl) : plan_walker(a, hw, B, do_grad, grad_only, mc, false, &pl);
  if (rc) return rc;
  out[0] = 1;
  out[1] = pl.nw;
  out[2] = pl.lpw;
  out[3] = pl.kjv;
  out[4] = pl.slots;
  out[5] = pl.wpc;
  out[6] = (int32_t)std::min<int64_t>(pl.n_batches, INT32_MAX);
  out[7] = pl.grid;
  out[8] = pl.ws ? 1 : 0;
  out[9] = pl.pt ? 1 : (pl.pt_global ? 2 : 0);
  out[10] = pl.tc_grad ? 1 : 0;
  out[11] = pl.fuse ? 1 : 0;
  // the walker kernel keeps a swept walker in registers for the next iteration
  // when every CTA has one batch
  out[12] = mc && pl.n_batches <= (int64_t)pl.grid ? 1 : 0;
  return CGSVMC_OK;
}

}  // namespace cgsvmc
