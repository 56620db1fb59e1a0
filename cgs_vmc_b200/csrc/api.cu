// extern "C" entry points of include/cgsvmc.h: argument checking, handle
// management and dispatch to the kernel launchers.
#include <cstdio>
#include <cstring>
#include <new>

#include <nvtx3/nvToolsExt.h>

#include "internal.h"

// NVTX ranges around the entry points (header-only nvtx3: a no-op function
// pointer check unless a profiler is attached), named after the kernel groups
// of SURVEY.md 2.2: K0 utility, K1 amplitudes, K2 sampler, K3 local energy,
// K4 weighted gradient sums, K5 statistics / loss.
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

namespace cgsvmc {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int cuda_fail(cudaError_t err, const char* what) {
  if (err == cudaSuccess) return CGSVMC_OK;
  g_last_error = std::string(what) + ": " + cudaGetErrorString(err);
  return CGSVMC_ERR_CUDA;
}

int ensure_scratch(cgsvmc_ansatz* a, size_t bytes) {
  if (bytes <= a->scratch_bytes) return CGSVMC_OK;
  if (a->scratch != nullptr) {
    // earlier launches -- and captured graphs -- may still use the old buffer
    a->retired.push_back(a->scratch);
    a->scratch = nullptr;
    a->scratch_bytes = 0;
  }
  if (int rc = cuda_fail(cudaMalloc(&a->scratch, bytes), "scratch alloc")) return rc;
  a->scratch_bytes = bytes;
  return CGSVMC_OK;
}

namespace {

int invalid(const char* msg) {
  set_error(msg);
  return CGSVMC_ERR_INVALID;
}

// Tensor sizes of the flat parameter layout (see cgsvmc.h).
bool layout(const cgsvmc_ansatz_desc& d, std::vector<int64_t>* sizes) {
  sizes->clear();
  const int64_t N = d.n_sites;
  switch (d.kind) {
    case CGSVMC_ANSATZ_FULLY_CONNECTED: {
      int64_t n_in = N;
      for (int l = 0; l < d.num_layers; ++l) {
        sizes->push_back(n_in * d.layer_size);
        sizes->push_back(d.layer_size);
        n_in = d.layer_size;
      }
      sizes->push_back(n_in);
      sizes->push_back(1);
      return true;
    }
    case CGSVMC_ANSATZ_RBM: {
      sizes->push_back(N);
      sizes->push_back(1);
      int64_t n_in = N;
      for (int l = 0; l < d.num_layers; ++l) {
        sizes->push_back(n_in * d.layer_size);
        sizes->push_back(d.layer_size);
        n_in = d.layer_size;
      }
      sizes->push_back(n_in * d.layer_size);
      sizes->push_back(d.layer_size);
      return true;
    }
    case CGSVMC_ANSATZ_CONV_1D:
    case CGSVMC_ANSATZ_CONV_2D: {
      int64_t c_in = 1;
      const int64_t taps = d.kind == CGSVMC_ANSATZ_CONV_1D ? d.kernel_size
                                                           : (int64_t)d.kernel_size * d.kernel_size;
      for (int l = 0; l < d.num_layers; ++l) {
        sizes->push_back(taps * c_in * d.num_filters);
        sizes->push_back(d.num_filters);
        c_in = d.num_filters;
      }
      return true;
    }
    case CGSVMC_ANSATZ_RESNET_1D:
    case CGSVMC_ANSATZ_RESNET_2D: {
      const int64_t taps = d.kind == CGSVMC_ANSATZ_RESNET_1D ? d.kernel_size
                                                             : (int64_t)d.kernel_size * d.kernel_size;
      const int64_t f = d.num_filters;
      sizes->push_back(taps * f);
      sizes->push_back(f);
      for (int l = 0; l < 2 * d.num_layers; ++l) {
        sizes->push_back(taps * f * f);
        sizes->push_back(f);
      }
      return true;
    }
    default:
      return false;
  }
}

int check_ready(const cgsvmc_ansatz* a) {
  if (a == nullptr) return invalid("ansatz handle is NULL");
  if (a->params == nullptr) return invalid("no parameters bound: call cgsvmc_ansatz_bind_params first");
  return CGSVMC_OK;
}

}  // namespace
}  // namespace cgsvmc

using namespace cgsvmc;

extern "C" {

int cgsvmc_version(void) { return CGSVMC_VERSION; }

const char* cgsvmc_last_error(void) { return g_last_error.c_str(); }

int cgsvmc_ansatz_create(const cgsvmc_ansatz_desc* desc, cgsvmc_ansatz** out) {
  if (desc == nullptr || out == nullptr) return invalid("ansatz_create: NULL argument");
  *out = nullptr;
  const cgsvmc_ansatz_desc& d = *desc;
  std::vector<int64_t> sizes;
  if (!layout(d, &sizes)) return invalid("Provided wavefunction_type is not registered.");
  if (d.n_sites < 2 || d.n_sites > CGSVMC_MAX_SITES)
    return invalid("ansatz_create: n_sites must be in [2, 256]");
  if (d.num_layers < 0) return invalid("ansatz_create: num_layers < 0");
  if (d.kind == CGSVMC_ANSATZ_FULLY_CONNECTED || d.kind == CGSVMC_ANSATZ_RBM) {
    if (d.layer_size < 1) return invalid("ansatz_create: layer_size < 1");
  } else {
    if (d.num_layers < 1 || d.num_filters < 1 || d.kernel_size < 1)
      return invalid("ansatz_create: conv needs num_layers, num_filters, kernel_size >= 1");
    if ((d.kind == CGSVMC_ANSATZ_CONV_2D || d.kind == CGSVMC_ANSATZ_RESNET_2D) &&
        (int64_t)d.size_x * d.size_y != d.n_sites)
      return invalid("ansatz_create: size_x * size_y must equal n_sites");
    if ((d.kind == CGSVMC_ANSATZ_RESNET_1D || d.kind == CGSVMC_ANSATZ_RESNET_2D) && d.num_layers > 7)
      return invalid("ansatz_create: at most 7 residual blocks");
  }
  if (d.nonlinearity < CGSVMC_ACT_RELU || d.nonlinearity > CGSVMC_ACT_SELU)
    return invalid("ansatz_create: unknown nonlinearity");
  cgsvmc_ansatz* a = new (std::nothrow) cgsvmc_ansatz();
  if (a == nullptr) return invalid("ansatz_create: out of host memory");
  a->desc = d;
  a->sizes = sizes;
  int64_t off = 0;
  for (int64_t s : sizes) { a->offsets.push_back(off); off += s; }
  a->n_params = off;
  cudaError_t e = cudaGetDevice(&a->device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&a->num_sms, cudaDevAttrMultiProcessorCount, a->device);
  if (e == cudaSuccess)
    e = cudaDeviceGetAttribute(&a->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, a->device);
  if (e != cudaSuccess) {
    delete a;
    return cuda_fail(e, "ansatz_create: device query");
  }
  *out = a;
  return CGSVMC_OK;
}

int cgsvmc_ansatz_destroy(cgsvmc_ansatz* a) {
  if (a == nullptr) return CGSVMC_OK;
  if (a->scratch != nullptr) cudaFree(a->scratch);
  for (void* p : a->retired) cudaFree(p);
  if (a->tables != nullptr) cudaFree(a->tables);
  if (a->acc_weights != nullptr) cudaFree(a->acc_weights);
  if (a->grid_sync != nullptr) cudaFree(a->grid_sync);
  for (auto& pt : a->pair_tables)
    if (pt.buf != nullptr) cudaFree(pt.buf);
  delete a;
  return CGSVMC_OK;
}

int64_t cgsvmc_ansatz_num_params(const cgsvmc_ansatz* a) { return a == nullptr ? -1 : a->n_params; }

int cgsvmc_ansatz_bind_params(cgsvmc_ansatz* a, const float* params_dev) {
  if (a == nullptr || params_dev == nullptr) return invalid("bind_params: NULL argument");
  a->params = params_dev;
  a->tables_valid = false;
  return CGSVMC_OK;
}

int cgsvmc_ansatz_track_params(cgsvmc_ansatz* a, int enabled) {
  if (a == nullptr) return invalid("track_params: NULL argument");
  a->track_params = enabled != 0;
  a->tables_valid = false;
  return CGSVMC_OK;
}

int cgsvmc_ansatz_params_changed(cgsvmc_ansatz* a) {
  if (a == nullptr) return invalid("params_changed: NULL argument");
  a->tables_valid = false;
  return CGSVMC_OK;
}

int cgsvmc_ham_create(const int32_t* ij_host, const float* jx_host, const float* jz_host,
                      int32_t n_bonds, int32_t n_sites, cgsvmc_ham** out) {
  if (out == nullptr) return invalid("ham_create: NULL out");
  *out = nullptr;
  if (n_bonds < 0 || (n_bonds > 0 && (ij_host == nullptr || jx_host == nullptr || jz_host == nullptr)))
    return invalid("ham_create: NULL bond arrays");
  if (n_sites < 2 || n_sites > CGSVMC_MAX_SITES) return invalid("ham_create: n_sites must be in [2, 256]");
  for (int k = 0; k < 2 * n_bonds; ++k)
    if (ij_host[k] < 0 || ij_host[k] >= n_sites) return invalid("ham_create: bond site index out of range");
  for (int k = 0; k < n_bonds; ++k)
    if (ij_host[2 * k] == ij_host[2 * k + 1]) return invalid("ham_create: bond connects a site to itself");
  cgsvmc_ham* h = new (std::nothrow) cgsvmc_ham();
  if (h == nullptr) return invalid("ham_create: out of host memory");
  static uint64_t next_uid = 0;
  h->uid = ++next_uid;
  h->n_bonds = n_bonds;
  h->n_sites = n_sites;
  const size_t nb = (size_t)std::max(n_bonds, 1);
  cudaError_t e = cudaMalloc(&h->ij, nb * sizeof(int2));
  if (e == cudaSuccess) e = cudaMalloc(&h->jx, nb * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&h->jz, nb * sizeof(float));
  if (e == cudaSuccess && n_bonds > 0) {
    e = cudaMemcpy(h->ij, ij_host, (size_t)n_bonds * sizeof(int2), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->jx, jx_host, (size_t)n_bonds * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->jz, jz_host, (size_t)n_bonds * sizeof(float), cudaMemcpyHostToDevice);
  }
  if (e != cudaSuccess) {
    cgsvmc_ham_destroy(h);
    return cuda_fail(e, "ham_create");
  }
  *out = h;
  return CGSVMC_OK;
}

int cgsvmc_ham_destroy(cgsvmc_ham* h) {
  if (h == nullptr) return CGSVMC_OK;
  if (h->ij) cudaFree(h->ij);
  if (h->jx) cudaFree(h->jx);
  if (h->jz) cudaFree(h->jz);
  delete h;
  return CGSVMC_OK;
}

int cgsvmc_pack_configs(const float* configs, int64_t B, int32_t N, uint64_t* packed, void* stream) {
  NvtxRange range("cgsvmc:K0 pack_configs");
  if (B < 0 || N < 1 || N > CGSVMC_MAX_SITES) return invalid("pack_configs: bad shape");
  if (B > 0 && (configs == nullptr || packed == nullptr)) return invalid("pack_configs: NULL buffer");
  return launch_pack(configs, B, N, packed, (cudaStream_t)stream);
}

int cgsvmc_pack_configs_host(const float* configs_host, int64_t B, int32_t N, uint64_t* packed_host,
                             int32_t n_threads) {
  NvtxRange range("cgsvmc:K0 pack_configs_host");
  if (B < 0 || N < 1 || N > CGSVMC_MAX_SITES) return invalid("pack_configs_host: bad shape");
  if (B > 0 && (configs_host == nullptr || packed_host == nullptr)) return invalid("pack_configs_host: NULL buffer");
  if (B == 0) return CGSVMC_OK;
  return pack_configs_host(configs_host, B, N, packed_host, n_threads);
}

int cgsvmc_upload_configs(const float* configs_host, int64_t B, int32_t N, uint64_t* staging_host,
                          void* dst, int32_t n_threads, void* stream) {
  NvtxRange range("cgsvmc:K0 upload_configs");
  if (B < 0 || N < 1 || N > CGSVMC_MAX_SITES) return invalid("upload_configs: bad shape");
  if (B == 0) return CGSVMC_OK;
  if (configs_host == nullptr || dst == nullptr) return invalid("upload_configs: NULL buffer");
  const void* src = configs_host;
  size_t bytes = (size_t)B * (size_t)N * sizeof(float);
  if (staging_host != nullptr) {
    if (int rc = pack_configs_host(configs_host, B, N, staging_host, n_threads)) return rc;
    src = staging_host;
    bytes = (size_t)B * (size_t)n_words(N) * sizeof(uint64_t);
  }
  return cuda_fail(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream),
                   "upload_configs copy");
}

int cgsvmc_unpack_configs(const uint64_t* packed, int64_t B, int32_t N, float* configs, void* stream) {
  NvtxRange range("cgsvmc:K0 unpack_configs");
  if (B < 0 || N < 1 || N > CGSVMC_MAX_SITES) return invalid("unpack_configs: bad shape");
  if (B > 0 && (configs == nullptr || packed == nullptr)) return invalid("unpack_configs: NULL buffer");
  return launch_unpack(packed, B, N, configs, (cudaStream_t)stream);
}

int cgsvmc_random_configs(uint64_t* packed, int64_t B, int32_t N, uint64_t seed, uint64_t walker_id0,
                          void* stream) {
  NvtxRange range("cgsvmc:K0 random_configs");
  if (B < 0 || N < 2 || N > CGSVMC_MAX_SITES) return invalid("random_configs: bad shape");
  if (B > 0 && packed == nullptr) return invalid("random_configs: NULL buffer");
  return launch_random_configs(packed, B, N, seed, walker_id0, (cudaStream_t)stream);
}

int cgsvmc_log_amp(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, float* log_amp,
                   void* stream) {
  NvtxRange range("cgsvmc:K1 log_amp");
  if (int rc = check_ready(a)) return rc;
  if (B < 0) return invalid("log_amp: n_walkers < 0");
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr || log_amp == nullptr) return invalid("log_amp: NULL buffer");
  if (rbm_fast_supported(a)) return rbm_log_amp(a, packed, B, log_amp, (cudaStream_t)stream);
  if (conv_tc_supported(a, nullptr))
    return conv_tc_log_amp(const_cast<cgsvmc_ansatz*>(a), packed, B, log_amp, (cudaStream_t)stream);
  if (fc_tc_supported(a, nullptr))
    return fc_tc_log_amp(const_cast<cgsvmc_ansatz*>(a), packed, B, log_amp, (cudaStream_t)stream);
  return net_log_amp(a, packed, B, log_amp, (cudaStream_t)stream);
}

int cgsvmc_mc_steps(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int32_t n_steps,
                    uint64_t seed, uint64_t walker_id0, uint64_t step0,
                    unsigned long long* accept_count, float* log_amp_out, void* stream) {
  NvtxRange range("cgsvmc:K2 mc_steps");
  if (int rc = check_ready(a)) return rc;
  if (B < 0 || n_steps < 0) return invalid("mc_steps: negative size");
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr) return invalid("mc_steps: NULL configs");
  if (rbm2_supported(a, nullptr))
    return rbm2_mc_steps(const_cast<cgsvmc_ansatz*>(a), packed, B, n_steps, seed, walker_id0, step0,
                         accept_count, log_amp_out, (cudaStream_t)stream);
  if (conv_tc_supported(a, nullptr))
    return conv_tc_mc_steps(const_cast<cgsvmc_ansatz*>(a), packed, B, n_steps, seed, walker_id0, step0,
                            accept_count, log_amp_out, (cudaStream_t)stream);
  if (fc_warp_supported(a, B))      // small batches: one warp per walker beats the 128-walker tensor-core tiles
    return fc_warp_mc_steps(a, packed, B, n_steps, seed, walker_id0, step0, accept_count, log_amp_out,
                            (cudaStream_t)stream);
  if (fc_tc_supported(a, nullptr))
    return fc_tc_mc_steps(const_cast<cgsvmc_ansatz*>(a), packed, B, n_steps, seed, walker_id0, step0,
                          accept_count, log_amp_out, (cudaStream_t)stream);
  return net_mc_steps(a, packed, B, n_steps, seed, walker_id0, step0, accept_count, log_amp_out,
                      (cudaStream_t)stream);
}

int cgsvmc_mc_steps_graph(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int32_t n_steps,
                          uint64_t seed, uint64_t walker_id0, uint64_t* step_counter,
                          unsigned long long* accept_count, float* log_amp_out, void* stream) {
  NvtxRange range("cgsvmc:K2 mc_steps_graph");
  if (a == nullptr) return invalid("ansatz handle is NULL");
  if (step_counter == nullptr) return invalid("mc_steps_graph: NULL step counter");
  cgsvmc_ansatz* am = const_cast<cgsvmc_ansatz*>(a);
  am->step_counter_dev = step_counter;
  const int rc = cgsvmc_mc_steps(a, packed, B, n_steps, seed, walker_id0, 0, accept_count, log_amp_out, stream);
  am->step_counter_dev = nullptr;
  if (rc != CGSVMC_OK || B == 0) return rc;
  return launch_advance_counter(step_counter, (uint64_t)n_steps, (cudaStream_t)stream);
}

int cgsvmc_mc_step_replay(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, const float* u_sites,
                          const float* u_acc, int32_t* down_site, int32_t* up_site,
                          float* log_ratio, uint8_t* accept_mask, void* stream) {
  NvtxRange range("cgsvmc:K2 mc_step_replay");
  if (int rc = check_ready(a)) return rc;
  if (B < 0) return invalid("mc_step_replay: n_walkers < 0");
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr || u_sites == nullptr || u_acc == nullptr)
    return invalid("mc_step_replay: NULL buffer");
  if (rbm_fast_supported(a))
    return rbm_mc_replay(a, packed, B, u_sites, u_acc, down_site, up_site, log_ratio, accept_mask,
                         (cudaStream_t)stream);
  return net_mc_replay(a, packed, B, u_sites, u_acc, down_site, up_site, log_ratio, accept_mask,
                       (cudaStream_t)stream);
}

int cgsvmc_flip_enum(const cgsvmc_ham* h, const uint64_t* packed, int64_t B, uint64_t* flipped,
                     uint32_t* active_mask, void* stream) {
  NvtxRange range("cgsvmc:K3 flip_enum");
  if (h == nullptr) return invalid("flip_enum: NULL hamiltonian");
  if (B < 0) return invalid("flip_enum: n_walkers < 0");
  if (B > 0 && packed == nullptr) return invalid("flip_enum: NULL configs");
  return launch_flip_enum(h, packed, B, flipped, active_mask, (cudaStream_t)stream);
}

int cgsvmc_local_energy(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed,
                        int64_t B, float* e_loc, float* log_amp_out, float* diag_out,
                        float* offdiag_ratio_out, void* stream) {
  NvtxRange range("cgsvmc:K3 local_energy");
  if (int rc = check_ready(a)) return rc;
  if (h == nullptr) return invalid("local_energy: NULL hamiltonian");
  if (h->n_sites != a->desc.n_sites) return invalid("local_energy: hamiltonian and ansatz n_sites differ");
  if (B < 0) return invalid("local_energy: n_walkers < 0");
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr || e_loc == nullptr) return invalid("local_energy: NULL buffer");
  if (rbm2_supported(a, h))
    return rbm2_walker(const_cast<cgsvmc_ansatz*>(a), h, packed, B, e_loc, log_amp_out, diag_out,
                       offdiag_ratio_out, false, nullptr, 0, nullptr, nullptr, (cudaStream_t)stream);
  if (rbm_fast_supported(a))
    return rbm_local_energy(a, h, packed, B, e_loc, log_amp_out, diag_out, offdiag_ratio_out,
                            (cudaStream_t)stream);
  if (conv_tc_supported(a, h))
    return conv_tc_local_energy(const_cast<cgsvmc_ansatz*>(a), h, packed, B, e_loc, log_amp_out, diag_out,
                                offdiag_ratio_out, (cudaStream_t)stream);
  if (fc_tc_supported(a, h))
    return fc_tc_local_energy(const_cast<cgsvmc_ansatz*>(a), h, packed, B, e_loc, log_amp_out, diag_out,
                              offdiag_ratio_out, (cudaStream_t)stream);
  return net_local_energy(a, h, packed, B, e_loc, log_amp_out, diag_out, offdiag_ratio_out,
                          (cudaStream_t)stream);
}

int cgsvmc_weighted_grad_sum(const cgsvmc_ansatz* a, const uint64_t* packed, const float* weights,
                             int64_t B, int32_t K, float* out, void* stream) {
  NvtxRange range("cgsvmc:K4 weighted_grad_sum");
  if (int rc = check_ready(a)) return rc;
  if (B < 0) return invalid("weighted_grad_sum: n_walkers < 0");
  if (K < 1 || K > 4) return invalid("weighted_grad_sum: n_weights must be in 1..4");
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr || weights == nullptr || out == nullptr)
    return invalid("weighted_grad_sum: NULL buffer");
  cgsvmc_ansatz* am = const_cast<cgsvmc_ansatz*>(a);   // scratch growth only
  if (rbm2_supported(a, nullptr)) {
    for (int k0 = 0; k0 < K; k0 += 2) {   // two weight columns per pass
      const int kk = K - k0 < 2 ? K - k0 : 2;
      if (int rc = rbm2_walker(am, nullptr, packed, B, nullptr, nullptr, nullptr, nullptr, true,
                               weights + (int64_t)k0 * B, kk, out + (int64_t)k0 * a->n_params,
                               nullptr, (cudaStream_t)stream))
        return rc;
    }
    return CGSVMC_OK;
  }
  if (fc_tc_grad_supported(a)) return fc_tc_grad(am, packed, weights, B, K, out, (cudaStream_t)stream);
  if (conv_tc_grad_supported(a)) return conv_tc_grad(am, packed, weights, B, K, out, (cudaStream_t)stream);
  return net_grad(am, packed, weights, B, K, out, (cudaStream_t)stream);
}

int cgsvmc_log_amp_jvp(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, const float* tangent,
                       float* jvp_out, void* stream) {
  NvtxRange range("cgsvmc:K1 log_amp_jvp");
  if (int rc = check_ready(a)) return rc;
  if (B < 0) return invalid("log_amp_jvp: n_walkers < 0");
  // before the empty-batch return, so that a call with no walkers probes for support
  if (!rbm_fast_supported(a)) {
    set_error("log_amp_jvp: built for the pure RBM only (rbm, no hidden layers, H <= 256, "
              "1, 2 or 4 spin words)");
    return CGSVMC_ERR_UNSUPPORTED;
  }
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr || tangent == nullptr || jvp_out == nullptr) return invalid("log_amp_jvp: NULL buffer");
  return rbm_log_amp_jvp(a, packed, B, tangent, jvp_out, (cudaStream_t)stream);
}

int cgsvmc_accumulate(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                      float* e_loc_out, float* log_amp_out, float* sums, double* stats, void* stream) {
  NvtxRange range("cgsvmc:K3+K4+K5 accumulate");
  if (int rc = check_ready(a)) return rc;
  if (h == nullptr) return invalid("accumulate: NULL hamiltonian");
  if (h->n_sites != a->desc.n_sites) return invalid("accumulate: hamiltonian and ansatz n_sites differ");
  if (B < 0) return invalid("accumulate: n_walkers < 0");
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr || sums == nullptr || stats == nullptr) return invalid("accumulate: NULL buffer");
  cgsvmc_ansatz* am = const_cast<cgsvmc_ansatz*>(a);
  cudaStream_t st = (cudaStream_t)stream;
  if (rbm2_supported(a, h))
    return rbm2_walker(am, h, packed, B, e_loc_out, log_amp_out, nullptr, nullptr, true, nullptr, 2, sums,
                       stats, st);
  // generic path: E_loc into the second weight row, then the two gradient sums
  const size_t need = (size_t)2 * B * sizeof(float);
  if (am->acc_weights_bytes < need) {
    if (am->acc_weights != nullptr) {
      am->retired.push_back(am->acc_weights);
      am->acc_weights = nullptr;
      am->acc_weights_bytes = 0;
    }
    if (int rc = cuda_fail(cudaMalloc(&am->acc_weights, need), "accumulate alloc")) return rc;
    am->acc_weights_bytes = need;
  }
  float* w = am->acc_weights;
  if (int rc = launch_fill(w, B, 1.0f, st)) return rc;
  if (int rc = cgsvmc_local_energy(a, h, packed, B, w + B, log_amp_out, nullptr, nullptr, stream)) return rc;
  if (e_loc_out != nullptr)
    if (int rc = cuda_fail(cudaMemcpyAsync(e_loc_out, w + B, (size_t)B * sizeof(float),
                                           cudaMemcpyDeviceToDevice, st), "accumulate copy")) return rc;
  if (int rc = cgsvmc_weighted_grad_sum(a, packed, w, B, 2, sums, stream)) return rc;
  return launch_energy_stats(w + B, B, stats, st);
}

static int batch_step_impl(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const float* configs_f32,
                           uint64_t* packed, int64_t B, float* e_loc_out, float* log_amp_out, float* sums,
                           double* stats, int32_t n_steps, uint64_t seed, uint64_t walker_id0, uint64_t step0,
                           uint64_t* step_counter, unsigned long long* accept_count, double* stats_out,
                           void* stream, int32_t n_iters = 1) {
  if (int rc = check_ready(a)) return rc;
  if (h == nullptr) return invalid("batch_step: NULL hamiltonian");
  if (h->n_sites != a->desc.n_sites) return invalid("batch_step: hamiltonian and ansatz n_sites differ");
  if (B < 0 || n_steps < 0) return invalid("batch_step: negative size");
  if (B == 0) return CGSVMC_OK;
  if (packed == nullptr || sums == nullptr || stats == nullptr) return invalid("batch_step: NULL buffer");
  cudaStream_t st = (cudaStream_t)stream;
  if (rbm2_supported(a, h)) {
    cgsvmc_ansatz* am = const_cast<cgsvmc_ansatz*>(a);
    Rbm2Sweep sw = {n_steps, seed, walker_id0, step_counter != nullptr ? 0 : step0, accept_count,
                    step_counter,   // the reduction advances the counter
                    configs_f32, stats_out, n_iters};
    am->step_counter_dev = step_counter;
    const int rc = rbm2_walker(am, h, packed, B, e_loc_out, log_amp_out, nullptr, nullptr, true, nullptr, 2,
                               sums, stats, st, &sw);
    am->step_counter_dev = nullptr;
    return rc;
  }
  if (configs_f32 != nullptr)
    if (int rc = launch_pack(configs_f32, B, a->desc.n_sites, packed, st)) return rc;
  if (int rc = cgsvmc_accumulate(a, h, packed, B, e_loc_out, log_amp_out, sums, stats, stream)) return rc;
  if (stats_out != nullptr)
    if (int rc = cuda_fail(cudaMemcpyAsync(stats_out, stats, 4 * sizeof(double), cudaMemcpyDefault, st),
                           "batch_step stats copy"))
      return rc;
  if (step_counter != nullptr)
    return cgsvmc_mc_steps_graph(a, packed, B, n_steps, seed, walker_id0, step_counter, accept_count,
                                 nullptr, stream);
  return cgsvmc_mc_steps(a, packed, B, n_steps, seed, walker_id0, step0, accept_count, nullptr, stream);
}

int cgsvmc_batch_step(const cgsvmc_ansatz* a, const cgsvmc_ham* h, uint64_t* packed, int64_t B,
                      float* e_loc_out, float* log_amp_out, float* sums, double* stats,
                      int32_t n_steps, uint64_t seed, uint64_t walker_id0, uint64_t step0,
                      uint64_t* step_counter, unsigned long long* accept_count, void* stream) {
  NvtxRange range("cgsvmc:K2+K3+K4+K5 batch_step");
  return batch_step_impl(a, h, nullptr, packed, B, e_loc_out, log_amp_out, sums, stats, n_steps, seed,
                         walker_id0, step0, step_counter, accept_count, nullptr, stream);
}

int cgsvmc_batch_steps(const cgsvmc_ansatz* a, const cgsvmc_ham* h, uint64_t* packed, int64_t B, int32_t n_batches,
                       float* e_loc_out, float* log_amp_out, float* sums, double* stats, int32_t n_steps,
                       uint64_t seed, uint64_t walker_id0, uint64_t step0, uint64_t* step_counter,
                       unsigned long long* accept_count, void* stream) {
  NvtxRange range("cgsvmc:K2+K3+K4+K5 batch_steps");
  if (n_batches < 0) return invalid("batch_steps: n_batches < 0");
  if (n_batches == 0) return CGSVMC_OK;
  if (int rc = check_ready(a)) return rc;
  if (h != nullptr && rbm2_supported(a, h))
    return batch_step_impl(a, h, nullptr, packed, B, e_loc_out, log_amp_out, sums, stats, n_steps, seed,
                           walker_id0, step0, step_counter, accept_count, nullptr, stream, n_batches);
  // tile networks: the launches of every iteration, one after another
  for (int32_t i = 0; i < n_batches; ++i) {
    if (int rc = batch_step_impl(a, h, nullptr, packed, B, e_loc_out != nullptr ? e_loc_out + (int64_t)i * B : nullptr,
                                 log_amp_out != nullptr ? log_amp_out + (int64_t)i * B : nullptr, sums, stats,
                                 n_steps, seed, walker_id0, step0 + (uint64_t)i * (uint64_t)n_steps, step_counter,
                                 accept_count, nullptr, stream))
      return rc;
  }
  return CGSVMC_OK;
}

int cgsvmc_rbm2_plan(const cgsvmc_ansatz* a, const cgsvmc_ham* h, int64_t B, int32_t mode, int32_t* out,
                     int32_t n_out) {
  if (a == nullptr) return invalid("ansatz handle is NULL");
  if (B < 1) return invalid("rbm2_plan: n_walkers < 1");
  if (n_out < 0 || (n_out > 0 && out == nullptr)) return invalid("rbm2_plan: bad output buffer");
  if (mode < CGSVMC_RBM2_PLAN_MC_STEPS || mode > CGSVMC_RBM2_PLAN_BATCH_STEPS) return invalid("rbm2_plan: unknown mode");
  const bool needs_ham = mode == CGSVMC_RBM2_PLAN_LOCAL_ENERGY || mode == CGSVMC_RBM2_PLAN_ACCUMULATE ||
                         mode == CGSVMC_RBM2_PLAN_BATCH_STEPS;
  if (needs_ham && h == nullptr) return invalid("rbm2_plan: NULL hamiltonian");
  if (needs_ham && h->n_sites != a->desc.n_sites) return invalid("rbm2_plan: hamiltonian and ansatz n_sites differ");
  int32_t fields[kRbm2PlanFields];
  const int rc = rbm2_plan(a, needs_ham ? h : nullptr, B, mode, fields);
  for (int i = 0; i < n_out && i < kRbm2PlanFields; ++i) out[i] = fields[i];
  return rc;
}

int cgsvmc_batch_step_fed(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const float* configs_f32,
                          uint64_t* packed_out, int64_t B, float* e_loc_out, float* log_amp_out,
                          float* sums, double* stats, int32_t n_steps, uint64_t seed, uint64_t walker_id0,
                          uint64_t step0, uint64_t* step_counter, unsigned long long* accept_count,
                          double* stats_out, void* stream) {
  NvtxRange range("cgsvmc:K0+K2+K3+K4+K5 batch_step_fed");
  return batch_step_impl(a, h, configs_f32, packed_out, B, e_loc_out, log_amp_out, sums, stats, n_steps, seed,
                         walker_id0, step0, step_counter, accept_count, stats_out, stream);
}

int cgsvmc_propose_exchange(const uint64_t* packed, int64_t B, int32_t N, uint64_t seed,
                            uint64_t walker_id0, uint64_t step, uint64_t* proposed, float* u_acc,
                            void* stream) {
  NvtxRange range("cgsvmc:K2 propose_exchange");
  if (B < 0 || N < 2 || N > CGSVMC_MAX_SITES) return invalid("propose_exchange: bad shape");
  if (B > 0 && (packed == nullptr || proposed == nullptr || u_acc == nullptr))
    return invalid("propose_exchange: NULL buffer");
  return launch_propose_exchange(packed, B, N, seed, walker_id0, step, proposed, u_acc, (cudaStream_t)stream);
}

int cgsvmc_accept_exchange(uint64_t* packed, const uint64_t* proposed, int64_t B, int32_t N,
                           float* logabs, float* sign, const float* logabs_new, const float* sign_new,
                           const float* u_acc, unsigned long long* accept_count, void* stream) {
  NvtxRange range("cgsvmc:K2 accept_exchange");
  if (B < 0 || N < 2 || N > CGSVMC_MAX_SITES) return invalid("accept_exchange: bad shape");
  if (B > 0 && (packed == nullptr || proposed == nullptr || logabs == nullptr || logabs_new == nullptr ||
                u_acc == nullptr))
    return invalid("accept_exchange: NULL buffer");
  if ((sign == nullptr) != (sign_new == nullptr)) return invalid("accept_exchange: sign and sign_new go together");
  return launch_accept_exchange(packed, proposed, B, N, logabs, sign, logabs_new, sign_new, u_acc,
                                accept_count, (cudaStream_t)stream);
}

int cgsvmc_local_energy_from_amps(const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                                  const float* logabs, const float* sign, const float* flipped_logabs,
                                  const float* flipped_sign, float* e_loc, float* diag_out,
                                  float* offdiag_ratio_out, void* stream) {
  NvtxRange range("cgsvmc:K3 local_energy_from_amps");
  if (h == nullptr) return invalid("local_energy_from_amps: NULL hamiltonian");
  if (B < 0) return invalid("local_energy_from_amps: n_walkers < 0");
  if (B > 0 && (packed == nullptr || logabs == nullptr || (h->n_bonds > 0 && flipped_logabs == nullptr)))
    return invalid("local_energy_from_amps: NULL buffer");
  return launch_eloc_from_amps(h, packed, B, logabs, sign, flipped_logabs, flipped_sign, e_loc, diag_out,
                               offdiag_ratio_out, (cudaStream_t)stream);
}

int cgsvmc_swo_weights(const float* log_amp, const float* sign, const float* log_amp_target,
                       const float* sign_target, int64_t B, float log_norm, float inv_total,
                       float* weights_out, double* loss_acc, void* stream) {
  NvtxRange range("cgsvmc:K5 swo_weights");
  if (B < 0) return invalid("swo_weights: n_walkers < 0");
  if (B > 0 && (log_amp == nullptr || log_amp_target == nullptr || weights_out == nullptr))
    return invalid("swo_weights: NULL buffer");
  return launch_swo_weights(log_amp, sign, log_amp_target, sign_target, B, log_norm, inv_total, weights_out,
                            loss_acc, (cudaStream_t)stream);
}

int cgsvmc_adam_step(float* params, float* m, float* v, int64_t n, const float* grad, const float* sums,
                     const double* stats, float inv_num_batches, float lr, const float* lr_dev,
                     float beta1, float beta2, float eps, uint64_t t, uint64_t* t_dev, void* stream) {
  NvtxRange range("cgsvmc:adam_step");
  if (n < 0) return invalid("adam_step: n < 0");
  if (n == 0) return CGSVMC_OK;
  if (params == nullptr || m == nullptr || v == nullptr) return invalid("adam_step: NULL buffer");
  if ((grad == nullptr) == (sums == nullptr)) return invalid("adam_step: give either grad or sums");
  if (sums != nullptr && stats == nullptr) return invalid("adam_step: sums need stats");
  if (t_dev == nullptr && t < 1) return invalid("adam_step: t starts at 1");
  if (int rc = launch_adam(params, m, v, n, grad, sums, stats, inv_num_batches, lr, lr_dev, beta1, beta2, eps,
                           t, t_dev, (cudaStream_t)stream))
    return rc;
  if (t_dev != nullptr) return launch_advance_counter(t_dev, 1, (cudaStream_t)stream);
  return CGSVMC_OK;
}

int cgsvmc_epoch_end(float* params, float* m, float* v, int64_t n, const float* total_sums,
                     const double* total_payload, const double* total_stats, float* local_sums,
                     double* local_stats, float inv_num_batches, float lr, float beta1, float beta2, float eps,
                     uint64_t t, double* stats_out, uint32_t* ticket, void* stream) {
  NvtxRange range("cgsvmc:epoch_end");
  if (n < 0) return invalid("epoch_end: n < 0");
  if (n == 0) return CGSVMC_OK;
  if (params == nullptr || m == nullptr || v == nullptr || ticket == nullptr) return invalid("epoch_end: NULL buffer");
  if ((total_sums == nullptr) == (total_payload == nullptr))
    return invalid("epoch_end: give either total_sums + total_stats or total_payload");
  if (total_sums != nullptr && total_stats == nullptr) return invalid("epoch_end: total_sums need total_stats");
  if (t < 1) return invalid("epoch_end: t starts at 1");
  // the float32 totals are scratch of the all-reduce when they are not the local accumulators
  float* zero_b = (total_sums != nullptr && total_sums != local_sums) ? const_cast<float*>(total_sums) : nullptr;
  double* zero_sb = (total_stats != nullptr && total_stats != local_stats) ? const_cast<double*>(total_stats) : nullptr;
  return launch_epoch_end(params, m, v, n, total_sums, total_payload, total_stats, local_sums, zero_b,
                          local_stats, zero_sb, inv_num_batches, lr, beta1, beta2, eps, t, stats_out, ticket,
                          (cudaStream_t)stream);
}

int cgsvmc_conv_periodic(const float* input, int64_t B, int32_t size_x, int32_t size_y, int32_t c_in, int32_t c_out,
                         int32_t kernel_size, int32_t rank, const float* weights, const float* bias, float* output,
                         void* stream) {
  NvtxRange range("cgsvmc:conv_periodic");
  if (rank != 1 && rank != 2) return invalid("conv_periodic: rank must be 1 or 2");
  if (B < 0 || size_x < 1 || size_y < 1 || c_in < 1 || c_out < 1 || kernel_size < 1)
    return invalid("conv_periodic: bad shape");
  if (rank == 1 && size_y != 1) return invalid("conv_periodic: rank 1 needs size_y = 1");
  if (B == 0) return CGSVMC_OK;
  if (input == nullptr || weights == nullptr || output == nullptr) return invalid("conv_periodic: NULL buffer");
  // wrap padding placed BEFORE the data: layers.py:64-73 (1-D: k/2 for even kernels) and
  // 132-141 (2-D: k/2 - 1 for even kernels); (k - 1) / 2 for odd kernels
  const int k = kernel_size;
  const int pad = k % 2 == 1 ? (k - 1) / 2 : (rank == 1 ? k / 2 : k / 2 - 1);
  return launch_conv_periodic(input, B, size_x, size_y, c_in, c_out, k, rank == 2 ? k : 1, pad, rank == 2 ? pad : 0,
                              weights, bias, output, (cudaStream_t)stream);
}

int cgsvmc_energy_stats(const float* e_loc, int64_t B, double* stats, void* stream) {
  NvtxRange range("cgsvmc:K5 energy_stats");
  if (B < 0) return invalid("energy_stats: n_walkers < 0");
  if (B > 0 && (e_loc == nullptr || stats == nullptr)) return invalid("energy_stats: NULL buffer");
  return launch_energy_stats(e_loc, B, stats, (cudaStream_t)stream);
}

}  // extern "C"
