// Internal (C++) side of the C-ABI: handle layouts and kernel launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/cgsvmc.h"

#ifndef CGSVMC_MAX_SITES
#define CGSVMC_MAX_WORDS 4      // 64-bit words per walker: n_sites <= 256
#define CGSVMC_MAX_SITES 256
#endif

struct cgsvmc_ansatz {
  cgsvmc_ansatz_desc desc;
  int64_t n_params = 0;
  const float* params = nullptr;   // borrowed device buffer, flat layout
  std::vector<int64_t> offsets;    // offset of every tensor of the flat layout
  std::vector<int64_t> sizes;
  int device = 0;
  int num_sms = 148;
  int max_smem_optin = 0;          // bytes
  float* scratch = nullptr;        // owned device scratch (gradient partials ...)
  size_t scratch_bytes = 0;
  // buffers outgrown by a later, larger request: kept until the handle is
  // destroyed because captured CUDA graphs may still point at them
  std::vector<void*> retired;
  float* tables = nullptr;         // owned: derived parameter image of the rbm2 kernels
  size_t tables_bytes = 0;
  bool tables_valid = false;       // tables match the bound parameters
  bool track_params = false;       // rebuild tables only after bind_params / params_changed
  const uint64_t* step_counter_dev = nullptr;   // set during cgsvmc_mc_steps_graph: device-side step offset
  unsigned int* grid_sync = nullptr;   // owned: arrive / depart counters of the in-kernel cross-CTA reduction (rbm2)
  float* acc_weights = nullptr;    // owned: [2, B] weight rows of cgsvmc_accumulate (tile networks)
  size_t acc_weights_bytes = 0;
  // owned: bond-pair tables of the rbm2 walker kernel ([2 n_bonds][HP]), one per
  // Hamiltonian this ansatz has been used with.  Entries are never moved or
  // evicted (captured CUDA graphs keep pointing at them); past kMaxPairTables
  // Hamiltonians the two-row path is used.
  struct PairTable {
    uint64_t ham_uid = 0;
    float* buf = nullptr;
    size_t bytes = 0;
    bool valid = false;            // matches the current tables
  };
  static constexpr int kMaxPairTables = 16;
  std::vector<PairTable> pair_tables;
};

struct cgsvmc_ham {
  uint64_t uid = 0;      // unique per created handle (cache key)
  int32_t n_bonds = 0;
  int32_t n_sites = 0;
  int2* ij = nullptr;    // device [n_bonds]
  float* jx = nullptr;   // device [n_bonds]
  float* jz = nullptr;   // device [n_bonds]
};

namespace cgsvmc {

void set_error(const std::string& msg);
int cuda_fail(cudaError_t err, const char* what);
// Grows ansatz->scratch to at least `bytes` (stream-ordered free/alloc is not
// needed: growth only happens on the first call of a given size).
int ensure_scratch(cgsvmc_ansatz* a, size_t bytes);

inline int n_words(int n_sites) { return (n_sites + 63) / 64; }

// ---- utility kernels (util_kernels.cu) ----
int launch_pack(const float* configs, int64_t B, int N, uint64_t* packed, cudaStream_t s);
int launch_unpack(const uint64_t* packed, int64_t B, int N, float* configs, cudaStream_t s);
int launch_random_configs(uint64_t* packed, int64_t B, int N, uint64_t seed, uint64_t walker0,
                          cudaStream_t s);
int launch_flip_enum(const cgsvmc_ham* h, const uint64_t* packed, int64_t B, uint64_t* flipped,
                     uint32_t* mask, cudaStream_t s);
int launch_advance_counter(uint64_t* counter, uint64_t by, cudaStream_t s);
int launch_propose_exchange(const uint64_t* packed, int64_t B, int N, uint64_t seed, uint64_t walker0,
                            uint64_t step, uint64_t* proposed, float* u_acc, cudaStream_t s);
int launch_accept_exchange(uint64_t* packed, const uint64_t* proposed, int64_t B, int N, float* logabs,
                           float* sign, const float* logabs_new, const float* sign_new,
                           const float* u_acc, unsigned long long* accept_count, cudaStream_t s);
int launch_eloc_from_amps(const cgsvmc_ham* h, const uint64_t* packed, int64_t B, const float* logabs,
                          const float* sign, const float* flipped_logabs, const float* flipped_sign,
                          float* e_loc, float* diag, float* off, cudaStream_t s);
int launch_fill(float* dst, int64_t n, float value, cudaStream_t s);
int launch_energy_stats(const float* e, int64_t B, double* stats, cudaStream_t s);
int launch_reduce_partials(const float* partials, int n_parts, int64_t n, float* out,
                           cudaStream_t s);
int launch_swo_weights(const float* z, const float* sign, const float* zt, const float* sign_t, int64_t B,
                       float log_norm, float inv_total, float* weights, double* acc, cudaStream_t s);
int pack_configs_host(const float* configs, int64_t B, int N, uint64_t* packed, int n_threads);
int launch_conv_periodic(const float* in, int64_t B, int X, int Y, int Cin, int Cout, int kx, int ky, int pad_x,
                         int pad_y, const float* w, const float* bias, float* out, cudaStream_t s);
int launch_epoch_end(float* params, float* m, float* v, int64_t n, const float* tot_sums,
                     const double* tot_payload, const double* tot_stats, float* zero_a, float* zero_b,
                     double* zero_stats_a, double* zero_stats_b, float inv_nb, float lr, float b1, float b2,
                     float eps, uint64_t t, double* stats_out, unsigned int* ticket, cudaStream_t s);
int launch_adam(float* params, float* m, float* v, int64_t n, const float* grad, const float* sums,
                const double* stats, float inv_nb, float lr, const float* lr_dev, float b1, float b2,
                float eps, uint64_t t, const uint64_t* t_dev, cudaStream_t s);

// ---- pure RBM (num_layers == 0): amplitudes, their directional derivative, replay and
//      large-bond local energy (rbm.cu) ----
bool rbm_fast_supported(const cgsvmc_ansatz* a);
int rbm_log_amp(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, float* out,
                cudaStream_t s);
// out[b] = sum_p (d z_b / d params_p) tangent[p]   (tangent: device float [P], flat layout)
int rbm_log_amp_jvp(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, const float* tangent,
                    float* out, cudaStream_t s);
int rbm_mc_replay(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, const float* u_sites,
                  const float* u_acc, int32_t* down, int32_t* up, float* log_ratio,
                  uint8_t* accept, cudaStream_t s);
int rbm_local_energy(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed,
                     int64_t B, float* e_loc, float* log_amp_out, float* diag_out,
                     float* off_out, cudaStream_t s);

// ---- pure RBM, second generation (rbm2.cu): ratio tables, 4 walkers per warp ----
// h may be NULL in rbm2_supported (sampler only).
bool rbm2_supported(const cgsvmc_ansatz* a, const cgsvmc_ham* h);
int rbm2_mc_steps(cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int n_steps, uint64_t seed,
                  uint64_t walker0, uint64_t step0, unsigned long long* accept_count,
                  float* log_amp_out, cudaStream_t s);
// One pass over the walkers: local energy when h != NULL (e_loc / log_amp /
// diag / off nullable), weighted gradient sums when do_grad (weights NULL =>
// rows (1, E_loc); out [K, P] +=; stats nullable double[4] +=).
// sweep != NULL fuses sweep->n_steps Metropolis steps after the estimators
// (`packed` is then written): one batch iteration in one launch.
struct Rbm2Sweep {
  int n_steps;
  uint64_t seed, walker0, step0;
  unsigned long long* accept_count;
  uint64_t* advance_counter;   // device step counter to advance by n_steps afterwards, or NULL
  const float* configs_f32;    // optional: the walkers as float32 [B][N] of +-1 (packed is then output only)
  double* stats_snapshot;      // optional: copy of the updated statistics (may be mapped host memory)
  int n_iters;                 // > 1: that many consecutive batch iterations in one launch (e_loc / log_amp: [n_iters][B])
};
int rbm2_walker(cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                float* e_loc, float* log_amp, float* diag, float* off, bool do_grad,
                const float* weights, int K, float* out, double* stats, cudaStream_t s,
                const Rbm2Sweep* sweep = nullptr);
// The launch plan of the entry point `mode` (CGSVMC_RBM2_PLAN_*) for B walkers,
// in the field order of cgsvmc_rbm2_plan; CGSVMC_ERR_UNSUPPORTED when rbm2 does
// not take the call.  No allocation, no launch.
constexpr int kRbm2PlanFields = 13;
int rbm2_plan(const cgsvmc_ansatz* a, const cgsvmc_ham* h, int64_t B, int mode, int32_t (&out)[kRbm2PlanFields]);

// ---- conv_1d / conv_2d forward on the tensor cores (conv_tc.cu): tcgen05 + TMEM ----
bool conv_tc_supported(const cgsvmc_ansatz* a, const cgsvmc_ham* h);
int conv_tc_log_amp(cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, float* out, cudaStream_t s);
int conv_tc_mc_steps(cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int n_steps, uint64_t seed,
                     uint64_t walker0, uint64_t step0, unsigned long long* accept_count,
                     float* log_amp_out, cudaStream_t s);
int conv_tc_local_energy(cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                         float* e_loc, float* log_amp_out, float* diag_out, float* off_out,
                         cudaStream_t s);

// weighted gradient sums of conv_1d / conv_2d on tcgen05 (conv_tc_grad.cu): forward,
// backward-data as the mirrored implicit GEMM, weight gradients as GEMMs over the
// rows (sites x configurations) of a batch with MN-major operands
struct ConvTcImage {
  const void *w1img, *wimg, *wimg_b;   // layer-1 B operand; forward / backward-data images of the tensor layers
  const float *bias, *wsum;            // [L-1][C]; [C] last-layer column sums, then N sum_c b_L[c]
};
int conv_tc_image(cgsvmc_ansatz* a, ConvTcImage* img, cudaStream_t s);
bool conv_tc_grad_supported(const cgsvmc_ansatz* a);
int conv_tc_grad(cgsvmc_ansatz* a, const uint64_t* packed, const float* weights, int64_t B, int K,
                 float* out, cudaStream_t s);

// ---- fully_connected forward on the tensor cores (fc_tc.cu): tcgen05 + TMEM ----
bool fc_tc_supported(const cgsvmc_ansatz* a, const cgsvmc_ham* h);
int fc_tc_log_amp(cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, float* out, cudaStream_t s);
int fc_tc_mc_steps(cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int n_steps, uint64_t seed,
                   uint64_t walker0, uint64_t step0, unsigned long long* accept_count,
                   float* log_amp_out, cudaStream_t s);
int fc_tc_local_energy(cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed, int64_t B,
                       float* e_loc, float* log_amp_out, float* diag_out, float* off_out,
                       cudaStream_t s);

// warp-per-walker sampler of the fully connected ansatz for small batches (fc_warp.cu)
bool fc_warp_supported(const cgsvmc_ansatz* a, int64_t B);
int fc_warp_mc_steps(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int n_steps, uint64_t seed,
                     uint64_t walker0, uint64_t step0, unsigned long long* accept_count, float* log_amp_out,
                     cudaStream_t s);

// weighted gradient sums of the fully connected ansatz on tcgen05 (fc_tc_grad.cu):
// forward, backward-data and the weight-gradient GEMMs dW_l = h_{l-1}^T (w delta_l)
int fc_tc_image(cgsvmc_ansatz* a, const void** wimg, const float** consts, cudaStream_t s);
bool fc_tc_grad_supported(const cgsvmc_ansatz* a);
int fc_tc_grad(cgsvmc_ansatz* a, const uint64_t* packed, const float* weights, int64_t B, int K,
               float* out, cudaStream_t s);

// ---- generic tile networks: fc, rbm with hidden layers, conv (net.cu) ----
int net_log_amp(const cgsvmc_ansatz* a, const uint64_t* packed, int64_t B, float* out,
                cudaStream_t s);
int net_mc_steps(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, int n_steps, uint64_t seed,
                 uint64_t walker0, uint64_t step0, unsigned long long* accept_count,
                 float* log_amp_out, cudaStream_t s);
int net_mc_replay(const cgsvmc_ansatz* a, uint64_t* packed, int64_t B, const float* u_sites,
                  const float* u_acc, int32_t* down, int32_t* up, float* log_ratio,
                  uint8_t* accept, cudaStream_t s);
int net_local_energy(const cgsvmc_ansatz* a, const cgsvmc_ham* h, const uint64_t* packed,
                     int64_t B, float* e_loc, float* log_amp_out, float* diag_out,
                     float* off_out, cudaStream_t s);
int net_grad(cgsvmc_ansatz* a, const uint64_t* packed, const float* weights, int64_t B, int K,
             float* out, cudaStream_t s);

}  // namespace cgsvmc
