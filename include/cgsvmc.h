/*
 * cgsvmc.h -- C-ABI of the B200-native variational-Monte-Carlo hot path.
 *
 * The reference (ClarkResearchGroup/cgs-vmc) has no FFI: its hot path is a
 * pure-Python object protocol on top of TensorFlow 1.x ops.  Each entry point
 * below replaces one group of those ops; the comment above it cites the
 * reference interface it stands in for (paths relative to cgs_vmc/ in the
 * reference tree).  INTEGRATION.md shows the ctypes binding a reference
 * maintainer would add.
 *
 * Conventions
 *  - plain C: opaque handles, raw pointers, sizes.  No C++/torch types.
 *  - every `*_dev` / unqualified data pointer is a DEVICE pointer borrowed for
 *    the duration of the stream-ordered call; `*_host` pointers are host
 *    memory read synchronously during the call.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default
 *    stream).  Calls enqueue work and return; they never synchronise.
 *  - return value: CGSVMC_OK or a negative error code; the message is kept in
 *    a thread-local string returned by cgsvmc_last_error().
 *  - handles are not thread-safe: one handle per (device, host thread).
 *
 * Walker configuration layout ("packed"): W = ceil(N / 64) uint64 words per
 * walker, row-major [B, W]; site i is bit (i & 63) of word (i >> 6);
 * bit = 1 <=> spin +1, bit = 0 <=> spin -1; unused high bits are zero.
 * cgsvmc_pack_configs / cgsvmc_unpack_configs convert from / to the
 * reference's float32 [B, N] tensor of +-1 (graph_builders.py:92-125).
 *
 * Amplitudes: all entry points work with z(sigma) = log psi(sigma) + shift,
 * i.e. the tensor the reference hands to add_exp_normalization + tf.exp
 * (wavefunctions.py:206-232); psi = exp(z - exp_norm_shift) is formed by the
 * host wrapper.  With output_activation = exp the amplitude is positive and
 * the fused sampler / local-energy / estimator entry points apply; signed
 * output activations and sum / difference / product composites evaluate
 * cgsvmc_log_amp of their parts and use the amplitude-agnostic entry points
 * (cgsvmc_propose_exchange, cgsvmc_accept_exchange,
 * cgsvmc_local_energy_from_amps) near the end of this header.
 *
 * Flat parameter layout (float32, row-major, Sonnet shapes):
 *   fully_connected : W_1[in,out], b_1[out], ..., W_L, b_L, W_out[in,1], b_out[1]
 *   rbm             : a[N], a0[1], (W_l, b_l) hidden layers ..., W[in,H], c[H]
 *   conv_1d         : per layer w[k, cin, cout], b[cout]
 *   conv_2d         : per layer w[k, k, cin, cout], b[cout]
 *   res_net_1d / 2d : initial conv w[k(, k), 1, F], b[F]; per block first_conv
 *                     w[k(, k), F, F], b[F], second_conv w[k(, k), F, F], b[F]
 */
#ifndef CGSVMC_H_
#define CGSVMC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGSVMC_VERSION 100 /* major * 10000 + minor * 100 + patch */

#define CGSVMC_OK 0
#define CGSVMC_ERR_INVALID (-1)     /* bad argument / shape mismatch */
#define CGSVMC_ERR_CUDA (-2)        /* CUDA runtime error */
#define CGSVMC_ERR_UNSUPPORTED (-3) /* valid request outside the built path */

/* wavefunctions.WAVEFUNCTION_TYPES keys (wavefunctions.py:1199-1211) */
#define CGSVMC_ANSATZ_FULLY_CONNECTED 1
#define CGSVMC_ANSATZ_RBM 2
#define CGSVMC_ANSATZ_CONV_1D 3
#define CGSVMC_ANSATZ_CONV_2D 4
/* ResNet1D / ResNet2D (wavefunctions.py:617-809): an initial periodic
 * convolution 1 -> F without nonlinearity, num_layers (= num_resnet_blocks)
 * residual blocks x <- x + conv2(selu(conv1(x))) (layers.py:163-296), then the
 * sum over sites and channels.  Flat layout: initial w, b; per block
 * first_conv w, b, second_conv w, b (Sonnet creation order).  `nonlinearity`
 * is ignored (selu is fixed in the blocks). */
#define CGSVMC_ANSATZ_RESNET_1D 5
#define CGSVMC_ANSATZ_RESNET_2D 6

/* layers.NONLINEARITIES keys (layers.py:13-21) */
#define CGSVMC_ACT_RELU 0
#define CGSVMC_ACT_TANH 1
#define CGSVMC_ACT_SIGMOID 2
#define CGSVMC_ACT_IDENTITY 3
#define CGSVMC_ACT_COS 4
#define CGSVMC_ACT_EXP 5
#define CGSVMC_ACT_TAN 6
#define CGSVMC_ACT_SELU 7   /* internal: the ResNet blocks */

typedef struct cgsvmc_ansatz cgsvmc_ansatz;
typedef struct cgsvmc_ham cgsvmc_ham;

/* Mirrors the hparams consumed by <Ansatz>.from_hparams
 * (wavefunctions.py:373-388, 438-452, 512-528, 597-615). */
typedef struct cgsvmc_ansatz_desc {
  int32_t kind;         /* CGSVMC_ANSATZ_*                                   */
  int32_t n_sites;      /* hparams.num_sites                                 */
  int32_t num_layers;   /* num_fc_layers (fc, rbm) / num_conv_layers (conv)  */
  int32_t layer_size;   /* fc_layer_size                                     */
  int32_t num_filters;  /* num_conv_filters                                  */
  int32_t kernel_size;  /* kernel_size                                       */
  int32_t size_x;       /* conv_2d: hparams.size_x                           */
  int32_t size_y;       /* conv_2d: hparams.size_y                           */
  int32_t nonlinearity; /* CGSVMC_ACT_* for hidden activations               */
} cgsvmc_ansatz_desc;

int cgsvmc_version(void);
const char* cgsvmc_last_error(void);

/* ---- handles ---------------------------------------------------------- */

/* Replaces wavefunctions.build_wavefunction / <Ansatz>.__init__
 * (wavefunctions.py:1157-1196).  Unknown kind -> CGSVMC_ERR_INVALID (the
 * reference raises ValueError, wavefunctions.py:1196). */
int cgsvmc_ansatz_create(const cgsvmc_ansatz_desc* desc, cgsvmc_ansatz** out);
int cgsvmc_ansatz_destroy(cgsvmc_ansatz* ansatz);
/* Number of float32 parameters P of the flat layout above
 * (len of get_trainable_variables flattened, wavefunctions.py:167-175). */
int64_t cgsvmc_ansatz_num_params(const cgsvmc_ansatz* ansatz);
/* Borrows a device buffer of P floats; it must stay valid until the next bind
 * or destroy.  The library only reads it. */
int cgsvmc_ansatz_bind_params(cgsvmc_ansatz* ansatz, const float* params_dev);
/* Some kernels read tables derived from the parameters (exp(+-4W) of the
 * pure RBM).  By default they are rebuilt by a small kernel at every call, so
 * the bound buffer may be modified in place at any time (the reference's
 * variables are updated in place by optimizer.apply_gradients,
 * training.py:565-567).  With tracking enabled the tables are rebuilt only
 * after cgsvmc_ansatz_bind_params or cgsvmc_ansatz_params_changed: the caller
 * promises to report every in-place modification. */
int cgsvmc_ansatz_track_params(cgsvmc_ansatz* ansatz, int enabled);
int cgsvmc_ansatz_params_changed(cgsvmc_ansatz* ansatz);

/* Replaces HeisenbergHamiltonian.__init__ (operators.py:212-225), with one
 * (j_x, j_z) per bond as in HeisenbergBond.__init__ (operators.py:131-135).
 * ij_host: int32 [n_bonds, 2]; jx_host, jz_host: float32 [n_bonds]; bonds may
 * repeat (list semantics). */
int cgsvmc_ham_create(const int32_t* ij_host, const float* jx_host,
                      const float* jz_host, int32_t n_bonds, int32_t n_sites,
                      cgsvmc_ham** out);
int cgsvmc_ham_destroy(cgsvmc_ham* ham);

/* ---- walker state ----------------------------------------------------- */

/* float32 [B, N] of +-1 (graph_builders.get_configs variable,
 * graph_builders.py:92-125) <-> packed uint64 [B, W]. */
int cgsvmc_pack_configs(const float* configs, int64_t n_walkers,
                        int32_t n_sites, uint64_t* packed, void* stream);
int cgsvmc_unpack_configs(const uint64_t* packed, int64_t n_walkers,
                          int32_t n_sites, float* configs, void* stream);
/* The same conversion on the HOST, for a caller that keeps the reference's
 * float32 [B, N] tensor in host memory and feeds a batch per step: 4 N bytes
 * per walker shrink to 8 W before the PCIe link (bit = 1 <=> value > 0, the
 * rule of cgsvmc_pack_configs).  Synchronous; n_threads <= 0 picks a thread
 * count from the size (persistent worker pool).  Layout conversion only. */
int cgsvmc_pack_configs_host(const float* configs_host, int64_t n_walkers,
                             int32_t n_sites, uint64_t* packed_host,
                             int32_t n_threads);
/* One host batch to the device, asynchronously on `stream` (the caller's copy
 * stream): with staging_host == NULL the float32 [B, N] tensor itself goes to
 * dst (float32 [B, N], for cgsvmc_batch_step_fed); otherwise the batch is
 * packed into staging_host (pinned, uint64 [B, W]; must not be in flight) by
 * cgsvmc_pack_configs_host and the packed words go to dst (uint64 [B, W]).
 * configs_host should be pinned for the copy to be asynchronous. */
int cgsvmc_upload_configs(const float* configs_host, int64_t n_walkers,
                          int32_t n_sites, uint64_t* staging_host, void* dst,
                          int32_t n_threads, void* stream);
/* Replaces utils.random_configurations (utils.py:169-192): uniformly random
 * configurations with n_sites / 2 spins down, Philox keyed by
 * (seed, walker_id0 + b). */
int cgsvmc_random_configs(uint64_t* packed, int64_t n_walkers, int32_t n_sites,
                          uint64_t seed, uint64_t walker_id0, void* stream);

/* ---- amplitudes ------------------------------------------------------- */

/* Replaces Wavefunction.__call__ / _build (wavefunctions.py:47-59, 355-371,
 * 419-436, 495-510, 578-595): z[b] = log psi(sigma_b) + shift. */
int cgsvmc_log_amp(const cgsvmc_ansatz* ansatz, const uint64_t* packed,
                   int64_t n_walkers, float* log_amp, void* stream);

/* ---- Metropolis sampler ----------------------------------------------- */

/* Replaces n_steps consecutive session.run(mc_step) of
 * graph_builders.build_monte_carlo_sampling (graph_builders.py:38-89;
 * loops at training.py:608-609, 616-617, 208-210, evaluation.py:143-149):
 * per walker and step, draw a uniformly random up site and a uniformly random
 * down site, exchange them, accept iff |psi'/psi|^2 > u (strict).  Randomness
 * is Philox4x32-10 with key = seed and counter = (step0 + s, walker_id0 + b),
 * so trajectories do not depend on how walkers are sharded over devices.
 * accept_count (uint64, device) is incremented by the number of accepted
 * moves (acceptance_count, graph_builders.py:86); log_amp_out (nullable)
 * receives z of the final configurations. */
int cgsvmc_mc_steps(const cgsvmc_ansatz* ansatz, uint64_t* packed_inout,
                    int64_t n_walkers, int32_t n_steps, uint64_t seed,
                    uint64_t walker_id0, uint64_t step0,
                    unsigned long long* accept_count, float* log_amp_out,
                    void* stream);

/* CUDA-graph friendly form of cgsvmc_mc_steps: the Philox step offset is read
 * from device memory (*step_counter, uint64) when the kernel runs and advanced
 * by n_steps afterwards on the same stream, so a captured graph of
 * "accumulate + sweep" (training.py:614-617) can be replayed every batch
 * without re-using random numbers. */
int cgsvmc_mc_steps_graph(const cgsvmc_ansatz* ansatz, uint64_t* packed_inout,
                          int64_t n_walkers, int32_t n_steps, uint64_t seed,
                          uint64_t walker_id0, uint64_t* step_counter,
                          unsigned long long* accept_count, float* log_amp_out,
                          void* stream);

/* One step in REPLAY mode (tests): consumes caller-supplied uniforms exactly
 * like graph_builders.py:59-79 -- u_sites float32 [B, N] (argmin / argmax of
 * sigma * u with first-occurrence ties), u_acc float32 [B] (accept iff
 * ratio > sqrt(u)).  Outputs (all nullable): down_site / up_site int32 [B],
 * log_ratio float32 [B] = z' - z, accept_mask uint8 [B]. */
int cgsvmc_mc_step_replay(const cgsvmc_ansatz* ansatz, uint64_t* packed_inout,
                          int64_t n_walkers, const float* u_sites,
                          const float* u_acc, int32_t* down_site,
                          int32_t* up_site, float* log_ratio,
                          uint8_t* accept_mask, void* stream);

/* ---- Hamiltonian ------------------------------------------------------ */

/* Parity hook for the integer part of HeisenbergBond.build
 * (operators.py:154-167): flipped uint64 [B, n_bonds, W] = configuration with
 * the bond's two spins exchanged, active_mask uint32 [B, ceil(n_bonds / 32)]
 * with bit (k & 31) of word (k >> 5) set iff bond k is antiparallel. */
int cgsvmc_flip_enum(const cgsvmc_ham* ham, const uint64_t* packed,
                     int64_t n_walkers, uint64_t* flipped,
                     uint32_t* active_mask, void* stream);

/* Replaces HeisenbergHamiltonian.local_value (operators.py:249-259):
 * e_loc[b] = sum_k jz_k/4 s_i s_j + jx_k/2 [s_i != s_j] psi(flip_k)/psi.
 * Nullable extra outputs: log_amp_out[b] = z(sigma_b); diag_out[b] and
 * offdiag_ratio_out[b] are the two terms of Operator.build
 * (operators.py:227-247) with the off-diagonal one divided by psi, so that
 * apply_in_place (operators.py:261-271) = (diag + offdiag_ratio) * psi. */
int cgsvmc_local_energy(const cgsvmc_ansatz* ansatz, const cgsvmc_ham* ham,
                        const uint64_t* packed, int64_t n_walkers,
                        float* e_loc, float* log_amp_out, float* diag_out,
                        float* offdiag_ratio_out, void* stream);

/* ---- estimators ------------------------------------------------------- */

/* Replaces the two tf.gradients + accumulators of
 * EnergyGradientOptimizer.build_opt_ops (training.py:545-558) and the
 * gradient of the SWO loss (training.py:169-175): for k < n_weights
 *   out[k, :] += sum_b weights[k, b] * d z_b / d params      (flat layout)
 * weights float32 [n_weights, B] (n_weights <= 4), out float32 [n_weights, P]
 * ACCUMULATED into (zero it to start an epoch, training.py:568).  The
 * reduction order is fixed (deterministic for a given B). */
int cgsvmc_weighted_grad_sum(const cgsvmc_ansatz* ansatz,
                             const uint64_t* packed, const float* weights,
                             int64_t n_walkers, int32_t n_weights, float* out,
                             void* stream);

/* The forward counterpart of cgsvmc_weighted_grad_sum (a Jacobian-vector
 * product of z):
 *   jvp_out[b] = sum_p (d z_b / d params_p) * tangent[p]   (flat layout, float32 [P])
 * With it the stochastic-reconfiguration matrix S = <O O^T> - <O><O>^T is
 * applied to a vector without forming S or the per-walker gradients: one call
 * here, one cgsvmc_weighted_grad_sum with the centred result as weights.
 * Built for the pure RBM (rbm with no hidden layers, H <= 256, 1, 2 or 4 spin
 * words); any other ansatz returns CGSVMC_ERR_UNSUPPORTED, also with
 * n_walkers == 0, so a call without walkers probes for support.  FP32 with a
 * fixed summation order (deterministic). */
int cgsvmc_log_amp_jvp(const cgsvmc_ansatz* ansatz, const uint64_t* packed,
                       int64_t n_walkers, const float* tangent, float* jvp_out,
                       void* stream);

/* Replaces one session.run(accumulate_gradients) of
 * EnergyGradientOptimizer (training.py:539-558, 615) in a single pass over the
 * walkers: psi and local energy of every walker (operators.py:249-259), then
 *   sums[0, :] += sum_b O_b,  sums[1, :] += sum_b E_b O_b   (O_b = d z_b / d params)
 *   stats     += { sum E, sum E^2, B, 0 }                   (double [4])
 * e_loc_out / log_amp_out (float32 [B]) are optional.  Equivalent to
 * cgsvmc_local_energy + cgsvmc_weighted_grad_sum with weights (1, E_loc) +
 * cgsvmc_energy_stats; the walker state (theta) is built once instead of
 * three times. */
int cgsvmc_accumulate(const cgsvmc_ansatz* ansatz, const cgsvmc_ham* ham,
                      const uint64_t* packed, int64_t n_walkers, float* e_loc_out,
                      float* log_amp_out, float* sums, double* stats, void* stream);

/* One batch iteration of EnergyGradientOptimizer.run_optimization_epoch
 * (training.py:614-617): session.run(accumulate_gradients) on the current
 * configurations, then num_monte_carlo_sweeps * num_sites x session.run(mc_step)
 * -- cgsvmc_accumulate followed by cgsvmc_mc_steps (same arguments, same
 * results).  For the pure RBM both run in ONE kernel: the walker state built
 * for the local energy is reused by the sampler and the ratio tables are
 * loaded into shared memory once.  step_counter, when non-NULL, is a device
 * uint64 holding the Philox step offset (step0 is then ignored); it is
 * advanced by n_steps on the stream, which makes the call CUDA-graph safe
 * (cf. cgsvmc_mc_steps_graph). */
int cgsvmc_batch_step(const cgsvmc_ansatz* ansatz, const cgsvmc_ham* ham,
                      uint64_t* packed_inout, int64_t n_walkers,
                      float* e_loc_out, float* log_amp_out, float* sums,
                      double* stats, int32_t n_steps, uint64_t seed,
                      uint64_t walker_id0, uint64_t step0,
                      uint64_t* step_counter, unsigned long long* accept_count,
                      void* stream);

/* n_batches consecutive batch iterations -- the whole inner loop of
 * EnergyGradientOptimizer.run_optimization_epoch (training.py:614-617:
 * `for _ in range(num_batches): accumulate_gradients; mc_step x sweeps`) -- in
 * one call: the same results as n_batches cgsvmc_batch_step calls with step0
 * advanced by n_steps each time (configurations and local energies bit for
 * bit; sums and statistics to float32 / float64 rounding, the partial sums are
 * reduced once instead of n_batches times).  For the pure RBM this is ONE
 * persistent kernel: ratio tables and bonds are loaded once, every walker
 * stays with its lane group across the iterations, the CTAs keep adding to
 * their partial sums and the cross-CTA reduction runs once.  e_loc_out /
 * log_amp_out (optional) are float32 [n_batches, n_walkers]; stats gains
 * { sum E, sum E^2, n_batches * B, 0 }; step_counter (optional, device) is
 * advanced by n_batches * n_steps. */
int cgsvmc_batch_steps(const cgsvmc_ansatz* ansatz, const cgsvmc_ham* ham,
                       uint64_t* packed_inout, int64_t n_walkers, int32_t n_batches,
                       float* e_loc_out, float* log_amp_out, float* sums,
                       double* stats, int32_t n_steps, uint64_t seed,
                       uint64_t walker_id0, uint64_t step0,
                       uint64_t* step_counter, unsigned long long* accept_count,
                       void* stream);

/* Which variant of the pure-RBM kernels (rbm2) an entry point would run for
 * n_walkers walkers with the current device, switches and pair-table slots,
 * without allocating or launching anything.  `mode` names the entry point:
 * CGSVMC_RBM2_PLAN_MC_STEPS, _LOCAL_ENERGY, _WEIGHTED_GRAD_SUM, _ACCUMULATE or
 * _BATCH_STEPS (cgsvmc_batch_step and cgsvmc_batch_steps).  `ham` is needed for
 * LOCAL_ENERGY, ACCUMULATE and BATCH_STEPS and ignored otherwise.  The first
 * n_out (at most 13) of these fields go to out:
 *   supported (1), words per walker, lanes per walker, HP / 32, walker slots
 *   per CTA, walkers per CTA batch, batches, grid, parameter tables in shared
 *   memory (0/1), bond-pair table (0 none, 1 shared, 2 global memory), gradient
 *   sums on the tensor cores (0/1), cross-CTA reduction inside the kernel
 *   (0/1), walkers kept in registers between the iterations of
 *   cgsvmc_batch_steps (0/1).
 * Returns CGSVMC_ERR_UNSUPPORTED (out zeroed) when rbm2 does not take the call:
 * another path serves it. */
#define CGSVMC_RBM2_PLAN_MC_STEPS 0
#define CGSVMC_RBM2_PLAN_LOCAL_ENERGY 1
#define CGSVMC_RBM2_PLAN_WEIGHTED_GRAD_SUM 2
#define CGSVMC_RBM2_PLAN_ACCUMULATE 3
#define CGSVMC_RBM2_PLAN_BATCH_STEPS 4
int cgsvmc_rbm2_plan(const cgsvmc_ansatz* ansatz, const cgsvmc_ham* ham,
                     int64_t n_walkers, int32_t mode, int32_t* out, int32_t n_out);

/* cgsvmc_batch_step for a caller that holds the walkers in the reference's own
 * layout (the float32 [B, N] variable of graph_builders.py:92-125) and reads
 * the energy statistics back every batch (training.py:619-620): configs_f32
 * (device float32 [n_walkers, n_sites] of +-1; NULL = take packed_out as the
 * input like cgsvmc_batch_step) is bit-packed by the walker kernel itself, the
 * swept configurations are written to packed_out, and the updated statistics
 * (double [4]) are also stored to stats_out when it is non-NULL -- stats_out may
 * be mapped pinned host memory, so no copy node follows the kernel. */
int cgsvmc_batch_step_fed(const cgsvmc_ansatz* ansatz, const cgsvmc_ham* ham,
                          const float* configs_f32, uint64_t* packed_out,
                          int64_t n_walkers, float* e_loc_out, float* log_amp_out,
                          float* sums, double* stats, int32_t n_steps,
                          uint64_t seed, uint64_t walker_id0, uint64_t step0,
                          uint64_t* step_counter, unsigned long long* accept_count,
                          double* stats_out, void* stream);

/* ---- amplitude-agnostic sampler / local energy ------------------------- */
/* For wavefunctions whose amplitude is not a single fused kernel: output
 * activations other than exp (layers.py:13-21, wavefunctions.py:350-353) give
 * signed amplitudes, and the sum / difference / product composites
 * (wavefunctions.py:61-165, 1178-1194) combine two ansaetze.  The caller
 * evaluates (log|psi|, sign psi) with cgsvmc_log_amp of the parts and combines
 * them; these three calls do the integer / reduction work around it.
 *
 * cgsvmc_propose_exchange replaces graph_builders.py:59-73 for one step:
 * proposed[b] = packed[b] with a uniformly random up site and a uniformly
 * random down site exchanged, u_acc[b] = the acceptance uniform; Philox
 * convention of cgsvmc_mc_steps (same proposals for the same seed, walker,
 * step).
 * cgsvmc_accept_exchange replaces graph_builders.py:74-89: walkers with
 * exp(2 (logabs_new - logabs)) > u_acc take the proposed configuration,
 * logabs (and sign when given); *accept_count += accepted.
 * cgsvmc_local_energy_from_amps replaces operators.py:165-169, 241-259:
 *   e_loc[b] = sum_k [ jz_k/4 s_i s_j + jx_k/2 [s_i != s_j] sign' sign exp(logabs' - logabs) ]
 * with flipped_logabs / flipped_sign float32 [B, n_bonds] for the configurations
 * of cgsvmc_flip_enum (entries of parallel bonds are ignored); sign arrays may
 * be NULL (all +1). */
int cgsvmc_propose_exchange(const uint64_t* packed, int64_t n_walkers,
                            int32_t n_sites, uint64_t seed, uint64_t walker_id0,
                            uint64_t step, uint64_t* proposed, float* u_acc,
                            void* stream);
int cgsvmc_accept_exchange(uint64_t* packed_inout, const uint64_t* proposed,
                           int64_t n_walkers, int32_t n_sites, float* logabs_inout,
                           float* sign_inout, const float* logabs_new,
                           const float* sign_new, const float* u_acc,
                           unsigned long long* accept_count, void* stream);
int cgsvmc_local_energy_from_amps(const cgsvmc_ham* ham, const uint64_t* packed,
                                  int64_t n_walkers, const float* logabs,
                                  const float* sign, const float* flipped_logabs,
                                  const float* flipped_sign, float* e_loc,
                                  float* diag_out, float* offdiag_ratio_out,
                                  void* stream);

/* Replaces tf.metrics.mean(local_energy) bookkeeping (training.py:555):
 * stats (double [4], device) += { sum e, sum e^2, B, 0 }. */
int cgsvmc_energy_stats(const float* e_loc, int64_t n_walkers, double* stats,
                        void* stream);

/* Replaces the loss / gradient-weight arithmetic of
 * SupervisedWavefunctionOptimizer.build_opt_ops (training.py:166-175) for one
 * batch, in one kernel: with r_b = psi_target(s_b) sqrt(2^N) / psi(s_b) formed
 * in the log domain from cgsvmc_log_amp of the two wavefunctions (log_norm =
 * N/2 log 2 plus the difference of the exp_norm_shifts; sign arrays NULL = +1),
 *   weights_out[b] = 2 (1 - r_b) * inv_total     (d loss / d log psi_b; feed to
 *                                                 cgsvmc_weighted_grad_sum)
 *   loss_acc (double [2], nullable) += { sum_b (1 - r_b)^2, B }
 * so that loss = loss_acc[0] / loss_acc[1] is tf.reduce_mean((psi - t)^2 /
 * stop_gradient(psi)^2). */
int cgsvmc_swo_weights(const float* log_amp, const float* sign,
                       const float* log_amp_target, const float* sign_target,
                       int64_t n_walkers, float log_norm, float inv_total,
                       float* weights_out, double* loss_acc, void* stream);

/* Replaces optimizer.apply_gradients / optimizer.minimize with
 * tf.train.AdamOptimizer(lr, beta2=hparams.beta2) (training.py:76-91, 175,
 * 565-567) on the flat parameter buffer, in one kernel:
 *   m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2
 *   params -= lr sqrt(1 - b2^t) / (1 - b1^t) m / (sqrt(v) + eps).
 * The gradient g is `grad` (float32 [n]) or, when `sums` is given instead, the
 * energy gradient of training.py:562-564 formed on the fly from the estimator
 * sums (float32 [2, n]) and statistics (double [4]) of cgsvmc_accumulate:
 *   g = (sums[1] - stats[0] / stats[2] * sums[0]) * inv_num_batches.
 * lr_dev / t_dev, when non-NULL, are device scalars read instead of lr / t
 * (t_dev holds the number of steps taken so far and is advanced by one on the
 * stream): the call is then CUDA-graph safe. */
int cgsvmc_adam_step(float* params, float* m, float* v, int64_t n,
                     const float* grad, const float* sums, const double* stats,
                     float inv_num_batches, float lr, const float* lr_dev,
                     float beta1, float beta2, float eps, uint64_t t,
                     uint64_t* t_dev, void* stream);

/* Replaces the three session.run calls that end an epoch of
 * EnergyGradientOptimizer.run_optimization_epoch (training.py:618-622) with one
 * kernel: apply_gradients (cgsvmc_adam_step on the energy gradient of the
 * all-reduced totals, training.py:562-567), metrics (the totals' statistics
 * [sum E, sum E^2, n, .] are stored to stats_out, which may be mapped pinned
 * host memory; training.py:555, 619-620) and reset_gradients (local_sums
 * [2, n] and local_stats [4] are zeroed; training.py:568, 621).
 * The totals are either total_sums (float32 [2, n]) + total_stats (double [4])
 * -- the same pointers as the local accumulators on one rank -- or
 * total_payload, the float64 all-reduce payload [2 n + 4] itself.  `ticket`:
 * one zero-initialised uint32 of device memory owned by the caller (returned
 * to zero by the kernel). */
int cgsvmc_epoch_end(float* params, float* m, float* v, int64_t n,
                     const float* total_sums, const double* total_payload,
                     const double* total_stats, float* local_sums,
                     double* local_stats, float inv_num_batches, float lr,
                     float beta1, float beta2, float eps, uint64_t t,
                     double* stats_out, uint32_t* ticket, void* stream);

/* Replaces one call of layers.Conv1dPeriodic / Conv2dPeriodic (layers.py:24-160):
 * periodic (wrap) padding followed by snt.Conv1D / snt.Conv2D with padding
 * VALID and stride 1.  input: float32 [B, size_x, size_y, c_in] (NHWC; rank 1:
 * size_y = 1, i.e. [B, L, c_in]), weights: [k, (k,) c_in, c_out] (Sonnet's
 * layout), bias: [c_out] or NULL, output: [B, size_x, size_y, c_out].  The
 * padding placed before the data is (k - 1) / 2 for odd k and, for even k,
 * k / 2 in 1-D (layers.py:64-73) but k / 2 - 1 in 2-D (layers.py:132-141).
 * The ansatz entry points fuse these layers into whole networks; this one makes
 * the layer callable by itself. */
int cgsvmc_conv_periodic(const float* input, int64_t n_batch, int32_t size_x,
                         int32_t size_y, int32_t c_in, int32_t c_out,
                         int32_t kernel_size, int32_t rank, const float* weights,
                         const float* bias, float* output, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CGSVMC_H_ */
