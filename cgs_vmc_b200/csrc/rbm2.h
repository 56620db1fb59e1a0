// Host-visible pieces of the second-generation pure-RBM kernels (rbm2_*.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cgsvmc {
namespace rbm2 {

// Parameter image (float offsets), built by prep_kernel from the flat
// parameter buffer: [2W | e^{4W} | e^{-4W} | A2 | base | a | a0, max|W| | select table].
struct Image {
  int N, H, HP, NP;
  int words;   // 64-bit words per walker in the packed layout (stride)
  int off_w2, off_f, off_g, off_a2, off_base, off_a, off_a0, off_lut, total;
};

struct Plan {
  Image im;
  int nw, lpw, kjv;     // words per walker, lanes per walker, HP / 32
  int slots;             // walkers per CTA batch the variant can hold
  bool ws;               // image in shared memory
  bool pt;               // walker kernel: bond-pair table in shared memory (E_loc reads one row per ratio)
  bool pt_global;        // walker kernel: bond-pair table in global memory (tables too large for shared memory)
  bool tc_grad;          // walker kernel: gradient sums on the tensor cores
  bool fuse;             // walker kernel: cross-CTA reduction inside the (cooperative) launch
  int wpc;               // walkers per CTA batch
  int64_t n_batches;
  int grid;
  size_t mc_smem, walker_smem;
  const uint64_t* step0_dev;   // optional device-side Philox step offset (CUDA graphs)
};

struct WalkerArgs;

// per-NW instantiation units
int launch_mc_nw1(const Plan&, const float*, uint64_t*, int64_t, int, uint64_t, uint64_t, uint64_t,
                  unsigned long long*, float*, cudaStream_t);
int launch_mc_nw2(const Plan&, const float*, uint64_t*, int64_t, int, uint64_t, uint64_t, uint64_t,
                  unsigned long long*, float*, cudaStream_t);
int launch_mc_nw4(const Plan&, const float*, uint64_t*, int64_t, int, uint64_t, uint64_t, uint64_t,
                  unsigned long long*, float*, cudaStream_t);
int launch_walker_nw1(const Plan&, const float*, const WalkerArgs&, cudaStream_t);
int launch_walker_nw2(const Plan&, const float*, const WalkerArgs&, cudaStream_t);
int launch_walker_nw4(const Plan&, const float*, const WalkerArgs&, cudaStream_t);

}  // namespace rbm2
}  // namespace cgsvmc
