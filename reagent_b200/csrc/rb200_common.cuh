// reagent_b200 -- common device/host helpers (sm_100a only).
//
// Data layout conventions used by every kernel in this library
//   * all batch tensors are dense row-major fp32, one transition per row;
//   * an MLP's parameters live in ONE flat fp32 arena laid out
//       [W0 (d1 x d0, row-major = nn.Linear.weight), b0 (d1), W1, b1, ...]
//     which is exactly torch's `parameters()` order for the reference's
//     FullyConnectedNetwork (reagent/models/fully_connected_network.py:101-153),
//     so Adam / Polyak / all-reduce are single launches over the arena;
//   * gradient partials, Adam moments and target networks use the same layout.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/reagent_b200.h"

namespace rb200 {

constexpr int kThreads = 256;          // every row-tile kernel uses 8 warps
constexpr int kMaxLayers = RB200_MAX_LAYERS;

// Device-side view of one MLP (passed by value as a kernel parameter).
struct Mlp {
  int n_layers;
  int dims[kMaxLayers + 1];
  int act[kMaxLayers];
  const float* params;                 // arena base (device)
  long long w_off[kMaxLayers];         // float offsets into the arena
  long long b_off[kMaxLayers];
  long long n_params;
};

inline Mlp make_mlp(const rb200_mlp_t* d) {
  Mlp m;
  m.n_layers = d->n_layers;
  for (int l = 0; l <= kMaxLayers; ++l) m.dims[l] = (l <= d->n_layers) ? d->dims[l] : 0;
  for (int l = 0; l < kMaxLayers; ++l) {
    const bool on = l < d->n_layers;
    m.act[l] = on ? d->act[l] : 0;
    m.w_off[l] = on ? d->w_off[l] : 0;
    m.b_off[l] = on ? d->b_off[l] : 0;
  }
  m.params = d->params;
  m.n_params = d->n_params;
  return m;
}
int validate_mlp(const rb200_mlp_t* d, const char* name);

__host__ __device__ __forceinline__ int round_up4(int x) { return (x + 3) & ~3; }
__host__ __device__ __forceinline__ int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ----------------------------------------------------------------------------
// activations (reagent/models/fully_connected_network.py:37-44)
// ----------------------------------------------------------------------------
__device__ __forceinline__ float act_fwd(float x, int act) {
  switch (act) {
    case RB200_ACT_RELU: return x > 0.f ? x : 0.f;
    case RB200_ACT_TANH: return tanhf(x);
    case RB200_ACT_LEAKY_RELU: return x > 0.f ? x : 0.01f * x;
    case RB200_ACT_SIGMOID: return 1.f / (1.f + expf(-x));
    case RB200_ACT_SOFTPLUS: return x > 20.f ? x : log1pf(expf(x));
    default: return x;
  }
}
// derivative of the activation expressed through its OUTPUT y
__device__ __forceinline__ float act_bwd_from_out(float y, int act) {
  switch (act) {
    case RB200_ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case RB200_ACT_TANH: return 1.f - y * y;
    case RB200_ACT_LEAKY_RELU: return y > 0.f ? 1.f : 0.01f;
    case RB200_ACT_SIGMOID: return y * (1.f - y);
    // softplus'(x) = sigmoid(x) = 1 - exp(-y); expm1 keeps it accurate for small y (x << 0),
    // where 1 - expf(-y) cancels (relative error ~0.5 at x = -16)
    case RB200_ACT_SOFTPLUS: return -expm1f(-y);
    default: return 1.f;
  }
}

// ----------------------------------------------------------------------------
// cp.async (LDGSTS) helpers
// ----------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Dynamic shared-memory opt-in of a kernel, remembered PER DEVICE (the attribute is per device
// and per function): a high-water mark indexed by the current device id, so the first launch on
// a second GPU of the same process opts in as well.  Racing threads at worst set the attribute
// twice.  Raised outside CUDA-graph capture by the first eager call.
struct SmemOptIn {
  size_t configured[64];
};
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, SmemOptIn& st, size_t bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev >= 0 && dev < 64 && st.configured[dev] >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && dev >= 0 && dev < 64) st.configured[dev] = bytes;
  return e;
}

// Error plumbing shared by the C-ABI translation units.
void set_last_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

}  // namespace rb200
