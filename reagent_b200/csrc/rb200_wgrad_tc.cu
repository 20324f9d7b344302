// reagent_b200 -- weight gradients on the 5th-generation tensor cores.
//
//   dW_l[n, k] = sum_b dZ_l[b, n] * A_{l-1}[b, k],   db_l[n] = sum_b dZ_l[b, n]
// (autograd's Linear backward reached from loss.backward() in the reference's Lightning loop,
// reagent/training/reagent_lightning_module.py:108-133) as tcgen05.mma kind::tf32 with 3xTF32
// error compensation and the accumulator in Tensor Memory.
//
// The contraction runs over the BATCH, and both factors are stored batch-row-major in HBM
// ([B, N] and [B, K]), i.e. transposed with respect to the K-major operand layout the MMA
// reads.  The kernel transposes while staging: a 32-row chunk of both matrices is loaded with
// 16-byte loads (a lane = one row x 4 features; 16 rows x 32 B per instruction: whole sectors),
// split into TF32 hi / lo in registers, and every scalar goes straight to its place in the
// canonical K-major no-swizzle layout
//     [batch row / 4][feature][4 batch rows]   (row-quad stride = LBO, 8 features = SBO = 128 B)
// with bank-conflict-free 4-byte stores (the padded row-quad stride spreads a warp's 32 stores
// over the 32 banks); every 8-row k step issues  D += A_hi.B_hi + A_lo.B_hi + A_hi.B_lo  with M = 128 output
// features of dZ_l and N <= 256 input features of A_{l-1}.
//
// One CTA = (layer, 128-feature tile of dZ_l, 256-feature tile of A_{l-1}, batch slab); the
// slabs are summed later by the Adam kernel in slab order (deterministic), exactly like the
// mma.sync kernel in rb200_optim.cu, which stays the default (RB200_WGRAD_TC=1 selects this one
// for every layer).  Two smem stages; the loads of chunk c+1 are in flight while chunk c's MMAs run.
#include <stdlib.h>

#include "rb200_umma.cuh"

namespace rb200 {

constexpr int kWtRows = 32;                       // batch rows per stage = 4 MMA k steps
constexpr int kWtM = 128;                         // dZ features per tile (UMMA M)
constexpr int kWtN = 256;                         // input features per tile (UMMA N, TMEM columns)
constexpr int kWtQuadA = kWtM * 16 + 16;          // bytes per 4-row group of the dZ operand
constexpr int kWtQuadB = kWtN * 16 + 16;          // ... of the activation operand
constexpr int kWtPlaneA = (kWtRows / 4) * kWtQuadA;
constexpr int kWtPlaneB = (kWtRows / 4) * kWtQuadB;
constexpr int kWtStage = 2 * (kWtPlaneA + kWtPlaneB);  // A_hi, A_lo, B_hi, B_lo
constexpr int kWtThreads = 256;
constexpr int kWtSmem = 2 * kWtStage + 64;

struct WtLayer {
  const float* A;   // [B, K]
  const float* dZ;  // [B, N]
  int K, N;
  long long w_off, b_off;
  int tiles_m, tiles_k, job_start;
};
struct WtParams {
  int dbg;  // profiling only: 1 skip the loads, 2 skip the split, 4 skip the MMAs, 8 skip the epilogue stores
  int n_layers;
  WtLayer L[kMaxLayers];
  int B, rows_per_split;
  float* gpart;
  long long P;
};

__global__ void __launch_bounds__(kWtThreads, 1) wgrad_tc_kernel(const WtParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int li = 0;
  while (li + 1 < p.n_layers && (int)blockIdx.x >= p.L[li + 1].job_start) ++li;
  const WtLayer& Ly = p.L[li];
  const int job = blockIdx.x - Ly.job_start;
  const int tm = job / Ly.tiles_k, tk = job - tm * Ly.tiles_k;
  const int n0 = tm * kWtM, k0 = tk * kWtN;
  const int N = Ly.N, K = Ly.K;
  const int nrows_m = min(kWtM, N - n0);             // valid dZ features of this tile
  const int ncols = min(kWtN, K - k0);               // valid input features of this tile
  const int n_mma = (ncols + 15) & ~15;              // UMMA N (multiple of 16 for M = 128)
  const int split = blockIdx.y;
  const int b_begin = split * p.rows_per_split;
  const int b_end = min(p.B, b_begin + p.rows_per_split);
  const int nchunks = ceil_div(max(b_end - b_begin, 0), kWtRows);

  uint64_t* mma_done = reinterpret_cast<uint64_t*>(smem + 2 * kWtStage);  // [2] stage reusable
  uint64_t* acc_done = mma_done + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_done + 1);

  // No zero-fill of the stages: every staged feature row is rewritten per chunk (zeros past the
  // slab end); features past the matrix are never written, and whatever they hold only reaches
  // accumulator rows / columns that are not stored (D[m][n] depends on A row m and B row n only).
  if (tid == 0) {
    mbar_init(mma_done, 1);
    mbar_init(mma_done + 1, 1);
    mbar_init(acc_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                     smem_u32(tmem_slot)), "n"(kWtN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // A chunk (32 batch rows) is moved in "units" of 16 rows x 8 features: lane = (row, 4-feature
  // piece) loads one float4 (16 rows x 32 B: whole sectors), splits it into TF32 hi / lo and
  // stores the 2 x 4 scalars transposed into the K-major planes -- element (row r, feature f)
  // at [r / 4][f][r % 4].  With the 16-byte padded row-quad stride the 32 stores of a warp hit
  // 32 different banks.  Units of a chunk: 2 halves x (feature pairs of A + of B), dealt to the
  // 8 warps round-robin; the loads of chunk c+1 are in flight while chunk c's MMAs run.
  const int fa = (nrows_m + 7) & ~7, fb = (ncols + 7) & ~7;  // staged features (multiples of 8)
  const int ua = 2 * (fa / 8), utotal = ua + 2 * (fb / 8);
  constexpr int kMaxUnits = (2 * (kWtM / 8) + 2 * (kWtN / 8)) / (kWtThreads / 32);  // 12
  const int r_l = lane & 15, qsel = lane >> 4;
  float4 regs[kMaxUnits];
  auto chunk_fetch = [&](int c) {
    const int r0 = b_begin + c * kWtRows;
#pragma unroll
    for (int u = 0; u < kMaxUnits; ++u) {
      const int unit = warp + u * (kWtThreads / 32);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (unit < utotal && !(p.dbg & 1)) {
        const bool isb = unit >= ua;
        const int j = isb ? unit - ua : unit;
        const int h = j & 1, fp = j >> 1;
        const int row = r0 + 16 * h + r_l;
        const int f = (isb ? k0 : n0) + 8 * fp + 4 * qsel;
        const int F = isb ? K : N;
        if (row < b_end && f < F) {
          const float* src = (isb ? Ly.A : Ly.dZ) + (size_t)row * F + f;
          if (f + 3 < F && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
            v = __ldg(reinterpret_cast<const float4*>(src));
          } else {
            v.x = src[0];
            if (f + 1 < F) v.y = src[1];
            if (f + 2 < F) v.z = src[2];
            if (f + 3 < F) v.w = src[3];
          }
        }
      }
      regs[u] = v;
    }
  };
  auto chunk_store = [&](int st) {
    unsigned char* base = smem + st * kWtStage;
#pragma unroll
    for (int u = 0; u < kMaxUnits; ++u) {
      const int unit = warp + u * (kWtThreads / 32);
      if (unit >= utotal) continue;
      const bool isb = unit >= ua;
      const int j = isb ? unit - ua : unit;
      const int h = j & 1, fp = j >> 1;
      const int r = 16 * h + r_l;
      const int fl = 8 * fp + 4 * qsel;
      float* hi = reinterpret_cast<float*>(base + (isb ? 2 * kWtPlaneA + (r >> 2) * kWtQuadB
                                                       : (r >> 2) * kWtQuadA) + fl * 16) + (r & 3);
      float* lo = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(hi) + (isb ? kWtPlaneB : kWtPlaneA));
      float4 hh, ll;
      split4(regs[u], hh, ll);
      hi[0] = hh.x; hi[4] = hh.y; hi[8] = hh.z; hi[12] = hh.w;
      lo[0] = ll.x; lo[4] = ll.y; lo[8] = ll.z; lo[12] = ll.w;
    }
  };
  // bias gradient: column sums of dZ over the chunk (hi + lo is the exact value)
  float bsum = 0.f;
  auto chunk_bias = [&](int st) {
    if (tk != 0 || tid >= kWtM) return;
    const unsigned char* base = smem + st * kWtStage;
#pragma unroll
    for (int rq = 0; rq < kWtRows / 4; ++rq) {
      const float4 a = *reinterpret_cast<const float4*>(base + rq * kWtQuadA + tid * 16);
      const float4 b = *reinterpret_cast<const float4*>(base + kWtPlaneA + rq * kWtQuadA + tid * 16);
      bsum += ((a.x + b.x) + (a.y + b.y)) + ((a.z + b.z) + (a.w + b.w));
    }
  };

  const uint32_t idesc = umma_idesc_tf32(kWtM, n_mma);
  uint32_t done_par[2] = {0u, 0u};
  if (nchunks > 0) chunk_fetch(0);
  for (int c = 0; c < nchunks; ++c) {
    const int st = c & 1;
    if (c >= 2) {  // the MMAs of chunk c-2 read this stage
      mbar_wait(mma_done + st, done_par[st]);
      done_par[st] ^= 1u;
    }
    if (!(p.dbg & 2)) chunk_store(st);
    if (c + 1 < nchunks) chunk_fetch(c + 1);  // in flight during the barrier and the MMAs
    fence_proxy_async_smem();
    __syncthreads();
    chunk_bias(st);
    if (tid == 0) {
      tc_fence_after();
      const uint32_t sb = smem_u32(smem + st * kWtStage);
      const uint32_t a_hi = sb, a_lo = sb + kWtPlaneA, b_hi = sb + 2 * kWtPlaneA, b_lo = b_hi + kWtPlaneB;
#pragma unroll
      for (int ks = 0; ks < ((p.dbg & 4) ? 0 : kWtRows / 8); ++ks) {
        // K-major no-swizzle: leading offset = next 4-row group, stride offset = 8 features
        const uint32_t oa = ks * 2 * kWtQuadA, ob = ks * 2 * kWtQuadB;
        const uint64_t dah = umma_desc(a_hi + oa, kWtQuadA, 128), dal = umma_desc(a_lo + oa, kWtQuadA, 128);
        const uint64_t dbh = umma_desc(b_hi + ob, kWtQuadB, 128), dbl = umma_desc(b_lo + ob, kWtQuadB, 128);
        umma_tf32(tmem, dah, dbh, idesc, (c > 0 || ks > 0) ? 1u : 0u);
        umma_tf32(tmem, dal, dbh, idesc, 1u);
        umma_tf32(tmem, dah, dbl, idesc, 1u);
      }
      umma_commit(mma_done + st);
      if (c == nchunks - 1) umma_commit(acc_done);
    }
  }

  // ---- epilogue: accumulator -> shared memory (the operand stages are dead) -> this slab's
  // gradient partial with coalesced 16-byte stores (a thread owns a TMEM lane = a row of dW;
  // writing it straight out would be 4-byte pieces 1 KB apart) ----
  float* gp = p.gpart + (size_t)split * p.P;
  constexpr int kLdT = kWtN + 4;  // floats per staged row: 16-byte aligned, conflict-free
  float* tile = reinterpret_cast<float*>(smem);
  if (nchunks > 0) {
    mbar_wait(acc_done, 0);
    tc_fence_after();
  }
  if (warp < 4) {
    const int nl = warp * 32 + lane;
    for (int c0 = 0; c0 < n_mma; c0 += 16) {
      uint32_t v[16];
      if (nchunks > 0) {
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
              "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
              "=r"(v[14]), "=r"(v[15])
            : "r"(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0));
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0u;
      }
      float4* d = reinterpret_cast<float4*>(tile + (size_t)nl * kLdT + c0);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        d[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                           __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
    }
    if (tk == 0 && n0 + nl < N) gp[Ly.b_off + n0 + nl] = bsum;
  }
  __syncthreads();
  {
    const bool v4 = ((K & 3) == 0) && ((k0 & 3) == 0) && ((Ly.w_off & 3) == 0) &&
                    ((reinterpret_cast<uintptr_t>(gp) & 15) == 0);
    for (int r = warp; r < ((p.dbg & 8) ? 0 : nrows_m); r += kWtThreads / 32) {
      float* dst = gp + Ly.w_off + (size_t)(n0 + r) * K + k0;
      const float* src = tile + (size_t)r * kLdT;
      if (v4) {
        for (int c = lane * 4; c < ncols; c += 128)
          *reinterpret_cast<float4*>(dst + c) = *reinterpret_cast<const float4*>(src + c);
      } else {
        for (int c = lane; c < ncols; c += 32) dst[c] = src[c];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "n"(kWtN));
  }
}

}  // namespace rb200

using namespace rb200;

// Launch the tcgen05 weight-gradient kernel.  Any layer shape fits (128 x 256 feature tiles,
// 32-row batch chunks, fixed shared-memory size), so there is no shape check here; a launch or
// opt-in error is returned as is: rb200_mlp_wgrad does not fall back to the mma.sync kernel.
int rb200_wgrad_tc_launch(const rb200_mlp_t* net, const float* net_input, int32_t batch,
                          const rb200_net_ws_t* ws, float* gpart, int32_t splits, void* stream) {
  WtParams p = {};
  { const char* e = getenv("RB200_WT_DBG"); p.dbg = e ? atoi(e) : 0; }
  p.n_layers = net->n_layers;
  p.B = batch;
  p.rows_per_split = ceil_div(ceil_div(batch, splits), kWtRows) * kWtRows;
  p.gpart = gpart;
  p.P = net->n_params;
  int jobs = 0;
  for (int l = 0; l < net->n_layers; ++l) {
    WtLayer& L = p.L[l];
    L.A = (l == 0) ? (net_input ? net_input : ws->input) : ws->hidden[l - 1];
    L.dZ = ws->dz[l];
    if (!L.A || !L.dZ) { set_last_error("rb200_mlp_wgrad: missing activation / dz for layer %d", l); return RB200_E_INVALID; }
    L.K = net->dims[l];
    L.N = net->dims[l + 1];
    L.w_off = net->w_off[l];
    L.b_off = net->b_off[l];
    L.tiles_m = ceil_div(L.N, kWtM);
    L.tiles_k = ceil_div(L.K, kWtN);
    L.job_start = jobs;
    jobs += L.tiles_m * L.tiles_k;
  }
  for (int l = net->n_layers; l < kMaxLayers; ++l) p.L[l].job_start = 1 << 30;
  static SmemOptIn optin = {};
  {
    cudaError_t e = ensure_dynamic_smem(wgrad_tc_kernel, optin, (size_t)kWtSmem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(wgrad_tc)");
  }
  dim3 grid(jobs, splits);
  wgrad_tc_kernel<<<grid, kWtThreads, kWtSmem, (cudaStream_t)stream>>>(p);
  return check_cuda(cudaGetLastError(), "wgrad_tc_kernel launch");
}
