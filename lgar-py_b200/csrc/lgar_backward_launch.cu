// =====================================================================================
// lgar_backward_launch.cu -- the reverse-mode kernel's own translation unit.
// Compiled separately from lgar_capi.cu (forward kernel): the two units compile in parallel (half the build time)
// and can make different code-generation trade-offs (e.g. pow-table placement, see lgar_pow.cuh).
// =====================================================================================
// every header symbol of this unit lives in its own namespace: the host-side stubs of the __device__ functions
// would otherwise collide with the forward unit's at link time (and the two units compile them differently)
#define lgar lgar_reverse_unit
#include <cstdio>

#include "lgar_backward.cuh"

namespace lgar {

#define BW_TRY(expr)                                                                      \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      std::snprintf(err, errlen, "%s failed: %s", #expr, cudaGetErrorString(e__));        \
      return LGAR_E_CUDA;                                                                 \
    }                                                                                     \
  } while (0)

// second stage of the shared-parameter reduction: block q sums partials[.][q] over the tiles in a fixed order
// (lane j takes tiles j, j+32, ... sequentially, then a butterfly over the 32 lane sums)
__global__ void lgar_reduce_tile_partials(const double* partials, int ntiles, int L, double* grad_alpha, double* grad_n,
                                          double* grad_ksat, double* grad_pdm) {
  const int q = blockIdx.x;  // 3 l + {0: alpha, 1: n, 2: ksat}
  double s = 0.0;
  for (int t = threadIdx.x; t < ntiles; t += 32) s += partials[(size_t)t * NPAR_IDS + q];
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if (threadIdx.x == 0) {
    const int l = q / 3;
    if (q == ID_PDM) {
      if (grad_pdm) grad_pdm[0] = s;
    } else if (l < L) {
      double* out = (q % 3 == 0) ? grad_alpha : ((q % 3 == 1) ? grad_n : grad_ksat);
      out[l] = s;
    }
  }
}

// resident warps that own a scratch slot.  Bounded by 160 SMs rather than the device's SM count, so that
// lgar_workspace_bytes needs no device.
static int scratch_slots(const KParams& K) {
  long long want = ((long long)K.ntiles * K.nchunks + WARPS - 1) / WARPS;
  long long grid = 160LL * BACKWARD_CTAS_PER_SM;
  if (grid > want) grid = want;
  return (int)grid * WARPS;
}

// Scratch of the reverse kernel, laid out from `scratch` (nullptr: sizing only): per slot the tape arena, the StepMeta
// ring and the adjoints; per tile the adjoint state and the parameter gradients between chunks, the overflow flags and
// the progress counter; then the item counter.  Reads the shape and the tape budget from P, sets P's scratch pointers
// and returns the bytes they span.
template <int FM>
static size_t carve_scratch(BParams& P, unsigned char* scratch) {
  const size_t slots = scratch_slots(P.K), ntiles = P.K.ntiles, nl = num_leaves<FM>();
  size_t o = 0;
  P.tape = at<TapeEntry>(scratch, o);               o = align_up(o + slots * P.arena_cap * 32 * sizeof(TapeEntry));
  P.meta = at<unsigned char>(scratch, o);           o = align_up(o + slots * P.ring_steps * 32 * sizeof(StepMeta<FM>));
  P.adj = at<double>(scratch, o);                   o = align_up(o + slots * (nl + P.step_cap) * 32 * sizeof(double));
  P.lam = at<double>(scratch, o);                   o = align_up(o + ntiles * nl * 32 * sizeof(double));
  P.gpar = at<double>(scratch, o);                  o = align_up(o + ntiles * NPAR_IDS * 32 * sizeof(double));
  P.rev_flags = at<int32_t>(scratch, o);            o = align_up(o + ntiles * 32 * sizeof(int32_t));
  P.rev_done = at<int32_t>(scratch, o);             o = align_up(o + ntiles * sizeof(int32_t));
  P.next_tile = at<unsigned long long>(scratch, o); o = align_up(o + 64);
  return o;
}

template <int FM, int GM>
static int launch_backward(const BParams& P, int num_sms, cudaStream_t st, char* err, size_t errlen) {
  auto kern = lgar_backward_kernel<FM, GM>;
  constexpr size_t smem = backward_smem_bytes<FM>();
  BW_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  BW_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NT, smem));
  if (per_sm < 1) {
    std::snprintf(err, errlen, "backward kernel does not fit on an SM");
    return LGAR_E_CUDA;
  }
  const int slots = scratch_slots(P.K);
  long long grid = (long long)num_sms * per_sm;
  if (grid > slots / WARPS) grid = slots / WARPS;
  if (grid < 1) grid = 1;
  BW_TRY(cudaMemsetAsync(P.next_tile, 0, 64, st));
  BW_TRY(cudaMemsetAsync(P.rev_done, 0, (size_t)P.K.ntiles * 4, st));
  kern<<<(unsigned)grid, NT, smem, st>>>(P);
  BW_TRY(cudaGetLastError());
  if (P.reduce) {
    lgar_reduce_tile_partials<<<NPAR_IDS, 32, 0, st>>>(P.partials, P.K.ntiles, P.K.p.num_layers, P.grad_alpha, P.grad_n,
                                                      P.grad_ksat, P.grad_pdm);
    BW_TRY(cudaGetLastError());
  }
  return 0;
}

}  // namespace lgar

// opaque-pointer entries used by lgar_capi.cu (BParams has the same layout in both units: same header)
size_t lgar_reverse_unit_scratch(int FM, void* params, unsigned char* scratch) {
  using namespace lgar;
  BParams& P = *static_cast<BParams*>(params);
  if (FM == 8) return carve_scratch<8>(P, scratch);
  if (FM == 12) return carve_scratch<12>(P, scratch);
  if (FM == 16) return carve_scratch<16>(P, scratch);
  return 0;  // max_fronts = 32 is forward-only: there is no reverse kernel to give scratch to
}

int lgar_reverse_unit_launch(int FM, const void* params, int num_sms, void* stream, char* err, size_t errlen) {
  using namespace lgar;
  const BParams& P = *static_cast<const BParams*>(params);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (FM == 8) return launch_backward<8, 2>(P, num_sms, st, err, errlen);
  if (FM == 12) return launch_backward<12, 2>(P, num_sms, st, err, errlen);
  // the default configuration gets a trapezoid-only instantiation (hot-path code size, see DESIGN.md 4.1)
  if (P.K.p.use_closed_form_G) return launch_backward<16, 2>(P, num_sms, st, err, errlen);
  return launch_backward<16, 0>(P, num_sms, st, err, errlen);
}
