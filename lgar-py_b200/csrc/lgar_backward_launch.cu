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

template <int FM, int GM>
static int launch_backward(BParams& P, int S, int chunk, int slots, int arena_cap, int step_cap, int num_sms,
                           unsigned char* scratch, cudaStream_t st, char* err, size_t errlen) {
  auto kern = lgar_backward_kernel<FM, GM>;
  const size_t smem = (size_t)5 * FM * NT * sizeof(double) + (size_t)WARPS * NODEBUF * sizeof(double) +
                      (size_t)5 * FM * NT * sizeof(short) + (size_t)FM * NT;
  BW_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  BW_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NT, smem));
  if (per_sm < 1) {
    std::snprintf(err, errlen, "backward kernel does not fit on an SM");
    return LGAR_E_CUDA;
  }
  long long grid = (long long)num_sms * per_sm;
  if (grid > slots / WARPS) grid = slots / WARPS;
  if (grid < 1) grid = 1;
  const int ntiles = P.K.ntiles;
  const size_t ring_steps = (size_t)chunk * S;
  const size_t nl = num_leaves<FM>();
  size_t o = 0;
  auto take = [&](size_t bytes) { unsigned char* q = scratch + o; o += (bytes + 255) / 256 * 256; return q; };
  P.tape = (TapeEntry*)take((size_t)slots * arena_cap * 32 * sizeof(TapeEntry));
  P.meta = (unsigned char*)take((size_t)slots * ring_steps * 32 * sizeof(StepMeta<FM>));
  P.adj = (double*)take((size_t)slots * (nl + step_cap) * 32 * 8);
  P.lam = (double*)take((size_t)ntiles * nl * 32 * 8);
  P.gpar = (double*)take((size_t)ntiles * NPAR_IDS * 32 * 8);
  P.rev_flags = (int32_t*)take((size_t)ntiles * 32 * 4);
  P.rev_done = (int32_t*)take((size_t)ntiles * 4);
  P.next_tile = (unsigned long long*)take(64);
  P.ring_steps = (int32_t)ring_steps;
  P.arena_cap = arena_cap;
  P.step_cap = step_cap;
  BW_TRY(cudaMemsetAsync(P.next_tile, 0, 64, st));
  BW_TRY(cudaMemsetAsync(P.rev_done, 0, (size_t)ntiles * 4, st));
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

// opaque-pointer entry used by lgar_capi.cu (BParams has the same layout in both units: same header)
int lgar_reverse_unit_launch(int FM, void* params, int S, int chunk, int slots, int arena_cap, int step_cap, int num_sms,
                             unsigned char* scratch, void* stream, char* err, size_t errlen) {
  using namespace lgar;
  BParams& P = *static_cast<BParams*>(params);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (FM == 8) return launch_backward<8, 2>(P, S, chunk, slots, arena_cap, step_cap, num_sms, scratch, st, err, errlen);
  if (FM == 12) return launch_backward<12, 2>(P, S, chunk, slots, arena_cap, step_cap, num_sms, scratch, st, err, errlen);
  // the default configuration gets a trapezoid-only instantiation (hot-path code size, see DESIGN.md 4.1)
  if (P.K.p.use_closed_form_G) return launch_backward<16, 2>(P, S, chunk, slots, arena_cap, step_cap, num_sms, scratch, st, err, errlen);
  return launch_backward<16, 0>(P, S, chunk, slots, arena_cap, step_cap, num_sms, scratch, st, err, errlen);
}
