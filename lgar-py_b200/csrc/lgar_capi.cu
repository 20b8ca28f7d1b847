// =====================================================================================
// lgar_capi.cu -- extern "C" entry points declared in include/lgar_b200.h.
// Host-side only does argument checking, workspace carving and ONE kernel launch per call.
// There is no CPU fallback: without an sm_100 device every compute entry point fails.
// =====================================================================================
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "lgar_forward.cuh"
#include "lgar_backward.cuh"

// the reverse kernel is compiled in its own translation unit (lgar_backward_launch.cu)
size_t lgar_reverse_unit_scratch(int FM, void* params, unsigned char* scratch);
int lgar_reverse_unit_launch(int FM, const void* params, int num_sms, void* stream, char* err, size_t errlen);

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, const char* detail = "") {
  std::snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}
#define CUDA_TRY(expr)                                                         \
  do {                                                                         \
    cudaError_t e__ = (expr);                                                  \
    if (e__ != cudaSuccess) {                                                  \
      std::snprintf(g_err, sizeof(g_err), "%s failed: %s", #expr, cudaGetErrorString(e__)); \
      return LGAR_E_CUDA;                                                      \
    }                                                                          \
  } while (0)

struct Shape {
  int B, Bp, L, T, S, FM, chunk, nchunks, ntiles;
  int t_begin, t_end;  // window of forcing rows (whole record: 0, T)
};

enum Entry { WORKSPACE_BYTES, FORWARD, BACKWARD };

// The argument rules of lgar_workspace_bytes, lgar_forward and lgar_backward_ex, checked before the device and before
// anything is enqueued.  `with_grad`: the call sizes, writes or reads checkpoints.  Fills s; returns the first rule
// the call breaks (0: none).
int check_args(Entry entry, const lgar_problem* p, int with_grad, const lgar_outputs* out, const lgar_gradients* g,
               Shape& s) {
  if (!p) return fail(LGAR_E_INVALID, "problem is NULL");
  if (p->abi_version != LGAR_ABI_VERSION) return fail(LGAR_E_INVALID, "abi_version mismatch");
  if (p->num_columns < 1 || p->num_steps < 1 || p->num_subcycles < 1) return fail(LGAR_E_INVALID, "empty problem");
  if (p->num_layers < 1 || p->num_layers > LGAR_MAX_LAYERS) return fail(LGAR_E_INVALID, "num_layers out of range");
  if (p->nint < 1 || p->nint > 128) return fail(LGAR_E_INVALID, "nint must be in [1,128]");
  if (p->num_giuh < 1 || p->num_giuh > LGAR_MAX_GIUH) return fail(LGAR_E_INVALID, "num_giuh out of range");
  s.B = p->num_columns;
  s.Bp = (s.B + 31) / 32 * 32;
  s.L = p->num_layers;
  s.T = p->num_steps;
  s.S = p->num_subcycles;
  s.FM = p->max_fronts == 0 ? 16 : p->max_fronts;
  if (s.FM != 8 && s.FM != 12 && s.FM != 16 && s.FM != 32)
    return fail(LGAR_E_INVALID, "max_fronts must be 8, 12, 16 or 32");
  // default: 64 sub-steps per scheduling / checkpoint chunk (64 forcing steps at S = 1, 5 at S = 12), which also
  // bounds the tape arena of the reverse pass (one chunk of sub-steps per resident warp)
  s.chunk = p->chunk_steps > 0 ? p->chunk_steps : (64 / s.S > 0 ? 64 / s.S : 1);
  s.t_begin = 0;
  s.t_end = s.T;
  if (p->step_begin != 0 || p->step_end != 0) {
    if (p->step_begin < 0 || p->step_end <= p->step_begin || p->step_end > s.T)
      return fail(LGAR_E_INVALID, "step window must satisfy 0 <= step_begin < step_end <= num_steps");
    s.t_begin = p->step_begin;
    s.t_end = p->step_end;
  }
  s.nchunks = (s.t_end - s.t_begin + s.chunk - 1) / s.chunk;
  s.ntiles = s.Bp / 32;
  if (with_grad && (long long)s.chunk * s.S > 512)
    return fail(LGAR_E_INVALID, "chunk_steps * num_subcycles > 512 with checkpoints: the tape arena of the reverse "
                                "pass (one chunk of sub-steps per resident warp) would not fit; use chunk_steps = 0 "
                                "(default) or a smaller value");
  if (entry == WORKSPACE_BYTES) return 0;
  if (s.FM == 32 && with_grad) return fail(LGAR_E_INVALID, "max_fronts = 32 is forward-only (no checkpoints)");
  if (with_grad && (s.t_begin != 0 || s.t_end != s.T))
    return fail(LGAR_E_INVALID, "a step window (step_begin, step_end) is forward-only: checkpoints and lgar_backward "
                                "need the whole record");
  if (p->num_depths < 0 || p->num_depths > LGAR_MAX_DEPTHS)
    return fail(LGAR_E_INVALID, "num_depths must be in [0, LGAR_MAX_DEPTHS]");
  for (int d = 0; d < p->num_depths; d++)
    if (!(std::isfinite(p->moisture_depths[d]) && p->moisture_depths[d] > 0.0))
      return fail(LGAR_E_INVALID, "moisture_depths: every used depth must be finite and > 0");
  if (entry == BACKWARD) {
    if (!g) return fail(LGAR_E_INVALID, "gradients is NULL");
    if (g->grad_moisture && p->num_depths == 0)
      return fail(LGAR_E_INVALID, "grad_moisture needs num_depths > 0");
    if (!g->grad_alpha || !g->grad_n || !g->grad_ksat)
      return fail(LGAR_E_INVALID, "a gradient output array (grad_alpha, grad_n, grad_ksat) is NULL");
    if (g->reduce && !g->partials) return fail(LGAR_E_INVALID, "reduce needs the partials scratch array");
    return 0;
  }
  if (!out) return fail(LGAR_E_INVALID, "outputs is NULL");
  if (!p->alpha || !p->n || !p->ksat || !p->theta_r || !p->theta_e || !p->thickness || !p->initial_psi ||
      !p->ponded_depth_max || !p->forcing)
    return fail(LGAR_E_INVALID, "a required problem array is NULL");
  if (p->num_sites < 1) return fail(LGAR_E_INVALID, "num_sites < 1");
  if (p->resume && with_grad) return fail(LGAR_E_INVALID, "resume is not available with keep_checkpoints");
  if (s.t_begin != 0 && !p->resume) return fail(LGAR_E_INVALID, "step_begin > 0 needs resume = 1");
  if (p->pipeline_seq < 0 || p->pipeline_seq >= (1 << 23)) return fail(LGAR_E_INVALID, "pipeline_seq out of range");
  if (p->pipeline_seq > 0 && with_grad) return fail(LGAR_E_INVALID, "pipeline_seq > 0 is forward-only");
  if (p->pipeline_seq > 1 && !p->resume) return fail(LGAR_E_INVALID, "pipeline_seq > 1 needs resume = 1");
  if (out->fronts && s.FM != 16) return fail(LGAR_E_INVALID, "front dumps (outputs.fronts) need max_fronts = 16");
  if (out->moisture && p->num_depths == 0) return fail(LGAR_E_INVALID, "outputs.moisture needs num_depths > 0");
  return 0;
}

struct Carve {
  size_t off_d, off_i, off_f, off_slog, off_slogc, off_done, off_item, total;
  int slog_cap;
};
// search log of the reverse pass (KParams::slog): average budget of entries per sub-step and lane; a lane that needs
// more in some chunk searches again from there on (correct, just slower)
#define LGAR_SLOG_AVG 5

Carve carve(const Shape& s, int with_grad) {
  using lgar::align_up;
  const size_t nck = with_grad ? (size_t)s.nchunks + 1 : 1;
  const size_t nd = 5 * (size_t)s.FM + lgar::S_COUNT;
  Carve c;
  size_t o = 0;
  c.off_d = o;   o = align_up(o + nck * nd * s.Bp * sizeof(double));
  c.off_i = o;   o = align_up(o + nck * lgar::NI_STATE * s.Bp * sizeof(int32_t));
  c.off_f = o;   o = align_up(o + nck * (size_t)s.FM * s.Bp);
  c.slog_cap = with_grad ? s.chunk * s.S * LGAR_SLOG_AVG : 0;
  c.off_slog = o;  o = align_up(o + (with_grad ? (size_t)s.nchunks * c.slog_cap * s.Bp * sizeof(double) : 0));
  c.off_slogc = o; o = align_up(o + (with_grad ? (size_t)s.nchunks * s.Bp * sizeof(int32_t) : 0));
  c.off_done = o; o = align_up(o + (size_t)s.ntiles * sizeof(int32_t));
  c.off_item = o; o = align_up(o + 64);
  c.total = o;
  return c;
}

// the kernel parameters both passes share; the settings of one pass are made by its caller
lgar::KParams kparams(const lgar_problem* p, const Shape& s, const Carve& c, unsigned char* w) {
  lgar::KParams K;
  std::memset(&K, 0, sizeof(K));
  K.p = *p;
  K.state_d = lgar::at<double>(w, c.off_d);
  K.state_i = lgar::at<int32_t>(w, c.off_i);
  K.state_f = lgar::at<uint8_t>(w, c.off_f);
  K.done = lgar::at<int32_t>(w, c.off_done);
  K.next_item = lgar::at<unsigned long long>(w, c.off_item);
  K.Bp = s.Bp;
  K.ntiles = s.ntiles;
  K.nchunks = s.nchunks;
  K.chunk_steps = s.chunk;
  K.iter_cap = p->iter_cap > 0 ? p->iter_cap : 1000000;
  return K;
}

int g_dev_checked = -2;
int g_num_sms = 0;

int ensure_device() {
  int dev = -1;
  if (cudaGetDevice(&dev) == cudaSuccess && dev == g_dev_checked) return 0;
  return lgar_device_check();
}

// Tape budget of the reverse pass.  step_cap: entries one sub-step may record; step_cap + leaves must stay below 32768
// because tape ids are stored as 16 bit in shared memory.  arena_cap: entries of one chunk per lane, on average 640 per
// sub-step (bench ensemble: 83 per sub-step on average, heavy-tailed; 320 overflows 0.1 % of the columns), and at
// least step_cap.  An exhausted arena flags the column (NaN gradient + tape_overflow).  LGAR_DEBUG_TAPE_CAP (tests
// only) sets step_cap and shrinks the arena to it, to provoke the overflow path
// (tests/test_gpu_gradients.py::test_tape_overflow_is_reported).
void set_tape_budget(lgar::BParams& P, const Shape& s) {
  constexpr int TAPE_CAP_MAX = 6144, TAPE_AVG = 640;
  const char* e = std::getenv("LGAR_DEBUG_TAPE_CAP");
  const int v = e ? std::atoi(e) : 0;
  P.step_cap = (v >= 16 && v <= TAPE_CAP_MAX) ? v : TAPE_CAP_MAX;
  P.arena_cap = e ? P.step_cap : std::max(s.chunk * s.S * TAPE_AVG, P.step_cap);  // chunk * S <= 512 (checked)
}

// Everything the reverse kernel reads except the caller's gradient arguments, over workspace w (nullptr: sizing only).
// Returns the bytes of workspace the reverse pass needs.
size_t backward_params(const lgar_problem* p, const Shape& s, unsigned char* w, lgar::BParams& P) {
  const Carve c = carve(s, 1);
  std::memset(&P, 0, sizeof(P));
  lgar::KParams& K = P.K;
  K = kparams(p, s, c, w);
  K.t_begin = 0;
  K.t_end = s.T;
  K.keep_ckpt = 1;
  K.slog = lgar::at<double>(w, c.off_slog);
  K.slog_count = lgar::at<int32_t>(w, c.off_slogc);
  K.slog_cap = c.slog_cap;
  P.ring_steps = s.chunk * s.S;
  set_tape_budget(P, s);
  return c.total + lgar_reverse_unit_scratch(s.FM, &P, lgar::at<unsigned char>(w, c.total));
}

// Launch plan of one lgar_forward call.  `pipeline_seq` k > 1 asks for a programmatic dependent launch behind
// window k-1 (no host memset between the kernels; see KParams::seq).  That is only sound while every launch of
// the sequence fills the device: then launch k-2 has left the SMs before launch k can become resident, so a ring
// of three ticket words is enough.  Smaller grids fall back to ordinary stream-ordered launches.
struct Plan {
  lgar::KParams K;
  const Carve* carve;
  unsigned char* w;
  int pipeline_seq;
};

template <int FM, bool COUNT, bool DUMP, bool LOGW = false>
int launch_forward(Plan& P, cudaStream_t st) {
  lgar::KParams& K = P.K;
  auto kern = lgar::lgar_forward_kernel<FM, COUNT, DUMP, LOGW>;
  constexpr size_t smem = lgar::forward_smem_bytes<FM>();
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, lgar::NT, smem));
  if (per_sm < 1) return fail(LGAR_E_CUDA, "forward kernel does not fit on an SM");
  long long want = ((long long)K.ntiles * K.nchunks + lgar::WARPS - 1) / lgar::WARPS;
  const long long full = (long long)g_num_sms * per_sm;
  long long grid = full;
  if (grid > want) grid = want;
  if (grid < 1) grid = 1;
  const bool pipelined = P.pipeline_seq >= 1 && grid == full;
  const bool overlap = pipelined && P.pipeline_seq > 1;
  K.seq = pipelined ? P.pipeline_seq : 0;
  K.slot = pipelined ? P.pipeline_seq % 3 : 0;
  K.overlap = overlap ? 1 : 0;
  if (!overlap)  // progress counters and ticket words start from zero (stream-ordered before the kernel)
    CUDA_TRY(cudaMemsetAsync(P.w + P.carve->off_done, 0, P.carve->total - P.carve->off_done, st));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(lgar::NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = overlap ? 1 : 0;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, K));
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---- host-buffer variant ------------------------------------------------------------
struct DevBuf {
  std::vector<void*> ptrs;
  struct Download { void* host; const void* dev; size_t bytes; };
  std::vector<Download> downloads;
  ~DevBuf() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <class T>
  int up(const T* host, size_t count, const T** dev_out) {
    *dev_out = nullptr;
    if (!host) return 0;
    void* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, count * sizeof(T)));
    ptrs.push_back(d);
    CUDA_TRY(cudaMemcpy(d, host, count * sizeof(T), cudaMemcpyHostToDevice));
    *dev_out = (const T*)d;
    return 0;
  }
  // device buffer for an output, copied back to `host` by download()
  template <class T>
  int out(T* host, size_t count, T** dev_out) {
    *dev_out = nullptr;
    if (!host) return 0;
    void* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, count * sizeof(T)));
    ptrs.push_back(d);
    downloads.push_back({host, d, count * sizeof(T)});
    *dev_out = (T*)d;
    return 0;
  }
  int download() {
    for (const Download& x : downloads) CUDA_TRY(cudaMemcpy(x.host, x.dev, x.bytes, cudaMemcpyDeviceToHost));
    return 0;
  }
};

}  // namespace

extern "C" {

int lgar_abi_version(void) { return LGAR_ABI_VERSION; }

const char* lgar_last_error_string(void) { return g_err; }

int lgar_device_check(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(LGAR_E_NO_DEVICE, "no CUDA device: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return fail(LGAR_E_NO_DEVICE, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10) return fail(LGAR_E_NO_DEVICE, "device is not sm_100 (B200): %s", prop.name);
  g_num_sms = prop.multiProcessorCount;
  g_dev_checked = dev;
  return 0;
}

size_t lgar_workspace_bytes(const lgar_problem* p, int with_grad) {
  Shape s;
  if (check_args(WORKSPACE_BYTES, p, with_grad, nullptr, nullptr, s)) return 0;
  if (!with_grad) return carve(s, 0).total;
  lgar::BParams P;
  return backward_params(p, s, nullptr, P);
}

int lgar_forward(const lgar_problem* p, const lgar_outputs* out, void* workspace_dev, size_t workspace_bytes,
                 int keep_checkpoints, void* stream) {
  Shape s;
  int rc = check_args(FORWARD, p, keep_checkpoints, out, nullptr, s);
  if (rc || (rc = ensure_device())) return rc;
  const Carve c = carve(s, keep_checkpoints);
  if (!workspace_dev || workspace_bytes < c.total) return fail(LGAR_E_WORKSPACE, "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* w = (unsigned char*)workspace_dev;

  Plan plan{kparams(p, s, c, w), &c, w, p->pipeline_seq};
  lgar::KParams& K = plan.K;
  K.o = *out;
  K.t_begin = s.t_begin;
  K.t_end = s.t_end;
  K.keep_ckpt = keep_checkpoints ? 1 : 0;
  // the search log is written by the default instantiation only (16 fronts, no counters); other configurations
  // leave it empty (slog_count = 0) and the reverse pass searches again
  const bool logw = keep_checkpoints && s.FM == 16 && !out->counters && !out->fronts && !p->use_closed_form_G;
  if (keep_checkpoints) {
    K.slog = (double*)(w + c.off_slog);
    K.slog_count = (int32_t*)(w + c.off_slogc);
    K.slog_cap = c.slog_cap;
    if (!logw) CUDA_TRY(cudaMemsetAsync(K.slog_count, 0, (size_t)s.nchunks * s.Bp * sizeof(int32_t), st));
  }
  if (p->pipeline_seq <= 1) {  // (a memset between two kernels of a pipelined sequence would serialise them)
    if (out->counters) CUDA_TRY(cudaMemsetAsync(out->counters, 0, 16 * sizeof(unsigned long long), st));
    if (out->tile_cycles)
      CUDA_TRY(cudaMemsetAsync(out->tile_cycles, 0, (size_t)(out->tile_diag_rows == 3 ? 3 : 1) * s.ntiles * sizeof(unsigned long long), st));
  }
  // the kernels without work counters are trapezoid-only (closed-form branch compiled out of the hot path)
  const bool count = out->counters != nullptr || p->use_closed_form_G != 0;
  if (out->fronts) return launch_forward<16, true, true>(plan, st);
  if (s.FM == 8) return count ? launch_forward<8, true, false>(plan, st) : launch_forward<8, false, false>(plan, st);
  if (s.FM == 12) return count ? launch_forward<12, true, false>(plan, st) : launch_forward<12, false, false>(plan, st);
  if (s.FM == 32) return launch_forward<32, true, false>(plan, st);  // large-capacity fallback (1 CTA per SM)
  if (logw) return launch_forward<16, false, false, true>(plan, st);
  return count ? launch_forward<16, true, false>(plan, st) : launch_forward<16, false, false>(plan, st);
}

int lgar_backward_ex(const lgar_problem* p, const lgar_gradients* g, void* workspace_dev, size_t workspace_bytes,
                     void* stream) {
  Shape s;
  int rc = check_args(BACKWARD, p, 1, nullptr, g, s);
  if (rc || (rc = ensure_device())) return rc;
  unsigned char* w = (unsigned char*)workspace_dev;
  lgar::BParams P;
  if (!w || workspace_bytes < backward_params(p, s, w, P))
    return fail(LGAR_E_WORKSPACE, "workspace too small for lgar_backward");
  P.grad_per_step = g->grad_per_step;
  P.grad_mask = g->grad_per_step ? g->grad_mask : 0;
  P.grad_sums = g->grad_sums;
  P.grad_alpha = g->grad_alpha;
  P.grad_n = g->grad_n;
  P.grad_ksat = g->grad_ksat;
  P.grad_pdm = g->grad_ponded_depth_max;
  P.grad_moisture = g->grad_moisture;
  P.grad_layer_water = g->grad_layer_water;
  P.tape_overflow = g->tape_overflow;
  P.reduce = g->reduce ? 1 : 0;
  P.partials = g->partials;
  P.counters = g->counters;
  P.K.time_phases = g->counters ? 1 : 0;
  if (g->counters) CUDA_TRY(cudaMemsetAsync(g->counters, 0, 8 * sizeof(unsigned long long), (cudaStream_t)stream));
  return lgar_reverse_unit_launch(s.FM, &P, g_num_sms, stream, g_err, sizeof(g_err));
}

int lgar_backward(const lgar_problem* p, const double* grad_per_step, uint32_t grad_mask, const double* grad_sums,
                  double* grad_alpha, double* grad_n, double* grad_ksat, void* workspace_dev, size_t workspace_bytes,
                  void* stream) {
  lgar_gradients g;
  std::memset(&g, 0, sizeof(g));
  g.grad_per_step = grad_per_step;
  g.grad_mask = grad_mask;
  g.grad_sums = grad_sums;
  g.grad_alpha = grad_alpha;
  g.grad_n = grad_n;
  g.grad_ksat = grad_ksat;
  return lgar_backward_ex(p, &g, workspace_dev, workspace_bytes, stream);
}

int lgar_forward_host(const lgar_problem* ph, const lgar_outputs* oh) {
  Shape s;
  int rc = check_args(FORWARD, ph, 0, oh, nullptr, s);
  if (rc || (rc = lgar_device_check())) return rc;
  DevBuf db;
  lgar_problem p = *ph;
  lgar_outputs o = *oh;
  const size_t LB = (size_t)s.L * s.B, B = s.B, T = s.T;
#define UP(field, count) if ((rc = db.up(ph->field, (count), &p.field))) return rc;
  UP(alpha, LB) UP(n, LB) UP(ksat, LB) UP(theta_r, LB) UP(theta_e, LB) UP(thickness, LB)
  UP(initial_psi, B) UP(ponded_depth_max, B) UP(forcing, (size_t)ph->num_sites * T * 2) UP(site_index, B) UP(column_order, B)
#undef UP
#define OUT(field, count) if ((rc = db.out(oh->field, (count), &o.field))) return rc;
  OUT(per_step, (size_t)__builtin_popcount(oh->per_step_mask) * T * B) OUT(sums, (size_t)LGAR_NUM_OUTPUTS * B)
  OUT(start_volume, B) OUT(status, B) OUT(crash_step, B) OUT(num_fronts, T * B) OUT(fronts, T * LGAR_MAX_FRONTS * 5 * B)
  OUT(front_layer, T * LGAR_MAX_FRONTS * B) OUT(front_to_bottom, T * LGAR_MAX_FRONTS * B) OUT(counters, 16)
  OUT(tile_cycles, (size_t)(oh->tile_diag_rows == 3 ? 3 : 1) * s.ntiles)
  OUT(moisture, (size_t)ph->num_depths * T * B) OUT(layer_water, LB * T)
#undef OUT
  const size_t wsb = lgar_workspace_bytes(&p, 0);
  void* ws = nullptr;
  CUDA_TRY(cudaMalloc(&ws, wsb));
  db.ptrs.push_back(ws);
  rc = lgar_forward(&p, &o, ws, wsb, 0, nullptr);
  if (rc) return rc;
  CUDA_TRY(cudaDeviceSynchronize());
  return db.download();
}

}  // extern "C"

// ---- FP64 peak probe ------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) dfma_probe(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x * 1e-9, x1 = x0 + 1.0, x2 = x0 + 2.0, x3 = x0 + 3.0;
  double x4 = x0 + 4.0, x5 = x0 + 5.0, x6 = x0 + 6.0, x7 = x0 + 7.0;
  for (int i = 0; i < iters; i++) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}
}  // namespace

extern "C" double lgar_measure_fp64_flops(int iters) {
  if (lgar_device_check()) return 0.0;
  if (iters < 1) iters = 4096;
  const int blocks = g_num_sms * 8, threads = 256;
  double* d = nullptr;
  if (cudaMalloc(&d, (size_t)blocks * threads * sizeof(double)) != cudaSuccess) return 0.0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  dfma_probe<<<blocks, threads>>>(d, iters, 0.999999, 1e-7);  // warm-up
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0);
    dfma_probe<<<blocks, threads>>>(d, iters, 0.999999, 1e-7);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) break;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * 8.0 * (double)iters * blocks * threads / (ms * 1e-3);
    if (flops > best) best = flops;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  return best;
}
