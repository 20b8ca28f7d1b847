/* =====================================================================================
 * lgar_b200.h -- C ABI of the B200-native LGAR time-stepping core (liblgar_b200.so).
 *
 * This library replaces, for MANY independent soil columns at once, the per-column
 * update loop of the reference (paths relative to /root/reference/dpLGAR/):
 *
 *   lgar_forward   <->  models/dpLGAR.py:154-299  dpLGAR.forward(x) applied to every row of the
 *                       forcing record (the loop of agents/DifferentiableLGAR.py:117-125 with
 *                       MassBalance.change_mass resetting the accumulators after each step),
 *                       starting from models/dpLGAR.py:97-147 set_internal_states().
 *   lgar_backward  <->  loss.backward() of agents/DifferentiableLGAR.py:163 restricted to the
 *                       model parameters alpha/n/ksat (models/dpLGAR.py:50-57): reverse-mode
 *                       through the same step loop (reference autograd semantics, SURVEY Q13/Q14).
 *   status[B]      <->  the Python exceptions the reference uses as error reporting
 *                       (physics/utils.py:17-27,181-183; physics/layers/Layer.py:1206-1208,
 *                       :980 (Q9), :876-881 (Q10), :1115).
 *
 * The reference has no FFI layer (it is pure Python); the binding a maintainer adds is the
 * ctypes stub shown in INTEGRATION.md (== lgar-py_b200/_capi.py).
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch types.  Every function returns 0 on success or a
 *     negative LGAR_E_* code; lgar_last_error_string() describes the last failure of the
 *     calling thread.  Nothing throws across the ABI.
 *   - `*_dev` pointers are device pointers on the current CUDA device; the caller owns all
 *     buffers.  `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are
 *     asynchronous with respect to the host unless stated otherwise.
 *   - re-entrant per (stream, workspace): no global mutable state besides the per-thread
 *     error string and a lazily cached device-attribute query.
 *   - all floating point data is IEEE fp64; layouts have the COLUMN index fastest so that a
 *     warp of 32 columns reads/writes 256 contiguous bytes.
 * ===================================================================================== */
#ifndef LGAR_B200_H
#define LGAR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGAR_ABI_VERSION 3     /* 3: soil-moisture outputs (num_depths, moisture_depths, moisture, layer_water) */
#define LGAR_MAX_LAYERS 4      /* soil layers per column (all reference configs use 3)            */
#define LGAR_MAX_FRONTS 16     /* capacity of the wetting-front list of one column                */
#define LGAR_MAX_GIUH 8        /* GIUH ordinates (reference: 5, data/config/Phillipsburg.yaml)    */
#define LGAR_NUM_OUTPUTS 10
#define LGAR_MAX_DEPTHS 8      /* sensor depths of the soil-moisture output (lgar_problem.moisture_depths)   */

/* Soil moisture (lgar_outputs.moisture / layer_water), read off the column state at the END of every forcing
 * step (after its last sub-step), the same point the rows of per_step are read at.  "The list of layer l" is the
 * l-th block of the front list, cnt(l) fronts long (Layer.wetting_fronts of the reference).
 *   layer water W_l (cm): the per-layer term of Layer.mass_balance (Layer.py:795-824) in its exact operation order:
 *       top_l = 0 for l = 0, else cum_l - thickness_l (cum_l = thickness_0 + ... + thickness_l, summed in that order);
 *       W_l = 0 + sum over the fronts i of the list except the last of (depth_i - top_l) * (theta_i - theta_{i+1}),
 *             then + (depth_last - top_l) * theta_last.
 *     W_0 + (W_1 + (W_2 ...)) is the column's mass balance, so on every step of an OK column it equals the
 *     ENDING_VOLUME output bit for bit.  The layer-average water content is W_l / thickness_l.
 *   theta at depth z (cm below the surface, z > 0): the layer l with cum_{l-1} < z <= cum_l (a depth on a layer
 *     bottom belongs to the upper layer); theta(z) is the theta of the FIRST front of layer l's list, in list order,
 *     whose depth >= z.  A selection, bit-identical to that front's theta; NaN if z > cum_{L-1} or no front of the
 *     list qualifies.  Its gradient flows into the theta of the selected front; the selection carries none.
 *   A column that crashed gets NaN from its crash step on (like per_step); earlier steps keep their values.   */
/* per-forcing-step output variables (index into the [NOUT][T][B] output array); the same
 * accumulators MassBalance.change_mass reads and zeroes (physics/MassBalance.py:31-53)          */
enum lgar_output {
  LGAR_OUT_RUNOFF = 0,
  LGAR_OUT_PERCOLATION = 1,
  LGAR_OUT_AET = 2,
  LGAR_OUT_INFILTRATION = 3,
  LGAR_OUT_ENDING_VOLUME = 4,   /* state at the end of the step (not an accumulator)              */
  LGAR_OUT_PONDED_WATER = 5,    /* state at the end of the step                                   */
  LGAR_OUT_GIUH_RUNOFF = 6,
  LGAR_OUT_PRECIP = 7,
  LGAR_OUT_PET = 8,
  LGAR_OUT_DISCHARGE = 9
};

/* per-column status: 0 = OK; otherwise the reference would have raised at `crash_step`.       */
enum lgar_status {
  LGAR_ST_OK = 0,
  LGAR_ST_NEG_POW = 1,        /* ValueError, negative base in safe_pow      utils.py:25-27        */
  LGAR_ST_NAN = 2,            /* ValueError, NaN in pow input/result        utils.py:17-19,181-183 */
  LGAR_ST_THETA_ORDER = 3,    /* ValueError, theta_1 > theta_2 in layer 0   Layer.py:1206-1208    */
  LGAR_ST_BOTTOM_REACHED = 4, /* AttributeError, front left the last layer  Layer.py:980 (Q9)     */
  LGAR_ST_NULL_NEIGHBOUR = 5, /* AttributeError/UnboundLocalError           Layer.py:876-881 (Q10)*/
  LGAR_ST_FRONT_OVERFLOW = 6, /* more than `max_fronts` fronts (capacity of this library)         */
  LGAR_ST_ITER_CAP = 7,       /* a root finder exceeded `iter_cap` iterations                     */
  LGAR_ST_INDEX_ERROR = 8     /* IndexError                                 Layer.py:1115         */
};

enum lgar_error {
  LGAR_E_OK = 0,
  LGAR_E_INVALID = -1,   /* bad argument                                                        */
  LGAR_E_CUDA = -2,      /* CUDA runtime error (see lgar_last_error_string)                     */
  LGAR_E_NO_DEVICE = -3, /* no sm_100 device: there is NO CPU fallback                          */
  LGAR_E_WORKSPACE = -4  /* workspace too small                                                 */
};

/* Problem description.  Array members are device pointers (lgar_forward/backward) or host
 * pointers (lgar_forward_host).  [L][B] means layer-major, column fastest.                    */
typedef struct lgar_problem {
  int32_t abi_version;     /* = LGAR_ABI_VERSION                                                */
  int32_t num_columns;     /* B                                                                 */
  int32_t num_layers;      /* L <= LGAR_MAX_LAYERS          cfg.data.layer_thickness            */
  int32_t num_steps;       /* T forcing steps                cfg.models.nsteps                  */
  int32_t num_subcycles;   /* S sub-steps per forcing step   cfg.models.num_subcycles           */
  int32_t num_sites;       /* number of forcing series                                          */
  int32_t nint;            /* Geff trapezoid intervals       cfg.constants.nint (120)           */
  int32_t num_giuh;        /* <= LGAR_MAX_GIUH               cfg.data.giuh_ordinates            */
  int32_t max_fronts;      /* 8, 12, 16 or 32 (0 = 16): front-list capacity per column; 32 is
                              forward-only (one CTA per SM): the fallback for LGAR_ST_FRONT_OVERFLOW  */
  int32_t chunk_steps;     /* forcing steps per scheduling/checkpoint chunk (0 = default 64)    */
  int32_t resume;          /* 0: start from set_internal_states() (models/dpLGAR.py:97-147);
                              1: continue from the column state the previous lgar_forward left in
                              this workspace (same B, L, max_fronts; keep_checkpoints == 0): lets a
                              caller advance one forcing row per call like dpLGAR.forward(x)         */
  int32_t use_closed_form_G; /* cfg.data.use_closed_form_G: 0 = trapezoid Geff (green_ampt.py:45-84),
                              1 = Brooks-Corey closed form (green_ampt.py:85-98); was reserved (0) before   */
  int32_t step_begin;      /* window [step_begin, step_end) of the forcing record advanced by this call   */
  int32_t step_end;        /* (0, 0 = the whole record).  num_steps stays the length of the record: it
                              fixes the layout of `forcing` and of the per-step outputs, and step indices
                              (crash_step, rows of per_step) stay absolute.  A window that does not start
                              at row 0 needs resume = 1; windows are forward-only (keep_checkpoints == 0).
                              Lets a caller stream a long record segment by segment (bench.py) the way the
                              reference's loop feeds dpLGAR.forward one row at a time
                              (agents/DifferentiableLGAR.py:117-125)                                       */
  int32_t pipeline_seq;    /* 0: every call is stream-ordered after the previous one (default).
                              k >= 1: the k-th call of a PIPELINED sequence of consecutive windows of one
                              record on one stream and workspace (window k starts at the row where window
                              k-1 ended; k = 1 starts the sequence).  Calls k > 1 are launched with
                              programmatic dependent launch: their CTAs start on the SMs the previous
                              window has already drained, and the per-tile progress counters in the
                              workspace order the column states, so the slowest columns of one window no
                              longer idle the GPU before the next.  Nothing else may be enqueued on the
                              stream between two calls of a sequence (it would serialise them again); the
                              results of all windows are complete when the stream has drained.           */
  int32_t num_depths;      /* 0..LGAR_MAX_DEPTHS sensor depths of lgar_outputs.moisture (0 = none); was reserved (0)
                              before ABI 3                                                                  */
  int64_t iter_cap;        /* root-finder iteration cap (0 = default 1,000,000)                 */
  double subcycle_length_h;   /* dt in hours                 cfg.models.subcycle_length_h       */
  double wilting_point_psi;   /* cm                          cfg.data.wilting_point_psi         */
  double frozen_factor;       /*                             cfg.constants.frozen_factor        */
  double giuh_ordinates[LGAR_MAX_GIUH];
  /* learnable parameters, models/dpLGAR.py:50-57 (ksat already multiplied by frozen_factor)   */
  const double* alpha;        /* [L][B]  1/cm                                                    */
  const double* n;            /* [L][B]                                                          */
  const double* ksat;         /* [L][B]  cm/h                                                    */
  /* static soil/site data                                                                      */
  const double* theta_r;      /* [L][B]                      soils table column theta_r         */
  const double* theta_e;      /* [L][B]                      soils table column theta_e         */
  const double* thickness;    /* [L][B]  cm                  cfg.data.layer_thickness           */
  const double* initial_psi;  /* [B]     cm                  cfg.data.initial_psi               */
  const double* ponded_depth_max; /* [B] cm                  cfg.data.ponded_depth_max          */
  /* forcing, data/Data.py:33-40: x[t] = (P, PET) in cm/h                                       */
  const double* forcing;      /* [num_sites][T][2]                                               */
  const int32_t* site_index;  /* [B] forcing series of each column (NULL = all use series 0)    */
  const int32_t* column_order; /* [B] permutation of 0..B-1 or NULL: the i-th thread of the launch grid works on
                              column column_order[i].  Every array of this struct and of lgar_outputs stays
                              indexed by COLUMN; only the placement of columns on warps changes (results do not
                              depend on it).  A warp advances its 32 columns in lock step, so grouping columns of
                              similar cost (e.g. sorted by top-layer ksat) raises lane utilisation.  lgar_backward
                              and resumed calls must pass the order of the lgar_forward they follow.           */
  double moisture_depths[LGAR_MAX_DEPTHS]; /* cm below the surface, each finite and > 0; the first num_depths are
                              used.  Shared by all columns; read by lgar_forward (moisture) and by
                              lgar_backward_ex (grad_moisture)                                              */
} lgar_problem;

/* Output buffers.  Any pointer may be NULL (that output is skipped).                           */
typedef struct lgar_outputs {
  double* per_step;        /* [popcount(per_step_mask)][T][B]: the selected outputs, compact, in
                              increasing output index                                            */
  uint32_t per_step_mask;  /* bit k = store output k                                            */
  int32_t tile_diag_rows;  /* rows of `tile_cycles` (0 = 1); see there                             */
  double* sums;            /* [NOUT][B]: sum over t of every output (ENDING_VOLUME and
                              PONDED_WATER: value after the last step)                          */
  double* start_volume;    /* [B] water in the column after set_internal_states()               */
  int32_t* status;         /* [B] lgar_status                                                   */
  int32_t* crash_step;     /* [B] forcing step at which status became non-zero, else -1         */
  int32_t* num_fronts;     /* [T][B] number of wetting fronts after every step                  */
  /* full front-list dump after every step (parity tests; small B only)                        */
  double* fronts;          /* [T][MAXF=16][5][B]: depth, theta, psi_cm, k_cm_per_h, dzdt        */
  int8_t* front_layer;     /* [T][16][B] layer_num (-1 = no front)                              */
  int8_t* front_to_bottom; /* [T][16][B]                                                        */
  /* work counters, summed over columns and steps: 0 geff calls, 1 theta_from_h, 2 h_from_se,
   * 3 k_from_se, 4 se_from_h, 5 theta root-finder iterations, 6 column-mass iterations,
   * 7 sub-steps.  Used for the algorithmic FLOP count of the roofline (DESIGN.md).            */
  unsigned long long* counters; /* [16]: 0-7 work counters; 8-11 warp cycles in insert-water Geff, move
                                   sweep, dry-depth Geff, calc_dzdt; 12 total warp cycles; 13-15 branch coverage:
                                   dry-over-wet fixes (Layer.py:1055-1096), insert_water equality fall-through
                                   (Layer.py:1509-1521), calc_bottom_sum_f_p with the free-drainage front in
                                   layer >= 2 (Layer.py:1538-1555)                                          */
  /* diagnostics: SM cycles spent on each tile of 32 consecutive columns, summed over chunks.  With
   * tile_diag_rows = 3 (and `counters` set: the counting kernel) two more rows follow: cycles the tile's chunks
   * spent WAITING for their predecessor chunk (a resident warp blocked on the per-tile progress counter), and the
   * global timer (ns) at the end of the tile's last chunk of this launch -- the scheduler's idle time and tail */
  unsigned long long* tile_cycles; /* [tile_diag_rows][ceil(B/32)]                              */
  /* soil moisture after every step (definitions above LGAR_MAX_DEPTHS); may be NULL                        */
  double* moisture;        /* [num_depths][T][B] theta at moisture_depths[d]; needs num_depths > 0            */
  double* layer_water;     /* [L][T][B] water stored in each layer, cm                                        */
} lgar_outputs;

/* Library / device probe.  Returns 0 if an sm_100 device is current and usable.               */
int lgar_abi_version(void);
int lgar_device_check(void);
const char* lgar_last_error_string(void);

/* Bytes of device workspace needed by lgar_forward/lgar_backward for this problem shape
 * (only B, L, T, S, max_fronts, chunk_steps are read).  `with_grad` != 0 adds the checkpoint
 * store and the reverse-sweep scratch.                                                         */
size_t lgar_workspace_bytes(const lgar_problem* p, int with_grad);

/* Forward: advance all B columns through all T forcing steps in ONE persistent launch.
 * Replaces the per-row calls `runoff, percolation = self.model(x)` of the reference's training loop
 * (dpLGAR/agents/DifferentiableLGAR.py:117-125 -> dpLGAR.forward, dpLGAR/models/dpLGAR.py:154-299) together with
 * set_internal_states (models/dpLGAR.py:97-147) and the accumulator resets of MassBalance.change_mass
 * (models/physics/MassBalance.py:31-53).
 * If `workspace_dev` was sized with with_grad != 0, state checkpoints for lgar_backward are
 * stored in it (pass keep_checkpoints != 0).                                                   */
int lgar_forward(const lgar_problem* p, const lgar_outputs* out, void* workspace_dev,
                 size_t workspace_bytes, int keep_checkpoints, void* stream);

/* Reverse mode: replaces `loss.backward()` w.r.t. model.alpha / n / ksat (dpLGAR/agents/DifferentiableLGAR.py:163)
 * with the reference's autograd semantics (straight-through root finders).
 * grad_per_step[popcount(grad_mask)][T][B] (same compact layout) and/or
 * grad_sums[NOUT][B] are dL/d(output); writes dL/d(alpha,n,ksat) as [L][B] arrays.
 * Must follow an lgar_forward with keep_checkpoints on the same workspace and problem.         */
int lgar_backward(const lgar_problem* p, const double* grad_per_step, uint32_t grad_mask,
                  const double* grad_sums, double* grad_alpha, double* grad_n, double* grad_ksat,
                  void* workspace_dev, size_t workspace_bytes, void* stream);

/* lgar_backward with options.  Everything lgar_backward takes, plus:
 *   reduce != 0     the parameters are SHARED by all columns (the reference's model: one alpha/n/ksat per layer,
 *                   models/dpLGAR.py:50-57, trained over many columns / sites at once): grad_alpha/n/ksat are [L]
 *                   arrays holding the SUM over columns, reduced inside the library in a fixed order (warp shuffle
 *                   per tile, then a fixed-order pass over the tile partials): bit-reproducible, no atomics, and the
 *                   all-reduce input of a data-parallel calibration step comes straight out of our kernels.
 *                   Columns whose tape overflowed contribute 0 (see tape_overflow).
 *   tape_overflow   [B] or NULL: 1 where a column's tape arena was exhausted -- its gradient is not available
 *                   (per-column mode: NaN) and the caller must not step on it.
 *   partials        [ceil(B/32)][3 LGAR_MAX_LAYERS + 1] doubles of scratch for reduce != 0.
 *   counters        [8] or NULL, diagnostics summed over warps: 0 cycles in the taped recompute, 1 cycles in the
 *                   reverse sweeps, 2 tape entries recorded (per lane), 3 sub-steps taped (per lane), 4 overflowed columns,
 *                   5-7 cycles of the taped recompute in the move sweep, in calc_dzdt (Geff), in the other Geff phases. */
typedef struct lgar_gradients {
  const double* grad_per_step;  /* [popcount(grad_mask)][T][B] dL/d(per-step outputs) or NULL                */
  uint32_t grad_mask;
  int32_t reduce;
  const double* grad_sums;      /* [NOUT][B] dL/d(sums) or NULL                                              */
  double* grad_alpha;           /* [L][B], or [L] with reduce                                                */
  double* grad_n;
  double* grad_ksat;
  double* partials;
  int32_t* tape_overflow;
  unsigned long long* counters;
  double* grad_ponded_depth_max; /* [B], or [1] with reduce; NULL = not wanted.  dL/d ponded_depth_max: the reference
                                    declares it as a parameter in a commented-out line (models/dpLGAR.py:48-49); as a
                                    leaf it reaches the loss through update_ponded_depth (models/dpLGAR.py:369-382) and
                                    insert_water (Layer.py:1509-1532)                                              */
  const double* grad_moisture;    /* [num_depths][T][B] dL/d(lgar_outputs.moisture) or NULL (needs num_depths > 0)  */
  const double* grad_layer_water; /* [L][T][B] dL/d(lgar_outputs.layer_water) or NULL                              */
} lgar_gradients;
int lgar_backward_ex(const lgar_problem* p, const lgar_gradients* g, void* workspace_dev, size_t workspace_bytes,
                     void* stream);

/* Convenience for non-CUDA hosts: same as lgar_forward but every pointer in `p` and `out` is a
 * HOST pointer; the library allocates device memory, copies in, runs, copies out, synchronises. */
int lgar_forward_host(const lgar_problem* p, const lgar_outputs* out);

/* FP64 peak probe used by bench.py for the roofline denominator: runs a dependent-chain-free
 * DFMA kernel for `iters` iterations on the current device and returns achieved FLOP/s
 * (0 on failure).  Synchronous.                                                                */
double lgar_measure_fp64_flops(int iters);

#ifdef __cplusplus
}
#endif
#endif /* LGAR_B200_H */
