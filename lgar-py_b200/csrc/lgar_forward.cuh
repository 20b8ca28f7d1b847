// =====================================================================================
// lgar_forward.cuh -- persistent forward kernel: all columns x all forcing steps in ONE launch.
//
// Scheduling.  Work item = (tile of 32 columns, chunk of `chunk_steps` forcing steps).  Items
// are handed out chunk-major from one atomic counter to the resident warps (grid = SMs x CTAs
// per SM); item (tile, c) needs item (tile, c-1), which was handed out `ntiles` items earlier
// and is therefore finished or running on a resident warp -- a short acquire-spin on
// done[tile] resolves it without any possibility of deadlock.  Between chunks the column state
// (<= 16 fronts x 5 doubles + a few scalars) round-trips through global memory (L2): this
// removes the tail of a static column->warp assignment, balances slow and fast columns, and
// the chunk-start states double as the checkpoints of the reverse-mode kernel.
//
// One sub-step follows models/dpLGAR.py:154-299 exactly; the three places that evaluate Geff
// (insert_water, calc_dry_depth, calc_dzdt) are warp-convergent: their requests go through the
// per-warp queue, one request per lane (GeffQueue, lgar_device.cuh).
// =====================================================================================
#pragma once
#include "lgar_device.cuh"

namespace lgar {

// slots of the per-column state record (doubles), after the 5*FM front fields
enum StateSlot {
  S_PONDED = 0, S_PREV_PRECIP = 1, S_END_VOL = 2, S_GIUH = 3, /* 8 */ S_SUMS = 11, /* NOUT */ S_COUNT = 11 + NOUT
};
// int state: n, cntpk, status, crash_step
constexpr int NI_STATE = 4;

// outputs that are states, not fluxes: a step's value is the END state of the step and their "sum" is the last value
__host__ __device__ constexpr bool is_state_output(int k) { return k == LGAR_OUT_ENDING_VOLUME || k == LGAR_OUT_PONDED_WATER; }

template <int FM>
__host__ __device__ constexpr int state_doubles() { return 5 * FM + S_COUNT; }

struct KParams {
  lgar_problem p;
  lgar_outputs o;
  // workspace
  double* state_d;       // [nckpt][state_doubles][Bp]
  int32_t* state_i;      // [nckpt][NI_STATE][Bp]
  uint8_t* state_f;      // [nckpt][FM][Bp]
  int32_t* done;         // [ntiles] chunks completed per tile
  unsigned long long* next_item;
  int32_t Bp;            // B rounded up to a multiple of 32
  int32_t ntiles, nchunks, chunk_steps;
  int32_t t_begin, t_end;  // window of forcing rows advanced by this launch (lgar_problem.step_begin / step_end)
  // work-item tickets: 64-bit word next_item[slot] = (epoch << 40) | items handed out.  Classic launches: epoch 0, the
  // host zeroes the word.  Pipelined launches (lgar_problem.pipeline_seq = k > 1, programmatic dependent launch): no
  // host memset may sit between the kernels, so block 0 publishes (k << 40) itself and the other warps wait for
  // their epoch; a warp that finds a NEWER epoch in its slot (ring of 3, only possible for a launch that is over)
  // leaves.  `overlap`: the previous window may still be running, so even the first chunk of a tile waits for the
  // tile's progress counter.
  int32_t seq, slot, overlap;
  double* slog;          // search log [nchunks][slog_cap][Bp] (only with keep_ckpt; see Column::logp), nullptr = none
  int32_t* slog_count;   // [nchunks][Bp] entries the forward pass produced per lane and chunk
  int32_t slog_cap;
  int32_t time_phases;   // reverse kernel diagnostics: accumulate the phase timers of substep() in Ctx::ph
  int32_t keep_ckpt;     // 1: state of chunk c is stored at index c (+ final at nchunks)
  long long iter_cap;
};

// host: every region of the workspace starts on a 256-byte boundary; without a workspace (sizing only) the region
// pointers stay null
inline size_t align_up(size_t x) { return (x + 255) / 256 * 256; }
template <class T>
T* at(unsigned char* w, size_t off) { return w ? reinterpret_cast<T*>(w + off) : nullptr; }

template <int FM, class R, int LM = 0>
struct Tile {
  Column<FM, R, LM> col;
  Ctx ctx;
  R acc[NOUT];        // per-forcing-step accumulators (reset every step)
  double sums[NOUT];  // running sums over time
  int crash_step;
  int psiwp_st;       // guard raised while precomputing psi_wp (reported on first AET use)
};

// ---- Layer.calc_aet (Layer.py:760-783) -> calc_aet (lgar/aet.py:17-51)
template <int FM, class R, int LM>
__device__ __forceinline__ void precompute_psi_wp(Tile<FM, R, LM>& T, double wilting_psi) {
  Ctx cc = T.ctx;
  cc.st = 0;
  const SoilT<R>& s = T.col.soil[0];
  double theta_fc = (s.the - s.thr) * 0.75 + s.thr;  // GlobalParams.py:75
  R wp_head_theta = thetaR(R(wilting_psi), s, cc);
  R theta_wp = (theta_fc - wp_head_theta) * 0.5 + wp_head_theta;
  R se = se_thetaR(theta_wp, s, cc);
  T.col.psi_wp = h_seR(se, s, cc);
  T.psiwp_st = cc.st;
}
__device__ __forceinline__ double pow3R(double x, Ctx& c) { return safe_pow(x, 3.0, c); }
__device__ __forceinline__ Var pow3R(const Var& x, Ctx& c) { return pow3_(x, safe_pow(x.v, 3.0, c)); }
template <int FM, class R, int LM>
__device__ __forceinline__ R calc_aet(Tile<FM, R, LM>& T, double pet, double dt) {
  Ctx& c = T.ctx;
  if (T.psiwp_st) raise(c, T.psiwp_st);
  c.cnt[C_THETA_H] += 1;
  c.cnt[C_H_SE] += 1;
  R h_ratio = 1.0 + pow3R(T.col.g(F_PSI, 0) / T.col.psi_wp, c);
  R aet_ = pet * (1.0 / h_ratio) * dt;
  return clamp_(aet_, 0.0, pet);  // torch.clamp(min=0, max=pet): upper clamp is the RATE (sic)
}

// set_internal_states (models/dpLGAR.py:97-147), Layer.__init__ (Layer.py:22-90),
// WettingFront.__init__ (WettingFront.py:18-49), generate_soil_metrics (data/utils.py:40-105)
template <int FM, class R, int LM>
__device__ void init_column(Tile<FM, R, LM>& T, double initial_psi, bool closed_form_G = false) {
  Column<FM, R, LM>& C = T.col;
  Ctx& c = T.ctx;
  C.n = 0;
  C.cntpk = 0;
  for (int l = 0; l < C.L; l++) {
    const SoilT<R>& s = C.soil[l];
    if (closed_form_G && isnan(bc_psib(s.alpha, s.m))) raise(c, LGAR_ST_NAN);  // error_check in calc_bc_psib (utils.py:99)
    R theta_init = thetaR(R(initial_psi), s, c);
    const int i = C.n;
    C.s(F_DEPTH, i, R(C.cum[l]));
    C.s(F_THETA, i, theta_init);
    C.s(F_DZDT, i, R(0.0));
    R se = se_thetaR(theta_init, s, c);
    C.s(F_PSI, i, R(initial_psi));
    C.s(F_K, i, k_seR(se, s, c));
    C.set_flag(i, l, true);
    C.n++;
    C.add_cnt(l, 1);
  }
  C.ending_volume = C.mass_balance();
  C.ponded_water = R(0.0);
  C.previous_precip = 0.0;
  for (int i = 0; i < NGIUH; i++) C.giuh[i] = R(0.0);
  for (int k = 0; k < NOUT; k++) T.sums[k] = 0.0;
}

// ---- one sub-step: models/dpLGAR.py:176-298.  Warp-convergent: every lane of the warp calls it;
//      lanes with act == false only take part in the warp's Geff batches.
template <int FM, class R, int GM, int LM>
__device__ void substep(Tile<FM, R, LM>& T, bool act, double precip_rate, double pet_rate, const KParams& K,
                        double* nodebuf) {
  Column<FM, R, LM>& C = T.col;
  Ctx& c = T.ctx;
  const double dt = K.p.subcycle_length_h;
  const int nint = (GM == 2 && K.p.use_closed_form_G) ? -1 : K.p.nint;  // nint < 0 selects the closed-form Geff (geff_closedR)
  const int L = C.L;
  GeffQueue* const gq = reinterpret_cast<GeffQueue*>(nodebuf);
  act = act && (c.st == 0);

  double precip_sub = 0.0;
  R ponded_depth_sub(0.0), ponded_water_sub(0.0), percolation_sub(0.0);
  R runoff_sub(0.0), infiltration_sub(0.0), AET_sub(0.0);
  R ending_volume_sub = C.ending_volume;
  bool create = false, saturated = false;
  int fd = 0;
  if (act) {
    c.cnt[C_SUB]++;
    precip_sub = precip_rate * dt;
    const double pet_sub = pet_rate * dt;
    ponded_depth_sub = precip_sub + C.ponded_water;
    create = (C.previous_precip == 0.0) && (precip_sub > 0.0) && (C.ponded_water == 0.0);  // :310-323
    fd = C.free_drainage_front();
    saturated = C.f(F_THETA, 0) >= C.soil[0].the;  // Layer.is_saturated (:785-793)
    if (pet_rate > 0.0) AET_sub = calc_aet(T, pet_rate, dt);
    T.acc[LGAR_OUT_PRECIP] = T.acc[LGAR_OUT_PRECIP] + precip_sub;
    T.acc[LGAR_OUT_PET] = T.acc[LGAR_OUT_PET] + fmax(pet_sub, 0.0);
  }
  const bool brA = act && create && !saturated;             // create a surficial front
  const bool brB = act && !create && (ponded_depth_sub > 0.0);  // insert water

  const bool timed = ((GM == 2) && K.o.counters != nullptr) || K.time_phases;  // counting instantiations / reverse diagnostics
  long long tph = timed ? clock64() : 0;
  // ---- phase 1: Layer.insert_water (Layer.py:1418-1536) for branch-B lanes
  {
    int lfp = 0, nx_fd = 0;
    bool needG = false;
    R theta_1(0.0), theta_2(0.0);
    if (brB) {
      lfp = C.lay(fd);
      const int o = C.off(lfp);
      // get_drainage_neighbors (:1584-1607, Q6): the front after the FIRST front of fd's layer list
      if (C.cnt(lfp) > 1 || lfp < L - 1) nx_fd = o + 1;
      else raise(c, LGAR_ST_NULL_NEIGHBOUR);
      if (c.st == 0 && C.n != L) {
        needG = true;
        theta_1 = C.g(F_THETA, nx_fd);
        theta_2 = R(C.soil[lfp].the);
      }
    }
    const R geff = geff_one_per_lane<GM, R>(needG, theta_1, theta_2, lfp, C.soil, K.p.num_layers, nint, gq, c);
    if (brB && c.st == 0) {
      const R h_p = clamp_min_((ponded_depth_sub - precip_sub) * dt, 0.0);  // clamp(min=0)
      const R fd_depth = C.g(F_DEPTH, fd);
      R f_p(0.0);
      if (lfp == 0) {
        f_p = C.soil[0].ksatR() * (1.0 + (geff + h_p) / fd_depth);
      } else if (C.n == L) {
        raise(c, LGAR_ST_NULL_NEIGHBOUR);  // `free_drainage_ksat` unbound in the reference
      } else {
        const R fd_ksat = C.soil[lfp].ksatR() * K.p.frozen_factor;
        R bottom_sum = (fd_depth - C.cum[lfp - 1]) / fd_ksat;
        // calc_bottom_sum_f_p (:1538-1555, Q18): saturated K for layer 0, then the
        // unsaturated calc_bottom_sum for the remaining upper layers
        const R k0 = C.soil[0].ksatR() * K.p.frozen_factor;
        bottom_sum = bottom_sum + ((C.cum[0] - 0.0) / k0);
        if (1 != lfp) {
          c.br[2]++;
          bottom_sum = C.calc_bottom_sum(1, bottom_sum, C.g(F_PSI, fd), lfp, c);
        }
        f_p = (fd_depth / bottom_sum) + ((geff + h_p) * fd_ksat / fd_depth);
      }
      const R ponded_temp = clamp_min_(ponded_depth_sub - f_p * dt - 0.0, 0.0);
      const R fp_cm = f_p * dt + 0.0 / dt;
      if (C.pdm > 0.0) {
        if (ponded_temp < C.pdm) {
          infiltration_sub = tmin(ponded_depth_sub, fp_cm);
          ponded_depth_sub = ponded_depth_sub - infiltration_sub;
        } else if (ponded_temp > C.pdm) {
          ponded_depth_sub = C.pdmR();
          infiltration_sub = fp_cm;
        } else {
          c.br[1]++;  // equality: neither branch of the reference runs (Q8)
        }
        runoff_sub = clamp_min_(ponded_temp - C.pdmR(), 0.0);
      } else {
        infiltration_sub = tmin(ponded_depth_sub, fp_cm);
        const R r_ = ponded_depth_sub - infiltration_sub;
        ponded_depth_sub = C.pdmR();
        runoff_sub = clamp_min_(r_, 0.0);
      }
      T.acc[LGAR_OUT_INFILTRATION] = T.acc[LGAR_OUT_INFILTRATION] + infiltration_sub;
      T.acc[LGAR_OUT_RUNOFF] = T.acc[LGAR_OUT_RUNOFF] + runoff_sub;
      percolation_sub = infiltration_sub;
      ponded_water_sub = ponded_depth_sub;
    }
  }

  if (timed) { const long long t = clock64(); c.ph[0] += (unsigned long long)(t - tph); tph = t; }
  // ---- phase 2: move the fronts (branch A moves without adding water; every non-create lane moves
  //      with its infiltration).  models/dpLGAR.py:206-212 and :249-266
  {
    const bool go = act && c.st == 0 && (brA || !create);
    const R infil_arg = create ? R(0.0) : infiltration_sub;
    const R bottom = C.move_wetting_front_warp(go, fd, infil_arg, AET_sub, ending_volume_sub, dt, c);
    if (go && !create) {
      percolation_sub = bottom;
      T.acc[LGAR_OUT_PERCOLATION] = T.acc[LGAR_OUT_PERCOLATION] + percolation_sub;
    }  // branch A drops the bottom flux (Q7)
  }

  if (timed) { const long long t = clock64(); c.ph[1] += (unsigned long long)(t - tph); tph = t; }
  // ---- phase 3: calc_dry_depth (Layer.py:1309-1334) + create_surficial_front (:1336-1416)
  {
    const bool needG = brA && c.st == 0;
    R theta_1(0.0), theta_2(0.0);
    if (needG) {
      theta_1 = C.g(F_THETA, 0);
      theta_2 = R(C.soil[0].the);
    }
    const R geff = geff_one_per_lane<GM, R>(needG, theta_1, theta_2, 0, C.soil, K.p.num_layers, nint, gq, c);
    if (needG && c.st == 0) {
      const SoilT<R>& s = C.soil[0];
      const R cur_theta = C.g(F_THETA, 0);
      const R delta_theta = s.the - cur_theta;
      const R tau = dt * s.ksatR() / delta_theta;
      R dry_depth = 0.5 * (tau + sqrt_(tau * tau + 4.0 * tau * geff));
      dry_depth = tmin(C.cum[0], dry_depth);
      R theta_new(0.0);
      bool to_bottom;
      if (dry_depth * delta_theta > ponded_depth_sub) {
        infiltration_sub = ponded_depth_sub;
        theta_new = tmin(cur_theta + ponded_depth_sub / dry_depth, s.the);
        to_bottom = false;
        ponded_depth_sub = R(0.0);
      } else {
        infiltration_sub = dry_depth * delta_theta;
        ponded_depth_sub = ponded_depth_sub - (dry_depth * delta_theta);
        theta_new = R(s.the);
        to_bottom = !(dry_depth < C.cum[0]);
      }
      if (C.insert_at(0, 0, c)) {
        C.s(F_DEPTH, 0, dry_depth);
        C.s(F_THETA, 0, theta_new);
        C.set_flag(0, 0, to_bottom);
        R se = se_thetaR(theta_new, s, c);
        C.s(F_PSI, 0, h_seR(se, s, c));
        C.s(F_K, 0, k_seR(se, s, c) * K.p.frozen_factor);
        C.s(F_DZDT, 0, R(0.0));
      }
      T.acc[LGAR_OUT_INFILTRATION] = T.acc[LGAR_OUT_INFILTRATION] + infiltration_sub;
    }
  }
  // update_ponded_depth (models/dpLGAR.py:369-382) for every lane that did not insert water
  if (act && !brB) {
    if (ponded_depth_sub < C.pdm) {
      runoff_sub = R(0.0);
      ponded_water_sub = ponded_depth_sub;
      ponded_depth_sub = R(0.0);
    } else {
      runoff_sub = ponded_depth_sub - C.pdmR();
      ponded_depth_sub = C.pdmR();
      ponded_water_sub = ponded_depth_sub;
    }
    T.acc[LGAR_OUT_RUNOFF] = T.acc[LGAR_OUT_RUNOFF] + runoff_sub;
  }

  if (timed) { const long long t = clock64(); c.ph[2] += (unsigned long long)(t - tph); tph = t; }
  // ---- phase 4: Layer.calc_dzdt (Layer.py:1176-1252): one Geff per moving front of every column.  All requests of
  //      the tile are known here, so they go through the per-warp queue in batches of 32, one lane per request
  //      (geff_batch_eval); each lane then finishes dzdt of its own fronts in front order.  With the closed-form Geff
  //      (nint < 0) the queue is not used: the owner lane evaluates each of its requests itself (geff_closedR).
  {
    const bool closed = GM == 2 && nint < 0;
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const bool go = act && c.st == 0;
    const int my_n = go ? C.n - 1 : 0;  // the deepest front of the domain is excluded
    // requests of this lane: the fronts that are not to_bottom, up to the first front whose pre-checks fail (the
    // reference raises there, after the fronts before it went through calc_geff)
    int nreq = 0, pre_err = 0;
    {
      int l = 0, o_next = go ? C.cnt(0) : 0;
      for (int i = 0; i < my_n; i++) {
        while (i >= o_next) {
          l++;
          o_next += C.cnt(l);
        }
        if (C.tb(i)) {
          C.s(F_DZDT, i, R(0.0));
          continue;
        }
        if (C.lay(i) > 0) {
          if (l == 0) pre_err = LGAR_ST_NULL_NEIGHBOUR;  // self.previous_layer is None
        } else if (C.f(F_THETA, i + 1) > C.f(F_THETA, i)) {
          pre_err = LGAR_ST_THETA_ORDER;
        }
        if (pre_err) break;
        nreq++;
      }
    }
    int incl = nreq;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(FULL, incl, d);
      if (lane >= d) incl += v;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    int g = incl - nreq;   // queue index of this lane's next request
    int cur = 0;           // next front to look at
    int rem = nreq;
    for (int lo = 0; lo < total;) {
      const int hi = lo + 32;
      if (!closed) {
        gq->meta[lane] = -1;
        __syncwarp();
        int i = cur, gg = g, r_ = rem;
        while (r_ > 0 && gg < hi) {
          if (!C.tb(i)) {
            geffq_put(gq, gg - lo, lane, C.list_layer(i), C.f(F_THETA, i + 1), C.f(F_THETA, i));
            gg++;
            r_--;
          }
          i++;
        }
        __syncwarp();
        geffq_eval(gq, C.soil, K.p.num_layers, nint);
      }
      while (rem > 0 && g < hi) {
        const int i = cur++;
        if (C.tb(i)) continue;
        const int slot = g - lo;
        g++;
        rem--;
        if (c.st != 0) continue;
        const int l = C.list_layer(i);
        const R theta_1 = C.g(F_THETA, i + 1), theta_2 = C.g(F_THETA, i);
        const SoilT<R>& s = C.soil[l];
        const R geff = closed ? geff_closedR(true, theta_1, theta_2, s, c) : geffq_get(gq, slot, theta_1, theta_2, s, nint, c);
        if (c.st != 0) continue;
        const R depth = C.g(F_DEPTH, i);
        const R delta_theta = theta_2 - theta_1;
        R dzdt(0.0);
        if (C.lay(i) == 0) {
          if (delta_theta > 0.0)
            dzdt = 1.0 / delta_theta * (s.ksatR() * (geff + ponded_depth_sub) / depth + C.g(F_K, i));
        } else {
          const R bottom_sum = 0.0 + (C.g(F_DEPTH, i) - C.cum[l - 1]) / C.g(F_K, i);
          const R denominator = C.calc_bottom_sum(0, bottom_sum, C.g(F_PSI, i), C.lay(i), c);
          if (delta_theta > 0.0)
            dzdt = (1.0 / delta_theta) * ((depth / denominator) + s.ksatR() * (geff + ponded_depth_sub) / depth);
        }
        C.s(F_DZDT, i, dzdt);
      }
      __syncwarp();
      lo = hi;
    }
    if (go && c.st == 0 && pre_err) raise(c, pre_err);
  }

  if (timed) { const long long t = clock64(); c.ph[3] += (unsigned long long)(t - tph); tph = t; }
  if (act) {
    ending_volume_sub = C.mass_balance();
    C.previous_precip = precip_sub;
    C.ending_volume = ending_volume_sub;
    T.acc[LGAR_OUT_AET] = T.acc[LGAR_OUT_AET] + AET_sub;
    C.ponded_water = ponded_water_sub;
    // GIUH (lgar/giuh.py:8-20, models/dpLGAR.py:292-298)
    const int ng = K.p.num_giuh;
    double qsum = 0.0;
    for (int i = 0; i < ng; i++) qsum = qsum + val(C.giuh[i]);
    if (qsum > 0.0 || runoff_sub > 0.0) {
      for (int i = 0; i < ng; i++) C.giuh[i] = C.giuh[i] + (K.p.giuh_ordinates[i] * runoff_sub);
      const R now = C.giuh[0];
      for (int i = 0; i + 1 < ng; i++) C.giuh[i] = C.giuh[i + 1];
      C.giuh[ng - 1] = R(0.0);
      T.acc[LGAR_OUT_GIUH_RUNOFF] = T.acc[LGAR_OUT_GIUH_RUNOFF] + now;
      T.acc[LGAR_OUT_DISCHARGE] = T.acc[LGAR_OUT_DISCHARGE] + now;
    }
  }
}

// ------------------------------------------------------------------------------------
// state save / restore (global memory, column fastest).  Loads bypass L1 (__ldcg): the
// record may have been written by a warp on another SM.
// ------------------------------------------------------------------------------------
template <int FM, class R, int LM>
__device__ void save_state(const KParams& K, int slot, int b, Tile<FM, R, LM>& T) {
  const size_t Bp = K.Bp;
  double* sd = K.state_d + (size_t)slot * state_doubles<FM>() * Bp + b;
  Column<FM, R, LM>& C = T.col;
  for (int i = 0; i < C.n; i++) {
#pragma unroll
    for (int k = 0; k < 5; k++) sd[(size_t)(k * FM + i) * Bp] = C.f(k, i);
  }
  double* ss = sd + (size_t)(5 * FM) * Bp;
  ss[(size_t)S_PONDED * Bp] = val(C.ponded_water);
  ss[(size_t)S_PREV_PRECIP * Bp] = C.previous_precip;
  ss[(size_t)S_END_VOL * Bp] = val(C.ending_volume);
  for (int i = 0; i < NGIUH; i++) ss[(size_t)(S_GIUH + i) * Bp] = val(C.giuh[i]);
  for (int k = 0; k < NOUT; k++) ss[(size_t)(S_SUMS + k) * Bp] = T.sums[k];
  int32_t* si = K.state_i + (size_t)slot * NI_STATE * Bp + b;
  si[0] = C.n;
  si[Bp] = (int32_t)C.cntpk;
  si[2 * Bp] = T.ctx.st;
  si[3 * Bp] = T.crash_step;
  uint8_t* sf = K.state_f + (size_t)slot * FM * Bp + b;
  for (int i = 0; i < C.n; i++) sf[(size_t)i * Bp] = C.gb[i * NT];
}
template <int FM, class R, int LM>
__device__ void load_state(const KParams& K, int slot, int b, Tile<FM, R, LM>& T) {
  const size_t Bp = K.Bp;
  const double* sd = K.state_d + (size_t)slot * state_doubles<FM>() * Bp + b;
  Column<FM, R, LM>& C = T.col;
  const int32_t* si = K.state_i + (size_t)slot * NI_STATE * Bp + b;
  C.n = __ldcg(si);
  C.cntpk = (unsigned)__ldcg(si + Bp);
  T.ctx.st = __ldcg(si + 2 * Bp);
  T.crash_step = __ldcg(si + 3 * Bp);
  for (int i = 0; i < C.n; i++) {
#pragma unroll
    for (int k = 0; k < 5; k++) C.f(k, i) = __ldcg(sd + (size_t)(k * FM + i) * Bp);
  }
  const double* ss = sd + (size_t)(5 * FM) * Bp;
  C.ponded_water = R(__ldcg(ss + (size_t)S_PONDED * Bp));
  C.previous_precip = __ldcg(ss + (size_t)S_PREV_PRECIP * Bp);
  C.ending_volume = R(__ldcg(ss + (size_t)S_END_VOL * Bp));
  for (int i = 0; i < NGIUH; i++) C.giuh[i] = R(__ldcg(ss + (size_t)(S_GIUH + i) * Bp));
  for (int k = 0; k < NOUT; k++) T.sums[k] = __ldcg(ss + (size_t)(S_SUMS + k) * Bp);
  const uint8_t* sf = K.state_f + (size_t)slot * FM * Bp + b;
  for (int i = 0; i < C.n; i++) C.gb[i * NT] = __ldcg(sf + (size_t)i * Bp);
}

// load the column's parameters and derive the per-layer constants
// (models/dpLGAR.py:41-57, data/utils.py:75-91 calc_m, GlobalParams.py:99-110)
template <int FM, class R, int LM>
__device__ void load_params(const KParams& K, int b, Tile<FM, R, LM>& T) {
  const lgar_problem& p = K.p;
  Column<FM, R, LM>& C = T.col;
  const size_t B = p.num_columns;
  C.L = p.num_layers;
  double cumv = 0.0;
  for (int l = 0; l < C.L; l++) {
    SoilT<R>& s = C.soil[l];
    s.alpha = __ldg(p.alpha + l * B + b);
    s.n = __ldg(p.n + l * B + b);
    s.ksat = __ldg(p.ksat + l * B + b);
    s.the = __ldg(p.theta_e + l * B + b);
    s.thr = __ldg(p.theta_r + l * B + b);
    s.m = 1.0 - (1.0 / s.n);
    s.inv_m = 1.0 / s.m;
    s.ninv_m = -1.0 / s.m;
    s.inv_n = 1.0 / s.n;
    const double th = __ldg(p.thickness + l * B + b);
    C.thick[l] = th;
    cumv = (l == 0) ? th : cumv + th;
    C.cum[l] = cumv;
  }
  C.pdm = __ldg(p.ponded_depth_max + b);
  C.id_pdm = -1;
}

// ------------------------------------------------------------------------------------
// Forcing tiles.  A warp's 32 columns normally share one forcing record (columns of a site are adjacent; the
// balanced placement keeps them together): the rows of the current chunk are then staged into shared memory in blocks of
// FORCING_BLOCK rows (1 KB) by ONE bulk asynchronous copy (TMA engine: cp.async.bulk global -> shared, completion
// signalled on an mbarrier) issued by lane 0, and every step reads its (P, PET) pair as a shared-memory broadcast.
// Warps whose lanes mix sites (tile straddling two sites, per-column records) read through the read-only path.
// ------------------------------------------------------------------------------------
constexpr int FORCING_BLOCK = 64;
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
               "l"(src), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LGAR_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra LGAR_DONE_%=;\n"
      "bra LGAR_WAIT_%=;\n"
      "LGAR_DONE_%=:\n"
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}

// soil-moisture outputs of forcing step t (lgar_b200.h): theta at the sensor depths and the water of every layer, read
// off the END state of the step; NaN where the column has crashed (ok == false) or no front qualifies
template <int FM, class R, int LM>
__device__ void store_soil_moisture(const KParams& K, Column<FM, R, LM>& C, bool ok, int t, int b) {
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  const size_t B = K.p.num_columns, Tn = K.p.num_steps;
  if (K.o.moisture) {
    for (int d = 0; d < K.p.num_depths; d++) {
      const int i = ok ? C.front_at_depth(K.p.moisture_depths[d]) : -1;
      K.o.moisture[((size_t)d * Tn + t) * B + b] = (i >= 0) ? C.f(F_THETA, i) : qnan;
    }
  }
  if (K.o.layer_water) {
    int o = 0;
    for (int l = 0; l < C.L; l++) {
      K.o.layer_water[((size_t)l * Tn + t) * B + b] = ok ? C.template layer_water_t<double>(l, o) : qnan;
      o += C.cnt(l);
    }
  }
}

// dynamic shared memory of lgar_forward_kernel<FM>: the carve at the top of the kernel
template <int FM>
constexpr size_t forward_smem_bytes() {
  return (size_t)5 * FM * NT * sizeof(double) + (size_t)WARPS * NODEBUF * sizeof(double) + (size_t)FM * NT;
}

// resident CTAs per SM are bounded by the shared-memory front lists: 1 (FM = 32, the fallback for the rare columns
// that overflow 16 fronts), 2 (FM = 16), 3 (FM = 12), 4 (FM = 8); the register cap follows from that
// LOGW: the instantiation launched with keep_checkpoints also logs the end points of the root finders (Column::logp);
// in every other instantiation that code is compiled out
template <int FM, bool COUNT, bool DUMP, bool LOGW = false>
__global__ void __launch_bounds__(NT, (FM == 32) ? 1 : ((FM == 16) ? 2 : ((FM == 12) ? 3 : 4))) lgar_forward_kernel(const KParams K) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm_fields = reinterpret_cast<double*>(smem_raw);                       // [5*FM][NT]
  double* sm_nodes = sm_fields + 5 * FM * NT;                                    // [WARPS][NODEBUF]
  uint8_t* sm_flags = reinterpret_cast<uint8_t*>(sm_nodes + WARPS * NODEBUF);    // [FM][NT]
  __shared__ unsigned long long sm_item[WARPS];
  __shared__ __align__(16) double2 sm_forcing[WARPS][FORCING_BLOCK];
  __shared__ __align__(8) uint64_t sm_fbar[WARPS];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  if (lane == 0) mbar_init(&sm_fbar[warp], 1);
  pow_tables_to_shared();  // (ends with __syncthreads: the barriers are initialised for everybody)
  unsigned fphase = 0;     // parity of the next completion of this warp's forcing barrier

  double* nodebuf = sm_nodes + warp * NODEBUF;
  const lgar_problem& p = K.p;
  const int Tn = p.num_steps;
  const int S = p.num_subcycles;
  const size_t B = p.num_columns;
  const unsigned long long nitems = (unsigned long long)K.ntiles * K.nchunks;
  constexpr unsigned long long TICKET_MASK = (1ULL << 40) - 1ULL;
  unsigned long long* const ticket = K.next_item + K.slot;
  if (K.seq > 0 && blockIdx.x == 0 && threadIdx.x == 0) {
    atomicExch(ticket, (unsigned long long)K.seq << 40);
    __threadfence();
  }
  // programmatic dependent launch: the next window's grid may be scheduled as soon as every CTA of this one is
  // resident (has passed this point) and SM resources free up, i.e. while this launch drains its last items
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  Tile<FM, double, LOGW ? 1 : 0> T;
  T.col.fb = sm_fields + threadIdx.x;
  T.col.ib = nullptr;
  T.col.gb = sm_flags + threadIdx.x;
  T.ctx.iter_cap = K.iter_cap;
  T.col.logp = nullptr;
  T.col.log_pos = T.col.log_valid = T.col.log_stride = 0;

  for (;;) {
    if (lane == 0) {
      unsigned long long got = ~0ULL;
      for (;;) {
        const unsigned long long v = *reinterpret_cast<volatile unsigned long long*>(ticket);
        const unsigned long long ep = v >> 40;
        if (ep != (unsigned long long)K.seq) {
          if (ep < (unsigned long long)K.seq) {  // block 0 has not published this launch's epoch yet
            __nanosleep(100);
            continue;
          }
          break;  // the slot belongs to a later launch: this one is over
        }
        if ((v & TICKET_MASK) >= nitems) break;
        if (atomicCAS(ticket, v, v + 1ULL) == v) {
          got = v & TICKET_MASK;
          break;
        }
      }
      sm_item[warp] = got;
    }
    __syncwarp();
    const unsigned long long item = sm_item[warp];
    __syncwarp();
    if (item >= nitems) break;
    const int chunk = (int)(item / K.ntiles);
    const int tile = (int)(item % K.ntiles);
    // slot = position in the tile grid (state / checkpoint records); b = column of the ensemble this lane works on
    // (lgar_problem.column_order: work-balanced placement; identity when NULL)
    const int slot_c = tile * 32 + lane;
    const bool valid = (size_t)slot_c < B;
    const int slot_cc = valid ? slot_c : (int)B - 1;  // clamp for loads; results of invalid lanes are never stored
    const int b = p.column_order ? __ldg(p.column_order + slot_cc) : slot_cc;

    // wait for the previous chunk of this tile (acquire): done[tile] = forcing rows completed (absolute row index)
    const int t0 = K.t_begin + chunk * K.chunk_steps;
    const int t1 = min(K.t_end, t0 + K.chunk_steps);
    long long wait_cyc = 0;  // (counting kernel: scheduler diagnostics, lgar_outputs.tile_diag_rows)
    if (chunk > 0 || K.overlap) {
      if (lane == 0) {
        const long long w0 = COUNT ? clock64() : 0;
        volatile int32_t* d = K.done + tile;
        while (*d < t0) __nanosleep(200);
        if (COUNT) wait_cyc = clock64() - w0;
      }
      __syncwarp();
      __threadfence();
    }
#pragma unroll
    for (int k = 0; k < 8; k++) T.ctx.cnt[k] = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) T.ctx.ph[k] = 0;
#pragma unroll
    for (int k = 0; k < 3; k++) T.ctx.br[k] = 0;
    const long long clk0 = clock64();
    load_params(K, b, T);
    const int slot_in = K.keep_ckpt ? chunk : 0;
    if (chunk == 0 && p.resume) {
      load_state(K, 0, slot_cc, T);  // continue from the state the previous launch left in the workspace
      if (T.crash_step >= 0) T.crash_step = -2 - T.crash_step;  // crashed in an earlier call
    } else if (chunk == 0) {
      T.ctx.st = 0;
      T.crash_step = -1;
      init_column(T, __ldg(p.initial_psi + b), p.use_closed_form_G != 0);
      if (T.ctx.st) T.crash_step = 0;
      if (valid && K.o.start_volume) K.o.start_volume[b] = T.col.ending_volume;
      if (K.keep_ckpt && valid) save_state(K, 0, slot_c, T);
    } else {
      load_state(K, slot_in, slot_cc, T);
    }
    precompute_psi_wp(T, p.wilting_point_psi);
    if (LOGW && K.slog && K.keep_ckpt) {  // log the end points of the root finders for the reverse pass
      T.col.logp = K.slog + (size_t)chunk * K.slog_cap * K.Bp + slot_cc;
      T.col.log_pos = 0;
      T.col.log_valid = valid ? K.slog_cap : 0;
      T.col.log_stride = K.Bp;
    }
    const int site = (p.site_index && valid) ? __ldg(p.site_index + b) : 0;
    const double* frc = p.forcing + (size_t)site * Tn * 2;
    // one forcing record for the whole warp?  (lanes beyond B follow lane 0)
    const int site0 = __shfl_sync(0xffffffffu, site, 0);
    const bool staged = __all_sync(0xffffffffu, !valid || site == site0);
    const double2* frc0 = reinterpret_cast<const double2*>(p.forcing + (size_t)site0 * Tn * 2);

    for (int t = t0; t < t1; t++) {
      const int fk = (t - t0) & (FORCING_BLOCK - 1);
      if (staged && fk == 0) {
        const int rows = min(t1 - t, FORCING_BLOCK);
        __syncwarp();  // every lane has read the previous block
        if (lane == 0) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // order those reads before the async write
          mbar_expect_tx(&sm_fbar[warp], (uint32_t)rows * 16u);
          bulk_copy_g2s(&sm_forcing[warp][0], frc0 + t, (uint32_t)rows * 16u, &sm_fbar[warp]);
        }
        mbar_wait(&sm_fbar[warp], fphase);
        fphase ^= 1u;
      }
      const double2 x = staged ? sm_forcing[warp][fk] : __ldg(reinterpret_cast<const double2*>(frc) + t);
#pragma unroll
      for (int k = 0; k < NOUT; k++) T.acc[k] = 0.0;
      const bool alive = valid && (T.ctx.st == 0);
      for (int sc = 0; sc < S; sc++) substep<FM, double, COUNT ? 2 : 0>(T, alive, x.x, x.y, K, nodebuf);
      if (alive && T.ctx.st != 0) T.crash_step = t;
      const bool ok = valid && (T.ctx.st == 0);
      T.acc[LGAR_OUT_ENDING_VOLUME] = T.col.ending_volume;
      T.acc[LGAR_OUT_PONDED_WATER] = T.col.ponded_water;
      if (valid) {
        const double qnan = __longlong_as_double(0x7ff8000000000000LL);
        if (K.o.per_step) {
#pragma unroll
          for (int k = 0; k < NOUT; k++)
            if (K.o.per_step_mask & (1u << k))
              K.o.per_step[((size_t)__popc(K.o.per_step_mask & ((1u << k) - 1u)) * Tn + t) * B + b] =
                  ok ? T.acc[k] : qnan;
        }
        if (ok) {
#pragma unroll
          for (int k = 0; k < NOUT; k++)
            T.sums[k] = is_state_output(k) ? T.acc[k] : T.sums[k] + T.acc[k];
        }
        if (K.o.num_fronts) K.o.num_fronts[(size_t)t * B + b] = ok ? T.col.n : 0;
        if (K.o.moisture || K.o.layer_water) store_soil_moisture(K, T.col, ok, t, b);
        if (DUMP && K.o.fronts) {
          for (int i = 0; i < LGAR_MAX_FRONTS; i++) {
            const bool has = ok && i < T.col.n;
#pragma unroll
            for (int k = 0; k < 5; k++)
              K.o.fronts[(((size_t)t * LGAR_MAX_FRONTS + i) * 5 + k) * B + b] = has ? T.col.f(k, i) : 0.0;
            if (K.o.front_layer) K.o.front_layer[((size_t)t * LGAR_MAX_FRONTS + i) * B + b] = has ? (int8_t)T.col.lay(i) : (int8_t)-1;
            if (K.o.front_to_bottom) K.o.front_to_bottom[((size_t)t * LGAR_MAX_FRONTS + i) * B + b] = has ? (int8_t)T.col.tb(i) : (int8_t)0;
          }
        }
      }
    }

    // publish the state for the next chunk of this tile (release)
    const int slot_out = K.keep_ckpt ? chunk + 1 : 0;
    if (valid) save_state(K, slot_out, slot_c, T);
    if (LOGW && K.slog && valid) K.slog_count[(size_t)chunk * K.Bp + slot_c] = T.col.log_pos;
    if (chunk == K.nchunks - 1 && valid) {
      if (K.o.sums) {
#pragma unroll
        for (int k = 0; k < NOUT; k++) K.o.sums[(size_t)k * B + b] = T.sums[k];
      }
      if (K.o.status) K.o.status[b] = T.ctx.st;
      if (K.o.crash_step) K.o.crash_step[b] = T.crash_step;
    }
    if (COUNT && K.o.counters && valid) {
#pragma unroll
      for (int k = 0; k < 8; k++)
        if (T.ctx.cnt[k]) atomicAdd(K.o.counters + k, (unsigned long long)T.ctx.cnt[k]);
#pragma unroll
      for (int k = 0; k < 3; k++)
        if (T.ctx.br[k]) atomicAdd(K.o.counters + 13 + k, (unsigned long long)T.ctx.br[k]);
      if (lane == 0) {  // phase timers of this warp (entries 8..11) and its total chunk time (12)
#pragma unroll
        for (int k = 0; k < 4; k++) atomicAdd(K.o.counters + 8 + k, T.ctx.ph[k]);
        atomicAdd(K.o.counters + 12, (unsigned long long)(clock64() - clk0));
      }
    }
    __threadfence();
    __syncwarp();
    if (lane == 0) {
      if (K.o.tile_cycles) atomicAdd(K.o.tile_cycles + tile, (unsigned long long)(clock64() - clk0));
      if (COUNT && K.o.tile_cycles && K.o.tile_diag_rows == 3) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        atomicAdd(K.o.tile_cycles + K.ntiles + tile, (unsigned long long)wait_cyc);
        atomicMax(K.o.tile_cycles + 2 * (size_t)K.ntiles + tile, now);
      }
      atomicExch(K.done + tile, t1);
    }
  }
}

}  // namespace lgar
