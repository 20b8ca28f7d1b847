// =====================================================================================
// lgar_backward.cuh -- hand-written reverse-mode kernel (checkpointed recompute).
//
// dL/d(alpha, n, ksat)[L][B] for L = sum_{k,t,b} g[k][t][b] * out[k][t][b] (+ the same with the
// per-column sums), with the reference's autograd semantics (SURVEY Q12-Q14).
//
// Work item = (tile of 32 columns, chunk of the forcing record), handed out from one counter LAST CHUNK FIRST to the
// resident warps; item (tile, c) needs the adjoint state that item (tile, c+1) left behind (lambda of the column
// state, the running parameter gradients), which was handed out `ntiles` items earlier and is therefore finished or
// running on a resident warp: an acquire-spin on rev_done[tile] orders them without any possibility of deadlock.
// (Tiles cost between 0.5x and 1.7x the mean; with whole records per warp the launch lasted as long as the
// unluckiest warp's three or four tiles.)  For its item a warp:
//   1. load the chunk-start checkpoint the forward kernel stored (lgar_forward(keep_checkpoints));
//   2. recompute the chunk forward with R = Var: every sub-step records its own tape (leaves = the
//      state in front of it; it takes exactly the forward kernel's branches because the values come
//      from the same cores) into a per-warp arena, plus a small record of which tape ids the END
//      state and the step outputs ended up with;
//   3. walk the sub-steps of the chunk backwards: seed the adjoints (dL/d out of this step + the
//      adjoint of the next state), sweep the tape, keep the adjoint of the state in front of the
//      sub-step and accumulate the parameter adjoints.
// Tapes and adjoints live in global memory (L2), laid out lane-fastest so the 32 lanes of a warp
// touch consecutive addresses when they are at the same entry.  The root finders are
// straight-through (they never appear on the tape); Geff is one macro entry whose partials are
// evaluated together with its value, one request per lane (geff_batch_eval_taped).  (A first
// version recomputed the chunk in plain fp64 and replayed each sub-step on the tape afterwards;
// carrying both code paths made the kernel 50k instructions and instruction-fetch bound:
// `no_instruction` 3.8 stalls per issue in ncu.)
// =====================================================================================
#pragma once
#include "lgar_forward.cuh"

namespace lgar {

constexpr int NPAR_IDS = 3 * MAXL + 1;  // alpha[l] = 3l, n[l] = 3l+1, ksat[l] = 3l+2; ponded_depth_max = 3 MAXL
constexpr int ID_PDM = 3 * MAXL;
template <int FM>
__host__ __device__ constexpr int leaf_fields() { return NPAR_IDS; }                  // + fld*FM + i
template <int FM>
__host__ __device__ constexpr int leaf_ponded() { return NPAR_IDS + 5 * FM; }
template <int FM>
__host__ __device__ constexpr int leaf_endvol() { return NPAR_IDS + 5 * FM + 1; }
template <int FM>
__host__ __device__ constexpr int leaf_giuh() { return NPAR_IDS + 5 * FM + 2; }
template <int FM>
__host__ __device__ constexpr int num_leaves() { return NPAR_IDS + 5 * FM + 2 + NGIUH; }

// per-sub-step record kept for the reverse sweep (16-bit ids; see Column::ib)
template <int FM>
struct StepMeta {
  int32_t n_entries;   // tape entries of this sub-step
  int32_t n_fronts;    // fronts at the END of the sub-step
  int16_t alive;       // the lane simulated this sub-step
  int16_t id_ponded, id_endvol;
  int16_t id_giuh[NGIUH];
  int16_t id_acc[NOUT];
  int16_t id_field[5 * FM];  // [fld * FM + i]: tape id of every field of the END state
};

struct BParams {
  KParams K;
  const double* grad_per_step;  // [popc(grad_mask)][T][B] or NULL
  uint32_t grad_mask;
  const double* grad_sums;      // [NOUT][B] or NULL
  double* grad_alpha;           // [L][B]
  double* grad_n;
  double* grad_ksat;
  double* grad_pdm;             // [B] (or [1] with reduce) dL/d ponded_depth_max, or NULL
  // per resident warp scratch
  TapeEntry* tape;              // [slots][arena_cap][32]: the tapes of all sub-steps of one chunk, back to back
  unsigned char* meta;          // [slots][ring_steps][32] StepMeta
  double* adj;                  // [slots][num_leaves + step_cap][32]
  double* lam;                  // [ntiles][num_leaves][32]: adjoint of the column state between chunks
  double* gpar;                 // [ntiles][NPAR_IDS][32]: running parameter gradients between chunks
  int32_t* rev_done;            // [ntiles] chunks of the reverse pass completed per tile
  int32_t* rev_flags;           // [ntiles][32] tape overflow seen so far
  unsigned long long* next_tile;  // item counter
  int32_t ring_steps;           // chunk_steps * S
  int32_t arena_cap;            // tape entries per lane for one chunk
  int32_t step_cap;             // max entries of one sub-step (ids are 16 bit)
  int32_t* tape_overflow;       // [B] set to 1 if a column's tape overflowed (gradient invalid)
  int32_t reduce;               // 1: shared parameters -- per-tile sums into `partials`, no per-column gradients
  double* partials;             // [ntiles][NPAR_IDS]
  unsigned long long* counters; // [8] diagnostics (lgar_gradients.counters)
};

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

__host__ inline size_t backward_meta_bytes(int FM) {
  return FM == 16 ? sizeof(StepMeta<16>) : (FM == 12 ? sizeof(StepMeta<12>) : sizeof(StepMeta<8>));
}
__host__ inline size_t backward_scratch_bytes(int S, int FM, int chunk, int slots, int arena_cap, int step_cap, int ntiles) {
  const size_t ring_steps = (size_t)chunk * S;
  const size_t nl = NPAR_IDS + 5 * (size_t)FM + 2 + NGIUH;
  size_t per = (size_t)arena_cap * 32 * sizeof(TapeEntry) + ring_steps * 32 * backward_meta_bytes(FM) +
               (nl + step_cap) * 32 * 8;
  size_t per_tile = nl * 32 * 8 + (size_t)NPAR_IDS * 32 * 8 + 32 * 4 + 4;
  return per * slots + per_tile * ntiles + 16384;
}

// GM = 0: trapezoid Geff only (closed-form branch compiled out of the taped sub-step); GM = 2: run-time switch
template <int FM, int GM>
__global__ void __launch_bounds__(NT, 2) lgar_backward_kernel(const BParams P) {  // 2 CTAs per SM: up to 255 registers
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm_fields = reinterpret_cast<double*>(smem_raw);                       // [5*FM][NT]
  double* sm_nodes = sm_fields + 5 * FM * NT;                                    // [WARPS][NODEBUF]
  short* sm_ids = reinterpret_cast<short*>(sm_nodes + WARPS * NODEBUF);          // [5*FM][NT]
  uint8_t* sm_flags = reinterpret_cast<uint8_t*>(sm_ids + 5 * FM * NT);          // [FM][NT]
  __shared__ unsigned long long sm_item[WARPS];
  pow_tables_to_shared();

  const KParams& K = P.K;
  const lgar_problem& p = K.p;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int slot = blockIdx.x * WARPS + warp;  // resident-warp scratch slot
  double* nodebuf = sm_nodes + warp * NODEBUF;
  const int Tn = p.num_steps, S = p.num_subcycles;
  const size_t B = p.num_columns;
  constexpr int NL = num_leaves<FM>();

  TapeEntry* arena = P.tape + (size_t)slot * P.arena_cap * 32 + lane;
  StepMeta<FM>* metas = reinterpret_cast<StepMeta<FM>*>(P.meta) + (size_t)slot * P.ring_steps * 32 + lane;  // [j * 32]
  double* adj = P.adj + (size_t)slot * (NL + P.step_cap) * 32 + lane;
  TapeCtl& tc = g_tapectl[threadIdx.x];
  tc.first_id = NL;
  // Geff partials of the taped recompute go through the warp's adjoint array (idle until the reverse sweep)
  if (lane == 0) g_geffq_partials[warp] = P.adj + (size_t)slot * (NL + P.step_cap) * 32;
  __syncwarp();

  Tile<FM, Var, 2> Tv;
  Tv.col.fb = sm_fields + threadIdx.x;
  Tv.col.ib = sm_ids + threadIdx.x;
  Tv.col.gb = sm_flags + threadIdx.x;
  Tv.ctx.iter_cap = K.iter_cap;
  Column<FM, Var, 2>& C = Tv.col;
  const unsigned long long nitems = (unsigned long long)K.ntiles * K.nchunks;

  for (;;) {
    if (lane == 0) sm_item[warp] = atomicAdd(P.next_tile, 1ULL);
    __syncwarp();
    const unsigned long long item = sm_item[warp];
    __syncwarp();
    if (item >= nitems) break;
    const int chunk = K.nchunks - 1 - (int)(item / K.ntiles);   // last chunk first
    const int tile = (int)(item % K.ntiles);
    const bool first_item = (chunk == K.nchunks - 1);
    if (!first_item) {  // wait for the adjoint state of chunk + 1 (acquire)
      if (lane == 0) {
        volatile int32_t* d = P.rev_done + tile;
        while (*d < K.nchunks - 1 - chunk) __nanosleep(200);
      }
      __syncwarp();
      __threadfence();
    }
    const int slot_c = tile * 32 + lane;   // position in the tile grid (checkpoints); b = ensemble column
    const bool valid = (size_t)slot_c < B;
    const int slot_cc = valid ? slot_c : (int)B - 1;
    const int b = p.column_order ? __ldg(p.column_order + slot_cc) : slot_cc;
    const int bb = b;
    double* lam = P.lam + (size_t)tile * NL * 32 + lane;
    double* gsave = P.gpar + (size_t)tile * NPAR_IDS * 32 + lane;

    // final status of the forward pass: steps at and after the crash step have no gradient
    const int final_st = __ldcg(K.state_i + ((size_t)K.nchunks * NI_STATE + 2) * K.Bp + slot_cc);
    const int final_crash = __ldcg(K.state_i + ((size_t)K.nchunks * NI_STATE + 3) * K.Bp + slot_cc);
    const int t_end = (final_st == 0) ? Tn : final_crash;  // steps [0, t_end) produced outputs

    load_params(K, bb, Tv);
    for (int l = 0; l < C.L; l++) {
      C.soil[l].id_alpha = 3 * l;
      C.soil[l].id_n = 3 * l + 1;
      C.soil[l].id_ksat = 3 * l + 2;
      C.soil[l].id_m = -1;
    }
    C.id_pdm = P.grad_pdm ? ID_PDM : -1;  // ponded_depth_max as a gradient leaf (models/dpLGAR.py:48, commented out upstream)
    const int site = (p.site_index && valid) ? __ldg(p.site_index + b) : 0;
    const double* frc = p.forcing + (size_t)site * Tn * 2;
    double gpar[NPAR_IDS];
    bool overflow = false;
    if (first_item) {
      for (int q = 0; q < NL; q++) __stcg(lam + (size_t)q * 32, 0.0);
#pragma unroll
      for (int q = 0; q < NPAR_IDS; q++) gpar[q] = 0.0;
    } else {
#pragma unroll
      for (int q = 0; q < NPAR_IDS; q++) gpar[q] = __ldcg(gsave + (size_t)q * 32);
      overflow = __ldcg(P.rev_flags + (size_t)tile * 32 + lane) != 0;
    }
    unsigned long long cyc_fwd = 0, cyc_rev = 0, n_entries = 0, n_sub = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) Tv.ctx.ph[k] = 0;

    {
      const long long clk_a = clock64();
      const int t0 = chunk * K.chunk_steps;
      const int t1 = min(Tn, t0 + K.chunk_steps);
      // ---- forward through the chunk ON THE TAPE, from the checkpoint the forward kernel stored
      load_state(K, chunk, slot_cc, Tv);
      if (K.slog) {  // end points of the root finders, logged by the forward pass
        C.logp = K.slog + (size_t)chunk * K.slog_cap * K.Bp + slot_cc;
        C.log_pos = 0;
        C.log_valid = valid ? min(__ldcg(K.slog_count + (size_t)chunk * K.Bp + slot_cc), K.slog_cap) : 0;
        C.log_stride = K.Bp;
      } else {
        C.logp = nullptr;
        C.log_pos = C.log_valid = C.log_stride = 0;
      }
      int arena_used = 0;
      for (int t = t0; t < t1; t++) {
        const double2 x = __ldg(reinterpret_cast<const double2*>(frc) + t);
        for (int sc = 0; sc < S; sc++) {
          const int j = (t - t0) * S + sc;
          const bool alive = valid && (t < t_end) && (Tv.ctx.st == 0) && !overflow;
          // the state in front of this sub-step becomes the leaves of its tape
          for (int i = 0; i < C.n; i++)
#pragma unroll
            for (int k = 0; k < 5; k++) C.fid(k, i) = (short)(leaf_fields<FM>() + k * FM + i);
          C.ponded_water.id = leaf_ponded<FM>();
          C.ending_volume.id = leaf_endvol<FM>();
          for (int i = 0; i < NGIUH; i++) C.giuh[i].id = leaf_giuh<FM>() + i;
          tc.base = arena + (size_t)arena_used * 32;
          tc.n = 0;
          tc.cap = min(P.step_cap, P.arena_cap - arena_used);
          // derived parameters on the tape: m = 1 - 1/n (data/utils.py:75), psi_wp (aet.py:37-43)
          for (int l = 0; l < C.L; l++) {
            SoilT<Var>& sl = C.soil[l];
            Var mV = 1.0 - (1.0 / Var(sl.n, sl.id_n));
            sl.id_m = mV.id;
          }
          if (x.y > 0.0) precompute_psi_wp(Tv, p.wilting_point_psi);
#pragma unroll
          for (int k = 0; k < NOUT; k++) Tv.acc[k] = Var(0.0);
          substep<FM, Var, GM>(Tv, alive, x.x, x.y, K, nodebuf);
          __syncwarp();
          if (tc.n > tc.cap) overflow = true;
          const int ne = min(tc.n, tc.cap);
          if (alive) {
            n_entries += (unsigned long long)ne;
            n_sub++;
          }
          StepMeta<FM>& M = metas[(size_t)j * 32];
          M.n_entries = ne;
          M.n_fronts = C.n;
          M.alive = (int16_t)(alive && Tv.ctx.st == 0 && !overflow);
          M.id_ponded = (int16_t)C.ponded_water.id;
          M.id_endvol = (int16_t)C.ending_volume.id;
          for (int i = 0; i < NGIUH; i++) M.id_giuh[i] = (int16_t)C.giuh[i].id;
#pragma unroll
          for (int k = 0; k < NOUT; k++) M.id_acc[k] = (int16_t)Tv.acc[k].id;
          for (int i = 0; i < C.n; i++)
#pragma unroll
            for (int k = 0; k < 5; k++) M.id_field[k * FM + i] = C.fid(k, i);
          arena_used += ne;
        }
      }
      __syncwarp();
      const long long clk_b = clock64();
      cyc_fwd += (unsigned long long)(clk_b - clk_a);
      // ---- reverse sweep over the sub-steps of the chunk
      for (int t = t1 - 1; t >= t0; t--) {
        for (int sc = S - 1; sc >= 0; sc--) {
          const int j = (t - t0) * S + sc;
          const StepMeta<FM>& M = metas[(size_t)j * 32];
          const int ne = M.n_entries;
          arena_used -= ne;
          if (!M.alive) continue;
          const TapeEntry* tape = arena + (size_t)arena_used * 32;
          for (int q = 0; q < NL + ne; q++) adj[(size_t)q * 32] = 0.0;
          for (int i = 0; i < M.n_fronts; i++)
#pragma unroll
            for (int k = 0; k < 5; k++) {
              const int id = M.id_field[k * FM + i];
              if (id >= 0) adj[(size_t)id * 32] += __ldcg(lam + (size_t)(leaf_fields<FM>() + k * FM + i) * 32);
            }
          if (M.id_ponded >= 0) adj[(size_t)M.id_ponded * 32] += __ldcg(lam + (size_t)leaf_ponded<FM>() * 32);
          if (M.id_endvol >= 0) adj[(size_t)M.id_endvol * 32] += __ldcg(lam + (size_t)leaf_endvol<FM>() * 32);
          for (int i = 0; i < NGIUH; i++)
            if (M.id_giuh[i] >= 0) adj[(size_t)M.id_giuh[i] * 32] += __ldcg(lam + (size_t)(leaf_giuh<FM>() + i) * 32);
          // dL / d(outputs of this forcing step)
#pragma unroll
          for (int k = 0; k < NOUT; k++) {
            double g = 0.0;
            const bool state_out = (k == LGAR_OUT_ENDING_VOLUME || k == LGAR_OUT_PONDED_WATER);
            if (P.grad_per_step && (P.grad_mask & (1u << k)))
              g += __ldg(P.grad_per_step + ((size_t)__popc(P.grad_mask & ((1u << k) - 1u)) * Tn + t) * B + b);
            if (P.grad_sums && (!state_out || t == Tn - 1)) g += __ldg(P.grad_sums + (size_t)k * B + b);
            if (g == 0.0) continue;
            int id = -1;
            if (k == LGAR_OUT_ENDING_VOLUME) id = (sc == S - 1) ? M.id_endvol : -1;
            else if (k == LGAR_OUT_PONDED_WATER) id = (sc == S - 1) ? M.id_ponded : -1;
            else id = M.id_acc[k];
            if (id >= 0) adj[(size_t)id * 32] += g;
          }
          // the tape comes back from DRAM (the arenas of all resident warps are far larger than L2): fetch eight
          // entries at a time, independently of the adjoints, so that the misses overlap instead of queueing behind
          // the dependent chain adj -> entry -> adj
          for (int e0 = ne - 1; e0 >= 0; e0 -= 8) {
            TapeEntry te8[8];
#pragma unroll
            for (int k = 0; k < 8; k++)
              if (e0 - k >= 0) te8[k] = tape[(size_t)(e0 - k) * 32];
#pragma unroll
            for (int k = 0; k < 8; k++) {
              const int e = e0 - k;
              if (e >= 0) {
                const double g = adj[(size_t)(NL + e) * 32];
                if (g != 0.0) {
                  const TapeEntry te = te8[k];
                  if (te.a >= 0) adj[(size_t)te.a * 32] += g * te.da;
                  if (te.b >= 0) adj[(size_t)te.b * 32] += g * te.db;
                }
              }
            }
          }
          for (int q = NPAR_IDS; q < NL; q++) __stcg(lam + (size_t)q * 32, adj[(size_t)q * 32]);
#pragma unroll
          for (int q = 0; q < NPAR_IDS; q++) gpar[q] += adj[(size_t)q * 32];
        }
      }
      __syncwarp();
      cyc_rev += (unsigned long long)(clock64() - clk_b);
    }
    if (chunk > 0) {
      // hand the running state to the item (tile, chunk - 1): lambda is already in place (global memory)
#pragma unroll
      for (int q = 0; q < NPAR_IDS; q++) gsave[(size_t)q * 32] = gpar[q];
      P.rev_flags[(size_t)tile * 32 + lane] = overflow ? 1 : 0;
    }
    // ---- the initial state depends on the parameters: theta_init = theta_l(psi_init), K_init
    //      (data/utils.py:82-84, WettingFront.py:38-48); ending_volume(0) = mass_balance()
    if (chunk == 0) {
      tc.base = arena;
      tc.n = 0;
      tc.cap = min(P.step_cap, P.arena_cap);
      Tv.ctx.st = 0;
      for (int l = 0; l < C.L; l++) {
        SoilT<Var>& sl = C.soil[l];
        Var mV = 1.0 - (1.0 / Var(sl.n, sl.id_n));
        sl.id_m = mV.id;
      }
      init_column(Tv, __ldg(p.initial_psi + bb), p.use_closed_form_G != 0);
      const int ne = min(tc.n, tc.cap);
      if (valid && Tv.ctx.st == 0) {
        for (int q = 0; q < NL + ne; q++) adj[(size_t)q * 32] = 0.0;
        for (int i = 0; i < C.n; i++)
#pragma unroll
          for (int k = 0; k < 5; k++) {
            const int id = C.fid(k, i);
            if (id >= 0) adj[(size_t)id * 32] += __ldcg(lam + (size_t)(leaf_fields<FM>() + k * FM + i) * 32);
          }
        if (C.ending_volume.id >= 0) adj[(size_t)C.ending_volume.id * 32] += __ldcg(lam + (size_t)leaf_endvol<FM>() * 32);
        for (int e = ne - 1; e >= 0; e--) {
          const double g = adj[(size_t)(NL + e) * 32];
          if (g != 0.0) {
            const TapeEntry te = arena[(size_t)e * 32];
            if (te.a >= 0) adj[(size_t)te.a * 32] += g * te.da;
            if (te.b >= 0) adj[(size_t)te.b * 32] += g * te.db;
          }
        }
#pragma unroll
        for (int q = 0; q < NPAR_IDS; q++) gpar[q] += adj[(size_t)q * 32];
      }
    }
    if (chunk > 0) {
      // (nothing to write yet)
    } else if (P.reduce) {
      // shared parameters: sum over the 32 columns of the tile in a fixed (butterfly) order; overflowed and
      // out-of-range lanes contribute 0
#pragma unroll
      for (int q = 0; q < NPAR_IDS; q++) {
        double v = (valid && !overflow) ? gpar[q] : 0.0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if (lane == 0) P.partials[(size_t)tile * NPAR_IDS + q] = v;
      }
    } else if (valid) {
      const double qnan = __longlong_as_double(0x7ff8000000000000LL);
      for (int l = 0; l < p.num_layers; l++) {
        P.grad_alpha[(size_t)l * B + b] = overflow ? qnan : gpar[3 * l];
        P.grad_n[(size_t)l * B + b] = overflow ? qnan : gpar[3 * l + 1];
        P.grad_ksat[(size_t)l * B + b] = overflow ? qnan : gpar[3 * l + 2];
      }
      if (P.grad_pdm) P.grad_pdm[b] = overflow ? qnan : gpar[ID_PDM];
    }
    if (chunk == 0 && valid && P.tape_overflow) P.tape_overflow[b] = overflow ? 1 : 0;
    if (P.counters) {
      if (lane == 0) {
        atomicAdd(P.counters + 0, cyc_fwd);
        atomicAdd(P.counters + 1, cyc_rev);
#pragma unroll
        for (int k = 0; k < 3; k++) atomicAdd(P.counters + 5 + k, Tv.ctx.ph[k == 0 ? 1 : (k == 1 ? 3 : 0)] + (k == 2 ? Tv.ctx.ph[2] : 0ULL));
      }
      if (valid) {
        atomicAdd(P.counters + 2, n_entries);
        atomicAdd(P.counters + 3, n_sub);
        if (chunk == 0 && overflow) atomicAdd(P.counters + 4, 1ULL);
      }
    }
    // publish (release): the adjoint state of this chunk is complete
    __threadfence();
    __syncwarp();
    if (lane == 0) atomicExch(P.rev_done + tile, K.nchunks - chunk);
  }
}

}  // namespace lgar
