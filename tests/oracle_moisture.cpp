// =====================================================================================
// tests/oracle_moisture.cpp -- soil-moisture outputs (include/lgar_b200.h) of the CPU oracle.
//
// TEST INFRASTRUCTURE ONLY, built by tests/oracle_moisture.py into a temporary directory.  It compiles the oracle
// (oracle/lgar_oracle.cpp, unchanged) into the same translation unit and reads the two outputs off the reference's own
// data structures -- one list of wetting fronts per layer -- after every forcing step:
//   W_l       the inner sum of Column::mass_balance_from(l) in the same order (0 for an empty list);
//   theta(z)  the theta of the first front of the list of the layer with cum[l-1] < z <= cum[l] whose depth >= z,
//             NaN below the column or when no front of that list qualifies.
// With the Dual scalar both come with their forward-mode tangents w.r.t. (alpha[L], n[L], ksat[L]): an independent
// check of the reverse-mode kernel's soil-moisture gradients.
// =====================================================================================
#include "../oracle/lgar_oracle.cpp"

template <class T>
static T layer_water(Column<T>& c, int l) {
  Layer<T>& ly = c.layers[l];
  T sum(0.0);
  const double base = (l == 0) ? 0.0 : (ly.cum - ly.thick);
  const int nf = (int)ly.wf.size();
  for (int i = 0; i < nf - 1; i++) sum = sum + (ly.wf[i]->depth - base) * (ly.wf[i]->theta - ly.wf[i + 1]->theta);
  if (nf > 0) sum = sum + (ly.wf[nf - 1]->depth - base) * ly.wf[nf - 1]->theta;
  return sum;
}

template <class T>
static const Front<T>* front_at_depth(const Column<T>& c, double z) {
  for (const auto& ly : c.layers) {
    if (z <= ly.cum) {
      for (const auto* f : ly.wf)
        if (val(f->depth) >= z) return f;
      return nullptr;
    }
  }
  return nullptr;
}

// One column: w[T][L], th[T][D]; with T = Dual also dw[T][L][3L], dth[T][D][3L].  Rows from the crash step on are left
// as the caller set them.
template <class T>
static void moisture_column(const lgar_oracle_cfg& cfg, const double* forcing, int T_, const double* depths, int nd,
                            double* w, double* dw, double* th, double* dth, int32_t* status, int32_t* crash_step) {
  const int L = cfg.num_layers, np = 3 * L;
  Column<T> col;
  int st = ST_OK, crash = -1, t = 0;
  const double qnan = std::nan("");
  try {
    if constexpr (std::is_same<T, Dual>::value) {
      Dual a[LGAR_LMAX], n[LGAR_LMAX], k[LGAR_LMAX];
      for (int l = 0; l < L; l++) {
        a[l] = Dual(cfg.alpha[l]); a[l].d[l] = 1.0;
        n[l] = Dual(cfg.n[l]); n[l].d[L + l] = 1.0;
        k[l] = Dual(cfg.ksat[l]); k[l].d[2 * L + l] = 1.0;
      }
      col.init(cfg, a, n, k);
    } else {
      col.init(cfg, cfg.alpha, cfg.n, cfg.ksat);
    }
    for (t = 0; t < T_; t++) {
      col.forward(forcing[2 * t], forcing[2 * t + 1]);
      for (int l = 0; l < L; l++) {
        const T v = layer_water(col, l);
        w[(size_t)t * L + l] = val(v);
        if constexpr (std::is_same<T, Dual>::value)
          if (dw) for (int q = 0; q < np; q++) dw[((size_t)t * L + l) * np + q] = v.d[q];
      }
      for (int d = 0; d < nd; d++) {
        const Front<T>* f = front_at_depth(col, depths[d]);
        th[(size_t)t * nd + d] = f ? val(f->theta) : qnan;
        if constexpr (std::is_same<T, Dual>::value)
          if (dth) for (int q = 0; q < np; q++) dth[((size_t)t * nd + d) * np + q] = f ? f->theta.d[q] : qnan;
      }
      col.reset_accumulators();
    }
  } catch (RefError& e) {
    st = e.code;
    crash = t;
  }
  if (status) *status = st;
  if (crash_step) *crash_step = crash;
}

extern "C" {
// B columns (column b reads forcing + site[b] * T * 2; site == NULL: record 0) on `nthreads` threads:
// w[B][T][L], th[B][T][D]; dw[B][T][L][3L] and dth[B][T][D][3L] optional (both NULL: plain double run).
int lgar_oracle_moisture_batch(const lgar_oracle_cfg* cfgs, int B, const double* forcing, const int32_t* site, int T_,
                               const double* depths, int nd, double* w, double* dw, double* th, double* dth,
                               int32_t* status, int32_t* crash_step, int nthreads) {
  if (nthreads < 1) nthreads = 1;
  std::atomic<int> next(0);
  auto work = [&]() {
    for (;;) {
      const int b = next.fetch_add(1);
      if (b >= B) return;
      const double* f = forcing + (site ? (size_t)site[b] * T_ * 2 : 0);
      const int L = cfgs[b].num_layers, np = 3 * L;
      double* wb = w + (size_t)b * T_ * L;
      double* thb = th + (size_t)b * T_ * nd;
      int32_t* sb = status ? status + b : nullptr;
      int32_t* cb = crash_step ? crash_step + b : nullptr;
      if (dw || dth)
        moisture_column<Dual>(cfgs[b], f, T_, depths, nd, wb, dw ? dw + (size_t)b * T_ * L * np : nullptr, thb,
                              dth ? dth + (size_t)b * T_ * nd * np : nullptr, sb, cb);
      else
        moisture_column<double>(cfgs[b], f, T_, depths, nd, wb, nullptr, thb, nullptr, sb, cb);
    }
  };
  std::vector<std::thread> pool;
  for (int i = 1; i < nthreads; i++) pool.emplace_back(work);
  work();
  for (auto& x : pool) x.join();
  return 0;
}
}  // extern "C"
