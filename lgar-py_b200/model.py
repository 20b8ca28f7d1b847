"""`dpLGAR`-compatible nn.Module on top of the B200 kernels (drop-in for the reference's model class).

Mirrors the public surface of dpLGAR/models/dpLGAR.py:30-430 that its callers use
(agents/DifferentiableLGAR.py:63-171, models/physics/MassBalance.py:31-108):

  * ctor `dpLGAR(cfg)`: the same cfg keys (SURVEY 8b): cfg.data.{layer_soil_type, layer_thickness, initial_psi,
    ponded_depth_max, wilting_point_psi, giuh_ordinates, soil_params_file, use_closed_form_G}, cfg.constants.{frozen_factor, nint},
    cfg.models.{subcycle_length_h, num_subcycles}; cfg may be an omegaconf DictConfig or any attribute/dict mapping;
  * parameters `.alpha/.n/.ksat` = nn.ParameterList of 0-dim float64 (initial values: the reference's
    read_test_params table, data/utils.py:108-180, rows = cfg.data.layer_soil_type, ksat * frozen_factor);
  * `forward(x[2]) -> (runoff, percolation)` advances ONE forcing row (state stays on the GPU; `resume` launches);
    accumulators `.precip .PET .AET .infiltration .runoff .percolation .giuh_runoff .discharge
    .groundwater_discharge`, `.ponded_water`, `.ending_volume` are kept and must be zeroed by the caller exactly like
    MassBalance.change_mass does;
  * `set_internal_states()` resets the column to its initial state with the current parameters;
  * soil moisture (definitions in include/lgar_b200.h): with `moisture_depths` (ctor kwarg, else
    cfg.data.moisture_depths) `forward_record` also returns `moisture[T,D]` (theta at those depths), `layer_water[T,L]`
    (cm) and `layer_theta[T,L]`; after every one-row `forward`, `.soil_moisture[D]` and `.layer_water[L]` hold the
    state at the end of that row (plain state, not accumulators: the caller's resets leave them alone).

Differences (by design): one-row `forward` is a no-grad convenience; training uses `forward_record(x[T,2])`, which runs
the whole record in one persistent launch and is differentiable through the reverse-mode kernel
(`y_hat = model.forward_record(data.x)["runoff"][warmup:]`).  A reference exception becomes `RuntimeError` carrying the
status name.  Several columns (`columns > 1`, identical configuration) can share the module for ensembles.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import torch
import torch.nn as nn

from . import _capi
from .columns import ColumnEnsemble, check_moisture_depths, forward_raw, lgar_columns
from ._capi import CAPACITY_STATUSES, OUT_NAMES, status_message  # noqa: F401 (CAPACITY_STATUSES: importable from here)

# data/utils.py:108-180 read_test_params (== alpha, n, Ks columns of data/vG_default_params.dat; rows 12-17 are
# Phillipsburg P-1..3 and Bushland B-1..3)
ALPHA_TABLE = (0.01, 0.02, 0.01, 0.03, 0.04, 0.03, 0.02, 0.03, 0.01, 0.02, 0.01, 0.01,
               0.0031297, 0.0083272, 0.0037454, 0.009567, 0.005288, 0.004467)
N_TABLE = (1.25, 1.42, 1.47, 1.75, 3.18, 1.21, 1.33, 1.45, 1.68, 1.32, 1.52, 1.66,
           1.6858, 1.299, 1.6151, 1.3579, 1.5276, 1.4585)
KSAT_TABLE = (0.612, 0.3348, 0.504, 4.32, 26.64, 0.468, 0.54, 1.584, 1.836, 0.432, 0.468, 0.756,
              0.45, 0.07, 0.45, 0.07, 0.02, 0.2)


def _get(cfg, path, default=None):
    cur = cfg
    for key in path.split("."):
        if cur is None:
            return default
        cur = cur.get(key) if isinstance(cur, dict) else getattr(cur, key, None)
    return default if cur is None else cur


def read_soil_table(path):
    """theta_r, theta_e columns of a vG_default_params*.dat file (whitespace separated, quoted texture names)."""
    thr, the = [], []
    with open(path) as f:
        next(f)
        for line in f:
            parts = line.replace('"', " ").split()
            if len(parts) >= 7:
                thr.append(float(parts[-6])); the.append(float(parts[-5]))
    return np.array(thr), np.array(the)


class dpLGAR(nn.Module):
    def __init__(self, cfg, theta_r=None, theta_e=None, columns: int = 1, device="cuda", moisture_depths=None) -> None:
        super().__init__()
        self.cfg = cfg
        soil_types = list(_get(cfg, "data.layer_soil_type"))
        self.thickness = np.array(_get(cfg, "data.layer_thickness"), dtype=np.float64)
        ff = float(_get(cfg, "constants.frozen_factor", 1.0))
        self.frozen_factor = ff
        self.ponded_depth_max = torch.tensor(float(_get(cfg, "data.ponded_depth_max", 0.0)), dtype=torch.float64)
        self.alpha = nn.ParameterList([nn.Parameter(torch.tensor(ALPHA_TABLE[i], dtype=torch.float64)) for i in soil_types])
        self.n = nn.ParameterList([nn.Parameter(torch.tensor(N_TABLE[i], dtype=torch.float64)) for i in soil_types])
        self.ksat = nn.ParameterList([nn.Parameter(torch.tensor(KSAT_TABLE[i] * ff, dtype=torch.float64)) for i in soil_types])
        if theta_r is None:
            thr, the = read_soil_table(_get(cfg, "data.soil_params_file"))
            theta_r, theta_e = thr[soil_types], the[soil_types]
        self.theta_r = np.asarray(theta_r, dtype=np.float64)
        self.theta_e = np.asarray(theta_e, dtype=np.float64)
        self.columns = int(columns)
        self.device = torch.device(device)
        self.dt_h = float(_get(cfg, "models.subcycle_length_h"))
        self.num_subcycles = int(_get(cfg, "models.num_subcycles"))
        giuh = tuple(float(g) for g in _get(cfg, "data.giuh_ordinates", (0.06, 0.51, 0.28, 0.12, 0.03)))
        self.global_params = SimpleNamespace(num_giuh_ordinates=len(giuh), giuh_runoff=torch.zeros(len(giuh), dtype=torch.float64),
                                             giuh_ordinates=giuh, num_layers=len(soil_types))
        self._ens_kw = dict(
            initial_psi=float(_get(cfg, "data.initial_psi", 2000.0)), ponded_depth_max=float(self.ponded_depth_max),
            subcycle_length_h=self.dt_h, num_subcycles=self.num_subcycles, nint=int(_get(cfg, "constants.nint", 120)),
            wilting_point_psi=float(_get(cfg, "data.wilting_point_psi", 15495.0)), frozen_factor=ff, giuh_ordinates=giuh,
            use_closed_form_G=bool(_get(cfg, "data.use_closed_form_G", False)))
        if moisture_depths is None:
            moisture_depths = _get(cfg, "data.moisture_depths")
        self.moisture_depths = check_moisture_depths(moisture_depths)
        self._ens_kw["moisture_depths"] = self.moisture_depths
        self._step_ens = None
        self._ws = None
        self.set_internal_states()

    # ---- helpers -----------------------------------------------------------------------
    def _params(self):
        a = torch.stack(list(self.alpha)); n = torch.stack(list(self.n)); k = torch.stack(list(self.ksat))
        return a, n, k

    def _ensemble(self, forcing, resume=False):
        L, B = len(self.alpha), self.columns
        rep = lambda v: np.repeat(np.asarray(v, dtype=np.float64).reshape(L, 1), B, axis=1)
        f = torch.as_tensor(forcing, dtype=torch.float64)
        site_index = None
        if f.dim() == 3 and f.shape[0] > 1:  # one forcing record per column (sites of a calibration batch)
            if f.shape[0] != B:
                raise ValueError(f"forcing has {f.shape[0]} sites but the module holds {B} columns")
            site_index = np.arange(B, dtype=np.int32)
        return ColumnEnsemble(theta_r=rep(self.theta_r), theta_e=rep(self.theta_e), thickness=rep(self.thickness),
                              forcing=f, site_index=site_index, resume=resume, device=self.device, **self._ens_kw)

    def _zero(self):
        return torch.tensor(0.0, dtype=torch.float64)

    # ---- reference API --------------------------------------------------------------------
    def set_internal_states(self):
        """models/dpLGAR.py:97-147: rebuild the column from the current parameters."""
        for name in ("precip", "PET", "AET", "infiltration", "runoff", "percolation", "giuh_runoff", "discharge",
                     "groundwater_discharge", "ponded_water", "previous_precip"):
            setattr(self, name, self._zero())
        self._started = False
        self._ws = None
        self.soil_moisture = None  # [D] theta at moisture_depths after the last one-row forward
        self.layer_water = None    # [L] cm
        # initial water volume: a zero-length-forcing run is not allowed, so use one dry row and read start_volume
        a, n, k = self._params()
        ens = self._ensemble(np.zeros((1, 2)))
        with torch.no_grad():
            res, _ = forward_raw(ens, a.detach(), n.detach(), k.detach(), outputs=("runoff",))
        self.ending_volume = res.start_volume[0].cpu()

    def forward(self, x):
        """One forcing row (P, PET in cm/h) -> cumulative (runoff, percolation) since the caller last zeroed them."""
        a, n, k = self._params()
        f = torch.as_tensor(x, dtype=torch.float64).reshape(1, 1, 2)
        ens = self._ensemble(f, resume=self._started)
        with torch.no_grad():
            res, self._ws = forward_raw(ens, a.detach(), n.detach(), k.detach(), outputs=OUT_NAMES, workspace=self._ws,
                                        moisture=len(self.moisture_depths) > 0, layer_water=True)
        self._started = True
        st = int(res.status[0])
        if st != 0:
            raise RuntimeError(status_message(0, st))
        v = {name: res[name][0, 0].cpu() for name in OUT_NAMES}
        for name in ("precip", "PET", "AET", "infiltration", "runoff", "percolation", "giuh_runoff", "discharge"):
            setattr(self, name, getattr(self, name) + v[name])
        self.ponded_water = v["ponded_water"]
        self.ending_volume = v["ending_volume"]
        self.soil_moisture = (res.moisture[:, 0, 0].cpu() if res.moisture is not None
                              else torch.zeros(0, dtype=torch.float64))
        self.layer_water = res.layer_water[:, 0, 0].cpu()
        return self.runoff, self.percolation

    def forward_record(self, x, outputs=("runoff", "percolation"), on_status="raise"):
        """Whole record `x[T,2]` in one persistent launch, from the initial state; differentiable in alpha/n/ksat.
        Returns a dict of `[T]` tensors (or `[T, columns]`).  on_status: what to do when a column ends with a non-zero
        status (its series are NaN from the crash step on): "raise" (default: the reference raises out of model(x)),
        "warn" or "ignore" (the caller inspects out["status"] itself, like the agent does).
        With moisture_depths configured the soil-moisture outputs are added: `moisture[T,D]`, `layer_water[T,L]`,
        `layer_theta[T,L]` (with `columns > 1`: `[T,D,columns]` and `[T,L,columns]`)."""
        a, n, k = self._params()
        outputs = tuple(outputs)
        if self.moisture_depths:
            outputs += tuple(nm for nm in ("moisture", "layer_water") if nm not in outputs)
        ens = self._ensemble(torch.as_tensor(x, dtype=torch.float64))
        self.last_ensemble = ens  # (the reverse pass leaves its tape-overflow flags there)
        # ponded_depth_max as a learnable parameter (models/dpLGAR.py:48, commented out upstream): make it one with
        # `model.ponded_depth_max = nn.Parameter(model.ponded_depth_max)` and it receives a gradient like alpha/n/ksat
        pdm = self.ponded_depth_max if getattr(self.ponded_depth_max, "requires_grad", False) else None
        out = lgar_columns(a, n, k, ens, outputs=outputs, ponded_depth_max=pdm)
        if on_status != "ignore":
            st = out["status"]
            if bool((st != 0).any()):
                first = int((st != 0).nonzero()[0, 0])
                msg = status_message(first, int(st[first]), int(out["crash_step"][first]))
                if on_status == "raise":
                    raise RuntimeError(msg)
                import warnings
                warnings.warn(msg)
        for key in ("moisture", "layer_water", "layer_theta"):  # [D or L, T, B] -> time first, like the other series
            if key in out:
                out[key] = out[key].permute(1, 0, 2)
        if self.columns == 1:
            out = {key: (val[..., 0] if val.dim() >= 1 and val.shape[-1] == 1 else val) for key, val in out.items()}
        return out

    def print_params(self):
        for name, plist in (("Alpha", self.alpha), ("n", self.n), ("Ksat", self.ksat)):
            for i, p in enumerate(plist):
                print(f"{name} for soil {i + 1}: {p.detach().item():.4f}")
        print(f"Max Ponded Depth: {float(self.ponded_depth_max):.4f}")
