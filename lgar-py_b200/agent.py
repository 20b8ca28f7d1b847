"""Calibration agent on top of the B200 kernels (SURVEY 8f N2): the reference's training loop with whole forcing
records per launch, several sites per rank, one gradient all-reduce per optimiser step and checkpoint save / load.

Mirrors dpLGAR/agents/DifferentiableLGAR.py:19-196 (same method names, same loss, same optimiser, same logging of the
global mass balance as models/physics/MassBalance.py:77-108), with these differences by design:

  * the reference feeds one forcing row per `model(x)` call and accumulates `y_hat_[i] = runoff`
    (DifferentiableLGAR.py:113-124); here an epoch is ONE persistent forward launch over the whole record
    (`model.forward_record`) and ONE reverse launch (`loss.backward()` -> lgar_backward);
  * `sites > 1`: every rank may hold several forcing records / observation series; the parameters are shared, the
    per-site losses are averaged, and with `torch.distributed` initialised the loss and the 3L parameter gradients
    are summed over ranks with a single all-reduce (NCCL on the GPU box, gloo in the CPU tests) -- the reference has
    no distributed code;
  * `save_checkpoint` / `load_checkpoint` are implemented (the reference raises NotImplementedError,
    agents/DifferentiableLGAR.py:179-196).

Host-side helpers (`derive_time_config`, `RangeBoundLoss`, `mse_loss`, `calculate_nse`, `mass_balance_report`) are
plain torch / numpy and are covered by CPU tests against the reference's own functions.
"""
from __future__ import annotations

import logging
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from . import parallel
from ._capi import OUT_NAMES, status_message
from .model import _get

log = logging.getLogger("agents.DifferentiableLGAR")


def _set(cfg, path, value):
    keys = path.split(".")
    cur = cfg
    for key in keys[:-1]:
        cur = cur[key] if isinstance(cur, dict) else getattr(cur, key)
    if isinstance(cur, dict):
        cur[keys[-1]] = value
    else:
        setattr(cur, keys[-1], value)


def derive_time_config(cfg):
    """agents/DifferentiableLGAR.py:35-52: fill cfg.models.{endtime_s, subcycle_length_h, forcing_resolution_h,
    time_per_step, nsteps, num_subcycles} from the user-facing keys, with the reference's arithmetic (Q17)."""
    hr_to_sec = float(_get(cfg, "conversions.hr_to_sec", 3600.0))
    endtime_s = _get(cfg, "models.endtime") * hr_to_sec
    subcycle_length_h = _get(cfg, "models.subcycle_length") * (1 / hr_to_sec)
    forcing_resolution_h = _get(cfg, "models.forcing_resolution") / hr_to_sec
    time_per_step = forcing_resolution_h * hr_to_sec
    _set(cfg, "models.endtime_s", endtime_s)
    _set(cfg, "models.subcycle_length_h", subcycle_length_h)
    _set(cfg, "models.forcing_resolution_h", forcing_resolution_h)
    _set(cfg, "models.time_per_step", time_per_step)
    _set(cfg, "models.nsteps", int(endtime_s / time_per_step))
    _set(cfg, "models.num_subcycles", int(forcing_resolution_h / subcycle_length_h))
    return cfg


def mse_loss(y_hat: torch.Tensor, y_t: torch.Tensor) -> torch.Tensor:
    """models/functions/loss.py:7 (nn.MSELoss, mean reduction)."""
    return torch.mean((y_hat - y_t) ** 2)


class RangeBoundLoss(torch.nn.Module):
    """models/functions/loss.py:10-40: penalty for parameters outside [lb, ub].  Quirks kept: the upper-bound term
    of a parameter list is a SUM, the lower-bound term a MEAN; the last entry of `params` is a plain tensor."""

    def __init__(self, lb, ub, factor=1.0):
        super().__init__()
        self.lb = torch.tensor(list(lb), dtype=torch.float64)
        self.ub = torch.tensor(list(ub), dtype=torch.float64)
        self.factor = torch.tensor(float(factor), dtype=torch.float64)

    def forward(self, params):
        loss = torch.tensor(0.0, dtype=torch.float64)
        for i in range(len(params) - 1):
            p = torch.stack([q.to("cpu") for q in params[i]])
            loss = loss + torch.sum(self.factor * torch.relu(p - self.ub[i])) \
                        + torch.mean(self.factor * torch.relu(self.lb[i] - p))
        last = torch.as_tensor(params[-1], dtype=torch.float64).to("cpu")
        return loss + self.factor * torch.relu(last - self.ub[-1]) + self.factor * torch.relu(self.lb[-1] - last)


def calculate_nse(modeled, observed) -> float:
    """data/metrics.py:4-8."""
    modeled, observed = np.asarray(modeled, dtype=np.float64), np.asarray(observed, dtype=np.float64)
    return float(1 - np.divide(np.sum(np.power(observed - modeled, 2)), np.sum(np.power(observed - observed.mean(), 2))))


def mass_balance_report(totals: dict, starting_volume: float, giuh_queue_sum: float = 0.0, emit=log.info) -> float:
    """models/physics/MassBalance.py:77-108 from the per-record totals of the kernel outputs.  Returns the global
    balance error (cm)."""
    giuh = totals["giuh_runoff"] + giuh_queue_sum
    err = (starting_volume + totals["precip"] - totals["runoff"] - totals["AET"] - totals["ponded_water"]
           - totals["percolation"] - totals["ending_volume"])
    emit("********************************************************* ")
    emit("-------------------- Simulation Summary ----------------- ")
    emit("------------------------ Mass balance ------------------- ")
    emit(f"Initial water in soil    = {starting_volume:14f} cm")
    emit(f"Total precipitation      = {totals['precip']:14f} cm")
    emit(f"Total infiltration       = {totals['infiltration']:14f} cm")
    emit(f"Final water in soil      = {totals['ending_volume']:14f} cm")
    emit(f"Surface ponded water     = {totals['ponded_water']:14f} cm")
    emit(f"Surface runoff           = {totals['runoff']:14f} cm")
    emit(f"GIUH runoff              = {giuh:14f} cm")
    emit(f"Total percolation        = {totals['percolation']:14f} cm")
    emit(f"Total AET                = {totals['AET']:14f} cm")
    emit(f"Total PET                = {totals['PET']:14f} cm")
    emit(f"Total discharge (Q)      = {totals['discharge']:14f} cm")
    emit(f"Global balance           =   {err:.6e} cm")
    return float(err)


def reference_observations(nsteps: int) -> torch.Tensor:
    """data/Data.py:40: the reference has no observation reader wired in; it trains against
    `torch.rand([T])` drawn right after the agent's `torch.manual_seed(0)` (float64 default dtype)."""
    g = torch.Generator().manual_seed(0)
    return torch.rand([nsteps], dtype=torch.float64, generator=g)


class DifferentiableLGAR:
    """Drop-in for agents/DifferentiableLGAR.py.  `model` is anything with the dpLGAR surface plus `forward_record`
    (lgar_b200.model.dpLGAR); it is built from cfg when not given.  `x`: `[T, 2]` or `[sites, T, 2]` forcing in cm/h
    (read from cfg.data.forcing_file when None); `y`: observations `[T]` / `[sites, T]` (the reference's seeded
    random series when None)."""

    OUTPUTS = OUT_NAMES

    def __init__(self, cfg, model=None, x=None, y=None, device="cuda", group=None, on_column_error="raise") -> None:
        """on_column_error: "raise" (reference semantics: an exception inside model(x) aborts the run) or "mask"
        (sites whose column failed in this epoch are left out of the loss; useful with many sites per rank)."""
        assert on_column_error in ("raise", "mask")
        self.on_column_error = on_column_error
        self.cfg = cfg
        torch.manual_seed(0)
        torch.set_default_dtype(torch.float64)
        derive_time_config(cfg)
        nsteps = int(_get(cfg, "models.nsteps"))
        if x is None:
            from .forcing import read_forcing
            x = read_forcing(_get(cfg, "data.forcing_file"), nrows=nsteps)
        x = torch.as_tensor(np.asarray(x), dtype=torch.float64)
        if x.dim() == 2:
            x = x[None]
        self.x = x[:, :nsteps].contiguous()                     # [sites, T, 2]
        T = self.x.shape[1]
        if y is None:
            y = reference_observations(T)[None].expand(self.x.shape[0], T)
        y = torch.as_tensor(np.asarray(y), dtype=torch.float64)
        self.y = (y[None] if y.dim() == 1 else y)[:, :T].contiguous()  # [sites, T]
        self.group = group
        if model is None:
            from .model import dpLGAR
            model = dpLGAR(cfg, columns=self.x.shape[0], device=device)
        self.model = model
        hp = "models.hyperparameters."
        self.warmup = int(_get(cfg, hp + "warmup", 0))
        self.epochs = int(_get(cfg, hp + "epochs", 1))
        self.criterion = mse_loss
        self.optimizer = torch.optim.Adam(self.model.parameters(), lr=float(_get(cfg, hp + "learning_rate", 1e-3)))
        self.range_bound_loss = RangeBoundLoss(_get(cfg, hp + "lb"), _get(cfg, hp + "ub"), factor=1.0)
        self.y_hat = None
        self.y_t = None
        self.current_epoch = 0
        self.history = []  # (epoch, loss, nse)
        self.last_balance_error = None

    # ---- reference surface -----------------------------------------------------------------
    def run(self):
        try:
            self.train()
        except KeyboardInterrupt:
            log.info("You have entered CTRL+C.. Wait to finalize")

    def train(self):
        self.model.train()
        for _ in range(1, self.epochs + 1):
            self.train_one_epoch()
            self.current_epoch += 1
            self.model.set_internal_states()

    def train_one_epoch(self):
        """One pass over the record(s): one forward launch, mass-balance report, then `validate()`."""
        self.optimizer.zero_grad()
        out = self.model.forward_record(self.x if self.x.shape[0] > 1 else self.x[0], outputs=self.OUTPUTS,
                                        on_status="ignore")
        st = out.get("status")
        keep = None
        failed = st is not None and bool((st != 0).any())
        msg = ""
        if failed:
            first = int((st.reshape(-1) != 0).nonzero()[0, 0])
            msg = status_message(first, int(st.reshape(-1)[first]), int(out["crash_step"].reshape(-1)[first]))
        if self.on_column_error == "raise" and self._any_rank(failed):
            # every rank leaves together: a lone raise would leave the others waiting in the gradient all-reduce
            raise RuntimeError(msg or "LGAR column failure on another rank")
        if failed:
            keep = (st.reshape(-1) == 0)
            log.warning(f"{int((~keep).sum())} of {keep.numel()} sites left out of this epoch: {msg}")
        self._report_mass(out)
        y_hat = out["runoff"]
        if y_hat.dim() == 1:
            y_hat = y_hat[:, None]
        y_hat = y_hat.transpose(0, 1)                           # [sites, T]
        y_t = self.y.to(y_hat.device)
        if keep is not None:
            y_hat, y_t = y_hat[keep], y_t[keep]
        self.y_hat = y_hat[:, self.warmup:]
        self.y_t = y_t[:, self.warmup:]
        self._no_sites = keep is not None and int(keep.sum()) == 0
        self.validate()

    def validate(self) -> None:
        """Loss = MSE(y_hat, y_t) + RangeBoundLoss(params); backward through the reverse-mode kernel; Adam step
        (agents/DifferentiableLGAR.py:136-171).  With several ranks the loss and gradients are averaged first."""
        if getattr(self, "_no_sites", False):
            # every site of this rank failed: contribute a zero loss and zero gradients (the collective still runs)
            nse = float("nan")
            loss_mse = self.y_hat.sum() * 0.0
        else:
            nse = calculate_nse(self.y_hat.detach().cpu().numpy().ravel(), self.y_t.cpu().numpy().ravel())
            loss_mse = self.criterion(self.y_hat, self.y_t)
        log.info(f"trained NSE: {nse:.4}")
        params = [self.model.alpha, self.model.n, self.model.ksat, self.model.ponded_depth_max]
        bound_loss = self.range_bound_loss(params).to(loss_mse.device)
        loss = loss_mse + bound_loss
        start = time.perf_counter()
        loss.backward()
        end = time.perf_counter()
        log.info(f"Back prop took : {(end - start):.6f} seconds")
        ens = getattr(self.model, "last_ensemble", None)
        overflowed = ens.check_tape_overflow(raise_error=False) if ens is not None else 0
        # one collective: the loss and the gradients averaged over the ranks (each rank counts 1), and whether any
        # rank's gradient is unusable
        ps = list(self.model.parameters())
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in ps]
        loss_val, mean_grads, unusable = parallel.allreduce_loss_and_grads(loss.detach(), 1, grads, self.group,
                                                                            overflowed > 0)
        log.info(f"Loss: {loss_val}")
        parallel.step_if_usable(ps, mean_grads, unusable, self.optimizer, overflowed)
        self.history.append((self.current_epoch, float(loss_val), nse))

    def save_checkpoint(self, file_name="checkpoint.pth.tar", is_best=0):
        if dist.is_available() and dist.is_initialized() and dist.get_rank(self.group) != 0:
            return  # the ranks hold identical parameters: rank 0 writes
        state = {"epoch": self.current_epoch, "model": self.model.state_dict(), "optimizer": self.optimizer.state_dict(),
                 "history": list(self.history)}
        tmp = file_name + ".tmp"
        torch.save(state, tmp)
        os.replace(tmp, file_name)
        if is_best:
            torch.save(state, os.path.join(os.path.dirname(file_name) or ".", "model_best.pth.tar"))

    def load_checkpoint(self, file_name):
        state = torch.load(file_name, map_location="cpu", weights_only=True)
        self.model.load_state_dict(state["model"])
        self.optimizer.load_state_dict(state["optimizer"])
        self.current_epoch = int(state["epoch"])
        self.history = list(state.get("history", []))
        self.model.set_internal_states()

    def finalize(self):
        self.save_checkpoint()

    # ---- helpers ----------------------------------------------------------------------------
    def _any_rank(self, flag: bool) -> bool:
        """Logical OR of a host flag over the ranks (so that all of them raise, or none)."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.group) == 1:
            return bool(flag)
        dev = next(self.model.parameters()).device if dist.get_backend(self.group) == "nccl" else torch.device("cpu")
        if dev.type != "cuda" and dist.get_backend(self.group) == "nccl":
            dev = torch.device("cuda", torch.cuda.current_device())
        t = torch.tensor([1.0 if flag else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return bool(t.item() > 0)

    def _report_mass(self, out):
        with torch.no_grad():
            col = lambda v: (v if v.dim() == 1 else v[:, 0]).detach()
            tot = {k: float(col(out[k]).nan_to_num().sum()) for k in self.OUTPUTS if k not in ("ending_volume", "ponded_water")}
            tot["ending_volume"] = float(col(out["ending_volume"])[-1])
            tot["ponded_water"] = float(col(out["ponded_water"])[-1])
            sv = out.get("start_volume")
            start = float(sv.reshape(-1)[0]) if sv is not None else float(self.model.ending_volume)
            self.last_balance_error = mass_balance_report(tot, start)
