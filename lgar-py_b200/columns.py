"""Batched LGAR columns on one B200: the torch-facing wrapper around the C ABI.

`ColumnEnsemble` holds what the reference keeps in `cfg` + `GlobalParams`
(dpLGAR/models/physics/GlobalParams.py:79-138) for B independent columns;
`lgar_columns(alpha, n, ksat, ens)` is the batched equivalent of running
`dpLGAR.forward(x[t])` for every row of the forcing record
(dpLGAR/agents/DifferentiableLGAR.py:117-125) and is differentiable in alpha/n/ksat through the
hand-written reverse-mode kernel (reference autograd semantics).

PyTorch is used for device memory, streams and autograd plumbing only; all arithmetic happens
in liblgar_b200.so.  There is no CPU path: tensors are moved to the CUDA device (H2D) if they
arrive on the host, and the call fails loudly if the library or an sm_100 GPU is missing.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Optional, Sequence

import torch

from . import _capi
from ._capi import NUM_OUTPUTS, OUT_NAMES, MAX_FRONTS, MAX_DEPTHS

F64 = torch.float64


def _dev_f64(x, device, shape=None):
    t = torch.as_tensor(x, dtype=F64)
    if shape is not None and tuple(t.shape) != tuple(shape):
        if t.dim() == 1 and len(shape) == 2 and t.shape[0] == shape[0]:
            t = t.unsqueeze(1)  # per-layer values shared by all columns
        t = t.expand(shape)
    return t.to(device, non_blocking=True).contiguous()


@dataclass
class ColumnEnsemble:
    """Static description of B soil columns with L layers each (everything except alpha/n/ksat).

    Array layouts follow the C ABI: `[L, B]` (layer-major, column fastest)."""
    theta_r: torch.Tensor           # [L,B]
    theta_e: torch.Tensor           # [L,B]
    thickness: torch.Tensor         # [L,B] cm
    forcing: torch.Tensor           # [sites,T,2] (P, PET) cm/h, or [T,2]
    site_index: Optional[torch.Tensor] = None   # [B] int32
    initial_psi: object = 2000.0    # scalar or [B]
    ponded_depth_max: object = 0.0  # scalar or [B]
    subcycle_length_h: float = 1.0
    num_subcycles: int = 1
    nint: int = 120
    wilting_point_psi: float = 15495.0
    frozen_factor: float = 1.0
    use_closed_form_G: bool = False  # cfg.data.use_closed_form_G (green_ampt.py:85-98)
    giuh_ordinates: Sequence[float] = (0.06, 0.51, 0.28, 0.12, 0.03)
    max_fronts: int = 16
    chunk_steps: int = 0             # forcing steps per scheduling / checkpoint chunk (0 = library default: 64 sub-steps)
    iter_cap: int = 0
    resume: bool = False             # continue from the state left in the workspace (see lgar_b200.h)
    column_order: Optional[torch.Tensor] = None  # [B] int32 permutation: placement of columns on warps (lgar_b200.h)
    reverse_counters: bool = False   # collect the reverse kernel's diagnostics counters (lgar_gradients.counters)
    last_tape_overflow: Optional[torch.Tensor] = field(default=None, repr=False)   # [B] int32 after a backward pass
    last_reverse_counters: Optional[torch.Tensor] = field(default=None, repr=False)
    device: object = "cuda"
    _keep: list = field(default_factory=list, repr=False)
    # sensor depths (cm below the surface, at most 8, each > 0) of the soil-moisture output theta(z), shared by all
    # columns (lgar_problem.moisture_depths; definition in lgar_b200.h).  Last, so positional arguments keep their meaning
    moisture_depths: Optional[Sequence[float]] = None

    def __post_init__(self):
        dev = torch.device(self.device)
        if dev.type != "cuda":
            raise _capi.LGARLibraryError("lgar_b200 has no CPU path: device must be a CUDA device")
        self.device = dev
        self.theta_r = _dev_f64(self.theta_r, dev)
        L, B = self.theta_r.shape
        self.theta_e = _dev_f64(self.theta_e, dev, (L, B))
        self.thickness = _dev_f64(self.thickness, dev, (L, B))
        f = torch.as_tensor(self.forcing, dtype=F64)
        if f.dim() == 2:
            f = f.unsqueeze(0)
        assert f.dim() == 3 and f.shape[2] == 2, "forcing must be [sites,T,2]"
        self.forcing = f.to(dev, non_blocking=True).contiguous()
        if self.site_index is not None:
            self.site_index = torch.as_tensor(self.site_index, dtype=torch.int32).to(dev).contiguous()
            assert self.site_index.shape == (B,)
        if self.column_order is not None:
            self.column_order = torch.as_tensor(self.column_order, dtype=torch.int32).to(dev).contiguous()
            assert self.column_order.shape == (B,)
        self.initial_psi = _dev_f64(self.initial_psi, dev, (B,))
        self.ponded_depth_max = _dev_f64(self.ponded_depth_max, dev, (B,))
        self.moisture_depths = check_moisture_depths(self.moisture_depths)

    @property
    def num_layers(self): return self.theta_r.shape[0]
    @property
    def num_columns(self): return self.theta_r.shape[1]
    @property
    def num_steps(self): return self.forcing.shape[1]
    @property
    def num_depths(self): return len(self.moisture_depths)

    def problem(self, alpha, n, ksat, ponded_depth_max=None) -> _capi.Problem:
        p = _capi.Problem()
        p.abi_version = _capi.ABI_VERSION
        p.num_columns, p.num_layers, p.num_steps = self.num_columns, self.num_layers, self.num_steps
        p.num_subcycles, p.num_sites = int(self.num_subcycles), self.forcing.shape[0]
        p.nint, p.num_giuh = int(self.nint), len(self.giuh_ordinates)
        p.max_fronts, p.chunk_steps, p.iter_cap = int(self.max_fronts), int(self.chunk_steps), int(self.iter_cap)
        p.resume = 1 if self.resume else 0
        p.use_closed_form_G = 1 if self.use_closed_form_G else 0
        p.subcycle_length_h = float(self.subcycle_length_h)
        p.wilting_point_psi = float(self.wilting_point_psi)
        p.frozen_factor = float(self.frozen_factor)
        for i, g in enumerate(self.giuh_ordinates):
            p.giuh_ordinates[i] = float(g)
        p.alpha, p.n, p.ksat = alpha.data_ptr(), n.data_ptr(), ksat.data_ptr()
        p.theta_r, p.theta_e, p.thickness = self.theta_r.data_ptr(), self.theta_e.data_ptr(), self.thickness.data_ptr()
        pdm = self.ponded_depth_max if ponded_depth_max is None else ponded_depth_max
        p.initial_psi, p.ponded_depth_max = self.initial_psi.data_ptr(), pdm.data_ptr()
        p.forcing = self.forcing.data_ptr()
        p.site_index = self.site_index.data_ptr() if self.site_index is not None else None
        p.column_order = self.column_order.data_ptr() if self.column_order is not None else None
        p.num_depths = self.num_depths
        for i, z in enumerate(self.moisture_depths):
            p.moisture_depths[i] = z
        return p

    def check_tape_overflow(self, raise_error=True) -> int:
        """Number of columns whose reverse-pass tape arena was exhausted in the last backward pass (synchronises).
        Their per-column gradients are NaN and the shared-parameter sums leave them out: do not step on them."""
        ov = self.last_tape_overflow
        cnt = int(ov.sum()) if ov is not None else 0
        if cnt and raise_error:
            raise _capi.LGARLibraryError(
                f"{cnt} column(s) exhausted the tape arena of the reverse pass: their gradients are not available "
                "(use a smaller chunk_steps, or mask these columns: ColumnEnsemble.last_tape_overflow)")
        return cnt

    def balance(self, ksat) -> "ColumnEnsemble":
        """Place columns of similar cost on the same warp.  A warp advances its 32 columns in lock step, so its time per
        step is that of its slowest lane.  Two things make lanes alike: (1) the same forcing record -- storms and dry
        spells then hit all lanes in the same steps (columns of one site stay together); (2) within a site, a similar
        top-layer conductivity: the number of root-finder iterations of a column follows ksat[0] (rank correlation 0.76
        on the bench ensemble: a conductive top layer sends the fronts into the deeper layers, where every move is a
        mass-balance root find).  Sets `column_order` = columns sorted by (site, ksat[0]); results do not depend on
        the placement (tests/test_gpu_properties.py)."""
        k0 = torch.as_tensor(ksat, dtype=F64)
        k0 = (k0[0] if k0.dim() == 2 else k0[0].expand(self.num_columns)).to(self.device)
        order = torch.argsort(k0, stable=True)
        if self.site_index is not None:
            order = order[torch.argsort(self.site_index[order].to(torch.int64), stable=True)]
        self.column_order = order.to(torch.int32).contiguous()
        return self


def check_moisture_depths(depths) -> tuple:
    """The sensor depths as a tuple of floats; raises ValueError for more than MAX_DEPTHS depths or a depth that is not
    finite and > 0 (before anything is launched)."""
    if depths is None:
        return ()
    z = tuple(float(v) for v in torch.as_tensor(depths, dtype=F64).reshape(-1).tolist())
    if len(z) > MAX_DEPTHS:
        raise ValueError(f"moisture_depths: at most {MAX_DEPTHS} depths, got {len(z)}")
    if not all(math.isfinite(v) and v > 0.0 for v in z):
        raise ValueError(f"moisture_depths: every depth must be finite and > 0 cm, got {z}")
    return z


def output_mask(names) -> int:
    m = 0
    for nme in names:
        m |= 1 << OUT_NAMES.index(nme)
    return m


@dataclass
class ForwardResult:
    per_step: Optional[torch.Tensor]   # [popcount(mask),T,B]: selected outputs in increasing index
    mask: int
    sums: torch.Tensor                 # [NOUT,B]
    start_volume: torch.Tensor         # [B]
    status: torch.Tensor               # [B] int32
    crash_step: torch.Tensor           # [B] int32
    num_fronts: Optional[torch.Tensor] = None      # [T,B]
    fronts: Optional[torch.Tensor] = None          # [T,16,5,B]
    front_layer: Optional[torch.Tensor] = None     # [T,16,B]
    front_to_bottom: Optional[torch.Tensor] = None # [T,16,B]
    counters: Optional[torch.Tensor] = None        # [16] int64: 8 work counters + phase timers (lgar_b200.h)
    tile_cycles: Optional[torch.Tensor] = None     # [ceil(B/32)] int64 (diagnostics); [3, ceil(B/32)] with counters
    moisture: Optional[torch.Tensor] = None        # [D,T,B] theta at ens.moisture_depths (lgar_b200.h)
    layer_water: Optional[torch.Tensor] = None     # [L,T,B] water stored in each layer, cm
    overflow_reruns: int = 0                       # columns rerun with the 32-front kernel (overflow_fallback)

    def __getitem__(self, name) -> torch.Tensor:
        k = OUT_NAMES.index(name)
        assert self.per_step is not None and (self.mask >> k) & 1, f"output {name} was not requested"
        return self.per_step[bin(self.mask & ((1 << k) - 1)).count("1")]


def _param(x, ens: ColumnEnsemble):
    t = torch.as_tensor(x, dtype=F64)
    if t.dim() == 1:  # one parameter set shared by all columns
        t = t.unsqueeze(1).expand(ens.num_layers, ens.num_columns)
    return t.to(ens.device, non_blocking=True).contiguous()


FRONT_OVERFLOW = 6  # lgar_status: more than max_fronts wetting fronts (capacity of the library, not a reference state)


def _rerun_overflowed(ens: ColumnEnsemble, alpha, n, ksat, res: "ForwardResult", outputs, per_step, moisture=False,
                      layer_water=False) -> int:
    """The reference's front lists are unbounded; the production kernels hold 16 fronts per column in shared memory.
    The (rare: ~0.07 % of the bench ensemble over a year) columns that overflow are run again with the 32-front
    instantiation (one CTA per SM) and their results scattered into `res`.  Returns the number of columns rerun."""
    idx = (res.status == FRONT_OVERFLOW).nonzero().flatten()
    if idx.numel() == 0 or int(ens.max_fronts) >= 32 or ens.resume:
        return 0
    sub = ColumnEnsemble(
        theta_r=ens.theta_r[:, idx], theta_e=ens.theta_e[:, idx], thickness=ens.thickness[:, idx], forcing=ens.forcing,
        site_index=(ens.site_index[idx] if ens.site_index is not None else None), initial_psi=ens.initial_psi[idx],
        ponded_depth_max=ens.ponded_depth_max[idx], subcycle_length_h=ens.subcycle_length_h,
        num_subcycles=ens.num_subcycles, nint=ens.nint, wilting_point_psi=ens.wilting_point_psi,
        frozen_factor=ens.frozen_factor, use_closed_form_G=ens.use_closed_form_G, giuh_ordinates=ens.giuh_ordinates,
        max_fronts=32, chunk_steps=ens.chunk_steps, iter_cap=ens.iter_cap, moisture_depths=ens.moisture_depths,
        device=ens.device)
    r2, _ = forward_raw(sub, alpha[:, idx].contiguous(), n[:, idx].contiguous(), ksat[:, idx].contiguous(), outputs=outputs,
                        per_step=per_step, num_fronts=res.num_fronts is not None, overflow_fallback=False,
                        moisture=moisture, layer_water=layer_water)
    if res.per_step is not None:
        res.per_step[:, :, idx] = r2.per_step
    if moisture:
        res.moisture[:, :, idx] = r2.moisture
    if layer_water:
        res.layer_water[:, :, idx] = r2.layer_water
    res.sums[:, idx] = r2.sums
    res.start_volume[idx] = r2.start_volume
    res.status[idx] = r2.status
    res.crash_step[idx] = r2.crash_step
    if res.num_fronts is not None:
        res.num_fronts[:, idx] = r2.num_fronts
    return int(idx.numel())


def forward_raw(ens: ColumnEnsemble, alpha, n, ksat, outputs=("runoff", "percolation"), per_step=True,
                num_fronts=False, dump_fronts=False, counters=False, tile_cycles=False, keep_checkpoints=False,
                workspace: Optional[torch.Tensor] = None, overflow_fallback=False, window=None,
                into: Optional[ForwardResult] = None, pipeline_seq: int = 0, ponded_depth_max=None, moisture=False,
                layer_water=False) -> tuple[ForwardResult, torch.Tensor]:
    """One persistent launch over all columns and all forcing steps (no autograd).
    overflow_fallback: rerun the columns that overflowed the front list with the 32-front kernel (synchronises:
    the status array is inspected on the host).
    window=(t0, t1): advance only forcing rows [t0, t1) of the record (lgar_problem.step_begin/step_end); t0 > 0
    continues from the state the previous call left in `workspace` (resume).  Rows of the per-step outputs and
    crash steps stay absolute, so `into=` (the ForwardResult of the previous window) lets consecutive windows fill
    one set of buffers; `sums` are the running totals since row 0.  A column that crashed in an EARLIER window
    reports crash_step = -2 - t (t = the absolute step).
    pipeline_seq=k (1, 2, ...): the k-th consecutive window of a pipelined sequence (lgar_problem.pipeline_seq):
    windows k > 1 start on the SMs the previous window has drained (programmatic dependent launch); enqueue nothing
    else on the stream between them.
    moisture / layer_water: also store the soil-moisture outputs of every step, `res.moisture[D,T,B]` (theta at
    ens.moisture_depths) and `res.layer_water[L,T,B]` (cm); definitions in lgar_b200.h.  Windows fill their rows like
    per_step."""
    L_ = _capi.lib()
    dev = ens.device
    if moisture and ens.num_depths == 0:
        raise ValueError("moisture=True needs ColumnEnsemble(moisture_depths=...)")
    alpha, n, ksat = _param(alpha, ens), _param(n, ens), _param(ksat, ens)
    B, T = ens.num_columns, ens.num_steps
    if ponded_depth_max is not None:  # [B] override of ens.ponded_depth_max (e.g. a learnable one)
        ponded_depth_max = _dev_f64(ponded_depth_max, dev, (B,))
    p = ens.problem(alpha, n, ksat, ponded_depth_max)
    if window is not None:
        p.step_begin, p.step_end = int(window[0]), int(window[1])
        if p.step_begin > 0:
            p.resume = 1
    p.pipeline_seq = int(pipeline_seq)
    need = L_.lgar_workspace_bytes(C.byref(p), 1 if keep_checkpoints else 0)
    if need == 0:
        _capi.check(-1, "lgar_workspace_bytes")
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    mask = output_mask(outputs) if per_step else 0
    o = _capi.Outputs()
    if into is not None:
        assert into.mask == mask and into.sums.shape[1] == B, "`into` must come from the same ensemble and outputs"
        res = into
    else:
        res = ForwardResult(
            per_step=torch.empty((bin(mask).count("1"), T, B), dtype=F64, device=dev) if mask else None, mask=mask,
            sums=torch.empty((NUM_OUTPUTS, B), dtype=F64, device=dev),
            start_volume=torch.empty(B, dtype=F64, device=dev),
            status=torch.empty(B, dtype=torch.int32, device=dev),
            crash_step=torch.empty(B, dtype=torch.int32, device=dev))
    o.per_step = res.per_step.data_ptr() if mask else None
    o.per_step_mask = mask
    o.sums, o.start_volume = res.sums.data_ptr(), res.start_volume.data_ptr()
    o.status, o.crash_step = res.status.data_ptr(), res.crash_step.data_ptr()
    if moisture:
        if res.moisture is None:
            res.moisture = torch.empty((ens.num_depths, T, B), dtype=F64, device=dev)
        o.moisture = res.moisture.data_ptr()
    if layer_water:
        if res.layer_water is None:
            res.layer_water = torch.empty((ens.num_layers, T, B), dtype=F64, device=dev)
        o.layer_water = res.layer_water.data_ptr()
    if num_fronts or dump_fronts:
        if res.num_fronts is None:
            res.num_fronts = torch.empty((T, B), dtype=torch.int32, device=dev)
        o.num_fronts = res.num_fronts.data_ptr()
    if dump_fronts:
        res.fronts = torch.empty((T, MAX_FRONTS, 5, B), dtype=F64, device=dev)
        res.front_layer = torch.empty((T, MAX_FRONTS, B), dtype=torch.int8, device=dev)
        res.front_to_bottom = torch.empty((T, MAX_FRONTS, B), dtype=torch.int8, device=dev)
        o.fronts, o.front_layer = res.fronts.data_ptr(), res.front_layer.data_ptr()
        o.front_to_bottom = res.front_to_bottom.data_ptr()
    if counters or dump_fronts:
        res.counters = torch.zeros(16, dtype=torch.int64, device=dev)
        o.counters = res.counters.data_ptr()
    if tile_cycles:
        # with the counting kernel: [3, tiles] = busy cycles, cycles waiting for the predecessor chunk, finish time (ns)
        rows = 3 if counters else 1
        res.tile_cycles = torch.zeros((rows, (B + 31) // 32) if rows == 3 else ((B + 31) // 32,), dtype=torch.int64, device=dev)
        o.tile_cycles = res.tile_cycles.data_ptr()
        o.tile_diag_rows = rows
    stream = torch.cuda.current_stream(dev).cuda_stream
    with torch.cuda.device(dev):
        rc = L_.lgar_forward(C.byref(p), C.byref(o), workspace.data_ptr(), workspace.numel(),
                             1 if keep_checkpoints else 0, C.c_void_p(stream))
    _capi.check(rc, "lgar_forward")
    res._keep = (alpha, n, ksat, ens, ponded_depth_max)  # keep inputs alive until the stream has consumed them
    if overflow_fallback and not keep_checkpoints and not dump_fronts:
        res.overflow_reruns = _rerun_overflowed(ens, alpha, n, ksat, res, outputs, per_step, moisture, layer_water)
    return res, workspace


class _LGARFunction(torch.autograd.Function):
    """autograd bridge: forward = lgar_forward (stores chunk checkpoints), backward = lgar_backward_ex.
    Parameters given as `[L]` vectors are SHARED by all columns: their gradient (the sum over columns) is reduced
    inside the library in a fixed order (no torch reduction kernel, bit-reproducible).  The soil-moisture outputs
    (moisture, layer_water) are outputs of their own, empty when not requested."""

    @staticmethod
    def forward(ctx, alpha, n, ksat, pdm, ens: ColumnEnsemble, mask: int, moisture: bool = False,
                layer_water: bool = False):
        outputs = [OUT_NAMES[k] for k in range(NUM_OUTPUTS) if (mask >> k) & 1]
        need_grad = any(ctx.needs_input_grad[:4])
        B = ens.num_columns
        pdm_b = None
        if pdm is not None:
            pdm_b = pdm.detach().to(ens.device, F64)
            pdm_b = (pdm_b.reshape(1).expand(B) if pdm_b.numel() == 1 else pdm_b.reshape(B)).contiguous()
        res, ws = forward_raw(ens, alpha.detach(), n.detach(), ksat.detach(), outputs=outputs,
                              keep_checkpoints=need_grad, ponded_depth_max=pdm_b, moisture=moisture,
                              layer_water=layer_water)
        ctx.ens, ctx.mask, ctx.ws = ens, mask, ws
        ctx.save_for_backward(*res._keep[:3])
        ctx.pdm_b = res._keep[4]
        ctx.pdm_shape = None if pdm is None else tuple(pdm.shape)
        ctx.want_pdm = pdm is not None and ctx.needs_input_grad[3]
        ctx.in_shapes = (alpha.shape, n.shape, ksat.shape)
        ctx.mark_non_differentiable(res.status, res.crash_step, res.start_volume)
        # an output the loss does not use gets no gradient (None): the soil-moisture outputs then pass NULL to the
        # reverse pass, which leaves it exactly as without them; per_step and sums keep their zero gradients
        ctx.set_materialize_grads(False)
        empty = lambda x: x if x is not None else torch.zeros(0, dtype=F64, device=ens.device)
        return (empty(res.per_step), res.sums, res.start_volume, res.status, res.crash_step, empty(res.moisture),
                empty(res.layer_water))

    @staticmethod
    def backward(ctx, g_per_step, g_sums, _gsv, _gst, _gcs, g_moisture, g_layer_water):
        L_ = _capi.lib()
        ens: ColumnEnsemble = ctx.ens
        alpha, n, ksat = ctx.saved_tensors
        if g_per_step is None:
            g_per_step = torch.zeros(bin(ctx.mask).count("1"), ens.num_steps, ens.num_columns, dtype=F64, device=ens.device)
        if g_sums is None:
            g_sums = torch.zeros(NUM_OUTPUTS, ens.num_columns, dtype=F64, device=ens.device)
        dev = ens.device
        Lr, B = ens.num_layers, ens.num_columns
        p = ens.problem(alpha, n, ksat, ctx.pdm_b)
        sa, sn, sk = ctx.in_shapes
        pdm_shared = ctx.pdm_shape is None or int(torch.Size(ctx.pdm_shape).numel()) == 1
        shared = len(sa) == 1 and len(sn) == 1 and len(sk) == 1 and (pdm_shared or not ctx.want_pdm)
        g = _capi.Gradients()
        gshape = (Lr,) if shared else (Lr, B)
        ga = torch.zeros(gshape, dtype=F64, device=dev)
        gn = torch.zeros_like(ga)
        gk = torch.zeros_like(ga)
        gp = None
        if ctx.want_pdm:
            gp = torch.zeros(1 if shared else B, dtype=F64, device=dev)
            g.grad_ponded_depth_max = gp.data_ptr()
        gps = g_per_step.contiguous() if (g_per_step is not None and g_per_step.numel()) else None
        gs = g_sums.contiguous() if g_sums is not None else None
        overflow = torch.empty(B, dtype=torch.int32, device=dev)
        g.grad_per_step = gps.data_ptr() if gps is not None else None
        g.grad_mask = ctx.mask
        g.grad_sums = gs.data_ptr() if gs is not None else None
        gm = g_moisture.contiguous() if (g_moisture is not None and g_moisture.numel()) else None
        gl = g_layer_water.contiguous() if (g_layer_water is not None and g_layer_water.numel()) else None
        g.grad_moisture = gm.data_ptr() if gm is not None else None
        g.grad_layer_water = gl.data_ptr() if gl is not None else None
        g.grad_alpha, g.grad_n, g.grad_ksat = ga.data_ptr(), gn.data_ptr(), gk.data_ptr()
        g.tape_overflow = overflow.data_ptr()
        partials = None
        if shared:
            partials = torch.empty(((B + 31) // 32, 3 * _capi.MAX_LAYERS + 1), dtype=F64, device=dev)
            g.reduce, g.partials = 1, partials.data_ptr()
        counters = None
        if ens.reverse_counters:
            counters = torch.zeros(8, dtype=torch.int64, device=dev)
            g.counters = counters.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            rc = L_.lgar_backward_ex(C.byref(p), C.byref(g), ctx.ws.data_ptr(), ctx.ws.numel(), C.c_void_p(stream))
        _capi.check(rc, "lgar_backward_ex")
        # the caller decides what to do with columns whose tape arena was exhausted (their per-column gradient is NaN;
        # shared-parameter sums leave them out): see ColumnEnsemble.check_tape_overflow()
        ens.last_tape_overflow = overflow
        ens.last_reverse_counters = counters

        def shape_back(gr, shp):
            return gr.sum(dim=1) if (len(shp) == 1 and gr.dim() == 2) else gr
        gp_out = None
        if gp is not None:
            gp_out = (gp.sum() if (pdm_shared and gp.numel() > 1) else gp).reshape(ctx.pdm_shape)
        return shape_back(ga, sa), shape_back(gn, sn), shape_back(gk, sk), gp_out, None, None, None, None


def lgar_columns(alpha, n, ksat, ens: ColumnEnsemble, outputs=("runoff", "percolation"), ponded_depth_max=None):
    """Differentiable batched run.  alpha/n/ksat: `[L,B]` (per column) or `[L]` (shared by all columns).
    ponded_depth_max (optional): a scalar (shared) or `[B]` tensor that replaces ens.ponded_depth_max; if it requires
    grad it is a gradient leaf like alpha/n/ksat (the reference's commented-out parameter, models/dpLGAR.py:48-49).
    Returns a dict: every requested output as `[T,B]`, plus `sums[NOUT,B]`, `start_volume[B]`,
    `status[B]`, `crash_step[B]`.
    Soil moisture (definitions in lgar_b200.h), also differentiable: "moisture" in `outputs` adds `moisture[D,T,B]`,
    theta at ens.moisture_depths; "layer_water" adds `layer_water[L,T,B]` (cm) and `layer_theta[L,T,B]` = layer_water /
    thickness, the layer-average water content."""
    outputs = tuple(outputs)
    moisture, layer_water = "moisture" in outputs, "layer_water" in outputs
    if moisture and ens.num_depths == 0:
        raise ValueError('"moisture" needs ColumnEnsemble(moisture_depths=...)')
    outputs = tuple(nm for nm in outputs if nm not in ("moisture", "layer_water"))
    mask = output_mask(outputs)
    dev = ens.device
    a = torch.as_tensor(alpha, dtype=F64).to(dev)
    nn_ = torch.as_tensor(n, dtype=F64).to(dev)
    k = torch.as_tensor(ksat, dtype=F64).to(dev)
    if not (a.dim() == 1 and nn_.dim() == 1 and k.dim() == 1):  # mixed: expand the shared ones (autograd sums them)
        a = a if a.dim() == 2 else a.unsqueeze(1).expand(ens.num_layers, ens.num_columns)
        nn_ = nn_ if nn_.dim() == 2 else nn_.unsqueeze(1).expand(ens.num_layers, ens.num_columns)
        k = k if k.dim() == 2 else k.unsqueeze(1).expand(ens.num_layers, ens.num_columns)
    pdm = None if ponded_depth_max is None else torch.as_tensor(ponded_depth_max, dtype=F64).to(dev)
    per_step, sums, sv, st, cs, moist, lw = _LGARFunction.apply(a.contiguous(), nn_.contiguous(), k.contiguous(), pdm,
                                                                ens, mask, moisture, layer_water)
    out = {name: per_step[bin(mask & ((1 << OUT_NAMES.index(name)) - 1)).count("1")] for name in outputs}
    out.update(sums=sums, start_volume=sv, status=st, crash_step=cs)
    if moisture:
        out["moisture"] = moist
    if layer_water:
        out["layer_water"] = lw
        out["layer_theta"] = lw / ens.thickness[:, None, :]
    return out
