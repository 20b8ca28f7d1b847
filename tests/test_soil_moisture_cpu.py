"""CPU: the soil-moisture part of the C ABI (struct layout, argument rules, workspace sizes), the Python-side checks of
the sensor depths, and the plain-Python restatement of the two definitions (include/lgar_b200.h) on hand-built front
lists.  No device needed: the argument rules run before the device check."""
import ctypes as C
import math
import os
import subprocess

import pytest

from conftest import ROOT
from lgar_b200 import _capi
from soil_moisture_ref import cumulative, layer_water, theta_at

E_INVALID, E_NO_DEVICE, E_WORKSPACE = -1, -3, -4

FIELDS = (("lgar_problem", "num_depths", _capi.Problem), ("lgar_problem", "moisture_depths", _capi.Problem),
          ("lgar_outputs", "moisture", _capi.Outputs), ("lgar_outputs", "layer_water", _capi.Outputs),
          ("lgar_gradients", "grad_moisture", _capi.Gradients),
          ("lgar_gradients", "grad_layer_water", _capi.Gradients))


def test_struct_layout_of_the_soil_moisture_fields(tmp_path):
    src = tmp_path / "sm.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lgar_b200.h"', 'int main(void){',
             'printf("%zu %zu %zu %d %d\\n", sizeof(lgar_problem), sizeof(lgar_outputs), sizeof(lgar_gradients), '
             'LGAR_MAX_DEPTHS, LGAR_ABI_VERSION);']
    for struct, field, _ in FIELDS:
        lines.append(f'printf("%zu %zu\\n", offsetof({struct}, {field}), sizeof((({struct}*)0)->{field}));')
    lines.append("return 0;}")
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "sm"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    rows = [[int(x) for x in ln.split()] for ln in subprocess.check_output([str(exe)]).decode().splitlines()]
    sp, so, sg, max_depths, abi = rows[0]
    assert (sp, so, sg) == (C.sizeof(_capi.Problem), C.sizeof(_capi.Outputs), C.sizeof(_capi.Gradients))
    assert max_depths == _capi.MAX_DEPTHS and abi == _capi.ABI_VERSION == 3
    for (struct, field, cls), (off, size) in zip(FIELDS, rows[1:]):
        assert getattr(cls, field).offset == off, field
        assert getattr(cls, field).size == size, field
    # num_depths took the place of the reserved word: every field before the appended ones keeps its offset
    assert _capi.Problem.num_depths.offset == 60 and _capi.Problem.iter_cap.offset == 64


_dummy = (C.c_double * 64)()
_ADDR = C.addressof(_dummy)  # never dereferenced: every call below has no workspace


def _problem(num_depths=0, depths=(), B=4, L=3, T=8, **fields):
    p = _capi.Problem()
    p.abi_version = _capi.ABI_VERSION
    p.num_columns, p.num_layers, p.num_steps, p.num_subcycles = B, L, T, 1
    p.num_sites, p.nint, p.num_giuh = 1, 120, 5
    p.num_depths = num_depths
    for i, z in enumerate(depths):
        p.moisture_depths[i] = z
    for k, v in fields.items():
        setattr(p, k, v)
    return p


def _forward(p, moisture=False, layer_water=False):
    for f in ("alpha", "n", "ksat", "theta_r", "theta_e", "thickness", "initial_psi", "ponded_depth_max", "forcing"):
        setattr(p, f, _ADDR)
    o = _capi.Outputs()
    o.moisture = _ADDR if moisture else None
    o.layer_water = _ADDR if layer_water else None
    return _capi.lib().lgar_forward(C.byref(p), C.byref(o), None, 0, 0, None)


def _backward(p, grad_moisture=False, grad_layer_water=False):
    g = _capi.Gradients()
    g.grad_alpha = g.grad_n = g.grad_ksat = _ADDR
    g.grad_moisture = _ADDR if grad_moisture else None
    g.grad_layer_water = _ADDR if grad_layer_water else None
    return _capi.lib().lgar_backward_ex(C.byref(p), C.byref(g), None, 0, None)


INVALID = {
    "num_depths_negative": (lambda: _forward(_problem(num_depths=-1)), "num_depths"),
    "num_depths_9": (lambda: _forward(_problem(num_depths=9, depths=[10.0] * 8)), "num_depths"),
    "depth_zero": (lambda: _forward(_problem(num_depths=2, depths=(10.0, 0.0)), moisture=True), "moisture_depths"),
    "depth_negative": (lambda: _forward(_problem(num_depths=1, depths=(-5.0,))), "moisture_depths"),
    "depth_nan": (lambda: _forward(_problem(num_depths=1, depths=(math.nan,)), moisture=True), "moisture_depths"),
    "depth_inf": (lambda: _forward(_problem(num_depths=1, depths=(math.inf,))), "moisture_depths"),
    "moisture_without_depths": (lambda: _forward(_problem(), moisture=True), "moisture"),
    "backward_depth_zero": (lambda: _backward(_problem(num_depths=1, depths=(0.0,)), grad_moisture=True),
                            "moisture_depths"),
    "backward_num_depths_9": (lambda: _backward(_problem(num_depths=9, depths=[10.0] * 8)), "num_depths"),
    "grad_moisture_without_depths": (lambda: _backward(_problem(), grad_moisture=True), "grad_moisture"),
}


@pytest.mark.parametrize("name", sorted(INVALID))
def test_invalid_soil_moisture_arguments_are_rejected(name):
    call, field = INVALID[name]
    assert call() == E_INVALID
    assert field.encode() in _capi.lib().lgar_last_error_string()


def test_valid_soil_moisture_calls_get_past_the_argument_rules():
    z = (5.0, 10.0, 20.0, 50.0, 100.0, 150.0, 199.9, 200.0)
    assert _forward(_problem(num_depths=8, depths=z), moisture=True, layer_water=True) in (E_NO_DEVICE, E_WORKSPACE)
    assert _forward(_problem(), layer_water=True) in (E_NO_DEVICE, E_WORKSPACE)   # layer water needs no depths
    # unused slots of moisture_depths are not read
    assert _forward(_problem(num_depths=1, depths=(5.0, 0.0, math.nan)), moisture=True) in (E_NO_DEVICE, E_WORKSPACE)
    assert _backward(_problem(num_depths=5, depths=z[:5]), grad_moisture=True, grad_layer_water=True) in \
        (E_NO_DEVICE, E_WORKSPACE)
    assert _backward(_problem(), grad_layer_water=True) in (E_NO_DEVICE, E_WORKSPACE)


@pytest.mark.parametrize("shape", [(1, 3, 1, 0), (64, 3, 8760, 16), (1000, 3, 600, 0), (4097, 4, 160, 8),
                                   (100, 3, 100, 12), (100, 3, 100, 32)])
def test_workspace_bytes_do_not_depend_on_the_depths(shape, monkeypatch):
    """The soil-moisture outputs need no workspace: neither forward nor with-gradient sizes change with the depths
    (the reverse pass keeps the outputs of a step as the last entries of its tape, not in the step records)."""
    monkeypatch.delenv("LGAR_DEBUG_TAPE_CAP", raising=False)
    B, L, T, FM = shape
    lib = _capi.lib()
    base = _problem(B=B, L=L, T=T, max_fronts=FM)
    deep = _problem(num_depths=8, depths=[5.0, 10, 20, 50, 100, 150, 175, 200], B=B, L=L, T=T, max_fronts=FM)
    for wg in (0, 1):
        assert lib.lgar_workspace_bytes(C.byref(deep), wg) == lib.lgar_workspace_bytes(C.byref(base), wg) > 0


def test_ensemble_rejects_bad_depths_before_any_launch():
    from lgar_b200.columns import check_moisture_depths
    assert check_moisture_depths(None) == ()
    assert check_moisture_depths([5, 10.5]) == (5.0, 10.5)
    for bad in ([1.0] * 9, [5.0, 0.0], [-1.0], [math.nan], [math.inf]):
        with pytest.raises(ValueError, match="moisture_depths"):
            check_moisture_depths(bad)


# ---- the restatement on hand-built front lists ------------------------------------------------------------------
THICK = (44.0, 131.0, 25.0)   # cum = 44, 175, 200


def test_layer_water_association_and_empty_and_single_front_layers():
    # layer 0: two fronts; layer 1: one front (its bottom); layer 2: one front
    depth = [10.0, 44.0, 175.0, 200.0]
    theta = [0.40, 0.30, 0.25, 0.20]
    W = layer_water(depth, theta, [2, 1, 1], THICK)
    assert W[0] == 0.0 + (10.0 - 0.0) * (0.40 - 0.30) + (44.0 - 0.0) * 0.30
    assert W[1] == 0.0 + (175.0 - (175.0 - 131.0)) * 0.25
    assert W[2] == 0.0 + (200.0 - (200.0 - 25.0)) * 0.20
    # the top of a layer is cum - thickness, not the cumulative sum of the layers above (they can differ in the last bit)
    thick = (0.1, 0.2, 0.3)
    cum = cumulative(thick)
    assert cum[2] - thick[2] != cum[1]
    assert layer_water([0.1, 0.3, 0.6], [0.3, 0.2, 0.1], [1, 1, 1], thick)[2] == 0.0 + (0.6 - (cum[2] - 0.3)) * 0.1
    # an empty list contributes 0
    assert layer_water([44.0, 200.0], [0.3, 0.2], [1, 0, 1], THICK)[1] == 0.0


def test_theta_at_depth_selection_rules():
    depth = [5.0, 20.0, 44.0, 100.0, 175.0, 200.0]
    theta = [0.45, 0.35, 0.30, 0.28, 0.25, 0.20]
    cnt = [3, 2, 1]
    at = lambda z: theta_at(z, depth, theta, cnt, THICK)
    assert at(1.0) == 0.45
    assert at(5.0) == 0.45          # a front exactly at z is selected
    assert at(5.000001) == 0.35
    assert at(44.0) == 0.30         # z on the bottom of layer 0 belongs to layer 0
    assert at(44.1) == 0.28         # the first front of layer 1's list with depth >= z
    assert at(175.0) == 0.25
    assert at(199.9) == 0.20        # a layer with one front
    assert at(200.0) == 0.20
    assert math.isnan(at(200.1))    # below the column
    # the selection is by list membership: a deep front in the list of layer 0 is never selected for a layer-1 depth
    assert theta_at(50.0, [60.0, 175.0, 200.0], [0.4, 0.3, 0.2], [1, 1, 1], THICK) == 0.3
    # no front of the layer's list reaches z: NaN
    assert math.isnan(theta_at(30.0, [10.0, 175.0, 200.0], [0.4, 0.3, 0.2], [1, 1, 1], THICK))


# ---- the oracle's soil-moisture entry point (tests/oracle_moisture.cpp) -------------------------------------------
@pytest.mark.parametrize("name", ["phil_4500_600", "bush_5500_600", "thin_crash"])
def test_oracle_outputs_match_the_reference_front_lists(name):
    """The oracle's W_l and theta(z) against the restatement on the reference's front lists (goldens), and
    W_0 + (W_1 + W_2) against the oracle's ending volume, bit for bit; the tangents of the layer waters sum to the
    tangent of the ending volume."""
    import numpy as np
    from conftest import load_golden, max_excess
    from oracle import lgar_oracle as O
    from oracle_moisture import moisture_batch
    from soil_moisture_ref import outputs_of_dump
    g = load_golden(name)
    T = 200
    forcing = g["forcing"][:T]
    cfg = O.cfg_from_golden(g)
    depths = (1.0, 10.0, 43.9, 44.0, 44.1, 100.0, 175.0, 200.0)
    r = moisture_batch([cfg], forcing, depths, tangents=True)
    ref = O.forward(cfg, forcing, fronts=False)
    n_ok = T if ref["status"] == 0 else ref["crash_step"]
    assert r["status"][0] == ref["status"] and (ref["status"] == 0 or r["crash_step"][0] == n_ok)
    thick = [float(x) for x in g["layer_thickness"]]
    W_ref, th_ref = outputs_of_dump(g["fronts"][:n_ok], g["front_layer"][:n_ok], g["nfronts"][:n_ok], thick, depths)
    W, th = r["layer_water"][0, :n_ok], r["moisture"][0, :n_ok]
    assert max_excess(W, W_ref) <= 1.0 and max_excess(th, th_ref) <= 1.0
    assert np.isnan(r["layer_water"][0, n_ok:]).all()
    total = W[:, 0] + (W[:, 1] + W[:, 2])
    assert np.array_equal(total.view(np.int64), ref["ending_volume"][:n_ok].view(np.int64))
    tan = O.forward_tangent(cfg, forcing)
    dW = r["dlayer_water"][0, :n_ok]
    dsum = dW[:, 0] + (dW[:, 1] + dW[:, 2])
    dev = tan["dout"][:n_ok, O.OUT_NAMES.index("ending_volume")]
    np.testing.assert_allclose(dsum, dev, rtol=1e-12, atol=1e-12 * np.abs(dev).max())
