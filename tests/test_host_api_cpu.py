"""CPU: workspace sizes of the C ABI and the argument rules of its entry points.  Neither needs a device: the rules run
before the device check, so a rejected call has touched neither the GPU nor the caller's buffers."""
import ctypes as C

import pytest

from lgar_b200 import _capi

E_INVALID, E_NO_DEVICE, E_WORKSPACE = -1, -3, -4


def _problem(B=4, L=3, T=8, S=1, max_fronts=0, chunk_steps=0, **fields):
    p = _capi.Problem()
    p.abi_version = _capi.ABI_VERSION
    p.num_columns, p.num_layers, p.num_steps, p.num_subcycles = B, L, T, S
    p.max_fronts, p.chunk_steps = max_fronts, chunk_steps
    p.num_sites, p.nint, p.num_giuh = 1, 120, 5
    for k, v in fields.items():
        setattr(p, k, v)
    return p


# (B, L, T, S, max_fronts, chunk_steps) -> bytes without / with gradients (nint 120, 5 GIUH ordinates, 1 site)
WORKSPACE_BYTES = [
    ((1, 3, 1, 1, 0, 0), 27392, 134129664),
    ((4, 3, 8, 1, 0, 0), 27392, 134129664),
    ((33, 3, 65, 1, 16, 0), 54272, 134512896),
    ((64, 3, 8760, 1, 16, 0), 54272, 9273390592),
    ((1000, 3, 600, 12, 0, 0), 860672, 40717202432),
    ((4097, 4, 160, 1, 8, 0), 2114560, 12969579264),
    ((100, 3, 100, 1, 12, 48), 87040, 306599936),
    ((125000, 3, 8760, 1, 16, 64), 105036288, 101394348032),
    # 32 fronts are forward-only: there is no reverse scratch, only the checkpoint store
    ((100, 3, 100, 1, 32, 0), 192000, 1231360),
]


@pytest.mark.parametrize("shape,without_grad,with_grad", WORKSPACE_BYTES)
def test_workspace_bytes(shape, without_grad, with_grad, monkeypatch):
    monkeypatch.delenv("LGAR_DEBUG_TAPE_CAP", raising=False)
    lib = _capi.lib()
    p = _problem(*shape)
    assert lib.lgar_workspace_bytes(C.byref(p), 0) == without_grad
    assert lib.lgar_workspace_bytes(C.byref(p), 1) == with_grad


@pytest.mark.parametrize("shape,without_grad,with_grad", [
    ((4, 3, 8, 1, 0, 0), 27392, 2271232),
    ((64, 3, 8760, 1, 16, 0), 54272, 175158784),
])
def test_workspace_bytes_with_debug_tape_cap(shape, without_grad, with_grad, monkeypatch):
    """LGAR_DEBUG_TAPE_CAP caps the entries of one sub-step and shrinks the tape arena of a chunk to that cap."""
    monkeypatch.setenv("LGAR_DEBUG_TAPE_CAP", "64")
    lib = _capi.lib()
    p = _problem(*shape)
    assert lib.lgar_workspace_bytes(C.byref(p), 0) == without_grad
    assert lib.lgar_workspace_bytes(C.byref(p), 1) == with_grad


_dummy = (C.c_double * 64)()
_ADDR = C.addressof(_dummy)  # never dereferenced: every call below has no workspace


def _forward(p, keep_checkpoints=0, fronts=False):
    for f in ("alpha", "n", "ksat", "theta_r", "theta_e", "thickness", "initial_psi", "ponded_depth_max", "forcing"):
        setattr(p, f, _ADDR)
    o = _capi.Outputs()
    if fronts:
        o.fronts = _ADDR
    return _capi.lib().lgar_forward(C.byref(p), C.byref(o), None, 0, keep_checkpoints, None)


def _backward(p, **fields):
    g = _capi.Gradients()
    g.grad_alpha = g.grad_n = g.grad_ksat = _ADDR
    for k, v in fields.items():
        setattr(g, k, v)
    return _capi.lib().lgar_backward_ex(C.byref(p), C.byref(g), None, 0, None)


def _workspace_bytes_rc(p, with_grad):
    return E_INVALID if _capi.lib().lgar_workspace_bytes(C.byref(p), with_grad) == 0 else 0


INVALID_CALLS = {
    "max_fronts_10": (lambda: _forward(_problem(max_fronts=10)), "max_fronts"),
    "max_fronts_32_with_checkpoints": (lambda: _forward(_problem(max_fronts=32), keep_checkpoints=1), "max_fronts"),
    "window_with_checkpoints": (lambda: _forward(_problem(step_end=4), keep_checkpoints=1), "step_end"),
    "window_after_row_0_without_resume": (lambda: _forward(_problem(step_begin=2, step_end=8)), "step_begin"),
    "resume_with_checkpoints": (lambda: _forward(_problem(resume=1), keep_checkpoints=1), "resume"),
    "pipeline_seq_negative": (lambda: _forward(_problem(pipeline_seq=-1)), "pipeline_seq"),
    "pipeline_seq_2_without_resume": (lambda: _forward(_problem(pipeline_seq=2)), "pipeline_seq"),
    "pipeline_seq_with_checkpoints": (lambda: _forward(_problem(pipeline_seq=1), keep_checkpoints=1), "pipeline_seq"),
    "long_chunk_workspace_bytes": (lambda: _workspace_bytes_rc(_problem(S=6, chunk_steps=100), 1), "chunk_steps"),
    "long_chunk_forward_with_checkpoints": (lambda: _forward(_problem(S=6, chunk_steps=100), keep_checkpoints=1),
                                            "chunk_steps"),
    "long_chunk_backward": (lambda: _backward(_problem(S=6, chunk_steps=100)), "chunk_steps"),
    "front_dump_with_8_fronts": (lambda: _forward(_problem(max_fronts=8), fronts=True), "max_fronts"),
    "backward_max_fronts_32": (lambda: _backward(_problem(max_fronts=32)), "max_fronts"),
    "backward_window": (lambda: _backward(_problem(step_end=4)), "step_end"),
    "backward_reduce_without_partials": (lambda: _backward(_problem(), reduce=1), "partials"),
    "backward_null_gradient": (lambda: _backward(_problem(), grad_n=None), "grad_n"),
}


@pytest.mark.parametrize("name", sorted(INVALID_CALLS))
def test_invalid_call_is_rejected_before_the_device(name):
    call, field = INVALID_CALLS[name]
    assert call() == E_INVALID
    assert field.encode() in _capi.lib().lgar_last_error_string()


def test_valid_calls_get_past_the_argument_rules():
    """The calls the rejected ones are built from are valid: they fail only at the device or the missing workspace."""
    assert _forward(_problem()) in (E_NO_DEVICE, E_WORKSPACE)
    assert _forward(_problem(), keep_checkpoints=1) in (E_NO_DEVICE, E_WORKSPACE)
    assert _forward(_problem(step_begin=2, step_end=8, resume=1, pipeline_seq=2)) in (E_NO_DEVICE, E_WORKSPACE)
    assert _forward(_problem(max_fronts=16), fronts=True) in (E_NO_DEVICE, E_WORKSPACE)
    assert _backward(_problem(S=6, chunk_steps=85)) in (E_NO_DEVICE, E_WORKSPACE)
    assert _capi.lib().lgar_workspace_bytes(C.byref(_problem(S=6, chunk_steps=85)), 1) > 0
    assert _capi.lib().lgar_workspace_bytes(C.byref(_problem(max_fronts=32)), 1) > 0
