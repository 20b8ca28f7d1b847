"""ctypes binding of tests/oracle_moisture.cpp: the soil-moisture outputs of the CPU oracle (test infrastructure).

The library is compiled on first use into a temporary directory (the source tree may be read-only), with the flags of
oracle/Makefile: `variant="glibc"` is the plain oracle, `variant="devpow"` the one with the CUDA path's pow."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle.lgar_oracle import OracleCfg, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "oracle_moisture.cpp")
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-pthread", "-ffp-contract=off", "-fno-fast-math", "-shared"]
_DIR = None
_libs = {}


def lib(variant: str = "glibc"):
    global _DIR
    if variant not in _libs:
        if _DIR is None:
            _DIR = tempfile.mkdtemp(prefix="lgar_oracle_moisture_")
            atexit.register(shutil.rmtree, _DIR, True)
        so = os.path.join(_DIR, f"liboracle_moisture_{variant}.so")
        extra = ["-mfma", "-DLGAR_ORACLE_DEVICE_POW"] if variant == "devpow" else []
        subprocess.check_call(["g++", *_FLAGS, *extra, "-o", so, _SRC])
        l = C.CDLL(so)
        assert l.lgar_oracle_sizeof_cfg() == C.sizeof(OracleCfg)
        l.lgar_oracle_moisture_batch.restype = C.c_int
        _libs[variant] = l
    return _libs[variant]


def moisture_batch(cfgs, forcing: np.ndarray, depths, site=None, nthreads: int = 1, tangents: bool = False,
                   variant: str = "glibc"):
    """Soil-moisture outputs (include/lgar_b200.h) of B columns after every forcing step: `layer_water[B,T,L]` and
    `moisture[B,T,D]` (theta at `depths`), NaN from a column's crash step on; with tangents=True also their forward-mode
    derivatives `dlayer_water[B,T,L,3L]`, `dmoisture[B,T,D,3L]` w.r.t. (alpha[L], n[L], ksat[L])."""
    forcing = np.ascontiguousarray(forcing, dtype=np.float64)
    T = forcing.shape[-2]
    B = len(cfgs)
    L = cfgs[0].num_layers if B else 0
    z = np.ascontiguousarray(depths, dtype=np.float64).reshape(-1)
    D = z.size
    arr = (OracleCfg * B)(*cfgs)
    w = np.full((B, T, L), np.nan)
    th = np.full((B, T, D), np.nan)
    dw = np.full((B, T, L, 3 * L), np.nan) if tangents else None
    dth = np.full((B, T, D, 3 * L), np.nan) if tangents else None
    status = np.zeros(B, dtype=np.int32)
    crash = np.zeros(B, dtype=np.int32)
    site_arr = None
    if forcing.ndim == 3:
        site_arr = np.ascontiguousarray(site if site is not None else np.zeros(B), dtype=np.int32)
    lib(variant).lgar_oracle_moisture_batch(
        arr, C.c_int(B), _p(forcing, C.c_double), _p(site_arr, C.c_int32), C.c_int(T), _p(z, C.c_double), C.c_int(D),
        _p(w, C.c_double), _p(dw, C.c_double), _p(th, C.c_double), _p(dth, C.c_double), _p(status, C.c_int32),
        _p(crash, C.c_int32), C.c_int(nthreads))
    r = dict(layer_water=w, moisture=th, status=status, crash_step=crash)
    if tangents:
        r.update(dlayer_water=dw, dmoisture=dth)
    return r
