"""ctypes front end of the CTA emulator build of the kernel source (tests/emu) — TEST INFRASTRUCTURE.

The emulator executes gomilp_b200/csrc/simplex_cta.cuh (the file nvcc compiles for sm_100a) on the CPU,
one emulated thread block at a time, so the kernel's control flow is tested where there is no GPU.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "emu", "emu_capi.cpp")
_OUT = os.path.join(_HERE, "emu", "_build", "libemu.so")
_DEPS = [_SRC, os.path.join(_HERE, "emu", "cta_emu.hpp"),
         os.path.join(_HERE, "..", "gomilp_b200", "csrc", "simplex_cta.cuh"),
         os.path.join(_HERE, "..", "gomilp_b200", "csrc", "cta_rt.cuh"),
         os.path.join(_HERE, "..", "gomilp_b200", "csrc", "bnb_host.cpp"),
         os.path.join(_HERE, "..", "include", "gomilp_b200.h"),
         os.path.join(_HERE, "..", "include", "gomilp_status.h")]
_lib = None


def build():
    os.makedirs(os.path.dirname(_OUT), exist_ok=True)
    if os.path.exists(_OUT) and all(os.path.getmtime(_OUT) >= os.path.getmtime(d) for d in _DEPS):
        return _OUT
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                    "-I" + os.path.join(_HERE, "emu"), "-o", _OUT, _SRC], check=True)
    return _OUT


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.emu_simplex_batch.restype = C.c_int
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def simplex_batch(c, A, b, tol=0.0, bvar=None, bsign=None, brhs=None, initial_basic=None, T=64,
                  max_pivots=0, refactor_period=0, shared_root=False, x_len=None, shuffle_order=False, reg=False, ring_stages=0, ring_stage_bytes=4096, quad=False):
    """Batch of LPs through the emulated kernel.

    Plain batch: A [count,m,n], c [count,n], b [count,m]. Wave mode (shared_root=True): one root
    A [m0,n0] plus bvar/bsign/brhs of shape [count,L].
    """
    A = np.ascontiguousarray(A, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    if shared_root:
        m0, n0 = A.shape
        count = bvar.shape[0]
        L = bvar.shape[1]
        cs = As = bs = 0
        bvar = np.ascontiguousarray(bvar, dtype=np.int32)
        bsign = np.ascontiguousarray(bsign, dtype=np.float64)
        brhs = np.ascontiguousarray(brhs, dtype=np.float64)
    else:
        count, m0, n0 = A.shape
        L = 0
        cs, As, bs = n0, m0 * n0, m0
    m, n = m0 + L, n0 + L
    if x_len is None:
        x_len = n0 if shared_root else n
    status = np.zeros(count, dtype=np.int32)
    optF = np.zeros(count)
    x = np.zeros((count, x_len))
    basis = np.zeros((count, m), dtype=np.int64)
    stats = np.zeros((count, 8), dtype=np.int32)
    ib = None if initial_basic is None else np.ascontiguousarray(initial_basic, dtype=np.int64)
    lib().emu_set_quad(C.c_int(int(quad)))
    rc = lib().emu_simplex_batch(C.c_int(count), _p(c), _p(A), _p(b), C.c_longlong(cs), C.c_longlong(As),
                                 C.c_longlong(bs), C.c_int(n0), C.c_int(m0), C.c_int(n0), C.c_int(L), _p(bvar),
                                 _p(bsign), _p(brhs), _p(ib), C.c_double(tol), C.c_int(max_pivots),
                                 C.c_int(refactor_period), _p(status), _p(optF), _p(x), C.c_longlong(x_len),
                                 C.c_int(x_len), _p(basis), _p(stats), C.c_int(256 if reg else T), C.c_int(int(shuffle_order)),
                                 C.c_int(int(reg)), C.c_int(ring_stages), C.c_int(ring_stage_bytes if ring_stages else 0))
    if rc != 0:
        raise RuntimeError("CTA emulator: barrier divergence" if rc == -1 else "CTA emulator: bad tier request")
    return {"status": status, "optF": optF, "x": x, "basis": basis, "stats": stats}


def coop_batch(c, A, b, tol=0.0, bvar=None, bsign=None, brhs=None, T=64, G=3, groups=1, max_pivots=0,
               refactor_period=0, shared_root=False, shuffle_order=False, trace_cap=0, trace_lp=0, smem_panel=True,
               initial_basic=None):
    """Batch of LPs through the emulated COOPERATIVE tier: `groups` groups of G CTAs (T threads each) share the work."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    if shared_root:
        m0, n0 = A.shape
        count, L = bvar.shape
        cs = As = bs = 0
        bvar = np.ascontiguousarray(bvar, dtype=np.int32)
        bsign = np.ascontiguousarray(bsign, dtype=np.float64)
        brhs = np.ascontiguousarray(brhs, dtype=np.float64)
    else:
        count, m0, n0 = A.shape
        L = 0
        cs, As, bs = n0, m0 * n0, m0
    m = m0 + L
    x_len = n0 if shared_root else n0 + L
    status = np.zeros(count, dtype=np.int32)
    optF = np.zeros(count)
    x = np.zeros((count, x_len))
    basis = np.zeros((count, m), dtype=np.int64)
    stats = np.zeros((count, 8), dtype=np.int32)
    trace = np.full((max(trace_cap, 1), 4), -1, dtype=np.int32)
    ib = None if initial_basic is None else np.ascontiguousarray(initial_basic, dtype=np.int64).reshape(count, m)
    lib().emu_set_coop_pan(C.c_int(int(smem_panel)))
    rc = lib().emu_coop_batch(C.c_int(count), _p(c), _p(A), _p(b), C.c_longlong(cs), C.c_longlong(As), C.c_longlong(bs),
                              C.c_int(n0), C.c_int(m0), C.c_int(n0), C.c_int(L), _p(bvar), _p(bsign), _p(brhs), _p(ib),
                              C.c_double(tol), C.c_int(max_pivots), C.c_int(refactor_period), _p(status), _p(optF),
                              _p(x), C.c_longlong(x_len), C.c_int(x_len), _p(basis), _p(stats), C.c_int(T), C.c_int(G),
                              C.c_int(groups), C.c_int(int(shuffle_order)), _p(trace) if trace_cap else None,
                              C.c_int(trace_cap), C.c_int(trace_lp))
    if rc != 0:
        raise RuntimeError("CTA emulator: barrier divergence" if rc == -1 else "CTA emulator: bad request")
    return {"status": status, "optF": optF, "x": x, "basis": basis, "stats": stats, "trace": trace}


class _MilpRes(C.Structure):
    _fields_ = [("status", C.c_int32), ("lp_status", C.c_int32), ("z", C.c_double), ("x_len", C.c_int64),
                ("nodes", C.c_int64), ("waves", C.c_int64), ("pivots", C.c_int64), ("device_ms", C.c_double)]


_DCB = C.CFUNCTYPE(None, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_int32,
                   C.c_double)
_WCB = C.CFUNCTYPE(None, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_double)


def set_robust(on: bool):
    lib().emu_set_robust(C.c_int(int(on)))


def milp_solve(c, A=None, b=None, G=None, h=None, integrality=None, heuristic=0, mode=0, node_limit=0,
               time_limit_s=0.0, T=64, reg=False, quad=False):
    """The product's gm_milp_solve (bnb_host.cpp) with every wave solved by the emulated kernel."""
    L = lib()
    L.emu_set_threads(C.c_int(256 if reg else T), C.c_int(int(reg)))
    L.emu_set_quad(C.c_int(int(quad)))
    c = np.ascontiguousarray(c, dtype=np.float64)
    nvar = c.shape[0]
    meq = 0 if A is None else np.asarray(A).shape[0]
    nineq = 0 if G is None else np.asarray(G).shape[0]
    Aa = np.ascontiguousarray(A, dtype=np.float64).reshape(meq, nvar) if meq else None
    ba = np.ascontiguousarray(b, dtype=np.float64) if meq else None
    Ga = np.ascontiguousarray(G, dtype=np.float64).reshape(nineq, nvar) if nineq else None
    ha = np.ascontiguousarray(h, dtype=np.float64) if nineq else None
    integ = np.ascontiguousarray(integrality, dtype=np.uint8)
    x = np.zeros(nvar + nineq + 1)
    res = _MilpRes()
    log = []

    def on_dec(_u, id_, parent, depth, lp_status, z, decision, bvar, bfloor):
        log.append((id_, parent, depth, lp_status, z, decision, bvar, bfloor))

    cb = _DCB(on_dec)
    L.gm_milp_solve.restype = C.c_int
    rc = L.gm_milp_solve(C.c_int64(nvar), _p(c), C.c_int64(meq), _p(Aa), _p(ba), C.c_int64(nineq), _p(Ga), _p(ha),
                         _p(integ), C.c_int32(heuristic), C.c_int32(mode), C.c_int64(node_limit),
                         C.c_double(time_limit_s), _p(x), C.byref(res), cb, C.cast(None, _WCB), None)
    xl = int(res.x_len)
    return {"rc": rc, "status": res.status, "lp_status": res.lp_status, "z": res.z,
            "x": x[:xl].copy() if xl else None, "nodes": res.nodes, "waves": res.waves, "pivots": res.pivots,
            "log": log}
