"""ctypes binding of oracle_field/liboracle_field.so: the oracle's unstructured entries with a nodal velocity field
u_ele(2,3,E) (test infrastructure only).  u_ele is passed as an (E, 3, 2) array, which in C order is the reference's layout."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELD_DIR = os.path.join(ROOT, "oracle_field")
LIB_PATH = os.path.join(FIELD_DIR, "liboracle_field.so")

f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


def build(force=False):
    src = [os.path.join(FIELD_DIR, "pamg_oracle_field.cpp"), os.path.join(FIELD_DIR, "Makefile"),
           os.path.join(ROOT, "oracle", "pamg_oracle.cpp"), os.path.join(ROOT, "oracle", "pamg_oracle.h")]
    if force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in src):
        subprocess.run(["make", "-C", FIELD_DIR], check=True, stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(LIB_PATH)
    ci, cd = C.c_int, C.c_double
    L.orc_unstr_explicit_field.argtypes = [ci, f64p, i32p, i32p, i32p, f64p, cd, ci, ci, ci, ci, ci, cd, f64p]
    L.orc_unstr_explicit_field.restype = None
    L.orc_unstr_implicit_assemble_diff_field.argtypes = [ci, f64p, i32p, i32p, f64p, cd, cd, ci, ci, f64p, f64p]
    L.orc_unstr_implicit_assemble_diff_field.restype = None
    L.orc_unstr_stab_field.argtypes = [ci, f64p, f64p, f64p, f64p, cd, f64p, f64p]
    L.orc_unstr_stab_field.restype = None
    L.orc_unstr_implicit_field.argtypes = [ci, f64p, i32p, i32p, f64p, cd, ci, ci, ci, f64p]
    L.orc_unstr_implicit_field.restype = ci
    L.orc_unstr_implicit_stab_field.argtypes = [ci, f64p, i32p, i32p, f64p, cd, ci, ci, ci, f64p]
    L.orc_unstr_implicit_stab_field.restype = ci
    _lib = L
    return L


def _c(a, dt=np.float64):
    return np.ascontiguousarray(a, dt)


def explicit(X, neig, fneig, u, T, dt, ntime, nits, njac, exact, use_dir, t_bc=0.0):
    E = X.shape[0]
    out = _c(T).copy()
    lib().orc_unstr_explicit_field(E, _c(X), _c(neig, np.int32), _c(fneig, np.int32), np.zeros((E, 3), np.int32), _c(u),
                                   dt, ntime, nits, njac, int(exact), int(use_dir), t_bc, out)
    return out


def assemble(X, neig, fneig, u, dt, k=0.0, use_dir=True, literal_target=False):
    """dense (lhs + flux [+ diffusion], M/dt), (3E)^2 each"""
    N = 3 * X.shape[0]
    A, M = np.zeros((N, N)), np.zeros((N, N))
    lib().orc_unstr_implicit_assemble_diff_field(X.shape[0], _c(X), _c(neig, np.int32), _c(fneig, np.int32), _c(u), k, dt,
                                                 int(use_dir), int(literal_target), A, M)
    return A, M


def stab(X, u, tnew, told, dt):
    E = X.shape[0]
    dc, st = np.zeros((E, 3)), np.zeros((E, 3, 3))
    lib().orc_unstr_stab_field(E, _c(X), _c(tnew), _c(told), _c(u), dt, dc, st)
    return dc, st


def implicit(X, neig, fneig, u, T, dt, ntime, nits, use_dir=True, with_stab=False):
    out = _c(T).copy()
    fn = lib().orc_unstr_implicit_stab_field if with_stab else lib().orc_unstr_implicit_field
    rc = fn(X.shape[0], _c(X), _c(neig, np.int32), _c(fneig, np.int32), _c(u), dt, ntime, nits, int(use_dir), out)
    if rc != 0:
        raise RuntimeError("singular operator (FINDInv errorflag = -1)")
    return out
