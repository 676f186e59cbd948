"""Python host mirror of the reference's operator interface, bound to libpamg_cuda.so through ctypes.

The reference has no plugin API; its hot path is the set of procedures contained in
Semi_implicit_iterative (transport_tri_semi.F90:407-889) plus update_overlaps / restrictor /
prolongator (splitting.F90) and the element loop of unstr_explicit (transport_tri_unstr.F90:600-791).
This module exposes those procedures under their reference names and argument meaning, all running on
the GPU.  There is no CPU fallback: constructing a solver without a CUDA device raises PamgError.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PAMG_LIB") or os.path.join(_HERE, "lib", "libpamg_cuda.so")   # PAMG_LIB: A/B builds

OK, ERR_ARG, ERR_CUDA, ERR_STATE, ERR_IO, ERR_SINGULAR, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
TNEW, TOLD, RHS, RES, TNONLIN = 0, 1, 2, 3, 5
JACOBI, RICHARDSON, GAUSS_SEIDEL = 1, 2, 3

_f64 = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_i32 = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


class PamgError(RuntimeError):
    def __init__(self, code, msg=""):
        super().__init__(f"pamg error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    """pamg_params (include/pamg.h): everything the reference hard-codes (main.F90:46-47,
    transport_tri_semi.F90:117-140) plus the LITERAL/INTENDED switches of SURVEY appendix B."""
    _fields_ = [
        ("n_split", C.c_int32), ("multi_levels", C.c_int32), ("n_smooth", C.c_int32), ("n_multigrid", C.c_int32),
        ("n_coarse_smooth", C.c_int32), ("solver", C.c_int32), ("face_terms", C.c_int32),
        ("literal_source", C.c_int32), ("transfer", C.c_int32), ("residual_sign", C.c_int32),
        ("halo_rule", C.c_int32), ("coarse_bc_zero", C.c_int32), ("keep_tnew_gs", C.c_int32), ("reserved", C.c_int32),
        ("theta", C.c_double), ("dt", C.c_double), ("k", C.c_double), ("omega", C.c_double),
        ("u_x", C.c_double), ("u_y", C.c_double), ("source_coef", C.c_double),
    ]


_lib = None


def lib():
    """Loads the in-tree CUDA library; fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PamgError(ERR_STATE, f"{LIB_PATH} is missing: run `python __graft_entry__.py build` "
                                   "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, ci, cd = C.c_void_p, C.c_int, C.c_double
    pvp = C.POINTER(C.c_void_p)
    pint = C.POINTER(C.c_int)
    pdbl = C.POINTER(C.c_double)
    sig = {
        "pamg_version": (C.c_char_p, []),
        "pamg_device_count": (ci, [pint]),
        "pamg_default_params": (None, [C.POINTER(Params), ci]),
        "pamg_mesh_read_msh": (ci, [C.c_char_p, pvp]),
        "pamg_mesh_synthetic": (ci, [ci, ci, pvp]),
        "pamg_mesh_from_arrays": (ci, [ci, _f64, vp, pvp]),
        "pamg_mesh_structured_tri": (ci, [ci, ci, cd, cd, pvp]),
        "pamg_mesh_size": (ci, [vp, pint]),
        "pamg_mesh_get": (ci, [vp, vp, vp, vp, vp, vp]),
        "pamg_mesh_free": (None, [vp]),
        "pamg_create": (ci, [C.POINTER(Params), ci, pvp]),
        "pamg_create_multi": (ci, [C.POINTER(Params), ci, vp, pvp]),
        "pamg_set_boundary_data": (ci, [vp, ci, _i32, vp]),
        "pamg_destroy": (None, [vp]),
        "pamg_last_error": (C.c_char_p, [vp]),
        "pamg_set_parents": (ci, [vp, ci, _f64, _i32, _i32, _i32]),
        "pamg_set_parents_partition": (ci, [vp, ci, _f64, _i32, _i32, _i32, ci, _i32, ci]),
        "pamg_ndof": (ci, [vp, ci, C.POINTER(C.c_int64)]),
        "pamg_upload_field": (ci, [vp, ci, ci, vp]),
        "pamg_download_field": (ci, [vp, ci, ci, vp]),
        "pamg_fill_field": (ci, [vp, ci, ci, cd]),
        "pamg_copy_field": (ci, [vp, ci, ci, ci]),
        "pamg_download_overlap": (ci, [vp, ci, ci, _f64]),
        "pamg_device_ptr": (ci, [vp, ci, ci, pvp]),
        "pamg_update_overlaps": (ci, [vp, ci]),
        "pamg_build_rhs": (ci, [vp]),
        "pamg_smooth": (ci, [vp, ci, ci, ci]),
        "pamg_residual": (ci, [vp, ci, pdbl, pdbl]),
        "pamg_convergence": (ci, [vp, ci, pdbl]),
        "pamg_restrict": (ci, [vp, ci]),
        "pamg_prolong": (ci, [vp, ci]),
        "pamg_vcycle_solve": (ci, [vp, ci, ci, ci, ci, ci, cd, pint, _f64]),
        "pamg_literal_timestep": (ci, [vp, ci, ci, ci]),
        "pamg_timestep_host": (ci, [vp, vp, vp, ci, cd, pint, pdbl]),
        "pamg_smooth_host": (ci, [vp, ci, ci, vp, vp]),
        "pamg_smoother_host": (ci, [vp, ci, ci, vp, vp]),
        "pamg_halo_sources": (ci, [ci, _f64, _i32, _i32, _i32, ci, ci, _i32, ci, ci,
                                   np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")]),
        "pamg_numbering": (ci, [ci, ci, C.c_int64, C.c_int64, _i32]),
        "pamg_parent_table": (ci, [C.POINTER(Params), ci, _f64, _i32, vp, ci, ci, cd, ci, _f64]),
        "pamg_halo_plan": (ci, [ci, _f64, _i32, _i32, _i32, ci, ci, _i32, ci, _i32, _i32, _i32, _i32, _i32, _i32]),
        "pamg_comm_unique_id": (ci, [C.c_char_p]),
        "pamg_comm_init": (ci, [vp, C.c_char_p, ci, ci]),
        "pamg_halo_peer_count": (ci, [vp, pint]),
        "pamg_halo_peer_info": (ci, [vp, ci, pint, pint]),
        "pamg_set_unstructured": (ci, [vp, ci, _f64, _i32, _i32]),
        "pamg_unstr_set_velocity": (ci, [vp, vp]),
        "pamg_unstr_upload": (ci, [vp, _f64]),
        "pamg_unstr_download": (ci, [vp, _f64]),
        "pamg_explicit_step": (ci, [vp, cd, cd, cd, cd, ci, ci, ci, ci, ci]),
        "pamg_implicit_assemble": (ci, [vp, cd, cd, cd, ci]),
        "pamg_implicit_assemble_diffusion": (ci, [vp, cd, cd, cd, cd, ci]),
        "pamg_implicit_spmv_time": (ci, [vp, ci, C.POINTER(C.c_float)]),
        "pamg_implicit_host_syncs": (ci, [vp, C.POINTER(C.c_int64)]),
        "pamg_implicit_get_bsr": (ci, [vp, vp, vp]),
        "pamg_implicit_apply": (ci, [vp, _f64, _f64]),
        "pamg_implicit_step": (ci, [vp, ci, ci, cd, ci, pint, pdbl]),
        "pamg_unstr_stab": (ci, [vp, _f64, cd, cd, cd, vp, vp]),
        "pamg_implicit_set_stab": (ci, [vp, ci]),
        "pamg_trans_rec": (ci, [vp, cd, ci, ci, cd, cd, cd, cd, cd, ci, ci, ci, ci, vp, vp, pint]),
        "pamg_apply_local_minv": (ci, [vp, ci, ci, _f64, vp, vp, vp, vp]),
        "pamg_output_fields": (ci, [vp, vp, vp, vp]),
        "pamg_write_vtu": (ci, [vp, C.c_char_p, C.c_char_p, ci]),
        "pamg_sync": (ci, [vp]),
        "pamg_event_record": (ci, [vp, ci]),
        "pamg_event_elapsed_ms": (ci, [vp, ci, ci, C.POINTER(C.c_float)]),
        "pamg_launch_count": (ci, [vp, C.POINTER(C.c_int64)]),
        "pamg_flush_l2": (ci, [vp]),
        "pamg_profile": (ci, [vp, ci]),
        "pamg_profile_read": (ci, [vp, pdbl, pint]),
        "pamg_host_alloc": (ci, [pvp, C.c_int64]),
        "pamg_host_free": (ci, [vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    L._signatures = sig
    _lib = L
    return L


def device_count():
    n = C.c_int(0)
    rc = lib().pamg_device_count(C.byref(n))
    return n.value if rc == OK else 0


def default_params(literal_head=False, **kw):
    p = Params()
    lib().pamg_default_params(C.byref(p), 1 if literal_head else 0)
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    if "k" in kw and "source_coef" not in kw:
        p.source_coef = (-2.0 if literal_head else 2.0) * p.k
    return p


def _ptr(a):
    if a is None or isinstance(a, (C.c_void_p, int)):
        return a
    return a.ctypes.data_as(C.c_void_p)


# ------------------------------------------------------------------------------ mesh (host)
class Mesh:
    """Parent triangles with the reference's Mesh%X / Neig / fNeig / Dir / region_id
    (Structures.F90:143-170) built by the O(N) host pipeline."""

    def __init__(self, handle):
        self._h = handle
        L = lib()
        n = C.c_int(0)
        L.pamg_mesh_size(handle, C.byref(n))
        self.U = n.value
        self.X = np.zeros((self.U, 3, 2))
        self.neig = np.zeros((self.U, 3), np.int32)
        self.fneig = np.zeros((self.U, 3), np.int32)
        self.dir = np.zeros((self.U, 3), np.int32)
        self.region = np.zeros(self.U, np.int32)
        L.pamg_mesh_get(handle, _ptr(self.X), _ptr(self.neig), _ptr(self.fneig), _ptr(self.dir), _ptr(self.region))
        L.pamg_mesh_free(handle)
        self._h = None

    @classmethod
    def read_msh(cls, path):
        """ReadMSH (Msh2Tri.F90:132) + getNeigDataMesh (:454)."""
        h = C.c_void_p()
        rc = lib().pamg_mesh_read_msh(os.fsencode(path), C.byref(h))
        if rc != OK:
            raise PamgError(rc, f"cannot read gmsh 2.2 ASCII mesh {path}")
        return cls(h)

    @classmethod
    def synthetic(cls, kp, G=1):
        h = C.c_void_p()
        rc = lib().pamg_mesh_synthetic(kp, G, C.byref(h))
        if rc != OK:
            raise PamgError(rc, "pamg_mesh_synthetic")
        return cls(h)

    @classmethod
    def structured_tri(cls, no_ele_row, no_ele_col, dx, dy):
        """Structured triangles of str_explicit (structured_meshgen.F90:190-298)."""
        h = C.c_void_p()
        rc = lib().pamg_mesh_structured_tri(no_ele_row, no_ele_col, dx, dy, C.byref(h))
        if rc != OK:
            raise PamgError(rc, "pamg_mesh_structured_tri")
        return cls(h)

    @classmethod
    def from_arrays(cls, X, region=None):
        X = np.ascontiguousarray(X, np.float64)
        reg = None if region is None else np.ascontiguousarray(region, np.int32)
        h = C.c_void_p()
        rc = lib().pamg_mesh_from_arrays(X.shape[0], X, _ptr(reg), C.byref(h))
        if rc != OK:
            raise PamgError(rc, "pamg_mesh_from_arrays")
        return cls(h)


def halo_plan(mesh, halo_rule=1, nparts=1, part_first=None, my_part=0):
    """Host-only description of where every halo strip lives (pamg_plan.cpp)."""
    U = mesh.U
    pf = np.ascontiguousarray(part_first if part_first is not None else [0, U], np.int32)
    ul = int(pf[my_part + 1] - pf[my_part])
    out = {k: np.zeros(ul * 3, np.int32) for k in ("strip_of", "dst_strip", "rev", "hmap")}
    peers = np.zeros(max(nparts, 1) * 4, np.int32)
    counts = np.zeros(5, np.int32)
    rc = lib().pamg_halo_plan(U, mesh.X, mesh.neig, mesh.fneig, mesh.dir, halo_rule, nparts, pf, my_part,
                              out["strip_of"], out["dst_strip"], out["rev"], out["hmap"], peers, counts)
    if rc != OK:
        raise PamgError(rc, "pamg_halo_plan")
    out["peers"] = peers.reshape(-1, 4)[: counts[0]].copy()
    out["nstrips"], out["nsend"], out["U_local"], out["first"] = (int(c) for c in counts[1:5])
    return out


def halo_sources(mesh, s, halo_rule=1, nparts=1, part_first=None, my_part=0):
    """Host-only: offsets of the strip-free exterior values, int64 [U_local, 3, 2**s, 2] (pamg_halo_sources)."""
    U = mesh.U
    pf = np.ascontiguousarray(part_first if part_first is not None else [0, U], np.int32)
    ul = int(pf[my_part + 1] - pf[my_part])
    out = np.zeros((ul, 3, 2 ** s, 2), np.int64)
    rc = lib().pamg_halo_sources(U, mesh.X, mesh.neig, mesh.fneig, mesh.dir, halo_rule, nparts, pf, my_part, s, out)
    if rc != OK:
        raise PamgError(rc, "pamg_halo_sources")
    return out


def numbering(what, s, first=0, count=None):
    """Host-only: the closed-form child numbering of the kernels (pamg_numbering), int32 array [count][4]."""
    if count is None:
        count = 4 ** s - first
    out = np.zeros((count, 4), np.int32)
    rc = lib().pamg_numbering(what, s, first, count, out)
    if rc != OK:
        raise PamgError(rc, "pamg_numbering")
    return out


def parent_table(params, mesh, parent, s, theta_weight=None, with_mass=True, bc_kind=None):
    """Host-only: the 88 folded coefficients of parent `parent` (0-based) on the level with split s (pamg_parent_table)."""
    out = np.zeros(88)
    bk = None if bc_kind is None else np.ascontiguousarray(bc_kind, np.int32)
    rc = lib().pamg_parent_table(C.byref(params), mesh.U, mesh.X, mesh.neig, _ptr(bk), parent, s,
                                 params.theta if theta_weight is None else theta_weight, 1 if with_mass else 0, out)
    if rc != OK:
        raise PamgError(rc, "pamg_parent_table")
    return out


# ------------------------------------------------------------------------------ solver handle
class SemiImplicitIterative:
    """GPU implementation of Semi_implicit_iterative's contained procedures
    (transport_tri_semi.F90:14-891).  Method names follow the reference."""

    def __init__(self, params, mesh, device=0, nparts=1, part_first=None, my_part=0, devices=None, bc_kind=None,
                 bc_value=None):
        """devices: list of CUDA devices driven by THIS process (pamg_create_multi; the mesh is partitioned inside the
        library); nparts / part_first / my_part: one process per GPU (torchrun), this handle owns block my_part.
        bc_kind / bc_value: (U,3) Dirichlet data of the domain-boundary faces (pamg_set_boundary_data)."""
        self.L = lib()
        self.params = params
        self.mesh = mesh
        h = C.c_void_p()
        if devices is not None:
            dev = np.ascontiguousarray(devices, np.int32)
            rc = self.L.pamg_create_multi(C.byref(params), len(dev), _ptr(dev), C.byref(h))
        else:
            rc = self.L.pamg_create(C.byref(params), device, C.byref(h))
        if rc != OK:
            raise PamgError(rc, "pamg_create failed (no CUDA device? there is no CPU fallback)")
        self.h = h
        if bc_kind is not None:
            kind = np.ascontiguousarray(bc_kind, np.int32).reshape(-1)
            val = None if bc_value is None else np.ascontiguousarray(bc_value, np.float64).reshape(-1)
            self._ck(self.L.pamg_set_boundary_data(h, mesh.U, kind, _ptr(val)))
        if nparts == 1:
            self._ck(self.L.pamg_set_parents(h, mesh.U, mesh.X, mesh.neig, mesh.fneig, mesh.dir))
            self.U = mesh.U
        else:
            pf = np.ascontiguousarray(part_first, np.int32)
            self._ck(self.L.pamg_set_parents_partition(h, mesh.U, mesh.X, mesh.neig, mesh.fneig, mesh.dir,
                                                       nparts, pf, my_part))
            self.U = int(pf[my_part + 1] - pf[my_part])

    def _ck(self, rc):
        if rc != OK:
            raise PamgError(rc, (self.L.pamg_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.pamg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- fields -------------------------------------------------------------------------------
    def split(self, level):
        return self.params.n_split - level + 1

    def shape(self, level=1):
        return (self.U, 4 ** self.split(level), 3)

    def ndof(self, level=1):
        n = C.c_int64()
        self._ck(self.L.pamg_ndof(self.h, level, C.byref(n)))
        return n.value

    def upload(self, field, level, array):
        a = np.ascontiguousarray(array, np.float64)
        assert a.size == self.ndof(level)
        self._ck(self.L.pamg_upload_field(self.h, field, level, _ptr(a)))

    def download(self, field, level=1):
        out = np.empty(self.shape(level))
        self._ck(self.L.pamg_download_field(self.h, field, level, _ptr(out)))
        return out

    def fill(self, field, level, value):
        self._ck(self.L.pamg_fill_field(self.h, field, level, float(value)))

    def copy(self, level, dst, src):
        self._ck(self.L.pamg_copy_field(self.h, level, dst, src))

    def overlap(self, level=1, old=False):
        S = 2 ** self.split(level)
        out = np.zeros((self.U, 3, S, 3))
        self._ck(self.L.pamg_download_overlap(self.h, level, 1 if old else 0, out))
        return out

    # -- the contained procedures ---------------------------------------------------------------
    def update_overlaps(self, level=1):
        """update_overlaps (splitting.F90:1210)."""
        self._ck(self.L.pamg_update_overlaps(self.h, level))

    def get_RHS(self):
        """get_RHS (transport_tri_semi.F90:452) for every level-1 child."""
        self._ck(self.L.pamg_build_rhs(self.h))

    def smoother(self, level=1, solver=None, n_smooth=None):
        """smoother (:543): n_smooth sweeps of solver 1 Jacobi / 2 Richardson / 3 Gauss-Seidel."""
        self._ck(self.L.pamg_smooth(self.h, level, solver or self.params.solver,
                                    self.params.n_smooth if n_smooth is None else n_smooth))

    def get_residual(self, level=1):
        """get_residual (:725); returns (||r||_2, ||r||_inf)."""
        l2, li = C.c_double(), C.c_double()
        self._ck(self.L.pamg_residual(self.h, level, C.byref(l2), C.byref(li)))
        return l2.value, li.value

    def get_convergence(self, level=1):
        """get_convergence (:876): signed max of the residual, floor 0."""
        c = C.c_double()
        self._ck(self.L.pamg_convergence(self.h, level, C.byref(c)))
        return c.value

    def restrictor(self, fine_level):
        """restrictor (splitting.F90:10)."""
        self._ck(self.L.pamg_restrict(self.h, fine_level))

    def prolongator(self, fine_level):
        """prolongator (splitting.F90:38)."""
        self._ck(self.L.pamg_prolong(self.h, fine_level))

    def vcycle_solve(self, solver=None, nu1=None, nu2=None, ncoarse=None, max_cycles=50, tol=1e-8):
        p = self.params
        hist = np.zeros(max_cycles + 2)
        cyc = C.c_int(0)
        self._ck(self.L.pamg_vcycle_solve(self.h, solver or p.solver, p.n_smooth if nu1 is None else nu1,
                                          p.n_smooth if nu2 is None else nu2,
                                          p.n_coarse_smooth if ncoarse is None else ncoarse, max_cycles, tol,
                                          C.byref(cyc), hist))
        return cyc.value, hist[: min(cyc.value, max_cycles) + 1]

    def literal_timestep(self, solver=None, n_multigrid=None, n_smooth=None):
        """One itime of the loop at transport_tri_semi.F90:316-379 exactly as checked in."""
        p = self.params
        self._ck(self.L.pamg_literal_timestep(self.h, solver or p.solver, n_multigrid or p.n_multigrid,
                                              n_smooth or p.n_smooth))

    def timestep_host(self, tnew_in, tnew_out, max_cycles=50, tol=1e-8):
        """Reference-facing time step with HOST buffers (upload, told=tnew, V-cycles, download)."""
        cyc, rel = C.c_int(0), C.c_double(0)
        self._ck(self.L.pamg_timestep_host(self.h, _ptr(tnew_in), _ptr(tnew_out), max_cycles, tol,
                                           C.byref(cyc), C.byref(rel)))
        return cyc.value, rel.value

    # -- distributed -----------------------------------------------------------------------------
    def comm_init(self, unique_id, nranks, rank):
        self._ck(self.L.pamg_comm_init(self.h, unique_id, nranks, rank))

    # -- timing ------------------------------------------------------------------------------------
    def sync(self):
        self._ck(self.L.pamg_sync(self.h))

    def event_record(self, slot):
        self._ck(self.L.pamg_event_record(self.h, slot))

    def elapsed_ms(self, a, b):
        ms = C.c_float()
        self._ck(self.L.pamg_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def launch_count(self):
        n = C.c_int64()
        self._ck(self.L.pamg_launch_count(self.h, C.byref(n)))
        return n.value

    def flush_l2(self):
        self._ck(self.L.pamg_flush_l2(self.h))

    def profile(self, on=True):
        self._ck(self.L.pamg_profile(self.h, 1 if on else 0))

    def profile_read(self):
        ms, n = C.c_double(), C.c_int()
        self._ck(self.L.pamg_profile_read(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def upload_ptr(self, field, level, host_ptr):
        self._ck(self.L.pamg_upload_field(self.h, field, level, host_ptr))

    def download_ptr(self, field, level, host_ptr):
        self._ck(self.L.pamg_download_field(self.h, field, level, host_ptr))

    def smoother_host(self, solver, nsweeps, in_ptr, out_ptr):
        """Blocking smoother call on HOST fields (the reference-facing form): out is valid on return."""
        self._ck(self.L.pamg_smoother_host(self.h, solver, nsweeps, in_ptr, out_ptr))

    def smooth_host(self, solver, nsweeps, in_ptr, out_ptr):
        """Smoother on a HOST field (pointers, e.g. PinnedBuffer.ptr); asynchronous: call sync() before reading out."""
        self._ck(self.L.pamg_smooth_host(self.h, solver, nsweeps, in_ptr, out_ptr))

    # -- output (get_vtu / get_error) --------------------------------------------------------------
    def output_fields(self):
        """(x_all_str (U,C,3,2), analytical, error) of level 1 (transport_tri_semi.F90:274,278,531-540)."""
        sh = self.shape(1)
        x = np.zeros(sh + (2,)); an = np.zeros(sh); er = np.zeros(sh)
        self._ck(self.L.pamg_output_fields(self.h, _ptr(x), _ptr(an), _ptr(er)))
        return x, an, er

    def get_vtu(self, path, solve_for="Concentration", binary=False):
        self._ck(self.L.pamg_write_vtu(self.h, str(path).encode(), solve_for.encode(), int(binary)))

    # -- unstructured explicit (unstr_explicit, transport_tri_unstr.F90:413) ------------------------
    def set_unstructured(self, mesh):
        self._ck(self.L.pamg_set_unstructured(self.h, mesh.U, mesh.X, mesh.neig, mesh.fneig))
        self._E = mesh.U

    def set_velocity(self, u_ele):
        """Nodal velocity field u_ele of the unstructured front-ends: shape (E, 3, 2) = (element, node, component), which in C
        order is the reference's u_ele(2,3,E); None returns to the uniform velocity.  While a field is set, the u_x, u_y
        arguments of unstr_explicit, implicit_assemble, unstr_stab and unstr_implicit are not used.  Call implicit_assemble
        again before the implicit entries: the operator of the previous velocity is stale."""
        if u_ele is None:
            self._ck(self.L.pamg_unstr_set_velocity(self.h, None))
            return
        u = np.ascontiguousarray(u_ele, np.float64)
        if hasattr(self, "_E") and u.shape != (self._E, 3, 2):      # (without a mesh the library answers ERR_STATE)
            raise ValueError(f"u_ele must have shape (E, 3, 2) = ({self._E}, 3, 2), got {u.shape}")
        self._ck(self.L.pamg_unstr_set_velocity(self.h, _ptr(u)))

    def unstr_explicit(self, tnew, dt, u_x, u_y, ntime=2, nits=2, njac_its=10, t_bc=0.0, exact_minv=False,
                       use_dir=False):
        t = np.ascontiguousarray(tnew, np.float64)
        self._ck(self.L.pamg_unstr_upload(self.h, t))
        self._ck(self.L.pamg_explicit_step(self.h, dt, u_x, u_y, t_bc, ntime, nits, njac_its, int(exact_minv),
                                           int(use_dir)))
        out = np.empty_like(t)
        self._ck(self.L.pamg_unstr_download(self.h, out))
        return out

    # -- unstructured implicit (unstr_implicit, transport_tri_unstr.F90:18) --------------------------
    def implicit_assemble(self, dt, u_x, u_y, use_dir=False, k=0.0):
        """Assemble (mass/dt - stiffness + upwind flux [+ k (volume diffusion + face penalty)]) into block-CSR on the
        device (:270-364; the diffusion operator is that of get_A_x, transport_tri_semi.F90:412-448)."""
        self._ck(self.L.pamg_implicit_assemble_diffusion(self.h, dt, u_x, u_y, float(k), int(use_dir)))

    def implicit_spmv_ms(self, reps=20):
        ms = C.c_float()
        self._ck(self.L.pamg_implicit_spmv_time(self.h, reps, C.byref(ms)))
        return ms.value

    def implicit_host_syncs(self):
        n = C.c_int64()
        self._ck(self.L.pamg_implicit_host_syncs(self.h, C.byref(n)))
        return n.value

    def implicit_bsr(self):
        """(val[E,4,3,3], col[E,4]) of the assembled operator; col is 0-based, -1 where a block is absent."""
        val = np.zeros((self._E, 4, 3, 3)); col = np.zeros((self._E, 4), np.int32)
        self._ck(self.L.pamg_implicit_get_bsr(self.h, _ptr(val), _ptr(col)))
        return val, col

    def implicit_apply(self, x):
        x = np.ascontiguousarray(x, np.float64); y = np.empty_like(x)
        self._ck(self.L.pamg_implicit_apply(self.h, x, y))
        return y

    def unstr_stab(self, tnew, told, dt, u_x, u_y):
        """Petrov-Galerkin diff_coe (E,3) and stab (E,3,3) (transport_tri_unstr.F90:239-267,278)."""
        t = np.ascontiguousarray(tnew, np.float64); o = np.ascontiguousarray(told, np.float64)
        self._ck(self.L.pamg_unstr_upload(self.h, t))
        dc = np.zeros((self._E, 3)); st = np.zeros((self._E, 3, 3))
        self._ck(self.L.pamg_unstr_stab(self.h, o, dt, u_x, u_y, _ptr(dc), _ptr(st)))
        return dc, st

    def unstr_implicit(self, tnew, dt, u_x, u_y, ntime=2, nits=1, use_dir=False, tol=1e-13, max_iters=500, with_stab=False):
        """Time loop of unstr_implicit; returns (tnew, Krylov iterations in total, worst relative residual)."""
        t = np.ascontiguousarray(tnew, np.float64)
        self.implicit_assemble(dt, u_x, u_y, use_dir)
        if with_stab:
            self._ck(self.L.pamg_implicit_set_stab(self.h, 1))
        self._ck(self.L.pamg_unstr_upload(self.h, t))
        it = C.c_int(0); rr = C.c_double(0.0)
        self._ck(self.L.pamg_implicit_step(self.h, ntime, nits, tol, max_iters, C.byref(it), C.byref(rr)))
        out = np.empty_like(t)
        self._ck(self.L.pamg_unstr_download(self.h, out))
        return out, it.value, rr.value

    def trans_rec(self, CFL, no_ele_row, no_ele_col, u_x, u_y, time, nits=2, njac_its=10, direct_solver=False,
                  volume_term=False, x_length=100.0, y_length=100.0):
        """trans_rec (transport_rect.F90:7); returns (x_all (E,4,2), tnew (E,4), ntime)."""
        E = no_ele_row * no_ele_col
        x = np.zeros((E, 4, 2)); t = np.zeros((E, 4)); nt = C.c_int(0)
        self._ck(self.L.pamg_trans_rec(self.h, CFL, no_ele_row, no_ele_col, x_length, y_length, u_x, u_y, time, nits, njac_its,
                                       int(direct_solver), int(volume_term), _ptr(x), _ptr(t), C.byref(nt)))
        return x, t, nt.value

    def findinv(self, M, rhs=None):
        """Batched FINDInv (matrices.F90:1618): returns (Minv, x, status)."""
        M = np.ascontiguousarray(M, np.float64)
        batch, n = M.shape[0], M.shape[1]
        Minv = np.zeros_like(M)
        status = np.zeros(batch, np.int32)
        r = None if rhs is None else np.ascontiguousarray(rhs, np.float64)
        x = None if rhs is None else np.zeros_like(r)
        rc = self.L.pamg_apply_local_minv(self.h, n, batch, M, _ptr(r), _ptr(x), _ptr(Minv), _ptr(status))
        if rc not in (OK, ERR_SINGULAR):
            self._ck(rc)
        return Minv, x, status


class PinnedBuffer:
    """cudaMallocHost buffer exposed as a numpy array (for the HOST-buffer entry points)."""

    def __init__(self, n_doubles):
        p = C.c_void_p()
        rc = lib().pamg_host_alloc(C.byref(p), int(n_doubles) * 8)
        if rc != OK:
            raise PamgError(rc, "pamg_host_alloc")
        self.ptr = p
        self.array = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(int(n_doubles),))

    def free(self):
        if self.ptr:
            self.array = None
            lib().pamg_host_free(self.ptr)
            self.ptr = None


def get_unique_id():
    buf = C.create_string_buffer(128)
    rc = lib().pamg_comm_unique_id(buf)
    if rc != OK:
        raise PamgError(rc, "pamg_comm_unique_id (libnccl.so.2 missing?)")
    return buf.raw
