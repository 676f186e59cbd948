#!/usr/bin/env python
"""Generates p-a_multigrids_b200/host/pamg_iface.F90 from include/pamg.h: one ISO_C_BINDING interface per extern "C"
entry, the pamg_params derived type and the constants.  Run after every change of the header:

    python tools/gen_fortran_iface.py            # rewrites the module
    python tools/gen_fortran_iface.py --check    # exit 1 if the committed module is stale

tests/test_fortran_iface.py checks that every entry of the header appears in the module with the same argument count.
(The image has no Fortran compiler, so the module is generated mechanically and syntax-checked structurally only.)"""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pamg.h")
OUT = os.path.join(ROOT, "p-a_multigrids_b200", "host", "pamg_iface.F90")

# pointer arguments that are ONE value written by the library (everything else with a '*' is an array)
SCALAR_OUT = {"n", "U", "ndof", "l2", "linf", "conv", "cycles", "relres", "npeers", "peer_part", "nfaces", "iters_total",
              "ntime", "ms", "total_ms", "launches"}
# array arguments the header documents as optional (NULL allowed): passed as type(c_ptr) so that c_null_ptr can be given
NULLABLE = {"part_first", "region", "devices", "bc_value", "val", "col", "diff_coe", "stab", "x_all", "analytical", "error",
            "Minv", "status", "rhs", "x", "hist", "strip_of", "dst_strip", "rev", "hmap", "peers", "counts", "X_out", "bc_kind",
            "u_ele"}
NULLABLE_IN = {"pamg_mesh_get": {"X", "neig", "fneig", "dir", "region"},
               "pamg_halo_plan": {"part_first", "strip_of", "dst_strip", "rev", "hmap", "peers", "counts"},
               "pamg_halo_sources": {"part_first"},
               "pamg_apply_local_minv": {"rhs", "x", "Minv", "status"},
               "pamg_trans_rec": {"x_all"}, "pamg_create_multi": {"devices"},
               "pamg_set_parents_partition": {"part_first"}, "pamg_mesh_from_arrays": {"region"},
               "pamg_set_boundary_data": {"bc_value"}, "pamg_implicit_get_bsr": {"val", "col"},
               "pamg_unstr_stab": {"diff_coe", "stab"}, "pamg_output_fields": {"x_all", "analytical", "error"},
               "pamg_vcycle_solve": {"cycles", "hist"}, "pamg_residual": {"l2", "linf"},
               "pamg_timestep_host": {"cycles", "relres"}, "pamg_implicit_step": {"iters_total", "relres"},
               "pamg_halo_peer_info": {"peer_part", "nfaces"}, "pamg_parent_table": {"bc_kind"},
               "pamg_unstr_set_velocity": {"u_ele"}}

FTYPE = {"int": "integer(c_int)", "int32_t": "integer(c_int32_t)", "int64_t": "integer(c_int64_t)", "double": "real(c_double)",
         "float": "real(c_float)"}
KIND = {"int": "c_int", "int32_t": "c_int32_t", "int64_t": "c_int64_t", "double": "c_double", "float": "c_float"}


def strip_comments(text):
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    return re.sub(r"//[^\n]*", " ", text)


def parse_header(path=HEADER):
    """-> (functions [(ret, name, [(ctype, name)])], params fields [(ctype, name)], defines [(name, value)], enums [(name, value)])"""
    raw = open(path).read()
    text = strip_comments(raw)
    defines = [(m.group(1), m.group(2)) for m in re.finditer(r"#define\s+(PAMG_\w+)\s+\(?(-?\d+)\)?", text)
               if m.group(1) != "PAMG_H"]
    enums = []
    for m in re.finditer(r"enum\s*\{([^}]*)\}", text):
        for item in m.group(1).split(","):
            item = item.strip()
            if "=" in item:
                k, v = item.split("=")
                enums.append((k.strip(), v.strip()))
    sm = re.search(r"typedef\s+struct\s+pamg_params\s*\{(.*?)\}\s*pamg_params\s*;", text, flags=re.S)
    fields = []
    for decl in sm.group(1).split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ctype, names = decl.split(None, 1)
        for nm in names.split(","):
            fields.append((ctype, nm.strip()))
    body = text[text.index('extern "C"'):]
    funcs = []
    for m in re.finditer(r"(const\s+char\s*\*|int|void)\s+(pamg_\w+)\s*\(([^;{]*?)\)\s*;", body, flags=re.S):
        ret, name, args = m.group(1), m.group(2), " ".join(m.group(3).split())
        alist = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                am = re.match(r"(.*?)(\w+)$", a)
                alist.append((am.group(1).strip(), am.group(2)))
        funcs.append((" ".join(ret.split()), name, alist))
    return funcs, fields, defines, enums


def fortran_arg(fn, ctype, name):
    """-> (declaration line, set of imported kinds)"""
    const = ctype.startswith("const ")
    base = ctype.replace("const ", "").strip()
    stars = base.count("*")
    base = base.replace("*", "").strip()
    if stars == 0:
        return f"{FTYPE[base]}, value :: {name}", {KIND[base]}
    if base in ("pamg_handle", "pamg_mesh"):
        return (f"type(c_ptr), value :: {name}" if stars == 1 else f"type(c_ptr), intent(out) :: {name}"), {"c_ptr"}
    if base == "pamg_params":
        return f"type(pamg_params), intent({'in' if const else 'inout'}) :: {name}", {"pamg_params"}
    if base == "void":
        return (f"type(c_ptr), value :: {name}" if stars == 1 else f"type(c_ptr), intent(out) :: {name}"), {"c_ptr"}
    if base == "char":
        return f"character(kind=c_char), intent({'in' if const else 'inout'}) :: {name}(*)", {"c_char"}
    if name in NULLABLE_IN.get(fn, ()):
        return f"type(c_ptr), value :: {name}   ! {base}(*) or c_null_ptr", {"c_ptr"}
    if name in SCALAR_OUT and not const:
        return f"{FTYPE[base]}, intent(out) :: {name}", {KIND[base]}
    return f"{FTYPE[base]}, intent({'in' if const else 'inout'}) :: {name}(*)", {KIND[base]}


def generate():
    funcs, fields, defines, enums = parse_header()
    L = []
    L.append("! pamg_iface.F90 -- ISO_C_BINDING interfaces to libpamg_cuda.so for the reference's own Fortran driver")
    L.append("! (main.F90 / transport_tri_semi.F90).  GENERATED by tools/gen_fortran_iface.py from include/pamg.h - do not edit;")
    L.append(f"! {len(funcs)} entries.  The build image has no Fortran compiler: the module is generated mechanically and checked")
    L.append("! against the header by tests/test_fortran_iface.py; the identical call sequence is exercised from C++")
    L.append("! (host/pamg_host.cpp) and Python (pamg.py).  INTEGRATION.md says where each call replaces a contained procedure of")
    L.append("! Semi_implicit_iterative.")
    L.append("!")
    L.append("! Layout: tracer(ilevel)%tnew(nloc, totele_str, totele_unst) is passed as is (column-major, contiguous);")
    L.append("! meshList(:)%X / Neig / fNeig / Dir are gathered once into X(2,3,U), neig(3,U), fneig(3,U), dir(3,U) (Dir: .true. -> 1).")
    L.append("! Every function returns 0 on success, < 0 on error (like ierr / errorflag); pamg_last_error gives the text.")
    L.append("! Arguments documented as optional in pamg.h are type(c_ptr), value: pass c_loc(array) or c_null_ptr.")
    L.append("module pamg_iface")
    L.append("  use, intrinsic :: iso_c_binding")
    L.append("  implicit none")
    L.append("")
    for k, v in defines + enums:
        L.append(f"  integer(c_int), parameter :: {k} = {v}")
    L.append("")
    L.append("  type, bind(c) :: pamg_params")
    for ctype, nm in fields:
        L.append(f"    {FTYPE[ctype]} :: {nm}")
    L.append("  end type pamg_params")
    L.append("")
    L.append("  interface")
    for ret, name, args in funcs:
        decls, imports = [], set()
        for ctype, an in args:
            d, imp = fortran_arg(name, ctype, an)
            decls.append(d)
            imports |= imp
        names, arglist, cur = [an for _, an in args], "", 0
        for i, an in enumerate(names):           # free-form lines are limited to 132 characters: wrap the dummy list
            piece = an + (", " if i + 1 < len(names) else "")
            if cur + len(piece) > 80:
                arglist += "&\n        "
                cur = 0
            arglist += piece
            cur += len(piece)
        if ret == "void":
            head, tail = f"subroutine {name}({arglist})", "end subroutine"
        elif ret == "int":
            head, tail = f"integer(c_int) function {name}({arglist})", "end function"
            imports.add("c_int")
        else:   # const char*: convert with c_f_pointer / a strlen loop on the Fortran side
            head, tail = f"type(c_ptr) function {name}({arglist})", "end function"
            imports.add("c_ptr")
        L.append(f'    {head} &\n        bind(c, name="{name}")')
        if imports:
            L.append("      import :: " + ", ".join(sorted(imports)))
        for d in decls:
            L.append("      " + d)
        L.append(f"    {tail}")
        L.append("")
    L.append("  end interface")
    L.append("end module pamg_iface")
    return "\n".join(L) + "\n"


if __name__ == "__main__":
    text = generate()
    if "--check" in sys.argv:
        cur = open(OUT).read() if os.path.exists(OUT) else ""
        if cur != text:
            print("pamg_iface.F90 is stale: run python tools/gen_fortran_iface.py")
            sys.exit(1)
        print("pamg_iface.F90 is up to date")
    else:
        with open(OUT, "w") as f:
            f.write(text)
        print(f"wrote {OUT}")
