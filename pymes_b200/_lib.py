"""ctypes binding of ``libpymes_b200.so`` (the C ABI in include/pymes_b200.h).

There is deliberately no fallback: if the shared library is missing or a call
returns an error the caller gets a ``RuntimeError``.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# PYMES_B200_LIB overrides the library path (A/B runs of kernel variants in tools/); the
# default is the in-tree build
LIB_PATH = os.environ.get("PYMES_B200_LIB") or os.path.join(_PKG, "libpymes_b200.so")

MAX_DIMS = 4
MAX_TERMS = 8

I64x4 = C.c_int64 * MAX_DIMS
I32x4 = C.c_int32 * 4


class Term(C.Structure):
    _fields_ = [("A", C.c_void_p), ("B", C.c_void_p), ("nk", C.c_int32), ("_pad", C.c_int32),
                ("k_ext", I64x4), ("a_kstr", I64x4), ("b_kstr", I64x4),
                ("a_mstr", I64x4), ("b_nstr", I64x4), ("alpha", C.c_double),
                ("a_gen", C.c_void_p)]      # const pmb_ueg_operand_t * (generated A operand) or NULL


class Contract(C.Structure):
    _fields_ = [("nm", C.c_int32), ("nn", C.c_int32), ("nterms", C.c_int32), ("_pad", C.c_int32),
                ("m_ext", I64x4), ("n_ext", I64x4), ("c_mstr", I64x4), ("c_nstr", I64x4),
                ("C", C.c_void_p), ("beta", C.c_double), ("terms", Term * MAX_TERMS)]


class Bdot(C.Structure):
    _fields_ = [("A", C.c_void_p), ("B", C.c_void_p), ("out", C.c_void_p), ("ni", C.c_int32), ("nr", C.c_int32),
                ("i_ext", I64x4), ("o_istr", I64x4), ("a_istr", I64x4), ("b_istr", I64x4),
                ("r_ext", I64x4), ("a_rstr", I64x4), ("b_rstr", I64x4),
                ("alpha", C.c_double), ("beta", C.c_double)]


class Gemv(C.Structure):
    _fields_ = [("vec", C.c_void_p), ("B", C.c_void_p), ("out", C.c_void_p), ("nk", C.c_int32), ("nx", C.c_int32),
                ("k_ext", I64x4), ("v_kstr", I64x4), ("b_kstr", I64x4),
                ("x_ext", I64x4), ("b_xstr", I64x4), ("o_xstr", I64x4),
                ("alpha", C.c_double), ("beta", C.c_double)]


class Ueg(C.Structure):
    _fields_ = [("n_orb", C.c_int32), ("imax", C.c_int32), ("n_occ", C.c_int32), ("n_ele", C.c_int32),
                ("omega", C.c_double), ("u_table", C.c_void_p), ("u_table_len", C.c_int32),
                ("_pad", C.c_int32), ("kvec", C.c_void_p), ("kp", C.c_void_p), ("index_map", C.c_void_p)]


class UegOperand(C.Structure):
    _fields_ = [("ueg", Ueg), ("W0a", C.c_void_p), ("W1a", C.c_void_p), ("W0s", C.c_void_p),
                ("lin", C.c_void_p), ("nz", C.c_void_p), ("lo", I32x4), ("m_axis", I32x4),
                ("k_axis", I32x4)]


class Blocked(C.Structure):
    _fields_ = [("A", C.c_void_p), ("B", C.c_void_p), ("C", C.c_void_p), ("a_moff", C.c_void_p),
                ("c_moff", C.c_void_p), ("a_koff", C.c_void_p), ("b_koff", C.c_void_p), ("tiles", C.c_void_p),
                ("n_tiles", C.c_int32), ("n0_ext", C.c_int32), ("n1_ext", C.c_int32), ("_pad", C.c_int32),
                ("b_n1str", C.c_int64), ("c_n1str", C.c_int64), ("alpha", C.c_double), ("beta", C.c_double)]


class Gather(C.Structure):
    _fields_ = [("val", C.c_void_p), ("idx", C.c_void_p), ("D", C.c_void_p), ("out", C.c_void_p),
                ("ext", I32x4), ("role", I32x4), ("x_str", C.c_int64 * 3), ("d_ystr", C.c_int64),
                ("d_jstr", C.c_int64), ("alpha", C.c_double), ("beta", C.c_double)]


class Group(C.Structure):
    _fields_ = [("A", C.c_void_p), ("B", C.c_void_p), ("C", C.c_void_p), ("a_row", C.c_void_p),
                ("a_ent", C.c_void_p), ("b_ent", C.c_void_p), ("b_col", C.c_void_p), ("c_row", C.c_void_p),
                ("c_col", C.c_void_p), ("tiles", C.c_void_p), ("n_tiles", C.c_int32), ("_pad", C.c_int32),
                ("alpha", C.c_double)]


class GroupBatched(C.Structure):
    _fields_ = [("g", Group), ("n_batch", C.c_int32), ("_pad", C.c_int32), ("a_bstr", C.c_int64),
                ("b_bstr", C.c_int64), ("c_bstr", C.c_int64)]


_SIGS = {
    "pmb_version": (C.c_int, []),
    "pmb_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "pmb_launch_count": (C.c_longlong, []),
    "pmb_launch_count_reset": (None, []),
    "pmb_error_string": (C.c_char_p, [C.c_int]),
    "pmb_contract_workspace": (C.c_size_t, [C.POINTER(Contract)]),
    "pmb_contract": (C.c_int, [C.POINTER(Contract), C.c_void_p, C.c_size_t, C.c_void_p]),
    "pmb_contract_set_tuning": (None, [C.c_int, C.c_int]),
    "pmb_contract_set_panel_bytes": (None, [C.c_longlong]),
    "pmb_axpby4": (C.c_int, [I64x4, C.c_double, C.c_void_p, I64x4, C.c_double, C.c_void_p, I64x4, C.c_void_p]),
    "pmb_mp2_amplitudes": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p,
                                     I64x4, C.c_void_p, C.c_void_p]),
    "pmb_update_doubles": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                     C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                     C.c_void_p]),
    "pmb_update_singles": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pmb_energy_doubles": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, I64x4, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pmb_tilde": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "pmb_sym_baji": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "pmb_dots": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                           C.c_size_t, C.c_void_p]),
    "pmb_lincomb": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_void_p), C.c_int64, C.c_double,
                              C.c_void_p, C.c_void_p]),
    "pmb_reduce_workspace": (C.c_size_t, []),
    "pmb_bdot": (C.c_int, [C.POINTER(Bdot), C.c_void_p]),
    "pmb_gemv": (C.c_int, [C.POINTER(Gemv), C.c_void_p]),
    "pmb_cdiv_shifted": (C.c_int, [C.c_int64, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pmb_sector_gather": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                    C.c_int64, C.c_void_p]),
    "pmb_sector_scatter": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                     C.c_int64, C.c_void_p]),
    "pmb_ueg_umat": (C.c_int, [C.POINTER(Ueg), C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_void_p]),
    "pmb_ueg_pair_tables": (C.c_int, [C.POINTER(Ueg), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "pmb_ueg_build_nz": (C.c_int, [C.POINTER(Ueg), C.c_void_p, C.c_void_p, C.c_void_p, I32x4, I32x4,
                                   C.c_void_p, C.c_void_p]),
    "pmb_blocked_contract": (C.c_int, [C.POINTER(Blocked), C.c_void_p]),
    "pmb_gather_expand": (C.c_int, [C.POINTER(Gather), C.c_void_p]),
    "pmb_group_contract": (C.c_int, [C.POINTER(Group), C.c_void_p]),
    "pmb_group_contract_batched": (C.c_int, [C.POINTER(GroupBatched), C.c_void_p]),
    "pmb_momentum_residue": (C.c_int, [C.c_int, I64x4, I64x4, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pmb_synth_block": (C.c_int, [C.c_int, C.c_ulonglong, C.c_double, C.c_void_p, I32x4, I32x4, C.c_void_p,
                                  C.c_void_p]),
    "pmb_ueg_build_block": (C.c_int, [C.POINTER(Ueg), C.c_void_p, C.c_void_p, C.c_void_p, I32x4, I32x4,
                                      C.c_void_p, C.c_void_p]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def load():
    """dlopen the library (once) and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "pymes_b200: %s is missing. Build it with `python -m pymes_b200.build` "
            "(needs nvcc; there is no CPU fallback)." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().pmb_error_string(rc)
        raise RuntimeError("pymes_b200 %s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))
