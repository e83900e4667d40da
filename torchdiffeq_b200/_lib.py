"""ctypes binding of libtdq.so (include/tdq.h).  The library is the product: if it is missing or does
not load, every solver entry point raises -- there is no CPU or PyTorch fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libtdq.so")

TDQ_MAX_STAGES = 16
TDQ_MAX_K = TDQ_MAX_STAGES + 1
TDQ_MAX_SEGS = 64
TDQ_F32, TDQ_F64, TDQ_C64, TDQ_C128 = 0, 1, 2, 3     # complex: interleaved (re, im) pairs, n counts complex elements
RUN_OK, RUN_DT_UNDERFLOW, RUN_NONFINITE, RUN_MAX_STEPS, RUN_EXCHANGE_TIMEOUT = 0, 1, 2, 3, 4
TDQ_MAX_RANKS = 16
ABI_VERSION = 2


class IpcHandle(C.Structure):
    _fields_ = [("bytes", C.c_ubyte * 64)]


class Tableau(C.Structure):
    _fields_ = [
        ("n_stages", C.c_int32), ("order", C.c_int32), ("fsal", C.c_int32), ("reserved", C.c_int32),
        ("alpha", C.c_double * TDQ_MAX_STAGES),
        ("beta", (C.c_double * TDQ_MAX_K) * TDQ_MAX_STAGES),
        ("c_sol", C.c_double * TDQ_MAX_K),
        ("c_err", C.c_double * TDQ_MAX_K),
        ("c_mid", C.c_double * TDQ_MAX_K),
    ]


class Options(C.Structure):
    _fields_ = [
        ("dtype", C.c_int32), ("ratio_f64", C.c_int32),
        ("rtol", C.c_double), ("atol", C.c_double),
        ("min_step", C.c_double), ("max_step", C.c_double),
        ("safety", C.c_double), ("ifactor", C.c_double), ("dfactor", C.c_double),
        ("t_sign", C.c_double),
        ("max_num_steps", C.c_int64), ("n_global", C.c_int64),
        ("ybuf", C.c_void_p * 2), ("kbuf", C.c_void_p * 2),
        ("always_fit", C.c_int32), ("reserved", C.c_int32),
        ("loop_handle", C.c_uint64),
    ]


class Mailbox(C.Structure):
    _fields_ = [
        ("seq", C.c_uint64),
        ("status", C.c_int32), ("accept", C.c_int32), ("done", C.c_int32), ("out_cursor", C.c_int32),
        ("n_accept", C.c_int64), ("n_reject", C.c_int64),
        ("t0", C.c_double), ("t1", C.c_double), ("dt", C.c_double),
        ("ratio", C.c_double), ("att_t0", C.c_double), ("att_dt", C.c_double),
        ("next_t0", C.c_double), ("next_dt", C.c_double),
        ("on_jump_t", C.c_int32), ("par", C.c_int32),
    ]


class TdqError(RuntimeError):
    pass


_vp, _i32, _i64, _sz, _dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t, C.c_double
_pp = C.POINTER(C.c_void_p)
_pi64 = C.POINTER(C.c_int64)
_pdbl = C.POINTER(C.c_double)
_ptab = C.POINTER(Tableau)

# name -> (restype, argtypes); mirrors include/tdq.h one to one
_SIGNATURES = {
    "tdq_abi_version": (C.c_int, []),
    "tdq_sizeof": (_sz, [_i32]),
    "tdq_last_error": (C.c_char_p, []),
    "tdq_device_sm_count": (C.c_int, [C.POINTER(C.c_int)]),
    "tdq_tableau_get": (C.c_int, [C.c_char_p, _ptab]),
    "tdq_mailbox_create": (C.c_int, [C.POINTER(C.POINTER(Mailbox)), _pp]),
    "tdq_mailbox_destroy": (C.c_int, [C.POINTER(Mailbox)]),
    "tdq_ctrl_size": (_sz, []),
    "tdq_ctrl_tstage_offset": (_sz, []),
    "tdq_ctrl_taux_offset": (_sz, []),
    "tdq_ctrl_init": (C.c_int, [_vp, _ptab, C.POINTER(Options), _vp, _dbl, _i32, _vp, _vp]),
    "tdq_ctrl_set_step_t": (C.c_int, [_vp, _vp, _i32, _vp]),
    "tdq_ctrl_set_jump_t": (C.c_int, [_vp, _vp, _i32, _vp]),
    "tdq_norm_table_fill": (_i64, [_pi64, _pi64, _i32, _i64, _i32, _pi64, _i64]),
    "tdq_norm_partials_len": (_sz, [_sz, _i64]),
    "tdq_scaled_sumsq": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _sz, _vp, _vp, _vp]),
    "tdq_initial_step_h0": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _i32, _vp]),
    "tdq_initial_step_probe": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _sz, _vp]),
    "tdq_initial_step_finish": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _vp]),
    "tdq_set_first_step": (C.c_int, [_vp, _dbl, _vp]),
    "tdq_prepare_attempt": (C.c_int, [_vp, _i32, _vp, _vp]),
    "tdq_stage_combine": (C.c_int, [_vp, _ptab, _i32, _i32, _vp, _vp, _pp, _sz, _vp]),
    "tdq_stage_combine_final": (C.c_int, [_vp, _ptab, _i32, _vp, _vp, _vp, _pp, _sz, _vp]),
    "tdq_error_norm_commit": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _sz, _vp, _vp,
                                        _vp, _vp]),
    "tdq_commit_candidates": (C.c_int, [_vp, _i32, _vp, _vp, _sz, _vp]),
    "tdq_controller": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _vp, _vp]),
    "tdq_interp_fit_eval": (C.c_int, [_vp, _ptab, _i32, _vp, _pp, _pp, _vp, _sz, _vp]),
    "tdq_interp_eval_at": (C.c_int, [_vp, _i32, _pp, _vp, _vp, _sz, _vp]),
    "tdq_poly_eval": (C.c_int, [_i32, _pp, _dbl, _vp, _sz, _vp]),
    "tdq_ctrl_reset_interval": (C.c_int, [_vp, _vp]),
    "tdq_loop_create": (C.c_int, [_vp, _pp, C.POINTER(C.c_uint64)]),
    "tdq_loop_launch": (C.c_int, [_vp, _vp]),
    "tdq_loop_destroy": (C.c_int, [_vp]),
    "tdq_ctrl_set_loop": (C.c_int, [_vp, C.c_uint64, _vp]),
    "tdq_rk4_stage": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "tdq_fixed_emit": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _sz, _vp]),
    "tdq_fixed_final_emit": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _i64, _sz, _vp]),
    "tdq_lincomb": (C.c_int, [_i32, _vp, _vp, _pp, _pdbl, _i32, _sz, _vp]),
    "tdq_linear_supported": (C.c_int, [_i32, _i32]),
    "tdq_linear_weights_bytes": (_sz, [_i32]),
    "tdq_linear_prepare": (C.c_int, [_i32, _vp, _i32, _vp, _vp]),
    "tdq_linear_apply": (C.c_int, [_i32, _vp, _vp, _i32, _sz, _vp, _vp]),
    "tdq_linear_stage": (C.c_int, [_vp, _ptab, _i32, _i32, _vp, _vp, _vp, _vp, _pp, _vp, _i32, _sz, _vp]),
    "tdq_linear_attempt_supported": (C.c_int, [_ptab, _i32, _i32]),
    "tdq_linear_attempt": (C.c_int, [_vp, _ptab, _i32, _pp, _vp, _vp, _vp, _vp, _vp, _i32, _sz, _vp, _vp, _vp, _i32, _vp]),
    "tdq_fixed_emit_cubic": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _sz, _vp]),
    "tdq_pack_segments": (C.c_int, [_i32, _vp, _pp, _pi64, _pi64, _pdbl, _i32, _vp]),
    "tdq_xchg_create": (C.c_int, [_pp, C.POINTER(IpcHandle)]),
    "tdq_xchg_open": (C.c_int, [C.POINTER(IpcHandle), _pp]),
    "tdq_xchg_close": (C.c_int, [_vp]),
    "tdq_xchg_destroy": (C.c_int, [_vp]),
    "tdq_ctrl_set_exchange": (C.c_int, [_vp, _pp, _i32, _i32, C.c_uint64, _vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load libtdq.so once; raises TdqError (never falls back) when it is absent or stale."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TdqError(
            "libtdq.so is not built (%s). Run `python -m torchdiffeq_b200.csrc.build` "
            "(or __graft_entry__.build()); there is no fallback path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise TdqError("libtdq.so does not export %s; rebuild it" % name) from e
        fn.restype = res
        fn.argtypes = args
    if lib.tdq_abi_version() != ABI_VERSION:
        raise TdqError("libtdq.so ABI version mismatch")
    for which, st in ((0, Tableau), (1, Options), (2, Mailbox)):
        if lib.tdq_sizeof(which) != C.sizeof(st):
            raise TdqError("libtdq.so struct layout mismatch for %s; rebuild it" % st.__name__)
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().tdq_last_error()
        raise TdqError("libtdq call failed (%d): %s" % (rc, msg.decode() if msg else "?"))


def tableau(name):
    t = Tableau()
    check(load().tdq_tableau_get(name.encode(), C.byref(t)))
    return t


def tableau_as_dict(name):
    """Dense float64 view of a named tableau (for tests and documentation)."""
    t = tableau(name)
    S = t.n_stages
    return {
        "n_stages": S, "order": t.order, "fsal": bool(t.fsal),
        "alpha": [t.alpha[i] for i in range(S)],
        "beta": [[t.beta[i][j] for j in range(i + 1)] for i in range(S)],
        "c_sol": [t.c_sol[j] for j in range(S + 1)],
        "c_err": [t.c_err[j] for j in range(S + 1)],
        "c_mid": [t.c_mid[j] for j in range(S + 1)],
    }


def norm_table(segs, n, dt_code):
    """Chunk table of tdq_norm_table_fill for segments [(offset, len), ...] of a flat state of n elements, as a
    host list of int64 words; table[1] = number of chunks, table[3] = 1 when every segment is 16-byte aligned."""
    lib = load()
    offs = i64_array([int(o) for o, _ in segs])
    lens = i64_array([int(l) for _, l in segs])
    words = lib.tdq_norm_table_fill(offs, lens, len(segs), int(n), dt_code, None, 0)
    if words < 0:
        check(1)
    buf = (C.c_int64 * words)()
    if lib.tdq_norm_table_fill(offs, lens, len(segs), int(n), dt_code, buf, words) != words:
        check(1)
    return list(buf)


def ptr_array(ptrs):
    """void*[] from a list of ints/None."""
    arr = (C.c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def i64_array(vals):
    return (C.c_int64 * len(vals))(*vals)


def dbl_array(vals):
    return (C.c_double * len(vals))(*vals)
