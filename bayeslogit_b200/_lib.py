"""ctypes binding of libbayeslogit_b200.so (the C ABI in include/bayeslogit_b200.h).

There is no fallback: if the shared library is missing or cannot be loaded the
import of any compute entry point raises.  This is exactly the stub a maintainer
of the reference's R package would replace `.C(..., PACKAGE="BayesLogit")` with
(INTEGRATION.md shows the R-side binding).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libbayeslogit_b200.so")

TRACE_W = 6


class Tape(C.Structure):
    _fields_ = [("tu", C.c_void_p), ("te", C.c_void_p), ("tn", C.c_void_p), ("tg", C.c_void_p),
                ("lu", C.c_int32), ("le", C.c_int32), ("ln", C.c_int32), ("lg", C.c_int32)]


class EngineError(RuntimeError):
    pass


_lib = None


def lib():
    """Load (once) and return the engine library; raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineError(
            f"{LIB_PATH} not found: build it with `python -m bayeslogit_b200.build` "
            "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i64, u64, u32, ci = C.c_void_p, C.c_int64, C.c_uint64, C.c_uint32, C.c_int
    # part 1: reference entry points
    L.rpg_gamma.argtypes = [vp, vp, vp, vp, vp]
    L.rpg_devroye.argtypes = [vp, vp, vp, vp]
    L.rpg_alt.argtypes = [vp, vp, vp, vp]
    L.rpg_sp.argtypes = [vp, vp, vp, vp, vp]
    L.rpg_hybrid.argtypes = [vp, vp, vp, vp]
    for f in (L.rpg_gamma, L.rpg_devroye, L.rpg_alt, L.rpg_sp, L.rpg_hybrid):
        f.restype = None
    for name, nargs in (("gibbs", 11), ("EM", 8), ("combine", 5), ("mult_gibbs", 12),
                        ("mult_combine", 6)):
        if hasattr(L, name):
            f = getattr(L, name)
            f.argtypes = [vp] * nargs
            f.restype = None
    # part 2: extensions
    L.bl_version.restype = ci
    L.bl_last_error.restype = C.c_char_p
    L.bl_set_device.argtypes = [ci]
    L.bl_set_seed.argtypes = [u64]
    L.bl_get_seed.restype = u64
    L.bl_get_call_counter.restype = u32
    L.bl_kernel_launches.restype = u64
    L.bl_probe_pipeline_schedule.argtypes = [i64, vp, ci]
    L.bl_probe_pipeline_schedule.restype = ci
    tail = [u64, u32, u64]
    L.bl_rpg_devroye_dev.argtypes = [vp, vp, vp, i64, *tail, vp]
    L.bl_rpg_devroye_plain_dev.argtypes = [vp, vp, vp, i64, *tail, vp]
    L.bl_rpg_devroye_loop_dev.argtypes = [vp, vp, vp, i64, *tail, vp]
    L.bl_rpg_gamma_dev.argtypes = [vp, vp, vp, i64, ci, *tail, vp]
    L.bl_rpg_alt_dev.argtypes = [vp, vp, vp, i64, *tail, vp]
    L.bl_rpg_sp_dev.argtypes = [vp, vp, vp, i64, vp, *tail, vp]
    L.bl_rpg_hybrid_dev.argtypes = [vp, vp, vp, i64, *tail, vp]
    L.bl_rpg_devroye_seeded.argtypes = [vp, vp, vp, i64, *tail]
    L.bl_rpg_gamma_seeded.argtypes = [vp, vp, vp, i64, ci, *tail]
    L.bl_rpg_alt_seeded.argtypes = [vp, vp, vp, i64, *tail]
    L.bl_rpg_sp_seeded.argtypes = [vp, vp, vp, i64, vp, *tail]
    L.bl_rpg_hybrid_seeded.argtypes = [vp, vp, vp, i64, *tail]
    tp = C.POINTER(Tape)
    L.bl_rpg_devroye_tape.argtypes = [vp, vp, vp, i64, tp, vp]
    L.bl_rpg_devroye_plain_tape.argtypes = [vp, vp, vp, i64, tp, vp]
    L.bl_rpg_gamma_tape.argtypes = [vp, vp, vp, i64, ci, tp, vp]
    L.bl_rpg_alt_tape.argtypes = [vp, vp, vp, i64, tp, vp]
    L.bl_rpg_sp_tape.argtypes = [vp, vp, vp, i64, vp, tp, vp]
    L.bl_rpg_hybrid_tape.argtypes = [vp, vp, vp, i64, tp, vp]
    cd = C.c_double
    L.bl_logit_gibbs.argtypes = [vp] * 7 + [ci, ci, ci, ci, u64, ci]
    L.bl_mlogit_gibbs.argtypes = [vp] * 7 + [ci, ci, ci, ci, ci, u64, ci]
    L.bl_nb_gibbs.argtypes = [vp, vp, vp, vp, cd, vp, vp, ci, ci, ci, u64]
    L.bl_nb_gibbs_df.argtypes = [vp, vp, vp, vp, vp, cd, vp, vp, ci, ci, ci, ci, u64]
    L.bl_nb_gibbs_dfreal.argtypes = [vp, vp, vp, vp, vp, cd, vp, vp, ci, ci, ci, ci, u64]
    L.bl_nb_gibbs_dfreal_dev.argtypes = [vp, vp, vp, vp, vp, cd, vp, vp, i64, ci, ci, ci, u64, u64, vp]
    L.bl_logit_gibbs_thin.argtypes = [vp] * 7 + [ci, ci, ci, ci, u64, ci, ci]
    L.bl_set_seed_r.argtypes = [vp]
    L.bl_set_seed_r.restype = None
    L.bl_nb_gibbs_df_dev.argtypes = [vp, vp, vp, vp, vp, cd, vp, vp, i64, ci, ci, ci, u64, u64, vp]
    L.bl_logit_gibbs_dev.argtypes = [vp] * 7 + [i64, ci, ci, ci, u64, ci, u64, vp]
    L.bl_mlogit_gibbs_dev.argtypes = [vp] * 7 + [i64, ci, ci, ci, ci, u64, ci, u64, vp]
    L.bl_nb_gibbs_dev.argtypes = [vp, vp, vp, vp, cd, vp, vp, i64, ci, ci, u64, u64, vp]
    L.bl_logit_chains.argtypes = [vp] * 6 + [ci, ci, ci, ci, ci, u64, ci]
    L.bl_logit_chains_dev.argtypes = [vp] * 6 + [ci, i64, ci, ci, ci, u64, ci, vp]
    L.bl_logit_multichain.argtypes = [vp] * 6 + [ci, ci, ci, ci, ci, u64, ci]
    L.bl_logit_multichain_dev.argtypes = [vp] * 6 + [ci, i64, ci, ci, ci, u64, ci, vp]
    L.bl_mlogit_multichain.argtypes = [vp] * 6 + [ci, ci, ci, ci, ci, ci, u64, ci]
    L.bl_mlogit_multichain_dev.argtypes = [vp] * 6 + [ci, i64, ci, ci, ci, ci, u64, ci, vp]
    L.bl_nb_multichain.argtypes = [vp, vp, vp, vp, cd, vp, vp, ci, ci, ci, ci, ci, u64, ci]
    L.bl_nb_multichain_dev.argtypes = [vp, vp, vp, vp, cd, vp, vp, ci, i64, ci, ci, ci, u64, ci, vp]
    L.bl_comm_unique_id.argtypes = [vp]
    L.bl_comm_init.argtypes = [vp, ci, ci]
    L.bl_comm_init_local.argtypes = [ci, ci]
    L.bl_vcomm_create.argtypes = [ci]
    L.bl_vcomm_bind.argtypes = [ci]
    L.bl_comm_peer_handle.argtypes = [vp]
    L.bl_comm_peer_open.argtypes = [vp]
    L.bl_probe_pg_moments.argtypes = [vp, vp, vp, vp, i64]
    L.bl_probe_v_eval.argtypes = [vp, vp, i64]
    L.bl_probe_specfun.argtypes = [vp, ci, vp, vp, vp, i64]
    L.bl_probe_philox.argtypes = [vp, vp, vp]
    L.bl_probe_nb_dispersion.argtypes = [vp, vp, vp, vp, ci, i64, u64, u32, ci]
    L.bl_probe_peaks.argtypes = [vp]
    L.bl_hybrid_timing.argtypes = [ci]
    L.bl_hybrid_timing_last.argtypes = [vp, vp]
    _lib = L
    return L


def check(status=0):
    """Raise EngineError if the last call reported an error."""
    L = lib()
    msg = L.bl_last_error()
    if status != 0 or msg:
        text = msg.decode() if msg else "engine call failed"
        L.bl_clear_error()
        raise EngineError(text)
