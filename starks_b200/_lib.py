"""ctypes loader for libstarks_b200.so (the C ABI declared in include/starks_b200.h).

There is no CPU fallback: if the library is missing or no CUDA device is present the
import of an engine fails loudly."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# STARKS_B200_LIB: an alternative build of the same ABI (kernel A/B experiments only)
LIB_PATH = os.environ.get("STARKS_B200_LIB") or os.path.join(_HERE, "libstarks_b200.so")

STK_OK, STK_EINVAL, STK_ECUDA, STK_EUNSUPPORTED, STK_EINDEX = 0, 1, 2, 3, 4


class StarksB200Error(RuntimeError):
  pass


_lib = None

u32p = ctypes.POINTER(ctypes.c_uint32)
u8p = ctypes.POINTER(ctypes.c_uint8)
u64p = ctypes.POINTER(ctypes.c_uint64)
vp = ctypes.c_void_p
u64 = ctypes.c_uint64
cint = ctypes.c_int

# name -> (restype, argtypes); mirrors include/starks_b200.h one to one
SIGNATURES = {
    "stk_version": (cint, []),
    "stk_init": (cint, [cint, ctypes.POINTER(vp)]),
    "stk_destroy": (None, [vp]),
    "stk_last_error": (ctypes.c_char_p, [vp]),
    "stk_set_stream": (cint, [vp, vp]),
    "stk_sync": (cint, [vp]),
    "stk_field_set": (cint, [vp, u32p]),
    "stk_dev_alloc": (cint, [vp, u64, ctypes.POINTER(vp)]),
    "stk_dev_free": (cint, [vp, vp]),
    "stk_host_alloc": (cint, [vp, u64, ctypes.POINTER(vp)]),
    "stk_host_free": (cint, [vp, vp]),
    "stk_memcpy_h2d": (cint, [vp, vp, vp, u64]),
    "stk_memcpy_d2h": (cint, [vp, vp, vp, u64]),
    "stk_memcpy_d2d": (cint, [vp, vp, vp, u64]),
    "stk_memset": (cint, [vp, vp, cint, u64]),
    "stk_ntt": (cint, [vp, vp, u64, u64, vp, u64, u64, u64, u32p, cint]),
    "stk_dft_generic": (cint, [vp, vp, u64, u64, vp, u64, u64, u64, u32p, cint]),
    "stk_ntt_host": (cint, [vp, vp, u64, u64, vp, u64, u64, u64, u32p, cint]),
    "stk_mul_polys": (cint, [vp, vp, u64, vp, u64, vp, u64, u32p]),
    "stk_poly_mul": (cint, [vp, vp, u64, vp, u64, vp]),
    "stk_poly_divmod": (cint, [vp, vp, u64, vp, u64, vp, vp]),
    "stk_poly_compose": (cint, [vp, vp, u64, vp, u64, vp]),
    "stk_poly_eval_multivar": (cint, [vp, vp, vp, u64, u64, vp, vp, vp, u64, u64, vp, u64]),
    "stk_vec_op": (cint, [vp, cint, vp, vp, vp, u64]),
    "stk_power_cycle": (cint, [vp, u32p, u64, vp]),
    "stk_ntt_dist_phase": (cint, [vp, cint, vp, vp, u64, u64, u64, u32p, u64, u64, cint]),
    "stk_ntt_dist_phase0_p2p": (cint, [vp, vp, u64, u32p, u64, u64, cint, u64p]),
    "stk_lde": (cint, [vp, vp, u64, u64, u64, u64, u32p, vp, u64, vp, u64]),
    "stk_lde_p2p": (cint, [vp, vp, u64, u64, u64, u64, u32p, u64, u64, u64p]),
    "stk_ntt_p2p": (cint, [vp, vp, u64, u64, u64, u64, u32p, u64, u64, u64p]),
    "stk_fri_fold4_rows": (cint, [vp, vp, u64, u32p, u32p, u64, u64, vp]),
    "stk_lde_commit_host": (cint, [vp, vp, u64, u64, u64, u64, u32p, vp, u64, vp, vp]),
    "stk_lde_commit": (cint, [vp, vp, u64, u64, u64, u64, u32p, vp, u64, vp, vp]),
    "stk_merkle_commit": (cint, [vp, vp, u64, u64, u64, vp, vp]),
    "stk_merkle_commit_raw": (cint, [vp, vp, u64, u64, vp, vp]),
    "stk_merkle_paths": (cint, [vp, vp, u64, u64, u64, vp, vp, u64, vp, u64]),
    "stk_verify_branches": (cint, [vp, vp, u64, u64, vp, u64, vp, u64, vp]),
    "stk_fri_fold4": (cint, [vp, vp, u64, u32p, u32p, vp]),
    "stk_pseudorandom_indices": (cint, [vp, vp, u64, u64, u64, vp]),
    "stk_fri_prove": (cint, [vp, vp, u64, vp, vp, u32p, u64, u64, u64, vp, u64, vp]),
    "stk_constraint_eval": (cint, [vp, vp, u64, u64, u64, u64, vp, vp, vp, u64, vp, u64]),
    "stk_quotient_eval": (cint, [vp, vp, u64, u64, u64, u64, vp, vp, vp, u64, u32p, u32p, vp, u64, u64, vp, u64]),
    "stk_boundary_eval": (cint, [vp, vp, u64, u64, u64, u64, u32p, u64, vp, vp, u64, vp, u64]),
    "stk_quotient_z": (cint, [vp, vp, u64, u64, u32p, vp, ctypes.POINTER(ctypes.c_uint32)]),
    "stk_div_linear": (cint, [vp, vp, u64, u32p, u64, vp]),
    "stk_lincomb": (cint, [vp, vp, u64, u64, u64, vp, vp]),
    "stk_trace_generate": (cint, [vp, vp, u64, u64, vp, vp, vp, u64, vp]),
    "stk_trace_generate_dev": (cint, [vp, vp, u64, u64, u64, vp, vp, vp, u64, vp, u64]),
    "stk_trace_generate_upload": (cint, [vp, vp, u64, u64, vp, vp, vp, u64, vp, vp, u64]),
    "stk_count_noncanonical": (cint, [vp, vp, u64, vp, cint]),
    "stk_microbench": (cint, [vp, cint, u64, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double)]),
    "stk_microbench_variant": (cint, [vp, cint, cint, u64, ctypes.POINTER(ctypes.c_float),
                                      ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]),
}


def load():
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise StarksB200Error(
        "libstarks_b200.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C starks_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
  lib = ctypes.CDLL(LIB_PATH)
  for name, (res, args) in SIGNATURES.items():
    fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
    fn.restype = res
    fn.argtypes = args
  _lib = lib
  return lib
