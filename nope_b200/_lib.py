"""ctypes binding of include/nope_b200.h.  There is no CPU fallback: if the shared
library is missing, or a call fails, the product path raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_DEFAULT_LIB_PATH = os.path.join(_HERE, "lib", "libnope_b200.so")
LIB_PATH = _DEFAULT_LIB_PATH

c_f32p = C.c_void_p   # raw device / host pointers travel as integers
c_i64p = C.c_void_p

# symbol -> (restype, argtypes); mirrors include/nope_b200.h one to one
SIGNATURES = {
    "nope_last_error": (C.c_char_p, []),
    "nope_abi_version": (C.c_int, []),
    "nope_build_arch": (C.c_char_p, []),
    "nope_unet_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int]),
    "nope_unet_destroy": (None, [C.c_void_p]),
    "nope_unet_load_tensor": (C.c_int, [C.c_void_p, C.c_char_p, c_f32p, C.POINTER(C.c_int64), C.c_int]),
    "nope_unet_finalize": (C.c_int, [C.c_void_p]),
    "nope_unet_set_chunk": (C.c_int, [C.c_void_p, C.c_int]),
    "nope_unet_set_conv_impl": (C.c_int, [C.c_void_p, C.c_int]),
    "nope_unet_sweep": (C.c_int, [C.c_void_p, c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, c_f32p,
                                  c_f32p, C.c_int, c_f32p, c_i64p, C.c_int64, C.c_void_p]),
    "nope_unet_last_launch_count": (C.c_int64, [C.c_void_p]),
    "nope_unet_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "nope_unet_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                         C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "nope_unet_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "nope_unet_get_option": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int)]),
    "nope_unet_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "nope_unet_set_workspace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int]),
    "nope_op_conv_gn_fused": (C.c_int, [C.c_int, C.c_int, c_f32p, C.c_int, c_f32p, C.c_int, c_f32p, c_f32p,
                                        c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, c_f32p, C.c_int, c_f32p,
                                        c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "nope_encoder_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int]),
    "nope_encoder_destroy": (None, [C.c_void_p]),
    "nope_encoder_load_tensor": (C.c_int, [C.c_void_p, C.c_char_p, c_f32p, C.POINTER(C.c_int64), C.c_int]),
    "nope_encoder_finalize": (C.c_int, [C.c_void_p]),
    "nope_encoder_encode": (C.c_int, [C.c_void_p, c_f32p, C.c_int, c_f32p, C.c_void_p]),
    "nope_encoder_last_launch_count": (C.c_int64, [C.c_void_p]),
    "nope_score_topk": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                  C.c_int, c_f32p, c_f32p, c_i64p, C.c_int64, C.c_void_p]),
    "nope_unet_set_metric": (C.c_int, [C.c_void_p, C.c_int, C.c_float]),
    "nope_topk": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_i64p, C.c_int64, C.c_void_p]),
    "nope_topk_pack_floats": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "nope_topk_merge": (C.c_int, [c_f32p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  c_f32p, c_f32p, c_i64p, C.c_void_p]),
    "nope_op_conv": (C.c_int, [C.c_int, C.c_int, c_f32p, C.c_int, c_f32p, C.c_int, c_f32p, c_f32p,
                               c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "nope_op_conv_gn": (C.c_int, [C.c_int, C.c_int, c_f32p, C.c_int, c_f32p, C.c_int, c_f32p, c_f32p,
                                  c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_void_p]),
    "nope_op_groupnorm": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p,
                                    C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "nope_op_linear_attention": (C.c_int, [C.c_int, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "nope_op_attention": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "nope_op_upsample2x": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "nope_ldm_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "nope_ldm_destroy": (None, [C.c_void_p]),
    "nope_ldm_load_tensor": (C.c_int, [C.c_void_p, C.c_char_p, c_f32p, C.POINTER(C.c_int64), C.c_int]),
    "nope_ldm_finalize": (C.c_int, [C.c_void_p]),
    "nope_ldm_set_chunk": (C.c_int, [C.c_void_p, C.c_int]),
    "nope_ldm_set_impl": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "nope_ldm_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "nope_ldm_sweep": (C.c_int, [C.c_void_p, c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, c_f32p,
                                 c_f32p, C.c_int, c_f32p, c_i64p, C.c_int64, C.c_void_p]),
    "nope_ldm_last_launch_count": (C.c_int64, [C.c_void_p]),
    "nope_ldm_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "nope_ldm_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                        C.POINTER(C.c_int64)]),
    "nope_ldm_debug_tap": (C.c_int, [C.c_void_p, c_f32p, c_f32p, C.c_int, C.c_char_p, c_f32p,
                                     C.c_int64, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]),
    "nope_ldm_run_block": (C.c_int, [C.c_void_p, C.c_char_p, c_f32p, C.c_int, c_f32p, C.c_int, C.c_int,
                                     C.c_int, c_f32p, c_f32p, C.c_void_p]),
    "nope_op_mh_attention": (C.c_int, [C.c_int, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "nope_unet_debug_tap": (C.c_int, [C.c_void_p, c_f32p, c_f32p, C.c_int, C.c_char_p, c_f32p,
                                      C.c_int64, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]),
    "nope_vsd_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "nope_vsd_render": (C.c_int, [c_f32p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, c_f32p, C.c_void_p,
                                  C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_int64, c_f32p,
                                  C.c_void_p]),
    "nope_vsd_error": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_float, C.c_double, c_i64p, C.c_void_p, C.c_void_p]),
}

EXPECTED_ABI = 2     # include/nope_b200.h "ABI version"; a stale build with other signatures must not bind

_lib = None


class NopeError(RuntimeError):
    pass


def load():
    """Load libnope_b200.so (raises if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if LIB_PATH == _DEFAULT_LIB_PATH and not os.environ.get("NOPE_NO_AUTOBUILD"):
        # the library is built in-tree by `python -m nope_b200.build` / __graft_entry__.build();
        # on a fresh checkout, or when a source file is newer than the binary, compile it now
        # (nvcc, sm_100a) -- still the CUDA path, never a fallback.  A box without nvcc keeps the
        # shipped binary (its ABI version is checked below).
        from . import build as _build
        if not os.path.exists(LIB_PATH) or (_build.is_stale() and _build.have_nvcc()):
            try:
                _build.build()
            except Exception as exc:
                if not os.path.exists(LIB_PATH):
                    raise NopeError(f"{LIB_PATH} is missing and building it failed: {exc}") from exc
    if not os.path.exists(LIB_PATH):
        raise NopeError(
            f"{LIB_PATH} is missing: build it with `python -m nope_b200.build` "
            "(nope_b200 has no CPU or PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.nope_abi_version.restype = C.c_int
    abi = lib.nope_abi_version()
    if abi != EXPECTED_ABI:
        raise NopeError(f"{LIB_PATH} has ABI version {abi}, this package binds version {EXPECTED_ABI}: "
                        "rebuild with `python -m nope_b200.build --force`")
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise NopeError(load().nope_last_error().decode("utf-8", "replace"))


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())
