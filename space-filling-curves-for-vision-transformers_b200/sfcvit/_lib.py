"""ctypes binding of include/sfcvit.h."""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_PK = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_PK, "lib", "libsfcvit_tl.so" if os.environ.get("SFC_ATTN_TIMELINE") else "libsfcvit.so")

_lock = threading.Lock()
_lib = None


class SfcGemmEpilogue(ctypes.Structure):
    _fields_ = [
        ("bias", ctypes.c_void_p), ("residual", ctypes.c_void_p), ("aux", ctypes.c_void_p),
        ("out", ctypes.c_void_p), ("out_pre", ctypes.c_void_p),
        ("ld_out", ctypes.c_longlong), ("ld_res", ctypes.c_longlong), ("ld_aux", ctypes.c_longlong),
        ("alpha", ctypes.c_float), ("act", ctypes.c_int), ("aux_mode", ctypes.c_int),
        ("out_fp32", ctypes.c_int), ("accumulate", ctypes.c_int), ("drop_p", ctypes.c_float),
        ("drop_seed", ctypes.c_ulonglong), ("colsum_out", ctypes.c_void_p), ("colsum_fp32", ctypes.c_int),
    ]


_vp, _i, _ll, _sz, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_size_t, ctypes.c_float

# name -> (restype, argtypes); must list every symbol declared in include/sfcvit.h
SIGNATURES = {
    "sfc_last_error": (ctypes.c_char_p, []),
    "sfc_abi_version": (_i, []),
    "sfc_device_sm_count": (_i, []),
    "sfc_set_dropout_epoch_ptr": (None, [_vp]),
    "sfc_curve_perm_scratch_bytes": (_sz, [_i, _i, _i]),
    "sfc_curve_perm": (_i, [_i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "sfc_block_stitch": (_i, [_i, _i, _i, _vp, _i, _vp, _i, _vp]),
    "sfc_hamiltonian_path": (_i, [_i, _i, _vp, _i, _ll, _vp]),
    "sfc_gemm_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "sfc_gemm_suggest_splits": (_i, [_i, _i, _i]),
    "sfc_gemm_colsum_splits": (_i, [_i, _i, _i, _i, _i]),
    "sfc_layernorm_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _f, _vp]),
    "sfc_layernorm_bwd_scratch_bytes": (_sz, [_ll, _i]),
    "sfc_layernorm_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, ctypes.c_ulonglong, _vp, _vp, _vp, _i, _i, _vp, _sz, _ll, _i, _vp]),
    "sfc_colsum_scratch_bytes": (_sz, [_ll, _i]),
    "sfc_colsum": (_i, [_vp, _ll, _ll, _i, _vp, _i, _i, _vp, _sz, _vp]),
    "sfc_interp_concat_fwd": (_i, [_vp, _ll, _i, _i, _i, _vp, _ll, _i, _vp]),
    "sfc_interp_concat_bwd": (_i, [_vp, _ll, _i, _i, _i, _vp, _ll, _i, _vp]),
    "sfc_patch_embed_kpad": (_i, [_i, _i, _i]),
    "sfc_patch_embed_fwd": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _ll, _vp, _ll, _i, _i, _i, _vp]),
    "sfc_patch_gather": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "sfc_act_bwd": (_i, [_vp, _vp, _vp, _ll, _i, _f, _f, ctypes.c_ulonglong, _vp]),
    "sfc_attn_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _f, ctypes.c_ulonglong, _vp]),
    "sfc_attn_bwd_scratch_bytes": (_sz, [_i, _i, _i]),
    "sfc_attn_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _i, _i, _i, _i, _f, _f, ctypes.c_ulonglong, _vp]),
    "sfc_grad_sumsq_scratch_bytes": (_sz, []),
    "sfc_grad_sumsq": (_i, [_vp, _i, _ll, _vp, _vp, _sz, _vp]),
    "sfc_adamw_step": (_i, [_vp, _vp, _vp, _vp, _ll, _i, _i, _f, _f, _f, _f, _f, _i, _f, _f, _vp, _vp, _vp]),
    "sfc_store_f32x4": (_i, [_vp, _f, _f, _f, _f, _vp]),
    "sfc_softce_scratch_bytes": (_sz, []),
    "sfc_softce_fwd": (_i, [_vp, _i, _ll, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "sfc_softce_bwd": (_i, [_vp, _i, _ll, _vp, _ll, _vp, _vp, _vp, _i, _i, _vp, _ll, _vp]),
    "sfc_gemm_bf16": (_i, [_vp, _i, _ll, _vp, _i, _ll, _i, _i, _i, ctypes.POINTER(SfcGemmEpilogue), _vp, _sz, _i, _vp]),
}


ABI_VERSION = 2


def _build_locked():
    """Runs build.py under an inter-process file lock when the library is stale: under torchrun all ranks import at
    once, and only one may compile / link; build.py links to a temporary file and renames. An up-to-date library is
    loaded without writing anything, so a built tree also works read-only."""
    import fcntl
    import importlib.util
    spec = importlib.util.spec_from_file_location("_sfcvit_build", os.path.join(_PK, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    if mod.up_to_date():
        return
    os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
    with open(LIB_PATH + ".lock", "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        try:
            mod.build()
        finally:
            fcntl.flock(lk, fcntl.LOCK_UN)


def load(build_if_missing: bool = True):
    """Loads libsfcvit.so (building it with nvcc when absent or older than its sources and nvcc exists). Raises if it
    cannot be loaded — there is no CPU fallback behind this library."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        have_nvcc = os.path.exists(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))
        if build_if_missing and have_nvcc and os.path.isdir(os.path.join(_PK, "csrc")):
            _build_locked()
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"libsfcvit.so not built: {LIB_PATH}")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if lib.sfc_abi_version() != ABI_VERSION:
            raise RuntimeError("libsfcvit ABI version mismatch")
        _lib = lib
        return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().sfc_last_error()
        raise RuntimeError(f"libsfcvit {what} failed (rc={rc}): {msg.decode() if msg else '?'}")
