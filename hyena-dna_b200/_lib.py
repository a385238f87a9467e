"""ctypes binding of libhyena_b200.so (C ABI declared in include/hyena_b200.h).

There is no CPU fallback: if the shared library is missing, or a call is made without a CUDA
device, the error is raised to the caller.
"""
import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# HYENA_B200_LIB: alternative build of the same library (A/B runs of kernel variants); default = the in-tree build
LIB_PATH = os.environ.get("HYENA_B200_LIB") or os.path.join(_HERE, "libhyena_b200.so")
CSRC = os.path.join(_HERE, "csrc")

_lib = None
_lock = threading.Lock()

c_fp = ctypes.c_void_p        # device pointers travel as integers
_i, _f, _sz, _vp = ctypes.c_int, ctypes.c_float, ctypes.c_size_t, ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/hyena_b200.h declares
SIGNATURES = {
    "hyena_b200_abi_version": (_i, []),
    "hyena_b200_last_error": (ctypes.c_char_p, []),
    "hyena_b200_launch_count": (ctypes.c_ulonglong, []),
    "hyena_b200_max_seqlen": (_i, []),
    "hyena_b200_profile_begin": (_i, []),
    "hyena_b200_profile_end": (_i, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_ulonglong), _i]),
    "hyena_b200_kind_name": (ctypes.c_char_p, [_i]),
    "hyena_b200_kind_count": (_i, []),
    "hyena_b200_spectrum_from_rfft": (_i, [c_fp, _i, c_fp, c_fp, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_spectrum_to_rfft": (_i, [c_fp, _i, c_fp, c_fp, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_spectrum_elems": (_sz, [_i]),
    "hyena_b200_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "hyena_b200_workspace_min_bytes": (_sz, [_i, _i, _i, _i]),
    "hyena_b200_filter_fwd": (_i, [c_fp, _i, c_fp] + [c_fp] * 7 + [c_fp, c_fp, _f, _i, _i, _i, _i, _i, c_fp, _vp]),
    "hyena_b200_filter_bwd_stage1": (_i, [c_fp, _i, c_fp] + [c_fp] * 7 + [c_fp, c_fp, _f, _i, _i, _i, _i, _i, c_fp, c_fp, c_fp, _vp]),
    "hyena_b200_filter_bwd_stage2": (_i, [c_fp] * 11 + [_i, _i, _i, _vp]),
    "hyena_b200_filter_spectrum": (_i, [c_fp, c_fp, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_core_fwd": (_i, [c_fp] * 9 + [_i, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_core_bwd": (_i, [c_fp] * 16 + [_i, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_fftconv_fwd": (_i, [c_fp] * 4 + [_i, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_fftconv_bwd": (_i, [c_fp] * 7 + [_i, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_gemm_available": (_i, []),
    "hyena_b200_proj_wimg_bytes": (_sz, [_i, _i]),
    "hyena_b200_proj_debug_buffer": (_i, [_vp]),
    "hyena_b200_proj_wgrad_scratch_bytes": (_sz, [_i, _i]),
    "hyena_b200_proj_wgrad": (_i, [c_fp, c_fp, c_fp, c_fp, _i, _f, _i, _i, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_proj_gemm": (_i, [c_fp, _i, c_fp, _i, _i, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "hyena_b200_filter_ddelta": (_i, [c_fp, c_fp, c_fp, c_fp, _f, _i, _i, c_fp, _vp]),
    "hyena_b200_filter_l1norm_fwd": (_i, [c_fp, c_fp, c_fp, _i, _i, _vp]),
    "hyena_b200_filter_l1norm_bwd": (_i, [c_fp, c_fp, c_fp, c_fp, _i, _i, _vp]),
    "hyena_b200_add_layernorm_scratch_bytes": (_sz, [ctypes.c_longlong, _i]),
    "hyena_b200_add_layernorm_fwd": (_i, [c_fp, c_fp, c_fp, c_fp, _f, c_fp, c_fp, c_fp, c_fp, ctypes.c_longlong, _i, _vp]),
    "hyena_b200_add_layernorm_bwd": (_i, [c_fp] * 9 + [ctypes.c_longlong, _i, _vp, _sz, _vp]),
    "hyena_b200_gemm": (_i, [_i, _i, _i, _i, _i, _f, c_fp, _i, ctypes.c_longlong, c_fp, _i, ctypes.c_longlong, _f, c_fp,
                             _i, ctypes.c_longlong, _i, c_fp, _i, _vp, _sz, _vp]),
    "hyena_b200_decode_workspace_bytes": (_sz, [_i, _i, _i]),
    "hyena_b200_decode_prefill": (_i, [c_fp] * 6 + [_i, _i, _i, _i, _vp]),
    "hyena_b200_decode_step": (_i, [c_fp] * 12 + [_i, _i, _i, _i, _vp, _sz, _vp]),
}


class HyenaB200Error(RuntimeError):
    pass


def build(verbose=False):
    """Compile csrc/*.cu for sm_100a into libhyena_b200.so (nvcc cross-compiles without a GPU)."""
    jobs = str(min(8, os.cpu_count() or 1))
    out = subprocess.run(["make", "-C", CSRC, "-j", jobs], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise HyenaB200Error("building libhyena_b200.so failed (see output above)")
    return LIB_PATH


def lib():
    """Load the shared library (once) and bind the signatures."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise HyenaB200Error(
                        f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "or `make -C hyena-dna_b200/csrc`. There is no CPU fallback.")
                L = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(L, name)
                    fn.restype, fn.argtypes = res, args
                if L.hyena_b200_abi_version() != 2:
                    raise HyenaB200Error("libhyena_b200.so ABI version mismatch")
                _lib = L
    return _lib


def check(status):
    if status != 0:
        raise HyenaB200Error(lib().hyena_b200_last_error().decode() or "hyena_b200 call failed")


def launch_count():
    return int(lib().hyena_b200_launch_count())


def profile_begin():
    check(lib().hyena_b200_profile_begin())


def profile_end():
    """-> {kernel class: (device ms, launches)} for the window opened by profile_begin()."""
    n = int(lib().hyena_b200_kind_count())
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_ulonglong * n)()
    check(lib().hyena_b200_profile_end(ms, cnt, n))
    return {lib().hyena_b200_kind_name(i).decode(): (ms[i], int(cnt[i])) for i in range(n) if cnt[i]}
