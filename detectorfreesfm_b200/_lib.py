"""ctypes binding of the C ABI in include/dfsfm_b200.h.  There is no CPU fallback: if the CUDA library is
missing or a call fails, an exception is raised."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdfsfm_b200.so")

_lib = None

c_void_p, c_int, c_float, c_char_p, c_int64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_char_p, ctypes.c_int64

# name -> (restype, argtypes); mirrors include/dfsfm_b200.h one to one
PROTOTYPES = {
    "dfsfm_last_error": (c_char_p, []),
    "dfsfm_version": (c_int, []),
    "dfsfm_launch_count": (c_int64, []),
    "dfsfm_thread_set_pdl": (None, [c_int]),
    "dfsfm_debug_gemm_slab": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                                      c_int, c_int, c_void_p]),
    "dfsfm_set_engine": (None, [c_int]),
    "dfsfm_get_engine": (c_int, []),
    "dfsfm_profile_enable": (None, [c_int]),
    "dfsfm_profile_report": (c_int, [c_char_p, c_int]),
    "dfsfm_post_create": (c_int, [ctypes.POINTER(c_void_p), c_int]),
    "dfsfm_post_destroy": (None, [c_void_p]),
    "dfsfm_post_merge_keypoints": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                           ctypes.POINTER(c_int64), c_void_p]),
    "dfsfm_resize_lanczos_gray": (c_int, [c_void_p, c_int, c_int, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                          c_void_p, c_void_p, c_void_p]),
    "dfsfm_debug_timeline_arm": (c_int, [c_int]),
    "dfsfm_debug_timeline_read": (c_int, [c_void_p, c_void_p, c_int]),
    "dfsfm_coarse_create": (c_int, [ctypes.POINTER(c_void_p), c_int]),
    "dfsfm_coarse_destroy": (None, [c_void_p]),
    "dfsfm_coarse_set_param": (c_int, [c_void_p, c_char_p, c_void_p, c_int64, c_int64, c_int]),
    "dfsfm_coarse_features": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dfsfm_coarse_features_pair": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dfsfm_coarse_features_fine": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dfsfm_coarse_fine_match": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                        c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "dfsfm_coarse_transformer": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "dfsfm_coarse_match": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_float, c_int, c_float,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "dfsfm_crop_and_resize_forward": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_float,
                                              c_int, c_int, c_void_p, c_void_p]),
    "dfsfm_refine_create": (c_int, [ctypes.POINTER(c_void_p), c_int, c_int, c_int]),
    "dfsfm_refine_destroy": (None, [c_void_p]),
    "dfsfm_refine_set_param": (c_int, [c_void_p, c_char_p, c_void_p, c_int64, c_int64, c_int]),
    "dfsfm_refine_chunk": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dfsfm_assign_bags": (c_int, [ctypes.POINTER(c_void_p), c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int]),
    "dfsfm_bags_sizes": (None, [c_void_p, ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), ctypes.POINTER(c_int64)]),
    "dfsfm_bags_export": (None, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dfsfm_bags_destroy": (None, [c_void_p]),
    "dfsfm_debug_pyset": (c_int, [c_int, c_void_p, c_int64, c_void_p, c_int64, c_void_p, ctypes.POINTER(c_int64)]),
    "dfsfm_debug_gemm": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                                 c_int, c_int, c_void_p]),
}


class DfsfmError(RuntimeError):
    pass


def load_library():
    """dlopen libdfsfm_b200.so and bind every symbol of the header.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DfsfmError(f"{LIB_PATH} not found: run `python __graft_entry__.py` (build()) first; "
                         "there is no CPU fallback for this engine")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != 0:
        msg = load_library().dfsfm_last_error()
        raise DfsfmError(msg.decode() if msg else f"dfsfm error {code}")


def ptr(t):
    """device/host pointer of a torch tensor (or None)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    """torch's current stream on ``device`` (default: the current device) -- the stream every C-ABI call is given"""
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
