"""ctypes binding of libsrst.so (the C ABI in include/srst.h).

There is deliberately no fallback: if the CUDA library is missing or fails to load, importing the
loss modules raises.  Build it with ``python -m srgan_st_b200.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsrst.so")

ABI_MAJOR = 2  # include/srst.h SRST_VERSION // 100

c_float_p = ctypes.POINTER(ctypes.c_float)
c_i64_p = ctypes.POINTER(ctypes.c_int64)
vp = ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/srst.h one to one
SIGNATURES = {
    "srst_version": (ctypes.c_int, []),
    "srst_error_string": (ctypes.c_char_p, [ctypes.c_int]),
    "srst_st_supported": (ctypes.c_int, [ctypes.c_int, ctypes.c_int]),
    "srst_st_num_cfgs": (ctypes.c_int, [ctypes.c_int]),
    "srst_st_force_cfg": (ctypes.c_int, [ctypes.c_int, ctypes.c_int]),
    "srst_st_force_chunk_blocks": (ctypes.c_int, [ctypes.c_int]),
    "srst_st_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 3),
    "srst_st_workspace_bytes_r": (ctypes.c_size_t, [ctypes.c_int] * 5),
    "srst_st_backward_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 5),
    "srst_st_ixy_floats": (ctypes.c_size_t, [ctypes.c_int] * 3),
    "srst_st_forward": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_float, vp, vp, vp, vp, vp,
                                       vp, ctypes.c_size_t, vp]),
    "srst_st_backward": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                        vp, vp]),
    "srst_st_backward_ws": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                           vp, vp, ctypes.c_size_t, vp]),
    "srst_st_forward_per_image": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                 c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                                 ctypes.c_int, ctypes.c_float, vp, vp, vp, vp, vp,
                                                 vp, ctypes.c_size_t, vp]),
    "srst_st_backward_per_image": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                  c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                                  vp, vp, ctypes.c_size_t, vp]),
    "srst_st_forward_map": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_float, vp, vp, vp, vp, vp, vp,
                                           vp, ctypes.c_size_t, vp]),
    "srst_st_backward_map_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 5),
    "srst_st_backward_map": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                            vp, vp, ctypes.c_size_t, vp]),
    "srst_st_features": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, vp, vp, vp, vp, vp]),
    "srst_stpx_forward": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_float, vp, vp, vp, vp, ctypes.c_size_t, vp]),
    "srst_stpx_backward": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, vp, vp]),
    "srst_stpx_forward_per_image": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                   c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                                   ctypes.c_int, ctypes.c_float, vp, vp, vp, vp, ctypes.c_size_t, vp]),
    "srst_stpx_backward_per_image": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                    c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, vp, vp]),
    "srst_bb_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 3),
    "srst_bb_forward": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp,
                                       vp, ctypes.c_size_t, vp]),
    "srst_bb_backward": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, vp, vp, ctypes.c_size_t, vp]),
    "srst_gram_forward": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp,
                                         vp, ctypes.c_size_t, vp]),
    "srst_gram_backward": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_int, vp, vp, ctypes.c_size_t, vp]),
    "srst_pst_forward": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                        ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp,
                                        vp, ctypes.c_size_t, vp]),
    "srst_pst_backward": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                         ctypes.c_int, vp, vp, ctypes.c_size_t, vp]),
    "srst_patch_backward_gt": (ctypes.c_int, [ctypes.c_int, vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                              c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                              ctypes.c_int, vp, vp, ctypes.c_size_t, vp]),
    "srst_patch_forward_per_image": (ctypes.c_int, [ctypes.c_int, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                    c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                                    ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp,
                                                    vp, ctypes.c_size_t, vp]),
    "srst_patch_backward_per_image": (ctypes.c_int, [ctypes.c_int, vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int,
                                                     ctypes.c_int, c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                                     ctypes.c_int, vp, vp, vp, ctypes.c_size_t, vp]),
    "srst_patch_forward_map": (ctypes.c_int, [ctypes.c_int, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                              c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                              ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp, vp,
                                              vp, ctypes.c_size_t, vp]),
    "srst_patch_backward_map": (ctypes.c_int, [ctypes.c_int, vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_int, c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_int,
                                               ctypes.c_int, vp, vp, vp, ctypes.c_size_t, vp]),
    "srst_bbg_supported": (ctypes.c_int, [ctypes.c_int] * 3),
    "srst_bbg_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 6),
    "srst_bbg_num_patches": (ctypes.c_longlong, [ctypes.c_int] * 5),
    "srst_bbg_forward": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp,
                                        vp, ctypes.c_size_t, vp]),
    "srst_bbg_backward": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp,
                                         vp, ctypes.c_size_t, vp]),
    "srst_bbg_forward_per_image": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                  ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                  ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp,
                                                  vp, ctypes.c_size_t, vp]),
    "srst_bbg_backward_per_image": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                   ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp,
                                                   vp, ctypes.c_size_t, vp]),
    "srst_bbg_forward_map": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_float, ctypes.c_float, ctypes.c_int, vp, vp, vp,
                                            vp, ctypes.c_size_t, vp]),
    "srst_bbg_backward_map": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp,
                                             vp, ctypes.c_size_t, vp]),
    "srst_bb_pyramid": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp]),
}


class SrstError(RuntimeError):
    pass


def bind(path: str) -> ctypes.CDLL:
    """Load a library exporting the srst C ABI and attach the prototypes."""
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SrstError(
                f"{LIB_PATH} not found. srgan_st_b200 has no CPU or PyTorch fallback: build the "
                "sm_100a library first with `python -m srgan_st_b200.build`.")
        _lib = bind(LIB_PATH)
        if _lib.srst_version() // 100 != ABI_MAJOR:
            raise SrstError(f"libsrst.so ABI version {_lib.srst_version()} does not match this package")
    return _lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().srst_error_string(code)
        raise SrstError(f"{what} failed ({code}): {msg.decode() if msg else '?'}")
