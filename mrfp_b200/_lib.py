"""ctypes binding of libmrfp_b200.so (the C ABI declared in include/mrfp_b200.h).

There is no fallback: if the shared library is missing or a symbol is absent, importing the ops fails
loudly.  `python -m mrfp_b200.build` (or `__graft_entry__.build()`) produces the library in-tree.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libmrfp_b200.so")

c_float_p = ctypes.c_void_p     # device pointers travel as integers (tensor.data_ptr())
c_void_pp = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); mirrors include/mrfp_b200.h one to one
SIGNATURES = {
    "mrfp_version": (ctypes.c_int, []),
    "mrfp_strerror": (ctypes.c_char_p, [ctypes.c_int]),
    "mrfp_npplus_ws_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "mrfp_npplus_ws_init": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "mrfp_npplus_fwd_f32": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                           ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_void_p]),
    "mrfp_npplus_bwd_f32": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                           ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_void_p]),
    "mrfp_relu_psum_f32": (ctypes.c_int, [c_float_p, c_float_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "mrfp_npplus_presummed_ws_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "mrfp_npplus_fwd_presummed_f32": (ctypes.c_int, [c_float_p, ctypes.c_void_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                                     c_float_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                                     ctypes.c_int, ctypes.c_void_p]),
    "mrfp_hrfp_plan_create": (ctypes.c_int, [c_void_pp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.c_int]),
    "mrfp_hrfp_plan_destroy": (None, [ctypes.c_void_p]),
    "mrfp_hrfp_plan_ws_bytes": (ctypes.c_size_t, [ctypes.c_void_p]),
    "mrfp_hrfp_plan_saved_bytes": (ctypes.c_size_t, [ctypes.c_void_p]),
    "mrfp_hrfp_plan_lut_bytes": (ctypes.c_size_t, [ctypes.c_void_p]),
    "mrfp_hrfp_plan_write_luts": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]),
    "mrfp_hrfp_plan_stage": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "mrfp_hrfp_plan_set_fusion": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "mrfp_hrfp_np_ws_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "mrfp_hrfp_fwd": (ctypes.c_int, [ctypes.c_void_p, c_float_p, c_void_pp, c_void_pp, c_void_pp, c_void_pp,
                                     c_void_pp, ctypes.c_float, ctypes.c_float, c_float_p, c_float_p, c_float_p,
                                     c_float_p, c_float_p, ctypes.c_void_p, c_float_p, c_float_p,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "mrfp_hrfp_bwd": (ctypes.c_int, [ctypes.c_void_p, c_float_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, c_void_pp,
                                     c_float_p, c_float_p, c_float_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                     c_float_p, ctypes.c_void_p, ctypes.c_void_p]),
    "mrfp_hrfp_plus_add": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, c_float_p,
                                          ctypes.c_void_p]),
    "mrfp_hrfp_plus_add_bilinear": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, ctypes.c_int,
                                                   ctypes.c_int, c_float_p, ctypes.c_void_p]),
    "mrfp_hrfp_tail_final2_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, ctypes.c_int,
                                                 ctypes.c_int, c_float_p, c_float_p, ctypes.c_int, c_float_p, ctypes.c_void_p]),
    "mrfp_hrfp_tail_final2_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, c_float_p,
                                                 ctypes.c_int, ctypes.c_void_p, c_float_p, c_float_p, ctypes.c_void_p]),
    "mrfp_hrfp_tail_final2_bwd_rk": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, c_float_p,
                                                    ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, c_float_p, c_float_p,
                                                    ctypes.c_void_p]),
    "mrfp_add_f32": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.c_size_t, ctypes.c_void_p]),
    "mrfp_bilinear_bwd_table_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "mrfp_bilinear_bwd_write_table": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t]),
    "mrfp_bilinear_up_bwd_f32": (ctypes.c_int, [c_float_p, c_float_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    "mrfp_instnorm_fwd_f32": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, c_float_p, c_float_p, ctypes.c_void_p,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int,
                                             ctypes.c_void_p]),
    "mrfp_instnorm_bwd_f32": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                             c_float_p, c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_void_p]),
    "mrfp_instnorm_bwd_np_f32": (ctypes.c_int, [c_float_p] * 9 + [ctypes.c_void_p, ctypes.c_size_t, c_float_p, c_float_p, c_float_p,
                                                ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
}

# test / bench hooks exported by the library but not declared in the public header (single kernels on caller buffers)
DEBUG_SIGNATURES = {
    "mrfp_debug_conv3x3_bf16": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 6 + [ctypes.c_void_p] * 4),
    "mrfp_debug_conv3x3_tf32": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 6 + [ctypes.c_void_p] * 4),
    "mrfp_debug_stage_op": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_void_p, ctypes.c_void_p]),
    "mrfp_debug_nchw_to_nhwc": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
}

_lib = None


class MrfpError(RuntimeError):
    pass


def load():
    """Loads the library once and binds every declared symbol (raises if any is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise MrfpError(f"{LIB_PATH} not found: build it with `python -m mrfp_b200.build` "
                        "(there is no CPU / PyTorch fallback for the MRFP kernels)")
    lib = ctypes.CDLL(LIB_PATH)
    for table in (SIGNATURES, DEBUG_SIGNATURES):
        for name, (res, args) in table.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
    _lib = lib
    return lib


# ----------------------------------------------------------------------------------------------------------------------
# scratch memory: ONE grow-only, zero-initialised buffer per (device, stream) and purpose, shared by every call on that
# stream (the kernels' scratch use is stream-ordered, nothing in it outlives a call).  Allocating per call costs a caching-
# allocator round trip on the launch path and, per HRFP plan, pinned 1.7 GB for the life of the process.
# ----------------------------------------------------------------------------------------------------------------------
_SCRATCH = {}


def scratch(device, nbytes: int, purpose: str = "ws"):
    """uint8 tensor of >= nbytes on `device`, private to the current stream; zero-filled when (re)allocated — the NP+
    kernels need their 64-byte control block zero on first use and re-arm it themselves afterwards (include/mrfp_b200.h)."""
    import torch
    device = torch.device(device)
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream, purpose)
    buf = _SCRATCH.get(key)
    if buf is None or buf.numel() < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise MrfpError("scratch buffer would be (re)allocated during CUDA-graph capture: run the same shapes once "
                            "eagerly on this stream before capturing")
        buf = torch.zeros(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _SCRATCH[key] = buf
    return buf


def release_scratch():
    """Drops every cached scratch buffer (they are re-created on demand)."""
    _SCRATCH.clear()


def check(rc: int, what: str):
    if rc != 0:
        msg = load().mrfp_strerror(rc).decode()
        raise MrfpError(f"{what} failed: rc={rc} ({msg})")
