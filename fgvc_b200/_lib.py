"""ctypes binding of libfgvc_b200.so (the C ABI declared in include/fgvc_b200.h).

There is no CPU fallback: if the library is missing it is built (nvcc); if that fails,
or a compute entry point is called without a CUDA device, the call raises.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int32, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfgvc_b200.so")

MASK_CIRCLE, MASK_SQUARE = 0, 1
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05 = 0, 1, 2
BANK_TF32, BANK_F16 = 0, 1
MEM_UNMASKED = 0x40000000
WEIGHT_COSINE, SIM_L2, HARD_PROP, ZERO_PAD = 1, 2, 4, 8


def zero_pad_flags(radius, W):
    """FGVC_ZERO_PAD_FLAGS of include/fgvc_b200.h"""
    assert 0 < radius <= 255 and 0 < W <= 65535
    return ZERO_PAD | (int(radius) << 8) | (int(W) << 16)


ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED = -1, -2, -3


class FgvcError(RuntimeError):
    def __init__(self, msg, rc=None):
        super().__init__(msg)
        self.rc = rc


class Job(ctypes.Structure):
    _fields_ = [("q_slot", c_int32), ("mem_begin", c_int32), ("mem_end", c_int32), ("out_slot", c_int32)]


class Lane(ctypes.Structure):
    """fgvc_lane: one recurrence of fgvc_point_clip_tail_lanes (offsets in floats)"""
    _fields_ = [("job_begin", c_int32), ("job_end", c_int32), ("L", c_int32), ("Lp", c_int32),
                ("lab_offset", c_int64), ("coord_offset", c_int64)]


class C2FLane(ctypes.Structure):
    """fgvc_c2f_lane: one recurrence of fgvc_c2f_point_clip_tail_lanes (offsets in floats)"""
    _fields_ = [("job_begin", c_int32), ("job_end", c_int32), ("L", c_int32), ("Lp", c_int32),
                ("lab_offset", c_int64), ("out_offset", c_int64), ("coord_offset", c_int64)]


P = c_void_p
I = c_int32
L64 = c_int64
F = c_float

# name -> (restype, argtypes); mirrors include/fgvc_b200.h one to one
SIGNATURES = {
    "fgvc_last_error": (c_char_p, []),
    "fgvc_version": (I, []),
    "fgvc_device_count": (I, []),
    "fgvc_launch_count": (L64, []),
    "fgvc_prep_features": (I, [P, L64, L64, I, I, I, I, I, P, I, I, P]),
    "fgvc_labels_to_pixmajor": (I, [P, L64, I, I, P, I, I, P]),
    "fgvc_labels_to_nchw": (I, [P, I, I, I, I, P, P]),
    "fgvc_gaussian_labels": (I, [P, I, I, I, I, F, P, I, I, P]),
    "fgvc_upsample_labels": (I, [P, I, I, I, P, I, I, I, P]),
    "fgvc_tc_supported": (I, [I, I, I, I, I]),
    "fgvc_topk_bytes": (L64, [I, I, I, I]),
    "fgvc_affinity_topk": (I, [P, I, I, I, I, I, P, I, P, I, I, I, I, P, P, I, P]),
    "fgvc_affinity_topk_seeded": (I, [P, I, I, I, I, I, P, I, P, I, I, I, I, P, P, P, I, P]),
    "fgvc_topk_floor": (I, [P, I, I, I, I, P, I, P, I, I, I, P, P]),
    "fgvc_affinity_topk_packed": (I, [P, I, I, I, I, P, P, I, P, P, I, I, I, I, I, I, P, P, P]),
    "fgvc_packed_tile_shape": (I, [I, I, I, I, I, P, P, P, P]),
    "fgvc_debug_affinity_boxes": (I, [P, I, I, I, I, I, P, I, P, I, I, I, P, P, P, P, I, P]),
    "fgvc_gather_labels": (I, [P, P, I, I, P, I, I, P, I, F, I, P, I, P]),
    "fgvc_dense_propagate": (I, [P, I, I, I, I, P, I, P, P, I, I, F, I, P, I, P]),
    "fgvc_heatmap_coords": (I, [P, I, I, I, I, I, I, P, P]),
    "fgvc_gaussian_coords": (I, [P, I, I, I, F, I, P, P]),
    "fgvc_decode_masks": (I, [P, I, I, I, I, I, P, P, P]),
    "fgvc_decode_masks_pixmajor": (I, [P, I, I, I, I, I, I, I, P, P, P]),
    "fgvc_chain_workspace_bytes": (L64, [I, I, I]),
    "fgvc_mask_clip_tail": (I, [P, P, I, I, P, P, I, I, P, I, I, F, I, P, I, I, I, I, P, P, P, P, L64, P]),
    "fgvc_point_clip_tail": (I, [P, P, I, I, P, P, I, I, P, I, I, F, I, P, I, I, I, I, I, P, P, P, L64, P]),
    "fgvc_point_clip_tail_shared": (I, [P, P, I, P, P, P, I, I, P, I, I, F, I, P, I, I, I, I, I, P, P, P, L64, P]),
    "fgvc_point_clip_tail_lanes": (I, [P, P, I, I, P, P, P, P, P, I, P, I, I, F, I, P, I, I, I, P, P, P, L64, P]),
    "fgvc_c2f_scratch_elems": (L64, [I, I]),
    "fgvc_c2f_propagate": (I, [P, I, I, I, I, I, P, I, I, I, P, P, P, P, I, I, I, I, F, P, I, P, P, P, L64, I, P]),
    "fgvc_c2f_clip_workspace_bytes": (L64, [P, I, I, I, I, I]),
    "fgvc_c2f_clip_weights": (I, [P, I, I, I, I, I, P, I, I, I, P, I, I, P, P, I, I, I, I, F, P, P, P, L64, I, P]),
    "fgvc_c2f_point_clip_tail_lanes": (I, [P, P, I, I, P, P, P, P, I, I, I, I, I, P, P, I, I, I, P, P, P, P]),
}

_lib = None


def load():
    """Load (building first if necessary) the CUDA library.  Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    if not _build.up_to_date():
        # torchrun starts every rank at once: one builds (exclusive file lock, the .so is replaced atomically),
        # the others wait for the lock and find the library current
        import fcntl
        with open(os.path.join(HERE, ".build.lock"), "w") as lk:
            fcntl.flock(lk, fcntl.LOCK_EX)
            try:
                _build.build()
            finally:
                fcntl.flock(lk, fcntl.LOCK_UN)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.fgvc_version() != 100:
        raise FgvcError(f"libfgvc_b200.so version {lib.fgvc_version()} does not match the Python host")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().fgvc_last_error().decode(errors="replace")
        raise FgvcError(f"fgvc_b200 error {rc}: {msg}", rc)


def call(name, *args):
    check(getattr(load(), name)(*args))


def require_cuda():
    import torch
    if not torch.cuda.is_available() or load().fgvc_device_count() < 1:
        raise FgvcError("fgvc_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def ptr(t):
    return c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def launch_count():
    return int(load().fgvc_launch_count())
