"""ctypes binding of libvidc_b200.so (include/vidc_b200.h).

The library is the product: if it is missing this module raises at import of the first symbol --
there is no PyTorch / CPU fallback anywhere in the package.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvidc_b200.so")

VIDC_OK = 0
VIDC_ERR_INVALID_ARGUMENT = -1
VIDC_ERR_BATCH_MISMATCH = -2
VIDC_ERR_CUDA = -3
VIDC_ERR_NO_DEVICE = -4
VIDC_BILINEAR = 0
VIDC_NEAREST = 1
VIDC_BICUBIC = 2

c_f32p = ctypes.c_void_p


class VidcCamera(ctypes.Structure):
    _fields_ = [
        ("W", ctypes.c_int32), ("H", ctypes.c_int32),
        ("K", ctypes.c_float * 9), ("Kinv", ctypes.c_float * 9),
        ("cx", ctypes.c_float), ("cy", ctypes.c_float),
        ("inv_half_w", ctypes.c_float), ("inv_half_h", ctypes.c_float),
        ("fx", ctypes.c_float), ("fy", ctypes.c_float),
    ]


class VidcImage(ctypes.Structure):
    _fields_ = [
        ("data", ctypes.c_void_p),
        ("n", ctypes.c_int32), ("c", ctypes.c_int32), ("h", ctypes.c_int32), ("w", ctypes.c_int32),
        ("sn", ctypes.c_int64), ("sc", ctypes.c_int64), ("sh", ctypes.c_int64), ("sw", ctypes.c_int64),
    ]


FRAME_PARAMS_FLOATS = 48  # sizeof(vidc_frame_params) / 4

_P = ctypes.POINTER
_SIGNATURES = {
    "vidc_abi_version": (ctypes.c_int, []),
    "vidc_last_error": (ctypes.c_char_p, []),
    "vidc_launch_count": (ctypes.c_uint64, []),
    "vidc_workspace_bytes": (ctypes.c_size_t, [_P(VidcCamera), ctypes.c_int32]),
    "vidc_camera_init": (ctypes.c_int, [ctypes.c_double] * 4 + [_P(VidcCamera)]),
    "vidc_frame_params_compute": (ctypes.c_int, [_P(VidcCamera), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]),
    "vidc_build_homography": (ctypes.c_int, [_P(VidcCamera), c_f32p, c_f32p, ctypes.c_int32, c_f32p, c_f32p, c_f32p, ctypes.c_void_p]),
    "vidc_warp_forward": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int,
                                         ctypes.c_void_p, c_f32p, _P(VidcImage), ctypes.c_void_p]),
    "vidc_warp_rgbd": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), _P(VidcImage), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int,
                                      ctypes.c_void_p, c_f32p, _P(VidcImage), _P(VidcImage), ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p]),
    "vidc_warp_rgbd_u8": (ctypes.c_int, [_P(VidcCamera), ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P(VidcImage),
                                         c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int, ctypes.c_void_p, c_f32p, _P(VidcImage),
                                         _P(VidcImage), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "vidc_warp_rgbd_packed": (ctypes.c_int, [_P(VidcCamera), c_f32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, c_f32p, c_f32p,
                                             ctypes.c_int32, ctypes.c_int, ctypes.c_void_p, c_f32p, c_f32p, ctypes.c_void_p,
                                             ctypes.c_void_p, ctypes.c_void_p]),
    "vidc_unwarp_normals": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int32,
                                           ctypes.c_void_p, c_f32p, _P(VidcImage), ctypes.c_void_p, ctypes.c_void_p]),
    "vidc_warp_backward": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int,
                                          ctypes.c_void_p, c_f32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]),
    "vidc_warp_backward_ordered": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int32,
                                                  ctypes.c_int, ctypes.c_void_p, c_f32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]),
    "vidc_warp_backward_params_scratch_bytes": (ctypes.c_size_t, [_P(VidcCamera), ctypes.c_int32]),
    "vidc_warp_backward_params": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), _P(VidcImage), c_f32p, c_f32p, ctypes.c_int32,
                                                 ctypes.c_int32, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                 ctypes.c_void_p]),
    "vidc_frame_params_backward": (ctypes.c_int, [_P(VidcCamera), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_void_p, c_f32p, c_f32p,
                                                  c_f32p, ctypes.c_void_p]),
    "vidc_sampler_forward_inverse":(ctypes.c_int, [_P(VidcCamera), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_void_p, c_f32p,
                                                    c_f32p, c_f32p, ctypes.c_void_p]),
    "vidc_warp_normals_forward": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int,
                                                 ctypes.c_void_p, c_f32p, _P(VidcImage), ctypes.c_void_p]),
    "vidc_warp_with_homography": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), c_f32p, ctypes.c_int32, ctypes.c_void_p,
                                                 _P(VidcImage), ctypes.c_void_p]),
    "vidc_validity_mask": (ctypes.c_int, [_P(VidcImage), ctypes.c_void_p, c_f32p, ctypes.c_void_p, ctypes.c_void_p]),
    "vidc_mask_nearest": (ctypes.c_int, [c_f32p] + [ctypes.c_int32] * 5 + [c_f32p, ctypes.c_void_p]),
    "vidc_mask_pyramid": (ctypes.c_int, [ctypes.c_void_p, c_f32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                         ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p]),
    "vidc_normalize3": (ctypes.c_int, [_P(VidcImage), _P(VidcImage), ctypes.c_void_p]),
    "vidc_normal_stats": (ctypes.c_int, [_P(VidcImage), _P(VidcImage), _P(VidcImage), ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]),
    "vidc_normal_loss_backward": (ctypes.c_int, [_P(VidcImage), _P(VidcImage), _P(VidcImage), ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                                 _P(VidcImage), ctypes.c_void_p]),
    "vidc_warp_unwarp_host": (ctypes.c_int, [_P(VidcCamera), ctypes.c_int32] + [ctypes.c_void_p] * 10),
    "vidc_release_workspace": (ctypes.c_int, []),
    "vidc_frame_params_prepare": (ctypes.c_int, [_P(VidcCamera), c_f32p, c_f32p, ctypes.c_int32, ctypes.c_void_p, c_f32p, ctypes.c_void_p]),
    "vidc_to_tensor_u8": (ctypes.c_int, [ctypes.c_void_p] + [ctypes.c_int32] * 4 + [c_f32p, ctypes.c_void_p]),
    "vidc_warp_unwarp_host_u8": (ctypes.c_int, [_P(VidcCamera), ctypes.c_int32] + [ctypes.c_void_p] * 10),
    "vidc_condition_gravity": (ctypes.c_int, [c_f32p, ctypes.c_int32, ctypes.c_int32, c_f32p, c_f32p, ctypes.c_void_p]),
    "vidc_rasterize_sparse_depth": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32] + [ctypes.c_double] * 4 +
                                    [ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, c_f32p, ctypes.c_void_p]),
    "vidc_warp_rgb_sparse_depth": (ctypes.c_int, [_P(VidcCamera), _P(VidcImage), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32] +
                                   [ctypes.c_double] * 4 + [c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int, ctypes.c_void_p, c_f32p,
                                                            _P(VidcImage), _P(VidcImage), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "vidc_debug_div": (ctypes.c_int, [c_f32p, c_f32p, c_f32p, ctypes.c_int64, c_f32p, ctypes.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib():
    """The loaded C-ABI library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension is the product and there is no fallback. "
                "Build it with `python -m vi_depth_completion_b200.build` (needs nvcc).")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if l.vidc_abi_version() != 3:
            raise RuntimeError(f"libvidc_b200.so ABI version {l.vidc_abi_version()} != 3; rebuild it")
        _lib = l
    return _lib


def check(rc: int):
    """Map a vidc_status to the exception the reference would raise at the same place."""
    if rc == VIDC_OK:
        return
    msg = lib().vidc_last_error().decode("utf-8", "replace")
    if rc == VIDC_ERR_BATCH_MISMATCH:
        raise AssertionError(msg)         # reference: `assert x.shape[0] == I_g.shape[0]`
    raise RuntimeError(f"vidc_b200: {msg} (status {rc})")
