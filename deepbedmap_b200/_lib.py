"""ctypes binding of libdeepbedmap_b200.so (the C ABI declared in include/deepbedmap_b200.h).

There is no CPU fallback: if the CUDA library is missing or fails to load, every product entry
point raises immediately.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# DEEPBEDMAP_B200_LIB: another build of the same library (A/B timing of two builds on one box, scripts/)
LIB_PATH = os.environ.get("DEEPBEDMAP_B200_LIB") or os.path.join(_HERE, "libdeepbedmap_b200.so")

_P, _L, _I, _F = ctypes.c_void_p, ctypes.c_long, ctypes.c_int, ctypes.c_float

# name -> argument ctypes, in the order of include/deepbedmap_b200.h
SIGNATURES = {
    "dbm_version": [],
    "dbm_launch_count": [],
    "dbm_set_sm_reserve": [_I],
    "dbm_set_deterministic": [_I],
    "dbm_conv2d_fwd_f32": [_P, _L, _P, _P, _P, _L, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "dbm_conv2d_bwd_data_f32": [_P, _L, _P, _P, _L, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "dbm_conv2d_bwd_weight_f32": [_P, _L, _P, _L, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "dbm_bias_grad_f32": [_P, _L, _P, _I, _I, _I, _P],
    "dbm_gemm_f32": [_P, _L, _L, _L, _P, _L, _L, _L, _P, _L, _L, _L, _P, _I, _I, _I, _I, _I, _I, _P],
    "dbm_gemm_bf16": [_P, _L, _L, _L, _P, _L, _L, _L, _P, _L, _L, _L, _P, _I, _I, _I, _I, _I, _I, _P],
    "dbm_axpby_f32": [_P, _L, _P, _L, _P, _L, _F, _F, _I, _L, _P],
    "dbm_lrelu_fwd_f32": [_P, _P, _L, _P],
    "dbm_lrelu_bwd_f32": [_P, _L, _P, _L, _P, _L, _I, _L, _I, _P],
    "dbm_upsample2_fwd_f32": [_P, _P, _L, _I, _I, _P],
    "dbm_upsample2_bwd_f32": [_P, _P, _L, _I, _I, _P],
    "dbm_fill_f32": [_P, _F, _L, _P],
    "dbm_nchw_to_slab8": [_P, _L, _P, _I, _I, _I, _I, _I, _I, _P],
    "dbm_slab8_to_nchw": [_P, _I, _I, _P, _L, _I, _I, _I, _I, _P],
    "dbm_nchw_to_slab4": [_P, _L, _P, _I, _I, _I, _I, _P],
    "dbm_slab4_to_nchw": [_P, _P, _L, _I, _I, _I, _I, _I, _P],
    "dbm_pack_conv3x3_weights": [_P, _P, _I, _I, _I, _I, _P],
    "dbm_pack_conv3x3_weights_slice": [_P, _I, _I, _P, _I, _I, _I, _I, _I, _P],
    "dbm_pack_conv3x3_table": [_P, _I, _L, _P],
    "dbm_trunk_umma": [_P, _I, _I, _I, _I, _P, _I, _P, _P, _I, _P, _P],
    "dbm_trunk_umma_split": [_P, _I, _I, _I, _I, _P, _I, _P, _P, _I, _P, _P],
    "dbm_nchw_to_slab8_split": [_P, _L, _P, _I, _I, _I, _I, _P],
    "dbm_slab8f_to_nchw": [_P, _P, _L, _I, _I, _I, _I, _P],
    "dbm_flat_geometry": [_I, _I, _I, _P],
    "dbm_flat_conv3x3_seq": [_P, _I, _I, _I, _I, _I, _I, _P],
    "dbm_flat_conv3x3_chain": [_P, _P, _I, _I, _I, _I, _I, _I, _P, _P],
    "dbm_trunk_local_fwd": [_P, _I, _I, _I, _I, _P, _P, _P, _P],
    "dbm_trunk_local_bwd": [_P, _I, _I, _I, _I, _P, _P, _P],
    "dbm_flat_wgrad": [_P, _I, _I, _I, _I, _P],
    "dbm_flat_wgrad_ctas": [_P, _I, _I, _I, _I, _I, _P],
    "dbm_flat_wgrad_reduce": [_P, _I, _P],
    "dbm_flat_bias_grad": [_P, _I, _I, _I, _I, _P],
    "dbm_flat_from_nchw": [_P, _I, _P, _P, _F, _I, _I, _I, _P],
    "dbm_flat_to_nchw": [_P, _P, _P, _I, _I, _I, _I, _P],
    "dbm_flat_from_nchw_ex": [_P, _I, _I, _I, _I, _P, _P, _F, _I, _I, _I, _P],
    "dbm_flat_to_nchw_ex": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "dbm_transpose_f32": [_P, _P, _I, _I, _P],
    "dbm_stem_fwd_slab8": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dbm_stem_w1_s2d": [_P, _P, _I, _I, _I, _P],
    "dbm_pack_stem_w1": [_P, _P, _P],
    "dbm_conv3x3_umma_valid": [_P, _I, _I, _P, _P, _I, _I, _I, _P, _I, _I, _P],
    "dbm_stem_fwd_flat": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "dbm_deform_conv_umma": [_P, _P, _I, _P, _P, _I, _I, _I, _I, _P, _I, _I, _P, _P, _P],
    "dbm_deform_conv_umma_nchw": [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P],
    "dbm_deform_sample_slab8_f32": [_P, _P, _P, _I, _I, _I, _P],
    "dbm_deform_out1_sample": [_P, _P, _I, _P, _P, _I, _I, _I, _P],
    "dbm_deform_conv_out1": [_P, _P, _I, _P, _P, _P, _P, _I, _I, _I, _P],
    "dbm_conv3x3_umma": [_P, _I, _I, _P, _P, _I, _I, _I, _I, _F, _I, _I, _P, _I, _I, _P, _I, _I, _P, _P, _P],
    "dbm_deform_sample_f32": [_P, _P, _P, _I, _I, _I, _I, _P],
    "dbm_deform_bwd_f32": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dbm_deform1_fwd_f32": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dbm_deform1_bwd_f32": [_P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P],
    "dbm_bn_lrelu_fwd_f32": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _F, _I, _P],
    "dbm_bn_lrelu_bwd_f32": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "dbm_bn_lrelu_fwd_groups_f32": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _F, _I, _P],
    "dbm_bn_lrelu_bwd_groups_f32": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dbm_ragan_loss_f32": [_P, _P, _I, _F, _F, _F, _P, _P, _P, _P],
    "dbm_gen_image_loss_f32": [_P, _P, _P, _I, _I, _I, _F, _F, _F, _P, _P, _P],
    "dbm_adam_step_f32": [_P, _P, _P, _P, _L, _F, _F, _F, _F, _I, _F, _P],
    "dbm_adam_step_dev_f32": [_P, _P, _P, _P, _L, _F, _F, _F, _F, _P, _F, _P],
    "dbm_crop_clip_f32": [_P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P],
    "dbm_place_tile_f32": [_P, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P],
    "dbm_f32_to_i16": [_P, _P, _L, _P],
    "dbm_copy2d_async": [_P, ctypes.c_size_t, _P, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, _P],
    "dbm_gather_rows_f32": [_P, _L, _P, _P, _L, _I, _P],
    # model-level entry points (handles are opaque pointers)
    "dbm_gen_create": [_I, _F, _I, ctypes.POINTER(_P)],
    "dbm_gen_destroy": [_P],
    "dbm_gen_count_params": [_P],
    "dbm_gen_num_arrays": [_P],
    "dbm_gen_array_info": [_P, _I, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(_I), ctypes.POINTER(_I),
                           ctypes.POINTER(_L)],
    "dbm_gen_set_param": [_P, ctypes.c_char_p, _P, _I, ctypes.POINTER(_I)],
    "dbm_gen_bind_params": [_P, _P],
    "dbm_gen_mark_updated": [_P],
    "dbm_gen_set_precision": [_P, _I],
    "dbm_gen_workspace_bytes": [_P, _I, _I, _I],
    "dbm_gen_forward": [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P, ctypes.c_size_t, _P],
    "dbm_disc_create": [ctypes.POINTER(_P)],
    "dbm_disc_destroy": [_P],
    "dbm_disc_set_precision": [_P, _I],
    "dbm_disc_count_params": [_P],
    "dbm_disc_num_arrays": [_P],
    "dbm_disc_array_info": [_P, _I, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(_I), ctypes.POINTER(_I),
                            ctypes.POINTER(_L)],
    "dbm_disc_set_param": [_P, ctypes.c_char_p, _P, _I, ctypes.POINTER(_I)],
    "dbm_disc_get_param": [_P, ctypes.c_char_p, _P],
    "dbm_disc_bind_params": [_P, _P],
    "dbm_disc_bind_grads": [_P, _P],
    "dbm_disc_mark_updated": [_P],
    "dbm_disc_zero_grads": [_P, _P],
    "dbm_disc_workspace_bytes": [_P, _I],
    "dbm_disc_forward": [_P, _P, _I, _I, _I, _I, _P, _P, ctypes.c_size_t, _P],
    "dbm_disc_backward": [_P, _P, _P, ctypes.c_size_t, _P],
}
# tuning / A-B switches (include/deepbedmap_b200_tuning.h): exported by the same library, not part of the boundary
TUNING_SIGNATURES = {
    "dbm_debug_set": [_I, _I],
    "dbm_debug_set_ptr": [_I, _P],
    "dbm_flat_debug_set": [_I, _I],
    "dbm_local_debug_set": [_I],
}
# entry points that return a value instead of a status
RESTYPES = {"dbm_launch_count": _L, "dbm_gen_count_params": _L, "dbm_gen_num_arrays": _I, "dbm_gen_workspace_bytes": ctypes.c_size_t,
            "dbm_disc_count_params": _L, "dbm_disc_num_arrays": _I, "dbm_disc_workspace_bytes": ctypes.c_size_t}

_lib: Optional[ctypes.CDLL] = None
launch_count = 0  # number of library calls that enqueue kernels (bench.py reports it)


class DeepBedMapError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load the shared library; raises loudly when it is missing (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DeepBedMapError(
            f"{LIB_PATH} is missing: build it with `python -m deepbedmap_b200.build` "
            "(nvcc, sm_100a). deepbedmap_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.dbm_last_error.restype = ctypes.c_char_p
    lib.dbm_last_error.argtypes = []
    for name, args in list(SIGNATURES.items()) + list(TUNING_SIGNATURES.items()):
        try:
            fn = getattr(lib, name)  # AttributeError if the library does not export it
        except AttributeError:
            if os.environ.get("DEEPBEDMAP_B200_LIB"):   # an older build under A/B test may lack newer entry points
                continue
            raise
        fn.argtypes = args
        fn.restype = RESTYPES.get(name, ctypes.c_int)
    _lib = lib
    return lib


def kernel_launches() -> int:
    """Kernels launched by the library so far (counted inside the library, one per launch)."""
    return int(load().dbm_launch_count())


def call(name: str, *args) -> None:
    """Invoke a C-ABI entry point; non-zero status -> ValueError (bad arguments, mirroring the
    reference's shape/type errors) or DeepBedMapError (CUDA failure)."""
    global launch_count
    lib = load()
    rc = getattr(lib, name)(*args)
    launch_count += 1
    if rc != 0:
        msg = lib.dbm_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"{name}: {msg}")
        raise DeepBedMapError(f"{name}: {msg}")
