"""ctypes binding of libc3d.so (C ABI declared in include/c3d.h).  No torch types cross it."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# C3D_LIB_PATH: developer override (the lab build libc3d_lab.so of csrc/Makefile `make lab`); never a fallback
LIB_PATH = os.environ.get("C3D_LIB_PATH") or os.path.join(_HERE, "libc3d.so")
_lib = None

C3D_OK, C3D_EINVAL, C3D_EWORKSPACE, C3D_ECUDA = 0, -1, -2, -3


class C3DError(RuntimeError):
    pass


def _sig(lib, name, restype, argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = argtypes
    return fn


def lib():
    """Load libc3d.so or raise — the product path has no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise C3DError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C omni3d_b200/csrc). omni3d_b200 has no CPU / library fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, i64, i32, f32, sz = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_size_t
    _sig(L, "c3d_last_error", ctypes.c_char_p, [])
    _sig(L, "c3d_abi_version", i32, [])
    _sig(L, "c3d_iou_box3d_workspace_bytes", sz, [i64, i64])
    _sig(L, "c3d_iou_box3d", i32, [vp, i64, vp, i64, vp, vp, vp, vp, sz, vp])
    _sig(L, "c3d_iou_box3d_paired", i32, [vp, vp, i64, vp, vp, vp, vp, sz, vp])
    _sig(L, "c3d_box3d_overlap", i32, [vp, i64, vp, i64, f32, f32, vp, vp, vp, sz, vp])
    _lib = L
    return L


# number of libc3d kernel launches issued through the python front-ends (bench.py's gpu_launches)
LAUNCHES = {"n": 0}


def check(code, launches=1):
    LAUNCHES["n"] += launches
    if code != C3D_OK:
        raise C3DError(f"libc3d error {code}: {lib().c3d_last_error().decode()}")


# every symbol include/c3d.h declares (tests/test_abi.py checks the .so exports each one)
EXPORTS = [
    "c3d_last_error", "c3d_abi_version", "c3d_iou_box3d_workspace_bytes", "c3d_iou_box3d",
    "c3d_iou_box3d_paired", "c3d_box3d_overlap", "c3d_conv2d_tiles", "c3d_conv2d_fwd", "c3d_conv2d_wgrad", "c3d_conv2d_wgrad_ex", "c3d_pack_conv_weight",
    "c3d_bn_scratch_bytes", "c3d_bn_finalize", "c3d_bn_apply", "c3d_bn_bwd_blocks", "c3d_bn_bwd", "c3d_maxpool2_fwd", "c3d_maxpool2_bwd", "c3d_maxpool2_bwd_acc",
    "c3d_preprocess_image", "c3d_grad_finite", "c3d_sgd_momentum", "c3d_roi_align_fwd", "c3d_roi_align_bwd",
    "c3d_nms_workspace_bytes", "c3d_nms_batched", "c3d_bias_act_bwd", "c3d_sumpool2", "c3d_zero_stuff2", "c3d_cube_loss_fwd", "c3d_cube_loss_bwd",
    "c3d_anchor_match", "c3d_preprocess_image_u8", "c3d_sgd_momentum_dev", "c3d_rpn_loss_fwd", "c3d_rpn_loss_bwd", "c3d_nms_batched_grouped", "c3d_rpn_decode_level",
    "c3d_maxpool3s2_fwd", "c3d_maxpool3s2_bwd",
    "c3d_pack_linear_weight", "c3d_linear_fwd", "c3d_linear_dgrad", "c3d_linear_wgrad",
    "c3d_box3d_overlap_segmented_workspace_bytes", "c3d_box3d_overlap_segmented",
    "c3d_topk_segments", "c3d_label_sample_proposals", "c3d_anchor_sample_keys", "c3d_anchor_sample_finish", "c3d_det_candidates",
    "c3d_box_loss_fwd", "c3d_box_loss_bwd", "c3d_cube_gather", "c3d_cube_reduce_fwd", "c3d_cube_reduce_bwd", "c3d_cube_scatter",
    "c3d_linear_fwd_blocks", "c3d_linear_dgrad_blocks", "c3d_linear_wgrad_blocks", "c3d_resize_bilinear_u8", "c3d_preprocess_batch", "c3d_pack_conv_weights_batched",
    "c3d_eval_match_workspace_bytes", "c3d_eval_match", "c3d_eval_accumulate",
]
