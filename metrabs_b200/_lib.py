"""ctypes binding of libmetrabs_b200.so (include/metrabs_b200.h).  There is no CPU or eager fallback: if the
shared library is missing or cannot be loaded, importing the compute entry points raises."""
import ctypes as C
import os

MTB_ABI_VERSION = 1
MTB_MAX_STAGES = 16

ARCH_EFFNET, ARCH_RESNET50, ARCH_MOBILENETV3_SMALL, ARCH_HEAD_ONLY = 0, 1, 2, 3
PRECISION_FP32, PRECISION_BF16_TC, PRECISION_BF16_SIMT, PRECISION_TF32X3 = 0, 1, 2, 3
DTYPE_F32, DTYPE_BF16, DTYPE_F16, DTYPE_I64 = 0, 1, 2, 3
LAYOUT_BDJHW, LAYOUT_BHWN = 0, 1

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'libmetrabs_b200.so')


class MtbStage(C.Structure):
    _fields_ = [('block', C.c_int32), ('expand', C.c_int32), ('kernel', C.c_int32), ('stride', C.c_int32),
                ('cin', C.c_int32), ('cout', C.c_int32), ('layers', C.c_int32), ('bottomright', C.c_int32)]


class MtbConfig(C.Structure):
    _fields_ = [('abi_version', C.c_int32), ('arch', C.c_int32), ('precision', C.c_int32), ('device', C.c_int32),
                ('proc_side', C.c_int32), ('stride_train', C.c_int32), ('stride_test', C.c_int32),
                ('centered_stride', C.c_int32), ('legacy_centered_stride_bug', C.c_int32),
                ('depth', C.c_int32), ('n_joints', C.c_int32), ('feature_channels', C.c_int32),
                ('box_size_mm', C.c_float), ('mix_3d_inside_fov', C.c_float), ('weak_perspective', C.c_int32),
                ('n_stages', C.c_int32), ('last_channel', C.c_int32), ('stages', MtbStage * MTB_MAX_STAGES)]


class MtbCropSetupArgs(C.Structure):
    _fields_ = [('boxes', C.c_void_p), ('box_stride', C.c_int32), ('intrinsics', C.c_void_p), ('distortion', C.c_void_p),
                ('n_dist', C.c_int32), ('camspace_up', C.c_void_p), ('aug_rotflipmat', C.c_void_p), ('aug_scales', C.c_void_p),
                ('n_boxes', C.c_int32), ('num_aug', C.c_int32), ('resolution', C.c_int32), ('antialias_factor', C.c_int32),
                ('new_intrinsics', C.c_void_p), ('rotations', C.c_void_p), ('inv_projections', C.c_void_p),
                ('pyramid_levels', C.c_void_p)]


class MtbWarpArgs(C.Structure):
    _fields_ = [('images', C.c_void_p), ('level1', C.c_void_p), ('level2', C.c_void_p), ('n_images', C.c_int32),
                ('height', C.c_int32), ('width', C.c_int32), ('intrinsics', C.c_void_p), ('distortion', C.c_void_p),
                ('n_dist', C.c_int32), ('image_ids', C.c_void_p), ('inv_projections', C.c_void_p),
                ('pyramid_levels', C.c_void_p), ('gamma_exponents', C.c_void_p), ('n_boxes', C.c_int32),
                ('num_aug', C.c_int32), ('resolution', C.c_int32), ('antialias_factor', C.c_int32), ('crops', C.c_void_p)]


class MtbTtaArgs(C.Structure):
    _fields_ = [('poses', C.c_void_p), ('rotations', C.c_void_p), ('aug_should_flip', C.c_void_p),
                ('mirror_mapping', C.c_void_p), ('joint_transform', C.c_void_p), ('skeleton', C.c_void_p),
                ('intrinsics', C.c_void_p), ('distortion', C.c_void_p), ('n_dist', C.c_int32),
                ('extrinsics_inv', C.c_void_p), ('n_boxes', C.c_int32), ('num_aug', C.c_int32), ('n_joints', C.c_int32),
                ('n_joints_transformed', C.c_int32), ('n_skeleton', C.c_int32), ('average_aug', C.c_int32),
                ('poses3d', C.c_void_p), ('poses2d', C.c_void_p)]


class MtbFilterArgs(C.Structure):
    _fields_ = [('poses3d', C.c_void_p), ('poses2d', C.c_void_p), ('boxes', C.c_void_p), ('box_stride', C.c_int32),
                ('bones', C.c_void_p), ('mean_bones', C.c_void_p), ('n_bones', C.c_int32), ('image_start', C.c_void_p),
                ('n_images', C.c_int32), ('n_boxes', C.c_int32), ('num_aug', C.c_int32), ('n_joints', C.c_int32),
                ('plausible', C.c_void_p), ('keep', C.c_void_p), ('scratch', C.c_void_p)]


class MetrabsB200Error(RuntimeError):
    pass


_SIGNATURES = {
    'mtb_create': (C.c_int, [C.POINTER(MtbConfig), C.POINTER(C.c_void_p)]),
    'mtb_destroy': (C.c_int, [C.c_void_p]),
    'mtb_last_error': (C.c_char_p, [C.c_void_p]),
    'mtb_version': (C.c_char_p, []),
    'mtb_load_weight': (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.c_int]),
    'mtb_finalize_weights': (C.c_int, [C.c_void_p]),
    'mtb_workspace_bytes': (C.c_size_t, [C.c_void_p, C.c_int]),
    'mtb_feature_shape': (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'mtb_backbone_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                       C.c_void_p]),
    'mtb_head_decode': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                  C.c_void_p]),
    'mtb_softargmax': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    'mtb_reconstruct_scratch_bytes': (C.c_size_t, [C.c_int]),
    'mtb_reconstruct_absolute': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    'mtb_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                              C.c_void_p]),
    'mtb_forward_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'mtb_forward_host_submit': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    'mtb_forward_host_wait': (C.c_int, [C.c_void_p, C.c_int]),
    'mtb_comm_unique_id': (C.c_int, [C.c_void_p]),
    'mtb_comm_init': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    'mtb_allgather_joints': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'mtb_sharded_scratch_bytes': (C.c_size_t, [C.c_void_p, C.c_int]),
    'mtb_forward_sharded': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_size_t, C.c_void_p]),
    'mtb_image_pyramid': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    'mtb_crop_setup': (C.c_int, [C.POINTER(MtbCropSetupArgs), C.c_void_p]),
    'mtb_warp_crops': (C.c_int, [C.POINTER(MtbWarpArgs), C.c_void_p]),
    'mtb_tta_merge': (C.c_int, [C.POINTER(MtbTtaArgs), C.c_void_p]),
    'mtb_filter_poses': (C.c_int, [C.POINTER(MtbFilterArgs), C.c_void_p]),
    'mtb_num_ops': (C.c_int, [C.c_void_p]),
    'mtb_op_name': (C.c_char_p, [C.c_void_p, C.c_int]),
    'mtb_debug_run_ops': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                    C.c_size_t, C.c_void_p]),
    'mtb_op_output_shape': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                      C.POINTER(C.c_int)]),
    'mtb_op_input_shape': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'mtb_debug_run_op': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    'mtb_op_is_fused_block': (C.c_int, [C.c_void_p, C.c_int]),
    'mtb_debug_run_fused_block': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                            C.c_size_t, C.c_void_p]),
    'mtb_op_is_expdw': (C.c_int, [C.c_void_p, C.c_int]),
    'mtb_debug_run_expdw': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                      C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    'mtb_profile_begin': (C.c_int, [C.c_void_p, C.c_uint]),
    'mtb_profile_end': (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                  C.POINTER(C.c_int64)]),
    'mtb_profile_op_times': (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                       C.POINTER(C.c_int), C.c_int]),
    'mtb_op_weight_bytes': (C.c_double, [C.c_void_p, C.c_int]),
    'mtb_num_kernel_classes': (C.c_int, []),
    'mtb_kernel_class_name': (C.c_char_p, [C.c_int]),
    'mtb_last_launch_count': (C.c_int64, [C.c_void_p]),
    'mtb_backbone_flops_per_crop': (C.c_double, [C.c_void_p]),
    'mtb_debug_dw_plan': (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                    C.POINTER(C.c_int)]),
    'mtb_debug_fmb_plan': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     C.POINTER(C.c_int)]),
    'mtb_debug_expdw_plan': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                       C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'mtb_debug_fmb_pack': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib():
    """Loads the shared library once; raises MetrabsB200Error when it is absent (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MetrabsB200Error(
                f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` or '
                f'metrabs_b200/csrc/build.sh. metrabs_b200 has no CPU/eager fallback.')
        handle = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def check(rc, handle=None):
    if rc != 0:
        msg = lib().mtb_last_error(handle)
        raise MetrabsB200Error(f'libmetrabs_b200 error {rc}: {msg.decode() if msg else "?"}')
