"""ctypes binding of ``libgsb200.so`` (the C ABI declared in ``include/gsb200.h``).

The product path has NO fallback: if the shared library is missing or fails to load this module
raises, and every wrapper raises ``RuntimeError`` with ``gsb200_last_error()`` on a non-zero return.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GSB200_LIB_PATH", os.path.join(_HERE, "libgsb200.so"))  # override: tuning experiments only

GSB_FLAG_EXACT_EXP = 1
GSB_FLAG_FORCE_KEY64 = 2
GSB_FLAG_Q_ALREADY_NORMALISED = 4
GSB_FLAG_KEEP_ALL_TILE_PAIRS = 8
GSB_FLAG_BACKWARD_TRANSPOSED = 16  # experimental, csrc/blend_bwd_transposed.cu
GSB_FLAG_NO_HOOK_STATS = 32
GSB_FLAG_COMPACT_GRADS = 64

c_i64, c_i32, c_u32, c_f32, c_vp = (ctypes.c_int64, ctypes.c_int32, ctypes.c_uint32, ctypes.c_float,
                                    ctypes.c_void_p)


class GsbWorkspaceLayout(ctypes.Structure):
    _fields_ = [
        ("total_bytes", c_i64), ("zero_bytes", c_i64), ("counters", c_i64), ("tickets", c_i64),
        ("scan_state", c_i64), ("sort_hist", c_i64), ("sort_state", c_i64), ("tile_start", c_i64),
        ("tile_end", c_i64), ("poses", c_i64), ("point_id", c_i64), ("point_offset", c_i64), ("num_tiles", c_i64),
        ("records", c_i64), ("point_in_camera", c_i64), ("keys_a", c_i64), ("keys_b", c_i64),
        ("vals_a", c_i64), ("vals_b", c_i64), ("keys_c", c_i64), ("vals_c", c_i64), ("key_bytes", c_i32), ("tile_bits", c_i32),
        ("depth_bits", c_i32), ("sort_passes", c_i32), ("key_capacity_padded", c_i64),
        ("sort_blocks", c_i32), ("scan_blocks", c_i32), ("radix_bits", c_i32), ("reserved", c_i32),
    ]


class GsbForwardArgs(ctypes.Structure):
    _fields_ = [
        ("num_points", c_i64), ("pointcloud", c_vp), ("pointcloud_features", c_vp),
        ("point_invalid_mask", c_vp), ("point_object_id", c_vp), ("num_objects", c_i32),
        ("q_pointcloud_camera", c_vp), ("t_pointcloud_camera", c_vp), ("camera_intrinsics", c_vp),
        ("camera_height", c_i32), ("camera_width", c_i32), ("near_plane", c_f32), ("far_plane", c_f32),
        ("depth_to_sort_key_scale", c_f32), ("rgb_only", c_i32), ("flags", c_u32), ("workspace", c_vp),
        ("workspace_bytes", c_i64), ("key_capacity", c_i64), ("rasterized_image", c_vp),
        ("rasterized_depth", c_vp), ("pixel_accumulated_alpha", c_vp),
        ("pixel_offset_of_last_effective_point", c_vp), ("pixel_valid_point_count", c_vp),
        ("stream", c_vp), ("host_counters", c_vp), ("host_counters_event", c_vp),
    ]


class GsbBackwardArgs(ctypes.Structure):
    _fields_ = [
        ("num_points", c_i64), ("pointcloud", c_vp), ("pointcloud_features", c_vp),
        ("point_object_id", c_vp), ("num_objects", c_i32), ("t_pointcloud_camera", c_vp),
        ("camera_intrinsics", c_vp), ("camera_height", c_i32), ("camera_width", c_i32),
        ("far_plane", c_f32), ("depth_to_sort_key_scale", c_f32), ("color_max_sh_band", c_i32),
        ("grad_q_factor", c_f32), ("grad_s_factor", c_f32), ("grad_alpha_factor", c_f32),
        ("grad_color_factor", c_f32), ("grad_high_order_color_factor", c_f32), ("flags", c_u32),
        ("workspace", c_vp), ("workspace_bytes", c_i64), ("key_capacity", c_i64),
        ("grad_rasterized_image", c_vp), ("pixel_accumulated_alpha", c_vp),
        ("pixel_offset_of_last_effective_point", c_vp), ("accum", c_vp), ("accum_rows", c_i64),
        ("grad_pointcloud", c_vp), ("grad_pointcloud_features", c_vp),
        ("magnitude_grad_viewspace_on_image", c_vp), ("stream", c_vp),
        ("grad_sum_compact", c_vp), ("grad_color_compact", c_vp),
        ("ctl_accumulated_num_in_camera", c_vp), ("ctl_accumulated_num_pixels", c_vp),
        ("ctl_accumulated_view_space_position_gradients", c_vp), ("ctl_accumulated_view_space_position_gradients_avg", c_vp),
        ("ctl_accumulated_position_gradients", c_vp), ("ctl_accumulated_position_gradients_norm", c_vp),
    ]


class GsbMultimemExchangeArgs(ctypes.Structure):
    _fields_ = [
        ("num_points", c_i64), ("num_objects", c_i32), ("rank", c_i32), ("world_size", c_i32), ("num_blocks", c_i32),
        ("phases", c_i32), ("reserved", c_i32), ("multicast_grad_sum", c_vp), ("multicast_blocks", c_vp), ("local_block", c_vp), ("block_stride", c_i64), ("stream", c_vp),
    ]


class GsbTrainStepArgs(ctypes.Structure):
    _fields_ = [
        ("forward", GsbForwardArgs), ("backward", GsbBackwardArgs), ("ground_truth_image", c_vp), ("lambda_value", c_f32),
        ("loss_out3", c_vp), ("loss_temp", c_vp), ("loss_temp_bytes", c_i64), ("feature_exp_avg", c_vp),
        ("feature_exp_avg_sq", c_vp), ("position_exp_avg", c_vp), ("position_exp_avg_sq", c_vp),
        ("feature_learning_rate", ctypes.c_double), ("position_learning_rate", ctypes.c_double), ("beta1", ctypes.c_double),
        ("beta2", ctypes.c_double), ("eps", ctypes.c_double), ("step", c_i32),
    ]


class GsbExpandArgs(ctypes.Structure):
    _fields_ = [
        ("num_points", c_i64), ("num_views", c_i32), ("num_objects", c_i32), ("grad_sum", c_vp),
        ("grad_color_views", c_vp), ("view_stride", c_i64), ("pointcloud", c_vp), ("point_object_id", c_vp),
        ("color_max_sh_band", c_i32), ("grad_color_factor", c_f32), ("grad_high_order_color_factor", c_f32),
        ("part", c_i32), ("grad_pointcloud", c_vp), ("grad_pointcloud_features", c_vp), ("stream", c_vp),
    ]


class GsbPoseGradArgs(ctypes.Structure):
    _fields_ = [
        ("q_pointcloud_camera", c_vp), ("t_pointcloud_camera", c_vp), ("grad_q_pointcloud_camera", c_vp),
        ("grad_t_pointcloud_camera", c_vp), ("temp", c_vp), ("temp_bytes", c_i64),
    ]


GSB_POSE_MAX_OBJECTS = 16

EXPORTS = (
    "gsb200_version", "gsb200_last_error", "gsb200_workspace_layout", "gsb200_forward",
    "gsb200_backward", "gsb200_stage_preprocess", "gsb200_stage_sort", "gsb200_stage_tile_ranges",
    "gsb200_stage_blend", "gsb200_sort_temp_bytes", "gsb200_sort_pairs", "gsb200_render_host", "gsb200_find_tile_start_and_end",
    "gsb200_forward_timed", "gsb200_backward_timed", "gsb200_abi_sizes", "gsb200_l1_loss_temp_bytes", "gsb200_l1_loss",
    "gsb200_image_loss_temp_bytes", "gsb200_image_loss", "gsb200_adam_step", "gsb200_controller_update",
    "gsb200_forward_blend_work", "gsb200_backward_blend_work", "gsb200_device_selftest", "gsb200_expand_view_gradients",
    "gsb200_train_step", "gsb200_abi_sizes_ext", "gsb200_exchange_multimem", "gsb200_pose_grad_temp_bytes",
    "gsb200_backward_with_pose",
)

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (building it is ``__graft_entry__.build()``'s job, never implicit)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m taichi_3d_gaussian_splatting_b200.build` "
            "(there is no CPU / PyTorch fallback for the rasteriser)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.gsb200_version.restype = ctypes.c_int
    lib.gsb200_last_error.restype = ctypes.c_char_p
    lib.gsb200_workspace_layout.argtypes = [c_i64, c_i32, c_i64, c_i32, c_i32, c_f32, c_f32, c_u32,
                                            ctypes.POINTER(GsbWorkspaceLayout)]
    for name in ("gsb200_forward", "gsb200_stage_preprocess", "gsb200_stage_sort",
                 "gsb200_stage_tile_ranges", "gsb200_stage_blend"):
        getattr(lib, name).argtypes = [ctypes.POINTER(GsbForwardArgs)]
        getattr(lib, name).restype = ctypes.c_int
    lib.gsb200_backward.argtypes = [ctypes.POINTER(GsbBackwardArgs)]
    lib.gsb200_backward.restype = ctypes.c_int
    has_pose = hasattr(lib, "gsb200_backward_with_pose")  # the pose gradients are detected by their symbol
    if has_pose:
        lib.gsb200_backward_with_pose.argtypes = [ctypes.POINTER(GsbBackwardArgs), ctypes.POINTER(GsbPoseGradArgs)]
        lib.gsb200_backward_with_pose.restype = ctypes.c_int
        lib.gsb200_pose_grad_temp_bytes.argtypes = [c_i32]
        lib.gsb200_pose_grad_temp_bytes.restype = c_i64
    lib.gsb200_sort_temp_bytes.argtypes = [c_i64, c_i32]
    lib.gsb200_sort_temp_bytes.restype = c_i64
    lib.gsb200_sort_pairs.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_vp, c_i64, c_vp]
    lib.gsb200_sort_pairs.restype = ctypes.c_int
    lib.gsb200_render_host.argtypes = [ctypes.POINTER(GsbForwardArgs), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.gsb200_render_host.restype = ctypes.c_int
    lib.gsb200_l1_loss_temp_bytes.argtypes = []
    lib.gsb200_l1_loss_temp_bytes.restype = c_i64
    lib.gsb200_l1_loss.argtypes = [c_vp, c_vp, c_i64, c_i32, c_f32, c_vp, c_vp, c_vp, c_i64, c_vp]
    lib.gsb200_l1_loss.restype = ctypes.c_int
    lib.gsb200_image_loss_temp_bytes.argtypes = [c_i32, c_i32]
    lib.gsb200_image_loss_temp_bytes.restype = c_i64
    lib.gsb200_image_loss.argtypes = [c_vp, c_vp, c_i32, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_i64, c_vp]
    lib.gsb200_image_loss.restype = ctypes.c_int
    lib.gsb200_adam_step.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                     ctypes.c_double, c_i32, c_vp]
    lib.gsb200_adam_step.restype = ctypes.c_int
    lib.gsb200_controller_update.argtypes = [c_vp, c_i64] + [c_vp] * 10
    lib.gsb200_controller_update.restype = ctypes.c_int
    lib.gsb200_forward_blend_work.argtypes = [ctypes.POINTER(GsbForwardArgs), ctypes.POINTER(ctypes.c_uint64)]
    lib.gsb200_forward_blend_work.restype = ctypes.c_int
    lib.gsb200_backward_blend_work.argtypes = [ctypes.POINTER(GsbBackwardArgs), ctypes.POINTER(ctypes.c_uint64)]
    lib.gsb200_backward_blend_work.restype = ctypes.c_int
    lib.gsb200_expand_view_gradients.argtypes = [ctypes.POINTER(GsbExpandArgs)]
    lib.gsb200_expand_view_gradients.restype = ctypes.c_int
    lib.gsb200_exchange_multimem.argtypes = [ctypes.POINTER(GsbMultimemExchangeArgs)]
    lib.gsb200_exchange_multimem.restype = ctypes.c_int
    lib.gsb200_train_step.argtypes = [ctypes.POINTER(GsbTrainStepArgs)]
    lib.gsb200_train_step.restype = ctypes.c_int
    lib.gsb200_device_selftest.argtypes = [c_vp]
    lib.gsb200_device_selftest.restype = ctypes.c_int
    sizes = (c_i64 * 3)()
    lib.gsb200_abi_sizes(sizes)
    mine = (ctypes.sizeof(GsbWorkspaceLayout), ctypes.sizeof(GsbForwardArgs), ctypes.sizeof(GsbBackwardArgs))
    if tuple(sizes) != mine:
        raise RuntimeError(f"libgsb200.so ABI mismatch: C struct sizes {tuple(sizes)} != ctypes mirrors {mine}; "
                           "rebuild with `python -m taichi_3d_gaussian_splatting_b200.build --force`")
    n_ext = 6 if has_pose else 5
    sizes_ext = (c_i64 * n_ext)()
    lib.gsb200_abi_sizes_ext(sizes_ext, n_ext)
    mine_ext = (mine + (ctypes.sizeof(GsbExpandArgs), ctypes.sizeof(GsbTrainStepArgs), ctypes.sizeof(GsbPoseGradArgs)))[:n_ext]
    if tuple(sizes_ext) != mine_ext:
        raise RuntimeError(f"libgsb200.so ABI mismatch: C struct sizes {tuple(sizes_ext)} != ctypes mirrors {mine_ext}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().gsb200_last_error()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def workspace_layout(num_points: int, num_objects: int, key_capacity: int, height: int, width: int,
                     far_plane: float, depth_scale: float, flags: int = 0) -> GsbWorkspaceLayout:
    out = GsbWorkspaceLayout()
    check(load().gsb200_workspace_layout(num_points, num_objects, key_capacity, height, width,
                                         far_plane, depth_scale, flags, ctypes.byref(out)),
          "gsb200_workspace_layout")
    return out
