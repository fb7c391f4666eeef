"""Drop-in replacement of the reference operator ``GaussianPointCloudRasterisation``.

Same public surface as ``taichi_3d_gaussian_splatting/GaussianPointCloudRasterisation.py:775-1204``
of the reference: ``GaussianPointCloudRasterisation(config, backward_valid_point_hook)`` is an
``nn.Module`` whose ``forward(GaussianPointCloudRasterisationInput)`` returns
``(image (H,W,3) f32, depth (H,W) f32, pixel_valid_point_count (H,W) i32)`` and whose autograd
backward produces dense ``(N,3)`` / ``(N,56)`` gradients, scales them with the fixed factors,
and calls the ``BackwardValidPointHookInput`` side channel -- but every kernel is hand-written
sm_100a CUDA behind the C ABI of ``libgsb200.so`` (``include/gsb200.h``).  PyTorch is used only
for device memory, streams and autograd plumbing.  There is no CPU fallback.

Contract details kept from the reference (SURVEY.md §8(b), §9):
* in-frustum rows of ``point_cloud_features[:, 0:4]`` are normalised IN PLACE each forward
  (GPCR:264-266);
* backward does nothing (all ``None``) unless xyz, features or a pose requires grad (GPCR:1028);
* the pose gradients, which the reference declares and leaves ``None`` (GPCR:1027, 1157-1163), are filled
  (``gsb200_backward_with_pose``) when ``q_pointcloud_camera`` or ``t_pointcloud_camera`` requires grad -- the gradient of
  the same surrogate the xyz gradient follows (DESIGN.md §9); a pose-only backward does not call the hook;
* the hook runs synchronously inside backward, after gradient scaling (GPCR:1127-1142);
* ``grad_*_factor`` are un-annotated class constants, i.e. not dataclass fields (GPCR:782-786);
* ``camera_width`` / ``camera_height`` must be multiples of 16 (GPCR:1193-1194).
Defined where the reference leaves memory uninitialised: an empty frame (no splat reaches a tile)
renders zeros, and with ``rgb_only=True`` the auxiliary outputs are zeros.
"""
import ctypes
import os
import threading
from dataclasses import dataclass
from typing import Callable, Optional

import torch

from . import _lib
from .Camera import CameraInfo, CameraView  # noqa: F401  (re-exported like the reference module)

BOUNDARY_TILES = 3
TILE_WIDTH = 16
TILE_HEIGHT = 16

_RECORD_FLOATS = 12
_ACCUM_FLOATS = 12


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require(t: torch.Tensor, name: str, dtype: torch.dtype, shape_tail=None) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device: the B200 rasteriser has no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if shape_tail is not None and tuple(t.shape[1:]) != tuple(shape_tail):
        raise ValueError(f"{name} must have shape (*, {', '.join(map(str, shape_tail))}), got {tuple(t.shape)}")
    return t


class _PinnedCounters:
    """Per-device pool of (pinned int64[4] read-back buffer, CUDA event) pairs, one per frame in flight."""
    _free = {}
    _lock = threading.Lock()  # operators of several threads (one per stream) share the pool

    @classmethod
    def acquire(cls, device: torch.device):
        key = device.index if device.index is not None else torch.cuda.current_device()
        with cls._lock:
            pool = cls._free.setdefault(key, [])
            if pool:
                return pool.pop()
        event = torch.cuda.Event()
        event.record()  # materialises the underlying cudaEvent_t so that its handle can cross the C ABI
        return torch.zeros(4, dtype=torch.int64).pin_memory(), event

    @classmethod
    def release(cls, device: torch.device, item) -> None:
        key = device.index if device.index is not None else torch.cuda.current_device()
        with cls._lock:
            cls._free.setdefault(key, []).append(item)


class Frame:
    """Per-call state shared by forward and backward: the workspace blob and typed views into it.

    The views expose the intermediates that the reference keeps as separate saved tensors
    (GPCR:998-1019); tests read them to compare stage by stage against the oracle.
    """

    def __init__(self, ws: torch.Tensor, layout: _lib.GsbWorkspaceLayout, num_points: int,
                 key_capacity: int, height: int, width: int, flags: int):
        self.ws = ws
        self.layout = layout
        self.num_points = num_points
        self.key_capacity = key_capacity
        self.height = height
        self.width = width
        self.flags = flags
        self.num_points_in_camera: Optional[int] = None  # M
        self.num_keys: Optional[int] = None  # K

    def _view(self, offset: int, count: int, dtype: torch.dtype) -> torch.Tensor:
        nbytes = count * torch.empty((), dtype=dtype).element_size()
        return self.ws[offset:offset + nbytes].view(dtype)

    @property
    def counters(self) -> torch.Tensor:
        return self._view(self.layout.counters, 8, torch.int64)

    def _m(self) -> int:
        if self.num_points_in_camera is None:
            raise RuntimeError("frame counters have not been read back yet")
        return self.num_points_in_camera

    @property
    def point_id_in_camera_list(self) -> torch.Tensor:
        return self._view(self.layout.point_id, self.num_points, torch.int32)[:self._m()]

    @property
    def num_overlap_tiles(self) -> torch.Tensor:
        return self._view(self.layout.num_tiles, self.num_points, torch.int32)[:self._m()]

    @property
    def records(self) -> torch.Tensor:
        """(M, 12): u v a b | c rescale opacity depth | r g b radius."""
        return self._view(self.layout.records, self.num_points * _RECORD_FLOATS,
                          torch.float32).view(-1, _RECORD_FLOATS)[:self._m()]

    @property
    def point_in_camera(self) -> torch.Tensor:
        return self._view(self.layout.point_in_camera, self.num_points * 3, torch.float32).view(-1, 3)[:self._m()]

    @property
    def point_uv(self) -> torch.Tensor:
        return self.records[:, 0:2]

    @property
    def point_uv_conic_and_rescale(self) -> torch.Tensor:
        r = self.records
        return torch.stack([r[:, 2], r[:, 3], r[:, 4], r[:, 5]], dim=-1)

    @property
    def point_alpha_after_activation(self) -> torch.Tensor:
        return self.records[:, 6]

    @property
    def point_color(self) -> torch.Tensor:
        return self.records[:, 8:11]

    @property
    def point_radii(self) -> torch.Tensor:
        return self.records[:, 11]

    @property
    def sorted_keys(self) -> torch.Tensor:
        """Sorted packed keys (tile << depth_bits | depth), int64 regardless of the device key width."""
        off = self.layout.keys_b  # the sort always ends in b
        n = min(self.num_keys, self.key_capacity)
        if self.layout.key_bytes == 4:
            return self._view(off, self.layout.key_capacity_padded, torch.int32)[:n].to(torch.int64) & 0xFFFFFFFF
        return self._view(off, self.layout.key_capacity_padded, torch.int64)[:n]

    @property
    def point_offset_with_sort_key(self) -> torch.Tensor:
        off = self.layout.vals_b
        n = min(self.num_keys, self.key_capacity)
        return self._view(off, self.layout.key_capacity_padded, torch.int32)[:n]

    @property
    def tile_points_start(self) -> torch.Tensor:
        T = (self.height // TILE_HEIGHT) * (self.width // TILE_WIDTH)
        return self._view(self.layout.tile_start, T, torch.int32)

    @property
    def tile_points_end(self) -> torch.Tensor:
        T = (self.height // TILE_HEIGHT) * (self.width // TILE_WIDTH)
        return self._view(self.layout.tile_end, T, torch.int32)


class GaussianPointCloudRasterisation(torch.nn.Module):
    @dataclass
    class GaussianPointCloudRasterisationConfig:
        # reference: GPCR:776-786 (a dataclass_wizard YAMLWizard there; plain dataclass here)
        near_plane: float = 0.8
        far_plane: float = 1000.
        depth_to_sort_key_scale: float = 100.
        rgb_only: bool = False
        # un-annotated on purpose: class constants, not dataclass fields (GPCR:782-786)
        grad_color_factor = 5.
        grad_high_order_color_factor = 1.
        grad_s_factor = 0.5
        grad_q_factor = 1.
        grad_alpha_factor = 20.

    @dataclass
    class GaussianPointCloudRasterisationInput:
        # reference: GPCR:788-804
        point_cloud: torch.Tensor  # Nx3
        point_cloud_features: torch.Tensor  # Nx56
        point_object_id: torch.Tensor  # N, int32
        point_invalid_mask: torch.Tensor  # N, int8
        camera_info: CameraInfo
        q_pointcloud_camera: torch.Tensor  # Kx4 (x, y, z, w), camera -> pointcloud
        t_pointcloud_camera: torch.Tensor  # Kx3
        color_max_sh_band: int = 2

    @dataclass
    class BackwardValidPointHookInput:
        # reference: GPCR:806-817
        point_id_in_camera_list: torch.Tensor  # M
        grad_point_in_camera: torch.Tensor  # Mx3
        grad_pointfeatures_in_camera: torch.Tensor  # Mx56
        grad_viewspace: torch.Tensor  # Mx2
        magnitude_grad_viewspace: torch.Tensor  # M
        magnitude_grad_viewspace_on_image: torch.Tensor  # HxWx2
        num_overlap_tiles: torch.Tensor  # M
        num_affected_pixels: torch.Tensor  # M
        point_depth: torch.Tensor  # M
        point_uv_in_camera: torch.Tensor  # Mx2

    def __init__(
        self,
        config: "GaussianPointCloudRasterisation.GaussianPointCloudRasterisationConfig",
        backward_valid_point_hook: Optional[Callable[["GaussianPointCloudRasterisation.BackwardValidPointHookInput"], None]] = None,
        *,
        exact_exp: bool = False,
        force_key64: bool = False,
        initial_key_capacity: Optional[int] = None,
        keep_all_tile_pairs: bool = False,
        backward_impl: Optional[str] = None,
        skip_unused_hook_statistics: Optional[bool] = None,
        gradient_exchange=None,
    ):
        """``exact_exp``: blend kernels use ``expf`` instead of ``ex2.approx`` (parity debugging).
        ``force_key64``: sort the reference's 64-bit ``tile << 32 | depth`` keys even when the live
        bits fit 32.  ``initial_key_capacity``: first guess for the number of (tile, splat) pairs;
        the buffers grow automatically when a frame needs more.  ``keep_all_tile_pairs``: emit a sort key for
        every tile of the reference's 3-sigma square instead of only the tiles the splat can actually reach with
        alpha >= 1/255 (same outputs, ~1.5x more keys; used by tests that compare the sorted list itself).
        ``backward_impl``: ``"transposed"`` (default; ``csrc/blend_bwd_transposed.cu``: splat-per-lane accumulation after a
        shared-memory transposition, 769 us at C3 on a B200) or ``"butterfly"`` (``csrc/blend_bwd.cu``: warp butterfly per
        (warp, splat), 997 us; kept as the second implementation the parity tests cross-check).  Constructor argument only:
        no environment variable can switch the kernel of a production run.  With no backward hook installed the transposed
        kernel does not compute the statistics only a hook reads (the reference's ``need_extra_info = False``, GPCR:521).
        ``skip_unused_hook_statistics``: the same switch for the butterfly kernel (opt-in; ``None`` reads
        ``GSB200_SKIP_HOOK_STATS``).
        ``gradient_exchange``: a ``parallel.ViewParallelExchange`` (view-parallel training, one process per GPU): backward
        then returns the gradients SUMMED over the ranks' views -- the per-point kernel writes compact rows, the ranks
        exchange 14 instead of 59 floats per Gaussian and ``gsb200_expand_view_gradients`` rebuilds the dense sum.  A
        backward hook still sees this rank's own view (``grad_pointfeatures_in_camera`` is ``None`` in this mode: the
        per-view dense feature gradients are never formed)."""
        super().__init__()
        self.config = config
        self.backward_valid_point_hook = backward_valid_point_hook
        self._flags = (_lib.GSB_FLAG_EXACT_EXP if exact_exp else 0) | (_lib.GSB_FLAG_FORCE_KEY64 if force_key64 else 0) | \
            (_lib.GSB_FLAG_KEEP_ALL_TILE_PAIRS if keep_all_tile_pairs else 0)
        backward_impl = backward_impl or "transposed"
        if backward_impl not in ("butterfly", "transposed"):
            raise ValueError(f"backward_impl must be 'butterfly' or 'transposed', got {backward_impl!r}")
        self.backward_impl = backward_impl
        if skip_unused_hook_statistics is None:
            skip_unused_hook_statistics = os.environ.get("GSB200_SKIP_HOOK_STATS", "0") not in ("", "0")
        self.skip_unused_hook_statistics = bool(skip_unused_hook_statistics)
        self.gradient_exchange = gradient_exchange
        self._key_capacity = int(initial_key_capacity) if initial_key_capacity else 0
        self.last_frame: Optional[Frame] = None
        self.last_gradient_buffer: Optional[torch.Tensor] = None  # flat storage behind the latest backward's grads
        self._layout_cache = {}
        _lib.load()  # fail loudly at construction time if the CUDA library is missing
        outer = self

        class _module_function(torch.autograd.Function):

            @staticmethod
            def forward(ctx, pointcloud, pointcloud_features, point_invalid_mask, point_object_id,
                        q_pointcloud_camera, t_pointcloud_camera, camera_info, color_max_sh_band):
                outs, frame, saved = outer._run_forward(
                    pointcloud, pointcloud_features, point_invalid_mask, point_object_id,
                    q_pointcloud_camera, t_pointcloud_camera, camera_info)
                image, depth, acc_alpha, last_effective, valid_count = outs
                ctx.save_for_backward(pointcloud, pointcloud_features, point_object_id,
                                      t_pointcloud_camera, saved["camera_intrinsics"], acc_alpha,
                                      last_effective, frame.ws, saved["q_pointcloud_camera"])
                ctx.frame = frame
                ctx.num_objects = q_pointcloud_camera.shape[0]
                ctx.q_shape, ctx.t_shape = q_pointcloud_camera.shape, t_pointcloud_camera.shape
                ctx.color_max_sh_band = color_max_sh_band
                ctx.mark_non_differentiable(depth, valid_count)
                return image, depth, valid_count

            @staticmethod
            def backward(ctx, grad_rasterized_image, grad_rasterized_depth, grad_pixel_valid_point_count):
                grad_pointcloud = grad_pointcloud_features = grad_q = grad_t = None
                scene = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]  # GPCR:1028
                pose = ctx.needs_input_grad[4] or ctx.needs_input_grad[5]
                if scene or pose:
                    if outer.config.rgb_only:
                        # the reference leaves accumulated alpha / last-effective offsets uninitialised in
                        # this mode (GPCR:478-484), so its backward is undefined; refuse instead
                        raise RuntimeError("rgb_only=True is an inference-only mode: backward needs the "
                                           "auxiliary per-pixel outputs")
                    if pose:
                        grad_pointcloud, grad_pointcloud_features, grad_q, grad_t = outer._run_backward(
                            ctx, grad_rasterized_image, pose=True, scene=scene)
                        if not scene:  # tracking against a frozen scene: no scene gradients, no hook
                            grad_pointcloud = grad_pointcloud_features = None
                        grad_q = grad_q.view(ctx.q_shape) if ctx.needs_input_grad[4] else None
                        grad_t = grad_t.view(ctx.t_shape) if ctx.needs_input_grad[5] else None
                    else:
                        grad_pointcloud, grad_pointcloud_features = outer._run_backward(ctx, grad_rasterized_image)
                return grad_pointcloud, grad_pointcloud_features, None, None, grad_q, grad_t, None, None

        self._module_function = _module_function

    # ------------------------------------------------------------------ forward plumbing
    def _default_key_capacity(self, num_points: int) -> int:
        return max(1 << 20, 8 * num_points)

    def _layout(self, N, n_obj, key_capacity, H, W):
        key = (N, n_obj, key_capacity, H, W, self.config.far_plane, self.config.depth_to_sort_key_scale, self._flags)
        cached = self._layout_cache.get(key)
        if cached is None:
            if len(self._layout_cache) > 64:
                self._layout_cache.clear()
            cached = _lib.workspace_layout(N, n_obj, key_capacity, H, W, self.config.far_plane,
                                           self.config.depth_to_sort_key_scale, self._flags)
            self._layout_cache[key] = cached
        return cached

    def _run_forward(self, pointcloud, pointcloud_features, point_invalid_mask, point_object_id,
                     q_pointcloud_camera, t_pointcloud_camera, camera_info):
        cfg = self.config
        lib = _lib.load()
        _require(pointcloud, "point_cloud", torch.float32, (3,))
        _require(pointcloud_features, "point_cloud_features", torch.float32, (56,))
        _require(point_invalid_mask, "point_invalid_mask", torch.int8)
        _require(point_object_id, "point_object_id", torch.int32)
        _require(q_pointcloud_camera, "q_pointcloud_camera", torch.float32, (4,))
        _require(t_pointcloud_camera, "t_pointcloud_camera", torch.float32, (3,))
        K = camera_info.camera_intrinsics
        _require(K, "camera_info.camera_intrinsics", torch.float32)
        for name, t in (("point_cloud", pointcloud), ("point_cloud_features", pointcloud_features),
                        ("point_invalid_mask", point_invalid_mask), ("point_object_id", point_object_id)):
            if not t.is_contiguous():  # Taichi rejects non-contiguous ndarrays as well
                raise ValueError(f"{name} must be contiguous")
        q_pc = q_pointcloud_camera.contiguous()
        t_pc = t_pointcloud_camera.contiguous()
        K = K.contiguous()
        device = pointcloud.device
        N = pointcloud.shape[0]
        n_obj = q_pc.shape[0]
        H, W = int(camera_info.camera_height), int(camera_info.camera_width)
        if self._key_capacity <= 0:
            self._key_capacity = self._default_key_capacity(N)

        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device)
            image = torch.empty((H, W, 3), dtype=torch.float32, device=device)
            if cfg.rgb_only:
                depth = torch.zeros((H, W), dtype=torch.float32, device=device)
                acc_alpha = torch.zeros((H, W), dtype=torch.float32, device=device)
                last_effective = torch.zeros((H, W), dtype=torch.int32, device=device)
                valid_count = torch.zeros((H, W), dtype=torch.int32, device=device)
            else:
                depth = torch.empty((H, W), dtype=torch.float32, device=device)
                acc_alpha = torch.empty((H, W), dtype=torch.float32, device=device)
                last_effective = torch.empty((H, W), dtype=torch.int32, device=device)
                valid_count = torch.empty((H, W), dtype=torch.int32, device=device)
            readback = _PinnedCounters.acquire(device)
            pinned, event = readback
            retry_flag = 0
            try:
                while True:
                    key_capacity = self._key_capacity
                    layout = self._layout(N, n_obj, key_capacity, H, W)
                    ws = torch.empty((layout.total_bytes,), dtype=torch.uint8, device=device)
                    args = _lib.GsbForwardArgs(
                        num_points=N, pointcloud=_ptr(pointcloud), pointcloud_features=_ptr(pointcloud_features),
                        point_invalid_mask=_ptr(point_invalid_mask), point_object_id=_ptr(point_object_id),
                        num_objects=n_obj, q_pointcloud_camera=_ptr(q_pc), t_pointcloud_camera=_ptr(t_pc),
                        camera_intrinsics=_ptr(K), camera_height=H, camera_width=W,
                        near_plane=cfg.near_plane, far_plane=cfg.far_plane,
                        depth_to_sort_key_scale=cfg.depth_to_sort_key_scale, rgb_only=1 if cfg.rgb_only else 0,
                        flags=self._flags | retry_flag, workspace=_ptr(ws), workspace_bytes=layout.total_bytes,
                        key_capacity=key_capacity, rasterized_image=_ptr(image), rasterized_depth=_ptr(depth),
                        pixel_accumulated_alpha=_ptr(acc_alpha),
                        pixel_offset_of_last_effective_point=_ptr(last_effective),
                        pixel_valid_point_count=_ptr(valid_count), stream=stream.cuda_stream,
                        host_counters=pinned.data_ptr(), host_counters_event=event.cuda_event)
                    # The whole frame is enqueued by this one call; the library copies {M, K, overflow} to pinned
                    # host memory right after the per-point stage and records `event` behind that copy.
                    _lib.check(lib.gsb200_forward(ctypes.byref(args)), "gsb200_forward")
                    frame = Frame(ws, layout, N, key_capacity, H, W, self._flags)
                    # ONE host wait per frame (the reference syncs twice, GPCR:864 and GPCR:916-931), and it ends
                    # when the first kernel is done: sort + blend are still in flight when we return.
                    event.synchronize()
                    frame.num_points_in_camera = int(pinned[0])
                    frame.num_keys = int(pinned[1])
                    if int(pinned[2]) == 0:
                        break
                    # more (tile, splat) pairs than capacity: grow and redo the frame.  The first pass already
                    # normalised the quaternions in place; the re-run must not normalise them a second time.
                    self._key_capacity = int(frame.num_keys * 1.25) + 4096
                    retry_flag = _lib.GSB_FLAG_Q_ALREADY_NORMALISED
            finally:  # also when the library call raises: the pooled pair goes back
                _PinnedCounters.release(device, readback)
        self.last_frame = frame
        return (image, depth, acc_alpha, last_effective, valid_count), frame, {"camera_intrinsics": K,
                                                                               "q_pointcloud_camera": q_pc}

    # ------------------------------------------------------------------ backward plumbing
    def _run_backward(self, ctx, grad_rasterized_image, pose: bool = False, scene: bool = True):
        """Dense gradients (and the hook).  ``pose``: also the gradients of q / t_pointcloud_camera (gsb200_backward_with_pose),
        returned as two more tensors; ``scene = False`` (pose only): the hook is not called and no gradient is exchanged."""
        cfg = self.config
        lib = _lib.load()
        (pointcloud, pointcloud_features, point_object_id, t_pointcloud_camera, K, acc_alpha,
         last_effective, ws, q_pointcloud_camera) = ctx.saved_tensors
        frame: Frame = ctx.frame
        device = pointcloud.device
        N = pointcloud.shape[0]
        M = frame.num_points_in_camera
        H, W = frame.height, frame.width
        band = ctx.color_max_sh_band
        band_i = int(band) if band in (0, 1, 2) else 3  # GPCR:1167-1182: anything else clears nothing
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device)
            grad_image = grad_rasterized_image.contiguous()
            if grad_image.dtype != torch.float32:
                grad_image = grad_image.float()
            # both dense gradients live in ONE allocation (xyz rows, pad to 16 B, feature rows) so that a
            # view-parallel trainer can sum them over ranks with a single collective (parallel.py)
            off = (3 * N + 3) // 4 * 4
            flat = torch.empty((off + 56 * N,), dtype=torch.float32, device=device)
            if off > 3 * N:
                flat[3 * N:off].zero_()
            grad_pointcloud = flat[:3 * N].view(N, 3)
            grad_pointcloud_features = flat[off:off + 56 * N].view(N, 56)
            self.last_gradient_buffer = flat
            accum = torch.empty((max(M, 1), _ACCUM_FLOATS), dtype=torch.float32, device=device)
            magnitude_on_image = torch.empty((H, W, 2), dtype=torch.float32, device=device)
            t_pc = t_pointcloud_camera.contiguous()
            backward_flags = self.backward_flags(frame.flags)
            exchange = self.gradient_exchange
            compact = exchange is not None and exchange.world > 1 and scene
            grad_sum = blocks = None
            if compact:
                n_obj = ctx.num_objects
                grad_sum, blocks = exchange.allocate(N, n_obj, device)
                blocks[exchange.rank, 3 * N:3 * N + 3 * n_obj] = t_pc.reshape(-1)
                backward_flags |= _lib.GSB_FLAG_COMPACT_GRADS
            args = _lib.GsbBackwardArgs(
                num_points=N, pointcloud=_ptr(pointcloud), pointcloud_features=_ptr(pointcloud_features),
                point_object_id=_ptr(point_object_id), num_objects=ctx.num_objects,
                t_pointcloud_camera=_ptr(t_pc), camera_intrinsics=_ptr(K), camera_height=H, camera_width=W,
                far_plane=cfg.far_plane, depth_to_sort_key_scale=cfg.depth_to_sort_key_scale,
                color_max_sh_band=band_i, grad_q_factor=cfg.grad_q_factor, grad_s_factor=cfg.grad_s_factor,
                grad_alpha_factor=cfg.grad_alpha_factor, grad_color_factor=cfg.grad_color_factor,
                grad_high_order_color_factor=cfg.grad_high_order_color_factor, flags=backward_flags,
                workspace=_ptr(ws), workspace_bytes=frame.layout.total_bytes, key_capacity=frame.key_capacity,
                grad_rasterized_image=_ptr(grad_image), pixel_accumulated_alpha=_ptr(acc_alpha),
                pixel_offset_of_last_effective_point=_ptr(last_effective), accum=_ptr(accum),
                accum_rows=M, grad_pointcloud=_ptr(grad_pointcloud),
                grad_pointcloud_features=_ptr(grad_pointcloud_features),
                magnitude_grad_viewspace_on_image=_ptr(magnitude_on_image), stream=stream.cuda_stream,
                grad_sum_compact=_ptr(grad_sum), grad_color_compact=_ptr(blocks[exchange.rank]) if compact else None)
            if pose:
                n_obj = ctx.num_objects
                if not hasattr(lib, "gsb200_backward_with_pose"):
                    raise RuntimeError(f"{_lib.LIB_PATH} has no gsb200_backward_with_pose: rebuild it for pose gradients")
                if n_obj > _lib.GSB_POSE_MAX_OBJECTS:
                    raise RuntimeError(f"pose gradients are available for at most {_lib.GSB_POSE_MAX_OBJECTS} objects, "
                                       f"got {n_obj}")
                grad_pose = torch.empty((7 * n_obj,), dtype=torch.float32, device=device)
                grad_q, grad_t = grad_pose[:4 * n_obj].view(n_obj, 4), grad_pose[4 * n_obj:].view(n_obj, 3)
                temp = torch.empty((lib.gsb200_pose_grad_temp_bytes(n_obj),), dtype=torch.uint8, device=device)
                pargs = _lib.GsbPoseGradArgs(
                    q_pointcloud_camera=_ptr(q_pointcloud_camera), t_pointcloud_camera=_ptr(t_pc),
                    grad_q_pointcloud_camera=_ptr(grad_q), grad_t_pointcloud_camera=_ptr(grad_t), temp=_ptr(temp),
                    temp_bytes=temp.numel())
                _lib.check(lib.gsb200_backward_with_pose(ctypes.byref(args), ctypes.byref(pargs)),
                           "gsb200_backward_with_pose")
            else:
                _lib.check(lib.gsb200_backward(ctypes.byref(args)), "gsb200_backward")
            own_view_grad_xyz = None
            if compact:
                exchange.rows_written(grad_sum, blocks)
                if self.backward_valid_point_hook is not None:  # the hook sees this rank's own view (before the sum)
                    own_view_grad_xyz = grad_sum[frame.point_id_in_camera_list.long(), 0:3]

                def expand(part: int) -> None:
                    """Dense gradients from the exchanged compact rows, on the CURRENT stream (part 0: everything; 1: the SH
                    columns, which need only the gathered blocks; 2: the summed columns) -- csrc/blend_bwd.cu."""
                    eargs = _lib.GsbExpandArgs(
                        num_points=N, num_views=exchange.world, num_objects=ctx.num_objects, grad_sum=_ptr(grad_sum),
                        grad_color_views=_ptr(blocks), view_stride=blocks.shape[1], pointcloud=_ptr(pointcloud),
                        point_object_id=_ptr(point_object_id), color_max_sh_band=band_i,
                        grad_color_factor=cfg.grad_color_factor,
                        grad_high_order_color_factor=cfg.grad_high_order_color_factor, part=part,
                        grad_pointcloud=_ptr(grad_pointcloud), grad_pointcloud_features=_ptr(grad_pointcloud_features),
                        stream=torch.cuda.current_stream(device).cuda_stream)
                    _lib.check(lib.gsb200_expand_view_gradients(ctypes.byref(eargs)), "gsb200_expand_view_gradients")

                exchange.run_and_expand(grad_sum, blocks, expand)

            hook = self.backward_valid_point_hook if scene else None
            if hook is not None:  # GPCR:1127-1142
                ids = frame.point_id_in_camera_list
                ids64 = ids.long()
                acc = accum[:M]
                hook(GaussianPointCloudRasterisation.BackwardValidPointHookInput(
                    point_id_in_camera_list=ids,
                    grad_point_in_camera=own_view_grad_xyz if compact else grad_pointcloud[ids64],
                    grad_pointfeatures_in_camera=None if compact else grad_pointcloud_features[ids64],
                    grad_viewspace=acc[:, 0:2].contiguous(),
                    magnitude_grad_viewspace=acc[:, 9].contiguous(),
                    magnitude_grad_viewspace_on_image=magnitude_on_image,
                    num_overlap_tiles=frame.num_overlap_tiles,
                    num_affected_pixels=acc[:, 10].round().to(torch.int32),
                    point_uv_in_camera=frame.point_uv.contiguous(),
                    point_depth=frame.point_in_camera[:, 2],
                ))
        if pose:
            return grad_pointcloud, grad_pointcloud_features, grad_q, grad_t
        return grad_pointcloud, grad_pointcloud_features

    def backward_flags(self, frame_flags: int) -> int:
        """Flags of the backward call for a frame rendered with ``frame_flags`` (adds the experimental kernel selection)."""
        if self.backward_impl == "transposed":
            frame_flags |= _lib.GSB_FLAG_BACKWARD_TRANSPOSED
        if self.backward_valid_point_hook is None and (self.backward_impl == "transposed" or self.skip_unused_hook_statistics):
            frame_flags |= _lib.GSB_FLAG_NO_HOOK_STATS  # the reference's need_extra_info = False, GPCR:521
        return frame_flags

    # ------------------------------------------------------------------ public forward (GPCR:1184-1204)
    def forward(self, input_data: "GaussianPointCloudRasterisation.GaussianPointCloudRasterisationInput"):
        camera_info = input_data.camera_info
        assert camera_info.camera_width % TILE_WIDTH == 0
        assert camera_info.camera_height % TILE_HEIGHT == 0
        return self._module_function.apply(
            input_data.point_cloud,
            input_data.point_cloud_features,
            input_data.point_invalid_mask,
            input_data.point_object_id,
            input_data.q_pointcloud_camera,
            input_data.t_pointcloud_camera,
            camera_info,
            input_data.color_max_sh_band,
        )


@dataclass
class GaussianPoint3D:
    """The fields of the reference's ``GaussianPoint3D`` Taichi struct (GaussianPoint3D.py:17-27) as tensors."""
    translation: torch.Tensor  # (3,)
    cov_rotation: torch.Tensor  # (4,) xyzw
    cov_scale: torch.Tensor  # (3,) log-scale
    alpha: torch.Tensor  # () opacity logit
    color_r: torch.Tensor  # (16,)
    color_g: torch.Tensor  # (16,)
    color_b: torch.Tensor  # (16,)


def load_point_cloud_row_into_gaussian_point_3d(pointcloud: torch.Tensor, pointcloud_features: torch.Tensor,
                                                point_id: int) -> GaussianPoint3D:
    """Same name, arguments and row layout as the reference's ``@ti.func`` (GPCR:208-236; imported by its controller,
    GaussianPointAdaptiveController.py:4, and pinned by its test ``test_load_point_cloud_row_into_gaussian_point_3d``):
    row ``point_id`` of the (N,3) / (N,56) tensors as a ``GaussianPoint3D`` -- q xyzw | log-scale | opacity logit |
    R, G, B SH x 16.  Host-side views; inside the kernels the same split is done by ``preprocess_kernel``."""
    f = pointcloud_features[point_id]
    return GaussianPoint3D(translation=pointcloud[point_id], cov_rotation=f[0:4], cov_scale=f[4:7], alpha=f[7],
                           color_r=f[8:24], color_g=f[24:40], color_b=f[40:56])


def find_tile_start_and_end(point_in_camera_sort_key: torch.Tensor, tile_points_start: torch.Tensor,
                            tile_points_end: torch.Tensor) -> None:
    """Same call shape as the reference kernel (GPCR:175-193; used by its tests): sorted int64 keys
    ``tile << 32 | depth`` -> per-tile [start, end) written into the two zero-initialised int32 outputs."""
    lib = _lib.load()
    _require(point_in_camera_sort_key, "point_in_camera_sort_key", torch.int64)
    _require(tile_points_start, "tile_points_start", torch.int32)
    _require(tile_points_end, "tile_points_end", torch.int32)
    fn = lib.gsb200_find_tile_start_and_end
    fn.argtypes = [_lib.c_vp, _lib.c_i64, _lib.c_vp, _lib.c_vp, _lib.c_i32, _lib.c_vp]
    fn.restype = ctypes.c_int
    with torch.cuda.device(point_in_camera_sort_key.device):
        stream = torch.cuda.current_stream(point_in_camera_sort_key.device)
        keys = point_in_camera_sort_key.contiguous()
        _lib.check(fn(keys.data_ptr(), keys.shape[0], tile_points_start.data_ptr(), tile_points_end.data_ptr(),
                      tile_points_start.shape[0], stream.cuda_stream), "gsb200_find_tile_start_and_end")
