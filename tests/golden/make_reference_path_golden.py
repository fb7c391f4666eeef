"""Golden vectors for the WHOLE hot path, produced by the reference's own kernels.

The reference's rasteriser (GaussianPointCloudRasterisation.py:31-1204 with GaussianPoint3D.py, SphericalHarmonics.py and
the ``ti.func`` helpers of utils.py) is imported from /root/reference and executed, unmodified, under ``taichi_shim``
(a minimal Taichi stand-in, see its docstring: float32 numpy arithmetic, by-value ``ti.func`` arguments, lock-step SIMT
emulation of the two shared-memory kernels).  For every scene of ``reference_path_scenes.py`` it runs
forward + backward through the reference's ``torch.autograd.Function`` on CPU tensors and stores: image, depth, valid
point count, the in-place-normalised feature tensor, both gradients, every tensor handed to the backward hook, and the
per-stage tensors the kernels write (projected attributes, sorted keys and offsets, tile ranges, accumulated alpha, last
effective offsets).

One deviation from a literal run: ``Tensor.sort`` is made stable.  The reference calls ``sort()`` on a CUDA tensor, where
it is CUB's (stable) radix sort; the CPU fallback is not, and tie order is part of the contract (SURVEY section 9.8).

    python tests/golden/make_reference_path_golden.py [--with-c1]   # build container only; writes reference_path_vectors.npz
                                                                    # (--with-c1: also BASELINE config 1 -> reference_path_c1.npz)
"""
import os
import sys
import time
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import taichi_shim  # noqa: E402
from reference_path_scenes import baseline_config_1, reduced_config_2, scenes  # noqa: E402


def validate_shim():
    """The shim is only trusted as far as the reference's OWN unit tests of the Taichi code on this path pass under it,
    run unmodified (they build Taichi fields, define kernels inside the test, compare with numpy / scipy / torch autograd):

    * tests/GaussianPoint3D_test.py (whole file): Sigma' projection, quaternion -> R;
    * tests/utils_test.py::Test2DGaussianPDF: 2-D Gaussian density and its mean / covariance gradients;
    * tests/GaussianPointCloudRasterisation_test.py: find_tile_start_and_end, the feature-row loader, the two-point
      scene rendered through the operator, and test_single_point (operator forward AND backward -- alpha, d/d uv,
      d/d cov, d/d xyz, d/d q, d/d s, d/d logit -- against torch autograd).  That file asks for cuda:0 tensors; its
      ``torch.device`` is redirected to the CPU, nothing else is touched.
    The operator's stress / optimisation tests of that file (1e5 points at 1080p, 1e4 Adam iterations) are too large for
    an interpreter and are restated in tests/test_reference_behaviour.py instead."""
    import contextlib
    import importlib
    import io
    import unittest
    sys.path.insert(0, "/root/reference/tests")
    loader, suite = unittest.defaultTestLoader, unittest.TestSuite()
    suite.addTests(loader.loadTestsFromModule(importlib.import_module("GaussianPoint3D_test")))
    suite.addTests(loader.loadTestsFromTestCase(importlib.import_module("utils_test").Test2DGaussianPDF))
    rast = importlib.import_module("GaussianPointCloudRasterisation_test")
    cpu = torch.device("cpu")
    rast.torch = types.SimpleNamespace(**{k: getattr(torch, k) for k in dir(torch) if not k.startswith("__")})
    rast.torch.device = lambda *a, **k: cpu
    wanted = ("test_find_tile_start_and_end", "test_load_point_cloud_row_into_gaussian_point_3d",
              "test_rasterisation_two_points", "test_single_point")
    for attr in vars(rast).values():
        if isinstance(attr, type) and issubclass(attr, unittest.TestCase):
            suite.addTests(attr(name) for name in wanted if hasattr(attr, name))
    with contextlib.redirect_stderr(io.StringIO()), contextlib.redirect_stdout(io.StringIO()):
        result = unittest.TextTestRunner(stream=io.StringIO(), verbosity=0).run(suite)
    assert result.testsRun == 7 and result.wasSuccessful(), (result.testsRun, result.failures, result.errors)
    print("shim check: 7 of the reference's own unit tests of this path pass with its kernels running under the shim")


def main():
    taichi_shim.install()
    sys.modules.setdefault("dataclass_wizard", types.SimpleNamespace(YAMLWizard=object))
    sys.path.insert(0, "/root/reference")
    plain_sort = torch.Tensor.sort
    torch.Tensor.sort = lambda self, *a, **k: plain_sort(self, *a, **{"stable": True, **k})
    validate_shim()
    from taichi_3d_gaussian_splatting.Camera import CameraInfo
    import taichi_3d_gaussian_splatting.GaussianPointCloudRasterisation as refmod
    from taichi_3d_gaussian_splatting.GaussianPointCloudRasterisation import GaussianPointCloudRasterisation as G

    # record the tensors the kernels write in place (the orchestration calls them by module-level name)
    stage = {}

    def recording(kernel_name, keys):
        kernel = getattr(refmod, kernel_name)

        def wrapped(**kwargs):
            kernel(**kwargs)
            for key in keys:
                stage[key] = kwargs[key].detach().clone()
        setattr(refmod, kernel_name, wrapped)

    recording("generate_point_attributes_in_camera_plane", ["point_uv", "point_in_camera", "point_uv_conic_and_rescale",
                                                            "point_alpha_after_activation", "point_color", "point_radii"])
    recording("find_tile_start_and_end", ["point_in_camera_sort_key", "tile_points_start", "tile_points_end"])
    recording("gaussian_point_rasterisation", ["point_offset_with_sort_key", "pixel_accumulated_alpha",
                                               "pixel_offset_of_last_effective_point"])

    with_c1 = "--with-c1" in sys.argv  # BASELINE config 1 takes a few minutes in the interpreter; its file is separate
    todo = dict(scenes())
    if with_c1:
        todo["C1_baseline_config_1"] = baseline_config_1()
    with_c2r = "--with-c2r" in sys.argv  # reduced BASELINE config 2: more than two and a half hours in the interpreter (1.2e8 pixel x splat iterations), sampled output
    if with_c2r:
        todo = {"C2R_reduced_config_2": reduced_config_2()} if "--only-c2r" in sys.argv else {**todo, "C2R_reduced_config_2": reduced_config_2()}
    out = {}
    for name, sc in todo.items():
        t0 = time.time()
        pc = sc["point_cloud"].clone().requires_grad_(True)
        feat = sc["point_cloud_features"].clone().requires_grad_(True)
        hook = {}
        module = G(config=G.GaussianPointCloudRasterisationConfig(
            near_plane=sc["near_plane"], far_plane=sc["far_plane"], depth_to_sort_key_scale=sc["depth_to_sort_key_scale"]),
            backward_valid_point_hook=lambda h: hook.update(h=h))
        info = CameraInfo(camera_intrinsics=sc["camera_intrinsics"].clone(), camera_height=sc["camera_height"],
                          camera_width=sc["camera_width"], camera_id=0)
        image, depth, count = module(G.GaussianPointCloudRasterisationInput(
            point_cloud=pc, point_cloud_features=feat, point_object_id=sc["point_object_id"],
            point_invalid_mask=sc["point_invalid_mask"], camera_info=info, q_pointcloud_camera=sc["q_pointcloud_camera"],
            t_pointcloud_camera=sc["t_pointcloud_camera"], color_max_sh_band=sc["color_max_sh_band"]))
        grad_image = torch.randn(image.shape, generator=torch.Generator().manual_seed(sc["grad_seed"]))
        image.backward(grad_image)
        h = hook["h"]
        rec = dict(image=image.detach(), depth=depth.detach(), count=count.detach(), features_after_forward=feat.detach(),
                   grad_pointcloud=pc.grad, grad_pointcloud_features=feat.grad,
                   hook_point_id_in_camera_list=h.point_id_in_camera_list, hook_grad_point_in_camera=h.grad_point_in_camera,
                   hook_grad_pointfeatures_in_camera=h.grad_pointfeatures_in_camera, hook_grad_viewspace=h.grad_viewspace,
                   hook_magnitude_grad_viewspace=h.magnitude_grad_viewspace,
                   hook_magnitude_grad_viewspace_on_image=h.magnitude_grad_viewspace_on_image,
                   hook_num_overlap_tiles=h.num_overlap_tiles, hook_num_affected_pixels=h.num_affected_pixels,
                   hook_point_depth=h.point_depth, hook_point_uv_in_camera=h.point_uv_in_camera)
        rec.update({f"stage_{k}": v for k, v in stage.items()})
        stage.clear()
        for key, value in rec.items():
            out[f"{name}/{key}"] = value.detach().cpu().numpy()
        print(f"{name}: {time.time() - t0:.1f} s, M={h.point_id_in_camera_list.shape[0]}, "
              f"max blended per pixel={int(count.max())}, image max={float(image.max()):.3f}")
    small = {k: v for k, v in out.items() if not k.startswith(("C1_", "C2R_"))}
    if small:
        np.savez_compressed(os.path.join(HERE, "reference_path_vectors.npz"), **small)
        print("wrote", len(small), "arrays")
    if with_c2r:
        # 976 x 544 pixels, 3.7e4 points, 4.9e5 pairs: keep hashes of everything that must be bit-equal and samples of the rest
        pre = "C2R_reduced_config_2/"
        full = {k[len(pre):]: v for k, v in out.items() if k.startswith(pre)}
        keep = {"sha256_" + key: digest(full[key]) for key in (
            "hook_point_id_in_camera_list", "hook_num_overlap_tiles", "hook_num_affected_pixels", "count",
            "stage_point_in_camera_sort_key", "stage_point_offset_with_sort_key", "stage_tile_points_start",
            "stage_tile_points_end", "stage_pixel_offset_of_last_effective_point", *PER_POINT_STAGE, "features_after_forward")}
        keep.update(samples(full, 6000, 1500))
        keep["sizes"] = np.array([full["hook_point_id_in_camera_list"].shape[0], full["stage_point_offset_with_sort_key"].shape[0],
                                  int(full["count"].max())])
        np.savez_compressed(os.path.join(HERE, "reference_path_c2_reduced.npz"), **keep)
        print("wrote", len(keep), "arrays for the reduced BASELINE config 2")
    if with_c1:
        pre = "C1_baseline_config_1/"
        full = {k[len(pre):]: v for k, v in out.items() if k.startswith(pre)}
        np.savez_compressed(os.path.join(HERE, "reference_path_c1.npz"), **reduce_c1(full))
        print("wrote the arrays for BASELINE config 1")


PER_POINT_STAGE = ("stage_point_uv", "stage_point_in_camera", "stage_point_uv_conic_and_rescale",
                   "stage_point_alpha_after_activation", "stage_point_color", "stage_point_radii")


def digest(a):
    import hashlib
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def samples(full, num_pixels, num_rows):
    """Seeded samples of the float outputs: pixels of image / depth / count / accumulated alpha, per-tile image sums, rows of
    the hook gradients with each gradient's L1 norm over all rows."""
    keep = {}
    rng = np.random.default_rng(0)
    h, w = full["count"].shape
    pix = rng.choice(h * w, num_pixels, replace=False)
    keep["pixel_index"] = pix
    for key in ("image", "depth", "count", "stage_pixel_accumulated_alpha"):
        keep["pixel_" + key] = full[key].reshape(h * w, -1)[pix]
    tiles = full["image"].reshape(h // 16, 16, w // 16, 16, 3).astype(np.float64).sum(axis=(1, 3))
    keep["tile_image_sum"] = tiles.astype(np.float32)
    m = full["hook_point_id_in_camera_list"].shape[0]
    rows = np.sort(rng.choice(m, num_rows, replace=False))
    keep["point_rows"] = rows
    for key in ("hook_grad_point_in_camera", "hook_grad_pointfeatures_in_camera", "hook_grad_viewspace",
                "hook_magnitude_grad_viewspace"):
        keep["rows_" + key] = full[key][rows]
        keep["l1_" + key] = np.array([np.abs(full[key].astype(np.float64)).sum()])
    return keep


def reduce_c1(full):
    """BASELINE config 1 (256 x 256, 9566 points in the frustum) within 1 MB: the integer outputs the GPU test compares with
    a tolerance are stored whole, every other array that must be bit-equal as a SHA-256, and the floats as a quarter of the
    pixels and of the in-frustum rows.  The dense gradients are zero outside the frustum (checked here) and equal the hook
    tensors inside it, so they are not stored."""
    ids = full["hook_point_id_in_camera_list"].astype(np.int64)
    for key, hook in (("grad_pointcloud", "hook_grad_point_in_camera"),
                      ("grad_pointcloud_features", "hook_grad_pointfeatures_in_camera")):
        rest = np.ones(full[key].shape[0], dtype=bool)
        rest[ids] = False
        assert not full[key][rest].any() and np.array_equal(full[key][ids], full[hook])
    keep = {key: full[key] for key in ("hook_point_id_in_camera_list", "hook_num_overlap_tiles", "hook_num_affected_pixels",
                                       "count", "stage_tile_points_start", "stage_tile_points_end")}
    keep.update({"sha256_" + key: digest(full[key]) for key in (
        "stage_point_in_camera_sort_key", "stage_point_offset_with_sort_key", "stage_pixel_offset_of_last_effective_point",
        *PER_POINT_STAGE)})
    keep.update(samples(full, 16384, 2400))
    return keep


if __name__ == "__main__":
    main()
