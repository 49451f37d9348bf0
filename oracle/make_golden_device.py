"""Golden fixtures of the reference's mesh-extraction grid and data loader, from the UNMODIFIED reference on a CUDA device.

    python oracle/make_golden_device.py [OUT.npz]     # default: tests/golden/device_outputs.npz

Needs the reference's own `extract_mesh.py` and `dataset/dataset.py` (a checkout, or the staged copy made by
oracle/make_ref.py) and a GPU: the reference creates its tensors on the default CUDA device, so its random pixel draws
come from the CUDA generator, and its grid query is driven with our UDF module's callbacks (as tests/test_gpu_grid.py
does).  Two groups, sampled with fixed seeds to keep the fixture small:
  * grid_*: get_udf_normals_grid_slow (extract_mesh.py:18-105) at N = 48 on the golden scene's UDF: the near-surface
    mask in full (packed bits), all seven columns of `samples` at 2048 lattice points, the normals at 1024 near-surface cells;
  * ds_* / rays_* / grid{l}_*: Dataset (dataset/dataset.py) on tests/runner_env.write_synthetic_dtu's scene: the camera
    tensors raygen reads, per-image sums of the loaded images / masks, gen_random_rays_patches_at after
    torch.manual_seed(1234) for the cases of tests/test_gpu_raygen.py, gen_rays_at(3, l) at up to 512 pixels.
"""
import importlib
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import refshim  # noqa: E402
from tests import runner_env  # noqa: E402
from tests.golden_util import load_golden  # noqa: E402
from tests.gpu_util import build_modules  # noqa: E402

GRID_N = 48
RAY_CASES = ((0, False), (5, True), (11, False))        # (img_idx, crop_patch) of tests/test_gpu_raygen.py
GRID_LEVELS = (1, 2, 4)


def np_(t):
    return t.detach().cpu().numpy()


def _ref_module(name):
    runner_env.install_stubs()
    if refshim.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, refshim.REFERENCE_ROOT)
    for k in [k for k in sys.modules if k == name or k.startswith(name + ".")]:
        del sys.modules[k]
    mod = importlib.import_module(name)
    assert mod.__file__.startswith(refshim.REFERENCE_ROOT), mod.__file__
    return mod


def grid_fixtures(fx):
    udf = build_modules(load_golden(), "cuda")[0]

    def func_grad(xyz):                                    # exp_runner_blending.py:767-771
        g = udf.gradient(xyz)
        return g / (torch.linalg.norm(g, ord=2, dim=-1, keepdim=True) + 1e-5)

    em = _ref_module("extract_mesh")
    torch.set_default_tensor_type("torch.cuda.FloatTensor")
    try:
        df, vec, samples = em.get_udf_normals_grid_slow(udf.udf, func_grad, N=GRID_N, max_batch=1 << 14)
    finally:
        torch.set_default_tensor_type("torch.FloatTensor")
    samples = np_(samples).astype(np.float32)
    mask = np_(vec.abs().sum(-1) > 0).reshape(-1)
    rng = np.random.default_rng(0)
    idx = np.sort(rng.choice(GRID_N ** 3, 2048, replace=False)).astype(np.int32)
    surf = np.flatnonzero(mask)
    sidx = np.sort(rng.choice(surf, min(1024, surf.size), replace=False)).astype(np.int32)
    fx["grid_n"] = np.array(GRID_N)
    fx["grid_mask_bits"] = np.packbits(mask)
    fx["grid_idx"], fx["grid_samples"] = idx, samples[idx]
    fx["grid_surface_idx"], fx["grid_surface_vec"] = sidx, samples[sidx, 4:]


def dataset_fixtures(fx, tmp):
    data = runner_env.write_synthetic_dtu(os.path.join(tmp, "synth"), n_images=12, width=96, height=72)
    mod = _ref_module("dataset.dataset")
    conf = runner_env.ConfigTree(data_dir=data + "/", render_cameras_name="cameras.npz", object_cameras_name="cameras.npz")
    torch.set_default_tensor_type("torch.cuda.FloatTensor")
    try:
        ds = mod.Dataset(conf)
        fx["ds_hw"] = np.array([ds.H, ds.W])
        fx["ds_pose_all"], fx["ds_intrinsics_all_inv"] = np_(ds.pose_all), np_(ds.intrinsics_all_inv)
        fx["ds_image_sums"] = np_(ds.images.double().sum(dim=(1, 2, 3)))
        fx["ds_mask_sums"] = np_(ds.masks.double().sum(dim=(1, 2, 3)))
        rng = np.random.default_rng(1)
        for img_idx, crop in RAY_CASES:
            torch.manual_seed(1234)
            ref = ds.gen_random_rays_patches_at(img_idx, 512, crop_patch=crop, h_patch_size=3)
            near, far = ds.near_far_from_sphere(ref["rays"][:, :3], ref["rays"][:, 3:6])
            p = "rays%d_" % img_idx
            fx[p + "rays"], fx[p + "ndc_uv"] = np_(ref["rays"]), np_(ref["rays_ndc_uv"])
            fx[p + "norm_xyz_cam"], fx[p + "near"], fx[p + "far"] = np_(ref["rays_norm_XYZ_cam"]), np_(near), np_(far)
            if crop:
                sel = np.sort(rng.choice(512, 64, replace=False)).astype(np.int32)
                fx[p + "patch_mask"] = np_(ref["rays_patch_mask"])
                fx[p + "patch_idx"], fx[p + "patch_color"] = sel, np_(ref["rays_patch_color"])[sel]
        for level in GRID_LEVELS:
            ro, rd = ds.gen_rays_at(3, resolution_level=level)
            near, far = ds.near_far_from_sphere(ro.reshape(-1, 3), rd.reshape(-1, 3))
            n = ro.shape[0] * ro.shape[1]
            sel = np.sort(rng.choice(n, min(512, n), replace=False)).astype(np.int32)
            p = "grid%d_" % level
            fx[p + "shape"], fx[p + "idx"] = np.array(ro.shape), sel
            fx[p + "origin"] = np_(ro.reshape(-1, 3)[0])
            assert bool((ro.reshape(-1, 3) == ro.reshape(-1, 3)[0]).all())
            fx[p + "dirs"] = np_(rd.reshape(-1, 3))[sel]
            fx[p + "near"], fx[p + "far"] = np_(near)[sel], np_(far)[sel]
    finally:
        torch.set_default_tensor_type("torch.FloatTensor")


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "device_outputs.npz")
    assert torch.cuda.is_available() and refshim.available(), "needs a CUDA device and the reference (oracle/make_ref.py)"
    fx = {}
    grid_fixtures(fx)
    with tempfile.TemporaryDirectory() as tmp:
        dataset_fixtures(fx, tmp)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    np.savez_compressed(out, **fx)
    print("wrote %d arrays, %.1f KB raw -> %s (%.1f KB)" % (len(fx), sum(v.nbytes for v in fx.values()) / 1e3, out,
                                                           os.path.getsize(out) / 1e3))


if __name__ == "__main__":
    main()
