"""Device ray generation (neuraludf_b200/raygen.py, csrc/raygen.cu) against the reference's own data loader
(dataset/dataset.py:151-164, 228-294, 329-335) on a synthetic DTU-layout scene.  The reference's outputs for the seeded
draws below are stored by oracle/make_golden_device.py in tests/golden/device_outputs.npz (the patch colours and the
full-image grids at seeded samples of their rays)."""
import glob
import os
import types

import numpy as np
import pytest
import torch

from tests.golden_util import load_device_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref_dataset(tmp_path_factory):
    """What raygen reads of the reference's Dataset: images and masks loaded as dataset.py:69-70 does, and its camera
    tensors as the reference computed them."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import cv2
    from tests import runner_env
    fx = load_device_golden()
    root = runner_env.write_synthetic_dtu(str(tmp_path_factory.mktemp("dtu") / "synth"), n_images=12, width=96, height=72)

    def load(sub):
        return torch.from_numpy((np.stack([cv2.imread(f) for f in sorted(glob.glob(os.path.join(root, sub, "*.png")))])
                                 / 256.0).astype(np.float32)).cuda()
    ds = types.SimpleNamespace(images=load("image"), masks=load("mask"), H=int(fx["ds_hw"][0]), W=int(fx["ds_hw"][1]),
                               pose_all=torch.from_numpy(fx["ds_pose_all"]).cuda(),
                               intrinsics_all_inv=torch.from_numpy(fx["ds_intrinsics_all_inv"]).cuda())
    assert tuple(ds.images.shape[1:3]) == (ds.H, ds.W)
    np.testing.assert_allclose(ds.images.double().sum(dim=(1, 2, 3)).cpu().numpy(), fx["ds_image_sums"], rtol=1e-12)
    np.testing.assert_allclose(ds.masks.double().sum(dim=(1, 2, 3)).cpu().numpy(), fx["ds_mask_sums"], rtol=1e-12)
    return ds


def test_random_rays_match_reference(ref_dataset):
    from neuraludf_b200 import raygen
    ds = ref_dataset
    fx = load_device_golden()
    for img_idx, crop in ((0, False), (5, True), (torch.tensor(11), False)):
        p = "rays%d_" % int(img_idx)
        ref = {k: torch.from_numpy(fx[p + k]).cuda() for k in ("rays", "ndc_uv", "norm_xyz_cam", "near", "far")}
        torch.manual_seed(1234)
        new = raygen.gen_random_rays_patches_at(ds, img_idx, 512, crop_patch=crop, h_patch_size=3, with_near_far=True)
        assert torch.equal(new["rays"][:, 6:], ref["rays"][:, 6:])                      # gathered colours and mask: exact
        assert torch.equal(new["rays"][:, :3], ref["rays"][:, :3])                      # origins: exact
        assert float((new["rays"][:, 3:6] - ref["rays"][:, 3:6]).abs().max()) < 2e-6    # unit directions
        assert float((new["rays_ndc_uv"] - ref["ndc_uv"]).abs().max()) < 1e-6
        assert float((new["rays_norm_XYZ_cam"] - ref["norm_xyz_cam"]).abs().max()) < 1e-5
        assert float((new["near"] - ref["near"]).abs().max()) < 1e-5 and float((new["far"] - ref["far"]).abs().max()) < 1e-5
        if crop:
            assert torch.equal(new["rays_patch_mask"].cpu(), torch.from_numpy(fx[p + "patch_mask"]))
            sel = torch.from_numpy(fx[p + "patch_idx"].astype(np.int64)).cuda()
            ref_c = torch.from_numpy(fx[p + "patch_color"]).cuda()
            assert new["rays_patch_color"].shape == (512,) + ref_c.shape[1:]
            assert float((new["rays_patch_color"][sel] - ref_c).abs().max()) < 1e-6
        else:
            assert new["rays_patch_color"] is None and new["rays_patch_mask"] is None


@pytest.mark.parametrize("level", [1, 2, 4])
def test_ray_grid_matches_reference(ref_dataset, level):
    from neuraludf_b200 import raygen
    ds = ref_dataset
    fx = load_device_golden()
    p = "grid%d_" % level
    no, nd, near, far = raygen.gen_rays_at(ds, 3, resolution_level=level, with_near_far=True)
    assert tuple(no.shape) == tuple(fx[p + "shape"]) and nd.shape == no.shape
    assert torch.equal(no.reshape(-1, 3).cpu(), torch.from_numpy(fx[p + "origin"]).expand(no.shape[0] * no.shape[1], 3))
    sel = torch.from_numpy(fx[p + "idx"].astype(np.int64)).cuda()
    assert float((nd.reshape(-1, 3)[sel].cpu() - torch.from_numpy(fx[p + "dirs"])).abs().max()) < 2e-6
    assert float((near.reshape(-1, 1)[sel].cpu() - torch.from_numpy(fx[p + "near"])).abs().max()) < 1e-5
    assert float((far.reshape(-1, 1)[sel].cpu() - torch.from_numpy(fx[p + "far"])).abs().max()) < 1e-5
