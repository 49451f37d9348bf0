"""CPU checks of the test-only runner environment (tests/runner_env.py): the HOCON-subset reader parses the reference's
four shipped confs (stored unmodified under tests/golden/confs) into the values the runner reads, the nudf modules accept
those conf blocks as constructor kwargs (exp_runner_blending.py:125-146), and the synthetic DTU-layout dataset has the
files / camera keys dataset.py loads."""
import os

import numpy as np
import pytest

from tests import runner_env
from tests.golden_util import GOLDEN

CONFS = ["confs/udf_dtu_blending.conf", "confs/udf_dtu_blending_ft.conf", "confs/udf_garment_blending.conf",
         "confs/udf_garment_blending_ft.conf"]


@pytest.mark.parametrize("name", CONFS)
def test_hocon_lite_parses_reference_confs(name):
    text = open(os.path.join(GOLDEN, name)).read().replace("CASE_NAME", "scan24")
    c = runner_env.ConfigFactory.parse_string(text)
    assert c["general.model_type"] == "udf"
    assert isinstance(c["general.recording"], list) and c["general.recording"][0] == "./"
    assert c.get_int("train.batch_size") == 512
    assert 1e-5 <= c.get_float("train.learning_rate") <= 1e-3
    assert c.get_bool("train.use_white_bkgd") is False
    assert c.get_string("dataset.dataset_name", default="general") in ("general", "dtu", "deepfashion3d")
    assert c.get_float("train.not_there", default=1.5) == 1.5
    with pytest.raises(KeyError):
        c.get_int("train.not_there")
    u = c["model.udf_network"]
    assert u["d_hidden"] == 256 and u["n_layers"] == 8 and u["skip_in"] == [4] and u["geometric_init"] is True
    assert c["model.nerf"]["skips"] == [4] and c["model.nerf"]["use_viewdirs"] is True
    assert c["model.beta_network"]["beta_min"] == pytest.approx(5e-5)
    r = c["model.udf_renderer"]
    assert r["n_samples"] == 64 and r["sdf2alpha_type"] == "numerical" and r["upsampling_type"] in ("classical", "mix")
    c["train"]["learning_rate"] = 1e-3                      # the runner's command-line overrides (:48-53)
    assert c.get_float("train.learning_rate") == 1e-3
    c["dataset.data_dir"] = c["dataset.data_dir"].replace("scan24", "x")
    assert "x" in c.get_string("dataset.data_dir")
    assert "udf_network" in runner_env.HOCONConverter.to_hocon(c)


@pytest.mark.parametrize("name", CONFS)
def test_modules_accept_conf_blocks(name):
    """exp_runner_blending.py:125-146 splats the conf blocks into the constructors"""
    from neuraludf_b200.models import fields as F
    from neuraludf_b200.models.udf_renderer_blending import UDFRendererBlending
    c = runner_env.ConfigFactory.parse_string(open(os.path.join(GOLDEN, name)).read())
    nerf = F.NeRF(**c["model.nerf"])
    udf = F.UDFNetwork(**c["model.udf_network"])
    var = F.SingleVarianceNetwork(**c["model.variance_network"])
    col = F.ResidualRenderingNetwork(**c["model.rendering_network"])
    beta = F.BetaNetwork(**c["model.beta_network"])
    ren = UDFRendererBlending(nerf, udf, var, col, beta, **c["model.udf_renderer"])
    assert ren.n_samples == c["model.udf_renderer"]["n_samples"]
    assert sum(p.numel() for p in udf.parameters()) == 529076


def test_synthetic_dtu_layout(tmp_path):
    root = runner_env.write_synthetic_dtu(str(tmp_path / "case"), n_images=4, width=32, height=24)
    assert sorted(os.listdir(os.path.join(root, "image"))) == ["000.png", "001.png", "002.png", "003.png"]
    assert len(os.listdir(os.path.join(root, "mask"))) == 4
    cams = np.load(os.path.join(root, "cameras.npz"))
    for i in range(4):
        assert cams["world_mat_%d" % i].shape == (4, 4) and cams["scale_mat_%d" % i].shape == (4, 4)
    import cv2
    K, R, t = cv2.decomposeProjectionMatrix(cams["world_mat_0"][:3, :4].astype(np.float32))[:3]
    c = (t[:3] / t[3])[:, 0]
    assert abs(np.linalg.norm(c) - 2.5) < 1e-3              # the camera sits outside the unit sphere (dataset.py:329-335)
    m = cv2.imread(os.path.join(root, "mask", "000.png"))
    assert 0.02 < (m > 0).mean() < 0.5                      # the sphere is visible and does not fill the image
    conf = runner_env.write_conf(GOLDEN, str(tmp_path / "t.conf"), root + "/", str(tmp_path / "exp") + "/", 3)
    c = runner_env.ConfigFactory.parse_string(open(conf).read())
    assert c.get_int("train.end_iter") == 3 and c.get_string("dataset.data_dir") == root + "/"
