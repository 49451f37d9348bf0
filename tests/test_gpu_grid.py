"""Device-side grid query / near-surface cell emission (neuraludf_b200/grid.py) against the reference's own
get_udf_normals_grid_slow (extract_mesh.py:18-105) driven with the same network callbacks, stored by
oracle/make_golden_device.py in tests/golden/device_outputs.npz (the full near-surface mask, seeded samples of the rest)."""
import numpy as np
import pytest
import torch

from tests.golden_util import load_device_golden
from tests.gpu_util import build_modules

pytestmark = pytest.mark.gpu


def test_grid_and_near_surface_cells_match_reference(golden):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from neuraludf_b200 import grid
    fx = load_device_golden()
    udf = build_modules(golden, "cuda")[0]
    N = int(fx["grid_n"])
    assert N == 48
    df, vec, samples = grid.get_udf_normals_grid_slow(udf, N=N, max_batch=1 << 15)
    assert df.shape == (N, N, N) and vec.shape == (N, N, N, 3) and samples.shape == (N ** 3, 7)
    idx = torch.from_numpy(fx["grid_idx"].astype(np.int64))
    ref = torch.from_numpy(fx["grid_samples"])
    assert float((samples[idx, :3] - ref[:, :3]).abs().max()) < 1e-6                # lattice coordinates
    assert float((samples[idx, 3] - ref[:, 3]).abs().max()) < 1e-6                  # same kernels, different batching
    assert float((samples[idx, 4:] - ref[:, 4:]).abs().max()) < 1e-4
    mask_ref = torch.from_numpy(np.unpackbits(fx["grid_mask_bits"])[:N ** 3].astype(bool))
    mask = (vec.abs().sum(-1) > 0).reshape(-1)
    assert torch.equal(mask, mask_ref) and int(mask.sum()) > 100                     # the same near-surface cells
    sidx = torch.from_numpy(fx["grid_surface_idx"].astype(np.int64))
    assert float((vec.reshape(-1, 3)[sidx] - torch.from_numpy(fx["grid_surface_vec"])).abs().max()) < 1e-4
    idx, normals = grid.near_surface_cells(udf, N)
    assert idx.numel() == int(mask.sum())
    assert float((normals.norm(dim=1) - 1).abs().max()) < 1e-4
    # slab partition (multi-GPU sweeps): two halves reproduce the whole grid
    half = N ** 3 // 2
    a = grid.udf_grid(udf, N, lo=0, hi=half)
    b = grid.udf_grid(udf, N, lo=half, hi=N ** 3)
    assert torch.equal(torch.cat([a, b]).cpu(), df.reshape(-1))
