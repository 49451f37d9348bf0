"""GPU unit tests of the tcgen05 (3xBF16 split) GEMM engine against fp64 matmuls, and end-to-end accuracy of the
renderer with the tensor engine enabled on the chains selected by the default mask."""
import ctypes

import pytest
import torch

from tests.gpu_util import build_modules, err_inf, parity, report, scale_inf

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _lib():
    from neuraludf_b200 import _lib as L
    return L, L.lib()


def _image(W, N, K, transposed, planes=2):
    L, lib = _lib()
    n = lib.nudf_tc_image_elems(N, K, planes)
    img = torch.zeros(n, dtype=torch.int16, device=DEV)
    L.check(lib.nudf_tc_prepare_weights(L.ptr(W), W.stride(0), N, K, transposed, planes, L.ptr(img), L.stream_ptr()), "prep")
    return img


@pytest.mark.parametrize("M,N,K", [(128, 256, 256), (300, 256, 256), (1000, 217, 256), (130, 128, 158), (128, 16, 39),
                                   (515, 257, 256), (4096, 256, 259), (77, 128, 64)])
def test_dense_forward_tc_vs_fp64(M, N, K):
    L, lib = _lib()
    g = torch.Generator().manual_seed(M + N + K)
    X = torch.randn(M, K, generator=g, dtype=torch.float64)
    W = torch.randn(N, K, generator=g, dtype=torch.float64) / K ** 0.5
    b = torch.randn(N, generator=g, dtype=torch.float64)
    ref = X @ W.t() + b
    Xd, Wd, bd = X.float().to(DEV).contiguous(), W.float().to(DEV).contiguous(), b.float().to(DEV)
    img = _image(Wd, N, K, 0)
    Y = torch.full((M, N), float("nan"), device=DEV)
    L.check(lib.nudf_dense_forward_tc(L.ptr(Xd), K, L.ptr(img), 2, L.ptr(bd), L.ptr(Y), N, M, N, K, 0, L.stream_ptr()), "dense_tc")
    torch.cuda.synchronize()
    e = err_inf(Y, ref) / scale_inf(ref)
    # 3-plane (6-product) variant: must be fp32-grade
    img3 = _image(Wd, N, K, 0, planes=3)
    Y3 = torch.full((M, N), float("nan"), device=DEV)
    L.check(lib.nudf_dense_forward_tc(L.ptr(Xd), K, L.ptr(img3), 3, L.ptr(bd), L.ptr(Y3), N, M, N, K, 0, L.stream_ptr()), "dense_tc3")
    e3 = err_inf(Y3, ref) / scale_inf(ref)
    report("tc.dense3[%d,%d,%d]" % (M, N, K), rel_tc3=e3)
    assert e3 < 2e-6, e3
    # fp32 engine for comparison
    Y0 = torch.empty(M, N, device=DEV)
    L.check(lib.nudf_dense_forward(L.ptr(Xd), K, L.ptr(Wd), K, L.ptr(bd), L.ptr(Y0), N, M, N, K, 0, L.stream_ptr()), "dense")
    e0 = err_inf(Y0, ref) / scale_inf(ref)
    report("tc.dense[%d,%d,%d]" % (M, N, K), rel_tc=e, rel_fp32=e0)
    assert torch.isfinite(Y).all()
    assert e < 5e-5, e
    # transposed image: Y2 = X2 @ W  (X2 [M,N], contraction over N)
    X2 = torch.randn(M, N, generator=g, dtype=torch.float64)
    ref2 = X2 @ W
    img2 = _image(Wd, K, N, 1)
    Y2 = torch.full((M, K), float("nan"), device=DEV)
    X2d = X2.float().to(DEV).contiguous()
    L.check(lib.nudf_dense_forward_tc(L.ptr(X2d), N, L.ptr(img2), 2, None, L.ptr(Y2), K, M, K, N, 0, L.stream_ptr()), "dense_tc_nn")
    e2 = err_inf(Y2, ref2) / scale_inf(ref2)
    report("tc.dense_nn[%d,%d,%d]" % (M, N, K), rel_tc=e2)
    assert e2 < 5e-5, e2


@pytest.mark.parametrize("P,n_out,n_in", [(65536, 256, 256), (20000, 257, 256), (65536, 3, 259)])
def test_wgrad_is_bitwise_reproducible(P, n_out, n_in):
    """The split-K partials are added in a fixed order: the same inputs give the same bits on every call, accumulating
    into a non-zero destination as the training step does."""
    L, lib = _lib()
    g = torch.Generator().manual_seed(P + n_in)
    dZd = torch.randn(P, n_out, generator=g).to(DEV)
    Xd = torch.randn(P, n_in, generator=g).to(DEV)
    base = torch.randn(n_out, n_in, generator=g).to(DEV)
    for engine in (1, 0):
        outs = []
        for _ in range(3):
            dW = base.clone()
            L.check(lib.nudf_wgrad(L.ptr(dZd), n_out, L.ptr(Xd), n_in, n_out, n_in, P, L.ptr(dW), n_in, engine, L.stream_ptr()),
                    "wgrad")
            outs.append(dW)
        torch.cuda.synchronize()
        assert all(torch.equal(o, outs[0]) for o in outs[1:]), engine
        assert not torch.equal(outs[0], base)


@pytest.mark.parametrize("P,n_out,n_in", [(1024, 256, 256), (5000, 217, 256), (3000, 128, 259), (700, 257, 256), (4096, 256, 39)])
def test_wgrad_tc_vs_fp64(P, n_out, n_in):
    L, lib = _lib()
    g = torch.Generator().manual_seed(P + n_out)
    dZ = torch.randn(P, n_out, generator=g, dtype=torch.float64)
    X = torch.randn(P, n_in, generator=g, dtype=torch.float64)
    ref = dZ.t() @ X
    dZd, Xd = dZ.float().to(DEV).contiguous(), X.float().to(DEV).contiguous()
    for engine in (1, 0):
        dW = torch.zeros(n_out, n_in, device=DEV)
        L.check(lib.nudf_wgrad(L.ptr(dZd), n_out, L.ptr(Xd), n_in, n_out, n_in, P, L.ptr(dW), n_in, engine, L.stream_ptr()), "wgrad")
        e = err_inf(dW, ref) / scale_inf(ref)
        report("tc.wgrad[%d,%d,%d].engine%d" % (P, n_out, n_in, engine), rel=e)
        assert e < 5e-5, (engine, e)


def _planes(L, lib, x):
    rows, cols = x.shape
    buf = torch.empty(lib.nudf_planes_elems(rows, cols) + 512, dtype=torch.int16, device=DEV)
    off = (-buf.data_ptr() % 1024) // 2
    pl = buf[off:off + lib.nudf_planes_elems(rows, cols)]
    pl.fill_(0x7FC0)                                  # bf16 NaN everywhere: pad rows must be rewritten by the packer
    L.check(lib.nudf_pack_planes(L.ptr(x), x.stride(0), rows, cols, L.ptr(pl), L.stream_ptr()), "pack")
    return pl


@pytest.mark.parametrize("rows,cols", [(1, 5), (130, 64), (257, 217), (4096, 256)])
def test_planes_round_trip(rows, cols):
    """fp32 -> split-bf16 planes -> fp32: 16 mantissa bits survive (relative error <= 2^-16)"""
    L, lib = _lib()
    g = torch.Generator().manual_seed(rows + cols)
    x = (torch.randn(rows, cols, generator=g) * torch.logspace(-3, 3, cols)[None, :]).to(DEV).contiguous()
    pl = _planes(L, lib, x)
    y = torch.full_like(x, float("nan"))
    L.check(lib.nudf_unpack_planes(L.ptr(pl), rows, cols, L.ptr(y), y.stride(0), L.stream_ptr()), "unpack")
    assert float(((y - x).abs() / x.abs().clamp(min=1e-30)).max()) <= 2.0 ** -16


@pytest.mark.parametrize("M,N,K,act", [(4096, 256, 256, 2), (300, 217, 256, 0), (129, 256, 39, 0), (1000, 39, 217, 0), (65536, 256, 256, 2)])
def test_dense_planes_vs_fp64(M, N, K, act):
    """one layer on the plane-fed weights-resident kernel (A operand fetched as plane blocks by cp.async.bulk)"""
    L, lib = _lib()
    g = torch.Generator().manual_seed(M + N + K)
    X = torch.randn(M, K, generator=g, dtype=torch.float64) * 0.5
    W = torch.randn(N, K, generator=g, dtype=torch.float64) / K ** 0.5
    b = torch.randn(N, generator=g, dtype=torch.float64) * 0.1
    ref = X @ W.t() + b
    if act == 2:
        ref = torch.nn.functional.softplus(ref, beta=100)
    Xd = X.float().to(DEV).contiguous()
    rows_pad = (M + 127) // 128 * 128
    buf = torch.empty(lib.nudf_planes_elems(rows_pad, K) + 512, dtype=torch.int16, device=DEV)
    off = (-buf.data_ptr() % 1024) // 2
    pl = buf[off:off + lib.nudf_planes_elems(rows_pad, K)]
    pl.fill_(0x7FC0)                                  # NaN in the rows beyond M: they must not leak into valid rows
    L.check(lib.nudf_pack_planes(L.ptr(Xd), K, M, K, L.ptr(pl), L.stream_ptr()), "pack")
    img = _image(W.float().to(DEV).contiguous(), N, K, 0)
    Y = torch.full((M, N), float("nan"), device=DEV)
    bd = b.float().to(DEV)
    L.check(lib.nudf_dense_forward_planes(L.ptr(pl), L.ptr(img), L.ptr(bd), L.ptr(Y), N, M, N, K, act, L.stream_ptr()), "dense_planes")
    e = err_inf(Y, ref) / scale_inf(ref)
    report("tc.dense_planes[%d,%d,%d]" % (M, N, K), rel=e)
    assert e < 3e-5, e


@pytest.mark.parametrize("P,n_out,n_in", [(4096, 256, 256), (1000, 128, 64), (70, 257, 39), (65536, 256, 256), (333, 217, 256)])
def test_wgrad_planes_vs_fp64(P, n_out, n_in):
    """weight-gradient contraction with both operands fetched as plane blocks (MN-major UMMA operands)"""
    L, lib = _lib()
    g = torch.Generator().manual_seed(P + n_out)
    dZ = torch.randn(P, n_out, generator=g, dtype=torch.float64)
    X = torch.randn(P, n_in, generator=g, dtype=torch.float64)
    ref = dZ.t() @ X
    dZp = _planes(L, lib, dZ.float().to(DEV).contiguous())
    Xp = _planes(L, lib, X.float().to(DEV).contiguous())
    dW = torch.zeros(n_out, n_in, device=DEV)
    L.check(lib.nudf_wgrad_planes(L.ptr(dZp), L.ptr(Xp), n_out, n_in, P, L.ptr(dW), n_in, L.stream_ptr()), "wgrad_planes")
    e = err_inf(dW, ref) / scale_inf(ref)
    report("tc.wgrad_planes[%d,%d,%d]" % (P, n_out, n_in), rel=e)
    assert e < 5e-5, e


@pytest.mark.parametrize("mask", [0, 62, -1, 63])
def test_render_core_accuracy_by_tc_mask(golden, mask):
    """How far each choice of tensor-engine chains moves render_core from the fp64 reference (reported; the default
    mask must stay within the parity bounds, the all-chains mask 63 is informational)."""
    from neuraludf_b200.models.udf_renderer_blending import UDFRendererBlending
    L, lib = _lib()
    old_engine, old_mask = lib.nudf_get_engine(), lib.nudf_get_tc_mask()
    lib.nudf_set_engine(1)
    if mask < 0:
        mask = lib.nudf_default_tc_mask()          # the shipped configuration
    lib.nudf_set_tc_mask(mask)
    try:
        g = golden
        udf, col, nerf, var, beta = build_modules(g, DEV)
        ren = UDFRendererBlending(nerf, udf, var, col, beta, n_samples=64, n_importance=0, n_outside=0, up_sample_steps=1,
                                  perturb=0.0)
        o, d = g.t("rays_o").to(DEV), g.t("rays_d").to(DEV)
        near, far = g.t("near").to(DEV), g.t("far").to(DEV)
        S = 128
        z = (near + (far - near) * torch.linspace(0.0, 1.0, S, device=DEV)[None, :]).contiguous()
        sd = ((far - near) / S).mean().item()
        ret = ren.render_core(o, d, z, sd, udf, var, col, beta_network=beta, cos_anneal_ratio=0.5, flip_saturation=0.3)
        tgt = torch.full((64, 3), 0.4, device=DEV)
        loss = ((ret["color"] - tgt).abs().mean() + 0.01 * (ret["color_base"] - tgt).abs().mean()
                + 0.1 * ret["gradient_error"] + 1e-3 * ret["sparse_error"] + 0.05 * ret["gradient_error_near_surface"]
                + 0.1 * ((ret["weight_sum"][:, 0] - 0.5) ** 2).mean())
        loss.backward()
        from oracle.make_golden import GRAD_STRIDE
        stats = {}
        for k in ("udf", "gradients", "color", "color_base", "depth", "weights", "alpha", "sparse_error", "gradient_error"):
            r64, r32 = g.t("rc_%s_f64" % k), g.t("rc_%s_f32" % k)
            stats[k] = err_inf(ret[k].reshape(r64.shape), r64) / scale_inf(r64)
            stats[k + "_refnoise"] = err_inf(r32, r64) / scale_inf(r64)
        worst = 0.0
        for mn, m in (("udf", udf), ("color", col)):
            for pn, p in m.named_parameters():
                key = "rc_grad.%s.%s_f64" % (mn, pn)
                ref = g.t(key) if g.has(key) else g.t(key + "_sub")
                new = p.grad.cpu() if g.has(key) else p.grad.reshape(-1)[::GRAD_STRIDE].cpu()
                worst = max(worst, err_inf(new, ref) / scale_inf(ref))
        stats["dparam_worst"] = worst
        report("tc.render_core.mask%d" % mask, **stats)
        assert all(v == v for v in stats.values())
        if mask != 63:
            # every reported tensor is held to the SURVEY 8(c) bound: max(tol, k x the reference's own fp32-vs-fp64 noise)
            assert stats["dparam_worst"] < 5e-3
            for k in ("udf", "gradients", "gradient_error"):
                assert stats[k] <= max(1e-4, 2.0 * stats[k + "_refnoise"]), (k, stats[k])
            for k in ("color", "color_base", "depth", "weights", "alpha"):
                assert stats[k] <= max(2e-4, 2.5 * stats[k + "_refnoise"]), (k, stats[k])
            assert stats["sparse_error"] <= max(2e-4, 4.0 * stats["sparse_error_refnoise"]), stats["sparse_error"]
    finally:
        lib.nudf_set_engine(old_engine)
        lib.nudf_set_tc_mask(old_mask)


def test_nerf_and_color_on_tensor_engine_vs_oracle(golden):
    """NeRF++ and colour networks with the tensor engine enabled (default chain mask) against fp64 oracle autograd."""
    from oracle import oracle_torch as O
    from tests.gpu_util import oracle_params
    L, lib = _lib()
    old_engine, old_mask = lib.nudf_get_engine(), lib.nudf_get_tc_mask()
    lib.nudf_set_engine(1)
    lib.nudf_set_tc_mask(126)
    try:
        g = golden
        _, col, nerf, _, _ = build_modules(g, DEV)
        gen = torch.Generator().manual_seed(21)
        P = 700
        pts4 = torch.randn(P, 4, generator=gen, dtype=torch.float64)
        pts4 = pts4 / pts4[:, :3].norm(dim=1, keepdim=True)
        dirs = torch.randn(P, 3, generator=gen, dtype=torch.float64)
        dirs = dirs / dirs.norm(dim=1, keepdim=True)
        ab = torch.randn(P, 1, generator=gen, dtype=torch.float64)
        rb = torch.randn(P, 3, generator=gen, dtype=torch.float64)
        # the 2^9 positional-encoding frequency amplifies fp32 input rounding to ~1e-4, which flips ReLU gates: the fp32
        # run of the oracle is the yardstick for that noise (parity protocol), the fp64 run the arbiter
        res = {}
        for dt in (torch.float64, torch.float32):
            pd = oracle_params(g, "nerf", dt, True)
            oa, orgb = O.nerf_mlp(pd, g.nerf_c, pts4.to(dt), dirs.to(dt))
            gr = dict(zip(pd.keys(), torch.autograd.grad((oa * ab.to(dt)).sum() + (orgb * rb.to(dt)).sum(), list(pd.values()))))
            res[dt] = (oa.detach(), orgb.detach(), gr)
        oa, orgb, gr = res[torch.float64]
        oa32, orgb32, gr32 = res[torch.float32]
        a, rgb = nerf(pts4.float().to(DEV), dirs.float().to(DEV))
        parity("tc.nerf.alpha", a, oa, oa32, tol=1e-4)
        parity("tc.nerf.rgb", rgb, orgb, orgb32, tol=1e-4)
        ((a * ab.float().to(DEV)).sum() + (rgb * rb.float().to(DEV)).sum()).backward()
        for k, v in nerf.named_parameters():
            parity("tc.nerf.dparam." + k, v.grad, gr[k], gr32[k], tol=5e-4, noise_mult=3.0)
        # colour network
        pts = g.t("col_pts").to(DEV); d3 = g.t("col_dirs").to(DEV); feat = g.t("col_feat").to(DEV).requires_grad_(True)
        cb, c, bl = col(pts, None, d3, feat)
        parity("tc.color.base", cb, g.t("col_base_f64"), None, tol=1e-4)
        parity("tc.color.color", c, g.t("col_color_f64"), None, tol=1e-4)
        parity("tc.color.blend", bl, g.t("col_blend_f64"), None, tol=1e-4)
        bars = [torch.randn(t.shape, generator=gen, dtype=torch.float64) for t in (cb, c, bl)]
        pc = oracle_params(g, "color", torch.float64, True)
        f64 = g.t("col_feat", torch.float64).clone().requires_grad_(True)
        o = O.color_mlp(pc, g.col_c, g.t("col_pts", torch.float64), g.t("col_dirs", torch.float64), f64)
        grc = torch.autograd.grad(sum((x * b).sum() for x, b in zip(o, bars)), list(pc.values()) + [f64])
        grc = dict(zip(list(pc.keys()) + ["feat"], grc))
        sum((x * b.float().to(DEV)).sum() for x, b in zip((cb, c, bl), bars)).backward()
        parity("tc.color.dfeat", feat.grad, grc["feat"], None, tol=5e-4)
        for k, v in col.named_parameters():
            parity("tc.color.dparam." + k, v.grad, grc[k], None, tol=5e-3)
    finally:
        lib.nudf_set_engine(old_engine)
        lib.nudf_set_tc_mask(old_mask)


def test_degenerate_sizes():
    """empty / single-point / ragged inputs go through both engines without touching memory they should not"""
    L, lib = _lib()
    from neuraludf_b200.models import fields as F
    for engine in (0, 1):
        lib.nudf_set_engine(engine)
        udf = F.UDFNetwork(d_in=3, d_out=257, d_hidden=64, n_layers=4, skip_in=(2,), multires=6).to(DEV)
        for P in (0, 1, 127, 129, 130):
            x = torch.rand(P, 3, device=DEV) - 0.5
            out, grad = udf.value_and_gradient(x)
            assert out.shape == (P, 257) and grad.shape == (P, 3)
            assert torch.isfinite(out).all() and torch.isfinite(grad).all()
            if P > 0:
                (out.sum() + grad.sum()).backward()
                assert all(torch.isfinite(p.grad).all() for p in udf.parameters())
    lib.nudf_set_engine(1)
