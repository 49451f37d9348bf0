#!/usr/bin/env python
"""Benchmark of the NeuralUDF volume-rendering hot path (BASELINE.json metric: ray-samples/s, render_core fwd+bwd).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], "C2" in SURVEY.md 8(d)): 512 rays x 128 uniform samples per GPU, UDF 8x256 +
ResidualRenderingNetwork 2x(4x128) (reference conf dims), synthetic seeded sphere scene.  One step = what one training
iteration of the reference does on this path: render_core forward, backward of  L1 colour + 0.01 L1 base colour + 0.1 eikonal
(exp_runner_blending.py:330-371), and the Adam update (exp_runner_blending.py:373-375) -- so the per-step weight-norm fold
and tensor-engine weight-image build are INSIDE the timed region.  For N > 1 (torchrun, one rank per GPU) rays are sharded
(weak scaling: 512 rays per GPU) and the gradients are all-reduced over NCCL before the update.

Prints ONE JSON line (rank 0):
  value      device-resident throughput (CUDA events on the launching stream, max over ranks);
  e2e        the same step driven from pinned HOST buffers through the public module API, H2D / D2H inside the timed region;
  families   per-kernel-family device time of the SAME step (cudaEvent pairs recorded by the library around each of its
             launches, nudf_set_launch_timing), share of the step, algorithmic TFLOP/s, fraction of the measured bf16 peak;
  roofline   the family with the largest share (i.e. picked from what the step actually launches);
  cpu_baseline  the UNMODIFIED reference's render_core (staged copy oracle/_ref, see oracle/make_ref.py) on the host cores,
             all 512 rays, thread count swept at the timed size; falls back to the pinned oracle port if no staged copy exists;
  workloads  the other BASELINE.json configs (C1 forward, C3 blending step, C4 whole training step incl. strong-scaling size,
             C5 256^3 grid sweep) so that the driver records them as well.
`--impl reference` times the same CPU arm alone; under torchrun only rank 0 works.
`--dump-outputs DIR` writes what the last timed C2 step computed (render_core outputs, loss, parameter gradients and the
parameters after the Adam update) as DIR/<name>.npy, so that two builds can be compared output for output on identical
seeded inputs.
"""
import argparse
import ctypes
import datetime
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_RAYS, N_SAMPLES = 512, 128
FLOP_FWD = 2274560           # per ray-sample, SURVEY 8(d): UDF value 1 049 088 + input-gradient sweep 918 016 + colour 307 456
FLOP_FWD_BWD = 6823680       # forward + backward (data-grad + weight-grad of every contraction)

# algorithmic MACs per sample point of the C2 step, by kernel family (layer dims of SURVEY App. B):
#   F value chain = all 9 layers; R reverse sweep / T tangent chain = layers 0..7; B backward chain = layers 8..1;
#   weight gradients = D^T Adot (layers 0..7) + Zbar^T A (layers 0..8); colour net: forward + data-grad + weight-grad
_UDF_MAC = [256 * 39, 256 * 256, 256 * 256, 217 * 256, 256 * 256, 256 * 256, 256 * 256, 256 * 256, 257 * 256]
_MAC_F = sum(_UDF_MAC)
_MAC_R = sum(_UDF_MAC[:8])
_MAC_B = sum(_UDF_MAC[1:])
_MAC_COL = 153728
FAMILY_MAC = {"udf_fwd_chain_fused": _MAC_F + _MAC_R, "udf_bwd_chain_fused": _MAC_R + _MAC_B, "tc_layer_reverse_sweep": _MAC_R,
              "tc_layer_tangent": _MAC_R, "tc_layer_backward": _MAC_B, "tc_weight_gradient": _MAC_R + _MAC_F + _MAC_COL}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def ncu_traffic(kernel_substr, launch=0):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes per launch) of the `launch`-th captured launch of a kernel from the
    newest committed `ncu --set full` summary under profiles/ (None if not captured)."""
    import glob
    best = None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    norm = lambda t: t.replace("nudf::", "").replace("tc::", "").replace("chain::", "").replace(" ", "")
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_gemm_kernels.txt")) +
                    glob.glob(os.path.join(ROOT, "profiles", "r*_kernel.txt"))):
        cur, rd, wr, seen, found = None, None, None, -1, None
        for line in open(f):
            if line.startswith("== "):
                cur, rd, wr = None, None, None
                if norm(kernel_substr) in norm(line):
                    seen += 1
                    if seen == launch:
                        cur = line
            elif cur:
                parts = line.split()
                if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    v = float(parts[1].replace(",", "")) * unit.get(parts[2], 1.0)
                    if parts[0].endswith("read.sum"):
                        rd = v
                    else:
                        wr = v
                if rd is not None and wr is not None:
                    found = rd + wr
                    cur = None
        if found is not None:
            best = found
    return best


def nerf_module(device):
    from neuraludf_b200 import synthetic as O
    from neuraludf_b200.models import fields as F
    nerf = F.NeRF(D=8, d_in=4, d_in_view=3, W=256, multires=10, multires_view=4, output_ch=4, skips=[4], use_viewdirs=True)
    nerf.load_state_dict(O.make_nerf_params(O.nerf_cfg(), seed=2))
    return nerf.to(device)


def scene(device, small_udf=False):
    from neuraludf_b200 import synthetic as O
    from neuraludf_b200.models import fields as F
    udf_c = O.udf_cfg(d_hidden=128, n_layers=4) if small_udf else O.udf_cfg()
    col_c = O.color_cfg()
    udf = F.UDFNetwork(d_in=3, d_out=257, d_hidden=udf_c["d_hidden"], n_layers=udf_c["n_layers"], skip_in=(4,), multires=6,
                       bias=0.5, scale=1.0, geometric_init=True, weight_norm=True, udf_type="abs")
    udf.load_state_dict(O.make_udf_params(udf_c, seed=3 if small_udf else 0))
    col = F.ResidualRenderingNetwork(d_feature=256, mode="no_normal", d_in=6, d_out=3, d_hidden=128, n_layers=4,
                                     weight_norm=True, multires_view=4, squeeze_out=True, blending_cand_views=10)
    col.load_state_dict(O.make_color_params(col_c, seed=1))
    var = F.SingleVarianceNetwork(0.6)
    beta = F.BetaNetwork(init_var_beta=0.5, init_var_gamma=0.3, init_var_zeta=0.3, beta_min=5e-5,
                         requires_grad_beta=True, requires_grad_gamma=False, requires_grad_zeta=False)
    return [m.to(device) for m in (udf, col, var, beta)]


def make_optimizer(udf, others, fused=True):
    """Adam with the reference's parameter groups and learning rates (exp_runner_blending.py:130-139, confs: 5e-4 / geo 1e-4)."""
    groups = [{"params": [p for p in udf.parameters() if p.requires_grad], "lr": 1e-4},
              {"params": [p for m in others for p in m.parameters() if p.requires_grad], "lr": 5e-4}]
    try:
        return torch.optim.Adam(groups, fused=fused, capturable=fused)      # capturable: the step can live in a CUDA graph
    except Exception:
        return torch.optim.Adam(groups)


def rays(seed, device=None, n_rays=N_RAYS, n_samples=N_SAMPLES):
    from neuraludf_b200 import synthetic as O
    o, d, near, far = O.make_rays(n_rays, seed=seed)
    z = near + (far - near) * torch.linspace(0.0, 1.0, n_samples)[None, :]
    sd = float(((far - near) / n_samples).mean())
    if device is not None:
        o, d, z = o.to(device), d.to(device), z.to(device).contiguous()
    return o, d, z, sd


class Clocks:
    """nvidia-smi sampler (B200_PROFILING.md clocks line).  Started BEFORE the warm-up (nvidia-smi needs ~0.2 s to come
    up), every sample is time-stamped, and only the samples inside the [begin(), end()] wall-clock window -- the timed
    region -- are reported."""

    def __init__(self, idx):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.t0 = self.t1 = None
        q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(idx), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                       "-lms", "10"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def begin(self):
        deadline = time.time() + 2.0            # the first sample must exist before the timed region starts
        while self.p is not None and os.path.getsize(self.f.name) == 0 and time.time() < deadline:
            time.sleep(0.01)
        self.t0 = datetime.datetime.now()

    def end(self):
        self.t1 = datetime.datetime.now()

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        parsed = []
        for r in rows:
            try:
                ts = datetime.datetime.strptime(r[0].strip(), "%Y/%m/%d %H:%M:%S.%f")
                parsed.append((ts, float(r[1]), float(r[2]), [n for n, v in zip(names, r[3:7])
                                                               if v.strip().lower() == "active"]))
            except Exception:
                pass
        slack = datetime.timedelta(milliseconds=15)
        inside = [x for x in parsed if self.t0 is not None and self.t0 - slack <= x[0] <= self.t1 + slack]
        window = "timed region"
        if not inside and parsed and self.t0 is not None:
            # region shorter than the sampling period: the sample closest to it
            inside = [min(parsed, key=lambda x: abs((x[0] - self.t0).total_seconds()))]
            window = "nearest sample (timed region shorter than the sampling period)"
        sm = sorted(x[1] for x in inside)
        reasons = sorted({n for x in inside for n in x[3]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(x[2] for x in inside) if inside else None,
                "reasons": reasons, "samples": len(sm), "window": window}


def loss_fn(ret, tgt):
    return ((ret["color"] - tgt).abs().mean() + 0.01 * (ret["color_base"] - tgt).abs().mean()
            + 0.1 * ret["gradient_error"])


def _timed(fn, steps, warmup):
    """ms per call of fn(), CUDA events on the current stream, after `warmup` untimed calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def read_families(lib, n_steps, ms_step, P, pk):
    """Per-family table from the library's event pairs (see the module docstring)."""
    from neuraludf_b200 import _lib
    nf = lib.nudf_launch_family_count()
    ms = (ctypes.c_float * nf)()
    cnt = (ctypes.c_int32 * nf)()
    _lib.check(lib.nudf_read_launch_timing(ms, cnt), "nudf_read_launch_timing")
    fam = {}
    tot = 0.0
    for i, name in enumerate(_lib.LAUNCH_FAMILIES[:nf]):
        if cnt[i] == 0:
            continue
        us = ms[i] * 1e3 / n_steps
        tot += us
        row = {"launches_per_step": cnt[i] / n_steps, "us_per_step": us, "share": us / (ms_step * 1e3)}
        if name in FAMILY_MAC:
            fl = 2.0 * FAMILY_MAC[name] * P
            row["algorithmic_tflops"] = fl / (us * 1e-6) / 1e12
            row["frac_of_bf16_sustained"] = row["algorithmic_tflops"] / pk["bf16_sustained"]
            row["us_per_launch"] = us / (cnt[i] / n_steps)
        fam[name] = row
    fam["torch_glue_and_idle"] = {"us_per_step": ms_step * 1e3 - tot, "share": 1.0 - tot / (ms_step * 1e3),
                                  "note": "step time minus the library's kernels: torch element-wise / reduction / optimiser "
                                          "kernels, launch gaps"}
    return fam


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, ret, loss, named_modules):
    """rank 0: every tensor the caller of the timed step receives, as float32 (float64 stays float64) .npy files."""
    arrays = {"loss": loss}
    arrays.update(("out." + k, v) for k, v in ret.items() if isinstance(v, torch.Tensor))
    for mname, m in named_modules:
        for pname, p in m.named_parameters():
            arrays["param.%s.%s" % (mname, pname)] = p
            if p.grad is not None:
                arrays["grad.%s.%s" % (mname, pname)] = p.grad
    arrays = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32).contiguous().numpy()
              for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return total


def run_ours(args):
    import torch.distributed as dist
    from neuraludf_b200 import _lib
    from neuraludf_b200.models.udf_renderer_blending import UDFRendererBlending
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()
    udf, col, var, beta = scene(dev)
    if args.workload in ("c3", "c4", "c5", "c1"):
        fn = {"c3": run_c3, "c4": run_c4, "c5": run_c5, "c1": run_c1}[args.workload]
        res = fn(args, dev, lib, rank, world)
        if rank == 0:
            print(json.dumps(res), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return None
    params = [p for m in (udf, col, var, beta) for p in m.parameters() if p.requires_grad]
    ren = UDFRendererBlending(None, udf, var, col, beta, n_samples=N_SAMPLES, n_importance=0, n_outside=0,
                              up_sample_steps=1, perturb=0.0)
    ren.want_diagnostics = False      # per-sample debug tensors are only consumed by validate() / visualize_one_ray()
    o, d, z, sd = rays(seed=rank, device=dev)
    tgt = torch.full((N_RAYS, 3), 0.4, device=dev)
    from neuraludf_b200.dp import GradBucket
    bucket = GradBucket(params, modules=(udf, col))      # backward kernels write dg / dv / db straight into the flat bucket
    opt = make_optimizer(udf, (col, var, beta))

    # outputs of the latest step (inside a graph: its static tensors), detached: a reference into the autograd graph of an
    # eager step would keep its AccumulateGrad nodes alive into the capture on the side stream and invalidate the capture
    last = {}

    def compute(o_, d_, z_):
        opt.zero_grad(set_to_none=True)
        ret = ren.render_core(o_, d_, z_, sd, udf, var, col, beta_network=beta, cos_anneal_ratio=0.5)
        loss = loss_fn(ret, tgt)
        loss.backward()
        last["ret"] = {k: v.detach() if isinstance(v, torch.Tensor) else v for k, v in ret.items()}
        last["loss"] = loss.detach()
        return loss

    def step(o_, d_, z_):
        loss = compute(o_, d_, z_)
        if world > 1:
            bucket.allreduce_mean()                    # NCCL all-reduce of the flat gradient bucket over NVLink
        opt.step()                                     # Adam: parameters change => fold + weight images rebuilt next step
        return loss

    # CUDA-graph replay.  One GPU: the whole step (forward, backward, Adam) is one graph.  Several GPUs: the graph holds forward
    # + backward only; the NCCL all-reduce of the flat bucket and Adam are launched after each replay (NCCL calls are kept out
    # of captured graphs; the per-region overlap of the eager path is given up for one 2.8 MB collective).
    def graph_body(o_, d_, z_):
        return step(o_, d_, z_) if world == 1 else compute(o_, d_, z_)

    def replay_step():
        graph.replay()
        if world > 1:
            bucket.allreduce_replayed()
            opt.step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def stage(msg):                                    # NUDF_BENCH_TRACE=1: progress on stderr (multi-GPU debugging aid)
        if os.environ.get("NUDF_BENCH_TRACE"):
            print("[bench rank %d] %s" % (rank, msg), file=sys.stderr, flush=True)

    clocks = Clocks(local) if rank == 0 else None
    stage("warm-up")
    for _ in range(max(args.warmup, 3)):
        step(o, d, z)
    barrier()
    stage("eager loop")
    # ---- eager loop: every kernel launched from Python (ctypes / torch) each step ----
    l0 = lib.nudf_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step(o, d, z)
    e1.record()
    barrier()
    ms_eager = e0.elapsed_time(e1)
    launches = lib.nudf_launch_count() - l0
    # ---- the same step captured ONCE into a CUDA graph and replayed (no host work per step; the step has no host read) ----
    graph, g_in, g_loss, graph_err, static_grads = None, None, None, None, []
    stage("graph capture")
    if not args.no_graph:
        try:
            g_in = [t.clone() for t in (o, d, z)]
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            bucket.overlap = world == 1                # no collective is issued from inside backward while capturing
            with torch.cuda.stream(side):
                for _ in range(2):
                    graph_body(*g_in)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                g_loss = graph_body(*g_in)
            static_grads = [(p, p.grad) for p in params]     # the tensors the captured kernels write
            for _ in range(3):
                replay_step()
            barrier()
        except Exception as e:                         # capture not possible here: the eager number stands
            graph, graph_err = None, "%s: %s" % (type(e).__name__, str(e)[:200])
            torch.cuda.synchronize()
        if graph is None:
            bucket.overlap = True
    stage("timed loop (graph=%s)" % (graph is not None))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if clocks:
        clocks.begin()
    barrier()
    e0.record()
    for _ in range(args.steps):
        if graph is not None:
            replay_step()
        else:
            step(o, d, z)
    e1.record()
    barrier()
    if clocks:
        clocks.end()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:               # before any further step changes the parameters
        dump_outputs(args.dump_outputs, last["ret"], last["loss"],
                     (("udf", udf), ("color", col), ("variance", var), ("beta", beta)))

    if args.quick:
        if rank == 0:
            print(json.dumps({"quick": True, "ms_per_step": ms / args.steps, "ms_per_step_eager": ms_eager / args.steps,
                              "cuda_graph": graph is not None, "gpu_launches": int(launches),
                              "value": world * N_RAYS * N_SAMPLES * args.steps / (ms * 1e-3)}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return None

    # ---- the same steps again with the library's per-family event pairs switched on ----
    # (every rank runs the steps -- they contain the gradient all-reduce --, rank 0 alone records the events)
    stage("family timing")
    fam = None
    n_fam_steps = min(args.steps, 10)
    if rank == 0:
        lib.nudf_set_launch_timing(1)
    for _ in range(n_fam_steps):
        step(o, d, z)
    torch.cuda.synchronize()
    if graph is not None:                              # the eager steps re-created the .grad tensors: point the parameters back
        for p, g in static_grads:                      # at the ones the graph writes (the eager finish of replay_step reads them)
            p.grad = g
    if rank == 0:
        fam = read_families(lib, n_fam_steps, ms / args.steps, N_RAYS * N_SAMPLES, peaks())
        lib.nudf_set_launch_timing(0)
    barrier()

    # ---- end-to-end: host (pinned) inputs, H2D + D2H inside the timed region, through the public module API ----
    ho, hd, hz, _ = rays(seed=rank)
    ho, hd, hz = ho.pin_memory(), hd.pin_memory(), hz.contiguous().pin_memory()
    def e2e_step():
        if graph is not None:                          # H2D into the graph's static inputs, replay, D2H of the loss
            g_in[0].copy_(ho, non_blocking=True); g_in[1].copy_(hd, non_blocking=True); g_in[2].copy_(hz, non_blocking=True)
            replay_step()
            return g_loss
        return step(ho.to(dev, non_blocking=True), hd.to(dev, non_blocking=True), hz.to(dev, non_blocking=True))

    stage("e2e")
    for _ in range(2):
        l = e2e_step()
    barrier()
    t0 = time.perf_counter()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        l = e2e_step()
        float(l.item())                                # D2H read of the step's result (loss)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    wall_e2e = (time.perf_counter() - t0) * 1e3
    ms_e2e = max(ms_e2e, wall_e2e)                     # host-driven loop: wall clock bounds it from above

    stage("reduce times")
    times = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(times[0]), float(times[1])

    graph_flag = graph is not None
    # ---- the other BASELINE.json configs (short runs) ----
    extra = {}
    if not args.no_extra:
        del ren, bucket, opt, graph, g_in, g_loss
        torch.cuda.empty_cache()
        sub = argparse.Namespace(steps=5, warmup=3)
        for name, fn in (("c1", run_c1), ("c3", run_c3), ("c4", run_c4), ("c5", run_c5)):
            stage("workload " + name)
            try:
                extra[name] = fn(sub, dev, lib, rank, world)
            except Exception as e:                     # a secondary workload must never take the headline down with it
                extra[name] = {"error": "%s: %s" % (type(e).__name__, e)}
            torch.cuda.empty_cache()

    out = None
    if rank == 0:
        pk = peaks()
        samples = world * N_RAYS * N_SAMPLES * args.steps
        value = samples / (ms * 1e-3)
        engine = lib.nudf_get_engine()
        graph_used = graph_flag
        step_tflops = value * FLOP_FWD_BWD / 1e12 / world
        # roofline: the kernel family with the largest share of the step's device time
        tens = {k: v for k, v in fam.items() if "algorithmic_tflops" in v}
        dom = max(tens, key=lambda k: tens[k]["share"]) if tens else None
        kernel_of = {"udf_fwd_chain_fused": "udf_chain_kernel", "udf_bwd_chain_fused": "udf_chain_kernel", "tc_layer_reverse_sweep": "gemm_wr_kernel<nudf::EpiRev>",
                     "tc_layer_tangent": "gemm_wr_kernel<nudf::EpiTan>", "tc_layer_backward": "gemm_wr_kernel<nudf::EpiBwd>",
                     "tc_weight_gradient": "gemm_tn2_kernel"}
        launch_of = {"udf_bwd_chain_fused": 1}         # profiles/r02_chain_kernel.txt: launch 0 = F + R, launch 1 = T + B
        roof = None
        if dom is not None:
            r = tens[dom]
            roof = {"bound": "tensor", "kernel": "%s (%s): %.1f launches/step, %.1f us each" % (
                        dom, kernel_of[dom], r["launches_per_step"], r["us_per_launch"]),
                    "achieved": r["algorithmic_tflops"], "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                    "frac": r["algorithmic_tflops"] / pk["bf16_sustained"], "share_of_step": r["share"],
                    "traffic": ncu_traffic(kernel_of[dom], launch_of.get(dom, 0)),
                    "traffic_unit": "bytes per launch (dram read+write, ncu --set full, profiles/)",
                    "peak_source": pk["source"] + ", bf16 sustained (kernel timed inside the step)",
                    "how": "largest-share family of the timed step; duration = cudaEvent pairs recorded by the library on the "
                           "launching stream around each launch of the family, in %d extra steps identical to the timed ones" % min(args.steps, 10),
                    "note": "algorithmic FLOPs (2 x MACs of the family's contractions); the tensor engine executes 3x that "
                            "(3-product bf16/fp16 split) or 5x (exact value chain)",
                    "step_level": {"algorithmic_tflops": step_tflops, "frac_of_bf16_sustained": step_tflops / pk["bf16_sustained"]}}
        cpu = cpu_baseline(steps=2, warmup=1) if world == 1 else None      # host baseline: N = 1 only
        out = {
            "metric": "ray-samples/sec (render_core fwd+bwd)", "value": value, "unit": "ray-samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "ms_per_step_eager": ms_eager / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (seeded geometric-init sphere scene, random-perturbed weights)",
            "config": {"workload": "C2: 512 rays x 128 uniform samples per GPU, UDF 8x256 + colour 2x(4x128), "
                                   "render_core forward + backward + Adam update (fold / weight images rebuilt every step)",
                       "rays_per_gpu": N_RAYS, "samples_per_ray": N_SAMPLES,
                       "parallelism": "dp%d (rays sharded, NCCL all-reduce of the flat gradient bucket)" % world,
                       "l2": "per-step working set (> 1 GB of saved activations) exceeds the 126 MB L2",
                       "launch": ("whole step captured once in a CUDA graph and replayed" if graph_used else
                                  "eager (every kernel launched from Python each step)" + (": graph capture failed -- " + graph_err if graph_err else "")),
                       "engine": ("tcgen05 (fused exact fp16-split value chain + 3xBF16 gradient chains), chain mask %d" % lib.nudf_get_tc_mask())
                       if engine == 1 else "fp32 FFMA",
                       "algorithmic_flop_per_sample": FLOP_FWD_BWD,
                       "step_algorithmic_tflops": step_tflops},
            "clocks": clk,
            "e2e": {"value": world * N_RAYS * N_SAMPLES * args.steps / (ms_e2e * 1e-3), "unit": "ray-samples/s",
                    "h2d_bytes_per_step": int((ho.numel() + hd.numel() + hz.numel()) * 4), "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "families": fam,
            "roofline": roof,
            "cpu_baseline": cpu,
            "workloads": extra,
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


# ---------------------------------------------------------------------------------------------------------------
# secondary workloads (the other BASELINE.json configs); each returns a small dict
# ---------------------------------------------------------------------------------------------------------------
def run_c1(args, dev, lib, rank, world):
    """BASELINE configs[0]: 512 rays x 64 uniform samples, 4-layer / 128-wide UDF, render_core FORWARD."""
    from neuraludf_b200.models.udf_renderer_blending import UDFRendererBlending
    udf, col, var, beta = scene(dev, small_udf=True)
    ren = UDFRendererBlending(None, udf, var, col, beta, n_samples=64, n_importance=0, n_outside=0, up_sample_steps=1,
                              perturb=0.0)
    ren.want_diagnostics = False
    o, d, z, sd = rays(seed=rank, device=dev, n_samples=64)

    def fwd():
        with torch.no_grad():
            return ren.render_core(o, d, z, sd, udf, var, col, beta_network=beta, cos_anneal_ratio=None)

    ms = _timed(fwd, max(args.steps, 10), max(args.warmup, 3))
    return {"workload": "c1: render_core forward, 512 rays x 64 samples, UDF 4x128", "ms_per_step": ms,
            "ray_samples_per_s": world * N_RAYS * 64 / (ms * 1e-3), "n_gpus": world}


def run_c4(args, dev, lib, rank, world):
    """BASELINE configs[3]: whole training step of confs/udf_dtu_blending.conf -- render() (64 + 50 importance samples, 32
    outside samples, perturb) forward + backward + gradient all-reduce + Adam.  Two sizes: 512 rays per GPU (weak) and
    4096 rays in total sharded over the ranks (strong; the conf's batch on 8 GPUs)."""
    import torch.distributed as dist
    from neuraludf_b200 import synthetic as O
    from neuraludf_b200.dp import GradBucket
    from neuraludf_b200.models.udf_renderer_blending import UDFRendererBlending
    udf, col, var, beta = scene(dev)
    nerf = nerf_module(dev)
    ren = UDFRendererBlending(nerf, udf, var, col, beta, n_samples=64, n_importance=50, n_outside=32, up_sample_steps=5,
                              perturb=1.0)
    ren.want_diagnostics = False
    params = [p for m in (udf, col, var, beta, nerf) for p in m.parameters() if p.requires_grad]
    bucket = GradBucket(params, modules=(udf, col, nerf))
    opt = make_optimizer(udf, (col, var, beta, nerf))
    res = {"workload": "c4: render() fwd+bwd + all-reduce + Adam, confs/udf_dtu_blending.conf shapes", "n_gpus": world}
    for tag, n_rays in (("weak_512_per_gpu", N_RAYS), ("strong_4096_total", 4096 // world)):
        o, d, near, far = [t.to(dev) for t in O.make_rays(n_rays, seed=rank)]
        tgt = torch.full((n_rays, 3), 0.4, device=dev)

        def step():
            opt.zero_grad(set_to_none=True)
            ret = ren.render(o, d, near, far, cos_anneal_ratio=0.5, flip_saturation=0.1)
            loss = loss_fn(ret, tgt)
            loss.backward()
            if world > 1:
                bucket.allreduce_mean()
            opt.step()
            return loss

        l0 = None
        for _ in range(max(args.warmup, 3)):
            step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = lib.nudf_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        res[tag] = {"rays_per_gpu": n_rays, "ms_per_step": ms, "rays_per_s": world * n_rays / (ms * 1e-3),
                    "fine_ray_samples_per_s": world * n_rays * 114 / (ms * 1e-3),
                    "gpu_launches_per_step": (lib.nudf_launch_count() - l0) / args.steps}
    return res


def run_c3(args, dev, lib, rank, world):
    """BASELINE configs[2]: whole render() of the fine-tuning stage on open-surface shapes: 1024 rays x (64 + 64 importance)
    samples, no outside samples, pixel + patch blending on (8 source views of 1024 x 1024, 7 x 7 patches), fwd + bwd + Adam."""
    import torch.distributed as dist
    from neuraludf_b200 import synthetic as O
    from neuraludf_b200.dp import GradBucket
    from neuraludf_b200.models.udf_renderer_blending import UDFRendererBlending
    udf, col, var, beta = scene(dev)
    n_rays = 1024
    ren = UDFRendererBlending(None, udf, var, col, beta, n_samples=64, n_importance=64, n_outside=0, up_sample_steps=4,
                              perturb=1.0, upsampling_type="classical", h_patch_size=3, use_norm_grad_for_cosine=True)
    ren.want_diagnostics = False
    params = [p for m in (udf, col, var, beta) for p in m.parameters() if p.requires_grad]
    bucket = GradBucket(params, modules=(udf, col))
    opt = make_optimizer(udf, (col, var, beta))
    v = {k: t.to(dev) for k, t in O.make_blend_views(n_rays, n_views=8, height=1024, width=1024, seed=rank).items()}
    tgt = torch.full((n_rays, 3), 0.4, device=dev)

    def step():
        opt.zero_grad(set_to_none=True)
        ret = ren.render(v["rays_o"], v["rays_d"], v["near"], v["far"], cos_anneal_ratio=1.0, flip_saturation=0.0,
                         color_maps=v["color_maps"], w2cs=v["w2cs"], intrinsics=v["intrinsics"], query_c2w=v["query_c2w"],
                         rays_uv=v["rays_uv"])
        pm = ret["patch_mask"].detach()
        loss = (loss_fn(ret, tgt) + 0.5 * (ret["color_pixel"] - tgt).abs().mean()
                + 0.5 * ((ret["patch_colors"] - 0.4).abs().mean(dim=(1, 2)) * pm).sum() / (pm.sum() + 1e-5))
        loss.backward()
        if world > 1:
            bucket.allreduce_mean()
        opt.step()
        return loss

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    l0 = lib.nudf_launch_count()
    ms = _timed(step, args.steps, 0)
    return {"workload": "c3: render() fwd+bwd + Adam with pixel + patch blending, 1024 rays x (64+64) samples, 8 views 1024x1024, "
                        "49-pixel patches", "ms_per_step": ms, "rays_per_s": world * n_rays / (ms * 1e-3),
            "fine_ray_samples_per_s": world * n_rays * 128 / (ms * 1e-3), "n_gpus": world,
            "gpu_launches_per_step": (lib.nudf_launch_count() - l0) / max(args.steps, 1)}


def run_c5(args, dev, lib, rank, world):
    """BASELINE configs[4]: 256^3 lattice on [-1,1]^3 -- UDF value at every point, then the normalised gradient where
    udf < 2 voxels (the reference's get_udf_normals_grid_slow, extract_mesh.py:18-105) and, as an upper bound, at every
    point.  Lattice generated, compacted and handed over on the device (neuraludf_b200/grid.py).  With N ranks the lattice is
    slab-partitioned along x (replicas only, no exchange)."""
    import torch.distributed as dist
    from neuraludf_b200 import grid
    udf, _, _, _ = scene(dev)
    R = 256
    n_pts = R ** 3
    lo, hi = rank * n_pts // world, (rank + 1) * n_pts // world

    def sweep_all_grads():
        n = 0
        for head in range(lo, hi, 1 << 20):
            m = min(1 << 20, hi - head)
            with torch.no_grad():
                g = udf.gradient(grid.lattice_points(head, m, R, dev)).squeeze(1)
                g = g / (g.norm(dim=-1, keepdim=True) + 1e-12)
            n += m
        return n

    def timed(fn):
        fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), r

    t_val, u = timed(lambda: grid.udf_grid(udf, R, lo=lo, hi=hi))
    t_gn, cells = timed(lambda: grid.near_surface_cells(udf, R, u, lo=lo))
    t_ga, _ = timed(sweep_all_grads)
    pk = peaks()
    return {"workload": "c5: 256^3 grid query (value everywhere; normalised gradient near the surface / everywhere), lattice "
                        "generated and compacted on the device", "n_gpus": world, "value_sweep_s": t_val,
            "value_Mpts_per_s": n_pts / t_val / 1e6, "value_algorithmic_tflops": n_pts * 918016 / t_val / 1e12,
            "value_hbm_gbs": n_pts * 4 / t_val / 1e9, "value_hbm_frac": n_pts * 4 / t_val / 1e9 / pk["hbm"],
            "near_surface_cells_this_rank": int(cells[0].numel()), "near_surface_gradient_sweep_s": t_gn,
            "all_points_gradient_sweep_s": t_ga, "all_points_value_and_gradient_Mpts_per_s": n_pts / t_ga / 1e6,
            "note": "compute-bound by construction (0.9-1.8 MFLOP per point vs 4 B of HBM traffic per point -- the lattice is "
                    "generated in place --): the HBM fraction is small and is not the bound (SURVEY 8(d))"}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation of the path on the host cores
# ---------------------------------------------------------------------------------------------------------------
def _reference_step_fn(n_rays):
    """one training step of the UNMODIFIED reference (staged copy, oracle/_ref) on the CPU, or None if it is not staged"""
    from oracle import refshim
    if not refshim.available():
        return None
    from neuraludf_b200 import synthetic as S
    F, R = refshim.load()
    torch.set_default_dtype(torch.float32)
    udf_c, col_c = S.udf_cfg(), S.color_cfg()
    udf = F.UDFNetwork(d_in=3, d_out=257, d_hidden=256, n_layers=8, skip_in=(4,), multires=6, scale=1.0, bias=0.5,
                       geometric_init=False, weight_norm=True, udf_type="abs")
    udf.load_state_dict(S.make_udf_params(udf_c, seed=0))
    col = F.ResidualRenderingNetwork(d_feature=256, mode="no_normal", d_in=6, d_out=3, d_hidden=128, n_layers=4,
                                     weight_norm=True, multires_view=4, squeeze_out=True, blending_cand_views=10)
    col.load_state_dict(S.make_color_params(col_c, seed=1))
    var = F.SingleVarianceNetwork(init_val=0.6)
    beta = F.BetaNetwork(init_var_beta=0.5, init_var_gamma=0.3, init_var_zeta=0.3, beta_min=5e-5, requires_grad_beta=True,
                         requires_grad_gamma=False, requires_grad_zeta=False)
    ren = R.UDFRendererBlending(None, udf, var, col, beta, n_samples=N_SAMPLES, n_importance=0, n_outside=0,
                                up_sample_steps=1, perturb=0.0)
    opt = make_optimizer(udf, (col, var, beta), fused=False)
    o, d, z, sd = rays(seed=0)
    o, d, z = o[:n_rays], d[:n_rays], z[:n_rays]
    tgt = torch.full((n_rays, 3), 0.4)

    def one():
        t0 = time.perf_counter()
        opt.zero_grad()
        ret = ren.render_core(o, d, z, sd, udf, var, col, beta_network=beta, cos_anneal_ratio=0.5)
        loss_fn(ret, tgt).backward()
        opt.step()
        return time.perf_counter() - t0
    return one


def _ref_origin():
    from oracle import refshim
    return "staged byte-for-byte copy oracle/_ref" if refshim.is_staged_copy() else "checkout " + refshim.REFERENCE_ROOT


def _port_step_fn(n_rays):
    from oracle import oracle_torch as O
    udf_c, col_c = O.udf_cfg(), O.color_cfg()
    up = {k: v.clone().requires_grad_(True) for k, v in O.make_udf_params(udf_c, seed=0).items()}
    cp = {k: v.clone().requires_grad_(True) for k, v in O.make_color_params(col_c, seed=1).items()}
    sc = {k: v.clone().requires_grad_(True) for k, v in O.make_scalars().items()}
    o, d, z, sd = rays(seed=0)
    o, d, z = o[:n_rays], d[:n_rays], z[:n_rays]
    tgt = torch.full((n_rays, 3), 0.4)
    leaves = list(up.values()) + list(cp.values()) + [sc["variance"], sc["beta"]]
    opt = torch.optim.Adam(leaves, lr=1e-4)

    def one():
        t0 = time.perf_counter()
        opt.zero_grad()
        ret = O.render_core(up, udf_c, cp, col_c, sc, o, d, z, sd, cos_anneal_ratio=0.5)
        loss_fn(ret, tgt).backward()
        opt.step()
        return time.perf_counter() - t0
    return one


def cpu_baseline(steps, warmup, n_rays=N_RAYS):
    """The reference's render_core training step on the host cores, on the SAME configuration as the CUDA arm (all 512 rays x
    128 samples, forward + backward + Adam).  The thread count is swept at the timed size."""
    one = _reference_step_fn(n_rays)
    kind = "reference"
    if one is None:
        one, kind = _port_step_fn(n_rays), "port"
    ncpu = os.cpu_count() or 1
    cands = sorted(set(c for c in (8, 16, 32, 64, ncpu) if c <= ncpu)) or [ncpu]
    sweep = {}
    one()                                               # first call pays allocator / thread-pool start-up
    for c in cands:
        torch.set_num_threads(c)
        sweep[c] = one()
    best = min(sweep, key=sweep.get)
    torch.set_num_threads(best)
    ts = []
    for i in range(warmup + steps):
        dt = one()
        if i >= warmup:
            ts.append(dt)
    per = sum(ts) / len(ts)
    what = ("the unmodified reference (xxlong0/NeuralUDF models/udf_renderer_blending.py render_core, %s)" % _ref_origin()
            if kind == "reference" else "the pinned oracle port of the reference's render_core (no staged reference copy found)")
    return {"value": n_rays * N_SAMPLES / per, "unit": "ray-samples/s", "cores": torch.get_num_threads(), "kind": kind,
            "host_cpus": ncpu,
            "sample": "%s: all %d rays x %d samples, forward + backward + Adam, %d timed steps after %d warm-up; thread count = "
                      "fastest of a sweep at this size %s" % (what, n_rays, N_SAMPLES, steps, warmup,
                                                             {k: round(v, 3) for k, v in sweep.items()}),
            "s_per_step": per}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    steps = max(1, min(args.steps, 8))                  # bounded: ~1 s per step on the host
    cpu = cpu_baseline(steps=steps, warmup=max(1, min(args.warmup, 2)))
    return {"impl": "reference", "metric": "ray-samples/sec (render_core fwd+bwd)", "value": cpu["value"],
            "unit": "ray-samples/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": steps,
            "warmup": args.warmup, "ms_per_step": cpu["s_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (same seeded scene as the CUDA arm)",
            "config": {"workload": "C2: 512 rays x 128 uniform samples, UDF 8x256 + colour 2x(4x128), render_core forward + "
                                   "backward + Adam update on the host CPU (%s)" % cpu["kind"],
                       "rays_per_gpu": N_RAYS, "samples_per_ray": N_SAMPLES, "requested_steps": args.steps},
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5"],
                    help="c2 (default, the BASELINE.json headline; also runs short versions of the others and reports them "
                         "under `workloads`); c1 / c3 / c4 / c5: that workload alone, reduced JSON line")
    ap.add_argument("--quick", action="store_true", help="main timed loop only (for profiler runs): no e2e leg, no "
                    "family table, no CPU baseline, no secondary workloads; prints a reduced JSON line")
    ap.add_argument("--no-extra", dest="no_extra", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--no-graph", dest="no_graph", action="store_true", help="time the eager loop only (no CUDA-graph capture)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed C2 step (render_core outputs, loss, parameter gradients, "
                         "updated parameters) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs applies to the C2 workload of --impl ours")
    out = run_reference(args) if args.impl == "reference" else run_ours(args)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
