#!/usr/bin/env python
"""bench.py — render+loss(+GAN) images/sec on B200 (BASELINE.json metric), one JSON line on stdout.

Workloads (SURVEY.md §8d):
  cfg3 (default; BASELINE.json configs[2], the configuration the metric is quoted on): per step THREE training
       iterations (G, D, D — main.py:691's 1 : d_steps_per_g alternation) at batch 32 per GPU, each iteration =
       cfg2's render+loss forward/backward on a FRESH batch + one conv-GAN step at 256^2 (nd = 2, class-conditional,
       SyncBN generator, hinge loss, Adam(0, 0.9), EMA generator).
  cfg2 (configs[1]): render+loss only, batch 16: (i) EffectiveLossFunction(V=128)(points[16,8000,3], q, scale) ->
       sum-MSE vs mask; (ii) mesh_map -> template vertices (482 v / 960 f) -> pose -> DIB-R render 256x256 with a
       128x128 texture -> RGBA MSE + 5e-4 * loss_flat (+ mIoU).
Synthetic, seeded inputs (no dataset exists offline).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2|cfg3] [--dump-outputs DIR]
N>1 is launched by torchrun (one rank per GPU, NCCL); every rank owns its own shard of the global batch (weak scaling).
cfg3's collectives: SyncBN statistics of the generator and the gradient all-reduce of G / D (captured in the step's CUDA
graph).  `--impl reference` times the reference's algorithm on the host cores (oracle/, torch CPU) on the same config.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "2dimageto3dmodel_b200")
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

_T0 = time.time()


def stage(msg):
    """Wall-clock breadcrumbs on stderr (rank 0): where a slow multi-GPU launch spends its time."""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)

N_PTS, V, H, TEX, FLAT_COEF = 8000, 128, 256, 128, 5e-4
WORKLOADS = {
    # BASELINE.json configs[1]
    "cfg2": dict(batch=16, gan=False, kind="render", iters=1,
                 metric="render+loss images/sec (cfg2: 8000-pt effective loss V=128 + CUB mesh render 256x256, fwd+bwd)",
                 name="cfg2: CUB 256x256, 8000-pt cloud, full render+loss, batch=16 per GPU"),
    # BASELINE.json configs[2] = the configuration the metric "render+loss+GAN images/sec" is quoted on
    "cfg3": dict(batch=32, gan=True, kind="render+gan", iters=3, res=256, nd=2,
                 metric="render+loss+GAN images/sec (cfg3: cfg2 render+loss at batch 32 + conv-GAN 256x256 G/D iteration, 1 G : 2 D, Adam)",
                 name="cfg3: CUB 256x256 render+loss + conv-GAN G/D step, batch=32 per GPU"),
    # BASELINE.json configs[3]: run_reconstruction.py's training iteration (network -> template -> pose with DatasetParams
    # deltas + z0 -> render -> MSE + flat warm-up -> two Adams) on the P3D template (962 v / 1920 f); the reference's batch
    # of 50 on one GPU, 13 per rank under DDP x4 (global 52: equal shards)
    "cfg4": dict(batch=50, gan=False, kind="recon", iters=1,
                 metric="reconstruction-training images/sec (cfg4: ReconstructionNetwork + P3D mesh render 256x256 + losses, optimize_z0, Adam x2)",
                 name="cfg4: Pascal3D+ 256x256, optimize_z0 reconstruction loop, batch=50 (13 per GPU under DDP)"),
    # BASELINE.json configs[4]: main.py's GAN iteration at 512^2 with three discriminators, 8 images per rank
    "cfg5": dict(batch=8, gan=True, kind="gan", iters=3, res=512, nd=3,
                 metric="GAN-training images/sec (cfg5: conv-GAN 512x512 class-conditional, nd=3, 1 G : 2 D, Adam, SyncBN)",
                 name="cfg5: CUB 512x512 class-conditional GAN training, batch=8 per GPU (64 on 8 GPUs)"),
}
GAN_RES = 256


def gan_args(res=256, nd=2):
    import types
    return types.SimpleNamespace(texture_resolution=res, conditional_class=True, conditional_color=False,
                                 conditional_text=False, norm_g='syncbatch', norm_d='none', n_classes=(200,),
                                 mask_output=True, texture_only=False, num_discriminators=nd, text_embedding_dim=256,
                                 latent_dim=64, loss='hinge', lr_g=1e-4, lr_d=4e-4, d_steps_per_g=2,
                                 mesh_regularization=1e-4, g_running_average_alpha=0.999, symmetric_g=True)


def recon_host_inputs(B, seed, pin, dataset_size=4722):
    """cfg4 (SURVEY §8d): RGBA images with a disk alpha, poses in the ranges of cache/p3d/poses_metadata.npz, image indices
    into a dataset of 4722 images and their mirrored copies."""
    g = torch.Generator().manual_seed(seed + 13)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, H), torch.linspace(-1, 1, H), indexing="ij")
    disk = ((yy * yy + xx * xx) < 0.45).float()
    x_real = torch.rand(B, 4, H, H, generator=g) * 2 - 1
    x_real[:, 3] = disk
    x_real[:, :3] *= disk
    d = dict(x_real=x_real, pscale=0.55 + 0.3 * torch.rand(B, 1, generator=g), ptrans=(torch.rand(B, 3, generator=g) - 0.5) * 0.3,
             rot=torch.nn.functional.normalize(torch.randn(B, 4, generator=g), dim=-1),
             idx=torch.randint(0, 2 * dataset_size, (B,), generator=g))
    return {k: (v.pin_memory() if pin else v) for k, v in d.items()}


def gan_host_inputs(B, seed, pin, R=256):
    g = torch.Generator().manual_seed(seed + 77)
    alpha = (torch.rand(B, 1, R // 8, R // 8, generator=g) > 0.4).float()
    d = dict(X_tex=torch.rand(B, 3, R, R, generator=g) * 2 - 1,
             X_alpha=torch.nn.functional.interpolate(alpha, size=(R, R), mode="bilinear", align_corners=False),
             X_mesh=torch.randn(B, 3, 32, 32, generator=g) * 0.05, C=torch.randint(0, 200, (B, 1), generator=g))
    return {k: (v.pin_memory() if pin else v) for k, v in d.items()}


def host_inputs(B, seed, pin):
    g = torch.Generator().manual_seed(seed)
    pts = (torch.rand(B, N_PTS, 3, generator=g) * 2 - 1) * 0.45
    shell = torch.nn.functional.normalize(torch.randn(B, N_PTS // 2, 3, generator=g), dim=-1)
    pts[:, : N_PTS // 2] = shell * (0.33 + 0.01 * torch.randn(B, N_PTS // 2, 1, generator=g))
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, H), torch.linspace(-1, 1, H), indexing="ij")
    disk = ((yy * yy + xx * xx) < 0.45).float()
    x_real = torch.rand(B, 4, H, H, generator=g) * 2 - 1
    x_real[:, 3] = disk
    x_real[:, :3] *= disk
    m = torch.nn.functional.interpolate(disk[None, None], size=(V, V), mode="bilinear", align_corners=True)[0, 0]
    d = dict(points=pts, quat=torch.randn(B, 4, generator=g), scale=0.5 + 0.5 * torch.rand(B, 1, generator=g),
             mask=m.expand(B, V, V).contiguous(), mesh_map=torch.randn(B, 3, 32, 32, generator=g) * 0.05,
             tex=torch.rand(B, 3, TEX, TEX, generator=g) * 2 - 1,
             rot=torch.nn.functional.normalize(torch.randn(B, 4, generator=g), dim=-1),
             pscale=0.55 + 0.3 * torch.rand(B, 1, generator=g), ptrans=(torch.rand(B, 3, generator=g) - 0.5) * 0.3,
             x_real=x_real)
    return {k: (v.pin_memory() if pin else v) for k, v in d.items()}


def template_path(rings=16):
    from tools.uvsphere import write_uvsphere_obj          # synthetic input (the shipped templates cannot travel)
    return write_uvsphere_obj(os.path.join(tempfile.mkdtemp(), f"uvsphere_{rings}rings.obj"), rings=rings)


# --------------------------------------------------------------------------------------------- CUDA arm
class CudaWorkload:
    def __init__(self, device, cfg):
        from rendering.mesh_template import MeshTemplate
        from rendering.renderer import Renderer
        from utils.effective_loss_function import EffectiveLossFunction
        self.dev, self.kind = device, cfg["kind"]
        self.gan = self.recon = None
        self.tpl = MeshTemplate(template_path(31 if self.kind == "recon" else 16), device=device)
        if "render" in self.kind:
            self.elf = EffectiveLossFunction(voxel_size=V).to(device)
            self.renderer = Renderer(H, H)
        if cfg["gan"]:
            from gan_training import GANTrainer
            torch.manual_seed(4321)                      # identical replicas on every rank
            self.gan = GANTrainer(gan_args(cfg["res"], cfg["nd"]), mesh_template=self.tpl, device=device, capturable=True)
        if self.kind == "recon":
            from reconstruction_training import ReconTrainer, default_args
            torch.manual_seed(4321)
            self.recon = ReconTrainer(default_args(optimize_z0=True), self.tpl, dataset_size=4722, device=device, capturable=True)

    def step(self, batches):
        """One step over `batches` (one input dict per training iteration).  cfg2: render+loss fwd+bwd.  cfg3: three
        iterations (G, D, D — the reference's 1 : d_steps_per_g alternation, main.py:691), each on its own batch =
        render+loss fwd+bwd + one GAN step with its optimiser.  cfg4: one run_reconstruction.py iteration.  cfg5: G, D, D.
        Returns the loss and, when the step renders, each iteration's input gradients (render_step)."""
        if self.kind == "render":
            loss, grads = self.render_step(batches[0])
            return loss, [grads]
        if self.kind == "recon":
            d = batches[0]
            return self.recon.step(d["x_real"], d["pscale"], d["ptrans"], d["rot"], d["idx"])[0], None
        loss, grads = None, []
        for it, d in enumerate(batches):
            if it == 0:
                gl = self.gan.g_step(d["X_alpha"], d["C"])
            else:
                gl = self.gan.d_step(d["X_tex"], d["X_alpha"], d["X_mesh"], d["C"])
            if "render" in self.kind:
                rl, rg = self.render_step(d)
                gl = gl + rl
                grads.append(rg)
            loss = gl if loss is None else loss + gl
        return loss, grads or None

    def render_step(self, d):
        from b3d.mesh import rgba_mse_iou
        from utils.losses import loss_flat
        p, q, s = (d[k].detach().requires_grad_(True) for k in ("points", "quat", "scale"))
        sil = self.elf(p, q, s)
        loss_pc = (sil - d["mask"]).square().sum() / sil.shape[0]        # unsupervised_part.py:111
        mm, tex = d["mesh_map"].detach().requires_grad_(True), d["tex"].detach().requires_grad_(True)
        # get_vertex_positions + transform_vertices in one launch (b3d.vertex; run_reconstruction.py:425-427)
        raw, vtx = self.tpl.vertices_and_pose(mm, d["pscale"], d["ptrans"], d["rot"])
        img, alpha = self.tpl.forward_renderer(self.renderer, vtx, tex)
        recon, miou = rgba_mse_iou(img, alpha, d["x_real"])
        flat = loss_flat(self.tpl.mesh, self.tpl.compute_normals(raw))
        loss = loss_pc + recon + FLAT_COEF * flat
        loss.backward()
        return loss.detach(), (p.grad, q.grad, s.grad, mm.grad, tex.grad)


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        return len(self.rows)

    def stop(self, lo=0, hi=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for r in self.rows[lo:hi] if len(r) >= 7] or [r for r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        f = lambda x: float(x) if x.replace(".", "", 1).isdigit() else None
        sm = [f(r[0]) for r in rows if f(r[0]) is not None]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": f(rows[0][1]),
                "power_w_max": max((f(r[2]) or 0) for r in rows), "samples": len(rows), "reasons": reasons}


def measure_tf32_peak(dev, seconds=2.0):
    """Dense tf32 tensor-core peak of THIS GPU, measured the way MEASURED_PEAKS.json measures bf16: torch.matmul (cuBLAS)
    8192^3 with allow_tf32, fp32 storage.  burst = best of 10 single calls, sustained = back to back for `seconds`."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a, b = torch.randn(n, n, device=dev), torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a, b, out=c); e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        reps = max(10, int(seconds * 1e3 / best))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        fl = 2.0 * n ** 3
        return {"burst": round(fl / (best * 1e-3) / 1e12, 1), "sustained": round(fl * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12, 1),
                "how": f"measured live: torch.matmul (cuBLAS) fp32 storage, allow_tf32, 8192^3; burst best of 10, sustained {reps} "
                       f"back-to-back calls (~{seconds:.0f} s)"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def chamfer_report(dev, B=32, N=8000):
    """Nearest-neighbour (chamfer) kernel on 8000 x 8000 point sets (north_star): CUDA events on the launching stream."""
    from b3d.chamfer import nearest

    def chamfer_nn(a, b):
        nearest(a, b)
        nearest(b, a)
    g = torch.Generator().manual_seed(5)
    a = (torch.rand(B, N, 3, generator=g) - 0.5).to(dev)
    b = (torch.rand(B, N, 3, generator=g) - 0.5).to(dev)
    for _ in range(3):
        chamfer_nn(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        chamfer_nn(a, b)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    fl = 8.0 * N * N * B * 2                      # both directions: (3 sub, 3 fma-equivalents, compare) ~ 8 flop per pair
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12     # 148 SMs x 128 FMA lanes x 2 flop x 1.965 GHz
    return {"kernel": "chamfer_nn_kernel (both directions)", "sets": f"{B} x ({N} vs {N})", "ms_per_launch_pair": round(ms, 4),
            "achieved": round(fl / (ms * 1e-3) / 1e12, 2), "peak": round(fp32_peak, 1), "unit": "TFLOP/s (fp32 CUDA cores)",
            "frac": round(fl / (ms * 1e-3) / 1e12 / fp32_peak, 4), "bound": "fp32 issue (8NM flop over 20(N+M) bytes)"}


def algorithmic_bytes(B, F_=960):
    """SURVEY.md §8(d) per-sample figures x the samples one launch processes (stated in DESIGN.md)."""
    pc_fwd = 8 * V**3 + 4 * V**2 + 12 * N_PTS
    pc_all = 20 * V**3 + 8 * V**2 + 36 * N_PTS
    Tw = TEX + 2
    mesh_fwd = 100 * F_ + 12 * TEX * Tw + H * H * 48
    mesh_bwd = H * H * 32 + 12 * TEX * Tw + 60 * F_
    return {"b3d_pc_silhouette_fwd_hosttaps": B * pc_fwd, "b3d_pc_silhouette_bwd_hosttaps": B * (pc_all - pc_fwd),
            "b3d_mesh_render_fwd": B * mesh_fwd, "b3d_mesh_render_bwd": B * mesh_bwd}


DUMP_LIMIT = 64 << 20          # bytes written in all


def dump_outputs(out_dir, loss, grads):
    """What the timed step returned last (CudaWorkload.step), as <out_dir>/<name>.npy in float32: the loss and, per
    training iteration that renders, the gradients of the loss with respect to the rendered inputs.  The trained networks'
    state is not written: Adam with betas (0, 0.9) moves every weight by about lr * sign(gradient) in its first steps, so
    gradients at rounding level (float atomics) make that state differ from run to run of the same build."""
    import numpy as np
    arrays = {"loss": loss.detach().reshape(-1)}
    for it, g in enumerate(grads or []):
        for name, t in zip(("points", "quat", "scale", "mesh_map", "tex"), g):
            arrays[f"iter{it}_grad_{name}"] = t
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    stage(f"dumped {len(arrays)} arrays ({total} bytes) to {out_dir}")


def run_cuda(args):
    import b3d
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference)")
    if os.environ.get("B3D_SINGLE_GPU"):      # development aid: all ranks share cuda:0 (use with B3D_DIST_BACKEND=gloo)
        local = 0
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        # NCCL collectives are captured into the step's CUDA graph: the watchdog must not poll CUDA during capture
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        import torch.distributed as dist
        backend = os.environ.get("B3D_DIST_BACKEND", "nccl")
        dist.init_process_group(backend, **({"device_id": dev} if backend == "nccl" else {}))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")

    stage("process group ready" if world > 1 else "start")
    cfg = WORKLOADS[args.workload]
    METRIC, WORKLOAD = cfg["metric"], cfg["name"]
    wl = CudaWorkload(dev, cfg)
    stage("workload built")
    B = cfg["batch"]
    if cfg["kind"] == "recon" and world > 1:
        B = 13                                              # DDP x4: 52 = 4 x 13 (equal shards of the reference's batch of 50)
    iters_per_step = cfg["iters"]
    host = []                                               # one pinned host batch per training iteration of the step;
    for it in range(iters_per_step):                        # each rank owns its shard of the global batch
        hb = {}
        if "render" in cfg["kind"]:
            hb.update(host_inputs(B, seed=1234 + rank + 1000 * it, pin=True))
        if cfg["gan"]:
            hb.update(gan_host_inputs(B, seed=1234 + rank + 1000 * it, pin=True, R=cfg["res"]))
        if cfg["kind"] == "recon":
            hb.update(recon_host_inputs(B, seed=1234 + rank + 1000 * it, pin=True))
        host.append(hb)
    h2d = sum(t.numel() * t.element_size() for hb in host for t in hb.values())
    resident = [{k: v.to(dev) for k, v in hb.items()} for hb in host]
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)  # > 126 MB L2

    def sync_all():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        sync_all()
        evs = []
        for _ in range(steps):
            flush.zero_()                                    # evict L2 between timed iterations
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        sync_all()
        total = sum(a.elapsed_time(b) for a, b in evs)
        if dist is not None:
            t = torch.tensor([total], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total = float(t)
        return total

    def fresh(batches):
        return [{k: v.detach() for k, v in d.items()} for d in batches]

    host_loss = torch.empty(1).pin_memory()
    graph = None
    # N > 1: the step contains NCCL collectives (gradient all-reduce, SyncBN statistics); they are captured into the
    # graph too (thread-local capture mode, NCCL async error handling off).  B3D_DDP_EAGER=1 launches eagerly instead.
    has_coll = cfg["gan"] or cfg["kind"] == "recon"
    capture_ok = world == 1 or not has_coll or (os.environ.get("B3D_DIST_BACKEND", "nccl") == "nccl"
                                                and not os.environ.get("B3D_DDP_EAGER"))
    if not args.no_graph and capture_ok:
        # the step has no host synchronisation: capture it once (forward + backward) and replay it
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                wl.step(fresh(resident))
        torch.cuda.current_stream().wait_stream(side)
        stage("eager warm-up done, capturing the step")
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, capture_error_mode="thread_local" if world > 1 else "global"):
            g_loss, g_grads = wl.step(fresh(resident))

    last = {}                                                # outputs of the latest step (the graph's are static)

    def step_resident():
        if graph is not None:
            graph.replay()
            last["loss"], last["grads"] = g_loss, g_grads
            return g_loss
        last["loss"], last["grads"] = wl.step(fresh(resident))
        return last["loss"]

    # End-to-end input pipeline (what a training loop with a prefetching loader does): the pinned host batches of step k+1
    # are uploaded into device STAGING buffers on a copy stream while step k computes; at the start of a step the staged
    # batches move device-to-device into the graph's static inputs.  Every step's H2D copies and its D2H loss read are inside
    # the timed region (the timed loop issues them); they overlap the previous step's kernels instead of serialising in front.
    copy_stream = torch.cuda.Stream()
    staging = [{k: torch.empty_like(v) for k, v in rb.items()} for rb in resident]
    staged, consumed = torch.cuda.Event(), torch.cuda.Event()
    consumed.record()

    def prefetch():
        copy_stream.wait_event(consumed)                     # the previous contents were moved into the graph inputs
        with torch.cuda.stream(copy_stream):
            for hb, sb in zip(host, staging):
                for k, v in hb.items():
                    sb[k].copy_(v, non_blocking=True)
            staged.record(copy_stream)

    prefetch()

    def step_e2e():
        main = torch.cuda.current_stream()
        main.wait_event(staged)                              # this step's inputs have arrived on the device
        if graph is not None:
            for sb, rb in zip(staging, resident):
                keys = list(sb)
                torch._foreach_copy_([rb[k] for k in keys], [sb[k] for k in keys])
            consumed.record(main)
            prefetch()                                       # next step's H2D overlaps this step's kernels
            graph.replay()
            loss = g_loss
        else:
            batches = [{k: v.clone() for k, v in sb.items()} for sb in staging]
            consumed.record(main)
            prefetch()
            loss, _ = wl.step(batches)
        host_loss.copy_(loss.reshape(1), non_blocking=True)
        main.synchronize()                                   # the user reads the loss every step
        return loss

    tf32 = measure_tf32_peak(dev) if (cfg["gan"] or cfg["kind"] == "recon") and rank == 0 else None
    stage("tf32 peak measured" if tf32 else "timing setup")
    clocks = ClockSampler(local) if rank == 0 else None
    time.sleep(0.3) if clocks else None
    n0 = b3d.launch_count()
    lo = clocks.mark() if clocks else 0
    stage("timing (resident inputs)")
    total_ms = timed(step_resident, args.steps, args.warmup)
    hi = clocks.mark() if clocks else 0
    if args.dump_outputs and rank == 0:                      # before the later passes overwrite the graph's outputs
        dump_outputs(args.dump_outputs, last["loss"], last["grads"])
    launches = (b3d.launch_count() - n0) // (args.steps + args.warmup)
    if graph is not None:                                    # replays do not pass through the C ABI counter
        n1 = b3d.launch_count()
        wl.step(fresh(resident))
        launches = b3d.launch_count() - n1
    stage("timing (end to end)")
    e2e_ms = timed(step_e2e, args.steps, args.warmup)
    clk = clocks.stop(lo, max(hi, lo + 1)) if clocks else None

    # per-entry-point device times (events on the launching stream), separate pass
    stage("per-entry-point profile pass")
    b3d.prof_enable()
    for _ in range(max(3, args.steps // 2)):
        flush.zero_()
        wl.step(fresh(resident))
    torch.cuda.synchronize()
    nprof = max(3, args.steps // 2)
    raw_prof = b3d.prof_disable()
    prof = {k: statistics.mean(v) for k, v in raw_prof.items()}
    prof_tot = {k: sum(v) / nprof for k, v in raw_prof.items()}     # ms per step per entry point
    if os.environ.get("B3D_PROF_SHAPES") == "1" and rank == 0:      # development aid: per-geometry conv times to stderr
        for k, v in sorted(prof_tot.items(), key=lambda kv: -kv[1])[:60]:
            print(f"{v:8.3f} ms/step x{len(raw_prof[k]) // nprof:3d}  {k}", file=sys.stderr)

    # collective work of one step (N > 1): the SyncBN statistic exchanges are libb3d entry points (timed above); the in-place
    # gradient all-reduces of the flat conv-weight buffers are timed here with CUDA events (all ranks take part)
    collectives = None
    if dist is not None and cfg["gan"]:
        import torch.distributed as tdist
        G_, D_ = wl.gan.trainer.generator, wl.gan.trainer.discriminator
        flats = [(n, getattr(m.__dict__.get('_bank'), 'last_dw', None)) for n, m in (("generator", G_), ("discriminator", D_))]
        ar_ms, ar_bytes = 0.0, 0
        if all(f is not None for _, f in flats) and tdist.get_backend() == "nccl":
            plan = [flats[0][1], flats[1][1], flats[1][1]]             # G step, two D steps
            for f in plan:
                tdist.all_reduce(f, op=tdist.ReduceOp.AVG)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                for f in plan:
                    tdist.all_reduce(f, op=tdist.ReduceOp.AVG)
            e1.record()
            torch.cuda.synchronize()
            ar_ms, ar_bytes = e0.elapsed_time(e1) / 5, sum(f.numel() * 4 for f in plan)
        sync_ms = sum(v for k, v in prof_tot.items() if k.endswith("_sync"))
        sync_n = sum(len(v) for k, v in raw_prof.items() if k.endswith("_sync")) // nprof
        collectives = {"syncbn_exchanges_per_step": sync_n, "syncbn_fused_kernels_ms_per_step": round(sync_ms, 3),
                       "syncbn_path": "fused one-shot all-reduce over NVLink peer memory" if sync_n else "NCCL all-reduce per layer",
                       "grad_allreduce_ms_per_step": round(ar_ms, 3), "grad_allreduce_bytes_per_step": ar_bytes}

    def finish():
        """All ranks leave together; with NCCL captured in a CUDA graph the communicator teardown can block, so multi-rank
        runs end with a barrier and a hard exit (the JSON line is flushed first)."""
        if dist is not None:
            torch.cuda.synchronize()
            dist.barrier()
            sys.stdout.flush()
            os._exit(0)

    if rank != 0:
        finish()
        return
    ms = total_ms / args.steps
    value = world * B * iters_per_step / (ms / 1e3)
    e2e_v = world * B * iters_per_step / (e2e_ms / args.steps / 1e3)
    alg = algorithmic_bytes(B, 1920 if cfg["kind"] == "recon" else 960)
    cand = {k: prof[k] for k in alg if k in prof}
    top = max(cand, key=cand.get) if cand else None
    ach = alg[top] / (cand[top] * 1e-3) / 1e9 if top else 0.0
    tensor = None
    if cfg["kind"] in ("recon", "gan"):
        # dense-conv FLOPs per image (SURVEY §8d / App. D): reconstruction network 12.21 GF fwd, x3 for fwd + dgrad + wgrad
        # (the first layer's input gradient is not executed: conv1e 5x5/s2 4->64, 0.21 GF); 512^2 GAN, nd=3: G 66.56, D 17.80
        # GF fwd; G-step 3G + 2D, D-step G + 6D minus the first-layer input gradients of the 2B batch
        # (d1.conv1 1.07 + d2.conv1 0.036 + d3.conv1 0.42 GF)
        gf_img = 3 * 12.21 - 0.21 if cfg["kind"] == "recon" else (3 * 66.56 + 2 * 17.80) + 2 * (66.56 + 6 * 17.80 - 2 * 1.526)
        conv_ms = sum(v for k, v in prof_tot.items() if k.startswith("b3d_conv2d"))
        tensor = {"kernel": "all conv entry points", "bound": "tensor",
                  "achieved": round(gf_img * B / (conv_ms * 1e-3) / 1e3, 1), "peak": tf32["sustained"], "unit": "TFLOP/s",
                  "frac": round(gf_img * B / (conv_ms * 1e-3) / 1e3 / tf32["sustained"], 4), "traffic": None,
                  "peak_source": tf32["how"], "peak_burst": tf32["burst"], "conv_ms_per_step": round(conv_ms, 3),
                  "gflop_per_step": round(gf_img * B, 1)}
    elif cfg["gan"]:
        # dense-conv FLOPs of one G + two D iterations (SURVEY §8d / App. D at 256^2, nd=2: G 17.09, D 14.76 GF/img fwd),
        # counting only what is executed: G-step = fwd G+D, dgrad+wgrad G, dgrad D (the reference's discarded D wgrad is
        # skipped) = 3G + 2D; D-step = G fwd + D fwd/dgrad/wgrad on 2B images = G + 6D — over the time spent inside the
        # tcgen05 conv entry points
        # ... minus the input gradient of the discriminators' first layers in the D-step (their input needs no gradient, so
        # it is not executed): d1.conv1 1.678 + d2.conv1 0.036 GF per image of the 2B batch
        gf_img = (3 * 17.09 + 2 * 14.76) + 2 * (17.09 + 6 * 14.76 - 2 * (1.678 + 0.036))
        conv_ms = sum(v for k, v in prof_tot.items() if k.startswith("b3d_conv2d"))
        tpeak, tpeak_src = tf32["sustained"], tf32["how"]
        tensor = {"kernel": "all conv entry points: conv_tf32_persistent + wgrad_tf32 (tcgen05 kind::tf32) + thin-head CUDA-core kernels", "bound": "tensor",
                  "achieved": round(gf_img * B / (conv_ms * 1e-3) / 1e3, 1), "peak": round(tpeak, 1), "unit": "TFLOP/s",
                  "frac": round(gf_img * B / (conv_ms * 1e-3) / 1e3 / tpeak, 4), "traffic": None,
                  "peak_source": tpeak_src, "peak_burst": tf32["burst"],
                  "conv_ms_per_step": round(conv_ms, 3), "gflop_per_step": round(gf_img * B, 1)}
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload, {})
        traffic = tj.get(top)
        if tensor is not None and "conv_dominant" in tj:      # DRAM bytes of the most expensive single conv launch (ncu)
            tensor["traffic"] = tj["conv_dominant"]["bytes"]
            tensor["traffic_kernel"] = tj["conv_dominant"]["kernel"]
    except (OSError, ValueError):
        pass
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms, 4), "higher_is_better": True,
        # cfg4 quotes a GLOBAL batch (50, run as 4 x 13 under DDP) that is split over the ranks; cfg2 / cfg3 / cfg5 fix the per-GPU batch
        "scaling": "strong" if cfg["kind"] == "recon" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": world * B,
                   "iterations_per_step": iters_per_step, "points": N_PTS, "voxels": V,
                   "image": cfg.get("res", H) if cfg["kind"] == "gan" else H, "faces": 1920 if cfg["kind"] == "recon" else 960,
                   "texture": TEX, "l2": "flushed between timed iterations (256 MB write)",
                   "parallelism": (f"dp{world}: batch shards; render/loss without collectives, GAN with SyncBN statistic "
                                   "all-reduces + gradient all-reduce (NCCL, captured in the step graph)") if cfg["gan"]
                   else (f"dp{world}: batch shards; SyncBN statistic exchange per BatchNorm layer + gradient all-reduce "
                         "(captured in the step graph)") if cfg["kind"] == "recon" and world > 1
                   else f"dp{world} (batch shards, no data-path collective)", "semantics": "R",
                   "fresh_batch_per_iteration": True,
                   "cuda_graph": graph is not None},
        "e2e": {"value": round(e2e_v, 2), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": round(e2e_ms / args.steps, 4),
                "pipeline": "pinned host -> device staging on a copy stream (prefetch of the next step, overlapped with compute), "
                            "staging -> graph inputs device-to-device, loss read back and host-synchronised every step"},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": {"kernel": top, "bound": "hbm", "achieved": round(ach, 1), "peak": hbm_peak, "unit": "GB/s",
                     "frac": round(ach / hbm_peak, 4), "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg[top], "ms_per_launch": round(cand[top], 4)} if top else None,
        "kernel_ms_per_step": {k: round(v, 4) for k, v in sorted(prof_tot.items(), key=lambda kv: -kv[1])},
    }
    try:
        out["chamfer"] = chamfer_report(dev)
    except Exception as e:                                   # reported, never fatal for the headline
        out["chamfer"] = {"error": str(e)[:200]}
    if collectives is not None:
        out["collectives"] = collectives
    if tensor is not None:
        # the convolutions dominate the step -> the tensor-core roofline is the primary one; the HBM-class kernel
        # roofline (point-cloud / raster backward) moves to roofline_hbm
        if out["roofline"] is not None:
            out["roofline_hbm"] = out["roofline"]
        out["roofline"] = tensor
        out["dtype"] = "tf32 (convs) / f32"
    if world == 1 and not os.environ.get("B3D_BENCH_NO_CPU") and cfg["kind"] != "recon":
        out["cpu_baseline"] = cpu_baseline(cfg, budget_s=25.0)
    print(json.dumps(out), flush=True)
    finish()


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_threads():
    """All the host threads torch can USE: its CPU kernels stop scaling (and regress) below the 100+ hardware threads of
    the GPU hosts, so a one-second probe (a ResBlock-sized fp32 convolution, forward + backward) picks the fastest of
    {32, 64, all} and that number is reported as `cores`."""
    ncpu = os.cpu_count() or 1
    cands = sorted({min(ncpu, 32), min(ncpu, 64), ncpu})
    if len(cands) == 1:
        torch.set_num_threads(cands[0])
        return cands[0]
    x = torch.randn(8, 64, 128, 66, requires_grad=True)
    w = torch.randn(64, 64, 3, 3, requires_grad=True)
    best, best_t = cands[0], 1e9
    for n in cands:
        torch.set_num_threads(n)
        torch.nn.functional.conv2d(x, w, padding=(1, 0)).sum().backward()
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.conv2d(x, w, padding=(1, 0)).sum().backward()
        t = time.perf_counter() - t0
        if t < best_t:
            best, best_t = n, t
    torch.set_num_threads(best)
    return best


class OracleWorkload:
    """The same step through oracle/ (the reference's algorithm restated in torch, on the CPU)."""

    def __init__(self, cfg):
        from oracle import mesh as M
        self.M = M
        path = template_path()
        self.T = M.TemplateData(M.load_obj(path), path)
        self.gan = None
        self.render = "render" in cfg["kind"]
        if cfg["gan"]:
            from oracle import gan as OG                    # the CPU arms never import the product package (libb3d.so)
            self.OG, self.args = OG, gan_args(cfg["res"], cfg["nd"])
            self.sg, self.sd = OG.init_state(self.args, seed=4321)
            for sdict in (self.sg, self.sd):
                for k in OG.trainable(sdict):
                    sdict[k].requires_grad_(True)
            self.opt_g = torch.optim.Adam([self.sg[k] for k in OG.trainable(self.sg)], lr=1e-4, betas=(0.0, 0.9))
            self.opt_d = torch.optim.Adam([self.sd[k] for k in OG.trainable(self.sd)], lr=4e-4, betas=(0.0, 0.9))
            self.gan = True

    def render_step(self, d):
        from oracle import pointcloud as O
        M, T = self.M, self.T
        p, q, s = (d[k].clone().requires_grad_(True) for k in ("points", "quat", "scale"))
        sil = O.effective_loss_forward(p, q, s, V=V, kernel_size=21, sigma=3.0, mode="R")
        loss_pc = O.silhouette_mse_sum(sil, d["mask"])
        mm, tex = d["mesh_map"].clone().requires_grad_(True), d["tex"].clone().requires_grad_(True)
        raw = M.get_vertex_positions(T, mm)
        vtx = M.transform_vertices(raw, d["pscale"], d["ptrans"], d["rot"])
        img, alpha, _ = M.forward_renderer(T, vtx, tex, H, H)
        xf = torch.cat((img, alpha), dim=3).permute(0, 3, 1, 2)
        recon = torch.nn.functional.mse_loss(xf, d["x_real"])
        flat = M.loss_flat(T.ff, T.faces.shape[0], M.compute_normals(T, raw))
        loss = loss_pc + recon + FLAT_COEF * flat
        loss.backward()
        return loss.detach()

    def step(self, batches):
        if self.gan is None:
            return self.render_step(batches[0])
        OG, M, T = self.OG, self.M, self.T
        total = 0.0
        for it, d in enumerate(batches):
            if self.render:
                total = total + self.render_step(d)
            B = d["C"].shape[0]
            z = torch.randn(B, 64)
            if it == 0:
                self.opt_g.zero_grad(set_to_none=True)
                loss, tex, mesh, _, _ = OG.g_loss(self.sg, self.sd, self.args, z, d["C"], d["X_alpha"])
                flat = M.loss_flat(T.ff, T.faces.shape[0], M.compute_normals(T, M.get_vertex_positions(T, mesh)))
                (loss + 1e-4 * flat).backward()
                self.opt_g.step()
            else:
                self.opt_d.zero_grad(set_to_none=True)
                lf, lr, _ = OG.d_loss(self.sg, self.sd, self.args, z, d["C"], d["X_alpha"], d["X_tex"], d["X_mesh"])
                (lf + lr).backward()
                self.opt_d.step()
                loss = lf + lr
            total = total + loss.detach()
        return total


def cpu_inputs(cfg, sample_b):
    out = []
    for it in range(cfg["iters"]):
        d = host_inputs(sample_b, seed=1234 + 1000 * it, pin=False) if "render" in cfg["kind"] else {}
        if cfg["gan"]:
            d.update(gan_host_inputs(sample_b, seed=1234 + 1000 * it, pin=False, R=cfg["res"]))
        out.append(d)
    return out


def cpu_baseline(cfg, budget_s, sample_b=2):
    cores = cpu_threads()
    wl = OracleWorkload(cfg)
    d = cpu_inputs(cfg, sample_b)
    iters = 3 if cfg["gan"] else 1
    t0 = time.perf_counter()
    wl.step(d)                                             # warm-up (also sizes the timed part)
    warm = time.perf_counter() - t0
    nmax = max(1, min(8, int(budget_s / max(warm, 1e-3))))
    t0, n = time.perf_counter(), 0
    while n < nmax:
        wl.step(d)
        n += 1
    el = time.perf_counter() - t0
    return {"value": round(sample_b * iters * n / el, 4), "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{n} steps ({iters} iteration(s) each) of batch {sample_b} of the same workload through oracle/ "
                      f"(the reference's algorithm in torch on the CPU, {cores} threads)"}


def run_reference(args):
    if WORKLOADS[args.workload]["kind"] == "recon":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"impl": "reference", "unavailable": "cfg4: oracle/ has no restatement of the reconstruction network "
                              "(its goldens come from the reference module itself in the authoring container); the reference tree "
                              "cannot be installed or travel"}))
        return
    _run_reference(args)


def _run_reference(args):
    """The reference's own CPU implementation of the path (its algorithm restated in torch under oracle/ — the reference
    tree itself cannot be installed or travel, DESIGN.md §6) on THIS arm's config: the same batch per step, the same
    three iterations per step; bounded to one timed step (a step is ~100 s of CPU work at batch 32)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = WORKLOADS[args.workload]
    cores = cpu_threads()
    B, iters = cfg["batch"], (3 if cfg["gan"] else 1)
    if os.environ.get("B3D_REF_BATCH"):                      # development aid
        B = int(os.environ["B3D_REF_BATCH"])
    wl = OracleWorkload(cfg)
    d = cpu_inputs(cfg, B)
    warm = 0 if cfg["gan"] else min(args.warmup, 1)
    for _ in range(warm):
        wl.step(d)
    steps = 1 if cfg["gan"] else max(1, min(args.steps, 3))
    t0 = time.perf_counter()
    for _ in range(steps):
        wl.step(d)
    el = time.perf_counter() - t0
    v = B * iters * steps / el
    sample = (f"{steps} step(s) ({iters} iteration(s) each) of batch {B} (the workload's own batch) through oracle/ = the "
              f"reference's algorithm in torch on the CPU, {cores} threads")
    print(json.dumps({
        "impl": "reference", "metric": cfg["metric"], "value": round(v, 4), "unit": "images/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": round(el / steps * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["name"], "batch_per_gpu": B, "global_batch": B, "iterations_per_step": iters,
                   "points": N_PTS, "voxels": V, "image": H, "faces": 960, "texture": TEX, "semantics": "R",
                   "fresh_batch_per_iteration": True},
        "cpu_baseline": {"value": round(v, 4), "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 4), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b3d", choices=["b3d", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to "
                    "DIR/<name>.npy (float32, seeded inputs: compare two builds output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b3d":
        args.warmup = 3
    (run_reference if args.impl == "reference" else run_cuda)(args)


if __name__ == "__main__":
    main()
