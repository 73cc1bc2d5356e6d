#!/usr/bin/env python
"""bench.py -- headline benchmark of the PermutoSDF hot path on B200 (contract: see DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA kernels through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  reference arm: the CPU (PyTorch-only) restatement of the
                                                           reference's encoding+MLP step on the host cores

Workload (BASELINE.json configs[1], "C2"): one training iteration of PermutoSDF (train_permuto_sdf.py:311-422,
--with_mask) on synthetic data: 512 rays x (96 occupancy-grid samples + 2x16 importance samples) = 128 samples/ray
(65 536 samples when every ray hits), 16-level permutohedral lattice (2^18 x 2 per level), 3x64 SDF MLP,
Lipschitz RGB MLP, 256^3 occupancy grid of the analytic sphere SDF |x|-0.3. A step = ray generation, sampling,
importance resampling, forward, losses, backward through the double backward, dense AdamW.
  python bench.py --rays 8192 ...                          same step with more rays per GPU (BASELINE config 4 = 8192 rays/GPU x 8 GPUs)
  python bench.py --workload sphere_trace [--gpus N]       sphere-traced render of one 1920x1080 frame (BASELINE config 5): px/s
  python bench.py ... --dump-outputs DIR                   training workload: after the timed steps, write what the last one computed
                                                           as DIR/<name>.npy

Metric: rays/s (whole job). `value`: inputs resident on the device. `e2e`: per step the ray indices come from pinned
host memory and the loss is read back. Multi-GPU: rays sharded by rank (weak scaling), one NCCL all-reduce of the
flat gradient buffer per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "compat")]

NR_RAYS = 512
SAMPLES_PER_RAY = 128
WORKLOAD = "C2: 512 rays x 128 samples (96 grid + 2x16 importance), 16-level lattice 2^18x2, 3x64 SDF MLP, RGB Lipschitz MLP, 256^3 occupancy, analytic sphere SDF"
METRIC = "rays/sec (train fwd+bwd+AdamW, 512 rays x 128 samples x 16 levels x 2 feat)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons during the timed region. NVML is polled every ~2 ms from a thread (a 34 ms timed region gets ~15
    samples); falls back to nvidia-smi (one sample per ~0.2 s) when the NVML binding is not importable."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.stop, self.th = index, [], False, None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run_nvml(self):
        n = self.nvml
        R = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        bits = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}
        while not self.stop:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                r = int(R(self.h))
                self.rows.append((sm, self.max_sm, [k for k, b in bits.items() if r & b]))
            except Exception:
                pass
            time.sleep(0.002)

    def _run_smi(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                if out:
                    c = [t.strip() for t in out.split(",")]
                    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                    self.rows.append((float(c[0]), float(c[1]), [nm for i, nm in enumerate(names) if c[2 + i].lower().startswith("active")]))
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.th = threading.Thread(target=self._run_nvml if self.nvml is not None else self._run_smi, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [r[0] for r in self.rows]
        reasons = sorted({x for r in self.rows for x in r[2]})
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(r[1] for r in self.rows), "reasons": reasons, "samples": len(self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def analytic_reel(nimg, H, W, f, device):
    """TensorReel-shaped synthetic data: cameras on a radius-1.2 sphere looking at a shaded sphere of radius 0.3"""
    g = torch.Generator().manual_seed(123)
    rgb = torch.zeros(nimg, 3, H, W)
    mask = torch.zeros(nimg, 1, H, W)
    K = torch.zeros(nimg, 3, 3)
    tf = torch.zeros(nimg, 4, 4)
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32) + 0.5, torch.arange(W, dtype=torch.float32) + 0.5, indexing="ij")
    for i in range(nimg):
        c = torch.randn(3, generator=g); c = 1.2 * c / c.norm()
        zaxis = -c / c.norm()
        up = torch.tensor([0.0, 1.0, 0.0])
        xaxis = torch.linalg.cross(up, zaxis); xaxis = xaxis / xaxis.norm()
        yaxis = torch.linalg.cross(zaxis, xaxis)
        R = torch.stack([xaxis, yaxis, zaxis], 1)
        K[i] = torch.tensor([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1.0]])
        tf[i, :3, :3], tf[i, :3, 3], tf[i, 3, 3] = R, c, 1.0
        dcam = torch.stack([(xs - W / 2.0) / f, (ys - H / 2.0) / f, torch.ones_like(xs)], -1)
        d = dcam @ R.t()
        d = d / d.norm(dim=-1, keepdim=True)
        b = (d * c).sum(-1); disc = b * b - (c.dot(c) - 0.09)
        hit = disc > 0
        t = -b - torch.sqrt(disc.clamp(min=0))
        n = torch.nn.functional.normalize(c + t[..., None] * d, dim=-1)
        col = (0.5 + 0.5 * n).permute(2, 0, 1)
        rgb[i] = col * hit[None]
        mask[i, 0] = hit.float()

    class Reel:
        pass
    r = Reel()
    r.rgb_reel, r.mask_reel, r.K_reel, r.tf_world_cam_reel = rgb.to(device), mask.to(device), K.to(device), tf.to(device)
    return r


def central_pixels(n, H, W, box, gen):
    """pixel indices inside the central box x box window (all those rays hit the object)"""
    x = torch.randint(W // 2 - box // 2, W // 2 + box // 2, (n,), generator=gen)
    y = torch.randint(H // 2 - box // 2, H // 2 + box // 2, (n,), generator=gen)
    return (y * W + x).to(torch.int32)


def run_ours(args):
    global NR_RAYS
    import torch.distributed as dist
    from permuto_sdf_b200 import _lib, load_library
    from permuto_sdf_b200.dist import FlatGrads
    from permuto_sdf_b200.permuto_sdf import PermutoSDF
    from permuto_sdf_b200.train import HyperParams, Trainer
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = load_library()
    assert lib.psdf_device_ok() == 1

    hp = HyperParams()
    hp.max_nr_samples_per_ray = SAMPLES_PER_RAY - 2 * 16
    hp.nr_samples_imp_sampling = 16
    NR_RAYS = int(args.rays)
    hp.nr_rays = NR_RAYS
    tr = Trainer(hp, nr_levels=16, capacity=2 ** 18, sdf_hidden=64, nr_images=8, occupancy_resolution=256, seed=0,
                 fused_inference=not args.modular, fused_training=not args.modular, optimizer="adamw" if args.modular else "fused")
    tr.set_analytic_scene()
    tr.iter_nr = 20000          # past coarse-to-fine: all 16 levels active, cos-anneal half way
    graphed = not (args.modular or args.eager)
    graphed_mode = graphed
    if graphed:
        tr.enable_cuda_graph(warmup_steps=3)
    H, W, f = 600, 800, 1000.0
    reel = analytic_reel(8, H, W, f, dev)
    flat = None
    if world > 1 and not hasattr(tr.optimizer, "flat_grad"):
        flat = FlatGrads(tr.params)

    total = args.steps + args.warmup
    gen = torch.Generator().manual_seed(1000 + rank)
    pix_host = [central_pixels(NR_RAYS, H, W, 300, gen).pin_memory() for _ in range(total)]
    img_host = [torch.randint(0, 8, (NR_RAYS,), generator=gen, dtype=torch.int32).pin_memory() for _ in range(total)]
    pix_dev = [p.to(dev) for p in pix_host]
    img_dev = [p.to(dev) for p in img_host]

    dp_mode = os.environ.get("PSDF_DP_MODE", "peer")        # peer | nccl | nccl_overlap | legacy
    if world > 1 and flat is None and dp_mode != "legacy":
        # peer: fused gradient reduction + AdamW + parameter broadcast over NVLink peer memory (no all-reduce); nccl: one all-reduce
        # captured in the optimizer graph; nccl_overlap: bucketed all-reduce overlapped with the SDF backward / AdamW
        tr.enable_data_parallel(world, overlap=(dp_mode == "nccl_overlap"), mode="peer" if dp_mode == "peer" else "nccl")
    start = StartState(tr) if args.dump_outputs else None      # before the first step (the peer mode above re-homes the buffers)

    def one_step(i, e2e):
        # e2e: the step's inputs start in pinned host memory; otherwise they are device resident
        pix, img = (pix_host[i], img_host[i]) if e2e else (pix_dev[i], img_dev[i])
        dp = tr._dp is not None
        # device-resident indices were materialised before the synchronize() that precedes the timed region (inputs_ready): the
        # parameter-free head of the iteration may then start beside the previous optimizer step
        # e2e: the loss is read through Trainer's HostLoss handle (device -> pinned host copy queued right behind the forward/backward
        # graph): float(loss) below waits for that copy, not for the optimizer step, so the host launches the next step's head beside it
        loss = tr.step_from_reel(reel, pix, img, update_occupancy=(i % 8 == 0), optimizer_step=(world == 1 or dp), inputs_ready=not e2e,
                                 loss_to_host=e2e and graphed_mode)
        if world > 1 and not dp:
            # legacy path (PSDF_DP_MODE=legacy): one blocking NCCL all-reduce of the flat gradient buffer between the two graphs
            dist.all_reduce(tr.optimizer.flat_grad if flat is None else flat.flat, op=dist.ReduceOp.SUM)
            tr.optimizer_step(grad_scale=1.0 / world)
        if e2e:
            return float(loss)          # device -> host read of the step's result
        return loss

    if graphed:
        # setup, not part of the W warm-up steps: 3 eager static-shape iterations + the iteration that captures the graphs
        for i in range(5):
            one_step(i % total, False)
        torch.cuda.synchronize()

    static_eager = False
    last = {}

    def timed(e2e, with_events, steps=None):
        steps = args.steps if steps is None else steps
        for i in range(args.warmup):
            one_step(i, e2e)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        _lib.stats_begin(with_events=with_events)
        evs = []
        nsamples = 0
        with ClockSampler(local) as cs:
            for i in range(args.warmup, args.warmup + steps):
                if start is not None and e2e and i == args.warmup + steps - 1:
                    start.restore()             # the last timed step: its inputs are the same in every run
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                last["loss"] = one_step(i, e2e)
                e.record()
                evs.append((s, e))
                if not graphed:
                    nsamples += int(tr.last["nr_samples_dev"]) if static_eager else tr.last["nr_samples"]
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = sum(s.elapsed_time(e) for s, e in evs)
        calls, launches, times = _lib.stats_end()
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, times, cs.summary(), nsamples / steps

    ms_dev, launches, ktimes, clocks, avg_samples = timed(e2e=False, with_events=not graphed)
    ms_e2e, _, _, clocks2, _ = timed(e2e=True, with_events=False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, training_outputs(tr, last["loss"]))
    ms_per_step = ms_dev / args.steps
    prof_steps = 0
    if graphed:
        # kernels inside the replayed graphs (counted at capture) + the eager calls of the timed region (occupancy refresh)
        launches += tr.graph_launches_per_step() * args.steps
        # per-kernel CUDA-event times and the sample count come from a few iterations of the same workload afterwards, outside the
        # timed region (events cannot bracket individual kernels of a replayed graph): same static-capacity containers and
        # device-resident generators / schedule as under replay, but every kernel launched from Python
        tr._cg["fb"], tr._cg["opt"], tr._cg["occ"], tr._cg["warm"] = None, {}, None, 1 << 30
        graphed, static_eager = False, True
        prof_steps = min(args.steps, 5)
        ms_prof, _, ktimes, _, avg_samples = timed(e2e=False, with_events=True, steps=prof_steps)
        sc = args.steps / prof_steps                                  # rescale to the timed region's step count
        ktimes = {k: (n * sc, t * sc) for k, (n, t) in ktimes.items()}
    rays_total = NR_RAYS * world * args.steps
    value = rays_total / (ms_dev / 1e3)
    e2e_value = rays_total / (ms_e2e / 1e3)

    # ---- roofline of the dominant kernel of OUR library inside the timed region (CUDA events on the launch stream)
    hbm, peak_src = peaks()
    L, C = 16, 36
    alg_bytes = {   # algorithmic bytes per SAMPLE, SURVEY.md 8(d); multiplied by the samples the timed launches actually processed
        "psdf_enc_forward": 12 + L * 4 * 8 + C * 4,
        "psdf_enc_backward": 12 + L * 8 + L * 4 * 8 + L * 4 * 8,
        "psdf_enc_double_backward": 12 + 12 + L * 8 + L * 4 * 8 + L * 4 * 8 + C * 4,
        "psdf_sdf_fused_forward": 12 + L * 4 * 8 + 4 + 12 + 128,
        "psdf_sdf_fused_backward": 12 + 2 * L * 4 * 8 + 4 + 12 + 128,
        "psdf_sdf_fused_forward_multi": 12 + L * 4 * 8 + 4 + 12 + 128,
        "psdf_sdf_fused_backward_multi": 12 + 2 * L * 4 * 8 + 4 + 12 + 128,
        "psdf_rgb_fused_forward": 12 + L * 4 * 8 + 12 + 12 + 128 + 12,
        "psdf_rgb_fused_backward": 12 + 2 * L * 4 * 8 + 12 + 12 + 128 + 12 + 12 + 128,
        "psdf_rgb_fused_backward_acc": 12 + 2 * L * 4 * 8 + 12 + 12 + 128 + 12 + 12 + 128,
    }
    units = dict(_lib.LAST_UNITS)
    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the tracked `ncu --set full` capture of this workload
    ncu_traffic = ncu_traffic_from_profiles()
    roof = None
    if ktimes:
        top = sorted(((v[1], k) for k, v in ktimes.items()), reverse=True)
        name = next((k for _, k in top if k in alg_bytes), top[0][1])
        n, tot_ms = ktimes[name]
        per_launch_s = tot_ms / n / 1e3
        # samples processed by the timed launches of this entry point (the profiling pass is rescaled to the timed step count)
        nsamp = units.get(name, 0) * (args.steps / prof_steps if prof_steps else 1.0)
        ach = (alg_bytes[name] * nsamp / (tot_ms / 1e3) / 1e9) if name in alg_bytes and nsamp else None
        roof = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": (ach / hbm) if ach else None,
                "traffic": ncu_traffic.get(name), "launches": n, "avg_us": per_launch_s * 1e6, "samples_per_launch": nsamp / n if n else None,
                "peak_source": peak_src,
                "share_of_step": tot_ms / ms_dev,
                "top5_ms_per_step": {k: round(v / args.steps, 4) for v, k in top[:5]},
                "calls_per_step": {k: round(ktimes[k][0] / args.steps, 2) for _, k in top[:12]}}

    out = None
    if rank == 0:
        cpu = cpu_baseline(sample_rays=8, steps=3, warmup=1)
        out = {
            "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "ours",
            "config": {"workload": WORKLOAD if NR_RAYS == 512 else WORKLOAD.replace("512 rays", "%d rays" % NR_RAYS).replace("C2:", "C2 shape at %d rays/GPU (BASELINE config 4 when 8192 x 8 GPUs):" % NR_RAYS),
                       "rays_per_gpu": NR_RAYS, "avg_samples_per_step": avg_samples, "parallelism": "dp%d" % world, "gradient_exchange": (dp_mode if world > 1 else None),
                       "l2": "per-step working set (2 lattice tables + grads + Adam moments ~0.4 GB) exceeds the 126 MB L2; no explicit flush",
                       "timed_region": "sum of per-step CUDA-event intervals",
                       "execution": "eager" if (args.modular or args.eager) else "CUDA graphs (forward+backward graph, optimizer graph), static-capacity containers"},
            "e2e": {"value": e2e_value, "unit": "rays/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": NR_RAYS * 4 * 2 * world,
                    "d2h_bytes_per_step": 4 * world},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        }
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def run_sphere_trace(args):
    """BASELINE config 5: sphere-traced render (train_permuto_sdf.py:211-242, sdf_utils.py:120-218) of one 1920x1080 frame, 256
    iterations max, occupancy grid on, normals + colour included. N GPUs: the image is tiled by rows, every rank traces its tile and
    one NCCL all_gather assembles the frame on all ranks. `value`: camera already on the device, image stays there; `e2e`: camera
    (K, pose) from pinned host memory, finished image copied back to pinned host memory inside the timed region."""
    import torch.distributed as dist
    import permuto_sdf_b200.train as T
    from permuto_sdf_b200 import _lib, load_library
    from permuto_sdf_b200.train import HyperParams, Trainer
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert load_library().psdf_device_ok() == 1
    W, H = args.width, args.height
    hp = HyperParams()
    tr = Trainer(hp, nr_levels=16, capacity=2 ** 18, sdf_hidden=64, nr_images=8, occupancy_resolution=256, seed=0, optimizer="fused")
    tr.set_analytic_scene()
    m = tr.model_sdf
    # fit the SDF to the analytic sphere of the scene (the reference's sphere initialisation, train_permuto_sdf.py:262-291): rays then
    # converge on a surface inside the occupied shell like on a trained model. Same seed on every rank -> identical replicas.
    for i in range(400):
        loss, _, _ = T.loss_sphere_init(30000, tr.aabb, m, 20000)
        tr.optimizer.zero_grad(set_to_none=False)
        loss.backward()
        tr.optimizer_step()
    m.eval(); tr.model_rgb.eval()
    m.last_iter_nr = 20000
    torch.set_grad_enabled(False)
    rows = [(H * r) // world for r in range(world + 1)]
    r0, r1 = rows[rank], rows[rank + 1]
    cam_host = torch.tensor([1.2 * W, W / 2.0, H / 2.0, 0.0, 0.0, -1.5], dtype=torch.float32).pin_memory()   # f, cx, cy, camera centre
    img_host = torch.empty(H, W, 3, dtype=torch.float32).pin_memory()
    cam_dev = cam_host.to(dev)
    tile_rows = max(b - a for a, b in zip(rows[:-1], rows[1:]))
    gathered = torch.zeros(world, tile_rows * W, 3, device=dev)
    stats = {"evals": 0, "rays": 0}

    def frame(e2e):
        cam = cam_host.to(dev, non_blocking=True) if e2e else cam_dev
        # primary rays of this rank's rows (pixel centres; CreateRaysModule of the reference, models/modules.py:170-230). The camera sits on
        # the -z side looking along +z: rays leave the grid through a POSITIVE face. Rays that leave through a negative face are never
        # flagged out of bounds by the reference's marcher (float -> uint saturation, SURVEY.md A.2, reproduced bit for bit): they alias
        # voxel column 0, exhaust the DDA step budget in every iteration and burn all 256 iterations far outside the scene.
        v, u = torch.meshgrid(torch.arange(r0, r1, device=dev, dtype=torch.float32), torch.arange(W, device=dev, dtype=torch.float32), indexing="ij")
        d = torch.stack([(u + 0.5 - cam[1]) / cam[0], (v + 0.5 - cam[2]) / cam[0], torch.ones_like(u)], -1).reshape(-1, 3)
        d = torch.nn.functional.normalize(d, dim=-1).contiguous()
        o = cam[3:6].expand_as(d).contiguous()
        rgb, normals, wsum = T.run_net_sphere_traced(o, d, hp, m, tr.model_rgb, tr.occupancy_grid, 20000, args.trace_iters, 0.9, 2e-4)
        if world > 1:
            mine = torch.zeros(tile_rows * W, 3, device=dev)
            mine[: rgb.shape[0]] = rgb
            dist.all_gather_into_tensor(gathered.view(-1), mine.view(-1))      # the single collective of this path
            img = torch.cat([gathered[r, : (rows[r + 1] - rows[r]) * W] for r in range(world)], 0)
        else:
            img = rgb
        if e2e:
            img_host.view(-1, 3).copy_(img, non_blocking=True)
        return img

    def timed(e2e, with_events):
        for _ in range(args.warmup):
            frame(e2e)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        _lib.stats_begin(with_events=with_events)
        evs = []
        with ClockSampler(local) as cs:
            for _ in range(args.steps):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                frame(e2e)
                if with_events and getattr(m.fused, "last_trace_stats", None) is not None:
                    stats["evals"] += int(m.fused.last_trace_stats[1]); stats["rays"] += 1
                e.record()
                evs.append((s, e))
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = sum(s.elapsed_time(e) for s, e in evs)
        calls, launches, times = _lib.stats_end()
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, times, cs.summary()

    ms_dev, launches, _, clocks = timed(False, False)
    ms_e2e, _, _, _ = timed(True, False)
    _, _, ktimes, _ = timed(False, True)               # per-kernel CUDA-event times (serialising events: outside the reported time)
    hbm, peak_src = peaks()
    roof = None
    name = "psdf_sdf_sphere_trace"
    if name in ktimes and stats["rays"]:
        n, tot_ms = ktimes[name]
        evals_per_launch = stats["evals"] / stats["rays"]
        alg = 12 + 16 * 4 * 8                      # per network evaluation: position + 16 levels x 4 vertices x 8 B (SURVEY.md 8d, fused: no feature write)
        ach = alg * evals_per_launch * n / (tot_ms / 1e3) / 1e9
        top = sorted(((v[1], k) for k, v in ktimes.items()), reverse=True)
        roof = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "traffic": ncu_traffic_from_profiles().get(name),
                "launches": n, "avg_us": tot_ms / n * 1e3, "network_evaluations_per_launch": evals_per_launch, "peak_source": peak_src,
                "share_of_step": tot_ms / n / (ms_dev / args.steps), "top5_ms_per_step": {k: round(v / args.steps, 4) for v, k in top[:5]}}
    if rank == 0:
        px = W * H * args.steps
        out = {"metric": "sphere-trace px/sec (%dx%d, %d iterations max, occupancy grid on, normals + colour)" % (W, H, args.trace_iters),
               "value": px / (ms_dev / 1e3), "unit": "px/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "impl": "ours",
               "config": {"workload": "C5: sphere-trace inference %dx%d, %d max steps, OccupancyGrid 256^3 on, 16-level lattice 2^18x2, 3x64 SDF MLP fitted "
                                      "to the analytic sphere, RGB Lipschitz MLP; image tiled by rows over the ranks + one all_gather" % (W, H, args.trace_iters),
                          "parallelism": "tiles%d" % world, "l2": "lattice table 33.5 MB + 16.8 MB occupancy are L2 resident by design; no flush",
                          "timed_region": "sum of per-frame CUDA-event intervals"},
               "e2e": {"value": px / (ms_e2e / 1e3), "unit": "px/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": 24 * world,
                       "d2h_bytes_per_step": W * H * 3 * 4},
               "gpu_launches": launches, "clocks": clocks, "roofline": roof}
        with torch.enable_grad():
            out["cpu_baseline"] = cpu_baseline(sample_rays=8, steps=3, warmup=1)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_SAMPLE = 1 << 20          # entries kept of each large state buffer by --dump-outputs
DUMP_LIMIT = 64 << 20


class StartState:
    """The model state a Trainer is built with (parameters, AdamW moments, occupancy grid), put back in place before the last timed
    step when outputs are dumped. Every training step accumulates gradients, losses and grid updates with floating-point atomics in
    an order that changes from run to run, and AdamW (eps 1e-15) and the curvature loss magnify those last-bit differences: after 25
    steps of this workload the losses of two runs differed by up to 15 % (B200, 1000 W). Restored, the last step reads the same
    parameters, grid and rays in every run, so its outputs differ only by the rounding of that one step."""

    def __init__(self, tr):
        opt, grid = tr.optimizer, tr.occupancy_grid
        if not hasattr(opt, "flat_param"):
            raise RuntimeError("--dump-outputs needs the flat-buffer optimizer (not --modular)")
        self.tr = tr
        self.live = [opt.flat_param, opt.exp_avg, opt.exp_avg_sq, grid.get_grid_values(), grid.get_grid_occupancy()]
        self.saved = [t.clone() for t in self.live]

    def restore(self):
        for dst, src in zip(self.live, self.saved):
            dst.copy_(src)
        fused = getattr(self.tr.model_sdf, "fused", None)
        if fused is not None:
            fused.repack()                      # the fused SDF kernels read a packed copy of the MLP weights
        torch.cuda.synchronize()                # graphs on other streams read these buffers too


def training_outputs(tr, loss):
    """What a training step leaves its caller: the loss and its terms, the sample count, and the parameters and AdamW moments the
    optimizer step wrote (a fixed seeded sample of DUMP_SAMPLE entries of each: the flat buffers hold ~17M floats apiece)."""
    out = {"loss": np.array([float(loss)], np.float64)}
    for k in ("loss_rgb", "loss_eikonal", "loss_curvature", "nr_samples_dev"):
        if torch.is_tensor(tr.last.get(k)):
            out[k] = tr.last[k].detach().double().cpu().numpy().reshape(-1)
    opt = tr.optimizer
    if hasattr(opt, "flat_param"):
        bufs = {"params": opt.flat_param, "adam_exp_avg": opt.exp_avg, "adam_exp_avg_sq": opt.exp_avg_sq}
    else:
        bufs = {"params": torch.cat([p.detach().reshape(-1) for p in tr.params])}
    for name, b in bufs.items():
        n = b.numel()
        idx = np.sort(np.random.RandomState(0).choice(n, min(n, DUMP_SAMPLE), replace=False))
        out[name + "_sample"] = b.detach().reshape(-1)[torch.from_numpy(idx).to(b.device)].float().cpu().numpy()
    return out


def dump_outputs(d, arrays):
    """DIR/<name>.npy per array (float32 / float64), at most DUMP_LIMIT bytes in all"""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d byte limit" % (total, DUMP_LIMIT))
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(d, name + ".npy"), a)


NCU_KERNEL_OF = {"psdf_sdf_fused_forward": "k_sdf_fused_dual", "psdf_sdf_fused_backward": "k_sdf_fused_backward",
                 "psdf_sdf_fused_forward_multi": "k_sdf_fused_dual", "psdf_sdf_fused_backward_multi": "k_sdf_fused_backward",
                 "psdf_rgb_fused_forward": "k_rgb_fused", "psdf_rgb_fused_backward": "k_rgb_fused_backward",
                 "psdf_rgb_fused_backward_acc": "k_rgb_fused_backward",
                 "psdf_sdf_sphere_trace": "k_sdf_sphere_trace"}


def ncu_traffic_from_profiles():
    """entry point -> DRAM bytes (read + write) per launch, read from the newest tracked profiles/r*_ncu_kernels.csv (65 536-sample
    launches of the bench workload). None for kernels the capture does not hold."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_kernels.csv")))
    out = {}
    if not files:
        return out
    rows = list(csv.DictReader(open(files[-1])))
    for entry, kern in NCU_KERNEL_OF.items():
        for r in rows:
            if r.get("kernel", "").startswith(kern):
                try:
                    out[entry] = (float(r["dram__bytes_read.sum [Mbyte]"]) + float(r["dram__bytes_write.sum [Mbyte]"])) * 1e6
                except (KeyError, ValueError):
                    pass
                break
    return out


def cpu_baseline(sample_rays, steps, warmup, threads=None):
    """the reference path restated on the CPU (PyTorch only), bounded sample of the same workload"""
    from oracle.cpu_step import time_cpu_step
    threads = threads or min(os.cpu_count() or 1, 32)      # the 65-sample-per-ray port does not scale past a few dozen threads
    med, ts = time_cpu_step(sample_rays, SAMPLES_PER_RAY, steps, warmup, threads)
    return {"value": sample_rays / med, "unit": "rays/s", "cores": threads, "cores_available": os.cpu_count(),
            "threads_note": "the port's per-step work (tens of samples per thread) stops scaling past ~32 threads; more threads measured slower",
            "kind": "port",
            "sample": "%d rays x %d samples per step, %d steps, median; SDF encoding + 3x64 MLP forward, d sdf/dx, eikonal + feature loss, backward "
                      "(double backward); the reference has no CPU path, this is the oracle restatement" % (sample_rays, SAMPLES_PER_RAY, steps),
            "seconds_per_step": med}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    sample_rays = 16
    cpu = cpu_baseline(sample_rays, steps=args.steps, warmup=min(args.warmup, 2))
    out = {"metric": METRIC, "value": cpu["value"], "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": cpu["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "impl": "reference",
           "config": {"workload": WORKLOAD, "note": "CPU PyTorch-only restatement on the host cores; each step is a bounded sample of %d rays" % sample_rays},
           "cpu_baseline": cpu, "e2e": {"value": cpu["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--eager", action="store_true", help="launch every kernel from Python (no CUDA-graph replay)")
    ap.add_argument("--modular", action="store_true", help="drop-in API path only (encoding kernels + torch MLP), no fused tcgen05 kernels")
    ap.add_argument("--rays", type=int, default=512, help="rays per GPU and step (512 = BASELINE config 2, 8192 = config 4 per GPU)")
    ap.add_argument("--workload", default="train", choices=["train", "sphere_trace"])
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--trace_iters", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "train" or args.impl != "ours"):
        # the sphere-trace frame is rendered from a 400-step SDF fit that accumulates with atomics like training (see StartState): two
        # runs gave frames differing in ~5 % of the pixel values (B200, 1000 W)
        ap.error("--dump-outputs covers the training workload of our implementation")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "sphere_trace":
        run_sphere_trace(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
