#!/usr/bin/env python
"""bench.py -- views/sec forward+backward of the feature-Gaussian rasterizer (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c3] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

Workload (config.workload): BASELINE.json configs[2] = "c3": 1M synthetic Gaussians, 1920x1080, SH degree 3,
feature dim 128, forward + backward.  One *step* = every rank renders `views_per_rank` distinct cameras
(forward + backward through the public GaussianRasterizer autograd API, gradients accumulating in one flat
fp32 buffer) and then the step's single gradient all-reduce (N > 1).  Weak scaling: per-rank work is fixed.

JSON keys beyond the base contract:
  value     device-resident throughput: cameras and upstream gradients already in HBM, CUDA-event timed.
  e2e       same metric through the same public API with the per-view camera coming from pinned host memory
            (H2D inside the timed region), a scalar loss built on the device and read back to the host every
            step (D2H).  The Gaussian parameters are the model state and stay resident, as in train.py.
  roofline  dominant kernel of OUR library: algorithmic bytes (SURVEY.md section 8d formulas with the measured V, R)
            / its mean launch duration, measured live with CUDA events on the launch stream inside the timed
            region (f3dgs_profile_*), against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline  the CPU oracle (oracle/, a port: the reference has no CPU implementation) on a bounded tile
            sample of the same workload, all host cores, rank 0 at N=1 only.
`--impl reference` runs the UNMODIFIED reference CUDA extension (oracle/_ref, built from /root/reference's own
sources for sm_100a) through the identical procedure: the north star compares against "the reference's own
rasterizer timed on the same box".  If oracle/_ref is missing it falls back to timing the CPU oracle port.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "feature-3dgs_b200"))

import scenegen  # noqa: E402

METRIC = "views/sec fwd+bwd @1M Gaussians/1080p/feat_dim=128"
STAGES = ["preprocess_fwd", "scan", "duplicate_keys", "sort", "tile_ranges", "composite_fwd", "composite_bwd",
          "preprocess_bwd"]


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                 "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 60 << 20  # array data; with the .npy headers the files stay under 64 MB


class OutputDump:
    """--dump-outputs: what the timed `value` path computed in its last step, written as DIR/<name>.npy in float32.
    Per-view outputs (color, feature_map, depth, radii and, through the autograd API, grad_means2D) are stacked over
    this rank's views; the parameter gradients are the step's accumulated (all-reduced) ones.  So that the whole dump stays within DUMP_BYTES, an array with more than
    `cap` elements is replaced by a fixed sample of its flat elements (sorted indices drawn with numpy PCG64 seed 0, the
    same for every view and every run with the same arguments), stored as [views, cap] / [cap]."""

    def __init__(self, n_views, n_arrays):
        self.n_views, self.cap = n_views, DUMP_BYTES // 4 // n_arrays
        self.sel, self.bufs = {}, {}

    def _select(self, name, x):
        import torch

        if name not in self.sel:
            n = x.numel()
            self.sel[name] = None if n <= self.cap else torch.from_numpy(
                np.sort(np.random.Generator(np.random.PCG64(0)).choice(n, self.cap, replace=False))).to(x.device)
        return self.sel[name]

    def keep(self, view, **outs):
        """Inside the timed step: device-side copies / gathers into buffers allocated on the first (warm-up) step."""
        import torch

        for name, x in outs.items():
            if x.numel() == 0:
                continue
            x = x.detach()
            sel = self._select(name, x)
            if name not in self.bufs:
                shape = tuple(x.shape) if sel is None else (sel.numel(),)
                self.bufs[name] = x.new_empty((self.n_views,) + shape)
            if sel is None:
                self.bufs[name][view].copy_(x)
            else:
                torch.index_select(x.reshape(-1), 0, sel, out=self.bufs[name][view])

    def write(self, out_dir, grads):
        arrays = dict(self.bufs)
        for name, g in grads.items():
            sel = self._select(name, g)
            arrays[name] = g.detach() if sel is None else g.detach().reshape(-1)[sel]
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())
        log(f"dump-outputs: {len(arrays)} arrays to {out_dir}: " + ", ".join(
            f"{k}{list(a.shape)}" for k, a in sorted(arrays.items())))


def algorithmic_bytes(V, R, tiles, HW, C):
    """SURVEY.md section 8(d): compulsory traffic of the two composite kernels, bytes per view."""
    fwd = V * (4 * C + 40) + 4 * R + 8 * tiles + HW * (4 * C + 24)
    bwd = V * 40 + 4 * R + 8 * tiles + HW * (4 * C + 24) + V * (4 * C + 48)
    return {"composite_fwd": fwd, "composite_bwd": bwd}


def cpu_baseline(scene, cfg, sample_div=16):
    """CPU oracle port on a bounded tile sample of the same view (preprocess + binning in full)."""
    import oracle

    cores = os.cpu_count() or 1
    oracle.set_threads(cores)
    cam = scene.cameras[0]
    W, H, C = cam.image_width, cam.image_height, scene.C
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    t0 = time.time()
    f = oracle.forward(scene, cam, render=False)
    t_front = time.time() - t0
    # contiguous band of tile rows through the image centre
    n = max(tiles // sample_div, 1)
    b = (tiles - n) // 2
    f.update(final_T=np.ones((H, W), np.float32), n_contrib=np.zeros((H, W), np.uint32),
             color=np.zeros((3, H, W), np.float32), feature_map=np.zeros((C, H, W), np.float32),
             depth=np.zeros((1, H, W), np.float32))
    L = oracle.lib()
    p = oracle._p
    feats = np.ascontiguousarray(scene.features.reshape(scene.P, C))
    t0 = time.time()
    L.oracle_render(W, H, C, p(f["ranges"]), p(f["point_list"]), p(f["means2D"]), p(f["colors"]), p(feats),
                    p(f["depths"]), p(f["conic_opacity"]), p(scene.bg), p(f["final_T"]), p(f["n_contrib"]),
                    p(f["color"]), p(f["feature_map"]), p(f["depth"]), b, b + n)
    t_fwd = time.time() - t0
    gc, gf, gd = (np.ones((3, H, W), np.float32), np.ones((C, H, W), np.float32), np.ones((1, H, W), np.float32))
    t0 = time.time()
    oracle.backward(scene, cam, f, gc, gf, gd, tile_range=(b, b + n))
    t_bwd = time.time() - t0
    est = t_front + (t_fwd + t_bwd) * (tiles / n)
    return {"value": 1.0 / est, "unit": "views/s", "cores": cores, "kind": "port",
            "sample": f"preprocess+binning in full ({t_front:.2f}s) + composite fwd ({t_fwd:.2f}s) and bwd+preprocess_bwd "
                      f"({t_bwd:.2f}s) on {n} of {tiles} tiles (centre band), composite time scaled by {tiles / n:.1f}; "
                      f"{cfg}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=list(scenegen.CONFIGS))
    ap.add_argument("--views-per-rank", type=int, default=8,
                    help="views each rank renders per step (weak scaling; 8 x 8 GPUs = the 64-view batch of BASELINE config 4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--api", default="batch", choices=["batch", "autograd"],
                    help="ours only: 'batch' = ViewBatch (autograd-free forward + in-kernel gradient accumulation, the "
                         "framework's own view-batch API); 'autograd' = the reference-compatible GaussianRasterizer autograd API. "
                         "The line's value/e2e use this API; the other one is measured too and reported under config.")
    ap.add_argument("--batch-views", type=int, default=64,
                    help="config c4 only: size of the view batch sharded over the ranks (BASELINE: 64)")
    ap.add_argument("--l2-flush", action="store_true",
                    help="write a 512 MB buffer between timed steps (outside the per-step event pairs)")
    ap.add_argument("--ref-debug", action="store_true",
                    help="reference arm only: debug=True, the reference scripts' default (arguments/__init__.py:71)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of `value`, write what its last step computed (per-view outputs and the "
                         "step's gradients) to DIR/<name>.npy, float32, at most 64 MB (larger arrays as a fixed seeded "
                         "sample); the copies run inside the timed steps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        log(f"note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    distributed = world > 1
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", f"ref_rast_C{scenegen.CONFIGS[args.config]['C'] or 1}.so"))

    cfgd = scenegen.CONFIGS[args.config]
    fwd_only = args.config == "c5"          # BASELINE.json configs[4]: forward-only render throughput
    strong = args.config == "c4"            # BASELINE.json configs[3]: one 64-view batch sharded over the ranks
    mode = "fwd-only" if fwd_only else "fwd+bwd"
    cfg_str = (f"{args.config}: {cfgd['P']} Gaussians, {cfgd['W']}x{cfgd['H']}, SH deg {cfgd['sh_degree']}, "
               f"feat_dim {cfgd['C']}, {mode}")
    metric = METRIC if args.config == "c3" else (
        f"views/sec {mode} @{cfgd['P']} Gaussians/{cfgd['W']}x{cfgd['H']}/feat_dim={cfgd['C']}")

    if args.impl == "reference" and not have_ref:
        # no reference build on this box: time the CPU port instead (rank 0 only)
        if rank == 0:
            sc = scenegen.make_config(args.config, views=1)
            cb = cpu_baseline(sc, cfg_str)
            print(json.dumps({"impl": "reference", "metric": metric, "value": cb["value"], "unit": "views/s",
                              "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                              "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True, "scaling": "weak",
                              "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                              "config": {"workload": cfg_str, "note": "oracle/_ref missing: CPU oracle port timed"},
                              "cpu_baseline": cb,
                              "e2e": {"value": cb["value"], "unit": "views/s", "h2d_bytes_per_step": 0,
                                      "d2h_bytes_per_step": 0}}))
        return

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if distributed:
        dist.init_process_group("nccl", device_id=dev)

    VPR = args.views_per_rank
    if strong:
        if args.batch_views % world:
            raise SystemExit("config c4 shards one view batch: WORLD_SIZE must divide --batch-views")
        VPR = args.batch_views // world
    n_views = VPR * world
    scene = scenegen.make_config(args.config, views=n_views)
    C, P = scene.C, scene.P
    W, H = scene.cameras[0].image_width, scene.cameras[0].image_height
    HW, tiles = W * H, ((W + 15) // 16) * ((H + 15) // 16)

    if args.impl == "ours":
        from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer, _C
        from diff_gaussian_rasterization.parallel import FlatGradBuffer, ViewBatch, shard_views
    else:
        # The reference arm must not map this repo's native libraries: the host-side helpers (flat gradient buffer, view
        # sharding -- pure torch) are loaded by FILE PATH so that the package __init__ (which imports _C) never runs.
        import importlib.util

        sys.path.insert(0, ROOT)
        from oracle import ref_wrapper as rw
        spec = importlib.util.spec_from_file_location(
            "f3dgs_parallel_helpers", os.path.join(ROOT, "feature-3dgs_b200", "diff_gaussian_rasterization", "parallel.py"))
        _par = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(_par)
        FlatGradBuffer, shard_views = _par.FlatGradBuffer, _par.shard_views
        _C = None

    t = scenegen.to_torch(scene, dev, requires_grad=True)
    params = [t[k] for k in ("means3D", "scales", "rotations", "opacities", "shs", "semantic_feature")]
    flat = FlatGradBuffer(params)
    my_views = shard_views(n_views, rank, world)
    bg = t["bg"]

    # per-view camera: device-resident copies (for `value`) and pinned host copies (for `e2e`)
    def cam_pack(cam):
        return np.concatenate([cam.viewmatrix.reshape(-1), cam.projmatrix.reshape(-1), cam.campos]).astype(np.float32)

    cams = [scene.cameras[v] for v in my_views]
    cam_host = [torch.from_numpy(cam_pack(c)).pin_memory() for c in cams]
    cam_dev = [h.to(dev) for h in cam_host]
    gc, gf, gd = [torch.from_numpy(g).to(dev) for g in scenegen.upstream_grads(H, W, C, seed=99)]

    def make_rasterizer(cam, packed):
        kw = dict(image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg, scale_modifier=1.0,
                  viewmatrix=packed[0:16].view(4, 4), projmatrix=packed[16:32].view(4, 4),
                  sh_degree=scene.sh_degree, campos=packed[32:35], prefiltered=False,
                  debug=bool(args.ref_debug and args.impl == "reference"))
        if args.impl == "ours":
            return GaussianRasterizer(GaussianRasterizationSettings(**kw))
        return rw.RefRasterizer(kw, C)

    def render(cam, packed):
        means2D = torch.zeros_like(t["means3D"], requires_grad=True)
        if dump:
            stats["means2D"] = means2D  # its .grad: the viewspace gradient a caller of the autograd API receives
        return make_rasterizer(cam, packed)(
            means3D=t["means3D"], means2D=means2D, opacities=t["opacities"], shs=t["shs"],
            semantic_feature=t["semantic_feature"] if C else None, scales=t["scales"], rotations=t["rotations"])

    # teacher feature map at the teacher's resolution (reference train.py:99: viewpoint_cam.semantic_feature), resident
    Hg, Wg = max(int(round(H / 2.25)), 1), max(int(round(W / 2.25)), 1)
    gt_feat = torch.rand(C, Hg, Wg, device=dev, generator=torch.Generator(dev).manual_seed(7)) if C else None

    stats = {}
    dump = OutputDump(len(cams), 5 * len(cams) + 8) if args.dump_outputs and rank == 0 else None
    use_batch = args.impl == "ours" and args.api == "batch" and not fwd_only
    if args.impl == "ours" and not fwd_only:
        vb = ViewBatch({k: t[k].detach() for k in ("means3D", "scales", "rotations", "opacities", "shs", "semantic_feature")})

        def settings_of(cam, packed):
            return GaussianRasterizationSettings(
                image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg, scale_modifier=1.0,
                viewmatrix=packed[0:16].view(4, 4), projmatrix=packed[16:32].view(4, 4), sh_degree=scene.sh_degree,
                campos=packed[32:35], prefiltered=False, debug=False)

        def step_device_batch():
            vb.zero_()
            for i, cam in enumerate(cams):
                color, feat, radii, depth, ctx = vb.forward(settings_of(cam, cam_dev[i]))
                if dump:
                    dump.keep(i, color=color, feature_map=feat, depth=depth, radii=radii)
                vb.backward(ctx, gc, gf if C else None, gd, last=(i == len(cams) - 1))
                stats["radii"] = radii
            vb.all_reduce()

        from diff_gaussian_rasterization import feature_head as fh

        def step_e2e_batch():
            # the reference's loss structure (train.py:96-104): a colour term on the rendered image through autograd
            # (small tensors) + the L1 feature loss against the teacher map after the bilinear resize -- the latter through
            # the fused feature head (csrc/feature_head.cu), which also returns dL/dfeature_map
            vb.zero_()
            total = torch.zeros((), device=dev)
            for i, cam in enumerate(cams):
                cam_stage[i].copy_(cam_host[i], non_blocking=True)  # H2D of this view's camera
                color, feat, radii, depth, ctx = vb.forward(settings_of(cam, cam_stage[i]))
                outs = [color.requires_grad_(), depth.requires_grad_()]
                loss = (outs[0] * gc).sum() + (outs[1] * gd).sum()
                loss.backward()  # the user's colour / depth loss: autograd only over two small maps
                gfeat = None
                if C:
                    lf, gfeat = fh.feature_l1_loss_and_grad(feat, gt_feat, 1.0)
                    loss = loss.detach() + lf
                vb.backward(ctx, color.grad, gfeat, depth.grad, last=(i == len(cams) - 1))
                total = total + loss.detach()
            vb.all_reduce()
            return float(total.item())  # D2H read of the step's result

    def step_device():
        if fwd_only:
            with torch.no_grad():
                for i, cam in enumerate(cams):
                    color, feat, radii, depth = render(cam, cam_dev[i])
                    if dump:
                        dump.keep(i, color=color, feature_map=feat, depth=depth, radii=radii)
                    stats["radii"] = radii
            return
        flat.zero_()
        for i, cam in enumerate(cams):
            color, feat, radii, depth = render(cam, cam_dev[i])
            if dump:
                dump.keep(i, color=color, feature_map=feat, depth=depth, radii=radii)
            outs, gos = [color, depth], [gc, gd]
            if C:
                outs.append(feat)
                gos.append(gf)
            torch.autograd.backward(outs, gos)
            if dump:
                dump.keep(i, grad_means2D=stats["means2D"].grad)
            stats["radii"] = radii
        flat.all_reduce()

    h2d_bytes = sum(h.numel() * 4 for h in cam_host)
    cam_stage = [torch.empty_like(d) for d in cam_dev]
    step_device_autograd = step_device

    def step_e2e():
        total = torch.zeros((), device=dev)
        if fwd_only:
            with torch.no_grad():
                for i, cam in enumerate(cams):
                    cam_stage[i].copy_(cam_host[i], non_blocking=True)
                    color, feat, radii, depth = render(cam, cam_stage[i])
                    total = total + (color * gc).sum() + (depth * gd).sum() + ((feat * gf).sum() if C else 0.0)
            return float(total.item())
        flat.zero_()
        for i, cam in enumerate(cams):
            cam_stage[i].copy_(cam_host[i], non_blocking=True)  # H2D of this view's camera
            color, feat, radii, depth = render(cam, cam_stage[i])
            loss = (color * gc).sum() + (depth * gd).sum()
            if C:  # the reference's feature loss, with the reference's own operators (train.py:100-104)
                fm = torch.nn.functional.interpolate(feat.unsqueeze(0), size=(Hg, Wg), mode="bilinear",
                                                     align_corners=True).squeeze(0)
                loss = loss + torch.abs(fm - gt_feat).mean()
            loss.backward()
            total = total + loss.detach()
        flat.all_reduce()
        return float(total.item())  # D2H read of the step's result

    def barrier():
        if distributed:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device=dev) if args.l2_flush else None

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        if flush_buf is None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            barrier()
            total_ms = e0.elapsed_time(e1)
        else:
            # one event pair per step; the L2 flush (a 512 MB fill, 4x the 126 MB L2) sits between the pairs
            pairs = []
            for _ in range(steps):
                flush_buf.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                pairs.append((a, b))
            barrier()
            total_ms = sum(a.elapsed_time(b) for a, b in pairs)
        ms = torch.tensor([total_ms], device=dev)
        if distributed:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)  # max over ranks
        return float(ms.item())

    # ---------------- timed region 1: device-resident `value`
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()  # nvidia-smi takes ~1 s to produce its first row: start before the warm-up
    main_step = step_device_batch if use_batch else step_device
    for _ in range(args.warmup):
        main_step()
    barrier()
    if _C is not None:
        _C.profile_read()
        _C.profile_enable(True)
        launches0 = _C.launch_count()
    ms_total = timed(main_step, args.steps, 0)
    if _C is not None:
        launches = _C.launch_count() - launches0
        _C.profile_enable(False)
        stage_ms, stage_cnt = _C.profile_read()
    views_per_step = n_views
    value = views_per_step * args.steps / (ms_total / 1000.0)
    if dump:
        if fwd_only:
            grads = {}
        elif use_batch:
            grads = {"grad_" + k: g for k, g in vb.grads.items()}
            grads.update(grad_accum=vb.grad_accum, denom=vb.denom)
        else:
            grads = {"grad_" + k: t[k].grad for k in ("means3D", "scales", "rotations", "opacities", "shs",
                                                      "semantic_feature") if t[k].grad is not None}
        dump.write(args.dump_outputs, grads)
        dump = None  # the later regions run the same step functions

    # ---------------- timed region 2: end to end
    ms_e2e = timed(step_e2e_batch if use_batch else step_e2e, args.steps, max(args.warmup, 3))
    e2e_value = views_per_step * args.steps / (ms_e2e / 1000.0)
    other_api = None
    if args.impl == "ours" and not fwd_only:
        # the other public API, same procedure, for the record
        o_dev, o_e2e = (step_device_autograd, step_e2e) if use_batch else (step_device_batch, step_e2e_batch)
        o_ms = timed(o_dev, args.steps, max(args.warmup, 3))
        o_ms_e2e = timed(o_e2e, args.steps, max(args.warmup, 3))
        other_api = {"api": "autograd" if use_batch else "batch",
                     "value": views_per_step * args.steps / (o_ms / 1000.0), "ms_per_step": o_ms / args.steps,
                     "e2e_value": views_per_step * args.steps / (o_ms_e2e / 1000.0), "e2e_ms_per_step": o_ms_e2e / args.steps}
    if sampler:
        clocks = sampler.stop()  # rows cover warm-up + both timed regions (the GPU is busy throughout)

    if rank != 0:
        if distributed:
            dist.destroy_process_group()
        return

    radii = stats["radii"]
    V = int((radii > 0).sum().item())
    out = {
        "metric": metric, "value": value, "unit": "views/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg_str, "views_per_rank_per_step": VPR, "views_per_step": views_per_step,
                   "parallelism": f"view-sharded dp{world}, 1 grad all-reduce/step" if distributed else "single GPU",
                   "l2": ("explicit flush: 512 MB fill between timed steps, outside the per-step event pairs" if args.l2_flush
                          else "inputs exceed the 126 MB L2 (per view: features P*C*4 B, upstream grads C*H*W*4 B); no explicit flush"),
                   "api": ("ViewBatch: _C.rasterize_gaussians forward + in-kernel gradient accumulation "
                           "(f3dgs_backward_accum) into one flat buffer, densification statistics folded in" if use_batch else
                           "GaussianRasterizer autograd API (forward" + ("" if fwd_only else " + torch.autograd.backward") + ")"),
                   "other_api": other_api,
                   "e2e_moves": "per view: 35 floats of camera state from pinned host memory (H2D); per step: the scalar loss "
                                "(D2H). Gaussian parameters, loss targets and rendered maps stay in HBM (model state and "
                                "dataset cache of a training loop, as in the reference train.py)",
                   "e2e_loss": ("colour/depth term sum(out * fixed weights) + the reference's feature loss (train.py:100-104): "
                                "L1 against a resident teacher map at 1/2.25 resolution after a bilinear resize "
                                "(align_corners=True). Autograd API / reference arm: PyTorch operators; batch API: the fused "
                                "feature head (csrc/feature_head.cu)")},
        "clocks": clocks,
        "dump_outputs": (None if not args.dump_outputs else
                         f"{args.dump_outputs}: the timed steps of `value` include the device-side copies of the dump"),
        "e2e": {"value": e2e_value, "unit": "views/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
    }
    if args.impl == "reference":
        out["impl"] = "reference"
        out["config"]["reference_kind"] = ("unmodified reference CUDA kernels + _C binding (oracle/_ref, sm_100a build), debug="
                                           + str(bool(args.ref_debug)) + "; its 60-line Python autograd shim is restated "
                                           "in oracle/ref_wrapper.py (the reference tree does not travel to the GPU box)")
        maps = open("/proc/self/maps").read()
        mine = sorted({ln.split("/")[-1] for ln in maps.splitlines()
                       if "libf3dgs_b200" in ln or "diff_gaussian_rasterization/_C" in ln})
        assert not mine, f"reference arm mapped this repo's native libraries: {mine}"
        out["config"]["native_libs_of_this_repo_mapped"] = mine
        out["gpu_launches"] = 0
    else:
        out["gpu_launches"] = int(launches)
        # roofline of the dominant kernel
        per_launch = {s: (stage_ms[i] / stage_cnt[i] if stage_cnt[i] else 0.0) for i, s in enumerate(STAGES)}
        # R of the last view: read from the profile? use the library's own count via a fresh forward
        with torch.no_grad():
            raw = _C.rasterize_gaussians(bg, t["means3D"], torch.Tensor([]), t["semantic_feature"] if C else torch.empty(0, device=dev),
                                         t["opacities"], t["scales"], t["rotations"], 1.0, torch.Tensor([]),
                                         cam_dev[-1][0:16].view(4, 4), cam_dev[-1][16:32].view(4, 4), cams[-1].tanfovx,
                                         cams[-1].tanfovy, H, W, t["shs"], scene.sh_degree, cam_dev[-1][32:35], False, False)
        R = int(raw[0])
        alg = algorithmic_bytes(V, R, tiles, HW, C)
        dom = "composite_fwd" if fwd_only else max(("composite_fwd", "composite_bwd"), key=lambda k: per_launch[k])
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = alg[dom] / (per_launch[dom] * 1e-3) / 1e9 if per_launch[dom] > 0 else 0.0
        traffic = None  # the ncu --set full capture under profiles/ was taken at config 3: null for the other configs
        try:
            if args.config == "c3":
                traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dom)
        except Exception:
            pass
        out["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                           "frac": achieved / peak, "traffic": traffic,
                           "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                           "algorithmic_bytes_per_launch": alg[dom], "launch_ms": per_launch[dom],
                           "V": V, "R": R, "stage_ms_per_launch": per_launch,
                           "other": {k: {"achieved": alg[k] / (per_launch[k] * 1e-3) / 1e9 if per_launch[k] else 0.0,
                                         "algorithmic_bytes_per_launch": alg[k], "launch_ms": per_launch[k]}
                                     for k in alg if k != dom}}
    if world == 1 and not args.no_cpu_baseline:
        try:
            out["cpu_baseline"] = cpu_baseline(scenegen.make_config(args.config, views=1), cfg_str)
        except Exception as ex:  # the checker must never take the bench down
            out["cpu_baseline"] = {"value": None, "unit": "views/s", "cores": os.cpu_count(), "kind": "port",
                                   "sample": f"failed: {ex}"}
        if args.impl == "reference":
            out["cpu_baseline"]["note"] = "reference arm = reference CUDA kernels; CPU port listed for context"
    print(json.dumps(out))
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
