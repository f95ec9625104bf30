#!/usr/bin/env python
"""bench.py -- Mrays/s fwd+bwd of the NeuS volume-rendering hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference algorithm's CPU implementation (oracle port) on the host cores

Workload (config.workload = "cfg2"): BASELINE.json configs[1], "neus_in_10_minutes BMVS-style object (LoTD + fused MLP),
800x600, 1 B200": a CFG-sized LoTDNeuS (16-level LoTD, 12.13 M params, 32->64->1 SDF decoder, 58->64->64->3 radiance net,
64^3 occupancy grid), synthetic sphere-like SDF, one full 800x600 frame (480 000 rays) per step, rendered in ray chunks.
A step = ray_test -> march -> 3-stage up-sampling -> boundary SDF (grad) -> alpha -> compression -> colour/normal query
-> compositing -> scalar loss over rgb/depth/normals/mask -> backward to every parameter (-> one NCCL all-reduce of the
flat gradient when N > 1).  Weak scaling: every rank renders its own full frame (its own camera pose).

Timing: CUDA events on the current stream, barrier + synchronize on both sides, max over ranks; L2 is flushed between
steps (256 MiB write, outside the per-step event pairs); clocks are sampled with nvidia-smi during the timed region.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W = 600, 800
N_VIEWS = 8


# ---------------------------------------------------------------------------------------------- synthetic scene (cfg 2)
def pinhole_rays(Hh, Ww, cam_pos, focal=None):
    focal = (Hh + Ww) / 2. if focal is None else focal
    cam = np.asarray(cam_pos, dtype=np.float64)
    fwd = -cam / np.linalg.norm(cam)
    right = np.cross(fwd, np.array([0., 0., 1.])); right /= np.linalg.norm(right)
    down = np.cross(fwd, right)
    j, i = np.meshgrid(np.arange(Hh, dtype=np.float64), np.arange(Ww, dtype=np.float64), indexing="ij")
    d = ((i + 0.5 - Ww / 2.) / focal)[..., None] * right + ((j + 0.5 - Hh / 2.) / focal)[..., None] * down + fwd
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    o = np.broadcast_to(cam, d.shape)
    return (torch.from_numpy(np.ascontiguousarray(o.reshape(-1, 3), dtype=np.float32)),
            torch.from_numpy(np.ascontiguousarray(d.reshape(-1, 3), dtype=np.float32)))


def orbit(k, n, radius=3.0, elev_deg=20.0):
    a, e = 2 * math.pi * k / n, math.radians(elev_deg)
    return (radius * math.cos(e) * math.cos(a), radius * math.cos(e) * math.sin(a), radius * math.sin(e))


def build_model(device, seed=42, radius=0.5, noise=2.0e-3, ln_inv_s_init=0.5298, k_pass=8.0, collect_samples=False):
    """CFG-sized model whose SDF is a noisy sphere (the state `pretrain_sdf_sphere` would reach; see oracle/scene.py for
    the same construction on the oracle side).  inv_s = exp(10 * 0.5298) ~ 200."""
    from neuralsim_b200.fields import LoTDNeuSModel
    gen = torch.Generator(device=device).manual_seed(seed)
    model = LoTDNeuSModel(
        surface_cfg=dict(bounding_size=2.0, encoding_cfg=dict(lotd_auto_compute_cfg=dict(type="gen_ngp", min_res=16, n_feats=2, log2_hashmap_size=19,
                                                                                         per_level_scale=1.382, num_levels=16),
                                                              param_init_cfg=dict(type="uniform_to_type", bound=noise))),
        radiance_cfg=dict(n_appear_embedding=4, dir_embed_cfg=dict(type="spherical", degree=4), D=2, W=64),
        var_ctrl_cfg=dict(ln_inv_s_init=ln_inv_s_init, ln_inv_s_factor=10.0),
        accel_cfg=dict(resolution=[64, 64, 64], occ_val_fn_cfg=dict(type="sdf", inv_s=256.0), occ_thre=0.3, ema_decay=0.95,
                       update_from_samples_cfg=dict() if collect_samples else None),
        ray_query_cfg=dict(query_mode="march_occ_multi_upsample_compressed", query_param=dict(
            nablas_has_grad=True, num_coarse=64, num_fine=[8, 8, 32], coarse_step_cfg=dict(step_mode="linear"),
            march_cfg=dict(step_size=0.005, max_steps=4096), upsample_inv_s=64.0, upsample_inv_s_factors=[1, 4, 16],
            upsample_use_estimate_alpha=True)),
        device=device, generator=gen)
    enc = model.implicit_surface.encoding
    meta = enc.meta
    lvl = 5
    res = meta.level_res_multidim[lvl]
    ax = [((torch.arange(r, dtype=torch.float64) - 0.5) / (r - 2) * 2 - 1) for r in res]
    gx, gy, gz = torch.meshgrid(*ax, indexing="ij")
    s = (torch.sqrt(gx * gx + gy * gy + gz * gz) - radius).float().to(device)
    with torch.no_grad():
        off, nf = meta.level_offsets[lvl], meta.level_n_feats[lvl]
        enc.flattened_params[off:off + meta.level_n_params[lvl]].view(*res, nf)[..., 0] = s
        f_idx = sum(meta.level_n_feats[:lvl])
        d0, d1 = model.implicit_surface.decoder.layers
        d0.weight[:, f_idx] = 0.
        d1.weight.mul_(0.05); d1.bias.zero_()
        d0.weight[0].zero_(); d0.weight[1].zero_()
        d0.weight[0, f_idx], d0.weight[1, f_idx] = k_pass, -k_pass
        d0.bias[0], d0.bias[1] = 0., 0.
        d1.weight[0, 0], d1.weight[0, 1] = 1. / k_pass, -1. / k_pass
        c = (torch.arange(64, dtype=torch.float64) + 0.5) / 64 * 2 - 1
        cx, cy, cz = torch.meshgrid(c, c, c, indexing="ij")
        occ = ((torch.sqrt(cx * cx + cy * cy + cz * cz) - radius).abs() < 0.012 + math.sqrt(3.) / 64)
        model.accel.occ.set_occ_grid(occ.to(device))
    return model


def strong_shard(o, d, rank, world, total_rays, rays_per_rank, seed=None):
    """The rays of ONE frame dealt to `world` ranks (strong scaling).  Image-ordered rays: row r of the frame -> rank r mod world (the ranks share
    the object's rows; rays stay image-ordered inside a row); random pixels (`seed`): ray j of the draw -> rank j mod world.  Every ray goes to
    exactly one rank."""
    if seed is not None:
        sel = torch.randperm(o.shape[0], generator=torch.Generator().manual_seed(seed))[:total_rays]
        o, d = o[sel][rank::world], d[sel][rank::world]
    elif total_rays == H * W and H % world == 0:
        o, d = o.view(H, W, 3)[rank::world].reshape(-1, 3), d.view(H, W, 3)[rank::world].reshape(-1, 3)
    else:
        o, d = o[:total_rays][rank * rays_per_rank:(rank + 1) * rays_per_rank], d[:total_rays][rank * rays_per_rank:(rank + 1) * rays_per_rank]
    return o.contiguous(), d.contiguous()


def flat_grad_views(model):
    """One flat fp32 buffer holding every gradient (p.grad are views) -> a single all-reduce per step."""
    params = [p for p in model.parameters() if p.requires_grad]
    flat = torch.zeros(sum(p.numel() for p in params), device=params[0].device)
    o = 0
    for p in params:
        p.grad = flat[o:o + p.numel()].view_as(p)
        o += p.numel()
    return flat, params


def loss_of(rendered):
    return rendered["rgb_volume"].mean() + rendered["depth_volume"].mean() + rendered["normals_volume"].mean() + rendered["mask_volume"].mean()


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons during the timed region.

    Measured on this pool (profiles/diag_clock_sampler.sh, /tmp logs of round 1): ANY concurrent poller -- a looping `nvidia-smi -lms 100..1000`,
    a thread forking nvidia-smi, an NVML thread -- makes 7 of 8 runs of this launch- and sync-heavy step show 80-230 ms stalls inside 15 ms steps
    (NVML queries disturb CUDA submission for ~100 ms; even a query made between two steps shows up in the next ones, profiles/diag_*.sh); with no
    poller -- and no NVML session inside this process -- steps are 14.2-15.8 ms.  So ONE sample is taken, by a separate one-shot `nvidia-smi`
    process, at the one moment it cannot perturb the measurement and is still "during" it: right after the LAST step of the resident loop has been
    enqueued -- the GPU is then executing the timed steps and nothing of ours is left to launch."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0, period_ms=100):
        self.index, self.enabled = index, period_ms > 0
        self.samples, self.reasons, self.max_mhz, self.how = [], set(), None, None
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        self.phys = vis.split(",")[index].strip() if vis and len(vis.split(",")) > index else str(index)

    def __enter__(self):
        return self

    def __exit__(self, *a):
        pass

    def sample(self):
        """ONE `nvidia-smi` query (a separate process; nothing NVML-related ever lives in this one), called by the timing loop once the
        last resident step has been enqueued: the GPU is executing the timed steps, and nothing of ours is left to launch."""
        if not self.enabled:
            return
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", self.phys], capture_output=True, text=True,
                                 timeout=10).stdout.strip().split(",")
            self.samples.append(float(out[0])); self.max_mhz = float(out[1])
            self.how = "one nvidia-smi query while the GPU executes the enqueued timed steps (after the last launch of the resident loop)"
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:6]):
                if "Active" in v and "Not" not in v:
                    self.reasons.add(name)
        except Exception:
            pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no sampler"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples),
                "how": self.how}


def effective_cpus():
    """host cores this container may actually use: min(visible cores, cgroup CPU-bandwidth quota) -- the GPU boxes of this pool show 128
    cores under a 16-CPU quota; 128 busy threads there are throttled for most of every 100 ms period."""
    n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# ---------------------------------------------------------------------------------------------- CPU baseline / reference arm
def cpu_baseline(sample_rays=1536, threads=None):
    """The reference algorithm's CPU implementation (oracle port of nr3d_lib's path) on a bounded sample of the same workload:
    `sample_rays` rays of the 800x600 frame (strided over the image), fwd+bwd.  Runs on the host cores."""
    from oracle import render as orender, scene as oscene
    threads = threads or effective_cpus()
    torch.set_num_threads(threads)
    P = oscene.make_sphere_params()
    occ = oscene.make_occ_grid()
    ro, rd = oscene.pinhole_rays(H, W, oscene.orbit_camera(0, N_VIEWS))
    sel = torch.linspace(0, ro.shape[0] - 1, sample_rays).long()
    ro, rd = ro[sel].contiguous(), rd[sel].contiguous()
    P.requires_grad_(True)
    t0 = time.perf_counter()
    rt = orender.ray_test(ro, rd, near=0.01)
    vb, _ = orender.neus_ray_query(P, occ, rt, rays_h_appear=torch.zeros(rt["num_rays"], P.n_appear))
    out = orender.volume_integration(vb, ro.shape[0])
    (out["rgb_volume"].mean() + out["depth_volume"].mean() + out["normals_volume"].mean() + out["mask_volume"].mean()).backward()
    dt = time.perf_counter() - t0
    return dict(value=sample_rays / dt / 1e6, unit="Mrays/s", cores=threads, kind="port",
                sample=f"{sample_rays} rays strided over the 800x600 frame of view 0, fwd+bwd, {dt:.1f} s wall "
                       f"(the numpy LoTD port walks its 16 levels on a thread pool, the torch MLP part uses {threads} threads)")


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    rays = args.ref_rays
    times = []
    for i in range(warm + steps):
        r = cpu_baseline(rays)
        if i >= warm:
            times.append(rays / r["value"] / 1e6)
    ms = 1e3 * float(np.mean(times))
    val = rays / (ms / 1e3) / 1e6
    base = dict(value=val, unit="Mrays/s", cores=effective_cpus(), kind="port",
                sample=f"{rays} rays of the 800x600 frame per step (bounded sample), fwd+bwd, oracle port of the reference path")
    print(json.dumps({
        "impl": "reference", "metric": "Mrays/sec fwd+bwd", "value": val, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": "cfg2", "frame": "800x600", "rays_per_step": rays, "note": "CPU, bounded sample"},
        "cpu_baseline": base, "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


def use_reference_cuda_kernels():
    """BASELINE.md B1: route the SAME host orchestration through the REFERENCE'S OWN CUDA kernels (oracle/_ref: `_lotd`,
    `_pack_ops`, `_occ_grid`, `_shencoder` compiled from /root/reference) and switch every fused path off, i.e. the op
    sequence nr3d_lib executes (16-level gather kernels, autocast cuBLAS MLPs, one-thread-per-pack pack_ops, fp16 atomics).
    Only used by `--impl reference-cuda` and the `reference_cuda` field; never by the product path."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_ref
    mods = {n: build_ref.load(n) for n in ("_lotd", "_pack_ops", "_occ_grid", "_shencoder")}
    if any(m is None for m in mods.values()):
        return False
    import neuralsim_b200.fields.encoding as E
    import neuralsim_b200.fields.networks as NW
    import neuralsim_b200.graphics.pack_ops as GP
    import neuralsim_b200.graphics.raymarch as GR
    import neuralsim_b200.fields.space as SP
    import neuralsim_b200.graphics.neus as GN
    E._backend, GP._backend, GR._backend, NW._shencoder = mods["_lotd"], mods["_pack_ops"], mods["_occ_grid"], mods["_shencoder"]
    NW.LoTDSDF._fusable = lambda self: False       # no fused SDF / colour kernels
    GN.FUSED_STAGES = False                        # the op-by-op chain of neus_ray_query.py / single_volume_renderer.py, every op a reference kernel or ATen
    SP.FUSED_RAY_TEST = False                      # the torch chain of aabb.py
    return True


# ---------------------------------------------------------------------------------------------- cfg3 arm
def run_cfg3(args, rank, world, local, device):
    """BASELINE.json configs[2] (bench_cfg3.py): per step 8192 camera rays (rgb + normals) and 8192 LiDAR rays (depth + normals) through the
    street-segment model, fwd + bwd; each ray kind is one CUDA-graph launch (graph mode) or the host-sized path (host mode)."""
    import torch.distributed as dist
    import bench_cfg3 as C
    from neuralsim_b200 import _lib
    from neuralsim_b200.renderer import SingleVolumeRenderer
    from neuralsim_b200.graphics.neus_static import StaticFrame
    mode = "host" if args.impl == "reference-cuda" else args.mode
    if args.impl == "reference-cuda" and not use_reference_cuda_kernels():
        raise SystemExit("bench.py: oracle/_ref is not built")
    model = C.build_model(device).train()
    flat, params = flat_grad_views(model)
    views_dev, views_host = [], []
    for k in range(N_VIEWS):
        (co, cd), (lo, ld) = C.make_views(k, rank, world)
        views_host.append(tuple(t.pin_memory() for t in (co, cd, lo, ld)))
        views_dev.append(tuple(t.to(device) for t in (co, cd, lo, ld)))
    n_rays = C.N_CAM + C.N_LIDAR
    ha = torch.zeros(C.N_CAM, 4, device=device)
    r_cam = SingleVolumeRenderer(dict(near=C.NEAR, far=C.FAR)).train()
    r_lidar = SingleVolumeRenderer(dict(near=C.NEAR, far=C.FAR, with_rgb=False, with_normal=True)).train()
    f_cam = f_lidar = None
    launches_per_step = None
    if mode != "host":
        f_cam = StaticFrame(model, C.N_CAM, loss_fn=C.loss_cam, near=C.NEAR, far=C.FAR, use_graph=(mode == "graph"), pre_hook=flat.zero_, slack=2.0)
        f_lidar = StaticFrame(model, C.N_LIDAR, loss_fn=C.loss_lidar, near=C.NEAR, far=C.FAR, with_rgb=False, use_graph=(mode == "graph"), slack=2.0)
        for k in range(N_VIEWS):
            f_cam.rays_o.copy_(views_dev[k][0]); f_cam.rays_d.copy_(views_dev[k][1]); f_cam._size()
            f_lidar.rays_o.copy_(views_dev[k][2]); f_lidar.rays_d.copy_(views_dev[k][3]); f_lidar._size()
        l0 = _lib.launch_count()
        f_cam.capture(); f_lidar.capture()
        launches_per_step = (_lib.launch_count() - l0) // (3 if mode == "graph" else 1) if mode == "graph" else None      # 2 warm-up runs + the captured one
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)
    loss_host = torch.zeros((), pin_memory=True)
    out_host = {"rgb": torch.zeros(C.N_CAM, 3).pin_memory(), "depth_cam": torch.zeros(C.N_CAM).pin_memory(), "depth_lidar": torch.zeros(C.N_LIDAR).pin_memory()}
    last = {}

    def step(v):
        co, cd, lo, ld = v
        if f_cam is not None:
            l1 = f_cam.step(co, cd, None)
            l2 = f_lidar.step(lo, ld, None)
            last["cam"], last["lidar"] = f_cam.rendered, f_lidar.rendered
            loss = l1 + l2
        else:
            flat.zero_()
            co, cd, lo, ld = (t.to(device, non_blocking=True) for t in v)
            a = r_cam.render(model, co, cd, rays_h_appear=ha)["rendered"]
            b = r_lidar.render(model, lo, ld)["rendered"]
            loss = C.loss_cam(a) + C.loss_lidar(b)
            if loss.requires_grad:
                loss.backward()
            last["cam"], last["lidar"] = a, b
            loss = loss.detach()
        if world > 1:
            dist.all_reduce(flat)
        return loss

    def timed(fn, k, sampler=None):
        evs = []
        for i in range(k):
            flush_buf.fill_(i & 0xff)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(i); b.record()
            evs.append((a, b))
        if sampler is not None:
            sampler.sample()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    n_views = max(1, min(N_VIEWS, args.warmup))

    def resident(i):
        return step(views_dev[i % n_views])

    def e2e(i):
        loss = step(views_host[i % n_views])
        out_host["rgb"].copy_(last["cam"]["rgb_volume"], non_blocking=True)
        out_host["depth_cam"].copy_(last["cam"]["depth_volume"], non_blocking=True)
        out_host["depth_lidar"].copy_(last["lidar"]["depth_volume"], non_blocking=True)
        loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    with ClockSampler(local, args.clock_period_ms) as clocks:
        for i in range(args.warmup):
            resident(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_e2e = timed(e2e, args.steps)
        if world > 1:
            dist.barrier()
        t_res = timed(resident, args.steps, clocks)
    st_res, st_e2e = stats_of(t_res), stats_of(t_e2e)
    ms = torch.tensor([st_res["mean"], st_e2e["mean"], st_res["median"], st_e2e["median"]], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if rank != 0:
            dist.destroy_process_group()
            return
    ms_res, ms_e2e, med_res, med_e2e = (float(x) for x in ms)
    tot = world * n_rays
    meta = model.implicit_surface.encoding.meta
    counts = {"cam": f_cam.counts(), "lidar": f_lidar.counts()} if f_cam is not None else None
    line = {"metric": "Mrays/sec fwd+bwd", "value": tot / (ms_res * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_res, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "median": {"ms_per_step": med_res, "value": tot / (med_res * 1e-3) / 1e6, "e2e_ms_per_step": med_e2e, "e2e_value": tot / (med_e2e * 1e-3) / 1e6},
            "config": {"workload": "cfg3", "what": "StreetSurf close-range model: cuboid aabb 40x150x15 m, cuboid LoTD (ngp auto config, 2^20 hash, max_num_levels 16 -- "
                       "the shipped config's 17 levels run op by op), 1 m occupancy voxels, step 0.2, 128 coarse + [8,8,32] fine; 8192 camera rays (rgb+normals) + "
                       "8192 LiDAR rays (with_rgb=False) per step", "lotd_levels": meta.n_levels, "lotd_params": int(meta.n_params),
                       "lotd_res": [list(r) for r in meta.level_res_multidim], "occ_grid": list(model.accel.occ.occ_grid.shape), "mode": mode,
                       "rays_per_step_per_gpu": n_rays, "parallelism": f"dp{world}", "l2": "256 MiB L2 flush between steps", "counts": counts},
            "e2e": {"value": tot / (ms_e2e * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(2 * n_rays * 3 * 4),
                    "d2h_bytes_per_step": int(sum(v.numel() * 4 for v in out_host.values()) + 4)},
            "gpu_launches": (int(launches_per_step * args.steps) if launches_per_step else None), "launches_per_step": launches_per_step,
            "host_launches_per_step": (2 if mode == "graph" else None), "clocks": clocks.summary(),
            "step_ms": {"resident": [round(x, 3) for x in t_res], "e2e": [round(x, 3) for x in t_e2e]}}
    if args.impl == "reference-cuda":
        line["impl"] = "reference-cuda"
    elif world == 1 and not args.no_ref_cuda:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-cuda", "--workload", "cfg3", "--steps", "10", "--warmup", "3"],
                               capture_output=True, text=True, timeout=900)
            rl = json.loads(r.stdout.strip().splitlines()[-1])
            line["reference_cuda"] = {"value": rl["value"], "ms_per_step": rl["ms_per_step"], "e2e": rl["e2e"]["value"], "steps": rl["steps"]}
            line["vs_reference_cuda"] = {"value_ratio": line["value"] / rl["value"], "e2e_ratio": line["e2e"]["value"] / rl["e2e"]["value"]}
        except Exception as ex:
            line["reference_cuda"] = {"unavailable": repr(ex)[:300]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------- cfg4 arm
def run_cfg4(args, rank, world, local, device):
    """BASELINE.json configs[3], the part of it that is built: N single-object NeuS models in one scene (8 instances of the cfg-2 object at
    different poses / scales in front of one camera), every object queried in its own frame (fused host-sized path), the buffers collected, sorted per
    ray and integrated jointly (neuralsim_b200/compose.py; reference app/renderers/buffer_compose_renderer.py:644-714), fwd + bwd.  The shared
    conditional (permutohedral) foreground models of code_multi are not built (DESIGN.md §8)."""
    import torch.distributed as dist
    from neuralsim_b200 import _lib
    from neuralsim_b200.compose import BufferComposeRenderer, ObjectPose
    if args.impl == "reference-cuda" and not use_reference_cuda_kernels():
        raise SystemExit("bench.py: oracle/_ref is not built")
    model = build_model(device).train()
    flat, params = flat_grad_views(model)
    rng = np.random.default_rng(0)
    n_obj = 8
    poses = []
    for i in range(n_obj):
        ang = 2 * math.pi * i / n_obj
        a = rng.uniform(0, 2 * math.pi)
        R = np.array([[math.cos(a), -math.sin(a), 0.], [math.sin(a), math.cos(a), 0.], [0., 0., 1.]])
        poses.append(ObjectPose(rotation=R, translation=[2.6 * math.cos(ang), 2.6 * math.sin(ang), 0.4 * math.sin(3 * ang)], scale=0.7 + 0.05 * i, device=device))
    objects = [(model, p) for p in poses]
    renderer = BufferComposeRenderer(dict(near=0.01)).train()
    views = []
    for k in range(N_VIEWS):
        a = 2 * math.pi * (k * world + rank) / (N_VIEWS * world)
        o, d = pinhole_rays(H, W, (9.0 * math.cos(a), 9.0 * math.sin(a), 3.0))
        views.append((o.to(device), d.to(device), o.pin_memory(), d.pin_memory()))
    n_rays = H * W
    ha = torch.zeros(n_rays, 4, device=device)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)
    loss_host = torch.zeros((), pin_memory=True)
    img_host = torch.zeros(n_rays, 3).pin_memory()

    def step(o, d):
        flat.zero_()
        out = renderer.render(objects, o, d, ha)["rendered"]
        loss = loss_of(out)
        if loss.requires_grad:
            loss.backward()
        if world > 1:
            dist.all_reduce(flat)
        return loss.detach(), out

    def timed(fn, k):
        ts = []
        for i in range(k):
            flush_buf.fill_(i & 0xff)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(i); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return ts

    def resident(i):
        v = views[i % N_VIEWS]
        step(v[0], v[1])

    def e2e(i):
        v = views[i % N_VIEWS]
        loss, out = step(v[2].to(device, non_blocking=True), v[3].to(device, non_blocking=True))
        img_host.copy_(out["rgb_volume"], non_blocking=True)
        loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for i in range(args.warmup):
        resident(i)
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    t_e2e = timed(e2e, args.steps)
    t_res = timed(resident, args.steps)
    launches = (_lib.launch_count() - l0) // (2 * args.steps)
    st_res, st_e2e = stats_of(t_res), stats_of(t_e2e)
    ms = torch.tensor([st_res["mean"], st_e2e["mean"], st_res["median"]], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if rank != 0:
            dist.destroy_process_group()
            return
    tot = world * n_rays
    line = {"metric": "Mrays/sec fwd+bwd", "value": tot / (float(ms[0]) * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": float(ms[0]), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "median": {"ms_per_step": float(ms[2]), "value": tot / (float(ms[2]) * 1e-3) / 1e6},
            "config": {"workload": "cfg4", "what": f"{n_obj} single-object NeuS models (the cfg-2 object at {n_obj} poses / scales) composed along the rays of one 800x600 "
                       "frame: per-object fused query (host-sized path) -> collect -> per-ray sort -> joint integration; no shared conditional models",
                       "rays_per_step_per_gpu": n_rays, "parallelism": f"dp{world}", "mode": "host"},
            "e2e": {"value": tot / (float(ms[1]) * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": float(ms[1]), "h2d_bytes_per_step": int(2 * n_rays * 12),
                    "d2h_bytes_per_step": int(n_rays * 12 + 4)},
            "gpu_launches": int(launches * args.steps), "launches_per_step": int(launches),
            "step_ms": {"resident": [round(x, 3) for x in t_res], "e2e": [round(x, 3) for x in t_e2e]}}
    if args.impl == "reference-cuda":
        line["impl"] = "reference-cuda"
    elif world == 1 and not args.no_ref_cuda:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-cuda", "--workload", "cfg4", "--steps", "5", "--warmup", "2"],
                               capture_output=True, text=True, timeout=900)
            rl = json.loads(r.stdout.strip().splitlines()[-1])
            line["reference_cuda"] = {"value": rl["value"], "ms_per_step": rl["ms_per_step"], "steps": rl["steps"]}
            line["vs_reference_cuda"] = {"value_ratio": line["value"] / rl["value"]}
        except Exception as ex:
            line["reference_cuda"] = {"unavailable": repr(ex)[:300]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------- main arm
def stats_of(ts):
    a = np.asarray(ts, dtype=np.float64)
    return dict(mean=float(a.mean()), median=float(np.median(a)), min=float(a.min()), max=float(a.max()))


DUMP_SAMPLE = 1 << 20


def step_outputs(model, rendered, loss):
    """what a caller of the step receives, as float32 host arrays: the rendered buffers, the loss and every parameter's gradient (a fixed
    seeded sample of DUMP_SAMPLE entries of a larger one, so that the whole dump stays far below 64 MB)"""
    out = {f"rendered.{k}": v for k, v in rendered.items() if torch.is_tensor(v) and v.is_floating_point()}
    out["loss"] = loss
    for name, p in model.named_parameters():
        if p.requires_grad and p.grad is not None:
            g = p.grad.reshape(-1)
            if g.numel() > DUMP_SAMPLE:
                idx = np.sort(np.random.default_rng(0).choice(g.numel(), DUMP_SAMPLE, replace=False))
                g = g[torch.from_numpy(idx).to(g.device)]
            out[f"grad.{name}"] = g
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--mode", default="graph", choices=["graph", "static", "host"],
                    help="graph: the whole fwd+bwd step is ONE CUDA-graph launch (sizes stay on the device; default).  static: the same step launched "
                         "kernel by kernel.  host: the host-sized path (three host reads per step; round-1 behaviour)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: every rank renders its own 800x600 frame; strong: the ranks share ONE frame (480000 / N rays each)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4"])
    ap.add_argument("--rayschunk", type=int, default=0, help="host mode only: rays per render call (0 = the whole batch in one call)")
    ap.add_argument("--rays", type=int, default=H * W, help="rays per step and GPU (default: the full 800x600 frame)")
    ap.add_argument("--random-rays", action="store_true", help="draw the --rays rays of every pose as random pixels (a training batch) instead of the first rows")
    ap.add_argument("--collect-samples", action="store_true", help="accel.update_from_samples_cfg = {} as in the shipped training config: every "
                    "training-time SDF query also feeds the occupancy grid's evidence buffer (in-kernel here, torch_scatter in the reference)")
    ap.add_argument("--clock-period-ms", type=int, default=100, help="0 = no clock sampler (diagnostics)")
    ap.add_argument("--ref-rays", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--dump-render", default=None, help="(internal) save the rendered buffers of view 0 to this file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="cfg2 only: after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32): the rendered "
                         "buffers, the loss and the gradient of every parameter (of a parameter with more than 2^20 entries, a fixed seeded "
                         "sample of 2^20 of them, in increasing index order)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl == "reference" or args.workload != "cfg2"):
        ap.error("--dump-outputs is implemented for the cfg2 workload of the GPU arms")

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    torch.set_num_threads(max(1, min(8, effective_cpus())))      # host side of the GPU arm is one launching thread; keep the intra-op pool small
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    from neuralsim_b200 import _lib
    from neuralsim_b200.renderer import SingleVolumeRenderer
    from neuralsim_b200.graphics.neus_static import StaticFrame
    mode = args.mode
    if args.impl == "reference-cuda":
        if not use_reference_cuda_kernels():
            raise SystemExit("bench.py: oracle/_ref is not built (python oracle/build_ref.py in the build container)")
        mode = "host"
    if args.workload == "cfg3":
        run_cfg3(args, rank, world, local, device)
        return
    if args.workload == "cfg4":
        run_cfg4(args, rank, world, local, device)
        return
    model = build_model(device, collect_samples=args.collect_samples).train()
    near = 0.01
    renderer = SingleVolumeRenderer(dict(near=near, rayschunk=0)).train()
    flat, params = flat_grad_views(model)
    n_rays = args.rays
    if args.scaling == "strong":
        n_rays = (args.rays + world - 1) // world
    views_host, views_dev = [], []
    for k in range(N_VIEWS):
        if args.scaling == "strong":           # ONE frame per step, its rows dealt to the ranks round-robin (row r -> rank r mod N): contiguous
            # blocks would give the ranks that own the object's rows most of the work (measured: 38 % efficiency at N = 8, profiles/r02s_*)
            o, d = pinhole_rays(H, W, orbit(k, N_VIEWS))
            o, d = strong_shard(o, d, rank, world, args.rays, n_rays, seed=(1000 + k) if args.random_rays else None)
            if o.shape[0] < n_rays:                # the last rank's block is padded with its own last ray
                pad = n_rays - o.shape[0]
                o, d = torch.cat([o, o[-1:].expand(pad, 3)]).contiguous(), torch.cat([d, d[-1:].expand(pad, 3)]).contiguous()
        else:
            o, d = pinhole_rays(H, W, orbit((k * world + rank) % (N_VIEWS * world), N_VIEWS * world))
            if args.random_rays:
                sel = torch.randperm(o.shape[0], generator=torch.Generator().manual_seed(1000 + k))[:n_rays]
                o, d = o[sel].contiguous(), d[sel].contiguous()
            else:
                o, d = o[:n_rays].contiguous(), d[:n_rays].contiguous()
        views_host.append((o.pin_memory(), d.pin_memory()))
        views_dev.append((o.to(device), d.to(device)))
    n_appear = 4
    h_appear = torch.zeros(n_rays, n_appear, device=device)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)
    chunk = args.rayschunk if args.rayschunk > 0 else n_rays
    keys = ("rgb_volume", "depth_volume", "normals_volume", "mask_volume")
    out_host = {"rgb_volume": torch.zeros(n_rays, 3).pin_memory(), "depth_volume": torch.zeros(n_rays).pin_memory(),
                "normals_volume": torch.zeros(n_rays, 3).pin_memory(), "mask_volume": torch.zeros(n_rays).pin_memory()}
    loss_host = torch.zeros((), pin_memory=True)
    d2h_bytes = int(sum(v.numel() * 4 for v in out_host.values()) + 4)

    # ------------------------------------------------------------------ the step
    frame = None
    if mode in ("graph", "static"):
        # flat.zero_() is part of the step (and of the graph); every size stays on the device; ONE launch per step in graph mode
        frame = StaticFrame(model, n_rays, loss_fn=loss_of, near=near, use_graph=(mode == "graph"), pre_hook=flat.zero_)
        frame.rays_o.copy_(views_dev[0][0]); frame.rays_d.copy_(views_dev[0][1])
        frame._size()                               # arenas from view 0 ...
        for k in range(1, N_VIEWS):                 # ... grown to the largest of the poses this run renders
            frame.rays_o.copy_(views_dev[k][0]); frame.rays_d.copy_(views_dev[k][1])
            frame._size()
        frame.capture()

    last = {}

    def step(o, d):
        """fwd+bwd of one batch of rays; gradients land in the flat buffer.  -> (loss, rendered)"""
        if frame is not None:
            loss = frame.step(o, d, None)
            rendered = frame.rendered
        else:
            flat.zero_()
            total = torch.zeros((), device=device)
            rendered = None
            for s0 in range(0, n_rays, chunk):
                e = min(s0 + chunk, n_rays)
                rendered = renderer.render(model, o[s0:e], d[s0:e], rays_h_appear=h_appear[:e - s0])["rendered"]
                loss = loss_of(rendered) * ((e - s0) / n_rays)
                if loss.requires_grad:             # a chunk whose rays all miss the object renders constants
                    loss.backward()
                total += loss.detach()
            loss = total
        if world > 1:
            dist.all_reduce(flat)                # the one collective of a step: sum of the flat gradient
        last["rendered"], last["loss"] = rendered, loss
        return loss

    def timed(fn, k, sampler=None):
        evs = []
        for i in range(k):
            flush_buf.fill_(i & 0xff)         # L2 flush, outside the event pair
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(i); b.record()
            evs.append((a, b))
        if sampler is not None:              # every step is enqueued and the GPU is still executing them: sample now, then drain
            sampler.sample()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    n_views = max(1, min(N_VIEWS, args.warmup))

    def resident(i):
        o, d = views_dev[i % n_views]
        return step(o, d)

    def e2e(i):
        oh, dh = views_host[i % n_views]
        if frame is not None:
            loss = step(oh, dh)                                                       # H2D of the step's rays straight into the graph's inputs
        else:
            loss = step(oh.to(device, non_blocking=True), dh.to(device, non_blocking=True))
        rendered = last["rendered"]
        if rendered is not None and chunk >= n_rays:
            for kk in keys:                                                           # D2H of the rendered buffers (15.4 MB for a frame) ...
                out_host[kk].copy_(rendered[kk], non_blocking=True)
        loss_host.copy_(loss, non_blocking=True)                                      # ... and of the loss
        torch.cuda.current_stream().synchronize()

    with ClockSampler(local, args.clock_period_ms) as clocks:          # see the class: one clock query after the last timed launch
        for i in range(args.warmup):
            resident(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        import gc
        gc.collect()
        gc.disable()                           # no collector pause inside a step; re-enabled right after the timed loops
        t_e2e = timed(e2e, args.steps)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t_res = timed(resident, args.steps, clocks)      # ... and the one clock query comes after its last launch (see ClockSampler)
        gc.enable()
        # the instrumented pass below reuses these buffers: keep what the last timed step computed
        timed_out = step_outputs(model, last["rendered"], last["loss"]) if args.dump_outputs else None
        overflow = int(frame.counts()["overflow"]) if frame is not None else 0
        # a separate, instrumented pass for the roofline: the same step launched kernel by kernel with CUDA events around every launch of
        # the hash-gather kernels (not part of `value`); sizes are read back after every step to count the points that were processed
        inst_steps = min(args.steps, 5)
        points = dict(gather=0, marched=0, boundary=0, kept=0)
        launches_per_step = None
        if frame is not None:
            inst = StaticFrame(model, n_rays, loss_fn=loss_of, near=near, use_graph=False, pre_hook=flat.zero_, march_cap=frame.march_cap,
                               kept_cap=frame.kept_cap, coherent=frame.coherent)
            inst.step(*views_dev[0])
            torch.cuda.synchronize()
            l0 = _lib.launch_count()
            inst.step(*views_dev[0])
            launches_per_step = _lib.launch_count() - l0
            _lib.KERNEL_TIMER.enable()
            t_inst = []
            for i in range(inst_steps):
                flush_buf.fill_(i & 0xff)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); inst.step(*views_dev[i % n_views]); b.record()
                torch.cuda.synchronize()
                t_inst.append(a.elapsed_time(b))
                c = inst.cnt.tolist()
                stages = [c[14 + q] for q in range(4) if c[14 + q]]
                fine_q = sum(stages[:-1]) if stages else 0         # the fine samples that are re-queried: every stage but the last
                points["marched"] += c[12]; points["boundary"] += c[18]; points["kept"] += c[19]
                points["gather"] += c[12] + fine_q + c[18]
            _lib.KERNEL_TIMER.disable()
        else:
            l0 = _lib.launch_count()
            _lib.KERNEL_TIMER.enable()
            t_inst = timed(resident, inst_steps)
            _lib.KERNEL_TIMER.disable()
            launches_per_step = (_lib.launch_count() - l0) // max(inst_steps, 1)
    st_res, st_e2e = stats_of(t_res), stats_of(t_e2e)
    ms = torch.tensor([st_res["mean"], st_e2e["mean"], st_res["median"], st_e2e["median"]], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_res, ms_e2e, med_res, med_e2e = (float(x) for x in ms)
    if args.dump_render and rank == 0:
        with torch.no_grad():
            model.eval()
            o0, d0 = pinhole_rays(H, W, orbit(0, N_VIEWS))
            out = SingleVolumeRenderer(dict(near=near)).eval().render(model, o0.to(device), d0.to(device), rays_h_appear=torch.zeros(o0.shape[0], n_appear, device=device))["rendered"]
            torch.save({k: v.cpu() for k, v in out.items()}, args.dump_render)
            model.train()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if timed_out is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in timed_out.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
    kt = _lib.KERNEL_TIMER.summary()
    # the dominant kernel: the boundary SDF query (k_fused_sdf_tc, "fused_sdf_fwd": hash gather + tcgen05 decoder over the 65 coarse + 51 fine
    # samples of every ray) -- 35-40 % of the step.  (The no-grad queries of the up-sampling half run inside the persistent per-ray kernel.)
    gather = dict(kt["fused_sdf_fwd"]) if "fused_sdf_fwd" in kt else None
    if gather and frame is not None:
        gather["units"] = points["boundary"]          # points actually processed (the launch is sized by capacity)
    traffic, traffic_note = None, None
    try:       # dram bytes of the dominant gather launch, from the committed ncu --set full capture (per launch, like `achieved`)
        tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        traffic = tj["traffic_bytes_per_launch"]
        traffic_note = {"unit": "bytes per launch (dram read + write)", "algorithmic_bytes_of_that_launch": tj["algorithmic_bytes_per_launch"], "source": tj["source"]}
    except Exception:
        pass
    roof = None
    if gather and gather["ms"] > 0:
        achieved = gather["units"] * 512.0 / (gather["ms"] * 1e-3) / 1e9     # 512 B of table per encoded point (SURVEY §8d)
        per_ms = {k: v["ms"] / inst_steps for k, v in kt.items()}
        roof = {"kernel": "LoTD hash gather: k_fused_sdf_tc (gather + tcgen05 decoder), the boundary SDF query of the step (one launch per step)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_note": traffic_note, "points_per_launch": gather["units"] / max(gather["launches"], 1), "launches": gather["launches"],
                "avg_launch_ms": gather["ms"] / max(gather["launches"], 1), "share_of_step": gather["ms"] / max(sum(t_inst), 1e-9),
                "per_kernel_ms_per_step": per_ms, "points_per_step": {k: v / inst_steps for k, v in points.items()} if frame is not None else None,
                "how": "CUDA events around every launch of these kernels in a separate kernel-by-kernel pass of the same step (events cannot sit inside the graph)"}
    tot_rays = world * n_rays
    line = {
        "metric": "Mrays/sec fwd+bwd", "value": tot_rays / (ms_res * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_res, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f16",
        "data": "synthetic",
        "median": {"ms_per_step": med_res, "value": tot_rays / (med_res * 1e-3) / 1e6, "e2e_ms_per_step": med_e2e, "e2e_value": tot_rays / (med_e2e * 1e-3) / 1e6},
        "config": {"workload": args.workload, "model": "LoTDNeuS 16x2 LoTD (12.13M params) + 32-64-1 SDF MLP + 58-64-64-3 radiance MLP",
                   "frame": "800x600", "rays_per_step_per_gpu": n_rays, "ray_order": "random pixels" if args.random_rays else "image rows",
                   "collect_samples": bool(args.collect_samples), "mode": mode,
                   "step": {"graph": "one CUDA-graph launch per step, no host read (sizes stay on the device)", "static": "kernel-by-kernel, no host read",
                            "host": "kernel-by-kernel, three host reads per step"}[mode],
                   "samples_per_ray": "<=116 boundary, <=1024 marched",
                   "parallelism": f"dp{world} ray-shard ({args.scaling}), 1 all-reduce/step", "l2": "256 MiB L2 flush between steps; per-step working set >> 126 MB",
                   "camera_poses": n_views, "arena_overflow": overflow,
                   "arenas": {"march_cap": frame.march_cap, "kept_cap": frame.kept_cap} if frame is not None else None},
        "e2e": {"value": tot_rays / (ms_e2e * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(2 * n_rays * 3 * 4), "d2h_bytes_per_step": d2h_bytes,
                "what": "pinned-host rays H2D -> step -> rendered rgb/depth/normals/mask + loss D2H, sync"},
        "gpu_launches": int(launches_per_step * args.steps), "launches_per_step": int(launches_per_step),
        "host_launches_per_step": (1 if mode == "graph" else int(launches_per_step)),
        "clocks": clocks.summary(), "roofline": roof,
        "step_ms": {"resident": [round(x, 3) for x in t_res], "e2e": [round(x, 3) for x in t_e2e],
                    "resident_stats": {k: round(v, 3) for k, v in st_res.items()}, "e2e_stats": {k: round(v, 3) for k, v in st_e2e.items()}},
    }
    if args.impl == "reference-cuda":
        line["impl"] = "reference-cuda"
        line["gpu_launches"] = 0
        line["config"]["note"] = "the reference's own CUDA kernels (oracle/_ref) under the same orchestration; no neuralsim_b200 kernel runs"
    elif world == 1 and not args.no_ref_cuda and args.workload == "cfg2":
        # B1 of BASELINE.md, measured in a child process so that none of its module patching can leak into this arm; it also dumps its
        # eval render of view 0, against which ours is compared (BASELINE.json: "PSNR vs ref"; north_star: 1e-4 relative L2)
        try:
            dump = f"/tmp/nsb_ref_render_{os.getpid()}.pt"
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-cuda", "--steps", "10", "--warmup", "3",
                                "--no-cpu-baseline", "--rays", str(args.rays), "--dump-render", dump] + (["--random-rays"] if args.random_rays else [])
                               + (["--collect-samples"] if args.collect_samples else []),
                               capture_output=True, text=True, timeout=900)
            rl = json.loads(r.stdout.strip().splitlines()[-1])
            line["reference_cuda"] = {"value": rl["value"], "unit": "Mrays/s", "ms_per_step": rl["ms_per_step"], "median_ms_per_step": rl["median"]["ms_per_step"],
                                      "e2e": rl["e2e"]["value"], "steps": rl["steps"], "warmup": rl["warmup"],
                                      "what": "reference nr3d_lib CUDA kernels compiled from /root/reference (oracle/_ref), same B200, same workload"}
            line["vs_reference_cuda"] = {"value_ratio": line["value"] / rl["value"], "e2e_ratio": line["e2e"]["value"] / rl["e2e"]["value"],
                                         "median_ratio": line["median"]["value"] / rl["median"]["value"]}
            if os.path.exists(dump):
                ref = torch.load(dump)
                with torch.no_grad():
                    model.eval()
                    o0, d0 = pinhole_rays(H, W, orbit(0, N_VIEWS))
                    ours = SingleVolumeRenderer(dict(near=near)).eval().render(model, o0.to(device), d0.to(device), rays_h_appear=torch.zeros(o0.shape[0], n_appear, device=device))["rendered"]
                    model.train()
                par = {}
                for kk in keys:
                    x, y = ours[kk].double().cpu(), ref[kk].double()
                    mse = float((x - y).square().mean())
                    par[kk] = {"rel_l2": float((x - y).norm() / y.norm().clamp_min(1e-30)), "psnr_db": (None if mse == 0 else -10.0 * math.log10(mse))}
                line["parity_vs_reference_kernels"] = {"what": "800x600 eval render of view 0, ours vs the reference's own kernels (same weights, rays, grid); "
                                                               "psnr_db null = identical", **par}
                os.remove(dump)
        except Exception as ex:
            line["reference_cuda"] = {"unavailable": repr(ex)[:300]}
    if not args.no_cpu_baseline and world == 1:
        try:
            line["cpu_baseline"] = cpu_baseline(args.ref_rays)
        except Exception as ex:  # the oracle is test infrastructure; never let it take the bench line down
            line["cpu_baseline"] = {"error": repr(ex)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
