#!/usr/bin/env python
"""bench.py -- headline benchmark of the per-ray sample pipeline (contract: task prompt ④).

    python bench.py --gpus N --steps K --warmup W            # product arm (one rank per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own training step on the host cores, rank 0 only
    python bench.py ... --dump-outputs DIR                   # also write what the last timed training step computed, DIR/<name>.npy

Headline (the half of BASELINE.json's metric that north_star sets its targets on): **train rays/s (fwd+bwd)** on configs[2] --
ScanNet scene0241_01-shaped hybrid training step, 640x480 frames, 4096-ray batch (8x8 dilated patches of 8x8), 8 reference-view
feature maps, 2M neural points.  One step = forward + loss + backward (+ NCCL gradient all-reduce for N > 1) + Adam of the network
and of the point tables.  N > 1 is data parallel exactly as north_star describes it: the point cloud, grid, weights are replicated,
every rank trains on its OWN 4096-ray raster (weak scaling), the gradients of the MLPs and of the dense point tables (39 floats x
2M points = 312 MB) are all-reduced over NCCL, overlapped with the next forward's query / pyramid / packing.
Also reported in the same JSON line: `render` (configs[1]: 800x800 full-frame render, Mpix/s, N = 1), `train_blur*` (configs[3]),
`large_scene` (configs[4]: 8M points, 1296x968 frames, 1.25 GB of point gradients per all-reduce; every N), `cpu_baseline` and
`reference_gpu` (the unmodified reference's training step on the host cores / on the same B200).
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
sys.path.insert(0, ROOT)

H = W = 800
N_POINTS = 1_000_000
V = 4
CHUNK = None          # whole frame per query (one host readback per frame)
RENDER_WORKLOAD = "NeRF-synthetic lego-shaped full-frame render 800x800, synthetic 1M neural points (voxel query + aggregation + compositing)"
FLOP_NBR_FWD = 542_720                                   # per valid neighbour row, SURVEY.md 8d
FLOP_NBR_DGRAD = 2 * (3 * 256 * 256 + 256 * 224)         # dZ_3 -> dZ_2 -> dZ_1 -> dZ_0 -> dX0 (224 needed input columns)
BYTES_WGRAD_ROW = 4 * (4 * 256 + 288 + 256 + 272 + 256)  # every dZ / input image read once, 4 bytes per element
# dram__bytes_read.sum + dram__bytes_write.sum of one configs[2] training step, from the committed `ncu --set full` capture
# profiles/r2f_train_kernels_ncu.md (same command as scripts/train_step_bench.py, one frame of the benchmark's frame set)
NCU_TRAFFIC = {"nbr_mlp": 0.132934e9 + 3.252108e9,
               "backward/nbr_bwd_chain": 1.588010e9 + 2.353657e9,
               "backward/wgrad_img": (0.102070 + 1.203327 + 0.282054 + 5.085762) * 1e9 + (3.554 + 5.230 + 6.924 + 5.667) * 1e6}   # its 4 launches
NCU_TRAFFIC_SOURCE = "profiles/r2f_train_kernels_ncu.md (ncu --set full, same step; summed over the kernel's launches of one step like `achieved`)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    d, kind = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"
    if os.path.exists(p):
        d, kind = json.load(open(p)), "measured"
    t = os.path.join(ROOT, "profiles", "r2_tf32_peak.json")            # scripts/measure_tf32_peak.py on this pool's B200
    if os.path.exists(t):
        d = dict(d, **{k: v for k, v in json.load(open(t)).items() if k.startswith("tf32_")})
    return d, kind


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML every 20 ms; nvidia-smi as a fallback)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self.run, daemon=True)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") else \
            n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        g = lambda name, alt: getattr(n, name, getattr(n, alt, 0))
        bits = [g("nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                g("nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                g("nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                g("nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap")]
        return [str(sm), str(mx)] + ["Active" if (b and (r & b)) else "Not Active" for b in bits]

    def run(self):
        while not self.stop:
            try:
                if self.nvml is not None:
                    self.rows.append(self.sample_nvml())
                    time.sleep(0.02)
                    continue
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                self.nvml = None
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows if len(r) > 2 + i)]
        # median over the samples taken under load (idle samples between steps sit at the idle clock)
        hot = [x for x in sm if x >= 0.6 * max(sm)] if sm else []
        return {"sm_mhz": hot[len(hot) // 2] if hot else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


DUMP_POINT_ROWS = 1 << 16       # rows of the point tables --dump-outputs writes: a fixed sample (seed 0) of the 2M points
DUMP_MAX_BYTES = 64 << 20


def dump_train_outputs(out_dir, net, loss, n_valid):
    """--dump-outputs: what the last timed training step leaves its caller, as DIR/<name>.npy (float32, counts and row ids float64):
    the loss and valid-ray count train_step returns, every trained network parameter after the optimiser step, and of the trained
    per-point tables the rows of DUMP_POINT_ROWS points.  The inputs are seeded, so two builds can be compared output for output."""
    arrays = {"loss": loss.detach().float().cpu().numpy(), "valid_rays": n_valid.detach().double().cpu().numpy()}
    rows = None
    for name, p in net.named_parameters():
        if not p.requires_grad:
            continue
        t = p.detach()
        if name.startswith("neural_points."):
            t = t.reshape(-1, t.shape[-1])                                   # (1, N, C) or (N, C) -> (N, C)
            if rows is None:
                rows = np.sort(np.random.default_rng(0).choice(t.shape[0], size=min(t.shape[0], DUMP_POINT_ROWS), replace=False))
                arrays["neural_points.sample_rows"] = rows.astype(np.float64)
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
        arrays[name] = t.float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes > {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ======================================================================================================================
# reference arm / cpu_baseline / reference_gpu: the reference's own training step (oracle/reference_pipeline.py)
# ======================================================================================================================
def train_scene(views=8, points=2_000_000):
    from hybridneuralrendering_b200 import make_opt
    from hybridneuralrendering_b200 import synthetic as syn
    from hybridneuralrendering_b200.synthetic import point_attributes
    opt = make_opt("scannet", use_nearest=views, SR=24, is_train=True, drop_ratio=0.5, dilation_setup="8_8_1_8", max_o=1_000_000)
    xyz = syn.room_scene(points, 0)
    att = point_attributes(np.random.default_rng(0), len(xyz))
    fr = syn.room_frame(H=480, W=640, V=views, patch_num=8, patch_size=8, seed=0)
    return opt, xyz, att, fr


def reference_step_times(device: str, rays: int, repeats: int, warmup: int):
    """times the reference's training step on the first `rays` rays (whole 8x8 patches) of the headline's 4096-ray raster.
    -> dict(rays/s over fwd+bwd of aggregation+compositing, with the query reported next to it)"""
    from oracle import reference_pipeline as rp
    from oracle import render_oracle as ro
    opt, xyz, att, fr = train_scene()
    # whole patch ROWS of the raster: the first `rays` rays of the (64 x 64)-pixel patch raster
    ids = np.arange(min(rays, fr["raydir"].shape[1]))
    # the reference's patch drop indexes the raster of the WHOLE batch (point_aggregators.py:1222-1237): on a sub-sample of the rays
    # its positions fall outside the compacted ray array, so the sample runs without the drop (the dropped rays cost the same)
    st = rp.ReferenceStep(xyz, att, fr, opt, ro.random_params(0), device, ray_ids=ids, drop_ratio=0.0)
    tq = st.query()
    f, b = [], []
    for i in range(warmup + repeats):
        tf, tb, kept, loss = st.fwd_bwd()
        if i >= warmup:
            f.append(tf); b.append(tb)
    tf, tb = float(np.mean(f)), float(np.mean(b))
    return {"rays": int(len(ids)), "kept_rays": kept, "s_fwd": tf, "s_bwd": tb, "s_query": tq, "value": len(ids) / (tf + tb), "value_with_query": len(ids) / (tf + tb + tq),
            "kind": rp.kind(), "query": st.query_kind, "loss": loss}


def run_reference(args, rank):
    """--impl reference: the reference's own implementation of the path on the box's host cores, all threads, the headline's
    metric / unit / workload; each step = fwd+bwd of a bounded sample of the 4096-ray batch."""
    if rank != 0:
        return
    from hybridneuralrendering_b200.benchmarks import TRAIN_WORKLOAD
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    rays = 1024 if cores >= 8 else 512            # ~2-3 s of host work per step: the K+W run ends within a few minutes
    r = reference_step_times("cpu", rays, args.steps, args.warmup)
    sample = (f"first {r['rays']} rays (16 whole patches of the 4096-ray raster, {r['kept_rays']} hit the scene) per step: PointAggregator.forward + ray_dist "
              f"+ ray_march + loss + backward ({r['kind']}: {'unmodified reference classes' if r['kind'] == 'reference' else 'oracle port'}), torch {torch.__version__} "
              f"CPU fp32, {cores} threads; fwd {r['s_fwd']:.2f} s + bwd {r['s_bwd']:.2f} s per step; the voxel query is not in the metric "
              f"(the reference has no CPU query; {r['query']} took {r['s_query']:.2f} s incl. its per-call grid build)")
    line = {"impl": "reference", "metric": "train rays/s (fwd+bwd)", "value": r["value"], "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": (r["s_fwd"] + r["s_bwd"]) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": TRAIN_WORKLOAD, "sample": sample},
            "cpu_baseline": {"value": r["value"], "unit": "rays/s", "cores": cores, "kind": r["kind"], "sample": sample},
            "e2e": {"value": r["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ======================================================================================================================
# configs[1]: full-frame render (N = 1 only; frames are independent units, no collective)
# ======================================================================================================================
FRAME_KEYS = ("campos", "camrotc2w", "raydir", "near", "far", "intrinsic", "bg_color", "images_nearest", "c2w_nearest", "campos_nearest",
              "intrinsic_nearest")


def render_benchmark(dev, steps, warmup, pk):
    from hybridneuralrendering_b200 import NeuralPoints, NeuralPointsRayMarching, PointAggregator, make_opt, ops, profiling
    from hybridneuralrendering_b200 import synthetic as syn
    from hybridneuralrendering_b200.renderer import render_rays
    xyz = syn.lego_scene(N_POINTS, 0)
    att = syn.point_attributes(np.random.default_rng(0), len(xyz))
    fr = syn.lego_frame(H=H, W=W, V=V, seed=0)
    opt = make_opt("lego", use_nearest=V, is_train=False)
    c = lambda a: torch.from_numpy(a).to(dev)
    pts = NeuralPoints(32, len(xyz), opt, dev)
    t0 = time.perf_counter()
    pts.set_points(c(xyz), c(att["emb"])[None], points_color=c(att["color"])[None], points_dir=c(att["dir"])[None],
                   points_conf=c(att["conf"])[None], parameter=True)
    torch.manual_seed(0)
    agg = PointAggregator(opt).to(dev)
    agg.load_state_dict(syn.random_aggregator_params(0), strict=False)
    net = NeuralPointsRayMarching(aggregator=agg, neural_points=pts, opt=opt).to(dev)
    net.near_far = (2.0, 6.0)
    host = {k: torch.from_numpy(np.ascontiguousarray(fr[k])).pin_memory() for k in FRAME_KEYS}
    resident = {k: v.to(dev) for k, v in host.items()}
    img = torch.empty((H * W, 3), device=dev)
    img_host = torch.empty((H * W, 3)).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    # grid build: once per point set (amortised, not in the Mpix/s), reported separately (SURVEY 8d)
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    pts.querier._ensure_grid(pts.xyz[None, ...])
    g1.record()
    torch.cuda.synchronize()
    grid_ms = g0.elapsed_time(g1)

    def step_resident():
        render_rays(net, resident, CHUNK, out=img)

    def step_e2e():
        f = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        render_rays(net, f, CHUNK, out=img)
        img_host.copy_(img, non_blocking=True)

    def timed(fn, n):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        torch.cuda.synchronize()
        for s, e in ev:
            flush.zero_()
            s.record()
            fn()
            e.record()
        torch.cuda.synchronize()
        return sum(s.elapsed_time(e) for s, e in ev) / 1e3

    for _ in range(warmup):
        step_resident()
    ops.LAUNCHES = 0
    t_res = timed(step_resident, steps)
    launches = ops.LAUNCHES
    step_e2e()
    t_e2e = timed(step_e2e, steps)
    mpix = H * W / 1e6
    roof = profiling.dominant_kernel_roofline(net, resident, CHUNK, pk)
    roof["step"] = profiling.step_roofline(roof["units"], V, H * W, int(opt.z_depth_dim), int(opt.SR), H, W, t_res / steps * 1e3, pk[0])
    return {"metric": "render Mpix/s", "value": steps * mpix / t_res, "unit": "Mpix/s", "ms_per_frame": t_res / steps * 1e3,
            "e2e": {"value": steps * mpix / t_e2e, "unit": "Mpix/s", "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in host.values()),
                    "d2h_bytes_per_step": img_host.numel() * 4},
            "grid_build_ms": grid_ms, "grid_build_note": "occupancy-grid build of the 1M points, once per point-set change (the reference rebuilds per forward)",
            "gpu_launches": launches, "roofline": roof,
            "config": {"workload": RENDER_WORKLOAD, "rays_per_step": H * W, "chunk_rays": CHUNK or H * W, "valid_samples_per_pass": agg.max_valid_chunk,
                       "use_nearest": V, "SR": int(opt.SR), "K": int(opt.K), "l2": "flushed between frames (256 MB write)"}}


def config0_product(dev, repeats=5, warmup=3):
    """BASELINE.json configs[0] on the product: the drop-in PointAggregator.forward on the SAME gathered tensors (1024 rays x 80 samples,
    K = 8 precomputed neighbours, 200K points, V = 4) + ray_dist + ray_march + loss, forward and backward, CUDA events"""
    from hybridneuralrendering_b200 import PointAggregator, make_opt
    from hybridneuralrendering_b200 import synthetic as syn
    from hybridneuralrendering_b200.diff_ray_marching import ray_march_from_depth
    d = syn.render_stage_inputs(seed=0)
    g = syn.gather_neighbours(d)
    c = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    agg = PointAggregator(make_opt(use_nearest=4, is_train=False)).to(dev)
    agg.load_state_dict(syn.random_aggregator_params(0), strict=False)
    leaf = {k: c(g[k]).requires_grad_(True) for k in ("sampled_embedding", "sampled_color", "sampled_dir", "sampled_conf")}
    fixed = [c(g["sampled_xyz_pers"]), c(g["sampled_xyz"]), c(g["sample_pnt_mask"]), c(d["sample_loc"]), c(d["sample_loc_w"]), c(d["sample_ray_dirs"])]
    img, xy, dv = c(d["images_nearest"]), c(d["sample_loc_i_n"]), c(d["delta_viewdir_n"])
    R = d["sample_pidx"].shape[1]
    gt = c(np.random.default_rng(7).random((1, R, 3), dtype=np.float32))
    bg = torch.ones(1, 3, device=dev)

    def step():
        for t in list(leaf.values()) + list(agg.parameters()):
            t.grad = None
        out = agg(leaf["sampled_color"], torch.eye(3, device=dev), leaf["sampled_dir"], leaf["sampled_conf"], leaf["sampled_embedding"], *fixed,
                  d["vsize"], 0, img_n=img, sample_loc_i_n=xy, delta_viewdir_n=dv)
        color = ray_march_from_depth(fixed[3], out[1], out[0], float(d["vsize"][2]), 1, bg)[0]
        loss = torch.nn.functional.mse_loss(color, gt)
        loss.backward()
        return loss
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(repeats):
        loss = step()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / repeats
    return {"value": R / (ms * 1e-3), "unit": "rays/s", "ms_fwd_bwd": ms, "rays": R, "loss": float(loss.detach()),
            "path": "drop-in PointAggregator.forward (gathered tensors, as the reference calls it) + ray_march, fwd + bwd"}


def train_kernel_rooflines(tr, pk):
    """roofline records of the three big kernels of the fused training path from the per-launch CUDA events of one step"""
    peaks_d, kind = pk
    M, rows = tr["valid_neighbours"], tr["valid_samples"] * 8
    rows_pad = (rows + 127) // 128 * 128
    tens = peaks_d["bf16_tflops_sustained"] / 3.0
    st = tr["stage_ms"]
    out = []

    def rec(name, tag, bound, work, peak, unit, note):
        ms = st.get(tag)
        if not ms:
            return
        ach = work / (ms * 1e-3) / (1e12 if bound == "tensor" else 1e9)
        out.append({"kernel": name, "bound": bound, "ms": ms, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak, "work_per_launch": work,
                    "traffic": NCU_TRAFFIC.get(tag), "note": note})

    rec("nbr_mlp_f16_kernel<2> (fused per-neighbour forward, training mode: saves its operands as split images)", "nbr_mlp", "tensor",
        FLOP_NBR_FWD * M, tens, "TFLOP/s", "542,720 FLOP x valid neighbours; peak = bf16_tflops_sustained/3 (3 f16 MMAs per fp32-accurate product)")
    rec("nbr_bwd_f16_kernel (fused data-gradient chain dZ_3 -> dX0)", "backward/nbr_bwd_chain", "tensor", FLOP_NBR_DGRAD * M, tens, "TFLOP/s",
        "2*(3*256*256 + 256*224) FLOP x valid neighbours; peak = bf16_tflops_sustained/3 (3 bf16 MMAs per product)")
    ws = st.get("backward/wgrad_img")
    if ws:
        # three wgrad_img launches per step (per-neighbour MLP + three chains); the per-neighbour one dominates: attribute by bytes
        v, nv = tr["views"], tr["valid_samples"]
        chain_bytes = 4 * (nv * (3 * 128 + 288 + 128 + 128) + v * nv * (3 * 64 + 176 + 64 + 64) + nv * (3 * 48 + 96 + 48 + 48))
        work = BYTES_WGRAD_ROW * rows_pad + chain_bytes
        ach = work / (ws * 1e-3) / 1e9
        out.append({"kernel": "wgrad_img_kernel (all weight/bias gradients from MN-major slab images, 4 launches per step)", "bound": "hbm", "ms": ws,
                    "achieved": ach, "peak": peaks_d["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks_d["hbm_gbs"], "work_per_launch": work,
                    "traffic": NCU_TRAFFIC["backward/wgrad_img"],
                    "note": "every dZ / input image read once (4 B per element); the two 128-row halves of a layer re-read the input image through L2"})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-render", action="store_true", help="skip the configs[1] full-frame render (N = 1)")
    ap.add_argument("--no-large", action="store_true", help="skip configs[4] (8M points)")
    ap.add_argument("--no-extras", action="store_true", help="skip configs[3] (blur) and the reference_gpu leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="product arm: write what the last timed training step computed to DIR/<name>.npy "
                                                          "(rank 0 writes; the ranks' parameters are identical after the all-reduce)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "product":
        ap.error("--dump-outputs applies to the product arm only")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch.distributed as dist
    from hybridneuralrendering_b200 import benchmarks, profiling

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback of the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    steps, warmup = args.steps, max(3, args.warmup)
    dump = None
    if args.dump_outputs and rank == 0:
        dump = lambda net, loss, n_valid: dump_train_outputs(args.dump_outputs, net, loss, n_valid)

    # ---------------------------------------------------------------- headline: configs[2] training step
    with ClockSampler(local) as clk:
        tr = benchmarks.train_step_benchmark(dev, steps=steps, warmup=warmup, world=world, rank=rank, stage_split=(world == 1), capture=dump)
    roofs = train_kernel_rooflines(tr, pk) if world == 1 else []
    top = max(roofs, key=lambda r: r["ms"]) if roofs else None
    # whole-step roofline (SURVEY 8d) against fwd+bwd time: backward on the f16 pipe like the forward (3 bf16 MMAs per product)
    step_roof = profiling.step_roofline(tr, tr["views"], tr["rays_per_step_per_gpu"], 400, 24, 480, 640, tr["ms_fwd_bwd"], pk[0], train=True,
                                        points=tr["points"])
    line = {"metric": "train rays/s (fwd+bwd)", "value": tr["value"], "unit": "rays/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": tr["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": benchmarks.TRAIN_WORKLOAD, "rays_per_step_per_gpu": tr["rays_per_step_per_gpu"], "points": tr["points"], "views": tr["views"],
                       "SR": 24, "K": 8, "step": tr["step"], "l2": "flushed between steps (256 MB write)",
                       "query": "the next step's voxel query is launched one step ahead (one query per step, software-pipelined)",
                       "mlp_engine": "3xFP16 tcgen05 fused forward, 3xBF16 tcgen05 fused backward (split images)",
                       "parallelism": (f"dp{world}: point cloud / grid / weights replicated, every rank its own 4096-ray raster, NCCL SUM all-reduce of the MLP bucket "
                                       "(1.8 MB) and of the dense point-gradient tables (312 MB) overlapped with the next forward's query / pyramid / packing")
                       if world > 1 else "1 GPU"},
            "e2e": tr.get("e2e"), "gpu_launches": tr["launches_per_step"] * steps, "clocks": clk.summary(),
            "train": {k: tr[k] for k in ("ms_per_step", "ms_fwd_bwd", "kept_rays", "valid_samples", "valid_neighbours", "loss", "launches_per_step", "stage_ms", "ranks") if k in tr}}
    if top is not None:
        line["roofline"] = {"bound": top["bound"], "achieved": top["achieved"], "peak": top["peak"], "unit": top["unit"], "frac": top["frac"],
                            "traffic": top.get("traffic"), "traffic_source": NCU_TRAFFIC_SOURCE, "kernel": top["kernel"], "kernel_ms": top["ms"],
                            "note": top["note"],
                            "peak_source": f"MEASURED_PEAKS.json ({pk[1]}), sustained figures (kernels timed inside a long step)",
                            "kernels": roofs, "step": step_roof}
    else:
        line["roofline"] = {"bound": "tensor", "achieved": None, "peak": None, "unit": "TFLOP/s", "frac": None, "traffic": None,
                            "note": "per-kernel events are taken at N = 1 only", "step": step_roof}
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- configs[4]: 8M points (every N; the 1.25 GB all-reduce)
    if not args.no_large:
        lg = benchmarks.train_step_benchmark(dev, steps=min(steps, 10), warmup=3, world=world, rank=rank, stage_split=False, points=8_000_000,
                                             size=(12.0, 10.0, 3.0), H=968, W=1296, max_o=4_000_000, e2e=False, workload=benchmarks.LARGE_WORKLOAD)
        line["large_scene"] = {k: lg[k] for k in ("metric", "value", "unit", "ms_per_step", "ms_fwd_bwd", "rays_per_step_per_gpu", "points", "views", "kept_rays",
                                                  "valid_samples", "step", "config")}
        line["large_scene"]["n_gpus"] = world
        if "ranks" in lg:
            line["large_scene"]["ranks"] = lg["ranks"]
        line["large_scene"]["allreduce_bytes"] = 39 * 4 * lg["points"] if world > 1 else 0
        torch.cuda.empty_cache()

    if world == 1:
        if not args.no_render:
            line["render"] = render_benchmark(dev, steps, warmup, pk)
            torch.cuda.empty_cache()
        if not args.no_extras:
            line["train_blur"] = benchmarks.blur_train_step_benchmark(dev, steps=3, warmup=3)      # BASELINE configs[3]
            line["train_blur_learnable"] = benchmarks.blur_train_step_benchmark(dev, steps=3, warmup=3, learnable=True)   # SURVEY 8f N3
            torch.cuda.empty_cache()
            try:
                r = reference_step_times("cuda", 4096, 3, 2)
                line["reference_gpu"] = {"value": r["value_with_query"], "unit": "rays/s", "value_without_query": r["value"], "kind": r["kind"], "rays": r["rays"],
                                         "s_query": r["s_query"], "s_fwd": r["s_fwd"], "s_bwd": r["s_bwd"],
                                         "what": f"the reference's own GPU path on this B200, same 4096-ray batch: {r['query']} (grid rebuilt per call) + "
                                                 "PointAggregator / ray_march (ATen, cuBLAS fp32) fwd + bwd; no optimiser step"}
            except Exception as e:      # the comparator must never break the product line
                line["reference_gpu"] = {"unavailable": repr(e)[:300]}
            torch.cuda.empty_cache()
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            try:
                r = reference_step_times("cpu", 2048 if cores >= 8 else 512, 3, 1)          # mean of 3 timed passes after one warm-up (~6 s of host work)
                line["cpu_baseline"] = {"value": r["value"], "unit": "rays/s", "cores": cores, "kind": r["kind"],
                                        "sample": (f"first {r['rays']} rays (whole patches) of the same 4096-ray batch, fwd {r['s_fwd']:.1f} s + bwd {r['s_bwd']:.1f} s of "
                                                   f"PointAggregator.forward + ray_dist + ray_march + loss + backward, torch {torch.__version__} CPU fp32; query "
                                                   f"({r['query']}, {r['s_query']:.1f} s) not in the metric")}
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "unit": "rays/s", "cores": cores, "kind": "port", "sample": "unavailable: " + repr(e)[:300]}
            # BASELINE.json configs[0] / BASELINE.md §3: the render stage on precomputed neighbours, reference on the host cores vs the product
            try:
                from oracle import reference_pipeline as rp
                c0 = rp.config0_reference("cpu", repeats=3, warmup=1)
                line["config0"] = {"workload": "render stage on CPU: diff_ray_marching + point_aggregators fwd/bwd, synthetic 200K neural points (32-ch), 1024 rays x 80 "
                                               "samples, K=8 precomputed neighbours",
                                   "reference_cpu": dict(c0, cores=cores, torch=torch.__version__), "product_gpu": config0_product(dev)}
            except Exception as e:
                line["config0"] = {"unavailable": repr(e)[:300]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
