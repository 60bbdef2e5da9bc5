#!/usr/bin/env python
"""bench.py — training rays/s of the F2-NeRF per-ray rendering hot path on B200.

One "step" = one pass of the hot path over one batch: Renderer.Render (perspective-warp ray march,
early-stop pass, hash encode, density + colour MLPs, composite) + the trainer's loss + backward down
to the parameter gradients (+ the NCCL gradient / octree-vote all-reduce when N > 1).  The optimizer
step is outside the path (SURVEY.md §8d).

Workload (``--config``, default ``wanjinyou`` = BASELINE.json configs[1], the configuration the metric is quoted on):
4096 rays x <= 1024 samples per ray per GPU, log2_table_size 19, confs/wanjinyou.yaml sampler settings, on the
REFERENCE'S OWN ngp_fox octree / warps / cameras (committed fixture tests/golden/ref_ngp_fox.npz — the blobs the
unmodified reference built), rays drawn like Dataset::RandRaysData under seed 2023, parameters initialised like
oracle/ref_driver.cpp — so `reference_gpu` (the compiled reference, oracle/_ref/ref_driver, timed on the same box)
runs the very same batch.  Other configs (tests/workloads.py): free, nerf360 (8192 rays global, strong scaling),
big20, big22, synthetic.

  python bench.py --gpus N --steps K --warmup W [--config C]      (torchrun launches N > 1)
  python bench.py --impl reference ...     the path's CPU port (oracle/) on the same config, all host threads, rank 0 only
  python bench.py ... --dump-outputs DIR   also write what the last step of the first timed pass returned (step_outputs)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import workloads as W  # noqa: E402   (numpy / torch-CPU only: does not load the CUDA library)


def config_dict(args, world):
    """The `config` object of the JSON line: a pure function of (--config, --rays, N) so both arms print the same one."""
    cfg = W.CONFIGS[args.config]
    rays = args.rays or cfg["rays"]
    per_gpu = rays // world if cfg["scaling"] == "strong" else rays
    scene = ("the reference's ngp_fox octree / warps / cameras (tests/golden/ref_ngp_fox.npz), rays as Dataset::RandRaysData seed 2023"
             if cfg["scene"] == "ngp_fox" else "synthetic 24-camera octree (tests/synth_scene.py)")
    return {"workload": f"{args.config}: BASELINE configs[{cfg['baseline_config']}] ({cfg['yaml']}) — {per_gpu} rays x <=1024 samples per GPU, "
                        f"near {cfg['near']}, scale_by_dis {cfg['scale_by_dis']}, use_app_emb {cfg['use_app_emb']}, sample_l 1/256, "
                        f"fineness 1, log2_table_size {cfg['log2_table']}; {scene}; table U(-1,1), field MLP x4 (as oracle/ref_driver.cpp); "
                        "Render + loss + backward",
            "name": args.config, "rays_per_gpu": per_gpu, "global_rays": per_gpu * world, "log2_table_size": cfg["log2_table"],
            "parallelism": f"dp{world} (rays sharded, params replicated)",
            "l2": "per-step working set (>=100 MB of samples + the table) exceeds the 126 MB L2; no explicit flush"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), tf=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, tf=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region, sampled in-process through NVML (no nvidia-smi
    subprocesses: they stall kernel launches for tens of ms each)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.err, self.h = index, [], False, None, None
        if index < 0:
            self.err = "not sampled on this rank"
            return
        try:                                     # nvmlInit takes ~0.3 s and a driver lock: do it before the timed region
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[index]) if vis and vis.split(",")[0].isdigit() else index
            self.h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.err = str(e)[:120]

    def poll(self):
        if self.h is None:
            return
        import pynvml as nv
        try:
            self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksEventReasons(self.h),
                              nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
        except Exception as e:  # noqa: BLE001
            self.err = str(e)[:120]

    def run(self):
        # An NVML query holds a driver lock for tens of ms on this driver and perturbs kernel submission for a while afterwards:
        # the first (slowest) queries happen before the warm-up, then one every 0.3 s.  A timed loop that one of them lands in is
        # rejected by the host-stall rule below and re-timed (all attempts are reported).
        while not self.stop_flag and self.h is not None:
            self.poll()
            time.sleep(0.3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {self.err}"]}
        import pynvml as nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(self.max_mhz), "reasons": [k for k, v in names.items() if bits & v],
                "power_w_max": max(r[2] for r in self.rows), "samples": len(self.rows)}


def build_problem(rank, world, args, device):
    import torch
    from f2nerf_b200 import TRAIN, GlobalDataPool, Hash3DAnchored, PersSampler, RayGenerator, Renderer, SHShader
    cfg = W.CONFIGS[args.config]
    sb = W.scene_blobs(args.config)                               # identical octree on every rank
    nodes, trans, edges = sb["nodes"], sb["trans"], sb["edges"]
    gdp = GlobalDataPool()
    sampler = PersSampler(gdp, nodes, trans, edges, near=cfg["near"], sample_l=cfg["sample_l"], scale_by_dis=cfg["scale_by_dis"],
                          device=device)
    par = W.init_params(args.config, gdp.n_volumes_, sb["n_images"], sb["prim"], sb["bias"])       # replicated parameters
    field = Hash3DAnchored(gdp, log2_table_size=cfg["log2_table"], device=device, prim_pool=par["prim"], bias_pool=par["bias"])
    field.feat_pool_.data.copy_(torch.from_numpy(par["table"]))
    field.mlp_.params_.data.copy_(torch.from_numpy(par["field_mlp"]))
    shader = SHShader(gdp, device=device)
    shader.mlp_.params_.data.copy_(torch.from_numpy(par["shader_mlp"]))
    renderer = Renderer(gdp, sampler, field, shader, n_images=sb["n_images"], use_app_emb=cfg["use_app_emb"], device=device)
    renderer.app_emb_.data.copy_(torch.from_numpy(par["app_emb"]))
    gdp.mode_ = TRAIN
    rays = args.rays or cfg["rays"]
    if cfg["scaling"] == "strong":                                 # one global batch, rank r renders its slice
        n_draw, seed, lo, hi = rays, 2023, rank * (rays // world), (rank + 1) * (rays // world)
    else:                                                          # rank-sharded i.i.d. batches (weak scaling)
        n_draw, seed, lo, hi = rays, 2023 + rank, 0, rays
    if sb["synthetic"] is not None:
        o, d, cam = sb["synthetic"].rays(n_draw, seed=1234 + (0 if cfg["scaling"] == "strong" else rank))
    else:                                                          # the product's own ray generation (N3) on the reference's cameras
        g = sb["golden"]
        gen = RayGenerator(g["ds_poses"].reshape(-1, 3, 4), g["ds_intri"].reshape(-1, 3, 3), g["ds_dist_params"], g["ds_bounds"],
                           images=None, height=int(g["ds_hw"][0]), width=int(g["ds_hw"][1]), train_set=g["ds_train_set"].tolist(),
                           device=device)
        torch.manual_seed(seed)
        (ro, rd, _), _, cam_d = gen.RandRaysData(n_draw)
        o, d, cam = ro.cpu().numpy(), rd.cpu().numpy(), cam_d.cpu().numpy()
        prob_gen = gen
    o, d, cam = (np.ascontiguousarray(x[lo:hi]) for x in (o, d, cam))
    rng = np.random.default_rng(99 + rank)
    gt = rng.random((hi - lo, 3), dtype=np.float32)
    return dict(gdp=gdp, sampler=sampler, field=field, shader=shader, renderer=renderer, cfg=cfg, n_rays=hi - lo,
                host=(o, d, cam, gt), blobs=(nodes, trans, edges), n_images=sb["n_images"],
                ray_gen=None if sb["synthetic"] is not None else prob_gen)


def train_step(prob, rays_o, rays_d, emb_idx, gt, dist_sync=None, next_rays=None):
    """ExpRunner::Train's use of the path (src/ExpRunner.cpp:93-130) minus the optimizer step.  ``next_rays``: the
    (rays_o, rays_d) the NEXT call will be given (or a callable producing them — the e2e loop uploads them here): their
    march is software-pipelined behind this step's loss + backward (Renderer.prefetch_next); every step still runs exactly
    one march."""
    import torch
    from f2nerf_b200 import CustomOps
    r = prob["renderer"]
    for p in (prob["field"].feat_pool_, prob["field"].mlp_.params_, prob["shader"].mlp_.params_, r.app_emb_):
        p.grad = None
    nxt = None
    if next_rays is not None:
        nxt = next_rays() if callable(next_rays) else next_rays
        if os.environ.get("F2B_EARLY_PREFETCH", "1") == "1":
            r.set_next_rays(nxt[0], nxt[1])                        # Render launches their march itself, behind its occupancy votes
    res = r.Render(rays_o, rays_d, None, emb_idx)
    if nxt is not None:
        r.prefetch_next(nxt[0], nxt[1])                            # no-op when Render already did
    color_loss = torch.sqrt((res.colors - gt) ** 2 + 1e-4).mean()
    var_loss = torch.sqrt(CustomOps.WeightVar(res.weights, res.idx_start_end) + 1e-2).mean()
    tv_loss = ((res.edge_feats[:, 0] - res.edge_feats[:, 1]) ** 2).mean()
    loss = color_loss + var_loss * 1e-2 + tv_loss * 1e-1
    loss.backward()
    if dist_sync is not None:
        dist_sync(prob)
    return loss, res


ALGO_BYTES = {  # algorithmic bytes per unit (sample) at the operator boundary — DESIGN.md "roofline accounting"
    "f2b_field_fwd": 16 + 512 + 64, "f2b_field_fwd_slots": 16 + 512 + 64, "f2b_sampler_march": 28, "f2b_compact_slots": 28 + 64 + 44 + 64,
    "f2b_hash_fwd": 16 + 512 + 64, "f2b_hash_bwd": 16 + 64 + 512, "f2b_sampler_fill": 44, "f2b_sampler_count": 0,
    "f2b_composite_fwd": 28, "f2b_composite_bwd": 24 + 16 + 16, "f2b_early_stop": 8 + 9, "f2b_compact_samples": 88,
    "f2b_shader_prep": 64 + 12 + 64, "f2b_shader_act": 32 + 12, "f2b_cast_f16_to_f32": 6, "f2b_cast_f32_to_f16": 6,
}


NCU_KERNEL = {"f2b_hash_bwd": "hash_bwd_kernel<1>", "f2b_sampler_march": "march16_kernel<2, 0>",
              "f2b_field_fwd_slots": "field_fwd_kernel<1, 4>", "f2b_field_fwd": "field_fwd_kernel<1, 4>",
              "f2b_mlp_bwd2": "mlp_bwd_rc_kernel<1>",
              "f2b_compact_slots": "compact_slots_kernel", "f2b_composite_fwd": "composite_fwd_kernel",
              "f2b_composite_bwd": "composite_bwd_kernel<0>", "f2b_composite_act_bwd": "composite_bwd_kernel<1>"}


def ncu_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel behind C-ABI call ``name``, from the
    committed `ncu --set full` capture of this same command (profiles/*_traffic.json, newest round); None if absent."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files or name not in NCU_KERNEL:
        return None
    try:
        k = json.load(open(files[-1]))["kernels"].get(NCU_KERNEL[name])
        return None if k is None else {"dram_bytes_per_launch": k["dram_bytes_per_launch"], "source": os.path.basename(files[-1])}
    except Exception:  # noqa: BLE001
        return None


GOVERNING_OK = True      # main() clears it for any workload other than the one the committed ncu capture was taken on


def governing_roofline(name, per_launch_ms):
    """The hardware rate that actually bounds the two table kernels, next to the HBM figure the contract asks for: both keep the
    table L2-resident (17 MB live at log2 19), so DRAM bytes say little.  `units` per launch come from the committed ncu capture of
    this same command (profiles/*_traffic.json: reduction / load sectors leaving the SM; deterministic for a seeded batch), the time
    is THIS run's, the peak is the microbenchmark of the same instruction mix on this GPU type (scripts/microbench_red.cu /
    microbench_gather.cu -> profiles/*_red_rate.json / *_gather_rate.json, random addresses in a table-sized L2-resident buffer)."""
    import glob
    spec = {"f2b_hash_bwd": ("l2_reduction_issue", "red_sectors_per_launch", "*_red_rate.json", "G lane-reductions/s"),
            "f2b_field_fwd_slots": ("l1_l2_gather_sectors", "ld_sectors_per_launch", "*_gather_rate.json", "G 32B-sectors/s"),
            "f2b_field_fwd": ("l1_l2_gather_sectors", "ld_sectors_per_launch", "*_gather_rate.json", "G 32B-sectors/s")}.get(name)
    tf = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if spec is None or not tf or name not in NCU_KERNEL or not GOVERNING_OK:
        return None
    try:
        k = json.load(open(tf[-1]))["kernels"][NCU_KERNEL[name]]
        units = float(k[spec[1]])
        mb = json.load(open(sorted(glob.glob(os.path.join(ROOT, "profiles", spec[2])))[-1]))
        if spec[0] == "l2_reduction_issue":
            peak = max(r["g_lane_red_per_s"] for r in mb["rows"] if r["kind"] == "v2f32" and r["pattern"] == "spread")
        else:
            peak = max(r["spread_g_lane_gathers_per_s"] for r in mb["rows"] if r["table_mb"] <= 34)
        ach = units / (per_launch_ms * 1e-3) / 1e9
        return {"bound": spec[0], "achieved": ach, "peak": peak, "unit": spec[3], "frac": ach / peak, "units_per_launch": units,
                "units_source": os.path.basename(tf[-1]), "peak_source": "microbenchmark, profiles/" + spec[2].replace("*", "rNN")}
    except Exception:  # noqa: BLE001
        return None


def unit_count(name, ints):
    """number of samples (units) a traced call processed, from its integer arguments."""
    pos = {"f2b_field_fwd": 3, "f2b_hash_fwd": 3, "f2b_hash_bwd": 3, "f2b_mlp_fwd": 1, "f2b_mlp_bwd": 1, "f2b_shader_prep": 0,
           "f2b_shader_act": 0, "f2b_shader_act_bwd": 0, "f2b_shader_prep_bwd": 0, "f2b_cast_f16_to_f32": 0,
           "f2b_cast_f32_to_f16": 0, "f2b_table_to_half": 0}
    if name in pos and len(ints) > pos[name]:
        return ints[pos[name]]
    return None


DUMP_CAP = 1 << 21        # elements kept of one dumped array (a dump of any config stays far below 64 MB)


def step_outputs(prob, loss, res):
    """What a caller of the timed path receives from one step, as host arrays (float32; integer outputs as float64): the loss,
    the RenderResult fields and the parameter gradients.  An array of more than DUMP_CAP elements is flattened and replaced by a
    fixed sample of DUMP_CAP of them (sorted indices from seed 0, a function of its size only), e.g. the 64 MB table gradient."""
    import torch
    field, shader, r = prob["field"], prob["shader"], prob["renderer"]
    arrays = {"loss": loss.reshape(1), "colors": res.colors, "disparity": res.disparity, "depth": res.depth,
              "first_oct_dis": res.first_oct_dis, "weights": res.weights, "idx_start_end": res.idx_start_end,
              "edge_feats": res.edge_feats, "grad_feat_pool": field.feat_pool_.grad, "grad_field_mlp": field.mlp_.params_.grad,
              "grad_shader_mlp": shader.mlp_.params_.grad, "grad_app_emb": r.app_emb_.grad}
    out = {}
    for name, t in arrays.items():
        if t is None:
            continue
        t = t.detach()
        if t.numel() > DUMP_CAP:
            idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), DUMP_CAP))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        out[name] = a.astype(np.float64 if a.dtype.kind in "iu" else np.float32)
    return out


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise RuntimeError(f"--dump-outputs: {total} bytes, over the 64 MB a dump may take")
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    print(f"bench.py: wrote {len(arrays)} arrays ({total / 1e6:.1f} MB) to {path}", file=sys.stderr)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from f2nerf_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist_sync = None
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
        from f2nerf_b200.dist import allreduce_step
        dist_sync = allreduce_step
    global GOVERNING_OK
    GOVERNING_OK = args.config == "wanjinyou" and not args.rays   # the sector counts in profiles/*_traffic.json are this batch's
    prob = build_problem(rank, world, args, device)
    n_rays = prob["n_rays"]                                     # rays THIS rank renders per step
    if world > 1:
        from f2nerf_b200.dist import install_grad_overlap, install_vote_sync
        install_vote_sync(prob["sampler"])
        # F2B_DP_OVERLAP=1: table-gradient all-reduce per level slab behind a per-slab scatter (dist.install_grad_overlap).  Measured
        # on B200 (profiles/r02f_*, r02g_*): the four per-slab scatter launches cost +0.17 ms against the single 16-level launch,
        # more than the overlapped all-reduce saves at N = 2 and 4 (4.64 / 4.73 vs 4.48 / 4.64 ms) — so the default is ONE
        # all-reduce of the live 34 MB behind the single scatter launch.
        if os.environ.get("F2B_DP_OVERLAP", "0") == "1":
            install_grad_overlap(prob["renderer"])
    o, d, cam, gt = prob["host"]
    pin = lambda a: torch.from_numpy(a).pin_memory()
    h_o, h_d, h_cam, h_gt = pin(o), pin(d), pin(cam), pin(gt)
    d_o, d_d, d_cam, d_gt = (x.to(device) for x in (h_o, h_d, h_cam, h_gt))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value): K steps bracketed by barrier + synchronize, CUDA events --------
    clocks = ClockSampler(local if rank == 0 else -1)   # rank 0 reports the clocks: only it polls (a poll on any rank stalls the
                                                 # whole job through the next collective); polling starts before the warm-up: the first NVML queries of a
    clocks.start()                               # process stall kernel submission for 100s of ms on this driver
    nxt = (d_o, d_d) if args.pipeline_march else None           # the same resident batch every step: the next rays are these
    for _ in range(args.warmup):                 # same object lifetimes as the timed loop (the caching allocator must have
        loss, res = train_step(prob, d_o, d_d, d_cam, d_gt, dist_sync, nxt)   # seen the steady-state peak before timing starts)
    barrier()
    clocks.rows.clear()                          # keep only samples taken under the timed regions
    def timed_loop(capture):
        import gc
        gc.collect()
        gc.disable()                              # like timeit: no cyclic-GC pause inside the timed region
        try:
            return _timed_loop(capture)
        finally:
            gc.enable()

    def _timed_loop(capture):
        barrier()
        l0 = _lib.LAUNCHES
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        ns = nk = 0
        w = []
        for _ in range(args.steps):
            w0 = time.perf_counter()
            loss, res = train_step(prob, d_o, d_d, d_cam, d_gt, dist_sync, nxt)
            ns += prob["renderer"].n_sampled_pts_
            nk += res.weights.shape[0]
            w.append(round((time.perf_counter() - w0) * 1e3, 2))
        eb.record()
        barrier()
        out = step_outputs(prob, loss, res) if capture else None      # outside the timed window, before another step runs
        return ea.elapsed_time(eb), w, ns, nk, _lib.LAUNCHES - l0, out

    # A step whose host wall time is far off the median (seen on fresh boxes: one NVML poll of the clock sampler
    # holding the driver lock for ~40 ms while the main thread launches) makes the whole K-step number a
    # measurement of that stall: such a run is rejected and the K steps are timed ONCE more; both are reported.
    def stalled(w):
        """A host-stall outlier on ANY rank (ranks must take the same branch: the verdict is all-reduced)."""
        med = sorted(w)[len(w) // 2]
        bad = max(w[1:] or w) > 1.5 * med and max(w[1:] or w) - med > 2.5
        if world > 1:
            t = torch.tensor([1.0 if bad else 0.0], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            bad = bool(t.item() > 0)
        return bool(bad)

    attempts, best = [], None
    for i in range(4):                            # at most three re-measurements, every attempt disclosed in `timing_attempts`
        # the dump is the first pass's last step: its inputs (RNG position, octree votes so far) depend on the arguments only
        res = timed_loop(capture=bool(args.dump_outputs) and rank == 0 and i == 0)
        if i == 0:
            dumped = res[5]
        outlier = stalled(res[1])
        attempts.append({"ms_per_step": res[0] / args.steps, "host_wall_ms_per_step": res[1], "rejected": bool(outlier)})
        if not outlier:
            best = res
            break
        if best is None or res[0] < best[0]:
            best = res                            # every attempt stalled: the least disturbed one stands, flagged as rejected
    ms, walls, n_samples, n_kept, launches, _ = best
    # ---- per-kernel CUDA-event trace over the same steps (separate loop: event pairs around every C-ABI call) --
    _lib.TRACE = []
    for _ in range(args.steps):
        train_step(prob, d_o, d_d, d_cam, d_gt, dist_sync, nxt)
    barrier()
    trace, _lib.TRACE = _lib.TRACE, None
    # ---- end-to-end timing: pinned host rays -> device, loss -> host, every step ----------------
    barrier()
    up = lambda: (h_o.to(device, non_blocking=True), h_d.to(device, non_blocking=True))
    prob["renderer"].pts_sampler_.take_prefetched(d_o, d_d)       # drop the resident loop's pending prefetch
    ro, rd = up()                                                 # pipeline fill (outside the timed region, like the warm-up)
    def e2e_loop(ro, rd):
        barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        w = []
        for _ in range(args.steps):                               # per step: ONE upload of a ray batch (the next step's when the march
            w0 = time.perf_counter()                              # is pipelined), cam + gt of this step, the loss back to the host
            rc, rg = h_cam.to(device, non_blocking=True), h_gt.to(device, non_blocking=True)
            if args.pipeline_march:
                box = []
                loss, res = train_step(prob, ro, rd, rc, rg, dist_sync, lambda: box.append(up()) or box[0])
                ro, rd = box[0]
            else:
                loss, res = train_step(prob, ro, rd, rc, rg, dist_sync)
                ro, rd = up()
            loss_host = float(loss.item())
            w.append(round((time.perf_counter() - w0) * 1e3, 2))
        e3.record()
        barrier()
        return e2.elapsed_time(e3), w, ro, rd

    e2e_attempts, best_e2e = [], None
    for _ in range(4):                                            # same host-stall rule as the resident loop
        t_e2e, e2e_walls, ro, rd = e2e_loop(ro, rd)
        outlier = stalled(e2e_walls)
        e2e_attempts.append({"ms_per_step": t_e2e / args.steps, "host_wall_ms_per_step": e2e_walls, "rejected": bool(outlier)})
        if not outlier:
            best_e2e = t_e2e
            break
        best_e2e = t_e2e if best_e2e is None else min(best_e2e, t_e2e)
    ms_e2e = best_e2e
    clocks.stop_flag = True
    clocks.join(timeout=2)
    clocks_note = "polled every 0.3 s from before the warm-up; rows kept from the first timed step on"
    need = torch.tensor([1.0 if (rank == 0 and not clocks.rows) else 0.0], device=device)
    if world > 1:
        dist.broadcast(need, src=0)               # every rank takes the same branch (the extra steps contain collectives)
    if float(need.item()) > 0:                    # a very short run: no poll landed in the timed regions — take one now, under the same load
        for _ in range(3):
            train_step(prob, d_o, d_d, d_cam, d_gt, dist_sync, nxt)
        clocks.poll()                             # (rank 0) the GPU is still working through the steps just queued
        clocks_note = "no poll landed inside the (short) timed regions: one sample taken right behind them under the same load"
        barrier()
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
        cnt = torch.tensor([n_samples, n_kept], device=device, dtype=torch.float64)
        dist.all_reduce(cnt)
        n_samples, n_kept = float(cnt[0]), float(cnt[1])
    # ---- per-kernel breakdown from the traced events --------------------------------------------
    agg = {}
    for name, a, b, ints in trace:
        u = unit_count(name, ints)
        rec = agg.setdefault(name, dict(ms=0.0, calls=0, units=0))
        rec["ms"] += a.elapsed_time(b); rec["calls"] += 1; rec["units"] += (u or 0)
    peaks = load_peaks()
    total_traced = sum(v["ms"] for v in agg.values())
    # dominant kernel ON THE STEP'S CRITICAL PATH: with the march software-pipelined it runs for the NEXT batch on a side stream
    # behind this step's backward (Renderer.prefetch_next); it is listed in `rooflines` below but it is not what the step waits for
    hidden = {"f2b_sampler_march"} if args.pipeline_march else set()
    top = max(((k, v) for k, v in agg.items() if k not in hidden), key=lambda kv: kv[1]["ms"])
    name, rec = top
    per_launch_ms = rec["ms"] / rec["calls"]
    if name in ("f2b_mlp_fwd", "f2b_mlp_bwd"):
        flops = {"f2b_mlp_fwd": 2 * 3072, "f2b_mlp_bwd": 4 * 3072}[name] * (rec["units"] / rec["calls"])
        roof = dict(bound="tensor", achieved=flops / (per_launch_ms * 1e-3) / 1e12, peak=peaks["tf"], unit="TFLOP/s")
    else:
        units = rec["units"] / rec["calls"] if rec["units"] else n_samples / args.steps / max(world, 1)
        byts = ALGO_BYTES.get(name, 0) * units
        roof = dict(bound="hbm", achieved=byts / (per_launch_ms * 1e-3) / 1e9, peak=peaks["hbm"], unit="GB/s")
    roof.update(frac=roof["achieved"] / roof["peak"], traffic=ncu_traffic(name), kernel=name, ms_per_launch=per_launch_ms,
                share_of_step=rec["ms"] / max(total_traced, 1e-9), peak_source=peaks["src"],
                governing=governing_roofline(name, rec["ms"] / args.steps))   # per STEP: the capture's units are the large launch
                                                                               # (ray samples; the 16 k TV edge points add 0.5 %)
    rooflines = []                                                  # the same two figures for the six largest kernels
    for kname, krec in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])[:6]:
        k_ms = krec["ms"] / krec["calls"]
        k_units = krec["units"] / krec["calls"] if krec["units"] else n_samples / args.steps / max(world, 1)
        hbm = ALGO_BYTES.get(kname, 0) * k_units / (k_ms * 1e-3) / 1e9 if kname in ALGO_BYTES else None
        rooflines.append({"kernel": kname, "ms_per_launch": k_ms, "off_critical_path": kname in hidden,
                          "hbm_frac_algorithmic": None if hbm is None else hbm / peaks["hbm"],
                          "governing": governing_roofline(kname, krec["ms"] / args.steps)})
    rays_total = n_rays * world * args.steps
    cfg = prob["cfg"]
    line = {
        "metric": "training rays/sec", "value": rays_total / (ms * 1e-3), "unit": "rays/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32 march/composite, f16 hash table + MLP operands (f32 accumulate)",
        "data": "synthetic", "samples_per_sec": n_samples / (ms * 1e-3),
        "config": config_dict(args, world),
        "workload_measured": {"samples_per_ray": n_samples / args.steps / world / n_rays, "kept_per_ray": n_kept / args.steps / world / n_rays,
                              "mlp_impl": int(_lib.lib.f2b_get_mlp_impl())},
        "e2e": {"value": rays_total / (ms_e2e * 1e-3), "unit": "rays/s",
                "h2d_bytes_per_step": int(sum(x.numel() * x.element_size() for x in (h_o, h_d, h_cam, h_gt))) * world,
                "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps, "timing_attempts": e2e_attempts},
        "gpu_launches": int(launches),
        "host_wall_ms_per_step": walls, "timing_attempts": attempts,
        "clocks": dict(clocks.summary(), note=clocks_note) if rank == 0 else None,
        "roofline": roof, "rooflines": rooflines,
        "kernels": {k: {"ms_per_step": v["ms"] / args.steps, "calls_per_step": v["calls"] / args.steps} for k, v in
                    sorted(agg.items(), key=lambda kv: -kv[1]["ms"])},
    }
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_port(args, budget_s=20.0)
        if world == 1:
            line["optimizer_step"] = optimizer_timing(prob)
            line["forward_only"] = forward_only_timing(prob, d_o, d_d, args)
            if prob["ray_gen"] is not None:
                line["ray_generation"] = ray_generation_timing(prob, args)
        ref_gpu = reference_gpu_timing(args)
        if ref_gpu is not None:
            line["reference_gpu"] = ref_gpu
        cpp = cpp_host_timing(args)
        if cpp is not None:
            line["cpp_host"] = cpp
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def forward_only_timing(prob, d_o, d_d, args, iters=20):
    """Forward-only rays/s (SURVEY 8d; the path ExpRunner::RenderWholeImage drives, ExpRunner.cpp:257-293): VALIDATE mode
    (noise == 1, bg 0.5, no octree votes / edge samples), no autograd, same ray batch as the headline."""
    import torch
    from f2nerf_b200 import TRAIN, VALIDATE
    gdp, r = prob["gdp"], prob["renderer"]
    gdp.mode_ = VALIDATE
    try:
        with torch.no_grad():
            for _ in range(3):
                r.Render(d_o, d_d, None, None)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                r.Render(d_o, d_d, None, None)
            e1.record()
            torch.cuda.synchronize()
    finally:
        gdp.mode_ = TRAIN
    ms = e0.elapsed_time(e1) / iters
    out = {"value": prob["n_rays"] / (ms * 1e-3), "unit": "rays/s", "ms_per_step": ms, "mode": "VALIDATE, no_grad",
           "note": "the reference's number is reference_gpu.ms_validate_median on the same ray count"}
    # the evaluation loop itself (ExpRunner::RenderWholeImage, ExpRunner.cpp:257-293): 8 x the batch as one "image", the
    # reference's 8192-ray chunks, results to the host — chunks alternate between two streams (f2nerf_b200/eval.py)
    from f2nerf_b200 import RenderWholeImage
    big_o, big_d = d_o.repeat(8, 1), d_d.repeat(8, 1)
    for _ in range(2):
        RenderWholeImage(r, big_o, big_d)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        RenderWholeImage(r, big_o, big_d)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / 5
    out["whole_image"] = {"rays": int(big_o.shape[0]), "ms_per_image": wall * 1e3, "rays_per_s": big_o.shape[0] / wall,
                          "note": "host wall time incl. the final device->host copy of the three images"}
    return out


def ray_generation_timing(prob, args, iters=20):
    """SURVEY 8f N3 (reported separately): one training batch of rays + ground-truth colours.  `ours` =
    RayGenerator.RandRaysData (CPU index draws, ONE 48 KB H2D copy, two kernels on HBM-resident images);
    `reference_style` = the same draws followed by what Dataset::RandRaysData does (Dataset.cpp:287-296): CPU gather from
    a CPU image tensor, three H2D copies, ray kernel.  ngp_fox geometry: 50 images of 960 x 540."""
    import torch
    from f2nerf_b200 import RayGenerator
    src = prob["ray_gen"]                                        # the reference's ngp_fox cameras (fixture)
    n_img, H, Wd = src.n_images_, src.height_, src.width_
    g = torch.Generator().manual_seed(0)
    images = torch.rand((n_img, H, Wd, 3), generator=g)
    gen = RayGenerator(src.poses_, src.intri_, src.dist_params_, src.bounds_, images=images, train_set=src.train_set_)
    n_b = prob["n_rays"]
    dev = gen.poses_.device
    flat = images.view(-1, 3)

    def ours():
        gen.RandRaysData(n_b)

    def ref_style():
        cam = torch.randint(n_img, (n_b,), dtype=torch.int64)
        i = torch.randint(0, H, (n_b,), dtype=torch.int64)
        j = torch.randint(0, Wd, (n_b,), dtype=torch.int64)
        ij = torch.stack([i, j], -1).to(dev).contiguous()
        gt = flat[cam * H * Wd + i * Wd + j].to(dev).contiguous()
        cam_d = cam.to(dev)
        gen.Img2WorldRayFlex(cam_d.to(torch.int32), ij.to(torch.int32))
        return gt, gen.bounds_[cam_d].contiguous()

    out = {}
    for name, fn in (("ours_ms", ours), ("reference_style_ms", ref_style)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
        out[name] = (time.perf_counter() - t0) / iters * 1e3
    out["note"] = "host wall time per 4096-ray batch incl. the CPU index draws; images 50x960x540x3 fp32"
    return out


def optimizer_timing(prob, iters=20):
    """SURVEY 8f N1, reported separately from the headline (the metric excludes the optimizer step): the hash
    table's Adam update as the reference runs it (torch::optim::Adam's ATen sequence, ExpRunner.cpp:136, plus the
    fp32->fp16 table copy the next forward makes) vs f2b_adam_step (one pass over the live prefix + fp16 shadow)."""
    import torch
    from f2nerf_b200 import FusedAdam, ops
    field = prob["field"]
    p = field.feat_pool_
    g = p.grad if p.grad is not None else torch.zeros_like(p)
    pa, m, v = p.detach().clone(), torch.zeros_like(p), torch.zeros_like(p)

    def aten(step):
        bc1, bc2 = 1 - 0.9 ** step, 1 - 0.99 ** step
        m.mul_(0.9).add_(g, alpha=0.1)
        v.mul_(0.99).addcmul_(g, g, value=0.01)
        pa.addcdiv_(m, (v.sqrt() / (bc2 ** 0.5)).add_(1e-15), value=-(1e-2 / bc1))
        ops.table_to_half(pa)

    saved = p.detach().clone()
    opt = FusedAdam([dict(params=[p], lr=1e-2, betas=(0.9, 0.99), eps=1e-15)], table_field=field)
    out = {}
    for name, fn in (("aten_sequence_ms", aten), ("fused_ms", lambda step: opt.step())):
        for i in range(3):
            fn(i + 1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i + 4)
        e1.record()
        torch.cuda.synchronize()
        out[name] = e0.elapsed_time(e1) / iters
    p.data.copy_(saved)                                            # leave the problem as it was
    field.manage_shadow(False)
    out.update(elements=int(p.numel()), live_elements=int(17 * field.local_size_),
               note="hash-table group only; ATen side includes the fp16 table copy of the next forward")
    return out


def cpp_host_timing(args):
    """Informational, N=1 only: the SAME harness (oracle/ref_driver.cpp: the reference's own program — Dataset, factories, autograd,
    loss — 20 timed Render + loss.backward() on the seeded batch) with Renderer::Render replaced by the C++/LibTorch host of this
    library (f2nerf_b200/shim/B200Renderer.cpp -> oracle/_ref/ref_driver_b200): the number a maintainer gets after the drop-in,
    no Python anywhere."""
    drv = os.path.join(ROOT, "oracle", "_ref", "ref_driver_b200")
    cfg = W.CONFIGS[args.config]
    if args.no_ref_gpu or int(os.environ.get("WORLD_SIZE", "1")) > 1 or cfg["ref_yaml"] is None or not os.path.exists(drv):
        return None
    try:
        out_dir = "/tmp/f2b_cpp_bench"
        r = subprocess.run([drv, os.path.join(ROOT, cfg["ref_yaml"]), out_dir, str(args.rays or cfg["rays"]), "20"],
                           cwd=ROOT, capture_output=True, text=True, timeout=900)
        if r.returncode != 0:
            return {"unavailable": ("ref_driver_b200 rc %d: " % r.returncode) + r.stderr[-160:]}
        t = json.load(open(os.path.join(out_dir, "ref_timing.json")))
        t["note"] = "the reference's program with the B200 C++ host linked in as Renderer::Render (no march pipelining in this harness)"
        return t
    except Exception as e:  # noqa: BLE001
        return {"unavailable": str(e)[:200]}


def reference_gpu_timing(args):
    """Informational, N=1 only: the compiled, unmodified reference (oracle/_ref/ref_driver, built by build() from
    /root/reference) timed on the same box, same config YAML, same ngp_fox scene, same seeded ray batch (seed 2023) and
    parameter state as the product arm.  CUDA events around its own Renderer::Render + loss.backward(), median of 20."""
    drv = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
    cfg = W.CONFIGS[args.config]
    if args.no_ref_gpu or int(os.environ.get("WORLD_SIZE", "1")) > 1:
        return None
    if cfg["ref_yaml"] is None:
        return {"unavailable": "synthetic scene: the reference builds its octree from a dataset"}
    if not os.path.exists(drv):
        return {"unavailable": "oracle/_ref/ref_driver not built (build() makes it when /root/reference is present)"}
    try:
        out_dir = "/tmp/f2b_ref_bench"
        r = subprocess.run([drv, os.path.join(ROOT, cfg["ref_yaml"]), out_dir, str(args.rays or cfg["rays"]), "20"],
                           cwd=ROOT, capture_output=True, text=True, timeout=900)
        if r.returncode != 0:
            return {"unavailable": ("ref_driver rc %d: " % r.returncode) + r.stderr[-160:]}
        t = json.load(open(os.path.join(out_dir, "ref_timing.json")))
        t["config_yaml"] = cfg["ref_yaml"]
        t["note"] = "unmodified Totoro97/f2-nerf + tiny-cuda-nn compiled for sm_100a; same scene / rays / parameters as the product arm"
        return t
    except Exception as e:  # noqa: BLE001
        return {"unavailable": str(e)[:200]}


class CpuPort:
    """The CPU restatement (oracle/) of the same step on the same config: same octree blobs, same parameter state, the
    same seeded ray batch (rays through the oracle's restatement of Img2WorldRayKernel).  Loads no product code."""

    def __init__(self, args):
        import oracle_lib as O
        self.O, self.args = O, args
        cfg = self.cfg = W.CONFIGS[args.config]
        sb = W.scene_blobs(args.config)
        V = sb["trans"].size // 544
        par = W.init_params(args.config, V, sb["n_images"], sb["prim"], sb["bias"])
        self.sc = dict(nodes=sb["nodes"], trans=sb["trans"], edges=sb["edges"], near=cfg["near"], sample_l=cfg["sample_l"],
                       scale_by_dis=cfg["scale_by_dis"], max_hits=1024)
        local = (((1 << cfg["log2_table"]) * 16 // 16) >> 4) << 4
        self.fld = dict(table16=par["table"].astype(np.float16), prim=par["prim"], bias=par["bias"], V=V, local_size=local,
                        mlp_params=par["field_mlp"])
        self.sp, self.emb = par["shader_mlp"], (par["app_emb"] if cfg["use_app_emb"] else None)
        self.rays = args.rays or cfg["rays"]
        o, d, cam = W.host_rays(args.config, self.rays, 2023 if sb["synthetic"] is None else 1234)
        self.o, self.cam = o, cam
        self.dn = (d / np.linalg.norm(d, axis=-1, keepdims=True)).astype(np.float32)
        self.rng = np.random.default_rng(0)
        self.gt = self.rng.random((self.rays, 3), dtype=np.float32)
        self.n_edges = sb["edges"].size // 64

    def step(self, n):
        import oracle_pipeline as OP
        rng = self.rng
        noise = (rng.random(1024 + n + 10, dtype=np.float32) + .5).astype(np.float32)
        bg = rng.random((n, 3), dtype=np.float32)
        edge = (rng.integers(0, self.n_edges, 8192).astype(np.int32), (rng.random((8192, 2), dtype=np.float32) * 2 - 1))
        t0 = time.time()
        OP.render_train(self.sc, self.o[:n], self.dn[:n], noise, bg, self.fld, self.sp, self.emb,
                        self.cam[:n] if self.emb is not None else None, edge, self.gt[:n])
        return time.time() - t0

    def size_for(self, budget_s, n0=32):
        """largest power-of-two ray count (<= the batch) whose step fits ``budget_s``; returns (n, seconds of the probe)."""
        n, t = n0, self.step(n0)
        while t < budget_s / 2 and n < self.rays:
            n = min(n * 2, self.rays)
            t = self.step(n)
        return n, t


def cpu_port(args, budget_s=20.0):
    import oracle_lib as O
    port = CpuPort(args)
    n, t = port.size_for(budget_s / 2)
    return {"value": n / t, "unit": "rays/s", "cores": O.num_threads(), "kind": "port",
            "sample": f"{n} of the {port.rays} rays of the same batch (all stages incl. backward), {t:.1f} s wall; "
                      "all stages OpenMP-parallel (oracle/f2_oracle.c)"}


def run_reference(args):
    """--impl reference: the reference has no CPU path (src/Common.h:9-13 hard-codes CUDA tensors; tiny-cuda-nn is CUDA-only)
    and is a C++/CUDA executable, not a pip package: this arm times the CPU port of its algorithm (oracle/) with all host
    threads on the product arm's config; every step is a bounded sample (the first n rays of the same seeded batch), n chosen
    so that the K + W steps end within ~2 minutes.  Imports nothing from the product package."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if "F2B_REF_THREADS" in os.environ or os.environ.get("OMP_NUM_THREADS") == "1":
        # torchrun pins OMP_NUM_THREADS=1 for its workers; the CPU arm is meant to use every host thread it can
        os.environ["OMP_NUM_THREADS"] = os.environ.get("F2B_REF_THREADS", str(os.cpu_count()))
    import oracle_lib as O
    port = CpuPort(args)
    n, _ = port.size_for(120.0 / max(args.steps + args.warmup, 1)) if not args.ref_rays else (min(args.ref_rays, port.rays), 0)
    for _ in range(args.warmup):
        port.step(n)
    t0 = time.time()
    for _ in range(args.steps):
        port.step(n)
    dt = time.time() - t0
    v = n * args.steps / dt
    world = int(os.environ.get("WORLD_SIZE", "1"))
    print(json.dumps({
        "impl": "reference", "metric": "training rays/sec", "value": v, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": W.CONFIGS[args.config]["scaling"], "vs_baseline": None, "dtype": "f32 (CPU port, fp16 table / MLP operands)",
        "data": "synthetic", "config": config_dict(args, world),
        "cpu_baseline": {"value": v, "unit": "rays/s", "cores": O.num_threads(), "kind": "port",
                         "sample": f"each step = the first {n} of the {port.rays} rays of the product arm's seeded batch x <=1024 samples, "
                                   "all stages incl. backward"},
        "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="wanjinyou", choices=sorted(W.CONFIGS))
    ap.add_argument("--rays", type=int, default=0, help="override the config's ray count (global for strong-scaling configs)")
    ap.add_argument("--ref-rays", dest="ref_rays", type=int, default=0, help="--impl reference: rays per step (0 = sized to ~2 min total)")
    ap.add_argument("--no-pipeline-march", dest="pipeline_march", action="store_false",
                    help="march every batch at the start of its own Render (default: the next batch's march runs behind this step's backward)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last step of the first timed pass returned (loss, render outputs, parameter gradients) "
                         "as DIR/<name>.npy; rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
