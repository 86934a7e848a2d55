#!/usr/bin/env python
"""bench.py -- stereo pairs rendered + TSDF-fused per second (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C1] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One STEP = one stereo pair of the synthetic scene: render the left and the right view
(forward rasterizer x2, float->u8 frames), then fuse the left view's depth + colour into the
TSDF volume.  With N > 1 GPUs the N*K views are sharded round-robin over the ranks (weak scaling:
K pairs per rank) and the timed region ends with the single NCCL sum-reduce of the volume.

`value`  : pairs/s with everything resident in HBM (Gaussians, camera table, volume).
`e2e`    : same metric through the public classes with HOST buffers: Renderer.render_image_pair()
           copies both uint8 frames and the left depth to pinned host memory, TSDF.integrate() takes
           host depth + host rgb and uploads them -- every step.
`--impl reference`: the reference's own implementation of the path on this box: the UNMODIFIED
           reference rasterizer built for sm_100a (oracle/_ref) called the way
           renderer_utils.py:378-390 calls it (float frame D2H, x255 -> uint8 on the host) and the
           Open3D-0.17-equivalent CPU TSDF (oracle port, all host threads).  PNG encoding and the
           stereo network are left out (both would only slow the reference arm down).
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step handed its caller as DIR/<name>.npy
           (float32 / float64, see dump_outputs), so that two builds can be compared output for output on the same
           seeded inputs.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "stereo_pairs_per_sec_rendered_and_tsdf_fused"
MERGE_DST = None if os.environ.get("BENCH_MERGE", "reduce") == "allreduce" else 0  # A/B: ncclReduce to rank 0 | ncclAllReduce
UNIT = "stereo-pairs/s"


class BenchArgs:
    """Reference defaults of the flags the hot path reads (argument_utils.py:29-42,74-90)."""

    GS_white_background = False
    TSDF_scale = 1.0
    TSDF_sdf_trunc = 0.04
    TSDF_dilate = 1
    TSDF_valid = None
    TSDF_skip = None
    TSDF_use_mask = False
    TSDF_use_occlusion_mask = False

    def __init__(self, cfg):
        self.TSDF_voxel = 2.0 * 512 / cfg["tsdf_res"]  # voxel_length = TSDF_voxel/512 = 2/tsdf_res
        self.TSDF_min_depth_baselines = cfg["min_db"]
        self.TSDF_max_depth_baselines = cfg["max_db"]
        self.TSDF_sdf_trunc = max(0.04, 3 * 2.0 / cfg["tsdf_res"])


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            v = json.load(f).get("hbm_gbs")
        if v:
            return float(v), "measured"
    except Exception:
        pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix="gsb_clocks_", suffix=".csv")
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1]))
                    mx.append(float(c[2]))
                except ValueError:
                    continue
                for k, name in enumerate(names):
                    if c[5 + k].lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def setup_dist(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    if n_gpus != world:
        if rank == 0:
            print(f"[bench] --gpus {n_gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    return rank, local, world


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def build_scene(cfg, total_views, seed=1):
    from gs2mesh_b200 import scene

    cloud = scene.make_gaussians(cfg["num_points"], seed=seed)
    rigs, baseline = scene.make_stereo_cameras(total_views, cfg["width"], cfg["height"], layout=cfg["layout"],
                                               principal_point=cfg.get("principal_point"))
    return cloud, rigs, baseline


def shared_config(args, cfg, total_views, world, pairs_per_rank):
    """`config` is identical in the `ours` and the `reference` line of one (N, K, W) run; arm-specific facts go to `details`."""
    return {"workload": workload_name(args.config, cfg, total_views), "pairs_per_rank": pairs_per_rank,
            "sharding": f"views round-robin x{world}", "scaling": args.scaling}


def workload_name(name, cfg, total_views):
    return (f"{name}: synthetic {cfg['num_points']}-Gaussian {'360' if cfg['layout'] == 'ring' else 'frontal-cap'} scene, "
            f"{total_views} stereo pairs @{cfg['width']}x{cfg['height']}, {cfg['tsdf_res']}^3 TSDF lattice (voxel 2/{cfg['tsdf_res']})")


# ------------------------------------------------------------------------------------------------ ours
DEFAULT_E2E_ORDER = "lagged"
DUMP_MAX_VALUES = 1 << 20  # per dumped array (4 MB as float32): the ten arrays stay well under 64 MB together


def _dump_values(t):
    """Device tensor -> float32 host array; above DUMP_MAX_VALUES values, the same seeded sample of positions on every run."""
    flat = t.reshape(-1)
    if flat.numel() <= DUMP_MAX_VALUES:
        return t.float().cpu().numpy()
    pick = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_MAX_VALUES, replace=False))
    return flat[torch.from_numpy(pick).to(flat.device)].float().cpu().numpy()


def dump_outputs(out_dir, out, vol):
    """What the last timed step handed its caller: the pair's float and uint8 frames, the left view's depth and
    transmittance, and the TSDF volume after its fusion.  Bricks are listed in lattice-index order (pool slots depend on
    the order in which blocks opened them): volume_brick_index [n,3] (float64) and the bricks' tsdf / weight / colour."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: _dump_values(out[k]) for k in ("left", "right", "left_u8", "right_u8", "depth", "final_T")}
    index = vol.brick_indices().cpu().numpy()
    order = np.lexsort(index.T[::-1])
    slots = torch.from_numpy(order).to(vol.device)
    arrays["volume_brick_index"] = index[order].astype(np.float64)
    bricks = vol.pool()[slots]
    arrays["volume_tsdf"] = _dump_values(bricks[..., 0])
    arrays["volume_weight"] = _dump_values(bricks[..., 1])
    if vol.color is not None:
        arrays["volume_color"] = _dump_values(vol.color.view(vol.pool_bricks, -1, 4)[slots][..., :3])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_ours(args, cfg, rank, local, world):
    from gs2mesh_b200 import _lib
    from gs2mesh_b200.renderer import Renderer
    from gs2mesh_b200.tsdf import TSDF, shard_views

    Wm = args.warmup
    if args.scaling == "strong":  # total work fixed: --steps pairs split over the ranks (round-robin)
        total_views = args.steps
        K = len(range(rank, total_views, world))
    else:
        K = args.steps
        total_views = K * world
    cloud, rigs, baseline = build_scene(cfg, total_views)
    bargs = BenchArgs(cfg)
    dev = f"cuda:{local}"
    renderer = Renderer.from_scene(rigs, baseline, cloud, output_dir_root=None, args=bargs, device=dev)
    # the caller's stream (TSDF fusion, the e2e copies) gets a higher priority than the renderer's side streams: with
    # several views in flight its short kernels and copies are otherwise queued behind thousands of blend CTAs
    if os.environ.get("BENCH_MAIN_PRIORITY", "-1") != "0":
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=int(os.environ.get("BENCH_MAIN_PRIORITY", "-1"))))
    renderer.prepare_renderer()
    stage = TSDF(renderer, None, bargs, "bench", window_resolution=cfg["tsdf_res"], device=dev)
    stage.volume = stage._make_volume()
    vol = stage.volume
    mine = shard_views(total_views, rank, world)
    assert len(mine) == K
    W, H = cfg["width"], cfg["height"]

    def step(i):
        out = renderer.render_image_pair(i, to_host=False)
        stage.integrate(out["depth"], out["left_u8"], rigs[i]["left"], final_T=out["final_T"])
        return out

    # ---- calibration (untimed): per-view workload statistics for the roofline formulas
    stats = dict(Pv=[], R=[], R_ref=[], bricks=[], V_upd=[])
    for i in mine[:3]:
        o = renderer.render_view(i, 0, want_depth=True, want_counts=True)
        rr = renderer.render_view(i, 0, want_counts=True)
        cnt = o["counts"].cpu().numpy()
        stats["R"].append(int(cnt[0]))
        stats["R_ref"].append(int(cnt[1]))
        from gs2mesh_b200 import rasterizer as rast

        rad = rast.rasterize_forward(means3D=renderer.means3D, opacities=renderer.opacity, viewmatrix=renderer._camera_table[i, 0, 0:16],
                                     projmatrix=renderer._camera_table[i, 0, 16:32], campos=renderer._camera_table[i, 0, 32:35],
                                     bg=renderer.background, width=W, height=H, tan_fovx=renderer._views[i][0].tan_fovx,
                                     tan_fovy=renderer._views[i][0].tan_fovy, shs=renderer.shs, scales=renderer.scales,
                                     rotations=renderer.rotations, sh_degree=renderer.sh_degree, want_depth=False, want_final_T=False)["radii"]
        stats["Pv"].append(int((rad > 0).sum().item()))
        del rad, rr
        w_before = float(vol.tsdf_weight.view(-1, 2)[:, 1].sum(dtype=torch.float64).item())
        step(i)
        stats["bricks"].append(vol.last_stats()[0])
        stats["V_upd"].append(float(vol.tsdf_weight.view(-1, 2)[:, 1].sum(dtype=torch.float64).item()) - w_before)
    vol.reset()
    mean = {k: float(np.mean(v)) for k, v in stats.items()}

    # ---- warm-up (incl. one merge, so NCCL's lazy connection set-up is not billed to the timed region)
    for i in (mine * ((Wm // max(len(mine), 1)) + 1))[:Wm]:
        step(i)
    if world > 1:
        vol.reduce_across_ranks(dst=MERGE_DST)
    vol.reset()
    barrier(world)
    _lib.profile_enable(False)

    # ---- timed region: K steps (+ the one volume reduce when sharded)
    sampler = ClockSampler(local)
    launches0 = _lib.lib().gsb_kernel_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    barrier(world)
    ev0.record()
    host_t0 = time.perf_counter()
    last = None
    for i in mine:
        last = step(i)
    host_enqueue_ms = 1e3 * (time.perf_counter() - host_t0) / max(K, 1)  # host time to ENQUEUE a step (no waiting)
    evr = torch.cuda.Event(enable_timing=True)
    evr.record()
    if world > 1:
        vol.reduce_across_ranks(dst=MERGE_DST)
    ev1.record()
    barrier(world)
    reduce_ms = max_over_ranks(evr.elapsed_time(ev1), world)
    pool_after = vol.pool_stats()
    assert pool_after["dropped_total"] == 0, "the brick pool overflowed during the timed region"
    renderer.check_status(mine)  # no asynchronously rendered frame overflowed its scratch
    clocks = sampler.stop()
    launches = int(_lib.lib().gsb_kernel_launch_count() - launches0)
    elapsed_ms = max_over_ranks(ev0.elapsed_time(ev1), world)
    value = total_views / (elapsed_ms / 1e3)
    if args.dump_outputs and rank == 0 and last is not None:
        dump_outputs(args.dump_outputs, last, vol)

    # ---- per-kernel durations: the same steps again with the two eyes serialised on one stream, every
    #      stage bracketed by CUDA events on the launching stream (in the timed loop above the eyes overlap
    #      on two streams, so a bracketed stage would also contain the other eye's kernels)
    vol.reset()
    renderer.overlap_eyes = False
    n_prof = max(1, min(K, 25))
    for i in mine[:2]:
        step(i)
    _lib.profile_collect()
    _lib.profile_enable(True)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for i in mine[:n_prof]:
        step(i)
    pe1.record()
    torch.cuda.synchronize()
    _lib.profile_enable(False)
    prof = _lib.profile_collect()
    serial_ms_per_step = pe0.elapsed_time(pe1) / n_prof
    renderer.overlap_eyes = True
    merge_phases = None
    if world > 1:  # the phases of one more merge of the volume just fused (CUDA events inside gsb_tsdf_reduce, this rank's view)
        _lib.profile_enable(True)
        barrier(world)
        vol.reduce_across_ranks(dst=MERGE_DST)
        torch.cuda.synchronize()
        _lib.profile_enable(False)
        merge_phases = {k: round(ms / max(n, 1), 4) for k, (ms, n) in _lib.profile_collect().items() if k.startswith("merge_") and n}
    prof = {k: v for k, v in prof.items() if not k.startswith("merge_")}

    # ---- e2e: public classes with host buffers, H2D + D2H every step
    vol.reset()
    host_depth = [torch.empty(H, W, dtype=torch.float32).pin_memory() for _ in range(2)]
    dev_depth = [torch.empty(H, W, dtype=torch.float32, device=dev) for _ in range(2)]
    depth_ready = [None, None]
    K_e2e = K
    barrier(world)
    t0 = time.perf_counter()
    # software-pipelined: while the host consumes pair i (waits for its frames in pinned memory, reads the depth back, hands
    # depth + colour to TSDF.integrate, which uploads them), the next `pairs_in_flight` pairs are already being rendered; the
    # depth read-back of pair i is consumed one iteration later, so no step waits for a copy it has just enqueued
    views = mine[:K_e2e]
    lag = max(1, int(renderer.pairs_in_flight))
    pending = [renderer.render_image_pair(v, to_host=True, wait=False) for v in views[:lag]]
    fuse_next = None  # (view, pinned host frame, buffer index) of the pair whose depth is still travelling to the host

    def fuse(item):
        i, rgb_host, k = item
        depth_ready[k].synchronize()  # the float depth of pair i is in pinned host memory
        # what a host-side stereo stage would hand back: float depth + the uint8 left frame, both on the host
        stage.integrate(host_depth[k], rgb_host, rigs[i]["left"])

    # BENCH_E2E_ORDER (A/B switch): "lagged" = pair n-1 is fused at the top of iteration n, right after its depth read-back
    # was enqueued (the host then idles for that copy before it enqueues the next render); "overlap" = the depth read-back of
    # pair n is enqueued, THEN the render of pair n + lag (the host is busy enqueueing while the depth travels), then pair n
    # is fused.  Both respect the renderer's buffer rotation: the tensors of call n are valid until call
    # n + pairs_in_flight + 1 is entered, and pair n is fused after call n + lag = n + pairs_in_flight was.
    order = os.environ.get("BENCH_E2E_ORDER", DEFAULT_E2E_ORDER)
    for n, i in enumerate(views):
        if order == "lagged":
            if fuse_next is not None:  # pair n-1
                fuse(fuse_next)
            out = pending.pop(0)
            if n + lag < len(views):
                pending.append(renderer.render_image_pair(views[n + lag], to_host=True, wait=False))
            out["ready"].synchronize()  # both uint8 frames of pair i are in pinned host memory
        else:
            out = pending.pop(0)
            out["ready"].synchronize()  # both uint8 frames of pair i are in pinned host memory
        k = n & 1
        vol.prepare_depth(out["depth"], W, H, final_T=out["final_T"], out=dev_depth[k])  # expected depth of the left view
        host_depth[k].copy_(dev_depth[k], non_blocking=True)
        depth_ready[k] = torch.cuda.current_stream().record_event()
        fuse_next = (i, out["host_left_u8"], k)
        if order != "lagged":
            if n + lag < len(views):
                pending.append(renderer.render_image_pair(views[n + lag], to_host=True, wait=False))
            fuse(fuse_next)
            fuse_next = None
    if fuse_next is not None:
        fuse(fuse_next)
    renderer.check_status(views)
    if world > 1:
        vol.reduce_across_ranks(dst=MERGE_DST)
    barrier(world)
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    e2e_value = total_views / e2e_s
    h2d = 4 * W * H + 3 * W * H + 16 * 8
    d2h = 2 * 3 * W * H + 4 * W * H

    if rank != 0:
        return None

    # ---- roofline of the dominant kernel
    peak, peak_kind = measured_peak_gbs()
    P = cfg["num_points"]
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    pre_per_step = prof.get("preprocess", (0, 0))[1] / n_prof  # 1 = one fused launch per pair, 2 = one per eye
    eyes_per_pre = 2 if pre_per_step < 1.5 else 1
    bytes_per_launch = {  # algorithmic bytes per launch, SURVEY.md 8(d) / DESIGN.md
        # fused pair launch: parameters read once (SURVEY 8(d): "a fused L/R preprocess may legitimately read params once"),
        # records written per eye
        "preprocess": 12 * P + 224 * mean["Pv"] + eyes_per_pre * (8 * P + 40 * mean["Pv"]),
        "depth_sort": 16 * P + 8 * P,
        "emit": 8 * mean["R"] + 36 * mean["Pv"] + 8 * P,
        "tile_sort": 16 * mean["R"],
        "tile_ranges": 8 * mean["R"] + 8 * tiles,
        "render": 40 * mean["R"] + 16 * W * H,
        "to_u8": 15 * W * H,
        "prepare_depth": 12 * W * H,
        "mark_bricks": 4 * W * H / 16,
        # SURVEY 8(d): (tsdf, weight) and the float4 colour of every UPDATED voxel are read and written, the depth and
        # rgb frames are read once; voxels the frame does not update are never touched
        # SURVEY 8(d) with 3 x f32 colour: 16 + 24 = 40 B per updated voxel (the store pads colour to float4: 48 B move)
        "integrate": 40 * mean["V_upd"] + 7 * W * H,
    }
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        pass
    kernels = {}
    for name, (ms, n) in prof.items():
        if n == 0:
            continue
        avg = ms / n
        gbs = bytes_per_launch[name] / (avg * 1e-3) / 1e9
        kernels[name] = {"avg_ms": round(avg, 5), "launches": n, "launches_per_step": round(n / n_prof, 3),
                         "share": round(ms / (serial_ms_per_step * n_prof), 4),
                         "achieved_gbs": round(gbs, 1), "frac": round(gbs / peak, 4)}
    dom = max(kernels, key=lambda k: kernels[k]["avg_ms"] * kernels[k]["launches"])
    roofline = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "peak_kind": f"of {peak_kind}",
                "unit": "GB/s", "frac": kernels[dom]["frac"], "traffic": traffic.get(dom),
                "algorithmic_bytes_per_launch": int(bytes_per_launch[dom]), "avg_ms": kernels[dom]["avg_ms"]}
    if dom == "render":
        # what ncu shows for this kernel (profiles/r02k_ncu_full_summary.txt): the records are L1/L2-resident and the
        # kernel is limited by instruction issue, so the HBM fraction above is a lower bound on its quality, not its limiter
        roofline["note"] = ("issue-bound: 76 % issue-slot utilisation while warps are resident (31 % of the warp slots), DRAM "
                            "throughput 2.9 % of peak in the ncu capture (profiles/r02k_ncu_full_summary.txt); algorithmic bytes = "
                            "40 B per (Gaussian, tile) instance + 16 B per pixel, measured DRAM traffic is 0.2x of that (records are "
                            "L1/L2 hits)")

    # ---- CPU baseline: Open3D-0.17-equivalent TSDF (oracle port) on a bounded sample, all host threads
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_tsdf_baseline(renderer, vol, stage, rigs, mine, cfg, bargs, baseline, budget_s=args.cpu_budget)

    line = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": round(elapsed_ms / max(K, 1), 4), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": shared_config(args, cfg, total_views, world, K),
        "details": {"volume_merge": None if world == 1 else {"kind": "gsb_tsdf_reduce: union of the ranks' bricks, one " + ("ncclReduce to rank 0" if MERGE_DST == 0 else "ncclAllReduce"),
                                                             "ms": round(reduce_ms, 3), "phases_ms_rank0": merge_phases},
                    "l2": f"inputs larger than L2: {236 * cfg['num_points'] / 1e6:.0f} MB of Gaussian parameters re-read per pair + brick store per view",
                    "tsdf_colour": "fused (float4 running mean)", "exact_tile_cull": True,
                    "pair_mode": os.environ.get("GSB_PAIR_MODE", "fused"),
                    "pairs_sharing_one_depth_sort": round(float(np.mean([renderer._shared_depth[i] for i in mine])), 3) if mine else None,
                    "pairs_in_flight": int(renderer.pairs_in_flight),
                    "frame_copies_on_own_streams": bool(renderer.copy_streams),
                    "spare_buffer_sets": int(renderer.spare_buffer_sets),
                    "e2e_loop_order": os.environ.get("BENCH_E2E_ORDER", DEFAULT_E2E_ORDER),
                    "host_enqueue_ms_per_step": round(host_enqueue_ms, 4),
                    "caller_stream_priority": int(torch.cuda.current_stream().priority),
                    "per_view": {k: round(v, 1) for k, v in mean.items()},
                    "tsdf_volume": {"kind": "unbounded hashed brick pool", "bricks_open_after_timed_region": int(pool_after["bricks"]),
                                    "bricks_dropped": int(pool_after["dropped_total"]), "pool_bricks": int(vol.pool_bricks)}},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": K_e2e},
        "gpu_launches": launches,
        "roofline": roofline,
        "kernels": kernels,
        "kernels_note": f"per-kernel CUDA-event durations from {n_prof} steps with the eyes serialised on one stream "
                        f"({round(serial_ms_per_step, 4)} ms/step); the timed region overlaps the two eyes on two streams.  "
                        "preprocess is ONE launch per stereo pair (both eyes), depth_sort one per pair when the eyes share "
                        "their view depths, else one per eye (launches_per_step)",
        "cpu_baseline": cpu_baseline,
    }
    return line


def cpu_tsdf_baseline(renderer, vol, stage, rigs, mine, cfg, bargs, baseline, budget_s=20.0):
    """The reference's CPU-path TSDF (Open3D ScalableTSDFVolume restated, oracle/tsdf_oracle.cpp) on the
    first few depth frames of the same workload; the oracle is only timed here, never used as a result."""
    from oracle import oracle as orc

    W, H = cfg["width"], cfg["height"]
    cores = os.cpu_count() or 1
    frames = []
    for i in mine[:8]:
        out = renderer.render_image_pair(i, to_host=True)
        d = vol.prepare_depth(out["depth"], W, H, final_T=out["final_T"], min_depth=bargs.TSDF_min_depth_baselines * baseline)
        frames.append((d.cpu().numpy(), out["host_left_u8"].numpy().copy(), rigs[i]["left"]))
    ovol = orc.OracleTSDFVolume(vol.voxel_length, vol.sdf_trunc, with_color=True)
    n, t0 = 0, time.perf_counter()
    for d, rgb, cam_ in frames:
        ovol.integrate(d, rgb, W, H, cam_["fx"], cam_["fy"], cam_["cx"], cam_["cy"], np.linalg.inv(cam_["extrinsic"]),
                       depth_scale=1.0, depth_trunc=baseline * bargs.TSDF_max_depth_baselines, threads=cores)
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": round(n / dt, 4), "unit": "stereo-pairs/s (TSDF fuse only, CPU)", "cores": cores, "kind": "port",
            "sample": f"first {n} left depth frames of the workload, Open3D-0.17-equivalent ScalableTSDFVolume restatement, {cores} OpenMP threads"}


# ------------------------------------------------------------------------------------------------ reference arm
def emit_depth_frames(args, cfg, local):
    """Child process of the reference arm (untimed set-up): the depth frames that stand in for the out-of-scope stereo
    network's output, rendered with this repository's rasterizer and written to a .npz.  Running it in a separate process
    keeps libgs2mesh_b200.so out of the process that times the reference."""
    from gs2mesh_b200.renderer import Renderer
    from gs2mesh_b200.tsdf import TSDFVolume

    n_sample = int(os.environ["GSB_BENCH_NSAMPLE"])
    total_views = int(os.environ["GSB_BENCH_TOTAL_VIEWS"])
    cloud, rigs, baseline = build_scene(cfg, total_views)
    bargs = BenchArgs(cfg)
    W, H = cfg["width"], cfg["height"]
    dev = torch.device("cuda", local)
    helper = Renderer.from_scene(rigs, baseline, cloud, output_dir_root=None, args=bargs, device=str(dev))
    helper.prepare_renderer()
    hv = TSDFVolume(2.0 / cfg["tsdf_res"], bargs.TSDF_sdf_trunc, with_color=False, device=dev, pool_bricks=16)
    frames = []
    for i in range(n_sample):
        out = helper.render_image_pair(i, to_host=False)
        frames.append(hv.prepare_depth(out["depth"], W, H, final_T=out["final_T"],
                                       min_depth=bargs.TSDF_min_depth_baselines * baseline).cpu().numpy())
    np.savez(args.emit_depth_frames, depth=np.stack(frames))


def run_reference(args, cfg, rank, local, world):
    if rank != 0:
        return None
    from oracle import oracle as orc

    K, Wm = args.steps, args.warmup
    total_views = K if args.scaling == "strong" else K * world
    cloud, rigs, baseline = build_scene(cfg, total_views)
    bargs = BenchArgs(cfg)
    W, H = cfg["width"], cfg["height"]
    cores = os.cpu_count() or 1
    dev = torch.device("cuda", local)
    have_ref = orc.ref_available()
    if not have_ref:
        return {"impl": "reference", "unavailable": "oracle/_ref/libref_dgr.so (reference rasterizer built for sm_100a) is missing"}

    from gs2mesh_b200 import camera as cam  # host-side pose maths only (numpy); does not load the CUDA library

    up = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    g = dict(xyz=up(cloud.xyz), sh=up(cloud.features), op=up(cloud.opacity).reshape(-1), sc=up(cloud.scaling), ro=up(cloud.rotation))
    bg = torch.zeros(3, device=dev)

    # Set-up only (untimed, in a CHILD process): depth frames standing in for the stereo network's output.
    n_sample = min(K + Wm, total_views)
    tmp = tempfile.mktemp(prefix="gsb_depth_frames_", suffix=".npz")
    env = dict(os.environ, GSB_BENCH_NSAMPLE=str(n_sample), GSB_BENCH_TOTAL_VIEWS=str(total_views))
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--config", args.config, "--emit-depth-frames", tmp, "--gpus", "1"],
                   check=True, env=env, stdout=sys.stderr)
    depth_frames = np.load(tmp)["depth"]
    os.unlink(tmp)
    assert "libgs2mesh_b200" not in open("/proc/self/maps").read(), "the reference process must not map the product library"

    ovol = orc.OracleTSDFVolume(2.0 / cfg["tsdf_res"], bargs.TSDF_sdf_trunc, with_color=True)

    raster_ms, raster_wall_ms = [], []

    def step(i):
        frames = []
        for side in ("left", "right"):  # renderer_utils.py:378-390
            c = rigs[i][side]
            vt = cam.view_transforms_from_camera(c)
            view, proj, pos = up(vt.world_view), up(vt.full_proj), up(vt.cam_center)  # cameras.py:54-57 uploads per view
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            res = orc.ref_forward_torch(g["xyz"], g["op"], view, proj, pos, W, H, vt.tan_fovx, vt.tan_fovy, bg, shs=g["sh"],
                                        scales=g["sc"], rotations=g["ro"], sh_degree=3)
            e1.record()
            e1.synchronize()
            raster_wall_ms.append(1e3 * (time.perf_counter() - t0))
            raster_ms.append(e0.elapsed_time(e1))
            rendering = (res["color"].permute(1, 2, 0) * 255).cpu().numpy()  # :389
            frames.append(np.clip(np.rint(rendering), 0, 255).astype(np.uint8))  # imwrite's float->u8
        c = rigs[i]["left"]
        ovol.integrate(depth_frames[i], frames[0], W, H, c["fx"], c["fy"], c["cx"], c["cy"], np.linalg.inv(c["extrinsic"]),
                       depth_scale=1.0, depth_trunc=baseline * bargs.TSDF_max_depth_baselines, threads=cores)

    order = list(range(n_sample))
    for i in order[:Wm]:
        step(i)
    torch.cuda.synchronize()
    raster_ms.clear()
    raster_wall_ms.clear()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = time.perf_counter()
    done = 0
    for i in order[Wm:Wm + K] if n_sample >= Wm + K else order[:K]:
        step(i)
        done += 1
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    value = done / dt
    return {
        "impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": UNIT, "n_gpus": world, "steps": done, "warmup": Wm,
        "ms_per_step": round(1e3 * dt / max(done, 1), 3), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": shared_config(args, cfg, total_views, world, K if args.scaling == "weak" else len(range(0, total_views, world))),
        "details": {"note": "reference rasterizer (oracle/_ref, sm_100a build of the unmodified sources) x2 per pair as called by "
                            "renderer_utils.py:378-390 + Open3D-0.17-equivalent CPU TSDF; rank 0 only; PNG encode and DLNR excluded; "
                            "the stand-in depth frames were rendered by a child process (this process never maps libgs2mesh_b200.so)",
                    "reference_rasterizer_ms_per_view": {
                        "cuda_events_around_the_call": round(float(np.mean(raster_ms)), 4) if raster_ms else None,
                        "host_wall": round(float(np.mean(raster_wall_ms)), 4) if raster_wall_ms else None,
                        "note": "as called: the reference blocks on a 4-byte D2H in the middle of every frame "
                                "(rasterizer_impl.cu:281) and grows three scratch buffers through callbacks, so its per-view time "
                                "follows the host's launch / copy latency (2.5 ms on one box, 5.0 ms on another in round 1), "
                                "not only its kernels"}},
        "clocks": clocks,
        "cpu_baseline": {"value": round(value, 4), "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{done} stereo pairs: reference rasterizer (unmodified sources, sm_100a build, GPU) + Open3D-0.17-equivalent CPU TSDF port on {cores} threads"},
        "e2e": {"value": round(value, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="C1")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (driver contract): --steps pairs PER RANK; strong: --steps pairs in total, split over the ranks")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the last step's outputs as DIR/<name>.npy (--impl ours)")
    ap.add_argument("--emit-depth-frames", default=None, help=argparse.SUPPRESS)  # child process of the reference arm
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is only implemented for --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    from gs2mesh_b200 import scene

    cfg = scene.CONFIGS[args.config]
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: gs2mesh_b200 has no CPU fallback")
    rank, local, world = setup_dist(args.gpus)
    if rank == 0:
        if args.impl == "reference" and not args.emit_depth_frames:
            from oracle import oracle as orc

            orc.build()  # the checker only: the reference process never loads the product library
        else:
            import __graft_entry__ as ge

            ge.build()
    barrier(world)
    if args.emit_depth_frames:
        emit_depth_frames(args, cfg, local)
        return
    if args.impl == "reference":
        line = run_reference(args, cfg, rank, local, world)
    else:
        line = run_ours(args, cfg, rank, local, world)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and line is not None:
        print(json.dumps(line))


if __name__ == "__main__":
    main()
