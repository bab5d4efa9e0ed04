#!/usr/bin/env python
"""bench.py -- the hot path's headline benchmark (BASELINE.json: "Gaussians/sec rasterized (fwd & fwd+bwd) @256^2").

A "step" is one pass of the rasterizer over one batch of synthetic input: configs[1] of BASELINE.json,
500k Gaussians x 8 views x 256x256, SH (25 coefficients, degree-3 evaluation), forward only.  Per rank the work is
fixed (weak scaling): rank r renders views [8r, 8r+8) of the same cloud; there is no collective in the data
path (views are independent), only an all-gather of per-view PSNR after the timed region.

Reported on ONE JSON line (see the task contract):
  value      forward Gaussians/s (= P * views / time), inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the C ABI's host-buffer entry gs_render_host (pinned host inputs copied to the
             device and images copied back inside the timed region)
  fwd_bwd    forward + backward (MSE to a random target) Gaussians/s, device-resident
  roofline   dominant kernel: algorithmic bytes per launch / its average duration (CUDA events on the launch
             stream, recorded by the library around each stage), against MEASURED_PEAKS.json's HBM GB/s
  cpu_baseline  the CPU oracle port (oracle/gs_oracle.c, OpenMP) timed on this box's host cores on a bounded
             sample (whole views of the same workload)
  moving_cloud  the forward when the cloud MOVES every step (means jittered by ~1 px, 5 % of the Gaussians re-drawn): the
             speculative bucket capacities are learned from the previous call, so this leg reports ms/step AND how often
             the speculation overflowed and the call was redone exactly
  c4         BASELINE.json configs[3] (2M Gaussians x 32 views x 512x512), the 32 views split over the N ranks (strong
             scaling): ms/step, 512x512 views/s
  parity     view 0 against the oracle: pixels over 1e-4, fragile fraction, worst non-fragile / fragile error (N = 1)
`--impl reference` times that CPU port alone (the reference's rasterizer is an absent external CUDA extension
and the reference has no CPU path of its own: SURVEY.md section 0, BASELINE.md section 2-3).
`--dump-outputs DIR` writes what the last timed forward step returned (DIR/color.npy, DIR/radii.npy; suffixed _rank<r>
under N > 1), at most DUMP_BUDGET bytes over all ranks (see write_outputs).  The inputs are seeded, so two builds run
with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D_SH = 25
# BASELINE.json configs: the metric is quoted on configs[1] (C2), which is the default and the only bench line the
# driver reads; C4 (configs[3]) is available for extra measurements with --workload c4
WORKLOADS = {
    "c2": (500_000, 8, 256, "C2: 500k Gaussians x 8 views x 256x256, SH 25 coeff (deg-3 eval), forward"),
    "c4": (2_000_000, 32, 512, "C4: 2M Gaussians x 32 views x 512x512, SH 25 coeff (deg-3 eval), forward"),
}
P_GAUSS, VIEWS, HW, WORKLOAD = WORKLOADS["c2"]


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU every 5 ms through NVML while the timed regions run."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self.thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes CUDA_VISIBLE_DEVICES; NVML enumerates physical devices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].strip().isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml unavailable: {type(e).__name__}")
            return

        def loop():
            while not self._stop.is_set():
                try:
                    self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in self.REASONS.items():
                        if mask & bit:
                            self.reasons.add(name)
                except Exception:  # noqa: BLE001
                    pass
                time.sleep(0.005)

        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        self._stop.set()
        if self.thread:
            self.thread.join(timeout=1)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def host_threads() -> int:
    """CPU threads this process may really use: the affinity mask and a cgroup CPU quota (containers) both cap
    os.cpu_count(); oversubscribing a quota with one OpenMP thread per visible CPU makes the CPU baseline slower."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:  # cgroup v2, then v1
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except (OSError, ValueError):
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0 and period > 0:
                n = min(n, max(1, -(-quota // period)))
        except (OSError, ValueError):
            pass
    return max(1, n)


DUMP_BUDGET = 64 * 10**6   # bytes --dump-outputs may write, all ranks together


def write_outputs(out_dir, outputs, world=1, rank=0, budget=DUMP_BUDGET):
    """Writes `outputs` (name -> array) as out_dir/<name>.npy in float32, suffixed _rank<r> under N > 1, in at most
    budget // world bytes per rank.  Arrays over that share are all replaced by a fixed sample of their elements, seeded
    by the rank and so the same in every run of the same workload: the values in <name>.npy, their flat indices into the
    full array in <name>_index.npy (float64, exact below 2**53).  Returns the bytes written."""
    import numpy as np
    share = budget // world
    header = 128                 # .npy header of these arrays
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in outputs.items()}
    if sum(a.nbytes + header for a in arrays.values()) > share:
        # one sampling fraction for all arrays: 4 bytes of value + 8 of index per kept element
        frac = max(0, share - 2 * header * len(arrays)) / (12 * sum(a.size for a in arrays.values()))
        rng = np.random.default_rng(rank)
        sampled = {}
        for k, a in arrays.items():
            idx = np.unique(rng.integers(0, a.size, int(a.size * frac)))
            sampled[k], sampled[k + "_index"] = a.reshape(-1)[idx], idx.astype(np.float64)
        arrays = sampled
    os.makedirs(out_dir, exist_ok=True)
    written = 0
    for k, a in arrays.items():
        path = os.path.join(out_dir, k + (f"_rank{rank}" if world > 1 else "") + ".npy")
        np.save(path, a)
        written += os.path.getsize(path)
    assert written <= share, f"--dump-outputs wrote {written} bytes, over this rank's {share}"
    return written


def run_reference(args):
    """CPU arm: the oracle port on the host cores, one whole view of the workload per step."""
    import numpy as np
    from oracle.gs_oracle import OracleRender
    from pf3plat_b200.synthetic import make_scene
    from tests.util import view_args
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import gs_oracle
    cores = gs_oracle.set_threads(host_threads())   # torchrun exports OMP_NUM_THREADS=1: ask for all usable cores
    sc = make_scene(P_GAUSS, VIEWS, HW, HW, seed=0)
    for _ in range(args.warmup):
        st, kw = view_args(sc, 0)
        OracleRender(st, frag_rel=0, **kw).close()
    t0 = time.perf_counter()
    for k in range(args.steps):
        st, kw = view_args(sc, k % VIEWS)
        OracleRender(st, frag_rel=0, **kw).close()
    dt = time.perf_counter() - t0
    val = P_GAUSS * args.steps / dt
    sample = f"{args.steps} steps x 1 view ({P_GAUSS} Gaussians, {HW}x{HW}) of the {WORKLOAD.split(':')[0]} workload, forward"
    print(json.dumps({
        "impl": "reference", "metric": "gaussians_per_sec_fwd_256", "value": val, "unit": "Gaussians/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "reference rasterizer is an absent external CUDA extension; this "
                   "is the CPU oracle port of its algorithm, OpenMP over tiles"},
        "cpu_baseline": {"value": val, "unit": "Gaussians/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Gaussians/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tuning", type=int, default=0, help="GS_TUNE_* flags (experiments)")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-c4", action="store_true", help="skip the C4 (2M x 32 views x 512x512) strong-scaling block")
    ap.add_argument("--no-moving", action="store_true", help="skip the moving-cloud leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed forward step returned (color, radii) to DIR/<name>.npy, in float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global P_GAUSS, VIEWS, HW, WORKLOAD
    P_GAUSS, VIEWS, HW, WORKLOAD = WORKLOADS[args.workload]
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from pf3plat_b200 import _capi, rasterizer
    from pf3plat_b200.cameras import make_view_batch
    from pf3plat_b200.rasterizer import BatchSettings, rasterize_batch
    from pf3plat_b200.sharding import gather_metric, interleave_views, shard_views
    from pf3plat_b200.synthetic import make_scene, make_target

    # on the GPU box NCCL prints a "NCCL version ..." banner on stdout (NCCL_DEBUG=VERSION via env or nccl.conf),
    # next to the one JSON line this script owes its caller; an explicit NCCL_DEBUG=INFO etc. is left alone
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists)"
    torch.cuda.set_device(local)
    from pf3plat_b200.sharding import SharedCloudUploader, numa_local_allocation
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- synthetic workload: this rank's 8 views of the shared cloud (SURVEY.md section 8(d)) ----
    # weak scaling: 8 views per rank out of world * 8 on the camera circle, dealt round-robin -- every rank gets the same
    # mix of the circle (at N = 1 these are the circle's 8 views; contiguous blocks gave every rank one arc, and the arcs'
    # tile-instance counts differ by a few per cent: the job then ran at the pace of the heaviest arc)
    my_views = interleave_views(world * VIEWS, rank, world)
    sc = make_scene(P_GAUSS, len(my_views), HW, HW, seed=0, first_view=my_views[0], total_views=world * VIEWS,
                    view_stride=world)
    vb = make_view_batch(sc.extrinsics, sc.intrinsics, sc.near, sc.far, scale_invariant=True)
    host = {
        "means3D": sc.means.reshape(1, P_GAUSS, 3), "opacities": sc.opacities.reshape(1, P_GAUSS),
        "shs": sc.harmonics.permute(0, 2, 1).contiguous().reshape(1, P_GAUSS, D_SH, 3),
        "cov3D_precomp": torch.stack([sc.covariances[:, 0, 0], sc.covariances[:, 0, 1], sc.covariances[:, 0, 2],
                                      sc.covariances[:, 1, 1], sc.covariances[:, 1, 2], sc.covariances[:, 2, 2]],
                                     -1).reshape(1, P_GAUSS, 6),
        "viewmatrix": vb.viewmatrix, "projmatrix": vb.projmatrix, "campos": vb.campos, "bg": sc.background,
        "tanfov": vb.tanfov,
    }
    # pinned staging buffers are allocated while the process sits on the GPU's own socket (first touch), then the
    # affinity is released again
    with numa_local_allocation(local) as numa:
        host = {k: v.contiguous().float().pin_memory() for k, v in host.items()}
        out_color = torch.empty((VIEWS, 3, HW, HW), dtype=torch.float32).pin_memory()
        out_radii = torch.empty((VIEWS, P_GAUSS), dtype=torch.int32).pin_memory()
    numa_cpus = numa.cpus
    d = {k: v.to(dev) for k, v in host.items()}
    bs = BatchSettings(image_height=HW, image_width=HW, viewmatrix=d["viewmatrix"], projmatrix=d["projmatrix"],
                       campos=d["campos"], bg=d["bg"], sh_degree=4, tanfov=d["tanfov"], tuning=args.tuning)

    def fwd():
        with torch.no_grad():
            return rasterize_batch(bs, d["means3D"], d["opacities"], shs=d["shs"], cov3D_precomp=d["cov3D_precomp"])

    target = make_target(VIEWS, HW, HW, seed=1 + rank).to(dev)
    leaves = {k: d[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "shs", "cov3D_precomp")}

    def fwd_bwd():
        for t in leaves.values():
            t.grad = None
        color, _ = rasterize_batch(bs, leaves["means3D"], leaves["opacities"], shs=leaves["shs"],
                                   cov3D_precomp=leaves["cov3D_precomp"])
        loss = ((color - target) ** 2).mean()
        loss.backward()
        return loss

    # ---- e2e through the C ABI with HOST buffers ----
    L = _capi.lib()
    hcfg = _capi.GsConfig()
    hcfg.P, hcfg.S, hcfg.V, hcfg.M, hcfg.sh_degree = P_GAUSS, 1, VIEWS, D_SH, 4
    hcfg.image_height = hcfg.image_width = HW
    hcfg.scale_modifier = 1.0
    hcfg.tuning = args.tuning
    for k in ("viewmatrix", "projmatrix", "campos", "bg", "tanfov"):
        setattr(hcfg, k, host[k].data_ptr())
    hin = _capi.GsInputs(means3D=host["means3D"].data_ptr(), opacities=host["opacities"].data_ptr(),
                         shs=host["shs"].data_ptr(), cov3D_precomp=host["cov3D_precomp"].data_ptr())
    hout = _capi.GsOutputs(color=out_color.data_ptr(), radii=out_radii.data_ptr(), depth=None)
    # Bytes that cross PCIe per step.  Everything but the SH block is copied whole; of the SH block (pinned, M = 25)
    # k_sh_colour pulls the 16-byte pieces that hold a coefficient of bands 0..3 straight out of the host buffer
    # (zero-copy feed): 51 of every 75 pieces (4 rows).  --tuning 131072 (GS_TUNE_NO_ZERO_COPY) copies it whole instead.
    zero_copy = D_SH > 16 and not (args.tuning & _capi.GS_TUNE_NO_ZERO_COPY)
    row_f = D_SH * 3
    pulled16 = sum(1 for q in range(row_f) if (4 * q) % row_f < 48 or (4 * q) % row_f + 3 >= row_f)   # per 4 rows = row_f pieces
    sh_bytes = host["shs"].numel() * 4
    sh_crossing = sh_bytes * pulled16 // row_f if zero_copy else sh_bytes
    h2d = sum(host[k].numel() * 4 for k in host if k != "shs") + sh_crossing
    d2h = out_color.numel() * 4 + out_radii.numel() * 4
    stream = torch.cuda.current_stream(dev)
    ctx = rasterizer.current_context(dev)

    def e2e_single():
        _capi.check(L.gs_render_host(ctx, ctypes.byref(hcfg), ctypes.byref(hin), ctypes.byref(hout), stream.cuda_stream))

    # N > 1: the ranks of one box render different views of the SAME cloud.  Every rank uploads 1/N of the per-Gaussian
    # arrays over its own PCIe link and one NCCL all-gather per array (NVLink) completes the cloud on every GPU
    # (pf3plat_b200.sharding.SharedCloudUploader); cameras are per rank.  Then the device entry, then the results back.
    uploader = None
    if world > 1:
        cloud_host = {"means3D": host["means3D"][0], "opacities": host["opacities"][0], "shs": host["shs"][0],
                      "cov3D_precomp": host["cov3D_precomp"][0]}
        uploader = SharedCloudUploader(cloud_host, dev)
        cam_keys = ("viewmatrix", "projmatrix", "campos", "bg", "tanfov")
        cam_dev = {k: torch.empty_like(host[k], device=dev) for k in cam_keys}
        h2d = uploader.bytes_per_step + sum(host[k].numel() * 4 for k in cam_keys)

    def e2e_shared():
        with torch.no_grad():
            for k in cam_keys:
                cam_dev[k].copy_(host[k], non_blocking=True)
            cl = uploader.upload()
            bs_e = BatchSettings(image_height=HW, image_width=HW, viewmatrix=cam_dev["viewmatrix"], projmatrix=cam_dev["projmatrix"],
                                 campos=cam_dev["campos"], bg=cam_dev["bg"], sh_degree=4, tanfov=cam_dev["tanfov"], tuning=args.tuning)
            c_, r_ = rasterize_batch(bs_e, cl["means3D"][None], cl["opacities"][None], shs=cl["shs"][None],
                                     cov3D_precomp=cl["cov3D_precomp"][None])
            out_color.copy_(c_, non_blocking=True)
            out_radii.copy_(r_, non_blocking=True)
        stream.synchronize()

    e2e = e2e_shared if world > 1 else e2e_single

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    per_rank_ms = {}

    def timed(fn, steps, warmup, tag=None, keep_last=False):
        """Device ms of `steps` calls of fn (max over ranks); with keep_last, also what the last call returned."""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps - 1):
            fn()
        last = fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            every = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(every, ms)                      # each rank's own device time: what the MAX below is taken over
            per_rank_ms[tag] = [float(t.item()) / steps for t in every]
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return (float(ms.item()), last) if keep_last else float(ms.item())

    gauss_per_step = P_GAUSS * VIEWS * world

    # correctness spot check + counters (outside every timed region)
    color, radii = fwd()
    torch.cuda.synchronize(dev)
    stats = rasterizer.last_stats(dev)
    launches_fwd = stats["kernel_launches"]
    D_ours = stats["num_rendered"]
    vis = int((radii > 0).sum().item())
    e2e()
    assert torch.equal(out_color.to(dev), color), "host-buffer entry and device entry disagree"
    if world > 1:
        e2e_single()    # the single-rank entry agrees with the shared upload
        assert torch.equal(out_color.to(dev), color)

    sampler = ClockSampler(local)
    sampler.start()
    ms_fwd, last_fwd = timed(fwd, args.steps, args.warmup, "fwd", keep_last=True)
    launches_fwd = rasterizer.last_stats(dev)["kernel_launches"]   # of the last timed step (steady state)
    dump = {name: t.float().cpu().numpy() for name, t in zip(("color", "radii"), last_fwd)} if args.dump_outputs else None
    del last_fwd
    ms_e2e = timed(e2e, args.steps, args.warmup, "e2e")
    launches_e2e = rasterizer.last_stats(dev)["kernel_launches"]   # 4 with the split pipeline (k_sh_colour), else 3
    ms_fb = timed(fwd_bwd, args.steps, args.warmup, "fwd_bwd")
    stats_fb = rasterizer.last_stats(dev)

    # ---- moving cloud: every step renders a different cloud (training moves the Gaussians between steps), so the bucket
    # capacities learned from step k-1 meet the counts of step k.  Means are jittered by ~1 px (sigma = 1 px worth of
    # camera-space x/y at the Gaussian's depth) and 5 % of the Gaussians are re-drawn somewhere else; all variants are
    # built before the timed region, each step only picks the next one.
    moving = None
    if not args.no_moving:
        g = torch.Generator(device="cpu").manual_seed(77 + rank)
        nvar = min(args.steps + args.warmup, 32)
        px_at_depth = (2.0 * (0.5 / 0.86) / HW)                     # camera-space x per pixel per unit depth
        variants = []
        base = sc.means
        for k in range(nvar):
            m = base + torch.randn(P_GAUSS, 3, generator=g) * (base[:, 2:3] * px_at_depth) * torch.tensor([1.0, 1.0, 0.0])
            # re-drawn Gaussians get a new position in the image at their OWN depth (their world-space size was drawn for
            # that depth: moving one from depth 20 to depth 1.5 would make it a 13x larger splat, a different workload)
            redraw = torch.rand(P_GAUSS, generator=g) < 0.05
            nr = int(redraw.sum())
            z = base[redraw, 2:3]
            m[redraw] = torch.cat([(torch.rand(nr, 2, generator=g) * 2.1 - 1.05) * (0.5 / 0.86) * z, z], dim=1)
            variants.append(m.reshape(1, P_GAUSS, 3).contiguous().to(dev))
        state = {"k": 0, "overflows": 0, "calls": 0}

        def fwd_moving():   # nothing but the call in the timed loop: overflows are counted by the library (GsStats.overflow_redos)
            with torch.no_grad():
                rasterize_batch(bs, variants[state["k"] % nvar], d["opacities"], shs=d["shs"], cov3D_precomp=d["cov3D_precomp"])
            state["k"] += 1
            state["calls"] += 1

        for _ in range(3 + nvar):                                  # exact -> trial -> steady state, then once through every
            fwd_moving()                                            # variant: the sticky capacities ratchet up to the largest
        state.update(calls=0)                                       # (each growth re-allocates ~100 MB of buckets, ~1 ms)
        redos0 = rasterizer.last_stats(dev)["overflow_redos"]
        ms_mov = timed(fwd_moving, args.steps, args.warmup, "moving_cloud")
        state["overflows"] = rasterizer.last_stats(dev)["overflow_redos"] - redos0
        rasterizer.set_profiling(True, dev)
        acc_m = {}
        for _ in range(5):
            fwd_moving()
            for k_, v_ in rasterizer.stage_ms(dev).items():
                acc_m.setdefault(k_, []).append(v_)
        rasterizer.set_profiling(False, dev)
        moving = {"stage_ms": {k_: statistics.mean(v_) for k_, v_ in acc_m.items()},
                  "tile_instances_last": rasterizer.last_stats(dev)["num_rendered"],
                  "ms_per_step": ms_mov / args.steps, "value": gauss_per_step * args.steps / (ms_mov * 1e-3),
                  "unit": "Gaussians/s", "overflow_rate": state["overflows"] / max(1, state["calls"]),
                  "calls": state["calls"], "variants": nvar,
                  "perturbation": "means jittered by N(0, 1 px) in x/y, 5 % of the Gaussians re-drawn at a new image position (same depth), every step"}
        del variants
        fwd()    # back to the static cloud's capacities for the stage profile below
        fwd()
    clocks = sampler.stop()   # covers the timed loops (warm-ups included: the GPU is under the same load)

    # ---- C4 (configs[3]): 2M Gaussians, 32 views of 512x512, the views split over the ranks (STRONG scaling) ----
    c4 = None
    if not args.no_c4 and args.workload == "c2" and 32 % world == 0:
        P4, V4, HW4 = 2_000_000, 32, 512
        mine4 = shard_views(V4, rank, world)
        sc4 = make_scene(P4, len(mine4), HW4, HW4, seed=0, first_view=mine4[0], total_views=V4)
        vb4 = make_view_batch(sc4.extrinsics, sc4.intrinsics, sc4.near, sc4.far, scale_invariant=True)
        cv = sc4.covariances
        d4 = {"means3D": sc4.means.reshape(1, P4, 3), "opacities": sc4.opacities.reshape(1, P4),
              "shs": sc4.harmonics.permute(0, 2, 1).contiguous().reshape(1, P4, D_SH, 3),
              "cov3D_precomp": torch.stack([cv[:, 0, 0], cv[:, 0, 1], cv[:, 0, 2], cv[:, 1, 1], cv[:, 1, 2], cv[:, 2, 2]],
                                           -1).reshape(1, P4, 6)}
        d4 = {k: v.contiguous().float().to(dev) for k, v in d4.items()}
        bs4 = BatchSettings(image_height=HW4, image_width=HW4, viewmatrix=vb4.viewmatrix.to(dev), projmatrix=vb4.projmatrix.to(dev),
                            campos=vb4.campos.to(dev), bg=sc4.background.to(dev), sh_degree=4, tanfov=vb4.tanfov.to(dev),
                            tuning=args.tuning)
        del sc4, cv

        def fwd4():
            with torch.no_grad():
                return rasterize_batch(bs4, d4["means3D"], d4["opacities"], shs=d4["shs"], cov3D_precomp=d4["cov3D_precomp"])

        steps4 = max(3, args.steps // 4)
        state4 = {"exact": 0, "calls": 0}

        def fwd4_counted():
            fwd4()
            state4["calls"] += 1
            state4["exact"] += int(rasterizer.last_stats(dev)["speculative"] == 0)

        for _ in range(3):
            fwd4()                      # exact -> trial -> steady state
        ms4_first = timed(fwd4_counted, steps4, 3, "c4_first_loop")
        ms4 = timed(fwd4_counted, steps4, 1, "c4")     # reported: the second timed loop (the first one is kept as `first_loop_ms`)
        st4 = rasterizer.last_stats(dev)
        # per-rank view of the same loop (its own CUDA events), gathered: who is the slowest and why
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record(stream)
        for _ in range(steps4):
            fwd4()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        mine = torch.tensor([e0.elapsed_time(e1) / steps4, float(st4["num_rendered"]), float(st4["speculative"]),
                             float(state4["exact"])], device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        if world > 1:
            dist.all_gather(allr, mine)
        else:
            allr = [mine]
        # forward + backward at this size too (MSE to a U(0,1) target, gradients to means / opacities / SH / covariances):
        # north_star asks for fwd and fwd+bwd views/s at 512x512
        leaves4 = {k: d4[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "shs", "cov3D_precomp")}
        target4 = make_target(len(mine4), HW4, HW4, seed=5).to(dev)

        def fwd_bwd4():
            for t in leaves4.values():
                t.grad = None
            col4, _ = rasterize_batch(bs4, leaves4["means3D"], leaves4["opacities"], shs=leaves4["shs"],
                                      cov3D_precomp=leaves4["cov3D_precomp"])
            ((col4 - target4) ** 2).mean().backward()

        steps4_fb = max(8, args.steps // 2)
        for _ in range(5):
            fwd_bwd4()
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps4_fb + 1)]
        evs[0].record(stream)
        for k_ in range(steps4_fb):                      # one event per step: a hiccup shows as max >> median
            fwd_bwd4()
            evs[k_ + 1].record(stream)
        barrier()
        per_step4 = [evs[k_].elapsed_time(evs[k_ + 1]) for k_ in range(steps4_fb)]
        ms4_fb_t = torch.tensor([evs[0].elapsed_time(evs[-1])], device=dev)
        if world > 1:
            dist.all_reduce(ms4_fb_t, op=dist.ReduceOp.MAX)
        ms4_fb = float(ms4_fb_t.item())
        del leaves4, target4
        c4 = {"workload": WORKLOADS["c4"][3], "scaling": "strong", "views_total": V4, "views_per_gpu": len(mine4),
              "fwd_bwd": {"ms_per_step": ms4_fb / steps4_fb, "views_per_sec_512": V4 * steps4_fb / (ms4_fb * 1e-3),
                          "gaussians_per_sec": P4 * V4 * steps4_fb / (ms4_fb * 1e-3), "loss": "MSE to U(0,1) target",
                          "steps": steps4_fb, "median_step_ms_rank0": statistics.median(per_step4),
                          "max_step_ms_rank0": max(per_step4)},
              "steps": steps4, "ms_per_step": ms4 / steps4, "views_per_sec_512": V4 * steps4 / (ms4 * 1e-3),
              "gaussians_per_sec": P4 * V4 * steps4 / (ms4 * 1e-3), "tile_instances_rank0": st4["num_rendered"],
              "speculative": st4["speculative"], "first_loop_ms_per_step": ms4_first / steps4,
              "per_rank": [{"ms_per_step": float(t[0]), "tile_instances": int(t[1]), "speculative": int(t[2]),
                            "exact_path_calls_in_timed_loop": int(t[3])} for t in allr]}
        del d4, bs4
        torch.cuda.empty_cache()
        rasterizer.trim_memory(dev)
        fwd()
        fwd()

    # per-stage device time (library-recorded CUDA events on the launch stream), separate pass
    rasterizer.set_profiling(True, dev)
    acc = {}
    for _ in range(max(3, args.steps // 2)):
        fwd_bwd()
        for k, v in rasterizer.stage_ms(dev).items():
            acc.setdefault(k, []).append(v)
    rasterizer.set_profiling(False, dev)
    stage = {k: statistics.mean(v) for k, v in acc.items()}

    # PSNR of each view against the target, gathered over ranks (the only collective of the job)
    from pf3plat_b200.metrics import compute_psnr
    psnr = gather_metric(compute_psnr(target, color))

    if rank == 0:
        hbm, hbm_src = peaks()
        # CPU baseline on a bounded sample + the oracle's own D (upstream's 3-sigma-square definition)
        cpu = None
        D_ref_per_view = None
        parity = None
        c1 = None
        if not args.no_cpu_baseline and world == 1:   # contract: the CPU baseline leg runs at N = 1 only
            from oracle import gs_oracle
            from oracle.gs_oracle import OracleRender
            from tests.util import view_args
            cores = gs_oracle.set_threads(host_threads())
            # (1) in this process, untimed: the oracle's tile-instance count D of every view of this rank (the D of the
            #     algorithmic-bytes formulas) and the worst RGB difference of view 0
            Ds = []
            for v in range(VIEWS):
                st, kw = view_args(sc, v)
                r = OracleRender(st, frag_rel=0, **kw)
                Ds.append(r.num_rendered)
                r.close()
            D_ref_per_view = sum(Ds) / VIEWS
            from tests.util import image_report, oracle_view
            r0 = oracle_view(sc, 0)                      # default fragility band (1e-4 relative), as in the tests
            parity = image_report(color[0], r0)
            parity["view"] = 0
            parity["tolerance"] = "1e-4 abs RGB on non-fragile pixels; fragile = an alpha>=1/255 / T<1e-4 / footprint decision within 1e-4 (relative) of its threshold in the oracle"
            err = max(parity["max_err_nonfragile"], parity["max_err_fragile"])
            r0.close()
            # C1 (BASELINE.json configs[0]: 10k Gaussians, 1 view, 256x256): both CPU restatements, forward, same box
            c1 = {}
            try:
                sc1 = make_scene(10_000, 1, 256, 256, seed=0)
                st1, kw1 = view_args(sc1, 0)
                OracleRender(st1, frag_rel=0, **kw1).close()
                t0 = time.perf_counter()
                for _ in range(5):
                    OracleRender(st1, frag_rel=0, **kw1).close()
                c1["c_oracle_ms"] = 1e3 * (time.perf_counter() - t0) / 5
                from oracle import torch_oracle
                torch.set_num_threads(cores)
                tk = {k: torch.from_numpy(np.ascontiguousarray(v)).float() for k, v in kw1.items()}
                with torch.no_grad():
                    t0 = time.perf_counter()
                    torch_oracle.render(st1, dtype=torch.float32, **tk)
                    c1["torch_oracle_ms"] = 1e3 * (time.perf_counter() - t0)
                c1["workload"] = "C1: 10k Gaussians x 1 view x 256x256, forward"
                c1["cores"] = cores
                c1["c_oracle_gaussians_per_sec"] = 10_000 / (c1["c_oracle_ms"] * 1e-3)
                c1["torch_oracle_gaussians_per_sec"] = 10_000 / (c1["torch_oracle_ms"] * 1e-3)
            except Exception as exc:  # noqa: BLE001
                c1["error"] = repr(exc)
            # (2) timed in a process of its own -- the same code as `--impl reference` -- so that this process's CUDA
            #     context, pinned buffers and thread pools do not perturb the CPU number (in-process it came out ~2.7x
            #     lower than the reference arm on the same box)
            import subprocess
            nsteps = min(3 * VIEWS, 24)
            cpu = None
            try:
                env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS")}
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(nsteps),
                                      "--warmup", "2", "--workload", args.workload], capture_output=True, text=True,
                                     timeout=900, env=env)
                ref = json.loads(out.stdout.strip().splitlines()[-1])
                cpu = {"value": ref["value"], "unit": "Gaussians/s", "cores": ref["cpu_baseline"]["cores"], "kind": "port",
                       "sample": f"{nsteps} views ({P_GAUSS} Gaussians, {HW}x{HW}) of this workload, forward, "
                                 "oracle/gs_oracle.c with OpenMP, timed in a separate process (= bench.py --impl reference)",
                       "max_abs_rgb_err_view0": float(err), "c1": c1}
            except Exception as exc:  # noqa: BLE001 -- fall back to timing it here
                sys.stderr.write(f"cpu_baseline subprocess failed ({exc}); timing in-process\n")
            if cpu is None:
                t0 = time.perf_counter()
                for v in range(VIEWS):
                    st, kw = view_args(sc, v)
                    OracleRender(st, frag_rel=0, **kw).close()
                dt = time.perf_counter() - t0
                cpu = {"value": P_GAUSS * VIEWS / dt, "unit": "Gaussians/s", "cores": cores, "kind": "port",
                       "sample": f"{VIEWS} views ({P_GAUSS} Gaussians, {HW}x{HW}), forward, oracle/gs_oracle.c with OpenMP, in-process",
                       "max_abs_rgb_err_view0": float(err), "c1": c1}
        # algorithmic bytes (SURVEY.md section 8(d)) with the kernels' OWN tile-instance count D (the tight binning walks
        # 27 % fewer instances than upstream's 3-sigma squares; using upstream's D would flatter every fraction)
        N = HW * HW
        D_up = (D_ref_per_view * VIEWS) if D_ref_per_view else None
        D_alg = D_ours
        S_sh = 12 * D_SH
        b_pre = 40 * P_GAUSS + S_sh * P_GAUSS + 48 * vis + 12 * P_GAUSS * VIEWS
        b_bin = 36 * D_alg
        b_comp = 40 * D_alg + 20 * N * VIEWS
        b_fwd = b_pre + b_bin + b_comp
        ms_bin = sum(stage.get(k) or 0.0 for k in ("bin_scan", "bin_emit", "bin_sort"))
        stages = {
            "preprocess": {"bytes": b_pre, "ms": stage.get("preprocess")},
            "bin": {"bytes": b_bin, "ms": ms_bin, "parts_ms": {k: stage.get(k) for k in ("bin_scan", "bin_emit", "bin_sort")}},
            "composite": {"bytes": b_comp, "ms": stage.get("composite")},
        }
        for s_ in stages.values():
            s_["achieved_gbs"] = s_["bytes"] / (s_["ms"] * 1e-3) / 1e9 if s_["ms"] else None
            s_["frac"] = s_["achieved_gbs"] / hbm if s_["ms"] else None
        # dominant single KERNEL of the forward (bin_scan also contains the host read-back, so it is not a candidate)
        sort_kernel = {0: "k_tile_sort", 1: "k_tile_sort_spec",
                       2: "k_stratum_sort" if (args.tuning & 64) else "k_stratum_rank_sort"}[stats_fb["speculative"]]
        kern_ms = {"k_preprocess": stage.get("preprocess"), "k_emit_buckets": stage.get("bin_emit"),
                   sort_kernel: stage.get("bin_sort"), "k_composite_fwd": stage.get("composite")}
        kern_bytes = {"k_preprocess": b_pre, "k_emit_buckets": 12 * D_alg, sort_kernel: 24 * D_alg, "k_composite_fwd": b_comp,
                      # backward split of SURVEY 8(d)'s B_bwd: compositor = dL/dpixel + T + n_contrib, staged records,
                      # per-(view,Gaussian) gradients written; preprocess backward = those re-read, inputs, outputs
                      "k_composite_bwd": 20 * N * VIEWS + 40 * D_alg + 44 * vis,
                      "k_preprocess_bwd": 88 * vis + 40 * P_GAUSS + S_sh * P_GAUSS + (40 + 12 * D_SH) * P_GAUSS}
        dom = max(kern_ms, key=lambda k: kern_ms[k] or 0)
        # ncu-derived per-launch figures of the same workload (profiles/r2_traffic.json, made by scripts/ncu_summary.py):
        # DRAM bytes and executed warp instructions.  The issue roofline is instructions / (SMs x 4 schedulers x clock).
        traffic, issue = None, None
        prof = {}
        for name in ("r2_traffic.json", "r1_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath) and args.workload == "c2":
                prof = json.load(open(tpath))
                break
        sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
        clock_hz = (clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0) * 1e6

        def issue_roofline(kernel, ms):
            winst = prof.get(kernel, {}).get("warp_instructions_per_launch") or prof.get(kernel, {}).get("warp_instructions")
            if not winst or not ms:
                return None
            floor_ms = winst / (sm_count * 4 * clock_hz) * 1e3
            return {"warp_instructions_per_launch": winst, "issue_slots_per_s": sm_count * 4 * clock_hz,
                    "floor_ms": floor_ms, "frac": floor_ms / ms,
                    "source": "ncu smsp__inst_executed.sum of this workload (profiles/), clock sampled in this run"}

        traffic = prof.get(dom, {}).get("dram_bytes_per_launch")
        issue = issue_roofline(dom, kern_ms[dom])
        dom_gbs = kern_bytes[dom] / (kern_ms[dom] * 1e-3) / 1e9
        issue_bound = dom in ("k_composite_fwd",) or (issue is not None and issue["frac"] > dom_gbs / hbm)
        bwd_kernels = {"k_composite_bwd": stage.get("composite_bwd"), "k_preprocess_bwd": stage.get("preprocess_bwd")}
        kernels_report = {k: {"ms": v, "hbm_frac": (kern_bytes[k] / (v * 1e-3) / 1e9 / hbm) if (v and k in kern_bytes) else None,
                              "issue": issue_roofline(k, v), "dram_bytes_per_launch": prof.get(k, {}).get("dram_bytes_per_launch")}
                          for k, v in {**kern_ms, **bwd_kernels}.items() if v}
        line = {
            "metric": "gaussians_per_sec_fwd_256", "value": gauss_per_step * args.steps / (ms_fwd * 1e-3),
            "unit": "Gaussians/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_fwd / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "views_per_gpu": VIEWS, "gaussians": P_GAUSS, "image": [HW, HW],
                       "parallelism": f"views dealt round-robin to {world} GPU(s) (rank r renders views r, r+N, ... of the {world * VIEWS} on the camera circle), no data-path collective",
                       "l2": "inputs+intermediates per step (~360 MB for C2) exceed the 126 MB L2; no explicit flush"},
            "views_per_sec": VIEWS * world * args.steps / (ms_fwd * 1e-3),
            "per_rank_ms_per_step": per_rank_ms or None,   # N > 1: every rank's own device time per step (value uses the max)
            "e2e": {"value": gauss_per_step * args.steps / (ms_e2e * 1e-3), "unit": "Gaussians/s",
                    "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "kernel_launches_per_call": launches_e2e,
                    "api": ("gs_render_host (C ABI, pinned host buffers; SH block pulled zero-copy by k_sh_colour: "
                            f"{sh_crossing} of its {sh_bytes} bytes requested in 16-byte pieces, the rest of the inputs copied)"
                            if zero_copy else "gs_render_host (C ABI, pinned host buffers, everything copied)") if world == 1 else
                           "SharedCloudUploader (1/N of the cloud per rank over PCIe + NCCL all-gather over NVLink) + "
                           "rasterize_batch + D2H of the results; pinned buffers allocated on the GPU's NUMA node",
                    "numa_cpus_rank0": len(numa_cpus)},
            "fwd_bwd": {"value": gauss_per_step * args.steps / (ms_fb * 1e-3), "unit": "Gaussians/s",
                        "ms_per_step": ms_fb / args.steps, "loss": "MSE to U(0,1) target"},
            "gpu_launches": (launches_fwd) * args.steps,
            "gpu_launches_note": f"{launches_fwd} own kernels per forward step (k_preprocess, the tile sort, "
                                 f"k_composite_fwd in steady state); fwd+bwd step: {stats_fb['kernel_launches']}",
            "roofline": {"kernel": dom, "bound": "issue" if issue_bound else "hbm", "achieved": dom_gbs, "peak": hbm,
                         "unit": "GB/s", "frac": dom_gbs / hbm, "traffic": traffic, "peak_source": hbm_src,
                         "algorithmic_bytes_per_launch": kern_bytes[dom], "ms_per_launch": kern_ms[dom],
                         "issue": issue,
                         "note": "achieved/peak/frac are the HBM figures the contract asks for, computed with the kernel's own "
                                 "tile-instance count; `bound` names what really limits the kernel: the compositors are "
                                 "instruction-issue bound (issue.frac = executed warp instructions / issue slots available in "
                                 "the measured time; DRAM < 15 % of peak)"},
            "kernels": kernels_report,
            "parity": parity,
            "moving_cloud": moving,
            "c4": c4,
            "roofline_stages": stages,
            "roofline_forward": {"bytes": b_fwd, "achieved_gbs": b_fwd / (ms_fwd / args.steps * 1e-3) / 1e9,
                                 "frac": b_fwd / (ms_fwd / args.steps * 1e-3) / 1e9 / hbm},
            "stage_ms": stage,
            "tile_instances": {"ours_tight": D_ours, "upstream_definition": D_up, "visible": vis},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "psnr_vs_target_mean": float(psnr.mean().item()),
        }
        sys.stdout.flush()
        print(json.dumps(line), flush=True)
    if dump is not None:
        write_outputs(args.dump_outputs, dump, world, rank)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
