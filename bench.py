#!/usr/bin/env python
"""bench.py -- scenes/sec of the 3D-SIS dense-voxel TEST forward on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg2|cfg3|cfg3s|cfg4|cfg5]
                  [--dump-outputs DIR]

A step = one pass of the hot path (back-projection -> 3D backbone -> RPN/NMS -> RoI pool + classifier -> per-RoI mask
head) over a batch of synthetic scenes; ENet-shaped 2D features are an input (ENet is upstream of the path, SURVEY 8f2).
Default workload = BASELINE.json configs[1] (cfg2: 96x48x96 ScanNet-shape chunks, 5 views); `--config` selects the other
BASELINE configs (SURVEY 8d): cfg3 whole scene 208x48x160 / 40 views (cfg3s: 88x44x88 / 40 views), cfg4 312 mixed-shape
scenes LPT-sharded over the ranks (strong scaling, NCCL all_gather of the detections inside the timed region), cfg5 SUNCG
backbone, 3 views, fp16-operand tensor-core math.  One process per GPU; scenes are independent, so ranks shard with no
data-path collective.  `value` times the scene loop with inputs resident in HBM, `e2e` the same loop from pinned HOST
buffers including the read-back of detections and thresholded masks.  No number here is taken under a profiler.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "3d-sis_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

MASK_BYTES_PER_VOXEL = 2712.0  # SURVEY 8(d): mask-head compulsory bytes per RoI voxel


# ------------------------------------------------------------------------------------------------ workloads
def alg_bytes(dims, cfgname="scannet"):
    """SURVEY 8(d) / appendix A: per-layer compulsory fp32 bytes of backbone + RPN.  cfg2 (96x48x96, ScanNet) = 806.8 MB;
    other shapes scale as 1824 B x N0 + 23 MB of weights (the cfg2 ratio, as 8(d) states); SUNCG chunk = 729.3 MB."""
    n0 = dims[0] * dims[1] * dims[2]
    if cfgname == "suncg":
        return 729.3e6 * n0 / (96 * 48 * 96)
    if tuple(dims) == (96, 48, 96):
        return 806.8e6
    return 1824.0 * n0 + 23e6


def flops(dims, cfgname="scannet"):
    base = 48.75e9 if cfgname == "suncg" else 53.86e9
    return base * dims[0] * dims[1] * dims[2] / (96 * 48 * 96)


CFG4_SHAPES = [((88, 44, 88), 8), ((96, 48, 96), 12), ((112, 48, 96), 16), ((128, 48, 112), 20), ((144, 48, 128), 24),
               ((160, 48, 128), 28), ((176, 48, 144), 32), ((208, 48, 160), 40)]


def workload(name, rank, world):
    """-> dict(metric, scenes=[(seed, dims, n_img)] (the distinct scenes this rank generates), ...)"""
    if name == "cfg2":
        return dict(metric="scenes_per_sec_96x48x96_5img", cfgname="scannet", math_default="exact", scaling="weak",
                    what="96x48x96 ScanNet-shape chunk, 5 views, full rpn_class_mask_5 TEST forward (cfg2)",
                    scenes=[(1000 + rank * 64 + j, (96, 48, 96), 5) for j in range(24)], chunks_default=320)
    if name in ("cfg3", "cfg3s"):
        dims = (208, 48, 160) if name == "cfg3" else (88, 44, 88)
        return dict(metric=f"scenes_per_sec_whole_scene_{dims[0]}x{dims[1]}x{dims[2]}_40img", cfgname="scannet",
                    math_default="exact", scaling="weak",
                    what=f"whole scene {dims[0]}x{dims[1]}x{dims[2]}, 40 views (every 20th frame), fully convolutional "
                         "rpn_class_mask_5 TEST forward (cfg3)",
                    scenes=[(3000 + rank * 16 + j, dims, 40) for j in range(4 if name == "cfg3" else 8)],
                    chunks_default=48 if name == "cfg3" else 160)
    if name == "cfg4":
        # 312 scenes (count of experiments/filelists/ScanNet/v1/test.txt), shape class and view count drawn per scene index
        # from 8 classes between 88x44x88/8 views and 208x48x160/40 views; the voxel/feature CONTENT of scene i is pool entry
        # (class_i, i % 2) -- 16 generated scenes -- because 312 distinct 1.6 M-voxel synthetic scenes would take minutes to
        # generate; every scene is still a full H2D + forward + D2H
        rng = np.random.default_rng(4)
        cls = rng.integers(0, len(CFG4_SHAPES), 312)
        pool = [(4000 + 2 * k + v, CFG4_SHAPES[k][0], CFG4_SHAPES[k][1]) for k in range(len(CFG4_SHAPES)) for v in range(2)]
        lst = [int(2 * cls[i] + i % 2) for i in range(312)]
        return dict(metric="scenes_per_sec_312_mixed_scenes", cfgname="scannet", math_default="exact", scaling="strong",
                    what="312 synthetic ScanNet-shape scenes, 8 shape classes 88x44x88/8 views .. 208x48x160/40 views, "
                         "LPT-sharded over the ranks, detections all_gathered over NCCL inside the timed region (cfg4)",
                    scenes=pool, scene_list=lst, chunks_default=312, graph_cache=8)
    if name == "cfg5":
        return dict(metric="scenes_per_sec_suncg_96x48x96_3img_fp16", cfgname="suncg", math_default="fp16", scaling="weak",
                    what="96x48x96 SUNCG-shape chunk, 3 views, SUNCG backbone, 26 classes, fp16-operand tensor-core convs (cfg5)",
                    scenes=[(5000 + rank * 64 + j, (96, 48, 96), 3) for j in range(24)], chunks_default=320)
    raise SystemExit(f"unknown --config {name}")


def case_of(wl, dims, n_img):
    return dict(cfgname=wl["cfgname"], dims=dims, n_img=n_img, seed=0, use_images=True, use_mask=True)


# ------------------------------------------------------------------------------------------------ helpers
def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), bf16_burst=float(p["bf16_tflops"]),
                    bf16_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    except Exception:
        return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


def measure_tf32_peak(dev):
    """cuBLAS TF32 GEMM (torch.matmul on fp32 tensors with allow_tf32), 8192^3, best of 10 -- the burst figure, which is
    the right denominator for a kernel timed in isolation."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(2):
            torch.matmul(a, b)
        best = float("inf")
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def sources_sha():
    """Hash of the kernel sources: profile-derived numbers (DRAM traffic) are only reported for the build they were taken on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "3d-sis_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def profile_traffic():
    """DRAM bytes from the committed ncu capture of THIS build (tools/ncu_traffic.py -> profiles/r2_traffic.json), else None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            t = json.load(f)
        return t if t.get("sources_sha") == sources_sha() else None
    except Exception:
        return None


def usable_cores():
    """Host threads this process may really use: affinity mask and cgroup CPU quota, not the box's core count."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


class Clocks:
    """nvidia-smi clock / throttle sampling during the timed region (one long-lived `-lms 100` process)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw"

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def summary(self):
        rows = []
        if self.proc is not None:
            try:
                self.proc.terminate()
                out, _ = self.proc.communicate(timeout=5)
                rows = [[t.strip() for t in ln.split(",")] for ln in out.splitlines() if ln.strip()]
            except Exception:
                pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in rows)]
        pw = [float(r[6]) for r in rows if len(r) > 6 and r[6].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(rows[0][1]) if rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(rows), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------ CPU arm
def reference_runner(wl):
    """The CPU implementation of the path: the torch-CPU oracle port of the reference (oracle/port.py, pinned to the
    unmodified reference by tests/test_oracle_golden.py) -- kind "port".  Returns (kind, run(seed, dims, n_img) -> seconds
    of one full forward)."""
    import sis3d_synth as synth
    from oracle import port
    ocfg = port.make_cfg(wl["cfgname"])
    w = synth.make_weights(seed=0, net=ocfg.NET, use_images=True, num_classes=ocfg.NUM_CLASSES, a1=ocfg.NUM_ANCHORS_LEVEL1,
                           a2=ocfg.NUM_ANCHORS_LEVEL2, use_mask=True)

    def run(seed, dims, n_img):
        data, boxes = synth.make_scene(seed, dims)
        v = synth.make_views(seed, dims, n_img, boxes, intrinsic=np.array(ocfg.INTRINSIC, dtype=np.float32))
        t0 = time.perf_counter()
        port.forward(ocfg, w, data, v)
        return time.perf_counter() - t0
    return "port", run


def best_threads(run, cores):
    """Thread count that is fastest for the CPU arm on this host (over-subscription makes intra-op threading slower, and
    the baseline should be the best the CPU can do): probed on a small scene."""
    best, best_t = cores, float("inf")
    for c in sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores}):
        torch.set_num_threads(c)
        run(7, (48, 32, 48), 2)
        dt = run(7, (48, 32, 48), 2)
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_arm(wl, seconds, min_scenes=1, max_scenes=10 ** 9):
    kind, run = reference_runner(wl)
    cores = best_threads(run, usable_cores())
    run(*wl["scenes"][0])  # warm
    ts, t0 = [], time.perf_counter()
    while len(ts) < min_scenes or (time.perf_counter() - t0 < seconds and len(ts) < max_scenes):
        ts.append(run(*wl["scenes"][len(ts) % len(wl["scenes"])]))
    what = "torch-CPU fp32 oracle port of the reference path"
    return dict(value=1.0 / float(np.mean(ts)), unit="scenes/s", cores=cores, kind=kind,
                sample=f"{len(ts)} full forwards of the workload's scenes in {sum(ts):.0f}s, {what}"), ts


def run_reference(args, rank, wl):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores, rank 0 only."""
    if rank != 0:
        return
    steps = max(1, args.steps if args.steps else 10)
    base, ts = cpu_arm(wl, 150.0, min_scenes=min(steps, 3), max_scenes=steps)
    ms = 1e3 * float(np.mean(ts))
    v = 1e3 / ms
    base["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": wl["metric"], "value": v, "unit": "scenes/s", "n_gpus": args.gpus, "steps": len(ts),
        "warmup": 1, "ms_per_step": ms, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["what"], "weights": "seeded synthetic", "threads": base["cores"],
                   "step": "one full forward of one scene of the workload (bounded sample, <= 150 s in total)"},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, scenes):
    """What the scene loop handed its caller for each scene of one step, in loop order, as the caller stores it
    (lib/model/trainval.py save_scene_results): the [n, 16] detection table (box, score, class, mask keep, crop, count) and
    the thresholded predicted-class mask of every kept detection.  float32 / float64 .npy files, DUMP_BYTES in all: mask
    voxels beyond that are replaced by a fixed, seeded sample of them (mask_voxel_index)."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"detections": np.concatenate([d for d, _, _ in scenes]).astype(np.float32),
           "detections_per_scene": np.array([len(d) for d, _, _ in scenes], dtype=np.float64),
           "masks_per_scene": np.array([0 if s is None else len(s) for _, _, s in scenes], dtype=np.float64),
           "mask_sizes": np.concatenate([np.zeros((0, 3))] + [s for _, _, s in scenes if s is not None]).astype(np.float64)}
    bits = np.concatenate([np.zeros(0, np.uint8)] + [b for _, b, _ in scenes if b is not None])
    room = (DUMP_BYTES - 1024 * (len(out) + 2) - sum(a.nbytes for a in out.values())) // 4  # float32 slots; 1 KB per header
    if bits.size > room:  # a sampled voxel costs 12 bytes: its value (float32) and its index (float64)
        idx = np.sort(np.random.default_rng(0).choice(bits.size, room // 3, replace=False))
        out["mask_voxel_index"] = idx.astype(np.float64)
        bits = bits[idx]
    out["mask_voxels"] = bits.astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=0, help="timed steps (default 20; cfg3/cfg4: 5)")
    ap.add_argument("--chunks-per-step", type=int, default=0,
                    help="scenes per rank in one step = one pass of the scene loop (default: sized so 20 steps time >= 3 s)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="sis3d")
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--enet", action="store_true",
                    help="inputs are RGB frames [n,3,256,328]: the 2-D ENet encoder (SURVEY row f2) runs inside the timed region")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=20.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lean", action="store_true", help="profiling runs: timed loops only (no latency / parity / CPU legs)")
    ap.add_argument("--host-profile", type=int, default=0, help="cProfile one pass -> stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step handed to its caller (rank 0: detection tables and thresholded "
                         "masks of its scenes) as DIR/<name>.npy")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    wl = workload(args.config, rank, world)
    if args.impl == "reference":
        return run_reference(args, rank, wl)
    args.warmup = max(args.warmup, 3)
    if not args.steps:
        args.steps = 20 if args.config in ("cfg2", "cfg5", "cfg3s") else 5
    if "graph_cache" in wl:
        os.environ.setdefault("SIS3D_GRAPH_CACHE", str(wl["graph_cache"]))

    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import sis3d_synth as synth
    from lib import _sis3d as S
    from lib.model.scene_shard import gather_detections, shard_scenes
    math = os.environ.get("SIS3D_CONV_MATH", wl["math_default"])
    s0 = wl["scenes"][0]
    st = dict(net=synth.make_net(case_of(wl, s0[1], s0[2]), keep_debug=False, math=math, enet=args.enet)[0])

    # distinct scenes rotate so that the inputs of consecutive scenes exceed the 126 MB L2: host (pinned) and device copies
    host_in, dev_in = [], []
    for seed, dims, n_img in wl["scenes"]:
        data, boxes = synth.make_scene(seed, dims)
        views = synth.make_views(seed, dims, n_img, boxes)
        if args.enet:  # normalised RGB frames instead of ENet-shaped features (lib/datasets/dataset.py:255-266)
            views["feats"] = np.random.default_rng(seed + 7).standard_normal((n_img, 3, 256, 328)).astype(np.float32)
        hb = synth.make_blobs(None, data, views, pin=True)
        host_in.append(hb)
        dev_in.append({"data": hb["data"].to(dev), "id": hb["id"],
                       "nearest_images": {"images": [hb["nearest_images"]["images"][0].to(dev)],
                                          "depths": [hb["nearest_images"]["depths"][0].to(dev)],
                                          "poses": hb["nearest_images"]["poses"], "world2grid": hb["nearest_images"]["world2grid"]}})

    def in_bytes(hb):
        return sum(t.numel() * t.element_size() for t in [hb["data"]] + [v[0] for v in hb["nearest_images"].values()])
    n_in = len(host_in)
    if "scene_list" in wl:   # cfg4: this rank's LPT share of the fixed 312-scene list (strong scaling)
        costs = [float(np.prod(wl["scenes"][k][1])) * (1 + wl["scenes"][k][2] / 40.0) for k in wl["scene_list"]]
        mine = shard_scenes(costs, rank, world)
        st["order"] = [wl["scene_list"][i] for i in mine]
    else:
        mine = None
        nb = max(1, args.chunks_per_step or wl["chunks_default"])
        st["order"] = [i % n_in for i in range(nb)]
    B = len(st["order"])
    l2_bytes = sum(in_bytes(host_in[k]) for k in sorted(set(st["order"])))

    def timed_loop(inputs, steps):
        """`steps` passes of the scene loop (Network.forward_pipelined, 7 scenes in flight) over this rank's scenes; every
        scene's detections and thresholded predicted-class masks are read back to the host.  CUDA events on the default
        stream bracket the region (it waits for the slot streams), barrier + synchronize on both sides, max over ranks."""
        net, order = st["net"], st["order"]
        # rank-0-only sections (after the other ranks have left: parity, other math modes) must not touch a collective
        multi = world > 1 and not st.get("solo", False)
        d2h = 0
        k0 = net.kernel_launches()
        if multi:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dets = []
        for _ in range(steps):
            local_det, st["last"] = [], []
            for j, (_, P) in enumerate(net.forward_pipelined(inputs[k] for k in order)):
                det = P["detections_host"]  # results of this scene are on the host: detection table + thresholded masks
                d2h += det.nbytes + (P["mask_bits_host"].nbytes if "mask_bits_host" in P else 0)
                dets.append(det)
                st["last"].append((det, P.get("mask_bits_host"), P.get("mask_sizes")))
                if mine is not None:
                    t = torch.from_numpy(det)
                    local_det.append((mine[j], t[:, :6], t[:, 7], t[:, 6]))
            if mine is not None and multi:  # cfg4: every rank ends a pass with all scenes' detections (NCCL all_gather)
                allres = gather_detections(local_det, device=dev)
                assert len(allres) == len(wl["scene_list"])
        for sl in net._slots:
            if sl["stream"] is not None:
                torch.cuda.current_stream().wait_stream(sl["stream"])
        e1.record()
        torch.cuda.synchronize()
        if multi:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if multi:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vox = nroi = nmask = 0
        for det in dets:  # workload statistics, outside the timed region
            k = det[det[:, 8] > 0.5]
            vox += int(((k[:, 12] - k[:, 9]) * (k[:, 13] - k[:, 10]) * (k[:, 14] - k[:, 11])).sum())
            nroi += det.shape[0]
            nmask += k.shape[0]
        n = max(1, len(dets))
        return float(t.item()), net.kernel_launches() - k0, d2h / n, vox / n, nroi / n, nmask / n

    def latency(inputs, steps):
        ts = []
        for i in range(steps):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st["net"].forward(inputs[st["order"][i % B]], "TEST", None)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    for i in range(args.warmup):
        st["net"].forward(dev_in[st["order"][i % B]], "TEST", None)
    wsteps = max(1, min(args.warmup, max(1, 64 // B)))
    timed_loop(dev_in, wsteps)   # warm-up passes; also capture the graphs of the pipeline slots
    timed_loop(host_in, wsteps)
    if args.host_profile and rank == 0 and world == 1:  # (a rank-0-only pass would wait at the barrier forever)
        import cProfile
        import io
        import pstats
        pr = cProfile.Profile()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pr.enable()
        timed_loop(host_in, 1)
        pr.disable()
        wall = (time.perf_counter() - t0) / B * 1e3
        buf = io.StringIO()
        pstats.Stats(pr, stream=buf).sort_stats("tottime").print_stats(40)
        print(f"wall ms per scene (pipelined loop, host inputs, under cProfile): {wall:.3f}\n" + buf.getvalue(), file=sys.stderr)
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    ms_dev, launches, _, vox, nroi, nmask = timed_loop(dev_in, args.steps)
    last_step = st["last"]
    ms_e2e, _, d2h, _, _, _ = timed_loop(host_in, args.steps)
    clock_summary = clocks.summary() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_step)
    n_scenes = args.steps * B  # scenes per rank inside each timed region
    total_scenes = n_scenes
    if world > 1:
        tot = torch.tensor([float(n_scenes)], dtype=torch.float64, device=dev)
        dist.all_reduce(tot)
        total_scenes = int(tot.item())

    # pinned-host -> device copy bandwidth of this box (explains the gap between `value` and `e2e`)
    probe_h = torch.empty(64 << 20, dtype=torch.uint8, pin_memory=True)
    probe_d = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
    probe_d.copy_(probe_h, non_blocking=True)
    torch.cuda.synchronize()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for _ in range(8):
        probe_d.copy_(probe_h, non_blocking=True)
    pe1.record()
    torch.cuda.synchronize()
    h2d_gbs = 8 * (64 << 20) / (pe0.elapsed_time(pe1) * 1e-3) / 1e9
    del probe_h, probe_d
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    st["solo"] = True  # from here on rank 0 works alone: no collective may be issued (the other ranks are gone)
    # single-GPU properties (latency, parity rate, other math modes, mask-heavy point, CPU arm) are reported by the N = 1 line only
    extras = not args.lean and world == 1
    lat_dev = latency(dev_in, 30) if extras else None
    lat_host = latency(host_in, 30) if extras else None

    # dominant tensor-core kernel, timed live through the C ABI: rpn_net_level{1,2} = 3x3x3 conv 128 -> 256 on the 24x12x24
    # level grid (12.231 GFLOP algorithmic), 40 back-to-back launches between two CUDA events on the launching stream
    # (inputs 3.5 MB: L2-resident, as in the forward where the producer has just written them), in the math of this run
    import ctypes as C
    net = st["net"]
    rx = torch.randn(24, 12, 24, 128, device=dev)
    rw = torch.randn(256, 128, 3, 3, 3, device=dev) * 0.02
    rb = torch.zeros(256, device=dev)
    ro = torch.empty(24, 12, 24, 256, device=dev)
    sh = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    h3 = net._math == "f16x3"
    x3 = net._math in ("tf32x3", "f16x3")
    wp = torch.empty(512 if x3 else 256, 27 * 128, device=dev, dtype=torch.float16 if h3 else torch.float32)
    S.check((S.lib.sis3d_pack_conv_weight_tc_h3 if h3 else S.lib.sis3d_pack_conv_weight_tc_x3 if x3
             else S.lib.sis3d_pack_conv_weight_tc)(S.ptr(rw), 256, 128, 3, S.ptr(wp), sh), "pack")

    def rpn_conv():
        if x3:
            S.check((S.lib.sis3d_conv3d_k3_tc_h3 if h3 else S.lib.sis3d_conv3d_k3_tc_x3)(
                S.ptr(rx), S.ptr(wp), S.ptr(rb), None, 0, 0, S.ptr(ro), 256, 0, 24, 12, 24, 128, 256, 3, 1, sh), "rpn conv x3")
        else:
            S.check(S.lib.sis3d_conv3d_k3_tc(S.ptr(rx), S.ptr(wp), S.ptr(rb), None, 0, 0, S.ptr(ro), 256, 0, 24, 12, 24, 128, 256, 3,
                                             None, 0, 1, sh), "rpn conv")
    for _ in range(5):
        rpn_conv()
    ke0, ke1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ke0.record()
    for _ in range(40):
        rpn_conv()
    ke1.record()
    torch.cuda.synchronize()
    rpn_ms = ke0.elapsed_time(ke1) / 40
    pk = peaks()
    tf32_peak = measure_tf32_peak(dev)
    mma_peak = pk["bf16_burst"] if (h3 or net._math == "fp16") else tf32_peak  # the tensor-pipe rate this kernel's MMAs run at
    traffic = profile_traffic()
    value = total_scenes / (ms_dev / 1e3)
    e2e_v = total_scenes / (ms_e2e / 1e3)
    per_gpu = value / world
    per_scene_ms = ms_dev / n_scenes
    order = st["order"]
    dims0 = wl["scenes"][order[0]][1]
    mean_alg = float(np.mean([alg_bytes(wl["scenes"][k][1], wl["cfgname"]) for k in order])) + MASK_BYTES_PER_VOXEL * vox
    mean_flops = float(np.mean([flops(wl["scenes"][k][1], wl["cfgname"]) for k in order])) + 0.894e6 * vox
    tf = 12.231e9 / (rpn_ms * 1e-3) / 1e12
    issued = tf * (3 if x3 else 1)
    tensor_roof = {
        "bound": "tensor",
        "kernel": f"conv3d_k3_tc_kernel<128,3{',X3=2' if h3 else ',X3=1' if x3 else ''}> (rpn_net_level1/2: 3x3x3, 128 -> 256 ch, 24x12x24; "
                  + ("error-compensated fp16 split: three tcgen05 kind::f16 MMAs per algorithmic product" if h3 else
                     "error-compensated 3xTF32: three tcgen05 MMAs per algorithmic product" if x3 else "TF32 in") + ", fp32 accumulate)",
        "achieved": tf, "peak": mma_peak, "unit": "TFLOP/s", "frac": tf / mma_peak,
        "peak_note": ("measured bf16/fp16 GEMM burst peak of MEASURED_PEAKS.json (the kernel's MMAs are kind::f16)" if mma_peak != tf32_peak
                      else "cuBLAS TF32 GEMM 8192^3 measured in this run (burst, best of 10)") + "; the kernel is timed in isolation; "
                     "`achieved` counts ALGORITHMIC flops, `issued_mma_tflops` the 3x MMA work of the compensated product",
        "flops_per_launch": 12.231e9, "ms_per_launch": rpn_ms, "launches_timed": 40,
        "issued_mma_tflops": issued, "issued_frac": issued / mma_peak,
        "traffic": traffic.get("rpn_kernel_dram_bytes_per_launch") if traffic else None,
        "traffic_note": "dram__bytes_read+write per launch, ncu --set full capture of this build (profiles/r2_traffic.json)"
                        if traffic else "null: no ncu capture of this exact build (sources hash) is committed"}
    dtype = {"exact": "f16 hi/lo split, error-compensated 3-MMA products (static-stage convs: fp32-class accuracy) / f16 operands (mask-stage convs) on tcgen05, fp32 accumulate, + f32",
             "f16x3": "f16 hi/lo split, error-compensated 3-MMA products (static stage) / tf32 (mask stage) on tcgen05, fp32 accumulate, + f32",
             "tf32x3": "3xTF32 error-compensated (static stage) / tf32 (mask stage) on tcgen05, fp32 accumulate, + f32",
             "tf32": "tf32 (convs on tcgen05, fp32 accumulate) + f32",
             "mixed": "tf32 (static-stage convs) / f16 operands (mask-stage convs) on tcgen05, fp32 accumulate, + f32",
             "fp16": "f16 operands (convs on tcgen05, fp32 accumulate) + f32"}.get(math, "f32")
    have_traffic = bool(traffic) and args.config == "cfg2" and traffic.get("forward_dram_bytes_per_scene")
    out = {
        "metric": wl["metric"] + ("_with_enet" if args.enet else ""), "value": value, "unit": "scenes/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
        "dtype": dtype, "data": "synthetic",
        "config": {"workload": wl["what"] + (" + 2-D ENet encoder on raw RGB frames (row f2)" if args.enet else ""), "conv_math": math,
                   "inputs": ("seeded synthetic TSDF + RGB frames [n,3,256,328]/depth/poses; seeded synthetic weights" if args.enet else
                              "seeded synthetic TSDF + ENet-shaped features/depth/poses; seeded synthetic weights"),
                   "l2": f"{len(set(order))} distinct scenes per rank rotate: {l2_bytes / 1e6:.0f} MB of inputs > 126 MB L2 (no flush kernel)",
                   "api": "Network.forward_pipelined (the scene loop; 7 scenes in flight on 7 streams: inputs uploaded one "
                          "scene ahead, 4 static stages overlapping)",
                   "scenes_per_step_per_rank": B, "step": f"one pass of the scene loop over {B} scenes per rank",
                   "rois_per_scene": nroi, "mask_rois_per_scene": nmask, "mask_voxels_per_scene": vox,
                   "scenes_per_rank": n_scenes, "timed_seconds": ms_dev / 1e3,
                   "parallelism": f"scene-sharded dp{world}" + (" (LPT by voxel count)" if mine is not None else "")},
        "e2e": {"value": e2e_v, "unit": "scenes/s", "h2d_bytes_per_step": float(np.mean([in_bytes(host_in[k]) for k in order])) * B,
                "d2h_bytes_per_step": d2h * B, "ms_per_step": ms_e2e / args.steps, "ms_per_scene": ms_e2e / n_scenes,
                "timed_seconds": ms_e2e / 1e3, "h2d_probe_gbs": round(h2d_gbs, 1),
                "what": "same loop from pinned HOST buffers: H2D of scene+features+depth+poses and D2H of detections + "
                        "thresholded predicted-class masks inside the timed region"},
        "latency_ms": {"sync_forward_device_inputs": lat_dev, "sync_forward_host_inputs": lat_host,
                       "note": "median of single synchronous Network.forward calls (no overlap between scenes)"},
        "gpu_launches": launches,
        # SURVEY 8(d): fraction of the 3D-conv HBM roofline = ALG_BYTES x scenes/s per GPU / HBM peak.  ALG_BYTES are the
        # per-layer compulsory fp32 bytes of the reference's dataflow; the fused/sparse design moves far fewer, so the
        # physically meaningful fractions are given next to it: measured DRAM traffic and algorithmic FLOPs.
        "roofline": {"bound": "hbm", "achieved": mean_alg * per_gpu / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                     "frac": mean_alg * per_gpu / 1e9 / pk["hbm"], "peak_source": pk["source"],
                     "traffic": traffic["forward_dram_bytes_per_scene"] if have_traffic else None,
                     "traffic_note": ("dram__bytes_read+write summed over the launches of one cfg2 scene, ncu --set full capture of "
                                      "this build (profiles/r2_traffic.json; caches flushed per kernel -> upper bound)")
                     if have_traffic else "null: no ncu capture of this exact build/config is committed",
                     "kernel": "whole forward = all libsis3d launches of one scene (graph replay + ragged mask stage)",
                     "algorithmic_bytes_per_scene": mean_alg, "gpu_ms_per_scene": per_scene_ms,
                     "dram_frac": (traffic["forward_dram_bytes_per_scene"] * per_gpu / 1e9 / pk["hbm"]) if have_traffic else None,
                     "algorithmic_tflops": mean_flops * per_gpu / 1e12,
                     "flop_frac_of_tf32_sustained": mean_flops * per_gpu / 1e12 / (tf32_peak * pk["bf16_sustained"] / pk["bf16_burst"]),
                     "note": "whole-step fractions use the sustained peak scale (long step), the isolated kernel below the burst "
                             "peak; per-kernel times and shares: profiles/ (ncu launch list + --set full capture)"},
        "roofline_tensor_kernel": tensor_roof,
        "peaks": {"hbm_gbs": pk["hbm"], "bf16_tflops_burst": pk["bf16_burst"], "bf16_tflops_sustained": pk["bf16_sustained"],
                  "tf32_tflops_burst_measured_here": tf32_peak, "source": pk["source"]},
        "clocks": clock_summary,
    }
    if extras:
        # ---- parity of THIS math mode on THESE inputs: fraction of scenes whose integer outputs equal the fp32 CUDA-core path
        from lib.utils.parity import parity_rate
        uniq = sorted(set(order))[:24]
        by_shape = {}
        for k in uniq:
            by_shape.setdefault((wl["scenes"][k][1], wl["scenes"][k][2]), []).append(dev_in[k])
        exact = n = 0
        fields, flips = {}, []
        for (dims, n_img), bl in by_shape.items():
            mk = lambda mode, d=dims, v=n_img: synth.make_net(case_of(wl, d, v), keep_debug=False, math=mode, enet=args.enet)[0]  # noqa: E731
            r, _ = parity_rate(mk, bl, math)
            exact += r["exact_scenes"]
            n += r["scenes"]
            for f, c in r["first_mismatch_fields"].items():
                fields[f] = fields.get(f, 0) + c
            if r["thresholded_mask_voxel_flip_fraction"] is not None:
                flips.append(r["thresholded_mask_voxel_flip_fraction"])
        out["parity_rate"] = {"value": exact / max(n, 1), "scenes": n, "exact_scenes": exact, "against": "fp32 CUDA-core mode "
                              "(pinned bit-exact to the unmodified reference on the golden cases by tests/test_gpu_forward.py)",
                              "compared": "proposal count + order, level ids, class argmax, mask-keep flags, crop bounds",
                              "first_mismatch_fields": fields,
                              "thresholded_mask_voxel_flip_fraction": float(np.mean(flips)) if flips else None}
        # ---- throughput of the other math modes on the same loop (short passes): fp32 CUDA-core path and the fast TF32 mode
        others = {}
        keep_net, keep_order = st["net"], st["order"]
        for m in ("fp32", "mixed"):
            if m == math:
                continue
            nn_ = min(B, 48 if m == "fp32" else 192)
            st["net"], st["order"] = synth.make_net(case_of(wl, s0[1], s0[2]), keep_debug=False, math=m, enet=args.enet)[0], keep_order[:nn_]
            try:
                timed_loop(dev_in, 1)
                ms_o = timed_loop(dev_in, 2)[0]
                others[m] = {"value": 2 * nn_ / (ms_o / 1e3), "unit": "scenes/s", "scenes_timed": 2 * nn_, "n_gpus": 1,
                             "what": "same scene loop, device-resident inputs, rank 0 only"}
            finally:
                st["net"], st["order"] = keep_net, keep_order
        out["other_math_modes"] = others
        # ---- mask-heavy workload point: 10 RoIs of 54x22x22 (SURVEY 8(a10) sizes a real RoI like this), mask stage only
        det = np.zeros((10, 16), dtype=np.float32)
        rngm = np.random.default_rng(0)
        for i in range(10):
            x0, y0, z0 = (int(rngm.integers(0, dims0[a] - s + 1)) for a, s in ((0, 54), (1, 22), (2, 22)))
            det[i, 7], det[i, 8], det[i, 9:15] = 1 + i, 1.0, (x0, y0, z0, x0 + 54, y0 + 22, z0 + 22)
        scene_t = dev_in[order[0]]["data"]
        for _ in range(3):
            net._mask_branch(scene_t, det, 10)
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for _ in range(10):
            net._mask_branch(scene_t, det, 10)
        m1.record()
        torch.cuda.synchronize()
        mh = m0.elapsed_time(m1) / 10
        mvox = 10 * 54 * 22 * 22
        out["mask_heavy"] = {"rois": 10, "crop": [54, 22, 22], "mask_voxels": mvox, "ms": mh,
                             "algorithmic_tflops": 0.894e6 * mvox / (mh * 1e-3) / 1e12,
                             "what": "ragged mask stage alone (plan + 6 layers + select) on 10 RoIs of 54x22x22, teacher-forced table"}
    if extras and not args.no_cpu_baseline:
        # the CPU arm runs in a process of its own (the same code path as `--impl reference`); only if that fails is it timed
        # in this process
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config", args.config,
                                "--steps", "6", "--warmup", "1"], capture_output=True, text=True, timeout=400,
                               env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
            out["cpu_baseline"] = json.loads(line)["cpu_baseline"]
        except Exception as e:
            print(f"[bench] reference subprocess failed ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
            out["cpu_baseline"], _ = cpu_arm(wl, args.cpu_baseline_seconds)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
