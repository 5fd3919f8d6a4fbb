#!/usr/bin/env python
"""bench.py -- images/sec of the YOLO forward hot path on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5                       # our CUDA path, one JSON line
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                           # one rank per GPU, images sharded
    python bench.py --impl reference --steps 3 --warmup 1                # the reference's own CPU path

A "step" is one forward pass of the network over one batch of synthetic images per GPU (workload = BASELINE.json
configs[1]: yolov3.cfg at 608x608, FP32-semantics convolutions, batch 16 per GPU; weak scaling: images are
independent, every rank runs its own batch, the only collective is ONE broadcast of the prepared weight arena at
init).  `value` = images processed by all ranks / max-over-ranks device time with inputs resident in HBM;
`e2e` = the same through the public predict call with pinned host buffers (H2D of the images and D2H of the
activated detection tensors inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (model builder key, size, per-GPU batch, quantized rule)
    "yolov3-608-fp32-b16": ("yolov3", 608, 16, 0),
    "yolov3-spp-608-fp32-b16": ("yolov3-spp", 608, 16, 0),
    "yolov3-tiny-416-int8-b64": ("yolov3-tiny", 416, 64, 1),
    "tiny-yolo-obj_xnor-416-b64": ("tiny-yolo-obj_xnor", 416, 64, 0),
    "yolov3-tiny-416-fp32-b1": ("yolov3-tiny", 416, 1, 0),
}
DEFAULT_WORKLOAD = "yolov3-608-fp32-b16"


def conv_flops(sections, batch):
    """Sum 2*n*k*k*c*out_h*out_w over convolutions == the reference's own `bflops` (additionally.c:2903)."""
    from yolo2_light_b200 import cfgs
    tot = 0
    for L in cfgs.conv_shapes(sections):
        if L["type"] in ("convolutional", "conv"):
            tot += 2 * L["n"] * L["size"] ** 2 * L["c"] * L["out_h"] * L["out_w"]
    return tot * batch


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every ~5 ms DURING the timed region (the nvidia-smi recipe of
    B200_PROFILING.md is too coarse for a ~0.2 s region); falls back to `nvidia-smi -lms` when pynvml is missing."""
    REASONS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}

    def __init__(self, gpu_index):
        self.gpu, self.samples, self.stop_flag, self.thread, self.max_mhz = gpu_index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[0].isdigit() else self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def loop():
                while not self.stop_flag:
                    try:
                        mhz = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                        try:
                            mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        except Exception:
                            mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.samples.append((time.time(), float(mhz), int(mask)))
                    except Exception:
                        pass
                    time.sleep(0.004)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def stop(self, t0, t1):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        sel = [(m, k) for ts, m, k in self.samples if t0 <= ts <= t1]
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        reasons = sorted(name for name, bit in self.REASONS.items() if any(k & bit for _, k in sel))
        return {"sm_mhz": float(np.median([m for m, _ in sel])), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sel)}


def host_cpu_info():
    """Usable hardware threads (affinity mask AND cgroup quota), physical cores among them, sockets, CPU model."""
    aff = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    model, cores, sockets = "unknown", set(), set()
    try:
        cur = {}
        for line in open("/proc/cpuinfo"):
            if ":" in line:
                k, v = [t.strip() for t in line.split(":", 1)]
                cur[k] = v
            elif not line.strip():
                if cur and int(cur.get("processor", -1)) in aff:
                    cores.add((cur.get("physical id", "0"), cur.get("core id", cur.get("processor"))))
                    sockets.add(cur.get("physical id", "0"))
                    model = cur.get("model name", model)
                cur = {}
    except Exception:
        pass
    threads = len(aff)
    if quota:
        threads = max(1, min(threads, int(quota + 0.5)))
    phys = max(1, min(len(cores) or threads, threads))
    return {"threads": threads, "physical_cores": phys, "sockets": max(1, len(sockets)), "model": model,
            "affinity": len(aff), "cgroup_quota": quota}


def reference_cpu_rate(cfg, wts, q, x1, n_images, max_seconds=40.0):
    """images/s of the reference's own CPU forward (oracle/_ref) on this box.  ONE code path for `--impl reference` and for
    `cpu_baseline`: OpenMP placement is pinned (OMP_PROC_BIND=close, OMP_PLACES=cores, set before the library loads), the
    thread count is set explicitly with omp_set_num_threads (torchrun exports OMP_NUM_THREADS=1, which the reference would
    silently inherit), the candidates {physical cores, one socket, every usable thread} are each tried on one image and the
    best is timed on `n_images`.  Returns (images/s, description dict)."""
    import ctypes
    info = host_cpu_info()
    os.environ["OMP_PROC_BIND"] = "close"
    os.environ["OMP_PLACES"] = "cores"
    os.environ["OMP_NUM_THREADS"] = str(info["threads"])
    os.environ.setdefault("OMP_WAIT_POLICY", "active")
    from oracle import ref
    kind = "fast" if ref.available("fast") else "scalar"
    rnet = ref.RefNet(cfg, wts, 1, q, 7, kind=kind)
    gomp = None
    if kind == "fast":
        try:
            gomp = ctypes.CDLL("libgomp.so.1")
        except OSError:
            gomp = None
    cands = sorted({info["threads"], info["physical_cores"], max(1, info["physical_cores"] // info["sockets"])}, reverse=True)
    if gomp is None:
        cands = [info["threads"] if kind == "fast" else 1]
    t_start = time.time()
    rnet.time_predict(x1, 1)          # first call: page faults on ~600 MB of buffers (SURVEY section 6)
    trial = {}
    for n in cands:
        if gomp is not None:
            gomp.omp_set_num_threads(int(n))
        trial[n] = rnet.time_predict(x1, 1)
        if time.time() - t_start > max_seconds * 0.6:
            break
    best = min(trial, key=trial.get)
    if gomp is not None:
        gomp.omp_set_num_threads(int(best))
    t = rnet.time_predict(x1, max(1, n_images))
    desc = {"cores": int(best) if kind == "fast" else 1, "kind": "reference", "cpu_model": info["model"],
            "usable_threads": info["threads"], "physical_cores": info["physical_cores"], "sockets": info["sockets"],
            "threads_tried": {str(k): round(1.0 / v, 4) for k, v in trial.items()},
            "build": "reference sources, AVX=1 OPENMP=1 -Ofast (oracle/_ref)" if kind == "fast" else "reference sources, scalar -O2",
            "omp": "OMP_PROC_BIND=close OMP_PLACES=cores, omp_set_num_threads(best)"}
    return 1.0 / t, desc


def traffic_per_launch(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per k_conv_tc launch, averaged over the launches of one step, from
    the committed ncu capture (profiles/r01_traffic.json, made with tools/ncu_traffic.sh); None when not captured."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            v = d.get(workload, {}).get("dram_bytes_per_launch")
            if v is not None:
                return v
        except Exception:
            pass
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(outdir, outputs):
    """What the timed path hands its caller -- the detection tensors [batch, ...] of one step -- as <outdir>/yolo_l<i>.npy
    (float32).  Inputs and weights are seeded, so two builds can be compared file by file.  A batch larger than DUMP_BYTES
    is cut to its leading images, the same ones on every run."""
    os.makedirs(outdir, exist_ok=True)
    per_image = sum(o[0].nbytes for o in outputs.values())
    keep = max(1, DUMP_BYTES // per_image)
    for i, o in outputs.items():
        np.save(os.path.join(outdir, f"yolo_l{i}.npy"), np.ascontiguousarray(o[:keep], np.float32))


def reference_run(args, workload):
    """`--impl reference`: the reference's own CPU implementation (oracle/_ref/libyolo2ref_fast.so = its sources
    compiled with the flags its Makefile recommends, AVX=1 OPENMP=1) on this box's host cores, batch 1 as its CLI
    runs it (main.c:160).  One step = one image."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from yolo2_light_b200 import cfgs
    model, size, batch, q = WORKLOADS[workload]
    secs = cfgs.MODELS[model](size, size)
    wd = tempfile.mkdtemp(prefix="yb_ref_")
    cfg = cfgs.write_cfg(secs, os.path.join(wd, "m.cfg"))
    wts = cfgs.write_weights(secs, os.path.join(wd, "m.weights"), seed=1)
    x = cfgs.synthetic_images(1, 3, size, size)
    val, desc = reference_cpu_rate(cfg, wts, q, x, max(args.steps, 1))
    t = 1.0 / val
    desc = dict(desc, value=val, unit="images/sec",
                sample=f"{max(args.steps, 1)} single-image forwards after warm-up and a thread-count trial")
    line = {
        "impl": "reference", "metric": "images/sec", "value": val, "unit": "images/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if not q else "s8", "data": "synthetic",
        "config": {"workload": workload, "model": model, "input": f"{size}x{size}", "batch_per_step": 1,
                   "rule": "network_predict_quantized" if q else "network_predict_cpu"},
        "cpu_baseline": desc,
        "e2e": {"value": val, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-images", type=int, default=4)
    ap.add_argument("--det-thresh", type=float, default=0.0,
                    help="objectness threshold of the end-to-end detection path; 0 (default) = the lowest threshold >= 0.5 at which no\n"
                         "image yields more than 300 candidates: random-init heads sit at logit ~0, so the reference's demo default\n"
                         "0.24 would pass every one of the 22743 boxes of every image")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the detection tensors of the last one as DIR/<name>.npy (float32, "
                         "at most 64 MB: a larger batch is cut to its leading images)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        reference_run(args, args.workload)
        return

    import torch
    import torch.distributed as dist

    import yolo2_light_b200 as yb
    from yolo2_light_b200 import cfgs

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this framework has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    model, size, batch, q = WORKLOADS[args.workload]
    secs = cfgs.MODELS[model](size, size)
    tag = os.environ.get("MASTER_PORT", "0")
    wd = os.path.join(tempfile.gettempdir(), f"yb_bench_{tag}_{os.getuid()}")
    cfg, wts = os.path.join(wd, "m.cfg"), os.path.join(wd, "m.weights")
    if rank == 0:
        os.makedirs(wd, exist_ok=True)
        cfgs.write_cfg(secs, cfg)
        cfgs.write_weights(secs, wts, seed=1)
    if world > 1:
        dist.barrier()

    # ---- model preparation: the reference's main.c:160-171 sequence -------------------------------------
    net = yb.parse_network_cfg(cfg, batch, q)
    if rank == 0:
        yb.load_weights_upto_cpu(net, wts)   # other ranks receive the prepared arena by broadcast
    yb.yolov2_fuse_conv_batchnorm(net)
    yb.calculate_binary_weights(net)
    if q:
        yb.quantinization_and_get_multipliers(net)
    net.set_device(local_rank)
    ptr, nbytes = net.weight_arena(quantized=bool(q), upload=(rank == 0))
    if world > 1:
        from yolo2_light_b200 import parallel
        arena = parallel.arena_tensor(ptr, nbytes, torch.device("cuda", local_rank))   # zero-copy view of the engine's arena
        parallel.broadcast_arena(arena, src=0)   # the ONLY collective of the whole job (NCCL over NVLink)
        torch.cuda.synchronize()

    # ---- inputs resident in HBM: 4 rotating batches (> L2 together with ~4 GB of activations per step) ----
    nrot = 4
    host_batches = [cfgs.synthetic_images(batch, 3, size, size, seed=1234 + (rank * nrot + r) * batch) for r in range(nrot)]
    dev_batches = [torch.from_numpy(h).cuda() for h in host_batches]
    tstream = torch.cuda.Stream()            # a real (non-default) stream: kernels, events and graphs all live on it
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def step(i):
        net.forward_device(dev_batches[i % nrot].data_ptr(), quantized=bool(q), stream=stream)

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    launches_per_step = net.last_launches()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record()
    for i in range(args.steps):
        step(i)
    ev1.record()
    torch.cuda.synchronize()
    t_wall1 = time.time()
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    tmax = torch.tensor([ms], device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total = float(tmax.item())
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    net.sync_outputs(quantized=bool(q), stream=stream)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, net.detection_outputs())
    sanity = {i: float(np.abs(o).mean()) for i, o in net.detection_outputs().items()}
    if not all(np.isfinite(v) and v > 0 for v in sanity.values()):
        raise SystemExit(f"bench.py: non-finite / empty detection outputs {sanity}")

    # ---- end to end through the public serving call (the reference app's loop, main.c:188-229, as one pipelined call per
    # batch): 8-bit frames in pinned host memory -> H2D + the reference's resize on the device -> forward -> decode + NMS on
    # the device (under the next batch's forward) -> candidate rows back to the host.  Three batches in flight.
    det_thresh, det_nms, det_cap = args.det_thresh, 0.45, 4096
    rng = np.random.default_rng(4321 + rank)
    frames = []
    for k in range(3):
        pb = yb.PinnedBuffer(batch * size * size * 3, dtype=np.uint8)
        pb.array[:] = rng.integers(0, 256, size=batch * size * size * 3, dtype=np.uint8)
        frames.append(pb)
    fshape = (batch, size, size, 3)
    if args.det_thresh <= 0:
        # untrained heads sit at logit ~0 (objectness ~0.5 everywhere): raise the threshold until an image yields at most a few
        # hundred candidates, which is what a trained detector hands to the NMS; outside every timed region
        net.predict_image_u8(frames[0].array.reshape(fshape), quantized=bool(q))
        det_thresh = 0.5
        while det_thresh < 0.95:
            _, cnts = net.detect(size, size, det_thresh, det_nms, max_rows=det_cap, quantized=bool(q))
            if int(cnts.max()) <= 300:
                break
            det_thresh = round(det_thresh + 0.01, 2)
    e2e_steps = max(6, min(args.steps, 30))
    e2e_stats = {"rows": 0, "d2h": 0, "maxcount": 0}

    def run_detect_pipeline(nsteps):
        inflight = []

        def take():
            dets, counts, moved = net.collect_detections(inflight.pop(0), quantized=bool(q), copy=False)
            e2e_stats["rows"] += int(sum(d.shape[0] for d in dets))
            e2e_stats["d2h"] += moved
            e2e_stats["maxcount"] = max(e2e_stats["maxcount"], int(counts.max()))
        for k in range(nsteps):
            if len(inflight) == 3:
                take()
            inflight.append(net.submit_u8(frames[k % 3].array.reshape(fshape), det_thresh, det_nms, max_rows=det_cap, quantized=bool(q)))
        while inflight:
            take()

    run_detect_pipeline(4)
    if world > 1:
        dist.barrier()
    e2e_stats.update(rows=0, d2h=0, maxcount=0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run_detect_pipeline(e2e_steps)
    t_e2e = time.perf_counter() - t0

    # the same loop with float images in and the raw yolo tensors out (round 1's e2e: 71 MB in / 124 MB out per batch)
    pinned = [yb.PinnedBuffer(batch * 3 * size * size) for _ in range(3)]
    for k, pb in enumerate(pinned):
        pb.array[:] = host_batches[k].ravel()

    def run_pipelined(nsteps):
        inflight = []
        for k in range(nsteps):
            if len(inflight) == 3:
                net.collect(inflight.pop(0), quantized=bool(q))
            inflight.append(net.submit(pinned[k % 3].array, quantized=bool(q)))
        while inflight:
            net.collect(inflight.pop(0), quantized=bool(q))

    run_pipelined(3)
    raw_steps = max(4, e2e_steps // 2)
    t0 = time.perf_counter()
    run_pipelined(raw_steps)
    t_raw = (time.perf_counter() - t0) / raw_steps
    t0 = time.perf_counter()
    nsync = max(3, e2e_steps // 3)
    for k in range(nsync):
        net.predict(pinned[k % 3].array, quantized=bool(q))
    t_sync = (time.perf_counter() - t0) / nsync
    te = torch.tensor([t_e2e, t_raw, t_sync], device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    t_e2e, t_raw, t_sync = float(te[0].item()), float(te[1].item()), float(te[2].item())
    h2d = batch * size * size * 3
    d2h = int(e2e_stats["d2h"] / max(e2e_steps, 1))
    raw_h2d = batch * 3 * size * size * 4
    raw_d2h = int(sum(o.size for o in net.detection_outputs().values()) * 4)

    # ---- decode + NMS alone (synchronous yb_network_detect on the tensors of the last forward) and what the pipeline exposes
    decode = None
    if rank == 0:
        try:
            net.predict(pinned[0].array, quantized=bool(q))
            net.detect(size, size, det_thresh, det_nms, max_rows=det_cap, quantized=bool(q))
            t0 = time.perf_counter()
            for _ in range(5):
                dets, counts = net.detect(size, size, det_thresh, det_nms, max_rows=det_cap, quantized=bool(q))
            t_det = (time.perf_counter() - t0) / 5
            decode = {"ms_per_batch_sync": t_det * 1e3, "thresh": det_thresh, "nms": det_nms, "max_rows": det_cap,
                      "candidates_per_image": e2e_stats["rows"] / max(1, e2e_steps * batch),
                      "max_candidates_in_an_image": e2e_stats["maxcount"],
                      "exposed_ms_per_batch_in_pipeline": max(0.0, t_e2e / e2e_steps * 1e3 - ms_total / args.steps),
                      "note": "random-init heads sit at logit ~0: the reference's demo threshold 0.24 would pass all 22743 boxes of "
                              "every image; thresh = the lowest value >= 0.5 at which no image yields more than 300 candidates, which is "
                              "what a trained detector hands to the NMS"}
        except Exception as e:
            decode = {"error": str(e)}

    # ---- the drop-in as a maintainer would build it: the reference's UNMODIFIED host code + integration/..._glue.c + the engine
    # (oracle/_ref/libyolo2ref_dropin.so), batch 1 like the reference CLI: network_predict_b200 (+ get_network_boxes_nms_b200)
    dropin = None
    if rank == 0 and world == 1:
        try:
            from oracle import ref
            if ref.available("dropin"):
                cfg1 = os.path.join(wd, "m_b1.cfg")
                cfgs.write_cfg(secs, cfg1)
                rnet = ref.RefNet(cfg1, wts, 1, q, 7, kind="dropin")
                x1 = host_batches[0][:1]
                rnet.time_predict_b200(x1, 3, decode=True, thresh=det_thresh, nms=det_nms)
                t_p = rnet.time_predict_b200(x1, 20, decode=False)
                t_pd = rnet.time_predict_b200(x1, 20, decode=True, thresh=det_thresh, nms=det_nms)
                dropin = {"predict_img_s": 1.0 / t_p, "predict_plus_device_decode_img_s": 1.0 / t_pd, "batch": 1,
                          "api": "network_predict_b200 + get_network_boxes_nms_b200 behind the reference's parser/loader (glue)"}
        except Exception as e:
            dropin = {"error": str(e)}

    # ---- roofline of the dominant kernel (tcgen05 implicit-GEMM conv), measured live with CUDA events ------
    roof = None
    if rank == 0:
        prof = net.profile(quantized=bool(q), d_input_ptr=dev_batches[0].data_ptr())
        by = {}
        for li, kind, t in prof:
            by.setdefault(kind, []).append((li, t))
        dom = max(by, key=lambda k: sum(t for _, t in by[k]))
        peaks, src = measured_peaks()
        shapes = cfgs.conv_shapes(secs)
        if dom in ("conv_tc", "conv_tc2", "conv_simt", "conv_tc_i8", "conv_int8", "conv_xnor"):
            fl = sum(2 * shapes[li]["n"] * shapes[li]["size"] ** 2 * shapes[li]["c"] * shapes[li]["out_h"] *
                     shapes[li]["out_w"] * batch for li, _ in by[dom])
            tsum = sum(t for _, t in by[dom]) * 1e-3
            ach = fl / tsum / 1e12
            peak = peaks.get("bf16_tflops_sustained", 1400.0)
            unit = "TFLOP/s"
            if dom in ("conv_tc_i8", "conv_int8"):
                # integer workloads: the denominator is the kind::i8 MMA rate measured on this pool (SURVEY 8d asks for it;
                # MEASURED_PEAKS.json only has bf16), scaled by what a real cuBLAS GEMM reaches of the bf16 MMA-only rate
                try:
                    ip = json.load(open(os.path.join(ROOT, "profiles", "r02_int8_peak.json")))
                    peak = ip["int8_tops_mma_only"] * peaks.get("bf16_tflops_sustained", 1393.7) / ip["bf16_tflops_mma_only"]
                    src = "kind::i8 MMA-only probe (profiles/r02_int8_peak.json) x cuBLAS-to-MMA-only bf16 ratio"
                    unit = "TOP/s"
                except Exception:
                    pass
            kname = {"conv_tc2": "k_conv_tc<2> (tcgen05 cta_group::2 implicit-GEMM conv)",
                     "conv_tc": "k_conv_tc<1> (tcgen05 implicit-GEMM conv)"}.get(dom, dom)
            all_tc = [(li, t) for k in ("conv_tc", "conv_tc2", "conv_tc_i8", "conv_tc_tf32") for li, t in by.get(k, [])]
            fl_all = sum(2 * shapes[li]["n"] * shapes[li]["size"] ** 2 * shapes[li]["c"] * shapes[li]["out_h"] *
                         shapes[li]["out_w"] * batch for li, _ in all_tc)
            t_all = sum(t for _, t in all_tc) * 1e-3
            roof = {"bound": "tensor", "kernel": kname, "achieved": ach, "peak": peak, "unit": unit,
                    "all_tensor_core_convs": {"achieved": fl_all / max(t_all, 1e-12) / 1e12, "launches": len(all_tc),
                                              "frac": fl_all / max(t_all, 1e-12) / 1e12 / peak,
                                              "share_of_step": t_all * 1e3 / sum(t for _, _, t in prof)},
                    "frac": ach / peak, "traffic": traffic_per_launch(args.workload), "launches": len(by[dom]),
                    "avg_launch_ms": tsum * 1e3 / len(by[dom]), "flops_per_launch": fl / len(by[dom]),
                    "share_of_step": tsum * 1e3 / sum(t for _, _, t in prof), "peak_source": src + " (sustained)"}

    # ---- CPU baseline: the reference's own forward on this box's cores (rank 0, N=1 only) ------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            n_img = args.cpu_baseline_images
            v, desc = reference_cpu_rate(cfg, wts, q, host_batches[0][:1], n_img)
            cpu = dict(desc, value=v, unit="images/sec",
                       sample=f"{n_img} single-image forwards of the same network after warm-up and a thread-count trial")
        except Exception as e:   # the checker must never take the bench down
            cpu = {"value": None, "unit": "images/sec", "cores": 0, "kind": "reference", "sample": f"failed: {e}"}

    if rank == 0:
        imgs = batch * world * args.steps
        value = imgs / (ms_total * 1e-3)
        line = {
            "metric": "images/sec", "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if not q else "s8", "data": "synthetic",
            "config": {"workload": args.workload, "model": model, "input": f"{size}x{size}", "batch_per_gpu": batch,
                       "global_batch": batch * world, "parallelism": f"dp{world} (images sharded, weights broadcast once)",
                       "weights": "random-init, seeded, BN folded", "l2": "inputs larger than L2: 4 rotating image "
                       "batches, ~4 GB of activations per step vs 126 MB L2",
                       "gflop_per_image": conv_flops(secs, 1) / 1e9},
            "e2e": {"value": batch * world * e2e_steps / t_e2e, "unit": "images/sec", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": "yb_network_submit_u8 / yb_network_collect_detections: 8-bit frames from pinned host memory -> device "
                           "resize -> forward -> device decode + NMS -> candidate rows on the host (3 batches in flight)",
                    "raw_tensors": {"value": batch * world / t_raw, "h2d_bytes_per_step": raw_h2d, "d2h_bytes_per_step": raw_d2h,
                                    "api": "yb_network_submit/collect: float images in, yolo tensors out"},
                    "sync_predict_value": batch * world / t_sync, "sync_predict_ms": t_sync * 1e3, "dropin": dropin},
            "gpu_launches": launches_per_step * args.steps * world,
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "device_decode": decode,
            "tflops": conv_flops(secs, batch * world) * args.steps / (ms_total * 1e-3) / 1e12,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
