#!/usr/bin/env python3
"""bench.py — camera frames/s @1080p multi-task on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python bench.py --steps K --dump-outputs DIR   # also write the last timed step's outputs (dump_outputs)
    python bench.py --autospeed ...      # row f.4: the AutoSpeed detector, 1080p frame -> boxes
    python bench.py --config5 ...        # row e: multi-camera all-gather + fusion, one rank per camera (torchrun)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one 1920x1080 RGB camera frame through the whole hot path: fused pre-process
(Pillow-bicubic resize + normalise) -> shared encoder -> SceneSeg / Scene3D / DomainSeg / EgoLanes
heads -> per-pixel post-process (BASELINE.json configs[2]; at N GPUs, N independent camera streams,
one per GPU, no data-path collective: configs[3], weak scaling).

Lines printed by rank 0:
  value      frames/s with the frames already resident in HBM (a pool of distinct frames larger
             than L2 is cycled so no step re-reads its input from cache), CUDA-event timed;
  e2e        the same metric through the reference-facing C-ABI call vp_engine_infer with pinned
             HOST frames: H2D of the frame + kernels + D2H of the masks/depth inside the timed
             region; also the p50 / p95 pre-proc->masks latency;
  roofline   the dominant kernel (the tensor-core kernel with the most device time per frame): ALGORITHMIC 2*MAC per
             launch (SURVEY.md 8d: of the reference graph's layers the launch computes) / mean launch duration, all its
             launches of the frame issued back to back for >= 2 s between one CUDA-event pair (vp_engine_time_kernel),
             against the measured SUSTAINED cuBLAS bf16 peak; achieved_executed / frac_executed = the same with the MACs
             the kernel actually executes (the composed ConvTranspose->Conv3x3 GEMM runs 44 % of the reference's);
             roofline.stages = one entry per kernel of the frame (HBM-bound ones against the measured copy peak);
  cpu_baseline  the oracle (CPU fp32 port of the reference's PyTorch path: PIL resize -> 4 networks
             -> post-process) on the host cores, a bounded sample, N=1 only.
  --impl reference  times that CPU path alone with all host threads (the reference's own
             implementation of the path is PyTorch-on-CPU; /root/reference is not on the GPU box,
             so the port in oracle/ — validated bit-equal against it — is what runs).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H_IN, W_IN = 1080, 1920
MODELS = ("scene_seg", "scene_3d", "domain_seg", "ego_lanes")
GFLOP_MT = 1153.25      # SURVEY.md §8d: algorithmic GFLOP / frame, shared-encoder multi-task
POOL_FRAMES = 24        # 24 x 6.22 MB = 149 MB > 126 MB L2


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"tflops_burst": d.get("bf16_tflops"), "tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "src": "measured"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "src": "fallback"}


def load_traffic(kernel):
    """Average DRAM bytes per launch of the dominant kernel from the newest committed ncu capture of THAT kernel
    (profiles/r*_traffic*.json, produced by scripts/ncu_conv_traffic.sh).  STATIC: read from the committed file, not
    measured in this run (ncu cannot run inside a timed bench)."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*traffic*.json")), reverse=True):
        with open(path) as f:
            d = json.load(f)
        if d.get("kernel") == kernel:
            return d.get("avg_dram_bytes"), os.path.relpath(path, ROOT)
    return None, None


TENSOR_KERNELS = ("conv_gemm_kernel", "conv3x3_lin_kernel", "conv3x3_pair_kernel", "conv3x3_splitk_kernel",
                  "convt_ws_kernel", "upconv_pair_kernel")


def stage_rooflines(eng, peaks):
    """One entry per kernel of the frame: all its launches issued back to back 20x between one CUDA-event pair
    (vp_engine_time_kernel).  HBM-bound stages: algorithmic bytes (SURVEY.md 8d: tensors in + out) / time against
    the measured HBM copy peak; tensor stages: algorithmic 2*MAC (SURVEY.md 8d: of the REFERENCE graph's layers the
    launches stand for) / time against the measured cuBLAS bf16 BURST peak (these are short isolated bursts).  The
    composed ConvTranspose->Conv3x3 GEMM executes fewer MACs than the reference layers it replaces: its row carries
    both figures (achieved = algorithmic, achieved_executed = what the tensor pipe actually does)."""
    st = eng.stats()
    extra_ref = max(0.0, st["reference_flops"] - st["total_flops"])      # per frame, all of it in upconv_pair_kernel
    rows, total_us = [], 0.0
    for k in eng.kernel_names():
        r = eng.time_kernel_name(k, reps=20)
        if r["launches"] == 0:
            continue
        us_frame = 1e3 * r["ms"] / 20
        total_us += us_frame
        tensor = k in TENSOR_KERNELS
        ach_exec = None
        if tensor:
            ach_exec = r["flops"] / (r["ms"] / 1e3) / 1e12
            fl = r["flops"] + (20 * extra_ref if k == "upconv_pair_kernel" else 0.0)
            ach, peak, unit = fl / (r["ms"] / 1e3) / 1e12, peaks["tflops_burst"], "TFLOP/s"
        else:
            ach, peak, unit = r["bytes"] / (r["ms"] / 1e3) / 1e9, peaks["hbm_gbs"], "GB/s"
        row = {"kernel": k, "bound": "tensor" if tensor else "hbm", "launches_per_frame": r["launches"] // 20,
               "us_per_frame": us_frame, "achieved": ach, "peak": peak, "unit": unit,
               "frac": ach / peak if peak else None}
        if k == "upconv_pair_kernel":
            row["achieved_executed"] = ach_exec
            row["frac_executed"] = ach_exec / peak if peak else None
        rows.append(row)
    for row in rows:
        row["share_of_kernel_time"] = row["us_per_frame"] / total_us if total_us else None
    return rows, total_us


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (one persistent
    `nvidia-smi -lms 100` child, killed by its own PID afterwards)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if line.strip():
                    self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


def usable_cpus() -> int:
    """Host threads this process may really use: affinity mask and cgroup CPU quota, not os.cpu_count()."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, n)


def pick_cpu_threads(sds, frame) -> int:
    """The CPU path is timed with the thread count that is fastest on this host (a 128-thread pool
    on a quota-limited container is ~20x slower than 8 threads): one SceneSeg forward per candidate."""
    import torch
    from oracle import net
    x = net.to_tensor_normalize(np.ascontiguousarray(frame[:320, :640]))
    best, best_t = 1, float("inf")
    cap = usable_cpus()
    for n in sorted({c for c in (4, 8, 16, 32, 64, cap) if c <= cap}):
        torch.set_num_threads(n)
        t = time.time()
        net.forward("scene_seg", sds["scene_seg"], x)
        t = time.time() - t
        if t < best_t:
            best, best_t = n, t
        elif t > 2.0 * best_t:
            break
    torch.set_num_threads(best)
    return best


def make_checkpoints(tmpdir: str):
    """Seeded synthetic checkpoints (no network access for the real ones) -> .vpw files."""
    from autoware_vision_pilot_b200 import weights as W
    from oracle import synth
    paths, sds = [], {}
    for m in MODELS:
        sd = synth.synth_state_dict(m)
        sds[m] = sd
        paths.append(W.write_vpw(sd, os.path.join(tmpdir, f"{m}.vpw")))
    return paths, sds


def dump_outputs(eng, out_dir):
    """What the engine's last frame returned to its caller, as float32 .npy files (6 MB in all):
    <model>_raw.npy = the fp32 NCHW tensor (logits, depth, lane masks), <model>_cls.npy = the class / mask map
    (absent for Scene3D)."""
    os.makedirs(out_dir, exist_ok=True)
    for i, m in enumerate(MODELS):
        eng.fetch_raw(i)                   # D2H on the engine's stream, after that frame, then a sync
        np.save(os.path.join(out_dir, f"{m}_raw.npy"), eng.raw(i).astype(np.float32))
        cls = eng.cls(i)
        if cls is not None:
            np.save(os.path.join(out_dir, f"{m}_cls.npy"), cls.astype(np.float32))


def cpu_reference_frame(sds, frame):
    """The reference's CPU path for one frame, multi-task the way the reference runs it (one
    helper per model, nothing shared): PIL bicubic resize -> ToTensor/Normalize -> network ->
    post-process (Models/inference/*_infer.py)."""
    import torch
    from PIL import Image
    from oracle import net
    small = np.asarray(Image.fromarray(frame).resize((640, 320)))
    outs = []
    for m in MODELS:
        x = net.to_tensor_normalize(small)
        outs.append(net.postprocess(m, net.forward(m, sds[m], x)))
    return outs


def run_reference(args, rank, world):
    if rank != 0:
        return
    import torch
    from oracle import synth
    sds = {m: synth.synth_state_dict(m) for m in MODELS}
    frames = [synth.synth_frame(i) for i in range(2)]
    nthreads = pick_cpu_threads(sds, frames[0])
    budget_s = 120.0
    t0 = time.time()
    cpu_reference_frame(sds, frames[0])
    t_first = time.time() - t0
    warm = max(0, min(args.warmup, int(20.0 / max(t_first, 1e-3))) - 1)
    for i in range(warm):
        cpu_reference_frame(sds, frames[i % 2])
    steps = max(1, min(args.steps, int(budget_s / max(t_first, 1e-3))))
    ts = []
    for i in range(steps):
        t = time.time()
        cpu_reference_frame(sds, frames[i % 2])
        ts.append(time.time() - t)
    fps = steps / sum(ts)
    line = {
        "impl": "reference", "metric": "camera frames/sec @1080p multi-task", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "steps_executed": steps,
        "ms_per_step": 1e3 / fps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "1080p multi-task (SceneSeg+Scene3D+DomainSeg+EgoLanes), CPU PyTorch fp32, "
                               "one helper per model as the reference runs it", "frame": [H_IN, W_IN, 3]},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": nthreads, "kind": "port",
                         "sample": f"{steps} frames x 4 networks, torch {torch.__version__} fp32, "
                                   f"{nthreads} threads = fastest of the candidates on this host "
                                   f"({usable_cpus()} usable CPUs, os.cpu_count()={os.cpu_count()}); capped to ~{int(budget_s)} s"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "p50_latency_ms": statistics.median(ts) * 1e3,
    }
    print(json.dumps(line), flush=True)


def run_config5(args, rank, local_rank, world):
    """BASELINE.json configs[4] (SURVEY.md 8e; an extension — the reference's PathFinder is single-camera):
    every rank = one camera: 1080p frame -> EgoLanes (fused pre-process, encoder, 1456-channel feature fusion,
    context, neck, head) -> lane masks -> device LaneFilter/LaneTracker/PathFinder measurement -> ONE ncclAllGather
    of (fused features 582 400 B + measurement 224 B) per rank, issued from C++ (vp_b200_multicam.h) -> Estimator
    fusion of the `world` measurements on every rank.  All of it is enqueued on one stream per rank."""
    import ctypes as C
    import tempfile
    import torch
    import torch.distributed as dist
    from autoware_vision_pilot_b200 import _lib as L
    from autoware_vision_pilot_b200 import engine as E
    from autoware_vision_pilot_b200 import lateral, multicam
    from autoware_vision_pilot_b200 import weights as W
    from oracle import synth   # synthetic frames / weights only

    dev = torch.device("cuda", local_rank)
    tmp = tempfile.mkdtemp(prefix="vpb_bench5_")
    vpw = W.write_vpw(synth.synth_state_dict("ego_lanes"), os.path.join(tmp, f"ego_{rank}.vpw"))
    stream = torch.cuda.Stream()
    eng = E.Engine([E.EGO_LANES], [vpw], gpu_id=local_rank, dtype=args.dtype, resize_mode=E.RESIZE_PIL_BICUBIC,
                   convention=E.CONV_RGB, fetch_raw=False, use_graph=True, stream=stream.cuda_stream)
    uid = multicam.exchange_unique_id(rank, dev) if world > 1 else multicam.make_unique_id()
    mc = multicam.MultiCamera(uid, rank, world, local_rank, stream=stream.cuda_stream)
    lat = lateral.LateralPostProcess(device=f"cuda:{local_rank}")
    lib = L.lib()
    lib.vpb_lane_masks.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_void_p]
    masks = torch.zeros((3, 80, 160), dtype=torch.float32, device=dev)
    host_frames = [synth.synth_frame(synth.stream_seed(rank, f)) for f in range(4)]
    pool = torch.empty((POOL_FRAMES, H_IN, W_IN, 3), dtype=torch.uint8, device=dev)
    for i in range(POOL_FRAMES):
        pool[i].copy_(torch.from_numpy(np.roll(host_frames[i % 4], 37 * i, axis=1)))
    torch.cuda.synchronize()
    raw_dev = eng.out_dev(0)[0]

    def step(i):
        eng.infer_device(pool[i % POOL_FRAMES].data_ptr(), H_IN, W_IN, W_IN * 3)
        L.check(lib.vpb_lane_masks(raw_dev, 3 * 80 * 160, 0.0, masks.data_ptr(), stream.cuda_stream), "vpb_lane_masks")
        lat.update_device(masks.data_ptr(), 80, 160, stream=stream.cuda_stream)
        mc.step_engine(eng, 0, lat._out.data_ptr(), predict=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(i)
    torch.cuda.synchronize()
    timed_steps = args.steps
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(timed_steps):
        step(i)
    e1.record(stream)
    barrier()
    ms = multicam.max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop()
    barrier()
    ag_us = multicam.max_over_ranks(mc.time_allgather(200), dev)
    feats, meas, state = mc.read()
    stats = eng.stats()
    mc.close()
    if rank != 0:
        return
    fps = world * timed_steps / (ms / 1e3)
    print(json.dumps({
        "metric": "camera frames/sec @1080p EgoLanes + multi-camera PathFinder fusion (config 5)", "value": fps,
        "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "timed_steps": timed_steps,
        "timed_region_s": ms / 1e3, "ms_per_step": ms / timed_steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16" if args.dtype == "fp16" else "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE configs[4]: per GPU one 1080p camera -> EgoLanes -> lane masks -> device "
                               "LaneFilter/LaneTracker/PathFinder measurement -> ONE ncclAllGather (C++, 582 624 B per rank) "
                               "-> Estimator fusion of all cameras on every rank",
                   "frame": [H_IN, W_IN, 3], "payload_bytes_per_rank": multicam.PAYLOAD_BYTES,
                   "l2": f"{POOL_FRAMES} distinct device-resident frames cycled (149 MB > L2)"},
        "allgather": {"us_per_call": ag_us, "bytes_per_rank": multicam.PAYLOAD_BYTES, "world": world,
                      "algbw_gbs": multicam.PAYLOAD_BYTES * world / (ag_us * 1e-6) / 1e9 if ag_us > 0 else None,
                      "how": "200 back-to-back ncclAllGather calls between one CUDA-event pair, max over ranks"},
        "fused_state_cte_yaw_curv": [state[3].tolist(), state[7].tolist(), state[11].tolist()],
        "cameras_with_measurement": int((~np.isnan(meas[:, 1, 0]) | ~np.isnan(meas[:, 2, 0])).sum()),
        "gpu_launches": (stats["n_launches"] + 4) * timed_steps, "clocks": clocks}), flush=True)


def run_autospeed(args, rank, local_rank, world):
    """SURVEY.md 8f rank 4: the AutoSpeed detector (letterbox -> YOLO-style network with CTX / C3K2 / SPPF / PSA attention
    -> DFL decode -> confidence filter + NMS) on 1080p frames; N>1 = one camera stream per GPU (independent frames)."""
    import tempfile
    import torch
    import torch.distributed as dist
    from autoware_vision_pilot_b200 import autospeed as AS
    from autoware_vision_pilot_b200 import multicam
    from autoware_vision_pilot_b200 import weights as W
    from oracle import autospeed as O      # synthetic weights + the CPU baseline leg only
    from oracle import synth
    dev = torch.device("cuda", local_rank)
    sd = O.synth_state_dict()
    vpw = W.write_vpw(sd, os.path.join(tempfile.mkdtemp(prefix="vpb_bench_as_"), f"autospeed_{rank}.vpw"))
    stream = torch.cuda.Stream()
    eng = AS.AutoSpeedEngine(vpw, gpu_id=local_rank, dtype=args.dtype, stream=stream.cuda_stream)
    host_frames = [synth.synth_frame(synth.stream_seed(rank, f)) for f in range(4)]
    pool = torch.empty((POOL_FRAMES, H_IN, W_IN, 3), dtype=torch.uint8, device=dev)
    for i in range(POOL_FRAMES):
        pool[i].copy_(torch.from_numpy(np.roll(host_frames[i % 4], 37 * i, axis=1)))
    torch.cuda.synchronize()

    def step(i):
        eng.infer_device(pool[i % POOL_FRAMES].data_ptr(), H_IN, W_IN, W_IN * 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(i)
    torch.cuda.synchronize()
    timed_steps = args.steps
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(timed_steps):
        step(i)
    e1.record(stream)
    barrier()
    ms = multicam.max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop()
    # end to end: pageable-host frame in, detections on the host (H2D + kernels + D2H + sync per frame)
    n_e2e = max(20, min(args.steps, 200))
    for i in range(3):
        eng.infer(host_frames[i % 4])
    barrier()
    t0 = time.time()
    lat = []
    for i in range(n_e2e):
        t = time.time()
        det = eng.infer(host_frames[i % 4])
        lat.append(time.time() - t)
    e2e_s = time.time() - t0
    stats = eng.stats()
    if rank != 0:
        return
    fps = world * timed_steps / (ms / 1e3)
    line = {"metric": "camera frames/sec @1080p AutoSpeed detector", "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "timed_steps": timed_steps, "timed_region_s": ms / 1e3,
            "ms_per_step": ms / timed_steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16" if args.dtype == "fp16" else "bf16", "data": "synthetic",
            "config": {"workload": "AutoSpeed 'n' (4 classes) on 1080p frames: letterbox 1024x512 -> network -> DFL decode -> "
                                   "confidence 0.6 + NMS 0.45 (Models/inference/auto_speed_infer.py)",
                       "gflop_per_frame": stats["flops"] / 1e9, "launches_per_frame": stats["n_launches"],
                       "weights": "seeded synthetic state_dict (oracle/autospeed.py)",
                       "l2": f"{POOL_FRAMES} distinct device-resident frames cycled (149 MB > L2)"},
            "e2e": {"value": world * n_e2e / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": H_IN * W_IN * 3,
                    "d2h_bytes_per_step": 1024 * 6 * 4 + 8, "p50_latency_ms": 1e3 * sorted(lat)[len(lat) // 2],
                    "how": "vp_autospeed_infer from host frames (H2D + kernels + D2H + sync), one frame at a time, wall clock"},
            "detections_last_frame": int(len(det)), "gpu_launches": stats["n_launches"] * timed_steps, "clocks": clocks}
    if world == 1 and not args.no_cpu_baseline:
        import torch as _t
        _t.set_num_threads(min(16, usable_cpus()))
        O.inference(sd, host_frames[0])
        ts = []
        while len(ts) < 40 and sum(ts) < 15.0:
            t = time.time()
            O.inference(sd, host_frames[len(ts) % 4])
            ts.append(time.time() - t)
        line["cpu_baseline"] = {"value": len(ts) / sum(ts), "unit": "frames/s", "cores": min(16, usable_cpus()), "kind": "port",
                                "sample": f"{len(ts)} frames, oracle/autospeed.py fp32 (pinned against the reference module)"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--dtype", default="fp16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--single-stream", action="store_true", help="disable the concurrent per-model lanes")
    ap.add_argument("--config5", action="store_true",
                    help="BASELINE configs[4]: per rank EgoLanes + device lateral post-process, ONE ncclAllGather of the "
                         "fused features + PathFinder measurements (C++, vp_b200_multicam.h), Estimator fusion")
    ap.add_argument("--autospeed", action="store_true", help="SURVEY 8f.4: the AutoSpeed detector instead of the 4-task frame")
    ap.add_argument("--inflight", type=int, default=4,
                    help="camera frames in flight per GPU (engine replicas on separate streams; the next "
                         "frame's latency-bound encoder overlaps the current frame's decoders)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (every model's fp32 tensor and "
                         "class / mask map) as DIR/<model>_{raw,cls}.npy, float32; the multi-task benchmark only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.autospeed or args.config5):
        ap.error("--dump-outputs applies to the multi-task benchmark only")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import tempfile
    import torch
    import torch.distributed as dist
    from autoware_vision_pilot_b200 import engine as E
    from autoware_vision_pilot_b200 import multicam
    from oracle import synth   # synthetic frames / weights only; never on the measured path

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.autospeed:
        run_autospeed(args, rank, local_rank, world)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.config5:
        run_config5(args, rank, local_rank, world)
        if world > 1:
            dist.destroy_process_group()
        return

    tmp = tempfile.mkdtemp(prefix="vpb_bench_")
    paths, sds = make_checkpoints(tmp)
    kinds = [E.KIND_BY_NAME[m] for m in MODELS]
    n_eng = max(1, args.inflight)
    streams = [torch.cuda.Stream() for _ in range(n_eng)]
    engs = [E.Engine(kinds, paths, gpu_id=local_rank, dtype=args.dtype, resize_mode=E.RESIZE_PIL_BICUBIC,
                     convention=E.CONV_RGB, fetch_raw=False, use_graph=True, stream=st.cuda_stream,
                     single_stream=args.single_stream) for st in streams]
    eng, stream = engs[0], streams[0]
    # camera stream `rank`: frames seeded 1000*rank + f (SURVEY.md §8d)
    host_frames = [synth.synth_frame(synth.stream_seed(rank, f)) for f in range(4)]
    pool = torch.empty((POOL_FRAMES, H_IN, W_IN, 3), dtype=torch.uint8, device="cuda")
    for i in range(POOL_FRAMES):
        pool[i].copy_(torch.from_numpy(np.roll(host_frames[i % 4], 37 * i, axis=1)))
    torch.cuda.synchronize()

    def step(i):
        engs[i % n_eng].infer_device(pool[i % POOL_FRAMES].data_ptr(), H_IN, W_IN, W_IN * 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def elapsed_all(start, ends):
        return max(start.elapsed_time(e) for e in ends)

    for i in range(max(args.warmup, 2 * n_eng)):
        step(i)
    torch.cuda.synchronize()
    timed_steps = args.steps

    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e0.record(streams[0])
    for st in streams[1:]:
        st.wait_event(e0)
    for i in range(timed_steps):
        step(i)
    ends = []
    for st in streams:
        e = torch.cuda.Event(enable_timing=True)
        e.record(st)
        ends.append(e)
    barrier()
    ms = elapsed_all(e0, ends)
    ms = multicam.max_over_ranks(ms, torch.device("cuda", local_rank))
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # before the end-to-end runs below overwrite the engines' outputs
        dump_outputs(engs[(timed_steps - 1) % n_eng], args.dump_outputs)

    # ---- end to end through the C-ABI with pinned host frames (H2D + kernels + D2H per step)
    # (a) latency: one engine, synchronous per frame
    pinned = [g.pinned_frame(H_IN, W_IN) for g in engs]
    for k, g in enumerate(engs):
        for i in range(3):
            pinned[k][...] = host_frames[i % 4]
            g.infer(pinned[k])
    barrier()
    n_e2e = max(20, min(args.steps, 200))
    evs = []
    for i in range(n_e2e):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        eng.infer(pinned[0])               # H2D + graph + D2H + stream sync
        b.record(stream)
        evs.append((a, b))
    barrier()
    lat = sorted(a.elapsed_time(b) for a, b in evs)
    # (b) throughput: the same per-frame work (H2D + kernels + D2H) with `inflight` frames in
    # flight: frame i is submitted to engine replica i % inflight after that replica's previous frame
    # has completed (vp_engine_submit / vp_engine_sync)
    f0 = torch.cuda.Event(enable_timing=True)
    f_ends = [torch.cuda.Event(enable_timing=True) for _ in engs]
    per = n_e2e // n_eng + 1
    f0.record(streams[0])
    for st in streams[1:]:
        st.wait_event(f0)
    for i in range(per * n_eng):
        k = i % n_eng
        if i >= n_eng:
            engs[k].sync()                 # frame i - inflight is complete, its host outputs are readable
        engs[k].submit(pinned[k])
    for k in range(n_eng):
        engs[k].sync()
        f_ends[k].record(streams[k])
    barrier()
    e2e_ms = multicam.max_over_ranks(elapsed_all(f0, f_ends), torch.device("cuda", local_rank))
    n_e2e_frames = per * n_eng
    d2h = 0
    for i, m in enumerate(MODELS):
        c, h, w = eng.out_dev(i)[2]
        if m in ("scene_seg", "domain_seg"):
            d2h += h * w
        elif m == "scene_3d":
            d2h += c * h * w * 4
        else:
            d2h += c * h * w * 4 + h * w

    # ---- roofline: every kernel's launches of one frame issued back to back between ONE CUDA-event pair
    # (vp_engine_time_kernel; no per-launch events or launch gaps inside the figure)
    peaks = load_peaks()
    stages, stages_us = stage_rooflines(eng, peaks)
    tens = [r for r in stages if r["bound"] == "tensor"]
    dom = max(tens, key=lambda r: r["us_per_frame"])["kernel"]
    # the dominant kernel again, now for >= 2 s of back-to-back launches: a SUSTAINED measurement (clocks and power
    # settle like in the long step), so the sustained cuBLAS peak is its denominator
    one = eng.time_kernel_name(dom, reps=5)
    reps_sus = max(10, int(np.ceil(2000.0 / max(one["ms"] / 5, 1e-3))))
    sus = eng.time_kernel_name(dom, reps=reps_sus)
    gemm_ms, gemm_fl, n_gemm = sus["ms"], sus["flops"], sus["launches"]
    all_us = sum(r["us_per_frame"] for r in tens)
    all_fl = sum(r.get("achieved_executed", r["achieved"]) * 1e12 * r["us_per_frame"] / 1e6 for r in tens)
    stats = eng.stats()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    fps = world * timed_steps / (ms / 1e3)
    e2e_fps = world * n_e2e_frames / (e2e_ms / 1e3)
    executed = gemm_fl / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    peak = peaks["tflops_sustained"]
    traffic, traffic_src = load_traffic(dom)
    # FLOPs the reference's layer-by-layer graph spends on what the fused ConvTranspose->Conv3x3 launches compute
    extra_ref = max(0.0, stats["reference_flops"] - stats["total_flops"]) if dom == "upconv_pair_kernel" else 0.0
    dom_per_frame = next(r["launches_per_frame"] for r in stages if r["kernel"] == dom)
    # SURVEY.md 8d: roofline.achieved counts the ALGORITHMIC FLOPs of the reference graph's layers these launches compute
    achieved = (gemm_fl + extra_ref * n_gemm / max(dom_per_frame, 1)) / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    line = {
        "metric": "camera frames/sec @1080p multi-task", "value": fps, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / timed_steps, "higher_is_better": True,
        "timed_steps": timed_steps, "timed_region_s": ms / 1e3,
        "timing": f"{timed_steps} steps back to back inside ONE device-timed region, max over ranks",
        "scaling": "weak", "vs_baseline": None, "dtype": "f16" if args.dtype == "fp16" else "bf16",
        "data": "synthetic",
        "config": {"workload": "1080p multi-task: SceneSeg+Scene3D+DomainSeg+EgoLanes, shared encoder "
                               "(BASELINE.json configs[2]); N>1 = one camera stream per GPU (configs[3])",
                   "frame": [H_IN, W_IN, 3], "net_input": [320, 640], "resize": "pil_bicubic (fused)",
                   "weights": "seeded synthetic state_dicts (oracle/synth.py)",
                   "l2": f"{POOL_FRAMES} distinct device-resident frames cycled (149 MB > L2); weights+activations "
                         f"{(stats['weight_bytes'] + stats['act_bytes']) / 1e6:.0f} MB",
                   "gflop_per_frame_algorithmic": GFLOP_MT, "gflop_per_frame_reference_graph": stats["reference_flops"] / 1e9,
                   "gflop_per_frame_executed": stats["total_flops"] / 1e9,
                   "shared_encoders": stats["shared_encoders"], "shared_trunks": stats["shared_trunks"],
                   "frames_in_flight_per_gpu": n_eng},
        "clocks": clocks,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": H_IN * W_IN * 3,
                "d2h_bytes_per_step": d2h,
                "how": f"vp_engine_infer (H2D + kernels + D2H + sync) from pinned host frames; throughput with "
                       f"{n_eng} frames in flight (vp_engine_submit on {n_eng} engine replicas); latency = one engine, one frame at a time",
                "p50_latency_ms": lat[len(lat) // 2], "p95_latency_ms": lat[int(len(lat) * 0.95)]},
        "gpu_launches": stats["n_launches"] * timed_steps,
        "launches_per_frame": stats["n_launches"],
        "tensor_tflops_whole_step": GFLOP_MT * fps / world / 1e3,
        "roofline": {"bound": "tensor", "kernel": f"{dom} (tcgen05 implicit-GEMM convolution)",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                     "flops_counted": "achieved / frac: ALGORITHMIC 2*MAC of the reference graph's layers these launches compute "
                                      "(SURVEY.md 8d); achieved_executed / frac_executed: the 2*MAC the kernel actually "
                                      "executes (the composed ConvTranspose->Conv3x3 GEMM runs 44 % of the reference "
                                      "layers' MACs for the same outputs, DESIGN.md 3e) = the tensor-pipe utilisation",
                     "achieved_executed": executed,
                     "frac_executed": executed / peak if peak else None,
                     "peak_src": f"{peaks['src']} bf16 cuBLAS, SUSTAINED: the kernel is timed over {gemm_ms / 1e3:.1f} s of "
                                 "back-to-back launches",
                     "frac_vs_burst_peak": achieved / peaks["tflops_burst"] if peaks["tflops_burst"] else None,
                     "burst_peak": peaks["tflops_burst"],
                     "launches_timed": n_gemm,
                     "share_of_kernel_time": next(r["share_of_kernel_time"] for r in stages if r["kernel"] == dom),
                     "traffic": traffic, "traffic_src": f"STATIC, {traffic_src} (ncu --set full of an earlier run of this "
                                                        "kernel; not measured in this run)" if traffic_src else None,
                     "flop_per_launch": achieved * 1e12 * (gemm_ms / 1e3) / max(n_gemm, 1),
                     "flop_per_launch_executed": gemm_fl / max(n_gemm, 1), "us_per_launch": 1e3 * gemm_ms / max(n_gemm, 1),
                     "all_tensor_kernels": {"achieved_executed": all_fl / (all_us / 1e6) / 1e12 if all_us else None,
                                            "us_per_frame": all_us},
                     "stages": stages, "stages_serial_us_per_frame": stages_us,
                     "how": "dominant kernel = the tensor-core kernel with the largest back-to-back device time per frame; "
                            "achieved = algorithmic 2*MAC of all its launches of the frame / their device time, issued "
                            f"back to back {reps_sus}x between one CUDA-event pair on the engine stream "
                            "(vp_engine_time_kernel); stages[] = the same for every kernel of the frame (20 reps, "
                            "isolated bursts: tensor stages against the burst peak, HBM stages = algorithmic bytes / time "
                            "against the measured copy bandwidth); share_of_kernel_time = the kernel's serial device time / "
                            "the sum over all kernels (what an ncu launch list measures)"},
    }
    if world == 1 and not args.no_cpu_baseline:
        import torch as _t
        nthreads = pick_cpu_threads(sds, host_frames[0])
        cpu_reference_frame(sds, host_frames[0])        # warm-up
        ts = []
        t_budget = time.time()
        while len(ts) < 8 and time.time() - t_budget < 25.0:
            t = time.time()
            cpu_reference_frame(sds, host_frames[len(ts) % 4])
            ts.append(time.time() - t)
        cfps = len(ts) / sum(ts)
        line["cpu_baseline"] = {"value": cfps, "unit": "frames/s", "cores": nthreads, "kind": "port",
                                "sample": f"{len(ts)} frames x 4 networks (PIL resize + oracle fp32 forward + "
                                          f"post-process), torch {_t.__version__}, {nthreads} threads (fastest "
                                          f"candidate; {usable_cpus()} usable CPUs)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
