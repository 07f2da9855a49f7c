#!/usr/bin/env python
"""Headline benchmark (BASELINE.json metric): frames/sec at 512x512 SD-Turbo 1-step img2img, stream-batch 1,
synthetic RGB frame feed, one independent video stream per GPU (weak scaling, NCCL weight broadcast at init
only, no per-step collective).

  python bench.py --gpus N --steps K --warmup W            # this repo (sm_100a engine through the public API)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (fp32 oracle on host cores)
  python bench.py --impl library --steps K ...             # torch fp16 library path (cuDNN + SDPA, CUDA graph) on the same GPU
  python bench.py --steps K --dump-outputs DIR             # also writes the last timed frame's output to DIR/output.npy

A "step" is one frame through StreamDiffusionPipeline.__call__.  `value` is timed on the device with the
input frame already resident in HBM; `e2e` includes, every step, the pinned-host -> device copy of the frame
and the device -> pinned-host read of the result.  Prints ONE JSON line on rank 0."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# workload table: BASELINE.json configs[1] is the default (the configuration the headline metric is quoted on);
# the others are the remaining single-GPU configs, selectable for additional measurements (--workload)
WORKLOADS = {
    "sd-turbo-512": dict(model="stabilityai/sd-turbo", t=[32], hw=512, gflop=1068.0,
                         metric="frames/sec at 512x512 SD-Turbo img2img (1-step, stream-batch 1)",
                         name="SD-Turbo 1-step img2img 512x512, stream-batch=1, synthetic RGB frame feed (BASELINE.json configs[1])"),
    "sd15-lcm4-512": dict(model="lykon/dreamshaper-8", t=[18, 26, 35, 45], hw=512, gflop=3476.9,
                          metric="frames/sec at 512x512 SD-1.5 + LCM 4-step img2img (stream-batch 4)",
                          name="SD-1.5 + LCM-LoRA 4-step img2img 512x512, stream-batch=4 (BASELINE.json configs[2])"),
    "sd15-lcm4-768": dict(model="lykon/dreamshaper-8", t=[18, 26, 35, 45], hw=768, gflop=9185.6,
                          metric="frames/sec at 768x768 SD-1.5 + LCM 4-step img2img (stream-batch 4)",
                          name="SD-1.5 + LCM-LoRA 4-step img2img 768x768, stream-batch=4, synthetic feed (BASELINE.json configs[4] without codecs)"),
}
MODEL_ID = "stabilityai/sd-turbo"
T_INDEX_LIST = [32]
H = W = 512
METRIC = WORKLOADS["sd-turbo-512"]["metric"]
GFLOP_PER_FRAME = 1068.0  # BASELINE.md section 3: 804.3 (UNet) + 122.3 (TAESD enc) + 141.4 (TAESD dec)
WORKLOAD = WORKLOADS["sd-turbo-512"]["name"]


def select_workload(key: str) -> None:
    global MODEL_ID, T_INDEX_LIST, H, W, METRIC, GFLOP_PER_FRAME, WORKLOAD
    w = WORKLOADS[key]
    MODEL_ID, T_INDEX_LIST, METRIC, GFLOP_PER_FRAME, WORKLOAD = w["model"], w["t"], w["metric"], w["gflop"], w["name"]
    H = W = w["hw"]


def bench_config(world: int) -> dict:
    """One config dict for every arm (the driver compares the arms' `config` keys)."""
    return {"workload": WORKLOAD, "t_index_list": T_INDEX_LIST, "weights": "seeded synthetic (no checkpoint offline)",
            "parallelism": f"dp{world}: one independent stream per GPU, NCCL weight broadcast at init only",
            "l2": "UNet weights (1.73 GB) are re-streamed from HBM every step (>> 126 MB L2); 64-frame input ring",
            "model": MODEL_ID}


def physical_cores() -> int:
    """Physical cores of the box (torchrun exports OMP_NUM_THREADS=1, which would hobble the CPU arm to one thread)."""
    try:
        pairs = set()
        phys = core = None
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("physical id"):
                    phys = line.split(":")[1].strip()
                elif line.startswith("core id"):
                    core = line.split(":")[1].strip()
                elif not line.strip():
                    if phys is not None and core is not None:
                        pairs.add((phys, core))
                    phys = core = None
        if pairs:
            return len(pairs)
    except OSError:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def pin_to_gpu_numa_node(dev_index: int):
    """Bind this rank's host threads to the CPUs of its GPU's NUMA node (pinned-memory copies and launches then stay
    local).  Returns a short description for the JSON line, or None when the topology files are not readable."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev_index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus), "pci": bdf}
    except Exception:   # noqa: BLE001 - best effort
        return None


def nccl_log_summary(log_glob: str):
    """What NCCL itself reported at init (NCCL_DEBUG=INFO written to NCCL_DEBUG_FILE): ranks, version, transports."""
    import glob
    import re
    nranks, version, nvls, p2p = set(), None, False, False
    for path in glob.glob(log_glob):
        try:
            with open(path, errors="replace") as f:
                for line in f:
                    m = re.search(r"nranks (\d+)", line)
                    if m and "Init COMPLETE" in line:
                        nranks.add(int(m.group(1)))
                    m = re.search(r"NCCL version ([0-9.]+)", line)
                    if m:
                        version = m.group(1)
                    nvls |= "NVLS" in line
                    p2p |= "P2P" in line
        except OSError:
            pass
    return {"init_complete_nranks": sorted(nranks), "version": version, "nvls_seen": nvls, "p2p_seen": p2p, "log": log_glob}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_uuid: str):
        self.lines = []
        self.proc = None
        self.uuid = gpu_uuid
        self.t = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.uuid, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()  # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU oracle arm
def run_oracle(steps: int, warmup: int, budget_s: float):
    """Times the fp32 oracle (the reference's CPU diffusers path restated, oracle/) on the host cores."""
    import torch
    from oracle import pipeline as opipe
    from oracle import stream as ostream
    from oracle import unet as ounet
    from oracle import weights as ow
    # every physical core, set explicitly: under torchrun OMP_NUM_THREADS=1 would otherwise leave this arm single-threaded
    # (oversubscribing the SMT siblings is slower, so not os.cpu_count())
    threads = min(physical_cores(), len(os.sched_getaffinity(0)))
    torch.set_num_threads(threads)
    cfg = ounet.config_for(MODEL_ID)
    usd = ow.to_float(ow.make_unet_weights(cfg))
    vsd = ow.to_float(ow.make_taesd_weights())
    orc = ostream.StreamOracle(usd, cfg, vsd, T_INDEX_LIST, W, H)
    orc.prepare(ow.make_prompt_embeds(cfg.cross_attention_dim).float(), guidance_scale=0.0)
    frames = [ow.make_frame(H, W, seed=i) for i in range(4)]
    t0 = time.perf_counter()
    opipe.frame_to_u8(orc, frames[0])  # at least one warm-up frame
    first = time.perf_counter() - t0
    w_done = 1
    while w_done < warmup and (time.perf_counter() - t0) + first < budget_s * 0.25:
        opipe.frame_to_u8(orc, frames[w_done % 4])
        w_done += 1
    times = []
    t_start = time.perf_counter()
    for i in range(steps):
        t1 = time.perf_counter()
        opipe.frame_to_u8(orc, frames[i % 4])
        times.append(time.perf_counter() - t1)
        if time.perf_counter() - t_start + times[-1] > budget_s:
            break
    total = sum(times)
    return {"fps": len(times) / total, "ms_per_step": 1000.0 * total / len(times), "steps": len(times), "warmup": w_done,
            "threads": threads}


def main_reference(args):
    rank = int(os.getenv("RANK", "0"))
    if rank != 0:
        return 0
    r = run_oracle(args.steps, args.warmup, budget_s=150.0)
    cb = {"value": r["fps"], "unit": "frames/s", "cores": r["threads"], "kind": "port",
          "sample": f"{r['steps']} full 512x512 SD-Turbo 1-step frames (UNet + TAESD enc/dec, fp32 torch oracle; the reference's "
                    "diffusers/StreamDiffusion packages are not installable offline), time-bounded to 150 s"}
    line = {"impl": "reference", "metric": METRIC, "value": r["fps"], "unit": "frames/s", "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(max(1, args.gpus)),
            "cpu_baseline": cb,
            "e2e": {"value": r["fps"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ library arm
def run_library(steps: int, warmup: int, dev, use_graph: bool = True):
    """The same frame program through torch's fp16 library kernels (cuDNN convolutions, cuBLAS GEMMs, fused SDPA), the whole
    frame captured in one CUDA graph: the stand-in for "the reference's TensorRT engines" that can be built offline
    (lib/wrapper.py:923-925 falls back to plain torch fp16 when TensorRT is unavailable).  oracle/torch_gpu.py."""
    import torch
    from oracle import torch_gpu as tg
    from oracle import unet as ounet
    from oracle import weights as ow
    torch.backends.cudnn.benchmark = True
    cfg = ounet.config_for(MODEL_ID)
    orc = tg.build(cfg, ow.make_unet_weights(cfg), ow.make_taesd_weights(), T_INDEX_LIST, H,
                   ow.make_prompt_embeds(cfg.cross_attention_dim), None, torch.float16, str(dev))
    frame = tg.GraphedFrame(orc, H, use_graph=use_graph)
    g = torch.Generator().manual_seed(999)
    ring = [torch.randint(0, 256, (1, H, W, 3), dtype=torch.uint8, generator=g).to(dev) for _ in range(16)]
    for i in range(max(warmup, 3)):
        frame(ring[i % 16])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        frame(ring[i % 16])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": 1000.0 / ms, "unit": "frames/s", "ms_per_step": ms, "steps": steps,
            "kind": "torch %s fp16: oracle modules .half().cuda(), cuDNN conv (benchmark mode) + fused SDPA + cuBLAS, whole frame in "
                    "one CUDA graph%s" % (torch.__version__, "" if use_graph else " (graph OFF)")}


def main_library(args):
    import torch
    rank = int(os.getenv("RANK", "0"))
    if rank != 0:
        return 0
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl library needs a CUDA device")
    dev = torch.device("cuda", int(os.getenv("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    r = run_library(args.steps, args.warmup, dev)
    line = {"impl": "library", "metric": METRIC, "value": r["value"], "unit": "frames/s", "n_gpus": 1, "steps": r["steps"],
            "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": bench_config(1),
            "library_baseline": {"value": r["value"], "unit": "frames/s", "kind": r["kind"]}, "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm
def _pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


def main_gpu(args):
    import gc
    import torch
    import torch.distributed as dist
    os.environ.setdefault("B200SD_SYNTHETIC_WEIGHTS", "1")
    world_env = int(os.getenv("WORLD_SIZE", "1"))
    nccl_glob = log_dir = None
    nccl_env = {k: v for k, v in os.environ.items() if k.startswith("NCCL_DEBUG")}
    if world_env > 1 and os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":   # unset, or the CUDA image's default
        # nobody asked for NCCL's log: keep stdout to the single JSON line, but still keep NCCL's own account of the job
        # (INFO level into per-process files, summarised in the line's "nccl" field).  A caller-provided NCCL_DEBUG is left
        # exactly as it is -- level and destination -- so a harness that reads NCCL's output from this process keeps seeing it.
        # The logs go to a directory of this launch under the temporary directory (the tree may be read-only).  Every rank
        # derives the same name: the user id and the torchrun run id, or, without one, the launcher's pid (ranks started by one
        # torchrun share it as their parent) and the rendezvous port.  Rank 0 removes the directory once it has summarised it.
        import tempfile
        launch = os.getenv("TORCHELASTIC_RUN_ID", "none")
        if launch == "none":
            launch = f"{os.getppid()}-{os.getenv('MASTER_PORT', '0')}"
        log_dir = os.path.join(tempfile.gettempdir(), f"b200sd-bench-nccl-{os.getuid()}-{launch}")
        os.makedirs(log_dir, exist_ok=True)
        if os.stat(log_dir).st_uid != os.getuid():     # a directory of that name owned by someone else: NCCL's defaults
            log_dir = None
        else:
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ["NCCL_DEBUG_FILE"] = os.path.join(log_dir, f"nccl_n{world_env}_%h_%p.log")
            nccl_glob = os.environ["NCCL_DEBUG_FILE"].replace("%h", "*").replace("%p", "*")
    os.environ["NVENC"] = "1"  # keep the output tensor in HBM (lib/pipeline.py:83,96)
    from ai_rtc_agent_b200.host import dist as bdist
    from ai_rtc_agent_b200.host.pipeline import StreamDiffusionPipeline
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the GPU arm has no CPU fallback; use --impl reference)")
    rank, world, local = bdist.init()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    numa = pin_to_gpu_numa_node(local) if not args.no_numa_pin else None
    bdist.load_and_broadcast(MODEL_ID, dev)          # rank 0 materialises, NCCL broadcast, once
    pipe = StreamDiffusionPipeline(MODEL_ID, t_index_list=T_INDEX_LIST, width=W, height=H)
    stream = pipe.model.stream

    g = torch.Generator().manual_seed(1000 + rank)
    ring_host = [torch.randint(0, 256, (1, H, W, 3), dtype=torch.uint8, generator=g).pin_memory() for _ in range(64)]
    ring_dev = [f.to(dev) for f in ring_host]
    out_host = torch.empty((1, 3, H, W), dtype=torch.uint8).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(vals):
        """list of floats of this rank -> [world][len] on every rank"""
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world == 1:
            return [t.tolist()]
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [o.tolist() for o in out]

    import collections
    lanes = pipe.lanes
    cur = torch.cuda.current_stream(dev)
    warm = max(args.warmup, 3)
    for i in range(warm * lanes):
        pipe(ring_dev[i % 64])
    torch.cuda.synchronize()

    def timed_device_loop(submit):
        """K frames, device-timed on the current stream; `submit(i)` returns a ticket or None (stream-ordered call).
        Returns the elapsed ms and the ticket of the last frame (None when `submit` returns no tickets)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = collections.deque(maxlen=lanes)
        for i in range(args.steps):
            t = submit(i)
            if t is not None:
                last.append(t)
        for t in last:
            t.wait(cur)            # the closing event is ordered after the last frame of every lane
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), (last[-1] if last else None)

    # ---- device-resident throughput (value): frames already in HBM, public non-blocking entry, `lanes` frames in flight
    sampler = ClockSampler("GPU-" + str(torch.cuda.get_device_properties(dev).uuid)) if rank == 0 else None
    gc.collect()
    gc.disable()   # a collection inside a 20-step timed loop is a multi-ms tail on that rank
    barrier()
    if sampler:
        sampler.start()
    my_ms, last_ticket = timed_device_loop(lambda i: pipe.enqueue(ring_dev[(warm + i) % 64]))
    barrier()
    clocks = sampler.stop() if sampler else None
    # what the caller of the timed path received for its last frame: (1, 3, H, W) u8, stored as float32
    dumped = {"output": last_ticket.result().float().cpu().numpy()} if args.dump_outputs and rank == 0 else None
    dev_ms = [r[0] for r in gather([my_ms])]
    ms_total = max(dev_ms)
    value = world * args.steps / (ms_total / 1000.0)
    # the same frames through the blocking call (one frame at a time, the reference's calling pattern): per-frame device latency
    barrier()
    seq_ms = max(r[0] for r in gather([timed_device_loop(lambda i: (pipe(ring_dev[(warm + i) % 64]), None)[1])[0]]))
    # ---- end to end through the public API with host buffers (e2e): every step copies its frame from pinned host memory and
    # reads its result back into pinned host memory; latency = submit -> result on the host.  Up to `lanes` frames are pending
    # (--e2e-pending): the next frame is submitted when the oldest has been retired, i.e. when its lane is free.  With lanes + 2
    # pending the upload / download phases no longer cost a compute slot (+3 %: 484-488 frames/s instead of 470), but a frame
    # can then queue behind a whole frame on its lane: p99 33 ms instead of 17.6 ms (profiles/bench_r02w_line.json).
    d2h = torch.cuda.Stream(dev)
    pending_max = max(1, args.e2e_pending if args.e2e_pending > 0 else lanes)
    out_ring = [torch.empty((1, 3, H, W), dtype=torch.uint8).pin_memory() for _ in range(pending_max + 1)]

    in_ring = [torch.empty((1, H, W, 3), dtype=torch.uint8, device=dev) for _ in range(pending_max + 1)]

    def e2e_submit(i):
        # no allocation on this path: the upload lands in a preallocated device slot (free again once its frame has been
        # retired), and the result tensor is kept alive until its download has completed instead of record_stream()ing it -- a
        # cudaMalloc in the middle of the loop would drain every frame in flight (a 16 ms stall seen once with .to() + record_stream)
        t0 = time.perf_counter()
        frame = in_ring[i % (pending_max + 1)]
        frame.copy_(ring_host[(warm + i) % 64], non_blocking=True)
        tk = pipe.enqueue(frame)
        tk.wait(d2h)
        with torch.cuda.stream(d2h):
            res = tk.result(wait=False)
            out_ring[i % (pending_max + 1)].copy_(res, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(d2h)
        return t0, ev, res

    def e2e_run(n, lat):
        pend = collections.deque()
        for i in range(n):
            pend.append(e2e_submit(i))
            while len(pend) >= pending_max:      # retire the oldest before submitting the next
                t0, ev, _res = pend.popleft()
                ev.synchronize()
                lat.append((time.perf_counter() - t0) * 1000.0)
        while pend:
            t0, ev, _res = pend.popleft()
            ev.synchronize()
            lat.append((time.perf_counter() - t0) * 1000.0)

    e2e_run(6 * pending_max, [])     # untimed: first use of the pinned rings / copy streams on this rank
    lat = []
    barrier()
    t_all = time.perf_counter()
    e2e_run(args.steps, lat)
    my_e2e_s = time.perf_counter() - t_all
    barrier()
    gc.enable()
    per = gather([my_e2e_s, statistics.median(lat), _pct(lat, 0.99), max(lat), float(lat.index(max(lat)))])
    e2e_s = max(r[0] for r in per)
    e2e_fps = world * args.steps / e2e_s
    p50 = max(r[1] for r in per)
    slowest = max(range(world), key=lambda r: per[r][0])
    per_rank = [{"rank": r, "device_ms_per_step": dev_ms[r] / args.steps, "e2e_s": per[r][0], "e2e_p50_ms": per[r][1],
                 "e2e_p99_ms": per[r][2], "e2e_max_ms": per[r][3], "e2e_max_at_step": int(per[r][4])} for r in range(world)]
    numa_all = gather([float(numa["numa_node"]) if numa else -1.0])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    # ---- roofline of the dominant kernel: per-launch device times from an eager replay outside the timed region
    prof = stream.profile(ring_dev[0], iters=3)
    by = {}
    for op in prof:
        kind = op["name"].split(" ")[0]
        d = by.setdefault(kind, {"ms": 0.0, "flops": 0.0, "launches": 0})
        d["ms"] += op["ms"]; d["flops"] += op["flops"]; d["launches"] += 1
    peaks, peak_src = measured_peaks()
    # dominant kernel: its launches alone, replayed from their own CUDA graph (same order, buffers, PDL edges and weight
    # streaming as inside the frame graph) -> average launch duration without the host-side gaps of the eager replay
    ig = stream.profile_kind("igemm", iters=20)
    ig_tflops_seq = ig["flops"] / (ig["ms"] * 1e-3) / 1e12

    def concurrent_kind(kind, iters=60):
        """The launches of one class of ALL lanes replayed at the same time (one host thread + CUDA stream per lane, like the
        frames in flight of the timed region): aggregate algorithmic FLOP/s of that kernel under the conditions it really runs in."""
        import threading
        from ai_rtc_agent_b200.host import capi
        res = [None] * lanes
        gate = threading.Barrier(lanes)
        capi.lib().b2sd_profile_gate(lanes)   # the lanes' timed replays start together (after capture / warm-up of all of them)

        def work(k):
            torch.cuda.set_device(dev)
            with torch.cuda.stream(torch.cuda.Stream(dev)):
                gate.wait()
                res[k] = pipe._engines[k].profile_kind(kind, iters=iters)

        th = [threading.Thread(target=work, args=(k,)) for k in range(lanes)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        capi.lib().b2sd_profile_gate(0)
        ms = sum(r["ms"] for r in res) / lanes
        return {"ms": ms, "flops": sum(r["flops"] for r in res), "launches": res[0]["launches"]}

    igc = concurrent_kind("igemm") if lanes > 1 else ig
    ig_tflops = igc["flops"] / (igc["ms"] * 1e-3) / 1e12
    kinds = {}
    for kind in ("tconv", "attn", "groupnorm", "layernorm"):
        try:
            r = stream.profile_kind(kind, iters=20)
            kinds[kind] = {"ms_per_step": round(r["ms"], 4), "launches": r["launches"],
                           "tflops": round(r["flops"] / (r["ms"] * 1e-3) / 1e12, 1) if r["flops"] else None}
        except Exception:   # noqa: BLE001 - kind not present in this program
            pass
    step_ms = ms_total / args.steps
    step_tflops = GFLOP_PER_FRAME * (value / world) / 1e3
    traffic, traffic_note = None, "no ncu capture found under profiles/"
    tpath = os.path.join(ROOT, "profiles", "igemm_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic, traffic_note = tj.get("dram_bytes_per_launch"), tj.get("note", "")
    roofline = {
        "bound": "tensor", "kernel": "igemm_kernel / igemm_pair_kernel (one source: tcgen05 implicit-GEMM conv/linear, single CTAs or cta_group::2 CTA pairs)",
        "achieved": ig_tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
        "frac": ig_tflops / peaks["bf16_tflops_sustained"], "traffic": traffic,
        "peak_source": peak_src + ", sustained figure (kernel timed inside a long step)",
        "traffic_note": traffic_note,
        "kernel_share_of_step": (igc["ms"] / lanes) / step_ms, "kernel_launches_per_step": ig["launches"],
        "kernel_ms_per_step": igc["ms"] / lanes, "kernel_avg_launch_us": 1e3 * (igc["ms"] / lanes) / max(ig["launches"], 1),
        "kernel_timing": f"CUDA events around graphs holding only the igemm launches of one frame; {lanes} such graphs (one per lane, as "
                         "many frames as the timed region keeps in flight) replayed concurrently on their own streams, 60 replays each: "
                         "achieved = their summed algorithmic FLOPs / the mean replay time; kernel_ms_per_step = that time / lanes",
        "kernel_algorithmic_gflop_per_step": ig["flops"] / 1e9,
        "one_frame_at_a_time": {"achieved": ig_tflops_seq, "frac": ig_tflops_seq / peaks["bf16_tflops_sustained"],
                                "kernel_ms_per_step": ig["ms"], "kernel_avg_launch_us": 1e3 * ig["ms"] / max(ig["launches"], 1),
                                "note": "the same launches of ONE frame alone on the GPU, a dependent chain.  They are planned for the number of frames in flight "
                                        "(>= 4: CTA pairs without split-K), so alone they are slower than a lanes=1 pipeline's latency plan "
                                        "(single CTAs, cluster split-K: frac 0.18-0.20, DESIGN.md 4.7)"},
        "step_achieved": step_tflops, "step_frac": step_tflops / peaks["bf16_tflops_sustained"],
        "step_algorithmic_gflop": GFLOP_PER_FRAME,
        "other_kernels_in_graph": kinds,
        "by_kernel_eager_ms": {k: round(v["ms"], 4) for k, v in sorted(by.items(), key=lambda kv: -kv[1]["ms"])},
    }
    # ---- baselines (reported, not the target), rank 0 at N=1 only: torch fp16 library path on this GPU, fp32 oracle on the host cores
    cpu = lib = None
    if world == 1 and not args.no_library_baseline:
        del ring_dev
        try:
            r = run_library(min(args.steps, 100), 3, dev)
            lib = {"value": r["value"], "unit": "frames/s", "ms_per_step": r["ms_per_step"], "kind": r["kind"],
                   "ratio": value / r["value"]}
        except Exception as exc:   # noqa: BLE001 - the baseline must not take the bench line down
            lib = {"value": None, "error": f"{type(exc).__name__}: {exc}"[:300]}
    if world == 1 and not args.no_cpu_baseline:
        r = run_oracle(steps=2, warmup=1, budget_s=40.0)
        cpu = {"value": r["fps"], "unit": "frames/s", "cores": r["threads"], "kind": "port",
               "sample": f"{r['steps']} full 512x512 SD-Turbo 1-step frames of the fp32 torch oracle (1 warm-up), same workload"}
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": bench_config(world),
        "frames_in_flight": lanes,
        "sequential": {"value": world * args.steps / (seq_ms / 1000.0), "unit": "frames/s", "ms_per_frame": seq_ms / args.steps,
                       "note": "same frames through the blocking call, one frame on the GPU at a time (the reference's calling pattern), on THIS "
                               "pipeline, whose launches are planned for its frames_in_flight; a lanes=1 pipeline plans for latency instead "
                               "(SD-Turbo 512x512: 4.15 ms per frame, DESIGN.md 4.5)"},
        "p50_ms": p50,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": H * W * 3, "d2h_bytes_per_step": H * W * 3,
                "p50_ms": p50, "p99_ms": max(r[2] for r in per), "max_ms": max(r[3] for r in per), "slowest_rank": slowest,
                "samples_per_rank": args.steps, "frames_pending_max": pending_max,
                "tails_note": None if args.steps >= 100 else f"p99/max come from only {args.steps} samples per rank"},
        "per_rank": per_rank,
        "numa": {"pinned": numa is not None, "rank0": numa, "nodes_by_rank": [int(r[0]) for r in numa_all]},
        "gpu_launches": stream.launches_per_step * args.steps,
        "launches_per_step": stream.launches_per_step,
        "roofline": roofline, "library_baseline": lib, "cpu_baseline": cpu, "clocks": clocks,
    }
    if world > 1:
        line["nccl"] = dict(nccl_log_summary(nccl_glob) if nccl_glob else {"log": "NCCL_DEBUG* set by the caller, left untouched"},
                            caller_env=nccl_env, world_size=world, backend=dist.get_backend(), collectives_per_step=0)
    if log_dir:
        import shutil
        shutil.rmtree(log_dir, ignore_errors=True)
    if dumped:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "library"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--no-numa-pin", action="store_true")
    ap.add_argument("--e2e-pending", type=int, default=0, help="frames pending in the end-to-end loop (0 = frames_in_flight)")
    ap.add_argument("--workload", default="sd-turbo-512", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step (rank 0: the (1,3,H,W) u8 frame the caller received, as float32) "
                         "to DIR/output.npy; the inputs are seeded, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs is supported by --impl b200 only")
    select_workload(a.workload)
    sys.exit(main_reference(a) if a.impl == "reference" else (main_library(a) if a.impl == "library" else main_gpu(a)))
