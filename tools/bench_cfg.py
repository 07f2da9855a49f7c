"""Cost of classifier-free guidance through the public pipeline (StreamDiffusionPipeline, seeded synthetic weights).

For each workload (SD-1.5 + LCM 4-step and SD-Turbo 1-step, 512x512) and each cfg_type (none; self / initialize / full with
guidance_scale 1.4) it reports
  * fps:    frames/s of `steps` frames enqueued back to back on the pipeline's default lanes, device-timed (CUDA events);
  * p50_ms: median latency of the blocking call (one frame at a time, host clock around a call that ends in a synchronise);
  * lanes, unet_batch, launches_per_step.
The GPU name and power limit are read in the same run.  Prints one JSON line and writes it to --out (default
profiles/bench_cfg_line.json); the source tree is not written otherwise.

    python tools/bench_cfg.py [--steps 200] [--warmup 10] [--out profiles/bench_cfg_line.json]"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {"sd15-lcm4-512": ("lykon/dreamshaper-8", [18, 26, 35, 45], 512),
             "sd-turbo-512": ("stabilityai/sd-turbo", [32], 512)}
CFG_TYPES = ("none", "self", "initialize", "full")
GUIDANCE = 1.4


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        name, power, clk = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit": power, "clocks_max_sm": clk}
    except Exception as exc:   # noqa: BLE001 - reported, not fatal
        return {"gpu": None, "error": str(exc)}


def run_one(torch, model_id, tl, hw, cfg_type, steps, warmup):
    from ai_rtc_agent_b200.host.pipeline import StreamDiffusionPipeline
    guided = cfg_type != "none"
    pipe = StreamDiffusionPipeline(model_id, t_index_list=tl, width=hw, height=hw, cfg_type=cfg_type,
                                   guidance_scale=GUIDANCE if guided else 0.0, negative_prompt="blurry, low quality")
    g = torch.Generator().manual_seed(1000)
    ring = [torch.randint(0, 256, (1, hw, hw, 3), dtype=torch.uint8, generator=g).cuda() for _ in range(32)]
    for i in range(max(warmup, 3) * pipe.lanes):
        pipe(ring[i % 32])
    torch.cuda.synchronize()
    cur = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gc.disable()
    e0.record()
    last = []
    for i in range(steps):
        last.append(pipe.enqueue(ring[i % 32]))
        last = last[-pipe.lanes:]
    for t in last:
        t.wait(cur)
    e1.record()
    torch.cuda.synchronize()
    fps = steps / (e0.elapsed_time(e1) / 1000.0)
    lat = []
    for i in range(steps):
        t0 = time.perf_counter()
        pipe(ring[i % 32])
        torch.cuda.synchronize()
        lat.append((time.perf_counter() - t0) * 1000.0)
    gc.enable()
    sd = pipe.model.stream
    row = {"cfg_type": cfg_type, "guidance_scale": GUIDANCE if guided else 0.0, "fps": round(fps, 2),
           "p50_ms": round(statistics.median(lat), 3), "lanes": pipe.lanes, "unet_batch": sd.trt_unet_batch_size,
           "launches_per_step": sd.launches_per_step}
    del pipe, sd, ring
    gc.collect()
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_cfg_line.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_cfg.py: no CUDA device (no CPU fallback)")
    os.environ.setdefault("B200SD_SYNTHETIC_WEIGHTS", "1")
    os.environ["NVENC"] = "1"
    from ai_rtc_agent_b200.host import dist as bdist
    from ai_rtc_agent_b200.host import weights as W
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    line = {"tool": "tools/bench_cfg.py", **gpu_info(), "steps": args.steps, "workloads": {}}
    for key in args.workloads.split(","):
        model_id, tl, hw = WORKLOADS[key]
        bdist.load_and_broadcast(model_id, dev)
        line["workloads"][key] = [run_one(torch, model_id, tl, hw, ct, args.steps, args.warmup) for ct in CFG_TYPES]
        W._PRELOADED.pop(model_id, None)
        gc.collect()
        torch.cuda.empty_cache()
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
