"""Throughput of `MIGAN_Pipeline.forward_batch` against the same requests served one by one through `pipe(image, mask)`, on
cuda:0.  Model resolution 512, padding 128, a hole of a quarter of each side (as tools/pipeline_latency.py).  Traffic mix:
32 requests = 8 x 512^2 + 16 x 1080x1920 + 8 x 2160x3840, images and masks already on the device (~420 MB of images, far
over the 126 MB of L2).  The two paths alternate in one run, each timed with a host clock around work that ends in
torch.cuda.synchronize(); then one row per size for a single request; then a separate torch.profiler run for launch counts
and kernel times.  Measurement tooling (seeded random weights, no oracle).

    python tools/pipeline_batch.py [out.json]      # default: r03_pipeline_batch_512.json in the current directory
"""
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import migan_b200  # noqa: E402
from migan_b200 import synthetic  # noqa: E402
from migan_b200.pipeline import MIGAN_Pipeline  # noqa: E402

RES, PAD = 512, 128
MIX = [(512, 512)] * 8 + [(1080, 1920)] * 16 + [(2160, 3840)] * 8


def requests(sizes, dev, seed=0):
    rng = np.random.RandomState(seed)
    images, masks = [], []
    for (H, W) in sizes:
        images.append(torch.from_numpy(rng.randint(0, 256, size=(1, 3, H, W), dtype=np.uint8)).to(dev))
        m = torch.full((1, 1, H, W), 255, dtype=torch.uint8, device=dev)
        m[:, :, H // 3: H // 3 + H // 4, W // 3: W // 3 + W // 4] = 0
        masks.append(m)
    return images, masks


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def stats(ms, n_req):
    s = sorted(ms)
    p50 = statistics.median(s)
    return {"p50_ms": p50, "p90_ms": s[int(0.9 * (len(s) - 1))], "requests_per_s": n_req / (p50 * 1e-3), "samples": len(s)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "r03_pipeline_batch_512.json"
    dev = torch.device("cuda", 0)
    sd = synthetic.export_style_state_dict(RES, seed=1)
    seq = MIGAN_Pipeline(sd, RES, padding=PAD, device=dev)          # its own generator: the batch-1 graph stays captured
    bat = MIGAN_Pipeline(sd, RES, padding=PAD, device=dev)
    images, masks = requests(MIX, dev)

    def run_seq(imgs=images, msks=masks):
        for im, m in zip(imgs, msks):
            seq(im, m)

    def run_batch(imgs=images, msks=masks):
        bat.forward_batch(imgs, msks)

    for _ in range(3):
        run_seq(); run_batch()
    t_seq, t_bat = [], []
    for _ in range(20):
        t_seq.append(timed(run_seq))
        t_bat.append(timed(run_batch))
    mix = {"requests": len(MIX), "sizes": {"512x512": 8, "1080x1920": 16, "2160x3840": 8},
           "sequential": stats(t_seq, len(MIX)), "forward_batch": stats(t_bat, len(MIX))}
    mix["speedup_requests_per_s"] = mix["forward_batch"]["requests_per_s"] / mix["sequential"]["requests_per_s"]
    print(json.dumps(mix), flush=True)

    single = []
    for size in [(512, 512), (1080, 1920), (2160, 3840)]:
        im, m = requests([size], dev, seed=1)
        for _ in range(5):
            run_seq(im, m); run_batch(im, m)
        a, b = [], []
        for _ in range(30):
            a.append(timed(lambda: run_seq(im, m)))
            b.append(timed(lambda: run_batch(im, m)))
        single.append({"image": list(size), "sequential": stats(a, 1), "forward_batch": stats(b, 1)})
        print(json.dumps(single[-1]), flush=True)

    # profiled run (separate from the timings): launches per batch, box kernel vs the flag stage on the 4K masks
    from torch.profiler import ProfilerActivity, profile
    k4 = [i for i, s in enumerate(MIX) if s == (2160, 3840)]
    im4, m4 = [images[i] for i in k4], [masks[i] for i in k4]
    run_batch(im4, m4); [seq.get_masked_bbox(m) for m in m4]
    torch.cuda.synchronize()
    prof_rows = {}
    for name, fn in (("sequential", run_seq), ("forward_batch", run_batch),
                     ("flags_4k_x8", lambda: [seq.get_masked_bbox(m) for m in m4]), ("batch_4k_x8", lambda: run_batch(im4, m4))):
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            fn()
            torch.cuda.synchronize()
        kern = [e for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in e.name and "Memset" not in e.name]
        copies = [e for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" in e.name]
        row = {"kernels": len(kern), "copies": len(copies), "kernel_ms": sum(e.device_time for e in kern) / 1e3}
        if name == "flags_4k_x8":
            row["hole_flags_ms"] = sum(e.device_time for e in kern if "HoleFlagsK" in e.name) / 1e3
            row["dtoh_copies"] = len([e for e in copies if "DtoH" in e.name])
        if name == "batch_4k_x8":
            row["hole_extents_ms"] = sum(e.device_time for e in kern if "hole_extents" in e.name) / 1e3
            row["box_stage_ms"] = sum(e.device_time for e in kern if any(k in e.name for k in ("hole_extents", "ExtentsInitK", "BoxFromExtentsK"))) / 1e3
            row["mask_bytes"] = 8 * 2160 * 3840
            row["hole_extents_GBps"] = row["mask_bytes"] / (row["hole_extents_ms"] * 1e-3) / 1e9 if row["hole_extents_ms"] else None
        by = {}
        for e in kern:
            key = e.name.split("(")[0][:120]
            b = by.setdefault(key, [0, 0.0])
            b[0] += 1; b[1] += e.device_time / 1e3
        row["by_kernel"] = {k: {"launches": v[0], "ms": round(v[1], 4)} for k, v in sorted(by.items(), key=lambda kv: -kv[1][1])[:12]}
        prof_rows[name] = row
        print(name, json.dumps({k: v for k, v in row.items() if k != "by_kernel"}), flush=True)

    result = {"what": "MIGAN_Pipeline.forward_batch vs sequential pipe(image, mask)", "resolution": RES, "padding": PAD,
              "hole": "a quarter of each side at (H/3, W/3)", "inputs": "device-resident, contiguous",
              "timing": "host clock around work ending in torch.cuda.synchronize(); paths alternated in one run",
              "card": card(), "mix": mix, "single_request": single, "profile": prof_rows}
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    json.dump(result, open(out_path, "w"), indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
