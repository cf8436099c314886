"""bench.py -- images/sec of the MI-GAN generator forward on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (torchrun for N > 1)
    python bench.py --impl reference [--steps K] [--warmup W]      # reference arm: CPU forward on host cores

One "step" = Generator.forward on one batch of synthetic input: migan-512, 32 images per GPU
(BASELINE.json configs[2]/[3]); at N GPUs every rank runs its own 32 images (weak scaling) and
the outputs are all-gathered over NCCL.  Prints ONE JSON line (rank 0).

  value        whole-job images/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          same metric through the host-buffer C-ABI call (pinned H2D + forward + D2H per step)
  roofline     dominant kernel: algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json HBM copy rate
  cpu_baseline the reference algorithm (oracle port, torch CPU ops) on this box's host cores
  parity       max-abs / mean-abs error of image 0 of the timed batch vs the CPU reference algorithm (same run)
  clocks       SM clock / throttle reasons sampled during the timed region

--dump-outputs DIR writes the images the timed path returned in its last step to DIR/img.npy (float32, NCHW; a batch
above 64 MB is cut to a fixed seeded sample of whole images).  Inputs and weights are seeded, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

DUMP_BYTES = 64_000_000
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
print_json = print


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="migan", choices=["migan", "comodgan"],
                    help="migan (default: BASELINE.json metric, configs[2]/[3]) or comodgan (configs[4], 256 / 16 images)")
    ap.add_argument("--res", type=int, default=None, help="default 512 (migan) / 256 (comodgan)")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU; default 32 (migan) / 16 (comodgan)")
    ap.add_argument("--path", default=os.environ.get("MIGAN_B200_PATH", "tc"))
    ap.add_argument("--comod-gemm", default=None, choices=["simt", "tc"],
                    help="comodgan workload: GEMM engine (tc = staged tcgen05 route, not yet run on hardware)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gather", action="store_true",
                    help="N > 1: skip the output all-gather (shows what the collective costs; not the north_star configuration)")
    ap.add_argument("--gather", default="auto", choices=["auto", "ce", "nccl"],
                    help="N > 1: output all-gather by copy-engine peer reads + an 8-byte NCCL ready signal (ce), NCCL all_gather_into_tensor "
                         "with 8 SMs left free for its 8 channels (nccl), or whichever measured faster at this world size (auto: ce at 2 GPUs, nccl above)")
    ap.add_argument("--masks", default="free_form", choices=["free_form", "blocks"], help="synthetic hole masks")
    ap.add_argument("--profile-out", default=None, help="write the per-launch table (JSON) here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the images of the last timed step to DIR/img.npy (float32; at most 64 MB, a seeded sample of whole images)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.res is None:
        args.res = 512 if args.workload == "migan" else 256
    if args.batch is None:
        args.batch = 32 if args.workload == "migan" else 16
    return args


def dump_outputs(out_dir: str, img: torch.Tensor) -> None:
    """img [N, 3, R, R] -> out_dir/img.npy as float32; above DUMP_BYTES, a seeded choice of whole images (in batch order)."""
    import numpy as np

    img = img.detach().to("cpu", torch.float32)
    keep = min(img.shape[0], (DUMP_BYTES - 128) // (img[0].numel() * 4))      # 128: the .npy header
    if keep < img.shape[0]:
        pick = torch.randperm(img.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        print("dump-outputs: images %s of %d" % (pick.tolist(), img.shape[0]), file=sys.stderr)
        img = img[pick]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "img.npy"), img.contiguous().numpy())


# ------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.02)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return HBM_FALLBACK_GBS, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def usable_cpus() -> int:
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:  # cgroup v2 CPU quota
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def pick_cpu_threads(res: int) -> int:
    """All the host threads the CPU path can actually use: oneDNN stops scaling (and collapses when
    the container's CPU quota is below the visible core count), so calibrate on a small case."""
    from oracle import migan_oracle as O

    limit = usable_cpus()
    cands = sorted({c for c in (8, 16, 32, 64, limit) if c <= limit} | {min(limit, 8)})
    r = min(res, 128)
    sd = O.make_state_dict(r, seed=1)
    x = O.make_input(r, 1, seed=1)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        O.generator_forward(sd, x, r)
        t0 = time.perf_counter()
        O.generator_forward(sd, x, r)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_reference_forward_rate(res: int, seconds: float, max_iters: int, warmup: int = 1):
    """The reference algorithm on the host cores: oracle port (same torch CPU ops as
    lib/model_zoo/migan_inference.py), batch 1 (fastest per image on CPU, BASELINE.md section 2)."""
    from oracle import migan_oracle as O  # checker / CPU baseline only

    threads = pick_cpu_threads(res)
    sd = O.make_state_dict(res, seed=1)
    x = O.make_input(res, 1, seed=1234)
    for _ in range(warmup):
        O.generator_forward(sd, x, res)
    times = []
    t_begin = time.perf_counter()
    while len(times) < max_iters and (time.perf_counter() - t_begin < seconds or not times):
        t0 = time.perf_counter()
        O.generator_forward(sd, x, res)
        times.append(time.perf_counter() - t0)
    return len(times) / sum(times), len(times), threads


# ------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm: the reference's own CPU forward (oracle port; /root/reference does not exist
    on the GPU box), all host threads, one bs=1 forward of migan-<res> per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import migan_oracle as O

    pick_cpu_threads(args.res)
    sd = O.make_state_dict(args.res, seed=1)
    x = O.make_input(args.res, 1, seed=1234)
    for _ in range(max(args.warmup, 1)):
        O.generator_forward(sd, x, args.res)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = O.generator_forward(sd, x, args.res)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y)
    value = args.steps / dt
    line = {
        "impl": "reference", "metric": "images/sec", "value": value, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "migan-%d Generator.forward, reference algorithm on host CPU, bs=1 per step" % args.res},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": "%d bs=1 forwards of migan-%d (torch %s CPU ops)" % (args.steps, args.res, torch.__version__)},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print_json(json.dumps(line), flush=True)


def run_b200(args):
    import torch.distributed as dist

    import migan_b200
    from migan_b200 import parallel, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        parallel.configure_overlap(gather=args.gather)              # nccl: few channels + SMs left free for them; ce: nothing reserved
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout = the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    R, B, K, Wm = args.res, args.batch, args.steps, max(args.warmup, 3)

    model = migan_b200.Generator(R, path=args.path)
    model.load_state_dict(synthetic.export_style_state_dict(R, seed=1))
    model = model.to(dev).eval()
    x_host = synthetic.synthetic_input(R, B, seed=1234 + rank, masks=args.masks).pin_memory()
    x = x_host.to(dev)
    sharded = parallel.ShardedGenerator(model, gather=args.gather) if (world > 1 and not args.no_gather) else None
    if sharded is not None:
        sharded.check_replicas(model.state_dict())

    def step():
        if sharded is None:
            return model(x)
        return sharded.forward_async(x)          # gather of step t overlaps compute of step t+1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(Wm):
        h = step()
    if sharded is not None:
        h.wait()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    handles = []
    for _ in range(K):
        h = step()
        if sharded is None:
            continue                             # the previous output is released: the caching allocator hands the same
                                                 # block to the next call, so no cudaMalloc lands in the timed region
        handles.append(h)
        if len(handles) > 2:
            handles.pop(0).wait()                # bound memory: at most 2 gathers in flight
    for h in handles:
        h.wait()
    ev1.record()
    barrier()
    clocks = sampler.stop()
    elapsed_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:                # h: the last step's output (its gather handle at N > 1)
        dump_outputs(args.dump_outputs, h if sharded is None else h.wait())
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    launches_per_step = model.last_launch_count()
    value = world * B * K / (elapsed_ms * 1e-3)

    # ---- end-to-end through the host-buffer C-ABI call (pinned H2D + forward + D2H, every step) ----
    y_host = torch.empty((B, 3, R, R), dtype=torch.float32).pin_memory()
    if sharded is None:
        for _ in range(2):
            model.forward_host(x_host, out=y_host)
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            model.forward_host(x_host, out=y_host, wait=False)   # serving loop: batches submitted back to back ...
        model.host_wait()                                         # ... every y has landed in host memory here
    else:   # N > 1: through ShardedGenerator -- host shard in, forward, all-gather, this rank's rows of the gathered tensor out
        for _ in range(2):
            sharded.forward_host_async(x_host, y_host)
        sharded.host_wait()
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            sharded.forward_host_async(x_host, y_host)
        sharded.host_wait()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": world * B * K / e2e_s, "unit": "images/s",
           "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": y_host.numel() * 4}

    # ---- same, through the uint8 request call (img + mask uint8 in, composed uint8 out: 7 B/px over PCIe, not 28) ----
    e2e_u8 = None
    if world == 1:
        try:
            g8 = torch.Generator().manual_seed(7)
            img8 = torch.randint(0, 256, (B, R, R, 3), dtype=torch.uint8, generator=g8).pin_memory()
            m8 = ((torch.rand(B, R, R, generator=g8) > 0.4).to(torch.uint8) * 255).pin_memory()
            o8 = torch.empty((B, R, R, 3), dtype=torch.uint8).pin_memory()
            for _ in range(2):
                model.forward_u8(img8, m8, out=o8)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for _ in range(K):
                model.forward_u8(img8, m8, out=o8, wait=False)   # serving loop, like the fp32 host call above
            model.host_wait()
            u8_s = time.perf_counter() - t0
            e2e_u8 = {"value": B * K / u8_s, "unit": "images/s", "h2d_bytes_per_step": img8.numel() + m8.numel(),
                      "d2h_bytes_per_step": o8.numel(), "api": "Generator.forward_u8(wait=False) + host_wait (migan_forward_u8_async)"}
        except Exception as exc:  # the uint8 path is an extra; the contract's e2e above does not depend on it
            e2e_u8 = {"error": str(exc)[:200]}

    if sharded is not None:
        sharded.close()
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- per-kernel pass: CUDA events around every launch, same inputs, K steps (rank 0) ----
    model.set_profiling(True)
    acc = {}
    for _ in range(K):
        model(x)
        torch.cuda.synchronize(dev)
        for label, ms, nbytes, flops in model.profile_steps():
            a = acc.setdefault(label, [0.0, nbytes, flops, 0])
            a[0] += ms
            a[3] += 1
    model.set_profiling(False)
    table = [{"launch": lb, "ms": v[0] / v[3], "alg_bytes": v[1], "flops": v[2],
              "GBps": v[1] / (v[0] / v[3] * 1e-3) / 1e9} for lb, v in acc.items()]
    by_kernel = {}
    for row in table:
        k = row["launch"].rsplit(".", 1)[-1]
        b = by_kernel.setdefault(k, {"ms": 0.0, "alg_bytes": 0.0, "launches": 0})
        b["ms"] += row["ms"]; b["alg_bytes"] += row["alg_bytes"]; b["launches"] += 1
    total_ms = sum(b["ms"] for b in by_kernel.values())
    dom = max(by_kernel, key=lambda k: by_kernel[k]["ms"])
    peak, peak_src = measured_peaks()
    d = by_kernel[dom]
    achieved = d["alg_bytes"] / (d["ms"] * 1e-3) / 1e9
    traffic, traffic_note = None, None
    try:  # DRAM bytes of one profiled launch of the dominant kernel (ncu --set full), committed under profiles/
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(dom)
        if tj:
            traffic, traffic_note = tj["dram_bytes"], tj
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_launch": traffic_note, "peak_source": peak_src,
                "launches_per_step": d["launches"], "share_of_step": d["ms"] / total_ms,
                "whole_step": {"alg_bytes": sum(b["alg_bytes"] for b in by_kernel.values()), "ms_sum_of_kernels": total_ms,
                               "GBps": sum(b["alg_bytes"] for b in by_kernel.values()) / (total_ms * 1e-3) / 1e9},
                "by_kernel": {k: {"ms": round(b["ms"], 4), "GBps": round(b["alg_bytes"] / (b["ms"] * 1e-3) / 1e9, 1),
                                  "launches": b["launches"]} for k, b in by_kernel.items()}}
    if R == 512:   # SURVEY.md 8(d): fully fused ideal = 1094.7 MB per image at 512 x 512 (every layer reads its input and writes its output once)
        ideal = 1094.7e6 * B
        roofline["whole_step"]["fused_ideal_bytes"] = ideal
        roofline["whole_step"]["frac_of_peak_vs_fused_ideal"] = ideal / (elapsed_ms / K * 1e-3) / 1e9 / peak if world == 1 else None
    if args.profile_out:
        os.makedirs(os.path.dirname(os.path.abspath(args.profile_out)), exist_ok=True)
        with open(args.profile_out, "w") as f:
            json.dump({"res": R, "batch": B, "path": args.path, "hbm_peak_GBps": peak, "launches": table}, f, indent=1)

    # ---- batch-1 latency through the CUDA-graph replay (the reference's primary caller is batch 1, scripts/demo.py:125-142) ----
    latency = None
    if world == 1:
        try:
            x1 = x[:1].contiguous()
            for _ in range(5):
                model(x1)
            torch.cuda.synchronize(dev)
            lat = []
            for _ in range(50):
                t0 = time.perf_counter()
                model(x1)
                torch.cuda.synchronize(dev)
                lat.append((time.perf_counter() - t0) * 1e3)
            latency = {"batch": 1, "p50_ms": statistics.median(lat), "p90_ms": sorted(lat)[44], "api": "Generator.forward (migan_forward_graph)",
                       "launches_replayed": model.last_launch_count()}
        except Exception as exc:
            latency = {"error": str(exc)[:200]}

    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        try:   # BASELINE.md section 3 item 6: parity in the same run, image 0 of the timed batch against the CPU reference algorithm
            from oracle import migan_oracle as O  # checker / CPU baseline only
            y0 = model(x)[:1].cpu()
            ref = O.generator_forward(O.make_state_dict(R, seed=1), x_host[:1], R)
            d = (y0 - ref).abs()
            parity = {"max_abs": float(d.max()), "mean_abs": float(d.mean()), "ref_abs_max": float(ref.abs().max()),
                      "isclose_rtol_1e-3_mismatch_frac": float((~torch.isclose(y0, ref, rtol=1e-3)).float().mean()),
                      "against": "oracle port (bit-exact with the reference on the committed fixtures), image 0 of the timed batch"}
        except Exception as exc:
            parity = {"error": str(exc)[:200]}
        rate, iters, cores = cpu_reference_forward_rate(R, seconds=12.0, max_iters=40)
        cpu = {"value": rate, "unit": "images/s", "cores": cores, "kind": "port",
               "sample": "%d bs=1 forwards of migan-%d with the oracle port (torch %s CPU ops, %d threads)"
                         % (iters, R, torch.__version__, cores)}

    line = {
        "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.path != "tc_fast" else "f16",
        "data": "synthetic",
        "config": {"workload": "migan-%d Generator.forward, %d images/GPU%s" % (R, B, (", all-gather of outputs (%s)" % ("copy-engine peer reads over NVLink + 8-byte NCCL ready signal" if sharded.gather == "ce" else "NCCL all_gather_into_tensor, %s channels, %s SMs left free for them" % (os.environ.get("NCCL_MAX_NCHANNELS", "?"), os.environ.get("MIGAN_TC_RESERVE_SMS", "0")))) if sharded is not None else (", no gather" if world > 1 else "")),
                   "masks": "free-form (rectangles + brush strokes, evaluate_fid_lpips.py protocol)" if args.masks == "free_form" else "8x8-cell blocks",
                   "path": args.path, "arithmetic": "fp32 CUDA-core depthwise/FIR; 1x1 convs on tcgen05 as fp16 hi/lo 3-pass split with fp32 accumulate"
                   if args.path == "tc" else args.path,
                   "global_batch": world * B, "weights": "seeded export-style random (unit-L2 filters)",
                   "l2": "per-step working set (input 134 MB + ~10 GB of activations at 512/32) exceeds the 126 MB L2; no flush needed",
                   "kernel_timing": "separate pass of K steps with cudaEvents around every launch",
                   "e2e": ("K host batches submitted back to back through migan_forward_host_async (pinned H2D + forward + D2H "
                           "per batch, two staging slots so the copies of batch t+1 / t-1 run under the kernels of batch t), timed until the last "
                           "output landed in host memory") if sharded is None else
                          ("K host shards per rank through ShardedGenerator.forward_host_async: pinned H2D, forward, all-gather, D2H of the "
                           "rank's rows of the gathered tensor; copies of batch t+1 / t-1 run under the kernels of batch t")},
        "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "clocks": clocks, "e2e": e2e, "e2e_u8": e2e_u8,
        "latency_bs1": latency,
        "gpu_launches": launches_per_step * K,
    }
    print_json(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def comodgan_gemm_flops(R: int) -> float:
    """2 x MACs of every GEMM one image goes through (closed form over the layer list of comodgan.py)."""
    ch = lambda r: min(32768 // r, 512)
    macs = 8 * 512 * 512 + 4 * ch(R) * R * R                          # mapping, fromrgb
    r = R
    while r >= 8:
        macs += 9 * ch(r) * ch(r) * r * r + 9 * ch(r) * ch(r // 2) * (r // 2) ** 2      # encoder conv0, conv1 (stride 2)
        r //= 2
    macs += 9 * 512 * 512 * 16 + 2 * 8192 * 1024                      # b4 conv, the two bottleneck dense layers
    macs += 9 * 512 * 512 * 16 + 512 * 3 * 16 + 2 * 1536 * 512        # synthesis b4 conv, torgb, affines
    r = 8
    while r <= R:
        macs += 9 * ch(r // 2) * ch(r) * (r // 2) ** 2 + 9 * ch(r) * ch(r) * r * r + 3 * ch(r) * r * r   # conv0 (transposed), conv1, torgb
        macs += 1536 * (ch(r // 2) + 2 * ch(r))
        r *= 2
    return 2.0 * macs


def run_comodgan(args):
    """BASELINE.json configs[4]: comodgan-256 Generator forward, batch 16, noise_mode='const'.  Round-1 path: exact fp32
    CUDA-core GEMMs (no tensor cores yet), so the roofline fraction against the tensor peak is small by construction."""
    from migan_b200 import comodgan

    if args.comod_gemm:
        os.environ["COMOD_GEMM"] = args.comod_gemm
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    R, B, K, Wm = args.res, args.batch, args.steps, max(args.warmup, 3)
    num_ws = 2 * (R.bit_length() - 1) - 2
    torch.manual_seed(1)
    model = comodgan.Generator(comodgan.Mapping(num_ws=num_ws), comodgan.Encoder(resolution=R), comodgan.Synthesis(resolution=R))
    with torch.no_grad():
        for k, p in model.named_parameters():                          # non-trivial biases / noise, like the parity tests
            if k.endswith("noise_strength") or (k.endswith(".bias") and "affine" not in k):
                p.copy_(0.1 * torch.randn(p.shape))
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(1234 + rank)
    mask = (torch.rand(B, 1, R, R, generator=g) > 0.4).float()
    img = torch.rand(B, 3, R, R, generator=g) * 2 - 1
    x_host = torch.cat([mask - 0.5, img * mask], 1).pin_memory()
    z_host = torch.randn(B, 512, generator=g).pin_memory()
    x, z = x_host.to(dev), z_host.to(dev)
    for _ in range(Wm):
        model(x, z=z, noise_mode="const")
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(K):
        y = model(x, z=z, noise_mode="const")
    ev1.record()
    torch.cuda.synchronize(dev)
    clocks = sampler.stop()
    elapsed_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y)
    y_host = torch.empty((B, 3, R, R), dtype=torch.float32).pin_memory()
    t0 = time.perf_counter()
    for _ in range(K):
        y = model(x_host.to(dev, non_blocking=True), z=z_host.to(dev, non_blocking=True), noise_mode="const")
        y_host.copy_(y, non_blocking=True)
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    if rank != 0:
        return
    flops = comodgan_gemm_flops(R) * B
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    tpeak = float(peaks.get("bf16_tflops_sustained", 0) or 0) or 1392.6
    achieved = flops / (elapsed_ms / K * 1e-3) / 1e12
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import comodgan_oracle as C  # checker / CPU baseline only
        from oracle import migan_oracle as O
        pick_cpu_threads(R)
        sd = C.make_state_dict(R, seed=1)
        xc, zc = O.make_input(R, 1, seed=1234), C.make_latent(1, seed=1235)
        C.generator_forward(sd, xc, zc, R)
        times = []
        while len(times) < 10 and (sum(times) < 10.0 or not times):
            t1 = time.perf_counter()
            C.generator_forward(sd, xc, zc, R)
            times.append(time.perf_counter() - t1)
        cpu = {"value": len(times) / sum(times), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "%d bs=1 forwards of comodgan-%d with the oracle port (torch %s CPU ops)" % (len(times), R, torch.__version__)}
    line = {
        "metric": "images/sec", "value": world * B * K / (elapsed_ms * 1e-3), "unit": "images/s", "n_gpus": world, "steps": K,
        "warmup": Wm, "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "comodgan-%d Generator.forward (z given, noise_mode=const), %d images/GPU" % (R, B),
                   "arithmetic": "exact fp32: im2col + CUDA-core GEMM (round-1 first path; tcgen05 implicit GEMM is the next step)"
                   if os.environ.get("COMOD_GEMM") != "tc" else "im2col fp16 hi/lo split + tcgen05 3-pass GEMM (staged route)",
                   "global_batch": world * B, "weights": "constructor-style N(0,1) + non-zero biases / noise strengths",
                   "l2": "col matrices are GBs per layer: far beyond the 126 MB L2"},
        "roofline": {"bound": "tensor", "kernel": "pw_gemm_simt (all GEMM launches)", "achieved": achieved, "peak": tpeak,
                     "unit": "TFLOP/s", "frac": achieved / tpeak, "traffic": None,
                     "note": "achieved = closed-form GEMM FLOPs of the step / whole step time (upper bound on the GEMM kernel's "
                             "own time); peak = MEASURED_PEAKS.json bf16_tflops_sustained"},
        "cpu_baseline": cpu, "clocks": clocks,
        "e2e": {"value": world * B * K / e2e_s, "unit": "images/s", "h2d_bytes_per_step": (x_host.numel() + z_host.numel()) * 4,
                "d2h_bytes_per_step": y_host.numel() * 4},
        "gpu_launches": model.last_launch_count() * K,
    }
    print_json(json.dumps(line), flush=True)


def main():
    args = parse_args()
    # stdout must carry exactly ONE JSON line: libraries (NCCL prints its version banner to stdout on some
    # configurations) get stderr for the whole run, the real stdout is restored only for the final print.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import builtins
    _print = builtins.print

    def emit(*a, **k):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        _print(*a, **k)
        sys.stdout.flush()
        os.dup2(2, 1)

    global print_json
    print_json = emit
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "comodgan":
        run_comodgan(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
