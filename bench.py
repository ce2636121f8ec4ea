#!/usr/bin/env python
"""Headline benchmark of the HardNet hot path on B200 (contract: see the task brief / DESIGN.md section 5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of HardNet.forward over this rank's shard of synthetic 32x32 patches
(BASELINE.json configs[2], bulk extraction: 4,194,304 patches over 8 GPUs = 524,288 patches per GPU per step,
weak scaling). Prints ONE JSON line on rank 0. Besides the headline keys the line carries three structured
sub-records, each with its own roofline / cpu_baseline / e2e:
    "matching": BASELINE configs[3], mutual-NN + ratio test on synth.make_match_set(65536, 65536, seed=11), query rows and
                gallery rows sharded over the ranks, output verified inside the run;
    "nas":      BASELINE configs[4], wang2 forward at batch 65 536;
    "config1":  BASELINE configs[1], forward x 2 + loss_HardNet at batch 1024 (B200 eager / CUDA graph, CPU, stock torch GPU).
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
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

METRIC = "descriptor_patches_per_sec"
UNIT = "patches/s"
PATCHES_PER_GPU = 524288          # configs[2] shard at 8 GPUs
FLOP_PER_PATCH = 78184448         # SURVEY.md section 8a
NAS_FLOP_PER_PATCH = 7272448      # wang2, SURVEY.md section 8d
NAS_ALGO_BYTES_PER_PATCH = 4608   # 4096 in + 512 out
MATCH_FLOP_PER_PAIR = 256
MATCH_N = 65536
GEN_CHUNK = 65536
REF_SAMPLE = 4096                 # patches per step of the CPU reference arm (bounded sample of the same workload)
DUMP_MAX_ROWS = 65536             # --dump-outputs: 32 MiB of 128-d fp32 descriptors at most


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--patches-per-gpu", type=int, default=PATCHES_PER_GPU)
    ap.add_argument("--no-extras", action="store_true", help="skip the matching / NAS / config-1 sub-records")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the descriptors of the last step (rank 0) as DIR/descriptors.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(directory, **arrays):
    """Write each array as DIR/<name>.npy in float32. An array of more than DUMP_MAX_ROWS rows is sampled: the same seeded,
    sorted row indices on every run, so the dumps of two builds of the project compare row for row."""
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        n = t.shape[0]
        if n > DUMP_MAX_ROWS:
            rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ROWS].sort().values
            t = t[rows.to(t.device)]
            print(f"[bench] {name}: {DUMP_MAX_ROWS} of {n} rows (seeded sample)", file=sys.stderr)
        np.save(d / f"{name}.npy", t.detach().float().cpu().numpy())


def workload_config(args, world):
    return {
        "workload": "BASELINE configs[2]: bulk descriptor extraction, HardNet fp32-in/fp32-out forward, "
                    f"{args.patches_per_gpu} synthetic 32x32 patches per GPU per step "
                    f"({args.patches_per_gpu * world} per step over {world} GPU(s); 4,194,304 at 8 GPUs)",
        "patches_per_gpu_per_step": args.patches_per_gpu,
        "weights": "reference init (torch.manual_seed(0), orthogonal gain 0.6), BN running stats randomised (seed 3), eval mode",
        "activations": "fp16 (10-bit mantissa) with fp32 accumulation",
        "l2_policy": "inputs (2 GiB per GPU per step) are larger than L2; no flush needed",
        "parallelism": f"dp{world} (patch shards, no data-path collective)",
        "reference_arm": f"--impl reference times the unmodified reference HardNet class (oracle/_ref, else the oracle port) on the "
                         f"host cores, one step = a bounded sample of {REF_SAMPLE} patches of this workload",
    }


# ---------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path on the box's host cores
# ---------------------------------------------------------------------------------------------------------
def reference_forward_fn():
    """-> (callable x -> descriptors, kind, description). The unmodified reference class when its sources are available
    (a checkout at ../reference, or the copy build() staged under oracle/_ref), else the oracle port."""
    from oracle import hardnet_oracle, ref_loader, synth
    root = ref_loader.root()
    if root is not None:
        try:
            ref_hardnet, _, _ = ref_loader.load_hardnet(root)
            torch.manual_seed(0)
            model = ref_hardnet.HardNet()
            model.load_state_dict(synth.randomize_bn_stats(model.state_dict(), 3))
            model.eval()

            def fwd(x):
                with torch.no_grad():
                    return model(x)
            return fwd, "reference", f"unmodified hardnet/HardNet.py class imported from {root}"
        except Exception as exc:   # fall back to the port, say why
            print(f"[bench] reference import failed ({exc!r}); timing the oracle port instead", file=sys.stderr)
    w, m, v = synth.hardnet_weights_from_seed(0, 3)
    return (lambda x: hardnet_oracle.hardnet_forward(x, w, m, v)), "port", \
        "oracle/hardnet_oracle.py (torch CPU fp32 restatement of hardnet/HardNet.py:312-315, pinned by tests/golden)"


def cpu_reference_throughput(sample: int, repeats: int = 1):
    from oracle import synth
    fwd, kind, desc = reference_forward_fn()
    x = synth.make_patches(sample, 1234, edge_cases=False)
    fwd(x[:256])  # warm the thread pool / oneDNN primitives
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        fwd(x)
        best = min(best, time.perf_counter() - t0)
    return sample / best, best, kind, desc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import synth
    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    fwd, kind, desc = reference_forward_fn()
    x = synth.make_patches(REF_SAMPLE, 1234, edge_cases=False)
    for _ in range(args.warmup):
        fwd(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = fwd(x)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, descriptors=y)
    value = REF_SAMPLE * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(world, args.gpus)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{REF_SAMPLE} patches per step (bounded sample of the workload); {desc}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, device_index: int):
        self.rows = []
        self.proc = None
        try:
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", uuid], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_start, t_end):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, power, reasons = [], [], [], set()
        for t, line in self.rows:
            if t < t_start or t > t_end + 0.2:
                continue
            f = [c.strip() for c in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(self.NAMES, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(device_index: int):
    """Pin this process to the CPU cores next to its GPU BEFORE it allocates pinned host memory, so the staging buffers are
    first-touched on the GPU's NUMA node (at N = 8 every rank otherwise pins on node 0 and shares one socket's uplinks)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(device_index).uuid)
        if not uuid.startswith("GPU-"):
            uuid = "GPU-" + uuid
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": len(cpus), "first": min(cpus), "last": max(cpus)}
    except Exception as exc:
        return {"error": repr(exc)}
    return None


def make_device_patches(n, device, first_chunk_id):
    """uniform noise smoothed 5x5, generated on the device chunk by chunk from seed 1000 + global chunk id."""
    out = torch.empty((n, 1, 32, 32), dtype=torch.float32, device=device)
    g = torch.Generator(device=device)
    for i, s in enumerate(range(0, n, GEN_CHUNK)):
        m = min(GEN_CHUNK, n - s)
        g.manual_seed(1000 + first_chunk_id + i)
        x = torch.rand((m, 1, 32, 32), generator=g, device=device)
        out[s:s + m] = torch.nn.functional.avg_pool2d(x, 5, 1, 2)
    return out


def randomize_bn_stats(state_dict, seed=3):
    """running_mean ~ 0.1 N(0,1), running_var ~ U(0.5,1.5) (same recipe and seed as the parity tests)."""
    g = torch.Generator().manual_seed(seed)
    out = dict(state_dict)
    for k in sorted(out.keys()):
        if k.endswith("running_mean"):
            out[k] = 0.1 * torch.randn(out[k].shape, generator=g)
        elif k.endswith("running_var"):
            out[k] = 0.5 + torch.rand(out[k].shape, generator=g)
    return out


def load_peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"tflops_sustained": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "tflops_burst": d.get("bf16_tflops"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def load_traffic(stage_name):
    p = REPO / "profiles" / "roofline_traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(stage_name)
        except Exception:
            return None
    return None


class Dist:
    """The few collectives the bench itself needs (timing reductions, barriers)."""

    def __init__(self, world, device):
        self.world, self.device = world, device

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max(self, x: float) -> float:
        if self.world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=self.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, x: float) -> float:
        if self.world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=self.device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())


def timeit(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def h2d_probe(device, D: Dist, nbytes=1 << 30):
    """Aggregate pinned host -> device bandwidth with every rank copying at once: the ceiling of any e2e number."""
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nbytes, dtype=torch.uint8, device=device)
    d.copy_(h, non_blocking=True)
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        d.copy_(h, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    ms = D.max(e0.elapsed_time(e1) / 3)
    D.barrier()
    del h, d
    return D.world * nbytes / (ms / 1e3) / 1e9


def run_b200(args):
    import torch.distributed as dist
    from hardnetnas_b200 import _lib
    from hardnetnas_b200.extract import DescriptorExtractor
    from hardnetnas_b200.hardnet import HardNet

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    D = Dist(world, device)

    lib = _lib.load()
    torch.manual_seed(0)
    model = HardNet()
    model.load_state_dict(randomize_bn_stats(model.state_dict(), 3))
    model = model.to(device).eval()

    P = args.patches_per_gpu
    chunks_per_rank = (P + GEN_CHUNK - 1) // GEN_CHUNK
    x = make_device_patches(P, device, rank * chunks_per_rank)
    out = torch.empty((P, 128), dtype=torch.float32, device=device)

    # ---- warm-up; the first warm-up step is instrumented stage by stage to find the dominant kernel ----
    model(x[:4096], out=out[:4096])
    model.profile_enable(0x7F)
    for w in range(max(args.warmup, 3)):
        model(x, out=out)
        if w == 0:
            torch.cuda.synchronize()
            ms_all, n_all = model.profile_read()
            model.profile_enable(0)
    torch.cuda.synchronize()
    stage_names, stage_macs = HardNet.stage_table(n_all)   # conv3 + conv4 are one kernel when the engine fuses them
    dom = max(range(7), key=lambda i: ms_all[i])
    stage_share = {stage_names[i]: round(ms_all[i] / max(sum(ms_all), 1e-9), 4) for i in range(7) if stage_macs[i] or ms_all[i]}

    # ---- timed region: device-resident inputs ------------------------------------------------------------
    model.profile_enable(1 << dom)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    D.barrier()
    launches0 = lib.hn_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        model(x, out=out)
    e1.record()
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    D.barrier()
    launches = lib.hn_launch_count() - launches0
    ms_total = D.max(e0.elapsed_time(e1))
    clocks = sampler.stop(t_start, t_end) if sampler else None
    dom_ms, dom_n = model.profile_read()
    model.profile_enable(0)
    value = world * P * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, descriptors=out)

    peaks = load_peaks()
    dom_flops = 2.0 * stage_macs[dom] * P * args.steps      # algorithmic FLOPs of that stage over the region
    achieved_tflops = dom_flops / (dom_ms[dom] / 1e3) / 1e12
    flops_per_launch = dom_flops / max(dom_n[dom], 1)
    roofline = {
        "kernel": stage_names[dom], "bound": "tensor", "achieved": achieved_tflops, "peak": peaks["tflops_sustained"],
        "unit": "TFLOP/s", "frac": achieved_tflops / peaks["tflops_sustained"], "traffic": load_traffic(stage_names[dom]),
        "peak_source": peaks["source"] + ", sustained bf16 dense (kernel timed inside a long step)",
        "launches": dom_n[dom], "avg_launch_ms": dom_ms[dom] / max(dom_n[dom], 1), "algorithmic_flop_per_launch": flops_per_launch,
        "stage_time_share_warmup": stage_share,
        "whole_path": {"achieved": value / world * FLOP_PER_PATCH / 1e12, "unit": "TFLOP/s",
                       "frac": value / world * FLOP_PER_PATCH / 1e12 / peaks["tflops_sustained"]},
    }

    # ---- end to end: pinned host buffers, H2D + forward + D2H inside the timed region ------------------------
    h_in = torch.empty((P, 1, 32, 32), dtype=torch.float32, pin_memory=True)
    h_in.copy_(x)
    h_out = torch.empty((P, 128), dtype=torch.float32, pin_memory=True)
    del x, out
    torch.cuda.empty_cache()
    ext = DescriptorExtractor(model, device=device)
    ext(h_in, h_out)
    e2e_steps = max(1, min(args.steps, 5))
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ext(h_in, h_out)
    torch.cuda.synchronize()
    t_e2e = D.max(time.perf_counter() - t0)
    D.barrier()
    e2e = {"value": world * P * e2e_steps / t_e2e, "unit": UNIT, "h2d_bytes_per_step": world * P * 4096,
           "d2h_bytes_per_step": world * P * 512, "steps": e2e_steps,
           "api": f"hardnetnas_b200.extract.DescriptorExtractor (pinned host in/out, {ext.batch}-patch pipelined batches)",
           "pinned_memory_numa_binding": numa}
    # the same pipeline fed with uint8 patches — what the reference's patch datasets hold on disk (hardnet/HardNet.py:174-273
    # reads uint8 PhotoTour bitmaps; input_norm makes the scale irrelevant): 1 KB instead of 4 KB per patch over PCIe
    h_u8 = torch.empty((P, 1, 32, 32), dtype=torch.uint8, pin_memory=True)
    h_u8.copy_((h_in * 255.0).round_().clamp_(0, 255))
    ext8 = DescriptorExtractor(model, device=device, in_dtype=torch.uint8)
    ext8(h_u8, h_out)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ext8(h_u8, h_out)
    torch.cuda.synchronize()
    t_u8 = D.max(time.perf_counter() - t0)
    D.barrier()
    del ext8, h_u8, ext
    e2e_u8 = {"value": world * P * e2e_steps / t_u8, "unit": UNIT, "h2d_bytes_per_step": world * P * 1024,
              "d2h_bytes_per_step": world * P * 512, "steps": e2e_steps, "input": "uint8 patches (dataset storage format)"}
    # host -> device ceiling of this box with all ranks copying at once; e2e as a fraction of what it allows
    h2d_gbs = h2d_probe(device, D)
    for rec, bytes_pp in ((e2e, 4096), (e2e_u8, 1024)):
        rec["h2d_ceiling_GBps_all_ranks"] = h2d_gbs
        rec["h2d_ceiling_patches_per_sec"] = h2d_gbs * 1e9 / bytes_pp
        rec["frac_of_min_h2d_ceiling_and_device_rate"] = rec["value"] / min(h2d_gbs * 1e9 / bytes_pp, value)
    del h_in, h_out
    torch.cuda.empty_cache()

    matching = nas = config1 = keypoints = None
    if not args.no_extras:
        matching = bench_matching(device, rank, world, D, peaks, with_cpu=(rank == 0 and world == 1 and not args.no_cpu_baseline))
        if rank == 0:
            nas = bench_nas(device, peaks, with_cpu=(world == 1 and not args.no_cpu_baseline))
            config1 = bench_config1(device, model, with_cpu=(world == 1 and not args.no_cpu_baseline))
            keypoints = bench_keypoints(device, model, with_cpu=(world == 1 and not args.no_cpu_baseline))
        D.barrier()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        v1, t1, kind, desc = cpu_reference_throughput(1024)
        sample = int(min(32768, max(1024, 1024 * round(10.0 / max(t1, 1e-3)))))
        v, t, kind, desc = cpu_reference_throughput(sample)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                        "sample": f"{sample} patches ({t:.1f} s); {desc}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic", "config": workload_config(args, world), "clocks": clocks, "e2e": e2e,
            "e2e_u8": e2e_u8, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "matching": matching, "nas": nas, "config1": config1, "keypoints": keypoints,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------
# BASELINE configs[3]: mutual-NN + ratio matching, 64k x 64k, rows sharded over the ranks
# ---------------------------------------------------------------------------------------------------------
def bench_matching(device, rank, world, D: Dist, peaks, with_cpu):
    import ctypes as C
    from hardnetnas_b200 import _lib, distributed as hd
    from hardnetnas_b200.matching import mutual_nn_ratio
    from hardnetnas_b200 import _ops
    from oracle import synth
    lib = _lib.load()
    n = MATCH_N
    # SURVEY section 8d match set: 80 % of the queries are noisy copies of gallery rows (d ~ 0.43 against ~1.41 for
    # distractors), 20 % fresh unit vectors (ratio rejections, non-mutual rows); identical on every rank
    q_all, g_all, truth = synth.make_match_set(n, n, seed=11)
    qlo, qhi = hd.shard_range(n, rank, world)
    glo, ghi = hd.shard_range(n, rank, world)
    q, g = q_all[qlo:qhi].to(device), g_all[glo:ghi].to(device)
    q_counts = [hd.shard_range(n, r, world)[1] - hd.shard_range(n, r, world)[0] for r in range(world)]
    rec = {"metric": "nn_match_pairs_per_sec", "unit": "pairs/s",
           "workload": f"BASELINE configs[3]: mutual-NN + ratio test (0.7), {n} x {n} 128-d descriptors, oracle/synth.make_match_set(seed=11) "
                       f"(80 % planted matches, 20 % unmatched queries), query and gallery rows sharded over {world} GPU(s)"}

    if world == 1:
        def step():
            return mutual_nn_ratio(q, g, 0.7, return_pairs=False)
        def fwd_only():
            return _ops.match_top2(q, g)
    else:
        def step():
            # one GEMM per rank + two small all_reduces; masks over this rank's rows
            return (None,) + tuple(hd.mutual_nn_ratio_sharded(q, g, q_counts, q_counts, 0.7))
        def fwd_only():
            return hd.match_sharded(q, g, g_counts=q_counts)

    # ---- correctness inside the run: planted matches recovered, mutual rows consistent, sample vs the CPU oracle ----
    res = step()
    mutual, ratio, fwd = res[1], res[2], res[3]
    t = truth[qlo:qhi].to(device)
    planted = t >= 0
    recovered = (fwd[planted] == t[planted]).float().mean().item()
    mutual_on_planted = mutual[planted].float().mean().item()
    ratio_on_planted = ratio[planted].float().mean().item()
    ratio_on_unmatched = ratio[~planted].float().mean().item() if (~planted).any() else 0.0
    from oracle import losses_oracle
    rows = torch.arange(0, qhi - qlo, max(1, (qhi - qlo) // 256))[:256]
    _, ia, da, db = losses_oracle.ratio_match(q_all[qlo:qhi][rows], g_all)
    sample_exact = bool(torch.equal(fwd[rows.to(device)].cpu(), ia))
    verified = bool(recovered >= 0.999 and mutual_on_planted >= 0.99 and ratio_on_planted >= 0.99 and ratio_on_unmatched <= 0.01
                    and sample_exact)
    verified = bool(D.sum(0.0 if verified else 1.0) == 0.0)
    rec["verified"] = {"ok": verified, "planted_matches_recovered": recovered, "mutual_on_planted": mutual_on_planted,
                       "ratio_accept_on_planted": ratio_on_planted, "ratio_accept_on_unmatched": ratio_on_unmatched,
                       "nn_index_equal_to_cpu_oracle_on_256_rows": sample_exact}
    if not verified:
        print(f"[bench] matching output FAILED verification on rank {rank}: {rec['verified']}", file=sys.stderr)

    # ---- device-resident timing: whole call (both directions) and the forward direction alone ----
    iters = 10
    D.barrier()
    ms = D.max(timeit(step, iters))
    D.barrier()
    ms_fwd = D.max(timeit(fwd_only, iters))
    D.barrier()
    rec["value"] = n * n / (ms / 1e3)
    rec["ms_mutual_plus_ratio"] = ms
    if world == 1:
        from hardnetnas_b200.matching import mutual_nn_ratio_two_pass
        rec["ms_mutual_plus_ratio_two_gemm_passes"] = timeit(lambda: mutual_nn_ratio_two_pass(q, g, 0.7, return_pairs=False), iters)
    rec["ms_forward_direction_only"] = ms_fwd
    rec["forward_only_pairs_per_sec"] = n * n / (ms_fwd / 1e3)
    # ---- roofline from the GEMM kernel's own in-run time (events around its launches inside hn_match) ----
    lib.hn_match_profile_enable(1)
    for _ in range(iters):
        step()
    torch.cuda.synchronize()
    msv, nv = (C.c_double * 3)(), (C.c_longlong * 3)()
    lib.hn_match_profile_read(msv, nv)
    lib.hn_match_profile_enable(0)
    gemm_ms, gemm_n = msv[1], max(nv[1], 1)
    pairs_per_launch = (qhi - qlo) * n          # the one GEMM launch of a step covers local rows x all columns
    ach = MATCH_FLOP_PER_PAIR * pairs_per_launch / (gemm_ms / gemm_n / 1e3) / 1e12
    # a matching call is a ~1 ms burst, not a long power-capped step: the burst bf16 figure is the denominator
    peak = peaks["tflops_burst"] or peaks["tflops_sustained"]
    rec["roofline"] = {"kernel": "match_pair_kernel (GEMM + top-4-chunk shortlist)", "bound": "tensor", "achieved": ach,
                       "peak": peak, "peak_kind": "burst bf16 dense (kernel timed alone in ~1 ms calls)", "unit": "TFLOP/s",
                       "frac": ach / peak, "traffic": None,
                       "avg_launch_ms": gemm_ms / gemm_n, "launches": int(nv[1]), "algorithmic_flop_per_launch": MATCH_FLOP_PER_PAIR * pairs_per_launch,
                       "stage_ms_per_step": {"pack_inside_call": msv[0] / iters, "gemm_shortlist_blockmax": msv[1] / iters,
                                             "exact_rerank": msv[2] / iters,
                                             "claims_and_column_verification": max(ms - (msv[0] + msv[1] + msv[2]) / iters, 0.0)},
                       "whole_call": {"achieved": MATCH_FLOP_PER_PAIR * n * n / world / (ms / 1e3) / 1e12,
                                      "frac": MATCH_FLOP_PER_PAIR * n * n / world / (ms / 1e3) / 1e12 / peak,
                                      "note": "whole mutual-NN + ratio call (GEMM, exact re-rank, claims, column verification) at 256 FLOP/pair"}}
    if world > 1:
        # compute-only: the same kernels on already gathered operands (no collective inside the timed region)
        import torch.distributed as dist
        g_full = hd.all_gather_rows(g, q_counts)
        g16 = _ops.pack_descriptors(g_full)
        ms_compute = D.max(timeit(lambda: _ops.match_top2(q, g_full, g16=g16), iters))
        rec["forward_only_compute_ms_no_collective"] = ms_compute
        rec["forward_only_comm_inclusive_ms"] = ms_fwd
        del g_full, g16
    # ---- e2e: host buffers in, host results out ----
    if world == 1:
        hq, hg = q_all.pin_memory(), g_all.pin_memory()
        dq, dg = torch.empty_like(q), torch.empty_like(g)
        hm = torch.empty(n, dtype=torch.bool, pin_memory=True)
        hr = torch.empty(n, dtype=torch.bool, pin_memory=True)
        hi = torch.empty(n, dtype=torch.int64, pin_memory=True)

        def e2e_step():
            dq.copy_(hq, non_blocking=True)
            dg.copy_(hg, non_blocking=True)
            _, m_, r_, i_, _, _ = mutual_nn_ratio(dq, dg, 0.7, return_pairs=False)
            hm.copy_(m_, non_blocking=True); hr.copy_(r_, non_blocking=True); hi.copy_(i_, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        e2e_step()
        t0 = time.perf_counter()
        for _ in range(5):
            e2e_step()
        dt = (time.perf_counter() - t0) / 5
        rec["e2e"] = {"value": n * n / dt, "unit": "pairs/s", "h2d_bytes_per_step": 2 * n * 512, "d2h_bytes_per_step": n * 10,
                      "api": "hardnetnas_b200.matching.mutual_nn_ratio on pinned host descriptors (H2D, match, D2H of masks + indices)"}
        del hq, hg, dq, dg
    if with_cpu:
        torch.set_num_threads(os.cpu_count() or 1)
        nq_s = 4096
        try:
            from oracle import ref_loader
            eval_utils, _ = ref_loader.load_fdl()
            kp = torch.zeros((n, 3))
            t0 = time.perf_counter()
            eval_utils.nearest_neighbor_distance_ratio_match(q_all[:nq_s], g_all, kp, 0.7)
            dt = time.perf_counter() - t0
            kind, what = "reference", "unmodified FDLNet-master/utils/eval_utils.py:168-175 (full distance matrix + row sort)"
        except Exception:
            t0 = time.perf_counter()
            losses_oracle.ratio_match(q_all[:nq_s], g_all, 0.7)
            dt = time.perf_counter() - t0
            kind, what = "port", "oracle/losses_oracle.ratio_match (top-2 instead of the reference's full row sort)"
        rec["cpu_baseline"] = {"value": nq_s * n / dt, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": kind,
                               "sample": f"{nq_s} x {n} query chunk, ratio test only, one direction ({dt:.1f} s); {what}"}
    return rec


# ---------------------------------------------------------------------------------------------------------
# BASELINE configs[4]: NAS-derived descriptor net (wang2) at batch 65 536
# ---------------------------------------------------------------------------------------------------------
def bench_nas(device, peaks, with_cpu):
    from hardnetnas_b200.extract import DescriptorExtractor
    from hardnetnas_b200.nas import SampledDescriptorNet
    from oracle import synth
    B = 65536
    torch.manual_seed(0)
    nas = SampledDescriptorNet("wang2")
    nas.load_state_dict(synth.randomize_nas_state(nas.state_dict(), 4))
    sd = {k: v.clone() for k, v in nas.state_dict().items()}
    nas = nas.to(device).eval()
    g = torch.Generator(device=device).manual_seed(5)
    xb = torch.nn.functional.avg_pool2d(torch.rand((B, 1, 32, 32), generator=g, device=device), 5, 1, 2)
    ob = torch.empty((B, 128), dtype=torch.float32, device=device)
    nas(xb, out=ob)
    ms = timeit(lambda: nas(xb, out=ob), 10)
    rate = B / (ms / 1e3)
    moved = load_traffic("nas_wang2_bytes_per_patch")
    rec = {"metric": "nas_descriptor_patches_per_sec", "unit": "patches/s", "value": rate, "ms_per_step": ms,
           "workload": f"BASELINE configs[4]: sampled NAS descriptor net wang2 (hardnetNAS fbnet_building_blocks), eval forward at batch {B}, "
                       "fp32 in / fp32 out, fp16 activations",
           "launch_plan": {"tail_launches": nas.resident_plan(), "launches_per_pass": 2 + len(nas.resident_plan()),
                           "note": "fused front kernel (stem + pw + stride-2 dw) + warpgroup-per-patch tail launches (first packed op, last packed op, "
                                   "patches in flight per CTA, 0) with the linear 1x1 convs folded into their consumers + head GEMM; "
                                   "ncu launch list profiles/r2_nas_launch_table_tail.txt"},
           "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peaks["hbm_gbs"],
                        "achieved": rate * NAS_ALGO_BYTES_PER_PATCH / 1e9, "frac": rate * NAS_ALGO_BYTES_PER_PATCH / 1e9 / peaks["hbm_gbs"],
                        "algorithmic_bytes_per_patch": NAS_ALGO_BYTES_PER_PATCH,
                        "moved_bytes_per_patch": moved, "moved_GBps": (rate * moved / 1e9) if moved else None,
                        "moved_frac": (rate * moved / 1e9 / peaks["hbm_gbs"]) if moved else None, "traffic": moved,
                        "tensor": {"achieved": rate * NAS_FLOP_PER_PATCH / 1e12, "unit": "TFLOP/s", "peak": peaks["tflops_sustained"],
                                   "frac": rate * NAS_FLOP_PER_PATCH / 1e12 / peaks["tflops_sustained"]}}}
    # e2e through the host pipeline
    h_in = torch.empty((B, 1, 32, 32), dtype=torch.float32, pin_memory=True)
    h_in.copy_(xb)
    h_out = torch.empty((B, 128), dtype=torch.float32, pin_memory=True)
    ext = DescriptorExtractor(nas, device=device)
    ext(h_in, h_out)
    t0 = time.perf_counter()
    for _ in range(5):
        ext(h_in, h_out)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 5
    rec["e2e"] = {"value": B / dt, "unit": "patches/s", "h2d_bytes_per_step": B * 4096, "d2h_bytes_per_step": B * 512,
                  "api": "hardnetnas_b200.extract.DescriptorExtractor(SampledDescriptorNet('wang2')) on pinned host buffers"}
    # the same pipeline fed with uint8 patches (1 KB instead of 4 KB per patch over PCIe: the fp32 line is bound by the host link)
    h_u8 = torch.empty((B, 1, 32, 32), dtype=torch.uint8, pin_memory=True)
    h_u8.copy_((h_in * 255.0).round_().clamp_(0, 255))
    ext8 = DescriptorExtractor(nas, device=device, in_dtype=torch.uint8)
    ext8(h_u8, h_out)
    t0 = time.perf_counter()
    for _ in range(5):
        ext8(h_u8, h_out)
    torch.cuda.synchronize()
    dt8 = (time.perf_counter() - t0) / 5
    rec["e2e_u8"] = {"value": B / dt8, "unit": "patches/s", "h2d_bytes_per_step": B * 1024, "d2h_bytes_per_step": B * 512,
                     "input": "uint8 patches (dataset storage format)"}
    del ext8, h_u8
    if with_cpu:
        from oracle import nas_oracle
        from hardnetnas_b200.nas.fbnet_modeldef import arch_ops
        torch.set_num_threads(os.cpu_count() or 1)
        xs = h_in[:2048].clone()
        nas_oracle.nas_forward(xs[:256], arch_ops("wang2"), sd)
        t0 = time.perf_counter()
        nas_oracle.nas_forward(xs, arch_ops("wang2"), sd)
        dtc = time.perf_counter() - t0
        rec["cpu_baseline"] = {"value": 2048 / dtc, "unit": "patches/s", "cores": torch.get_num_threads(), "kind": "port",
                               "sample": f"2048 patches ({dtc:.1f} s), oracle/nas_oracle.py (functional restatement of the sampled net; "
                                         "the reference has no class that builds it, SURVEY.md section 3.4)"}
    return rec


# ---------------------------------------------------------------------------------------------------------
# BASELINE configs[1]: forward x 2 + loss_HardNet at batch 1024
# ---------------------------------------------------------------------------------------------------------
def bench_config1(device, model, with_cpu):
    from hardnetnas_b200.losses import _masked_matrix, loss_HardNet
    g = torch.Generator(device=device).manual_seed(7)
    a = torch.nn.functional.avg_pool2d(torch.rand((1024, 1, 32, 32), generator=g, device=device), 5, 1, 2)
    p = a + 0.1 * torch.randn(a.shape, generator=g, device=device)
    rec = {"workload": "BASELINE configs[1]: HardNet forward of 1024 anchors + 1024 positives and loss_HardNet (min, triplet_margin, "
                       "anchor swap), one step", "unit": "ms"}

    def step():
        da, dp = model(a), model(p)
        return loss_HardNet(da, dp, anchor_swap=True)
    rec["b200_eager_ms"] = timeit(step, 20)
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            step()
        rec["b200_cuda_graph_ms"] = timeit(graph.replay, 50)
        del graph
    except Exception as exc:   # a capture problem must not take the bench line down
        rec["b200_cuda_graph_ms"] = None
        print(f"[bench] CUDA graph capture of the config-1 step failed: {exc}", file=sys.stderr)
    da, dp = model(a), model(p)
    rec["b200_loss_only_ms"] = timeit(lambda: loss_HardNet(da, dp, anchor_swap=True), 50)

    # The same step with the anchors and positives in ONE forward of 2048 patches (eval-mode BatchNorm: identical descriptors;
    # the concatenation is inside the timed step). Seven kernel prologues instead of fourteen.
    def step_one_forward():
        d = model(torch.cat([a, p]))
        return loss_HardNet(d[:1024], d[1024:], anchor_swap=True)
    try:
        rec["b200_one_forward_of_2048_eager_ms"] = timeit(step_one_forward, 20)
        # (the split-K factor of the head GEMM follows the batch size: last-bit differences between the two forms)
        rec["one_forward_vs_two_max_abs_diff"] = float((model(torch.cat([a, p])) - torch.cat([da, dp])).abs().max().item())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            step_one_forward()
        rec["b200_one_forward_of_2048_cuda_graph_ms"] = timeit(graph.replay, 50)
        del graph
    except Exception as exc:
        print(f"[bench] single-forward variant of the config-1 step failed: {exc}", file=sys.stderr)

    # the reference's own op sequence on the same GPU (stock torch modules: cuDNN / cuBLAS, TF32 allowed) for the same step
    def stock_step():
        with torch.no_grad():
            xa, xp = model.forward_stock(a), model.forward_stock(p)
            pos, d = _masked_matrix(xa, xp)
            mn = torch.min(d.min(dim=1)[0], d.min(dim=0)[0])
            return torch.clamp(1.0 + pos - mn, min=0.0).mean()
    rec["stock_torch_gpu_ms"] = timeit(stock_step, 10)
    xs = torch.nn.functional.avg_pool2d(torch.rand((65536, 1, 32, 32), generator=g, device=device), 5, 1, 2)
    with torch.no_grad():
        rec["stock_torch_gpu_tf32_patches_per_sec_batch65536"] = 65536 / (timeit(lambda: model.forward_stock(xs), 5) / 1e3)
        with torch.autocast("cuda", dtype=torch.float16):
            rec["stock_torch_gpu_fp16_autocast_patches_per_sec_batch65536"] = 65536 / (timeit(lambda: model.forward_stock(xs), 5) / 1e3)
    del xs
    if with_cpu:
        from oracle import losses_oracle
        torch.set_num_threads(os.cpu_count() or 1)
        fwd, kind, desc = reference_forward_fn()
        ac, pc = a.cpu(), p.cpu()
        fwd(ac[:64])

        def cpu_step():
            return losses_oracle.loss_hardnet(fwd(ac), fwd(pc), True)
        cpu_step()
        t0 = time.perf_counter()
        for _ in range(3):
            cpu_step()
        rec["cpu_ms"] = (time.perf_counter() - t0) / 3 * 1e3
        rec["cpu_kind"] = f"{kind} forward ({desc}) + oracle loss (hardnet/Losses.py:87-154 without its hard-coded .cuda()), {torch.get_num_threads()} threads"
    return rec


# ---------------------------------------------------------------------------------------------------------
# SURVEY.md section 8f row 2: keypoints -> descriptors (the caller right upstream of the descriptor in RFNetSO.inference,
# FDLNet-master/latency/rfnet/model/rf_net_so.py:160-180: clip_patch, then des(patches))
# ---------------------------------------------------------------------------------------------------------
def bench_keypoints(device, model, with_cpu):
    from hardnetnas_b200.image_utils import clip_patch
    B, k, H, W = 16, 16384, 480, 640
    g = torch.Generator().manual_seed(1)
    images = torch.nn.functional.avg_pool2d(torch.rand(B, 1, H, W, generator=g), 5, 1, 2)
    img8 = (images * 255).round().to(torch.uint8).to(device)
    imgf = img8.float()
    ys, xs = torch.randint(0, H // 2, (B, k), generator=g), torch.randint(0, W // 2, (B, k), generator=g)
    bs = torch.arange(B)[:, None].expand(B, k)
    byxc_h = torch.stack([bs, ys, xs, torch.zeros_like(ys)], dim=-1).view(-1, 4).long()
    scale_h = 6.0 + 34.0 * torch.rand(B * k, generator=g)
    ang = 6.2831853 * torch.rand(B * k, generator=g)
    ori_h = torch.stack([torch.cos(ang), torch.sin(ang)], dim=-1)
    info_h = torch.full((B, 2), 0.5)
    byxc, scale, ori, info = byxc_h.to(device), scale_h.to(device), ori_h.to(device), info_h.to(device)
    n = B * k
    two = model(clip_patch(byxc, scale, ori, info, imgf, 32))
    one = model.forward_clip(byxc, scale, ori, info, img8)
    patches = clip_patch(byxc, scale, ori, info, imgf, 32)
    t_clip = timeit(lambda: clip_patch(byxc, scale, ori, info, imgf, 32), 5)
    t_fwd = timeit(lambda: model(patches), 5)
    del patches
    t_two = timeit(lambda: model(clip_patch(byxc, scale, ori, info, imgf, 32)), 5)
    t_one = timeit(lambda: model.forward_clip(byxc, scale, ori, info, img8), 5)
    rec = {"workload": f"keypoints -> descriptors: clip_patch (scale / orientation / bilinear, psize 32) + HardNet forward, {n} keypoints "
                       f"on {B} images of {H}x{W} (scales 6-40 px, random orientation), images resident on the device",
           "metric": "keypoint_descriptors_per_sec", "unit": "keypoints/s",
           "value": n / t_two * 1e3,
           "ms_clip_patch_then_forward": t_two, "ms_clip_patch_alone": t_clip, "ms_forward_of_ready_patches": t_fwd,
           "forward_clip": {"value": n / t_one * 1e3, "ms": t_one, "input": "uint8 images, no patch tensor (crop inside the front kernel)",
                            "bit_identical_to_two_calls": bool(torch.equal(one, two)),
                            "device_memory_saved_bytes": n * 4096},
           "roofline": {"kernel": "clip_patch32_kernel", "bound": "hbm", "unit": "GB/s", "achieved": n * 4096 / t_clip / 1e6,
                        "peak": load_peaks()["hbm_gbs"], "traffic": None,
                        "note": "algorithmic bytes = the 4 KiB patch written (the gathered image pixels stay in L2)"}}
    if rec["roofline"]["peak"]:
        rec["roofline"]["frac"] = rec["roofline"]["achieved"] / rec["roofline"]["peak"]
    if with_cpu:
        from oracle import clip_oracle
        torch.set_num_threads(os.cpu_count() or 1)
        m = 4096
        fwd, kind, desc = reference_forward_fn()
        t0 = time.perf_counter()
        pc = clip_oracle.clip_patch(byxc_h[:m], scale_h[:m], ori_h[:m], info_h[:1], images[:1], 32)
        with torch.no_grad():
            fwd(pc)
        dt = time.perf_counter() - t0
        rec["cpu_baseline"] = {"value": m / dt, "unit": "keypoints/s", "cores": torch.get_num_threads(), "kind": "port+" + kind,
                               "sample": f"{m} keypoints of image 0 ({dt:.1f} s): oracle/clip_oracle.py (restatement of image_utils.py:11-158) + {desc}"}
    return rec


def emit(line: dict):
    """The ONE JSON line goes to the real stdout; everything else any library prints was diverted to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    args = parse_args()
    # libraries (NCCL's version banner, torchrun, the reference's import-time prints) write to fd 1: keep stdout clean for the
    # single result line
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
