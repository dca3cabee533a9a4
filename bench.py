#!/usr/bin/env python
"""bench.py -- images/sec of the ViT-B/16 224^2 bf16 forward pass (BASELINE.json `metric`, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config vit_b16|vit_l16_384|...]
                    [--dump-outputs DIR]

One "step" is one forward pass over one synthetic batch (256 images per GPU).  N > 1 is launched by torchrun, one
rank per GPU: the batch is sharded data-parallel (weak scaling: 256 images per GPU), the forward has no
communication and ends with ONE NCCL all-gather of the logits.  Rank 0 prints ONE JSON line.

`value`        whole-job images/s with the inputs already resident in HBM (device-timed with CUDA events,
               barrier + synchronize on both sides, max over ranks).
`e2e`          the same metric through the public host-buffer API (vit_tensorflow_b200.runtime.HostPipeline):
               every step copies its images from pinned host memory and reads the logits back to the host.
`roofline`     tcgen05 GEMM kernel (>= 95 % of the FLOPs): algorithmic FLOPs / device time of its launches, timed
               inside the timed region with CUDA events on the launch stream, against MEASURED_PEAKS.json.
`cpu_baseline` the oracle's torch-CPU restatement of the reference (TensorFlow is not installable here) on a
               bounded sample, on the host cores of the same box.
`--impl reference` times that CPU restatement as the reference arm.

`--dump-outputs DIR` writes, after the timed steps, what the timed path returned in its last step: `DIR/logits.npy`, float32
[global batch, classes] (for `--impl reference`, the CPU restatement's logits of its sample).  Weights and images come from
fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from untouched (no __pycache__)

CONFIGS = {
    # BASELINE.json configs[1] -- the configuration the metric is quoted on
    "vit_b16": dict(kind="vit", image_size=224, patch_size=16, num_classes=1000, dim=768, depth=12, heads=12, mlp_dim=3072, batch=256),
    # parity-test configurations, runnable as bench lines on request
    "vit_tiny_gate": dict(kind="vit", image_size=224, patch_size=16, num_classes=1000, dim=192, depth=1, heads=3, mlp_dim=768, batch=2),
    "deepvit": dict(kind="deepvit", image_size=224, patch_size=16, num_classes=1000, dim=1024, depth=24, heads=16, mlp_dim=4096, batch=128),
    "cait_s36": dict(kind="cait", image_size=224, patch_size=16, num_classes=1000, dim=384, depth=36, cls_depth=2, heads=8,
                     mlp_dim=1536, dim_head=48, batch=128),
    "vit_l16_384": dict(kind="vit", image_size=384, patch_size=16, num_classes=1000, dim=1024, depth=24, heads=16, mlp_dim=4096, batch=128),
    # the reference README's usage examples of the two remaining hot-path model classes (README.md:327-345, :208-216)
    "crossvit_readme": dict(kind="crossvit", image_size=256, num_classes=1000, depth=4, sm_dim=192, sm_patch_size=16, sm_enc_depth=2,
                            sm_enc_heads=8, sm_enc_mlp_dim=2048, lg_dim=384, lg_patch_size=64, lg_enc_depth=3, lg_enc_heads=8,
                            lg_enc_mlp_dim=2048, cross_attn_depth=2, cross_attn_heads=8, batch=256),
    "t2t_readme": dict(kind="t2t_vit", image_size=224, num_classes=1000, dim=512, depth=5, heads=8, mlp_dim=512,
                       t2t_layers=((7, 4), (3, 2), (3, 2)), batch=64),
}
METRIC = "images/sec ViT-B/16 224^2 bf16 forward"


def metric_name(workload):
    """BASELINE.json's metric for the configuration it is quoted on; the other configurations are labelled as what they are."""
    return METRIC if workload == "vit_b16" else f"images/sec {workload} bf16 forward (not the configuration BASELINE.json's metric is quoted on)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(source="measured", hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]))
    # fallback stated by /opt/skills/guides/B200_PROFILING.md
    return dict(source="fallback", hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.limit")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def wait_ready(self, timeout=4.0):
        """nvidia-smi needs ~1 s before its first sample; make sure it is sampling before the timed region starts."""
        t0 = time.perf_counter()
        while self.p is not None and time.perf_counter() - t0 < timeout:
            try:
                if os.path.getsize(self.f.name) > 0:
                    return
            except OSError:
                pass
            time.sleep(0.05)

    def stop(self):
        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons, limit = [], [], [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.strip().lower() == "active":
                    reasons.add(n)
            try:
                limit = float(r[7])      # enforced board power limit: boxes of this pool differ (about 500 W ... 1000 W)
            except Exception:
                pass
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
        return dict(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), power_w_max=max(pw), power_limit_w=limit, samples=len(sm),
                    reasons=sorted(reasons))


def oracle_cfg(c):
    import oracle
    kw = {k: v for k, v in c.items() if k not in ("kind", "batch")}
    return oracle.make_config(c["kind"], **kw)


def ncu_dram_traffic(config):
    """DRAM bytes (read + write) per GEMM launch from the committed ncu capture of this bench command, or None.
    The number is from a profiler run (cold caches, serialised kernels); it is reported next to the live timing, never
    measured inside it."""
    root = os.path.dirname(os.path.abspath(__file__))
    for rnd in ("r02", "r01"):                      # newest committed capture first
        path = os.path.join(root, "profiles", f"{rnd}_dram_traffic_{config}.json")
        try:
            with open(path) as fh:
                d = json.load(fh)
            return d["gemm_class"]["dram_bytes_per_launch"], os.path.relpath(path, root)
        except (OSError, KeyError, ValueError):
            continue
    return None, None


def usable_cores():
    """Host threads this process may really use: scheduler affinity capped by the cgroup CPU quota (a container that
    sees 128 logical CPUs but owns a fraction of them thrashes with 128 torch threads)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


# --------------------------------------------------------------------------------------------- CPU arm
def time_cpu_reference(c, budget_s, steps, warmup, log=None):
    """Restated reference (oracle/ref_torch.py, torch CPU fp32, all host threads) on a bounded sample.  `budget_s` (None: no
    budget) stops the timed loop early once exceeded; returns (summary, ms per forward, batch, logits of the last forward)."""
    import numpy as np
    import torch
    import oracle
    from oracle import ref_torch
    cores = usable_cores()
    torch.set_num_threads(cores)
    cfg = oracle_cfg(c)
    w = oracle.init_weights(cfg, 0)
    ref = ref_torch.TorchReference(w, cfg)
    b = int(min(32, c["batch"]))
    img = oracle.make_image(cfg, b, 1)
    t_start = time.perf_counter()
    for _ in range(warmup):
        ref(img)
    ts = []
    out = None
    for _ in range(steps):
        t0 = time.perf_counter(); out = ref(img); ts.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_start > budget_s:
            break
    steps = len(ts)
    t = sum(ts) / len(ts)
    return dict(value=b / t, unit="images/s", cores=cores, kind="port",
                sample=f"{steps} timed forwards of a {b}-image batch after {warmup} warm-up (torch {torch.__version__} CPU fp32 "
                       f"restatement of vit_tensorflow; TensorFlow not installable in this image)"), t * 1e3, b, out


def run_reference(args, c):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, ms, b, out = time_cpu_reference(c, budget_s=None, steps=args.steps, warmup=args.warmup)
    if args.dump_outputs:
        dump_logits(args.dump_outputs, out)
    line = dict(impl="reference", metric=metric_name(args.config), value=cb["value"], unit="images/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", config=dict(workload=args.config, kind=c["kind"], sample_batch=b,
                                              note="CPU arm: the reference has no GPU/distributed path; rank 0 only"),
                cpu_baseline=cb, e2e=dict(value=cb["value"], unit="images/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- GPU arm
def run_ours(args, c):
    import numpy as np
    import torch
    import torch.distributed as dist
    import oracle
    from vit_tensorflow_b200 import build, from_config
    from vit_tensorflow_b200.runtime import DataParallel, HostPipeline, NativeDataParallel, bind_to_gpu_numa, init_distributed

    numa_node = bind_to_gpu_numa(int(os.environ.get("LOCAL_RANK", "0")))   # before any pinned allocation (first touch)
    rank, world, local = init_distributed("nccl")
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()

    cfg = oracle_cfg(c)
    B, H, W = c["batch"], cfg["image_h"], cfg["image_w"]
    model = from_config(cfg, precision=args.precision, device=local, seed=0)     # random-init weights, same on all ranks
    # N > 1: the C-ABI's own data-parallel entry (vb_dp_init / vb_forward_allgather: forward + in-place ncclAllGather of the
    # logits on one stream); N = 1: the plain forward (no collective exists)
    native_dp = world > 1 and not args.torch_dp
    dp = NativeDataParallel(model, B, (H, W), rank, world) if native_dp else DataParallel(model, B, (H, W), rank, world)
    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)
    img_host = torch.randn((B, H, W, 3), generator=gen, dtype=torch.float32).pin_memory()
    img_dev = img_host.to(dev)
    flops_img = oracle.flops_per_image(cfg)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput ----------------------------------------------------------------
    sampler = ClockSampler(local)
    for _ in range(max(args.warmup, 3)):
        dp.forward_device(img_dev)
    barrier()
    sampler.wait_ready()
    for _ in range(3):                      # keep the GPU under load while the first samples are taken
        dp.forward_device(img_dev)
    barrier()
    launches_per_step = model.last_launch_count + (1 if world > 1 else 0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out_dev = dp.forward_device(img_dev)
    ev1.record()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    last_logits = out_dev.float().cpu().numpy() if args.dump_outputs else None     # the buffer is reused by the passes below
    # the same K steps again with per-kernel-class CUDA events on the launch stream (roofline numbers); the event
    # records between kernels defeat programmatic dependent launch, so this pass is a little slower than `value`
    model.profile(True)
    model.profile_read(reset=True)
    pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    pv0.record()
    for _ in range(args.steps):
        dp.forward_device(img_dev)
    pv1.record()
    barrier()
    ms_profiled = pv0.elapsed_time(pv1)
    prof = model.profile_read(reset=True)
    model.profile(False)
    clocks = sampler.stop()
    logits = dp.gathered.float().cpu().numpy()
    assert np.isfinite(logits).all()
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)

    # ---- end to end through the public host-buffer API ---------------------------------------------
    pipe = HostPipeline(dp)
    for _ in range(3):
        pipe.submit(img_host)
    pipe.flush()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(pipe.copy_stream)
    checksum = 0.0
    for _ in range(args.steps):
        prev = pipe.submit(img_host)
        if prev is not None:
            checksum += float(prev[0, 0])
    last = pipe.flush()
    checksum += float(last[0, 0])
    e1.record(pipe.compute_stream)
    torch.cuda.synchronize(dev)
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), wall_ms)) / args.steps
    e2e = dict(value=world * B / (e2e_ms * 1e-3), unit="images/s", h2d_bytes_per_step=pipe.h2d_bytes,
               d2h_bytes_per_step=pipe.d2h_bytes, ms_per_step=e2e_ms,
               api="vit_tensorflow_b200.runtime.HostPipeline.submit (pinned host images in, host logits out, "
                   "H2D of step i overlapped with compute of step i-1)")

    # ---- roofline of the dominant kernel (tcgen05 GEMM), timed inside the timed region ---------------
    peaks = load_peaks()
    gemm_classes = ("gemm_tcgen05", "gemm_tcgen05_gelu", "gemm_tcgen05_residual")
    g = {k: sum(prof[c][k] for c in gemm_classes) for k in ("ms", "flops", "bytes", "launches")}
    roof = None
    if g["launches"] > 0 and g["ms"] > 0:
        achieved = g["flops"] / (g["ms"] * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        traffic, traffic_src = ncu_dram_traffic(args.config)
        roof = dict(bound="tensor", kernel="gemm_bf16_kernel (tcgen05, all epilogue variants)", achieved=achieved, peak=peak,
                    unit="TFLOP/s", frac=achieved / peak, traffic=traffic, traffic_source=traffic_src,
                    algorithmic_bytes_per_launch=g["bytes"] / g["launches"],
                    peak_source=f"{peaks['source']} MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step); "
                                f"burst peak {peaks['bf16_tflops']}",
                    launches=g["launches"], avg_launch_ms=g["ms"] / g["launches"],
                    share_of_step=g["ms"] / ms_profiled, profiled_ms_per_step=ms_profiled / args.steps,
                    end_to_end_frac=(value / world) * flops_img / 1e12 / peak,
                    # the same two fractions against the BURST cuBLAS figure (a kernel timed alone, not under the power cap)
                    frac_of_burst=achieved / peaks["bf16_tflops"],
                    end_to_end_frac_of_burst=(value / world) * flops_img / 1e12 / peaks["bf16_tflops"],
                    by_epilogue={k: dict(ms_per_step=prof[k]["ms"] / args.steps, launches_per_step=prof[k]["launches"] / args.steps,
                                         tflops=prof[k]["flops"] / (prof[k]["ms"] * 1e-3) / 1e12)
                                 for k in gemm_classes if prof[k]["launches"]},
                    other_kernels={k: dict(ms_per_step=v["ms"] / args.steps, launches_per_step=v["launches"] / args.steps,
                                           gbps=(v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else None),
                                           tflops=(v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 and v["flops"] else None))
                                   for k, v in prof.items() if k not in gemm_classes and v["launches"]})

    all_clocks = [clocks]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, clocks)
        all_clocks = gathered
    if rank == 0:
        sm = [c_["sm_mhz"] for c_ in all_clocks if c_.get("sm_mhz")]
        reasons = sorted(set(r for c_ in all_clocks for r in c_.get("reasons", [])))
        clocks_out = dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=clocks.get("sm_max_mhz"), reasons=reasons,
                          power_w_max=clocks.get("power_w_max"), power_limit_w=clocks.get("power_limit_w"))
        cb = None
        if world == 1 and not args.no_cpu_baseline:
            cb, _, _, _ = time_cpu_reference(c, budget_s=20.0, steps=3, warmup=1)
        line = dict(metric=metric_name(args.config), value=value, unit="images/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="bf16" if args.precision == "bf16" else "f32", data="synthetic",
                    config=dict(workload=args.config, kind=c["kind"], per_gpu_batch=B, global_batch=world * B,
                                image=[H, W], parallelism=f"dp{world}", flops_per_image=flops_img,
                                collective=("vb_forward_allgather (C-ABI, NCCL all-gather of the logits)" if native_dp else
                                            ("torch.distributed all_gather_into_tensor" if world > 1 else "none")),
                                numa_node_rank0=numa_node,
                                l2="inputs larger than L2 (154 MB images, >1 GB activations per step; no flush needed)",
                                weights="random init (reference distributions), seed 0"),
                    e2e=e2e, gpu_launches=int(launches_per_step * args.steps), clocks=clocks_out, roofline=roof,
                    cpu_baseline=cb, tflops_end_to_end=value * flops_img / 1e12, e2e_checksum=checksum)
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_logits(args.dump_outputs, last_logits)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_logits(directory, logits):
    """DIR/logits.npy, float32; at most 64 MB (the logits of every configuration here at its default batch are about 1 MB)."""
    import numpy as np
    a = np.ascontiguousarray(logits, dtype=np.float32)
    if a.nbytes > 64 << 20:
        raise SystemExit(f"--dump-outputs: logits of {a.nbytes >> 20} MB exceed the 64 MB a dump may take")
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "logits.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="vit_b16", choices=sorted(CONFIGS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=None, help="override the per-GPU batch of the config")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--torch-dp", action="store_true", help="N > 1: torch.distributed for the all-gather instead of the C-ABI's own NCCL path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's logits to DIR/logits.npy (float32) for output-for-output comparison of builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    c = dict(CONFIGS[args.config])
    if args.batch:
        c["batch"] = args.batch
    if args.impl == "reference":
        run_reference(args, c)
    else:
        run_ours(args, c)


if __name__ == "__main__":
    main()
