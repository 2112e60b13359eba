#!/usr/bin/env python
"""Benchmark of the UniDepthV2.infer() hot path (see BASELINE.json / SURVEY.md section 8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|torch-gpu] [--workload default|hires|v1]
                    [--dump-outputs DIR]

A "step" = one `infer` pass over one batch of synthetic uint8 RGB.  Workloads (BASELINE.json `configs`):
  default  configs[1]/[2]: ViT-L/14, 8 x 3x480x640 per GPU  (the configuration the metric is quoted on)
  hires    configs[4]:     ViT-L/14, 4 x 3x1024x1536 per GPU (infer resizes to 644x952 -> 3129 tokens)
  v1       configs[3]:     UniDepthV1 ConvNeXt-L, 16 x 3x480x640 per GPU (fixed network shape 462x616; conv path)
Rank 0 prints ONE JSON line.  `value` = images/s with inputs resident in HBM (whole job, max over
ranks); `e2e` = images/s through the public API with pinned-host input -> H2D -> infer -> D2H of
depth + intrinsics inside the timed region (`e2e_full`: D2H of the whole seven-tensor output dict).
`--impl reference` times the reference algorithm's CPU implementation (the torch-fp32 oracle port;
/root/reference does not exist on the GPU box).  `--impl torch-gpu` is an INFORMATIVE extra arm, never the
product: the same oracle port run by stock PyTorch on the GPU under fp16 autocast (what the reference itself does
on a GPU, unidepthv2.py:239-241) -- the "kernel to beat on the same box" of BASELINE.md section 4.
`--dump-outputs DIR` writes the outputs of the last timed step as DIR/<name>.npy (see dump_outputs) so that two builds
can be compared output for output: weights and inputs are seeded, identical from run to run with the same arguments.
"""
from __future__ import annotations

import argparse
import copy
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: no bytecode cache next to the sources

import torch  # noqa: E402

# algorithmic FLOPs per image: SURVEY.md section 8d / BASELINE.md section 2
WORKLOADS = {
    "default": dict(flops=1648.56e9, batch=8, hw=(480, 640),
                    desc=dict(model="UniDepthV2 ViT-L/14", batch_per_gpu=8, input="3x480x640 uint8", net_input="490x644",
                              baseline_config="configs[1] (N=1) / configs[2] (N=8)")),
    "hires": dict(flops=3708.02e9, batch=4, hw=(1024, 1536),
                  desc=dict(model="UniDepthV2 ViT-L/14", batch_per_gpu=4, input="3x1024x1536 uint8", net_input="644x952 (3129 tokens)",
                            baseline_config="configs[4] (long-sequence attention)")),
    # SURVEY.md section 8a row a20: encoder 375.35 GF + decoder ~145 GF (the Nystrom part approximate); the line also reports
    # the flops the launched GEMM / attention kernels declared (roofline.declared_tflop_per_step)
    "v1": dict(flops=520.0e9, batch=16, hw=(480, 640), v1=True,
               desc=dict(model="UniDepthV1 ConvNeXt-L", batch_per_gpu=16, input="3x480x640 uint8", net_input="462x616 (fixed)",
                         baseline_config="configs[3] (conv path)")),
}


def load_config(workload="default"):
    name = "config_v1_cnvnxtl.json" if WORKLOADS[workload].get("v1") else "config_v2_vitl14.json"
    return json.load(open(os.path.join(ROOT, "tests", "golden", name)))


def oracle_for(workload):
    """(make_state_dict(cfg, seed), infer(sd, cfg, rgb)) of the CPU oracle for this workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from fixture import make_state_dict, make_v1_state_dict
    if WORKLOADS[workload].get("v1"):
        import unidepth_v1_oracle as O1
        return make_v1_state_dict, lambda sd, cfg, rgb: O1.infer_v1(sd, copy.deepcopy(cfg), rgb)
    import unidepth_oracle as O
    return make_state_dict, lambda sd, cfg, rgb: O.infer_v2(sd, copy.deepcopy(cfg), rgb)


DUMP_BYTES = 63 * 10**6          # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(out, path):
    """Write each output tensor of one infer as <path>/<name>.npy in float32, at most DUMP_BYTES in all.  Smallest first,
    each output gets an equal share of the budget still left; one larger than its share is replaced by a fixed sample of
    its elements (flattened, at indices drawn with seed 0 and sorted), so runs with the same arguments sample the same
    elements."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    left, n = DUMP_BYTES // 4, len(out)
    for name, t in sorted(out.items(), key=lambda kv: kv[1].numel()):
        a = t.detach().float().cpu()
        cap = left // n
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a.numpy())
        left, n = left - a.numel(), n - 1


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1446.4), d.get("bf16_tflops", 1695.9), d.get("hbm_gbs", 6555.5), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.lines = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def pick_cpu_threads(fn):
    """Best of {32, 64, 128} torch threads (capped at the core count) for one call of `fn`; returns (threads, seconds)."""
    best = None
    ncpu = os.cpu_count() or 1
    for t in sorted({min(c, ncpu) for c in (32, 64, 128)}):
        torch.set_num_threads(t)
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best is None or dt < best[1]:
            best = (t, dt)
    torch.set_num_threads(best[0])
    return best


def metric_name(wl):
    if WORKLOADS[wl].get("v1"):
        return "images/sec UniDepthV1.infer ConvNeXt-L 480x640"
    return "images/sec UniDepthV2.infer ViT-L/14 " + ("480x640" if wl == "default" else "1024x1536")


def run_reference(args, rank, world):
    """CPU arm: the oracle port of the reference's infer on the host cores.  Each step is a batch of the workload's
    own batch size when the whole run fits ~4 minutes, else the largest batch that does (stated in `sample`)."""
    if rank != 0:
        return
    make_sd, oracle_infer = oracle_for(args.workload)
    cfg = load_config(args.workload)
    W = WORKLOADS[args.workload]
    sd = make_sd(cfg, 0)
    g = torch.Generator().manual_seed(0)
    H, Wd = W["hw"]
    rgb = torch.randint(0, 256, (W["batch"], 3, H, Wd), dtype=torch.uint8, generator=g)
    oracle_infer(sd, cfg, rgb[:1])                      # page in
    cores, t1 = pick_cpu_threads(lambda: oracle_infer(sd, cfg, rgb[:1]))
    steps = max(1, args.steps)
    n_warm = max(0, min(args.warmup, 1))
    budget_s = 240.0
    b = int(max(1, min(W["batch"], budget_s / (t1 * (steps + n_warm)))))
    x = rgb[:b]
    for _ in range(n_warm):
        oracle_infer(sd, cfg, x)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = oracle_infer(sd, cfg, x)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    val = steps * b / dt
    sample = (f"{steps} steps x batch {b} of the workload's {W['batch']}-image batch, torch fp32, {cores} threads "
              f"(best of 32/64/128) of {os.cpu_count()} cores")
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": n_warm, "ms_per_step": 1000 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": W["desc"], "sample": sample, "same_batch_as_gpu_arm": b == W["batch"]},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_torch_gpu(args, rank, world):
    """INFORMATIVE arm (not the product, not the reference arm): the oracle port executed by stock PyTorch on the GPU
    under fp16 autocast -- cuBLAS / cuDNN / SDPA kernels, i.e. what the reference does on a GPU (unidepthv2.py:239-241).
    Also reports that path's drift against the fp32 CPU forward (the declared fp16 noise floor)."""
    if rank != 0:
        return
    make_sd, oracle_infer = oracle_for(args.workload)
    cfg = load_config(args.workload)
    W = WORKLOADS[args.workload]
    dev = torch.device("cuda", 0)
    sd = make_sd(cfg, 0)
    sd_dev = {k: v.to(dev) for k, v in sd.items()}
    g = torch.Generator().manual_seed(0)
    H, Wd = W["hw"]
    rgb = torch.randint(0, 256, (W["batch"], 3, H, Wd), dtype=torch.uint8, generator=g)
    rgb_dev = rgb.to(dev)

    def step():
        # torch.device(dev): the oracle's constant tensors (mean/std, pixel grids) are created on the GPU too
        with torch.no_grad(), torch.device(dev), torch.autocast("cuda", dtype=torch.float16):
            return oracle_infer(sd_dev, cfg, rgb_dev)

    for _ in range(max(3, args.warmup)):
        out = step()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(args.steps):
        out = step()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e)
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    torch.set_num_threads(min(64, os.cpu_count()))
    ref = oracle_infer(sd, cfg, rgb[:1])
    d, dr = out["depth"][:1].float().cpu(), ref["depth"]
    rel = (d - dr).abs() / dr
    k, kr = out["intrinsics"][:1].float().cpu(), ref["intrinsics"]
    kerr = {n: ((k[:, i, j] - kr[:, i, j]).abs() / kr[:, i, j].abs()).max().item()
            for n, (i, j) in dict(fx=(0, 0), fy=(1, 1), cx=(0, 2), cy=(1, 2)).items()}
    line = {
        "impl": "torch-gpu", "metric": metric_name(args.workload), "value": args.steps * W["batch"] / (ms / 1000.0),
        "unit": "images/s", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "dtype": "fp16 autocast (stock PyTorch kernels)", "data": "synthetic",
        "config": {"workload": W["desc"], "note": "informative: oracle port through stock PyTorch eager on the GPU, "
                   "inputs resident in HBM; not the product path and not the reference arm"},
        "fp16_autocast_drift_vs_fp32_cpu": {"depth_arel": rel.mean().item(), "depth_max_rel": rel.max().item(), "intrinsics_rel": kerr},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-gpu"])
    ap.add_argument("--workload", default="default", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fuse-ln", action="store_true", help="A/B: fold norm1 / norm2 into the qkv / fc1 GEMMs (UniDepthV2.fuse_ln)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                    "(float32; rank 0's images; a fixed seeded sample of an output above its share of 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.impl == "torch-gpu":
        run_torch_gpu(args, rank, world)
        return
    warmup = max(3, args.warmup)
    W = WORKLOADS[args.workload]
    FLOPS_PER_IMAGE = W["flops"]
    H_in, W_in = W["hw"]

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from unidepth_b200 import UniDepthV1, UniDepthV2
    from unidepth_b200 import _cabi
    from unidepth_b200.synthetic import synthetic_state_dict, synthetic_state_dict_v1
    from unidepth_b200.parallel import gather_outputs

    is_v1 = bool(W.get("v1"))
    cfg = load_config(args.workload)
    if is_v1:
        model = UniDepthV1(copy.deepcopy(cfg))
        model.load_state_dict(synthetic_state_dict_v1(cfg, 0, device=dev), strict=True)
        model = model.to(dev).eval()
    else:
        model = UniDepthV2(copy.deepcopy(cfg))
        model.load_state_dict(synthetic_state_dict(cfg, 0, device=dev), strict=True)   # same seed on every rank
        model = model.to(dev).eval()
        model.resolution_level = None
        model.fuse_ln = bool(args.fuse_ln)
    B = args.batch or W["batch"]
    g = torch.Generator().manual_seed(rank)
    rgb_host = torch.randint(0, 256, (B, 3, H_in, W_in), dtype=torch.uint8, generator=g).pin_memory()
    rgb_dev = rgb_host.to(dev)
    import warnings
    warnings.simplefilter("ignore")

    # N > 1: one all-gather of the packed outputs per step (unidepth_b200/parallel.py); `pipelined` gathers are left in
    # flight under the next step's compute (depth-1 pipeline) and every gather is waited for inside the timed region.
    pending = {"dev": None, "e2e": None}
    from unidepth_b200 import parallel
    pipelined = world > 1 and parallel.gather_mode() != "nccl"
    no_gather = os.environ.get("UDB_BENCH_NOGATHER") == "1"     # diagnosis only: N independent replicas, max over ranks

    last_out = {"v": None}

    def infer_into_slot(x):
        # N > 1 with the peer-memory gather: outputs go straight into the send slot (no clone, no pack)
        if world > 1 and pipelined and last_out["v"] is not None:
            model.output_buffers = parallel.output_views(last_out["v"])
        out = model.infer(x)
        last_out["v"] = out
        return out

    def step_device():
        out = infer_into_slot(rgb_dev)
        if no_gather:
            return out
        if world > 1 and pipelined:
            nxt = gather_outputs(out, world, async_op=True)
            if pending["dev"] is not None:
                pending["dev"].wait()
            pending["dev"] = nxt
        elif world > 1:
            out = gather_outputs(out, world)
        return out

    depth_host = torch.empty((B, 1, H_in, W_in), dtype=torch.float32).pin_memory()
    k_host = torch.empty((B, 3, 3), dtype=torch.float32).pin_memory()
    full_host = {}

    def _d2h(out, full=False, local=False):
        lo = rank * B if (world > 1 and not local) else 0
        depth_host.copy_(out["depth"][lo:lo + B], non_blocking=True)
        k_host.copy_(out["intrinsics"][lo:lo + B], non_blocking=True)
        if full:
            for k, v in out.items():
                if k in ("depth", "intrinsics"):
                    continue
                if k not in full_host:
                    full_host[k] = torch.empty((B,) + tuple(v.shape[1:]), dtype=torch.float32).pin_memory()
                full_host[k].copy_(v[lo:lo + B], non_blocking=True)

    def make_e2e(full):
        def step_e2e():
            x = rgb_host.to(dev, non_blocking=True)
            out = infer_into_slot(x)
            if no_gather:
                _d2h(out, full, local=True)
                return out
            if world > 1 and pipelined:
                nxt = gather_outputs(out, world, async_op=True)
                if pending["e2e"] is not None:
                    _d2h(pending["e2e"].wait(), full)
                pending["e2e"] = nxt
            else:
                if world > 1:
                    out = gather_outputs(out, world)
                _d2h(out, full)
            return out
        return step_e2e

    flush_full = [False]

    def flush():
        if pending["dev"] is not None:
            pending["dev"].wait()
            pending["dev"] = None
        if pending["e2e"] is not None:
            _d2h(pending["e2e"].wait(), flush_full[0])
            pending["e2e"] = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        flush()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    l0 = _cabi.launch_count()
    model.use_cuda_graph = False
    step_device()                                   # eager once: counts our launches per forward
    flush()
    torch.cuda.synchronize()
    launches_per_step = _cabi.launch_count() - l0
    model.use_cuda_graph = True
    for _ in range(warmup):
        step_device()
    flush()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(last_out["v"], args.dump_outputs)
    step_e2e = make_e2e(False)
    for _ in range(2):
        step_e2e()
    flush()
    ms_e2e = timed(step_e2e, args.steps)
    step_e2e_full = make_e2e(True)
    flush_full[0] = True
    for _ in range(2):
        step_e2e_full()
    flush()
    ms_e2e_full = timed(step_e2e_full, args.steps)
    flush_full[0] = False
    d2h_full_bytes = (depth_host.numel() + k_host.numel() + sum(t.numel() for t in full_host.values())) * 4

    # per-kernel rooflines: one eager pass through the engine with the library's per-launch profile on (a CUDA event after
    # every kernel on the launching stream, include/udb.h udb_profile_begin / udb_profile_end)
    roof = None
    if rank == 0:
        model.use_cuda_graph = False
        # keep the GPU busy while the host enqueues the whole eager pass (launches + event records),
        # so consecutive events bracket back-to-back kernel executions, not host launch gaps
        torch.cuda._sleep(int(0.15 * 1.9e9))
        stream_ptr = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        prof = _cabi.profile(lambda: model.infer(rgb_dev), stream_ptr, cap=8192)
        torch.cuda.synchronize()
        model.use_cuda_graph = True
        agg = {}
        for name, kms, flops, nbytes in prof:            # the profile's start event fires when the spin kernel ends
            key = "gemm_f16_kernel" if name.startswith("gemm") else name
            a = agg.setdefault(key, [0.0, 0.0, 0, 0.0])
            a[0] += flops
            a[1] += kms
            a[2] += 1
            a[3] += nbytes
        sustained, burst, hbm, how = measured_peaks()
        tot_ms = sum(a[1] for a in agg.values())
        kern = {}
        for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            ent = {"launches": a[2], "ms": round(a[1], 3), "share": round(a[1] / tot_ms, 3)}
            if a[0] > 0 and a[1] > 0:
                ent["tflops"] = round(a[0] / a[1] / 1e9, 1)
                ent["frac_of_sustained_tensor_peak"] = round(a[0] / a[1] / 1e9 / sustained, 3)
            if a[3] > 0 and a[1] > 0 and not k.startswith(("gemm", "attn", "conv3x3_halo")):
                ent["gbs"] = round(a[3] / a[1] / 1e6, 1)           # algorithmic bytes / event time
                ent["frac_of_hbm_peak"] = round(a[3] / a[1] / 1e6 / hbm, 3)
            kern[k] = ent
        gm = agg.get("gemm_f16_kernel", [0.0, 1.0, 1, 0.0])
        ach = gm[0] / gm[1] / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
        if os.path.exists(tpath) and args.workload == "default":
            traffic = json.load(open(tpath)).get("bytes_per_launch_avg")   # ncu capture of the 4 encoder GEMM flavours
        declared = sum(a[0] for a in agg.values())
        roof = {"bound": "tensor", "kernel": "gemm_f16_kernel / gemm2_f16_kernel (linear + conv + convT launches)",
                "achieved": round(ach, 1), "peak": sustained, "unit": "TFLOP/s", "frac": round(ach / sustained, 4),
                "peak_source": f"{how} bf16_tflops_sustained (MEASURED_PEAKS.json)", "traffic": traffic,
                "launches": gm[2], "avg_launch_us": round(1000 * gm[1] / max(gm[2], 1), 2),
                "flops_per_launch_avg": round(gm[0] / max(gm[2], 1) / 1e9, 2),
                "step_tflops": round(B * FLOPS_PER_IMAGE / (ms / args.steps) / 1e9, 1),
                "step_frac": round(B * FLOPS_PER_IMAGE / (ms / args.steps) / 1e9 / sustained, 4),
                "declared_tflop_per_step": round(declared / 1e12, 3),
                "profiled_launches": len(prof), "profiled_ms": round(tot_ms, 3),
                "hbm_peak_gbs": hbm, "kernels": kern}
        at = agg.get("attn_fwd_kernel")
        if at:
            roof["attention"] = {"bound": "tensor", "kernel": "attn_fwd_kernel", "achieved": round(at[0] / at[1] / 1e9, 1),
                                 "peak": sustained, "unit": "TFLOP/s", "frac": round(at[0] / at[1] / 1e9 / sustained, 4),
                                 "launches": at[2], "avg_launch_us": round(1000 * at[1] / at[2], 2)}

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        _, oracle_infer = oracle_for(args.workload)
        sd_cpu = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        one = rgb_host[:1].clone()
        oracle_infer(sd_cpu, cfg, one)
        cores, _ = pick_cpu_threads(lambda: oracle_infer(sd_cpu, cfg, one))
        n = 1 if args.workload == "hires" else 3
        t0 = time.perf_counter()
        for _ in range(n):
            ref = oracle_infer(sd_cpu, cfg, one)
        dt = time.perf_counter() - t0
        got = model.infer(rgb_dev[:1])
        d, dr = got["depth"].cpu(), ref["depth"]
        rel = (d - dr).abs() / dr
        k, kr = got["intrinsics"].cpu(), ref["intrinsics"]
        kerr = {nm: ((k[:, i, j] - kr[:, i, j]).abs() / kr[:, i, j].abs()).max().item()
                for nm, (i, j) in dict(fx=(0, 0), fy=(1, 1), cx=(0, 2), cy=(1, 2)).items()}
        cpu_base = {"value": n / dt, "unit": "images/s", "cores": cores, "kind": "port",
                    "sample": f"{n} x batch-1 infer of the same weights/input (torch fp32 oracle, {cores} threads "
                              f"(best of 32/64/128) of {os.cpu_count()} cores)",
                    "depth_arel_vs_cpu": rel.mean().item(), "depth_max_rel_vs_cpu": rel.max().item(),
                    "intrinsics_rel_vs_cpu": kerr}

    if rank == 0:
        total_images = B * world * args.steps
        line = {
            "metric": metric_name(args.workload), "value": total_images / (ms / 1000.0),
            "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands, f32 accumulate/residual", "data": "synthetic",
            "config": {"workload": W["desc"], "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2": "per-step working set (f16 weights 0.4-0.7 GB + activations > 4 GB) exceeds the 126 MB L2",
                       "fused_layernorm": (not is_v1) and bool(args.fuse_ln),
                       "cuda_graph": True, "engine": ("udb_infer_v1" if is_v1 else "udb_infer_v2") + " (one C call per infer)",
                       **({"collective": "NONE (UDB_BENCH_NOGATHER=1 diagnosis run: independent replicas)" if no_gather
                           else parallel.gather_description()} if world > 1 else {}),
                       **({"peer_memory_unavailable": parallel._p2p_failed[0]} if parallel._p2p_failed[0] else {})},
            "e2e": {"value": total_images / (ms_e2e / 1000.0), "unit": "images/s",
                    "h2d_bytes_per_step": rgb_host.numel(), "d2h_bytes_per_step": depth_host.numel() * 4 + k_host.numel() * 4,
                    "d2h": "depth + intrinsics of this rank's images (the reference returns device tensors; these two are "
                           "what a caller reads back); e2e_full copies the whole output dict"},
            "e2e_full": {"value": total_images / (ms_e2e_full / 1000.0), "unit": "images/s",
                         "h2d_bytes_per_step": rgb_host.numel(), "d2h_bytes_per_step": d2h_full_bytes,
                         "d2h": "every output tensor of this rank's images"},
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu_base,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
