"""UniDepthV1 with the DINOv2 ViT-L/14 encoder on one GPU: the same workload as `bench.py --workload v1` (16 x 3x480x640
uint8 per step, network input 462x616 fixed), so the two V1 encoders compare directly.  Prints one JSON line:

  value / ms_per_step   CUDA-graph replays, input resident in HBM
  e2e                   host input -> H2D -> infer -> D2H of depth + intrinsics
  roofline              one eager pass under the library's per-launch profile (udb_profile_begin / end): GEMM and
                        attention TF/s from the flops the kernels declare, every kernel's time and share, the ViT tap kernel
  torch_gpu             the fp32 oracle run by stock PyTorch under fp16 autocast on the same GPU (what bench.py
                        --impl torch-gpu does for the other workloads), its images/s and its drift against the fp32 CPU oracle
  drift_vs_cpu          this path's drift against the same fp32 CPU oracle (image 0)
  gpu                   name, power limit and max SM clock, read in the same run

    python tools/bench_v1_vitl.py --steps 20 --warmup 3 [--out profiles/<name>.json]
FLOPs per image come from shapes (encoder_flops / decoder_flops below), not from a measurement."""
import argparse
import copy
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
sys.dont_write_bytecode = True

import torch  # noqa: E402

from bench import ClockSampler, measured_peaks  # noqa: E402

BATCH, HW, NET = 16, (480, 640), (462, 616)


def encoder_flops(gh=33, gw=44, d=1024, depth=24):
    """Multiply-adds x 2 of the DINOv2 encoder from its shapes: per block qkv + proj + fc1 + fc2 GEMMs (12 d^2 per token)
    and attention (QK^T and PV: 4 T^2 d), plus the 588-wide patch embedding."""
    n = gh * gw
    t = n + 1
    gemm = depth * 2 * t * 12 * d * d
    attn = depth * 4 * t * t * d
    patch = 2 * n * 588 * d
    return dict(gemm=gemm, attention=attn, patch_embed=patch, total=gemm + attn + patch)


def decoder_flops(gh=33, gw=44, d=1024, hid=512, depths=(3, 2, 1)):
    """The V1 decoder's GEMM-shaped work from its shapes (adapters, camera context, rays, depth head with dense and
    Nystrom attention, ConvUpsample); the small fp32 camera-head pieces are left out (< 0.1 GF)."""
    n = gh * gw
    f = 0
    f += 2 * 2 * 4 * n * d * hid                          # input adapters (tokens + channel copy)
    f += 2 * 4 * n * (hid * 2 * hid * 2) + 2 * (4 * n + 4) * hid * 2 * hid   # camera in_features MLP + kv
    for s in range(3):                                    # ray MLPs 128 -> 384 -> C
        r = n * 4 ** s
        f += 2 * r * (128 * 384 + 384 * (hid >> s))
    f += 2 * n * 4 * hid * hid + 2 * n * (hid * 2 * hid * 2)   # features_channel_cat + to_latents
    for nk in (4 * n, n):                                 # aggregate_16 / prompt_camera: dense single head
        f += 2 * n * hid * hid * 2 + 2 * nk * hid * hid * 2 + 2 * 2 * n * nk * hid + 2 * n * (hid * 4 * hid * 2)
    blk = lambda r, c: 2 * r * (c * c * 4) + 2 * r * (c * 4 * c * 2)   # q, kv, out + MLP
    f += depths[0] * (blk(n, hid) + 4 * n * n * hid)
    for s, dep in ((1, depths[1]), (2, depths[2])):
        r, c = n * 4 ** s, hid >> s
        f += dep * (blk(r, c) + 2 * 2 * 2 * r * 128 * c)   # Nystrom: two r x 128 attentions
    for s in range(3):                                    # ConvUpsample: 2 ConvNeXt blocks, 1x1, 3x3
        r, c = n * 4 ** s, hid >> s
        f += 2 * (2 * r * c * 4 * c * 2 + 2 * r * 49 * c) + 2 * r * c * c // 2 + 2 * 4 * r * 9 * (c // 2) ** 2
    return f


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, plim, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": plim, "clocks_max_sm": clk, "torch_name": torch.cuda.get_device_name(0)}


def drift(out, ref):
    d, dr = out["depth"][:1].float().cpu(), ref["depth"]
    rel = (d - dr).abs() / dr
    k, kr = out["intrinsics"][:1].float().cpu(), ref["intrinsics"]
    kerr = max(((k[:, i, j] - kr[:, i, j]).abs() / kr[:, i, j].abs()).max().item() for i, j in ((0, 0), (1, 1), (0, 2), (1, 2)))
    return {"depth_arel": rel.mean().item(), "depth_max_rel": rel.max().item(), "intrinsics_rel": kerr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_v1_vitl.py needs a CUDA device")
    import unidepth_v1_vit_oracle as OV
    from unidepth_b200 import UniDepthV1, _cabi
    dev = torch.device("cuda", 0)
    cfg = json.load(open(os.path.join(ROOT, "unidepth_b200", "configs", "config_v1_vitl14.json")))
    sd = OV.make_v1_vit_state_dict(cfg, 0)
    model = UniDepthV1(copy.deepcopy(cfg))
    model.load_state_dict(sd, strict=True)
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(0)
    rgb_host = torch.randint(0, 256, (BATCH, 3, *HW), dtype=torch.uint8, generator=g).pin_memory()
    rgb_dev = rgb_host.to(dev)
    info = gpu_info()

    def timed(fn, steps):
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e)

    l0 = _cabi.launch_count()
    model.use_cuda_graph = False
    model.infer(rgb_dev)
    torch.cuda.synchronize()
    launches = _cabi.launch_count() - l0
    model.use_cuda_graph = True
    for _ in range(max(3, args.warmup)):
        out = model.infer(rgb_dev)
    sampler = ClockSampler(0)
    sampler.start()
    ms = timed(lambda: model.infer(rgb_dev), args.steps)
    clocks = sampler.stop()
    depth_host = torch.empty((BATCH, 1, *HW), dtype=torch.float32).pin_memory()
    k_host = torch.empty((BATCH, 3, 3), dtype=torch.float32).pin_memory()

    def e2e():
        o = model.infer(rgb_host.to(dev, non_blocking=True))
        depth_host.copy_(o["depth"], non_blocking=True)
        k_host.copy_(o["intrinsics"], non_blocking=True)

    for _ in range(2):
        e2e()
    ms_e2e = timed(e2e, args.steps)

    # per-launch profile of one eager pass (GPU kept busy while the host enqueues, as bench.py does)
    model.use_cuda_graph = False
    torch.cuda._sleep(int(0.3 * 1.9e9))
    prof = _cabi.profile(lambda: model.infer(rgb_dev), C.c_void_p(torch.cuda.current_stream().cuda_stream), cap=16384)
    torch.cuda.synchronize()
    model.use_cuda_graph = True
    agg = {}
    for name, kms, flops, nbytes in prof:
        key = "gemm_f16_kernel" if name.startswith("gemm") else name
        a = agg.setdefault(key, [0.0, 0.0, 0, 0.0])
        a[0] += flops
        a[1] += kms
        a[2] += 1
        a[3] += nbytes
    tot = sum(a[1] for a in agg.values())
    sustained, _, hbm, how = measured_peaks()
    kern = {}
    for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        ent = {"launches": a[2], "ms": round(a[1], 3), "share": round(a[1] / tot, 4)}
        if a[0] > 0 and a[1] > 0:
            ent["tflops"] = round(a[0] / a[1] / 1e9, 1)
        kern[k] = ent
    tap_bytes = BATCH * (24 * (33 * 44 * 1024 * (4 + 2)) + 19 * 33 * 44 * 1024 * 2)   # f32 rows read, f16 written, f16 max read
    tap = agg.get("vit_tap_kernel", [0, 0.0, 0, 0])
    enc, dec = encoder_flops(), decoder_flops()
    per_img = enc["total"] + dec

    # stock PyTorch arm: the oracle on the GPU under fp16 autocast, and both paths' drift against the fp32 CPU oracle
    sd_dev = {k: v.to(dev) for k, v in sd.items()}

    def torch_step():
        with torch.no_grad(), torch.device(dev), torch.autocast("cuda", dtype=torch.float16):
            return OV.infer_v1_vit(sd_dev, cfg, rgb_dev)

    for _ in range(3):
        tout = torch_step()
    tsteps = max(3, args.steps // 4)
    ms_torch = timed(torch_step, tsteps)
    torch.set_num_threads(min(64, os.cpu_count()))
    ref = OV.infer_v1_vit(sd, cfg, rgb_host[:1].clone())
    ours = model.infer(rgb_dev[:1])

    line = {
        "metric": "unidepth_v1_vitl14_images_per_s", "value": args.steps * BATCH / (ms / 1000.0), "unit": "images/s",
        "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
        "config": {"model": "UniDepthV1 ViT-L/14 (config_v1_vitl14.json)", "batch": BATCH, "input": "3x480x640 uint8",
                   "net_input": "462x616 (fixed), 33x44 patches", "cuda_graph": True, "engine": "udb_infer_v1",
                   "weights": "seeded fixture (oracle/unidepth_v1_vit_oracle.py, seed 0)"},
        "gpu": info, "clocks": clocks, "gpu_launches_per_step": launches,
        "e2e": {"value": args.steps * BATCH / (ms_e2e / 1000.0), "unit": "images/s",
                "h2d_bytes_per_step": rgb_host.numel(), "d2h_bytes_per_step": (depth_host.numel() + k_host.numel()) * 4},
        "flops_per_image_from_shapes": {"encoder": enc, "decoder": dec, "total": per_img},
        "step_tflops": round(BATCH * per_img / (ms / args.steps) / 1e9, 1),
        "roofline": {"profiled_ms": round(tot, 3), "profiled_launches": len(prof), "peak_source": how,
                     "sustained_tensor_tflops": sustained, "hbm_gbs": hbm,
                     "gemm_tflops": kern.get("gemm_f16_kernel", {}).get("tflops"),
                     "attention_tflops": kern.get("attn_fwd_kernel", {}).get("tflops"),
                     "tap": {"kernel": "vit_tap_kernel", "launches": tap[2], "ms": round(tap[1], 3),
                             "share": round(tap[1] / tot, 4) if tot else None,
                             "gbs": round(tap_bytes / tap[1] / 1e6, 1) if tap[1] else None},
                     "kernels": kern},
        "torch_gpu": {"value": tsteps * BATCH / (ms_torch / 1000.0), "unit": "images/s",
                      "dtype": "fp16 autocast, stock PyTorch kernels (oracle port, inputs resident in HBM)",
                      "drift_vs_fp32_cpu": drift(tout, ref)},
        "drift_vs_cpu": drift(ours, ref),
    }
    line["speedup_vs_torch_gpu"] = round(line["value"] / line["torch_gpu"]["value"], 3)
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
