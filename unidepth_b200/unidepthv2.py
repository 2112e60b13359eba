"""UniDepthV2 -- drop-in for the reference's inference API, running on libudb.so (sm_100a).

Mirrors `unidepth.models.UniDepthV2` for the inference path only
(reference: unidepth/models/unidepthv2/unidepthv2.py:111-127 constructor, :239-339 `infer`,
:414-416 `device`, :381-394 `load_pretrained`; HF-hub mixin `from_pretrained`):

    model = UniDepthV2.from_pretrained(dir_with_config_json_and_safetensors)   # or UniDepthV2(config)
    model = model.to("cuda").eval()
    out = model.infer(rgb_uint8)        # dict: confidence intrinsics radius depth points rays depth_features

The module owns `nn.Parameter`s under exactly the reference's state-dict names, so reference
checkpoints (`model.safetensors` / `pytorch_model.bin`) load unchanged.  The forward itself is not
PyTorch: `infer` packs the weights once (f16 GEMM operands, f32 epilogue vectors) and drives the
hand-written kernels through the C ABI (include/udb.h) on torch's current stream, optionally as a
captured CUDA graph.  There is no CPU / eager fallback: a missing library or a CPU-resident model
raises.
"""
from __future__ import annotations

import ctypes as C
import json
import math
import os
import warnings
from collections import OrderedDict
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _cabi as cabi
from . import ops
from .spec import ModelSpec, PATCH, get_paddings, get_resize_factor, param_shapes, pixel_bounds

try:  # same mixin as the reference (unidepthv2.py:111-117)
    from huggingface_hub import PyTorchModelHubMixin
    _HAS_HF = True
except Exception:  # pragma: no cover
    _HAS_HF = False

    class PyTorchModelHubMixin:  # minimal stand-in: local directories only
        def __init_subclass__(cls, **kwargs):
            super().__init_subclass__()

f16, f32 = torch.float16, torch.float32


class _Node(nn.Module):
    """Anonymous container used to reproduce the reference's dotted parameter names."""


def _enc16(w: torch.Tensor, split: bool) -> torch.Tensor:
    """Encoder GEMM weight [N, K]: f16, or in split mode [N, 3K] = [hi | hi | lo] with w ~= hi + lo."""
    w = w.to(f32)
    hi = w.to(f16)
    if not split:
        return hi.contiguous()
    lo = (w - hi.to(f32)).to(f16)
    return torch.cat([hi, hi, lo], dim=1).contiguous()


def _ln_fold(w, b, lnw, lnb):
    """LayerNorm folded into the Linear that follows it:  LN(x) W^T + b = rstd (x W'^T - mean c1) + c2  with
    W' = W diag(ln_w) (f16, what the MMA multiplies), c1 = row sums of the ROUNDED W', c2 = W ln_b + b."""
    w, b, lnw, lnb = w.float(), b.float(), lnw.float(), lnb.float()
    wf = (w * lnw.unsqueeze(0)).to(f16)
    return wf.contiguous(), wf.float().sum(dim=1).contiguous(), (w @ lnb + b).contiguous()


def pack_vit_blocks(sd: dict, pe: str, depth: int, split: bool = False, fuse: bool = False) -> list:
    """Per-block operand dicts of a DINOv2 encoder (state dict `sd`, prefix `pe`), the names the engines' shared block
    (engine_common.h `vit_block`) reads as blocks.<i>.<name>: default f16, split precision or fused LayerNorm."""
    h16 = lambda t: t.to(f16).contiguous()
    c32 = lambda t: t.to(f32).contiguous()
    enc16 = lambda w: _enc16(w, split)
    blocks = []
    for i in range(depth):
        b = f"{pe}blocks.{i}."
        if fuse:
            qw, qc1, qc2 = _ln_fold(sd[b + "attn.qkv.weight"], sd[b + "attn.qkv.bias"], sd[b + "norm1.weight"], sd[b + "norm1.bias"])
            fw, fc1, fc2 = _ln_fold(sd[b + "mlp.fc1.weight"], sd[b + "mlp.fc1.bias"], sd[b + "norm2.weight"], sd[b + "norm2.bias"])
            blocks.append(dict(
                qkv_wf=qw, qkv_c1=qc1, qkv_c2=qc2, fc1_wf=fw, fc1_c1=fc1, fc1_c2=fc2,
                proj_w=h16(sd[b + "attn.proj.weight"]), proj_b=c32(sd[b + "attn.proj.bias"]), ls1=c32(sd[b + "ls1.gamma"]),
                fc2_w=h16(sd[b + "mlp.fc2.weight"]), fc2_b=c32(sd[b + "mlp.fc2.bias"]), ls2=c32(sd[b + "ls2.gamma"])))
            continue
        blocks.append(dict(
            n1w=c32(sd[b + "norm1.weight"]), n1b=c32(sd[b + "norm1.bias"]),
            qkv_w=enc16(sd[b + "attn.qkv.weight"]), qkv_b=c32(sd[b + "attn.qkv.bias"]),
            proj_w=enc16(sd[b + "attn.proj.weight"]), proj_b=c32(sd[b + "attn.proj.bias"]),
            ls1=c32(sd[b + "ls1.gamma"]),
            n2w=c32(sd[b + "norm2.weight"]), n2b=c32(sd[b + "norm2.bias"]),
            fc1_w=enc16(sd[b + "mlp.fc1.weight"]), fc1_b=c32(sd[b + "mlp.fc1.bias"]),
            fc2_w=enc16(sd[b + "mlp.fc2.weight"]), fc2_b=c32(sd[b + "mlp.fc2.bias"]),
            ls2=c32(sd[b + "ls2.gamma"])))
    return blocks


def _register(root: nn.Module, dotted: str, tensor: torch.Tensor):
    parts = dotted.split(".")
    mod = root
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, _Node())
        mod = mod._modules[p]
    mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))


class UniDepthV2(nn.Module, PyTorchModelHubMixin,
                 **(dict(library_name="UniDepth", repo_url="https://github.com/lpiccinelli-eth/UniDepth",
                         tags=["monocular-metric-depth-estimation"]) if _HAS_HF else {})):
    def __init__(self, config: dict, eps: float = 1e-6, **kwargs):
        super().__init__()
        self.config = config
        self.eps = eps
        self.spec = ModelSpec(config)
        s = self.spec
        if not s.use_norm:
            raise NotImplementedError("pixel_encoder.use_norm=false is not used by any shipped UniDepthV2 config")
        for key, shape in param_shapes(config).items():
            _register(self, key, torch.zeros(shape, dtype=f32))
        self.shape_constraints = dict(s.shape_constraints)   # mutable, read by infer (unidepthv2.py:459)
        self.interpolation_mode = "bilinear"                 # unidepthv2.py:460
        self.use_cuda_graph = True
        self.use_engine = True        # False: schedule the same kernels from Python (ops.*; debugging taps / per-kernel timing)
        # "f16": f16 GEMM / attention operands with f32 accumulation (the reference's own GPU dtype, unidepthv2.py:240).
        # "split": parity / debugging mode -- every f16 operand of the ENCODER is a hi + lo pair fed through the same
        # tcgen05 GEMM (three products hi.W_hi + lo.W_hi + hi.W_lo, include/udb.h udb_gemm_t.a_split_k) and attention
        # runs in fp32; ~4x slower.  It shows that the default mode's residual against the fp32 reference is operand
        # rounding: the intrinsics (fp32 camera head on the encoder's cls tokens) then meet north_star's 1e-4.
        self.precision = "f16"
        # optional dict of preallocated output tensors (same keys / shapes as infer's result): graph-mode infer copies its
        # static outputs there instead of cloning them (parallel.PeerGather.views(): the multi-GPU send slot)
        self.output_buffers = None
        # Fused LayerNorm (north_star: "fused LayerNorm + QKV projection"): norm1 / norm2 of the encoder blocks folded into
        # the qkv / fc1 GEMMs (include/udb.h udb_gemm_t.ln_*), no stand-alone LayerNorm pass.  Engine path, f16 mode.
        # OFF by default: measured on the B200 (same box, profiles/r02_fused_ln_ab.txt) it removes 0.89 ms of LayerNorm
        # kernels per 8-image step but adds 1.30 ms to the GEMMs (the producers' extra f16 store + row statistics land in
        # the attn.proj epilogue, which is already longer than its K=1024 main loop): 18.39 vs 18.02 ms/step.
        self.fuse_ln = False
        self._engine = None
        self._engine_key = None
        # Bounded caches (LRU): the reference handles arbitrary shapes in constant memory, so a stream of
        # differently-sized images must not grow device memory without limit.  A captured graph keeps its own
        # reference to the workspace it was captured with, so evicting a workspace never frees memory a live
        # graph still replays into.
        self.max_cached_graphs = 8
        self.max_cached_workspaces = 8
        self.max_engine_shapes = 64       # per-(gh,gw) tables live inside the engine; beyond this everything is rebuilt
        self._workspaces: "OrderedDict[tuple, torch.Tensor]" = OrderedDict()
        self._packed: Optional[dict] = None
        self._packed_key = None
        self._graphs: "OrderedDict[tuple, dict]" = OrderedDict()
        self._posembed_cache: Dict[tuple, torch.Tensor] = {}
        self._scales_cache: Dict[tuple, torch.Tensor] = {}      # ray-embedding frequency tables: shape constants, never dropped
        self._engine_shapes: set = set()

    # ------------------------------------------------------------------ reference-compatible API
    @property
    def device(self):
        return next(self.parameters()).device

    def load_pretrained(self, model_file: str):
        """unidepthv2.py:381-394: torch checkpoint, optional 'model' key, strip 'module.'."""
        sd = torch.load(model_file, map_location="cpu", weights_only=False)
        if "model" in sd:
            sd = sd["model"]
        sd = {k.replace("module.", ""): v for k, v in sd.items()}
        info = self.load_state_dict(sd, strict=False)
        print(f"Loaded from {model_file} for {self.__class__.__name__} results in:", info)

    if not _HAS_HF:
        @classmethod
        def from_pretrained(cls, path: str, **kwargs):
            config = json.load(open(os.path.join(path, "config.json")))
            model = cls(config=config.get("config", config))
            st = os.path.join(path, "model.safetensors")
            if os.path.exists(st):
                from safetensors.torch import load_file
                model.load_state_dict(load_file(st), strict=False)
            else:
                model.load_state_dict(torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu"),
                                      strict=False)
            return model

    # ------------------------------------------------------------------ weight packing
    def _fuse(self) -> bool:
        return bool(self.fuse_ln and self.use_engine and self.precision == "f16")

    def _fingerprint(self):
        return (self.precision, self._fuse()) + tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _pack(self):
        """One-time (per weight version) repack into kernel operand layouts."""
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("unidepth_b200.UniDepthV2.infer needs the model on a CUDA device "
                               "(model.to('cuda')); there is no CPU fallback")
        torch.cuda.set_device(dev)      # callers hold `with torch.cuda.device(self.device)`
        self._packed = self._pack_tensors(dev)
        self._packed_key = self._fingerprint()
        self._drop_engine()

    def _pack_tensors(self, dev) -> dict:
        """The packed operands as tensors on `dev` (plain torch layout work, no kernel involved).  `_pack` is the only
        product caller (CUDA device); tests/test_engine_schedule_cpu.py runs it on the CPU to check, through the engine's
        dry run, that every packing mode registers exactly the operands the C schedule asks for."""
        s = self.spec
        if s.kernel_size != 3:
            raise NotImplementedError(f"pixel_decoder.kernel_size={s.kernel_size}: the residual conv units run as 3x3 "
                                      "convolutions (every shipped UniDepthV2 config sets 3)")
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        h16 = lambda t: t.to(f16).contiguous()
        c32 = lambda t: t.to(f32).contiguous()
        if self.precision not in ("f16", "split"):
            raise ValueError(f"precision must be 'f16' or 'split', not {self.precision!r}")
        split = self.precision == "split"

        fuse = self._fuse()
        P: dict = {"split": split, "fuse_ln": fuse}
        d, hid = s.embed_dim, s.hidden
        # The attention kernel works on 64-wide heads.  Narrower decoder heads (ViT-S: 256/8 = 32) are
        # zero-padded to 64 in the packed q / kv / out weights: padded q,k columns add 0 to q.k, padded
        # v columns produce zeros that meet zero columns of the out projection; the softmax scale stays
        # 1/sqrt(true head dim).
        hd = hid // s.dec_heads
        if d // s.enc_heads != 64 or hd > 64:
            raise NotImplementedError(f"head dims (encoder {d // s.enc_heads}, decoder {hd}) not supported")
        for cch in list(s.cur) + list(s.outd[:-1]):
            if cch % 64:
                raise NotImplementedError(f"decoder channel count {cch} is not a multiple of 64")
        # The last stage's output map (ViT-B: 96 channels) and the "lr" convs' outputs (48 / 32) are
        # zero-padded to multiples of 64 channels: zero weight rows produce zero channels, which meet
        # zero weight columns downstream; LayerNorm statistics use the real count (dim_valid).
        pad64 = lambda c: (c + 63) // 64 * 64
        c_hr_real, c_hr = s.outd[-1], pad64(s.outd[-1])
        if c_hr_real % 8 or c_hr > 256:
            raise NotImplementedError(f"high-resolution feature width {c_hr_real} not supported")
        P["dec_hd"], P["dec_hp"] = hd, s.dec_heads * 64
        pe = "pixel_encoder."
        wpe = torch.zeros((d, 640), device=dev, dtype=f32)
        wpe[:, :588] = sd[pe + "patch_embed.proj.weight"].reshape(d, 588).to(f32)
        P["patch_w"], P["patch_b"] = _enc16(wpe, split), c32(sd[pe + "patch_embed.proj.bias"])
        P["cls"] = c32(sd[pe + "cls_token"].reshape(d))
        P["pos"] = c32(sd[pe + "pos_embed"].reshape(-1, d))
        P["blocks"] = pack_vit_blocks(sd, pe, s.depth, split, fuse)
        P["norm_w"], P["norm_b"] = c32(sd[pe + "norm.weight"]), c32(sd[pe + "norm.bias"])

        pd = "pixel_decoder."
        P["adapt"] = [(h16(sd[f"{pd}input_adapter.input_adapters.{i}.weight"]),
                       c32(sd[f"{pd}input_adapter.input_adapters.{i}.bias"])) for i in range(4)]
        P["cam_adapt"] = [(c32(sd[f"{pd}camera_token_adapter.input_adapters.{i}.weight"]),
                           c32(sd[f"{pd}camera_token_adapter.input_adapters.{i}.bias"])) for i in range(4)]
        cl = pd + "camera_layer."

        def mlp32(prefix):
            return dict(nw=c32(sd[prefix + ".norm.weight"]), nb=c32(sd[prefix + ".norm.bias"]),
                        w1=c32(sd[prefix + ".proj1.weight"]), b1=c32(sd[prefix + ".proj1.bias"]),
                        w2=c32(sd[prefix + ".proj2.weight"]), b2=c32(sd[prefix + ".proj2.bias"]))

        def agg32(prefix):
            return dict(mlp=mlp32(prefix + ".mlp"), kv=c32(sd[prefix + ".kv.weight"]), q=c32(sd[prefix + ".q.weight"]),
                        nxw=c32(sd[prefix + ".norm_attnx.weight"]), nxb=c32(sd[prefix + ".norm_attnx.bias"]),
                        ncw=c32(sd[prefix + ".norm_attnctx.weight"]), ncb=c32(sd[prefix + ".norm_attnctx.bias"]),
                        out=c32(sd[prefix + ".out.weight"]), ls1=c32(sd[prefix + ".ls1.gamma"]),
                        ls2=c32(sd[prefix + ".ls2.gamma"]))

        P["cam"] = dict(pos=c32(sd[cl + "latents_pos"].reshape(4, hid)), agg1=agg32(cl + "aggregate1"),
                        agg2=agg32(cl + "aggregate2"), project=mlp32(cl + "project"),
                        pinhole=mlp32(cl + "out_pinhole"))
        dl = pd + "depth_layer."
        nh_dec = s.dec_heads

        def pad_heads_rows(w):      # [heads*hd, K] -> [heads*64, K], zero rows for the padded head dims
            if hd == 64:
                return w
            out_w = torch.zeros((nh_dec, 64, w.shape[1]), device=w.device, dtype=w.dtype)
            out_w[:, :hd] = w.reshape(nh_dec, hd, w.shape[1])
            return out_w.reshape(nh_dec * 64, w.shape[1])

        def pad_heads_cols(w):      # [N, heads*hd] -> [N, heads*64]
            if hd == 64:
                return w
            out_w = torch.zeros((w.shape[0], nh_dec, 64), device=w.device, dtype=w.dtype)
            out_w[:, :, :hd] = w.reshape(w.shape[0], nh_dec, hd)
            return out_w.reshape(w.shape[0], nh_dec * 64)

        P["prompt"] = []
        for i in range(4):
            p = f"{dl}prompt_camera.{i}.layers.0"
            P["prompt"].append(dict(
                nxw=c32(sd[p + ".norm_attnx.weight"]), nxb=c32(sd[p + ".norm_attnx.bias"]),
                ncw=c32(sd[p + ".norm_attnctx.weight"]), ncb=c32(sd[p + ".norm_attnctx.bias"]),
                q=h16(pad_heads_rows(sd[p + ".q.weight"])),
                kv=h16(torch.cat([pad_heads_rows(sd[p + ".kv.weight"][:hid]), pad_heads_rows(sd[p + ".kv.weight"][hid:])], 0)),
                out=h16(pad_heads_cols(sd[p + ".out.weight"])),
                mnw=c32(sd[p + ".mlp.norm.weight"]), mnb=c32(sd[p + ".mlp.norm.bias"]),
                w1=h16(sd[p + ".mlp.proj1.weight"]), b1=c32(sd[p + ".mlp.proj1.bias"]),
                w2=h16(sd[p + ".mlp.proj2.weight"]), b2=c32(sd[p + ".mlp.proj2.bias"])))
        P["lat_w"], P["lat_b"] = h16(sd[dl + "to_latents.weight"]), c32(sd[dl + "to_latents.bias"])
        conv_pack = lambda w: h16(w.permute(0, 2, 3, 1).reshape(w.shape[0], -1))   # [Cout,(dy,dx,ci)]
        P["ups"] = []
        for i in range(len(s.dec_depths)):
            k = max(1, 2 * i)
            wt = sd[f"{dl}process_features.{i}.weight"]                            # [Cin,Cout,k,k]
            cout = wt.shape[1]
            st = dict(k=k, cout=cout,
                      ct_w=h16(wt.permute(2, 3, 1, 0).reshape(k * k * cout, wt.shape[0])),
                      ct_b=c32(sd[f"{dl}process_features.{i}.bias"].repeat(k * k)), rcus=[])
            for j in range(s.dec_depths[i]):
                u = f"{dl}ups.{i}.convs.{j}."
                st["rcus"].append(dict(w1=conv_pack(sd[u + "conv1.weight"]), b1=c32(sd[u + "conv1.bias"]),
                                       w2=conv_pack(sd[u + "conv2.weight"]), b2=c32(sd[u + "conv2.bias"]),
                                       gamma=c32(sd[u + "gamma"].reshape(-1))))
            uw = sd[f"{dl}ups.{i}.up.0.weight"]
            uw, ub = uw.reshape(uw.shape[0], uw.shape[1]).float(), sd[f"{dl}ups.{i}.up.0.bias"].float()
            if uw.shape[0] % 64:            # last stage of ViT-B: 96 -> 128 output channels (zeros)
                extra = pad64(uw.shape[0]) - uw.shape[0]
                uw = torch.cat([uw, torch.zeros((extra, uw.shape[1]), device=dev)], 0)
                ub = torch.cat([ub, torch.zeros(extra, device=dev)], 0)
            st["up_w"], st["up_b"] = h16(uw), c32(ub)
            P["ups"].append(st)
        last = len(s.dec_depths) - 1
        # heads: LN(x) = xhat * w + b with the SAME xhat for depth and confidence, so the two
        # LN -> Linear pairs fold into one GEMM on xhat with W' = W * w (per input channel) and
        # b' = W b + bias, depth rows first then confidence rows (decoder.py:190-199, 288, 306-307)
        P["heads"] = []
        wm, bm = [], []
        zpad = lambda t, dim, n: t if t.shape[dim] == n else torch.cat(
            [t, torch.zeros(tuple(n - t.shape[dim] if i == dim else sz for i, sz in enumerate(t.shape)), device=dev)], dim)
        for mlp_p, lr, hr, add in ((f"{dl}depth_mlp.{last}", "to_depth_lr", "to_depth_hr", 2.0),
                                   (f"{dl}confidence_mlp", "to_confidence_lr", "to_confidence_hr", 0.0)):
            lnw, lnb = sd[mlp_p + ".0.weight"].float(), sd[mlp_p + ".0.bias"].float()
            w, bb = sd[mlp_p + ".1.weight"].float(), sd[mlp_p + ".1.bias"].float()
            # [c_hr, c_hr] block of the merged GEMM: real rows / columns first, zero padding after
            wm.append(zpad(zpad(w * lnw.unsqueeze(0), 1, c_hr), 0, c_hr))
            bm.append(zpad(w @ lnb + bb, 0, c_hr))
            lr_w, lr_b, hr_w = sd[f"{dl}{lr}.weight"].float(), sd[f"{dl}{lr}.bias"].float(), sd[f"{dl}{hr}.0.weight"].float()
            lr_c = pad64(lr_w.shape[0])       # ViT-S: 32 -> 64, ViT-B: 48 -> 64 output channels of the lr conv
            lr_w = zpad(zpad(lr_w, 1, c_hr), 0, lr_c)
            lr_b = zpad(lr_b, 0, lr_c)
            hr_w = zpad(hr_w, 1, lr_c)
            P["heads"].append(dict(
                lr_w=conv_pack(lr_w), lr_b=c32(lr_b),
                hr_w=conv_pack(hr_w), hr_b=c32(sd[f"{dl}{hr}.0.bias"]),
                head_w=c32(sd[f"{dl}{hr}.2.weight"].reshape(32)), head_b=float(sd[f"{dl}{hr}.2.bias"].item()),
                add=add))
        P["head_mlp_w"], P["head_mlp_b"] = h16(torch.cat(wm, 0)), c32(torch.cat(bm, 0))
        P["c_hr_valid"] = c_hr_real
        ones = torch.zeros(c_hr, device=dev, dtype=f32)
        ones[:c_hr_real] = 1.0               # padded channels: weight 0 -> normalised value 0
        P["ln_ones"] = ones
        P["ln_zeros"] = torch.zeros(c_hr, device=dev, dtype=f32)
        return P

    # ------------------------------------------------------------------ C engine (udb_create / udb_infer_v2)
    def _drop_engine(self):
        """Destroy the engine AND everything that holds raw pointers into it: captured graphs replay kernels whose
        arguments point at the engine's per-shape tables and at the workspaces, so they go first."""
        self._graphs.clear()
        self._posembed_cache.clear()
        if self._engine is not None:
            dev = getattr(self, "_engine_device", None)
            if dev is not None:
                torch.cuda.synchronize(dev)       # nothing may still be running out of the tables we free
            cabi.lib().udb_destroy(self._engine)
        self._engine, self._engine_key = None, None
        self._workspaces.clear()
        self._engine_shapes = set()

    def __del__(self):
        try:
            self._drop_engine()
        except Exception:
            pass

    @staticmethod
    def _flatten_packed(P: dict):
        """Packed-weight dict -> ({engine tensor name: tensor}, {scalar name: float}) (names: include/udb.h,
        DESIGN.md 'packed tensors')."""
        T, S = {}, {}
        for k in ("patch_w", "patch_b", "cls", "pos", "norm_w", "norm_b", "lat_w", "lat_b", "head_mlp_w", "head_mlp_b",
                  "ln_ones", "ln_zeros"):
            T[k] = P[k]
        S["precision"] = 1.0 if P.get("split") else 0.0
        S["fuse_ln"] = 1.0 if P.get("fuse_ln") else 0.0
        for i, blk in enumerate(P["blocks"]):
            for k, v in blk.items():
                T[f"blocks.{i}.{k}"] = v
        for l in range(4):
            T[f"adapt.{l}.w"], T[f"adapt.{l}.b"] = P["adapt"][l]
            T[f"cam_adapt.{l}.w"], T[f"cam_adapt.{l}.b"] = P["cam_adapt"][l]
            for k, v in P["prompt"][l].items():
                T[f"prompt.{l}.{k}"] = v
        cam = P["cam"]
        T["cam.pos"] = cam["pos"]
        for name in ("project", "pinhole"):
            for k, v in cam[name].items():
                T[f"cam.{name}.{k}"] = v
        for name in ("agg1", "agg2"):
            for k, v in cam[name].items():
                if k == "mlp":
                    for k2, v2 in v.items():
                        T[f"cam.{name}.mlp.{k2}"] = v2
                else:
                    T[f"cam.{name}.{k}"] = v
        for i, st in enumerate(P["ups"]):
            for k in ("ct_w", "ct_b", "up_w", "up_b"):
                T[f"ups.{i}.{k}"] = st[k]
            for j, r in enumerate(st["rcus"]):
                for k, v in r.items():
                    T[f"ups.{i}.rcu.{j}.{k}"] = v
        for i, hd in enumerate(P["heads"]):
            for k in ("lr_w", "lr_b", "hr_w", "hr_b", "head_w"):
                T[f"heads.{i}.{k}"] = hd[k]
            S[f"heads.{i}.head_b"] = hd["head_b"]
            S[f"heads.{i}.add"] = hd["add"]
        return T, S

    def _engine_config(self, P: dict) -> "cabi.Config":
        """udb_config_t of this model (include/udb.h)."""
        s, sc = self.spec, self.shape_constraints
        cfg = cabi.Config()
        cfg.embed_dim, cfg.depth, cfg.enc_heads = s.embed_dim, s.depth, s.enc_heads
        for i, t in enumerate(s.taps):
            cfg.taps[i] = t
        cfg.pos_grid = int(math.isqrt(P["pos"].shape[0] - 1))
        cfg.hidden, cfg.dec_heads, cfg.expansion, cfg.out_dim = s.hidden, s.dec_heads, s.expansion, s.out_dim
        cfg.n_stages = len(s.dec_depths)
        for i, dd in enumerate(s.dec_depths):
            cfg.dec_depths[i] = dd
        cfg.ratio_min, cfg.ratio_max = sc["ratio_bounds"]
        cfg.pixels_min, cfg.pixels_max = sc["pixels_min"], sc["pixels_max"]
        return cfg

    @staticmethod
    def _register(handle, tensors: dict, scalars: dict):
        """udb_set_weight / udb_set_scalar for every packed operand (the engine borrows the pointers)."""
        for name, t in tensors.items():
            assert t.is_contiguous() and t.dtype in (f16, f32), name
            shape = (C.c_int64 * max(t.ndim, 1))(*t.shape)
            cabi.check(cabi.lib().udb_set_weight(handle, name.encode(), C.c_void_p(t.data_ptr()), shape, t.ndim,
                                                 cabi.DT_F32 if t.dtype == f32 else cabi.DT_F16), f"udb_set_weight({name})")
        for name, v in scalars.items():
            cabi.check(cabi.lib().udb_set_scalar(handle, name.encode(), float(v)), f"udb_set_scalar({name})")

    def _get_engine(self):
        P = self._weights()
        sc = self.shape_constraints
        key = (tuple(sc["ratio_bounds"]), sc["pixels_min"], sc["pixels_max"])
        if self._engine is not None and self._engine_key == key:
            return self._engine
        self._drop_engine()
        handle = C.c_void_p()
        cabi.check(cabi.lib().udb_create(C.byref(self._engine_config(P)), C.byref(handle)), "udb_create")
        tensors, scalars = self._flatten_packed(P)
        for name, t in tensors.items():
            assert t.is_cuda, name
        self._register(handle, tensors, scalars)
        self._engine, self._engine_key = handle, key
        self._engine_device = self.device
        self._engine_tensors = tensors          # the engine borrows these pointers
        return handle

    def _forward_engine(self, rgb: torch.Tensor, geom: dict, normalize: bool, level, camera_k=None, rays_in=None):
        """The whole path as ONE C call (udb_infer_v2): torch only allocates outputs / workspace."""
        eng = self._get_engine()
        lib = cabi.lib()
        dev = rgb.device
        B, _, H, W = rgb.shape
        lvl = -1 if level is None else int(level)      # -2: network-only (identity geometry)
        g = cabi.Geometry()
        cabi.check(lib.udb_geometry(eng, H, W, lvl, C.byref(g)), "udb_geometry")
        assert (g.net_h, g.net_w) == tuple(geom["net_hw"]) and (g.pad_l, g.pad_r, g.pad_t, g.pad_b) == tuple(geom["paddings"])
        wkey = (B, H, W, lvl)
        ws = self._workspaces.get(wkey)
        if ws is None:
            nbytes = lib.udb_workspace_bytes(eng, B, H, W, lvl)
            if nbytes == 0:
                raise RuntimeError(f"udb_workspace_bytes failed: {lib.udb_last_error().decode()}")
            ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            self._workspaces[wkey] = ws
            self._engine_shapes.add((g.gh, g.gw))
            while len(self._workspaces) > self.max_cached_workspaces:
                self._workspaces.popitem(last=False)
        else:
            self._workspaces.move_to_end(wkey)
        self._last_ws = ws
        hid = self.spec.hidden
        E = lambda *shape: torch.empty(shape, device=dev, dtype=f32)
        out = {"confidence": E(B, 1, H, W), "intrinsics": E(B, 3, 3), "radius": E(B, 1, H, W), "depth": E(B, 1, H, W),
               "points": E(B, 3, H, W), "rays": E(B, 3, H, W)}
        feats = E(B, g.gh, g.gw, hid)
        a = cabi.InferArgs()
        a.rgb, a.rgb_is_u8, a.normalize = rgb.data_ptr(), int(rgb.dtype == torch.uint8), int(normalize)
        a.B, a.H, a.W, a.resolution_level = B, H, W, lvl
        a.camera_k = camera_k.data_ptr() if camera_k is not None else None
        a.camera_rays = rays_in.data_ptr() if rays_in is not None else None
        a.ray_scales = geom["scales"].data_ptr()
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        for k, v in out.items():
            setattr(a, k, v.data_ptr())
        a.depth_features = feats.data_ptr()
        cabi.check(lib.udb_infer_v2(eng, C.byref(a), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "udb_infer_v2")
        out["depth_features"] = feats.permute(0, 3, 1, 2)
        return out

    def _weights(self):
        if self._packed is None or self._packed_key != self._fingerprint():
            self._pack()
        return self._packed

    def _pos_embed(self, gh: int, gw: int) -> torch.Tensor:
        """[1+gh*gw, D] f32: row 0 = cls position, rest = bicubic-resized grid (cached per shape)."""
        key = (gh, gw)
        if key not in self._posembed_cache:
            P = self._weights()
            pos = P["pos"]
            m = int(math.isqrt(pos.shape[0] - 1))
            d = pos.shape[1]
            if (gh, gw) == (m, m):
                full = pos.clone()
            else:
                grid = ops.posembed_bicubic(pos[1:].contiguous(), m, d, gh, gw)
                full = torch.cat([pos[:1], grid], dim=0).contiguous()
            self._posembed_cache[key] = full
        return self._posembed_cache[key]

    # ------------------------------------------------------------------ the forward (kernel launches only)
    def _forward(self, rgb: torch.Tensor, geom: dict, normalize: bool, gt_intr4=None, taps: Optional[dict] = None,
                 rays_in=None):
        P = self._weights()
        s = self.spec
        dev = rgb.device
        B = rgb.shape[0]
        nh, nw = geom["net_hw"]
        gh, gw = nh // PATCH, nw // PATCH
        N, T, D, hid = gh * gw, gh * gw + 1, s.embed_dim, s.hidden
        E = lambda *shape, dtype=f16: torch.empty(shape, device=dev, dtype=dtype)

        # a2/a3/a4: preprocess + patch embed + cls/pos
        patches = E(B * N, 640)
        ops.preprocess_patchify(rgb, geom["paddings"], (nh, nw), patches, normalize)
        pos = self._pos_embed(gh, gw)
        x = E(B * T, D, dtype=f32)
        ops.gemm(patches, P["patch_w"], bias=P["patch_b"], resid=pos, out=x, rows_per_group=N, group_stride=T,
                 row_offset=1, resid_mod=N, resid_row_offset=1)
        ops.set_cls_rows(x, P["cls"], pos, B, T, D)
        if taps is not None:
            taps["tokens0"] = x.clone().view(B, T, D)

        # a5-a8: transformer blocks
        h = E(B * T, D)
        qkv = E(B * T, 3 * D)
        att = E(B * T, D)
        mid = E(B * T, 4 * D)
        feats, clss = [], []
        for i, blk in enumerate(P["blocks"]):
            ops.layernorm(x, blk["n1w"], blk["n1b"], 1e-6, out=h)
            ops.gemm(h, blk["qkv_w"], bias=blk["qkv_b"], out=qkv)
            ops.attention(qkv, qkv, qkv, att, B=B, heads=s.enc_heads, seq_q=T, seq_k=T, head_dim=64,
                          q_col0=0, k_col0=D, v_col0=2 * D)
            ops.gemm(att, blk["proj_w"], bias=blk["proj_b"], gamma=blk["ls1"], resid=x, out=x)
            ops.layernorm(x, blk["n2w"], blk["n2b"], 1e-6, out=h)
            ops.gemm(h, blk["fc1_w"], bias=blk["fc1_b"], act=ops.ACT_GELU, out=mid)
            ops.gemm(mid, blk["fc2_w"], bias=blk["fc2_b"], gamma=blk["ls2"], resid=x, out=x)
            if taps is not None and i == 0:
                taps["block0"] = x.clone().view(B, T, D)
            if (i + 1) in s.taps:
                feats.append(ops.layernorm(x, P["norm_w"], P["norm_b"], 1e-5, out=E(B * N, D), rows=B * N,
                                           rows_per_group=N, group_stride=T, row_offset=1))
                clss.append(ops.layernorm(x, P["norm_w"], P["norm_b"], 1e-5, out=E(B, D, dtype=f32), rows=B,
                                          rows_per_group=1, group_stride=T, row_offset=0))
        if taps is not None:
            taps["feat3"] = feats[-1].clone().view(B, gh, gw, D)
            taps["cls3"] = clss[-1].clone().view(B, 1, D)

        # a9: adapters
        F = [ops.gemm(feats[l], P["adapt"][l][0], bias=P["adapt"][l][1], out_dtype=f32) for l in range(4)]
        tokens = E(B, 4, hid, dtype=f32)
        tok2 = tokens.view(B, 4 * hid)
        for l in range(4):
            ops.small_linear(clss[l], P["cam_adapt"][l][0], P["cam_adapt"][l][1], out=tok2[:, l * hid:(l + 1) * hid])

        # a10: camera head (fp32)
        cam = P["cam"]
        t = tokens.view(B * 4, hid)

        def mlp32(x_in, m, resid=None, gamma=None):
            y = ops.layernorm(x_in, m["nw"], m["nb"], 1e-5, out_dtype=f32)
            y = ops.small_linear(y, m["w1"], m["b1"], act=ops.ACT_GELU)
            return ops.small_linear(y, m["w2"], m["b2"], gamma=gamma, resid=resid)

        t = mlp32(t, cam["project"])
        for agg in (cam["agg1"], cam["agg2"]):
            xn = ops.layernorm(t, agg["nxw"], agg["nxb"], 1e-5, out_dtype=f32)
            cn = ops.layernorm(t, agg["ncw"], agg["ncb"], 1e-5, out_dtype=f32)
            q = ops.small_linear(xn, agg["q"])
            kv = ops.small_linear(cn, agg["kv"])
            a4 = ops.camera_attn4(q, kv, cam["pos"], B, hid, s.dec_heads)
            t = ops.small_linear(a4, agg["out"], gamma=agg["ls1"], resid=t)
            t = mlp32(t, agg["mlp"], resid=t, gamma=agg["ls2"])
        x4 = mlp32(t, cam["pinhole"])                       # [B*4, 1] == [B,4]
        intr4, k_net, k_out = ops.camera_intrinsics(x4, B, (nh, nw), geom["factor"], geom["paddings"][0],
                                                    geom["paddings"][2])

        # a11/a12: ray embedding
        scales = geom["scales"]
        # GT-camera branch (unidepthv2.py:299-303,361-362; decoder.py:400): rays come from the given
        # pinhole K instead of the predicted one; the returned intrinsics stay the predicted ones.
        ray_intr = intr4 if gt_intr4 is None else gt_intr4
        remb = ops.ray_embed(ray_intr, scales, B, (nh, nw), (gh, gw), out_dtype=f32, rays_in=rays_in)
        if taps is not None:
            taps["ray_embedding"] = remb.clone().view(B, N, hid)
            taps["intrinsics4"] = intr4.clone()

        # a13: prompt blocks
        cond = []
        xn, cn = E(B * N, hid), E(B * N, hid)
        hp = P["dec_hp"]                               # heads * 64 (heads zero-padded to 64 dims)
        qb, kvb, ab = E(B * N, hp), E(B * N, 2 * hp), E(B * N, hp)
        mb = E(B * N, s.expansion * hid)
        for l in range(4):
            pr = P["prompt"][l]
            ops.layernorm(F[l], pr["nxw"], pr["nxb"], 1e-5, out=xn)
            ops.layernorm(remb, pr["ncw"], pr["ncb"], 1e-5, out=cn)
            ops.gemm(xn, pr["q"], out=qb)
            ops.gemm(cn, pr["kv"], out=kvb)
            ops.attention(qb, kvb, kvb, ab, B=B, heads=s.dec_heads, seq_q=N, seq_k=N, head_dim=64, k_col0=0, v_col0=hp,
                          scale=P["dec_hd"] ** -0.5)
            ops.gemm(ab, pr["out"], resid=F[l], out=F[l])
            ops.layernorm(F[l], pr["mnw"], pr["mnb"], 1e-5, out=xn)
            ops.gemm(xn, pr["w1"], bias=pr["b1"], act=ops.ACT_GELU, out=mb)
            if taps is not None and l == 0:
                c32_ = ops.gemm(mb, pr["w2"], bias=pr["b2"], resid=F[l], out_dtype=f32)
                taps["cond0"] = c32_.view(B, N, hid)
            cond.append(ops.gemm(mb, pr["w2"], bias=pr["b2"], resid=F[l], out=E(B * N, hid)))

        # a14/a15: latents + up-sampling stages
        init_latents = ops.gemm(cond[0], P["lat_w"], bias=P["lat_b"], out_dtype=f32)      # [B*N, hid] == NHWC
        cur_h, cur_w = gh, gw
        prev = init_latents.view(B, gh, gw, hid)
        for i, st in enumerate(P["ups"]):
            k, cout = st["k"], st["cout"]
            oh, ow = cur_h, cur_w                      # spatial size of this stage (prev already at it)
            lat = E(B, oh, ow, cout, dtype=f32)
            act = E(B, oh, ow, cout)
            ops.conv_transpose_ks(cond[i + 1], st["ct_w"], k, cout, (gh, gw), bias=st["ct_b"], resid=prev, out=lat,
                                  out2=act, out2_leaky=True)
            n_rcu = len(st["rcus"])
            tmp = E(B, oh, ow, cout)
            for j, r in enumerate(st["rcus"]):
                ops.conv3x3(act, r["w1"], bias=r["b1"], act=ops.ACT_LEAKY, out=tmp)
                ops.conv3x3(tmp, r["w2"], bias=r["b2"], gamma=r["gamma"], resid=lat, out=lat, out2=act,
                            out2_leaky=(j + 1 < n_rcu))
            up_c = st["up_w"].shape[0]
            u = ops.gemm(act.view(B * oh * ow, cout), st["up_w"], bias=st["up_b"], out=E(B * oh * ow, up_c))
            prev = ops.upsample2x(u.view(B, oh, ow, up_c))
            cur_h, cur_w = 2 * oh, 2 * ow
            if taps is not None:
                taps[f"ups{i}"] = prev.clone()
        feat_hr = prev                                  # [B, 8gh, 8gw, C] f16
        C_hr = feat_hr.shape[-1]
        hh, hw = feat_hr.shape[1], feat_hr.shape[2]

        # a16/a17: depth + confidence heads (shared normalisation, merged LN->Linear GEMM written
        # straight into the reflect-padded buffer the 3x3 "lr" convs read)
        xhat = ops.layernorm(feat_hr, P["ln_ones"], P["ln_zeros"], 1e-5, out=E(B * hh * hw, C_hr),
                             dim_valid=P["c_hr_valid"] if P["c_hr_valid"] != C_hr else 0)
        n_mlp = P["head_mlp_w"].shape[0]                      # 2 * out_dim: [depth | confidence]
        mp = E(B, hh + 2, hw + 2, n_mlp)
        ops.conv_transpose_ks(xhat, P["head_mlp_w"], 1, n_mlp, (hh, hw), bias=P["head_mlp_b"], out=mp, pad=1)
        ops.reflect_border_fill(mp)
        planes = []
        for i, hd in enumerate(P["heads"]):
            # small-Cout convs: halo-reuse kernel (input tile loaded once for the nine taps)
            lr = ops.conv3x3_halo(mp, hd["lr_w"], bias=hd["lr_b"], c_off=i * (n_mlp // 2), c_used=n_mlp // 2)
            up = ops.resize_ac_pad(lr, nh, nw, 1)
            planes.append(ops.conv3x3_halo(up, hd["hr_w"], bias=hd["hr_b"], act=ops.ACT_LEAKY,
                                           head_w=hd["head_w"], head_b=hd["head_b"], head_add=hd["add"]))
        radius, confidence = planes
        if taps is not None:
            taps["radius_net"] = radius.clone()

        # a18: output assembly
        pl, pr_, pt, pb = geom["paddings"]
        out = ops.postprocess(radius, confidence, ray_intr, B, (nh, nw), geom["padded_hw"], pl, pt, geom["out_hw"],
                              rays_in=rays_in)
        out["intrinsics"] = k_out
        out["depth_features"] = init_latents.view(B, gh, gw, hid).permute(0, 3, 1, 2)
        return out

    @staticmethod
    def _gt_intrinsics(camera, B, paddings, factor, dev):
        """`camera=` argument of infer: a (...,3,3) pinhole K (unidepthv2.py:267-279).  The reference
        wraps it in Pinhole/BatchCamera, shifts the principal point by the paddings (`crop`,
        utils/camera.py:115-120) and scales by the resize factor (`resize`, :78-81); rays are then
        K^-1 [u,v,1] at pixel centres (Pinhole.unproject :252-263).  Here the adjusted
        (fx,fy,cx,cy) is handed to the ray kernels, which evaluate the same expression."""
        assert camera.shape[-1] == 3 and camera.shape[-2] == 3, \
            "camera tensor should be of shape (..., 3, 3): assume pinhole"
        K = camera.to(dev, f32).reshape(-1, 3, 3)
        if K.shape[0] not in (1, B):
            raise ValueError(f"camera holds {K.shape[0]} intrinsics for a batch of {B} images (need 1 or {B})")
        if K.shape[0] == 1 and B > 1:
            K = K.expand(B, 3, 3)
        if float(K[:, 0, 1].abs().max()) != 0.0:
            raise NotImplementedError("pinhole K with skew is not supported")
        pl, _, pt, _ = paddings
        return torch.stack([K[:, 0, 0] * factor, K[:, 1, 1] * factor, (K[:, 0, 2] + pl) * factor,
                            (K[:, 1, 2] + pt) * factor], dim=1).contiguous()

    # ------------------------------------------------------------------ infer
    @staticmethod
    def _camera_rays(camera, B, paddings, factor, net_hw, dev):
        """`camera=` given as a camera OBJECT (the reference's `Camera` / `BatchCamera` family,
        utils/camera.py, or anything with the same three methods): the reference crops it by the
        paddings, resizes it by the factor and asks it for unit rays at network-input resolution
        (unidepthv2.py:299-303, :361-362); those rays replace the predicted ones (decoder.py:400).
        The object's own host/torch code generates the rays; they enter the kernels as a
        [B, net_h*net_w, 3] f32 tensor.  The caller's object is not mutated (the reference does)."""
        import copy
        for name in ("crop", "resize", "get_rays"):
            if not callable(getattr(camera, name, None)):
                raise TypeError(f"camera must be a (...,3,3) tensor or an object with crop/resize/get_rays (missing {name})")
        cam = copy.deepcopy(camera)
        if callable(getattr(cam, "to", None)):
            cam = cam.to(dev)
        pl, pr_, pt, pb = paddings
        cam = cam.crop(left=-pl, top=-pt, right=-pr_, bottom=-pb)
        cam = cam.resize(factor)
        nh, nw = net_hw
        rays = cam.get_rays(shapes=(B, nh, nw))
        if rays.ndim == 3:
            rays = rays.unsqueeze(0)
        assert rays.shape[-3:] == (3, nh, nw), f"camera.get_rays returned {tuple(rays.shape)}"
        if rays.shape[0] not in (1, B):
            raise ValueError(f"camera.get_rays returned {rays.shape[0]} ray maps for a batch of {B} images")
        if rays.shape[0] == 1 and B > 1:
            rays = rays.expand(B, 3, nh, nw)
        return rays.to(dev, f32).permute(0, 2, 3, 1).reshape(B, nh * nw, 3).contiguous()

    @torch.no_grad()
    def infer(self, rgb: torch.Tensor, camera=None, normalize: bool = True):
        """Same contract as the reference `UniDepthV2.infer` (unidepthv2.py:239-339)."""
        if self.interpolation_mode != "bilinear":
            raise NotImplementedError("interpolation_mode other than 'bilinear' is not implemented")
        level = getattr(self, "resolution_level", None)
        if level is None:
            warnings.warn("!! self.resolution_level not set, using default bounds !!")
        bounds = pixel_bounds(self.shape_constraints, level)
        if rgb.ndim == 3:
            rgb = rgb.unsqueeze(0)
        B, _, H, W = rgb.shape
        rgb = self._to_device_input(rgb)
        paddings, (ph, pw) = get_paddings((H, W), self.shape_constraints["ratio_bounds"])
        factor, (nh, nw) = get_resize_factor((ph, pw), bounds)
        geom = dict(paddings=paddings, padded_hw=(ph, pw), factor=factor, net_hw=(nh, nw), out_hw=(H, W))
        key = (level, tuple(self.shape_constraints["ratio_bounds"]), bounds)
        return self._run(rgb, geom, level, normalize, camera, key)

    NETWORK_ONLY = -2      # udb.h: UDB_LEVEL_NETWORK_ONLY

    @torch.no_grad()
    def network_forward(self, rgbs: torch.Tensor, rays: Optional[torch.Tensor] = None):
        """The network alone, as the reference's ONNX wrappers expose it (unidepthv2/export.py:27-45 `forward(rgbs)`
        and :58-79 `forward(rgbs, rays)`): `rgbs` is the NORMALISED float network input [B,3,H,W] with H, W
        multiples of 14; no padding / resizing / cropping.  Returns (pts_3d [B,3,H,W], confidence [B,1,H,W],
        intrinsics [B,3,3])."""
        out = self._network_outputs(rgbs, rays)
        return out["points"], out["confidence"], out["intrinsics"]

    def _network_outputs(self, rgbs, rays=None):
        assert rgbs.ndim == 4 and rgbs.shape[1] == 3, "rgbs must be [B,3,H,W]"
        B, _, H, W = rgbs.shape
        if H % PATCH or W % PATCH:
            raise ValueError(f"network input {H}x{W} must be a multiple of {PATCH}")
        rgbs = self._to_device_input(rgbs.float())
        geom = dict(paddings=(0, 0, 0, 0), padded_hw=(H, W), factor=1.0, net_hw=(H, W), out_hw=(H, W))
        rays_in = None
        if rays is not None:
            assert tuple(rays.shape) == (B, 3, H, W), "rays must be [B,3,H,W] at the network resolution"
            rays_in = rays.to(rgbs.device, f32).permute(0, 2, 3, 1).reshape(B, H * W, 3).contiguous()
        return self._run(rgbs, geom, self.NETWORK_ONLY, False, None, ("network_only",), rays_in=rays_in)

    @torch.no_grad()
    def forward_test(self, inputs: dict, image_metas=None):
        """Validation forward of the reference (unidepthv2.py:134-160): `inputs["image"]` is the data
        pipeline's normalised network input, `inputs["depth"]` the ground truth whose size the predictions
        are matched to, `inputs["paddings"]` the per-image (l, r, t, b) paddings of the network input,
        optional `inputs["camera"]` a camera object for GT rays (:361-362)."""
        from .validation import match_gt, match_intrinsics
        image = inputs["image"]
        rays = None
        cam = inputs.get("camera", None)
        if cam is not None:
            B, _, H, W = image.shape
            rays = cam.get_rays(shapes=(B, H, W))
        out = self._network_outputs(image, rays)
        gt, pads = inputs["depth"], inputs.get("paddings", None)
        res = {k: match_gt(out[k], gt, padding1=pads, padding2=None) for k in ("depth", "points", "confidence")}
        res["rays"] = out["rays"] / torch.norm(out["rays"], dim=1, keepdim=True).clip(min=1e-5)
        res["intrinsics"] = match_intrinsics(out["intrinsics"], image, gt, padding1=pads, padding2=None)
        return res

    def forward(self, inputs=None, image_metas=None, *args, **kwargs):
        """Evaluation-mode `forward` of the reference dispatches to `forward_test` (unidepthv2.py:162-166);
        training is out of scope."""
        if self.training or not isinstance(inputs, dict):
            raise NotImplementedError("training forward is out of scope; use .infer() / .forward_test() in eval mode")
        return self.forward_test(inputs, image_metas)

    def _to_device_input(self, rgb):
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("unidepth_b200 has no CPU path: move the model to a CUDA device")
        rgb = rgb.to(dev)
        if rgb.dtype not in (torch.uint8, f32):
            rgb = rgb.float()
        return rgb.contiguous()

    def _run(self, rgb, geom, level, normalize, camera, key_extra, rays_in=None):
        """Common tail of infer / network_forward: camera handling, engine or Python schedule, CUDA graph cache.
        Everything runs with the model's device current (streams, cudaMalloc of the engine tables, the per-device
        kernel attributes on the C side), so a model on cuda:1 works while cuda:0 is the process default."""
        with torch.cuda.device(self.device):
            return self._run_on_device(rgb, geom, level, normalize, camera, key_extra, rays_in)

    def _run_on_device(self, rgb, geom, level, normalize, camera, key_extra, rays_in=None):
        B, _, H, W = rgb.shape
        dev = rgb.device
        nh, nw = geom["net_hw"]
        gh, gw = nh // PATCH, nw // PATCH
        bands = self.spec.hidden // 2
        # Weights first: packing drops the engine and every cache that depends on it.  (Round-1/2 bug: the frequency table
        # below used to live in _posembed_cache and be created BEFORE this call; the first infer then packed, cleared the
        # cache, captured the graph with the table's pointer and let the tensor die with `geom` -- later allocations reused
        # its memory and replays of that first graph computed the ray embedding from garbage.  It surfaced only when the
        # freed block happened to be reused, e.g. by the peer-memory gather's output tensors.)
        self._weights()
        skey = (gh, gw, bands, dev.index)
        if skey not in self._scales_cache:
            # positional_embedding.py:231-233 -- computed with the same torch expression (host, once per grid)
            self._scales_cache[skey] = (2.0 ** torch.linspace(0.0, math.log2(max(gh, gw) // 2), steps=bands)).to(dev)
        geom["scales"] = self._scales_cache[skey]

        gt_intr4, camera_k = None, None
        if camera is not None and not isinstance(camera, torch.Tensor):
            rays_in = self._camera_rays(camera, B, geom["paddings"], geom["factor"], (nh, nw), dev)
        elif camera is not None:
            gt_intr4 = self._gt_intrinsics(camera, B, geom["paddings"], geom["factor"], dev)     # validates the argument
            camera_k = camera.to(dev, f32).reshape(-1, 3, 3)
            if camera_k.shape[0] == 1 and B > 1:
                camera_k = camera_k.expand(B, 3, 3)
            camera_k = camera_k.contiguous()

        self._weights()
        if len(self._engine_shapes) > self.max_engine_shapes:
            self._drop_engine()       # too many distinct grids seen: rebuild (frees the engine's per-shape tables)

        def run(inp):
            if not self.use_engine and self.precision != "f16":
                raise NotImplementedError("precision='split' runs through the C engine only (use_engine=True)")
            if self.use_engine:
                return self._forward_engine(inp, geom, normalize, level, camera_k=camera_k, rays_in=rays_in)
            self._pos_embed(gh, gw)
            return self._forward(inp, geom, normalize, gt_intr4=gt_intr4, rays_in=rays_in)

        if not self.use_cuda_graph or camera is not None or rays_in is not None:
            return run(rgb)

        key = (B, H, W, rgb.dtype, bool(normalize), bool(self.use_engine)) + tuple(key_extra)
        entry = self._graphs.get(key)
        if entry is None:
            static_in = rgb.clone()
            # warm-up on a side stream (allocator, per-shape tables, workspace), then capture
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                run(static_in)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = run(static_in)
            # the entry owns everything whose address the captured kernels read
            entry = dict(graph=graph, inp=static_in, out=static_out, ws=getattr(self, "_last_ws", None), scales=geom["scales"])
            self._graphs[key] = entry
            while len(self._graphs) > self.max_cached_graphs:
                self._graphs.popitem(last=False)
        else:
            self._graphs.move_to_end(key)
        if os.environ.get("UDB_SKIP_INPUT_COPY") != "1":      # (experiment switch: isolates copy-engine contention)
            entry["inp"].copy_(rgb, non_blocking=True)
        entry["graph"].replay()
        bufs = self.output_buffers
        if bufs is not None:       # caller-provided destinations (e.g. the send slot of parallel.PeerGather): one copy, no clone
            for k, v in entry["out"].items():
                bufs[k].copy_(v)
            return {k: bufs[k] for k in entry["out"]}
        return {k: v.clone() for k, v in entry["out"].items()}
