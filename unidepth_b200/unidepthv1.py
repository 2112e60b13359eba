"""UniDepthV1 (ConvNeXt or DINOv2 ViT encoder) -- drop-in for the reference's inference API, running on libudb.so (sm_100a).

Mirrors `unidepth.models.UniDepthV1` for the inference path only (reference:
unidepth/models/unidepthv1/unidepthv1.py:96-110 constructor, :288-373 `infer`, :375-392 `load_pretrained`,
:418-420 `device`; HF-hub mixin `from_pretrained`):

    model = UniDepthV1.from_pretrained(dir_with_config_json_and_safetensors)    # or UniDepthV1(config)
    model = model.to("cuda").eval()
    out = model.infer(rgb_uint8, intrinsics=None, skip_camera=False)             # dict: intrinsics points depth

The module owns `nn.Parameter`s under exactly the reference's state-dict names (unidepth_b200/spec_v1.py), so reference
checkpoints load unchanged.  `infer` packs the weights once and makes ONE C call (`udb_infer_v1`, include/udb.h) that
enqueues the hand-written kernels on torch's current stream, optionally captured as a CUDA graph.  No CPU / eager fallback.

The 1/8 and 1/4 decoder levels use Nystrom attention (reference: xformers NystromAttention, absent here); this
implementation follows the published algorithm as restated in oracle/unidepth_v1_oracle.py -- parity for that one
function is unpinned (see DESIGN.md).
"""
from __future__ import annotations

import ctypes as C
import json
import math
import os
from collections import OrderedDict
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi as cabi
from .spec_v1 import V1Spec, level_grid, param_shapes, v1_paddings, v1_shapes
from .unidepthv2 import PyTorchModelHubMixin, _HAS_HF, _register, pack_vit_blocks

f16, f32 = torch.float16, torch.float32


def _sine_position_embedding(h: int, w: int, num_pos_feats: int, device) -> torch.Tensor:
    """PositionEmbeddingSine(num_pos_feats, normalize=True) of an all-valid h x w grid -> [h*w, 2*num_pos_feats]
    (layers/positional_encoding.py:15-59: y features then x features, sin on even / cos on odd feature indices).
    Evaluated once per weight version on the host side (a constant of the shape)."""
    eps, scale = 1e-6, 2 * math.pi
    y = torch.arange(1, h + 1, dtype=f32, device=device)[:, None].expand(h, w) / (h + eps) * scale
    x = torch.arange(1, w + 1, dtype=f32, device=device)[None, :].expand(h, w) / (w + eps) * scale
    dim_t = torch.arange(num_pos_feats, dtype=f32, device=device)
    dim_t = 10000.0 ** (2 * torch.div(dim_t, 2, rounding_mode="floor") / num_pos_feats)
    px, py = x[..., None] / dim_t, y[..., None] / dim_t
    px = torch.stack((px[..., 0::2].sin(), px[..., 1::2].cos()), dim=3).flatten(2)
    py = torch.stack((py[..., 0::2].sin(), py[..., 1::2].cos()), dim=3).flatten(2)
    return torch.cat((py, px), dim=2).reshape(h * w, 2 * num_pos_feats)


class UniDepthV1(nn.Module, PyTorchModelHubMixin,
                 **(dict(library_name="UniDepth", repo_url="https://github.com/lpiccinelli-eth/UniDepth",
                         tags=["monocular-metric-depth-estimation"]) if _HAS_HF else {})):
    def __init__(self, config: dict, eps: float = 1e-6, **kwargs):
        super().__init__()
        self.config = config
        self.eps = eps
        self.spec = V1Spec(config)
        for key, shape in param_shapes(config).items():
            _register(self, key, torch.zeros(shape, dtype=f32))
        self.image_shape = list(self.spec.image_shape)        # unidepthv1.py:447
        self.use_cuda_graph = True
        self.max_cached_graphs = 8
        self.output_buffers = None      # see UniDepthV2.output_buffers
        self._engine = None
        self._packed: Optional[dict] = None
        self._packed_key = None
        self._graphs: "OrderedDict[tuple, dict]" = OrderedDict()
        self._workspaces: "OrderedDict[tuple, torch.Tensor]" = OrderedDict()

    # ------------------------------------------------------------------ reference-compatible API
    @property
    def device(self):
        return next(self.parameters()).device

    def load_pretrained(self, model_file: str):
        """unidepthv1.py:375-392."""
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
                model.load_state_dict(torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu"), strict=False)
            return model

    # ------------------------------------------------------------------ weight packing
    def _fingerprint(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _pack(self):
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("unidepth_b200.UniDepthV1.infer needs the model on a CUDA device (model.to('cuda')); "
                               "there is no CPU fallback")
        torch.cuda.set_device(dev)
        T, S = self._pack_tensors(dev)
        self._packed = dict(T=T, S=S)
        self._packed_key = self._fingerprint()
        self._drop_engine()

    def _pack_tensors(self, dev):
        """({engine tensor name: tensor on `dev`}, {scalar name: float}): plain torch layout work.  `_pack` is the only
        product caller (CUDA device); tests/test_engine_schedule_cpu.py runs it on the CPU to check, through the engine's
        dry run, that the packer registers exactly the operands the C schedule asks for."""
        s = self.spec
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        h16 = lambda t: t.to(f16).contiguous()
        c32 = lambda t: t.to(f32).contiguous()
        T: Dict[str, torch.Tensor] = {}
        S: Dict[str, float] = {}
        pe, pd = "pixel_encoder.", "pixel_decoder."
        hid = s.hidden

        def zpad(t, rows, cols):
            out = torch.zeros((rows, cols), device=dev, dtype=f32)
            out[:t.shape[0], :t.shape[1]] = t
            return out

        def zpad1(t, n):
            out = torch.zeros(n, device=dev, dtype=f32)
            out[:t.shape[0]] = t
            return out

        def block(dst, src, conv_names):
            """ConvNeXt block operands: depthwise weights tap-major [49, C] f32, MLP weights f16."""
            dw, norm, fc1, fc2 = conv_names
            w = sd[f"{src}{dw}.weight"]
            T[dst + "dw_w"] = c32(w.reshape(w.shape[0], 49).t())
            T[dst + "dw_b"] = c32(sd[f"{src}{dw}.bias"])
            T[dst + "ln_w"], T[dst + "ln_b"] = c32(sd[f"{src}{norm}.weight"]), c32(sd[f"{src}{norm}.bias"])
            T[dst + "w1"], T[dst + "b1"] = h16(sd[f"{src}{fc1}.weight"]), c32(sd[f"{src}{fc1}.bias"])
            T[dst + "w2"], T[dst + "b2"] = h16(sd[f"{src}{fc2}.weight"]), c32(sd[f"{src}{fc2}.bias"])
            T[dst + "gamma"] = c32(sd[f"{src}gamma"])

        # ---- encoder
        hc, wc = level_grid(s)
        if s.vit:
            d = s.embed_dim
            T["patch_w"] = h16(zpad(sd[pe + "patch_embed.proj.weight"].reshape(d, 588).float(), d, 640))
            T["patch_b"], T["cls"] = c32(sd[pe + "patch_embed.proj.bias"]), c32(sd[pe + "cls_token"].reshape(d))
            # dinov2.py:267-304 with interpolate_offset 0.1 (unidepthv1.py:418-424): the bicubic resampling of the 37x37
            # table takes its sample positions from the scale factor; the network shape is fixed, so the resampled table
            # is a constant of the weights, folded here with the reference's own call
            pos = sd[pe + "pos_embed"].float()
            m = math.isqrt(pos.shape[1] - 1)
            grid = F.interpolate(pos[:, 1:].reshape(1, m, m, d).permute(0, 3, 1, 2), mode="bicubic", antialias=False,
                                 scale_factor=((hc + 0.1) / m, (wc + 0.1) / m))
            assert tuple(grid.shape[-2:]) == (hc, wc), grid.shape
            T["pos"] = c32(torch.cat([pos[0, :1], grid.permute(0, 2, 3, 1).reshape(hc * wc, d)], 0))
            for i, blk in enumerate(pack_vit_blocks(sd, pe, s.enc_depth)):
                for k, v in blk.items():
                    T[f"blocks.{i}.{k}"] = v
        else:
            T["stem_w"] = h16(zpad(sd[pe + "stem.0.weight"].reshape(s.dims[0], 48), s.dims[0], 64))
            T["stem_b"] = c32(sd[pe + "stem.0.bias"])
            T["stem_ln_w"], T["stem_ln_b"] = c32(sd[pe + "stem.1.weight"]), c32(sd[pe + "stem.1.bias"])
            for i, depth in enumerate(s.depths):
                st = f"{pe}stages.{i}."
                if i > 0:
                    w = sd[st + "downsample.1.weight"]                               # [C, Cp, 2, 2] -> [C, (dy,dx,ci)]
                    T[f"ds{i}.ln_w"], T[f"ds{i}.ln_b"] = c32(sd[st + "downsample.0.weight"]), c32(sd[st + "downsample.0.bias"])
                    T[f"ds{i}.w"], T[f"ds{i}.b"] = h16(w.permute(0, 2, 3, 1).reshape(w.shape[0], -1)), c32(sd[st + "downsample.1.bias"])
                for j in range(depth):
                    block(f"s{i}.b{j}.", f"{st}blocks.{j}.", ("conv_dw", "norm", "mlp.fc1", "mlp.fc2"))

        # ---- decoder: adapters, embeddings
        for l in range(4):
            a = f"{pd}input_adapter.input_adapters.{l}"
            T[f"adapt.{l}.ln_w"], T[f"adapt.{l}.ln_b"] = c32(sd[a + ".0.weight"]), c32(sd[a + ".0.bias"])
            T[f"adapt.{l}.w"], T[f"adapt.{l}.b"] = h16(sd[a + ".1.weight"]), c32(sd[a + ".1.bias"])
            t = f"{pd}token_adapter.input_adapters.{l}"
            T[f"tok.{l}.ln_w"], T[f"tok.{l}.ln_b"] = c32(sd[t + ".0.weight"]), c32(sd[t + ".0.bias"])
            T[f"tok.{l}.w"], T[f"tok.{l}.b"] = c32(sd[t + ".1.weight"]), c32(sd[t + ".1.bias"])
        # level embedding MLP of the four learned level vectors + sine position embedding of the common grid
        # (decoder.py:410-433): constants of (weights, network shape), folded once here
        le = F.linear(F.gelu(F.linear(sd[pd + "level_embeds"].float(), sd[pd + "level_embed_layer.0.weight"].float(),
                                      sd[pd + "level_embed_layer.0.bias"].float())),
                      sd[pd + "level_embed_layer.2.weight"].float(), sd[pd + "level_embed_layer.2.bias"].float())
        le = F.layer_norm(le, (hid,), sd[pd + "level_embed_layer.3.weight"].float(), sd[pd + "level_embed_layer.3.bias"].float(), 1e-5)
        pos = _sine_position_embedding(hc, wc, hid // 2, dev)
        T["tokens_pos"] = c32((pos[None, :, :] + le[:, None, :]).reshape(4 * hc * wc, hid))

        def mlp32(dst, src):
            T[dst + ".nw"], T[dst + ".nb"] = c32(sd[src + ".norm.weight"]), c32(sd[src + ".norm.bias"])
            T[dst + ".w1"], T[dst + ".b1"] = c32(sd[src + ".proj1.weight"]), c32(sd[src + ".proj1.bias"])
            T[dst + ".w2"], T[dst + ".b2"] = c32(sd[src + ".proj2.weight"]), c32(sd[src + ".proj2.bias"])

        cl = pd + "camera_layer."
        T["cam.cls.nw"], T["cam.cls.nb"] = c32(sd[cl + "cls_project.0.weight"]), c32(sd[cl + "cls_project.0.bias"])
        T["cam.cls.w1"], T["cam.cls.b1"] = c32(sd[cl + "cls_project.1.weight"]), c32(sd[cl + "cls_project.1.bias"])
        T["cam.cls.w2"], T["cam.cls.b2"] = c32(sd[cl + "cls_project.3.weight"]), c32(sd[cl + "cls_project.3.bias"])
        T["cam.inf.nw"], T["cam.inf.nb"] = c32(sd[cl + "in_features.norm.weight"]), c32(sd[cl + "in_features.norm.bias"])
        T["cam.inf.w1"], T["cam.inf.b1"] = h16(sd[cl + "in_features.proj1.weight"]), c32(sd[cl + "in_features.proj1.bias"])
        T["cam.inf.w2"], T["cam.inf.b2"] = h16(sd[cl + "in_features.proj2.weight"]), c32(sd[cl + "in_features.proj2.bias"])
        T["cam.pos"] = c32(sd[cl + "latents_pos"].reshape(4, hid))

        def cam_block(dst, src, kv_half):
            for a, b in (("nxw", "norm_attnx.weight"), ("nxb", "norm_attnx.bias"), ("ncw", "norm_attnctx.weight"),
                         ("ncb", "norm_attnctx.bias"), ("q_w", "q.weight"), ("q_b", "q.bias"), ("kv_b", "kv.bias"),
                         ("out_w", "out.weight"), ("out_b", "out.bias"), ("ls1", "ls1.gamma"), ("ls2", "ls2.gamma")):
                T[dst + a] = c32(sd[src + b])
            T[dst + "kv_w"] = h16(sd[src + "kv.weight"]) if kv_half else c32(sd[src + "kv.weight"])
            mlp32(dst + "mlp", src + "mlp")

        cam_block("cam.agg.", cl + "aggregate.", True)
        for i in range(2):
            cam_block(f"cam.l{i}.", f"{cl}layers.{i}.", False)
        mlp32("cam.out", cl + "out")

        dl = pd + "depth_layer."
        for name, outd in (("16", hid), ("8", hid // 2), ("4", hid // 4)):
            src = f"{dl}project_rays{name}"
            T[f"rays.{name}.ln_w"], T[f"rays.{name}.ln_b"] = zpad1(sd[src + ".norm.weight"].float(), 84), zpad1(sd[src + ".norm.bias"].float(), 84)
            T[f"rays.{name}.w1"] = h16(zpad(sd[src + ".proj1.weight"].float(), 384, 128))       # [324, 81] zero-extended
            T[f"rays.{name}.b1"] = zpad1(sd[src + ".proj1.bias"].float(), 384)
            T[f"rays.{name}.w2"] = h16(zpad(sd[src + ".proj2.weight"].float(), outd, 384))
            T[f"rays.{name}.b2"] = c32(sd[src + ".proj2.bias"])
        T["fcc_w"], T["fcc_b"] = h16(sd[dl + "features_channel_cat.weight"]), c32(sd[dl + "features_channel_cat.bias"])
        T["lat.nw"], T["lat.nb"] = c32(sd[dl + "to_latents.norm.weight"]), c32(sd[dl + "to_latents.norm.bias"])
        T["lat.w1"], T["lat.b1"] = h16(sd[dl + "to_latents.proj1.weight"]), c32(sd[dl + "to_latents.proj1.bias"])
        T["lat.w2"], T["lat.b2"] = h16(sd[dl + "to_latents.proj2.weight"]), c32(sd[dl + "to_latents.proj2.bias"])

        def attn_block(dst, src, split_kv):
            for a, b in (("nxw", "norm_attnx.weight"), ("nxb", "norm_attnx.bias"), ("ncw", "norm_attnctx.weight"),
                         ("ncb", "norm_attnctx.bias"), ("q_b", "q.bias"), ("out_b", "out.bias"), ("ls1", "ls1.gamma"),
                         ("ls2", "ls2.gamma"), ("mnw", "mlp.norm.weight"), ("mnb", "mlp.norm.bias"), ("mb1", "mlp.proj1.bias"),
                         ("mb2", "mlp.proj2.bias")):
                T[dst + a] = c32(sd[src + b])
            for a, b in (("q_w", "q.weight"), ("out_w", "out.weight"), ("mw1", "mlp.proj1.weight"), ("mw2", "mlp.proj2.weight")):
                T[dst + a] = h16(sd[src + b])
            kvw, kvb = sd[src + "kv.weight"], sd[src + "kv.bias"]
            d = kvw.shape[1]
            if split_kv:       # dense single-head blocks: k and v projections are separate GEMM operands
                T[dst + "k_w"], T[dst + "k_b"] = h16(kvw[:d]), c32(kvb[:d])
                T[dst + "v_w"], T[dst + "v_b"] = h16(kvw[d:]), c32(kvb[d:])
            else:
                T[dst + "kv_w"], T[dst + "kv_b"] = h16(kvw), c32(kvb)

        attn_block("agg16.", dl + "aggregate_16.", True)
        attn_block("prompt.", dl + "prompt_camera.", True)
        for name, dst, n in (("layers_16", "l16", s.dec_depths[0]), ("layers_8", "l8", s.dec_depths[1]), ("layers_4", "l4", s.dec_depths[2])):
            for i in range(n):
                attn_block(f"{dst}.{i}.", f"{dl}{name}.{i}.", False)
        for name in ("up8", "up4", "up2"):
            for j in range(2):
                block(f"{name}.c{j}.", f"{dl}{name}.convs.{j}.", ("dwconv", "norm", "pwconv1", "pwconv2"))
            uw = sd[f"{dl}{name}.up.0.weight"]
            T[f"{name}.up_w"], T[f"{name}.up_b"] = h16(uw.reshape(uw.shape[0], uw.shape[1])), c32(sd[f"{dl}{name}.up.0.bias"])
            cw = sd[f"{dl}{name}.up.2.weight"]
            T[f"{name}.conv_w"] = h16(cw.permute(0, 2, 3, 1).reshape(cw.shape[0], -1))
            T[f"{name}.conv_b"] = c32(sd[f"{dl}{name}.up.2.bias"])
        for name in ("out8", "out4", "out2"):
            w = sd[f"{dl}{name}.weight"]                                             # [1, C, 3, 3] -> [9, C]
            T[f"{name}.w"] = c32(w.permute(0, 2, 3, 1).reshape(9, w.shape[1]))
            S[f"{name}.b"] = float(sd[f"{dl}{name}.bias"].item())
        return T, S

    def _weights(self):
        if self._packed is None or self._packed_key != self._fingerprint():
            self._pack()
        return self._packed

    # ------------------------------------------------------------------ engine
    def _drop_engine(self):
        self._graphs.clear()
        if self._engine is not None:
            torch.cuda.synchronize(self._engine_device)
            cabi.lib().udb_v1_destroy(self._engine)
        self._engine = None
        self._workspaces.clear()

    def __del__(self):
        try:
            self._drop_engine()
        except Exception:
            pass

    def _engine_config(self) -> "cabi.V1Config":
        """udb_v1_config_t of this model (include/udb.h)."""
        s = self.spec
        cfg = cabi.V1Config()
        for i in range(4):
            cfg.depths[i], cfg.dims[i] = s.depths[i], s.dims[i]
        cfg.hidden, cfg.heads, cfg.expansion = s.hidden, s.heads, s.expansion
        for i in range(3):
            cfg.dec_depths[i] = s.dec_depths[i]
        cfg.net_h, cfg.net_w = self.image_shape
        return cfg

    @staticmethod
    def _register(handle, tensors: dict, scalars: dict):
        """udb_v1_set_weight / udb_v1_set_scalar for every packed operand (the engine borrows the pointers)."""
        lib = cabi.lib()
        for name, t in tensors.items():
            assert t.is_contiguous() and t.dtype in (f16, f32), name
            shape = (C.c_int64 * max(t.ndim, 1))(*t.shape)
            cabi.check(lib.udb_v1_set_weight(handle, name.encode(), C.c_void_p(t.data_ptr()), shape, t.ndim,
                                             cabi.DT_F32 if t.dtype == f32 else cabi.DT_F16), f"udb_v1_set_weight({name})")
        for name, v in scalars.items():
            cabi.check(lib.udb_v1_set_scalar(handle, name.encode(), float(v)), f"udb_v1_set_scalar({name})")

    def _get_engine(self):
        P = self._weights()
        if self._engine is not None:
            return self._engine
        handle = C.c_void_p()
        if self.spec.vit:
            cabi.check(cabi.lib().udb_v1_create_vit(C.byref(self._engine_config()), self.spec.enc_heads, C.byref(handle)),
                       "udb_v1_create_vit")
        else:
            cabi.check(cabi.lib().udb_v1_create(C.byref(self._engine_config()), C.byref(handle)), "udb_v1_create")
        for name, t in P["T"].items():
            assert t.is_cuda, name
        self._register(handle, P["T"], P["S"])
        self._engine, self._engine_device = handle, self.device
        return handle

    def _forward_engine(self, rgb: torch.Tensor, K: Optional[torch.Tensor], skip_camera: bool, scale255: bool, normalize: bool):
        eng = self._get_engine()
        lib = cabi.lib()
        dev = rgb.device
        B, _, H, W = rgb.shape
        wkey = (B, H, W)
        ws = self._workspaces.get(wkey)
        if ws is None:
            nbytes = lib.udb_v1_workspace_bytes(eng, B, H, W)
            if nbytes == 0:
                raise RuntimeError(f"udb_v1_workspace_bytes failed: {lib.udb_last_error().decode()}")
            ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            self._workspaces[wkey] = ws
            while len(self._workspaces) > 4:
                self._workspaces.popitem(last=False)
        self._last_ws = ws
        out = {"intrinsics": torch.empty((B, 3, 3), device=dev, dtype=f32),
               "points": torch.empty((B, 3, H, W), device=dev, dtype=f32),
               "depth": torch.empty((B, 1, H, W), device=dev, dtype=f32)}
        a = cabi.InferV1Args()
        a.rgb, a.rgb_is_u8, a.scale255, a.normalize = rgb.data_ptr(), int(rgb.dtype == torch.uint8), int(scale255), int(normalize)
        a.B, a.H, a.W = B, H, W
        a.intrinsics = K.data_ptr() if K is not None else None
        a.skip_camera = int(bool(skip_camera and K is not None))
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        a.out_intrinsics, a.out_points, a.out_depth = out["intrinsics"].data_ptr(), out["points"].data_ptr(), out["depth"].data_ptr()
        cabi.check(lib.udb_infer_v1(eng, C.byref(a), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "udb_infer_v1")
        return out

    # ------------------------------------------------------------------ infer
    @torch.no_grad()
    def infer(self, rgbs: torch.Tensor, intrinsics=None, skip_camera: bool = False):
        """Same contract as the reference `UniDepthV1.infer` (unidepthv1.py:288-373)."""
        if rgbs.ndim == 3:
            rgbs = rgbs.unsqueeze(0)
        if intrinsics is not None and intrinsics.ndim == 2:
            intrinsics = intrinsics.unsqueeze(0)
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("unidepth_b200 has no CPU path: move the model to a CUDA device")
        with torch.cuda.device(dev):
            rgbs = rgbs.to(dev)
            B = rgbs.shape[0]
            # unidepthv1.py:301-308: "/255" when the data looks like 0..255, ImageNet normalisation when it then lies in [0, 1]
            if rgbs.dtype == torch.uint8:
                scale255, normalize = True, True
            else:
                rgbs = rgbs.float()
                mx, mn = float(rgbs.max()), float(rgbs.min())
                scale255 = mx > 5
                if scale255:
                    mx, mn = mx / 255.0, mn / 255.0
                normalize = mn >= 0.0 and mx <= 1.0
            rgbs = rgbs.contiguous()
            K = None
            if intrinsics is not None:
                K = intrinsics.to(dev, f32).reshape(-1, 3, 3)
                if K.shape[0] != B:
                    raise ValueError(f"intrinsics holds {K.shape[0]} matrices for a batch of {B} images")
                K = K.contiguous()
            self._weights()
            run = lambda x, k: self._forward_engine(x, k, skip_camera, scale255, normalize)
            if not self.use_cuda_graph:
                return run(rgbs, K)
            key = (tuple(rgbs.shape), rgbs.dtype, scale255, normalize, K is not None, bool(skip_camera))
            entry = self._graphs.get(key)
            if entry is None:
                static_in = rgbs.clone()
                static_k = K.clone() if K is not None else None
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    run(static_in, static_k)
                torch.cuda.current_stream().wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    static_out = run(static_in, static_k)
                entry = dict(graph=graph, inp=static_in, k=static_k, out=static_out, ws=self._last_ws)
                self._graphs[key] = entry
                while len(self._graphs) > self.max_cached_graphs:
                    self._graphs.popitem(last=False)
            else:
                self._graphs.move_to_end(key)
            entry["inp"].copy_(rgbs, non_blocking=True)
            if K is not None:
                entry["k"].copy_(K, non_blocking=True)
            entry["graph"].replay()
            bufs = self.output_buffers
            if bufs is not None:
                for k, v in entry["out"].items():
                    bufs[k].copy_(v)
                return {k: bufs[k] for k in entry["out"]}
            return {k: v.clone() for k, v in entry["out"].items()}

    def forward(self, *args, **kwargs):
        raise NotImplementedError("training / validation forward of UniDepthV1 is out of scope; use .infer()")
