"""Torch-fp32 functional restatement of `UniDepthV1.infer()` with the DINOv2 ViT encoder (configs/config_v1_vitl14.json),
and the seeded weights it runs on.  TEST INFRASTRUCTURE ONLY, like oracle/unidepth_v1_oracle.py, whose decoder and pre /
post-processing it reuses unchanged; only the encoder differs from the ConvNeXt model.

Reference walk (file:line under the reference's unidepth/):
  models/unidepthv1/unidepthv1.py:418-424   build: encoder config with interpolate_offset 0.1 -> interpolate_pos_embed(offset=0.1)
                                  :322-326  encoder outputs + their cls token          -> vit_encoder_v1
  models/encoder.py:177-192                 dinov2_vitl14: output_idx [5,12,18,24], use_norm False
  models/backbones/dinov2.py:267-347        interpolate_pos_encoding, prepare_tokens, forward (every block returned)
  models/unidepthv1/decoder.py:364-396      max_stack over [0,5) [5,12) [12,18) [18,24); one grid -> flat_interpolate is the
                                            identity (utils/geometric.py:235)                   -> unidepth_v1_oracle.decoder_v1
"""
import math
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

import unidepth_v1_oracle as O1
from unidepth_oracle import _lin, _ln, _sdpa
from unidepth_v1_parts import spherical_zbuffer_to_euclidean, v1_paddings, v1_postprocess, v1_preprocess, v1_shapes
from unidepth_v1_oracle import generate_rays

PATCH = 14
VIT = {"dinov2_vits14": (384, 12, 6, [3, 6, 9, 12]), "dinov2_vitb14": (768, 12, 12, [3, 6, 9, 12]),
       "dinov2_vitl14": (1024, 24, 16, [5, 12, 18, 24])}


def interpolate_pos_embed(pos_embed: torch.Tensor, gh: int, gw: int, offset: float = 0.0) -> torch.Tensor:
    """dinov2.py:267-304: the 37x37 table resampled bicubically (antialias off) to gh x gw.  offset 0 (V2): by output
    size; offset > 0 (V1: 0.1): by scale_factor ((gh + offset) / 37, (gw + offset) / 37), whose sample positions differ."""
    n = pos_embed.shape[1] - 1
    m = int(math.sqrt(n))
    assert m * m == n
    dim = pos_embed.shape[-1]
    if gh == m and gw == m:
        return pos_embed
    grid = pos_embed[:, 1:].reshape(1, m, m, dim).permute(0, 3, 1, 2)
    if offset:
        grid = F.interpolate(grid, scale_factor=((gh + offset) / m, (gw + offset) / m), mode="bicubic", antialias=False)
    else:
        grid = F.interpolate(grid, size=(gh, gw), mode="bicubic", antialias=False)
    assert tuple(grid.shape[-2:]) == (gh, gw)
    return torch.cat([pos_embed[:, :1], grid.permute(0, 2, 3, 1).reshape(1, gh * gw, dim)], dim=1)


def vit_encoder_v1(sd: Dict[str, torch.Tensor], image: torch.Tensor, depth: int, heads: int,
                   offset: float = 0.1) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
    """DinoVisionTransformer.forward with use_norm False (dinov2.py:324-347) + unidepthv1.py:322-326: every block's patch
    map with its cls token added [B, gh, gw, D], and every block's cls token [B, 1, D]."""
    p = "pixel_encoder."
    b, _, hh, ww = image.shape
    gh, gw = hh // PATCH, ww // PATCH
    x = F.conv2d(image, sd[p + "patch_embed.proj.weight"], sd[p + "patch_embed.proj.bias"], stride=PATCH)
    x = torch.cat([sd[p + "cls_token"].expand(b, -1, -1), x.flatten(2).transpose(1, 2)], dim=1)
    x = x + interpolate_pos_embed(sd[p + "pos_embed"].float(), gh, gw, offset)
    d = x.shape[-1]
    outs, clss = [], []
    for i in range(depth):
        bp = f"{p}blocks.{i}."
        # metadinov2/block.py:84-109, attention.py:51-62, mlp.py:35-41; LayerNorm eps 1e-6
        qkv = _lin(_ln(x, sd, bp + "norm1", 1e-6), sd, bp + "attn.qkv").view(b, -1, 3, heads, d // heads).permute(2, 0, 3, 1, 4)
        x = x + _lin(_sdpa(qkv[0], qkv[1], qkv[2]).transpose(1, 2).reshape(b, -1, d), sd, bp + "attn.proj") * sd[bp + "ls1.gamma"]
        x = x + _lin(F.gelu(_lin(_ln(x, sd, bp + "norm2", 1e-6), sd, bp + "mlp.fc1")), sd, bp + "mlp.fc2") * sd[bp + "ls2.gamma"]
        clss.append(x[:, :1])
        outs.append((x[:, 1:] + x[:, :1]).reshape(b, gh, gw, d))
    return outs, clss


@torch.no_grad()
def infer_v1_vit(sd: Dict[str, torch.Tensor], cfg: dict, rgbs: torch.Tensor, intrinsics: Optional[torch.Tensor] = None,
                 skip_camera: bool = False) -> Dict[str, torch.Tensor]:
    """unidepthv1.py:288-373 for a DINOv2 encoder: the same steps as unidepth_v1_oracle.infer_v1 around vit_encoder_v1."""
    if rgbs.ndim == 3:
        rgbs = rgbs.unsqueeze(0)
    if intrinsics is not None and intrinsics.ndim == 2:
        intrinsics = intrinsics.unsqueeze(0)
    B, _, H, W = rgbs.shape
    if rgbs.max() > 5 or rgbs.dtype == torch.uint8:
        rgbs = rgbs.to(torch.float32).div(255)
    if rgbs.min() >= 0.0 and rgbs.max() <= 1.0:
        mean = torch.tensor(O1.IMAGENET_MEAN, dtype=rgbs.dtype).view(1, 3, 1, 1)
        std = torch.tensor(O1.IMAGENET_STD, dtype=rgbs.dtype).view(1, 3, 1, 1)
        rgbs = (rgbs - mean) / std
    net_hw = tuple(cfg["data"]["image_shape"])
    enc = cfg["model"]["pixel_encoder"]
    _, depth, heads, taps = VIT[enc["name"]]
    output_idx = enc.get("output_idx", taps)
    (h, w), ratio = v1_shapes((H, W), net_hw)
    pads = v1_paddings((h, w), net_hw)
    x, gt_k = v1_preprocess(rgbs, intrinsics, (h, w), pads, ratio)
    enc_outs, cls_all = vit_encoder_v1(sd, x, depth, heads)
    K, outs, _ = O1.decoder_v1(sd, enc_outs, cls_all, net_hw, output_idx, cfg["model"]["num_heads"], gt_k=gt_k,
                               skip_camera=skip_camera and gt_k is not None)
    pred, K_out = v1_postprocess(outs, K.clone(), net_hw, pads, ratio, (H, W))
    use_k = gt_k if gt_k is not None else K_out          # unidepthv1.py:354-356, as in infer_v1
    angles = generate_rays(use_k, (H, W))[1].transpose(1, 2).reshape(B, 2, H, W)
    pts = spherical_zbuffer_to_euclidean(torch.cat((angles, pred), dim=1).permute(0, 2, 3, 1)).permute(0, 3, 1, 2)
    return {"intrinsics": K_out, "points": pts, "depth": pred[:, -1:]}


def make_v1_vit_state_dict(config: dict, seed: int = 0) -> Dict[str, torch.Tensor]:
    """Seeded fixture for UniDepthV1 with a ViT encoder, the recipe of fixture.make_v1_state_dict (one generator per
    tensor, seeded from (seed, index in spec_v1.param_shapes)) plus the DINOv2-only tensors: cls_token and pos_embed
    0.2 N(0,1), register_tokens N(0,1) (unused on the infer path), mask_token 0."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    from unidepth_b200.spec_v1 import param_shapes as v1_shapes
    sd: Dict[str, torch.Tensor] = {}
    for idx, (key, shape) in enumerate(v1_shapes(config).items()):
        g = torch.Generator().manual_seed(seed * 1_000_003 + idx)
        n = lambda *s: torch.randn(*s, generator=g)
        u = lambda *s: torch.rand(*s, generator=g)
        leaf = key.rsplit(".", 1)[-1]
        is_norm = ("norm" in key or key.endswith((".0.weight", ".0.bias")) and "input_adapters" in key
                   or "cls_project.0." in key or "level_embed_layer.3." in key)
        if key.endswith("mask_token"):
            t = torch.zeros(*shape)
        elif key.endswith(("cls_token", "pos_embed")):
            t = 0.2 * n(*shape)
        elif key.endswith("register_tokens"):
            t = n(*shape)
        elif key.endswith(("level_embeds", "latents_pos")):
            t = 0.5 * n(*shape)
        elif ".ls1.gamma" in key or ".ls2.gamma" in key:
            t = 0.3 * (0.5 + u(*shape))
        elif leaf == "gamma":
            t = 0.4 * (0.5 + u(*shape))
        elif is_norm and len(shape) == 1:
            t = 1.0 + 0.1 * n(*shape) if leaf == "weight" else 0.05 * n(*shape)
        elif leaf == "bias":
            t = 0.05 * n(*shape)
        elif leaf == "weight":
            t = n(*shape) / math.prod(shape[1:]) ** 0.5
            if key.endswith(("camera_layer.out.proj2.weight", "out2.weight", "out4.weight", "out8.weight")):
                t = 0.3 * t
        else:
            raise KeyError(key)
        sd[key] = t.float().contiguous()
    return sd
