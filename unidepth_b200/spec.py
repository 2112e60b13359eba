"""Shape arithmetic and state-dict layout of the UniDepthV2 inference path (host side, pure
Python).  Mirrors the reference's config handling and pre-processing integer/float arithmetic:
unidepth/models/unidepthv2/unidepthv2.py:36-77,247-262,418-460 and
unidepth/models/unidepthv2/decoder.py:470-524."""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Optional

PATCH = 14

# unidepth/models/backbones/dinov2.py:388-427 ; default taps unidepth/models/encoder.py:139-193
_VIT = {
    "dinov2_vits14": (384, 12, 6, [3, 6, 9, 12]),
    "dinov2_vitb14": (768, 12, 12, [3, 6, 9, 12]),
    "dinov2_vitl14": (1024, 24, 16, [5, 12, 18, 24]),
}


class ModelSpec:
    def __init__(self, config: dict):
        enc = config["model"]["pixel_encoder"]
        dec = config["model"]["pixel_decoder"]
        name = enc["name"]
        if name not in _VIT:
            raise NotImplementedError(
                f"pixel_encoder '{name}': only the DINOv2 ViT encoders of UniDepthV2 are implemented")
        d, depth, heads, taps = _VIT[name]
        over = enc.get("arch_override", {})
        self.name = name
        self.embed_dim = over.get("embed_dim", d)
        self.depth = over.get("depth", depth)
        self.enc_heads = over.get("num_heads", heads)
        self.taps = list(enc.get("output_idx", taps))
        self.use_norm = bool(enc.get("use_norm", False))
        self.hidden = dec["hidden_dim"]
        self.dec_heads = config["model"]["num_heads"]
        self.expansion = config["model"]["expansion"]
        self.dec_depths = list(dec["depths"])
        self.out_dim = dec["out_dim"]
        self.kernel_size = dec.get("kernel_size", 7)
        sc = config["data"]["augmentations"]["shape_constraints"]
        self.shape_constraints = dict(sc)
        h = self.hidden
        self.cur, self.nxt, self.outd = [], [], []
        for i in range(len(self.dec_depths)):
            self.cur.append(min(h, 2 * h // int(2 ** i)))
            self.nxt.append(2 * h // int(2 ** (i + 1)))
            self.outd.append(max(self.nxt[-1], self.out_dim))


def get_paddings(original_shape, aspect_ratio_range):
    """unidepthv2.py:36-58 -> (pad_left, pad_right, pad_top, pad_bottom), (H_new, W_new)."""
    h_ori, w_ori = original_shape
    ratio = w_ori / h_ori
    lo, hi = aspect_ratio_range
    target = min(hi, max(lo, ratio))
    if ratio > target:
        w_new, h_new = w_ori, int(w_ori / target)
        top = (h_new - h_ori) // 2
        return (0, 0, top, h_new - h_ori - top), (h_new, w_new)
    h_new, w_new = h_ori, int(h_ori * target)
    left = (w_new - w_ori) // 2
    return (left, w_new - w_ori - left, 0, 0), (h_new, w_new)


def get_resize_factor(original_shape, pixels_range, shape_multiplier=PATCH):
    """unidepthv2.py:61-77 -> factor, (new_H, new_W)."""
    h_ori, w_ori = original_shape
    n_ori = w_ori * h_ori
    lo, hi = pixels_range
    target = min(hi, max(lo, n_ori))
    factor = (target / n_ori) ** 0.5
    new_w = int(w_ori * factor)
    new_h = int(h_ori * factor)
    new_h = math.ceil(new_h / shape_multiplier) * shape_multiplier
    new_w = math.ceil(new_w / shape_multiplier) * shape_multiplier
    return factor, (new_h, new_w)


def pixel_bounds(shape_constraints: dict, resolution_level: Optional[int]):
    """unidepthv2.py:247-262."""
    lo, hi = shape_constraints["pixels_min"], shape_constraints["pixels_max"]
    if resolution_level is None:
        return (lo, hi)
    assert 0 <= resolution_level < 10, "resolution_level should be in [0, 10)"
    interval = (hi - lo) / 10
    return (resolution_level * interval + lo, (resolution_level + 1) * interval + lo)


def vit_encoder_param_shapes(out: "OrderedDict[str, tuple]", pe: str, d: int, depth: int):
    """The DINOv2 encoder's state-dict entries (dinov2.py:186-257; one register token slot, no registers used), added to
    `out` under the prefix `pe`; shared by UniDepthV2 and UniDepthV1 with a ViT encoder."""
    out[pe + "cls_token"] = (1, 1, d)
    out[pe + "pos_embed"] = (1, 1 + 37 * 37, d)
    out[pe + "register_tokens"] = (1, 1, d)
    out[pe + "mask_token"] = (1, d)
    out[pe + "patch_embed.proj.weight"] = (d, 3, PATCH, PATCH)
    out[pe + "patch_embed.proj.bias"] = (d,)
    for i in range(depth):
        b = f"{pe}blocks.{i}."
        for nm, shp in (("norm1.weight", (d,)), ("norm1.bias", (d,)), ("attn.qkv.weight", (3 * d, d)),
                        ("attn.qkv.bias", (3 * d,)), ("attn.proj.weight", (d, d)), ("attn.proj.bias", (d,)),
                        ("ls1.gamma", (d,)), ("norm2.weight", (d,)), ("norm2.bias", (d,)),
                        ("mlp.fc1.weight", (4 * d, d)), ("mlp.fc1.bias", (4 * d,)),
                        ("mlp.fc2.weight", (d, 4 * d)), ("mlp.fc2.bias", (d,)), ("ls2.gamma", (d,))):
            out[b + nm] = shp
    out[pe + "norm.weight"] = (d,)
    out[pe + "norm.bias"] = (d,)


def param_shapes(config: dict) -> "OrderedDict[str, tuple]":
    """key -> shape of every tensor in the reference UniDepthV2 `state_dict()` (same names, same
    order of magnitude as SURVEY.md section 8b), so reference checkpoints load unchanged."""
    s = ModelSpec(config)
    d, h = s.embed_dim, s.hidden
    out: "OrderedDict[str, tuple]" = OrderedDict()
    pe = "pixel_encoder."
    vit_encoder_param_shapes(out, pe, d, s.depth)

    pd = "pixel_decoder."
    out[pd + "level_embeds"] = (1, 1, 4, h)
    for adapter in ("input_adapter", "camera_token_adapter"):
        for i in range(4):
            out[f"{pd}{adapter}.input_adapters.{i}.weight"] = (h, d)
            out[f"{pd}{adapter}.input_adapters.{i}.bias"] = (h,)

    def mlp(prefix, hid, od):
        out[prefix + ".norm.weight"] = (h,)
        out[prefix + ".norm.bias"] = (h,)
        out[prefix + ".proj1.weight"] = (hid, h)
        out[prefix + ".proj1.bias"] = (hid,)
        out[prefix + ".proj2.weight"] = (od, hid)
        out[prefix + ".proj2.bias"] = (od,)

    def block(prefix, layer_scale):
        mlp(prefix + ".mlp", s.expansion * h, h)
        out[prefix + ".kv.weight"] = (2 * h, h)
        out[prefix + ".q.weight"] = (h, h)
        for nm in ("norm_attnx", "norm_attnctx"):
            out[f"{prefix}.{nm}.weight"] = (h,)
            out[f"{prefix}.{nm}.bias"] = (h,)
        out[prefix + ".out.weight"] = (h, h)
        if layer_scale:
            out[prefix + ".ls1.gamma"] = (h,)
            out[prefix + ".ls2.gamma"] = (h,)

    cl = pd + "camera_layer."
    out[cl + "latents_pos"] = (1, 4, h)
    block(cl + "aggregate1", True)
    block(cl + "aggregate2", True)
    mlp(cl + "project", h, h)
    mlp(cl + "out_pinhole", h, 1)

    dl = pd + "depth_layer."
    n_up = len(s.dec_depths)
    ks = s.kernel_size
    for i in range(n_up):
        for j in range(s.dec_depths[i]):
            u = f"{dl}ups.{i}.convs.{j}."
            out[u + "gamma"] = (1, s.cur[i], 1, 1)
            for cv in ("conv1", "conv2"):
                out[f"{u}{cv}.weight"] = (s.cur[i], s.cur[i], ks, ks)
                out[f"{u}{cv}.bias"] = (s.cur[i],)
        out[f"{dl}ups.{i}.up.0.weight"] = (s.outd[i], s.cur[i], 1, 1)
        out[f"{dl}ups.{i}.up.0.bias"] = (s.outd[i],)
    last = n_up - 1
    out[f"{dl}depth_mlp.{last}.0.weight"] = (s.nxt[last],)
    out[f"{dl}depth_mlp.{last}.0.bias"] = (s.nxt[last],)
    out[f"{dl}depth_mlp.{last}.1.weight"] = (s.outd[last], s.nxt[last])
    out[f"{dl}depth_mlp.{last}.1.bias"] = (s.outd[last],)
    for i in range(n_up):
        k = max(1, 2 * i)
        out[f"{dl}process_features.{i}.weight"] = (h, s.cur[i], k, k)
        out[f"{dl}process_features.{i}.bias"] = (s.cur[i],)
    for i in range(4):
        block(f"{dl}prompt_camera.{i}.layers.0", False)
    out[dl + "to_latents.weight"] = (h, h)
    out[dl + "to_latents.bias"] = (h,)
    out[dl + "confidence_mlp.0.weight"] = (s.nxt[last],)
    out[dl + "confidence_mlp.0.bias"] = (s.nxt[last],)
    out[dl + "confidence_mlp.1.weight"] = (s.outd[last], s.nxt[last])
    out[dl + "confidence_mlp.1.bias"] = (s.outd[last],)
    od = s.outd[last]
    for nm in ("to_depth_lr", "to_confidence_lr"):
        out[f"{dl}{nm}.weight"] = (od // 2, od, 3, 3)
        out[f"{dl}{nm}.bias"] = (od // 2,)
    for nm in ("to_depth_hr", "to_confidence_hr"):
        out[f"{dl}{nm}.0.weight"] = (32, od // 2, 3, 3)
        out[f"{dl}{nm}.0.bias"] = (32,)
        out[f"{dl}{nm}.2.weight"] = (1, 32, 1, 1)
        out[f"{dl}{nm}.2.bias"] = (1,)
    return out
