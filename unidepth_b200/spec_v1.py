"""Static description of UniDepthV1 (ConvNeXt or DINOv2 ViT encoder) for the inference path: hyper-parameters read from the
reference's config format, the parameter table under the reference's state-dict names, and the fixed-shape
arithmetic of `infer` (reference: unidepth/models/unidepthv1/unidepthv1.py:30-46 `_paddings` / `_shapes`,
:423-447 `build`; unidepthv1/decoder.py:465-533 `Decoder.build`; backbones/convnext.py:301-448)."""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, Tuple

from .spec import PATCH, _VIT, vit_encoder_param_shapes

CONVNEXT_ARCHS = {
    # encoder.py:127-136 (`convnext_large`): depths / dims / per-stage end indices used as `output_idx`
    "convnext_large": dict(depths=(3, 3, 27, 3), dims=(192, 384, 768, 1536)),
    "convnext_large_pt": dict(depths=(3, 3, 27, 3), dims=(192, 384, 768, 1536)),
}


class V1Spec:
    def __init__(self, config: dict):
        m = config["model"]
        enc = m["pixel_encoder"]
        name = enc["name"]
        self.vit = name in _VIT
        if self.vit:
            # encoder.py:139-193: every block is an output; `depths` are the lengths of the four block ranges the decoder
            # max-stacks (decoder.py:371-374) and every range has the embedding width
            d, depth, heads, taps = _VIT[name]
            self.embed_dim, self.enc_depth, self.enc_heads = d, depth, heads
            self.output_idx = tuple(enc.get("output_idx", taps))
            idx = (0,) + self.output_idx
            if len(self.output_idx) != 4 or any(b <= a for a, b in zip(idx, idx[1:])) or self.output_idx[-1] != depth:
                raise NotImplementedError(f"output_idx {list(self.output_idx)}: needs 4 increasing block indices ending at "
                                          f"the depth ({depth})")
            self.depths = tuple(b - a for a, b in zip(idx, idx[1:]))
            self.dims = (d,) * 4
        else:
            if name not in CONVNEXT_ARCHS and "arch" not in enc:
                raise NotImplementedError(f"UniDepthV1 encoder '{name}': only the ConvNeXt and DINOv2 ViT encoders "
                                          "are implemented")
            arch = enc.get("arch", CONVNEXT_ARCHS.get(name))       # "arch": test-only override {depths, dims}
            self.depths = tuple(arch["depths"])
            self.dims = tuple(arch["dims"])
            ends, acc = [], 0
            for d in self.depths:
                acc += d
                ends.append(acc)
            self.output_idx = tuple(enc.get("output_idx", ends))   # encoder.py:131 default [3, 6, 33, 36]
            if tuple(self.output_idx) != tuple(ends):
                raise NotImplementedError("output_idx must be the last block of each ConvNeXt stage")
        self.hidden = m["pixel_decoder"]["hidden_dim"]
        self.dec_depths = tuple(m["pixel_decoder"]["depths"])    # blocks at 1/16, 1/8 (Nystrom), 1/4 (Nystrom)
        self.heads = m["num_heads"]
        self.expansion = m["expansion"]
        self.image_shape = tuple(config["data"]["image_shape"])  # fixed network input (462, 616)
        if self.vit and (self.image_shape[0] % PATCH or self.image_shape[1] % PATCH):
            raise NotImplementedError(f"network shape {self.image_shape} is not a multiple of the patch size {PATCH}")
        # decoder.py:489-492: token adapters read the cls tokens of the last four BLOCKS, newest first
        per_block = [c for d, c in zip(self.depths, self.dims) for _ in range(d)]
        self.cls_dims = tuple(per_block[-i - 1] for i in range(4))
        if self.hidden % 64 or (self.hidden // self.heads) != 64:
            raise NotImplementedError("decoder needs 64-wide heads (hidden_dim / num_heads == 64)")


def v1_shapes(image_hw: Tuple[int, int], network_hw: Tuple[int, int]):
    """unidepthv1.py:38-46: ((h', w'), ratio) of the aspect-preserving resize into the fixed network shape."""
    h, w = image_hw
    if network_hw[1] / network_hw[0] > w / h:
        ratio = network_hw[0] / h
    else:
        ratio = network_hw[1] / w
    return (math.ceil(h * ratio - 0.5), math.ceil(w * ratio - 0.5)), ratio


def v1_paddings(resized_hw: Tuple[int, int], network_hw: Tuple[int, int]):
    """unidepthv1.py:30-35: (left, right, top, bottom)."""
    dh, dw = network_hw[0] - resized_hw[0], network_hw[1] - resized_hw[1]
    return dw // 2, dw - dw // 2, dh // 2, dh - dh // 2


def param_shapes(config: dict) -> "OrderedDict[str, tuple]":
    """name -> shape of every parameter of the reference `UniDepthV1(config)` state dict."""
    s = V1Spec(config)
    out: "OrderedDict[str, tuple]" = OrderedDict()
    pe = "pixel_encoder."
    if s.vit:
        vit_encoder_param_shapes(out, pe, s.embed_dim, s.enc_depth)
    else:
        _convnext_param_shapes(out, pe, s)
    _decoder_param_shapes(out, s)
    return out


def level_grid(spec: V1Spec) -> Tuple[int, int]:
    """The decoder's common grid (decoder.py:381-392): the ViT patch grid, or the ConvNeXt pyramid's 1/16 level."""
    if spec.vit:
        return spec.image_shape[0] // PATCH, spec.image_shape[1] // PATCH
    sh = [(spec.image_shape[0] - 4) // 4 + 1, (spec.image_shape[1] - 4) // 4 + 1]
    return sh[0] // 4, sh[1] // 4


def _convnext_param_shapes(out, pe: str, s: V1Spec):
    d0 = s.dims[0]
    out[pe + "mask_token"] = (1, d0, 1, 1)
    out[pe + "stem.0.weight"], out[pe + "stem.0.bias"] = (d0, 3, 4, 4), (d0,)
    out[pe + "stem.1.weight"], out[pe + "stem.1.bias"] = (d0,), (d0,)
    prev = d0
    for i, (depth, c) in enumerate(zip(s.depths, s.dims)):
        st = f"{pe}stages.{i}."
        if i > 0:
            out[st + "downsample.0.weight"], out[st + "downsample.0.bias"] = (prev,), (prev,)
            out[st + "downsample.1.weight"], out[st + "downsample.1.bias"] = (c, prev, 2, 2), (c,)
        for j in range(depth):
            b = f"{st}blocks.{j}."
            out[b + "gamma"] = (c,)
            out[b + "conv_dw.weight"], out[b + "conv_dw.bias"] = (c, 1, 7, 7), (c,)
            out[b + "norm.weight"], out[b + "norm.bias"] = (c,), (c,)
            out[b + "mlp.fc1.weight"], out[b + "mlp.fc1.bias"] = (4 * c, c), (4 * c,)
            out[b + "mlp.fc2.weight"], out[b + "mlp.fc2.bias"] = (c, 4 * c), (c,)
        prev = c


def _decoder_param_shapes(out, s: V1Spec):
    pd = "pixel_decoder."
    hid, ex = s.hidden, s.expansion

    def ln(p, c):
        out[p + ".weight"], out[p + ".bias"] = (c,), (c,)

    def lin(p, cout, cin):
        out[p + ".weight"], out[p + ".bias"] = (cout, cin), (cout,)

    def mlp(p, c, expansion, outd=None):
        ln(p + ".norm", c)
        lin(p + ".proj1", int(c * expansion), c)
        lin(p + ".proj2", outd if outd is not None else c, int(c * expansion))

    def attn_block(p, c):
        mlp(p + ".mlp", c, ex)
        lin(p + ".kv", 2 * c, c)
        lin(p + ".q", c, c)
        ln(p + ".norm_attnx", c)
        ln(p + ".norm_attnctx", c)
        lin(p + ".out", c, c)
        out[p + ".ls1.gamma"], out[p + ".ls2.gamma"] = (c,), (c,)

    def conv_upsample(p, c):
        for j in range(2):
            b = f"{p}.convs.{j}"
            out[b + ".gamma"] = (c,)
            out[b + ".dwconv.weight"], out[b + ".dwconv.bias"] = (c, 1, 7, 7), (c,)
            ln(b + ".norm", c)
            lin(b + ".pwconv1", ex * c, c)
            lin(b + ".pwconv2", c, ex * c)
        out[p + ".up.0.weight"], out[p + ".up.0.bias"] = (c // 2, c, 1, 1), (c // 2,)
        out[p + ".up.2.weight"], out[p + ".up.2.bias"] = (c // 2, c // 2, 3, 3), (c // 2,)

    out[pd + "level_embeds"] = (4, hid)
    for i, c in enumerate(s.dims):
        ln(f"{pd}input_adapter.input_adapters.{i}.0", c)
        lin(f"{pd}input_adapter.input_adapters.{i}.1", hid, c)
    for i, c in enumerate(s.cls_dims):
        ln(f"{pd}token_adapter.input_adapters.{i}.0", c)
        lin(f"{pd}token_adapter.input_adapters.{i}.1", hid, c)
    cl = pd + "camera_layer"
    out[cl + ".latents_pos"] = (1, 4, hid)
    attn_block(cl + ".aggregate", hid)
    for i in range(2):
        attn_block(f"{cl}.layers.{i}", hid)
    mlp(cl + ".in_features", hid, 2)
    mlp(cl + ".out", hid, 2, 1)
    ln(cl + ".cls_project.0", hid)
    lin(cl + ".cls_project.1", hid // 2, hid)
    lin(cl + ".cls_project.3", hid, hid // 2)
    dl = pd + "depth_layer"
    for name, outd in (("16", hid), ("8", hid // 2), ("4", hid // 4)):
        mlp(f"{dl}.project_rays{name}", 81, ex, outd)
    mlp(dl + ".to_latents", hid, 2)
    lin(dl + ".features_channel_cat", hid, 4 * hid)
    conv_upsample(dl + ".up8", hid)
    conv_upsample(dl + ".up4", hid // 2)
    conv_upsample(dl + ".up2", hid // 4)
    for name, c, n in (("layers_16", hid, s.dec_depths[0]), ("layers_8", hid // 2, s.dec_depths[1]),
                       ("layers_4", hid // 4, s.dec_depths[2])):
        for i in range(n):
            attn_block(f"{dl}.{name}.{i}", c)
    attn_block(dl + ".aggregate_16", hid)
    attn_block(dl + ".prompt_camera", hid)
    for name, c in (("out2", hid // 8), ("out4", hid // 4), ("out8", hid // 2)):
        out[f"{dl}.{name}.weight"], out[f"{dl}.{name}.bias"] = (1, c, 3, 3), (1,)
    lin(pd + "level_embed_layer.0", hid, hid)
    lin(pd + "level_embed_layer.2", hid, hid)
    ln(pd + "level_embed_layer.3", hid)
