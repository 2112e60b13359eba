"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from
/root/reference through oracle/ref_shims) on the seeded fixture weights.

Run here (CPU container, has /root/reference):   python oracle/make_golden.py
The GPU box has no /root/reference; it only reads the committed .npz files.
TEST INFRASTRUCTURE ONLY.
"""
import copy
import json
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
sys.path[:0] = [REF, os.path.join(HERE, "ref_shims"), HERE]

from fixture import make_state_dict, param_shapes  # noqa: E402

CASES = [
    # name, config, seed, (B,H,W), resolution_level[, strides as in BIG_CASES; default (1, 1, 4)]
    ("vits_120x160", "config_v2_vits14.json", 0, (1, 120, 160), None),
    ("vits_pad_96x288_rl3", "config_v2_vits14.json", 1, (2, 96, 288), 3, (1, 2, 16)),
    ("vitb_112x160", "config_v2_vitb14.json", 2, (1, 112, 160), None),
]
# The benchmark configuration itself (BASELINE.json configs[1]: ViT-L/14, 3x480x640), full depth, one image.
# Takes a few minutes on CPU, so it is generated on request:  python oracle/make_golden.py vitl
# Stored: intrinsics in full; depth every 2nd pixel; the other maps every 4th pixel; depth_features every 32nd channel.
# `python oracle/make_golden.py vitl` also writes BASELINE configs[4]'s shape (3x1024x1536 -> 644x952, 3129 tokens) at full
# depth: depth every 4th pixel, the other maps every 16th, depth_features every 32nd channel.
# The strides keep every file under 1 MB.
BIG_CASES = [
    # name, config, seed, (B,H,W), resolution_level, (depth stride, spatial stride, depth_features channel stride)
    ("vitl_480x640", "config_v2_vitl14.json", 0, (1, 480, 640), None, (2, 4, 32)),
    ("vitl_1024x1536", "config_v2_vitl14.json", 3, (1, 1024, 1536), None, (4, 16, 32)),
]


def seeded_rgb(shape, seed):
    g = torch.Generator().manual_seed(1234 + seed)
    b, h, w = shape
    return torch.randint(0, 256, (b, 3, h, w), dtype=torch.uint8, generator=g)


def main():
    warnings.simplefilter("ignore")
    from unidepth.models import UniDepthV2
    out_dir = os.path.join(HERE, "..", "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    big = len(sys.argv) > 1 and sys.argv[1] == "vitl"
    only = sys.argv[2] if len(sys.argv) > 2 else None
    for name, cfg_name, seed, shape, level, *rest in (BIG_CASES if big else CASES):
        if only and name != only:
            continue
        sd_, ss_, sc_ = rest[0] if rest else (1, 1, 4)
        cfg = json.load(open(os.path.join(REF, "configs", cfg_name)))
        model = UniDepthV2(copy.deepcopy(cfg)).eval()
        ref_sd = model.state_dict()
        shapes = param_shapes(cfg)
        assert list(shapes.keys()) == list(ref_sd.keys()) or set(shapes) == set(ref_sd), \
            (set(shapes) ^ set(ref_sd))
        for k, v in ref_sd.items():
            assert tuple(v.shape) == tuple(shapes[k]), (k, v.shape, shapes[k])
        sd = make_state_dict(cfg, seed)
        info = model.load_state_dict(sd, strict=True)
        if level is not None:
            model.resolution_level = level
        rgb = seeded_rgb(shape, seed)
        out = model.infer(rgb)
        arrays = {k: v.detach().cpu().numpy() for k, v in out.items()}
        # depth_features is large; keep every sc_-th channel (the restatement is checked on those)
        arrays["depth_features"] = arrays["depth_features"][:, ::sc_]
        arrays["depth"] = arrays["depth"][:, :, ::sd_, ::sd_]
        for k in ("confidence", "radius", "points", "rays"):
            arrays[k] = arrays[k][:, :, ::ss_, ::ss_]
        meta = dict(config=cfg_name, seed=seed, shape=list(shape), resolution_level=level,
                    strides=dict(depth=sd_, spatial=ss_, depth_features=sc_))
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), __meta__=json.dumps(meta), **arrays)
        d = arrays["depth"]
        print(name, "depth range", float(d.min()), float(d.max()), "conf", float(arrays["confidence"].min()),
              float(arrays["confidence"].max()), "K", arrays["intrinsics"][0].tolist())
    if big:
        return
    # reference outputs of the validation glue (misc.py:596-690, evaluation_depth.py:93-110) on seeded inputs
    from unidepth.utils.misc import match_gt, match_intrinsics
    from unidepth.utils.evaluation_depth import DICT_METRICS
    g = torch.Generator().manual_seed(99)
    pred = torch.rand(3, 2, 28, 42, generator=g) + 0.5
    gt = torch.rand(3, 1, 37, 61, generator=g) + 0.5
    img = torch.zeros(3, 3, 28, 42)
    pads1 = [(0, 0, 0, 0), (2, 3, 0, 0), (0, 0, 4, 1)]
    pads2 = [(1, 0, 0, 2), (0, 0, 0, 0), (3, 3, 1, 1)]
    K = torch.tensor([[30.0, 0, 20.5], [0, 31.0, 14.0], [0, 0, 1]]).repeat(3, 1, 1) + torch.rand(3, 3, 3, generator=g) * torch.tensor([[1.0, 0, 1], [0, 1, 1], [0, 0, 0]])
    arrays = dict(pred=pred.numpy(), gt=gt.numpy(), K=K.numpy(), pads1=np.array(pads1), pads2=np.array(pads2),
                  m_none=match_gt(pred, gt, None, None).numpy(), m_p1=match_gt(pred, gt, pads1, None).numpy(),
                  m_p12=match_gt(pred, gt, pads1, pads2).numpy(),
                  k_p1=match_intrinsics(K, img, gt, pads1, None).numpy(), k_p12=match_intrinsics(K, img, gt, pads1, pads2).numpy())
    a, b = gt[0, 0].flatten(), (gt[0, 0] * (1 + 0.2 * (torch.rand(37, 61, generator=g) - 0.5))).flatten()
    arrays["met_gt"], arrays["met_pred"] = a.numpy(), b.numpy()
    for name in ("d1", "d2", "d3", "rmse", "rmselog", "arel", "sqrel", "log10", "silog"):
        arrays["met_" + name] = np.array(float(DICT_METRICS[name](a, b).mean()))
    np.savez_compressed(os.path.join(out_dir, "validation_glue.npz"), **arrays)
    # V1 ray embedding basis (next row): the reference's rsh_cart_8 on seeded unit vectors (sht.py:833-1393)
    from unidepth.utils.sht import rsh_cart_8
    v = torch.randn(256, 3, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    v = v / v.norm(dim=-1, keepdim=True)
    np.savez_compressed(os.path.join(out_dir, "sh81.npz"), xyz=v.numpy(), rsh=rsh_cart_8(v).numpy())
    # V1 host-side pieces (unidepthv1.py:30-94, geometric.py:13-73) on seeded inputs
    from unidepth.models.unidepthv1.unidepthv1 import _paddings, _postprocess, _preprocess, _shapes
    from unidepth.utils.geometric import generate_rays as ref_rays, spherical_zbuffer_to_euclidean as ref_s2e
    g = torch.Generator().manual_seed(21)
    net = (462, 616)
    cases = [(480, 640), (375, 1242), (1000, 400), (231, 308)]
    arr = {"cases": np.array(cases)}
    for i, (h, w) in enumerate(cases):
        (rh, rw), ratio = _shapes((h, w), net)
        pads = _paddings((rh, rw), net)
        arr[f"shape{i}"] = np.array([rh, rw, *pads], dtype=np.int64)
        arr[f"ratio{i}"] = np.array(ratio)
    h, w = 60, 99
    rgb = torch.rand(2, 3, h, w, generator=g)
    K = torch.tensor([[[75.0, 0, 50.0], [0, 76.0, 30.5], [0, 0, 1]], [[70.0, 0, 49.0], [0, 69.5, 29.25], [0, 0, 1]]])
    small_net = (42, 56)
    (rh, rw), ratio = _shapes((h, w), small_net)
    pads = _paddings((rh, rw), small_net)
    x, k2 = _preprocess(rgb, K, (rh, rw), pads, ratio, small_net)
    preds = [torch.rand(2, 3, small_net[0] // s, small_net[1] // s, generator=g) for s in (1, 2, 4)]
    post, k3 = _postprocess(preds, k2.clone(), small_net, pads, ratio, (h, w))
    rays, angles = ref_rays(k2, small_net)
    tpz = torch.cat([angles, 1.0 + torch.rand(2, small_net[0] * small_net[1], 1, generator=g)], dim=-1)
    arr.update(rgb=rgb.numpy(), K=K.numpy(), pre=x.numpy(), k_pre=k2.numpy(), post=post.numpy(), k_post=k3.numpy(),
               rays=rays.numpy(), angles=angles.numpy(), tpz=tpz.numpy(), xyz=ref_s2e(tpz).numpy(),
               **{f"pred{j}": p.numpy() for j, p in enumerate(preds)})
    np.savez_compressed(os.path.join(out_dir, "v1_parts.npz"), **arr)
    # ConvNeXt encoder (UniDepthV1's cnvnxtl pixel_encoder, scaled down): the reference's module on seeded weights
    from unidepth.models.backbones.convnext import ConvNeXt
    from fixture import convnext_param_shapes, make_convnext_state_dict
    depths, dims = (2, 2, 3, 2), (32, 64, 96, 128)
    enc = ConvNeXt(depths=depths, dims=dims, output_idx=[2, 4, 7, 9]).eval()
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == dict(convnext_param_shapes(depths, dims))
    big = ConvNeXt(depths=(3, 3, 27, 3), dims=(192, 384, 768, 1536), output_idx=[3, 6, 33, 36])     # config_v1_cnvnxtl.json
    assert {k: tuple(v.shape) for k, v in big.state_dict().items()} == dict(convnext_param_shapes((3, 3, 27, 3), (192, 384, 768, 1536)))
    del big
    csd = make_convnext_state_dict(depths, dims, 4)
    enc.load_state_dict(csd, strict=True)
    xin = torch.randn(2, 3, 64, 96, generator=torch.Generator().manual_seed(8))
    with torch.no_grad():
        feats, toks = enc(xin)
    ends = [1, 3, 6, 8]      # last block of each stage
    np.savez_compressed(os.path.join(out_dir, "convnext_small.npz"), x=xin.numpy(),
                        **{f"tok{j}": t.numpy() for j, t in enumerate(toks)}, **{f"feat{j}": feats[j].numpy() for j in ends})
    # also copy the configs the tests need (JSON input format, not code)
    for cfg_name in ("config_v2_vits14.json", "config_v2_vitl14.json", "config_v2_vitb14.json"):
        cfg = json.load(open(os.path.join(REF, "configs", cfg_name)))
        keep = {"model": cfg["model"],
                "data": {"augmentations": {"shape_constraints": cfg["data"]["augmentations"]["shape_constraints"]}},
                "training": {"losses": {}}}
        json.dump(keep, open(os.path.join(out_dir, cfg_name), "w"), indent=1)


if __name__ == "__main__":
    main()
