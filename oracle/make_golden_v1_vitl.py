"""Generate tests/golden/v1_vitl14_*.npz: outputs of the UNMODIFIED reference `UniDepthV1.infer` with the DINOv2 ViT-L/14
encoder (configs/config_v1_vitl14.json), on the seeded fixture of oracle/unidepth_v1_vit_oracle.py, with the same one
substitution as oracle/make_golden_v1.py (the Nystrom stand-in for the missing xformers class).  Same strides as the
ConvNeXt V1 goldens (points every 4th pixel, depth every 2nd), each file under 1 MB.

    python oracle/make_golden_v1_vitl.py       (CPU; the GPU box only reads the .npz files)
TEST INFRASTRUCTURE ONLY."""
import copy
import json
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
sys.path[:0] = [REF, os.path.join(HERE, "ref_shims"), HERE, os.path.join(HERE, "..")]

from make_golden_v1 import OracleNystrom, seeded_rgb  # noqa: E402
from unidepth_v1_vit_oracle import make_v1_vit_state_dict  # noqa: E402

CASES = [
    # name, seed, (B,H,W), with GT intrinsics, skip_camera
    ("v1_vitl14_480x640", 0, (1, 480, 640), False, False),
    ("v1_vitl14_gtK_375x1242", 1, (1, 375, 1242), True, False),
]


def main():
    warnings.simplefilter("ignore")
    torch.set_num_threads(os.cpu_count() or 1)
    import unidepth.layers.nystrom_attention as NA
    NA.NystromAttention = OracleNystrom
    from unidepth.models import UniDepthV1
    from unidepth_b200.spec_v1 import param_shapes
    out_dir = os.path.join(HERE, "..", "tests", "golden")
    cfg = json.load(open(os.path.join(REF, "configs", "config_v1_vitl14.json")))
    keep = {"model": cfg["model"], "data": {"image_shape": cfg["data"]["image_shape"]}, "training": {}}
    json.dump(keep, open(os.path.join(out_dir, "config_v1_vitl14.json"), "w"), indent=1)
    model = UniDepthV1(copy.deepcopy(cfg)).eval()
    ref_shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    mine = dict(param_shapes(cfg))
    assert ref_shapes == mine, (set(ref_shapes) ^ set(mine), [k for k in mine if k in ref_shapes and mine[k] != ref_shapes[k]])
    print("state dict:", len(ref_shapes), "keys")
    for name, seed, shape, with_k, skip in CASES:
        sd = make_v1_vit_state_dict(cfg, seed)
        model.load_state_dict(sd, strict=True)
        rgb = seeded_rgb(shape, seed)
        K = None
        if with_k:
            K = torch.tensor([[[720.0, 0.0, 610.0], [0.0, 725.0, 180.0], [0.0, 0.0, 1.0]]])
        out = model.infer(rgb, K.clone() if K is not None else None, skip_camera=skip)
        arrays = {k: v.detach().cpu().numpy() for k, v in out.items()}
        arrays["points"] = arrays["points"][:, :, ::4, ::4]
        arrays["depth"] = arrays["depth"][:, :, ::2, ::2]
        meta = dict(config="config_v1_vitl14.json", seed=seed, shape=list(shape), with_k=with_k, skip_camera=skip,
                    strides=dict(points=4, depth=2))
        if K is not None:
            arrays["K_in"] = K.numpy()
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), __meta__=json.dumps(meta), **arrays)
        d = arrays["depth"]
        print(name, "depth range", float(d.min()), float(d.max()), "K", arrays["intrinsics"][0].tolist())


if __name__ == "__main__":
    main()
