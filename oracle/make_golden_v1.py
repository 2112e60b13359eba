"""Generate tests/golden/v1_*.npz: outputs of the UNMODIFIED reference `UniDepthV1.infer` (imported from /root/reference
through oracle/ref_shims) on the seeded fixture, with ONE substitution: xformers' NystromAttention, which is not
installed here, is replaced by the restatement in oracle/unidepth_v1_oracle.py (`nystrom_attention`), so the goldens pin
everything except that function's arithmetic ("parity unpinned" for Nystrom, see that module's header).

    python oracle/make_golden_v1.py            (CPU container; the GPU box only reads the .npz files)
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

from fixture import make_v1_state_dict  # noqa: E402
import unidepth_v1_oracle as O1  # noqa: E402


class OracleNystrom:
    """Stand-in with xformers' call signature: q, k, v [b, n, h, d] -> [b, n, h, d]."""

    def __init__(self, num_landmarks=128, num_heads=1, dropout=0.0, **kw):
        self.num_landmarks = num_landmarks

    def __call__(self, q, k, v, key_padding_mask=None, **kw):
        o = O1.nystrom_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), self.num_landmarks)
        return o.transpose(1, 2)


def seeded_rgb(shape, seed):
    g = torch.Generator().manual_seed(4321 + seed)
    b, h, w = shape
    return torch.randint(0, 256, (b, 3, h, w), dtype=torch.uint8, generator=g)


CASES = [
    # name, seed, (B,H,W), with GT intrinsics, skip_camera
    ("v1_cnvnxtl_480x640", 0, (1, 480, 640), False, False),
    ("v1_cnvnxtl_gtK_375x1242", 1, (1, 375, 1242), True, False),
]


def main():
    warnings.simplefilter("ignore")
    import unidepth.layers.nystrom_attention as NA
    NA.NystromAttention = OracleNystrom
    from unidepth.models import UniDepthV1
    from unidepth_b200.spec_v1 import param_shapes
    out_dir = os.path.join(HERE, "..", "tests", "golden")
    cfg = json.load(open(os.path.join(REF, "configs", "config_v1_cnvnxtl.json")))
    keep = {"model": cfg["model"], "data": {"image_shape": cfg["data"]["image_shape"]}, "training": {}}
    json.dump(keep, open(os.path.join(out_dir, "config_v1_cnvnxtl.json"), "w"), indent=1)
    model = UniDepthV1(copy.deepcopy(cfg)).eval()
    ref_shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    mine = dict(param_shapes(cfg))
    assert ref_shapes == mine, (set(ref_shapes) ^ set(mine), [k for k in mine if k in ref_shapes and mine[k] != ref_shapes[k]])
    for name, seed, shape, with_k, skip in CASES:
        sd = make_v1_state_dict(cfg, seed)
        model.load_state_dict(sd, strict=True)
        rgb = seeded_rgb(shape, seed)
        K = None
        if with_k:
            K = torch.tensor([[[720.0, 0.0, 610.0], [0.0, 725.0, 180.0], [0.0, 0.0, 1.0]]])
        out = model.infer(rgb, K.clone() if K is not None else None, skip_camera=skip)
        arrays = {k: v.detach().cpu().numpy() for k, v in out.items()}
        # every 4th pixel of the points and every 2nd of the depth keep each file under 1 MB
        arrays["points"] = arrays["points"][:, :, ::4, ::4]
        arrays["depth"] = arrays["depth"][:, :, ::2, ::2]
        meta = dict(config="config_v1_cnvnxtl.json", seed=seed, shape=list(shape), with_k=with_k, skip_camera=skip,
                    strides=dict(points=4, depth=2))
        if K is not None:
            arrays["K_in"] = K.numpy()
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), __meta__=json.dumps(meta), **arrays)
        d = arrays["depth"]
        print(name, "depth range", float(d.min()), float(d.max()), "K", arrays["intrinsics"][0].tolist())


if __name__ == "__main__":
    main()
