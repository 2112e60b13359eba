"""Generate tests/golden/vits_cam*.npz: `UniDepthV2.infer(rgb, camera=...)` of the UNMODIFIED reference (GT-camera
branch, unidepthv2.py:267-303,361-362; decoder.py:400) for a K tensor, a Pinhole object and a non-pinhole camera object,
with and without padding / resolution level.  Pins the oracle's GT-camera branch (tests/test_oracle_golden.py).

Run here (CPU container, has /root/reference):   python oracle/make_golden_camera_infer.py
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

from fixture import make_state_dict  # noqa: E402
from make_golden import seeded_rgb  # noqa: E402

# name, config, seed, (B,H,W), resolution_level, camera = (kind, params): kind "K" = (...,3,3) tensor from fx fy cx cy,
# otherwise a reference camera class name (utils/camera.py) with its parameter vector; spatial stride of the stored
# confidence / radius / points / rays (2 keeps the larger image under 1 MB)
CASES = [
    ("vits_camK_120x160", "config_v2_vits14.json", 5, (1, 120, 160), None, ("K", [125.0, 127.0, 79.0, 61.5]), 1),
    ("vits_campinhole_pad_96x288_rl3", "config_v2_vits14.json", 6, (1, 96, 288), 3, ("Pinhole", [150.0, 148.0, 140.0, 50.0]), 2),
    ("vits_cameucm_pad_200x70_rl0", "config_v2_vits14.json", 7, (1, 200, 70), 0, ("EUCM", [60.0, 61.0, 36.0, 98.0, 0.6, 1.1]), 1),
]


def main():
    warnings.simplefilter("ignore")
    from unidepth.models import UniDepthV2
    import unidepth.utils.camera as C
    out_dir = os.path.join(HERE, "..", "tests", "golden")
    for name, cfg_name, seed, shape, level, (kind, params), ss in CASES:
        cfg = json.load(open(os.path.join(REF, "configs", cfg_name)))
        model = UniDepthV2(copy.deepcopy(cfg)).eval()
        model.load_state_dict(make_state_dict(cfg, seed), strict=True)
        if level is not None:
            model.resolution_level = level
        p = torch.tensor([params], dtype=torch.float32)
        if kind == "K":
            cam = torch.tensor([[[params[0], 0.0, params[2]], [0.0, params[1], params[3]], [0.0, 0.0, 1.0]]])
        else:
            cam = getattr(C, kind)(params=p.clone())
        out = model.infer(seeded_rgb(shape, seed), cam)
        arrays = {k: v.detach().cpu().numpy() for k, v in out.items()}
        arrays["depth_features"] = arrays["depth_features"][:, ::4]
        for k in ("confidence", "radius", "points", "rays"):
            arrays[k] = arrays[k][:, :, ::ss, ::ss]
        meta = dict(config=cfg_name, seed=seed, shape=list(shape), resolution_level=level, camera=dict(kind=kind, params=params),
                    strides=dict(depth=1, spatial=ss, depth_features=4))
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), __meta__=json.dumps(meta), **arrays)
        d = arrays["depth"]
        print(name, "depth range", float(d.min()), float(d.max()), "K out", arrays["intrinsics"][0].tolist())


if __name__ == "__main__":
    main()
