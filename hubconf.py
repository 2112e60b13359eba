"""torch.hub entry point with the reference's name and arguments (reference: hubconf.py:25-41):

    model = torch.hub.load(<this repo>, "UniDepth", version="v2", backbone="vitl14", pretrained=True, source="local")

UniDepthV2 (ViT-L/B/S) and UniDepthV1 with the ConvNeXt-L encoder load through this entry; UniDepthV1 with ViT-L runs on the
B200 path through `UniDepthV1(config_v1_vitl14.json)` but not through the hub entry yet.  The other entries the reference
lists raise NotImplementedError instead of silently loading something else."""
dependencies = ["torch"]

import json
import os

_HERE = os.path.dirname(os.path.realpath(__file__))
_SUPPORTED = {"v2": ("vitl14", "vitb14", "vits14"), "v1": ("cnvnxtl",)}
_KNOWN_ELSEWHERE = {"v1": ("vitl14",), "v2old": ("vitl14", "vits14")}


def UniDepth(version="v2", backbone="vitl14", pretrained=True):
    from unidepth_b200 import UniDepthV1, UniDepthV2

    if version not in _SUPPORTED and version not in _KNOWN_ELSEWHERE:
        raise AssertionError(f"version must be one of {sorted(set(_SUPPORTED) | set(_KNOWN_ELSEWHERE))}")
    if backbone not in _SUPPORTED.get(version, ()):
        if backbone in _KNOWN_ELSEWHERE.get(version, ()):
            if version == "v1":
                raise NotImplementedError(f"UniDepth v1 {backbone}: not available through the hub entry yet; build it with "
                                          f"UniDepthV1(json.load(open('unidepth_b200/configs/config_v1_{backbone}.json'))) "
                                          "or UniDepthV1.from_pretrained(...)")
            raise NotImplementedError(f"UniDepth {version} {backbone} is not part of the B200 inference path")
        raise AssertionError(f"backbone for version {version} must be one of {list(_SUPPORTED.get(version, ()))}")
    cfg_path = os.path.join(_HERE, "unidepth_b200", "configs", f"config_{version}_{backbone}.json")
    with open(cfg_path) as fh:
        model = (UniDepthV1 if version == "v1" else UniDepthV2)(json.load(fh))
    if pretrained:
        # same checkpoint location as the reference; needs network access (or a warm HF cache)
        import torch
        from huggingface_hub import hf_hub_download
        weights = hf_hub_download(repo_id=f"lpiccinelli/unidepth-{version}-{backbone}", filename="pytorch_model.bin",
                                  repo_type="model")
        report = model.load_state_dict(torch.load(weights, map_location="cpu"), strict=False)
        print(f"UniDepth_{version}_{backbone}: missing {report.missing_keys}, unexpected {report.unexpected_keys}")
    return model
