"""UniDepthV1 with the DINOv2 ViT-L/14 encoder (config_v1_vitl14.json) without a GPU: the parameter table against the
fixture and the reference's state dict, the oracle against the unmodified reference's `infer` outputs
(tests/golden/v1_vitl14_*.npz, oracle/make_golden_v1_vitl.py), and the packer / C schedule contract through the engine's
dry run (`udb_v1_workspace_bytes` walks every stage without touching a device)."""
import copy
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CPU = torch.device("cpu")
VIT_CASES = ["v1_vitl14_480x640", "v1_vitl14_gtK_375x1242"]


def _cfg(name="config_v1_vitl14.json"):
    return json.load(open(os.path.join(GOLDEN, name)))


def vit_case_inputs(name):
    """(config, state dict, rgb, K or None, meta, golden arrays) of one tests/golden/v1_vitl14_*.npz case."""
    from unidepth_v1_vit_oracle import make_v1_vit_state_dict
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    meta = json.loads(str(z["__meta__"]))
    cfg = _cfg(meta["config"])
    g = torch.Generator().manual_seed(4321 + meta["seed"])
    b, h, w = meta["shape"]
    rgb = torch.randint(0, 256, (b, 3, h, w), dtype=torch.uint8, generator=g)
    K = torch.from_numpy(z["K_in"]) if meta["with_k"] else None
    return cfg, make_v1_vit_state_dict(cfg, meta["seed"]), rgb, K, meta, z


def test_param_shapes_match_fixture_and_reference():
    """The golden's config is the reference's own (oracle/make_golden_v1_vitl.py asserts param_shapes equals the live
    reference state dict, 698 keys); the fixture fills exactly those tensors."""
    from unidepth_b200.spec_v1 import V1Spec, param_shapes
    from unidepth_v1_vit_oracle import make_v1_vit_state_dict
    cfg = _cfg()
    shapes = param_shapes(cfg)
    assert len(shapes) == 698
    assert {k: tuple(v.shape) for k, v in make_v1_vit_state_dict(cfg, 0).items()} == dict(shapes)
    assert shapes["pixel_encoder.pos_embed"] == (1, 1 + 37 * 37, 1024) and shapes["pixel_encoder.register_tokens"] == (1, 1, 1024)
    assert shapes["pixel_decoder.input_adapter.input_adapters.3.1.weight"] == (512, 1024)
    s = V1Spec(cfg)
    assert s.depths == (5, 7, 6, 6) and s.dims == (1024,) * 4 and s.cls_dims == (1024,) * 4
    # the package's config is the golden's
    assert json.load(open(os.path.join(ROOT, "unidepth_b200", "configs", "config_v1_vitl14.json"))) == cfg
    for bad in ([5, 12, 18], [5, 12, 12, 24], [5, 12, 18, 23]):
        c = copy.deepcopy(cfg)
        c["model"]["pixel_encoder"]["output_idx"] = bad
        with pytest.raises(NotImplementedError):
            V1Spec(c)


def test_pos_embed_offset_uses_the_scale_factor():
    """interpolate_offset 0.1 samples the 37x37 table at other positions than the size form would."""
    from unidepth_v1_vit_oracle import interpolate_pos_embed
    g = torch.Generator().manual_seed(0)
    pos = torch.randn(1, 1 + 37 * 37, 8, generator=g)
    a, b = interpolate_pos_embed(pos, 33, 44, 0.1), interpolate_pos_embed(pos, 33, 44)
    assert a.shape == b.shape == (1, 1 + 33 * 44, 8)
    assert torch.equal(a[:, 0], pos[:, 0]) and (a - b).abs().max().item() > 1e-3


@pytest.mark.parametrize("name", VIT_CASES)
def test_vit_oracle_matches_reference_golden(name):
    import unidepth_v1_vit_oracle as OV
    cfg, sd, rgb, K, meta, z = vit_case_inputs(name)
    out = OV.infer_v1_vit(sd, cfg, rgb, K, skip_camera=meta["skip_camera"])
    assert set(out) == {"intrinsics", "points", "depth"}
    for k in ("intrinsics", "depth", "points"):
        ref = torch.from_numpy(z[k])
        s = meta["strides"].get(k, 1)
        got = out[k][:, :, ::s, ::s] if k in ("depth", "points") else out[k]
        assert got.shape == ref.shape, (k, got.shape, ref.shape)
        floor = 0.1 * ref.abs().mean().item()
        err = ((got - ref).abs() / ref.abs().clamp(min=floor)).max().item()
        print(k, "max rel err", err)
        # depth and intrinsics to 2e-6; the points add the back-projection's float trigonometry on top (measured 4.7e-6)
        assert err < (1e-5 if k == "points" else 2e-6), (k, err)


def _vit_model():
    from unidepth_b200 import UniDepthV1
    return UniDepthV1(copy.deepcopy(_cfg())).eval()


def _engine(m, tensors, S, heads=16):
    from unidepth_b200 import _cabi
    h = C.c_void_p()
    _cabi.check(_cabi.lib().udb_v1_create_vit(C.byref(m._engine_config()), heads, C.byref(h)), "udb_v1_create_vit")
    m._register(h, tensors, S)
    return h


def test_vit_packer_and_schedule_agree():
    from unidepth_b200 import _cabi
    lib = _cabi.lib()
    m = _vit_model()
    T, S = m._pack_tensors(CPU)
    assert T["pos"].shape == (1 + 33 * 44, 1024) and T["patch_w"].shape == (1024, 640)
    assert T["tokens_pos"].shape == (4 * 33 * 44, 512)
    h = _engine(m, T, S)
    try:
        for B in (1, 4):
            for H, W in ((480, 640), (375, 1242), (1000, 400)):
                assert lib.udb_v1_workspace_bytes(h, B, H, W) > 0, (B, H, W, lib.udb_last_error().decode())
        assert lib.udb_v1_workspace_bytes(h, 4, 480, 640) > lib.udb_v1_workspace_bytes(h, 1, 480, 640)
    finally:
        lib.udb_v1_destroy(h)
    # one operand short: reported by name
    for name in ["patch_w", "pos", "cls", "blocks.0.qkv_w", "blocks.23.ls2", "tokens_pos", "adapt.3.w", "up2.conv_w"]:
        h = _engine(m, {k: v for k, v in T.items() if k != name}, S)
        try:
            assert lib.udb_v1_workspace_bytes(h, 1, 480, 640) == 0
            assert name in lib.udb_last_error().decode(), (name, lib.udb_last_error().decode())
        finally:
            lib.udb_v1_destroy(h)
    # a transposed fc1 weight or a position table for another grid is refused, not read with the wrong shape
    for name in ("blocks.0.fc1_w", "pos"):
        bad = dict(T)
        bad[name] = T[name].t().contiguous() if name != "pos" else T[name][:-44].contiguous()
        h = _engine(m, bad, S)
        try:
            assert lib.udb_v1_workspace_bytes(h, 1, 480, 640) == 0
            assert name in lib.udb_last_error().decode(), lib.udb_last_error().decode()
        finally:
            lib.udb_v1_destroy(h)


def test_create_vit_rejects_bad_heads_or_width():
    from unidepth_b200 import _cabi
    lib = _cabi.lib()
    m = _vit_model()
    for heads, dims, net in ((15, None, None), (8, None, None), (0, None, None), (16, (1024, 1024, 1024, 768), None),
                             (16, (1000,) * 4, None), (16, None, (462, 620))):
        cfg = m._engine_config()
        if dims:
            for i in range(4):
                cfg.dims[i] = dims[i]
        if net:
            cfg.net_h, cfg.net_w = net
        h = C.c_void_p()
        assert lib.udb_v1_create_vit(C.byref(cfg), heads, C.byref(h)) != 0, (heads, dims, net)
        assert b"udb_v1_create_vit" in lib.udb_last_error()


def test_convnext_v1_dry_run_unchanged():
    """The ConvNeXt-L schedule sizes its workspace exactly as before the ViT encoder was added."""
    from unidepth_b200 import UniDepthV1, _cabi
    lib = _cabi.lib()
    m = UniDepthV1(_cfg("config_v1_cnvnxtl.json")).eval()
    T, S = m._pack_tensors(CPU)
    h = C.c_void_p()
    _cabi.check(lib.udb_v1_create(C.byref(m._engine_config()), C.byref(h)), "udb_v1_create")
    try:
        m._register(h, T, S)
        assert lib.udb_v1_workspace_bytes(h, 1, 480, 640) == 142151424
        assert lib.udb_v1_workspace_bytes(h, 4, 480, 640) == 568405504
        assert lib.udb_v1_workspace_bytes(h, 16, 480, 640) == 2273422336
    finally:
        lib.udb_v1_destroy(h)


def test_v1_vit_load_state_dict_and_from_pretrained(tmp_path):
    """Reference checkpoint keys load strictly; from_pretrained reads config.json + weights from a directory."""
    from unidepth_b200 import UniDepthV1
    from unidepth_v1_vit_oracle import make_v1_vit_state_dict
    cfg = _cfg()
    sd = make_v1_vit_state_dict(cfg, 0)
    m = UniDepthV1(copy.deepcopy(cfg))
    m.load_state_dict(sd, strict=True)
    m.save_pretrained(str(tmp_path))
    m2 = UniDepthV1.from_pretrained(str(tmp_path))
    assert m2.spec.vit
    for k, v in m.state_dict().items():
        assert torch.equal(v, m2.state_dict()[k]), k
