"""Pin the oracle: the torch-fp32 restatement (oracle/unidepth_oracle.py) must reproduce the
outputs of the unmodified reference stored in tests/golden/*.npz (made by oracle/make_golden.py).
Both are fp32 on CPU, so the tolerance is only summation-order noise."""
import json
import os

import numpy as np
import pytest
import torch

import unidepth_oracle as O
from fixture import make_state_dict

CASES = ["vits_120x160", "vits_pad_96x288_rl3", "vitb_112x160", "vitl_480x640"]


def subsample_like_golden(out, meta):
    """Apply the sub-sampling oracle/make_golden.py used when it stored the big maps."""
    st = {"depth": 1, "spatial": 1, "depth_features": 4, **meta.get("strides", {})}
    res = {}
    for k, v in out.items():
        if k == "depth_features":
            res[k] = v[:, ::st["depth_features"]]
        elif k == "depth":
            res[k] = v[:, :, ::st["depth"], ::st["depth"]]
        elif k in ("confidence", "radius", "points", "rays"):
            res[k] = v[:, :, ::st["spatial"], ::st["spatial"]]
        else:
            res[k] = v
    return res


def _rgb(shape, seed):
    g = torch.Generator().manual_seed(1234 + seed)
    b, h, w = shape
    return torch.randint(0, 256, (b, 3, h, w), dtype=torch.uint8, generator=g)


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name, golden_dir):
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    meta = json.loads(str(z["__meta__"]))
    cfg = json.load(open(os.path.join(golden_dir, meta["config"])))
    sd = make_state_dict(cfg, meta["seed"])
    out = O.infer_v2(sd, cfg, _rgb(meta["shape"], meta["seed"]), resolution_level=meta["resolution_level"])
    assert set(out) == {"confidence", "intrinsics", "radius", "depth", "points", "rays", "depth_features"}
    out = subsample_like_golden(out, meta)
    for k, v in out.items():
        ref = torch.from_numpy(z[k])
        got = v
        assert got.shape == ref.shape, (k, got.shape, ref.shape)
        # error relative to |ref|, floored at 10% of the tensor's mean magnitude so that
        # zero-crossings of signed tensors (points.x, depth_features) do not blow it up
        floor = 0.1 * ref.abs().mean().item()
        err = ((got - ref).abs() / ref.abs().clamp(min=floor)).max().item()
        print(k, "max rel err", err)
        assert err < 3e-4, (k, err)
    rel_depth = ((out["depth"] - torch.from_numpy(z["depth"])).abs() / torch.from_numpy(z["depth"])).max().item()
    assert rel_depth < 5e-5, rel_depth
    kk = out["intrinsics"]
    kr = torch.from_numpy(z["intrinsics"])
    for (i, j) in ((0, 0), (1, 1), (0, 2), (1, 2)):
        assert ((kk[:, i, j] - kr[:, i, j]).abs() / kr[:, i, j].abs()).max().item() < 1e-5


CAMERA_CASES = ["vits_camK_120x160", "vits_campinhole_pad_96x288_rl3", "vits_cameucm_pad_200x70_rl0"]


@pytest.mark.parametrize("name", CAMERA_CASES)
def test_oracle_gt_camera_branch_matches_reference_golden(name, golden_dir):
    """infer(rgb, camera=...) of the unmodified reference (oracle/make_golden_camera_infer.py): K tensor, Pinhole object with
    padding + resolution level, a non-pinhole (EUCM) object on a portrait image.  The camera objects handed to the oracle
    are this repo's own classes (unidepth_b200/camera.py), so this also checks them inside the whole forward."""
    from unidepth_b200 import camera as C
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    meta = json.loads(str(z["__meta__"]))
    cfg = json.load(open(os.path.join(golden_dir, meta["config"])))
    sd = make_state_dict(cfg, meta["seed"])
    kind, params = meta["camera"]["kind"], meta["camera"]["params"]
    if kind == "K":
        cam = torch.tensor([[[params[0], 0.0, params[2]], [0.0, params[1], params[3]], [0.0, 0.0, 1.0]]])
    else:
        cam = getattr(C, kind)(params=torch.tensor([params], dtype=torch.float32))
    out = O.infer_v2(sd, cfg, _rgb(meta["shape"], meta["seed"]), resolution_level=meta["resolution_level"], camera=cam)
    out = subsample_like_golden(out, meta)
    for k, v in out.items():
        ref = torch.from_numpy(z[k])
        assert v.shape == ref.shape, (k, v.shape, ref.shape)
        floor = 0.1 * ref.abs().mean().item()
        err = ((v - ref).abs() / ref.abs().clamp(min=floor)).max().item()
        print(name, k, "max rel err", err)
        assert err < 3e-4, (k, err)
    assert (out["rays"] - torch.from_numpy(z["rays"])).abs().max().item() < 2e-6       # the GT rays themselves
    if kind != "K":      # the oracle works on a copy, like the product (the reference mutates the caller's object)
        assert torch.equal(cam.params, torch.tensor([params], dtype=torch.float32))


def test_shape_arithmetic_examples():
    # SURVEY.md section 8 a1 (values produced by the reference functions)
    assert O.get_resize_factor((480, 640), (2e5, 6e5))[1] == (490, 644)
    assert O.get_resize_factor((1024, 1536), (2e5, 6e5))[1] == (644, 952)
    pads, shp = O.get_paddings((480, 1600), (0.5, 2.5))
    assert pads == (0, 0, 80, 80) and shp == (640, 1600)
    pads, shp = O.get_paddings((1000, 400), (0.5, 2.5))
    assert pads == (50, 50, 0, 0) and shp == (1000, 500)
    levels = {0: (434, 574), 2: (490, 644), 5: (560, 742), 9: (658, 868)}
    for lvl, hw in levels.items():
        assert O.get_resize_factor((480, 640), O.resolve_pixel_bounds((2e5, 6e5), lvl))[1] == hw


def test_sh81_recurrence_matches_reference_polynomials(golden_dir):
    """oracle/sh81.py (definition + recurrences) vs the reference's expanded degree-8 polynomials
    (unidepth/utils/sht.py:833-1393) on seeded unit vectors: the oracle of V1's ray embedding basis."""
    from sh81 import rsh_cart
    z = np.load(os.path.join(golden_dir, "sh81.npz"))
    xyz, ref = torch.from_numpy(z["xyz"]), torch.from_numpy(z["rsh"])
    got = rsh_cart(xyz)
    assert got.shape == ref.shape == (256, 81)
    assert float((got - ref).abs().max()) < 5e-8          # the reference's literals carry ~15 digits
    assert float((rsh_cart(xyz.float()) - ref.float()).abs().max()) < 1e-5


def test_v1_host_pieces_match_reference(golden_dir):
    """oracle/unidepth_v1_parts.py vs the reference's V1 helpers (unidepthv1.py:30-94, geometric.py:13-73):
    fixed-shape resize / pad arithmetic (incl. the reference's benchmark shape 480x640 -> 462x616),
    pre/post-processing with the K updates, ray generation, (theta, phi, z) -> xyz."""
    import unidepth_v1_parts as V
    z = np.load(os.path.join(golden_dir, "v1_parts.npz"))
    net = (462, 616)
    for i, (h, w) in enumerate(z["cases"]):
        (rh, rw), ratio = V.v1_shapes((int(h), int(w)), net)
        assert [rh, rw, *V.v1_paddings((rh, rw), net)] == list(z[f"shape{i}"]) and ratio == float(z[f"ratio{i}"])
    assert list(z["shape0"]) == [462, 616, 0, 0, 0, 0]
    rgb, K = torch.from_numpy(z["rgb"]), torch.from_numpy(z["K"])
    small_net = (42, 56)
    (rh, rw), ratio = V.v1_shapes(tuple(rgb.shape[-2:]), small_net)
    pads = V.v1_paddings((rh, rw), small_net)
    x, k2 = V.v1_preprocess(rgb, K, (rh, rw), pads, ratio)
    assert torch.equal(x, torch.from_numpy(z["pre"])) and torch.allclose(k2, torch.from_numpy(z["k_pre"]), rtol=0, atol=0)
    preds = [torch.from_numpy(z[f"pred{j}"]) for j in range(3)]
    post, k3 = V.v1_postprocess(preds, k2, small_net, pads, ratio, tuple(rgb.shape[-2:]))
    assert torch.allclose(post, torch.from_numpy(z["post"]), atol=1e-6, rtol=0)
    assert torch.allclose(k3, torch.from_numpy(z["k_post"]), atol=1e-4, rtol=1e-6)
    rays, angles = V.generate_rays(k2, small_net)
    assert torch.allclose(rays, torch.from_numpy(z["rays"]), atol=2e-6, rtol=0)
    assert torch.allclose(angles, torch.from_numpy(z["angles"]), atol=2e-6, rtol=0)
    xyz = V.spherical_zbuffer_to_euclidean(torch.from_numpy(z["tpz"]))
    assert torch.allclose(xyz, torch.from_numpy(z["xyz"]), atol=0, rtol=0)


def test_convnext_encoder_restatement_matches_reference_module(golden_dir):
    """oracle/convnext_oracle.py vs the reference's ConvNeXt module (backbones/convnext.py, run by
    oracle/make_golden.py with the timm stand-ins) on a scaled-down encoder: every block's mean token and the
    last feature map of each stage."""
    from convnext_oracle import convnext_encoder
    from fixture import convnext_param_shapes, make_convnext_state_dict
    z = np.load(os.path.join(golden_dir, "convnext_small.npz"))
    depths, dims = (2, 2, 3, 2), (32, 64, 96, 128)
    sd = make_convnext_state_dict(depths, dims, 4)
    feats, toks = convnext_encoder(sd, torch.from_numpy(z["x"]), depths)
    assert len(feats) == sum(depths)
    for j, t in enumerate(toks):
        assert torch.allclose(t, torch.from_numpy(z[f"tok{j}"]), atol=2e-5, rtol=1e-5), j
    for j in (1, 3, 6, 8):
        ref = torch.from_numpy(z[f"feat{j}"])
        assert feats[j].shape == ref.shape and float((feats[j] - ref).abs().max()) < 5e-5, j
    # the benchmark configuration's parameter census (config_v1_cnvnxtl.json: ConvNeXt-L, 196.2 M parameters)
    n = sum(int(np.prod(s)) for s in convnext_param_shapes((3, 3, 27, 3), (192, 384, 768, 1536)).values())
    assert 196.0e6 < n < 196.5e6


V1_CASES = ["v1_cnvnxtl_480x640", "v1_cnvnxtl_gtK_375x1242"]


def v1_case_inputs(golden_dir, name):
    """(config, state dict, rgb, K or None, meta, golden arrays) of one tests/golden/v1_*.npz case."""
    from fixture import make_v1_state_dict
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    meta = json.loads(str(z["__meta__"]))
    cfg = json.load(open(os.path.join(golden_dir, meta["config"])))
    g = torch.Generator().manual_seed(4321 + meta["seed"])
    b, h, w = meta["shape"]
    rgb = torch.randint(0, 256, (b, 3, h, w), dtype=torch.uint8, generator=g)
    K = torch.from_numpy(z["K_in"]) if meta["with_k"] else None
    return cfg, make_v1_state_dict(cfg, meta["seed"]), rgb, K, meta, z


@pytest.mark.parametrize("name", V1_CASES)
def test_v1_oracle_matches_reference_golden(name, golden_dir):
    """UniDepthV1 (ConvNeXt-L, config_v1_cnvnxtl.json) oracle vs the unmodified reference's `infer` outputs
    (oracle/make_golden_v1.py; the one substitution -- Nystrom attention -- is described there)."""
    import unidepth_v1_oracle as O1
    cfg, sd, rgb, K, meta, z = v1_case_inputs(golden_dir, name)
    out = O1.infer_v1(sd, cfg, rgb, K, skip_camera=meta["skip_camera"])
    assert set(out) == {"intrinsics", "points", "depth"}
    for k in ("intrinsics", "depth", "points"):
        ref = torch.from_numpy(z[k])
        s = meta["strides"].get(k, 1)
        got = out[k][:, :, ::s, ::s] if k in ("depth", "points") else out[k]
        assert got.shape == ref.shape, (k, got.shape, ref.shape)
        floor = 0.1 * ref.abs().mean().item()
        err = ((got - ref).abs() / ref.abs().clamp(min=floor)).max().item()
        print(k, "max rel err", err)
        assert err < 5e-5, (k, err)


def test_nystrom_restatement_properties():
    """The Nystrom restatement has no reference output to be pinned to (xformers absent: "parity unpinned"), so check
    what the published algorithm guarantees: with as many landmarks as keys it IS softmax attention, rows of the
    reconstruction are close to exact attention for smooth inputs, and the Newton-Schulz iteration inverts a
    well-conditioned row-stochastic matrix."""
    import unidepth_v1_oracle as O1
    g = torch.Generator().manual_seed(3)
    q, k, v = (torch.randn(2, 3, 128, 64, generator=g) for _ in range(3))
    exact = torch.softmax(q @ k.transpose(-1, -2) / 8.0, -1) @ v
    assert torch.allclose(O1.nystrom_attention(q, k, v, 128), exact, atol=1e-6)
    m = torch.softmax(torch.randn(4, 128, 128, generator=g) * 0.1 + 8 * torch.eye(128), -1)
    inv = O1._iterative_pinv(m, 12)
    assert (inv @ m - torch.eye(128)).abs().max() < 1e-3
    # ragged segment means: 300 rows into 128 landmarks = 84 segments of 2 rows + 44 of 3
    x = torch.arange(300.0).reshape(1, 1, 300, 1)
    lm = O1._avg_landmarks(x, 128)[0, 0, :, 0]
    assert lm[0] == 0.5 and lm[83] == 166.5 and lm[84] == 169.0 and lm[-1] == 298.0


def test_nystrom_restatement_matches_independent_implementation():
    """Second anchor for the one "parity unpinned" function: HuggingFace transformers ships the Nystromformer authors'
    own implementation of the same published algorithm (segment-mean landmarks, three softmax kernels, 6 Newton-Schulz
    iterations).  With its skip-connection convolution zeroed and the exact 1/||K||_1 initialisation (xformers'
    default `pinverse_original_init=False`) it must agree with `nystrom_attention` to fp32 rounding wherever the
    sequence length is a multiple of the landmark count (HF supports nothing else).  xformers' own arithmetic stays
    unpinned only for the ragged pooling (checked by hand in the test above) and the s == landmarks shortcut."""
    pytest.importorskip("transformers")
    from transformers import NystromformerConfig
    from transformers.models.nystromformer.modeling_nystromformer import NystromformerSelfAttention
    import unidepth_v1_oracle as O1
    torch.manual_seed(0)
    # (heads, head_dim, tokens, landmarks, input scale): the V1 decoder's 1/8-scale block shape, a long peaky one, a small one
    for heads, d, s, m, scale in ((4, 64, 1024, 128, 1.0), (8, 64, 2304, 128, 3.0), (2, 32, 640, 64, 2.0)):
        cfg = NystromformerConfig(hidden_size=heads * d, num_attention_heads=heads, num_landmarks=m,
                                  segment_means_seq_len=s, conv_kernel_size=3, attention_probs_dropout_prob=0.0)
        att = NystromformerSelfAttention(cfg).eval()
        att.init_option = "exact"            # any value but "original": per-matrix 1/||K||_1, as in xformers
        att.conv.weight.data.zero_()         # xformers' NystromAttention default: no convolutional skip connection
        x = torch.randn(2, s, heads * d) * scale
        with torch.no_grad():
            want = att(x)[0]
            split = lambda t: t.view(2, s, heads, d).transpose(1, 2)
            got = O1.nystrom_attention(split(att.query(x)), split(att.key(x)), split(att.value(x)), m)
        got = got.transpose(1, 2).reshape(2, s, heads * d)
        err = (got - want).abs().max().item()
        print(f"nystrom vs HF Nystromformer heads={heads} d={d} s={s} m={m}: max abs {err:.2e} (mean |out| {want.abs().mean():.3f})")
        assert err < 5e-6, err
