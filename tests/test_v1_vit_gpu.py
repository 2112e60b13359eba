"""UniDepthV1 with the DINOv2 ViT-L/14 encoder on the GPU: the two ViT-only kernels (14x14 pre-processing, the tap after each
block) against PyTorch, and the whole `infer` (udb_infer_v1 through udb_v1_create_vit) against the unmodified reference's
outputs (tests/golden/v1_vitl14_*.npz) and the oracle."""
import copy
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
f16, f32 = torch.float16, torch.float32


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def test_v1_preprocess_vit_patches():
    """14x14 patch rows [B*33*44, 640] vs the oracle's v1_preprocess + F.unfold(k=14, s=14); columns 588.. stay zero."""
    from unidepth_b200 import _cabi as cabi
    import unidepth_v1_parts as P1
    lib = cabi.lib()
    dev = _dev()
    g = torch.Generator().manual_seed(1)
    mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
    for (H, W) in ((480, 640), (375, 1242), (1000, 400), (231, 308)):
        rgb = torch.randint(0, 256, (2, 3, H, W), dtype=torch.uint8, generator=g)
        (rh, rw), ratio = P1.v1_shapes((H, W), (462, 616))
        pads = P1.v1_paddings((rh, rw), (462, 616))
        xr, _ = P1.v1_preprocess((rgb.float() / 255 - mean) / std, None, (rh, rw), pads, ratio)
        ref = F.unfold(xr, kernel_size=14, stride=14).transpose(1, 2).reshape(-1, 588)      # (c, py, px) columns
        patches = torch.full((2 * 33 * 44, 640), float("nan"), device=dev, dtype=f16)
        p = cabi.V1Preprocess()
        rd = rgb.to(dev)
        p.rgb, p.rgb_is_u8, p.scale255, p.normalize, p.B, p.H, p.W = _p(rd), 1, 1, 1, 2, H, W
        p.rh, p.rw, p.pad_l, p.pad_t, p.net_h, p.net_w, p.patches = rh, rw, pads[0], pads[2], 462, 616, _p(patches)
        cabi.check(lib.udb_v1_preprocess_vit(C.byref(p), _st()), "v1_preprocess_vit")
        got = patches[:, :588].float().cpu()
        err = ((got - ref).abs().max() / ref.abs().max()).item()
        print(f"v1_preprocess_vit {H}x{W}: max rel err {err:.2e}")
        assert err < 2e-3 and patches[:, 588:].abs().max().item() == 0


def test_vit_tap_kernel_bit_exact():
    """dst = f16(x[:,1:] + x[:,:1]) on the first block, running max after; the cls row copied in f32; odd B / T."""
    from unidepth_b200 import _cabi as cabi
    lib = cabi.lib()
    dev = _dev()
    g = torch.Generator().manual_seed(2)
    for B, T, D in ((1, 1453, 1024), (3, 37, 384), (5, 2, 8), (2, 1001, 768)):
        dst = torch.empty(B, T - 1, D, device=dev, dtype=f16)
        ref = None
        for blk in range(3):
            x = (torch.randn(B, T, D, generator=g) * (3.0 + blk)).to(dev)
            cls = torch.full((B, D), float("nan"), device=dev) if blk == 2 else None
            cabi.check(lib.udb_vit_tap_f16(_p(x), _p(dst), _p(cls), B, T, D, int(blk == 0), _st()), "vit_tap")
            cur = (x[:, 1:] + x[:, :1]).half()
            ref = cur if ref is None else torch.maximum(ref, cur)
            assert torch.equal(dst, ref), (B, T, D, blk)
            if cls is not None:
                assert torch.equal(cls, x[:, 0])
    x = torch.zeros(1, 4, 12, device=dev)
    assert lib.udb_vit_tap_f16(_p(x), _p(x), None, 1, 4, 12, 1, _st()) != 0          # D % 8


def _model(cfg, sd):
    from unidepth_b200 import UniDepthV1
    m = UniDepthV1(copy.deepcopy(cfg))
    m.load_state_dict(sd, strict=True)
    return m.to("cuda:0").eval()


# measured on the B200 (profiles/r03_v1_vitl_parity_gpu.log), asserted with a 1.5x margin: (depth ARel, depth max-rel,
# intrinsics rel); all under the ceilings of 1e-3 (depth ARel) and 5e-4 (intrinsics)
MEASURED = {
    "golden_v1_vitl14_480x640": (2.090e-4, 8.671e-4, 5.242e-5),
    "golden_v1_vitl14_gtK_375x1242": (4.048e-4, 1.053e-3, 2.499e-4),
    "oracle_v1_vitl14_480x640": (2.092e-4, 9.096e-4, 5.242e-5),
    "skip_camera_480x640": (1.736e-4, 7.581e-4, 1e-6),
}


def _check(out, ref_depth, ref_K, ref_pts, tag, pts_stride=1, depth_stride=1):
    d = out["depth"].float().cpu()[:, :, ::depth_stride, ::depth_stride]
    rel = (d - ref_depth).abs() / ref_depth
    k = out["intrinsics"].cpu()
    kerr = max(((k[:, i, j] - ref_K[:, i, j]).abs() / ref_K[:, i, j].abs()).max().item() for i, j in ((0, 0), (1, 1), (0, 2), (1, 2)))
    pts = out["points"].float().cpu()[:, :, ::pts_stride, ::pts_stride]
    perr = ((pts - ref_pts).abs() / ref_pts.abs().clamp(min=0.1 * ref_pts.abs().mean())).mean().item()
    print(f"V1VITPARITY {tag}: depth ARel {rel.mean().item():.3e} max {rel.max().item():.3e}; intrinsics rel {kerr:.3e}; "
          f"points mean rel {perr:.3e}")
    m = MEASURED[tag]
    assert rel.mean().item() < 1.5 * m[0] and rel.max().item() < 1.5 * m[1] and kerr < 1.5 * m[2], (tag, rel.mean().item(),
                                                                                                     rel.max().item(), kerr)
    assert perr < 5e-3


@pytest.mark.parametrize("name", ["v1_vitl14_480x640", "v1_vitl14_gtK_375x1242"])
def test_v1_vit_infer_against_reference_golden(name):
    _dev()
    from test_v1_vit_cpu import vit_case_inputs
    cfg, sd, rgb, K, meta, z = vit_case_inputs(name)
    m = _model(cfg, sd)
    out = m.infer(rgb, K, skip_camera=meta["skip_camera"])
    assert set(out) == {"intrinsics", "points", "depth"}
    _check(out, torch.from_numpy(z["depth"]), torch.from_numpy(z["intrinsics"]), torch.from_numpy(z["points"]), "golden_" + name,
           meta["strides"]["points"], meta["strides"]["depth"])
    # graph replay equals eager bit for bit
    again = m.infer(rgb, K, skip_camera=meta["skip_camera"])
    assert all(torch.equal(again[k], out[k]) for k in out)
    m.use_cuda_graph = False
    eager = m.infer(rgb, K, skip_camera=meta["skip_camera"])
    assert all(torch.equal(eager[k], out[k]) for k in out)


def test_v1_vit_oracle_batch_and_skip_camera():
    _dev()
    import unidepth_v1_vit_oracle as OV
    from test_v1_vit_cpu import vit_case_inputs
    cfg, sd, rgb, _, meta, z = vit_case_inputs("v1_vitl14_480x640")
    m = _model(cfg, sd)
    one = m.infer(rgb)
    ref = OV.infer_v1_vit(sd, copy.deepcopy(cfg), rgb)
    _check(one, ref["depth"], ref["intrinsics"], ref["points"], "oracle_v1_vitl14_480x640")
    # the golden image inside a batch of 16 gives its single-image result
    g = torch.Generator().manual_seed(9)
    batch = torch.cat([torch.randint(0, 256, (7, 3, 480, 640), dtype=torch.uint8, generator=g), rgb,
                       torch.randint(0, 256, (8, 3, 480, 640), dtype=torch.uint8, generator=g)], 0)
    out = m.infer(batch)
    assert all(torch.equal(out[k][7:8], one[k]) for k in one)
    # skip_camera with GT intrinsics: the GT K comes back, rays / points use it
    K = torch.tensor([[[520.0, 0.0, 318.0], [0.0, 515.0, 242.0], [0.0, 0.0, 1.0]]])
    ref = OV.infer_v1_vit(sd, copy.deepcopy(cfg), rgb, K.clone(), skip_camera=True)
    got = m.infer(rgb, K.clone(), skip_camera=True)
    _check(got, ref["depth"], ref["intrinsics"], ref["points"], "skip_camera_480x640")
