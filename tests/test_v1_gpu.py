"""UniDepthV1 (ConvNeXt-L, BASELINE config 4) on the GPU: every V1-only kernel against a PyTorch fp32 reference of the
same op, and the whole `infer` (through udb_infer_v1) against outputs of the unmodified reference (tests/golden/v1_*.npz;
the Nystrom function substitution is described in oracle/make_golden_v1.py) and against the oracle."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f16, f32 = torch.float16, torch.float32


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _lib():
    from unidepth_b200 import _cabi
    return _cabi, _cabi.lib()


def _rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp(min=1e-12)).item()


def test_dwconv7_and_layernorm_any():
    cabi, lib = _lib()
    dev = _dev()
    g = torch.Generator().manual_seed(0)
    for (B, H, W, Cc) in ((2, 29, 39, 192), (1, 14, 19, 1536), (3, 9, 70, 64)):
        x = torch.randn(B, H, W, Cc, generator=g).to(dev).half()
        w = (torch.randn(Cc, 1, 7, 7, generator=g) / 7).to(dev)
        b = torch.randn(Cc, generator=g).to(dev)
        y = torch.empty_like(x)
        cabi.check(lib.udb_dwconv7_nhwc_f16(_p(x), _p(w.reshape(Cc, 49).t().contiguous()), _p(b), _p(y), B, H, W, Cc, _st()), "dwconv")
        ref = F.conv2d(x.double().permute(0, 3, 1, 2), w.double(), b.double(), padding=3, groups=Cc).permute(0, 2, 3, 1)
        err = _rel(y.float(), ref)
        print(f"dwconv7 {B}x{H}x{W}x{Cc}: {err:.2e}")
        assert err < 2e-3                      # one f16 rounding of the output
    for dim in (192, 384, 768, 1536, 512):
        rows = 777
        x = (torch.randn(rows, dim, generator=g) * 2 + 0.5).to(dev)
        lw, lb = torch.randn(dim, generator=g).to(dev), torch.randn(dim, generator=g).to(dev)
        add = torch.randn(37, dim, generator=g).to(dev)
        for in16 in (False, True):
            for with_add in (False, True):
                xin = x.half() if in16 else x
                out = torch.empty(rows, dim, device=dev, dtype=f32)
                p = cabi.LayerNormAny()
                p.inp, p.in_f32, p.out, p.out_f32, p.weight, p.bias = _p(xin), int(not in16), _p(out), 1, _p(lw), _p(lb)
                p.rows, p.dim, p.ld_in, p.ld_out, p.eps = rows, dim, dim, dim, 1e-6
                if with_add:
                    p.add, p.add_mod = _p(add), 37
                cabi.check(lib.udb_layernorm_any(C.byref(p), _st()), "ln_any")
                xi = xin.float() + (add[torch.arange(rows, device=dev) % 37] if with_add else 0)
                ref = F.layer_norm(xi, (dim,), lw, lb, 1e-6)
                assert _rel(out, ref) < 2e-5, (dim, in16, with_add)
    # space-to-depth output: LayerNorm2d + the k2 s2 downsample's im2col (odd sizes drop the last row / column)
    B, H, W, dim = 2, 7, 9, 192
    x = torch.randn(B, H, W, dim, generator=g).to(dev)
    lw, lb = torch.randn(dim, generator=g).to(dev), torch.randn(dim, generator=g).to(dev)
    out = torch.zeros(B * (H // 2) * (W // 2), 4 * dim, device=dev, dtype=f16)
    p = cabi.LayerNormAny()
    p.inp, p.in_f32, p.out, p.out_f32, p.weight, p.bias = _p(x), 1, _p(out), 0, _p(lw), _p(lb)
    p.rows, p.dim, p.ld_in, p.ld_out, p.eps, p.s2d_h, p.s2d_w = B * H * W, dim, dim, 4 * dim, 1e-6, H, W
    cabi.check(lib.udb_layernorm_any(C.byref(p), _st()), "ln_any s2d")
    y = F.layer_norm(x, (dim,), lw, lb, 1e-6)[:, :H // 2 * 2, :W // 2 * 2]
    ref = y.reshape(B, H // 2, 2, W // 2, 2, dim).permute(0, 1, 3, 2, 4, 5).reshape(B * (H // 2) * (W // 2), 4 * dim)
    assert _rel(out.float(), ref) < 2e-3
    # and the conv k2 s2 as a GEMM on it equals F.conv2d
    from unidepth_b200 import ops
    cw = (torch.randn(384, dim, 2, 2, generator=g) / 28).to(dev)
    o = ops.gemm(out, cw.permute(0, 2, 3, 1).reshape(384, -1).half().contiguous(), out_dtype=f32)
    refc = F.conv2d(F.layer_norm(x, (dim,), lw, lb, 1e-6).double().permute(0, 3, 1, 2), cw.double(), stride=2).permute(0, 2, 3, 1).reshape(-1, 384)
    assert _rel(o, refc) < 3e-3


def test_aa_resize_preprocess_and_postprocess():
    cabi, lib = _lib()
    dev = _dev()
    g = torch.Generator().manual_seed(1)
    for (H, W, oh, ow) in ((115, 154, 28, 38), (57, 77, 28, 38), (14, 19, 28, 38), (30, 41, 30, 41)):
        x = torch.randn(2, H, W, 64, generator=g).to(dev).half()
        out = torch.empty(2, oh, ow, 64, device=dev, dtype=f16)
        cabi.check(lib.udb_aa_resize_nhwc_f16(_p(x), _p(out), 2, H, W, 64, oh, ow, _st()), "aa")
        ref = F.interpolate(x.float().permute(0, 3, 1, 2), size=(oh, ow), mode="bilinear", align_corners=False, antialias=True).permute(0, 2, 3, 1)
        err = _rel(out.float(), ref)
        print(f"aa_resize {H}x{W}->{oh}x{ow}: {err:.2e}")
        assert err < 2e-3
    # pre-processing + 4x4 patches vs the oracle's v1_preprocess + unfold
    import unidepth_v1_parts as P1
    for (H, W) in ((480, 640), (375, 1242), (1000, 400), (231, 308)):
        rgb = torch.randint(0, 256, (2, 3, H, W), dtype=torch.uint8, generator=g)
        (rh, rw), ratio = P1.v1_shapes((H, W), (462, 616))
        pads = P1.v1_paddings((rh, rw), (462, 616))
        mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)
        std = torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
        xr, _ = P1.v1_preprocess((rgb.float() / 255 - mean) / std, None, (rh, rw), pads, ratio)
        ref = F.unfold(xr, kernel_size=4, stride=4).transpose(1, 2).reshape(-1, 48)          # (c, py, px) columns
        gh, gw = (462 - 4) // 4 + 1, (616 - 4) // 4 + 1
        patches = torch.empty(2 * gh * gw, 64, device=dev, dtype=f16)
        p = cabi.V1Preprocess()
        rd = rgb.to(dev)
        p.rgb, p.rgb_is_u8, p.scale255, p.normalize, p.B, p.H, p.W = _p(rd), 1, 1, 1, 2, H, W
        p.rh, p.rw, p.pad_l, p.pad_t, p.net_h, p.net_w, p.patches = rh, rw, pads[0], pads[2], 462, 616, _p(patches)
        cabi.check(lib.udb_v1_preprocess(C.byref(p), _st()), "v1_preprocess")
        err = (patches[:, :48].float().cpu() - ref).abs().max().item()
        print(f"v1_preprocess {H}x{W}: max abs err {err:.2e}")
        assert err < 3e-3 and patches[:, 48:].abs().max().item() == 0
    # mean of the three maps + final resize + back-projection vs the oracle's v1_postprocess / zbuffer conversion
    B, gh, gw = 2, 28, 38
    outs = [torch.rand(B, 1, gh << s, gw << s, generator=g) + 0.5 for s in (1, 2, 3)]
    for (H, W) in ((480, 640), (375, 1242)):
        (rh, rw), ratio = P1.v1_shapes((H, W), (462, 616))
        pads = P1.v1_paddings((rh, rw), (462, 616))
        K = torch.tensor([[[500.0, 0, 310.0], [0, 505.0, 240.0], [0, 0, 1]]]).repeat(B, 1, 1)
        pred, _ = P1.v1_postprocess(outs, K.clone(), (462, 616), pads, ratio, (H, W))
        ang = P1.generate_rays(K, (H, W))[1].transpose(1, 2).reshape(B, 2, H, W)
        pts = P1.spherical_zbuffer_to_euclidean(torch.cat((ang, pred), 1).permute(0, 2, 3, 1)).permute(0, 3, 1, 2)
        d = [o.to(dev).contiguous() for o in outs]
        mean = torch.empty(B, 462, 616, device=dev)
        cabi.check(lib.udb_v1_mean_maps(_p(d[0]), _p(d[1]), _p(d[2]), _p(mean), B, gh, gw, 462, 616, _st()), "mean")
        k4 = torch.tensor([[500.0, 505.0, 310.0, 240.0]]).repeat(B, 1).to(dev)
        od, op = torch.empty(B, 1, H, W, device=dev), torch.empty(B, 3, H, W, device=dev)
        pp = cabi.V1Postprocess()
        pp.mean, pp.k4, pp.B, pp.net_h, pp.net_w = _p(mean), _p(k4), B, 462, 616
        pp.pad_l, pp.pad_r, pp.pad_t, pp.pad_b, pp.H, pp.W, pp.out_depth, pp.out_points = *pads, H, W, _p(od), _p(op)
        cabi.check(lib.udb_v1_postprocess(C.byref(pp), _st()), "post")
        assert _rel(od.cpu(), pred) < 1e-5 and _rel(op.cpu(), pts) < 1e-4, (H, W)


def test_rays_sh81_embedding():
    cabi, lib = _lib()
    dev = _dev()
    import unidepth_v1_oracle as O1
    from sh81 import rsh_cart
    import math
    B = 2
    K = torch.tensor([[[380.0, 0, 300.0], [0, 400.0, 250.0], [0, 0, 1]], [[700.0, 0, 320.0], [0, 650.0, 200.0], [0, 0, 1]]])
    rays = O1.generate_rays(K, (462, 616))[0]
    g = torch.Generator().manual_seed(2)
    lw, lb = 1 + 0.1 * torch.randn(81, generator=g), 0.1 * torch.randn(81, generator=g)
    shk = [0.0] * 81
    for l in range(9):
        for m in range(l + 1):
            shk[l * 9 + m] = math.sqrt((2 * l + 1) / (4 * math.pi) * math.factorial(l - m) / math.factorial(l + m)) * (math.sqrt(2) if m else 1)
    for s in (1, 2, 4):
        gh, gw = 28 * s, 38 * s
        r = F.normalize(O1.flat_interpolate(rays, (462, 616), (gh, gw)), dim=-1)
        ref = F.layer_norm(rsh_cart(r, 8), (81,), lw, lb, 1e-5)
        out = torch.empty(B * gh * gw, 128, device=dev, dtype=f16)
        p = cabi.V1Rays()
        intr4 = torch.stack([K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2]], 1).contiguous().to(dev)
        lwd, lbd = F.pad(lw, (0, 3)).to(dev), F.pad(lb, (0, 3)).to(dev)
        p.intr4, p.B, p.net_h, p.net_w, p.gh, p.gw, p.ln_w, p.ln_b, p.out = _p(intr4), B, 462, 616, gh, gw, _p(lwd), _p(lbd), _p(out)
        for i in range(81):
            p.sh_k[i] = shk[i]
        cabi.check(lib.udb_v1_rays_sh81(C.byref(p), _st()), "rays_sh81")
        err = (out[:, :81].float().cpu() - ref.reshape(-1, 81)).abs().max().item()
        print(f"rays_sh81 level x{s}: max abs err {err:.2e}")
        assert err < 5e-3 and out[:, 81:].abs().max().item() == 0


def test_small_attention_pieces_and_nystrom():
    cabi, lib = _lib()
    dev = _dev()
    import unidepth_v1_oracle as O1
    g = torch.Generator().manual_seed(3)
    # row softmax
    s = torch.randn(300, 1088, generator=g).to(dev) * 5
    pr = torch.empty(300, 1088, device=dev, dtype=f16)
    cabi.check(lib.udb_softmax_rows(_p(s), _p(pr), 300, 1064, 1088, 1088, 0.3, _st()), "softmax")
    ref = torch.softmax(s[:, :1064] * 0.3, -1)
    assert (pr[:, :1064].float() - ref).abs().max().item() < 1e-3 and pr[:, 1064:].abs().max().item() == 0
    # 4-query cross attention
    B, nq, nk, D = 2, 4, 333, 512
    q, pos = torch.randn(B * nq, D, generator=g).to(dev), torch.randn(nq, D, generator=g).to(dev)
    kv = torch.randn(B * nk, 2 * D, generator=g).to(dev).half()
    out = torch.empty(B * nq, D, device=dev)
    scratch = torch.empty(B * 16 * nq * (D + 2), device=dev)
    cabi.check(lib.udb_cross_attn_small(_p(q), _p(pos), _p(kv), _p(out), _p(scratch), B, nq, nk, D, D ** -0.5, _st()), "cross")
    qq = (q.view(B, nq, D) + pos)
    kk, vv = kv.float().view(B, nk, 2 * D)[..., :D], kv.float().view(B, nk, 2 * D)[..., D:]
    ref = torch.softmax(qq @ kk.transpose(1, 2) * D ** -0.5, -1) @ vv
    assert _rel(out.view(B, nq, D), ref) < 1e-4
    # single-output 3x3 conv + exp(clamp)
    x = torch.randn(2, 20, 31, 128, generator=g).to(dev).half()
    w = (torch.randn(1, 128, 3, 3, generator=g) / 30).to(dev)
    o = torch.empty(2, 20, 31, device=dev)
    cabi.check(lib.udb_conv3x3_c1_exp(_p(x), _p(w.permute(0, 2, 3, 1).reshape(9, 128).contiguous()), 0.1, _p(o), 2, 20, 31, 128, _st()), "c1")
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), w.double(), torch.tensor([0.1], device=dev, dtype=torch.float64), padding=1).clamp(-10, 10).exp()[:, 0]
    assert _rel(o, ref) < 1e-5
    # Nystrom attention assembled from the pieces (as engine_v1.cu's mh_attn_block does) vs the oracle's restatement
    from unidepth_b200 import ops
    B, n, heads = 2, 1000, 2
    Cc = heads * 64
    qf, kf, vf = (torch.randn(B, n, Cc, generator=g) * 0.7 for _ in range(3))
    qh = qf.to(dev).half().reshape(B * n, Cc).contiguous()
    kvh = torch.cat([kf, vf], -1).to(dev).half().reshape(B * n, 2 * Cc).contiguous()
    lm = torch.empty(B * 128, 2 * Cc, device=dev, dtype=f16)
    cabi.check(lib.udb_nystrom_landmarks(_p(qh), Cc, _p(kvh), 2 * Cc, _p(lm), B, n, heads, _st()), "landmarks")
    mm = B * heads * 128 * 128
    k2, z, tmp = torch.empty(mm, device=dev), torch.empty(mm, device=dev), torch.empty(3 * mm, device=dev)
    cabi.check(lib.udb_nystrom_k2_pinv(_p(lm), _p(k2), _p(z), _p(tmp), B, heads, 6, _st()), "pinv")
    k3 = torch.empty(B * 128, Cc, device=dev, dtype=f16)
    ops.attention(lm, kvh, kvh, k3, B=B, heads=heads, seq_q=128, seq_k=n, head_dim=64, q_col0=0, k_col0=0, v_col0=Cc)
    w2 = torch.empty(B * 128, Cc, device=dev, dtype=f16)
    cabi.check(lib.udb_nystrom_zk3(_p(z), _p(k3), Cc, _p(w2), Cc, B, heads, _st()), "zk3")
    o = torch.empty(B * n, Cc, device=dev, dtype=f16)
    ops.attention(qh, lm, w2, o, B=B, heads=heads, seq_q=n, seq_k=128, head_dim=64, q_col0=0, k_col0=Cc, v_col0=0)
    hsplit = lambda t: t.half().float().reshape(B, n, heads, 64).transpose(1, 2)
    ref = O1.nystrom_attention(hsplit(qf), hsplit(kf), hsplit(vf)).transpose(1, 2).reshape(B * n, Cc)
    err = _rel(o.float().cpu(), ref)
    print(f"nystrom attention vs oracle restatement: {err:.2e}")
    assert err < 2e-2


def _v1_model(cfg, sd):
    from unidepth_b200 import UniDepthV1
    import copy
    m = UniDepthV1(copy.deepcopy(cfg))
    m.load_state_dict(sd, strict=True)
    return m.to("cuda:0").eval()


# measured on the B200 (profiles/r02_v1_parity_gpu.log), asserted with a 1.5x margin: (depth ARel, depth max-rel, K rel)
V1_MEASURED = {
    "golden_v1_cnvnxtl_480x640": (1.724e-4, 8.849e-4, 7.815e-5),
    "golden_v1_cnvnxtl_gtK_375x1242": (1.312e-4, 7.532e-4, 1.148e-4),
    "skip_camera_480x640": (1.702e-4, 9.559e-4, 1e-6),
    "default": (2.0e-4, 1.0e-3, 1.2e-4),
}


def _check_v1(out, ref_depth, ref_K, ref_pts, tag, pts_stride=1, depth_stride=1):
    d, dr = out["depth"].float().cpu()[:, :, ::depth_stride, ::depth_stride], ref_depth
    rel = (d - dr).abs() / dr
    k, kr = out["intrinsics"].cpu(), ref_K
    kerr = max(((k[:, i, j] - kr[:, i, j]).abs() / kr[:, i, j].abs()).max().item() for i, j in ((0, 0), (1, 1), (0, 2), (1, 2)))
    pts = out["points"].float().cpu()[:, :, ::pts_stride, ::pts_stride]
    perr = ((pts - ref_pts).abs() / ref_pts.abs().clamp(min=0.1 * ref_pts.abs().mean())).mean().item()
    print(f"V1PARITY {tag}: depth ARel {rel.mean().item():.3e} max {rel.max().item():.3e}; intrinsics rel {kerr:.3e}; points mean rel {perr:.3e}")
    m = V1_MEASURED.get(tag, V1_MEASURED["default"])
    assert rel.mean().item() < 1.5 * m[0] and rel.max().item() < 1.5 * m[1] and kerr < 1.5 * m[2], (tag, rel.mean().item(), rel.max().item(), kerr)
    assert perr < 5e-3


@pytest.mark.parametrize("name", ["v1_cnvnxtl_480x640", "v1_cnvnxtl_gtK_375x1242"])
def test_v1_infer_against_reference_golden(name, golden_dir):
    _dev()
    from test_oracle_golden import v1_case_inputs
    cfg, sd, rgb, K, meta, z = v1_case_inputs(golden_dir, name)
    m = _v1_model(cfg, sd)
    out = m.infer(rgb, K, skip_camera=meta["skip_camera"])
    assert set(out) == {"intrinsics", "points", "depth"}
    _check_v1(out, torch.from_numpy(z["depth"]), torch.from_numpy(z["intrinsics"]), torch.from_numpy(z["points"]), "golden_" + name,
              meta["strides"]["points"], meta["strides"]["depth"])
    # graph replay and eager agree bit for bit; a batch returns each image's single-image result
    again = m.infer(rgb, K, skip_camera=meta["skip_camera"])
    assert all(torch.equal(again[k], out[k]) for k in out)
    m.use_cuda_graph = False
    eager = m.infer(rgb, K, skip_camera=meta["skip_camera"])
    assert all(torch.equal(eager[k], out[k]) for k in out)


def test_v1_batch_float_input_and_skip_camera(golden_dir):
    _dev()
    import copy
    import unidepth_v1_oracle as O1
    from test_oracle_golden import v1_case_inputs
    cfg, sd, rgb, _, meta, z = v1_case_inputs(golden_dir, "v1_cnvnxtl_480x640")
    m = _v1_model(cfg, sd)
    g = torch.Generator().manual_seed(9)
    batch = torch.cat([rgb, torch.randint(0, 256, (2, 3, 480, 640), dtype=torch.uint8, generator=g)], 0)
    out = m.infer(batch)
    one = m.infer(rgb)
    assert torch.equal(out["depth"][:1], one["depth"]) and torch.equal(out["intrinsics"][:1], one["intrinsics"])
    # float input in [0, 1] takes the same path as uint8 (unidepthv1.py:301-308)
    fl = m.infer(rgb.float() / 255.0)
    assert (fl["depth"] - one["depth"]).abs().max().item() < 2e-3 * one["depth"].max().item()
    # skip_camera with GT intrinsics: the GT K comes back, rays / points use it
    K = torch.tensor([[[520.0, 0.0, 318.0], [0.0, 515.0, 242.0], [0.0, 0.0, 1.0]]])
    ref = O1.infer_v1(sd, copy.deepcopy(cfg), rgb, K.clone(), skip_camera=True)
    got = m.infer(rgb, K.clone(), skip_camera=True)
    _check_v1(got, ref["depth"], ref["intrinsics"], ref["points"], "skip_camera_480x640")
