"""CPU-side checks: host logic (shape arithmetic, state-dict layout, HF round trip), the C ABI
surface (library loads, exports every symbol of include/udb.h, ctypes structs match the C structs),
and the no-fallback rule.  No GPU compute here."""
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(name="config_v2_vitl14.json"):
    return json.load(open(os.path.join(ROOT, "tests", "golden", name)))


def test_library_exports_every_header_symbol():
    from unidepth_b200 import _cabi
    from unidepth_b200.build import build
    build()
    hdr = open(os.path.join(ROOT, "include", "udb.h")).read()
    names = set(re.findall(r"\b(udb_[a-z0-9_]+)\s*\(", hdr))
    assert names, "no functions parsed from udb.h"
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for n in sorted(names):
        assert hasattr(lib, n), f"libudb.so does not export {n}"
    assert set(_cabi.EXPORTS) == names, (set(_cabi.EXPORTS) ^ names)
    assert _cabi.lib().udb_version() == 1
    # a freshly loaded library has launched nothing; checked in a new process because GPU tests earlier in this one
    # have already advanced the counter
    fresh = subprocess.check_output([sys.executable, "-c", "import sys; sys.path.insert(0, sys.argv[1]); "
                                     "from unidepth_b200 import _cabi; print(_cabi.lib().udb_launch_count())", ROOT], text=True)
    assert int(fresh) == 0


def test_ctypes_structs_match_c_layout():
    from unidepth_b200 import _cabi
    structs = {"udb_gemm_t": _cabi.Gemm, "udb_conv_halo_t": _cabi.ConvHalo, "udb_attn_t": _cabi.Attn, "udb_layernorm_t": _cabi.LayerNorm,
               "udb_preprocess_t": _cabi.Preprocess, "udb_small_linear_t": _cabi.SmallLinear,
               "udb_ray_embed_t": _cabi.RayEmbed, "udb_postprocess_t": _cabi.Postprocess,
               "udb_config_t": _cabi.Config, "udb_geometry_t": _cabi.Geometry, "udb_infer_args_t": _cabi.InferArgs,
               "udb_v1_preprocess_t": _cabi.V1Preprocess, "udb_layernorm_any_t": _cabi.LayerNormAny, "udb_v1_rays_t": _cabi.V1Rays,
               "udb_v1_postprocess_t": _cabi.V1Postprocess, "udb_v1_config_t": _cabi.V1Config, "udb_infer_v1_args_t": _cabi.InferV1Args,
               "udb_v1_geometry_t": _cabi.V1Geometry, "udb_profile_entry_t": _cabi.ProfileEntry}
    last = {"udb_gemm_t": "ln_eps", "udb_conv_halo_t": "head_out", "udb_attn_t": "lo_off_o", "udb_layernorm_t": "out_split", "udb_preprocess_t": "split",
            "udb_small_linear_t": "ldr", "udb_ray_embed_t": "out_f32", "udb_postprocess_t": "out_rays",
            "udb_config_t": "pixels_max", "udb_geometry_t": "factor", "udb_infer_args_t": "depth_features",
            "udb_v1_preprocess_t": "patches", "udb_layernorm_any_t": "s2d_w", "udb_v1_rays_t": "sh_k", "udb_v1_postprocess_t": "out_points",
            "udb_v1_config_t": "net_w", "udb_infer_v1_args_t": "out_depth", "udb_v1_geometry_t": "ratio", "udb_profile_entry_t": "bytes"}
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "udb.h"\nint main(){\n'
    for n in structs:
        src += f'printf("{n} %zu %zu\\n", sizeof({n}), offsetof({n}, {last[n]}));\n'
    src += "return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")])
        out = subprocess.check_output([os.path.join(d, "t")], text=True)
    for line in out.strip().splitlines():
        n, size, off = line.split()
        cs = structs[n]
        assert ctypes.sizeof(cs) == int(size), (n, ctypes.sizeof(cs), size)
        field = cs._fields_[-1][0]
        assert getattr(cs, field).offset == int(off), (n, field)


def test_param_layout_matches_oracle_fixture():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fixture
    from unidepth_b200.spec import param_shapes
    for name in ("config_v2_vits14.json", "config_v2_vitb14.json", "config_v2_vitl14.json"):
        cfg = _cfg(name)
        assert list(param_shapes(cfg).items()) == list(fixture.param_shapes(cfg).items())


def test_shape_arithmetic_matches_oracle_and_reference_examples():
    import unidepth_oracle as O
    from unidepth_b200 import spec
    g = torch.Generator().manual_seed(0)
    for _ in range(300):
        h = int(torch.randint(16, 2200, (1,), generator=g))
        w = int(torch.randint(16, 2200, (1,), generator=g))
        a = spec.get_paddings((h, w), (0.5, 2.5))
        assert a == O.get_paddings((h, w), (0.5, 2.5))
        for lvl in (None, 0, 4, 9):
            b1 = spec.pixel_bounds({"pixels_min": 200000, "pixels_max": 600000}, lvl)
            assert b1 == O.resolve_pixel_bounds((200000, 600000), lvl)
            f, (nh, nw) = spec.get_resize_factor(a[1], b1)
            assert (f, (nh, nw)) == O.get_resize_factor(a[1], b1)
            assert nh % 14 == 0 and nw % 14 == 0
    assert spec.get_resize_factor((480, 640), (2e5, 6e5))[1] == (490, 644)
    assert spec.get_resize_factor((1024, 1536), (2e5, 6e5))[1] == (644, 952)
    assert spec.get_paddings((480, 1600), (0.5, 2.5)) == ((0, 0, 80, 80), (640, 1600))


def test_state_dict_round_trip_and_no_cpu_fallback():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fixture
    from unidepth_b200 import UniDepthV2
    cfg = _cfg("config_v2_vits14.json")
    m = UniDepthV2(cfg)
    sd = fixture.make_state_dict(cfg, 3)
    info = m.load_state_dict(sd, strict=True)
    assert not info.missing_keys and not info.unexpected_keys
    with tempfile.TemporaryDirectory() as d:
        m.save_pretrained(d)
        assert os.path.exists(os.path.join(d, "config.json")) and os.path.exists(os.path.join(d, "model.safetensors"))
        m2 = UniDepthV2.from_pretrained(d)
    for k, v in m.state_dict().items():
        assert torch.equal(v, m2.state_dict()[k]), k
    assert m.device.type == "cpu"
    with pytest.raises(RuntimeError, match="no CPU"):
        m.infer(torch.zeros(3, 64, 64, dtype=torch.uint8))
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1))


def test_unknown_encoder_is_rejected():
    from unidepth_b200 import UniDepthV2
    cfg = _cfg("config_v2_vits14.json")
    cfg["model"]["pixel_encoder"]["name"] = "convnext_large"
    with pytest.raises(NotImplementedError):
        UniDepthV2(cfg)


def test_engine_geometry_matches_python_and_reference_examples():
    """udb_geometry (C, include/udb.h) == spec.get_paddings / get_resize_factor (== the oracle's) on
    random shapes and every resolution level; host-only calls, no GPU needed."""
    import ctypes as C
    from unidepth_b200 import _cabi, spec
    lib = _cabi.lib()
    cfg = _cabi.Config()
    cfg.embed_dim, cfg.depth, cfg.enc_heads = 1024, 24, 16
    for i, t in enumerate((6, 12, 18, 24)):
        cfg.taps[i] = t
    cfg.pos_grid, cfg.hidden, cfg.dec_heads, cfg.expansion, cfg.out_dim, cfg.n_stages = 37, 512, 8, 4, 64, 3
    for i in range(3):
        cfg.dec_depths[i] = 2
    cfg.ratio_min, cfg.ratio_max, cfg.pixels_min, cfg.pixels_max = 0.5, 2.5, 200000.0, 600000.0
    h = C.c_void_p()
    assert lib.udb_create(C.byref(cfg), C.byref(h)) == 0
    try:
        g = _cabi.Geometry()
        gen = torch.Generator().manual_seed(1)
        shapes = [(480, 640), (1024, 1536), (480, 1600), (1000, 400)]
        shapes += [(int(torch.randint(16, 2200, (1,), generator=gen)), int(torch.randint(16, 2200, (1,), generator=gen)))
                   for _ in range(300)]
        for (H, W) in shapes:
            pads, padded = spec.get_paddings((H, W), (0.5, 2.5))
            for lvl in (None, 0, 2, 5, 9):
                bounds = spec.pixel_bounds({"pixels_min": 200000, "pixels_max": 600000}, lvl)
                f, (nh, nw) = spec.get_resize_factor(padded, bounds)
                assert lib.udb_geometry(h, H, W, -1 if lvl is None else lvl, C.byref(g)) == 0
                assert (g.pad_l, g.pad_r, g.pad_t, g.pad_b) == pads and (g.padded_h, g.padded_w) == padded
                assert (g.net_h, g.net_w, g.gh, g.gw) == (nh, nw, nh // 14, nw // 14) and g.factor == f, (H, W, lvl)
        assert lib.udb_geometry(h, 480, 640, -1, C.byref(g)) == 0 and (g.net_h, g.net_w) == (490, 644)
        assert lib.udb_geometry(h, 480, 640, 10, C.byref(g)) != 0          # resolution_level out of range
        # unprepared / incomplete handles fail loudly instead of computing anything
        a = _cabi.InferArgs()
        assert lib.udb_infer_v2(h, C.byref(a), None) != 0
        assert b"null" in lib.udb_last_error()
    finally:
        lib.udb_destroy(h)
    bad = _cabi.Config()
    bad.embed_dim, bad.enc_heads, bad.hidden, bad.dec_heads, bad.n_stages = 1000, 16, 512, 8, 3
    assert lib.udb_create(C.byref(bad), C.byref(h)) != 0


def test_hubconf_entry_point():
    """hubconf.UniDepth(version, backbone, pretrained) as in the reference (hubconf.py:25-41), offline."""
    sys.path.insert(0, ROOT)
    import hubconf
    from unidepth_b200 import UniDepthV2
    for bb, d in (("vits14", 384), ("vitb14", 768), ("vitl14", 1024)):
        m = hubconf.UniDepth("v2", bb, pretrained=False)
        assert isinstance(m, UniDepthV2) and m.spec.embed_dim == d
    from unidepth_b200 import UniDepthV1
    m1 = hubconf.UniDepth("v1", "cnvnxtl", pretrained=False)
    assert isinstance(m1, UniDepthV1) and m1.image_shape == [462, 616]
    with pytest.raises(NotImplementedError):
        hubconf.UniDepth("v1", "vitl14", pretrained=False)
    with pytest.raises(AssertionError):
        hubconf.UniDepth("v2", "resnet50", pretrained=False)


def test_engine_fails_loudly_without_a_gpu_or_weights():
    """No CPU fallback anywhere in the C engine: preparing a shape needs the device, and an engine whose
    packed tensors were never registered reports which one is missing instead of computing."""
    import ctypes as C
    from unidepth_b200 import _cabi
    lib = _cabi.lib()
    cfg = _cabi.Config()
    cfg.embed_dim, cfg.depth, cfg.enc_heads, cfg.pos_grid = 384, 12, 6, 37
    for i, t in enumerate((3, 6, 9, 12)):
        cfg.taps[i] = t
    cfg.hidden, cfg.dec_heads, cfg.expansion, cfg.out_dim, cfg.n_stages = 256, 8, 4, 32, 3
    for i in range(3):
        cfg.dec_depths[i] = 2
    cfg.ratio_min, cfg.ratio_max, cfg.pixels_min, cfg.pixels_max = 0.5, 2.5, 200000.0, 600000.0
    h = C.c_void_p()
    assert lib.udb_create(C.byref(cfg), C.byref(h)) == 0
    try:
        assert lib.udb_workspace_bytes(h, 1, 120, 160, -1) == 0          # 'pos' not registered
        assert b"pos" in lib.udb_last_error()
        buf = (C.c_float * 64)()
        shape = (C.c_int64 * 2)(4, 4)
        addr = C.addressof(buf)
        assert lib.udb_set_weight(h, b"pos", C.c_void_p(addr + 4), shape, 2, _cabi.DT_F32) != 0      # misaligned pointer
        assert b"aligned" in lib.udb_last_error()
        if not torch.cuda.is_available():
            aligned = (addr + 15) & ~15
            assert lib.udb_set_weight(h, b"pos", C.c_void_p(aligned), shape, 2, _cabi.DT_F32) == 0
            assert lib.udb_workspace_bytes(h, 1, 120, 160, -1) == 0      # cudaMalloc of the tables fails: no device
            assert lib.udb_last_error() != b""
    finally:
        lib.udb_destroy(h)


def test_c_example_links_and_runs_against_the_abi():
    """examples/engine_minimal.c: plain C, no torch, links libudb.so and prints the reference's geometry
    examples (SURVEY 8a1): 480x640 -> 490x644, 1024x1536 -> 644x952, 480x1600 -> pad 80/80, 1000x400 -> pad 50/50."""
    from unidepth_b200 import _cabi
    from unidepth_b200.build import build
    build()
    libdir = os.path.dirname(_cabi.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "engine_minimal")
        subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                               os.path.join(ROOT, "examples", "engine_minimal.c"), "-L", libdir, "-ludb",
                               f"-Wl,-rpath,{libdir}", "-o", exe])
        out = subprocess.check_output([exe], text=True)
    assert "480x640 -> pad l0 r0 t0 b0, network 490x644 (grid 35x46)" in out
    assert "1024x1536 -> pad l0 r0 t0 b0, network 644x952 (grid 46x68)" in out
    assert "480x1600 -> pad l0 r0 t80 b80" in out and "1000x400 -> pad l50 r50 t0 b0" in out
    assert "as expected:" in out and "udb version 1" in out


def test_v1_geometry_and_fail_loudly():
    """V1's fixed-shape arithmetic (unidepthv1.py:30-46) against the values the reference functions produced
    (tests/golden/v1_parts.npz), and the V1 class has no CPU path."""
    import numpy as np
    from unidepth_b200 import UniDepthV1
    from unidepth_b200.spec_v1 import v1_paddings, v1_shapes
    z = np.load(os.path.join(ROOT, "tests", "golden", "v1_parts.npz"))
    for i, (h, w) in enumerate(z["cases"]):
        (rh, rw), ratio = v1_shapes((int(h), int(w)), (462, 616))
        assert [rh, rw, *v1_paddings((rh, rw), (462, 616))] == z[f"shape{i}"].tolist()
        assert abs(ratio - float(z[f"ratio{i}"])) < 1e-12
    # the C engine's own copy of that arithmetic (engine_v1.cu v1_geometry, exported as udb_v1_geometry) against the Python
    # functions -- themselves checked against the reference just above -- on the golden cases and 400 random shapes
    import ctypes as C
    from unidepth_b200 import _cabi
    lib, g = _cabi.lib(), _cabi.V1Geometry()
    gen = torch.Generator().manual_seed(2)
    shapes = [tuple(int(v) for v in c) for c in z["cases"]] + [(462, 616), (1, 1), (3000, 17), (17, 3000)]
    shapes += [(int(torch.randint(8, 2600, (1,), generator=gen)), int(torch.randint(8, 2600, (1,), generator=gen))) for _ in range(400)]
    for net in ((462, 616), (42, 56), (616, 462)):
        for (h, w) in shapes:
            (rh, rw), ratio = v1_shapes((h, w), net)
            pl, pr, pt, pb = v1_paddings((rh, rw), net)
            assert lib.udb_v1_geometry(h, w, net[0], net[1], C.byref(g)) == 0
            assert (g.resized_h, g.resized_w, g.pad_l, g.pad_r, g.pad_t, g.pad_b) == (rh, rw, pl, pr, pt, pb), (h, w, net)
            assert g.ratio == ratio, (h, w, net)
    assert lib.udb_v1_geometry(0, 5, 462, 616, C.byref(g)) != 0
    cfg = json.load(open(os.path.join(ROOT, "tests", "golden", "config_v1_cnvnxtl.json")))
    cfg["model"]["pixel_encoder"]["arch"] = {"depths": [1, 1, 1, 1], "dims": [64, 64, 64, 64]}
    m = UniDepthV1(cfg)
    with pytest.raises(RuntimeError):
        m.infer(torch.zeros(3, 32, 32, dtype=torch.uint8))
