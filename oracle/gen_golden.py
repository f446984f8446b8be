"""Generate tests/golden/*.npz by running the REAL reference (nagadomi/nunif,
imported read-only from /root/reference) on seeded inputs.

Run in the build container only (the GPU box has no /root/reference):
    NUNIF_HOME=/tmp/nunif_home PYTHONDONTWRITEBYTECODE=1 \
    PYTHONPATH=/root/reference:/root/repo python oracle/gen_golden.py

The committed .npz files pin the oracle (tests/test_oracle_golden.py) and are
the fixtures the GPU parity tests compare against.  Inputs are regenerated at
test time from nunif_b200.synth with the seeds stored in each file, and the
inputs themselves are stored too so a synth drift is detected.
"""
import os
import sys
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("NUNIF_HOME", "/tmp/nunif_home")
sys.path.insert(0, "/root/reference")

from nunif_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
torch.set_grad_enabled(False)
torch.manual_seed(0)


def save(name, **arrays):
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **{k: (v.numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()})
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def gen_seam_config():
    from nunif.utils.seam_blending import SeamBlending
    rows = []
    cases = []
    for (scale, offset, blend) in [(1, 28, 0), (2, 36, 0), (1, 8, 4), (2, 16, 8), (4, 32, 16), (1, 8, 16)]:
        for tile in (64, 112, 160, 256, 400):
            for (h, w) in [(1, 1), (17, 33), (220, 220), (240, 240), (256, 256), (300, 420), (1080, 1920),
                           (2160, 3840), (4320, 7680), (236, 237), (471, 12)]:
                if tile - (2 * -(-offset // scale) + -(-blend // scale)) <= 0:
                    continue
                p = SeamBlending.create_config((h, w), scale, offset, tile, blend)
                cases.append([h, w, scale, offset, tile, blend])
                rows.append([p["y_h"], p["y_w"], p["h_blocks"], p["w_blocks"], *p["pad"],
                             p["y_buffer_h"], p["y_buffer_w"], p["input_tile_step"], p["output_tile_step"]])
    filters = {}
    for (scale, offset, tile, blend) in [(4, 32, 64, 16), (2, 16, 64, 8), (1, 8, 64, 4), (1, 8, 64, 16)]:
        filters[f"filter_{scale}_{offset}_{tile}_{blend}"] = SeamBlending.create_blend_filter(scale, offset, tile, blend, 3)
    save("seam_config", cases=np.array(cases, dtype=np.int64), configs=np.array(rows, dtype=np.int64), **filters)

    # find_valid_tile_size for both validators (model.py:51-62)
    import waifu2x.models  # noqa
    from nunif.models import create_model
    up = create_model("waifu2x.upcunet")
    sw = create_model("waifu2x.swin_unet_4x")
    q = np.arange(64, 600)
    save("tile_size", query=q,
         cunet=np.array([up.find_valid_tile_size(int(t)) for t in q]),
         swin=np.array([sw.find_valid_tile_size(int(t)) for t in q]))


def gen_models():
    import waifu2x.models  # noqa
    from nunif.models import create_model
    from nunif.utils.render import tiled_render
    # --- cunet family
    for name, sdf, n in [("waifu2x.upcunet", synth.upcunet_state_dict, "upcunet"),
                         ("waifu2x.cunet", synth.cunet_state_dict, "cunet")]:
        m = create_model(name).eval()
        m.load_state_dict(sdf(0), strict=True)
        x = synth.synth_image(11, 3, 104, 104).unsqueeze(0)
        z = m(x)
        img = synth.synth_image(12, 3, 150, 170)
        y = tiled_render(img, m, tile_size=104, batch_size=3)
        save(n, x=x, z=z, img=img, render=y, tile_size=104, batch_size=3)
    # --- swin family
    m4 = create_model("waifu2x.swin_unet_4x").eval()
    m4.load_state_dict(synth.swin_unet_state_dict(0, 4), strict=True)
    x = synth.synth_image(21, 3, 64, 64).unsqueeze(0).repeat(2, 1, 1, 1)
    x[1] = synth.synth_image(22, 3, 64, 64)
    z4 = m4(x)
    m2 = m4.to_2x().eval()  # waifu2x/utils.py:99-100 (_setup -> .eval())
    z2 = m2(x)
    m1 = m4.to_1x().eval()
    z1 = m1(x)
    img = synth.synth_image(23, 3, 70, 100)
    y4 = tiled_render(img, m4, tile_size=64, batch_size=4)
    y2 = tiled_render(img, m2, tile_size=64, batch_size=4)
    save("swin_unet_4x", x=x, z4=z4, z2=z2, z1=z1, img=img, render4=y4, render2=y2, tile_size=64, batch_size=4)
    for sf, name in [(2, "waifu2x.swin_unet_2x"), (1, "waifu2x.swin_unet_1x")]:
        m = create_model(name).eval()
        m.load_state_dict(synth.swin_unet_state_dict(0, sf), strict=True)
        save(f"swin_unet_{sf}x", x=x[:1], z=m(x[:1]))


def gen_iw3():
    from iw3.backward_warp import apply_divergence_grid_sample
    from iw3.forward_warp import apply_divergence_forward_warp
    from iw3.dilation import dilate_edge
    from iw3.depth_scaler import minmax_normalize
    from iw3.mapper import get_mapper
    from iw3.anaglyph import apply_anaglyph_redcyan

    B, H, W, h, w = 2, 72, 128, 28, 49
    c = torch.stack([synth.synth_image(31 + i, 3, H, W) for i in range(B)])
    d_lo = synth.synth_depth(41, B, h, w)
    d_hi = synth.synth_depth(42, B, H, W)

    out = {}
    for sv in ("both", "left", "right"):
        l, r = apply_divergence_grid_sample(c, d_lo, 2.0, 0.5, sv)
        out[f"bw_{sv}_l"], out[f"bw_{sv}_r"] = l, r
    l, r = apply_divergence_grid_sample(c, d_hi, 5.0, 0.3, "both")
    out["bw_hi_l"], out["bw_hi_r"] = l, r
    save("backward_warp", c=c, d_lo=d_lo, d_hi=d_hi, **out)

    out = {}
    for tag, depth, div, conv, wb in [("hi", d_hi, 4.0, 0.5, False), ("hi_wb", d_hi, 10.0, 0.3, True),
                                      ("lo", d_lo, 4.0, 0.5, False)]:
        for method in ("forward_fill", "forward"):
            l, r, lm, rm = apply_divergence_forward_warp(c.clone(), depth.clone(), div, conv, method=method,
                                                         synthetic_view="both", return_mask=True, width_base=wb)
            out[f"fw_{tag}_{method}_l"], out[f"fw_{tag}_{method}_r"] = l, r
            out[f"fw_{tag}_{method}_lm"], out[f"fw_{tag}_{method}_rm"] = lm, rm
    for sv in ("left", "right"):
        l, r = apply_divergence_forward_warp(c.clone(), d_hi.clone(), 2.0, 0.5, method="forward_fill",
                                             synthetic_view=sv, width_base=False)
        out[f"fw_{sv}_l"], out[f"fw_{sv}_r"] = l, r
    # long holes: > 100 px (iteration cap, forward_warp.py:18,45)
    Wl = 1280
    cl = synth.synth_image(35, 3, 12, Wl).unsqueeze(0)
    dl = synth.synth_depth(45, 1, 12, Wl)
    l, r = apply_divergence_forward_warp(cl.clone(), dl.clone(), 60.0, 0.0, method="forward_fill",
                                         synthetic_view="both", width_base=True)
    out["fw_long_l"], out["fw_long_r"] = l, r
    save("forward_warp", c=c, d_lo=d_lo, d_hi=d_hi, cl=cl, dl=dl, **out)

    dd = synth.synth_depth(51, 2, 56, 98) * 7.0 + 0.25
    out = {"x": dd}
    for n in ([2, 1], [1, 2], 2, [0, 0], [3, 0]):
        key = "dil_" + "_".join(str(v) for v in (n if isinstance(n, list) else [n]))
        out[key] = dilate_edge(dd.clone(), n)
    mn, mx = dd[0].amin(), dd[0].amax()
    out["minmax0"] = minmax_normalize(dd[0].clone(), mn, mx)
    out["div_6"] = get_mapper("div_6")(out["minmax0"])
    out["div_1"] = get_mapper("div_1")(out["minmax0"])
    save("dilation", **out)

    le, re = synth.synth_image(61, 3, 40, 64), synth.synth_image(62, 3, 40, 64)
    out = {"l": le, "r": re}
    for t in ("dubois", "dubois2", "color", "gray", "half-color", "wimmer", "wimmer2"):
        out[t.replace("-", "_")] = apply_anaglyph_redcyan(le.clone(), re.clone(), t)
    save("anaglyph", **out)


def gen_alpha_tta():
    """AlphaBorderPadding (nunif/utils/alpha.py) and tta_split/tta_merge (nunif/transforms/tta.py)."""
    from nunif.utils.alpha import AlphaBorderPadding
    from nunif.transforms.tta import tta_split, tta_merge
    g = torch.Generator().manual_seed(7)
    H, W = 45, 61
    rgb = torch.rand(3, H, W, generator=g)
    # alpha: two opaque blobs with soft edges, a hole, and a fully transparent corner region
    yy, xx = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
    a = torch.clamp(1.3 - ((yy - 14) ** 2 + (xx - 18) ** 2).sqrt() / 9, 0, 1)
    a = torch.maximum(a, torch.clamp(1.2 - ((yy - 33) ** 2 / 30 + (xx - 44) ** 2 / 90).sqrt(), 0, 1))
    a[12:16, 16:20] = 0
    alpha = a.unsqueeze(0)
    pad = AlphaBorderPadding().eval()
    out = {"rgb": rgb, "alpha": alpha}
    for off in (0, 1, 8, 17, 36):
        out[f"pad_{off}"] = pad(rgb, alpha, off)
    x = torch.rand(3, 22, 31, generator=g)
    views = tta_split(x)
    for k, v in enumerate(views):
        out[f"view_{k}"] = v.contiguous()
    zs = [torch.rand(v.shape, generator=g) * 1.2 - 0.1 for v in views]
    for k, z in enumerate(zs):
        out[f"z_{k}"] = z
    out["x"] = x
    out["merged"] = tta_merge(zs)
    out["merged_identity"] = tta_merge([v.clone() for v in views])
    save("alpha_tta", **out)


def gen_frames():
    """Frame conversions (nunif/utils/video.py, iw3/utils.py:274-289) and DepthAnything batch_preprocess."""
    # iw3/utils.py imports PyAV (absent in this image) at module scope, so the pure-tensor helper
    # hwc_to_chw_float (iw3/utils.py:274-289) is executed from the reference source file without importing the module.
    import ast
    src = open("/root/reference/iw3/utils.py").read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "hwc_to_chw_float")
    ns = {"torch": torch}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "/root/reference/iw3/utils.py", "exec"), ns)
    hwc_to_chw_float = ns["hwc_to_chw_float"]
    from iw3.depth_anything_model import batch_preprocess
    g = torch.Generator().manual_seed(11)
    out = {}
    u8 = torch.randint(0, 256, (2, 37, 53, 3), generator=g, dtype=torch.uint8)
    u16 = torch.randint(0, 65536, (37, 53, 3), generator=g, dtype=torch.int32).to(torch.uint16)
    out["u8"], out["u16"] = u8, u16.view(torch.int16)
    out["u8_f"] = hwc_to_chw_float(u8, "cpu")
    out["u16_f"] = hwc_to_chw_float(u16, "cpu")
    f = torch.rand(3, 41, 29, generator=g)
    f[0, 0, :8] = torch.tensor([0.5 / 255, 1.5 / 255, 2.5 / 255, 254.5 / 255, 0.0, 1.0, 0.49999 / 255, 127.5 / 255])
    out["f"] = f
    # from_tensor's tensor part (video.py:244)
    out["f_u8"] = (f.permute(1, 2, 0).contiguous() * 255.0).round_().to(torch.uint8)
    out["f_u16"] = (f.permute(1, 2, 0).contiguous() * 65535.0).round_().to(torch.uint16).view(torch.int16)
    x = torch.rand(2, 3, 135, 240, generator=g)
    out["x"] = x
    out["prep_126"] = batch_preprocess(x.clone(), lower_bound=126)
    out["prep_98_limit"] = batch_preprocess(x.clone(), lower_bound=392, limit_resolution=True)
    xt = torch.rand(1, 3, 300, 64, generator=g)   # tall: aspect cap + width floor
    out["xt"] = xt
    out["prep_tall"] = batch_preprocess(xt.clone(), lower_bound=70)
    sizes = []
    for (H, W) in ((1080, 1920), (2160, 3840), (720, 1280), (480, 854), (1920, 1080), (300, 3000), (100, 100), (393, 699)):
        for lb, lim in ((392, False), (518, False), (392, True), (224, True)):
            y = batch_preprocess(torch.zeros(1, 3, H, W), lower_bound=lb, limit_resolution=lim)
            sizes.append((H, W, lb, int(lim), y.shape[2], y.shape[3]))
    out["sizes"] = np.array(sizes, dtype=np.int64)
    # ZoeDepth batch_preprocess (iw3/zoedepth_model.py:30-85)
    from iw3.zoedepth_model import batch_preprocess as zoe_prep
    y, ph, pw = zoe_prep(x.clone(), h_height=96, v_height=128)
    out["zoe_land"], out["zoe_land_pad"] = y, np.array([ph, pw])
    y, ph, pw = zoe_prep(xt.clone(), h_height=96, v_height=128)
    out["zoe_port"], out["zoe_port_pad"] = y, np.array([ph, pw])
    zs = []
    for (H, W) in ((1080, 1920), (2160, 3840), (720, 1280), (480, 854), (1920, 1080), (300, 300), (200, 3000), (393, 699), (100, 64)):
        y, ph, pw = zoe_prep(torch.zeros(1, 3, H, W))
        zs.append((H, W, y.shape[2], y.shape[3], ph, pw))
    out["zoe_sizes"] = np.array(zs, dtype=np.int64)
    save("frames", **out)


def gen_row_flow():
    """sbs.row_flow_v3 (iw3/models/row_flow_v3.py) + apply_divergence_nn_LR (iw3/backward_warp.py:124-232), steps=1."""
    from nunif.models import create_model
    import iw3.models  # noqa: F401  (registers sbs.*)
    from iw3.backward_warp import apply_divergence_nn_LR, make_input_tensor
    m = create_model("sbs.row_flow_v3").eval()
    sd = synth.row_flow_v3_state_dict(0)
    m.load_state_dict(sd, strict=True)
    m.delta_output = True
    out = {}
    d = synth.synth_depth(3, 2, 70, 130)
    x = torch.stack([make_input_tensor(None, d[i], divergence=2.0, convergence=0.5, image_width=130) for i in range(2)])
    out["d"], out["x"] = d, x
    out["delta"] = m(x)[:, 0:1]
    c = torch.stack([synth.synth_image(4 + i, 3, 140, 260) for i in range(2)])
    out["c"] = c
    l, r = apply_divergence_nn_LR(m, c, d, 2.0, 0.5, steps=1, enable_amp=False)
    out["left"], out["right"] = l, r
    l, r = apply_divergence_nn_LR(m, c, d, 2.5, 0.3, steps=1, synthetic_view="right", enable_amp=False)
    out["sv_right_l"], out["sv_right_r"] = l, r
    d2 = synth.synth_depth(5, 1, 96, 192)                      # sizes that are already multiples of 12 / 96
    c2 = synth.synth_image(9, 3, 96, 192).unsqueeze(0)
    out["d2"], out["c2"] = d2, c2
    l, r = apply_divergence_nn_LR(m, c2, d2, 4.0, 0.6, steps=1, enable_amp=False)
    out["left2"], out["right2"] = l, r
    save("row_flow", **out)


def gen_row_flow_steps():
    """apply_divergence_nn_LR with steps > 1 (iterative re-warping of the depth, iw3/backward_warp.py:205-226) and with
    preserve_screen_border (make_input_tensor, :33-47) through the REAL sbs.row_flow_v3."""
    from nunif.models import create_model
    import iw3.models  # noqa: F401  (registers sbs.*)
    from iw3.backward_warp import apply_divergence_nn_LR
    m = create_model("sbs.row_flow_v3").eval()
    m.load_state_dict(synth.row_flow_v3_state_dict(0), strict=True)
    m.delta_output = True
    d = synth.synth_depth(3, 2, 70, 130)
    c = torch.stack([synth.synth_image(4 + i, 3, 140, 260) for i in range(2)])
    out = {"d": d, "c": c}
    out["s2_left"], out["s2_right"] = apply_divergence_nn_LR(m, c, d, 2.0, 0.5, steps=2, enable_amp=False)
    out["s3b_left"], out["s3b_right"] = apply_divergence_nn_LR(m, c, d, 4.0, 0.4, steps=3, preserve_screen_border=True, enable_amp=False)
    out["b_left"], out["b_right"] = apply_divergence_nn_LR(m, c, d, 5.0, 0.5, steps=1, synthetic_view="left", preserve_screen_border=True,
                                                            enable_amp=False)
    save("row_flow_steps", **out)


POSTPROCESS_CASES = [
    ("sbs", {}),
    ("half_sbs", {"half_sbs": True}),
    ("half_tb", {"half_tb": True}),
    ("tb", {"tb": True}),
    ("cross", {"cross_eyed": True}),
    ("ipd", {"ipd_offset": 3.0}),
    ("ipd_neg_pad_tblr", {"ipd_offset": -2.0, "pad": 0.1, "pad_mode": "tblr"}),
    ("pad_top", {"pad": 0.07, "pad_mode": "top"}),
    ("pad_169", {"pad_mode": "16:9"}),
    ("ana_wimmer2_half", {"anaglyph": "wimmer2", "half_sbs": True}),
    ("maxw", {"max_output_width": 200, "keep_aspect_ratio": True}),
    ("maxh_nokeep", {"max_output_height": 70}),
]


def gen_postprocess():
    """postprocess_image / postprocess_padding (iw3/utils.py:394-487) executed from the reference source (iw3/utils.py
    imports PyAV at module scope, which this image lacks, so the two functions are compiled out of the file by AST)."""
    import ast
    import types
    import torchvision.transforms.functional as TF
    from torchvision.transforms import InterpolationMode
    from iw3.anaglyph import apply_anaglyph_redcyan
    src = open("/root/reference/iw3/utils.py").read()
    fns = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name in ("postprocess_padding", "postprocess_image")]
    ns = {"torch": torch, "TF": TF, "InterpolationMode": InterpolationMode, "apply_anaglyph_redcyan": apply_anaglyph_redcyan,
          "equirectangular_projection": None}
    exec(compile(ast.Module(body=fns, type_ignores=[]), "/root/reference/iw3/utils.py", "exec"), ns)
    base = dict(ipd_offset=0, rgbd=False, half_rgbd=False, pad=None, pad_mode=None, vr180=False, half_sbs=False, half_tb=False, tb=False,
                cross_eyed=False, anaglyph=None, max_output_height=None, max_output_width=None, keep_aspect_ratio=False)
    g = torch.Generator().manual_seed(31)
    l = torch.rand(3, 90, 150, generator=g) * 1.1 - 0.05
    r = torch.rand(3, 90, 150, generator=g) * 1.1 - 0.05
    out = {"l": l, "r": r}
    for name, kw in POSTPROCESS_CASES:
        out["pp_" + name] = ns["postprocess_image"](l.clone(), r.clone(), types.SimpleNamespace(**{**base, **kw}))
    from iw3.equirectangular import equirectangular_projection
    out["vr180_l"] = equirectangular_projection(l.clamp(0, 1))
    save("postprocess", **out)


def gen_depth_scaler():
    """EMAMinMaxScaler (iw3/depth_scaler.py:64-142) over a sequence of frames, look-ahead buffering and flush included."""
    from iw3.depth_scaler import EMAMinMaxScaler
    g = torch.Generator().manual_seed(41)
    frames = [torch.rand(1, 12, 17, generator=g) * (1.0 + 0.5 * i) + 0.1 * ((-1) ** i) * i for i in range(9)]
    frames[4] = torch.zeros(1, 12, 17)        # an all-equal frame (scale == 0 branch of a stateless scaler)
    out = {"frames": torch.stack(frames)}
    for tag, kw in (("simple", dict(decay=0, buffer_size=1)), ("ema", dict(decay=0.75, buffer_size=1)),
                    ("window", dict(decay=0.9, buffer_size=4)), ("max", dict(decay=0.5, buffer_size=2, mode="max"))):
        sc = EMAMinMaxScaler(**kw)
        res = []
        for f in frames:
            r = sc.update(f)
            res.append(torch.full_like(f, float("nan")) if r is None else r)
        tail = sc.flush()
        out[tag + "_update"] = torch.stack(res)
        out[tag + "_flush"] = torch.stack(tail) if tail else torch.zeros(0, 1, 12, 17)
    save("depth_scaler", **out)


def gen_depth_aa():
    """iw3.depth_aa (iw3/models/depth_aa.py): forward (eval clamp) and infer."""
    from nunif.models import create_model
    import iw3.models  # noqa: F401
    m = create_model("iw3.depth_aa").eval()
    m.load_state_dict(synth.depth_aa_state_dict(0), strict=True)
    g = torch.Generator().manual_seed(51)
    x = torch.rand(2, 1, 70, 90, generator=g)
    xi = synth.synth_depth(7, 1, 98, 130) * 6.0 + 1.5
    save("depth_aa", x=x, y=m(x), xi=xi, yi=m.infer(xi))


def gen_mlbw():
    """sbs.mlbw (iw3/models/mlbw.py) in delta_output mode + apply_divergence_nn_LR -> apply_divergence_nn_delta_weight."""
    from nunif.models import create_model
    import iw3.models  # noqa: F401
    from iw3.backward_warp import apply_divergence_nn_LR, make_input_tensor
    m = create_model("sbs.mlbw").eval()
    m.load_state_dict(synth.mlbw_state_dict(0), strict=True)
    m.delta_output = True
    d = synth.synth_depth(3, 2, 70, 130)
    x = torch.stack([make_input_tensor(None, d[i], divergence=2.0, convergence=0.5, image_width=130) for i in range(2)])
    delta, lw = m(x)
    c = torch.stack([synth.synth_image(4 + i, 3, 140, 260) for i in range(2)])
    l, r = apply_divergence_nn_LR(m, c, d, 2.0, 0.5, steps=1, enable_amp=False)
    save("mlbw", d=d, x=x, delta=delta, layer_weight=lw, left=l, right=r)


def gen_mlbw_variants():
    """sbs.mlbw with num_layers=4 and the `small` layout (two blocks, shift along x only): delta / layer weights of the REAL model."""
    from nunif.models import create_model
    import iw3.models  # noqa: F401
    from iw3.backward_warp import make_input_tensor
    out = {}
    for tag, L, small, (B, h, w) in [("l4", 4, False, (1, 70, 130)), ("l2s", 2, True, (2, 33, 96))]:
        m = create_model("sbs.mlbw", num_layers=L, small=small).eval()
        sd = synth.mlbw_state_dict(1, num_layers=L)
        if small:
            sd = {k: v for k, v in sd.items() if not (k.startswith("lv2.2.") or k.startswith("lv2.3."))}
        m.load_state_dict(sd, strict=True)
        m.delta_output = True
        d = synth.synth_depth(7, B, h, w)
        x = torch.stack([make_input_tensor(None, d[i], divergence=2.5, convergence=0.4, image_width=max(h, w)) for i in range(B)])
        delta, lw = m(x)
        out[tag + "_delta"], out[tag + "_lw"] = delta, lw                    # _forward_delta_only (:232-240): L x-flow layers + weights
    save("mlbw_variants", **out)


def gen_zoedepth_infer():
    """The REAL iw3/zoedepth_model.py batch_infer (:89-148: batch_preprocess, flip TTA, crop of the reflection pad, dilation in
    negative space, negation) around a stand-in network: the third-party ZoeD_N module is replaced by the oracle's restatement
    (oracle/zoedepth.py, reduced widths) exposed through the same `model(x)['metric_depth']` interface, so the golden pins the
    reference's wrapper logic (SURVEY 8a row B4) while the network itself stays pinned to transformers (test_oracle_golden)."""
    from iw3.zoedepth_model import batch_infer as ref_batch_infer
    from oracle import zoedepth as oz
    sd = synth.zoedepth_state_dict(5, synth.ZOED_MINI)

    class Stub:
        device = torch.device("cpu")
        prep_h_height, prep_v_height, prep_mod = 96, 128, 32

        def __call__(self, x):
            return {"metric_depth": oz.zoedepth_forward(sd, x, oz.ZOED_MINI)}

    land = torch.stack([synth.synth_image(71 + i, 3, 180, 320, smooth=False) for i in range(2)])
    port = synth.synth_image(73, 3, 240, 160, smooth=False)
    out = {"land": land, "port": port}
    for flip in (0, 1):
        for dil in (0, 2):
            out[f"land_f{flip}_d{dil}"] = ref_batch_infer(Stub(), land.clone(), flip_aug=bool(flip), enable_amp=False, edge_dilation=dil)
            out[f"port_f{flip}_d{dil}"] = ref_batch_infer(Stub(), port.clone(), flip_aug=bool(flip), enable_amp=False, edge_dilation=dil)
    save("zoedepth_infer", **out)


def gen_transformers():
    """transformers' Depth-Anything-V2 and ZoeDepth models, the independent implementations the depth-network oracles are
    pinned to, on the seeded cases of tests/test_oracle_golden.py: the pin then holds without transformers installed."""
    import transformers
    from tests import test_oracle_golden as tog
    save("transformers_depth", depth_anything=tog.hf_depth_anything(*tog.da_case()), zoedepth=tog.hf_zoedepth(*tog.zoe_case()),
         transformers_version=np.asarray(transformers.__version__))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ["seam", "models", "iw3", "alpha_tta", "frames", "row_flow", "row_flow_steps", "postprocess", "depth_scaler",
                             "depth_aa", "mlbw", "mlbw_variants", "zoedepth_infer", "transformers"]
    if "seam" in which:
        gen_seam_config()
    if "models" in which:
        gen_models()
    if "iw3" in which:
        gen_iw3()
    if "alpha_tta" in which:
        gen_alpha_tta()
    if "frames" in which:
        gen_frames()
    if "row_flow" in which:
        gen_row_flow()
    if "row_flow_steps" in which:
        gen_row_flow_steps()
    if "postprocess" in which:
        gen_postprocess()
    if "depth_scaler" in which:
        gen_depth_scaler()
    if "depth_aa" in which:
        gen_depth_aa()
    if "mlbw" in which:
        gen_mlbw()
    if "mlbw_variants" in which:
        gen_mlbw_variants()
    if "zoedepth_infer" in which:
        gen_zoedepth_infer()
    if "transformers" in which:
        gen_transformers()
