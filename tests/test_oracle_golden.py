"""Pin the CPU oracle to the committed outputs of the real reference
(tests/golden/*.npz, produced by oracle/gen_golden.py).  CPU only."""
import importlib.util
import os
import numpy as np
import pytest
import torch

from nunif_b200 import synth
from oracle import seam_blending as osb
from oracle import cunet as ocu
from oracle import swin_unet as osw
from oracle import iw3 as oiw
from tests.util import load_golden

G = os.path.join(os.path.dirname(__file__), "golden")
torch.set_grad_enabled(False)


def load(name):
    return {k: v for k, v in np.load(os.path.join(G, name + ".npz")).items()}


def t(a):
    return torch.from_numpy(np.asarray(a))


def maxdiff(a, b):
    return float((t(a).double() - t(b).double()).abs().max())


def test_create_config_bit_exact():
    g = load("seam_config")
    for case, want in zip(g["cases"], g["configs"]):
        h, w, scale, offset, tile, blend = (int(v) for v in case)
        p = osb.create_config(h, w, scale, offset, tile, blend)
        got = [p["y_h"], p["y_w"], p["h_blocks"], p["w_blocks"], *p["pad"],
               p["y_buffer_h"], p["y_buffer_w"], p["input_tile_step"], p["output_tile_step"]]
        assert got == [int(v) for v in want], (case, got, want)


def test_survey_table_counts():
    # SURVEY.md section 8a A4: swin4x@256: 4K 10x17=170, 8K 19x33=627; upcunet 4K 10x18
    p = osb.create_config(2160, 3840, 4, 32, 256, 16)
    assert (p["h_blocks"], p["w_blocks"], p["input_tile_step"]) == (10, 17, 236)
    p = osb.create_config(4320, 7680, 2, 16, 256, 8)
    assert (p["h_blocks"], p["w_blocks"]) == (19, 33)
    p = osb.create_config(2160, 3840, 2, 36, 256, 0)
    assert (p["h_blocks"], p["w_blocks"], p["input_tile_step"]) == (10, 18, 220)


def test_blend_filter_bit_exact():
    g = load("seam_config")
    for k, v in g.items():
        if k.startswith("filter_"):
            scale, offset, tile, blend = (int(s) for s in k.split("_")[1:])
            f = osb.create_blend_filter(scale, offset, tile, blend, 3)
            assert torch.equal(f, t(v)), k


def test_find_valid_tile_size():
    g = load("tile_size")
    for q, c, s in zip(g["query"], g["cunet"], g["swin"]):
        assert osb.find_valid_tile_size(osb.cunet_tile_validator, int(q)) == int(c)
        assert osb.find_valid_tile_size(osb.swin_tile_validator, int(q)) == int(s)


@pytest.mark.parametrize("name,up", [("upcunet", True), ("cunet", False)])
def test_cunet_forward_and_render(name, up):
    g = load(name)
    sd = synth.upcunet_state_dict(0) if up else synth.cunet_state_dict(0)
    assert torch.equal(synth.synth_image(11, 3, 104, 104).unsqueeze(0), t(g["x"]))
    z = ocu.cunet_forward(sd, t(g["x"]), upscale=up)
    assert maxdiff(z, g["z"]) < 2e-5
    spec = ocu.UPCUNET if up else ocu.CUNET
    y = osb.tiled_render(t(g["img"]), lambda b: ocu.cunet_forward(sd, b, upscale=up),
                         spec["scale"], spec["offset"], spec["blend_size"], int(g["tile_size"]), int(g["batch_size"]))
    assert y.shape == t(g["render"]).shape
    assert maxdiff(y, g["render"]) < 2e-5


def test_swin_unet_4x_family():
    g = load("swin_unet_4x")
    sd = synth.swin_unet_state_dict(0, 4)
    x = t(g["x"])
    assert maxdiff(osw.swin_unet_forward(sd, x, 4), g["z4"]) < 5e-5
    assert maxdiff(osw.swin_unet_forward(sd, x, 4, 2), g["z2"]) < 5e-5
    assert maxdiff(osw.swin_unet_forward(sd, x, 4, 4), g["z1"]) < 5e-5
    y4 = osb.tiled_render(t(g["img"]), lambda b: osw.swin_unet_forward(sd, b, 4), 4, 32, 16, 64, 4)
    assert maxdiff(y4, g["render4"]) < 5e-5
    y2 = osb.tiled_render(t(g["img"]), lambda b: osw.swin_unet_forward(sd, b, 4, 2), 2, 16, 8, 64, 4)
    assert maxdiff(y2, g["render2"]) < 5e-5
    # closed-form (order independent) blend == raster-order reference (SURVEY 7.2)
    y4c = osb.tiled_render_closed_form(t(g["img"]), lambda b: osw.swin_unet_forward(sd, b, 4), 4, 32, 16, 64, 4)
    assert maxdiff(y4c, g["render4"]) < 5e-5


@pytest.mark.parametrize("sf", [1, 2])
def test_swin_unet_native(sf):
    g = load(f"swin_unet_{sf}x")
    sd = synth.swin_unet_state_dict(0, sf)
    assert maxdiff(osw.swin_unet_forward(sd, t(g["x"]), sf), g["z"]) < 5e-5


def test_bicubic_aa_weights_match_aten():
    import torch.nn.functional as F
    x = torch.rand(1, 1, 48, 48)
    for factor in (2, 4):
        starts, w = osw.bicubic_aa_weights(48, 48 // factor)
        # separable application
        taps = w.shape[1]
        idx = (starts.view(-1, 1) + torch.arange(taps).view(1, -1)).clamp(max=47)
        tmp = (x[0, 0][:, idx] * w.view(1, -1, taps)).sum(-1)             # H, out
        out = (tmp[idx, :] * w.view(-1, taps, 1)).sum(1)                   # out, out
        ref = F.interpolate(x, size=(48 // factor,) * 2, mode="bicubic", align_corners=False, antialias=True)[0, 0]
        assert float((out - ref).abs().max()) < 2e-6


def test_backward_warp():
    g = load("backward_warp")
    c, d_lo, d_hi = t(g["c"]), t(g["d_lo"]), t(g["d_hi"])
    for sv in ("both", "left", "right"):
        l, r = oiw.apply_divergence_grid_sample(c, d_lo, 2.0, 0.5, sv)
        assert maxdiff(l, g[f"bw_{sv}_l"]) < 2e-5 and maxdiff(r, g[f"bw_{sv}_r"]) < 2e-5
    l, r = oiw.apply_divergence_grid_sample(c, d_hi, 5.0, 0.3, "both")
    assert maxdiff(l, g["bw_hi_l"]) < 2e-5 and maxdiff(r, g["bw_hi_r"]) < 2e-5


def test_forward_warp_bit_exact():
    g = load("forward_warp")
    c, d_lo, d_hi = t(g["c"]), t(g["d_lo"]), t(g["d_hi"])
    for tag, depth, div, conv, wb in [("hi", d_hi, 4.0, 0.5, False), ("hi_wb", d_hi, 10.0, 0.3, True),
                                      ("lo", d_lo, 4.0, 0.5, False)]:
        for method in ("forward_fill", "forward"):
            l, r, lm, rm = oiw.forward_warp(c, depth, div, conv, fill=(method == "forward_fill"),
                                            return_mask=True, width_base=wb)
            for got, key in ((l, "l"), (r, "r"), (lm, "lm"), (rm, "rm")):
                assert maxdiff(got, g[f"fw_{tag}_{method}_{key}"]) == 0.0, (tag, method, key)
    for sv in ("left", "right"):
        l, r = oiw.forward_warp(c, d_hi, 2.0, 0.5, fill=True, synthetic_view=sv, width_base=False)
        assert maxdiff(l, g[f"fw_{sv}_l"]) == 0.0 and maxdiff(r, g[f"fw_{sv}_r"]) == 0.0
    l, r = oiw.forward_warp(t(g["cl"]), t(g["dl"]), 60.0, 0.0, fill=True, width_base=True)
    assert maxdiff(l, g["fw_long_l"]) == 0.0 and maxdiff(r, g["fw_long_r"]) == 0.0
    # the >100 px iteration cap really is exercised (unfilled cells stay negative)
    assert (t(g["fw_long_l"]) < 0).any() or (t(g["fw_long_r"]) < 0).any()


def test_dilation_minmax_mapper():
    g = load("dilation")
    x = t(g["x"])
    for key in g:
        if key.startswith("dil_"):
            n = [int(v) for v in key.split("_")[1:]]
            n = n[0] if len(n) == 1 else n
            assert maxdiff(oiw.dilate_edge(x, n), g[key]) < 1e-5, key
    mm = oiw.minmax_normalize(x[:1])[0]
    assert maxdiff(mm, g["minmax0"]) == 0.0
    assert maxdiff(oiw.mapper(mm, "div_6"), g["div_6"]) < 1e-6
    assert maxdiff(oiw.mapper(mm, "div_1"), g["div_1"]) < 1e-6
    with pytest.raises(ValueError):
        oiw.edge_dilation_parse("3")


def test_anaglyph():
    g = load("anaglyph")
    l, r = t(g["l"]), t(g["r"])
    assert maxdiff(oiw.dubois(l, r, True), g["dubois"]) < 1e-6
    assert maxdiff(oiw.dubois(l, r, False), g["dubois2"]) < 1e-6


def test_alpha_border_padding_oracle_matches_reference():
    from oracle import alpha_tta as oat
    g = load_golden("alpha_tta")
    for off in (0, 1, 8, 17, 36):
        got = oat.alpha_border_padding(g["rgb"], g["alpha"], off)
        # the reference sums its 3x3 box with a depthwise conv whose accumulation order is not specified
        assert np.abs(got - g[f"pad_{off}"]).max() < 2e-6, off


def test_tta_oracle_matches_reference():
    from oracle import alpha_tta as oat
    g = load_golden("alpha_tta")
    views = oat.tta_split(g["x"])
    for k in range(8):
        assert np.array_equal(views[k], g[f"view_{k}"]), k
    assert np.array_equal(oat.tta_merge([g[f"z_{k}"] for k in range(8)]), g["merged"])
    assert np.abs(oat.tta_merge(list(views)) - g["merged_identity"]).max() == 0


def test_frame_conversion_oracle_matches_reference():
    from oracle import frames as ofr
    g = load_golden("frames")
    assert np.array_equal(ofr.hwc_to_chw_float(g["u8"]), g["u8_f"])
    assert np.array_equal(ofr.hwc_to_chw_float(g["u16"].view(np.uint16)), g["u16_f"])
    assert np.array_equal(ofr.chw_float_to_hwc(g["f"]), g["f_u8"])
    assert np.array_equal(ofr.chw_float_to_hwc(g["f"], use_16bit=True), g["f_u16"].view(np.uint16))


def test_da_preprocess_oracle_matches_reference():
    from oracle import frames as ofr
    g = load_golden("frames")
    for H, W, lb, lim, nh, nw in g["sizes"]:
        assert ofr.preprocess_size(int(H), int(W), int(lb), 4, bool(lim)) == (int(nh), int(nw)), (H, W, lb, lim)
    # ATen's CPU kernel accumulates the separable passes in a different order: a few fp32 ulps
    assert np.abs(ofr.batch_preprocess(g["x"], lower_bound=126) - g["prep_126"]).max() < 3e-6
    assert np.abs(ofr.batch_preprocess(g["x"], lower_bound=392, limit_resolution=True) - g["prep_98_limit"]).max() < 3e-6
    assert np.abs(ofr.batch_preprocess(g["xt"], lower_bound=70) - g["prep_tall"]).max() < 3e-6


def _da_to_hf(sd, depth=12):
    """oracle (upstream Depth-Anything-V2 key names) -> transformers.DepthAnythingForDepthEstimation key names."""
    out = {}
    out["backbone.embeddings.cls_token"] = sd["pretrained.cls_token"]
    out["backbone.embeddings.mask_token"] = sd["pretrained.mask_token"]
    out["backbone.embeddings.position_embeddings"] = sd["pretrained.pos_embed"]
    out["backbone.embeddings.patch_embeddings.projection.weight"] = sd["pretrained.patch_embed.proj.weight"]
    out["backbone.embeddings.patch_embeddings.projection.bias"] = sd["pretrained.patch_embed.proj.bias"]
    for i in range(depth):
        p, q = f"pretrained.blocks.{i}.", f"backbone.encoder.layer.{i}."
        dim = sd[p + "norm1.weight"].shape[0]
        for n in ("norm1", "norm2"):
            out[q + n + ".weight"], out[q + n + ".bias"] = sd[p + n + ".weight"], sd[p + n + ".bias"]
        w, b = sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]
        for j, n in enumerate(("query", "key", "value")):
            out[q + f"attention.attention.{n}.weight"] = w[j * dim:(j + 1) * dim]
            out[q + f"attention.attention.{n}.bias"] = b[j * dim:(j + 1) * dim]
        out[q + "attention.output.dense.weight"], out[q + "attention.output.dense.bias"] = sd[p + "attn.proj.weight"], sd[p + "attn.proj.bias"]
        out[q + "layer_scale1.lambda1"], out[q + "layer_scale2.lambda1"] = sd[p + "ls1.gamma"], sd[p + "ls2.gamma"]
        for n in ("fc1", "fc2"):
            out[q + f"mlp.{n}.weight"], out[q + f"mlp.{n}.bias"] = sd[p + f"mlp.{n}.weight"], sd[p + f"mlp.{n}.bias"]
    out["backbone.layernorm.weight"], out["backbone.layernorm.bias"] = sd["pretrained.norm.weight"], sd["pretrained.norm.bias"]
    for i in range(4):
        out[f"neck.reassemble_stage.layers.{i}.projection.weight"] = sd[f"depth_head.projects.{i}.weight"]
        out[f"neck.reassemble_stage.layers.{i}.projection.bias"] = sd[f"depth_head.projects.{i}.bias"]
        if i != 2:
            out[f"neck.reassemble_stage.layers.{i}.resize.weight"] = sd[f"depth_head.resize_layers.{i}.weight"]
            out[f"neck.reassemble_stage.layers.{i}.resize.bias"] = sd[f"depth_head.resize_layers.{i}.bias"]
        out[f"neck.convs.{i}.weight"] = sd[f"depth_head.scratch.layer{i + 1}_rn.weight"]
        p, q = f"depth_head.scratch.refinenet{4 - i}.", f"neck.fusion_stage.layers.{i}."
        out[q + "projection.weight"], out[q + "projection.bias"] = sd[p + "out_conv.weight"], sd[p + "out_conv.bias"]
        for u in (1, 2):
            for cv in (1, 2):
                for wb in ("weight", "bias"):
                    out[q + f"residual_layer{u}.convolution{cv}.{wb}"] = sd[p + f"resConfUnit{u}.conv{cv}.{wb}"]
    s = "depth_head.scratch."
    for hf, up in (("conv1", "output_conv1"), ("conv2", "output_conv2.0"), ("conv3", "output_conv2.2")):
        out[f"head.{hf}.weight"], out[f"head.{hf}.bias"] = sd[s + up + ".weight"], sd[s + up + ".bias"]
    return out


DA_GRID = 6


def da_case():
    """(weights, input) of the Depth-Anything-V2 comparison with transformers."""
    sd = synth.depth_anything_v2_state_dict(3, pos_grid=DA_GRID)
    x = torch.randn(2, 3, 14 * DA_GRID, 14 * DA_GRID, generator=torch.Generator().manual_seed(5))
    return sd, x


def hf_depth_anything(sd, x):
    """transformers.DepthAnythingForDepthEstimation loaded with the oracle's weights: predicted depth for x."""
    from transformers import DepthAnythingConfig, DepthAnythingForDepthEstimation, Dinov2Config
    grid = DA_GRID
    cfg = DepthAnythingConfig(
        backbone_config=Dinov2Config(hidden_size=384, num_hidden_layers=12, num_attention_heads=6, mlp_ratio=4, image_size=14 * grid,
                                     patch_size=14, out_features=["stage3", "stage6", "stage9", "stage12"],
                                     reshape_hidden_states=False, apply_layernorm=True, layer_norm_eps=1e-6),
        reassemble_hidden_size=384, neck_hidden_sizes=[48, 96, 192, 384], fusion_hidden_size=64, head_hidden_size=32,
        patch_size=14, reassemble_factors=[4, 2, 1, 0.5])
    hf = DepthAnythingForDepthEstimation(cfg).eval()
    missing, unexpected = hf.load_state_dict(_da_to_hf(sd), strict=False)
    assert not unexpected and all("position_ids" in m or "rel" in m for m in missing), (missing, unexpected)
    with torch.no_grad():
        return hf(pixel_values=x).predicted_depth


def transformers_wants(key, fn, *args):
    """What transformers computes for a case: the output stored in tests/golden/transformers_depth.npz (oracle/gen_golden.py
    transformers), so the pin holds where the package is not installed, plus a fresh run where it is."""
    wants = [t(load("transformers_depth")[key])]
    if importlib.util.find_spec("transformers") is not None:
        wants.append(fn(*args))
    return wants


def test_depth_anything_oracle_matches_transformers():
    """The Depth-Anything-V2 network is third-party code that the reference fetches through torch.hub.  Pin the oracle's
    restatement against an independent public implementation (transformers), same weights."""
    from oracle import depth_anything as oda
    sd, x = da_case()
    with torch.no_grad():
        got = oda.depth_anything_forward(sd, x)
    for want in transformers_wants("depth_anything", hf_depth_anything, sd, x):
        assert got.shape == want.shape == (2, 14 * DA_GRID, 14 * DA_GRID)
        assert float(want.std()) > 0.1
        assert float((got - want).abs().max()) < 2e-4 * float(want.abs().max())


def test_zoe_preprocess_oracle_matches_reference():
    from oracle import frames as ofr
    g = load_golden("frames")
    for H, W, oh, ow, ph, pw in g["zoe_sizes"]:
        nh, nw, p_h, p_w, fh, fw = ofr.zoe_preprocess_size(int(H), int(W))
        assert (fh + 2 * p_h, fw + 2 * p_w, p_h, p_w) == (int(oh), int(ow), int(ph), int(pw)), (H, W)
    y, ph, pw = ofr.zoe_batch_preprocess(g["x"], 96, 128)
    assert (ph, pw) == tuple(g["zoe_land_pad"]) and np.abs(y - g["zoe_land"]).max() < 3e-6
    y, ph, pw = ofr.zoe_batch_preprocess(g["xt"], 96, 128)
    assert (ph, pw) == tuple(g["zoe_port_pad"]) and np.abs(y - g["zoe_port"]).max() < 3e-6


def test_row_flow_oracle_matches_reference():
    from oracle import row_flow as orf
    g = load_golden("row_flow")
    sd = synth.row_flow_v3_state_dict(0)
    with torch.no_grad():
        x = orf.make_input(t(g["d"]), 2.0, 0.5)
        assert torch.equal(x, t(g["x"]))
        assert float((orf.row_flow_delta(sd, x) - t(g["delta"])).abs().max()) < 1e-5
        l, r = orf.apply_divergence_nn_LR(sd, t(g["c"]), t(g["d"]), 2.0, 0.5)
        assert float((l - t(g["left"])).abs().max()) < 1e-5 and float((r - t(g["right"])).abs().max()) < 1e-5
        l, r = orf.apply_divergence_nn_LR(sd, t(g["c"]), t(g["d"]), 2.5, 0.3, "right")
        assert torch.equal(l, t(g["sv_right_l"])) and float((r - t(g["sv_right_r"])).abs().max()) < 1e-5
        l, r = orf.apply_divergence_nn_LR(sd, t(g["c2"]), t(g["d2"]), 4.0, 0.6)
        assert float((l - t(g["left2"])).abs().max()) < 1e-5 and float((r - t(g["right2"])).abs().max()) < 1e-5


def test_row_flow_steps_oracle_matches_reference():
    """steps > 1 and preserve_screen_border of apply_divergence_nn_LR, pinned against the real reference model."""
    from oracle import row_flow as orf
    g = load_golden("row_flow_steps")
    sd = synth.row_flow_v3_state_dict(0)
    c, d = t(g["c"]), t(g["d"])
    with torch.no_grad():
        l, r = orf.apply_divergence_nn_LR(sd, c, d, 2.0, 0.5, steps=2)
        assert float((l - t(g["s2_left"])).abs().max()) < 1e-5 and float((r - t(g["s2_right"])).abs().max()) < 1e-5
        l, r = orf.apply_divergence_nn_LR(sd, c, d, 4.0, 0.4, steps=3, preserve_screen_border=True)
        assert float((l - t(g["s3b_left"])).abs().max()) < 1e-5 and float((r - t(g["s3b_right"])).abs().max()) < 1e-5
        l, r = orf.apply_divergence_nn_LR(sd, c, d, 5.0, 0.5, "left", preserve_screen_border=True)
        assert float((l - t(g["b_left"])).abs().max()) < 1e-5 and torch.equal(r, t(g["b_right"]))


def test_mlbw_variants_oracle_matches_reference():
    """sbs.mlbw with 4 layers and the `small` layout against the real reference model (tests/golden/mlbw_variants.npz)."""
    from oracle import mlbw as om
    from oracle.row_flow import make_input
    g = load_golden("mlbw_variants")
    for tag, L, small, (B, h, w) in [("l4", 4, False, (1, 70, 130)), ("l2s", 2, True, (2, 33, 96))]:
        sd = synth.mlbw_state_dict(1, num_layers=L)
        if small:
            sd = {k: v for k, v in sd.items() if not (k.startswith("lv2.2.") or k.startswith("lv2.3."))}
        x = make_input(synth.synth_depth(7, B, h, w), 2.5, 0.4)
        with torch.no_grad():
            delta, lw = om.mlbw_delta(sd, x, num_layers=L, small=small)
        assert float((delta - t(g[tag + "_delta"])).abs().max()) < 1e-4, tag
        assert float((lw - t(g[tag + "_lw"])).abs().max()) < 1e-5, tag


def _pp_kwargs(kw):
    kw = dict(kw)
    if "anaglyph" in kw:
        kw["anaglyph_type"] = kw.pop("anaglyph")
    return kw


def test_anaglyph_family_and_postprocess_oracle_match_reference():
    from oracle import postprocess as opp
    g = load_golden("anaglyph")
    for kind in ("color", "gray", "half-color", "wimmer", "wimmer2"):
        got = opp.anaglyph(g["l"], g["r"], kind)
        assert np.abs(got - g[kind.replace("-", "_")]).max() < 1e-6, kind
    pg = load_golden("postprocess")
    cases = _postprocess_cases()
    dub = lambda l, r, cb: oiw.dubois(torch.from_numpy(l), torch.from_numpy(r), cb).numpy()   # noqa: E731
    for name, kw in cases:
        got = opp.postprocess_image(pg["l"], pg["r"], dubois=dub, **_pp_kwargs(kw))
        want = pg["pp_" + name]
        assert got.shape == want.shape, (name, got.shape, want.shape)
        assert np.abs(got - want).max() < 1e-5, (name, np.abs(got - want).max())   # fractional-scale AA weights: fp32 order


def _postprocess_cases():
    """POSTPROCESS_CASES of oracle/gen_golden.py without importing it (it imports the reference tree)."""
    import ast
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "gen_golden.py")).read()
    for node in ast.parse(src).body:
        if isinstance(node, ast.Assign) and getattr(node.targets[0], "id", "") == "POSTPROCESS_CASES":
            return ast.literal_eval(node.value)
    raise AssertionError("POSTPROCESS_CASES not found")


def test_ema_minmax_scaler_oracle_matches_reference():
    """Stateful normaliser of --ema-normalize (SURVEY 8f rank 4): pinned now, ported in a later round."""
    from oracle.depth_scaler import EMAMinMaxScaler
    g = load_golden("depth_scaler")
    frames = g["frames"]
    for tag, kw in (("simple", dict(decay=0, buffer_size=1)), ("ema", dict(decay=0.75, buffer_size=1)),
                    ("window", dict(decay=0.9, buffer_size=4)), ("max", dict(decay=0.5, buffer_size=2, mode="max"))):
        sc = EMAMinMaxScaler(**kw)
        for i, f in enumerate(frames):
            r = sc.update(f)
            want = g[tag + "_update"][i]
            if r is None:
                assert np.isnan(want).all(), (tag, i)
            else:
                assert np.abs(r - want).max() < 1e-6, (tag, i, np.abs(r - want).max())
        tail = sc.flush()
        assert len(tail) == g[tag + "_flush"].shape[0], tag
        for r, want in zip(tail, g[tag + "_flush"]):
            assert np.abs(r - want).max() < 1e-6, tag


def test_equirectangular_oracle_matches_reference():
    """VR180 projection (iw3/equirectangular.py): pinned now, ported in a later round."""
    from oracle import postprocess as opp
    g = load_golden("postprocess")
    got = opp.equirectangular_projection(np.clip(g["l"], 0, 1))
    want = g["vr180_l"]
    assert got.shape == want.shape
    d = np.abs(got - want)
    assert d.max() < 5e-5 and d.mean() < 1e-6, (d.max(), d.mean())


def test_depth_aa_oracle_matches_reference():
    """iw3.depth_aa learned post-filter (SURVEY 8f rank 4): pinned now, ported in a later round."""
    from oracle import depth_aa as oaa
    g = load_golden("depth_aa")
    sd = synth.depth_aa_state_dict(0)
    with torch.no_grad():
        assert float((oaa.depth_aa_forward(sd, t(g["x"])) - t(g["y"])).abs().max()) < 1e-5
        yi = oaa.depth_aa_infer(sd, t(g["xi"]))
        assert float((yi - t(g["yi"])).abs().max()) < 1e-4 * float(t(g["yi"]).abs().max())


def test_mlbw_oracle_matches_reference():
    """sbs.mlbw multi-layer learned warp (SURVEY 8f rank 2): pinned now, ported in a later round."""
    from oracle import mlbw as om
    g = load_golden("mlbw")
    sd = synth.mlbw_state_dict(0)
    c = torch.stack([synth.synth_image(4 + i, 3, 140, 260) for i in range(2)])
    with torch.no_grad():
        delta, lw = om.mlbw_delta(sd, t(g["x"]))
        assert float((delta - t(g["delta"])).abs().max()) < 1e-5 and float((lw - t(g["layer_weight"])).abs().max()) < 1e-6
        l = om.apply_divergence_mlbw(sd, c, t(g["d"]), 2.0, 0.5, -1)
        r = om.apply_divergence_mlbw(sd, c, t(g["d"]), 2.0, 0.5, 1)
        assert float((l - t(g["left"])).abs().max()) < 1e-5 and float((r - t(g["right"])).abs().max()) < 1e-5


def _zoe_to_hf(sd, cfg):
    """oracle (upstream ZoeD_M12_N.pt key names) -> transformers.ZoeDepthForDepthEstimation key names (the published
    conversion table: q/k/v split of attn.qkv, gamma -> lambda, act_postprocess -> reassemble stage, refinenet{4-i} ->
    fusion layer i, output_conv -> relative_head, _net.{0,2} -> conv{1,2})."""
    out = {}
    bb, pp, sc = "core.core.pretrained.model.", "core.core.pretrained.", "core.core.scratch."
    dim = cfg["dim"]
    out["backbone.embeddings.cls_token"] = sd[bb + "cls_token"]
    out["backbone.embeddings.patch_embeddings.projection.weight"] = sd[bb + "patch_embed.proj.weight"]
    out["backbone.embeddings.patch_embeddings.projection.bias"] = sd[bb + "patch_embed.proj.bias"]
    for i in range(cfg["depth"]):
        p, q = f"{bb}blocks.{i}.", f"backbone.encoder.layer.{i}."
        out[q + "lambda_1"], out[q + "lambda_2"] = sd[p + "gamma_1"], sd[p + "gamma_2"]
        for a, b in (("norm1", "layernorm_before"), ("norm2", "layernorm_after")):
            out[q + b + ".weight"], out[q + b + ".bias"] = sd[p + a + ".weight"], sd[p + a + ".bias"]
        w = sd[p + "attn.qkv.weight"]
        for j, n in enumerate(("query", "key", "value")):
            out[q + f"attention.attention.{n}.weight"] = w[j * dim:(j + 1) * dim]
        out[q + "attention.attention.query.bias"] = sd[p + "attn.q_bias"]
        out[q + "attention.attention.value.bias"] = sd[p + "attn.v_bias"]
        out[q + "attention.attention.relative_position_bias.relative_position_bias_table"] = sd[p + "attn.relative_position_bias_table"]
        out[q + "attention.output.dense.weight"], out[q + "attention.output.dense.bias"] = sd[p + "attn.proj.weight"], sd[p + "attn.proj.bias"]
        out[q + "intermediate.dense.weight"], out[q + "intermediate.dense.bias"] = sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"]
        out[q + "output.dense.weight"], out[q + "output.dense.bias"] = sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"]
    for i in range(4):
        p = f"{pp}act_postprocess{i + 1}."
        for wb in ("weight", "bias"):
            out[f"neck.reassemble_stage.readout_projects.{i}.0.{wb}"] = sd[p + "0.project.0." + wb]
            out[f"neck.reassemble_stage.layers.{i}.projection.{wb}"] = sd[p + "3." + wb]
            if i != 2:
                out[f"neck.reassemble_stage.layers.{i}.resize.{wb}"] = sd[p + "4." + wb]
        out[f"neck.convs.{i}.weight"] = sd[f"{sc}layer{i + 1}_rn.weight"]
        p, q = f"{sc}refinenet{4 - i}.", f"neck.fusion_stage.layers.{i}."
        for wb in ("weight", "bias"):
            out[q + "projection." + wb] = sd[p + "out_conv." + wb]
            for u in (1, 2):
                for cv in (1, 2):
                    out[q + f"residual_layer{u}.convolution{cv}.{wb}"] = sd[p + f"resConfUnit{u}.conv{cv}.{wb}"]
    for wb in ("weight", "bias"):
        for hf, up in (("conv1", "0"), ("conv2", "2"), ("conv3", "4")):
            out[f"relative_head.{hf}.{wb}"] = sd[f"{sc}output_conv.{up}.{wb}"]
        out["metric_head.conv2." + wb] = sd["conv2." + wb]
        mods = ["seed_bin_regressor", "seed_projector"] + [f"projectors.{i}" for i in range(4)] + [f"attractors.{i}" for i in range(4)]
        for m in mods:
            out[f"metric_head.{m}.conv1.{wb}"] = sd[f"{m}._net.0.{wb}"]
            out[f"metric_head.{m}.conv2.{wb}"] = sd[f"{m}._net.2.{wb}"]
        for j in (0, 2):
            out[f"metric_head.conditional_log_binomial.mlp.{j}.{wb}"] = sd[f"conditional_log_binomial.mlp.{j}.{wb}"]
    return out


def zoe_case():
    """(weights, input) of the ZoeD_N comparison with transformers: non-square, so the relative-position table is resampled."""
    sd = synth.zoedepth_state_dict(3, synth.ZOED_MINI)
    x = torch.randn(2, 3, 64, 96, generator=torch.Generator().manual_seed(5))
    return sd, x


def hf_zoedepth(sd, x):
    """transformers.ZoeDepthForDepthEstimation at the reduced widths of ZOED_MINI, loaded with the oracle's weights."""
    from transformers import ZoeDepthConfig, ZoeDepthForDepthEstimation, BeitConfig
    from oracle import zoedepth as oz
    cfg = oz.ZOED_MINI
    hf_cfg = ZoeDepthConfig(
        backbone_config=BeitConfig(image_size=16 * cfg["old_grid"], patch_size=16, hidden_size=cfg["dim"], num_hidden_layers=cfg["depth"],
                                   num_attention_heads=cfg["heads"], intermediate_size=4 * cfg["dim"], use_relative_position_bias=True,
                                   use_absolute_position_embeddings=False, use_mask_token=False, layer_scale_init_value=0.1,
                                   reshape_hidden_states=False, layer_norm_eps=1e-6,
                                   out_features=[f"stage{h + 1}" for h in cfg["hooks"]]),
        neck_hidden_sizes=list(cfg["oc"]), fusion_hidden_size=cfg["feat"], bottleneck_features=cfg["feat"], readout_type="project",
        reassemble_factors=[4, 2, 1, 0.5], num_relative_features=32, bin_embedding_dim=128, num_attractors=[16, 8, 4, 1],
        bin_centers_type="softplus", bin_configurations=[{"n_bins": 64, "min_depth": 0.001, "max_depth": 10.0}])
    hf = ZoeDepthForDepthEstimation(hf_cfg).eval()
    missing, unexpected = hf.load_state_dict(_zoe_to_hf(sd, cfg), strict=False)
    assert not unexpected and all("relative_position_index" in m or "k_idx" in m or "k_minus_1" in m for m in missing), (missing, unexpected)
    with torch.no_grad():
        return hf(pixel_values=x).predicted_depth


def test_zoedepth_oracle_matches_transformers():
    """ZoeD_N (BEiT-L + DPT + metric bins) is third-party code that the reference fetches through torch.hub.  Pin the oracle's
    restatement against an independent public implementation (transformers), same weights, on a non-square input so that
    the relative-position table is resampled."""
    from oracle import zoedepth as oz
    sd, x = zoe_case()
    with torch.no_grad():
        got = oz.zoedepth_forward(sd, x, oz.ZOED_MINI)[:, 0]
    for want in transformers_wants("zoedepth", hf_zoedepth, sd, x):
        assert got.shape == want.shape == (2, 64, 96)
        assert float(want.std()) > 0.05
        assert float((got - want).abs().max()) < 2e-4 * float(want.abs().max())


def test_zoedepth_batch_infer_oracle_matches_reference():
    """oracle/zoedepth.batch_infer against the REAL iw3/zoedepth_model.batch_infer (golden generated around a stand-in network,
    oracle/gen_golden.py:gen_zoedepth_infer): preprocessing incl. the square-padded portrait case, flip TTA, pad crop,
    dilation in negative space, negation, single-image squeeze."""
    from oracle import zoedepth as oz
    g = load_golden("zoedepth_infer")
    sd = synth.zoedepth_state_dict(5, synth.ZOED_MINI)
    with torch.no_grad():
        for flip in (0, 1):
            for dil in (0, 2):
                got = oz.batch_infer(sd, t(g["land"]), flip_aug=bool(flip), edge_dilation=dil, h_height=96, v_height=128, cfg=oz.ZOED_MINI)
                want = t(g[f"land_f{flip}_d{dil}"])
                assert got.shape == want.shape and float((got - want).abs().max()) < 2e-4 * float(want.abs().max()), (flip, dil)
                got = oz.batch_infer(sd, t(g["port"]).unsqueeze(0), flip_aug=bool(flip), edge_dilation=dil, h_height=96, v_height=128,
                                     cfg=oz.ZOED_MINI)[0]
                want = t(g[f"port_f{flip}_d{dil}"])
                assert got.shape == want.shape and float((got - want).abs().max()) < 2e-4 * float(want.abs().max()), (flip, dil)
