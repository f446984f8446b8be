#!/usr/bin/env python
"""bench.py - the driver's measurement contract for nunif_b200.

Default workload (BASELINE.json configs[1]): waifu2x swin_unet/art scale4x, one synthetic 4K
(3x2160x3840) frame per step through `tiled_render(tile_size=256, batch_size=16)` = 170 tiles,
random-init weights (seed 0), fp16 tensor-core compute.  Metric = input megapixels / second.

  python bench.py --gpus N --steps K --warmup W            # this repo's engine (one rank per GPU under torchrun)
  python bench.py --impl reference ...                      # the reference algorithm on the host CPU cores (oracle port)
  python bench.py --dump-outputs DIR ...                    # also write the last timed step's output to DIR/*.npy

One JSON line is printed by rank 0.  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME = {"4k": (2160, 3840), "1080p": (1080, 1920), "8k": (4320, 7680)}
TILE, BATCH = 256, 16
# --workload: (model variant, frame, name in the JSON line).  swin4x_4k is BASELINE.json configs[1] (the headline);
# swin2x_4k the north-star `to_2x` path on the same frame; swin2x_8k configs[3] (one 8K frame per GPU).
WORKLOADS = {
    "swin4x_4k": dict(down=1, frame="4k", text="waifu2x swin_unet/art scale4x"),
    "swin2x_4k": dict(down=2, frame="4k", text="waifu2x swin_unet/art scale2x (SwinUNet4x.to_2x: 4x network + antialiased bicubic /2)"),
    "swin2x_8k": dict(down=2, frame="8k", text="waifu2x swin_unet/photo scale2x (SwinUNet4x.to_2x), 8K frame per GPU (configs[3])"),
}
# iw3 workloads (BASELINE.json configs[2] and configs[4]): a step = one batch of frames through depth model -> dilation ->
# min/max (+ mapper) -> warp -> composed stereo frame; metric = frames/s
IW3_WORKLOADS = {
    "iw3_1080p": dict(frame="1080p", batch=4, depth="Any_V2_S", method="forward_fill", mapper="none", anaglyph=None, edge_dilation=[2, 1],
                      text="iw3 Depth-Anything-V2-Small + dilate_edge [2,1] + forward_fill warp + SBS, 1080p stream (configs[2])"),
    "iw3_4k_zoe": dict(frame="4k", batch=2, depth="ZoeD_N", method="backward", mapper="div_6", anaglyph="dubois", edge_dilation=2,
                       text="iw3 ZoeD_N (BEiT-L) + dilate_edge 2 + backward (grid_sample) warp + dubois anaglyph, 4K stream (configs[4])"),
}
SWIN4X_TILE_GFLOP = 155.7           # BASELINE.md section 2 (conv 8.6 + addmm 140.1 + bmm 7.0)
# --dump-outputs keeps at most this many float32 values in all (32 MiB): the 4K swin4x output alone is 4e8 values (1.6 GB)
DUMP_ELEMS = 1 << 23


def dump_outputs(path, outputs, seed=0):
    """Write each output tensor as <path>/<name>.npy in float32: whole if it fits its share of DUMP_ELEMS, otherwise that many
    flat elements at sorted indices drawn from a generator seeded with `seed`, so two runs with the same arguments (two builds
    of the project) dump the same positions.  Returns {name: {"shape": full shape, "dumped": elements written}}."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    share = DUMP_ELEMS // len(outputs)
    info = {}
    for name, t in outputs.items():
        if t.numel() > share:
            idx = torch.randint(t.numel(), (share,), generator=torch.Generator().manual_seed(seed)).sort().values
            a = t.reshape(-1)[idx.to(t.device)]
        else:
            a = t
        np.save(os.path.join(path, name + ".npy"), a.float().cpu().numpy())
        info[name] = {"shape": list(t.shape), "dumped": a.numel()}
    return info


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mx = max(int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_reference_sample(n_tiles, threads):
    """The reference algorithm on the CPU (oracle port, fp32 like nunif/device.py:59-65 on CPU):
    n_tiles 256x256 tiles of swin_unet_4x through model(minibatch).  Returns seconds."""
    import torch
    from nunif_b200 import synth
    from oracle import swin_unet as osw
    torch.set_num_threads(threads)
    sd = synth.swin_unet_state_dict(0, 4)
    x = torch.stack([synth.synth_image(100 + i, 3, TILE, TILE) for i in range(n_tiles)])
    with torch.inference_mode():
        t0 = time.perf_counter()
        osw.swin_unet_forward(sd, x, 4)
        return time.perf_counter() - t0


def cpu_worker_main(n_tiles, threads):
    """`bench.py --cpu-worker N T`: one tile batch on T threads; prints wall-clock start / end (time.time) as JSON."""
    import torch
    from nunif_b200 import synth
    from oracle import swin_unet as osw
    torch.set_num_threads(threads)
    sd = synth.swin_unet_state_dict(0, 4)
    x = torch.stack([synth.synth_image(100 + i, 3, TILE, TILE) for i in range(n_tiles)])
    with torch.inference_mode():
        osw.swin_unet_forward(sd, x[:1, :, :64, :64].contiguous(), 4)     # warm: allocator, oneDNN primitives
        t0 = time.time()
        osw.swin_unet_forward(sd, x, 4)
        t1 = time.time()
    print(json.dumps({"t0": t0, "t1": t1}), flush=True)


def cpu_reference_concurrent(workers, tiles_per_worker, threads):
    """`workers` processes, each pushing one batch of `tiles_per_worker` tiles through the model on `threads` threads at the
    same time - how a CPU run of the reference keeps a many-core host busy (one torch process scales poorly past a few dozen
    threads on the small per-tile GEMMs).  Returns (seconds from the first start to the last finish, tiles done)."""
    procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-worker", str(tiles_per_worker), str(threads)],
                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
                              env={**os.environ, "OMP_NUM_THREADS": str(threads), "MKL_NUM_THREADS": str(threads)})
             for _ in range(workers)]
    spans = []
    for pr in procs:
        out, _ = pr.communicate()
        lines = [ln for ln in out.splitlines() if ln.startswith("{")]
        if pr.returncode == 0 and lines:
            spans.append(json.loads(lines[-1]))
    if not spans:
        raise RuntimeError("CPU reference workers failed")
    return max(sp["t1"] for sp in spans) - min(sp["t0"] for sp in spans), len(spans) * tiles_per_worker


def cpu_plan(cores):
    """(workers, threads per worker): at least 8 concurrent tile batches, every core used."""
    workers = 8 if cores >= 16 else max(1, cores // 2)
    return workers, max(1, cores // workers)


def frame_tiles(h, w, scale=4, offset=32, blend=16):
    """Tiles per frame from the library's host integer planner (nb200_tile_config_create == SeamBlending.create_config)."""
    from nunif_b200.nunif.render import create_config
    cfg = create_config((h, w), scale, offset, TILE, blend)
    return cfg["h_blocks"] * cfg["w_blocks"]


def cpu_baseline_object(h, w, ntiles, tiles_per_worker=1):
    cores = host_cores()
    workers, threads = cpu_plan(cores)
    t, done = cpu_reference_concurrent(workers, tiles_per_worker, threads)
    mp = h * w / 1e6
    val = mp * done / ntiles / t
    return t, {"value": val, "unit": "MP/s", "cores": workers * threads, "kind": "port", "host_cores": cores,
               "workers": workers, "threads_per_worker": threads,
               "sample": f"{done} of the {ntiles} 256x256 tiles of one frame: {workers} concurrent processes x {tiles_per_worker} tile(s) "
                         f"through oracle/swin_unet.py (torch-CPU fp32, {threads} threads each), {t:.1f} s wall from first start "
                         f"to last finish; MP/s = frame MP * {done}/{ntiles} / t"}


def _default_frame(args):
    if args.frame is None:
        args.frame = WORKLOADS[args.workload]["frame"]


def run_reference(args):
    """The reference arm: the reference's algorithm (oracle port; the reference itself is Python with no installable package
    and cannot travel to the GPU box) on ALL host cores - several tile batches at a time, every core busy."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _default_frame(args)
    h, w = FRAME[args.frame]
    ntiles = frame_tiles(h, w)
    ts, cb = [], None
    for _ in range(max(1, args.steps)):
        t, cb = cpu_baseline_object(h, w, ntiles)
        ts.append((t, cb["value"]))
    val = sum(v for _, v in ts) / len(ts)
    t = sum(tt for tt, _ in ts) / len(ts)
    cb["value"] = val
    line = {
        "impl": "reference", "metric": "waifu2x_input_megapixels_per_sec", "value": val, "unit": "MP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"waifu2x swin_unet/art scale4x, {args.frame} input 3x{h}x{w}, tile_size=256 batch=16, "
                               f"{ntiles} tiles/frame, 1 frame/GPU/step",
                   "warmup_note": "each worker warms its allocator / oneDNN primitives on a 64x64 tile before its timed batch"},
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_torch_gpu(args):
    """`--impl torch_gpu`: what the reference itself does on a CUDA device - its PyTorch modules (oracle restatement, same ops)
    under torch.autocast(fp16) (nunif/device.py:58-71), eager or torch.compile'd (waifu2x/utils.py:25-39 `compile`), through
    the reference's tiling loop (oracle/seam_blending.py) with the frame resident in HBM.  Same metric and workload as the
    default arm; a BASELINE only (SURVEY 8d / BASELINE.md section 3), never part of the product path."""
    import torch
    from nunif_b200 import synth
    from oracle import swin_unet as osw, seam_blending as osb
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    _default_frame(args)
    h, w = FRAME[args.frame]
    ntiles = frame_tiles(h, w)
    sd = {k: v.to(dev) for k, v in synth.swin_unet_state_dict(0, 4).items()}
    x = synth.synth_image(1000, 3, h, w, smooth=False).to(dev)

    def fwd(b):
        return osw.swin_unet_forward(sd, b, 4)
    model = torch.compile(fwd) if args.compile else fwd

    def amp_model(b):
        with torch.autocast("cuda", dtype=torch.float16):
            return model(b.to(dev))

    def step():
        return osb.tiled_render(x, amp_model, 4, 32, 16, TILE, BATCH)
    with torch.no_grad():
        for _ in range(max(1, args.warmup)):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(dev.index or 0) as clocks:
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    val = args.steps * (h * w / 1e6) / (ms / 1e3)
    print(json.dumps({
        "impl": "torch_gpu", "metric": "waifu2x_input_megapixels_per_sec", "value": val, "unit": "MP/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic", "clocks": clocks.summary(),
        "config": {"workload": f"waifu2x swin_unet/art scale4x, {args.frame} input 3x{h}x{w}, tile_size=256 batch=16, {ntiles} tiles/frame",
                   "engine": "PyTorch " + torch.__version__ + (" torch.compile" if args.compile else " eager") + ", torch.autocast(fp16)",
                   "frames_per_sec": args.steps / (ms / 1e3)}}), flush=True)


def bench_iw3(dev, lib, peaks_gbs, B=4, iters=20):
    """Secondary numbers (BASELINE.json configs[2], post-depth stages only - the DepthAnything body is not part of this
    round): dilate_edge[2,1] + per-frame min/max + warp + SBS compose on B 1080p frames resident in HBM, device-timed.
    Algorithmic bytes per frame (SURVEY.md 8d): (3 in + 6 out planes) * 4 B * H*W + the depth map = 75.7 MB."""
    import ctypes
    import torch
    from nunif_b200 import synth, _lib
    from nunif_b200.iw3 import stereo_sbs
    H, W, h, w = 1080, 1920, 392, 686
    c = torch.stack([synth.synth_image(50 + i, 3, H, W, smooth=False) for i in range(B)]).to(dev)
    d = synth.synth_depth(60, B, h, w).to(dev) * 7.0 + 0.5
    out = {}
    for method in ("forward_fill", "backward"):
        for _ in range(3):
            y = stereo_sbs(c, d, 2.0, 0.5, method=method, edge_dilation=[2, 1])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            y = stereo_sbs(c, d, 2.0, 0.5, method=method, edge_dilation=[2, 1])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        _lib.check(lib.nb200_profile_enable(1))
        y = stereo_sbs(c, d, 2.0, 0.5, method=method, edge_dilation=[2, 1])
        buf = ctypes.create_string_buffer(8192)
        _lib.check(lib.nb200_profile_report(buf, 8192))
        _lib.check(lib.nb200_profile_enable(0))
        prof = json.loads(buf.value.decode())
        k = prof.get("forward_warp" if method == "forward_fill" else "backward_warp", {"ms": 0, "work": 0})
        gbs = k["work"] / (k["ms"] / 1e3) / 1e9 if k["ms"] > 0 else 0.0
        out[method] = {"fps": B / (ms / 1e3), "ms_per_batch": ms, "batch": B,
                       "warp_kernel_ms": k["ms"], "warp_kernel_GBps_algorithmic": gbs, "warp_frac_of_hbm_peak": gbs / peaks_gbs,
                       "kernel_classes_ms": {kk: round(v["ms"], 4) for kk, v in prof.items()}}
        del y
    out["note"] = "forward_fill / backward: post-depth stages only (dilate_edge [2,1], minmax, warp, SBS) on a synthetic depth map"
    # ---- the whole per-frame path of BASELINE configs[2]: Depth-Anything-V2-S (seeded weights) at resolution 392 +
    # dilate_edge [2,1] + min/max + forward_fill warp + SBS, frames resident in HBM as float CHW
    from nunif_b200.iw3 import DepthAnythingModel
    dam = DepthAnythingModel().load_state_dict(synth.depth_anything_v2_state_dict(0), gpu=dev.index or 0)

    def full(method):
        with torch.inference_mode():
            depth = dam.infer(c, edge_dilation=[2, 1])
            return stereo_sbs(c, depth, 2.0, 0.5, method=method, edge_dilation=0, side_model=rfm)
    from nunif_b200.iw3 import RowFlowV3
    rfm = RowFlowV3(synth.row_flow_v3_state_dict(0), dev)
    for method in ("forward_fill", "backward", "row_flow_v3"):
        for _ in range(3):
            y = full(method)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            y = full(method)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        _lib.check(lib.nb200_profile_enable(1))
        y = full(method)
        buf = ctypes.create_string_buffer(8192)
        _lib.check(lib.nb200_profile_report(buf, 8192))
        _lib.check(lib.nb200_profile_enable(0))
        prof = json.loads(buf.value.decode())
        out["with_depth_" + method] = {"fps": B / (ms / 1e3), "ms_per_batch": ms, "batch": B,
                                       "depth_model": "Depth-Anything-V2 ViT-S (seeded random weights), 392x686 network input",
                                       "kernel_classes_ms": {kk: round(v["ms"], 4) for kk, v in prof.items()}}
        del y
    # ---- BASELINE configs[4] warp stage: 4K frame, grid_sample warp with the fused dubois anaglyph epilogue
    c4k = torch.stack([synth.synth_image(90 + i, 3, 2160, 3840, smooth=False) for i in range(2)]).to(dev)
    d4k = synth.synth_depth(61, 2, 384, 704).to(dev)

    def ana():
        return stereo_sbs(c4k, d4k, 2.0, 0.5, method="backward", mapper="div_6", edge_dilation=[2, 1], anaglyph="dubois")
    for _ in range(3):
        y = ana()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        y = ana()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    out["backward_dubois_4k"] = {"fps": 2 / (ms / 1e3), "ms_per_batch": ms, "batch": 2,
                                 "note": "post-depth stages of configs[4] only (dilate_edge, minmax + div_6 mapper, grid_sample warp, dubois) on a synthetic depth map"}
    del y, d4k
    # ---- the whole per-frame path of BASELINE configs[4]: ZoeD_N (BEiT-L, seeded weights) at 384x704 + dilate_edge 2 + min/max +
    # div_6 mapper + grid_sample warp + dubois anaglyph on two 4K frames resident in HBM (the standalone line is --workload iw3_4k_zoe)
    from nunif_b200.iw3 import ZoeDepthModel
    zm = ZoeDepthModel("ZoeD_N").load_state_dict(synth.zoedepth_state_dict(0), gpu=dev.index or 0)

    def zoe_ana():
        with torch.inference_mode():
            depth = zm.infer(c4k, edge_dilation=2)
            return stereo_sbs(c4k, depth, 2.0, 0.5, method="backward", mapper="div_6", edge_dilation=0, anaglyph="dubois")
    for _ in range(3):
        y = zoe_ana()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        y = zoe_ana()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    _lib.check(lib.nb200_profile_enable(1))
    y = zoe_ana()
    buf = ctypes.create_string_buffer(8192)
    _lib.check(lib.nb200_profile_report(buf, 8192))
    _lib.check(lib.nb200_profile_enable(0))
    prof = json.loads(buf.value.decode())
    out["zoe_anaglyph_4k"] = {"fps": 2 / (ms / 1e3), "ms_per_batch": ms, "batch": 2,
                              "depth_model": "ZoeD_N = BEiT-L/16 + DPT + metric bins (seeded random weights), 384x704 network input",
                              "kernel_classes_ms": {kk: round(v["ms"], 4) for kk, v in prof.items()}}
    del y, c4k, zm
    # ---- the same path end to end from HOST uint8 frames (video.py to_tensor / from_tensor edges): pinned uint8 HWC in,
    # H2D, uint8->float CHW, depth, warp, SBS, float->uint8 HWC, D2H of the SBS frames
    from nunif_b200.iw3 import hwc_to_chw_float, chw_float_to_hwc
    u8_in = (c.permute(0, 2, 3, 1) * 255.0).round().to(torch.uint8).contiguous().cpu().pin_memory()   # contiguous HWC, like a decoder's frame

    # FrameBatchPipeline (nunif_b200/nunif/video.py): 3-slot ring, H2D | uint8->float, depth, warp, SBS, float->uint8 | D2H on three
    # streams, frames returned in ticket order - what FrameCallbackPool + per-thread streams do in the reference
    from nunif_b200.nunif.video import FrameBatchPipeline

    def sbs_callback(xf):
        depth = dam.infer(xf, edge_dilation=[2, 1])
        return stereo_sbs(xf, depth, 2.0, 0.5, method="forward_fill", edge_dilation=0)
    frames_host = [u8_in[i] for i in range(B)]
    pipe = FrameBatchPipeline(sbs_callback, B, dev, depth=3, copy_output=False)
    n_frames = B * (iters + 3)
    done = 0
    for i in range(3 * B):                      # warm: fills the ring
        done += len(pipe(frames_host[i % B]))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(iters * B):
        done += len(pipe(frames_host[i % B]))
    done += len(pipe.finish())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert done == n_frames, (done, n_frames)
    out["e2e_uint8_host_forward_fill"] = {"fps": iters * B / dt, "ms_per_batch": dt * 1e3 / iters, "batch": B,
                                          "h2d_bytes_per_batch": int(u8_in.numel()), "d2h_bytes_per_batch": int(B * H * 2 * W * 3),
                                          "pipeline": "FrameBatchPipeline depth 3 (copy-in | compute | copy-out streams), host wall clock over "
                                                      f"{iters} batches incl. the final drain, frames pushed one by one from pinned uint8"}
    return out


def bench_8k_downscaled(dev, model4x, iters=2):
    """Secondary: BASELINE configs[3] per GPU - SwinUNetDownscaled(2x) derived from the 4x weights on one 8K frame
    (3x4320x7680, 627 tiles of 256, batch 16, 97.6 TFLOP), device-timed, frame resident in HBM."""
    import torch
    from nunif_b200 import synth
    from nunif_b200.nunif.render import tiled_render
    m2 = model4x.to_2x()
    x8 = synth.synth_image(77, 3, 4320, 7680, smooth=False).to(dev)
    with torch.no_grad():
        y = tiled_render(x8, m2, tile_size=TILE, batch_size=BATCH)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            y = tiled_render(x8, m2, tile_size=TILE, batch_size=BATCH)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        shape = tuple(y.shape)
        del y
    return {"ms_per_frame": ms, "frames_per_sec": 1e3 / ms, "input_megapixels_per_sec": 4320 * 7680 / 1e6 / (ms / 1e3),
            "tiles": 627, "output_shape": shape, "model_tflops_per_sec": 627 * 155.7 / 1e3 / (ms / 1e3)}


def bench_to2x_4k(dev, model4x, x, iters=3):
    """Secondary: the north-star workload itself - swin_unet/art 2x (the released 2x model IS the 4x network followed by the
    antialiased bicubic /2, waifu2x/utils.py:128-176) on the same 4K frame, tile 256, batch 16, device-timed."""
    import torch
    from nunif_b200.nunif.render import tiled_render
    m2 = model4x.to_2x()
    with torch.no_grad():
        y = tiled_render(x, m2, tile_size=TILE, batch_size=BATCH)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            y = tiled_render(x, m2, tile_size=TILE, batch_size=BATCH)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        shape = tuple(y.shape)
        del y
    h, w = x.shape[1], x.shape[2]
    return {"ms_per_frame": ms, "frames_per_sec": 1e3 / ms, "input_megapixels_per_sec": h * w / 1e6 / (ms / 1e3), "output_shape": shape}


def bench_upcunet(dev, lib, x, iters=3):
    """Secondary: the 2x model of BASELINE configs[0] (UpCUNet, cunet/art noise1_scale2x layout, seeded weights) on the same
    4K frame, tile 256, batch 16 (180 tiles, 81.9 GFLOP each): device-timed, frame resident in HBM."""
    import ctypes
    import torch
    from nunif_b200 import synth, _lib
    from nunif_b200.nunif.models import create_model
    from nunif_b200.nunif.render import tiled_render
    m = create_model("waifu2x.upcunet", synth.upcunet_state_dict(0), dev)
    with torch.no_grad():
        for _ in range(2):
            y = tiled_render(x, m, tile_size=TILE, batch_size=BATCH)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            y = tiled_render(x, m, tile_size=TILE, batch_size=BATCH)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        _lib.check(lib.nb200_profile_enable(1))
        y = tiled_render(x, m, tile_size=TILE, batch_size=BATCH)
        buf = ctypes.create_string_buffer(8192)
        _lib.check(lib.nb200_profile_report(buf, 8192))
        _lib.check(lib.nb200_profile_enable(0))
        prof = json.loads(buf.value.decode())
        del y
    h, w = x.shape[1], x.shape[2]
    gemm = prof.get("gemm", {"ms": 0.0, "work": 0.0})
    return {"ms_per_frame": ms, "input_megapixels_per_sec": h * w / 1e6 / (ms / 1e3), "tiles": 180,
            "model_tflops_per_sec": 180 * 81.9 / 1e3 / (ms / 1e3),
            "gemm_tflops_per_sec": gemm["work"] / (gemm["ms"] / 1e3) / 1e12 if gemm["ms"] else None,
            "kernel_classes_ms": {k: round(v["ms"], 3) for k, v in prof.items()}}


def _iw3_models(wl, dev=None):
    """(state_dict, engine depth model or None) for an iw3 workload."""
    from nunif_b200 import synth
    sd = synth.zoedepth_state_dict(0) if wl["depth"] == "ZoeD_N" else synth.depth_anything_v2_state_dict(0)
    if dev is None:
        return sd, None
    from nunif_b200.iw3 import DepthAnythingModel, ZoeDepthModel
    gpu = dev.index or 0
    dm = ZoeDepthModel("ZoeD_N").load_state_dict(sd, gpu=gpu) if wl["depth"] == "ZoeD_N" else DepthAnythingModel().load_state_dict(sd, gpu=gpu)
    return sd, dm


def iw3_cpu_frames(wl, n_frames, threads):
    """The reference algorithm of an iw3 workload on the CPU (oracle port, fp32): n_frames frames through depth network ->
    dilate_edge -> min/max (+ mapper) -> warp -> composed frame.  Returns seconds."""
    import numpy as np
    import torch
    from nunif_b200 import synth
    from oracle import iw3 as oiw3, frames as ofr
    torch.set_num_threads(threads)
    h, w = FRAME[wl["frame"]]
    sd, _ = _iw3_models(wl)
    c = torch.stack([synth.synth_image(50 + i, 3, h, w, smooth=False) for i in range(n_frames)])
    with torch.inference_mode():
        t0 = time.perf_counter()
        if wl["depth"] == "ZoeD_N":
            from oracle import zoedepth as oz
            depth = oz.batch_infer(sd, c, flip_aug=False, edge_dilation=wl["edge_dilation"])
        else:
            from oracle import depth_anything as oda
            x = torch.from_numpy(np.ascontiguousarray(ofr.batch_preprocess(c.numpy(), 392)))
            depth = oiw3.dilate_edge(oda.depth_anything_forward(sd, x).unsqueeze(1), wl["edge_dilation"])
        depth = oiw3.mapper(oiw3.minmax_normalize(depth), wl["mapper"])
        if wl["method"] == "backward":
            left, right = oiw3.apply_divergence_grid_sample(c, depth, 2.0, 0.5)
        else:
            left, right = oiw3.forward_warp(c, depth, 2.0, 0.5, fill=True)
        ys = [oiw3.dubois(lf, rt) if wl["anaglyph"] else oiw3.sbs(lf, rt) for lf, rt in zip(left, right)]
        assert len(ys) == n_frames
        return time.perf_counter() - t0


def iw3_cpu_baseline_object(wl, n_frames=1):
    cores = host_cores()
    threads = min(cores, 32)          # one torch process stops scaling on these layer sizes well before 128 threads
    t = iw3_cpu_frames(wl, n_frames, threads)
    return t, {"value": n_frames / t, "unit": "frames/s", "cores": threads, "kind": "port", "host_cores": cores,
               "sample": f"{n_frames} {wl['frame']} frame(s) through the oracle port of the whole path (oracle/zoedepth.py | depth_anything.py, "
                         f"iw3.py; torch-CPU fp32, {threads} threads), {t:.1f} s"}


def run_iw3_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = IW3_WORKLOADS[args.workload]
    ts, cb = [], None
    for _ in range(max(1, min(args.steps, 3))):      # bounded: a step is ONE frame on the host cores
        t, cb = iw3_cpu_baseline_object(wl, 1)
        ts.append(t)
    t = sum(ts) / len(ts)
    cb["value"] = 1.0 / t
    h, w = FRAME[wl["frame"]]
    print(json.dumps({
        "impl": "reference", "metric": "iw3_frames_per_sec", "value": 1.0 / t, "unit": "frames/s", "n_gpus": args.gpus, "steps": len(ts),
        "warmup": 0, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": f"{wl['text']}, {w}x{h} frames, 1 frame per step (bounded sample of the stream)",
                                        "workload_key": args.workload},
        "cpu_baseline": cb, "e2e": {"value": 1.0 / t, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def _init_b200(args):
    import torch
    import torch.distributed as dist
    from nunif_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.lib()
    _lib.check(lib.nb200_check_device(local))
    return world, rank, local, dev, lib


def run_b200_iw3(args):
    """--workload iw3_1080p | iw3_4k_zoe: frame-parallel stream, B frames per GPU per step (weak scaling, no data-path collective;
    every rank packs the same seeded weights).  `value`: frames resident in HBM as float CHW, device-timed.  `e2e`: pinned uint8
    HWC frames on the host -> FrameBatchPipeline (H2D | compute | D2H streams, ticket order) -> uint8 stereo frames on the host."""
    import ctypes
    import torch
    import torch.distributed as dist
    from nunif_b200 import synth, _lib
    from nunif_b200.iw3 import stereo_sbs
    from nunif_b200.nunif.video import FrameBatchPipeline
    world, rank, local, dev, lib = _init_b200(args)
    wl = IW3_WORKLOADS[args.workload]
    h, w = FRAME[wl["frame"]]
    B = wl["batch"]
    _, dm = _iw3_models(wl, dev)
    c = torch.stack([synth.synth_image(50 + 16 * rank + i, 3, h, w, smooth=False) for i in range(B)]).to(dev)

    def frames_to_stereo(xf):
        depth = dm.infer(xf, edge_dilation=wl["edge_dilation"])
        return stereo_sbs(xf, depth, 2.0, 0.5, method=wl["method"], mapper=wl["mapper"], edge_dilation=0, anaglyph=wl["anaglyph"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.inference_mode():
        for _ in range(args.warmup):
            y = frames_to_stereo(c)
        barrier()
        launches0 = lib.nb200_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clocks:
            e0.record()
            for _ in range(args.steps):
                y = frames_to_stereo(c)
            e1.record()
            barrier()
        launches = lib.nb200_launch_count() - launches0
        ms = e0.elapsed_time(e1)
        out_shape = list(y.shape)
        dumped = dump_outputs(args.dump_outputs, {"stereo_frames": y}) if args.dump_outputs and rank == 0 else None
    # ---- end to end from host uint8 frames (outside inference_mode: the pipeline enters it around the callback itself)
    u8_in = (c.permute(0, 2, 3, 1) * 255.0).round().to(torch.uint8).contiguous().cpu().pin_memory()   # contiguous HWC, like a decoder's frame
    frames_host = [u8_in[i] for i in range(B)]
    pipe = FrameBatchPipeline(frames_to_stereo, B, dev, depth=3, copy_output=False)
    e2e_steps = min(max(args.steps, 10), 50)
    done = 0
    for i in range(3 * B):
        done += len(pipe(frames_host[i % B]))
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps * B):
        done += len(pipe(frames_host[i % B]))
    t_loop = time.perf_counter() - t0
    done += len(pipe.finish())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert done == (e2e_steps + 3) * B, done
    if os.environ.get("NB200_PIPE_TRACE"):
        print(f"[pipe trace] loop {t_loop * 1e3:.1f} ms, drain {(dt - t_loop) * 1e3:.1f} ms, frames pinned: {frames_host[0].is_pinned()}", file=sys.stderr)
        for name, cb in (("trivial", lambda xf: torch.cat([xf, xf], dim=3)), ("real", frames_to_stereo)):
            p2 = FrameBatchPipeline(cb, B, dev, depth=3, copy_output=False)
            for i in range(4 * B):
                p2(frames_host[i % B])
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            for i in range(40 * B):
                p2(frames_host[i % B])
            p2.finish()
            torch.cuda.synchronize()
            print(f"[pipe trace] second pipeline [{name}]: {40 * B / (time.perf_counter() - t1):.0f} fps", file=sys.stderr)
    with torch.inference_mode():
        # ---- kernel classes
        _lib.check(lib.nb200_profile_enable(1))
        y = frames_to_stereo(c)
        buf = ctypes.create_string_buffer(8192)
        _lib.check(lib.nb200_profile_report(buf, 8192))
        _lib.check(lib.nb200_profile_enable(0))
        prof = json.loads(buf.value.decode())
    t = torch.tensor([ms, dt * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    fps = world * args.steps * B / (ms / 1e3)
    fps_e2e = world * e2e_steps * B / (ms_e2e / 1e3)
    peaks, peak_src = load_peaks()
    peak_tf = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    total = sum(v["ms"] for v in prof.values()) or 1.0
    dom = max(prof, key=lambda k: prof[k]["ms"])
    d = prof[dom]
    if dom in ("gemm", "window_attention"):
        ach = d["work"] / (d["ms"] / 1e3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf}
    else:
        ach = d["work"] / (d["ms"] / 1e3) / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"]}
    roof.update({"kernel": {"gemm": "gemm_conv_persistent (tcgen05 implicit GEMM: every Linear / conv of the depth network)",
                            "window_attention": "flash_attention_kernel (mma.sync, d = 64, relative-position bias for BEiT)"}.get(dom, dom),
                 "class": dom, "launches": d.get("launches"), "avg_launch_us": d["ms"] * 1e3 / max(1, d.get("launches", 1)),
                 "share_of_step": d["ms"] / total, "peak_source": f"{peak_src} MEASURED_PEAKS.json", "traffic": None,
                 "note": "achieved = algorithmic FLOPs (2*M*N*K per GEMM launch; 4*T*N*d per attention launch) or bytes of every launch of the "
                         "dominant kernel class in one step / their CUDA-event time (nb200_profile_report)"})
    line = {
        "metric": "iw3_frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"{wl['text']}, {w}x{h} frames, {B} frames/GPU/step", "workload_key": args.workload,
                   "parallelism": f"frame-parallel x{world} (no data-path collective)", "weights": "random-init seed 0 (nunif_b200.synth)",
                   "l2": "frames + activations per step exceed the 126 MB L2; no explicit flush", "output_shape": out_shape,
                   "input_megapixels_per_sec": fps * h * w / 1e6},
        "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(u8_in.numel()),
                "d2h_bytes_per_step": int(out_shape[0] * out_shape[1] * out_shape[2] * out_shape[3]), "steps": e2e_steps,
                "note": "pinned uint8 HWC frames -> FrameBatchPipeline depth 3 (H2D | uint8->float, depth, warp, compose, float->uint8 | D2H on "
                        "three streams, ticket order) -> uint8 frames on the host; host wall clock incl. the final drain"},
        "gpu_launches": int(launches), "clocks": clocks.summary(), "roofline": roof,
        "kernel_classes_ms": {k: round(v["ms"], 4) for k, v in prof.items()},
    }
    if dumped:
        line["dump_outputs"] = dumped
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = iw3_cpu_baseline_object(wl, 1)[1]
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_b200(args):
    import torch
    import torch.distributed as dist
    from nunif_b200 import synth, _lib
    from nunif_b200.nunif.models import create_model
    from nunif_b200.nunif.render import tiled_render
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout; keep stdout for the single JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.lib()
    _lib.check(lib.nb200_check_device(local))
    if os.environ.get("NB200_GRAPHS"):
        _lib.check(lib.nb200_tune_set(9, int(os.environ["NB200_GRAPHS"])))   # CUDA-graph replay of the tile-batch forward (A/B)
    for kv in filter(None, os.environ.get("NB200_TUNE", "").split(",")):    # A/B knobs of csrc/gemm.cu g_tune, e.g. NB200_TUNE=12=1
        k, v = kv.split("=")
        _lib.check(lib.nb200_tune_set(int(k), int(v)))

    wl = WORKLOADS[args.workload]
    if args.frame is None:
        args.frame = wl["frame"]
    h, w = FRAME[args.frame]
    down = wl["down"]
    oscale = 4 // down
    ntiles = frame_tiles(h, w, scale=oscale, offset=32 // down, blend=16 if down == 1 else 4 * down)
    # every rank builds the same container; rank 0's packed weight blob is broadcast once over NCCL
    # (replaces torch.nn.parallel.replicate, nunif/models/data_parallel.py:16,58)
    model4x = create_model("waifu2x.swin_unet_4x", synth.swin_unet_state_dict(0, 4), dev)
    if world > 1:
        from nunif_b200 import parallel
        parallel.broadcast_model_weights(model4x, src=0)
    model = model4x if down == 1 else model4x.to_2x()
    # per-rank frame (weak scaling: one frame per GPU per step), already resident in HBM
    x = synth.synth_image(1000 + rank, 3, h, w, smooth=False).to(dev)
    x_host = synth.synth_image(1000 + rank, 3, h, w, smooth=False).pin_memory()
    out_host = torch.empty((3, h * oscale, w * oscale), dtype=torch.float32).pin_memory()

    def step():
        return tiled_render(x, model, tile_size=TILE, batch_size=BATCH)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(args.warmup):
            y = step()
        y = None
        barrier()
        launches0 = lib.nb200_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clocks:
            e0.record()
            for _ in range(args.steps):
                y = step()
            e1.record()
            barrier()
        launches = lib.nb200_launch_count() - launches0
        ms = e0.elapsed_time(e1)
        dumped = dump_outputs(args.dump_outputs, {"output": y}) if args.dump_outputs and rank == 0 else None
        del y
        # ---- end-to-end through the public API with host buffers (H2D + render + D2H every step)
        e2e_steps = max(1, min(args.steps, 3))
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tiled_render(x_host, model, tile_size=TILE, batch_size=BATCH, out=out_host)   # warm the side stream / pool
        barrier()
        g0.record()
        for _ in range(e2e_steps):
            # host tensor in -> host tensor out: nb200_tiled_render_host (H2D of the frame, render, band-pipelined D2H)
            tiled_render(x_host, model, tile_size=TILE, batch_size=BATCH, out=out_host)
        g1.record()
        barrier()
        ms_e2e = g0.elapsed_time(g1)
        # ---- kernel-class timing for the roofline (one extra, untimed-for-`value` step)
        _lib.check(lib.nb200_profile_enable(1))
        y = step()
        import ctypes
        buf = ctypes.create_string_buffer(8192)
        _lib.check(lib.nb200_profile_report(buf, 8192))
        _lib.check(lib.nb200_profile_enable(0))
        prof = json.loads(buf.value.decode())
        del y

        # secondary objects (rank 0 only): never allowed to take the headline line down with them
        def guarded(fn, *a, **k):
            try:
                return fn(*a, **k)
            except Exception as e:  # noqa: BLE001
                torch.cuda.synchronize()
                return {"error": f"{type(e).__name__}: {e}"}
        secondaries = rank == 0 and args.workload == "swin4x_4k" and not os.environ.get("NB200_BENCH_MINIMAL")   # (set for the ncu launch-list pass)
        to2x = guarded(bench_to2x_4k, dev, model4x, x) if secondaries else None
        iw3 = guarded(bench_iw3, dev, lib, peaks_gbs=load_peaks()[0]["hbm_gbs"]) if secondaries else None
        upc = guarded(bench_upcunet, dev, lib, x) if secondaries else None
        cfg4 = guarded(bench_8k_downscaled, dev, model4x) if secondaries else None

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    mp = h * w / 1e6
    value = world * args.steps * mp / (ms / 1e3)
    e2e = world * e2e_steps * mp / (ms_e2e / 1e3)
    peaks, peak_src = load_peaks()
    peak_tf = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])     # kernels timed inside a long step: the sustained figure
    total_prof_ms = sum(v["ms"] for v in prof.values())
    KERNEL_OF = {"fused_attn": "swin_attn_tc_kernel (tcgen05 qkv GEMM, QK^T and PV; q/k/v/S/P in shared / tensor memory)",
                 "fused_mlp": "swin_mlp_fused2_kernel / swin_mlp_fused_kernel (tcgen05 [proj +] fc1 + GELU + fc2, hidden in smem/TMEM)",
                 "gemm": "gemm_conv_persistent (tcgen05 implicit GEMM: convs, patch up/down, proj of the C=192 blocks, to_image)"}

    def tensor_view(name):
        c = prof.get(name)
        if not c or c["ms"] <= 0:
            return None
        tf = c["work"] / (c["ms"] / 1e3) / 1e12
        gbs = c.get("hbm_bytes", 0.0) / (c["ms"] / 1e3) / 1e9
        return {"kernel": KERNEL_OF[name], "tflops": tf, "tensor_frac": tf / peak_tf, "launches": c["launches"],
                "avg_launch_us": c["ms"] * 1e3 / max(1, c["launches"]), "ms_per_frame": c["ms"],
                "share_of_step": c["ms"] / total_prof_ms if total_prof_ms else None,
                "hbm_GBps_algorithmic": gbs, "hbm_frac": gbs / peaks["hbm_gbs"],
                "flop_per_launch": c["work"] / max(1, c["launches"]), "hbm_bytes_per_launch": c.get("hbm_bytes", 0.0) / max(1, c["launches"])}
    views = {k: tensor_view(k) for k in KERNEL_OF}
    views = {k: v for k, v in views.items() if v}
    dom = max(views, key=lambda k: views[k]["ms_per_frame"]) if views else None
    # dram__bytes_read.sum + dram__bytes_write.sum of the shipped kernels, parsed from an ncu --set full capture by
    # profiles/ncu_traffic.py into profiles/r2/ncu_traffic.json (per launch of the largest launch class); null until captured
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2", "ncu_traffic.json")
    if dom and os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(dom)
        except (OSError, ValueError):
            traffic = None
    line = {
        "metric": "waifu2x_input_megapixels_per_sec", "value": value, "unit": "MP/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"{wl['text']}, {args.frame} input 3x{h}x{w}, tile_size=256 batch=16, "
                               f"{ntiles} tiles/frame, 1 frame/GPU/step",
                   "workload_key": args.workload,
                   "parallelism": f"frame-parallel x{world} (no data-path collective; NCCL weight broadcast at load)",
                   "weights": "random-init seed 0 (nunif_b200.synth)",
                   "l2": "inputs/activations per step (>1 GB) exceed the 126 MB L2; no explicit flush",
                   "frames_per_sec": world * args.steps / (ms / 1e3),
                   "output_megapixels_per_sec": value * oscale * oscale,
                   "model_tflops_per_sec": world * args.steps * ntiles * SWIN4X_TILE_GFLOP / 1e3 / (ms / 1e3)},
        "e2e": {"value": e2e, "unit": "MP/s", "h2d_bytes_per_step": 3 * h * w * 4, "d2h_bytes_per_step": 3 * h * w * oscale * oscale * 4,
                "steps": e2e_steps, "note": "pinned host frame -> tiled_render (nb200_tiled_render_host: H2D, render, output blended and copied back in bands "
                        "of finished tile rows on a side stream) -> pinned host fp32 output; every step moves all bytes"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": ({"bound": "tensor", "kernel": views[dom]["kernel"], "class": dom,
                      "achieved": views[dom]["tflops"], "peak": peak_tf, "unit": "TFLOP/s", "frac": views[dom]["tensor_frac"],
                      "peak_source": f"{peak_src} MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)",
                      "launches": views[dom]["launches"], "avg_launch_us": views[dom]["avg_launch_us"],
                      "share_of_step": views[dom]["share_of_step"],
                      "note": "SURVEY 8(d): path A is judged against the tensor roofline.  achieved = algorithmic FLOPs of every launch of "
                              "the dominant kernel class in one frame (2*M*N*K of its GEMMs + 4*T*36*C for QK^T/PV) / their CUDA-event "
                              "time (nb200_profile_report, events on the launching stream)",
                      "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                      "traffic_launch": (traffic or {}).get("launch"),
                      "traffic_algorithmic": (traffic or {}).get("algorithmic_bytes_per_launch")} if dom else None),
        "roofline_by_class": views,
        "kernel_classes_ms": {k: round(v["ms"], 3) for k, v in prof.items()},
    }
    if to2x is not None:
        line["swin_to_2x_4k"] = to2x
    if upc is not None:
        line["upcunet_4k_2x"] = upc
    if cfg4 is not None:
        line["swin_downscaled2x_8k"] = cfg4
    if iw3 is not None:
        line["iw3_1080p"] = iw3
    if dumped:
        line["dump_outputs"] = dumped
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = guarded(lambda: cpu_baseline_object(h, w, ntiles)[1])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_gpu"])
    ap.add_argument("--compile", action="store_true", help="--impl torch_gpu: wrap the forward in torch.compile")
    ap.add_argument("--cpu-worker", nargs=2, type=int, metavar=("TILES", "THREADS"), help=argparse.SUPPRESS)
    ap.add_argument("--frame", default=None, choices=list(FRAME), help="frame size (default: the workload's)")
    ap.add_argument("--workload", default="swin4x_4k", choices=list(WORKLOADS) + list(IW3_WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl b200: after the timed steps, write the last step's output to DIR/<name>.npy (float32; a fixed "
                         "seeded sample of it when it exceeds 32 MiB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs is implemented for --impl b200")
    if args.cpu_worker:
        cpu_worker_main(*args.cpu_worker)
    elif args.workload in IW3_WORKLOADS:
        if args.impl == "torch_gpu":
            raise SystemExit("--impl torch_gpu is defined for the waifu2x workloads")
        run_iw3_reference(args) if args.impl == "reference" else run_b200_iw3(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_gpu":
        run_torch_gpu(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
