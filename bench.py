#!/usr/bin/env python
"""bench.py — SSGI+denoise Mpixels/s at 3840x2160 on N B200s (BASELINE.json metric; N = 1 workload = config C3).

One "step" = one frame of the SSGI chain over one batch of synthetic G-buffer planes:
  K1 SSGI trace (steps 20 / refine 5) -> K2 temporal reprojection (2 planes) ->
  K3 Poisson denoise x4 (denoiseIterations = 2) -> K4 GI compose          (432 B/px algorithmic, SURVEY.md §8d)

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N = 1 : one 3840x2160 frame per step on one GPU (the configuration the metric is quoted on).
N > 1 : the SAME 3840x2160 frame, strong scaling: row bands over N ranks (rfx_group_*: halo rows recomputed locally, last frame's
        history read in place on the owning rank over NVLink, one tiny NCCL collective per frame).  The line also carries
        config C5 (7680x4320 over the same N GPUs) under "c5_8k".
value   : whole-job Mpixels/s with the input planes resident in HBM (CUDA events on the launching stream, max over ranks).
e2e     : the same metric through host buffers (pinned host planes -> H2D -> chain -> D2H of `composed`), copies inside the
          timed region; at N = 1 this is rfx_ssgi_chain_submit_host / wait_host (sync_call_ms: rfx_ssgi_chain_render_host).
roofline: the dominant kernel's algorithmic bytes / its mean CUDA-event duration over the timed frames, against the measured
          HBM copy bandwidth in MEASURED_PEAKS.json (+ the chain-level figure).
parity  : the first frame of the timed workload against the CPU oracle's frame (the one cpu_baseline times anyway).
configs : device time + roofline of the other single-GPU BASELINE configs (C1 motion blur 256^2, C2 SSGI 1080p, C4 HBAO 4K).
cpu_baseline / --impl reference: the reference's own shaders compiled for the CPU (oracle/_ref, when built) or the CPU restatement in
oracle/ (the reference's run time is WebGL-only and cannot run here: no GL,
          no JS engine) on the box's host cores, bounded sample, thread count pinned and reported.
--dump-outputs DIR: after the timed steps, the `composed` plane of the last timed step (what a caller of the chain receives) as
          DIR/composed.npy, float32.  A plane larger than 64 MB (the 4K frame) is stored as a fixed, seeded sample of its pixels, shape
          (pixels, 4), the same pixels on every run at that size.  The inputs are synthetic and deterministic, so two builds run with the
          same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

WIDTH, HEIGHT = 3840, 2160
DENOISE_ITERATIONS = 2
DUMP_BYTES, DUMP_SEED = 64_000_000, 20261017  # --dump-outputs: size bound of all files together, seed of the pixel sample
ALGO_BYTES = {  # SURVEY.md §8(d): algorithmic bytes per output pixel
    "K1_ssgi_trace": 76, "K2_temporal_reproject": 80, "K3_poisson_pass0": 68, "K3_poisson_pass1plus": 52, "K4_gi_compose": 52,
}


def chain_bytes_per_px(iterations: int) -> int:
    n = 2 * iterations
    return 76 + 80 + (68 + max(n - 1, 0) * 52 if n else 0) + 52


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.p = gpu_index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.gpu)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.25)  # let the sampler come up before the timed region starts
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def make_gpu_frames(width, height, n, device, aspect=None):
    """Synthetic planes generated on the device with torch (plumbing)."""
    import torch

    from realism_effects_b200 import synth

    frames = []
    for t in range(n):
        fr = synth.render_frame(width, height, t + 1, device=device, aspect=aspect or width / height)
        frames.append(dict(depth=fr.depth, gbuffer=fr.gbuffer, velocity=fr.velocity, direct=fr.direct_light, cam=fr.cam.uniforms(), moved=True, soa=fr.soa))
    torch.cuda.synchronize()
    return frames


def tensor_plane(t, fmt):
    from realism_effects_b200 import abi

    p = abi.Plane()
    p.ptr = t.data_ptr()
    p.height, p.width = t.shape[0], t.shape[1]
    p.pitch = t.shape[1] * abi.FMT_BYTES[fmt]
    p.format = fmt
    return p


class _PW:  # adapter so SsgiChain.render can take raw planes
    def __init__(self, p):
        self.p = p


def frame_planes(f):
    from realism_effects_b200 import abi

    return (_PW(tensor_plane(f["depth"], abi.FMT_R32F)), _PW(tensor_plane(f["gbuffer"], abi.FMT_RGBA32F)), _PW(tensor_plane(f["velocity"], abi.FMT_RGBA32F)),
            _PW(tensor_plane(f["direct"], abi.FMT_RGBA16F)))


def env_for_bench():
    """The reference demo's environment (example/public/hdr/spree_bank_1k.hdr, 1024x512, SURVEY.md §8d) decoded like three's RGBELoader, and its
    importance-sampling tables as `gatherData` builds them for a flipY texture (EquirectHdrInfoUniform.js:149-245, incl. the mirroring un-flip, A4)"""
    from realism_effects_b200 import synth

    img, gl = synth.load_reference_env()
    marg, cond, total = synth.build_env_cdf(img.astype(np.float32), flip_y=True)
    return gl, marg, cond, total


def chain_options(ch, o, W, H):
    class _I:
        width, height = W, H

    return ch.chain_options(_I, o)


def dump_outputs(out_dir: str, **planes) -> None:
    """--dump-outputs: each (H, W, C) plane as <out_dir>/<name>.npy in float32; one over its share of DUMP_BYTES becomes a seeded
    sample of its pixels (sorted pixel order)"""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in planes.items():
        a = np.asarray(a, np.float32)
        n = (DUMP_BYTES // len(planes) - 4096) // a[0, 0].nbytes  # pixels that fit the share (less the .npy header)
        note = ""
        if a.shape[0] * a.shape[1] > n:
            px = a.reshape(a.shape[0] * a.shape[1], -1)
            a = px[np.sort(np.random.default_rng(DUMP_SEED).choice(px.shape[0], n, replace=False))]
            note = " (seeded pixel sample)"
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        print(f"bench.py: wrote {path} {a.shape}{note}", file=sys.stderr)


def time_frames(stream, render, K):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(K):
        render(i)
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / K


# ---------------------------------------------------------------------------------------------------------------------------
def other_configs(ctx, ch, dev, stream, peak):
    """Device time + roofline of the other single-GPU BASELINE configs (SURVEY.md §8d byte counts)."""
    import torch

    from realism_effects_b200 import abi, engine, synth

    out = {}

    def line(ms, W, H, bpp, extra=None):
        gbs = bpp * W * H / (ms * 1e-3) / 1e9
        d = {"ms_per_frame": round(ms, 4), "Mpixels_per_s": round(W * H / 1e6 / (ms * 1e-3), 1), "algorithmic_B_per_px": bpp, "achieved_GBps": round(gbs, 1),
             "frac_of_measured_hbm": round(gbs / peak, 4)}
        d.update(extra or {})
        return d

    # C2: SSGIEffect 1920x1080, steps 20 / refine 5, denoiseIterations 1 (the effect's default)
    W, H = 1920, 1080
    o = ch.Opts(denoise_iterations=1)
    frames = make_gpu_frames(W, H, 2, dev)
    chain = engine.SsgiChain(ctx, chain_options(ch, o, W, H))
    pl = [frame_planes(f) for f in frames]
    cams = [abi.make_camera(f["cam"]) for f in frames]
    r = lambda i: chain.render(cams[i % 2], *pl[i % 2], frames[i % 2]["cam"]["position"], True)  # noqa: E731
    for i in range(6):
        r(i)
    out["C2_ssgi_1080p"] = line(time_frames(stream, r, 50), W, H, chain_bytes_per_px(1), {"workload": "SSGIEffect 1920x1080 steps=20 refineSteps=5 denoiseIterations=1"})
    chain.close()
    del frames, pl
    # C4: HBAOEffect 3840x2160 (spp form) + 2 single-plane Poisson passes (velocity-layout normals) + ao_compose
    W, H = WIDTH, HEIGHT
    f = make_gpu_frames(W, H, 1, dev)[0]
    d, g, v, dl = (pw.p for pw in frame_planes(f))
    ao, tA, tB, outp = (ctx.alloc(abi.FMT_RGBA16F, W, H) for _ in range(4))
    hp = ch.hbao_params(f["cam"], 778)
    pps = []
    for i in range(2):
        p = ch.poisson_params(ch.Opts(), 1234568 + i, False)
        p.texture_count, p.gbuffer_texture, p.input_linear = 1, 0, 1
        p.is_texture_specular[:] = [0, 0]
        p.normal_phi, p.depth_phi, p.roughness_phi, p.specular_phi = 3.25, 2.0, 0.0, 0.0
        pps.append(p)
    acp = ch.ao_compose_params()

    def c4(_i):
        ctx.hbao(hp, d, ao)
        ctx.poisson_denoise(pps[0], d, v, ao, None, tA, None)
        ctx.poisson_denoise(pps[1], d, v, tA, None, tB, None)
        ctx.ao_compose(acp, d, tB, dl, outp)

    for i in range(4):
        c4(i)
    out["C4_hbao_4k"] = line(time_frames(stream, c4, 30), W, H, 112, {"workload": "HBAO (spp 8) + 2 Poisson passes (1 plane) + ao_compose, 3840x2160"})
    ms_h = time_frames(stream, lambda _i: ctx.hbao(hp, d, ao), 30)
    out["C4_hbao_4k"]["hbao_kernel_ms"] = round(ms_h, 4)
    out["C4_hbao_4k"]["hbao_kernel_GBps"] = round(12 * W * H / (ms_h * 1e-3) / 1e9, 1)
    for p in (ao, tA, tB, outp):
        p.free()
    # G-buffer ingest (SURVEY §8f row 2) at 3840x2160: albedo RGBA8 + normal RGBA16F + material RGBA8 + emissive RGBA16F + motion RGBA16F + depth in
    # (4 + 8 + 4 + 8 + 8 + 4 = 36 B/px), gBuffer + velocity RGBA32F out (32 B/px): a pure stream
    soa = f["soa"]
    keep = [soa["albedo"], soa["normal"].to(torch.float16).contiguous(), (soa["material"].float() * 255).round().to(torch.uint8).contiguous(), soa["emissive"],
            soa["motion"].to(torch.float16).contiguous()]  # the tensors own the memory the planes point at
    ing = [tensor_plane(t, fm) for t, fm in zip(keep, (abi.FMT_RGBA8, abi.FMT_RGBA16F, abi.FMT_RGBA8, abi.FMT_RGBA16F, abi.FMT_RGBA16F))]
    og, ov = ctx.alloc(abi.FMT_RGBA32F, W, H), ctx.alloc(abi.FMT_RGBA32F, W, H)
    ingest = lambda _i: ctx.gbuffer_ingest(*ing, d, og, ov)  # noqa: E731
    for i in range(5):
        ingest(i)
    out["gbuffer_ingest_4k"] = line(time_frames(stream, ingest, 50), W, H, 68, {"workload": "rfx_gbuffer_ingest_launch 3840x2160: 6 SoA planes (36 B/px) -> packed gBuffer + velocity (32 B/px)"})
    og.free()
    ov.free()
    del keep
    # cosmetic effects tail (SURVEY §8f row 3) at 3840x2160: Sharpness + GradualBackground + Sparkle merged in one launch
    # (input 8 + depth 4 + velocity 16 in, 8 out = 36 B/px; the reference spends one full-frame round trip per effect)
    fxp = ch.fx_params(f["cam"], [abi.FX_SHARPNESS, abi.FX_GRADUAL_BACKGROUND, abi.FX_SPARKLE])
    fxo = ctx.alloc(abi.FMT_RGBA16F, W, H)
    fxr = lambda _i: ctx.effects(fxp, dl, d, v, fxo)  # noqa: E731
    for i in range(5):
        fxr(i)
    out["fx_tail_4k"] = line(time_frames(stream, fxr, 50), W, H, 36, {"workload": "rfx_effects_launch 3840x2160: Sharpness + GradualBackground + Sparkle merged (EffectPass semantics), one launch"})
    tp = abi.TaaParams()
    tp.camera_not_moved_frames, tp.srgb_output = 3.0, 1
    th, to = ctx.alloc(abi.FMT_RGBA8, W, H), ctx.alloc(abi.FMT_RGBA8, W, H)
    tr_ = lambda _i: ctx.taa(tp, dl, th, to)  # noqa: E731
    for i in range(5):
        tr_(i)
    out["taa_pass_4k"] = line(time_frames(stream, tr_, 50), W, H, 16, {"workload": "rfx_taa_launch 3840x2160 (input RGBA16F 8 + history RGBA8 4 in, canvas RGBA8 4 out)"})
    for pl in (fxo, th, to):
        pl.free()
    # C1: MotionBlurEffect 256x256 (plumbing config)
    W, H = 256, 256
    inp = ch.make_inputs(W, H, 1)
    fr = inp.frames[0]
    vel = ctx.upload(ch.rotation_velocity_field(W, H, fr["depth"]))
    src, dst = ctx.upload(fr["direct"]), ctx.alloc(abi.FMT_RGBA16F, W, H)
    mp = ch.motion_blur_params(W, H, frame=7)
    mb = lambda _i: ctx.motion_blur(mp, vel, src, dst)  # noqa: E731
    for i in range(10):
        mb(i)
    out["C1_motion_blur_256"] = line(time_frames(stream, mb, 200), W, H, 32, {"workload": "MotionBlurEffect 256x256, 16 samples (launch-latency bound at this size)"})
    torch.cuda.synchronize()
    return out


def run_single(args):
    import torch

    from realism_effects_b200 import abi, engine, synth

    import chain_harness as ch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path (use --impl reference for the CPU oracle timing)")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    o = ch.Opts(denoise_iterations=DENOISE_ITERATIONS)
    W, H, K, Wm = args.width, args.height, args.steps, args.warmup
    ctx = engine.Context(0)
    env, marg, cond, total = env_for_bench()
    ctx.set_env(env, marg, cond, total)
    copt = chain_options(ch, o, W, H)
    frames = make_gpu_frames(W, H, 2, dev)
    planes = [frame_planes(f) for f in frames]
    cams = [abi.make_camera(f["cam"]) for f in frames]
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    peak, peak_src = measured_peak()

    # ---- parity: frame 0 of the workload on a fresh chain (kept on the device until the oracle's frame exists) ---------------------
    chain = engine.SsgiChain(ctx, copt)
    chain.render(cams[0], *planes[0], frames[0]["cam"]["position"], True)
    gpu_frame0 = chain.download(0)
    chain.close()

    chain = engine.SsgiChain(ctx, copt)

    def render(i):
        j = i % 2
        chain.render(cams[j], *planes[j], frames[j]["cam"]["position"], True)

    for i in range(Wm):
        render(i)
    ctx.sync()
    launches0 = ctx.launch_count
    chain.set_profiling(True)
    chain.get_profile()
    clocks = ClockSampler(0)
    clocks.start()
    ms_per_step = time_frames(stream, lambda i: render(Wm + i), K)
    clk = clocks.stop()
    prof = chain.get_profile()
    chain.set_profiling(False)
    launches = ctx.launch_count - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, composed=chain.download(0))
    mpx = W * H / 1e6
    value = mpx / (ms_per_step / 1e3)

    per_kernel = {}
    for k, (ms, n) in prof.items():
        if n:
            per_kernel[k] = {"ms_per_launch": ms / n, "launches": n, "share_of_step": ms / (ms_per_step * K), "algo_GBps": ALGO_BYTES[k] * W * H / (ms / n * 1e-3) / 1e9}
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms_per_launch"] * per_kernel[k]["launches"])
    ach = per_kernel[dom]["algo_GBps"]
    chain_ach = chain_bytes_per_px(DENOISE_ITERATIONS) * W * H / (ms_per_step * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4), "traffic": None, "peak_source": peak_src,
            "chain_achieved": round(chain_ach, 1), "chain_frac": round(chain_ach / peak, 4),
            "note": "the fast chain fuses K4 into the last Poisson pass (its time is inside K3_poisson_pass1plus); this path is instruction-issue bound, not HBM bound "
                    "(DESIGN.md §4): ncu DRAM traffic is at or below the algorithmic bytes",
            "per_kernel": {k: {kk: round(vv, 4) for kk, vv in v.items()} for k, v in per_kernel.items()}}
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    if (W, H) == (WIDTH, HEIGHT) and os.path.exists(tf):  # measured once per round under ncu (tools/ncu_traffic.py), quoted here
        t = json.load(open(tf))
        if dom in t.get("bytes_per_launch", {}):
            roof["traffic"] = t["bytes_per_launch"][dom]
            roof["algorithmic_bytes_per_launch"] = ALGO_BYTES[dom] * W * H
            roof["traffic_source"] = t.get("source")

    # ---- e2e through host buffers ----------------------------------------------------------------------------------------------
    host = [{k: f[k].cpu().pin_memory() for k in ("depth", "gbuffer", "velocity", "direct")} for f in frames]
    h2d = sum(host[0][k].numel() * host[0][k].element_size() for k in host[0])
    outs = [torch.empty((H, W, 4), dtype=torch.float32).pin_memory() for _ in range(2)]
    hfs = []
    for j, hb in enumerate(host):
        hf = abi.SsgiHostFrame()
        hf.cam = cams[j]
        hf.depth, hf.gbuffer, hf.velocity, hf.direct_light = hb["depth"].data_ptr(), hb["gbuffer"].data_ptr(), hb["velocity"].data_ptr(), hb["direct"].data_ptr()
        hf.camera_pos[:] = [float(x) for x in frames[j]["cam"]["position"]]
        hf.camera_moved = 1
        hf.out_composed = outs[j].data_ptr()
        hfs.append(hf)
    ke = max(3, min(K, 20))
    for i in range(3):
        chain.submit_host(hfs[i % 2])
        chain.wait_host(1)
    chain.wait_host(0)
    t0 = time.perf_counter()
    for i in range(ke):  # pipelined host path: frame i's H2D / kernels / D2H on three streams; every step moves its own 365 MB in and 133 MB out
        chain.submit_host(hfs[i % 2])
        chain.wait_host(1)
    chain.wait_host(0)
    e2e_s = (time.perf_counter() - t0) / ke
    t0 = time.perf_counter()
    for i in range(3):
        chain.render_host(hfs[i % 2])
    sync_ms = (time.perf_counter() - t0) / 3 * 1e3
    e2e = {"value": round(mpx / e2e_s, 2), "unit": "Mpixels/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(outs[0].numel() * 4), "ms_per_step": round(e2e_s * 1e3, 3),
           "steps": ke, "result_checksum": float(outs[0][::97, ::89, :3].double().sum()), "sync_call_ms": round(sync_ms, 3),
           "mode": "pipelined rfx_ssgi_chain_submit_host / wait_host, 2 frames in flight (PCIe-bound: the kernels hide under the upload); sync_call_ms = rfx_ssgi_chain_render_host"}
    chain.close()

    # ---- CPU baseline + parity: one full-resolution frame (frame 0, empty history) through the oracle -----------------------------
    cpu, parity = None, None
    if not args.no_cpu_baseline:
        f0 = frames[0]
        fr = dict(depth=f0["depth"].cpu().numpy(), gbuffer=f0["gbuffer"].cpu().numpy(), velocity=f0["velocity"].cpu().numpy(), direct=f0["direct"].cpu().numpy(), cam=f0["cam"], moved=True)
        cpu_inp = ch.Inputs(W, H, [fr], env, marg, cond, total, synth.load_blue_noise())
        cpu, ref0 = cpu_baseline_sample(ch, o, cpu_inp)
        c = ch.compare(ref0, gpu_frame0)
        c4 = ch.compare(ref0, gpu_frame0, rtol=4e-3)
        parity = {"config": "C3", "plane": "composed", "frame": "first frame of the timed workload (empty history)", "frac_bad_1e-3": c["frac_bad"], "n_bad": c["n_bad"],
                  "frac_bad_4e-3": c4["frac_bad"], "max_rel_of_conforming": c["max_rel_ok"], "bit_equal_fraction": c["bit_equal"],
                  "note": "GPU fast variant vs the CPU oracle on identical planes; multi-frame / all-plane parity at C2 and C3 sizes: tests/test_gpu_parity_at_size.py"}

    configs = None
    if not args.no_configs:
        configs = other_configs(ctx, ch, dev, stream, peak)

    cfg = {"workload": f"C3 SSGI+PoissonDenoise(denoiseIterations={DENOISE_ITERATIONS} => {2 * DENOISE_ITERATIONS} passes)+compose, steps=20 refineSteps=5, {W}x{H}",
           "inputs": f"2 alternating synthetic G-buffer frames ({h2d / 1e6:.0f} MB of input planes per frame > 126 MB L2), moving camera, the reference demo's env map (spree_bank_1k.hdr, 1024x512) + its CDF tables",
           "l2": "inputs larger than L2; no explicit flush", "fast_math": True}
    line = {"metric": "SSGI+denoise Mpixels/s at 4K", "value": round(value, 2), "unit": "Mpixels/s", "n_gpus": 1, "steps": K, "warmup": Wm, "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp16 accumulate planes)", "data": "synthetic", "impl": "ours", "config": cfg,
            "gpu_launches": int(launches), "e2e": e2e, "roofline": roof, "cpu_baseline": cpu, "parity": parity, "configs": configs, "clocks": clk}
    print(json.dumps(line))
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------------
def run_sharded(args):
    import torch
    import torch.distributed as dist

    from realism_effects_b200 import abi, engine, parallel

    import chain_harness as ch

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    o = ch.Opts(denoise_iterations=DENOISE_ITERATIONS)
    K, Wm = args.steps, args.warmup
    ctx = engine.Context(local)
    env, marg, cond, total = env_for_bench()
    ctx.set_env(env, marg, cond, total)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    peak, peak_src = measured_peak()

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    def reduce(x: float, op) -> float:
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def measure(W, H, steps, warm, check_frames, settle):
        """strong scaling of one W x H frame over the ranks; returns (ms/frame max over ranks, info)"""
        copt = chain_options(ch, o, W, H)
        frames = make_gpu_frames(W, H, 2, dev)
        planes = [frame_planes(f) for f in frames]
        cams = [abi.make_camera(f["cam"]) for f in frames]
        sh = parallel.ShardedSsgiChain(ctx, copt, rebalance_every=4, rebalance_lag=2)
        bit_exact = None
        if check_frames:  # every rank also renders the whole frame alone and compares its band's bytes, frame after frame
            single = engine.SsgiChain(ctx, copt)
            ok = True
            for t in range(check_frames):
                j = t % 2
                single.render(cams[j], *planes[j], frames[j]["cam"]["position"], True)
                sh.render(cams[j], *planes[j], frames[j]["cam"]["position"], True)
                b0, b1 = sh.band_of_last_frame
                ok = ok and single.download(0)[b0:b1].tobytes() == sh.chain.download(0)[b0:b1].tobytes()
            single.close()
            bit_exact = reduce(1.0 if ok else 0.0, dist.ReduceOp.MIN) == 1.0
        rr = lambda i: sh.render(cams[i % 2], *planes[i % 2], frames[i % 2]["cam"]["position"], True)  # noqa: E731
        for i in range(settle + warm):  # the band borders settle (cost-driven) before the timed region
            rr(i)
        barrier()
        launches0 = ctx.launch_count
        ms = time_frames(stream, lambda i: rr(warm + i), steps)
        barrier()
        ms = reduce(ms, dist.ReduceOp.MAX)
        info = {"bounds": list(sh.bounds), "per_rank_kernel_ms": [round(c, 4) for c in sh.last_costs], "launches_per_frame": (ctx.launch_count - launches0) / steps,
                "multi_gpu_bit_exact": bit_exact, "peer_reads": sh.uses_peer_reads}
        return ms, info, sh, frames, cams

    clocks = ClockSampler(local)
    clocks.start()
    ms_per_step, info, sh, frames, cams = measure(args.width, args.height, K, Wm, 3, 24)
    clk = clocks.stop()
    W, H = args.width, args.height
    mpx = W * H / 1e6
    value = mpx / (ms_per_step / 1e3)
    chain_ach = chain_bytes_per_px(DENOISE_ITERATIONS) * W * H / (ms_per_step * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": "chain (all kernels of a frame, all ranks)", "achieved": round(chain_ach, 1), "peak": peak * world, "unit": "GB/s", "frac": round(chain_ach / (peak * world), 4),
            "traffic": None, "peak_source": peak_src + f" x {world} GPUs", "note": "whole-job algorithmic bytes per frame / max-over-ranks frame time; per-kernel figures are in the N = 1 line"}

    # ---- e2e: sharded host path (each rank uploads its share; depth / velocity rows exchanged over NCCL; own rows read back) ----------
    host = [{k: f[k].cpu().pin_memory() for k in ("depth", "gbuffer", "velocity", "direct")} for f in frames]
    outs = [torch.empty((H, W, 4), dtype=torch.float32).pin_memory() for _ in range(2)]
    ke = max(3, min(K, 20))

    def e2e_step(i):
        j = i % 2
        sh.submit_host(cams[j], host[j], frames[j]["cam"]["position"], True, outs[j])
        sh.wait_host(1)

    for i in range(8):
        e2e_step(i)
    sh.wait_host(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(ke):
        e2e_step(i)
    sh.wait_host(0)
    barrier()
    e2e_s = reduce((time.perf_counter() - t0) / ke, dist.ReduceOp.MAX)
    h2d, d2h = sh.host_bytes_per_frame
    e2e = {"value": round(mpx / e2e_s, 2), "unit": "Mpixels/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": round(e2e_s * 1e3, 3), "steps": ke,
           "bytes_are": "per rank (own rows of depth / velocity + K1-range rows of gBuffer / direct light in; own rows of composed out)",
           "result_checksum": float(outs[0][: 64, ::89, :3].double().sum())}
    sh.close()
    del frames, host, outs

    c5 = None
    if not args.no_c5:  # config C5: the full chain at 7680x4320 over the same N GPUs
        try:
            ms8, info8, sh8, _f8, _c8 = measure(7680, 4320, max(10, K // 4), 3, 0, 16)
            c5 = {"workload": f"C5 7680x4320 row bands over {world} GPUs", "ms_per_step": round(ms8, 4), "value": round(7680 * 4320 / 1e6 / (ms8 / 1e3), 2), "unit": "Mpixels/s",
                  "bounds": info8["bounds"], "per_rank_kernel_ms": info8["per_rank_kernel_ms"]}
            sh8.close()
        except Exception as e:  # noqa: BLE001
            c5 = {"error": str(e)[:200]}

    if rank == 0:
        cfg = {"workload": f"C3 SSGI+PoissonDenoise(denoiseIterations={DENOISE_ITERATIONS})+compose, steps=20 refineSteps=5, ONE {W}x{H} frame per step row-sharded over {world} GPUs (strong scaling)",
               "inputs": "2 alternating synthetic G-buffer frames resident on every rank (365 MB per frame > 126 MB L2), moving camera", "l2": "inputs larger than L2; no explicit flush",
               "fast_math": True,
               "multi_gpu": {"sharding": "one contiguous row band per rank, borders rebalanced every 4 frames from the ranks' device-timed kernel cost; halo rows recomputed locally",
                             "exchange": ("none per pass; last frame's composed / dn history is read in place on the owning rank (CUDA IPC peer mappings over NVLink); one NCCL all-gather of "
                                          f"{world} floats per frame (kernel costs) doubles as the frame barrier") if info["peer_reads"] else
                                         "FALLBACK: peer mappings unavailable (or RFX_GROUP_EXCHANGE=allgather) - composed + dn rows replicated with an NCCL exchange after every frame",
                             "bounds_during_timed_frames": info["bounds"], "per_rank_kernel_ms_per_frame": info["per_rank_kernel_ms"], "launches_per_frame_per_rank": info["launches_per_frame"]}}
        line = {"metric": "SSGI+denoise Mpixels/s at 4K", "value": round(value, 2), "unit": "Mpixels/s", "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms_per_step, 4),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp16 accumulate planes)", "data": "synthetic", "impl": "ours", "config": cfg,
                "gpu_launches": int(round(info["launches_per_frame"] * K)), "e2e": e2e, "roofline": roof, "cpu_baseline": None, "multi_gpu_bit_exact": info["multi_gpu_bit_exact"],
                "c5_8k": c5, "clocks": clk}
        print(json.dumps(line))
    ctx.close()
    dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------------
def oracle_threads() -> int:
    """Pin the oracle's OpenMP thread count BEFORE the library is loaded: all host cores this process may use (a launcher such as
    torchrun sets OMP_NUM_THREADS=1 for its children, which would silently turn the 'all host threads' baseline into one thread)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ.pop("OMP_THREAD_LIMIT", None)
    return n


def cpu_baseline_sample(ch, o, inp):
    """Times the CPU oracle chain on the frames of `inp` (all host threads); returns (cpu_baseline dict, composed of the last frame)."""
    want = oracle_threads()
    import orc

    width, height, frames_n = inp.width, inp.height, len(inp.frames)
    orc.lib()
    t0 = time.perf_counter()
    ref = ch.run_oracle_chain(inp, o, capture=("composed",), lean=True)
    dt = time.perf_counter() - t0
    cores = int(orc.lib().orc_num_threads())
    out = {"value": round(width * height * frames_n / 1e6 / dt, 4), "unit": "Mpixels/s", "cores": cores, "threads_requested": want, "kind": "port",
           "sample": f"{frames_n} frame(s) of the same chain at {width}x{height} ({dt:.1f} s of CPU work; first frame => empty history)"}
    rs = reference_shaders()
    if rs is not None:  # the reference's own shaders on the same cores, on a 1/16 sample (the port above also supplies the parity pixels)
        small = ch.make_inputs(960, 540, 1, reference_env=True)
        t0 = time.perf_counter()
        ch.run_oracle_chain(small, o, capture=("composed",), lean=True, impl=rs)
        dts = time.perf_counter() - t0
        out["reference_shaders"] = {"value": round(960 * 540 / 1e6 / dts, 4), "unit": "Mpixels/s", "kind": "reference", "cores": cores,
                                    "sample": f"one 960x540 frame of the same chain through oracle/_ref ({dts:.1f} s)"}
    return (out, ref[-1]["composed"])


def reference_shaders():
    """tests/refglsl.py when the reference's own shaders, compiled for the CPU, can run the C3 chain here (oracle/_ref/*.so built by
    __graft_entry__.build() from the reference checkout; they travel to the GPU box), else None"""
    try:
        import refglsl

        return refglsl if refglsl.chain_available(0) else None
    except Exception:  # noqa: BLE001
        return None


def run_reference(args):
    """--impl reference: the reference's run time is WebGL (no GL / JS engine here), so the arm runs the reference's OWN FRAGMENT
    SHADERS compiled for the host CPU (oracle/_ref, kind "reference": the GLSL text of the reference on the GLSL runtime
    oracle/ref/glsl_rt.h, driven by the reference's frame logic) with all host threads, each step a bounded sample of the workload.
    Without those libraries it falls back to the C++ restatement in oracle/ (kind "port")."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    want = oracle_threads()
    import chain_harness as ch
    import orc

    ref = reference_shaders()

    o = ch.Opts(denoise_iterations=DENOISE_ITERATIONS)
    sw, sh = (960, 540) if (args.cpu_width, args.cpu_height) == (0, 0) else (args.cpu_width, args.cpu_height)
    K, Wm = args.steps, args.warmup
    inp = ch.make_inputs(sw, sh, 2, reference_env=True)
    frames = inp.frames
    cores = int(orc.lib().orc_num_threads())

    def step_block(n):
        inp.frames = [frames[i % 2] for i in range(n)]
        return ch.run_oracle_chain(inp, o, capture=("composed",), lean=True, impl=ref)

    step_block(Wm)
    t0 = time.perf_counter()
    last = step_block(K)[-1]["composed"]
    dt = (time.perf_counter() - t0) / K
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, composed=last)
    v = round(sw * sh / 1e6 / dt, 4)
    line = {"metric": "SSGI+denoise Mpixels/s at 4K", "value": v, "unit": "Mpixels/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": K, "warmup": Wm,
            "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"C3 SSGI+PoissonDenoise(denoiseIterations={DENOISE_ITERATIONS})+compose, " +
                                   ("the reference's own fragment shaders compiled for the CPU (oracle/_ref)" if ref else "CPU restatement (oracle/)") +
                                   f", bounded sample {sw}x{sh} per step (1/16 of the 4K frame), {cores} OpenMP threads"},
            "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": cores, "threads_requested": want, "kind": "reference" if ref else "port",
                             "sample": f"{K} steps x one {sw}x{sh} frame (1/16 of the 4K frame)"},
            "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, help="timed steps (default 100; --impl reference: 20, a CPU step takes ~0.5 s)")
    ap.add_argument("--warmup", type=int, help="untimed steps before them (default 10; --impl reference: 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", type=int, default=WIDTH)
    ap.add_argument("--height", type=int, default=HEIGHT)
    ap.add_argument("--cpu-width", type=int, default=0, help="--impl reference: sample size per step (default 960x540)")
    ap.add_argument("--cpu-height", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="N = 1: skip the CPU oracle frame (and the parity field computed from it)")
    ap.add_argument("--no-configs", action="store_true", help="N = 1: skip the C1 / C2 / C4 block")
    ap.add_argument("--no-c5", action="store_true", help="N > 1: skip the 7680x4320 measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the last timed step to DIR/composed.npy (N = 1 and --impl reference)")
    args = ap.parse_args()
    cpu = args.impl == "reference"
    if args.steps is None:
        args.steps = 20 if cpu else 100
    if args.warmup is None:
        args.warmup = 3 if cpu else 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.dump_outputs and not cpu and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs: the row-sharded run (N > 1) has no single output plane to write")
    if args.impl == "reference":
        run_reference(args)
    elif int(os.environ.get("WORLD_SIZE", "1")) > 1:
        run_sharded(args)
    else:
        run_single(args)


if __name__ == "__main__":
    main()
