"""Randomised pinning: the oracle against the reference's own shaders (tests/refglsl.py) on random option sets.

    python tools/fuzz_pin.py --cases 40 --seed 1 [--json profiles/r02_fuzz_pin.json]

tools/pin_oracle.py checks a fixed matrix; this draws the options — every uniform-valued option of the chain (distance, thickness, envBlur,
radius, the five phis, blue-noise start, camera motion and field of view, frame size incl. odd and portrait, frame count), the shader-variant
options from small sets (steps, refineSteps, the four SSGI flags, SSGI/SSR, denoiseMode, denoiseIterations, resolutionScale), and the
parameters of the single passes (HBAO, ao_compose, motion blur, ssgi_compose fog, the cosmetic effects, TAAPass) — and compares every output
plane bit for bit.  Exits 1 on any differing pixel.  Needs the reference checkout; TEST INFRASTRUCTURE (tools/ is not the product).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import chain_harness as ch  # noqa: E402
import orc  # noqa: E402
import refglsl  # noqa: E402
from pin_oracle import PLANES, diff  # noqa: E402
from realism_effects_b200 import abi  # noqa: E402


def draw_chain(rng) -> tuple:
    W = int(rng.choice([33, 48, 57, 64, 80, 96]))
    H = int(rng.choice([24, 31, 40, 54, 72, 101]))  # some portrait (H > W): the Poisson taps' row reach grows with H/W
    F = int(rng.integers(1, 4))
    use_env = bool(rng.random() < 0.8)
    scale = float(rng.choice([1.0, 1.0, 0.5, 0.6, 0.75]))
    okw = dict(
        distance=float(rng.uniform(1.0, 25.0)), thickness=float(rng.uniform(0.2, 15.0)), env_blur=float(rng.uniform(0.0, 1.0)),
        radius=float(rng.uniform(1.0, 6.0)), phi=float(rng.uniform(0.05, 1.0)), luma_phi=float(rng.uniform(0.5, 20.0)),
        depth_phi=float(rng.uniform(0.5, 10.0)), normal_phi=float(rng.uniform(1.0, 80.0)), roughness_phi=float(rng.uniform(1.0, 80.0)),
        specular_phi=float(rng.uniform(1.0, 80.0)), denoise_iterations=int(rng.integers(1, 4)),
        steps=int(rng.choice([3, 8, 12, 20, 31])), refine_steps=int(rng.choice([0, 1, 3, 5])),
        importance_sampling=bool(rng.random() < 0.6), missed_rays=bool(rng.random() < 0.3), use_direct_light=bool(rng.random() < 0.7),
        use_envmap=use_env, mode=int(rng.choice([abi.MODE_SSGI, abi.MODE_SSGI, abi.MODE_SSR])), blue_noise_start=int(rng.integers(0, 1 << 20)),
        resolution_scale=scale, denoise_mode=int(rng.choice([0, 0, 0, 1, 2])))
    ikw = dict(static=bool(rng.random() < 0.2), fov=float(rng.uniform(25.0, 80.0)),
               cam_step=(float(rng.uniform(-0.08, 0.08)), float(rng.uniform(-0.03, 0.03)), float(rng.uniform(-0.1, 0.1))),
               orthographic=bool(rng.random() < 0.2))
    return W, H, F, okw, ikw


def run_chain(W, H, F, okw, ikw, ref=refglsl):
    o = ch.Opts(**okw)
    inp = ch.make_inputs(W, H, F, **ikw)
    planes = [p for p in PLANES if not (o.mode == abi.MODE_SSR and p in ("tr1", "dn1")) and not (o.denoise_mode != 0 and p in ("dn0", "dn1"))]
    if o.denoise_mode == 2:
        planes = [p for p in planes if p != "composed"]
    a = ch.run_oracle_chain(inp, o, capture=planes, lean=True)
    b = ch.run_oracle_chain(inp, o, capture=planes, lean=True, impl=ref)
    bad = {}
    for f, (x, y) in enumerate(zip(a, b)):
        for k in planes:
            d = diff(x[k], y[k])
            if d["n_px"]:
                bad[f"f{f}_{k}"] = d["n_px"]
    return len(planes) * F, bad


def run_passes(rng, ref=refglsl):
    """one random draw of every single-pass surface; returns (planes compared, {plane: differing pixels}).  `ref`: what the oracle is
    compared with (the reference's shaders, or tests/refpin.py's record / replay of them)"""
    W, H = int(rng.choice([40, 64, 96])), int(rng.choice([30, 54, 77]))
    ortho = bool(rng.random() < 0.3)
    inp = ch.make_inputs(W, H, 2, fov=float(rng.uniform(30.0, 75.0)), orthographic=ortho)
    f0, f1 = inp.frames
    z = np.zeros((H, W, 4), np.float16)
    n, bad = 0, {}

    def both(tag, fn):
        nonlocal n
        for i, (x, y) in enumerate(zip(fn(orc), fn(ref))):
            n += 1
            d = diff(x, y)
            if d["n_px"]:
                bad[f"{tag}[{i}]"] = d["n_px"]

    # K6 with random parameters (spp is a shader variant), one Poisson pass on it, K7
    hp = ch.hbao_params(f1["cam"], int(rng.integers(0, 1 << 20)), spp=int(rng.choice([4, 8, 16])))
    hp.ao_distance, hp.distance_power, hp.bias, hp.thickness = float(rng.uniform(0.5, 6.0)), float(rng.uniform(0.5, 3.0)), float(rng.uniform(5.0, 80.0)), float(rng.uniform(0.02, 0.5))
    acp = ch.ao_compose_params(power=float(rng.uniform(0.5, 4.0)), color=tuple(float(c) for c in rng.uniform(0, 1, 3)))

    def hbao(m):
        ao = m.hbao(hp, f1["depth"], inp.blue, z)
        p = ch.poisson_params(ch.Opts(radius=float(hp.ao_distance) + 1.0), 99, False)
        p.texture_count, p.gbuffer_texture, p.input_linear = 1, 0, 1
        p.is_texture_specular[:] = [0, 0]
        p.normal_phi, p.depth_phi, p.roughness_phi, p.specular_phi = 3.25, 2.0, 0.0, 0.0
        dn, _ = m.poisson_denoise(p, f1["depth"], f1["velocity"], ao, None, inp.blue, z, None)
        return ao, dn, m.ao_compose(acp, f1["depth"], dn, f1["direct"])

    both("hbao", hbao)

    # K8: samples is a shader variant; intensity/jitter uniforms; window size != buffer size
    vel = ch.rotation_velocity_field(W, H, f1["depth"], vmax=float(rng.uniform(0.005, 0.2)))
    mp = ch.motion_blur_params(W, H, frame=int(rng.integers(0, 4096)), samples=int(rng.choice([4, 8, 16])), delta_time=float(rng.uniform(1 / 240, 1 / 20)),
                               resolution=(int(rng.integers(200, 2000)), int(rng.integers(200, 1200))))
    for k in ("intensity", "jitter"):
        if hasattr(mp, k):
            setattr(mp, k, float(rng.uniform(0.2, 3.0)))
    both("motion_blur", lambda m: (m.motion_blur(mp, vel, f1["direct"], inp.blue),))

    # K5 with fog
    gi = rng.uniform(0, 3, (H, W, 4)).astype(np.float32)
    sp = abi.SsgiComposeParams()
    sp.use_fog, sp.fog_exp2, sp.perspective, sp.is_debug = int(rng.random() < 0.7), int(rng.random() < 0.5), int(not ortho), int(rng.random() < 0.2)
    sp.fog_color[:] = [float(c) for c in rng.uniform(0, 1, 3)]
    sp.fog_near, sp.fog_far, sp.fog_density = float(rng.uniform(0.5, 10.0)), float(rng.uniform(15.0, 60.0)), float(rng.uniform(0.005, 0.2))
    sp.camera_near, sp.camera_far = float(f1["cam"]["near"]), float(f1["cam"]["far"])
    both("ssgi_compose", lambda m: (m.ssgi_compose(f1["depth"], gi, f1["direct"], sp),))

    # K2 alone, SSGI form (2 planes), on frame 1 of a chain (real history), with the uniform-valued options drawn: maxBlend, neighborhoodClampIntensity,
    # keepData, fullAccumulate; and the shader-variant ones: logTransform, confidencePower
    rec = ch.run_oracle_chain(inp, ch.Opts(), capture=("ssgi",))[1]
    tp = rec["_k2_params"]
    tp.max_blend, tp.neighborhood_clamp_intensity = float(rng.uniform(0.5, 1.0)), float(rng.uniform(0.0, 1.0))
    tp.keep_data, tp.full_accumulate = float(rng.integers(0, 2)), int(rng.random() < 0.3)
    tp.log_transform, tp.confidence_power = int(rng.random() < 0.7), float(rng.choice([0.125, 0.75, 1.0, 4.0]))
    both("temporal_reproject", lambda m: m.temporal_reproject(tp, rec["ssgi"], f1["velocity"], rec["_k2_hist"][0], rec["_k2_hist"][1],
                                                               rec["_k2_prev_out"][0], rec["_k2_prev_out"][1]))

    # TRAA (K2 single plane + K9)
    both("traa", lambda m: ch.traa_two_frames(m, f0, f1))

    # cosmetic effects with random parameters, in a random EffectPass order
    ids = [abi.FX_SHARPNESS, abi.FX_LENS_DISTORTION, abi.FX_GRADUAL_BACKGROUND, abi.FX_SPARKLE]
    effs = [int(e) for e in rng.permutation(ids)[: int(rng.integers(1, 5))]]
    if abi.FX_LENS_DISTORTION in effs:  # a uv-transforming effect comes first in a merged EffectPass (postprocessing sorts by attributes); keep one order
        effs = [abi.FX_LENS_DISTORTION] + [e for e in effs if e != abi.FX_LENS_DISTORTION]
    fp = abi.make_effects_params(f1["cam"], effs, sharpness=float(rng.uniform(0.0, 3.0)), alphax=float(rng.uniform(-0.2, 0.2)), alphay=float(rng.uniform(-0.2, 0.2)),
                                 aberration=float(rng.uniform(0.0, 3.0)), background_color=tuple(float(c) for c in rng.uniform(0, 1, 3)),
                                 max_distance=float(rng.uniform(3.0, 40.0)), spread=float(rng.uniform(0.2, 3.0)), intensity=float(rng.uniform(0.2, 5.0)),
                                 sparkle_perspective=bool(rng.random() < 0.5), perspective=not ortho)
    both("cosmetic_effects", lambda m: (m.effects(fp, f1["direct"], f1["depth"], f1["velocity"]),))

    # TAAPass
    hist = rng.integers(0, 256, (H, W, 4), dtype=np.uint8)
    tp = abi.TaaParams()
    tp.camera_not_moved_frames, tp.srgb_output = float(rng.integers(0, 200)), int(rng.random() < 0.5)
    both("taa_pass", lambda m: (m.taa(tp, f1["direct"], hist),))
    return n, bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=20)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--json", type=str)
    ap.add_argument("--only", choices=("chain", "passes"))
    a = ap.parse_args()
    if not refglsl.assemble.available():
        sys.exit("the reference checkout is needed to build the shaders")
    rng = np.random.default_rng(a.seed)
    report, total_bad, total_planes = [], 0, 0
    t0 = time.time()
    for i in range(a.cases):
        if a.only != "passes":
            W, H, F, okw, ikw = draw_chain(rng)
            n, bad = run_chain(W, H, F, okw, ikw)
            total_planes += n
            total_bad += sum(bad.values())
            report.append(dict(kind="chain", size=[W, H], frames=F, opts=okw, inputs=ikw, planes=n, differing=bad))
            print(f"[{i:3d}] chain {W}x{H}x{F} mode={okw['mode']} dm={okw['denoise_mode']} it={okw['denoise_iterations']} steps={okw['steps']}/{okw['refine_steps']} "
                  f"scale={okw['resolution_scale']} ortho={int(ikw['orthographic'])} env={int(okw['use_envmap'])} is={int(okw['importance_sampling'])} mr={int(okw['missed_rays'])}: "
                  f"{n} planes, {'OK' if not bad else bad}", flush=True)
        if a.only != "chain":
            n, bad = run_passes(rng)
            total_planes += n
            total_bad += sum(bad.values())
            report.append(dict(kind="passes", planes=n, differing=bad))
            print(f"[{i:3d}] passes: {n} planes, {'OK' if not bad else bad}", flush=True)
    out = dict(seed=a.seed, cases=a.cases, planes_compared=total_planes, differing_pixels=total_bad, seconds=round(time.time() - t0, 1), cases_detail=report)
    print(f"fuzz: {a.cases} cases, {total_planes} planes compared, {total_bad} differing pixels, {out['seconds']} s")
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)
    sys.exit(1 if total_bad else 0)


if __name__ == "__main__":
    main()
