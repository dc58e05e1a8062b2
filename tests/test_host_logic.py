"""CPU tests of the host-side logic that surrounds the kernels: camera math, blue-noise index sequence,
env-map CDF tables, the synthetic generator's plane layouts."""
import json
import os

import numpy as np
import torch

import chain_harness as ch
from realism_effects_b200 import abi, synth


def test_camera_matrices_follow_threejs_conventions():
    cam = synth.Camera(aspect=16 / 9)
    u = cam.uniforms()
    P = u["projection"].reshape(4, 4).T
    # three.js makePerspective: te[11] = -1, te[15] = 0, te[14] = -2fn/(f-n)
    assert P[3, 2] == -1 and P[3, 3] == 0
    assert np.isclose(P[2, 3], -2 * 250 * 0.01 / (250 - 0.01))
    assert np.isclose(P[1, 1], 1 / np.tan(np.radians(20)))
    assert np.allclose(P @ u["projection_inverse"].reshape(4, 4).T, np.eye(4), atol=1e-4)
    Wm = u["camera_matrix_world"].reshape(4, 4).T
    assert np.allclose(Wm @ u["view_matrix"].reshape(4, 4).T, np.eye(4), atol=1e-5)
    assert np.allclose(Wm[:3, 3], [0, 8.75, 25]) and np.allclose(Wm[:3, 2], [0, 0, 1])  # looks down -z


def test_blue_noise_index_sequence():
    """BlueNoiseUtils.js:19-28: index_n = (start + index_{n-1} + 1) % 0x7fffffff, index_0 = 0"""
    start, c, seen = 1234567, 0, []
    for _ in range(5):
        c = ch.next_blue(start, c)
        seen.append(c)
    assert seen == [1234568, 2469136, 3703704, 4938272, 6172840]
    assert ch.next_blue(0x7FFFFFF0, 0x7FFFFFF0) == (0x7FFFFFF0 * 2 + 1) % 0x7FFFFFFF


def test_env_cdf_tables():
    env = synth.synthetic_env(64, 32).astype(np.float32)
    marg, cond, total = synth.build_env_cdf(env)
    assert marg.shape == (32,) and cond.shape == (32, 64)
    assert (np.diff(marg) >= 0).all() and (np.diff(cond, axis=1) >= 0).all()
    assert ((marg * 32 - 0.5) % 1 == 0).all() and ((cond * 64 - 0.5) % 1 == 0).all()  # half-texel centred indices
    lum = 0.2126 * env[..., 0] + 0.7152 * env[..., 1] + 0.0722 * env[..., 2]
    assert np.isclose(total, lum.astype(np.float64).sum(), rtol=1e-6)
    # importance: the brightest row must own more of the [0,1) range than a dark one
    rows = ((marg * 32 - 0.5)).astype(int)
    counts = np.bincount(rows, minlength=32)
    assert counts[np.argmax(lum.sum(1))] >= counts[np.argmin(lum.sum(1))]
    # A4: with flipY the reference's in-place "un-flip" mirrors the top half
    m2, c2, t2 = synth.build_env_cdf(env, flip_y=True)
    mirrored = env.copy()
    for y in range(32):
        mirrored[31 - y] = mirrored[y]
    m3, c3, t3 = synth.build_env_cdf(mirrored)
    assert np.array_equal(m2, m3) and np.array_equal(c2, c3) and t2 == t3
    assert not np.array_equal(m2, marg)


def test_synthetic_planes_follow_reference_layouts():
    fr = synth.render_frame(64, 36, t=1)
    d, g, v = fr.depth.numpy(), fr.gbuffer.numpy(), fr.velocity.numpy()
    bg = d == 1.0
    assert 0.05 < bg.mean() < 0.5 and (d[~bg] < 1).all() and (d[~bg] > 0.99).all()
    assert (g[bg] == [0, 0, 0, 1]).all() and (v[bg] == [0, 0, 0, 1]).all()         # cleared targets
    assert np.array_equal(v[..., 3], d)                                             # velocity.a = depth
    assert np.array_equal(v[~bg][:, 2].view(np.uint32), g[~bg][:, 1].view(np.uint32))  # same packed oct normal
    assert np.abs(v[~bg][:, :2]).max() > 1e-5                                       # camera moved between t-1 and t
    st = synth.render_frame(64, 36, t=1, static=True)
    assert not st.velocity.numpy()[..., :2].any()
    # packed albedo byte 3 (alpha = 1.0 -> 254 after the ONE_SAFE clamp) keeps the float away from NaN/Inf bit patterns
    bits = g[~bg][:, 0].view(np.uint32)
    assert ((bits >> 24) == 254).all()
    assert fr.direct_light.dtype == torch.float16 and tuple(fr.direct_light.shape) == (36, 64, 4)


def test_chain_option_mirrors_defaults():
    """Opts defaults == src/ssgi/SSGIOptions.js:26-48"""
    o = ch.Opts()
    assert (o.distance, o.thickness, o.denoise_iterations, o.radius, o.phi, o.luma_phi, o.depth_phi, o.normal_phi, o.roughness_phi, o.specular_phi,
            o.env_blur, o.steps, o.refine_steps) == (10, 10, 1, 3, 0.5, 5, 2, 50, 50, 50, 0.5, 20, 5)
    assert o.flags == abi.SSGI_IMPORTANCE_SAMPLING | abi.SSGI_USE_DIRECT_LIGHT | abi.SSGI_USE_ENVMAP
    assert ch.max_mip_level(1024, 512) == 11.0


def test_traa_jitter_r2_sequence_and_view_offset():
    """TRAA projection jitter (VERDICT r1 row V1): generateR2 (QuasirandomGenerator.js:11-24), r2Sequence / jitter (TAAUtils.js:3-11),
    three.js PerspectiveCamera.setViewOffset -> updateProjectionMatrix, and the un-jittered projection K2 uploads
    (TemporalReprojectPass.js:168-186)."""
    from realism_effects_b200 import effects

    g = 1.32471795724474602596090885447809
    pts = effects.generateR2(5)
    base = 1.1127756842787055
    for n, (a, b) in enumerate(pts):
        assert a == (base + n / g) % 1 and b == (base + n / (g * g)) % 1 and 0 <= a < 1 and 0 <= b < 1
    assert len(effects.r2Sequence) == 256 and all(-0.5 <= x < 0.5 and -0.5 <= y < 0.5 for x, y in effects.r2Sequence)
    # low discrepancy: 256 points cover a 8x8 grid with every cell hit
    cells = {(int((x + 0.5) * 8), int((y + 0.5) * 8)) for x, y in effects.r2Sequence}
    assert len(cells) == 64
    W, H = 1920, 1080
    cam = synth.Camera(aspect=W / H)
    P0 = cam.proj.copy()
    frame = 37
    effects.jitter(W, H, cam, frame)
    x, y = effects.r2Sequence[frame]
    # a view offset of (x, y) pixels shifts the frustum: only the third column of the projection changes, by 2x/W and -2y/H (NDC per pixel)
    assert np.allclose(cam.proj[:, [0, 1, 3]], P0[:, [0, 1, 3]])
    assert np.isclose(cam.proj[0, 2] - P0[0, 2], 2 * x / W) and np.isclose(cam.proj[1, 2] - P0[1, 2], -2 * y / H)
    # a point at the centre of the image moves by exactly (x, y) pixels... in the opposite direction of the window shift
    p = np.array([0.3, -0.2, -5.0, 1.0])
    ndc0, ndc1 = (P0 @ p)[:2] / (P0 @ p)[3], (cam.proj @ p)[:2] / (cam.proj @ p)[3]
    assert np.allclose((ndc1 - ndc0) * np.array([W, H]) / 2, [-x, y])
    # K2 sees the un-jittered matrix while the camera stays jittered
    assert np.array_equal(cam.unjittered_uniforms()["projection"], synth.col_major32(P0)) and not np.array_equal(cam.proj, P0)
    cam.clearViewOffset()
    assert np.array_equal(cam.proj, P0)
    effects.jitter(W, H, object(), 3)  # cameras without setViewOffset are left alone (TAAUtils.js:8)


JS_TABLES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_js_tables.json")


def reference_js_tables() -> dict:
    """the reference's option tables and index exports, as tests/golden/make_golden.py parsed them from its JS files"""
    with open(JS_TABLES, encoding="utf-8") as f:
        return json.load(f)


def test_option_defaults_equal_the_reference_js_tables():
    """the option tables of effects.py and js/index.js against the reference's own files (SSGIOptions.js, TemporalReprojectPass.js,
    PoissonDenoisePass.js, AOEffect.js, MotionBlurEffect.js)"""
    import re

    from realism_effects_b200 import effects

    ref = reference_js_tables()
    tables = [("defaultSSGIOptions", effects.defaultSSGIOptions), ("defaultTemporalReprojectPassOptions", effects.defaultTemporalReprojectPassOptions),
              ("defaultPoissonBlurOptions", effects.defaultPoissonBlurOptions), ("defaultAOOptions", effects.defaultAOOptions)]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    js = open(os.path.join(root, "js", "index.js"), encoding="utf-8").read()
    for name, mine in tables:
        want = ref[name]
        assert len(want) >= 5, (name, want)
        for k, v in want.items():
            assert k in mine, (name, k)
            got = mine[k]
            assert (got == v) or (isinstance(v, float) and float(got) == v), (name, k, got, v)
        # the ES-module mirror carries the same literal values
        m = re.search(r"export const " + name + r"\s*=\s*\{(.*?)\n\}", js, flags=re.S)
        assert m, f"js/index.js lacks {name}"
        for k, v in want.items():
            lit = "true" if v is True else "false" if v is False else "null" if v is None else (f'"{v}"' if isinstance(v, str) else None)
            if lit is None:
                assert re.search(r"\b" + k + r":\s*" + re.escape(("%g" % v)) + r"\b", m.group(1)), (name, k, v)
            else:
                assert re.search(r"\b" + k + r":\s*" + re.escape(lit), m.group(1)), (name, k, v)
    assert ref["MotionBlurEffect.defaultOptions"] == {k: float(v) for k, v in effects.defaultMotionBlurOptions.items()}


def test_plugin_surface_exports_every_class_of_the_reference_index():
    """src/index.js:16-31 exports 14 names; effects.py and js/index.js carry all of them (the compute behind each is an rfx_* entry point)"""
    import re

    names = set(reference_js_tables()["index.js exports"])
    assert len(names) == 14
    from realism_effects_b200 import effects

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    js = set(re.findall(r"export class (\w+)", open(os.path.join(root, "js", "index.js"), encoding="utf-8").read()))
    for n in names:
        assert hasattr(effects, n), f"effects.py lacks {n}"
        assert n in js, f"js/index.js lacks {n}"
