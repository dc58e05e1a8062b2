"""The reference's own shaders run on the CPU (tests/refglsl.py) against the oracle, plus known-answer tests of the GLSL runtime
that executes them (oracle/ref/glsl_rt.h + oracle/ref/transpile.py).

* runtime tests: small GLSL programs written here whose results are known in closed form — they check the language semantics the
  reference shaders rely on (swizzle l-values, inout copy-back, array constructors, uint arithmetic, quad derivatives with
  helper lanes, discard / early return, sampler state).  They need only g++.
* pinning tests: the oracle must equal the reference shaders BIT FOR BIT, in every output of every pass call.  The reference's runs
  are stored as digests (tests/refpin.py, tests/golden/reference_pins.json, minted by tests/golden/make_golden.py), so these tests
  need no reference checkout.
"""
import numpy as np
import pytest

import chain_harness as ch
import orc
import refglsl
import refpin
from realism_effects_b200 import abi

F32, F16 = refglsl.F_RGBA32F, refglsl.F_RGBA16F


def run_glsl(name, body, W=8, H=6, uniforms=None, textures=(), outs=None):
    s = refglsl.Shader(name, glsl="varying vec2 vUv;\nuniform vec2 resolution;\n" + body)
    s.set(resolution=[W, H], **(uniforms or {}))
    for t in textures:
        s.tex(*t[:3], **(t[3] if len(t) > 3 else {}))
    return s.run(W, H, outs or [(F32, None)])


def test_runtime_swizzles_inout_arrays_and_uint_math():
    out = run_glsl("rt_lang", """
      struct P { vec3 c; float w; };
      void twice(inout vec3 v) { v *= 2.0; }
      void split(vec4 e, out vec2 a, out vec2 b) { a = e.xy; b = e.zw; }
      vec2 TAB[3] = vec2[](vec2(1.0, 2.0), vec2(3.0, 4.0), vec2(5.0, 6.0));
      void main() {
        vec4 v = vec4(1.0, 2.0, 3.0, 4.0);
        v.xy = v.yx;                 // aliasing swizzle assignment -> (2,1,3,4)
        twice(v.yzw);                // inout through a swizzle    -> (2,2,6,8)
        vec2 a, b;
        split(v, a, b);
        P p = P(vec3(a, b.x), b.y);  // struct constructor
        uvec4 u = uvec4(7, 7 * 15843, 7 * 31 + 4566, 7 * 2345 + 58585);
        u = u * 1664525u + 1013904223u;
        u.x += u.y * u.w;
        u = u ^ (u >> 16u);
        float s = 0.0;
        for (int i = 0; i < 3; i++) s += TAB[i].x * TAB[i].y;   // 2 + 12 + 30
        float h = unpackHalf2x16(packHalf2x16(vec2(0.1, -3.0))).y;
        gl_FragColor = vec4(p.c.x + p.c.y * 10.0 + p.c.z * 100.0 + p.w * 1000.0, float(u.x % 1000u), s, h);
      }""")[0]
    u = np.array([7, 7 * 15843, 7 * 31 + 4566, 7 * 2345 + 58585], np.uint32)
    u = u * np.uint32(1664525) + np.uint32(1013904223)
    u[0] += u[1] * u[3]
    u = u ^ (u >> np.uint32(16))
    assert np.all(out[..., 0] == 2 + 20 + 600 + 8000)
    assert np.all(out[..., 1] == float(int(u[0]) % 1000))
    assert np.all(out[..., 2] == 44.0) and np.all(out[..., 3] == -3.0)


def test_runtime_quad_derivatives_discard_and_helper_lanes():
    """fwidth over a quad is taken from all four pixels even when some of them left main() early or were discarded; a discarded
    fragment keeps the target's previous texel"""
    W, H = 8, 6
    prev = np.full((H, W, 4), 7.0, np.float32)
    out = run_glsl("rt_deriv", """
      void main() {
        vec2 p = vUv * resolution;            // pixel centre: x + 0.5
        if (p.x < 2.0) { gl_FragColor = vec4(-1.0); return; }     // columns 0,1 leave early (uniform within their quads)
        if (p.y > 4.0 && p.x > 6.0) { discard; return; }          // the last quad column of the last quad row is discarded
        float keyed = (p.x > 3.0 && p.x < 4.0) ? 100.0 : 0.0;     // column 3 carries a different value than column 2
        gl_FragColor = vec4(fwidth(p.x * p.y), dFdx(keyed), dFdy(p.y * p.y), 1.0);
      }""", W, H, outs=[(F32, prev)])[0]
    assert np.all(out[:, :2] == -1.0)
    assert np.all(out[4:, 6:] == 7.0)                                    # discarded: previous contents
    y, x = 1, 4                                                          # quad (4..5, 0..1): d/dx (x*y) = y + .5, d/dy = x + .5
    assert out[y, x, 0] == pytest.approx((y + 0.5) + (x + 0.5))
    assert np.all(out[:4, 2:4, 1] == 100.0)                              # fine derivative inside the quad of columns 2,3
    assert out[2, 4, 2] == pytest.approx(3.5 * 3.5 - 2.5 * 2.5)


def test_runtime_sampler_state_and_null_sampler():
    W, H = 4, 4
    tex = np.zeros((2, 2, 4), np.float32)
    tex[0, 0], tex[0, 1], tex[1, 0], tex[1, 1] = [0, 0, 0, 1], [1, 0, 0, 1], [0, 1, 0, 1], [1, 1, 0, 1]
    body = """
      uniform sampler2D a; uniform sampler2D b; uniform sampler2D none;
      void main() {
        vec4 n = textureLod(a, vec2(0.5), 0.0);       // NEAREST at the centre: texel (1,1)
        vec4 l = textureLod(b, vec2(0.5), 0.0);       // LINEAR at the centre: the mean of the four texels
        gl_FragColor = vec4(n.x + n.y, l.x, textureLod(none, vUv, 0.0).a, float(textureSize(a, 0).x) + texelFetch(a, ivec2(1, 0), 0).x);
      }"""
    out = run_glsl("rt_tex", body, W, H, textures=[("a", tex, F32), ("b", tex, F32, dict(linear=True))])[0]
    assert np.all(out[..., 0] == 2.0) and np.all(out[..., 1] == 0.5) and np.all(out[..., 2] == 1.0) and np.all(out[..., 3] == 3.0)


needs_ref = pytest.mark.skipif(not refglsl.available(), reason="neither the reference checkout nor prebuilt oracle/_ref libraries")


def bits(a):
    return np.ascontiguousarray(a).tobytes()


# ---- pinning cases: pass sequences run on the reference's shaders by tests/golden/make_golden.py (refpin.Record) and on the oracle by the
# tests below (refpin.Replay); `m` executes the passes
def chain_case(m, mode):
    """K1 -> K2 -> K3 x2 -> K4 with history over 3 frames, default options"""
    return ch.run_oracle_chain(ch.make_inputs(80, 45, 3), ch.Opts(mode=mode), capture=("composed",), lean=True, impl=m)


def effect_passes_case(m):
    """K5 (fog), K6 + AO denoise + K7, K8, TRAA K2 + K9"""
    inp = ch.make_inputs(64, 36, 2)
    f0, f1 = inp.frames
    H, W = f1["depth"].shape
    ao = m.hbao(ch.hbao_params(f1["cam"], 991), f1["depth"], inp.blue, np.zeros((H, W, 4), np.float16))
    ch.ao_denoise(m, f1, inp.blue, ao)
    m.ao_compose(ch.ao_compose_params(), f1["depth"], ao, f1["direct"])
    ch.traa_two_frames(m, f0, f1)
    m.traa_compose(f1["direct"])
    m.motion_blur(ch.motion_blur_params(W, H, frame=7), ch.rotation_velocity_field(W, H, f1["depth"]), f1["direct"], inp.blue)
    gi = np.random.default_rng(5).uniform(0, 2, (H, W, 4)).astype(np.float32)
    for exp2 in (False, True):
        m.ssgi_compose(f1["depth"], gi, f1["direct"], ch.fog_params(f1["cam"], exp2))
    m.ssgi_compose(f1["depth"], gi, f1["direct"])
    return ao


def cosmetic_case(m):
    """SharpnessEffect / LensDistortionEffect / GradualBackgroundEffect / SparkleEffect alone and merged in EffectPass order, and TAAPass"""
    inp = ch.make_inputs(96, 54, 2)
    f1 = inp.frames[1]
    outs = [m.effects(ch.fx_params(f1["cam"], effs, sp), f1["direct"], f1["depth"], f1["velocity"]) for effs, sp in ch.FX_CASES]
    hist = np.random.default_rng(1).integers(0, 256, (54, 96, 4), dtype=np.uint8)
    for p in ch.taa_cases():
        m.taa(p, f1["direct"], hist)
    return inp, outs


def orthographic_case(m, mode):
    """the `#else` branches of PERSPECTIVE_CAMERA (K1 ray set-up, getViewZ, the view directions of K2 and K4) through a three.js OrthographicCamera"""
    inp = ch.make_inputs(64, 40, 2, orthographic=True)
    return inp, ch.run_oracle_chain(inp, ch.Opts(mode=mode), capture=("composed",), lean=True, impl=m)


def random_option_sets_case(m):
    """tools/fuzz_pin.py in small: random uniform values, shader variants, frame sizes (odd, portrait) and camera motion, through the chain and
    each single pass"""
    import os
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import fuzz_pin

    rng = np.random.default_rng(20260923)
    for _ in range(4):
        n, bad = fuzz_pin.run_chain(*fuzz_pin.draw_chain(rng), ref=m)
        assert n > 0 and not bad, bad
    n, bad = fuzz_pin.run_passes(rng, ref=m)
    assert n == 11 and not bad, bad


PINNED = {  # case name in tests/golden/reference_pins.json -> pass sequence
    **{f"chain_mode{mode}": (lambda m, mode=mode: chain_case(m, mode)) for mode in (abi.MODE_SSGI, abi.MODE_SSR)},
    "effect_passes": effect_passes_case,
    "cosmetic_effects_and_taa": cosmetic_case,
    **{f"orthographic_mode{mode}": (lambda m, mode=mode: orthographic_case(m, mode)) for mode in (abi.MODE_SSGI, abi.MODE_SSR)},
    "random_option_sets": random_option_sets_case,
}


@pytest.mark.parametrize("mode", [abi.MODE_SSGI, abi.MODE_SSR])
def test_oracle_equals_reference_shaders_chain(mode):
    """every pass of every frame, bit for bit"""
    pin = refpin.Replay(f"chain_mode{mode}")
    out = chain_case(pin, mode)
    pin.finish()
    assert float(np.abs(out[2]["composed"]).max()) > 0.1  # the comparison is not of empty planes


def test_oracle_equals_reference_shaders_effect_passes():
    pin = refpin.Replay("effect_passes")
    ao = effect_passes_case(pin)
    pin.finish()
    assert float(ao[..., 3].astype(np.float32).min()) < 0.99


def test_oracle_equals_reference_shaders_cosmetic_effects_and_taa():
    pin = refpin.Replay("cosmetic_effects_and_taa")
    inp, outs = cosmetic_case(pin)
    pin.finish()
    f1 = inp.frames[1]
    for (effs, sp), a in zip(ch.FX_CASES, outs):
        if effs != [abi.FX_SPARKLE] or sp:  # (with the reference's orthographic getViewZ branch the sparkle term underflows on this scene)
            assert bits(a) != bits(f1["direct"])  # the effect does something
    fade = orc.effects(ch.fx_params(f1["cam"], [abi.FX_GRADUAL_BACKGROUND]), f1["direct"], f1["depth"], f1["velocity"]).astype(np.float32)
    assert len(np.unique(fade[..., 0])) > 50       # the blend towards the background colour is exercised, not saturated


@needs_ref
def test_prebuilt_reference_shaders_run_without_the_checkout():
    """what the GPU box does: no /root/reference there, only the libraries __graft_entry__.build() left in oracle/_ref (bench.py --impl reference, the
    `reference_shaders` leg of cpu_baseline).  A subprocess with RFX_REFERENCE_DIR pointing nowhere must still run the default chain through them."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    refglsl.prebuild()  # here (checkout present) this is a cache hit; it guarantees the manifest lists every standard variant
    code = ("import sys; sys.path.insert(0, 'tests'); import numpy as np, chain_harness as ch, refglsl, orc\n"
            "assert not refglsl.assemble.available() and refglsl.chain_available(0) and refglsl.chain_available(1)\n"
            "inp = ch.make_inputs(48, 32, 2); o = ch.Opts()\n"
            "a = ch.run_oracle_chain(inp, o, capture=('composed',), lean=True); b = ch.run_oracle_chain(inp, o, capture=('composed',), lean=True, impl=refglsl)\n"
            "assert a[1]['composed'].tobytes() == b[1]['composed'].tobytes(); print('ok')")
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "RFX_REFERENCE_DIR": "/nonexistent"}, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("mode", [abi.MODE_SSGI, abi.MODE_SSR])
def test_oracle_equals_reference_shaders_orthographic_camera(mode):
    pin = refpin.Replay(f"orthographic_mode{mode}")
    inp, a = orthographic_case(pin, mode)
    pin.finish()
    assert inp.frames[0]["cam"]["perspective"] is False and abi.make_camera(inp.frames[0]["cam"]).perspective == 0
    assert float(np.abs(np.asarray(a[1]["composed"], np.float32)).max()) > 0.1
    p = ch.Opts()  # and it is a different image from the perspective one on the same planes
    assert bits(ch.run_oracle_chain(ch.make_inputs(64, 40, 1), p, capture=("composed",), lean=True)[0]["composed"]) != bits(a[0]["composed"])


def test_random_option_sets_oracle_equals_reference_shaders():
    """every plane of the chain and of each single pass bit-equal between the oracle and the reference's shaders
    (profiles/r02_fuzz_pin_seed*.json: 460 cases, 0 differing pixels)"""
    pin = refpin.Replay("random_option_sets")
    random_option_sets_case(pin)
    pin.finish()
