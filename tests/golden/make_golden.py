"""Mint the golden fixtures from THE REFERENCE'S OWN SHADERS, compiled for the CPU (tests/refglsl.py: the GLSL under the reference's
src/, assembled like the reference's JS assembles it, run on oracle/ref/glsl_rt.h), and from the reference's JS option tables.

    python tests/golden/make_golden.py [chains] [pins] [js]     # all three by default; needs the reference checkout (RFX_REFERENCE_DIR)

The reference ships no golden vectors of its own (SURVEY.md §4/§8c); these are outputs of the reference itself run here.
tests/test_oracle_chain_cpu.py checks the C++ oracle against them on any machine (no checkout needed), the `-m gpu` tests check
the CUDA engine against them.  Inputs are stored with the outputs so the fixtures do not depend on the synthetic generator.
  chain_96x54.npz      SSGI chain (K1 -> K2 -> K3 x2 -> K4), 2 frames, steps 12 / refine 3  + K5..K9 and the AO denoise on frame 1
  chain_ssr_64x36.npz  SSR chain (mode "ssr": 1-plane K2/K3, TYPE_SPECULAR compose), 3 frames
  reference_pins.json  the pinning cases of tests/test_reference_glsl.py (PINNED) run on the reference's shaders: per pass call, digests
                       of its inputs and outputs (tests/refpin.py); and the packGBuffer / packNormal probe of tests/test_ingest_cpu.py.
                       Inputs come from the synthetic generator: a change to it needs a re-mint.
  reference_js_tables.json  the reference's option defaults and index exports (tests/test_host_logic.py)
"""
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import chain_harness as ch  # noqa: E402
import refglsl as ref  # noqa: E402  (the reference shaders; NOT the oracle)
from realism_effects_b200 import abi  # noqa: E402


def store_inputs(d, inp):
    d.update(env_map=inp.env_map, env_marginal=inp.env_marginal, env_conditional=inp.env_conditional, env_total=np.float64(inp.env_total))
    for t, fr in enumerate(inp.frames):
        for k in ("depth", "gbuffer", "velocity", "direct"):
            d[f"f{t}_{k}"] = fr[k]
        for k, v in fr["cam"].items():
            d[f"f{t}_cam_{k}"] = np.asarray(v)
        d[f"f{t}_moved"] = np.int32(fr["moved"])


def mint_chains():
    o = ch.Opts(steps=12, refine_steps=3)
    inp = ch.make_inputs(96, 54, 2)
    out = ch.run_oracle_chain(inp, o, impl=ref)
    d = {}
    store_inputs(d, inp)
    for t in range(2):
        for k in ("ssgi", "tr0", "tr1", "dn0", "dn1", "composed"):
            d[f"f{t}_out_{k}"] = out[t][k]
    f0, f1 = inp.frames
    H, W = f1["depth"].shape
    ao = ref.hbao(ch.hbao_params(f1["cam"], 4242), f1["depth"], inp.blue, np.zeros((H, W, 4), np.float16))
    d["hbao"] = ao
    d["ao_composed"] = ref.ao_compose(ch.ao_compose_params(), f1["depth"], ao, f1["direct"])
    vel = ch.rotation_velocity_field(W, H, f1["depth"])
    d["mb_velocity"] = vel
    d["motion_blur"] = ref.motion_blur(ch.motion_blur_params(W, H), vel, f1["direct"], inp.blue)
    d["traa_compose"] = ref.traa_compose(f1["direct"])
    d["ao_dn_a"], d["ao_dn_b"] = ch.ao_denoise(ref, f1, inp.blue, ao)
    d["traa_h0"], d["traa_h1"] = ch.traa_two_frames(ref, f0, f1)
    d["k5_plain"] = ref.ssgi_compose(f1["depth"], out[1]["composed"], f1["direct"])
    d["k5_fog"] = ref.ssgi_compose(f1["depth"], out[1]["composed"], f1["direct"], ch.fog_params(f1["cam"], False))
    d["k5_fog_exp2"] = ref.ssgi_compose(f1["depth"], out[1]["composed"], f1["direct"], ch.fog_params(f1["cam"], True))
    path = os.path.join(HERE, "chain_96x54.npz")
    np.savez_compressed(path, **d)
    print("wrote", path, os.path.getsize(path), "bytes")

    o = ch.Opts(mode=abi.MODE_SSR)
    inp = ch.make_inputs(64, 36, 3)
    out = ch.run_oracle_chain(inp, o, impl=ref)
    d = {}
    store_inputs(d, inp)
    for t in range(3):
        for k in ("ssgi", "tr0", "dn0", "composed"):
            d[f"f{t}_out_{k}"] = out[t][k]
    path = os.path.join(HERE, "chain_ssr_64x36.npz")
    np.savez_compressed(path, **d)
    print("wrote", path, os.path.getsize(path), "bytes")


GLSL_INGEST = """
uniform sampler2D tAlbedo; uniform sampler2D tNormal; uniform sampler2D tMaterial; uniform sampler2D tEmissive;
layout(location = 0) out vec4 oG;
layout(location = 1) out vec4 oN;
%s
void main() {
  vec4 m = textureLod(tMaterial, vUv, 0.);
  vec3 n = textureLod(tNormal, vUv, 0.).xyz;
  oG = packGBuffer(textureLod(tAlbedo, vUv, 0.), n, m.r, m.g, textureLod(tEmissive, vUv, 0.).rgb);
  oN = vec4(packNormal(n), 0., 0., 1.);
}
"""


def mint_pins():
    import refpin
    import test_ingest_cpu
    import test_reference_glsl

    pins = {}
    for name, case in test_reference_glsl.PINNED.items():
        rec = refpin.Record(ref)
        case(rec)
        pins[name] = rec.log
        print(name, len(rec.log), "pass calls")
    fr, s, fg, lit, inputs = test_ingest_cpu.ingest_probe_inputs()
    H, W = fr.depth.shape
    sh = ref.Shader("ingest_probe", glsl="varying vec2 vUv;\n" + GLSL_INGEST % ref.assemble.read("gbuffer/shader/gbuffer_packing.glsl"))
    sh.tex("tAlbedo", s["albedo"], ref.F_RGBA8)
    sh.tex("tNormal", s["normal"], ref.F_RGBA32F)
    sh.tex("tMaterial", s["material"], ref.F_RGBA16F)
    sh.tex("tEmissive", s["emissive"], ref.F_RGBA16F)
    ref_g, ref_n = sh.run(W, H, [(ref.F_RGBA32F, None), (ref.F_RGBA32F, None)])
    pins["ingest_packgbuffer"] = dict(inputs=inputs, words=[refpin.digest(w) for w in test_ingest_cpu.packer_words(ref_g, ref_n[..., 0], fg, lit)])
    path = os.path.join(HERE, "reference_pins.json")
    with open(path, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v, separators=(',', ':'))}" for k, v in pins.items()) + "\n}\n")
    print("wrote", path, os.path.getsize(path), "bytes")


def _js_object(text: str, name: str) -> dict:
    """the flat `const <name> = { key: literal, ... }` object literal of a reference JS file -> dict (numbers, booleans, strings, null)"""
    m = re.search(r"(?:const|let)\s+" + re.escape(name) + r"\s*=\s*\{(.*?)\n\}", text, flags=re.S)
    assert m, name
    out = {}
    for key, val in re.findall(r"^\s*(\w+)\s*:\s*([^,\n/]+?)\s*,?\s*(?://.*)?$", m.group(1), flags=re.M):
        v = val.strip()
        if v in ("true", "false"):
            out[key] = v == "true"
        elif v == "null":
            out[key] = None
        elif v[0] in "\"'":
            out[key] = v[1:-1]
        else:
            try:
                out[key] = float(v)
            except ValueError:
                pass  # an expression (new Color(...), a spread): compared elsewhere
    return out


def mint_js_tables():
    rd = ref.assemble.read  # paths under the reference's src/
    d = {name: _js_object(rd(rel), name) for rel, name in [
        ("ssgi/SSGIOptions.js", "defaultSSGIOptions"), ("temporal-reproject/TemporalReprojectPass.js", "defaultTemporalReprojectPassOptions"),
        ("denoise/pass/PoissonDenoisePass.js", "defaultPoissonBlurOptions"), ("ao/AOEffect.js", "defaultAOOptions")]}
    mb = re.search(r"const defaultOptions = \{([^}]*)\}", rd("motion-blur/MotionBlurEffect.js")).group(1)
    d["MotionBlurEffect.defaultOptions"] = {k: float(v) for k, v in re.findall(r"(\w+):\s*([\d.]+)", mb)}
    idx = re.search(r"export \{(.*?)\}", rd("index.js"), flags=re.S).group(1)
    d["index.js exports"] = sorted(re.findall(r"^\s*(\w+),?\s*$", idx, flags=re.M))
    path = os.path.join(HERE, "reference_js_tables.json")
    with open(path, "w") as f:
        json.dump(d, f, indent=1)
        f.write("\n")
    print("wrote", path)


def main():
    assert ref.assemble.available(), "the reference checkout is needed"
    which = sys.argv[1:] or ["chains", "pins", "js"]
    for name, fn in (("chains", mint_chains), ("pins", mint_pins), ("js", mint_js_tables)):
        if name in which:
            fn()


if __name__ == "__main__":
    main()
