"""G-buffer ingest (SURVEY.md §8f row 2): the oracle's orc_gbuffer_ingest against (a) the torch restatement of the reference's packers
in realism_effects_b200/synth.py on identical inputs and (b) the reference's own packGBuffer / packNormal GLSL
(src/gbuffer/shader/gbuffer_packing.glsl) run through the GLSL runtime, stored as digests."""
import numpy as np
import torch

import orc
import refpin
from realism_effects_b200 import synth


def soa_frame(W=96, H=54, t=1):
    fr = synth.render_frame(W, H, t)
    s = {k: v.cpu().numpy() for k, v in fr.soa.items()}
    return fr, s


def test_oracle_ingest_equals_torch_packers():
    fr, s = soa_frame()
    gb, vel = orc.gbuffer_ingest(s["albedo"], s["normal"], s["material"], s["emissive"], s["motion"], fr.depth.numpy(), normalize_normals=False)
    # the torch packers on the same (quantised) inputs
    diffuse4 = torch.from_numpy(s["albedo"]).float() / 255.0
    mat = torch.from_numpy(s["material"]).float()
    em = torch.from_numpy(s["emissive"]).float()[..., :3]
    nrm = torch.from_numpy(s["normal"])[..., :3]
    want = synth.pack_gbuffer(diffuse4, nrm, mat[..., 0], mat[..., 1], em)
    clear = torch.tensor([0.0, 0.0, 0.0, 1.0])
    bg = fr.background
    want = torch.where(bg.unsqueeze(-1), clear, want).numpy()
    assert gb.view(np.uint32).tobytes() == want.view(np.uint32).tobytes()
    # with fp16-exact material values the ingested planes ARE the generator's planes; the velocity plane always is
    assert vel.view(np.uint32).tobytes() == fr.velocity.numpy().view(np.uint32).tobytes()
    assert (gb[..., :2].view(np.uint32) == fr.gbuffer.numpy()[..., :2].view(np.uint32)).all()      # diffuse + normal words


def test_ingest_options_and_formats():
    fr, s = soa_frame(64, 40)
    d = fr.depth.numpy()
    n16 = s["normal"].astype(np.float16)
    gb_a, vel_a = orc.gbuffer_ingest(s["albedo"], n16, s["material"], None, None, d)                     # no emissive, static, fp16 normals, normalised
    fg = d < 1.0
    assert (vel_a[..., :2] == 0).all() and (gb_a[fg][:, 3].view(np.uint32) == 0).all()
    assert (vel_a[..., 3] == d).all()
    gb_b, vel_b = orc.gbuffer_ingest(s["albedo"].astype(np.float16) / np.float16(255), s["normal"], (s["material"].astype(np.float32) * 255).round().astype(np.uint8),
                                     s["emissive"], s["motion"].astype(np.float16), d, motion_scale=(0.5, 0.5))
    assert np.allclose(vel_b[fg][:, :2], 0.5 * s["motion"][fg][:, :2], rtol=2e-3, atol=1e-7)
    bg = ~fg
    assert (gb_b[bg] == np.array([0, 0, 0, 1], np.float32)).all() and (vel_b[bg] == np.array([0, 0, 0, 1], np.float32)).all()


def packer_words(gbuffer, normal_word, fg, lit):
    """the words the ingest shares with the reference's packGBuffer / packNormal: diffuse, normal, roughness/metalness on the foreground,
    the RGBE8 emissive word where the shader's path is defined (`lit`), and the packed normal of the velocity plane"""
    return gbuffer[fg][:, :3].view(np.uint32), gbuffer[lit][:, 3].view(np.uint32), normal_word[fg].view(np.uint32)


def ingest_probe_inputs():
    """-> frame, SoA planes, foreground and lit masks, digest of the planes the packers read"""
    fr, s = soa_frame()
    depth = fr.depth.numpy()
    fg = depth < 1.0
    lit = fg & (s["emissive"][..., :3].astype(np.float32).max(-1) > 0)
    return fr, s, fg, lit, refpin.digest(s["albedo"], s["normal"], s["material"], s["emissive"], depth)


def test_oracle_ingest_equals_the_reference_packgbuffer_glsl():
    """against the outputs of the reference's gbuffer_packing.glsl run through the GLSL runtime (stored as digests by tests/golden/make_golden.py)"""
    fr, s, fg, lit, inputs = ingest_probe_inputs()
    want = refpin.load("ingest_packgbuffer")
    assert inputs == want["inputs"], "not the inputs the reference's packers were run on"
    gb, vel = orc.gbuffer_ingest(s["albedo"], s["normal"], s["material"], s["emissive"], s["motion"], fr.depth.numpy(), normalize_normals=False)
    assert lit.any()
    got = [refpin.digest(w) for w in packer_words(gb, vel[..., 2], fg, lit)]
    assert got == want["words"], "diffuse/normal/roughness-metalness, emissive, packNormal words vs the reference: " + str([g == w for g, w in zip(got, want["words"])])
