"""Pins the CPU oracle against the REFERENCE's own shader sources.

tests/golden/ref_shader.npz holds frames shaded by src/shaders/shading_pass.frag.glsl (+ includes) compiled as C++
(oracle/build_ref.py, oracle/glsl_compat/). The oracle must reproduce them bit for bit, for every sampling strategy
and MIS heuristic of the projected-solid-angle technique and for the related-work techniques ("_q<technique>": Turk, Urena, Arvo, Hart; SURVEY 8 f4).
tests/golden/ref_shader_digests.json holds the sha256 of more of the reference shader's frames and of their inputs (tools/make_ref_golden.py digests):
the fixtures shaded again, and a spread of configurations at other resolutions.
"""
import hashlib
import json
import os
import re

import numpy as np
import pytest

from tests import harness as H
from tests.ref_frames import WIDTH, HEIGHT, dataset_for, digest, host_constants, oracle_cfg, sample_difference

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_shader.npz")
DIGESTS = os.path.join(os.path.dirname(GOLDEN), "ref_shader_digests.json")


def _golden():
	return np.load(GOLDEN)


def _digests(width, height):
	"""{configuration name: {"inputs_sha256", "rgba_sha256"[, "rgba_sample"]}} of the reference shader's frames at this resolution."""
	with open(DIGESTS) as f:
		suffix = "@%dx%d" % (width, height)
		return {k[:-len(suffix)]: v for k, v in json.load(f).items() if k.endswith(suffix)}


def _config_from_name(name):
	m = re.match(r"s(\d+)_h(\d+)_b(\d+)_L(\d+)_V(\d+)(?:m(\d+))?_S(\d+)_t(\d+)_l(\d+)_M(\d+)(?:_q(\d+))?(?:_e(\d))?(?:_x(\d))?(?:_y(\d))?(?:_o(\d)(\d))?$", name)
	s, h, b, L, V, Vmin, S, t, l, M, q, e, x, y, srgb, frame_bits = (int(x) if x is not None else None for x in m.groups())
	return dict(name=name, entry="ref_shade_" + name.replace("_x1", "").replace("_y1", ""), strategy=s, heuristic=h, biased=b, lights=L, max_vertices=V, min_vertices=V if Vmin is None else Vmin,
		samples=S, trace=t, show_lights=l, materials=M, technique=11 if q is None else q, error_display=e or 0, textured=x or 0, light_textures=y or 0, srgb=srgb or 0, frame_bits=frame_bits or 0)


def _names():
	return sorted({k.split("/")[0] for k in _golden().files})


@pytest.mark.parametrize("name", _names())
def test_oracle_reproduces_reference_shader_bit_for_bit(name):
	g = _golden(); cfg = _config_from_name(name)
	info = H.dataset(dataset_for(cfg)); oi = H.OracleInputs(info)
	sha = hashlib.sha256(open(info["vks"], "rb").read()).digest()
	assert bytes(g[name + "/vks_sha256"]) == sha, "the synthetic scene generator drifted: regenerate with tools/make_ref_golden.py"
	constants = host_constants(info, WIDTH, HEIGHT, cfg["lights"], frame_bits=cfg["frame_bits"])
	assert constants == bytes(g[name + "/constants"]), "the constant block drifted"
	vis = oi.visibility(WIDTH, HEIGHT, constants)
	assert np.array_equal(vis, g[name + "/visibility"])
	gb = oi.gbuffer(WIDTH, HEIGHT, constants, vis)
	out, _ = oi.shade(oracle_cfg(cfg), constants, gb)
	ref = g[name + "/rgba"]
	assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)), H.compare_radiance(out, ref)
	assert float(ref[..., :3].max()) > 0.0


def test_live_reference_shader_matches_fixture():
	"""Does not run the reference shader: each fixture frame, and its inputs, must match the sha256 of the frame the reference shader computed from
	those inputs, stored in ref_shader_digests.json (tools/make_ref_golden.py digests). This keeps the fixtures the oracle and the kernels are held
	to equal to what the reference computes."""
	g = _golden()
	stored = _digests(WIDTH, HEIGHT)
	assert sorted(stored) == _names()
	for name in _names():
		assert digest(bytes(g[name + "/constants"]), g[name + "/visibility"]) == stored[name]["inputs_sha256"], name
		assert digest(g[name + "/rgba"]) == stored[name]["rgba_sha256"], name


@pytest.mark.parametrize("width,height", [(40, 30), (97, 41)])
def test_oracle_follows_the_live_reference_shader_at_other_resolutions(width, height):
	"""The fixtures are 64x48; other resolutions move every pixel ray, sample and noise fetch. Does not run the reference shader: a spread of
	configurations (every strategy, related-work techniques, error display, textures) was shaded by it and stored as the sha256 of the inputs and
	frames plus a fixed sample of pixels (ref_shader_digests.json); the oracle's frames must match the digests, i.e. be bit-identical again."""
	stored = _digests(width, height)
	assert len(stored) == 15
	for name, digests in sorted(stored.items()):
		cfg = _config_from_name(name)
		info = H.dataset(dataset_for(cfg)); oi = H.OracleInputs(info)
		constants = host_constants(info, width, height, cfg["lights"])
		vis = oi.visibility(width, height, constants)
		assert digest(constants, vis) == digests["inputs_sha256"], (name, "the inputs drifted: regenerate with tools/make_ref_golden.py")
		gb = oi.gbuffer(width, height, constants, vis)
		out, _ = oi.shade(oracle_cfg(cfg, width, height), constants, gb)
		assert digest(out) == digests["rgba_sha256"], (name, "sampled pixels", sample_difference(out, digests["rgba_sample"]))


def test_every_light_texturing_technique_shapes_the_textured_fixture():
	"""The "_y1" fixtures exercise all three branches of get_polygon_radiance() (shading_pass.frag.glsl:155-181): replacing the texture of any one
	light (area, portal, IES profile) by white changes the oracle's frame, and the frame with all three equals the reference shader's (test above)."""
	g = _golden(); name = "s3_h3_b0_L3_V4_S3_t1_l1_M8_y1"; cfg = _config_from_name(name)
	info = H.dataset(dataset_for(cfg)); oi = H.OracleInputs(info)
	assert [l["texturing_technique"] for l in info["lights"][:3]] == [1, 2, 3]
	constants = bytes(g[name + "/constants"])
	gb = oi.gbuffer(WIDTH, HEIGHT, constants, g[name + "/visibility"])
	ref = g[name + "/rgba"]
	dims, offsets, data = oi.light_textures
	for i in range(3):
		d = dims.copy(); o = offsets.copy(); white = np.concatenate([data, np.ones(4, dtype=np.float32)])
		d[i] = (1, 1, 1); o[i] = len(data)
		out, _ = H.oracle.shade(oracle_cfg(cfg), constants, gb, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris, light_textures=(d, o, white))
		changed = (out.view(np.uint32) != ref.view(np.uint32)).any(axis=-1).mean()
		assert changed > 0.02, "light %d (technique %d) leaves the frame unchanged" % (i, i + 1)
