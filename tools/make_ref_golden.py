#!/usr/bin/env python3
"""Freezes outputs of the REFERENCE's own code (its shader sources compiled as C++ and its host loaders compiled against shim/, both by
oracle/build_ref.py into oracle/_ref) as golden fixtures, so that the tests compare with the reference without needing it.

  python tools/make_ref_golden.py [shader] [digests] [fuzz] [host]      (default: all; needs the reference's sources)

shader   tests/golden/ref_shader.npz: for every configuration in oracle/_ref/configs.json a 64x48 frame of a seeded synthetic scene
         shaded by the reference shader; inputs are identified by sha256 of the scene file and the constant block is stored, so a drift
         of the synthetic-data generator is detected instead of silently changing the fixture's meaning.
digests  tests/golden/ref_shader_digests.json: sha256 of the reference shader's frames and of their inputs (constant block, visibility
         buffer), keyed "<configuration>@<width>x<height>": every fixture of ref_shader.npz shaded again from the fixture's inputs, and a
         spread of configurations at 40x30 and 97x41 (with a fixed sample of their pixels, tests/ref_frames.pixel_sample).
fuzz     tests/golden/ref_fuzz.json: the same digests and pixel samples for the random frames of tools/fuzz_parity.py, seed 202 (tests/test_fuzz_parity.py).
host     tests/golden/ref_host.json: what the reference's loaders and host maths produce for the synthetic data sets and the random lights
         and cameras of tests/test_ref_host.py (small values as they are, large buffers as sha256).
"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import harness as H  # noqa: E402
from tests.ref_frames import WIDTH, HEIGHT, camera_trials, dataset_for, digest, host_constants, light_trials, pixel_sample  # noqa: E402
from oracle import ref_binding as R  # noqa: E402
from vulkan_renderer_b200 import api  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# tests/test_ref_shader.py::test_oracle_follows_the_live_reference_shader_at_other_resolutions: every strategy, related-work techniques, error display, textures
RESOLUTION_PICKS = ["s0_h0_b0_L3_V4_S3_t1_l1_M8", "s1_h1_b0_L3_V4_S3_t1_l1_M8", "s2_h0_b0_L3_V4_S3_t1_l1_M8", "s3_h3_b0_L3_V4_S3_t1_l1_M8", "s4_h0_b0_L3_V4_S3_t1_l1_M8",
	"s3_h4_b0_L3_V4_S3_t1_l1_M8", "s3_h3_b1_L3_V4_S3_t1_l1_M8", "s3_h3_b0_L3_V7m5_S3_t1_l1_M8", "s3_h3_b0_L32_V4_S2_t1_l1_M8",
	"s0_h0_b0_L3_V4_S3_t1_l1_M8_q3", "s0_h0_b0_L3_V4_S3_t1_l1_M8_q9", "s1_h0_b0_L3_V4_S3_t1_l1_M8_q10", "s0_h0_b0_L3_V7m5_S3_t1_l1_M8_q7",
	"s3_h3_b0_L3_V4_S3_t1_l1_M8_e4", "s3_h3_b0_L3_V4_S3_t1_l1_M8_x1"]
RESOLUTIONS = [(40, 30), (97, 41)]
FUZZ_FRAMES, FUZZ_SEED = 16, 202


def _write_json(name, data):
	with open(os.path.join(GOLDEN, name), "w") as f:
		json.dump(data, f, indent=1, sort_keys=True)
		f.write("\n")


def shader():
	out = {}
	for cfg in R.configs():
		name = dataset_for(cfg)
		info = H.dataset(name); oi = H.OracleInputs(info)
		constants = host_constants(info, WIDTH, HEIGHT, cfg["lights"], frame_bits=cfg.get("frame_bits", 0))
		vis = oi.visibility(WIDTH, HEIGHT, constants)
		ref = R.shade(cfg["entry"], WIDTH, HEIGHT, cfg, constants, vis, oi.vks, oi.material_params, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris, textures=oi.textures, light_textures=oi.light_textures)
		key = cfg["name"]
		out[key + "/rgba"] = ref
		out[key + "/visibility"] = vis
		out[key + "/constants"] = np.frombuffer(constants, dtype=np.uint8)
		out[key + "/vks_sha256"] = np.frombuffer(hashlib.sha256(open(info["vks"], "rb").read()).digest(), dtype=np.uint8)
		print(key, "mean radiance", float(ref[..., :3].mean()))
	np.savez_compressed(os.path.join(GOLDEN, "ref_shader.npz"), **out)


def digests():
	live = {c["name"]: c for c in R.configs()}
	out = {}
	g = np.load(os.path.join(GOLDEN, "ref_shader.npz"))
	for name in sorted({k.split("/")[0] for k in g.files}):   # the fixtures' own inputs, as tests/test_ref_shader.py feeds them to the live shader
		cfg = live[name]
		info = H.dataset(dataset_for(cfg)); oi = H.OracleInputs(info)
		constants = bytes(g[name + "/constants"]); vis = g[name + "/visibility"]
		ref = R.shade(cfg["entry"], WIDTH, HEIGHT, cfg, constants, vis, oi.vks, oi.material_params, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris, textures=oi.textures, light_textures=oi.light_textures)
		out["%s@%dx%d" % (name, WIDTH, HEIGHT)] = {"inputs_sha256": digest(constants, vis), "rgba_sha256": digest(ref)}
	for width, height in RESOLUTIONS:
		for name in RESOLUTION_PICKS:
			cfg = live[name]
			info = H.dataset(dataset_for(cfg)); oi = H.OracleInputs(info)
			constants = host_constants(info, width, height, cfg["lights"])
			vis = oi.visibility(width, height, constants)
			ref = R.shade(cfg["entry"], width, height, cfg, constants, vis, oi.vks, oi.material_params, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris, textures=oi.textures, light_textures=oi.light_textures)
			out["%s@%dx%d" % (name, width, height)] = {"inputs_sha256": digest(constants, vis), "rgba_sha256": digest(ref), "rgba_sample": pixel_sample(ref)}
	_write_json("ref_shader_digests.json", out)


def fuzz():
	sys.path.insert(0, os.path.join(ROOT, "tools"))
	import fuzz_parity
	record = {}
	mismatches, compared, _ = fuzz_parity.run(frames=FUZZ_FRAMES, seed=FUZZ_SEED, with_reference=True, verbose=True, record=record)
	assert compared["reference vs oracle"] == FUZZ_FRAMES and not any(mismatches.values())
	_write_json("ref_fuzz.json", {"frames": FUZZ_FRAMES, "seed": FUZZ_SEED, "reference": record})


def host():
	lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_host.so"))
	lib.ref_probe_material_name.restype = C.c_char_p
	lib.ref_probe_material_name.argtypes = [C.c_uint64]
	lib.ref_probe_sizes.restype = C.c_uint32
	out = {"struct_sizes": [lib.ref_probe_sizes(i) for i in range(5)], "scenes": {}}
	for name in ("cornell", "mini_city"):
		info = H.dataset(name)
		tri = C.c_uint64(); mat = C.c_uint64(); fs = (C.c_float * 6)(); pos = C.c_void_p(); nuv = C.c_void_p(); mi = C.c_void_p(); soup = C.POINTER(C.c_float)(); ntri = C.c_uint64()
		assert lib.ref_probe_load_scene(info["vks"].encode(), info["textures"].encode(), C.byref(tri), C.byref(mat), fs, C.byref(pos), C.byref(nuv), C.byref(mi), C.byref(soup), C.byref(ntri)) == 0
		n = tri.value
		texels = []
		for m in range(mat.value):
			texels.append([])
			for t in range(3):
				texel = (C.c_uint16 * 8)()
				fmt = lib.ref_probe_material_texel(C.c_uint64(m), t, texel)
				texels[-1].append({"format": fmt, "rgba": [float(v) for v in np.frombuffer(bytes(texel), dtype=np.float16)[:4]]})
		out["scenes"][name] = {
			"vks_sha256": digest(open(info["vks"], "rb").read()), "triangle_count": n, "material_count": mat.value, "dequantization": list(fs),
			"positions_sha256": digest(np.ctypeslib.as_array(C.cast(pos, C.POINTER(C.c_uint32)), (3 * n, 2))),
			"normals_uv_sha256": digest(np.ctypeslib.as_array(C.cast(nuv, C.POINTER(C.c_uint16)), (3 * n, 4))),
			"material_indices_sha256": digest(np.ctypeslib.as_array(C.cast(mi, C.POINTER(C.c_uint8)), (n,))),
			"soup_triangle_count": ntri.value, "soup_sha256": digest(np.ctypeslib.as_array(soup, (ntri.value, 9))),
			"material_names": [lib.ref_probe_material_name(m).decode() for m in range(mat.value)], "material_texels": texels}
		lib.ref_probe_destroy_scene()
	info = H.dataset("cornell")
	res = C.c_uint32(); t0 = C.c_void_p(); t1 = C.c_void_p(); consts = (C.c_float * 8)()
	assert lib.ref_probe_load_ltc(info["ltc"].encode(), 51, C.byref(res), C.byref(t0), C.byref(t1), consts) == 0
	r = res.value
	out["ltc"] = {"resolution": r, "table0_sha256": digest(np.ctypeslib.as_array(C.cast(t0, C.POINTER(C.c_uint16)), (51, r, r, 4))),
		"table1_sha256": digest(np.ctypeslib.as_array(C.cast(t1, C.POINTER(C.c_uint16)), (51, r, r, 2))), "constants": bytes(consts).hex()}
	lib.ref_probe_destroy_ltc()
	out["noise"] = []
	for animate in (0, 1):
		data = C.c_void_p(); masks = (C.c_uint32 * 7)()
		assert lib.ref_probe_load_noise(256, 256, 64, 0, C.byref(data), masks, animate) == 0
		out["noise"].append({"data_sha256": digest(np.ctypeslib.as_array(C.cast(data, C.POINTER(C.c_uint16)), (64 * 256 * 256 * 4,))), "masks": list(masks)})
		lib.ref_probe_destroy_noise()
	rng = np.random.default_rng(11)
	out["lights_sha256"] = []
	for n, light, vp in light_trials(rng):
		ref_bytes = (C.c_uint8 * 160).from_buffer_copy(bytes(light)[:160])
		vw = np.zeros((n, 4), dtype=np.float32); fa = np.zeros((n - 2, 4), dtype=np.float32)
		lib.ref_probe_update_light(ref_bytes, n, vp.ctypes.data, vw.ctypes.data, fa.ctypes.data)
		out["lights_sha256"].append(digest(bytes(ref_bytes), vw, fa))
	out["cameras_sha256"] = []
	for cam, aspect in camera_trials(rng):
		a = (C.c_float * 16)()
		lib.ref_probe_world_to_projection(C.byref(cam), C.c_float(aspect), a)
		out["cameras_sha256"].append(digest(bytes(a)))
	cb = host_constants(H.dataset("mini_city"), 320, 200, 3)
	w2p = np.frombuffer(cb[32:96], dtype=np.float32).reshape(4, 4).copy()
	w2p[:3, 3] = 0.0
	inv = (C.c_float * 16)()
	lib.ref_probe_matrix_inverse(w2p.ctypes.data, inv)
	out["inverse"] = {"input": w2p.tobytes().hex(), "output": bytes(inv).hex()}
	out["constants"] = {}
	for name, lights, width, height in [("cornell", 1, 128, 96), ("mini_city", 3, 320, 192), ("mini_room", 32, 64, 48)]:
		block = H.reference_constants(H.dataset(name), width, height, lights, sample_count=4)
		out["constants"]["%s_%d_%dx%d" % (name, lights, width, height)] = {"size": len(block), "sha256": digest(block)}
	_write_json("ref_host.json", out)


def main():
	if not R.available():
		sys.path.insert(0, os.path.join(ROOT, "oracle"))
		import build_ref
		build_ref.build()
	steps = {"shader": shader, "digests": digests, "fuzz": fuzz, "host": host}
	for name in sys.argv[1:] or list(steps):
		steps[name]()
		print("make_ref_golden: %s written" % name)


if __name__ == "__main__":
	main()
