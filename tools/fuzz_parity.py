#!/usr/bin/env python3
"""Randomised differential test (TEST INFRASTRUCTURE; needs /root/reference, i.e. the build container):

  python tools/fuzz_parity.py [--frames 200] [--seed 0]

Every frame: one of the built shader configurations (oracle/_ref/configs.json), a random camera inside the scene, randomly moved / turned /
scaled lights (also behind surfaces, grazing, partly below horizons), random exposure / roughness factor / MIS visibility estimate. Then
  (1) the REFERENCE shader compiled as C++  vs  the oracle                                   -- pins the oracle beyond the frozen fixtures,
  (2) the DEVICE code compiled for the CPU (tests/device_on_host.cpp, rays off)  vs  the oracle -- the arithmetic the GPU kernels run.
All comparisons are bit for bit. Prints one line per mismatch and a summary; exit code 1 if anything differs."""
import argparse
import re
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import harness as H  # noqa: E402
from tests.ref_frames import dataset_for, digest, oracle_cfg, pixel_sample, sample_difference  # noqa: E402
from oracle import ref_binding as R  # noqa: E402
from vulkan_renderer_b200 import api  # noqa: E402


def perturb(lib, spec, st, info, cfg, rng, wild=False):
	"""Random camera, light transforms / fluxes and settings, written into the scene specification and render settings (shared with tests/test_gpu_zzw_fuzz.py)."""
	cam = spec.camera
	base = np.array(info["camera"]["position"], dtype=np.float64)
	for a in range(3):
		cam.position_world_space[a] = float(base[a] + rng.uniform(-2.0, 2.0) * (0.3 if a == 2 else 1.0))
	cam.rotation_z = float(info["camera"]["rotation_z"] + rng.uniform(-1.2, 1.2)); cam.rotation_x = float(np.clip(info["camera"]["rotation_x"] + rng.uniform(-0.7, 0.7), 0.05, 3.0))
	cam.vertical_fov = float(rng.uniform(0.5, 1.6))
	for i in range(cfg["lights"]):
		light = spec.polygonal_lights[i]
		for a in range(3):
			light.rotation_angles[a] = float(light.rotation_angles[a] + rng.uniform(-1.0, 1.0) * (1.0 if rng.random() < 0.7 else 3.0))
			light.translation[a] = float(light.translation[a] + rng.uniform(-1.5, 1.5) * (0.5 if a == 2 else 1.0))
			light.radiant_flux[a] = float(rng.uniform(1.0, 30.0))
		light.scaling_x = float(rng.uniform(0.1, 3.0)); light.scaling_y = float(rng.uniform(0.1, 3.0))
		if wild:   # needles, specks and walls of light; lights dropped into the ground plane or next to the camera
			light.scaling_x = float(10.0 ** rng.uniform(-3.0, 1.5)); light.scaling_y = float(10.0 ** rng.uniform(-3.0, 1.5))
			if rng.random() < 0.3: light.translation[2] = float(rng.uniform(-0.05, 0.05))
			if rng.random() < 0.2:
				for a in range(3): light.translation[a] = float(cam.position_world_space[a] + rng.uniform(-0.3, 0.3))
		lib.vkr_update_polygonal_light(C.byref(light))
	lib.vkr_specify_default_render_settings(C.byref(st)); st.animate_noise = 0
	st.exposure_factor = float(rng.uniform(0.5, 4.0)); st.roughness_factor = float(rng.uniform(0.3, 1.5)); st.mis_visibility_estimate = float(rng.uniform(0.0, 1.0))
	if wild:
		st.roughness_factor = float(10.0 ** rng.uniform(-2.0, 0.7)); st.mis_visibility_estimate = float(rng.choice([0.0, 1.0, rng.uniform(0.0, 1.0)])); st.exposure_factor = float(10.0 ** rng.uniform(-3.0, 3.0))
	st.error_min_exponent = float(rng.uniform(-7.0, -3.0)); st.sample_count = cfg["samples"]


def random_constants(info, cfg, width, height, rng, wild=False):
	lib = api.load_library()
	scene = api.Scene(); ltc = api.LtcTable(); noise = api.NoiseTable(); spec = api.SceneSpecification(); st = api.RenderSettings()
	assert lib.vkr_load_scene(C.byref(scene), None, info["vks"].encode(), info["textures"].encode(), 0) == 0
	assert lib.vkr_load_ltc_table(C.byref(ltc), None, info["ltc"].encode(), 51) == 0
	assert lib.vkr_load_noise_table(C.byref(noise), None, 256, 256, 64, api.NOISE_WHITE) == 0
	assert lib.vkr_quick_load(C.byref(spec), info["save"].encode()) == 0
	assert lib.vkr_create_and_assign_light_textures(None, None, C.byref(spec)) == 0
	count = spec.polygonal_light_count
	spec.polygonal_light_count = cfg["lights"]
	perturb(lib, spec, st, info, cfg, rng, wild)
	size = lib.vkr_get_constants_size(C.byref(spec)); buf = (C.c_uint8 * size)()
	lib.vkr_write_constants(buf, C.byref(spec), C.byref(st), C.byref(scene), C.byref(ltc), C.byref(noise), width, height)
	if cfg.get("frame_bits", 0):
		lib.vkr_set_frame_bits(buf, cfg["frame_bits"])
	spec.polygonal_light_count = count
	lib.vkr_destroy_scene_specification(C.byref(spec)); lib.vkr_destroy_noise_table(C.byref(noise), None); lib.vkr_destroy_ltc_table(C.byref(ltc), None); lib.vkr_destroy_scene(C.byref(scene), None)
	return bytes(buf)


_primary_bvh = {}


def device_on_host_visibility(dev, oi, constants, width, height):
	"""The body of visibility_kernel on the CPU: shader-side vertex decode (device function), the product's host BVH builder, closest_hit per pixel."""
	P = lambda a: a.ctypes.data_as(C.c_void_p)
	q = np.ascontiguousarray(oi.vks["positions"], dtype=np.uint32)
	key = (id(oi), constants[:32])   # the dequantisation constants decide the vertices
	if key not in _primary_bvh:
		cb = (C.c_uint8 * len(constants)).from_buffer_copy(constants)
		verts = np.zeros((len(q), 3), dtype=np.float32)
		dev.vkr_device_on_host_decode_positions(cb, P(q), C.c_uint64(len(q)), P(verts))
		lib = api.load_library(); PT = C.POINTER
		nodes = PT(C.c_float)(); tri = PT(C.c_float)(); ids = PT(C.c_uint32)(); nc = C.c_uint64(); md = C.c_uint32()
		tris = np.ascontiguousarray(verts.reshape(-1, 9))
		assert lib.vkr_bvh_build_probe(tris.ctypes.data, len(tris), C.byref(nodes), C.byref(nc), C.byref(tri), C.byref(ids), C.byref(md)) == 0
		n = len(tris)
		_primary_bvh[key] = (np.ctypeslib.as_array(nodes, (nc.value, 16)).copy(), np.ctypeslib.as_array(tri, (n, 12)).copy(), np.ctypeslib.as_array(ids, (n,)).copy())
		lib.vkr_bvh_free_probe(nodes, tri, ids)
	nodes, tri, ids = _primary_bvh[key]
	out = np.zeros((height, width), dtype=np.uint32)
	cb = (C.c_uint8 * len(constants)).from_buffer_copy(constants)
	dev.vkr_device_on_host_visibility(C.c_uint32(width), C.c_uint32(height), cb, P(nodes), P(tri), P(ids), C.c_uint32(len(ids)), P(out))
	return out


def device_on_host_gbuffer(dev, oi, constants, vis, width, height):
	"""The per-pixel body of the G-buffer kernel (csrc/vkr_gbuffer.cuh) on the CPU."""
	P = lambda a: a.ctypes.data_as(C.c_void_p)
	out = np.zeros((4, height, width, 4), dtype=np.float32)
	q = np.ascontiguousarray(oi.vks["positions"], dtype=np.uint32); nt = np.ascontiguousarray(oi.vks["normals_uv"], dtype=np.uint16)
	mi = np.ascontiguousarray(oi.vks["material_indices"], dtype=np.uint8); mp = np.ascontiguousarray(oi.material_params, dtype=np.float32)
	vis = np.ascontiguousarray(vis, dtype=np.uint32)
	if oi.textures is not None:
		dims3, offsets, data = oi.textures
		dims = np.zeros((len(dims3), 4), dtype=np.uint32); dims[:, :3] = dims3
		offsets_texels = (offsets // 4).astype(np.uint64); data = np.ascontiguousarray(data, dtype=np.float32)
		tex = (P(dims), P(offsets_texels), P(data))
	else:
		tex = (None, None, None)
	cb = (C.c_uint8 * len(constants)).from_buffer_copy(constants)
	dev.vkr_device_on_host_gbuffer(C.c_uint32(width), C.c_uint32(height), cb, P(vis), P(q), P(nt), P(mi), P(mp), tex[0], tex[1], tex[2], P(out))
	return out


def device_on_host_frame(dev, cfg, oi, constants, gb, width, height):
	"""Rays off. Returns None where tests/device_on_host.cpp has no entry for the configuration (error display with an sRGB / half-bit output stage)."""
	if cfg.get("error_display", 0) and (cfg.get("srgb", 0) or cfg.get("frame_bits", 0)):
		return None
	P = lambda a: a.ctypes.data_as(C.c_void_p)
	out = np.zeros((height, width, 4), dtype=np.float32)
	noise = np.ascontiguousarray(oi.noise, dtype=np.uint16); ltc0 = np.ascontiguousarray(oi.ltc0, dtype=np.uint16); ltc1 = np.ascontiguousarray(oi.ltc1, dtype=np.uint16)
	gb = np.ascontiguousarray(gb, dtype=np.float32)
	cb = (C.c_uint8 * len(constants)).from_buffer_copy(constants)
	table = (P(noise), C.c_uint32(noise.shape[2]), C.c_uint32(noise.shape[1]), C.c_uint32(noise.shape[0]), P(ltc0), P(ltc1), C.c_uint32(ltc0.shape[1]), C.c_uint32(ltc0.shape[0]))
	if cfg.get("error_display", 0):
		technique = cfg["technique"] if cfg["technique"] != 11 else (12 if cfg["biased"] else 11)
		rc = dev.vkr_device_on_host_error_display_frame(C.c_uint32(width), C.c_uint32(height), C.c_uint32(cfg["max_vertices"]), C.c_uint32(cfg["lights"]), C.c_uint32(technique),
			C.c_uint32(cfg["error_display"]), C.c_int(cfg["show_lights"]), cb, P(gb), *table, P(out))
	else:
		if oi.light_textures is not None:
			dims3, offsets, data = oi.light_textures
			dims = np.zeros((len(dims3), 4), dtype=np.uint32); dims[:, :3] = dims3
			offsets_texels = np.ascontiguousarray(offsets // 4, dtype=np.uint64); data = np.ascontiguousarray(data, dtype=np.float32)
			tex = (C.c_uint32(len(dims)), P(dims), P(offsets_texels), P(data))
		else:
			tex = (C.c_uint32(0), None, None, None)
		rc = dev.vkr_device_on_host_shade_frame(C.c_uint32(width), C.c_uint32(height), C.c_uint32(cfg["max_vertices"]), C.c_uint32(cfg["lights"]), C.c_uint32(cfg["technique"]), C.c_uint32(cfg["strategy"]),
			C.c_uint32(cfg["heuristic"]), C.c_int(cfg["biased"]), C.c_uint32(cfg["samples"]), C.c_int(cfg["show_lights"]), cb, P(gb), *table, C.c_int(cfg.get("srgb", 0)), *tex, P(out))
	assert rc == 0, cfg["name"]
	return out


def fixture_configs():
	"""The configurations of the frozen fixtures (tests/golden/ref_shader.npz): available without oracle/_ref."""
	from tests.test_ref_shader import _config_from_name
	g = np.load(os.path.join(ROOT, "tests", "golden", "ref_shader.npz"))
	return [_config_from_name(n) for n in sorted({k.split("/")[0] for k in g.files})]


def random_config(rng):
	"""Any legal combination of the run-time settings (src/user_interface.cpp:90-180), not only the ones a reference shader was compiled for: for the device code
	against the oracle. Vertex counts come with the data set."""
	dataset, vmax, vmin = [("mini_tri", 3, 3), ("mini_city", 4, 4), ("mini_mixed", 4, 3), ("mini_v5", 5, 5), ("mini_v6", 6, 6), ("mini_v7", 7, 7), ("mini_poly", 7, 5), ("mini_lit", 4, 4)][int(rng.integers(8))]
	cfg = dict(strategy=int(rng.integers(5)), heuristic=0, biased=0, lights=int(rng.integers(1, 4)), max_vertices=vmax, min_vertices=vmin, samples=int(rng.integers(1, 6)), trace=1,
		show_lights=int(rng.integers(2)), materials=8, technique=11, error_display=0, textured=0, light_textures=int(dataset == "mini_lit"), srgb=int(rng.random() < 0.2), frame_bits=int(rng.choice([0, 0, 0, 1, 2])))
	if dataset == "mini_poly" and cfg["lights"] < 3: cfg["min_vertices"] = [5, 5][cfg["lights"] - 1]   # lights are pentagon, heptagon, hexagon
	if dataset == "mini_mixed" and cfg["lights"] == 1: cfg["min_vertices"] = 3; 
	if dataset == "mini_mixed" and cfg["lights"] == 1: cfg["max_vertices"] = 4
	roll = rng.random()
	if roll < 0.35:   # related work (also under textured lights): diffuse only, or GGX MIS where the density stands alone
		cfg["technique"] = int(rng.integers(0, 11))
		ggx_ok = cfg["technique"] in (2, 3, 4, 5, 10)
		cfg["strategy"] = int(rng.integers(2)) if ggx_ok else 0
	elif roll < 0.5:
		cfg["biased"] = 1
	if cfg["strategy"] == 1: cfg["heuristic"] = int(rng.integers(2))
	if cfg["strategy"] == 3: cfg["heuristic"] = int(rng.integers(5))
	if cfg["technique"] in (10, 11) and rng.random() < 0.15 and not cfg["light_textures"]:
		cfg["error_display"] = int(rng.integers(1, 7)); cfg["srgb"] = 0; cfg["frame_bits"] = 0
		if cfg["error_display"] >= 4 and cfg["strategy"] < 2: cfg["strategy"] = 2 + int(rng.integers(3)); cfg["heuristic"] = 0
		if cfg["technique"] == 10:
			cfg["strategy"] = 0; cfg["heuristic"] = 0
			if cfg["error_display"] >= 3: cfg["error_display"] = 1 + int(rng.integers(2))
		if cfg["strategy"] == 3: cfg["heuristic"] = int(rng.integers(5))
	cfg["name"] = "any:%s s%d h%d b%d L%d S%d q%d e%d o%d%d" % (dataset, cfg["strategy"], cfg["heuristic"], cfg["biased"], cfg["lights"], cfg["samples"], cfg["technique"], cfg["error_display"], cfg["srgb"], cfg["frame_bits"])
	cfg["dataset"] = dataset
	return cfg


def run(frames, seed, width=48, height=32, max_samples=8, with_reference=True, verbose=True, only=None, wild=False, any_config=False, reference_digests=None, record=None):
	"""Returns (mismatches, compared): dicts with the keys "reference vs oracle" and "device code vs oracle".
	reference_digests: {frame index (str): {"inputs_sha256", "rgba_sha256", "rgba_sample"}} of the reference shader's frames for these arguments (tests/golden/ref_fuzz.json,
	written by tools/make_ref_golden.py); the oracle's frames are compared with them instead of running the reference shader. record: a dict that the
	live reference arm fills with those digests."""
	import __graft_entry__
	dev = C.CDLL(__graft_entry__.build_device_on_host())
	rng = np.random.default_rng(seed)
	# the fixture configurations (the same frames with and without the reference arm), or a second set compiled with
	# `python oracle/build_ref.py --random <count> <seed> <name>` and selected with VKR_REF_SET=<name>
	source = R.configs() if os.environ.get("VKR_REF_SET") else fixture_configs()
	configs = [dict(technique=11, error_display=0, srgb=0, frame_bits=0, textured=0, light_textures=0, **{"min_vertices": c["max_vertices"]}) | c for c in source if c["samples"] <= max_samples and (only is None or re.search(only, c["name"]))]
	keys = ("reference vs oracle", "device code vs oracle", "device G-buffer code vs oracle", "device visibility code vs oracle")
	mismatches = {k: 0 for k in keys}; compared = {k: 0 for k in keys}; lit = 0; pink = 0
	inputs = {}
	for f in range(frames):
		cfg = random_config(rng) if any_config else configs[int(rng.integers(len(configs)))]
		name = cfg.get("dataset") or dataset_for(cfg)
		if name not in inputs:
			info = H.dataset(name); inputs[name] = (info, H.OracleInputs(info))
		info, oi = inputs[name]
		w0, h0 = width, height
		width, height = w0 + int(rng.integers(0, 17)), h0 + int(rng.integers(0, 9))
		constants = random_constants(info, cfg, width, height, rng, wild)
		vis = oi.visibility(width, height, constants)
		gb = oi.gbuffer(width, height, constants, vis)
		host_vis = device_on_host_visibility(dev, oi, constants, width, height)
		compared["device visibility code vs oracle"] += 1
		if not np.array_equal(host_vis, vis):
			mismatches["device visibility code vs oracle"] += 1
			print("MISMATCH device visibility code vs oracle: frame %d seed %d %s %dx%d, %d pixels" % (f, seed, cfg["name"], width, height, int((host_vis != vis).sum())), flush=True)
		host_gb = device_on_host_gbuffer(dev, oi, constants, vis, width, height)
		compared["device G-buffer code vs oracle"] += 1
		if not np.array_equal(host_gb.view(np.uint32), np.ascontiguousarray(gb, dtype=np.float32).view(np.uint32)):
			mismatches["device G-buffer code vs oracle"] += 1
			print("MISMATCH device G-buffer code vs oracle: frame %d seed %d %s %dx%d" % (f, seed, cfg["name"], width, height), flush=True)
		out, _ = oi.shade(oracle_cfg(cfg, width, height), constants, gb)
		lit += int((out[..., :3].sum(-1) > 0).any()); pink += int(((out[..., 1] == 0) & (out[..., 0] > 0) & (out[..., 2] > 0)).any())
		if with_reference and reference_digests is not None:
			stored = reference_digests[str(f)]
			compared["reference vs oracle"] += 1
			if digest(constants, vis) != stored["inputs_sha256"]:
				mismatches["reference vs oracle"] += 1
				print("MISMATCH reference vs oracle: frame %d seed %d %s %dx%d: the inputs (constant block, visibility) differ from the stored frame's" % (f, seed, cfg["name"], width, height), flush=True)
			elif digest(out) != stored["rgba_sha256"]:
				mismatches["reference vs oracle"] += 1
				print("MISMATCH reference vs oracle: frame %d seed %d %s %dx%d, sampled pixels: %s" % (f, seed, cfg["name"], width, height, sample_difference(out, stored["rgba_sample"])), flush=True)
		elif with_reference:
			ref = R.shade(cfg["entry"], width, height, cfg, constants, vis, oi.vks, oi.material_params, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris, textures=oi.textures, light_textures=oi.light_textures)
			if record is not None:
				record[str(f)] = {"inputs_sha256": digest(constants, vis), "rgba_sha256": digest(ref), "rgba_sample": pixel_sample(ref)}
			compared["reference vs oracle"] += 1
			if not np.array_equal(out.view(np.uint32), ref.view(np.uint32)):
				mismatches["reference vs oracle"] += 1
				print("MISMATCH reference vs oracle: frame %d seed %d %s %dx%d %s" % (f, seed, cfg["name"], width, height, H.compare_radiance(out, ref)), flush=True)
		host = device_on_host_frame(dev, cfg, oi, constants, gb, width, height)
		if host is not None:
			no_rays, _ = oi.shade(oracle_cfg(dict(cfg, trace=0), width, height), constants, gb)
			compared["device code vs oracle"] += 1
			if not np.array_equal(host.view(np.uint32), no_rays.view(np.uint32)):
				mismatches["device code vs oracle"] += 1
				print("MISMATCH device code vs oracle: frame %d seed %d %s %dx%d %s" % (f, seed, cfg["name"], width, height, H.compare_radiance(host, no_rays)), flush=True)
		width, height = w0, h0
	if verbose:
		print("fuzz_parity: seed %d, %d frames (%d lit, %d with NaN-pink pixels); " % (seed, frames, lit, pink)
			+ "; ".join("%s: %d of %d differ" % (k, mismatches[k], compared[k]) for k in compared))
	return mismatches, compared, lit


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument("--frames", type=int, default=200)
	ap.add_argument("--seed", type=int, default=0)
	ap.add_argument("--width", type=int, default=48)
	ap.add_argument("--height", type=int, default=32)
	ap.add_argument("--max-samples", type=int, default=8, help="skip configurations with more samples per pixel (time)")
	ap.add_argument("--only", default=None, help="regular expression on the configuration name, e.g. '^s[0124]_' for the strategies other than MIS")
	ap.add_argument("--wild", action="store_true", help="extreme light sizes and positions, roughness factors, exposures")
	ap.add_argument("--any-config", action="store_true", help="any legal combination of settings instead of the compiled shader configurations (implies --no-reference)")
	ap.add_argument("--no-reference", action="store_true", help="device code vs oracle only (where oracle/_ref is not built)")
	args = ap.parse_args()
	if not (args.no_reference or args.any_config) and not R.available():
		raise SystemExit("oracle/_ref/libref_shader.so is not built (needs /root/reference); --no-reference compares the device code with the oracle only")
	mismatches, _, _ = run(args.frames, args.seed, args.width, args.height, args.max_samples, with_reference=not (args.no_reference or args.any_config), only=args.only, wild=args.wild, any_config=args.any_config)
	return 1 if any(mismatches.values()) else 0


if __name__ == "__main__":
	sys.exit(main())
