"""Frame set-up and random inputs shared by tools/make_ref_golden.py and the tests that compare with its fixtures (host-only, no GPU)."""
import ctypes as C
import hashlib

import numpy as np

from vulkan_renderer_b200 import api

WIDTH, HEIGHT = 64, 48


def digest(*parts):
	"""sha256 (hex) of the bytes of arrays / bytes objects, in order: equal digests mean bit-identical contents."""
	h = hashlib.sha256()
	for p in parts:
		h.update(p if isinstance(p, (bytes, bytearray)) else np.ascontiguousarray(p).tobytes())
	return h.hexdigest()


SAMPLE_PIXELS = 32


def pixel_sample(frame):
	"""A fixed, seeded sample of a frame's pixels (the same pixels for the same frame size): the hex of their float32 RGBA bits, stored next to a
	frame's digest so that a frame which no longer matches can be told how it differs."""
	h, w = frame.shape[:2]
	pixels = np.ascontiguousarray(frame, dtype=np.float32).reshape(h * w, -1)
	return [pixels[i].tobytes().hex() for i in np.sort(np.random.default_rng(0).choice(h * w, min(SAMPLE_PIXELS, h * w), replace=False))]


def sample_difference(frame, stored):
	"""How a frame's sampled pixels differ from a stored pixel_sample() (tests.harness.compare_radiance of the two samples)."""
	from tests import harness as H
	ours = np.array([np.frombuffer(bytes.fromhex(s), dtype=np.float32) for s in pixel_sample(frame)])
	theirs = np.array([np.frombuffer(bytes.fromhex(s), dtype=np.float32) for s in stored])
	return H.compare_radiance(ours, theirs)


def light_trials(rng, count=200):
	"""Random polygonal lights for the host maths (both windings: the plane gets flipped for clockwise polygons). Yields (vertex count, light
	before vkr_update_polygonal_light, plane-space vertices float32 [n, 4])."""
	for trial in range(count):
		n = int(rng.integers(3, 8))
		light = api.PolygonalLight()
		for i in range(3):
			light.rotation_angles[i] = rng.uniform(-3.2, 3.2); light.translation[i] = rng.uniform(-50, 50); light.radiant_flux[i] = rng.uniform(0.1, 100)
		light.scaling_x = rng.uniform(0.1, 5); light.scaling_y = rng.uniform(0.1, 5)
		ang = np.sort(rng.uniform(0, 2 * np.pi, n))
		if trial % 2: ang = ang[::-1]
		vp = np.zeros((n, 4), dtype=np.float32); vp[:, 0] = np.cos(ang) * rng.uniform(0.5, 1.5); vp[:, 1] = np.sin(ang) * rng.uniform(0.5, 1.5)
		yield n, light, vp


def camera_trials(rng, count=200):
	"""Random cameras and aspect ratios for the world-to-projection matrix. Yields (camera, aspect)."""
	for _ in range(count):
		cam = api.Camera()
		for i in range(3): cam.position_world_space[i] = rng.uniform(-100, 100)
		cam.rotation_z = rng.uniform(-7, 7); cam.rotation_x = rng.uniform(0, 3.14); cam.vertical_fov = rng.uniform(0.3, 2.0); cam.near_plane = 0.05; cam.far_plane = 1000.0
		yield cam, np.float32(rng.uniform(0.5, 2.5))


def dataset_for(cfg):
	if cfg.get("textured", 0):
		return "mini_textured"
	if cfg.get("light_textures", 0):
		return "mini_lit"
	if cfg["materials"] == 3:
		return "cornell"
	if cfg["lights"] > 3:
		return "mini_room"
	if cfg["max_vertices"] >= 5:
		vmin = cfg.get("min_vertices", cfg["max_vertices"])
		return "mini_poly" if vmin != cfg["max_vertices"] else "mini_v%d" % cfg["max_vertices"]
	if cfg["max_vertices"] == 3:
		return "mini_tri"
	return "mini_mixed" if cfg.get("min_vertices", cfg["max_vertices"]) != cfg["max_vertices"] else "mini_city"


def host_constants(info, width, height, lights, sample_count=1, frame_bits=0):
	"""Constant block through the library's host-only loaders (device = NULL)."""
	lib = api.load_library()
	scene = api.Scene(); ltc = api.LtcTable(); noise = api.NoiseTable(); spec = api.SceneSpecification(); st = api.RenderSettings()
	assert lib.vkr_load_scene(C.byref(scene), None, info["vks"].encode(), info["textures"].encode(), 0) == 0
	assert lib.vkr_load_ltc_table(C.byref(ltc), None, info["ltc"].encode(), 51) == 0
	assert lib.vkr_load_noise_table(C.byref(noise), None, 256, 256, 64, api.NOISE_WHITE) == 0
	assert lib.vkr_quick_load(C.byref(spec), info["save"].encode()) == 0
	assert lights <= spec.polygonal_light_count
	assert lib.vkr_create_and_assign_light_textures(None, None, C.byref(spec)) == 0   # texture indices only (src/main.c:2167)
	spec_count = spec.polygonal_light_count
	spec.polygonal_light_count = lights
	lib.vkr_specify_default_render_settings(C.byref(st)); st.animate_noise = 0; st.exposure_factor = 1.0; st.sample_count = sample_count
	size = lib.vkr_get_constants_size(C.byref(spec)); buf = (C.c_uint8 * size)()
	lib.vkr_write_constants(buf, C.byref(spec), C.byref(st), C.byref(scene), C.byref(ltc), C.byref(noise), width, height)
	if frame_bits:
		lib.vkr_set_frame_bits(buf, frame_bits)
	spec.polygonal_light_count = spec_count
	lib.vkr_destroy_scene_specification(C.byref(spec)); lib.vkr_destroy_noise_table(C.byref(noise), None); lib.vkr_destroy_ltc_table(C.byref(ltc), None); lib.vkr_destroy_scene(C.byref(scene), None)
	return bytes(buf)


def oracle_cfg(cfg, width=WIDTH, height=HEIGHT):
	return dict(width=width, height=height, light_count=cfg["lights"], max_light_vertex_count=cfg["max_vertices"], min_light_vertex_count=cfg.get("min_vertices", cfg["max_vertices"]),
		sample_count=cfg["samples"], sampling_strategies=cfg["strategy"], mis_heuristic=cfg["heuristic"], biased_sampling=cfg["biased"],
		trace_shadow_rays=cfg["trace"], show_polygonal_lights=cfg["show_lights"], output_srgb=cfg.get("srgb", 0), polygon_sampling_technique=cfg.get("technique", 11), error_display=cfg.get("error_display", 0))
