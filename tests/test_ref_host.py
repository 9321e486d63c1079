"""Boundary B1 (SURVEY 8b): the reference's UNCHANGED loader and host-maths sources, compiled against shim/ into
oracle/_ref/libref_host.so, load the synthetic datasets; what they upload through the shim must equal, byte for byte,
what libvkr_b200.so's own loaders produce. Also pins the host maths (update_polygonal_light, camera matrices,
matrix_inverse) of vkr_host.cpp against the reference's code. What the reference's code produced is stored in
tests/golden/ref_host.json (tools/make_ref_golden.py host): small values as they are, large buffers as sha256 digests."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from tests import harness as H
from tests.ref_frames import camera_trials, digest, host_constants, light_trials
from vulkan_renderer_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_host.json")


@pytest.fixture(scope="module")
def ref():
	with open(GOLDEN) as f:
		return json.load(f)


def test_struct_sizes(ref):
	assert ref["struct_sizes"] == [C.sizeof(api.Camera), C.sizeof(api.PolygonalLight), 88, 160, C.sizeof(api.LtcConstants)]


@pytest.mark.parametrize("name", ["cornell", "mini_city"])
def test_reference_load_scene_through_the_shim_equals_our_loader(ref, name):
	g = ref["scenes"][name]
	info = H.dataset(name)
	assert digest(open(info["vks"], "rb").read()) == g["vks_sha256"], "the synthetic scene generator drifted: regenerate with tools/make_ref_golden.py"
	n = g["triangle_count"]
	lib = api.load_library()
	scene = api.Scene()
	assert lib.vkr_load_scene(C.byref(scene), None, info["vks"].encode(), info["textures"].encode(), 1) == 0
	assert n == scene.triangle_count == info["triangle_count"] and g["material_count"] == scene.material_count
	assert g["dequantization"] == list(scene.dequantization_factor) + list(scene.dequantization_summand)
	vks = H.read_vks(info["vks"])
	assert digest(vks["positions"]) == g["positions_sha256"]
	assert digest(vks["normals_uv"]) == g["normals_uv_sha256"]
	assert digest(vks["material_indices"]) == g["material_indices_sha256"]
	# the triangle soup handed to vkCmdBuildAccelerationStructuresKHR (scene.c:175-209) == what our shadow BVH is built from
	assert g["soup_triangle_count"] == n
	assert digest(H.oracle.dequantize_for_bvh(vks["positions"], vks["factor"], vks["summand"]).astype(np.float32)) == g["soup_sha256"]
	# materials: names and the texel our constant-material model takes from each *.vkt
	mp = np.ctypeslib.as_array(scene.material_params, (scene.material_count, 8))
	for m in range(g["material_count"]):
		assert g["material_names"][m].encode() == scene.material_names[m]
		for t, cols in ((0, (0, 1, 2)), (1, (None, 3, 4)), (2, (5, 6, None))):
			texel = g["material_texels"][m][t]
			assert texel["format"] == 97
			for k, col in enumerate(cols):
				if col is not None:
					assert texel["rgba"][k] == mp[m, col]
	lib.vkr_destroy_scene(C.byref(scene), None)


def test_reference_ltc_and_noise_tables_through_the_shim(ref):
	info = H.dataset("cornell")
	lib = api.load_library()
	g = ref["ltc"]
	ltc = api.LtcTable()
	assert lib.vkr_load_ltc_table(C.byref(ltc), None, info["ltc"].encode(), 51) == 0
	r = g["resolution"]
	assert r == ltc.roughness_count == 64
	assert digest(np.ctypeslib.as_array(ltc.h_table0, (51, r, r, 4))) == g["table0_sha256"]
	assert digest(np.ctypeslib.as_array(ltc.h_table1, (51, r, r, 2))) == g["table1_sha256"]
	assert bytes(ltc.constants).hex() == g["constants"]
	lib.vkr_destroy_ltc_table(C.byref(ltc), None)
	for animate in (0, 1):
		g = ref["noise"][animate]
		noise = api.NoiseTable()
		assert lib.vkr_load_noise_table(C.byref(noise), None, 256, 256, 64, api.NOISE_WHITE) == 0
		assert digest(np.ctypeslib.as_array(noise.h_noise, (64 * 256 * 256 * 4,))) == g["data_sha256"]
		masks = (C.c_uint32 * 2)(); layer = C.c_uint32(); rnd = (C.c_uint32 * 4)()
		lib.vkr_set_noise_constants(masks, C.byref(layer), rnd, C.byref(noise), animate)
		assert g["masks"] == list(masks) + [layer.value] + list(rnd)
		lib.vkr_destroy_noise_table(C.byref(noise), None)


def test_host_maths_matches_the_reference_bit_for_bit(ref):
	"""Per trial, the digest of what the reference's update_polygonal_light left (the first 160 bytes of the light, world-space vertices, fan areas)
	and of its world-to-projection matrix."""
	lib = api.load_library()
	rng = np.random.default_rng(11)
	for trial, (n, light, vp) in enumerate(light_trials(rng)):
		lib.vkr_set_polygonal_light_vertex_count(C.byref(light), n)
		C.memmove(light.vertices_plane_space, vp.ctypes.data, vp.nbytes)
		lib.vkr_update_polygonal_light(C.byref(light))
		ours = digest(bytes(light)[:160], np.ctypeslib.as_array(light.vertices_world_space, (n, 4)), np.ctypeslib.as_array(light.fan_areas, (n - 2, 4)))
		assert ours == ref["lights_sha256"][trial], trial
		lib.vkr_destroy_polygonal_light(C.byref(light))
	for trial, (cam, aspect) in enumerate(camera_trials(rng)):
		b = (C.c_float * 16)()
		lib.vkr_get_world_to_projection_space(b, C.byref(cam), C.c_float(aspect))
		assert digest(bytes(b)) == ref["cameras_sha256"][trial], trial


def test_constant_block_pixel_to_ray_uses_the_reference_inverse(ref):
	"""vkr_write_constants inverts the projection with the reference's cofactor expansion (math_utilities.h:24-46)."""
	info = H.dataset("mini_city")
	cb = host_constants(info, 320, 200, 3)
	w2p = np.frombuffer(cb[32:96], dtype=np.float32).reshape(4, 4).copy()
	w2p[:3, 3] = 0.0
	assert w2p.tobytes().hex() == ref["inverse"]["input"], "the constant block drifted: regenerate with tools/make_ref_golden.py"
	inv = np.frombuffer(bytes.fromhex(ref["inverse"]["output"]), dtype=np.float32).reshape(4, 4)
	vt = np.array([np.float32(2.0) / np.float32(320), np.float32(2.0) / np.float32(200)], dtype=np.float32)
	p2p = np.array([[vt[0], 0, np.float32(0.5) * vt[0] - np.float32(1)], [0, vt[1], np.float32(0.5) * vt[1] - np.float32(1)], [0, 0, 1], [0, 0, 1]], dtype=np.float32)
	expect = np.zeros((3, 4), dtype=np.float32)
	for i in range(3):
		for j in range(3):
			acc = np.float32(0)
			for k in range(4):
				acc = np.float32(acc + np.float32(inv[i, k] * p2p[k, j]))
			expect[i, j] = acc
	got = np.frombuffer(cb[96:144], dtype=np.float32).reshape(3, 4)
	assert np.array_equal(got.view(np.uint32), expect.view(np.uint32))


@pytest.mark.parametrize("name,lights,width,height", [("cornell", 1, 128, 96), ("mini_city", 3, 320, 192), ("mini_room", 32, 64, 48)])
def test_constant_block_equals_the_reference_host_code(ref, name, lights, width, height):
	"""vkr_write_constants against quick_load + write_constants of the reference (restated over its own structs and functions in oracle/ref_host_probe.c)."""
	info = H.dataset(name)
	ours = host_constants(info, width, height, lights, sample_count=4)
	theirs = ref["constants"]["%s_%d_%dx%d" % (name, lights, width, height)]
	assert len(ours) == theirs["size"]
	assert digest(ours) == theirs["sha256"]


def test_noise_blob_files_are_read_as_the_reference_lays_them_out(tmp_path, monkeypatch):
	"""The *.blob branch of load_noise_table (src/noise_table.c:76-107; the reference's timing runs use noise_type_ahmed, src/experiment_list.c:371): raw uint16 RGBA
	cells, layer-major, under data/noise/<type>_<w>x<h>_<layers>.blob. The reference's own loader cannot be the judge here: it formats the path with
	sprintf(file_path, file_path, ...) onto itself (noise_table.c:96, undefined behaviour; with this C library the path comes out empty and the load fails),
	so a synthetic blob is compared with what vkr_load_noise_table hands to the device; a missing file fails."""
	lib = api.load_library()
	monkeypatch.chdir(tmp_path)
	os.makedirs("data/noise")
	w, h, layers = 16, 8, 4
	rng = np.random.default_rng(3)
	cells = rng.integers(0, 65536, w * h * layers * 4, dtype=np.uint16)
	for noise_type, pattern in ((api.NOISE_AHMED, "data/noise/ahmed_2d_rgba_%02dx%02d_%02d.blob"), (api.NOISE_BLUE, "data/noise/blue_noise_rgba_%02dx%02d_%02d.blob")):
		noise = api.NoiseTable()
		assert lib.vkr_load_noise_table(C.byref(noise), None, w, h, layers, noise_type) != 0    # no file yet
		cells.tofile(pattern % (w, h, layers))
		assert lib.vkr_load_noise_table(C.byref(noise), None, w, h, layers, noise_type) == 0
		assert (noise.width, noise.height, noise.layers) == (w, h, layers)
		assert np.array_equal(np.ctypeslib.as_array(noise.h_noise, (len(cells),)), cells)
		masks = (C.c_uint32 * 2)(); layer = C.c_uint32(); rnd = (C.c_uint32 * 4)()
		lib.vkr_set_noise_constants(masks, C.byref(layer), rnd, C.byref(noise), 0)
		assert list(masks) == [w - 1, h - 1] and layer.value == layers - 1
		lib.vkr_destroy_noise_table(C.byref(noise), None)
