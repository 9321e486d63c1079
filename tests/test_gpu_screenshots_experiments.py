"""After the pass on the GPU (SURVEY 8 row f3): screenshots through vkr_take_screenshot and a short run of the experiment list.

The writers and the frame timer are tested on the CPU (tests/test_output.py); here the frames come from the shading kernel:
the *.png must hold the 8-bit quantisation of the sRGB frame, the *.hdr the half-precision linear frame rebuilt from the two
half-bit frames -- both compared with the oracle's frame for the same inputs (exact up to the file formats' precision)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from tests import harness as H
from tests.test_output import _read_hdr, _read_png
from vulkan_renderer_b200 import api, experiments as E

pytestmark = pytest.mark.gpu


def _frame_and_inputs(width, height):
	info = H.dataset("mini_city"); oi = H.OracleInputs(info)
	frame = H.open_frame(info)
	frame.configure(sample_count=2, strategy=api.STRATEGY_DIFFUSE_SPECULAR_MIS, heuristic=api.MIS_OPTIMAL_CLAMPED, trace_shadow_rays=1, show_lights=1)
	constants = frame.constants(width, height)
	vis = oi.visibility(width, height, constants); gb = oi.gbuffer(width, height, constants, vis)
	targets = api.RenderTargets()
	assert frame.lib.vkr_create_render_targets(C.byref(targets), C.byref(frame.device), width, height) == 0
	assert frame.lib.vkr_upload_gbuffer(C.byref(targets), C.byref(frame.device), np.ascontiguousarray(gb, dtype=np.float32).ctypes.data_as(C.c_void_p)) == 0
	return frame, oi, constants, gb, targets


def test_png_screenshot_is_the_quantised_srgb_frame(tmp_path):
	width, height = 96, 56
	frame, oi, constants, gb, targets = _frame_and_inputs(width, height)
	try:
		p = frame.create_pass(width, height)
		path = str(tmp_path / "shot.png")
		assert frame.lib.vkr_take_screenshot(C.byref(p), C.byref(frame.device), constants, len(constants), targets.d_gbuffer, path.encode(), None) == 0
		assert frame.lib.vkr_take_screenshot(C.byref(p), C.byref(frame.device), constants, len(constants), targets.d_gbuffer, path.encode(), path.encode()) == 1   # cannot mix LDR and HDR
		ref, _ = oi.shade(dict(H.oracle_config(frame, width, height), output_srgb=1), constants, gb)
	finally:
		frame.lib.vkr_destroy_render_targets(C.byref(targets), C.byref(frame.device)); frame.close()
	expected = np.floor(np.clip(ref[..., :3], 0.0, 1.0).astype(np.float32) * np.float32(255.0) + np.float32(0.5)).astype(np.uint8)
	shot = _read_png(path)
	assert shot.shape == (height, width, 3) and np.array_equal(shot, expected)
	assert shot.max() > 32


def test_hdr_screenshot_is_the_half_precision_linear_frame(tmp_path):
	width, height = 96, 56
	frame, oi, constants, gb, targets = _frame_and_inputs(width, height)
	try:
		p = frame.create_pass(width, height)
		path = str(tmp_path / "shot.hdr")
		assert frame.lib.vkr_take_screenshot(C.byref(p), C.byref(frame.device), constants, len(constants), targets.d_gbuffer, None, path.encode()) == 0
		assert p.desc.output_srgb == 0                                  # the pass is left as it was
		ref, _ = oi.shade(H.oracle_config(frame, width, height), constants, gb)
	finally:
		frame.lib.vkr_destroy_render_targets(C.byref(targets), C.byref(frame.device)); frame.close()
	half = ref[..., :3].astype(np.float16).astype(np.float64)          # packHalf2x16: round to nearest even
	shot = _read_hdr(path)
	peak = half.max(axis=-1, keepdims=True)
	assert (np.abs(shot - half) <= peak / 128.0 + 1e-30).all()
	assert shot.max() > 0.05


def test_a_slice_of_the_experiment_list_runs_and_reports(tmp_path):
	"""Three entries of the timing matrix (128 quads, central) at a reduced resolution: records, file names with the frame time, pictures."""
	todo = [e for e in E.timing_experiments() if e["name"] in ("timings_central_4_128_projected_solid_angle_ours", "timings_central_4_128_solid_angle_ours", "timings_central_4_128_area_turk")]
	assert len(todo) == 3
	records = E.run(todo, str(tmp_path / "data"), str(tmp_path / "out"), json_path=str(tmp_path / "out" / "timings.json"), frames=5, warmup=2, width=160, height=90)
	assert [r["name"] for r in records] == [e["name"] for e in todo]
	assert json.load(open(tmp_path / "out" / "timings.json")) == records
	pictures = []
	for r in records:
		assert r["light_count"] == 128 and r["light_vertex_counts"] == [4] and r["frame_time_ms"] > 0.0 and r["kernel_ms_min"] <= r["frame_time_ms"] <= r["kernel_ms_max"]
		# the name carries the raw median time at 3 decimals, the record the same time rounded to 4: the name is what a time within half a unit
		# of the record's last digit prints as
		t = r["frame_time_ms"]
		assert os.path.basename(r["screenshot"]) in {"%s_%.3f.png" % (r["name"], t + d) for d in (-0.00005, 0.0, 0.00005)}
		pictures.append(_read_png(r["screenshot"]).astype(np.float64))
		assert pictures[-1].shape == (90, 160, 3) and pictures[-1].mean() > 2.0
	# unbiased techniques of the same scene: the same picture up to noise
	assert abs(pictures[1].mean() / pictures[0].mean() - 1.0) < 0.2 and abs(pictures[2].mean() / pictures[0].mean() - 1.0) < 0.2
