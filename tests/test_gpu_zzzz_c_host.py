"""Boundaries B1 + B2 with a plain C host (SURVEY 8b, INTEGRATION.md): tests/c_host/route_b.c loads a data set with the reference's UNCHANGED loaders
(compiled from /root/reference against shim/), hands their buffers and images to libvkr_b200.so and renders a frame through the C-ABI. The frame
must equal the oracle's, bit for bit. build() compiles the binary into oracle/_ref/route_b where the reference's sources are present; it travels prebuilt."""
import os
import subprocess

import numpy as np
import pytest

from tests import harness as H
from tests.ref_frames import host_constants
from vulkan_renderer_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BINARY = os.path.join(ROOT, "oracle", "_ref", "route_b")
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not os.path.exists(BINARY), reason="oracle/_ref/route_b not built (needs the reference's loader sources)")]


@pytest.mark.parametrize("name,width,height,spp", [("cornell", 128, 96, 2), ("mini_city", 160, 96, 2)])
def test_c_host_over_the_reference_loaders_renders_the_oracle_frame(tmp_path, name, width, height, spp):
	info = H.dataset(name)
	out = tmp_path / "frame.f32"
	run = subprocess.run([BINARY, info["vks"], info["textures"], info["save"], info["ltc"], str(width), str(height), str(spp), str(out)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
	assert run.returncode == 0, run.stdout
	frame = np.fromfile(out, dtype=np.float32).reshape(height, width, 4)
	oi = H.OracleInputs(info)
	lights = len(info["lights"])
	constants = host_constants(info, width, height, lights, sample_count=spp)
	vis = oi.visibility(width, height, constants)
	gb = oi.gbuffer(width, height, constants, vis)
	cfg = dict(width=width, height=height, light_count=lights, max_light_vertex_count=4, min_light_vertex_count=4, sample_count=spp,
		sampling_strategies=api.STRATEGY_DIFFUSE_SPECULAR_MIS, mis_heuristic=api.MIS_OPTIMAL_CLAMPED, biased_sampling=0, trace_shadow_rays=1, show_polygonal_lights=1, row_begin=0, row_end=0)
	ref, _ = H.oracle.shade(cfg, constants, gb, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris)
	assert np.array_equal(frame.view(np.uint32), ref.view(np.uint32)), H.compare_radiance(frame, ref)
