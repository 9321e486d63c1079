#!/usr/bin/env python3
"""Compiles the REFERENCE's own shading-pass sources into oracle/_ref/libref_shader.so (TEST INFRASTRUCTURE).

The reference's hot path is GLSL (src/shaders/shading_pass.frag.glsl and its includes). GLSL is close enough
to C++ that g++ compiles it against oracle/glsl_compat/glsl_compat.hpp after a mechanical syntax pass:

  * '#version' / '#extension' lines dropped, 'layout(...)' qualifiers stripped,
  * the uniform block 'per_frame_constants { ... }' opened up (its members become globals),
  * 'inout T x' / 'out T x' parameters become 'T& x' (arrays stay arrays: they decay to pointers),
  * shader in/out variables become thread_local globals,
  * the one float -> int conversion whose NaN case GLSL leaves undefined (error_to_color) goes through glsl_float_to_int().

No arithmetic is touched. The transformed copies go to oracle/_ref/gen/ (git-ignored, never committed), the
sources are read where they lie under /root/reference. One translation unit per configuration because the
reference bakes its settings into the shader as -D defines (src/main.c:752-792).
"""
import json
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SHADERS = "/root/reference/src/shaders"
OUT = os.path.join(HERE, "_ref")
GEN = os.path.join(OUT, "gen")
CXX = "/usr/bin/g++"

STRATEGIES = ["DIFFUSE_ONLY", "DIFFUSE_GGX_MIS", "DIFFUSE_SPECULAR_SEPARATELY", "DIFFUSE_SPECULAR_MIS", "DIFFUSE_SPECULAR_RANDOM"]
HEURISTICS = ["BALANCE", "POWER", "WEIGHTED", "OPTIMAL_CLAMPED", "OPTIMAL"]
# index = sample_polygon_technique_t (src/polygonal_light.h:30-66); 12 = the biased variant of 11 (c["biased"])
TECHNIQUES = ["BASELINE", "AREA_TURK", "RECTANGLE_SOLID_ANGLE_URENA", "SOLID_ANGLE_ARVO", "SOLID_ANGLE", "CLIPPED_SOLID_ANGLE", "BILINEAR_COSINE_WARP_HART",
	"BILINEAR_COSINE_WARP_CLIPPING_HART", "BIQUADRATIC_COSINE_WARP_HART", "BIQUADRATIC_COSINE_WARP_CLIPPING_HART", "PROJECTED_SOLID_ANGLE_ARVO", "PROJECTED_SOLID_ANGLE"]
CLIPPING_TECHNIQUES = (5, 7, 9, 10, 11)   # get_max_polygon_vertex_count (src/main.c:194-216): clipping may add one vertex
# error_display_t (src/main.h:95-112) -> (ERROR_DISPLAY_DIFFUSE, ERROR_DISPLAY_SPECULAR, ERROR_INDEX), src/main.c:735-750
ERROR_DISPLAYS = {0: (0, 0, 0), 1: (1, 0, 0), 2: (1, 0, 1), 3: (1, 0, 2), 4: (0, 1, 0), 5: (0, 1, 1), 6: (0, 1, 2)}


def config_name(c):
	vertices = "%d" % c["max_vertices"] if c.get("min_vertices", c["max_vertices"]) == c["max_vertices"] else "%dm%d" % (c["max_vertices"], c["min_vertices"])
	name = "s%d_h%d_b%d_L%d_V%s_S%d_t%d_l%d_M%d" % (c["strategy"], c["heuristic"], c["biased"], c["lights"], vertices, c["samples"], c["trace"], c["show_lights"], c["materials"])
	if c.get("technique", 11) != 11:                 # related-work sampling technique: q<sample_polygon_technique_t>
		name += "_q%d" % c["technique"]
	if c.get("error_display", 0):
		name += "_e%d" % c["error_display"]
	if c.get("textured", 0):                          # same -D defines, material textures that need filtering (data set mini_textured)
		name += "_x1"
	if c.get("light_textures", 0):                    # same -D defines, lights with area / portal / IES textures (data set mini_lit)
		name += "_y1"
	if c.get("srgb", 0) or c.get("frame_bits", 0):   # output stage: o<srgb><frame_bits>
		name += "_o%d%d" % (c.get("srgb", 0), c.get("frame_bits", 0))
	return name


def defines(c):
	"""The -D list of create_shading_pass (src/main.c:752-792) for one configuration."""
	d = {
		"MATERIAL_COUNT": c["materials"], "POLYGONAL_LIGHT_COUNT": c["lights"], "POLYGONAL_LIGHT_ARRAY_SIZE": max(c["lights"], 1),
		"POLYGONAL_LIGHT_COUNT_CLAMPED": min(c["lights"], 33), "LIGHT_TEXTURE_COUNT": 4,
		"MIN_POLYGON_VERTEX_COUNT_BEFORE_CLIPPING": c.get("min_vertices", c["max_vertices"]), "MAX_POLYGONAL_LIGHT_VERTEX_COUNT": c["max_vertices"],
		"MAX_POLYGON_VERTEX_COUNT": c["max_vertices"] + (1 if c.get("technique", 11) in CLIPPING_TECHNIQUES else 0), "SAMPLE_COUNT": c["samples"], "SAMPLE_COUNT_CLAMPED": min(c["samples"], 33),
		"TRACE_SHADOW_RAYS": c["trace"], "SHOW_POLYGONAL_LIGHTS": c["show_lights"],
		"ERROR_DISPLAY_DIFFUSE": ERROR_DISPLAYS[c.get("error_display", 0)][0], "ERROR_DISPLAY_SPECULAR": ERROR_DISPLAYS[c.get("error_display", 0)][1],
		"ERROR_INDEX": ERROR_DISPLAYS[c.get("error_display", 0)][2], "OUTPUT_LINEAR_RGB": 0 if c.get("srgb", 0) else 1,
	}
	for i, s in enumerate(STRATEGIES):
		d["SAMPLING_STRATEGIES_" + s] = int(c["strategy"] == i)
	for i, h in enumerate(HEURISTICS):
		d["MIS_HEURISTIC_" + h] = int(c["heuristic"] == i)
	for t in TECHNIQUES:
		d["SAMPLE_POLYGON_" + t] = int(t == TECHNIQUES[c.get("technique", 11)])
	flags = ["-D%s=%s" % kv for kv in d.items()]
	flags.append("-DUSE_BIASED_PROJECTED_SOLID_ANGLE_SAMPLING" if c["biased"] else "-DDONT_USE_BIASED_PROJECTED_SOLID_ANGLE_SAMPLING")
	return flags


def transform(text):
	text = re.sub(r"^\s*#(version|extension)[^\n]*\n", "\n", text, flags=re.M)
	# open up the uniform block: drop its header line and its closing '};'
	m = re.search(r"layout\s*\([^)]*\)\s*uniform\s+\w+\s*\{", text)
	if m:
		depth = 0; i = m.end() - 1
		while True:
			if text[i] == "{": depth += 1
			elif text[i] == "}":
				depth -= 1
				if depth == 0: break
			i += 1
		close_end = text.index(";", i) + 1
		text = text[:m.start()] + text[m.end():i] + text[close_end:]
	# shader stage inputs/outputs -> thread_local globals; resource bindings -> plain globals
	text = re.sub(r"layout\s*\([^)]*\)\s*in\s+", "thread_local ", text)
	text = re.sub(r"layout\s*\([^)]*\)\s*out\s+", "thread_local ", text)
	text = re.sub(r"layout\s*\([^)]*\)\s*uniform\s+", "", text)
	# parameter qualifiers
	def param(mm):
		return "%s %s[" % (mm.group(2), mm.group(3)) if mm.group(4) else "%s& %s" % (mm.group(2), mm.group(3))
	text = re.sub(r"\b(inout|out)\s+(\w+)\s+(\w+)(\s*\[)?", param, text)
	# error_to_color() (shading_pass.frag.glsl:114) indexes its colour table with int(color_index); for a NaN error GLSL leaves the
	# result undefined and a C++ cast reads out of bounds. glsl_float_to_int() maps everything outside the table to its first entry.
	text = text.replace("tab20b_colors[int(color_index)]", "tab20b_colors[glsl_float_to_int(color_index)]")
	return text


def generate_sources():
	os.makedirs(GEN, exist_ok=True)
	for name in sorted(os.listdir(REF_SHADERS)):
		if name.endswith(".glsl"):
			with open(os.path.join(REF_SHADERS, name)) as f:
				text = f.read()
			with open(os.path.join(GEN, name), "w") as f:
				f.write(transform(text))


def default_configs():
	base = dict(strategy=3, heuristic=3, biased=0, lights=3, max_vertices=4, samples=3, trace=1, show_lights=1, materials=8)
	configs = []
	for strategy, heuristic in [(0, 0), (1, 0), (1, 1), (2, 0), (3, 0), (3, 1), (3, 2), (3, 3), (3, 4), (4, 0)]:
		configs.append(dict(base, strategy=strategy, heuristic=heuristic))
	configs.append(dict(base, biased=1))
	configs.append(dict(base, samples=40, lights=2))                       # loop instead of unrolled code (SAMPLE_COUNT_CLAMPED = 33)
	configs.append(dict(base, lights=1, samples=1, trace=0, materials=3, strategy=0, heuristic=3))   # BASELINE config 1 (Cornell)
	configs.append(dict(base, lights=1, samples=2, trace=1, materials=3))  # Cornell with MIS and rays
	configs.append(dict(base, max_vertices=3))                             # triangle lights (data set mini_tri)
	configs.append(dict(base, max_vertices=3, strategy=1, heuristic=0))
	configs.append(dict(base, max_vertices=4, min_vertices=3))             # triangle, quad, triangle (data set mini_mixed)
	configs.append(dict(base, max_vertices=4, min_vertices=3, strategy=1, heuristic=1))
	configs.append(dict(base, max_vertices=7, min_vertices=5))             # pentagon, heptagon, hexagon (data set mini_poly)
	configs.append(dict(base, max_vertices=7, min_vertices=5, strategy=0, heuristic=0))
	configs.append(dict(base, max_vertices=7, min_vertices=5, strategy=1, heuristic=0))
	configs.append(dict(base, max_vertices=5))                             # pentagons (mini_v5)
	configs.append(dict(base, max_vertices=6, strategy=2, heuristic=0))    # hexagons (mini_v6)
	configs.append(dict(base, max_vertices=7, strategy=4, heuristic=0))    # heptagons (mini_v7)
	configs.append(dict(base, lights=32, samples=2))                       # many lights (data set mini_room): the shape of BASELINE config 4
	configs.append(dict(base, lights=16, samples=1, strategy=1, heuristic=0))
	configs.append(dict(base, lights=1, samples=256))                      # config 4's sample count: 4 periods of the noise sequence
	configs.append(dict(base, trace=0))                                    # TRACE_SHADOW_RAYS=0 with the other strategies
	configs.append(dict(base, trace=0, strategy=1, heuristic=1))
	configs.append(dict(base, trace=0, heuristic=4))
	configs.append(dict(base, lights=8, samples=64, materials=64))           # BASELINE config 3 as bench.py runs it (8 quads, 64 spp, clamped optimal MIS, 64 materials): the CPU reference arm
	# related-work sampling techniques (SURVEY 8 f4; shading_pass.frag.glsl:332-481), sample_polygon_technique_t 0..10: diffuse only, then GGX MIS
	# for the techniques the reference's interface allows it with (user_interface.cpp:130-140)
	for technique in range(0, 11):
		configs.append(dict(base, strategy=0, heuristic=0, technique=technique))
	for technique, heuristic in [(2, 0), (3, 1), (4, 0), (5, 1), (10, 0)]:
		configs.append(dict(base, strategy=1, heuristic=heuristic, technique=technique))
	for technique in (1, 3, 4, 6, 8):                                        # techniques without clipping: MAX_POLYGON_VERTEX_COUNT = light vertices
		configs.append(dict(base, strategy=0, heuristic=0, technique=technique, max_vertices=3))
	for technique in (4, 5, 7, 9, 10):
		configs.append(dict(base, strategy=0, heuristic=0, technique=technique, max_vertices=7, min_vertices=5))
	configs.append(dict(base, strategy=0, heuristic=0, technique=1, max_vertices=6))
	configs.append(dict(base, strategy=0, heuristic=0, technique=10, max_vertices=5, trace=0))
	configs.append(dict(base, strategy=0, heuristic=0, technique=9, lights=16, samples=1))
	configs.append(dict(base, strategy=0, heuristic=0, technique=2, lights=1, samples=2, materials=3))   # Cornell box, Urena's rectangle sampling
	# error display of the sampling procedure (error_display_t 1..6, src/main.h:92-112; shading_pass.frag.glsl:462-481, 549-563)
	for error_display, extra in [(1, dict(strategy=0, heuristic=0)), (2, dict()), (3, dict(strategy=1, heuristic=0)), (4, dict()), (5, dict(strategy=2, heuristic=0)), (6, dict(strategy=4, heuristic=0)),
			(1, dict(biased=1)), (4, dict(biased=1)), (3, dict(max_vertices=7, min_vertices=5)), (6, dict(max_vertices=3)), (1, dict(strategy=0, heuristic=0, technique=10)), (2, dict(strategy=0, heuristic=0, technique=10, max_vertices=5))]:
		configs.append(dict(base, error_display=error_display, **extra))
	configs.append(dict(base, textured=1))                                   # get_shading_data with filtered material textures (SURVEY 8 f1)
	configs.append(dict(base, textured=1, strategy=1, heuristic=1, trace=0))
	# lights with textures (get_polygon_radiance, shading_pass.frag.glsl:151-185): an area texture, a light probe behind a portal, an IES profile
	configs.append(dict(base, light_textures=1))
	configs.append(dict(base, light_textures=1, strategy=1, heuristic=0))
	configs.append(dict(base, light_textures=1, strategy=0, heuristic=0))
	configs.append(dict(base, light_textures=1, trace=0))
	configs.append(dict(base, light_textures=1, trace=0, heuristic=4))
	configs.append(dict(base, light_textures=1, strategy=0, heuristic=0, technique=4))
	for srgb, frame_bits in [(1, 0), (0, 1), (0, 2), (1, 1), (1, 2)]:         # output stage: sRGB conversion, half-bit split for HDR screenshots (frame_bits is a uniform)
		configs.append(dict(base, srgb=srgb, frame_bits=frame_bits))
	return configs


def build(configs=None, verbose=False, set_name=""):
	if not os.path.isdir(REF_SHADERS):
		print("build_ref: /root/reference is not present; keeping the prebuilt oracle/_ref as it is")
		return None
	configs = configs or default_configs()
	generate_sources()
	compat = os.path.join(HERE, "glsl_compat")
	common = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-mfma", "-mavx2", "-fopenmp", "-w", "-I", GEN, "-I", compat]
	objects = []
	procs = []
	obj = os.path.join(OUT, "ref_common.o")
	procs.append(("common", subprocess.Popen([CXX] + common + ["-c", os.path.join(compat, "ref_common.cpp"), "-o", obj], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
	objects.append(obj)
	names = []
	for c in configs:
		name = config_name(c)
		if c.get("textured", 0) or c.get("light_textures", 0):   # textures are inputs, not defines: the entry point of the untextured configuration serves
			names.append(dict(c, name=name, entry="ref_shade_" + config_name(dict(c, textured=0, light_textures=0))))
			continue
		names.append(dict(c, name=name, entry="ref_shade_" + name))
		obj = os.path.join(OUT, name + ".o")
		objects.append(obj)
		cmd = [CXX] + common + defines(c) + ["-DREF_NS=cfg_" + name, "-DREF_ENTRY=ref_shade_" + name, "-c", os.path.join(compat, "ref_driver.cpp"), "-o", obj]
		procs.append((name, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
	failed = False
	for name, p in procs:
		out, _ = p.communicate()
		if p.returncode != 0:
			failed = True
			sys.stderr.write("---- %s\n%s\n" % (name, out[-6000:]))
	if failed:
		raise SystemExit("build_ref: compiling the reference shader as C++ failed")
	compiled = {n["entry"] for n in names if not (n.get("textured", 0) or n.get("light_textures", 0))}
	missing = [n["name"] for n in names if n["entry"] not in compiled]
	if missing:
		raise SystemExit("build_ref: textured configurations without an untextured twin: %s" % missing)
	lib = os.path.join(OUT, "libref_shader%s.so" % (("_" + set_name) if set_name else ""))
	subprocess.check_call([CXX, "-shared", "-fopenmp", "-o", lib] + objects)
	with open(os.path.join(OUT, "configs%s.json" % (("_" + set_name) if set_name else "")), "w") as f:
		json.dump(names, f, indent=1)
	for o in objects:
		os.remove(o)
	print("build_ref: %d configurations -> %s" % (len(configs), lib))
	if not set_name:
		build_host()
	return lib


def random_configs(count, seed):
	"""Legal combinations of the settings (src/user_interface.cpp:90-180) beyond default_configs(), for tools/fuzz_parity.py --ref-set: the oracle takes all of
	them as run-time parameters, the reference needs one compiled shader each."""
	import random
	rng = random.Random(seed)
	out, seen = [], {config_name(c) for c in default_configs()}
	while len(out) < count:
		vmax, vmin = rng.choice([(3, 3), (4, 4), (4, 3), (5, 5), (6, 6), (7, 7), (7, 5)])
		c = dict(strategy=rng.randrange(5), heuristic=0, biased=0, lights=3, max_vertices=vmax, min_vertices=vmin, samples=rng.randrange(1, 5), trace=rng.randrange(2), show_lights=rng.randrange(2), materials=8)
		roll = rng.random()
		if roll < 0.35:
			c["technique"] = rng.randrange(11)
			c["strategy"] = rng.randrange(2) if c["technique"] in (2, 3, 4, 5, 10) else 0
		elif roll < 0.55:
			c["biased"] = 1
		if c["strategy"] == 1: c["heuristic"] = rng.randrange(2)
		if c["strategy"] == 3: c["heuristic"] = rng.randrange(5)
		if c.get("technique", 11) in (10, 11) and rng.random() < 0.2:
			c["error_display"] = rng.randrange(1, 7)
			if c.get("technique", 11) == 10: c["strategy"] = 0; c["heuristic"] = 0; c["error_display"] = rng.randrange(1, 3)
			elif c["error_display"] >= 4 and c["strategy"] < 2: c["strategy"] = rng.randrange(2, 5); c["heuristic"] = rng.randrange(5) if c["strategy"] == 3 else 0
		elif rng.random() < 0.25:
			c["srgb"] = rng.randrange(2); c["frame_bits"] = rng.randrange(3)
		if vmin == vmax: c.pop("min_vertices")
		name = config_name(c)
		if name not in seen:
			seen.add(name); out.append(c)
			# textures are inputs, not defines: a twin of the same shader under textured lights (data set mini_lit: three quads) or with filtered material textures
			if vmax == 4 and vmin == 4 and not c.get("error_display", 0) and rng.random() < 0.3:
				out.append(dict(c, light_textures=1))
			elif vmax == 4 and vmin == 4 and rng.random() < 0.15:
				out.append(dict(c, textured=1))
	return out


def build_host():
	"""The reference's UNCHANGED loader / host-maths C files (SURVEY 8b boundary B1), compiled from where they lie
	against shim/ (a host-memory stand-in for the Vulkan allocation helpers they call) -> oracle/_ref/libref_host.so.
	tests/test_ref_host.py holds vkr_host.cpp against it byte for byte."""
	ref_src = "/root/reference/src"
	if not os.path.isdir(ref_src):
		return None
	root = os.path.dirname(HERE)
	shim = os.path.join(root, "shim")
	lib = os.path.join(OUT, "libref_host.so")
	sources = [os.path.join(ref_src, n) for n in ("scene.c", "textures.c", "ltc_table.c", "noise_table.c", "polygonal_light.c", "camera.c")]
	cmd = ["/usr/bin/gcc", "-O2", "-std=gnu11", "-fPIC", "-shared", "-w", "-ffp-contract=off", "-I", shim, "-I", ref_src,
		os.path.join(shim, "vkr_shim.c")] + sources + [os.path.join(HERE, "ref_host_probe.c"), "-lm", "-o", lib]
	subprocess.check_call(cmd)
	print("build_ref: reference loaders over the shim -> %s" % lib)
	return lib


def build_c_host():
	"""tests/c_host/route_b.c: a plain C host that loads a data set with the reference's UNCHANGED loaders (over shim/), hands their buffers to
	libvkr_b200.so and renders a frame through the C-ABI (INTEGRATION.md, Routes B and A) -> oracle/_ref/route_b, next to the other binaries built from
	the reference's sources. Needs the reference's sources and the built library."""
	ref_src = "/root/reference/src"
	root = os.path.dirname(HERE)
	package = os.path.join(root, "vulkan_renderer_b200")
	if not os.path.isdir(ref_src) or not os.path.exists(os.path.join(package, "libvkr_b200.so")):
		return None
	shim = os.path.join(root, "shim")
	os.makedirs(OUT, exist_ok=True)
	binary = os.path.join(OUT, "route_b")
	sources = [os.path.join(ref_src, n) for n in ("scene.c", "textures.c", "ltc_table.c", "noise_table.c")]
	cmd = ["/usr/bin/gcc", "-O2", "-std=gnu11", "-w", "-ffp-contract=off", "-I", shim, "-I", ref_src, "-I", os.path.join(root, "include"),
		os.path.join(root, "tests", "c_host", "route_b.c"), os.path.join(shim, "vkr_shim.c")] + sources + ["-L", package, "-l:libvkr_b200.so", "-Wl,-rpath,$ORIGIN/../../vulkan_renderer_b200", "-lm", "-o", binary]
	subprocess.check_call(cmd)
	print("build_ref: C host over the reference's loaders and the C-ABI -> %s" % binary)
	return binary


if __name__ == "__main__":
	if "--random" in sys.argv:   # python oracle/build_ref.py --random <count> <seed> <set name>
		i = sys.argv.index("--random")
		build(random_configs(int(sys.argv[i + 1]), int(sys.argv[i + 2])), set_name=sys.argv[i + 3])
	else:
		build(verbose="-v" in sys.argv)
		build_c_host()
