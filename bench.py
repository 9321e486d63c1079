#!/usr/bin/env python3
"""Benchmark of the shading pass hot path (BASELINE.json: Msamples/s at 1920x1080x64spp).

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C3|C2|C4|C1|mini] [--dump-outputs DIR]

A "step" is one pass of the shading megakernel over one frame of a synthetic scene. The default workload is BASELINE config 3, the
one the metric is quoted on: the Bistro-like city (2.8 M triangles) at 1920x1080, 8 quad lights, 64 spp, diffuse+specular MIS with the
clamped optimal heuristic, shadow rays on. C2 (1 light, 4 spp, diffuse only) and C4 (the attic-like room at 3840x2160, 32 lights,
256 spp: the configuration north_star shards over 8 GPUs) are selectable; results of those runs live under profiles/.

  value  whole-job Msamples/s (pixels*spp / time), inputs resident in HBM, CUDA events on the launching stream, L2 flushed between
         steps, max over ranks
  e2e    same metric through the C-ABI call with HOST buffers (H2D of the G-buffer and D2H of the frame inside the timed region)
  N > 1  every GPU shades the screen tiles (tx + ty / 8) % N == rank of the frame (strong scaling); the shading kernel stores finished pixels into
         the frames of all GPUs over NVLink (vkr_frame_exchange_t), two one-block kernels form the barrier: all of it inside the timed
         region. After the timed loop every rank's frame is hashed and compared with a single-GPU render of the same frame.

--impl reference times the reference's shader sources compiled for the CPU (oracle/_ref, all host threads) on a bounded sample of
the same frame; the reference's Vulkan path itself cannot run on this box (no ICD, no glslangValidator).
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# sampling_strategies_t / mis_heuristic_t (src/main.h:45-92)
DIFFUSE_ONLY, DIFFUSE_SPECULAR_MIS, OPTIMAL_CLAMPED = 0, 3, 3
WORKLOADS = {
	"C3": dict(dataset="city", scene="Bistro-like synthetic city", width=1920, height=1080, lights=8, spp=64, strategy=DIFFUSE_SPECULAR_MIS),
	"C2": dict(dataset="city", scene="Bistro-like synthetic city", width=1920, height=1080, lights=1, spp=4, strategy=DIFFUSE_ONLY),
	"C4": dict(dataset="room", scene="attic-like synthetic room", width=3840, height=2160, lights=32, spp=256, strategy=DIFFUSE_SPECULAR_MIS),
	"C1": dict(dataset="cornell", scene="Cornell box", width=256, height=256, lights=1, spp=1, strategy=DIFFUSE_ONLY, rays=0),
	"mini": dict(dataset="mini_city", scene="small synthetic city", width=320, height=192, lights=3, spp=8, strategy=DIFFUSE_SPECULAR_MIS),
}


def log(*a):
	print(*a, file=sys.stderr, flush=True)


def workload_text(name, w, tri_count):
	strategy = "diffuse+specular MIS (clamped optimal)" if w["strategy"] == DIFFUSE_SPECULAR_MIS else "diffuse-only projected solid angle sampling"
	return "%s: %s %dx%d, %d quad light%s, %d spp, %s, shadow rays %s, %d triangles" % (name, w["scene"], w["width"], w["height"], w["lights"],
		"" if w["lights"] == 1 else "s", w["spp"], strategy, "on" if w.get("rays", 1) else "off", tri_count)


def metric_text(w):
	return "Msamples/s (pixels x spp) at %dx%dx%dspp; achieved HBM GB/s vs roofline" % (w["width"], w["height"], w["spp"])


class ClockSampler:
	"""Samples nvidia-smi clocks and throttle reasons while the timed region runs."""
	QUERY = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

	def __init__(self, gpu_index):
		self.gpu_index = gpu_index; self.samples = []; self.proc = None; self.thread = None

	def start(self):
		try:
			self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
		except OSError:
			self.proc = None
			return
		def reader():
			for line in self.proc.stdout:
				parts = [p.strip() for p in line.split(",")]
				if len(parts) >= 9:
					self.samples.append(parts)
		self.thread = threading.Thread(target=reader, daemon=True); self.thread.start()

	def stop(self):
		if self.proc is None:
			return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
		time.sleep(0.15)
		self.proc.terminate()
		try:
			self.proc.wait(timeout=2)
		except subprocess.TimeoutExpired:
			self.proc.kill()
		clocks, max_clocks, reasons = [], [], set()
		for p in self.samples:
			try:
				clocks.append(float(p[1])); max_clocks.append(float(p[2]))
			except ValueError:
				continue
			for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
				if val.lower().startswith("active"):
					reasons.add(name)
		return {"sm_mhz": float(np.median(clocks)) if clocks else None, "sm_max_mhz": max(max_clocks) if max_clocks else None,
			"reasons": sorted(reasons), "samples": len(clocks), "power_w_max": max([float(p[3]) for p in self.samples if p[3].replace(".", "", 1).isdigit()] or [0.0])}


def algorithmic_bytes(width, height, tri_count, light_count, noise_fetches_per_pixel, ltc_res, ltc_layers_touched, rays):
	"""SURVEY 8d: compulsory bytes per frame, every byte counted once (BVH and triangles only when shadow rays are traced)."""
	return (width * height * (64 + 16)
		+ ((64 * (tri_count - 1) + 48 * tri_count) if rays else 0)
		+ 256 + 320 * light_count
		+ min(33554432, width * height * noise_fetches_per_pixel * 8)
		+ ltc_res * ltc_res * 12 * ltc_layers_touched)


def measured_peak():
	path = os.path.join(ROOT, "MEASURED_PEAKS.json")
	if os.path.exists(path):
		with open(path) as f:
			return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
	return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_capture(workload):
	"""What only a profiler can count (DRAM bytes, issued warp instructions, pipe utilisation): the committed `ncu --set full` capture of this
	workload, profiles/kernel_counters.json (written by tools/summarize_ncu.py together with the git hash of the kernel that was captured)."""
	path = os.path.join(ROOT, "profiles", "kernel_counters.json")
	if os.path.exists(path):
		with open(path) as f:
			return json.load(f).get(workload) or {}
	return {}


def build_frame(workload):
	from vulkan_renderer_b200 import synth
	w = WORKLOADS[workload]
	data_root = os.environ.get("VKR_BENCH_DATA", os.path.join("/tmp", "vkr_b200_data"))
	t0 = time.time()
	info = synth.build_dataset(os.path.join(data_root, w["dataset"]), w["dataset"])
	log("[bench] dataset %s: %d triangles (%.1f s)" % (w["dataset"], info["triangle_count"], time.time() - t0))
	return info, w


def run_b200(args):
	import torch
	import torch.distributed as dist
	from vulkan_renderer_b200 import Frame, api
	from vulkan_renderer_b200.stripes import ShareGather, connect_exchange
	world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
	if world > 1:
		os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
		dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
		# torchrun exports OMP_NUM_THREADS=1; every rank builds the scene's BVH on the host (OpenMP tasks), so give each its share of the cores
		os.environ["OMP_NUM_THREADS"] = str(max(1, host_threads() // world))
		try:
			C.CDLL("libgomp.so.1").omp_set_num_threads(max(1, host_threads() // world))
		except OSError:
			pass
	torch.cuda.set_device(local_rank)
	dev = torch.device("cuda", local_rank)
	# A dedicated stream shared by torch and the library: the default stream's handle is 0, which the C-ABI
	# reads as "create your own stream"; CUDA events must be recorded on the stream the kernels run on.
	stream = torch.cuda.Stream(dev)
	torch.cuda.set_stream(stream)
	assert stream.cuda_stream != 0
	if world > 1 and rank != 0:
		dist.barrier()  # rank 0 writes the dataset first
	info, w = build_frame(args.workload)
	width, height, lights, spp, rays = w["width"], w["height"], w["lights"], w["spp"], w.get("rays", 1)
	if world > 1 and rank == 0:
		dist.barrier()
	frame = Frame(info["vks"], info["textures"], info["save"], info["ltc"], cuda_device=local_rank, stream=stream.cuda_stream)
	frame.configure(sample_count=spp, strategy=w["strategy"], heuristic=OPTIMAL_CLAMPED, technique=api.TECHNIQUE_PSA, trace_shadow_rays=rays, show_lights=1, light_count=lights)
	lib = frame.lib
	log("[bench] rank %d: BVH %d node pairs, depth %d, build %.2f s (%s)" % (rank, frame.scene.shadow_node_count, frame.scene.shadow_max_depth, frame.scene.build_seconds, os.environ.get("VKR_BVH_BUILDER", "sah on the host")))
	constants = frame.constants(width, height)
	# --- inputs: the G-buffer is produced on the device once, outside the timed region
	vis = torch.empty((height, width), dtype=torch.int32, device=dev)
	gb = torch.empty((4, height, width, 4), dtype=torch.float32, device=dev)
	out = torch.zeros((height, width, 4), dtype=torch.float32, device=dev)
	assert lib.vkr_run_visibility_pass(C.byref(frame.device), C.byref(frame.scene), constants, width, height, vis.data_ptr()) == 0
	assert lib.vkr_run_gbuffer_pass(C.byref(frame.device), C.byref(frame.scene), constants, width, height, vis.data_ptr(), gb.data_ptr()) == 0
	torch.cuda.synchronize()
	valid = gb[1, :, :, 3] != 0
	f0_lum = (gb[3, :, :, :3] * torch.tensor([0.2126, 0.7152, 0.0722], device=dev)).sum(-1)
	ltc_layers = int(torch.unique(torch.round(f0_lum[valid].clamp(0, 1) * 50.0)).numel()) if bool(valid.any()) else 0
	p = frame.create_pass(width, height, stripe_index=rank, stripe_count=world)
	flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

	# --- N > 1: the frame exchange (peer stores from the kernel epilogue); the all_gather edition only if the GPUs cannot map each other's memory
	exchange = None; gather = None; exchange_kind = "single GPU"
	if world > 1:
		exchange = api.FrameExchange()
		ok = lib.vkr_create_frame_exchange(C.byref(exchange), C.byref(frame.device), width, height, rank, world) == 0
		if ok:
			try:
				connect_exchange(lib, exchange, frame.device)
			except RuntimeError as e:
				log("[bench] rank %d: %s" % (rank, e)); ok = False
		flags = torch.tensor([1.0 if ok else 0.0], device=dev); dist.all_reduce(flags, op=dist.ReduceOp.MIN)
		if flags.item() < 0.5:
			if ok: lib.vkr_destroy_frame_exchange(C.byref(exchange), C.byref(frame.device))
			exchange = None; gather = ShareGather(height, width, rank, world, dev)
			exchange_kind = "screen tiles (tx + ty / 8) %% %d == rank, one NCCL all_gather of the HDR tiles (no peer access between the GPUs)" % world
		else:
			exchange_kind = "screen tiles (tx + ty / 8) %% %d == rank, pixels stored into every GPU's frame from the kernel epilogue over NVLink peer memory, two one-block barrier kernels" % world

	def step_device():
		if exchange is not None:
			rc = lib.vkr_shading_pass_run_exchange(C.byref(p), C.byref(frame.device), constants, len(constants), gb.data_ptr(), C.byref(exchange))
			assert rc == 0
		else:
			rc = lib.vkr_shading_pass_run(C.byref(p), C.byref(frame.device), constants, len(constants), gb.data_ptr(), out.data_ptr())
			assert rc == 0
			if gather is not None:
				gather.gather_frame(out)

	def timed(step_fn, steps, warmup):
		for _ in range(warmup):
			flush.zero_(); step_fn()
		torch.cuda.synchronize()
		if world > 1:
			dist.barrier()
		torch.cuda.synchronize()
		events = []
		for _ in range(steps):
			flush.zero_()
			e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
			e0.record(stream); step_fn(); e1.record(stream)
			events.append((e0, e1))
		torch.cuda.synchronize()
		if world > 1:
			dist.barrier()
		torch.cuda.synchronize()
		total_ms = sum(a.elapsed_time(b) for a, b in events)
		t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
		if world > 1:
			dist.all_reduce(t, op=dist.ReduceOp.MAX)
		return float(t.item())

	def frame_of_this_rank():
		if exchange is None:
			return out.cpu().numpy()
		host = np.empty((height, width, 4), dtype=np.float32)
		assert lib.vkr_frame_exchange_download(C.byref(exchange), C.byref(frame.device), host.ctypes.data) == 0
		return host

	# kernel-only timing (per launch, CUDA events inside the library on the launching stream)
	p.timing_enabled = 1
	if world > 1:
		dist.barrier()   # the first exchanged frame must not wait for a rank that is still building its BVH
	sampler = ClockSampler(local_rank)
	if rank == 0:
		sampler.start()
	for _ in range(args.warmup):
		flush.zero_(); step_device()
	launches_before = int(p.kernel_launches)
	total_ms = timed(step_device, args.steps, 0)
	launches = (int(p.kernel_launches) - launches_before) * world * (3 if exchange is not None else 1)   # every rank: the shading kernel (+ signal and wait of the exchange)
	clocks = sampler.stop() if rank == 0 else None
	if args.dump_outputs and rank == 0:
		dump_outputs(args.dump_outputs, {"frame": frame_of_this_rank()})
	# one more step to read the kernel's own duration on every rank
	flush.zero_(); step_device(); lib.vkr_shading_pass_wait(C.byref(p), C.byref(frame.device))
	if exchange is not None:
		assert lib.vkr_frame_exchange_wait(C.byref(exchange), C.byref(frame.device)) == 0
	kernel_ms = float(p.last_kernel_ms)
	kernel_ms_all = [kernel_ms]
	if world > 1:
		t = torch.zeros(world, dtype=torch.float64, device=dev); t[rank] = kernel_ms
		dist.all_reduce(t); kernel_ms_all = [float(v) for v in t.tolist()]
	ms_per_step = total_ms / args.steps
	samples = width * height * spp
	value = samples / (ms_per_step * 1e-3) / 1e6

	# --- the frame every rank holds now against a single-GPU render of the same frame (rank 0 renders it alone)
	frame_check = None
	if world > 1:
		mine = hashlib.sha256(frame_of_this_rank().tobytes()).hexdigest()
		single = None
		if rank == 0:
			whole = frame.create_pass(width, height)
			solo = torch.zeros((height, width, 4), dtype=torch.float32, device=dev)
			assert lib.vkr_shading_pass_run(C.byref(whole), C.byref(frame.device), constants, len(constants), gb.data_ptr(), solo.data_ptr()) == 0
			lib.vkr_shading_pass_wait(C.byref(whole), C.byref(frame.device))
			single = hashlib.sha256(solo.cpu().numpy().tobytes()).hexdigest()
			frame.destroy_pass(whole); del solo
		hashes = [None] * world
		dist.all_gather_object(hashes, mine)
		ref = [single]; dist.broadcast_object_list(ref, src=0); single = ref[0]
		frame_check = {"sha256": hashes[0][:16], "single_gpu_sha256": single[:16], "ranks_equal": len(set(hashes)) == 1, "equal_to_single_gpu": all(h == single for h in hashes)}
		if not frame_check["equal_to_single_gpu"]:
			log("[bench] ERROR: the exchanged frame differs from the single-GPU frame: %s vs %s" % (hashes, single))

	# --- e2e: host buffers in, host buffers out (pinned), through the library's own host entry points
	gb_host = torch.empty((4, height, width, 4), dtype=torch.float32).pin_memory(); gb_host.copy_(gb)
	out_host = torch.zeros((height, width, 4), dtype=torch.float32).pin_memory()

	def step_e2e():
		if exchange is not None:   # upload this GPU's tile columns, shade + exchange, rank 0 reads the whole frame back
			rc = lib.vkr_shading_pass_run_host_exchange(C.byref(p), C.byref(frame.device), constants, len(constants), gb_host.data_ptr(), C.byref(exchange), out_host.data_ptr() if rank == 0 else None)
			assert rc == 0
		elif world == 1:
			rc = lib.vkr_shading_pass_run_host(C.byref(p), C.byref(frame.device), constants, len(constants), gb_host.data_ptr(), out_host.data_ptr())
			assert rc == 0
		else:   # all_gather edition: the host entry point moves this GPU's tile columns both ways, the gather runs on the device frame
			gb.copy_(gb_host, non_blocking=True); step_device()
			if rank == 0:
				out_host.copy_(out, non_blocking=True)
	e2e_steps = max(1, min(args.steps, 5)); e2e_warm = max(1, min(args.warmup, 2))
	e2e_ms = timed(step_e2e, e2e_steps, e2e_warm) / e2e_steps
	e2e_value = samples / (e2e_ms * 1e-3) / 1e6
	# host -> device, summed over the GPUs: every GPU uploads its own tile columns of the G-buffer (the all_gather edition: the whole G-buffer) and the constant block
	h2d = (4 * height * width * 16) * (world if (world > 1 and exchange is None) else 1) + len(constants) * world
	d2h = height * width * 16
	if world == 1 and e2e_steps:
		assert hashlib.sha256(out_host.numpy().tobytes()).hexdigest() == hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest(), "the host path and the device path shade different frames"

	# --- what the trace warps did: the counters edition of the kernel (same frame), one untimed launch on rank 0's share
	trace = None
	if rays and rank == 0 and not args.no_counters:
		counters = (C.c_uint64 * api.TRACE_COUNTER_COUNT)()
		scratch = torch.zeros((height, width, 4), dtype=torch.float32, device=dev)
		if lib.vkr_shading_pass_run_with_counters(C.byref(p), C.byref(frame.device), constants, len(constants), gb.data_ptr(), scratch.data_ptr(), counters) == 0:
			c = dict(zip(api.TRACE_COUNTER_NAMES, [int(v) for v in counters]))
			n = max(1, c["rays"])
			trace = {"shadow_rays": c["rays"] * world, "rays_per_sample": round(c["rays"] * world / samples, 4), "grays_per_s": round(c["rays"] / (kernel_ms * 1e-3) / 1e9, 3) if kernel_ms else None,
				"node_visits_per_ray": round(c["node_visits"] / n, 3), "leaf_visits_per_ray": round(c["leaf_visits"] / n, 3), "triangle_tests_per_ray": round(c["triangle_tests"] / n, 3),
				"occluded_frac": round(c["occluded"] / n, 4), "occluder_cache_hit_frac": round(c["cache_hits"] / n, 4), "lanes_per_node_step": round(c["node_visits"] / max(1, c["warp_node_steps"]), 2),
				"traffic_model_bytes": (c["node_visits"] * 64 + c["triangle_tests"] * 48) * world, "trace_warp_idle_polls": c["idle_polls"], "shading_warp_result_polls": c["resolve_polls"],
				"from": "in-kernel counters of one extra untimed launch of the counters edition of the kernel (same frame%s)" % ("" if world == 1 else "; rank 0's share, totals scaled by the GPU count")}
		del scratch

	result = None
	if rank == 0:
		tri_count = int(frame.scene.triangle_count)
		fetches = lights * spp if w["strategy"] == DIFFUSE_SPECULAR_MIS else (lights * spp + 1) // 2   # one RGBA16 texel holds two 2D random numbers
		bytes_alg = algorithmic_bytes(width, height, tri_count, lights, fetches, int(frame.ltc.roughness_count), ltc_layers, rays)
		peak, peak_kind = measured_peak()
		capture = recorded_capture(args.workload) if world == 1 else {}
		slowest_kernel_ms = max(kernel_ms_all)
		achieved = bytes_alg / (slowest_kernel_ms * 1e-3) / 1e9 if world == 1 else bytes_alg / (ms_per_step * 1e-3) / 1e9
		sm_clock_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6 if clocks else 1965.0e6
		roofline = {"bound": "hbm", "achieved": round(achieved, 3), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 6), "traffic": capture.get("dram_bytes_per_launch"),
			"peak_source": peak_kind, "algorithmic_bytes": int(bytes_alg), "algorithmic_bytes_per_sample": round(bytes_alg / samples, 3),
			"note": "the HBM line is the contract's; what bounds this kernel is instruction issue and the L1 data pipe (SURVEY 8d: ~0.5 GB of compulsory traffic against >1 G shadow rays), see `issue` and `trace`"}
		if trace is not None:
			roofline["trace"] = trace
		if capture:
			inst = capture.get("warp_instructions")
			issue = {"peak_warp_inst_per_s": round(int(frame.device.sm_count) * 4 * sm_clock_hz / 1e9, 1), "unit": "G warp-instructions/s", "capture": capture.get("source"), "capture_git": capture.get("git"),
				"issue_active_frac": capture.get("issue_active_frac"), "lanes_per_instruction": capture.get("lanes_per_instruction"), "l1_data_pipe_frac": capture.get("l1_data_pipe_frac"),
				"pipe_fma_frac": capture.get("pipe_fma_frac"), "pipe_alu_frac": capture.get("pipe_alu_frac"), "pipe_xu_frac": capture.get("pipe_xu_frac"), "pipe_lsu_frac": capture.get("pipe_lsu_frac")}
			if inst:
				issue["warp_instructions_per_launch"] = inst
				issue["achieved_warp_inst_per_s"] = round(inst / (kernel_ms * 1e-3) / 1e9, 1)   # instructions of the captured kernel over THIS run's kernel time
				issue["frac"] = round(issue["achieved_warp_inst_per_s"] / issue["peak_warp_inst_per_s"], 4)
				issue["warp_instructions_per_sample"] = round(inst / samples, 2)
			roofline["issue"] = issue
		result = {
			"metric": metric_text(w), "value": round(value, 3), "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
			"higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
			"config": {"workload": workload_text(args.workload, w, tri_count), "parallelism": exchange_kind,
				"l2": "flushed between steps (512 MiB memset); inputs %d MB > 126 MB L2" % ((4 * width * height * 16 + 112 * tri_count) // 1000000),
				"rays_per_sample_pair": 2 if w["strategy"] == DIFFUSE_SPECULAR_MIS else 1, "sample_pairs": width * height * lights * spp,
				"tile_order": "tiles launched dearest first by the cost measured in the previous frame" if p.reorder_tiles else "row-major"},
			"e2e": {"value": round(e2e_value, 3), "unit": "Msamples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": round(e2e_ms, 4)},
			"gpu_launches": launches,
			"kernel_ms": round(kernel_ms, 4),
			"roofline": roofline,
			"clocks": clocks,
		}
		if world > 1:
			result["kernel_ms_per_rank"] = {"min": round(min(kernel_ms_all), 4), "max": round(max(kernel_ms_all), 4), "all": [round(v, 3) for v in kernel_ms_all]}
			result["exchange_ms"] = round(ms_per_step - max(kernel_ms_all), 4)   # step minus the slowest rank's kernel: barrier + waiting, ~0 when the peer stores hide in the kernel
			result["frame_check"] = frame_check
		if world == 1 and not args.no_cpu_baseline:
			result["cpu_baseline"] = cpu_baseline(args, info, w, constants, visibility=vis.cpu().numpy().view(np.uint32))
	ok = frame_check is None or frame_check["equal_to_single_gpu"]
	frame.destroy_pass(p)
	if exchange is not None:
		dist.barrier()   # nobody unmaps a frame a peer may still be writing to
		lib.vkr_destroy_frame_exchange(C.byref(exchange), C.byref(frame.device))
	frame.close()
	if world > 1:
		dist.barrier()
		dist.destroy_process_group()
	if rank == 0:
		print(json.dumps(result), flush=True)
	if not ok:
		sys.exit(3)


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(directory, arrays):
	"""Writes each array as <directory>/<name>.npy (float32) so that two builds can be compared output for output. An array over its share of
	DUMP_LIMIT_BYTES is cut to a fixed, seeded sample of its rows (the same rows for the same shape), in ascending row order."""
	os.makedirs(directory, exist_ok=True)
	share = DUMP_LIMIT_BYTES // len(arrays)
	for name, a in arrays.items():
		a = np.ascontiguousarray(a, dtype=np.float32)
		if a.nbytes > share:
			keep = share // (a.nbytes // a.shape[0])
			a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
			log("[bench] %s: %d of its rows written (fixed sample, seed 0)" % (name, keep))
		np.save(os.path.join(directory, name + ".npy"), a)


def host_threads():
	"""All host threads, whatever the launcher put into OMP_NUM_THREADS (torchrun sets it to 1)."""
	try:
		return len(os.sched_getaffinity(0))
	except AttributeError:
		return os.cpu_count() or 1


def cpu_baseline(args, info, w, constants, band_stride_tiles=None, visibility=None, repeat=1, shaded_rows=None):
	"""Times the reference's path on the host cores on a bounded sample: 8-row bands spread over the frame, full light count and spp.
	kind "reference": the reference's own shader sources compiled for the CPU (oracle/_ref/libref_shader.so, built by
	oracle/build_ref.py where /root/reference exists and shipped prebuilt; it starts from the visibility buffer like the
	shader does, i.e. it includes get_shading_data). kind "port": the C restatement (oracle/) when that library or this
	configuration is not available. Both use OpenMP over 64-pixel pieces of rows with all host threads. shaded_rows: a list that receives the rows
	of the sample as shaded by the last repetition, float32 [rows, width, 4]."""
	from tests import harness as H
	width, height, lights, spp, rays = w["width"], w["height"], w["lights"], w["spp"], w.get("rays", 1)
	oi = H.OracleInputs(info)
	band_stride = 8 * (band_stride_tiles or args.cpu_band_stride)
	rows = sum(1 for y in range(height) if y % band_stride < 8)
	ref_cfg = None
	if not args.cpu_port:
		try:
			from oracle import ref_binding as R
			ref_cfg = R.find_config(strategy=w["strategy"], heuristic=OPTIMAL_CLAMPED, biased=0, lights=lights, max_vertices=4, min_vertices=4,
				samples=spp, trace=rays, show_lights=1, technique=11, srgb=0, frame_bits=0)
			if ref_cfg is not None and ref_cfg["materials"] < len(oi.material_params):
				ref_cfg = None
		except Exception as e:   # a broken prebuilt library must not take the bench down
			log("[bench] reference shader library unusable (%s); timing the C restatement instead" % e)
			ref_cfg = None
	seconds_all = []
	for _ in range(repeat):
		t0 = time.time()
		if ref_cfg is not None:
			if visibility is None:
				visibility = oi.visibility(width, height, constants)
			t0 = time.time()
			R.set_threads(host_threads())
			frame = R.shade(ref_cfg["entry"], width, height, ref_cfg, constants, visibility, oi.vks, oi.material_params, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris, band_height=8, band_stride=band_stride)
			seconds = R.last_shade_seconds(); cores = R.thread_count(); kind = "reference"
			what = "the reference's shader sources (shading_pass.frag.glsl + includes) compiled as C++ with g++ -O2, fp32, OpenMP, ray queries on a CPU BVH"
			log("[bench] cpu reference shader: %d rows in %.2f s on %d threads (+ %.1f s BVH build)" % (rows, seconds, cores, time.time() - t0 - seconds))
		else:
			cfg = dict(width=width, height=height, light_count=lights, max_light_vertex_count=4, min_light_vertex_count=4, sample_count=spp,
				sampling_strategies=w["strategy"], mis_heuristic=OPTIMAL_CLAMPED, biased_sampling=0, trace_shadow_rays=rays, show_polygonal_lights=1,
				row_begin=0, row_end=0, band_height=8, band_stride=band_stride)
			gbuffer = oi.gbuffer(width, height, constants, visibility if visibility is not None else oi.visibility(width, height, constants))
			H.oracle.set_threads(host_threads())
			frame, n_rays = H.oracle.shade(cfg, constants, gbuffer, oi.noise, oi.ltc0, oi.ltc1, oi.shadow_tris)
			seconds = H.oracle.last_shade_seconds(); cores = H.oracle.thread_count(); kind = "port"
			what = "scalar fp32 C oracle, OpenMP"
			log("[bench] cpu oracle: %d rows in %.2f s on %d threads (+ %.1f s BVH build), %d shadow rays" % (rows, seconds, cores, time.time() - t0 - seconds, n_rays))
		seconds_all.append(seconds)
	if shaded_rows is not None:
		shaded_rows.append(frame[[y for y in range(height) if y % band_stride < 8]])
	seconds = float(np.mean(seconds_all))
	value = rows * width * spp / seconds / 1e6
	return {"value": round(value, 4), "unit": "Msamples/s", "cores": cores, "kind": kind,
		"sample": "%d of %d rows (8-row bands every %d rows), all %d lights, %d spp, %s; BVH build excluded" % (rows, height, band_stride, lights, spp, what),
		"seconds": round(seconds, 3), "seconds_all": [round(s, 3) for s in seconds_all]}


def run_reference(args):
	"""The reference's own implementation of this path is a GLSL fragment shader driven through Vulkan (no ICD, no glslangValidator
	on this box). Its CPU-runnable form is that shader compiled as C++ (oracle/_ref, kind 'reference', see cpu_baseline); without the
	prebuilt library the C restatement is timed (kind 'port'). Rank 0 only; nothing of libvkr_b200.so is loaded here: the constant block comes
	from the reference's own host code (oracle/_ref/libref_host.so: quick-load, update_polygonal_light, camera and table constants)."""
	rank = int(os.environ.get("RANK", "0"))
	if rank != 0:
		return
	os.environ["OMP_NUM_THREADS"] = str(host_threads())   # torchrun exports OMP_NUM_THREADS=1
	os.environ["VKR_B200_NO_AUTOLOAD"] = "1"              # the package's data-set generator is used here, its CUDA library is not
	from tests import harness as H
	info, w = build_frame(args.workload)
	width, height, lights, spp = w["width"], w["height"], w["lights"], w["spp"]
	constants = H.reference_constants(info, width, height, lights, spp)
	oi = H.OracleInputs(info)
	t0 = time.time()
	vis = oi.visibility(width, height, constants)
	log("[bench] reference arm: oracle visibility buffer in %.1f s" % (time.time() - t0))
	# a step = the same bounded sample of the frame every time; the sample is sized so that warm-up + steps stay within a few minutes
	values = []
	budget_s = float(os.environ.get("VKR_REFERENCE_BUDGET_S", "240"))
	# one thin probe (an 8-row band every 32 tile rows) gives seconds per row; the sample of a step is the densest set of bands that fits the budget
	probe = cpu_baseline(args, info, w, constants, band_stride_tiles=32, visibility=vis)
	probe_rows = sum(1 for y in range(height) if y % (8 * 32) < 8)
	rows_allowed = budget_s / (args.steps + args.warmup) / (probe["seconds"] / probe_rows)
	stride = args.cpu_band_stride
	while stride < 64 and sum(1 for y in range(height) if y % (8 * stride) < 8) > rows_allowed:
		stride *= 2
	shaded_rows = []
	for i in range(args.warmup + args.steps):
		r = cpu_baseline(args, info, w, constants, band_stride_tiles=stride, visibility=vis, shaded_rows=shaded_rows)
		if i >= args.warmup:
			values.append(r)
	if args.dump_outputs:
		dump_outputs(args.dump_outputs, {"frame": shaded_rows[-1]})
	seconds = sum(r["seconds"] for r in values)
	value = float(np.mean([r["value"] for r in values]))
	base = values[-1]
	try:
		load = os.getloadavg()[0]
	except OSError:
		load = None
	cpu_model = ""
	try:
		with open("/proc/cpuinfo") as f:
			cpu_model = [l.split(":", 1)[1].strip() for l in f if l.startswith("model name")][0]
	except (OSError, IndexError):
		pass
	native = sorted({l.split()[-1] for l in open("/proc/self/maps") if l.rstrip().endswith(".so") and ROOT in l})
	print(json.dumps({
		"impl": "reference", "metric": metric_text(w), "value": round(value, 4), "unit": "Msamples/s",
		"n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * seconds / max(1, len(values)), 3),
		"higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
		"config": {"workload": workload_text(args.workload, w, info["triangle_count"]),
			"note": "each step = a bounded sample of the frame on the host cores; the reference's GLSL/Vulkan path itself cannot run here (no Vulkan ICD / glslangValidator)",
			"host": {"cpu": cpu_model, "threads": base["cores"], "load_average_1min": load}, "libraries": [os.path.relpath(p, ROOT) for p in native]},
		"cpu_baseline": {"value": round(value, 4), "unit": "Msamples/s", "cores": base["cores"], "kind": base["kind"], "sample": base["sample"]},
		"e2e": {"value": round(value, 4), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
		"gpu_launches": 0,
	}), flush=True)


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument("--gpus", type=int, default=1)
	ap.add_argument("--steps", type=int, default=5)
	ap.add_argument("--warmup", type=int, default=3)
	ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
	ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
	ap.add_argument("--no-cpu-baseline", action="store_true")
	ap.add_argument("--no-counters", action="store_true", help="skip the extra untimed launch of the counters edition of the kernel")
	ap.add_argument("--cpu-port", action="store_true", help="time the C restatement (oracle/) on the CPU legs even if the compiled reference shader is available")
	ap.add_argument("--cpu-band-stride", type=int, default=4, help="the CPU sample takes one 8-row band every this many tile rows")
	ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step shaded to DIR/frame.npy (float32 [rows, width, 4]: the whole frame; "
		"with --impl reference the rows of its sample; above 64 MiB a fixed, seeded sample of those rows)")
	args = ap.parse_args()
	if args.steps < 1:
		ap.error("--steps must be at least 1")
	if args.warmup < 3:
		log("[bench] note: the timing rules ask for at least 3 warm-up steps (got %d)" % args.warmup)
	if args.impl == "reference":
		run_reference(args)
	else:
		run_b200(args)


if __name__ == "__main__":
	main()
