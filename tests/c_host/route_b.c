/* tests/c_host/route_b.c -- TEST INFRASTRUCTURE: a C host that follows INTEGRATION.md literally (boundary B1 + B2, SURVEY 8b).
 *
 * Route B: the reference's UNCHANGED loaders -- load_scene (src/scene.c), load_ltc_table (src/ltc_table.c), load_noise_table (src/noise_table.c),
 * compiled from where they lie under /root/reference against shim/ (host memory instead of Vulkan allocations) -- read the data set; their staging
 * buffers, images and the triangle soup of the acceleration structure build are handed to libvkr_b200.so (vkr_scene_from_buffers,
 * vkr_ltc_table_from_images, vkr_noise_table_from_image). Route A from there on: the frame-side C-ABI renders one frame (visibility pass, G-buffer
 * pass, shading pass) and the program writes it as raw float32 RGBA. No Python, no ctypes: this is what a maintainer of the reference would link.
 * Built by oracle/build_ref.py (needs the reference's sources) into oracle/_ref/route_b; tests/test_gpu_zzzz_c_host.py runs it on the GPU box and compares the
 * frame with the oracle.
 *
 *   route_b <scene.vks> <texture dir> <quicksave> <ltc dir> <width> <height> <sample count> <out.f32>
 */
#include "scene.h"
#include "ltc_table.h"
#include "noise_table.h"
#include "vkr_b200.h"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

int main(int argc, char** argv) {
	if (argc != 9) { printf("usage: route_b <scene.vks> <texture dir> <quicksave> <ltc dir> <width> <height> <sample count> <out.f32>\n"); return 2; }
	const uint32_t width = (uint32_t) atoi(argv[5]), height = (uint32_t) atoi(argv[6]), sample_count = (uint32_t) atoi(argv[7]);
	/* ---- B1: the reference's loaders over the shim */
	device_t ref_device; memset(&ref_device, 0, sizeof(ref_device));
	ref_device.device = vkr_shim_device(); ref_device.instance = vkr_shim_instance();
	ref_device.ray_tracing_supported = VK_TRUE;
	ref_device.acceleration_structure_properties.minAccelerationStructureScratchOffsetAlignment = 128;
	ref_device.physical_device_properties.limits.nonCoherentAtomSize = 64;
	scene_t ref_scene; ltc_table_t ref_ltc; noise_table_t ref_noise;
	if (load_scene(&ref_scene, &ref_device, argv[1], argv[2], VK_TRUE)) return 1;
	if (load_ltc_table(&ref_ltc, &ref_device, argv[4], 51)) return 1;
	VkExtent3D noise_resolution = { 256, 256, 64 };
	if (load_noise_table(&ref_noise, &ref_device, noise_resolution, noise_type_white)) return 1;
	/* ---- hand-over */
	vkr_device_t device;
	if (vkr_create_device(&device, 0, NULL)) return 1;
	const uint64_t material_count = ref_scene.materials.material_count;
	vkr_texture_t* textures = (vkr_texture_t*) calloc(3 * material_count, sizeof(vkr_texture_t));
	for (uint64_t i = 0; i != 3 * material_count; ++i) {
		const image_t* image = &ref_scene.materials.textures.images[i];
		const uint32_t mip_count = image->image_info.mipLevels;
		const void* levels[32]; uint64_t sizes[32];
		for (uint32_t k = 0; k != mip_count && k != 32; ++k) { VkDeviceSize size = 0; levels[k] = vkr_shim_image_data(image->image, k, 0, &size); sizes[k] = size; }
		if (vkr_texture_from_levels(&textures[i], image->image_info.extent.width, image->image_info.extent.height, mip_count, (uint32_t) image->image_info.format, levels, sizes)) return 1;
	}
	vkr_scene_buffers_t buffers; memset(&buffers, 0, sizeof(buffers));
	buffers.triangle_count = ref_scene.mesh.triangle_count; buffers.material_count = material_count;
	memcpy(buffers.dequantization_factor, ref_scene.mesh.dequantization_factor, 12); memcpy(buffers.dequantization_summand, ref_scene.mesh.dequantization_summand, 12);
	buffers.material_names = (const char* const*) ref_scene.materials.material_names;
	buffers.quantized_positions = (const uint32_t*) vkr_shim_buffer_data(ref_scene.mesh.positions.buffer, NULL);
	buffers.normals_and_tex_coords = (const uint16_t*) vkr_shim_buffer_data(ref_scene.mesh.normals_and_tex_coords.buffer, NULL);
	buffers.material_indices = (const uint8_t*) vkr_shim_buffer_data(ref_scene.mesh.material_indices.buffer, NULL);
	uint64_t soup_triangles = 0;
	buffers.acceleration_structure_vertices = vkr_shim_acceleration_structure_vertices(ref_scene.acceleration_structure.bottom_level, &soup_triangles);
	if (soup_triangles != buffers.triangle_count) { printf("The acceleration structure build saw %llu triangles, the mesh has %llu.\n", (unsigned long long) soup_triangles, (unsigned long long) buffers.triangle_count); return 1; }
	buffers.material_textures = textures;
	vkr_scene_t scene; vkr_ltc_table_t ltc; vkr_noise_table_t noise;
	if (vkr_scene_from_buffers(&scene, &device, &buffers, 1)) return 1;
	for (uint64_t i = 0; i != 3 * material_count; ++i) vkr_destroy_texture(&textures[i]);
	free(textures);
	vkr_ltc_constants_t ltc_constants; memcpy(&ltc_constants, &ref_ltc.constants, sizeof(ltc_constants));
	if (vkr_ltc_table_from_images(&ltc, &device, ref_ltc.roughness_count, ref_ltc.inclination_count, ref_ltc.fresnel_count,
		(const uint16_t*) vkr_shim_image_data(ref_ltc.texture_arrays.images[0].image, 0, 0, NULL), (const uint16_t*) vkr_shim_image_data(ref_ltc.texture_arrays.images[1].image, 0, 0, NULL), &ltc_constants)) return 1;
	if (vkr_noise_table_from_image(&noise, &device, 256, 256, 64, (const uint16_t*) vkr_shim_image_data(ref_noise.noise_array.images[0].image, 0, 0, NULL), ref_noise.random_seed)) return 1;
	destroy_noise_table(&ref_noise, &ref_device); destroy_ltc_table(&ref_ltc, &ref_device); destroy_scene(&ref_scene, &ref_device);
	/* ---- B2: one frame through the frame-side C-ABI (what render_frame + write_constants do, src/main.c:2114-2270) */
	vkr_scene_specification_t spec; vkr_render_settings_t settings;
	memset(&spec, 0, sizeof(spec));
	if (vkr_quick_load(&spec, argv[3])) return 1;
	if (vkr_create_and_assign_light_textures(NULL, NULL, &spec)) return 1;
	vkr_specify_default_render_settings(&settings);
	settings.animate_noise = 0; settings.exposure_factor = 1.0f; settings.sample_count = sample_count;
	const size_t constants_size = vkr_get_constants_size(&spec);
	void* constants = malloc(constants_size);
	vkr_write_constants(constants, &spec, &settings, &scene, &ltc, &noise, width, height);
	vkr_render_targets_t targets;
	if (vkr_create_render_targets(&targets, &device, width, height)) return 1;
	if (vkr_run_visibility_pass(&device, &scene, constants, width, height, targets.d_visibility)) return 1;
	if (vkr_run_gbuffer_pass(&device, &scene, constants, width, height, targets.d_visibility, targets.d_gbuffer)) return 1;
	uint32_t max_vertices = 3, min_vertices = 7;
	for (uint32_t i = 0; i != spec.polygonal_light_count; ++i) {
		if (max_vertices < spec.polygonal_lights[i].vertex_count) max_vertices = spec.polygonal_lights[i].vertex_count;
		if (min_vertices > spec.polygonal_lights[i].vertex_count) min_vertices = spec.polygonal_lights[i].vertex_count;
	}
	vkr_shading_pass_desc_t desc; memset(&desc, 0, sizeof(desc));
	desc.width = width; desc.height = height;
	desc.polygonal_light_count = spec.polygonal_light_count; desc.min_polygonal_light_vertex_count = min_vertices; desc.max_polygonal_light_vertex_count = max_vertices;
	desc.sample_count = settings.sample_count; desc.sampling_strategies = settings.sampling_strategies; desc.mis_heuristic = settings.mis_heuristic;
	desc.polygon_sampling_technique = settings.polygon_sampling_technique; desc.trace_shadow_rays = settings.trace_shadow_rays; desc.show_polygonal_lights = settings.show_polygonal_lights;
	desc.scene = &scene; desc.ltc_table = &ltc; desc.noise_table = &noise;
	vkr_shading_pass_t pass;
	if (vkr_create_shading_pass(&pass, &device, &desc)) return 1;
	if (vkr_shading_pass_run(&pass, &device, constants, constants_size, targets.d_gbuffer, targets.d_frame)) return 1;
	if (vkr_shading_pass_wait(&pass, &device)) return 1;
	float* frame = (float*) malloc(sizeof(float) * 4 * (size_t) width * height);
	if (vkr_download_frame(&targets, &device, frame)) return 1;
	FILE* file = fopen(argv[8], "wb");
	if (!file || fwrite(frame, sizeof(float) * 4, (size_t) width * height, file) != (size_t) width * height) { printf("Failed to write %s.\n", argv[8]); return 1; }
	fclose(file);
	printf("route_b: %ux%u frame of %llu triangles, %u lights, %u spp written to %s\n", width, height, (unsigned long long) scene.triangle_count, spec.polygonal_light_count, sample_count, argv[8]);
	free(frame); free(constants);
	vkr_destroy_shading_pass(&pass, &device); vkr_destroy_render_targets(&targets, &device);
	vkr_destroy_scene_specification(&spec);
	vkr_destroy_noise_table(&noise, &device); vkr_destroy_ltc_table(&ltc, &device); vkr_destroy_scene(&scene, &device); vkr_destroy_device(&device);
	return 0;
}
