/* pt_b200.h — C ABI of the B200-native trace path (libpt_b200.so).
 *
 * Drop-in seam: the public interface of the reference's `class Pathtracer`
 * (reference: PathtracerCUDA/src/pathtracer/Pathtracer.h:12-69).  Each entry point below cites the reference
 * method it replaces.  Plain pointers and sizes only; no C++/torch types.  All calls are blocking, like the
 * reference (Pathtracer.cpp:199 cudaDeviceSynchronize after every launch).
 *
 * Conventions
 *   - every int-returning call returns PT_OK (0) or a negative PT_E_* code; pt_last_error() gives the text
 *     (the reference prints "CUDA error = ..." and exit()s, Pathtracer.cpp:17-28; the CLI reproduces that).
 *   - images are bottom-row-first (pixel y=0 is the bottom of the view), RGBA, exactly as the reference's
 *     accumulation buffer (kernels/trace.cu:181,196-198).
 *   - there is NO CPU fallback: without a CUDA device pt_create fails with PT_E_NO_DEVICE.
 */
#ifndef PT_B200_H
#define PT_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PT_OK 0
#define PT_E_INVALID (-1)
#define PT_E_NO_DEVICE (-2)
#define PT_E_CUDA (-3)
#define PT_E_IO (-4)
#define PT_E_PARSE (-5)
#define PT_E_LIMIT (-6)

/* reference: enum class HittableType, Hittable.h:9-12 (same numeric values) */
enum { PT_SPHERE = 0, PT_CYLINDER = 1, PT_DISK = 2, PT_CONE = 3, PT_PARABOLOID = 4, PT_QUAD = 5, PT_CUBE = 6 };
/* reference: enum class MaterialType, Material.h:9-12 */
enum { PT_LAMBERT = 0, PT_GGX = 1, PT_LAMBERT_GGX = 2 };

/* arguments of the reference Material ctor (Material.h:17): type, baseColor, emissive, roughness, metalness,
 * textureIndex (1-based texture handle, 0 = none). */
typedef struct pt_material_desc {
	uint32_t type;
	float base_color[3];
	float emissive[3];
	float roughness;
	float metalness;
	uint32_t texture;
} pt_material_desc;

/* arguments of the reference CpuHittable ctor (Hittable.h:45): type, position, rotation (Euler XYZ, RADIANS),
 * scale, material. */
typedef struct pt_object_desc {
	uint32_t type;
	float position[3];
	float rotation[3];
	float scale[3];
	pt_material_desc material;
} pt_object_desc;

/* arguments of the reference Camera ctor (Camera.h:7): position, lookat, up, fovy (RADIANS), aspectRatio. */
typedef struct pt_camera_desc {
	float position[3];
	float look_at[3];
	float up[3];
	float fovy;
	float aspect;
} pt_camera_desc;

/* counters of the last pt_render call (SURVEY.md §5 "Tracing"). */
typedef struct pt_stats {
	uint64_t samples;      /* paths started (= W*H*spp) */
	uint64_t rays;         /* closest-hit queries (camera + scattered segments, <=5 per sample) */
	uint64_t node_visits;  /* BVH node box-pair tests (only counted when option "count_work" = 1) */
	uint64_t prim_tests;   /* primitive intersection tests (idem) */
	uint64_t shades;       /* Material::sample evaluations (idem) */
	uint64_t misses;       /* environment lookups (idem) */
	float gpu_ms;          /* CUDA-event time of the trace stage, same as pt_get_timing_ms */
	uint32_t bvh_nodes;
	uint32_t bvh_depth;
	uint32_t scene_bytes;  /* device bytes of nodes + primitives + materials */
	uint32_t scene_in_smem;/* 1 if the scene was staged into shared memory by TMA bulk copy */
} pt_stats;

/* What a reference CpuHittable still holds after its ctor (Hittable.h:41-59): the world->local rows (m_invTransformRow0..2),
 * the world AABB (getAABB()), the type and the material - position / rotation / scale are gone.  pt_set_scene_xform takes
 * that, so the reference's own SceneLoader.cpp can drive this library through an unmodified `class Pathtracer` interface
 * (integration/Pathtracer_b200.cpp). */
typedef struct pt_object_xform_desc {
	uint32_t type;
	float world_to_local[12]; /* three rows of four, as Hittable.h:22-24 */
	float aabb_min[3];
	float aabb_max[3];
	pt_material_desc material;
} pt_object_xform_desc;

/* The four vectors Camera::getRay uses (Camera.h:15-18, Camera.inl:25-28): origin, lower-left corner, horizontal, vertical. */
typedef struct pt_camera_vectors {
	float origin[3];
	float lower_left[3];
	float horizontal[3];
	float vertical[3];
} pt_camera_vectors;

typedef struct pt_context pt_context;

/* Pathtracer::Pathtracer(width, height, openglPixelBuffer = 0)   Pathtracer.h:15, Pathtracer.cpp:30-68.
 * `device` is the CUDA ordinal (the reference hard-wires 0, Pathtracer.cpp:40).  No GL interop. */
int pt_create(uint32_t width, uint32_t height, int device, pt_context **out);
/* Pathtracer::~Pathtracer   Pathtracer.cpp:70-109 */
void pt_destroy(pt_context *ctx);

/* Multi-GPU context (SURVEY.md §8b / §8e; the reference is fixed to device 0, Pathtracer.cpp:40).  `device_mask` bit i = CUDA
 * ordinal i; the lowest set bit is the ROOT device, whose buffers the image getters read.  The returned context is used
 * with the SAME entry points as a single-device one: pt_set_scene builds the BVH once and replicates it, textures / skybox /
 * options go to every device, pt_render splits the work and runs one host thread per GPU (blocking, like every call), the
 * image getters, pt_get_timing_ms (slowest device + exchange) and pt_get_stats (sums) answer for the whole job.
 * Options of a multi-GPU context:
 *  "partition"  0 (default): PIXELS - device i renders all samples of the pixels i, i + N, ... (row-major); the image is
 *               bit-identical to the single-GPU one.  1: SAMPLES - device i renders the global sample indices i, i + N, ... of
 *               every pixel (north_star's split); equal up to float summation order (and to the per-launch stratification).
 *  "exchange"   how the image comes together on the root.  1 / -1 (default, when the devices have peer access): pixel
 *               partition only - the kernels of the other devices store their finished pixels directly into the root's
 *               accumulation buffer over NVLink (16 B per pixel, no collective).  0: ONE ncclReduce (sum, float32, 4*W*H
 *               elements) of the per-device accumulation buffers into a buffer on the root; always used by the sample
 *               partition.  NCCL (libnccl.so.2) is loaded with dlopen the first time it is needed. */
int pt_create_multi(uint32_t width, uint32_t height, uint32_t device_mask, pt_context **out);
/* devices of the context (1 for pt_create), whether the last / next pt_render exchanges by peer-to-peer stores, and the two
 * parts of pt_get_timing_ms of the last pt_render: slowest device's trace time, device time of the ncclReduce (0 with p2p). */
int pt_get_multi_info(const pt_context *ctx, int *devices, int *peer_to_peer, float *trace_ms, float *exchange_ms);

/* Pathtracer::setScene(count, hittables)   Pathtracer.h:22, Pathtracer.cpp:111-160.  Copies the input, builds the
 * BVH, replaces the previous scene.  count == 0 prints the reference's message and is a no-op returning PT_OK. */
int pt_set_scene(pt_context *ctx, size_t count, const pt_object_desc *objects);

/* Pathtracer::setScene for callers that hold reference CpuHittables (see pt_object_xform_desc): same semantics as
 * pt_set_scene, the transforms and boxes are taken as given instead of being derived from position / rotation / scale. */
int pt_set_scene_xform(pt_context *ctx, size_t count, const pt_object_xform_desc *objects);

/* Pathtracer::loadTexture(path)   Pathtracer.h:35, Pathtracer.cpp:234-292.  Returns a 1-based handle, 0 on failure or
 * when 64 textures exist.  ".hdr" (Radiance RGBE) -> float RGBA, anything else (PNG) -> 8-bit RGBA. */
uint32_t pt_load_texture(pt_context *ctx, const char *path);
/* same, from decoded RGBA texels already in host memory (is_hdr: float[4] per texel, else uint8[4]). */
uint32_t pt_load_texture_mem(pt_context *ctx, uint32_t width, uint32_t height, int is_hdr, const void *rgba);

/* Pathtracer::setSkyboxTextureHandle(handle)   Pathtracer.h:38, Pathtracer.cpp:294-297.  0 = black environment. */
int pt_set_skybox(pt_context *ctx, uint32_t handle);

/* Pathtracer::render(camera, spp, ignoreHistory)   Pathtracer.h:26, Pathtracer.cpp:162-227.  Synchronous.  Adds `spp`
 * samples per pixel to the accumulation (or restarts it).  spp == 0 or no scene -> no kernel. */
int pt_render(pt_context *ctx, const pt_camera_desc *camera, uint32_t spp, int ignore_history);

/* Pathtracer::render for callers that hold a reference Camera object: its four ray vectors as they stand (pt_camera_vectors),
 * no re-derivation from position / look-at / fovy. */
int pt_render_vectors(pt_context *ctx, const pt_camera_vectors *camera, uint32_t spp, int ignore_history);

/* Pathtracer::getTiming()   Pathtracer.h:29, Pathtracer.cpp:229-232.  GPU ms of the last pt_render. */
float pt_get_timing_ms(const pt_context *ctx);

/* Pathtracer::getHDRImageData()   Pathtracer.h:41, Pathtracer.cpp:299-315.  Library-owned W*H*4 floats, valid until
 * the next call on ctx.  Normalised exactly like the reference: accumulation / number of render() calls
 * (SURVEY.md Q1), all four channels scaled. */
const float *pt_get_hdr(pt_context *ctx);
/* Pathtracer::getImageData()   Pathtracer.h:44, Pathtracer.cpp:317-339 + kernels/tonemap.cu:4-27.  Library-owned
 * W*H*4 bytes RGBA8 (A = 255): mean -> Reinhard -> gamma 1/2.2 -> truncate. */
const uint8_t *pt_get_ldr(pt_context *ctx);

/* ---- extensions (not in the reference class; used by the CLI, the tests and the bench) ---- */

/* W*H*4 floats of the TRUE per-sample mean (accumulation / total samples), library-owned. */
const float *pt_get_hdr_mean(pt_context *ctx);
/* W*H*4 floats of the raw accumulation buffer (per-pixel sums, alpha = 1; what kernels/tonemap.cu reads), library-owned. */
const float *pt_get_hdr_sum(pt_context *ctx);

/* Options (all doubles):
 *  "seed"            Philox key (default 1984, cf. kernels/initRandState.cu:16)
 *  "sample_offset"   global index of the first sample of the next pt_render (multi-GPU sample partition)
 *  "sample_stride"   distance between this context's consecutive global sample indices (1 = contiguous)
 *  "pixel_offset"    multi-GPU pixel partition: this context renders the pixels offset, offset + stride, ... (row-major index)
 *  "pixel_stride"    with all of their samples; with stride > 1 a pt_render that restarts the accumulation zeroes the buffer first,
 *                    so that the sum of the ranks' buffers is the image (default 0 / 1: every pixel)
 *  "total_samples" / "accumulated_frames"  overwrite the counts the image getters normalise by (after a multi-GPU reduce the
 *                    destination's buffer holds the samples of all ranks)
 *  "alpha"           what pt_render writes into the fourth channel of the accumulation buffer (default 1, kernels/trace.cu:198); ranks > 0
 *                    of a multi-process sample partition set 0 so that the reduced alpha is 1
 *  "frames_per_spp"  k>0: a pt_render of spp samples counts ceil(spp/k) frames for the Q1 normalisation
 *                    (k=8 reproduces the reference headless CLI, main.cpp:271-278); 0: one frame per call
 *  "count_work"      1: count node visits / primitive tests / shades / misses (slower)
 *  "smem_scene"      0: never stage the scene in shared memory; 1: auto (default)
 *  "max_bounces"     path segments, default 5 (kernels/trace.cu:109)
 *  "max_leaf"        primitives per BVH leaf at most (default 4, the reference's Pathtracer.cpp:121; set before the scene)
 *  "bvh_builder"     0: binned SAH, as good a tree as the reference's (BVH.cpp:66-228); 1: LBVH - Morton order of the centroids +
 *                    Karras' radix tree, one primitive per leaf - built by all cores in a tenth of the time, traversal ~2 % slower
 *                    (measured on 10 k ... 1 M objects); 2 (default): LBVH from 2^19 objects, SAH below (set before the scene)
 *  "max_global"      how many scene-spanning primitives are hoisted out of the BVH (default 8; set before the scene)
 *  "variant"         trace kernel: 0 (default) = 12 from 64 spp, 4 below; 4 = one pixel per lane; 12 = one pixel per warp, with
 *                    separate passes for camera rays and scattered rays.  Any other value returns PT_E_INVALID
 *  "beam"            pixel beams for camera rays (one-pixel-per-warp kernels): 1 on, 0 off, -1 auto (default: on from 128 spp)
 *  "regen_low"       one-pixel-per-warp kernels: idle lanes wait until this many can start new samples together (0 = default)
 *  "stratify"        one-pixel-per-warp kernels: stratify the two randoms of the FIRST scattering direction over the samples of a
 *                    pixel (2^k cells of equal sample count, k <= 8; the cell is the top bits, the Philox draw the rest).  Same
 *                    expectation as the reference's plain draws (Material.inl:40-41), never more variance, and the lanes of a
 *                    warp scatter into the same cell (coherent traversal): 1 on, 0 off, -1 auto (default: on from 128 spp)
 *  "smem_stack"      traversal stack in shared memory instead of local memory: 1 / -1 (default) when it fits, 0 off
 *  "jitter"          0: every sample goes through the pixel centre, u = (x + 0.5) / W (parity aid; default 1 = trace.cu:190-191)
 *  "first_hit"       1: pt_render also records, per pixel, the scene index and t of the closest hit of the camera ray AS FOUND BY
 *                    THE RENDER KERNEL ITSELF (pt_get_first_hit); with "jitter" = 0 this is the primary-pass gate on the
 *                    production traversal (beams, MUFU reciprocals and all).  Both aids are compiled into a twin instantiation
 *                    of each trace kernel - same template, same arguments - which renders the same bits
 *                    as the instantiation without them (checked in tests/test_gpu_baseline_sizes.py)
 *  "env_is"          1: every scattering vertex also draws one direction from the sky's importance distribution
 *                    (pt_env_distribution) and the sky light reaching it is estimated by multiple importance sampling (balance
 *                    heuristic) of that draw and the BSDF's own.  The same integral as the reference's estimator (paths of at
 *                    most max_bounces segments, sky light through a miss) - the image converges to the same picture, with less
 *                    variance per sample under a sky with a sun; one more ray per vertex.  Default 0 (trace.cu:115-134).
 *  "light_is"        1: every scattering vertex also draws one point on an emissive object (pt_light_distribution picks the object,
 *                    the point is uniform over its surface) and traces a shadow ray to it; the light of the emitters is estimated by
 *                    multiple importance sampling (balance heuristic) of that point and the BSDF's own direction.  The same integral as
 *                    the reference's estimator (emission added where a path segment hits an emitter) - the image converges to the same
 *                    picture, with less variance per sample in scenes lit by small emitters; one more ray per vertex.  A scene without
 *                    emitters renders as without the option.  Not combinable with "env_is" or the parity aids (pt_render returns
 *                    PT_E_INVALID).  Default 0 (trace.cu:136-151).
 *  "tex_unit"        1 (default): texture taps through CUDA texture objects, as the reference (Pathtracer.cpp:259-288);
 *                    0: fp32 bilinear filter in software over the packed texels */
int pt_set_option(pt_context *ctx, const char *key, double value);
int pt_get_stats(const pt_context *ctx, pt_stats *out);

/* Camera::rotate(pitch, yaw, roll) / Camera::translate(x, y, z)   Camera.h:10-11, Camera.inl:30-52 (the reference's
 * interactive controls, main.cpp:404-420).  Host-only helpers on the POD camera: angles in radians, pitch about the
 * camera's right axis, yaw about the world up axis, roll ignored (as in the reference); the translation is along the camera's
 * right / up / backward axes.  The next pt_render with the changed camera should pass ignore_history = 1. */
void pt_camera_rotate(pt_camera_desc *camera, float pitch, float yaw, float roll);
void pt_camera_translate(pt_camera_desc *camera, float x, float y, float z);

/* Deterministic primary-ray pass (parity gate): pixel-centre rays u=(x+0.5)/W, v=(y+0.5)/H, t_min=0.001; writes the
 * scene-order object index (or -1) and hit t (0 on miss) per pixel into HOST buffers of W*H elements. */
int pt_primary_pass(pt_context *ctx, const pt_camera_desc *camera, int32_t *hit_index, float *hit_t);

/* After a pt_render with option "first_hit" = 1: scene-order object index (-1: miss) and t (0 on a miss) of the camera ray's
 * closest hit per pixel, as found by the render kernel, into HOST buffers of W*H elements. */
int pt_get_first_hit(pt_context *ctx, int32_t *hit_index, float *hit_t);

/* Closest-hit queries for caller-supplied rays (n rays, origin/direction as xyz triples in host memory). */
int pt_trace_rays(pt_context *ctx, size_t n, const float *origins, const float *directions, float t_min,
                  int32_t *hit_index, float *hit_t, float *hit_normal);

/* Device pointer of the float4 accumulation buffer (W*H*4 floats) for the multi-GPU reduce, and a setter so the
 * caller can supply its own allocation (e.g. a torch tensor reduced with torch.distributed / NCCL). */
void *pt_accum_device_ptr(pt_context *ctx);
int pt_set_accum_device_ptr(pt_context *ctx, void *device_ptr);

/* loadScene(pathtracer, params)   SceneLoader.cpp:124-348: parse the JSON scene, load its textures (paths relative to
 * the process CWD), set scene + skybox, return the camera for aspect = width/height of ctx. */
int pt_load_scene_file(pt_context *ctx, const char *json_path, pt_camera_desc *camera_out);
/* parse only: fills up to `capacity` objects, returns the object count (or a negative error).  Texture paths are
 * returned as indices into a '\n'-joined list written to tex_paths (may be NULL). */
int pt_parse_scene_file(const char *json_path, pt_object_desc *objects, size_t capacity, pt_camera_desc *camera_out,
                        float aspect, char *tex_paths, size_t tex_paths_cap, int32_t *skybox_tex_index);

/* stbi_write_png / stbi_write_hdr with flip-on-write   main.cpp:180-199.  data is bottom-row-first RGBA. */
int pt_write_png(const char *path, uint32_t width, uint32_t height, const uint8_t *rgba);
int pt_write_hdr(const char *path, uint32_t width, uint32_t height, const float *rgba);
/* decoders used by pt_load_texture (stbi_load / stbi_loadf replacement).  Caller frees with pt_free. */
int pt_read_image(const char *path, uint32_t *width, uint32_t *height, int *is_hdr, void **rgba);
void pt_free(void *p);

/* The importance distribution option "env_is" samples the sky with (no counterpart in the reference, which evaluates the sky only
 * where a path misses, kernels/trace.cu:115-134): a grid of cols x rows cells (at most 512 x 256) over the equirectangular map
 * `rgba` (width x height, float RGBA when is_hdr, else RGBA8), cell weight = sum over its texels of luminance x sin(theta).
 * alias: 2 words per cell (float bits of the acceptance threshold, alias cell) - one table over all cells; density: per cell
 * P(cell) x cells / (2 pi^2), so that the solid-angle pdf of a direction in the cell is density / sin(theta).  Host only.
 * Call with alias = density = NULL for the grid size; returns the cell count or a negative error. */
int pt_env_distribution(uint32_t width, uint32_t height, int is_hdr, const void *rgba, uint32_t *cols, uint32_t *rows, uint32_t *alias, float *density);

/* The emitter table option "light_is" samples (no counterpart in the reference, which finds an emitter only when a BSDF-sampled ray
 * hits it): every object with a non-zero emissive channel is one emitter, in the order of `objects`; selection weight = mean emissive x
 * world surface area (exact for disks, quads and cubes under any transform, the uniform-scale value for the curved shapes).  Writes per
 * emitter its index in `objects`, its selection probability and its alias-table entry (2 words: float bits of the acceptance threshold,
 * alias emitter).  Host only.  Call with NULL buffers for the count; returns the emitter count (0 when nothing emits) or a negative error. */
int pt_light_distribution(size_t count, const pt_object_desc *objects, uint32_t *scene_index, float *probability, uint32_t *alias);

const char *pt_last_error(void);
const char *pt_version(void);

#ifdef __cplusplus
}
#endif
#endif
