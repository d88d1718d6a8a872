/* pt_oracle.h — CPU restatement of the reference trace path.  TEST INFRASTRUCTURE ONLY: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may load this library; the
 * product (pathtracercuda_b200/) never links or calls it.  See pt_oracle.c for the per-function citations. */
#ifndef PT_ORACLE_H
#define PT_ORACLE_H
#include "../include/pt_b200.h"
#ifdef __cplusplus
extern "C" {
#endif
typedef struct orc_scene orc_scene;

orc_scene *orc_scene_create(size_t count, const pt_object_desc *objects);
void orc_scene_destroy(orc_scene *s);
/* textures: 1-based handles in load order, like Pathtracer::loadTexture */
uint32_t orc_add_texture(orc_scene *s, uint32_t w, uint32_t h, int is_hdr, const void *rgba);
void orc_set_skybox(orc_scene *s, uint32_t handle);
/* NOT THE REFERENCE: the product's "env_is" estimator (csrc/env_sampling.h), restated so that the CUDA path can be checked path for path */
void orc_set_env_is(orc_scene *s, int on);
uint32_t orc_env_tables(const orc_scene *s, uint32_t *cols, uint32_t *rows, float *q, uint32_t *alias, float *density);
void orc_env_sample(const orc_scene *s, uint32_t r0, uint32_t r1, uint32_t r2, float *out6);
/* NOT THE REFERENCE: the product's "light_is" estimator (csrc/light_sampling.h), restated likewise.  Not to be combined with
 * env_is, which pt_render refuses too */
void orc_set_light_is(orc_scene *s, int on);
uint32_t orc_light_table(const orc_scene *s, uint32_t *scene, float *prob, float *q, uint32_t *alias);
void orc_light_sample_point(const orc_scene *s, const uint32_t *q, float *out8);
void orc_bvh_info(const orc_scene *s, uint32_t *nodes, uint32_t *depth, int32_t *valid);
/* per object: 12 floats world->local rows, 6 floats AABB (min, max) */
void orc_object_info(const orc_scene *s, size_t i, float *rows12, float *aabb6);
void orc_camera_ray(const pt_camera_desc *cam, float s, float t, float *out6);
int orc_hit_object(const orc_scene *s, size_t i, const float *o, const float *d, float tmin, float tmax, float *out10);
void orc_material_sample(const pt_material_desc *m, const float *N, const float *in_dir, float rnd0, float rnd1, float *out9);
void orc_primary_pass(const orc_scene *s, const pt_camera_desc *cam, uint32_t w, uint32_t h, int32_t *idx, float *t, uint64_t *stats2);
void orc_trace_rays(const orc_scene *s, size_t n, const float *o, const float *d, float tmin, int32_t *idx, float *t, float *nrm);
/* accum (W*H*4 floats) = sum of spp samples per pixel with global sample indices sample_offset + k*sample_stride;
 * returns rays traced.  add != 0 accumulates onto the buffer (ignoreHistory = false). */
uint64_t orc_render(const orc_scene *s, const pt_camera_desc *cam, uint32_t w, uint32_t h, uint32_t spp, uint64_t seed,
                    uint32_t sample_offset, uint32_t sample_stride, int add, int max_bounces, float *accum);
/* first-bounce stratification of the product's one-pixel-per-warp kernels (not in the reference; see pt_oracle.c) */
/* distance of a ray from the nearest accept / reject decision of one object, in units of float32 rounding noise (test aid) */
double orc_decision_margin(const orc_scene *s, size_t i, const float *o, const float *d);
void orc_set_stratify(int on);
int orc_threads(int n);
void orc_tonemap(const float *accum, size_t pixels, uint32_t sample_count, uint8_t *out);
void orc_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out4);
float orc_uniform(uint32_t x);
void orc_texture_lookup(const orc_scene *s, uint32_t handle, float u, float v, float *out4);
#ifdef __cplusplus
}
#endif
#endif
