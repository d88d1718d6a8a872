/* pt_oracle.c — CPU ORACLE for the trace hot path.  TEST INFRASTRUCTURE ONLY (see pt_oracle.h).
 *
 * A plain-C restatement of the reference's algorithm, function by function, each citing the reference lines it
 * follows (paths relative to /root/reference/PathtracerCUDA/src/pathtracer/).  Floating-point operation ORDER follows
 * the reference expressions so that, compiled with -ffp-contract=off like oracle/_ref/libref_host.so (the reference's
 * own headers built with g++), the deterministic parts agree bit for bit.
 *
 * PINNING (tests/test_oracle_vs_reference.py, run in the build container where /root/reference exists; results
 * frozen as tests/golden/ fixtures for boxes without it):
 *   - transforms / AABBs / BVH shape / camera rays / per-shape hits / primary pass: bit-exact vs libref_host.so
 *   - Material::sample at the reference's own (rnd0, rnd1) draws: bit-exact vs libref_host.so
 *   - full path tracing: the RNG differs BY DESIGN (Philox4x32-10 keyed on pixel/sample/bounce instead of per-pixel
 *     XORWOW, north_star item 4), so images agree statistically: RMSE(oracle, ref seed A) <= 1.1 x RMSE(ref A, ref B).
 * Texture filtering: the reference uses the texture unit (tex2D, 9-bit weights); this oracle and the product use
 * the same rule in fp32 (normalized coords, texel centres at +0.5, wrap U, clamp V, Pathtracer.cpp:276-281).
 */
#include "pt_oracle.h"
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define PI_F (3.14159265358979323846f) /* vec3.h:5 */

typedef struct { float x, y, z; } v3;
typedef struct { v3 o, d; } ray_t;
typedef struct { v3 mn, mx; } aabb_t;

typedef struct
{
	float r0[4], r1[4], r2[4]; /* world->local rows (Hittable.h:22-24) */
	uint32_t type;
	/* Material (Material.h:22-27) */
	v3 baseColor; float roughness; v3 emissive; float metalness; uint32_t texture; uint32_t mtype;
	aabb_t box;
} obj_t;

typedef struct { aabb_t box; uint32_t offset; uint32_t countAxis; } node_t; /* BVH.h:6-11 */

typedef struct { uint32_t w, h; int hdr; float *f; uint8_t *b; } tex_t;

/* NOT THE REFERENCE: one emitter of the "light_is" estimator (csrc/light_sampling.h) */
typedef struct
{
	float m[12];    /* local -> world rows */
	float pdfScale; /* P_sel / (A_l |det M|) */
	float q;        /* alias threshold */
	uint32_t alias, scene, type;
	float prob;
} light_t;

struct orc_scene
{
	size_t n;
	obj_t *objs;      /* BVH order */
	int32_t *toScene; /* BVH order -> scene order */
	obj_t *sceneObjs; /* scene order */
	node_t *nodes; uint32_t nodeCount, nodeCap;
	tex_t tex[64]; uint32_t texCount; uint32_t skybox;
	/* NOT THE REFERENCE: importance distribution of the sky (option "env_is" of the product, csrc/env_sampling.h) */
	int envIS; uint32_t envCols, envRows; float *envQ; uint32_t *envAlias; float *envDensity;
	/* NOT THE REFERENCE: emitter table (option "light_is" of the product, csrc/light_sampling.h); lightCount is 0 unless the option is
	 * on and the scene emits.  lightOf: scene index -> emitter index, -1: not an emitter */
	uint32_t lightCount; light_t *lights; int32_t *lightOf;
};

/* ---- vec3.inl ------------------------------------------------------------------------------------------ */
static inline v3 V(float x, float y, float z) { v3 r = { x, y, z }; return r; }
static inline v3 vadd(v3 a, v3 b) { return V(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 vsub(v3 a, v3 b) { return V(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 vmul(v3 a, v3 b) { return V(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline v3 vscale(float t, v3 v) { return V(t * v.x, t * v.y, t * v.z); }             /* vec3.inl:126-129 */
static inline v3 vneg(v3 a) { return V(-a.x, -a.y, -a.z); }
static inline float vdot(v3 u, v3 v) { return u.x * v.x + u.y * v.y + u.z * v.z; }            /* vec3.inl:156-161 */
static inline v3 vcross(v3 u, v3 v) { return V(u.y * v.z - u.z * v.y, u.z * v.x - u.x * v.z, u.x * v.y - u.y * v.x); }
static inline float vlen(v3 v) { return sqrtf(v.x * v.x + v.y * v.y + v.z * v.z); }
static inline v3 vdivf(v3 v, float t) { return vscale(1.0f / t, v); }                        /* vec3.inl:141-144 */
static inline v3 vnorm(v3 v) { return vdivf(v, vlen(v)); }                                   /* vec3.inl:197-200 */
static inline v3 vreflect(v3 v, v3 n) { return vsub(v, vscale(2.0f * vdot(v, n), n)); }      /* vec3.inl:202-205 */
static inline float clampf(float x, float a, float b) { x = x < a ? a : x; x = x > b ? b : x; return x; }
static inline v3 vmin(v3 a, v3 b) { return V(a.x < b.x ? a.x : b.x, a.y < b.y ? a.y : b.y, a.z < b.z ? a.z : b.z); }
static inline v3 vmax(v3 a, v3 b) { return V(a.x >= b.x ? a.x : b.x, a.y >= b.y ? a.y : b.y, a.z >= b.z ? a.z : b.z); }
static inline float vget(v3 v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : v.z); }
static inline v3 rat(ray_t r, float t) { return vadd(r.o, vscale(t, r.d)); }                 /* Ray.h:19-22 */

/* ---- Hittable.cpp:6-103 worldTransform ------------------------------------------------------------------- */
static void quatToRotMat(const float q[4] /* x y z w */, float m[3][3])
{
	float qxx = q[0] * q[0], qyy = q[1] * q[1], qzz = q[2] * q[2], qxz = q[0] * q[2], qxy = q[0] * q[1], qyz = q[1] * q[2];
	float qwx = q[3] * q[0], qwy = q[3] * q[1], qwz = q[3] * q[2];
	m[0][0] = 1.0f - 2.0f * (qyy + qzz); m[0][1] = 2.0f * (qxy + qwz); m[0][2] = 2.0f * (qxz - qwy);
	m[1][0] = 2.0f * (qxy - qwz); m[1][1] = 1.0f - 2.0f * (qxx + qzz); m[1][2] = 2.0f * (qyz + qwx);
	m[2][0] = 2.0f * (qxz + qwy); m[2][1] = 2.0f * (qyz - qwx); m[2][2] = 1.0f - 2.0f * (qxx + qyy);
}

static void worldTransform(v3 position, v3 rotation, v3 scale, float l2w[3][4], float w2l[3][4])
{
	float q[4], invQ[4];
	{
		v3 c = V(cosf(rotation.x * 0.5f), cosf(rotation.y * 0.5f), cosf(rotation.z * 0.5f));
		v3 s = V(sinf(rotation.x * 0.5f), sinf(rotation.y * 0.5f), sinf(rotation.z * 0.5f));
		q[3] = c.x * c.y * c.z + s.x * s.y * s.z;
		q[0] = s.x * c.y * c.z - c.x * s.y * s.z;
		q[1] = c.x * s.y * c.z + s.x * c.y * s.z;
		q[2] = c.x * c.y * s.z - s.x * s.y * c.z;
	}
	{
		float invDot = (1.0f / (q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]));
		invQ[0] = -q[0] * invDot; invQ[1] = -q[1] * invDot; invQ[2] = -q[2] * invDot; invQ[3] = q[3] * invDot;
	}
	{
		float m[3][3];
		quatToRotMat(invQ, m);
		v3 invScale = V(1.0f / scale.x, 1.0f / scale.y, 1.0f / scale.z);
		v3 np = vneg(position);
		w2l[0][0] = invScale.x * m[0][0]; w2l[0][1] = invScale.x * m[1][0]; w2l[0][2] = invScale.x * m[2][0];
		w2l[0][3] = invScale.x * vdot(V(m[0][0], m[1][0], m[2][0]), np);
		w2l[1][0] = invScale.y * m[0][1]; w2l[1][1] = invScale.y * m[1][1]; w2l[1][2] = invScale.y * m[2][1];
		w2l[1][3] = invScale.y * vdot(V(m[0][1], m[1][1], m[2][1]), np);
		w2l[2][0] = invScale.z * m[0][2]; w2l[2][1] = invScale.z * m[1][2]; w2l[2][2] = invScale.z * m[2][2];
		w2l[2][3] = invScale.z * vdot(V(m[0][2], m[1][2], m[2][2]), np);
	}
	{
		float m[3][3];
		quatToRotMat(q, m);
		l2w[0][0] = scale.x * m[0][0]; l2w[0][1] = scale.y * m[1][0]; l2w[0][2] = scale.z * m[2][0]; l2w[0][3] = position.x;
		l2w[1][0] = scale.x * m[0][1]; l2w[1][1] = scale.y * m[1][1]; l2w[1][2] = scale.z * m[2][1]; l2w[1][3] = position.y;
		l2w[2][0] = scale.x * m[0][2]; l2w[2][1] = scale.y * m[1][2]; l2w[2][2] = scale.z * m[2][2]; l2w[2][3] = position.z;
	}
}

/* Hittable.cpp:115-179 CpuHittable ctor, Material.inl:8-18 Material ctor */
static void makeObject(const pt_object_desc *d, obj_t *o)
{
	v3 scale = V(d->scale[0], d->scale[1], d->scale[2]);
	if (d->type == PT_DISK || d->type == PT_QUAD) scale.y = 1.0f;
	float l2w[3][4], w2l[3][4];
	worldTransform(V(d->position[0], d->position[1], d->position[2]), V(d->rotation[0], d->rotation[1], d->rotation[2]), scale, l2w, w2l);
	memcpy(o->r0, w2l[0], 16); memcpy(o->r1, w2l[1], 16); memcpy(o->r2, w2l[2], 16);
	o->type = d->type;
	o->baseColor = V(d->material.base_color[0], d->material.base_color[1], d->material.base_color[2]);
	o->emissive = V(d->material.emissive[0], d->material.emissive[1], d->material.emissive[2]);
	o->roughness = d->material.roughness < 0.04f ? 0.04f : d->material.roughness;
	o->metalness = d->material.metalness;
	o->texture = d->material.texture;
	o->mtype = d->material.type;
	float xe[2] = { -1.0f, 1.0f }, ye[2] = { -1.0f, 1.0f }, ze[2] = { -1.0f, 1.0f };
	if (d->type == PT_DISK || d->type == PT_QUAD) { ye[0] = -0.01f; ye[1] = 0.01f; }
	else if (d->type == PT_PARABOLOID) { ye[0] = 0.0f; }
	o->box.mn = V(FLT_MAX, FLT_MAX, FLT_MAX);
	o->box.mx = V(-FLT_MAX, -FLT_MAX, -FLT_MAX);
	for (int z = 0; z < 2; ++z) for (int y = 0; y < 2; ++y) for (int x = 0; x < 2; ++x)
	{
		v3 c = V(xe[x], ye[y], ze[z]), p;
		p.x = vdot(c, V(l2w[0][0], l2w[0][1], l2w[0][2])) + l2w[0][3];
		p.y = vdot(c, V(l2w[1][0], l2w[1][1], l2w[1][2])) + l2w[1][3];
		p.z = vdot(c, V(l2w[2][0], l2w[2][1], l2w[2][2])) + l2w[2][3];
		o->box.mn = vmin(o->box.mn, p);
		o->box.mx = vmax(o->box.mx, p);
	}
}

/* ---- AABB.inl:22-44 / 46-69 ------------------------------------------------------------------------------ */
static inline int aabbSlab(aabb_t b, ray_t r, float tMin, float tMax, float *tEntry)
{
	for (int a = 0; a < 3; ++a)
	{
		float invD = 1.0f / vget(r.d, a);
		float t0 = (vget(b.mn, a) - vget(r.o, a)) * invD;
		float t1 = (vget(b.mx, a) - vget(r.o, a)) * invD;
		if (invD < 0.0f) { float tmp = t0; t0 = t1; t1 = tmp; }
		tMin = t0 > tMin ? t0 : tMin;
		tMax = t1 < tMax ? t1 : tMax;
		if (tMax <= tMin) return 0;
	}
	if (tEntry) *tEntry = tMin;
	return 1;
}
static inline aabb_t aabbUnion(aabb_t a, aabb_t b) { aabb_t r; r.mn = vmin(a.mn, b.mn); r.mx = vmax(a.mx, b.mx); return r; }

/* ---- BVH.cpp:54-228 -------------------------------------------------------------------------------------- */
static float calcSurfaceArea(v3 mn, v3 mx)
{
	v3 e = vsub(mx, mn);
	if (e.x <= 0.0f || e.y <= 0.0f || e.z <= 0.0f) return 0.0f;
	return (e.x * e.y + e.x * e.z + e.y * e.z) * 2.0f;
}
static aabb_t emptyBox(void) { aabb_t b; b.mn = V(FLT_MAX, FLT_MAX, FLT_MAX); b.mx = V(-FLT_MAX, -FLT_MAX, -FLT_MAX); return b; }

static int g_sortAxis;
static int cmpCentroid(const void *pa, const void *pb)
{
	const obj_t *a = (const obj_t *)pa, *b = (const obj_t *)pb;
	float ca = vget(vscale(0.5f, vadd(a->box.mn, a->box.mx)), g_sortAxis), cb = vget(vscale(0.5f, vadd(b->box.mn, b->box.mx)), g_sortAxis);
	return ca < cb ? -1 : (ca > cb ? 1 : 0);
}

typedef struct { obj_t o; int32_t scene; } bobj_t;
static int cmpCentroidB(const void *pa, const void *pb) { return cmpCentroid(&((const bobj_t *)pa)->o, &((const bobj_t *)pb)->o); }

static uint32_t buildRecursive(orc_scene *s, bobj_t *e, size_t begin, size_t end, uint32_t maxLeaf)
{
	uint32_t nodeIndex = s->nodeCount++;
	node_t node; memset(&node, 0, sizeof node);
	node.box = emptyBox();
	for (size_t i = begin; i < end; ++i) node.box = aabbUnion(node.box, e[i].o.box);
	if ((end - begin) > maxLeaf)
	{
		uint32_t binCount[3][8]; aabb_t binBox[3][8];
		for (int a = 0; a < 3; ++a) for (int b = 0; b < 8; ++b) { binCount[a][b] = 0; binBox[a][b] = emptyBox(); }
		v3 ext = vmax(vsub(node.box.mx, node.box.mn), V(0.00000001f, 0.00000001f, 0.00000001f));
		for (size_t i = begin; i < end; ++i)
		{
			aabb_t eb = e[i].o.box;
			v3 centroid = vscale(0.5f, vadd(eb.mn, eb.mx));
			v3 diff = vsub(centroid, node.box.mn);
			/* operator/(vec3, vec3) = vec3(1/t.x, 1/t.y, 1/t.z) * v   (vec3.inl:136-139) */
			v3 rel = vmul(V(1.0f / ext.x, 1.0f / ext.y, 1.0f / ext.z), diff);
			for (int j = 0; j < 3; ++j)
			{
				int binIdx = (int)(vget(rel, j) * 8.0f);
				binIdx = binIdx < 0 ? 0 : binIdx > 7 ? 7 : binIdx;
				binCount[j][binIdx] += 1;
				binBox[j][binIdx] = aabbUnion(binBox[j][binIdx], eb);
			}
		}
		float sa = calcSurfaceArea(node.box.mn, node.box.mx);
		float invSA = 1.0f / (sa > 0.000000001f ? sa : 0.000000001f);
		float lowest = FLT_MAX; uint32_t bestAxis = 0, bestBin = 0;
		for (uint32_t i = 0; i < 3; ++i) for (uint32_t j = 0; j < 7; ++j)
		{
			aabb_t b0 = emptyBox(), b1 = emptyBox(); uint32_t c0 = 0, c1 = 0;
			for (uint32_t k = 0; k <= j; ++k) { b0 = aabbUnion(b0, binBox[i][k]); c0 += binCount[i][k]; }
			for (uint32_t k = j + 1; k < 8; ++k) { b1 = aabbUnion(b1, binBox[i][k]); c1 += binCount[i][k]; }
			float a0 = calcSurfaceArea(b0.mn, b0.mx), a1 = calcSurfaceArea(b1.mn, b1.mx);
			float cost = 0.125f + (c0 * a0 + c1 * a1) * invSA;
			cost = (c0 == 0 || c1 == 0) ? FLT_MAX : cost;
			if (cost < lowest) { lowest = cost; bestAxis = i; bestBin = j; }
		}
		/* std::partition (BVH.cpp:176-186): any partition into {bin <= bestBin} | {bin > bestBin} */
		size_t lo = begin, hi = end;
		while (lo < hi)
		{
			aabb_t eb = e[lo].o.box;
			v3 centroid = vscale(0.5f, vadd(eb.mn, eb.mx));
			/* float / float here (BVH.cpp:180): a true division, not reciprocal-multiply */
			float rel = (vget(centroid, bestAxis) - vget(node.box.mn, bestAxis)) / vget(ext, bestAxis);
			int binIdx = (int)(8.0f * rel);
			binIdx = binIdx < 0 ? 0 : binIdx > 7 ? 7 : binIdx;
			if ((uint32_t)binIdx <= bestBin) ++lo;
			else { --hi; bobj_t tmp = e[lo]; e[lo] = e[hi]; e[hi] = tmp; }
		}
		size_t split = lo;
		if (split == begin || split == end)
		{
			bestAxis = (ext.x < ext.y) ? 0 : (ext.y < ext.z) ? 1 : 2;
			split = (begin + end) / 2;
			g_sortAxis = (int)bestAxis; /* std::nth_element (BVH.cpp:195-207): a full sort is one valid outcome */
			qsort(e + begin, end - begin, sizeof(bobj_t), cmpCentroidB);
		}
		buildRecursive(s, e, begin, split, maxLeaf);
		node.offset = buildRecursive(s, e, split, end, maxLeaf);
		node.countAxis |= (bestAxis << 8);
	}
	else
	{
		node.offset = (uint32_t)begin;
		node.countAxis |= (uint32_t)(end - begin) << 16;
	}
	s->nodes[nodeIndex] = node;
	return nodeIndex;
}

static uint32_t bvhDepth(const orc_scene *s, uint32_t n)
{
	if (s->nodes[n].countAxis >> 16) return 1;
	uint32_t a = bvhDepth(s, n + 1), b = bvhDepth(s, s->nodes[n].offset);
	return 1 + (a > b ? a : b);
}

/* ---- Hittable.inl ---------------------------------------------------------------------------------------- */
static inline int quadratic(float a, float b, float c, float *t0, float *t1) /* Hittable.inl:7-39 */
{
	const float disc = b * b - 4.0f * a * c;
	if (disc < 0.0f) return 0;
	const float root = sqrtf(disc);
	const float q = b < 0.0f ? -0.5f * (b - root) : -0.5f * (b + root);
	*t0 = q / a;
	*t1 = c / q;
	if (*t0 > *t1) { float tmp = *t0; *t0 = *t1; *t1 = tmp; }
	return 1;
}

/* hitQuadric<A..J> (Hittable.inl:42-55) with the template constants written out as float products in the reference's
 * term order (int * float promotes to float; "0 * x" terms contribute +0/-0 and are kept for NaN/sign fidelity only
 * where they could matter - they cannot change a finite sum, so they are dropped). */
static inline int hitQuadricABC(int A, int B, int C, int Hc, int J, v3 o, v3 d, float *t0, float *t1)
{
	float a = (A * d.x * d.x) + (B * d.y * d.y) + (C * d.z * d.z) + (0 * d.x * d.y) + (0 * d.x * d.z) + (0 * d.y * d.z);
	float b = (2.0f * A * o.x * d.x) + (2.0f * B * o.y * d.y) + (2.0f * C * o.z * d.z) + (0 * (o.x * d.y + o.y * d.x))
		+ (0 * (o.x * d.z + o.z * d.x)) + (0 * (o.y * d.z + d.y * o.z)) + (0 * d.x) + (Hc * d.y) + (0 * d.z);
	float c = (A * o.x * o.x) + (B * o.y * o.y) + (C * o.z * o.z) + (0 * o.x * o.y) + (0 * o.x * o.z) + (0 * o.y * o.z) + (0 * o.x) + (Hc * o.y) + (0 * o.z) + J;
	return quadratic(a, b, c, t0, t1);
}

typedef struct { float t; v3 p, n; float u, v; int front; int hit; } hit_t;

static int hitLocal(uint32_t type, ray_t r, float tMin, float tMax, float *t, v3 *normal, float *u, float *v)
{
	float t0 = 0.0f, t1 = 0.0f;
	switch (type)
	{
	case PT_SPHERE: /* Hittable.inl:147-169 */
	{
		if (!hitQuadricABC(1, 1, 1, 0, -1, r.o, r.d, &t0, &t1) || t0 > tMax || t1 <= tMin) return 0;
		*t = t0 > tMin ? t0 : t1;
		*normal = vnorm(rat(r, *t));
		float theta = acosf(normal->y), phi = atan2f(normal->z, normal->x);
		*u = 1.0f - phi / (2.0f * PI_F);
		*v = theta / PI_F;
		return 1;
	}
	case PT_CYLINDER: /* Hittable.inl:171-203 */
	case PT_CONE:     /* Hittable.inl:237-266 */
	case PT_PARABOLOID: /* Hittable.inl:268-297 */
	{
		int ok = type == PT_CYLINDER ? hitQuadricABC(1, 0, 1, 0, -1, r.o, r.d, &t0, &t1)
			: type == PT_CONE ? hitQuadricABC(1, -1, 1, 0, 0, r.o, r.d, &t0, &t1)
			: hitQuadricABC(1, 0, 1, -1, 0, r.o, r.d, &t0, &t1);
		if (!ok || t0 > tMax || t1 <= tMin) return 0;
		const float h0 = r.d.y * t0 + r.o.y, h1 = r.d.y * t1 + r.o.y;
		const int v0 = t0 > tMin && t0 <= tMax && h0 >= -1.0f && h0 <= 1.0f;
		const int v1 = t1 > tMin && t1 <= tMax && h1 >= -1.0f && h1 <= 1.0f;
		if (!v0 && !v1) return 0;
		*t = v0 ? t0 : t1;
		v3 p = rat(r, *t);
		if (type == PT_CYLINDER)
		{
			*normal = V(p.x, 0.0f, p.z);
			float phi = atan2f(normal->z, normal->x);
			*u = 1.0f - phi / (2.0f * PI_F);
			*v = 1.0f - (p.y * 0.5f + 0.5f);
		}
		else if (type == PT_CONE) /* quadricNormal<1,-1,1> Hittable.inl:58-67 */
			*normal = V(2.0f * (1 * p.x) + (0 * p.y) + (0 * p.z) + 0, 2.0f * (-1 * p.y) + (0 * p.x) + (0 * p.z) + 0, 2.0f * (1 * p.z) + (0 * p.x) + (0 * p.y) + 0);
		else /* quadricNormal<1,0,1,0,0,0,0,-1> */
			*normal = V(2.0f * (1 * p.x) + (0 * p.y) + (0 * p.z) + 0, 2.0f * (0 * p.y) + (0 * p.x) + (0 * p.z) + -1, 2.0f * (1 * p.z) + (0 * p.x) + (0 * p.y) + 0);
		return 1;
	}
	case PT_DISK: /* Hittable.inl:205-235 */
	case PT_QUAD: /* Hittable.inl:299-329 */
	{
		if (r.d.y == 0.0f) return 0;
		*t = -r.o.y / r.d.y;
		if (*t <= tMin || *t > tMax) return 0;
		float hx = r.o.x + r.d.x * *t, hz = r.o.z + r.d.z * *t;
		if (type == PT_DISK) { if ((hx * hx + hz * hz) >= 1.0f) return 0; }
		else { if (fabsf(hx) > 1.0f || fabsf(hz) > 1.0f) return 0; }
		*normal = V(0.0f, 1.0f, 0.0f);
		*u = hx * 0.5f + 0.5f;
		*v = 1.0f - (hz * 0.5f + 0.5f);
		return 1;
	}
	case PT_CUBE: /* Hittable.inl:331-358 */
	{
		aabb_t b; b.mn = V(-1.0f, -1.0f, -1.0f); b.mx = V(1.0f, 1.0f, 1.0f);
		if (!aabbSlab(b, r, tMin, tMax, t)) return 0;
		v3 n = rat(r, *t);
		v3 an = V(fabsf(n.x), fabsf(n.y), fabsf(n.z));
		if (an.x > an.y && an.x > an.z) *normal = V(n.x > 0.0f ? 1.0f : -1.0f, 0.0f, 0.0f);
		else if (an.y > an.x && an.y > an.z) *normal = V(0.0f, n.y > 0.0f ? 1.0f : -1.0f, 0.0f);
		else *normal = V(0.0f, 0.0f, n.z > 0.0f ? 1.0f : -1.0f);
		return 1;
	}
	default: return 0;
	}
}

/* Hittable::hit  Hittable.inl:88-145.  Cone/paraboloid u,v are uninitialised in the reference (SURVEY.md Q3): 0 here. */
static int hitObject(const obj_t *h, ray_t r, float tMin, float tMax, hit_t *rec)
{
	ray_t lr;
	lr.o.x = vdot(r.o, V(h->r0[0], h->r0[1], h->r0[2])) + h->r0[3];
	lr.o.y = vdot(r.o, V(h->r1[0], h->r1[1], h->r1[2])) + h->r1[3];
	lr.o.z = vdot(r.o, V(h->r2[0], h->r2[1], h->r2[2])) + h->r2[3];
	lr.d.x = vdot(r.d, V(h->r0[0], h->r0[1], h->r0[2]));
	lr.d.y = vdot(r.d, V(h->r1[0], h->r1[1], h->r1[2]));
	lr.d.z = vdot(r.d, V(h->r2[0], h->r2[1], h->r2[2]));
	float t, u = 0.0f, v = 0.0f; v3 normal;
	if (!hitLocal(h->type, lr, tMin, tMax, &t, &normal, &u, &v)) return 0;
	v3 tmp;
	tmp.x = vdot(normal, V(h->r0[0], h->r1[0], h->r2[0]));
	tmp.y = vdot(normal, V(h->r0[1], h->r1[1], h->r2[1]));
	tmp.z = vdot(normal, V(h->r0[2], h->r1[2], h->r2[2]));
	rec->t = t;
	rec->p = rat(r, t);
	v3 on = vnorm(tmp);
	rec->front = vdot(r.d, on) < 0.0f; /* HitRecord.h:18-24 */
	rec->n = rec->front ? on : vneg(on);
	rec->u = u; rec->v = v;
	return 1;
}

/* hitBVH  kernels/trace.cu:28-98 */
static int hitBVH(const orc_scene *s, ray_t r, float tMin, float tMax, hit_t *rec, uint32_t *elem, uint64_t *nv, uint64_t *np)
{
	v3 inv;
	inv.x = 1.0f / (r.d.x != 0.0f ? r.d.x : 1e-7f);
	inv.y = 1.0f / (r.d.y != 0.0f ? r.d.y : 1e-7f);
	inv.z = 1.0f / (r.d.z != 0.0f ? r.d.z : 1e-7f);
	int neg[3] = { inv.x < 0.0f, inv.y < 0.0f, inv.z < 0.0f };
	uint32_t stack[64], sp = 0, cur = 0, elemIdx = UINT32_MAX;
	if (s->nodeCount == 0) return 0;
	for (;;)
	{
		const node_t *node = &s->nodes[cur];
		if (nv) ++*nv;
		if (aabbSlab(node->box, r, tMin, tMax, NULL))
		{
			const uint32_t pc = node->countAxis >> 16;
			if (pc > 0)
			{
				for (uint32_t i = 0; i < pc; ++i)
				{
					if (np) ++*np;
					if (hitObject(&s->objs[node->offset + i], r, tMin, tMax, rec)) { tMax = rec->t; elemIdx = node->offset + i; }
				}
				if (sp == 0) break;
				cur = stack[--sp];
			}
			else
			{
				int isNeg = neg[(node->countAxis >> 8) & 0xFF];
				stack[sp++] = isNeg ? (cur + 1) : node->offset;
				cur = isNeg ? node->offset : (cur + 1);
			}
		}
		else
		{
			if (sp == 0) break;
			cur = stack[--sp];
		}
	}
	*elem = elemIdx;
	return elemIdx != UINT32_MAX;
}

/* ---- Camera.inl:4-28,54-62 ------------------------------------------------------------------------------- */
typedef struct { v3 origin, ll, horiz, vert; } cam_t;
static cam_t makeCamera(const pt_camera_desc *c)
{
	cam_t k;
	float tanHalf = tanf(c->fovy * 0.5f);
	k.origin = V(c->position[0], c->position[1], c->position[2]);
	v3 backward = vnorm(vsub(k.origin, V(c->look_at[0], c->look_at[1], c->look_at[2])));
	v3 right = vnorm(vcross(V(c->up[0], c->up[1], c->up[2]), backward));
	v3 up = vcross(backward, right);
	float halfHeight = tanHalf, halfWidth = c->aspect * halfHeight;
	k.ll = vsub(vadd(vscale(-halfWidth, right), vscale(-halfHeight, up)), backward);
	k.horiz = vscale(2.0f * halfWidth, right);
	k.vert = vscale(2.0f * halfHeight, up);
	return k;
}
static inline ray_t cameraRay(const cam_t *k, float s, float t)
{
	ray_t r; r.o = k->origin;
	r.d = vnorm(vadd(vadd(k->ll, vscale(s, k->horiz)), vscale(t, k->vert)));
	return r;
}

/* ---- RNG: Philox4x32-10 (Salmon et al. 2011), counter = (pixel, sample, slot, 0), key = (seed lo, seed hi) ---- */
void orc_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out)
{
	for (int i = 0; i < 10; ++i)
	{
		uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
		uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
		c0 = n0; c1 = n1; c2 = n2; c3 = n3;
		k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
	}
	out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
/* same map as cuRAND's curand_uniform (curand_kernel.h _curand_uniform): (0, 1] */
float orc_uniform(uint32_t x) { return fmaf((float)x, 2.3283064365386963e-10f, 1.16415321826934814453125e-10f); }

/* ---- textures: tex2D<float4> linear / normalized / wrap-U clamp-V (Pathtracer.cpp:276-281) in fp32 --------- */
static void texLookup(const tex_t *t, float u, float v, float out[4])
{
	float x = u * (float)t->w - 0.5f, y = v * (float)t->h - 0.5f;
	float fx = floorf(x), fy = floorf(y);
	float ax = x - fx, ay = y - fy;
	int x0 = (int)fx, y0 = (int)fy, W = (int)t->w, H = (int)t->h;
	int xa = x0 % W; if (xa < 0) xa += W;
	int xb = (x0 + 1) % W; if (xb < 0) xb += W;
	int ya = y0 < 0 ? 0 : (y0 > H - 1 ? H - 1 : y0);
	int yb = y0 + 1 < 0 ? 0 : (y0 + 1 > H - 1 ? H - 1 : y0 + 1);
	for (int c = 0; c < 4; ++c)
	{
		float t00, t10, t01, t11;
		if (t->hdr)
		{
			t00 = t->f[((size_t)ya * W + xa) * 4 + c]; t10 = t->f[((size_t)ya * W + xb) * 4 + c];
			t01 = t->f[((size_t)yb * W + xa) * 4 + c]; t11 = t->f[((size_t)yb * W + xb) * 4 + c];
		}
		else
		{
			t00 = t->b[((size_t)ya * W + xa) * 4 + c] * (1.0f / 255.0f); t10 = t->b[((size_t)ya * W + xb) * 4 + c] * (1.0f / 255.0f);
			t01 = t->b[((size_t)yb * W + xa) * 4 + c] * (1.0f / 255.0f); t11 = t->b[((size_t)yb * W + xb) * 4 + c] * (1.0f / 255.0f);
		}
		out[c] = (1.0f - ay) * ((1.0f - ax) * t00 + ax * t10) + ay * ((1.0f - ax) * t01 + ax * t11);
	}
}

/* ---- brdf.h / MonteCarlo.h ------------------------------------------------------------------------------- */
static inline float pow5(float v) { float v2 = v * v; return v2 * v2 * v; }                                   /* brdf.h:4-8 */
static inline float D_GGX(float NdotH, float a2) { float d = (NdotH * a2 - NdotH) * NdotH + 1.0f; return a2 / (PI_F * d * d); } /* brdf.h:11-15 */
static inline float V_SmithGGXCorrelated(float NdotV, float NdotL, float a2)                                  /* brdf.h:18-24 */
{
	float lv = NdotL * sqrtf((-NdotV * a2 + NdotV) * NdotV + a2);
	float ll = NdotV * sqrtf((-NdotL * a2 + NdotL) * NdotL + a2);
	return 0.5f / (lv + ll + 1e-5f);
}
static inline v3 F_Schlick(v3 F0, float VdotH)                                                                /* brdf.h:27-32 */
{
	float p = pow5(1.0f - VdotH);
	/* pow5Term + F0 * (1.0f - pow5Term): operator*(vec3,float) then operator+(float,vec3) = v + u */
	v3 a = vscale(1.0f - p, F0);
	return V(a.x + p, a.y + p, a.z + p);
}
static inline v3 Specular_GGX(v3 F0, float NdotV, float NdotL, float NdotH, float VdotH, float a2)            /* brdf.h:56-62 */
{
	float D = D_GGX(NdotH, a2);
	float Vis = V_SmithGGXCorrelated(NdotV, NdotL, a2);
	v3 F = F_Schlick(F0, VdotH);
	return vscale(D * Vis, F); /* D * V * F: (float*float)*vec3 */
}
static inline v3 tangentToWorld(v3 N, v3 v)                                                                   /* MonteCarlo.h:5-12 */
{
	v3 up = fabsf(N.z) < 0.999f ? V(0.0f, 0.0f, 1.0f) : V(1.0f, 0.0f, 0.0f);
	v3 tangent = vnorm(vcross(up, N));
	v3 bitangent = vcross(N, tangent);
	/* tangent * v.x = v.x * tangent (vec3.inl:131-134) */
	return vnorm(vadd(vadd(vscale(v.x, tangent), vscale(v.y, bitangent)), vscale(v.z, N)));
}
static inline v3 worldToTangent(v3 N, v3 v)                                                                   /* MonteCarlo.h:15-22 */
{
	v3 up = fabsf(N.z) < 0.999f ? V(0.0f, 0.0f, 1.0f) : V(1.0f, 0.0f, 0.0f);
	v3 tangent = vnorm(vcross(up, N));
	v3 bitangent = vcross(N, tangent);
	return vnorm(vadd(vadd(vscale(v.x, V(tangent.x, bitangent.x, N.x)), vscale(v.y, V(tangent.y, bitangent.y, N.y))), vscale(v.z, V(tangent.z, bitangent.z, N.z))));
}
static inline v3 cosineSampleHemisphere(float u0, float u1)                                                   /* MonteCarlo.h:24-30 */
{
	const float phi = 2.0f * PI_F * u0, cosTheta = sqrtf(u1), sinTheta = sqrtf(1.0f - u1);
	return V(cosf(phi) * sinTheta, sinf(phi) * sinTheta, cosTheta);
}
static inline v3 importanceSampleGGXVNDF(v3 Vv, float u0, float u1, float a)                                  /* MonteCarlo.h:73-101 */
{
	v3 Vh = vnorm(V(a * Vv.x, a * Vv.y, Vv.z));
	float lensq = Vh.x * Vh.x + Vh.y * Vh.y;
	v3 T1 = lensq > 0.0f ? vscale(1.0f / sqrtf(lensq), V(-Vh.y, Vh.x, 0.0f)) : V(1.0f, 0.0f, 0.0f);
	v3 T2 = vcross(Vh, T1);
	float r = sqrtf(u0), phi = 2.0f * PI_F * u1;
	float t1 = r * cosf(phi), t2 = r * sinf(phi);
	float s = 0.5f * (1.0f + Vh.z);
	t2 = (1.0f - s) * sqrtf(1.0f - t1 * t1) + s * t2;
	v3 Nh = vadd(vadd(vscale(t1, T1), vscale(t2, T2)), vscale(sqrtf(clampf(1.0f - t1 * t1 - t2 * t2, 0.0f, 1.0f)), Vh));
	return vnorm(V(a * Nh.x, a * Nh.y, clampf(Nh.z, 0.0f, 1.0f)));
}
static inline float importanceSampleGGXVNDFPdf(v3 H, v3 Vv, float a)                                          /* MonteCarlo.h:104-114 */
{
	float a2 = a * a, NdotH = H.z, VdotH = clampf(vdot(Vv, H), 0.0f, 1.0f);
	float G1 = (2.0f * Vv.z) / (Vv.z + sqrtf(a2 + (1.0f - a2) * (Vv.z * Vv.z)));
	float Dv = (G1 * VdotH * D_GGX(NdotH, a2)) / Vv.z;
	return Dv / (4.0f * VdotH);
}
static inline v3 lerp3(v3 x, v3 y, float a) { return vadd(vscale(1.0f - a, x), vscale(a, y)); }               /* vec3.inl:225-228 */

/* Material::sample  Material.inl:20-60 (+ sampleLambert :67-72, sampleGGX :74-99, sampleLambertGGX :101-144).
 * Returns attenuation; *pdf, *scatteredDir (world).  baseColor already texture-resolved by the caller. */
/* NOT THE REFERENCE (a helper of the "env_is" and "light_is" estimators): attenuation and pdf of Material::sample for a GIVEN tangent-space
 * direction - the same expressions as in materialSample below (Material.inl:67-72, :89-98, :124-143), which are functions of the
 * view vector and the scattered direction alone. */
static v3 materialEval(uint32_t mtype, v3 baseColor, float roughness, float metalness, v3 Vv, v3 sdir, float *pdf)
{
	v3 att = V(0.0f, 0.0f, 0.0f);
	*pdf = 0.0f;
	if (mtype == PT_LAMBERT) { *pdf = sdir.z / PI_F; att = vscale(1.0f / PI_F, baseColor); }
	else if (mtype == PT_GGX || mtype == PT_LAMBERT_GGX)
	{
		const float a = roughness * roughness, a2 = a * a;
		if (sdir.z < 0.0f) { *pdf = 1.0f; return att; }
		const float NdotV = fabsf(Vv.z) + 1e-5f;
		const v3 H = vnorm(vadd(Vv, sdir));
		const float VdotH = clampf(vdot(Vv, H), 0.0f, 1.0f), NdotH = clampf(H.z, 0.0f, 1.0f), NdotL = clampf(sdir.z, 0.0f, 1.0f);
		const v3 F0 = lerp3(V(0.04f, 0.04f, 0.04f), baseColor, metalness);
		const v3 kS = Specular_GGX(F0, NdotV, NdotL, NdotH, VdotH, a2);
		if (mtype == PT_GGX) { *pdf = importanceSampleGGXVNDFPdf(H, Vv, a); att = kS; }
		else
		{
			const float cosinePdf = sdir.z / PI_F, ggxPdf = importanceSampleGGXVNDFPdf(H, Vv, a);
			*pdf = (ggxPdf + cosinePdf) * 0.5f;
			att = vadd(vscale(1.0f - metalness, vscale(1.0f / PI_F, baseColor)), kS);
		}
	}
	return att;
}

static v3 materialSample(uint32_t mtype, v3 baseColor, float roughness, float metalness, v3 N, v3 inDir, float rnd0, float rnd1, v3 *scattered, float *pdf)
{
	const v3 Vv = worldToTangent(N, vneg(inDir));
	v3 sdir = V(0.0f, 0.0f, 0.0f), att = V(0.0f, 0.0f, 0.0f);
	*pdf = 0.0f; /* trace.cu:143 */
	if (mtype == PT_LAMBERT)
	{
		sdir = cosineSampleHemisphere(rnd0, rnd1);
		*pdf = sdir.z / PI_F;
		att = vscale(1.0f / PI_F, baseColor);
	}
	else if (mtype == PT_GGX || mtype == PT_LAMBERT_GGX)
	{
		const float a = roughness * roughness, a2 = a * a;
		if (mtype == PT_GGX) sdir = vreflect(vneg(Vv), importanceSampleGGXVNDF(Vv, rnd0, rnd1, a));
		else if (rnd0 < 0.5f) { rnd0 = 2.0f * rnd0; sdir = cosineSampleHemisphere(rnd0, rnd1); }
		else { rnd0 = 2.0f * (rnd0 - 0.5f); sdir = vreflect(vneg(Vv), importanceSampleGGXVNDF(Vv, rnd0, rnd1, a)); }
		if (sdir.z < 0.0f) { *pdf = 1.0f; att = V(0.0f, 0.0f, 0.0f); }
		else
		{
			const float NdotV = fabsf(Vv.z) + 1e-5f;
			const v3 H = vnorm(vadd(Vv, sdir));
			const float VdotH = clampf(vdot(Vv, H), 0.0f, 1.0f), NdotH = clampf(H.z, 0.0f, 1.0f), NdotL = clampf(sdir.z, 0.0f, 1.0f);
			const v3 F0 = lerp3(V(0.04f, 0.04f, 0.04f), baseColor, metalness);
			const v3 kS = Specular_GGX(F0, NdotV, NdotL, NdotH, VdotH, a2);
			if (mtype == PT_GGX) { *pdf = importanceSampleGGXVNDFPdf(H, Vv, a); att = kS; }
			else
			{
				const float cosinePdf = sdir.z / PI_F, ggxPdf = importanceSampleGGXVNDFPdf(H, Vv, a);
				*pdf = (ggxPdf + cosinePdf) * 0.5f;
				const v3 kD = vscale(1.0f / PI_F, baseColor);
				att = vadd(vscale(1.0f - metalness, kD), kS);
			}
		}
	}
	*scattered = vnorm(tangentToWorld(N, sdir));
	return att;
}

static v3 resolveBaseColor(const orc_scene *s, const obj_t *o, float u, float v)                              /* Material.inl:25-35 */
{
	v3 bc = o->baseColor;
	if (o->texture != 0 && o->texture <= s->texCount)
	{
		float tap[4];
		texLookup(&s->tex[o->texture - 1], u, v, tap);
		bc = V(powf(tap[0], 2.2f), powf(tap[1], 2.2f), powf(tap[2], 2.2f));
	}
	return bc;
}

/* ---- NOT THE REFERENCE: the sky's importance distribution (the product's option "env_is"; csrc/env_sampling.h states the
 * estimator).  Restated here so that the CUDA path can be checked path for path: a grid of at most 512 x 256 cells over the
 * equirectangular map, weight = sum over the cell's texels of luminance x sin(theta) plus a floor of 1e-4 of the mean, one alias
 * table over all cells (Vose, work lists filled in index order, used as stacks), density = P(cell) cells / (2 pi^2). ---- */
static void envBuild(orc_scene *s)
{
	free(s->envQ); free(s->envAlias); free(s->envDensity);
	s->envQ = NULL; s->envAlias = NULL; s->envDensity = NULL; s->envCols = s->envRows = 0;
	if (s->skybox == 0 || s->skybox > s->texCount) return;
	const tex_t *t = &s->tex[s->skybox - 1];
	const uint32_t bw = (t->w + 511u) / 512u, bh = (t->h + 255u) / 256u;
	const uint32_t cols = (t->w + bw - 1u) / bw, rows = (t->h + bh - 1u) / bh;
	const size_t n = (size_t)cols * rows;
	double *w = (double *)calloc(n, sizeof(double)), *scaled = (double *)malloc(n * sizeof(double));
	const double pi = 3.14159265358979323846;
	for (uint32_t y = 0; y < t->h; ++y)
	{
		const double sinTheta = sin(pi * ((double)y + 0.5) / (double)t->h);
		for (uint32_t x = 0; x < t->w; ++x)
		{
			const size_t k = ((size_t)y * t->w + x) * 4;
			double r, g, b;
			if (t->hdr) { r = t->f[k]; g = t->f[k + 1]; b = t->f[k + 2]; }
			else { r = t->b[k] / 255.0; g = t->b[k + 1] / 255.0; b = t->b[k + 2] / 255.0; }
			double lum = 0.2126 * r + 0.7152 * g + 0.0722 * b;
			if (!(lum > 0.0) || !(lum < 1e30)) lum = 0.0;
			w[(size_t)(y / bh) * cols + x / bw] += lum * sinTheta;
		}
	}
	double total = 0.0;
	for (size_t i = 0; i < n; ++i) total += w[i];
	if (!(total > 0.0)) { for (size_t i = 0; i < n; ++i) w[i] = 1.0; total = (double)n; }
	const double floorW = 1e-4 * total / (double)n;
	double total2 = 0.0;
	for (size_t i = 0; i < n; ++i) { w[i] += floorW; total2 += w[i]; }
	s->envQ = (float *)malloc(n * sizeof(float)); s->envAlias = (uint32_t *)malloc(n * sizeof(uint32_t)); s->envDensity = (float *)malloc(n * sizeof(float));
	for (size_t i = 0; i < n; ++i)
	{
		const double p = w[i] / total2;
		s->envDensity[i] = (float)(p * (double)n / (2.0 * pi * pi));
		scaled[i] = p * (double)n;
	}
	uint32_t *small = (uint32_t *)malloc(n * sizeof(uint32_t)), *large = (uint32_t *)malloc(n * sizeof(uint32_t));
	size_t ns = 0, nl = 0;
	for (size_t i = 0; i < n; ++i) { if (scaled[i] < 1.0) small[ns++] = (uint32_t)i; else large[nl++] = (uint32_t)i; }
#define ENV_PUT(cell, q, other) do { double q_ = (q); s->envQ[cell] = (float)(q_ < 0.0 ? 0.0 : (q_ > 1.0 ? 1.0 : q_)); s->envAlias[cell] = (other); } while (0)
	while (ns > 0 && nl > 0)
	{
		const uint32_t sm = small[--ns], lg = large[nl - 1];
		ENV_PUT(sm, scaled[sm], lg);
		scaled[lg] = (scaled[lg] + scaled[sm]) - 1.0;
		if (scaled[lg] < 1.0) { --nl; small[ns++] = lg; }
	}
	for (size_t i = 0; i < nl; ++i) ENV_PUT(large[i], 1.0, large[i]);
	for (size_t i = 0; i < ns; ++i) ENV_PUT(small[i], 1.0, small[i]);
#undef ENV_PUT
	free(small); free(large); free(w); free(scaled);
	s->envCols = cols; s->envRows = rows;
}
/* one direction ~ the distribution from three random words (cell by the alias table with integer arithmetic, position inside the
 * cell from the other two), its lookup coordinates and solid-angle pdf */
static v3 envSample(const orc_scene *s, uint32_t r0, uint32_t r1, uint32_t r2, float *u, float *v, float *pdf)
{
	const uint32_t cells = s->envCols * s->envRows;
	const uint64_t x = (uint64_t)r0 * cells;
	const uint32_t i = (uint32_t)(x >> 32);
	const float frac = (float)(uint32_t)x * 2.3283064365386963e-10f;
	const uint32_t cell = frac < s->envQ[i] ? i : s->envAlias[i];
	const uint32_t row = cell / s->envCols, col = cell - row * s->envCols;
	*u = ((float)col + orc_uniform(r1)) * (1.0f / (float)s->envCols);
	*v = ((float)row + orc_uniform(r2)) * (1.0f / (float)s->envRows);
	const float phi = 2.0f * PI_F * *u, theta = PI_F * *v;
	const float st = sinf(theta), ct = cosf(theta);
	*pdf = s->envDensity[cell] * (1.0f / fmaxf(st, 1e-6f));
	return V(st * cosf(phi), ct, st * sinf(phi));
}
static float envPdf(const orc_scene *s, float u, float v, float dirY)
{
	const float uw = u - floorf(u);
	uint32_t col = (uint32_t)(uw * (float)s->envCols), row = (uint32_t)(fmaxf(v, 0.0f) * (float)s->envRows);
	if (col > s->envCols - 1u) col = s->envCols - 1u;
	if (row > s->envRows - 1u) row = s->envRows - 1u;
	return s->envDensity[row * s->envCols + col] * (1.0f / sqrtf(fmaxf(1.0f - dirY * dirY, 1e-12f)));
}

/* ---- NOT THE REFERENCE: the emitters' importance distribution (the product's option "light_is"; csrc/light_sampling.h states the
 * estimator).  Restated here so that the CUDA path can be checked path for path: one alias table over the objects with a non-zero
 * emissive channel, weight = mean emission x world area (the same double arithmetic as the product; Vose, work lists filled in index
 * order, used as stacks), a uniform point on the chosen emitter's surface with its solid-angle pdf, and a shadow ray through the BVH
 * that stops just short of the point. ---- */
static double lightLocalArea(uint32_t type)
{
	const double pi = 3.14159265358979323846;
	switch (type)
	{
	case PT_SPHERE: return 4.0 * pi;
	case PT_CYLINDER: return 4.0 * pi;
	case PT_DISK: return pi;
	case PT_CONE: return 2.0 * sqrt(2.0) * pi;
	case PT_PARABOLOID: return pi * (5.0 * sqrt(5.0) - 1.0) / 6.0;
	case PT_QUAD: return 4.0;
	default: return 24.0;
	}
}
static void lightBuild(orc_scene *s)
{
	s->lightOf = (int32_t *)malloc((s->n ? s->n : 1) * sizeof(int32_t));
	uint32_t n = 0;
	for (size_t i = 0; i < s->n; ++i)
	{
		const obj_t *o = &s->sceneObjs[i];
		s->lightOf[i] = (o->emissive.x != 0.0f || o->emissive.y != 0.0f || o->emissive.z != 0.0f) ? (int32_t)n++ : -1;
	}
	s->lights = (light_t *)calloc(n ? n : 1, sizeof(light_t));
	double *w = (double *)calloc(n ? n : 1, sizeof(double)), *det = (double *)calloc(n ? n : 1, sizeof(double)), *scaled = (double *)calloc(n ? n : 1, sizeof(double));
	double total = 0.0;
	for (size_t i = 0; i < s->n; ++i)
	{
		if (s->lightOf[i] < 0) continue;
		const uint32_t k = (uint32_t)s->lightOf[i];
		const obj_t *o = &s->sceneObjs[i];
		light_t *L = &s->lights[k];
		L->scene = (uint32_t)i;
		L->type = o->type <= PT_CUBE ? o->type : PT_SPHERE;
		const float *rows[3] = { o->r0, o->r1, o->r2 };
		double W[3][3], tr[3];
		for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) W[r][c] = rows[r][c]; tr[r] = rows[r][3]; }
		const double dW = W[0][0] * (W[1][1] * W[2][2] - W[1][2] * W[2][1]) - W[0][1] * (W[1][0] * W[2][2] - W[1][2] * W[2][0]) +
		                  W[0][2] * (W[1][0] * W[2][1] - W[1][1] * W[2][0]);
		if (!(isfinite(dW) && dW != 0.0)) continue;
		double M[3][3];
		M[0][0] = (W[1][1] * W[2][2] - W[1][2] * W[2][1]) / dW;
		M[0][1] = (W[0][2] * W[2][1] - W[0][1] * W[2][2]) / dW;
		M[0][2] = (W[0][1] * W[1][2] - W[0][2] * W[1][1]) / dW;
		M[1][0] = (W[1][2] * W[2][0] - W[1][0] * W[2][2]) / dW;
		M[1][1] = (W[0][0] * W[2][2] - W[0][2] * W[2][0]) / dW;
		M[1][2] = (W[0][2] * W[1][0] - W[0][0] * W[1][2]) / dW;
		M[2][0] = (W[1][0] * W[2][1] - W[1][1] * W[2][0]) / dW;
		M[2][1] = (W[0][1] * W[2][0] - W[0][0] * W[2][1]) / dW;
		M[2][2] = (W[0][0] * W[1][1] - W[0][1] * W[1][0]) / dW;
		for (int r = 0; r < 3; ++r)
		{
			for (int c = 0; c < 3; ++c) L->m[4 * r + c] = (float)M[r][c];
			L->m[4 * r + 3] = (float)(-(M[r][0] * tr[0] + M[r][1] * tr[1] + M[r][2] * tr[2]));
		}
		const double dM = fabs(1.0 / dW);
		double len[3];
		for (int r = 0; r < 3; ++r) len[r] = sqrt(W[r][0] * W[r][0] + W[r][1] * W[r][1] + W[r][2] * W[r][2]);
		double area;
		if (L->type == PT_QUAD || L->type == PT_DISK) area = lightLocalArea(L->type) * dM * len[1];
		else if (L->type == PT_CUBE) area = 8.0 * dM * (len[0] + len[1] + len[2]);
		else area = lightLocalArea(L->type) * cbrt(dM * dM);
		const double mean = ((double)o->emissive.x + (double)o->emissive.y + (double)o->emissive.z) / 3.0;
		w[k] = mean > 0.0 && isfinite(area) ? mean * area : 0.0;
		det[k] = dM;
		total += w[k];
	}
	if (!(total > 0.0 && isfinite(total))) n = 0;
	s->lightCount = n;
	for (uint32_t k = 0; k < n; ++k)
	{
		const double P = w[k] / total;
		s->lights[k].pdfScale = P > 0.0 ? (float)(P / (lightLocalArea(s->lights[k].type) * det[k])) : 0.0f;
		s->lights[k].prob = (float)P;
		scaled[k] = P * (double)n;
	}
	uint32_t *small = (uint32_t *)malloc((n ? n : 1) * sizeof(uint32_t)), *large = (uint32_t *)malloc((n ? n : 1) * sizeof(uint32_t));
	size_t ns = 0, nl = 0;
	for (uint32_t i = 0; i < n; ++i) { if (scaled[i] < 1.0) small[ns++] = i; else large[nl++] = i; }
#define LIGHT_PUT(i, qq, other) do { double q_ = (qq); s->lights[i].q = (float)(q_ < 0.0 ? 0.0 : (q_ > 1.0 ? 1.0 : q_)); s->lights[i].alias = (other); } while (0)
	while (ns > 0 && nl > 0)
	{
		const uint32_t sm = small[--ns], lg = large[nl - 1];
		LIGHT_PUT(sm, scaled[sm], lg);
		scaled[lg] = (scaled[lg] + scaled[sm]) - 1.0;
		if (scaled[lg] < 1.0) { --nl; small[ns++] = lg; }
	}
	for (size_t i = 0; i < nl; ++i) LIGHT_PUT(large[i], 1.0, large[i]);
	for (size_t i = 0; i < ns; ++i) LIGHT_PUT(small[i], 1.0, small[i]);
#undef LIGHT_PUT
	free(small); free(large); free(w); free(det); free(scaled);
}
static v3 lightUnitNormal(uint32_t type, v3 lp)
{
	v3 n;
	switch (type)
	{
	case PT_SPHERE: n = lp; break;
	case PT_CYLINDER: n = V(lp.x, 0.0f, lp.z); break;
	case PT_CONE: n = V(lp.x, -lp.y, lp.z); break;
	case PT_PARABOLOID: n = V(2.0f * lp.x, -1.0f, 2.0f * lp.z); break;
	case PT_CUBE:
	{
		const float ax = fabsf(lp.x), ay = fabsf(lp.y), az = fabsf(lp.z);
		if (ax > ay && ax > az) n = V(1.0f, 0.0f, 0.0f);
		else if (ay > ax && ay > az) n = V(0.0f, 1.0f, 0.0f);
		else n = V(0.0f, 0.0f, 1.0f);
		break;
	}
	default: n = V(0.0f, 1.0f, 0.0f); break;
	}
	return vnorm(n);
}
/* W^T n_l: the (unnormalised) world normal */
static v3 lightWorldNormal(const obj_t *o, v3 nl)
{
	return V(nl.x * o->r0[0] + nl.y * o->r1[0] + nl.z * o->r2[0], nl.x * o->r0[1] + nl.y * o->r1[1] + nl.z * o->r2[1], nl.x * o->r0[2] + nl.y * o->r1[2] + nl.z * o->r2[2]);
}
/* local point of the canonical surface from two uniforms and one word (face / nappe) */
static v3 lightLocalPoint(uint32_t type, float u, float v, uint32_t w)
{
	const float ph = 2.0f * PI_F * v, cp = cosf(ph), sp = sinf(ph);
	switch (type)
	{
	case PT_SPHERE: { const float y = 1.0f - 2.0f * u, r = sqrtf(fmaxf(1.0f - y * y, 0.0f)); return V(r * cp, y, r * sp); }
	case PT_CYLINDER: return V(cp, 2.0f * u - 1.0f, sp);
	case PT_DISK: { const float r = sqrtf(u); return V(r * cp, 0.0f, r * sp); }
	case PT_CONE: { const float h = sqrtf(u); return V(h * cp, (w & 1u) ? h : -h, h * sp); }
	case PT_PARABOLOID:
	{
		const float g = cbrtf(1.0f + u * 10.180339887498949f);
		const float r2 = fmaxf((g * g - 1.0f) * 0.25f, 0.0f), r = sqrtf(r2);
		return V(r * cp, r2, r * sp);
	}
	case PT_QUAD: return V(2.0f * u - 1.0f, 0.0f, 2.0f * v - 1.0f);
	default:
	{
		const uint32_t face = (uint32_t)(((uint64_t)w * 6u) >> 32);
		const float s = (face & 1u) ? 1.0f : -1.0f, a = 2.0f * u - 1.0f, b = 2.0f * v - 1.0f;
		return face < 2u ? V(s, a, b) : (face < 4u ? V(a, s, b) : V(a, b, s));
	}
	}
}
/* one light sample from the four words q seen from p: emitter k, world point x, unit direction, distance, solid-angle pdf; 0 = unusable */
static int lightSample(const orc_scene *s, const uint32_t q[4], v3 p, uint32_t *k, v3 *x, v3 *wdir, float *dist, float *pdf)
{
	const uint64_t xx = (uint64_t)q[0] * s->lightCount;
	const uint32_t i = (uint32_t)(xx >> 32);
	const float frac = (float)(uint32_t)xx * 2.3283064365386963e-10f;
	*k = frac < s->lights[i].q ? i : s->lights[i].alias;
	const light_t *L = &s->lights[*k];
	const v3 lp = lightLocalPoint(L->type, orc_uniform(q[1]), orc_uniform(q[2]), q[3]);
	*x = V(L->m[0] * lp.x + L->m[1] * lp.y + L->m[2] * lp.z + L->m[3], L->m[4] * lp.x + L->m[5] * lp.y + L->m[6] * lp.z + L->m[7],
	       L->m[8] * lp.x + L->m[9] * lp.y + L->m[10] * lp.z + L->m[11]);
	const v3 dv = vsub(*x, p);
	const float d2 = vdot(dv, dv);
	*dist = sqrtf(d2);
	*wdir = vscale(1.0f / *dist, dv);
	const v3 wn = lightWorldNormal(&s->sceneObjs[L->scene], lightUnitNormal(L->type, lp));
	*pdf = L->pdfScale * d2 / fmaxf(fabsf(vdot(wn, *wdir)), 1e-30f);
	return d2 > 0.0f && *pdf > 0.0f && *pdf < 3.0e38f;
}
/* solid-angle pdf of the light sampler for a BSDF-sampled ray that hit emitter L (object o) at t */
static float lightPdf(const light_t *L, const obj_t *o, ray_t ray, float t)
{
	v3 lo;
	lo.x = vdot(ray.o, V(o->r0[0], o->r0[1], o->r0[2])) + o->r0[3];
	lo.y = vdot(ray.o, V(o->r1[0], o->r1[1], o->r1[2])) + o->r1[3];
	lo.z = vdot(ray.o, V(o->r2[0], o->r2[1], o->r2[2])) + o->r2[3];
	const v3 ld = V(vdot(ray.d, V(o->r0[0], o->r0[1], o->r0[2])), vdot(ray.d, V(o->r1[0], o->r1[1], o->r1[2])), vdot(ray.d, V(o->r2[0], o->r2[1], o->r2[2])));
	const v3 lp = vadd(lo, vscale(t, ld));
	const v3 wn = lightWorldNormal(o, lightUnitNormal(L->type, lp));
	return L->pdfScale * t * t / fmaxf(fabsf(vdot(wn, ray.d)), 1e-30f);
}
/* the shadow ray of a light sample: any primitive hit in (tMin, tMax] */
static int occludedBVH(const orc_scene *s, ray_t r, float tMin, float tMax)
{
	uint32_t stack[64], sp = 0, cur = 0;
	if (s->nodeCount == 0) return 0;
	v3 inv;
	inv.x = 1.0f / (r.d.x != 0.0f ? r.d.x : 1e-7f);
	inv.y = 1.0f / (r.d.y != 0.0f ? r.d.y : 1e-7f);
	inv.z = 1.0f / (r.d.z != 0.0f ? r.d.z : 1e-7f);
	int neg[3] = { inv.x < 0.0f, inv.y < 0.0f, inv.z < 0.0f };
	for (;;)
	{
		const node_t *node = &s->nodes[cur];
		if (aabbSlab(node->box, r, tMin, tMax, NULL))
		{
			const uint32_t pc = node->countAxis >> 16;
			if (pc > 0)
			{
				for (uint32_t i = 0; i < pc; ++i)
				{
					hit_t rec;
					if (hitObject(&s->objs[node->offset + i], r, tMin, tMax, &rec) && rec.t <= tMax) return 1;
				}
				if (sp == 0) break;
				cur = stack[--sp];
			}
			else
			{
				int isNeg = neg[(node->countAxis >> 8) & 0xFF];
				stack[sp++] = isNeg ? (cur + 1) : node->offset;
				cur = isNeg ? node->offset : (cur + 1);
			}
		}
		else
		{
			if (sp == 0) break;
			cur = stack[--sp];
		}
	}
	return 0;
}

/* getColor  kernels/trace.cu:101-156 */
static v3 getColor(const orc_scene *s, ray_t ray, uint32_t pixel, uint32_t sample, uint32_t k0, uint32_t k1, const uint32_t rng0[4], int maxBounces, uint64_t *rays)
{
	v3 throughput = V(1.0f, 1.0f, 1.0f), L = V(0.0f, 0.0f, 0.0f);
	float lastPdf = 0.0f;
	uint32_t rng[4] = { rng0[0], rng0[1], rng0[2], rng0[3] };
	for (int it = 0; it < maxBounces; ++it)
	{
		hit_t rec; uint32_t elem;
		++*rays;
		if (!hitBVH(s, ray, 0.001f, FLT_MAX, &rec, &elem, NULL, NULL))
		{
			v3 c = V(0.0f, 0.0f, 0.0f);
			if (s->skybox != 0 && s->skybox <= s->texCount)
			{
				float theta = acosf(ray.d.y), phi = atan2f(ray.d.z, ray.d.x);
				float v = theta / PI_F, u = phi / (2.0f * PI_F), tap[4];
				texLookup(&s->tex[s->skybox - 1], u, v, tap);
				c = V(tap[0], tap[1], tap[2]);
			}
			if (s->envIS && it > 0 && s->skybox != 0 && s->skybox <= s->texCount)
			{
				/* NOT THE REFERENCE: balance-heuristic weight of a BSDF-sampled direction that reached the sky */
				const float theta = acosf(ray.d.y), phi = atan2f(ray.d.z, ray.d.x);
				const float pe = envPdf(s, phi / (2.0f * PI_F), theta / PI_F, ray.d.y);
				c = vscale(lastPdf / (lastPdf + pe), c);
			}
			L = vadd(L, vmul(throughput, c));
			break;
		}
		const obj_t *o = &s->objs[elem];
		v3 em = o->emissive;
		const int32_t ek = s->lightCount ? s->lightOf[s->toScene[elem]] : -1;
		if (it > 0 && ek >= 0) /* NOT THE REFERENCE: balance-heuristic weight of a BSDF-sampled direction that hit an emitter */
			em = vscale(lastPdf / (lastPdf + lightPdf(&s->lights[ek], o, ray, rec.t)), em);
		L = vadd(L, vmul(throughput, em));
		/* uniforms: slot 0 = (jitter x, jitter y, bounce0 r0, bounce0 r1); slot k>=1 = (bounce 2k-1 r0 r1, bounce 2k r0 r1) */
		float rnd0, rnd1;
		if (it == 0) { rnd0 = orc_uniform(rng[2]); rnd1 = orc_uniform(rng[3]); }
		else
		{
			if (it & 1) orc_philox(pixel, sample, (uint32_t)(it + 1) / 2, 0, k0, k1, rng);
			rnd0 = orc_uniform(rng[(it & 1) ? 0 : 2]); rnd1 = orc_uniform(rng[(it & 1) ? 1 : 3]);
		}
		v3 sdir; float pdf;
		const v3 base = resolveBaseColor(s, o, rec.u, rec.v);
		if (s->envIS && s->skybox != 0 && s->skybox <= s->texCount && it + 1 < maxBounces)
		{
			/* NOT THE REFERENCE: one direction from the sky's distribution per scattering vertex (Philox counter word 3 = 1,
			 * slot = bounce), weighted against the BSDF's pdf for the same direction; shadow ray with the path's own tMin */
			uint32_t q[4];
			orc_philox(pixel, sample, (uint32_t)it, 1, k0, k1, q);
			float lu, lv, pe;
			const v3 wl = envSample(s, q[0], q[1], q[2], &lu, &lv, &pe);
			const v3 Vv = worldToTangent(rec.n, vneg(ray.d)), sl = worldToTangent(rec.n, wl);
			float pbL;
			const v3 attL = materialEval(o->mtype, base, o->roughness, o->metalness, Vv, sl, &pbL);
			if (sl.z > 0.0f && !((attL.x == 0.0f && attL.y == 0.0f && attL.z == 0.0f) || pbL == 0.0f))
			{
				float tap[4];
				texLookup(&s->tex[s->skybox - 1], lu, lv, tap);
				ray_t sh; sh.o = rec.p; sh.d = wl;
				hit_t srec; uint32_t selem;
				++*rays;
				if (!hitBVH(s, sh, 0.001f, FLT_MAX, &srec, &selem, NULL, NULL))
					L = vadd(L, vmul(vmul(throughput, vscale(sl.z / (pe + pbL), attL)), V(tap[0], tap[1], tap[2])));
			}
		}
		if (s->lightCount && it + 1 < maxBounces)
		{
			/* NOT THE REFERENCE: one point on an emitter per scattering vertex (Philox counter word 3 = 2, slot = bounce), weighted
			 * against the BSDF's pdf for the same direction; the shadow ray stops just short of the point */
			uint32_t q[4], k; v3 x, wl; float dist, pl;
			orc_philox(pixel, sample, (uint32_t)it, 2, k0, k1, q);
			if (lightSample(s, q, rec.p, &k, &x, &wl, &dist, &pl))
			{
				const v3 Vv = worldToTangent(rec.n, vneg(ray.d)), sl = worldToTangent(rec.n, wl);
				float pbL;
				const v3 attL = materialEval(o->mtype, base, o->roughness, o->metalness, Vv, sl, &pbL);
				if (sl.z > 0.0f && !((attL.x == 0.0f && attL.y == 0.0f && attL.z == 0.0f) || pbL == 0.0f))
				{
					ray_t sh; sh.o = rec.p; sh.d = wl;
					++*rays;
					if (!occludedBVH(s, sh, 0.001f, dist * (1.0f - 1e-4f)))
						L = vadd(L, vmul(vmul(throughput, vscale(sl.z / (pl + pbL), attL)), s->sceneObjs[s->lights[k].scene].emissive));
				}
			}
		}
		v3 att = materialSample(o->mtype, base, o->roughness, o->metalness, rec.n, ray.d, rnd0, rnd1, &sdir, &pdf);
		lastPdf = pdf;
		if ((att.x == 0.0f && att.y == 0.0f && att.z == 0.0f) || pdf == 0.0f) break;
		/* throughput *= attenuation * abs(dot(scattered.m_dir, rec.m_normal)) / pdf   (trace.cu:150):
		 * (att * |dot|) / pdf = (1/pdf) * (|dot| * att) */
		v3 w = vdivf(vscale(fabsf(vdot(sdir, rec.n)), att), pdf);
		throughput = vmul(throughput, w);
		ray.o = rec.p; ray.d = sdir;
	}
	return L;
}

/* ---- public ---------------------------------------------------------------------------------------------- */
orc_scene *orc_scene_create(size_t count, const pt_object_desc *objects)
{
	orc_scene *s = (orc_scene *)calloc(1, sizeof *s);
	s->n = count;
	if (count == 0) return s;
	bobj_t *e = (bobj_t *)malloc(count * sizeof *e);
	s->sceneObjs = (obj_t *)malloc(count * sizeof(obj_t));
	for (size_t i = 0; i < count; ++i) { makeObject(&objects[i], &e[i].o); e[i].scene = (int32_t)i; s->sceneObjs[i] = e[i].o; }
	s->nodeCap = (uint32_t)(2 * count);
	s->nodes = (node_t *)malloc(s->nodeCap * sizeof(node_t));
	buildRecursive(s, e, 0, count, 4); /* Pathtracer.cpp:121 */
	s->objs = (obj_t *)malloc(count * sizeof(obj_t));
	s->toScene = (int32_t *)malloc(count * sizeof(int32_t));
	for (size_t i = 0; i < count; ++i) { s->objs[i] = e[i].o; s->toScene[i] = e[i].scene; }
	free(e);
	return s;
}
void orc_scene_destroy(orc_scene *s)
{
	if (!s) return;
	for (uint32_t i = 0; i < s->texCount; ++i) { free(s->tex[i].f); free(s->tex[i].b); }
	free(s->envQ); free(s->envAlias); free(s->envDensity);
	free(s->lights); free(s->lightOf);
	free(s->objs); free(s->toScene); free(s->sceneObjs); free(s->nodes); free(s);
}
uint32_t orc_add_texture(orc_scene *s, uint32_t w, uint32_t h, int is_hdr, const void *rgba)
{
	if (s->texCount >= 64) return 0;
	tex_t *t = &s->tex[s->texCount];
	t->w = w; t->h = h; t->hdr = is_hdr; t->f = NULL; t->b = NULL;
	size_t bytes = (size_t)w * h * 4 * (is_hdr ? 4 : 1);
	void *p = malloc(bytes); memcpy(p, rgba, bytes);
	if (is_hdr) t->f = (float *)p; else t->b = (uint8_t *)p;
	return ++s->texCount;
}
void orc_set_skybox(orc_scene *s, uint32_t handle) { s->skybox = handle; if (s->envIS) envBuild(s); }
/* NOT THE REFERENCE: switch the "env_is" estimator on / off (builds the distribution of the current sky) */
void orc_set_env_is(orc_scene *s, int on) { s->envIS = on != 0; if (s->envIS) envBuild(s); }
/* the tables, for tests: returns the cell count (0 = none); q / alias / density may be NULL */
uint32_t orc_env_tables(const orc_scene *s, uint32_t *cols, uint32_t *rows, float *q, uint32_t *alias, float *density)
{
	const uint32_t n = s->envCols * s->envRows;
	if (cols) *cols = s->envCols;
	if (rows) *rows = s->envRows;
	if (n && q) memcpy(q, s->envQ, n * sizeof(float));
	if (n && alias) memcpy(alias, s->envAlias, n * sizeof(uint32_t));
	if (n && density) memcpy(density, s->envDensity, n * sizeof(float));
	return n;
}
/* one sample of the distribution (tests): out6 = direction, u, v, pdf */
void orc_env_sample(const orc_scene *s, uint32_t r0, uint32_t r1, uint32_t r2, float *out6)
{
	float u, v, pdf;
	const v3 d = envSample(s, r0, r1, r2, &u, &v, &pdf);
	out6[0] = d.x; out6[1] = d.y; out6[2] = d.z; out6[3] = u; out6[4] = v; out6[5] = pdf;
}
/* NOT THE REFERENCE: switch the "light_is" estimator on (builds the emitter table of the scene) / off (drops it) */
void orc_set_light_is(orc_scene *s, int on)
{
	free(s->lights); free(s->lightOf);
	s->lights = NULL; s->lightOf = NULL; s->lightCount = 0;
	if (on) lightBuild(s);
}
/* the table, for tests: returns the emitter count; scene / prob / q / alias may be NULL */
uint32_t orc_light_table(const orc_scene *s, uint32_t *scene, float *prob, float *q, uint32_t *alias)
{
	for (uint32_t k = 0; k < s->lightCount; ++k)
	{
		if (scene) scene[k] = s->lights[k].scene;
		if (prob) prob[k] = s->lights[k].prob;
		if (q) q[k] = s->lights[k].q;
		if (alias) alias[k] = s->lights[k].alias;
	}
	return s->lightCount;
}
/* one sample of the emitter sampler (tests): out8 = world point, area pdf without the selection probability
 * (pdfScale / P_sel / |W^T n_l|), emitter, local point */
void orc_light_sample_point(const orc_scene *s, const uint32_t *q, float *out8)
{
	uint32_t k; v3 x, wd; float dist, pdf;
	lightSample(s, q, V(0.0f, 0.0f, 0.0f), &k, &x, &wd, &dist, &pdf);
	const light_t *L = &s->lights[k];
	const v3 lp = lightLocalPoint(L->type, orc_uniform(q[1]), orc_uniform(q[2]), q[3]);
	const v3 wn = lightWorldNormal(&s->sceneObjs[L->scene], lightUnitNormal(L->type, lp));
	out8[0] = x.x; out8[1] = x.y; out8[2] = x.z;
	out8[3] = (float)((double)L->pdfScale / (double)L->prob / sqrt((double)wn.x * wn.x + (double)wn.y * wn.y + (double)wn.z * wn.z));
	out8[4] = (float)k; out8[5] = lp.x; out8[6] = lp.y; out8[7] = lp.z;
}
void orc_bvh_info(const orc_scene *s, uint32_t *nodes, uint32_t *depth, int32_t *valid)
{
	*nodes = s->nodeCount; *depth = s->nodeCount ? bvhDepth(s, 0) : 0;
	/* BVH::validate (BVH.cpp:36-52,230-255): every primitive in exactly one leaf */
	uint8_t *seen = (uint8_t *)calloc(s->n ? s->n : 1, 1); int ok = 1;
	for (uint32_t i = 0; i < s->nodeCount; ++i)
	{
		uint32_t pc = s->nodes[i].countAxis >> 16;
		for (uint32_t k = 0; k < pc; ++k) { if (seen[s->nodes[i].offset + k]) ok = 0; seen[s->nodes[i].offset + k] = 1; }
	}
	for (size_t i = 0; i < s->n; ++i) if (!seen[i]) ok = 0;
	free(seen); *valid = ok;
}
void orc_object_info(const orc_scene *s, size_t i, float *rows12, float *aabb6)
{
	const obj_t *o = &s->sceneObjs[i];
	memcpy(rows12, o->r0, 16); memcpy(rows12 + 4, o->r1, 16); memcpy(rows12 + 8, o->r2, 16);
	aabb6[0] = o->box.mn.x; aabb6[1] = o->box.mn.y; aabb6[2] = o->box.mn.z; aabb6[3] = o->box.mx.x; aabb6[4] = o->box.mx.y; aabb6[5] = o->box.mx.z;
}
void orc_camera_ray(const pt_camera_desc *cam, float s, float t, float *out6)
{
	cam_t k = makeCamera(cam); ray_t r = cameraRay(&k, s, t);
	out6[0] = r.o.x; out6[1] = r.o.y; out6[2] = r.o.z; out6[3] = r.d.x; out6[4] = r.d.y; out6[5] = r.d.z;
}
int orc_hit_object(const orc_scene *s, size_t i, const float *o, const float *d, float tmin, float tmax, float *out10)
{
	ray_t r; r.o = V(o[0], o[1], o[2]); r.d = V(d[0], d[1], d[2]);
	hit_t rec;
	if (!hitObject(&s->sceneObjs[i], r, tmin, tmax, &rec)) return 0;
	out10[0] = rec.t; out10[1] = rec.p.x; out10[2] = rec.p.y; out10[3] = rec.p.z; out10[4] = rec.n.x; out10[5] = rec.n.y; out10[6] = rec.n.z;
	out10[7] = rec.u; out10[8] = rec.v; out10[9] = rec.front ? 1.0f : 0.0f;
	return 1;
}
/* How far a ray is from the nearest accept / reject DECISION of one object's intersection routine (Hittable.inl:147-358),
 * in units of the rounding noise of the float32 evaluation.  Test infrastructure for the first-hit gate: two float32
 * implementations of the same formulas (the reference's GPU build, ours with MUFU reciprocals) may only disagree about an
 * object where this is small.  Computed in double precision from the object's world->local rows:
 *   quadrics : tangency |disc| against the magnitude of its two terms b*b and 4*a*c (far from an object the local origin is
 *              ~10^3 units away and the float32 discriminant has lost ~7 digits), and for the open quadrics the height test
 *              |y| <= 1 at both roots against the magnitude of the terms of y = o.y + t * d.y
 *   disk/quad: the edge tests at the plane hit against the magnitude of o + t * d;   cube: the slab interval's length
 * Returns min over the decisions of |quantity - threshold| / (2^-23 * magnitude of the terms): < ~100 means "within float32
 * rounding of flipping".  Also tMin / tMax are ignored (closest-hit competition between objects is judged by t). */
double orc_decision_margin(const orc_scene *s, size_t i, const float *of, const float *df)
{
	const obj_t *ob = &s->sceneObjs[i];
	const double eps = 1.1920929e-7;
	double o[3], d[3], mo[3], md[3]; /* local origin / direction, and the magnitude of the terms that formed them */
	const float *rows[3] = { ob->r0, ob->r1, ob->r2 };
	for (int k = 0; k < 3; ++k)
	{
		const float *r = rows[k];
		o[k] = (double)r[0] * of[0] + (double)r[1] * of[1] + (double)r[2] * of[2] + (double)r[3];
		d[k] = (double)r[0] * df[0] + (double)r[1] * df[1] + (double)r[2] * df[2];
		mo[k] = fabs((double)r[0] * of[0]) + fabs((double)r[1] * of[1]) + fabs((double)r[2] * of[2]) + fabs((double)r[3]);
		md[k] = fabs((double)r[0] * df[0]) + fabs((double)r[1] * df[1]) + fabs((double)r[2] * df[2]);
	}
	double best = 1e300;
#define MARGIN(q, mag) do { const double m_ = fabs(q) / (eps * ((mag) + 1e-300)); if (m_ < best) best = m_; } while (0)
	const uint32_t type = ob->type;
	if (type == PT_DISK || type == PT_QUAD)
	{
		if (d[1] == 0.0) return 0.0;
		const double t = -o[1] / d[1];
		const double hx = o[0] + d[0] * t, hz = o[2] + d[2] * t;
		const double mx = mo[0] + fabs(d[0] * t) + md[0] * fabs(t), mz = mo[2] + fabs(d[2] * t) + md[2] * fabs(t);
		if (type == PT_DISK) MARGIN(hx * hx + hz * hz - 1.0, 2.0 * (fabs(hx) * mx + fabs(hz) * mz) + 1.0);
		else { MARGIN(fabs(hx) - 1.0, mx + 1.0); MARGIN(fabs(hz) - 1.0, mz + 1.0); }
		MARGIN(t, fabs(t)); /* t == 0 never decides anything here; keeps best finite */
		return best < 1e299 ? best : 1e299;
	}
	if (type == PT_CUBE)
	{
		double tn = -1e300, tf = 1e300, mag = 0.0;
		for (int k = 0; k < 3; ++k)
		{
			if (d[k] == 0.0) continue;
			double t0 = (-1.0 - o[k]) / d[k], t1 = (1.0 - o[k]) / d[k];
			if (t0 > t1) { const double x = t0; t0 = t1; t1 = x; }
			if (t0 > tn) tn = t0;
			if (t1 < tf) tf = t1;
			const double m = (mo[k] + 1.0) / fabs(d[k]) + fabs(t1) * md[k] / fabs(d[k]);
			if (m > mag) mag = m;
		}
		MARGIN(tf - tn, mag);
		return best;
	}
	const double B = type == PT_SPHERE ? 1.0 : (type == PT_CONE ? -1.0 : 0.0), Hc = type == PT_PARABOLOID ? -1.0 : 0.0;
	const double J = (type == PT_SPHERE || type == PT_CYLINDER) ? -1.0 : 0.0;
	const double a = d[0] * d[0] + B * d[1] * d[1] + d[2] * d[2];
	const double b = 2.0 * (o[0] * d[0] + B * o[1] * d[1] + o[2] * d[2]) + Hc * d[1];
	const double c = o[0] * o[0] + B * o[1] * o[1] + o[2] * o[2] + Hc * o[1] + J;
	/* magnitudes of the float32 evaluations of b and c (their own terms cancel, then b*b - 4ac cancels again) */
	const double mb = 2.0 * (fabs(o[0] * d[0]) + fabs(o[1] * d[1]) + fabs(o[2] * d[2])) + 2.0 * (mo[0] * fabs(d[0]) + mo[1] * fabs(d[1]) + mo[2] * fabs(d[2]));
	const double mc = o[0] * o[0] + o[1] * o[1] + o[2] * o[2] + 2.0 * (mo[0] * fabs(o[0]) + mo[1] * fabs(o[1]) + mo[2] * fabs(o[2])) + 1.0;
	const double disc = b * b - 4.0 * a * c;
	MARGIN(disc, 2.0 * fabs(b) * mb + 4.0 * fabs(a) * mc + fabs(b * b) + fabs(4.0 * a * c));
	if (disc >= 0.0 && type != PT_SPHERE && a != 0.0)
	{
		const double root = sqrt(disc);
		const double q = b < 0.0 ? -0.5 * (b - root) : -0.5 * (b + root);
		const double ts[2] = { q / a, q != 0.0 ? c / q : 0.0 };
		/* the roots inherit the discriminant's noise through sqrt(disc): dt ~ d(disc) / (2 * root * 2a) */
		const double dDisc = eps * (2.0 * fabs(b) * mb + 4.0 * fabs(a) * mc + fabs(b * b) + fabs(4.0 * a * c));
		for (int k = 0; k < 2; ++k)
		{
			const double h = o[1] + d[1] * ts[k];
			const double dt = root > 0.0 ? dDisc / (4.0 * fabs(a) * root) : 1e300;
			const double magH = mo[1] + fabs(d[1] * ts[k]) + md[1] * fabs(ts[k]) + fabs(d[1]) * dt / eps + 1.0;
			MARGIN(fabs(h) - 1.0, magH);
		}
	}
#undef MARGIN
	return best;
}
void orc_material_sample(const pt_material_desc *m, const float *N, const float *in_dir, float rnd0, float rnd1, float *out9)
{
	v3 sdir; float pdf;
	float rough = m->roughness < 0.04f ? 0.04f : m->roughness;
	v3 att = materialSample(m->type, V(m->base_color[0], m->base_color[1], m->base_color[2]), rough, m->metalness, V(N[0], N[1], N[2]), V(in_dir[0], in_dir[1], in_dir[2]), rnd0, rnd1, &sdir, &pdf);
	out9[0] = att.x; out9[1] = att.y; out9[2] = att.z; out9[3] = pdf; out9[4] = sdir.x; out9[5] = sdir.y; out9[6] = sdir.z; out9[7] = 0.0f; out9[8] = 0.0f;
}
void orc_primary_pass(const orc_scene *s, const pt_camera_desc *cam, uint32_t w, uint32_t h, int32_t *idx, float *t, uint64_t *stats2)
{
	cam_t k = makeCamera(cam);
	uint64_t nv = 0, np = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : nv, np)
	for (int y = 0; y < (int)h; ++y)
		for (uint32_t x = 0; x < w; ++x)
		{
			ray_t r = cameraRay(&k, (x + 0.5f) / (float)w, (y + 0.5f) / (float)h);
			hit_t rec; uint32_t elem;
			int hit = hitBVH(s, r, 0.001f, FLT_MAX, &rec, &elem, &nv, &np);
			idx[(size_t)y * w + x] = hit ? s->toScene[elem] : -1;
			t[(size_t)y * w + x] = hit ? rec.t : 0.0f;
		}
	if (stats2) { stats2[0] = nv; stats2[1] = np; }
}
void orc_trace_rays(const orc_scene *s, size_t n, const float *o, const float *d, float tmin, int32_t *idx, float *t, float *nrm)
{
#pragma omp parallel for schedule(static, 256)
	for (long i = 0; i < (long)n; ++i)
	{
		ray_t r; r.o = V(o[3 * i], o[3 * i + 1], o[3 * i + 2]); r.d = V(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
		hit_t rec; uint32_t elem;
		int hit = hitBVH(s, r, tmin, FLT_MAX, &rec, &elem, NULL, NULL);
		idx[i] = hit ? s->toScene[elem] : -1; t[i] = hit ? rec.t : 0.0f;
		if (nrm) { nrm[3 * i] = hit ? rec.n.x : 0.0f; nrm[3 * i + 1] = hit ? rec.n.y : 0.0f; nrm[3 * i + 2] = hit ? rec.n.z : 0.0f; }
	}
}
/* First-bounce stratification — NOT in the reference; the product's one-pixel-per-warp kernels apply it by default from
 * 128 spp (include/pt_b200.h option "stratify", csrc/trace_kernels.h RenderParams::strataPer) and the path-for-path tests
 * need the checker to draw the same numbers.  The launch's first per << k samples of a pixel (local index i) take the two
 * randoms of the first scattering direction from cell i / per of a 2^bitsA x 2^bitsB grid: the cell gives the top bits, the
 * Philox draw the bits below.  Integer arithmetic only, so CPU and GPU agree to the bit.  Same rule as pt_render. */
/* threads orc_render will use; n > 0 sets the count first (see refh_threads, oracle/ref_harness/ref_host.cpp) */
#include <omp.h>
int orc_threads(int n)
{
	if (n > 0) omp_set_num_threads(n);
	return omp_get_max_threads();
}
static int g_stratify = 0;
void orc_set_stratify(int on) { g_stratify = on; }
static void strataFor(uint32_t spp, uint32_t *per, uint32_t *bitsA, uint32_t *bitsB)
{
	*per = 0; *bitsA = *bitsB = 0;
	if (!g_stratify || spp < 4u || spp >= (1u << 21)) return;
	uint32_t k = 2;
	while (k < 8u && (spp >> (k + 1u)) >= 16u) ++k;
	while (k > 2u && (spp >> k) == 0u) --k;
	*bitsA = (k + 1u) / 2u; *bitsB = k / 2u; *per = spp >> k;
}
/* traceKernel  kernels/trace.cu:158-199 with the Philox stream of north_star item 4 */
uint64_t orc_render(const orc_scene *s, const pt_camera_desc *cam, uint32_t w, uint32_t h, uint32_t spp, uint64_t seed,
                    uint32_t sample_offset, uint32_t sample_stride, int add, int max_bounces, float *accum)
{
	cam_t k = makeCamera(cam);
	uint64_t rays = 0;
	const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
	uint32_t per, bitsA, bitsB;
	strataFor(spp, &per, &bitsA, &bitsB);
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : rays)
	for (int y = 0; y < (int)h; ++y)
		for (uint32_t x = 0; x < w; ++x)
		{
			uint32_t pixel = x + (uint32_t)y * w;
			v3 color = V(0.0f, 0.0f, 0.0f);
			for (uint32_t i = 0; i < spp; ++i)
			{
				uint32_t sample = sample_offset + i * sample_stride, rng[4];
				orc_philox(pixel, sample, 0, 0, k0, k1, rng);
				if (per && i < (per << (bitsA + bitsB)))
				{
					const uint32_t cell = i / per, a = cell >> bitsB, bMask = (1u << bitsB) - 1u;
					const uint32_t b = (a & 1u) ? bMask - (cell & bMask) : (cell & bMask);
					rng[2] = (a << (32u - bitsA)) | (rng[2] >> bitsA);
					rng[3] = (b << (32u - bitsB)) | (rng[3] >> bitsB);
				}
				float u = (x + orc_uniform(rng[0])) / (float)w;
				float v = (y + orc_uniform(rng[1])) / (float)h;
				ray_t r = cameraRay(&k, u, v);
				color = vadd(color, s->nodeCount ? getColor(s, r, pixel, sample, k0, k1, rng, max_bounces, &rays) : V(0.0f, 0.0f, 0.0f));
			}
			float *a = accum + (size_t)pixel * 4;
			if (add) { color = vadd(color, V(a[0], a[1], a[2])); }
			a[0] = color.x; a[1] = color.y; a[2] = color.z; a[3] = 1.0f;
		}
	return rays;
}
/* tonemap  kernels/tonemap.cu:4-27 */
void orc_tonemap(const float *accum, size_t pixels, uint32_t sample_count, uint8_t *out)
{
	for (size_t i = 0; i < pixels; ++i)
	{
		v3 c = vdivf(V(accum[i * 4], accum[i * 4 + 1], accum[i * 4 + 2]), (float)sample_count);
		/* resultColor / (resultColor + 1.0f): operator/(vec3, vec3) = vec3(1/t) * v */
		c = V((1.0f / (c.x + 1.0f)) * c.x, (1.0f / (c.y + 1.0f)) * c.y, (1.0f / (c.z + 1.0f)) * c.z);
		c = V(powf(c.x, 1.0f / 2.2f), powf(c.y, 1.0f / 2.2f), powf(c.z, 1.0f / 2.2f));
		out[i * 4] = (unsigned char)(c.x * 255.0f); out[i * 4 + 1] = (unsigned char)(c.y * 255.0f); out[i * 4 + 2] = (unsigned char)(c.z * 255.0f); out[i * 4 + 3] = 255;
	}
}
void orc_texture_lookup(const orc_scene *s, uint32_t handle, float u, float v, float *out4)
{
	if (handle == 0 || handle > s->texCount) { out4[0] = out4[1] = out4[2] = out4[3] = 0.0f; return; }
	texLookup(&s->tex[handle - 1], u, v, out4);
}
