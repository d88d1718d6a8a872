/* light_oracle.c — TEST INFRASTRUCTURE ONLY.  NOT THE REFERENCE: the product's option "light_is" (next-event estimation of the
 * emitters with multiple importance sampling, pathtracercuda_b200/csrc/light_sampling.h) restated on top of the oracle, which is
 * included as it stands, so that the CUDA path can be checked path for path.  Same table (bit for bit: the same double arithmetic,
 * Vose's method with index-ordered work lists), same point sampler and pdf, shadow rays through the oracle's BVH with a tMax, the same
 * balance-heuristic weights.  Built by tests/test_light_sampling.py into a temporary directory. */
#include "../oracle/pt_oracle.c"

typedef struct
{
	float m[12];    /* local -> world rows */
	float pdfScale; /* P_sel / (A_l |det M|) */
	float q;        /* alias threshold */
	uint32_t alias, scene, type;
	float prob;
} lrec_t;
typedef struct
{
	uint32_t n;
	lrec_t *r;
	int32_t *ofScene; /* scene index -> emitter index, -1: not an emitter */
} lor_table;

static double lorLocalArea(uint32_t type)
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

lor_table *lor_build(const orc_scene *s)
{
	lor_table *t = (lor_table *)calloc(1, sizeof *t);
	t->ofScene = (int32_t *)malloc((s->n ? s->n : 1) * sizeof(int32_t));
	uint32_t n = 0;
	for (size_t i = 0; i < s->n; ++i)
	{
		const obj_t *o = &s->sceneObjs[i];
		t->ofScene[i] = (o->emissive.x != 0.0f || o->emissive.y != 0.0f || o->emissive.z != 0.0f) ? (int32_t)n++ : -1;
	}
	t->r = (lrec_t *)calloc(n ? n : 1, sizeof(lrec_t));
	double *w = (double *)calloc(n ? n : 1, sizeof(double)), *det = (double *)calloc(n ? n : 1, sizeof(double)), *scaled = (double *)calloc(n ? n : 1, sizeof(double));
	double total = 0.0;
	for (size_t i = 0; i < s->n; ++i)
	{
		if (t->ofScene[i] < 0) continue;
		const uint32_t k = (uint32_t)t->ofScene[i];
		const obj_t *o = &s->sceneObjs[i];
		lrec_t *L = &t->r[k];
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
		if (L->type == PT_QUAD || L->type == PT_DISK) area = lorLocalArea(L->type) * dM * len[1];
		else if (L->type == PT_CUBE) area = 8.0 * dM * (len[0] + len[1] + len[2]);
		else area = lorLocalArea(L->type) * cbrt(dM * dM);
		const double mean = ((double)o->emissive.x + (double)o->emissive.y + (double)o->emissive.z) / 3.0;
		w[k] = mean > 0.0 && isfinite(area) ? mean * area : 0.0;
		det[k] = dM;
		total += w[k];
	}
	if (!(total > 0.0 && isfinite(total))) n = 0;
	t->n = n;
	for (uint32_t k = 0; k < n; ++k)
	{
		const double P = w[k] / total;
		t->r[k].pdfScale = P > 0.0 ? (float)(P / (lorLocalArea(t->r[k].type) * det[k])) : 0.0f;
		t->r[k].prob = (float)P;
		scaled[k] = P * (double)n;
	}
	uint32_t *small = (uint32_t *)malloc((n ? n : 1) * sizeof(uint32_t)), *large = (uint32_t *)malloc((n ? n : 1) * sizeof(uint32_t));
	size_t ns = 0, nl = 0;
	for (uint32_t i = 0; i < n; ++i) { if (scaled[i] < 1.0) small[ns++] = i; else large[nl++] = i; }
#define LPUT(i, qq, other) do { double q_ = (qq); t->r[i].q = (float)(q_ < 0.0 ? 0.0 : (q_ > 1.0 ? 1.0 : q_)); t->r[i].alias = (other); } while (0)
	while (ns > 0 && nl > 0)
	{
		const uint32_t sm = small[--ns], lg = large[nl - 1];
		LPUT(sm, scaled[sm], lg);
		scaled[lg] = (scaled[lg] + scaled[sm]) - 1.0;
		if (scaled[lg] < 1.0) { --nl; small[ns++] = lg; }
	}
	for (size_t i = 0; i < nl; ++i) LPUT(large[i], 1.0, large[i]);
	for (size_t i = 0; i < ns; ++i) LPUT(small[i], 1.0, small[i]);
#undef LPUT
	free(small); free(large); free(w); free(det); free(scaled);
	return t;
}
void lor_free(lor_table *t) { if (t) { free(t->r); free(t->ofScene); free(t); } }
uint32_t lor_table_get(const lor_table *t, uint32_t *scene, float *prob, uint32_t *alias2)
{
	for (uint32_t k = 0; k < t->n; ++k)
	{
		if (scene) scene[k] = t->r[k].scene;
		if (prob) prob[k] = t->r[k].prob;
		if (alias2) { memcpy(&alias2[2 * k], &t->r[k].q, 4); alias2[2 * k + 1] = t->r[k].alias; }
	}
	return t->n;
}

static v3 lorUnitNormal(uint32_t type, v3 lp)
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
static v3 lorWorldNormal(const obj_t *o, v3 nl)
{
	return V(nl.x * o->r0[0] + nl.y * o->r1[0] + nl.z * o->r2[0], nl.x * o->r0[1] + nl.y * o->r1[1] + nl.z * o->r2[1], nl.x * o->r0[2] + nl.y * o->r1[2] + nl.z * o->r2[2]);
}
/* local point of the canonical surface from two uniforms and one word (face / nappe) */
static v3 lorLocalPoint(uint32_t type, float u, float v, uint32_t w)
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
static int lorSample(const orc_scene *s, const lor_table *t, const uint32_t q[4], v3 p, uint32_t *k, v3 *x, v3 *wdir, float *dist, float *pdf)
{
	const uint64_t xx = (uint64_t)q[0] * t->n;
	const uint32_t i = (uint32_t)(xx >> 32);
	const float frac = (float)(uint32_t)xx * 2.3283064365386963e-10f;
	*k = frac < t->r[i].q ? i : t->r[i].alias;
	const lrec_t *L = &t->r[*k];
	const v3 lp = lorLocalPoint(L->type, orc_uniform(q[1]), orc_uniform(q[2]), q[3]);
	*x = V(L->m[0] * lp.x + L->m[1] * lp.y + L->m[2] * lp.z + L->m[3], L->m[4] * lp.x + L->m[5] * lp.y + L->m[6] * lp.z + L->m[7],
	       L->m[8] * lp.x + L->m[9] * lp.y + L->m[10] * lp.z + L->m[11]);
	const v3 dv = vsub(*x, p);
	const float d2 = vdot(dv, dv);
	*dist = sqrtf(d2);
	*wdir = vscale(1.0f / *dist, dv);
	const v3 wn = lorWorldNormal(&s->sceneObjs[L->scene], lorUnitNormal(L->type, lp));
	*pdf = L->pdfScale * d2 / fmaxf(fabsf(vdot(wn, *wdir)), 1e-30f);
	return d2 > 0.0f && *pdf > 0.0f && *pdf < 3.0e38f;
}
/* sampler test aid: out8 = world point, area pdf p_A = pdf_sel-free (pdfScale / P_sel / |W^T n_l|), emitter, local point */
void lor_sample_point(const orc_scene *s, const lor_table *t, const uint32_t *q, float *out8)
{
	uint32_t k; v3 x, wd; float dist, pdf;
	lorSample(s, t, q, V(0.0f, 0.0f, 0.0f), &k, &x, &wd, &dist, &pdf);
	const lrec_t *L = &t->r[k];
	const v3 lp = lorLocalPoint(L->type, orc_uniform(q[1]), orc_uniform(q[2]), q[3]);
	const v3 wn = lorWorldNormal(&s->sceneObjs[L->scene], lorUnitNormal(L->type, lp));
	out8[0] = x.x; out8[1] = x.y; out8[2] = x.z;
	out8[3] = (float)((double)L->pdfScale / (double)L->prob / sqrt((double)wn.x * wn.x + (double)wn.y * wn.y + (double)wn.z * wn.z));
	out8[4] = (float)k; out8[5] = lp.x; out8[6] = lp.y; out8[7] = lp.z;
}

/* occlusion: any primitive hit in (tMin, tMax] */
static int lorOccluded(const orc_scene *s, ray_t r, float tMin, float tMax)
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

/* getColor (pt_oracle.c) with the light sample at every scattering vertex: Philox counter word 3 = 2, slot = bounce */
static v3 lorGetColor(const orc_scene *s, const lor_table *t, ray_t ray, uint32_t pixel, uint32_t sample, uint32_t k0, uint32_t k1, const uint32_t rng0[4],
                      int maxBounces, uint64_t *rays)
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
			if (s->skybox != 0 && s->skybox <= s->texCount)
			{
				float theta = acosf(ray.d.y), phi = atan2f(ray.d.z, ray.d.x);
				float v = theta / PI_F, u = phi / (2.0f * PI_F), tap[4];
				texLookup(&s->tex[s->skybox - 1], u, v, tap);
				L = vadd(L, vmul(throughput, V(tap[0], tap[1], tap[2])));
			}
			break;
		}
		const obj_t *o = &s->objs[elem];
		v3 em = o->emissive;
		const int32_t ek = t->n ? t->ofScene[s->toScene[elem]] : -1;
		if (it > 0 && ek >= 0)
		{
			/* balance-heuristic weight of a BSDF-sampled direction that hit an emitter */
			v3 lo;
			lo.x = vdot(ray.o, V(o->r0[0], o->r0[1], o->r0[2])) + o->r0[3];
			lo.y = vdot(ray.o, V(o->r1[0], o->r1[1], o->r1[2])) + o->r1[3];
			lo.z = vdot(ray.o, V(o->r2[0], o->r2[1], o->r2[2])) + o->r2[3];
			const v3 ld = V(vdot(ray.d, V(o->r0[0], o->r0[1], o->r0[2])), vdot(ray.d, V(o->r1[0], o->r1[1], o->r1[2])), vdot(ray.d, V(o->r2[0], o->r2[1], o->r2[2])));
			const v3 lp = vadd(lo, vscale(rec.t, ld));
			const v3 wn = lorWorldNormal(o, lorUnitNormal(t->r[ek].type, lp));
			const float pl = t->r[ek].pdfScale * rec.t * rec.t / fmaxf(fabsf(vdot(wn, ray.d)), 1e-30f);
			em = vscale(lastPdf / (lastPdf + pl), em);
		}
		L = vadd(L, vmul(throughput, em));
		float rnd0, rnd1;
		if (it == 0) { rnd0 = orc_uniform(rng[2]); rnd1 = orc_uniform(rng[3]); }
		else
		{
			if (it & 1) orc_philox(pixel, sample, (uint32_t)(it + 1) / 2, 0, k0, k1, rng);
			rnd0 = orc_uniform(rng[(it & 1) ? 0 : 2]); rnd1 = orc_uniform(rng[(it & 1) ? 1 : 3]);
		}
		v3 sdir; float pdf;
		const v3 base = resolveBaseColor(s, o, rec.u, rec.v);
		if (t->n && it + 1 < maxBounces)
		{
			uint32_t q[4], k; v3 x, wl; float dist, pl;
			orc_philox(pixel, sample, (uint32_t)it, 2, k0, k1, q);
			if (lorSample(s, t, q, rec.p, &k, &x, &wl, &dist, &pl))
			{
				const v3 Vv = worldToTangent(rec.n, vneg(ray.d)), sl = worldToTangent(rec.n, wl);
				float pbL;
				const v3 attL = materialEval(o->mtype, base, o->roughness, o->metalness, Vv, sl, &pbL);
				if (sl.z > 0.0f && !((attL.x == 0.0f && attL.y == 0.0f && attL.z == 0.0f) || pbL == 0.0f))
				{
					ray_t sh; sh.o = rec.p; sh.d = wl;
					++*rays;
					if (!lorOccluded(s, sh, 0.001f, dist * (1.0f - 1e-4f)))
						L = vadd(L, vmul(vmul(throughput, vscale(sl.z / (pl + pbL), attL)), s->sceneObjs[t->r[k].scene].emissive));
				}
			}
		}
		v3 att = materialSample(o->mtype, base, o->roughness, o->metalness, rec.n, ray.d, rnd0, rnd1, &sdir, &pdf);
		lastPdf = pdf;
		if ((att.x == 0.0f && att.y == 0.0f && att.z == 0.0f) || pdf == 0.0f) break;
		v3 w = vdivf(vscale(fabsf(vdot(sdir, rec.n)), att), pdf);
		throughput = vmul(throughput, w);
		ray.o = rec.p; ray.d = sdir;
	}
	return L;
}

/* orc_render with the light sample; the same sample indices, stratification and accumulation */
uint64_t lor_render(const orc_scene *s, const lor_table *t, const pt_camera_desc *cam, uint32_t w, uint32_t h, uint32_t spp, uint64_t seed,
                    uint32_t sample_offset, uint32_t sample_stride, int max_bounces, float *accum)
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
				color = vadd(color, s->nodeCount ? lorGetColor(s, t, r, pixel, sample, k0, k1, rng, max_bounces, &rays) : V(0.0f, 0.0f, 0.0f));
			}
			float *a = accum + (size_t)pixel * 4;
			a[0] = color.x; a[1] = color.y; a[2] = color.z; a[3] = 1.0f;
		}
	return rays;
}
