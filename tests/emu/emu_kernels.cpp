// emu_kernels.cpp — TEST-ONLY host emulation of the CUDA trace path.
//
// Compiles pathtracercuda_b200/csrc/trace_device.cuh (the exact per-ray device functions the sm_100a kernels call) for the
// CPU, with host stand-ins for the CUDA intrinsics, and drives them with plain loops that mirror the kernel bodies in
// trace_kernels.cu.  Purpose: on a box WITHOUT a GPU, the `-m "not gpu"` tests can still check the kernel LOGIC
// (two-box BVH traversal, shared quadric routine, tie-breaking, Philox draw schedule, shading) against the oracle.
// It is not a fallback: nothing in pathtracercuda_b200/ builds, links or loads this file, and its numbers are never
// reported.  What it cannot cover - the persistent-thread scheduler, the warp-aggregated pixel queue, the TMA staging -
// is covered by the `-m gpu` tests.
#define PTB_HOST_EMULATION
#define PTB_DEV static inline
#define PTB_MEMBER inline
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>
#include <string>
#include <vector>

static inline float rcpApprox(float x) { return 1.0f / x; }
static inline float sqrtApprox(float x) { return sqrtf(x); }
static inline float rsqrtApprox(float x) { return 1.0f / sqrtf(x); }
static inline float divExact(float a, float b) { return a / b; }
static inline float sqrtExact(float a) { return sqrtf(a); }
static inline float invSqrtExact(float x) { return 1.0f / sqrtf(x); }
template <typename T> static inline T __ldg(const T *p) { return *p; }
static inline float __fmaf_rn(float a, float b, float c) { return fmaf(a, b, c); }
static inline float __uint2float_rn(uint32_t x) { return (float)x; }
static inline uint32_t __umulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
static inline int __float_as_int(float f) { int i; memcpy(&i, &f, 4); return i; }
static inline uint32_t __float_as_uint(float f) { uint32_t i; memcpy(&i, &f, 4); return i; }
static inline float __uint_as_float(uint32_t i) { float f; memcpy(&f, &i, 4); return f; }
static inline uint32_t __float2uint_rz(float f) { return f > 0.0f ? (uint32_t)f : 0u; }
static inline void fastSinCos(float x, float *s, float *c) { *s = sinf(x); *c = cosf(x); }
static inline float fastPow(float a, float b) { return powf(a, b); }
using std::max;
using std::min;

#include "../../pathtracercuda_b200/csrc/scene_compile.h"
#include "../../pathtracercuda_b200/csrc/trace_device.cuh"

using namespace ptb;

namespace
{
struct EmuScene
{
	CompiledScene cs;
	std::vector<float4> blob;
	std::vector<std::vector<uint8_t>> texData;
	TexDesc tex[64];
	uint32_t texCount = 0, skybox = 0;
	SceneView<false> view() const
	{
		SceneView<false> sv;
		sv.nodes = blob.data();
		sv.prims = blob.data() + cs.nodes.size() * 4;
		sv.globalCount = cs.globalCount;
		return sv;
	}
};
} // namespace

static uint64_t g_lastWork[2] = { 0, 0 };
static int g_beam = 0;              // emu_render: camera rays through the pixel beam lists (trace_device.cuh beamLeaves)
static uint64_t g_beamStats[4] = { 0, 0, 0, 0 }; // pixels, list entries, overflows, longest list

extern "C"
{
void *emu_scene_create2(size_t n, const pt_object_desc *objs, uint32_t maxLeaf, int builder);
void *emu_scene_create(size_t n, const pt_object_desc *objs, uint32_t maxLeaf) { return emu_scene_create2(n, objs, maxLeaf, kBuilderSah); }
void *emu_scene_create2(size_t n, const pt_object_desc *objs, uint32_t maxLeaf, int builder)
{
	EmuScene *s = new EmuScene();
	std::string err;
	if (!compileScene(n, objs, maxLeaf, s->cs, err, kMaxGlobalPrims, nullptr, builder)) { delete s; return nullptr; }
	s->blob.resize((s->cs.nodes.size() + s->cs.prims.size()) * 4);
	memcpy(s->blob.data(), s->cs.nodes.data(), s->cs.nodes.size() * 64);
	memcpy(s->blob.data() + s->cs.nodes.size() * 4, s->cs.prims.data(), s->cs.prims.size() * 64);
	memset(s->tex, 0, sizeof s->tex);
	return s;
}
void emu_scene_destroy(void *p) { delete (EmuScene *)p; }
uint32_t emu_add_texture(void *p, uint32_t w, uint32_t h, int isHdr, const void *rgba)
{
	EmuScene *s = (EmuScene *)p;
	if (s->texCount >= 64) return 0;
	const size_t bytes = size_t(w) * h * (isHdr ? 16 : 4);
	s->texData.emplace_back((const uint8_t *)rgba, (const uint8_t *)rgba + bytes);
	TexDesc &t = s->tex[s->texCount];
	t.texels = s->texData.back().data();
	t.width = w; t.height = h; t.isHdr = isHdr ? 1u : 0u;
	return ++s->texCount;
}
void emu_set_skybox(void *p, uint32_t h) { ((EmuScene *)p)->skybox = h; }
uint32_t emu_global_count(void *p) { return ((EmuScene *)p)->cs.globalCount; }
void emu_scene_info(void *p, uint32_t *nodes, uint32_t *depth, uint32_t *leaves)
{
	EmuScene *s = (EmuScene *)p;
	*nodes = (uint32_t)s->cs.treeNodeCount; *depth = s->cs.depth; *leaves = s->cs.leafCount;
}
// raw compiled arrays for structural validation by the tests (Node = 16 x 4 bytes, Prim = 16 x 4 bytes)
void emu_scene_arrays(void *p, void *nodesOut, void *primsOut)
{
	EmuScene *s = (EmuScene *)p;
	memcpy(nodesOut, s->cs.nodes.data(), size_t(s->cs.treeNodeCount) * 64); // the tree (not the hoisted-box records behind it)
	memcpy(primsOut, s->cs.prims.data(), s->cs.prims.size() * 64);
}

// mirrors primaryKernel (trace_kernels.cu)
void emu_primary(void *p, const pt_camera_desc *cd, uint32_t width, uint32_t height, int32_t *hitIndex, float *hitT, uint64_t *stats2)
{
	EmuScene *s = (EmuScene *)p;
	CameraDev cam;
	computeCamera(*cd, cam);
	const SceneView<false> sv = s->view();
	uint64_t nvTot = 0, ptTot = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : nvTot, ptTot)
	for (int y = 0; y < (int)height; ++y)
		for (uint32_t x = 0; x < width; ++x)
		{
			const uint32_t i = x + uint32_t(y) * width;
			uint32_t nv = 0, pt = 0;
			const float u = (float(x) + 0.5f) / float(width), v = (float(y) + 0.5f) / float(height);
			const V3 o = mk(cam.origin[0], cam.origin[1], cam.origin[2]);
			const V3 d = cameraDir(cam, u, v);
			const Hit h = closestHit<false, true>(sv, o, d, 0.001f, nv, pt);
			hitIndex[i] = h.prim < 0 ? -1 : int32_t(primSceneIndex(sv.prims[h.prim * 4 + 3]));
			hitT[i] = h.prim < 0 ? 0.0f : h.t;
			nvTot += nv; ptTot += pt;
		}
	if (stats2) { stats2[0] = nvTot; stats2[1] = ptTot; }
}

// mirrors what the production kernel does for the camera ray of a pixel with option jitter = 0: the pixel's beam list
// (beamLeaves), then closestHitWW with the hot-path arithmetic - the first-hit gate of tests/test_gpu_baseline_sizes.py on the CPU
void emu_first_hit(void *p, const pt_camera_desc *cd, uint32_t width, uint32_t height, int useBeam, int32_t *hitIndex, float *hitT)
{
	EmuScene *s = (EmuScene *)p;
	CameraDev cam;
	computeCamera(*cd, cam);
	const SceneView<false> sv = s->view();
	const float invW = 1.0f / float(width), invH = 1.0f / float(height);
#pragma omp parallel for schedule(dynamic, 4)
	for (int y = 0; y < (int)height; ++y)
		for (uint32_t x = 0; x < width; ++x)
		{
			const uint32_t i = x + uint32_t(y) * width;
			uint32_t nv = 0, pt = 0;
			BeamEntry beam[kBeamMax];
			BeamBox boxes[kBeamMax];
			int nBeam = -1;
			const float m = 1.0f / 64.0f;
			if (useBeam)
				nBeam = beamLeaves<false>(sv.nodes, s->cs.treeNodeCount, uint32_t(s->cs.nodes.size()), cam, (float(x) - m) * invW, (float(x) + 1.0f + m) * invW, (float(y) - m) * invH,
				                          (float(y) + 1.0f + m) * invH, beam, true, boxes);
			const float u = (float(x) + 0.5f) / float(width), v = (float(y) + 0.5f) / float(height);
			const V3 o = mk(cam.origin[0], cam.origin[1], cam.origin[2]);
			const V3 d = cameraDir<2>(cam, u, v);
			const Hit h = closestHitWW<false, true, kHotExact>(sv, o, d, 0.001f, nv, pt, beam, nBeam, 0, boxes);
			hitIndex[i] = h.prim < 0 ? -1 : int32_t(primSceneIndex(sv.prims[h.prim * 4 + 3]));
			hitT[i] = h.prim < 0 ? 0.0f : h.t;
		}
}

// mirrors traceRaysKernel
void emu_trace_rays(void *p, size_t n, const float *origins, const float *directions, float tMin, int32_t *hitIndex, float *hitT, float *hitNormal)
{
	EmuScene *s = (EmuScene *)p;
	const SceneView<false> sv = s->view();
#pragma omp parallel for schedule(static, 256)
	for (long i = 0; i < (long)n; ++i)
	{
		uint32_t nv = 0, pt = 0;
		const V3 o = mk(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2]);
		const V3 d = mk(directions[3 * i], directions[3 * i + 1], directions[3 * i + 2]);
		const Hit h = closestHit<false, false>(sv, o, d, tMin, nv, pt);
		hitIndex[i] = h.prim < 0 ? -1 : int32_t(primSceneIndex(sv.prims[h.prim * 4 + 3]));
		hitT[i] = h.prim < 0 ? 0.0f : h.t;
		if (hitNormal)
		{
			V3 nn = mk(0.0f, 0.0f, 0.0f);
			if (h.prim >= 0) nn = surfaceAt<false>(sv, h.prim, o, d, h.t).n;
			hitNormal[3 * i] = nn.x; hitNormal[3 * i + 1] = nn.y; hitNormal[3 * i + 2] = nn.z;
		}
	}
}

// mirrors the per-lane body of traceKernel (generate -> traverse -> miss | shade -> accumulate), one pixel at a time
uint64_t emu_render(void *p, const pt_camera_desc *cd, uint32_t width, uint32_t height, uint32_t spp, uint64_t seed, uint32_t sampleOffset,
                    uint32_t sampleStride, int add, uint32_t maxBounces, float *accum)
{
	EmuScene *s = (EmuScene *)p;
	CameraDev cam;
	computeCamera(*cd, cam);
	const SceneView<false> sv = s->view();
	const uint32_t seedLo = (uint32_t)seed, seedHi = (uint32_t)(seed >> 32);
	const float invW = 1.0f / float(width), invH = 1.0f / float(height);
	const V3 camO = mk(cam.origin[0], cam.origin[1], cam.origin[2]);
	uint64_t raysTot = 0, nvTot = 0, ptTot = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : raysTot, nvTot, ptTot)
	for (int y = 0; y < (int)height; ++y)
		for (uint32_t x = 0; x < width; ++x)
		{
			const uint32_t pixel = x + uint32_t(y) * width;
			V3 color = mk(0.0f, 0.0f, 0.0f);
			BeamEntry beam[kBeamMax];
			BeamBox boxes[kBeamMax];
			int nBeam = -1;
			if (g_beam)
			{
				const float m = 1.0f / 64.0f;
				nBeam = beamLeaves<false>(sv.nodes, s->cs.treeNodeCount, uint32_t(s->cs.nodes.size()), cam, (float(x) - m) * invW, (float(x) + 1.0f + m) * invW, (float(y) - m) * invH, (float(y) + 1.0f + m) * invH, beam, true, boxes);
#pragma omp critical
				{
					++g_beamStats[0];
					if (nBeam < 0) ++g_beamStats[2];
					else { g_beamStats[1] += uint64_t(nBeam); g_beamStats[3] = std::max<uint64_t>(g_beamStats[3], uint64_t(nBeam)); }
				}
			}
			for (uint32_t sample = 0; sample < spp; ++sample)
			{
				const uint32_t sampleIdx = sampleOffset + sample * sampleStride;
				const uint4 r = philox4x32_10(pixel, sampleIdx, 0u, 0u, seedLo, seedHi);
				const float u = (float(x) + uniform01(r.x)) * (1.0f / float(width)), v = (float(y) + uniform01(r.y)) * (1.0f / float(height));
				uint32_t rz = r.z, rw = r.w;
				V3 ro = camO, rd = cameraDir<2>(cam, u, v), thr = mk(1.0f, 1.0f, 1.0f), L = mk(0.0f, 0.0f, 0.0f);
				uint32_t bounce = 0;
				while (true)
				{
					++raysTot;
					uint32_t nv = 0, pt = 0;
					const Hit h = g_beam ? closestHitWW<false, true, kHotExact>(sv, ro, rd, 0.001f, nv, pt, beam, bounce == 0 ? nBeam : -1, 0, boxes)
					                     : closestHit<false, true, kHotExact>(sv, ro, rd, 0.001f, nv, pt);
					nvTot += nv; ptTot += pt;
					if (h.prim < 0)
					{
						if (s->skybox != 0)
						{
							const float theta = fastAcos(rd.y), phi = fastAtan2(rd.z, rd.x);
							const V3 sky = texLookup(s->tex, s->skybox, phi * (0.5f / PT_PI), theta * (1.0f / PT_PI));
							L = L + thr * sky;
						}
						break;
					}
					const Surface sf = surfaceAt<false>(sv, h.prim, ro, rd, h.t);
					const Mat &m = s->cs.mats[h.prim];
					L = L + thr * mk(m.emissive[0], m.emissive[1], m.emissive[2]);
					V3 base = mk(m.baseColor[0], m.baseColor[1], m.baseColor[2]);
					if (m.texture != 0 && m.texture <= s->texCount)
					{
						const V3 tap = texLookup(s->tex, m.texture, sf.u, sf.v);
						base = mk(fastPow(tap.x, 2.2f), fastPow(tap.y, 2.2f), fastPow(tap.z, 2.2f));
					}
					float rnd0, rnd1;
					if (bounce == 0) { rnd0 = uniform01(rz); rnd1 = uniform01(rw); }
					else if (bounce & 1u)
					{
						const uint4 q = philox4x32_10(pixel, sampleIdx, (bounce + 1u) >> 1, 0u, seedLo, seedHi);
						rnd0 = uniform01(q.x); rnd1 = uniform01(q.y); rz = q.z; rw = q.w;
					}
					else { rnd0 = uniform01(rz); rnd1 = uniform01(rw); }
					V3 wi, weight;
					if (!sampleMaterial(m.type, base, m.roughness, m.metalness, sf.n, rd, rnd0, rnd1, wi, weight)) break;
					thr = thr * weight;
					ro = sf.p; rd = wi;
					if (++bounce >= maxBounces) break;
				}
				color = color + L;
			}
			float *a = accum + size_t(pixel) * 4;
			if (add) { color.x += a[0]; color.y += a[1]; color.z += a[2]; }
			a[0] = color.x; a[1] = color.y; a[2] = color.z; a[3] = 1.0f;
		}
	g_lastWork[0] = nvTot; g_lastWork[1] = ptTot;
	return raysTot;
}
// the compact atan2 / acos used for the equirectangular lookups (accuracy test)
void emu_fast_angles(size_t n, const float *y, const float *x, float *atan2Out, float *acosOut)
{
	for (size_t i = 0; i < n; ++i) { atan2Out[i] = fastAtan2(y[i], x[i]); acosOut[i] = fastAcos(x[i]); }
}
// node visits / primitive tests of the last emu_render (BVH quality experiments)
void emu_last_work(uint64_t *out) { out[0] = g_lastWork[0]; out[1] = g_lastWork[1]; }
// pixel beams on/off for emu_render + their statistics since the last call (pixels, entries, overflows, longest list)
void emu_set_beam(int on) { g_beam = on; for (auto &v : g_beamStats) v = 0; }
void emu_beam_stats(uint64_t *out) { for (int i = 0; i < 4; ++i) out[i] = g_beamStats[i]; }
}
