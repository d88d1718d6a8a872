// device_probe.cu — TEST-ONLY: the trace kernels' per-call device routines (trace_device.cuh), one thread per input, behind
// extern "C" host wrappers, so that tests/test_device_functions.py and tests/test_texture_lookups.py can compare each routine on the
// GPU with the reference's stored outputs and with float64 statements.  Never part of libpt_b200.so: the test builds it into a
// temporary directory, together with the product's own host code (scene_compile.cpp, light_sampling.cpp, env_sampling.cpp) that
// makes the records the kernels read.
// Every wrapper allocates, copies in, launches, copies out and frees; errors come back as a negative return value.
#include "../pathtracercuda_b200/csrc/trace_device.cuh"
#include "../pathtracercuda_b200/csrc/env_sampling.h"
#include "../pathtracercuda_b200/csrc/light_sampling.h"
#include "../pathtracercuda_b200/csrc/scene_compile.h"
#include <cstring>
#include <string>
#include <vector>

using namespace ptb;

namespace
{
constexpr int kBlock = 128;
inline uint32_t gridFor(uint32_t n) { return (n + kBlock - 1) / kBlock; }

template <typename T>
T *toDevice(const void *src, size_t bytes)
{
	T *d = nullptr;
	if (cudaMalloc(&d, bytes ? bytes : 16) != cudaSuccess) return nullptr;
	if (bytes && cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return nullptr; }
	return d;
}
// launch finished + result copied back
int finish(void *host, const void *dev, size_t bytes)
{
	if (cudaGetLastError() != cudaSuccess) return -2;
	if (cudaDeviceSynchronize() != cudaSuccess) return -3;
	return cudaMemcpy(host, dev, bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -4;
}
} // namespace

// ---------------------------------------------------------------------------------------------------------------------------------
// materials.  in[20]: type, base rgb, roughness, metalness, N xyz (world), inDir xyz (world), rnd0, rnd1, sdir xyz (tangent), -, -, -
// out[32]: [0] ok, [1..3] wi, [4..6] weight, [7] pdfOut                 sampleMaterial(frame form, pdfOut)
//          [8] ok, [9..11] wi, [12..14] weight                          sampleMaterial(N, inDir form)
//          [15] ok, [16..18] att, [19] pdf                              evalMaterial(V, sdir)
//          [20] ok, [21..23] att, [24] pdf                              evalMaterial(V, toTangent(frame, wi)) of the first form
//          [25..27] V (tangent), [28..30] toTangent(frame, wi)
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void materialKernel(uint32_t n, const float *in, float *out)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float *a = in + 20 * size_t(i);
	float *o = out + 32 * size_t(i);
	const uint32_t mtype = uint32_t(a[0]);
	const V3 base = mk(a[1], a[2], a[3]), N = mk(a[6], a[7], a[8]), inDir = mk(a[9], a[10], a[11]), sdir = mk(a[14], a[15], a[16]);
	const Frame fr = makeFrame(N);
	const V3 Vv = toTangent(fr, -inDir);
	V3 wi = mk(0.f, 0.f, 0.f), w = mk(0.f, 0.f, 0.f);
	float pdf = 0.f;
	const bool ok = sampleMaterial(mtype, base, a[4], a[5], fr, Vv, a[12], a[13], wi, w, &pdf);
	o[0] = ok; o[1] = wi.x; o[2] = wi.y; o[3] = wi.z; o[4] = w.x; o[5] = w.y; o[6] = w.z; o[7] = pdf;
	V3 wi2 = mk(0.f, 0.f, 0.f), w2 = mk(0.f, 0.f, 0.f);
	const bool ok2 = sampleMaterial(mtype, base, a[4], a[5], N, inDir, a[12], a[13], wi2, w2);
	o[8] = ok2; o[9] = wi2.x; o[10] = wi2.y; o[11] = wi2.z; o[12] = w2.x; o[13] = w2.y; o[14] = w2.z;
	V3 att = mk(0.f, 0.f, 0.f);
	float pe = 0.f;
	const bool okE = evalMaterial(mtype, base, a[4], a[5], Vv, sdir, att, pe);
	o[15] = okE; o[16] = att.x; o[17] = att.y; o[18] = att.z; o[19] = pe;
	const V3 back = toTangent(fr, wi);
	V3 attR = mk(0.f, 0.f, 0.f);
	float pr = 0.f;
	const bool okR = ok && evalMaterial(mtype, base, a[4], a[5], Vv, back, attR, pr);
	o[20] = okR; o[21] = attR.x; o[22] = attR.y; o[23] = attR.z; o[24] = pr;
	o[25] = Vv.x; o[26] = Vv.y; o[27] = Vv.z; o[28] = back.x; o[29] = back.y; o[30] = back.z; o[31] = 0.f;
}

extern "C" int probe_material(uint32_t n, const float *in, float *out)
{
	float *dIn = toDevice<float>(in, size_t(n) * 20 * 4), *dOut = nullptr;
	if (!dIn || cudaMalloc(&dOut, size_t(n) * 32 * 4) != cudaSuccess) { cudaFree(dIn); return -1; }
	materialKernel<<<gridFor(n), kBlock>>>(n, dIn, dOut);
	const int rc = finish(out, dOut, size_t(n) * 32 * 4);
	cudaFree(dIn);
	cudaFree(dOut);
	return rc;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// scenes: the product's scene compiler and emitter table, uploaded as the kernels see them (Prim rows in BVH order, LightRecs)
// ---------------------------------------------------------------------------------------------------------------------------------
struct ProbeScene
{
	CompiledScene cs;
	LightTable lt;
	float4 *prims = nullptr;   // device, 4 quads per primitive
	float4 *lights = nullptr;  // device, 4 quads per emitter
	int *emitterOf = nullptr;  // device, per primitive: its emitter index (Mat::pad[0] - 1), -1 when not an emitter
	std::vector<int> primOf;   // per scene object: its primitive index (BVH order)
};

extern "C" void *probe_scene_create(size_t count, const pt_object_desc *objects)
{
	ProbeScene *s = new ProbeScene;
	std::string err;
	if (!compileScene(count, objects, 4, s->cs, err)) { delete s; return nullptr; }
	buildLightTable(s->cs, s->lt);
	const size_t np = s->cs.prims.size();
	s->primOf.assign(count, -1);
	std::vector<int> em(np);
	for (size_t p = 0; p < np; ++p)
	{
		s->primOf[s->cs.prims[p].packed & kPrimSceneMask] = int(p);
		em[p] = int(s->cs.mats[p].pad[0]) - 1;
	}
	s->prims = toDevice<float4>(s->cs.prims.data(), np * sizeof(Prim));
	s->lights = toDevice<float4>(s->lt.recs.data(), s->lt.recs.size() * sizeof(LightRec));
	s->emitterOf = toDevice<int>(em.data(), np * sizeof(int));
	if (!s->prims || !s->lights || !s->emitterOf) { cudaFree(s->prims); cudaFree(s->lights); cudaFree(s->emitterOf); delete s; return nullptr; }
	return s;
}

extern "C" void probe_scene_destroy(void *h)
{
	ProbeScene *s = static_cast<ProbeScene *>(h);
	if (!s) return;
	cudaFree(s->prims);
	cudaFree(s->lights);
	cudaFree(s->emitterOf);
	delete s;
}

// primOf[count]: primitive index of every scene object; returns the number of emitters
extern "C" uint32_t probe_scene_info(void *h, int *primOf)
{
	const ProbeScene *s = static_cast<const ProbeScene *>(h);
	if (primOf) memcpy(primOf, s->primOf.data(), s->primOf.size() * sizeof(int));
	return uint32_t(s->lt.recs.size());
}

// ---------------------------------------------------------------------------------------------------------------------------------
// hit: testPrimInline<false, EXACT, CLIP> on one primitive with best.t = tMax, then surfaceAt.
// out[12]: hit, t, p xyz, n xyz, u, v, -, -
// ---------------------------------------------------------------------------------------------------------------------------------
template <bool EXACT, bool CLIP>
__global__ void hitKernel(const float4 *prims, uint32_t n, const int *prim, const float *o, const float *d, float tMin, const float *tMax, float *out)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const V3 O = mk(o[3 * i], o[3 * i + 1], o[3 * i + 2]), D = mk(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
	Best best;
	best.t = tMax[i]; best.prim = -1; best.scene = 0;
	best = testPrimInline<false, EXACT, CLIP>(prims, uint32_t(prim[i]), makeRayOD(O, D), tMin, best);
	float *r = out + 12 * size_t(i);
	for (int k = 0; k < 12; ++k) r[k] = 0.f;
	r[0] = best.prim >= 0;
	r[1] = best.t;
	if (best.prim < 0) return;
	SceneView<false> sv;
	sv.nodes = prims; sv.prims = prims; sv.globalCount = 0;
	const Surface s = surfaceAt<false>(sv, best.prim, O, D, best.t);
	r[2] = s.p.x; r[3] = s.p.y; r[4] = s.p.z; r[5] = s.n.x; r[6] = s.n.y; r[7] = s.n.z; r[8] = s.u; r[9] = s.v;
}

// mode: bit 0 = EXACT (the parity kernels' IEEE division / square root; else kHotExact, what the render kernels run), bit 1 = CLIP
extern "C" int probe_hit(void *h, int mode, uint32_t n, const int *prim, const float *o, const float *d, float tMin, const float *tMax, float *out)
{
	const ProbeScene *s = static_cast<const ProbeScene *>(h);
	int *dPrim = toDevice<int>(prim, size_t(n) * 4);
	float *dO = toDevice<float>(o, size_t(n) * 12), *dD = toDevice<float>(d, size_t(n) * 12), *dT = toDevice<float>(tMax, size_t(n) * 4), *dOut = nullptr;
	int rc = -1;
	if (dPrim && dO && dD && dT && cudaMalloc(&dOut, size_t(n) * 48) == cudaSuccess)
	{
		switch (mode & 3)
		{
		case 0: hitKernel<kHotExact, false><<<gridFor(n), kBlock>>>(s->prims, n, dPrim, dO, dD, tMin, dT, dOut); break;
		case 1: hitKernel<true, false><<<gridFor(n), kBlock>>>(s->prims, n, dPrim, dO, dD, tMin, dT, dOut); break;
		case 2: hitKernel<kHotExact, true><<<gridFor(n), kBlock>>>(s->prims, n, dPrim, dO, dD, tMin, dT, dOut); break;
		default: hitKernel<true, true><<<gridFor(n), kBlock>>>(s->prims, n, dPrim, dO, dD, tMin, dT, dOut); break;
		}
		rc = finish(out, dOut, size_t(n) * 48);
	}
	cudaFree(dPrim); cudaFree(dO); cudaFree(dD); cudaFree(dT); cudaFree(dOut);
	return rc;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// light: sampleLight<false>, then lightPdfHit<false> for the ray from the same origin along the returned direction to the returned
// distance.  out[8]: ok, w xyz, dist, pdf, prim (BVH order), lightPdfHit
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void lightKernel(LightDev L, const float4 *prims, const int *emitterOf, uint32_t n, const uint4 *q, const float *p, float *out)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	SceneView<false> sv;
	sv.nodes = prims; sv.prims = prims; sv.globalCount = 0;
	V3 w = mk(0.f, 0.f, 0.f);
	float dist = 0.f, pdf = 0.f;
	int prim = -1;
	const V3 P = mk(p[3 * i], p[3 * i + 1], p[3 * i + 2]);
	const bool ok = sampleLight<false>(L, sv, q[i], P, w, dist, pdf, prim);
	float *r = out + 8 * size_t(i);
	r[0] = ok; r[1] = w.x; r[2] = w.y; r[3] = w.z; r[4] = dist; r[5] = pdf; r[6] = float(prim);
	r[7] = ok ? lightPdfHit<false>(L, sv, uint32_t(emitterOf[prim]), prim, P, w, dist) : 0.f;
}

extern "C" int probe_light(void *h, uint32_t n, const uint32_t *q, const float *p, float *out)
{
	const ProbeScene *s = static_cast<const ProbeScene *>(h);
	if (s->lt.recs.empty()) return -5;
	uint4 *dQ = toDevice<uint4>(q, size_t(n) * 16);
	float *dP = toDevice<float>(p, size_t(n) * 12), *dOut = nullptr;
	int rc = -1;
	if (dQ && dP && cudaMalloc(&dOut, size_t(n) * 32) == cudaSuccess)
	{
		LightDev L;
		L.recs = s->lights;
		L.count = uint32_t(s->lt.recs.size());
		lightKernel<<<gridFor(n), kBlock>>>(L, s->prims, s->emitterOf, n, dQ, dP, dOut);
		rc = finish(out, dOut, size_t(n) * 32);
	}
	cudaFree(dQ); cudaFree(dP); cudaFree(dOut);
	return rc;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// sky: the product's distribution of an RGBA float (isHdr) or RGBA8 texture; sampleEnv then envPdf at the returned (u, v), and envPdf
// alone at given (u, v, dir.y).
// env out[8]: d xyz, u, v, pdf, envPdf(u, v, d.y), -          pdf out[1]: envPdf
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void envKernel(EnvDev e, uint32_t n, const uint4 *q, float *out)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	float u = 0.f, v = 0.f, pdf = 0.f;
	const V3 d = sampleEnv(e, q[i].x, q[i].y, q[i].z, u, v, pdf);
	float *r = out + 8 * size_t(i);
	r[0] = d.x; r[1] = d.y; r[2] = d.z; r[3] = u; r[4] = v; r[5] = pdf; r[6] = envPdf(e, u, v, d.y); r[7] = 0.f;
}
__global__ void envPdfKernel(EnvDev e, uint32_t n, const float *uvy, float *out)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	out[i] = envPdf(e, uvy[3 * i], uvy[3 * i + 1], uvy[3 * i + 2]);
}

// mode 0: n draws of sampleEnv from q[4 n] (the fourth word unused), out[8 n];  mode 1: envPdf at q = float (u, v, dir.y)[3 n], out[n]
extern "C" int probe_env(uint32_t width, uint32_t height, int isHdr, const void *texels, int mode, uint32_t n, const void *q, float *out)
{
	EnvDistribution dist;
	buildEnvDistribution(width, height, isHdr != 0, texels, dist);
	EnvDev e;
	uint2 *dAlias = toDevice<uint2>(dist.alias.data(), dist.alias.size() * 4);
	float *dDens = toDevice<float>(dist.density.data(), dist.density.size() * 4);
	e.alias = dAlias;
	e.density = dDens;
	e.cols = dist.cols;
	e.rows = dist.rows;
	const size_t inBytes = size_t(n) * (mode == 0 ? 16 : 12), outBytes = size_t(n) * (mode == 0 ? 32 : 4);
	void *dQ = toDevice<char>(q, inBytes);
	float *dOut = nullptr;
	int rc = -1;
	if (dAlias && dDens && dQ && cudaMalloc(&dOut, outBytes) == cudaSuccess)
	{
		if (mode == 0) envKernel<<<gridFor(n), kBlock>>>(e, n, static_cast<const uint4 *>(dQ), dOut);
		else envPdfKernel<<<gridFor(n), kBlock>>>(e, n, static_cast<const float *>(dQ), dOut);
		rc = finish(out, dOut, outBytes);
	}
	cudaFree(dAlias); cudaFree(dDens); cudaFree(dQ); cudaFree(dOut);
	return rc;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// textures: texLookup on a one-entry TexDesc table (handle 1) over the caller's texels - RGBA8 words or float4, row-major.
// unit 0: texObj = 0, the fp32 software filter (option tex_unit = 0).  unit 1: a texture object over a copy of the texels in a CUDA
// array with the descriptor of pt_capi.cu loadTextureMemOne (wrap U, clamp V, linear filter, normalised coordinates, RGBA8 read as
// normalised floats).  This object is the probe's own; the end-to-end tests of tests/test_texture_lookups.py are what tie the
// product's object to it.  in: (u, v)[2 n]; out[3 n]: the tap's rgb.
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void texKernel(const TexDesc *table, uint32_t n, const float *uv, float *out)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const V3 r = texLookup(table, 1u, uv[2 * i], uv[2 * i + 1]);
	out[3 * i] = r.x; out[3 * i + 1] = r.y; out[3 * i + 2] = r.z;
}

extern "C" int probe_tex(uint32_t width, uint32_t height, int isHdr, const void *texels, int unit, uint32_t n, const float *uv, float *out)
{
	const size_t pitch = size_t(width) * (isHdr ? 16 : 4);
	TexDesc t;
	memset(&t, 0, sizeof t);
	t.texels = toDevice<char>(texels, pitch * height);
	t.width = width;
	t.height = height;
	t.isHdr = isHdr ? 1u : 0u;
	cudaArray_t arr = nullptr;
	cudaTextureObject_t obj = 0;
	int rc = -1;
	if (t.texels && unit)
	{
		cudaChannelFormatDesc fmt = isHdr ? cudaCreateChannelDesc<float4>() : cudaCreateChannelDesc<uchar4>();
		bool ok = cudaMallocArray(&arr, &fmt, width, height) == cudaSuccess;
		ok = ok && cudaMemcpy2DToArray(arr, 0, 0, texels, pitch, pitch, height, cudaMemcpyHostToDevice) == cudaSuccess;
		if (ok)
		{
			cudaResourceDesc rd;
			memset(&rd, 0, sizeof rd);
			rd.resType = cudaResourceTypeArray;
			rd.res.array.array = arr;
			cudaTextureDesc td;
			memset(&td, 0, sizeof td);
			td.addressMode[0] = cudaAddressModeWrap;
			td.addressMode[1] = cudaAddressModeClamp;
			td.filterMode = cudaFilterModeLinear;
			td.readMode = isHdr ? cudaReadModeElementType : cudaReadModeNormalizedFloat;
			td.normalizedCoords = 1;
			ok = cudaCreateTextureObject(&obj, &rd, &td, nullptr) == cudaSuccess;
		}
		t.texObj = ok ? (unsigned long long)obj : 0ull;
	}
	TexDesc *dTab = (t.texels && (!unit || t.texObj)) ? toDevice<TexDesc>(&t, sizeof t) : nullptr;
	float *dUV = toDevice<float>(uv, size_t(n) * 8), *dOut = nullptr;
	if (dTab && dUV && cudaMalloc(&dOut, size_t(n) * 12) == cudaSuccess)
	{
		texKernel<<<gridFor(n), kBlock>>>(dTab, n, dUV, dOut);
		rc = finish(out, dOut, size_t(n) * 12);
	}
	if (obj) cudaDestroyTextureObject(obj);
	if (arr) cudaFreeArray(arr);
	cudaFree(const_cast<void *>(t.texels)); cudaFree(dTab); cudaFree(dUV); cudaFree(dOut);
	return rc;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// the equirectangular angles and the gamma step.  in[4 n]: y, x, c, p.
// out[4 n]: fastAtan2(y, x), fastAtan2Inline(y, x), fastAcos(c), fastPow(p, 2.2f)
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void angleKernel(uint32_t n, const float *in, float *out)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float *a = in + 4 * size_t(i);
	float *o = out + 4 * size_t(i);
	o[0] = fastAtan2(a[0], a[1]); o[1] = fastAtan2Inline(a[0], a[1]); o[2] = fastAcos(a[2]); o[3] = fastPow(a[3], 2.2f);
}

extern "C" int probe_angles(uint32_t n, const float *in, float *out)
{
	float *dIn = toDevice<float>(in, size_t(n) * 16), *dOut = nullptr;
	int rc = -1;
	if (dIn && cudaMalloc(&dOut, size_t(n) * 16) == cudaSuccess)
	{
		angleKernel<<<gridFor(n), kBlock>>>(n, dIn, dOut);
		rc = finish(out, dOut, size_t(n) * 16);
	}
	cudaFree(dIn); cudaFree(dOut);
	return rc;
}
