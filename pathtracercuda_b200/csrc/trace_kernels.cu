// trace_kernels.cu — the trace hot path as hand-written sm_100a CUDA.
//
// Replaces the reference's three kernels (kernels/trace.cu traceKernel :158-199 + getColor :101-156 + hitBVH :28-98,
// kernels/initRandState.cu, kernels/tonemap.cu) and the device halves of Hittable.inl / Material.inl / MonteCarlo.h /
// brdf.h / Camera.inl.  Same estimator, different machine mapping:
//
//   * persistent CTAs (one wave sized to the SM count) with path regeneration, so warps stay full through all five path
//     segments instead of idling until the longest path of the warp ends (the reference runs one thread per pixel with no
//     compaction).  Long renders (SHARE, from 64 spp): ONE PIXEL PER WARP - the lanes trace samples of the same
//     pixel; the leaves its camera rays can reach are found once per pixel (pixel beams, trace_device.cuh beamLeaves); a
//     pass of the main loop is either for camera rays or for scattered rays; the first bounce is stratified (RenderParams::
//     strataPer).  Short renders: one pixel per lane, pixels handed out by a warp-aggregated atomic (ballot + popc prefix);
//   * no per-pixel RNG state, no 48 B/pixel buffer: Philox4x32-10 keyed on (seed), counter (pixel, sample, bounce slot);
//   * the BVH is 64-byte two-box nodes + 64-byte primitives read with 128-bit loads; when nodes+primitives fit in
//     shared memory they are staged there once per CTA with a TMA bulk copy (cp.async.bulk + mbarrier);
//   * ray/box tests use a precomputed reciprocal direction (12 FMA per node instead of the reference's 3 IEEE
//     divisions per box, AABB.inl:26); the four quadrics share one intersection routine selected by coefficients, the
//     two flat shapes share another: 3 divergent classes instead of 7;
//   * normals, UVs, the tangent frame and the material fetch happen once per path segment at the closest hit, not once
//     per accepted candidate (Hittable.inl:129-142).
#include "trace_common.cuh"
#include <algorithm>

namespace ptb
{

// a finished pixel: the sum of its samples into the accumulation buffer (trace.cu:196-198)
static __device__ __forceinline__ void storePixel(const RenderParams &p, uint32_t pixel, V3 color)
{
	float4 out = make_float4(color.x, color.y, color.z, p.alpha);
	if (!p.ignoreHistory)
	{
		const float4 prev = p.accum[pixel];
		out.x += prev.x; out.y += prev.y; out.z += prev.z;
	}
	p.accum[pixel] = out;
}

// the base colour of a hit (Material.inl:26-35): the material's own, or the tap of its texture at (u, v) taken to linear by the 2.2 power;
// one statement for the trace kernels and the guide-buffer kernel, so that the albedo guide is the colour the paths are shaded with
static __device__ __forceinline__ V3 baseColour(const SceneDev &scene, float4 m0, uint32_t tex, float u, float v)
{
	V3 base = mk(m0.x, m0.y, m0.z);
	if (tex != 0 && tex <= scene.texCount)
	{
		const V3 tap = texLookup(scene.textures, tex, u, v); // Material.inl:26-35
		base = mk(fastPow(tap.x, 2.2f), fastPow(tap.y, 2.2f), fastPow(tap.z, 2.2f));
	}
	return base;
}

// a contribution of a lane's path: the one-pixel-per-warp kernel (SHARE) adds it to the warp's partial sums of the pixel as it comes, the
// one-pixel-per-lane kernel to the path's own sum L, which goes to the pixel's when the path ends (the two orders of the additions give
// different bits).  The contribution is a x b.  ADAPT: the one-pixel-per-warp kernel also sums the luminance of the path's contributions
// (the luminance of the path's total, one register instead of three), for the stopping test of option "adaptive"; the weights are those of
// env_sampling.cpp.  Its product is its own, never contracted (__fmul_rn): a product with two uses is not fused into the addition to
// `color`, which would then round differently from the kernel without the option
template <bool SHARE, bool ADAPT = false>
static __device__ __forceinline__ void accumulate(V3 &color, V3 &L, float &y, V3 a, V3 b)
{
	if constexpr (SHARE) color = color + a * b;
	else L = L + a * b;
	if constexpr (ADAPT) y += 0.2126f * __fmul_rn(a.x, b.x) + 0.7152f * __fmul_rn(a.y, b.y) + 0.0722f * __fmul_rn(a.z, b.z);
}

// first-bounce stratification of the one-pixel-per-warp kernel (RenderParams::strataPer): the cell of the sample with local index m (m / per)
// becomes the top bits of the two randoms of the first scattering direction, the Philox draw fills the bits below
static __device__ __forceinline__ void stratify(uint32_t m, uint32_t per, uint32_t bitsA, uint32_t bitsB, float invPer, uint32_t &rz, uint32_t &rw)
{
	if (m < (per << (bitsA + bitsB)))
	{
		const uint32_t cell = __float2uint_rz((__uint2float_rn(m) + 0.5f) * invPer);
		const uint32_t a = cell >> bitsB, bMask = (1u << bitsB) - 1u;
		const uint32_t b = (a & 1u) ? bMask - (cell & bMask) : (cell & bMask); // snake: neighbouring cells are neighbouring directions
		rz = (a << (32u - bitsA)) | (rz >> bitsA);
		rw = (b << (32u - bitsB)) | (rw >> bitsB);
	}
}

// ---------------------------------------------------------------------------------------------------------------
// the trace kernel
// ---------------------------------------------------------------------------------------------------------------
// SMEM: the scene staged in shared memory; COUNT: work counters (option "count_work"); SHARE: one pixel per warp; SSTACK: the
// traversal stack in shared memory; TWIN: the options compiled into an instantiation of their own (trace_kernels.h Twin); ADAPT (SHARE only):
// option "adaptive", a pixel's samples stop at the first checkpoint whose stopping test passes (RenderParams::adapt)
template <bool SMEM, bool COUNT, bool SHARE, bool SSTACK, Twin TWIN, bool ADAPT = false>
__global__ void __launch_bounds__(kTraceThreads, 1) traceKernel(const __grid_constant__ RenderParams p)
{
	extern __shared__ __align__(128) float4 smemScene[];
	// shared-window address of the dynamic shared memory, made opaque to the compiler: left alone it RE-DERIVES the address at
	// every use (S2UR SR_CgaCtaId, UMOV, UIADD3, ULEA ... five issue slots per primitive test) instead of keeping one register
	uint32_t smemBase = uint32_t(__cvta_generic_to_shared(smemScene));
	asm volatile("" : "+r"(smemBase));
	// SSTACK: this thread's column of the shared-memory traversal stack (trace_device.cuh TravStack<true>), behind the scene copy
	// (pinning this address, or the warp's index, in a register - as is done for smemBase - was measured: no gain / +1.3 ms; the
	// compiler recomputes both where they are used)
	const uint32_t stackColumn = SSTACK ? smemBase + p.stackOffset + threadIdx.x * 4u : 0u;
	__shared__ uint64_t mbar;
	SceneView<SMEM> sv;
	if constexpr (SMEM)
	{
		stageSceneToSmem(smemScene, p.scene.sceneBlob, (p.scene.nodeCount + p.scene.primCount) * 64u + p.scene.primCount * uint32_t(sizeof(Mat)), &mbar);
		sv.nodes = reinterpret_cast<const float4 *>(uintptr_t(smemBase));
		sv.prims = sv.nodes + size_t(p.scene.nodeCount) * 4;
		sv.globalCount = p.scene.globalCount;
	}
	else
	{
		sv.nodes = p.scene.sceneBlob;
		sv.prims = p.scene.sceneBlob + size_t(p.scene.nodeCount) * 4;
		sv.globalCount = p.scene.globalCount;
	}
	// the material table sits behind the primitives, in the shared-memory copy too: the three quads of a material are read once per
	// path segment, and from L1 / L2 they were a long-scoreboard stall at the head of every shade
	const float4 *const matTable = sv.prims + size_t(p.scene.primCount) * 4;

	// SHARE: the leaves the camera rays of the warp's pixel can reach (beamLeaves), nearest first
	__shared__ BeamEntry beamList[SHARE ? kTraceThreads / 32 : 1][kBeamMax];
	__shared__ BeamBox beamBoxes[SHARE && !SMEM ? kTraceThreads / 32 : 1][kBeamMax]; // scenes in global memory: the leaves' boxes (trace_device.cuh BeamBox)
	int nBeam = -1;
	__shared__ float2 pixelXY[SHARE ? kTraceThreads / 32 : 1]; // SHARE: (x, y) of the warp's pixel, once per pixel instead of once per sample

	const uint32_t lane = threadIdx.x & 31u;
	// the work counter hands out LOCAL indices: pixel = local * pixelStride + pixelOffset (all pixels for stride 1)
	const uint32_t allPixels = p.width * p.height;
	const uint32_t totalPixels = allPixels > p.pixelOffset ? (allPixels - p.pixelOffset + p.pixelStride - 1u) / p.pixelStride : 0u;
	const float invW = 1.0f / float(p.width), invH = 1.0f / float(p.height);
	const V3 camO = mk(p.cam.origin[0], p.cam.origin[1], p.cam.origin[2]);

	uint32_t pixel = kInvalid, sample = p.spp;
	bool active = true, alive = false;
	V3 color = mk(0.0f, 0.0f, 0.0f);
	V3 ro = camO, rd = mk(0.0f, 0.0f, 1.0f), thr = mk(1.0f, 1.0f, 1.0f), L = mk(0.0f, 0.0f, 0.0f);
	uint32_t bounce = 0, rz = 0, rw = 0, sampleIdx = 0;
	uint32_t rays = 0, nodeVisits = 0, primTests = 0, shades = 0, misses = 0;
	float lastPdf = 0.0f;   // EnvIS / LightIS: pdf with which the BSDF sampled the direction the lane is tracing (weights the sky at a miss, an emitter at a hit)
	uint32_t wNext = p.spp; // SHARE: next sample of the warp's pixel to hand out (warp-uniform)
	// ADAPT: the pixel's current interval (warp-uniform; it ends at the next checkpoint); the luminance y of the lane's path, the lane's sums
	// of y and y^2
	uint32_t ckIdx = 0;
	float yPath = 0.0f, s1 = 0.0f, s2 = 0.0f;
	unsigned long long passStat[6] = { 0, 0, 0, 0, 0, 0 }; // COUNT + SHARE (lane 0): camera passes, lanes, clocks; scattered passes, lanes, clocks
	unsigned long long travClk[2] = { 0, 0 };               // COUNT + SHARE: clocks up to the end of the traversal, camera / scattered passes
	const long long kernelT0 = COUNT && SHARE ? clock64() : 0;

	while (true)
	{
		bool generate;
		uint32_t nGen = 0; // SHARE: lanes that start a new sample in this pass (warp-uniform)
		if constexpr (SHARE)
		{
			// ---- the 32 lanes of the warp work on the SAME pixel: a lane without a path takes the pixel's next sample.
			// Camera rays of one warp are then (nearly) the same ray, the first hits the same primitive, the scattered rays
			// start from the same place: coherent node fetches (shared-memory broadcast) and fewer divergent branches ----
			generate = false;
			nGen = 0;
			const uint32_t needMask = __ballot_sync(0xffffffffu, !alive);
			if (needMask)
			{
				// hand out new samples only to groups of >= regenLow idle lanes (or when nobody is left tracing): the camera
				// rays of one group are nearly the same ray and stay in step through their first hit.  Everything here but the
				// lane's own place in the group is warp-uniform: one vote per pass, the rest is arithmetic on its result
				const uint32_t idle = uint32_t(__popc(needMask));
				// (each form written out on its own here and at the stratification below: a shared statement moved the register allocation of
				// the instantiations without ADAPT)
				if constexpr (ADAPT)
				{
					// samples up to the pixel's next checkpoint
					const uint32_t end = p.adapt[ckIdx].end;
					if (pixel != kInvalid && wNext < end && (idle >= p.regenLow || needMask == 0xffffffffu || end - wNext < 32u))
					{
						nGen = min(idle, end - wNext);
						const uint32_t place = __popc(needMask & ((1u << lane) - 1u));
						if (!alive && place < nGen)
						{
							sample = wNext + place;
							generate = true;
						}
						wNext += nGen;
					}
				}
				else if (pixel != kInvalid && wNext < p.spp && (idle >= p.regenLow || needMask == 0xffffffffu || p.spp - wNext < 32u))
				{
					nGen = min(idle, p.spp - wNext);
					const uint32_t place = __popc(needMask & ((1u << lane) - 1u));
					if (!alive && place < nGen)
					{
						sample = wNext + place;
						generate = true;
					}
					wNext += nGen;
				}
				if (needMask == 0xffffffffu && nGen == 0u)
				{
					// the pixel is complete: add the lanes' partial sums in a fixed order (butterfly), one lane writes
					if (pixel != kInvalid)
					{
						if constexpr (ADAPT)
						{
							// a checkpoint below spp: the stopping test on copies of the lanes' sums (the lanes keep their own for the
							// next checkpoint), warp-uniform.  var / n <= (tau x max(mean, floor))^2 is the test of the standard error
							// without a square root; 1 / n and 1 / (n (n - 1)) come from the host
							if (wNext < p.spp)
							{
								float a = s1, b = s2;
#pragma unroll
								for (int o = 16; o > 0; o >>= 1)
								{
									a += __shfl_xor_sync(0xffffffffu, a, o);
									b += __shfl_xor_sync(0xffffffffu, b, o);
								}
								const AdaptInterval &iv = p.adapt[ckIdx];
								const float se2 = fmaxf(b - a * a * iv.invN, 0.0f) * iv.invNN1;
								const float bound = p.adaptTau * fmaxf(a * iv.invN, p.adaptFloor);
								if (!(se2 <= bound * bound))
								{
									++ckIdx; // the same pixel: its beam list and pixelXY stay
									continue;
								}
							}
						}
#pragma unroll
						for (int o = 16; o > 0; o >>= 1)
						{
							color.x += __shfl_xor_sync(0xffffffffu, color.x, o);
							color.y += __shfl_xor_sync(0xffffffffu, color.y, o);
							color.z += __shfl_xor_sync(0xffffffffu, color.z, o);
						}
						if constexpr (ADAPT)
						{
							// the sum of n samples scaled to spp (x spp / n, worked out by the host; not at all when n = spp): the
							// accumulation buffer holds mean x spp, as without the option
							if (lane == 0)
							{
								if (wNext != p.spp) color = p.adapt[ckIdx].scale * color;
								storePixel(p, pixel, color);
								p.sampleCounts[pixel] = wNext;
								atomicAdd(&p.counters[kCtrSamples], (unsigned long long)wNext);
							}
						}
						else if (lane == 0) storePixel(p, pixel, color);
					}
					color = mk(0.0f, 0.0f, 0.0f);
					if constexpr (ADAPT)
					{
						s1 = s2 = 0.0f;
						ckIdx = 0;
					}
					unsigned long long next = 0;
					if (lane == 0) next = atomicAdd(&p.counters[kCtrWork], 1ull);
					next = __shfl_sync(0xffffffffu, next, 0);
					if (next >= totalPixels) break;
					pixel = uint32_t(next) * p.pixelStride + p.pixelOffset;
					wNext = 0;
					{
						uint32_t px, py;
						pixelToXY(pixel, p.width, p.height, px, py);
						if (lane == 0) pixelXY[(threadIdx.x >> 5)] = make_float2(float(px), float(py));
						__syncwarp();
					}
					if (p.beam)
					{
						uint32_t px, py;
						pixelToXY(pixel, p.width, p.height, px, py);
						const float m = 1.0f / 64.0f; // footprint widened: the jittered (s, t) are rounded products
						nBeam = beamLeaves<SMEM>(sv.nodes, p.scene.treeNodeCount, p.scene.nodeCount, p.cam, (float(px) - m) * invW, (float(px) + 1.0f + m) * invW, (float(py) - m) * invH,
						                         (float(py) + 1.0f + m) * invH, beamList[(threadIdx.x >> 5)], lane == 0, SMEM ? nullptr : beamBoxes[(threadIdx.x >> 5)]);
						__syncwarp();
					}
					continue;
				}
			}
		}
		else
		{
		// ---- accumulate + fetch the next pixel (warp-aggregated atomic: ballot + popc prefix) ----
		const bool need = active && !alive && sample == p.spp;
		if (need && pixel != kInvalid) storePixel(p, pixel, color);
		const uint32_t needMask = __ballot_sync(0xffffffffu, need);
		if (needMask)
		{
			const uint32_t leader = __ffs(needMask) - 1;
			unsigned long long base = 0;
			if (lane == leader) base = atomicAdd(&p.counters[kCtrWork], (unsigned long long)__popc(needMask));
			base = __shfl_sync(0xffffffffu, base, leader);
			if (need)
			{
				const unsigned long long mine = base + __popc(needMask & ((1u << lane) - 1u));
				if (mine >= totalPixels) { active = false; pixel = kInvalid; }
				else { pixel = uint32_t(mine) * p.pixelStride + p.pixelOffset; sample = 0; color = mk(0.0f, 0.0f, 0.0f); }
			}
		}
		if (!__any_sync(0xffffffffu, active)) break;
		generate = active && !alive;
		}

		bool takePart = SHARE ? (alive || generate) : active;
		if constexpr (SHARE)
		{
			// a pass is EITHER for the camera rays just generated (coherent: same pixel, leaves from the pixel's beam list,
			// no tree walk, usually the same material) OR for the scattered rays, where every live lane then walks the tree
			// together.  Mixed passes kept ~11 of 32 lanes in the node loop: the lanes with camera rays had nothing to walk.
			if (nGen != 0u) takePart = generate;
		}
		// COUNT + SHARE: passes, participating lanes and clocks per pass kind (tools/exp.py prints them)
		long long passT0 = 0;
		bool camPassNow = false;
		if constexpr (COUNT && SHARE)
		{
			camPassNow = __any_sync(0xffffffffu, generate);
			const uint32_t part = __popc(__ballot_sync(0xffffffffu, takePart));
			if (lane == 0) { passStat[camPassNow ? 0 : 3] += 1; passStat[camPassNow ? 1 : 4] += part; }
			passT0 = clock64();
		}
		if (takePart)
		{
			// ---- generate (trace.cu:187-192) ----
			if (generate)
			{
				sampleIdx = p.sampleOffset + sample * p.sampleStride;
				const uint4 r = philox4x32_10_keyed(pixel, sampleIdx, 0u, 0u, p.philoxKeys);
				float pxf, pyf;
				if constexpr (SHARE) { const float2 xy = pixelXY[(threadIdx.x >> 5)]; pxf = xy.x; pyf = xy.y; }
				else
				{
					uint32_t px, py;
					pixelToXY(pixel, p.width, p.height, px, py);
					pxf = float(px); pyf = float(py);
				}
				float u = (pxf + uniform01(r.x)) * invW; // trace.cu:190
				float v = (pyf + uniform01(r.y)) * invH;
				// option "jitter" = 0 (parity aid): every sample through the pixel centre, u = (x + 0.5) / W with the IEEE division of the
				// reference's primary pass - read from two small tables the host worked out (a division routine here, even out of
				// line, cost the hot loop 2 %: its call constrains the register allocation of everything around it)
				if constexpr (TWIN == Twin::Aids)
					if (p.aids & kAidPixelCentre) { u = __ldg(p.centreU + __float2uint_rz(pxf)); v = __ldg(p.centreV + __float2uint_rz(pyf)); }
				rz = r.z; rw = r.w;
				if constexpr (SHARE)
				{
					// first-bounce stratification: the cell of this sample (its local index / samples per cell) becomes the top bits of
					// the two randoms of the first scattering direction, the Philox draw fills the bits below (RenderParams::strataPer)
					// (ADAPT: the sample's index within its interval, and the interval's own grid)
					if constexpr (ADAPT)
					{
						const AdaptInterval &iv = p.adapt[ckIdx];
						stratify(sample - iv.start, iv.strataPer, iv.strataBitsA, iv.strataBitsB, iv.strataInvPer, rz, rw);
					}
					else if (sample < (p.strataPer << (p.strataBitsA + p.strataBitsB)))
					{
						const uint32_t cell = __float2uint_rz((__uint2float_rn(sample) + 0.5f) * p.strataInvPer);
						const uint32_t a = cell >> p.strataBitsB, bMask = (1u << p.strataBitsB) - 1u;
						const uint32_t b = (a & 1u) ? bMask - (cell & bMask) : (cell & bMask); // snake: neighbouring cells are neighbouring directions
						rz = (a << (32u - p.strataBitsA)) | (rz >> p.strataBitsA);
						rw = (b << (32u - p.strataBitsB)) | (rw >> p.strataBitsB);
					}
				}
				ro = camO;
				// IEEE square root and division here, as in the reference's Camera::getRay: far from an object the quadratic of the
				// primitive test cancels ~7 digits, so a direction that differs in its last bit re-rolls which silhouette pixels
				// hit - with the exact direction (and toLocalOD's rounding order) the render kernel's first hits are the reference's
				rd = cameraDir<2>(p.cam, u, v);
				thr = mk(1.0f, 1.0f, 1.0f);
				L = mk(0.0f, 0.0f, 0.0f);
				if constexpr (ADAPT) yPath = 0.0f;
				bounce = 0;
				alive = true;
			}

			// ---- traverse + intersect (trace.cu:112) ----
			++rays;
			const Hit h = closestHitWW<SMEM, COUNT, kHotExact, SSTACK>(sv, ro, rd, 0.001f, nodeVisits, primTests, beamList[SHARE ? (threadIdx.x >> 5) : 0],
			                                                           SHARE && bounce == 0 ? nBeam : -1, stackColumn, SMEM ? nullptr : beamBoxes[SHARE ? (threadIdx.x >> 5) : 0]);
			if constexpr (TWIN == Twin::Aids)
			{
				// parity aid: what THIS kernel's traversal found for the camera ray (scene-order index, t), per pixel
				if ((p.aids & kAidFirstHit) && bounce == 0)
				{
					p.firstHitIndex[pixel] = h.prim < 0 ? -1 : int32_t(primSceneIndex(sv.ld(sv.prims + h.prim * 4 + 3)));
					p.firstHitT[pixel] = h.prim < 0 ? 0.0f : h.t;
				}
			}

			if constexpr (COUNT && SHARE)
			{
				// clocks of the traversal part of the pass, as seen by the first participating lane (debug statistics)
				if (lane == uint32_t(__ffs(__activemask()) - 1)) travClk[camPassNow ? 0 : 1] += (unsigned long long)(clock64() - passT0);
			}
			bool terminate;
			if (h.prim < 0)
			{
				// ---- environment miss (trace.cu:115-134) ----
				if (COUNT) ++misses;
				if (p.scene.skybox != 0)
				{
					// (both inlined: as calls - one copy each, shared with the texture-coordinate code - they cost the hot loop 3 %: two
					// call / return pairs per miss, and the calling convention fixes registers around them)
					const float theta = fastAcos(rd.y), phi = fastAtan2Inline(rd.z, rd.x);
					V3 sky = texLookup(p.scene.textures, p.scene.skybox, phi * (0.5f / PT_PI), theta * (1.0f / PT_PI));
					if constexpr (TWIN == Twin::EnvIS)
					{
						// a scattered ray that reaches the sky: the direction could also have come from the sky's own distribution
						// (balance heuristic; the camera ray's miss has no such rival and keeps weight 1)
						if (bounce != 0u) sky = balanceWeight(lastPdf, envPdf(p.scene.env, phi * (0.5f / PT_PI), theta * (1.0f / PT_PI), rd.y)) * sky;
					}
					accumulate<SHARE, ADAPT>(color, L, yPath, thr, sky);
				}
				terminate = true;
			}
			else
			{
				// ---- shade / sample (trace.cu:136-151) ----
				const float4 *mp = matTable + h.prim * 3;
				const float4 m1 = sv.ld(mp + 1);
				V3 emitted = mk(m1.x, m1.y, m1.z); // getEmitted, Material.inl:62-65
				if constexpr (TWIN == Twin::LightIS)
				{
					// a scattered ray that hits an emitter: the point could also have come from the light sample of the vertex it left
					// (balance heuristic; the camera ray's hit has no such rival and keeps weight 1).  Mat::pad[0] = emitter index + 1
					const uint32_t emitter = __float_as_uint(sv.ld(mp + 2).z);
					if (bounce != 0u && emitter != 0u) emitted = balanceWeight(lastPdf, lightPdfHit<SMEM>(p.lights, sv, emitter - 1u, h.prim, ro, rd, h.t)) * emitted;
				}
				accumulate<SHARE, ADAPT>(color, L, yPath, thr, emitted);
				terminate = true;
				// The last segment of a path only contributes what it hits: the direction the reference still samples there
				// (trace.cu:139-151 in its fifth loop trip) is never traced and its weight never reaches the image - no normal,
				// texture tap or BSDF sample for it.
				if (bounce + 1u < p.maxBounces)
				{
					if (COUNT) ++shades;
					const Surface s = surfaceAt<SMEM>(sv, h.prim, ro, rd, h.t);
					const float4 m0 = sv.ld(mp), m2 = sv.ld(mp + 2);
					const uint32_t tex = __float_as_uint(m2.x), mtype = __float_as_uint(m2.y);
					const V3 base = baseColour(p.scene, m0, tex, s.u, s.v);
					float rnd0, rnd1;
					if (bounce == 0) { rnd0 = uniform01(rz); rnd1 = uniform01(rw); }
					else if (bounce & 1u)
					{
						const uint4 r = philox4x32_10_keyed(pixel, sampleIdx, (bounce + 1u) >> 1, 0u, p.philoxKeys);
						rnd0 = uniform01(r.x); rnd1 = uniform01(r.y);
						rz = r.z; rw = r.w;
					}
					else { rnd0 = uniform01(rz); rnd1 = uniform01(rw); }
					V3 wi, weight;
					bool scattered;
					if constexpr (TWIN == Twin::EnvIS)
					{
						const Frame fr = makeFrame(s.n);
						const V3 Vv = toTangent(fr, -rd);
						// one direction from the sky's distribution (its own Philox stream: fourth counter word 1, slot = bounce - the
						// draws of the path itself are those of a render without "env_is"), the same f and pdf the BSDF sample would
						// have had for it, and a ray towards it: sky x f x cos / (pdf_sky + pdf_bsdf) if nothing is in the way
						const uint4 q = philox4x32_10_keyed(pixel, sampleIdx, bounce, 1u, p.philoxKeys);
						float lu, lv, pe;
						const V3 wl = sampleEnv(p.scene.env, q.x, q.y, q.z, lu, lv, pe);
						const V3 sl = toTangent(fr, wl);
						V3 attL;
						float pbL;
						V3 contrib = mk(0.0f, 0.0f, 0.0f);
						const bool lit = sl.z > 0.0f && evalMaterial(mtype, base, m0.w, m1.w, Vv, sl, attL, pbL);
						if (lit)
						{
							const V3 sky = texLookup(p.scene.textures, p.scene.skybox, lu, lv);
							contrib = thr * ((sl.z * rcpApprox(pe + pbL)) * attL) * sky;
						}
						// (the BSDF sample first, the shadow ray behind it: frame, view vector and material are dead by then and only
						// the light sample's direction and value live across the walk)
						scattered = sampleMaterial(mtype, base, m0.w, m1.w, fr, Vv, rnd0, rnd1, wi, weight, &lastPdf);
						if (lit)
						{
							++rays;
							uint32_t nv = 0, pt = 0;
							const Hit hs = closestHitWW<SMEM, false, kHotExact, SSTACK, true>(sv, s.p, wl, 0.001f, nv, pt, beamList[0], -1, stackColumn, nullptr);
							if (hs.prim < 0) accumulate<SHARE, ADAPT>(color, L, yPath, contrib, mk(1.0f, 1.0f, 1.0f));
						}
					}
					else if constexpr (TWIN == Twin::LightIS)
					{
						const Frame fr = makeFrame(s.n);
						const V3 Vv = toTangent(fr, -rd);
						// one point on an emitter (its own Philox stream: fourth counter word 2, slot = bounce - the draws of the path
						// itself are those of a render without "light_is"), the f and pdf the BSDF sample would have had for its
						// direction, and a shadow ray that stops short of it: Le x f x cos / (pdf_light + pdf_bsdf) if nothing is in the way
						const uint4 q = philox4x32_10_keyed(pixel, sampleIdx, bounce, 2u, p.philoxKeys);
						V3 wl;
						float dist, pl;
						int lprim;
						const bool onLight = sampleLight<SMEM>(p.lights, sv, q, s.p, wl, dist, pl, lprim);
						const V3 sl = toTangent(fr, wl);
						V3 attL;
						float pbL;
						V3 contrib = mk(0.0f, 0.0f, 0.0f);
						const bool lit = onLight && sl.z > 0.0f && evalMaterial(mtype, base, m0.w, m1.w, Vv, sl, attL, pbL);
						if (lit)
						{
							const float4 le = sv.ld(matTable + lprim * 3 + 1);
							contrib = thr * ((sl.z * rcpApprox(pl + pbL)) * attL) * mk(le.x, le.y, le.z);
						}
						scattered = sampleMaterial(mtype, base, m0.w, m1.w, fr, Vv, rnd0, rnd1, wi, weight, &lastPdf);
						if (lit)
						{
							++rays;
							uint32_t nv = 0, pt = 0;
							const Hit hs = closestHitWW<SMEM, false, kHotExact, SSTACK, true, true>(sv, s.p, wl, 0.001f, nv, pt, beamList[0], -1, stackColumn, nullptr,
							                                                                      dist * (1.0f - 1e-4f));
							if (hs.prim < 0) accumulate<SHARE, ADAPT>(color, L, yPath, contrib, mk(1.0f, 1.0f, 1.0f));
						}
					}
					else scattered = sampleMaterial(mtype, base, m0.w, m1.w, s.n, rd, rnd0, rnd1, wi, weight);
					if (scattered)
					{
						thr = thr * weight;
						ro = s.p;
						rd = wi;
						++bounce;
						terminate = false;
					}
				}
			}
			if (terminate)
			{
				if constexpr (!SHARE) color = color + L;
				if constexpr (ADAPT)
				{
					s1 += yPath;
					s2 += yPath * yPath;
				}
				++sample;
				alive = false;
			}
		}
		if constexpr (COUNT && SHARE)
		{
			__syncwarp();
			if (lane == 0) passStat[camPassNow ? 2 : 5] += (unsigned long long)(clock64() - passT0);
		}
	}

	// ---- counters: one atomic per warp ----
	unsigned long long r64 = rays;
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) r64 += __shfl_xor_sync(0xffffffffu, r64, o);
	if (lane == 0) atomicAdd(&p.counters[kCtrRays], r64);
	if constexpr (COUNT && SHARE)
	{
		if (lane == 0)
		{
			for (int k = 0; k < 6; ++k) atomicAdd(&p.counters[kCtrPassStats + k], passStat[k]);
			atomicAdd(&p.counters[kCtrPassStats + 6], (unsigned long long)(clock64() - kernelT0));
		}
		atomicAdd(&p.counters[kCtrPassStats + 7], travClk[0]);
		atomicAdd(&p.counters[kCtrPassStats + 8], travClk[1]);
	}
	if (COUNT)
	{
		unsigned long long c[4] = { nodeVisits, primTests, shades, misses };
#pragma unroll
		for (int k = 0; k < 4; ++k)
		{
#pragma unroll
			for (int o = 16; o > 0; o >>= 1) c[k] += __shfl_xor_sync(0xffffffffu, c[k], o);
			if (lane == 0) atomicAdd(&p.counters[kCtrNodes + k], c[k]);
		}
	}
}

// ---------------------------------------------------------------------------------------------------------------
// deterministic primary pass / generic ray queries (parity gates) and the output stage
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) primaryKernel(SceneDev scene, CameraDev cam, uint32_t width, uint32_t height, int32_t *hitIndex, float *hitT)
{
	SceneView<false> sv;
	sv.nodes = scene.sceneBlob;
	sv.prims = scene.sceneBlob + size_t(scene.nodeCount) * 4;
	sv.globalCount = scene.globalCount;
	const uint32_t total = width * height;
	uint32_t nv = 0, pt = 0;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x)
	{
		const uint32_t x = i % width, y = i / width;
		const float u = divExact(float(x) + 0.5f, float(width)), v = divExact(float(y) + 0.5f, float(height));
		const V3 o = mk(cam.origin[0], cam.origin[1], cam.origin[2]);
		const V3 d = cameraDir(cam, u, v);
		const Hit h = closestHit<false, false>(sv, o, d, 0.001f, nv, pt);
		hitIndex[i] = h.prim < 0 ? -1 : int32_t(primSceneIndex(__ldg(sv.prims + h.prim * 4 + 3)));
		hitT[i] = h.prim < 0 ? 0.0f : h.t;
	}
}

__global__ void __launch_bounds__(kThreads) traceRaysKernel(SceneDev scene, uint32_t n, const float *origins, const float *directions, float tMin,
                                                            int32_t *hitIndex, float *hitT, float *hitNormal)
{
	SceneView<false> sv;
	sv.nodes = scene.sceneBlob;
	sv.prims = scene.sceneBlob + size_t(scene.nodeCount) * 4;
	sv.globalCount = scene.globalCount;
	uint32_t nv = 0, pt = 0;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
	{
		const V3 o = mk(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2]);
		const V3 d = mk(directions[3 * i], directions[3 * i + 1], directions[3 * i + 2]);
		const Hit h = closestHit<false, false>(sv, o, d, tMin, nv, pt);
		hitIndex[i] = h.prim < 0 ? -1 : int32_t(primSceneIndex(__ldg(sv.prims + h.prim * 4 + 3)));
		hitT[i] = h.prim < 0 ? 0.0f : h.t;
		if (hitNormal)
		{
			V3 nn = mk(0.0f, 0.0f, 0.0f);
			if (h.prim >= 0) nn = surfaceAt<false>(sv, h.prim, o, d, h.t).n;
			hitNormal[3 * i] = nn.x; hitNormal[3 * i + 1] = nn.y; hitNormal[3 * i + 2] = nn.z;
		}
	}
}

// the guide buffers of the denoiser (pt_render_aov): one thread per pixel, spp camera rays each, through the scene in global memory
// (a pass this short does not pay for the shared-memory staging); the means over the pixel's samples of the first hit's base colour
// (a miss counts as white; w = the fraction of rays that hit), its normal facing the ray (a miss counts as 0), and over the hits only
// its position (w = t)
__global__ void __launch_bounds__(kThreads) aovKernel(const __grid_constant__ AovParams p)
{
	const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
	if (pixel >= p.width * p.height) return;
	SceneView<false> sv;
	sv.nodes = p.scene.sceneBlob;
	sv.prims = p.scene.sceneBlob + size_t(p.scene.nodeCount) * 4;
	sv.globalCount = p.scene.globalCount;
	const float4 *const matTable = sv.prims + size_t(p.scene.primCount) * 4;
	uint32_t px, py;
	pixelToXY(pixel, p.width, p.height, px, py);
	const float invW = 1.0f / float(p.width), invH = 1.0f / float(p.height);
	const V3 o = mk(p.cam.origin[0], p.cam.origin[1], p.cam.origin[2]);
	V3 albedo = mk(0.0f, 0.0f, 0.0f), normal = mk(0.0f, 0.0f, 0.0f), position = mk(0.0f, 0.0f, 0.0f);
	float tSum = 0.0f;
	uint32_t hits = 0, nv = 0, pt = 0;
	for (uint32_t sample = 0; sample < p.spp; ++sample)
	{
		float u, v;
		if (p.centreU) { u = __ldg(p.centreU + px); v = __ldg(p.centreV + py); } // option "jitter" = 0: the rays of pt_primary_pass
		else
		{
			// a Philox stream of its own (fourth counter word 3): no draw of a render is reused
			const uint4 r = philox4x32_10_keyed(pixel, sample, 0u, 3u, p.philoxKeys);
			u = (float(px) + uniform01(r.x)) * invW;
			v = (float(py) + uniform01(r.y)) * invH;
		}
		const V3 d = cameraDir<2>(p.cam, u, v);
		// (the primitive tests with IEEE division and square root, as pt_primary_pass / pt_trace_rays: the guides of pixel-centre rays are
		// those queries' hits)
		const Hit h = closestHitWW<false, false, true>(sv, o, d, 0.001f, nv, pt);
		if (h.prim < 0)
		{
			albedo = albedo + mk(1.0f, 1.0f, 1.0f);
			continue;
		}
		const Surface s = surfaceAt<false>(sv, h.prim, o, d, h.t);
		const float4 *mp = matTable + h.prim * 3;
		albedo = albedo + baseColour(p.scene, __ldg(mp), __float_as_uint(__ldg(mp + 2).x), s.u, s.v);
		normal = normal + s.n;
		position = position + s.p;
		tSum += h.t;
		++hits;
	}
	const float n = float(p.spp), k = float(hits);
	p.albedo[pixel] = make_float4(albedo.x / n, albedo.y / n, albedo.z / n, k / n);
	p.normal[pixel] = make_float4(normal.x / n, normal.y / n, normal.z / n, 0.0f);
	p.position[pixel] = hits ? make_float4(position.x / k, position.y / k, position.z / k, tSum / k) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

// debugging aid: invSqrtExact against the library routines it stands in for
__global__ void invSqrtCheckKernel(uint32_t n, const float *x, float *fast, float *ieee)
{
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
	{
		fast[i] = invSqrtExact(x[i]);
		ieee[i] = divExact(1.0f, sqrtExact(x[i]));
	}
}
int launchInvSqrtCheck(uint32_t n, const float *x, float *fast, float *ieee, cudaStream_t stream)
{
	invSqrtCheckKernel<<<148 * 4, 256, 0, stream>>>(n, x, fast, ieee);
	return 1;
}

// tonemap (kernels/tonemap.cu:4-27): mean -> Reinhard -> gamma 1/2.2 -> truncating RGBA8.  HBM-bound: 16 B in, 4 B out.
__global__ void __launch_bounds__(kThreads) tonemapKernel(const float4 *__restrict__ accum, uchar4 *__restrict__ out, uint32_t pixels, float invSampleCount)
{
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < pixels; i += gridDim.x * blockDim.x)
	{
		const float4 a = __ldg(accum + i);
		float r = a.x * invSampleCount, g = a.y * invSampleCount, b = a.z * invSampleCount;
		r = r * (1.0f / (r + 1.0f)); g = g * (1.0f / (g + 1.0f)); b = b * (1.0f / (b + 1.0f));
		r = powf(r, 1.0f / 2.2f); g = powf(g, 1.0f / 2.2f); b = powf(b, 1.0f / 2.2f);
		out[i] = make_uchar4((unsigned char)(r * 255.0f), (unsigned char)(g * 255.0f), (unsigned char)(b * 255.0f), 255);
	}
}

// getHDRImageData's host loop (Pathtracer.cpp:307-312) on the device: all four channels scaled
__global__ void __launch_bounds__(kThreads) scaleKernel(const float4 *__restrict__ accum, float4 *__restrict__ out, uint32_t pixels, float scale)
{
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < pixels; i += gridDim.x * blockDim.x)
	{
		const float4 a = __ldg(accum + i);
		out[i] = make_float4(a.x * scale, a.y * scale, a.z * scale, a.w * scale);
	}
}

// ---------------------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------------------
// Launch one persistent wave.  Returns the number of kernels launched (1), 0 when this instantiation cannot run with
// `smemBytes` of dynamic shared memory (the caller then falls back to a configuration that needs less), -1 on a CUDA error.
template <typename K>
static int launchKernel(K kern, const RenderParams &p, const LaunchConfig &cfg, size_t smemBytes, cudaStream_t stream)
{
	// opt in whenever dynamic shared memory is used: the 48 KB default limit covers static + dynamic together, and the
	// one-pixel-per-warp kernels carry ~20 KB of static shared memory (beam lists)
	if (smemBytes > 0 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemBytes)) != cudaSuccess)
	{
		cudaGetLastError();
		return 0;
	}
	int blocksPerSm = 0;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocksPerSm, kern, kTraceThreads, smemBytes) != cudaSuccess)
	{
		cudaGetLastError();
		return 0;
	}
	if (blocksPerSm < 1) return 0;
	const int grid = cfg.smCount * blocksPerSm;
	kern<<<grid, kTraceThreads, smemBytes, stream>>>(p);
	return cudaPeekAtLastError() == cudaSuccess ? 1 : -1;
}

// static shared memory of the trace kernels (beam lists, per-warp pixel coordinates, barrier; + the beam boxes of
// the global-memory instantiations) - an upper bound; launchKernel has the last word (occupancy query)
constexpr size_t kStaticSmemBound = 8192; // (the instantiations that stage the scene carry 4.5 KB: the beam boxes belong to the global-memory ones)

// the instantiation of traceKernel for one scheduling form, stack form and twin; the twins exist without work counters only
// (count_work is ignored for them)
template <bool SHARE, bool SSTACK, Twin TWIN>
static int launchTraceKernel(const RenderParams &p, const LaunchConfig &cfg, bool smem, size_t smemBytes, cudaStream_t stream)
{
	if constexpr (TWIN == Twin::Plain)
		if (cfg.countWork)
			return launchKernel(smem ? traceKernel<true, true, SHARE, SSTACK, TWIN> : traceKernel<false, true, SHARE, SSTACK, TWIN>, p, cfg, smemBytes, stream);
	return launchKernel(smem ? traceKernel<true, false, SHARE, SSTACK, TWIN> : traceKernel<false, false, SHARE, SSTACK, TWIN>, p, cfg, smemBytes, stream);
}

// option "adaptive": the one-pixel-per-warp form without work counters, for the plain kernel and the env_is / light_is twins
template <bool SSTACK, Twin TWIN>
static int launchAdaptive(const RenderParams &p, const LaunchConfig &cfg, bool smem, size_t smemBytes, cudaStream_t stream)
{
	return launchKernel(smem ? traceKernel<true, false, true, SSTACK, TWIN, true> : traceKernel<false, false, true, SSTACK, TWIN, true>, p, cfg, smemBytes, stream);
}

template <bool SHARE, bool SSTACK>
static int launchTwin(const RenderParams &p, const LaunchConfig &cfg, bool smem, size_t smemBytes, cudaStream_t stream)
{
	if constexpr (SHARE)
	{
		if (cfg.adaptive)
		{
			switch (cfg.twin)
			{
			case Twin::EnvIS: return launchAdaptive<SSTACK, Twin::EnvIS>(p, cfg, smem, smemBytes, stream);
			case Twin::LightIS: return launchAdaptive<SSTACK, Twin::LightIS>(p, cfg, smem, smemBytes, stream);
			case Twin::Plain: return launchAdaptive<SSTACK, Twin::Plain>(p, cfg, smem, smemBytes, stream);
			default: return -1; // (pt_render refuses the parity aids with the option)
			}
		}
	}
	switch (cfg.twin)
	{
	case Twin::Aids: return launchTraceKernel<SHARE, SSTACK, Twin::Aids>(p, cfg, smem, smemBytes, stream);
	case Twin::EnvIS: return launchTraceKernel<SHARE, SSTACK, Twin::EnvIS>(p, cfg, smem, smemBytes, stream);
	case Twin::LightIS: return launchTraceKernel<SHARE, SSTACK, Twin::LightIS>(p, cfg, smem, smemBytes, stream);
	default: return launchTraceKernel<SHARE, SSTACK, Twin::Plain>(p, cfg, smem, smemBytes, stream);
	}
}

int launchTrace(const RenderParams &pIn, const LaunchConfig &cfg, cudaStream_t stream, int *usedSmem)
{
	RenderParams p = pIn;
	const size_t sceneBytes = (size_t(p.scene.nodeCount) + p.scene.primCount) * 64 + size_t(p.scene.primCount) * sizeof(Mat); // nodes | primitives | materials
	// one pixel per warp: camera passes and scattered passes alternate
	const bool share = cfg.adaptive || onePixelPerWarp(cfg, p.spp);
	const size_t stackBytes = size_t(cfg.stackLevels) * kStackStride;
	// what goes into shared memory: the scene when it fits (a scene larger than the opt-in limit stays in L2/HBM), the traversal
	// stack when it fits beside it
	bool smem = cfg.smemScene && sceneBytes + kStaticSmemBound <= cfg.maxSmemOptin;
	bool sstack = cfg.smemStack != 0 && cfg.stackLevels > 0 && (smem ? sceneBytes : 0) + stackBytes + kStaticSmemBound <= cfg.maxSmemOptin;
	for (int attempt = 0; attempt < 3; ++attempt)
	{
		if (usedSmem) *usedSmem = smem ? 1 : 0;
		p.stackOffset = uint32_t(smem ? sceneBytes : 0); // records are 64 bytes: the stack starts 16-byte aligned
		const size_t sb = (smem ? sceneBytes : 0) + (sstack ? stackBytes : 0);
		const int n = share ? (sstack ? launchTwin<true, true>(p, cfg, smem, sb, stream) : launchTwin<true, false>(p, cfg, smem, sb, stream))
		                    : (sstack ? launchTwin<false, true>(p, cfg, smem, sb, stream) : launchTwin<false, false>(p, cfg, smem, sb, stream));
		if (n != 0) return n;
		// the instantiation does not fit with this much shared memory: first without the stack, then without the scene
		if (sstack) sstack = false;
		else if (smem) smem = false;
		else return -1;
	}
	return -1;
}

int launchPrimary(const SceneDev &scene, const CameraDev &cam, uint32_t width, uint32_t height, int32_t *hitIndex, float *hitT, cudaStream_t stream)
{
	const uint32_t total = width * height;
	const int grid = int((total + kThreads - 1) / kThreads);
	primaryKernel<<<grid, kThreads, 0, stream>>>(scene, cam, width, height, hitIndex, hitT);
	return 1;
}

int launchTraceRays(const SceneDev &scene, size_t n, const float *origins, const float *directions, float tMin, int32_t *hitIndex, float *hitT,
                    float *hitNormal, cudaStream_t stream)
{
	const int grid = int((n + kThreads - 1) / kThreads);
	traceRaysKernel<<<grid, kThreads, 0, stream>>>(scene, uint32_t(n), origins, directions, tMin, hitIndex, hitT, hitNormal);
	return 1;
}

int launchAov(const AovParams &p, cudaStream_t stream)
{
	const uint32_t total = p.width * p.height;
	aovKernel<<<int((total + kThreads - 1) / kThreads), kThreads, 0, stream>>>(p);
	return 1;
}

int launchTonemap(const float4 *accum, uchar4 *out, uint32_t pixels, float invSampleCount, cudaStream_t stream)
{
	const int grid = int(min((pixels + kThreads - 1) / kThreads, 148u * 8u));
	tonemapKernel<<<grid, kThreads, 0, stream>>>(accum, out, pixels, invSampleCount);
	return 1;
}

int launchScale(const float4 *accum, float4 *out, uint32_t pixels, float scale, cudaStream_t stream)
{
	const int grid = int(min((pixels + kThreads - 1) / kThreads, 148u * 8u));
	scaleKernel<<<grid, kThreads, 0, stream>>>(accum, out, pixels, scale);
	return 1;
}

} // namespace ptb
