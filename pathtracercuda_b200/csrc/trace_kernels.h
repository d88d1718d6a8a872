// trace_kernels.h — launch interface of the CUDA trace path (implemented in trace_kernels.cu).
#pragma once
#include "pt_types.h"
#include <cuda_runtime.h>

namespace ptb
{

// counters[] layout (device, unsigned long long)
enum { kCtrWork = 0, kCtrRays = 1, kCtrNodes = 2, kCtrPrims = 3, kCtrShades = 4, kCtrMisses = 5,
       // pass statistics of the one-pixel-per-warp kernel (count_work = 1), 9 slots from kCtrPassStats: camera passes, their lanes,
       // their clocks; scattered passes, lanes, clocks; kernel clocks; traversal clocks of camera / scattered passes
       kCtrPassStats = 8, kCtrCount = 24 };

// option "env_is": the sky's importance distribution (env_sampling.h), on the read-only path
struct EnvDev
{
	const uint2 *alias = nullptr; // per cell: (float bits of the acceptance threshold, alias cell)
	const float *density = nullptr; // per cell: P(cell) cols rows / (2 pi^2); solid-angle pdf = density / sin(theta)
	uint32_t cols = 0, rows = 0;
};

// option "light_is": the emitter table (light_sampling.h LightRec, 64 bytes each), on the read-only path
struct LightDev
{
	const float4 *recs = nullptr; // 4 quads per emitter
	uint32_t count = 0;
};

struct SceneDev
{
	const float4 *sceneBlob = nullptr; // [nodes | prims | materials], 16-byte records, one allocation (bulk-copied to smem)
	const Mat *mats = nullptr;         // = the third part of the blob
	const TexDesc *textures = nullptr;
	uint32_t nodeCount = 0, primCount = 0, texCount = 0, skybox = 0;
	uint32_t globalCount = 0; // prims[0..globalCount): tested by every ray before the traversal (pt_types.h)
	uint32_t treeNodeCount = 0; // nodes[treeNodeCount..nodeCount): boxes of the hoisted primitives, for the pixel-beam walk only
	EnvDev env;                 // set (alias != nullptr) when the launch samples the sky directly (option "env_is")
};

struct RenderParams
{
	SceneDev scene;
	CameraDev cam;
	float4 *accum;
	unsigned long long *counters;
	uint32_t width, height, spp, ignoreHistory;
	uint32_t sampleOffset, sampleStride;
	uint32_t pixelOffset = 0, pixelStride = 1; // this launch renders pixels offset, offset + stride, ... (multi-GPU pixel partition)
	uint32_t seedLo, seedHi;
	// the ten round keys of Philox4x32-10 (key + i * Weyl constants), worked out once on the host: in the kernel they are
	// constant-bank operands of the rounds' XORs instead of two additions per round (a third of the generator's instructions)
	uint32_t philoxKeys[20];
	uint32_t maxBounces;
	uint32_t regenLow = 1; // one-pixel-per-warp kernel: idle lanes wait until this many can start new samples together
	uint32_t beam = 0;     // one-pixel-per-warp kernel: camera rays take their leaves from the pixel's beam list (trace_device.cuh)
	// First-bounce stratification (one-pixel-per-warp kernels).  The launch's first strataPer << (strataBitsA + strataBitsB)
	// samples of a pixel (local index m) take the first scattering direction's two randoms from cell m / strataPer of a
	// 2^bitsA x 2^bitsB grid over the unit square (top bits = the cell, low bits = the Philox draw), so that (a) every cell gets
	// exactly strataPer samples - stratified sampling of the first bounce, same expectation, never more variance - and (b) the
	// lanes of a pass, which hold consecutive m, scatter into the SAME cell: what the sample sort bought, without sort, scratch
	// or second Philox evaluation.  strataPer = 0: off.
	uint32_t strataPer = 0, strataBitsA = 0, strataBitsB = 0;
	float strataInvPer = 0.0f;
	// parity aid (option "jitter" = 0): every sample through the pixel centre; centreU[x] = (x + 0.5f) / W, centreV[y] = (y + 0.5f) / H with
	// IEEE division, like the reference's primary pass - tables made by the host (pt_render); nullptr = jittered samples
	const float *centreU = nullptr, *centreV = nullptr;
	uint32_t aids = 0;              // kAid* bits: which parity aids are on (ONE warp-uniform test per site in the kernel)
	int32_t *firstHitIndex = nullptr; // parity aid: scene index (-1: miss) and t of the camera ray's closest hit, per pixel, written by
	float *firstHitT = nullptr;       // the render kernel itself (with noJitter every sample of a pixel writes the same values)
	float alpha = 1.0f;             // what the kernel writes to the accumulation buffer's fourth channel (trace.cu:198 writes 1); a multi-GPU
	                                // sample partition lets only its first device write 1, so that the summed alpha is 1 as on one GPU
	uint32_t stackOffset = 0;       // SSTACK kernels: byte offset of the shared-memory traversal stack in dynamic shared memory
	// (launch parameters added from here on go at the END: the constant-bank offsets of the fields above stay where the existing
	// kernels read them)
	LightDev lights; // set (count != 0) when the launch samples the emitters directly (option "light_is")
};

constexpr uint32_t kAidPixelCentre = 1u, kAidFirstHit = 2u;

struct LaunchConfig
{
	int smCount = 148;
	int smemScene = 1;   // stage the scene in shared memory when it fits
	int countWork = 0;   // node/prim/shade/miss counters
	int variant = 0;     // kernel variant (0 = default: 12 for spp >= 64, else 4.  4: one pixel per lane, while-while traversal; 1: if/else traversal;
	                     //  5: + leaf parking; 8: one pixel per WARP (lanes = samples), while-while; 9/10: its other traversals;
	                     //  12: 8 with separate passes for camera rays and scattered rays)
	int regenLow = 0;    // see RenderParams::regenLow (0 = default)
	int beam = -1;       // pixel beams for the camera rays of the one-pixel-per-warp kernel: 1 on, 0 off, -1 = on from 128 spp
	int stratify = -1;   // first-bounce stratification (RenderParams::strataPer): 1 on, 0 off, -1 = on from 128 spp (one-pixel-per-warp kernels)
	int strataK = 0;     // experiments: log2 of the cell count (0 = the rule of pt_render: at least 32 samples per cell, at most 128 cells)
	int smemStack = -1;  // traversal stack in shared memory (TravStack<true>): 1 on, 0 off, -1 = on when it fits beside the scene
	int envIS = 0;       // next-event estimation of the sky with multiple importance sampling (RenderParams::scene.env; one-pixel-per-warp kernel)
	int lightIS = 0;     // next-event estimation of the emitters with multiple importance sampling (RenderParams::lights; variants 4 / 12)
	int stackLevels = 0; // BVH depth + 2: levels the shared-memory stack needs (set by pt_render from the compiled scene)
	size_t maxSmemOptin = 0;
};

// Returns the number of kernels launched; *usedSmem = 1 when the scene was staged in shared memory.
int launchTrace(const RenderParams &p, const LaunchConfig &cfg, cudaStream_t stream, int *usedSmem);
int launchPrimary(const SceneDev &scene, const CameraDev &cam, uint32_t width, uint32_t height, int32_t *hitIndex, float *hitT, cudaStream_t stream);
int launchTraceRays(const SceneDev &scene, size_t n, const float *origins, const float *directions, float tMin, int32_t *hitIndex, float *hitT,
                    float *hitNormal, cudaStream_t stream);
int launchInvSqrtCheck(uint32_t n, const float *x, float *fast, float *ieee, cudaStream_t stream); // debugging aid
int launchTonemap(const float4 *accum, uchar4 *out, uint32_t pixels, float invSampleCount, cudaStream_t stream);
int launchScale(const float4 *accum, float4 *out, uint32_t pixels, float scale, cudaStream_t stream);

} // namespace ptb
