// pt_capi.cu — the C ABI of include/pt_b200.h: a resource-owning context that mirrors the reference's `class Pathtracer`
// (Pathtracer.h:12-69, Pathtracer.cpp:30-339) method for method.  Blocking calls, one CUDA stream per context,
// no CPU fallback (pt_create fails without a device).
#include "../../include/pt_b200.h"
#include "image_io.h"
#include "env_sampling.h"
#include "light_sampling.h"
#include "scene_compile.h"
#include "scene_loader.h"
#include "trace_kernels.h"
#include <cmath>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <nccl.h>
#include <string>
#include <thread>
#include <vector>

using namespace ptb;

namespace
{
thread_local std::string g_lastError;
int setError(int code, const std::string &msg)
{
	g_lastError = msg;
	return code;
}
constexpr uint32_t kMaxTextures = 64; // MAX_TEXTURE_COUNT, Pathtracer.cpp:15
} // namespace

struct pt_context
{
	int device = 0;
	uint32_t width = 0, height = 0;
	cudaStream_t stream = nullptr;
	cudaEvent_t evStart = nullptr, evStop = nullptr;
	float4 *accum = nullptr;
	bool ownAccum = true;
	float4 *scaledDev = nullptr;
	uchar4 *ldrDev = nullptr;
	float *hostHdr = nullptr;     // pinned
	uint8_t *hostLdr = nullptr;   // pinned
	unsigned long long *counters = nullptr;
	int32_t *firstHitIndex = nullptr; // option "first_hit": the render kernel's own first-hit (index, t) per pixel (parity aid)
	float *firstHitT = nullptr;
	bool firstHit = false, noJitter = false;
	// option "env_is": the sky's importance distribution (env_sampling.h), built for texture handle envHandle on first use
	bool envIS = false;
	uint32_t envHandle = 0;
	void *envAlias = nullptr;
	float *envDensity = nullptr;
	uint32_t envCols = 0, envRows = 0;
	// option "light_is": the emitter table of the current scene (light_sampling.h), built with the compiled scene
	bool lightIS = false;
	float4 *lightRecs = nullptr;
	uint32_t lightCount = 0;
	float *centreUV = nullptr; // option "jitter" = 0: pixel-centre coordinates (RenderParams::centreU / centreV), made on first use
	// scene
	float4 *sceneBlob = nullptr;
	Mat *mats = nullptr;
	uint32_t nodeCount = 0, treeNodeCount = 0, primCount = 0, bvhDepth = 0, globalCount = 0, maxGlobal = ptb::kMaxGlobalPrims;
	int bvhBuilder = ptb::kBuilderAuto; // option "bvh_builder" (scene_compile.h): SAH, from 2^19 objects the LBVH
	// textures
	std::vector<void *> texMem;
	TexDesc texHost[kMaxTextures];
	std::vector<cudaArray_t> texArrays;
	std::vector<cudaTextureObject_t> texObjects;
	int texUnit = 1; // filter textures with the texture unit (0: in software from linear memory)
	TexDesc *texDev = nullptr;
	uint32_t textureCount = 0, skybox = 0;
	// state mirrored from the reference
	float timingMs = 0.0f;
	uint32_t accumulatedFrames = 0;
	unsigned long long totalSamples = 0;
	// options
	uint64_t seed = 1984;
	uint32_t sampleOffset = 0, sampleStride = 1, sampleCursor = 0;
	uint32_t pixelOffset = 0, pixelStride = 1; // multi-GPU pixel partition: this context renders pixels offset, offset + stride, ...
	uint32_t framesPerSpp = 0, maxBounces = 5, maxLeaf = 4;
	LaunchConfig launch;
	pt_stats stats;
	unsigned long long rawCounters[ptb::kCtrCount] = {};
	// ---- multi-GPU (pt_create_multi).  This context is the ROOT: the first device of the mask, the one whose buffers the
	// image getters read.  `peers` are ordinary single-device contexts on the other devices; every call on the root is
	// carried out on all of them (scene, textures, options) or split over them (pt_render, one host thread per GPU).
	std::vector<pt_context *> peers;
	int partition = 0;            // how pt_render splits the work: 0 = pixels (device i: pixels i, i + N, ...), 1 = samples
	int exchange = -1;            // how the image comes together: 1 = peer-to-peer stores into the root's buffer (pixels only),
	                              // 0 = one ncclReduce of the float4 accumulation buffers, -1 = p2p when the devices allow it
	bool p2pReady = false;        // peer access root <- peers enabled
	struct NcclState *nccl = nullptr;
	float4 *reduced = nullptr;    // NCCL exchange: the sum over devices lands here (the per-device partial sums stay intact)
	const float4 *imageSource = nullptr; // what the image getters read: null = accum
	float reduceMs = 0.0f;        // device time of the last exchange (0 with peer-to-peer stores: there is none)
	unsigned long long jobSamples = 0; // samples per pixel / render calls of the whole job since the last restart
	uint32_t jobFrames = 0;
	float multiTraceMs = 0.0f;    // slowest device's trace time of the last pt_render
	pt_stats multiStats = {};     // statistics of the last pt_render summed over the devices
	float alpha = 1.0f;           // RenderParams::alpha
	bool skipPartitionClear = false; // p2p: the other devices write their pixels into this very buffer - nothing to zero
};

#define CK(expr)                                                                                                      \
	do                                                                                                                \
	{                                                                                                                 \
		cudaError_t e_ = (expr);                                                                                      \
		if (e_ != cudaSuccess)                                                                                        \
		{                                                                                                             \
			char buf[512];                                                                                            \
			snprintf(buf, sizeof buf, "CUDA error = %u at %s:%d '%s' (%s)", (unsigned)e_, __FILE__, __LINE__, #expr, cudaGetErrorString(e_)); \
			return setError(PT_E_CUDA, buf);                                                                          \
		}                                                                                                             \
	} while (0)

namespace
{
// device allocation freed on every return path
struct DevBuf
{
	void *p = nullptr;
	~DevBuf() { if (p) cudaFree(p); }
	cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes); }
	template <typename T> T *as() const { return static_cast<T *>(p); }
};
} // namespace

// NCCL is loaded at run time (dlopen, local scope), only when a multi-GPU context first needs a reduce: the library keeps
// no link-time dependency on it - a host process that already carries its own NCCL (PyTorch's) is left alone, and single-GPU
// users need none.  <nccl.h> is used for its types only.
struct NcclState
{
	void *lib = nullptr;
	ncclResult_t (*commInitAll)(ncclComm_t *, int, const int *) = nullptr;
	ncclResult_t (*commDestroy)(ncclComm_t) = nullptr;
	ncclResult_t (*groupStart)() = nullptr;
	ncclResult_t (*groupEnd)() = nullptr;
	ncclResult_t (*reduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
	const char *(*getErrorString)(ncclResult_t) = nullptr;
	std::vector<ncclComm_t> comms;
	cudaEvent_t ev0 = nullptr, ev1 = nullptr; // on the root's stream, around the reduce
	bool warm = false;                        // the communicators have run their first collective
};

// No C++ exception may cross the C boundary (std::bad_alloc from a huge scene or image would otherwise terminate the host)
#define PT_TRY try {
#define PT_CATCH(ret)                                                                                                 \
	}                                                                                                                 \
	catch (const std::bad_alloc &) { setError(PT_E_LIMIT, std::string(__func__) + ": out of memory"); return ret; }    \
	catch (const std::exception &e) { setError(PT_E_LIMIT, std::string(__func__) + ": " + e.what()); return ret; }     \
	catch (...) { setError(PT_E_LIMIT, std::string(__func__) + ": unknown exception"); return ret; }

extern "C"
{

const char *pt_last_error(void) { return g_lastError.c_str(); }
const char *pt_version(void) { return "pathtracercuda_b200 0.1 (sm_100a)"; }
void pt_free(void *p) { free(p); }

int pt_create(uint32_t width, uint32_t height, int device, pt_context **out)
{
	PT_TRY
	if (!out || width == 0 || height == 0) return setError(PT_E_INVALID, "pt_create: bad arguments");
	*out = nullptr;
	int count = 0;
	if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
	{
		cudaGetLastError();
		return setError(PT_E_NO_DEVICE, "pt_create: no CUDA device (this library has no CPU fallback)");
	}
	if (device < 0 || device >= count) return setError(PT_E_INVALID, "pt_create: device ordinal out of range");
	pt_context *c = new pt_context();
	c->device = device;
	c->width = width;
	c->height = height;
	memset(&c->stats, 0, sizeof c->stats);
	memset(c->texHost, 0, sizeof c->texHost);
	const size_t px = size_t(width) * height;
#define CKC(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { char buf[512]; snprintf(buf, sizeof buf, "CUDA error = %u at %s:%d '%s' (%s)", (unsigned)e_, __FILE__, __LINE__, #expr, cudaGetErrorString(e_)); g_lastError = buf; pt_destroy(c); return PT_E_CUDA; } } while (0)
	CKC(cudaSetDevice(device));
	// (two attributes, not cudaGetDeviceProperties: that call fills in everything the driver knows about the device and is one of
	// the slower ones of a process's start)
	int smCount = 0, smemOptin = 0;
	CKC(cudaDeviceGetAttribute(&smCount, cudaDevAttrMultiProcessorCount, device));
	CKC(cudaDeviceGetAttribute(&smemOptin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
	c->launch.smCount = smCount;
	c->launch.maxSmemOptin = size_t(smemOptin);
	CKC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	CKC(cudaEventCreate(&c->evStart));
	CKC(cudaEventCreate(&c->evStop));
	CKC(cudaMalloc(&c->accum, px * sizeof(float4)));
	CKC(cudaMemsetAsync(c->accum, 0, px * sizeof(float4), c->stream));
	// (the read-back buffers - device staging and pinned host memory for the HDR and the LDR image - are allocated by the first
	// getter that needs them: pinned allocations are slow, a peer context of a multi-GPU job never reads back, and a run that
	// writes a PNG does not need the 33 MB HDR pair)
	CKC(cudaMalloc(&c->counters, kCtrCount * sizeof(unsigned long long)));
	CKC(cudaMalloc(&c->texDev, kMaxTextures * sizeof(TexDesc)));
	CKC(cudaMemsetAsync(c->texDev, 0, kMaxTextures * sizeof(TexDesc), c->stream));
	CKC(cudaStreamSynchronize(c->stream));
#undef CKC
	*out = c;
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

int pt_create_multi(uint32_t width, uint32_t height, uint32_t device_mask, pt_context **out)
{
	PT_TRY
	if (!out || device_mask == 0) return setError(PT_E_INVALID, "pt_create_multi: bad arguments");
	*out = nullptr;
	std::vector<int> devs;
	for (int d = 0; d < 32; ++d)
		if (device_mask & (1u << d)) devs.push_back(d);
	pt_context *root = nullptr;
	int r = pt_create(width, height, devs[0], &root);
	if (r != PT_OK) return r;
	for (size_t i = 1; i < devs.size(); ++i)
	{
		pt_context *peer = nullptr;
		r = pt_create(width, height, devs[i], &peer);
		if (r != PT_OK) { const std::string e = g_lastError; pt_destroy(root); g_lastError = e; return r; }
		root->peers.push_back(peer);
	}
	// peer access root <- every other device: their kernels can then store finished pixels straight into the root's buffer
	root->p2pReady = !root->peers.empty();
	for (pt_context *peer : root->peers)
	{
		int can = 0;
		if (cudaSetDevice(peer->device) != cudaSuccess || cudaDeviceCanAccessPeer(&can, peer->device, root->device) != cudaSuccess || !can) { root->p2pReady = false; continue; }
		const cudaError_t e = cudaDeviceEnablePeerAccess(root->device, 0);
		if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) root->p2pReady = false;
		cudaGetLastError();
	}
	cudaSetDevice(root->device);
	*out = root;
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

int pt_get_multi_info(const pt_context *c, int *devices, int *peer_to_peer, float *trace_ms, float *exchange_ms)
{
	if (!c) return setError(PT_E_INVALID, "pt_get_multi_info: null context");
	if (devices) *devices = int(c->peers.size()) + 1;
	if (peer_to_peer) *peer_to_peer = (c->partition == 0 && c->p2pReady && c->exchange != 0) ? 1 : 0;
	if (trace_ms) *trace_ms = c->peers.empty() ? c->timingMs : c->multiTraceMs;
	if (exchange_ms) *exchange_ms = c->reduceMs;
	return PT_OK;
}

void pt_destroy(pt_context *c)
{
	if (!c) return;
	for (pt_context *peer : c->peers)
	{
		if (peer->accum == c->accum) { peer->accum = nullptr; peer->ownAccum = false; } // p2p: the buffer is the root's
		pt_destroy(peer);
	}
	c->peers.clear();
	if (c->nccl)
	{
		for (ncclComm_t comm : c->nccl->comms) if (comm && c->nccl->commDestroy) c->nccl->commDestroy(comm);
		cudaSetDevice(c->device);
		if (c->nccl->ev0) cudaEventDestroy(c->nccl->ev0);
		if (c->nccl->ev1) cudaEventDestroy(c->nccl->ev1);
		if (c->nccl->lib) dlclose(c->nccl->lib);
		delete c->nccl;
		c->nccl = nullptr;
	}
	cudaSetDevice(c->device);
	if (c->reduced) cudaFree(c->reduced);
	if (c->stream) cudaStreamSynchronize(c->stream);
	if (c->ownAccum && c->accum) cudaFree(c->accum);
	if (c->scaledDev) cudaFree(c->scaledDev);
	if (c->ldrDev) cudaFree(c->ldrDev);
	if (c->hostHdr) cudaFreeHost(c->hostHdr);
	if (c->hostLdr) cudaFreeHost(c->hostLdr);
	if (c->counters) cudaFree(c->counters);
	if (c->firstHitIndex) cudaFree(c->firstHitIndex);
	if (c->firstHitT) cudaFree(c->firstHitT);
	if (c->centreUV) cudaFree(c->centreUV);
	if (c->envAlias) cudaFree(c->envAlias);
	if (c->envDensity) cudaFree(c->envDensity);
	if (c->lightRecs) cudaFree(c->lightRecs);
	if (c->texDev) cudaFree(c->texDev);
	if (c->sceneBlob) cudaFree(c->sceneBlob); // (the material table lives in the same allocation)
	for (void *p : c->texMem) cudaFree(p);
	for (cudaTextureObject_t o : c->texObjects) cudaDestroyTextureObject(o);
	for (cudaArray_t a : c->texArrays) cudaFreeArray(a);
	if (c->evStart) cudaEventDestroy(c->evStart);
	if (c->evStop) cudaEventDestroy(c->evStop);
	if (c->stream) cudaStreamDestroy(c->stream);
	delete c;
}

// upload a compiled scene and its emitter table to one device (replaces the previous ones)
static int uploadScene(pt_context *c, const CompiledScene &cs, const LightTable &lt)
{
	CK(cudaSetDevice(c->device));
	CK(cudaStreamSynchronize(c->stream));
	if (c->sceneBlob) { CK(cudaFree(c->sceneBlob)); c->sceneBlob = nullptr; }
	if (c->lightRecs) { CK(cudaFree(c->lightRecs)); c->lightRecs = nullptr; }
	c->lightCount = 0;
	if (!lt.recs.empty())
	{
		CK(cudaMalloc(&c->lightRecs, lt.recs.size() * sizeof(LightRec)));
		CK(cudaMemcpyAsync(c->lightRecs, lt.recs.data(), lt.recs.size() * sizeof(LightRec), cudaMemcpyHostToDevice, c->stream));
		c->lightCount = uint32_t(lt.recs.size());
	}
	c->mats = nullptr;
	// one allocation, nodes | primitives | materials: a scene that fits is staged in shared memory whole, by one bulk copy
	const size_t nodeBytes = cs.nodes.size() * sizeof(Node), primBytes = cs.prims.size() * sizeof(Prim), matBytes = cs.mats.size() * sizeof(Mat);
	CK(cudaMalloc(&c->sceneBlob, nodeBytes + primBytes + matBytes));
	c->mats = reinterpret_cast<Mat *>(reinterpret_cast<char *>(c->sceneBlob) + nodeBytes + primBytes);
	CK(cudaMemcpyAsync(c->sceneBlob, cs.nodes.data(), nodeBytes, cudaMemcpyHostToDevice, c->stream));
	CK(cudaMemcpyAsync(reinterpret_cast<char *>(c->sceneBlob) + nodeBytes, cs.prims.data(), primBytes, cudaMemcpyHostToDevice, c->stream));
	CK(cudaMemcpyAsync(c->mats, cs.mats.data(), matBytes, cudaMemcpyHostToDevice, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	c->nodeCount = uint32_t(cs.nodes.size());
	c->primCount = uint32_t(cs.prims.size());
	c->globalCount = cs.globalCount;
	c->treeNodeCount = cs.treeNodeCount;
	c->bvhDepth = cs.depth;
	c->stats.bvh_nodes = c->treeNodeCount;
	c->stats.bvh_depth = c->bvhDepth;
	c->stats.scene_bytes = uint32_t(nodeBytes + primBytes + cs.mats.size() * sizeof(Mat));
	return PT_OK;
}

int pt_set_scene(pt_context *c, size_t count, const pt_object_desc *objects)
{
	PT_TRY
	if (!c) return setError(PT_E_INVALID, "pt_set_scene: null context");
	if (count == 0)
	{
		printf("Setting an empty scene is not allowed!\n"); // Pathtracer.cpp:115
		return PT_OK;
	}
	if (!objects) return setError(PT_E_INVALID, "pt_set_scene: null objects");
	CompiledScene cs;
	std::string err;
	if (!compileScene(count, objects, c->maxLeaf, cs, err, c->maxGlobal, nullptr, c->bvhBuilder)) return setError(PT_E_LIMIT, "pt_set_scene: " + err);
	LightTable lt;
	buildLightTable(cs, lt);
	// the BVH (and the emitter table) is built ONCE on the host; a multi-GPU context replicates the compiled scene on every device
	int r = uploadScene(c, cs, lt);
	for (size_t i = 0; r == PT_OK && i < c->peers.size(); ++i) r = uploadScene(c->peers[i], cs, lt);
	return r;
	PT_CATCH(PT_E_LIMIT)
}

int pt_set_scene_xform(pt_context *c, size_t count, const pt_object_xform_desc *objects)
{
	PT_TRY
	if (!c) return setError(PT_E_INVALID, "pt_set_scene_xform: null context");
	if (count == 0)
	{
		printf("Setting an empty scene is not allowed!\n"); // Pathtracer.cpp:115
		return PT_OK;
	}
	if (!objects) return setError(PT_E_INVALID, "pt_set_scene_xform: null objects");
	std::vector<pt_object_desc> descs(count);
	std::vector<ObjectXform> xf(count);
	for (size_t i = 0; i < count; ++i)
	{
		memset(&descs[i], 0, sizeof descs[i]);
		descs[i].type = objects[i].type;
		descs[i].scale[0] = descs[i].scale[1] = descs[i].scale[2] = 1.0f;
		descs[i].material = objects[i].material;
		memset(&xf[i], 0, sizeof xf[i]);
		memcpy(xf[i].w2l, objects[i].world_to_local, sizeof xf[i].w2l);
		memcpy(xf[i].bmin, objects[i].aabb_min, 12);
		memcpy(xf[i].bmax, objects[i].aabb_max, 12);
	}
	CompiledScene cs;
	std::string err;
	if (!compileScene(count, descs.data(), c->maxLeaf, cs, err, c->maxGlobal, xf.data(), c->bvhBuilder)) return setError(PT_E_LIMIT, "pt_set_scene_xform: " + err);
	LightTable lt;
	buildLightTable(cs, lt);
	int r = uploadScene(c, cs, lt);
	for (size_t i = 0; r == PT_OK && i < c->peers.size(); ++i) r = uploadScene(c->peers[i], cs, lt);
	return r;
	PT_CATCH(PT_E_LIMIT)
}

// device copy of the texture table; with tex_unit = 0 the texture objects are left out and the kernels filter in software
static int uploadTextureTable(pt_context *c)
{
	TexDesc tmp[kMaxTextures];
	memcpy(tmp, c->texHost, sizeof tmp);
	if (!c->texUnit)
		for (TexDesc &t : tmp) t.texObj = 0;
	if (cudaMemcpyAsync(c->texDev, tmp, sizeof tmp, cudaMemcpyHostToDevice, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
		return setError(PT_E_CUDA, "pt_load_texture: table upload failed");
	return PT_OK;
}

static uint32_t loadTextureMemOne(pt_context *c, uint32_t width, uint32_t height, int is_hdr, const void *rgba)
{
	PT_TRY
	if (!c || !rgba || width == 0 || height == 0) return 0;
	if (c->textureCount >= kMaxTextures) return 0; // Pathtracer.cpp:236-240
	if (cudaSetDevice(c->device) != cudaSuccess) return 0;
	const size_t bytes = size_t(width) * height * (is_hdr ? 16 : 4);
	void *dev = nullptr;
	if (cudaMalloc(&dev, bytes) != cudaSuccess) { setError(PT_E_CUDA, "pt_load_texture: cudaMalloc failed"); return 0; }
	if (cudaMemcpyAsync(dev, rgba, bytes, cudaMemcpyHostToDevice, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
	{
		cudaFree(dev);
		setError(PT_E_CUDA, "pt_load_texture: upload failed");
		return 0;
	}
	TexDesc &t = c->texHost[c->textureCount];
	t.texels = dev;
	t.width = width;
	t.height = height;
	t.isHdr = is_hdr ? 1u : 0u;
	t.pad = 0;
	t.texObj = 0;
	c->texMem.push_back(dev);
	// the same texels behind a texture object (Pathtracer.cpp:259-288: array, wrap U / clamp V, linear filter, normalised
	// coordinates; 8-bit texels read as normalised floats)
	{
		cudaChannelFormatDesc fmt = is_hdr ? cudaCreateChannelDesc<float4>() : cudaCreateChannelDesc<uchar4>();
		cudaArray_t arr = nullptr;
		cudaTextureObject_t obj = 0;
		bool ok = cudaMallocArray(&arr, &fmt, width, height) == cudaSuccess;
		const size_t pitch = size_t(width) * (is_hdr ? 16 : 4);
		ok = ok && cudaMemcpy2DToArray(arr, 0, 0, rgba, pitch, pitch, height, cudaMemcpyHostToDevice) == cudaSuccess;
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
			td.readMode = is_hdr ? cudaReadModeElementType : cudaReadModeNormalizedFloat;
			td.normalizedCoords = 1;
			ok = cudaCreateTextureObject(&obj, &rd, &td, nullptr) == cudaSuccess;
		}
		if (!ok)
		{
			if (arr) cudaFreeArray(arr);
			cudaGetLastError();
			setError(PT_E_CUDA, "pt_load_texture: texture object creation failed");
			return 0;
		}
		t.texObj = (unsigned long long)obj;
		c->texArrays.push_back(arr);
		c->texObjects.push_back(obj);
	}
	++c->textureCount;
	if (uploadTextureTable(c) != PT_OK) { --c->textureCount; return 0; }
	return c->textureCount;
	PT_CATCH(0u)
}

uint32_t pt_load_texture_mem(pt_context *c, uint32_t width, uint32_t height, int is_hdr, const void *rgba)
{
	const uint32_t h = loadTextureMemOne(c, width, height, is_hdr, rgba);
	if (h != 0 && c)
		for (pt_context *peer : c->peers)
			if (loadTextureMemOne(peer, width, height, is_hdr, rgba) != h) { setError(PT_E_CUDA, "pt_load_texture: the devices of a multi-GPU context disagree on the texture handle"); return 0; }
	return h;
}

uint32_t pt_load_texture(pt_context *c, const char *path)
{
	PT_TRY
	if (!c || !path) return 0;
	if (c->textureCount >= kMaxTextures) return 0;
	Image img;
	std::string err;
	if (!readImage(path, img, err)) { g_lastError = err; return 0; } // failed load -> handle 0, no error (Pathtracer.cpp:253-257)
	return pt_load_texture_mem(c, img.width, img.height, img.isHdr ? 1 : 0, img.isHdr ? (const void *)img.hdr.data() : (const void *)img.ldr.data());
	PT_CATCH(0u)
}

int pt_set_skybox(pt_context *c, uint32_t handle)
{
	if (!c) return setError(PT_E_INVALID, "pt_set_skybox: null context");
	c->skybox = handle;
	for (pt_context *peer : c->peers) peer->skybox = handle;
	return PT_OK;
}

static SceneDev sceneDev(const pt_context *c)
{
	SceneDev s;
	s.sceneBlob = c->sceneBlob;
	s.mats = c->mats;
	s.textures = c->texDev;
	s.nodeCount = c->nodeCount;
	s.primCount = c->primCount;
	s.globalCount = c->globalCount;
	s.treeNodeCount = c->treeNodeCount;
	s.texCount = c->textureCount;
	s.skybox = (c->skybox <= c->textureCount) ? c->skybox : 0;
	return s;
}

// option "env_is": make sure the device holds the importance distribution of the current sky texture (texels read back from the
// linear device copy the loader keeps)
static int ensureEnvDistribution(pt_context *c, uint32_t handle)
{
	if (c->envHandle == handle && c->envAlias) return PT_OK;
	const TexDesc &t = c->texHost[handle - 1];
	const size_t bytes = size_t(t.width) * t.height * (t.isHdr ? 16 : 4);
	std::vector<unsigned char> texels(bytes);
	CK(cudaMemcpyAsync(texels.data(), t.texels, bytes, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	EnvDistribution d;
	buildEnvDistribution(t.width, t.height, t.isHdr != 0, texels.data(), d);
	if (c->envAlias) { CK(cudaFree(c->envAlias)); c->envAlias = nullptr; }
	if (c->envDensity) { CK(cudaFree(c->envDensity)); c->envDensity = nullptr; }
	CK(cudaMalloc(&c->envAlias, d.alias.size() * 4));
	CK(cudaMalloc(&c->envDensity, d.density.size() * 4));
	CK(cudaMemcpyAsync(c->envAlias, d.alias.data(), d.alias.size() * 4, cudaMemcpyHostToDevice, c->stream));
	CK(cudaMemcpyAsync(c->envDensity, d.density.data(), d.density.size() * 4, cudaMemcpyHostToDevice, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	c->envCols = d.cols;
	c->envRows = d.rows;
	c->envHandle = handle;
	return PT_OK;
}

static int renderOne(pt_context *c, const CameraDev *camera, uint32_t spp, int ignore_history)
{
	PT_TRY
	if (!c || !camera) return setError(PT_E_INVALID, "pt_render: bad arguments");
	CK(cudaSetDevice(c->device));
	if (ignore_history)
	{
		c->accumulatedFrames = 0; // Pathtracer.cpp:164-167
		c->totalSamples = 0;
		c->sampleCursor = c->sampleOffset;
	}
	c->timingMs = 0.0f;
	int launches = 0, usedSmem = 0;
	CK(cudaMemsetAsync(c->counters, 0, kCtrCount * sizeof(unsigned long long), c->stream));
	const bool run = c->nodeCount >= 1 && c->primCount >= 1 && spp > 0; // Pathtracer.cpp:174
	if (run)
	{
		RenderParams p;
		p.scene = sceneDev(c);
		p.cam = *camera;
		p.accum = c->accum;
		p.counters = c->counters;
		p.width = c->width;
		p.height = c->height;
		p.spp = spp;
		p.ignoreHistory = ignore_history ? 1u : 0u;
		p.sampleOffset = c->sampleCursor;
		p.sampleStride = c->sampleStride;
		p.pixelOffset = c->pixelOffset;
		p.pixelStride = c->pixelStride;
		p.seedLo = uint32_t(c->seed);
		p.seedHi = uint32_t(c->seed >> 32);
		for (uint32_t i = 0; i < 10; ++i) { p.philoxKeys[2 * i] = p.seedLo + i * 0x9E3779B9u; p.philoxKeys[2 * i + 1] = p.seedHi + i * 0xBB67AE85u; }
		p.maxBounces = c->maxBounces;
		p.regenLow = c->launch.regenLow > 0 ? uint32_t(c->launch.regenLow) : 16u;
		// first-bounce stratification (RenderParams::strataPer): 2^k cells, k <= 8, at least 16 samples per cell - the lanes of a
		// pass of the one-pixel-per-warp kernel then hold samples of one or two neighbouring cells
		const int v = c->launch.variant;
		const bool perWarpKernel = v == 0 ? spp >= 64u : v == 12; // launchTrace's choice
		const bool wantStrata = perWarpKernel && (c->launch.stratify < 0 ? spp >= 128u : c->launch.stratify != 0) && spp >= 4u && spp < (1u << 21);
		if (wantStrata)
		{
			uint32_t k = 2;
			while (k < 8u && (spp >> (k + 1u)) >= 16u) ++k; // measured at 4096 spp: 32 / 64 / 128 / 256 / 512 cells -> 489 / 479 / 470 / 465 / 468 ms
			if (c->launch.strataK > 0) k = uint32_t(c->launch.strataK); // (experiments: another cell count than the rule's)
			while (k > 2u && (spp >> k) == 0u) --k;
			p.strataBitsA = (k + 1u) / 2u;
			p.strataBitsB = k / 2u;
			p.strataPer = spp >> k;
			p.strataInvPer = 1.0f / float(p.strataPer);
		}
		p.beam = c->launch.beam < 0 ? (spp >= 128u ? 1u : 0u) : uint32_t(c->launch.beam != 0);
		p.alpha = c->alpha;
		c->launch.envIS = 0;
		if (c->envIS && p.scene.skybox != 0)
		{
			const int rc = ensureEnvDistribution(c, p.scene.skybox);
			if (rc != PT_OK) return rc;
			p.scene.env.alias = static_cast<const uint2 *>(c->envAlias);
			p.scene.env.density = c->envDensity;
			p.scene.env.cols = c->envCols;
			p.scene.env.rows = c->envRows;
			c->launch.envIS = 1;
		}
		if (c->noJitter)
		{
			if (!c->centreUV)
			{
				// (this file is compiled without FMA contraction: the division is the IEEE one of the reference's primary pass)
				std::vector<float> uv(size_t(c->width) + c->height);
				for (uint32_t x = 0; x < c->width; ++x) uv[x] = (float(x) + 0.5f) / float(c->width);
				for (uint32_t y = 0; y < c->height; ++y) uv[c->width + y] = (float(y) + 0.5f) / float(c->height);
				CK(cudaMalloc(&c->centreUV, uv.size() * sizeof(float)));
				CK(cudaMemcpy(c->centreUV, uv.data(), uv.size() * sizeof(float), cudaMemcpyHostToDevice));
			}
			p.centreU = c->centreUV;
			p.centreV = c->centreUV + c->width;
			p.aids |= kAidPixelCentre;
		}
		p.firstHitIndex = c->firstHit ? c->firstHitIndex : nullptr;
		p.firstHitT = c->firstHit ? c->firstHitT : nullptr;
		if (c->firstHit) p.aids |= kAidFirstHit;
		if (p.aids && c->launch.envIS) return setError(PT_E_INVALID, "pt_render: the parity aids and env_is cannot be combined");
		c->launch.lightIS = 0;
		if (c->lightIS)
		{
			if (c->envIS) return setError(PT_E_INVALID, "pt_render: light_is and env_is cannot be combined (one sampled light source per kernel)");
			if (c->noJitter || c->firstHit) return setError(PT_E_INVALID, "pt_render: light_is and the parity aids (jitter = 0, first_hit = 1) cannot be combined");
			// a scene without emitters renders with the plain kernel: the same bits as without the option
			if (c->lightCount != 0)
			{
				p.lights.recs = c->lightRecs;
				p.lights.count = c->lightCount;
				c->launch.lightIS = 1;
			}
		}
		c->launch.stackLevels = int(c->bvhDepth) + 2;
		CK(cudaEventRecord(c->evStart, c->stream)); // (all allocations are behind us: the events bracket the device work alone)
		// pixel partition: the pixels of the other ranks hold zeros, so that the sum over ranks is the image
		if (ignore_history && c->pixelStride > 1u && !c->skipPartitionClear) CK(cudaMemsetAsync(c->accum, 0, size_t(c->width) * c->height * sizeof(float4), c->stream));
		launches = launchTrace(p, c->launch, c->stream, &usedSmem);
		if (launches < 0) return setError(PT_E_CUDA, std::string("pt_render: kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()));
	}
	if (!run) CK(cudaEventRecord(c->evStart, c->stream));
	CK(cudaEventRecord(c->evStop, c->stream));
	CK(cudaGetLastError());
	CK(cudaStreamSynchronize(c->stream));
	CK(cudaEventElapsedTime(&c->timingMs, c->evStart, c->evStop));
	if (run)
	{
		unsigned long long h[kCtrCount];
		CK(cudaMemcpy(h, c->counters, sizeof h, cudaMemcpyDeviceToHost));
		{
			const unsigned long long all = (unsigned long long)c->width * c->height;
			const unsigned long long own = all > c->pixelOffset ? (all - c->pixelOffset + c->pixelStride - 1u) / c->pixelStride : 0ull;
			c->stats.samples = own * spp;
		}
		memcpy(c->rawCounters, h, sizeof h);
		c->stats.rays = h[kCtrRays];
		c->stats.node_visits = h[kCtrNodes];
		c->stats.prim_tests = h[kCtrPrims];
		c->stats.shades = h[kCtrShades];
		c->stats.misses = h[kCtrMisses];
		c->stats.scene_in_smem = uint32_t(usedSmem);
		c->sampleCursor += spp * c->sampleStride;
		c->totalSamples += spp;
	}
	c->stats.gpu_ms = c->timingMs;
	(void)launches;
	// the reference counts render() CALLS, not samples (Pathtracer.cpp:226, quirk Q1); "frames_per_spp" = k makes one
	// call count as ceil(spp / k) calls so a single launch reproduces the reference CLI's 8-spp slicing (main.cpp:271-278)
	c->accumulatedFrames += (c->framesPerSpp > 0) ? (spp + c->framesPerSpp - 1) / c->framesPerSpp : 1u;
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

static int loadNccl(pt_context *c)
{
	if (c->nccl) return PT_OK;
	NcclState *n = new NcclState();
	c->nccl = n;
	const char *names[] = { "libnccl.so.2", "libnccl.so" };
	for (const char *name : names)
		if (!n->lib) n->lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
	if (!n->lib) return setError(PT_E_CUDA, std::string("multi-GPU: cannot load NCCL (libnccl.so.2): ") + dlerror());
#define PT_SYM(field, sym) n->field = reinterpret_cast<decltype(n->field)>(dlsym(n->lib, sym)); if (!n->field) return setError(PT_E_CUDA, std::string("multi-GPU: NCCL lacks ") + sym)
	PT_SYM(commInitAll, "ncclCommInitAll");
	PT_SYM(commDestroy, "ncclCommDestroy");
	PT_SYM(groupStart, "ncclGroupStart");
	PT_SYM(groupEnd, "ncclGroupEnd");
	PT_SYM(reduce, "ncclReduce");
	PT_SYM(getErrorString, "ncclGetErrorString");
#undef PT_SYM
	std::vector<int> devs = { c->device };
	for (pt_context *peer : c->peers) devs.push_back(peer->device);
	n->comms.assign(devs.size(), nullptr);
	const ncclResult_t r = n->commInitAll(n->comms.data(), int(devs.size()), devs.data());
	if (r != ncclSuccess) return setError(PT_E_CUDA, std::string("multi-GPU: ncclCommInitAll failed: ") + n->getErrorString(r));
	CK(cudaSetDevice(c->device));
	CK(cudaEventCreate(&n->ev0));
	CK(cudaEventCreate(&n->ev1));
	return PT_OK;
}

// pt_render on a multi-GPU context: the work is split over the devices (option "partition"), every device renders its share
// on its own host thread, and the image comes together on the root either by itself - pixel partition with peer access: the
// kernels of the other devices store their pixels straight into the root's accumulation buffer over NVLink, 16 bytes per
// pixel, no collective at all - or by ONE ncclReduce of the float4 accumulation buffers (option "exchange").
static int renderMulti(pt_context *c, const CameraDev *camera, uint32_t spp, int ignore_history)
{
	std::vector<pt_context *> all = { c };
	all.insert(all.end(), c->peers.begin(), c->peers.end());
	const uint32_t N = uint32_t(all.size());
	const size_t px = size_t(c->width) * c->height;
	const bool pixels = c->partition == 0;
	const bool p2p = pixels && c->p2pReady && c->exchange != 0;
	std::vector<uint32_t> share(N, spp);
	for (uint32_t i = 0; i < N; ++i)
	{
		pt_context *d = all[i];
		d->pixelOffset = pixels ? i : 0u;
		d->pixelStride = pixels ? N : 1u;
		d->sampleStride = pixels ? 1u : N;
		const uint32_t off = pixels ? 0u : i;
		if (d->sampleOffset != off) { d->sampleOffset = off; d->sampleCursor = off; } // (an unchanged offset must not rewind a progressive render)
		if (!pixels) share[i] = spp > i ? (spp - i + N - 1u) / N : 0u;
		d->skipPartitionClear = p2p;
		d->alpha = (pixels || i == 0u) ? 1.0f : 0.0f; // sample partition: the summed alpha is 1, as on one GPU
		if (i > 0)
		{
			// p2p: the peer renders into the ROOT's buffer; NCCL: into its own
			float4 *want = p2p ? c->accum : nullptr;
			if (want && d->accum != want)
			{
				CK(cudaSetDevice(d->device));
				if (d->ownAccum && d->accum) CK(cudaFree(d->accum));
				d->accum = want;
				d->ownAccum = false;
			}
			else if (!want && !d->ownAccum)
			{
				CK(cudaSetDevice(d->device));
				d->accum = nullptr;
				CK(cudaMalloc(&d->accum, px * sizeof(float4)));
				CK(cudaMemset(d->accum, 0, px * sizeof(float4)));
				d->ownAccum = true;
			}
		}
	}
	if (!p2p && loadNccl(c) != PT_OK) return PT_E_CUDA;
	// a device whose share of a restarting call is empty (sample partition, spp < devices) must not leave old sums in the reduce
	for (uint32_t i = 0; i < N; ++i)
		if (!p2p && ignore_history && share[i] == 0u)
		{
			CK(cudaSetDevice(all[i]->device));
			CK(cudaMemsetAsync(all[i]->accum, 0, px * sizeof(float4), all[i]->stream));
		}
	// one host thread per GPU
	std::vector<int> rc(N, PT_OK);
	std::vector<std::string> errs(N);
	std::vector<std::thread> threads;
	for (uint32_t i = 1; i < N; ++i)
		threads.emplace_back([&, i]() { rc[i] = renderOne(all[i], camera, share[i], ignore_history); if (rc[i] != PT_OK) errs[i] = g_lastError; });
	rc[0] = renderOne(c, camera, share[0], ignore_history);
	if (rc[0] != PT_OK) errs[0] = g_lastError;
	for (std::thread &t : threads) t.join();
	for (uint32_t i = 0; i < N; ++i)
		if (rc[i] != PT_OK) return setError(rc[i], "device " + std::to_string(all[i]->device) + ": " + errs[i]);
	float traceMs = 0.0f;
	for (pt_context *d : all) traceMs = fmaxf(traceMs, d->timingMs);
	c->reduceMs = 0.0f;
	c->imageSource = nullptr;
	if (!p2p)
	{
		NcclState *n = c->nccl;
		CK(cudaSetDevice(c->device));
		if (!c->reduced) CK(cudaMalloc(&c->reduced, px * sizeof(float4)));
		ncclResult_t r = ncclSuccess;
		// the communicators' first collective sets up the NVLink connections (~150 ms): done once, by an untimed reduce of the same
		// buffers (into the same destination - the timed one below just repeats it), so that exchange_ms is the transfer
		for (int pass = n->warm ? 1 : 0; pass < 2 && r == ncclSuccess; ++pass)
		{
			if (pass == 1) CK(cudaEventRecord(n->ev0, c->stream));
			r = n->groupStart();
			for (uint32_t i = 0; r == ncclSuccess && i < N; ++i)
				r = n->reduce(all[i]->accum, c->reduced, px * 4, ncclFloat, ncclSum, 0, n->comms[i], all[i]->stream);
			const ncclResult_t r2 = n->groupEnd();
			if (r == ncclSuccess) r = r2;
			if (pass == 0)
				for (pt_context *d : all)
				{
					CK(cudaSetDevice(d->device));
					CK(cudaStreamSynchronize(d->stream));
				}
			CK(cudaSetDevice(c->device));
		}
		n->warm = true;
		if (r != ncclSuccess) return setError(PT_E_CUDA, std::string("multi-GPU: ncclReduce failed: ") + n->getErrorString(r));
		CK(cudaSetDevice(c->device));
		CK(cudaEventRecord(n->ev1, c->stream));
		for (pt_context *d : all)
		{
			CK(cudaSetDevice(d->device));
			CK(cudaStreamSynchronize(d->stream));
		}
		CK(cudaSetDevice(c->device));
		CK(cudaEventElapsedTime(&c->reduceMs, n->ev0, n->ev1));
		c->imageSource = c->reduced;
	}
	// the root answers for the whole job: timing (slowest device + exchange), counts for the normalisation, summed statistics
	c->multiTraceMs = traceMs;
	c->timingMs = traceMs + c->reduceMs;
	if (ignore_history) { c->jobSamples = 0; c->jobFrames = 0; }
	c->jobSamples += spp;
	c->jobFrames += (c->framesPerSpp > 0) ? (spp + c->framesPerSpp - 1) / c->framesPerSpp : 1u;
	c->totalSamples = c->jobSamples;
	c->accumulatedFrames = c->jobFrames;
	pt_stats sum = c->stats;
	for (uint32_t i = 1; i < N; ++i)
	{
		const pt_stats &s = all[i]->stats;
		sum.samples += s.samples; sum.rays += s.rays; sum.node_visits += s.node_visits; sum.prim_tests += s.prim_tests; sum.shades += s.shades; sum.misses += s.misses;
	}
	sum.gpu_ms = c->timingMs;
	c->multiStats = sum;
	return PT_OK;
}

int pt_render(pt_context *c, const pt_camera_desc *camera, uint32_t spp, int ignore_history)
{
	PT_TRY
	if (!c || !camera) return setError(PT_E_INVALID, "pt_render: bad arguments");
	CameraDev cam;
	computeCamera(*camera, cam);
	return c->peers.empty() ? renderOne(c, &cam, spp, ignore_history) : renderMulti(c, &cam, spp, ignore_history);
	PT_CATCH(PT_E_LIMIT)
}

int pt_render_vectors(pt_context *c, const pt_camera_vectors *camera, uint32_t spp, int ignore_history)
{
	PT_TRY
	if (!c || !camera) return setError(PT_E_INVALID, "pt_render_vectors: bad arguments");
	CameraDev cam;
	memcpy(cam.origin, camera->origin, 12);
	memcpy(cam.lowerLeft, camera->lower_left, 12);
	memcpy(cam.horizontal, camera->horizontal, 12);
	memcpy(cam.vertical, camera->vertical, 12);
	return c->peers.empty() ? renderOne(c, &cam, spp, ignore_history) : renderMulti(c, &cam, spp, ignore_history);
	PT_CATCH(PT_E_LIMIT)
}

float pt_get_timing_ms(const pt_context *c) { return c ? c->timingMs : 0.0f; }

static const float *readHdr(pt_context *c, float scale)
{
	if (cudaSetDevice(c->device) != cudaSuccess) return nullptr;
	const uint32_t px = c->width * c->height;
	if ((!c->scaledDev && cudaMalloc(&c->scaledDev, size_t(px) * sizeof(float4)) != cudaSuccess) ||
	    (!c->hostHdr && cudaMallocHost(&c->hostHdr, size_t(px) * sizeof(float4)) != cudaSuccess))
	{
		setError(PT_E_CUDA, std::string("pt_get_hdr: ") + cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	launchScale(c->imageSource ? c->imageSource : c->accum, c->scaledDev, px, scale, c->stream);
	if (cudaMemcpyAsync(c->hostHdr, c->scaledDev, size_t(px) * sizeof(float4), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
	    cudaStreamSynchronize(c->stream) != cudaSuccess)
	{
		setError(PT_E_CUDA, std::string("pt_get_hdr: ") + cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	return c->hostHdr;
}

const float *pt_get_hdr(pt_context *c)
{
	if (!c) return nullptr;
	return readHdr(c, 1.0f / fmaxf(float(c->accumulatedFrames), 1.0f)); // Pathtracer.cpp:307
}

const float *pt_get_hdr_mean(pt_context *c)
{
	if (!c) return nullptr;
	return readHdr(c, 1.0f / fmaxf(float(c->totalSamples), 1.0f));
}

const float *pt_get_hdr_sum(pt_context *c)
{
	if (!c) return nullptr;
	return readHdr(c, 1.0f);
}

const uint8_t *pt_get_ldr(pt_context *c)
{
	if (!c) return nullptr;
	if (cudaSetDevice(c->device) != cudaSuccess) return nullptr;
	const uint32_t px = c->width * c->height;
	if ((!c->ldrDev && cudaMalloc(&c->ldrDev, size_t(px) * sizeof(uchar4)) != cudaSuccess) ||
	    (!c->hostLdr && cudaMallocHost(&c->hostLdr, size_t(px) * sizeof(uchar4)) != cudaSuccess))
	{
		setError(PT_E_CUDA, std::string("pt_get_ldr: ") + cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	// tonemap.cu:17 divides by float(accumulatedSampleCount) via reciprocal-multiply; 0 frames -> division by zero in the
	// reference; here the accumulation is zero in that case and the scale is clamped like getHDRImageData's
	launchTonemap(c->imageSource ? c->imageSource : c->accum, c->ldrDev, px, 1.0f / fmaxf(float(c->accumulatedFrames), 1.0f), c->stream);
	if (cudaMemcpyAsync(c->hostLdr, c->ldrDev, size_t(px) * sizeof(uchar4), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
	    cudaStreamSynchronize(c->stream) != cudaSuccess)
	{
		setError(PT_E_CUDA, std::string("pt_get_ldr: ") + cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	return c->hostLdr;
}

static int setOptionOne(pt_context *c, const char *key, double value)
{
	PT_TRY
	if (!c || !key) return setError(PT_E_INVALID, "pt_set_option: bad arguments");
	const std::string k(key);
	if (k == "seed") c->seed = uint64_t(value);
	else if (k == "sample_offset")
	{
		// (setting the SAME offset again - a multi-GPU driver configuring its partition before every call - must not rewind
		// the sample cursor of a progressive render: the next call would replay the same Philox indices)
		if (uint32_t(value) != c->sampleOffset) { c->sampleOffset = uint32_t(value); c->sampleCursor = c->sampleOffset; }
	}
	// after a multi-GPU reduce the destination buffer holds the samples / frames of ALL ranks: let the driver say so, so that
	// pt_get_hdr / pt_get_hdr_mean / pt_get_ldr normalise by the right count
	else if (k == "total_samples") c->totalSamples = value < 0 ? 0ull : (unsigned long long)(value);
	else if (k == "accumulated_frames") c->accumulatedFrames = value < 0 ? 0u : uint32_t(value);
	else if (k == "sample_stride") c->sampleStride = value < 1 ? 1u : uint32_t(value);
	else if (k == "pixel_offset") c->pixelOffset = value < 0 ? 0u : uint32_t(value);
	else if (k == "pixel_stride") c->pixelStride = value < 1 ? 1u : uint32_t(value);
	else if (k == "frames_per_spp") c->framesPerSpp = uint32_t(value);
	else if (k == "count_work") c->launch.countWork = value != 0;
	else if (k == "smem_scene") c->launch.smemScene = value != 0;
	else if (k == "max_bounces") c->maxBounces = value < 1 ? 1u : uint32_t(value);
	else if (k == "max_leaf") c->maxLeaf = value < 1 ? 1u : uint32_t(value);
	else if (k == "variant")
	{
		if (!(value == 0 || value == 4 || value == 12)) return setError(PT_E_INVALID, "pt_set_option: variant must be 0 (default), 4 (one pixel per lane) or 12 (one pixel per warp)");
		c->launch.variant = int(value);
	}
	else if (k == "max_global") c->maxGlobal = uint32_t(value < 0 ? 0 : value);
	else if (k == "bvh_builder") c->bvhBuilder = value == 1 ? kBuilderLbvh : (value == 0 ? kBuilderSah : kBuilderAuto);
	else if (k == "regen_low") c->launch.regenLow = int(value);
	else if (k == "beam") c->launch.beam = int(value);
	else if (k == "alpha") c->alpha = float(value);
	else if (k == "stratify") c->launch.stratify = int(value);
	else if (k == "strata_k") c->launch.strataK = value < 2 ? 0 : (value > 10 ? 10 : int(value));
	else if (k == "smem_stack") c->launch.smemStack = int(value);
	else if (k == "jitter") c->noJitter = value == 0;
	else if (k == "env_is") c->envIS = value != 0;
	else if (k == "light_is") c->lightIS = value != 0;
	else if (k == "first_hit")
	{
		c->firstHit = value != 0;
		if (c->firstHit && !c->firstHitIndex)
		{
			const size_t px = size_t(c->width) * c->height;
			CK(cudaSetDevice(c->device));
			CK(cudaMalloc(&c->firstHitIndex, px * 4));
			CK(cudaMalloc(&c->firstHitT, px * 4));
			CK(cudaMemset(c->firstHitIndex, 0xff, px * 4));
			CK(cudaMemset(c->firstHitT, 0, px * 4));
		}
	}
	else if (k == "tex_unit") { c->texUnit = value != 0; return uploadTextureTable(c); }
	else return setError(PT_E_INVALID, "pt_set_option: unknown option " + k);
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

int pt_set_option(pt_context *c, const char *key, double value)
{
	if (!c || !key) return setError(PT_E_INVALID, "pt_set_option: bad arguments");
	const std::string k(key);
	if (k == "partition") { c->partition = value != 0 ? 1 : 0; return PT_OK; }
	if (k == "exchange") { c->exchange = value < 0 ? -1 : (value != 0 ? 1 : 0); return PT_OK; }
	if (!c->peers.empty() && (k == "pixel_offset" || k == "pixel_stride" || k == "sample_offset" || k == "sample_stride"))
		return setError(PT_E_INVALID, "pt_set_option: a multi-GPU context sets the partition options of its devices itself (use \"partition\")");
	int r = setOptionOne(c, key, value);
	for (size_t i = 0; r == PT_OK && i < c->peers.size(); ++i) r = setOptionOne(c->peers[i], key, value);
	return r;
}

/* debugging aid (not in the header): raw device counters of the last pt_render, see trace_kernels.h kCtr* */
extern "C" int pt_debug_counters(const pt_context *c, unsigned long long *out, int n)
{
	if (!c || !out) return 0;
	const int m = n < int(kCtrCount) ? n : int(kCtrCount);
	for (int i = 0; i < m; ++i) out[i] = c->rawCounters[i];
	return m;
}

/* debugging aid (not in the header): the render kernels' 1 / sqrt(x) (trace_device.cuh invSqrtExact) next to the IEEE routines */
extern "C" int pt_debug_inv_sqrt(pt_context *c, uint32_t n, const float *x, float *fast, float *ieee)
{
	if (!c || !x || !fast || !ieee) return setError(PT_E_INVALID, "pt_debug_inv_sqrt: bad arguments");
	CK(cudaSetDevice(c->device));
	DevBuf dx, df, di;
	CK(dx.alloc(size_t(n) * 4)); CK(df.alloc(size_t(n) * 4)); CK(di.alloc(size_t(n) * 4));
	CK(cudaMemcpyAsync(dx.p, x, size_t(n) * 4, cudaMemcpyHostToDevice, c->stream));
	launchInvSqrtCheck(n, dx.as<float>(), df.as<float>(), di.as<float>(), c->stream);
	CK(cudaGetLastError());
	CK(cudaMemcpyAsync(fast, df.p, size_t(n) * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaMemcpyAsync(ieee, di.p, size_t(n) * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	return PT_OK;
}

int pt_get_stats(const pt_context *c, pt_stats *out)
{
	if (!c || !out) return setError(PT_E_INVALID, "pt_get_stats: bad arguments");
	*out = c->peers.empty() ? c->stats : c->multiStats;
	return PT_OK;
}

void pt_camera_rotate(pt_camera_desc *camera, float pitch, float yaw, float roll)
{
	if (camera) cameraRotate(*camera, pitch, yaw, roll);
}
void pt_camera_translate(pt_camera_desc *camera, float x, float y, float z)
{
	if (camera) cameraTranslate(*camera, x, y, z);
}

int pt_primary_pass(pt_context *c, const pt_camera_desc *camera, int32_t *hit_index, float *hit_t)
{
	if (!c || !camera || !hit_index || !hit_t) return setError(PT_E_INVALID, "pt_primary_pass: bad arguments");
	const size_t px = size_t(c->width) * c->height;
	if (c->nodeCount == 0)
	{
		for (size_t i = 0; i < px; ++i) { hit_index[i] = -1; hit_t[i] = 0.0f; }
		return PT_OK;
	}
	CK(cudaSetDevice(c->device));
	DevBuf dIdx, dT;
	CK(dIdx.alloc(px * 4));
	CK(dT.alloc(px * 4));
	CameraDev cam;
	computeCamera(*camera, cam);
	launchPrimary(sceneDev(c), cam, c->width, c->height, dIdx.as<int32_t>(), dT.as<float>(), c->stream);
	CK(cudaGetLastError());
	CK(cudaMemcpyAsync(hit_index, dIdx.p, px * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaMemcpyAsync(hit_t, dT.p, px * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	return PT_OK;
}

int pt_trace_rays(pt_context *c, size_t n, const float *origins, const float *directions, float t_min, int32_t *hit_index, float *hit_t, float *hit_normal)
{
	if (!c || !origins || !directions || !hit_index || !hit_t) return setError(PT_E_INVALID, "pt_trace_rays: bad arguments");
	if (n == 0) return PT_OK;
	if (c->nodeCount == 0) return setError(PT_E_INVALID, "pt_trace_rays: no scene");
	CK(cudaSetDevice(c->device));
	DevBuf dO, dD, dT, dI, dN;
	CK(dO.alloc(n * 12)); CK(dD.alloc(n * 12)); CK(dT.alloc(n * 4)); CK(dI.alloc(n * 4));
	if (hit_normal) CK(dN.alloc(n * 12));
	CK(cudaMemcpyAsync(dO.p, origins, n * 12, cudaMemcpyHostToDevice, c->stream));
	CK(cudaMemcpyAsync(dD.p, directions, n * 12, cudaMemcpyHostToDevice, c->stream));
	launchTraceRays(sceneDev(c), n, dO.as<float>(), dD.as<float>(), t_min, dI.as<int32_t>(), dT.as<float>(), dN.as<float>(), c->stream);
	CK(cudaGetLastError());
	CK(cudaMemcpyAsync(hit_index, dI.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaMemcpyAsync(hit_t, dT.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
	if (hit_normal) CK(cudaMemcpyAsync(hit_normal, dN.p, n * 12, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	return PT_OK;
}

int pt_get_first_hit(pt_context *c, int32_t *hit_index, float *hit_t)
{
	if (!c || !hit_index || !hit_t) return setError(PT_E_INVALID, "pt_get_first_hit: bad arguments");
	if (!c->firstHitIndex) return setError(PT_E_INVALID, "pt_get_first_hit: option first_hit was not set before pt_render");
	const size_t px = size_t(c->width) * c->height;
	CK(cudaSetDevice(c->device));
	CK(cudaMemcpyAsync(hit_index, c->firstHitIndex, px * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaMemcpyAsync(hit_t, c->firstHitT, px * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	return PT_OK;
}

void *pt_accum_device_ptr(pt_context *c) { return c ? (void *)c->accum : nullptr; }

int pt_set_accum_device_ptr(pt_context *c, void *device_ptr)
{
	if (!c || !device_ptr) return setError(PT_E_INVALID, "pt_set_accum_device_ptr: bad arguments");
	if (!c->peers.empty()) return setError(PT_E_INVALID, "pt_set_accum_device_ptr: not on a multi-GPU context (it owns the exchange)");
	CK(cudaSetDevice(c->device));
	CK(cudaStreamSynchronize(c->stream));
	if (c->ownAccum && c->accum) CK(cudaFree(c->accum));
	c->accum = reinterpret_cast<float4 *>(device_ptr);
	c->ownAccum = false;
	return PT_OK;
}

int pt_parse_scene_file(const char *json_path, pt_object_desc *objects, size_t capacity, pt_camera_desc *camera_out, float aspect, char *tex_paths,
                        size_t tex_paths_cap, int32_t *skybox_tex_index)
{
	PT_TRY
	if (!json_path) return setError(PT_E_INVALID, "pt_parse_scene_file: null path");
	ParsedScene ps;
	std::string err;
	int code = PT_E_PARSE;
	if (!parseSceneFile(json_path, aspect, ps, err, &code)) return setError(code, err);
	if (objects)
		for (size_t i = 0; i < ps.objects.size() && i < capacity; ++i) objects[i] = ps.objects[i];
	if (camera_out) *camera_out = ps.camera;
	if (skybox_tex_index) *skybox_tex_index = int32_t(ps.skyboxTexture);
	if (tex_paths && tex_paths_cap)
	{
		std::string joined;
		for (size_t i = 0; i < ps.texturePaths.size(); ++i) { if (i) joined += '\n'; joined += ps.texturePaths[i]; }
		snprintf(tex_paths, tex_paths_cap, "%s", joined.c_str());
	}
	return int(ps.objects.size());
	PT_CATCH(PT_E_LIMIT)
}

int pt_load_scene_file(pt_context *c, const char *json_path, pt_camera_desc *camera_out)
{
	PT_TRY
	if (!c || !json_path) return setError(PT_E_INVALID, "pt_load_scene_file: bad arguments");
	ParsedScene ps;
	std::string err;
	int code = PT_E_PARSE;
	if (!parseSceneFile(json_path, float(c->width) / float(c->height), ps, err, &code)) return setError(code, err);
	for (const std::string &m : ps.messages) printf("%s\n", m.c_str());
	// textures load in first-use order; a failed load maps to handle 0 and does not consume a slot (SceneLoader.cpp:127-149)
	std::vector<uint32_t> handles(ps.texturePaths.size(), 0);
	auto loadIdx = [&](uint32_t idx) -> uint32_t { return idx == 0 ? 0u : handles[idx - 1]; };
	for (size_t i = 0; i < ps.texturePaths.size(); ++i) handles[i] = pt_load_texture(c, ps.texturePaths[i].c_str());
	for (pt_object_desc &o : ps.objects) o.material.texture = loadIdx(o.material.texture);
	if (ps.hasObjectsArray)
	{
		const int r = pt_set_scene(c, ps.objects.size(), ps.objects.data());
		if (r != PT_OK) return r;
	}
	// setSkyboxTextureHandle is called whenever "skybox" is a string (SceneLoader.cpp:327-332) - with handle 0 for "" or a
	// failed load, so a context reused for another scene does not keep the previous sky
	if (ps.hasSkyboxString) pt_set_skybox(c, loadIdx(ps.skyboxTexture));
	if (camera_out) *camera_out = ps.camera;
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

int pt_write_png(const char *path, uint32_t width, uint32_t height, const uint8_t *rgba)
{
	PT_TRY
	std::string err;
	if (!path || !rgba) return setError(PT_E_INVALID, "pt_write_png: bad arguments");
	if (!writePng(path, width, height, rgba, err)) return setError(PT_E_IO, err);
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

int pt_write_hdr(const char *path, uint32_t width, uint32_t height, const float *rgba)
{
	PT_TRY
	std::string err;
	if (!path || !rgba) return setError(PT_E_INVALID, "pt_write_hdr: bad arguments");
	if (!writeHdr(path, width, height, rgba, err)) return setError(PT_E_IO, err);
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

int pt_env_distribution(uint32_t width, uint32_t height, int is_hdr, const void *rgba, uint32_t *cols, uint32_t *rows, uint32_t *alias, float *density)
{
	PT_TRY
	if (!rgba || width == 0 || height == 0) return setError(PT_E_INVALID, "pt_env_distribution: bad arguments");
	EnvDistribution d;
	buildEnvDistribution(width, height, is_hdr != 0, rgba, d);
	if (cols) *cols = d.cols;
	if (rows) *rows = d.rows;
	if (alias) memcpy(alias, d.alias.data(), d.alias.size() * 4);
	if (density) memcpy(density, d.density.data(), d.density.size() * 4);
	return int(d.density.size());
	PT_CATCH(PT_E_LIMIT)
}

int pt_light_distribution(size_t count, const pt_object_desc *objects, uint32_t *scene_index, float *probability, uint32_t *alias)
{
	PT_TRY
	if (count == 0 || !objects) return setError(PT_E_INVALID, "pt_light_distribution: bad arguments");
	CompiledScene cs;
	std::string err;
	if (!compileScene(count, objects, 4, cs, err)) return setError(PT_E_LIMIT, "pt_light_distribution: " + err);
	LightTable lt;
	buildLightTable(cs, lt);
	for (size_t k = 0; k < lt.recs.size(); ++k)
	{
		if (scene_index) scene_index[k] = lt.sceneIndex[k];
		if (probability) probability[k] = lt.probability[k];
		if (alias)
		{
			memcpy(&alias[2 * k], &lt.recs[k].aliasQ, 4);
			alias[2 * k + 1] = lt.recs[k].alias;
		}
	}
	return int(lt.recs.size());
	PT_CATCH(PT_E_LIMIT)
}

int pt_read_image(const char *path, uint32_t *width, uint32_t *height, int *is_hdr, void **rgba)
{
	PT_TRY
	if (!path || !width || !height || !is_hdr || !rgba) return setError(PT_E_INVALID, "pt_read_image: bad arguments");
	Image img;
	std::string err;
	if (!readImage(path, img, err)) return setError(PT_E_IO, err);
	*width = img.width;
	*height = img.height;
	*is_hdr = img.isHdr ? 1 : 0;
	const size_t bytes = size_t(img.width) * img.height * (img.isHdr ? 16 : 4);
	*rgba = malloc(bytes);
	if (!*rgba) return setError(PT_E_LIMIT, "pt_read_image: out of memory");
	memcpy(*rgba, img.isHdr ? (const void *)img.hdr.data() : (const void *)img.ldr.data(), bytes);
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

} // extern "C"
