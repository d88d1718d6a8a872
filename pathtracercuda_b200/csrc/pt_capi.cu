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
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <memory>
#include <nccl.h>
#include <string>
#include <thread>
#include <utility>
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

// Memory of one CUDA allocator, freed when its holder goes.  Move-only; a holder is freed or replaced only where its device is
// current and no queued work can still use it.
template <cudaError_t (*Alloc)(void **, size_t), cudaError_t (*Free)(void *)>
struct Buf
{
	void *p = nullptr;
	Buf() = default;
	Buf(Buf &&o) noexcept : p(std::exchange(o.p, nullptr)) {}
	Buf &operator=(Buf o) noexcept { std::swap(p, o.p); return *this; } // (the memory held before goes with `o`)
	~Buf() { if (p) Free(p); }
	cudaError_t alloc(size_t bytes) // (on an empty holder; it stays empty when the allocation fails)
	{
		void *q = nullptr;
		const cudaError_t e = Alloc(&q, bytes);
		if (e == cudaSuccess) p = q;
		return e;
	}
	template <typename T> T *as() const { return static_cast<T *>(p); }
};
using DevBuf = Buf<cudaMalloc, cudaFree>;          // device memory
using HostBuf = Buf<cudaMallocHost, cudaFreeHost>; // pinned host memory

// one loaded texture: the linear copy (software filter, env_is tables) and the texture object over a CUDA array of the same
// texels; freed in the order object, array, linear copy
struct Texture
{
	DevBuf texels;
	cudaArray_t array = nullptr;
	cudaTextureObject_t object = 0;
	Texture() = default;
	Texture(Texture &&o) noexcept : texels(std::move(o.texels)), array(std::exchange(o.array, nullptr)), object(std::exchange(o.object, 0)) {}
	~Texture() { if (object) cudaDestroyTextureObject(object); if (array) cudaFreeArray(array); }
};
} // namespace

struct pt_context
{
	int device = 0;
	uint32_t width = 0, height = 0;
	cudaStream_t stream = nullptr;
	cudaEvent_t evStart = nullptr, evStop = nullptr;
	float4 *accum = nullptr;
	bool ownAccum = true;
	DevBuf scaledDev, ldrDev;    // read-back staging (float4 / uchar4 per pixel)
	HostBuf hostHdr, hostLdr;
	DevBuf counters;             // kCtrCount unsigned long long
	DevBuf firstHitIndex, firstHitT; // option "first_hit": the render kernel's own first-hit (index, t) per pixel (parity aid)
	bool firstHit = false, noJitter = false;
	// option "env_is": the sky's importance distribution (env_sampling.h), built for texture handle envHandle on first use
	bool envIS = false;
	uint32_t envHandle = 0;
	DevBuf envAlias, envDensity;
	uint32_t envCols = 0, envRows = 0;
	// option "light_is": the emitter table of the current scene (light_sampling.h), built with the compiled scene
	bool lightIS = false;
	DevBuf lightRecs;
	uint32_t lightCount = 0;
	DevBuf centreUV; // option "jitter" = 0: pixel-centre coordinates (RenderParams::centreU / centreV), made on first use
	// option "adaptive": threshold tau (0 = off) and first checkpoint m; the samples each pixel took in the last pt_render (made on first
	// use), valid when that render was adaptive
	float adaptTau = 0.0f;
	uint32_t adaptMinSpp = 128;
	DevBuf sampleCounts;
	bool countsValid = false;
	// scene
	DevBuf sceneBlob;
	Mat *mats = nullptr; // (the material table at the end of sceneBlob)
	uint32_t nodeCount = 0, treeNodeCount = 0, primCount = 0, bvhDepth = 0, globalCount = 0, maxGlobal = ptb::kMaxGlobalPrims;
	int bvhBuilder = ptb::kBuilderAuto; // option "bvh_builder" (scene_compile.h): SAH, from 2^19 objects the LBVH
	// textures: handle h is textures[h - 1] and texHost[h - 1]
	std::vector<Texture> textures;
	TexDesc texHost[kMaxTextures];
	int texUnit = 1; // filter textures with the texture unit (0: in software from linear memory)
	DevBuf texDev;   // the device copy of texHost
	uint32_t skybox = 0;
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
	// denoiser (pt_render_aov / pt_denoise; on the root device), allocated on first use
	DevBuf aov[3];                // guide buffers: albedo, normal, position (PT_AOV_*)
	bool aovValid = false;        // rendered, and no scene set since
	DevBuf denoised, denoiseTmp;  // the filtered sum buffer, and the other side of the ping-pong
	bool hasDenoised = false;
	uint32_t denoisedFrames = 0;  // accumulatedFrames / totalSamples of the image pt_denoise filtered
	unsigned long long denoisedSamples = 0;
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
	std::unique_ptr<pt_context, void (*)(pt_context *)> c(new pt_context(), pt_destroy); // (destroyed on every early return)
	c->device = device;
	c->width = width;
	c->height = height;
	memset(&c->stats, 0, sizeof c->stats);
	memset(c->texHost, 0, sizeof c->texHost);
	const size_t px = size_t(width) * height;
	CK(cudaSetDevice(device));
	// (two attributes, not cudaGetDeviceProperties: that call fills in everything the driver knows about the device and is one of
	// the slower ones of a process's start)
	int smCount = 0, smemOptin = 0;
	CK(cudaDeviceGetAttribute(&smCount, cudaDevAttrMultiProcessorCount, device));
	CK(cudaDeviceGetAttribute(&smemOptin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
	c->launch.smCount = smCount;
	c->launch.maxSmemOptin = size_t(smemOptin);
	CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	CK(cudaEventCreate(&c->evStart));
	CK(cudaEventCreate(&c->evStop));
	CK(cudaMalloc(&c->accum, px * sizeof(float4)));
	CK(cudaMemsetAsync(c->accum, 0, px * sizeof(float4), c->stream));
	// (the read-back buffers - device staging and pinned host memory for the HDR and the LDR image - are allocated by the first
	// getter that needs them: pinned allocations are slow, a peer context of a multi-GPU job never reads back, and a run that
	// writes a PNG does not need the 33 MB HDR pair)
	CK(c->counters.alloc(kCtrCount * sizeof(unsigned long long)));
	CK(c->texDev.alloc(kMaxTextures * sizeof(TexDesc)));
	CK(cudaMemsetAsync(c->texDev.p, 0, kMaxTextures * sizeof(TexDesc), c->stream));
	CK(cudaStreamSynchronize(c->stream));
	*out = c.release();
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
	if (c->evStart) cudaEventDestroy(c->evStart);
	if (c->evStop) cudaEventDestroy(c->evStop);
	if (c->stream) cudaStreamDestroy(c->stream);
	delete c; // (the holders free the rest: the device is current and the stream has finished)
}

// upload a compiled scene and its emitter table to one device; they replace the previous ones once they are complete
static int uploadScene(pt_context *c, const CompiledScene &cs, const LightTable &lt)
{
	CK(cudaSetDevice(c->device));
	DevBuf lights;
	if (!lt.recs.empty())
	{
		CK(lights.alloc(lt.recs.size() * sizeof(LightRec)));
		CK(cudaMemcpyAsync(lights.p, lt.recs.data(), lt.recs.size() * sizeof(LightRec), cudaMemcpyHostToDevice, c->stream));
	}
	// one allocation, nodes | primitives | materials: a scene that fits is staged in shared memory whole, by one bulk copy
	const size_t nodeBytes = cs.nodes.size() * sizeof(Node), primBytes = cs.prims.size() * sizeof(Prim), matBytes = cs.mats.size() * sizeof(Mat);
	DevBuf blob;
	CK(blob.alloc(nodeBytes + primBytes + matBytes));
	char *const b = blob.as<char>();
	CK(cudaMemcpyAsync(b, cs.nodes.data(), nodeBytes, cudaMemcpyHostToDevice, c->stream));
	CK(cudaMemcpyAsync(b + nodeBytes, cs.prims.data(), primBytes, cudaMemcpyHostToDevice, c->stream));
	CK(cudaMemcpyAsync(b + nodeBytes + primBytes, cs.mats.data(), matBytes, cudaMemcpyHostToDevice, c->stream));
	CK(cudaStreamSynchronize(c->stream)); // (also: no render still reads the scene replaced here)
	c->sceneBlob = std::move(blob);
	c->mats = reinterpret_cast<Mat *>(b + nodeBytes + primBytes);
	c->lightRecs = std::move(lights);
	c->lightCount = uint32_t(lt.recs.size());
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

// pt_set_scene (objects) and pt_set_scene_xform (xobjects: objects given by their world-to-local transform and box)
static int setScene(pt_context *c, const std::string &fn, size_t count, const pt_object_desc *objects, const pt_object_xform_desc *xobjects)
{
	if (!c) return setError(PT_E_INVALID, fn + ": null context");
	if (count == 0)
	{
		printf("Setting an empty scene is not allowed!\n"); // Pathtracer.cpp:115
		return PT_OK;
	}
	if (!objects && !xobjects) return setError(PT_E_INVALID, fn + ": null objects");
	std::vector<pt_object_desc> descs;
	std::vector<ObjectXform> xf;
	if (xobjects)
	{
		descs.resize(count);
		xf.resize(count);
		for (size_t i = 0; i < count; ++i)
		{
			memset(&descs[i], 0, sizeof descs[i]);
			descs[i].type = xobjects[i].type;
			descs[i].scale[0] = descs[i].scale[1] = descs[i].scale[2] = 1.0f;
			descs[i].material = xobjects[i].material;
			memset(&xf[i], 0, sizeof xf[i]);
			memcpy(xf[i].w2l, xobjects[i].world_to_local, sizeof xf[i].w2l);
			memcpy(xf[i].bmin, xobjects[i].aabb_min, 12);
			memcpy(xf[i].bmax, xobjects[i].aabb_max, 12);
		}
		objects = descs.data();
	}
	CompiledScene cs;
	std::string err;
	if (!compileScene(count, objects, c->maxLeaf, cs, err, c->maxGlobal, xobjects ? xf.data() : nullptr, c->bvhBuilder)) return setError(PT_E_LIMIT, fn + ": " + err);
	LightTable lt;
	buildLightTable(cs, lt);
	// the BVH (and the emitter table) is built ONCE on the host; a multi-GPU context replicates the compiled scene on every device
	int r = uploadScene(c, cs, lt);
	if (r == PT_OK) c->aovValid = false; // the guide buffers show the previous scene
	for (size_t i = 0; r == PT_OK && i < c->peers.size(); ++i) r = uploadScene(c->peers[i], cs, lt);
	return r;
}

int pt_set_scene(pt_context *c, size_t count, const pt_object_desc *objects)
{
	PT_TRY
	return setScene(c, "pt_set_scene", count, objects, nullptr);
	PT_CATCH(PT_E_LIMIT)
}

int pt_set_scene_xform(pt_context *c, size_t count, const pt_object_xform_desc *objects)
{
	PT_TRY
	return setScene(c, "pt_set_scene_xform", count, nullptr, objects);
	PT_CATCH(PT_E_LIMIT)
}

// device copy of the texture table; with tex_unit = 0 the texture objects are left out and the kernels filter in software
static int uploadTextureTable(pt_context *c)
{
	TexDesc tmp[kMaxTextures];
	memcpy(tmp, c->texHost, sizeof tmp);
	if (!c->texUnit)
		for (TexDesc &t : tmp) t.texObj = 0;
	if (cudaMemcpyAsync(c->texDev.p, tmp, sizeof tmp, cudaMemcpyHostToDevice, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
		return setError(PT_E_CUDA, "pt_load_texture: table upload failed");
	return PT_OK;
}

static uint32_t loadTextureMemOne(pt_context *c, uint32_t width, uint32_t height, int is_hdr, const void *rgba)
{
	PT_TRY
	if (!c || !rgba || width == 0 || height == 0) return 0;
	if (c->textures.size() >= kMaxTextures) return 0; // Pathtracer.cpp:236-240
	if (cudaSetDevice(c->device) != cudaSuccess) return 0;
	const size_t bytes = size_t(width) * height * (is_hdr ? 16 : 4);
	Texture tex;
	if (tex.texels.alloc(bytes) != cudaSuccess) { setError(PT_E_CUDA, "pt_load_texture: cudaMalloc failed"); return 0; }
	if (cudaMemcpyAsync(tex.texels.p, rgba, bytes, cudaMemcpyHostToDevice, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
	{
		setError(PT_E_CUDA, "pt_load_texture: upload failed");
		return 0;
	}
	// the same texels behind a texture object (Pathtracer.cpp:259-288: array, wrap U / clamp V, linear filter, normalised
	// coordinates; 8-bit texels read as normalised floats)
	cudaChannelFormatDesc fmt = is_hdr ? cudaCreateChannelDesc<float4>() : cudaCreateChannelDesc<uchar4>();
	cudaTextureObject_t obj = 0;
	bool ok = cudaMallocArray(&tex.array, &fmt, width, height) == cudaSuccess;
	const size_t pitch = size_t(width) * (is_hdr ? 16 : 4);
	ok = ok && cudaMemcpy2DToArray(tex.array, 0, 0, rgba, pitch, pitch, height, cudaMemcpyHostToDevice) == cudaSuccess;
	if (ok)
	{
		cudaResourceDesc rd;
		memset(&rd, 0, sizeof rd);
		rd.resType = cudaResourceTypeArray;
		rd.res.array.array = tex.array;
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
		cudaGetLastError();
		setError(PT_E_CUDA, "pt_load_texture: texture object creation failed");
		return 0;
	}
	tex.object = obj;
	// the record is complete: it becomes the next handle
	c->texHost[c->textures.size()] = TexDesc{tex.texels.p, width, height, is_hdr ? 1u : 0u, 0u, (unsigned long long)obj};
	c->textures.push_back(std::move(tex));
	if (uploadTextureTable(c) != PT_OK) { c->textures.pop_back(); return 0; }
	return uint32_t(c->textures.size());
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
	if (c->textures.size() >= kMaxTextures) return 0;
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
	s.sceneBlob = c->sceneBlob.as<float4>();
	s.mats = c->mats;
	s.textures = c->texDev.as<TexDesc>();
	s.nodeCount = c->nodeCount;
	s.primCount = c->primCount;
	s.globalCount = c->globalCount;
	s.treeNodeCount = c->treeNodeCount;
	s.texCount = uint32_t(c->textures.size());
	s.skybox = (c->skybox <= s.texCount) ? c->skybox : 0;
	return s;
}

// option "env_is": make sure the device holds the importance distribution of the current sky texture (texels read back from the
// linear device copy the loader keeps)
static int ensureEnvDistribution(pt_context *c, uint32_t handle)
{
	if (c->envHandle == handle && c->envAlias.p) return PT_OK;
	const TexDesc &t = c->texHost[handle - 1];
	const size_t bytes = size_t(t.width) * t.height * (t.isHdr ? 16 : 4);
	std::vector<unsigned char> texels(bytes);
	CK(cudaMemcpyAsync(texels.data(), t.texels, bytes, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	EnvDistribution d;
	buildEnvDistribution(t.width, t.height, t.isHdr != 0, texels.data(), d);
	DevBuf alias, density;
	CK(alias.alloc(d.alias.size() * 4));
	CK(density.alloc(d.density.size() * 4));
	CK(cudaMemcpyAsync(alias.p, d.alias.data(), d.alias.size() * 4, cudaMemcpyHostToDevice, c->stream));
	CK(cudaMemcpyAsync(density.p, d.density.data(), d.density.size() * 4, cudaMemcpyHostToDevice, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	// the tables of `handle` are complete: they replace the cached ones together with their size and handle
	c->envAlias = std::move(alias);
	c->envDensity = std::move(density);
	c->envCols = d.cols;
	c->envRows = d.rows;
	c->envHandle = handle;
	return PT_OK;
}

// the ten Philox round keys of `seed` (RenderParams::philoxKeys)
static void philoxKeys(uint64_t seed, uint32_t (&keys)[20])
{
	const uint32_t lo = uint32_t(seed), hi = uint32_t(seed >> 32);
	for (uint32_t i = 0; i < 10; ++i) { keys[2 * i] = lo + i * 0x9E3779B9u; keys[2 * i + 1] = hi + i * 0xBB67AE85u; }
}

// option "jitter" = 0: the pixel-centre coordinates (RenderParams::centreU / centreV), made on first use
static int ensureCentreTables(pt_context *c)
{
	if (c->centreUV.p) return PT_OK;
	// (this file is compiled without FMA contraction: the division is the IEEE one of the reference's primary pass)
	std::vector<float> uv(size_t(c->width) + c->height);
	for (uint32_t x = 0; x < c->width; ++x) uv[x] = (float(x) + 0.5f) / float(c->width);
	for (uint32_t y = 0; y < c->height; ++y) uv[c->width + y] = (float(y) + 0.5f) / float(c->height);
	DevBuf centres;
	CK(centres.alloc(uv.size() * sizeof(float)));
	CK(cudaMemcpy(centres.p, uv.data(), uv.size() * sizeof(float), cudaMemcpyHostToDevice));
	c->centreUV = std::move(centres);
	return PT_OK;
}

// the first-bounce stratification of `len` samples (RenderParams::strataPer): 2^k cells, k <= 8, at least 16 samples per cell - the lanes of
// a pass of the one-pixel-per-warp kernel then hold samples of one or two neighbouring cells; fewer than 4 samples are not stratified
static void strataRule(const LaunchConfig &cfg, uint32_t len, uint32_t &per, uint32_t &bitsA, uint32_t &bitsB, float &invPer)
{
	per = bitsA = bitsB = 0;
	invPer = 0.0f;
	if (len < 4u || len >= (1u << 21)) return;
	uint32_t k = 2;
	while (k < 8u && (len >> (k + 1u)) >= 16u) ++k; // measured at 4096 spp: 32 / 64 / 128 / 256 / 512 cells -> 489 / 479 / 470 / 465 / 468 ms
	if (cfg.strataK > 0) k = uint32_t(cfg.strataK);  // (experiments: another cell count than the rule's)
	while (k > 2u && (len >> k) == 0u) --k;
	bitsA = (k + 1u) / 2u;
	bitsB = k / 2u;
	per = len >> k;
	invPer = 1.0f / float(per);
}

// option "adaptive": the intervals of a pixel's samples, [0, c0), [c0, c1), ... with c0 = min(m, spp), c_{j+1} = min(2 c_j, spp), each
// stratified on its own when the launch stratifies, and the constants of the stopping test and the scaling at their ends
static void adaptIntervals(const LaunchConfig &cfg, uint32_t spp, uint32_t minSpp, bool stratify, RenderParams &p)
{
	uint32_t start = 0, end = minSpp < spp ? minSpp : spp, j = 0;
	for (;; ++j)
	{
		AdaptInterval &iv = p.adapt[j];
		iv.start = start;
		iv.end = end;
		if (stratify) strataRule(cfg, end - start, iv.strataPer, iv.strataBitsA, iv.strataBitsB, iv.strataInvPer);
		else { iv.strataPer = iv.strataBitsA = iv.strataBitsB = 0; iv.strataInvPer = 0.0f; }
		iv.invN = float(1.0 / double(end));
		iv.invNN1 = end > 1u ? float(1.0 / (double(end) * double(end - 1u))) : 0.0f;
		iv.scale = float(spp) / float(end); // (this file is compiled without FMA contraction: the IEEE quotient)
		if (end == spp) break;
		start = end;
		end = end > spp / 2u ? spp : 2u * end;
	}
	p.adaptIntervals = j + 1u;
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
	CK(cudaMemsetAsync(c->counters.p, 0, kCtrCount * sizeof(unsigned long long), c->stream));
	const bool run = c->nodeCount >= 1 && c->primCount >= 1 && spp > 0; // Pathtracer.cpp:174
	if (run)
	{
		RenderParams p;
		p.scene = sceneDev(c);
		p.cam = *camera;
		p.accum = c->accum;
		p.counters = c->counters.as<unsigned long long>();
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
		philoxKeys(c->seed, p.philoxKeys);
		p.maxBounces = c->maxBounces;
		p.regenLow = c->launch.regenLow > 0 ? uint32_t(c->launch.regenLow) : 16u;
		// first-bounce stratification (RenderParams::strataPer); option "adaptive" always runs the one-pixel-per-warp kernel
		const bool adaptive = c->adaptTau > 0.0f;
		const bool stratify = (adaptive || onePixelPerWarp(c->launch, spp)) && (c->launch.stratify < 0 ? spp >= 128u : c->launch.stratify != 0);
		if (stratify) strataRule(c->launch, spp, p.strataPer, p.strataBitsA, p.strataBitsB, p.strataInvPer);
		p.beam = c->launch.beam < 0 ? (spp >= 128u ? 1u : 0u) : uint32_t(c->launch.beam != 0);
		c->launch.adaptive = adaptive;
		if (adaptive)
		{
			if (c->noJitter || c->firstHit) return setError(PT_E_INVALID, "pt_render: adaptive and the parity aids (jitter = 0, first_hit = 1) cannot be combined");
			if (c->launch.variant == 4) return setError(PT_E_INVALID, "pt_render: adaptive runs in the one-pixel-per-warp kernel only (variant 0 or 12, not 4)");
			if (!c->sampleCounts.p) CK(c->sampleCounts.alloc(size_t(c->width) * c->height * sizeof(uint32_t)));
			adaptIntervals(c->launch, spp, c->adaptMinSpp, stratify, p);
			p.sampleCounts = c->sampleCounts.as<uint32_t>();
			p.adaptTau = c->adaptTau;
			p.adaptFloor = PT_ADAPTIVE_FLOOR;
		}
		p.alpha = c->alpha;
		// which twin of the trace kernel runs: the options compiled into twins are exclusive
		c->launch.twin = Twin::Plain;
		if (c->envIS && p.scene.skybox != 0)
		{
			const int rc = ensureEnvDistribution(c, p.scene.skybox);
			if (rc != PT_OK) return rc;
			p.scene.env.alias = c->envAlias.as<const uint2>();
			p.scene.env.density = c->envDensity.as<float>();
			p.scene.env.cols = c->envCols;
			p.scene.env.rows = c->envRows;
			c->launch.twin = Twin::EnvIS;
		}
		if (c->noJitter)
		{
			const int rc = ensureCentreTables(c);
			if (rc != PT_OK) return rc;
			p.centreU = c->centreUV.as<float>();
			p.centreV = c->centreUV.as<float>() + c->width;
			p.aids |= kAidPixelCentre;
		}
		p.firstHitIndex = c->firstHit ? c->firstHitIndex.as<int32_t>() : nullptr;
		p.firstHitT = c->firstHit ? c->firstHitT.as<float>() : nullptr;
		if (c->firstHit) p.aids |= kAidFirstHit;
		if (p.aids)
		{
			if (c->launch.twin == Twin::EnvIS) return setError(PT_E_INVALID, "pt_render: the parity aids and env_is cannot be combined");
			c->launch.twin = Twin::Aids;
		}
		if (c->lightIS)
		{
			if (c->envIS) return setError(PT_E_INVALID, "pt_render: light_is and env_is cannot be combined (one sampled light source per kernel)");
			if (c->noJitter || c->firstHit) return setError(PT_E_INVALID, "pt_render: light_is and the parity aids (jitter = 0, first_hit = 1) cannot be combined");
			// a scene without emitters renders with the plain kernel: the same bits as without the option
			if (c->lightCount != 0)
			{
				p.lights.recs = c->lightRecs.as<float4>();
				p.lights.count = c->lightCount;
				c->launch.twin = Twin::LightIS;
			}
		}
		c->launch.stackLevels = int(c->bvhDepth) + 2;
		CK(cudaEventRecord(c->evStart, c->stream)); // (all allocations are behind us: the events bracket the device work alone)
		// pixel partition: the pixels of the other ranks hold zeros, so that the sum over ranks is the image
		if (ignore_history && c->pixelStride > 1u && !c->skipPartitionClear) CK(cudaMemsetAsync(c->accum, 0, size_t(c->width) * c->height * sizeof(float4), c->stream));
		if (adaptive && c->pixelStride > 1u) CK(cudaMemsetAsync(c->sampleCounts.p, 0, size_t(c->width) * c->height * sizeof(uint32_t), c->stream)); // (the other ranks' pixels: 0)
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
		CK(cudaMemcpy(h, c->counters.p, sizeof h, cudaMemcpyDeviceToHost));
		{
			const unsigned long long all = (unsigned long long)c->width * c->height;
			const unsigned long long own = all > c->pixelOffset ? (all - c->pixelOffset + c->pixelStride - 1u) / c->pixelStride : 0ull;
			c->stats.samples = c->launch.adaptive ? h[kCtrSamples] : own * spp;
		}
		c->countsValid = c->launch.adaptive;
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
	if (c->adaptTau > 0.0f && c->partition != 0)
		return setError(PT_E_INVALID, "pt_render: adaptive and the multi-GPU sample partition cannot be combined (each device would stop a pixel on its own share of the samples)");
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

// the image getters: the accumulation x scale (HDR) or tone-mapped (LDR) into device staging, copied to pinned host memory (both
// allocated by the first call).  `src`: the float4 buffer to read, null = the image (the accumulation, or a multi-GPU job's reduce)
static const void *readBack(pt_context *c, bool ldr, float scale, const float4 *src = nullptr)
{
	if (cudaSetDevice(c->device) != cudaSuccess) return nullptr;
	const uint32_t px = c->width * c->height;
	const size_t bytes = size_t(px) * (ldr ? sizeof(uchar4) : sizeof(float4));
	DevBuf &dev = ldr ? c->ldrDev : c->scaledDev;
	HostBuf &host = ldr ? c->hostLdr : c->hostHdr;
	const std::string fn = ldr ? "pt_get_ldr: " : "pt_get_hdr: ";
	if ((!dev.p && dev.alloc(bytes) != cudaSuccess) || (!host.p && host.alloc(bytes) != cudaSuccess))
	{
		setError(PT_E_CUDA, fn + cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	if (!src) src = c->imageSource ? c->imageSource : c->accum;
	if (ldr) launchTonemap(src, dev.as<uchar4>(), px, scale, c->stream);
	else launchScale(src, dev.as<float4>(), px, scale, c->stream);
	if (cudaMemcpyAsync(host.p, dev.p, bytes, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
	{
		setError(PT_E_CUDA, fn + cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	return host.p;
}

const float *pt_get_hdr(pt_context *c)
{
	if (!c) return nullptr;
	return static_cast<const float *>(readBack(c, false, 1.0f / fmaxf(float(c->accumulatedFrames), 1.0f))); // Pathtracer.cpp:307
}

const float *pt_get_hdr_mean(pt_context *c)
{
	if (!c) return nullptr;
	return static_cast<const float *>(readBack(c, false, 1.0f / fmaxf(float(c->totalSamples), 1.0f)));
}

const float *pt_get_hdr_sum(pt_context *c)
{
	if (!c) return nullptr;
	return static_cast<const float *>(readBack(c, false, 1.0f));
}

const uint8_t *pt_get_ldr(pt_context *c)
{
	if (!c) return nullptr;
	// tonemap.cu:17 divides by float(accumulatedSampleCount) via reciprocal-multiply; 0 frames -> division by zero in the
	// reference; here the accumulation is zero in that case and the scale is clamped like getHDRImageData's
	return static_cast<const uint8_t *>(readBack(c, true, 1.0f / fmaxf(float(c->accumulatedFrames), 1.0f)));
}

int pt_render_aov(pt_context *c, const pt_camera_desc *camera, uint32_t spp)
{
	PT_TRY
	if (!c || !camera) return setError(PT_E_INVALID, "pt_render_aov: bad arguments");
	if (spp == 0) return setError(PT_E_INVALID, "pt_render_aov: spp must be at least 1");
	if (c->nodeCount == 0) return setError(PT_E_INVALID, "pt_render_aov: no scene");
	CK(cudaSetDevice(c->device));
	const size_t bytes = size_t(c->width) * c->height * sizeof(float4);
	for (DevBuf &b : c->aov)
		if (!b.p) CK(b.alloc(bytes));
	AovParams p;
	p.scene = sceneDev(c);
	computeCamera(*camera, p.cam);
	p.width = c->width;
	p.height = c->height;
	p.spp = spp;
	philoxKeys(c->seed, p.philoxKeys);
	if (c->noJitter)
	{
		const int rc = ensureCentreTables(c);
		if (rc != PT_OK) return rc;
		p.centreU = c->centreUV.as<float>();
		p.centreV = c->centreUV.as<float>() + c->width;
	}
	p.albedo = c->aov[PT_AOV_ALBEDO].as<float4>();
	p.normal = c->aov[PT_AOV_NORMAL].as<float4>();
	p.position = c->aov[PT_AOV_POSITION].as<float4>();
	launchAov(p, c->stream);
	CK(cudaGetLastError());
	CK(cudaStreamSynchronize(c->stream));
	c->aovValid = true;
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

const float *pt_get_aov(pt_context *c, int kind)
{
	if (!c || kind < PT_AOV_ALBEDO || kind > PT_AOV_POSITION) { setError(PT_E_INVALID, "pt_get_aov: bad arguments"); return nullptr; }
	if (!c->aov[kind].p) { setError(PT_E_INVALID, "pt_get_aov: no pt_render_aov yet"); return nullptr; }
	return static_cast<const float *>(readBack(c, false, 1.0f, c->aov[kind].as<float4>())); // (x 1: the buffer's own bits)
}

int pt_denoise(pt_context *c, const pt_denoise_params *params)
{
	PT_TRY
	if (!c) return setError(PT_E_INVALID, "pt_denoise: null context");
	const pt_denoise_params q = params ? *params
	                                   : pt_denoise_params{ PT_DENOISE_DEFAULT_ITERATIONS, PT_DENOISE_DEFAULT_SIGMA_COLOR, PT_DENOISE_DEFAULT_SIGMA_NORMAL,
	                                                        PT_DENOISE_DEFAULT_SIGMA_POSITION };
	if (q.iterations > 12) return setError(PT_E_INVALID, "pt_denoise: at most 12 iterations");
	for (float s : { q.sigma_color, q.sigma_normal, q.sigma_position })
		if (!(s >= 0.0f) || !std::isfinite(s)) return setError(PT_E_INVALID, "pt_denoise: every sigma must be finite and not negative");
	if (!c->aov[0].p) return setError(PT_E_INVALID, "pt_denoise: no guide buffers (pt_render_aov first)");
	if (!c->aovValid) return setError(PT_E_INVALID, "pt_denoise: the guide buffers are stale (the scene changed since pt_render_aov)");
	CK(cudaSetDevice(c->device));
	const size_t bytes = size_t(c->width) * c->height * sizeof(float4);
	if (!c->denoised.p) CK(c->denoised.alloc(bytes));
	if (q.iterations > 1 && !c->denoiseTmp.p) CK(c->denoiseTmp.alloc(bytes));
	const float4 *src = c->imageSource ? c->imageSource : c->accum;
	if (q.iterations == 0) CK(cudaMemcpyAsync(c->denoised.p, src, bytes, cudaMemcpyDeviceToDevice, c->stream));
	// the filter runs on the sums: the colour term's sigma is scaled by the sample count, which in exact arithmetic is the filter of the
	// per-sample mean
	const double n = double(c->totalSamples > 0 ? c->totalSamples : 1ull);
	auto inverseSquare = [](double s) { return float(std::fmin(1.0 / (s * s), double(FLT_MAX))); }; // (sigma 0: FLT_MAX, see denoise.cu)
	for (uint32_t i = 0; i < q.iterations; ++i)
	{
		AtrousParams a;
		a.in = src;
		a.out = ((q.iterations - 1u - i) & 1u) ? c->denoiseTmp.as<float4>() : c->denoised.as<float4>(); // the last iteration lands in `denoised`
		a.albedo = c->aov[PT_AOV_ALBEDO].as<float4>();
		a.normal = c->aov[PT_AOV_NORMAL].as<float4>();
		a.position = c->aov[PT_AOV_POSITION].as<float4>();
		a.width = c->width;
		a.height = c->height;
		a.step = 1u << i;
		a.invColor2 = inverseSquare(double(q.sigma_color) * n / double(a.step));
		a.invNormal2 = inverseSquare(double(q.sigma_normal));
		a.sigmaPosition = q.sigma_position;
		a.demodulate = i == 0;
		a.remodulate = i + 1u == q.iterations;
		launchAtrous(a, c->stream);
		src = a.out;
	}
	CK(cudaGetLastError());
	CK(cudaStreamSynchronize(c->stream));
	c->hasDenoised = true;
	c->denoisedFrames = c->accumulatedFrames;
	c->denoisedSamples = c->totalSamples;
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
}

// the denoised sum buffer through readBack, with the counts of the image it was made from
static const void *readDenoised(pt_context *c, bool ldr, bool mean)
{
	if (!c) return nullptr;
	if (!c->hasDenoised) { setError(PT_E_INVALID, "pt_get_denoised_*: no pt_denoise yet"); return nullptr; }
	const float count = mean ? float(c->denoisedSamples) : float(c->denoisedFrames);
	return readBack(c, ldr, 1.0f / fmaxf(count, 1.0f), c->denoised.as<float4>());
}

const float *pt_get_denoised_hdr(pt_context *c) { return static_cast<const float *>(readDenoised(c, false, false)); }
const float *pt_get_denoised_hdr_mean(pt_context *c) { return static_cast<const float *>(readDenoised(c, false, true)); }
const uint8_t *pt_get_denoised_ldr(pt_context *c) { return static_cast<const uint8_t *>(readDenoised(c, true, false)); }

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
	else if (k == "adaptive")
	{
		if (!(value >= 0.0) || !std::isfinite(value)) return setError(PT_E_INVALID, "pt_set_option: adaptive must be a finite threshold >= 0 (0 = off)");
		c->adaptTau = float(value);
	}
	else if (k == "adaptive_min_spp")
	{
		if (!(value >= 32.0) || !(value <= 4294967295.0)) return setError(PT_E_INVALID, "pt_set_option: adaptive_min_spp must be at least 32");
		c->adaptMinSpp = uint32_t(value);
	}
	else if (k == "first_hit")
	{
		if (value != 0 && !c->firstHitIndex.p)
		{
			const size_t px = size_t(c->width) * c->height;
			CK(cudaSetDevice(c->device));
			DevBuf index, t;
			CK(index.alloc(px * 4));
			CK(t.alloc(px * 4));
			CK(cudaMemset(index.p, 0xff, px * 4));
			CK(cudaMemset(t.p, 0, px * 4));
			c->firstHitIndex = std::move(index);
			c->firstHitT = std::move(t);
		}
		c->firstHit = value != 0;
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
	if (!c->firstHitIndex.p) return setError(PT_E_INVALID, "pt_get_first_hit: option first_hit was not set before pt_render");
	const size_t px = size_t(c->width) * c->height;
	CK(cudaSetDevice(c->device));
	CK(cudaMemcpyAsync(hit_index, c->firstHitIndex.p, px * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaMemcpyAsync(hit_t, c->firstHitT.p, px * 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	return PT_OK;
}

int pt_get_sample_counts(pt_context *c, uint32_t *counts)
{
	PT_TRY
	if (!c || !counts) return setError(PT_E_INVALID, "pt_get_sample_counts: bad arguments");
	if (!c->countsValid) return setError(PT_E_INVALID, "pt_get_sample_counts: the last pt_render was not adaptive (option \"adaptive\" > 0)");
	const size_t px = size_t(c->width) * c->height;
	if (c->peers.empty())
	{
		CK(cudaSetDevice(c->device));
		CK(cudaMemcpyAsync(counts, c->sampleCounts.p, px * 4, cudaMemcpyDeviceToHost, c->stream));
		CK(cudaStreamSynchronize(c->stream));
		return PT_OK;
	}
	// pixel partition: device i rendered the pixels i, i + N, ... and holds their counts in its own buffer
	std::vector<pt_context *> all = { c };
	all.insert(all.end(), c->peers.begin(), c->peers.end());
	std::vector<uint32_t> part(px);
	for (size_t i = 0; i < all.size(); ++i)
	{
		pt_context *d = all[i];
		CK(cudaSetDevice(d->device));
		CK(cudaMemcpyAsync(part.data(), d->sampleCounts.p, px * 4, cudaMemcpyDeviceToHost, d->stream));
		CK(cudaStreamSynchronize(d->stream));
		for (size_t q = i; q < px; q += all.size()) counts[q] = part[q];
	}
	CK(cudaSetDevice(c->device));
	return PT_OK;
	PT_CATCH(PT_E_LIMIT)
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
