// C ABI of libgarden_sceneprep.so (include/garden_sceneprep.h): context, staging uploads, frame orchestration, results.
// Orchestration mirrors MeshRenderSystem::prepareMeshes (source/system/render/mesh.cpp:331-553) for all views of a frame.
#include "sceneprep_internal.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <functional>
#include <new>

using namespace gsp;

static std::string gCreateError;

#define GSP_CUDA(call)                                                                             \
	do {                                                                                           \
		cudaError_t err__ = (call);                                                                \
		if (err__ != cudaSuccess) {                                                                \
			c.error = std::string(#call) + ": " + cudaGetErrorString(err__);                       \
			return GSP_ERR_CUDA;                                                                   \
		}                                                                                          \
	} while (0)

extern "C" { static int fetchWait(Context& c); }
template<class F> static void parallelFor(uint32_t n, F fn, uint32_t minParallel = 1u << 18);

static int fail(Context& c, int code, const char* message)
{
	c.error = message;
	return code;
}

template<class T>
static cudaError_t ensureDevice(T*& ptr, size_t& cap, size_t need, bool keep = false, cudaStream_t stream = nullptr)
{
	if (need <= cap && ptr)
		return cudaSuccess;
	size_t newCap = std::max(need, cap + cap / 2);
	if (newCap == 0) newCap = 1;
	T* fresh = nullptr;
	cudaError_t err = cudaMalloc((void**)&fresh, newCap * sizeof(T));
	if (err != cudaSuccess)
		return err;
	if (ptr)
	{
		if (keep && cap)
			cudaMemcpyAsync(fresh, ptr, cap * sizeof(T), cudaMemcpyDeviceToDevice, stream);
		cudaStreamSynchronize(stream);
		cudaFree(ptr);
	}
	ptr = fresh; cap = newCap;
	return cudaSuccess;
}
template<class T>
static cudaError_t ensureDevice32(T*& ptr, uint32_t& cap, size_t need)
{
	size_t cap64 = cap;
	cudaError_t err = ensureDevice(ptr, cap64, need);
	cap = (uint32_t)cap64;
	return err;
}

extern "C"
{

const char* gsp_version(void) { return "garden_sceneprep 0.1 sm_100a"; }

int gsp_create(int device, gsp_context** out)
{
	if (!out)
		return GSP_ERR_INVALID;
	*out = nullptr;
	int deviceCount = 0;
	cudaError_t err = cudaGetDeviceCount(&deviceCount);
	if (err != cudaSuccess || deviceCount == 0)
	{
		gCreateError = std::string("no CUDA device available (") + cudaGetErrorString(err) +
			"); this library has no CPU fallback";
		return GSP_ERR_CUDA;
	}
	if (device < 0 || device >= deviceCount)
	{
		gCreateError = "device index out of range";
		return GSP_ERR_INVALID;
	}
	cudaDeviceProp prop;
	err = cudaGetDeviceProperties(&prop, device);
	if (err != cudaSuccess || prop.major < 10)
	{
		gCreateError = "device is not sm_100 class (kernels are built for sm_100a only)";
		return GSP_ERR_CUDA;
	}
	auto ctx = new (std::nothrow) gsp_context();
	if (!ctx)
		return GSP_ERR_NOMEM;
	Context& c = ctx->c;
	c.device = device;
	c.smCount = (uint32_t)std::max(1, prop.multiProcessorCount);
	memset(c.segOf, -1, sizeof(c.segOf));
	if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c.ownStream, cudaStreamNonBlocking) != cudaSuccess ||
		cudaStreamCreateWithFlags(&c.copyStream, cudaStreamNonBlocking) != cudaSuccess ||
		cudaEventCreateWithFlags(&c.copyEvent, cudaEventDisableTiming) != cudaSuccess ||
		cudaMalloc((void**)&c.dCounters, kCtrCount * sizeof(uint32_t)) != cudaSuccess ||
		cudaMallocHost((void**)&c.hCounters, (kCtrCount + 16) * sizeof(uint32_t)) != cudaSuccess)
	{
		gCreateError = std::string("context allocation failed: ") + cudaGetErrorString(cudaGetLastError());
		delete ctx;
		return GSP_ERR_CUDA;
	}
	c.stream = c.ownStream;
	c.dError = c.dCounters + kCtrError;
	cudaMemset(c.dCounters, 0, kCtrCount * sizeof(uint32_t));
	memset(c.hCounters, 0, kCtrCount * sizeof(uint32_t));
	*out = ctx;
	return GSP_OK;
}

void gsp_destroy(gsp_context* ctx)
{
	if (!ctx)
		return;
	Context& c = ctx->c;
	cudaSetDevice(c.device);
	cudaStreamSynchronize(c.stream);
	destroyExchange(c);
	if (c.copyStream) cudaStreamSynchronize(c.copyStream);
	auto& t = c.tf;
	cudaFree(t.rot); cudaFree(t.posSx); cudaFree(t.sYZ); cudaFree(t.parent); cudaFree(t.entity);
	cudaFree(t.parentEntity); cudaFree(t.flags); cudaFree(t.bound); cudaFree(t.record); cudaFree(t.rho); cudaFree(t.chainRoot); cudaFree(t.rootW); cudaFree(t.poolMask); cudaFree(t.entityToSlot);
	cudaFree(t.tBits); cudaFree(t.tBlockCount); cudaFree(t.tList); cudaFree(t.tIndex); cudaFree(t.tWorld);
	for (auto& p : c.pools)
	{
		cudaFree(p.aabbA); cudaFree(p.aabbB); cudaFree(p.entity); cudaFree(p.tslot); cudaFree(p.flags);
		cudaFree(p.ready); cudaFree(p.world); cudaFree(p.worldPos); cudaFree(p.visible); cudaFree(p.visBits);
		cudaFree(p.radius); cudaFree(p.surList); cudaFree(p.surTs); cudaFree(p.surBits); cudaFree(p.blockCount);
	}
	cudaFree(c.frameZero);
	cudaFree(c.dSegments); cudaFree(c.keys[0]); cudaFree(c.keys[1]); cudaFree(c.payloads[0]); cudaFree(c.payloads[1]);
	cudaFree(c.records); cudaFree(c.dCounters); cudaFree(c.sortStatus);
	cudaFree(c.segTileOffset); cudaFree(c.dAosScratch);
	cudaFreeHost(c.hCounters); cudaFreeHost(c.hGather); cudaFreeHost(c.hRecords); cudaFreeHost(c.hVisible); cudaFree(c.dVisScratch);
	if (c.phaseEventsCreated)
	{
		for (auto& e : c.phaseEvents)
			cudaEventDestroy(e);
		for (auto& pe : c.poolEvents)
			for (auto& e : pe)
				cudaEventDestroy(e);
		for (auto& e : c.splitEvents)
			cudaEventDestroy(e);
	}
	cudaStreamSynchronize(c.copyStream);
	cudaStreamDestroy(c.copyStream);
	cudaEventDestroy(c.copyEvent);
	cudaStreamDestroy(c.ownStream);
	delete ctx;
}

const char* gsp_last_error(const gsp_context* ctx)
{
	return ctx ? ctx->c.error.c_str() : gCreateError.c_str();
}

int gsp_set_stream(gsp_context* ctx, void* cudaStream)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	GSP_CUDA(cudaSetDevice(c.device));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	c.stream = cudaStream ? (cudaStream_t)cudaStream : c.ownStream;
	return GSP_OK;
}

//----------------------------------------------------------------------------------------------------------------------
// Where the staging kernels read the caller's AoS bytes from:
//  * pinned / registered host memory (cudaMallocHost, cudaHostRegister, gsp_pin_host): read in place over PCIe by the
//    staging kernel ("zero copy") — no intermediate device buffer, the re-layout overlaps the transfer;
//  * device memory: read in place;
//  * pageable host memory: copied into a device scratch buffer first (cudaMemcpyAsync stages it through the driver), at
//    `scratchOffset`. A call with two sources puts the second behind the first and reserves room for both BEFORE the first
//    resolveSource: growing the scratch here would free the buffer the first source's pointer points into.
static int resolveSource(Context& c, const void* aos, size_t bytes, const void** src, size_t scratchOffset = 0)
{
	cudaPointerAttributes attr = {};
	cudaError_t err = cudaPointerGetAttributes(&attr, aos);
	if (err != cudaSuccess)
	{
		cudaGetLastError(); // (older drivers report unregistered host memory as an error)
		attr.type = cudaMemoryTypeUnregistered;
	}
	if ((attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) && attr.devicePointer)
	{
		*src = attr.devicePointer;
		return GSP_OK;
	}
	if (attr.type == cudaMemoryTypeHost && attr.devicePointer)
	{
		*src = attr.devicePointer;
		c.zeroCopyBytes += bytes;
		return GSP_OK;
	}
	size_t cap = c.dAosScratchCap;
	uint8_t* ptr = (uint8_t*)c.dAosScratch;
	GSP_CUDA(ensureDevice(ptr, cap, scratchOffset + bytes, false, c.stream));
	c.dAosScratch = ptr; c.dAosScratchCap = cap;
	GSP_CUDA(cudaMemcpyAsync((uint8_t*)c.dAosScratch + scratchOffset, aos, bytes, cudaMemcpyHostToDevice, c.stream));
	*src = (uint8_t*)c.dAosScratch + scratchOffset;
	return GSP_OK;
}

static bool isDevicePointer(const void* p)
{
	cudaPointerAttributes attr = {};
	if (cudaPointerGetAttributes(&attr, p) != cudaSuccess)
	{
		cudaGetLastError();
		return false;
	}
	return attr.type == cudaMemoryTypeDevice;
}

// A scattered dirty set as ONE upload: slots[count], then the components aos[slots[i]] back to back, then (ready != nullptr)
// the bytes ready[slots[i]], packed in pinned memory and copied into the device scratch buffer. Host memory only.
struct Gathered
{
	const uint32_t* slots;
	const uint8_t* aos;
	const uint8_t* ready;
};
static int uploadGathered(Context& c, const void* aos, uint32_t stride, const uint32_t* slots, uint32_t count,
	const uint8_t* ready, Gathered* out)
{
	const size_t listBytes = ((size_t)count * sizeof(uint32_t) + 15) & ~(size_t)15;
	const size_t aosBytes = (size_t)count * stride;
	const size_t bytes = listBytes + aosBytes + (ready ? count : 0);
	if (c.hGatherCap < bytes)
	{
		GSP_CUDA(cudaStreamSynchronize(c.stream));
		cudaFreeHost(c.hGather); c.hGather = nullptr; c.hGatherCap = 0;
		const size_t cap = bytes + bytes / 2;
		GSP_CUDA(cudaMallocHost((void**)&c.hGather, cap));
		c.hGatherCap = cap;
	}
	memcpy(c.hGather, slots, (size_t)count * sizeof(uint32_t));
	const uint8_t* src = (const uint8_t*)aos;
	uint8_t* packed = c.hGather + listBytes;
	uint8_t* packedReady = packed + aosBytes;
	parallelFor(count, [=](uint32_t first, uint32_t last)
	{
		for (uint32_t i = first; i < last; i++)
		{
			memcpy(packed + (size_t)i * stride, src + (size_t)slots[i] * stride, stride);
			if (ready)
				packedReady[i] = ready[slots[i]];
		}
	}, 1u << 14); // (each row is a cache miss at a scattered address: workers pay off far below the default threshold)
	size_t cap = c.dAosScratchCap;
	uint8_t* ptr = (uint8_t*)c.dAosScratch;
	GSP_CUDA(ensureDevice(ptr, cap, bytes, false, c.stream));
	c.dAosScratch = ptr; c.dAosScratchCap = cap;
	GSP_CUDA(cudaMemcpyAsync(c.dAosScratch, c.hGather, bytes, cudaMemcpyHostToDevice, c.stream));
	const uint8_t* d = (const uint8_t*)c.dAosScratch;
	out->slots = (const uint32_t*)d;
	out->aos = d + listBytes;
	out->ready = ready ? d + listBytes + aosBytes : nullptr;
	return GSP_OK;
}

int gsp_pin_host(void* ptr, size_t bytes)
{
	if (!ptr || !bytes)
		return GSP_ERR_INVALID;
	cudaError_t err = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
	if (err == cudaErrorHostMemoryAlreadyRegistered)
	{
		cudaGetLastError();
		return GSP_OK;
	}
	return err == cudaSuccess ? GSP_OK : GSP_ERR_CUDA;
}

int gsp_unpin_host(void* ptr)
{
	if (!ptr)
		return GSP_ERR_INVALID;
	cudaError_t err = cudaHostUnregister(ptr);
	if (err != cudaSuccess)
		cudaGetLastError();
	return err == cudaSuccess ? GSP_OK : GSP_ERR_CUDA;
}

int gsp_set_transforms(gsp_context* ctx, const void* aos, uint32_t stride, uint32_t occupancy)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if ((!aos && occupancy) || stride < kTfMinStride || (stride & 3))
		return fail(c, GSP_ERR_INVALID, "gsp_set_transforms: bad pointer or stride (need >= 80, multiple of 4)");
	GSP_CUDA(cudaSetDevice(c.device));
	auto& t = c.tf;
	if (occupancy > t.capacity || !t.rot)
	{
		uint32_t cap = std::max<uint32_t>(occupancy, t.capacity + t.capacity / 2);
		if (cap == 0) cap = 1;
		GSP_CUDA(cudaStreamSynchronize(c.stream));
		cudaFree(t.rot); cudaFree(t.posSx); cudaFree(t.sYZ); cudaFree(t.parent); cudaFree(t.entity);
		cudaFree(t.parentEntity); cudaFree(t.flags); cudaFree(t.bound); cudaFree(t.record); cudaFree(t.rho); cudaFree(t.chainRoot); cudaFree(t.rootW); cudaFree(t.poolMask);
		cudaFree(t.tBits); cudaFree(t.tBlockCount); cudaFree(t.tList); cudaFree(t.tIndex); cudaFree(t.tWorld);
		t.tBits = nullptr; t.tBlockCount = nullptr; t.tList = nullptr; t.tIndex = nullptr; t.tWorld = nullptr; t.splitCap = 0;
		t.bound = nullptr; t.record = nullptr; t.rho = nullptr; t.chainRoot = nullptr; t.rootW = nullptr; t.poolMask = nullptr;
		c.layoutDirty = true; // (tBucketCount is carved out of the per-frame zero block)
		t.rot = nullptr; t.posSx = nullptr; t.sYZ = nullptr; t.parent = nullptr; t.entity = nullptr;
		t.parentEntity = nullptr; t.flags = nullptr; t.capacity = 0;
		GSP_CUDA(cudaMalloc((void**)&t.rot, (size_t)cap * sizeof(float4)));
		GSP_CUDA(cudaMalloc((void**)&t.posSx, (size_t)cap * sizeof(float4)));
		GSP_CUDA(cudaMalloc((void**)&t.sYZ, (size_t)cap * sizeof(float2)));
		GSP_CUDA(cudaMalloc((void**)&t.parent, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.entity, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.parentEntity, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.bound, (size_t)cap * sizeof(float2)));
		GSP_CUDA(cudaMalloc((void**)&t.record, (size_t)cap * sizeof(float4)));
		GSP_CUDA(cudaMalloc((void**)&t.rho, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.chainRoot, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.rootW, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.poolMask, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.flags, (((size_t)cap + 1) & ~(size_t)1) * sizeof(uint16_t))); // whole 32-bit words: gsp_set_active updates a flag entry through the word that holds it
		t.capacity = cap;
	}
	t.occupancy = occupancy;
	t.cyclic = false;
	c.linkDirty = true; c.chainDirty = true; c.resultsValid = false; c.frameEnqueued = false;
	if (occupancy == 0)
		return GSP_OK;
	const void* src = nullptr;
	int rc = resolveSource(c, aos, (size_t)stride * occupancy, &src);
	if (rc) return rc;
	// one pass over the caller's bytes: SoA streams, entity / parent-entity ids, the largest live entity id
	uint32_t* dMax = c.dCounters + kCtrError + 1;
	GSP_CUDA(cudaMemsetAsync(dMax, 0, sizeof(uint32_t), c.stream));
	GSP_CUDA(cudaMemsetAsync(c.dError, 0, sizeof(uint32_t), c.stream));
	launchStageTransforms(c, src, stride, 0, occupancy, true, dMax);
	uint32_t* hScalars = c.hCounters + kCtrCount; // two pinned words past the frame counters
	GSP_CUDA(cudaMemcpyAsync(&hScalars[0], dMax, sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream)); // the caller's memory is free again
	const uint32_t maxEntity = hScalars[0];
	// entity -> slot map sized by the largest live entity id, then parent slots and chain lengths from the SoA copy
	GSP_CUDA(ensureDevice32(t.entityToSlot, t.entityCap, (size_t)maxEntity + 1));
	GSP_CUDA(cudaMemsetAsync(t.entityToSlot, 0, (size_t)t.entityCap * sizeof(uint32_t), c.stream));
	uint32_t* dFlag = dMax; // (read already) set when some chain is 255 links or longer, then when some chain is cyclic
	GSP_CUDA(cudaMemsetAsync(dFlag, 0, sizeof(uint32_t), c.stream));
	launchBuildHierarchy(c, dFlag);
	GSP_CUDA(cudaMemcpyAsync(&hScalars[1], c.dError, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream)); // error, flag
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	GSP_CUDA(cudaGetLastError());
	if (hScalars[1])
		return fail(c, GSP_ERR_HIERARCHY, "gsp_set_transforms: a parent entity has no TransformComponent");
	if (hScalars[2])
	{
		// deep chains are legal; cycles are recorded here and refused by every call that walks the chains (gsp_run,
		// gsp_set_active, gsp_animate), so those walks need no per-frame cycle guard
		GSP_CUDA(cudaMemsetAsync(dFlag, 0, sizeof(uint32_t), c.stream));
		launchFindCycles(c, dFlag);
		GSP_CUDA(cudaMemcpyAsync(&hScalars[2], dFlag, sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
		GSP_CUDA(cudaStreamSynchronize(c.stream));
		GSP_CUDA(cudaGetLastError());
		t.cyclic = hScalars[2] != 0;
	}
	return GSP_OK;
}

int gsp_update_transforms(gsp_context* ctx, const void* aos, uint32_t stride, uint32_t first, uint32_t count)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if ((!aos && count) || stride < kTfMinStride || (stride & 3) || (uint64_t)first + count > c.tf.occupancy)
		return fail(c, GSP_ERR_INVALID, "gsp_update_transforms: bad pointer, stride or range");
	if (count == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	// `aos` is the pool base (same pointer meaning as gsp_set_transforms); only the dirty range is uploaded.
	const void* src = nullptr;
	int rc = resolveSource(c, (const uint8_t*)aos + (size_t)first * stride, (size_t)stride * count, &src);
	if (rc) return rc;
	launchStageTransforms(c, src, stride, first, count, false, nullptr);
	c.chainDirty = true;
	GSP_CUDA(cudaStreamSynchronize(c.stream)); // the scratch buffer and the caller's memory are free again
	GSP_CUDA(cudaGetLastError());
	c.resultsValid = false; c.frameEnqueued = false;
	return GSP_OK;
}

int gsp_update_transforms_indexed(gsp_context* ctx, const void* aos, uint32_t stride, const uint32_t* slots, uint32_t count)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (((!aos || !slots) && count) || stride < kTfMinStride || (stride & 3))
		return fail(c, GSP_ERR_INVALID, "gsp_update_transforms_indexed: bad pointer or stride");
	if (count == 0)
		return GSP_OK;
	for (uint32_t i = 0; i < count; i++)
		if (slots[i] >= c.tf.occupancy)
			return fail(c, GSP_ERR_INVALID, "gsp_update_transforms_indexed: slot index out of range");
	GSP_CUDA(cudaSetDevice(c.device));
	Gathered g;
	int rc = uploadGathered(c, aos, stride, slots, count, nullptr, &g);
	if (rc) return rc;
	launchStageTransforms(c, g.aos, stride, 0, count, false, nullptr, g.slots);
	c.chainDirty = true;
	GSP_CUDA(cudaStreamSynchronize(c.stream)); // the pinned gather buffer is free again
	GSP_CUDA(cudaGetLastError());
	c.resultsValid = false; c.frameEnqueued = false;
	return GSP_OK;
}

int gsp_set_pool_count(gsp_context* ctx, uint32_t poolCount)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (poolCount > (uint32_t)kMaxPools)
		return fail(c, GSP_ERR_INVALID, "gsp_set_pool_count: too many pools");
	bool changed = c.poolCount != poolCount;
	for (uint32_t i = poolCount; i < (uint32_t)kMaxPools; i++)
	{
		changed = changed || c.pools[i].set;
		c.pools[i].set = false;
	}
	c.poolCount = poolCount;
	if (changed) // (re-stating the same count every frame, as a caller without dirty tracking does, keeps the list layout)
		c.layoutDirty = true;
	c.resultsValid = false; c.frameEnqueued = false;
	return GSP_OK;
}

int gsp_set_mesh_pool(gsp_context* ctx, uint32_t pool, uint32_t renderType, uint32_t drawReady, const void* aos,
	uint32_t stride, uint32_t occupancy, uint32_t count, const uint8_t* readyCounts)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (pool >= (uint32_t)kMaxPools || renderType > GSP_RT_UI || (!aos && occupancy) || stride < kMcMinStride || (stride & 3) ||
		occupancy > 0x0FFFFFFFu)
		return fail(c, GSP_ERR_INVALID, "gsp_set_mesh_pool: bad pool index, render type, pointer, stride or occupancy");
	GSP_CUDA(cudaSetDevice(c.device));
	auto& p = c.pools[pool];
	if (occupancy > p.capacity || !p.aabbA)
	{
		uint32_t cap = std::max<uint32_t>(occupancy, p.capacity + p.capacity / 2);
		if (cap == 0) cap = 1;
		GSP_CUDA(cudaStreamSynchronize(c.stream));
		cudaFree(p.aabbA); cudaFree(p.aabbB); cudaFree(p.entity); cudaFree(p.tslot); cudaFree(p.flags);
		cudaFree(p.ready); cudaFree(p.world); cudaFree(p.worldPos); cudaFree(p.visible); cudaFree(p.visBits);
		cudaFree(p.radius); cudaFree(p.surList); cudaFree(p.surTs); cudaFree(p.surBits); cudaFree(p.blockCount);
		p.visBits = nullptr; p.radius = nullptr; p.surList = nullptr; p.surTs = nullptr; p.surBits = nullptr; p.blockCount = nullptr; p.bucketCount = nullptr;
		p.aabbA = nullptr; p.aabbB = nullptr; p.entity = nullptr; p.tslot = nullptr; p.flags = nullptr; p.ready = nullptr;
		p.world = nullptr; p.worldPos = nullptr; p.visible = nullptr; p.cullStatus = nullptr; p.capacity = 0;
		GSP_CUDA(cudaMalloc((void**)&p.aabbA, (size_t)cap * sizeof(float4)));
		GSP_CUDA(cudaMalloc((void**)&p.aabbB, (size_t)cap * sizeof(float2)));
		GSP_CUDA(cudaMalloc((void**)&p.entity, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&p.tslot, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&p.flags, (size_t)cap));
		GSP_CUDA(cudaMalloc((void**)&p.ready, (size_t)cap));
		GSP_CUDA(cudaMalloc((void**)&p.world, (size_t)cap * kWorldStride * sizeof(float4)));
		GSP_CUDA(cudaMalloc((void**)&p.worldPos, (size_t)cap * sizeof(float4)));
		GSP_CUDA(cudaMalloc((void**)&p.visible, (size_t)cap));
		GSP_CUDA(cudaMalloc((void**)&p.radius, (size_t)cap * sizeof(float)));
		GSP_CUDA(cudaMalloc((void**)&p.surList, (size_t)cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&p.surTs, (size_t)cap * sizeof(uint32_t)));
		{
			const size_t preBlocks = ((size_t)cap + kPreTile - 1) / kPreTile;
			GSP_CUDA(cudaMalloc((void**)&p.surBits, preBlocks * (kPreTile / 32) * sizeof(uint32_t)));
			GSP_CUDA(cudaMalloc((void**)&p.blockCount, preBlocks * sizeof(uint32_t)));
		}
		p.cullTilesCap = (cap + kCullTile - 1) / kCullTile;
		GSP_CUDA(cudaMalloc((void**)&p.visBits, (size_t)p.cullTilesCap * kMaxViews * (kCullTile / 32) * sizeof(uint32_t)));
		p.capacity = cap;
		c.layoutDirty = true; // (the per-frame scratch of the pool is carved out of the context's zeroed block)
	}
	if (p.occupancy != occupancy || p.renderType != renderType || p.stride != stride || !p.set ||
		(p.count == 0) != (count == 0) || p.drawReady != drawReady)
		c.layoutDirty = true;
	p.occupancy = occupancy; p.count = count; p.stride = stride; p.renderType = renderType; p.drawReady = drawReady;
	p.hasReady = readyCounts != nullptr; p.set = true; p.visibleValid = false;
	if (pool >= c.poolCount) { c.poolCount = pool + 1; c.layoutDirty = true; }
	c.linkDirty = true; c.chainDirty = true; c.resultsValid = false; c.frameEnqueued = false;
	if (occupancy == 0)
		return GSP_OK;
	const void* src = nullptr;
	int rc = resolveSource(c, aos, (size_t)stride * occupancy, &src);
	if (rc) return rc;
	launchStagePool(c, pool, src, stride, 0, occupancy);
	if (readyCounts)
		GSP_CUDA(cudaMemcpyAsync(p.ready, readyCounts, occupancy, cudaMemcpyHostToDevice, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	GSP_CUDA(cudaGetLastError());
	return GSP_OK;
}

// Arguments every gsp_update_mesh_pool* call checks before it changes anything.
static int checkMeshUpdate(Context& c, uint32_t pool, uint32_t stride, bool pointers, const uint8_t* readyCounts, const char* who)
{
	if (pool >= (uint32_t)kMaxPools)
		return fail(c, GSP_ERR_INVALID, (std::string(who) + ": bad pool index").c_str());
	auto& p = c.pools[pool];
	if (!p.set)
		return fail(c, GSP_ERR_STATE, (std::string(who) + ": the pool has not been set (gsp_set_mesh_pool)").c_str());
	if (stride != p.stride || !pointers || (readyCounts != nullptr) != p.hasReady)
		return fail(c, GSP_ERR_INVALID, (std::string(who) + ": null pointer, a stride other than the staged one, or ready "
			"counts given for a pool staged without them (or the reverse)").c_str());
	return GSP_OK;
}

// The listed slots were restaged by kStagePool (dSlotMap, else first + i). Links them incrementally instead of marking the link
// dirty: the next frame then launches what a frame after no change launches. Ends in a stream synchronisation.
static int relinkMeshSlots(Context& c, uint32_t pool, const uint32_t* dSlotMap, uint32_t first, uint32_t count,
	uint32_t componentCount)
{
	auto& p = c.pools[pool];
	// a pending full link / chain pass of the next frame covers these slots (and needs the current rho, tslot)
	const bool link = !c.linkDirty, walk = link && !c.chainDirty;
	uint32_t* dGrew = c.dCounters + kCtrError + 1;
	uint32_t* hGrew = c.hCounters + kCtrCount;
	if (link)
	{
		GSP_CUDA(cudaMemsetAsync(dGrew, 0, sizeof(uint32_t), c.stream));
		launchLinkSlots(c, pool, dSlotMap, first, count, walk, dGrew);
		GSP_CUDA(cudaMemcpyAsync(hGrew, dGrew, sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	}
	GSP_CUDA(cudaStreamSynchronize(c.stream)); // the scratch buffer and the caller's memory are free again
	GSP_CUDA(cudaGetLastError());
	if (walk && *hGrew)
	{
		launchChainRecords(c);
		GSP_CUDA(cudaStreamSynchronize(c.stream));
		GSP_CUDA(cudaGetLastError());
	}
	if ((p.count == 0) != (componentCount == 0))
		c.layoutDirty = true;
	p.count = componentCount;
	p.visibleValid = false;
	c.resultsValid = false; c.frameEnqueued = false;
	return GSP_OK;
}

int gsp_update_mesh_pool(gsp_context* ctx, uint32_t pool, const void* aos, uint32_t stride, uint32_t first, uint32_t count,
	uint32_t componentCount, const uint8_t* readyCounts)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkMeshUpdate(c, pool, stride, aos || !count, readyCounts, "gsp_update_mesh_pool");
	if (rc) return rc;
	auto& p = c.pools[pool];
	if ((uint64_t)first + count > p.occupancy)
		return fail(c, GSP_ERR_INVALID, "gsp_update_mesh_pool: range past the staged occupancy (gsp_set_mesh_pool grows it)");
	if (count == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	// `aos` / `readyCounts` are the pool bases; only the range is read, each from where it lives (resolveSource)
	const size_t aosBytes = (size_t)stride * count;
	const size_t readyOffset = (aosBytes + 15) & ~(size_t)15;
	{
		// room for both sources before either is resolved (see resolveSource)
		size_t cap = c.dAosScratchCap;
		uint8_t* ptr = (uint8_t*)c.dAosScratch;
		GSP_CUDA(ensureDevice(ptr, cap, readyCounts ? readyOffset + count : aosBytes, false, c.stream));
		c.dAosScratch = ptr; c.dAosScratchCap = cap;
	}
	const void* src = nullptr;
	const void* readySrc = nullptr;
	rc = resolveSource(c, (const uint8_t*)aos + (size_t)first * stride, aosBytes, &src);
	if (rc) return rc;
	if (readyCounts)
	{
		rc = resolveSource(c, readyCounts + first, count, &readySrc, readyOffset);
		if (rc) return rc;
	}
	launchStagePool(c, pool, src, stride, first, count, nullptr, (const uint8_t*)readySrc);
	return relinkMeshSlots(c, pool, nullptr, first, count, componentCount);
}

int gsp_update_mesh_pool_indexed(gsp_context* ctx, uint32_t pool, const void* aos, uint32_t stride, const uint32_t* slots,
	uint32_t count, uint32_t componentCount, const uint8_t* readyCounts)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkMeshUpdate(c, pool, stride, (aos && slots) || !count, readyCounts, "gsp_update_mesh_pool_indexed");
	if (rc) return rc;
	if (count == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	// the library reads all three on the host while it packs them
	if (isDevicePointer(aos) || isDevicePointer(slots) || (readyCounts && isDevicePointer(readyCounts)))
		return fail(c, GSP_ERR_INVALID, "gsp_update_mesh_pool_indexed: the components, slots and ready counts must be host memory");
	auto& p = c.pools[pool];
	for (uint32_t i = 0; i < count; i++)
		if (slots[i] >= p.occupancy)
			return fail(c, GSP_ERR_INVALID, "gsp_update_mesh_pool_indexed: slot index past the staged occupancy");
	Gathered g;
	rc = uploadGathered(c, aos, stride, slots, count, readyCounts, &g);
	if (rc) return rc;
	launchStagePool(c, pool, g.aos, stride, 0, count, g.slots, g.ready);
	return relinkMeshSlots(c, pool, g.slots, 0, count, componentCount);
}

int gsp_set_pool_view_mask(gsp_context* ctx, uint32_t pool, uint32_t viewMask)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (pool >= (uint32_t)kMaxPools)
		return fail(c, GSP_ERR_INVALID, "gsp_set_pool_view_mask: bad pool index");
	auto& p = c.pools[pool];
	if (p.viewMask != viewMask)
	{
		p.viewMask = viewMask;
		c.layoutDirty = true; c.resultsValid = false; c.frameEnqueued = false;
	}
	return GSP_OK;
}

int gsp_set_views(gsp_context* ctx, uint32_t viewCount, const gsp_view* views, const float cameraPosition[3])
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (viewCount == 0 || viewCount > (uint32_t)kMaxViews || !views || !cameraPosition)
		return fail(c, GSP_ERR_INVALID, "gsp_set_views: bad view count or null pointer");
	for (uint32_t v = 0; v < viewCount; v++)
	{
		if (views[v].planeCount == 0 || views[v].planeCount > 6 || views[v].uiPlaneCount > 6)
			return fail(c, GSP_ERR_INVALID, "gsp_set_views: plane count must be 1..6 (Frustum::setPlaneCount, frustum.hpp:71-76)");
	}
	bool shapeChanged = c.views.size() != viewCount;
	for (uint32_t v = 0; v < viewCount && !shapeChanged; v++)
		shapeChanged = (c.views[v].shadowPass < 0) != (views[v].shadowPass < 0) ||
			(c.views[v].uiPlaneCount == 0) != (views[v].uiPlaneCount == 0);
	c.views.assign(views, views + viewCount);
	memcpy(c.cameraPos, cameraPosition, sizeof(c.cameraPos));
	c.viewsSet = true; c.resultsValid = false; c.frameEnqueued = false;
	if (shapeChanged)
		c.layoutDirty = true;
	return GSP_OK;
}

//----------------------------------------------------------------------------------------------------------------------
// Buffer bookkeeping of prepareMeshes (mesh.cpp:341-375,408-423,476-483) for every view, plus arena allocation.
static int rebuildLayout(Context& c)
{
	c.segments.clear();
	memset(c.segOf, -1, sizeof(c.segOf));
	memset(c.prevPool, -1, sizeof(c.prevPool));
	memset(c.participates, 0, sizeof(c.participates));
	memset(c.bufferIndexOf, 0, sizeof(c.bufferIndexOf));
	uint64_t offset = 0;
	for (uint32_t v = 0; v < (uint32_t)c.views.size(); v++)
	{
		const bool mainView = c.views[v].shadowPass < 0;
		uint32_t unsortedIndex = 0, sortedIndex = 0;
		int transSeg = -1, uiSeg = -1, lastTrans = -1, lastUi = -1;
		for (uint32_t p = 0; p < c.poolCount; p++)
		{
			auto& pool = c.pools[p];
			if (!pool.set)
			{
				c.error = "pool " + std::to_string(p) + " was declared by gsp_set_pool_count but never set";
				return GSP_ERR_STATE;
			}
			const bool active = pool.count > 0 && pool.drawReady && ((pool.viewMask >> v) & 1u) && pool.occupancy > 0; // isDrawReady(shadowPass) per view, mesh.cpp:426,482
			if (pool.renderType == GSP_RT_TRANSLUCENT || pool.renderType == GSP_RT_UI)
			{
				const bool isUI = pool.renderType == GSP_RT_UI;
				if (isUI && !mainView) // mesh.cpp:365,416-417
					continue;
				if (isUI && active && c.views[v].uiPlaneCount == 0)
				{
					c.error = "a UI mesh pool needs uiPlanes in main views (the reference dereferences uiFrustum, mesh.cpp:440)";
					return GSP_ERR_INVALID;
				}
				c.bufferIndexOf[v][p] = sortedIndex++;
				int& segIndex = isUI ? uiSeg : transSeg;
				int& last = isUI ? lastUi : lastTrans;
				if (segIndex < 0)
				{
					Segment s;
					s.view = v; s.pool = p; s.kind = isUI ? 2 : 1; s.descending = 1; s.key2D = isUI ? 1 : 0;
					s.sorted = 1; s.capacity = 0; s.lastPool = kNone;
					segIndex = (int)c.segments.size();
					c.segments.push_back(s);
				}
				c.segOf[v][p] = segIndex;
				if (active)
				{
					c.participates[v][p] = true;
					c.prevPool[v][p] = last;
					last = (int)p;
					c.segments[segIndex].capacity += pool.occupancy;
					c.segments[segIndex].lastPool = p;
				}
			}
			else
			{
				Segment s;
				s.view = v; s.pool = p; s.kind = 0; s.listIndex = (int)unsortedIndex;
				s.sorted = pool.renderType == GSP_RT_OIT ? 0 : 1; // mesh.cpp:273-277
				s.capacity = active ? pool.occupancy : 0;
				s.lastPool = active ? p : kNone;
				c.bufferIndexOf[v][p] = unsortedIndex++;
				c.segOf[v][p] = (int)c.segments.size();
				c.participates[v][p] = active;
				c.segments.push_back(s);
			}
		}
		c.unsortedCount[v] = unsortedIndex; c.sortedCount[v] = sortedIndex;
	}
	// arena offsets (16-element aligned so that 64-byte records and vector loads stay aligned)
	std::vector<SegmentDev> dev(c.segments.size());
	std::vector<uint32_t> tileOffsets(c.segments.size() + 1, 0);
	uint32_t tiles = 0;
	for (size_t i = 0; i < c.segments.size(); i++)
	{
		auto& s = c.segments[i];
		s.offset = (uint32_t)offset;
		offset += (s.capacity + 15u) & ~15u;
		if (offset > 0xFFFFFFF0ull)
		{
			c.error = "draw-list arena exceeds 2^32 elements";
			return GSP_ERR_NOMEM;
		}
		dev[i].offset = s.offset; dev[i].capacity = s.capacity;
		dev[i].countIndex = s.lastPool == kNone ? kNone : ctrPoolEnd(s.lastPool, s.view);
		dev[i].sorted = s.sorted; dev[i].descending = s.descending; dev[i].key2D = s.key2D; dev[i].pad0 = dev[i].pad1 = 0;
		tileOffsets[i] = tiles;
		tiles += (s.capacity + kSortTile - 1) / kSortTile;
	}
	tileOffsets[c.segments.size()] = tiles;
	c.arenaElems = (uint32_t)offset;
	c.sortTilesTotal = tiles;

	GSP_CUDA(cudaStreamSynchronize(c.stream));
	const size_t nseg = c.segments.size();
	if (nseg > c.dSegmentsCap || !c.dSegments)
	{
		cudaFree(c.dSegments); cudaFree(c.segTileOffset);
		c.dSegments = nullptr; c.segTileOffset = nullptr;
		size_t cap = std::max<size_t>(nseg, 8);
		GSP_CUDA(cudaMalloc((void**)&c.dSegments, cap * sizeof(SegmentDev)));
		GSP_CUDA(cudaMalloc((void**)&c.segTileOffset, (cap + 1) * sizeof(uint32_t)));
		c.dSegmentsCap = (uint32_t)cap;
	}
	if (nseg)
	{
		GSP_CUDA(cudaMemcpy(c.dSegments, dev.data(), nseg * sizeof(SegmentDev), cudaMemcpyHostToDevice));
		GSP_CUDA(cudaMemcpy(c.segTileOffset, tileOffsets.data(), (nseg + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice));
	}
	{
		// Everything that must be zero at the start of a frame lives in ONE block cleared by ONE memset per frame:
		// sort histograms and tickets of every segment, per pool the chunk counts and the survivor bucket counts.
		const size_t tBuckets = (((size_t)c.tf.capacity + kPreTile - 1) / kPreTile) / 64 + 1;
		size_t words = nseg * 4 * 256 + nseg * 4 + tBuckets;
		for (uint32_t p = 0; p < (uint32_t)kMaxPools; p++)
		{
			auto& pool = c.pools[p];
			const size_t chunksCap = ((size_t)pool.cullTilesCap + 7) / 8, preBlocks = ((size_t)pool.capacity + kPreTile - 1) / kPreTile;
			words += chunksCap * kMaxViews + preBlocks / 64 + 1;
		}
		if (words > c.frameZeroCap || !c.frameZero)
		{
			cudaFree(c.frameZero); c.frameZero = nullptr;
			GSP_CUDA(cudaMalloc((void**)&c.frameZero, words * sizeof(uint32_t)));
			c.frameZeroCap = words;
		}
		c.frameZeroWords = words;
		uint32_t* at = c.frameZero;
		c.sortHist = at; at += nseg * 4 * 256;
		c.sortTickets = at; at += nseg * 4;
		c.tf.tBucketCount = at; at += tBuckets;
		for (uint32_t p = 0; p < (uint32_t)kMaxPools; p++)
		{
			auto& pool = c.pools[p];
			const size_t chunksCap = ((size_t)pool.cullTilesCap + 7) / 8, preBlocks = ((size_t)pool.capacity + kPreTile - 1) / kPreTile;
			pool.cullStatus = at; at += chunksCap * kMaxViews;
			pool.bucketCount = at; at += preBlocks / 64 + 1;
		}
	}
	if (c.arenaElems > c.arenaCap || !c.keys[0])
	{
		for (int i = 0; i < 2; i++)
		{
			cudaFree(c.keys[i]); cudaFree(c.payloads[i]);
			c.keys[i] = nullptr; c.payloads[i] = nullptr;
		}
		cudaFree(c.records); c.records = nullptr;
		size_t cap = std::max<size_t>(c.arenaElems, 16);
		for (int i = 0; i < 2; i++)
		{
			GSP_CUDA(cudaMalloc((void**)&c.keys[i], cap * sizeof(uint32_t)));
			GSP_CUDA(cudaMalloc((void**)&c.payloads[i], cap * sizeof(uint32_t)));
		}
		GSP_CUDA(cudaMalloc((void**)&c.records, cap * sizeof(gsp_record)));
		c.arenaCap = (uint32_t)cap;
	}
	const size_t statusNeed = (size_t)tiles * 256;
	if (statusNeed > c.sortStatusCap || !c.sortStatus)
	{
		cudaFree(c.sortStatus); c.sortStatus = nullptr;
		size_t cap = std::max<size_t>(statusNeed, 1024);
		GSP_CUDA(cudaMalloc((void**)&c.sortStatus, cap * sizeof(unsigned long long)));
		GSP_CUDA(cudaMemset(c.sortStatus, 0, cap * sizeof(unsigned long long))); // epoch 0 = never published
		c.sortStatusCap = cap;
	}
	c.segDownloaded.assign(nseg, 0);
	c.layoutDirty = false;
	return GSP_OK;
}

// After linking: which pools take the split path (cull.cu)? A pool whose chains mostly find their ancestors among the pool's
// own components (every node of a hierarchy carries a mesh of that pool) is handled by the fused kernel; when more than 2 %
// of its slots have a parent without a mesh in the pool — hierarchies spread over several mesh systems, or inner nodes
// without meshes — world matrices are computed once per surviving transform instead. GSP_SPLIT=0 / 1 forces the choice.
static int decideSplit(Context& c)
{
	uint32_t* hCross = c.hCounters + kCtrCount + 2;
	GSP_CUDA(cudaMemcpyAsync(hCross, c.dCounters + kCtrCross, kMaxPools * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	static const int forced = []{ const char* e = getenv("GSP_SPLIT"); return !e ? -1 : (!strcmp(e, "0") ? 0 : 1); }();
	c.anySplit = false;
	for (uint32_t p = 0; p < c.poolCount; p++)
	{
		auto& pool = c.pools[p];
		const bool eligible = pool.set && pool.occupancy > 0 && pool.renderType != GSP_RT_UI;
		bool split = eligible && (uint64_t)hCross[p] * 50u > pool.occupancy;
		if (forced >= 0)
			split = eligible && forced == 1;
		pool.split = split;
		c.anySplit = c.anySplit || split;
	}
	auto& t = c.tf;
	if (c.anySplit && t.splitCap < t.capacity)
	{
		cudaFree(t.tBits); cudaFree(t.tBlockCount); cudaFree(t.tList); cudaFree(t.tIndex); cudaFree(t.tWorld);
		t.tBits = nullptr; t.tBlockCount = nullptr; t.tList = nullptr; t.tIndex = nullptr; t.tWorld = nullptr; t.splitCap = 0;
		const size_t cap = t.capacity, preBlocks = (cap + kPreTile - 1) / kPreTile;
		GSP_CUDA(cudaMalloc((void**)&t.tBits, preBlocks * (kPreTile / 32) * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.tBlockCount, preBlocks * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.tList, cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.tIndex, cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMemset(t.tIndex, 0xFF, cap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&t.tWorld, cap * kWorldStride * sizeof(float4)));
		t.splitCap = (uint32_t)cap;
	}
	return GSP_OK;
}

int gsp_run_async(gsp_context* ctx)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.viewsSet)
		return fail(c, GSP_ERR_STATE, "gsp_run: gsp_set_views has not been called");
	if (c.tf.cyclic)
		return fail(c, GSP_ERR_HIERARCHY, "gsp_run: the transform hierarchy is cyclic");
	GSP_CUDA(cudaSetDevice(c.device));
	c.fetchedValid = false; // the record arena and the counters are about to be rewritten
	if (c.fetchInFlight) // the previous frame's lists are still travelling out of the record arena
	{
		int rc = fetchWait(c);
		if (rc) return rc;
	}
	if (c.layoutDirty)
	{
		int rc = rebuildLayout(c);
		if (rc) return rc;
	}
	uint32_t launches = 0;
	const bool prof = c.profiling;
	if (prof && !c.phaseEventsCreated)
	{
		for (auto& e : c.phaseEvents)
			GSP_CUDA(cudaEventCreate(&e));
		for (auto& pe : c.poolEvents)
			for (auto& e : pe)
				GSP_CUDA(cudaEventCreate(&e));
		for (auto& e : c.splitEvents)
			GSP_CUDA(cudaEventCreate(&e));
		c.phaseEventsCreated = true;
	}
	if (prof) cudaEventRecord(c.phaseEvents[0], c.stream);
	if (c.linkDirty)
	{
		launches += launchLink(c);
		int rc = decideSplit(c); // (one host synchronisation per structural change)
		if (rc) return rc;
		c.linkDirty = false;
	}
	if (c.chainDirty)
	{
		launches += launchChainBounds(c); // prepass bounds of every transform (only after the transform pool changed)
		c.chainDirty = false;
	}
	if (prof) cudaEventRecord(c.phaseEvents[1], c.stream);
	GSP_CUDA(cudaMemsetAsync(c.dCounters, 0, kCtrCount * sizeof(uint32_t), c.stream));
	GSP_CUDA(cudaMemsetAsync(c.frameZero, 0, c.frameZeroWords * sizeof(uint32_t), c.stream));
	{
		const uint32_t n = launchSplitWorld(c, prof ? c.splitEvents[0] : nullptr, prof ? c.splitEvents[1] : nullptr);
		c.splitRan = n != 0;
		launches += n;
	}
	for (uint32_t p = 0; p < c.poolCount; p++)
		launches += launchCull(c, p, prof ? c.poolEvents[p][0] : nullptr, prof ? c.poolEvents[p][1] : nullptr, prof ? c.poolEvents[p][2] : nullptr);
	launches += launchSort(c, prof ? c.phaseEvents[2] : nullptr);
	if (prof) cudaEventRecord(c.phaseEvents[3], c.stream);
	launches += launchEmit(c);
	if (prof) cudaEventRecord(c.phaseEvents[4], c.stream);
	c.phaseTimesValid = prof;
	GSP_CUDA(cudaMemcpyAsync(c.hCounters, c.dCounters, kCtrCount * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaGetLastError());
	c.launchCount = launches;
	std::fill(c.segDownloaded.begin(), c.segDownloaded.end(), 0);
	c.resultsValid = false;
	c.frameEnqueued = true;
	return GSP_OK;
}

int gsp_sync(gsp_context* ctx)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	GSP_CUDA(cudaSetDevice(c.device));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	GSP_CUDA(cudaGetLastError());
	// results only exist for a frame enqueued AFTER the last change of transforms / pools / views (anything else would hand
	// out the counters and segments of an older frame, possibly of an older layout)
	if (!c.frameEnqueued || c.layoutDirty)
		return fail(c, GSP_ERR_STATE, "gsp_sync: no frame has been enqueued (gsp_run_async) since the last change");
	if (c.hCounters[kCtrError])
		return fail(c, GSP_ERR_HIERARCHY, "gsp_run: a parent chain is longer than the transform pool");
	c.resultsValid = true;
	return GSP_OK;
}

int gsp_run(gsp_context* ctx)
{
	int rc = gsp_run_async(ctx);
	return rc ? rc : gsp_sync(ctx);
}

//----------------------------------------------------------------------------------------------------------------------
static int findSegment(Context& c, uint32_t view, int kind, uint32_t listIndex)
{
	for (size_t i = 0; i < c.segments.size(); i++)
	{
		auto& s = c.segments[i];
		if (s.view == view && s.kind == kind && (kind != 0 || (uint32_t)s.listIndex == listIndex))
			return (int)i;
	}
	return -1;
}
static uint32_t segmentCount(Context& c, const Segment& s)
{
	return s.lastPool == kNone ? 0 : c.hCounters[ctrPoolEnd(s.lastPool, s.view)];
}
static uint32_t poolDrawCount(Context& c, uint32_t view, uint32_t pool)
{
	if (!c.participates[view][pool])
		return 0;
	uint32_t end = c.hCounters[ctrPoolEnd(pool, view)];
	int prev = c.prevPool[view][pool];
	return end - (prev >= 0 ? c.hCounters[ctrPoolEnd((uint32_t)prev, view)] : 0);
}
static uint32_t poolInstanceCount(Context& c, uint32_t view, uint32_t pool)
{
	if (!c.participates[view][pool])
		return 0;
	return c.pools[pool].hasReady ? c.hCounters[ctrPoolInst(pool, view)] : poolDrawCount(c, view, pool);
}

static int checkResults(Context& c, uint32_t view)
{
	// valid: a completed frame nobody has touched since — or the snapshot gsp_fetch_all_async took of one, which survives the
	// staging of the next frame's inputs (the lists of frame k travel to the host while frame k+1 is uploaded); a layout
	// change or the next gsp_run_async ends it
	if (!c.resultsValid && !(c.fetchedValid && !c.layoutDirty))
		return fail(c, GSP_ERR_STATE, "results requested before a completed gsp_run");
	if (view >= c.views.size())
		return fail(c, GSP_ERR_INVALID, "view index out of range");
	return GSP_OK;
}

static int downloadSegment(Context& c, int seg, const gsp_record** records)
{
	const Segment& s = c.segments[seg];
	if (c.hRecordsCap < c.arenaElems || !c.hRecords)
	{
		cudaFreeHost(c.hRecords); c.hRecords = nullptr; c.hRecordsCap = 0;
		GSP_CUDA(cudaMallocHost((void**)&c.hRecords, std::max<size_t>(c.arenaElems, 16) * sizeof(gsp_record)));
		c.hRecordsCap = std::max<size_t>(c.arenaElems, 16);
		std::fill(c.segDownloaded.begin(), c.segDownloaded.end(), 0);
	}
	uint32_t count = segmentCount(c, s);
	if (c.segDownloaded[seg] == 2)
	{
		int rc = fetchWait(c);
		if (rc) return rc;
	}
	if (!c.segDownloaded[seg] && count)
	{
		GSP_CUDA(cudaMemcpyAsync(c.hRecords + s.offset, c.records + s.offset, (size_t)count * sizeof(gsp_record),
			cudaMemcpyDeviceToHost, c.stream));
		GSP_CUDA(cudaStreamSynchronize(c.stream));
		c.segDownloaded[seg] = 1;
	}
	*records = c.hRecords + s.offset;
	return GSP_OK;
}

// Enqueues the download of every list that has not travelled yet on the context's COPY stream (ordered after the frame by
// an event), so the caller — and gsp_writeback_visible's host-side scatter — overlap the transfer.
static int fetchAllAsync(Context& c)
{
	if (!c.resultsValid)
		return fail(c, GSP_ERR_STATE, "results requested before a completed gsp_run");
	GSP_CUDA(cudaSetDevice(c.device));
	if (c.hRecordsCap < c.arenaElems || !c.hRecords)
	{
		GSP_CUDA(cudaStreamSynchronize(c.copyStream));
		cudaFreeHost(c.hRecords); c.hRecords = nullptr; c.hRecordsCap = 0;
		GSP_CUDA(cudaMallocHost((void**)&c.hRecords, std::max<size_t>(c.arenaElems, 16) * sizeof(gsp_record)));
		c.hRecordsCap = std::max<size_t>(c.arenaElems, 16);
		std::fill(c.segDownloaded.begin(), c.segDownloaded.end(), 0);
	}
	bool any = false;
	for (size_t seg = 0; seg < c.segments.size(); seg++)
	{
		const Segment& s = c.segments[seg];
		const uint32_t count = segmentCount(c, s);
		if (c.segDownloaded[seg] || !count)
			continue;
		if (!any)
		{
			GSP_CUDA(cudaEventRecord(c.copyEvent, c.stream));
			GSP_CUDA(cudaStreamWaitEvent(c.copyStream, c.copyEvent, 0));
			any = true;
		}
		GSP_CUDA(cudaMemcpyAsync(c.hRecords + s.offset, c.records + s.offset, (size_t)count * sizeof(gsp_record),
			cudaMemcpyDeviceToHost, c.copyStream));
		c.segDownloaded[seg] = 2; // in flight
	}
	c.fetchInFlight = c.fetchInFlight || any;
	c.fetchedValid = true;
	return GSP_OK;
}

static int fetchWait(Context& c)
{
	if (!c.fetchInFlight)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	GSP_CUDA(cudaStreamSynchronize(c.copyStream));
	for (auto& d : c.segDownloaded)
		if (d == 2) d = 1;
	c.fetchInFlight = false;
	return GSP_OK;
}

int gsp_fetch_all_async(gsp_context* ctx)
{
	return ctx ? fetchAllAsync(ctx->c) : GSP_ERR_INVALID;
}

int gsp_fetch_all(gsp_context* ctx)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	int rc = fetchAllAsync(ctx->c);
	return rc ? rc : fetchWait(ctx->c);
}

uint32_t gsp_unsorted_buffer_count(const gsp_context* ctx, uint32_t view)
{
	return (ctx && view < ctx->c.views.size() && !ctx->c.layoutDirty) ? ctx->c.unsortedCount[view] : 0;
}
uint32_t gsp_sorted_buffer_count(const gsp_context* ctx, uint32_t view)
{
	return (ctx && view < ctx->c.views.size() && !ctx->c.layoutDirty) ? ctx->c.sortedCount[view] : 0;
}

static int getUnsorted(gsp_context* ctx, uint32_t view, uint32_t buffer, const gsp_record** records,
	uint32_t* drawCount, uint32_t* instanceCount, bool device)
{
	if (!ctx || !records || !drawCount || !instanceCount)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkResults(c, view);
	if (rc) return rc;
	int seg = findSegment(c, view, 0, buffer);
	if (seg < 0)
		return fail(c, GSP_ERR_INVALID, "unsorted buffer index out of range");
	const Segment& s = c.segments[seg];
	*drawCount = segmentCount(c, s);
	*instanceCount = poolInstanceCount(c, view, s.pool);
	if (device)
	{
		*records = c.records + s.offset;
		return GSP_OK;
	}
	GSP_CUDA(cudaSetDevice(c.device));
	return downloadSegment(c, seg, records);
}

int gsp_get_unsorted(gsp_context* ctx, uint32_t view, uint32_t buffer, const gsp_record** records,
	uint32_t* drawCount, uint32_t* instanceCount)
{
	return getUnsorted(ctx, view, buffer, records, drawCount, instanceCount, false);
}
int gsp_get_unsorted_device(gsp_context* ctx, uint32_t view, uint32_t buffer, const gsp_record** records,
	uint32_t* drawCount, uint32_t* instanceCount)
{
	return getUnsorted(ctx, view, buffer, records, drawCount, instanceCount, true);
}

int gsp_get_sorted_counts(gsp_context* ctx, uint32_t view, uint32_t buffer, uint32_t* drawCount, uint32_t* instanceCount)
{
	if (!ctx || !drawCount || !instanceCount)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkResults(c, view);
	if (rc) return rc;
	for (uint32_t p = 0; p < c.poolCount; p++)
	{
		auto rt = c.pools[p].renderType;
		if ((rt == GSP_RT_TRANSLUCENT || rt == GSP_RT_UI) && c.segOf[view][p] >= 0 && c.bufferIndexOf[view][p] == buffer)
		{
			*drawCount = poolDrawCount(c, view, p);
			*instanceCount = poolInstanceCount(c, view, p);
			return GSP_OK;
		}
	}
	return fail(c, GSP_ERR_INVALID, "sorted buffer index out of range");
}

static int getSorted(gsp_context* ctx, uint32_t view, int which, const gsp_record** records, uint32_t* drawCount, bool device)
{
	if (!ctx || !records || !drawCount || (which != 0 && which != 1))
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkResults(c, view);
	if (rc) return rc;
	int seg = findSegment(c, view, which == 0 ? 1 : 2, 0);
	if (seg < 0) // no translucent / UI system in this view: empty list (transDrawIndex == 0)
	{
		*records = nullptr; *drawCount = 0;
		return GSP_OK;
	}
	const Segment& s = c.segments[seg];
	*drawCount = segmentCount(c, s);
	if (device)
	{
		*records = c.records + s.offset;
		return GSP_OK;
	}
	GSP_CUDA(cudaSetDevice(c.device));
	return downloadSegment(c, seg, records);
}
int gsp_get_sorted(gsp_context* ctx, uint32_t view, int which, const gsp_record** records, uint32_t* drawCount)
{
	return getSorted(ctx, view, which, records, drawCount, false);
}
int gsp_get_sorted_device(gsp_context* ctx, uint32_t view, int which, const gsp_record** records, uint32_t* drawCount)
{
	return getSorted(ctx, view, which, records, drawCount, true);
}

int gsp_get_sorted_run_device(gsp_context* ctx, uint32_t view, int listKind, uint32_t buffer,
	const uint32_t** keys, const uint32_t** payloads, uint32_t* count)
{
	if (!ctx || !keys || !payloads || !count || listKind < 0 || listKind > 2)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkResults(c, view);
	if (rc) return rc;
	int seg = findSegment(c, view, listKind, buffer);
	if (seg < 0)
	{
		*keys = nullptr; *payloads = nullptr; *count = 0;
		return GSP_OK;
	}
	const Segment& s = c.segments[seg];
	*keys = c.keys[0] + s.offset; *payloads = c.payloads[0] + s.offset; *count = segmentCount(c, s);
	return GSP_OK;
}

uint32_t gsp_list_count(const gsp_context* ctx)
{
	return (ctx && !ctx->c.layoutDirty) ? (uint32_t)ctx->c.segments.size() : 0;
}

int gsp_get_list_counts(gsp_context* ctx, uint32_t* counts, uint32_t capacity)
{
	if (!ctx || !counts)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.resultsValid)
		return fail(c, GSP_ERR_STATE, "results requested before a completed gsp_run");
	if (capacity < c.segments.size())
		return fail(c, GSP_ERR_INVALID, "gsp_get_list_counts: capacity too small");
	for (size_t i = 0; i < c.segments.size(); i++)
		counts[i] = segmentCount(c, c.segments[i]);
	return GSP_OK;
}

int gsp_export_runs(gsp_context* ctx, uint32_t* dKeys, uint32_t* dPayloads, uint32_t capacity)
{
	if (!ctx || !dKeys || !dPayloads)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.resultsValid)
		return fail(c, GSP_ERR_STATE, "results requested before a completed gsp_run");
	GSP_CUDA(cudaSetDevice(c.device));
	uint64_t offset = 0;
	for (auto& s : c.segments)
	{
		const uint32_t n = segmentCount(c, s);
		if (offset + n > capacity)
			return fail(c, GSP_ERR_INVALID, "gsp_export_runs: destination too small");
		if (n)
		{
			GSP_CUDA(cudaMemcpyAsync(dKeys + offset, c.keys[0] + s.offset, (size_t)n * 4, cudaMemcpyDeviceToDevice, c.stream));
			GSP_CUDA(cudaMemcpyAsync(dPayloads + offset, c.payloads[0] + s.offset, (size_t)n * 4, cudaMemcpyDeviceToDevice, c.stream));
		}
		offset += n;
	}
	return GSP_OK;
}

// ---- SURVEY.md §8f rows -------------------------------------------------------------------------------------------------
static int emitInstances(gsp_context* ctx, uint32_t view, int listKind, uint32_t buffer, const float* viewProj, void* dst,
	uint32_t stride, uint32_t mvpOffset, uint32_t capacity, bool deviceDst)
{
	if (!ctx || !viewProj || listKind < 0 || listKind > 2)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if ((!dst && capacity) || stride < 64 || (stride & 15) || (mvpOffset & 15) || (uint64_t)mvpOffset + 64 > stride)
		return fail(c, GSP_ERR_INVALID, "gsp_emit_instances: need stride >= 64, stride and mvpOffset multiples of 16, mvp inside the stride");
	if (deviceDst ? (!c.frameEnqueued || c.layoutDirty) : !c.resultsValid)
		return fail(c, GSP_ERR_STATE, "gsp_emit_instances: no frame to read (gsp_run_async for device output, completed gsp_run for host output)");
	if (view >= c.views.size())
		return fail(c, GSP_ERR_INVALID, "view index out of range");
	const int seg = findSegment(c, view, listKind, buffer);
	if (seg < 0 || capacity == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	if (deviceDst)
	{
		launchInstances(c, seg, viewProj, dst, stride, mvpOffset, capacity);
		GSP_CUDA(cudaGetLastError());
		return GSP_OK;
	}
	const uint32_t count = std::min(capacity, segmentCount(c, c.segments[seg]));
	if (count == 0)
		return GSP_OK;
	// host destination: packed 64-byte matrices on the device, then one strided copy into the caller's instance buffer
	size_t cap = c.dAosScratchCap;
	uint8_t* ptr = (uint8_t*)c.dAosScratch;
	GSP_CUDA(ensureDevice(ptr, cap, (size_t)count * 64, false, c.stream));
	c.dAosScratch = ptr; c.dAosScratchCap = cap;
	launchInstances(c, seg, viewProj, c.dAosScratch, 64, 0, count);
	GSP_CUDA(cudaMemcpy2DAsync((uint8_t*)dst + mvpOffset, stride, c.dAosScratch, 64, 64, count, cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	GSP_CUDA(cudaGetLastError());
	return GSP_OK;
}
int gsp_emit_instances(gsp_context* ctx, uint32_t view, int listKind, uint32_t buffer, const float* viewProj, void* instances,
	uint32_t stride, uint32_t mvpOffset, uint32_t capacity)
{
	return emitInstances(ctx, view, listKind, buffer, viewProj, instances, stride, mvpOffset, capacity, false);
}
int gsp_emit_instances_device(gsp_context* ctx, uint32_t view, int listKind, uint32_t buffer, const float* viewProj,
	void* dInstances, uint32_t stride, uint32_t mvpOffset, uint32_t capacity)
{
	return emitInstances(ctx, view, listKind, buffer, viewProj, dInstances, stride, mvpOffset, capacity, true);
}

// f4 (host part): Frustum(viewProj), libraries/math/include/math/frustum.hpp:51-61 — Gribb & Hartmann on the transposed
// matrix with the Vulkan Y flip; planes stay unnormalised, exactly what prepareMeshes receives (mesh.cpp:815,869,902).
void gsp_frustum_planes(const float* viewProj, float* planes)
{
	if (!viewProj || !planes)
		return;
	const volatile float* m = viewProj; // (volatile: every sum below is one separately rounded float operation)
	for (int l = 0; l < 4; l++)
	{
		// t = transpose4x4(viewProj): lane l of t.c_i = lane i of viewProj.c_l
		const float t0 = m[l * 4 + 0], t1 = m[l * 4 + 1], t2 = m[l * 4 + 2], t3 = m[l * 4 + 3];
		planes[0 * 4 + l] = t3 + t0;
		planes[1 * 4 + l] = t3 - t0;
		planes[2 * 4 + l] = t3 - t1;
		planes[3 * 4 + l] = t3 + t1;
		planes[4 * 4 + l] = t2;
		planes[5 * 4 + l] = t3 - t2;
	}
}

int gsp_view_from_viewproj(const float* viewProj, const float* cameraOffset, int32_t shadowPass, gsp_view* view)
{
	if (!viewProj || !view)
		return GSP_ERR_INVALID;
	memset(view, 0, sizeof(*view));
	gsp_frustum_planes(viewProj, &view->planes[0][0]);
	view->planeCount = 6;
	if (cameraOffset)
		memcpy(view->cameraOffset, cameraOffset, sizeof(view->cameraOffset));
	view->shadowPass = shadowPass;
	return GSP_OK;
}

int gsp_set_active(gsp_context* ctx, const uint32_t* entityIds, uint32_t count, int active)
{
	if (!ctx || (!entityIds && count))
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	auto& t = c.tf;
	if (!t.flags || !t.entityToSlot)
		return fail(c, GSP_ERR_STATE, "gsp_set_active: gsp_set_transforms has not been called");
	if (t.cyclic)
		return fail(c, GSP_ERR_HIERARCHY, "gsp_set_active: the transform hierarchy is cyclic (nothing was applied)");
	GSP_CUDA(cudaSetDevice(c.device));
	uint32_t* dIds = nullptr;
	if (count)
	{
		size_t cap = c.dAosScratchCap;
		uint8_t* ptr = (uint8_t*)c.dAosScratch;
		GSP_CUDA(ensureDevice(ptr, cap, (size_t)count * sizeof(uint32_t), false, c.stream));
		c.dAosScratch = ptr; c.dAosScratchCap = cap;
		dIds = (uint32_t*)c.dAosScratch;
		GSP_CUDA(cudaMemcpyAsync(dIds, entityIds, (size_t)count * sizeof(uint32_t), cudaMemcpyHostToDevice, c.stream));
	}
	GSP_CUDA(cudaMemsetAsync(c.dError, 0, sizeof(uint32_t), c.stream));
	launchSetActive(c, dIds, count, active);
	c.chainDirty = true; // the prepass records carry isActive()
	uint32_t* hScalars = c.hCounters + kCtrCount;
	GSP_CUDA(cudaMemcpyAsync(&hScalars[1], c.dError, sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream)); // the caller's id array is free again
	GSP_CUDA(cudaGetLastError());
	c.resultsValid = false; c.frameEnqueued = false;
	if (hScalars[1] == (uint32_t)GSP_ERR_HIERARCHY)
		return fail(c, GSP_ERR_HIERARCHY, "gsp_set_active: a parent chain is longer than the transform pool");
	if (hScalars[1])
		return fail(c, GSP_ERR_INVALID, "gsp_set_active: an entity id has no TransformComponent (the other ids were applied)");
	return GSP_OK;
}

// f2: TransformSystem::animateAsync for `count` entities, entirely on the device (next.cu: kAnimate).
int gsp_animate(gsp_context* ctx, const uint32_t* entityIds, const uint8_t* flags, const float* frameA, const float* frameB,
	const float* t, uint32_t count)
{
	if (!ctx || ((!entityIds || !flags || !frameA || !frameB || !t) && count))
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	auto& tf = c.tf;
	if (!tf.flags || !tf.entityToSlot)
		return fail(c, GSP_ERR_STATE, "gsp_animate: gsp_set_transforms has not been called");
	if (count == 0)
		return GSP_OK;
	if (tf.cyclic)
		return fail(c, GSP_ERR_HIERARCHY, "gsp_animate: the transform hierarchy is cyclic (nothing was animated)");
	GSP_CUDA(cudaSetDevice(c.device));
	// one upload: ids | t | frameA | frameB | flags
	const size_t idBytes = (size_t)count * 4, frameBytes = (size_t)count * 40, flagBytes = ((size_t)count + 15) & ~(size_t)15;
	const size_t bytes = 2 * idBytes + 2 * frameBytes + flagBytes;
	if (c.hGatherCap < bytes)
	{
		GSP_CUDA(cudaStreamSynchronize(c.stream));
		cudaFreeHost(c.hGather); c.hGather = nullptr; c.hGatherCap = 0;
		GSP_CUDA(cudaMallocHost((void**)&c.hGather, bytes + bytes / 2));
		c.hGatherCap = bytes + bytes / 2;
	}
	uint8_t* h = c.hGather;
	memcpy(h, entityIds, idBytes); memcpy(h + idBytes, t, idBytes);
	memcpy(h + 2 * idBytes, frameA, frameBytes); memcpy(h + 2 * idBytes + frameBytes, frameB, frameBytes);
	memcpy(h + 2 * idBytes + 2 * frameBytes, flags, count);
	size_t cap = c.dAosScratchCap;
	uint8_t* d = (uint8_t*)c.dAosScratch;
	GSP_CUDA(ensureDevice(d, cap, bytes, false, c.stream));
	c.dAosScratch = d; c.dAosScratchCap = cap;
	GSP_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, c.stream));
	GSP_CUDA(cudaMemsetAsync(c.dError, 0, sizeof(uint32_t), c.stream));
	launchAnimate(c, (const uint32_t*)d, d + 2 * idBytes + 2 * frameBytes, (const float*)(d + 2 * idBytes),
		(const float*)(d + 2 * idBytes + frameBytes), (const float*)(d + idBytes), count);
	uint32_t* hScalars = c.hCounters + kCtrCount;
	GSP_CUDA(cudaMemcpyAsync(&hScalars[1], c.dError, sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream)); // the caller's arrays (and the pinned staging block) are free again
	GSP_CUDA(cudaGetLastError());
	c.chainDirty = true; c.resultsValid = false; c.frameEnqueued = false;
	if (hScalars[1] == (uint32_t)GSP_ERR_HIERARCHY)
		return fail(c, GSP_ERR_HIERARCHY, "gsp_animate: a parent chain is longer than the transform pool");
	if (hScalars[1])
		return fail(c, GSP_ERR_INVALID, "gsp_animate: an entity id has no TransformComponent (the other entities were animated)");
	return GSP_OK;
}

// Stores position / scale / rotation of every live transform (bytes 16..27, 32..43, 48..63; lane W of position and scale —
// childCount / childCapacity — is left alone) into the caller's pool: what the ECS needs back after gsp_animate.
int gsp_writeback_trs(gsp_context* ctx, void* aos, uint32_t stride)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	auto& t = c.tf;
	if ((!aos && t.occupancy) || stride < kTfMinStride)
		return fail(c, GSP_ERR_INVALID, "gsp_writeback_trs: bad pointer or stride");
	if (!t.flags || t.occupancy == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	const uint32_t n = t.occupancy;
	std::vector<float4> rot(n), ps(n);
	std::vector<float2> syz(n);
	std::vector<uint16_t> flags(n);
	GSP_CUDA(cudaMemcpyAsync(rot.data(), t.rot, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaMemcpyAsync(ps.data(), t.posSx, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaMemcpyAsync(syz.data(), t.sYZ, (size_t)n * sizeof(float2), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaMemcpyAsync(flags.data(), t.flags, (size_t)n * sizeof(uint16_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	uint8_t* base = (uint8_t*)aos;
	parallelFor(n, [&](uint32_t first, uint32_t last) {
		for (uint32_t i = first; i < last; i++)
		{
			if (!(flags[i] & kTfLive))
				continue;
			uint8_t* p = base + (size_t)i * stride;
			const float pos[3] = { ps[i].x, ps[i].y, ps[i].z }, scl[3] = { ps[i].w, syz[i].x, syz[i].y };
			memcpy(p + kTfPos, pos, 12); memcpy(p + kTfScale, scl, 12); memcpy(p + kTfRot, &rot[i], 16);
		}
	});
	return GSP_OK;
}

int gsp_writeback_active(gsp_context* ctx, void* aos, uint32_t stride)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	auto& t = c.tf;
	if ((!aos && t.occupancy) || stride < kTfMinStride)
		return fail(c, GSP_ERR_INVALID, "gsp_writeback_active: bad pointer or stride");
	if (!t.flags || t.occupancy == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	std::vector<uint16_t> flags(t.occupancy);
	GSP_CUDA(cudaMemcpyAsync(flags.data(), t.flags, (size_t)t.occupancy * sizeof(uint16_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	uint8_t* base = (uint8_t*)aos;
	for (uint32_t i = 0; i < t.occupancy; i++)
	{
		if (!(flags[i] & kTfLive))
			continue; // freed slots keep their default-constructed bytes
		base[(size_t)i * stride + kTfSelfActive] = (flags[i] & kTfSelfBit) ? 1 : 0;
		base[(size_t)i * stride + kTfAncestorsActive] = (flags[i] & kTfAncBit) ? 1 : 0;
	}
	return GSP_OK;
}

int gsp_export_runs_packed(gsp_context* ctx, uint32_t* dBlock, uint32_t capacityElems)
{
	if (!ctx || !dBlock)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.frameEnqueued || c.layoutDirty)
		return fail(c, GSP_ERR_STATE, "gsp_export_runs_packed: no frame has been enqueued (gsp_run_async) since the last change");
	if (c.segments.empty() || c.segments.size() > kExMaxLists)
		return fail(c, GSP_ERR_INVALID, "gsp_export_runs_packed: the frame has no lists (or more than the block header holds)");
	GSP_CUDA(cudaSetDevice(c.device));
	launchExportPacked(c, dBlock, capacityElems);
	GSP_CUDA(cudaGetLastError());
	return GSP_OK;
}

} // extern "C"

// Runs fn(first, last) over [0, n) on the library's host workers (the write-back scatter touches every cache line of a pool).
// The workers are PERSISTENT (created on first use, parked on a condition variable between calls) and their number is
// hardware_concurrency divided by the number of GPU processes sharing the host (LOCAL_WORLD_SIZE, as torchrun / mpirun set it),
// at most 16; GSP_HOST_THREADS overrides. Eight ranks on a 32-core host thus run 4 workers each instead of 8 x 16 fresh threads.
namespace
{
class HostWorkers
{
public:
	static HostWorkers& get()
	{
		static HostWorkers pool;
		return pool;
	}
	uint32_t size() const { return (uint32_t)threads.size() + 1; } // the caller works too
	template<class F> void run(uint32_t n, F fn)
	{
		const uint32_t parts = size();
		const uint32_t per = ((n + parts - 1) / parts + 31u) & ~31u;
		std::function<void(uint32_t)> job = [&](uint32_t part)
		{
			const uint32_t first = (uint32_t)std::min<uint64_t>((uint64_t)part * per, n);
			const uint32_t last = (uint32_t)std::min<uint64_t>((uint64_t)first + per, n);
			if (first < last)
				fn(first, last);
		};
		{
			std::lock_guard<std::mutex> serial(callers); // (contexts of several caller threads share the workers)
			{
				std::lock_guard<std::mutex> lock(m);
				current = &job; pending = (uint32_t)threads.size(); generation++;
			}
			wake.notify_all();
			job(parts - 1);
			std::unique_lock<std::mutex> lock(m);
			done.wait(lock, [&]{ return pending == 0; });
			current = nullptr;
		}
	}
private:
	HostWorkers()
	{
		uint32_t n = std::max(1u, std::thread::hardware_concurrency());
		if (const char* e = getenv("LOCAL_WORLD_SIZE"))
			n = std::max(1u, n / (uint32_t)std::max(1, atoi(e)));
		n = std::min(n, 16u);
		if (const char* e = getenv("GSP_HOST_THREADS"))
			n = (uint32_t)std::max(1, std::min(64, atoi(e)));
		for (uint32_t i = 0; i + 1 < n; i++)
			threads.emplace_back([this, i]{ loop(i); });
	}
	~HostWorkers()
	{
		{
			std::lock_guard<std::mutex> lock(m);
			quit = true;
		}
		wake.notify_all();
		for (auto& t : threads) t.join();
	}
	void loop(uint32_t index)
	{
		uint64_t seen = 0;
		while (true)
		{
			std::function<void(uint32_t)>* job;
			{
				std::unique_lock<std::mutex> lock(m);
				wake.wait(lock, [&]{ return quit || generation != seen; });
				if (quit) return;
				seen = generation; job = current;
			}
			(*job)(index);
			{
				std::lock_guard<std::mutex> lock(m);
				if (--pending == 0) done.notify_one();
			}
		}
	}
	std::vector<std::thread> threads;
	std::mutex m, callers;
	std::condition_variable wake, done;
	std::function<void(uint32_t)>* current = nullptr;
	uint32_t pending = 0;
	uint64_t generation = 0;
	bool quit = false;
};
} // namespace

template<class F>
static void parallelFor(uint32_t n, F fn, uint32_t minParallel)
{
	if (n < minParallel || HostWorkers::get().size() == 1)
	{
		fn(0u, n);
		return;
	}
	HostWorkers::get().run(n, fn);
}

// Mapped pinned host words the write-back kernels store into directly (+2 trailing words: device counter mirror).
static int ensureVisibleScratch(Context& c, size_t words)
{
	if (c.visScratchCap >= words && c.hVisible)
		return GSP_OK;
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	cudaFreeHost(c.hVisible);
	c.hVisible = nullptr; c.dVisMapped = nullptr; c.visScratchCap = 0;
	GSP_CUDA(cudaHostAlloc((void**)&c.hVisible, (words + 2) * sizeof(uint32_t), cudaHostAllocMapped));
	GSP_CUDA(cudaHostGetDevicePointer((void**)&c.dVisMapped, c.hVisible, 0));
	if (!c.dVisScratch)
		GSP_CUDA(cudaMalloc((void**)&c.dVisScratch, 2 * sizeof(uint32_t)));
	c.visScratchCap = words;
	return GSP_OK;
}

static int checkWriteback(Context& c, uint32_t pool, void* aos, uint32_t stride, const char* who)
{
	if (pool >= c.poolCount || !aos || stride < kMcMinStride)
	{
		c.error = std::string(who) + ": bad pool, pointer or stride";
		return GSP_ERR_INVALID;
	}
	if (!c.resultsValid)
		return fail(c, GSP_ERR_STATE, "results requested before a completed gsp_run");
	return GSP_OK;
}

extern "C"
{

int gsp_writeback_visible(gsp_context* ctx, uint32_t pool, void* aos, uint32_t stride)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkWriteback(c, pool, aos, stride, "gsp_writeback_visible");
	if (rc) return rc;
	auto& p = c.pools[pool];
	if (!p.visibleValid || p.occupancy == 0)
		return GSP_OK; // the reference does not touch isVisible of pools the main view skipped (mesh.cpp:426,482)
	GSP_CUDA(cudaSetDevice(c.device));
	const size_t words = ((size_t)p.occupancy + 31) / 32;
	rc = ensureVisibleScratch(c, words);
	if (rc) return rc;
	launchPackVisible(c, pool, c.dVisMapped);
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	GSP_CUDA(cudaGetLastError());
	uint8_t* dst = (uint8_t*)aos + kMcVisible;
	const uint32_t* bits = c.hVisible;
	parallelFor(p.occupancy, [=](uint32_t first, uint32_t last) {
		for (uint32_t i = first; i < last; i++)
		{
			const uint8_t v = (uint8_t)((bits[i >> 5] >> (i & 31u)) & 1u);
			uint8_t* d = dst + (size_t)i * stride;
			if (*d != v) // (unchanged bytes are only read: no dirty cache lines to write back)
				*d = v;
		}
	});
	return GSP_OK;
}

int gsp_writeback_visible_delta(gsp_context* ctx, uint32_t pool, void* aos, uint32_t stride, uint32_t* changedOut)
{
	if (changedOut)
		*changedOut = 0;
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	int rc = checkWriteback(c, pool, aos, stride, "gsp_writeback_visible_delta");
	if (rc) return rc;
	auto& p = c.pools[pool];
	if (!p.visibleValid || p.occupancy == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	rc = ensureVisibleScratch(c, p.occupancy); // worst case every slot changes
	if (rc) return rc;
	uint32_t* dCount = c.dVisScratch;
	GSP_CUDA(cudaMemsetAsync(dCount, 0, sizeof(uint32_t), c.stream));
	launchVisibleDelta(c, pool, c.dVisMapped, dCount, c.dVisMapped + c.visScratchCap);
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	GSP_CUDA(cudaGetLastError());
	const uint32_t changed = c.hVisible[c.visScratchCap];
	if (changed)
	{
		uint8_t* dst = (uint8_t*)aos + kMcVisible;
		const uint32_t* list = c.hVisible;
		parallelFor(changed, [=](uint32_t first, uint32_t last) {
			for (uint32_t k = first; k < last; k++)
				dst[(size_t)(list[k] & 0x7fffffffu) * stride] = (uint8_t)(list[k] >> 31);
		});
	}
	if (changedOut)
		*changedOut = changed;
	return GSP_OK;
}

int gsp_download_models(gsp_context* ctx, uint32_t pool, float* out)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (pool >= c.poolCount || !out)
		return fail(c, GSP_ERR_INVALID, "gsp_download_models: bad pool or pointer");
	if (!c.resultsValid)
		return fail(c, GSP_ERR_STATE, "results requested before a completed gsp_run");
	auto& p = c.pools[pool];
	if (p.occupancy == 0)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	// world matrices are stored per SURVIVOR of the prepass (compact, in slot order): scatter them back to slots here
	const uint32_t survivors = c.hCounters[kCtrSurvivors + pool];
	if (survivors == 0 || !c.poolLaunched[pool])
		return GSP_OK;
	std::vector<uint32_t> list(survivors);
	std::vector<float> compact((size_t)survivors * 12);
	GSP_CUDA(cudaMemcpyAsync(list.data(), p.surList, (size_t)survivors * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaMemcpy2DAsync(compact.data(), 12 * sizeof(float), p.world, kWorldStride * sizeof(float4), 12 * sizeof(float), survivors,
		cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	for (uint32_t i = 0; i < survivors; i++)
		memcpy(out + (size_t)list[i] * 12, compact.data() + (size_t)i * 12, 12 * sizeof(float));
	return GSP_OK;
}

int gsp_set_profiling(gsp_context* ctx, int enabled)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	ctx->c.profiling = enabled != 0;
	return GSP_OK;
}

int gsp_get_phase_times(gsp_context* ctx, float* ms)
{
	if (!ctx || !ms)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	for (int i = 0; i < GSP_PHASE_COUNT; i++)
		ms[i] = 0.0f;
	if (!c.phaseTimesValid || !c.resultsValid)
		return GSP_OK;
	GSP_CUDA(cudaSetDevice(c.device));
	// link | per pool: prepass, cull, then scan + scatter | sort passes | emission
	GSP_CUDA(cudaEventElapsedTime(&ms[0], c.phaseEvents[0], c.phaseEvents[1]));
	cudaEvent_t prev = c.phaseEvents[1];
	if (c.anySplit && c.splitRan)
	{
		// split path: transform-level prepass + compaction + world matrices, booked under phase 1 (world matrices)
		float pre = 0.0f, w = 0.0f;
		GSP_CUDA(cudaEventElapsedTime(&pre, prev, c.splitEvents[0]));
		GSP_CUDA(cudaEventElapsedTime(&w, c.splitEvents[0], c.splitEvents[1]));
		ms[3] += pre; ms[1] += w;
		prev = c.splitEvents[1];
	}
	for (uint32_t p = 0; p < c.poolCount; p++)
	{
		if (!c.poolLaunched[p])
			continue;
		float pre = 0.0f, a = 0.0f, b = 0.0f;
		GSP_CUDA(cudaEventElapsedTime(&pre, prev, c.poolEvents[p][0]));
		GSP_CUDA(cudaEventElapsedTime(&a, c.poolEvents[p][0], c.poolEvents[p][1]));
		GSP_CUDA(cudaEventElapsedTime(&b, c.poolEvents[p][1], c.poolEvents[p][2]));
		ms[3] += pre; ms[1] += a; ms[2] += b;
		prev = c.poolEvents[p][2];
	}
	GSP_CUDA(cudaEventElapsedTime(&ms[4], c.phaseEvents[2], c.phaseEvents[3]));
	GSP_CUDA(cudaEventElapsedTime(&ms[5], c.phaseEvents[3], c.phaseEvents[4]));
	return GSP_OK;
}

uint32_t gsp_last_launch_count(const gsp_context* ctx) { return ctx ? ctx->c.launchCount : 0; }

uint64_t gsp_last_visible_total(gsp_context* ctx)
{
	if (!ctx || !ctx->c.resultsValid)
		return 0;
	Context& c = ctx->c;
	uint64_t total = 0;
	for (auto& s : c.segments)
		total += segmentCount(c, s);
	return total;
}

} // extern "C"
