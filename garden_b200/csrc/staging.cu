// Component staging: AoS ECS pools (as uploaded raw from the host) -> SoA mirrors in HBM.
//
// Replaces, once per structural change instead of per entity per view, the reference's
//   Manager::tryGet<TransformComponent>(entity)  (libraries/ecsm/include/ecsm.hpp:898-905, Entity::findComponent :274-278)
// with a device-resident entity -> transform-slot map, and the AoS field reads of
//   TransformComponent  (include/garden/system/transform.hpp:31-60)   and
//   MeshRenderComponent (include/garden/system/render/mesh.hpp:45-55).
#include "sceneprep_internal.h"
#include "sceneprep_math.cuh"
#include <algorithm>

namespace gsp
{

static inline uint32_t blocksFor(uint32_t n, uint32_t per) { return (n + per - 1) / per; }

__device__ __forceinline__ uint32_t ldU32(const uint8_t* p) { return *reinterpret_cast<const uint32_t*>(p); }
__device__ __forceinline__ float ldF32(const uint8_t* p) { return *reinterpret_cast<const float*>(p); }

// ---- tile loader ------------------------------------------------------------------------------------------------------------
// A block pulls `tileSlots` consecutive AoS slots (tileSlots * stride bytes, a multiple of 16) into shared memory with
// coalesced 128-bit loads, many in flight per thread, and the fields are picked out of shared memory afterwards. The source
// may be device memory (the upload scratch), or PINNED HOST memory read directly over PCIe ("zero copy": no intermediate
// device buffer, the re-layout overlaps the transfer). Sources that are not 16-byte aligned use 32-bit loads.
constexpr uint32_t kStageThreads = 256;

__device__ __forceinline__ uint4 ldStream128(const uint4* p)
{
	uint4 v;
	asm volatile("ld.global.cs.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
	return v;
}

__device__ __forceinline__ void loadTile(uint8_t* sTile, const uint8_t* __restrict__ src, uint32_t bytes)
{
	if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0)
	{
		const uint4* s4 = reinterpret_cast<const uint4*>(src);
		uint4* d4 = reinterpret_cast<uint4*>(sTile);
		const uint32_t n = bytes >> 4; // (bytes is a multiple of 4; the tail below handles the rest)
		constexpr uint32_t kBatch = 5;
		for (uint32_t i0 = threadIdx.x; i0 < n; i0 += kStageThreads * kBatch)
		{
			uint4 v[kBatch];
			#pragma unroll
			for (uint32_t b = 0; b < kBatch; b++)
				if (i0 + b * kStageThreads < n)
					v[b] = ldStream128(s4 + i0 + b * kStageThreads);
			#pragma unroll
			for (uint32_t b = 0; b < kBatch; b++)
				if (i0 + b * kStageThreads < n)
					d4[i0 + b * kStageThreads] = v[b];
		}
		for (uint32_t i = (n << 2) + threadIdx.x; i < (bytes >> 2); i += kStageThreads)
			reinterpret_cast<uint32_t*>(sTile)[i] = reinterpret_cast<const uint32_t*>(src)[i];
	}
	else
	{
		const uint32_t* s1 = reinterpret_cast<const uint32_t*>(src);
		uint32_t* d1 = reinterpret_cast<uint32_t*>(sTile);
		for (uint32_t i = threadIdx.x; i < (bytes >> 2); i += kStageThreads)
			d1[i] = s1[i];
	}
	__syncthreads();
}

// One block per tile of transform slots. `full` also (re)builds the hierarchy inputs (entity, parent entity, the largest
// entity id); the entity -> slot map is built from the SoA copy afterwards (kBuildEntityMap), once its size is known.
__global__ void __launch_bounds__(kStageThreads) kStageTransforms(const uint8_t* __restrict__ aos, uint32_t stride,
	uint32_t first, uint32_t count, int full, uint32_t tileSlots, float4* __restrict__ rot, float4* __restrict__ posSx,
	float2* __restrict__ sYZ, uint16_t* __restrict__ flags, float2* __restrict__ bound, uint32_t* __restrict__ entity,
	uint32_t* __restrict__ parentEntity, uint32_t* __restrict__ maxEntity, const uint32_t* __restrict__ slotMap)
{
	extern __shared__ __align__(16) uint8_t sTile[];
	const uint32_t tileFirst = blockIdx.x * tileSlots;
	const uint32_t n = min(tileSlots, count - tileFirst);
	loadTile(sTile, aos + (size_t)tileFirst * stride, n * stride);
	uint32_t emax = 0;
	for (uint32_t j = threadIdx.x; j < n; j += kStageThreads)
	{
		// slotMap: the j-th staged component belongs to slot slotMap[j] (scattered dirty set), else to first + j (a range)
		const uint32_t slot = slotMap ? slotMap[tileFirst + j] : first + tileFirst + j;
		const uint8_t* t = sTile + (size_t)j * stride;
		const uint32_t e = ldU32(t + kTfEntity);
		const float4 q = make_float4(ldF32(t + kTfRot), ldF32(t + kTfRot + 4), ldF32(t + kTfRot + 8), ldF32(t + kTfRot + 12));
		const float4 ps = make_float4(ldF32(t + kTfPos), ldF32(t + kTfPos + 4), ldF32(t + kTfPos + 8), ldF32(t + kTfScale));
		const float2 syz = make_float2(ldF32(t + kTfScale + 4), ldF32(t + kTfScale + 8));
		rot[slot] = q; posSx[slot] = ps; sYZ[slot] = syz;
		const uint32_t w = ldU32(t + kTfSelfActive); // bytes 72..75: selfActive, ancestorsActive, modelWithAncestors, pad
		uint16_t f = 0;
		Mat43 unused;
		if (!localModel43Fast<true>(ps.x, ps.y, ps.z, q.x, q.y, q.z, q.w, ps.w, syz.x, syz.y, unused))
			f |= kTfExactLocal; // the per-frame kernel must use the guarded 4-lane code for this transform
		bound[slot] = transformBound(ps.x, ps.y, ps.z, ps.w, syz.x, syz.y, q.x, q.y, q.z, q.w);
		if (e) f |= kTfLive;
		if (w & 0xffu) f |= kTfSelfBit;
		if (w & 0xff00u) f |= kTfAncBit;
		if ((w & 0xffu) && (w & 0xff00u)) f |= kTfActive;   // isActive(), transform.hpp:110
		if (w & 0xff0000u) f |= kTfAncestors;                // modelWithAncestors, transform.hpp:60,200
		// the upper byte holds the chain length (kComputeDepth); a TRS-only update keeps it
		flags[slot] = full ? f : (uint16_t)(f | (flags[slot] & ~((1u << kTfDepthShift) - 1u)));
		if (full)
		{
			entity[slot] = e;
			parentEntity[slot] = e ? ldU32(t + kTfParent) : 0;
			emax = max(emax, e);
		}
	}
	if (full)
	{
		emax = __reduce_max_sync(0xffffffffu, emax);
		if ((threadIdx.x & 31) == 0 && emax)
			atomicMax(maxEntity, emax);
	}
}

// entity id -> transform slot + 1 (0 = the entity has no TransformComponent)
__global__ void __launch_bounds__(256) kBuildEntityMap(uint32_t count, const uint32_t* __restrict__ entity,
	uint32_t* __restrict__ entityToSlot)
{
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	const uint32_t e = entity[i];
	if (e)
		entityToSlot[e] = i + 1;
}

// parent entity id -> parent transform slot. A live parent id without a TransformComponent is an error
// (the reference's Manager::get throws, ecsm.hpp:863-873).
__global__ void __launch_bounds__(256) kResolveParents(uint32_t count, const uint32_t* __restrict__ parentEntity,
	const uint32_t* __restrict__ entityToSlot, uint32_t entityCap, uint32_t* __restrict__ parent, uint32_t* __restrict__ error)
{
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	uint32_t pe = parentEntity[i];
	uint32_t p = kNone;
	if (pe)
	{
		uint32_t s = pe < entityCap ? entityToSlot[pe] : 0;
		if (s) p = s - 1;
		else atomicExch(error, (uint32_t)GSP_ERR_HIERARCHY);
	}
	parent[i] = p;
}

// Chain length of every transform (number of ancestors, saturating at 255) into the upper flag byte. The cull kernel uses
// it as the trip count of its chain loop and to group work of equal chain length into the same warp; a wrong value only
// costs time (the links decide), never correctness. *deep = 1 when some walk saturates: only then can a chain be cyclic.
__global__ void __launch_bounds__(256) kComputeDepth(uint32_t count, const uint32_t* __restrict__ parent, uint16_t* __restrict__ flags,
	uint32_t* __restrict__ deep)
{
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	uint32_t depth = 0;
	uint32_t p = parent[i];
	while (p != kNone && depth < kTfDepthMax)
	{
		depth++;
		p = parent[p];
	}
	if (depth == kTfDepthMax)
		*deep = 1;
	flags[i] = (uint16_t)((flags[i] & ((1u << kTfDepthShift) - 1u)) | (depth << kTfDepthShift));
}

// Cycle detection by pointer jumping. up[i] starts as the parent link; every round replaces it by the link of the slot it
// points at, so after r rounds it points at least 2^r steps up the chain, or is kNone past the root. A round may read a link
// that another thread of the same round has already advanced: that only moves further up the same chain. An acyclic chain has
// at most count - 1 links, so after ceil(log2(count)) rounds every link still set lies on a cycle or leads into one.
__global__ void __launch_bounds__(256) kJumpParents(uint32_t count, uint32_t* up, uint32_t* __restrict__ cyclic)
{
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	uint32_t p = up[i];
	if (p == kNone)
		return;
	p = up[p];
	up[i] = p;
	if (cyclic && p != kNone)
		*cyclic = 1;
}

// One block per tile of mesh-component slots: AABB, owner entity, the static part of the filter at mesh.cpp:140-147, and the
// isVisible byte the host currently holds (for the changed-slots-only write-back). `readySrc` (nullable): the ready counts of
// the staged components, in the same order.
__global__ void __launch_bounds__(kStageThreads) kStagePool(const uint8_t* __restrict__ aos, uint32_t stride, uint32_t first,
	uint32_t count, uint32_t tileSlots, const uint32_t* __restrict__ slotMap, const uint8_t* __restrict__ readySrc,
	float4* __restrict__ aabbA, float2* __restrict__ aabbB, uint32_t* __restrict__ entity, uint8_t* __restrict__ flags,
	float* __restrict__ radius, uint8_t* __restrict__ ready)
{
	extern __shared__ __align__(16) uint8_t sTile[];
	const uint32_t tileFirst = blockIdx.x * tileSlots;
	const uint32_t n = min(tileSlots, count - tileFirst);
	loadTile(sTile, aos + (size_t)tileFirst * stride, n * stride);
	for (uint32_t j = threadIdx.x; j < n; j += kStageThreads)
	{
		// slotMap: the j-th staged component belongs to slot slotMap[j] (scattered dirty set), else to first + j (a range)
		const uint32_t i = slotMap ? slotMap[tileFirst + j] : first + tileFirst + j;
		const uint8_t* m = sTile + (size_t)j * stride;
		uint32_t e = ldU32(m + kMcEntity);
		uint32_t w = ldU32(m + 12); // bytes 12..15: reserved2 (u16), isEnabled, isVisible
		float mnx = ldF32(m + kMcAabbMin), mny = ldF32(m + kMcAabbMin + 4), mnz = ldF32(m + kMcAabbMin + 8);
		float mxx = ldF32(m + kMcAabbMax), mxy = ldF32(m + kMcAabbMax + 4), mxz = ldF32(m + kMcAabbMax + 8);
		aabbA[i] = make_float4(mnx, mny, mnz, mxx);
		aabbB[i] = make_float2(mxy, mxz);
		radius[i] = aabbRadiusBound(mnx, mny, mnz, mxx, mxy, mxz);
		entity[i] = e;
		// aabb.getSize() = max - min, fixW(), areAllTrue(size <= 0)  (mesh.cpp:140-142, aabb.hpp:142)
		bool degenerate = (__fsub_rn(mxx, mnx) <= 0.0f) && (__fsub_rn(mxy, mny) <= 0.0f) && (__fsub_rn(mxz, mnz) <= 0.0f);
		bool enabled = (w & 0xff0000u) != 0;
		uint8_t f = (e && enabled && !degenerate) ? kMfCandidate : 0;
		const uint32_t hostVisible = w >> 24;
		if (hostVisible == 1) f |= kMfHostVisible;          // the host byte is a clean `true`
		else if (hostVisible != 0) f |= kMfHostVisibleOdd;  // neither 0 nor 1: always rewritten
		flags[i] = f;
		if (readySrc)
			ready[i] = readySrc[tileFirst + j];
	}
}

// Also folds the slot's box radius into its transform's `rho` (largest radius of any mesh on the transform, over all pools):
// radii are >= +0 or NaN, whose bit patterns order like unsigned integers with NaN on top, so atomicMax on the bits works and
// a NaN box keeps its transform from ever being culled by the prepass.
__global__ void __launch_bounds__(256) kLinkPool(uint32_t count, const uint32_t* __restrict__ entity,
	const uint32_t* __restrict__ entityToSlot, uint32_t entityCap, uint32_t* __restrict__ tslot,
	const float* __restrict__ radius, uint32_t* __restrict__ tRho, uint32_t* __restrict__ tPoolMask, uint32_t poolBit)
{
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	uint32_t e = entity[i];
	uint32_t s = (e && e < entityCap) ? entityToSlot[e] : 0;
	tslot[i] = s ? s - 1 : kNone;
	if (s)
	{
		atomicMax(&tRho[s - 1], __float_as_uint(radius[i]));
		atomicOr(&tPoolMask[s - 1], poolBit);
	}
}

// How many slots of the pool walk a chain whose first ancestor carries no mesh of the SAME pool: such chains cannot be found
// among the pool's own survivors, and when they are common the pool takes the split path (world matrices per transform).
__global__ void __launch_bounds__(256) kPoolLocality(uint32_t count, const uint32_t* __restrict__ tslot,
	const uint32_t* __restrict__ tParent, const uint16_t* __restrict__ tFlags, const uint32_t* __restrict__ tPoolMask,
	uint32_t poolBit, uint32_t* __restrict__ cross)
{
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	bool outside = false;
	if (i < count)
	{
		const uint32_t ts = tslot[i];
		if (ts != kNone)
		{
			const uint16_t f = tFlags[ts];
			const uint32_t p = tParent[ts];
			outside = (f & kTfLive) && (f & kTfAncestors) && p != kNone && !(tPoolMask[p] & poolBit);
		}
	}
	const uint32_t n = __popc(__ballot_sync(0xffffffffu, outside));
	if ((threadIdx.x & 31) == 0 && n)
		atomicAdd(cross, n);
}

// Slots per tile: a multiple of 4 (tile bytes stay a multiple of 16) that fits the shared-memory budget.
static uint32_t tileSlotsFor(uint32_t stride, size_t& smemBytes)
{
	const size_t budget = 60 * 1024;
	uint32_t slots = (uint32_t)std::min<size_t>(kStageThreads, budget / stride) & ~3u;
	if (slots == 0) slots = 1; // (stride > 15 KB: one slot per tile, still correct)
	smemBytes = (size_t)slots * stride;
	return slots;
}

uint32_t launchStageTransforms(Context& c, const void* dAos, uint32_t stride, uint32_t first, uint32_t count, bool full,
	uint32_t* dMaxEntity, const uint32_t* dSlotMap)
{
	if (count == 0)
		return 0;
	auto& t = c.tf;
	size_t smem;
	const uint32_t tileSlots = tileSlotsFor(stride, smem);
	cudaFuncSetAttribute(kStageTransforms, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	kStageTransforms<<<blocksFor(count, tileSlots), kStageThreads, smem, c.stream>>>((const uint8_t*)dAos, stride, first, count,
		full ? 1 : 0, tileSlots, t.rot, t.posSx, t.sYZ, t.flags, t.bound, t.entity, t.parentEntity, dMaxEntity, dSlotMap);
	return 1;
}

// After a full staging pass: entity map, parent slots, chain lengths (all from the SoA copy in HBM). *dDeep (zeroed by the
// caller) is set when some chain is 255 links or longer.
uint32_t launchBuildHierarchy(Context& c, uint32_t* dDeep)
{
	auto& t = c.tf;
	const uint32_t count = t.occupancy;
	if (count == 0)
		return 0;
	kBuildEntityMap<<<blocksFor(count, 256), 256, 0, c.stream>>>(count, t.entity, t.entityToSlot);
	kResolveParents<<<blocksFor(count, 256), 256, 0, c.stream>>>(count, t.parentEntity, t.entityToSlot, t.entityCap,
		t.parent, c.dError);
	kComputeDepth<<<blocksFor(count, 256), 256, 0, c.stream>>>(count, t.parent, t.flags, dDeep);
	return 3;
}

// *dCyclic (zeroed by the caller) = 1 iff some parent chain is cyclic. Only run when launchBuildHierarchy found a deep chain.
// The jump links live in chainRoot, which gsp_set_transforms marks stale (kChainBounds rewrites it before it is read).
uint32_t launchFindCycles(Context& c, uint32_t* dCyclic)
{
	auto& t = c.tf;
	const uint32_t count = t.occupancy;
	if (count == 0)
		return 0;
	uint32_t rounds = 1;
	while ((1ull << rounds) < count)
		rounds++;
	cudaMemcpyAsync(t.chainRoot, t.parent, (size_t)count * sizeof(uint32_t), cudaMemcpyDeviceToDevice, c.stream);
	for (uint32_t r = 0; r < rounds; r++)
		kJumpParents<<<blocksFor(count, 256), 256, 0, c.stream>>>(count, t.chainRoot, r + 1 == rounds ? dCyclic : nullptr);
	return rounds;
}

uint32_t launchStagePool(Context& c, uint32_t pool, const void* dAos, uint32_t stride, uint32_t first, uint32_t count,
	const uint32_t* dSlotMap, const uint8_t* dReady)
{
	if (count == 0)
		return 0;
	auto& p = c.pools[pool];
	size_t smem;
	const uint32_t tileSlots = tileSlotsFor(stride, smem);
	cudaFuncSetAttribute(kStagePool, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	kStagePool<<<blocksFor(count, tileSlots), kStageThreads, smem, c.stream>>>((const uint8_t*)dAos, stride, first, count,
		tileSlots, dSlotMap, dReady, p.aabbA, p.aabbB, p.entity, p.flags, p.radius, p.ready);
	return 1;
}

uint32_t launchLink(Context& c)
{
	uint32_t n = 0;
	if (c.tf.occupancy)
	{
		cudaMemsetAsync(c.tf.rho, 0, (size_t)c.tf.occupancy * sizeof(uint32_t), c.stream);
		cudaMemsetAsync(c.tf.poolMask, 0, (size_t)c.tf.occupancy * sizeof(uint32_t), c.stream);
	}
	cudaMemsetAsync(c.dCounters + kCtrCross, 0, kMaxPools * sizeof(uint32_t), c.stream);
	for (uint32_t i = 0; i < c.poolCount; i++)
	{
		auto& p = c.pools[i];
		if (!p.set || p.occupancy == 0)
			continue;
		kLinkPool<<<blocksFor(p.occupancy, 256), 256, 0, c.stream>>>(p.occupancy, p.entity, c.tf.entityToSlot,
			c.tf.entityCap, p.tslot, p.radius, c.tf.rho, c.tf.poolMask, 1u << i);
		n++;
	}
	for (uint32_t i = 0; i < c.poolCount; i++)
	{
		auto& p = c.pools[i];
		if (!p.set || p.occupancy == 0)
			continue;
		kPoolLocality<<<blocksFor(p.occupancy, 256), 256, 0, c.stream>>>(p.occupancy, p.tslot, c.tf.parent, c.tf.flags,
			c.tf.poolMask, 1u << i, c.dCounters + kCtrCross + i);
		n++;
	}
	return n;
}

} // namespace gsp
