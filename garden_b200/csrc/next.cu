// The callers either side of the hot path (SURVEY.md §8f), to the same bit-exact bar:
//   f1  instance data of a draw list: mvp = (float4x4)(viewProj * f32x4x4(bakedModel, (0,0,0,1))) per record, in draw order
//       — what renderUnsorted / renderSorted hand to IMeshRenderSystem::drawAsync and what every setInstanceData stores
//       first (source/system/render/mesh.cpp:600-603,632-635; source/system/render/sprite.cpp:122-130);
//   f3  TransformComponent::setActive (source/system/transform.cpp:75-127) on the staged hierarchy: selfActive flips for a
//       set of entities, ancestorsActive re-derived for every transform by walking its parent links.
#include "sceneprep_internal.h"
#include "sceneprep_math.cuh"
#include <algorithm>

namespace gsp
{

// ---- f1 ----------------------------------------------------------------------------------------------------------------
// Four lanes per record: lane q produces column q of the product (16 bytes), so a warp stores 8 x 64 contiguous bytes when
// the instance stride is 64. f32x4x4::operator* (simd/matrix/float.hpp:197-204): r = VP.c0 * b.x; r = fma(VP.c1, b.y, r);
// r = fma(VP.c2, b.z, r); r = fma(VP.c3, b.w, r) with b = column q of the model, whose lane W is 0, 0, 0, 1.
struct InstanceArgs
{
	const gsp_record* __restrict__ records;
	const uint32_t* __restrict__ counters; // draw count = counters[countIndex] (read on the device: no host sync needed)
	uint8_t* __restrict__ dst;
	float vp[16];
	uint32_t countIndex, capacity, stride, offset;
};

__global__ void __launch_bounds__(256) kInstances(const __grid_constant__ InstanceArgs A)
{
	const uint32_t count = min(A.countIndex == kNone ? 0u : A.counters[A.countIndex], A.capacity);
	const uint32_t q = threadIdx.x & 3;
	const float bw = q == 3 ? 1.0f : 0.0f;
	for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 2; i < count; i += (gridDim.x * blockDim.x) >> 2)
	{
		const float* m = reinterpret_cast<const float*>(A.records + i) + 2 + q * 3; // bakedModel starts at byte 8
		const float bx = m[0], by = m[1], bz = m[2];
		float4 r;
		r.x = __fmul_rn(A.vp[0], bx); r.y = __fmul_rn(A.vp[1], bx); r.z = __fmul_rn(A.vp[2], bx); r.w = __fmul_rn(A.vp[3], bx);
		r.x = __fmaf_rn(A.vp[4], by, r.x); r.y = __fmaf_rn(A.vp[5], by, r.y); r.z = __fmaf_rn(A.vp[6], by, r.z); r.w = __fmaf_rn(A.vp[7], by, r.w);
		r.x = __fmaf_rn(A.vp[8], bz, r.x); r.y = __fmaf_rn(A.vp[9], bz, r.y); r.z = __fmaf_rn(A.vp[10], bz, r.z); r.w = __fmaf_rn(A.vp[11], bz, r.w);
		r.x = __fmaf_rn(A.vp[12], bw, r.x); r.y = __fmaf_rn(A.vp[13], bw, r.y); r.z = __fmaf_rn(A.vp[14], bw, r.z); r.w = __fmaf_rn(A.vp[15], bw, r.w);
		*reinterpret_cast<float4*>(A.dst + (size_t)i * A.stride + A.offset + q * 16) = r;
	}
}

uint32_t launchInstances(Context& c, int seg, const float* viewProj, void* dDst, uint32_t stride, uint32_t offset,
	uint32_t capacity)
{
	const Segment& s = c.segments[seg];
	InstanceArgs A;
	A.records = c.records + s.offset; A.counters = c.dCounters;
	A.countIndex = s.lastPool == kNone ? kNone : ctrPoolEnd(s.lastPool, s.view);
	A.dst = (uint8_t*)dDst; A.capacity = std::min(capacity, s.capacity); A.stride = stride; A.offset = offset;
	for (int i = 0; i < 16; i++) A.vp[i] = viewProj[i];
	const uint32_t groups = (A.capacity + 63) / 64;
	if (groups == 0)
		return 0;
	kInstances<<<std::min<uint32_t>(groups, c.smCount * 8u), 256, 0, c.stream>>>(A);
	return 1;
}

// ---- f3 ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kSetSelfActive(const uint32_t* __restrict__ ids, uint32_t count, int active,
	const uint32_t* __restrict__ entityToSlot, uint32_t entityCap, uint16_t* __restrict__ flags, uint32_t* __restrict__ error)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	const uint32_t e = ids[i];
	const uint32_t s = (e && e < entityCap) ? entityToSlot[e] : 0;
	if (!s)
	{
		atomicExch(error, (uint32_t)GSP_ERR_INVALID); // Manager::get<TransformComponent> would throw (ecsm.hpp:863-873)
		return;
	}
	// the same entity may be listed twice (same value): 16-bit flag words share a 32-bit word with their neighbour, so use
	// an atomic on the containing word
	uint32_t* word = reinterpret_cast<uint32_t*>(flags) + ((s - 1) >> 1);
	const uint32_t bit = (uint32_t)kTfSelfBit << (((s - 1) & 1) * 16);
	if (active) atomicOr(word, bit); else atomicAnd(word, ~bit);
}

// ancestorsActive(x) = AND of selfActive over the strict ancestors of x — the invariant every TransformComponent::setActive
// call maintains (deactivation clears it in the whole subtree, transform.cpp:109-125; activation sets it along paths of
// self-active nodes, :85-107). isActive() = selfActive && ancestorsActive (transform.hpp:110) is what the cull filter reads.
__global__ void __launch_bounds__(256) kPropagateActive(uint32_t count, const uint32_t* __restrict__ parent,
	uint16_t* __restrict__ flags, uint32_t* __restrict__ error)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	const uint16_t f = flags[i];
	if (!(f & kTfLive))
		return;
	bool anc = true;
	uint32_t p = parent[i], depth = 0;
	while (p != kNone && anc)
	{
		if (++depth > count) // (cannot happen: cyclic hierarchies are refused before launch)
		{
			atomicExch(error, (uint32_t)GSP_ERR_HIERARCHY);
			break;
		}
		anc = (flags[p] & kTfSelfBit) != 0; // (only the self bit of other slots is read, and nobody writes it here)
		p = parent[p];
	}
	uint16_t g = (uint16_t)(f & ~(kTfAncBit | kTfActive));
	if (anc) g |= kTfAncBit;
	if (anc && (f & kTfSelfBit)) g |= kTfActive;
	if (g != f)
	{
		// neighbours share the 32-bit word: update only my half, atomically
		uint32_t* word = reinterpret_cast<uint32_t*>(flags) + (i >> 1);
		const uint32_t shift = (i & 1) * 16;
		const uint32_t changed = (uint32_t)(g ^ f) << shift;
		atomicXor(word, changed);
	}
}

// ---- f2: TransformSystem::animateAsync (source/system/transform.cpp:609-623) on the staged transforms ----------------------------
// lerp(f32x4 a, f32x4 b, float t) = a * (1 - t) + b * t (simd/vector/float.hpp:1469: two lane-wise products and a sum, no FMA):
// position and scale are bit-exact. slerp (quaternion.hpp:175-193): dot4, shortest path, lerp when cosTheta > 1 - FLT_EPSILON,
// else (a * sin((1 - t) * angle) + c * sin(t * angle)) / sin(angle) — the reference calls the HOST libm (acosf / sinf), the
// device has its own (<= 2 ulp each), so the rotation carries a stated tolerance (tests/test_gpu_next.py). isActive goes through
// the self bit + kPropagateActive like gsp_set_active. The per-transform data derived from TRS (exact-local flag, prepass
// bound) is refreshed here; the chain records are marked stale by the caller.
struct AnimateArgs
{
	const uint32_t* __restrict__ ids;
	const uint8_t* __restrict__ flags;
	const float* __restrict__ frameA;
	const float* __restrict__ frameB;
	const float* __restrict__ t;
	const uint32_t* __restrict__ entityToSlot;
	float4* __restrict__ rot;
	float4* __restrict__ posSx;
	float2* __restrict__ sYZ;
	uint16_t* __restrict__ tflags;
	float2* __restrict__ bound;
	uint32_t* __restrict__ error;
	uint32_t count, entityCap;
};
__global__ void __launch_bounds__(256) kAnimate(const __grid_constant__ AnimateArgs A)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= A.count)
		return;
	const uint32_t e = A.ids[i];
	const uint32_t s1 = (e && e < A.entityCap) ? A.entityToSlot[e] : 0;
	if (!s1)
	{
		atomicExch(A.error, (uint32_t)GSP_ERR_INVALID); // Manager::get<TransformComponent> would throw (ecsm.hpp:863-873)
		return;
	}
	const uint32_t s = s1 - 1;
	const uint32_t f = A.flags[i];
	const float* a = A.frameA + (size_t)i * 10;
	const float* b = A.frameB + (size_t)i * 10;
	const float t = A.t[i], u = __fsub_rn(1.0f, t);
	float4 ps = A.posSx[s];
	float2 syz = A.sYZ[s];
	float4 q = A.rot[s];
	if (f & 1u) // animatePosition
	{
		ps.x = __fadd_rn(__fmul_rn(a[0], u), __fmul_rn(b[0], t));
		ps.y = __fadd_rn(__fmul_rn(a[1], u), __fmul_rn(b[1], t));
		ps.z = __fadd_rn(__fmul_rn(a[2], u), __fmul_rn(b[2], t));
	}
	if (f & 2u) // animateScale
	{
		ps.w = __fadd_rn(__fmul_rn(a[3], u), __fmul_rn(b[3], t));
		syz.x = __fadd_rn(__fmul_rn(a[4], u), __fmul_rn(b[4], t));
		syz.y = __fadd_rn(__fmul_rn(a[5], u), __fmul_rn(b[5], t));
	}
	if (f & 4u) // animateRotation
	{
		const float* qa = a + 6;
		float c[4] = { b[6], b[7], b[8], b[9] };
		float cosTheta = __fadd_rn(__fadd_rn(__fmul_rn(qa[0], c[0]), __fmul_rn(qa[1], c[1])), __fadd_rn(__fmul_rn(qa[2], c[2]), __fmul_rn(qa[3], c[3])));
		if (cosTheta < 0.0f)
		{
			#pragma unroll
			for (int l = 0; l < 4; l++) c[l] = -c[l];
			cosTheta = -cosTheta;
		}
		float v[4];
		if (cosTheta > 1.0f - 1.1920928955078125e-07f)
		{
			#pragma unroll
			for (int l = 0; l < 4; l++) v[l] = __fadd_rn(__fmul_rn(qa[l], u), __fmul_rn(c[l], t));
		}
		else
		{
			const float angle = acosf(cosTheta);
			const float w0 = sinf(__fmul_rn(u, angle)), w1 = sinf(__fmul_rn(t, angle)), w2 = sinf(angle);
			#pragma unroll
			for (int l = 0; l < 4; l++) v[l] = __fdiv_rn(__fadd_rn(__fmul_rn(qa[l], w0), __fmul_rn(c[l], w1)), w2);
		}
		q = make_float4(v[0], v[1], v[2], v[3]);
	}
	if (f & 7u)
	{
		A.posSx[s] = ps; A.sYZ[s] = syz; A.rot[s] = q;
		Mat43 unused;
		const bool exact = !localModel43Fast<true>(ps.x, ps.y, ps.z, q.x, q.y, q.z, q.w, ps.w, syz.x, syz.y, unused);
		A.bound[s] = transformBound(ps.x, ps.y, ps.z, ps.w, syz.x, syz.y, q.x, q.y, q.z, q.w);
		uint32_t* word = reinterpret_cast<uint32_t*>(A.tflags) + (s >> 1);
		const uint32_t bit = (uint32_t)kTfExactLocal << ((s & 1) * 16);
		if (exact) atomicOr(word, bit); else atomicAnd(word, ~bit);
	}
	if (f & 8u) // animateIsActive: setActive(round(t) ? b.isActive : a.isActive), transform.cpp:620-621
	{
		const bool active = roundf(t) != 0.0f ? ((f >> 5) & 1u) : ((f >> 4) & 1u);
		uint32_t* word = reinterpret_cast<uint32_t*>(A.tflags) + (s >> 1);
		const uint32_t bit = (uint32_t)kTfSelfBit << ((s & 1) * 16);
		if (active) atomicOr(word, bit); else atomicAnd(word, ~bit);
	}
}

uint32_t launchAnimate(Context& c, const uint32_t* dIds, const uint8_t* dFlags, const float* dA, const float* dB, const float* dT,
	uint32_t count)
{
	auto& t = c.tf;
	if (!count)
		return 0;
	AnimateArgs A;
	A.ids = dIds; A.flags = dFlags; A.frameA = dA; A.frameB = dB; A.t = dT; A.entityToSlot = t.entityToSlot;
	A.rot = t.rot; A.posSx = t.posSx; A.sYZ = t.sYZ; A.tflags = t.flags; A.bound = t.bound; A.error = c.dError;
	A.count = count; A.entityCap = t.entityCap;
	kAnimate<<<(count + 255) / 256, 256, 0, c.stream>>>(A);
	kPropagateActive<<<(t.occupancy + 255) / 256, 256, 0, c.stream>>>(t.occupancy, t.parent, t.flags, c.dError);
	return 2;
}

uint32_t launchSetActive(Context& c, const uint32_t* dIds, uint32_t count, int active)
{
	auto& t = c.tf;
	uint32_t launches = 0;
	if (count)
	{
		kSetSelfActive<<<(count + 255) / 256, 256, 0, c.stream>>>(dIds, count, active, t.entityToSlot, t.entityCap, t.flags, c.dError);
		launches++;
	}
	if (t.occupancy)
	{
		kPropagateActive<<<(t.occupancy + 255) / 256, 256, 0, c.stream>>>(t.occupancy, t.parent, t.flags, c.dError);
		launches++;
	}
	return launches;
}

} // namespace gsp
