// Fused hot loop: world matrix (leaf-first parent-chain product) -> AABB-vs-frustum test for EVERY view of the frame ->
// visibility ballots -> deterministic stream compaction (per-chunk counts, one scan, warp-per-chunk scatter with keys).
//
// Replaces prepareUnsortedMeshes / prepareSortedMeshes (source/system/render/mesh.cpp:111-184,187-262) and what they call:
//   TransformComponent::calcModel        include/garden/system/transform.hpp:197-214
//   IMeshRenderSystem::getReadyMeshesAsync / isBehindFrustum   mesh.hpp:142-146, libraries/math/include/math/aabb.hpp:438-464
//   the key                              mesh.cpp:172,250-251
//   thread-local lists + fetch_add append mesh.cpp:177-183,257-261  (here: slot-ordered compaction, so ties sort by slot)
// The reference runs this loop once per view; here an entity's chain and corners are computed once and tested against
// all views (the camera position subtracted from the model is the same for every view, mesh.cpp:401,500).
#include "sceneprep_internal.h"
#include "sceneprep_math.cuh"
#include <math.h>
#include <algorithm>
#include <cmath>
#include <string.h>
#include <stdlib.h>

namespace gsp
{

struct CullArgs
{
	const float4* __restrict__ tRot;
	const float4* __restrict__ tPosSx;
	const float2* __restrict__ tSYZ;
	const uint32_t* __restrict__ tParent;
	const uint16_t* __restrict__ tFlags;
	const float4* __restrict__ tRecord; // per transform: prepass sphere (centre xyz, radius; < 0: not a candidate)
	const float4* __restrict__ aabbA;
	const float2* __restrict__ aabbB;
	const uint32_t* __restrict__ tslot;
	const uint8_t* __restrict__ mflags;
	const uint8_t* __restrict__ ready;
	uint32_t* __restrict__ surList;  // survivor index -> slot (written by kCompactSurvivors in slot order)
	uint32_t* __restrict__ surTs;    // survivor index -> transform slot of the owning entity
	float4* __restrict__ world;      // [survivor][kWorldStride]
	float4* __restrict__ worldPos;   // [survivor] translation column of the same matrix (what the sort key is made of)
	uint8_t* __restrict__ visible;
	uint32_t* __restrict__ visBits;  // [kMaxViews][tiles * 8] one ballot word per 32 SURVIVORS and view
	uint32_t* __restrict__ chunkCount; // [kMaxViews][chunks] visible survivors per chunk and view; scanned in place to list offsets
	uint32_t* __restrict__ counters;
	uint32_t* __restrict__ keys;
	uint32_t* __restrict__ payloads;
	uint32_t* __restrict__ sortHist; // [segment][4][256] digit histograms of the sort, accumulated by kScatter
	uint32_t* __restrict__ surBits;     // [prepass blocks][32] survivor bit per slot
	uint32_t* __restrict__ blockCount;  // [prepass blocks] survivors per prepass block
	uint32_t* __restrict__ bucketCount; // [prepass blocks / kPreBucket] survivors per bucket of blocks (zeroed per frame)
	uint32_t histOffset[kMaxViews];  // element offset of the list's histograms in sortHist (kNone = list is not sorted)
	uint32_t segOffset[kMaxViews];   // arena offset of this pool's list in view v
	uint32_t baseCounter[kMaxViews]; // counter index holding the list length before this pool (kNone = 0)
	uint32_t visibleView;            // view whose result is stored to isVisible (kNone = none)
	uint32_t tiles;                  // capacity in 256-survivor tiles (stride of visBits)
	uint32_t chunks;                 // capacity in chunks (stride of chunkCount)
	uint32_t prepassCull;            // 0: the prepass only applies the filter (GSP_PREPASS=0, for A/B measurements)
	uint32_t surCounter;             // counter index holding the length of surList (pool survivors, or surviving transforms)
	// ---- split path (pools whose hierarchies do not live in the pool itself): world matrices per surviving TRANSFORM ----
	const uint32_t* __restrict__ tList;   // surviving transforms in slot order (kPrepassT + kCompactSurvivors<true>)
	const uint32_t* __restrict__ tIndex;  // transform slot -> index in tList (only meaningful where tList[index] == slot)
	float4* __restrict__ tWorld;          // [surviving transform][kWorldStride] chain product, camera NOT subtracted
	uint32_t tCounter;                    // counter index holding the length of tList
	uint32_t tOccupancy;                  // transform slots: no acyclic chain has more links
};

constexpr uint32_t kChunkTiles = 8;                                // 256-survivor tiles per compaction chunk
constexpr uint32_t kChunkWords = kChunkTiles * (kCullTile / 32);   // ballot words per chunk (one warp of kScatter per chunk)
constexpr uint32_t kChunkItems = kChunkWords * 32;                 // survivors per chunk

// ---- conservative classification -------------------------------------------------------------------------------------------
// The reference culls an entity for a view iff some plane has all eight transformed corners at d < 0 (aabb.hpp:452-462).
// All corners lie in a sphere (centre cw, radius r), so with unit-normal planes
//   min_i (n_i . cw + d_i) < -(r + band)   =>  some plane has every corner certainly behind: culled;
//   min_i (n_i . cw + d_i) >  (r + band)   =>  every plane has every corner certainly in front: visible;
// anything else (the box straddles a plane, or NaN/Inf anywhere) runs the reference's exact 8-corner arithmetic, so the
// boolean is identical by construction. `band` absorbs every rounding difference between this real-arithmetic argument
// and the floats on either side: computed plane distances differ from real arithmetic by a few ulp of
// |n|_1 * A + |d| (A bounds every |corner lane| and every partial sum of the corner transform); kBandR * A + kBandD * |d|
// = 2^-15 * (sqrt(3) A + |d|) leaves a factor > 30 of head room over the ~2^-21 worst case.
// Cost per plane: 3 FMA + 1 MIN (the view loop is unrolled, every plane constant is a constant-bank operand).
constexpr float kBandR = 1.7321f / 32768.0f, kBandD = 1.0f / 32768.0f;

__device__ __forceinline__ float sqrtApprox(float x)
{
	float r;
	asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
	return r;
}

// smallest unit-plane distance of the point c over the view's planes (slots past planeCount are neutral: +inf)
__device__ __forceinline__ float minPlaneDistance(const ViewConst& V, float cx, float cy, float cz)
{
	// planes (2j, 2j+1) share one packed FMA chain
	f32x2 d[3];
	#pragma unroll
	for (int j = 0; j < 3; j++)
		d[j] = fma2(pack2(V.ux[j].x, V.ux[j].y), pack2(cx, cx), fma2(pack2(V.uy[j].x, V.uy[j].y), pack2(cy, cy),
			fma2(pack2(V.uz[j].x, V.uz[j].y), pack2(cz, cz), pack2(V.ud[j].x, V.ud[j].y))));
	return fminf(fminf(fminf(lo2(d[0]), hi2(d[0])), fminf(lo2(d[1]), hi2(d[1]))), fminf(lo2(d[2]), hi2(d[2])));
}

// One test for all box-shaped views of the frame (CullParams::boxMask; they share their orientation, e.g. the cascades of
// one light): with a_j the common unit face normals and [lo_j, hi_j] the union of the boxes' extents along a_j, a sphere
// (c, r) with a_j . c > hi_j + r (or < lo_j - r) for some j is behind the (j, +) (or (j, -)) face plane of EVERY box.
// `reach` = r + the classifier's band, as in the per-plane test (the band also covers the <= 1e-6 by which the boxes'
// normals may differ from the common ones, prepareBoxGroup). False for NaN / Inf.
__device__ __forceinline__ bool boxesCulled(const CullParams& P, float cx, float cy, float cz, float reach)
{
	const float r = reach + P.boxSlack;
	bool outside = false;
	#pragma unroll
	for (int j = 0; j < 3; j++)
	{
		const float t = fmaf(P.boxAxis[j][0], cx, fmaf(P.boxAxis[j][1], cy, P.boxAxis[j][2] * cz));
		outside = outside || t > P.boxHi[j] + r || t < P.boxLo[j] - r;
	}
	return outside;
}

// The prepass' view loop: true if the sphere (c, reach) may touch some enabled view. The box views of the group share the
// three dot products with their common axes, so each of them costs six comparisons against its own extents
// (CullParams::boxViewLo / boxViewHi) instead of six plane equations; when every lane of the warp is outside the union of
// the boxes they are skipped altogether. All lanes of the warp call it (`test` masks lanes that have nothing to test).
template<uint32_t kViews>
__device__ __forceinline__ bool sphereMaySurvive(const CullParams& P, bool test, float cx, float cy, float cz, float reach)
{
	float rm[3] = { 0.f, 0.f, 0.f }, rp[3] = { 0.f, 0.f, 0.f };
	bool outsideBoxes = false;
	if (P.boxMask != 0) // (uniform)
	{
		const float r = reach + P.boxSlack;
		#pragma unroll
		for (int j = 0; j < 3; j++)
		{
			const float t = fmaf(P.boxAxis[j][0], cx, fmaf(P.boxAxis[j][1], cy, P.boxAxis[j][2] * cz));
			rm[j] = t - r; rp[j] = t + r;
			outsideBoxes = outsideBoxes | (rm[j] > P.boxHi[j]) | (rp[j] < P.boxLo[j]);
		}
	}
	const uint32_t skipViews = __all_sync(0xffffffffu, outsideBoxes || !test) ? P.boxMask : 0u;
	bool maybe = false;
	if (test)
	{
		#pragma unroll
		for (uint32_t v = 0; v < kViews; v++)
		{
			if (v < P.viewCount && !((skipViews >> v) & 1u)) // warp-uniform
			{
				const ViewConst& V = P.views[v];
				bool behind; // false for NaN / infinite bounds in both forms
				// (no short-circuit evaluation: the lanes of a warp rarely agree, and a chain of predicated compares
				// is cheaper than the reconvergence of early exits)
				if ((P.boxMask >> v) & 1u) // (uniform)
					behind = (rm[0] > P.boxViewHi[v][0]) | (rp[0] < P.boxViewLo[v][0]) | (rm[1] > P.boxViewHi[v][1]) | (rp[1] < P.boxViewLo[v][1]) |
						(rm[2] > P.boxViewHi[v][2]) | (rp[2] < P.boxViewLo[v][2]);
				else
					behind = minPlaneDistance(V, cx, cy, cz) < -(reach + V.slack);
				maybe = maybe | ((V.enabled != 0) & !behind);
			}
		}
	}
	return maybe;
}

// ---- prepass: filter + hierarchical conservative culling + ordered compaction of the survivors ---------------------------
// In a large scene most entities are outside every view, and the expensive part of the path — the leaf-first product of the
// parent chain (transform.hpp:197-214) — is only needed for entities that might be visible. The prepass bounds the world box
// of a slot WITHOUT any matrix: with sigma_i >= |linear part of L_i| and tau_i >= |translation of L_i| (staging.cu,
// transformBound) for the chain e = n_0, n_1 = parent, ..., n_k = root, every corner x of the box satisfies
//     | M x - p_k |  <=  u_k,     u_0 = sigma_0 * rho,   u_i = sigma_i * (tau_(i-1) + u_(i-1))
// (rho >= |x|; p_k = the root's position, which IS the translation of its local matrix), so all eight corners lie in the
// sphere (p_k - cam, u_k). u_k is linear in rho: u_k = D + S * rho with D_0 = 0, S_0 = sigma_0, D_i = sigma_i * (tau_(i-1) +
// D_(i-1)), S_i = sigma_i * S_(i-1). Every step is inflated by 2^-8, far more than the rounding of the float product the
// bound stands for (a 4x3 product perturbs its result by < 2^-20 of the same norms), so the bound also holds for the FLOAT
// world matrix the exact path computes.
// These are quantities of the transform pool alone, so they are computed when it CHANGES, not per frame: kChainBounds walks
// every transform's chain once (D, S, root) and folds u = D + S * rho_t (rho_t = largest box of any mesh on the transform,
// kLinkPool) into W[root] = max over the hierarchy; kChainRecords then gives every transform the sphere (position of its
// root, W[root]). One sphere per hierarchy: it survives or is dropped as a whole, so the survivors' ancestors are survivors
// too and sit right before them in the list. gsp_set_transforms / gsp_update_transforms* / gsp_set_mesh_pool /
// gsp_set_active / gsp_animate mark the records stale; the next frame recomputes them before anything reads them.
// Per frame, kPrepass only streams: a slot is dropped iff, for every view it takes part in, its sphere is certainly behind one
// of the view's planes — then the reference's 8-corner test culls it too (all corners behind that plane). Everything else
// "survives": kPrepass writes one survivor bit per slot and the survivor count of its block, kCompactSurvivors turns the
// bits into surList (slot order, no inter-block dependency) and kCull does the exact work on the survivors alone.
// Non-finite or out-of-range inputs make the bound infinite or NaN (survive).
constexpr uint32_t kPreThreads = 256, kPreItems = kPreTile / kPreThreads, kPreWarps = kPreThreads / 32;
constexpr uint32_t kPreWords = kPreTile / 32;      // survivor-bit words per prepass block
constexpr uint32_t kPreBucket = 64;                // prepass blocks per bucket of the two-level survivor count
static_assert(kPreBucket == 64, "kCompactSurvivors reads the blocks of a bucket as two per lane");
constexpr uint32_t kPreMaxWalk = 255;
static_assert(kPreWords == 32, "kCompactSurvivors handles one prepass block per warp, one word per lane");

struct ChainArgs
{
	const float2* __restrict__ bound;
	const uint32_t* __restrict__ parent;
	const uint16_t* __restrict__ flags;
	const float4* __restrict__ posSx;
	const uint32_t* __restrict__ rho;
	uint32_t* __restrict__ chainRoot;
	uint32_t* __restrict__ rootW;
	float4* __restrict__ record;
	uint32_t count;
};
// Walks the parent chain of transform t (D, S above) and returns its root; `beyond`: the chain is longer than the walk allows.
__device__ __forceinline__ uint32_t chainWalk(const float2* __restrict__ bound, const uint32_t* __restrict__ parent, uint32_t t,
	float& D, float& S, bool& beyond)
{
	const float2 own = bound[t];
	float tauPrev = own.y;
	D = 0.0f; S = own.x;
	uint32_t root = t, p = parent[t], n = 0;
	while (p != kNone && n < kPreMaxWalk)
	{
		const float2 b = bound[p];
		const float d = b.x * (tauPrev + D), s = b.x * S;
		D = fmaf(d, 0x1p-8f, d); S = fmaf(s, 0x1p-8f, s);
		tauPrev = b.y; root = p; p = parent[p]; n++;
	}
	beyond = p != kNone;
	return root;
}
// u = D + S * rho, the reach of a mesh of box radius rho on the transform from its root's position
__device__ __forceinline__ float chainReach(float D, float S, float rho, bool beyond)
{
	float u = rho == 0.0f ? D : fmaf(S, rho, D); // (0 * inf would poison a transform that carries no mesh)
	if (beyond) // longer than the walk allows (or cyclic): nothing of this hierarchy is ever culled by the prepass
		u = __int_as_float(0x7f800000);
	return u;
}
__global__ void __launch_bounds__(256) kChainBounds(const __grid_constant__ ChainArgs A)
{
	const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= A.count)
		return;
	float D, S;
	bool beyond;
	const uint32_t root = chainWalk(A.bound, A.parent, t, D, S, beyond);
	const float u = chainReach(D, S, __uint_as_float(A.rho[t]), beyond);
	A.chainRoot[t] = root;
	// u >= +0, +inf or NaN: the bit patterns order like unsigned integers (NaN on top)
	if ((A.flags[t] & kTfLive) && (A.flags[root] & kTfLive))
		atomicMax(&A.rootW[root], __float_as_uint(u));
}
// Incremental link of the pool slots that gsp_update_mesh_pool[_indexed] restaged (slotMap[i], else first + i): the slot's
// transform slot, and its box radius folded into rho as kLinkPool does. rho only grows here: a smaller or moved box keeps the
// larger sphere, still conservative, until the next full link. *grew = 1 when some rho grew; with `walk` (the chain bounds
// are current) such a transform's chain is walked as kChainBounds walks it and its reach folded into rootW[root]. Each thread
// folds its own radius: the largest one that raised rho reaches rootW, so rootW covers the final rho. The records then need
// kChainRecords.
__global__ void __launch_bounds__(256) kLinkSlots(const uint32_t* __restrict__ slotMap, uint32_t first, uint32_t count,
	const uint32_t* __restrict__ entity, const uint32_t* __restrict__ entityToSlot, uint32_t entityCap,
	uint32_t* __restrict__ tslot, const float* __restrict__ radius, uint32_t* rho, int walk, const float2* __restrict__ bound,
	const uint32_t* __restrict__ parent, const uint16_t* __restrict__ tFlags, uint32_t* rootW, uint32_t* __restrict__ grew)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
		return;
	const uint32_t slot = slotMap ? slotMap[i] : first + i;
	const uint32_t e = entity[slot];
	const uint32_t s = (e && e < entityCap) ? entityToSlot[e] : 0;
	tslot[slot] = s ? s - 1 : kNone;
	if (!s)
		return;
	const uint32_t t = s - 1, r = __float_as_uint(radius[slot]);
	if (atomicMax(&rho[t], r) >= r)
		return;
	*grew = 1;
	if (!walk)
		return;
	float D, S;
	bool beyond;
	const uint32_t root = chainWalk(bound, parent, t, D, S, beyond);
	const float u = chainReach(D, S, __uint_as_float(r), beyond);
	if ((tFlags[t] & kTfLive) && (tFlags[root] & kTfLive))
		atomicMax(&rootW[root], __float_as_uint(u));
}
__global__ void __launch_bounds__(256) kChainRecords(const __grid_constant__ ChainArgs A)
{
	const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= A.count)
		return;
	const uint16_t f = A.flags[t];
	float4 rec = make_float4(0.f, 0.f, 0.f, -__int_as_float(0x7f800000)); // dead slot
	if (f & kTfLive)
	{
		float w;
		if (f & kTfAncestors)
		{
			const uint32_t root = A.chainRoot[t];
			const float4 c = A.posSx[root];
			rec = make_float4(c.x, c.y, c.z, 0.f);
			w = __uint_as_float(A.rootW[root]);
		}
		else
		{
			// modelWithAncestors == false: the model is the local matrix alone (transform.hpp:200)
			const float4 c = A.posSx[t];
			const float rho = __uint_as_float(A.rho[t]);
			rec = make_float4(c.x, c.y, c.z, 0.f);
			w = rho == 0.0f ? 0.0f : A.bound[t].x * rho;
		}
		if (w != w)
			w = __int_as_float(0x7f800000); // NaN bound: never culled (and the sign below stays meaningful)
		// the sign carries isActive() (mesh.cpp:149-155): a mesh on an inactive transform is never a candidate, but the
		// transform may still be an ancestor of active ones, so the sphere itself is kept
		rec.w = (f & kTfActive) ? w : -w;
		if (!(f & kTfActive) && w == 0.0f)
			rec.w = -0.0f;
	}
	A.record[t] = rec;
}

template<uint32_t kViews>
__global__ void __launch_bounds__(kPreThreads) kPrepass(const __grid_constant__ CullParams P, const __grid_constant__ CullArgs A)
{
	__shared__ uint32_t sCount[kPreWarps];
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t blockBase = blockIdx.x * kPreTile;

	uint32_t slot[kPreItems], ts[kPreItems];
	bool cand[kPreItems];
	#pragma unroll
	for (uint32_t k = 0; k < kPreItems; k++)
	{
		slot[k] = blockBase + k * kPreThreads + threadIdx.x;
		const bool inRange = slot[k] < P.occupancy;
		cand[k] = inRange && (A.mflags[slot[k]] & kMfCandidate);
		ts[k] = inRange ? A.tslot[slot[k]] : kNone;
		if (P.hasReady && inRange && A.ready[slot[k]] == 0) // a getReadyMeshesAsync override's extra predicate (e.g. sprite.cpp:90-97)
			cand[k] = false;
		// isVisible of the (last) main view is written for every slot like mesh.cpp:144-146,152-153,161-167: zero here,
		// kCull stores the ones
		if (A.visibleView != kNone && inRange)
			A.visible[slot[k]] = 0;
	}
	float4 rec[kPreItems];
	#pragma unroll
	for (uint32_t k = 0; k < kPreItems; k++)
	{
		cand[k] = cand[k] && ts[k] != kNone;
		rec[k] = make_float4(0.f, 0.f, 0.f, -1.0f);
		if (cand[k])
			rec[k] = A.tRecord[ts[k]];
		cand[k] = cand[k] && !signbit(rec[k].w); // live and active transform (kChainRecords stores -W otherwise)
	}
	uint32_t total = 0;
	#pragma unroll
	for (uint32_t k = 0; k < kPreItems; k++)
	{
		bool survive = cand[k];
		const bool test = cand[k] && A.prepassCull != 0;
		const float u = rec[k].w;
		const float cx = rec[k].x - P.cam[0], cy = rec[k].y - P.cam[1], cz = rec[k].z - P.cam[2];
		const float magnitude = (fabsf(cx) + fabsf(cy)) + (fabsf(cz) + u);
		const float reach = fmaf(magnitude, kBandR, u * 1.0001f);
		const bool maybe = sphereMaySurvive<kViews>(P, test, cx, cy, cz, reach);
		if (test)
			survive = maybe;
		// slots of a block are ordered (round, warp, lane): word k * kPreWarps + warp holds 32 consecutive slots
		const uint32_t votes = __ballot_sync(0xffffffffu, survive);
		if (lane == 0)
			A.surBits[(size_t)blockIdx.x * kPreWords + k * kPreWarps + warp] = votes;
		total += __popc(votes);
	}
	if (lane == 0)
		sCount[warp] = total;
	__syncthreads();
	if (threadIdx.x == 0)
	{
		uint32_t sum = 0;
		#pragma unroll
		for (uint32_t w = 0; w < kPreWarps; w++)
			sum += sCount[w];
		A.blockCount[blockIdx.x] = sum;
		if (sum)
			atomicAdd(&A.bucketCount[blockIdx.x / kPreBucket], sum);
	}
}

// Split path: the same test per TRANSFORM, for the views any split pool takes part in (P.views[].enabled). The records are
// per hierarchy, so whole hierarchies survive and a surviving mesh always finds its transform — and its ancestors — here.
template<uint32_t kViews>
__global__ void __launch_bounds__(kPreThreads) kPrepassT(const __grid_constant__ CullParams P, const __grid_constant__ CullArgs A)
{
	__shared__ uint32_t sCount[kPreWarps];
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t blockBase = blockIdx.x * kPreTile;
	uint32_t total = 0;
	#pragma unroll
	for (uint32_t k = 0; k < kPreItems; k++)
	{
		const uint32_t t = blockBase + k * kPreThreads + threadIdx.x;
		const bool live = t < P.occupancy && (A.tFlags[t] & kTfLive);
		const float4 rec = live ? A.tRecord[t] : make_float4(0.f, 0.f, 0.f, 0.f);
		const float u = fabsf(rec.w); // (the sign only says "inactive": an inactive transform may still be somebody's ancestor)
		const float cx = rec.x - P.cam[0], cy = rec.y - P.cam[1], cz = rec.z - P.cam[2];
		const float magnitude = (fabsf(cx) + fabsf(cy)) + (fabsf(cz) + u);
		const float reach = fmaf(magnitude, kBandR, u * 1.0001f);
		const bool test = live && A.prepassCull != 0;
		const bool maybe = sphereMaySurvive<kViews>(P, test, cx, cy, cz, reach);
		const bool survive = test ? maybe : live;
		const uint32_t votes = __ballot_sync(0xffffffffu, survive);
		if (lane == 0)
			A.surBits[(size_t)blockIdx.x * kPreWords + k * kPreWarps + warp] = votes;
		total += __popc(votes);
	}
	if (lane == 0)
		sCount[warp] = total;
	__syncthreads();
	if (threadIdx.x == 0)
	{
		uint32_t sum = 0;
		#pragma unroll
		for (uint32_t w = 0; w < kPreWarps; w++)
			sum += sCount[w];
		A.blockCount[blockIdx.x] = sum;
		if (sum)
			atomicAdd(&A.bucketCount[blockIdx.x / kPreBucket], sum);
	}
}

// Survivor bits -> surList (+ the survivors' transform slots) in slot order. One WARP per prepass block (lane = one word of
// 32 slots). The block's position in the list = survivors of all earlier blocks = (sum of the earlier buckets) + (sum of
// the earlier blocks of its own bucket): a few hundred L2-resident words read by the 32 lanes in parallel, so no block ever
// waits for another one. The set bits are expanded into shared memory first, so that the list is written (and the
// transform links are gathered) by whole warps.
constexpr uint32_t kCompactWarps = 8;
struct CompactArgs
{
	const uint32_t* __restrict__ bits;        // [blocks][32]
	const uint32_t* __restrict__ blockCount;  // [blocks]
	const uint32_t* __restrict__ bucketCount; // [blocks / kPreBucket + 1]
	uint32_t* __restrict__ list;              // out: survivor index -> slot
	uint32_t* __restrict__ aux;               // out: kTransforms ? slot -> survivor index : survivor index -> tslot[slot]
	const uint32_t* __restrict__ tslot;
	uint32_t* __restrict__ counters;
	uint32_t counterIndex, blocks;
};
template<bool kTransforms>
__global__ void __launch_bounds__(kCompactWarps * 32) kCompactSurvivors(const __grid_constant__ CompactArgs A)
{
	const uint32_t preBlocks = A.blocks;
	__shared__ uint16_t sOffsets[kCompactWarps][kPreTile];
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.x * kCompactWarps + warp;
	if (b >= preBlocks)
		return; // (whole warps; nothing below synchronises across warps)
	uint32_t before = 0;
	const uint32_t bucket = b / kPreBucket;
	// everything this warp reads before it can write is requested up front: its own word of survivor bits, the counts of the
	// earlier blocks of its bucket, the earlier buckets
	const uint32_t bits = A.bits[(size_t)b * kPreWords + lane];
	{
		const uint32_t i0 = bucket * kPreBucket + lane, i1 = i0 + 32; // (kPreBucket == 64: two blocks per lane)
		const uint32_t v0 = i0 < b ? A.blockCount[i0] : 0u, v1 = i1 < b ? A.blockCount[i1] : 0u;
		before = v0 + v1;
	}
	for (uint32_t j0 = lane; j0 < bucket; j0 += 32 * 8) // 8 independent loads in flight per lane
	{
		uint32_t v[8];
		#pragma unroll
		for (uint32_t q = 0; q < 8; q++)
			v[q] = j0 + 32 * q < bucket ? A.bucketCount[j0 + 32 * q] : 0u;
		#pragma unroll
		for (uint32_t q = 0; q < 8; q++)
			before += v[q];
	}
	before = __reduce_add_sync(0xffffffffu, before);
	const uint32_t c = __popc(bits);
	uint32_t inc = c;
	#pragma unroll
	for (int o = 1; o < 32; o <<= 1)
	{
		const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
		if (lane >= (uint32_t)o) inc += t;
	}
	const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
	{
		uint32_t pos = inc - c, rest = bits;
		while (rest)
		{
			sOffsets[warp][pos++] = (uint16_t)(lane * 32 + __ffs(rest) - 1);
			rest &= rest - 1;
		}
	}
	__syncwarp();
	// four list positions per lane and round: the transform links are gathered with four loads in flight
	for (uint32_t j0 = lane; j0 < total; j0 += 32 * 4)
	{
		uint32_t slot[4], link[4];
		#pragma unroll
		for (uint32_t q = 0; q < 4; q++)
		{
			const uint32_t j = j0 + 32 * q;
			slot[q] = b * kPreTile + (j < total ? sOffsets[warp][j] : 0u);
			link[q] = (!kTransforms && j < total) ? A.tslot[slot[q]] : 0u;
		}
		#pragma unroll
		for (uint32_t q = 0; q < 4; q++)
		{
			const uint32_t j = j0 + 32 * q;
			if (j < total)
			{
				A.list[before + j] = slot[q];
				if (kTransforms)
					A.aux[slot[q]] = before + j;
				else
					A.aux[before + j] = link[q];
			}
		}
	}
	if (b == preBlocks - 1 && lane == 0)
		A.counters[A.counterIndex] = before + total;
}

// ---- shared-memory cache of local matrices ----------------------------------------------------------------------------------
// Leaf-first association (transform.hpp:204-210) forces every entity to multiply its own chain, but the chain's factors —
// the ancestors' LOCAL matrices — are shared. Each WARP owns a tile of kWarpTile consecutive SURVIVORS and a private slice
// of shared memory holding kEntries local matrices: entry i < kWarpTile is the own transform of the tile's i-th survivor,
// the rest is the ANCESTOR CLOSURE of the tile — every lane walks up its parent links and the first lane to meet a transform
// that has no entry yet computes its local matrix (bit-identical wherever it is computed, SURVEY.md §7), so chains whose
// ancestors live in another pool, or anywhere else in the transform pool, still run out of shared memory. A small hash
// table (transform slot -> entry) is only used while the tile is set up: every entry then resolves its parent link to an
// ENTRY INDEX once (kLinkEnd = root, kLinkMiss = no entry: table full), so a chain step in the hot loop is one 16-bit
// link load, three 128-bit matrix loads, 24 packed multiply-adds. Entries are handed out in survivor order, so the lanes
// of a warp — which walk neighbouring chains — read neighbouring entries (no bank conflicts on the 128-bit loads).
// Warps never synchronise with each other (only __syncwarp): while one warp waits for its loads, the others compute.
constexpr uint32_t kWarpTile = 64, kWarpItems = kWarpTile / 32;       // survivors per warp tile, survivors per lane
constexpr uint32_t kEntries = 96;                                     // kWarpTile own transforms + closure
constexpr uint32_t kHalo = 16;                                        // survivors before the tile that may get an entry speculatively
constexpr uint32_t kHashBits = 7, kHashSize = 1u << kHashBits, kHashProbes = 16;
constexpr uint32_t kEntryNone = 0xFFu;
constexpr uint32_t kDepthBins = 32;
constexpr uint32_t kLinkEnd = 0xFFFFu, kLinkMiss = 0xFFFEu, kLinkTodo = 0xFFFDu;
constexpr uint32_t kDepthUnknown = kTfDepthMax; // chain-length hint saturates here: such chains take the guarded slow path
static_assert(kWarpItems == 2, "work items are dealt as a deep half and a shallow half");
static_assert(kEntries >= kWarpTile && kEntries < kEntryNone, "entry indices fit a byte");

struct CullShared // one per warp
{
	float4 L[kEntries][3];      // per entry: row l = (c0[l], c1[l], c2[l], c3[l]); 48-byte stride: 128-bit accesses conflict-free
	uint32_t hkey[kHashSize];   // hash table: transform slot (kNone = empty) ...
	uint32_t par[kEntries];     // per entry: parent transform slot
	uint32_t closure[kEntries - kWarpTile]; // transform slot of each closure entry (until its matrix has been computed)
	uint32_t slotOf[kWarpTile]; // per owner: pool slot (kNone = past the end of the survivor list)
	uint32_t hist[kDepthBins];
	uint32_t inst[kMaxViews];
	uint32_t nEntries;
	uint16_t lnk[kEntries];     // entry index of the parent's entry, kLinkEnd or kLinkMiss
	uint16_t maskOf[kWarpTile]; // per owner: visibility bit per view
	uint8_t hval[kHashSize];    // ... -> entry index (kEntryNone: the transform is known to have no entry)
	uint8_t perm[kWarpTile];    // work item -> owner, ordered by chain length (deepest first)
	uint8_t ownSteps[kWarpTile]; // per owner: ancestors to multiply in (0 when modelWithAncestors == false)
};

__device__ __forceinline__ uint32_t hashOf(uint32_t t) { return (t * 0x9E3779B1u) >> (32 - kHashBits); }

// entry index of transform slot t, or kEntryNone
__device__ __forceinline__ uint32_t cacheFind(const CullShared& sh, uint32_t t)
{
	uint32_t h = hashOf(t);
	for (uint32_t i = 0; i < kHashProbes; i++)
	{
		const uint32_t k = sh.hkey[h];
		if (k == t) return sh.hval[h];
		if (k == kNone) return kEntryNone;
		h = (h + 1) & (kHashSize - 1);
	}
	return kEntryNone;
}
// 0: the key was inserted by this call (the caller owns sh.hval[h]); 1: it was there already; 2: no room
__device__ __forceinline__ int cacheClaim(CullShared& sh, uint32_t t, uint32_t& h)
{
	h = hashOf(t);
	for (uint32_t i = 0; i < kHashProbes; i++)
	{
		const uint32_t old = atomicCAS(&sh.hkey[h], kNone, t);
		if (old == kNone) return 0;
		if (old == t) return 1;
		h = (h + 1) & (kHashSize - 1);
	}
	return 2;
}

__device__ __forceinline__ Mat43 loadLocal43(const CullArgs& a, uint32_t t)
{
	float4 q = a.tRot[t];
	float4 p = a.tPosSx[t];
	float2 s = a.tSYZ[t];
	return localModel43(p.x, p.y, p.z, q.x, q.y, q.z, q.w, p.w, s.x, s.y, (a.tFlags[t] & kTfExactLocal) != 0);
}

__device__ __forceinline__ void entryStore(CullShared& sh, uint32_t e, uint32_t parent, const Mat43& L)
{
	#pragma unroll
	for (int l = 0; l < 3; l++)
		sh.L[e][l] = make_float4(L.c[0][l], L.c[1][l], L.c[2][l], L.c[3][l]);
	sh.par[e] = parent;
}

__device__ __forceinline__ Mat43 cachedLocal(const CullShared& sh, uint32_t e)
{
	Mat43 L;
	#pragma unroll
	for (int l = 0; l < 3; l++)
	{
		const float4 a = sh.L[e][l];
		L.c[0][l] = a.x; L.c[1][l] = a.y; L.c[2][l] = a.z; L.c[3][l] = a.w;
	}
	return L;
}

// Local matrix + parent link of transform slot t: from its entry when it has one, else recomputed from the SoA streams.
__device__ __forceinline__ Mat43 fetchLocal(const CullShared& sh, const CullArgs& a, uint32_t t, uint32_t& parent)
{
	const uint32_t e = cacheFind(sh, t);
	Mat43 L;
	if (e != kEntryNone)
	{
		L = cachedLocal(sh, e);
		parent = sh.par[e];
	}
	else
	{
		L = loadLocal43(a, t);
		parent = a.tParent[t];
	}
	return L;
}

// Guarded generic chain walk (cold): continues M = L(p) * M from transform slot p to the root.
static __device__ __forceinline__ void walkChainSlow(const CullShared& sh, const CullArgs& a, uint32_t p, Mat43& M)
{
	uint32_t depth = 0;
	while (p != kNone)
	{
		if (++depth > a.tOccupancy) // (cannot happen: cyclic hierarchies are refused before launch)
		{
			atomicExch(&a.counters[kCtrError], (uint32_t)GSP_ERR_HIERARCHY);
			break;
		}
		uint32_t next;
		const Mat43 L = fetchLocal(sh, a, p, next);
		M = matMul43(L, M);
		p = next;
	}
}

// ---- phase 3: the world box against every view -------------------------------------------------------------------------------
// M = the model matrix (camera position already subtracted, transform.hpp:211), box = the component's AABB. Returns the bit
// mask of views in which the reference's isBehindFrustum (aabb.hpp:438-464) does NOT cull the box. Called by all lanes of a
// warp (it votes); lanes with work == false return 0.
template<uint32_t kViews>
__device__ __forceinline__ uint32_t classifyBox(const CullParams& P, const Mat43& M, const float4 boxA, const float2 boxB, const bool work)
{
	constexpr uint32_t kFull = 0xffffffffu;
	uint32_t mask = 0;
	float mn[3], mx[3];
	{
		const float4 ba = boxA;
		const float2 bb = boxB;
		mn[0] = ba.x; mn[1] = ba.y; mn[2] = ba.z; mx[0] = ba.w; mx[1] = bb.x; mx[2] = bb.y;
	}

	// ---- phase 3a: bounding sphere of the transformed box + error band (any rounding is fine here, the band absorbs it) ----
	float cw[3]; // world-space centre
	float reach; // sphere radius + band
	bool finite;
	{
		float ctr[3], ext[3], amax[3];
		#pragma unroll
		for (int k = 0; k < 3; k++)
		{
			ctr[k] = 0.5f * (mn[k] + mx[k]);
			ext[k] = 0.5f * fabsf(mx[k] - mn[k]);
			amax[k] = fmaxf(fabsf(mn[k]), fabsf(mx[k]));
		}
		#pragma unroll
		for (int l = 0; l < 3; l++)
			cw[l] = fmaf(M.c[0][l], ctr[0], fmaf(M.c[1][l], ctr[1], fmaf(M.c[2][l], ctr[2], M.c[3][l])));
		// sum_i |c_i| * e_i <= sqrt(3 * sum_i |c_i|^2 e_i^2): with e = ext it bounds the corner distance from the centre,
		// with e = amax (plus |c3|) it bounds every |corner lane| and every partial sum of the corner transform
		float rr = 0.0f, ra = 0.0f;
		#pragma unroll
		for (int i = 0; i < 3; i++)
		{
			const float len2 = fmaf(M.c[i][0], M.c[i][0], fmaf(M.c[i][1], M.c[i][1], M.c[i][2] * M.c[i][2]));
			rr = fmaf(len2, ext[i] * ext[i], rr);
			ra = fmaf(len2, amax[i] * amax[i], ra);
		}
		const float c3max = fmaxf(fmaxf(fabsf(M.c[3][0]), fabsf(M.c[3][1])), fabsf(M.c[3][2]));
		const float magnitude = fmaf(sqrtApprox(3.0f * ra), 1.0001f, c3max);
		reach = fmaf(magnitude, kBandR, sqrtApprox(3.0f * rr) * 1.0001f);
		// NaN / Inf anywhere in the matrix poisons this sum: such entities always take the exact test
		finite = fabsf(((cw[0] + cw[1]) + (cw[2] + rr)) + ra) < __int_as_float(0x7f800000);
	}

	// ---- phase 3b: per view, the smallest unit-plane distance of the centre decides (see above) ----
	uint32_t exactViews = 0; // views that need the exact test
	// box views (cascades) are skipped by the whole warp when every lane's box is certainly outside all of them
	const bool outsideBoxes = P.boxMask != 0 && finite && boxesCulled(P, cw[0], cw[1], cw[2], reach);
	const uint32_t skipViews = __all_sync(kFull, outsideBoxes || !work) ? P.boxMask : 0u;
	#pragma unroll
	for (uint32_t v = 0; v < kViews; v++)
	{
		if (v < P.viewCount && !((skipViews >> v) & 1u)) // warp-uniform
		{
			const ViewConst& V = P.views[v];
			const float dmin = minPlaneDistance(V, cw[0], cw[1], cw[2]);
			const float t = reach + V.slack;
			const bool front = dmin > t, behind = dmin < -t;
			if (V.enabled)
			{
				if (front && finite)
					mask |= 1u << v;
				else if (!(behind && finite))
					exactViews |= 1u << v;
			}
		}
	}
	if (!work)
	{
		mask = 0; exactViews = 0;
	}
	if (exactViews) // rare: the box straddles a plane
	{
		float vx[8], vy[8], vz[8];
		#pragma unroll
		for (int k = 0; k < 8; k++)
			transformCorner43(M, (k & 4) ? mx[0] : mn[0], (k & 2) ? mx[1] : mn[1], (k & 1) ? mx[2] : mn[2], vx[k], vy[k], vz[k]);
		while (exactViews)
		{
			const uint32_t v = __ffs(exactViews) - 1;
			exactViews &= exactViews - 1;
			const ViewConst& V = P.views[v];
			bool culled = false;
			for (uint32_t i = 0; i < V.planeCount && !culled; i++)
			{
				const float nx = V.planes[i][0], ny = V.planes[i][1], nz = V.planes[i][2], nd = V.planes[i][3];
				bool allBehind = true;
				#pragma unroll
				for (int k = 0; k < 8; k++)
					allBehind = allBehind && (planeDistance(nx, ny, nz, nd, vx[k], vy[k], vz[k]) < 0.0f);
				culled = allBehind;
			}
			if (!culled)
				mask |= 1u << v;
		}
	}
	return mask;
}

// One block = kCullWarps independent warps; every warp walks the survivor list in tiles of kWarpTile with a grid stride.
// Inside a tile the work items are ordered by chain length (deepest first); lane i takes item i of the deep half and item i
// of the shallow half, so the warp walks chains of similar length together and every lane carries about the same total.
constexpr uint32_t kCullThreads = 128, kCullWarps = kCullThreads / 32, kCullBlocksPerSM = 8;
static_assert(kCullWarps * kWarpTile == kCullTile, "a block covers one kCullTile per round");

// kWorldOnly: the split path's first half — the items are surviving TRANSFORMS (A.surList = tList, A.surTs = tList), the
// chain product goes to A.tWorld without the camera translation, nothing is classified.
template<uint32_t kViews, bool kWorldOnly>
__global__ void __launch_bounds__(kCullThreads, kCullBlocksPerSM) kCull(const __grid_constant__ CullParams P, const __grid_constant__ CullArgs A)
{
	__shared__ CullShared shAll[kCullWarps];
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	CullShared& sh = shAll[warp];
	constexpr uint32_t kFull = 0xffffffffu;
	const uint32_t survivors = A.counters[A.surCounter];
	const uint32_t tileCount = (survivors + kWarpTile - 1) / kWarpTile;
	const uint32_t words = A.tiles * (kCullTile / 32);

	#pragma unroll 1
	for (uint32_t tile = blockIdx.x * kCullWarps + warp; tile < tileCount; tile += gridDim.x * kCullWarps)
	{
	const uint32_t tileBase = tile * kWarpTile;
	__syncwarp(); // the previous tile's readers are done with this warp's slice
	for (uint32_t i = lane; i < kHashSize; i += 32)
		sh.hkey[i] = kNone;
	sh.hist[lane] = 0;
	if (lane < kMaxViews)
		sh.inst[lane] = 0;
	if (lane == 0)
		sh.nEntries = kWarpTile;
	__syncwarp();

	// ---- phase 1: local matrix of the own transform into entry `own` (every survivor passed the filter, mesh.cpp:140-155) ----
	// Both survivors of the lane move through the dependent load levels together, and their local matrices are computed by
	// straight-line code so the two dependency chains interleave.
	uint32_t depthKey[kWarpItems], rankInBin[kWarpItems], steps[kWarpItems], parentLink[kWarpItems];
	bool valid[kWarpItems];
	// halo: the survivors right before the tile. Hierarchies survive the prepass as a whole and are usually laid out
	// parent-first, so the ancestors of the tile's first chains are exactly these; their links are fetched together with
	// the tile's own loads and `haloNeed` of them get an entry below without any walk.
	uint32_t haloTs = kNone, haloParent = kNone, haloNeed = 0;
	{
		uint32_t ts[kWarpItems];
		if (lane < kHalo && tileBase > lane)
			haloTs = A.surTs[tileBase - 1 - lane];
		#pragma unroll
		for (uint32_t r = 0; r < kWarpItems; r++)
		{
			const uint32_t own = lane + r * 32;
			valid[r] = tileBase + own < survivors;
			const uint32_t slot = valid[r] ? A.surList[tileBase + own] : kNone;
			ts[r] = valid[r] ? A.surTs[tileBase + own] : kNone;
			sh.slotOf[own] = slot;
		}
		uint16_t tf[kWarpItems];
		float4 tq[kWarpItems], tp[kWarpItems];
		float2 tsyz[kWarpItems];
		#pragma unroll
		for (uint32_t r = 0; r < kWarpItems; r++)
		{
			// flags, TRS and parent link depend only on `ts`: all loads of both survivors are issued together
			tf[r] = 0; tq[r] = make_float4(0.f, 0.f, 0.f, 1.f); tp[r] = make_float4(0.f, 0.f, 0.f, 1.f);
			tsyz[r] = make_float2(1.f, 1.f); parentLink[r] = kNone;
			if (valid[r])
			{
				tf[r] = A.tFlags[ts[r]]; tq[r] = A.tRot[ts[r]]; tp[r] = A.tPosSx[ts[r]]; tsyz[r] = A.tSYZ[ts[r]];
				parentLink[r] = A.tParent[ts[r]];
			}
		}
		if (haloTs != kNone)
			haloParent = A.tParent[haloTs];
		Mat43 L[kWarpItems];
		#pragma unroll
		for (uint32_t r = 0; r < kWarpItems; r++)
			localModel43Fast<false>(tp[r].x, tp[r].y, tp[r].z, tq[r].x, tq[r].y, tq[r].z, tq[r].w, tp[r].w, tsyz[r].x, tsyz[r].y, L[r]);
		#pragma unroll
		for (uint32_t r = 0; r < kWarpItems; r++)
		{
			const uint32_t own = lane + r * 32;
			// Survivors are in slot order and hierarchies are usually laid out parent-first, so the parent of a survivor's
			// transform is very often the transform of the survivor right before it: its entry is then own - 1, no lookup.
			uint32_t prevTs = __shfl_up_sync(kFull, ts[r], 1);
			if (r != 0)
			{
				const uint32_t wrap = __shfl_sync(kFull, ts[0], 31);
				if (lane == 0) prevTs = wrap;
			}
			else if (lane == 0)
				prevTs = kNone;
			const bool parentIsPrev = valid[r] && parentLink[r] != kNone && parentLink[r] == prevTs;
			if (valid[r])
			{
				if (tf[r] & kTfExactLocal) // zero / subnormal entries, out-of-range inputs: the exact 4-lane code (rare)
					L[r] = localModel43Slow(tp[r].x, tp[r].y, tp[r].z, tq[r].x, tq[r].y, tq[r].z, tq[r].w, tp[r].w, tsyz[r].x, tsyz[r].y);
				entryStore(sh, own, parentLink[r], L[r]);
				uint32_t h;
				if (cacheClaim(sh, ts[r], h) == 0)
					sh.hval[h] = (uint8_t)own;
				sh.lnk[own] = (uint16_t)(parentLink[r] == kNone ? kLinkEnd : parentIsPrev ? own - 1 : kLinkTodo);
			}
			else
			{
				sh.par[own] = kNone;
				sh.lnk[own] = (uint16_t)kLinkEnd;
			}
			// chain length (capped) orders the tile's work; modelWithAncestors == false means no walk at all (transform.hpp:200)
			const bool walk = valid[r] && (tf[r] & kTfAncestors);
			steps[r] = walk ? (uint32_t)(tf[r] >> kTfDepthShift) : 0u;
			if (!walk || parentIsPrev) parentLink[r] = kNone; // (nothing to look for above this lane's item)
			if (walk && steps[r] != kDepthUnknown && steps[r] > own)
				haloNeed = max(haloNeed, steps[r] - own); // ancestors of a chain that starts before the tile
			depthKey[r] = min(steps[r], kDepthBins - 1);
			sh.ownSteps[own] = (uint8_t)steps[r];
			rankInBin[r] = atomicAdd(&sh.hist[depthKey[r]], 1u);
		}
	}
	__syncwarp();
	// ---- ancestor closure: transforms on the tile's chains that have no entry yet (ancestors outside the tile: another pool,
	// a parent that was culled by the prepass, a hierarchy that is not laid out in order). The first lane to claim a
	// transform computes its local matrix; a lane that meets a claimed one stops (its claimer walks on from there).
	// Three steps, so that the matrices are computed by all lanes at once: (h) the halo survivors claim entries without any
	// walk; (a) every lane whose parent is still unknown walks the links, claims entries and notes the transform slot of each
	// new entry (with the halo in place this finds everything present in an ordered hierarchy); (b) one local matrix per lane.
	haloNeed = min(__reduce_max_sync(kFull, haloNeed), kHalo);
	if (lane < haloNeed && haloTs != kNone)
	{
		uint32_t h;
		if (cacheClaim(sh, haloTs, h) == 0)
		{
			const uint32_t e = atomicAdd(&sh.nEntries, 1u);
			if (e < kEntries)
			{
				sh.hval[h] = (uint8_t)e;
				sh.closure[e - kWarpTile] = haloTs;
				sh.par[e] = haloParent;
				sh.lnk[e] = (uint16_t)(haloParent == kNone ? kLinkEnd : kLinkTodo);
			}
			else
				sh.hval[h] = (uint8_t)kEntryNone;
		}
	}
	__syncwarp();
	#pragma unroll 1
	for (uint32_t r = 0; r < kWarpItems; r++)
	{
		uint32_t p = parentLink[r];
		for (uint32_t budget = steps[r]; p != kNone && budget != 0; budget--)
		{
			uint32_t h;
			if (cacheClaim(sh, p, h) != 0)
				break;
			const uint32_t e = atomicAdd(&sh.nEntries, 1u);
			if (e >= kEntries)
			{
				sh.hval[h] = (uint8_t)kEntryNone; // known, but no room: chains through it finish on the generic path
				break;
			}
			sh.hval[h] = (uint8_t)e;
			sh.closure[e - kWarpTile] = p;
			const uint32_t next = A.tParent[p];
			sh.par[e] = next;
			sh.lnk[e] = (uint16_t)(next == kNone ? kLinkEnd : kLinkTodo);
			p = next;
		}
	}
	__syncwarp();
	for (uint32_t e = kWarpTile + lane; e < min(sh.nEntries, kEntries); e += 32)
	{
		const Mat43 H = loadLocal43(A, sh.closure[e - kWarpTile]);
		#pragma unroll
		for (int l = 0; l < 3; l++)
			sh.L[e][l] = make_float4(H.c[0][l], H.c[1][l], H.c[2][l], H.c[3][l]);
	}
	{
		// exclusive scan of the depth histogram, deepest chains first: lane i owns bin (kDepthBins - 1 - i)
		const uint32_t c = sh.hist[kDepthBins - 1 - lane];
		uint32_t inc = c;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1)
		{
			uint32_t t = __shfl_up_sync(kFull, inc, o);
			if (lane >= (uint32_t)o) inc += t;
		}
		const uint32_t exclusive = inc - c;
		#pragma unroll
		for (uint32_t r = 0; r < kWarpItems; r++)
		{
			const uint32_t start = __shfl_sync(kFull, exclusive, kDepthBins - 1 - depthKey[r]);
			sh.perm[start + rankInBin[r]] = (uint8_t)(lane + r * 32);
		}
	}
	__syncwarp();
	// parent links as entry indices (once per entry instead of once per chain step)
	{
		const uint32_t n = min(sh.nEntries, kEntries);
		for (uint32_t e = lane; e < n; e += 32)
		{
			if (sh.lnk[e] == kLinkTodo) // (the others were settled when the entry was made)
			{
				const uint32_t pe = cacheFind(sh, sh.par[e]);
				sh.lnk[e] = (uint16_t)(pe != kEntryNone ? pe : kLinkMiss);
			}
		}
	}
	__syncwarp();

	// ---- phases 2 + 3 run per WORK ITEM: r = 0 the deep half, r = 1 the shallow half ----
	#pragma unroll 1
	for (uint32_t r = 0; r < kWarpItems; r++)
	{
		const uint32_t owner = sh.perm[r * 32 + lane];
		const uint32_t wslot = sh.slotOf[owner];
		const bool work = wslot != kNone;
		uint32_t mask = 0;
		// the box is only needed after the chain product: its loads fly meanwhile
		float4 boxA = make_float4(0.f, 0.f, 0.f, 0.f);
		float2 boxB = make_float2(0.f, 0.f);
		if (work && !kWorldOnly)
		{
			boxA = A.aabbA[wslot];
			boxB = A.aabbB[wslot];
		}

		// ---- phase 2: world matrix, leaf-first chain product (transform.hpp:199-211) ----
		Mat43 M;
		#pragma unroll
		for (int i = 0; i < 4; i++)
			for (int l = 0; l < 3; l++)
				M.c[i][l] = (i == l) ? 1.0f : 0.0f;
		if (work)
		{
			const uint32_t steps = sh.ownSteps[owner];
			uint32_t e = owner;
			uint32_t slowFrom = kNone; // transform slot the slow path continues from
			bool slow = false;
			if (steps != kDepthUnknown)
			{
				Mat43P Mp; // column pairs straight out of the row-major entry
				#pragma unroll
				for (int l = 0; l < 3; l++)
				{
					const float4 a = sh.L[e][l];
					Mp.p[l][0] = pack2(a.x, a.y); Mp.p[l][1] = pack2(a.z, a.w);
				}
				uint32_t link = steps ? (uint32_t)sh.lnk[e] : kLinkEnd;
				#pragma unroll 2
				for (uint32_t s = 0; s < steps && link < kLinkMiss; s++)
				{
					e = link;
					const float4 a[3] = { sh.L[e][0], sh.L[e][1], sh.L[e][2] };
					Mp = matMul43P(a, Mp);
					link = sh.lnk[e];
				}
				M = unpairMat(Mp);
				// the hint and the links agree unless an ancestor has no entry (or the hint is stale): finish generically
				if (link != kLinkEnd)
				{
					slow = true; slowFrom = sh.par[e];
				}
			}
			else
			{
				M = cachedLocal(sh, e);
				slow = true; slowFrom = sh.par[e];
			}
			if (slow)
				walkChainSlow(sh, A, slowFrom, M);
		}
		if (kWorldOnly)
		{
			if (work)
			{
				float4* w = A.tWorld + (size_t)(tileBase + owner) * kWorldStride;
				w[0] = make_float4(M.c[0][0], M.c[0][1], M.c[0][2], M.c[1][0]);
				w[1] = make_float4(M.c[1][1], M.c[1][2], M.c[2][0], M.c[2][1]);
				w[2] = make_float4(M.c[2][2], M.c[3][0], M.c[3][1], M.c[3][2]);
			}
			continue;
		}
		// translate(-cameraPosition, model): c3.xyz += -cam, w kept (matrix/transform.hpp:71-74)
		M.c[3][0] = __fadd_rn(M.c[3][0], -P.cam[0]);
		M.c[3][1] = __fadd_rn(M.c[3][1], -P.cam[1]);
		M.c[3][2] = __fadd_rn(M.c[3][2], -P.cam[2]);

		mask = classifyBox<kViews>(P, M, boxA, boxB, work);
		uint32_t readyCount = 1;
		if (P.hasReady && mask) // a getReadyMeshesAsync override's extra predicate (e.g. sprite.cpp:90-97)
		{
			readyCount = A.ready[wslot];
			if (readyCount == 0) mask = 0;
		}
		if (mask) // bakedModel = (float4x3)model (mesh.cpp:171,249)
		{
			float4* w = A.world + (size_t)(tileBase + owner) * kWorldStride;
			w[0] = make_float4(M.c[0][0], M.c[0][1], M.c[0][2], M.c[1][0]);
			w[1] = make_float4(M.c[1][1], M.c[1][2], M.c[2][0], M.c[2][1]);
			w[2] = make_float4(M.c[2][2], M.c[3][0], M.c[3][1], M.c[3][2]);
			A.worldPos[tileBase + owner] = make_float4(M.c[3][0], M.c[3][1], M.c[3][2], 0.f);
			if (P.hasReady)
			{
				for (uint32_t v = 0; v < P.viewCount; v++)
					if ((mask >> v) & 1u)
						atomicAdd(&sh.inst[v], readyCount);
			}
		}
		sh.maskOf[owner] = (uint16_t)mask;
	}
	__syncwarp();
	if (kWorldOnly)
		continue;

	// ---- back to survivor order: isVisible, one ballot word per 32 survivors and view, the tile's visible count per view ----
	// (no inter-tile dependency in this kernel: list positions are assigned by kScanChunks + kScatter below)
	uint32_t visibleCount = 0; // lane v: visible survivors of the tile in view v
	#pragma unroll
	for (uint32_t r = 0; r < kWarpItems; r++)
	{
		const uint32_t own = lane + r * 32;
		const uint32_t mask = sh.maskOf[own];
		// isVisible of the (last) main view: the prepass stored 0 for every slot, the visible survivors get their 1 here
		if (A.visibleView != kNone && ((mask >> A.visibleView) & 1u))
			A.visible[sh.slotOf[own]] = 1;
		uint32_t mine = 0; // lane v keeps the ballot word of view v
		#pragma unroll
		for (uint32_t v = 0; v < kViews; v++)
		{
			const uint32_t b = __ballot_sync(kFull, (mask >> v) & 1u);
			if (lane == v) mine = b;
		}
		if (lane < P.viewCount)
		{
			A.visBits[(size_t)lane * words + tile * kWarpItems + r] = mine;
			visibleCount += __popc(mine);
		}
	}
	if (lane < P.viewCount)
	{
		// visible slots per chunk of kChunkTiles tiles: the only cross-tile quantity the compaction needs
		if (visibleCount)
			atomicAdd(&A.chunkCount[(size_t)lane * A.chunks + tileBase / kChunkItems], visibleCount);
		if (P.hasReady && sh.inst[lane])
			atomicAdd(&A.counters[ctrPoolInst(P.poolIndex, lane)], sh.inst[lane]);
	}
	} // tile loop
}

// ---- split path, second half: the pool's survivors pick up their transform's world matrix and are classified ----------------
// One survivor per lane, one ballot word per warp step. The matrix comes from tWorld (kCull<.., true> over the surviving
// transforms); a survivor whose transform is not there (cannot happen while the two prepasses see the same spheres; kept as
// a guard) multiplies its chain from the SoA streams right here. Everything after the matrix is the fused kernel's phase 3.
constexpr uint32_t kClassifyThreads = 256;
static __device__ __noinline__ Mat43 chainFromStreams(const CullArgs& a, uint32_t ts)
{
	Mat43 M = loadLocal43(a, ts);
	if (!(a.tFlags[ts] & kTfAncestors))
		return M;
	uint32_t p = a.tParent[ts], depth = 0;
	while (p != kNone)
	{
		if (++depth > a.tOccupancy) // (cannot happen: cyclic hierarchies are refused before launch)
		{
			atomicExch(&a.counters[kCtrError], (uint32_t)GSP_ERR_HIERARCHY);
			break;
		}
		M = matMul43(loadLocal43(a, p), M);
		p = a.tParent[p];
	}
	return M;
}

template<uint32_t kViews>
__global__ void __launch_bounds__(kClassifyThreads) kClassify(const __grid_constant__ CullParams P, const __grid_constant__ CullArgs A)
{
	constexpr uint32_t kFull = 0xffffffffu;
	const uint32_t lane = threadIdx.x & 31;
	const uint32_t survivors = A.counters[A.surCounter], transforms = A.counters[A.tCounter];
	const uint32_t liveWords = ((survivors + kWarpTile - 1) / kWarpTile) * kWarpItems; // kScatter reads the words in pairs
	const uint32_t words = A.tiles * (kCullTile / 32);
	const uint32_t warpsTotal = gridDim.x * (kClassifyThreads / 32);
	for (uint32_t word = blockIdx.x * (kClassifyThreads / 32) + (threadIdx.x >> 5); word < liveWords; word += warpsTotal)
	{
		const uint32_t idx = word * 32 + lane;
		const bool valid = idx < survivors;
		uint32_t slot = kNone, ts = kNone, tidx = kNone;
		if (valid)
		{
			slot = A.surList[idx]; ts = A.surTs[idx];
		}
		float4 boxA = make_float4(0.f, 0.f, 0.f, 0.f);
		float2 boxB = make_float2(0.f, 0.f);
		if (valid)
		{
			tidx = A.tIndex[ts];
			boxA = A.aabbA[slot]; boxB = A.aabbB[slot];
		}
		Mat43 M;
		#pragma unroll
		for (int i = 0; i < 4; i++)
			for (int l = 0; l < 3; l++)
				M.c[i][l] = (i == l) ? 1.0f : 0.0f;
		const bool found = valid && tidx < transforms && A.tList[tidx] == ts;
		if (found)
		{
			const float4* w = A.tWorld + (size_t)tidx * kWorldStride;
			const float4 w0 = w[0], w1 = w[1], w2 = w[2];
			M.c[0][0] = w0.x; M.c[0][1] = w0.y; M.c[0][2] = w0.z; M.c[1][0] = w0.w;
			M.c[1][1] = w1.x; M.c[1][2] = w1.y; M.c[2][0] = w1.z; M.c[2][1] = w1.w;
			M.c[2][2] = w2.x; M.c[3][0] = w2.y; M.c[3][1] = w2.z; M.c[3][2] = w2.w;
		}
		else if (valid)
			M = chainFromStreams(A, ts);
		// translate(-cameraPosition, model): c3.xyz += -cam, w kept (matrix/transform.hpp:71-74)
		M.c[3][0] = __fadd_rn(M.c[3][0], -P.cam[0]);
		M.c[3][1] = __fadd_rn(M.c[3][1], -P.cam[1]);
		M.c[3][2] = __fadd_rn(M.c[3][2], -P.cam[2]);
		uint32_t mask = classifyBox<kViews>(P, M, boxA, boxB, valid);
		uint32_t readyCount = 1;
		if (P.hasReady && mask) // a getReadyMeshesAsync override's extra predicate (e.g. sprite.cpp:90-97)
		{
			readyCount = A.ready[slot];
			if (readyCount == 0) mask = 0;
		}
		if (mask) // bakedModel = (float4x3)model (mesh.cpp:171,249)
		{
			float4* w = A.world + (size_t)idx * kWorldStride;
			w[0] = make_float4(M.c[0][0], M.c[0][1], M.c[0][2], M.c[1][0]);
			w[1] = make_float4(M.c[1][1], M.c[1][2], M.c[2][0], M.c[2][1]);
			w[2] = make_float4(M.c[2][2], M.c[3][0], M.c[3][1], M.c[3][2]);
			A.worldPos[idx] = make_float4(M.c[3][0], M.c[3][1], M.c[3][2], 0.f);
			if (A.visibleView != kNone && ((mask >> A.visibleView) & 1u))
				A.visible[slot] = 1; // (the prepass stored 0 for every slot)
		}
		uint32_t mine = 0, inst = 0; // lane v keeps the ballot word / instance count of view v
		#pragma unroll
		for (uint32_t v = 0; v < kViews; v++)
		{
			const bool bit = (mask >> v) & 1u;
			const uint32_t b = __ballot_sync(kFull, bit);
			if (lane == v) mine = b;
			if (P.hasReady)
			{
				const uint32_t n = __reduce_add_sync(kFull, bit ? readyCount : 0u);
				if (lane == v) inst = n;
			}
		}
		if (lane < P.viewCount)
		{
			A.visBits[(size_t)lane * words + word] = mine;
			if (mine)
				atomicAdd(&A.chunkCount[(size_t)lane * A.chunks + idx / kChunkItems], (uint32_t)__popc(mine));
			if (P.hasReady && inst)
				atomicAdd(&A.counters[ctrPoolInst(P.poolIndex, lane)], inst);
		}
	}
}

// Exclusive scan of the per-chunk visible counts of one view (one block per view) -> list offset of every chunk.
// Also publishes the list length after this pool (poolEnd), which is the draw count the host reads back.
constexpr uint32_t kScanThreads = 1024;
__global__ void __launch_bounds__(kScanThreads) kScanChunks(const __grid_constant__ CullParams P, const __grid_constant__ CullArgs A)
{
	const uint32_t v = blockIdx.x;
	if (!P.views[v].enabled)
		return;
	__shared__ uint32_t sWarp[kScanThreads / 32];
	__shared__ uint32_t sCarry;
	uint32_t* counts = A.chunkCount + (size_t)v * A.chunks;
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t chunks = (A.counters[A.surCounter] + kChunkItems - 1) / kChunkItems; // chunks that hold survivors
	if (threadIdx.x == 0)
		sCarry = A.baseCounter[v] != kNone ? A.counters[A.baseCounter[v]] : 0;
	__syncthreads();
	for (uint32_t base = 0; base < chunks; base += kScanThreads)
	{
		const uint32_t i = base + threadIdx.x;
		const uint32_t c = i < chunks ? counts[i] : 0;
		uint32_t inc = c;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1)
		{
			uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
			if (lane >= (uint32_t)o) inc += t;
		}
		if (lane == 31)
			sWarp[warp] = inc;
		__syncthreads();
		if (warp == 0)
		{
			uint32_t w = sWarp[lane], winc = w;
			#pragma unroll
			for (int o = 1; o < 32; o <<= 1)
			{
				uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
				if (lane >= (uint32_t)o) winc += t;
			}
			sWarp[lane] = winc - w;
		}
		__syncthreads();
		const uint32_t carry = sCarry;
		const uint32_t exclusive = carry + sWarp[warp] + inc - c;
		if (i < chunks)
			counts[i] = exclusive;
		__syncthreads();
		if (threadIdx.x == kScanThreads - 1)
			sCarry = exclusive + c;
		__syncthreads();
	}
	if (threadIdx.x == 0)
		A.counters[ctrPoolEnd(P.poolIndex, v)] = sCarry;
}

// Compaction + key + sort histograms. Work unit = one chunk (kChunkWords ballot words = 2048 slots) of one view, handled by
// ONE WARP with no block-level synchronisation: each lane owns 2 consecutive words (one 64-bit load), a warp scan of the
// popcounts gives every lane its offset inside the chunk, each lane expands its set bits into a shared-memory list of
// slot offsets, and then the OUTPUT positions are dealt round-robin to the lanes, so every lane gathers and stores on
// every iteration no matter how the visible slots cluster. Units are dealt to the warps of a persistent grid view-fastest,
// so the views' gathers of one region of world matrices run together (L2 reuse). Lists come out in slot order, so the
// stable radix sort breaks ties by slot. The four 8-bit digit histograms of the keys are accumulated in shared memory on
// the way and added to the list's global histograms once per block (this replaces a separate histogram pass over the keys).
constexpr uint32_t kScatterWarps = 8, kScatterThreads = kScatterWarps * 32, kWordsPerLane = kChunkWords / 32;
static_assert(kWordsPerLane == 2, "one 64-bit load per lane");
__global__ void __launch_bounds__(kScatterThreads) kScatter(const __grid_constant__ CullParams P, const __grid_constant__ CullArgs A)
{
	__shared__ uint16_t sList[kScatterWarps][kChunkWords * 32]; // slot offsets inside the chunk, in list order
	extern __shared__ uint32_t sHistDyn[]; // [viewCount][4][256]
	uint32_t (*sHist)[4][256] = reinterpret_cast<uint32_t (*)[4][256]>(sHistDyn);
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (uint32_t i = threadIdx.x; i < P.viewCount * 4 * 256; i += kScatterThreads)
		sHistDyn[i] = 0;
	__syncthreads();
	const uint32_t words = A.tiles * (kCullTile / 32);
	const uint32_t survivors = A.counters[A.surCounter];
	const uint32_t liveWords = ((survivors + kWarpTile - 1) / kWarpTile) * kWarpItems; // ballot words kCull wrote
	const uint32_t chunks = (survivors + kChunkItems - 1) / kChunkItems;
	const uint32_t units = chunks * P.viewCount;
	for (uint32_t u = blockIdx.x * kScatterWarps + warp; u < units; u += gridDim.x * kScatterWarps)
	{
		// chunks are walked from the END of the list: the world matrices kCull wrote last are still in L2 when this kernel
		// starts, the ones it wrote first were evicted long ago either way (list positions come from the scan, not the order)
		const uint32_t v = u % P.viewCount, chunk = chunks - 1 - u / P.viewCount;
		const ViewConst& V = P.views[v];
		if (!V.enabled) // warp-uniform
			continue;
		const uint32_t firstWord = chunk * kChunkWords + lane * kWordsPerLane;
		uint2 w = make_uint2(0u, 0u);
		if (firstWord + kWordsPerLane <= liveWords) // (kCull writes kWarpItems == kWordsPerLane words per warp tile)
			w = *reinterpret_cast<const uint2*>(A.visBits + (size_t)v * words + firstWord);
		const uint32_t sum = __popc(w.x) + __popc(w.y);
		uint32_t inc = sum;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1)
		{
			uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
			if (lane >= (uint32_t)o) inc += t;
		}
		const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
		if (total == 0)
			continue;
		__syncwarp(); // the previous unit's readers are done with this warp's list
		{
			uint32_t pos = inc - sum;
			uint32_t bits = w.x, offset = lane * 64;
			while (bits)
			{
				sList[warp][pos++] = (uint16_t)(offset + __ffs(bits) - 1);
				bits &= bits - 1;
			}
			bits = w.y; offset += 32;
			while (bits)
			{
				sList[warp][pos++] = (uint16_t)(offset + __ffs(bits) - 1);
				bits &= bits - 1;
			}
		}
		__syncwarp();
		const uint32_t base = A.chunkCount[(size_t)v * A.chunks + chunk];
		uint32_t* keys = A.keys + A.segOffset[v];
		uint32_t* pays = A.payloads + A.segOffset[v];
		const float ox = V.cameraOffset[0], oy = V.cameraOffset[1], oz = V.cameraOffset[2];
		const bool sorted = A.histOffset[v] != kNone; // OIT buffers are never sorted (mesh.cpp:273-277): no histogram
		// kGatherBatch independent gathers in flight per lane (the loop is bound by their latency, not by bandwidth;
		// measured on C4: 4 -> 0.098 ms, 8 -> 0.086, 16 -> 0.077, 32 -> 0.103 for kScanChunks + kScatter)
		constexpr uint32_t kGatherBatch = 16;
		for (uint32_t j0 = lane; j0 < total; j0 += 32 * kGatherBatch)
		{
			uint32_t slot[kGatherBatch];
			float4 w2[kGatherBatch];
			#pragma unroll
			for (uint32_t b = 0; b < kGatherBatch; b++)
			{
				const uint32_t j = j0 + 32 * b;
				slot[b] = chunk * kChunkItems + (j < total ? sList[warp][j] : sList[warp][j0]); // (a survivor index)
				w2[b] = A.worldPos[slot[b]]; // (c3.x, c3.y, c3.z, 0): the dense copy of the world matrices' translation
			}
			#pragma unroll
			for (uint32_t b = 0; b < kGatherBatch; b++)
			{
				const uint32_t j = j0 + 32 * b;
				if (j >= total)
					break;
				float key;
				if (P.key2D)
					key = __fadd_rn(w2[b].z, 1.0f); // mesh.cpp:250
				else
					key = lengthSq3(__fadd_rn(w2[b].x, ox), __fadd_rn(w2[b].y, oy), __fadd_rn(w2[b].z, oz)); // mesh.cpp:172,251
				uint32_t k = floatToOrdered(key);
				if (P.descending)
					k = ~k;
				keys[base + j] = k;
				pays[base + j] = (P.poolIndex << 28) | slot[b];
				if (sorted)
				{
					atomicAdd(&sHist[v][0][k & 255u], 1u);
					atomicAdd(&sHist[v][1][(k >> 8) & 255u], 1u);
					atomicAdd(&sHist[v][2][(k >> 16) & 255u], 1u);
					atomicAdd(&sHist[v][3][k >> 24], 1u);
				}
			}
		}
	}
	__syncthreads();
	for (uint32_t i = threadIdx.x; i < P.viewCount * 4 * 256; i += kScatterThreads)
	{
		const uint32_t v = i >> 10;
		const uint32_t c = sHistDyn[i];
		if (c && A.histOffset[v] != kNone)
			atomicAdd(&A.sortHist[A.histOffset[v] + (i & 1023u)], c);
	}
}

// Unit-normal copies of a view's planes for the conservative classifier (see kCull). Scaling a plane by a positive
// factor does not change which side a point is on; the factor is computed in double and its rounding is far inside the
// band. A plane with a zero normal has the same distance d for every finite point: it either never culls (d >= 0 or NaN,
// neutral) or culls every finite entity (d < 0). Anything that cannot be normalised safely forces the exact test.
static void prepareClassifier(ViewConst& V)
{
	const float inf = INFINITY;
	float maxAbsD = 0.0f;
	bool forceExact = false;
	for (uint32_t i = 0; i < 6; i++)
	{
		float* ux = i & 1 ? &V.ux[i >> 1].y : &V.ux[i >> 1].x;
		float* uy = i & 1 ? &V.uy[i >> 1].y : &V.uy[i >> 1].x;
		float* uz = i & 1 ? &V.uz[i >> 1].y : &V.uz[i >> 1].x;
		float* ud = i & 1 ? &V.ud[i >> 1].y : &V.ud[i >> 1].x;
		*ux = *uy = *uz = 0.0f; *ud = inf;
		if (i >= V.planeCount)
			continue;
		const float* pl = V.planes[i];
		const double nx = pl[0], ny = pl[1], nz = pl[2], d = pl[3];
		if (!std::isfinite(nx) || !std::isfinite(ny) || !std::isfinite(nz) || !std::isfinite(d))
		{
			forceExact = true;
			continue;
		}
		const double len = std::sqrt(nx * nx + ny * ny + nz * nz);
		if (len == 0.0)
		{
			if (d < 0.0) *ud = -inf;
			continue;
		}
		const double nux = nx / len, nuy = ny / len, nuz = nz / len, nud = d / len;
		if (len < 1e-30 || !std::isfinite(nud) || std::fabs(nud) > 1e30)
		{
			forceExact = true;
			continue;
		}
		*ux = (float)nux; *uy = (float)nuy; *uz = (float)nuz; *ud = (float)nud;
		maxAbsD = std::max(maxAbsD, std::fabs(*ud));
	}
	V.slack = forceExact ? inf : maxAbsD * kBandD * 1.0001f;
}

// Is the view a box (three pairs of opposite planes with orthonormal normals, e.g. an orthographic cascade)? Then its face
// normals and its extent [lo, hi] along each, in the camera-relative space the planes live in. Planes are expected in
// Frustum(viewProj) order (frustum.hpp:53-60: the pairs are (0,1), (2,3), (4,5)); anything else simply is not recognised
// (no shortcut, same result).
static bool viewBox(const ViewConst& V, double n[3][3], double lo[3], double hi[3])
{
	if (V.planeCount != 6 || !(V.slack < INFINITY))
		return false;
	for (int j = 0; j < 3; j++)
	{
		const double a[3] = { V.ux[j].x, V.uy[j].x, V.uz[j].x }, b[3] = { V.ux[j].y, V.uy[j].y, V.uz[j].y };
		const double da = V.ud[j].x, db = V.ud[j].y;
		double len2 = 0.0;
		for (int k = 0; k < 3; k++)
		{
			if (std::fabs(a[k] + b[k]) > 1e-6)
				return false;
			n[j][k] = a[k]; len2 += a[k] * a[k];
		}
		if (std::fabs(len2 - 1.0) > 1e-5 || !std::isfinite(da) || !std::isfinite(db))
			return false;
		lo[j] = -da; hi[j] = db; // inside: -da <= n . x <= db
		if (!(hi[j] >= lo[j]))
			return false;
	}
	for (int i = 0; i < 3; i++)
		for (int j = i + 1; j < 3; j++)
			if (std::fabs(n[i][0] * n[j][0] + n[i][1] * n[j][1] + n[i][2] * n[j][2]) > 1e-5)
				return false;
	return true;
}

// One bounding description for all box views of the frame that share the first one's orientation (see boxesCulled).
static void prepareBoxGroup(CullParams& P)
{
	P.boxMask = 0; P.boxSlack = 0.0f;
	double axis[3][3] = {}, glo[3] = {}, ghi[3] = {}, slack = 0.0;
	bool groupBroken = false;
	for (uint32_t v = 0; v < P.viewCount; v++)
	{
		double n[3][3], lo[3], hi[3];
		if (!P.views[v].enabled || !viewBox(P.views[v], n, lo, hi))
			continue;
		if (P.boxMask == 0)
		{
			memcpy(axis, n, sizeof(axis)); memcpy(glo, lo, sizeof(glo)); memcpy(ghi, hi, sizeof(ghi));
		}
		else
		{
			double dev = 0.0;
			for (int j = 0; j < 3; j++)
				for (int k = 0; k < 3; k++)
					dev = std::max(dev, std::fabs(n[j][k] - axis[j][k]));
			if (dev > 1e-6)
				continue; // another orientation: tested per plane as usual
			for (int j = 0; j < 3; j++)
			{
				glo[j] = std::min(glo[j], lo[j]); ghi[j] = std::max(ghi[j], hi[j]);
			}
		}
		P.boxMask |= 1u << v;
		slack = std::max(slack, (double)P.views[v].slack);
		for (int j = 0; j < 3; j++)
		{
			// rounded outwards like the union below
			P.boxViewLo[v][j] = (float)(lo[j] - std::fabs(lo[j]) * 1e-5 - 1e-30);
			P.boxViewHi[v][j] = (float)(hi[j] + std::fabs(hi[j]) * 1e-5 + 1e-30);
			if (!std::isfinite(P.boxViewLo[v][j]) || !std::isfinite(P.boxViewHi[v][j]))
				groupBroken = true;
		}
	}
	if (groupBroken)
		P.boxMask = 0;
	if (!P.boxMask)
		return;
	for (int j = 0; j < 3; j++)
	{
		for (int k = 0; k < 3; k++) P.boxAxis[j][k] = (float)axis[j][k];
		// rounded outwards (the float conversion and the kBandD-style slack of the extents themselves)
		P.boxLo[j] = (float)(glo[j] - std::fabs(glo[j]) * 1e-5 - 1e-30);
		P.boxHi[j] = (float)(ghi[j] + std::fabs(ghi[j]) * 1e-5 + 1e-30);
		if (!std::isfinite(P.boxLo[j]) || !std::isfinite(P.boxHi[j]))
		{
			P.boxMask = 0;
			return;
		}
	}
	P.boxSlack = (float)(slack * 1.0001);
}

static ChainArgs chainArgs(const TransformsDev& t)
{
	ChainArgs A;
	A.bound = t.bound; A.parent = t.parent; A.flags = t.flags; A.posSx = t.posSx; A.rho = t.rho;
	A.chainRoot = t.chainRoot; A.rootW = t.rootW; A.record = t.record; A.count = t.occupancy;
	return A;
}

// Prepass spheres of every transform: once per change of transforms, pools or active flags (after launchLink: needs rho)
uint32_t launchChainBounds(Context& c)
{
	auto& t = c.tf;
	if (t.occupancy == 0)
		return 0;
	const ChainArgs A = chainArgs(t);
	cudaMemsetAsync(t.rootW, 0, (size_t)t.occupancy * sizeof(uint32_t), c.stream);
	kChainBounds<<<(t.occupancy + 255) / 256, 256, 0, c.stream>>>(A);
	kChainRecords<<<(t.occupancy + 255) / 256, 256, 0, c.stream>>>(A);
	return 2;
}

// The records alone, from rho and rootW as they stand (after kLinkSlots grew some of them)
uint32_t launchChainRecords(Context& c)
{
	auto& t = c.tf;
	if (t.occupancy == 0)
		return 0;
	kChainRecords<<<(t.occupancy + 255) / 256, 256, 0, c.stream>>>(chainArgs(t));
	return 1;
}

// *dGrew (zeroed by the caller) = 1 when some rho grew. `walk` needs rootW and chainRoot of the current transforms.
uint32_t launchLinkSlots(Context& c, uint32_t pool, const uint32_t* dSlotMap, uint32_t first, uint32_t count, bool walk,
	uint32_t* dGrew)
{
	auto& t = c.tf;
	auto& p = c.pools[pool];
	if (count == 0)
		return 0;
	kLinkSlots<<<(count + 255) / 256, 256, 0, c.stream>>>(dSlotMap, first, count, p.entity, t.entityToSlot, t.entityCap,
		p.tslot, p.radius, t.rho, walk ? 1 : 0, t.bound, t.parent, t.flags, t.rootW, dGrew);
	return 1;
}

static void setKernelAttributes(Context& c)
{
	// 8 resident blocks x 26 KB of shared memory need the large carve-out (function attributes are per device, and one
	// context = one device, so the flag lives in the context)
	if (c.cullAttrsSet)
		return;
	#define GSP_CARVEOUT(V) do { \
		cudaFuncSetAttribute(kCull<V, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); \
		cudaFuncSetAttribute(kCull<V, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); } while (0)
	GSP_CARVEOUT(1); GSP_CARVEOUT(2); GSP_CARVEOUT(3); GSP_CARVEOUT(4); GSP_CARVEOUT(5); GSP_CARVEOUT(6); GSP_CARVEOUT(8); GSP_CARVEOUT(16);
	#undef GSP_CARVEOUT
	c.cullAttrsSet = true;
}

static void commonArgs(Context& c, CullArgs& A)
{
	A.tRot = c.tf.rot; A.tPosSx = c.tf.posSx; A.tSYZ = c.tf.sYZ; A.tParent = c.tf.parent; A.tFlags = c.tf.flags;
	A.tRecord = c.tf.record;
	A.tOccupancy = c.tf.occupancy;
	A.counters = c.dCounters;
	A.tList = c.tf.tList; A.tIndex = c.tf.tIndex; A.tWorld = c.tf.tWorld; A.tCounter = kCtrSurvivorsT;
	static const bool prepassOff = []{ const char* e = getenv("GSP_PREPASS"); return e && !strcmp(e, "0"); }();
	A.prepassCull = prepassOff ? 0u : 1u;
}

// view count -> template instantiation (the view loops are unrolled at compile time: plane constants become direct
// constant-bank operands)
#define GSP_FOR_VIEW_COUNT(N, LAUNCH) do { \
	if ((N) <= 1) { LAUNCH(1); } else if ((N) <= 2) { LAUNCH(2); } else if ((N) <= 3) { LAUNCH(3); } else if ((N) <= 4) { LAUNCH(4); } \
	else if ((N) <= 5) { LAUNCH(5); } else if ((N) <= 6) { LAUNCH(6); } else if ((N) <= 8) { LAUNCH(8); } else { LAUNCH(16); } } while (0)

// Split path, once per frame for all split pools: surviving transforms (for the views any split pool takes part in), their
// list, and their world matrices.
uint32_t launchSplitWorld(Context& c, cudaEvent_t before, cudaEvent_t after)
{
	auto& t = c.tf;
	if (!c.anySplit || t.occupancy == 0)
		return 0;
	CullParams P = {};
	CullArgs A = {};
	bool any = false;
	for (uint32_t v = 0; v < (uint32_t)c.views.size(); v++)
	{
		const gsp_view& gv = c.views[v];
		ViewConst& V = P.views[v];
		V.enabled = 0;
		for (uint32_t p = 0; p < c.poolCount; p++)
			if (c.pools[p].split && c.segOf[v][p] >= 0 && c.participates[v][p])
				V.enabled = 1;
		if (!V.enabled)
			continue;
		any = true;
		memcpy(V.planes, gv.planes, sizeof(V.planes));
		V.planeCount = gv.planeCount;
		prepareClassifier(V);
	}
	if (!any)
		return 0;
	for (int i = 0; i < 3; i++)
		P.cam[i] = c.cameraPos[i];
	P.viewCount = (uint32_t)c.views.size();
	P.occupancy = t.occupancy;
	static const bool boxesOff = []{ const char* e = getenv("GSP_BOXGROUP"); return e && !strcmp(e, "0"); }();
	if (!boxesOff)
		prepareBoxGroup(P);
	commonArgs(c, A);
	A.surBits = t.tBits; A.blockCount = t.tBlockCount; A.bucketCount = t.tBucketCount;
	A.surList = t.tList; A.surTs = t.tList; // the items of the world-only kCull ARE transform slots
	A.surCounter = kCtrSurvivorsT;
	A.visibleView = kNone;
	A.tiles = (t.occupancy + kCullTile - 1) / kCullTile;
	A.chunks = (A.tiles + kChunkTiles - 1) / kChunkTiles;
	setKernelAttributes(c);
	if (before) cudaEventRecord(before, c.stream);
	const uint32_t preBlocks = (t.occupancy + kPreTile - 1) / kPreTile;
	const uint32_t cullBlocks = std::max(1u, std::min(A.tiles, c.smCount * kCullBlocksPerSM));
	CompactArgs K;
	K.bits = t.tBits; K.blockCount = t.tBlockCount; K.bucketCount = t.tBucketCount; K.list = t.tList; K.aux = t.tIndex;
	K.tslot = nullptr; K.counters = c.dCounters; K.counterIndex = kCtrSurvivorsT; K.blocks = preBlocks;
	#define GSP_LAUNCH_WORLD(V) do { \
		kPrepassT<V><<<preBlocks, kPreThreads, 0, c.stream>>>(P, A); \
		kCompactSurvivors<true><<<(preBlocks + kCompactWarps - 1) / kCompactWarps, kCompactWarps * 32, 0, c.stream>>>(K); \
		kCull<V, true><<<cullBlocks, kCullThreads, 0, c.stream>>>(P, A); } while (0)
	GSP_FOR_VIEW_COUNT(P.viewCount, GSP_LAUNCH_WORLD);
	#undef GSP_LAUNCH_WORLD
	if (after) cudaEventRecord(after, c.stream);
	return 3;
}

uint32_t launchCull(Context& c, uint32_t pool, cudaEvent_t afterPrepass, cudaEvent_t afterCull, cudaEvent_t afterScatter)
{
	auto& p = c.pools[pool];
	c.poolLaunched[pool] = false;
	p.visibleValid = false; // only a frame whose main view processed this pool owns its isVisible bytes (mesh.cpp:426,482)
	if (!p.set || p.occupancy == 0)
		return 0;
	CullParams P = {};
	CullArgs A = {};
	const bool isUI = p.renderType == GSP_RT_UI;
	const bool sortedList = isUI || p.renderType == GSP_RT_TRANSLUCENT;
	bool any = false;
	A.visibleView = kNone;
	for (uint32_t v = 0; v < (uint32_t)c.views.size(); v++)
	{
		const gsp_view& gv = c.views[v];
		ViewConst& V = P.views[v];
		int seg = c.segOf[v][pool];
		V.enabled = seg >= 0 && c.participates[v][pool];
		A.segOffset[v] = 0; A.baseCounter[v] = kNone; A.histOffset[v] = kNone;
		if (!V.enabled)
			continue;
		any = true;
		memcpy(V.planes, isUI ? gv.uiPlanes : gv.planes, sizeof(V.planes));
		V.planeCount = isUI ? gv.uiPlaneCount : gv.planeCount;
		prepareClassifier(V);
		memcpy(V.cameraOffset, gv.cameraOffset, sizeof(V.cameraOffset));
		A.segOffset[v] = c.segments[seg].offset;
		A.histOffset[v] = c.segments[seg].sorted ? (uint32_t)seg * 4u * 256u : kNone;
		int prev = c.prevPool[v][pool];
		A.baseCounter[v] = prev >= 0 ? ctrPoolEnd((uint32_t)prev, v) : kNone;
		if (gv.shadowPass < 0)
			A.visibleView = v; // the last main view wins, as repeated prepareMeshes calls would overwrite isVisible
	}
	if (!any)
		return 0;
	for (int i = 0; i < 3; i++)
		P.cam[i] = isUI ? 0.0f : c.cameraPos[i]; // mesh.cpp:435,441
	P.viewCount = (uint32_t)c.views.size();
	P.occupancy = p.occupancy;
	P.poolIndex = pool;
	P.key2D = isUI ? 1 : 0;
	P.descending = sortedList ? 1 : 0;
	P.hasReady = p.hasReady ? 1 : 0;
	static const bool boxesOff = []{ const char* e = getenv("GSP_BOXGROUP"); return e && !strcmp(e, "0"); }();
	if (!boxesOff)
		prepareBoxGroup(P);

	commonArgs(c, A);
	A.aabbA = p.aabbA; A.aabbB = p.aabbB; A.tslot = p.tslot; A.mflags = p.flags; A.ready = p.ready;
	A.surList = p.surList; A.surTs = p.surTs; A.world = p.world; A.worldPos = p.worldPos; A.visible = p.visible;
	A.visBits = p.visBits; A.chunkCount = p.cullStatus;
	A.keys = c.keys[0]; A.payloads = c.payloads[0]; A.sortHist = c.sortHist;
	A.surBits = p.surBits; A.blockCount = p.blockCount; A.bucketCount = p.bucketCount;
	A.surCounter = kCtrSurvivors + pool;
	A.tiles = (p.occupancy + kCullTile - 1) / kCullTile;
	A.chunks = (A.tiles + kChunkTiles - 1) / kChunkTiles;
	p.visibleValid = A.visibleView != kNone;
	setKernelAttributes(c);

	const uint32_t preBlocks = (p.occupancy + kPreTile - 1) / kPreTile;
	// kCull / kClassify are persistent: their warps stride over the survivors (the count only exists on the device)
	const uint32_t cullBlocks = std::max(1u, std::min(A.tiles, c.smCount * kCullBlocksPerSM));
	const uint32_t classifyBlocks = std::max(1u, std::min((p.occupancy + kClassifyThreads - 1) / kClassifyThreads, c.smCount * 8u));
	const bool split = p.split && !isUI && c.anySplit;
	CompactArgs K;
	K.bits = p.surBits; K.blockCount = p.blockCount; K.bucketCount = p.bucketCount; K.list = p.surList; K.aux = p.surTs;
	K.tslot = p.tslot; K.counters = c.dCounters; K.counterIndex = kCtrSurvivors + pool; K.blocks = preBlocks;
	#define GSP_LAUNCH_CULL(V) do { \
		kPrepass<V><<<preBlocks, kPreThreads, 0, c.stream>>>(P, A); \
		kCompactSurvivors<false><<<(preBlocks + kCompactWarps - 1) / kCompactWarps, kCompactWarps * 32, 0, c.stream>>>(K); \
		if (afterPrepass) cudaEventRecord(afterPrepass, c.stream); \
		if (split) kClassify<V><<<classifyBlocks, kClassifyThreads, 0, c.stream>>>(P, A); \
		else kCull<V, false><<<cullBlocks, kCullThreads, 0, c.stream>>>(P, A); } while (0)
	GSP_FOR_VIEW_COUNT(P.viewCount, GSP_LAUNCH_CULL);
	#undef GSP_LAUNCH_CULL
	if (afterCull) cudaEventRecord(afterCull, c.stream);
	if (c.arenaFreePending)
	{
		cudaStreamWaitEvent(c.stream, c.arenaFree, 0); // (exchange.cu: the last frame's runs have left the arenas)
		c.arenaFreePending = false;
	}
	kScanChunks<<<P.viewCount, kScanThreads, 0, c.stream>>>(P, A);
	{
		// persistent grid: one wave of blocks, every warp strides over (chunk, view) units
		const uint32_t units = A.chunks * P.viewCount;
		const uint32_t blocks = std::max(1u, std::min((units + kScatterWarps - 1) / kScatterWarps, c.smCount * 4u));
		const size_t histBytes = (size_t)P.viewCount * 4 * 256 * sizeof(uint32_t);
		if (!c.scatterAttrSet)
		{
			cudaFuncSetAttribute(kScatter, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxViews * 4 * 256 * sizeof(uint32_t));
			c.scatterAttrSet = true;
		}
		kScatter<<<blocks, kScatterThreads, histBytes, c.stream>>>(P, A);
	}
	if (afterScatter) cudaEventRecord(afterScatter, c.stream);
	c.poolLaunched[pool] = true;
	return 5;
}

} // namespace gsp
