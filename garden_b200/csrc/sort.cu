// Segmented one-sweep LSD radix sort of (key, payload) pairs: 8-bit digits, 4 passes over 32-bit keys, stable.
//
// Replaces MeshRenderSystem::sortMeshes (source/system/render/mesh.cpp:265-328): one std::sort per unsorted buffer plus the
// translucent and UI lists. Here every list of every view is one segment and all segments are sorted by the same launches.
// Keys are order-preserving integer images of distanceSq (ascending lists) or their complement (descending lists,
// mesh.hpp:204), payload = pool << 28 | slot. The compaction emits each list in (pool, slot) order and the sort is stable,
// so equal keys keep ascending (pool, slot) order — the canonical tie-break (the reference's order on ties is unspecified).
//
// Algorithm (Adinets & Merrill, "Onesweep"): the 4 digit histograms of every segment are built up front (by kScatter, while
// it writes the keys); each pass then reads a tile once, ranks it in shared memory, resolves the tile's global digit offsets
// with a decoupled look-back over the preceding tiles and scatters. Per element traffic: 4 x (8 B read + 8 B write).
// Look-back status words carry the launch's epoch in their upper half, so they never need clearing: a word written by an
// earlier pass or frame simply reads as "not published yet".
#include "sceneprep_internal.h"
#include <algorithm>

namespace gsp
{

constexpr uint32_t kRadixBits = 8, kRadix = 1u << kRadixBits, kPasses = 4;
constexpr uint32_t kWarps = kSortThreads / 32;
constexpr uint32_t kFlagAggregate = 1u << 30, kFlagInclusive = 2u << 30, kValueMask = (1u << 30) - 1;

struct SortArgs
{
	const SegmentDev* __restrict__ segments;
	const uint32_t* __restrict__ counters; // segment length = counters[countIndex] (kNone -> 0)
	uint32_t* __restrict__ hist;           // [segment][pass][256]
	unsigned long long* __restrict__ status; // [tileBase(segment) + tile][256]: epoch << 32 | flag << 30 | value
	uint32_t* __restrict__ tickets;        // [segment][pass]
	const uint32_t* __restrict__ segTileOffset; // first status tile of each segment
	uint32_t epoch;                        // unique per (frame, pass) launch
	uint32_t segmentCountTotal;            // number of segments
};

__device__ __forceinline__ uint32_t segmentCount(const SortArgs& a, const SegmentDev& s)
{
	return s.countIndex == kNone ? 0u : a.counters[s.countIndex];
}
__device__ __forceinline__ unsigned long long ldRelaxed(const unsigned long long* p)
{
	unsigned long long v;
	asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
	return v;
}
// The status word is the only thing a successor tile reads from this tile, so a relaxed store is enough. (A release
// store would first drain this thread's scattered output stores of the previous tile and delay the publication.)
__device__ __forceinline__ void stRelaxed(unsigned long long* p, unsigned long long v)
{
	asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// Block-wide exclusive scan of one value per thread (kSortThreads == kRadix values).
__device__ __forceinline__ uint32_t blockExclusiveScan(uint32_t v, uint32_t* sWarpTotals /*[kWarps]*/)
{
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint32_t inc = v;
	#pragma unroll
	for (int o = 1; o < 32; o <<= 1)
	{
		uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
		if (lane >= (uint32_t)o) inc += t;
	}
	if (lane == 31)
		sWarpTotals[warp] = inc;
	__syncthreads();
	uint32_t offset = 0;
	#pragma unroll
	for (uint32_t w = 0; w < kWarps; w++)
		if (w < warp) offset += sWarpTotals[w];
	__syncthreads();
	return offset + inc - v;
}

// One step of the peer search: keeps in `peers` the lanes whose digit agrees with mine in the bit `mask`. Four SASS
// instructions (test, vote, and / and-not under the predicate); the plain C++ form compiled to nine.
__device__ __forceinline__ uint32_t ballotPeers(uint32_t peers, uint32_t digit, uint32_t mask)
{
	asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 v, w;\n\t"
		"and.b32 v, %1, %2;\n\tsetp.ne.u32 p, v, 0;\n\t"
		"vote.sync.ballot.b32 v, p, 0xffffffff;\n\t"
		"not.b32 w, v;\n\t"
		"selp.b32 v, v, w, p;\n\t"
		"and.b32 %0, %0, v;\n\t}"
		: "+r"(peers) : "r"(digit), "r"(mask));
	return peers;
}

#ifndef GSP_SORT_BLOCKS_PER_SM
#define GSP_SORT_BLOCKS_PER_SM (kSortItems >= 16 ? 3 : 5)
#endif
constexpr uint32_t kSortBlocksPerSM = GSP_SORT_BLOCKS_PER_SM; // resident blocks the pass is sized for
constexpr uint32_t kLookbackBatch = 4; // predecessor tiles inspected per step (independent loads in flight; 16 measured slower, 8 / 4 / 2 within 2 %)

__global__ void __launch_bounds__(kSortThreads, kSortBlocksPerSM) kSortPass(const __grid_constant__ SortArgs A, uint32_t pass, uint32_t epoch,
	const uint32_t* __restrict__ keysIn, const uint32_t* __restrict__ payIn,
	uint32_t* __restrict__ keysOut, uint32_t* __restrict__ payOut)
{
	__shared__ uint32_t sKeys[kSortTile];
	__shared__ uint32_t sPay[kSortTile];
	__shared__ uint32_t sWarpHist[kWarps][kRadix];
	__shared__ uint32_t sBinStart[kRadix];  // tile-local exclusive start of each digit
	__shared__ int32_t sGlobal[kRadix];     // global position = sGlobal[d] + local index
	__shared__ uint32_t sWarpTotals[kWarps];
	__shared__ uint32_t sSegTileEnd[kMaxViews * kMaxPools]; // inclusive prefix of tiles over the segments
	__shared__ uint32_t sWork[2];           // claimed (segment, tile)

	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t shift = pass * kRadixBits;
	const uint32_t d = threadIdx.x; // the digit this thread owns in the per-digit phases

	// Tiles of ALL segments form one ticket space (segment lengths differ by orders of magnitude between a near cascade and
	// the main view, so per-segment grids would leave most blocks idle). Tickets are claimed in order => within a segment
	// tiles start in order and the look-back never waits on a tile that has not been claimed.
	if (threadIdx.x == 0)
	{
		uint32_t running = 0;
		for (uint32_t i = 0; i < A.segmentCountTotal; i++)
		{
			const SegmentDev sg = A.segments[i];
			const uint32_t c = sg.sorted ? segmentCount(A, sg) : 0u;
			running += (c + kSortTile - 1) / kSortTile;
			sSegTileEnd[i] = running;
		}
	}
	__syncthreads();
	const uint32_t totalTiles = sSegTileEnd[A.segmentCountTotal - 1];

	while (true)
	{
		__syncthreads();
		if (threadIdx.x == 0)
		{
			const uint32_t g = atomicAdd(&A.tickets[pass], 1u);
			uint32_t sgi = 0;
			if (g < totalTiles)
				while (sSegTileEnd[sgi] <= g) sgi++;
			sWork[0] = g < totalTiles ? sgi : kNone;
			sWork[1] = g - (sgi ? sSegTileEnd[sgi - 1] : 0u);
		}
		for (uint32_t i = threadIdx.x; i < kWarps * kRadix; i += kSortThreads)
			(&sWarpHist[0][0])[i] = 0;
		__syncthreads();
		const uint32_t segIndex = sWork[0];
		if (segIndex == kNone)
			break;
		const uint32_t tile = sWork[1];
		const SegmentDev seg = A.segments[segIndex];
		const uint32_t count = segmentCount(A, seg);
		unsigned long long* statusBase = A.status + (size_t)A.segTileOffset[segIndex] * kRadix + d;
		const unsigned long long tag = (unsigned long long)epoch << 32;
		// global exclusive start of digit d in this pass = exclusive scan of the segment histogram
		const uint32_t histD = A.hist[((size_t)segIndex * kPasses + pass) * kRadix + d];
		const uint32_t base = tile * kSortTile;
		const uint32_t n = min(kSortTile, count - base);
		const uint32_t* kin = keysIn + seg.offset + base;
		const uint32_t* pin = payIn + seg.offset + base;

		// ---- load (warp-striped: tile order = warp, item, lane) and rank within the warp, in order ----
		uint32_t key[kSortItems], pay[kSortItems], rank[kSortItems];
		#pragma unroll
		for (uint32_t i = 0; i < kSortItems; i++)
		{
			uint32_t idx = warp * (kSortItems * 32) + i * 32 + lane;
			key[i] = idx < n ? kin[idx] : 0xFFFFFFFFu; // padding ranks after every real key of the tile
			pay[i] = idx < n ? pin[idx] : 0u;
		}
		// lanes holding the same digit ("peers"): eight ballots, one per digit bit (cheaper than match.any here, and all
		// sixteen items' masks are independent, so they pipeline)
		uint32_t peerMask[kSortItems];
		#pragma unroll
		for (uint32_t i = 0; i < kSortItems; i++)
		{
			const uint32_t dg = (key[i] >> shift) & (kRadix - 1);
			uint32_t peers = 0xffffffffu;
			#pragma unroll
			for (uint32_t b = 0; b < kRadixBits; b++)
				peers = ballotPeers(peers, dg, 1u << b);
			peerMask[i] = peers;
		}
		#pragma unroll
		for (uint32_t i = 0; i < kSortItems; i++)
		{
			const uint32_t dg = (key[i] >> shift) & (kRadix - 1);
			const uint32_t peers = peerMask[i];
			const uint32_t leader = __ffs(peers) - 1;
			uint32_t pre = 0;
			if (lane == leader)
			{
				pre = sWarpHist[warp][dg];
				sWarpHist[warp][dg] = pre + __popc(peers);
			}
			pre = __shfl_sync(0xffffffffu, pre, leader);
			rank[i] = pre + __popc(peers & ((1u << lane) - 1u));
			__syncwarp();
		}
		__syncthreads();

		// ---- per digit (thread d owns digit d): warp offsets, tile count, global offset by look-back ----
		uint32_t tileCount = 0;
		#pragma unroll
		for (uint32_t w = 0; w < kWarps; w++)
		{
			uint32_t c = sWarpHist[w][d];
			sWarpHist[w][d] = tileCount;
			tileCount += c;
		}
		// padding keys (digit 255 in every pass) are excluded from what is published to other tiles
		uint32_t realCount = tileCount;
		if (d == kRadix - 1)
			realCount -= kSortTile - n;
		unsigned long long* st = statusBase + (size_t)tile * kRadix;
		stRelaxed(st, tag | (tile == 0 ? kFlagInclusive : kFlagAggregate) | realCount);
		const uint32_t binStart = blockExclusiveScan(tileCount, sWarpTotals);
		const uint32_t digitBase = blockExclusiveScan(histD, sWarpTotals);

		uint32_t exclusive = 0;
		if (tile != 0)
		{
			int32_t t = (int32_t)tile - 1;
			bool done = false;
			while (!done)
			{
				unsigned long long sv[kLookbackBatch];
				#pragma unroll
				for (uint32_t j = 0; j < kLookbackBatch; j++)
				{
					const int32_t idx = t - (int32_t)j;
					sv[j] = idx >= 0 ? ldRelaxed(statusBase + (size_t)idx * kRadix) : (tag | kFlagInclusive);
				}
				#pragma unroll
				for (uint32_t j = 0; j < kLookbackBatch; j++)
				{
					if (!done)
					{
						// published by this launch? (any other epoch is a stale word of an earlier pass or frame)
						while ((sv[j] >> 32) != epoch)
							sv[j] = ldRelaxed(statusBase + (size_t)(t - (int32_t)j) * kRadix);
						const uint32_t word = (uint32_t)sv[j];
						exclusive += word & kValueMask;
						done = (word & kFlagInclusive) != 0;
					}
				}
				t -= (int32_t)kLookbackBatch;
			}
			stRelaxed(st, tag | kFlagInclusive | (exclusive + realCount));
		}
		sBinStart[d] = binStart;
		sGlobal[d] = (int32_t)(digitBase + exclusive) - (int32_t)binStart;
		__syncthreads();

		// ---- scatter into shared memory in digit order, then write runs out ----
		#pragma unroll
		for (uint32_t i = 0; i < kSortItems; i++)
		{
			const uint32_t dg = (key[i] >> shift) & (kRadix - 1);
			const uint32_t local = sBinStart[dg] + sWarpHist[warp][dg] + rank[i];
			sKeys[local] = key[i];
			sPay[local] = pay[i];
		}
		__syncthreads();
		uint32_t* kout = keysOut + seg.offset;
		uint32_t* pout = payOut + seg.offset;
		#pragma unroll
		for (uint32_t u = 0; u < kSortItems; u++)
		{
			const uint32_t j = threadIdx.x + u * kSortThreads;
			if (j < n)
			{
				const uint32_t k = sKeys[j];
				const uint32_t dg = (k >> shift) & (kRadix - 1);
				const uint32_t pos = (uint32_t)(sGlobal[dg] + (int32_t)j);
				kout[pos] = k;
				pout[pos] = sPay[j];
			}
		}
	}
}

uint32_t launchSort(Context& c, cudaEvent_t afterHistogram)
{
	if (afterHistogram) cudaEventRecord(afterHistogram, c.stream); // (the histograms are built by kScatter)
	const uint32_t nseg = (uint32_t)c.segments.size();
	uint32_t totalCapTiles = 0;
	for (auto& sgm : c.segments)
		if (sgm.sorted) totalCapTiles += (sgm.capacity + kSortTile - 1) / kSortTile;
	if (nseg == 0 || totalCapTiles == 0)
		return 0;
	SortArgs A;
	A.segments = c.dSegments; A.counters = c.dCounters; A.hist = c.sortHist; A.status = c.sortStatus;
	A.tickets = c.sortTickets; A.segTileOffset = c.segTileOffset; A.epoch = 0;
	A.segmentCountTotal = nseg;
	// sort passes are persistent (tiles claimed by ticket): 3 resident blocks per SM, split over the segments
	dim3 passGrid(std::min<uint32_t>(totalCapTiles, c.smCount * kSortBlocksPerSM));
	uint32_t launches = 0;
	for (uint32_t pass = 0; pass < kPasses; pass++)
	{
		const uint32_t in = pass & 1, out = in ^ 1;
		if (++c.sortEpoch == 0) ++c.sortEpoch; // 0 is what freshly allocated (zeroed) status memory holds
		kSortPass<<<passGrid, kSortThreads, 0, c.stream>>>(A, pass, c.sortEpoch, c.keys[in], c.payloads[in], c.keys[out], c.payloads[out]);
		launches++;
	}
	return launches; // 4 passes: sorted data ends in buffer 0
}

} // namespace gsp
