// Multi-GPU exchange step: k-way merge of the per-GPU sorted (key, payload) runs once they have been exchanged (exchange.cu).
//
// The reference has no counterpart (one process, one std::sort per list, mesh.cpp:265-328); this is what makes the sharded
// path produce the same draw order as a single sort over all entities: every GPU culls + sorts its contiguous entity
// range, the runs travel over NVLink, and each GPU merges ONE key range of every list. Either the runs were cut by common
// splitters before they travelled (all-to-all: every received element is mine), or every rank received every run
// (all-gather) and kMergeBounds cuts my range out of each (splitters are taken from the longest run, which every rank holds,
// so all ranks agree without further communication). The sub-ranges are then merged two by two by a merge-path tree
// (kTreePartition + kMergeTree). Ties are broken by (rank, payload), i.e. by global entity order, because shards are
// contiguous ranges in rank order and runs are already tie-ordered by payload (stable radix sort of a slot-ordered compaction).
#include "sceneprep_internal.h"
#include <algorithm>

namespace gsp
{

struct MergeArgs
{
	const uint32_t* __restrict__ keys;      // gathered: rank r's block starts at r * rankStride
	const uint32_t* __restrict__ payloads;
	const uint32_t* __restrict__ offsets;   // [ranks][lists] start of (rank, list) inside the rank's block
	const uint32_t* __restrict__ counts;    // [ranks][lists]
	uint32_t* __restrict__ bounds;          // [lists][ranks][2] sub-range [lo, hi) of each run that falls into my key range
	uint32_t* __restrict__ sliceInfo;       // [lists][2] global position of my slice start, slice length
	uint32_t* __restrict__ outKeys;         // my slice of every list, list l at outOffsets[l]
	uint32_t* __restrict__ outPayloads;
	uint8_t* __restrict__ outRanks;
	const uint32_t* __restrict__ outOffsets; // [lists]
	uint32_t rankStride, ranks, lists, myRank;
	uint32_t preSplit; // the runs were cut by common splitters before they travelled (all-to-all): every element is mine
};

// Warp-cooperative bound: all 32 lanes call it with the same arguments. Every round probes 32 evenly spaced positions of the
// remaining range and keeps the 1/33 of it that contains the answer, so a run of millions of keys takes 4-5 dependent
// memory round trips instead of 22 (the searches are pure latency). Returns the first index with a[i] >= key.
__device__ __forceinline__ uint32_t warpBound(const uint32_t* __restrict__ a, uint32_t n, uint32_t key)
{
	const uint32_t lane = threadIdx.x & 31;
	uint32_t lo = 0, hi = n; // the answer lies in [lo, hi]
	while (hi - lo > 32)
	{
		const uint64_t span = hi - lo;
		const uint32_t p = lo + (uint32_t)(((uint64_t)(lane + 1) * span) / 33); // lo < p < hi, increasing with the lane
		const uint32_t v = a[p];
		const uint32_t before = __ballot_sync(0xffffffffu, v < key); // a prefix of the lanes
		const uint32_t t = __popc(before);
		const uint32_t pPrev = __shfl_sync(0xffffffffu, p, t ? t - 1 : 0), pNext = __shfl_sync(0xffffffffu, p, t < 32 ? t : 31);
		if (t) lo = pPrev + 1;
		if (t < 32) hi = pNext;
	}
	const uint32_t i = lo + lane;
	const uint32_t v = i < hi ? a[i] : 0u;
	const uint32_t before = __ballot_sync(0xffffffffu, i < hi && v < key);
	return lo + __popc(before);
}

// One WARP per (list, run): the sub-range of the run inside my key range [splitLo, splitHi).
// Splitter k = key at position k * count / ranks of the longest run (k = 1..ranks-1); range 0 starts at -inf, the last
// ends at +inf. (If every run is empty there is nothing to split.)
__global__ void __launch_bounds__(1024) kMergeBounds(const __grid_constant__ MergeArgs A)
{
	const uint32_t list = blockIdx.x, run = threadIdx.x >> 5, lane = threadIdx.x & 31;
	if (run < A.ranks) // (whole warps)
	{
		// splitter source: the longest run of this list (lowest rank on ties); every rank sees the same counts
		uint32_t src = 0;
		for (uint32_t r = 1; r < A.ranks; r++)
			if (A.counts[r * A.lists + list] > A.counts[src * A.lists + list]) src = r;
		const uint32_t count0 = A.counts[src * A.lists + list];
		const uint32_t* run0 = A.keys + (size_t)src * A.rankStride + A.offsets[src * A.lists + list];
		const uint32_t me = A.myRank;
		const bool hasLo = me > 0 && count0 > 0, hasHi = me + 1 < A.ranks && count0 > 0;
		const uint32_t keyLo = hasLo ? run0[(uint64_t)me * count0 / A.ranks] : 0u;
		const uint32_t keyHi = hasHi ? run0[(uint64_t)(me + 1) * count0 / A.ranks] : 0u;
		const uint32_t n = A.counts[run * A.lists + list];
		const uint32_t* a = A.keys + (size_t)run * A.rankStride + A.offsets[run * A.lists + list];
		// a key equal to a splitter belongs to the range that starts at the splitter
		uint32_t lo = 0u, hi = n;
		if (!A.preSplit)
		{
			lo = hasLo ? warpBound(a, n, keyLo) : 0u;
			hi = hasHi ? warpBound(a, n, keyHi) : n;
		}
		if (hi < lo) hi = lo; // equal splitters
		if (lane == 0)
		{
			A.bounds[(list * A.ranks + run) * 2 + 0] = lo;
			A.bounds[(list * A.ranks + run) * 2 + 1] = hi;
		}
	}
	__syncthreads();
	if (threadIdx.x == 0)
	{
		uint32_t start = 0, length = 0;
		for (uint32_t r = 0; r < A.ranks; r++)
		{
			start += A.bounds[(list * A.ranks + r) * 2 + 0];
			length += A.bounds[(list * A.ranks + r) * 2 + 1] - A.bounds[(list * A.ranks + r) * 2 + 0];
		}
		A.sliceInfo[list * 2 + 0] = A.preSplit ? 0u : start; // (all-to-all: the global start comes from the length exchange)
		A.sliceInfo[list * 2 + 1] = length;
	}
}

// ---- pairwise merge tree -------------------------------------------------------------------------------------------------
// The runs of a list are merged two by two with merge-path partitioning: ceil(log2 ranks) passes, each reading and writing
// every element of my slice once (9 bytes in, 9 out), whatever the rank count. (Ranking every element in every other run
// instead takes ranks - 1 searches per element, which at 8 ranks costs more than the sort that produced the runs.) Level 1
// reads the sub-ranges [lo, hi) of the received runs (the rank is implicit), the later levels read the previous level from
// a scratch buffer; the groups of a list stay back to back in run order at every level, so the two inputs of a merge are
// adjacent and its output covers exactly their union — one region per list, the same in the two scratch buffers and in the
// final output. Ties go to the lower group (lower ranks hold lower global entity indices).
constexpr uint32_t kTreeThreads = 256, kTreeItems = 8, kTreeTile = kTreeThreads * kTreeItems;
// one job per (list, pair of runs) at level 1: every list the layout allows at the largest rank count
constexpr uint32_t kTreeMaxJobs = kMaxViews * kMaxPools * 16;
static_assert(kTreeMaxJobs >= kMaxViews * kMaxPools * ((kMaxRanks + 1) / 2), "the job table must hold every list at kMaxRanks ranks");
// shared arrays skip one word in 33: a thread's outputs are kTreeItems apart from its neighbour's, which would put
// every fourth lane into the same bank
constexpr uint32_t kTreePadded = kTreeTile + kTreeTile / 32, kTreeBlocksPerSM = 4;
__device__ __forceinline__ uint32_t treePad(uint32_t i) { return i + (i >> 5); }

struct TreeArgs
{
	MergeArgs M;
	const uint32_t* __restrict__ srcKeys;   // previous level (levels > 1)
	const uint32_t* __restrict__ srcPays;
	const uint8_t* __restrict__ srcRanks;
	uint32_t* __restrict__ dstKeys;
	uint32_t* __restrict__ dstPays;
	uint8_t* __restrict__ dstRanks;
	uint32_t half;                          // runs per input group: 1, 2, 4 ...
};

// Merge path: how many of the first `diag` outputs of merge(a, b) come from a (a wins ties). All 32 lanes call it with the
// same arguments; 32 probes per round like warpBound.
__device__ __forceinline__ uint32_t warpMergePath(const uint32_t* __restrict__ a, uint32_t na, const uint32_t* __restrict__ b, uint32_t nb,
	uint32_t diag)
{
	const uint32_t lane = threadIdx.x & 31;
	uint32_t lo = diag > nb ? diag - nb : 0u, hi = min(diag, na); // the answer lies in [lo, hi]
	while (hi - lo > 32)
	{
		const uint64_t span = hi - lo;
		const uint32_t p = lo + (uint32_t)(((uint64_t)(lane + 1) * span) / 33); // lo < p < hi
		const uint32_t taken = __ballot_sync(0xffffffffu, a[p] <= b[diag - 1 - p]); // a prefix of the lanes
		const uint32_t t = __popc(taken);
		const uint32_t pPrev = __shfl_sync(0xffffffffu, p, t ? t - 1 : 0), pNext = __shfl_sync(0xffffffffu, p, t < 32 ? t : 31);
		if (t) lo = pPrev + 1;
		if (t < 32) hi = pNext;
	}
	const uint32_t i = lo + lane;
	const uint32_t taken = __ballot_sync(0xffffffffu, i < hi && a[i] <= b[diag - 1 - i]);
	return lo + __popc(taken);
}

// One launch per level cuts the level's merges into tiles: the tiles of every (list, pair) job are numbered through, two
// warps per tile search the two diagonals that bound it, and a 32-byte record tells kMergeTree all it needs — the merge
// kernel itself then has no dependent global searches left, only streaming loads and stores.
//   record = { dst, na, nb, rankA | rankB << 8, srcA, 0, srcB, 0 }   (element indices into the level's key array)
constexpr uint32_t kTreeRecordWords = 8, kPartitionTilesPerBlock = kTreeThreads / 64;
template<bool kFirst>
__global__ void __launch_bounds__(kTreeThreads) kTreePartition(const __grid_constant__ TreeArgs T, uint32_t* __restrict__ records /* [0] = tiles, records from word 8 */)
{
	__shared__ uint32_t sTileStart[kTreeMaxJobs + 1];
	__shared__ uint32_t sCut[kTreeThreads / 32];
	const MergeArgs& A = T.M;
	const uint32_t ranks = A.ranks, half = T.half, pairs = (ranks + 2 * half - 1) / (2 * half), jobs = A.lists * pairs;
	const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

	// tiles of every job (list, pair), then their running sum
	for (uint32_t job = threadIdx.x; job < jobs; job += kTreeThreads)
	{
		const uint32_t list = job / pairs, a0 = (job % pairs) * 2 * half, a2 = min(a0 + 2 * half, ranks);
		uint32_t n = 0;
		for (uint32_t r = a0; r < a2; r++)
			n += A.bounds[(list * ranks + r) * 2 + 1] - A.bounds[(list * ranks + r) * 2 + 0];
		sTileStart[job + 1] = (n + kTreeTile - 1) / kTreeTile;
	}
	if (threadIdx.x == 0)
		sTileStart[0] = 0;
	__syncthreads();
	if (warp == 0)
	{
		uint32_t running = 0;
		for (uint32_t base = 0; base < jobs; base += 32)
		{
			uint32_t v = base + lane < jobs ? sTileStart[base + lane + 1] : 0u;
			#pragma unroll
			for (uint32_t o = 1; o < 32; o <<= 1)
			{
				const uint32_t up = __shfl_up_sync(0xffffffffu, v, o);
				if (lane >= o) v += up;
			}
			if (base + lane < jobs)
				sTileStart[base + lane + 1] = running + v;
			running += __shfl_sync(0xffffffffu, v, 31);
		}
	}
	__syncthreads();
	const uint32_t tiles = sTileStart[jobs];
	if (blockIdx.x == 0 && threadIdx.x == 0)
		records[0] = tiles;

	const uint32_t tile = blockIdx.x * kPartitionTilesPerBlock + (warp >> 1);
	const bool live = tile < tiles; // (uniform per warp pair; the barrier below is reached by everyone)
	uint32_t region = 0, nA = 0, nB = 0, a0 = 0, a1 = 0, d0 = 0, d1 = 0;
	size_t baseA = 0, baseB = 0;
	if (live)
	{
		uint32_t job = 0;
		{
			uint32_t lo = 0, hi = jobs; // first job whose tiles end beyond `tile`
			while (lo < hi)
			{
				const uint32_t mid = (lo + hi) >> 1;
				if (sTileStart[mid + 1] <= tile) lo = mid + 1; else hi = mid;
			}
			job = lo;
		}
		const uint32_t list = job / pairs;
		a0 = (job % pairs) * 2 * half; a1 = min(a0 + half, ranks);
		const uint32_t a2 = min(a0 + 2 * half, ranks);
		uint32_t before = 0;
		{
			const uint32_t n = lane < ranks ? A.bounds[(list * ranks + lane) * 2 + 1] - A.bounds[(list * ranks + lane) * 2 + 0] : 0u;
			before = lane < a0 ? n : 0u; nA = lane >= a0 && lane < a1 ? n : 0u; nB = lane >= a1 && lane < a2 ? n : 0u;
			#pragma unroll
			for (int o = 16; o > 0; o >>= 1)
			{
				before += __shfl_xor_sync(0xffffffffu, before, o);
				nA += __shfl_xor_sync(0xffffffffu, nA, o);
				nB += __shfl_xor_sync(0xffffffffu, nB, o);
			}
		}
		region = A.outOffsets[list] + before;
		const uint32_t* keys;
		if (kFirst)
		{
			keys = A.keys;
			baseA = (size_t)a0 * A.rankStride + A.offsets[a0 * A.lists + list] + A.bounds[(list * ranks + a0) * 2 + 0];
			baseB = baseA;
			if (a1 < a2)
				baseB = (size_t)a1 * A.rankStride + A.offsets[a1 * A.lists + list] + A.bounds[(list * ranks + a1) * 2 + 0];
		}
		else
		{
			keys = T.srcKeys;
			baseA = region; baseB = (size_t)region + nA;
		}
		d0 = (tile - sTileStart[job]) * kTreeTile; d1 = min(d0 + kTreeTile, nA + nB);
		const uint32_t cut = warpMergePath(keys + baseA, nA, keys + baseB, nB, (warp & 1) ? d1 : d0);
		if (lane == 0)
			sCut[warp] = cut;
	}
	__syncthreads();
	if (live && !(warp & 1) && lane == 0)
	{
		const uint32_t i0 = sCut[warp], i1 = sCut[warp + 1], j0 = d0 - i0;
		const size_t srcA = baseA + i0, srcB = baseB + j0;
		uint4* rec = (uint4*)(records + kTreeRecordWords * (1 + (size_t)tile));
		rec[0] = make_uint4(region + d0, i1 - i0, (d1 - i1) - j0, a0 | a1 << 8);
		rec[1] = make_uint4((uint32_t)srcA, 0u, (uint32_t)srcB, 0u);
	}
}

template<bool kFirst>
__global__ void __launch_bounds__(kTreeThreads, kTreeBlocksPerSM) kMergeTree(const __grid_constant__ TreeArgs T, const uint32_t* __restrict__ records)
{
	__shared__ uint32_t sKeys[kTreePadded], sPays[kTreePadded];
	__shared__ uint16_t sSrc[kTreePadded];
	__shared__ uint8_t sRanks[kTreePadded];
	const uint32_t* __restrict__ keys = kFirst ? T.M.keys : T.srcKeys;
	const uint32_t* __restrict__ pays = kFirst ? T.M.payloads : T.srcPays;
	const uint32_t tiles = records[0];
	// padded positions of what this thread touches: o = threadIdx.x + u * kTreeThreads -> oBase + u * (kTreeThreads + kTreeThreads / 32),
	// d + u = threadIdx.x * kTreeItems + u -> dBase + u   (kTreeItems divides 32)
	const uint32_t oBase = treePad(threadIdx.x), dBase = threadIdx.x * kTreeItems + (threadIdx.x * kTreeItems >> 5);
	constexpr uint32_t oStep = kTreeThreads + kTreeThreads / 32;
	uint4 r0 = make_uint4(0, 0, 0, 0), r1 = r0;
	if (blockIdx.x < tiles)
	{
		r0 = ((const uint4*)(records + kTreeRecordWords * (1 + (size_t)blockIdx.x)))[0];
		r1 = ((const uint4*)(records + kTreeRecordWords * (1 + (size_t)blockIdx.x)))[1];
	}
	for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x)
	{
		const uint32_t dst = r0.x, na = r0.y, nb = r0.z, n = na + nb, rankA = r0.w & 255u, rankB = r0.w >> 8;
		// 32-bit element indices relative to the key array (the launcher refuses layouts beyond 2^32 elements); b's index is
		// biased by -na so that position o of the staged pair reads index (o < na ? srcA : srcB) + o
		const uint32_t srcA = r1.x, srcB = r1.z - na;
		// the next tile's record travels while this one is merged
		if (tile + gridDim.x < tiles)
		{
			r0 = ((const uint4*)(records + kTreeRecordWords * (1 + (size_t)tile + gridDim.x)))[0];
			r1 = ((const uint4*)(records + kTreeRecordWords * (1 + (size_t)tile + gridDim.x)))[1];
		}
		// stage both ranges, [a | b] (keys, payloads, source ranks): coalesced, every load of the thread in flight at once
		{
			uint32_t k[kTreeItems], q[kTreeItems], r[kTreeItems];
			#pragma unroll
			for (uint32_t u = 0; u < kTreeItems; u++)
			{
				const uint32_t o = threadIdx.x + u * kTreeThreads;
				if (o < n)
				{
					const bool fromB = o >= na;
					const uint32_t g = (fromB ? srcB : srcA) + o;
					k[u] = keys[g];
					q[u] = pays[g];
					r[u] = kFirst ? (fromB ? rankB : rankA) : (uint32_t)T.srcRanks[g];
				}
			}
			#pragma unroll
			for (uint32_t u = 0; u < kTreeItems; u++)
			{
				const uint32_t o = threadIdx.x + u * kTreeThreads;
				if (o < n)
				{
					sKeys[oBase + u * oStep] = k[u];
					sPays[oBase + u * oStep] = q[u];
					sRanks[oBase + u * oStep] = (uint8_t)r[u];
				}
			}
		}
		__syncthreads();
		{
			// my kTreeItems outputs start at diagonal d of the staged pair
			const uint32_t d = min(threadIdx.x * kTreeItems, n);
			uint32_t lo = d > nb ? d - nb : 0u, hi = min(d, na);
			while (lo < hi)
			{
				const uint32_t mid = (lo + hi) >> 1;
				if (sKeys[treePad(mid)] <= sKeys[treePad(na + (d - 1 - mid))]) lo = mid + 1; else hi = mid;
			}
			uint32_t ai = lo, bi = na + (d - lo); // positions in the staged array
			bool hasA = ai < na, hasB = bi < n;
			uint32_t ka = hasA ? sKeys[treePad(ai)] : 0u, kb = hasB ? sKeys[treePad(bi)] : 0u;
			// (no divergent branches: one shared load per step whichever side advances)
			#pragma unroll
			for (uint32_t u = 0; u < kTreeItems; u++)
			{
				const bool takeA = !hasB || (hasA && ka <= kb);
				const uint32_t taken = takeA ? ai : bi, next = taken + 1;
				if (d + u < n)
					sSrc[dBase + u] = (uint16_t)taken;
				const bool has = next < (takeA ? na : n);
				const uint32_t v = has ? sKeys[treePad(next)] : 0u;
				ai = takeA ? next : ai; bi = takeA ? bi : next;
				ka = takeA ? v : ka; kb = takeA ? kb : v;
				hasA = takeA ? has : hasA; hasB = takeA ? hasB : has;
			}
		}
		__syncthreads();
		#pragma unroll
		for (uint32_t u = 0; u < kTreeItems; u++)
		{
			const uint32_t o = threadIdx.x + u * kTreeThreads;
			if (o < n)
			{
				const uint32_t src = treePad(sSrc[oBase + u * oStep]);
				T.dstKeys[dst + o] = sKeys[src];
				T.dstPays[dst + o] = sPays[src];
				T.dstRanks[dst + o] = sRanks[src];
			}
		}
		__syncthreads(); // the next tile reuses the shared arrays
	}
}

// scratch words of the tree for an output of outCapacity elements: 2 x (keys | payloads | ranks), then the tile records
static inline size_t mergeTreeDataWords(uint32_t outCapacity)
{
	return (4ull * outCapacity + 2ull * ((outCapacity + 3ull) / 4ull) + 3ull) & ~3ull; // (records are read as uint4)
}
static inline size_t mergeTreeScratchWords(uint32_t outCapacity)
{
	return mergeTreeDataWords(outCapacity) + kTreeRecordWords * (2ull + outCapacity / kTreeTile + kTreeMaxJobs);
}

uint32_t launchMergeTree(cudaStream_t stream, const MergeArgs& A, uint32_t outCapacity, uint32_t* scratch, uint32_t smCount)
{
	if (A.lists == 0 || A.ranks == 0)
		return 0;
	kMergeBounds<<<A.lists, 32 * A.ranks, 0, stream>>>(A);
	uint32_t levels = 1;
	while ((1u << levels) < A.ranks) levels++;
	uint32_t* tmpK[2] = { scratch, scratch + 2ull * outCapacity };
	uint32_t* tmpP[2] = { scratch + outCapacity, scratch + 3ull * outCapacity };
	uint8_t* tmpR[2] = { (uint8_t*)(scratch + 4ull * outCapacity), (uint8_t*)(scratch + 4ull * outCapacity + (outCapacity + 3ull) / 4ull) };
	uint32_t* records = scratch + mergeTreeDataWords(outCapacity);
	const uint32_t worstTiles = outCapacity / kTreeTile + A.lists * ((A.ranks + 1) / 2) + 1;
	const uint32_t blocks = std::max(1u, std::min(worstTiles, smCount * kTreeBlocksPerSM));
	const uint32_t partitionBlocks = (worstTiles + kPartitionTilesPerBlock - 1) / kPartitionTilesPerBlock;
	for (uint32_t lv = 1; lv <= levels; lv++)
	{
		TreeArgs T;
		T.M = A; T.half = 1u << (lv - 1);
		T.srcKeys = tmpK[(lv - 1) & 1]; T.srcPays = tmpP[(lv - 1) & 1]; T.srcRanks = tmpR[(lv - 1) & 1];
		const bool last = lv == levels;
		T.dstKeys = last ? A.outKeys : tmpK[lv & 1]; T.dstPays = last ? A.outPayloads : tmpP[lv & 1]; T.dstRanks = last ? A.outRanks : tmpR[lv & 1];
		if (lv == 1)
		{
			kTreePartition<true><<<partitionBlocks, kTreeThreads, 0, stream>>>(T, records);
			kMergeTree<true><<<blocks, kTreeThreads, 0, stream>>>(T, records);
		}
		else
		{
			kTreePartition<false><<<partitionBlocks, kTreeThreads, 0, stream>>>(T, records);
			kMergeTree<false><<<blocks, kTreeThreads, 0, stream>>>(T, records);
		}
	}
	return 1 + 2 * levels;
}


// ---- host-synchronisation-free exchange ---------------------------------------------------------------------------------
// The per-list lengths only exist on the device when the frame has just been enqueued, so the whole exchange is laid out
// around a fixed-capacity BLOCK per rank that carries its own description:
//   words [0, kExHeaderWords): header = { kExMagic, lists, total, capacity, overflow, 0, 0, 0, count[0 .. lists) }
//   words [H, H + capacity): keys of all lists back to back;   words [H + capacity, H + 2 * capacity): payloads
// One all-gather of equal-sized blocks moves everything; kMergePlan then derives offsets / totals from the gathered
// headers on the device. A block whose lists do not fit its capacity is flagged (and carries no elements): the host finds
// out from the plan flags one frame later, grows the capacity and repeats that frame.
struct ExportArgs
{
	const SegmentDev* __restrict__ segments;
	const uint32_t* __restrict__ counters;
	const uint32_t* __restrict__ keys;
	const uint32_t* __restrict__ payloads;
	uint32_t* __restrict__ block;
	uint32_t lists, capacity;
};

__global__ void __launch_bounds__(256) kExportPacked(const __grid_constant__ ExportArgs A)
{
	__shared__ uint32_t sCount[kExMaxLists], sStart[kExMaxLists], sFrom[kExMaxLists];
	__shared__ uint32_t sTotal;
	if (threadIdx.x == 0)
	{
		uint32_t running = 0;
		for (uint32_t l = 0; l < A.lists; l++)
		{
			const SegmentDev sg = A.segments[l];
			const uint32_t c = sg.countIndex == kNone ? 0u : A.counters[sg.countIndex];
			sCount[l] = c; sStart[l] = running; sFrom[l] = sg.offset;
			running += c;
		}
		sTotal = running;
	}
	__syncthreads();
	const bool overflow = sTotal > A.capacity;
	if (blockIdx.x == 0)
	{
		for (uint32_t i = threadIdx.x; i < kExHeaderWords; i += blockDim.x)
		{
			uint32_t w = 0;
			if (i == 0) w = kExMagic;
			else if (i == 1) w = A.lists;
			else if (i == 2) w = sTotal;
			else if (i == 3) w = A.capacity;
			else if (i == 4) w = overflow ? 1u : 0u;
			else if (i >= kExHeaderFixed && i < kExHeaderFixed + A.lists) w = overflow ? 0u : sCount[i - kExHeaderFixed];
			A.block[i] = w;
		}
	}
	if (overflow)
		return;
	uint32_t* dk = A.block + kExHeaderWords;
	uint32_t* dp = dk + A.capacity;
	for (uint32_t l = 0; l < A.lists; l++)
	{
		const uint32_t n = sCount[l], from = sFrom[l], to = sStart[l];
		// 4 independent elements in flight per thread and array
		const uint32_t stride = gridDim.x * blockDim.x;
		for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += 4 * stride)
		{
			uint32_t k[4], q[4];
			#pragma unroll
			for (uint32_t u = 0; u < 4; u++)
				if (i + u * stride < n)
				{
					k[u] = A.keys[from + i + u * stride];
					q[u] = A.payloads[from + i + u * stride];
				}
			#pragma unroll
			for (uint32_t u = 0; u < 4; u++)
				if (i + u * stride < n)
				{
					dk[to + i + u * stride] = k[u];
					dp[to + i + u * stride] = q[u];
				}
		}
	}
}

uint32_t launchExportPacked(Context& c, uint32_t* dBlock, uint32_t capacity)
{
	ExportArgs A;
	A.segments = c.dSegments; A.counters = c.dCounters; A.keys = c.keys[0]; A.payloads = c.payloads[0];
	A.block = dBlock; A.lists = (uint32_t)c.segments.size(); A.capacity = capacity;
	kExportPacked<<<c.smCount * 4, 256, 0, c.stream>>>(A);
	return 1;
}

// One block: offsets / counts / output offsets of the merge from the gathered headers; flags for the host.
// plan layout (uint32 words): offsets[ranks*lists] | counts[ranks*lists] | outOffsets[lists] | bounds[lists*ranks*2] | flags[8]
//   flags = { error bits (1 = a rank overflowed its block, 2 = bad header, 4 = merged lists exceed outCapacity),
//             merged total, largest per-rank total (what the block capacity must hold), 0... }
__global__ void kMergePlan(const uint32_t* __restrict__ gathered, uint32_t blockWords, uint32_t ranks, uint32_t lists,
	uint32_t outCapacity, uint32_t* __restrict__ plan)
{
	uint32_t* offsets = plan;
	uint32_t* counts = plan + ranks * lists;
	uint32_t* outOffsets = counts + ranks * lists;
	uint32_t* flags = outOffsets + lists + lists * ranks * 2;
	__shared__ uint32_t sError, sMaxTotal;
	if (threadIdx.x == 0) { sError = 0; sMaxTotal = 0; }
	__syncthreads();
	if (threadIdx.x < ranks)
	{
		const uint32_t* h = gathered + (size_t)threadIdx.x * blockWords;
		uint32_t e = 0;
		if (h[0] != kExMagic || h[1] != lists) e |= 2u;
		if (h[4]) e |= 1u;
		if (e) atomicOr(&sError, e);
		atomicMax(&sMaxTotal, h[2]);
	}
	__syncthreads();
	const bool bad = sError != 0;
	if (threadIdx.x < ranks)
	{
		const uint32_t r = threadIdx.x;
		const uint32_t* h = gathered + (size_t)r * blockWords + kExHeaderFixed;
		uint32_t running = 0;
		for (uint32_t l = 0; l < lists; l++)
		{
			const uint32_t c = bad ? 0u : h[l];
			offsets[r * lists + l] = running;
			counts[r * lists + l] = c;
			running += c;
		}
	}
	__syncthreads();
	if (threadIdx.x == 0)
	{
		uint64_t running = 0;
		for (uint32_t l = 0; l < lists; l++)
		{
			outOffsets[l] = (uint32_t)running;
			for (uint32_t r = 0; r < ranks; r++)
				running += counts[r * lists + l];
		}
		uint32_t e = sError;
		if (running > outCapacity)
		{
			// nothing may be written: drop every run (kMergeBounds and the tree then see empty lists)
			e |= 4u;
			for (uint32_t i = 0; i < ranks * lists; i++)
				counts[i] = 0;
		}
		flags[0] = e; flags[1] = (uint32_t)running; flags[2] = sMaxTotal;
		flags[3] = 0; flags[4] = 0; flags[5] = 0; flags[6] = 0; flags[7] = 0;
	}
}

} // namespace gsp

using namespace gsp;

extern "C" uint32_t gsp_exchange_block_words(uint32_t capacityElems)
{
	return kExHeaderWords + 2u * capacityElems;
}

extern "C" uint32_t gsp_merge_plan_words(uint32_t ranks, uint32_t lists)
{
	return 2u * ranks * lists + lists + 2u * lists * ranks + 8u;
}

namespace gsp
{
// plan + bounds + merge of `ranks` packed blocks (block r at r * (kExHeaderWords + 2 * capacityElems) words).
// Preconditions: lists * ceil(ranks / 2) <= kTreeMaxJobs, exchangeBlocksIndexable(capacityElems, ranks).
uint32_t launchMergePacked(cudaStream_t stream, uint32_t ranks, uint32_t myRank, uint32_t lists, uint32_t capacityElems,
	const uint32_t* dGathered, uint32_t* dPlan, uint32_t* dSliceInfo, uint32_t* dOutKeys, uint32_t* dOutPays, uint8_t* dOutRanks,
	uint32_t outCapacity, bool preSplit, uint32_t* dTreeScratch, uint32_t smCount)
{
	const uint32_t blockWords = kExHeaderWords + 2u * capacityElems;
	kMergePlan<<<1, 32, 0, stream>>>(dGathered, blockWords, ranks, lists, outCapacity, dPlan);
	MergeArgs A;
	A.keys = dGathered + kExHeaderWords; A.payloads = dGathered + kExHeaderWords + capacityElems;
	A.offsets = dPlan; A.counts = dPlan + ranks * lists;
	A.outOffsets = dPlan + 2 * ranks * lists; A.bounds = dPlan + 2 * ranks * lists + lists;
	A.sliceInfo = dSliceInfo; A.outKeys = dOutKeys; A.outPayloads = dOutPays; A.outRanks = dOutRanks;
	A.rankStride = blockWords; A.ranks = ranks; A.lists = lists; A.myRank = myRank; A.preSplit = preSplit ? 1u : 0u;
	return 1 + launchMergeTree(stream, A, outCapacity, dTreeScratch, smCount);
}

// ---- all-to-all protocol: common splitters from samples, one sub-block per destination --------------------------------------
constexpr uint32_t kSamples = 64, kSampleWords = kSamples + 1; // (exchange.cu: kExSamples)

// samples[list][k] = key at position (2k + 1) * count / (2 * kSamples) of my sorted run, samples[list][kSamples] = count
__global__ void kSampleRuns(const SegmentDev* __restrict__ segments, const uint32_t* __restrict__ counters,
	const uint32_t* __restrict__ keys, uint32_t lists, uint32_t* __restrict__ samples)
{
	const uint32_t l = blockIdx.x, k = threadIdx.x;
	if (l >= lists || k > kSamples)
		return;
	const SegmentDev sg = segments[l];
	const uint32_t c = sg.countIndex == kNone ? 0u : counters[sg.countIndex];
	uint32_t v = c;
	if (k < kSamples)
		v = c ? keys[sg.offset + (uint32_t)(((uint64_t)(2 * k + 1) * c) / (2 * kSamples))] : 0xFFFFFFFFu;
	samples[l * kSampleWords + k] = v;
}

// One block per list, one warp per splitter j = 1 .. ranks-1; lane r looks after rank r's samples.
// Splitter j = the smallest key x whose weighted rank  W(x) = sum_r count_r * #(samples of r <= x)  reaches j/ranks of the
// total weight (integer arithmetic, identical on every rank). Then the position of the splitter in MY run: bounds[list][j].
struct SplitArgs
{
	const SegmentDev* __restrict__ segments;
	const uint32_t* __restrict__ counters;
	const uint32_t* __restrict__ keys;
	const uint32_t* __restrict__ gathered; // [ranks][lists][kSampleWords]
	const uint32_t* __restrict__ mine;     // [lists][kSampleWords]: my own samples (their last word = my run length)
	uint32_t* __restrict__ splitters;      // [lists][ranks - 1], then bounds [lists][ranks + 1]
	uint32_t lists, ranks;
};
__global__ void __launch_bounds__(1024) kSplitRuns(const __grid_constant__ SplitArgs A)
{
	const uint32_t l = blockIdx.x, j = (threadIdx.x >> 5) + 1, lane = threadIdx.x & 31;
	uint32_t* bounds = A.splitters + A.lists * (A.ranks - 1) + l * (A.ranks + 1);
	const SegmentDev sg = A.segments[l];
	// (the frame counters may already belong to the NEXT frame when this runs on the exchange stream: the length travels
	// with the samples)
	const uint32_t myCount = A.mine[l * kSampleWords + kSamples];
	if (threadIdx.x == 0)
	{
		bounds[0] = 0; bounds[A.ranks] = myCount;
	}
	// every rank's samples of this list into shared memory (the value search below probes them ~200 times per lane)
	__shared__ uint32_t sSamples[kMaxRanks][kSampleWords];
	for (uint32_t i = threadIdx.x; i < A.ranks * kSampleWords; i += blockDim.x)
		sSamples[i / kSampleWords][i % kSampleWords] = A.gathered[((size_t)(i / kSampleWords) * A.lists + l) * kSampleWords + i % kSampleWords];
	__syncthreads();
	if (j >= A.ranks)
		return; // (whole warps)
	const uint32_t* mine = lane < A.ranks ? sSamples[lane] : nullptr;
	const unsigned long long weight = mine ? mine[kSamples] : 0ull;
	unsigned long long totalWeight = 0;
	{
		// exact 64-bit sum over the lanes
		unsigned long long w = weight;
		#pragma unroll
		for (int o = 16; o > 0; o >>= 1)
			w += __shfl_xor_sync(0xffffffffu, w, o);
		totalWeight = w * kSamples;
	}
	const unsigned long long target = (totalWeight * j + A.ranks - 1) / A.ranks;
	// binary search on the key value: smallest x with W(x) >= target  (W is monotone in x, W(0xFFFFFFFF) = totalWeight)
	uint32_t lo = 0, hi = 0xFFFFFFFFu;
	while (lo < hi)
	{
		const uint32_t mid = lo + ((hi - lo) >> 1);
		uint32_t cnt = 0;
		if (mine && weight)
		{
			uint32_t a = 0, b = kSamples; // #samples <= mid
			while (a < b)
			{
				const uint32_t m = (a + b) >> 1;
				if (mine[m] <= mid) a = m + 1; else b = m;
			}
			cnt = a;
		}
		unsigned long long w = weight * cnt;
		#pragma unroll
		for (int o = 16; o > 0; o >>= 1)
			w += __shfl_xor_sync(0xffffffffu, w, o);
		if (w >= target) hi = mid; else lo = mid + 1;
	}
	const uint32_t splitter = totalWeight ? lo : 0xFFFFFFFFu;
	const uint32_t pos = warpBound(A.keys + sg.offset, myCount, splitter); // keys equal to a splitter start the next range
	if (lane == 0)
	{
		A.splitters[l * (A.ranks - 1) + (j - 1)] = splitter;
		bounds[j] = pos;
	}
}

// Packs my runs into `ranks` sub-blocks (block d = what rank d merges), each laid out like kExportPacked's block.
struct PackArgs
{
	const SegmentDev* __restrict__ segments;
	const uint32_t* __restrict__ keys;
	const uint32_t* __restrict__ payloads;
	const uint32_t* __restrict__ bounds; // [lists][ranks + 1]
	uint32_t* __restrict__ blocks;       // [ranks][kExHeaderWords + 2 * capacity]
	uint32_t lists, ranks, capacity;
};
__global__ void __launch_bounds__(256) kPackByDestination(const __grid_constant__ PackArgs A)
{
	__shared__ uint32_t sBound[kMaxRanks + 1];
	__shared__ uint32_t sTotal[kMaxRanks], sBefore[kMaxRanks]; // per destination: all lists / the lists before this one
	const size_t blockWords = kExHeaderWords + 2ull * A.capacity;
	if (threadIdx.x < A.ranks)
	{
		uint32_t total = 0;
		for (uint32_t l = 0; l < A.lists; l++)
			total += A.bounds[l * (A.ranks + 1) + threadIdx.x + 1] - A.bounds[l * (A.ranks + 1) + threadIdx.x];
		sTotal[threadIdx.x] = total;
	}
	__syncthreads();
	if (blockIdx.x == 0)
	{
		// headers: { magic, lists, total, capacity, overflow, 0, 0, 0, count[lists], before[lists] }
		for (uint32_t d = 0; d < A.ranks; d++)
		{
			const bool overflow = sTotal[d] > A.capacity;
			uint32_t* h = A.blocks + d * blockWords;
			for (uint32_t i = threadIdx.x; i < kExHeaderWords; i += blockDim.x)
			{
				uint32_t w = 0;
				if (i == 0) w = kExMagic;
				else if (i == 1) w = A.lists;
				else if (i == 2) w = sTotal[d];
				else if (i == 3) w = A.capacity;
				else if (i == 4) w = overflow ? 1u : 0u;
				else if (i >= kExHeaderFixed && i < kExHeaderFixed + A.lists && !overflow)
					w = A.bounds[(i - kExHeaderFixed) * (A.ranks + 1) + d + 1] - A.bounds[(i - kExHeaderFixed) * (A.ranks + 1) + d];
				else if (i >= kExHeaderFixed + A.lists && i < kExHeaderFixed + 2 * A.lists)
					w = A.bounds[(i - kExHeaderFixed - A.lists) * (A.ranks + 1) + d]; // elements of my run BEFORE d's key range
				h[i] = w;
			}
		}
	}
	if (threadIdx.x < A.ranks)
		sBefore[threadIdx.x] = 0;
	for (uint32_t l = 0; l < A.lists; l++)
	{
		__syncthreads();
		if (threadIdx.x <= A.ranks)
			sBound[threadIdx.x] = A.bounds[l * (A.ranks + 1) + threadIdx.x];
		__syncthreads();
		const uint32_t n = sBound[A.ranks], from = A.segments[l].offset;
		const uint32_t stride = gridDim.x * blockDim.x;
		for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
		{
			uint32_t d = 0;
			while (d + 1 < A.ranks && i >= sBound[d + 1]) d++;
			if (sTotal[d] > A.capacity)
				continue; // that block overflowed: it carries no elements
			uint32_t* dk = A.blocks + d * blockWords + kExHeaderWords;
			const uint32_t at = sBefore[d] + (i - sBound[d]);
			dk[at] = A.keys[from + i];
			dk[A.capacity + at] = A.payloads[from + i];
		}
		__syncthreads();
		if (threadIdx.x < A.ranks)
			sBefore[threadIdx.x] += sBound[threadIdx.x + 1] - sBound[threadIdx.x];
	}
}

// Where my slice of every list starts in the merged list: the elements every rank holds below my key range. Each source
// wrote that number into the header of the sub-block it sent me, so no further exchange is needed.
__global__ void kSliceStarts(uint32_t ranks, uint32_t lists, const uint32_t* __restrict__ received, size_t blockWords,
	uint32_t* __restrict__ sliceInfo)
{
	const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
	if (l >= lists)
		return;
	uint32_t start = 0;
	for (uint32_t r = 0; r < ranks; r++)
		start += received[r * blockWords + kExHeaderFixed + lists + l];
	sliceInfo[l * 2 + 0] = start;
}

uint32_t launchSampleRuns(Context& c, uint32_t* dSamples)
{
	const uint32_t lists = (uint32_t)c.segments.size();
	kSampleRuns<<<lists, 96, 0, c.stream>>>(c.dSegments, c.dCounters, c.keys[0], lists, dSamples);
	return 1;
}
uint32_t launchSplitAndPack(Context& c, cudaStream_t stream, uint32_t ranks, const uint32_t* dMySamples, const uint32_t* dGatheredSamples,
	uint32_t* dSplitters, uint32_t* dSendBlocks, uint32_t capacityPerDest)
{
	const uint32_t lists = (uint32_t)c.segments.size();
	SplitArgs S;
	S.segments = c.dSegments; S.counters = c.dCounters; S.keys = c.keys[0]; S.gathered = dGatheredSamples; S.mine = dMySamples; S.splitters = dSplitters;
	S.lists = lists; S.ranks = ranks;
	kSplitRuns<<<lists, 32 * std::max(1u, ranks - 1), 0, stream>>>(S);
	PackArgs P;
	P.segments = c.dSegments; P.keys = c.keys[0]; P.payloads = c.payloads[0];
	P.bounds = dSplitters + lists * (ranks - 1); P.blocks = dSendBlocks; P.lists = lists; P.ranks = ranks; P.capacity = capacityPerDest;
	kPackByDestination<<<c.smCount * 4, 256, 0, stream>>>(P);
	return 2;
}
uint32_t launchSliceStarts(cudaStream_t stream, uint32_t ranks, uint32_t lists, const uint32_t* dReceived, uint32_t capacityPerDest,
	uint32_t* dSliceInfo)
{
	kSliceStarts<<<(lists + 127) / 128, 128, 0, stream>>>(ranks, lists, dReceived, kExHeaderWords + 2ull * capacityPerDest, dSliceInfo);
	return 1;
}
} // namespace gsp

extern "C" uint64_t gsp_merge_tree_scratch_words(uint32_t outCapacity)
{
	return gsp::mergeTreeScratchWords(outCapacity);
}

extern "C" int gsp_merge_gathered_packed_tree(void* cudaStream, uint32_t ranks, uint32_t myRank, uint32_t lists, uint32_t capacityElems,
	const uint32_t* dGathered, uint32_t* dPlan, uint32_t* dSliceInfo, uint32_t* dOutKeys, uint32_t* dOutPayloads,
	uint8_t* dOutRanks, uint32_t outCapacity, uint32_t* dScratch)
{
	if (ranks == 0 || ranks > kMaxRanks || myRank >= ranks || lists == 0 || lists > kExMaxLists || !dGathered || !dPlan ||
		!dSliceInfo || !dOutKeys || !dOutPayloads || !dOutRanks || !dScratch || lists * ((ranks + 1) / 2) > gsp::kTreeMaxJobs ||
		!exchangeBlocksIndexable(capacityElems, ranks))
		return GSP_ERR_INVALID;
	int device = 0, sms = 148;
	cudaGetDevice(&device);
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
	gsp::launchMergePacked((cudaStream_t)cudaStream, ranks, myRank, lists, capacityElems, dGathered, dPlan, dSliceInfo, dOutKeys,
		dOutPayloads, dOutRanks, outCapacity, false, dScratch, (uint32_t)sms);
	return cudaGetLastError() == cudaSuccess ? GSP_OK : GSP_ERR_CUDA;
}
