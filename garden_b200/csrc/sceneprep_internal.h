// Internal declarations shared by the translation units of libgarden_sceneprep.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/garden_sceneprep.h"

namespace gsp
{

constexpr uint32_t kNone = 0xFFFFFFFFu;
constexpr int kMaxPools = GSP_MAX_POOLS;
constexpr int kMaxViews = GSP_MAX_VIEWS;

// ---- AoS field offsets of the reference's components (SURVEY.md §8 a1/a2, verified with offsetof in oracle/ref_harness) ----
// TransformComponent, include/garden/system/transform.hpp:31-60
constexpr uint32_t kTfEntity = 0, kTfParent = 4, kTfPos = 16, kTfScale = 32, kTfRot = 48, kTfSelfActive = 72,
	kTfAncestorsActive = 73, kTfWithAncestors = 74, kTfMinStride = 80;
// MeshRenderComponent, include/garden/system/render/mesh.hpp:45-55
constexpr uint32_t kMcEntity = 0, kMcEnabled = 14, kMcVisible = 15, kMcAabbMin = 16, kMcAabbMax = 32, kMcMinStride = 48;

// transform flags (SoA, 16 bits)
constexpr uint16_t kTfLive = 1, kTfActive = 2, kTfAncestors = 4;
// the local matrix of this transform needs the guarded 4-lane code (zero / subnormal entries, out-of-range or non-finite
// TRS): decided once at staging time by localModel43Fast<true>, so the per-frame kernel carries no guards
constexpr uint16_t kTfExactLocal = 8;
// the component's own selfActive / ancestorsActive bytes (transform.hpp:57-58); kTfActive = both (isActive(), :110)
constexpr uint16_t kTfSelfBit = 16, kTfAncBit = 32;
constexpr uint32_t kTfDepthShift = 8; // bits 8..15: chain length, saturating at 255 (= unknown: guarded generic walk)
constexpr uint32_t kTfDepthMax = 255;
// mesh flags (SoA): static filter of mesh.cpp:140-147 (entity != 0 && isEnabled && !degenerate AABB)
constexpr uint8_t kMfCandidate = 1;
// the isVisible byte the HOST currently holds for this slot (as uploaded, or as last written back): bit set = 1;
// kMfHostVisibleOdd = the host byte is neither 0 nor 1 (always rewritten by the delta write-back)
constexpr uint8_t kMfHostVisible = 2, kMfHostVisibleOdd = 4;

// ---- device SoA mirrors -------------------------------------------------------------------------------------------
struct TransformsDev
{
	uint32_t occupancy = 0, capacity = 0;
	float4* rot = nullptr;    // quaternion xyzw
	float4* posSx = nullptr;  // position xyz, scale x
	float2* sYZ = nullptr;    // scale y, z
	uint32_t* parent = nullptr; // parent transform slot or kNone
	uint32_t* entity = nullptr; // owner entity id (0 = free slot)
	uint32_t* parentEntity = nullptr;
	uint16_t* flags = nullptr;
	// conservative bound inputs of the prepass (cull.cu): x = largest |scale| component, y = |position|, both rounded up by
	// 2^-10; x = +inf for transforms whose local matrix needs the guarded code (the prepass then never culls below them)
	float2* bound = nullptr;
	// Prepass sphere of every mesh on this transform (kChainBounds + kChainRecords, refreshed whenever transforms, pools or
	// active flags changed): xyz = centre (the chain root's position), w = radius W >= 0 — ONE sphere per hierarchy (the
	// largest bound of any mesh below the root), so a hierarchy survives or is dropped as a whole; w < 0: the transform is
	// dead or inactive (never a candidate); w = +inf / NaN: never culled by the prepass.
	float4* record = nullptr;
	uint32_t* rho = nullptr;       // bits of the largest box radius of any mesh on the transform (kLinkPool)
	uint32_t* chainRoot = nullptr; // root slot of the transform's parent chain
	uint32_t* rootW = nullptr;     // per ROOT slot: bits of max over its hierarchy of D + S * rho
	uint32_t* poolMask = nullptr;  // bit p: pool p holds a mesh on this transform (kLinkPool)
	// split path (allocated when a pool needs it): surviving transforms and their world matrices
	uint32_t* tBits = nullptr; uint32_t* tBlockCount = nullptr; uint32_t* tBucketCount = nullptr; // (tBucketCount inside frameZero)
	uint32_t* tList = nullptr; uint32_t* tIndex = nullptr; float4* tWorld = nullptr;
	uint32_t splitCap = 0;
	uint32_t* entityToSlot = nullptr; // entity id -> slot + 1
	uint32_t entityCap = 0;
	// some parent chain is cyclic (decided once per gsp_set_transforms, staging.cu: kJumpParents): nothing walks the chains
	// then, so an acyclic hierarchy of any depth is walked to its roots and the per-frame walks only keep `occupancy` as a
	// bound against corrupted links
	bool cyclic = false;
};

struct PoolDev
{
	uint32_t occupancy = 0, capacity = 0, count = 0, stride = 0, renderType = 0, drawReady = 0;
	uint32_t viewMask = 0xFFFFFFFFu; // bit v: isDrawReady(views[v].shadowPass) (gsp_set_pool_view_mask)
	bool hasReady = false, set = false;
	bool split = false; // the pool's hierarchies reach outside the pool: world matrices per transform, then kClassify (cull.cu)
	float4* aabbA = nullptr;  // min xyz, max x
	float2* aabbB = nullptr;  // max y, z
	uint32_t* entity = nullptr;
	uint32_t* tslot = nullptr; // transform slot or kNone (resolved by the link kernel)
	uint8_t* flags = nullptr;
	uint8_t* ready = nullptr;
	float* radius = nullptr;   // per slot: distance of the farthest AABB corner from the local origin, rounded up (prepass)
	// ---- per frame. The prepass compacts the slots that survive the filter and its conservative bound into a list in slot
	// order; everything downstream (world matrices, ballots, chunks, payloads) is indexed by SURVIVOR INDEX ----
	uint32_t* surList = nullptr;  // survivor index -> slot
	uint32_t* surTs = nullptr;    // survivor index -> transform slot
	float4* world = nullptr;   // kWorldStride x float4 per SURVIVOR: float4x3 world matrix (c0..c3 lanes xyz), written when visible anywhere
	float4* worldPos = nullptr; // (c3.x, c3.y, c3.z, 0) of the same matrices, dense: all the key computation (kScatter) reads
	uint8_t* visible = nullptr; // isVisible of the last main view, per slot
	uint32_t* cullStatus = nullptr; // [kMaxViews][chunks] visible count per chunk of survivors and view, scanned in place to list offsets
	uint32_t* visBits = nullptr;    // [kMaxViews][tiles * 8] visibility ballot words over survivor indices
	uint32_t* surBits = nullptr;     // [prepass blocks][32] survivor bit per slot
	uint32_t* blockCount = nullptr;  // [prepass blocks]
	uint32_t* bucketCount = nullptr; // [prepass blocks / 64 + 1]
	uint32_t cullTiles = 0, cullTilesCap = 0;
	bool visibleValid = false;
};

// Per-view constants handed to the cull kernel by value (__grid_constant__).
struct ViewConst
{
	float planes[6][4];  // the caller's planes, verbatim: only the exact 8-corner test reads them
	// Conservative classifier: the same planes scaled to unit normals (host, double precision); slots past planeCount
	// and planes that can never cull hold (0, 0, 0, +inf), planes that cull everything hold (0, 0, 0, -inf).
	// Stored as pairs of planes (2j, 2j+1) per coefficient so that one packed FMA serves two planes.
	float2 ux[3], uy[3], uz[3], ud[3];
	float slack;         // max_i |unit d_i| * kBandD (rounded up); +inf forces the exact test for the whole view
	float cameraOffset[4];
	uint32_t planeCount;
	uint32_t enabled;   // pool participates in this view
};
struct CullParams
{
	ViewConst views[kMaxViews];
	float cam[4];          // camera position subtracted from c3 (zero for UI pools, mesh.cpp:441)
	uint32_t viewCount;
	uint32_t occupancy;
	uint32_t poolIndex;    // goes into payload bits 28..31
	uint32_t key2D;        // UI: key = model.c3.z + 1.0f (mesh.cpp:250)
	uint32_t descending;   // translucent / UI lists sort descending (mesh.hpp:204)
	uint32_t hasReady;
	// Views whose six planes form a box (orthographic frusta: the CSM cascades) with the SAME orientation. boxAxis are the
	// three common face normals, [boxLo, boxHi] the union of the views' extents along each: a sphere that lies beyond that
	// interval on some axis is behind a face plane of EVERY such view, so one test of three dot products stands for all of
	// them (cull.cu: boxesCulled); boxMask == 0: no such view in this frame.
	uint32_t boxMask;
	float boxAxis[3][3];
	float boxLo[3], boxHi[3];
	float boxSlack;
	float boxViewLo[kMaxViews][3], boxViewHi[kMaxViews][3]; // each group view's own extents along boxAxis (the prepass)
};

// A segment = one output list of one view: (view, canonical pool). Unsorted buffers own a segment each;
// all translucent pools of a view share one, all UI pools share one.
struct Segment
{
	uint32_t offset = 0;    // element offset into the key/payload/record arenas
	uint32_t capacity = 0;
	uint32_t view = 0, pool = 0; // canonical (first) pool
	uint32_t lastPool = 0;  // last pool appending to it (its poolEnd is the final count)
	uint32_t sorted = 1;    // 0 for OIT buffers (mesh.cpp:273-277)
	uint32_t descending = 0, key2D = 0, stride = 0;
	int kind = 0;           // 0 unsorted, 1 translucent, 2 ui
	int listIndex = 0;      // unsorted buffer index within the view
};

struct SegmentDev // device-visible part
{
	uint32_t offset, capacity, countIndex /* index into poolEnd of lastPool,view */, sorted;
	uint32_t descending, key2D, pad0, pad1;
};

struct Exchange; // multi-GPU exchange state (exchange.cu)

struct Context
{
	int device = 0;
	Exchange* exchange = nullptr;
	// all-to-all exchange: the previous frame's runs are still being packed out of the key / payload arenas on the exchange
	// stream; the next frame's first kScatter waits for this event (its prepass and kCull run meanwhile)
	cudaEvent_t arenaFree = nullptr; bool arenaFreePending = false;
	uint32_t smCount = 148; // cudaDevAttrMultiProcessorCount of `device` (grid sizes of the persistent kernels)
	cudaStream_t ownStream = nullptr, stream = nullptr;
	cudaStream_t copyStream = nullptr; cudaEvent_t copyEvent = nullptr; // list downloads overlap the caller / the write-back
	bool fetchInFlight = false;
	bool fetchedValid = false; // gsp_fetch_all_async took a snapshot of the frame's lists: the list getters keep serving it while the
	                           // NEXT frame's inputs are staged (until gsp_run_async or a layout change)
	std::string error;

	TransformsDev tf;
	PoolDev pools[kMaxPools];
	uint32_t poolCount = 0;

	std::vector<gsp_view> views;
	float cameraPos[3] = {0, 0, 0};
	bool viewsSet = false, linkDirty = true, layoutDirty = true, resultsValid = false;
	bool chainDirty = true; // the transform pool changed since kChainBounds last ran
	bool anySplit = false;  // some pool takes the split path this frame
	bool splitRan = false;
	cudaEvent_t splitEvents[2] = {};
	bool cullAttrsSet = false, scatterAttrSet = false; // kernel function attributes applied on this context's device
	bool frameEnqueued = false; // a frame has been enqueued since the last structural change (its results may still be in flight)

	// segments
	std::vector<Segment> segments;
	int segOf[kMaxViews][kMaxPools]; // view,pool -> segment index or -1
	int prevPool[kMaxViews][kMaxPools]; // previous pool appending to the same list (-1 = first)
	bool participates[kMaxViews][kMaxPools]; // pool is processed in this view (count > 0 && isDrawReady, mesh.cpp:426,482)
	uint32_t bufferIndexOf[kMaxViews][kMaxPools]; // unsorted / sorted buffer index of the pool in the view
	uint32_t unsortedCount[kMaxViews], sortedCount[kMaxViews];
	SegmentDev* dSegments = nullptr; uint32_t dSegmentsCap = 0;
	uint32_t arenaElems = 0, arenaCap = 0;
	uint32_t* keys[2] = {nullptr, nullptr};
	uint32_t* payloads[2] = {nullptr, nullptr};
	gsp_record* records = nullptr; size_t recordsCap = 0;

	// per-frame device counters: [0, P*V) poolEnd, [P*V, 2*P*V) poolInst, then tickets, then error flag
	uint32_t* dCounters = nullptr;
	uint32_t* hCounters = nullptr; // pinned
	// sort scratch
	uint32_t* frameZero = nullptr; size_t frameZeroWords = 0, frameZeroCap = 0; // per-frame scratch that starts at zero (one memset)
	uint32_t* sortHist = nullptr;   // [segments][4][256] (inside frameZero)
	unsigned long long* sortStatus = nullptr; // [tiles][256] look-back words tagged with the launch epoch (never cleared)
	uint32_t sortEpoch = 0;
	uint32_t* sortTickets = nullptr; // [segments][4]
	uint32_t* segTileOffset = nullptr; // device: prefix of tiles per segment (capacity based)
	uint32_t sortTilesTotal = 0, sortScratchSegs = 0;
	size_t sortStatusCap = 0;

	// host staging
	void* dAosScratch = nullptr; size_t dAosScratchCap = 0;
	uint8_t* hGather = nullptr; size_t hGatherCap = 0; // pinned: scattered dirty components packed for one upload
	uint64_t zeroCopyBytes = 0; // bytes the staging kernels read straight from pinned host memory
	gsp_record* hRecords = nullptr; size_t hRecordsCap = 0; // pinned download area (arena-shaped)
	std::vector<uint8_t> segDownloaded;
	uint32_t* hVisible = nullptr; uint32_t* dVisMapped = nullptr; uint32_t* dVisScratch = nullptr; size_t visScratchCap = 0; // isVisible write-back: bit words / changed-slot list (+1 count word)
	uint32_t launchCount = 0;
	bool profiling = false;
	cudaEvent_t phaseEvents[8] = {};
	cudaEvent_t poolEvents[kMaxPools][3] = {}; // after the prepass, after kCull, after the scatter
	bool poolLaunched[kMaxPools] = {};
	bool phaseEventsCreated = false, phaseTimesValid = false;
	uint32_t* dError = nullptr;
};

// counters layout helpers
__host__ __device__ inline uint32_t ctrPoolEnd(uint32_t pool, uint32_t view) { return pool * kMaxViews + view; }
__host__ __device__ inline uint32_t ctrPoolInst(uint32_t pool, uint32_t view) { return kMaxPools * kMaxViews + pool * kMaxViews + view; }
constexpr uint32_t kCtrCullTicket = 2 * kMaxPools * kMaxViews; // + pool (unused)
constexpr uint32_t kCtrSurvivors = kCtrCullTicket + kMaxPools;  // + pool: survivors of the prepass
constexpr uint32_t kCtrSurvivorsT = kCtrSurvivors + kMaxPools; // surviving transforms (split path)
constexpr uint32_t kCtrCross = kCtrSurvivorsT + 1;            // + pool: slots whose parent transform has no mesh in the pool (link time)
constexpr uint32_t kCtrError = kCtrCross + kMaxPools;
constexpr uint32_t kCtrCount = kCtrError + 8;  // (the pinned host mirror has 16 more words: staging scalars, link-time statistics)

// float4 per slot in PoolDev::world: the 48-byte matrix, unpadded. (Padding it to one 64-byte DRAM line was measured and is
// slower: neighbouring slots are usually visible together and then share lines; 0.980 -> 1.012 ms per frame on C4.)
constexpr uint32_t kWorldStride = 3;
constexpr uint32_t kCullTile = 256;       // survivors per cull block (4 warp tiles of 64)
constexpr uint32_t kPreTile = 1024;       // slots per prepass block
constexpr uint32_t kSortItems = 16;       // keys per thread in the radix sort
constexpr uint32_t kSortThreads = 256;
constexpr uint32_t kSortTile = kSortItems * kSortThreads;

// ---- packed exchange block of the multi-GPU path (merge.cu) ----
constexpr uint32_t kExHeaderWords = 256, kExHeaderFixed = 8, kExMaxLists = kExHeaderWords - kExHeaderFixed;
constexpr uint32_t kExMagic = 0x47535031u; // "GSP1"
constexpr uint32_t kMaxRanks = 32;          // GPUs of one communicator (gsp_comm_init)
// The merge tree (merge.cu) indexes the received blocks with 32-bit element indices: the `ranks` blocks of
// kExHeaderWords + 2 * capacityElems words each must stay below 2^32 words together.
inline bool exchangeBlocksIndexable(uint32_t capacityElems, uint32_t ranks)
{
	return ((uint64_t)kExHeaderWords + 2ull * capacityElems) * ranks < (1ull << 32);
}

// ---- kernel launchers (each returns the number of kernels it launched, or throws nothing; errors via cudaGetLastError) ----
uint32_t launchStageTransforms(Context& c, const void* dAos, uint32_t stride, uint32_t first, uint32_t count, bool full,
	uint32_t* dMaxEntity, const uint32_t* dSlotMap = nullptr);
uint32_t launchBuildHierarchy(Context& c, uint32_t* dDeep);
uint32_t launchFindCycles(Context& c, uint32_t* dCyclic);
uint32_t launchStagePool(Context& c, uint32_t pool, const void* dAos, uint32_t stride, uint32_t first, uint32_t count,
	const uint32_t* dSlotMap = nullptr, const uint8_t* dReady = nullptr);
uint32_t launchLink(Context& c);
uint32_t launchChainBounds(Context& c);
uint32_t launchLinkSlots(Context& c, uint32_t pool, const uint32_t* dSlotMap, uint32_t first, uint32_t count, bool walk,
	uint32_t* dGrew);
uint32_t launchChainRecords(Context& c);
uint32_t launchSplitWorld(Context& c, cudaEvent_t before, cudaEvent_t after);
uint32_t launchCull(Context& c, uint32_t pool, cudaEvent_t afterPrepass, cudaEvent_t afterCull, cudaEvent_t afterScatter);
uint32_t launchSort(Context& c, cudaEvent_t afterHistogram);
uint32_t launchEmit(Context& c);
uint32_t launchInstances(Context& c, int seg, const float* viewProj, void* dDst, uint32_t stride, uint32_t offset, uint32_t capacity);
uint32_t launchSetActive(Context& c, const uint32_t* dIds, uint32_t count, int active);
uint32_t launchAnimate(Context& c, const uint32_t* dIds, const uint8_t* dFlags, const float* dA, const float* dB, const float* dT,
	uint32_t count);
uint32_t launchExportPacked(Context& c, uint32_t* dBlock, uint32_t capacity);
void destroyExchange(Context& c);
uint32_t launchPackVisible(Context& c, uint32_t pool, uint32_t* dBits);
uint32_t launchVisibleDelta(Context& c, uint32_t pool, uint32_t* list, uint32_t* dCount, uint32_t* hCountMapped);

} // namespace gsp

struct gsp_context
{
	gsp::Context c;
};
