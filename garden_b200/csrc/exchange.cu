// Multi-GPU exchange behind the C ABI: NCCL lives INSIDE libgarden_sceneprep.so (loaded at run time, so single-GPU users do
// not need it), one context per GPU, one communicator over the contexts of a frame.
//
// The reference has no counterpart (one process, one std::sort per list, mesh.cpp:265-328). Every GPU prepares a contiguous
// entity range with the single-GPU path; what has to be exchanged so that the sharded result equals ONE sort over all
// entities are the sorted (key, payload) runs. Per frame, without any host synchronisation:
//   compute stream:   gsp_run_async -> export of the runs into fixed-capacity blocks (lengths read on the device)
//   exchange stream:  collective(s) -> merge plan from the received headers -> k-way merge of this rank's key range
// and frame k's exchange overlaps frame k+1's culling (double-buffered sets, reuse guarded by events).
// Two protocols (GSP_EXCHANGE=allgather|alltoall, default alltoall):
//   allgather  every rank receives every run (one ncclAllGather of equal blocks) and cuts out its key range itself;
//   alltoall   the runs are cut by common splitters BEFORE they travel: a small all-gather of samples gives every rank the
//              same weighted quantiles, each rank packs one sub-block per destination, grouped ncclSend/ncclRecv move them,
//              and a rank receives only what it merges: 1/ranks of the all-gather's volume. Sub-block headers also carry
//              "elements of the sender's run below your key range", whose sum is where the slice starts in the merged list.
// Both protocols merge with the same pairwise merge-path tree (merge.cu: kTreePartition + kMergeTree).
// The block capacity is speculative: an overflow is flagged in the header and in the plan flags, nothing is merged for
// that frame, and the host — which reads the flags from pinned memory — grows the blocks and repeats the frame.
#include "sceneprep_internal.h"

#include <dlfcn.h>
#include <nccl.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

namespace gsp
{

// ---- NCCL, resolved at run time -------------------------------------------------------------------------------------------
struct NcclApi
{
	void* handle = nullptr;
	ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
	ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
	ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
	ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
	ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*GroupStart)() = nullptr;
	ncclResult_t (*GroupEnd)() = nullptr;
	const char* (*GetErrorString)(ncclResult_t) = nullptr;
	std::string error;
};

static NcclApi& nccl()
{
	static NcclApi api;
	static std::once_flag once;
	std::call_once(once, [] {
		// a copy that is already in the process (e.g. the one PyTorch ships) wins: RTLD_NOLOAD first
		const char* names[] = { "libnccl.so.2", "libnccl.so" };
		for (const char* n : names)
			if (!api.handle) api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
		for (const char* n : names)
			if (!api.handle) api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
		if (!api.handle)
		{
			api.error = std::string("libnccl.so.2 could not be loaded: ") + (dlerror() ? dlerror() : "?");
			return;
		}
		#define GSP_NCCL_SYM(field, name) \
			api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.handle, name)); \
			if (!api.field) api.error = std::string("symbol missing in libnccl: ") + name;
		GSP_NCCL_SYM(GetUniqueId, "ncclGetUniqueId") GSP_NCCL_SYM(CommInitRank, "ncclCommInitRank")
		GSP_NCCL_SYM(CommInitAll, "ncclCommInitAll") GSP_NCCL_SYM(CommDestroy, "ncclCommDestroy")
		GSP_NCCL_SYM(AllGather, "ncclAllGather") GSP_NCCL_SYM(AllReduce, "ncclAllReduce")
		GSP_NCCL_SYM(Send, "ncclSend") GSP_NCCL_SYM(Recv, "ncclRecv")
		GSP_NCCL_SYM(GroupStart, "ncclGroupStart") GSP_NCCL_SYM(GroupEnd, "ncclGroupEnd")
		GSP_NCCL_SYM(GetErrorString, "ncclGetErrorString")
		#undef GSP_NCCL_SYM
	});
	return api;
}

// ---- per-context exchange state --------------------------------------------------------------------------------------------
constexpr uint32_t kExSets = 2;
constexpr uint32_t kExSamples = 64;                       // keys sampled per list and rank for the common splitters
constexpr uint32_t kExSampleWords = kExSamples + 1;       // + the run length

struct ExchangeSet
{
	uint32_t* send = nullptr;       // allgather: one block; alltoall: `ranks` sub-blocks back to back
	uint32_t* recv = nullptr;       // `ranks` blocks
	uint32_t* plan = nullptr;
	uint32_t* sliceInfo = nullptr;  // [lists][2]: global start of my slice (alltoall: filled by the length exchange), length
	uint32_t* outKeys = nullptr; uint32_t* outPays = nullptr; uint8_t* outRanks = nullptr;
	uint32_t* samples = nullptr;    // alltoall: [lists][kExSampleWords] mine, then [ranks][lists][kExSampleWords] gathered
	uint32_t* splitters = nullptr;  // alltoall: [lists][ranks - 1] common splitters, then per-rank scratch
	uint32_t* hFlags = nullptr;     // pinned: the 8 plan flags of the frame
	cudaEvent_t exported = nullptr, done = nullptr;
	cudaEvent_t t[4] = {};          // optional timing: export | collective | merge
	bool used = false, pending = false;
	uint64_t frame = 0;
};

struct Exchange
{
	ncclComm_t comm = nullptr;
	uint32_t ranks = 0, rank = 0;
	cudaStream_t stream = nullptr;
	ExchangeSet sets[kExSets];
	uint32_t capacity = 0;      // elements per rank block (allgather) / per destination sub-block (alltoall)
	uint32_t outCapacity = 0;
	uint32_t lists = 0;
	uint64_t frameIndex = 0;
	bool allToAll = true, timing = false;
	uint32_t* dScalar = nullptr; // 2 words for the autosize reduction
	uint32_t* mergeScratch = nullptr; // the two intermediate levels of the merge tree (merges are serialised on `stream`)
};

} // namespace gsp

using namespace gsp;

namespace gsp
{
uint32_t launchMergePacked(cudaStream_t stream, uint32_t ranks, uint32_t myRank, uint32_t lists, uint32_t capacityElems,
	const uint32_t* dGathered, uint32_t* dPlan, uint32_t* dSliceInfo, uint32_t* dOutKeys, uint32_t* dOutPays, uint8_t* dOutRanks,
	uint32_t outCapacity, bool preSplit, uint32_t* dTreeScratch, uint32_t smCount);
uint32_t launchSampleRuns(Context& c, uint32_t* dSamples);
uint32_t launchSplitAndPack(Context& c, cudaStream_t stream, uint32_t ranks, const uint32_t* dMySamples, const uint32_t* dGatheredSamples,
	uint32_t* dSplitters, uint32_t* dSendBlocks, uint32_t capacityPerDest);
uint32_t launchSliceStarts(cudaStream_t stream, uint32_t ranks, uint32_t lists, const uint32_t* dReceived, uint32_t capacityPerDest,
	uint32_t* dSliceInfo);
}

#define GSP_CUDA(call)                                                                             \
	do {                                                                                           \
		cudaError_t err__ = (call);                                                                \
		if (err__ != cudaSuccess) {                                                                \
			c.error = std::string(#call) + ": " + cudaGetErrorString(err__);                       \
			return GSP_ERR_CUDA;                                                                   \
		}                                                                                          \
	} while (0)
#define GSP_NCCL(call)                                                                             \
	do {                                                                                           \
		ncclResult_t res__ = (call);                                                               \
		if (res__ != ncclSuccess) {                                                                \
			c.error = std::string(#call) + ": " + N.GetErrorString(res__);                         \
			return GSP_ERR_CUDA;                                                                   \
		}                                                                                          \
	} while (0)

static int failEx(Context& c, int code, const char* message)
{
	c.error = message;
	return code;
}

static void freeSets(Exchange& x)
{
	for (auto& s : x.sets)
	{
		cudaFree(s.send); cudaFree(s.recv); cudaFree(s.plan); cudaFree(s.sliceInfo); cudaFree(s.outKeys); cudaFree(s.outPays);
		cudaFree(s.outRanks); cudaFree(s.samples); cudaFree(s.splitters); cudaFreeHost(s.hFlags);
		s.send = s.recv = s.plan = s.sliceInfo = s.outKeys = s.outPays = s.samples = s.splitters = s.hFlags = nullptr;
		s.outRanks = nullptr;
		s.used = s.pending = false;
	}
	cudaFree(x.mergeScratch);
	x.mergeScratch = nullptr;
	x.capacity = x.outCapacity = 0;
}

namespace gsp
{
void destroyExchange(Context& c)
{
	Exchange* x = c.exchange;
	if (!x)
		return;
	cudaSetDevice(c.device);
	if (x->stream) cudaStreamSynchronize(x->stream);
	freeSets(*x);
	for (auto& s : x->sets)
	{
		if (s.exported) cudaEventDestroy(s.exported);
		if (s.done) cudaEventDestroy(s.done);
		for (auto& e : s.t) if (e) cudaEventDestroy(e);
	}
	cudaFree(x->dScalar);
	if (c.arenaFree) { cudaEventDestroy(c.arenaFree); c.arenaFree = nullptr; c.arenaFreePending = false; }
	if (x->comm && nccl().CommDestroy) nccl().CommDestroy(x->comm);
	if (x->stream) cudaStreamDestroy(x->stream);
	delete x;
	c.exchange = nullptr;
}
} // namespace gsp

static int attachComm(Context& c, ncclComm_t comm, uint32_t ranks, uint32_t rank)
{
	destroyExchange(c);
	Exchange* x = new (std::nothrow) Exchange();
	if (!x)
		return GSP_ERR_NOMEM;
	x->comm = comm; x->ranks = ranks; x->rank = rank;
	const char* mode = getenv("GSP_EXCHANGE");
	x->allToAll = !(mode && !strcmp(mode, "allgather"));
	c.exchange = x;
	GSP_CUDA(cudaSetDevice(c.device));
	GSP_CUDA(cudaStreamCreateWithFlags(&x->stream, cudaStreamNonBlocking));
	GSP_CUDA(cudaMalloc((void**)&x->dScalar, 2 * sizeof(uint32_t)));
	for (auto& s : x->sets)
	{
		GSP_CUDA(cudaEventCreateWithFlags(&s.exported, cudaEventDisableTiming));
		GSP_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
		for (auto& e : s.t) GSP_CUDA(cudaEventCreate(&e));
	}
	return GSP_OK;
}

static int allocateSets(Context& c, uint32_t capacity)
{
	Exchange& x = *c.exchange;
	GSP_CUDA(cudaSetDevice(c.device));
	GSP_CUDA(cudaStreamSynchronize(x.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	freeSets(x);
	x.lists = (uint32_t)c.segments.size();
	if (x.allToAll && 2u * x.lists > kExMaxLists)
		x.allToAll = false; // the sub-block headers carry two words per list: beyond that, the all-gather protocol
	const uint32_t lists = std::max(1u, x.lists), ranks = x.ranks;
	const size_t blockWords = kExHeaderWords + 2ull * capacity;
	// allgather: every rank's slice fits even if one key range swallowed everything; alltoall: what can be received
	const size_t outCap = (size_t)capacity * ranks;
	if (outCap > 0xFFFFFFF0ull)
		return failEx(c, GSP_ERR_NOMEM, "exchange capacity exceeds 2^32 elements");
	if (!exchangeBlocksIndexable(capacity, ranks))
		return failEx(c, GSP_ERR_NOMEM, "exchange blocks of all ranks reach 2^32 words (the merge indexes them with 32 bits)");
	const size_t planWords = 2ull * ranks * lists + lists + 2ull * lists * ranks + 8;
	for (auto& s : x.sets)
	{
		GSP_CUDA(cudaMalloc((void**)&s.send, blockWords * (x.allToAll ? ranks : 1) * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&s.recv, blockWords * ranks * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&s.plan, planWords * sizeof(uint32_t)));
		GSP_CUDA(cudaMemset(s.plan, 0, planWords * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&s.sliceInfo, lists * 2 * sizeof(uint32_t)));
		GSP_CUDA(cudaMemset(s.sliceInfo, 0, lists * 2 * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&s.outKeys, outCap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&s.outPays, outCap * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&s.outRanks, outCap));
		GSP_CUDA(cudaMalloc((void**)&s.samples, (size_t)(ranks + 1) * lists * kExSampleWords * sizeof(uint32_t)));
		GSP_CUDA(cudaMalloc((void**)&s.splitters, (size_t)lists * (ranks + 1) * 2 * sizeof(uint32_t)));
		GSP_CUDA(cudaMallocHost((void**)&s.hFlags, 8 * sizeof(uint32_t)));
		memset(s.hFlags, 0, 8 * sizeof(uint32_t));
	}
	GSP_CUDA(cudaMalloc((void**)&x.mergeScratch, gsp_merge_tree_scratch_words((uint32_t)outCap) * sizeof(uint32_t)));
	x.capacity = capacity; x.outCapacity = (uint32_t)outCap;
	return GSP_OK;
}

extern "C"
{

int gsp_comm_unique_id(uint8_t id[GSP_COMM_ID_BYTES])
{
	NcclApi& N = nccl();
	if (!id || !N.GetUniqueId)
		return GSP_ERR_CUDA;
	static_assert(GSP_COMM_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "id size");
	ncclUniqueId u;
	if (N.GetUniqueId(&u) != ncclSuccess)
		return GSP_ERR_CUDA;
	memcpy(id, u.internal, NCCL_UNIQUE_ID_BYTES);
	return GSP_OK;
}

int gsp_comm_init(gsp_context* ctx, const uint8_t id[GSP_COMM_ID_BYTES], uint32_t ranks, uint32_t rank)
{
	if (!ctx || !id)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (ranks == 0 || ranks > kMaxRanks || rank >= ranks)
		return failEx(c, GSP_ERR_INVALID, "gsp_comm_init: need 1 <= ranks <= 32 and rank < ranks");
	NcclApi& N = nccl();
	if (!N.CommInitRank)
		return failEx(c, GSP_ERR_CUDA, N.error.empty() ? "NCCL is not available" : N.error.c_str());
	GSP_CUDA(cudaSetDevice(c.device));
	ncclUniqueId u;
	memcpy(u.internal, id, NCCL_UNIQUE_ID_BYTES);
	ncclComm_t comm = nullptr;
	GSP_NCCL(N.CommInitRank(&comm, (int)ranks, u, (int)rank));
	return attachComm(c, comm, ranks, rank);
}

int gsp_comm_init_all(gsp_context** contexts, uint32_t count)
{
	if (!contexts || count == 0 || count > kMaxRanks)
		return GSP_ERR_INVALID;
	for (uint32_t i = 0; i < count; i++)
		if (!contexts[i]) return GSP_ERR_INVALID;
	Context& c = contexts[0]->c;
	NcclApi& N = nccl();
	if (!N.CommInitAll)
		return failEx(c, GSP_ERR_CUDA, N.error.empty() ? "NCCL is not available" : N.error.c_str());
	int devices[kMaxRanks];
	ncclComm_t comms[kMaxRanks];
	for (uint32_t i = 0; i < count; i++)
		devices[i] = contexts[i]->c.device;
	GSP_NCCL(N.CommInitAll(comms, (int)count, devices));
	for (uint32_t i = 0; i < count; i++)
	{
		int rc = attachComm(contexts[i]->c, comms[i], count, i);
		if (rc) return rc;
	}
	return GSP_OK;
}

int gsp_comm_destroy(gsp_context* ctx)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	destroyExchange(ctx->c);
	return GSP_OK;
}

int gsp_comm_info(const gsp_context* ctx, uint32_t* ranks, uint32_t* rank, uint32_t* capacity, uint32_t* allToAll)
{
	if (!ctx || !ctx->c.exchange)
		return GSP_ERR_STATE;
	const Exchange& x = *ctx->c.exchange;
	if (ranks) *ranks = x.ranks;
	if (rank) *rank = x.rank;
	if (capacity) *capacity = x.capacity;
	if (allToAll) *allToAll = x.allToAll ? 1u : 0u;
	return GSP_OK;
}

int gsp_exchange_configure(gsp_context* ctx, uint32_t capacityElems)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.exchange)
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_configure: gsp_comm_init has not been called");
	if (c.layoutDirty || c.segments.empty() || c.segments.size() > kExMaxLists)
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_configure: run a frame first (the lists of the frame define the exchange)");
	return allocateSets(c, std::max(capacityElems, 16u));
}

// Collective: one synchronous frame, the largest per-rank total over all ranks (ncclAllReduce max), head room, allocation.
// alltoall: the capacity is per DESTINATION sub-block: (largest total / ranks) with more head room, since the split follows
// sampled quantiles.
int gsp_exchange_autosize(gsp_context* ctx, uint32_t* capacityOut)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.exchange)
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_autosize: gsp_comm_init has not been called");
	Exchange& x = *c.exchange;
	NcclApi& N = nccl();
	int rc = gsp_run(ctx);
	if (rc) return rc;
	uint32_t total = (uint32_t)std::min<uint64_t>(gsp_last_visible_total(ctx), 0xFFFFFFFFull);
	GSP_CUDA(cudaMemcpyAsync(x.dScalar, &total, sizeof(uint32_t), cudaMemcpyHostToDevice, c.stream));
	GSP_NCCL(N.AllReduce(x.dScalar, x.dScalar + 1, 1, ncclUint32, ncclMax, x.comm, c.stream));
	uint32_t largest = 0;
	GSP_CUDA(cudaMemcpyAsync(&largest, x.dScalar + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
	GSP_CUDA(cudaStreamSynchronize(c.stream));
	uint64_t cap = x.allToAll ? (uint64_t)largest * 4 / (3 * x.ranks) + 8192 : (uint64_t)largest * 5 / 4 + 4096;
	if (capacityOut) *capacityOut = (uint32_t)cap;
	return allocateSets(c, (uint32_t)cap);
}

int gsp_exchange_set_timing(gsp_context* ctx, int enabled)
{
	if (!ctx || !ctx->c.exchange)
		return GSP_ERR_STATE;
	ctx->c.exchange->timing = enabled != 0;
	return GSP_OK;
}

// Enqueues the exchange of the frame that has just been enqueued (gsp_run_async).
int gsp_exchange_async(gsp_context* ctx)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	Exchange* xp = c.exchange;
	if (!xp || !xp->capacity)
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_async: gsp_comm_init + gsp_exchange_configure / _autosize first");
	if (!c.frameEnqueued || c.layoutDirty)
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_async: no frame has been enqueued (gsp_run_async) since the last change");
	Exchange& x = *xp;
	if (x.lists != c.segments.size())
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_async: the frame's lists changed, call gsp_exchange_configure again");
	NcclApi& N = nccl();
	GSP_CUDA(cudaSetDevice(c.device));
	ExchangeSet& s = x.sets[x.frameIndex % kExSets];
	if (s.pending)
	{
		// its flags have not been looked at yet: do that before the set is overwritten (an unseen overflow must not vanish)
		GSP_CUDA(cudaEventSynchronize(s.done));
		if (s.hFlags[0])
			return failEx(c, GSP_ERR_NOMEM, "gsp_exchange_async: an earlier frame overflowed its exchange blocks (gsp_exchange_poll)");
		s.pending = false;
	}
	if (s.used)
		GSP_CUDA(cudaStreamWaitEvent(c.stream, s.done, 0)); // the exchange that last read this set's blocks has finished
	const uint32_t lists = x.lists, ranks = x.ranks;
	const size_t blockWords = kExHeaderWords + 2ull * x.capacity;
	if (x.timing) cudaEventRecord(s.t[0], c.stream);
	if (!x.allToAll)
	{
		launchExportPacked(c, s.send, x.capacity);
		GSP_CUDA(cudaEventRecord(s.exported, c.stream));
		GSP_CUDA(cudaStreamWaitEvent(x.stream, s.exported, 0));
		if (x.timing) cudaEventRecord(s.t[1], x.stream);
		GSP_NCCL(N.AllGather(s.send, s.recv, blockWords, ncclUint32, x.comm, x.stream));
		if (x.timing) cudaEventRecord(s.t[2], x.stream);
		launchMergePacked(x.stream, ranks, x.rank, lists, x.capacity, s.recv, s.plan, s.sliceInfo, s.outKeys, s.outPays, s.outRanks,
			x.outCapacity, false, x.mergeScratch, c.smCount);
	}
	else
	{
		// samples of my runs (compute stream: the runs are final there), then everything else on the exchange stream
		launchSampleRuns(c, s.samples);
		GSP_CUDA(cudaEventRecord(s.exported, c.stream));
		GSP_CUDA(cudaStreamWaitEvent(x.stream, s.exported, 0));
		if (x.timing) cudaEventRecord(s.t[1], x.stream);
		const size_t sampleWords = (size_t)lists * kExSampleWords;
		GSP_NCCL(N.AllGather(s.samples, s.samples + sampleWords, sampleWords, ncclUint32, x.comm, x.stream));
		launchSplitAndPack(c, x.stream, ranks, s.samples, s.samples + sampleWords, s.splitters, s.send, x.capacity);
		if (!c.arenaFree)
			GSP_CUDA(cudaEventCreateWithFlags(&c.arenaFree, cudaEventDisableTiming));
		GSP_CUDA(cudaEventRecord(c.arenaFree, x.stream));
		c.arenaFreePending = true;
		GSP_NCCL(N.GroupStart());
		for (uint32_t r = 0; r < ranks; r++)
		{
			GSP_NCCL(N.Send(s.send + (size_t)r * blockWords, blockWords, ncclUint32, (int)r, x.comm, x.stream));
			GSP_NCCL(N.Recv(s.recv + (size_t)r * blockWords, blockWords, ncclUint32, (int)r, x.comm, x.stream));
		}
		GSP_NCCL(N.GroupEnd());
		if (x.timing) cudaEventRecord(s.t[2], x.stream);
		launchMergePacked(x.stream, ranks, x.rank, lists, x.capacity, s.recv, s.plan, s.sliceInfo, s.outKeys, s.outPays, s.outRanks,
			x.outCapacity, true, x.mergeScratch, c.smCount);
		// where my slices start in the merged lists: every source put "elements below your range" into its sub-block header
		launchSliceStarts(x.stream, ranks, lists, s.recv, x.capacity, s.sliceInfo);
	}
	if (x.timing) cudaEventRecord(s.t[3], x.stream);
	const size_t planWords = 2ull * ranks * lists + lists + 2ull * lists * ranks + 8;
	GSP_CUDA(cudaMemcpyAsync(s.hFlags, s.plan + planWords - 8, 8 * sizeof(uint32_t), cudaMemcpyDeviceToHost, x.stream));
	GSP_CUDA(cudaEventRecord(s.done, x.stream));
	GSP_CUDA(cudaGetLastError());
	s.used = true; s.pending = true; s.frame = x.frameIndex;
	x.frameIndex++;
	return GSP_OK;
}

// Looks at the flags of the exchanges that have finished (wait != 0: of all that were enqueued). errorBits: 1 a block
// overflowed, 2 bad header, 4 merged lists exceed the output capacity; needed = capacity that would have sufficed.
int gsp_exchange_poll(gsp_context* ctx, int wait, uint32_t* errorBits, uint32_t* needed)
{
	if (errorBits) *errorBits = 0;
	if (needed) *needed = 0;
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.exchange)
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_poll: gsp_comm_init has not been called");
	Exchange& x = *c.exchange;
	GSP_CUDA(cudaSetDevice(c.device));
	for (auto& s : x.sets)
	{
		if (!s.pending)
			continue;
		if (wait)
			GSP_CUDA(cudaEventSynchronize(s.done));
		else if (cudaEventQuery(s.done) != cudaSuccess)
		{
			cudaGetLastError();
			continue;
		}
		s.pending = false;
		if (s.hFlags[0])
		{
			if (errorBits) *errorBits |= s.hFlags[0];
			// flags[2] = largest per-rank (allgather) / per-block (alltoall) total that was offered
			if (needed) *needed = std::max(*needed, s.hFlags[2]);
		}
	}
	return GSP_OK;
}

// The compute stream waits for every enqueued exchange (device side), the host for their flags.
int gsp_exchange_finish(gsp_context* ctx, uint32_t* errorBits, uint32_t* needed)
{
	if (!ctx)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.exchange)
		return failEx(c, GSP_ERR_STATE, "gsp_exchange_finish: gsp_comm_init has not been called");
	for (auto& s : c.exchange->sets)
		if (s.used)
			GSP_CUDA(cudaStreamWaitEvent(c.stream, s.done, 0));
	return gsp_exchange_poll(ctx, 1, errorBits, needed);
}

// This rank's merged slice of list `list` of the most recently enqueued exchange (device pointers, valid until the set is
// reused two frames later): start = position of the slice in the merged list, ranks[i] = the GPU element i came from.
int gsp_get_merged_device(gsp_context* ctx, uint32_t list, const uint32_t** keys, const uint32_t** payloads, const uint8_t** ranks,
	uint32_t* start, uint32_t* count)
{
	if (!ctx || !keys || !payloads || !ranks || !start || !count)
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	if (!c.exchange || c.exchange->frameIndex == 0)
		return failEx(c, GSP_ERR_STATE, "gsp_get_merged_device: no exchange has been enqueued");
	Exchange& x = *c.exchange;
	if (list >= x.lists)
		return failEx(c, GSP_ERR_INVALID, "gsp_get_merged_device: list index out of range");
	GSP_CUDA(cudaSetDevice(c.device));
	ExchangeSet& s = x.sets[(x.frameIndex - 1) % kExSets];
	GSP_CUDA(cudaEventSynchronize(s.done));
	const uint32_t lists = x.lists, rk = x.ranks;
	std::vector<uint32_t> info(lists * 2), outOffsets(lists);
	GSP_CUDA(cudaMemcpy(info.data(), s.sliceInfo, lists * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
	GSP_CUDA(cudaMemcpy(outOffsets.data(), s.plan + 2ull * rk * lists, lists * sizeof(uint32_t), cudaMemcpyDeviceToHost));
	*keys = s.outKeys + outOffsets[list]; *payloads = s.outPays + outOffsets[list]; *ranks = s.outRanks + outOffsets[list];
	*start = info[list * 2]; *count = info[list * 2 + 1];
	return GSP_OK;
}

// Milliseconds of the last enqueued exchange's steps (gsp_exchange_set_timing): export / sampling, collective(s), merge.
int gsp_exchange_times(gsp_context* ctx, float ms[3])
{
	if (!ctx || !ms || !ctx->c.exchange || ctx->c.exchange->frameIndex == 0)
		return GSP_ERR_STATE;
	Context& c = ctx->c;
	Exchange& x = *c.exchange;
	ExchangeSet& s = x.sets[(x.frameIndex - 1) % kExSets];
	GSP_CUDA(cudaSetDevice(c.device));
	GSP_CUDA(cudaEventSynchronize(s.done));
	ms[0] = ms[1] = ms[2] = 0.0f;
	if (!x.timing)
		return GSP_OK;
	GSP_CUDA(cudaEventElapsedTime(&ms[0], s.t[0], s.t[1]));
	GSP_CUDA(cudaEventElapsedTime(&ms[1], s.t[1], s.t[2]));
	GSP_CUDA(cudaEventElapsedTime(&ms[2], s.t[2], s.t[3]));
	return GSP_OK;
}

// Copies `bytes` from a device pointer handed out by this library (merged slices, device lists) to host memory.
int gsp_copy_to_host(gsp_context* ctx, const void* devicePtr, void* host, size_t bytes)
{
	if (!ctx || (!devicePtr && bytes) || (!host && bytes))
		return GSP_ERR_INVALID;
	Context& c = ctx->c;
	GSP_CUDA(cudaSetDevice(c.device));
	if (bytes)
		GSP_CUDA(cudaMemcpy(host, devicePtr, bytes, cudaMemcpyDeviceToHost));
	return GSP_OK;
}

uint64_t gsp_exchange_bytes_received(const gsp_context* ctx)
{
	if (!ctx || !ctx->c.exchange)
		return 0;
	const Exchange& x = *ctx->c.exchange;
	return (uint64_t)(kExHeaderWords + 2ull * x.capacity) * x.ranks * sizeof(uint32_t);
}

} // extern "C"
