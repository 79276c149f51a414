/* garden_sceneprep.h — C ABI of the B200 scene-preparation library (libgarden_sceneprep.so).
 *
 * Drop-in boundary for ONE path of cfnptr/garden: the body of
 *     MeshRenderSystem::prepareMeshes(const Frustum&, const Frustum*, f32x4 cameraOffset, int8 shadowPass)
 *     (reference: source/system/render/mesh.cpp:331-553, callers mesh.cpp:815,869,902)
 * and everything it calls per component (TransformComponent::calcModel, isBehindFrustum, the distance key, the thread-local
 * compaction and the std::sort of the draw lists), hoisted so that all views of a frame run in one call.
 *
 * Plain pointers and sizes only; no C++ or torch types cross this boundary; no exceptions (status codes + gsp_last_error).
 * One caller thread per context; calls are synchronous from the caller's view unless stated otherwise.
 * There is NO CPU fallback: every entry point that computes fails with GSP_ERR_CUDA if no sm_100 device is usable.
 *
 * The reference-side binding a maintainer would add is shown in INTEGRATION.md.
 */
#ifndef GARDEN_SCENEPREP_H
#define GARDEN_SCENEPREP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSP_MAX_POOLS 8   /* mesh systems per context (IMeshRenderSystem group members) */
#define GSP_MAX_VIEWS 16  /* views per frame (main camera + shadow passes + probes) */

typedef enum gsp_status
{
	GSP_OK = 0,
	GSP_ERR_INVALID = 1,  /* bad argument */
	GSP_ERR_CUDA = 2,     /* CUDA runtime / device error (see gsp_last_error) */
	GSP_ERR_NOMEM = 3,    /* host or device allocation failed */
	GSP_ERR_STATE = 4,    /* call sequence error (e.g. gsp_run before gsp_set_views) */
	GSP_ERR_HIERARCHY = 5 /* a parent entity has no TransformComponent (gsp_set_transforms; the reference throws EcsmError
	                         from Manager::get, ecsm.hpp:863-873), or the hierarchy is cyclic (gsp_run, gsp_set_active,
	                         gsp_animate). Acyclic chains of any depth are valid. */
} gsp_status;

/* MeshRenderType — include/garden/system/render/mesh.hpp:30-40 (same numeric values). */
typedef enum gsp_render_type
{
	GSP_RT_COLOR = 0, GSP_RT_OPAQUE = 1, GSP_RT_TRANSLUCENT = 2, GSP_RT_OIT = 3,
	GSP_RT_REFRACTED = 4, GSP_RT_TRANS_DEPTH = 5, GSP_RT_UI = 6
} gsp_render_type;

/* Draw-list record: byte-identical to MeshRenderSystem::UnsortedMesh / SortedMesh
 * (include/garden/system/render/mesh.hpp:191-205): 64 bytes, bakedModel = float4x3 column-major (c0..c3, lanes xyz).
 * bufferIndex is only meaningful in the translucent / UI lists (SortedMesh); it is 0 in unsorted buffers. */
typedef struct gsp_record
{
	uint64_t componentOffset; /* slot * componentStride, mesh.cpp:170,248 */
	float bakedModel[12];
	float distanceSq;
	uint32_t bufferIndex;
} gsp_record;

/* One view = one reference prepareMeshes() call. Planes are what math::Frustum holds after Frustum(viewProj)
 * (libraries/math/include/math/frustum.hpp:51-61): normal xyz + distance, unnormalised, computed by the caller. */
typedef struct gsp_view
{
	float planes[6][4];
	uint32_t planeCount;     /* Frustum::getPlaneCount(), 1..6 */
	float uiPlanes[6][4];    /* the `uiFrustum` argument; used for UI mesh systems in the main view only */
	uint32_t uiPlaneCount;   /* 0 = nullptr */
	float cameraOffset[4];   /* the `cameraOffset` argument (zero for the main view, csm.cpp:304 for a cascade) */
	int32_t shadowPass;      /* the `shadowPass` argument: < 0 main view (writes isVisible), >= 0 shadow pass */
} gsp_view;

typedef struct gsp_context gsp_context;

/* ---- lifetime -------------------------------------------------------------------------------------------------- */
/* Creates a context on CUDA device `device`. Replaces MeshRenderSystem's constructor-time state (mesh.cpp:31-36).
 * Buffers of MeshRenderType::OIT systems are filled but left unsorted, as in sortMeshes (mesh.cpp:273-277). */
int gsp_create(int device, gsp_context** out);
void gsp_destroy(gsp_context* ctx);
/* Last error message of this context (never NULL). With ctx == NULL: the message of the last failed gsp_create. */
const char* gsp_last_error(const gsp_context* ctx);
/* All work of this context is enqueued on `cudaStream` (a cudaStream_t; NULL = the context's own stream). */
int gsp_set_stream(gsp_context* ctx, void* cudaStream);

/* ---- component staging (AoS ECS pools -> SoA in HBM) ------------------------------------------------------------ */
/* Replaces the per-entity Manager::tryGet<TransformComponent>() + field reads (mesh.cpp:149; ecsm.hpp:898-905).
 * `aos` = LinearPool<TransformComponent>::getData() (linear-pool.hpp:717), `stride` = sizeof(TransformComponent) = 80
 * (include/garden/system/transform.hpp:31-60), `occupancy` = getOccupancy() (linear-pool.hpp:734).
 * The memory is consumed during the call and may change afterwards. Pinned / registered host memory (cudaMallocHost,
 * cudaHostRegister, gsp_pin_host) is read IN PLACE over PCIe by the staging kernel (no intermediate device buffer, the
 * AoS -> SoA re-layout overlaps the transfer); device pointers are read in place; pageable memory is copied to a device
 * scratch buffer first (slower: the driver stages it). */
int gsp_set_transforms(gsp_context* ctx, const void* aos, uint32_t stride, uint32_t occupancy);
/* Dirty range: re-stages position/rotation/scale/active flags of slots [first, first+count); `aos` is the pool base
 * (same pointer meaning as gsp_set_transforms), only the bytes of the range are read and uploaded. The hierarchy
 * (entity and parent fields) must be unchanged since the last gsp_set_transforms. The ECS has no dirty tracking
 * (transform.hpp:74-104 are plain stores), so the range comes from the caller. */
int gsp_update_transforms(gsp_context* ctx, const void* aos, uint32_t stride, uint32_t first, uint32_t count);
/* Same for a SCATTERED dirty set (e.g. the animated tenth of configuration C3): `slots[count]` are transform-pool slot
 * indices, `aos` is the pool base. Only those components travel (packed into one pinned upload by the library). */
int gsp_update_transforms_indexed(gsp_context* ctx, const void* aos, uint32_t stride, const uint32_t* slots, uint32_t count);
/* Declares how many mesh systems the frame has (meshSystems.size() after prepareSystems, mesh.cpp:69-108). */
int gsp_set_pool_count(gsp_context* ctx, uint32_t poolCount);
/* Replaces reading IMeshRenderSystem::{getMeshRenderType,getMeshComponentPool,getMeshComponentSize,isDrawReady}
 * (mesh.hpp:60-147) inside prepareMeshes. `pool` is the index in meshSystems order. `count` = getCount()
 * (linear-pool.hpp:729). `readyCounts` (nullable, `occupancy` bytes) carries the result of a system's
 * getReadyMeshesAsync override beyond the frustum test (e.g. sprite.cpp:90-97): ready instance count per slot. */
int gsp_set_mesh_pool(gsp_context* ctx, uint32_t pool, uint32_t renderType, uint32_t drawReady, const void* aos,
	uint32_t stride, uint32_t occupancy, uint32_t count, const uint8_t* readyCounts);
/* MeshRenderComponent changes (mesh.hpp:45-55: entity, isEnabled, isVisible, aabb) of slots [first, first + count) of a pool
 * staged by gsp_set_mesh_pool: a mesh hidden or shown, a box swapped, a sprite that became ready, a component destroyed
 * (entity = 0) or a freed slot reused by an entity that already has a transform. `aos` and `readyCounts` are the pool /
 * ready-count bases (same meaning as gsp_set_mesh_pool); only the listed slots are read, from pinned, device or pageable memory
 * as in gsp_set_transforms. componentCount = LinearPool::getCount() after the change (linear-pool.hpp:729).
 * Every result afterwards is what a context would give that had staged the same bytes with gsp_set_mesh_pool, but the pool is
 * not re-uploaded and the next frame does not relink: a grown box widens its hierarchy's prepass sphere in place, a shrunken
 * or moved box keeps the larger sphere (only a gsp_set_mesh_pool or gsp_set_transforms tightens it again). Like
 * gsp_set_mesh_pool, the call ends the frame's results (gsp_writeback_visible* are no-ops until the next run), keeps a
 * gsp_fetch_all_async snapshot unless componentCount changes between zero and non-zero (a new list layout), and takes the
 * library's copy of the host's isVisible byte of the listed slots from the uploaded bytes.
 * GSP_ERR_STATE: the pool was never set. GSP_ERR_INVALID: pool >= GSP_MAX_POOLS, a stride other than the staged one, a slot at
 * or past the staged occupancy (growing it is gsp_set_mesh_pool's), readyCounts given for a pool staged without ready counts
 * or the reverse, a null pointer with count > 0. A refused call changes nothing. These checks come first: a call that passes
 * them with count == 0 is a no-op (so a range must still start at or below the occupancy, and the pool must have been set,
 * as for gsp_update_transforms). */
int gsp_update_mesh_pool(gsp_context* ctx, uint32_t pool, const void* aos, uint32_t stride, uint32_t first, uint32_t count,
	uint32_t componentCount, const uint8_t* readyCounts);
/* Same for a scattered set: slots[count] (any order, duplicates allowed). `aos`, `slots` and `readyCounts` are host memory
 * (a device pointer is refused with GSP_ERR_INVALID); the listed components travel packed in one pinned upload. */
int gsp_update_mesh_pool_indexed(gsp_context* ctx, uint32_t pool, const void* aos, uint32_t stride, const uint32_t* slots,
	uint32_t count, uint32_t componentCount, const uint8_t* readyCounts);
/* IMeshRenderSystem::isDrawReady(shadowPass) is asked once per prepareMeshes call, i.e. per VIEW (mesh.cpp:426,482), and
 * systems answer per kind of pass: InstanceRenderSystem checks the base pipeline for shadowPass < 0 and the shadow pipeline
 * otherwise (source/system/render/instance.cpp:61-113; createShadowPipeline() returns {} by default), UiLabelSystem returns
 * false for every shadow pass (source/system/ui/label.cpp:262-265). Bit v of `viewMask` = isDrawReady(views[v].shadowPass)
 * for the views of gsp_set_views; a pool takes part in view v iff drawReady (gsp_set_mesh_pool) != 0 AND bit v is set.
 * The mask persists across gsp_set_mesh_pool calls until it is set again; the default is all ones. */
int gsp_set_pool_view_mask(gsp_context* ctx, uint32_t pool, uint32_t viewMask);

/* Page-locks and maps `bytes` of caller memory (e.g. a LinearPool's storage after it (re)allocates, linear-pool.hpp:620-628)
 * so that gsp_set_* / gsp_update_transforms read it in place. Already-registered ranges are accepted. Process-wide. */
int gsp_pin_host(void* ptr, size_t bytes);
int gsp_unpin_host(void* ptr);

/* ---- per frame ---------------------------------------------------------------------------------------------------- */
/* cameraPosition = CommonConstants::cameraPos (mesh.cpp:401), shared by every view of the frame. */
int gsp_set_views(gsp_context* ctx, uint32_t viewCount, const gsp_view* views, const float cameraPosition[3]);
/* Runs the whole frame on the device: world matrices, culling for every view, keys, compaction, sort, record
 * emission. Results stay in HBM until fetched. Returns after the work has been enqueued AND completed. */
int gsp_run(gsp_context* ctx);
/* Same, but only enqueues (no host synchronisation); pair with gsp_sync. Used for device-side timing. */
int gsp_run_async(gsp_context* ctx);
int gsp_sync(gsp_context* ctx);

/* ---- results (replace reading unsortedBuffers / transSortedMeshes / uiSortedMeshes, mesh.cpp:556-770) ------------ */
uint32_t gsp_unsorted_buffer_count(const gsp_context* ctx, uint32_t view);
uint32_t gsp_sorted_buffer_count(const gsp_context* ctx, uint32_t view);
/* unsortedBuffers[buffer]->{combinedMeshes, drawCount, instanceCount}. `records` receives a pointer to pinned host
 * memory owned by the library, valid until the next gsp_run / gsp_destroy; the list is downloaded on first request. */
int gsp_get_unsorted(gsp_context* ctx, uint32_t view, uint32_t buffer, const gsp_record** records,
	uint32_t* drawCount, uint32_t* instanceCount);
/* Downloads every list of the frame that has not travelled yet: all copies are enqueued back to back with ONE host
 * synchronisation (gsp_get_unsorted / gsp_get_sorted afterwards return pointers without further copies). */
int gsp_fetch_all(gsp_context* ctx);
/* Same, but only enqueues the copies (on the context's copy stream, ordered after the frame): the transfer overlaps whatever
 * the caller does next, e.g. gsp_writeback_visible. The first gsp_get_unsorted / gsp_get_sorted (or gsp_fetch_all) waits.
 * The call also takes a SNAPSHOT of the frame's lists: the list getters keep serving it while the inputs of the NEXT frame are
 * staged (gsp_set_transforms / gsp_update_transforms* / gsp_set_mesh_pool / gsp_set_views with the same shape), so the lists
 * of frame k travel to the host while frame k+1 is uploaded — the renderer consumes frame k meanwhile, as the reference's
 * render passes do after prepareMeshes. The snapshot ends with the next gsp_run[_async] or any change of the list layout
 * (pool count, a pool's capacity or render type, the number or kind of views). */
int gsp_fetch_all_async(gsp_context* ctx);
/* sortedBuffers[buffer]->{drawCount, instanceCount} */
int gsp_get_sorted_counts(gsp_context* ctx, uint32_t view, uint32_t buffer, uint32_t* drawCount, uint32_t* instanceCount);
/* which = 0: transSortedMeshes / transDrawIndex, which = 1: uiSortedMeshes / uiDrawIndex */
int gsp_get_sorted(gsp_context* ctx, uint32_t view, int which, const gsp_record** records, uint32_t* drawCount);
/* Device-resident variants (no copy): `records` receives a device pointer (for CUDA/Vulkan interop consumers). */
int gsp_get_unsorted_device(gsp_context* ctx, uint32_t view, uint32_t buffer, const gsp_record** records,
	uint32_t* drawCount, uint32_t* instanceCount);
int gsp_get_sorted_device(gsp_context* ctx, uint32_t view, int which, const gsp_record** records, uint32_t* drawCount);
/* Sorted (key, payload) runs of one list on the device, before record emission: keys are the radix keys
 * (ascending order == draw order), payload = pool << 28 | slot. Used by the multi-GPU gather + merge. */
int gsp_get_sorted_run_device(gsp_context* ctx, uint32_t view, int listKind, uint32_t buffer,
	const uint32_t** keys, const uint32_t** payloads, uint32_t* count);
/* ---- multi-GPU exchange (no reference counterpart: one process, one std::sort per list) ---------------------------- */
/* Number of draw lists of the frame, in (view, meshSystems order) with the shared translucent / UI lists counted once. */
uint32_t gsp_list_count(const gsp_context* ctx);
/* Length of every list of the last completed frame (`capacity` >= gsp_list_count entries). */
int gsp_get_list_counts(gsp_context* ctx, uint32_t* counts, uint32_t capacity);
/* Packs the sorted (key, payload) runs of all lists back to back into caller-provided DEVICE buffers (list l follows list
 * l - 1, lengths as gsp_get_list_counts). Enqueued on the context's stream. */
int gsp_export_runs(gsp_context* ctx, uint32_t* dKeys, uint32_t* dPayloads, uint32_t capacity);
/* The multi-GPU exchange step without host synchronisation. A frame only has to be ENQUEUED (gsp_run_async): list lengths
 * are read on the device. Every rank fills one fixed-capacity block
 *   [0, 256) header { magic, lists, total, capacity, overflow, 0, 0, 0, count[lists] } | keys[capacity] | payloads[capacity]
 * (gsp_exchange_block_words(capacity) 32-bit words) with gsp_export_runs_packed, and ONE all-gather of equal blocks moves
 * everything. */
uint32_t gsp_exchange_block_words(uint32_t capacityElems);
uint32_t gsp_merge_plan_words(uint32_t ranks, uint32_t lists);
int gsp_export_runs_packed(gsp_context* ctx, uint32_t* dBlock, uint32_t capacityElems);
/* K-way merge of the `ranks` gathered blocks (block r at r * gsp_exchange_block_words(capacityElems) words): this rank merges
 * ITS key range of every list (splitters = quantiles of the longest run, identical on every rank) with a pairwise
 * merge-path tree, ceil(log2 ranks) passes over its slice; what gsp_exchange_async uses. The merge plans itself from the
 * gathered headers. All pointers are device pointers. dPlan = gsp_merge_plan_words(ranks, lists) words of device scratch;
 * its last 8 words are flags the caller reads back whenever convenient: { error bits (1 a block overflowed its capacity,
 * 2 bad header, 4 merged lists exceed outCapacity), merged total, largest per-rank total, 0... }. With a non-zero error
 * word nothing was merged: grow the capacity to hold flags[2] (or outCapacity to hold flags[1]) and repeat the frame.
 * dSliceInfo: [lists][2] out = (global position of my slice, slice length); dOutKeys/dOutPayloads/dOutRanks: my slices,
 * list l at the merged list's offset (plan words [2 * ranks * lists, + lists)). Ties resolve to (rank, payload) order.
 * dScratch = gsp_merge_tree_scratch_words(outCapacity) 32-bit words. Refused (GSP_ERR_INVALID) when ranks exceeds 32,
 * lists exceeds 248, lists * ceil(ranks / 2) exceeds 2048 (every layout of up to 128 lists at 32 ranks fits), or the
 * gathered blocks reach 2^32 words: (256 + 2 * capacityElems) * ranks >= 2^32. */
uint64_t gsp_merge_tree_scratch_words(uint32_t outCapacity);
int gsp_merge_gathered_packed_tree(void* cudaStream, uint32_t ranks, uint32_t myRank, uint32_t lists, uint32_t capacityElems,
	const uint32_t* dGathered, uint32_t* dPlan, uint32_t* dSliceInfo, uint32_t* dOutKeys, uint32_t* dOutPayloads,
	uint8_t* dOutRanks, uint32_t outCapacity, uint32_t* dScratch);

/* ---- the same exchange with NCCL inside the library: one context per GPU, any host language ------------------------------------
 * (SURVEY.md 8b: "one context may drive 1-8 GPUs" — here: n contexts, one per device, joined by one communicator.)
 * Process-per-GPU: rank 0 calls gsp_comm_unique_id, the id travels out of band (MPI, a socket, torch.distributed), every rank
 * calls gsp_comm_init. Single process: gsp_comm_init_all over its contexts; then drive every context from its own thread (NCCL's
 * rule for several devices per process). libnccl.so.2 is loaded at run time on the first call; single-GPU users never need it.
 * Per frame:  gsp_run_async(ctx); gsp_exchange_async(ctx);  — no host synchronisation, frame k's exchange (exchange stream)
 * overlaps frame k+1. The blocks have a fixed capacity (gsp_exchange_autosize measures one frame; collective): a frame whose
 * runs do not fit is flagged, nothing of it is merged, gsp_exchange_poll / _finish report it with the capacity that would
 * have sufficed; the caller then calls gsp_exchange_configure (same value on every rank) and repeats the frame.
 * GSP_EXCHANGE=allgather|alltoall selects the protocol (default alltoall: runs are cut by common, sample-based splitters
 * before they travel, every rank receives only the key range it merges: two collectives per frame — a small all-gather of
 * samples and grouped send/recv of the sub-blocks, whose headers also carry where each slice starts; falls back to allgather
 * beyond 124 lists). Both protocols merge with gsp_merge_gathered_packed_tree's merge-path tree. */
#define GSP_COMM_ID_BYTES 128
int gsp_comm_unique_id(uint8_t id[GSP_COMM_ID_BYTES]);
int gsp_comm_init(gsp_context* ctx, const uint8_t id[GSP_COMM_ID_BYTES], uint32_t ranks, uint32_t rank);
int gsp_comm_init_all(gsp_context** contexts, uint32_t count);
int gsp_comm_destroy(gsp_context* ctx);
int gsp_comm_info(const gsp_context* ctx, uint32_t* ranks, uint32_t* rank, uint32_t* capacity, uint32_t* allToAll);
int gsp_exchange_configure(gsp_context* ctx, uint32_t capacityElems);
int gsp_exchange_autosize(gsp_context* ctx, uint32_t* capacityOut);
int gsp_exchange_async(gsp_context* ctx);
/* errorBits: 1 a block overflowed, 2 bad header, 4 merged lists exceed the output capacity. wait != 0: blocks until every
 * enqueued exchange has finished. gsp_exchange_finish additionally makes the context's stream wait for them. */
int gsp_exchange_poll(gsp_context* ctx, int wait, uint32_t* errorBits, uint32_t* neededCapacity);
int gsp_exchange_finish(gsp_context* ctx, uint32_t* errorBits, uint32_t* neededCapacity);
/* This rank's key-range slice of merged list `list` (gsp_list_count order) of the most recent exchange: device pointers,
 * valid until two more exchanges have been enqueued. start = position of the slice in the merged list; ranks[i] = the GPU
 * element i came from; payload = pool << 28 | slot ON THAT GPU. Ties resolve to (rank, payload) order. */
int gsp_get_merged_device(gsp_context* ctx, uint32_t list, const uint32_t** keys, const uint32_t** payloads, const uint8_t** ranks,
	uint32_t* start, uint32_t* count);
int gsp_exchange_set_timing(gsp_context* ctx, int enabled);
/* ms = { export / sampling, collective(s), merge } of the most recent exchange (needs gsp_exchange_set_timing) */
int gsp_exchange_times(gsp_context* ctx, float ms[3]);
uint64_t gsp_exchange_bytes_received(const gsp_context* ctx);
/* Device -> host copy of memory this library handed out as a device pointer (merged slices, device-resident lists). */
int gsp_copy_to_host(gsp_context* ctx, const void* devicePtr, void* host, size_t bytes);

/* ---- the callers either side of the path (SURVEY.md 8f) ----------------------------------------------------------------- */
/* Instance data of one draw list, in draw order: for record i, mvp = (float4x4)(viewProj * f32x4x4(bakedModel, (0,0,0,1)))
 * stored at instances + i * stride + mvpOffset (64 bytes, column-major) — what renderUnsorted / renderSorted pass to
 * IMeshRenderSystem::drawAsync and every setInstanceData stores first (mesh.cpp:600-603,632-635, sprite.cpp:122-130;
 * instanceIndex == drawIndex for the default getInstancesAsync() == 1). viewProj: 16 floats, column-major.
 * listKind: 0 = unsortedBuffers[buffer], 1 = transSortedMeshes, 2 = uiSortedMeshes. stride and mvpOffset are multiples of 16.
 * At most `capacity` instances are written. The host variant needs a completed gsp_run; the device variant only needs the
 * frame to be enqueued (the draw count is read on the device) and leaves the result in caller-owned device memory, e.g. a
 * Vulkan buffer imported as CUDA external memory. */
int gsp_emit_instances(gsp_context* ctx, uint32_t view, int listKind, uint32_t buffer, const float* viewProj, void* instances,
	uint32_t stride, uint32_t mvpOffset, uint32_t capacity);
int gsp_emit_instances_device(gsp_context* ctx, uint32_t view, int listKind, uint32_t buffer, const float* viewProj,
	void* dInstances, uint32_t stride, uint32_t mvpOffset, uint32_t capacity);
/* View setup helpers (host code, no context): Frustum(viewProj) (libraries/math/include/math/frustum.hpp:51-61) — the six
 * unnormalised planes [6][4] of a column-major view-projection matrix, Vulkan Y flip included — and a gsp_view filled from a
 * viewProj the way the callers of prepareMeshes build their arguments (mesh.cpp:815,869,902; no UI frustum). */
void gsp_frustum_planes(const float* viewProj, float* planes);
int gsp_view_from_viewproj(const float* viewProj, const float* cameraOffset, int32_t shadowPass, gsp_view* view);
/* The matrices themselves, in the reference's float operation order (host code; csrc/viewsetup.cu), so that a caller that hands
 * over camera parameters instead of planes gets the reference's planes bit for bit. All matrices: 16 floats, column-major.
 *   gsp_camera_view_proj   GraphicsSystem::prepareCommonConstants for a perspective camera without a parent entity
 *                          (source/system/graphics.cpp:168-172,192-203,241; camera.hpp:111-121): the camera-relative view
 *                          (translation zeroed), calcPerspProjInfRevZ, viewProj = projection * view
 *   gsp_camera_view_proj_chain  the same for a camera WITH ancestors: calcRelativeView (graphics.cpp:173-189) multiplies
 *                          calcModel(ancestor) onto the view, nearest ancestor first; parents[i] = { position xyz, rotation
 *                          xyzw, scale xyz } (10 floats per ancestor)
 *   gsp_camera_view_proj_ortho  the same for an orthographic CameraComponent: calcOrthoProjRevZ(width, height, depth)
 *                          (camera.hpp:119-120, matrix/projection.hpp:92-99); ancestors as above (parentCount may be 0)
 *   gsp_light_view_proj    calcLightViewProj (source/system/render/csm.cpp:260-308): cascade viewProj + cameraOffset for the
 *                          camera sub-frustum [nearPlane, farPlane]
 *   gsp_cascade_views      CsmRenderSystem::prepareShadowRender for passes 0 .. cascadeCount-1 (csm.cpp:311-329): `splits`
 *                          holds cascadeCount-1 fractions of shadowDistance (csm.hpp:89); fills views[i] (planes, offset,
 *                          shadowPass = i) and, if not NULL, viewProjs[i][16] */
int gsp_camera_view_proj(const float* position, const float* rotation, const float* scale, float fieldOfView, float aspectRatio,
	float nearPlane, float* view, float* projection, float* viewProj);
int gsp_camera_view_proj_chain(const float* position, const float* rotation, const float* scale, const float* parents,
	uint32_t parentCount, float fieldOfView, float aspectRatio, float nearPlane, float* view, float* projection, float* viewProj);
int gsp_camera_view_proj_ortho(const float* position, const float* rotation, const float* scale, const float* parents,
	uint32_t parentCount, const float width[2], const float height[2], const float depth[2], float* view, float* projection,
	float* viewProj);
int gsp_light_view_proj(const float* view, const float* lightDir, float fieldOfView, float aspectRatio, float nearPlane, float farPlane,
	float zCoeff, uint32_t shadowMapSize, float* viewProj, float* cameraOffset);
int gsp_cascade_views(const float* view, const float* lightDir, float fieldOfView, float aspectRatio, float cameraNear,
	float shadowDistance, const float* splits, uint32_t cascadeCount, float zCoeff, uint32_t shadowMapSize, gsp_view* views,
	float* viewProjs);
/* TransformComponent::setActive(active) (source/system/transform.cpp:75-127) for `count` entities (1-based ECS ids) on the
 * staged hierarchy: selfActive is set, ancestorsActive is re-derived for every transform (AND of its ancestors' selfActive,
 * the invariant every setActive call maintains), and the next gsp_run filters on the new isActive() values.
 * gsp_writeback_active stores the resulting selfActive / ancestorsActive bytes (offsets 72 / 73) into the caller's pool.
 * A later gsp_set_transforms / gsp_update_transforms re-reads these bytes from the caller's memory. */
int gsp_set_active(gsp_context* ctx, const uint32_t* entityIds, uint32_t count, int active);
/* TransformSystem::animateAsync (source/system/transform.cpp:609-623; AnimationSystem::update, animation.cpp:155-190) for
 * `count` entities (1-based ECS ids, each listed once) on the staged transforms — the keyframe pair never becomes an upload of
 * whole components. flags[i]: bit 0 animatePosition, 1 animateScale, 2 animateRotation, 3 animateIsActive, 4 frameA.isActive,
 * 5 frameB.isActive; frameA / frameB: [count][10] floats = position xyz, scale xyz, rotation xyzw; t[count].
 * position / scale = lerp, bit-exact (a * (1 - t) + b * t, simd/vector/float.hpp:1469); rotation = slerp (quaternion.hpp:175-193):
 * same branches and operation order, but acosf / sinf are the device's (<= 2 ulp each) where the reference calls the host
 * libm: components agree within 4e-6 for unit quaternions (tests/test_gpu_next.py states and checks it); isActive =
 * setActive(round(t) ? b.isActive : a.isActive) with the semantics of gsp_set_active.
 * gsp_writeback_trs stores position / scale / rotation of every live transform into the caller's pool (bytes 16-27, 32-43,
 * 48-63), gsp_writeback_active the flags. */
int gsp_animate(gsp_context* ctx, const uint32_t* entityIds, const uint8_t* flags, const float* frameA, const float* frameB,
	const float* t, uint32_t count);
int gsp_writeback_trs(gsp_context* ctx, void* aos, uint32_t stride);
int gsp_writeback_active(gsp_context* ctx, void* aos, uint32_t stride);

/* Stores MeshRenderComponent::isVisible (offset 15) for every slot of `pool` exactly as the reference's main-view pass
 * does (mesh.cpp:144-146,152-153,161-167). No-op for pools the main view did not process. */
int gsp_writeback_visible(gsp_context* ctx, uint32_t pool, void* aos, uint32_t stride);
/* Same result, but only the slots whose value differs from the byte the HOST holds are transferred and stored. The library
 * knows that byte for every slot: it was uploaded with the pool by the last gsp_set_mesh_pool, or written by the previous
 * gsp_writeback_visible[_delta]. Precondition: `aos` is that pool and nobody else changed its isVisible bytes since.
 * `changed` (nullable) receives the number of bytes stored. */
int gsp_writeback_visible_delta(gsp_context* ctx, uint32_t pool, void* aos, uint32_t stride, uint32_t* changed);
/* World matrices (TransformComponent::calcModel(cameraPosition), transform.hpp:197-214) of pool slots as float4x3,
 * valid for slots that were visible in at least one view of the last frame. `out` = occupancy * 12 floats on the host. */
int gsp_download_models(gsp_context* ctx, uint32_t pool, float* out);

/* ---- introspection for benchmarks --------------------------------------------------------------------------------- */
/* Per-phase device timing with CUDA events recorded on the context's stream around each kernel group of gsp_run.
 * Phases: 0 link (entity -> transform slot, only after structural changes), 1 world matrices + culling (kCull, all pools),
 * 2 compaction + keys + sort histograms (kScanChunks + kScatter), 3 unused (always 0), 4 sort passes, 5 record emission. */
#define GSP_PHASE_COUNT 6
int gsp_set_profiling(gsp_context* ctx, int enabled);
/* Milliseconds of each phase of the last completed gsp_run (zeros when profiling is off). `ms` = GSP_PHASE_COUNT floats. */
int gsp_get_phase_times(gsp_context* ctx, float* ms);
/* Number of CUDA kernels the last gsp_run launched. */
uint32_t gsp_last_launch_count(const gsp_context* ctx);
/* Sum over views and lists of drawCount for the last frame (needs results to be complete). */
uint64_t gsp_last_visible_total(gsp_context* ctx);
/* Device self-test of the exact-arithmetic shortcuts of the hot kernel (shared-reciprocal division, sqrt fast path, packed
 * 4x3 products): `blocks` x 256 threads x `iterations` random / adversarial TRS inputs run through the shortcut and through
 * the reference's 4-lane IEEE operation order, compared bit for bit on the device.
 * results = { inputs tested, inputs that took the shortcut, shortcut mismatches, matrix products tested, product mismatches }. */
int gsp_selftest_math(int device, uint32_t blocks, uint32_t iterations, uint64_t seed, uint64_t results[5]);
/* Library version string, e.g. "garden_sceneprep 0.1 sm_100a". */
const char* gsp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GARDEN_SCENEPREP_H */
