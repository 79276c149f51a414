"""ctypes binding of the C ABI in include/garden_sceneprep.h (libgarden_sceneprep.so).

This is the Python face of the product used by bench.py and tests/: it only marshals plain pointers and sizes.
There is no fallback path: if the library is missing, or no sm_100 GPU is usable, construction raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from .layout import RECORD_DTYPE, VIEW_DTYPE

LIB_PATH = Path(__file__).resolve().parent / "libgarden_sceneprep.so"

GSP_OK, GSP_ERR_INVALID, GSP_ERR_CUDA, GSP_ERR_NOMEM, GSP_ERR_STATE, GSP_ERR_HIERARCHY = range(6)
GSP_MAX_POOLS, GSP_MAX_VIEWS = 8, 16

# every symbol include/garden_sceneprep.h declares: name -> (restype, argtypes)
_u32, _i32, _u64, _vp = C.c_uint32, C.c_int, C.c_uint64, C.c_void_p
_pp = C.POINTER(C.c_void_p)
_pu32 = C.POINTER(C.c_uint32)
SYMBOLS = {
    "gsp_version": (C.c_char_p, []),
    "gsp_create": (_i32, [_i32, _pp]),
    "gsp_destroy": (None, [_vp]),
    "gsp_last_error": (C.c_char_p, [_vp]),
    "gsp_set_stream": (_i32, [_vp, _vp]),
    "gsp_set_transforms": (_i32, [_vp, _vp, _u32, _u32]),
    "gsp_update_transforms": (_i32, [_vp, _vp, _u32, _u32, _u32]),
    "gsp_update_transforms_indexed": (_i32, [_vp, _vp, _u32, _vp, _u32]),
    "gsp_set_pool_count": (_i32, [_vp, _u32]),
    "gsp_set_mesh_pool": (_i32, [_vp, _u32, _u32, _u32, _vp, _u32, _u32, _u32, _vp]),
    "gsp_update_mesh_pool": (_i32, [_vp, _u32, _vp, _u32, _u32, _u32, _u32, _vp]),
    "gsp_update_mesh_pool_indexed": (_i32, [_vp, _u32, _vp, _u32, _vp, _u32, _u32, _vp]),
    "gsp_set_pool_view_mask": (_i32, [_vp, _u32, _u32]),
    "gsp_set_views": (_i32, [_vp, _u32, _vp, _vp]),
    "gsp_run": (_i32, [_vp]),
    "gsp_run_async": (_i32, [_vp]),
    "gsp_sync": (_i32, [_vp]),
    "gsp_unsorted_buffer_count": (_u32, [_vp, _u32]),
    "gsp_sorted_buffer_count": (_u32, [_vp, _u32]),
    "gsp_get_unsorted": (_i32, [_vp, _u32, _u32, _pp, _pu32, _pu32]),
    "gsp_get_sorted_counts": (_i32, [_vp, _u32, _u32, _pu32, _pu32]),
    "gsp_get_sorted": (_i32, [_vp, _u32, _i32, _pp, _pu32]),
    "gsp_get_unsorted_device": (_i32, [_vp, _u32, _u32, _pp, _pu32, _pu32]),
    "gsp_get_sorted_device": (_i32, [_vp, _u32, _i32, _pp, _pu32]),
    "gsp_get_sorted_run_device": (_i32, [_vp, _u32, _i32, _u32, _pp, _pp, _pu32]),
    "gsp_list_count": (_u32, [_vp]),
    "gsp_get_list_counts": (_i32, [_vp, _vp, _u32]),
    "gsp_export_runs": (_i32, [_vp, _vp, _vp, _u32]),
    "gsp_exchange_block_words": (_u32, [_u32]),
    "gsp_merge_plan_words": (_u32, [_u32, _u32]),
    "gsp_export_runs_packed": (_i32, [_vp, _vp, _u32]),
    "gsp_merge_tree_scratch_words": (_u64, [_u32]),
    "gsp_merge_gathered_packed_tree": (_i32, [_vp, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _vp]),
    "gsp_comm_unique_id": (_i32, [_vp]),
    "gsp_comm_init": (_i32, [_vp, _vp, _u32, _u32]),
    "gsp_comm_init_all": (_i32, [_vp, _u32]),
    "gsp_comm_destroy": (_i32, [_vp]),
    "gsp_comm_info": (_i32, [_vp, _pu32, _pu32, _pu32, _pu32]),
    "gsp_exchange_configure": (_i32, [_vp, _u32]),
    "gsp_exchange_autosize": (_i32, [_vp, _pu32]),
    "gsp_exchange_async": (_i32, [_vp]),
    "gsp_exchange_poll": (_i32, [_vp, _i32, _pu32, _pu32]),
    "gsp_exchange_finish": (_i32, [_vp, _pu32, _pu32]),
    "gsp_get_merged_device": (_i32, [_vp, _u32, _pp, _pp, _pp, _pu32, _pu32]),
    "gsp_exchange_set_timing": (_i32, [_vp, _i32]),
    "gsp_exchange_times": (_i32, [_vp, _vp]),
    "gsp_exchange_bytes_received": (_u64, [_vp]),
    "gsp_copy_to_host": (_i32, [_vp, _vp, _vp, C.c_size_t]),
    "gsp_emit_instances": (_i32, [_vp, _u32, _i32, _u32, _vp, _vp, _u32, _u32, _u32]),
    "gsp_emit_instances_device": (_i32, [_vp, _u32, _i32, _u32, _vp, _vp, _u32, _u32, _u32]),
    "gsp_frustum_planes": (None, [_vp, _vp]),
    "gsp_view_from_viewproj": (_i32, [_vp, _vp, _i32, _vp]),
    "gsp_camera_view_proj": (_i32, [_vp, _vp, _vp, C.c_float, C.c_float, C.c_float, _vp, _vp, _vp]),
    "gsp_camera_view_proj_chain": (_i32, [_vp, _vp, _vp, _vp, _u32, C.c_float, C.c_float, C.c_float, _vp, _vp, _vp]),
    "gsp_camera_view_proj_ortho": (_i32, [_vp, _vp, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gsp_light_view_proj": (_i32, [_vp, _vp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _u32, _vp, _vp]),
    "gsp_cascade_views": (_i32, [_vp, _vp, C.c_float, C.c_float, C.c_float, C.c_float, _vp, _u32, C.c_float, _u32, _vp, _vp]),
    "gsp_set_active": (_i32, [_vp, _vp, _u32, _i32]),
    "gsp_writeback_active": (_i32, [_vp, _vp, _u32]),
    "gsp_animate": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _u32]),
    "gsp_writeback_trs": (_i32, [_vp, _vp, _u32]),
    "gsp_writeback_visible": (_i32, [_vp, _u32, _vp, _u32]),
    "gsp_writeback_visible_delta": (_i32, [_vp, _u32, _vp, _u32, _pu32]),
    "gsp_fetch_all": (_i32, [_vp]),
    "gsp_fetch_all_async": (_i32, [_vp]),
    "gsp_pin_host": (_i32, [_vp, C.c_size_t]),
    "gsp_unpin_host": (_i32, [_vp]),
    "gsp_download_models": (_i32, [_vp, _u32, _vp]),
    "gsp_set_profiling": (_i32, [_vp, _i32]),
    "gsp_get_phase_times": (_i32, [_vp, _vp]),
    "gsp_last_launch_count": (_u32, [_vp]),
    "gsp_last_visible_total": (_u64, [_vp]),
    "gsp_selftest_math": (_i32, [_i32, _u32, _u32, _u64, _vp]),
}


class ScenePrepError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"gsp error {code}: {message}")
        self.code = code


_lib = None


def load_library() -> C.CDLL:
    """Loads libgarden_sceneprep.so and binds every declared symbol. Raises if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise FileNotFoundError(
            f"{LIB_PATH} is missing: build it with `python -m garden_b200.build` (or __graft_entry__.build()). "
            "There is no CPU fallback for the scene-preparation path.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def _ptr(a) -> int:
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a)


def pin_host(arr: np.ndarray):
    """cudaHostRegister of a numpy buffer: the staging kernels then read it in place over PCIe."""
    rc = load_library().gsp_pin_host(arr.ctypes.data, arr.nbytes)
    if rc != GSP_OK:
        raise ScenePrepError(rc, "gsp_pin_host failed")


def unpin_host(arr: np.ndarray):
    load_library().gsp_unpin_host(arr.ctypes.data)


class ScenePrep:
    """One gsp_context. Mirrors the call sequence of MeshRenderSystem (prepareSystems -> prepareMeshes per view)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        handle = C.c_void_p()
        rc = self.lib.gsp_create(device, C.byref(handle))
        if rc != GSP_OK:
            raise ScenePrepError(rc, self.lib.gsp_last_error(None).decode())
        self.h = handle
        self.view_count = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.gsp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != GSP_OK:
            raise ScenePrepError(rc, self.lib.gsp_last_error(self.h).decode())

    # ---- staging ----
    def set_stream(self, cuda_stream: int):
        self._check(self.lib.gsp_set_stream(self.h, cuda_stream))

    def set_transforms(self, aos, stride: int, occupancy: int):
        self._check(self.lib.gsp_set_transforms(self.h, _ptr(aos), stride, occupancy))

    def update_transforms(self, aos, stride: int, first: int, count: int):
        self._check(self.lib.gsp_update_transforms(self.h, _ptr(aos), stride, first, count))

    def update_transforms_indexed(self, aos, stride: int, slots):
        slots = np.ascontiguousarray(slots, dtype=np.uint32)
        self._check(self.lib.gsp_update_transforms_indexed(self.h, _ptr(aos), stride, slots.ctypes.data, slots.size))

    def set_pool_count(self, n: int):
        self._check(self.lib.gsp_set_pool_count(self.h, n))

    def set_mesh_pool(self, pool: int, render_type: int, aos, stride: int, occupancy: int, count: int | None = None,
                      draw_ready: bool = True, ready_counts=None):
        if count is None:
            count = occupancy
        if ready_counts is not None:
            ready_counts = np.ascontiguousarray(ready_counts, dtype=np.uint8)
            assert ready_counts.size >= occupancy
        self._check(self.lib.gsp_set_mesh_pool(self.h, pool, render_type, 1 if draw_ready else 0, _ptr(aos), stride,
                                               occupancy, count, _ptr(ready_counts)))

    def update_mesh_pool(self, pool: int, aos, stride: int, first: int, count: int, component_count: int,
                         ready_counts=None):
        """Restages slots [first, first + count) of a pool set by set_mesh_pool; aos / ready_counts are the pool bases
        (numpy arrays or raw pointers, host or device)."""
        self._check(self.lib.gsp_update_mesh_pool(self.h, pool, _ptr(aos), stride, first, count, component_count,
                                                  _ptr(ready_counts)))

    def update_mesh_pool_indexed(self, pool: int, aos, stride: int, slots, component_count: int, ready_counts=None):
        """Same for a scattered set of slots (any order, duplicates allowed); aos / ready_counts are host memory."""
        slots = np.ascontiguousarray(slots, dtype=np.uint32)
        self._check(self.lib.gsp_update_mesh_pool_indexed(self.h, pool, _ptr(aos), stride, slots.ctypes.data, slots.size,
                                                          component_count, _ptr(ready_counts)))

    def set_pool_view_mask(self, pool: int, view_mask: int):
        """bit v = isDrawReady(views[v].shadowPass) of the pool's mesh system (mesh.cpp:426,482)."""
        self._check(self.lib.gsp_set_pool_view_mask(self.h, pool, view_mask & 0xFFFFFFFF))

    def set_views(self, views: np.ndarray, camera_pos):
        views = np.ascontiguousarray(views, dtype=VIEW_DTYPE)
        cam = np.ascontiguousarray(camera_pos, dtype=np.float32)
        self._check(self.lib.gsp_set_views(self.h, views.size, views.ctypes.data, cam.ctypes.data))
        self.view_count = views.size

    # ---- frame ----
    def run(self):
        self._check(self.lib.gsp_run(self.h))

    def run_async(self):
        self._check(self.lib.gsp_run_async(self.h))

    def sync(self):
        self._check(self.lib.gsp_sync(self.h))

    # ---- results ----
    def unsorted_buffer_count(self, view: int) -> int:
        return self.lib.gsp_unsorted_buffer_count(self.h, view)

    def sorted_buffer_count(self, view: int) -> int:
        return self.lib.gsp_sorted_buffer_count(self.h, view)

    def _records(self, ptr: C.c_void_p, count: int, copy: bool) -> np.ndarray:
        if count == 0 or not ptr.value:
            return np.zeros(0, dtype=RECORD_DTYPE)
        buf = (C.c_uint8 * (count * 64)).from_address(ptr.value)
        arr = np.frombuffer(buf, dtype=RECORD_DTYPE, count=count)
        return arr.copy() if copy else arr

    def get_unsorted(self, view: int, buffer: int, copy: bool = True):
        ptr, draw, inst = C.c_void_p(), C.c_uint32(), C.c_uint32()
        self._check(self.lib.gsp_get_unsorted(self.h, view, buffer, C.byref(ptr), C.byref(draw), C.byref(inst)))
        return self._records(ptr, draw.value, copy), draw.value, inst.value

    def get_sorted_counts(self, view: int, buffer: int):
        draw, inst = C.c_uint32(), C.c_uint32()
        self._check(self.lib.gsp_get_sorted_counts(self.h, view, buffer, C.byref(draw), C.byref(inst)))
        return draw.value, inst.value

    def get_sorted(self, view: int, which: int, copy: bool = True):
        ptr, draw = C.c_void_p(), C.c_uint32()
        self._check(self.lib.gsp_get_sorted(self.h, view, which, C.byref(ptr), C.byref(draw)))
        return self._records(ptr, draw.value, copy), draw.value

    def get_unsorted_device(self, view: int, buffer: int):
        ptr, draw, inst = C.c_void_p(), C.c_uint32(), C.c_uint32()
        self._check(self.lib.gsp_get_unsorted_device(self.h, view, buffer, C.byref(ptr), C.byref(draw), C.byref(inst)))
        return ptr.value, draw.value, inst.value

    def get_sorted_run_device(self, view: int, kind: int, buffer: int = 0):
        keys, pays, count = C.c_void_p(), C.c_void_p(), C.c_uint32()
        self._check(self.lib.gsp_get_sorted_run_device(self.h, view, kind, buffer, C.byref(keys), C.byref(pays),
                                                       C.byref(count)))
        return keys.value, pays.value, count.value

    def list_count(self) -> int:
        return self.lib.gsp_list_count(self.h)

    def list_counts(self) -> np.ndarray:
        n = self.list_count()
        counts = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(self.lib.gsp_get_list_counts(self.h, counts.ctypes.data, counts.size))
        return counts[:n]

    def export_runs(self, d_keys: int, d_payloads: int, capacity: int):
        self._check(self.lib.gsp_export_runs(self.h, d_keys, d_payloads, capacity))

    def export_runs_packed(self, d_block: int, capacity: int):
        """Enqueues the packed export of the frame that has just been enqueued (no host synchronisation)."""
        self._check(self.lib.gsp_export_runs_packed(self.h, d_block, capacity))

    def emit_instances(self, view: int, kind: int, buffer: int, view_proj, count: int, stride: int = 64, mvp_offset: int = 0):
        """Host instance buffer of one draw list: returns [count, stride] bytes with mvp at mvp_offset of every instance."""
        vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
        out = np.zeros((max(count, 1), stride), dtype=np.uint8)
        self._check(self.lib.gsp_emit_instances(self.h, view, kind, buffer, vp.ctypes.data, out.ctypes.data, stride, mvp_offset, count))
        return out[:count]

    def emit_instances_device(self, view: int, kind: int, buffer: int, view_proj, d_instances: int, capacity: int,
                              stride: int = 64, mvp_offset: int = 0):
        vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
        self._check(self.lib.gsp_emit_instances_device(self.h, view, kind, buffer, vp.ctypes.data, d_instances, stride,
                                                       mvp_offset, capacity))

    def set_active(self, entity_ids, active: bool):
        ids = np.ascontiguousarray(entity_ids, dtype=np.uint32)
        self._check(self.lib.gsp_set_active(self.h, ids.ctypes.data, ids.size, 1 if active else 0))

    def animate(self, entity_ids, flags, frame_a, frame_b, t):
        """TransformSystem::animateAsync on the device; frames are [n, 10] = position, scale, rotation."""
        ids = np.ascontiguousarray(entity_ids, dtype=np.uint32)
        fl = np.ascontiguousarray(flags, dtype=np.uint8)
        fa = np.ascontiguousarray(frame_a, dtype=np.float32); fb = np.ascontiguousarray(frame_b, dtype=np.float32)
        tt = np.ascontiguousarray(t, dtype=np.float32)
        assert fa.shape == (ids.size, 10) and fb.shape == (ids.size, 10) and fl.size == ids.size and tt.size == ids.size
        self._check(self.lib.gsp_animate(self.h, ids.ctypes.data, fl.ctypes.data, fa.ctypes.data, fb.ctypes.data, tt.ctypes.data, ids.size))

    def writeback_trs(self, aos, stride: int):
        self._check(self.lib.gsp_writeback_trs(self.h, _ptr(aos), stride))

    def writeback_active(self, aos, stride: int):
        self._check(self.lib.gsp_writeback_active(self.h, _ptr(aos), stride))

    def writeback_visible(self, pool: int, aos, stride: int):
        self._check(self.lib.gsp_writeback_visible(self.h, pool, _ptr(aos), stride))

    def writeback_visible_delta(self, pool: int, aos, stride: int) -> int:
        changed = C.c_uint32()
        self._check(self.lib.gsp_writeback_visible_delta(self.h, pool, _ptr(aos), stride, C.byref(changed)))
        return changed.value

    def fetch_all(self):
        self._check(self.lib.gsp_fetch_all(self.h))

    def fetch_all_async(self):
        self._check(self.lib.gsp_fetch_all_async(self.h))

    def download_models(self, pool: int, occupancy: int) -> np.ndarray:
        out = np.zeros((occupancy, 12), dtype=np.float32)
        self._check(self.lib.gsp_download_models(self.h, pool, out.ctypes.data))
        return out

    def set_profiling(self, enabled: bool):
        self._check(self.lib.gsp_set_profiling(self.h, 1 if enabled else 0))

    def phase_times(self) -> np.ndarray:
        ms = np.zeros(6, dtype=np.float32)
        self._check(self.lib.gsp_get_phase_times(self.h, ms.ctypes.data))
        return ms

    def last_launch_count(self) -> int:
        return self.lib.gsp_last_launch_count(self.h)

    def last_visible_total(self) -> int:
        return self.lib.gsp_last_visible_total(self.h)
