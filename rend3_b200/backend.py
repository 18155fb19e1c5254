"""ctypes binding of the C ABI declared in include/rend3_b200.h.

`Backend` wraps one context of a shared library exporting that ABI.  The product library is
librend3_b200.so (prefix ``r3_``); loading it is `load_cuda_backend()`.  The test suite binds
its CPU checker through the same class with another prefix — this module knows nothing about
it and never falls back to it: if the CUDA library is missing, loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from .layouts import (
    BATCH_DTYPE,
    CAMERA_HEADER_DTYPE,
    INDIRECT_CALL_DTYPE,
    OBJECT_MATRICES_DTYPE,
    REGION_DTYPE,
)

CAMERA_VIEWPORT = 0xFFFFFFFF
CB_BAKE, CB_CULL = 1, 2

_ROOT = os.path.dirname(os.path.abspath(__file__))
CUDA_LIB_PATH = os.path.join(_ROOT, "librend3_b200.so")

# every entry point of include/rend3_b200.h (tests check the .so exports all of them)
ENTRY_POINTS = [
    "abi_version", "ctx_create", "ctx_destroy", "last_error", "sync", "get_stream", "launch_count", "set_stage_timing", "stage_times", "frame_begin", "frame_end", "frame_graph_stats",
    "set_objects", "update_objects", "set_objects_device", "set_object_sort_info", "set_mesh_buffer", "set_textures", "set_skybox",
    "set_materials", "set_directional_lights", "set_point_lights", "set_frame_uniforms",
    "object_uniform_upload", "visible_count", "readback_visible", "readback_object_matrices",
    "batch_objects", "batch_counts", "readback_batches", "batching_info", "cull", "readback_indices",
    "readback_draw_calls", "readback_culling_results", "set_render_target", "clear_shadow_atlas",
    "shadow_pass", "forward_begin", "forward_pass", "hiz_build", "forward_resolve", "forward_blend", "tonemap",
    "set_parity_target", "readback_hdr_f32", "readback_hdr_f16", "readback_depth", "readback_ldr", "readback_shadow_atlas",
    "readback_hiz", "forward_stats", "forward_light_evaluations", "device_ptr", "set_scissor_rows", "skin", "readback_mesh_buffer",
    "exchange_create", "exchange_connect", "exchange_words", "exchange_merge", "exchange_merged", "exchange_count", "exchange_counts", "exchange_destroy",
    "peer_create", "peer_connect", "peer_send_atlas_rect", "peer_send_rows", "peer_signal", "peer_wait", "peer_destroy", "clear_shadow_rect", "set_cull_shard",
    "generate_mipmaps", "readback_texels", "stage_times_n",
]


class R3Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"rend3_b200 error {code}: {message}")
        self.code = code


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Backend:
    """One context.  Method names follow the C ABI one to one."""

    def __init__(self, lib: C.CDLL, prefix: str = "r3_", device: int = 0):
        self.lib, self.prefix = lib, prefix
        self.ctx = C.c_void_p()
        self._fn("last_error").restype = C.c_char_p
        self._fn("abi_version").restype = C.c_uint32
        rc = self._fn("ctx_create")(C.c_int(device), C.byref(self.ctx))
        if rc != 0:
            raise R3Error(rc, "context creation failed (no CUDA device?)")

    def _fn(self, name):
        return getattr(self.lib, self.prefix + name)

    def _call(self, name, *args):
        rc = self._fn(name)(self.ctx, *args)
        if rc != 0:
            raise R3Error(rc, (self._fn("last_error")(self.ctx) or b"?").decode())

    def close(self):
        if self.ctx:
            self._fn("ctx_destroy")(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- context
    def sync(self):
        self._call("sync")

    def stream(self) -> int:
        s = C.c_void_p()
        self._call("get_stream", C.byref(s))
        return s.value or 0

    def launch_count(self) -> int:
        n = C.c_uint64()
        self._call("launch_count", C.byref(n))
        return n.value

    STAGES = ("triangle_test", "raster_setup_colour", "raster_setup_depth", "raster_bands", "resolve", "sort", "cull_bake", "triangle_compact")

    def frame_begin(self):
        self._call("frame_begin")

    def frame_end(self):
        self._call("frame_end")

    def frame_graph_stats(self):
        s = (C.c_uint64 * 4)()
        self._call("frame_graph_stats", s)
        return {"frames": int(s[0]), "graphed": int(s[1]), "flushed": int(s[2]), "instantiations": int(s[3])}

    def set_stage_timing(self, enabled: bool = True):
        self._call("set_stage_timing", C.c_int(1 if enabled else 0))

    def stage_times(self):
        ms, n = (C.c_double * 8)(), (C.c_uint32 * 8)()
        self._call("stage_times", ms, n)
        return {name: {"ms": float(ms[i]), "launches": int(n[i])} for i, name in enumerate(self.STAGES)}

    def mipmap_stage_time(self):
        """Stage 8 of the stage timer (r3_stage_times_n): r3_generate_mipmaps calls since the last read, ms summed over them."""
        ms, n = (C.c_double * 9)(), (C.c_uint32 * 9)()
        self._call("stage_times_n", C.c_uint32(9), ms, n)
        return {"ms": float(ms[8]), "launches": int(n[8])}

    # ---- world data
    def set_objects(self, records: np.ndarray):
        records = np.ascontiguousarray(records)
        assert records.dtype.itemsize == 128
        self._call("set_objects", _ptr(records), C.c_uint32(len(records)))

    def set_objects_device(self, device_ptr: int, n_slots: int):
        self._call("set_objects_device", C.c_void_p(device_ptr), C.c_uint32(n_slots))

    def update_objects(self, slots: np.ndarray, records: np.ndarray):
        slots = np.ascontiguousarray(slots, dtype=np.uint32)
        records = np.ascontiguousarray(records)
        self._call("update_objects", _ptr(slots), _ptr(records), C.c_uint32(len(slots)))

    def set_object_sort_info(self, material_key, flags, location):
        k = np.ascontiguousarray(material_key, dtype=np.uint64)
        f = np.ascontiguousarray(flags, dtype=np.uint8)
        l = np.ascontiguousarray(location, dtype=np.float32).reshape(-1)
        assert len(f) == len(k) and len(l) == 3 * len(k)
        self._call("set_object_sort_info", _ptr(k), _ptr(f), _ptr(l), C.c_uint32(len(k)))

    def set_mesh_buffer(self, words: np.ndarray):
        words = np.ascontiguousarray(words, dtype=np.uint32)
        self._call("set_mesh_buffer", _ptr(words), C.c_uint64(words.nbytes))

    def set_materials(self, records: np.ndarray):
        records = np.ascontiguousarray(records)
        assert records.dtype.itemsize == 208
        self._call("set_materials", _ptr(records), C.c_uint32(len(records)))

    def set_textures(self, descs: np.ndarray, texels: np.ndarray):
        descs = np.ascontiguousarray(descs)
        texels = np.ascontiguousarray(texels).view(np.uint8).reshape(-1)
        assert descs.dtype.itemsize == 32
        self._call("set_textures", _ptr(descs) if len(descs) else None, C.c_uint32(len(descs)), _ptr(texels) if len(texels) else None, C.c_uint64(len(texels)))

    def generate_mipmaps(self, texture_indices):
        """MipmapGenerator::generate_mipmaps for MipmapSource::Generated textures: levels 1.. of the listed table entries from level 0 (rule R12)."""
        idx = np.ascontiguousarray(texture_indices, dtype=np.uint32).reshape(-1)
        self._call("generate_mipmaps", _ptr(idx) if len(idx) else None, C.c_uint32(len(idx)))

    def readback_texels(self, byte_offset: int, nbytes: int) -> np.ndarray:
        out = np.zeros(nbytes, dtype=np.uint8)
        self._call("readback_texels", C.c_uint64(byte_offset), _ptr(out) if nbytes else None, C.c_uint64(nbytes))
        return out

    def set_skybox(self, desc: Optional[np.ndarray], texels: Optional[np.ndarray]):
        if desc is None:
            self._call("set_skybox", None, None, C.c_uint64(0))
            return
        desc = np.ascontiguousarray(desc).reshape(1)
        texels = np.ascontiguousarray(texels).view(np.uint8).reshape(-1)
        self._call("set_skybox", _ptr(desc), _ptr(texels), C.c_uint64(len(texels)))

    def set_directional_lights(self, data: bytes, atlas_w: int, atlas_h: int):
        self._call("set_directional_lights", C.c_char_p(data), C.c_uint64(len(data)), C.c_uint32(atlas_w), C.c_uint32(atlas_h))

    def set_point_lights(self, data: bytes):
        self._call("set_point_lights", C.c_char_p(data), C.c_uint64(len(data)))

    def set_frame_uniforms(self, record: np.ndarray):
        b = record.tobytes()
        assert len(b) == 496
        self._call("set_frame_uniforms", C.c_char_p(b))

    # ---- skinning
    def skin(self, inputs: np.ndarray, joint_matrices: np.ndarray):
        inputs = np.ascontiguousarray(inputs)
        assert inputs.dtype.itemsize == 40
        jm = np.ascontiguousarray(joint_matrices, dtype=np.float32).reshape(-1, 16)
        self._call("skin", _ptr(inputs), C.c_uint32(len(inputs)), _ptr(jm), C.c_uint32(len(jm)))

    def readback_mesh_buffer(self, n_words: int) -> np.ndarray:
        out = np.empty(n_words, dtype=np.uint32)
        self._call("readback_mesh_buffer", _ptr(out), C.c_uint64(out.nbytes))
        return out

    # ---- object cull + bake
    def object_uniform_upload(self, camera: int, header: np.ndarray, mode: int = CB_BAKE | CB_CULL):
        b = header.tobytes()
        assert len(b) == CAMERA_HEADER_DTYPE.itemsize
        self._call("object_uniform_upload", C.c_uint32(camera), C.c_char_p(b), C.c_uint32(mode))

    def visible_count(self, camera: int) -> int:
        n = C.c_uint32()
        self._call("visible_count", C.c_uint32(camera), C.byref(n))
        return n.value

    def readback_visible(self, camera: int) -> np.ndarray:
        n = self.visible_count(camera)
        out = np.empty(max(n, 1), dtype=np.uint32)
        cnt = C.c_uint32()
        self._call("readback_visible", C.c_uint32(camera), _ptr(out), C.c_uint32(len(out)), C.byref(cnt))
        return out[: cnt.value]

    def readback_object_matrices(self, camera: int, first: int, n: int) -> np.ndarray:
        out = np.empty(max(n, 1), dtype=OBJECT_MATRICES_DTYPE)
        self._call("readback_object_matrices", C.c_uint32(camera), _ptr(out), C.c_uint32(first), C.c_uint32(n))
        return out[:n]

    # ---- batching + triangle cull
    def batch_objects(self, camera: int, viewport_location, max_dispatch_count: int = 65535):
        loc = np.ascontiguousarray(viewport_location, dtype=np.float32)
        self._call("batch_objects", C.c_uint32(camera), _ptr(loc), C.c_uint32(max_dispatch_count))

    def batch_counts(self, camera: int):
        a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self._call("batch_counts", C.c_uint32(camera), C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def readback_batches(self, camera: int):
        nb, nr, _ = self.batch_counts(camera)
        batches = np.zeros(max(nb, 1), dtype=BATCH_DTYPE)
        regions = np.zeros(max(nr, 1), dtype=REGION_DTYPE)
        self._call("readback_batches", C.c_uint32(camera), _ptr(batches), _ptr(regions))
        return batches[:nb], regions[:nr]

    def batching_info(self, camera: int):
        info = (C.c_uint32 * 4)()
        self._call("batching_info", C.c_uint32(camera), info)
        return {"path": {0: "none", 1: "device", 2: "host", 3: "device, frame-wide sort"}[info[0]], "overflow": int(info[1]), "batches": int(info[2]), "regions": int(info[3])}

    def cull(self, camera: int, batches: Optional[np.ndarray] = None, regions: Optional[np.ndarray] = None):
        if batches is None:
            self._call("cull", C.c_uint32(camera), None, C.c_uint32(0), None, C.c_uint32(0))
        else:
            batches, regions = np.ascontiguousarray(batches), np.ascontiguousarray(regions)
            self._call("cull", C.c_uint32(camera), _ptr(batches), C.c_uint32(len(batches)), _ptr(regions), C.c_uint32(len(regions)))

    def _readback_counted(self, name, camera, partition, dtype, count_type=C.c_uint64):
        n = count_type()
        self._call(name, C.c_uint32(camera), C.c_int(partition), None, count_type(0), C.byref(n))
        out = np.empty(max(n.value, 1), dtype=dtype)
        self._call(name, C.c_uint32(camera), C.c_int(partition), _ptr(out), count_type(len(out)), C.byref(n))
        return out[: n.value]

    def readback_indices(self, camera: int, partition: int) -> np.ndarray:
        return self._readback_counted("readback_indices", camera, partition, np.uint32)

    def readback_draw_calls(self, camera: int, partition: int) -> np.ndarray:
        return self._readback_counted("readback_draw_calls", camera, partition, INDIRECT_CALL_DTYPE, C.c_uint32)

    def readback_culling_results(self, camera: int, partition: int) -> np.ndarray:
        return self._readback_counted("readback_culling_results", camera, partition, np.uint32)

    # ---- forward
    def set_render_target(self, width: int, height: int, samples: int = 1, clear=(0, 0, 0, 0)):
        c = (C.c_float * 4)(*[float(v) for v in clear])
        self._call("set_render_target", C.c_uint32(width), C.c_uint32(height), C.c_uint32(samples), c)
        self.width, self.height = width, height

    def set_scissor_rows(self, begin: int, end: int):
        self._call("set_scissor_rows", C.c_uint32(begin), C.c_uint32(end))

    def clear_shadow_atlas(self):
        self._call("clear_shadow_atlas")

    def shadow_pass(self, index: int, ox: int, oy: int, size: int):
        self._call("shadow_pass", C.c_uint32(index), C.c_uint32(ox), C.c_uint32(oy), C.c_uint32(size))

    def forward_begin(self):
        self._call("forward_begin")

    def forward_pass(self, source: int):
        self._call("forward_pass", C.c_int(source))

    def hiz_build(self):
        self._call("hiz_build")

    def forward_resolve(self):
        self._call("forward_resolve")

    # ---- multi-GPU exchange of the visible set over NVLink peer memory
    def exchange_create(self, camera: int, n_ranks: int, my_rank: int, max_objects_per_rank: int) -> bytes:
        h = (C.c_uint8 * 64)()
        self._call("exchange_create", C.c_uint32(camera), C.c_uint32(n_ranks), C.c_uint32(my_rank), C.c_uint32(max_objects_per_rank), h)
        return bytes(h)

    def exchange_connect(self, camera: int, handles: bytes):
        buf = (C.c_uint8 * len(handles)).from_buffer_copy(handles)
        self._call("exchange_connect", C.c_uint32(camera), buf)

    def exchange_words(self, camera: int):
        p, n, w = C.c_void_p(), C.c_uint64(), C.c_uint32()
        self._call("exchange_words", C.c_uint32(camera), C.byref(p), C.byref(n), C.byref(w))
        return p.value, n.value, w.value

    def exchange_merge(self, camera: int, rank_objects, rank_base=None):
        ro = np.ascontiguousarray(rank_objects, dtype=np.uint32)
        rb = None if rank_base is None else np.ascontiguousarray(rank_base, dtype=np.uint32)
        self._call("exchange_merge", C.c_uint32(camera), _ptr(ro), _ptr(rb))

    def exchange_count(self, camera: int, rank_objects):
        ro = np.ascontiguousarray(rank_objects, dtype=np.uint32)
        self._call("exchange_count", C.c_uint32(camera), _ptr(ro))

    def exchange_counts(self, camera: int, n_ranks: int) -> np.ndarray:
        out = np.zeros(n_ranks + 1, dtype=np.uint32)
        self._call("exchange_counts", C.c_uint32(camera), _ptr(out))
        return out

    def exchange_merged(self, camera: int):
        lst, cnt, cap = C.c_void_p(), C.c_void_p(), C.c_uint64()
        self._call("exchange_merged", C.c_uint32(camera), C.byref(lst), C.byref(cnt), C.byref(cap))
        return lst.value, cnt.value, cap.value

    def exchange_destroy(self, camera: int):
        self._call("exchange_destroy", C.c_uint32(camera))

    # ---- peer-memory plumbing of the multi-GPU forward pass
    def peer_create(self, n_ranks: int, my_rank: int) -> bytes:
        h = (C.c_uint8 * 256)()
        self._call("peer_create", C.c_uint32(n_ranks), C.c_uint32(my_rank), h)
        return bytes(h)

    def peer_connect(self, handles: bytes):
        buf = (C.c_uint8 * len(handles)).from_buffer_copy(handles)
        self._call("peer_connect", buf)

    def peer_send_atlas_rect(self, ox: int, oy: int, w: int, h: int):
        self._call("peer_send_atlas_rect", C.c_uint32(ox), C.c_uint32(oy), C.c_uint32(w), C.c_uint32(h))

    def peer_send_rows(self, row_begin: int, row_end: int, root: int = -1):
        self._call("peer_send_rows", C.c_uint32(row_begin), C.c_uint32(row_end), C.c_int(root))

    def peer_signal(self, kind: int):
        self._call("peer_signal", C.c_uint32(kind))

    def peer_wait(self, kind: int, expected):
        e = np.ascontiguousarray(expected, dtype=np.uint32)
        self._call("peer_wait", C.c_uint32(kind), _ptr(e))

    def set_cull_shard(self, index: int, count: int):
        self._call("set_cull_shard", C.c_uint32(index), C.c_uint32(count))

    def peer_destroy(self):
        self._call("peer_destroy")

    def clear_shadow_rect(self, ox: int, oy: int, w: int, h: int):
        self._call("clear_shadow_rect", C.c_uint32(ox), C.c_uint32(oy), C.c_uint32(w), C.c_uint32(h))

    def forward_blend(self):
        self._call("forward_blend")

    def tonemap(self, srgb_target: bool = True):
        self._call("tonemap", C.c_int(1 if srgb_target else 0))

    def set_parity_target(self, enabled: bool = True):
        self._call("set_parity_target", C.c_int(1 if enabled else 0))

    def readback_hdr_f32(self) -> np.ndarray:
        out = np.empty((self.height, self.width, 4), dtype=np.float32)
        self._call("readback_hdr_f32", _ptr(out), C.c_uint64(out.size))
        return out

    def readback_hdr_f16(self) -> np.ndarray:
        out = np.empty((self.height, self.width, 4), dtype=np.float16)
        self._call("readback_hdr_f16", _ptr(out), C.c_uint64(out.size))
        return out

    def readback_depth(self) -> np.ndarray:
        out = np.empty((self.height, self.width), dtype=np.float32)
        self._call("readback_depth", _ptr(out), C.c_uint64(out.size))
        return out

    def readback_ldr(self) -> np.ndarray:
        out = np.empty((self.height, self.width, 4), dtype=np.uint8)
        self._call("readback_ldr", _ptr(out), C.c_uint64(out.size))
        return out

    def readback_shadow_atlas(self, w: int, h: int) -> np.ndarray:
        out = np.empty((h, w), dtype=np.float32)
        self._call("readback_shadow_atlas", _ptr(out), C.c_uint64(out.size))
        return out

    def readback_hiz(self, mip: int) -> np.ndarray:
        w, h = C.c_uint32(), C.c_uint32()
        self._call("readback_hiz", C.c_uint32(mip), None, C.c_uint64(0), C.byref(w), C.byref(h))
        out = np.empty((h.value, w.value), dtype=np.float32)
        self._call("readback_hiz", C.c_uint32(mip), _ptr(out), C.c_uint64(out.size), C.byref(w), C.byref(h))
        return out

    def forward_stats(self):
        s = (C.c_uint64 * 4)()
        self._call("forward_stats", s)
        return list(s)

    def forward_light_evaluations(self) -> int:
        n = C.c_uint64()
        self._call("forward_light_evaluations", C.byref(n))
        return n.value

    def device_ptr(self, camera: int, which: int):
        p, n = C.c_void_p(), C.c_uint64()
        self._call("device_ptr", C.c_uint32(camera), C.c_int(which), C.byref(p), C.byref(n))
        return p.value or 0, n.value


def load_cuda_library() -> C.CDLL:
    """dlopen librend3_b200.so (built in-tree by __graft_entry__.build()).  No fallback."""
    if not os.path.exists(CUDA_LIB_PATH):
        raise FileNotFoundError(
            f"{CUDA_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` first. "
            "rend3_b200 has no CPU fallback."
        )
    return C.CDLL(CUDA_LIB_PATH)


def load_cuda_backend(device: int = 0, parity_target: Optional[bool] = None) -> Backend:
    """`parity_target` switches the library's rgba32f parity instrumentation on (r3_set_parity_target); left at None it follows the
    R3_PARITY_TARGET environment variable, which only the test suite sets — bench.py and the tools run the production configuration."""
    b = Backend(load_cuda_library(), "r3_", device)
    if parity_target is None:
        parity_target = os.environ.get("R3_PARITY_TARGET", "0") not in ("", "0")
    if parity_target:
        b.set_parity_target(True)
    return b
