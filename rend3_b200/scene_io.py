"""Scene files for the C++ host driver (rend3_b200/host/r3_frame.cpp): the bytes the engine's managers hand to the routines for one
target — object / material / light buffers, the PerCameraUniform header of every camera, FrameUniforms.  Sections are
u32 tag_len | tag | u64 nbytes | payload."""
from __future__ import annotations

import struct
from typing import Dict, Tuple

import numpy as np

from .backend import CAMERA_VIEWPORT
from .routines import BaseRenderGraphSettings, frame_uniforms, per_camera_header
from .world import EvalOutput


def _section(f, tag: str, payload: bytes):
    f.write(struct.pack("<I", len(tag)))
    f.write(tag.encode())
    f.write(struct.pack("<Q", len(payload)))
    f.write(payload)


def dump_scene(path: str, ev: EvalOutput, resolution: Tuple[int, int], samples: int = 1,
               settings: BaseRenderGraphSettings = BaseRenderGraphSettings(), srgb_target: bool = True, frames: int = 1):
    n = len(ev.object_buffer)
    flags = ((ev.object_live & 1) | ((ev.object_atomic & 1) << 1) | ((ev.object_back_to_front & 1) << 2)).astype(np.uint8)
    with open(path, "wb") as f:
        _section(f, "objects", np.ascontiguousarray(ev.object_buffer).tobytes())
        _section(f, "material_key", np.ascontiguousarray(ev.object_material_key, dtype=np.uint64).tobytes())
        _section(f, "sort_flags", flags.tobytes())
        _section(f, "location", np.ascontiguousarray(ev.object_location, dtype=np.float32).tobytes())
        _section(f, "mesh", np.ascontiguousarray(ev.mesh_buffer).tobytes())
        _section(f, "materials", np.ascontiguousarray(ev.material_buffer).tobytes())
        _section(f, "tex_descs", np.ascontiguousarray(ev.texture_descs).tobytes())
        _section(f, "texels", np.ascontiguousarray(ev.texture_texels).tobytes())
        if len(ev.generated_textures):   # older scene files have no such section: r3_frame reads it as empty
            _section(f, "tex_generated", np.ascontiguousarray(ev.generated_textures, dtype=np.uint32).tobytes())
        _section(f, "skybox_desc", b"" if ev.skybox_desc is None else np.ascontiguousarray(ev.skybox_desc).tobytes())
        _section(f, "skybox_texels", b"" if ev.skybox_texels is None else np.ascontiguousarray(ev.skybox_texels).tobytes())
        _section(f, "dir_lights", bytes(ev.directional_buffer))
        _section(f, "point_lights", bytes(ev.point_buffer))
        _section(f, "shadow_target", struct.pack("<II", *ev.shadow_target_size))
        shadows = b""
        for i, s in enumerate(ev.shadows):
            shadows += per_camera_header(s.camera, i, (s.size, s.size), 1, n).tobytes() + struct.pack("<IIII", s.offset[0], s.offset[1], s.size, 0)
        _section(f, "shadows", shadows)
        _section(f, "viewport_header", per_camera_header(ev.camera, CAMERA_VIEWPORT, resolution, samples, n).tobytes())
        _section(f, "uniforms", frame_uniforms(ev.camera, settings.ambient_color, resolution).tobytes())
        _section(f, "viewport_location", np.asarray(ev.camera.location(), dtype=np.float32).tobytes())
        _section(f, "settings", np.asarray(list(settings.ambient_color) + list(settings.clear_color), dtype=np.float32).tobytes())
        _section(f, "target", struct.pack("<IIIII", resolution[0], resolution[1], samples, 1 if srgb_target else 0, frames))


def load_outputs(path: str) -> Dict[str, np.ndarray]:
    out = {}
    with open(path, "rb") as f:
        while True:
            head = f.read(4)
            if len(head) < 4:
                break
            (tl,) = struct.unpack("<I", head)
            tag = f.read(tl).decode()
            (n,) = struct.unpack("<Q", f.read(8))
            out[tag] = f.read(n)
    return {"hdr": np.frombuffer(out["hdr"], dtype=np.float32), "depth": np.frombuffer(out["depth"], dtype=np.float32),
            "ldr": np.frombuffer(out["ldr"], dtype=np.uint8), "visible": np.frombuffer(out["visible"], dtype=np.uint32),
            "stats": np.frombuffer(out["stats"], dtype=np.uint64)}
