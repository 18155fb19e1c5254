"""Host-side mirror of rend3-routine's interface for the hot path, driving the C ABI.

Names, argument meaning and call order follow the reference so that the parity tests read like
rend3-test's own tests:

  GpuCuller.object_uniform_upload     rend3-routine/src/culling/culler.rs:427-529
  GpuCuller.cull (+ batch_objects)    culler.rs:531-659, 682-713; batching.rs:120-250
  ForwardRoutine / shadow rendering   forward.rs:192-315; base.rs:366-448
  FrameUniforms.new                   uniforms.rs:30-49
  BaseRenderGraph.add_to_graph        base.rs:129-185 (node order)
  TonemappingRoutine.add_to_graph     tonemapping.rs:108-147

There is no render graph here: the graph's job (ordering + resource lifetime) collapses to a
fixed, stream-ordered call sequence on one CUDA stream.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np

from . import glam
from .backend import CAMERA_VIEWPORT, CB_BAKE, CB_CULL, Backend
from .layouts import CAMERA_HEADER_DTYPE, FRAME_UNIFORMS_DTYPE, PCU_MULTISAMPLED, PCU_POSITIVE_AREA_VISIBLE
from .world import LEFT, CameraState, EvalOutput, frustum_from_matrix

f32 = np.float32


def triangle_visibility_positive(handedness: str, shadow: bool) -> bool:
    """TriangleVisibility::from_winding_and_face (culler.rs:127-149): winding = handedness.into()
    (Left -> Cw, rend3-types lib.rs:1190-1197); viewport culls Back, shadow cameras cull Front."""
    cw = handedness == LEFT
    front_culled = shadow
    # (Ccw,Back)|(Cw,Front) -> positive ; (Ccw,Front)|(Cw,Back) -> negative
    return (not cw and not front_culled) or (cw and front_culled)


def per_camera_header(camera: CameraState, camera_specifier: int, resolution: Tuple[int, int], samples: int,
                      object_count: int) -> np.ndarray:
    """PerCameraUniform header written by object_uniform_upload (culler.rs:484-505)."""
    h = np.zeros((), dtype=CAMERA_HEADER_DTYPE)
    h["view"] = camera.view.reshape(16)
    h["view_proj"] = camera.view_proj.reshape(16)
    h["shadow_index"] = camera_specifier
    h["frustum"] = camera.world_frustum
    h["resolution"] = np.array(resolution, dtype=f32)
    flags = 0
    if triangle_visibility_positive(camera.handedness, camera_specifier != CAMERA_VIEWPORT):
        flags |= PCU_POSITIVE_AREA_VISIBLE
    if samples != 1:
        flags |= PCU_MULTISAMPLED
    h["flags"] = flags
    h["object_count"] = object_count
    return h


def frame_uniforms(camera: CameraState, ambient, resolution: Tuple[int, int]) -> np.ndarray:
    """FrameUniforms::new (uniforms.rs:30-49)."""
    u = np.zeros((), dtype=FRAME_UNIFORMS_DTYPE)
    u["view"] = camera.view.reshape(16)
    u["view_proj"] = camera.view_proj.reshape(16)
    u["origin_view_proj"] = camera.origin_view_proj.reshape(16)
    u["inv_view"] = glam.inverse(camera.view).reshape(16)
    try:
        u["inv_view_proj"] = glam.inverse(camera.view_proj).reshape(16)
        u["inv_origin_view_proj"] = glam.inverse(camera.origin_view_proj).reshape(16)
    except np.linalg.LinAlgError:  # singular raw projections are never inverted on the hot path
        pass
    u["frustum"] = frustum_from_matrix(camera.proj)
    u["ambient"] = np.asarray(ambient, dtype=f32)
    u["resolution"] = np.asarray(resolution, dtype=np.uint32)
    return u


@dataclass
class BaseRenderGraphSettings:
    """base.rs:95-98."""

    ambient_color: Tuple[float, float, float, float] = (0.0, 0.0, 0.0, 0.0)
    clear_color: Tuple[float, float, float, float] = (0.0, 0.0, 0.0, 0.0)


class GpuCuller:
    """culling/culler.rs:185-714, bound to one backend context."""

    def __init__(self, backend: Backend):
        self.backend = backend

    def object_uniform_upload(self, eval_output: EvalOutput, camera: CameraState, camera_specifier: int,
                              resolution: Tuple[int, int], samples: int = 1, mode: int = CB_BAKE | CB_CULL):
        header = per_camera_header(camera, camera_specifier, resolution, samples, len(eval_output.object_buffer))
        self.backend.object_uniform_upload(camera_specifier, header, mode)

    def cull(self, eval_output: EvalOutput, camera_specifier: int):
        """add_culling_to_graph (culler.rs:682-713): batch_objects then cull."""
        self.backend.batch_objects(camera_specifier, eval_output.camera.location())
        self.backend.cull(camera_specifier)


class BaseRenderGraph:
    """base.rs:103-186 collapsed to a call sequence."""

    def __init__(self, backend: Backend):
        self.backend = backend
        self.gpu_culler = GpuCuller(backend)
        self._resolution: Optional[Tuple[int, int]] = None

    def upload_world(self, ev: EvalOutput):
        """What evaluate_instructions leaves in wgpu buffers (renderer/eval.rs:157-181)."""
        b = self.backend
        b.set_objects(ev.object_buffer)
        flags = (ev.object_live & 1) | ((ev.object_atomic & 1) << 1) | ((ev.object_back_to_front & 1) << 2)
        loc = np.ascontiguousarray(ev.object_location, dtype=f32)
        b.set_object_sort_info(ev.object_material_key, flags.astype(np.uint8), loc)
        b.set_mesh_buffer(ev.mesh_buffer)
        b.set_textures(ev.texture_descs, ev.texture_texels)
        if len(ev.generated_textures):                                            # TextureManager::add, MipmapSource::Generated (texture.rs:146-180)
            b.generate_mipmaps(ev.generated_textures)
        b.set_skybox(ev.skybox_desc, ev.skybox_texels)
        b.set_materials(ev.material_buffer)
        b.set_directional_lights(ev.directional_buffer, ev.shadow_target_size[0], ev.shadow_target_size[1])
        b.set_point_lights(ev.point_buffer)

    def add_to_graph(self, ev: EvalOutput, resolution: Tuple[int, int], samples: int = 1,
                     settings: BaseRenderGraphSettings = BaseRenderGraphSettings(), srgb_target: bool = True,
                     upload: bool = True, scissor_rows: Optional[Tuple[int, int]] = None, shadow_filter=None, after_shadows=None,
                     after_target=None, tonemap: bool = True, skinning=None, frame_graph: Optional[bool] = None, before_resolve=None):
        """One frame in the node order of base.rs:135-185.  `scissor_rows` restricts rasterisation and shading
        to a band of pixel rows (the screen-tile split of the multi-GPU forward pass); `shadow_filter(i)` selects the shadow
        maps this rank renders — it then clears only their rects, the others arrive from their owners — and `after_shadows()`
        runs once they are in the atlas (the ranks send their maps to the peers there) and `before_resolve()` right before the
        shading reads the atlas (the ranks wait for the peers' maps there: the exchange overlaps the viewport cull and raster); `after_target()` runs once the render target and
        the atlas exist (peer mappings are created there); `tonemap=False` leaves the blit to the caller (the assembling rank
        runs it after the other ranks' rows have arrived); `frame_graph` records the frame's stream work and submits it as ONE CUDA
        graph launch (r3_frame_begin / r3_frame_end; the reference submits once per frame, graph.rs:510) — default: the R3_FRAME_GRAPH
        environment variable."""
        import os
        if frame_graph is None:
            frame_graph = os.environ.get("R3_FRAME_GRAPH", "0") not in ("", "0")
        b, culler = self.backend, self.gpu_culler
        if upload:
            self.upload_world(ev)
        if self._resolution != (resolution, samples, tuple(settings.clear_color)):
            b.set_render_target(resolution[0], resolution[1], samples, settings.clear_color)
            self._resolution = (resolution, samples, tuple(settings.clear_color))
        if scissor_rows is not None:
            b.set_scissor_rows(scissor_rows[0], scissor_rows[1])
        if after_target is not None:
            after_target()
        if frame_graph:
            b.frame_begin()
        if shadow_filter is None:
            b.clear_shadow_atlas()                                                # base.rs:139
        else:
            for i, s in enumerate(ev.shadows):
                if shadow_filter(i):
                    b.clear_shadow_rect(s.offset[0], s.offset[1], s.size, s.size)
        b.set_frame_uniforms(frame_uniforms(ev.camera, settings.ambient_color, resolution))  # :142
        if skinning is not None:                                                  # :145 state.skinning: (skeleton records, joint matrices)
            b.skin(skinning[0], skinning[1])
        mine = [(i, s) for i, s in enumerate(ev.shadows) if shadow_filter is None or shadow_filter(i)]
        for i, s in mine:                                                         # :148
            culler.object_uniform_upload(ev, s.camera, i, (s.size, s.size), 1)
        for i, s in mine:                                                         # :150
            culler.cull(ev, i)
        for i, s in mine:                                                         # :153
            b.shadow_pass(i, s.offset[0], s.offset[1], s.size)
        if after_shadows is not None:
            after_shadows()
        culler.object_uniform_upload(ev, ev.camera, CAMERA_VIEWPORT, resolution, samples)   # :156
        b.forward_begin()
        b.forward_pass(0)                                                         # :159 predicted triangles
        b.hiz_build()                                                             # :162
        culler.cull(ev, CAMERA_VIEWPORT)                                          # :169
        b.forward_pass(1)                                                         # :172 residual triangles
        if before_resolve is not None:
            before_resolve()
        b.forward_resolve()                                                       # fs_main of the opaque + cutout fragments
        # skybox (:175) is outside this path
        b.forward_blend()                                                         # :181 transparent objects, back to front
        if tonemap:
            b.tonemap(srgb_target)                                                # :184
        if frame_graph:
            b.frame_end()
