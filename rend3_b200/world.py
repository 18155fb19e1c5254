"""Stand-in for rend3's Rust managers: produces the exact std430 bytes they upload.

In a real integration the Rust `Renderer` and its managers stay untouched and hand their
buffers to the C ABI (see INTEGRATION.md).  No Rust toolchain exists in this image, so the
tests and the bench need *something* that builds those buffers; this module restates the
managers' data provenance — nothing here is on the product's hot path.

Mirrors (names kept so tests read like rend3-test/tests/*.rs):
  * `MeshBuilder` / `Mesh`            rend3-types/src/lib.rs:337-706 (smooth normals :662-706)
  * `PbrMaterial` -> ShaderMaterial   rend3-routine/src/pbr/material.rs:455-583
  * `Renderer.add_*`                  rend3/src/renderer/mod.rs:133-423
  * object records                    rend3/src/managers/object.rs:23-36,230-293
  * mesh megabuffer                   rend3/src/managers/mesh.rs:99-166
  * bounding spheres / frustum        rend3/src/util/frustum.rs:15-161
  * `CameraState`                     rend3/src/managers/camera.rs:23-109
  * directional lights + shadow atlas rend3/src/managers/directional.rs:99-157,
                                      directional/shadow_alloc.rs:59-136, shadow_camera.rs:6-33
  * point lights                      rend3/src/managers/point.rs:58-74
  * freelist buffer growth            rend3/src/util/freelist/buffer.rs:19-92
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np

from . import glam
from .layouts import (
    ATTR_ABSENT,
    MAT_ALBEDO_ACTIVE,
    MAT_ALBEDO_BLEND,
    MAT_AOMR_BW_SPLIT,
    MAT_AOMR_SPLIT,
    MAT_AOMR_SWIZZLED_SPLIT,
    MAT_BICOMPONENT_NORMAL,
    MAT_CC_BW_SPLIT,
    MAT_CC_GLTF_SPLIT,
    MAT_NEAREST,
    MAT_SWIZZLED_NORMAL,
    MAT_YDOWN_NORMAL,
    TEXTURE_DESC_DTYPE,
    TEXFMT_RGBA8_UNORM,
    TEXFMT_RGBA8_UNORM_SRGB,
    TEXFMT_RGBA32_FLOAT,
    TEXFMT_R8_UNORM,
    TEXFMT_RG8_UNORM,
    MAT_ALBEDO_VERTEX_SRGB,
    MAT_AOMR_COMBINED,
    MAT_CC_GLTF_COMBINED,
    MAT_UNLIT,
    MATERIAL_DTYPE,
    OBJECT_DTYPE,
    DIRECTIONAL_LIGHT_DTYPE,
    POINT_LIGHT_DTYPE,
)

f32 = np.float32

LEFT = "Left"
RIGHT = "Right"

# Transparency -> (material key, sorting reason, sorting order); pbr/material.rs:382-417,497-503
# SortingReason::Optimization = opaque/cutout front-to-back, Requirement = blend back-to-front
OPAQUE, CUTOUT, BLEND = 0, 1, 2


# ----------------------------------------------------------------------------- meshes
@dataclass
class Mesh:
    """SoA mesh; `attributes` is an ordered list of (slot, array) like Mesh::attributes."""

    attributes: List[Tuple[int, np.ndarray]]
    vertex_count: int
    indices: np.ndarray


class MeshBuilder:
    """rend3-types/src/lib.rs:337-514."""

    def __init__(self, vertex_positions, handedness: str):
        self.positions = np.asarray(vertex_positions, dtype=f32).reshape(-1, 3)
        self.handedness = handedness
        self.normals = None
        self.uv0 = None
        self.color0 = None
        self.indices = None

    @staticmethod
    def new(vertex_positions, handedness: str) -> "MeshBuilder":
        return MeshBuilder(vertex_positions, handedness)

    def with_indices(self, indices) -> "MeshBuilder":
        self.indices = np.asarray(indices, dtype=np.uint32)
        return self

    def with_vertex_normals(self, normals) -> "MeshBuilder":
        self.normals = np.asarray(normals, dtype=f32).reshape(-1, 3)
        return self

    def with_vertex_texture_coordinates_0(self, uv) -> "MeshBuilder":
        self.uv0 = np.asarray(uv, dtype=f32).reshape(-1, 2)
        return self

    def with_vertex_color_0(self, colors) -> "MeshBuilder":
        self.color0 = np.asarray(colors, dtype=np.uint8).reshape(-1, 4)
        return self

    def build(self) -> Mesh:
        n = len(self.positions)
        indices = self.indices if self.indices is not None else np.arange(n, dtype=np.uint32)
        if len(indices) % 3 != 0:
            raise ValueError("IndexCountNotMultipleOfThree")
        if len(indices) and int(indices.max()) >= n:
            raise ValueError("IndexOutOfBounds")
        attrs: List[Tuple[int, np.ndarray]] = [(0, self.positions)]
        if self.normals is not None:
            attrs.append((1, self.normals))
        if self.uv0 is not None:
            attrs.append((3, self.uv0))
        if self.color0 is not None:
            attrs.append((5, self.color0))
        if self.normals is None:
            attrs.append((1, calculate_normals(self.positions, indices, self.handedness == LEFT)))
        # tangents are generated only when uv0 exists (lib.rs:720-728)
        if self.uv0 is not None:
            normals = next(a for slot, a in attrs if slot == 1)
            attrs.append((2, calculate_tangents(self.positions, normals, self.uv0, indices)))
        return Mesh(attrs, n, indices)


def calculate_normals(positions: np.ndarray, indices: np.ndarray, left_handed: bool) -> np.ndarray:
    """Mesh::calculate_normals_for_buffers (rend3-types/src/lib.rs:662-706): per-face
    edge1 x edge2 (LH) / edge2 x edge1 (RH) accumulated in index order, normalize_or_zero."""
    normals = np.zeros_like(positions, dtype=f32)
    tri = indices.reshape(-1, 3)
    for i0, i1, i2 in tri:
        p1, p2, p3 = positions[i0], positions[i1], positions[i2]
        e1 = (p2 - p1).astype(f32)
        e2 = (p3 - p1).astype(f32)
        nrm = glam.cross(e1, e2) if left_handed else glam.cross(e2, e1)
        normals[i0] = normals[i0] + nrm
        normals[i1] = normals[i1] + nrm
        normals[i2] = normals[i2] + nrm
    for i in range(len(normals)):
        normals[i] = glam.normalize_or_zero3(normals[i])
    return normals


def calculate_tangents(positions: np.ndarray, normals: np.ndarray, uvs: np.ndarray, indices: np.ndarray) -> np.ndarray:
    """Mesh::calculate_tangents_for_buffers (rend3-types/src/lib.rs:784-836), including its operator precedence:
    tangent = edge1 * uv2.y - (edge2 * uv1.y) * r; then Gram-Schmidt against the normal, normalize_or_zero."""
    tangents = np.zeros_like(positions, dtype=f32)
    with np.errstate(all="ignore"):
        for i0, i1, i2 in indices.reshape(-1, 3):
            e1 = (positions[i1] - positions[i0]).astype(f32)
            e2 = (positions[i2] - positions[i0]).astype(f32)
            uv1 = (uvs[i1] - uvs[i0]).astype(f32)
            uv2 = (uvs[i2] - uvs[i0]).astype(f32)
            r = f32(1.0) / f32(f32(uv1[0] * uv2[1]) - f32(uv1[1] * uv2[0]))
            t = ((e1 * uv2[1]).astype(f32) - ((e2 * uv1[1]).astype(f32) * r).astype(f32)).astype(f32)
            for i in (i0, i1, i2):
                tangents[i] = (tangents[i] + t).astype(f32)
        for i in range(len(tangents)):
            t = (tangents[i] - (normals[i] * glam.dot3(normals[i], tangents[i])).astype(f32)).astype(f32)
            tangents[i] = glam.normalize_or_zero3(np.nan_to_num(t, nan=0.0, posinf=0.0, neginf=0.0).astype(f32))
    return tangents


def bounding_sphere_from_mesh(positions: np.ndarray):
    """BoundingSphere::from_mesh (util/frustum.rs:15-56): AABB centre, max distance."""
    if len(positions) == 0:
        return np.zeros(3, dtype=f32), f32(0)
    mx = positions.max(axis=0).astype(f32)
    mn = positions.min(axis=0).astype(f32)
    center = ((mx + mn) / f32(2.0)).astype(f32)
    d = (positions - center).astype(f32)
    dist = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]).astype(f32) + d[:, 2] * d[:, 2]).astype(f32)
    return center, f32(dist.max())


def sphere_apply_transform(center, radius, m):
    """BoundingSphere::apply_transform (util/frustum.rs:22-32)."""
    ls = [glam.dot3(m[i, :3], m[i, :3]) for i in range(3)]
    max_scale = f32(np.sqrt(max(ls[0], max(ls[1], ls[2]))))
    c = glam.mul_vec4(m, [center[0], center[1], center[2], 1.0])[:3]
    return c.astype(f32), f32(max_scale * radius)


# ----------------------------------------------------------------------------- materials
@dataclass
class Texture:
    """rend3_types::Texture (rend3-types/src/lib.rs:843-870): RGBA texels + MipmapSource.  `data` is (h, w, 4) uint8 (Rgba8Unorm /
    Rgba8UnormSrgb) or float32 (Rgba32Float); mips = "generated" (box filter, MipmapCount::Maximum) or 1 level; mips = "device":
    MipmapSource::Generated as rend3 does it — level 0 plus a zero-filled chain of MipmapCount::Maximum levels that r3_generate_mipmaps
    fills on the device (rule R12)."""

    data: np.ndarray
    srgb: bool = False
    mips: str = "generated"
    channels: int = 4          # 1 / 2: R8Unorm / Rg8Unorm — only the first channels of `data` are stored, the others read (0, 0, 1)
    block_format: Optional[str] = None   # "bc1" | "bc2" | "bc3" | "bc4" | "bc4s" | "bc5" | "bc5s": the levels are stored as 4x4 blocks (bc.py stands in
                                         # for the ktx2 / dds asset rend3-gltf would load); `srgb` picks the *UnormSrgb variant of bc1 - bc3
    storage: Optional[str] = None        # one of texformats.STORAGE ("rgba16f", "bgra8_srgb", "rgb10a2", "rg8s", ...): the levels are stored in that format
    block_levels: Optional[List[np.ndarray]] = None   # the asset's own blocks per level (flat uint8); then `data` only carries the level-0 shape

    def levels(self) -> List[np.ndarray]:
        lv = [np.ascontiguousarray(self.data)]
        if self.mips != "generated":
            return lv
        while lv[-1].shape[0] > 1 or lv[-1].shape[1] > 1:
            a = lv[-1].astype(np.float64)
            if self.srgb and a.dtype != np.float32 and self.data.dtype == np.uint8:
                lin = a / 255.0
                rgb = np.where(lin[..., :3] > 0.04045, ((lin[..., :3] + 0.055) / 1.055) ** 2.4, lin[..., :3] / 12.92)
                a = np.concatenate([rgb, lin[..., 3:]], axis=-1)
            elif self.data.dtype == np.uint8:
                a = a / 255.0
            h, w = a.shape[:2]
            nh, nw = max(h // 2, 1), max(w // 2, 1)
            a = a[: nh * 2 if h > 1 else 1, : nw * 2 if w > 1 else 1]
            a = a.reshape(nh, 2 if h > 1 else 1, nw, 2 if w > 1 else 1, 4).mean(axis=(1, 3))
            if self.data.dtype == np.uint8:
                if self.srgb:
                    rgb = np.where(a[..., :3] > 0.0031308, 1.055 * a[..., :3] ** (1 / 2.4) - 0.055, a[..., :3] * 12.92)
                    a = np.concatenate([rgb, a[..., 3:]], axis=-1)
                lv.append(np.clip(np.rint(a * 255.0), 0, 255).astype(np.uint8))
            else:
                lv.append(a.astype(np.float32))
        return lv

    def format(self) -> int:
        if self.storage is not None:
            from .texformats import STORAGE
            return STORAGE[self.storage][0]
        if self.block_format is not None:
            from .bc import BLOCK_FORMATS
            plain, srgb, _ = BLOCK_FORMATS[self.block_format]
            return srgb if (self.srgb and srgb is not None) else plain
        if self.data.dtype == np.float32:
            return TEXFMT_RGBA32_FLOAT
        if self.channels in (1, 2):
            return TEXFMT_R8_UNORM if self.channels == 1 else TEXFMT_RG8_UNORM
        return TEXFMT_RGBA8_UNORM_SRGB if self.srgb else TEXFMT_RGBA8_UNORM

    def stored_levels(self) -> List[np.ndarray]:
        """The mip levels as they are stored: narrow formats keep only their channels."""
        lv = self.levels()
        if self.storage is not None:
            from .texformats import pack
            lv = [pack(self.storage, l) for l in lv]
        elif self.block_format is not None:
            from .bc import encode
            if self.block_levels is not None:
                return [np.ascontiguousarray(l, dtype=np.uint8).reshape(-1) for l in self.block_levels]
            return [encode(self.block_format, l) for l in lv]
        elif self.channels in (1, 2) and self.data.dtype == np.uint8:
            lv = [np.ascontiguousarray(l[..., : self.channels]) for l in lv]
        if self.mips == "device":
            h, w = self.data.shape[:2]
            bpp = np.ascontiguousarray(lv[0]).nbytes // (w * h)
            lv = lv + [np.zeros(max(w >> l, 1) * max(h >> l, 1) * bpp, dtype=np.uint8) for l in range(1, max(w, h).bit_length())]
        return lv


@dataclass
class PbrMaterial:
    """Untextured subset of rend3-routine's PbrMaterial (pbr/material.rs:455-474)."""

    albedo_value: Optional[Tuple[float, float, float, float]] = None  # AlbedoComponent::Value / ValueVertex
    albedo_vertex: Optional[str] = None  # None | "linear" | "srgb"  (Vertex{srgb})
    unlit: bool = False
    transparency: int = OPAQUE
    alpha_cutout: float = 0.0
    roughness_factor: Optional[float] = None
    metallic_factor: Optional[float] = None
    reflectance: Optional[float] = None
    ao_factor: Optional[float] = None
    clearcoat_factor: Optional[float] = None
    clearcoat_roughness_factor: Optional[float] = None
    emissive: Optional[Tuple[float, float, float]] = None
    anisotropy: Optional[float] = None
    # texture handles (Renderer.add_texture_2d) per slot of GpuMaterialData (material.wgsl:21-35); None = no texture
    albedo_texture: Optional[int] = None            # AlbedoComponent::Texture / TextureValue / TextureVertex...
    normal_texture: Optional[int] = None            # NormalTexture::{Tricomponent, Bicomponent, BicomponentSwizzled}
    normal_kind: str = "tricomponent"               # | "bicomponent" | "bicomponent_swizzled"
    normal_y_down: bool = False                     # NormalTextureYDirection::Down
    aomr_kind: str = "combined"                     # AoMRTextures: "combined" | "swizzled_split" | "split" | "bw_split"
    roughness_texture: Optional[int] = None         # the mr / aomr texture slot
    metallic_texture: Optional[int] = None
    ao_texture: Optional[int] = None
    reflectance_texture: Optional[int] = None
    clearcoat_kind: str = "gltf_combined"           # ClearcoatTextures: "gltf_combined" | "gltf_split" | "bw_split"
    clearcoat_texture: Optional[int] = None
    clearcoat_roughness_texture: Optional[int] = None
    emissive_texture: Optional[int] = None
    anisotropy_texture: Optional[int] = None
    sample_type: str = "linear"                     # SampleType::{Linear, Nearest}
    uv_transform0: Optional[np.ndarray] = None      # 3x3, column-major like glam Mat3

    def key(self) -> int:  # Material::key (pbr/material.rs:497-499)
        return int(self.transparency)

    def atomic_capable(self) -> bool:  # SortingReason::Optimization (pbr/material.rs:411-416)
        return self.transparency != BLEND

    def back_to_front(self) -> bool:
        return self.transparency == BLEND

    def to_record(self) -> np.ndarray:
        """ShaderMaterial::from_material (pbr/material.rs:549-582) inside the Gpu wrapper."""
        r = np.zeros((), dtype=MATERIAL_DTYPE)
        r["uv_transform0"] = [[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0]]
        if self.uv_transform0 is not None:
            u = np.asarray(self.uv_transform0, dtype=f32).reshape(3, 3)   # u[col][row]
            r["uv_transform0"] = [[u[0][0], u[0][1], u[0][2], 0], [u[1][0], u[1][1], u[1][2], 0], [u[2][0], u[2][1], u[2][2], 0]]
        for slot, handle in enumerate((self.albedo_texture, self.normal_texture, self.roughness_texture, self.metallic_texture, self.reflectance_texture,
                                       self.clearcoat_texture, self.clearcoat_roughness_texture, self.emissive_texture, self.anisotropy_texture, self.ao_texture)):
            r["textures"][slot] = 0 if handle is None else handle + 1            # NonZeroU32 index + 1 (managers/texture.rs)
        r["uv_transform1"] = [[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0]]
        r["albedo"] = self.albedo_value if self.albedo_value is not None else (1, 1, 1, 1)
        r["emissive"] = self.emissive if self.emissive is not None else (0, 0, 0)
        r["roughness"] = self.roughness_factor or 0.0
        r["metallic"] = self.metallic_factor or 0.0
        r["reflectance"] = 0.5 if self.reflectance is None else self.reflectance
        r["clear_coat"] = self.clearcoat_factor or 0.0
        r["clear_coat_roughness"] = self.clearcoat_roughness_factor or 0.0
        r["anisotropy"] = self.anisotropy or 0.0
        r["ambient_occlusion"] = 1.0 if self.ao_factor is None else self.ao_factor
        r["alpha_cutout"] = self.alpha_cutout if self.transparency == CUTOUT else 0.0
        flags = 0
        if self.albedo_value is not None or self.albedo_vertex is not None or self.albedo_texture is not None:
            flags |= MAT_ALBEDO_ACTIVE
        if self.albedo_vertex is not None:
            flags |= MAT_ALBEDO_BLEND
            if self.albedo_vertex == "srgb":
                flags |= MAT_ALBEDO_VERTEX_SRGB
        # pbr/material.rs:296-305,354-362: the texture-layout enums map to one flag each (None counts as Combined)
        flags |= {"combined": MAT_AOMR_COMBINED, "swizzled_split": MAT_AOMR_SWIZZLED_SPLIT, "split": MAT_AOMR_SPLIT, "bw_split": MAT_AOMR_BW_SPLIT}[self.aomr_kind]
        flags |= {"gltf_combined": MAT_CC_GLTF_COMBINED, "gltf_split": MAT_CC_GLTF_SPLIT, "bw_split": MAT_CC_BW_SPLIT}[self.clearcoat_kind]
        if self.normal_texture is not None:
            if self.normal_kind != "tricomponent":
                flags |= MAT_BICOMPONENT_NORMAL
            if self.normal_kind == "bicomponent_swizzled":
                flags |= MAT_SWIZZLED_NORMAL
            if self.normal_y_down:
                flags |= MAT_YDOWN_NORMAL
        if self.sample_type == "nearest":
            flags |= MAT_NEAREST
        if self.unlit:
            flags |= MAT_UNLIT
        r["flags"] = flags
        return r


# ----------------------------------------------------------------------------- scene types
@dataclass
class Object:
    mesh: int
    material: int
    transform: np.ndarray


@dataclass
class Camera:
    """rend3-types Camera: projection = ("raw", mat4) | ("perspective", vfov_deg, near) |
    ("orthographic", (sx, sy, sz))."""

    projection: tuple
    view: np.ndarray


@dataclass
class DirectionalLight:
    color: Tuple[float, float, float]
    intensity: float
    direction: Tuple[float, float, float]
    distance: float
    resolution: int


@dataclass
class PointLight:
    position: Tuple[float, float, float]
    color: Tuple[float, float, float]
    radius: float
    intensity: float


def frustum_from_matrix(m: np.ndarray) -> np.ndarray:
    """Frustum::from_matrix (util/frustum.rs:96-145). m[c][r]; returns (5,4) f32 planes
    left,right,top,bottom,near, each normalised by |abc|."""
    a = m.astype(f32)

    def plane(sign, r):
        p = np.array([a[c][3] + sign * a[c][r] for c in range(4)], dtype=f32)
        mag = glam.length3(p[:3])
        return (p / mag).astype(f32)

    return np.array([plane(+1, 0), plane(-1, 0), plane(-1, 1), plane(+1, 1), plane(-1, 2)], dtype=f32)


class CameraState:
    """rend3/src/managers/camera.rs:10-109."""

    def __init__(self, data: Camera, handedness: str, aspect_ratio: Optional[float]):
        self.handedness = handedness
        self.data = data
        self.aspect_ratio = f32(1.0 if aspect_ratio is None else aspect_ratio)
        self.proj = self._projection()
        self.view = data.view.astype(f32)
        self.orig_view = self.view.copy()
        self.orig_view[3] = [0, 0, 0, 1]
        self.inv_view = glam.inverse(self.view)
        self.view_proj = glam.mul(self.proj, self.view)
        self.origin_view_proj = glam.mul(self.proj, self.orig_view)
        self.world_frustum = frustum_from_matrix(self.view_proj)

    def _projection(self) -> np.ndarray:
        p = self.data.projection
        lh = self.handedness == LEFT
        if p[0] == "raw":
            return np.asarray(p[1], dtype=f32)
        if p[0] == "perspective":
            fn = glam.perspective_infinite_reverse_lh if lh else glam.perspective_infinite_reverse_rh
            return fn(glam.to_radians(p[1]), self.aspect_ratio, p[2])
        if p[0] == "orthographic":
            half = np.asarray(p[1], dtype=f32) * f32(0.5)
            fn = glam.orthographic_lh if lh else glam.orthographic_rh
            return fn(-half[0], half[0], -half[1], half[1], half[2], -half[2])
        raise ValueError(p[0])

    def location(self) -> np.ndarray:
        return self.inv_view[3, :3].astype(f32)


def shadow_camera(light: DirectionalLight, user_camera: CameraState) -> CameraState:
    """directional/shadow_camera.rs:6-33: texel-snapped ortho camera centred on the viewer."""
    cam_loc = user_camera.location()
    texel = f32(f32(light.distance) / f32(light.resolution))
    look_at = glam.look_at_lh if user_camera.handedness == LEFT else glam.look_at_rh
    direction = np.asarray(light.direction, dtype=f32)
    origin_view = look_at(np.zeros(3, dtype=f32), direction, glam.vec3(0, 1, 0))
    cov = glam.transform_point3(origin_view, cam_loc)
    offset = np.fmod(cov[:2], texel).astype(f32)
    shadow_loc = (cov - np.array([offset[0], offset[1], 0], dtype=f32)).astype(f32)
    new_loc = glam.transform_point3(glam.inverse(origin_view), shadow_loc)
    d = f32(light.distance)
    return CameraState(
        Camera(("orthographic", (d, d, d)), look_at(new_loc, (new_loc + direction).astype(f32), glam.vec3(0, 1, 0))),
        user_camera.handedness,
        None,
    )


def allocate_shadow_atlas(maps: List[Tuple[int, int]], max_dimension: int = 8192):
    """Quadtree atlas packing with the same observable results as
    directional/shadow_alloc.rs:59-136: maps sorted by descending resolution (stable), each
    placed in the first root whose quadtree has a free node of its order; roots laid out
    row-major.  Returns ((width, height), [(offset_x, offset_y, size, handle)]) in BFS order."""
    if not maps or max_dimension == 0:
        return None
    order_sorted = sorted(maps, key=lambda hr: -hr[1])
    root_size = order_sorted[0][1]
    root_lz = 16 - root_size.bit_length()

    VAC, LEAF, KIDS = 0, 1, 2
    nodes: list = [[VAC, None]]
    roots = [0]

    def try_alloc(idx, rel, handle) -> bool:
        kind, payload = nodes[idx]
        if kind == VAC:
            if rel == 0:
                nodes[idx] = [LEAF, handle]
                return True
            base = len(nodes)
            nodes[idx] = [KIDS, [base, base + 1, base + 2, base + 3]]
            nodes.extend([[VAC, None] for _ in range(4)])
            return try_alloc(idx, rel, handle)
        if kind == LEAF:
            return False
        if rel == 0:
            return False
        return any(try_alloc(c, rel - 1, handle) for c in payload)

    for handle, res in order_sorted:
        rel = (16 - res.bit_length()) - root_lz
        while not try_alloc(roots[-1], rel, handle):
            nodes.append([VAC, None])
            roots.append(len(nodes) - 1)

    cols_avail = max_dimension // root_size
    n_roots = len(roots)
    rows = int(np.ceil(n_roots / cols_avail))
    cols = int(np.ceil(n_roots / rows))
    dims = (cols * root_size, rows * root_size)
    out = []
    queue = [(1, ((i % cols) * root_size, (i // cols) * root_size), r) for i, r in enumerate(roots)]
    while queue:
        div, off, idx = queue.pop(0)
        size = root_size // div
        kind, payload = nodes[idx]
        if kind == LEAF:
            out.append((off[0], off[1], size, payload))
        elif kind == KIDS:
            half = size // 2
            for ci, c in enumerate(payload):
                queue.append((div * 2, (off[0] + half * (ci % 2), off[1] + half * (ci // 2)), c))
    return dims, out


MINIMUM_SHADOW_MAP_SIZE = 32  # directional.rs:24


@dataclass
class ShadowDesc:
    offset: Tuple[int, int]
    size: int
    handle: int
    camera: CameraState


@dataclass
class EvalOutput:
    """What `Renderer::evaluate_instructions` leaves on the GPU + the host-side facts the
    routines read from the managers (renderer/eval.rs:9-181)."""

    object_buffer: np.ndarray          # (capacity,) OBJECT_DTYPE — object_manager.buffer::<M>()
    object_material_key: np.ndarray    # (capacity,) u64   material.inner.key()
    object_atomic: np.ndarray          # (capacity,) u8    sorting.reason == Optimization
    object_back_to_front: np.ndarray   # (capacity,) u8
    object_live: np.ndarray            # (capacity,) u8    slot is Some(..) in data_vec (enumerated_objects)
    object_location: np.ndarray        # (capacity,3) f32  InternalObject::location (object.rs:256,306)
    mesh_buffer: np.ndarray            # (nwords,) u32
    material_buffer: np.ndarray        # (n,) MATERIAL_DTYPE
    texture_descs: np.ndarray          # (n,) TEXTURE_DESC_DTYPE — the bindless d2 table
    texture_texels: np.ndarray         # u8 blob holding every mip level
    directional_buffer: bytes          # u32 count @0, array @16 (stride 128)
    point_buffer: bytes                # u32 count @0, array @16 (stride 32)
    shadows: List[ShadowDesc]
    shadow_target_size: Tuple[int, int]
    camera: CameraState
    skybox_desc: Optional[np.ndarray] = None    # TEXTURE_DESC_DTYPE scalar (width = face size), None = no skybox
    skybox_texels: Optional[np.ndarray] = None  # six faces (+X -X +Y -Y +Z -Z), each with its mip chain
    generated_textures: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.uint32))   # table indices of mips="device" textures


class Renderer:
    """Subset of rend3::Renderer's world-mutation API (renderer/mod.rs:133-423)."""

    STARTING_SIZE = 16  # util/freelist/buffer.rs:19

    def __init__(self, handedness: str = LEFT, aspect_ratio: Optional[float] = None):
        self.handedness = handedness
        self.aspect_ratio = aspect_ratio
        self.meshes: list = []
        self.mesh_words = np.zeros(0, dtype=np.uint32)
        self.materials: List[PbrMaterial] = []
        self.textures: List[Texture] = []
        self.skybox: Optional[List[Texture]] = None
        self.objects: List[Optional[dict]] = []
        self.free_objects: List[int] = []
        self.delayed: List[int] = []
        self.to_delete: List[int] = []
        self.obj_capacity = self.STARTING_SIZE
        self.obj_reserved = self.STARTING_SIZE
        self.obj_gpu = np.zeros(self.STARTING_SIZE, dtype=OBJECT_DTYPE)
        self.stale: List[int] = []
        self.dir_lights: List[Optional[DirectionalLight]] = []
        self.point_lights: List[Optional[PointLight]] = []
        self.camera = CameraState(Camera(("raw", glam.identity()), glam.identity()), handedness, aspect_ratio)

    # ---- meshes (managers/mesh.rs:99-166): attributes then indices, bump-allocated bytes
    def add_mesh(self, mesh: Mesh) -> int:
        ranges = {}
        words = [self.mesh_words]
        cursor = len(self.mesh_words) * 4
        for slot, arr in mesh.attributes:
            raw = np.ascontiguousarray(arr).view(np.uint8).reshape(-1)
            assert len(raw) % 4 == 0
            ranges[slot] = cursor
            words.append(raw.view(np.uint32))
            cursor += len(raw)
        index_start = cursor
        words.append(mesh.indices.astype(np.uint32))
        self.mesh_words = np.concatenate(words)
        center, radius = bounding_sphere_from_mesh(mesh.attributes[0][1])
        self.meshes.append(
            dict(ranges=ranges, index_start=index_start, index_count=len(mesh.indices), center=center, radius=radius)
        )
        return len(self.meshes) - 1

    def add_texture_2d(self, texture: Texture) -> int:   # Renderer::add_texture_2d (renderer/mod.rs:213-241)
        self.textures.append(texture)
        return len(self.textures) - 1

    def set_skybox(self, faces, srgb: bool = True, mips: str = "generated"):
        """SkyboxRoutine::set_background_texture with a cube texture (rend3-routine/src/skybox.rs:47-60): six square RGBA faces
        in the order +X, -X, +Y, -Y, +Z, -Z; None removes it."""
        self.skybox = None if faces is None else [Texture(np.ascontiguousarray(f), srgb=srgb, mips=mips) for f in faces]

    def _skybox_blob(self):
        if self.skybox is None:
            return None, None
        lv0 = self.skybox[0].levels()
        desc = np.zeros((), dtype=TEXTURE_DESC_DTYPE)
        desc["width"], desc["height"], desc["mip_count"], desc["format"], desc["byte_offset"] = lv0[0].shape[1], lv0[0].shape[0], len(lv0), self.skybox[0].format(), 0
        raw = [np.ascontiguousarray(l).view(np.uint8).reshape(-1) for f in self.skybox for l in f.levels()]
        return desc, np.concatenate(raw)

    def _texture_table(self):
        descs = np.zeros(len(self.textures), dtype=TEXTURE_DESC_DTYPE)
        blobs, cursor = [], 0
        for i, t in enumerate(self.textures):
            lv = t.stored_levels()
            descs[i]["width"], descs[i]["height"] = t.data.shape[1], t.data.shape[0]
            descs[i]["mip_count"], descs[i]["format"], descs[i]["byte_offset"] = len(lv), t.format(), cursor
            raw = np.concatenate([np.ascontiguousarray(l).view(np.uint8).reshape(-1) for l in lv])
            pad = (-len(raw)) % 16
            blobs.append(np.concatenate([raw, np.zeros(pad, dtype=np.uint8)]))
            cursor += len(raw) + pad
        return descs, (np.concatenate(blobs) if blobs else np.zeros(0, dtype=np.uint8))

    def add_material(self, material: PbrMaterial) -> int:
        self.materials.append(material)
        return len(self.materials) - 1

    # ---- objects (managers/object.rs:230-293, handle_alloc.rs:46-77)
    def _alloc_object_handle(self) -> int:
        if self.free_objects:
            return self.free_objects.pop()
        self.objects.append(None)
        return len(self.objects) - 1

    def _use_index(self, idx: int):  # FreelistDerivedBuffer::use_index (buffer.rs:48-54), `>` as written
        if idx > self.obj_reserved:
            self.obj_reserved = 1 << (idx - 1).bit_length()
        self.stale.append(idx)

    def add_object(self, obj: Object) -> int:
        h = self._alloc_object_handle()
        mesh = self.meshes[obj.mesh]
        rec = np.zeros((), dtype=OBJECT_DTYPE)
        t = np.asarray(obj.transform, dtype=f32)
        c, r = sphere_apply_transform(mesh["center"], mesh["radius"], t)
        rec["transform"] = t.reshape(16)
        rec["sphere_center"] = c
        rec["sphere_radius"] = r
        rec["first_index"] = mesh["index_start"] // 4
        rec["index_count"] = mesh["index_count"]
        rec["material_index"] = obj.material
        rec["attr_offset"] = [mesh["ranges"].get(s, ATTR_ABSENT) for s in range(6)]
        rec["enabled"] = 1
        self.objects[h] = dict(rec=rec, obj=obj, mesh_center=mesh["center"], mesh_radius=mesh["radius"], location=c)
        self._use_index(h)
        return h

    def duplicate_object(self, src: int, transform=None, material=None) -> int:
        o = self.objects[src]["obj"]
        return self.add_object(
            Object(o.mesh, o.material if material is None else material, o.transform if transform is None else transform)
        )

    def set_object_transform(self, h: int, transform):
        e = self.objects[h]
        t = np.asarray(transform, dtype=f32)
        e["rec"]["transform"] = t.reshape(16)
        c, r = sphere_apply_transform(e["mesh_center"], e["mesh_radius"], t)
        e["rec"]["sphere_center"], e["rec"]["sphere_radius"] = c, r
        e["location"] = glam.transform_point3(t, np.zeros(3, dtype=f32))
        e["obj"].transform = t
        self._use_index(h)

    def remove_object(self, h: int):
        """Dropping an ObjectHandle: disabled now, physically removed one frame later
        (object.rs:330-342, handle_alloc.rs:21-29)."""
        self.to_delete.append(h)

    def add_directional_light(self, light: DirectionalLight) -> int:
        self.dir_lights.append(light)
        return len(self.dir_lights) - 1

    def add_point_light(self, light: PointLight) -> int:
        self.point_lights.append(light)
        return len(self.point_lights) - 1

    def set_camera_data(self, camera: Camera):
        self.camera = CameraState(camera, self.handedness, self.aspect_ratio)

    def set_aspect_ratio(self, aspect_ratio: Optional[float]):
        self.aspect_ratio = aspect_ratio
        self.camera = CameraState(self.camera.data, self.handedness, aspect_ratio)

    # ---- Renderer::evaluate_instructions (renderer/eval.rs:9-181)
    def evaluate(self) -> EvalOutput:
        # delayed handles reclaimed at the top of the frame; their slots are taken out
        deferred = self.delayed
        self.delayed = []
        self.free_objects.extend(deferred)
        for h in self.to_delete:  # Delete instructions of this frame: mark disabled, delay reclamation
            self._use_index(h)
            self.objects[h]["rec"]["enabled"] = 0
            self.delayed.append(h)
        self.to_delete = []
        for h in deferred:
            self.objects[h] = None
        # FreelistDerivedBuffer::apply
        if self.obj_capacity != self.obj_reserved:
            grown = np.zeros(self.obj_reserved, dtype=OBJECT_DTYPE)
            grown[: self.obj_capacity] = self.obj_gpu
            self.obj_gpu = grown
            self.obj_capacity = self.obj_reserved
        for idx in self.stale:
            if idx < self.obj_capacity:  # out-of-range scatter writes are dropped (robust buffer access)
                e = self.objects[idx]
                self.obj_gpu[idx] = e["rec"] if e is not None else np.zeros((), dtype=OBJECT_DTYPE)
        self.stale = []

        cap = self.obj_capacity
        key = np.zeros(cap, dtype=np.uint64)
        atomic = np.zeros(cap, dtype=np.uint8)
        b2f = np.zeros(cap, dtype=np.uint8)
        live = np.zeros(cap, dtype=np.uint8)
        location = np.zeros((cap, 3), dtype=f32)
        for i, e in enumerate(self.objects[:cap]):
            if e is None:
                continue
            m = self.materials[int(e["rec"]["material_index"])]
            key[i], atomic[i], b2f[i], live[i] = m.key(), m.atomic_capable(), m.back_to_front(), 1
            location[i] = e["location"]

        mats = np.zeros(max(len(self.materials), 1), dtype=MATERIAL_DTYPE)
        for i, m in enumerate(self.materials):
            mats[i] = m.to_record()

        # directional lights + shadow atlas (directional.rs:99-157)
        live_lights = [(i, l) for i, l in enumerate(self.dir_lights) if l is not None]
        atlas = allocate_shadow_atlas([(i, l.resolution) for i, l in live_lights])
        shadows: List[ShadowDesc] = []
        size = (MINIMUM_SHADOW_MAP_SIZE, MINIMUM_SHADOW_MAP_SIZE)
        dl = np.zeros(0, dtype=DIRECTIONAL_LIGHT_DTYPE)
        if atlas is not None:
            dims, maps = atlas
            size = (max(dims[0], MINIMUM_SHADOW_MAP_SIZE), max(dims[1], MINIMUM_SHADOW_MAP_SIZE))
            size_f = np.array(size, dtype=f32)
            dl = np.zeros(len(maps), dtype=DIRECTIONAL_LIGHT_DTYPE)
            for k, (ox, oy, sz, handle) in enumerate(maps):
                light = self.dir_lights[handle]
                cam = shadow_camera(light, self.camera)
                shadows.append(ShadowDesc((ox, oy), sz, handle, cam))
                dl[k]["view_proj"] = cam.view_proj.reshape(16)
                dl[k]["color"] = np.asarray(light.color, dtype=f32) * f32(light.intensity)
                dl[k]["direction"] = np.asarray(light.direction, dtype=f32)
                dl[k]["inv_resolution"] = f32(1.0) / size_f
                dl[k]["atlas_offset"] = np.array([ox, oy], dtype=f32) / size_f
                dl[k]["atlas_size"] = f32(sz) / size_f
        dbytes = np.array([len(dl), 0, 0, 0], dtype=np.uint32).tobytes() + dl.tobytes()

        pls = [l for l in self.point_lights if l is not None]
        pl = np.zeros(len(pls), dtype=POINT_LIGHT_DTYPE)
        for k, l in enumerate(pls):
            pl[k]["position"] = [l.position[0], l.position[1], l.position[2], 1.0]
            pl[k]["color"] = np.asarray(l.color, dtype=f32) * f32(l.intensity)
            pl[k]["radius"] = l.radius
        pbytes = np.array([len(pl), 0, 0, 0], dtype=np.uint32).tobytes() + pl.tobytes()

        tex_descs, tex_blob = self._texture_table()
        sky_desc, sky_blob = self._skybox_blob()
        return EvalOutput(
            object_buffer=self.obj_gpu.copy(),
            object_material_key=key,
            object_atomic=atomic,
            object_back_to_front=b2f,
            object_live=live,
            object_location=location,
            mesh_buffer=self.mesh_words.copy(),
            material_buffer=mats,
            texture_descs=tex_descs,
            texture_texels=tex_blob,
            skybox_desc=sky_desc,
            skybox_texels=sky_blob,
            generated_textures=np.array([i for i, t in enumerate(self.textures) if t.mips == "device"], dtype=np.uint32),
            directional_buffer=dbytes,
            point_buffer=pbytes,
            shadows=shadows,
            shadow_target_size=size,
            camera=self.camera,
        )
