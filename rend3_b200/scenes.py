"""Seeded synthetic scenes for the BASELINE.json configurations (SURVEY.md 8d), built vectorised.

Everything here produces the same `EvalOutput` the manager stand-in (world.py) produces, only in bulk:
object records for 10^4..10^7 objects cannot go through per-object Python calls.  Meshes, materials,
lights and cameras still go through `world.Renderer` so their bytes follow the same code as the tests.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

from . import glam
from .layouts import ATTR_ABSENT, OBJECT_DTYPE
from .runner import cube_mesh
from .world import LEFT, Camera, DirectionalLight, EvalOutput, MeshBuilder, Object, PbrMaterial, PointLight, Renderer

f32 = np.float32


def random_unit_quaternions(rng: np.random.Generator, n: int) -> np.ndarray:
    q = rng.standard_normal((n, 4)).astype(f32)
    q /= np.linalg.norm(q, axis=1, keepdims=True).astype(f32)
    return q.astype(f32)


def trs_matrices(translation: np.ndarray, quat: np.ndarray, scale: np.ndarray) -> np.ndarray:
    """Mat4::from_scale_rotation_translation, vectorised; returns (n, 4, 4) f32 as [col][row]."""
    x, y, z, w = (quat[:, i].astype(f32) for i in range(4))
    x2, y2, z2 = x + x, y + y, z + z
    xx, xy, xz = x * x2, x * y2, x * z2
    yy, yz, zz = y * y2, y * z2, z * z2
    wx, wy, wz = w * x2, w * y2, w * z2
    one = f32(1.0)
    n = len(x)
    m = np.zeros((n, 4, 4), dtype=f32)
    s = scale.astype(f32).reshape(n, scale.shape[1] if scale.ndim > 1 else 1)
    if s.shape[1] == 1:
        s = np.repeat(s, 3, axis=1)
    m[:, 0, 0] = (one - (yy + zz)) * s[:, 0]; m[:, 0, 1] = (xy + wz) * s[:, 0]; m[:, 0, 2] = (xz - wy) * s[:, 0]
    m[:, 1, 0] = (xy - wz) * s[:, 1]; m[:, 1, 1] = (one - (xx + zz)) * s[:, 1]; m[:, 1, 2] = (yz + wx) * s[:, 1]
    m[:, 2, 0] = (xz + wy) * s[:, 2]; m[:, 2, 1] = (yz - wx) * s[:, 2]; m[:, 2, 2] = (one - (xx + yy)) * s[:, 2]
    m[:, 3, :3] = translation.astype(f32)
    m[:, 3, 3] = one
    return m


def bulk_object_records(renderer: Renderer, transforms: np.ndarray, mesh_ids: np.ndarray, material_ids: np.ndarray,
                        enabled: Optional[np.ndarray] = None, capacity: Optional[int] = None):
    """Vectorised object_add_callback (rend3/src/managers/object.rs:230-293) for n objects in slots 0..n-1.
    Returns (records[capacity], location[capacity,3])."""
    n = len(transforms)
    cap = capacity or max(Renderer.STARTING_SIZE, 1 << max(n - 1, 0).bit_length())
    rec = np.zeros(cap, dtype=OBJECT_DTYPE)
    t = transforms.astype(f32)
    rec["transform"][:n] = t.reshape(n, 16)
    centers = np.array([m["center"] for m in renderer.meshes], dtype=f32)[mesh_ids]
    radii = np.array([m["radius"] for m in renderer.meshes], dtype=f32)[mesh_ids]
    # BoundingSphere::apply_transform (util/frustum.rs:22-32) in glam's accumulation order
    c = t[:, 0, :3] * centers[:, 0:1]
    c = c + t[:, 1, :3] * centers[:, 1:2]
    c = c + t[:, 2, :3] * centers[:, 2:3]
    c = (c + t[:, 3, :3]).astype(f32)
    ls = [((t[:, k, 0] * t[:, k, 0] + t[:, k, 1] * t[:, k, 1]).astype(f32) + t[:, k, 2] * t[:, k, 2]).astype(f32) for k in range(3)]
    max_scale = np.sqrt(np.maximum(ls[0], np.maximum(ls[1], ls[2]))).astype(f32)
    rec["sphere_center"][:n] = c
    rec["sphere_radius"][:n] = (max_scale * radii).astype(f32)
    rec["first_index"][:n] = np.array([m["index_start"] // 4 for m in renderer.meshes], dtype=np.uint32)[mesh_ids]
    rec["index_count"][:n] = np.array([m["index_count"] for m in renderer.meshes], dtype=np.uint32)[mesh_ids]
    rec["material_index"][:n] = material_ids
    offs = np.array([[m["ranges"].get(s, ATTR_ABSENT) for s in range(6)] for m in renderer.meshes], dtype=np.uint32)
    rec["attr_offset"][:n] = offs[mesh_ids]
    rec["enabled"][:n] = 1 if enabled is None else enabled.astype(np.uint32)
    loc = np.zeros((cap, 3), dtype=f32)
    loc[:n] = c
    return rec, loc


def eval_with_bulk_objects(renderer: Renderer, rec: np.ndarray, loc: np.ndarray, n_live: int) -> EvalOutput:
    ev = renderer.evaluate()
    cap = len(rec)
    mats = renderer.materials
    mi = rec["material_index"][:n_live]
    key_of = np.array([m.key() for m in mats], dtype=np.uint64)
    atomic_of = np.array([m.atomic_capable() for m in mats], dtype=np.uint8)
    b2f_of = np.array([m.back_to_front() for m in mats], dtype=np.uint8)
    ev.object_buffer = rec
    ev.object_material_key = np.zeros(cap, dtype=np.uint64); ev.object_material_key[:n_live] = key_of[mi]
    ev.object_atomic = np.zeros(cap, dtype=np.uint8); ev.object_atomic[:n_live] = atomic_of[mi]
    ev.object_back_to_front = np.zeros(cap, dtype=np.uint8); ev.object_back_to_front[:n_live] = b2f_of[mi]
    ev.object_live = np.zeros(cap, dtype=np.uint8); ev.object_live[:n_live] = 1
    ev.object_location = loc
    return ev


def cube_example_camera(pull_back: float = 1.0) -> Camera:
    """examples/src/cube/mod.rs:99-107: view = euler XYZ(-0.55, 0.5, 0) * translate(-(3, 3, -5) * pull_back)."""
    loc = np.array([3.0, 3.0, -5.0], dtype=f32) * f32(pull_back)
    view = glam.mul(glam.from_euler_xyz(-0.55, 0.5, 0.0), glam.from_translation(-loc))
    return Camera(("perspective", 60.0, 0.1), view)


def subdivided_cube_mesh(k: int, with_uv: bool = False, vertex_alpha_seed: Optional[int] = None):
    """Cube [-1,1]^3 whose faces are k x k quads (12 k^2 triangles), same winding as rend3-test's cube.  with_uv: every face
    carries texture coordinates [0,1]^2 (MeshBuilder then derives tangents, lib.rs:720-836)."""
    if k == 1 and not with_uv and vertex_alpha_seed is None:
        return cube_mesh()
    faces = [  # origin corner, u edge, v edge chosen so (o, o+u, o+u+v, o+v) matches helpers.rs:78-109
        ((-1, -1, 1), (2, 0, 0), (0, 2, 0)), ((-1, 1, -1), (2, 0, 0), (0, -2, 0)), ((1, -1, -1), (0, 2, 0), (0, 0, 2)),
        ((-1, -1, 1), (0, 2, 0), (0, 0, -2)), ((1, 1, -1), (-2, 0, 0), (0, 0, 2)), ((1, -1, 1), (-2, 0, 0), (0, 0, -2)),
    ]
    pos, idx, uvs = [], [], []
    for o, u, v in faces:
        o, u, v = (np.array(a, dtype=np.float64) for a in (o, u, v))
        base = len(pos)
        for j in range(k + 1):
            for i in range(k + 1):
                pos.append(o + u * (i / k) + v * (j / k))
                uvs.append((i / k, j / k))
        for j in range(k):
            for i in range(k):
                a = base + j * (k + 1) + i
                b, c, d = a + 1, a + 1 + (k + 1), a + (k + 1)
                idx += [a, b, c, c, d, a]
    mb = MeshBuilder.new(np.array(pos, dtype=f32), LEFT).with_indices(idx)
    if with_uv:
        mb = mb.with_vertex_texture_coordinates_0(np.array(uvs, dtype=f32))
    if vertex_alpha_seed is not None:   # vertex colours whose alpha straddles a 0.5 cutout
        col = np.random.default_rng(vertex_alpha_seed).integers(0, 256, (len(pos), 4), dtype=np.uint8)
        mb = mb.with_vertex_color_0(col)
    return mb.build()


def textured_cube_scene(n_objects: int = 300, seed: int = 41, resolution: Tuple[int, int] = (320, 180), texture_size: int = 32,
                        sample_type: str = "linear", cutout: bool = False, block_compressed: bool = False, device_mips: bool = False) -> EvalOutput:
    """Cubes with texture coordinates and materials that exercise every texture slot and layout flag of PbrMaterial
    (opaque.wgsl:203-424): sRGB albedo, tri- and bi-component normal maps, combined / split AO-metallic-roughness, reflectance,
    clear coat, emissive, a scaled uv_transform0; one shadowed directional light and two point lights."""
    from .world import Texture

    rng = np.random.default_rng(seed)
    r = Renderer(LEFT, aspect_ratio=resolution[0] / resolution[1])
    meshes = [r.add_mesh(subdivided_cube_mesh(k, with_uv=True)) for k in (1, 2)]

    def smooth(channels_lo, channels_hi):   # low-frequency random texture: a few random texels upsampled bilinearly
        coarse = rng.uniform(channels_lo, channels_hi, (5, 5, 4))
        t = np.linspace(0, 4, texture_size, endpoint=False)
        i0 = np.floor(t).astype(int)
        f = (t - i0)[:, None]
        rows = coarse[i0] * (1 - f[..., None]) + coarse[np.minimum(i0 + 1, 4)] * f[..., None]
        img = rows[:, i0] * (1 - f[None, :, :]) + rows[:, np.minimum(i0 + 1, 4)] * f[None, :, :]
        return np.clip(np.rint(img * 255), 0, 255).astype(np.uint8)

    albedo = r.add_texture_2d(Texture(smooth(0.2, 1.0), srgb=True))
    normal = r.add_texture_2d(Texture(smooth((0.35, 0.35, 0.8, 0.35), (0.65, 0.65, 1.0, 0.65))))
    aomr = r.add_texture_2d(Texture(smooth((0.6, 0.3, 0.0, 0.0), (1.0, 0.9, 0.6, 1.0))))
    single = r.add_texture_2d(Texture(smooth(0.3, 0.9)))
    single_r8 = r.add_texture_2d(Texture(smooth(0.3, 0.9), channels=1))                                   # R8Unorm: reads (r, 0, 0, 1)
    normal_rg8 = r.add_texture_2d(Texture(smooth((0.35, 0.35, 0.0, 0.0), (0.65, 0.65, 0.0, 0.0)), channels=2))   # Rg8Unorm: bicomponent normal map
    emissive = r.add_texture_2d(Texture(smooth(0.0, 0.4), srgb=True))
    f32tex = r.add_texture_2d(Texture(rng.uniform(0.2, 0.8, (8, 8, 4)).astype(f32), mips="none"))
    ut = np.array([[2.0, 0, 0], [0, 1.5, 0], [0.25, 0.1, 1]], dtype=f32)
    mats = [
        PbrMaterial(albedo_texture=albedo, roughness_factor=0.5, sample_type=sample_type),
        PbrMaterial(albedo_texture=albedo, albedo_value=(0.9, 0.8, 0.7, 1.0), normal_texture=normal, roughness_texture=aomr, roughness_factor=0.9, metallic_factor=0.8,
                    ao_factor=0.9, sample_type=sample_type),
        PbrMaterial(albedo_value=(0.6, 0.6, 0.6, 1.0), normal_texture=normal_rg8, normal_kind="bicomponent", normal_y_down=True, aomr_kind="bw_split",
                    roughness_texture=single_r8, metallic_texture=single, ao_texture=single_r8, roughness_factor=0.8, metallic_factor=0.5, sample_type=sample_type),
        PbrMaterial(albedo_texture=albedo, normal_texture=normal, normal_kind="bicomponent_swizzled", aomr_kind="swizzled_split", roughness_texture=aomr, ao_texture=single,
                    roughness_factor=1.0, metallic_factor=1.0, reflectance_texture=single, reflectance=0.8, emissive=(1.0, 0.8, 0.6), emissive_texture=emissive,
                    uv_transform0=ut, sample_type=sample_type),
        PbrMaterial(albedo_texture=f32tex, aomr_kind="split", roughness_texture=aomr, roughness_factor=0.7, metallic_factor=0.4, clearcoat_factor=0.6,
                    clearcoat_roughness_factor=0.5, clearcoat_texture=aomr, clearcoat_kind="gltf_combined", sample_type=sample_type),
        PbrMaterial(albedo_texture=albedo, roughness_factor=0.6, clearcoat_factor=0.5, clearcoat_roughness_factor=0.8, clearcoat_kind="gltf_split",
                    clearcoat_texture=single, clearcoat_roughness_texture=aomr, anisotropy=0.3, anisotropy_texture=single, sample_type=sample_type),
        PbrMaterial(albedo_texture=albedo, unlit=True, sample_type=sample_type),
    ]
    if cutout:
        # cutout routine with per-fragment alpha: from the albedo texture, from the vertex colour, from both (opaque.wgsl:231-235,
        # depth.wgsl:101-127); the holes also show in the shadow map
        from .world import CUTOUT
        meshes += [r.add_mesh(subdivided_cube_mesh(3, with_uv=True, vertex_alpha_seed=seed + 1))]
        alpha_tex = r.add_texture_2d(Texture(smooth((0.3, 0.3, 0.3, 0.0), (1.0, 1.0, 1.0, 1.0)), srgb=True))
        mats += [
            PbrMaterial(albedo_texture=alpha_tex, roughness_factor=0.6, transparency=CUTOUT, alpha_cutout=0.5, sample_type=sample_type, uv_transform0=ut),
            PbrMaterial(albedo_value=(0.8, 0.7, 0.3, 1.0), albedo_vertex="linear", roughness_factor=0.6, transparency=CUTOUT, alpha_cutout=0.5),
            PbrMaterial(albedo_texture=alpha_tex, albedo_value=(1.0, 1.0, 1.0, 1.3), albedo_vertex="srgb", roughness_factor=0.6, transparency=CUTOUT, alpha_cutout=0.4,
                        sample_type=sample_type),
        ]
    if block_compressed:
        # the same images as the ktx2 / dds assets rend3-gltf would load (rend3-gltf/src/lib.rs:1300-1335): BC1 / BC3 sRGB colour maps, BC1 / BC2
        # linear maps, BC4 single-channel and BC5 two-channel maps, BC7 (mode 6) for a linear and an sRGB map; the float texture stays uncompressed
        for handle, name in ((albedo, "bc1"), (normal, "bc3"), (aomr, "bc2"), (single, "bc7"), (single_r8, "bc4"), (normal_rg8, "bc5"), (emissive, "bc7")):
            r.textures[handle].block_format = name
        if cutout:
            r.textures[alpha_tex].block_format = "bc3"
    if device_mips:   # MipmapSource::Generated as rend3 does it: level 0 uploaded, the chain rendered on the device (r3_generate_mipmaps, rule R12)
        for t in r.textures:
            if t.mips == "generated" and t.block_format is None:
                t.mips = "device"
    mat_ids = [r.add_material(m) for m in mats]
    r.set_camera_data(cube_example_camera(8.0))
    r.add_directional_light(DirectionalLight(color=(1, 1, 1), intensity=1.0, direction=(-1.0, -4.0, 2.0), distance=80.0, resolution=256))
    for _ in range(2):
        r.add_point_light(PointLight(position=tuple(rng.uniform(-10, 10, 3)), color=tuple(rng.uniform(0.3, 1.0, 3)), radius=18.0, intensity=3.0))
    centers = rng.uniform(-14.0, 14.0, (n_objects, 3)).astype(f32)
    scale = rng.uniform(0.8, 3.0, (n_objects, 1)).astype(f32)
    transforms = trs_matrices(centers, random_unit_quaternions(rng, n_objects), scale)
    for i in range(n_objects):
        mi = mat_ids[i % len(mat_ids)]
        vertex_coloured = cutout and (i % len(mat_ids)) >= len(mat_ids) - 2
        r.add_object(Object(meshes[2] if vertex_coloured else meshes[i % 2], mi, transforms[i]))
    return r.evaluate()


def cube_field_scene(n_objects: int = 10_000, seed: int = 1, resolution: Tuple[int, int] = (1920, 1080), extent: float = 50.0,
                     pull_back: float = 20.0, n_point_lights: int = 0, n_dir_lights: int = 1, shadow_resolution: int = 2048,
                     shadow_distance: float = 400.0, roughness: float = 0.5, subdivisions=(1,), material_count: int = 1,
                     scale_range: Tuple[float, float] = (0.2, 1.0), slabs: bool = False, mixed_transparency: bool = False) -> EvalOutput:
    """BASELINE config C1 family (SURVEY.md 8d): n cubes, centres U([-extent, extent]^3), uniform scale U(0.2, 1),
    random rotation, PBR material albedo 0.5, directional light(s) like examples/src/cube, camera pulled back."""
    rng = np.random.default_rng(seed)
    r = Renderer(LEFT, aspect_ratio=resolution[0] / resolution[1])
    mesh_ids_avail = [r.add_mesh(subdivided_cube_mesh(k)) for k in subdivisions]
    for m in range(material_count):
        g = 0.5 if material_count == 1 else 0.25 + 0.5 * (m / max(material_count - 1, 1))
        # mixed_transparency: materials cycle opaque / cutout / blend, i.e. material keys 0 / 1 / 2 (pbr/material.rs:497-503)
        transparency = (m % 3) if mixed_transparency else 0
        # every other cutout material has alpha below its cutout threshold: its objects are discarded in the forward and shadow passes
        alpha = 0.3 if (mixed_transparency and m % 6 == 1) else 1.0
        if mixed_transparency and m % 3 == 2:
            alpha = 0.25 + 0.5 * (m / max(material_count - 1, 1))   # blend materials are actually translucent
        r.add_material(PbrMaterial(albedo_value=(0.5, g, 0.5 if material_count == 1 else 1.0 - g, alpha), roughness_factor=roughness,
                                   transparency=transparency, alpha_cutout=0.5))
    r.set_camera_data(cube_example_camera(pull_back))
    dirs = [(-1.0, -4.0, 2.0), (2.0, -3.0, -1.0), (-2.0, -5.0, -3.0), (1.0, -2.0, 3.0)]
    for i in range(n_dir_lights):
        r.add_directional_light(DirectionalLight(color=(1, 1, 1), intensity=1.0 / max(n_dir_lights, 1), direction=dirs[i % 4],
                                                 distance=shadow_distance, resolution=shadow_resolution))
    for i in range(n_point_lights):
        p = rng.uniform(-extent, extent, 3)
        col = rng.uniform(0.2, 1.0, 3)
        r.add_point_light(PointLight(position=tuple(p), color=tuple(col), radius=float(rng.uniform(5.0, 20.0)), intensity=4.0))
    centers = rng.uniform(-extent, extent, (n_objects, 3)).astype(f32)
    scale = rng.uniform(scale_range[0], scale_range[1], (n_objects, 1)).astype(f32)
    quat = random_unit_quaternions(rng, n_objects)
    transforms = trs_matrices(centers, quat, scale)
    mesh_ids = np.asarray(mesh_ids_avail, dtype=np.int64)[rng.integers(0, len(mesh_ids_avail), n_objects)]
    material_ids = rng.integers(0, material_count, n_objects).astype(np.uint32)
    if slabs:
        # a floor and two back walls (one 12-triangle box each) so that the frame is fully covered, as in an interior scene;
        # their screen-filling triangles exercise the banded large-triangle path
        slab_mesh = r.add_mesh(cube_mesh())
        e, t = f32(extent * 1.25), f32(0.5)
        sc = np.array([[e, t, e], [t, e, e], [e, e, t]], dtype=f32)
        tr = np.array([[0, -e, 0], [-e, 0, 0], [0, 0, e]], dtype=f32)
        ident = np.tile(np.array([[0, 0, 0, 1]], dtype=f32), (3, 1))
        transforms = np.concatenate([transforms, trs_matrices(tr, ident, sc)])
        mesh_ids = np.concatenate([mesh_ids, np.full(3, slab_mesh, dtype=np.int64)])
        material_ids = np.concatenate([material_ids, np.zeros(3, dtype=np.uint32)])
        n_objects += 3
    rec, loc = bulk_object_records(r, transforms, mesh_ids, material_ids)
    return eval_with_bulk_objects(r, rec, loc, n_objects)


def object_cloud_records(n: int, seed: int = 2, extent: float = 1000.0, disabled_fraction: float = 0.01) -> np.ndarray:
    """BASELINE configs C2 / C4: object records only (no mesh work).  Centres U([-extent, extent]^3), uniform scale
    log-U(0.1, 10), random rotation, bounding radius sqrt(3) * scale (unit cube mesh), 1% disabled."""
    rng = np.random.default_rng(seed)
    rec = np.zeros(n, dtype=OBJECT_DTYPE)
    chunk = 1 << 20
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        m = e - s
        centers = rng.uniform(-extent, extent, (m, 3)).astype(f32)
        scale = np.exp(rng.uniform(np.log(0.1), np.log(10.0), (m, 1))).astype(f32)
        t = trs_matrices(centers, random_unit_quaternions(rng, m), scale)
        rec["transform"][s:e] = t.reshape(m, 16)
        rec["sphere_center"][s:e] = centers
        ls = [((t[:, k, 0] * t[:, k, 0] + t[:, k, 1] * t[:, k, 1]).astype(f32) + t[:, k, 2] * t[:, k, 2]).astype(f32) for k in range(3)]
        rec["sphere_radius"][s:e] = (np.sqrt(np.maximum(ls[0], np.maximum(ls[1], ls[2]))).astype(f32) * f32(np.sqrt(f32(3.0)))).astype(f32)
        rec["index_count"][s:e] = 36
        rec["attr_offset"][s:e] = [0, 288, ATTR_ABSENT, ATTR_ABSENT, ATTR_ABSENT, ATTR_ABSENT]
        rec["first_index"][s:e] = 144
        rec["enabled"][s:e] = (rng.random(m) >= disabled_fraction).astype(np.uint32)
    return rec


def cloud_camera(resolution: Tuple[int, int] = (1920, 1080), pull_back: float = 150.0):
    """Camera family of the cull-only configs: the cube-example view pulled back into the cloud."""
    from .world import CameraState

    return CameraState(cube_example_camera(pull_back), LEFT, resolution[0] / resolution[1])
