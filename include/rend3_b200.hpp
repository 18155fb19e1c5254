// rend3_b200.hpp — C++17 host-side mirror of rend3-routine's interface for the hot path, header-only, on top of the C ABI
// (include/rend3_b200.h).  The reference's host side is compiled code (Rust); no Rust toolchain exists in this image, so this is
// the native stand-in a C++ engine — or a Rust shim through the same C symbols (INTEGRATION.md) — would drive.  Names, argument
// meaning and call order follow the reference:
//
//   r3::GpuCuller::object_uniform_upload      rend3-routine/src/culling/culler.rs:427-529
//   r3::GpuSkinner::add_skinning_to_graph     skinning.rs:54-199 (node position base.rs:145)
//   r3::GpuCuller::add_culling_to_graph       culler.rs:682-713 (batch_objects, batching.rs:120-250, then cull, culler.rs:531-659)
//   r3::ForwardRoutine::add_forward_to_graph  forward.rs:192-315      r3::HiZRoutine::add_hi_z_to_graph   hi_z.rs:161-234
//   r3::TonemappingRoutine::add_to_graph      tonemapping.rs:108-147  r3::BaseRenderGraph::add_to_graph   base.rs:129-185
//
// What stays with the engine's managers is INPUT here, as the bytes they upload today: the object / material / light buffers,
// the PerCameraUniform header of every camera (culler.rs:484-505) and FrameUniforms (uniforms.rs:30-49).
// Error behaviour: the reference panics inside graph nodes (e.g. culler.rs:439,572); here every failure throws r3::Error carrying
// the C ABI's code and r3_last_error text — nothing unwinds across the C boundary.
#ifndef REND3_B200_HPP
#define REND3_B200_HPP

#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "rend3_b200.h"

namespace r3 {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};

enum class SampleCount : uint32_t { One = 1, Four = 4 };        // rend3-types SampleCount
enum class CullingSource { Predicted, Residual };               // forward.rs:134-142

// CameraSpecifier (rend3-routine/src/common/camera.rs): Viewport or Shadow(index); to_shader_index() is what the kernels see
struct CameraSpecifier {
    uint32_t index;
    static CameraSpecifier Viewport() { return {R3_CAMERA_VIEWPORT}; }
    static CameraSpecifier Shadow(uint32_t i) { return {i}; }
    bool is_shadow() const { return index != R3_CAMERA_VIEWPORT; }
    uint32_t to_shader_index() const { return index; }
};

// One shadow map of a directional light: its camera's PerCameraUniform header + the atlas viewport (directional.rs:24-119)
struct ShadowMap {
    r3_camera_header header;
    uint32_t offset[2];
    uint32_t size;
};

// What Renderer::evaluate_instructions leaves for the routines (renderer/eval.rs:9-181), as spans over the managers' bytes
struct EvalOutput {
    const r3_object* objects = nullptr; uint32_t n_slots = 0;                                   // object_manager.buffer::<M>()
    const uint64_t* material_key = nullptr; const uint8_t* sort_flags = nullptr; const float* location = nullptr;   // per slot
    const void* mesh_buffer = nullptr; uint64_t mesh_bytes = 0;
    const r3_material* materials = nullptr; uint32_t n_materials = 0;
    const r3_texture_desc* textures = nullptr; uint32_t n_textures = 0; const void* texels = nullptr; uint64_t texel_bytes = 0;
    const uint32_t* generated_textures = nullptr; uint32_t n_generated = 0;   // table entries added with MipmapSource::Generated (texture.rs:146-180)
    const r3_texture_desc* skybox = nullptr; const void* skybox_texels = nullptr; uint64_t skybox_bytes = 0;     // SkyboxRoutine's cube map (null = none)
    const void* directional_lights = nullptr; uint64_t directional_bytes = 0; uint32_t shadow_target_size[2] = {0, 0};
    const void* point_lights = nullptr; uint64_t point_bytes = 0;
    std::vector<ShadowMap> shadows;
    r3_camera_header viewport{};              // PerCameraUniform header of the viewport camera for this target
    r3_frame_uniforms uniforms{};             // FrameUniforms::new
    float viewport_location[3] = {0, 0, 0};   // CameraState::location()
    // GPU skinning (skinning.rs:54-199): one record per skeleton + the global joint matrices; empty = no animated meshes this frame
    const r3_skinning_input* skinning_inputs = nullptr; uint32_t n_skeletons = 0; const float* joint_matrices = nullptr; uint32_t n_joints = 0;
};

struct BaseRenderGraphSettings {              // base.rs:95-98
    std::array<float, 4> ambient_color{0, 0, 0, 0};
    std::array<float, 4> clear_color{0, 0, 0, 0};
};

// Owns the device context (one per GPU); calls are externally serialised like rend3's data_core lock (graph.rs:265)
class Renderer {
public:
    explicit Renderer(int device) {
        const int rc = r3_ctx_create(device, &ctx_);
        if (rc != R3_OK) throw Error(rc, rc == R3_E_NO_DEVICE ? "no CUDA device (there is no CPU fallback)" : "r3_ctx_create failed");
    }
    ~Renderer() { if (ctx_) r3_ctx_destroy(ctx_); }
    Renderer(const Renderer&) = delete;
    Renderer& operator=(const Renderer&) = delete;
    r3_ctx* raw() const { return ctx_; }
    void check(int rc) const { if (rc != R3_OK) throw Error(rc, r3_last_error(ctx_)); }

    // renderer/eval.rs:157-181 — the buffers evaluate_instructions (re)uploads
    void upload_world(const EvalOutput& ev) {
        check(r3_set_objects(ctx_, ev.objects, ev.n_slots));
        if (ev.material_key) check(r3_set_object_sort_info(ctx_, ev.material_key, ev.sort_flags, ev.location, ev.n_slots));
        check(r3_set_mesh_buffer(ctx_, ev.mesh_buffer, ev.mesh_bytes));
        check(r3_set_textures(ctx_, ev.textures, ev.n_textures, ev.texels, ev.texel_bytes));
        if (ev.n_generated) check(r3_generate_mipmaps(ctx_, ev.generated_textures, ev.n_generated));   // MipmapGenerator::generate_mipmaps
        check(r3_set_skybox(ctx_, ev.skybox, ev.skybox_texels, ev.skybox_bytes));
        check(r3_set_materials(ctx_, ev.materials, ev.n_materials));
        check(r3_set_directional_lights(ctx_, ev.directional_lights, ev.directional_bytes, ev.shadow_target_size[0], ev.shadow_target_size[1]));
        check(r3_set_point_lights(ctx_, ev.point_lights, ev.point_bytes));
    }
    void sync() { check(r3_sync(ctx_)); }

private:
    r3_ctx* ctx_ = nullptr;
};

class GpuCuller {   // culling/culler.rs:185-714
public:
    // object_uniform_upload: MV / MVP for every enabled slot + (fused here) the sphere-frustum filter of batch_objects
    void object_uniform_upload(Renderer& r, CameraSpecifier camera, const r3_camera_header& header) const {
        r.check(r3_object_uniform_upload(r.raw(), camera.to_shader_index(), &header, R3_CB_BAKE | R3_CB_CULL));
    }
    // add_culling_to_graph: batch_objects, then the per-triangle cull into the ping-pong CullingBuffers
    void add_culling_to_graph(Renderer& r, CameraSpecifier camera, const float viewport_location[3], uint32_t max_compute_workgroups_per_dimension = 65535) const {
        r.check(r3_batch_objects(r.raw(), camera.to_shader_index(), viewport_location, max_compute_workgroups_per_dimension));
        r.check(r3_cull(r.raw(), camera.to_shader_index(), nullptr, 0, nullptr, 0));
    }
};

class GpuSkinner {   // skinning.rs:54-199: add_skinning_to_graph — skinned positions / normals / tangents into the skeletons' overridden mesh ranges
public:
    void add_skinning_to_graph(Renderer& r, const EvalOutput& ev) const {
        if (ev.n_skeletons) r.check(r3_skin(r.raw(), ev.skinning_inputs, ev.n_skeletons, ev.joint_matrices, ev.n_joints));
    }
};

class ForwardRoutine {   // forward.rs:85-315; opaque + cutout routines share one call, the blend routine has its own
public:
    void add_forward_to_graph(Renderer& r, CullingSource source) const { r.check(r3_forward_pass(r.raw(), source == CullingSource::Predicted ? 0 : 1)); }
    void add_shadow_to_graph(Renderer& r, uint32_t shadow_index, const ShadowMap& map) const {   // pbr_shadow_rendering, base.rs:366-396
        r.check(r3_shadow_pass(r.raw(), shadow_index, map.offset[0], map.offset[1], map.size));
    }
    void resolve(Renderer& r) const { r.check(r3_forward_resolve(r.raw())); }                     // fs_main of the winning fragments (+ SkyboxRoutine, base.rs:175)
    void add_transparent_to_graph(Renderer& r) const { r.check(r3_forward_blend(r.raw())); }       // pbr_forward_rendering_transparent
};

class HiZRoutine {
public:
    void add_hi_z_to_graph(Renderer& r) const { r.check(r3_hiz_build(r.raw())); }
};

class TonemappingRoutine {
public:
    void add_to_graph(Renderer& r, bool target_is_srgb) const { r.check(r3_tonemap(r.raw(), target_is_srgb ? 1 : 0)); }
};

// BaseRenderGraph::add_to_graph (base.rs:129-185): the node order of one frame, collapsed to a stream-ordered call sequence
class BaseRenderGraph {
public:
    GpuCuller gpu_culler;
    GpuSkinner gpu_skinner;
    ForwardRoutine forward;
    HiZRoutine hi_z;
    TonemappingRoutine tonemapping;
    bool submit_as_graph = false;             // record the frame and submit it as one CUDA graph launch (graph.rs:510: one submit per frame)

    void add_to_graph(Renderer& r, const EvalOutput& ev, uint32_t width, uint32_t height, SampleCount samples, const BaseRenderGraphSettings& settings,
                      bool target_is_srgb = true) {
        r.check(r3_set_render_target(r.raw(), width, height, (uint32_t)samples, settings.clear_color.data()));
        if (submit_as_graph) r.check(r3_frame_begin(r.raw()));
        r.check(r3_clear_shadow_atlas(r.raw()));                                                     // base.rs:139
        r.check(r3_set_frame_uniforms(r.raw(), &ev.uniforms));                                       // :142
        gpu_skinner.add_skinning_to_graph(r, ev);                                                    // :145 state.skinning — before any camera culls
        for (uint32_t i = 0; i < ev.shadows.size(); ++i) gpu_culler.object_uniform_upload(r, CameraSpecifier::Shadow(i), ev.shadows[i].header);   // :148
        for (uint32_t i = 0; i < ev.shadows.size(); ++i) gpu_culler.add_culling_to_graph(r, CameraSpecifier::Shadow(i), ev.viewport_location);     // :150
        for (uint32_t i = 0; i < ev.shadows.size(); ++i) forward.add_shadow_to_graph(r, i, ev.shadows[i]);                                         // :153
        gpu_culler.object_uniform_upload(r, CameraSpecifier::Viewport(), ev.viewport);               // :156
        r.check(r3_forward_begin(r.raw()));
        forward.add_forward_to_graph(r, CullingSource::Predicted);                                   // :159
        hi_z.add_hi_z_to_graph(r);                                                                   // :162
        gpu_culler.add_culling_to_graph(r, CameraSpecifier::Viewport(), ev.viewport_location);       // :169
        forward.add_forward_to_graph(r, CullingSource::Residual);                                    // :172
        forward.resolve(r);
        forward.add_transparent_to_graph(r);                                                         // :181
        tonemapping.add_to_graph(r, target_is_srgb);                                                 // :184
        if (submit_as_graph) r.check(r3_frame_end(r.raw()));
    }
};

}  // namespace r3
#endif
