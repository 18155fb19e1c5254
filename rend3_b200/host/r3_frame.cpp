// r3_frame — renders frames of a dumped scene through the C++ host mirror (include/rend3_b200.hpp) and writes the artefacts
// the parity tests compare.  usage: r3_frame <scene.r3s> <out.r3o> [device]
// The scene file is what the engine's managers would hand over each frame (rend3_b200/scene_io.py writes it from the Python
// scene generators); sections are  u32 tag_len | tag | u64 nbytes | payload.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <string>

#include "rend3_b200.hpp"

using Blob = std::vector<uint8_t>;

static std::map<std::string, Blob> read_sections(const char* path) {
    std::ifstream f(path, std::ios::binary);
    if (!f) throw std::runtime_error(std::string("cannot open ") + path);
    std::map<std::string, Blob> out;
    for (;;) {
        uint32_t tl = 0;
        if (!f.read(reinterpret_cast<char*>(&tl), 4)) break;
        std::string tag(tl, '\0');
        uint64_t n = 0;
        f.read(&tag[0], tl);
        f.read(reinterpret_cast<char*>(&n), 8);
        Blob b(n);
        if (n) f.read(reinterpret_cast<char*>(b.data()), (std::streamsize)n);
        if (!f) throw std::runtime_error("truncated scene file");
        out[tag] = std::move(b);
    }
    return out;
}
static void write_section(std::ofstream& f, const std::string& tag, const void* p, uint64_t n) {
    const uint32_t tl = (uint32_t)tag.size();
    f.write(reinterpret_cast<const char*>(&tl), 4);
    f.write(tag.data(), tl);
    f.write(reinterpret_cast<const char*>(&n), 8);
    if (n) f.write(reinterpret_cast<const char*>(p), (std::streamsize)n);
}
template <typename T>
static const T* as(const std::map<std::string, Blob>& s, const char* tag, uint64_t* count = nullptr) {
    const auto it = s.find(tag);
    if (it == s.end()) throw std::runtime_error(std::string("scene file lacks section ") + tag);
    if (count) *count = it->second.size() / sizeof(T);
    return it->second.empty() ? nullptr : reinterpret_cast<const T*>(it->second.data());
}

int main(int argc, char** argv) {
    if (argc < 3) { std::fprintf(stderr, "usage: r3_frame <scene.r3s> <out.r3o> [device]\n"); return 2; }
    try {
        const auto s = read_sections(argv[1]);
        r3::EvalOutput ev;
        uint64_t n = 0;
        ev.objects = as<r3_object>(s, "objects", &n); ev.n_slots = (uint32_t)n;
        ev.material_key = as<uint64_t>(s, "material_key"); ev.sort_flags = as<uint8_t>(s, "sort_flags"); ev.location = as<float>(s, "location");
        ev.mesh_buffer = as<uint8_t>(s, "mesh", &n); ev.mesh_bytes = n;
        ev.materials = as<r3_material>(s, "materials", &n); ev.n_materials = (uint32_t)n;
        ev.textures = as<r3_texture_desc>(s, "tex_descs", &n); ev.n_textures = (uint32_t)n;
        ev.texels = as<uint8_t>(s, "texels", &n); ev.texel_bytes = n;
        if (s.count("tex_generated")) { ev.generated_textures = as<uint32_t>(s, "tex_generated", &n); ev.n_generated = (uint32_t)n; }   // absent: none
        if (s.count("skybox_desc") && !s.at("skybox_desc").empty()) {
            ev.skybox = as<r3_texture_desc>(s, "skybox_desc");
            ev.skybox_texels = as<uint8_t>(s, "skybox_texels", &n); ev.skybox_bytes = n;
        }
        ev.directional_lights = as<uint8_t>(s, "dir_lights", &n); ev.directional_bytes = n;
        ev.point_lights = as<uint8_t>(s, "point_lights", &n); ev.point_bytes = n;
        const uint32_t* st = as<uint32_t>(s, "shadow_target");
        ev.shadow_target_size[0] = st[0]; ev.shadow_target_size[1] = st[1];
        struct ShadowRec { r3_camera_header header; uint32_t ox, oy, size, pad; };
        static_assert(sizeof(ShadowRec) == 256, "shadow record");
        const ShadowRec* sh = as<ShadowRec>(s, "shadows", &n);
        for (uint64_t i = 0; i < n; ++i) ev.shadows.push_back(r3::ShadowMap{sh[i].header, {sh[i].ox, sh[i].oy}, sh[i].size});
        ev.viewport = *as<r3_camera_header>(s, "viewport_header");
        ev.uniforms = *as<r3_frame_uniforms>(s, "uniforms");
        std::memcpy(ev.viewport_location, as<float>(s, "viewport_location"), 12);
        const float* set = as<float>(s, "settings");
        r3::BaseRenderGraphSettings settings;
        for (int k = 0; k < 4; ++k) { settings.ambient_color[k] = set[k]; settings.clear_color[k] = set[4 + k]; }
        const uint32_t* tg = as<uint32_t>(s, "target");   // width, height, samples, srgb target, frames
        const uint32_t width = tg[0], height = tg[1], frames = tg[4] ? tg[4] : 1;

        r3::Renderer renderer(argc > 3 ? std::atoi(argv[3]) : 0);
        renderer.check(r3_set_parity_target(renderer.raw(), 1));   // this driver exists for the parity tests: keep the f32 shading result
        r3::BaseRenderGraph graph;
        graph.submit_as_graph = std::getenv("R3_FRAME_GRAPH") && std::getenv("R3_FRAME_GRAPH")[0] != '0';
        renderer.upload_world(ev);
        for (uint32_t f = 0; f < frames; ++f)
            graph.add_to_graph(renderer, ev, width, height, tg[2] == 4 ? r3::SampleCount::Four : r3::SampleCount::One, settings, tg[3] != 0);
        renderer.sync();

        const uint64_t px = (uint64_t)width * height;
        std::vector<float> hdr(px * 4), depth(px);
        std::vector<uint8_t> ldr(px * 4);
        std::vector<uint32_t> visible(ev.n_slots ? ev.n_slots : 1);
        uint32_t n_visible = 0;
        uint64_t stats[4] = {0, 0, 0, 0};
        renderer.check(r3_readback_hdr_f32(renderer.raw(), hdr.data(), hdr.size()));
        renderer.check(r3_readback_depth(renderer.raw(), depth.data(), depth.size()));
        renderer.check(r3_readback_ldr(renderer.raw(), ldr.data(), ldr.size()));
        renderer.check(r3_readback_visible(renderer.raw(), R3_CAMERA_VIEWPORT, visible.data(), (uint32_t)visible.size(), &n_visible));
        renderer.check(r3_forward_stats(renderer.raw(), stats));
        std::ofstream o(argv[2], std::ios::binary);
        write_section(o, "hdr", hdr.data(), hdr.size() * 4);
        write_section(o, "depth", depth.data(), depth.size() * 4);
        write_section(o, "ldr", ldr.data(), ldr.size());
        write_section(o, "visible", visible.data(), (uint64_t)n_visible * 4);
        write_section(o, "stats", stats, sizeof stats);
        std::printf("r3_frame: %u frame(s) %ux%u, %u visible objects, %llu fragments shaded\n", frames, width, height, n_visible, (unsigned long long)stats[2]);
        return 0;
    } catch (const r3::Error& e) {
        std::fprintf(stderr, "r3_frame: library error %d: %s\n", e.code, e.what());
        return 1;
    } catch (const std::exception& e) {
        std::fprintf(stderr, "r3_frame: %s\n", e.what());
        return 1;
    }
}
