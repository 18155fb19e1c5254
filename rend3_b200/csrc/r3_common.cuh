// r3_common.cuh — shared declarations of librend3_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/rend3_b200.h"

#define R3_EXPORT extern "C" __attribute__((visibility("default")))

constexpr int R3_MAX_CAMERAS = 64;          // slot 0 = viewport, 1+i = shadow i
constexpr int R3_SM_COUNT = 148;            // B200: 2 dies x 74 SMs

struct r3_iobuf {                           // InputOutputBuffer, rend3-routine/src/culling/suballoc.rs:17-223
    uint8_t* d = nullptr;
    uint64_t capacity_elements = 0, out_elems = 0, in_elems = 0, elem_size = 0;
    bool flipped = false, clear_on_swap = false, created = false;
    uint64_t out_off() const { return flipped ? capacity_elements / 2 : 0; }
    uint64_t in_off() const { return flipped ? 0 : capacity_elements / 2; }
};

// device-side description of the draw calls of one camera/frame (what forward.rs:290-313 walks)
struct r3_jobs {
    r3_batch_data* d_batches = nullptr; uint32_t batches_cap = 0, n_batches = 0;
    r3_region* d_regions = nullptr; uint32_t regions_cap = 0, n_regions = 0;
    uint32_t* d_region_first_inv = nullptr;   // [n_regions+1] first global invocation of each region
    // device-side job header the downstream kernels read their counts from (so a frame needs no host sync):
    // [0] n_visible  [1] n_batches  [2] n_regions  [3] total_invocations  [4] overflow flag
    uint32_t* d_header = nullptr;
    uint32_t total_invocations = 0;           // exact (host batching) or an upper bound (device batching)
    bool device_built = false;                // host vectors are filled lazily by readbacks
    std::vector<r3_batch_data> batches;      // host copies (batch_objects builds these on the CPU)
    std::vector<r3_region> regions;
    bool valid = false;
};

// optional per-stage device timing (r3_set_stage_timing / r3_stage_times): CUDA event pairs around the kernels named below, so that
// bench.py can put a measured duration next to each kernel's algorithmic bytes / flops.  Off by default: no events are recorded.
enum { R3_STAGE_TRIANGLE_TEST = 0, R3_STAGE_RASTER_SETUP_COLOUR, R3_STAGE_RASTER_SETUP_DEPTH, R3_STAGE_RASTER_BANDS, R3_STAGE_RESOLVE, R3_STAGE_SORT,
       R3_STAGE_CULL_BAKE, R3_STAGE_TRIANGLE_COMPACT, R3_STAGE_MIPMAPS, R3_STAGE_COUNT };
struct r3_stage_timer {
    bool enabled = false;
    std::vector<cudaEvent_t> pool;            // recycled events: [2 k] start, [2 k + 1] stop
    std::vector<int> stage_of;                // stage of pair k
    size_t used = 0;
};
constexpr int R3_MAX_EXCHANGE_RANKS = 16;
constexpr int R3_EXCHANGE_SLOTS = 4;         // row sets of the visible-set exchange in flight (epoch % slots)
// peer-memory plumbing of the multi-GPU forward pass (r3_peer.cu): kinds of epoch flags
constexpr uint32_t R3_PEER_KINDS = 4;        // 0 shadow atlas rects, 1 colour rows, 2 frame done, 3 visibility words of the sharded triangle test
struct r3_peer_state {
    bool created = false, connected = false, has_atlas = false;
    uint32_t n_ranks = 0, rank = 0;
    uint32_t* d_flags = nullptr;              // this rank's flags[R3_PEER_KINDS][R3_MAX_EXCHANGE_RANKS]
    uint32_t* flags[R3_MAX_EXCHANGE_RANKS] = {}; float* atlas[R3_MAX_EXCHANGE_RANKS] = {}; uint16_t* hdr16[R3_MAX_EXCHANGE_RANKS] = {};   // peer mappings
    uint32_t sent[R3_PEER_KINDS] = {0, 0, 0, 0};
    uint32_t* d_tri_words = nullptr; uint64_t tri_cap_words = 0; uint32_t* tri_words[R3_MAX_EXCHANGE_RANKS] = {};   // staging arrays of the sharded triangle test
    const void* atlas_at_create = nullptr; const void* hdr_at_create = nullptr;
    cudaEvent_t side_event = nullptr; bool atlas_on_side = false;   // atlas copies run on the context's side stream
};
struct r3_camera {
    bool header_set = false;
    r3_camera_header header{};
    r3_object_matrices* d_matrices = nullptr; uint32_t matrices_cap = 0;
    uint32_t* d_visible = nullptr; uint32_t visible_cap = 0;
    uint32_t* d_visible_count = nullptr;      // device scalar
    unsigned long long* d_tile_state = nullptr; uint32_t tile_state_cap = 0;   // visibility words + per-CTA counts (two alternating sets)
    uint32_t* d_words = nullptr; uint32_t words_set = 0;                       // the set the last cull wrote
    // multi-GPU exchange of the visible set over NVLink peer memory (r3_exchange_*): gathered[n_ranks][words_per_rank]
    uint32_t* d_gathered = nullptr; uint32_t ex_ranks = 0, ex_rank = 0, ex_words_per_rank = 0; bool ex_connected = false;
    uint32_t* ex_peers[R3_MAX_EXCHANGE_RANKS] = {};   // peer-mapped gathered buffers (ex_peers[ex_rank] == d_gathered)
    uint32_t ex_epoch = 0, ex_objects = 0; uint32_t* d_ex_done = nullptr;       // step counter (parity = epoch & 1), CTA arrival counter of the publishing kernel
    cudaEvent_t ex_cull_done[R3_EXCHANGE_SLOTS] = {}, ex_merge_done[R3_EXCHANGE_SLOTS] = {}; bool ex_merge_pending[R3_EXCHANGE_SLOTS] = {}; uint32_t ex_consumed[R3_EXCHANGE_SLOTS] = {};   // consumers on the side stream; last epoch consumed per slot
    uint32_t* d_global_visible = nullptr; uint64_t global_visible_cap = 0; uint32_t* d_merge_counts = nullptr; uint64_t merge_counts_cap = 0;   // r3_exchange_merge
    int visible_count_host = -1;              // cached after a readback, -1 = unknown
    r3_jobs jobs[2]; int cur = 0;             // jobs[cur] = this frame, jobs[cur^1] = cached DrawCallSet (forward.rs:219)
    int batching_path = 0;                    // which batch_objects ran last for this camera: 0 none, 1 device, 2 host, 3 device with the frame-wide sort (r3_batching_info)
    uint64_t gsort_epoch_used = ~0ull;        // frame epoch in which this camera last batched (r3_gpu_batching.cu)
    bool has_draw_call_set = false; int cache_idx = -1;   // cache_idx: which jobs[] the forward routine cached, -1 = none
    std::vector<uint32_t> prev_invocation;    // PerCameraPreviousInvocationsMap (batching.rs:102-118), host batching
    uint32_t* d_prev_inv[2] = {nullptr, nullptr}; uint32_t prev_inv_cap = 0; int prev_inv_cur = 0;   // same map, device batching
    unsigned long long* d_sort_keys[2] = {nullptr, nullptr}; uint64_t sort_keys_cap = 0, sort_keys_cap2 = 0;
    uint32_t* d_sort_hist = nullptr; uint64_t sort_hist_cap = 0;
    uint32_t* d_batch_tmp = nullptr; uint64_t batch_tmp_cap = 0;
    r3_iobuf index_buffer, draw_call_buffer, results_buffer;   // CullingBuffers (culler.rs:88-125)
    // scratch of the ordered triangle compaction
    uint32_t* d_resid_bits = nullptr; uint64_t resid_bits_cap = 0;
    unsigned long long* d_word_scan = nullptr; uint64_t word_scan_cap = 0;
    unsigned long long* d_block_sums = nullptr; uint64_t block_sums_cap = 0;
};

// one job of r3_generate_mipmaps' work list (r3_mipmap.cu): a texture's source level and how many levels one launch derives from it
struct r3_mip_job {
    uint64_t src_off;                         // byte offset of the source level in the texel blob
    uint32_t sw, sh, fmt, levels;             // source size, format, levels produced (head: fused levels, level kernel: 1, tail: the rest)
    uint32_t tiles_x;                         // head: 64x64 tiles per row; level kernel: 256-texel segments per destination row
    uint32_t item_begin;                      // first work item of the job within its launch
};
static_assert(sizeof(r3_mip_job) == 32, "mip job");

struct r3_tri_record { float xyw[3][3]; uint32_t object_id; uint32_t vid[3]; uint32_t _pad[3]; };   // 64 B
static_assert(sizeof(r3_tri_record) == 64, "triangle record");

struct r3_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t side_stream = nullptr;       // low-priority stream of the exchange consumer (r3_exchange_merge), created on first use
    std::string err;
    uint64_t launches = 0;
    bool coop_launch_ok = false;              // cudaDevAttrCooperativeLaunch (grid-wide barriers inside one launch)
    // world
    r3_object* d_objects = nullptr; uint32_t n_slots = 0, objects_cap = 0; bool objects_borrowed = false;
    // dense copies of the fields the cull + bake stream reads (r3_cull_bake.cu): transform columns, bounding spheres, enabled bits
    float4* d_hot_transform = nullptr; float4* d_hot_sphere = nullptr; uint32_t* d_enabled_bits = nullptr; uint64_t hot_cap = 0; bool hot_valid = false;
    std::vector<uint64_t> sort_key; std::vector<uint8_t> sort_flags; std::vector<float> sort_loc;
    uint32_t* d_live_bits = nullptr; uint32_t live_bits_cap = 0; bool have_live = false;
    uint8_t* d_sort_key8 = nullptr; float* d_sort_loc = nullptr; uint32_t sort_dev_cap = 0; bool gpu_batching_ok = false;
    // frame-wide sort shared by the cameras of one frame (r3_gpu_batching.cu)
    unsigned long long* d_gsort_keys[2] = {nullptr, nullptr}; uint64_t gsort_cap[2] = {0, 0}; uint32_t* d_gsort_hist = nullptr; uint64_t gsort_hist_cap = 0;
    uint32_t* d_gsort_header = nullptr; int gsort_src = 0; uint32_t gsort_n = 0; bool gsort_valid = false; float gsort_loc[3] = {0, 0, 0};
    uint64_t gsort_epoch = 0, gsort_sorted_epoch = ~0ull; uint32_t gsort_cameras_this_epoch = 0, gsort_cameras_last_epoch = 0;
    uint64_t max_total_invocations = 0, max_object_invocations = 0; bool max_invocations_valid = false;   // sum / max over all slots of round_up(tris, 256)
    uint32_t* d_mesh = nullptr; uint64_t mesh_words = 0, mesh_cap = 0;
    r3_material* d_materials = nullptr; uint32_t n_materials = 0, materials_cap = 0;
    bool has_skybox = false; r3_texture_desc sky_desc{}; uint8_t* d_sky_texels = nullptr; uint64_t sky_cap = 0;   // cube map of the skybox routine
    r3_texture_desc* d_tex_descs = nullptr; uint32_t n_textures = 0, tex_descs_cap = 0; uint8_t* d_texels = nullptr; uint64_t texels_cap = 0;
    std::vector<r3_texture_desc> tex_descs_host; uint64_t texel_bytes = 0;   // host copy of the table (r3_generate_mipmaps plans from it)
    r3_mip_job* d_mip_jobs = nullptr; uint64_t mip_jobs_cap = 0; std::vector<uint8_t> mip_plan_host;   // work list of the last r3_generate_mipmaps
    // pinned staging of work lists uploaded inside a recorded frame (the captured copy reads it when the graph runs): appended to, and
    // rewound once the stream has drained (r3_stream_sync); a full arena is replaced by one twice as large and kept until the context goes
    uint8_t* mip_staging = nullptr; uint64_t mip_staging_cap = 0, mip_staging_used = 0; std::vector<void*> mip_staging_retired;
    bool mip_tail_smem_set = false;           // mip_tail_kernel's dynamic shared-memory limit raised
    r3_directional_light* d_dir = nullptr; uint32_t n_dir = 0, dir_cap = 0;
    r3_point_light* d_point = nullptr; uint32_t n_point = 0, point_cap = 0;
    float* d_light_mats = nullptr; uint64_t light_mats_cap = 0;   // view-space light tables built by light_prep_kernel
    r3_frame_uniforms uniforms{}; bool uniforms_set = false;
    float* d_atlas = nullptr; uint32_t atlas_w = 0, atlas_h = 0;
    r3_camera cams[R3_MAX_CAMERAS];
    // render targets
    uint32_t width = 0, height = 0, samples = 1; float clear_color[4] = {0, 0, 0, 0};
    uint32_t row_begin = 0, row_end = 0;
    unsigned long long* d_vis = nullptr;      // (depth bits << 32) | (pass << 31) | record
    bool parity_target = false;               // also keep the f32 shading result before the rgba16f store (tests; off in production)
    float* d_hdr32 = nullptr; uint16_t* d_hdr16 = nullptr; float* d_depth = nullptr; uint8_t* d_ldr = nullptr;
    std::vector<float*> d_hiz; std::vector<uint32_t> hiz_w, hiz_h;
    float** d_hiz_ptrs = nullptr; uint32_t* d_hiz_dims = nullptr;
    r3_tri_record* d_tris[4] = {nullptr, nullptr, nullptr, nullptr}; uint64_t tris_cap[4] = {0, 0, 0, 0}; uint64_t n_tris[4] = {0, 0, 0, 0};   // predicted, residual, blend, shadow scratch
    bool any_frag_alpha = false;              // a material discards per fragment (cutout alpha from its albedo texture / vertex colour)
    unsigned long long* d_stats = nullptr;    // [8]: [0..3] forward statistics, [4] scratch of r3_compute_max_invocations
    // blend routine: per-sample fragment lists (head = node index + 1, 0 = empty; node = {record, depth bits, next, 0})
    bool any_blend = false;                   // some live object carries material key 2 (TransparencyType::Blend)
    uint32_t* d_frag_heads = nullptr; uint64_t frag_heads_cap = 0;
    uint4* d_frag_nodes = nullptr; uint64_t frag_nodes_cap = 0;
    void* d_scratch = nullptr; uint64_t scratch_cap = 0;
    r3_stage_timer timer;
    r3_peer_state peer;
    uint32_t tri_shard_index = 0, tri_shard_count = 1;   // r3_set_cull_shard
    // frame graph
    bool capturing = false;                   // between r3_frame_begin and the submission (or an early flush)
    cudaGraphExec_t frame_exec[2] = {nullptr, nullptr};   // instantiated graphs of even / odd frames (the culling buffers ping-pong), updated in place
    uint64_t frame_index = 0, frames_graphed = 0, frames_flushed = 0, graph_reinstantiations = 0;
};

// ---- error plumbing (nothing throws across the C boundary)
int r3_fail(r3_ctx* c, int code, const char* msg);
int r3_cuda_fail(r3_ctx* c, cudaError_t e, const char* where);
#define R3_CUDA(c, call)                                                  \
    do {                                                                  \
        cudaError_t e__ = (call);                                         \
        if (e__ != cudaSuccess) return r3_cuda_fail((c), e__, #call);     \
    } while (0)
#define R3_CHECK_LAUNCH(c, name)                                          \
    do {                                                                  \
        (c)->launches++;                                                  \
        cudaError_t e__ = cudaGetLastError();                             \
        if (e__ != cudaSuccess) return r3_cuda_fail((c), e__, name);      \
    } while (0)
#define R3_TRY(expr)                                                      \
    do {                                                                  \
        int rc__ = (expr);                                                \
        if (rc__ != R3_OK) return rc__;                                   \
    } while (0)

// Frame graph (r3_frame_begin / r3_frame_end): the stream work of one frame is recorded by stream capture and submitted as ONE CUDA graph
// launch (the reference submits once per frame, graph.rs:510).  Anything that has to wait for the stream inside a frame first flushes what
// was recorded so far (r3_stream_sync does that), after which the rest of the frame runs eagerly.
cudaError_t r3_stream_sync(r3_ctx* c);
// stage timing: no-ops unless enabled
void r3_stage_begin(r3_ctx* c, int stage);
void r3_stage_end(r3_ctx* c);
static inline int r3_cam_slot(uint32_t camera) { return camera == R3_CAMERA_VIEWPORT ? 0 : (int)camera + 1; }
static inline r3_camera* r3_get_camera(r3_ctx* c, uint32_t camera) {
    if (!c || (camera != R3_CAMERA_VIEWPORT && camera >= R3_MAX_SHADOWS)) return nullptr;
    return &c->cams[r3_cam_slot(camera)];
}
#define R3_CAM_OR_FAIL(ctx, camera)                                                                              \
    if (!(ctx)) return R3_E_INVALID;                                                                             \
    if ((camera) != R3_CAMERA_VIEWPORT && (camera) >= R3_MAX_SHADOWS) return r3_fail((ctx), R3_E_INVALID, "bad camera"); \
    r3_camera* cam = &(ctx)->cams[r3_cam_slot(camera)]

// grow-only device allocation helper: keeps contents when `keep` is set
int r3_reserve(r3_ctx* c, void** ptr, uint64_t* cap_elems, uint64_t need_elems, size_t elem_size, bool keep, bool zero_new);
template <typename T, typename C>
int r3_reserve_t(r3_ctx* c, T** ptr, C* cap, uint64_t need, bool keep = false, bool zero_new = false) {
    uint64_t cap64 = *cap;
    int rc = r3_reserve(c, (void**)ptr, &cap64, need, sizeof(T), keep, zero_new);
    *cap = (C)cap64;
    return rc;
}

// stages implemented in the other translation units
int r3_launch_cull_bake(r3_ctx* c, r3_camera* cam, uint32_t mode);
int r3_split_objects(r3_ctx* c);
int r3_split_slots(r3_ctx* c, const uint32_t* d_slots, uint32_t n);
int r3_launch_triangle_cull(r3_ctx* c, r3_camera* cam);
int r3_host_batch_objects(r3_ctx* c, r3_camera* cam, const float vp_loc[3], uint32_t max_dispatch_count);
int r3_upload_jobs(r3_ctx* c, r3_camera* cam);
int r3_device_batch_objects(r3_ctx* c, r3_camera* cam, const float vp_loc[3], uint32_t max_dispatch_count);
int r3_download_jobs(r3_ctx* c, r3_camera* cam);          // device-built jobs -> host vectors (readbacks / tests)
int r3_compute_max_invocations(r3_ctx* c);
void r3_new_frame_epoch(r3_ctx* c);          // the frame-wide sort of the previous frame is stale from here on
int r3_blend_collect(r3_ctx* c, bool* ran);   // r3_raster.cu: per-sample fragment lists of the blend routine
int r3_launch_mipmaps(r3_ctx* c, const uint32_t* indices, uint32_t count);   // r3_mipmap.cu: rule R12 over validated table indices
int r3_iobuf_new(r3_ctx* c, r3_iobuf* b, uint64_t elems, uint64_t elem_size, bool clear_on_swap);
int r3_iobuf_swap(r3_ctx* c, r3_iobuf* b, uint64_t new_elems);

#ifdef __CUDACC__
// IEEE, never-contracted arithmetic for the bit-exact stages (SURVEY D7)
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
// M * (x, y, z, w): column-major, accumulated x,y,z,w like WGSL's mat4x4*vec4
__device__ __forceinline__ float4 mat_vec_rn(const float* __restrict__ m, float x, float y, float z, float w) {
    float4 r;
    r.x = mul_rn(m[0], x); r.y = mul_rn(m[1], x); r.z = mul_rn(m[2], x); r.w = mul_rn(m[3], x);
    r.x = add_rn(r.x, mul_rn(m[4], y)); r.y = add_rn(r.y, mul_rn(m[5], y)); r.z = add_rn(r.z, mul_rn(m[6], y)); r.w = add_rn(r.w, mul_rn(m[7], y));
    r.x = add_rn(r.x, mul_rn(m[8], z)); r.y = add_rn(r.y, mul_rn(m[9], z)); r.z = add_rn(r.z, mul_rn(m[10], z)); r.w = add_rn(r.w, mul_rn(m[11], z));
    r.x = add_rn(r.x, mul_rn(m[12], w)); r.y = add_rn(r.y, mul_rn(m[13], w)); r.z = add_rn(r.z, mul_rn(m[14], w)); r.w = add_rn(r.w, mul_rn(m[15], w));
    return r;
}
// M * (x, y, z, 1)
__device__ __forceinline__ float4 mat_point_rn(const float* __restrict__ m, float x, float y, float z) {
    float4 r;
    r.x = mul_rn(m[0], x); r.y = mul_rn(m[1], x); r.z = mul_rn(m[2], x); r.w = mul_rn(m[3], x);
    r.x = add_rn(r.x, mul_rn(m[4], y)); r.y = add_rn(r.y, mul_rn(m[5], y)); r.z = add_rn(r.z, mul_rn(m[6], y)); r.w = add_rn(r.w, mul_rn(m[7], y));
    r.x = add_rn(r.x, mul_rn(m[8], z)); r.y = add_rn(r.y, mul_rn(m[9], z)); r.z = add_rn(r.z, mul_rn(m[10], z)); r.w = add_rn(r.w, mul_rn(m[11], z));
    r.x = add_rn(r.x, m[12]); r.y = add_rn(r.y, m[13]); r.z = add_rn(r.z, m[14]); r.w = add_rn(r.w, m[15]);
    return r;
}
#endif
