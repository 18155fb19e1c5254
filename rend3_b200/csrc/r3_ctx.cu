// r3_ctx.cu — context, uploads, readbacks and the C ABI glue of librend3_b200.so (include/rend3_b200.h).
// Host logic only; the kernels live in r3_cull_bake.cu, r3_tri_cull.cu, r3_raster.cu, r3_shade.cu.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "r3_common.cuh"

int r3_fail(r3_ctx* c, int code, const char* msg) {
    if (c) c->err = msg;
    return code;
}
int r3_cuda_fail(r3_ctx* c, cudaError_t e, const char* where) {
    if (c) {
        c->err = std::string(where) + ": " + cudaGetErrorString(e);
    }
    cudaGetLastError();   // clear the sticky-less error so later calls report their own
    return e == cudaErrorMemoryAllocation ? R3_E_OOM : R3_E_CUDA;
}

int r3_reserve(r3_ctx* c, void** ptr, uint64_t* cap, uint64_t need, size_t elem, bool keep, bool zero_new) {
    if (*ptr && *cap >= need) return R3_OK;
    uint64_t ncap = need < 16 ? 16 : need;
    void* n = nullptr;
    R3_CUDA(c, cudaMalloc(&n, ncap * elem));
    if (zero_new) R3_CUDA(c, cudaMemsetAsync(n, 0, ncap * elem, c->stream));
    if (*ptr) {
        if (keep && *cap) R3_CUDA(c, cudaMemcpyAsync(n, *ptr, *cap * elem, cudaMemcpyDeviceToDevice, c->stream));
        R3_CUDA(c, r3_stream_sync(c));
        cudaFree(*ptr);
    }
    *ptr = n;
    *cap = ncap;
    return R3_OK;
}

// ------------------------------------------------------------------ context
R3_EXPORT uint32_t r3_abi_version(void) { return R3_ABI_VERSION; }

R3_EXPORT int r3_ctx_create(int device, r3_ctx** out) {
    if (!out) return R3_E_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return R3_E_NO_DEVICE;   // there is no CPU fallback: the caller must fail (RendererInitializationError::MissingAdapter)
    }
    r3_ctx* c = new (std::nothrow) r3_ctx();
    if (!c) return R3_E_OOM;
    c->device = device;
    // the context's stream gets the greatest priority: the exchange consumer's side stream (least priority) then only fills the SMs it leaves idle
    int prio_least = 0, prio_greatest = 0;
    if (cudaSetDevice(device) == cudaSuccess) cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) {
        delete c;
        cudaGetLastError();
        return R3_E_CUDA;
    }
    { int coop = 0; cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device); c->coop_launch_ok = coop != 0 && !getenv("R3_NO_COOP_SORT"); }
    if (cudaMalloc((void**)&c->d_stats, 8 * sizeof(unsigned long long)) != cudaSuccess) { delete c; return R3_E_OOM; }
    cudaMemsetAsync(c->d_stats, 0, 64, c->stream);
    *out = c;
    return R3_OK;
}

static void free_jobs(r3_jobs& j) { cudaFree(j.d_batches); cudaFree(j.d_regions); cudaFree(j.d_region_first_inv); cudaFree(j.d_header); }

R3_EXPORT int r3_ctx_destroy(r3_ctx* c) {
    if (!c) return R3_E_INVALID;
    cudaSetDevice(c->device);
    r3_stream_sync(c);
    if (c->side_stream) cudaStreamSynchronize(c->side_stream);
    r3_peer_destroy(c);
    if (!c->objects_borrowed) cudaFree(c->d_objects);
    cudaFree(c->d_hot_transform); cudaFree(c->d_hot_sphere); cudaFree(c->d_enabled_bits); cudaFree(c->d_tex_descs); cudaFree(c->d_texels); cudaFree(c->d_sky_texels);
    cudaFree(c->d_mip_jobs);
    if (c->mip_staging) cudaFreeHost(c->mip_staging);
    for (void* p : c->mip_staging_retired) cudaFreeHost(p);
    cudaFree(c->d_sort_key8); cudaFree(c->d_sort_loc); cudaFree(c->d_gsort_keys[0]); cudaFree(c->d_gsort_keys[1]); cudaFree(c->d_gsort_hist); cudaFree(c->d_gsort_header);
    cudaFree(c->d_live_bits); cudaFree(c->d_mesh); cudaFree(c->d_materials); cudaFree(c->d_dir); cudaFree(c->d_point);
    cudaFree(c->d_light_mats); cudaFree(c->d_atlas);
    for (auto& k : c->cams) {
        cudaFree(k.d_matrices); cudaFree(k.d_visible); cudaFree(k.d_visible_count); cudaFree(k.d_tile_state);
        if (k.d_gathered) {   // visible-set exchange: unmap the peers' buffers, free ours
            for (uint32_t r = 0; r < k.ex_ranks; ++r)
                if (k.ex_connected && r != k.ex_rank && k.ex_peers[r]) cudaIpcCloseMemHandle(k.ex_peers[r]);
            cudaFree(k.d_gathered);
        }
        cudaFree(k.d_ex_done); cudaFree(k.d_global_visible); cudaFree(k.d_merge_counts);
        for (int q = 0; q < R3_EXCHANGE_SLOTS; ++q) { if (k.ex_cull_done[q]) cudaEventDestroy(k.ex_cull_done[q]); if (k.ex_merge_done[q]) cudaEventDestroy(k.ex_merge_done[q]); }
        free_jobs(k.jobs[0]); free_jobs(k.jobs[1]);
        cudaFree(k.index_buffer.d); cudaFree(k.draw_call_buffer.d); cudaFree(k.results_buffer.d);
        cudaFree(k.d_resid_bits); cudaFree(k.d_word_scan); cudaFree(k.d_block_sums);
        cudaFree(k.d_prev_inv[0]); cudaFree(k.d_prev_inv[1]); cudaFree(k.d_sort_keys[0]); cudaFree(k.d_sort_keys[1]); cudaFree(k.d_sort_hist); cudaFree(k.d_batch_tmp);
    }
    cudaFree(c->d_vis); cudaFree(c->d_hdr32); cudaFree(c->d_hdr16); cudaFree(c->d_depth); cudaFree(c->d_ldr);
    for (float* p : c->d_hiz) cudaFree(p);
    cudaFree(c->d_hiz_ptrs); cudaFree(c->d_hiz_dims);
    cudaFree(c->d_tris[0]); cudaFree(c->d_tris[1]); cudaFree(c->d_tris[2]); cudaFree(c->d_tris[3]); cudaFree(c->d_stats); cudaFree(c->d_scratch);
    cudaFree(c->d_frag_heads); cudaFree(c->d_frag_nodes);
    for (cudaEvent_t e : c->timer.pool) cudaEventDestroy(e);
    for (auto& x : c->frame_exec) if (x) cudaGraphExecDestroy(x);
    if (c->side_stream) cudaStreamDestroy(c->side_stream);
    cudaStreamDestroy(c->stream);
    delete c;
    return R3_OK;
}
R3_EXPORT const char* r3_last_error(const r3_ctx* c) { return c ? c->err.c_str() : "null context"; }
R3_EXPORT int r3_sync(r3_ctx* c) {
    if (!c) return R3_E_INVALID;
    cudaSetDevice(c->device);
    R3_CUDA(c, r3_stream_sync(c));
    if (c->side_stream) R3_CUDA(c, cudaStreamSynchronize(c->side_stream));   // exchange consumers in flight
    return R3_OK;
}
R3_EXPORT int r3_get_stream(r3_ctx* c, void** s) {
    if (!c || !s) return R3_E_INVALID;
    *s = (void*)c->stream;
    return R3_OK;
}
R3_EXPORT int r3_launch_count(r3_ctx* c, uint64_t* n) {
    if (!c || !n) return R3_E_INVALID;
    *n = c->launches;
    return R3_OK;
}

// ------------------------------------------------------------------ frame graph
// End the capture (if one is running) and submit what it recorded.  `slot` >= 0: keep the instantiated graph of that frame parity and
// update it in place next time (cudaGraphExecUpdate: same topology, new kernel arguments / pointers); slot < 0: one-off (an early flush).
static cudaError_t r3_submit_capture(r3_ctx* c, int slot) {
    if (!c->capturing) return cudaSuccess;
    c->capturing = false;
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(c->stream, &g);
    if (e != cudaSuccess || !g) return e != cudaSuccess ? e : cudaErrorUnknown;
    if (slot < 0) {
        cudaGraphExec_t x = nullptr;
        e = cudaGraphInstantiate(&x, g, 0);
        if (e == cudaSuccess) e = cudaGraphLaunch(x, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);   // the one-off exec is destroyed right away: wait for it
        if (x) cudaGraphExecDestroy(x);
        cudaGraphDestroy(g);
        return e;
    }
    cudaGraphExec_t& x = c->frame_exec[slot];
    if (x) {
        cudaGraphExecUpdateResultInfo info;
        if (cudaGraphExecUpdate(x, g, &info) != cudaSuccess) {   // another topology (new buffers sizes, another routine set): instantiate again
            cudaGetLastError();
            cudaGraphExecDestroy(x);
            x = nullptr;
        }
    }
    if (!x) {
        e = cudaGraphInstantiate(&x, g, 0);
        c->graph_reinstantiations++;
    }
    if (e == cudaSuccess) e = cudaGraphLaunch(x, c->stream);
    cudaGraphDestroy(g);
    return e;
}
cudaError_t r3_stream_sync(r3_ctx* c) {
    if (c->capturing) {
        // a stage needs the stream to drain in the middle of a recorded frame (a buffer grows, a host path reads back): submit what
        // was recorded, wait, and let the rest of the frame run eagerly
        const cudaError_t e = r3_submit_capture(c, -1);
        c->frames_flushed++;
        if (e != cudaSuccess) { c->mip_plan_host.clear(); return e; }   // the recorded work-list copy never ran
    }
    const cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) c->mip_staging_used = 0;   // every recorded copy out of the staging arena has run
    return e;
}
R3_EXPORT int r3_frame_begin(r3_ctx* c) {
    if (!c) return R3_E_INVALID;
    cudaSetDevice(c->device);
    if (c->capturing) return r3_fail(c, R3_E_STATE, "frame_begin: a frame is already being recorded");
    if (c->timer.enabled) return R3_OK;       // per-kernel timing needs real event records: the frame runs eagerly
    R3_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed));
    c->capturing = true;
    return R3_OK;
}
R3_EXPORT int r3_frame_end(r3_ctx* c) {
    if (!c) return R3_E_INVALID;
    cudaSetDevice(c->device);
    const bool was = c->capturing;
    const cudaError_t e = r3_submit_capture(c, (int)(c->frame_index & 1u));
    c->frame_index++;
    if (was) c->frames_graphed++;
    if (e != cudaSuccess) {
        c->mip_plan_host.clear();   // the recorded work-list copy never ran: the next r3_generate_mipmaps uploads its list again
        return r3_cuda_fail(c, e, "frame_end (graph submission)");
    }
    return R3_OK;
}
R3_EXPORT int r3_frame_graph_stats(r3_ctx* c, uint64_t stats[4]) {
    if (!c || !stats) return R3_E_INVALID;
    stats[0] = c->frame_index; stats[1] = c->frames_graphed; stats[2] = c->frames_flushed; stats[3] = c->graph_reinstantiations;
    return R3_OK;
}

// ------------------------------------------------------------------ stage timing
void r3_stage_begin(r3_ctx* c, int stage) {
    r3_stage_timer& t = c->timer;
    if (!t.enabled || c->capturing) return;
    if (t.pool.size() < 2 * (t.used + 1)) {
        cudaEvent_t a = nullptr, b = nullptr;
        if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) { t.enabled = false; return; }
        t.pool.push_back(a); t.pool.push_back(b); t.stage_of.push_back(stage);
    }
    t.stage_of[t.used] = stage;
    cudaEventRecord(t.pool[2 * t.used], c->stream);
}
void r3_stage_end(r3_ctx* c) {
    r3_stage_timer& t = c->timer;
    if (!t.enabled || c->capturing) return;
    cudaEventRecord(t.pool[2 * t.used + 1], c->stream);
    t.used++;
}
R3_EXPORT int r3_set_stage_timing(r3_ctx* c, int enabled) {
    if (!c) return R3_E_INVALID;
    cudaSetDevice(c->device);
    c->timer.enabled = enabled != 0;
    c->timer.used = 0;
    return R3_OK;
}
R3_EXPORT int r3_stage_times_n(r3_ctx* c, uint32_t n_stages, double* ms, uint32_t* launches) {
    if (!c || !ms || !launches || n_stages > R3_STAGE_COUNT) return r3_fail(c, R3_E_INVALID, "stage_times: bad arguments");
    cudaSetDevice(c->device);
    R3_CUDA(c, r3_stream_sync(c));
    for (uint32_t k = 0; k < n_stages; ++k) { ms[k] = 0.0; launches[k] = 0; }
    r3_stage_timer& t = c->timer;
    for (size_t k = 0; k < t.used; ++k) {
        float e = 0.f;
        if (cudaEventElapsedTime(&e, t.pool[2 * k], t.pool[2 * k + 1]) == cudaSuccess && t.stage_of[k] >= 0 && t.stage_of[k] < (int)n_stages) { ms[t.stage_of[k]] += e; launches[t.stage_of[k]]++; }
    }
    t.used = 0;
    return R3_OK;
}
R3_EXPORT int r3_stage_times(r3_ctx* c, double ms[8], uint32_t launches[8]) { return r3_stage_times_n(c, 8, ms, launches); }

// ------------------------------------------------------------------ world data
R3_EXPORT int r3_set_objects(r3_ctx* c, const r3_object* recs, uint32_t n) {
    if (!c || (!recs && n)) return r3_fail(c, R3_E_INVALID, "set_objects: null records");
    cudaSetDevice(c->device);
    if (c->objects_borrowed) { c->d_objects = nullptr; c->objects_cap = 0; c->objects_borrowed = false; }
    R3_TRY(r3_reserve_t(c, &c->d_objects, &c->objects_cap, n));
    if (n) R3_CUDA(c, cudaMemcpyAsync(c->d_objects, recs, (size_t)n * sizeof(r3_object), cudaMemcpyHostToDevice, c->stream));
    c->n_slots = n;
    c->max_invocations_valid = false;
    R3_TRY(r3_split_objects(c));
    R3_CUDA(c, r3_stream_sync(c));   // host pointer is only borrowed for the call
    return R3_OK;
}
R3_EXPORT int r3_set_objects_device(r3_ctx* c, const void* dptr, uint32_t n) {
    if (!c || (!dptr && n)) return r3_fail(c, R3_E_INVALID, "set_objects_device: null pointer");
    if (!c->objects_borrowed) { cudaFree(c->d_objects); }
    c->d_objects = (r3_object*)dptr;
    c->objects_cap = n; c->n_slots = n; c->objects_borrowed = true;
    c->max_invocations_valid = false;
    cudaSetDevice(c->device);
    return r3_split_objects(c);   // snapshot of the hot fields: call again after changing the records
}

__global__ void scatter_objects_kernel(r3_object* dst, const r3_object* src, const uint32_t* slots, uint32_t n, uint32_t n_slots) {
    // ScatterCopy (rend3/shaders/scatter_copy.wgsl): one 16-byte lane per float4 of the 128-byte record
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, k = threadIdx.x & 7;
    if (i >= n) return;
    const uint32_t s = slots[i];
    if (s >= n_slots) return;   // out-of-range writes are dropped (robust buffer access)
    reinterpret_cast<float4*>(dst)[(size_t)s * 8 + k] = reinterpret_cast<const float4*>(src)[(size_t)i * 8 + k];
}
R3_EXPORT int r3_update_objects(r3_ctx* c, const uint32_t* slots, const r3_object* recs, uint32_t n) {
    if (!c || !slots || !recs) return r3_fail(c, R3_E_INVALID, "update_objects: null");
    if (n == 0) return R3_OK;
    cudaSetDevice(c->device);
    const uint64_t bytes = (uint64_t)n * (sizeof(r3_object) + 4);
    R3_TRY(r3_reserve(c, &c->d_scratch, &c->scratch_cap, bytes, 1, false, false));
    r3_object* d_recs = (r3_object*)c->d_scratch;
    uint32_t* d_slots = (uint32_t*)((uint8_t*)c->d_scratch + (size_t)n * sizeof(r3_object));
    R3_CUDA(c, cudaMemcpyAsync(d_recs, recs, (size_t)n * sizeof(r3_object), cudaMemcpyHostToDevice, c->stream));
    R3_CUDA(c, cudaMemcpyAsync(d_slots, slots, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
    scatter_objects_kernel<<<(n * 8 + 255) / 256, 256, 0, c->stream>>>(c->d_objects, d_recs, d_slots, n, c->n_slots);
    R3_CHECK_LAUNCH(c, "scatter_objects_kernel");
    R3_TRY(r3_split_slots(c, d_slots, n));
    c->max_invocations_valid = false;
    R3_CUDA(c, r3_stream_sync(c));
    return R3_OK;
}
R3_EXPORT int r3_set_object_sort_info(r3_ctx* c, const uint64_t* key, const uint8_t* flags, const float* loc, uint32_t n) {
    if (!c || !key || !flags || !loc) return r3_fail(c, R3_E_INVALID, "set_object_sort_info: null");
    cudaSetDevice(c->device);
    c->sort_key.assign(key, key + n);
    c->sort_flags.assign(flags, flags + n);
    c->sort_loc.assign(loc, loc + 3 * (size_t)n);
    const uint32_t words = (n + 31) / 32;
    std::vector<uint32_t> bits(words ? words : 1, 0u);
    for (uint32_t i = 0; i < n; ++i)
        if (flags[i] & 1) bits[i >> 5] |= 1u << (i & 31);
    R3_TRY(r3_reserve_t(c, &c->d_live_bits, &c->live_bits_cap, words));
    R3_CUDA(c, cudaMemcpyAsync(c->d_live_bits, bits.data(), (size_t)words * 4, cudaMemcpyHostToDevice, c->stream));
    // device copies for the on-device batch_objects: key8 = ((material_key << 1 | reason) << 1) | back_to_front
    bool ok = true;
    std::vector<uint8_t> key8(n ? n : 1, 0);
    c->any_blend = false;
    for (uint32_t i = 0; i < n; ++i) {
        if (key[i] >= 64) ok = false;
        if (key[i] == 2 && (flags[i] & 1)) c->any_blend = true;   // TransparencyType::Blend as u64 (pbr/material.rs:497-503)
        const uint32_t reason = (flags[i] & 2) ? 0u : 1u;
        key8[i] = (uint8_t)(((((uint32_t)key[i] & 63u) << 1 | reason) << 1) | ((flags[i] & 4) ? 1u : 0u));
    }
    uint32_t cap2 = c->sort_dev_cap;
    R3_TRY(r3_reserve_t(c, &c->d_sort_key8, &c->sort_dev_cap, n));
    if (!c->d_sort_loc || cap2 != c->sort_dev_cap) {
        cudaFree(c->d_sort_loc);
        c->d_sort_loc = nullptr;
        R3_CUDA(c, cudaMalloc((void**)&c->d_sort_loc, ((size_t)c->sort_dev_cap * 3 + 4) * 4));
    }
    if (n) {
        R3_CUDA(c, cudaMemcpyAsync(c->d_sort_key8, key8.data(), n, cudaMemcpyHostToDevice, c->stream));
        R3_CUDA(c, cudaMemcpyAsync(c->d_sort_loc, loc, (size_t)n * 12, cudaMemcpyHostToDevice, c->stream));
    }
    R3_CUDA(c, r3_stream_sync(c));
    r3_new_frame_epoch(c);
    c->have_live = true;
    c->gpu_batching_ok = ok && n < (1u << 24) && !getenv("R3_HOST_BATCHING");
    return R3_OK;
}
R3_EXPORT int r3_set_mesh_buffer(r3_ctx* c, const void* bytes, uint64_t nbytes) {
    if (!c || (!bytes && nbytes) || (nbytes & 3)) return r3_fail(c, R3_E_INVALID, "set_mesh_buffer: bad size");
    cudaSetDevice(c->device);
    R3_TRY(r3_reserve_t(c, &c->d_mesh, &c->mesh_cap, nbytes / 4 + 4));
    if (nbytes) R3_CUDA(c, cudaMemcpyAsync(c->d_mesh, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    R3_CUDA(c, r3_stream_sync(c));
    c->mesh_words = nbytes / 4;
    return R3_OK;
}
R3_EXPORT int r3_set_materials(r3_ctx* c, const r3_material* recs, uint32_t n) {
    if (!c || (!recs && n)) return r3_fail(c, R3_E_INVALID, "set_materials: null");
    cudaSetDevice(c->device);
    R3_TRY(r3_reserve_t(c, &c->d_materials, &c->materials_cap, n));
    if (n) R3_CUDA(c, cudaMemcpyAsync(c->d_materials, recs, (size_t)n * sizeof(r3_material), cudaMemcpyHostToDevice, c->stream));
    R3_CUDA(c, r3_stream_sync(c));
    c->n_materials = n;
    c->any_frag_alpha = false;
    for (uint32_t i = 0; i < n; ++i)
        if ((recs[i].flags & R3_MAT_ALBEDO_ACTIVE) && recs[i].alpha_cutout > 0.0f && (recs[i].textures[R3_TEX_ALBEDO] || (recs[i].flags & R3_MAT_ALBEDO_BLEND))) c->any_frag_alpha = true;
    return R3_OK;
}
R3_EXPORT int r3_set_textures(r3_ctx* c, const r3_texture_desc* descs, uint32_t n, const void* texels, uint64_t nbytes) {
    if (!c || (!descs && n) || (!texels && nbytes)) return r3_fail(c, R3_E_INVALID, "set_textures: null");
    for (uint32_t i = 0; i < n; ++i) {   // validated once here so the samplers index without checks
        const r3_texture_desc& d = descs[i];
        if (!d.width || !d.height || !d.mip_count || d.mip_count > 32 || d.format >= R3_TEXFMT_COUNT) return r3_fail(c, R3_E_INVALID, "set_textures: bad descriptor");
        uint64_t total = 0;
        for (uint32_t l = 0; l < d.mip_count; ++l) total += R3_TEXFMT_LEVEL_BYTES(d.format, (d.width >> l) ? (d.width >> l) : 1u, (d.height >> l) ? (d.height >> l) : 1u);
        if (d.byte_offset % 16 || d.byte_offset + total > nbytes) return r3_fail(c, R3_E_INVALID, "set_textures: mip chain outside the texel blob");
    }
    cudaSetDevice(c->device);
    R3_TRY(r3_reserve_t(c, &c->d_tex_descs, &c->tex_descs_cap, n));
    R3_TRY(r3_reserve_t(c, &c->d_texels, &c->texels_cap, nbytes + 16));
    if (n) R3_CUDA(c, cudaMemcpyAsync(c->d_tex_descs, descs, (size_t)n * sizeof(r3_texture_desc), cudaMemcpyHostToDevice, c->stream));
    if (nbytes) R3_CUDA(c, cudaMemcpyAsync(c->d_texels, texels, nbytes, cudaMemcpyHostToDevice, c->stream));
    R3_CUDA(c, r3_stream_sync(c));
    c->n_textures = n;
    c->tex_descs_host.assign(descs, descs + n);
    c->texel_bytes = nbytes;
    return R3_OK;
}
// the formats wgpu guarantees FILTERABLE and RENDER_ATTACHMENT: what rend3-gltf asks MipmapSource::Generated for (rend3-gltf/src/lib.rs:1082-1087)
static bool mip_format_ok(uint32_t f) {
    return f == R3_TEXFMT_RGBA8_UNORM || f == R3_TEXFMT_RGBA8_UNORM_SRGB || f == R3_TEXFMT_BGRA8_UNORM || f == R3_TEXFMT_BGRA8_UNORM_SRGB || f == R3_TEXFMT_R8_UNORM ||
           f == R3_TEXFMT_RG8_UNORM || f == R3_TEXFMT_RGB10A2_UNORM || f == R3_TEXFMT_R16_FLOAT || f == R3_TEXFMT_RG16_FLOAT || f == R3_TEXFMT_RGBA16_FLOAT;
}
R3_EXPORT int r3_generate_mipmaps(r3_ctx* c, const uint32_t* indices, uint32_t count) {
    if (!c || (!indices && count)) return r3_fail(c, R3_E_INVALID, "generate_mipmaps: null");
    // the whole list is checked before anything is launched: a rejected call changes no byte
    std::vector<std::pair<uint64_t, uint64_t>> chains;
    std::vector<uint8_t> seen(c->n_textures, 0);
    for (uint32_t n = 0; n < count; ++n) {
        const uint32_t i = indices[n];
        if (i >= c->n_textures) return r3_fail(c, R3_E_INVALID, "generate_mipmaps: index outside the texture table");
        if (seen[i]) return r3_fail(c, R3_E_INVALID, "generate_mipmaps: index listed twice");
        seen[i] = 1;
        const r3_texture_desc& d = c->tex_descs_host[i];
        if (!mip_format_ok(d.format)) return r3_fail(c, R3_E_INVALID, "generate_mipmaps: format is not filterable and renderable");
        uint32_t max_mips = 0;
        for (uint32_t m = d.width > d.height ? d.width : d.height; m; m >>= 1) ++max_mips;   // floor(log2(max(w, h))) + 1
        if (d.mip_count > max_mips) return r3_fail(c, R3_E_INVALID, "generate_mipmaps: mip_count exceeds floor(log2(max(w, h))) + 1");
        uint64_t total = 0;
        for (uint32_t l = 0; l < d.mip_count; ++l) total += R3_TEXFMT_LEVEL_BYTES(d.format, (d.width >> l) ? (d.width >> l) : 1u, (d.height >> l) ? (d.height >> l) : 1u);
        chains.emplace_back(d.byte_offset, d.byte_offset + total);
    }
    std::sort(chains.begin(), chains.end());
    for (size_t k = 1; k < chains.size(); ++k)
        if (chains[k].first < chains[k - 1].second) return r3_fail(c, R3_E_INVALID, "generate_mipmaps: two listed mip chains overlap");
    cudaSetDevice(c->device);
    return r3_launch_mipmaps(c, indices, count);
}
R3_EXPORT int r3_readback_texels(r3_ctx* c, uint64_t byte_offset, void* dst, uint64_t nbytes) {
    if (!c || (!dst && nbytes)) return r3_fail(c, R3_E_INVALID, "readback_texels: null");
    if (byte_offset > c->texel_bytes || nbytes > c->texel_bytes - byte_offset) return r3_fail(c, R3_E_INVALID, "readback_texels: range outside the texel blob");
    cudaSetDevice(c->device);
    if (nbytes) R3_CUDA(c, cudaMemcpyAsync(dst, c->d_texels + byte_offset, nbytes, cudaMemcpyDeviceToHost, c->stream));
    R3_CUDA(c, r3_stream_sync(c));
    return R3_OK;
}
R3_EXPORT int r3_set_skybox(r3_ctx* c, const r3_texture_desc* desc, const void* texels, uint64_t nbytes) {
    if (!c) return R3_E_INVALID;
    c->has_skybox = false;
    if (!desc) return R3_OK;
    if (!texels || !desc->width || !desc->mip_count || desc->mip_count > 32 || desc->format > R3_TEXFMT_RGBA32_FLOAT) return r3_fail(c, R3_E_INVALID, "set_skybox: bad descriptor");
    const uint64_t bpp = desc->format == R3_TEXFMT_RGBA32_FLOAT ? 16 : 4;
    uint64_t face = 0;
    for (uint32_t l = 0; l < desc->mip_count; ++l) { const uint64_t w = (desc->width >> l) ? (desc->width >> l) : 1u; face += w * w * bpp; }
    if (desc->byte_offset % 16 || desc->byte_offset + 6 * face > nbytes) return r3_fail(c, R3_E_INVALID, "set_skybox: faces outside the texel blob");
    cudaSetDevice(c->device);
    R3_TRY(r3_reserve_t(c, &c->d_sky_texels, &c->sky_cap, nbytes + 16));
    R3_CUDA(c, cudaMemcpyAsync(c->d_sky_texels, texels, nbytes, cudaMemcpyHostToDevice, c->stream));
    R3_CUDA(c, r3_stream_sync(c));
    c->sky_desc = *desc; c->sky_desc.height = desc->width; c->has_skybox = true;
    return R3_OK;
}
R3_EXPORT int r3_set_directional_lights(r3_ctx* c, const void* bytes, uint64_t nbytes, uint32_t aw, uint32_t ah) {
    if (!c || !bytes || nbytes < 16) return r3_fail(c, R3_E_INVALID, "set_directional_lights: short buffer");
    cudaSetDevice(c->device);
    const uint32_t n = *(const uint32_t*)bytes;
    if (nbytes < 16 + (uint64_t)n * sizeof(r3_directional_light)) return r3_fail(c, R3_E_INVALID, "set_directional_lights: short buffer");
    R3_TRY(r3_reserve_t(c, &c->d_dir, &c->dir_cap, n));
    if (n) R3_CUDA(c, cudaMemcpyAsync(c->d_dir, (const uint8_t*)bytes + 16, (size_t)n * sizeof(r3_directional_light), cudaMemcpyHostToDevice, c->stream));
    c->n_dir = n;
    if (aw != c->atlas_w || ah != c->atlas_h || !c->d_atlas) {
        R3_CUDA(c, r3_stream_sync(c));
        cudaFree(c->d_atlas);
        c->d_atlas = nullptr;
        R3_CUDA(c, cudaMalloc((void**)&c->d_atlas, (size_t)aw * ah * 4 + 16));
        R3_CUDA(c, cudaMemsetAsync(c->d_atlas, 0, (size_t)aw * ah * 4, c->stream));
        c->atlas_w = aw; c->atlas_h = ah;
    }
    R3_CUDA(c, r3_stream_sync(c));
    return R3_OK;
}
R3_EXPORT int r3_set_point_lights(r3_ctx* c, const void* bytes, uint64_t nbytes) {
    if (!c || !bytes || nbytes < 16) return r3_fail(c, R3_E_INVALID, "set_point_lights: short buffer");
    cudaSetDevice(c->device);
    const uint32_t n = *(const uint32_t*)bytes;
    if (nbytes < 16 + (uint64_t)n * sizeof(r3_point_light)) return r3_fail(c, R3_E_INVALID, "set_point_lights: short buffer");
    R3_TRY(r3_reserve_t(c, &c->d_point, &c->point_cap, n));
    if (n) R3_CUDA(c, cudaMemcpyAsync(c->d_point, (const uint8_t*)bytes + 16, (size_t)n * sizeof(r3_point_light), cudaMemcpyHostToDevice, c->stream));
    R3_CUDA(c, r3_stream_sync(c));
    c->n_point = n;
    return R3_OK;
}
void r3_new_frame_epoch(r3_ctx* c) {
    c->gsort_epoch++;
    c->gsort_valid = false;
    if (c->gsort_cameras_this_epoch) c->gsort_cameras_last_epoch = c->gsort_cameras_this_epoch;
    c->gsort_cameras_this_epoch = 0;
}
R3_EXPORT int r3_set_frame_uniforms(r3_ctx* c, const r3_frame_uniforms* u) {
    if (!c || !u) return r3_fail(c, R3_E_INVALID, "set_frame_uniforms: null");
    r3_new_frame_epoch(c);   // base.rs:142: once per frame, before any camera batches
    c->uniforms = *u;
    c->uniforms_set = true;
    return R3_OK;
}

// ------------------------------------------------------------------ cull + bake
R3_EXPORT int r3_object_uniform_upload(r3_ctx* c, uint32_t camera, const r3_camera_header* h, uint32_t mode) {
    R3_CAM_OR_FAIL(c, camera);
    if (!h) return r3_fail(c, R3_E_INVALID, "object_uniform_upload: null header");
    cudaSetDevice(c->device);
    if (h->object_count > c->n_slots) return r3_fail(c, R3_E_INVALID, "object_count exceeds the object buffer");
    cam->header = *h;
    cam->header_set = true;
    const uint32_t n = h->object_count;
    if (mode & R3_CB_BAKE) {
        // a resized per-camera buffer starts zeroed (culler.rs:459-476: new buffer when the size changes)
        if (cam->matrices_cap < n || !cam->d_matrices) {
            R3_CUDA(c, r3_stream_sync(c));
            cudaFree(cam->d_matrices);
            cam->d_matrices = nullptr;
            R3_CUDA(c, cudaMalloc((void**)&cam->d_matrices, ((size_t)n + 1) * sizeof(r3_object_matrices)));
            R3_CUDA(c, cudaMemsetAsync(cam->d_matrices, 0, ((size_t)n + 1) * sizeof(r3_object_matrices), c->stream));
            cam->matrices_cap = n;
        }
    }
    if (!cam->d_visible_count) {
        R3_CUDA(c, cudaMalloc((void**)&cam->d_visible_count, 16));
        R3_CUDA(c, cudaMemsetAsync(cam->d_visible_count, 0, 16, c->stream));
    }
    if (mode & R3_CB_CULL) R3_TRY(r3_reserve_t(c, &cam->d_visible, &cam->visible_cap, (uint64_t)n + 1));
    cam->visible_count_host = -1;
    return r3_launch_cull_bake(c, cam, mode);
}
R3_EXPORT int r3_visible_count(r3_ctx* c, uint32_t camera, uint32_t* count) {
    R3_CAM_OR_FAIL(c, camera);
    if (!count) return r3_fail(c, R3_E_INVALID, "null");
    cudaSetDevice(c->device);
    if (!cam->d_visible_count) { *count = 0; return R3_OK; }
    if (cam->visible_count_host < 0) {
        uint32_t v = 0;
        R3_CUDA(c, cudaMemcpyAsync(&v, cam->d_visible_count, 4, cudaMemcpyDeviceToHost, c->stream));
        R3_CUDA(c, r3_stream_sync(c));
        cam->visible_count_host = (int)v;
    }
    *count = (uint32_t)cam->visible_count_host;
    return R3_OK;
}
R3_EXPORT int r3_readback_visible(r3_ctx* c, uint32_t camera, uint32_t* out, uint32_t cap, uint32_t* count) {
    uint32_t n = 0;
    R3_TRY(r3_visible_count(c, camera, &n));
    r3_camera* cam = &c->cams[r3_cam_slot(camera)];
    if (count) *count = n;
    if (out && n) {
        if (cap < n) return r3_fail(c, R3_E_INVALID, "readback_visible: capacity too small");
        R3_CUDA(c, cudaMemcpyAsync(out, cam->d_visible, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
        R3_CUDA(c, r3_stream_sync(c));
    }
    return R3_OK;
}
R3_EXPORT int r3_readback_object_matrices(r3_ctx* c, uint32_t camera, r3_object_matrices* out, uint32_t first, uint32_t n) {
    R3_CAM_OR_FAIL(c, camera);
    if (!out || (uint64_t)first + n > cam->matrices_cap) return r3_fail(c, R3_E_INVALID, "readback_object_matrices: range");
    cudaSetDevice(c->device);
    if (n) R3_CUDA(c, cudaMemcpyAsync(out, cam->d_matrices + first, (size_t)n * sizeof *out, cudaMemcpyDeviceToHost, c->stream));
    R3_CUDA(c, r3_stream_sync(c));
    return R3_OK;
}

// ------------------------------------------------------------------ InputOutputBuffer (suballoc.rs:66-222)
static uint64_t next_pow2_u64(uint64_t v) { uint64_t p = 1; while (p < v) p <<= 1; return p; }
static uint64_t io_capacity(uint64_t in, uint64_t out) { return next_pow2_u64(in > out ? in : out) * 2; }

int r3_iobuf_new(r3_ctx* c, r3_iobuf* b, uint64_t elems, uint64_t elem_size, bool clear_on_swap) {
    b->capacity_elements = io_capacity(elems, elems);
    b->out_elems = b->in_elems = elems; b->flipped = false; b->clear_on_swap = clear_on_swap; b->elem_size = elem_size;
    R3_CUDA(c, cudaMalloc((void**)&b->d, b->capacity_elements * elem_size + 16));
    R3_CUDA(c, cudaMemsetAsync(b->d, 0, b->capacity_elements * elem_size, c->stream));   // wgpu buffers start zeroed
    b->created = true;
    return R3_OK;
}
int r3_iobuf_swap(r3_ctx* c, r3_iobuf* b, uint64_t new_elems) {
    const uint64_t old_out = b->out_off(), old_cap = b->capacity_elements;
    b->in_elems = b->out_elems; b->out_elems = new_elems; b->flipped = !b->flipped;
    const uint64_t ncap = io_capacity(b->in_elems, b->out_elems);
    if (ncap != b->capacity_elements) {
        uint8_t* nd = nullptr;
        R3_CUDA(c, cudaMalloc((void**)&nd, ncap * b->elem_size + 16));
        R3_CUDA(c, cudaMemsetAsync(nd, 0, ncap * b->elem_size, c->stream));
        b->capacity_elements = ncap;
        if (!b->clear_on_swap) {
            uint64_t bytes = b->in_elems * b->elem_size, room = (old_cap - old_out) * b->elem_size;
            if (bytes > room) bytes = room;
            if (bytes) R3_CUDA(c, cudaMemcpyAsync(nd + b->in_off() * b->elem_size, b->d + old_out * b->elem_size, bytes, cudaMemcpyDeviceToDevice, c->stream));
        }
        R3_CUDA(c, r3_stream_sync(c));
        cudaFree(b->d);
        b->d = nd;
    } else if (b->clear_on_swap) {
        R3_CUDA(c, cudaMemsetAsync(b->d, 0, b->capacity_elements * b->elem_size, c->stream));
    }
    return R3_OK;
}

static int io_read(r3_ctx* c, const r3_iobuf* b, int partition, void* out, uint64_t cap, uint64_t* count) {
    if (!b->created) { if (count) *count = 0; return R3_OK; }
    uint64_t elems = partition ? b->in_elems : b->out_elems, off = partition ? b->in_off() : b->out_off();
    const uint64_t room = b->capacity_elements / 2;
    if (elems > room) elems = room;
    if (count) *count = elems;
    if (out && elems) {
        if (cap < elems) return r3_fail(c, R3_E_INVALID, "readback: capacity too small");
        R3_CUDA(c, cudaMemcpyAsync(out, b->d + off * b->elem_size, elems * b->elem_size, cudaMemcpyDeviceToHost, c->stream));
        R3_CUDA(c, r3_stream_sync(c));
    }
    return R3_OK;
}
R3_EXPORT int r3_readback_indices(r3_ctx* c, uint32_t camera, int partition, uint32_t* out, uint64_t cap, uint64_t* count) {
    R3_CAM_OR_FAIL(c, camera);
    cudaSetDevice(c->device);
    return io_read(c, &cam->index_buffer, partition, out, cap, count);
}
R3_EXPORT int r3_readback_draw_calls(r3_ctx* c, uint32_t camera, int partition, r3_indirect_call* out, uint32_t cap, uint32_t* count) {
    R3_CAM_OR_FAIL(c, camera);
    cudaSetDevice(c->device);
    uint64_t n = 0;
    int rc = io_read(c, &cam->draw_call_buffer, partition, out, cap, &n);
    if (count) *count = (uint32_t)n;
    return rc;
}
R3_EXPORT int r3_readback_culling_results(r3_ctx* c, uint32_t camera, int partition, uint32_t* out, uint64_t cap, uint64_t* count) {
    R3_CAM_OR_FAIL(c, camera);
    cudaSetDevice(c->device);
    return io_read(c, &cam->results_buffer, partition, out, cap, count);
}

// ------------------------------------------------------------------ batching glue
R3_EXPORT int r3_batch_objects(r3_ctx* c, uint32_t camera, const float vp_loc[3], uint32_t max_dispatch_count) {
    R3_CAM_OR_FAIL(c, camera);
    if (!vp_loc) return r3_fail(c, R3_E_INVALID, "batch_objects: null location");
    cudaSetDevice(c->device);
    // The device path never splits a batch at the dispatch limit (batching.rs:196); it is only taken when no batch can reach it:
    // 256 objects x the largest padded triangle count of any slot stays below max_dispatch_count x 256 invocations.  Worlds with
    // such meshes (> ~65k triangles in one object), material keys >= 64 or >= 2^24 slots take the host path, which splits.
    bool device = c->gpu_batching_ok && c->sort_key.size() >= cam->header.object_count;
    if (device) {
        R3_TRY(r3_compute_max_invocations(c));   // cached: one small reduction per object upload, never per frame
        device = c->max_object_invocations * R3_BATCH_SIZE < (uint64_t)max_dispatch_count * R3_WORKGROUP_SIZE;
    }
    cam->batching_path = device ? 1 : 2;   // the device path raises it to 3 when it takes the frame-wide sort
    if (device) return r3_device_batch_objects(c, cam, vp_loc, max_dispatch_count);
    return r3_host_batch_objects(c, cam, vp_loc, max_dispatch_count);
}
R3_EXPORT int r3_batching_info(r3_ctx* c, uint32_t camera, uint32_t info[4]) {
    R3_CAM_OR_FAIL(c, camera);
    if (!info) return r3_fail(c, R3_E_INVALID, "batching_info: null");
    cudaSetDevice(c->device);
    info[0] = (uint32_t)cam->batching_path; info[1] = 0; info[2] = 0; info[3] = 0;
    const r3_jobs& j = cam->jobs[cam->cur];
    if ((cam->batching_path == 1 || cam->batching_path == 3) && j.d_header) {
        uint32_t hdr[8] = {0};
        R3_CUDA(c, cudaMemcpyAsync(hdr, j.d_header, 32, cudaMemcpyDeviceToHost, c->stream));
        R3_CUDA(c, r3_stream_sync(c));
        info[1] = hdr[4]; info[2] = hdr[1]; info[3] = hdr[2];
    } else if (cam->batching_path == 2) {
        info[2] = (uint32_t)j.batches.size(); info[3] = (uint32_t)j.regions.size();
    }
    return R3_OK;
}
R3_EXPORT int r3_batch_counts(r3_ctx* c, uint32_t camera, uint32_t* nb, uint32_t* nr, uint32_t* tot) {
    R3_CAM_OR_FAIL(c, camera);
    cudaSetDevice(c->device);
    R3_TRY(r3_download_jobs(c, cam));
    const r3_jobs& j = cam->jobs[cam->cur];
    if (nb) *nb = (uint32_t)j.batches.size();
    if (nr) *nr = (uint32_t)j.regions.size();
    if (tot) {
        uint64_t t = 0;
        for (const auto& b : j.batches) t += b.total_invocations;
        *tot = (uint32_t)t;
    }
    return R3_OK;
}
R3_EXPORT int r3_readback_batches(r3_ctx* c, uint32_t camera, r3_batch_data* b, r3_region* r) {
    R3_CAM_OR_FAIL(c, camera);
    cudaSetDevice(c->device);
    R3_TRY(r3_download_jobs(c, cam));
    const r3_jobs& j = cam->jobs[cam->cur];
    if (b && !j.batches.empty()) memcpy(b, j.batches.data(), j.batches.size() * sizeof *b);
    if (r && !j.regions.empty()) memcpy(r, j.regions.data(), j.regions.size() * sizeof *r);
    return R3_OK;
}

R3_EXPORT int r3_cull(r3_ctx* c, uint32_t camera, const r3_batch_data* batches, uint32_t n_batches, const r3_region* regions,
                      uint32_t n_regions) {
    R3_CAM_OR_FAIL(c, camera);
    cudaSetDevice(c->device);
    if (!cam->header_set) return r3_fail(c, R3_E_STATE, "cull before object_uniform_upload");
    if (batches) cam->cur = (cam->cache_idx == 0) ? 1 : 0;   // never overwrite the cached DrawCallSet
    r3_jobs& j = cam->jobs[cam->cur];
    if (batches) {
        if (!regions) return r3_fail(c, R3_E_INVALID, "cull: batches without regions");
        j.batches.assign(batches, batches + n_batches);
        j.regions.assign(regions, regions + n_regions);
        uint64_t tot = 0;
        for (const auto& b : j.batches) tot += b.total_invocations;
        j.total_invocations = (uint32_t)tot;
        j.device_built = false;
    }
    if (!j.device_built) {
        if (j.batches.empty()) { cam->has_draw_call_set = false; return R3_OK; }   // culler.rs:705-707
        R3_TRY(r3_upload_jobs(c, cam));
    }
    return r3_launch_triangle_cull(c, cam);
}

// ------------------------------------------------------------------ multi-GPU plumbing
R3_EXPORT int r3_device_ptr(r3_ctx* c, uint32_t camera, int which, void** p, uint64_t* nbytes) {
    R3_CAM_OR_FAIL(c, camera);
    if (!p || !nbytes) return r3_fail(c, R3_E_INVALID, "device_ptr: null");
    if (which == 0) { *p = cam->d_visible; *nbytes = (uint64_t)cam->visible_cap * 4; }
    else if (which == 1) { *p = c->d_hdr16; *nbytes = (uint64_t)c->width * c->height * 8; }
    else if (which == 2) { *p = cam->d_matrices; *nbytes = (uint64_t)cam->matrices_cap * 128; }
    else if (which == 3) { *p = cam->d_visible_count; *nbytes = 4; }
    else if (which == 4) { *p = cam->d_words; *nbytes = (((uint64_t)cam->header.object_count + 31) / 32) * 4; }   // 1 bit per object
    else if (which == 5) { *p = c->d_atlas; *nbytes = (uint64_t)c->atlas_w * c->atlas_h * 4; }   // shadow atlas (depth32f; reverse-Z depths order like their bits)
    else return r3_fail(c, R3_E_INVALID, "device_ptr: which");
    return R3_OK;
}
