/* rend3_b200.h — C ABI of librend3_b200.so: rend3's GPU-driven per-object hot path on B200.
 *
 * The library replaces, beneath rend3's public Renderer/Object/Material/RenderGraph API, the
 * work that `rend3-routine` records into wgpu for:
 *     GpuCuller::object_uniform_upload  + uniform_prep.wgsl     (culling/culler.rs:427-529)
 *     batch_objects                                              (culling/batching.rs:120-250)
 *     GpuCuller::cull                   + cull.wgsl              (culling/culler.rs:531-659)
 *     ForwardRoutine::add_forward_to_graph + opaque.wgsl/depth.wgsl (forward.rs:192-315)
 *     HiZRoutine::add_hi_z_to_graph     + hi_z.wgsl              (hi_z.rs:161-234)
 *     TonemappingRoutine::add_to_graph  + blit.wgsl              (tonemapping.rs:108-147)
 * in the node order of BaseRenderGraph::add_to_graph (base.rs:129-185).
 *
 * Conventions
 *   - every entry point returns 0 on success, a negative R3_E_* code otherwise; the message is
 *     available from r3_last_error().  Nothing unwinds, aborts or exits across the boundary
 *     (the reference panics inside graph nodes, culler.rs:439,572 — a C ABI cannot).
 *   - host pointers are borrowed for the duration of the call only; the library owns all
 *     device memory.  Buffers are the std430 bytes rend3's managers already produce
 *     (r3_layouts.h), so the Rust side uploads exactly what it uploads to wgpu today.
 *   - one context per GPU; calls on a context must be externally serialised (this is the
 *     `data_core` mutex of the reference, rend3/src/graph/graph.rs:265).  The per-frame entry points
 *     (r3_object_uniform_upload, r3_batch_objects, r3_cull, r3_shadow_pass, r3_forward_*, r3_hiz_build, r3_tonemap,
 *     r3_skin's kernel, r3_exchange_merge, r3_peer_*) only enqueue work on the context's stream and return.
 *     What BLOCKS the calling thread until the stream has drained: r3_sync, every r3_readback_*, r3_visible_count,
 *     r3_batch_counts / r3_batching_info / r3_forward_stats / r3_stage_times (small device-to-host reads), and the
 *     uploads that borrow a HOST pointer — r3_set_objects, r3_update_objects, r3_set_object_sort_info,
 *     r3_set_mesh_buffer, r3_set_materials, r3_set_textures, r3_set_skybox, r3_set_*_lights, r3_skin's joint upload —
 *     because the pointer is only valid for the duration of the call (they are the counterpart of queue.write_buffer,
 *     which copies before it returns).  r3_set_objects_device borrows device memory and does not block.  A buffer that
 *     has to grow (first frame, larger world, new resolution) is reallocated with a stream synchronisation as well.
 *   - `camera` is R3_CAMERA_VIEWPORT or a shadow index 0..R3_MAX_SHADOWS-1
 *     (CameraSpecifier, rend3-routine/src/common/camera.rs).
 */
#ifndef REND3_B200_H
#define REND3_B200_H

#include <stddef.h>
#include <stdint.h>

#include "r3_layouts.h"

#ifdef __cplusplus
extern "C" {
#endif

#define R3_ABI_VERSION 1u
#define R3_MAX_SHADOWS 63u

enum {
    R3_OK = 0,
    R3_E_INVALID = -1,   /* bad argument / call order (the reference's assert!/unwrap sites) */
    R3_E_CUDA = -2,      /* CUDA runtime failure; message carries cudaGetErrorString */
    R3_E_OOM = -3,       /* allocation failed (MeshCreationError::BufferAllocationFailed analogue) */
    R3_E_NO_DEVICE = -4, /* RendererInitializationError::MissingAdapter analogue */
    R3_E_STATE = -5      /* required earlier stage has not run for this camera/frame */
};

typedef struct r3_ctx r3_ctx;

/* ------------------------------------------------------------------ context */
uint32_t r3_abi_version(void);
/* replaces rend3::create_iad + GpuCuller::new/PbrRoutine::new pipeline creation (base.rs:111-124) */
int r3_ctx_create(int device, r3_ctx** out);
int r3_ctx_destroy(r3_ctx* ctx);
const char* r3_last_error(const r3_ctx* ctx);
int r3_sync(r3_ctx* ctx);
/* the CUDA stream all work of this context is enqueued on (cudaStream_t as void*) */
int r3_get_stream(r3_ctx* ctx, void** stream);
/* number of kernel launches issued by this context since creation (bench.py gpu_launches) */
int r3_launch_count(r3_ctx* ctx, uint64_t* launches);

/* Frame submission as ONE CUDA graph launch (the reference submits once per frame, rend3/src/graph/graph.rs:510).  Optional: bracket
 * the per-frame calls (r3_clear_shadow_atlas ... r3_tonemap) with r3_frame_begin / r3_frame_end.  The stream work in between is recorded
 * by stream capture instead of being launched; r3_frame_end turns it into a graph — the instantiated graph of the previous frame of the
 * same parity is updated in place (cudaGraphExecUpdate: same kernels, this frame's arguments and ping-pong pointers), so steady-state
 * frames pay no instantiation — and launches it.  A call that has to wait for the stream inside the bracket (a buffer that must grow, a
 * host-side batch_objects, a readback) submits what was recorded so far, waits, and the rest of the frame runs eagerly; results are the
 * same either way.  stats: [0] frames ended, [1] frames submitted as a graph, [2] early flushes, [3] graph (re)instantiations. */
int r3_frame_begin(r3_ctx* ctx);
int r3_frame_end(r3_ctx* ctx);
int r3_frame_graph_stats(r3_ctx* ctx, uint64_t stats[4]);

/* optional per-stage device timing (off by default): when enabled, CUDA event pairs are recorded around the kernels below and
 * r3_stage_times returns, per stage, the summed duration in ms and the number of launches since the last call (it synchronises).
 * stage ids: 0 triangle_test_kernel, 1 raster_setup_kernel (colour passes), 2 raster_setup_kernel (shadow passes), 3 raster_band_kernel,
 * 4 resolve_kernel, 5 the batch_objects sort, 6 cull_bake_kernel, 7 triangle_compact_kernel, 8 r3_generate_mipmaps (read with r3_stage_times_n). */
int r3_set_stage_timing(r3_ctx* ctx, int enabled);
int r3_stage_times(r3_ctx* ctx, double ms[8], uint32_t launches[8]);
/* the same for the first n_stages stages (at most 9): stage 8 = r3_generate_mipmaps (mip_head / mip_level / mip_tail kernels of one call
 * timed as one pair, launches = calls) */
int r3_stage_times_n(r3_ctx* ctx, uint32_t n_stages, double* ms, uint32_t* launches);

/* ------------------------------------------------------------------ world data
 * same bytes as the wgpu buffers named on the right */
int r3_set_objects(r3_ctx*, const r3_object* records, uint32_t n_slots);           /* object_manager.buffer::<M>() (object.rs:193) */
int r3_update_objects(r3_ctx*, const uint32_t* slots, const r3_object* records, uint32_t n); /* ScatterCopy (object.rs:344-364) */
/* borrow an object buffer that already lives in device memory (zero copy; caller keeps it alive) */
int r3_set_objects_device(r3_ctx*, const void* device_records, uint32_t n_slots);
/* facts batch_objects reads from the object/material managers (batching.rs:144-167):
 * flags bit0 = slot is live (enumerated_objects), bit1 = SortingReason::Optimization
 * ("atomic capable"), bit2 = SortingOrder::BackToFront.  location = InternalObject::location. */
int r3_set_object_sort_info(r3_ctx*, const uint64_t* material_key, const uint8_t* flags,
                            const float* location_xyz, uint32_t n_slots);
int r3_set_mesh_buffer(r3_ctx*, const void* bytes, uint64_t nbytes);               /* eval_output.mesh_buffer (mesh.rs:99) */
int r3_set_materials(r3_ctx*, const r3_material* records, uint32_t count);         /* material_manager.archetype_view::<M>().buffer() */
/* the bindless d2 texture table the material records index (TextureManager::add / fill, rend3/src/managers/texture.rs;
 * `textures[material.albedo_tex - 1u]`, opaque.wgsl:152-161): descriptors + one blob with every mip level.  Sampling is
 * textureSampleGrad with the linear or nearest Repeat sampler of common/samplers.rs:42-56 (trilinear, no anisotropy). */
int r3_set_textures(r3_ctx*, const r3_texture_desc* descs, uint32_t count, const void* texels, uint64_t nbytes);
/* SkyboxRoutine::set_background_texture (rend3-routine/src/skybox.rs:47-60): the cube map skybox.wgsl samples wherever the depth buffer
 * still holds its clear value.  desc->width = face size (height is ignored), six faces in the order +X, -X, +Y, -Y, +Z, -Z, each with
 * its `mip_count` levels stored tightly, face after face, from desc->byte_offset.  desc == NULL removes the skybox. */
int r3_set_skybox(r3_ctx*, const r3_texture_desc* desc, const void* texels, uint64_t nbytes);
/* MipmapGenerator::generate_mipmaps (rend3/src/util/mipmap.rs:139-219) for the textures TextureManager::add created with
 * MipmapSource::Generated: levels 1 .. mip_count-1 of each listed table entry are computed from its level 0 by rule R12 and
 * written into the resident texel blob.  The bytes of those levels that r3_set_textures uploaded are ignored.  Stream-ordered,
 * no host synchronisation (capturable inside r3_frame_begin / r3_frame_end).  The whole list is validated first; R3_E_INVALID, with
 * no byte changed, for an index outside the table or listed twice, mip_count > floor(log2(max(w, h))) + 1, two listed chains that
 * overlap in the blob, or a format outside Rgba8Unorm(Srgb), Bgra8Unorm(Srgb), R8Unorm, Rg8Unorm, Rgb10a2Unorm, R16Float, Rg16Float,
 * Rgba16Float (the formats wgpu guarantees FILTERABLE and RENDER_ATTACHMENT).  mip_count == 1 is a valid no-op. */
int r3_generate_mipmaps(r3_ctx*, const uint32_t* texture_indices, uint32_t count);
/* test / tool path: blocking copy of texel-blob bytes [byte_offset, byte_offset + nbytes) */
int r3_readback_texels(r3_ctx*, uint64_t byte_offset, void* dst, uint64_t nbytes);
int r3_set_directional_lights(r3_ctx*, const void* bytes, uint64_t nbytes,
                              uint32_t atlas_width, uint32_t atlas_height);         /* directional.rs:135-156 */
int r3_set_point_lights(r3_ctx*, const void* bytes, uint64_t nbytes);              /* point.rs:58-74 */
int r3_set_frame_uniforms(r3_ctx*, const r3_frame_uniforms* uniforms);             /* uniforms.rs:94-106 */

/* ------------------------------------------------------------------ GPU skinning
 * add_skinning_to_graph / GpuSkinner::execute_pass (rend3-routine/src/skinning.rs:54-199) + skinning.wgsl:37-94:
 * 4-joint linear blend of position / normal / tangent from the unskinned attribute ranges into the skeleton's
 * overridden ranges of the mesh buffer, one launch for all skeletons.  joint_matrices = global_joint_count mat4. */
int r3_skin(r3_ctx*, const r3_skinning_input* inputs, uint32_t n_skeletons, const float* joint_matrices, uint32_t n_joints);
int r3_readback_mesh_buffer(r3_ctx*, void* bytes, uint64_t capacity_bytes);

/* ------------------------------------------------------------------ per-object cull + uniform bake
 * GpuCuller::object_uniform_upload (culler.rs:427-529) fused with the sphere-frustum test of
 * batch_objects (batching.rs:144-148, util/frustum.rs:148-161): for every slot < object_count
 * bakes MV/MVP when `enabled`, and appends the slot to the camera's ascending visible list when
 * it is live and its world sphere is inside the 5 planes. */
#define R3_CB_BAKE 1u
#define R3_CB_CULL 2u
int r3_object_uniform_upload(r3_ctx*, uint32_t camera, const r3_camera_header* header, uint32_t mode);
int r3_visible_count(r3_ctx*, uint32_t camera, uint32_t* count);
int r3_readback_visible(r3_ctx*, uint32_t camera, uint32_t* out, uint32_t capacity, uint32_t* count);
int r3_readback_object_matrices(r3_ctx*, uint32_t camera, r3_object_matrices* out, uint32_t first, uint32_t n);

/* ------------------------------------------------------------------ batching + per-triangle cull
 * batch_objects (batching.rs:120-250) over the camera's visible list: sort by ShaderJobSortingKey,
 * pack <=256 objects per ShaderBatchData, split regions on key change, remember each object's
 * global invocation for next frame.  `viewport_location` = viewport_camera_state.location(). */
int r3_batch_objects(r3_ctx*, uint32_t camera, const float viewport_location[3], uint32_t max_dispatch_count);
int r3_batch_counts(r3_ctx*, uint32_t camera, uint32_t* n_batches, uint32_t* n_regions, uint32_t* total_invocations);
int r3_readback_batches(r3_ctx*, uint32_t camera, r3_batch_data* batches, r3_region* regions);
/* which implementation of batch_objects ran last for this camera, and what it built: info[0] = 0 none / 1 on the device (radix sort +
 * block scans, no host sync) / 2 on the host (material keys >= 64, >= 2^24 slots, or a mesh large enough that a batch could reach the
 * max_dispatch_count x 256 split of batching.rs:196, which only the host path implements) / 3 on the device, order taken from the
 * frame-wide sort the cameras of one frame share (the sort key does not depend on the camera, batching.rs:156-157); info[1] = device overflow flag (always 0
 * given the check above; kept as a tripwire); info[2] = batches, info[3] = regions.  Blocks (one 32-byte readback). */
int r3_batching_info(r3_ctx*, uint32_t camera, uint32_t info[4]);
/* GpuCuller::cull (culler.rs:531-659) + cull.wgsl.  batches/regions == NULL uses the jobs of the last
 * r3_batch_objects call; otherwise the caller's own ShaderBatchDatas (a Rust batch_objects). */
int r3_cull(r3_ctx*, uint32_t camera, const r3_batch_data* batches, uint32_t n_batches,
            const r3_region* regions, uint32_t n_regions);
/* CullingBuffers readback (culler.rs:88-125).  `partition`: 0 = Output (predicted, kept for next
 * frame), 1 = Input (residual / previous frame).  Sizes in elements. */
int r3_readback_indices(r3_ctx*, uint32_t camera, int partition, uint32_t* out, uint64_t capacity, uint64_t* count);
int r3_readback_draw_calls(r3_ctx*, uint32_t camera, int partition, r3_indirect_call* out, uint32_t capacity, uint32_t* count);
int r3_readback_culling_results(r3_ctx*, uint32_t camera, int partition, uint32_t* out, uint64_t capacity, uint64_t* count);

/* ------------------------------------------------------------------ forward path
 * render targets of BaseRenderGraphIntermediateState::new (base.rs:212-290): hdr colour rgba16f,
 * depth32f (reverse-Z, cleared to 0.0, compare GreaterEqual), shadow atlas depth32f. */
int r3_set_render_target(r3_ctx*, uint32_t width, uint32_t height, uint32_t samples, const float clear_color[4]);
int r3_clear_shadow_atlas(r3_ctx*);                                                /* clear.rs / base.rs:293-295 */
/* pbr_shadow_rendering (base.rs:366-396): depth.wgsl over the shadow camera's culled list, into
 * the atlas viewport (offset, size). */
int r3_shadow_pass(r3_ctx*, uint32_t shadow_index, uint32_t offset_x, uint32_t offset_y, uint32_t size);
/* begin the primary render pass: colour = clear colour, depth = 0.0 (base.rs:257-264) */
int r3_forward_begin(r3_ctx*);
/* ForwardRoutine::add_forward_to_graph for the opaque + cutout routines.
 * source 0 = CullingSource::Predicted (last frame's list, forward.rs:224-232),
 *        1 = CullingSource::Residual (this frame's residual list, forward.rs:212-222). */
int r3_forward_pass(r3_ctx*, int source);
int r3_hiz_build(r3_ctx*);                                                          /* hi_z.rs:161-234 */
/* run opaque.wgsl::fs_main for the winning fragment of every covered pixel */
int r3_forward_resolve(r3_ctx*);
/* pbr_forward_rendering_transparent (base.rs:181,450-466): the blend routine (pbr/routine.rs:129; material key 2,
 * BlendState::ALPHA_BLENDING, depth test + write) over this frame's residual list, whose non-atomic regions keep the
 * back-to-front object order of batch_objects (cull.wgsl:374-380).  Call after r3_forward_resolve: it blends into the
 * shaded rgba16f target.  A no-op when no object carries material key 2. */
int r3_forward_blend(r3_ctx*);
int r3_tonemap(r3_ctx*, int srgb_target);                                           /* tonemapping.rs:108-147 */

/* Parity instrumentation, OFF by default: when enabled the shading kernels also store their f32 result before the rgba16f rounding
 * (16 B per pixel more than the reference's targets write) so that tests can hold fs_main to 1e-4 without the half-precision step.
 * r3_readback_hdr_f32 fails with R3_E_STATE while it is off. */
int r3_set_parity_target(r3_ctx*, int enabled);
int r3_readback_hdr_f32(r3_ctx*, float* rgba, uint64_t capacity_floats);            /* pre-f16 shading result (parity target) */
int r3_readback_hdr_f16(r3_ctx*, uint16_t* rgba, uint64_t capacity_halfs);          /* the Rgba16Float target */
int r3_readback_depth(r3_ctx*, float* depth, uint64_t capacity);
int r3_readback_ldr(r3_ctx*, uint8_t* rgba8, uint64_t capacity);
int r3_readback_shadow_atlas(r3_ctx*, float* depth, uint64_t capacity);
int r3_readback_hiz(r3_ctx*, uint32_t mip, float* depth, uint64_t capacity, uint32_t* width, uint32_t* height);
/* forward statistics of the last frame: [0] triangles set up, [1] fragments rasterised (covered samples sent
 * to the depth test), [2] fragments shaded by r3_forward_resolve (fs_main invocations), [3] sample fragments blended by
 * r3_forward_blend (depth-test survivors of the blend routine) */
int r3_forward_stats(r3_ctx*, uint64_t stats[4]);
/* surface_shading evaluations (opaque.wgsl:440-468) of the last r3_forward_resolve, summed over its fragments (single-sampled targets):
 * directional lights + the point lights that survived the tile culling and the per-fragment range test — the flop count of the pass */
int r3_forward_light_evaluations(r3_ctx*, uint64_t* evaluations);

/* ------------------------------------------------------------------ multi-GPU plumbing
 * raw device views so torch.distributed / NCCL can move the visible list and tile rows without a
 * host bounce.  which: 0 visible list (u32), 1 hdr f16 colour, 2 object matrices, 3 visible count (u32),
 * 4 visibility words (1 bit per object slot, bit i of word w = slot 32*w + i), 5 shadow atlas (depth32f: ranks that render
 * different shadow maps merge them with an integer MAX all-reduce, the atlas being cleared to 0.0) */
int r3_device_ptr(r3_ctx*, uint32_t camera, int which, void** device_ptr, uint64_t* nbytes);
/* Exchange of the visible set between the GPUs of one node over NVLink / NVSwitch peer memory (one process per GPU, objects
 * sharded in contiguous ranges, SURVEY 8e).  r3_exchange_create allocates this rank's buffer — epoch flags, acknowledgements and
 * rows[4][n_ranks][words_per_rank] (1 bit per object slot, rows 256-byte aligned, four row sets) — and returns its CUDA IPC handle; the
 * caller all-gathers the handles with whatever it already uses (torch.distributed, MPI) and hands them to r3_exchange_connect.  From then on
 * every r3_object_uniform_upload(CULL) on that camera is one EPOCH e: its compaction kernel also stores the visibility words into row
 * (e % 4, my_rank) of EVERY rank's buffer and publishes them with flags[e % 4][my_rank] = e (st.release.sys, after system-scope fences) —
 * no collective kernel runs.  Consumers run on the context's least-priority side stream, chained on the flags ON THE DEVICE (ld.acquire.sys,
 * no host barrier), overlapping the next culls: r3_exchange_count (visible objects of every shard) and r3_exchange_merge (the global
 * ascending visible list; r3_exchange_merged hands out its device pointers, rank_base == NULL numbers the shards r * max_objects_per_rank).
 * A consumer acknowledges its epoch to every producer; a producer that is about to overwrite a row set waits — on the device — until the
 * epoch it held has been acknowledged by all ranks.  Protocol: the ranks cull in lockstep and an epoch that one rank consumes, every rank
 * consumes (the acknowledgements are awaited on that assumption); consumers may lag up to three epochs before a producer blocks. */
#define R3_IPC_HANDLE_BYTES 64
int r3_exchange_create(r3_ctx*, uint32_t camera, uint32_t n_ranks, uint32_t my_rank, uint32_t max_objects_per_rank,
                       uint8_t handle_out[R3_IPC_HANDLE_BYTES]);
int r3_exchange_connect(r3_ctx*, uint32_t camera, const uint8_t* handles /* n_ranks x R3_IPC_HANDLE_BYTES, rank order */);
/* rows [n_ranks][words_per_rank] of the LAST epoch in this rank's buffer (complete for a host reader after a stream sync + a barrier) */
int r3_exchange_words(r3_ctx*, uint32_t camera, void** device_ptr, uint64_t* nbytes, uint32_t* words_per_rank);
int r3_exchange_merge(r3_ctx*, uint32_t camera, const uint32_t* rank_objects /* n_ranks */, const uint32_t* rank_base /* n_ranks or NULL */);
int r3_exchange_merged(r3_ctx*, uint32_t camera, void** device_list /* u32 global ids */, void** device_count /* u32 */, uint64_t* capacity);
/* the light consumer: waits for the flags like r3_exchange_merge but only counts — visible objects of every shard and their total — without
 * expanding the list (4 B per visible object of the WHOLE world on every rank: a cost that grows with the number of ranks);
 * r3_exchange_counts reads counts[0 .. n_ranks] (the last one is the total) back, blocking */
int r3_exchange_count(r3_ctx*, uint32_t camera, const uint32_t* rank_objects /* n_ranks */);
int r3_exchange_counts(r3_ctx*, uint32_t camera, uint32_t* counts /* n_ranks + 1 */);
int r3_exchange_destroy(r3_ctx*, uint32_t camera);
/* Peer-memory plumbing of the multi-GPU forward pass (SURVEY 8e: shadow maps split by light, screen split in row tiles; one process per
 * GPU on one NVLink / NVSwitch node).  r3_peer_create (after r3_set_directional_lights and r3_set_render_target: the atlas and the rgba16f
 * target must exist and must not be reallocated afterwards; the objects must be uploaded) returns four CUDA IPC handles — flag block,
 * shadow atlas, colour target, staging arrays of the sharded triangle test; the
 * caller all-gathers them and calls r3_peer_connect.  Then, all stream-ordered and without host synchronisation:
 *   r3_peer_send_atlas_rect  copies a rect of the local atlas into the same rect of EVERY peer's atlas (plain stores over NVLink);
 *   r3_peer_send_rows        copies rows of the local rgba16f target into the peers' targets (root >= 0: only into that rank's);
 *   r3_peer_signal(kind)     publishes everything sent so far: flags[kind][my_rank] = ++epoch on every rank (st.release.sys);
 *   r3_peer_wait(kind, e[])  a one-CTA kernel on this context's stream that spins (ld.acquire.sys) until flags[kind][r] >= e[r] for all r.
 * kinds: 0 shadow atlas, 1 colour rows, 2 frame done, 3 visibility words of the sharded triangle test (used by r3_cull itself).  rend3_b200/parallel.py::ForwardSplit shows the per-frame protocol. */
int r3_peer_create(r3_ctx*, uint32_t n_ranks, uint32_t my_rank, uint8_t handles_out[4 * R3_IPC_HANDLE_BYTES]);
int r3_peer_connect(r3_ctx*, const uint8_t* handles /* n_ranks x 4 x R3_IPC_HANDLE_BYTES, rank order */);
/* SURVEY 8e "triangle cull: shard by batch": with count = n_ranks (> 1), r3_cull of the VIEWPORT camera tests only this rank's run of
 * workgroups — they are laid out batch after batch, so a shard is a run of batches — stores its visibility words into the staging arrays
 * of every rank, publishes them (flag kind 3) and, once everybody's words have arrived, continues with the scan / compaction on the full
 * set: every rank ends up with the same index lists and draw records.  Falls back to testing everything while translucent (non-atomic)
 * objects exist, whose in-place index slots are not exchanged. */
int r3_set_cull_shard(r3_ctx*, uint32_t shard_index, uint32_t shard_count);
int r3_peer_send_atlas_rect(r3_ctx*, uint32_t offset_x, uint32_t offset_y, uint32_t width, uint32_t height);
int r3_peer_send_rows(r3_ctx*, uint32_t row_begin, uint32_t row_end, int root /* -1 = every peer */);
int r3_peer_signal(r3_ctx*, uint32_t kind);
int r3_peer_wait(r3_ctx*, uint32_t kind, const uint32_t* expected_epochs /* n_ranks */);
int r3_peer_destroy(r3_ctx*);
/* clear one shadow map's rect (a rank that renders only some of the lights clears only theirs; the others arrive from their owners) */
int r3_clear_shadow_rect(r3_ctx*, uint32_t offset_x, uint32_t offset_y, uint32_t width, uint32_t height);
/* restrict rasterisation + shading to pixel rows [row_begin, row_end) (screen-tile split, SURVEY 8e) */
int r3_set_scissor_rows(r3_ctx*, uint32_t row_begin, uint32_t row_end);

#ifdef __cplusplus
}
#endif
#endif /* REND3_B200_H */
