// r3_mipmap.cu — MipmapGenerator::generate_mipmaps (rend3/src/util/mipmap.rs:139-219, mipmap.wgsl) for r3_generate_mipmaps:
// levels 1 .. mip_count-1 of listed table entries computed from level 0 by rule R12 (oracle_mipmaps/r3_oracle_mipmaps.c, DESIGN.md §2).
//
// One call is a fixed sequence of launches, whatever the number of textures:
//   mip_head_kernel   a CTA owns a 64x64 tile of level 0 of every texture whose first levels have even sizes (or size 1); under R12 the
//                     footprint of every destination texel then stays inside the tile, so the CTA produces the next levels (up to six,
//                     64x64 -> 1x1) in shared memory;
//   mip_level_kernel  one launch per remaining level depth across all textures (odd sizes: footprints cross tiles), grid-stride over
//                     destination row segments;
//   mip_tail_kernel   one CTA per texture finishes every level whose source fits in shared memory.
// Each destination texel comes from ONE function, mip_texel(), over a source accessor (global or shared memory).  Every level is
// stored in the texture's own format and the next level decodes those stored bits again, so the fused levels equal the per-level
// result bit for bit.  Compiled with -fmad=false: the blend is the oracle's operation sequence.
#include <cuda_fp16.h>

#include <algorithm>
#include <cstring>

#include "r3_common.cuh"
#define R3_SRGB_TABLE __device__ const
#include "../../include/r3_srgb_tables.h"

namespace {

constexpr uint32_t MIP_TILE = 64;                        // head tile edge (level-0 texels)
constexpr uint32_t MIP_MAX_FUSED = 6;                    // 64 -> 1
constexpr uint32_t MIP_SMEM_TEXELS = MIP_TILE * MIP_TILE;   // largest source region a CTA holds (head tile, tail source)
constexpr uint32_t MIP_THREADS = 256;
constexpr uint32_t MIP_SEGMENT = 256;                    // destination texels per work item of mip_level_kernel

__device__ __forceinline__ uint32_t fmt_bpp(uint32_t f) { return R3_TEXFMT_BPP(f); }

// stored bits of one texel (at most 8 bytes: Rgba16Float) <-> linear values; channels the format does not store are ignored
__device__ __forceinline__ uint2 load_raw(const uint8_t* p, uint32_t bpp) {
    if (bpp == 8) return *reinterpret_cast<const uint2*>(p);
    if (bpp == 4) return make_uint2(*reinterpret_cast<const uint32_t*>(p), 0u);
    if (bpp == 2) return make_uint2(*reinterpret_cast<const uint16_t*>(p), 0u);
    return make_uint2(*p, 0u);
}
__device__ __forceinline__ void store_raw(uint8_t* p, uint32_t bpp, uint2 v) {
    if (bpp == 8) *reinterpret_cast<uint2*>(p) = v;
    else if (bpp == 4) *reinterpret_cast<uint32_t*>(p) = v.x;
    else if (bpp == 2) *reinterpret_cast<uint16_t*>(p) = (uint16_t)v.x;
    else *p = (uint8_t)v.x;
}
// per-CTA copies in shared memory of what decode / encode look up: k / 255 (the same correctly rounded quotients as div_rn), the sRGB
// decode table, the sRGB encode thresholds (padded with +inf)
struct MipLut { float unorm8[256], srgb_dec[256], srgb_enc[256]; };
__device__ __forceinline__ void lut_load(MipLut& L) {
    for (uint32_t k = threadIdx.x; k < 256u; k += blockDim.x) {
        L.unorm8[k] = div_rn((float)k, 255.0f);
        L.srgb_dec[k] = r3_srgb_decode[k];
        L.srgb_enc[k] = k < 255u ? r3_srgb_encode[k] : __int_as_float(0x7F800000);
    }
    __syncthreads();
}
__device__ __forceinline__ float half_of(uint32_t h) { return __half2float(__ushort_as_half((unsigned short)h)); }
__device__ __forceinline__ float4 decode(uint2 r, uint32_t f, const MipLut& L) {
    const uint32_t v = r.x;
    switch (f) {
    case R3_TEXFMT_RGBA8_UNORM: return make_float4(L.unorm8[v & 255u], L.unorm8[(v >> 8) & 255u], L.unorm8[(v >> 16) & 255u], L.unorm8[v >> 24]);
    case R3_TEXFMT_RGBA8_UNORM_SRGB: return make_float4(L.srgb_dec[v & 255u], L.srgb_dec[(v >> 8) & 255u], L.srgb_dec[(v >> 16) & 255u], L.unorm8[v >> 24]);
    case R3_TEXFMT_BGRA8_UNORM: return make_float4(L.unorm8[(v >> 16) & 255u], L.unorm8[(v >> 8) & 255u], L.unorm8[v & 255u], L.unorm8[v >> 24]);
    case R3_TEXFMT_BGRA8_UNORM_SRGB: return make_float4(L.srgb_dec[(v >> 16) & 255u], L.srgb_dec[(v >> 8) & 255u], L.srgb_dec[v & 255u], L.unorm8[v >> 24]);
    case R3_TEXFMT_R8_UNORM: return make_float4(L.unorm8[v & 255u], 0.0f, 0.0f, 0.0f);
    case R3_TEXFMT_RG8_UNORM: return make_float4(L.unorm8[v & 255u], L.unorm8[(v >> 8) & 255u], 0.0f, 0.0f);
    case R3_TEXFMT_RGB10A2_UNORM:
        return make_float4(div_rn((float)(v & 1023u), 1023.0f), div_rn((float)((v >> 10) & 1023u), 1023.0f), div_rn((float)((v >> 20) & 1023u), 1023.0f), div_rn((float)(v >> 30), 3.0f));
    case R3_TEXFMT_R16_FLOAT: return make_float4(half_of(v & 0xFFFFu), 0.0f, 0.0f, 0.0f);
    case R3_TEXFMT_RG16_FLOAT: return make_float4(half_of(v & 0xFFFFu), half_of(v >> 16), 0.0f, 0.0f);
    default: return make_float4(half_of(v & 0xFFFFu), half_of(v >> 16), half_of(r.y & 0xFFFFu), half_of(r.y >> 16));   // Rgba16Float
    }
}
__device__ __forceinline__ uint32_t enc_unorm(float v, float full) {
    if (!(v == v)) return 0u;
    v = fminf(fmaxf(v, 0.0f), 1.0f);
    return (uint32_t)rintf(mul_rn(v, full));
}
__device__ __forceinline__ uint32_t enc_srgb(float v, const MipLut& L) {   // number of k with v >= T[k] (NaN compares false: 0)
    uint32_t n = 0u;
#pragma unroll
    for (uint32_t step = 128u; step; step >>= 1)   // branch-free search over the 256 padded thresholds (T[255] = +inf)
        if (v >= L.srgb_enc[n + step - 1u]) n += step;
    return n;
}
__device__ __forceinline__ uint32_t enc_half(float v) {
    if (!(v == v)) return 0x7E00u;
    return (uint32_t)__half_as_ushort(__float2half_rn(v));   // round to nearest even, overflow to +-inf
}
__device__ __forceinline__ uint2 encode(float4 c, uint32_t f, const MipLut& L) {
    switch (f) {
    case R3_TEXFMT_RGBA8_UNORM: return make_uint2(enc_unorm(c.x, 255.0f) | enc_unorm(c.y, 255.0f) << 8 | enc_unorm(c.z, 255.0f) << 16 | enc_unorm(c.w, 255.0f) << 24, 0u);
    case R3_TEXFMT_RGBA8_UNORM_SRGB: return make_uint2(enc_srgb(c.x, L) | enc_srgb(c.y, L) << 8 | enc_srgb(c.z, L) << 16 | enc_unorm(c.w, 255.0f) << 24, 0u);
    case R3_TEXFMT_BGRA8_UNORM: return make_uint2(enc_unorm(c.z, 255.0f) | enc_unorm(c.y, 255.0f) << 8 | enc_unorm(c.x, 255.0f) << 16 | enc_unorm(c.w, 255.0f) << 24, 0u);
    case R3_TEXFMT_BGRA8_UNORM_SRGB: return make_uint2(enc_srgb(c.z, L) | enc_srgb(c.y, L) << 8 | enc_srgb(c.x, L) << 16 | enc_unorm(c.w, 255.0f) << 24, 0u);
    case R3_TEXFMT_R8_UNORM: return make_uint2(enc_unorm(c.x, 255.0f), 0u);
    case R3_TEXFMT_RG8_UNORM: return make_uint2(enc_unorm(c.x, 255.0f) | enc_unorm(c.y, 255.0f) << 8, 0u);
    case R3_TEXFMT_RGB10A2_UNORM: return make_uint2(enc_unorm(c.x, 1023.0f) | enc_unorm(c.y, 1023.0f) << 10 | enc_unorm(c.z, 1023.0f) << 20 | enc_unorm(c.w, 3.0f) << 30, 0u);
    case R3_TEXFMT_R16_FLOAT: return make_uint2(enc_half(c.x), 0u);
    case R3_TEXFMT_RG16_FLOAT: return make_uint2(enc_half(c.x) | enc_half(c.y) << 16, 0u);
    default: return make_uint2(enc_half(c.x) | enc_half(c.y) << 16, enc_half(c.z) | enc_half(c.w) << 16);
    }
}

// rule R12 for destination texel (i, j) of a (dw, dh) level from its (sw, sh) source: the bilinear ClampToEdge sample of the fullscreen
// triangle at the texel centre, footprint x = ((2i + 1) sw - dw) / (2 dw) as an exact integer quotient plus an f32 remainder ratio
template <class Src>
__device__ __forceinline__ float4 mip_texel(const Src& src, uint32_t sw, uint32_t sh, uint32_t dw, uint32_t dh, uint32_t i, uint32_t j) {
    uint32_t x0, y0, rx, ry;
    if (sw < 65536u && sh < 65536u) {   // (2i + 1) sw - dw < 2^32: 32-bit integer division (64-bit division is a long software sequence)
        const uint32_t nx = (2u * i + 1u) * sw - dw, ny = (2u * j + 1u) * sh - dh;
        x0 = nx / (2u * dw); rx = nx - x0 * (2u * dw); y0 = ny / (2u * dh); ry = ny - y0 * (2u * dh);
    } else {
        const unsigned long long nx = (2ull * i + 1ull) * sw - dw, ny = (2ull * j + 1ull) * sh - dh;
        x0 = (uint32_t)(nx / (2ull * dw)); rx = (uint32_t)(nx % (2ull * dw)); y0 = (uint32_t)(ny / (2ull * dh)); ry = (uint32_t)(ny % (2ull * dh));
    }
    const float fx = div_rn((float)rx, (float)(2ull * dw)), fy = div_rn((float)ry, (float)(2ull * dh));
    const uint32_t x1 = min(x0 + 1u, sw - 1u), y1 = min(y0 + 1u, sh - 1u);
    const float gx = sub_rn(1.0f, fx), gy = sub_rn(1.0f, fy);
    const float4 t00 = src(x0, y0), t10 = src(x1, y0), t01 = src(x0, y1), t11 = src(x1, y1);
    auto blend = [&](float a00, float a10, float a01, float a11) {
        return add_rn(mul_rn(add_rn(mul_rn(a00, gx), mul_rn(a10, fx)), gy), mul_rn(add_rn(mul_rn(a01, gx), mul_rn(a11, fx)), fy));
    };
    return make_float4(blend(t00.x, t10.x, t01.x, t11.x), blend(t00.y, t10.y, t01.y, t11.y), blend(t00.z, t10.z, t01.z, t11.z), blend(t00.w, t10.w, t01.w, t11.w));
}

// a source level in global memory (level coordinates)
struct GlobalSrc {
    const uint8_t* base; uint32_t pitch_texels, bpp, fmt; const MipLut& L;
    __device__ float4 operator()(uint32_t x, uint32_t y) const { return decode(load_raw(base + ((unsigned long long)y * pitch_texels + x) * bpp, bpp), fmt, L); }
};
// a region [ox, ox + ex) x [oy, oy + ey) of a source level held in shared memory, stored bits, rows of ex texels
struct SharedSrc {
    const uint8_t* base; uint32_t ox, oy, ex, bpp, fmt; const MipLut& L;
    __device__ float4 operator()(uint32_t x, uint32_t y) const { return decode(load_raw(base + ((y - oy) * ex + (x - ox)) * bpp, bpp), fmt, L); }
};

__device__ __forceinline__ uint32_t job_of(const r3_mip_job* jobs, uint32_t n_jobs, uint32_t item) {   // last job with item_begin <= item
    uint32_t lo = 0u, hi = n_jobs;
    while (hi - lo > 1u) {
        const uint32_t mid = (lo + hi) >> 1;
        if (jobs[mid].item_begin <= item) lo = mid; else hi = mid;
    }
    return lo;
}

// `levels` levels of one region: the source region is copied into shared memory (16-byte vectors when its rows allow), then every
// level goes from shared memory to shared memory, each stored to the blob as well
__device__ void mip_region_chain(uint8_t* texels, const r3_mip_job& jb, uint32_t ox, uint32_t oy, uint32_t ex, uint32_t ey, uint8_t* buf_a, uint8_t* buf_b,
                                 const MipLut& L) {
    const uint32_t bpp = fmt_bpp(jb.fmt), row_bytes = ex * bpp;
    const uint8_t* src = texels + jb.src_off;
    const unsigned long long pitch = (unsigned long long)jb.sw * bpp;
    if ((pitch & 15ull) == 0ull && (row_bytes & 15u) == 0u && ((jb.src_off + ox * bpp) & 15ull) == 0ull) {
        const uint32_t vec_per_row = row_bytes >> 4;
        for (uint32_t k = threadIdx.x; k < vec_per_row * ey; k += blockDim.x) {
            const uint32_t r = k / vec_per_row, v = k - r * vec_per_row;
            reinterpret_cast<uint4*>(buf_a + r * row_bytes)[v] = __ldg(reinterpret_cast<const uint4*>(src + (oy + r) * pitch + ox * bpp) + v);
        }
    } else {
        for (uint32_t k = threadIdx.x; k < ex * ey; k += blockDim.x) {
            const uint32_t r = k / ex, x = k - r * ex;
            store_raw(buf_a + k * bpp, bpp, load_raw(src + (oy + r) * pitch + (unsigned long long)(ox + x) * bpp, bpp));
        }
    }
    __syncthreads();
    uint32_t sw = jb.sw, sh = jb.sh;
    unsigned long long dst_off = jb.src_off + (unsigned long long)sw * sh * bpp;
    uint8_t *cur = buf_a, *nxt = buf_b;
    for (uint32_t l = 0; l < jb.levels; ++l) {
        const uint32_t dw = max(sw >> 1, 1u), dh = max(sh >> 1, 1u);
        const uint32_t dox = ox >> 1, doy = oy >> 1, dex = min((ox + ex + 1u) >> 1, dw) - dox, dey = min((oy + ey + 1u) >> 1, dh) - doy;
        const SharedSrc s{cur, ox, oy, ex, bpp, jb.fmt, L};
        uint8_t* dst = texels + dst_off;
        for (uint32_t k = threadIdx.x; k < dex * dey; k += blockDim.x) {
            const uint32_t r = k / dex, x = dox + (k - r * dex), y = doy + r;
            const uint2 v = encode(mip_texel(s, sw, sh, dw, dh, x, y), jb.fmt, L);
            store_raw(dst + ((unsigned long long)y * dw + x) * bpp, bpp, v);
            store_raw(nxt + k * bpp, bpp, v);
        }
        __syncthreads();
        uint8_t* t = cur; cur = nxt; nxt = t;
        dst_off += (unsigned long long)dw * dh * bpp;
        sw = dw; sh = dh; ox = dox; oy = doy; ex = dex; ey = dey;
    }
}

}  // namespace

// kernel names are stable (global scope): profiles and traces find them as mip_head_kernel / mip_level_kernel / mip_tail_kernel
__global__ void __launch_bounds__(MIP_THREADS) mip_head_kernel(uint8_t* __restrict__ texels, const r3_mip_job* __restrict__ jobs, uint32_t n_jobs, uint32_t n_items) {
    __shared__ __align__(16) uint8_t buf_a[MIP_SMEM_TEXELS * 8];
    __shared__ __align__(16) uint8_t buf_b[MIP_SMEM_TEXELS * 8 / 4];
    __shared__ MipLut L;
    lut_load(L);
    for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x) {
        const r3_mip_job jb = jobs[job_of(jobs, n_jobs, item)];
        const uint32_t t = item - jb.item_begin, tx = t % jb.tiles_x, ty = t / jb.tiles_x;
        const uint32_t ox = tx * MIP_TILE, oy = ty * MIP_TILE;
        mip_region_chain(texels, jb, ox, oy, min(MIP_TILE, jb.sw - ox), min(MIP_TILE, jb.sh - oy), buf_a, buf_b, L);
    }
}

__global__ void __launch_bounds__(MIP_THREADS) mip_level_kernel(uint8_t* __restrict__ texels, const r3_mip_job* __restrict__ jobs, uint32_t n_jobs, uint32_t n_items) {
    __shared__ MipLut L;
    lut_load(L);
    for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x) {
        const r3_mip_job& jb = jobs[job_of(jobs, n_jobs, item)];
        const uint32_t bpp = fmt_bpp(jb.fmt), sw = jb.sw, sh = jb.sh, dw = max(sw >> 1, 1u), dh = max(sh >> 1, 1u);
        const uint32_t t = item - jb.item_begin, y = t / jb.tiles_x, x = (t - y * jb.tiles_x) * MIP_SEGMENT + threadIdx.x;
        if (x >= dw) continue;
        const GlobalSrc s{texels + jb.src_off, sw, bpp, jb.fmt, L};
        store_raw(texels + jb.src_off + (unsigned long long)sw * sh * bpp + ((unsigned long long)y * dw + x) * bpp, bpp, encode(mip_texel(s, sw, sh, dw, dh, x, y), jb.fmt, L));
    }
}

__global__ void __launch_bounds__(MIP_THREADS) mip_tail_kernel(uint8_t* __restrict__ texels, const r3_mip_job* __restrict__ jobs, uint32_t n_jobs) {
    extern __shared__ __align__(16) uint8_t mip_tail_smem[];   // MIP_TAIL_SMEM bytes: buf_a | buf_b | tables (over the 48 KB static limit)
    uint8_t *buf_a = mip_tail_smem, *buf_b = buf_a + MIP_SMEM_TEXELS * 8;
    MipLut& L = *reinterpret_cast<MipLut*>(buf_b + MIP_SMEM_TEXELS * 8 / 2);
    lut_load(L);
    for (uint32_t j = blockIdx.x; j < n_jobs; j += gridDim.x) {
        const r3_mip_job jb = jobs[j];
        mip_region_chain(texels, jb, 0u, 0u, jb.sw, jb.sh, buf_a, buf_b, L);
        __syncthreads();
    }
}

constexpr size_t MIP_TAIL_SMEM = MIP_SMEM_TEXELS * 8 + MIP_SMEM_TEXELS * 8 / 2 + sizeof(MipLut);

static uint64_t level_bytes(uint32_t f, uint32_t w, uint32_t h) { return R3_TEXFMT_LEVEL_BYTES(f, w, h); }

// The work list of one call (host side, from the descriptor copy r3_set_textures keeps): head jobs, then the jobs of every level
// depth, then the tail jobs, uploaded with one copy.  `indices` were validated by r3_generate_mipmaps.
int r3_launch_mipmaps(r3_ctx* c, const uint32_t* indices, uint32_t count) {
    std::vector<r3_mip_job> head, tail;
    std::vector<std::vector<r3_mip_job>> depth;
    for (uint32_t n = 0; n < count; ++n) {
        const r3_texture_desc& d = c->tex_descs_host[indices[n]];
        uint32_t left = d.mip_count - 1u, w = d.width, h = d.height;
        uint64_t off = d.byte_offset;
        if (!left) continue;
        auto advance = [&](uint32_t levels) {
            for (uint32_t l = 0; l < levels; ++l) { off += level_bytes(d.format, w, h); w = std::max(w >> 1, 1u); h = std::max(h >> 1, 1u); }
            left -= levels;
        };
        if ((uint64_t)w * h > MIP_SMEM_TEXELS) {
            uint32_t fused = 0, fw = w, fh = h;
            while (fused < left && fused < MIP_MAX_FUSED && (fw % 2 == 0 || fw == 1) && (fh % 2 == 0 || fh == 1)) { fw = std::max(fw >> 1, 1u); fh = std::max(fh >> 1, 1u); ++fused; }
            if (fused) {
                const uint32_t tx = (w + MIP_TILE - 1) / MIP_TILE, ty = (h + MIP_TILE - 1) / MIP_TILE;
                head.push_back(r3_mip_job{off, w, h, d.format, fused, tx, tx * ty});
                advance(fused);
            }
        }
        for (uint32_t k = 0; left && (uint64_t)w * h > MIP_SMEM_TEXELS; ++k) {
            if (depth.size() <= k) depth.emplace_back();
            const uint32_t segs = (std::max(w >> 1, 1u) + MIP_SEGMENT - 1) / MIP_SEGMENT;
            depth[k].push_back(r3_mip_job{off, w, h, d.format, 1u, segs, segs * std::max(h >> 1, 1u)});
            advance(1);
        }
        if (left) tail.push_back(r3_mip_job{off, w, h, d.format, left, 1u, 1u});
    }
    // item_begin: `items` of each job turned into the first item of the job within its launch
    std::vector<r3_mip_job> plan;
    std::vector<uint32_t> launch_first, launch_jobs, launch_items;
    auto add = [&](std::vector<r3_mip_job>& jobs) {
        uint32_t items = 0;
        launch_first.push_back((uint32_t)plan.size());
        launch_jobs.push_back((uint32_t)jobs.size());
        for (r3_mip_job& j : jobs) { const uint32_t n = j.item_begin; j.item_begin = items; items += n; plan.push_back(j); }
        launch_items.push_back(items);
    };
    add(head);
    for (auto& v : depth) add(v);
    add(tail);
    if (plan.empty()) return R3_OK;
    const uint64_t bytes = plan.size() * sizeof(r3_mip_job);
    // the list of the previous call is still on the device when nothing changed (the frame-after-frame case): no copy at all
    if (c->mip_plan_host.size() != bytes || std::memcmp(c->mip_plan_host.data(), plan.data(), bytes) != 0) {
        R3_TRY(r3_reserve_t(c, &c->d_mip_jobs, &c->mip_jobs_cap, plan.size()));
        const void* src = plan.data();
        if (c->capturing) {   // a captured copy reads its source when the graph runs: stage it in pinned memory that outlives this call
            if (c->mip_staging_used + bytes > c->mip_staging_cap) {
                const uint64_t cap = std::max<uint64_t>(2 * c->mip_staging_cap, std::max<uint64_t>(bytes, 64 * 1024));
                void* p = nullptr;
                R3_CUDA(c, cudaMallocHost(&p, cap));
                if (c->mip_staging) c->mip_staging_retired.push_back(c->mip_staging);   // earlier copies in this recording may still read it
                c->mip_staging = (uint8_t*)p; c->mip_staging_cap = cap; c->mip_staging_used = 0;
            }
            uint8_t* dst = c->mip_staging + c->mip_staging_used;
            std::memcpy(dst, plan.data(), bytes);
            c->mip_staging_used += (bytes + 15) & ~15ull;
            src = dst;
        }
        R3_CUDA(c, cudaMemcpyAsync(c->d_mip_jobs, src, bytes, cudaMemcpyHostToDevice, c->stream));
        c->mip_plan_host.assign((const uint8_t*)plan.data(), (const uint8_t*)plan.data() + bytes);
    }
    if (!c->mip_tail_smem_set) {
        R3_CUDA(c, cudaFuncSetAttribute(mip_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MIP_TAIL_SMEM));
        c->mip_tail_smem_set = true;
    }
    const r3_mip_job* jobs = c->d_mip_jobs;
    const size_t last = launch_first.size() - 1;
    r3_stage_begin(c, R3_STAGE_MIPMAPS);   // the three kernels of one call are one stage
    if (launch_jobs[0]) {
        mip_head_kernel<<<std::min(launch_items[0], (uint32_t)R3_SM_COUNT * 8u), MIP_THREADS, 0, c->stream>>>(c->d_texels, jobs, launch_jobs[0], launch_items[0]);
        R3_CHECK_LAUNCH(c, "mip_head_kernel");
    }
    for (size_t k = 1; k < last; ++k) {
        mip_level_kernel<<<std::min(launch_items[k], (uint32_t)R3_SM_COUNT * 16u), MIP_THREADS, 0, c->stream>>>(c->d_texels, jobs + launch_first[k], launch_jobs[k], launch_items[k]);
        R3_CHECK_LAUNCH(c, "mip_level_kernel");
    }
    if (launch_jobs[last]) {
        mip_tail_kernel<<<std::min(launch_jobs[last], (uint32_t)R3_SM_COUNT * 8u), MIP_THREADS, MIP_TAIL_SMEM, c->stream>>>(c->d_texels, jobs + launch_first[last], launch_jobs[last]);
        R3_CHECK_LAUNCH(c, "mip_tail_kernel");
    }
    r3_stage_end(c);
    return R3_OK;
}
