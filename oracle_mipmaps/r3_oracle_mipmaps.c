/* r3_oracle_mipmaps.c — CPU ORACLE of r3_generate_mipmaps / r3_readback_texels (TEST INFRASTRUCTURE; never linked into or called by
 * the product).  It works on the context of the CPU oracle (oracle/r3_oracle.h: the texture table and texel blob r3o_set_textures
 * keeps) and exports r3o_generate_mipmaps / r3o_readback_texels; oracle_mipmaps/__init__.py binds both next to the oracle's own
 * entry points.  Level by level, no fusion; OpenMP over destination rows; -ffp-contract=off like the rest of the oracle.
 *
 * Rule R12 — MipmapGenerator::generate_mipmaps (rend3/src/util/mipmap.rs:139-219, mipmap.wgsl).  The reference renders each level with
 * a fullscreen triangle that samples the previous level through a linear ClampToEdge sampler, so the arithmetic belongs to the
 * rasteriser, the sampler and the render-target encoder; R12 fixes it:
 *   sizes      destination level l+1 is (w', h') = (max(w >> 1, 1), max(h >> 1, 1)); level l is the source;
 *   footprint  texel (i, j) of level l+1: tex_coords at the pixel centre is (i + 0.5) / w', the sampler looks at u w - 0.5, i.e.
 *              num = (2i + 1) w - w', den = 2 w', x0 = num / den (integer division), fx = (float)(num % den) / (float)den (one IEEE
 *              division of exact operands; even sizes give fx = 0.5 exactly, the 2x2 box); y0, fy the same way with h;
 *   addressing ClampToEdge: x0 + 1 and y0 + 1 are clamped to the level;
 *   blend      per channel, on decoded values, in this order, never contracted, gx = 1 - fx, gy = 1 - fy:
 *              (t00 gx + t10 fx) gy + (t01 gx + t11 fx) fy;
 *   decode     unorm k / (2^b - 1) (Rgb10a2's alpha / 3); *Srgb rgb through the table D of include/r3_srgb_tables.h (the correctly
 *              rounded f32 of the exact EOTF; no powf), alpha linear; f16 widened exactly; Bgra8 swizzled;
 *   encode     into the texture's own format (the reference renders into it and the next level samples the quantised level):
 *              unorm: NaN -> 0, clamp to [0, 1], rint(v (2^b - 1)) ties to even; *Srgb rgb: the number of k in 0..254 with v >= T[k]
 *              (T of r3_srgb_tables.h: the correctly rounded OETF, ties up; NaN -> 0); f16: round to nearest even, overflow to +-inf,
 *              every NaN to 0x7E00; channels the format does not store are not written.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>

#include "../include/rend3_b200.h"
#include "../oracle/r3_oracle.h"
#include "../include/r3_srgb_tables.h"

#define API __attribute__((visibility("default")))

static int fail(r3o_ctx* c, const char* msg) {
    if (c) snprintf(c->err, sizeof c->err, "%s", msg);
    return R3_E_INVALID;
}

static int format_ok(uint32_t f) {   /* FILTERABLE and RENDER_ATTACHMENT in wgpu: what rend3-gltf asks Generated for (lib.rs:1082-1087) */
    return f == R3_TEXFMT_RGBA8_UNORM || f == R3_TEXFMT_RGBA8_UNORM_SRGB || f == R3_TEXFMT_BGRA8_UNORM || f == R3_TEXFMT_BGRA8_UNORM_SRGB ||
           f == R3_TEXFMT_R8_UNORM || f == R3_TEXFMT_RG8_UNORM || f == R3_TEXFMT_RGB10A2_UNORM || f == R3_TEXFMT_R16_FLOAT ||
           f == R3_TEXFMT_RG16_FLOAT || f == R3_TEXFMT_RGBA16_FLOAT;
}

/* ---- f16 by hand (no compiler conversion): f16 -> f32 exact, f32 -> f16 round to nearest even */
static float h2f(uint16_t h) {
    uint32_t sign = (uint32_t)(h & 0x8000u) << 16, e = (h >> 10) & 31u, m = h & 0x3FFu, bits;
    if (e == 0) {
        float v = (float)m * 5.9604644775390625e-8f;   /* m 2^-24, exact */
        return (h & 0x8000u) ? -v : v;
    }
    bits = e == 31 ? (sign | 0x7F800000u | (m << 13)) : (sign | ((e + 112u) << 23) | (m << 13));
    float f; memcpy(&f, &bits, 4);
    return f;
}
static uint16_t f2h(float f) {
    uint32_t x; memcpy(&x, &f, 4);
    const uint32_t sign = (x >> 16) & 0x8000u, exp = (x >> 23) & 255u;
    uint32_t mant = x & 0x7FFFFFu;
    if (exp == 255u) return mant ? 0x7E00u : (uint16_t)(sign | 0x7C00u);    /* every NaN -> 0x7E00 */
    const int32_t e = (int32_t)exp - 127 + 15;                               /* biased f16 exponent */
    if (e >= 31) return (uint16_t)(sign | 0x7C00u);
    if (e <= 0) {                                                            /* subnormal result (or zero) */
        if (e < -10) return (uint16_t)sign;
        mant |= 0x800000u;
        const uint32_t shift = (uint32_t)(14 - e), q = mant >> shift, rem = mant & ((1u << shift) - 1u), half = 1u << (shift - 1u);
        return (uint16_t)(sign | (q + (rem > half || (rem == half && (q & 1u)))));
    }
    const uint32_t q = ((uint32_t)e << 10) | (mant >> 13), rem = mant & 0x1FFFu;
    return (uint16_t)(sign | (q + (rem > 0x1000u || (rem == 0x1000u && (q & 1u)))));   /* a carry may reach 0x7C00: +-inf */
}

static uint32_t bpp_of(uint32_t f) { return R3_TEXFMT_BPP(f); }
static float un(uint32_t k, float full) { return (float)k / full; }
static void decode(const uint8_t* p, uint32_t f, float* o) {
    uint32_t v = 0;
    switch (f) {
    case R3_TEXFMT_RGBA8_UNORM: for (int k = 0; k < 4; ++k) o[k] = un(p[k], 255.0f); break;
    case R3_TEXFMT_RGBA8_UNORM_SRGB: for (int k = 0; k < 3; ++k) o[k] = r3_srgb_decode[p[k]]; o[3] = un(p[3], 255.0f); break;
    case R3_TEXFMT_BGRA8_UNORM: for (int k = 0; k < 3; ++k) o[k] = un(p[2 - k], 255.0f); o[3] = un(p[3], 255.0f); break;
    case R3_TEXFMT_BGRA8_UNORM_SRGB: for (int k = 0; k < 3; ++k) o[k] = r3_srgb_decode[p[2 - k]]; o[3] = un(p[3], 255.0f); break;
    case R3_TEXFMT_R8_UNORM: o[0] = un(p[0], 255.0f); break;
    case R3_TEXFMT_RG8_UNORM: o[0] = un(p[0], 255.0f); o[1] = un(p[1], 255.0f); break;
    case R3_TEXFMT_RGB10A2_UNORM:
        memcpy(&v, p, 4);
        for (int k = 0; k < 3; ++k) o[k] = un((v >> (10 * k)) & 1023u, 1023.0f);
        o[3] = un(v >> 30, 3.0f);
        break;
    default: {   /* R16 / RG16 / RGBA16 float */
        const int n = f == R3_TEXFMT_R16_FLOAT ? 1 : f == R3_TEXFMT_RG16_FLOAT ? 2 : 4;
        for (int k = 0; k < n; ++k) { uint16_t h; memcpy(&h, p + 2 * k, 2); o[k] = h2f(h); }
    }
    }
}
static uint32_t enc_unorm(float v, float full) {
    if (v != v) return 0;
    v = v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v);
    return (uint32_t)rintf(v * full);
}
static uint8_t enc_srgb(float v) {   /* the number of k with v >= T[k] */
    uint32_t n = 0;
    while (n < 255 && v >= r3_srgb_encode[n]) ++n;
    return (uint8_t)n;
}
static void encode(const float* c, uint32_t f, uint8_t* p) {
    uint32_t v;
    switch (f) {
    case R3_TEXFMT_RGBA8_UNORM: for (int k = 0; k < 4; ++k) p[k] = (uint8_t)enc_unorm(c[k], 255.0f); break;
    case R3_TEXFMT_RGBA8_UNORM_SRGB: for (int k = 0; k < 3; ++k) p[k] = enc_srgb(c[k]); p[3] = (uint8_t)enc_unorm(c[3], 255.0f); break;
    case R3_TEXFMT_BGRA8_UNORM: for (int k = 0; k < 3; ++k) p[2 - k] = (uint8_t)enc_unorm(c[k], 255.0f); p[3] = (uint8_t)enc_unorm(c[3], 255.0f); break;
    case R3_TEXFMT_BGRA8_UNORM_SRGB: for (int k = 0; k < 3; ++k) p[2 - k] = enc_srgb(c[k]); p[3] = (uint8_t)enc_unorm(c[3], 255.0f); break;
    case R3_TEXFMT_R8_UNORM: p[0] = (uint8_t)enc_unorm(c[0], 255.0f); break;
    case R3_TEXFMT_RG8_UNORM: p[0] = (uint8_t)enc_unorm(c[0], 255.0f); p[1] = (uint8_t)enc_unorm(c[1], 255.0f); break;
    case R3_TEXFMT_RGB10A2_UNORM:
        v = enc_unorm(c[0], 1023.0f) | enc_unorm(c[1], 1023.0f) << 10 | enc_unorm(c[2], 1023.0f) << 20 | enc_unorm(c[3], 3.0f) << 30;
        memcpy(p, &v, 4);
        break;
    default: {
        const int n = f == R3_TEXFMT_R16_FLOAT ? 1 : f == R3_TEXFMT_RG16_FLOAT ? 2 : 4;
        for (int k = 0; k < n; ++k) { uint16_t h = f2h(c[k]); memcpy(p + 2 * k, &h, 2); }
    }
    }
}

/* one level: dst (dw x dh) from src (sw x sh) */
static void mip_level(const uint8_t* src, uint8_t* dst, uint32_t f, uint32_t sw, uint32_t sh) {
    const uint32_t dw = sw >> 1 ? sw >> 1 : 1, dh = sh >> 1 ? sh >> 1 : 1, bpp = bpp_of(f);
#pragma omp parallel for schedule(static)
    for (int64_t j = 0; j < (int64_t)dh; ++j) {
        const uint64_t ny = (2 * (uint64_t)j + 1) * sh - dh, dy = 2 * (uint64_t)dh;
        const uint32_t y0 = (uint32_t)(ny / dy), y1 = y0 + 1 < sh ? y0 + 1 : sh - 1;
        const float fy = (float)(ny % dy) / (float)dy, gy = 1.0f - fy;
        for (uint32_t i = 0; i < dw; ++i) {
            const uint64_t nx = (2 * (uint64_t)i + 1) * sw - dw, dx = 2 * (uint64_t)dw;
            const uint32_t x0 = (uint32_t)(nx / dx), x1 = x0 + 1 < sw ? x0 + 1 : sw - 1;
            const float fx = (float)(nx % dx) / (float)dx, gx = 1.0f - fx;
            float t00[4] = {0}, t10[4] = {0}, t01[4] = {0}, t11[4] = {0}, out[4];
            decode(src + ((uint64_t)y0 * sw + x0) * bpp, f, t00);
            decode(src + ((uint64_t)y0 * sw + x1) * bpp, f, t10);
            decode(src + ((uint64_t)y1 * sw + x0) * bpp, f, t01);
            decode(src + ((uint64_t)y1 * sw + x1) * bpp, f, t11);
            for (int k = 0; k < 4; ++k) {
                const float top = t00[k] * gx + t10[k] * fx, bot = t01[k] * gx + t11[k] * fx;
                out[k] = top * gy + bot * fy;
            }
            encode(out, f, dst + ((uint64_t)j * dw + i) * bpp);
        }
    }
}

static uint64_t chain_bytes(const r3_texture_desc* d) {
    uint64_t total = 0;
    for (uint32_t l = 0; l < d->mip_count; ++l) total += R3_TEXFMT_LEVEL_BYTES(d->format, (d->width >> l) ? (d->width >> l) : 1u, (d->height >> l) ? (d->height >> l) : 1u);
    return total;
}

API int r3o_generate_mipmaps(r3o_ctx* c, const uint32_t* indices, uint32_t count) {
    if (!c || (!indices && count)) return fail(c, "generate_mipmaps: null");
    for (uint32_t n = 0; n < count; ++n) {   /* the whole list first: a rejected call changes no byte */
        const uint32_t i = indices[n];
        if (i >= c->n_textures) return fail(c, "generate_mipmaps: index outside the texture table");
        for (uint32_t m = 0; m < n; ++m)
            if (indices[m] == i) return fail(c, "generate_mipmaps: index listed twice");
        const r3_texture_desc* d = &c->tex_descs[i];
        if (!format_ok(d->format)) return fail(c, "generate_mipmaps: format is not filterable and renderable");
        uint32_t max_mips = 0;
        for (uint32_t s = d->width > d->height ? d->width : d->height; s; s >>= 1) ++max_mips;
        if (d->mip_count > max_mips) return fail(c, "generate_mipmaps: mip_count exceeds floor(log2(max(w, h))) + 1");
        for (uint32_t m = 0; m < n; ++m) {
            const r3_texture_desc* e = &c->tex_descs[indices[m]];
            if (d->byte_offset < e->byte_offset + chain_bytes(e) && e->byte_offset < d->byte_offset + chain_bytes(d))
                return fail(c, "generate_mipmaps: two listed mip chains overlap");
        }
    }
    for (uint32_t n = 0; n < count; ++n) {
        const r3_texture_desc* d = &c->tex_descs[indices[n]];
        uint32_t w = d->width, h = d->height;
        uint8_t* lv = c->texels + d->byte_offset;
        for (uint32_t l = 1; l < d->mip_count; ++l) {
            uint8_t* next = lv + R3_TEXFMT_LEVEL_BYTES(d->format, w, h);
            mip_level(lv, next, d->format, w, h);
            lv = next;
            w = w >> 1 ? w >> 1 : 1;
            h = h >> 1 ? h >> 1 : 1;
        }
    }
    return R3_OK;
}

API int r3o_readback_texels(r3o_ctx* c, uint64_t byte_offset, void* dst, uint64_t nbytes) {
    if (!c || (!dst && nbytes)) return fail(c, "readback_texels: null");
    if (byte_offset > c->texel_bytes || nbytes > c->texel_bytes - byte_offset) return fail(c, "readback_texels: range outside the texel blob");
    if (nbytes) memcpy(dst, c->texels + byte_offset, nbytes);
    return R3_OK;
}
