"""r3_generate_mipmaps (MipmapGenerator::generate_mipmaps, rule R12): the sRGB tables, the oracle against a float64 statement of R12, the
validation, the harness plumbing, and — on a B200 — the CUDA kernels bit for bit against the oracle."""
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from rend3_b200 import layouts as L
from rend3_b200.backend import R3Error, load_cuda_backend

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-4
SENTINEL = 0xA5

# accepted format -> (bytes per texel, stored channels)
FORMATS = {
    L.TEXFMT_RGBA8_UNORM: (4, 4), L.TEXFMT_RGBA8_UNORM_SRGB: (4, 4), L.TEXFMT_BGRA8_UNORM: (4, 4), L.TEXFMT_BGRA8_UNORM_SRGB: (4, 4),
    L.TEXFMT_R8_UNORM: (1, 1), L.TEXFMT_RG8_UNORM: (2, 2), L.TEXFMT_RGB10A2_UNORM: (4, 4),
    L.TEXFMT_R16_FLOAT: (2, 1), L.TEXFMT_RG16_FLOAT: (4, 2), L.TEXFMT_RGBA16_FLOAT: (8, 4),
}
SRGB = (L.TEXFMT_RGBA8_UNORM_SRGB, L.TEXFMT_BGRA8_UNORM_SRGB)


def oracle_backend():
    import oracle_mipmaps

    return oracle_mipmaps.load_oracle_backend()


def srgb_tables():
    text = open(os.path.join(ROOT, "include", "r3_srgb_tables.h")).read()
    vals = [float.fromhex(v) for v in re.findall(r"(-?0x[0-9a-f.]+p[-+]?\d+|0x0\.0p\+0)f", text)]
    assert len(vals) == 511
    return np.array(vals[:256], dtype=np.float32), np.array(vals[256:], dtype=np.float32)


def max_mips(w, h):
    return max(w, h).bit_length()


def dims(w, h, l):
    return max(w >> l, 1), max(h >> l, 1)


def chain_bytes(fmt, w, h, mips):
    return sum(dims(w, h, l)[0] * dims(w, h, l)[1] * FORMATS[fmt][0] for l in range(mips))


def make_table(specs, rng, gap=48):
    """specs: [(format, w, h, mip_count)] -> (descs, blob): random level 0, every other byte the sentinel, `gap` sentinel bytes
    between chains (all offsets 16-byte aligned)."""
    descs = np.zeros(len(specs), dtype=L.TEXTURE_DESC_DTYPE)
    parts, cursor = [np.full(gap, SENTINEL, np.uint8)], gap
    for i, (fmt, w, h, mips) in enumerate(specs):
        n = chain_bytes(fmt, w, h, mips)
        chain = np.full(n, SENTINEL, np.uint8)
        chain[: w * h * FORMATS[fmt][0]] = rng.integers(0, 256, w * h * FORMATS[fmt][0], dtype=np.uint8)
        descs[i]["width"], descs[i]["height"], descs[i]["mip_count"], descs[i]["format"], descs[i]["byte_offset"] = w, h, mips, fmt, cursor
        pad = (-n) % 16 + gap
        parts += [chain, np.full(pad, SENTINEL, np.uint8)]
        cursor += n + pad
    return descs, np.concatenate(parts)


def level_offsets(desc):
    fmt, w, h = int(desc["format"]), int(desc["width"]), int(desc["height"])
    off, out = int(desc["byte_offset"]), []
    for l in range(int(desc["mip_count"])):
        lw, lh = dims(w, h, l)
        out.append((off, lw, lh))
        off += lw * lh * FORMATS[fmt][0]
    return out


def run(backend, descs, blob, indices):
    backend.set_textures(descs, blob)
    backend.generate_mipmaps(np.asarray(indices, dtype=np.uint32))
    return backend.readback_texels(0, len(blob))


# ------------------------------------------------------------------ float64 statement of R12
def decode64(fmt, raw, w, h):
    """stored bytes of a w x h level -> (h, w, 4) float64 (channels the format does not store are 0)."""
    D, _ = srgb_tables()
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    out = np.zeros((h, w, 4))
    if fmt in (L.TEXFMT_RGBA8_UNORM, L.TEXFMT_RGBA8_UNORM_SRGB, L.TEXFMT_BGRA8_UNORM, L.TEXFMT_BGRA8_UNORM_SRGB):
        b = raw.reshape(h, w, 4)
        if fmt in (L.TEXFMT_BGRA8_UNORM, L.TEXFMT_BGRA8_UNORM_SRGB):
            b = b[..., [2, 1, 0, 3]]
        out = b / 255.0
        if fmt in SRGB:
            out[..., :3] = D[b[..., :3]].astype(np.float64)
    elif fmt in (L.TEXFMT_R8_UNORM, L.TEXFMT_RG8_UNORM):
        n = FORMATS[fmt][1]
        out[..., :n] = raw.reshape(h, w, n) / 255.0
    elif fmt == L.TEXFMT_RGB10A2_UNORM:
        v = raw.view("<u4").reshape(h, w).astype(np.int64)
        for k in range(3):
            out[..., k] = ((v >> (10 * k)) & 1023) / 1023.0
        out[..., 3] = (v >> 30) / 3.0
    else:
        n = FORMATS[fmt][1]
        out[..., :n] = raw.view("<f2").reshape(h, w, n).astype(np.float64)
    return out


def srgb_oetf(v):
    v = np.clip(v, 0.0, 1.0)
    return np.where(v <= 0.0031308, v * 12.92, 1.055 * np.power(v, 1 / 2.4) - 0.055)


def encode64(fmt, v):
    """(h, w, 4) float64 -> stored bytes (flat uint8) of the format, the exact-arithmetic statement of R12's encode."""
    h, w = v.shape[:2]
    v = np.where(np.isnan(v), 0.0, v) if fmt not in (L.TEXFMT_R16_FLOAT, L.TEXFMT_RG16_FLOAT, L.TEXFMT_RGBA16_FLOAT) else v
    un = lambda x, full: np.rint(np.clip(x, 0.0, 1.0) * full).astype(np.int64)
    if fmt in FORMATS and FORMATS[fmt][0] == 4 and fmt != L.TEXFMT_RGB10A2_UNORM and fmt not in (L.TEXFMT_RG16_FLOAT,):
        b = np.zeros((h, w, 4), np.int64)
        b[..., :3] = np.floor(srgb_oetf(v[..., :3]) * 255.0 + 0.5) if fmt in SRGB else un(v[..., :3], 255.0)
        b[..., 3] = un(v[..., 3], 255.0)
        if fmt in (L.TEXFMT_BGRA8_UNORM, L.TEXFMT_BGRA8_UNORM_SRGB):
            b = b[..., [2, 1, 0, 3]]
        return b.astype(np.uint8).reshape(-1)
    if fmt in (L.TEXFMT_R8_UNORM, L.TEXFMT_RG8_UNORM):
        return un(v[..., : FORMATS[fmt][1]], 255.0).astype(np.uint8).reshape(-1)
    if fmt == L.TEXFMT_RGB10A2_UNORM:
        c = un(v[..., :3], 1023.0)
        return np.ascontiguousarray((c[..., 0] | (c[..., 1] << 10) | (c[..., 2] << 20) | (un(v[..., 3], 3.0) << 30)).astype("<u4")).view(np.uint8).reshape(-1)
    hv = v[..., : FORMATS[fmt][1]].astype(np.float16)   # round to nearest even, overflow to inf
    bits = np.ascontiguousarray(hv).view(np.uint16).copy()
    bits[np.isnan(hv)] = 0x7E00
    return bits.astype("<u2").view(np.uint8).reshape(-1)


def r12_level64(src, sw, sh):
    """(sh, sw, 4) float64 decoded source -> (dh, dw, 4) float64 destination, R12's footprint and weights in exact arithmetic."""
    dw, dh = max(sw >> 1, 1), max(sh >> 1, 1)

    def axis(s, d):
        num = (2 * np.arange(d) + 1) * s - d
        i0 = num // (2 * d)
        return i0, np.minimum(i0 + 1, s - 1), (num % (2 * d)) / (2.0 * d)

    x0, x1, fx = axis(sw, dw)
    y0, y1, fy = axis(sh, dh)
    fx, fy = fx[None, :, None], fy[:, None, None]
    with np.errstate(invalid="ignore"):   # inf * 0 is NaN in R12 as in IEEE
        return _blend64(src, x0, x1, y0, y1, fx, fy)


def _blend64(src, x0, x1, y0, y1, fx, fy):
    top = src[y0][:, x0] * (1 - fx) + src[y0][:, x1] * fx
    bot = src[y1][:, x0] * (1 - fx) + src[y1][:, x1] * fx
    return top * (1 - fy) + bot * fy


def assert_level_matches_r12(fmt, got, src_raw, sw, sh):
    """The oracle's level against the float64 statement applied to the oracle's own source level: equal wherever the float64 value is not
    within 1e-6 (relative above 1) of a rounding boundary of the format."""
    dw, dh = max(sw >> 1, 1), max(sh >> 1, 1)
    v = r12_level64(decode64(fmt, src_raw, sw, sh), sw, sh)
    eps = 1e-6 * np.maximum(1.0, np.abs(np.nan_to_num(v, nan=0.0, posinf=0.0, neginf=0.0)))
    want, lo, hi = encode64(fmt, v), encode64(fmt, v - eps), encode64(fmt, v + eps)
    bpp = FORMATS[fmt][0]
    per_texel = lambda a: a.reshape(dh * dw, bpp)
    stable = np.all(per_texel(lo) == per_texel(hi), axis=1)
    bad = np.any(per_texel(got) != per_texel(want), axis=1) & stable
    assert not bad.any(), f"format {fmt} {sw}x{sh}: {bad.sum()} of {dw * dh} texels differ from the float64 statement of R12"
    assert stable.any() or dw * dh < 8


# ------------------------------------------------------------------ 1. sRGB tables
def test_srgb_tables_match_a_fresh_derivation():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import derive_srgb_tables

    assert open(os.path.join(ROOT, "include", "r3_srgb_tables.h")).read() == derive_srgb_tables.header()
    D, T = srgb_tables()
    assert np.all(np.diff(T.astype(np.float64)) > 0), "T must be strictly increasing"
    assert [int(np.sum(D[k] >= T)) for k in range(256)] == list(range(256)), "encode(D[k]) must give k back"


# ------------------------------------------------------------------ 2. the oracle against float64 R12
@pytest.mark.parametrize("fmt", sorted(FORMATS))
@pytest.mark.parametrize("w,h", [(8, 6), (5, 7), (13, 3), (33, 17)])
def test_oracle_levels_follow_r12(fmt, w, h):
    rng = np.random.default_rng(fmt * 100 + w * 10 + h)
    descs, blob = make_table([(fmt, w, h, max_mips(w, h))], rng)
    got = run(oracle_backend(), descs, blob, [0])
    lv = level_offsets(descs[0])
    for (so, sw, sh), (do, dw, dh) in zip(lv[:-1], lv[1:]):
        bpp = FORMATS[fmt][0]
        assert_level_matches_r12(fmt, got[do: do + dw * dh * bpp], got[so: so + sw * sh * bpp], sw, sh)


def test_oracle_even_size_is_the_2x2_box():
    src = np.array([[10, 20, 30, 40], [50, 60, 70, 80]], dtype=np.uint8)    # R8, 4 x 2 -> 2 x 1
    descs, blob = make_table([(L.TEXFMT_R8_UNORM, 4, 2, 2)], np.random.default_rng(0))
    off = int(descs[0]["byte_offset"])
    blob[off: off + 8] = src.reshape(-1)
    got = run(oracle_backend(), descs, blob, [0])
    assert list(got[off + 8: off + 10]) == [35, 55]


def _row(values, w, h=1):
    descs, blob = make_table([(L.TEXFMT_R8_UNORM, w, h, 2)], np.random.default_rng(1))
    off = int(descs[0]["byte_offset"])
    blob[off: off + w * h] = np.asarray(values, dtype=np.uint8)
    got = run(oracle_backend(), descs, blob, [0])
    return list(got[off + w * h: off + w * h + max(w >> 1, 1) * max(h >> 1, 1)])


def test_oracle_odd_sizes_hand_derived_weights():
    t = [0, 100, 200, 40, 240]
    # 5 -> 2: 1/4 t0 + 3/4 t1 and 3/4 t3 + 1/4 t4; t2 unused
    assert _row(t, 5) == [round(0.25 * t[0] + 0.75 * t[1]), round(0.75 * t[3] + 0.25 * t[4])]
    assert _row([0, 100, 7, 40, 240], 5) == _row(t, 5)
    # 7 -> 3: fx = 2/3, 0, 1/3 at x0 = 0, 3, 5: (1/3) 30 + (2/3) 90 = 70, t3, (2/3) 210 + (1/3) 255 = 225
    assert _row([30, 90, 11, 150, 13, 210, 255], 7) == [70, 150, 225]
    # 3 -> 1: the centre texel
    assert _row([0, 123, 255], 3) == [123]
    # the same along y (a 1-wide column)
    assert _row(t, 1, 5) == _row(t, 5)


@pytest.mark.parametrize("w,h", [(1, 1000), (1000, 1), (1, 7), (9, 1)])
def test_oracle_thin_chains(w, h):
    rng = np.random.default_rng(w + h)
    descs, blob = make_table([(L.TEXFMT_RGBA8_UNORM_SRGB, w, h, max_mips(w, h))], rng)
    got = run(oracle_backend(), descs, blob, [0])
    lv = level_offsets(descs[0])
    assert lv[-1][1:] == (1, 1)
    for (so, sw, sh), (do, dw, dh) in zip(lv[:-1], lv[1:]):
        assert_level_matches_r12(L.TEXFMT_RGBA8_UNORM_SRGB, got[do: do + dw * dh * 4], got[so: so + sw * sh * 4], sw, sh)


def test_oracle_one_texel_texture_is_a_no_op():
    descs, blob = make_table([(L.TEXFMT_RGBA8_UNORM, 1, 1, 1)], np.random.default_rng(3))
    assert np.array_equal(run(oracle_backend(), descs, blob, [0]), blob)


def test_oracle_f16_rounding_overflow_subnormals_nan():
    h = lambda x: int(np.float16(x).view(np.uint16))
    tiny = np.uint16(1).view(np.float16)                         # 2^-24
    one_ulp = np.float16(1.0) + np.float16(2.0 ** -10)
    cases = [  # (t0, t1): a 2 x 2 level whose rows are both (t0, t1) -> the 1 x 1 level, weights 1/2 exactly
        (h(1.0), h(one_ulp), h(1.0)),                            # 1 + ulp/2: tie to even (down)
        (h(one_ulp), h(np.float16(1.0) + np.float16(2.0 ** -9)), h(np.float16(1.0) + np.float16(2.0 ** -9))),   # 1 + 3 ulp/2: tie to even (up)
        (h(tiny), h(0.0), 0),                                    # 2^-25: tie to even -> 0
        (h(tiny), h(2 * tiny), h(2 * tiny)),                     # 1.5 * 2^-24 -> 2^-23 (even)
        (h(65504.0), h(65504.0), h(65504.0)),
        (0x7BFF, 0x7C00, 0x7C00),                                # inf stays inf
        (0xFC00, 0x7C00, 0x7E00),                                # -inf + inf: NaN -> 0x7E00
        (0x7D01, h(1.0), 0x7E00),                                # a NaN payload -> 0x7E00
        (0xFE00, h(1.0), 0x7E00),                                # a negative NaN -> 0x7E00
    ]
    for a, b, want in cases:
        descs, blob = make_table([(L.TEXFMT_R16_FLOAT, 2, 2, 2)], np.random.default_rng(4))
        off = int(descs[0]["byte_offset"])
        blob[off: off + 8] = np.array([a, b, a, b], dtype="<u2").view(np.uint8)
        got = run(oracle_backend(), descs, blob, [0])
        assert int(got[off + 8: off + 10].view("<u2")[0]) == int(want), (hex(a), hex(b))
    # a 1-high level: the clamped second row has weight 0, and inf * 0 is NaN
    descs, blob = make_table([(L.TEXFMT_R16_FLOAT, 2, 1, 2)], np.random.default_rng(4))
    off = int(descs[0]["byte_offset"])
    blob[off: off + 4] = np.array([0x7C00, h(1.0)], dtype="<u2").view(np.uint8)
    assert int(run(oracle_backend(), descs, blob, [0])[off + 4: off + 6].view("<u2")[0]) == 0x7E00, "inf * 0 (R12's unused row) is NaN"


def test_oracle_fewer_levels_and_untouched_bytes():
    rng = np.random.default_rng(5)
    specs = [(L.TEXFMT_RGBA8_UNORM, 37, 21, 3), (L.TEXFMT_RGBA16_FLOAT, 16, 16, 5), (L.TEXFMT_R8_UNORM, 9, 9, 4)]
    descs, blob = make_table(specs, rng)
    got = run(oracle_backend(), descs, blob, [2, 0])        # the 16 x 16 texture is not listed
    changed = np.zeros(len(blob), bool)
    for i in (0, 2):
        lv = level_offsets(descs[i])
        bpp = FORMATS[specs[i][0]][0]
        for o, w, h in lv[1:]:
            changed[o: o + w * h * bpp] = True
        o0, w0, h0 = lv[0]
        assert np.array_equal(got[o0: o0 + w0 * h0 * bpp], blob[o0: o0 + w0 * h0 * bpp]), "level 0 must not change"
    assert np.array_equal(got[~changed], blob[~changed]), "bytes outside the listed chains changed"
    assert (got[changed] != SENTINEL).mean() > 0.9


# ------------------------------------------------------------------ 3. rejections
def _rejection_cases():
    rng = np.random.default_rng(6)
    base = [(L.TEXFMT_RGBA8_UNORM, 8, 8, 4), (L.TEXFMT_RGBA8_UNORM, 4, 4, 3)]
    descs, blob = make_table(base, rng, gap=2048)   # room for the wider formats of the rejected descriptors
    yield "index outside the table", descs, blob, [0, 2]
    yield "index listed twice", descs, blob, [1, 0, 1]
    d2 = descs.copy(); d2[1]["mip_count"] = 4; d2[1]["width"] = 4; d2[1]["height"] = 4
    d2[0]["width"], d2[0]["height"], d2[0]["mip_count"] = 2, 1, 2     # max_mips(2, 1) = 2: fine; 3 is not
    d2[0]["mip_count"] = 3
    yield "mip_count above the maximum", d2, blob, [0]
    d3 = descs.copy(); d3[1]["byte_offset"] = d3[0]["byte_offset"] + 256   # inside the first chain (8x8x4 + ... bytes)
    yield "overlapping chains", d3, blob, [0, 1]
    for fmt in (L.TEXFMT_RGBA8_SNORM, L.TEXFMT_RGBA32_FLOAT, L.TEXFMT_R32_FLOAT, L.TEXFMT_RGBA16_UNORM, L.TEXFMT_BC1_RGBA_UNORM, L.TEXFMT_BC7_RGBA_UNORM_SRGB):
        d4 = descs.copy(); d4[1]["format"] = fmt
        yield f"format {fmt}", d4, blob, [0, 1]


REJECTIONS = list(_rejection_cases())


@pytest.mark.parametrize("case", REJECTIONS, ids=[c[0] for c in REJECTIONS])
def test_oracle_rejections_change_no_byte(case):
    what, descs, blob, idx = case
    b = oracle_backend()
    b.set_textures(descs, blob)
    with pytest.raises(R3Error) as e:
        b.generate_mipmaps(np.asarray(idx, dtype=np.uint32))
    assert e.value.code == -1, what
    assert np.array_equal(b.readback_texels(0, len(blob)), blob), what


def test_oracle_readback_range_is_checked():
    descs, blob = make_table([(L.TEXFMT_R8_UNORM, 4, 4, 1)], np.random.default_rng(7))
    b = oracle_backend()
    b.set_textures(descs, blob)
    with pytest.raises(R3Error):
        b.readback_texels(len(blob) - 4, 8)


# ------------------------------------------------------------------ 4. the harness
def test_texture_device_mips_descriptors():
    from rend3_b200.world import Renderer, Texture

    r = Renderer()
    img = np.random.default_rng(8).integers(0, 256, (75, 100, 4), dtype=np.uint8)
    a = r.add_texture_2d(Texture(img, srgb=True))                     # host box filter: unchanged
    b = r.add_texture_2d(Texture(img, srgb=True, mips="device"))
    c = r.add_texture_2d(Texture(img[..., :1].copy(), channels=1, mips="device"))
    d = r.add_texture_2d(Texture(img, storage="rgba16f", mips="device"))
    descs, blob = r._texture_table()
    assert descs[a]["mip_count"] == descs[b]["mip_count"] == 7 == max_mips(100, 75)
    for i, fmt in ((b, L.TEXFMT_RGBA8_UNORM_SRGB), (c, L.TEXFMT_R8_UNORM), (d, L.TEXFMT_RGBA16_FLOAT)):
        assert descs[i]["format"] == fmt and descs[i]["width"] == 100 and descs[i]["height"] == 75
        n0 = 100 * 75 * FORMATS[fmt][0]
        o = int(descs[i]["byte_offset"])
        assert not blob[o + n0: o + chain_bytes(fmt, 100, 75, 7)].any(), "the generated chain starts zeroed"
    o = int(descs[b]["byte_offset"])
    assert np.array_equal(blob[o: o + 100 * 75 * 4], img.reshape(-1))
    assert int(descs[b + 1]["byte_offset"]) >= o + chain_bytes(L.TEXFMT_RGBA8_UNORM_SRGB, 100, 75, 7)
    assert list(r.evaluate().generated_textures) == [b, c, d]


def test_scene_lists_generated_textures():
    from rend3_b200.scenes import textured_cube_scene

    ev = textured_cube_scene(n_objects=8, texture_size=27, device_mips=True)
    assert len(ev.generated_textures) == 7
    for i in ev.generated_textures:
        assert ev.texture_descs[i]["mip_count"] == max_mips(27, 27)
    assert len(textured_cube_scene(n_objects=8).generated_textures) == 0


# ------------------------------------------------------------------ 5. build
def test_mip_kernels_do_not_spill():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([nvcc, "-x", "cu", "-c", os.path.join(ROOT, "rend3_b200", "csrc", "r3_mipmap.cu"), "-o", os.path.join(tmp, "m.o"), "-std=c++17", "-O3",
                            "-gencode", "arch=compute_100a,code=sm_100a", "-prec-div=true", "-fmad=false", "-Xptxas", "-v"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    props = re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    kernels = {name: (int(a), int(b), int(c)) for name, a, b, c in props if "mip_" in name and "_kernel" in name}
    assert len(kernels) == 3, kernels
    assert all(v == (0, 0, 0) for v in kernels.values()), kernels


# ------------------------------------------------------------------ GPU
SHAPES = [(1, 1), (1, 1000), (333, 1), (256, 256), (255, 129), (640, 480), (3000, 17), (4096, 4096)]


@pytest.fixture()
def cuda():
    b = load_cuda_backend(0)
    yield b
    b.close()


@pytest.mark.gpu
def test_cuda_bit_exact_against_the_oracle_every_format_and_shape(cuda):
    import oracle

    oracle.set_threads(os.cpu_count() or 1)
    specs = [(fmt, w, h, max_mips(w, h)) for fmt in sorted(FORMATS) for (w, h) in SHAPES]
    descs, blob = make_table(specs, np.random.default_rng(9))
    order = list(np.random.default_rng(10).permutation(len(specs)))
    got = run(cuda, descs, blob, order)
    want = run(oracle_backend(), descs, blob, order)
    for i, (fmt, w, h, mips) in enumerate(specs):
        o, n = int(descs[i]["byte_offset"]), chain_bytes(fmt, w, h, mips)
        assert np.array_equal(got[o: o + n], want[o: o + n]), f"format {fmt} {w}x{h}: generated levels differ from the oracle"
        n0 = w * h * FORMATS[fmt][0]
        assert np.array_equal(got[o: o + n0], blob[o: o + n0])
    assert np.array_equal(got, want), "bytes outside the chains differ"


@pytest.mark.gpu
def test_cuda_launch_count_does_not_grow_with_textures(cuda):
    counts = []
    for n in (1, 64):
        descs, blob = make_table([(L.TEXFMT_RGBA8_UNORM_SRGB, 1000, 750, max_mips(1000, 750))] * n, np.random.default_rng(11), gap=0)
        cuda.set_textures(descs, blob)
        before = cuda.launch_count()
        cuda.generate_mipmaps(np.arange(n, dtype=np.uint32))
        cuda.sync()
        counts.append(cuda.launch_count() - before)
    assert counts[0] == counts[1] and 2 <= counts[0] <= 8, counts


@pytest.mark.gpu
def test_cuda_inside_a_recorded_frame_matches_an_eager_call(cuda):
    specs = [(fmt, 640, 480, max_mips(640, 480)) for fmt in sorted(FORMATS)] + [(L.TEXFMT_RGBA8_UNORM, 3000, 17, 12)]
    descs, blob = make_table(specs, np.random.default_rng(12))
    eager = run(cuda, descs, blob, range(len(specs)))
    for b in (cuda, load_cuda_backend(0)):        # the same work list again (cached on the device), and a fresh context (pinned upload)
        b.set_textures(descs, blob)
        b.frame_begin()
        b.generate_mipmaps(np.arange(len(specs), dtype=np.uint32))
        b.frame_end()
        assert b.frame_graph_stats()["graphed"] >= 1
        assert np.array_equal(b.readback_texels(0, len(blob)), eager)


def _hdr_close(a, b):
    err = np.abs(a.astype(np.float64) - b.astype(np.float64)) / np.maximum(1.0, np.abs(b.astype(np.float64)))
    assert np.nanmax(err) <= TOL, f"pixels differ by {np.nanmax(err):.3e}"


@pytest.mark.gpu
def test_device_mips_scene_renders_like_the_oracle(cuda):
    from rend3_b200.routines import BaseRenderGraph, BaseRenderGraphSettings
    from rend3_b200.scenes import textured_cube_scene

    res = (320, 180)
    settings = BaseRenderGraphSettings(clear_color=(0.1, 0.05, 0.1, 1.0))
    out = {}
    for name, b, dev in (("cuda", cuda, True), ("oracle", oracle_backend(), True), ("box", load_cuda_backend(0), False)):
        ev = textured_cube_scene(n_objects=300, seed=41, resolution=res, texture_size=27, device_mips=dev)
        BaseRenderGraph(b).add_to_graph(ev, res, 1, settings)
        w, h = ev.shadow_target_size
        out[name] = (b.readback_hdr_f32().copy(), b.readback_depth().copy(), b.readback_shadow_atlas(w, h).copy())
    (hc, dc, ac), (ho, do, ao), (hb, _, _) = out["cuda"], out["oracle"], out["box"]
    assert np.array_equal(dc.view(np.uint32), do.view(np.uint32)), "depth differs from the oracle"
    assert np.array_equal(ac.view(np.uint32), ao.view(np.uint32)), "shadow atlas differs from the oracle"
    _hdr_close(hc, ho)
    assert np.abs(hc.astype(np.float64) - hb).max() > 1e-3, "the generated levels are not what the image samples"


@pytest.mark.gpu
def test_cpp_host_mirror_generates_mipmaps(tmp_path):
    from rend3_b200.routines import BaseRenderGraph, BaseRenderGraphSettings
    from rend3_b200.scene_io import dump_scene, load_outputs
    from rend3_b200.scenes import textured_cube_scene

    res = (256, 144)
    ev = textured_cube_scene(n_objects=200, seed=43, resolution=res, texture_size=27, device_mips=True)
    settings = BaseRenderGraphSettings(clear_color=(0.1, 0.2, 0.3, 1.0))
    scene, out = tmp_path / "scene.r3s", tmp_path / "out.r3o"
    dump_scene(str(scene), ev, res, 1, settings, True)
    r = subprocess.run([os.path.join(ROOT, "rend3_b200", "host", "r3_frame"), str(scene), str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = load_outputs(str(out))
    orc = oracle_backend()
    BaseRenderGraph(orc).add_to_graph(ev, res, 1, settings)
    assert np.array_equal(got["depth"].view(np.uint32), orc.readback_depth().reshape(-1).view(np.uint32))
    _hdr_close(got["hdr"], orc.readback_hdr_f32().reshape(-1))


@pytest.mark.gpu
@pytest.mark.parametrize("case", REJECTIONS, ids=[c[0] for c in REJECTIONS])
def test_cuda_rejections_change_no_byte(cuda, case):
    what, descs, blob, idx = case
    cuda.set_textures(descs, blob)
    with pytest.raises(R3Error) as e:
        cuda.generate_mipmaps(np.asarray(idx, dtype=np.uint32))
    assert e.value.code == -1, what
    assert np.array_equal(cuda.readback_texels(0, len(blob)), blob), what


@pytest.mark.gpu
def test_cuda_mipmaps_are_one_timed_stage(cuda):
    descs, blob = make_table([(L.TEXFMT_RGBA8_UNORM_SRGB, 1000, 750, max_mips(1000, 750))] * 4, np.random.default_rng(13))
    cuda.set_textures(descs, blob)
    cuda.set_stage_timing(True)
    for _ in range(3):
        cuda.generate_mipmaps(np.arange(4, dtype=np.uint32))
    st = cuda.mipmap_stage_time()
    cuda.set_stage_timing(False)
    assert st["launches"] == 3 and st["ms"] > 0.0, st


@pytest.mark.gpu
def test_cuda_recorded_frames_with_changing_lists(cuda):
    """Work lists that change from one recorded frame to the next go through the pinned staging arena; every frame's chains are right."""
    specs = [(fmt, 300 + 37 * k, 200 + 11 * k, max_mips(300 + 37 * k, 200 + 11 * k)) for k, fmt in enumerate(sorted(FORMATS))]
    descs, blob = make_table(specs, np.random.default_rng(14))
    want = run(oracle_backend(), descs, blob, range(len(specs)))
    cuda.set_textures(descs, blob)
    for k in range(len(specs)):
        cuda.frame_begin()
        cuda.generate_mipmaps(np.array([k], dtype=np.uint32))
        cuda.frame_end()
    assert cuda.frame_graph_stats()["graphed"] == len(specs)
    assert np.array_equal(cuda.readback_texels(0, len(blob)), want)
