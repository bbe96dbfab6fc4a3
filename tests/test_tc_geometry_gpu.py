"""The tcgen05 conv kernels (csrc/tc_conv.cu) on every tile geometry the bf16 chain planner can send them, against fp64
on bf16-rounded operands.

The chain routes a k4 s2 p1 stage to these kernels on geometry alone (``chain._tc_ok`` / ``chain._thin_ok``): a small
map of p x q with p and q powers of two, q <= 128 (forward and input gradient) or q <= 64 (weight gradient), any batch.
A tile of 128 (64 for the weight gradients) pixels is Tw = q columns x Th rows x Tb images, and the kernels use p, q,
Tw, Th, Tb and tiles_y = p / Th as separate quantities: in the pixel-major epilogue's row_info, the producer's b0 / y0,
the channel-major epilogue's rel() and valid-column prefix, the TMA boxes of map_big_s2d / map_small / map_thin and the
thin input gradient's 4-row tiles.  The older tests all use square maps, where swapping p and q, Tw and Th or OH and OW
goes unnoticed; this file uses non-square maps throughout.

GEOMETRY names, for each kernel entry point, the shapes (n, c, p, q, k) -- c channels of the big map (2p x 2q), k of
the small map -- with the test hook each runs under and the regime it must take.  The *_regime helpers restate the C
launch plans (pick_tile, pick_cfg with the EADGAN_TC_CG hook, fprop_plan, dgrad_plan and thin_fprop_plan with the
EADGAN_TC_DGRADT hook, wgrad_plan, thin_wgrad_plan), which also take the SM count as an argument.  test_geometry_table (no GPU) checks every entry at the B200's 148 SMs, and every GPU test asserts that
its shape still takes its regime on the device it runs on.

What each shape checks, against fp64 on the same bf16 operands (tolerances of tests/test_tc_gpu.py: 2e-3 for fp32
outputs and statistics, 1e-2 for bf16 outputs):
  tc fprop / tc dgrad / thin fprop: bias + LeakyReLU + 1/sigma (fp32 NCHW where the entry is pixel-major, padded NHWC
    bf16 with a zero halo), bias with the BatchNorm statistics (sum, sum of squares), the fused activation backward
    (mask) of a Tanh producer with the per-channel sums of the result (stats_mode 2), and of a LeakyReLU producer;
  tc wgrad / thin wgrad: dw, bitwise identical on a second run;
  thin dgrad: bias + Tanh + 1/sigma into the fp32 NCHW image.
Every stored output is also written once into a buffer with guard bands (tests/test_guard_gpu.py): nothing in front,
behind or in the halo may change, and the interior must equal the unguarded launch bit for bit.

CHAIN runs a few non-square stacks through the chain executor against the fp64 referee of tests/test_chain_stages_gpu.py
at its bounds; it adds geometry, not plan rows, so it is not part of that file's STAGES."""
import pytest
import torch
import torch.nn.functional as TF

from conftest import rel_err

B200_SMS = 148
SIGMA = 1.25
SLOPE = 0.1


def _cdiv(a, b):
    return -(-a // b)


def _pow2(v):
    return v > 0 and v & (v - 1) == 0


# ---- regime selection, restated from csrc/tc_conv.cu ----------------------------------------------------------------
def pick_tile(p, q, pixels):
    """-> (Tw, Th, Tb): q columns, as many rows as fit (at most p), then whole images"""
    assert _pow2(p) and _pow2(q) and q <= pixels, (p, q, pixels)
    th = min(pixels // q, p)
    return q, th, pixels // (q * th)


def pick_bn_tiles(nch, m_tiles_x_par, sms):
    if nch % 256 == 0 and m_tiles_x_par * (nch // 256) >= 2 * sms:
        return 256
    return next(bn for bn in (128, 64, 32) if nch % bn == 0)


def pick_cfg(nch, m_tiles, parities, allow_pair, sms, env, force_bn=0):
    """-> (BLOCK_N, MT, cta_group)"""
    bn = force_bn or pick_bn_tiles(nch, m_tiles * parities, sms)
    tiles = m_tiles * parities * (nch // bn)
    cg = 2 if allow_pair and bn >= 128 and m_tiles >= 2 and tiles >= 2 * sms else 1
    if env.get("EADGAN_TC_CG") in ("1", "2") and allow_pair and bn >= 128:
        cg = int(env["EADGAN_TC_CG"])
    mt = 2 if bn <= 128 and tiles >= 4 * sms * cg else 1
    return bn, mt, cg


def _tile(n, p, q, pixels):
    tw, th, tb = pick_tile(p, q, pixels)
    return (tw, th, tb, p // th), _cdiv(n, tb) * (p // th)


def _tile_str(t):
    return "tile %dx%dx%d ty%d" % t


def tc_fprop_regime(shape, sms, env):
    n, c, p, q, k = shape
    t, m_tiles = _tile(n, p, q, 128)
    bn, mt, cg = pick_cfg(k, m_tiles, 1, True, sms, env)
    return f"{_tile_str(t)} bn{bn} mt{mt} cg{cg} qb{2 * c // 64}"


def tc_dgrad_regime(shape, sms, env):
    """padded NHWC output (the channel-major kernel never writes fp32 NCHW)"""
    n, c, p, q, k = shape
    t, m_tiles = _tile(n, p, q, 128)
    transposed = c == 128 and k % 64 == 0
    enough = m_tiles * 4 >= 8 * sms
    if env.get("EADGAN_TC_DGRADT") == "0":
        transposed = False
    elif env.get("EADGAN_TC_DGRADT") == "2":
        enough = True
    if transposed and enough:
        return f"{_tile_str(t)} channel-major m{m_tiles} qb{_cdiv(k, 64)}"
    bn, mt, cg = pick_cfg(c, m_tiles, 4, True, sms, env)
    return f"{_tile_str(t)} bn{bn} mt{mt} cg{cg} qb{_cdiv(k, 64)}"


def thin_fprop_regime(shape, sms, env):
    n, c, p, q, k = shape
    t, m_tiles = _tile(n, p, q, 128)
    bn = next(b for b in (128, 64, 32) if k % b == 0)
    major = k % 128 == 0 and m_tiles * (k // 128) >= 8 * sms
    if env.get("EADGAN_TC_DGRADT") == "0":
        major = False
    elif env.get("EADGAN_TC_DGRADT") == "2":
        major = k % 128 == 0
    if major:
        return f"{_tile_str(t)} channel-major m{m_tiles}"
    bn, mt, cg = pick_cfg(k, m_tiles, 1, False, sms, env, bn)
    return f"{_tile_str(t)} bn{bn} mt{mt} cg{cg}"


def _wgrad_splits(steps_total, tiles, bn, ktot, k, units):
    """wgrad_plan's split of the pixel reduction: the count minimising modelled MMA time plus partial-sum traffic"""
    k_pad = _cdiv(k, 128) * 128
    best, best_s = 1e300, 1
    for s in range(1, min(_cdiv(steps_total, 8), 4 * units) + 1):
        sps = _cdiv(steps_total, s)
        s_eff = _cdiv(steps_total, sps)
        waves = _cdiv(tiles * s_eff, units)
        t = waves * (sps * bn * 2.0 + 1500.0) / 1.9e9 / 0.9 + float(s_eff) * k_pad * ktot * 8.0 / 6.0e12
        if t < best:
            best, best_s = t, s_eff
    return _cdiv(steps_total, _cdiv(steps_total, best_s))


def tc_wgrad_regime(shape, sms, env):
    n, c, p, q, k = shape
    t, steps = _tile(n, p, q, 64)
    ktot = 16 * c
    bn = 256 if ktot % 256 == 0 else (128 if ktot % 128 == 0 else 64)
    cg = 2 if bn == 256 and k % 256 == 0 and steps >= 256 else 1
    if env.get("EADGAN_TC_CG") in ("1", "2") and bn == 256 and k % 256 == 0:
        cg = int(env["EADGAN_TC_CG"])
    tiles = (ktot // bn) * _cdiv(k, 128) // cg
    splits = _wgrad_splits(steps, tiles, bn, ktot, k, sms // cg)
    return f"{_tile_str(t)} bn{bn} cg{cg} qb{2 * c // 64} steps{steps} splits{splits}"


def thin_wgrad_regime(shape, sms, env):
    n, c, p, q, k = shape
    t, steps = _tile(n, p, q, 64)
    s = max(1, min(sms // _cdiv(k, 128), _cdiv(steps, 8)))
    return f"{_tile_str(t)} steps{steps} splits{_cdiv(steps, _cdiv(steps, s))}"


def thin_dgrad_regime(shape, sms, env):
    """one tile = 2 owned rows of one image (4 rows of the small map with its neighbours)"""
    n, c, p, q, k = shape
    assert q == 32 and p >= 2 and p % 2 == 0, (p, q)
    return f"tiles/img {p // 2} tiles {n * p // 2} kb{_cdiv(k, 64)}"


REGIME_OF = {"tc_fprop": tc_fprop_regime, "tc_dgrad": tc_dgrad_regime, "tc_wgrad": tc_wgrad_regime,
             "thin_fprop": thin_fprop_regime, "thin_wgrad": thin_wgrad_regime, "thin_dgrad": thin_dgrad_regime}

PM = {"EADGAN_TC_DGRADT": "0"}     # pixel-major dgrad / thin fprop
CM = {"EADGAN_TC_DGRADT": "2"}     # channel-major wherever the kernel applies
CG2 = {"EADGAN_TC_CG": "2"}        # CTA pairs wherever BLOCK_N >= 128
CG2_PM = {"EADGAN_TC_CG": "2", "EADGAN_TC_DGRADT": "0"}

# kernel -> [((n, c, p, q, k), test hooks, regime it must take, why)]
GEOMETRY = {
    "tc_fprop": [
        ((5, 64, 2, 16, 64), {}, "tile 16x2x4 ty1 bn64 mt1 cg1 qb2", "p < q, 4 images per tile, ragged batch"),
        ((3, 64, 16, 4, 128), {}, "tile 4x16x2 ty1 bn128 mt1 cg1 qb2", "p > q, 2 images per tile, ragged batch"),
        ((2, 32, 64, 8, 64), {}, "tile 8x16x1 ty4 bn64 mt1 cg1 qb1", "p > q, 4 tiles down each image"),
        ((5, 32, 32, 1, 64), {}, "tile 1x32x4 ty1 bn64 mt1 cg1 qb1", "q = 1: one column, 4 images per tile"),
        ((2, 32, 256, 1, 32), {}, "tile 1x128x1 ty2 bn32 mt1 cg1 qb1", "q = 1, 2 tiles down each image"),
        ((3, 64, 8, 2, 64), {}, "tile 2x8x8 ty1 bn64 mt1 cg1 qb2", "q = 2: 8 images per tile, 3 present"),
        ((6, 32, 1, 32, 64), {}, "tile 32x1x4 ty1 bn64 mt1 cg1 qb1", "p = 1: a single-row map"),
        ((2, 32, 4, 128, 64), {}, "tile 128x1x1 ty4 bn64 mt1 cg1 qb1", "q = 128, the widest: one map row per tile"),
        ((1, 64, 8, 32, 128), {}, "tile 32x4x1 ty2 bn128 mt1 cg1 qb2", "n = 1"),
        ((3, 128, 4, 32, 256), CG2, "tile 32x4x1 ty1 bn128 mt1 cg2 qb4",
         "CTA pairs on 3 M tiles: the peer of the second pair has no rows"),
        ((3, 96, 8, 16, 64), {}, "tile 16x8x1 ty1 bn64 mt1 cg1 qb3", "c = 96: 3 K blocks per tap, a box straddles dx"),
        ((600, 32, 4, 32, 64), {}, "tile 32x4x1 ty1 bn64 mt2 cg1 qb1", "two M tiles per CTA tile on a non-square map"),
    ],
    "tc_dgrad": [
        ((5, 64, 2, 16, 64), {}, "tile 16x2x4 ty1 bn64 mt1 cg1 qb1", "p < q, 4 images per tile, ragged batch"),
        ((3, 128, 16, 4, 64), PM, "tile 4x16x2 ty1 bn128 mt1 cg1 qb1", "p > q, 2 images per tile, ragged batch"),
        ((2, 32, 64, 8, 64), {}, "tile 8x16x1 ty4 bn32 mt1 cg1 qb1", "p > q, 4 tiles down each image"),
        ((5, 32, 32, 1, 64), {}, "tile 1x32x4 ty1 bn32 mt1 cg1 qb1", "q = 1: a 2-wide output"),
        ((2, 64, 256, 1, 32), {}, "tile 1x128x1 ty2 bn64 mt1 cg1 qb1", "q = 1, 2 tiles down each image, k = 32"),
        ((3, 64, 8, 2, 32), {}, "tile 2x8x8 ty1 bn64 mt1 cg1 qb1", "q = 2, k = 32: half of each channel box is zero"),
        ((6, 32, 1, 32, 64), {}, "tile 32x1x4 ty1 bn32 mt1 cg1 qb1", "p = 1: a 2-row output"),
        ((2, 64, 4, 128, 64), {}, "tile 128x1x1 ty4 bn64 mt1 cg1 qb1", "q = 128, the widest: one map row per tile"),
        ((1, 128, 8, 32, 128), PM, "tile 32x4x1 ty2 bn128 mt1 cg1 qb2", "n = 1"),
        ((3, 256, 4, 32, 128), CG2_PM, "tile 32x4x1 ty1 bn128 mt1 cg2 qb2",
         "CTA pairs on 3 M tiles x 4 parities"),
        ((3, 64, 8, 16, 192), {}, "tile 16x8x1 ty1 bn64 mt1 cg1 qb3", "k = 192: 3 K blocks per tap"),
        ((150, 64, 4, 32, 64), {}, "tile 32x4x1 ty1 bn64 mt2 cg1 qb1", "two M tiles per CTA tile on a non-square map"),
        # the channel-major kernel: two 128-pixel M tiles per tile, so an odd count leaves the second one empty
        ((3, 128, 4, 32, 64), CM, "tile 32x4x1 ty1 channel-major m3 qb1", "p < q, 3 M tiles"),
        ((1, 128, 32, 4, 64), CM, "tile 4x32x1 ty1 channel-major m1 qb1", "p > q, n = 1, 1 M tile"),
        ((1, 128, 64, 8, 64), CM, "tile 8x16x1 ty4 channel-major m4 qb1", "p > q, 4 tiles down the image"),
        ((5, 128, 2, 16, 64), CM, "tile 16x2x4 ty1 channel-major m2 qb1", "4 images per tile, ragged batch"),
        ((5, 128, 32, 1, 64), CM, "tile 1x32x4 ty1 channel-major m2 qb1", "q = 1"),
        ((3, 128, 8, 2, 128), CM, "tile 2x8x8 ty1 channel-major m1 qb2", "q = 2"),
        ((6, 128, 1, 32, 64), CM, "tile 32x1x4 ty1 channel-major m2 qb1", "p = 1"),
        ((1, 128, 2, 128, 64), CM, "tile 128x1x1 ty2 channel-major m2 qb1", "q = 128"),
        ((3, 128, 8, 16, 192), CM, "tile 16x8x1 ty1 channel-major m3 qb3", "k = 192, 3 M tiles"),
    ],
    "tc_wgrad": [
        ((5, 64, 2, 16, 64), {}, "tile 16x2x2 ty1 bn256 cg1 qb2 steps3 splits1", "p < q, 2 images per step"),
        ((2, 32, 64, 8, 64), {}, "tile 8x8x1 ty8 bn256 cg1 qb1 steps16 splits2", "p > q, 8 steps down each image"),
        ((5, 32, 32, 1, 64), {}, "tile 1x32x2 ty1 bn256 cg1 qb1 steps3 splits1", "q = 1"),
        ((2, 32, 256, 1, 32), {}, "tile 1x64x1 ty4 bn256 cg1 qb1 steps8 splits1", "q = 1, 4 steps down each image"),
        ((3, 64, 8, 2, 32), {}, "tile 2x8x4 ty1 bn256 cg1 qb2 steps1 splits1", "q = 2"),
        ((6, 32, 1, 32, 64), {}, "tile 32x1x2 ty1 bn256 cg1 qb1 steps3 splits1", "p = 1"),
        ((2, 32, 4, 64, 64), {}, "tile 64x1x1 ty4 bn256 cg1 qb1 steps8 splits1", "q = 64, the widest: one row per step"),
        ((1, 64, 16, 8, 128), {}, "tile 8x8x1 ty2 bn256 cg1 qb2 steps2 splits1", "n = 1"),
        ((3, 32, 8, 16, 256), CG2, "tile 16x4x1 ty2 bn256 cg2 qb1 steps6 splits1", "CTA pairs"),
        ((3, 96, 8, 16, 64), {}, "tile 16x4x1 ty2 bn256 cg1 qb3 steps6 splits1", "c = 96: 3 K blocks per tap"),
        ((37, 32, 16, 8, 64), {}, "tile 8x8x1 ty2 bn256 cg1 qb1 steps74 splits10", "split reduction, ragged last split"),
    ],
    "thin_fprop": [
        ((5, 3, 2, 16, 64), {}, "tile 16x2x4 ty1 bn64 mt1 cg1", "p < q, 4 images per tile, ragged batch"),
        ((2, 1, 64, 8, 32), {}, "tile 8x16x1 ty4 bn32 mt1 cg1", "p > q, 4 tiles down each image"),
        ((3, 2, 16, 4, 128), PM, "tile 4x16x2 ty1 bn128 mt1 cg1", "c = 2, p > q, 2 images per tile"),
        ((5, 3, 32, 1, 64), {}, "tile 1x32x4 ty1 bn64 mt1 cg1", "q = 1"),
        ((3, 2, 8, 2, 32), {}, "tile 2x8x8 ty1 bn32 mt1 cg1", "q = 2, c = 2"),
        ((6, 3, 1, 32, 64), {}, "tile 32x1x4 ty1 bn64 mt1 cg1", "p = 1"),
        ((2, 4, 4, 128, 64), {}, "tile 128x1x1 ty4 bn64 mt1 cg1", "q = 128, c = 4"),
        ((1, 3, 16, 8, 96), {}, "tile 8x16x1 ty1 bn32 mt1 cg1", "n = 1"),
        ((3, 3, 4, 32, 128), CM, "tile 32x4x1 ty1 channel-major m3", "p < q, 3 M tiles"),
        ((1, 2, 32, 4, 128), CM, "tile 4x32x1 ty1 channel-major m1", "p > q, n = 1, c = 2"),
        ((1, 3, 64, 8, 128), CM, "tile 8x16x1 ty4 channel-major m4", "4 tiles down the image"),
        ((5, 3, 2, 16, 128), CM, "tile 16x2x4 ty1 channel-major m2", "4 images per tile, ragged batch"),
        ((5, 4, 32, 1, 128), CM, "tile 1x32x4 ty1 channel-major m2", "q = 1, c = 4"),
        ((3, 1, 8, 2, 256), CM, "tile 2x8x8 ty1 channel-major m1", "q = 2, 2 channel blocks"),
        ((6, 3, 1, 32, 128), CM, "tile 32x1x4 ty1 channel-major m2", "p = 1"),
        ((1, 3, 2, 128, 128), CM, "tile 128x1x1 ty2 channel-major m2", "q = 128"),
    ],
    "thin_wgrad": [
        ((5, 3, 2, 16, 64), {}, "tile 16x2x2 ty1 steps3 splits1", "p < q, 2 images per step"),
        ((2, 1, 64, 8, 32), {}, "tile 8x8x1 ty8 steps16 splits2", "p > q, 8 steps down each image"),
        ((5, 3, 32, 1, 64), {}, "tile 1x32x2 ty1 steps3 splits1", "q = 1"),
        ((3, 2, 8, 2, 32), {}, "tile 2x8x4 ty1 steps1 splits1", "q = 2, c = 2"),
        ((6, 3, 1, 32, 64), {}, "tile 32x1x2 ty1 steps3 splits1", "p = 1"),
        ((2, 4, 4, 64, 64), {}, "tile 64x1x1 ty4 steps8 splits1", "q = 64, the widest, c = 4"),
        ((1, 3, 16, 8, 128), {}, "tile 8x8x1 ty2 steps2 splits1", "n = 1"),
        ((37, 2, 16, 8, 64), {}, "tile 8x8x1 ty2 steps74 splits10", "split reduction, ragged last split, c = 2"),
    ],
    "thin_dgrad": [
        ((5, 1, 2, 32, 32), {}, "tiles/img 1 tiles 5 kb1", "p = 2: one tile per image, c = 1, k = 32"),
        ((3, 2, 2, 32, 64), {}, "tiles/img 1 tiles 3 kb1", "p = 2, c = 2"),
        ((2, 3, 64, 32, 192), {}, "tiles/img 32 tiles 64 kb3", "p = 64 > q, k = 192"),
        ((1, 2, 8, 32, 64), {}, "tiles/img 4 tiles 4 kb1", "n = 1"),
        ((3, 3, 4, 32, 64), {}, "tiles/img 2 tiles 6 kb1", "p < q"),
        ((4, 1, 16, 32, 192), {}, "tiles/img 8 tiles 32 kb3", "c = 1, k = 192"),
    ],
}


def _cases(kernel):
    return [pytest.param(s, env, id="-".join(map(str, s)) + "".join(f"-{k[10:]}{v}" for k, v in sorted(env.items())))
            for s, env, _, _ in GEOMETRY[kernel]]


def _on_regime(kernel, shape, env, sms):
    want = next(r for s, e, r, _ in GEOMETRY[kernel] if s == shape and e == env)
    got = REGIME_OF[kernel](shape, sms, env)
    assert got == want, f"{kernel} {shape} {env} takes '{got}' at {sms} SMs, not '{want}'"


def test_geometry_table():
    """every table shape takes its named regime at the B200's SM count, and the table holds the geometries it is there
    for (no GPU needed)"""
    for kernel, entries in GEOMETRY.items():
        for shape, env, regime, _ in entries:
            assert REGIME_OF[kernel](shape, B200_SMS, env) == regime, (kernel, shape, REGIME_OF[kernel](shape, B200_SMS, env))
        ps, qs = {s[2] for s, _, _, _ in entries}, {s[3] for s, _, _, _ in entries}
        assert any(s[2] > s[3] for s, _, _, _ in entries) and any(s[2] < s[3] for s, _, _, _ in entries), kernel
        assert 1 in {s[0] for s, _, _, _ in entries}, kernel
        if kernel != "thin_dgrad":     # its guard: q == 32, p even
            assert {1, 2} <= qs and 1 in ps, kernel
            assert max(qs) == (64 if "wgrad" in kernel else 128), kernel
    # the channel-major kernels on an odd number of M tiles, CTA pairs, three K blocks per tap, thin dgrad extremes
    assert any("channel-major m3" in r for _, _, r, _ in GEOMETRY["tc_dgrad"])
    assert any("channel-major m3" in r for _, _, r, _ in GEOMETRY["thin_fprop"])
    for kernel in ("tc_fprop", "tc_dgrad", "tc_wgrad"):
        assert any("cg2" in r for _, _, r, _ in GEOMETRY[kernel]), kernel
        assert any("qb3" in r for _, _, r, _ in GEOMETRY[kernel]), kernel
    dg = [s for s, _, _, _ in GEOMETRY["thin_dgrad"]]
    assert {2, 64} <= {s[2] for s in dg} and {s[1] for s in dg} == {1, 2, 3} and {s[4] for s in dg} == {32, 64, 192}
    for kernel in ("thin_fprop", "thin_wgrad"):
        assert {2, 4} <= {s[1] for s, _, _, _ in GEOMETRY[kernel] if s[2] != s[3]}, kernel


# ---- chain stacks on non-square maps --------------------------------------------------------------------------------
# The two single-row plans the thin input gradient (2-row tiles) rejects: the image gradient of a thin conv on a 2-row
# image, and the forward of a ConvTranspose onto one (tests/test_cpu.py pins where the planner sends them).
P1_CONVT_LAST = ("p1_convT_last", [("convT", 64, 64, 3, 1, 1), ("relu",), ("convT", 64, 3, 4, 2, 1), ("tanh",)],
                 (4, 64, 1, 32))
P1_THIN_FIRST = ("p1_thin_first", [("conv", 3, 64, 4, 2, 1), ("lrelu", 0.2), ("conv", 64, 64, 3, 1, 1)], (4, 3, 2, 64))
CHAIN = [
    # CelebA-style discriminator trunk on a 32 x 128 image: thin first stage (16 x 64), BatchNorm stages down to 2 x 8
    ("celeba_D_wide", [("conv", 3, 64, 4, 2, 1), ("lrelu", 0.2), ("conv", 64, 128, 4, 2, 1, False), ("bn", 128),
                       ("lrelu", 0.2), ("conv", 128, 256, 4, 2, 1, False), ("bn", 256), ("lrelu", 0.2),
                       ("conv", 256, 32, 4, 2, 1)], (3, 3, 32, 128)),
    # generator growing from a 1 x 8 map to a 3-channel 8 x 64 image (thin ConvTranspose last on a 4 x 32 small map)
    ("G_from_1x8", [("convT", 64, 128, 4, 2, 1, False), ("bn", 128), ("relu",), ("convT", 128, 64, 4, 2, 1, False),
                    ("bn", 64), ("relu",), ("convT", 64, 3, 4, 2, 1), ("tanh",)], (3, 64, 1, 8)),
    # maps down to a single column (32 x 4 -> 16 x 2 -> 8 x 1) and a ConvTranspose back up from it
    ("down_to_q1", [("conv", 32, 64, 4, 2, 1), ("lrelu", 0.2), ("conv", 64, 128, 4, 2, 1), ("relu",),
                    ("convT", 128, 64, 4, 2, 1)], (5, 32, 32, 4)),
    P1_CONVT_LAST,
    P1_THIN_FIRST,
]


# ---- GPU tests ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sms(cuda):
    from eadgan_b200 import _lib
    return _lib.lib().eadgan_sm_count()


@pytest.fixture
def hooks(monkeypatch):
    def apply(env):
        for name in ("EADGAN_TC_CG", "EADGAN_TC_DGRADT"):
            monkeypatch.delenv(name, raising=False)
        for name, value in env.items():
            monkeypatch.setenv(name, value)
    return apply


def _bf(t):
    return t.bfloat16().float()


def _operands(shape, dev, seed, w_scale):
    """bf16-rounded big map x [n, c, 2p, 2q], small map y [n, k, p, q] and weight w [k, c, 4, 4]"""
    n, c, p, q, k = shape
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = _bf(torch.randn(n, c, 2 * p, 2 * q, generator=g)).to(dev)
    y = _bf(torch.randn(n, k, p, q, generator=g)).to(dev)
    w = _bf(torch.randn(k, c, 4, 4, generator=g) * w_scale).to(dev)
    bk, bc = torch.randn(k, generator=g).to(dev), torch.randn(c, generator=g).to(dev)
    return x, y, w, bk, bc


def _stored(launch, shape, dtype, dev, halo):
    """launch(None) into a fresh buffer, then launch(out) into one with guard bands: the guard bands (and a padded
    output's halo) must be untouched and the two results equal bit for bit -> the first result"""
    from test_guard_gpu import _check, _guarded
    first = launch(None).clone()
    if halo:
        assert float(first[:, 0].abs().max()) == 0 and float(first[:, -1].abs().max()) == 0, "halo rows not zero"
        assert float(first[:, :, 0].abs().max()) == 0 and float(first[:, :, -1].abs().max()) == 0, "halo columns not zero"
    big, out = _guarded(shape, dtype, dev)
    launch(out)
    _check(big, out, first, halo)
    return first


def _stats_errs(stats, pre, ch):
    return {"sum": rel_err(stats[:ch], pre.sum((0, 2, 3))), "sumsq": rel_err(stats[ch:], (pre * pre).sum((0, 2, 3)))}


def _sums_err(sums, ref):
    """per-channel sums against fp64, relative to the largest per-channel sum of |value| (test_tc_gpu._check_sums)"""
    return float((sums - ref.sum((0, 2, 3))).abs().max() / ref.abs().sum((0, 2, 3)).max())


def _assert_errs(kernel, shape, env, errs):
    """fp32 outputs and statistics <= 2e-3, bf16 outputs (keys starting with "bf16") <= 1e-2"""
    print(f"{kernel} {shape} {env}: " + " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v <= (1e-2 if k.startswith("bf16") else 2e-3)}
    assert not bad, (kernel, shape, env, bad)


def _epilogue_checks(dev, launch, pre_nobias, bias, out_ch, padded_shape, nchw_shape, f32):
    """the epilogue variants of a conv whose accumulator (/ sigma) is ``pre_nobias`` (fp64 NCHW):
    launch(bias, act, slope, mask, mask_mode, stats, stats_mode, sigma, out_f32, out) -> output tensor"""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU, ACT_NONE, ACT_TANH
    from test_tc_gpu import _act_grad_ref, _saved_output
    sigma = torch.tensor([SIGMA], device=dev)
    pre = pre_nobias / SIGMA + bias.double()[None, :, None, None]
    ref = TF.leaky_relu(pre, SLOPE)
    errs = {}
    if f32:
        out = _stored(lambda o: launch(bias, ACT_LRELU, SLOPE, None, 0, None, 1, sigma, True, o), nchw_shape,
                      torch.float32, dev, False)
        errs["f32"] = rel_err(out, ref)
    out = _stored(lambda o: launch(bias, ACT_LRELU, SLOPE, None, 0, None, 1, sigma, False, o), padded_shape,
                  torch.bfloat16, dev, True)
    errs["bf16"] = rel_err(tc.interior(out), ref)
    # BatchNorm statistics of the (pre-activation) output
    stats = torch.zeros(2 * out_ch, device=dev, dtype=torch.float64)
    out = launch(bias, ACT_NONE, 0.0, None, 0, stats, 1, sigma, False, None)
    errs["bf16_bn"] = rel_err(tc.interior(out), pre)
    errs.update(_stats_errs(stats, pre, out_ch))
    # fused activation backward of the producer (mask = its saved output), with and without the result's sums
    for name, mode, with_sums in (("tanh", ACT_TANH, True), ("lrelu", ACT_LRELU, False)):
        saved = _saved_output(name, nchw_shape, dev)
        ref_m = pre_nobias / SIGMA * _act_grad_ref(saved, name)
        mask = tc.to_padded(saved)
        sums = torch.zeros(out_ch, device=dev, dtype=torch.float64) if with_sums else None

        def masked(o):
            if sums is not None:
                sums.zero_()
            return launch(None, ACT_NONE, 0.2, mask, mode, sums, 2, sigma, False, o)
        out = _stored(masked, padded_shape, torch.bfloat16, dev, True)
        errs[f"bf16_mask_{name}"] = rel_err(tc.interior(out), ref_m)
        if sums is not None:
            errs["mask_sums"] = _sums_err(sums, ref_m)
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("shape,env", _cases("tc_fprop"))
def test_tc_fprop_geometry(cuda, sms, hooks, shape, env):
    from eadgan_b200 import tc
    hooks(env)
    _on_regime("tc_fprop", shape, env, sms)
    n, c, p, q, k = shape
    x, _, w, bk, _ = _operands(shape, cuda, 1, 0.05)
    xp, wpk = tc.to_padded(x), tc.pack_w(w, None, "fprop")

    def launch(bias, act, slope, mask, mode, stats, smode, sigma, f32, out):
        return tc.fprop(xp, wpk, bias, k, act, slope, out_f32_nchw=f32, mask=mask, mask_mode=mode, stats=stats,
                        stats_mode=smode, sigma=sigma, out=out)
    pre = TF.conv2d(x.double(), w.double(), None, stride=2, padding=1)
    errs = _epilogue_checks(cuda, launch, pre, bk, k, (n, p + 2, q + 2, k), (n, k, p, q), True)
    _assert_errs("tc_fprop", shape, env, errs)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,env", _cases("tc_dgrad"))
def test_tc_dgrad_geometry(cuda, sms, hooks, shape, env):
    from eadgan_b200 import tc
    hooks(env)
    _on_regime("tc_dgrad", shape, env, sms)
    n, c, p, q, k = shape
    _, y, w, _, bc = _operands(shape, cuda, 2, 0.05)
    yp, wpk = tc.to_padded(y), tc.pack_w(w, None, "dgrad")

    def launch(bias, act, slope, mask, mode, stats, smode, sigma, f32, out):
        return tc.dgrad(yp, wpk, bias, c, act, slope, out_f32_nchw=f32, mask=mask, mask_mode=mode, stats=stats,
                        stats_mode=smode, sigma=sigma, out=out)
    pre = TF.conv_transpose2d(y.double(), w.double(), None, stride=2, padding=1)
    # the fp32 NCHW epilogue only exists on the pixel-major kernel
    errs = _epilogue_checks(cuda, launch, pre, bc, c, (n, 2 * p + 2, 2 * q + 2, c), (n, c, 2 * p, 2 * q),
                            "channel-major" not in REGIME_OF["tc_dgrad"](shape, sms, env))
    _assert_errs("tc_dgrad", shape, env, errs)


def _wgrad_ref(x, y, c):
    return torch.nn.grad.conv2d_weight(x.double(), (y.shape[1], c, 4, 4), y.double(), stride=2, padding=1)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,env", _cases("tc_wgrad"))
def test_tc_wgrad_geometry(cuda, sms, hooks, shape, env):
    from eadgan_b200 import tc
    hooks(env)
    _on_regime("tc_wgrad", shape, env, sms)
    x, y, _, _, _ = _operands(shape, cuda, 3, 0.05)
    xp, yp = tc.to_padded(x), tc.to_padded(y)
    dw = tc.wgrad(xp, yp)
    assert torch.equal(dw, tc.wgrad(xp, yp)), "split partials must be summed in a fixed order"
    _assert_errs("tc_wgrad", shape, env, {"dw": rel_err(dw, _wgrad_ref(x, y, shape[1]))})


@pytest.mark.gpu
@pytest.mark.parametrize("shape,env", _cases("thin_fprop"))
def test_thin_fprop_geometry(cuda, sms, hooks, shape, env):
    from eadgan_b200 import tc
    hooks(env)
    _on_regime("thin_fprop", shape, env, sms)
    n, c, p, q, k = shape
    x, _, w, bk, _ = _operands(shape, cuda, 4, 0.1)
    r, wpk = tc.thin_expand(x), tc.thin_pack_w(w, "fprop")

    def launch(bias, act, slope, mask, mode, stats, smode, sigma, f32, out):
        assert not f32
        return tc.thin_fprop(r, wpk, bias, c, k, act, slope, mask=mask, mask_mode=mode, stats=stats, stats_mode=smode,
                             sigma=sigma, out=out)
    pre = TF.conv2d(x.double(), w.double(), None, stride=2, padding=1)
    errs = _epilogue_checks(cuda, launch, pre, bk, k, (n, p + 2, q + 2, k), (n, k, p, q), False)
    _assert_errs("thin_fprop", shape, env, errs)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,env", _cases("thin_wgrad"))
def test_thin_wgrad_geometry(cuda, sms, hooks, shape, env):
    from eadgan_b200 import tc
    hooks(env)
    _on_regime("thin_wgrad", shape, env, sms)
    c = shape[1]
    x, y, _, _, _ = _operands(shape, cuda, 5, 0.1)
    r, yp = tc.thin_expand(x), tc.to_padded(y)
    dw = tc.thin_wgrad(r, yp, c)
    assert torch.equal(dw, tc.thin_wgrad(r, yp, c)), "split partials must be summed in a fixed order"
    _assert_errs("thin_wgrad", shape, env, {"dw": rel_err(dw, _wgrad_ref(x, y, c))})


@pytest.mark.gpu
@pytest.mark.parametrize("shape,env", _cases("thin_dgrad"))
def test_thin_dgrad_geometry(cuda, sms, hooks, shape, env):
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_TANH
    hooks(env)
    _on_regime("thin_dgrad", shape, env, sms)
    n, c, p, q, k = shape
    _, y, w, _, bc = _operands(shape, cuda, 6, 0.1)
    yp, wpk = tc.to_padded(y), tc.thin_pack_w(w, "dgrad")
    sigma = torch.tensor([SIGMA], device=cuda)
    ref = torch.tanh(TF.conv_transpose2d(y.double(), w.double(), None, stride=2, padding=1) / SIGMA
                     + bc.double()[None, :, None, None])
    out = _stored(lambda o: tc.thin_dgrad(yp, wpk, bc, c, ACT_TANH, sigma=sigma, out=o), (n, c, 2 * p, 2 * q),
                  torch.float32, cuda, False)
    _assert_errs("thin_dgrad", shape, env, {"f32": rel_err(out, ref)})


@pytest.mark.gpu
@pytest.mark.parametrize("name,spec,shape", CHAIN, ids=[name for name, _, _ in CHAIN])
def test_chain_geometry_against_fp64_referee(cuda, name, spec, shape):
    """forward, every gradient and running statistic against tests/bf16_emul.py in fp64 on the chain's own gates; the
    frozen and no-input-gradient runs must repeat the full run"""
    from test_chain_stages_gpu import SAME_MAX, STAGE_MAX, run_entry
    errs, same = run_entry(spec, shape, cuda)
    print(f"chain {name}: worst {max(errs.values()):.2e}")
    bad = {k: v for k, v in errs.items() if not v <= STAGE_MAX}
    assert not bad, (name, bad)
    bad = {k: v for k, v in same.items() if not v <= SAME_MAX}
    assert not bad, (name, bad)
