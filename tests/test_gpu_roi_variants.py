"""Every RoIPool / RoIAlign kernel variant, at shapes that select it (148 SMs).

Each case names the kernel the dispatch must pick (frr_roi_variant) and fails, never skips, if the pick moves, so a change
to a heuristic cannot silently drop coverage.  Inputs carry the edges where these kernels go wrong: masked rois (index -1)
and rois with an index >= B, rois outside the map (empty bins), post-ReLU zero plateaus (argmax ties), windows of -inf,
NaN, -FLT_MAX and both signs of zero.  References:
  * RoIPool forward: the C oracle (torchvision CPU), out and argmax compared bitwise; the output without argmax must be
    bitwise the output with it (the 7x7 flat kernel may hold +0.0 for its -0.0); rows of masked rois must stay untouched.
  * backward (both ops) and the RoIAlign forward: a float64 restatement, checked per element against the fp32 rounding
    bound of that element's own terms, plus the fp32 oracle (1e-5) as before.
"""
import re
import zlib

import numpy as np
import pytest
import torch

from faster_rcnn_pytorch_b200 import _lib, ops, synth

DEV = "cuda:0"
f32 = np.float32
U = 2.0 ** -24       # unit roundoff of fp32
TINY = 1e-30         # below the scale of any nonzero term here
FLT_MAX = np.finfo(f32).max


# ------------------------------------------------------------------------------------------------
# the table: (name, B, C, H, W, K, output_size, spatial_scale, forward pick, backward pick, layouts)
# a pick is (kernel, channels per CTA, CTAs per (image, channel group))
# ------------------------------------------------------------------------------------------------
POOL_CASES = [
    # configs[2]: 500 rois per image (> 252 bin geometries per group, > 448 per list round), one CTA per image
    ("cfg2_cb8", 4, 512, 37, 62, 2000, (7, 7), 1.0, ("pool_fwd_flat", 8, 1), ("pool_bwd_color_tail", 8, 1), (False, True)),
    ("cb8_partial_group", 4, 300, 37, 62, 600, (7, 7), 1.0, ("pool_fwd_flat", 8, 1), ("pool_bwd_color_tail", 8, 1), (False, True)),
    # 75 x 80: 8 planes fit once per SM only (HW in [5977, 6652])
    ("cb8_one_per_sm", 2, 64, 75, 80, 300, (7, 7), 1.0, ("pool_fwd_flat", 8, 4), ("pool_bwd_tail", 0, 1), (False, True)),
    # configs[3]: 933 rois per image at one CTA per image, 2800 rois (> 2688: two scan rounds)
    ("cfg3_cb4", 3, 512, 50, 83, 2800, (7, 7), 1.0, ("pool_fwd_flat", 4, 1), ("pool_bwd_tail", 0, 1), (False,)),
    ("cfg0_cb4_z2", 1, 512, 37, 62, 300, (7, 7), 1.0, ("pool_fwd_flat", 4, 2), ("pool_bwd_color_tail", 8, 1), (False,)),
    ("cb4_z4", 1, 64, 37, 62, 300, (7, 7), 1.0, ("pool_fwd_flat", 4, 4), ("pool_bwd_color_tail", 8, 1), (True,)),
    ("planes_14x14", 2, 16, 37, 62, 200, (14, 14), 1.0, ("fwd_planes", 1, 1), ("bwd_planes", 1, 1), (False, True)),
    ("planes_3x5_img", 2, 160, 37, 62, 200, (3, 5), 1 / 16, ("fwd_planes", 2, 1), ("bwd_planes", 2, 1), (False,)),
    ("direct_14x14_img", 1, 8, 200, 336, 120, (14, 14), 1 / 16, ("fwd_direct", 0, 1), ("bwd_direct", 0, 1), (False, True)),
    # 7x7 bins on a plane too large for shared memory: generic forward, but the 7x7 backward still streams every roi
    ("direct_7x7_img", 1, 8, 200, 336, 120, (7, 7), 1 / 16, ("fwd_direct", 0, 1), ("pool_bwd_tail", 0, 1), (False,)),
    ("direct_3x5", 2, 4, 200, 336, 80, (3, 5), 1.0, ("fwd_direct", 0, 1), ("bwd_direct", 0, 1), (False,)),
]

# (name, B, C, H, W, K, spatial_scale, sampling_ratios, forward pick, backward pick, layouts); 7x7 bins.
# A sampling ratio other than 2 always takes the generic kernels, so the picks hold for ratio 2 and those cases list 2 only.
ALIGN_CASES = [
    ("fast_cb8", 2, 32, 37, 62, 200, 1.0, (2,), ("align_fwd_fast", 8, 1), ("align_bwd_fast", 4, 1), (False, True)),
    ("fast_cb4_two_per_sm", 2, 40, 50, 84, 200, 1.0, (2,), ("align_fwd_fast", 4, 1), ("align_bwd_stream", 0, 1), (False, True)),
    ("fast_cb8_one_per_sm", 2, 32, 78, 80, 150, 1.0, (2,), ("align_fwd_fast", 8, 1), ("align_bwd_stream", 0, 1), (False,)),
    ("fast_cb4_one_per_sm", 1, 16, 96, 128, 150, 1.0, (2,), ("align_fwd_fast", 4, 1), ("bwd_planes", 1, 1), (False, True)),
    # FPN level 3 / level 2 sized maps at full width: the separable backward with 16 and 8 planes per CTA
    ("bwd_cb16", 10, 240, 25, 42, 300, 0.5, (2,), ("align_fwd_fast", 8, 1), ("align_bwd_fast", 16, 1), (False,)),
    ("bwd_cb8", 4, 300, 25, 42, 200, 0.5, (2,), ("align_fwd_fast", 8, 1), ("align_bwd_fast", 8, 1), (True,)),
    # FPN level 1 of a COCO image: W = 168 > 128 columns, the plane does not fit the fast forward
    ("fpn1_planes", 2, 160, 100, 168, 100, 0.25, (2, 0, -1), ("fwd_planes", 2, 1), ("bwd_planes", 2, 1), (False, True)),
    ("adaptive_planes", 2, 32, 37, 62, 150, 1.0, (0, -1, 3), ("fwd_planes", 1, 1), ("bwd_planes", 1, 1), (False,)),
    ("direct", 1, 8, 200, 336, 60, 1.0, (2, 0, -1), ("fwd_direct", 0, 1), ("bwd_direct", 0, 1), (False, True)),
]

REACHABLE = {"pool_fwd_flat", "align_fwd_fast", "fwd_planes", "fwd_direct", "pool_bwd_color_tail", "pool_bwd_tail",
             "align_bwd_fast", "align_bwd_stream", "bwd_planes", "bwd_direct"}


def pick(op, K, B, C, H, W, output_size=(7, 7), sampling_ratio=2, want_argmax=True):
    v = ops.roi_variant(op, K, B, C, H, W, output_size, sampling_ratio, want_argmax)
    return v["kernel"], v["cb"], v["nz"]


def pool_picks(case):
    _, B, C, H, W, K, osz, _, _, _, _ = case
    return pick("roi_pool_fwd", K, B, C, H, W, osz), pick("roi_pool_bwd", K, B, C, H, W, osz)


def align_picks(case, sr):
    _, B, C, H, W, K, _, _, _, _, _ = case
    return pick("roi_align_fwd", K, B, C, H, W, (7, 7), sr), pick("roi_align_bwd", K, B, C, H, W, (7, 7), sr)


# ------------------------------------------------------------------------------------------------
# host checks of the table (no device needed: without one the dispatch assumes 148 SMs)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", POOL_CASES, ids=[c[0] for c in POOL_CASES])
def test_pool_case_selects_its_variant(case):
    assert pool_picks(case) == (case[8], case[9])


@pytest.mark.parametrize("case", ALIGN_CASES, ids=[c[0] for c in ALIGN_CASES])
def test_align_case_selects_its_variant(case):
    for sr in case[7]:
        want = (case[8], case[9]) if sr == 2 else None
        got = align_picks(case, sr)
        if want is not None:
            assert got == want, sr
        else:
            assert got[0][0] in ("fwd_planes", "fwd_direct") and got[1][0] in ("bwd_planes", "bwd_direct"), (sr, got)


def test_cases_cover_every_reachable_kernel():
    seen = set()
    for case in POOL_CASES:
        seen |= {p[0] for p in pool_picks(case)}
    for case in ALIGN_CASES:
        for sr in case[7]:
            seen |= {p[0] for p in align_picks(case, sr)}
    assert seen == REACHABLE, sorted(REACHABLE - seen)


def test_variant_query_edges():
    assert pick("roi_pool_fwd", 0, 2, 8, 37, 62)[0] == "none"                 # no rois: nothing launched
    assert pick("roi_pool_bwd", 0, 1, 4, 200, 336, (3, 5))[0] == "none"       # no rois, plane too large: memset only
    assert pick("roi_pool_bwd", 0, 1, 4, 37, 62, (3, 5))[0] == "bwd_planes"   # no rois: the planes kernel writes zeros
    with pytest.raises(ValueError):
        ops.roi_variant("roi_pool_fwd", 10, 0, 8, 37, 62)
    with pytest.raises(ValueError):
        _lib.check(_lib.load().frr_roi_variant(4, 10, 1, 8, 37, 62, 7, 7, 2, 1, (np.zeros(4, np.int32)).ctypes.data),
                   "frr_roi_variant")


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
N_SPECIAL = 10  # leading special rows of make_rois


def make_rois(seed, K, B, H, W, scale):
    """[K,5] rois in input coordinates (feature coordinates / scale), feature-map geometry:
    rows 0-9: index -1, index B, index B + 3, two rois outside the map, the -inf block, the mixed-sign zero block,
    the whole map, a sub-pixel roi, a roi crossing the top-left corner; then a quarter with integer corners and a rounded
    side of exactly 5, 6 or 7 pixels (the colour / tail split of the RoIPool backward), a quarter on x.5 (rounding
    boundaries once scaled), the rest random; 2 % of those masked."""
    rs = np.random.RandomState(seed)
    r = synth.random_rois(seed, K, H, W, B).astype(np.float64)
    rest = np.arange(N_SPECIAL, K)
    n = len(rest) // 4
    side = rs.choice([5, 6, 7], size=(n, 2))
    x1, y1 = rs.randint(0, W - 7, n), rs.randint(0, H - 7, n)
    r[rest[:n], 1:] = np.stack([x1, y1, x1 + side[:, 0] - 1, y1 + side[:, 1] - 1], axis=1)
    half = rest[n:2 * n]
    a = rs.randint(-1, W - 2, (len(half), 2)) + 0.5
    b = rs.randint(-1, H - 2, (len(half), 2)) + 0.5
    r[half, 1:] = np.stack([a.min(1), b.min(1), a.max(1) + 1, b.max(1) + 1], axis=1)
    r[rest, 0] = rs.randint(0, B, len(rest))
    r[rest[rs.rand(len(rest)) < 0.02], 0] = -1
    r[:N_SPECIAL, 0] = rs.randint(0, B, N_SPECIAL)
    r[0, 0], r[1, 0], r[2, 0] = -1, B, B + 3
    r[3, 1:] = [-60, -60, -50, -50]
    r[4, 1:] = [W + 20, H + 20, W + 40, H + 40]
    r[5, 1:] = [0, 0, 3, 3]              # the -inf block
    r[6, 1:] = [4, 4, 11, 11]            # the mixed-sign zero block
    r[7, 1:] = [0, 0, W - 1, H - 1]
    r[8, 1:] = [3.2, 3.2, 3.3, 3.4]
    r[9, 1:] = [-3.0, -2.0, 5.0, 4.0]
    r[:, 1:] /= scale
    return r.astype(f32)


def make_feat(seed, B, C, H, W, specials):
    """post-ReLU even channels (zero plateaus), zeros of both signs; with specials: -inf / NaN / -FLT_MAX sprinkled, an
    all -inf 4x4 block at the origin and an 8x8 block of mixed-sign zeros at (4, 4)"""
    rs = np.random.RandomState(seed)
    f = synth.features(seed, B, C, H, W)
    f[:, ::2] = np.maximum(f[:, ::2], 0.0)
    f[:, :, 4:12, 4:12] = 0.0
    f[(f == 0) & (rs.rand(*f.shape) < 0.5)] = -0.0
    if specials:
        m = rs.rand(*f.shape)
        f[m < 0.01] = -np.inf
        f[(m >= 0.01) & (m < 0.015)] = np.nan
        f[(m >= 0.015) & (m < 0.02)] = -FLT_MAX
        f[:, :, 0:4, 0:4] = -np.inf
    return f


def seed_of(name):
    return zlib.crc32(name.encode()) % 1000


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def bits(a):
    return np.ascontiguousarray(a, dtype=f32).view(np.uint32)


def within_bound(got, ref, n, s, what):
    """|got - ref| <= 2 (n + 2) u S per element: n = terms summed into the element, S = sum of their absolute values
    (each term carries up to three roundings of its own -- weight product, product with the gradient, division by the
    sample count -- and the fp32 sum n - 1 more)."""
    err = np.abs(got.astype(np.float64) - ref)
    bound = 2.0 * (n + 2) * U * s + TINY
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {int(bad.sum())} elements outside the bound, first at {np.argwhere(bad)[0]}: "
                           f"got {got[bad][0]!r} ref {ref[bad][0]!r} bound {bound[bad][0]!r}")


# ------------------------------------------------------------------------------------------------
# float64 references
# ------------------------------------------------------------------------------------------------
def align_taps(r, H, W, scale, PH, PW, sr, aligned):
    """torchvision's RoIAlign sampling restated with numpy: geometry and bilinear weights in fp32 (the same rounded
    operations), returned as (bin, pixel, weight / count in float64) for every tap of every valid sample."""
    off = f32(0.5) if aligned else f32(0.0)
    sc = f32(scale)
    sw, sh = f32(r[1]) * sc - off, f32(r[2]) * sc - off
    ew, eh = f32(r[3]) * sc - off, f32(r[4]) * sc - off
    rw, rh = ew - sw, eh - sh
    if not aligned:
        rw, rh = max(rw, f32(1.0)), max(rh, f32(1.0))
    bh, bw = rh / f32(PH), rw / f32(PW)
    gh = sr if sr > 0 else int(np.ceil(rh / f32(PH)))
    gw = sr if sr > 0 else int(np.ceil(rw / f32(PW)))
    count = max(gh * gw, 1)
    if gh <= 0 or gw <= 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0)

    def axis(start, bsz, P, g, size):
        p = np.repeat(np.arange(P), g).astype(f32)
        i = np.tile(np.arange(g), P).astype(f32)
        v = (start + p * bsz) + ((i + f32(0.5)) * bsz) / f32(g)
        ok = ~((v < f32(-1.0)) | (v > f32(size)))
        v = np.where(v <= 0, f32(0.0), v).astype(f32)
        lo = v.astype(np.int64)
        top = lo >= size - 1
        lo = np.where(top, size - 1, lo)
        hi = np.where(top, size - 1, lo + 1)
        v = np.where(top, lo.astype(f32), v)
        l = (v - lo.astype(f32)).astype(f32)
        return ok, lo, hi, l, (f32(1.0) - l).astype(f32)

    yok, ylo, yhi, ly, hy = axis(sh, bh, PH, gh, H)   # [PH * gh]
    xok, xlo, xhi, lx, hx = axis(sw, bw, PW, gw, W)   # [PW * gw]
    Y, X = np.meshgrid(np.arange(PH * gh), np.arange(PW * gw), indexing="ij")
    ok = (yok[Y] & xok[X]).ravel()
    Y, X = Y.ravel()[ok], X.ravel()[ok]
    binx = (Y // gh) * PW + (X // gw)
    pix = [ylo[Y] * W + xlo[X], ylo[Y] * W + xhi[X], yhi[Y] * W + xlo[X], yhi[Y] * W + xhi[X]]
    wts = [hy[Y] * hx[X], hy[Y] * lx[X], ly[Y] * hx[X], ly[Y] * lx[X]]   # fp32 products, as torchvision
    return (np.concatenate([binx] * 4), np.concatenate(pix),
            np.concatenate(wts).astype(np.float64) / count)


def align_ref64(feat, go, rois, scale, PH, PW, sr, aligned):
    """float64 RoIAlign forward and backward with per-element term counts and absolute sums (live rois only)."""
    B, C, H, W = feat.shape
    K = rois.shape[0]
    out = np.zeros((K, C, PH * PW)); out_n = np.zeros((K, 1, PH * PW)); out_s = np.zeros((K, C, PH * PW))
    gin = np.zeros((B, C, H * W)); gin_n = np.zeros((B, 1, H * W)); gin_s = np.zeros((B, C, H * W))
    f64 = feat.reshape(B, C, H * W).astype(np.float64)
    g64 = go.reshape(K, C, PH * PW).astype(np.float64)
    for k in range(K):
        b = int(rois[k, 0])
        if b < 0 or b >= B:
            continue
        binx, pix, w = align_taps(rois[k], H, W, scale, PH, PW, sr, aligned)
        if len(w) == 0:
            continue
        up, inv = np.unique(pix, return_inverse=True)
        M = np.zeros((PH * PW, len(up)))
        np.add.at(M, (binx, inv), w)
        fb = f64[b][:, up]
        out[k] = fb @ M.T
        out_s[k] = np.abs(fb) @ M.T
        out_n[k, 0] = np.bincount(binx, minlength=PH * PW)
        gin[b][:, up] += g64[k] @ M
        gin_s[b][:, up] += np.abs(g64[k]) @ M
        gin_n[b, 0, up] += np.bincount(inv, minlength=len(up))
    shp = (B, C, H, W)
    return ((out.reshape(go.shape), out_n.reshape(K, 1, PH, PW), out_s.reshape(go.shape)),
            (gin.reshape(shp), gin_n.reshape(B, 1, H, W), gin_s.reshape(shp)))


def pool_bwd_ref64(go, argmax, rois, shape):
    """grad_in[b, c, argmax] += grad_out in float64 over the given argmax (rois with an index outside [0, B) skipped),
    with per-element term counts and absolute sums."""
    B, C, H, W = shape
    K = rois.shape[0]
    bidx = rois[:, 0].astype(np.int64)
    live = (bidx >= 0) & (bidx < B)
    a = argmax.reshape(K, C, -1).astype(np.int64)
    g = go.reshape(K, C, -1).astype(np.float64)
    take = live[:, None, None] & (a >= 0)
    plane = (bidx[:, None, None] * C + np.arange(C)[None, :, None]) * (H * W)
    idx = (plane + a)[take]
    n = B * C * H * W
    ref = np.bincount(idx, weights=g[take], minlength=n).reshape(shape)
    cnt = np.bincount(idx, minlength=n).reshape(shape)
    s = np.bincount(idx, weights=np.abs(g[take]), minlength=n).reshape(shape)
    return ref, cnt, s


def close_accum(got, want):
    scale = max(float(np.abs(want).max()), 1e-30)
    assert float(np.abs(got - want).max()) <= 1e-5 * scale


# ------------------------------------------------------------------------------------------------
# raw ABI calls with NaN-filled outputs (rows of masked rois must stay untouched, as frr.h promises)
# ------------------------------------------------------------------------------------------------
def pool_fwd_abi(feat, rois, osz, scale, want_argmax):
    lib = _lib.load()
    f, cl = ops._feat_layout(feat)
    B, C, H, W = f.shape
    K = rois.shape[0]
    out = torch.full((K, C) + tuple(osz), float("nan"), device=DEV)
    arg = torch.full((K, C) + tuple(osz), -7, dtype=torch.int32, device=DEV) if want_argmax else None
    _lib.check(lib.frr_roi_pool_fwd(f.data_ptr(), rois.data_ptr(), K, B, C, H, W, osz[0], osz[1], float(scale), cl, None, 0,
                                    out.data_ptr(), arg.data_ptr() if want_argmax else None, ops._stream()),
               "frr_roi_pool_fwd")
    return out.cpu().numpy(), (arg.cpu().numpy() if want_argmax else None)


def layout(t, channels_last):
    return t.contiguous(memory_format=torch.channels_last) if channels_last else t


POOL_RUNS = [(c, cl) for c in POOL_CASES for cl in c[10]]
ALIGN_RUNS = [(c, sr, al, cl) for c in ALIGN_CASES for sr in c[7] for al in (False, True) for cl in c[10]
              if al is False or sr == 2]


@pytest.mark.gpu
@pytest.mark.parametrize("case,channels_last", POOL_RUNS, ids=[f"{c[0]}-{'nhwc' if cl else 'nchw'}" for c, cl in POOL_RUNS])
def test_roi_pool_variant_uniform(oracle, case, channels_last):
    name, B, C, H, W, K, osz, scale, want_fwd, want_bwd, _ = case
    assert pool_picks(case) == (want_fwd, want_bwd)
    feat = make_feat(seed_of(name) + 900, B, C, H, W, specials=True)
    rois = make_rois(seed_of(name) + 901, K, B, H, W, scale)
    go = np.random.RandomState(902).standard_normal((K, C) + tuple(osz)).astype(f32)
    live = (rois[:, 0] >= 0) & (rois[:, 0] < B)
    f = layout(dev(feat), channels_last)
    r = dev(rois)

    out, arg = pool_fwd_abi(f, r, osz, scale, True)
    wo, wa = oracle.roi_pool_forward(feat, rois[live], osz, scale)
    assert np.array_equal(bits(out[live]), bits(wo)), "max differs from torchvision (bitwise)"
    assert np.array_equal(arg[live], wa), "argmax differs from torchvision"
    assert np.isnan(out[~live]).all() and (arg[~live] == -7).all(), "rows of masked rois were written"
    out_na, _ = pool_fwd_abi(f, r, osz, scale, False)
    same = bits(out_na) == bits(out)
    if want_fwd[0] == "pool_fwd_flat":
        # its maximum without argmax is fmaxf: +0.0 may stand where the first strict maximum is -0.0 (frr.h)
        same |= (bits(out) == 0x80000000) & (bits(out_na) == 0)
    assert same.all(), "output without argmax differs from the output with it"

    gin = ops.roi_pool_backward(dev(go), dev(arg), r, feat.shape, spatial_scale=scale, channels_last=channels_last)
    got = gin.cpu().numpy()
    ref, n, s = pool_bwd_ref64(go, arg, rois, feat.shape)
    within_bound(got, ref, n, s, "roi_pool backward")
    close_accum(got, oracle.roi_pool_backward(go[live], wa, rois[live], feat.shape))


@pytest.mark.gpu
@pytest.mark.parametrize("case,sr,aligned,channels_last", ALIGN_RUNS,
                         ids=[f"{c[0]}-sr{sr}-{'aligned' if al else 'legacy'}-{'nhwc' if cl else 'nchw'}"
                              for c, sr, al, cl in ALIGN_RUNS])
def test_roi_align_variant(oracle, case, sr, aligned, channels_last):
    name, B, C, H, W, K, scale, _, want_fwd, want_bwd, _ = case
    fwd, bwd = align_picks(case, sr)
    if sr == 2:
        assert (fwd, bwd) == (want_fwd, want_bwd)
    else:
        assert fwd[0] in ("fwd_planes", "fwd_direct") and bwd[0] in ("bwd_planes", "bwd_direct")
    feat = make_feat(seed_of(name) + 950, B, C, H, W, specials=False)
    rois = make_rois(seed_of(name) + 951, K, B, H, W, scale)
    go = np.random.RandomState(952).standard_normal((K, C, 7, 7)).astype(f32)
    live = (rois[:, 0] >= 0) & (rois[:, 0] < B)
    f = layout(dev(feat), channels_last)
    r = dev(rois)

    out_t = torch.full((K, C, 7, 7), float("nan"), device=DEV)
    ops.roi_align_forward(f, r, (7, 7), scale, sr, aligned, out=out_t)
    out = out_t.cpu().numpy()
    assert np.isnan(out[~live]).all(), "rows of masked rois were written"
    want = oracle.roi_align_forward(feat, rois[live], (7, 7), scale, sr, aligned)
    np.testing.assert_allclose(out[live], want, rtol=1e-5, atol=1e-6)
    (o64, on, os_), (g64, gn, gs) = align_ref64(feat, go, rois, scale, 7, 7, sr, aligned)
    within_bound(out[live], o64[live], on[live], os_[live], "roi_align forward")

    gin = ops.roi_align_backward(dev(go), r, feat.shape, scale, sr, aligned, channels_last=channels_last)
    got = gin.cpu().numpy()
    within_bound(got, g64, gn, gs, "roi_align backward")
    close_accum(got, oracle.roi_align_backward(go[live], rois[live], feat.shape, (7, 7), scale, sr, aligned))


# ------------------------------------------------------------------------------------------------
# the query describes what launches
# ------------------------------------------------------------------------------------------------
KERNEL_NAMES = {
    "pool_fwd_flat": ["roi_pool_fwd_flat_kernel<{cb}"], "align_fwd_fast": ["roi_align_fwd_fast_kernel<{cb}"],
    "fwd_planes": ["roi_fwd_planes_kernel<"], "fwd_direct": ["roi_fwd_direct_kernel<"],
    "pool_bwd_color_tail": ["roi_pool_bwd_color_kernel<{cb}", "roi_pool_bwd_tail_kernel"],
    "pool_bwd_tail": ["roi_pool_bwd_tail_kernel"], "align_bwd_fast": ["roi_align_bwd_fast_kernel<{cb}"],
    "align_bwd_stream": ["roi_align_bwd_stream_kernel"], "bwd_planes": ["roi_bwd_planes_kernel<"],
    "bwd_direct": ["roi_bwd_direct_kernel<"],
}


def launched_roi_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return sorted(re.sub(r"\s+", "", re.sub(r"^void\s+", "", n)).replace("frr::", "") for n in names if "roi_" in n)


def expected_names(p):
    kernel, cb, _ = p
    return sorted(s.format(cb=cb) for s in KERNEL_NAMES[kernel])


@pytest.mark.gpu
def test_profiled_launches_match_the_query():
    """every pool case and every align case at sampling ratio 2 (a few rois each): the RoI kernels the profiler records
    are exactly the ones the query names, with the channels per CTA it names"""
    checked = set()
    for case in POOL_CASES:
        _, B, C, H, W, _, osz, scale, _, _, _ = case
        K = 64
        pf, pb = pick("roi_pool_fwd", K, B, C, H, W, osz), pick("roi_pool_bwd", K, B, C, H, W, osz)
        feat = dev(make_feat(1, B, C, H, W, specials=False))
        rois = dev(make_rois(2, K, B, H, W, scale))
        res = {}
        got = launched_roi_kernels(lambda: res.update(fa=ops.roi_pool_forward(feat, rois, osz, scale)))
        assert _match(got, expected_names(pf)), (case[0], got, pf)
        go = torch.ones((K, C) + tuple(osz), device=DEV)
        got = launched_roi_kernels(lambda: ops.roi_pool_backward(go, res["fa"][1], rois, (B, C, H, W), scale))
        assert _match(got, expected_names(pb)), (case[0], got, pb)
        checked |= {pf[0], pb[0]}
    for case in ALIGN_CASES:
        _, B, C, H, W, _, scale, _, _, _, _ = case
        K = 64
        pf, pb = pick("roi_align_fwd", K, B, C, H, W), pick("roi_align_bwd", K, B, C, H, W)
        feat = dev(make_feat(1, B, C, H, W, specials=False))
        rois = dev(make_rois(2, K, B, H, W, scale))
        got = launched_roi_kernels(lambda: ops.roi_align_forward(feat, rois, (7, 7), scale, 2))
        assert _match(got, expected_names(pf)), (case[0], got, pf)
        go = torch.ones((K, C, 7, 7), device=DEV)
        got = launched_roi_kernels(lambda: ops.roi_align_backward(go, rois, (B, C, H, W), scale, 2))
        assert _match(got, expected_names(pb)), (case[0], got, pb)
        checked |= {pf[0], pb[0]}
    assert checked == REACHABLE


def _match(got, want):
    """each expected name prefix is the prefix of exactly one recorded kernel, and nothing else was recorded"""
    if len(got) != len(want):
        return False
    return all(any(g.startswith(w) for g in got) for w in want)
