"""Parity of every CUDA kernel (through the C ABI) against the CPU oracle on identical seeded
inputs, plus the reference-generated golden fixtures.  Integer / byte outputs are bit-exact;
floating point carries the north_star tolerances written next to each assert."""
import numpy as np
import pytest
import torch

import pylc_oracle as orc

pytestmark = pytest.mark.gpu

STITCH_RTOL = 1e-5     # north_star: stitched probabilities within 1e-5 relative (fp32)
LOSS_RTOL = 1e-4       # north_star: loss values within 1e-4 relative
ARGMAX_MARGIN = 1e-6   # labels must agree wherever the reference's top-1 beats top-2 by more than this


@pytest.fixture(scope="module")
def ops():
    from pylc_b200 import ops as _ops
    _ops._lib.load()
    return _ops


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---------------------------------------------------------------------------------------------
# tile gather
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("H,W,ch,T,S", [
    (1100, 1300, 1, 512, 512), (1100, 1300, 3, 512, 512), (1536, 1024, 1, 512, 256), (1024, 1536, 3, 512, 256),
    (75, 101, 1, 32, 32), (80, 96, 3, 32, 16), (70, 200, 1, 64, 16), (512, 512, 3, 512, 512),
    (300, 300, 1, 512, 512),
])
def test_tile_gather(ops, H, W, ch, T, S, monkeypatch):
    img = orc.synth_image(3, W, H, ch)
    d, pitch = ops.upload_image(img)
    ref = orc.split_tiles(img, T, S)
    for no_tma in ("0", "1"):       # the switch must not change anything here (the image gathers are cp.async forms)
        monkeypatch.setenv("PYLC_NO_TMA", no_tma)
        tiles, stat = ops.tile_gather_u8(d, H, W, ch, pitch, T, S, stats=True)
        assert tuple(tiles.shape) == ref.shape
        assert np.array_equal(tiles.cpu().numpy(), ref)
        if ref.shape[0]:
            x = ref.astype(np.int64).reshape(ref.shape[0], ch, -1)
            want = np.stack([x.sum(-1), (x * x).sum(-1)], axis=-1)
            assert np.array_equal(stat.cpu().numpy(), want)
        plain = ops.tile_gather_u8(d, H, W, ch, pitch, T, S)          # the form without moments
        assert np.array_equal(plain.cpu().numpy(), ref)


def test_tile_gather_unaligned_source(ops):
    # contiguous rows of 1001 bytes: base/pitch not 16-byte aligned -> byte-wise path, same result
    img = orc.synth_image(4, 1001, 700, 1)
    d = dev(img)
    tiles = ops.tile_gather_u8(d, 700, 1001, 1, 1001, 512, 256)
    assert np.array_equal(tiles.cpu().numpy(), orc.split_tiles(img, 512, 256))
    img3 = orc.synth_image(5, 601, 600, 3)
    tiles = ops.tile_gather_u8(dev(img3), 600, 601, 3, 601 * 3, 512, 512)
    assert np.array_equal(tiles.cpu().numpy(), orc.split_tiles(img3, 512, 512))


def test_tile_gather_rejects_bad_geometry(ops):
    d, pitch = ops.upload_image(orc.synth_image(0, 640, 640, 1))
    with pytest.raises(ops.PylcError):
        ops.tile_gather_u8(d, 640, 640, 1, pitch, 500, 250)   # T % 16 != 0
    with pytest.raises(ops.PylcError):
        ops.tile_gather_u8(d, 640, 640, 1, pitch, 512, 384)   # T % S != 0


def test_split_golden(ops, golden):
    g = golden("split")
    for name in ("gray_s32", "gray_s16", "rgb_s32", "rgb_s16"):
        img = g["split_%s_img" % name]
        T, S = [int(v) for v in g["split_%s_TS" % name]]
        ch = 3 if img.ndim == 3 else 1
        d, pitch = ops.upload_image(img)
        tiles = ops.tile_gather_u8(d, img.shape[0], img.shape[1], ch, pitch, T, S)
        assert np.array_equal(tiles.cpu().numpy(), g["split_%s_tiles" % name])


@pytest.mark.parametrize("ch", [1, 3])
def test_gather_norm_bit_exact(ops, ch):
    H, W, T, S = 1024, 1536, 512, 256
    img = orc.synth_image(6, W, H, ch)
    mean = [127.3, 131.9, 120.1][:ch]
    std = [61.2, 58.7, 63.3][:ch]
    d, pitch = ops.upload_image(img)
    got = ops.tile_gather_norm_f32(d, H, W, ch, pitch, T, S, mean, std, 255.0, out_ch=3).cpu()
    tiles = torch.from_numpy(orc.split_tiles(img, T, S)).float()
    # models/model.py:434-445 in f32
    m = torch.tensor(mean, dtype=torch.float32)[None, :, None, None]
    s = torch.tensor(std, dtype=torch.float32)[None, :, None, None]
    want = ((tiles - m) / s) / 255
    if ch == 1:
        want = torch.cat((want, want, want), 1)   # models/model.py:376-377
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------
# mask gather + encode + histogram
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pk,H,W,T,S,skew", [
    ("a", 1100, 1300, 512, 512, False), ("b", 1100, 1300, 512, 512, True), ("a", 1024, 1536, 512, 256, True),
    ("b", 80, 96, 32, 16, False), ("a", 2000, 3000, 512, 512, True),
])
def test_mask_gather_encode_hist(ops, palettes, pk, H, W, T, S, skew):
    pal = palettes[pk]
    C = len(pal)
    mask = orc.synth_mask(7, W, H, pal, skew=skew, off_palette=0.002)
    d, pitch = ops.upload_image(mask)
    tiles, px_dist = ops.mask_gather_encode_hist(d, H, W, pitch, T, S, pal)
    ref = orc.class_encode(orc.split_tiles(mask, T, S), pal)
    assert np.array_equal(tiles.cpu().numpy(), ref)
    assert np.array_equal(px_dist.cpu().numpy(), orc.tile_histograms(ref, C))
    assert int(px_dist.sum()) == ref.size                       # utils/profile.py:125-126
    assert (ref == 1).sum() > 0


@pytest.mark.parametrize("pattern", ["noise", "uniform", "stripes3", "stripes4", "sparse", "pairs"])
@pytest.mark.parametrize("S,C", [(512, 9), (256, 9), (512, 20)])
def test_mask_gather_run_patterns(ops, palettes, pattern, S, C):
    """The TMA form encodes one pixel per 4-pixel group and re-encodes the groups whose 12 bytes are not
    one repeated pixel (palette_warp.cuh): masks built to hit every branch -- pure noise (dense
    fall-back), one colour (no fix-up), runs of 3 / 4 pixels (every / no group mixed), a few isolated
    off-palette pixels (queue path), pixels that differ from the group's anchor in ONE channel only."""
    rng = np.random.default_rng(11)
    pal = palettes["a"] if C == 9 else rng.integers(0, 256, size=(C, 3)).tolist()
    H, W, T = 1100, 1600, 512
    pal_a = np.asarray(pal, dtype=np.uint8)
    if pattern == "noise":
        lab = rng.integers(0, C, size=(H, W))
        mask = pal_a[lab]
        mask[rng.random((H, W)) < 0.3] = rng.integers(0, 256, size=3, dtype=np.uint8)
    elif pattern == "uniform":
        mask = np.broadcast_to(pal_a[C - 1], (H, W, 3)).copy()
    elif pattern in ("stripes3", "stripes4"):
        k = int(pattern[-1])
        mask = pal_a[(np.arange(W) // k + np.arange(H)[:, None]) % C]
    elif pattern == "sparse":
        mask = pal_a[orc.synth_labels(4, W, H, C, skew=False, block=200)]
        ys, xs = rng.integers(0, H, 300), rng.integers(0, W, 300)
        mask[ys, xs] = rng.integers(0, 256, size=(300, 3), dtype=np.uint8)
    else:   # pairs: neighbours equal in two channels, off by one in the third -> class 1 next to a palette colour
        mask = pal_a[orc.synth_labels(5, W, H, C, skew=False, block=64)]
        ch = rng.integers(0, 3, size=(H, W))
        hit = rng.random((H, W)) < 0.05
        for k in range(3):
            sel = hit & (ch == k)
            mask[..., k][sel] ^= 1
    mask = np.ascontiguousarray(mask)
    d, pitch = ops.upload_image(mask)
    tiles, px_dist = ops.mask_gather_encode_hist(d, H, W, pitch, T, S, pal)
    ref = orc.class_encode(orc.split_tiles(mask, T, S), pal)
    assert np.array_equal(tiles.cpu().numpy(), ref)
    assert np.array_equal(px_dist.cpu().numpy(), orc.tile_histograms(ref, C))


def test_mask_gather_wide_palette_duplicates_unaligned(ops):
    rng = np.random.default_rng(8)
    pal = rng.integers(0, 256, size=(20, 3)).tolist()
    pal[7] = pal[3]      # duplicate colour: the later index (7) wins
    mask = orc.synth_mask(9, 1001, 600, pal, off_palette=0.01)
    ref = orc.class_encode(orc.split_tiles(mask, 512, 512), pal)
    assert (ref == 7).any() and not (ref == 3).any()
    d, pitch = ops.upload_image(mask)
    tiles, px_dist = ops.mask_gather_encode_hist(d, 600, 1001, pitch, 512, 512, pal)
    assert np.array_equal(tiles.cpu().numpy(), ref)
    assert np.array_equal(px_dist.cpu().numpy(), orc.tile_histograms(ref, 20))
    # unpitched source -> byte-wise loads
    tiles2, px2 = ops.mask_gather_encode_hist(dev(mask), 600, 1001, 1001 * 3, 512, 512, pal)
    assert torch.equal(tiles, tiles2) and torch.equal(px_dist, px2)


@pytest.mark.parametrize("pk,n_img,H,W,T,S,ch", [
    ("b", 5, 1500, 2000, 512, 512, 1),     # configs[3]: gray image + schema_b mask pairs, one launch per stack (TMA form)
    ("a", 3, 1024, 1536, 512, 256, 3),     # 50 % overlap: a box goes to up to four tiles of its own image only
    ("b", 4, 80, 96, 32, 16, 1),           # small tiles: per-thread kernels, one launch per image inside the call
    ("a", 2, 600, 1001, 512, 512, 3),      # ragged width
    ("b", 1, 1100, 1300, 512, 512, 1),     # a stack of one
])
def test_extraction_stack_equals_per_image(ops, palettes, pk, n_img, H, W, T, S, ch, monkeypatch):
    """pylc_tile_gather_u8_stack / pylc_mask_gather_encode_hist_stack: the file loop of Extractor.extract
    (utils/extract.py:136-222) over equally sized pairs as one call -- tiles, moments and histograms in file
    order, bit-identical to the oracle and to per-image calls."""
    pal = palettes[pk]
    C = len(pal)
    imgs = [orc.synth_image(20 + i, W, H, ch) for i in range(n_img)]
    masks = [orc.synth_mask(20 + i, W, H, pal, skew=bool(i & 1), off_palette=0.002) for i in range(n_img)]
    d_imgs, ip, staging = ops.upload_stack(imgs)
    d_masks, mp, _ = ops.upload_stack(masks)
    assert tuple(d_imgs.shape) == (n_img, H, ip) and tuple(d_masks.shape) == (n_img, H, mp)
    tiles, stat = ops.tile_gather_u8_stack(d_imgs, H, W, ch, ip, T, S, stats=True)
    m_tiles, px_dist = ops.mask_gather_encode_hist_stack(d_masks, H, W, mp, T, S, pal)
    monkeypatch.setenv("PYLC_NO_TMA", "1")          # the per-thread / cp.async twins give the same bytes
    tiles_b, stat_b = ops.tile_gather_u8_stack(d_imgs, H, W, ch, ip, T, S, stats=True)
    m_tiles_b, px_dist_b = ops.mask_gather_encode_hist_stack(d_masks, H, W, mp, T, S, pal)
    monkeypatch.delenv("PYLC_NO_TMA")
    assert torch.equal(tiles, tiles_b) and torch.equal(stat, stat_b)
    assert torch.equal(m_tiles, m_tiles_b) and torch.equal(px_dist, px_dist_b)
    ref_i = np.concatenate([orc.split_tiles(im, T, S) for im in imgs])
    ref_m = np.concatenate([orc.class_encode(orc.split_tiles(m, T, S), pal) for m in masks])
    assert np.array_equal(tiles.cpu().numpy(), ref_i)
    assert np.array_equal(m_tiles.cpu().numpy(), ref_m)
    assert np.array_equal(px_dist.cpu().numpy(), orc.tile_histograms(ref_m, C))
    x = ref_i.astype(np.int64).reshape(ref_i.shape[0], ch, -1)
    assert np.array_equal(stat.cpu().numpy(), np.stack([x.sum(-1), (x * x).sum(-1)], axis=-1))
    # the same through the single-image entry points
    per = ref_i.shape[0] // n_img
    for i in range(n_img):
        t1, s1 = ops.tile_gather_u8(d_imgs[i], H, W, ch, ip, T, S, stats=True)
        m1, p1 = ops.mask_gather_encode_hist(d_masks[i], H, W, mp, T, S, pal)
        sl = slice(i * per, (i + 1) * per)
        assert torch.equal(t1, tiles[sl]) and torch.equal(s1, stat[sl])
        assert torch.equal(m1, m_tiles[sl]) and torch.equal(p1, px_dist[sl])
    # histograms accumulate into a caller's buffer; the tile-only form writes no histogram
    m2, p2 = ops.mask_gather_encode_hist_stack(d_masks, H, W, mp, T, S, pal, px_dist=px_dist.clone())
    assert torch.equal(p2, 2 * px_dist) and torch.equal(m2, m_tiles)
    m3, p3 = ops.mask_gather_encode_hist_stack(d_masks, H, W, mp, T, S, pal, hist=False)
    assert p3 is None and torch.equal(m3, m_tiles)


def test_extraction_stack_padded_image_stride(ops, palettes):
    """The image stride of a stack may exceed H * pitch (a pool with slack rows between images)."""
    pal = palettes["a"]
    H, W, T, S, n_img = 1024, 1024, 512, 256, 3
    masks = [orc.synth_mask(40 + i, W, H, pal) for i in range(n_img)]
    imgs = [orc.synth_image(40 + i, W, H, 3) for i in range(n_img)]
    pitch = ops.pitch_for(W * 3)
    pool_m = torch.full((n_img, H + 7, pitch), 255, dtype=torch.uint8, device="cuda")
    pool_i = torch.full((n_img, H + 7, pitch), 255, dtype=torch.uint8, device="cuda")
    for i in range(n_img):
        pool_m[i, :H, :W * 3] = dev(masks[i].reshape(H, W * 3))
        pool_i[i, :H, :W * 3] = dev(imgs[i].reshape(H, W * 3))
    lib = ops._lib.load()
    pal_c, C = ops._lib.palette_array(pal)
    n = 9 * n_img
    tiles = torch.empty((n, T, T), dtype=torch.uint8, device="cuda")
    px = torch.zeros((n, C), dtype=torch.int64, device="cuda")
    ops.check(lib.pylc_mask_gather_encode_hist_stack(ops._p(pool_m), n_img, (H + 7) * pitch, H, W, pitch, T, S, pal_c, C,
                                                     ops._p(tiles), ops._p(px), ops._stream()), "stack")
    ref_m = np.concatenate([orc.class_encode(orc.split_tiles(m, T, S), pal) for m in masks])
    assert np.array_equal(tiles.cpu().numpy(), ref_m)
    assert np.array_equal(px.cpu().numpy(), orc.tile_histograms(ref_m, C))
    it = torch.empty((n, 3, T, T), dtype=torch.uint8, device="cuda")
    ops.check(lib.pylc_tile_gather_u8_stack(ops._p(pool_i), n_img, (H + 7) * pitch, H, W, 3, pitch, T, S, ops._p(it), None,
                                            ops._stream()), "stack")
    assert np.array_equal(it.cpu().numpy(), np.concatenate([orc.split_tiles(im, T, S) for im in imgs]))
    # a stride shorter than one image is rejected
    with pytest.raises(ops.PylcError):
        ops.check(lib.pylc_tile_gather_u8_stack(ops._p(pool_i), n_img, H * pitch - 16, H, W, 3, pitch, T, S, ops._p(it), None,
                                                ops._stream()), "stack")


def test_extraction_stack_unaligned_rows(ops, palettes):
    """A stack whose rows are not 16-byte aligned (tightly packed 1001-pixel rows): the byte-wise per-thread kernels
    run once per image inside the one call; results as for aligned stacks."""
    pal = palettes["b"]
    H, W, T, S, n_img = 600, 1001, 512, 512, 3
    masks = np.stack([orc.synth_mask(60 + i, W, H, pal, off_palette=0.01) for i in range(n_img)])
    imgs = np.stack([orc.synth_image(60 + i, W, H, 1) for i in range(n_img)])
    d_m, d_i = dev(masks.reshape(n_img, H, W * 3)), dev(imgs.reshape(n_img, H, W))
    m_tiles, px_dist = ops.mask_gather_encode_hist_stack(d_m, H, W, W * 3, T, S, pal)
    tiles, stat = ops.tile_gather_u8_stack(d_i, H, W, 1, W, T, S, stats=True)
    ref_m = np.concatenate([orc.class_encode(orc.split_tiles(m, T, S), pal) for m in masks])
    ref_i = np.concatenate([orc.split_tiles(im, T, S) for im in imgs])
    assert np.array_equal(m_tiles.cpu().numpy(), ref_m) and np.array_equal(tiles.cpu().numpy(), ref_i)
    assert np.array_equal(px_dist.cpu().numpy(), orc.tile_histograms(ref_m, len(pal)))
    x = ref_i.astype(np.int64).reshape(ref_i.shape[0], 1, -1)
    assert np.array_equal(stat.cpu().numpy(), np.stack([x.sum(-1), (x * x).sum(-1)], axis=-1))


def test_class_encode_golden_and_layouts(ops, golden, palettes):
    g = golden("encode")
    for name in ("a", "b", "dup"):
        pal = g["palette_%s" % name].tolist()
        x = g["encode_%s_in" % name]
        out, hist = ops.class_encode_nchw(dev(x), pal, hist=True)
        assert np.array_equal(out.cpu().numpy(), g["encode_%s_out" % name])
        assert np.array_equal(hist.cpu().numpy(), np.bincount(g["encode_%s_out" % name].ravel(), minlength=len(pal)))
    pal = palettes["b"]
    for (h, w) in [(37, 53), (64, 48), (1500, 2000)]:
        mask = orc.synth_mask(h, w, h, pal, off_palette=0.01)
        want = orc.class_encode_hwc(mask, pal)
        # planar (the reference's NCHW argument), arbitrary size
        out = ops.class_encode_nchw(dev(np.moveaxis(mask, 2, 0)[None]), pal)
        assert np.array_equal(out.cpu().numpy()[0], want)
        # interleaved, pitched and unpitched
        d, pitch = ops.upload_image(mask)
        out, hist = ops.class_encode_hwc(d, h, w, pitch, pal, hist=True)
        assert np.array_equal(out.cpu().numpy()[0], want)
        assert np.array_equal(hist.cpu().numpy(), np.bincount(want.ravel(), minlength=len(pal)))
        out = ops.class_encode_hwc(dev(mask), h, w, w * 3, pal)
        assert np.array_equal(out.cpu().numpy()[0], want)


@pytest.mark.parametrize("rows,cols,n_img", [(45, 272, 1), (100, 1008, 1), (33, 16, 1), (70, 528, 3), (1500, 2000, 1), (64, 250, 1)])
@pytest.mark.parametrize("C", [9, 20])
def test_class_encode_hwc_box_edges(ops, palettes, rows, cols, n_img, C):
    """Interleaved class_encode through the TMA form (cols % 16 == 0: partial boxes on the right and bottom
    edges are zero-filled on load, clipped on store, and must not reach the histogram) and through the
    per-thread form (cols = 250); several images stacked as one tall image."""
    rng = np.random.default_rng(rows * 7 + cols)
    pal = palettes["a"] if C == 9 else rng.integers(0, 256, size=(C, 3)).tolist()
    imgs = [orc.synth_mask(40 + i, cols, rows, pal, skew=False, off_palette=0.01) for i in range(n_img)]
    stack = np.ascontiguousarray(np.concatenate(imgs, axis=0))
    d, pitch = ops.upload_image(stack)
    out, hist = ops.class_encode_hwc(d, rows, cols, pitch, pal, n_img=n_img, hist=True)
    ref = np.stack([orc.class_encode_hwc(im, pal) for im in imgs])
    assert np.array_equal(out.cpu().numpy(), ref)
    assert np.array_equal(hist.cpu().numpy(), np.bincount(ref.ravel(), minlength=C))
    out2 = ops.class_encode_hwc(d, rows, cols, pitch, pal, n_img=n_img)
    assert torch.equal(out, out2)


def test_class_encode_rejects_non_rgb(ops):
    with pytest.raises(ops.PylcError):   # utils/tools.py:433
        ops.class_encode_nchw(torch.zeros((1, 4, 8, 8), dtype=torch.uint8, device="cuda"), [[0, 0, 0]])


@pytest.mark.parametrize("ch,C,T", [(1, 9, 512), (3, 11, 512), (1, 20, 64), (3, 9, 32)])
def test_profile_tiles(ops, ch, C, T):
    rng = np.random.default_rng(10)
    n = 5
    imgs = rng.integers(0, 256, size=(n, ch, T, T), dtype=np.uint8)
    masks = rng.integers(0, C, size=(n, T, T), dtype=np.uint8)
    masks[0] = 0
    stat, px_dist = ops.profile_tiles(dev(imgs), dev(masks), C)
    assert np.array_equal(px_dist.cpu().numpy(), orc.tile_histograms(masks, C))
    x = imgs.astype(np.int64).reshape(n, ch, -1)
    assert np.array_equal(stat.cpu().numpy(), np.stack([x.sum(-1), (x * x).sum(-1)], axis=-1))


def test_extract_profile_golden(ops, golden, palettes):
    """extract + profile of the reference run in gen_golden.py, reproduced through the kernels."""
    g = golden("extract_profile")
    for name, ch, pk in (("gray_a", 1, "a"), ("rgb_b", 3, "b")):
        pal = palettes[pk]
        imgs, masks, dists = [], [], []
        for k in g["exprof_%s_order" % name]:
            img, mask = g["exprof_%s_img%d" % (name, k)], g["exprof_%s_mask%d" % (name, k)]
            d, p = ops.upload_image(img)
            imgs.append(ops.tile_gather_u8(d, img.shape[0], img.shape[1], ch, p, 32, 32))
            d, p = ops.upload_image(mask)
            t, pd = ops.mask_gather_encode_hist(d, mask.shape[0], mask.shape[1], p, 32, 32, pal)
            masks.append(t)
            dists.append(pd)
        assert np.array_equal(torch.cat(imgs).cpu().numpy(), g["exprof_%s_tiles_img" % name])
        assert np.array_equal(torch.cat(masks).cpu().numpy(), g["exprof_%s_tiles_mask" % name])
        assert np.array_equal(torch.cat(dists).cpu().numpy(), g["exprof_%s_px_dist" % name])


# ---------------------------------------------------------------------------------------------
# stitch + softmax + argmax + colourise
# ---------------------------------------------------------------------------------------------

def check_stitch(ops, tiles, nr, nc, T, S, pal, ref_map=None, batches=None):
    C = tiles.shape[1]
    lut = orc.colourize_lut(C, pal).tolist()
    if ref_map is None:
        ref_map = orc.stitch_map(tiles, nr, nc, T, S)
    if batches:
        src = [dev(tiles[i:i + batches]) for i in range(0, len(tiles), batches)]
    else:
        src = dev(tiles)
    labels, rgb, stitched = ops.stitch_argmax_colour(src, nr, nc, T, S, lut_rgb=lut, want_rgb=True, want_stitched=True)
    got = stitched.cpu().numpy()
    np.testing.assert_allclose(got, ref_map, rtol=STITCH_RTOL, atol=1e-7)
    lab = labels.cpu().numpy()
    # our labels are the exact first-argmax of our own map ...
    assert np.array_equal(lab, np.argmax(got, axis=0))
    # ... and agree with the reference wherever its top-1 is separated from top-2
    ref_lab = orc.stitch_labels(ref_map)
    margin = orc.top2_margin(ref_map)
    mism = lab != ref_lab
    assert not (mism & (margin > ARGMAX_MARGIN)).any(), "argmax mismatch above margin"
    assert np.array_equal(rgb.cpu().numpy(), np.asarray(lut, dtype=np.uint8)[lab])
    return int(mism.sum()), lab.size


@pytest.mark.parametrize("case", ["a_2x3", "a_3x2", "a_3x3", "a_2x1", "b_4x5", "a_s32_2x3"])
def test_stitch_golden(ops, golden, palettes, case):
    g = golden("reconstruct")
    nr, nc, T, S, h, w, w_full, h_full, C = [int(v) for v in g["recon_%s_geom" % case]]
    pal = palettes["b" if case.startswith("b") else "a"]
    tiles = orc.reconstruct_fixture_tiles(g, case)
    check_stitch(ops, tiles, nr, nc, T, S, pal, ref_map=g["recon_%s_map" % case])
    check_stitch(ops, tiles, nr, nc, T, S, pal, ref_map=g["recon_%s_map" % case], batches=4)
    # end of tools.reconstruct: NN-resample to (w_full, h_full) and colourise == reference RGB
    labels, _, _ = ops.stitch_argmax_colour(dev(tiles), nr, nc, T, S)
    res = ops.resample_encode_confusion(labels, w_full, h_full, lut_rgb=orc.colourize_lut(C, pal).tolist(), want_rgb=True)
    ref_rgb = g["recon_%s_rgb" % case]
    ours = res["pred_rgb"].cpu().numpy().astype(np.float32)
    ref_map = g["recon_%s_map" % case]
    near_tie = orc.resample_labels((orc.top2_margin(ref_map) <= ARGMAX_MARGIN).astype(np.uint8), w_full, h_full) > 0
    assert np.array_equal(ours[~near_tie], ref_rgb[~near_tie])


@pytest.mark.parametrize("C,nr,nc,T,S", [(9, 2, 3, 512, 256), (11, 3, 2, 512, 256), (9, 2, 2, 512, 512),
                                        (5, 3, 3, 64, 32), (12, 2, 2, 64, 32), (20, 2, 3, 64, 32), (2, 1, 1, 32, 16),
                                        (9, 3, 1, 32, 16), (16, 2, 2, 32, 32)])
def test_stitch_vs_oracle(ops, C, nr, nc, T, S):
    g = torch.Generator().manual_seed(C * 100 + nr * 10 + nc)
    tiles = (torch.randn(nr * nc, C, T, T, generator=g) * 3).numpy()
    pal = np.random.default_rng(C).integers(0, 256, size=(C, 3)).tolist()
    check_stitch(ops, tiles, nr, nc, T, S, pal)
    if nr * nc > 2:
        check_stitch(ops, tiles, nr, nc, T, S, pal, batches=2)


def test_stitch_exact_ties_pick_first_class(ops):
    # identical logits in every class: every softmax is uniform, np.argmax returns class 0
    tiles = np.zeros((4, 9, 32, 32), dtype=np.float32)
    labels, _, _ = ops.stitch_argmax_colour(dev(tiles), 2, 2, 32, 16)
    assert int(labels.max()) == 0
    tiles[:, 4] = 1.0
    labels, _, _ = ops.stitch_argmax_colour(dev(tiles), 2, 2, 32, 16)
    assert int(labels.min()) == 4 and int(labels.max()) == 4


def test_stitch_fitted_3000x2000(ops, palettes):
    """BASELINE config 2 geometry: 3000x2000 fits to 2560x1536 -> 5 x 9 tiles, C = 9."""
    nr, nc, T, S, C = 5, 9, 512, 256, 9
    g = torch.Generator().manual_seed(2)
    tiles = (torch.randn(nr * nc, C, T, T, generator=g) * 3).numpy()
    mism, total = check_stitch(ops, tiles, nr, nc, T, S, palettes["a"], batches=8)
    assert mism <= total * 1e-5


@pytest.mark.parametrize("C,nr,nc,T,S,tpb", [(9, 3, 5, 512, 256, 8), (11, 2, 2, 512, 256, 4), (5, 2, 3, 512, 512, 6),
                                             (12, 1, 2, 512, 256, 2), (9, 2, 2, 256, 128, 3)])
def test_stitch_fused_upsample_equals_two_kernel_route(ops, palettes, C, nr, nc, T, S, tpb):
    """SURVEY.md 8f-1: the stitch that reads the decoder's [b, T/4, T/4, C] channels-last output and evaluates
    the network's final x4 bilinear up-sample itself (models/architectures/deeplab.py:38) is BIT-identical to
    up-sample-to-logits followed by the stitch -- stitched map, labels and RGB -- and within the north-star
    tolerances of the reference sequence F.interpolate -> tools.reconstruct evaluated by the oracle."""
    n, hs = nr * nc, T // 4
    g = torch.Generator().manual_seed(C * 100 + n)
    dec_all = (torch.randn(n, C, hs, hs, generator=g) * 3).cuda().contiguous(memory_format=torch.channels_last)
    batches = [dec_all[i:i + tpb].contiguous(memory_format=torch.channels_last) for i in range(0, n, tpb)]
    lut = (palettes["a"] + palettes["b"])[:C]
    logits = [ops.upsample_nhwc_to_nchw(b, (T, T)) for b in batches]
    lab2, rgb2, map2 = ops.stitch_argmax_colour(logits if len(logits) > 1 else logits[0], nr, nc, T, S, lut_rgb=lut,
                                                want_rgb=True, want_stitched=True, tiles_per_batch=tpb)
    lab1, rgb1, map1 = ops.stitch_upsample_argmax_colour(batches, nr, nc, T, S, lut_rgb=lut, want_rgb=True,
                                                         want_stitched=True, tiles_per_batch=tpb)
    assert torch.equal(map1, map2)
    assert torch.equal(lab1, lab2) and torch.equal(rgb1, rgb2)
    # labels only (the pipeline's call)
    lab0, _, _ = ops.stitch_upsample_argmax_colour(batches, nr, nc, T, S, tiles_per_batch=tpb)
    assert torch.equal(lab0, lab1)
    if n * T * T <= 4 * 512 * 512 and S < T:
        up = torch.nn.functional.interpolate(dec_all.cpu().contiguous(), size=(T, T), mode="bilinear", align_corners=True)
        ref_map = orc.stitch_map(up.numpy(), nr, nc, T, S)
        np.testing.assert_allclose(map1.cpu().numpy(), ref_map, rtol=1e-5, atol=2e-6)
        bad = lab1.cpu().numpy() != orc.stitch_labels(ref_map)
        assert not (bad & (orc.top2_margin(ref_map) > 1e-5)).any()


def test_colourise(ops, golden, palettes):
    g = golden("colourize")
    for name in ("a", "b"):
        pal = palettes[name]
        lab = g["colourize_%s_in" % name].astype(np.uint8)
        lut = orc.colourize_lut(len(pal), pal).tolist()
        rgb = ops.colourise_u8(dev(lab), lut)
        assert np.array_equal(rgb.cpu().numpy().astype(np.int64), g["colourize_%s_out" % name])


# ---------------------------------------------------------------------------------------------
# test-time fit resize (cv2 INTER_AREA on the device)
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("W,H,T,ch", [(2000, 1500, 512, 1), (3000, 2000, 512, 3), (1300, 900, 256, 3), (1500, 1100, 512, 1),
                                      (1025, 2300, 512, 3), (6000, 4000, 512, 1), (2560, 1536, 512, 3)])
def test_fit_resize_area_bit_exact(ops, W, H, T, ch):
    """Device INTER_AREA == the installed OpenCV (what tools.adjust_to_tile calls), every byte; the
    source is uploaded unpitched and pitched."""
    import cv2
    w, h = orc.fit_dims(W, H, T)
    assert ops.area_supported(W, H, w, h)
    img = orc.synth_image(4, W, H, ch)
    img = (img.astype(np.int32) + np.random.default_rng(W).integers(-40, 40, size=img.shape)).clip(0, 255).astype(np.uint8)
    ref = cv2.resize(img, (w, h), interpolation=cv2.INTER_AREA).reshape(h, w * ch)
    got, pitch = ops.fit_resize_area(dev(img), H, W, ch, W * ch, h, w)
    assert np.array_equal(got.cpu().numpy()[:, :w * ch], ref)
    d_img, sp = ops.upload_pitched(torch.from_numpy(img).pin_memory())
    got2, _ = ops.fit_resize_area(d_img, H, W, ch, sp, h, w)
    assert torch.equal(got, got2)


def test_fit_resize_area_golden_and_refusals(ops, golden):
    g = golden("fit")      # the reference's own adjust_to_tile outputs
    for name in ("g", "c", "n"):
        src, ref = g["fitimg_%s_in" % name], g["fitimg_%s_out" % name]
        ch = 1 if src.ndim == 2 else 3
        H, W = src.shape[:2]
        h, w = ref.shape[:2]
        got, _ = ops.fit_resize_area(dev(src), H, W, ch, W * ch, h, w)
        assert np.array_equal(got.cpu().numpy()[:, :w * ch], ref.reshape(h, w * ch))
    # integer factors are OpenCV's separate "fast area" code, up-scales its linear filter: refused, the
    # caller keeps the host cv2 call
    assert not ops.area_supported(1024, 1024, 512, 512)
    assert not ops.area_supported(500, 500, 512, 512)
    assert ops.area_supported(1024, 1000, 512, 512)
    with pytest.raises(ops.PylcError):
        ops.fit_resize_area(dev(np.zeros((1024, 1024), np.uint8)), 1024, 1024, 1, 1024, 512, 512)


# ---------------------------------------------------------------------------------------------
# resample + encode + confusion
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pk,h,w,h_full,w_full", [("a", 1024, 1536, 1500, 2000), ("a", 1536, 2560, 2000, 3000),
                                                  ("b", 64, 96, 70, 100), ("a", 512, 512, 512, 512),
                                                  ("a", 96, 64, 131, 77)])
def test_resample_encode_confusion(ops, palettes, pk, h, w, h_full, w_full):
    pal = palettes[pk]
    C = len(pal)
    rng = np.random.default_rng(h + w)
    labels = orc.synth_labels(11, w, h, C, block=37)
    gt = orc.synth_mask(12, w_full, h_full, pal, skew=True, off_palette=0.003)
    d_gt, pitch = ops.upload_image(gt)
    lut = orc.colourize_lut(C, pal).tolist()
    res = ops.resample_encode_confusion(dev(labels), w_full, h_full, gt_rgb=d_gt, gt_pitch=pitch, palette=pal,
                                        lut_rgb=lut, n_inject=C, want_pred=True, want_rgb=True, want_gt=True)
    pred_full = orc.resample_labels(labels, w_full, h_full)
    gt_lab = orc.class_encode_hwc(gt, pal)
    # label / RGB outputs are the plain resample and encode; only the counts see the coverage injection
    assert np.array_equal(res["pred_full"].cpu().numpy(), pred_full)
    assert np.array_equal(res["gt_full"].cpu().numpy(), gt_lab)
    yt, yp = orc.inject_coverage(gt_lab, pred_full, C)
    assert np.array_equal(res["conf"].cpu().numpy(), orc.confusion_counts(yt, yp, C))
    assert int(res["conf"].sum()) == h_full * w_full
    assert np.array_equal(res["pred_rgb"].cpu().numpy(), np.asarray(lut, dtype=np.uint8)[pred_full])
    # aggregate path: flat vectors
    conf2 = ops.confusion_u8(dev(gt_lab), dev(pred_full), C, n_inject=C)
    assert torch.equal(conf2, res["conf"])
    # random (incoherent) labels stress the run-length path
    a = rng.integers(0, C, size=100003, dtype=np.uint8)
    b = rng.integers(0, C, size=100003, dtype=np.uint8)
    assert np.array_equal(ops.confusion_u8(dev(a), dev(b), C).cpu().numpy(), orc.confusion_counts(a, b, C))


@pytest.mark.parametrize("C,h,w,h_full,w_full,pitched", [
    (9, 1536, 2560, 2000, 3000, True),      # the bench geometry, counts only (pre-multiplied pair codes)
    (11, 256, 512, 301, 777, False),        # ragged width, unpitched ground truth (byte-wise loads)
    (15, 64, 160, 50, 100, True),           # down-sampling by < 2: still the PRMT gather
    (9, 300, 400, 100, 130, True),          # down-sampling by ~3: per-pixel gather
    (9, 97, 131, 120, 150, True),           # label row pitch not a multiple of 4: per-pixel gather
    (20, 128, 192, 150, 250, True),         # C > 15: u32 pair codes, per-warp atomic tables
    (32, 64, 64, 64, 64, False),            # identity maps, maximum class count
])
def test_resample_confusion_counts_only(ops, C, h, w, h_full, w_full, pitched):
    rng = np.random.default_rng(C * 1000 + w)
    pal = rng.permutation(256 ** 3)[:C]
    pal = [[int(v) & 255, (int(v) >> 8) & 255, int(v) >> 16] for v in pal]
    labels = orc.synth_labels(5, w, h, C, block=23)
    gt = orc.synth_mask(6, w_full, h_full, pal, skew=False, off_palette=0.01)
    if pitched:
        d_gt, pitch = ops.upload_image(gt)
    else:
        d_gt, pitch = dev(gt), w_full * 3
    conf = torch.zeros((C, C), dtype=torch.int64, device="cuda")
    res = ops.resample_encode_confusion(dev(labels), w_full, h_full, gt_rgb=d_gt, gt_pitch=pitch, palette=pal,
                                        n_inject=min(C, 9), conf=conf, want_pred=True)
    pred_full = orc.resample_labels(labels, w_full, h_full)
    gt_lab = orc.class_encode_hwc(gt, pal)
    assert np.array_equal(res["pred_full"].cpu().numpy(), pred_full)
    yt, yp = orc.inject_coverage(gt_lab, pred_full, min(C, 9))
    assert np.array_equal(conf.cpu().numpy(), orc.confusion_counts(yt, yp, C))
    # accumulates into the caller's matrix, and the optional ground-truth output does not change the counts
    res2 = ops.resample_encode_confusion(dev(labels), w_full, h_full, gt_rgb=d_gt, gt_pitch=pitch, palette=pal,
                                         n_inject=min(C, 9), conf=conf, want_gt=True)
    assert np.array_equal(res2["gt_full"].cpu().numpy(), gt_lab)
    assert np.array_equal(conf.cpu().numpy(), 2 * orc.confusion_counts(yt, yp, C))


@pytest.mark.parametrize("C,h,w,h_full,w_full,block,noise", [
    (9, 1536, 2560, 2000, 3000, 50, False),   # the bench geometry: 12 column blocks, ragged last unit (3000 = 187.5 units)
    (9, 1536, 2560, 2000, 3000, 50, True),    # per-pixel noise predictions: every group mixed (the dense branch)
    (11, 256, 512, 301, 777, 23, False),      # ragged width (777 % 4 = 1: a partial group), 301 rows = 18.8 boxes
    (9, 64, 160, 50, 100, 9, False),          # down-sampling by < 2: window lanes and per-pixel lanes in one warp
    (9, 304, 400, 100, 130, 7, False),        # down-sampling by ~3: every lane gathers from global memory
    (11, 512, 1024, 7, 2050, 3, False),       # fewer rows than one box, width just past a column block
    (9, 1024, 1536, 1500, 2000, 200, False),  # configs[0]: large uniform regions (anchor path almost everywhere)
    (2, 16, 16, 16, 16, 4, True),             # identity maps, two classes
])
def test_resample_confusion_tma_route(ops, monkeypatch, C, h, w, h_full, w_full, block, noise):
    """Counts-only calls with 16-byte aligned rows take the TMA kernel (confusion_tma.cu): bit-exact against
    the oracle's sklearn-equivalent counts, and equal to the per-thread kernel (PYLC_NO_TMA=1)."""
    rng = np.random.default_rng(C * 1000 + w_full)
    pal = rng.permutation(256 ** 3)[:C]
    pal = [[int(v) & 255, (int(v) >> 8) & 255, int(v) >> 16] for v in pal]
    labels = rng.integers(0, C, size=(h, w), dtype=np.uint8) if noise else orc.synth_labels(5, w, h, C, block=block)
    gt = orc.synth_mask(6, w_full, h_full, pal, skew=False, off_palette=0.01)
    d_gt, pitch = ops.upload_image(gt)
    pred_full = orc.resample_labels(labels, w_full, h_full)
    gt_lab = orc.class_encode_hwc(gt, pal)
    for n_inject in (min(C, w_full), 0):
        yt, yp = orc.inject_coverage(gt_lab, pred_full, n_inject)
        want = orc.confusion_counts(yt, yp, C)
        got = {}
        for no_tma in ("0", "1"):
            monkeypatch.setenv("PYLC_NO_TMA", no_tma)
            res = ops.resample_encode_confusion(dev(labels), w_full, h_full, gt_rgb=d_gt, gt_pitch=pitch, palette=pal, n_inject=n_inject)
            got[no_tma] = res["conf"].cpu().numpy()
        assert np.array_equal(got["0"], want)
        assert np.array_equal(got["1"], want)
        assert int(got["0"].sum()) == h_full * w_full


def test_resample_confusion_uniform_tall_image(ops, palettes):
    """A single (truth, prediction) pair over a tall narrow image: every lane counter of one code
    column carries the whole count, and ragged 48-px rows take the byte-wise ground-truth loads."""
    pal = palettes["a"]
    C = len(pal)
    h_full, w_full = 9000, 48
    labels = np.full((4500, 24), 3, dtype=np.uint8)
    gt = np.empty((h_full, w_full, 3), dtype=np.uint8)
    gt[:] = np.asarray(pal[5], dtype=np.uint8)
    res = ops.resample_encode_confusion(dev(labels), w_full, h_full, gt_rgb=dev(gt), gt_pitch=w_full * 3, palette=pal, n_inject=0)
    ref = np.zeros((C, C), dtype=np.int64)
    ref[5, 3] = h_full * w_full
    assert np.array_equal(res["conf"].cpu().numpy(), ref)


def test_evaluate_golden(ops, golden, palettes):
    g = golden("evaluate")
    pal = palettes["a"]
    C = len(pal)
    gt = g["eval_gt_rgb"]
    pred_rgb = g["eval_pred_rgb"].astype(np.uint8)
    h, w = gt.shape[:2]
    # Evaluator.load class-encodes the predicted RGB mask back to labels (utils/evaluate.py:104-107)
    d_pred, pp = ops.upload_image(pred_rgb)
    pred_lab = ops.class_encode_hwc(d_pred, h, w, pp, pal)[0]
    assert np.array_equal(pred_lab.cpu().numpy().ravel(), g["eval_y_pred_raw"])
    d_gt, gp = ops.upload_image(gt)
    res = ops.resample_encode_confusion(pred_lab, w, h, gt_rgb=d_gt, gt_pitch=gp, palette=pal, n_inject=C,
                                        want_pred=True, want_gt=True)
    # the golden vectors are the reference's y_true / y_pred AFTER validate()'s in-place injection
    yt, yp = orc.inject_coverage(res["gt_full"].cpu().numpy(), res["pred_full"].cpu().numpy(), C)
    assert np.array_equal(yt, g["eval_y_true"])
    assert np.array_equal(yp, g["eval_y_pred"])
    assert np.array_equal(res["conf"].cpu().numpy(), orc.confusion_counts(g["eval_y_true"], g["eval_y_pred"], C))
    M = res["conf"].cpu().numpy()
    m = orc.metrics_from_confusion(M)
    np.testing.assert_allclose([m["f1"], m["iou"], m["mcc"]], g["eval_scalars"], rtol=1e-12)
    np.testing.assert_allclose(m["cmatrix"], g["eval_cmatrix"], rtol=1e-15)


# ---------------------------------------------------------------------------------------------
# multi-loss
# ---------------------------------------------------------------------------------------------

def run_loss(ops, z, t, C, w=None, weighted=False, **kw):
    cfg = ops.loss_cfg(**kw)
    dz, dt = dev(z), dev(t)
    cw = dev(np.asarray(w, dtype=np.float32)) if weighted else None
    part = ops.multiloss_reduce(dz, dt, cfg, class_w=cw)
    vals = ops.multiloss_finalize(part, C, t.size, cfg)
    grad = ops.multiloss_grad(dz, dt, cfg, part, t.size, class_w=cw)
    return vals.cpu().numpy(), grad.cpu().numpy(), part.cpu().numpy()


@pytest.mark.parametrize("name,C,weighted", [("a_unw", 9, False), ("a_w", 9, True), ("b_w", 11, True)])
def test_multiloss_golden(ops, golden, name, C, weighted):
    g = golden("loss")
    z, t, w = g["loss_%s_z" % name], g["loss_%s_t" % name], g["loss_%s_w" % name]
    vals, grad, _ = run_loss(ops, z, t, C, w, weighted)
    np.testing.assert_allclose(vals, g["loss_%s_vals" % name], rtol=LOSS_RTOL)
    np.testing.assert_allclose(grad, g["loss_%s_grad" % name], rtol=1e-3, atol=2e-9)
    # u8 targets take the same path
    vals8, grad8, _ = run_loss(ops, z, t.astype(np.uint8), C, w, weighted)
    assert np.array_equal(vals, vals8) or np.allclose(vals, vals8, rtol=1e-6)
    np.testing.assert_allclose(grad8, grad, rtol=1e-5, atol=1e-10)


@pytest.mark.parametrize("B,C,H,W,weighted", [(4, 9, 128, 128, False), (2, 11, 64, 96, True), (3, 5, 17, 23, True),
                                              (2, 20, 32, 32, False), (1, 12, 64, 64, True), (2, 2, 16, 16, False)])
def test_multiloss_vs_oracle(ops, B, C, H, W, weighted):
    rng = np.random.default_rng(B * 1000 + C)
    z = (rng.standard_normal((B, C, H, W)) * 3).astype(np.float32)
    t = rng.integers(0, C, size=(B, H, W)).astype(np.int64)
    w = (rng.random(C) * 0.9 + 0.1).astype(np.float32)
    vals, grad, part = run_loss(ops, z, t, C, w, weighted)
    loss, ce, dice, focal, ref_grad, ref_part = orc.multiloss(z, t, C, weights=w, weighted=weighted)
    np.testing.assert_allclose(vals, [loss, ce, dice, focal], rtol=LOSS_RTOL)
    np.testing.assert_allclose(part, ref_part, rtol=1e-5)
    np.testing.assert_allclose(grad, ref_grad, rtol=1e-3, atol=1e-9)
    # the port (torch autograd, what the reference runs) agrees too
    port = orc.multiloss_port(z, t, C, weights=w, weighted=weighted)
    np.testing.assert_allclose(vals, port[:4], rtol=LOSS_RTOL)
    np.testing.assert_allclose(grad, port[4], rtol=1e-3, atol=2e-9)


def test_multiloss_other_hyperparameters(ops):
    rng = np.random.default_rng(77)
    z = (rng.standard_normal((2, 9, 32, 32)) * 2).astype(np.float32)
    t = rng.integers(0, 9, size=(2, 32, 32)).astype(np.int64)
    kw = dict(ce=0.3, dice=1.2, focal=0.7, smooth=0.5, gamma=3.0, alpha=0.4)
    vals, grad, _ = run_loss(ops, z, t, 9, **kw)
    ref = orc.multiloss(z, t, 9, **kw)
    np.testing.assert_allclose(vals, ref[:4], rtol=LOSS_RTOL)
    np.testing.assert_allclose(grad, ref[4], rtol=1e-3, atol=1e-9)


def test_multiloss_partials_are_additive_across_shards(ops):
    """Data-parallel contract: partials of two half-batches add up to the full-batch partials,
    so an all-reduce between the two passes reproduces the single-GPU loss and gradient."""
    rng = np.random.default_rng(5)
    z = (rng.standard_normal((4, 9, 64, 64)) * 3).astype(np.float32)
    t = rng.integers(0, 9, size=(4, 64, 64)).astype(np.int64)
    cfg = ops.loss_cfg()
    full = ops.multiloss_reduce(dev(z), dev(t), cfg)
    part = ops.multiloss_reduce(dev(z[:2]), dev(t[:2]), cfg)
    part = ops.multiloss_reduce(dev(z[2:]), dev(t[2:]), cfg, partials=part)
    np.testing.assert_allclose(part.cpu().numpy(), full.cpu().numpy(), rtol=1e-12)
    g_full = ops.multiloss_grad(dev(z), dev(t), cfg, full, t.size)
    g_half = ops.multiloss_grad(dev(z[2:]), dev(t[2:]), cfg, part, t.size)
    np.testing.assert_allclose(g_half.cpu().numpy(), g_full.cpu().numpy()[2:], rtol=1e-6, atol=1e-12)


@pytest.mark.parametrize("B,C,H,W,weighted,u8", [(4, 9, 128, 128, False, False), (2, 11, 64, 96, True, False),
                                                 (3, 5, 17, 23, True, True), (2, 20, 32, 32, False, True),
                                                 (8, 9, 512, 512, True, False)])
def test_multiloss_fused_equals_two_pass(ops, B, C, H, W, weighted, u8):
    """The single cooperative launch (reduce -> grid barrier -> gradient, back to front) against the
    two-launch path and the oracle: same loss values (1e-4 relative, north_star) and gradient."""
    rng = np.random.default_rng(B * C + H)
    z = (rng.standard_normal((B, C, H, W)) * 3).astype(np.float32)
    t = rng.integers(0, C, size=(B, H, W)).astype(np.uint8 if u8 else np.int64)
    w = (rng.random(C) + 0.3).astype(np.float32)
    cfg = ops.loss_cfg()
    dz, dt = dev(z), dev(t)
    cw = dev(w) if weighted else None
    out4, grad, part = ops.multiloss_fwd_bwd(dz, dt, cfg, class_w=cw)
    part2 = ops.multiloss_reduce(dz, dt, cfg, class_w=cw)
    vals2 = ops.multiloss_finalize(part2, C, t.size, cfg)
    grad2 = ops.multiloss_grad(dz, dt, cfg, part2, t.size, class_w=cw)
    np.testing.assert_allclose(part.cpu().numpy(), part2.cpu().numpy(), rtol=1e-9)
    np.testing.assert_allclose(out4.cpu().numpy(), vals2.cpu().numpy(), rtol=1e-6)
    np.testing.assert_allclose(grad.cpu().numpy(), grad2.cpu().numpy(), rtol=1e-5, atol=1e-12)
    if B * H * W <= 1 << 17:
        ref = orc.multiloss(z, t.astype(np.int64), C, weights=w if weighted else None, weighted=weighted)
        np.testing.assert_allclose(out4.cpu().numpy(), ref[:4], rtol=LOSS_RTOL)
        np.testing.assert_allclose(grad.cpu().numpy(), ref[4], rtol=2e-3, atol=1e-9)
    # upstream-gradient rescale: untouched for 1, scaled otherwise
    g1 = grad.clone()
    ops.scale_unless_one_(g1, torch.ones((), device="cuda"))
    assert torch.equal(g1, grad)
    ops.scale_unless_one_(g1, torch.full((), 0.5, device="cuda"))
    assert torch.equal(g1, grad * 0.5)


@pytest.mark.parametrize("B,C,H,W", [(4, 9, 128, 128), (3, 11, 31, 37), (2, 5, 64, 64)])
def test_multiloss_u8_target_workspace(ops, B, C, H, W):
    """int64 targets (the reference dtype): the reduce pass leaves a one-byte copy of the targets, the
    gradient pass reads that instead -- identical partials, loss values and gradient with and without it,
    in the two-launch and the single-launch form."""
    rng = np.random.default_rng(B + C + H)
    dz = dev((rng.standard_normal((B, C, H, W)) * 3).astype(np.float32))
    t = rng.integers(0, C, size=(B, H, W)).astype(np.int64)
    dt = dev(t)
    cfg = ops.loss_cfg()
    t8 = torch.full((t.size,), 255, dtype=torch.uint8, device="cuda")
    part = ops.multiloss_reduce(dz, dt, cfg, target_u8_out=t8)
    assert torch.equal(t8.view(B, H, W), dt.to(torch.uint8))
    part0 = ops.multiloss_reduce(dz, dt, cfg)
    assert torch.equal(part, part0)
    g8 = ops.multiloss_grad(dz, t8.view(B, H, W), cfg, part, t.size)
    g64 = ops.multiloss_grad(dz, dt, cfg, part, t.size)
    assert torch.equal(g8, g64)
    o_ws, g_ws, p_ws = ops.multiloss_fwd_bwd(dz, dt, cfg)                     # workspace on (default)
    o_no, g_no, p_no = ops.multiloss_fwd_bwd(dz, dt, cfg, use_u8_ws=False)
    assert torch.equal(o_ws, o_no) and torch.equal(g_ws, g_no)
    np.testing.assert_allclose(p_ws.cpu().numpy(), p_no.cpu().numpy(), rtol=1e-12)


def test_multiloss_out_of_range_target_is_loud(ops):
    """A target outside [0, C) (a mask encoded with another schema, a 255 'ignore' label): the reference's
    CrossEntropyLoss / one_hot raise (loss.py:66-69,137).  The kernels turn every value and gradient of the
    batch into NaN instead of silently using another class's weight; the host mirror raises."""
    from pylc_b200.models.modules.loss import MultiLoss
    C = 9
    g = torch.Generator().manual_seed(5)
    z = (torch.randn(2, C, 32, 32, generator=g) * 3).cuda()
    t = torch.randint(0, C, (2, 32, 32), generator=g).cuda()
    t[1, 7, 9] = C + 2
    cfg = ops.loss_cfg()
    part = ops.multiloss_reduce(z, t, cfg)
    vals = ops.multiloss_finalize(part, C, t.numel(), cfg)
    assert bool(torch.isnan(vals[0])) and bool(torch.isnan(vals[1]))
    out4, grad, _ = ops.multiloss_fwd_bwd(z, t, cfg)
    assert bool(torch.isnan(out4[0])) and bool(torch.isnan(grad).any())
    crit = MultiLoss({"weighted": False, "weights": None, "ce": 0.5, "dice": 0.5, "focal": 0.5},
                     {"n_classes": C, "class_codes": list("abcdefghi"), "class_labels": list("abcdefghi")})
    with pytest.raises(IndexError):
        crit(z, t)
    t[1, 7, 9] = 0
    assert bool(torch.isfinite(crit(z, t)))


def test_multiloss_second_backward_over_retained_graph(ops):
    """retain_graph=True / gradient checkpointing: the single-launch path hands its stashed gradient to the
    first backward and recomputes it from the saved tensors for any later one -- same values."""
    from pylc_b200.models.modules.loss import MultiLoss
    C = 9
    g = torch.Generator().manual_seed(6)
    z = (torch.randn(2, C, 48, 48, generator=g) * 3).cuda().requires_grad_(True)
    t = torch.randint(0, C, (2, 48, 48), generator=g).cuda()
    crit = MultiLoss({"weighted": True, "weights": list(np.linspace(0.2, 1.0, C)), "ce": 0.5, "dice": 0.5, "focal": 0.5},
                     {"n_classes": C, "class_codes": list("abcdefghi"), "class_labels": list("abcdefghi")})
    loss = crit(z, t)
    loss.backward(retain_graph=True)
    g1 = z.grad.clone()
    z.grad = None
    (2.0 * loss).backward()
    np.testing.assert_allclose(z.grad.cpu().numpy(), 2.0 * g1.cpu().numpy(), rtol=1e-5, atol=1e-12)


# ---------------------------------------------------------------------------------------------
# network glue kernels (channels-last activations) against the eager PyTorch ops they replace
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("B,Cx,h,w,Cl,H,W", [(3, 256, 32, 32, 48, 128, 128), (2, 64, 5, 7, 8, 19, 23), (1, 512, 4, 4, 4, 9, 9),
                                              (2, 128, 8, 8, 48, 8, 8)])
def test_upsample_concat_nhwc(ops, B, Cx, h, w, Cl, H, W):
    g = torch.Generator(device="cuda").manual_seed(B * Cx)
    x = torch.randn((B, Cx, h, w), device="cuda", generator=g).contiguous(memory_format=torch.channels_last)
    low = torch.randn((B, Cl, H, W), device="cuda", generator=g).contiguous(memory_format=torch.channels_last)
    ref = torch.cat((torch.nn.functional.interpolate(x, size=(H, W), mode="bilinear", align_corners=True), low), dim=1)
    got = ops.upsample_concat_nhwc(x, low)
    assert got.shape == ref.shape and got.is_contiguous(memory_format=torch.channels_last)
    torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-6)     # float rounding of the same bilinear formula
    assert torch.equal(got[:, Cx:], low)                            # the concatenated channels are a copy


@pytest.mark.parametrize("B,C,H,W", [(2, 64, 256, 256), (1, 8, 7, 9), (3, 16, 10, 5), (1, 4, 1, 1)])
def test_maxpool3x3s2_nhwc(ops, B, C, H, W):
    x = torch.randn((B, C, H, W), device="cuda").contiguous(memory_format=torch.channels_last)
    ref = torch.nn.functional.max_pool2d(x, 3, stride=2, padding=1)
    got = ops.maxpool3x3s2_nhwc(x)
    assert torch.equal(got, ref)


@pytest.mark.parametrize("B,C,h,w,H,W", [(3, 9, 128, 128, 512, 512), (2, 11, 16, 16, 64, 64), (1, 20, 5, 6, 8, 12), (2, 9, 32, 32, 32, 32)])
def test_upsample_nhwc_to_nchw(ops, B, C, h, w, H, W):
    x = torch.randn((B, C, h, w), device="cuda").contiguous(memory_format=torch.channels_last)
    ref = torch.nn.functional.interpolate(x.contiguous(), size=(H, W), mode="bilinear", align_corners=True)
    got = ops.upsample_nhwc_to_nchw(x, (H, W))
    assert got.is_contiguous()
    torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("ch,H,W,T,S", [(3, 1024, 1536, 512, 256), (1, 700, 650, 128, 64), (3, 96, 64, 32, 32)])
def test_gather_norm_s2d_layout(ops, ch, H, W, T, S):
    """The space-to-depth stem layout is the normalised tiles of pylc_tile_gather_norm_f32, re-indexed:
    bit-equal values, zero border (2 before, 1 after) and zero channels 12..15."""
    img = orc.synth_image(7, W, H, ch)
    d, pitch = ops.upload_image(img)
    mean, std = ([120.0], [40.0]) if ch == 1 else ([130.0, 140.0, 150.0], [25.0, 22.0, 19.0])
    planar = ops.tile_gather_norm_f32(d, H, W, ch, pitch, T, S, mean, std, 255.0, 3)          # [n,3,T,T]
    s2d = ops.tile_gather_norm_s2d(d, H, W, ch, pitch, T, S, mean, std, 255.0)                # [n,16,T/2+3,T/2+3]
    n, Hs = planar.shape[0], T // 2 + 3
    assert s2d.shape == (n, 16, Hs, Hs) and s2d.is_contiguous(memory_format=torch.channels_last)
    ref = torch.zeros((n, 16, Hs, Hs), device="cuda")
    for py in range(2):
        for px in range(2):
            ref[:, (py * 2 + px) * 3:(py * 2 + px) * 3 + 3, 2:2 + T // 2, 2:2 + T // 2] = planar[:, :, py::2, px::2]
    assert torch.equal(s2d, ref)


def test_s2d_stem_equals_7x7_stem(ops):
    """FusedDeepLab's rearranged 4x4 stem on the space-to-depth tiles == its 7x7 stride-2 stem on the
    planar tiles (same products; TF32 convolution noise only), and so are the final logits."""
    from pylc_b200.models.deeplab import DeepLab
    from pylc_b200.models.fused import FusedDeepLab
    torch.manual_seed(0)
    net = DeepLab(n_classes=9).cuda().eval().to(memory_format=torch.channels_last)
    plan = FusedDeepLab(net, channels_last=True)
    assert plan.stem_s2d is not None
    img = orc.synth_image(5, 768, 512, 3)
    d, pitch = ops.upload_image(img)
    mean, std = [130.0, 140.0, 150.0], [25.0, 22.0, 19.0]
    planar = ops.tile_gather_norm_f32(d, 512, 768, 3, pitch, 256, 128, mean, std, 255.0, 3)
    s2d = ops.tile_gather_norm_s2d(d, 512, 768, 3, pitch, 256, 128, mean, std, 255.0)
    a = plan.stem(planar.contiguous(memory_format=torch.channels_last))
    b = plan.stem_s2d(s2d)
    assert a.shape == b.shape
    assert (a - b).abs().max() <= 2e-3 * a.abs().max()
    ya, yb = plan(planar), plan.forward_s2d(s2d)
    assert ya.shape == yb.shape == (planar.shape[0], 9, 256, 256)
    assert (ya - yb).abs().max() <= 5e-3 * ya.abs().max()


@pytest.mark.parametrize("H,W,d,cin,cout,B", [(32, 32, 18, 2048, 256, 5), (32, 32, 12, 256, 64, 3), (24, 40, 6, 64, 32, 2), (32, 32, 24, 128, 16, 1)])
def test_tap_split_route_equals_cudnn_convolution(ops, H, W, d, cin, cout, B):
    """The inference plan's third convolution route (models/fused.py::_Conv._tap_split): a 3x3 convolution with
    padding == dilation as cuBLAS GEMMs over the tap windows that miss the zero padding.  Same TF32 products and
    fp32 sums as the cuDNN convolution of the same folded weights, in another order: equal to TF32 rounding."""
    import torch.nn as nn
    import torch.nn.functional as F
    from pylc_b200.models.fused import _Conv
    torch.manual_seed(d)
    conv = nn.Conv2d(cin, cout, 3, padding=d, dilation=d, bias=False).cuda()
    bn = nn.BatchNorm2d(cout).cuda().eval()
    with torch.no_grad():
        bn.running_mean.normal_()
        bn.running_var.uniform_(0.5, 2.0)
        bn.weight.normal_()
        bn.bias.normal_()
    c = _Conv(conv, bn, True, True)
    x = torch.randn(B, cin, H, W, device="cuda").contiguous(memory_format=torch.channels_last)
    assert c._tap_split_applies(x, None)
    with torch.no_grad():
        want = F.relu(F.conv2d(x, c.w, c.b, 1, d, d))
        exact = F.relu(F.conv2d(x.double(), c.w.double(), c.b.double(), 1, d, d))
        got = c._tap_split(x)
    assert got.shape == want.shape and got.is_contiguous(memory_format=torch.channels_last)
    scale = float(exact.abs().max())
    err_split, err_cudnn = float((got - exact).abs().max()), float((want - exact).abs().max())
    assert err_split <= 3e-3 * scale                       # TF32 inputs (10-bit mantissa), fp32 accumulation
    assert err_split <= 4 * err_cudnn + 1e-6 * scale       # no worse than the library convolution it replaces
    # and the plan's call returns the same thing whichever route its geometry rule picks
    y = c(x)
    assert float((y - exact).abs().max()) <= 3e-3 * scale


@pytest.mark.parametrize("W,H", [(1300, 1100), (2000, 1500)])
def test_tma_and_per_thread_routes_agree(ops, palettes, monkeypatch, W, H):
    """Every entry point with a TMA form (16-byte pitched rows) returns the same bytes from its per-thread kernels
    (PYLC_NO_TMA=1): mask gather + encode + histogram, class_encode, fit-resize."""
    pal = palettes["b"]
    mask = orc.synth_mask(21, W, H, pal, skew=True, off_palette=0.01)
    img = orc.synth_image(22, W, H, 3)
    d_mask, mp = ops.upload_image(mask)
    d_img, ip = ops.upload_image(img)
    w, h = orc.fit_dims(W, H, 512)
    got = {}
    for no_tma in ("0", "1"):
        monkeypatch.setenv("PYLC_NO_TMA", no_tma)
        tiles, hist = ops.mask_gather_encode_hist(d_mask, H, W, mp, 512, 512, pal)
        enc = ops.class_encode_hwc(d_mask, H, W, mp, pal, hist=True)
        fit, _ = ops.fit_resize_area(d_img, H, W, 3, ip, h, w)
        got[no_tma] = (tiles.clone(), hist.clone(), enc[0].clone(), enc[1].clone(), fit[:, :w * 3].clone())
    for a, b in zip(got["0"], got["1"]):
        assert torch.equal(a, b)
    assert np.array_equal(got["0"][0].cpu().numpy(), orc.class_encode(orc.split_tiles(mask, 512, 512), pal))


@pytest.mark.parametrize("seed", range(6))
def test_fit_resize_random_geometries_bit_exact(ops, seed):
    """Random down-scales with factors in [1, 1.9) on both axes, gray and colour, pitched rows (the TMA + f32x2
    kernel, incl. its byte-load fallback for column blocks whose taps spread too far): every byte equals OpenCV's."""
    import cv2
    rng = np.random.default_rng(100 + seed)
    for _ in range(4):
        ch = int(rng.choice([1, 3]))
        w, h = int(rng.integers(40, 900)), int(rng.integers(33, 700))
        W, H = min(int(w * rng.uniform(1.0, 1.89)), int(w * 1.89)), min(int(h * rng.uniform(1.0, 1.95)), int(h * 1.95))
        W, H = max(W, w), max(H, h)
        if not ops.area_supported(W, H, w, h):
            continue
        img = rng.integers(0, 256, size=(H, W) if ch == 1 else (H, W, 3), dtype=np.uint8)
        d_img, pitch = ops.upload_image(img)
        out, po = ops.fit_resize_area(d_img, H, W, ch, pitch, h, w)
        want = cv2.resize(img, (w, h), interpolation=cv2.INTER_AREA)
        got = out.cpu().numpy()[:, :w * ch].reshape(want.shape)
        assert np.array_equal(got, want), (W, H, w, h, ch)


@pytest.mark.parametrize("seed", range(6))
def test_resample_confusion_tma_random_geometries(ops, seed):
    """Random label-map / ground-truth geometries (up- and down-sampling, ragged widths, few rows) and class counts
    through the counts-only route: equal to the oracle's counts."""
    rng = np.random.default_rng(200 + seed)
    for _ in range(4):
        C = int(rng.integers(2, 12))
        w, h = 16 * int(rng.integers(1, 40)), int(rng.integers(1, 300))
        w_full, h_full = int(rng.integers(C, 900)), int(rng.integers(1, 500))
        pal = rng.permutation(256 ** 3)[:C]
        pal = [[int(v) & 255, (int(v) >> 8) & 255, int(v) >> 16] for v in pal]
        labels = orc.synth_labels(int(rng.integers(1 << 20)), w, h, C, block=int(rng.integers(1, 40)))
        gt = orc.synth_mask(int(rng.integers(1 << 20)), w_full, h_full, pal, skew=False, off_palette=0.02)
        d_gt, pitch = ops.upload_image(gt)
        n_inject = int(rng.integers(0, C + 1))
        res = ops.resample_encode_confusion(dev(labels), w_full, h_full, gt_rgb=d_gt, gt_pitch=pitch, palette=pal, n_inject=n_inject)
        yt, yp = orc.inject_coverage(orc.class_encode_hwc(gt, pal), orc.resample_labels(labels, w_full, h_full), n_inject)
        assert np.array_equal(res["conf"].cpu().numpy(), orc.confusion_counts(yt, yp, C)), (C, w, h, w_full, h_full, n_inject)


# ---------------------------------------------------------------------------------------------
# augmentation copies on the device (tools.augment_transform, utils/tools.py:452-594)
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ch", [1, 3])
def test_augment_tiles_device_equals_reference_golden_and_opencv(ops, golden, ch):
    """pylc_augment_tiles_u8: the bytes the reference's augment_transform produced for the fixture tile and
    RandomState(0 / 1 / 3) (golden warp vectors), and the OpenCV call chain on noise tiles with other seeds and a
    job table that re-uses and re-orders sources.  Bit-exact: image and mask."""
    from pylc_b200.utils import tools
    g = golden("warp")
    img, mask = orc.augment_fixture_tile(ch)
    seeds = [0, 1, 3]
    params = [tools.augment_params(np.random.RandomState(s), 512) for s in seeds]
    out_i, out_m = ops.augment_tiles(dev(img), dev(mask), [0, 0, 0], np.stack([p[0] for p in params]), [p[1] for p in params])
    out_i, out_m = out_i.cpu().numpy(), out_m.cpu().numpy()
    for j, s in enumerate(seeds):
        want = g["warp_ch%d_s%d_img" % (ch, s)]
        assert np.array_equal(out_i[j].reshape(want.shape), want)
        assert np.array_equal(out_m[j], g["warp_ch%d_s%d_mask" % (ch, s)])
    rng = np.random.default_rng(ch)
    img = rng.integers(0, 256, size=(2, ch, 512, 512), dtype=np.uint8)
    mask = rng.integers(0, 11, size=(2, 512, 512)).astype(np.uint8)
    seeds, srcs = [2, 5, 8], [1, 0, 1]
    params = [tools.augment_params(np.random.RandomState(s), 512) for s in seeds]
    out_i, out_m = ops.augment_tiles(dev(img), dev(mask), srcs, np.stack([p[0] for p in params]), [p[1] for p in params])
    for j, (s, k) in enumerate(zip(seeds, srcs)):
        a, b = tools.augment_transform(img[k:k + 1].astype(np.float32), mask[k:k + 1].astype(np.int64), np.random.RandomState(s))
        assert np.array_equal(np.asarray(a).reshape(out_i[j].shape), out_i[j].cpu().numpy())
        assert np.array_equal(np.asarray(b), out_m[j].cpu().numpy())
    with pytest.raises(ops.PylcError):
        ops.augment_tiles(dev(img), dev(mask), [2], np.stack([params[0][0]]), [10])      # source index out of range

