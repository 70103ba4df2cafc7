"""Pins the CPU oracle (oracle/hoh_oracle.c) to the real reference compiled from its own sources
(oracle/_ref/libhohref.so).  CPU only.  The comparisons skip when the reference library was never built."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol

needs_ref = pytest.mark.skipif(not ol.have_ref(), reason="oracle/_ref/libhohref.so not built")

STOCK = [0x0001, 0x0002, 0x0020, 0x0010, 0xffbf, 0x0003, 0xfffd, 0xfffb, 0xfff7, 0xffef, 0xffdf,
         0xff7f, 0xfdff, 0xffff]


def _symbols(rng, kind, n, rangev):
    if kind == 0:
        s = rng.integers(0, rangev, n)
    elif kind == 1:
        s = np.clip(np.rint(rng.laplace(rangev / 2, rangev / 40 + 0.3, n)), 0, rangev - 1)
    elif kind == 2:
        s = np.full(n, int(rng.integers(0, rangev)))
    elif kind == 3:
        s = np.clip(rng.geometric(0.3, n) - 1, 0, rangev - 1)
    elif kind == 4:
        s = np.clip(np.rint(rng.laplace(rangev / 2, 1.0, n)), 0, rangev - 1)
        if n > 3:
            s[:3] = [0, rangev - 1, rangev // 3]
    else:
        s = rng.integers(0, max(1, rangev // 8), n)
    return s.astype(np.uint16)


@needs_ref
def test_encode_entropy_random_streams():
    """entropy_encoding.hpp:8 — header, table modes 1/2, rANS payload, stored fallback, n = 0."""
    rng = np.random.default_rng(0)
    checked = 0
    for it in range(1500):
        rangev = int(rng.choice([1, 2, 3, 5, 14, 16, 255, 256, 257, 512]))
        pb = int(rng.integers(8, 20))
        if (1 << pb) < rangev:
            pb = 10
        n = int(rng.choice([1, 2, 7, 20, 49, 100, 1000, 5000, 70000])) if it % 50 else 0
        sym = _symbols(rng, it % 6, n, rangev)
        a, st = ol.orc_encode_entropy(sym, rangev, pb)
        if st != 0:
            continue  # the reference would assert() here
        b = ol.ref_encode_entropy(sym, rangev, pb)
        assert a.tobytes() == b.tobytes(), (it, rangev, pb, n)
        checked += 1
    assert checked > 1000


@needs_ref
def test_decode_entropy_matches_reference_where_it_can_parse():
    """entropy_decoding.hpp:134 with reference semantics (flags=0), prob_bits <= 15 (D9)."""
    rng = np.random.default_rng(3)
    for it in range(300):
        rangev = int(rng.choice([2, 14, 256, 512]))
        pb = int(rng.integers(9, 16))
        n = int(rng.choice([1, 5, 49, 1000, 20000]))
        sym = _symbols(rng, it % 6, n, rangev)
        if len(np.unique(sym)) < 2:
            continue  # freq == 2^prob_bits is not representable: the reference decoder asserts
        stream, st = ol.orc_encode_entropy(sym, rangev, pb)
        assert st == 0
        _, _, emode, _, tmode = ol.peek_stream(stream)
        if emode == 1 and tmode == 1:
            continue  # D6: raw tables keep only maxbits bits per freq; the reference cannot decode them
        d_ref, bp_ref = ol.ref_decode_entropy(stream)
        d_orc, bp_orc, st = ol.orc_decode_entropy(stream, flags=0)
        assert bp_ref == bp_orc
        assert (d_ref == d_orc).all() and (d_ref == sym).all()
        d_fix, bp_fix, st = ol.orc_decode_entropy(stream, flags=7)
        assert (d_fix == sym).all() and bp_fix == len(stream)


def test_decode_roundtrip_all_prob_bits_fixed_mode():
    rng = np.random.default_rng(4)
    for pb in range(8, 20):
        sym = _symbols(rng, 1, 30000, 512 if pb >= 9 else 256)
        stream, st = ol.orc_encode_entropy(sym, 512 if pb >= 9 else 256, pb)
        d, bp, st = ol.orc_decode_entropy(stream, flags=7)
        assert (d == sym).all() and bp == len(stream)


@needs_ref
def test_normalize_freqs():
    """stattools.hpp:13"""
    rng = np.random.default_rng(1)
    O, R = ol.oracle(), ol.ref()
    for it in range(1500):
        size = int(rng.choice([1, 2, 5, 14, 256, 512]))
        pb = int(rng.integers(8, 20))
        if (1 << pb) < size:
            continue
        k = it % 4
        if k == 0:
            f = rng.integers(0, 1000, size)
        elif k == 1:
            f = (rng.random(size) < 0.3) * rng.integers(1, 5, size)
        elif k == 2:
            f = np.rint(70000 * np.exp(-np.abs(np.arange(size) - size / 2) / (size / 30 + 0.5))).astype(np.int64)
            f[rng.integers(0, size, 5)] += 1
        else:
            f = rng.integers(0, 3, size)
        f = f.astype(np.uint32)
        if f.sum() == 0:
            f[0] = 1
        fa, fb = f.copy(), f.copy()
        ca, cb = np.zeros(size + 1, np.uint32), np.zeros(size + 1, np.uint32)
        if O.orc_normalize_freqs(fa, ca, size, 1 << pb):
            continue
        R.ref_normalize_freqs(fb, cb, size, 1 << pb)
        assert (fa == fb).all() and (ca == cb).all()


def _plane(rng, w, h, depth, kind):
    c = 1 << depth
    if kind == 0:
        return rng.integers(0, c, w * h).astype(np.uint16)
    if kind == 1:
        rgb = ol.synth_rgb(w, h, int(rng.integers(1, 1000)))
        g, rg, bg = (np.zeros(w * h, np.uint16) for _ in range(3))
        ol.oracle().orc_subtract_green(rgb, rgb.size, g, rg, bg)
        return g if depth == 8 else rg
    if kind == 2:
        base = np.cumsum(rng.integers(-3, 4, w * h)).astype(np.int64) + c // 2
        return np.clip(base, 0, c - 1).astype(np.uint16)
    return np.full(w * h, int(rng.integers(0, c)), np.uint16)


@needs_ref
def test_prediction_and_unprediction():
    """prediction.hpp:6/46/153, unprediction.hpp:6 incl. LZ back-references and clipped cells."""
    rng = np.random.default_rng(2)
    O, R = ol.oracle(), ol.ref()
    for it in range(250):
        w = int(rng.choice([1, 2, 3, 5, 37, 40, 41, 64, 81, 100, 256]))
        h = int(rng.choice([1, 2, 4, 39, 40, 41, 80, 97, 130]))
        depth = int(rng.choice([8, 9]))
        p = _plane(rng, w, h, depth, it % 4)
        a, b = np.zeros(w * h, np.uint16), np.zeros(w * h, np.uint16)
        O.orc_predict_fastpath(p, w, h, depth, a)
        R.ref_predict_fastpath(p, p.size, w, h, depth, b)
        assert (a == b).all()
        xt, yt = (w + 39) // 40, (h + 39) // 40
        for t in range(xt * yt):
            mask = int(rng.choice(STOCK + [int(rng.integers(1, 65536))]))
            ca, cb = np.zeros(1700, np.uint16), np.zeros(1700, np.uint16)
            na = O.orc_predict_section(p, w, h, depth, xt, yt, t % xt, t // xt, mask, ca)
            nb = R.ref_predict_section(p, p.size, w, h, depth, xt, yt, t % xt, t // xt, mask, cb)
            assert na == nb and (ca[:na] == cb[:nb]).all()
        tm = rng.choice(STOCK + [int(rng.integers(0, 65536))], xt * yt).astype(np.uint16)
        O.orc_predict_all(p, w, h, depth, xt, yt, tm, a)
        R.ref_predict_all(p, p.size, w, h, depth, xt, yt, tm, b)
        assert (a == b).all()
        br = np.zeros(w * h, np.uint16)
        if it % 3 == 0 and w * h > 10:
            idx = rng.integers(5, w * h, size=max(1, w * h // 10))
            br[idx] = rng.integers(1, 5, size=idx.size)
        dense = np.concatenate([a[br == 0], np.zeros(4, np.uint16)])
        ua, ub = np.zeros(w * h, np.uint16), np.zeros(w * h, np.uint16)
        O.orc_unpredict_all(dense, w, h, depth, xt, yt, tm, br.ctypes.data, ua)
        R.ref_unpredict_all(dense, dense.size - 4, w, h, depth, xt, yt, tm, br, ub)
        assert (ua == ub).all()
        if not br.any():
            assert (ua == p).all()
        fa, fu = np.zeros(w * h, np.uint16), np.zeros(w * h, np.uint16)
        O.orc_predict_fastpath(p, w, h, depth, fa)
        O.orc_unpredict_fastpath(fa, w, h, depth, None, fu)
        assert (fu == p).all()


@needs_ref
def test_colour_transform():
    """channel.hpp:63-79 and its algebraic inverse."""
    rng = np.random.default_rng(5)
    O, R = ol.oracle(), ol.ref()
    rgb = rng.integers(0, 256, 3 * 1000).astype(np.uint8)
    ga, ra, ba = (np.zeros(1000, np.uint16) for _ in range(3))
    gb, rb, bb = (np.zeros(1000, np.uint16) for _ in range(3))
    O.orc_subtract_green(rgb, rgb.size, ga, ra, ba)
    R.ref_subtract_green(rgb, rgb.size, gb, rb, bb)
    assert (ga == gb).all() and (ra == rb).all() and (ba == bb).all()
    back = np.zeros_like(rgb)
    O.orc_add_green(ga, ra, ba, 1000, back)
    assert (back == rgb).all()
    for t in range(3):
        pa, pb = np.zeros(1000, np.uint16), np.zeros(1000, np.uint16)
        O.orc_channel_picker(rgb, rgb.size, 3, t, pa)
        R.ref_channel_picker(rgb, rgb.size, 3, t, pb)
        assert (pa == pb).all()


@needs_ref
def test_layer_encode_all_modes():
    """layer_encode.hpp:11 byte-for-byte, modes 0-4, depth 8/9, with and without NUKE (D7 incl.)."""
    rng = np.random.default_rng(6)
    for it in range(40):
        w = int(rng.choice([5, 40, 41, 64, 100, 256]))
        h = int(rng.choice([4, 40, 41, 80, 130, 256]))
        depth = int(rng.choice([8, 9]))
        mode = it % 5
        kind = [1, 2, 1, 0, 3][it % 5] if it % 7 else 1
        p = _plane(rng, w, h, depth, kind)
        nuke = np.zeros(w * h, np.uint8)
        if it % 4 == 1:
            nuke[rng.integers(0, w * h, w * h // 8)] = 1
        a, _ = ol.orc_layer_encode(p, w, h, depth, mode, nuke)
        b = ol.ref_layer_encode(p, w, h, depth, mode, nuke)
        assert a.tobytes() == b.tobytes(), (w, h, depth, mode)


@needs_ref
def test_static_table_rans():
    """rans64.hpp:262 (reciprocal form) == divide form, rans64.hpp:107-142 decode (config 4)."""
    O, R = ol.oracle(), ol.ref()
    sym = ol.synth_symbols(1 << 16, 7).astype(np.uint16)
    freqs = np.bincount(sym, minlength=256).astype(np.uint32)
    cum = np.zeros(257, np.uint32)
    assert O.orc_normalize_freqs(freqs, cum, 256, 1 << 12) == 0
    oa, ob = np.zeros(4 * sym.size + 64, np.uint8), np.zeros(4 * sym.size + 64, np.uint8)
    na = O.orc_rans_encode_static(sym, sym.size, freqs, cum, 256, 12, oa)
    nb = R.ref_rans_encode_static(sym, sym.size, freqs, cum, 256, 12, ob)
    assert na == nb and (oa[:na] == ob[:nb]).all()
    da, db = np.zeros(sym.size, np.uint16), np.zeros(sym.size, np.uint16)
    O.orc_rans_decode_static(oa[:na].copy(), na, sym.size, freqs, cum, 256, 12, da)
    R.ref_rans_decode_static(ob[:nb].copy(), nb, sym.size, freqs, cum, 256, 12, db)
    assert (da == sym).all() and (db == sym).all()



@needs_ref
def test_find_lz_rgb_pinned_against_reference():
    """lz.hpp:6 — oracle restatement vs the compiled reference: LZ bytes and nuke map, every seek distance
    encode_tile uses (6, 10, 11, 12, 14) and every break-even bonus, on images that contain matches."""
    rng = np.random.default_rng(77)
    total_matches = 0
    for it in range(40):
        kind = ["flat", "pattern", "rows", "few", "photo"][it % 5]
        w, h = int(rng.integers(5, 70)), int(rng.integers(4, 50))
        img = ol.lz_test_image(rng, w, h, kind)
        for distance in (6, 10, 11, 12, 14):
            bonus = [0, 2, 10, 20, 32][int(rng.integers(0, 5))]
            want, want_nuke = ol.ref_find_lz_rgb(img, w, h, distance, bonus)
            got, got_nuke, side = ol.orc_find_lz_rgb(img, w, distance, bonus)
            assert np.array_equal(got, want), (it, kind, w, h, distance, bonus)
            assert np.array_equal(got_nuke, want_nuke), (it, kind, w, h, distance, bonus)
            total_matches += len(side[1])
    assert total_matches > 1000



@needs_ref
def test_lz_params_pinned_against_reference():
    rng = np.random.default_rng(5)
    for it in range(30):
        ncol = [1, 3, 4, 5, 8, 9, 16, 17, 32, 33, 255, 256, 257, 400][it % 14]
        pal = np.unique(rng.integers(0, 256, (ncol * 3, 3)).astype(np.uint8), axis=0)[:ncol]
        while len(pal) < ncol:
            pal = np.unique(np.concatenate([pal, rng.integers(0, 256, (ncol, 3)).astype(np.uint8)]), axis=0)[:ncol]
        idx = np.concatenate([np.arange(ncol), rng.integers(0, ncol, 500)])
        rng.shuffle(idx)
        img = pal[idx].ravel()
        want = ol.ref().ref_count_colours(img, img.size)
        assert ol.oracle().orc_count_colours(img, img.size) == want == (ncol if ncol <= 256 else -1)


@needs_ref
def test_encode_tile_subgreen_with_lz_pinned_against_reference():
    """choh.cpp:104-382 at -s0 on photographic tiles with repeats: the oracle's pieces (find_lz_rgb, NUKE-aware
    layer_encode) assembled by encode_tile's rules give the reference's tile bytes."""
    rng = np.random.default_rng(9)
    nuked = 0
    for it, (w, h) in enumerate([(64, 64), (120, 75), (256, 256)]):
        img = ol.photo_with_repeats(rng, w, h, 100 + it)
        got, nuke = ol.orc_encode_tile_subgreen(img, 0)
        buf = np.zeros(img.size * 3 + 4096, np.uint8)
        n = ol.ref().ref_encode_tile(np.ascontiguousarray(img).ravel(), img.size, buf, w, h, 0)
        assert got == buf[:n].tobytes(), (it, w, h)
        nuked += int(nuke.sum())
    assert nuked > 50


@needs_ref
def test_encode_tile_all_modes_pinned_against_reference():
    """encode_tile at cruncher modes 1-4 (wider LZ windows, predictor search, prob_bits search, the plain-RGB
    alternative at modes 3-4) on photographic tiles with repeats; one tile is built so that plain RGB wins."""
    rng = np.random.default_rng(10)
    modes_seen, colour_modes = set(), set()
    for it, (w, h, mode) in enumerate([(96, 80, 1), (100, 64, 2), (90, 70, 3), (64, 96, 4), (80, 80, 3)]):
        img = ol.photo_with_repeats(rng, w, h, 200 + it)
        if it == 4:  # decorrelate the channels: subtracting green then only adds noise
            img[..., 0] = rng.integers(0, 256, (h, w))
            img[..., 2] = rng.integers(0, 256, (h, w))
        got, _ = ol.orc_encode_tile_subgreen(img, mode)
        buf = np.zeros(img.size * 3 + 4096, np.uint8)
        n = ol.ref().ref_encode_tile(np.ascontiguousarray(img).ravel(), img.size, buf, w, h, mode)
        assert got == buf[:n].tobytes(), (it, w, h, mode)
        modes_seen.add(mode)
        colour_modes.add(got[2])
    assert modes_seen == {1, 2, 3, 4} and colour_modes == {128, 2}
