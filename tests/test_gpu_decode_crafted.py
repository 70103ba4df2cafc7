"""hoh_decode_images / hoh_decode_regions on tiles written here, independently of this library's encoder.

The decoders must accept any valid .hoh tile: stock `choh` output, other encoder versions, hand-made files.  The
encoder only ever emits its own choices (stock masks picked by the search, the prob_bits ladder, greedy LZ matches),
so a round trip leaves most of what the decoder accepts untested.  `write_tile` below builds tile bytes from an
explicit description of every choice out of the oracle's primitives (oracle/hoh_oracle.c): predictor masks and
per-cell maps, the prob_bits and table form of every entropy stream, and the LZ match list.  The CPU tests pin the
writer to the reference (its bytes equal the oracle's encode_tile / layer_encode for the reference's own choices)
and decode every crafted tile with the oracle's inverse.  The GPU tests decode the same tiles with the library and
check which un-prediction walk ran:
  - grouped: k_dt_unpredict's 8-pixel group walk, tile widths that are multiples of 8 and >= 16;
  - half-warp: k_dt_unpredict16 for predictor-grid planes, other widths at <= 16 384 planes in one pass;
  - scalar: k_dt_unpredict's one-thread-per-plane walk, other widths above 16 384 planes in one pass.
"""
import collections
import functools

import numpy as np
import pytest

import gpu_lib
import oracle_lib as ol

STOCK = [0x0001, 0x0002, 0x0020, 0x0010, 0xffbf, 0x0003, 0xfffd, 0xfffb, 0xfff7, 0xffef, 0xffdf,
         0xff7f, 0xfdff, 0xffff]
GRID = 40                 # predictor grid cell, layer_encode.hpp:124
MED = 0x0010              # the single predictor of the header 10 00 00 00 10
HALF_WARP_MAX_PLANES = 16384
u16 = np.uint16


# ---------------------------------------------------------------------------------------------
# the tile writer
# ---------------------------------------------------------------------------------------------
# One channel's choices.  masks None: the single-predictor header 10 00 00 00 10 (MED, fastpath residuals).
# Otherwise a predictor grid: `masks` is the listed masks, `cells` the index into them of every grid cell (raster
# order), idx_pb the prob_bits of the index stream.  pb: prob_bits of the residual stream.  flat / idx_flat: write
# that stream with table mode 0 (no frequency table: the decoder spreads 2^pb evenly over the range).
Chan = collections.namedtuple("Chan", "masks cells idx_pb pb flat idx_flat", defaults=(None, None, 8, 15, False, False))
# One written entropy stream: what it holds, its header fields and, for a lone-symbol stream (one distinct symbol
# owns all of 2^pb: HOH_FIX_CARRY territory, which the oracle does not have), its symbols; its length in bytes.
Rec = collections.namedtuple("Rec", "kind n range pb table_mode stored lone symbols size")


class LossyTable(ValueError):
    """The table-mode-1 stream cannot hold a frequency (SURVEY D6): not a valid file."""


def grid_of(w, h):
    return -(-w // GRID), -(-h // GRID)


def tile_geometry(w, h):
    """choh.cpp:454-460 -> (x_tiles, y_tiles, tile_w, tile_h)."""
    xt, yt = (w // 256, h // 256) if (w >= 512 or h >= 512) and w >= 256 and h >= 256 else (1, 1)
    return xt, yt, -(-w // xt), -(-h // yt)


def _flat_stream(symbols, range_, pb):
    """entropy_decoding.hpp:174-179 table mode 0: metadata byte, payload size, rANS payload under the flat counts."""
    n = len(symbols)
    freqs = np.ones(range_, np.uint32)
    cum = np.zeros(range_ + 1, np.uint32)
    assert ol.oracle().orc_normalize_freqs(freqs, cum, range_, 1 << pb) == 0
    out = np.zeros(4 * n + 64, np.uint8)
    k = ol.oracle().orc_rans_encode_static(np.ascontiguousarray(symbols, u16), n, freqs, cum, range_, pb, out)
    return (ol.varint_bytes(range_ - 1) + ol.varint_bytes(n) + bytes([0x80 | pb << 2]) + ol.varint_bytes(k) +
            out[:k].tobytes())


def write_stream(symbols, range_, pb, kind, recs, flat=False):
    """One entropy stream: encode_entropy's own choice of table / stored form, or table mode 0 (flat).  Every stream
    must decode back with the oracle, except a lone-symbol one (recorded with its symbols).  A prob_bits whose
    stream would be a lossy table-mode-1 one is not a valid file: the next lower prob_bits is taken instead (at
    2^pb <= 2^maxbits every frequency fits its field)."""
    assert (1 << pb) >= range_ and 1 <= pb <= 19
    while True:
        try:
            return _write_stream(symbols, range_, pb, kind, recs, flat)
        except LossyTable:
            pb -= 1
            assert (1 << pb) >= range_


def _write_stream(symbols, range_, pb, kind, recs, flat):
    symbols = np.ascontiguousarray(symbols, u16)
    if flat and len(symbols):
        data = _flat_stream(symbols, range_, pb)
    else:
        enc, st = ol.orc_encode_entropy(symbols, range_, pb)
        assert st == 0, (kind, range_, pb)
        data = enc.tobytes()
    r, n, em, pb5, tm = ol.peek_stream(np.frombuffer(data + bytes(4), np.uint8))
    assert (r, n) == (range_, len(symbols))
    lone = n > 0 and em == 1 and tm != 0 and len(np.unique(symbols)) == 1
    if lone:
        assert tm == 2, "HOH_FIX_CARRY recovers a lone symbol from table mode 2 only"
    elif n:
        got, end, st = ol.orc_decode_entropy(np.frombuffer(data, np.uint8), 0, flags=7, cap=n)
        if st != 0 or not np.array_equal(got, symbols):
            raise LossyTable((kind, range_, pb, tm))
        assert end == len(data)
    recs.append(Rec(kind, n, range_, pb5 if em else None, tm if em else None, em == 0 and n > 0, lone,
                    symbols if lone else None, len(data)))
    return data


def _layer(plane, w, h, depth, ch, covered, recs):
    """layer_encode's emission for the given choices: header, [index stream], residuals of the uncovered pixels."""
    plane = np.ascontiguousarray(plane, u16)
    res = np.zeros(w * h, u16)
    if ch.masks is None:
        ol.oracle().orc_predict_fastpath(plane, w, h, depth, res)
        head = bytes([0x10, 0, 0, MED >> 8, MED & 0xff])
    else:
        xt, yt = grid_of(w, h)
        assert xt * yt > 1, "a one-cell grid reads as the single-predictor header"
        assert 1 <= len(ch.masks) <= 14 and len(ch.cells) == xt * yt
        tmap = np.array([ch.masks[i] for i in ch.cells], u16)
        ol.oracle().orc_predict_all(plane, w, h, depth, xt, yt, tmap, res)
        head = (bytes([0x10, xt - 1, yt - 1, len(ch.masks)]) + b"".join(int(m).to_bytes(2, "big") for m in ch.masks) +
                write_stream(ch.cells, len(ch.masks), ch.idx_pb, "idx", recs, ch.idx_flat))
    return head + write_stream(res[~covered], 1 << depth, ch.pb, "resid", recs, ch.flat)


def write_tile(img, colour_mode=128, chans=(Chan(), Chan(), Chan()), matches=(), wide=False, lz_pb=(10, 10, 10, 10),
               lz_flat=False):
    """img (h, w, 3) u8 -> (tile bytes, the image the tile decodes to, [Rec] in stream order).

    matches: (pos, len, back) in pixels, ascending; the image is made consistent with them by forward copying
    before any residual is computed.  The LZ record is the one find_lz_rgb writes (hoh_oracle.c orc_find_lz_rgb):
    tag 0x03, since_last (a gap of g pixels is g // 255 entries of 255 then g % 255; the pixels after the last match
    add entries of 255 only), len - 4, back % 256 and, when wide, back / 256."""
    img = np.array(img, np.uint8)
    h, w = img.shape[:2]
    npx = w * h
    px = img.reshape(npx, 3)
    backref = np.zeros(npx, u16)
    side = [[], [], [], []]
    end = 0
    for pos, ln, back in matches:
        assert end <= pos and 4 <= ln <= 259 and 1 <= back <= pos and pos + ln <= npx
        assert back < (65536 if wide else 256)
        gap = pos - end
        side[0] += [255] * (gap // 255) + [gap % 255]
        side[1].append(ln - 4)
        side[2].append(back % 256)
        side[3].append(back // 256)
        for k in range(ln):
            px[pos + k] = px[pos + k - back]
        backref[pos:pos + ln] = back
        end = pos + ln
    side[0] += [255] * ((npx - end) // 255)
    recs = []
    lz = b"\x03" + b"".join(write_stream(side[k], 256, lz_pb[k], "lz", recs, lz_flat) for k in range(4 if wide else 3))
    covered = backref != 0
    if colour_mode == 128:
        planes = zip(ol.orc_subtract_green(img), (8, 9, 9))
    else:
        assert colour_mode == 2
        planes = ((px[:, c].astype(u16), 8) for c in (1, 0, 2))
    body = [_layer(p, w, h, d, ch, covered, recs) for (p, d), ch in zip(planes, chans)]
    return ol.assemble_tile(lz, colour_mode, body), img, recs


# ---------------------------------------------------------------------------------------------
# the oracle's inverse of a tile (the expected answer, independent of the writer's source image)
# ---------------------------------------------------------------------------------------------
def oracle_decode_tile(tile, w, h, recs):
    """Parse the tile bytes and invert them with the oracle: orc_decode_entropy, the LZ expansion into a
    back-reference map, orc_unpredict_all / orc_unpredict_fastpath, the colour inverse.  Lone-symbol streams take
    the symbols and length from their Rec (the oracle cannot read them back)."""
    b = np.frombuffer(tile, np.uint8)
    npx = w * h
    todo = iter(recs)
    at = 0

    def stream(pos):
        rec = next(todo)
        if rec.lone:
            return rec.symbols, pos + rec.size
        syms, end, st = ol.orc_decode_entropy(b, pos, flags=7, cap=npx + 16)
        assert st == 0 and len(syms) == rec.n and end == pos + rec.size
        return syms, end

    def varint():  # varint.hpp:6-27
        nonlocal at
        b0 = int(b[at]); at += 1
        if not b0 & 0x80:
            return b0
        b1 = int(b[at]); at += 1
        if not b1 & 0x80:
            return ((b0 & 0x7f) << 7) + b1
        b2 = int(b[at]); at += 1
        return ((b0 & 0x7f) << 14) + ((b1 & 0x7f) << 7) + b2

    assert b[0] == 0 and b[1] == 0 and b[3] == 0x03
    colour_mode = int(b[2])
    at = 4
    side = []
    for k in range(4):
        if k == 3 and not (b[at] == 0x81 and b[at + 1] == 0x7f):  # the D3 rule: a 4th stream has range 256
            break
        s, at = stream(at)
        side.append(s)
    backref = np.zeros(npx, u16)
    pos = group = i = 0
    s0 = side[0]
    while i < len(s0):                                           # un_lz.hpp:150-170, D12
        count = 0
        while i < len(s0) and s0[i] == 255:
            count += 255
            i += 1
        if i >= len(s0):
            break
        count += int(s0[i]); i += 1
        pos += count
        back = int(side[2][group]) + (int(side[3][group]) << 8 if len(side) == 4 else 0)
        ln = int(side[1][group]) + 4
        group += 1
        assert 1 <= back <= pos and pos + ln <= npx
        backref[pos:pos + ln] = back
        pos += ln
    assert b[at] == 0x24
    at += 1
    sizes = [varint(), varint()]
    starts = [at, at + sizes[0], at + sizes[0] + sizes[1], len(b)]
    planes = []
    for c in range(3):
        q = starts[c]
        depth = 8 if c == 0 or colour_mode == 2 else 9
        assert b[q] == 0x10
        gx, gy = int(b[q + 1]) + 1, int(b[q + 2]) + 1
        out = np.zeros(npx, u16)
        if gx == gy == 1:
            assert (int(b[q + 3]) << 8 | int(b[q + 4])) == MED
            res, end = stream(q + 5)
            ol.oracle().orc_unpredict_fastpath(np.ascontiguousarray(res, u16), w, h, depth, backref.ctypes.data, out)
        else:
            assert (gx, gy) == grid_of(w, h)
            nm = int(b[q + 3])
            masks = [int(b[q + 4 + 2 * m]) << 8 | int(b[q + 5 + 2 * m]) for m in range(nm)]
            idx, end = stream(q + 4 + 2 * nm)
            tmap = np.array([masks[k] for k in idx], u16)
            res, end = stream(end)
            ol.oracle().orc_unpredict_all(np.ascontiguousarray(res, u16), w, h, depth, gx, gy, tmap,
                                          backref.ctypes.data, out)
        assert end == starts[c + 1] and len(res) == int((backref == 0).sum())
        planes.append(out)
    if colour_mode == 128:
        rgb = np.zeros(npx * 3, np.uint8)
        ol.oracle().orc_add_green(*planes, npx, rgb)
        return rgb.reshape(h, w, 3)
    assert colour_mode == 2
    return np.stack([planes[1], planes[0], planes[2]], axis=-1).astype(np.uint8).reshape(h, w, 3)


# ---------------------------------------------------------------------------------------------
# content and choices
# ---------------------------------------------------------------------------------------------
def photo(rng, w, h):
    return ol.synth_rgb(w, h, int(rng.integers(1, 1 << 30))).reshape(h, w, 3)


def noise(rng, w, h):
    return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


def wide_chroma(rng, w, h):
    """Smooth green, red and blue far from it: the 9-bit R-G / B-G residuals take > 256 distinct values but are
    not uniform, so their streams are coded (not stored) with a table of more than 256 symbols."""
    img = photo(rng, w, h).astype(np.int64)
    for c in (0, 2):
        img[..., c] = np.clip(img[..., 1] + np.rint(rng.laplace(0, 45, (h, w))), 0, 255)
    return img.astype(np.uint8)


def random_matches(rng, w, h, count, max_back, max_len=40):
    """Non-overlapping (pos, len, back), ascending, at random gaps."""
    npx, out, pos = w * h, [], 1
    while len(out) < count:
        pos += int(rng.integers(0, 3 * max_len))
        ln = int(rng.integers(4, max_len + 1))
        if pos + ln > npx:
            break
        out.append((pos, ln, int(rng.integers(1, min(pos, max_back) + 1))))
        pos += ln
    return out


MASK_POOL = [0x0001, 0x8000, 0xffff, 0xffef, 0x0021, 0x4000, 0x0300, 0xfffe]   # single bits, all, no MED ...


def random_masks(rng, k):
    """k distinct non-zero masks, none of them stock (0xffff excepted: it is in the pool on purpose)."""
    out = list(rng.permutation(MASK_POOL)[:min(k, len(MASK_POOL))])
    while len(out) < k:
        m = int(rng.integers(1, 1 << 16))
        if m not in STOCK and m not in out:
            out.append(m)
    return [int(m) for m in out]


def grid_chan(rng, w, h, masks, used=None, **kw):
    """A predictor-grid channel whose cells draw from the first `used` listed masks (default: all)."""
    xt, yt = grid_of(w, h)
    cells = rng.integers(0, used or len(masks), xt * yt)
    if used is None and xt * yt >= len(masks):
        cells[:len(masks)] = rng.permutation(len(masks))      # every listed mask is used
    return Chan(masks=list(masks), cells=[int(c) for c in cells], **kw)


def mask_chans(rng, w, h, i):
    """Rotates through the mask situations: stock masks shuffled, random non-stock masks, 14 masks, a listed mask no
    cell uses, a one-mask list, and the single-predictor header."""
    kind = i % 6
    if kind == 0:
        a = grid_chan(rng, w, h, rng.permutation(STOCK)[:int(rng.integers(2, 15))])
    elif kind == 1:
        a = grid_chan(rng, w, h, random_masks(rng, int(rng.integers(2, 8))))
    elif kind == 2:
        a = grid_chan(rng, w, h, random_masks(rng, 7) + list(rng.permutation(STOCK)[:7]))
    elif kind == 3:
        a = grid_chan(rng, w, h, random_masks(rng, 3), used=2)
    elif kind == 4:
        a = grid_chan(rng, w, h, random_masks(rng, 1))
    else:
        a = Chan()
    b = grid_chan(rng, w, h, rng.permutation(STOCK)[:4])
    c = grid_chan(rng, w, h, [0x8000, 0x0001])
    return [a, b, c][i % 3:] + [a, b, c][:i % 3]


# ---------------------------------------------------------------------------------------------
# the decoder matrix
# ---------------------------------------------------------------------------------------------
Case = collections.namedtuple("Case", "w h n tiles rgb recs distinct walks")


def walks_of(w, h, n):
    """The un-prediction walks hoh_decode_images takes for n images of w x h in one pass per tile shape
    (tile_classes and decode_pass in hoh_api.cu): {walk: [tile shapes]}."""
    xt, yt, tw, th = tile_geometry(w, h)

    def split(size, tiles, t):  # (extent, tiles of that extent) along one axis
        last = size - (tiles - 1) * t
        return [(t, tiles)] if last == t else [(t, tiles - 1), (last, 1)]  # last != t needs tiles > 1

    out = collections.defaultdict(list)
    for sw, cx in split(w, xt, tw):
        for sh, cy in split(h, yt, th):
            if sw % 8 == 0 and sw >= 16:
                walk = "grouped"
            else:
                walk = "halfwarp" if 3 * n * cx * cy <= HALF_WARP_MAX_PLANES else "scalar"
            out[walk].append((sw, sh))
    return dict(out)


def build_case(w, h, n, make_tile, seed, distinct=None):
    """n images of w x h; tile k is make_tile(rng, tile_w, tile_h, k) -> write_tile(...).  distinct: write that many
    tiles and repeat them (the many-plane batches)."""
    rng = np.random.default_rng(seed)
    xt, yt, tw, th = tile_geometry(w, h)
    rgb = np.zeros((n, h, w, 3), np.uint8)
    tiles, recs, made = [], [], {}
    for i in range(n):
        for ty in range(yt):
            for tx in range(xt):
                k = len(tiles)
                j = k if distinct is None else k % distinct
                x0, y0 = tx * tw, ty * th
                sw, sh = min(tw, w - x0), min(th, h - y0)
                if j not in made:
                    made[j] = make_tile(rng, sw, sh, j)
                t, img, rc = made[j]
                assert img.shape == (sh, sw, 3)
                tiles.append(t)
                recs.append(rc)
                rgb[i, y0:y0 + sh, x0:x0 + sw] = img
    return Case(w, h, n, tiles, rgb.ravel(), recs, len(made), walks_of(w, h, n))


def _t_masks(rng, w, h, k):
    """Photographic tile, every mask situation across the tiles, a few LZ matches, colour mode 2 on every 4th."""
    m = random_matches(rng, w, h, int(rng.integers(0, 12)), 255)
    return write_tile(photo(rng, w, h), 2 if k % 4 == 3 else 128, mask_chans(rng, w, h, k), m)


def checker(rng, w, h):
    """A checkerboard of two levels 128 apart, a little noise: MED misses by about half the range, so the residuals
    sit at both ends of it (0, 1, .. and .., 254, 255) and encode_entropy picks table mode 1 (every frequency on
    maxbits bits) over the clamped table."""
    yy, xx = np.mgrid[0:h, 0:w]
    g = ((xx + yy) % 2) * 128 + rng.integers(0, 4, (h, w))
    return np.stack([g + 1, g, g + 2], axis=-1).astype(np.uint8)


def _t_prob_bits(rng, w, h, k):
    """Tile k of the prob_bits sweep: residual streams at 8 + k % 12 (G) and 9 + k % 11 / 19 - k % 11 (R-G, B-G),
    index streams at every value from 1 to 19 across the tiles (flat tables: coded whatever their length; their
    mask count fits 2^pb), the four LZ side streams at 8 .. 19 (flat tables on odd tiles).  B-G takes the flat
    table on odd tiles.  Tile 12 is noise (stored residual streams), tile 13 has wide R-G / B-G residuals (a table
    of more than 256 symbols), tile 14 has G residuals at both ends of the range (table mode 1)."""
    img = {12: noise, 13: wide_chroma, 14: checker}.get(k, photo)(rng, w, h)
    flat = k % 2 == 1
    chans = []
    for c, pb in enumerate((8 if k == 14 else 8 + k % 12, 9 + k % 11, 19 - k % 11)):
        ipb = 1 + (3 * k + c) % 19
        n_masks = min(1 << ipb, 2 + (k + c) % 13)
        chans.append(grid_chan(rng, w, h, random_masks(rng, n_masks), pb=pb, idx_pb=ipb, idx_flat=True,
                               flat=flat and c == 2))
    if k == 14:
        chans[0] = Chan(pb=8)  # MED: a predictor grid's masks would blur the two ends
    m = random_matches(rng, w, h, 160 if k != 14 else 0, 255, max_len=12)  # copies would break the checkerboard
    return write_tile(img, 128, chans, m, wide=True, lz_pb=tuple(8 + (4 * k + s) % 12 for s in range(4)), lz_flat=flat)


def lz_edge_matches(w, h, k):
    """The LZ record's edges: back = 1 over a run, back = pos (copies of pixel 0), back = width, lengths 4 and 259,
    gaps of 254, 255, 256 and 510, a match ending on the last pixel (k = 0) or trailing uncovered pixels (k = 1),
    every pixel but pixel 0 covered (k = 2), no match (k = 3)."""
    npx = w * h
    if k == 2:
        out, pos = [], 1
        while pos < npx:
            out.append((pos, min(259, npx - pos), 1))
            pos += out[-1][1]
        return out
    if k == 3:
        return []
    out = [(1, 4, 1), (100, 20, 100), (374, 259, 1)]          # ends 633
    pos = 633
    for gap, ln, back in ((255, 10, w), (256, 30, 200), (510, 4, 255), (0, 259, w)):
        pos += gap
        out.append((pos, ln, back))
        pos += ln
    if k == 0:
        out.append((npx - 72, 72, 128))
    else:
        out.append((pos + 3, 4, 2))
        assert npx - (pos + 7) > 600
    return out


def _t_lz_edges(rng, w, h, k):
    """Tiles 0 .. 3: lz_edge_matches(k); tile 4: flat grey 128 (every plane at the predictors' start value c / 2)
    and no match, so every residual stream holds one symbol (a lone-symbol table, HOH_FIX_CARRY)."""
    chans = [Chan(), grid_chan(rng, w, h, random_masks(rng, 3)), grid_chan(rng, w, h, rng.permutation(STOCK)[:5])]
    if k == 4:
        return write_tile(np.full((h, w, 3), 128, np.uint8), 128, chans)
    return write_tile(photo(rng, w, h), 2 if k % 2 else 128, chans, lz_edge_matches(w, h, k))


def _t_lz_wide(rng, w, h, k):
    """Tile 0: a 4-stream record with distances up to 65 535 (back = pos = 65 535 copies pixel 0; back = 65 535,
    whole rows, 256, 257, gaps of many 255s).  Tile 1: a 4-stream record whose distances are all < 256 (its 4th
    stream holds zeros only and must still be found by the D3 rule)."""
    npx = w * h
    if k % 2 == 0:
        m = [x for x in random_matches(rng, w, h, 40, 255) if x[0] + x[1] < 65535]
        m += [(65535, 100, 65535), (70000, 259, 65535), (80000, 50, 200 * w), (85000, 20, 256), (86000, 8, 257),
              (npx - 41, 41, 60000)]
    else:
        m = random_matches(rng, w, h, 300, 255, max_len=60)
    # channel 0: four listed masks, every cell on the first (a lone-symbol index stream)
    chans = [grid_chan(rng, w, h, random_masks(rng, 4), used=1), Chan(),
             grid_chan(rng, w, h, rng.permutation(STOCK)[:14])]
    return write_tile(photo(rng, w, h), 2 if k % 2 else 128, chans, m, wide=True)


# name -> (w, h, images, tile maker, distinct tiles or None, the walks the shapes must take)
CASES = {
    "grouped_96x80": (96, 80, 6, _t_masks, None, {"grouped"}),
    "halfwarp_44x30": (44, 30, 6, _t_masks, None, {"halfwarp"}),
    "halfwarp_8x90": (8, 90, 6, _t_masks, None, {"halfwarp"}),
    "scalar_44x30": (44, 30, 5462, _t_masks, 40, {"scalar"}),
    "scalar_8x90": (8, 90, 5462, _t_masks, 40, {"scalar"}),
    "tiled_601x523": (601, 523, 2, _t_masks, None, {"halfwarp"}),
    "tiled_527x523": (527, 523, 2, _t_masks, None, {"grouped", "halfwarp"}),
    "prob_bits_120x100": (120, 100, 15, _t_prob_bits, None, {"grouped"}),
    "lz_edges_64x48": (64, 48, 5, _t_lz_edges, None, {"grouped"}),
    "lz_edges_60x52": (60, 52, 5, _t_lz_edges, None, {"halfwarp"}),
    "lz_wide_300x300": (300, 300, 2, _t_lz_wide, None, {"halfwarp"}),
    "lz_wide_304x300": (304, 300, 2, _t_lz_wide, None, {"grouped"}),
}


@functools.lru_cache(maxsize=None)
def case(name):
    w, h, n, make, distinct, _ = CASES[name]
    return build_case(w, h, n, make, seed=sum(map(ord, name)), distinct=distinct)


def tile_windows(c):
    """(tile index, image, x0, y0, w, h) of every tile of a case, in batch order."""
    xt, yt, tw, th = tile_geometry(c.w, c.h)
    k = 0
    for i in range(c.n):
        for ty in range(yt):
            for tx in range(xt):
                yield k, i, tx * tw, ty * th, min(tw, c.w - tx * tw), min(th, c.h - ty * th)
                k += 1


def matches_of(side, wide):
    """The (pos, len, back) list of find_lz_rgb's raw side streams."""
    out, pos, g, i = [], 0, 0, 0
    while i < len(side[0]):
        if side[0][i] == 255:
            pos += 255
        else:
            pos += int(side[0][i])
            back = int(side[2][g]) + (int(side[3][g]) << 8 if wide else 0)
            out.append((pos, int(side[1][g]) + 4, back))
            pos += out[-1][1]
            g += 1
        i += 1
    return out


# ---------------------------------------------------------------------------------------------
# CPU: the writer against the reference
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["no_lz", "photo_with_repeats"])
def test_writer_equals_encode_tile_at_mode0(kind):
    """With the reference's choices at -s0 (MED header, prob_bits 15, LZ side streams at 10, the matches find_lz_rgb
    takes at distance 6, colour mode 128) the writer's bytes are encode_tile's."""
    rng = np.random.default_rng(5)
    w, h = 96, 80
    tile = photo(rng, w, h) if kind == "no_lz" else ol.photo_with_repeats(rng, w, h, 41)
    distance, bonus = ol.orc_lz_params(tile, 0)
    _, nuke, side = ol.orc_find_lz_rgb(tile, w, distance, bonus)
    m = matches_of(side, distance > 8)
    assert (len(m) == 0) == (kind == "no_lz") and int(nuke.sum()) == sum(x[1] for x in m)
    got, img, _ = write_tile(tile, 128, [Chan(pb=15)] * 3, m, wide=distance > 8)
    want, _ = ol.orc_encode_tile_subgreen(tile, 0)
    assert got == want
    assert np.array_equal(img, tile)  # the matches are the image's own repeats


def test_writer_equals_layer_encode_for_a_grid_plane():
    """A mode-2 plane whose kept stream is the one coded after the predictor search (prob_bits 12, not the stale
    15-bit trial of SURVEY D7): with the masks, cell map and prob_bits layer_encode chose, the writer's layer is
    layer_encode's."""
    w, h = 120, 100
    img = ol.synth_rgb(w, h, 1).reshape(h, w, 3)
    plane = ol.orc_subtract_green(img)[1]
    want, trace = ol.orc_layer_encode(plane, w, h, 9, 2)
    assert trace[0] == 12 and trace[1:3] == list(grid_of(w, h))
    n = int(want[3])
    masks = [int(want[4 + 2 * m]) << 8 | int(want[5 + 2 * m]) for m in range(n)]
    at = 4 + 2 * n
    cells, end, st = ol.orc_decode_entropy(want, at, flags=7, cap=64)
    assert st == 0 and len(cells) == w // GRID * -(-h // GRID)
    _, _, coded, idx_pb, _ = ol.peek_stream(want, at)
    idx_pb = idx_pb if coded else 8  # a stored stream does not record it; layer_encode codes index streams at 8
    res_pb = ol.peek_stream(want, end)[3]
    got = _layer(plane, w, h, 9, Chan(masks, [int(c) for c in cells], idx_pb, res_pb), np.zeros(w * h, bool), [])
    assert got == want.tobytes()


@pytest.mark.parametrize("name", sorted(CASES))
def test_crafted_tiles_decode_with_the_oracle(name):
    """Every tile of the decoder matrix, parsed and inverted by the oracle, gives the image the writer made
    consistent with its matches; and the case's tile shapes take the walks it is named for."""
    c = case(name)
    assert set(c.walks) == CASES[name][5], c.walks
    want = c.rgb.reshape(c.n, c.h, c.w, 3)
    seen = set()
    for k, i, x0, y0, sw, sh in tile_windows(c):
        if c.tiles[k] in seen:
            continue
        seen.add(c.tiles[k])
        got = oracle_decode_tile(c.tiles[k], sw, sh, c.recs[k])
        assert np.array_equal(got, want[i, y0:y0 + sh, x0:x0 + sw]), (name, k)
    assert len(seen) == c.distinct


def test_crafted_streams_cover_every_prob_bits_and_table_form():
    """What the decoder matrix feeds the decoder: residual streams at every prob_bits from the plane's depth to 19,
    index streams from 1 to 19, LZ side streams from 8 to 19, table modes 0, 1 and 2, stored streams, lone-symbol
    streams, 3- and 4-stream LZ records and both colour modes."""
    seen = collections.defaultdict(set)
    records = set()
    for name in CASES:
        c = case(name)
        for t, rc in zip(c.tiles, c.recs):
            records.add((t[2], sum(r.kind == "lz" for r in rc)))
            for r in rc:
                if r.stored:
                    seen["stored", r.kind].add(r.range)
                elif r.pb is not None:
                    seen[r.kind, r.range].add(r.pb)
                    seen["table mode"].add(r.table_mode)
                if r.lone:
                    seen["lone"].add(r.kind)
    every = set(range(1, 20))
    assert seen["resid", 256] >= every - set(range(1, 8))
    assert seen["resid", 512] >= every - set(range(1, 9))
    assert set().union(*(seen["idx", r] for r in range(2, 15))) >= every
    assert seen["lz", 256] >= every - set(range(1, 8))
    assert seen["table mode"] == {0, 1, 2}
    assert {256, 512} <= seen["stored", "resid"] and seen["stored", "idx"] and seen["lone"] >= {"idx", "resid"}
    assert {cm for cm, _ in records} == {2, 128} and {s for _, s in records} == {3, 4}


# ---------------------------------------------------------------------------------------------
# GPU: the decoder matrix
# ---------------------------------------------------------------------------------------------
def check_regions(g, c, seed):
    """hoh_decode_regions over the same batch: one seeded random window size at seeded origins, then the window
    that is the whole image.  Every crop equals the source, sliced."""
    rng = np.random.default_rng(seed)
    want = c.rgb.reshape(c.n, c.h, c.w, 3)
    cw, ch = int(rng.integers(1, c.w + 1)), int(rng.integers(1, c.h + 1))
    windows = [(cw, ch, np.stack([rng.integers(0, c.w - cw + 1, c.n), rng.integers(0, c.h - ch + 1, c.n)], axis=1)),
               (c.w, c.h, np.zeros((c.n, 2), np.int64))]
    for cw, ch, org in windows:
        crops, st = g.decode_regions(c.tiles, c.n, c.w, c.h, org, cw, ch)
        assert (st == 0).all(), (cw, ch, np.flatnonzero(st)[:8])
        for i, (x, y) in enumerate(org):
            assert np.array_equal(crops[i], want[i, y:y + ch, x:x + cw]), (cw, ch, i, x, y)


def decode_profiled(g, c):
    g.profile_begin()
    back, st = g.decode_images(c.tiles, c.n, c.w, c.h)
    return back, st, g.profile_end()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_decoder_matrix(name):
    """Every crafted tile decodes with status 0 to the source pixels, through the walk the case is named for
    (k_dt_unpredict16 runs exactly when a shape takes the half-warp walk); without the profiler (which serialises
    the side streams) the output is the same; the region decoder crops the same pixels."""
    c = case(name)
    g = gpu_lib.gpu()
    back, st, prof = decode_profiled(g, c)
    assert (st == 0).all(), (np.flatnonzero(st)[:8], st[st != 0][:8])
    assert np.array_equal(back, c.rgb), int(np.count_nonzero(back != c.rgb))
    assert ("k_dt_unpredict16" in prof) == ("halfwarp" in c.walks), (c.walks, sorted(prof))
    again, st2 = g.decode_images(c.tiles, c.n, c.w, c.h)
    assert (st2 == 0).all() and np.array_equal(again, back)
    check_regions(g, c, seed=len(name))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["scalar_44x30", "scalar_8x90"])
def test_scalar_batches_through_the_half_warp_walk(name, monkeypatch):
    """The scalar cases' batches again, cut by a small scratch budget into chunks of at most a few thousand planes:
    each chunk takes the half-warp walk, and both walks give the source."""
    c = case(name)
    g = gpu_lib.gpu()
    monkeypatch.setenv("HOH_SCRATCH_GB", "0.05")  # >= 12 KB of scratch per tile: < 4 500 tiles, 13 500 planes a chunk
    back, st, prof = decode_profiled(g, c)
    assert "k_dt_unpredict16" in prof and prof["k_dt_unpredict"][1] >= 2, sorted(prof)
    assert (st == 0).all() and np.array_equal(back, c.rgb)
