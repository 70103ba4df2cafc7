"""hoh_decode_images: the working tile decoder (all cruncher modes, LZ back-references, both photographic colour
modes) against hoh_encode_images — exact round trips at every mode with HOH_FIX_STALE (the decodable variant of
SURVEY D7), at mode 0 also for the byte-exact reference output and for a stock `choh` file."""
import os

import numpy as np
import pytest

import gpu_lib
import oracle_lib as ol

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIX_STALE = 24  # HOH_FIX_ENCODER = HOH_FIX_STALE | HOH_FIX_LONE


def _images(rng, w, h, n, seed, mode):
    imgs = [ol.photo_with_repeats(rng, w, h, seed + i) for i in range(n)]
    if mode > 2 and n > 1:  # uncorrelated channels: the plain-RGB colour mode wins
        imgs[1][..., 0] = rng.integers(0, 256, (h, w))
        imgs[1][..., 2] = rng.integers(0, 256, (h, w))
    return np.concatenate([i.ravel() for i in imgs])


@pytest.mark.parametrize("w,h,mode,n", [(512, 512, 0, 3), (96, 80, 1, 4), (512, 256, 2, 2), (90, 70, 3, 4), (64, 96, 4, 3),
                                        (768, 540, 2, 1), (33, 27, 2, 3)])
def test_roundtrip_all_modes_with_lz(w, h, mode, n):
    g = gpu_lib.gpu()
    rng = np.random.default_rng(17 * mode + w)
    rgb = _images(rng, w, h, n, 700 + mode, mode)
    tiles, rec = g.encode_images(rgb, n, w, h, mode, FIX_STALE)
    assert (rec["status"] == 0).all()
    back, st = g.decode_images(tiles, n, w, h)
    assert (st == 0).all(), st
    assert np.array_equal(back, rgb), int(np.count_nonzero(back != rgb))
    if mode > 2 and n > 1:
        assert 2 in set(rec["colour_mode"])
    # the LZ records are not empty: some pixels really are copies
    assert sum(int(r) for r in rec["lz_size"]) > 20 * len(tiles)


def test_reference_bytes_decode_at_mode0():
    """Without HOH_FIX_STALE the tiles are the reference's bytes; at -s0 those are decodable (D7 needs mode >= 1)."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(2)
    w, h, n = 512, 512, 2
    rgb = _images(rng, w, h, n, 900, 0)
    tiles, rec = g.encode_images(rgb, n, w, h, 0, 0)
    back, st = g.decode_images(tiles, n, w, h)
    assert (st == 0).all() and np.array_equal(back, rgb)


def test_stock_choh_file_decodes():
    """A file written by the real `choh -s0` (tests/golden): the container is parsed here on the host
    (choh.cpp:436-506 read backwards), the tiles are decoded on the device -> the generator image."""
    g = gpu_lib.gpu()
    data = np.load(os.path.join(G, "layer_tile.npz"))["file_512x512_s0"].tobytes()
    assert data[:6] == bytes([153, 72, 79, 72, 2, 8])
    pos = 6

    def varint():
        nonlocal pos
        b0 = data[pos]; pos += 1
        if not b0 & 0x80:
            return b0
        b1 = data[pos]; pos += 1
        if not b1 & 0x80:
            return ((b0 & 0x7f) << 7) + b1
        b2 = data[pos]; pos += 1
        return ((b0 & 0x7f) << 14) + ((b1 & 0x7f) << 7) + b2

    w, h = varint() + 1, varint() + 1
    xt, yt = data[pos] + 1, data[pos + 1] + 1
    pos += 2
    assert (w, h, xt, yt) == (512, 512, 2, 2)
    sizes = [varint() for _ in range(xt * yt - 1)]
    tiles = []
    for s in sizes:
        tiles.append(data[pos:pos + s])
        pos += s
    tiles.append(data[pos:])
    back, st = g.decode_images(tiles, 1, w, h)
    assert (st == 0).all()
    assert np.array_equal(back, ol.synth_rgb(512, 512, 1))


def test_damaged_tiles_are_reported_not_decoded():
    g = gpu_lib.gpu()
    rng = np.random.default_rng(4)
    w, h, n = 96, 80, 4
    rgb = _images(rng, w, h, n, 950, 2)
    tiles, rec = g.encode_images(rgb, n, w, h, 2, FIX_STALE)
    bad = [bytearray(t) for t in tiles]
    bad[0][2] = 77                      # unknown colour mode
    bad[1][3] = 0                       # LZ tag
    bad[2] = bad[2][: len(bad[2]) // 3]  # truncated
    back, st = g.decode_images([bytes(b) for b in bad], n, w, h)
    assert st[0] != 0 and st[1] != 0 and st[3] == 0
    per = w * h * 3
    assert np.array_equal(back[3 * per:], rgb[3 * per:])


def test_reference_bytes_of_flat_and_matchless_images_decode():
    """Reference-format tiles (no encoder-side fixes) whose streams have ONE distinct symbol — the LZ stream of
    255s of every photograph without matches, the residual planes of a flat image — carry the over-wide
    frequency field of SURVEY D6; HOH_FIX_CARRY recognises the pattern and undoes it."""
    g = gpu_lib.gpu()
    w = h = 256
    flat = np.full((h, w, 3), (10, 200, 77), np.uint8)
    flat[100:130, 50:90] = (255, 0, 255)          # 2 colours: palette territory, sub-green bytes are still produced
    photo = ol.synth_rgb(w, h, 3).reshape(h, w, 3)
    rgb = np.concatenate([flat.ravel(), photo.ravel()])
    tiles, rec = g.encode_images(rgb, 2, w, h, 0, 0)
    assert list(rec["flags"]) == [2, 0]
    back, st = g.decode_images(tiles, 2, w, h)
    assert (st == 0).all(), st
    assert np.array_equal(back, rgb)


@pytest.mark.parametrize("w,h,mode,n", [(601, 523, 0, 3), (601, 523, 2, 2), (1000, 700, 1, 2), (530, 300, 4, 2)])
def test_roundtrip_unequal_tiles(w, h, mode, n):
    """Tile grids with up to four tile shapes, batches of several images."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(w + mode)
    rgb = _images(rng, w, h, n, 1200 + mode, mode)
    tiles, rec = g.encode_images(rgb, n, w, h, mode, FIX_STALE)
    assert (rec["status"] == 0).all()
    back, st = g.decode_images(tiles, n, w, h)
    assert (st == 0).all(), st
    assert np.array_equal(back, rgb)


def test_decoder_survives_random_damage():
    """Fuzz: tiles with random byte flips, truncations and garbage tails must never hang or corrupt the decoding of
    their neighbours; a damaged tile either reports a status or decodes to something (it cannot be told apart from
    valid data), and every undamaged tile still decodes exactly."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(99)
    w, h, n = 64, 48, 48
    for mode in (0, 2):
        rgb = _images(rng, w, h, n, 2000 + mode, mode)
        tiles, rec = g.encode_images(rgb, n, w, h, mode, FIX_STALE)
        damaged = []
        bad = set()
        for i, t in enumerate(tiles):
            b = bytearray(t)
            kind = i % 4
            if kind == 1:
                for _ in range(int(rng.integers(1, 6))):
                    b[int(rng.integers(0, len(b)))] = int(rng.integers(0, 256))
            elif kind == 2:
                b = b[: int(rng.integers(1, len(b)))]
            elif kind == 3:
                cut = int(rng.integers(4, len(b)))
                b = b[:cut] + bytes(rng.integers(0, 256, len(b) - cut, dtype=np.uint8))
            if kind:
                bad.add(i)
            damaged.append(bytes(b))
        back, st = g.decode_images(damaged, n, w, h)
        per = w * h * 3
        for i in range(n):
            if i not in bad:
                assert st[i] == 0 and np.array_equal(back[i * per:(i + 1) * per], rgb[i * per:(i + 1) * per]), (mode, i)
        # truncations are always noticed (a stream or channel no longer ends where the tile says); flipped payload
        # bytes are not: rANS carries no checksum
        assert all(st[i] != 0 for i in bad if i % 4 == 2)


def test_roundtrip_many_small_tiles():
    """6 000 tiles = 18 000 planes in one call.  The tiles are 64 wide, a multiple of 8, so every plane takes the
    grouped un-prediction walk whatever the plane count; the one-thread-per-plane walk of other widths above 16 384
    planes is tested in test_gpu_decode_crafted.py."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(8)
    w, h, n = 64, 48, 6000
    base = [ol.photo_with_repeats(rng, w, h, 3000 + i) for i in range(40)]
    rgb = np.concatenate([base[i % 40].ravel() for i in range(n)])
    tiles, rec = g.encode_images(rgb, n, w, h, 2, FIX_STALE)
    assert (rec["status"] == 0).all()
    back, st = g.decode_images(tiles, n, w, h)
    assert (st == 0).all() and np.array_equal(back, rgb)
    # the same batch in the reference's format (this many planes take the two-round candidate schedule of
    # hoh_layer_encode_batch): sampled tiles against the oracle's encode_tile
    ref_tiles, rec = g.encode_images(rgb, n, w, h, 2, 0)
    for i in (0, 7, 1234, 5999):
        want, _ = ol.orc_encode_tile_subgreen(base[i % 40], 2)
        assert ref_tiles[i] == want, i


def test_chunked_walks_equal_one_pass(monkeypatch):
    """hoh_encode_images / hoh_decode_images cut a batch into chunks of whole images under a scratch budget
    (normally a fraction of the device's memory; HOH_SCRATCH_GB overrides).  With a budget of a few megabytes six
    small images take several chunks: same tile bytes as the one-pass call, same decoded pixels."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(99)
    w, h, n = 256, 192, 6
    rgb = _images(rng, w, h, n, 4100, 2)
    tiles_one, rec_one = g.encode_images(rgb, n, w, h, 2, FIX_STALE)
    back_one, st_one = g.decode_images(tiles_one, n, w, h)
    assert (st_one == 0).all() and np.array_equal(back_one, rgb)
    for budget in ("0.004", "0.02"):
        monkeypatch.setenv("HOH_SCRATCH_GB", budget)
        tiles, rec = g.encode_images(rgb, n, w, h, 2, FIX_STALE)
        assert (rec["status"] == 0).all()
        assert tiles == tiles_one, budget
        back, st = g.decode_images(tiles, n, w, h)
        assert (st == 0).all() and np.array_equal(back, rgb), budget


def test_row_distance_65536_stays_decodable_with_the_encoder_fix():
    """lz.hpp:54 accepts whole-row distances up to 65536 inclusive and lz.hpp:88-89 stores a distance in two bytes, so
    65536 is written as 0 — byte-exact with the reference, but undecodable.  A 256-wide tile whose rows repeat 256
    rows further up hits exactly that distance.  flags = 0 must still reproduce the reference's bytes; with
    HOH_FIX_ENCODER the finder stops at 65535 and the tile round-trips."""
    g = gpu_lib.gpu()
    w, h = 256, 300
    img = ol.synth_rgb(w, h, 77).reshape(h, w, 3).copy()
    img[256:] = img[:44]                                    # rows 256.. repeat rows 0..: distance 256 * 256
    flat = img.ravel()
    tiles0, rec0 = g.encode_images(flat, 1, w, h, 2, 0)
    want, nuke = ol.orc_encode_tile_subgreen(img, 2)
    assert tiles0[0] == want and nuke[256 * w:].sum() > 1000   # the reference does take the 65536-distance matches
    tiles, rec = g.encode_images(flat, 1, w, h, 2, 24)
    assert rec["status"][0] == 0
    back, st = g.decode_images(tiles, 1, w, h)
    assert st[0] == 0 and np.array_equal(back, flat)


def test_decode_after_encode_when_device_memory_is_short():
    """The codec's scratch stays cached between calls.  A decode right after an encode must not fail because the
    encoder's cached scratch holds the memory it needs: stale scratch (last used by an earlier top-level call) is freed
    when an allocation fails (hoh_api.cu scratch()).  A ballast leaves less free memory than the decode's scratch."""
    torch = pytest.importorskip("torch")
    mod = gpu_lib.hohgpu()
    g = mod.HohGpu(0)  # its own context: nothing cached from other tests
    try:
        w = h = 256
        n = 768
        rgb = np.concatenate([ol.synth_rgb(w, h, 3000 + i % 7) for i in range(n)])
        geo = g.tile_geometry(w, h)
        n_tiles = n * geo.tiles_per_image
        raw = rgb.size
        cap = raw + raw // 2 + 8192 * n_tiles + 64
        bufs = [g.alloc(raw), g.alloc(cap), g.alloc((n_tiles + 1) * 8), g.alloc(n_tiles * mod.TILE_DT.itemsize),
                g.alloc(raw), g.alloc(n_tiles * 4)]
        d_rgb, d_packed, d_off, d_tiles, d_back, d_st = bufs
        d_rgb.upload(rgb)
        g._ck(g.lib.hoh_encode_images(g.ctx, d_rgb.ptr, n, w, h, 2, FIX_STALE, d_packed.ptr, cap, d_off.ptr, d_tiles.ptr),
              "hoh_encode_images")
        g.sync()
        free_b, _total = torch.cuda.mem_get_info(0)
        ballast = g.alloc(max(free_b - (384 << 20), 1 << 20))  # what is left is far less than the decoder plans for
        bufs.append(ballast)
        g._ck(g.lib.hoh_decode_images(g.ctx, d_packed.ptr, cap, d_off.ptr, n, w, h, d_back.ptr, d_st.ptr), "hoh_decode_images")
        assert (d_st.download(np.int32, n_tiles) == 0).all()
        assert np.array_equal(d_back.download(np.uint8, raw), rgb)
    finally:
        for b in bufs:
            b.free()
        g.close()
