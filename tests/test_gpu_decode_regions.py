"""hoh_decode_regions / hoh_decode_regions_host: a window of every image, decoding only the tiles it touches, against
hoh_decode_images' output sliced in numpy — every tile shape, untiled images, LZ matches, the reference's own bytes, a
stock `choh -s0` file; untouched tiles overwritten, damaged touched tiles, bad windows, the host form over two chunks,
and `dhoh_batch --crop`."""
import os
import subprocess

import numpy as np
import pytest

import gpu_lib
import oracle_lib as ol

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G = os.path.join(HERE, "golden")
FIX_ENCODER = 24  # HOH_FIX_STALE | HOH_FIX_LONE: tiles hoh_decode_images can always invert
E_ARG = 2
S_BAD_WINDOW = 8


def _images(rng, w, h, n, seed):
    return np.concatenate([ol.photo_with_repeats(rng, w, h, seed + i).ravel() for i in range(n)])


def _packed(tiles):
    off = np.zeros(len(tiles) + 1, np.uint64)
    off[1:] = np.cumsum([len(t) for t in tiles])
    return np.frombuffer(b"".join(tiles), np.uint8).copy(), off


_BATCHES = {}


def _batch(w, h, mode, n, flags=FIX_ENCODER):
    """n encoded images (cached per module) and hoh_decode_images' output as (n, h, w, 3)."""
    key = (w, h, mode, n, flags)
    if key not in _BATCHES:
        g = gpu_lib.gpu()
        rgb = _images(np.random.default_rng(w * 7 + h + mode), w, h, n, 300 + 11 * mode)
        tiles, rec = g.encode_images(rgb, n, w, h, mode, flags)
        assert (rec["status"] == 0).all()
        full, st = g.decode_images(tiles, n, w, h)
        assert (st == 0).all() and np.array_equal(full, rgb)
        _BATCHES[key] = (tiles, full.reshape(n, h, w, 3))
    return _BATCHES[key]


def _expect(full, origins, cw, ch):
    return np.stack([full[i, y:y + ch, x:x + cw] for i, (x, y) in enumerate(origins)])


def _both_forms(g, tiles, full, w, h, origins, cw, ch):
    """Device and host form of one window batch: exact crops, status 0."""
    n = full.shape[0]
    want = _expect(full, origins, cw, ch)
    crops, st = g.decode_regions(tiles, n, w, h, origins, cw, ch)
    assert (st == 0).all(), (st, origins, cw, ch)
    assert np.array_equal(crops, want), (origins, cw, ch, int(np.count_nonzero(crops != want)))
    packed, off = _packed(tiles)
    crops_h, st_h = g.decode_regions_host(packed, off, n, w, h, origins, cw, ch)
    assert (st_h == 0).all(), (st_h, origins, cw, ch)
    assert np.array_equal(crops_h, want), (origins, cw, ch)


def _windows(geom, w, h, n, rng):
    """(origins, crop_w, crop_h) batches: random per-image windows, the full image, 1x1 at both corners, one whole tile,
    a four-tile corner, the narrow last column / row, and windows touching the right and bottom edges."""
    tw, th = geom.tile_w, geom.tile_h
    out = []
    for cw, ch in ((min(w, 64), min(h, 48)), (min(w, 300), min(h, 200)), (max(1, w // 3), max(1, h // 2))):
        out.append(([(int(rng.integers(0, w - cw + 1)), int(rng.integers(0, h - ch + 1))) for _ in range(n)], cw, ch))
    out.append(([(0, 0)] * n, w, h))
    out.append(([(0, 0) if i % 2 == 0 else (w - 1, h - 1) for i in range(n)], 1, 1))
    x1 = tw if geom.x_tiles > 1 else 0
    out.append(([(x1, 0)] * n, min(tw, w - x1), th))  # exactly one tile
    if geom.x_tiles > 1 and geom.y_tiles > 1:
        out.append(([(tw - 10, th - 7)] * n, 20, 14))  # straddles the corner of four tiles
    rw, bh = w - (geom.x_tiles - 1) * tw, h - (geom.y_tiles - 1) * th
    out.append(([(w - rw, h - bh)] * n, rw, bh))  # the corner tile of the last column and row
    out.append(([(w - rw + (rw > 1), 1)] * n, max(1, rw - 2), min(5, h - 1)))  # inside the last column
    out.append(([(2, h - bh)] * n, min(9, w - 2), bh))  # inside the last row
    out.append(([(w - min(w, 77), h - min(h, 61))] * n, min(w, 77), min(h, 61)))  # right and bottom edges
    return out


@pytest.mark.parametrize("w,h,mode,n", [(601, 523, 0, 3), (601, 523, 2, 3), (1000, 700, 4, 2), (601, 523, 4, 2),
                                        (3840, 2160, 2, 2), (256, 256, 2, 3), (33, 27, 0, 3), (33, 27, 4, 2)])
def test_windows_equal_full_decode(w, h, mode, n):
    g = gpu_lib.gpu()
    tiles, full = _batch(w, h, mode, n)
    rng = np.random.default_rng(w + mode)
    for origins, cw, ch in _windows(g.tile_geometry(w, h), w, h, n, rng):
        _both_forms(g, tiles, full, w, h, origins, cw, ch)


def test_reference_bytes_at_mode0():
    """flags 0: the reference's own bytes (decodable at -s0)."""
    g = gpu_lib.gpu()
    w, h, n = 601, 523, 2
    tiles, full = _batch(w, h, 0, n, flags=0)
    for origins, cw, ch in _windows(g.tile_geometry(w, h), w, h, n, np.random.default_rng(5))[:4]:
        _both_forms(g, tiles, full, w, h, origins, cw, ch)


def test_stock_choh_file_window():
    """The file the real `choh -s0` wrote (tests/golden, 512x512, 2x2 tiles): its tiles through a window."""
    g = gpu_lib.gpu()
    data = np.load(os.path.join(G, "layer_tile.npz"))["file_512x512_s0"].tobytes()
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
    full, st = g.decode_images(tiles, 1, w, h)
    assert (st == 0).all()
    full = full.reshape(1, h, w, 3)
    for origins, cw, ch in (([(200, 230)], 100, 50), ([(256, 0)], 256, 256), ([(0, 300)], 512, 10)):
        _both_forms(g, tiles, full, w, h, origins, cw, ch)


def _touched(geom, x, y, cw, ch):
    return {ty * geom.x_tiles + tx for ty in range(y // geom.tile_h, (y + ch - 1) // geom.tile_h + 1)
            for tx in range(x // geom.tile_w, (x + cw - 1) // geom.tile_w + 1)}


def test_untouched_tiles_are_never_read():
    """Every tile a window does not touch is overwritten with 0xFF (lengths kept): the crops stay exact."""
    g = gpu_lib.gpu()
    w, h, n = 601, 523, 3
    tiles, full = _batch(w, h, 2, n)
    geom = g.tile_geometry(w, h)
    origins, cw, ch = [(10, 20), (290, 250), (400, 300)], 150, 120
    tpi = geom.tiles_per_image
    wrecked = list(tiles)
    for i, (x, y) in enumerate(origins):
        keep = _touched(geom, x, y, cw, ch)
        for t in range(tpi):
            if t not in keep:
                wrecked[i * tpi + t] = b"\xff" * len(tiles[i * tpi + t])
    assert sum(t == b"\xff" * len(t) for t in wrecked) >= 4
    _both_forms(g, wrecked, full, w, h, origins, cw, ch)


def test_damaged_touched_tile():
    """A flipped payload byte in one touched tile of image 1: that image's status is the tile's, the tile's part of the
    crop keeps the sentinel (device) or is zero (host), everything else is exact."""
    g = gpu_lib.gpu()
    w, h, n = 601, 523, 3
    tiles, full = _batch(w, h, 2, n)
    geom = g.tile_geometry(w, h)
    tpi = geom.tiles_per_image
    origins, cw, ch = [(250, 200)] * n, 100, 100  # the four tiles around (301, 262)
    bad = 1 * tpi + 3  # image 1, bottom-right tile
    damaged = list(tiles)
    b = bytearray(tiles[bad])
    b[len(b) * 2 // 3] ^= 0x5a
    damaged[bad] = bytes(b)
    _, st_full = g.decode_images(damaged, n, w, h)
    assert st_full[bad] != 0 and np.count_nonzero(st_full) == 1
    want = _expect(full, origins, cw, ch)
    # crop pixels that belong to the damaged tile: x >= tile_w, y >= tile_h in image coordinates
    in_bad = np.zeros((ch, cw), bool)
    in_bad[geom.tile_h - 200:, geom.tile_w - 250:] = True
    crops, st = g.decode_regions(damaged, n, w, h, origins, cw, ch, fill=0xA5)
    assert list(st) == [0, int(st_full[bad]), 0]
    assert np.array_equal(crops[[0, 2]], want[[0, 2]])
    assert (crops[1][in_bad] == 0xA5).all()
    assert np.array_equal(crops[1][~in_bad], want[1][~in_bad])
    packed, off = _packed(damaged)
    crops_h, st_h = g.decode_regions_host(packed, off, n, w, h, origins, cw, ch)
    assert list(st_h) == list(st)
    assert np.array_equal(crops_h[[0, 2]], want[[0, 2]])
    assert (crops_h[1][in_bad] == 0).all()
    assert np.array_equal(crops_h[1][~in_bad], want[1][~in_bad])


def test_bad_windows():
    """A window past the right edge fails that image only; an empty or over-wide crop is HOH_E_ARG."""
    g, mod = gpu_lib.gpu(), gpu_lib.hohgpu()
    w, h, n = 601, 523, 3
    tiles, full = _batch(w, h, 0, n)
    origins, cw, ch = [(0, 0), (w - 50, 10), (100, h - 40)], 51, 40
    crops, st = g.decode_regions(tiles, n, w, h, origins, cw, ch, fill=0x3c)
    assert list(st) == [0, S_BAD_WINDOW, 0]
    want = _expect(full, [origins[0], (0, 0), origins[2]], cw, ch)
    assert np.array_equal(crops[[0, 2]], want[[0, 2]]) and (crops[1] == 0x3c).all()
    packed, off = _packed(tiles)
    crops_h, st_h = g.decode_regions_host(packed, off, n, w, h, origins, cw, ch)
    assert list(st_h) == [0, S_BAD_WINDOW, 0]
    assert np.array_equal(crops_h[[0, 2]], want[[0, 2]]) and (crops_h[1] == 0).all()
    for bad_w, bad_h in ((0, 10), (10, 0), (w + 1, 10), (10, h + 1)):
        with pytest.raises(mod.HohError) as e:
            g.decode_regions(tiles, n, w, h, [(0, 0)] * n, bad_w, bad_h)
        assert e.value.status == E_ARG
        with pytest.raises(mod.HohError) as e:
            g.decode_regions_host(packed, off, n, w, h, [(0, 0)] * n, bad_w, bad_h)
        assert e.value.status == E_ARG


def test_host_form_over_two_chunks(monkeypatch):
    """HOH_PIPE_CHUNK_KB lowers the chunk floor: the host form runs two chunks and returns what the device form does,
    a damaged tile and a bad window included; backwards offsets are HOH_E_ARG and leave the context usable."""
    g, mod = gpu_lib.gpu(), gpu_lib.hohgpu()
    w, h, n = 601, 523, 6
    tiles, full = _batch(w, h, 2, n)
    tpi = g.tile_geometry(w, h).tiles_per_image
    damaged = list(tiles)
    b = bytearray(tiles[4 * tpi])
    b[len(b) // 2] ^= 0x81
    damaged[4 * tpi] = bytes(b)
    rng = np.random.default_rng(11)
    cw, ch = 200, 150
    origins = [(int(rng.integers(0, w - cw + 1)), int(rng.integers(0, h - ch + 1))) for _ in range(n)]
    origins[4] = (0, 0)  # touches the damaged tile
    origins[2] = (w - cw + 1, 0)  # does not fit
    crops, st = g.decode_regions(damaged, n, w, h, origins, cw, ch)
    assert st[2] == S_BAD_WINDOW and st[4] != 0 and np.count_nonzero(st) == 2
    monkeypatch.setenv("HOH_PIPE_CHUNK_KB", "256")
    packed, off = _packed(damaged)
    crops_h, st_h = g.decode_regions_host(packed, off, n, w, h, origins, cw, ch)
    assert list(st_h) == list(st)
    ok = [i for i in range(n) if st[i] == 0]
    assert np.array_equal(crops_h[ok], crops[ok])
    inside = [(0, 0) if i == 2 else o for i, o in enumerate(origins)]  # image 2's window does not fit: not compared
    assert np.array_equal(crops_h[ok], _expect(full, inside, cw, ch)[ok])
    backwards = off.copy()  # inside the first tile row of image 1's window
    t0 = 1 * tpi + min(_touched(g.tile_geometry(w, h), origins[1][0], origins[1][1], cw, ch))
    backwards[t0 + 1] = backwards[t0] - 1
    with pytest.raises(mod.HohError) as e:
        g.decode_regions_host(packed, backwards, n, w, h, origins, cw, ch)
    assert e.value.status == E_ARG
    crops_h2, st_h2 = g.decode_regions_host(packed, off, n, w, h, origins, cw, ch)
    assert list(st_h2) == list(st) and np.array_equal(crops_h2[ok], crops[ok])


def test_dhoh_batch_crop(tmp_path):
    """choh_batch --decodable -> dhoh_batch --crop: the .rgb written is the window of the image; a window outside an
    image exits 1."""
    exe_dir = os.path.join(ROOT, "dropin", "_bin")
    if not os.path.exists(os.path.join(exe_dir, "dhoh_batch")):
        subprocess.run(["make", "-C", os.path.join(ROOT, "dropin"), "tools"], check=True, capture_output=True)
    w, h, mode = 601, 523, 2
    rng = np.random.default_rng(23)
    names, imgs = [], []
    for i in range(3):
        img = ol.photo_with_repeats(rng, w, h, 40 + i)
        p = tmp_path / f"p{i}.rgb"
        p.write_bytes(img.tobytes())
        names.append(str(p))
        imgs.append(img)
    enc, dec = tmp_path / "enc", tmp_path / "dec"
    enc.mkdir()
    dec.mkdir()
    run = lambda cmd: subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    r = run([os.path.join(exe_dir, "choh_batch"), "--batch", "--decodable", str(w), str(h), f"-s{mode}", str(enc)] + names)
    assert r.returncode == 0, r.stderr
    hoh = [str(enc / f"p{i}.hoh") for i in range(3)]
    x, y, cw, ch = 280, 240, 123, 45
    r = run([os.path.join(exe_dir, "dhoh_batch"), "--crop", str(x), str(y), str(cw), str(ch), "--batch", str(dec)] + hoh)
    assert r.returncode == 0, r.stderr
    for i in range(3):
        assert (dec / f"p{i}.rgb").read_bytes() == imgs[i][y:y + ch, x:x + cw].tobytes(), i
    r = run([os.path.join(exe_dir, "dhoh_batch"), "--crop", str(w - 10), "0", "11", "5", hoh[0], str(tmp_path / "o.rgb")])
    assert r.returncode == 1
