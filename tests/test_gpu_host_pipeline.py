"""The pipelined host-buffer calls (hoh_{en,de}code_images[_s0]_host) where the other suites do not reach them: the
whole-tile calls over more than one chunk, a capacity failure with chunks still in flight, and offset tables the
decoders must refuse."""
import numpy as np
import pytest

import gpu_lib
import oracle_lib as ol

pytestmark = pytest.mark.gpu

W = H = 1024
N = 90  # 270 MB of pixels: just above the 256 MB floor of a whole-tile chunk, so chunks of 86 and 4 images
PERIOD = 5
FIX_ENCODER = 24  # HOH_FIX_ENCODER: tiles hoh_decode_images can always invert


@pytest.fixture(scope="module")
def big_batch():
    """N images repeating with period PERIOD in pinned memory, with pinned buffers for the codes and the pixels."""
    g = gpu_lib.gpu()
    geom = g.tile_geometry(W, H)
    n_tiles = N * geom.tiles_per_image
    raw1 = W * H * 3
    rng = np.random.default_rng(7)
    imgs = [ol.photo_with_repeats(rng, W, H, 90 + i).ravel() for i in range(PERIOD)]
    rgb = g.host_alloc(N * raw1)
    for i in range(N):
        rgb[i * raw1:(i + 1) * raw1] = imgs[i % PERIOD]
    cap = N * raw1 + N * raw1 // 2 + 8192 * n_tiles
    return dict(g=g, geom=geom, n_tiles=n_tiles, rgb=rgb, cap=cap, packed=g.host_alloc(cap),
                back=g.host_alloc(N * raw1))


def _encode_host(b, mode, cap):
    g, mod = b["g"], gpu_lib.hohgpu()
    off = np.zeros(b["n_tiles"] + 1, np.uint64)
    rec = np.zeros(b["n_tiles"], mod.TILE_DT)
    st = g.lib.hoh_encode_images_host(g.ctx, b["rgb"].ctypes.data, N, W, H, mode, FIX_ENCODER, b["packed"].ctypes.data,
                                      cap, off.ctypes.data, rec.ctypes.data)
    return st, off, rec


@pytest.mark.parametrize("mode", [0, 2])
def test_whole_tile_host_calls_over_two_chunks(big_batch, mode):
    """Two chunks of whole images through hoh_encode_images_host / hoh_decode_images_host: the same tiles and offsets
    as the device form, tile records rebased across the chunks, and an exact round trip."""
    b, mod = big_batch, gpu_lib.hohgpu()
    g = b["g"]
    st, off, rec = _encode_host(b, mode, b["cap"])
    g._ck(st, "hoh_encode_images_host")
    assert (rec["status"] == 0).all()
    tiles, rec_dev = g.encode_images(b["rgb"], N, W, H, mode, FIX_ENCODER)
    assert np.array_equal(off, np.concatenate([[0], np.cumsum([len(t) for t in tiles])]).astype(np.uint64))
    assert b["packed"][:int(off[-1])].tobytes() == b"".join(tiles)
    assert np.array_equal(rec["start"], off[:-1])
    assert np.array_equal(rec["size"], rec_dev["size"])
    status = np.full(b["n_tiles"], -1, np.int32)
    g._ck(g.lib.hoh_decode_images_host(g.ctx, b["packed"].ctypes.data, int(off[-1]), off.ctypes.data, N, W, H,
                                       b["back"].ctypes.data, status.ctypes.data), "hoh_decode_images_host")
    assert (status == 0).all()
    assert np.array_equal(b["back"], b["rgb"])


def test_whole_tile_encode_capacity_failure_drains(big_batch):
    """A packed_cap that holds the first chunk but not the second: HOH_E_CAPACITY while the first chunk's fetch is in
    flight, then the same context encodes the batch correctly."""
    b, mod = big_batch, gpu_lib.hohgpu()
    st, off, _ = _encode_host(b, 0, b["cap"])
    b["g"]._ck(st, "hoh_encode_images_host")
    want = b["packed"][:int(off[-1])].tobytes()
    first_chunk = int(off[86 * b["geom"].tiles_per_image])
    st, _, _ = _encode_host(b, 0, first_chunk + 1)
    assert st == mod.HOH_E_CAPACITY
    st, off2, rec = _encode_host(b, 0, b["cap"])
    b["g"]._ck(st, "hoh_encode_images_host")
    assert np.array_equal(off2, off) and b["packed"][:int(off[-1])].tobytes() == want
    assert np.array_equal(rec["start"], off[:-1])


def test_s0_encode_capacity_failure_drains(monkeypatch):
    """hoh_encode_images_s0_host with several chunks queued (the ramped plan of test_host_buffer_pipeline_ramped_chunks)
    and a packed_cap too small for the first one: HOH_E_CAPACITY, then the same context returns the device path's
    bytes."""
    monkeypatch.setenv("HOH_PIPE_CHUNK_KB", "200")
    g, mod = gpu_lib.gpu(), gpu_lib.hohgpu()
    w = h = 128
    n = 64
    rgb = g.host_alloc(n * w * h * 3)
    for i in range(n):
        rgb[i * w * h * 3:(i + 1) * w * h * 3] = ol.synth_rgb(w, h, 31 + i)
    ns = n * g.tile_geometry(w, h).streams_per_image
    cap = rgb.size * 2 + 4096 * ns
    packed = g.host_alloc(cap)
    off = np.zeros(ns + 1, np.uint64)
    res = np.zeros(ns, mod.RESULT_DT)

    def encode(c):
        return g.lib.hoh_encode_images_s0_host(g.ctx, rgb.ctypes.data, n, w, h, packed.ctypes.data, c, off.ctypes.data,
                                               res.ctypes.data)

    assert encode(1000) == mod.HOH_E_CAPACITY
    g._ck(encode(cap), "hoh_encode_images_s0_host")
    assert (res["status"] == 0).all()
    ref_packed, ref_off, _ = g.encode_images_s0(np.asarray(rgb), n, w, h)
    assert np.array_equal(off, ref_off)
    assert packed[:int(ref_off[-1])].tobytes() == ref_packed.tobytes()


def test_decoders_refuse_bad_offsets():
    """Both host decoders: an offset table that runs backwards, or ends beyond packed_bytes, is HOH_E_ARG."""
    g, mod = gpu_lib.gpu(), gpu_lib.hohgpu()
    w = h = 256
    n = 2
    rng = np.random.default_rng(3)
    rgb = np.concatenate([ol.photo_with_repeats(rng, w, h, 5 + i).ravel() for i in range(n)])
    out = np.zeros(rgb.size, np.uint8)
    packed, off, _ = g.encode_images_s0(rgb, n, w, h)
    tiles, _ = g.encode_images(rgb, n, w, h, 0, FIX_ENCODER)
    tile_packed = np.frombuffer(b"".join(tiles), np.uint8)
    tile_off = np.concatenate([[0], np.cumsum([len(t) for t in tiles])]).astype(np.uint64)
    for fn, data, o in [(g.lib.hoh_decode_images_s0_host, packed, off),
                        (g.lib.hoh_decode_images_host, tile_packed, tile_off)]:
        status = np.zeros(len(o) - 1, np.int32)

        def decode(offsets, nbytes):
            offsets = np.ascontiguousarray(offsets, np.uint64)
            return fn(g.ctx, data.ctypes.data, nbytes, offsets.ctypes.data, n, w, h, out.ctypes.data,
                      status.ctypes.data)

        assert decode(o[::-1], data.size) == mod.HOH_E_ARG
        assert decode(o, data.size - 1) == mod.HOH_E_ARG
        g._ck(decode(o, data.size), "host decode")
        assert (status == 0).all() and np.array_equal(out, rgb)
