#!/usr/bin/env python
"""Region decode against full decode: N frames of 3840x2160 (BASELINE config 3's frame size) encoded at cruncher
modes 0 and 2 with HOH_FIX_ENCODER, and one seeded random 512x512 window per frame.

    python tools/bench_regions.py [--frames 64] [--steps 5] [--warmup 1] [--size 512] [--modes 0,2]

Per mode:
  device: ms per call of hoh_decode_images vs hoh_decode_regions on device-resident payloads (CUDA events), and the
          tiles the windows touch vs all tiles;
  host:   ms end to end of hoh_decode_images_host vs hoh_decode_regions_host from pinned buffers (host clock around
          the synchronous calls), and the payload bytes each sends host-to-device: every tile (tile_off[-1]) vs the
          touched tile rows; and the time to move those rows: one copy per row (what the library does) vs a gather
          into pinned staging and one copy;
  exact:  every crop equals the full decode, sliced, and every status is 0.
Prints one JSON line.  Development tool: bench.py stays the judged benchmark."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gpu_lib  # noqa: E402
import oracle_lib as ol  # noqa: E402

FIX_ENCODER = 24
W, H = 3840, 2160
PERIOD = 4  # distinct frames; the batch repeats them (each tile is decoded on its own either way)


def gpu_name():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def touched(geom, x, y, cw, ch):
    """Tile rows [a, b) of the image's tile grid the window touches (what the host form copies)."""
    tx0, tx1 = x // geom.tile_w, (x + cw - 1) // geom.tile_w
    return [(ty * geom.x_tiles + tx0, ty * geom.x_tiles + tx1 + 1)
            for ty in range(y // geom.tile_h, (y + ch - 1) // geom.tile_h + 1)]


def run_mode(g, mod, frames, mode, size, steps, warmup, rng):
    lib, ctx = g.lib, g.ctx
    geom = g.tile_geometry(W, H)
    tpi, raw1 = geom.tiles_per_image, W * H * 3
    n_tiles = frames * tpi
    base = [ol.photo_with_repeats(np.random.default_rng(100 + i), W, H, 500 + i).ravel() for i in range(PERIOD)]
    rgb = np.concatenate([base[i % PERIOD] for i in range(frames)])
    cap = rgb.nbytes * 2 + 8192 * n_tiles
    d_rgb = g.alloc(rgb.nbytes).upload(rgb)
    d_packed = g.alloc(cap)
    d_off = g.alloc((n_tiles + 1) * 8)
    d_rec = g.alloc(n_tiles * mod.TILE_DT.itemsize)
    g._ck(lib.hoh_encode_images(ctx, d_rgb.ptr, frames, W, H, mode, FIX_ENCODER, d_packed.ptr, cap, d_off.ptr,
                                d_rec.ptr), "hoh_encode_images")
    off = d_off.download(np.uint64, n_tiles + 1)
    total = int(off[-1])
    packed_bytes = total + 64  # the device input contract: zero padding behind the last tile
    g._ck(lib.hoh_dev_memset(ctx, d_packed.ptr + total, 0, 64), "hoh_dev_memset")
    origins = np.stack([rng.integers(0, W - size + 1, frames), rng.integers(0, H - size + 1, frames)], 1).astype(np.uint32)
    d_org = g.alloc(origins.nbytes).upload(origins)
    crop1 = size * size * 3
    d_crops = g.alloc(frames * crop1)
    d_st = g.alloc(n_tiles * 4)
    d_rst = g.alloc(frames * 4)

    def full():
        g._ck(lib.hoh_decode_images(ctx, d_packed.ptr, packed_bytes, d_off.ptr, frames, W, H, d_rgb.ptr, d_st.ptr),
              "hoh_decode_images")

    def region():
        g._ck(lib.hoh_decode_regions(ctx, d_packed.ptr, packed_bytes, d_off.ptr, frames, W, H, d_org.ptr, size, size,
                                     d_crops.ptr, d_rst.ptr), "hoh_decode_regions")

    def device_ms(fn):
        for _ in range(warmup):
            fn()
        g.sync()
        g.timer_start(0)
        for _ in range(steps):
            fn()
        g.timer_stop(0)
        return g.timer_ms(0) / steps

    # alternate the two calls so that both see the same state of the shared machine
    ms_full, ms_region = [], []
    for _ in range(2):
        ms_full.append(device_ms(full))
        ms_region.append(device_ms(region))
    whole = d_rgb.download(np.uint8, frames * raw1).reshape(frames, H, W, 3)
    crops = d_crops.download(np.uint8, frames * crop1).reshape(frames, size, size, 3)
    st_full, st_reg = d_st.download(np.int32, n_tiles), d_rst.download(np.int32, frames)
    exact_dev = bool((st_full == 0).all() and (st_reg == 0).all() and all(
        np.array_equal(crops[i], whole[i, y:y + size, x:x + size]) for i, (x, y) in enumerate(origins)))
    runs = [touched(geom, int(x), int(y), size, size) for x, y in origins]
    tiles_touched = sum(b - a for r in runs for a, b in r)
    h2d_region = sum(int(off[i * tpi + b] - off[i * tpi + a]) for i, r in enumerate(runs) for a, b in r)

    # host-buffer forms from pinned memory
    packed_h = g.host_alloc(total)
    packed_h[:] = d_packed.download(np.uint8, total)
    rgb_h = g.host_alloc(frames * raw1)
    crops_h = g.host_alloc(frames * crop1)
    st_h = np.zeros(n_tiles, np.int32)
    rst_h = np.zeros(frames, np.int32)

    def full_host():
        g._ck(lib.hoh_decode_images_host(ctx, packed_h.ctypes.data, total, off.ctypes.data, frames, W, H,
                                         rgb_h.ctypes.data, st_h.ctypes.data), "hoh_decode_images_host")

    def region_host():
        g._ck(lib.hoh_decode_regions_host(ctx, packed_h.ctypes.data, total, off.ctypes.data, frames, W, H,
                                          origins.ctypes.data, size, size, crops_h.ctypes.data, rst_h.ctypes.data),
              "hoh_decode_regions_host")

    def host_ms(fn):
        for _ in range(warmup):
            fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        return (time.perf_counter() - t0) * 1e3 / steps

    hms_full, hms_region = [], []
    for _ in range(2):
        hms_full.append(host_ms(full_host))
        hms_region.append(host_ms(region_host))
    exact_host = bool((rst_h == 0).all() and np.array_equal(crops_h.reshape(frames, size, size, 3), crops))

    # how the host form moves the touched tile rows: one cudaMemcpyAsync per run from the caller's pinned buffer (what
    # hoh_decode_regions_host does) against a host-side gather into pinned staging followed by one copy
    spans = [(int(off[i * tpi + a]), int(off[i * tpi + b])) for i, r in enumerate(runs) for a, b in r]
    stage = g.host_alloc(h2d_region)
    d_stage = g.alloc(h2d_region)

    def per_run():
        at = 0
        for lo, hi in spans:
            g._ck(lib.hoh_h2d(ctx, d_stage.ptr + at, packed_h.ctypes.data + lo, hi - lo), "hoh_h2d")
            at += hi - lo
        g.sync()

    def gather():
        at = 0
        for lo, hi in spans:
            stage[at:at + hi - lo] = packed_h[lo:hi]
            at += hi - lo
        g._ck(lib.hoh_h2d(ctx, d_stage.ptr, stage.ctypes.data, h2d_region), "hoh_h2d")
        g.sync()

    copy_runs, copy_gather = [], []
    for _ in range(2):
        copy_runs.append(host_ms(per_run))
        copy_gather.append(host_ms(gather))
    d_stage.free()
    g.host_free(stage)
    for b in (d_rgb, d_packed, d_off, d_rec, d_org, d_crops, d_st, d_rst):
        b.free()
    for a in (packed_h, rgb_h, crops_h):
        g.host_free(a)
    dev_full, dev_reg = min(ms_full), min(ms_region)
    host_full, host_reg = min(hms_full), min(hms_region)
    return {"mode": mode, "frames": frames, "window": size,
            "device": {"ms_full": round(dev_full, 2), "ms_region": round(dev_reg, 2),
                       "speedup": round(dev_full / dev_reg, 2), "ms_full_runs": [round(v, 2) for v in ms_full],
                       "ms_region_runs": [round(v, 2) for v in ms_region],
                       "tiles_touched": tiles_touched, "tiles_total": n_tiles},
            "host": {"ms_full": round(host_full, 2), "ms_region": round(host_reg, 2),
                     "speedup": round(host_full / host_reg, 2), "ms_full_runs": [round(v, 2) for v in hms_full],
                     "ms_region_runs": [round(v, 2) for v in hms_region],
                     "h2d_bytes_full": total, "h2d_bytes_region": h2d_region, "h2d_copies_region": len(spans),
                     "copy_ms_per_run": round(min(copy_runs), 3), "copy_ms_gather": round(min(copy_gather), 3)},
            "exact": exact_dev and exact_host}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--modes", default="0,2")
    a = ap.parse_args()
    if a.frames < 1 or a.steps < 1 or not 1 <= a.size <= min(W, H):
        ap.error("--frames and --steps must be >= 1, --size in 1..2160")
    g, mod = gpu_lib.gpu(), gpu_lib.hohgpu()
    rng = np.random.default_rng(2026)
    out = {"gpu": gpu_name(), "width": W, "height": H,
           "modes": [run_mode(g, mod, a.frames, int(m), a.size, a.steps, a.warmup, rng) for m in a.modes.split(",")]}
    out["exact"] = all(m["exact"] for m in out["modes"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
