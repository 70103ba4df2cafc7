#!/usr/bin/env python
"""bench.py — hoh-ANS hot path on B200: raw RGB MB/s, encode + decode, cruncher mode 0.

Workload (BASELINE.json configs[1]): a batch of 4096 synthetic 512x512 RGB images per GPU at -s0.
One "step" = encode the whole batch (RGB -> channel payloads + offset table) and decode it back
(payloads -> RGB).  `value` counts every raw byte once per direction:
    value = 2 * raw_bytes_all_ranks / (t_encode + t_decode)      [MB/s, 1 MB = 1e6 B]
with inputs already resident in HBM; `e2e` is the same metric through the host-buffer C-ABI calls
(hoh_encode_images_s0_host / hoh_decode_images_s0_host) with H2D/D2H inside the timed region.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
N > 1: launched by torchrun, one rank per GPU, images sharded by index, no data-path collective.
"""
import argparse
import atexit
import ctypes as C
import importlib.util
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
W = H = 512
MODE = 0


def _load(name, path):
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------------------
# synthetic inputs (tools/synth_gen.c, SURVEY section 8(d))
# ------------------------------------------------------------------------------------------------
_SYNTH_DIR = None


def synth_lib():
    """tools/synth_gen.c compiled into a per-process temporary directory: the tree may be read-only."""
    global _SYNTH_DIR
    if _SYNTH_DIR is None:
        _SYNTH_DIR = tempfile.mkdtemp(prefix="hoh_bench_")
        atexit.register(shutil.rmtree, _SYNTH_DIR, True)
    so = os.path.join(_SYNTH_DIR, "libsynth.so")
    if not os.path.exists(so):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-o", so, os.path.join(ROOT, "tools", "synth_gen.c")])
    L = C.CDLL(so)
    L.synth_rgb_batch.restype = None
    L.synth_rgb_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_size_t]
    return L


def fill_images(dst, first_seed, count, w, h, threads):
    """dst: uint8 array of count*w*h*3; image i uses seed first_seed + i."""
    L = synth_lib()
    per = w * h * 3
    base = dst.ctypes.data
    chunk = max(1, (count + threads - 1) // threads)
    jobs = []
    for lo in range(0, count, chunk):
        n = min(chunk, count - lo)
        t = threading.Thread(target=L.synth_rgb_batch, args=(base + lo * per, w, h, first_seed + lo, n))
        t.start()
        jobs.append(t)
    for t in jobs:
        t.join()


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region.  NVML is polled from a thread every ~2 ms (the
    timed region of a default run is ~150 ms, shorter than one nvidia-smi start-up); when NVML cannot be
    loaded an `nvidia-smi -lms` child started at construction is used and only the lines it printed between
    start() and stop() are counted."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index):
        import threading
        self.idx = gpu_index
        self.sm, self.reason_bits, self.mx = [], 0, None
        self.recording = False
        self.alive = True
        self.nvml = None
        self.proc = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = gpu_index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                phys = int(vis.split(",")[gpu_index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self.nvml = None
            self.path = os.path.join(tempfile.gettempdir(), f"hoh_clocks_{os.getpid()}.csv")
            try:
                self.out = open(self.path, "w")
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                              "--format=csv,noheader,nounits", "-lms", "20"],
                                             stdout=self.out, stderr=subprocess.DEVNULL)
            except Exception:
                self.proc = None

    def _poll(self):
        nv = self.nvml
        while self.alive:
            if self.recording:
                try:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                    try:
                        self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                    except Exception:
                        self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                except Exception:
                    pass
            time.sleep(0.002)

    def start(self):
        if self.proc:
            self.out.flush()
            self.pos0 = os.path.getsize(self.path)
        self.recording = True

    def stop(self):
        self.recording = False
        self.alive = False
        if self.nvml:
            self.thread.join(timeout=2)
            if not self.sm:
                return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": ["no samples"]}
            reasons = sorted(k for k, bit in self.BITS.items() if self.reason_bits & bit)
            return {"sm_mhz": float(np.median(self.sm)), "sm_min_mhz": float(np.min(self.sm)), "sm_max_mhz": self.mx,
                    "reasons": reasons, "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        pos1 = os.path.getsize(self.path)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as fh:
            fh.seek(self.pos0)
            text = fh.read(max(0, pos1 - self.pos0))
        for line in text.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own hot path (oracle/_ref, else the oracle port) on host cores
# ------------------------------------------------------------------------------------------------
class TileGrid:
    """choh.cpp:454-460: the 256-pixel tiling rule (host arithmetic for the CPU arm)."""

    def __init__(self, w, h):
        if (w >= 512 or h >= 512) and w >= 256 and h >= 256:
            self.x_tiles, self.y_tiles = w // 256, h // 256
        else:
            self.x_tiles = self.y_tiles = 1
        self.tile_w = (w + self.x_tiles - 1) // self.x_tiles
        self.tile_h = (h + self.y_tiles - 1) // self.y_tiles
        self.tiles_per_image = self.x_tiles * self.y_tiles


def tile_grid(w, h):
    return TileGrid(w, h)


def load_reference_in_parent():
    """dlopen oracle/_ref/libhohref.so (or the oracle port) in THIS process before the workers are forked, so that
    a driver looking at the process's mapped libraries sees what the CPU arm really runs."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    ol.oracle()
    if ol.have_ref():
        ol.ref()
        return "reference"
    return "port"


def _whole_tool_worker(args):
    """Stock `choh` (choh.cpp:394 main, through oracle/_ref's ref_choh_main): file in, file out, LZ included."""
    first_seed, count, w, h, mode, tmpdir = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    if not ol.have_ref():
        return None
    R = ol.ref()
    rgb = np.zeros(w * h * 3, np.uint8)
    busy = 0.0
    out_bytes = 0
    for i in range(count):
        synth_lib().synth_rgb_batch(rgb.ctypes.data, w, h, first_seed + i, 1)
        src = os.path.join(tmpdir, f"in_{os.getpid()}_{i}.rgb")
        dst = os.path.join(tmpdir, f"out_{os.getpid()}_{i}.hoh")
        rgb.tofile(src)
        t0 = time.perf_counter()
        devnull = os.open(os.devnull, os.O_WRONLY)  # choh prints the size
        saved = os.dup(1)
        os.dup2(devnull, 1)
        try:
            rc = R.ref_choh_main(src.encode(), dst.encode(), w, h, mode)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
            os.close(devnull)
        busy += time.perf_counter() - t0
        assert rc == 0
        out_bytes += os.path.getsize(dst)
        os.remove(src)
        os.remove(dst)
    return busy, count * w * h * 3, out_bytes


def cpu_whole_tool(images, w, h, mode, cores, seed0=1):
    """BASELINE.md section 3.1: stock choh, one process per core, over `images` images.  MB/s of raw RGB over the
    busy time of the slowest worker.  Encode only: the reference's dhoh cannot decode choh's output."""
    import multiprocessing as mp
    synth_lib()  # compiled once, before the workers fork
    per = [images // cores + (1 if i < images % cores else 0) for i in range(cores)]
    with tempfile.TemporaryDirectory() as tmp:
        jobs, seed = [], seed0
        for n in per:
            if n:
                jobs.append((seed, n, w, h, mode, tmp))
                seed += n
        with mp.get_context("fork").Pool(len(jobs)) as pool:
            res = pool.map(_whole_tool_worker, jobs)
    if any(r is None for r in res):
        return None
    raw = sum(r[1] for r in res)
    slowest = max(r[0] for r in res)
    return {"encode_mbs": raw / slowest / 1e6, "cores": len(jobs), "images": images, "mode": mode,
            "compressed_ratio": sum(r[2] for r in res) / raw,
            "what": "stock choh main() file to file (host LZ, colour-mode competition, container), one process per "
                    "core; decode has no whole-tool figure because dhoh cannot read choh's files"}


def _tile_worker(args):
    """reference encode_tile (choh.cpp:104) on whole tiles of a given shape and mode: the CPU figure beside the
    mode >= 1 configurations."""
    first_seed, count, w, h, mode = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    busy = 0.0
    for i in range(count):
        rgb = ol.synth_rgb(w, h, first_seed + i)
        t0 = time.perf_counter()
        if ol.have_ref():
            buf = np.zeros(rgb.size * 3 + 4096, np.uint8)
            ol.ref().ref_encode_tile(rgb, rgb.size, buf, w, h, mode)
        else:
            ol.orc_encode_tile_subgreen(rgb.reshape(h, w, 3), mode)
        busy += time.perf_counter() - t0
    return busy


def cpu_encode_tiles(tiles, w, h, mode, cores):
    import multiprocessing as mp
    per = [tiles // cores + (1 if i < tiles % cores else 0) for i in range(cores)]
    jobs = [(1000 + 97 * i, n, w, h, mode) for i, n in enumerate(per) if n]
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        res = pool.map(_tile_worker, jobs)
    return {"encode_mbs": tiles * w * h * 3 / max(res) / 1e6, "cores": len(jobs), "tiles": tiles,
            "ms_per_tile_one_core": 1e3 * sum(res) / tiles}


def _cpu_worker(args):
    first_seed, count, w, h = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    use_ref = ol.have_ref()
    R = ol.ref() if use_ref else None
    O = ol.oracle()
    rgb = np.zeros(count * w * h * 3, np.uint8)
    synth_lib().synth_rgb_batch(rgb.ctypes.data, w, h, first_seed, count)
    g = tile_grid(w, h)  # choh.cpp:454-460 in Python: the reference arm loads nothing of this repo's product
    t_enc = t_dec = t_lz = 0.0
    nuke = np.zeros(g.tile_w * g.tile_h, np.uint8)
    lz_out = np.zeros(g.tile_w * g.tile_h * 2 + 8192, np.uint8)
    mask = np.array([0x0010], np.uint16)
    no_backref = np.zeros(g.tile_w * g.tile_h, np.uint16)
    for i in range(count):
        img = rgb[i * w * h * 3:(i + 1) * w * h * 3].reshape(h, w, 3)
        for t in range(g.tiles_per_image):
            x0, y0 = (t % g.x_tiles) * g.tile_w, (t // g.x_tiles) * g.tile_h
            t0 = time.perf_counter()
            tile = np.ascontiguousarray(img[y0:y0 + g.tile_h, x0:x0 + g.tile_w])  # choh.cpp:478-484
            th, tw = tile.shape[:2]
            px = tw * th
            tile = tile.ravel()
            planes = [np.empty(px, np.uint16) for _ in range(3)]
            if use_ref:
                R.ref_subtract_green(tile, tile.size, *planes)
            else:
                O.orc_subtract_green(tile, tile.size, *planes)
            chans = []
            for p, d in zip(planes, (8, 9, 9)):
                out = np.empty(px * 4 + 4096, np.uint8)
                if use_ref:
                    n = R.ref_layer_encode(p, px, tw, th, d, MODE, nuke[:px], out)
                else:
                    n = O.orc_layer_encode(p, px, tw, th, d, MODE, nuke[:px], out, None)
                chans.append(out[:n + 16])
            t1 = time.perf_counter()
            dec = []
            for ch, d in zip(chans, (8, 9, 9)):
                sym = np.empty(px + 8, np.uint16)
                bp = C.c_size_t(5)  # after the channel header 10 00 00 00 10
                pl = np.empty(px, np.uint16)
                if use_ref:
                    R.ref_decode_entropy(ch, len(ch), C.byref(bp), sym, px)
                    R.ref_unpredict_all(sym, px, tw, th, d, 1, 1, mask, no_backref[:px], pl)
                else:
                    st = C.c_int(0)
                    O.orc_decode_entropy(ch, len(ch), C.byref(bp), sym, px, 7, C.byref(st))
                    O.orc_unpredict_fastpath(sym, tw, th, d, None, pl)
                dec.append(pl)
            back = np.empty(px * 3, np.uint8)
            O.orc_add_green(dec[0], dec[1], dec[2], px, back)  # the reference has no inverse (D4)
            t2 = time.perf_counter()
            # the LZ match finder (lz.hpp:6, seek distance 6 at -s0): timed on its own, not part of `value`
            lz_nuke = np.zeros(px, np.uint8)
            if use_ref:
                R.ref_find_lz_rgb(tile, tile.size, tw, th, lz_out, lz_nuke, 6, 0)
            else:
                O.orc_find_lz_rgb(tile, tile.size, tw, 6, 0, lz_out, lz_nuke, None, None)
            t3 = time.perf_counter()
            t_enc += t1 - t0
            t_dec += t2 - t1
            t_lz += t3 - t2
    return t_enc, t_dec, count * w * h * 3, use_ref, t_lz


def cpu_hot_path(sample_images, w, h, cores, seed0=1):
    """Times the reference CPU hot path (encode + decode, LZ excluded: NUKE == 0) on `cores`
    processes over `sample_images` images.  Returns dict(value MB/s, t_enc, t_dec, kind)."""
    import multiprocessing as mp
    synth_lib()  # compiled once, before the workers fork
    per = [sample_images // cores + (1 if i < sample_images % cores else 0) for i in range(cores)]
    jobs, seed = [], seed0
    for n in per:
        if n:
            jobs.append((seed, n, w, h))
            seed += n
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    raw = sum(r[2] for r in res)
    slowest = max(r[0] + r[1] for r in res)
    return {"value": 2 * raw / slowest / 1e6, "encode_mbs": raw / max(r[0] for r in res) / 1e6,
            "decode_mbs": raw / max(r[1] for r in res) / 1e6, "lz_mbs": raw / max(r[4] for r in res) / 1e6,
            "kind": "reference" if res[0][3] else "port",
            "cores": len(jobs), "wall_s": wall, "busy_s": slowest, "images": sample_images}


METRIC = "raw RGB MB/s, encode+decode (BASELINE.json: raw RGB MB/s encode & decode, % of HBM peak)"


# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(gpu_index):
    """Pins this process to the CPUs next to its GPU (the PCI device's local_cpulist) BEFORE the pinned staging
    buffers are allocated, so that first touch puts them on the GPU's own NUMA node: with one rank per GPU and the
    buffers on whichever node the ranks happened to start on, the host copies of an 8-GPU box cross the socket
    link.  Returns what was done, for the JSON line; does nothing on a single-node host."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        phys = gpu_index
        if vis and all(v.strip().isdigit() for v in vis.split(",")):
            phys = int(vis.split(",")[gpu_index])
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dev = "/sys/bus/pci/devices/" + bus.lower()[-12:]
        node = int(open(dev + "/numa_node").read().strip())
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if node < 0 or len(nodes) < 2:
            return {"node": node, "nodes": len(nodes), "bound": False}
        cpus = set()
        for part in open(dev + "/local_cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"node": node, "nodes": len(nodes), "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"node": node, "nodes": len(nodes), "bound": True, "cpus": len(cpus)}
    except Exception as e:  # no NVML, no sysfs: run unbound
        return {"bound": False, "why": type(e).__name__}


def host_memory_allows(need_bytes, reserve=8 << 30):
    """True when `need_bytes` more (summed over the ranks of this box) fit under /proc/meminfo's MemAvailable and
    the cgroup's limit with `reserve` to spare."""
    avail = None
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
    except OSError:
        return True
    try:
        lim = open("/sys/fs/cgroup/memory.max").read().strip()
        cur = int(open("/sys/fs/cgroup/memory.current").read().strip())
        if lim != "max":
            avail = min(avail, int(lim) - cur) if avail is not None else int(lim) - cur
    except (OSError, ValueError):
        pass
    return avail is None or need_bytes + reserve <= avail


def kernel_source_sha1():
    import hashlib
    h = hashlib.sha1()
    for f in ("hoh_kernels.cuh", "hoh_api.cu", "hoh_format.cuh"):
        h.update(open(os.path.join(ROOT, "hoh-ans_b200", "csrc", f), "rb").read())
    return h.hexdigest()


def pcie_probe(g, lib, ctx, h_src, h_dst, d_a, d_b, nbytes, reps=3):
    """H2D alone, D2H alone, both at once (pinned host memory; the context's stream and a second context's)."""
    other = type(g)(g.device)

    def run(h2d, d2h):
        g.sync()
        other.sync()
        t0 = time.perf_counter()
        for _ in range(reps):
            if h2d:
                g._ck(lib.hoh_h2d(ctx, d_a.ptr, h_src.ctypes.data, nbytes), "h2d")
            if d2h:
                g._ck(lib.hoh_d2h(other.ctx, h_dst.ctypes.data, d_b.ptr, nbytes), "d2h")
        g.sync()
        other.sync()
        return reps * nbytes / (time.perf_counter() - t0) / 1e9

    run(True, True)
    out = {"h2d_alone_gbs": run(True, False), "d2h_alone_gbs": run(False, True)}
    both = run(True, True)
    out["h2d_both_gbs"] = both
    out["d2h_both_gbs"] = both
    other.close()
    return out


def run_config_tiles(g, mod, shard, rank, world, host_threads, hbm_peak, barrier, name, w, h, mode, total_images, strong,
                     parity_tiles, steps, e2e_leg=True):
    """Whole tiles at cruncher mode >= 1 (hoh_encode_images / hoh_decode_images, device resident): BASELINE configs 3
    and 5.  strong: total_images is the whole job, split by image index; else total_images per rank."""
    lib, ctx = g.lib, g.ctx
    if strong:
        lo, hi = shard.shard_range(total_images, rank, world)
    else:
        lo, hi = rank * total_images, (rank + 1) * total_images
    n = hi - lo
    geo = g.tile_geometry(w, h)
    n_tiles = n * geo.tiles_per_image
    raw = n * w * h * 3
    rgb = np.zeros(max(raw, 1), np.uint8)
    if n:
        fill_images(rgb, 1 + lo, n, w, h, host_threads)
    cap = raw + raw // 2 + 8192 * n_tiles + 64
    bufs = [g.alloc(max(raw, 16)), g.alloc(cap), g.alloc((n_tiles + 1) * 8), g.alloc(max(n_tiles, 1) * mod.TILE_DT.itemsize),
            g.alloc(max(raw, 16)), g.alloc(max(n_tiles, 1) * 4)]
    d_rgb, d_packed, d_off, d_tiles, d_back, d_st = bufs
    if n:
        d_rgb.upload(rgb[:raw])
    FIX_ENCODER = 24

    def enc(flags=FIX_ENCODER):
        if n:
            g._ck(lib.hoh_encode_images(ctx, d_rgb.ptr, n, w, h, mode, flags, d_packed.ptr, cap, d_off.ptr, d_tiles.ptr), "hoh_encode_images")

    def dec():
        if n:
            g._ck(lib.hoh_decode_images(ctx, d_packed.ptr, cap, d_off.ptr, n, w, h, d_back.ptr, d_st.ptr), "hoh_decode_images")

    enc()
    dec()
    g.sync()
    g.layer_stats()  # reset: what follows counts the timed calls only
    l0 = g.launch_count()
    barrier()
    cfg_clocks = ClockSampler(int(os.environ.get("LOCAL_RANK", 0)))  # the clocks of THIS timed region
    cfg_clocks.start()
    # every call timed on its own (CUDA events on the context's stream) and the MEDIAN reported: a call of these paths is
    # ~100 launches spread over child contexts and side streams, and how the block scheduler interleaves them varies from
    # call to call (tools/jitter_probe.py: decode 33.8 ms eleven times out of twelve, 69 ms once); all samples are kept
    enc_calls, dec_calls = [], []
    for _ in range(steps):
        g.timer_start(4)
        enc()
        g.timer_stop(4)
        enc_calls.append(g.timer_ms(4))
    for _ in range(steps):
        g.timer_start(5)
        dec()
        g.timer_stop(5)
        dec_calls.append(g.timer_ms(5))
    enc_ms, dec_ms = float(np.median(enc_calls)), float(np.median(dec_calls))
    cfg_clk = cfg_clocks.stop()
    barrier()
    launches = g.launch_count() - l0
    coded, unsettled, planes = g.layer_stats()
    comp = int(d_off.download(np.uint64, n_tiles + 1)[-1]) if n else 0
    ok = True
    if n:
        rec = d_tiles.download(mod.TILE_DT, n_tiles)
        ok = bool((rec["status"] == 0).all() and (d_st.download(np.int32, n_tiles) == 0).all()
                  and np.array_equal(d_back.download(np.uint8, raw), rgb[:raw]))
    # sampled byte parity with the oracle at flags = 0 (stock choh bytes), rank 0 only: the oracle needs 0.6 s
    # (mode 2) to 3 s (mode 4) per tile, so the sample is small here; tests/test_gpu_config_sizes.py compares 64+
    parity = None
    if rank == 0 and n and parity_tiles:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as ol
        from concurrent.futures import ThreadPoolExecutor
        first = rgb[: w * h * 3]
        tiles, _ = g.encode_images(first, 1, w, h, mode, 0)
        img = first.reshape(h, w, 3)
        picks = sorted({(k * (geo.tiles_per_image - 1)) // max(parity_tiles - 1, 1) for k in range(parity_tiles)})

        def check(t):
            x0, y0 = (t % geo.x_tiles) * geo.tile_w, (t // geo.x_tiles) * geo.tile_h
            want, _ = ol.orc_encode_tile_subgreen(np.ascontiguousarray(img[y0:y0 + geo.tile_h, x0:x0 + geo.tile_w]), mode)
            return tiles[t] == want
        ol.oracle()
        with ThreadPoolExecutor(len(picks)) as pool:
            parity = {"tiles_compared": len(picks), "byte_exact": bool(all(pool.map(check, picks)))}
    for b in bufs:
        b.free()
    # end to end through the host-buffer C-ABI calls the C++ tools use (hoh_encode_images_host / hoh_decode_images_host):
    # pinned buffers, chunked H2D / kernels / D2H inside the library, copies inside the timed region
    e2e = None
    if n and e2e_leg:
        src = g.host_alloc(raw)
        src[:] = rgb[:raw]
        packed = g.host_alloc(cap)
        back = g.host_alloc(raw)
        off = np.zeros(n_tiles + 1, np.uint64)
        rec = np.zeros(n_tiles, mod.TILE_DT)
        st = np.zeros(n_tiles, np.int32)

        def e2e_once():
            ta = time.perf_counter()
            g._ck(lib.hoh_encode_images_host(ctx, src.ctypes.data, n, w, h, mode, FIX_ENCODER, packed.ctypes.data, cap,
                                             off.ctypes.data, rec.ctypes.data), "hoh_encode_images_host")
            tb = time.perf_counter()
            g._ck(lib.hoh_decode_images_host(ctx, packed.ctypes.data, int(off[-1]), off.ctypes.data, n, w, h,
                                             back.ctypes.data, st.ctypes.data), "hoh_decode_images_host")
            return tb - ta, time.perf_counter() - tb
        e2e_once()
        barrier()
        te = td = 0.0
        for _ in range(steps):
            a, b = e2e_once()
            te, td = te + a / steps, td + b / steps
        e2e = {"encode_ms": 1e3 * te, "decode_ms": 1e3 * td,
               "ok": bool((rec["status"] == 0).all() and (st == 0).all() and np.array_equal(back, src)),
               "h2d": raw + int(off[-1]), "d2h": raw + int(off[-1])}
        for a in (src, packed, back):
            g.host_free(a)
        del src, packed, back
    elif e2e_leg:
        barrier()
    e2e_out = None
    if e2e_leg:
        e_ms = shard.reduce_max(e2e["encode_ms"] + e2e["decode_ms"] if e2e else 0.0, world, device="cuda")
        e_ok = shard.reduce_sum(1.0 if (e2e is None or e2e["ok"]) else 0.0, world, device="cuda") == world
        e2e_out = {"value_mbs": 2 * shard.reduce_sum(float(raw), world, device="cuda") / e_ms / 1e3, "ms_per_step": e_ms,
                   "encode_ms_this_rank": e2e["encode_ms"] if e2e else None, "decode_ms_this_rank": e2e["decode_ms"] if e2e else None,
                   "h2d_bytes_per_step": e2e["h2d"] if e2e else 0, "d2h_bytes_per_step": e2e["d2h"] if e2e else 0, "verified": e_ok}
    enc_ms, dec_ms = shard.reduce_max(enc_ms, world, device="cuda"), shard.reduce_max(dec_ms, world, device="cuda")
    job_raw = shard.reduce_sum(float(raw), world, device="cuda")
    job_comp = shard.reduce_sum(float(comp), world, device="cuda")
    all_ok = shard.reduce_sum(1.0 if ok else 0.0, world, device="cuda") == world
    alg = job_raw + job_comp
    return {"workload": name, "scaling": "strong" if strong else "weak", "images_in_job": int(job_raw // (w * h * 3)),
            "images_this_rank": n, "mode": mode, "encode_ms": enc_ms, "decode_ms": dec_ms,
            "timing": f"median of {steps} calls, each timed with CUDA events; this rank's samples follow",
            "encode_ms_calls": [round(v, 2) for v in enc_calls], "decode_ms_calls": [round(v, 2) for v in dec_calls],
            "encode_mbs": job_raw / enc_ms / 1e3, "decode_mbs": job_raw / dec_ms / 1e3,
            "value_mbs": 2 * job_raw / (enc_ms + dec_ms) / 1e3, "compressed_ratio": job_comp / max(job_raw, 1),
            "hbm_frac_encode": alg / world / enc_ms / 1e6 / hbm_peak, "hbm_frac_decode": alg / world / dec_ms / 1e6 / hbm_peak,
            "roundtrip_exact": all_ok, "oracle_parity_sample": parity, "gpu_launches": int(launches), "clocks": cfg_clk,
            "entropy_candidates": {"planes": planes, "coded_per_plane": coded / max(planes, 1),
                                   "planes_coded_in_full_frac": unsettled / max(planes, 1),
                                   "what": "layer_encode tries six rANS candidates per plane; their sizes follow from histogram "
                                           "and table up to one word, so only the kept one is coded unless a comparison is open"},
            "e2e": e2e_out,
            "limit": "a launch of the entropy / un-prediction kernels lasts as long as ONE stream's serial chain however few "
                     "streams a rank holds, so strong scaling flattens once the per-rank batch no longer fills the SMs"
                     if strong else "throughput-bound: six to nine rANS candidates per plane plus the predictor search"}


def run_config_static(g, mod, shard, rank, world, hbm_peak, barrier, log2n, steps):
    """BASELINE config 4: rans64 sweep point — 2^log2n symbols per GPU over an 8-bit alphabet, one static 12-bit
    table, 65 536-symbol streams (tools/bench_static.py walks the whole 1 MB .. 4 GB range)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    lib, ctx = g.lib, g.ctx
    STREAM, PB = 65536, 12
    n = 1 << log2n
    n_streams = n // STREAM
    base = ol.synth_symbols(1 << 24, 7 + rank)
    f = np.bincount(base, minlength=256).astype(np.uint32)
    cum = np.zeros(257, np.uint32)
    assert ol.oracle().orc_normalize_freqs(f, cum, 256, 1 << PB) == 0
    d_cum = g.alloc(cum.nbytes).upload(cum)
    slab = (STREAM * PB // 8 + 64 + 15) & ~15
    sym = base.astype(np.uint16)
    d_sym, d_out, d_len, d_dec = g.alloc(n * 2 + 64), g.alloc(n_streams * slab), g.alloc(n_streams * 4), g.alloc(n * 2 + 64)
    piece = sym[:min(n, sym.size)]
    for r in range(max(1, n // sym.size)):
        g._ck(lib.hoh_h2d(ctx, d_sym.ptr + r * piece.nbytes, piece.ctypes.data, piece.nbytes), "h2d")

    def enc():
        g._ck(lib.hoh_rans_encode_static(ctx, d_sym.ptr, n, STREAM, d_cum.ptr, 256, PB, d_out.ptr, slab, d_len.ptr), "enc")

    def dec():
        g._ck(lib.hoh_rans_decode_static(ctx, d_out.ptr, slab, d_len.ptr, n, STREAM, d_cum.ptr, 256, PB, d_dec.ptr), "dec")
    enc()
    dec()
    g.sync()
    barrier()
    g.timer_start(4)
    for _ in range(steps):
        enc()
    g.timer_stop(4)
    g.timer_start(5)
    for _ in range(steps):
        dec()
    g.timer_stop(5)
    e_ms, d_ms = g.timer_ms(4) / steps, g.timer_ms(5) / steps
    barrier()
    lens = d_len.download(np.uint32, n_streams)
    back = d_dec.download(np.uint16, min(n, 1 << 24))
    ok = bool(np.array_equal(back, sym[:back.size]))
    # oracle parity on a sample of streams: payload bytes of the reference's Rans64 loop with the same table
    buf = np.zeros(STREAM * 2 + 64, np.uint8)
    exact = True
    for k in (0, n_streams // 2, n_streams - 1):
        part = np.ascontiguousarray(sym[(k * STREAM) % sym.size:(k * STREAM) % sym.size + STREAM])
        nb = ol.oracle().orc_rans_encode_static(part, STREAM, f, cum, 256, PB, buf)
        got = d_out.download(np.uint8, (k + 1) * slab)[k * slab:]
        exact = exact and int(lens[k]) == nb and got[slab - nb:].tobytes() == buf[:nb].tobytes()
    comp = int(lens.astype(np.uint64).sum())
    for b in (d_sym, d_out, d_len, d_dec, d_cum):
        b.free()
    e_ms, d_ms = shard.reduce_max(e_ms, world, device="cuda"), shard.reduce_max(d_ms, world, device="cuda")
    job_n = shard.reduce_sum(float(n), world, device="cuda")
    job_comp = shard.reduce_sum(float(comp), world, device="cuda")
    all_ok = shard.reduce_sum(1.0 if (ok and exact) else 0.0, world, device="cuda") == world
    alg = job_n + job_comp  # SURVEY 8(d): 1 B per symbol + H/8 B
    return {"workload": f"rans64 static-table stream sweep point: 2^{log2n} symbols per GPU, 8-bit alphabet, one 12-bit table, "
                        f"65 536-symbol streams", "scaling": "weak", "symbols_in_job": int(job_n), "encode_ms": e_ms, "decode_ms": d_ms,
            "encode_msym_s": job_n / e_ms / 1e3, "decode_msym_s": job_n / d_ms / 1e3, "bits_per_symbol": job_comp * 8 / job_n,
            "hbm_frac_encode": alg / world / e_ms / 1e6 / hbm_peak, "hbm_frac_decode": alg / world / d_ms / 1e6 / hbm_peak,
            "roundtrip_exact_and_oracle_parity": all_ok}


DUMP_IMAGES = 4  # images whose payload bytes and decoded RGB are written: ~20 MB as float32
DUMP_STREAMS = 1 << 18  # per-stream records written at most: 9 float64 each, ~19 MB
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, mod, geom, n_img, d_res, d_packed, d_off, d_back, d_st):
    """What a caller of hoh_encode_images_s0 + hoh_decode_images_s0 receives after the last timed step, so that two
    builds can be compared file by file: per-stream records (payload start / end, encode result fields, decode
    status) as float64 for every stream, or for a fixed, seeded sample of DUMP_STREAMS of them, and the payload
    bytes and decoded RGB of a fixed, seeded sample of DUMP_IMAGES images as float32 (the batch is gigabytes)."""
    spi = geom.streams_per_image
    n_streams = n_img * spi
    off = d_off.download(np.uint64, n_streams + 1)
    res = d_res.download(mod.RESULT_DT, n_streams)
    keep = np.arange(n_streams)
    if n_streams > DUMP_STREAMS:
        keep = np.sort(np.random.default_rng(1).choice(n_streams, DUMP_STREAMS, replace=False))
    arrays = {"streams": keep, "stream_start": off[keep], "stream_end": off[keep + 1],
              "decode_status": d_st.download(np.int32, n_streams)[keep]}
    for f in mod.RESULT_DT.names:
        arrays[f"encode_{f}"] = res[f][keep]
    arrays = {k: a.astype(np.float64) for k, a in arrays.items()}
    pick = np.sort(np.random.default_rng(0).choice(n_img, min(DUMP_IMAGES, n_img), replace=False))
    payload, rgb = [], []
    for i in pick:
        lo, hi = int(off[i * spi]), int(off[(i + 1) * spi])
        payload.append(d_packed.download(np.uint8, hi - lo, offset=lo))
        rgb.append(d_back.download(np.uint8, W * H * 3, offset=int(i) * W * H * 3).reshape(H, W, 3))
    arrays["sample_images"] = pick.astype(np.float64)
    arrays["sample_payload"] = np.concatenate(payload).astype(np.float32)
    arrays["sample_decoded_rgb"] = np.stack(rgb).astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--images", type=int, default=4096, help="images per GPU")
    ap.add_argument("--no-lz", action="store_true", help="skip the LZ match finder timing")
    ap.add_argument("--cpu-sample", type=int, default=0, help="images in the cpu_baseline sample (0 = 4 per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--configs", default="3,4,5", help="BASELINE.json configs reported beside the config-2 headline "
                    "(comma list of 3, 4, 5; empty = headline only)")
    ap.add_argument("--frames", type=int, default=256, help="config 3: 3840x2160 frames in the whole job (strong scaling)")
    ap.add_argument("--thumbs", type=int, default=8192, help="config 5: 256x256 thumbnails per GPU")
    ap.add_argument("--static-log2", type=int, default=30, help="config 4: log2 of the symbols per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    extra = [int(x) for x in args.configs.split(",") if x.strip()]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps, warmup = args.steps, max(args.warmup, 0)
    config = {"workload": f"{args.images} synthetic {W}x{H} RGB images per GPU, cruncher mode -s0 "
                          f"(BASELINE.json configs[1]), subtract-green + MED fastpath + rANS prob_bits 15, "
                          f"encode then decode", "images_per_gpu": args.images, "width": W, "height": H,
              "mode": MODE, "cold_cache": "inputs (3.2 GB per GPU) are larger than the 126 MB L2",
              "sharding": f"images by index across {world} GPU(s), no collective in the data path"}

    # ---------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        cores = os.cpu_count() or 1
        sample = args.cpu_sample or max(cores * 2, 16)
        load_reference_in_parent()
        vals = []
        for it in range(warmup + steps):
            r = cpu_hot_path(sample, W, H, cores, seed0=1)
            if it >= warmup:
                vals.append(r)
        busy = sum(v["busy_s"] for v in vals)
        raw = sum(v["images"] for v in vals) * W * H * 3
        value = 2 * raw / busy / 1e6
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "MB/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * busy / max(steps, 1),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16/u64 integer",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": "MB/s", "cores": vals[0]["cores"], "kind": vals[0]["kind"],
                                 "sample": f"{sample} images of {W}x{H} per step (of {args.images}), one process per "
                                           f"core, reference hot path only (subtract_green + layer_encode x3, "
                                           f"decode_entropy + unpredict_all x3; host LZ excluded on both arms)"},
                "e2e": {"value": value, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "encode_mbs": float(np.mean([v["encode_mbs"] for v in vals])),
                "decode_mbs": float(np.mean([v["decode_mbs"] for v in vals]))}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- B200 arm
    # one rank alone keeps every core (the cpu_baseline leg forks its workers from this process)
    numa = bind_to_gpu_numa(local_rank) if world > 1 else {"bound": False, "why": "single rank"}
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    mod = _load("hohgpu", os.path.join(ROOT, "hoh-ans_b200", "host", "hohgpu.py"))
    shard = _load("hoh_shard", os.path.join(ROOT, "hoh-ans_b200", "host", "shard.py"))
    g = mod.HohGpu(local_rank)
    lib, ctx = g.lib, g.ctx
    geom = g.tile_geometry(W, H)
    n_img = args.images
    raw = n_img * W * H * 3
    n_streams = n_img * geom.streams_per_image
    host_threads = max(1, (os.cpu_count() or 8) // max(world, 1))

    # inputs: distinct image per global index (seed = 1 + index), pinned host memory
    rgb_host = g.host_alloc(raw)
    fill_images(rgb_host, shard.weak_first_seed(n_img, rank), n_img, W, H, host_threads)
    out_bytes = int(lib.hoh_encode_images_out_bytes(C.byref(geom), n_img))
    packed_cap = raw + raw // 4 + 4096 * n_streams
    d_rgb, d_back = g.alloc(raw), g.alloc(raw)
    d_out, d_packed = g.alloc(out_bytes), g.alloc(packed_cap)
    d_res, d_off, d_st = g.alloc(n_streams * 24), g.alloc((n_streams + 1) * 8), g.alloc(n_streams * 4)
    g._ck(lib.hoh_h2d(ctx, d_rgb.ptr, rgb_host.ctypes.data, raw), "h2d")
    g.sync()

    def encode_dev():
        g._ck(lib.hoh_encode_images_s0(ctx, d_rgb.ptr, n_img, W, H, None, d_out.ptr, out_bytes, d_res.ptr,
                                       d_packed.ptr, packed_cap, d_off.ptr), "hoh_encode_images_s0")

    def decode_dev():
        g._ck(lib.hoh_decode_images_s0(ctx, d_packed.ptr, packed_cap, d_off.ptr, n_img, W, H, None, d_back.ptr,
                                       d_st.ptr), "hoh_decode_images_s0")

    def barrier():
        g.sync()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up + correctness of what is being timed
    clocks = ClockSampler(local_rank)
    for _ in range(max(warmup, 1)):
        encode_dev()
        decode_dev()
    g.sync()
    off = d_off.download(np.uint64, n_streams + 1)
    comp_bytes = int(off[-1])
    st = d_st.download(np.int32, n_streams)
    res = d_res.download(mod.RESULT_DT, n_streams)
    back = d_back.download(np.uint8, raw)
    verified = bool((st == 0).all() and (res["status"] == 0).all() and np.array_equal(back, rgb_host))
    del back

    # timed region: device resident
    launches0 = g.launch_count()
    barrier()
    clocks.start()
    t_enc = t_dec = 0.0
    g.timer_start(0)
    for k in range(steps):
        g.timer_start(2)
        encode_dev()
        g.timer_stop(2)
        g.timer_start(3)
        decode_dev()
        g.timer_stop(3)
        t_enc += g.timer_ms(2)
        t_dec += g.timer_ms(3)
    g.timer_stop(0)
    total_ms = g.timer_ms(0)
    barrier()
    clk = clocks.stop()
    launches = g.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, mod, geom, n_img, d_res, d_packed, d_off, d_back, d_st)

    # per-kernel profile of one step (separate pass, CUDA events after every launch)
    g.profile_begin()
    encode_dev()
    decode_dev()
    prof = g.profile_end()

    # the LZ match finder on the same resident batch (SURVEY 8(f) row 1; reported beside `value`, not in it)
    lz = None
    if not args.no_lz:
        geo = g.tile_geometry(W, H)
        n_tiles = n_img * geo.tiles_per_image
        nuke_stride = (geo.tile_w * geo.tile_h + 7) & ~7
        lz_stride = int(lib.hoh_find_lz_stride(geo.tile_w, geo.tile_h))
        lz_bufs = [g.alloc(n_tiles * nuke_stride), g.alloc(n_tiles * lz_stride), g.alloc(n_tiles * 4), g.alloc(n_tiles * 4)]

        def lz_dev():
            g._ck(lib.hoh_find_lz_images(ctx, d_rgb.ptr, n_img, W, H, 6, 0, None, lz_bufs[0].ptr, lz_bufs[1].ptr, lz_stride,
                                         lz_bufs[2].ptr, lz_bufs[3].ptr), "hoh_find_lz_images")
        lz_dev()
        g.sync()
        l0 = g.launch_count()
        g.timer_start(1)
        for _ in range(steps):
            lz_dev()
        g.timer_stop(1)
        lz_ms = g.timer_ms(1) / steps
        lz_ok = bool((lz_bufs[3].download(np.int32, n_tiles) == 0).all())
        lz = {"ms": lz_ms, "mbs": raw / (lz_ms / 1e3) / 1e6, "launches_per_call": (g.launch_count() - l0) // steps,
              "ok": lz_ok, "nuked_pixels": int(np.count_nonzero(lz_bufs[0].download(np.uint8, min(n_tiles, 64) * nuke_stride)))}
        for b in lz_bufs:
            b.free()

    # e2e: host buffers through the C-ABI, copies inside the timed region
    e2e = None
    barrier()
    short = 0.0 if host_memory_allows(world * (packed_cap + raw + (n_streams + 1) * 8)) else 1.0
    if not args.no_e2e and shard.reduce_max(short, world, device="cuda") > 0:  # one decision for all ranks
        # every rank pins ~7.4 GB more for this leg: a host that cannot hold that loses the leg, not the box
        sys.stderr.write("bench: e2e leg skipped, not enough free host memory for the pinned buffers\n")
        args.no_e2e = True
    if not args.no_e2e:
        packed_host = g.host_alloc(packed_cap)
        off_host = g.host_alloc((n_streams + 1) * 8, np.uint64)
        back_host = g.host_alloc(raw)

        e2e_split = [0.0, 0.0]

        def e2e_step():
            ta = time.perf_counter()
            g._ck(lib.hoh_encode_images_s0_host(ctx, rgb_host.ctypes.data, n_img, W, H, packed_host.ctypes.data,
                                                packed_cap, off_host.ctypes.data, None), "encode_host")
            tb = time.perf_counter()
            total = int(off_host[n_streams])
            g._ck(lib.hoh_decode_images_s0_host(ctx, packed_host.ctypes.data, total, off_host.ctypes.data, n_img, W,
                                                H, back_host.ctypes.data, None), "decode_host")
            e2e_split[0] += tb - ta
            e2e_split[1] += time.perf_counter() - tb
            return total

        e2e_step()
        e2e_ok = bool(np.array_equal(back_host, rgb_host))
        e2e_split[0] = e2e_split[1] = 0.0
        barrier()
        g.timer_start(1)
        t0 = time.perf_counter()
        e_steps = steps
        for _ in range(e_steps):
            total = e2e_step()
        g.timer_stop(1)
        e2e_ms = g.timer_ms(1)
        wall_ms = 1e3 * (time.perf_counter() - t0)
        barrier()
        e2e_ms = max(e2e_ms, wall_ms)
        e2e = {"ms": e2e_ms / e_steps, "ok": e2e_ok, "enc_ms": 1e3 * e2e_split[0] / e_steps,
               "dec_ms": 1e3 * e2e_split[1] / e_steps,
               "h2d": raw + total + (n_streams + 1) * 8, "d2h": total + (n_streams + 1) * 8 + raw}

    # max over ranks of the device time, sum over ranks of the bytes (hoh-ans_b200/host/shard.py)
    def rmax(x):
        return shard.reduce_max(x, world, device="cuda")

    def rsum(x):
        return shard.reduce_sum(x, world, device="cuda")

    def rmin(x):
        return -shard.reduce_max(-x, world, device="cuda")

    # what the PCIe links of THIS box give when every rank copies at once (both directions together): the ceiling
    # of the e2e leg, measured in the same run so that a low e2e number can be told apart from a slow box
    pcie = None
    if not args.no_e2e:
        probe_bytes = min(raw, 1 << 30)
        barrier()
        pcie = pcie_probe(g, lib, ctx, rgb_host, back_host, d_rgb, d_back, probe_bytes)
        barrier()
        pcie = {k: rmin(v) for k, v in pcie.items()}
        g.host_free(packed_host)
        g.host_free(off_host)
        g.host_free(back_host)
        del packed_host, off_host, back_host
    for b in (d_rgb, d_back, d_out, d_packed, d_res, d_off, d_st):
        b.free()
    g.host_free(rgb_host)
    del rgb_host

    configs_out = {}
    hbm_peak_all = 6650.0
    try:
        hbm_peak_all = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
    except Exception:
        pass
    for c in extra:
        barrier()
        g.release_scratch()
        if c == 3:
            configs_out["config3"] = run_config_tiles(g, mod, shard, rank, world, host_threads, hbm_peak_all, barrier,
                                                      name="256 x 3840x2160 -s2, frames sharded across the GPUs (strong scaling)",
                                                      w=3840, h=2160, mode=2, total_images=args.frames, strong=True,
                                                      parity_tiles=4, steps=steps, e2e_leg=not args.no_e2e)
        elif c == 5:
            configs_out["config5"] = run_config_tiles(g, mod, shard, rank, world, host_threads, hbm_peak_all, barrier,
                                                      name=f"slice of the 1M 256x256 thumbnails at -s4: {args.thumbs} per GPU "
                                                           f"(weak scaling; the full 10^6 / 8 GPUs = {125000 // args.thumbs + 1} such chunks per GPU)",
                                                      w=256, h=256, mode=4, total_images=args.thumbs, strong=False,
                                                      parity_tiles=2, steps=steps, e2e_leg=not args.no_e2e)
        elif c == 4:
            configs_out["config4"] = run_config_static(g, mod, shard, rank, world, hbm_peak_all, barrier, args.static_log2, steps)

    total_ms = rmax(total_ms)
    t_enc, t_dec = rmax(t_enc), rmax(t_dec)
    job_raw = rsum(float(raw))
    job_comp = rsum(float(comp_bytes))
    all_verified = rsum(1.0 if verified else 0.0) == world
    if e2e:
        e2e["ms"] = rmax(e2e["ms"])
        e2e_all_ok = rsum(1.0 if e2e["ok"] else 0.0) == world

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        value = 2 * job_raw * steps / (total_ms / 1e3) / 1e6
        # dominant kernel by device time in the profiled step
        top = max(prof.items(), key=lambda kv: kv[1][0])
        top_name, (top_ms, top_cnt) = top
        step_ms_prof = sum(v[0] for v in prof.values())
        per_launch_ms = top_ms / top_cnt
        # algorithmic bytes of one launch (DESIGN.md section 4): encode-side kernels move 3*W*H in + C out
        # per image, decode-side kernels C in + 3*W*H out; a launch covers the rank's whole batch
        alg_bytes = raw + comp_bytes
        # DRAM bytes per launch come from an `ncu --set full` capture (profiles/ncu_traffic.json); the file is stamped
        # with the hash of the kernel source it was captured from and is only quoted while that source is unchanged
        traffic, traffic_note = None, "no capture"
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            ent = tj.get(top_name.split("<")[0].split("[")[0])
            if ent and ent.get("images"):
                if tj.get("_kernel_source_sha1") == kernel_source_sha1():
                    traffic = ent["dram_bytes_per_launch"] * n_img / ent["images"]
                    traffic_note = f"ncu --set full capture at kernel source {tj['_kernel_source_sha1'][:12]}"
                else:
                    traffic_note = "capture is older than the kernel source: not quoted"
        except Exception:
            pass
        achieved = alg_bytes / (per_launch_ms / 1e3) / 1e9
        line = {
            "metric": METRIC,
            "value": value, "unit": "MB/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u16 pixels, u32 freqs, u64 rANS state (integer)", "data": "synthetic",
            "config": config, "verified_bit_exact_roundtrip": all_verified,
            "encode_mbs": job_raw * steps / (t_enc / 1e3) / 1e6, "decode_mbs": job_raw * steps / (t_dec / 1e3) / 1e6,
            "compressed_ratio": job_comp / job_raw,
            "hbm_frac_whole_step": ((job_raw + job_comp) * 2 * steps / world / (total_ms / 1e3) / 1e9) / hbm_peak,
            "gpu_launches": launches, "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": top_name, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": per_launch_ms,
                         "share_of_step": top_ms / step_ms_prof},
            "kernels_ms": {k: round(v[0], 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])},
        }
        if lz:
            line["lz_find"] = {"what": "find_lz_rgb (lz.hpp:6) for every tile of the batch on the device, seek distance 6; "
                                       "not included in value/e2e (BASELINE keeps LZ beside the metric)",
                               "ms_per_batch": lz["ms"], "raw_mbs_per_gpu": lz["mbs"], "gpu_launches": lz["launches_per_call"],
                               "status_ok": lz["ok"], "nuked_pixels_first_tiles": lz["nuked_pixels"]}
        if e2e:
            line["e2e"] = {"value": 2 * job_raw / (e2e["ms"] / 1e3) / 1e6, "unit": "MB/s",
                           "h2d_bytes_per_step": int(e2e["h2d"]), "d2h_bytes_per_step": int(e2e["d2h"]),
                           "ms_per_step": e2e["ms"], "encode_ms": e2e["enc_ms"], "decode_ms": e2e["dec_ms"],
                           "verified": e2e_all_ok, "numa_rank0": numa}
        if e2e and pcie:
            h2d_gbs, d2h_gbs = pcie["h2d_both_gbs"], pcie["d2h_both_gbs"]
            # encode moves raw in / C out, decode C in / raw out, overlapped: the longer direction of each phase bounds it
            bound_s = (raw / 1e9) / h2d_gbs + (raw / 1e9) / d2h_gbs
            line["e2e"]["pcie_bound_gbs"] = {"h2d_alone": pcie["h2d_alone_gbs"], "d2h_alone": pcie["d2h_alone_gbs"],
                                             "h2d_with_d2h": h2d_gbs, "d2h_with_h2d": d2h_gbs,
                                             "what": f"per rank, min over the {world} ranks copying at the same time, pinned memory"}
            line["e2e"]["pcie_bound_value"] = 2 * raw * world / bound_s / 1e6
            line["e2e"]["frac_of_pcie_bound"] = line["e2e"]["value"] / line["e2e"]["pcie_bound_value"]
        if configs_out:
            line["configs"] = configs_out
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            sample = args.cpu_sample or max(cores * 4, 32)
            load_reference_in_parent()
            whole = cpu_whole_tool(max(cores * 4, 32), W, H, MODE, cores)
            if whole:
                line["cpu_whole_tool"] = whole
            if "config3" in configs_out:
                configs_out["config3"]["cpu_reference"] = cpu_encode_tiles(cores, 256, 270, 2, cores)
            if "config5" in configs_out:
                configs_out["config5"]["cpu_reference"] = cpu_encode_tiles(cores, 256, 256, 4, cores)
            cb = cpu_hot_path(sample, W, H, cores, seed0=1)
            line["cpu_baseline"] = {"value": cb["value"], "unit": "MB/s", "cores": cb["cores"], "kind": cb["kind"],
                                    "encode_mbs": cb["encode_mbs"], "decode_mbs": cb["decode_mbs"],
                                    "lz_find_mbs": cb["lz_mbs"],
                                    "sample": f"{sample} of the {n_img} images, one process per core, hot path only "
                                              f"(host LZ excluded on both arms), busy time of the slowest worker"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    g.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
