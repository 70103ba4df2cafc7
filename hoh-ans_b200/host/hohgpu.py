"""Host-side mirror of the hoh-ANS hot-path interface over the C-ABI of libhohgpu.so.

The reference is header-only C++ with no Python; this module exists so that tests and the bench can
call the GPU path with the reference's own function names and argument meaning
(encode_entropy, decode_entropy, subtract_green, channelpredict_*, unpredict_all ...).  It does no
computation itself: every method forwards to an `extern "C"` entry point of include/hohgpu.h.
There is no CPU fallback — constructing HohGpu without a CUDA device raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# (HOH_GPU_LIB: another build of the same library, for A/B measurements of kernel variants)
LIB_PATH = os.environ.get("HOH_GPU_LIB") or os.path.join(os.path.dirname(_HERE), "csrc", "libhohgpu.so")

HOH_OK = 0
HOH_E_CUDA, HOH_E_ARG, HOH_E_UNSUPPORTED, HOH_E_CAPACITY, HOH_E_STREAM = 1, 2, 3, 4, 5
FIX_PROB_BITS5, FIX_ADVANCE, FIX_EMPTY, FIX_ALL = 1, 2, 4, 7
MAX_RANGE = 512
STOCK_MASKS = [0x0001, 0x0002, 0x0020, 0x0010, 0xffbf, 0x0003, 0xfffd, 0xfffb, 0xfff7, 0xffef, 0xffdf,
               0xff7f, 0xfdff, 0xffff]  # layer_encode.hpp:159-175


class HohError(RuntimeError):
    def __init__(self, status, where, detail=""):
        super().__init__(f"{where}: status {status} {detail}")
        self.status = status


class EncStream(C.Structure):
    _fields_ = [("sym_off", C.c_uint64), ("n", C.c_uint32), ("range", C.c_uint32), ("prob_bits", C.c_uint32),
                ("prefix_len", C.c_uint32), ("prefix", C.c_uint8 * 8), ("out_off", C.c_uint64),
                ("out_cap", C.c_uint32), ("reserved", C.c_uint32)]


class StreamResult(C.Structure):
    _fields_ = [("start", C.c_uint64), ("size", C.c_uint32), ("status", C.c_int32),
                ("payload_bytes", C.c_uint32), ("stored", C.c_uint32)]


class DecStream(C.Structure):
    _fields_ = [("in_off", C.c_uint64), ("sym_off", C.c_uint64), ("sym_cap", C.c_uint32), ("flags", C.c_uint32)]


class DecResult(C.Structure):
    _fields_ = [("end_off", C.c_uint64), ("n", C.c_uint32), ("status", C.c_int32), ("range", C.c_uint32),
                ("prob_bits", C.c_uint32), ("stored", C.c_uint32), ("table_mode", C.c_uint32)]


class TileGeometry(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("x_tiles", C.c_uint32), ("y_tiles", C.c_uint32),
                ("tile_w", C.c_uint32), ("tile_h", C.c_uint32), ("tiles_per_image", C.c_uint32),
                ("streams_per_image", C.c_uint32)]


ENC_STREAM_DT = np.dtype([("sym_off", "<u8"), ("n", "<u4"), ("range", "<u4"), ("prob_bits", "<u4"),
                          ("prefix_len", "<u4"), ("prefix", "u1", (8,)), ("out_off", "<u8"), ("out_cap", "<u4"),
                          ("reserved", "<u4")])
RESULT_DT = np.dtype([("start", "<u8"), ("size", "<u4"), ("status", "<i4"), ("payload_bytes", "<u4"),
                      ("stored", "<u4")])
TILE_DT = np.dtype([("start", np.uint64), ("size", np.uint32), ("status", np.int32), ("colour_mode", np.uint32),
                    ("lz_size", np.uint32), ("chan_size", np.uint32, (3,)), ("flags", np.uint32)])
DEC_STREAM_DT = np.dtype([("in_off", "<u8"), ("sym_off", "<u8"), ("sym_cap", "<u4"), ("flags", "<u4")])
DEC_RESULT_DT = np.dtype([("end_off", "<u8"), ("n", "<u4"), ("status", "<i4"), ("range", "<u4"),
                          ("prob_bits", "<u4"), ("stored", "<u4"), ("table_mode", "<u4")])
assert ENC_STREAM_DT.itemsize == C.sizeof(EncStream) == 48
assert RESULT_DT.itemsize == C.sizeof(StreamResult) == 24
assert DEC_STREAM_DT.itemsize == C.sizeof(DecStream) == 24
assert DEC_RESULT_DT.itemsize == C.sizeof(DecResult) == 32

_vp, _sz, _u32, _int = C.c_void_p, C.c_size_t, C.c_uint32, C.c_int

# name -> (restype, argtypes); every symbol include/hohgpu.h declares
SIGNATURES = {
    "hoh_ctx_create": (_int, [_int, _vp, C.POINTER(_vp)]),
    "hoh_ctx_destroy": (None, [_vp]),
    "hoh_sync": (_int, [_vp]),
    "hoh_release_scratch": (_int, [_vp]),
    "hoh_debug_layer_stats": (_int, [_vp, C.POINTER(C.c_uint64)]),
    "hoh_strerror": (C.c_char_p, [_int]),
    "hoh_last_cuda_error": (C.c_char_p, [_vp]),
    "hoh_launch_count": (C.c_uint64, [_vp]),
    "hoh_dev_alloc": (_int, [_vp, _sz, C.POINTER(_vp)]),
    "hoh_dev_free": (_int, [_vp, _vp]),
    "hoh_dev_memset": (_int, [_vp, _vp, _int, _sz]),
    "hoh_host_alloc": (_int, [_vp, _sz, C.POINTER(_vp)]),
    "hoh_host_free": (_int, [_vp, _vp]),
    "hoh_h2d": (_int, [_vp, _vp, _vp, _sz]),
    "hoh_d2h": (_int, [_vp, _vp, _vp, _sz]),
    "hoh_timer_start": (_int, [_vp, _int]),
    "hoh_timer_stop": (_int, [_vp, _int]),
    "hoh_timer_elapsed_ms": (_int, [_vp, _int, C.POINTER(C.c_float)]),
    "hoh_flush_l2": (_int, [_vp]),
    "hoh_profile_begin": (_int, [_vp]),
    "hoh_profile_end": (_int, [_vp]),
    "hoh_profile_count": (_int, [_vp]),
    "hoh_profile_entry": (_int, [_vp, _int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "hoh_encode_images_s0_host": (_int, [_vp, _vp, _sz, _u32, _u32, _vp, _sz, _vp, _vp]),
    "hoh_decode_images_s0_host": (_int, [_vp, _vp, _sz, _vp, _sz, _u32, _u32, _vp, _vp]),
    "hoh_enc_slab_bytes": (_sz, [_sz, _u32]),
    "hoh_encode_entropy_batch": (_int, [_vp, _vp, _sz, _vp, _vp, _vp, _u32, _u32, _u32]),
    "hoh_decode_entropy_batch": (_int, [_vp, _vp, _sz, _vp, _sz, _vp, _vp, _u32]),
    "hoh_rans_encode_static": (_int, [_vp, _vp, _sz, _u32, _vp, _u32, _u32, _vp, _u32, _vp]),
    "hoh_rans_decode_static": (_int, [_vp, _vp, _u32, _vp, _sz, _u32, _vp, _u32, _u32, _vp]),
    "hoh_tile_geometry_for": (_int, [_u32, _u32, C.POINTER(TileGeometry)]),
    "hoh_encode_images_out_bytes": (_sz, [C.POINTER(TileGeometry), _sz]),
    "hoh_encode_images_s0": (_int, [_vp, _vp, _sz, _u32, _u32, _vp, _vp, _sz, _vp, _vp, _sz, _vp]),
    "hoh_decode_images_s0": (_int, [_vp, _vp, _sz, _vp, _sz, _u32, _u32, _vp, _vp, _vp]),
    "hoh_subtract_green_dev": (_int, [_vp, _vp, _sz, _vp, _vp, _vp]),
    "hoh_add_green_dev": (_int, [_vp, _vp, _vp, _vp, _sz, _vp]),
    "hoh_predict_fastpath_dev": (_int, [_vp, _vp, _sz, _int, _int, _int, _vp]),
    "hoh_unpredict_fastpath_dev": (_int, [_vp, _vp, _sz, _int, _int, _int, _vp, _vp]),
    "hoh_predict_all_dev": (_int, [_vp, _vp, _sz, _int, _int, _int, _int, _int, _vp, _vp]),
    "hoh_unpredict_all_dev": (_int, [_vp, _vp, _sz, _int, _int, _int, _int, _int, _vp, _vp, _vp]),
    "hoh_predict_section_dev": (_int, [_vp, _vp, _sz, _int, _int, _int, _int, _int, _vp, _int, _vp, _u32, _vp]),
    "hoh_predictor_search_dev": (_int, [_vp, _vp, _sz, _int, _int, _int, _int, _vp, _vp, _vp]),
    "hoh_encode_images": (_int, [_vp, _vp, _sz, _u32, _u32, _int, C.c_uint, _vp, _sz, _vp, _vp]),
    "hoh_decode_images": (_int, [_vp, _vp, _sz, _vp, _sz, _u32, _u32, _vp, _vp]),
    "hoh_encode_images_host": (_int, [_vp, _vp, _sz, _u32, _u32, _int, C.c_uint, _vp, _sz, _vp, _vp]),
    "hoh_decode_images_host": (_int, [_vp, _vp, _sz, _vp, _sz, _u32, _u32, _vp, _vp]),
    "hoh_decode_regions": (_int, [_vp, _vp, _sz, _vp, _sz, _u32, _u32, _vp, _u32, _u32, _vp, _vp]),
    "hoh_decode_regions_host": (_int, [_vp, _vp, _sz, _vp, _sz, _u32, _u32, _vp, _u32, _u32, _vp, _vp]),
    "hoh_find_lz_stride": (_sz, [_int, _int]),
    "hoh_find_lz_rgb_batch": (_int, [_vp, _vp, _sz, _int, _int, _int, C.c_uint, _vp, _vp, _vp, _sz, _vp, _vp]),
    "hoh_find_lz_images": (_int, [_vp, _vp, _sz, _u32, _u32, _int, C.c_uint, _vp, _vp, _vp, _sz, _vp, _vp]),
    "hoh_find_lz_rgb": (_int, [_vp, _vp, _sz, _int, _int, _vp, _sz, _vp, _int, _int, C.POINTER(_sz)]),
    "hoh_layer_encode_out_bytes": (_sz, [_sz, _int, _int, _int, _int]),
    "hoh_layer_encode_batch": (_int, [_vp, _vp, _sz, _int, _int, _int, _int, C.c_uint, _vp, _sz, _u32, _vp, _sz, _vp, _vp,
                                      _sz, _vp]),
    "hoh_channel_picker_dev": (_int, [_vp, _vp, _sz, _int, _int, _vp]),
    "hoh_channel_picker": (_int, [_vp, _vp, _sz, _int, _int, _vp]),
    "hoh_encode_entropy": (_int, [_vp, _vp, _sz, _sz, _vp, _sz, _u32, C.POINTER(_sz), C.POINTER(_int)]),
    "hoh_encode_entropy_8bit": (_int, [_vp, _vp, _sz, _sz, _vp, _sz, _u32, C.POINTER(_sz), C.POINTER(_int)]),
    "hoh_decode_entropy": (_int, [_vp, _vp, _sz, C.POINTER(_sz), _vp, _sz, C.POINTER(_sz), C.c_uint,
                                  C.POINTER(_int)]),
    "hoh_normalize_freqs": (_int, [_vp, _vp, _vp, _sz, _u32, C.POINTER(_int)]),
    "hoh_subtract_green": (_int, [_vp, _vp, _sz, _vp, _vp, _vp]),
    "hoh_add_green": (_int, [_vp, _vp, _vp, _vp, _sz, _vp]),
    "hoh_channelpredict_fastpath": (_int, [_vp, _vp, _int, _int, _int, _vp]),
    "hoh_channelpredict_section": (_int, [_vp, _vp, _int, _int, _int, _int, _int, _int, _int, C.c_uint16, _vp, _sz,
                                          C.POINTER(_sz)]),
    "hoh_channelpredict_all": (_int, [_vp, _vp, _int, _int, _int, _int, _int, _vp, _vp]),
    "hoh_unpredict_all": (_int, [_vp, _vp, _sz, _int, _int, _int, _int, _int, _vp, _vp, _vp]),
    "hoh_unpredict_fastpath": (_int, [_vp, _vp, _sz, _int, _int, _int, _vp, _vp]),
    "hoh_predictor_search": (_int, [_vp, _vp, _int, _int, _int, _int, _vp, _vp, _vp]),
}

_lib = None


def load_library(path=LIB_PATH):
    """dlopen libhohgpu.so and type every entry point.  Raises if the library is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} not built: run `python hoh-ans_b200/build.py` (no CPU fallback exists)")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class DeviceBuffer:
    """A device allocation owned through the C-ABI (hoh_dev_alloc / hoh_dev_free)."""

    def __init__(self, gpu, nbytes):
        self.gpu, self.nbytes = gpu, int(nbytes)
        p = C.c_void_p()
        gpu._ck(gpu.lib.hoh_dev_alloc(gpu.ctx, self.nbytes, C.byref(p)), "hoh_dev_alloc")
        self.ptr = p.value

    def upload(self, arr, offset=0):
        arr = np.ascontiguousarray(arr)
        assert offset + arr.nbytes <= self.nbytes
        self.gpu._ck(self.gpu.lib.hoh_h2d(self.gpu.ctx, self.ptr + offset, _ptr(arr), arr.nbytes), "hoh_h2d")
        self.gpu.sync()
        return self

    def download(self, dtype, count, offset=0):
        out = np.empty(count, dtype)
        assert offset + out.nbytes <= self.nbytes
        self.gpu._ck(self.gpu.lib.hoh_d2h(self.gpu.ctx, _ptr(out), self.ptr + offset, out.nbytes), "hoh_d2h")
        self.gpu.sync()
        return out

    def zero(self):
        self.gpu._ck(self.gpu.lib.hoh_dev_memset(self.gpu.ctx, self.ptr, 0, self.nbytes), "hoh_dev_memset")

    def free(self):
        if self.ptr:
            self.gpu.lib.hoh_dev_free(self.gpu.ctx, self.ptr)
            self.ptr = None


class HohGpu:
    """One context = one GPU + one stream.  Methods carry the reference's function names."""

    def __init__(self, device=0, cuda_stream=None):
        self.lib = load_library()
        ctx = C.c_void_p()
        st = self.lib.hoh_ctx_create(device, cuda_stream, C.byref(ctx))
        if st != HOH_OK:
            raise HohError(st, "hoh_ctx_create", "(no CUDA device? this library has no CPU fallback)")
        self.ctx = ctx
        self.device = device

    def close(self):
        if self.ctx:
            self.lib.hoh_ctx_destroy(self.ctx)
            self.ctx = None

    def _ck(self, st, where):
        if st != HOH_OK:
            detail = self.lib.hoh_strerror(st).decode()
            if st == HOH_E_CUDA:
                detail += " | " + self.lib.hoh_last_cuda_error(self.ctx).decode()
            raise HohError(st, where, detail)

    def sync(self):
        self._ck(self.lib.hoh_sync(self.ctx), "hoh_sync")

    def release_scratch(self):
        self._ck(self.lib.hoh_release_scratch(self.ctx), "hoh_release_scratch")

    def layer_stats(self):
        """(candidates coded, planes coded in full, planes) of the mode >= 1 encoder since the last call."""
        out = (C.c_uint64 * 3)()
        self._ck(self.lib.hoh_debug_layer_stats(self.ctx, out), "hoh_debug_layer_stats")
        return int(out[0]), int(out[1]), int(out[2])

    def launch_count(self):
        return int(self.lib.hoh_launch_count(self.ctx))

    def alloc(self, nbytes):
        return DeviceBuffer(self, nbytes)

    def timer_start(self, slot=0):
        self._ck(self.lib.hoh_timer_start(self.ctx, slot), "hoh_timer_start")

    def timer_stop(self, slot=0):
        self._ck(self.lib.hoh_timer_stop(self.ctx, slot), "hoh_timer_stop")

    def timer_ms(self, slot=0):
        ms = C.c_float()
        self._ck(self.lib.hoh_timer_elapsed_ms(self.ctx, slot, C.byref(ms)), "hoh_timer_elapsed_ms")
        return float(ms.value)

    def flush_l2(self):
        self._ck(self.lib.hoh_flush_l2(self.ctx), "hoh_flush_l2")

    def profile_begin(self):
        self._ck(self.lib.hoh_profile_begin(self.ctx), "hoh_profile_begin")

    def profile_end(self):
        """-> {kernel name: (total_ms, launches)} since profile_begin."""
        self._ck(self.lib.hoh_profile_end(self.ctx), "hoh_profile_end")
        out = {}
        for i in range(self.lib.hoh_profile_count(self.ctx)):
            name, ms, cnt = C.c_char_p(), C.c_double(), C.c_uint64()
            self._ck(self.lib.hoh_profile_entry(self.ctx, i, C.byref(name), C.byref(ms), C.byref(cnt)),
                     "hoh_profile_entry")
            out[name.value.decode()] = (ms.value, int(cnt.value))
        return out

    def host_alloc(self, nbytes, dtype=np.uint8):
        """Pinned host memory as a numpy array (hoh_host_alloc); keep the HohGpu alive while it is used."""
        p = C.c_void_p()
        self._ck(self.lib.hoh_host_alloc(self.ctx, int(nbytes), C.byref(p)), "hoh_host_alloc")
        buf = (C.c_uint8 * int(nbytes)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=np.uint8).view(dtype)
        return arr

    def host_free(self, arr):
        """Release an array from host_alloc (the caller drops every view of it)."""
        self._ck(self.lib.hoh_host_free(self.ctx, C.c_void_p(arr.ctypes.data)), "hoh_host_free")

    # ---- compat shims: reference names, reference value semantics -------------------------------
    def encode_entropy(self, symbols, range_, prob_bits):
        """entropy_encoding.hpp:8 -> (bytes, stream_status)."""
        symbols = np.ascontiguousarray(symbols, dtype=np.uint16)
        cap = 4096 + 4 * int(range_) + 4 * len(symbols)
        out = np.zeros(cap, np.uint8)
        size, sst = C.c_size_t(0), C.c_int(0)
        st = self.lib.hoh_encode_entropy(self.ctx, _ptr(symbols), len(symbols), range_, _ptr(out), cap, prob_bits,
                                         C.byref(size), C.byref(sst))
        if st == HOH_E_STREAM:
            return out[:0].copy(), sst.value
        self._ck(st, "hoh_encode_entropy")
        return out[:size.value].copy(), sst.value

    def encode_entropy_8bit(self, symbols, range_, prob_bits):
        symbols = np.ascontiguousarray(symbols, dtype=np.uint8)
        cap = 4096 + 4 * int(range_) + 4 * len(symbols)
        out = np.zeros(cap, np.uint8)
        size, sst = C.c_size_t(0), C.c_int(0)
        st = self.lib.hoh_encode_entropy_8bit(self.ctx, _ptr(symbols), len(symbols), range_, _ptr(out), cap,
                                              prob_bits, C.byref(size), C.byref(sst))
        if st == HOH_E_STREAM:
            return out[:0].copy(), sst.value
        self._ck(st, "hoh_encode_entropy_8bit")
        return out[:size.value].copy(), sst.value

    def decode_entropy(self, stream, byte_pointer=0, flags=FIX_ALL, cap=1 << 22):
        """entropy_decoding.hpp:134 -> (symbols, byte_pointer_after, stream_status)."""
        stream = np.ascontiguousarray(stream, dtype=np.uint8)
        out = np.zeros(cap, np.uint16)
        bp, n, sst = C.c_size_t(byte_pointer), C.c_size_t(0), C.c_int(0)
        st = self.lib.hoh_decode_entropy(self.ctx, _ptr(stream), len(stream), C.byref(bp), _ptr(out), cap,
                                         C.byref(n), flags, C.byref(sst))
        if st not in (HOH_OK, HOH_E_STREAM, HOH_E_CAPACITY):
            self._ck(st, "hoh_decode_entropy")
        return out[:min(n.value, cap)].copy(), bp.value, sst.value

    def normalize_freqs(self, freqs, target_total):
        """stattools.hpp:13 -> (freqs, cum_freqs, status)."""
        f = np.ascontiguousarray(freqs, dtype=np.uint32).copy()
        cum = np.zeros(len(f) + 1, np.uint32)
        sst = C.c_int(0)
        st = self.lib.hoh_normalize_freqs(self.ctx, _ptr(f), _ptr(cum), len(f), target_total, C.byref(sst))
        if st == HOH_E_STREAM:
            return f, cum, sst.value
        self._ck(st, "hoh_normalize_freqs")
        return f, cum, 0

    def subtract_green(self, rgb):
        """channel.hpp:73 -> (G, R-G+256, B-G+256) as u16 planes."""
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).ravel()
        px = rgb.size // 3
        g, rg, bg = (np.zeros(px, np.uint16) for _ in range(3))
        self._ck(self.lib.hoh_subtract_green(self.ctx, _ptr(rgb), rgb.size, _ptr(g), _ptr(rg), _ptr(bg)),
                 "hoh_subtract_green")
        return g, rg, bg

    def add_green(self, g, rg, bg):
        g, rg, bg = (np.ascontiguousarray(a, dtype=np.uint16) for a in (g, rg, bg))
        rgb = np.zeros(g.size * 3, np.uint8)
        self._ck(self.lib.hoh_add_green(self.ctx, _ptr(g), _ptr(rg), _ptr(bg), g.size, _ptr(rgb)), "hoh_add_green")
        return rgb

    def channelpredict_fastpath(self, data, w, h, depth):
        data = np.ascontiguousarray(data, dtype=np.uint16)
        out = np.zeros(w * h, np.uint16)
        self._ck(self.lib.hoh_channelpredict_fastpath(self.ctx, _ptr(data), w, h, depth, _ptr(out)),
                 "hoh_channelpredict_fastpath")
        return out

    def channelpredict_section(self, data, w, h, depth, x_tiles, y_tiles, x, y, predictor):
        data = np.ascontiguousarray(data, dtype=np.uint16)
        out = np.zeros(w * h, np.uint16)
        cnt = C.c_size_t(0)
        self._ck(self.lib.hoh_channelpredict_section(self.ctx, _ptr(data), w, h, depth, x_tiles, y_tiles, x, y,
                                                     predictor, _ptr(out), out.size, C.byref(cnt)),
                 "hoh_channelpredict_section")
        return out[:cnt.value].copy()

    def channelpredict_all(self, data, w, h, depth, x_tiles, y_tiles, tile_map):
        data = np.ascontiguousarray(data, dtype=np.uint16)
        tile_map = np.ascontiguousarray(tile_map, dtype=np.uint16)
        out = np.zeros(w * h, np.uint16)
        self._ck(self.lib.hoh_channelpredict_all(self.ctx, _ptr(data), w, h, depth, x_tiles, y_tiles, _ptr(tile_map),
                                                 _ptr(out)), "hoh_channelpredict_all")
        return out

    def unpredict_all(self, resid, w, h, depth, x_tiles, y_tiles, tile_map, backref=None):
        resid = np.ascontiguousarray(resid, dtype=np.uint16)
        tile_map = np.ascontiguousarray(tile_map, dtype=np.uint16)
        if backref is not None:
            backref = np.ascontiguousarray(backref, dtype=np.uint16)
        out = np.zeros(w * h, np.uint16)
        self._ck(self.lib.hoh_unpredict_all(self.ctx, _ptr(resid), resid.size, w, h, depth, x_tiles, y_tiles,
                                            _ptr(tile_map), _ptr(backref), _ptr(out)), "hoh_unpredict_all")
        return out

    def unpredict_fastpath(self, resid, w, h, depth, backref=None):
        resid = np.ascontiguousarray(resid, dtype=np.uint16)
        if backref is not None:
            backref = np.ascontiguousarray(backref, dtype=np.uint16)
        out = np.zeros(w * h, np.uint16)
        self._ck(self.lib.hoh_unpredict_fastpath(self.ctx, _ptr(resid), resid.size, w, h, depth, _ptr(backref),
                                                 _ptr(out)), "hoh_unpredict_fastpath")
        return out

    def predictor_search(self, plane, w, h, depth, mode):
        """layer_encode.hpp:126-272 -> (tile_map, index_list, final residuals)."""
        plane = np.ascontiguousarray(plane, dtype=np.uint16)
        cells = ((w + 39) // 40) * ((h + 39) // 40)
        tmap = np.zeros(cells, np.uint16)
        idx = np.zeros(cells, np.uint8)
        resid = np.zeros(w * h, np.uint16)
        self._ck(self.lib.hoh_predictor_search(self.ctx, _ptr(plane), w, h, depth, mode, _ptr(tmap), _ptr(idx),
                                               _ptr(resid)), "hoh_predictor_search")
        return tmap, idx, resid

    # ---- batched, device resident ----------------------------------------------------------------
    def tile_geometry(self, width, height):
        g = TileGeometry()
        self._ck(self.lib.hoh_tile_geometry_for(width, height, C.byref(g)), "hoh_tile_geometry_for")
        return g

    def enc_slab_bytes(self, n, prob_bits):
        return int(self.lib.hoh_enc_slab_bytes(n, prob_bits))

    def encode_entropy_batch(self, symbol_arrays, ranges, prob_bits_list, prefixes=None):
        """Many encode_entropy calls in one launch sequence -> list of (bytes, status, stored)."""
        k = len(symbol_arrays)
        desc = np.zeros(k, ENC_STREAM_DT)
        sym_off = out_off = 0
        for i, (s, r, pb) in enumerate(zip(symbol_arrays, ranges, prob_bits_list)):
            desc[i]["sym_off"], desc[i]["n"], desc[i]["range"], desc[i]["prob_bits"] = sym_off, len(s), r, pb
            cap = self.enc_slab_bytes(len(s), pb)
            desc[i]["out_off"], desc[i]["out_cap"] = out_off, cap
            if prefixes is not None:
                p = prefixes[i]
                desc[i]["prefix_len"] = len(p)
                desc[i]["prefix"][:len(p)] = np.frombuffer(bytes(p), np.uint8)
            sym_off += (len(s) + 7) & ~7
            out_off += cap
        syms = np.zeros(max(sym_off, 8), np.uint16)
        for i, s in enumerate(symbol_arrays):
            o = int(desc[i]["sym_off"])
            syms[o:o + len(s)] = s
        d_sym = self.alloc(syms.nbytes).upload(syms)
        d_desc = self.alloc(desc.nbytes).upload(desc)
        d_out = self.alloc(max(out_off, 16))
        d_res = self.alloc(k * RESULT_DT.itemsize)
        try:
            self._ck(self.lib.hoh_encode_entropy_batch(self.ctx, d_desc.ptr, k, d_sym.ptr, d_out.ptr, d_res.ptr,
                                                       int(max(ranges)), int(max(prob_bits_list)),
                                                       int(max(len(s) for s in symbol_arrays))),
                     "hoh_encode_entropy_batch")
            res = d_res.download(RESULT_DT, k)
            blob = d_out.download(np.uint8, max(out_off, 16))
        finally:
            for b in (d_sym, d_desc, d_out, d_res):
                b.free()
        return [(blob[int(r["start"]):int(r["start"]) + int(r["size"])].copy(), int(r["status"]), int(r["stored"]))
                for r in res]

    def decode_entropy_batch(self, blob, offsets, caps, flags=FIX_ALL):
        """Many decode_entropy calls -> list of (symbols, end_off, status)."""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        k = len(offsets)
        desc = np.zeros(k, DEC_STREAM_DT)
        sym_off = 0
        for i, (o, cpt) in enumerate(zip(offsets, caps)):
            desc[i]["in_off"], desc[i]["sym_off"], desc[i]["sym_cap"], desc[i]["flags"] = o, sym_off, cpt, flags
            sym_off += (cpt + 7) & ~7
        padded = np.concatenate([blob, np.zeros(48 - len(blob) % 16, np.uint8)])
        d_in = self.alloc(padded.nbytes).upload(padded)
        d_desc = self.alloc(desc.nbytes).upload(desc)
        d_sym = self.alloc(max(sym_off, 8) * 2)
        d_res = self.alloc(k * DEC_RESULT_DT.itemsize)
        try:
            self._ck(self.lib.hoh_decode_entropy_batch(self.ctx, d_desc.ptr, k, d_in.ptr, padded.nbytes, d_sym.ptr,
                                                       d_res.ptr, int(max(caps))), "hoh_decode_entropy_batch")
            res = d_res.download(DEC_RESULT_DT, k)
            self.last_dec_results = res  # the full records (stored, prob_bits, table_mode ...) of the last call
            syms = d_sym.download(np.uint16, max(sym_off, 8))
        finally:
            for b in (d_in, d_desc, d_sym, d_res):
                b.free()
        out = []
        for i, r in enumerate(res):
            o = int(desc[i]["sym_off"])
            n = min(int(r["n"]), int(caps[i]))
            out.append((syms[o:o + n].copy(), int(r["end_off"]), int(r["status"])))
        return out

    def encode_images_s0(self, rgb, n_images, width, height):
        """Host-buffer convenience over hoh_encode_images_s0: rgb (n_images*H*W*3 u8) ->
        (packed bytes, offsets[n_streams+1], results).  H2D and D2H copies included."""
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).ravel()
        g = self.tile_geometry(width, height)
        n_streams = n_images * g.streams_per_image
        out_bytes = int(self.lib.hoh_encode_images_out_bytes(C.byref(g), n_images))
        d_rgb = self.alloc(rgb.nbytes).upload(rgb)
        d_out = self.alloc(out_bytes)
        d_res = self.alloc(n_streams * RESULT_DT.itemsize)
        packed_cap = rgb.nbytes * 2 + 4096 * n_streams
        d_packed = self.alloc(packed_cap)
        d_off = self.alloc((n_streams + 1) * 8)
        try:
            self._ck(self.lib.hoh_encode_images_s0(self.ctx, d_rgb.ptr, n_images, width, height, None, d_out.ptr,
                                                   out_bytes, d_res.ptr, d_packed.ptr, packed_cap, d_off.ptr),
                     "hoh_encode_images_s0")
            off = d_off.download(np.uint64, n_streams + 1)
            res = d_res.download(RESULT_DT, n_streams)
            packed = d_packed.download(np.uint8, int(off[-1]))
        finally:
            for b in (d_rgb, d_out, d_res, d_packed, d_off):
                b.free()
        return packed, off, res

    def find_lz_rgb(self, rgb, width, height, distance, bonus):
        """lz.hpp:6 -> (lz bytes, nuke map)."""
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).ravel()
        cap = int(self.lib.hoh_find_lz_stride(width, height))
        out = np.zeros(cap, np.uint8)
        nuke = np.zeros(rgb.size // 3, np.uint8)
        n = _sz(0)
        self._ck(self.lib.hoh_find_lz_rgb(self.ctx, _ptr(rgb), rgb.size, width, height, _ptr(out), cap, _ptr(nuke),
                                          distance, bonus, C.byref(n)), "hoh_find_lz_rgb")
        return out[:n.value].copy(), nuke

    def find_lz_rgb_batch(self, tiles, n_tiles, width, height, distance, bonus=None):
        """tiles: n_tiles*H*W*3 u8; bonus: per-tile int32 array or None (derived from the colour count on the
        device) -> list of (lz bytes, nuke map, status)."""
        tiles = np.ascontiguousarray(tiles, dtype=np.uint8).ravel()
        npx = width * height
        assert tiles.size == n_tiles * npx * 3
        stride = int(self.lib.hoh_find_lz_stride(width, height))
        d_rgb = self.alloc(tiles.nbytes).upload(tiles)
        d_nuke = self.alloc(n_tiles * npx)
        d_lz = self.alloc(n_tiles * stride)
        d_size = self.alloc(n_tiles * 4)
        d_st = self.alloc(n_tiles * 4)
        d_bonus = None
        if bonus is not None:
            b = np.ascontiguousarray(bonus, dtype=np.int32)
            d_bonus = self.alloc(b.nbytes).upload(b)
        try:
            self._ck(self.lib.hoh_find_lz_rgb_batch(self.ctx, d_rgb.ptr, n_tiles, width, height, distance, 0,
                                                    d_bonus.ptr if d_bonus else None, d_nuke.ptr, d_lz.ptr, stride,
                                                    d_size.ptr, d_st.ptr), "hoh_find_lz_rgb_batch")
            sizes = d_size.download(np.uint32, n_tiles)
            st = d_st.download(np.int32, n_tiles)
            lz = d_lz.download(np.uint8, n_tiles * stride).reshape(n_tiles, stride)
            nuke = d_nuke.download(np.uint8, n_tiles * npx).reshape(n_tiles, npx)
        finally:
            for buf in (d_rgb, d_nuke, d_lz, d_size, d_st, d_bonus):
                if buf is not None:
                    buf.free()
        return [(lz[i, :int(sizes[i])].copy(), nuke[i].copy(), int(st[i])) for i in range(n_tiles)]

    def encode_tiles_s0_lz(self, rgb, n_images, width, height):
        """Device-side pieces of encode_tile (choh.cpp:104) at mode 0 for photographic tiles: LZ records +
        NUKE maps (hoh_find_lz_images) and the three channel payloads coded with those maps
        (hoh_encode_images_s0) -> (list of lz bytes per tile, packed, offsets, results)."""
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).ravel()
        g = self.tile_geometry(width, height)
        n_tiles = n_images * g.tiles_per_image
        n_streams = n_tiles * 3
        nuke_stride = (g.tile_w * g.tile_h + 7) & ~7
        lz_stride = int(self.lib.hoh_find_lz_stride(g.tile_w, g.tile_h))
        out_bytes = int(self.lib.hoh_encode_images_out_bytes(C.byref(g), n_images))
        packed_cap = rgb.nbytes * 2 + 4096 * n_streams
        bufs = [self.alloc(rgb.nbytes).upload(rgb), self.alloc(n_tiles * nuke_stride), self.alloc(n_tiles * lz_stride),
                self.alloc(n_tiles * 4), self.alloc(n_tiles * 4), self.alloc(out_bytes),
                self.alloc(n_streams * RESULT_DT.itemsize), self.alloc(packed_cap), self.alloc((n_streams + 1) * 8)]
        d_rgb, d_nuke, d_lz, d_size, d_st, d_out, d_res, d_packed, d_off = bufs
        try:
            self._ck(self.lib.hoh_find_lz_images(self.ctx, d_rgb.ptr, n_images, width, height, 6, 0, None, d_nuke.ptr,
                                                 d_lz.ptr, lz_stride, d_size.ptr, d_st.ptr), "hoh_find_lz_images")
            self._ck(self.lib.hoh_encode_images_s0(self.ctx, d_rgb.ptr, n_images, width, height, d_nuke.ptr, d_out.ptr,
                                                   out_bytes, d_res.ptr, d_packed.ptr, packed_cap, d_off.ptr),
                     "hoh_encode_images_s0")
            assert (d_st.download(np.int32, n_tiles) == 0).all()
            sizes = d_size.download(np.uint32, n_tiles)
            lz = d_lz.download(np.uint8, n_tiles * lz_stride).reshape(n_tiles, lz_stride)
            off = d_off.download(np.uint64, n_streams + 1)
            res = d_res.download(RESULT_DT, n_streams)
            packed = d_packed.download(np.uint8, int(off[-1]))
        finally:
            for b in bufs:
                b.free()
        return [lz[t, :int(sizes[t])].copy() for t in range(n_tiles)], packed, off, res

    def channel_picker(self, src, total, target):
        """channel.hpp:63"""
        src = np.ascontiguousarray(src, dtype=np.uint8).ravel()
        out = np.zeros(src.size // total, np.uint16)
        self._ck(self.lib.hoh_channel_picker(self.ctx, _ptr(src), src.size, total, target, _ptr(out)), "hoh_channel_picker")
        return out

    def encode_images(self, rgb, n_images, width, height, mode, flags=0):
        """hoh_encode_images: encode_tile for every tile -> (list of tile bytes, TILE_DT records)."""
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).ravel()
        g = self.tile_geometry(width, height)
        n_tiles = n_images * g.tiles_per_image
        packed_cap = rgb.nbytes * 2 + 8192 * n_tiles
        d_rgb = self.alloc(rgb.nbytes).upload(rgb)
        d_packed = self.alloc(packed_cap)
        d_off = self.alloc((n_tiles + 1) * 8)
        d_tiles = self.alloc(n_tiles * TILE_DT.itemsize)
        try:
            self._ck(self.lib.hoh_encode_images(self.ctx, d_rgb.ptr, n_images, width, height, mode, flags, d_packed.ptr,
                                                packed_cap, d_off.ptr, d_tiles.ptr), "hoh_encode_images")
            off = d_off.download(np.uint64, n_tiles + 1)
            rec = d_tiles.download(TILE_DT, n_tiles)
            packed = d_packed.download(np.uint8, int(off[-1]))
        finally:
            for b in (d_rgb, d_packed, d_off, d_tiles):
                b.free()
        return [packed[int(off[t]):int(off[t + 1])].tobytes() for t in range(n_tiles)], rec

    def decode_images(self, tiles, n_images, width, height):
        """hoh_decode_images: list of tile byte strings (n_images * tiles_per_image) -> (rgb u8, status per tile)."""
        off = np.zeros(len(tiles) + 1, np.uint64)
        off[1:] = np.cumsum([len(t) for t in tiles])
        blob = np.frombuffer(b"".join(tiles) + bytes(64), np.uint8)
        d_packed = self.alloc(blob.nbytes).upload(blob)
        d_off = self.alloc(off.nbytes).upload(off)
        d_rgb = self.alloc(n_images * width * height * 3)
        d_rgb.zero()
        d_st = self.alloc(len(tiles) * 4)
        try:
            self._ck(self.lib.hoh_decode_images(self.ctx, d_packed.ptr, blob.nbytes, d_off.ptr, n_images, width, height,
                                                d_rgb.ptr, d_st.ptr), "hoh_decode_images")
            rgb = d_rgb.download(np.uint8, n_images * width * height * 3)
            st = d_st.download(np.int32, len(tiles))
        finally:
            for b in (d_packed, d_off, d_rgb, d_st):
                b.free()
        return rgb, st

    def encode_images_host(self, rgb, n_images, width, height, mode, flags=0):
        """hoh_encode_images_host: pinned host buffers in and out, chunked and pipelined inside the library ->
        (packed u8 view, tile offsets, TILE_DT records)."""
        g = self.tile_geometry(width, height)
        n_tiles = n_images * g.tiles_per_image
        raw = n_images * width * height * 3
        src = self.host_alloc(raw)
        src[:] = np.asarray(rgb, dtype=np.uint8).ravel()
        cap = raw + raw // 2 + 8192 * n_tiles
        packed = self.host_alloc(cap)
        off = np.zeros(n_tiles + 1, np.uint64)
        rec = np.zeros(n_tiles, TILE_DT)
        self._ck(self.lib.hoh_encode_images_host(self.ctx, _ptr(src), n_images, width, height, mode, flags, _ptr(packed),
                                                 cap, _ptr(off), _ptr(rec)), "hoh_encode_images_host")
        return packed[:int(off[-1])], off, rec

    def decode_images_host(self, packed, off, n_images, width, height):
        """hoh_decode_images_host: exact-size host buffers -> (rgb, per-tile status)."""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        rgb = self.host_alloc(n_images * width * height * 3)
        st = np.zeros(len(off) - 1, np.int32)
        self._ck(self.lib.hoh_decode_images_host(self.ctx, _ptr(packed), packed.size, _ptr(off), n_images, width, height,
                                                 _ptr(rgb), _ptr(st)), "hoh_decode_images_host")
        return rgb, st

    def decode_regions(self, tiles, n_images, width, height, origins, crop_w, crop_h, fill=0):
        """hoh_decode_regions: list of tile byte strings (n_images * tiles_per_image), origins (n_images x 2: x, y of
        each window) -> (crops u8 (n_images, crop_h, crop_w, 3), status per image).  fill: the byte the crops hold
        before the call (what a failing tile leaves)."""
        off = np.zeros(len(tiles) + 1, np.uint64)
        off[1:] = np.cumsum([len(t) for t in tiles])
        blob = np.frombuffer(b"".join(tiles) + bytes(64), np.uint8)
        org = np.ascontiguousarray(origins, dtype=np.uint32).reshape(n_images, 2)
        crop_bytes = n_images * crop_w * crop_h * 3
        d_packed = self.alloc(blob.nbytes).upload(blob)
        d_off = self.alloc(off.nbytes).upload(off)
        d_org = self.alloc(max(org.nbytes, 8)).upload(org)
        d_crops = self.alloc(max(crop_bytes, 1))
        self._ck(self.lib.hoh_dev_memset(self.ctx, d_crops.ptr, fill, max(crop_bytes, 1)), "hoh_dev_memset")
        d_st = self.alloc(max(n_images, 1) * 4)
        try:
            self._ck(self.lib.hoh_decode_regions(self.ctx, d_packed.ptr, blob.nbytes, d_off.ptr, n_images, width, height,
                                                 d_org.ptr, crop_w, crop_h, d_crops.ptr, d_st.ptr), "hoh_decode_regions")
            crops = d_crops.download(np.uint8, crop_bytes)
            st = d_st.download(np.int32, n_images)
        finally:
            for b in (d_packed, d_off, d_org, d_crops, d_st):
                b.free()
        return crops.reshape(n_images, crop_h, crop_w, 3), st

    def decode_regions_host(self, packed, off, n_images, width, height, origins, crop_w, crop_h):
        """hoh_decode_regions_host: exact-size host buffers and origins (n_images x 2) -> (crops (n_images, crop_h,
        crop_w, 3), status per image).  Only the touched tiles' bytes are copied to the device."""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        org = np.ascontiguousarray(origins, dtype=np.uint32).reshape(n_images, 2)
        crops = self.host_alloc(n_images * crop_w * crop_h * 3)
        st = np.zeros(n_images, np.int32)
        self._ck(self.lib.hoh_decode_regions_host(self.ctx, _ptr(packed), packed.size, _ptr(off), n_images, width, height,
                                                  _ptr(org), crop_w, crop_h, _ptr(crops), _ptr(st)),
                 "hoh_decode_regions_host")
        return crops.reshape(n_images, crop_h, crop_w, 3), st

    def layer_encode_batch(self, planes, n_planes, w, h, depth, mode, nuke=None, planes_per_map=1, flags=0):
        """layer_encode.hpp:11 for n_planes planes of the same shape -> list of (payload bytes, status, kept slot).
        nuke: (n_planes / planes_per_map) maps of w*h bytes, or None."""
        planes = np.ascontiguousarray(planes, dtype=np.uint16).ravel()
        assert planes.size == n_planes * w * h
        d_nuke = None
        if nuke is not None:
            nuke = np.ascontiguousarray(nuke, dtype=np.uint8).ravel()
            assert nuke.size * planes_per_map == n_planes * w * h
            d_nuke = self.alloc(nuke.nbytes).upload(nuke)
        out_bytes = int(self.lib.hoh_layer_encode_out_bytes(n_planes, w, h, depth, mode))
        d_pl = self.alloc(planes.nbytes).upload(planes)
        d_out = self.alloc(out_bytes)
        d_res = self.alloc(n_planes * RESULT_DT.itemsize)
        packed_cap = planes.nbytes * 2 + 4096 * n_planes
        d_packed = self.alloc(packed_cap)
        d_off = self.alloc((n_planes + 1) * 8)
        try:
            self._ck(self.lib.hoh_layer_encode_batch(self.ctx, d_pl.ptr, n_planes, w, h, depth, mode, flags,
                                                     d_nuke.ptr if d_nuke else None, w * h, planes_per_map, d_out.ptr,
                                                     out_bytes, d_res.ptr, d_packed.ptr, packed_cap, d_off.ptr),
                     "hoh_layer_encode_batch")
            off = d_off.download(np.uint64, n_planes + 1)
            res = d_res.download(RESULT_DT, n_planes)
            packed = d_packed.download(np.uint8, int(off[-1]))
        finally:
            for b in (d_pl, d_out, d_res, d_packed, d_off, d_nuke):
                if b is not None:
                    b.free()
        return [(packed[int(off[i]):int(off[i + 1])].tobytes(), int(res[i]["status"]), int(res[i]["stored"]))
                for i in range(n_planes)]

    def decode_images_s0(self, packed, offsets, n_images, width, height, backref=None):
        """Host-buffer convenience over hoh_decode_images_s0 -> (rgb, per-stream status).  backref: u16 maps, tile t's
        at t * plane_stride (tile_w*tile_h rounded up to 8), or None."""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        g = self.tile_geometry(width, height)
        n_streams = n_images * g.streams_per_image
        padded = np.concatenate([packed, np.zeros(48 - len(packed) % 16, np.uint8)])
        d_packed = self.alloc(padded.nbytes).upload(padded)
        d_off = self.alloc(offsets.nbytes).upload(offsets)
        d_rgb = self.alloc(n_images * width * height * 3)
        d_rgb.zero()
        d_st = self.alloc(n_streams * 4)
        d_br = None
        if backref is not None:
            backref = np.ascontiguousarray(backref, dtype=np.uint16).ravel()
            d_br = self.alloc(backref.nbytes).upload(backref)
        try:
            self._ck(self.lib.hoh_decode_images_s0(self.ctx, d_packed.ptr, padded.nbytes, d_off.ptr, n_images, width,
                                                   height, d_br.ptr if d_br else None, d_rgb.ptr, d_st.ptr),
                     "hoh_decode_images_s0")
            rgb = d_rgb.download(np.uint8, n_images * width * height * 3)
            st = d_st.download(np.int32, n_streams)
        finally:
            for b in (d_packed, d_off, d_rgb, d_st, d_br):
                if b is not None:
                    b.free()
        return rgb, st
