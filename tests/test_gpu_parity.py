"""GPU parity: every stage of the CUDA path, called through the C-ABI, against the CPU oracle
(oracle/hoh_oracle.c, pinned to the real reference) and the committed golden vectors.
Bit-exact everywhere: this is integer / byte work."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

import gpu_lib
import oracle_lib as ol

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
STOCK = [0x0001, 0x0002, 0x0020, 0x0010, 0xffbf, 0x0003, 0xfffd, 0xfffb, 0xfff7, 0xffef, 0xffdf,
         0xff7f, 0xfdff, 0xffff]


def _cases(npz, suffix):
    return sorted({k[: -len(suffix)] for k in npz.files if k.endswith(suffix)})


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


def _smooth_plane(rng, w, h, depth):
    yy, xx = np.mgrid[0:h, 0:w]
    c = 1 << depth
    base = (np.sin(xx / 9.0) + np.cos(yy / 7.0) + (xx + yy) / (w + h)) * c / 6 + c / 2
    return np.clip(np.rint(base + rng.normal(0, 2.0, (h, w))), 0, c - 1).astype(np.uint16).ravel()


# ---------------------------------------------------------------------------------------------
# entropy coder
# ---------------------------------------------------------------------------------------------
def test_encode_entropy_golden_vectors():
    """entropy_encoding.hpp:8 — reference-generated fixtures incl. the 817-byte known answer."""
    g = gpu_lib.gpu()
    z = np.load(os.path.join(G, "entropy.npz"))
    for name in _cases(z, "__sym"):
        sym, (rangev, pb), want = z[name + "__sym"], z[name + "__par"], z[name + "__out"]
        got, st = g.encode_entropy(sym, int(rangev), int(pb))
        assert st == 0 and got.tobytes() == want.tobytes(), name
    out, _ = g.encode_entropy(z["text817__sym"], 256, 12)
    assert hashlib.md5(out.tobytes()).hexdigest() == "c5d8fa190d78049ed26a5ebcf06e3ddd"
    out8, _ = g.encode_entropy_8bit(z["text817__sym"].astype(np.uint8), 256, 12)
    assert out8.tobytes() == out.tobytes()


def test_encode_entropy_batch_random_streams_vs_oracle():
    """Ragged batch: ranges 1..512, prob_bits 1..19, empty / single-symbol / stored-mode streams."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(11)
    syms, ranges, pbs, want = [], [], [], []
    for it in range(700):
        rangev = int(rng.choice([1, 2, 3, 5, 14, 16, 255, 256, 257, 512]))
        pb = int(rng.integers(8, 20))
        if (1 << pb) < rangev:
            pb = 10
        n = int(rng.choice([1, 2, 7, 20, 49, 63, 64, 65, 100, 1000, 5000, 70000])) if it % 40 else 0
        s = _symbols(rng, it % 6, n, rangev)
        w, st = ol.orc_encode_entropy(s, rangev, pb)
        syms.append(s)
        ranges.append(rangev)
        pbs.append(pb)
        want.append((w, st))
    # prob_bits 1..7 (the C-ABI takes 1..19), ranges up to 2^prob_bits; drawn after the streams above so that
    # those stay as they were
    low = np.random.default_rng(12)
    first_low = len(syms)
    for pb in range(1, 8):
        for rangev in sorted({1, 2, (1 << pb) // 2 + 1, 1 << pb}):
            for kind in range(6):
                s = _symbols(low, kind, int(low.choice([1, 7, 64, 1000, 20000])), rangev)
                syms.append(s)
                ranges.append(rangev)
                pbs.append(pb)
                want.append(ol.orc_encode_entropy(s, rangev, pb))
    got = g.encode_entropy_batch(syms, ranges, pbs)
    n_ok = n_stored = n_low_coded = 0
    for i, ((gb, gst, stored), (wb, wst)) in enumerate(zip(got, want)):
        if wst != 0:
            assert gst == wst, (i, ranges[i], pbs[i], len(syms[i]))
            continue
        assert gst == 0 and gb.tobytes() == wb.tobytes(), (i, ranges[i], pbs[i], len(syms[i]))
        n_ok += 1
        n_stored += stored
        n_low_coded += i >= first_low and not stored
    assert n_ok > 500 and n_stored > 10
    assert n_low_coded > 40


def test_encode_entropy_prefix_and_slab_layout():
    g = gpu_lib.gpu()
    rng = np.random.default_rng(2)
    syms = [_symbols(rng, 1, 3000, 256), _symbols(rng, 1, 10, 512), np.zeros(0, np.uint16)]
    got = g.encode_entropy_batch(syms, [256, 512, 256], [15, 15, 15], prefixes=[b"\x10\x00\x00\x00\x10", b"", b"\xaa"])
    for (gb, st, _), s, r, p in zip(got, syms, [256, 512, 256], [b"\x10\x00\x00\x00\x10", b"", b"\xaa"]):
        w, _ = ol.orc_encode_entropy(s, r, 15)
        assert st == 0 and gb.tobytes() == p + w.tobytes()


def test_decode_entropy_vs_oracle_and_roundtrip():
    """entropy_decoding.hpp:134 — fixed semantics (flags 7) at prob_bits 1..19 and reference semantics (flags 0)."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(3)
    blobs, offs, caps, exp = [], [], [], []
    pos = lossless = 0
    for it in range(400):
        rangev = int(rng.choice([2, 3, 14, 256, 257, 512]))
        pb = int(rng.integers(9, 20))
        n = int(rng.choice([1, 5, 49, 64, 65, 1000, 20000, 66000]))
        s = _symbols(rng, it % 6, n, rangev)
        if len(np.unique(s)) < 2:
            s[0] = (int(s[0]) + 1) % rangev  # a lone symbol owning 2^pb is unrepresentable (see oracle tests)
        enc, st = ol.orc_encode_entropy(s, rangev, pb)
        if st != 0:
            continue
        lead = int(rng.integers(0, 7))  # arbitrary byte alignment of the stream (SURVEY H3)
        # expected = what the oracle's decoder reads: table mode 1 is lossy when a frequency needs
        # more than maxbits bits (SURVEY D6), and then the decoded symbols are not the input
        want, _, wst = ol.orc_decode_entropy(enc, 0, flags=7, cap=n)
        assert wst == 0
        ok = np.array_equal(want, s)
        lossless += int(ok)
        if not ok:
            want = None  # garbage table: the state collapses and the decoder runs off the payload, so what
                         # it reads (oracle and reference alike) is whatever follows in memory
        blobs.append(np.zeros(lead, np.uint8))
        blobs.append(enc)
        offs.append(pos + lead)
        caps.append(n)
        exp.append((want, pos + lead + len(enc)))
        pos += lead + len(enc)
    assert lossless > 250
    # prob_bits 1..7 (k_rans_decode's direct lookup, lut_shift 0), ranges 2..2^prob_bits; drawn after the streams
    # above so that those stay as they were
    low = np.random.default_rng(4)
    first_low = len(exp)
    for pb in range(1, 8):
        for rangev in sorted({2, (1 << pb) // 2 + 1, 1 << pb}):
            for kind in range(6):
                n = int(low.choice([2, 7, 64, 1000, 20000, 66000]))
                s = _symbols(low, kind, n, rangev)
                if len(np.unique(s)) < 2:
                    s[0] = (int(s[0]) + 1) % rangev
                enc, st = ol.orc_encode_entropy(s, rangev, pb)
                assert st == 0
                want, _, wst = ol.orc_decode_entropy(enc, 0, flags=7, cap=n)
                assert wst == 0
                lead = int(low.integers(0, 7))
                blobs += [np.zeros(lead, np.uint8), enc]
                offs.append(pos + lead)
                caps.append(n)
                exp.append((want if np.array_equal(want, s) else None, pos + lead + len(enc)))
                pos += lead + len(enc)
    blob = np.concatenate(blobs)
    got = g.decode_entropy_batch(blob, offs, caps, flags=7)
    low_coded = 0
    for i, ((sym, end, st), (s, e)) in enumerate(zip(got, exp)):
        if s is None:  # garbage table (lossy mode 1): decoded without faulting, or refused as a bad table
            assert st in (0, 3, 6), i  # 6 = HOH_S_BAD_STATE: the final rANS state gives the garbage away
            continue
        assert st == 0 and end == e and np.array_equal(sym, s), i
        r = g.last_dec_results[i]
        low_coded += i >= first_low and not r["stored"] and r["prob_bits"] < 8
    assert low_coded > 30
    # single-call shim, reference semantics: byte_pointer stops at the payload (D8), 4-bit prob_bits (D9)
    checked_ref = 0
    for it in range(40):
        rangev, pb, n = int(rng.choice([14, 256, 512])), int(rng.integers(9, 16)), int(rng.choice([5, 1000, 20000]))
        s = _symbols(rng, 1 + it % 3, n, rangev)
        s[0] = (int(s[0]) + 1) % rangev
        enc, st = ol.orc_encode_entropy(s, rangev, pb)
        if st:
            continue
        a, bpa, sta = ol.orc_decode_entropy(enc, 0, flags=0, cap=n)
        if not np.array_equal(a, s):
            continue  # lossy table (D6): what the decoder reads past the payload is undefined
        b, bpb, stb = g.decode_entropy(enc, 0, flags=0, cap=n)
        assert sta == stb == 0 and bpa == bpb and np.array_equal(a, b)
        checked_ref += 1
    assert checked_ref > 15


def test_final_state_check_flags_damaged_payloads():
    """The decoder's only integrity check (the format has no checksum): a sound stream ends in the state the encoder
    started from, 2^31.  Streams with one payload byte changed report HOH_S_BAD_STATE (6) and still hand out their
    symbols; their intact neighbours decode exactly with status 0."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(61)
    encs, syms = [], []
    for it in range(96):
        n = int(rng.choice([700, 5000, 65536]))
        s = _symbols(rng, 1 + it % 3, n, 256)
        s[0] = (int(s[0]) + 1) % 256
        enc, st = ol.orc_encode_entropy(s, 256, 15)
        assert st == 0
        encs.append(np.array(enc, np.uint8))
        syms.append(s)
    offs, pos = [], 0
    for e in encs:
        offs.append(pos)
        pos += len(e)
    caps = [len(s) for s in syms]
    clean = g.decode_entropy_batch(np.concatenate(encs), offs, caps, flags=7)
    decodable = [st == 0 and np.array_equal(sym, s) for (sym, _, st), s in zip(clean, syms)]
    assert sum(decodable) > 80  # the rest: lossy mode-1 tables (SURVEY D6)
    coded = [int(r["stored"]) == 0 for r in g.last_dec_results]  # stored-mode streams have no state to check
    damaged = [e.copy() for e in encs]
    # (a near-constant stream is a table and a bare final state: only streams with a real payload are damaged)
    hit = [i for i in range(len(encs)) if i % 2 and decodable[i] and coded[i] and len(encs[i]) > 400]
    assert len(hit) > 20
    for i in hit:
        at = int(rng.integers(len(encs[i]) * 2 // 3, len(encs[i]) - 8))  # well inside the payload
        damaged[i][at] ^= int(rng.integers(1, 256))
    got = g.decode_entropy_batch(np.concatenate(damaged), offs, caps, flags=7)
    for i, ((sym, _, st), s) in enumerate(zip(got, syms)):
        if i in hit:
            assert st == 6 and len(sym) == len(s), (i, st)
        elif decodable[i]:
            assert st == 0 and np.array_equal(sym, s), i


def test_decode_entropy_golden_and_empty():
    g = gpu_lib.gpu()
    z = np.load(os.path.join(G, "entropy.npz"))
    for name in _cases(z, "__sym"):
        sym, want = z[name + "__sym"], z[name + "__out"]
        if len(np.unique(sym)) > 1:
            dec, bp, st = g.decode_entropy(want, 0, flags=7, cap=max(len(sym), 1))
            assert st == 0 and np.array_equal(dec, sym) and bp == len(want), name
    dec, bp, st = g.decode_entropy(z["empty__out"], 0, flags=7, cap=8)
    assert len(dec) == 0 and bp == len(z["empty__out"]) and st == 0


def test_normalize_freqs_vs_oracle():
    """stattools.hpp:13 incl. the steal loop and both assert conditions."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(4)
    for it in range(120):
        size = int(rng.choice([1, 2, 5, 14, 256, 512]))
        pb = int(rng.integers(8, 20))
        f = np.zeros(size, np.uint32)
        k = int(rng.integers(1, size + 1))
        idx = rng.choice(size, k, replace=False)
        f[idx] = (rng.pareto(0.7, k) * 3 + 1).astype(np.uint32)
        of, oc = f.copy(), np.zeros(size + 1, np.uint32)
        ost = ol.oracle().orc_normalize_freqs(of, oc, size, 1 << pb)
        gf, gc, gst = g.normalize_freqs(f, 1 << pb)
        assert gst == ost, (it, size, pb)
        if ost == 0:
            assert np.array_equal(gf, of) and np.array_equal(gc, oc), (it, size, pb)


def test_normalize_freqs_many_thieves():
    """Small prob_bits against a wide, almost fully used alphabet: dozens to hundreds of symbols round to zero
    and steal (the binary-search form of the steal loop).  (Running out of donors cannot happen once
    target >= size: the scaled counts sum to the target, so the spare counts always cover the thieves.)"""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(44)
    seen_many = 0
    for it in range(150):
        size = int(rng.choice([256, 512]))
        pb = int(rng.integers(8, 15))
        if (1 << pb) < size:
            pb = 9 if size == 512 else 8
        k = int(rng.integers(size // 2, size + 1))
        f = np.zeros(size, np.uint32)
        idx = rng.choice(size, k, replace=False)
        shape = [rng.geometric(0.02, k), (rng.pareto(1.2, k) * 5 + 1), rng.integers(1, 4, k),
                 np.where(rng.random(k) < 0.1, 5000, 1)][it % 4]
        f[idx] = np.maximum(1, np.asarray(shape)).astype(np.uint32)
        of, oc = f.copy(), np.zeros(size + 1, np.uint32)
        ost = ol.oracle().orc_normalize_freqs(of, oc, size, 1 << pb)
        gf, gc, gst = g.normalize_freqs(f, 1 << pb)
        assert gst == ost, (it, size, pb, gst, ost)
        if ost == 0:
            assert np.array_equal(gf, of) and np.array_equal(gc, oc), (it, size, pb)
            scaled = np.diff((np.concatenate([[0], np.cumsum(f, dtype=np.uint64)]) * (1 << pb)) // int(f.sum()))
            seen_many += int(np.count_nonzero((f > 0) & (scaled == 0)) > 16)
    assert seen_many > 20


def test_rans_static_table_sweep_sample():
    """Config 4 shape: 8-bit alphabet, one static prob_bits-12 table, 65 536-symbol streams."""
    mod = gpu_lib.hohgpu()
    g = gpu_lib.gpu()
    n, stream_len, pb = (1 << 20) + 12345, 65536, 12
    sym8 = ol.synth_symbols(n, 7)
    f = np.bincount(sym8, minlength=256).astype(np.uint32)
    cum = np.zeros(257, np.uint32)
    assert ol.oracle().orc_normalize_freqs(f, cum, 256, 1 << pb) == 0
    sym = sym8.astype(np.uint16)
    n_streams = (n + stream_len - 1) // stream_len
    slab = (stream_len * pb // 8 + 64 + 15) & ~15
    d_sym = g.alloc(sym.nbytes + 64).upload(sym)
    d_cum = g.alloc(cum.nbytes).upload(cum)
    d_out = g.alloc(n_streams * slab)
    d_len = g.alloc(n_streams * 4)
    d_dec = g.alloc(sym.nbytes + 64)
    g._ck(g.lib.hoh_rans_encode_static(g.ctx, d_sym.ptr, n, stream_len, d_cum.ptr, 256, pb, d_out.ptr, slab,
                                       d_len.ptr), "enc")
    g._ck(g.lib.hoh_rans_decode_static(g.ctx, d_out.ptr, slab, d_len.ptr, n, stream_len, d_cum.ptr, 256, pb,
                                       d_dec.ptr), "dec")
    lens = d_len.download(np.uint32, n_streams)
    blob = d_out.download(np.uint8, n_streams * slab)
    dec = d_dec.download(np.uint16, n)
    assert np.array_equal(dec, sym)
    for i in [0, 1, n_streams // 2, n_streams - 1]:
        part = sym[i * stream_len:(i + 1) * stream_len]
        want = np.zeros(len(part) * 2 + 64, np.uint8)
        wl = ol.oracle().orc_rans_encode_static(part, len(part), f, cum, 256, pb, want)
        assert lens[i] == wl
        assert blob[(i + 1) * slab - wl:(i + 1) * slab].tobytes() == want[:wl].tobytes(), i
    for b in (d_sym, d_cum, d_out, d_len, d_dec):
        b.free()
    assert mod.MAX_RANGE == 512


# ---------------------------------------------------------------------------------------------
# colour transform and prediction
# ---------------------------------------------------------------------------------------------
def test_subtract_green_and_inverse():
    g = gpu_lib.gpu()
    rgb = np.random.default_rng(0).integers(0, 256, 3 * 5000, dtype=np.uint8)
    a = [np.zeros(5000, np.uint16) for _ in range(3)]
    ol.oracle().orc_subtract_green(rgb, rgb.size, *a)
    b = g.subtract_green(rgb)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(g.add_green(*b), rgb)


def test_predict_golden_vectors():
    """prediction.hpp:6/:46/:153, unprediction.hpp:6 on the reference-generated fixtures."""
    g = gpu_lib.gpu()
    z = np.load(os.path.join(G, "predict.npz"))
    for name in _cases(z, "__plane"):
        w, h, depth, xt, yt = (int(v) for v in z[name + "__par"])
        plane, tm = z[name + "__plane"], z[name + "__map"]
        assert np.array_equal(g.channelpredict_fastpath(plane, w, h, depth), z[name + "__fast"]), name
        allr = g.channelpredict_all(plane, w, h, depth, xt, yt, tm)
        assert np.array_equal(allr, z[name + "__all"]), name
        assert np.array_equal(g.unpredict_all(allr, w, h, depth, xt, yt, tm), plane), name
        assert np.array_equal(g.unpredict_fastpath(z[name + "__fast"], w, h, depth), plane), name
        sec, secn = z[name + "__sec"], z[name + "__secn"]
        off = 0
        for t in range(xt * yt):
            r = g.channelpredict_section(plane, w, h, depth, xt, yt, t % xt, t // xt, int(tm[t]))
            assert len(r) == secn[t] and np.array_equal(r, sec[off:off + len(r)]), (name, t)
            off += len(r)
            if xt * yt > 6 and t > 8:
                break


def test_predict_random_vs_oracle():
    g = gpu_lib.gpu()
    O = ol.oracle()
    rng = np.random.default_rng(8)
    for it in range(30):
        w, h = int(rng.integers(1, 130)), int(rng.integers(1, 90))
        depth = int(rng.choice([8, 9]))
        xt, yt = (w + 39) // 40, (h + 39) // 40
        plane = _smooth_plane(rng, w, h, depth) if it % 3 else rng.integers(0, 1 << depth, w * h).astype(np.uint16)
        tm = rng.choice(STOCK, xt * yt).astype(np.uint16)
        a = np.zeros(w * h, np.uint16)
        O.orc_predict_fastpath(plane, w, h, depth, a)
        assert np.array_equal(g.channelpredict_fastpath(plane, w, h, depth), a), (it, w, h)
        assert np.array_equal(g.unpredict_fastpath(a, w, h, depth), plane), (it, w, h)
        O.orc_predict_all(plane, w, h, depth, xt, yt, tm, a)
        assert np.array_equal(g.channelpredict_all(plane, w, h, depth, xt, yt, tm), a), (it, w, h)
        assert np.array_equal(g.unpredict_all(a, w, h, depth, xt, yt, tm), plane), (it, w, h)
        t = int(rng.integers(0, xt * yt))
        buf = np.zeros(w * h + 8, np.uint16)
        n = O.orc_predict_section(plane, w, h, depth, xt, yt, t % xt, t // xt, int(tm[t]), buf)
        r = g.channelpredict_section(plane, w, h, depth, xt, yt, t % xt, t // xt, int(tm[t]))
        assert len(r) == n and np.array_equal(r, buf[:n]), (it, w, h, t)
    # back-references (unprediction.hpp:63-65)
    w, h, depth = 64, 40, 8
    plane = _smooth_plane(rng, w, h, depth)
    br = np.zeros(w * h, np.uint16)
    for at in rng.choice(np.arange(w + 2, w * h), 200, replace=False):
        br[at] = int(rng.integers(1, min(at, 300)))
    tm = rng.choice(STOCK, 2).astype(np.uint16)
    resid = np.zeros(w * h, np.uint16)
    O.orc_predict_all(plane, w, h, depth, 2, 1, tm, resid)
    dense = np.concatenate([resid[br == 0], np.zeros(8, np.uint16)])
    want = np.zeros(w * h, np.uint16)
    O.orc_unpredict_all(dense, w, h, depth, 2, 1, tm, br.ctypes.data, want)
    assert np.array_equal(g.unpredict_all(dense, w, h, depth, 2, 1, tm, backref=br), want)
    O.orc_predict_fastpath(plane, w, h, depth, resid)
    dense = np.concatenate([resid[br == 0], np.zeros(8, np.uint16)])
    O.orc_unpredict_fastpath(dense, w, h, depth, br.ctypes.data, want)
    assert np.array_equal(g.unpredict_fastpath(dense, w, h, depth, backref=br), want)


def test_predictor_search_vs_oracle():
    """layer_encode.hpp:126-272 — double-precision raster-order cost sums, strict-< argmin."""
    g = gpu_lib.gpu()
    O = ol.oracle()
    rng = np.random.default_rng(9)
    for it, (w, h, depth, mode) in enumerate([(96, 80, 8, 1), (96, 80, 9, 2), (130, 50, 8, 3), (256, 256, 8, 2),
                                              (256, 256, 9, 4), (41, 41, 8, 4)]):
        plane = _smooth_plane(rng, w, h, depth)
        cells = ((w + 39) // 40) * ((h + 39) // 40)
        tm, idx, res = np.zeros(cells, np.uint16), np.zeros(cells, np.uint8), np.zeros(w * h, np.uint16)
        O.orc_predictor_search(plane, w * h, w, h, depth, mode, tm, idx, res.ctypes.data)
        gtm, gidx, gres = g.predictor_search(plane, w, h, depth, mode)
        assert np.array_equal(gtm, tm) and np.array_equal(gidx, idx), (it, w, h, depth, mode)
        assert np.array_equal(gres, res), (it, w, h, depth, mode)


# ---------------------------------------------------------------------------------------------
# tile codec, mode 0
# ---------------------------------------------------------------------------------------------
def _oracle_channels(rgb_tile, w, h):
    px = w * h
    planes = [np.zeros(px, np.uint16) for _ in range(3)]
    ol.oracle().orc_subtract_green(rgb_tile, rgb_tile.size, *planes)
    return [ol.orc_layer_encode(p, w, h, d, 0)[0] for p, d in zip(planes, (8, 9, 9))]


def _tiles(rgb, W, H, geom):
    img = rgb.reshape(H, W, 3)
    for t in range(geom.tiles_per_image):
        x0, y0 = (t % geom.x_tiles) * geom.tile_w, (t // geom.x_tiles) * geom.tile_h
        sub = img[y0:y0 + geom.tile_h, x0:x0 + geom.tile_w]
        yield np.ascontiguousarray(sub).ravel(), sub.shape[1], sub.shape[0]


@pytest.mark.parametrize("W,H,n_images", [(512, 512, 3), (256, 256, 2), (600, 530, 1), (100, 37, 2), (2, 2, 1),
                                          (1000, 300, 1)])
def test_encode_images_s0_vs_oracle_and_roundtrip(W, H, n_images):
    """choh.cpp:454-506 tiling + channel.hpp:73 + layer_encode.hpp:11 (mode 0): every channel payload
    equals layer_encode's bytes; decode returns the original RGB."""
    g = gpu_lib.gpu()
    rgb = np.concatenate([ol.synth_rgb(W, H, 1 + i) for i in range(n_images)])
    packed, off, res = g.encode_images_s0(rgb, n_images, W, H)
    geom = g.tile_geometry(W, H)
    assert (res["status"] == 0).all()
    s = 0
    for i in range(n_images):
        for tile_rgb, tw, th in _tiles(rgb[i * W * H * 3:(i + 1) * W * H * 3], W, H, geom):
            for want in _oracle_channels(tile_rgb, tw, th):
                got = packed[int(off[s]):int(off[s + 1])]
                assert got.tobytes() == want.tobytes(), (i, s, tw, th)
                s += 1
    back, st = g.decode_images_s0(packed, off, n_images, W, H)
    assert (st == 0).all()
    assert np.array_equal(back, rgb)


def test_encode_images_s0_matches_stock_choh_file():
    """The 512x512 seed-1 file written by stock `choh -s0` (golden, md5 78c14f89...): every channel
    payload inside it is reproduced byte for byte by the GPU path."""
    g = gpu_lib.gpu()
    z = np.load(os.path.join(G, "layer_tile.npz"))
    ref_file = z["file_512x512_s0"].tobytes()
    rgb = ol.synth_rgb(512, 512, 1)
    packed, off, res = g.encode_images_s0(rgb, 1, 512, 512)
    cursor = 0
    for s in range(12):
        chan = packed[int(off[s]):int(off[s + 1])].tobytes()
        at = ref_file.find(chan, cursor)
        assert at >= 0, s
        cursor = at + len(chan)
    assert cursor == len(ref_file)  # the last channel ends the file


def test_decode_images_s0_noisy_and_flat_images():
    g = gpu_lib.gpu()
    rng = np.random.default_rng(5)
    W, H = 512, 256
    imgs = [rng.integers(0, 256, W * H * 3, dtype=np.uint8),          # incompressible: stored-mode streams
            np.full(W * H * 3, 77, np.uint8),                         # flat: single-symbol streams
            np.clip(rng.normal(128, 30, W * H * 3), 0, 255).astype(np.uint8)]
    rgb = np.concatenate(imgs)
    packed, off, res = g.encode_images_s0(rgb, 3, W, H)
    assert res["stored"][:6].any()
    geom = g.tile_geometry(W, H)
    s = 0
    for i in range(3):
        for tile_rgb, tw, th in _tiles(imgs[i], W, H, geom):
            for want in _oracle_channels(tile_rgb, tw, th):
                assert packed[int(off[s]):int(off[s + 1])].tobytes() == want.tobytes(), (i, s)
                s += 1
    back, st = g.decode_images_s0(packed, off, 3, W, H)
    # a flat plane's lone symbol owns 2^15 and cannot be represented by the table format (the
    # reference's own decoder fails on it too), so image 1 is only checked on the encode side
    assert np.array_equal(back[:W * H * 3], imgs[0])
    assert np.array_equal(back[2 * W * H * 3:], imgs[2])


def test_host_buffer_pipeline_matches_device_path():
    """hoh_encode_images_s0_host / hoh_decode_images_s0_host (chunked H2D / kernels / D2H pipeline, 3 chunks
    here) return exactly what the one-shot device-resident calls return."""
    import ctypes as C
    g = gpu_lib.gpu()
    mod = gpu_lib.hohgpu()
    W = H = 512
    n = 200  # 157 MB of pixels: above the pipeline's 64 MB minimum chunk, so several chunks
    rgb = g.host_alloc(n * W * H * 3)
    for i in range(n):
        rgb[i * W * H * 3:(i + 1) * W * H * 3] = ol.synth_rgb(W, H, 1 + (i % 7))
    geom = g.tile_geometry(W, H)
    ns = n * geom.streams_per_image
    cap = rgb.size * 2
    packed = g.host_alloc(cap)
    off = g.host_alloc((ns + 1) * 8, np.uint64)
    res = np.zeros(ns, mod.RESULT_DT)
    g._ck(g.lib.hoh_encode_images_s0_host(g.ctx, rgb.ctypes.data, n, W, H, packed.ctypes.data, cap, off.ctypes.data,
                                          res.ctypes.data), "encode_host")
    assert (res["status"] == 0).all()
    ref_packed, ref_off, _ = g.encode_images_s0(rgb[:7 * W * H * 3], 7, W, H)
    per_img = geom.streams_per_image
    assert np.array_equal(np.diff(off.astype(np.int64))[:7 * per_img], np.diff(ref_off.astype(np.int64)))
    assert packed[:int(ref_off[-1])].tobytes() == ref_packed.tobytes()
    # images repeat with period 7, so every image's payload sizes must repeat too
    sizes = np.diff(off.astype(np.int64)).reshape(n, per_img)
    assert all(np.array_equal(sizes[i], sizes[i % 7]) for i in range(n))
    back = g.host_alloc(rgb.size)
    st = np.zeros(ns, np.int32)
    g._ck(g.lib.hoh_decode_images_s0_host(g.ctx, packed.ctypes.data, int(off[ns]), off.ctypes.data, n, W, H,
                                          back.ctypes.data, st.ctypes.data), "decode_host")
    assert (st == 0).all()
    assert np.array_equal(back, rgb)


def test_host_buffer_pipeline_ramped_chunks(monkeypatch):
    """The pipelined host calls cut a large batch into short chunks at both ends and steady ones between them
    (chunk_plan in hoh_api.cu).  HOH_PIPE_CHUNK_KB lowers the chunk floor so that a small batch takes that path: 64 images
    of 128x128 become chunks of 4, 8 x 7, 4 images over 4 buffers, and must give the one-shot device path's bytes."""
    monkeypatch.setenv("HOH_PIPE_CHUNK_KB", "200")
    g = gpu_lib.gpu()
    mod = gpu_lib.hohgpu()
    W = H = 128
    n = 64
    rgb = g.host_alloc(n * W * H * 3)
    for i in range(n):
        rgb[i * W * H * 3:(i + 1) * W * H * 3] = ol.synth_rgb(W, H, 11 + i)
    geom = g.tile_geometry(W, H)
    ns = n * geom.streams_per_image
    cap = rgb.size * 2 + 4096 * ns
    packed = g.host_alloc(cap)
    off = g.host_alloc((ns + 1) * 8, np.uint64)
    res = np.zeros(ns, mod.RESULT_DT)
    g._ck(g.lib.hoh_encode_images_s0_host(g.ctx, rgb.ctypes.data, n, W, H, packed.ctypes.data, cap, off.ctypes.data,
                                          res.ctypes.data), "encode_host")
    assert (res["status"] == 0).all()
    ref_packed, ref_off, _ = g.encode_images_s0(np.asarray(rgb), n, W, H)
    assert np.array_equal(off, ref_off)
    assert packed[:int(ref_off[-1])].tobytes() == ref_packed.tobytes()
    back = g.host_alloc(rgb.size)
    st = np.zeros(ns, np.int32)
    g._ck(g.lib.hoh_decode_images_s0_host(g.ctx, packed.ctypes.data, int(off[ns]), off.ctypes.data, n, W, H,
                                          back.ctypes.data, st.ctypes.data), "decode_host")
    assert (st == 0).all()
    assert np.array_equal(back, rgb)


def test_predictor_search_batched_planes_vs_oracle():
    """hoh_predictor_search_dev over several planes at once (the BASELINE config 3 / 5 shape: every
    channel of every tile is one plane) equals the per-plane oracle."""
    g = gpu_lib.gpu()
    O = ol.oracle()
    rng = np.random.default_rng(31)
    w, h, depth, mode, n_planes = 128, 96, 9, 2, 6
    planes = np.concatenate([_smooth_plane(rng, w, h, depth) for _ in range(n_planes)])
    cells = ((w + 39) // 40) * ((h + 39) // 40)
    d_pl = g.alloc(planes.nbytes).upload(planes)
    d_map, d_idx, d_res = g.alloc(n_planes * cells * 2), g.alloc(n_planes * cells), g.alloc(planes.nbytes)
    g._ck(g.lib.hoh_predictor_search_dev(g.ctx, d_pl.ptr, n_planes, w, h, depth, mode, d_map.ptr, d_idx.ptr,
                                         d_res.ptr), "search_dev")
    maps = d_map.download(np.uint16, n_planes * cells).reshape(n_planes, cells)
    idxs = d_idx.download(np.uint8, n_planes * cells).reshape(n_planes, cells)
    res = d_res.download(np.uint16, planes.size).reshape(n_planes, w * h)
    for p in range(n_planes):
        tm, idx, r = np.zeros(cells, np.uint16), np.zeros(cells, np.uint8), np.zeros(w * h, np.uint16)
        O.orc_predictor_search(np.ascontiguousarray(planes[p * w * h:(p + 1) * w * h]), w * h, w, h, depth, mode,
                               tm, idx, r.ctypes.data)
        assert np.array_equal(maps[p], tm) and np.array_equal(idxs[p], idx) and np.array_equal(res[p], r), p
    # and the batched inverse: unpredict_all over all planes returns the planes
    d_back = g.alloc(planes.nbytes)
    g._ck(g.lib.hoh_unpredict_all_dev(g.ctx, d_res.ptr, n_planes, w, h, depth, (w + 39) // 40, (h + 39) // 40,
                                      d_map.ptr, None, d_back.ptr), "unpredict_all_dev")
    assert np.array_equal(d_back.download(np.uint16, planes.size), planes)
    for b in (d_pl, d_map, d_idx, d_res, d_back):
        b.free()


def test_round_trip_4k_images_and_larger_batch():
    """Size-independent property at BASELINE shapes: 3840x2160 (15x8 tiles of 256x270, choh.cpp:455-460) and
    a 256-image batch of 512x512 round-trip exactly; payload sizes of identical images are identical."""
    g = gpu_lib.gpu()
    W, H = 3840, 2160
    rgb = np.concatenate([ol.synth_rgb(W, H, 1), ol.synth_rgb(W, H, 2)])
    packed, off, res = g.encode_images_s0(rgb, 2, W, H)
    assert (res["status"] == 0).all() and len(off) == 2 * 360 + 1
    assert hashlib.md5(rgb[:W * H * 3].tobytes()).hexdigest() == "2517cea8921e09ee393f541b4a3a4f51"  # SURVEY 8(c)
    back, st = g.decode_images_s0(packed, off, 2, W, H)
    assert (st == 0).all() and np.array_equal(back, rgb)
    # one tile against the oracle
    tile = np.ascontiguousarray(rgb[:W * H * 3].reshape(H, W, 3)[270:540, 256:512]).ravel()
    s = (1 * 15 + 1) * 3
    for k, want in enumerate(_oracle_channels(tile, 256, 270)):
        assert packed[int(off[s + k]):int(off[s + k + 1])].tobytes() == want.tobytes()
    n = 256
    base = [ol.synth_rgb(512, 512, 1 + i) for i in range(4)]
    rgb = np.concatenate([base[i % 4] for i in range(n)])
    packed, off, res = g.encode_images_s0(rgb, n, 512, 512)
    sizes = np.diff(off.astype(np.int64)).reshape(n, 12)
    assert all(np.array_equal(sizes[i], sizes[i % 4]) for i in range(n))
    back, st = g.decode_images_s0(packed, off, n, 512, 512)
    assert (st == 0).all() and np.array_equal(back, rgb)


def test_rans_static_sweep_64mb_round_trip():
    """Config 4 at a larger size: 64 Mi geometric symbols in 65 536-symbol streams, one static table;
    decode(encode(x)) == x and the payload total matches the entropy within 1 %."""
    g = gpu_lib.gpu()
    n, stream_len, pb = 1 << 26, 65536, 12
    sym8 = np.tile(ol.synth_symbols(1 << 22, 11), 16)
    f = np.bincount(sym8[:1 << 22], minlength=256).astype(np.uint32)
    cum = np.zeros(257, np.uint32)
    assert ol.oracle().orc_normalize_freqs(f, cum, 256, 1 << pb) == 0
    sym = sym8.astype(np.uint16)
    n_streams = n // stream_len
    slab = (stream_len * pb // 8 + 64 + 15) & ~15
    d_sym, d_cum = g.alloc(sym.nbytes).upload(sym), g.alloc(cum.nbytes).upload(cum)
    d_out, d_len, d_dec = g.alloc(n_streams * slab), g.alloc(n_streams * 4), g.alloc(sym.nbytes)
    g._ck(g.lib.hoh_rans_encode_static(g.ctx, d_sym.ptr, n, stream_len, d_cum.ptr, 256, pb, d_out.ptr, slab,
                                       d_len.ptr), "enc")
    g._ck(g.lib.hoh_rans_decode_static(g.ctx, d_out.ptr, slab, d_len.ptr, n, stream_len, d_cum.ptr, 256, pb,
                                       d_dec.ptr), "dec")
    assert np.array_equal(d_dec.download(np.uint16, n), sym)
    lens = d_len.download(np.uint32, n_streams)
    p = f[f > 0] / float(1 << pb)
    counts = np.bincount(sym8[:1 << 22], minlength=256)[f > 0]
    ideal_bits = float(-(counts * np.log2(p)).sum()) * 16
    assert abs(lens.sum() * 8.0 / ideal_bits - 1.0) < 0.01
    for b in (d_sym, d_cum, d_out, d_len, d_dec):
        b.free()


@pytest.mark.parametrize("total,target,n_px", [(3, 0, 1000), (3, 1, 65536), (3, 2, 70001), (4, 3, 513), (1, 0, 77), (2, 1, 4096)])
def test_channel_picker_direct(total, target, n_px):
    """channel.hpp:63-71 on the device, compared with the oracle and with plain slicing."""
    g = gpu_lib.gpu()
    rng = np.random.default_rng(100 * total + target)
    src = rng.integers(0, 256, n_px * total, dtype=np.uint8)
    got = g.channel_picker(src, total, target)
    assert got.dtype == np.uint16 and np.array_equal(got, src[target::total].astype(np.uint16))
    assert np.array_equal(got, ol.orc_channel_picker(src, total, target))


def _backref_maps(rgb, n_images, w, h, geo, nukes):
    """LEMPEL_BACKREF maps for decode: a covered pixel copies the nearest earlier pixel of its tile with the same
    colour (any in-tile distance that reproduces the pixel is a valid back-reference for the decoder)."""
    stride = (geo.tile_w * geo.tile_h + 7) & ~7
    maps = np.zeros(n_images * geo.tiles_per_image * stride, np.uint16)
    for i in range(n_images):
        img = rgb[i * w * h * 3:(i + 1) * w * h * 3].reshape(h, w, 3)
        for t in range(geo.tiles_per_image):
            x0, y0 = (t % geo.x_tiles) * geo.tile_w, (t // geo.x_tiles) * geo.tile_h
            tile = img[y0:y0 + geo.tile_h, x0:x0 + geo.tile_w].reshape(-1, 3).astype(np.uint32)
            key = (tile[:, 0] << 16) | (tile[:, 1] << 8) | tile[:, 2]
            k = i * geo.tiles_per_image + t
            nuke = nukes[k * stride:k * stride + key.size]
            last = {}
            for p in range(key.size):
                if nuke[p]:
                    assert int(key[p]) in last, "a covered pixel must have an earlier equal pixel"
                    maps[k * stride + p] = p - last[int(key[p])]
                last[int(key[p])] = p
    return maps


@pytest.mark.parametrize("w,h,n", [(96, 80, 3), (512, 256, 2), (601, 523, 1)])
def test_decode_images_s0_with_backrefs(w, h, n):
    """hoh_decode_images_s0 with LEMPEL_BACKREF maps (unprediction.hpp:63-65): streams coded with the NUKE maps of
    the LZ finder hold residuals only for uncovered pixels; the decoder copies the covered ones."""
    g = gpu_lib.gpu()
    mod = gpu_lib.hohgpu()
    rng = np.random.default_rng(w + h)
    rgb = np.concatenate([ol.photo_with_repeats(rng, w, h, 40 + i).ravel() for i in range(n)])
    geo = g.tile_geometry(w, h)
    n_tiles = n * geo.tiles_per_image
    n_streams = n_tiles * 3
    stride = (geo.tile_w * geo.tile_h + 7) & ~7
    lz_stride = int(g.lib.hoh_find_lz_stride(geo.tile_w, geo.tile_h))
    out_bytes = int(g.lib.hoh_encode_images_out_bytes(C.byref(geo), n))
    cap = rgb.nbytes * 2 + 4096 * n_streams
    bufs = [g.alloc(rgb.nbytes).upload(rgb), g.alloc(n_tiles * stride), g.alloc(n_tiles * lz_stride), g.alloc(n_tiles * 4),
            g.alloc(n_tiles * 4), g.alloc(out_bytes), g.alloc(n_streams * mod.RESULT_DT.itemsize), g.alloc(cap),
            g.alloc((n_streams + 1) * 8)]
    d_rgb, d_nuke, d_lz, d_size, d_st, d_out, d_res, d_packed, d_off = bufs
    try:
        d_nuke.zero()
        g._ck(g.lib.hoh_find_lz_images(g.ctx, d_rgb.ptr, n, w, h, 6, 0, None, d_nuke.ptr, d_lz.ptr, lz_stride, d_size.ptr,
                                       d_st.ptr), "lz")
        g._ck(g.lib.hoh_encode_images_s0(g.ctx, d_rgb.ptr, n, w, h, d_nuke.ptr, d_out.ptr, out_bytes, d_res.ptr,
                                         d_packed.ptr, cap, d_off.ptr), "encode")
        nukes = d_nuke.download(np.uint8, n_tiles * stride)
        off = d_off.download(np.uint64, n_streams + 1)
        packed = d_packed.download(np.uint8, int(off[-1]))
    finally:
        for b in bufs:
            b.free()
    assert nukes.sum() > 50
    maps = _backref_maps(rgb, n, w, h, geo, nukes)
    back, st = g.decode_images_s0(packed, off, n, w, h, backref=maps)
    assert (st == 0).all() and np.array_equal(back, rgb)
    # without the maps the dense streams cannot fill the tiles: every tile with a match is reported, not mis-decoded
    back2, st2 = g.decode_images_s0(packed, off, n, w, h)
    assert (st2 != 0).any()
    # a map that disagrees with the stream (one more covered pixel) is caught as well
    wrong = maps.copy()
    first_free = int(np.flatnonzero(wrong[:geo.tile_w * geo.tile_h] == 0)[5])
    wrong[first_free] = 1
    back3, st3 = g.decode_images_s0(packed, off, n, w, h, backref=wrong)
    assert st3[0] == 5 and st3[1] == 5 and st3[2] == 5


def test_fused_tile_decoder_reports_damage_and_leaves_the_tile_alone():
    """k_rans_decode_tiles_s0 (entropy decode + un-prediction + colour inverse + scatter in one kernel): a changed
    payload byte shows up as HOH_S_BAD_STATE on its stream, a broken channel header as HOH_S_BAD_LAYER and its tile is
    not written; every other tile of the batch still decodes exactly."""
    g = gpu_lib.gpu()
    W, H, n = 512, 512, 3
    rgb = np.concatenate([ol.synth_rgb(W, H, 20 + i) for i in range(n)])
    packed, off, res = g.encode_images_s0(rgb, n, W, H)
    geom = g.tile_geometry(W, H)
    bad = packed.copy()
    s_state, s_layer = 7, 22                       # stream 7 = tile 2 of image 0, stream 22 = tile 3 of image 1
    bad[int(off[s_state]) + 900] ^= 0x10           # inside the rANS payload
    bad[int(off[s_layer])] = 0x11                  # channel header byte (layer_encode.hpp:57)
    back, st = g.decode_images_s0(bad, off, n, W, H)
    assert st[s_state] == 6 and st[s_layer] == 5
    assert np.count_nonzero(st) == 2
    img = back.reshape(n, H, W, 3)
    want = rgb.reshape(n, H, W, 3)
    for i in range(n):
        for t in range(geom.tiles_per_image):
            x0, y0 = (t % geom.x_tiles) * geom.tile_w, (t // geom.x_tiles) * geom.tile_h
            got_t = img[i, y0:y0 + geom.tile_h, x0:x0 + geom.tile_w]
            k = i * geom.tiles_per_image + t
            if k == s_layer // 3:
                assert not got_t.any()             # the wrapper zeroes the output: the tile was never written
            elif k != s_state // 3:                # (a BAD_STATE tile is written: its symbols are still delivered)
                assert np.array_equal(got_t, want[i, y0:y0 + geom.tile_h, x0:x0 + geom.tile_w]), (i, t)
