// dhoh_batch — host-side .hoh container reader on top of libhohgpu.so.
//
// The reader half of the batched drop-in: the host parses the container (magic, pixel format, depth, size varints,
// tile grid, tile-size varints — dhoh.cpp:297-396 and :22-46, varint.hpp:6-27) and hands the tile byte ranges of ALL
// files to one C-ABI call, hoh_decode_images_host, which does everything inside the tiles on the GPU (tile header,
// LZ side streams, channel layout, layer headers, rANS, un-prediction with LZ copies, colour inverse, tile scatter —
// dhoh.cpp:87-290, un_lz.hpp, layer_decode.hpp as they have to work: the reference's own dhoh cannot parse what
// choh writes, SURVEY D2/D3/D4/D8/D9/D10/D12).
//
//   dhoh_batch infile.hoh outfile.rgb                    the reference tool's command line (dhoh.cpp:306-318)
//   dhoh_batch --batch outdir in1.hoh [in2.hoh ...]      many files in one GPU call per image size -> outdir/<name>.rgb
//   options: --device N
//            --crop X Y W H   write only the W x H window at (X, Y) of every file (W * H * 3 bytes of RGB); only the
//                             tiles the window touches are read and decoded (hoh_decode_regions_host).  A window that
//                             does not lie inside an image is a CLI error (exit 1).
// Exit codes follow dhoh.cpp:283-295: 0 ok, 1 CLI, 2 I/O, 3 unexpected end of file / no GPU, 4 incorrect bitstream,
// 5 not implemented.
#include <cerrno>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "hohgpu.h"

namespace {

struct Parsed {
    std::string in, out;
    std::vector<uint8_t> bytes;
    uint32_t width = 0, height = 0;
    std::vector<uint64_t> tile_begin;  // offsets into bytes, n_tiles + 1 entries
};

bool read_file(const std::string& path, std::vector<uint8_t>& out) {
    FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) {
        std::fprintf(stderr, "dhoh_batch: cannot open %s: %s\n", path.c_str(), std::strerror(errno));
        return false;
    }
    std::fseek(f, 0, SEEK_END);
    const long sz = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    out.resize(sz > 0 ? (size_t)sz : 0);
    const bool ok = out.empty() || std::fread(out.data(), 1, out.size(), f) == out.size();
    std::fclose(f);
    return ok;
}

// varint.hpp:6-27: up to three 7-bit groups, continuation bit on all but the last
bool get_varint(const std::vector<uint8_t>& b, size_t& at, size_t& value) {
    value = 0;
    for (int k = 0; k < 3; k++) {
        if (at >= b.size()) return false;
        const uint8_t byte = b[at++];
        if (k == 2) {
            value = (value << 7) + byte;  // the third byte is taken whole (varint.hpp:16)
            return true;
        }
        value = (value << 7) + (byte & 0x7f);
        if (!(byte & 0x80)) return true;
    }
    return true;
}

// 0 ok, else dhoh's exit code
int parse_container(Parsed& p) {
    const std::vector<uint8_t>& b = p.bytes;
    if (b.size() < 8) {
        std::fprintf(stderr, "dhoh_batch: %s: not a valid hoh file!\n", p.in.c_str());  // dhoh.cpp:323
        return 3;
    }
    if (b[0] != 153 || b[1] != 72 || b[2] != 79 || b[3] != 72) {
        std::fprintf(stderr, "dhoh_batch: %s: not a valid hoh file!\n", p.in.c_str());  // dhoh.cpp:333
        return 4;
    }
    if (b[4] != 2 || b[5] != 8) {  // the encoder only writes RGB at 8 bits (choh.cpp:443-446)
        std::fprintf(stderr, "dhoh_batch: %s: pixel format %d at depth %d is not implemented\n", p.in.c_str(), b[4], b[5]);
        return 5;
    }
    size_t at = 6, w1 = 0, h1 = 0;
    if (!get_varint(b, at, w1) || !get_varint(b, at, h1)) return 3;
    p.width = (uint32_t)w1 + 1;
    p.height = (uint32_t)h1 + 1;
    hoh_tile_geometry g;
    hoh_tile_geometry_for(p.width, p.height, &g);
    if (at + 2 > b.size()) {
        std::fprintf(stderr, "dhoh_batch: %s holds a header and no tile: stock choh never writes the tile of an untiled image (SURVEY D1)\n",
                     p.in.c_str());
        return 3;
    }
    const uint32_t xt = b[at] + 1u, yt = b[at + 1] + 1u;  // dhoh.cpp:32-33
    if (xt == 1 && yt == 1) {  // an untiled image: what follows IS the tile, whose own first bytes are this 00 00 marker
        if (g.tiles_per_image != 1) return 4;
        p.tile_begin = {at, b.size()};
        return 0;
    }
    at += 2;
    if (xt != g.x_tiles || yt != g.y_tiles) {
        std::fprintf(stderr, "dhoh_batch: %s: tile grid %ux%u is not the encoder's %ux%u for %ux%u pixels\n", p.in.c_str(), xt, yt,
                     g.x_tiles, g.y_tiles, p.width, p.height);
        return 5;
    }
    std::vector<size_t> sizes(g.tiles_per_image - 1);
    for (size_t& s : sizes)
        if (!get_varint(b, at, s)) return 3;  // dhoh.cpp:41-45
    p.tile_begin.assign(1, at);
    for (size_t s : sizes) {
        at += s;
        if (at > b.size()) return 3;
        p.tile_begin.push_back(at);
    }
    p.tile_begin.push_back(b.size());  // the last tile takes the rest of the file
    return 0;
}

std::string stem_of(const std::string& path) {
    const size_t slash = path.find_last_of('/');
    std::string name = slash == std::string::npos ? path : path.substr(slash + 1);
    const size_t dot = name.find_last_of('.');
    return dot == std::string::npos || dot == 0 ? name : name.substr(0, dot);
}

}  // namespace

int main(int argc, char** argv) {
    bool batch = false, crop = false;
    int device = 0;
    uint32_t cx = 0, cy = 0, cw = 0, ch = 0;
    std::vector<std::string> pos;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        if (a == "--batch") batch = true;
        else if (a == "--device" && i + 1 < argc) device = std::atoi(argv[++i]);
        else if (a == "--crop" && i + 4 < argc) {
            crop = true;
            uint32_t* v[4] = {&cx, &cy, &cw, &ch};
            for (int k = 0; k < 4; k++) {
                char* end = nullptr;
                const long x = std::strtol(argv[++i], &end, 10);
                if (!end || *end || x < 0 || x > 0x7fffffffL) {
                    std::fprintf(stderr, "dhoh_batch: --crop takes four non-negative integers X Y W H\n");
                    return 1;
                }
                *v[k] = (uint32_t)x;
            }
            if (cw == 0 || ch == 0) {
                std::fprintf(stderr, "dhoh_batch: --crop: the window must not be empty\n");
                return 1;
            }
        } else if (a == "--help" || a == "-h") {
            std::printf("usage: dhoh_batch [--crop X Y W H] infile.hoh outfile.rgb\n"
                        "       dhoh_batch [--crop X Y W H] --batch outdir in1.hoh [in2.hoh ...]\n");
            return 0;
        } else pos.push_back(a);
    }
    std::vector<Parsed> files;
    if (!batch) {
        if (pos.size() < 2) {
            std::printf("not enough arguments!\n");  // dhoh.cpp:312
            return 1;
        }
        files.emplace_back();
        files[0].in = pos[0];
        files[0].out = pos[1];
    } else {
        if (pos.size() < 2) return 1;
        for (size_t i = 1; i < pos.size(); i++) {
            files.emplace_back();
            files.back().in = pos[i];
            files.back().out = pos[0] + "/" + stem_of(pos[i]) + ".rgb";
        }
    }
    std::map<std::pair<uint32_t, uint32_t>, std::vector<size_t>> by_size;  // one GPU call per image size
    for (size_t i = 0; i < files.size(); i++) {
        if (!read_file(files[i].in, files[i].bytes)) return 2;
        if (int rc = parse_container(files[i])) return rc;
        if (crop && ((uint64_t)cx + cw > files[i].width || (uint64_t)cy + ch > files[i].height)) {
            std::fprintf(stderr, "dhoh_batch: --crop %u %u %u %u does not lie inside %s (%ux%u)\n", cx, cy, cw, ch,
                         files[i].in.c_str(), files[i].width, files[i].height);
            return 1;
        }
        by_size[{files[i].width, files[i].height}].push_back(i);
    }
    hoh_ctx* ctx = nullptr;
    int st = hoh_ctx_create(device, nullptr, &ctx);
    if (st != HOH_OK) {
        std::fprintf(stderr, "dhoh_batch: no usable CUDA device %d: %s (there is no CPU fallback)\n", device, hoh_strerror(st));
        return 3;
    }
    int rc = 0;
    for (const auto& group : by_size) {
        const uint32_t w = group.first.first, h = group.first.second;
        const std::vector<size_t>& idx = group.second;
        hoh_tile_geometry g;
        hoh_tile_geometry_for(w, h, &g);
        const size_t n = idx.size(), n_tiles = n * g.tiles_per_image;
        const size_t raw1 = crop ? (size_t)cw * ch * 3 : (size_t)w * h * 3;  // bytes written per file
        size_t total = 0;
        for (size_t i : idx) total += files[i].tile_begin.back() - files[i].tile_begin.front();
        uint8_t *packed = nullptr, *rgb = nullptr;
        if (hoh_host_alloc(ctx, total + 16, (void**)&packed) != HOH_OK || hoh_host_alloc(ctx, n * raw1, (void**)&rgb) != HOH_OK) {
            std::fprintf(stderr, "dhoh_batch: cannot pin host memory: %s\n", hoh_last_cuda_error(ctx));
            return 3;
        }
        std::vector<uint64_t> off(n_tiles + 1);
        std::vector<int32_t> status(n_tiles);
        size_t at = 0, t = 0;
        for (size_t i : idx) {
            const Parsed& p = files[i];
            for (size_t k = 0; k + 1 < p.tile_begin.size(); k++) off[t++] = at + (p.tile_begin[k] - p.tile_begin[0]);
            const size_t len = p.tile_begin.back() - p.tile_begin.front();
            std::memcpy(packed + at, p.bytes.data() + p.tile_begin.front(), len);
            at += len;
        }
        off[t] = at;
        if (crop) {  // one status per file: its failing touched tile with the lowest index
            std::vector<uint32_t> origin(2 * n);
            for (size_t k = 0; k < n; k++) origin[2 * k] = cx, origin[2 * k + 1] = cy;
            st = hoh_decode_regions_host(ctx, packed, total, off.data(), n, w, h, origin.data(), cw, ch, rgb, status.data());
        } else {
            st = hoh_decode_images_host(ctx, packed, total, off.data(), n, w, h, rgb, status.data());
        }
        if (st != HOH_OK) {
            std::fprintf(stderr, "dhoh_batch: %s: %s (%s)\n", crop ? "hoh_decode_regions_host" : "hoh_decode_images_host",
                         hoh_strerror(st), hoh_last_cuda_error(ctx));
            return 3;
        }
        for (size_t k = 0; k < n; k++) {
            const Parsed& p = files[idx[k]];
            if (crop && status[k] != HOH_S_OK) {
                std::fprintf(stderr, "dhoh_batch: %s: a tile of the window cannot be decoded (stream status %d)\n",
                             p.in.c_str(), status[k]);
                rc = 4;
            }
            for (size_t j = 0; j < (crop ? 0 : g.tiles_per_image); j++)
                if (status[k * g.tiles_per_image + j] != HOH_S_OK) {
                    std::fprintf(stderr, "dhoh_batch: %s tile %zu cannot be decoded (stream status %d%s)\n", p.in.c_str(), j,
                                 status[k * g.tiles_per_image + j],
                                 status[k * g.tiles_per_image + j] == HOH_S_BAD_LAYER
                                     ? ": a channel does not end where the container says - stock choh -s1..4 output under SURVEY D7?"
                                     : "");
                    rc = 4;
                }
            FILE* f = std::fopen(p.out.c_str(), "wb");
            if (!f || std::fwrite(rgb + k * raw1, 1, raw1, f) != raw1 || std::fclose(f) != 0) {
                std::fprintf(stderr, "dhoh_batch: cannot write %s\n", p.out.c_str());
                return 2;
            }
        }
        hoh_host_free(ctx, packed);
        hoh_host_free(ctx, rgb);
    }
    hoh_ctx_destroy(ctx);
    return rc;
}
