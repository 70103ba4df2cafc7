/* hohgpu.h — C-ABI of libhohgpu.so: the B200 (sm_100a) implementation of the hoh-ANS hot path.
 *
 * What this replaces.  hoh-ANS (hohMiyazawa/hoh-ANS) has no plugin / FFI interface: its hot path is a
 * set of free C++ functions defined in headers which the container code (choh.cpp, dhoh.cpp,
 * layer_encode.hpp, layer_decode.hpp, lz.hpp, un_lz.hpp) calls directly.  Every entry point below
 * names the reference function it stands in for (file:line into the reference tree).  Two tiers:
 *
 *   (i)  compat shims  — one call = one reference call, HOST pointers in and out, the reference's
 *        value semantics (same bytes, same symbols, same planes).  They exist so that the
 *        reference's own host code can be relinked against the GPU (see INTEGRATION.md) and so that
 *        parity tests read like the reference's tests.  Each call is a batch of one: H2D copy,
 *        kernels, D2H copy.
 *   (ii) batched entry points — DEVICE pointers, many independent streams / tiles / images per
 *        call; this is where the throughput is.  No host work other than launching kernels.
 *
 * Conventions: plain C, plain pointers and sizes, no exceptions, no stdout, every function returns
 * an int status (HOH_OK == 0) unless stated otherwise; the library owns its scratch device memory
 * (grown on demand, cached in the context), the caller owns every buffer it passes in and states
 * its capacity.  A context is bound to one CUDA device and one stream; calls on one context must
 * not overlap in time, different contexts are independent (one per GPU / per host thread).
 * There is NO CPU fallback: without a CUDA device hoh_ctx_create fails with HOH_E_CUDA.
 */
#ifndef HOHGPU_H
#define HOHGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------ */
/* status codes                                                                               */
/* ------------------------------------------------------------------------------------------ */
#define HOH_OK 0
#define HOH_E_CUDA 1          /* a CUDA runtime call failed (hoh_last_cuda_error has the text)   */
#define HOH_E_ARG 2           /* bad argument (null pointer, zero size, misaligned offset)       */
#define HOH_E_UNSUPPORTED 3   /* outside the hot path's domain (range > 512, prob_bits > 19 ...) */
#define HOH_E_CAPACITY 4      /* caller's output buffer too small                                */
#define HOH_E_STREAM 5        /* at least one stream failed; see the per-stream status array      */

/* per-stream status (hoh_stream_result.status) */
#define HOH_S_OK 0
#define HOH_S_RANGE_GT_TOTAL 1 /* stattools.hpp:14  assert(target_total >= size) would fire        */
#define HOH_S_NO_DONOR 2       /* stattools.hpp:42  assert(best_steal != -1) would fire            */
#define HOH_S_BAD_TABLE 3      /* decode: table storage mode 3                                     */
#define HOH_S_OVERFLOW 4       /* output slab / symbol capacity too small                          */
#define HOH_S_BAD_LAYER 5      /* tile decode: channel header is not the mode-0 form 10 00 00 00 10 */
#define HOH_S_BAD_STATE 6      /* decode: the rANS state after the last symbol is not 2^31, the value the
                                * encoder starts from (rans64.hpp:65): the table or the payload is damaged.
                                * The symbols are still delivered (the reference would not notice).      */
#define HOH_S_BAD_ESTIMATE 7   /* encode: the payload length computed from the histogram alone (used to pick a
                                * channel's candidate without coding the others) does not contain the coded
                                * length: an internal error, never expected                               */

/* decode flags: 0 reproduces entropy_decoding.hpp byte for byte including its defects; the FIX
 * bits turn individual defects off (SURVEY.md section 8.0). */
#define HOH_FIX_PROB_BITS5 1u /* D9: prob_bits is a 5-bit field (mask 0x7C), reference masks 4 bits */
#define HOH_FIX_ADVANCE 2u    /* D8: leave *byte_pointer after the rANS payload, not at its start   */
#define HOH_FIX_EMPTY 4u      /* D2: a zero-symbol stream has no metadata byte                      */
#define HOH_FIX_ALL 7u
/* Decoder side: recognise the table of a stream with ONE distinct symbol, whose over-wide frequency field reads 0
 * and increments the clamp bits sharing its first byte (D6: every stock `choh -s0` file of a photograph has such
 * a stream — the LZ stream of 255s), and give that symbol the whole range.
 * The pattern cannot be produced by a valid table, so the flag never changes how a valid stream decodes. */
#define HOH_FIX_CARRY 32u
#define HOH_FIX_DECODER 39u /* HOH_FIX_ALL | HOH_FIX_CARRY: what hoh_decode_images uses */
/* Encoder side (hoh_layer_encode_batch, hoh_encode_images): D7 — keep the winning candidate's own bytes
 * instead of the reference's stale buffer, and give the plain fastpath stream its own single-predictor header
 * when it beats the searched candidates.  0 = byte-for-byte reference output (not decodable where D7 strikes). */
#define HOH_FIX_STALE 8u
/* Encoder side: a stream with ONE distinct symbol would give it all of 2^prob_bits, which the table's
 * prob_bits-wide field cannot hold (D6): neither the reference's decoder nor any other can read it back.
 * With this flag one count goes to a neighbouring symbol that never occurs (a few bits per stream), and table
 * mode 1 (maxbits-wide fields) is not chosen when a frequency does not fit its field. */
#define HOH_FIX_LONE 16u
#define HOH_FIX_ENCODER 24u /* HOH_FIX_STALE | HOH_FIX_LONE: what hoh_decode_images can always invert */

#define HOH_MAX_RANGE 512     /* largest alphabet on the hot path (depth-9 sub-green planes)        */
#define HOH_MAX_PROB_BITS 19  /* layer_encode.hpp:359-392 tries up to 19                            */
#define HOH_HEAD_CAP 1536     /* bytes reserved in front of a payload for varints + metadata + table */

typedef struct hoh_ctx hoh_ctx;

/* ------------------------------------------------------------------------------------------ */
/* context, memory and timing helpers                                                         */
/* ------------------------------------------------------------------------------------------ */
/* cuda_stream: a cudaStream_t to launch on (e.g. torch.cuda.current_stream().cuda_stream), or NULL
 * to let the context create its own non-blocking stream. */
int hoh_ctx_create(int device, void* cuda_stream, hoh_ctx** out);
void hoh_ctx_destroy(hoh_ctx* ctx);
int hoh_sync(hoh_ctx* ctx);
/* Development aid: what hoh_layer_encode_batch / hoh_encode_images (cruncher mode >= 1) did since the last call of this
 * function, summed over the context and its child contexts: out[0] = candidates that went through the rANS coder,
 * out[1] = planes whose candidate sizes the histogram-derived intervals could not settle (their whole path was coded, as
 * the reference does for every plane), out[2] = planes.  Synchronises the context. */
int hoh_debug_layer_stats(hoh_ctx* ctx, uint64_t out[3]);
/* Frees the scratch device memory the context (and its internal child contexts) caches between calls.  The
 * chunked entry points do this themselves when the image shape or mode changes, and an allocation that fails
 * first frees whatever scratch the CURRENT top-level call has not asked for (e.g. the encoder's, during a decode)
 * and tries again, so a caller never has to call this for correctness — only to hand the memory back early. */
int hoh_release_scratch(hoh_ctx* ctx);
const char* hoh_strerror(int status);
const char* hoh_last_cuda_error(hoh_ctx* ctx);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches claim). */
uint64_t hoh_launch_count(hoh_ctx* ctx);

int hoh_dev_alloc(hoh_ctx* ctx, size_t bytes, void** dptr);
int hoh_dev_free(hoh_ctx* ctx, void* dptr);
int hoh_dev_memset(hoh_ctx* ctx, void* dptr, int value, size_t bytes);
int hoh_host_alloc(hoh_ctx* ctx, size_t bytes, void** hptr); /* pinned */
int hoh_host_free(hoh_ctx* ctx, void* hptr);
int hoh_h2d(hoh_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes); /* async on the ctx stream */
int hoh_d2h(hoh_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes); /* async on the ctx stream */
/* CUDA-event timer on the context's stream: start/stop record events, elapsed synchronises. */
int hoh_timer_start(hoh_ctx* ctx, int slot); /* slot 0..15 */
int hoh_timer_stop(hoh_ctx* ctx, int slot);
int hoh_timer_elapsed_ms(hoh_ctx* ctx, int slot, float* ms);
/* Writes a scratch buffer larger than L2 so that the next timed launch starts cold. */
int hoh_flush_l2(hoh_ctx* ctx);
/* Per-kernel device timing: between begin and end every kernel launch is followed by a CUDA event on
 * the context's stream; end synchronises and sums the intervals per kernel name.  For profiling
 * passes only (the events add a little launch overhead). */
int hoh_profile_begin(hoh_ctx* ctx);
int hoh_profile_end(hoh_ctx* ctx);
int hoh_profile_count(hoh_ctx* ctx);
int hoh_profile_entry(hoh_ctx* ctx, int index, const char** name, double* total_ms, uint64_t* launches);

/* ------------------------------------------------------------------------------------------ */
/* (ii) batched entropy coding — entropy_encoding.hpp:8 / entropy_decoding.hpp:134 over N streams */
/* ------------------------------------------------------------------------------------------ */
/* One stream to encode.  Arrays of these live in DEVICE memory. */
typedef struct hoh_enc_stream {
    uint64_t sym_off;    /* element offset of the first symbol in the u16 symbol buffer; multiple of 8 */
    uint32_t n;          /* symbols in this stream (< 2^21: varint.hpp:39-45)                           */
    uint32_t range;      /* alphabet size, 1..HOH_MAX_RANGE                                             */
    uint32_t prob_bits;  /* 1..HOH_MAX_PROB_BITS, 2^prob_bits >= range                                  */
    uint32_t prefix_len; /* literal bytes emitted in front of the stream (channel header), 0..8         */
    uint8_t prefix[8];
    uint64_t out_off;    /* byte offset of this stream's slab in the output buffer; multiple of 16      */
    uint32_t out_cap;    /* slab bytes, multiple of 16; see hoh_enc_slab_bytes                          */
    uint32_t reserved;   /* 0, or HOH_FIX_LONE                                                          */
} hoh_enc_stream;

typedef struct hoh_stream_result {
    uint64_t start;  /* byte offset in the output buffer where prefix+stream begin           */
    uint32_t size;   /* prefix_len + bytes encode_entropy would have returned                */
    int32_t status;  /* HOH_S_*                                                              */
    uint32_t payload_bytes; /* rANS payload length (0 in stored mode / empty stream)         */
    uint32_t stored;        /* 1 if the stored-mode fallback won (entropy_encoding.hpp:244)  */
} hoh_stream_result;

/* Slab size that can never overflow for a stream of n symbols at prob_bits. */
size_t hoh_enc_slab_bytes(size_t n, uint32_t prob_bits);

/* encode_entropy for every stream: histogram -> normalize_freqs -> header + table -> rANS -> length
 * varint -> stored-mode fallback.  d_streams, d_symbols, d_out, d_results are device pointers.
 * max_range / max_prob_bits / max_n are upper bounds over the batch (they size shared memory and
 * loop trip counts; the host does not read the descriptors). */
int hoh_encode_entropy_batch(hoh_ctx* ctx, const hoh_enc_stream* d_streams, size_t n_streams,
                             const uint16_t* d_symbols, uint8_t* d_out, hoh_stream_result* d_results,
                             uint32_t max_range, uint32_t max_prob_bits, uint32_t max_n);

/* One stream to decode. */
typedef struct hoh_dec_stream {
    uint64_t in_off;   /* byte offset of the stream header (varint(range-1)) in the input buffer */
    uint64_t sym_off;  /* element offset for the decoded u16 symbols; multiple of 8              */
    uint32_t sym_cap;  /* symbols that may be written                                            */
    uint32_t flags;    /* HOH_FIX_*                                                              */
} hoh_dec_stream;

typedef struct hoh_dec_result {
    uint64_t end_off;  /* *byte_pointer after the call (reference semantics, see HOH_FIX_ADVANCE) */
    uint32_t n;        /* symbols decoded                                                         */
    int32_t status;
    uint32_t range;
    uint32_t prob_bits;
    uint32_t stored;
    uint32_t table_mode;
} hoh_dec_result;

/* decode_entropy for every stream.  in_bytes = size of d_in.
 * INPUT CONTRACT of every device-pointer decode entry point (this one, hoh_decode_images_s0, hoh_decode_images):
 * the payload words are fetched as aligned 16-byte vectors and never at or past the last whole 16-byte line of the
 * buffer, so d_in must be READABLE AND ZERO for at least 32 bytes behind the last stream byte, and in_bytes must
 * include that padding (pass in_bytes = data bytes + 32, rounded as you like).  in_bytes < 32 is HOH_E_ARG.  The
 * host-pointer forms (hoh_decode_entropy, hoh_decode_images_s0_host, hoh_decode_images_host) take exact sizes and
 * add the padding themselves. */
int hoh_decode_entropy_batch(hoh_ctx* ctx, const hoh_dec_stream* d_streams, size_t n_streams,
                             const uint8_t* d_in, size_t in_bytes, uint16_t* d_symbols,
                             hoh_dec_result* d_results, uint32_t max_n);

/* rans64.hpp:262 / :107-142 loops with ONE caller-supplied table shared by all streams (config 4:
 * static-table symbol-stream sweep).  Stream i covers symbols [i*stream_len, min(n, (i+1)*stream_len));
 * its payload is written at d_out + i*slab_bytes, END-aligned inside the slab; d_payload_bytes[i]
 * receives its length.  stream_len multiple of 8, slab_bytes multiple of 16. */
int hoh_rans_encode_static(hoh_ctx* ctx, const uint16_t* d_symbols, size_t n, uint32_t stream_len,
                           const uint32_t* d_cum /* range+1 */, uint32_t range, uint32_t prob_bits,
                           uint8_t* d_out, uint32_t slab_bytes, uint32_t* d_payload_bytes);
int hoh_rans_decode_static(hoh_ctx* ctx, const uint8_t* d_in, uint32_t slab_bytes,
                           const uint32_t* d_payload_bytes, size_t n, uint32_t stream_len,
                           const uint32_t* d_cum, uint32_t range, uint32_t prob_bits,
                           uint16_t* d_symbols);

/* ------------------------------------------------------------------------------------------ */
/* (ii) batched tile codec, cruncher mode 0 — choh.cpp:454-506 tiling, channel.hpp:73,            */
/*      layer_encode.hpp:11 (mode 0 branch), and their inverses                                   */
/* ------------------------------------------------------------------------------------------ */
typedef struct hoh_tile_geometry {
    uint32_t width, height;     /* image                                             */
    uint32_t x_tiles, y_tiles;  /* choh.cpp:455-456 (1,1 when the image is not tiled) */
    uint32_t tile_w, tile_h;    /* choh.cpp:459-460 nominal tile size                */
    uint32_t tiles_per_image;
    uint32_t streams_per_image; /* 3 * tiles_per_image (G, R-G, B-G)                 */
} hoh_tile_geometry;

/* choh.cpp:454-460: the 256-pixel image tiling rule. */
int hoh_tile_geometry_for(uint32_t width, uint32_t height, hoh_tile_geometry* out);

/* Bytes of device output needed by hoh_encode_images_s0 for n_images (slabs, worst case). */
size_t hoh_encode_images_out_bytes(const hoh_tile_geometry* g, size_t n_images);

/* Encode n_images interleaved RGB8 images (d_rgb: n_images * height * width * 3 bytes) at cruncher
 * mode 0 with the subtract-green colour mode (choh.cpp:219-255) and no LZ matches (NUKE == 0; pass
 * d_nuke = NULL) or the LEMPEL_NUKE map hoh_find_lz_images writes (d_nuke: one byte per pixel, tile t's
 * map in raster order at t * nuke_stride, nuke_stride = tile_w*tile_h rounded up to 8): the residuals of
 * covered pixels are dropped before entropy coding (layer_encode.hpp:93-99).
 * For stream s = (image * tiles_per_image + tile) * 3 + channel, d_results[s] gives the byte range in
 * d_out holding exactly what layer_encode() writes for that channel ("10 00 00 00 10" + stream).
 * If d_packed != NULL the channel payloads are also gathered back to back in stream order into
 * d_packed (capacity packed_cap bytes) and d_packed_off[s] (n_streams+1 entries, u64) receives their
 * offsets — the "final gather" the host container writer consumes. */
int hoh_encode_images_s0(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_images, uint32_t width,
                         uint32_t height, const uint8_t* d_nuke, uint8_t* d_out, size_t out_bytes,
                         hoh_stream_result* d_results, uint8_t* d_packed, size_t packed_cap,
                         uint64_t* d_packed_off);

/* Inverse: channel payloads (as produced above: d_packed + d_packed_off, n_images*streams_per_image
 * of them, each starting with the 5-byte mode-0 channel header) -> interleaved RGB8 images.
 * The un-prediction is the exact inverse of channelpredict_fastpath (pure MED, SURVEY D10) and the
 * colour inverse is the algebraic inverse of channel.hpp:73-79 (SURVEY D4).  d_backref = NULL (the fused
 * wavefront kernel) or the LEMPEL_BACKREF maps for the copies of unprediction.hpp:63-65: one u16 per pixel, tile
 * t's map in raster order at t * plane_stride, plane_stride = tile_w*tile_h rounded up to 8 (the layout of d_nuke
 * on the encode side); 0 = coded pixel, b > 0 = copy of the pixel b positions earlier in the tile.  With a map the
 * residual streams are dense (covered pixels have none) and the un-prediction is a raster walk per plane; a stream
 * whose symbol count differs from the number of uncovered pixels gets HOH_S_BAD_LAYER.
 * packed_bytes: see the input contract at hoh_decode_entropy_batch (32 zero bytes of padding included). */
int hoh_decode_images_s0(hoh_ctx* ctx, const uint8_t* d_packed, size_t packed_bytes,
                         const uint64_t* d_packed_off, size_t n_images, uint32_t width,
                         uint32_t height, const uint16_t* d_backref, uint8_t* d_rgb,
                         int32_t* d_status /* n_images*streams_per_image */);

/* Host-buffer forms of the two calls above — what a host container writer / reader calls: the batch is
 * cut into chunks of whole images that are pipelined, up to four in flight: while one chunk is copied in,
 * earlier ones are coded (each in a child context of its own, so their kernels run concurrently) and
 * copied out, on copy streams of the context.  Work queued on the context's stream before the call
 * happens first.  Device staging lives in the context and is reused across calls.  Pass pinned buffers
 * (hoh_host_alloc) for full copy bandwidth.  encode: packed_host/packed_cap receive the channel
 * payloads back to back, off_host (n_streams+1 u64) their offsets, results_host (n_streams, may be
 * NULL) the per-stream results; HOH_E_CAPACITY when packed_cap is too small.  decode: exact sizes, no
 * padding needed; status_host (n_streams, may be NULL); HOH_E_ARG when off_host runs backwards or past
 * packed_bytes between chunks (a bad range inside a chunk fails its stream's status).  On any failure
 * of these two calls, or of the whole-tile host calls below, every copy and kernel of the call has been
 * drained before it returns, and the context stays usable. */
int hoh_encode_images_s0_host(hoh_ctx* ctx, const uint8_t* rgb_host, size_t n_images, uint32_t width,
                              uint32_t height, uint8_t* packed_host, size_t packed_cap, uint64_t* off_host,
                              hoh_stream_result* results_host);
int hoh_decode_images_s0_host(hoh_ctx* ctx, const uint8_t* packed_host, size_t packed_bytes,
                              const uint64_t* off_host, size_t n_images, uint32_t width, uint32_t height,
                              uint8_t* rgb_host, int32_t* status_host);

/* ------------------------------------------------------------------------------------------ */
/* (ii) batched plane kernels (device pointers; planes are u16, raster order, back to back)     */
/* ------------------------------------------------------------------------------------------ */
/* channel_picker channel.hpp:63-71: channel `target` of `total`-byte interleaved pixels -> u16 plane. */
int hoh_channel_picker_dev(hoh_ctx* ctx, const uint8_t* d_src, size_t n_px, int total, int target, uint16_t* d_out);

/* channel.hpp:73 subtract_green over `pixels` interleaved RGB8 pixels. */
int hoh_subtract_green_dev(hoh_ctx* ctx, const uint8_t* d_rgb, size_t pixels, uint16_t* d_g,
                           uint16_t* d_rg, uint16_t* d_bg);
/* algebraic inverse (SURVEY D4) */
int hoh_add_green_dev(hoh_ctx* ctx, const uint16_t* d_g, const uint16_t* d_rg, const uint16_t* d_bg,
                      size_t pixels, uint8_t* d_rgb);
/* prediction.hpp:6 channelpredict_fastpath on n_planes planes of w*h. */
int hoh_predict_fastpath_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h,
                             int depth, uint16_t* d_resid);
/* exact inverse of the above (with optional back-reference copies, n_planes*w*h u16 or NULL);
 * residuals are dense per plane (w*h of them when d_backref == NULL). */
int hoh_unpredict_fastpath_dev(hoh_ctx* ctx, const uint16_t* d_resid, size_t n_planes, int w, int h,
                               int depth, const uint16_t* d_backref, uint16_t* d_planes);
/* prediction.hpp:153 channelpredict_all: per plane its own tile_map (x_tiles*y_tiles u16 masks). */
int hoh_predict_all_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h,
                        int depth, int x_tiles, int y_tiles, const uint16_t* d_tile_maps,
                        uint16_t* d_resid);
/* unprediction.hpp:6 unpredict_all.  Residuals of plane p start at d_resid + p*w*h. */
int hoh_unpredict_all_dev(hoh_ctx* ctx, const uint16_t* d_resid, size_t n_planes, int w, int h,
                          int depth, int x_tiles, int y_tiles, const uint16_t* d_tile_maps,
                          const uint16_t* d_backref, uint16_t* d_planes);
/* prediction.hpp:46 channelpredict_section for every (plane, grid cell, mask): writes the cell's
 * residuals (cell-raster order) to d_resid + ((p*cells + cell)*n_masks + m)*cell_cap and the count to
 * d_counts (same index without cell_cap); cell_cap >= tile_w*tile_h of the predictor grid. */
int hoh_predict_section_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h,
                            int depth, int x_tiles, int y_tiles, const uint16_t* d_masks, int n_masks,
                            uint16_t* d_resid, uint32_t cell_cap, uint32_t* d_counts);
/* layer_encode.hpp:126-272: the predictor search (histogram -> -log2 cost table -> per cell argmin
 * over the first min(14, 5*mode) stock masks, costs summed in raster order in double precision,
 * strict <; refinement pass when mode > 2) followed by channelpredict_all.  Outputs per plane:
 * tile_map (cells u16), index_list (cells u8, index into the 14 stock masks) and the final residual
 * plane.  The grid is ceil(w/40) x ceil(h/40) (layer_encode.hpp:124,150-151). */
int hoh_predictor_search_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h,
                             int depth, int mode, uint16_t* d_tile_maps, uint8_t* d_index_lists,
                             uint16_t* d_resid);

/* ------------------------------------------------------------------------------------------ */
/* (vi) whole tiles — encode_tile choh.cpp:104-382 for every tile of N images, any cruncher mode   */
/* ------------------------------------------------------------------------------------------ */
#define HOH_TILE_GREY 1u    /* every pixel grey: encode_tile takes the greyscale branch (choh.cpp:180-213)      */
#define HOH_TILE_PALETTE 2u /* <= 256 colours: encode_tile also tries the indexed mode (choh.cpp:298-307)       */

typedef struct hoh_tile_result {
    uint64_t start;        /* byte offset of the tile's bytes in d_packed                                  */
    uint32_t size;         /* bytes of the tile as emitted here; = encode_tile's return value when flags == 0
                            * (a tile with HOH_TILE_GREY / HOH_TILE_PALETTE is emitted in subtract-green mode, where
                            * the reference would have taken its greyscale / indexed branch: the bytes are a valid
                            * tile but NOT what choh writes — the host must notice the flag)                    */
    int32_t status;        /* HOH_S_* of the first failing stage                                           */
    uint32_t colour_mode;  /* 128 subtract-green, 2 plain RGB (choh.cpp:295-327)                           */
    uint32_t lz_size;      /* bytes of the LZ record inside the tile                                       */
    uint32_t chan_size[3]; /* the three channel payloads                                                   */
    uint32_t flags;        /* HOH_TILE_*: the reference would (also) take a colour mode that stays on the host */
} hoh_tile_result;

/* encode_tile for every tile of n_images interleaved RGB8 images at cruncher mode 0..4, entirely on the
 * device: LZ match finder with the mode's seek window (choh.cpp:123-156), subtract-green planes (and the plain
 * R, B alternatives at mode > 2), layer_encode of every plane with the NUKE maps, the colour-mode comparison
 * and the emission of the tile's bytes (header 00 00, colour mode, LZ record, channel-order byte, size varints,
 * channels).  Tile t = image * tiles_per_image + tile occupies d_packed[d_tile_off[t], d_tile_off[t+1]).
 * The host keeps only the file header and the tile offset table (choh.cpp:436-506).  Tiles the reference would
 * code in greyscale / indexed mode are flagged (they still get their sub-green bytes).  Image sizes whose last
 * tile column / row is narrower than the others (choh.cpp:459-474) are handled one tile shape at a time.  Large
 * batches are processed in chunks of whole images sized by an internal scratch budget (half of the device's
 * memory, at most 55 % of what is free, or the HOH_SCRATCH_GB environment variable). */
int hoh_encode_images(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_images, uint32_t width, uint32_t height,
                      int mode, unsigned flags /* 0 or HOH_FIX_ENCODER */, uint8_t* d_packed, size_t packed_cap, uint64_t* d_tile_off,
                      hoh_tile_result* d_tiles);

/* The inverse: tiles as hoh_encode_images (or stock `choh`) wrote them -> interleaved RGB8 images, entirely on
 * the device.  This is the decoder the format needs rather than the reference's (dhoh.cpp:22-141,
 * un_lz.hpp:66-180, layer_decode.hpp:127-277 cannot parse choh's output: SURVEY D2, D3, D4, D8, D9, D10, D12 are
 * corrected here; none of the corrections changes hot-path arithmetic): tile header, the 3 or 4 LZ side streams,
 * channel order and sizes, per channel the layer header / predictor masks / predictor-index stream / residual
 * stream, LZ expansion into back-references, un-prediction (pure-MED inverse for the single-predictor header,
 * unpredict_all otherwise) with the copies of unprediction.hpp:63-65, colour inverse, tile scatter.
 * Tile t's bytes are d_packed[d_tile_off[t], d_tile_off[t+1]).  d_status[t] != 0: the tile could not be decoded
 * (its pixels are left untouched).  Every stream has to end where the container says it ends, so truncated tiles
 * and the channels the reference emits under defect D7 (a stale buffer cut to another candidate's length, see
 * HOH_FIX_STALE) are reported rather than decoded to wrong pixels; a changed payload byte is caught by the final
 * rANS state (HOH_S_BAD_STATE: a sound stream ends in the encoder's initial state 2^31) — the format carries no
 * checksum, so that is a 2^-32-ish guarantee per stream, not a proof. */
int hoh_decode_images(hoh_ctx* ctx, const uint8_t* d_packed, size_t packed_bytes, const uint64_t* d_tile_off,
                      size_t n_images, uint32_t width, uint32_t height, uint8_t* d_rgb, int32_t* d_status);

/* Host-buffer forms of the two calls above — what a batched container writer / reader calls (tools/choh_batch.cpp,
 * tools/dhoh_batch.cpp): the batch is cut into chunks of whole images, chunk c+1 is copied in while chunk c is coded
 * and chunk c-1 is copied out (own copy streams; pass pinned buffers from hoh_host_alloc for full PCIe bandwidth).
 * encode: packed_host[0, tile_off_host[n_tiles]) receives the tiles back to back, tile_off_host has n_tiles+1
 * entries, tiles_host n_tiles records (start rebased to packed_host).  decode: exact sizes, no padding needed;
 * status_host has n_tiles entries; pixels of tiles that fail to decode are zero.  On any failure every copy has
 * been drained before the call returns. */
int hoh_encode_images_host(hoh_ctx* ctx, const uint8_t* rgb_host, size_t n_images, uint32_t width, uint32_t height,
                           int mode, unsigned flags, uint8_t* packed_host, size_t packed_cap, uint64_t* tile_off_host,
                           hoh_tile_result* tiles_host);
int hoh_decode_images_host(hoh_ctx* ctx, const uint8_t* packed_host, size_t packed_bytes, const uint64_t* tile_off_host,
                           size_t n_images, uint32_t width, uint32_t height, uint8_t* rgb_host, int32_t* status_host);

#define HOH_S_BAD_WINDOW 8  /* decode_regions: the window does not lie inside the image */

/* Region decode (random access into tiled images): the crop_w x crop_h window at (origin[2i], origin[2i+1]) of image
 * i, for every image of a batch that hoh_encode_images (or stock choh) wrote.  Only the tiles the window touches are
 * decoded.  d_crops: n_images * crop_h * crop_w * 3 bytes, dense (crop i at i * crop_h * crop_w * 3, row-major RGB8).
 * d_status[i] (n_images entries) is HOH_S_OK when every tile the window touches decoded.  Otherwise it is the status
 * of the failing touched tile with the lowest tile index; that tile's part of the crop is left untouched, as in
 * hoh_decode_images.  A window that does not lie inside its image gets HOH_S_BAD_WINDOW and its crop is untouched.
 * The bytes of tiles the window does not touch are never decoded: they may be anything, as long as d_tile_off stays
 * ascending.  Input contract as for hoh_decode_images (32 zero bytes of padding).  crop_w == 0, crop_h == 0,
 * crop_w > width or crop_h > height is HOH_E_ARG; the origins are device memory, so a window that does not fit is
 * reported per image. */
int hoh_decode_regions(hoh_ctx* ctx, const uint8_t* d_packed, size_t packed_bytes, const uint64_t* d_tile_off,
                       size_t n_images, uint32_t width, uint32_t height, const uint32_t* d_origin,
                       uint32_t crop_w, uint32_t crop_h, uint8_t* d_crops, int32_t* d_status);
/* Host-buffer form, pipelined like hoh_decode_images_host.  Exact sizes, no padding.  Only the byte ranges of touched
 * tiles cross PCIe (one copy per touched tile row of each window).  Pixels of a failing tile, and the crop of a bad
 * window, are zero.  HOH_E_ARG when the offsets of a touched tile row run backwards or past packed_bytes.  Drains on
 * every failure, like the other host calls. */
int hoh_decode_regions_host(hoh_ctx* ctx, const uint8_t* packed_host, size_t packed_bytes,
                            const uint64_t* tile_off_host, size_t n_images, uint32_t width, uint32_t height,
                            const uint32_t* origin_host, uint32_t crop_w, uint32_t crop_h,
                            uint8_t* crops_host, int32_t* status_host);

/* ------------------------------------------------------------------------------------------ */
/* (v) LZ match finder — find_lz_rgb lz.hpp:6-145 (SURVEY 8(f) row 1) over N tiles                 */
/* ------------------------------------------------------------------------------------------ */
/* Bytes of one tile's LEMPEL record buffer (tag byte + up to four entropy-coded side streams). */
size_t hoh_find_lz_stride(int w, int h);

/* find_lz_rgb for n_tiles tiles of w x h pixels (tile t = RGB8 bytes [t*w*h*3, (t+1)*w*h*3): matches
 * never cross tiles, exactly like the per-tile call at choh.cpp:156).  distance = log2 of the near seek
 * window (choh.cpp:123-136: 6, 10, 11, 12, 14 for cruncher modes 0-4).  d_bonus: per-tile break-even
 * bonus, or NULL to derive it on the device from the tile's colour count (count_colours choh.cpp:17-50 and
 * the table at :138-154).  Outputs: d_nuke[n_tiles*w*h] (0/1, fully written), d_lz[n_tiles * lz_stride]
 * with lz_stride >= hoh_find_lz_stride(w, h), d_lz_size[n_tiles] = find_lz_rgb's return value,
 * d_status[n_tiles] (optional) = HOH_S_*. */
int hoh_find_lz_rgb_batch(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_tiles, int w, int h, int distance,
                          unsigned flags /* 0 or HOH_FIX_LONE */, const int32_t* d_bonus, uint8_t* d_nuke, uint8_t* d_lz, size_t lz_stride,
                          uint32_t* d_lz_size, int32_t* d_status);

/* The same for whole images: every image is cut into tiles as choh.cpp:454-484 cuts it and find_lz_rgb runs
 * on each tile (tile index = image * tiles_per_image + tile, as everywhere in this header).  d_nuke holds
 * n_tiles * nuke_stride bytes with nuke_stride = tile_w*tile_h rounded up to 8 (tile t's map starts at
 * t * nuke_stride; it is the map hoh_encode_images_s0 takes); lz_stride >= hoh_find_lz_stride(tile_w, tile_h). */
int hoh_find_lz_images(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_images, uint32_t width, uint32_t height,
                       int distance, unsigned flags /* 0 or HOH_FIX_LONE */, const int32_t* d_bonus, uint8_t* d_nuke, uint8_t* d_lz, size_t lz_stride,
                       uint32_t* d_lz_size, int32_t* d_status);

/* layer_encode.hpp:11 for n_planes planes of the same geometry (w x h, depth, cruncher mode 0..4): the
 * reference's decision sequence — which candidates are entropy-coded, in which order,
 * which buffer is finally emitted, including the stale-buffer behaviour of SURVEY D7 — replayed with the
 * batched kernels (fastpath residuals, predictor search, up to seven entropy-coding passes per plane).
 * d_results[p] (start, size) locates plane p's channel payload in d_out (capacity out_bytes >=
 * hoh_layer_encode_out_bytes); .stored holds the index of the candidate whose bytes were kept.
 * d_nuke = NULL, or LEMPEL_NUKE maps (one byte per pixel): plane p uses the map at
 * d_nuke + (p / planes_per_map) * nuke_stride — e.g. planes_per_map = 3 when the planes are the G, R-G, B-G
 * planes of consecutive tiles — and the residuals of covered pixels are dropped (layer_encode.hpp:93-99, 328-333).
 * If d_packed != NULL the payloads are also gathered back to back (d_packed_off: n_planes+1 offsets). */
size_t hoh_layer_encode_out_bytes(size_t n_planes, int w, int h, int depth, int mode);
int hoh_layer_encode_batch(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth,
                           int mode, unsigned flags /* 0 or HOH_FIX_STALE | HOH_FIX_LONE */, const uint8_t* d_nuke, size_t nuke_stride, uint32_t planes_per_map,
                           uint8_t* d_out, size_t out_bytes, hoh_stream_result* d_results, uint8_t* d_packed,
                           size_t packed_cap, uint64_t* d_packed_off);

/* ------------------------------------------------------------------------------------------ */
/* (i) compat shims — host pointers, one reference call each                                    */
/* ------------------------------------------------------------------------------------------ */
/* entropy_encoding.hpp:8  size_t encode_entropy(symbols, n, range, out, prob_bits, diagnostics).
 * Returns the byte count through *out_size; out_cap is the capacity the reference never checked. */
int hoh_encode_entropy(hoh_ctx* ctx, const uint16_t* symbols, size_t n, size_t range, uint8_t* out,
                       size_t out_cap, uint32_t prob_bits, size_t* out_size, int* stream_status);
/* entropy_encoding.hpp:283 (8-bit symbols overload) */
int hoh_encode_entropy_8bit(hoh_ctx* ctx, const uint8_t* symbols, size_t n, size_t range, uint8_t* out,
                            size_t out_cap, uint32_t prob_bits, size_t* out_size, int* stream_status);
/* entropy_decoding.hpp:134  uint16_t* decode_entropy(in, in_size, &byte_pointer, &symbol_size, diag).
 * The caller supplies the symbol buffer instead of receiving a new[] array. */
int hoh_decode_entropy(hoh_ctx* ctx, const uint8_t* in, size_t in_size, size_t* byte_pointer,
                       uint16_t* symbols, size_t symbols_cap, size_t* symbol_size, unsigned flags,
                       int* stream_status);
/* stattools.hpp:13 normalize_freqs (in place; cum_freqs has size+1 entries). */
int hoh_normalize_freqs(hoh_ctx* ctx, uint32_t* freqs, uint32_t* cum_freqs, size_t size,
                        uint32_t target_total, int* stream_status);
/* channel.hpp:63 (host pointers; size = bytes of src) */
int hoh_channel_picker(hoh_ctx* ctx, const uint8_t* src, size_t size, int total, int target, uint16_t* out);

/* channel.hpp:73 / :63 */
int hoh_subtract_green(hoh_ctx* ctx, const uint8_t* rgb, size_t size, uint16_t* green, uint16_t* red_g,
                       uint16_t* blue_g);
int hoh_add_green(hoh_ctx* ctx, const uint16_t* green, const uint16_t* red_g, const uint16_t* blue_g,
                  size_t pixels, uint8_t* rgb);
/* prediction.hpp:6, :46, :153; unprediction.hpp:6 (+ the pure-MED inverse) */
int hoh_channelpredict_fastpath(hoh_ctx* ctx, const uint16_t* data, int w, int h, int depth, uint16_t* out);
int hoh_channelpredict_section(hoh_ctx* ctx, const uint16_t* data, int w, int h, int depth, int x_tiles,
                               int y_tiles, int x, int y, uint16_t predictor, uint16_t* out,
                               size_t out_cap, size_t* out_count);
int hoh_channelpredict_all(hoh_ctx* ctx, const uint16_t* data, int w, int h, int depth, int x_tiles,
                           int y_tiles, const uint16_t* tile_map, uint16_t* out);
int hoh_unpredict_all(hoh_ctx* ctx, const uint16_t* resid, size_t n_resid, int w, int h, int depth,
                      int x_tiles, int y_tiles, const uint16_t* tile_map, const uint16_t* backref,
                      uint16_t* out);
int hoh_unpredict_fastpath(hoh_ctx* ctx, const uint16_t* resid, size_t n_resid, int w, int h, int depth,
                           const uint16_t* backref, uint16_t* out);
/* lz.hpp:6 — one tile, host pointers.  lz_symbols receives *lz_size <= lz_cap bytes; nukemap (size/3
 * bytes) is OR-ed like the reference does (the caller zeroes it, choh.cpp:118-121). */
int hoh_find_lz_rgb(hoh_ctx* ctx, const uint8_t* source, size_t size, int width, int height, uint8_t* lz_symbols,
                    size_t lz_cap, uint8_t* nukemap, int distance, int break_even_bonus, size_t* lz_size);

/* layer_encode.hpp:126-272 for one plane */
int hoh_predictor_search(hoh_ctx* ctx, const uint16_t* plane, int w, int h, int depth, int mode,
                         uint16_t* tile_map, uint8_t* index_list, uint16_t* final_resid);

#ifdef __cplusplus
}
#endif
#endif /* HOHGPU_H */
