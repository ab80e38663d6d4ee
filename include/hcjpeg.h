/*
 * hcjpeg.h — C ABI of libhcjpeg: a B200-native (sm_100a) baseline-JPEG decode / encode path that is a
 * drop-in for the software model of hardcamls/video-coding (jpeg/model/src, common/src).
 *
 * The reference has no FFI of its own (it is 100 % OCaml); the entry points below are what thin OCaml
 * `external` stubs bind so that `Hardcaml_jpeg_model.Decoder` / `.Encoder` can run on the GPU.  Each
 * entry point cites the reference interface (file:line, relative to the reference root) it replaces.
 * The matching stubs are in video-coding_b200/ocaml/ and described in INTEGRATION.md.
 *
 * Conventions: plain C, no exceptions across the boundary, the library never keeps a caller pointer
 * after a call returns.  Every function returns an hcj_status (0 = ok).  Batched calls also fill a
 * per-image status array: a bad image never poisons the rest of the batch.  There is NO CPU fallback:
 * without a CUDA device every compute entry point returns HCJ_ERR_CUDA_*.
 */
#ifndef HCJPEG_H
#define HCJPEG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HCJ_VERSION 100 /* 0.1.0 */

/* ---- status codes: one per exception the model can raise, plus stated extensions ------------- */
typedef enum hcj_status {
  HCJ_OK = 0,
  HCJ_ERR_UNSUPPORTED_MARKER = -1,   /* decoder.ml:67  "unsupported marker code" */
  HCJ_ERR_NO_DC_CODE = -2,           /* decoder.ml:92  "Can't find dc code" */
  HCJ_ERR_NO_AC_CODE = -3,           /* decoder.ml:101 "Can't find ac code" */
  HCJ_ERR_COEF_INDEX = -4,           /* decoder.ml:136 "coefficient index out of range:" */
  HCJ_ERR_NO_COMPONENT = -5,         /* decoder.ml:228 "unable to find component identifier" */
  HCJ_ERR_NO_QUANT_TABLE = -6,       /* decoder.ml:234 "unable to find quantisation table" */
  HCJ_ERR_NO_HUFFMAN_TABLE = -7,     /* decoder.ml:243 "unable to find huffman table" */
  HCJ_ERR_NO_FRAME_OR_SCAN = -8,     /* decoder.ml:291 "From start of frame or start of scan marker" */
  HCJ_ERR_BITS_OUT_OF_BOUNDS = -9,   /* common/src/bitstream_reader.ml:32 "Bitstream_reader out of bounds" */
  HCJ_ERR_PLANE_BOUNDS = -10,        /* common/src/plane.ml:47-59 "[Plane.get/set] out of bounds" */
  HCJ_ERR_FRAME_INFER = -11,         /* common/src/frame.ml:44,55 chroma planes mismatch / cannot infer */
  HCJ_ERR_NEED_3_COMPONENTS = -12,   /* decoder.ml:415-420 get_yuv_frame needs components.(1), .(2) */
  HCJ_ERR_ENCODER_PARAMS = -13,      /* encoder.ml:274-282 "Failed to find identifier", bin/model.ml:76-82 */
  /* stated extensions, and inputs on which the model does not terminate */
  HCJ_ERR_NO_TERMINATOR = -20,       /* decoder.ml:261-281 loops forever when no marker follows the scan */
  HCJ_ERR_RESTART_COUNT = -21,       /* restart extension: number of RSTn != ceil(MCUs / Ri) - 1 */
  HCJ_ERR_UNSUPPORTED_GEOMETRY = -22,/* >4 scan components, sampling factor 0 or >4, >10 blocks/MCU, DC category >15, Pq>1 */
  HCJ_ERR_DC_RANGE = -23,            /* an absolute DC value does not fit the int16 coefficient store */
  HCJ_ERR_TRUNCATED = -24,           /* decoder.ml:24-29 find_marker spins forever on a truncated header */
  HCJ_ERR_BAD_HUFFMAN_TABLE = -25,   /* tables.ml:497-499 array index out of bounds (over-subscribed DHT) */
  HCJ_ERR_BUFFER_TOO_SMALL = -30,
  HCJ_ERR_INVALID_ARG = -31,
  HCJ_ERR_OUT_OF_MEMORY = -32,
  HCJ_ERR_CUDA = -1000               /* -1000 - cudaError_t */
} hcj_status;

const char *hcj_strerror(int status);
int hcj_version(void);

/* ---- Decoder.Header (decoder.mli:5-21, decoder.ml:5-71; Markers, markers.ml) ------------------ */
#define HCJ_MAX_COMPONENTS 4
#define HCJ_MAX_TABLE_SEGMENTS 64

typedef struct hcj_component { /* Markers.Component.t, markers.ml:6-13 */
  int identifier, horizontal_sampling_factor, vertical_sampling_factor, quantization_table_identifier;
} hcj_component;

typedef struct hcj_scan_component { /* Markers.Scan_component.t, markers.ml:75-82 */
  int selector, dc_coef_selector, ac_coef_selector;
} hcj_scan_component;

typedef struct hcj_dqt { /* Markers.Dqt.t, markers.ml:153-160 */
  int length, element_precision, table_identifier;
  int elements[64]; /* file (zig-zag) order */
} hcj_dqt;

typedef struct hcj_dht { /* Markers.Dht.t, markers.ml:200-208 */
  int length, table_class, destination_identifier;
  int lengths[16];
  int nvalues;
  uint8_t values[256];
} hcj_dht;

typedef struct hcj_header { /* Decoder.Header.t, decoder.ml:6-13 */
  int has_frame; /* frame : Sof.t option */
  int sof_length, sample_precision, width, height, number_of_components;
  hcj_component components[HCJ_MAX_COMPONENTS];
  int has_scan; /* scan : Sos.t option */
  int sos_length, number_of_image_components;
  hcj_scan_component scan_components[HCJ_MAX_COMPONENTS];
  int start_of_predictor_selection, end_of_predictor_selection;
  int successive_approximation_bit_high, successive_approximation_bit_low;
  int has_restart_interval; /* restart_interval : Dri.t option */
  int dri_length, restart_interval;
  int n_quant_tables; /* list order: most recently parsed first (decoder.ml:51) */
  hcj_dqt quant_tables[HCJ_MAX_TABLE_SEGMENTS];
  int n_huffman_tables; /* likewise (decoder.ml:55) */
  hcj_dht huffman_tables[HCJ_MAX_TABLE_SEGMENTS];
  int64_t scan_byte_pos; /* Bits.bit_pos / 8 after the SOS header: first entropy-coded byte */
} hcj_header;

/* Decoder.Header.decode : Bits.t -> Header.t (decoder.ml:37-70).  Host only. */
int hcj_header_decode(const uint8_t *jpeg, size_t len, hcj_header *out);
/* The same with HCJ_FLAG_* (below): HCJ_FLAG_T81_TABLES reads every table of a DQT / DHT segment. */
int hcj_header_decode_ex(const uint8_t *jpeg, size_t len, unsigned flags, hcj_header *out);

/* Geometry fixed by Decoder.init (decoder.ml:304-345) and decode_seq (:374-383).  Host only. */
typedef struct hcj_frame_info {
  int width, height, ncomp;
  int chroma; /* 420 / 422 / 444 as inferred by Frame.of_planes (frame.ml:42-61); 0 if not a YUV frame */
  int hs[HCJ_MAX_COMPONENTS], vs[HCJ_MAX_COMPONENTS];
  int decoded_width[HCJ_MAX_COMPONENTS], decoded_height[HCJ_MAX_COMPONENTS]; /* padded planes */
  int actual_width[HCJ_MAX_COMPONENTS], actual_height[HCJ_MAX_COMPONENTS];   /* cropped planes */
  int mcus_wide, mcus_high, blocks_per_mcu;
  int64_t nblocks;
  int restart_interval; /* 0 when absent */
  size_t yuv_bytes;     /* Frame.output size: cropped planar Y,U,V (0 if chroma == 0) */
  size_t planes_bytes;  /* get_decoded_planes: padded planes, scan order */
  size_t rgb_bytes;     /* width*height*3 (0 if chroma == 0) */
} hcj_frame_info;

int hcj_frame_info_get(const uint8_t *jpeg, size_t len, hcj_frame_info *out); /* flags = HCJ_FLAG_DEFAULT */
int hcj_frame_info_get_ex(const uint8_t *jpeg, size_t len, unsigned flags, hcj_frame_info *out);

/* ---- context: one per GPU (the model's `Decoder.t` / `Encoder.t` values own no device state) -- */
typedef struct hcj_ctx hcj_ctx;

/* `cuda_stream` is a cudaStream_t (or NULL for a private stream); all work of this context is issued on it. */
int hcj_ctx_create(int device, void *cuda_stream, hcj_ctx **out);
void hcj_ctx_destroy(hcj_ctx *ctx);
int hcj_ctx_synchronize(hcj_ctx *ctx);
/* Pinned host memory for zero-staging transfers (callers may also pass ordinary memory everywhere). */
void *hcj_host_alloc(size_t bytes);
void hcj_host_free(void *p);

/* ---- decode --------------------------------------------------------------------------------- */
typedef enum hcj_out_mode {
  HCJ_OUT_YUV = 0,    /* Decoder.get_yuv_frame -> Frame.output: cropped planar Y,U,V (decoder.ml:403-420, frame.ml:66-70) */
  HCJ_OUT_PLANES = 1, /* Decoder.get_decoded_planes: padded planes in scan order (decoder.ml:399-401) */
  HCJ_OUT_RGB24 = 2,  /* extension: Planar_444 up-sampling (tools/src/planar_444.ml:25-33,82-103) + stated YCbCr->RGB */
  HCJ_OUT_YUV444 = 3  /* `oyuv convert` to 4:4:4 on the device: Planar_444.convert_from_420 / convert_from_422
                         (tools/src/planar_444.ml:52-61,122-131) of the cropped frame, planar Y,U,V of width*height
                         bytes each (hcj_frame_info.rgb_bytes in total) */
} hcj_out_mode;

#define HCJ_FLAG_RESTART_EXT 1u /* honour DRI / RSTn (T.81 semantics).  Without it: pure model semantics (decoder.ml:261-281) */
/* Stated extension for files the model's parser cannot read (markers.ml:162-168,210-220 take ONE table per DQT / DHT
 * segment and then hunt for the next FF): every table of a segment is read, parsing continues at the end of the
 * segment, and 0xFF fill bytes in front of a marker code are skipped (T.81 B.1.1.2, B.2.4.1, B.2.4.2).  Files the
 * model reads correctly decode identically with and without it. */
#define HCJ_FLAG_T81_TABLES 2u
/* Stated extension (the model has no scaled decode): decode at 1/2, 1/4 or 1/8 size, like libjpeg's scale_num /
 * scale_denom (and Pillow's Image.draft).  Every block of every component is reconstructed straight to k x k samples,
 * k = 8 / s, with libjpeg's reduced inverse DCTs (jidctred.c: jpeg_idct_4x4, _2x2, _1x1) on the dequantised
 * coefficients (coefficient x quant entry, natural order, absolute DC), in exact integer arithmetic, output
 * clamp(x + 128, 0, 255).  Block (bx, by) of component c lands at (bx k, by k) of a padded plane of
 * decoded_width[c] / s x decoded_height[c] / s.  The frame is then the frame of W' = ceil(width / s) x
 * H' = ceil(height / s) with the same sampling factors (libjpeg's output size): hcj_frame_info reports width W',
 * height H', actual_* of that frame, the scaled padded planes and yuv_bytes / planes_bytes / rgb_bytes of those
 * sizes, while mcus_*, blocks_per_mcu, nblocks and restart_interval keep describing the coded blocks.  Every output
 * mode works on the scaled planes exactly as on any frame of that size; the coefficient taps are not scaled.
 * Honoured by hcj_frame_info_get_ex, hcj_decode_batch(_multi), hcj_decode_a_frame, hcj_decode_stream and
 * hcj_batch_create; hcj_header_decode_ex ignores it.  s = 1 (no bit set) is the ordinary decode. */
#define HCJ_FLAG_SCALE_1_2 0x10u
#define HCJ_FLAG_SCALE_1_4 0x20u
#define HCJ_FLAG_SCALE_1_8 0x30u
#define HCJ_FLAG_SCALE_MASK 0x30u
/* Stated extension (the model reconstructs with Chen-Wang and Planar_444): reconstruct samples as libjpeg-turbo's default
 * decompressor does (dct_method JDCT_ISLOW, do_fancy_upsampling TRUE; its C code paths are the specification), so that
 * RGB24 equals what Pillow, OpenCV and torchvision's CPU decoder give.
 *  - Every block of every component, in every output mode: jidctint.c jpeg_idct_islow on the dequantised coefficients
 *    (coefficient x quant entry, natural order, absolute DC), columns first, 64-bit intermediates, column-pass results
 *    truncated to 32 bits, row pass descaled by 18, then libjpeg's range-limit table with its wrap:
 *    clamp(((v + 512) & 1023) - 512 + 128, 0, 255).
 *  - HCJ_OUT_RGB24 / HCJ_OUT_YUV444: jdsample.c up-sampling of each component's real plane, ceil(W h_c / h_max) x
 *    ceil(H v_c / v_max) samples, by (h_max / h_c, v_max / v_c): (1, 1) copy; (2, 1) / (2, 2) / (1, 2) the fancy
 *    (triangle) filters h2v1 / h2v2 / h1v2, edges replicated, (2, 1) and (2, 2) plain replication when the real plane is
 *    at most 2 samples wide; any other integral ratio replication (int_upsample); a non-integral ratio is
 *    HCJ_ERR_UNSUPPORTED_GEOMETRY.  Cropped to W x H; colour as without the flag (the formula is jdcolor.c's).
 *    RGB24 equals Image.open(f).convert("RGB"), YUV444 Image.draft("YCbCr", size).
 *  - HCJ_OUT_YUV / HCJ_OUT_PLANES keep their layout and the model's crop rules, with islow samples.
 *  - hcj_frame_info is unchanged except that a 3-component frame with chroma 0 but integral ratios (4:4:0, 4:1:1)
 *    reports rgb_bytes = W H 3 and decodes to RGB24 / YUV444.  4-component frames give HCJ_ERR_UNSUPPORTED_GEOMETRY in
 *    RGB24 / YUV444 (libjpeg would take them as CMYK / YCCK); fewer than 3 components keep HCJ_ERR_NEED_3_COMPONENTS.
 *  - Honoured by hcj_frame_info_get_ex, hcj_decode_batch(_multi), hcj_decode_a_frame, hcj_decode_stream and
 *    hcj_batch_create; hcj_header_decode_ex and the debug taps (coefficients, entropy, block log, hcj_idct_blocks)
 *    ignore it.  Together with an HCJ_FLAG_SCALE_* bit it is HCJ_ERR_INVALID_ARG.
 * libjpeg-turbo's x86 SIMD IDCT works in 16-bit lanes and differs from its C code on blocks whose dequantised
 * coefficients do not fit 16 bits; this flag follows the C code there. */
#define HCJ_FLAG_LIBJPEG 0x40u
#define HCJ_FLAG_DEFAULT HCJ_FLAG_RESTART_EXT

/* Decoder.decode_a_frame (decoder.ml:422-427) for n independent images; host buffers in and out.
 * out[i] must hold at least the size hcj_frame_info_get reports for `mode`.  Returns the first
 * non-image error (CUDA, arguments); per-image results are in status[i]. */
int hcj_decode_batch(hcj_ctx *ctx, const uint8_t *const *jpeg, const size_t *len, int n, int mode, unsigned flags,
                     uint8_t *const *out, const size_t *out_capacity, int *status);

/* One process, several GPUs (the model's callers are single processes: jpeg/bin/model.ml:29-44).  Images are
 * independent (decoder.ml:422-427), so context k - one per device, all distinct - decodes the contiguous index range
 * hcj_shard_range(n, k, nctx) on its own host thread with its own streams; no data moves between devices.  Arguments
 * and results as hcj_decode_batch; returns the first failing context's code. */
int hcj_decode_batch_multi(hcj_ctx *const *ctx, int nctx, const uint8_t *const *jpeg, const size_t *len, int n, int mode,
                           unsigned flags, uint8_t *const *out, const size_t *out_capacity, int *status);
/* [*lo, *hi) = the batch indices part `part` of `nparts` handles: floor(n part / nparts) .. floor(n (part + 1) / nparts). */
void hcj_shard_range(int n, int part, int nparts, int *lo, int *hi);
int hcj_device_count(void); /* CUDA devices visible to the process (0 without a driver) */

/* Decoder.decode_a_frame (decoder.ml:422-427) for one image: a batch of one; returns the image's status. */
int hcj_decode_a_frame(hcj_ctx *ctx, const uint8_t *jpeg, size_t len, int mode, unsigned flags, uint8_t *out, size_t out_capacity);

/* Motion JPEG (jpeg/README.md:33 lists it as the model's next step: "just testing processing of multiple frames"):
 * a stream of whole JPEG files back to back.  hcj_mjpeg_split finds the frames (host only; pass offsets = NULL to
 * count them); hcj_decode_stream decodes all of them like hcj_decode_batch (files up, kernels and frames down
 * overlapped chunk by chunk) into one buffer: frame i at out + out_offsets[i], out_offsets[nframes] = bytes used
 * (each frame starts at a 256-byte boundary; out_offsets needs capacity + 1 entries). */
int hcj_mjpeg_split(const uint8_t *stream, size_t len, size_t *offsets, size_t *lengths, int capacity, int *nframes);
int hcj_decode_stream(hcj_ctx *ctx, const uint8_t *stream, size_t len, int mode, unsigned flags, uint8_t *out,
                      size_t out_capacity, size_t *out_offsets, int *status, int capacity, int *nframes);

/* The same in three steps, for pipelines that keep data resident in HBM. */
typedef struct hcj_batch hcj_batch;
/* Header.decode + init for every image, then upload (H2D) of the compressed bytes and tables.
 * n <= HCJ_MAX_BATCH (the image index is a CUDA grid dimension); larger jobs are split by the caller. */
#define HCJ_MAX_BATCH 65535
int hcj_batch_create(hcj_ctx *ctx, const uint8_t *const *jpeg, const size_t *len, int n, int mode, unsigned flags,
                     int *status, hcj_batch **out);
/* Decoder.decode for the whole batch: kernels only, asynchronous on the context's stream. */
int hcj_batch_decode(hcj_ctx *ctx, hcj_batch *b);
/* D2H of the outputs and of the per-image statuses; synchronises. */
int hcj_batch_fetch(hcj_ctx *ctx, hcj_batch *b, uint8_t *const *out, const size_t *out_capacity, int *status);
/* Device pointer / size of image i's output (valid until the batch is destroyed). */
int hcj_batch_device_output(hcj_batch *b, int i, void **dptr, size_t *bytes);
int hcj_batch_count_kernels(const hcj_batch *b); /* kernels hcj_batch_decode launches */
void hcj_batch_destroy(hcj_ctx *ctx, hcj_batch *b);

/* Debug taps mirroring Decoder.For_testing (decoder.mli:62-85). */
/* Component.coefs for every block of image i in decode_seq order: int16, zig-zag, DC *resolved* (absolute). */
int hcj_batch_fetch_coefficients(hcj_ctx *ctx, hcj_batch *b, int i, int16_t *coefs, size_t capacity_blocks);
/* For_testing.extract_entropy_coded_bits (decoder.ml:261-281): destuffed entropy-coded segment of image i. */
int hcj_batch_fetch_entropy(hcj_ctx *ctx, hcj_batch *b, int i, uint8_t *out, size_t capacity, size_t *len);
/* `model decode log` (jpeg/bin/model.ml:46-68): Decoder.Component.Summary (decoder.ml:189-203) of blocks
 * [first_block, first_block + count) of image i in decode_seq order, computed on the device from the decoded
 * coefficient blocks with the model's 64-bit arithmetic. */
typedef struct hcj_block_log {
  int32_t x, y;        /* origin of the block in its component's padded plane (decoder.ml:353-360) */
  int32_t dc_pred;     /* the component's predictor after the block */
  int32_t component;   /* scan component index; its identifier is hcj_header.scan_components[component].selector */
  int16_t coefs[64];   /* zig-zag order, coefs[0] = the DC differential as decoded (Component.coefs) */
  int32_t dequant[64]; /* natural order (Component.dequant) */
  int32_t idct[64];    /* Dct.Chen.inverse_8x8 of dequant, before clipping (Component.idct) */
  uint8_t recon[64];   /* clip + level shift (Component.recon) */
} hcj_block_log;
int hcj_batch_fetch_block_log(hcj_ctx *ctx, hcj_batch *b, int i, size_t first_block, size_t count, hcj_block_log *out);
/* dequantize + Dct.Chen.inverse_8x8 + recon (decoder.ml:142-149,213-224; dct.ml:100-107) on caller-provided
 * zig-zag blocks (DC absolute): out = nblocks*64 reconstructed samples, block-major (Component.recon). */
int hcj_idct_blocks(hcj_ctx *ctx, const int16_t *coefs, size_t nblocks, const uint16_t quant_table[64], uint8_t *out);

/* ---- encode --------------------------------------------------------------------------------- */
/* Encoder.encode_420 / encode_422 / encode_444 / encode_monochrome (encoder.ml:522-552) for n frames of identical
 * geometry.  yuv[i]: planar Y,U,V as Frame.input reads it (frame.ml:72-76).  chroma: 420/422/444, or 400 for
 * encode_monochrome (one plane of width * height bytes; like the model, the plane is copied into its padded
 * plane linearly, so a width that is not a multiple of 8 shears the image: Plane.blit, plane.ml:20).
 * restart_interval 0 reproduces the model byte-for-byte; >0 is the stated DRI/RSTn extension.
 * out_len[i] is the length of frame i's file whether or not it fitted: with HCJ_ERR_BUFFER_TOO_SMALL in status[i] it is
 * the capacity a second call needs (hcj_encode_bound is the bound that never fails).
 * The frames go through the device in chunks (64 by default) on three streams - upload of the next chunk, kernels,
 * download of the previous chunk's files - so with pinned frame buffers (hcj_host_alloc) the call runs at the link's
 * host-to-device rate; frames that lie back to back in host memory go up as one copy per chunk. */
int hcj_encode_batch(hcj_ctx *ctx, const uint8_t *const *yuv, int n, int width, int height, int chroma, int quality,
                     int restart_interval, uint8_t *const *out, const size_t *out_capacity, size_t *out_len,
                     int *status);
/* The same over several GPUs from one process: context k encodes frames hcj_shard_range(n, k, nctx) (see hcj_decode_batch_multi). */
int hcj_encode_batch_multi(hcj_ctx *const *ctx, int nctx, const uint8_t *const *yuv, int n, int width, int height, int chroma,
                           int quality, int restart_interval, uint8_t *const *out, const size_t *out_capacity, size_t *out_len,
                           int *status);
/* The same for RGB24 frames (extension; the model's encoder takes planar frames only): rgb[i] is width*height*3 bytes,
 * R, G, B interleaved, rows top to bottom, no padding - the layout HCJ_OUT_RGB24 decodes to.  On the device, every frame
 * is taken to the planar frame of `chroma` that hcj_encode_batch would be given, in two steps:
 *   1. JFIF full-range forward conversion, libjpeg's jccolor.c in 16-bit fixed point with arithmetic shifts (every
 *      result lies in [0, 255]; each channel is within 1 of OpenCV's COLOR_RGB2YCrCb and Pillow's "YCbCr"):
 *        Y  = ( 19595 R + 38470 G +  7471 B + 32768)               >> 16
 *        Cb = (-11059 R - 21709 G + 32768 B + (128 << 16) + 32767) >> 16
 *        Cr = ( 32768 R - 27439 G -  5329 B + (128 << 16) + 32767) >> 16
 *   2. chroma 420 / 422: Planar_444.convert_to_420 / convert_to_422 (tools/src/planar_444.ml:18-23,68-80) of the
 *      rounded 4:4:4 Cb / Cr planes: planes of floor(width/2) x floor(height/2) (or x height), the average of each 2x2
 *      (2x1) group with rounding, an odd last column or row dropped.  444 keeps the planes, 400 keeps Y only.
 * That frame is then encoded exactly as hcj_encode_batch encodes it: the files are byte-identical, statuses (for
 * example HCJ_ERR_PLANE_BOUNDS), out_len, HCJ_ERR_BUFFER_TOO_SMALL, hcj_encode_bound and hcj_encode_last_device_ms
 * (which includes the conversion) behave the same.  Without flags the frames are in host memory and go up chunk by
 * chunk like planar frames (3 bytes a pixel instead of 1.5 for 4:2:0).  flags: HCJ_ENC_SRC_DEVICE, or 0; other bits
 * are HCJ_ERR_INVALID_ARG. */
#define HCJ_ENC_SRC_DEVICE 1u /* rgb[i] are device pointers on the context's device */
/* With HCJ_ENC_SRC_DEVICE nothing is uploaded: the conversion reads the caller's buffers, on the context's stream (the
 * one passed to hcj_ctx_create), so work the caller enqueued on that stream before the call is ordered before the
 * reads; work on other streams must be synchronised by the caller.  Every pointer is checked before any work is
 * enqueued: one that is not device (or managed) memory of the context's device makes the call return
 * HCJ_ERR_INVALID_ARG with nothing written.  As everywhere, nothing reads caller memory after the call returns. */
int hcj_encode_rgb_batch(hcj_ctx *ctx, const uint8_t *const *rgb, int n, int width, int height, int chroma, int quality,
                         int restart_interval, unsigned flags, uint8_t *const *out, const size_t *out_capacity,
                         size_t *out_len, int *status);
/* The conversion alone (steps 1-2), one frame, host buffers: the planar frame hcj_encode_rgb_batch encodes
 * (width*height bytes of Y, then Cb and Cr; Y only for 400).  HCJ_ERR_BUFFER_TOO_SMALL if dst_capacity is less. */
int hcj_rgb_to_yuv(hcj_ctx *ctx, const uint8_t *rgb, int width, int height, int chroma, uint8_t *dst, size_t dst_capacity);
size_t hcj_encode_bound(int width, int height, int chroma); /* worst-case bytes of one encoded frame */
int hcj_encode_count_kernels(void); /* kernels one hcj_encode_batch launches */
/* Encoder.write_headers (encoder.ml:371-418).  Host only. */
int hcj_write_headers(int width, int height, int chroma, int quality, int restart_interval, uint8_t *out,
                      size_t capacity, size_t *len);
/* Block.quant (encoder.ml:56-66): quantised zig-zag blocks of one frame in encode_seq order. */
int hcj_encode_quantized(hcj_ctx *ctx, const uint8_t *yuv, int width, int height, int chroma, int quality,
                         int16_t *quant, size_t capacity_blocks);

/* `model encode log [-verbose]` (jpeg/bin/model.ml:108-142): Encoder.Block.t (encoder.ml:56-66) of blocks
 * [first_block, first_block + count) of one frame in encode_seq order (encoder.ml:476-505), computed on the device
 * with the model's arithmetic; the reconstruction (Block.decoded, encoder.ml:37-55,110-125) is always filled. */
typedef struct hcj_encoder_block {
  int32_t x_pos, y_pos;      /* origin of the block in its component's padded plane (encoder.ml:486-489) */
  int32_t dc_pred;           /* the component's predictor after the block (= quant[0]) */
  int32_t component;         /* scan component index */
  int32_t nrle;              /* entries of rle_run / rle_value in use */
  uint8_t input_pixels[64];  /* Block.input_pixels (before the level shift) */
  int32_t fdct[64];          /* Dct.Chen.forward_8x8 of the level-shifted block, natural order (4 x the orthonormal DCT) */
  int16_t quant[64];         /* zig-zag order, quant[0] absolute */
  int16_t rle_run[64];       /* Block.rle (encoder.ml:127-141): entry 0 = { run = 0; value = DC differential }, */
  int16_t rle_value[64];     /*   then the AC pairs; position 63 is always emitted (value 0 = end of block) */
  int32_t dequant[64];       /* Decoded.dequant, natural order */
  int32_t idct[64];          /* Decoded.idct */
  uint8_t recon[64];         /* Decoded.recon = clamp (idct + 128) */
  uint8_t error[64];         /* Decoded.error = |recon - input_pixels| */
} hcj_encoder_block;
int hcj_encode_block_log(hcj_ctx *ctx, const uint8_t *yuv, int width, int height, int chroma, int quality, int restart_interval,
                         size_t first_block, size_t count, hcj_encoder_block *out);

/* Scalar helpers the reference exposes for its tests, evaluated on the host by the same functions the kernels call:
 * Decoder.For_testing.mag (decoder.mli:64-65, decoder.ml:73-79: signed value of `cat` magnitude bits `code`),
 * Encoder.size and Encoder.magnitude (encoder.ml:143-147; pinned by test_encode_codewords.ml). */
/* Quant_tables.scale luma / chroma (quant_tables.ml:139-147; test_quant_tables.ml) and one entry of
 * Tables.Encoder.dc_table / ac_table for the default specifications (tables.ml:504-545; test_tables.ml):
 * table 0 dc_luma, 1 dc_chroma, 2 ac_luma, 3 ac_chroma; *length = 0 when the table has no such code. */
int hcj_quant_scale(int chroma_table, int quality, uint16_t out[64]);
int hcj_encoder_code(int table, int run, int size, int *bits, int *length);
int hcj_mag(int cat, int code);
int hcj_size(int value);
int hcj_magnitude(int size, int value);

/* ---- on-device frame tools (tools/src) ------------------------------------------------------- */
/* Ocompare.square_error / max_difference per plane (tools/src/ocompare.ml:8-52) of two host frames. */
int hcj_compare_planes(hcj_ctx *ctx, const uint8_t *a, const uint8_t *b, size_t n, int64_t *square_error,
                       int *max_difference);
/* The same with Ocompare.total_difference (tools/src/ocompare.ml:20-30): what `oyuv compare mean-difference` divides. */
int hcj_compare_planes_ex(hcj_ctx *ctx, const uint8_t *a, const uint8_t *b, size_t n, int64_t *square_error,
                          int *max_difference, int64_t *total_difference);

/* `oyuv convert` on the device (tools/src/oconv.ml:111-133): a planar frame of `chroma` (420 / 422 / 444, planes as
 * Frame.create lays them out) is taken to 4:4:4 (Planar_444.convert_from_420 / _422), cropped to dst_width x dst_height
 * at (x_off, y_off) with the edge clamp of Yuv.crop (yuv.ml:43-62), and sub-sampled to `dst_chroma`
 * (Planar_444.convert_to_420 / _422).  Host buffers in and out. */
int hcj_yuv_convert(hcj_ctx *ctx, const uint8_t *src, int width, int height, int chroma, int x_off, int y_off, uint8_t *dst,
                    int dst_width, int dst_height, int dst_chroma, size_t dst_capacity);

/* `oyuv compare` for a whole decoded batch, on the device: Ocompare.square_error / total_difference / max_difference
 * (tools/src/ocompare.ml:8-46) per plane between image i's output resident in HBM (after hcj_batch_decode) and the
 * reference frame ref[i] in host memory, which has the layout and size of the batch's output mode.  Planes: Y,U,V
 * for HCJ_OUT_YUV / HCJ_OUT_YUV444, one per scan component for HCJ_OUT_PLANES, one (all bytes) for HCJ_OUT_RGB24.
 * mean_square_error = square_error / samples; psnr = 10 log10(255^2 / mean_square_error) (ocompare.ml:48-56). */
typedef struct hcj_plane_metrics {
  int status;                  /* the image's status; metrics are zero unless it is HCJ_OK */
  int max_difference[4];
  int64_t square_error[4];
  int64_t total_difference[4];
  int64_t samples[4];          /* width * height of the plane; 0 = no such plane */
} hcj_plane_metrics;
int hcj_batch_compare(hcj_ctx *ctx, hcj_batch *b, const uint8_t *const *ref, const size_t *ref_len, hcj_plane_metrics *out);

/* ---- timing helpers for benchmarks --------------------------------------------------------------- */
/* One decode pass with a CUDA event between consecutive stages (on the context's stream); fills
 * ms[0..*nstages) in launch order and synchronises.  Stage names: hcj_decode_stage_name(i). */
int hcj_batch_decode_stages(hcj_ctx *ctx, hcj_batch *b, float *ms, int capacity, int *nstages);
const char *hcj_decode_stage_name(int i);
/* Kernel time of the latest hcj_encode_batch on this context, summed over its chunks (CUDA events around the two
 * kernel phases of every chunk; the host's sizing step between them is not device work). */
int hcj_encode_last_device_ms(hcj_ctx *ctx, float *ms);
/* ms between two points on the context's stream */
int hcj_timer_start(hcj_ctx *ctx);
int hcj_timer_stop(hcj_ctx *ctx, float *ms); /* synchronises */

#ifdef __cplusplus
}
#endif
#endif /* HCJPEG_H */
