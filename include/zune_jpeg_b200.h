/*
 * zune_jpeg_b200.h -- C ABI of the B200-native pixel-reconstruction path of
 * etemesi254/zune-jpeg (snapshot 0.2.0).
 *
 * The reference has no FFI; its boundary for this path is the crate-private
 *
 *   worker::post_process(coeff:&[&[i16];3], component_data:&[Components], idct_func, color_convert_16,
 *                        input_colorspace, output_colorspace, output:&mut [u8], width)   (src/worker.rs:32-41)
 *
 * called once per MCU-row strip from src/mcu.rs:356-368 (baseline) and src/mcu_prog.rs:205-233
 * (progressive).  A strip is far too small a GPU launch, so this ABI takes WHOLE-IMAGE coefficient planes
 * (the layout mcu_prog.rs:73-79 allocates, and that the concatenation of mcu.rs's per-strip buffers equals)
 * and performs every strip's post_process -- dequantise + IDCT + upsample + colour-convert + row de-padding --
 * for a batch of images in one call.  See INTEGRATION.md for the Rust `extern "C"` block that binds it.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns 0 (ZJ_OK) or a negative
 * zj_status and never unwinds; the caller owns every buffer; a call is thread-safe per (device, stream).
 * There is NO CPU fallback: without a CUDA device every compute entry point returns ZJ_ERR_NO_DEVICE.
 */
#ifndef ZUNE_JPEG_B200_H
#define ZUNE_JPEG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define ZJ_API __declspec(dllexport)
#else
#define ZJ_API __attribute__((visibility("default")))
#endif

/* ------------------------------------------------------------------ enums */

/* Ordinals of `ColorSpace` (src/misc.rs:88-106). */
typedef enum zj_colorspace {
    ZJ_CS_RGB = 0,
    ZJ_CS_GRAYSCALE = 1,
    ZJ_CS_YCBCR = 2,
    ZJ_CS_CMYK = 3,
    ZJ_CS_YCCK = 4,
    ZJ_CS_RGBA = 5,
    ZJ_CS_RGBX = 6
} zj_colorspace;

/* Which of the reference's two CPU code paths the output must be bit-identical to.
 * X86    = ZuneJpegOptions::use_unsafe == true on an AVX2+SSE4.1 host (the default, src/options.rs:31):
 *          AVX2 IDCT (src/idct/avx2.rs), SSE H upsampler (src/upsampler/sse.rs), scalar V, AVX2 HV
 *          (src/upsampler/avx2.rs, scalar below 500 samples), AVX2 RGB (src/color_convert/avx.rs).
 * SCALAR = use_unsafe == false or `--no-default-features`: src/idct/scalar.rs, src/upsampler/scalar.rs,
 *          src/color_convert/scalar.rs. */
typedef enum zj_variant { ZJ_VARIANT_X86 = 0, ZJ_VARIANT_SCALAR = 1, ZJ_VARIANT_SPEC = 2 } zj_variant;

/* ZJ_VARIANT_SPEC -- not in the reference: spec-correct output, none of its pixel-path quirks (DESIGN.md section 4.6).  The
 * output is a function of the coefficient planes, bit-exact:
 *   1. Samples: every block of every component goes through the X86 IDCT above (dequantise, rows then columns, the DC-only
 *      shortcut, clamp to [0, 255]); a component plane is the raster of its blocks.
 *   2. Sizes: luma is width x height; chroma is cw = ceil(width / hs) by ch = ceil(height / vs), (hs, vs) = comp[0]'s factors.
 *      Samples beyond these sizes (block padding) are never read: every neighbour index below is clamped to
 *      [0, ch-1] x [0, cw-1].
 *   3. Up-sampling (libjpeg jdsample.c, integer "fancy" forms), c[j][i] a chroma sample:
 *        none  C(y, x) = c[y][x]
 *        H     C(y, 2i) = (3c[y][i] + c[y][i-1] + 1) >> 2         C(y, 2i+1) = (3c[y][i] + c[y][i+1] + 2) >> 2
 *        V     C(2j, x) = (3c[j][x] + c[j-1][x] + 1) >> 2         C(2j+1, x) = (3c[j][x] + c[j+1][x] + 2) >> 2
 *        HV    s[i] = 3c[j][i] + c[j'][i], j' = j-1 for output row 2j and j+1 for row 2j+1 (indices of s clamped alike):
 *              C(., 2i) = (3s[i] + s[i-1] + 8) >> 4                C(., 2i+1) = (3s[i] + s[i+1] + 7) >> 4
 *      then cut to width x height.
 *   4. Colour (libjpeg jdcolor.c, 16-bit fixed point, arithmetic shifts), cb' = Cb - 128, cr' = Cr - 128:
 *        R = clamp(Y + ((91881 cr' + 32768) >> 16))
 *        G = clamp(Y + ((-22554 cb' - 46802 cr' + 32768) >> 16))
 *        B = clamp(Y + ((116130 cb' + 32768) >> 16))
 *   5. Output: RGB = R, G, B; RGBA and RGBX = R, G, B, 255; YCBCR = Y, Cb, Cr; GRAYSCALE = Y.  One-component input: GRAYSCALE = Y,
 *      RGB / RGBA / RGBX = Y, Y, Y (, 255).  Every other pair is ZJ_ERR_UNSUPPORTED.
 * Every byte of the width*height*nc output is written.  Every strip of the image is reconstructed (4:2:2 and 4:2:0: ceil(mcu_y/2)
 * strips), so the planes must cover them (ZJ_ERR_SHORT_PLANE otherwise, e.g. for planes of an as-written host stage that dropped
 * an odd last MCU row); none of the reference's panic rules applies.  Such an image cannot be cut into strip ranges: the rows of a
 * strip need chroma from its neighbours (zj_image_strip_range returns ZJ_ERR_UNSUPPORTED for any cut).  The host stage produces
 * it with zj_options.use_unsafe = ZJ_USE_SPEC_OUTPUT. */
enum { ZJ_USE_SPEC_OUTPUT = 2 };

/* ZJ_VARIANT_SPEC with ZJ_FLAG_ISLOW in zj_image.flags -- libjpeg-turbo-exact output (DESIGN.md section 4.6.1).  The statement
 * above with one alternative step 1; steps 2-5 stay as they are:
 *   1'. Samples: every block of every component goes through jpeg_idct_islow of libjpeg-turbo's jidctint.c, in 32-bit
 *       two's-complement arithmetic that wraps (as the X86 IDCT does), shifts arithmetic.  CONST_BITS 13, PASS1_BITS 2, the
 *       FIX_* constants 2446 3196 4433 6270 7373 9633 12299 15137 16069 16819 20995 25172; dequantise (coefficient x table
 *       entry); pass 1 down the columns, DESCALE(x, 11); pass 2 along the rows, DESCALE(x, 18); DESCALE(x, n) = (x + 2^(n-1)) >> n.
 *       The sample is range_limit[v & 1023]: v + 128 for v in [0, 127], 255 for [128, 511], 0 for [512, 895], v - 896 for
 *       [896, 1023].  A column whose coefficients in rows 1-7 are all zero takes jidctint.c's pass-1 shortcut: its 8 values are
 *       (DC x table entry) << 2.  (That equals the full pass unless the dequantised DC is 2^18 or more in magnitude, where the
 *       full pass would wrap.)  The pass-2 shortcut for rows whose AC is zero equals the full pass, so it is not part of the
 *       statement.  Whenever no intermediate leaves 32 bits -- every block an 8-bit JPEG encoder produces -- this equals
 *       jidctint.c with a 64-bit JLONG; with libjpeg-turbo's fancy up-sampling (step 3) and colour conversion (step 4) it is
 *       then the decode of libjpeg-turbo's default settings (JDCT_ISLOW, do_fancy_upsampling), i.e. Pillow's.
 * The flag is valid with ZJ_VARIANT_SPEC only (ZJ_ERR_INVALID_ARG otherwise).  The host stage produces such images with
 * zj_options.use_unsafe = ZJ_USE_LIBJPEG_OUTPUT: it decodes exactly as for ZJ_USE_SPEC_OUTPUT and sets the flag. */
enum { ZJ_USE_LIBJPEG_OUTPUT = 3 };

/* ZJ_VARIANT_SPEC | ZJ_FLAG_ISLOW with a scale k = (flags & ZJ_FLAG_SCALE_MASK) >> ZJ_FLAG_SCALE_SHIFT in {1, 2, 3} -- libjpeg-turbo's
 * DCT-scaled decode to 1/d, d = 2^k (DESIGN.md section 4.6.2): what Pillow's Image.draft(mode, size) gives.  s0 = 8 / d; (hmax, vmax)
 * = comp[0]'s factors, (h_z, v_z) = component z's.
 *   1''. Block size per component (jdmaster.c): ss_z = s0, doubled while ss_z < 8, (hmax s0) mod (2 h_z ss_z) = 0 and (vmax s0) mod
 *       (2 v_z ss_z) = 0.  Luma gets s0; 4:2:0 chroma 2 s0; 4:4:4, 4:2:2 and 4:4:0 chroma s0.
 *   2''. Samples: every block of component z becomes ss_z x ss_z samples.  ss = 8: step 1'.  Otherwise jidctred.c, in the
 *       arithmetic of step 1' (32-bit two's complement that wraps, arithmetic shifts, CONST_BITS 13, PASS1_BITS 2, dequantise =
 *       coefficient x table entry, DESCALE and range_limit[v & 1023] as there):
 *       ss = 4 (jpeg_idct_4x4): pass 1 down columns 0-3 and 5-7 (column 4 is never used); a column whose coefficients in rows 1, 2,
 *         3, 5, 6, 7 are all zero gives 4 values (DC x q) << 2; otherwise, with z_r the dequantised row r,
 *           t0 = z_0 << 14, t2 = 15137 z_2 - 6270 z_6, t10 = t0 + t2, t12 = t0 - t2,
 *           a = -1730 z_7 + 11893 z_5 - 17799 z_3 + 8697 z_1, b = -4176 z_7 - 4926 z_5 + 7373 z_3 + 20995 z_1,
 *           values DESCALE(t10 + b, 12), DESCALE(t12 + a, 12), DESCALE(t12 - a, 12), DESCALE(t10 - b, 12).
 *         Pass 2 along each of the 4 rows w: a row whose w_1, w_2, w_3, w_5, w_6, w_7 are all zero gives 4 samples
 *         range_limit[DESCALE(w_0, 5)]; otherwise the same formulas on w (t0 = w_0 << 14) with DESCALE(., 19).
 *       ss = 2 (jpeg_idct_2x2): only rows and columns 0, 1, 3, 5, 7 are read.  Pass 1 down columns 0, 1, 3, 5, 7: a column whose rows
 *         1, 3, 5, 7 are zero gives 2 values (DC x q) << 2; otherwise t10 = z_0 << 15, t0 = -5906 z_7 + 6967 z_5 - 10426 z_3 +
 *         29692 z_1, values DESCALE(t10 + t0, 13), DESCALE(t10 - t0, 13).  Pass 2 along each of the 2 rows w: w_1, w_3, w_5, w_7 all
 *         zero gives range_limit[DESCALE(w_0, 5)] twice; otherwise the same formulas on w with DESCALE(., 20).
 *       ss = 1 (jpeg_idct_1x1): range_limit[DESCALE(DC x q, 3)].
 *       The zero tests read the coefficients (pass 1) and the pass-1 values (pass 2), as jidctred.c does.  Whenever no intermediate
 *       leaves 32 bits -- every block an 8-bit JPEG encoder produces -- this equals jidctred.c with a 64-bit JLONG.
 *   3''. Sizes: the output is W' x H' = ceil(width / d) x ceil(height / d); component z is dw_z = ceil(width h_z ss_z / (hmax 8)) by
 *       dh_z = ceil(height v_z ss_z / (vmax 8)) samples, and samples beyond these sizes are never read.
 *   4''. Up-sampling by (hmax s0 / (h_z ss_z), vmax s0 / (v_z ss_z)), fancy = (s0 > 1): (1, 1) none; (2, 1) step 3's H filter when
 *       fancy and dw_z > 2, else each sample twice; (1, 2) step 3's V filter when fancy, else each row twice.  Neighbour indices are
 *       clamped to [0, dh_z-1] x [0, dw_z-1]; the result is cut to W' x H'.
 *   5''. Steps 4 and 5 as they are, over W' x H' pixels: GRAYSCALE output is the luma plane.
 * A non-zero scale on any other image is ZJ_ERR_INVALID_ARG; k = 0 is the statement above.  Everything downstream of reconstruction
 * (zj_output_size, the consumers' shapes, rois, resizes) sees the W' x H' image.  The host stage produces such images with
 * zj_options.use_unsafe = ZJ_USE_LIBJPEG_OUTPUT | k << 4: it decodes exactly as for ZJ_USE_LIBJPEG_OUTPUT and sets the scale. */
#define ZJ_FLAG_SCALE_SHIFT 2
#define ZJ_FLAG_SCALE_MASK (3u << ZJ_FLAG_SCALE_SHIFT)

/* ZJ_VARIANT_SPEC (with or without ZJ_FLAG_ISLOW and a scale) with an orientation o = ((flags & ZJ_FLAG_ORIENT_MASK) >>
 * ZJ_FLAG_ORIENT_SHIFT) + 1 in {2, ..., 8} -- the EXIF orientation applied (DESIGN.md section 4.6.3): what Pillow 12.2's
 * ImageOps.exif_transpose gives.  The W' x H' image the statements above give (after any DCT scaling, as draft then
 * exif_transpose) goes through Pillow's Transpose for o, each pixel's nc bytes moving together:
 *   o = 2 FLIP_LEFT_RIGHT  out(X, Y) = in(W'-1-X, Y)          o = 5 TRANSPOSE   out(X, Y) = in(Y, X)
 *   o = 3 ROTATE_180       out(X, Y) = in(W'-1-X, H'-1-Y)     o = 6 ROTATE_270  out(X, Y) = in(Y, H'-1-X)
 *   o = 4 FLIP_TOP_BOTTOM  out(X, Y) = in(X, H'-1-Y)          o = 7 TRANSVERSE  out(X, Y) = in(W'-1-Y, H'-1-X)
 *                                                             o = 8 ROTATE_90   out(X, Y) = in(W'-1-Y, X)
 * The output is W' x H' for o = 2-4 and H' x W' for o = 5-8 (the same byte count).  Everything downstream of reconstruction
 * (zj_output_size, the consumers' shapes, rois -- given in the displayed frame -- and resizes) sees the oriented image.  The bits
 * are valid with ZJ_VARIANT_SPEC only (ZJ_ERR_INVALID_ARG otherwise); 0 is no transform.
 *
 * The host stage finds o (zj_decoder_orientation) the way Pillow 12.2's Image.getexif() does (PIL/Image.py, JpegImagePlugin.py
 * APP()), reading only the markers before the first SOS:
 *   - EXIF: the APP1 segments that start with "Exif\0\0" -- the first one's payload, with each later one's bytes after its 6-byte
 *     header appended, every leading "Exif\0\0" of the result stripped.  Nothing left: no EXIF.  Otherwise an 8-byte TIFF header
 *     ("II*\0" or "MM\0*" and IFD0's offset); a shorter or other header gives o = 1 and the XMP is not read (Pillow raises there).
 *   - IFD0: its entry count, then its 12-byte entries in order, up to the first one that cannot be read whole -- its 12 bytes, or
 *     the data it points at when its count x type size (types 1-13: 1 1 2 4 8 1 1 2 4 8 4 8 4 bytes) exceeds 4.  Entries of another
 *     type or of size 0 are skipped; a later entry of a tag replaces an earlier one.  IFD0's offset past the data: no entries.
 *   - Tag 0x0112 of type SHORT, LONG, SSHORT or SLONG: its first value, whatever the count (Pillow keeps the first value when the
 *     count is not 1).  Of any other type: a value that is not an orientation (Pillow compares a RATIONAL or FLOAT value with
 *     2-8; this does not).
 *   - XMP, only when IFD0 has no tag 0x0112: the last APP1 segment that starts with "http://ns.adobe.com/xap/1.0/\0"; the first
 *     match of tiff:Orientation(="|>)([0-9]) in it.
 *   Any value other than 2-8 means no transform, and so does a missing tag.  torchvision's decode_jpeg(apply_exif_orientation=True)
 *   reads the EXIF only (and a single SHORT); an XMP-only orientation is applied here, as Pillow applies it, and not there.  A bad
 *   EXIF never fails a decode.
 * With zj_options.use_unsafe = ZJ_USE_SPEC_OUTPUT, ZJ_USE_LIBJPEG_OUTPUT or ZJ_USE_LIBJPEG_OUTPUT | k << 4, ORed with
 * ZJ_USE_EXIF_ORIENTATION, the host stage decodes as without it and sets o in the images' flags. */
#define ZJ_FLAG_ORIENT_SHIFT 4
#define ZJ_FLAG_ORIENT_MASK (7u << ZJ_FLAG_ORIENT_SHIFT)
enum { ZJ_USE_EXIF_ORIENTATION = 0x100 };

typedef enum zj_status {
    ZJ_OK = 0,
    ZJ_ERR_INVALID_ARG = -1,     /* null pointer, bad enum, inconsistent descriptor                        */
    ZJ_ERR_UNSUPPORTED = -2,     /* sampling the reference rejects (decoder.rs:512-519, :609-646)          */
    ZJ_ERR_SHORT_PLANE = -3,     /* a coefficient plane is smaller than the strips it must feed            */
    ZJ_ERR_SHORT_OUTPUT = -4,    /* out_len[i] < width*height*out_components                               */
    ZJ_ERR_REF_PANIC = -5,       /* the reference panics on this geometry (tiny widths, see DESIGN.md)     */
    ZJ_ERR_NO_DEVICE = -6,       /* no CUDA device / bad ordinal -- there is no CPU fallback               */
    ZJ_ERR_CUDA = -7,            /* a CUDA runtime call failed; zj_gpu_last_cuda_error() has the text      */
    ZJ_ERR_OOM = -8,             /* device or pinned allocation failed                                     */
    ZJ_ERR_DECODE = -9           /* host front-end (headers/entropy) error; zj_decoder_error() has details */
} zj_status;

/* ------------------------------------------------------------ descriptors */

/* One image component as the path sees it: the fields of `Components` (src/components.rs:18-43) that
 * post_process reads, plus the coefficient plane. */
typedef struct zj_component {
    const int16_t *coeff;  /* whole-image plane: blocks in raster order, width_stride/8 blocks per block-row,
                              64 i16 per block in NATURAL (de-zigzagged, row-major) order -- what
                              bitstream.rs:343,359 / mcu_prog.rs:298,404-406 produce.  Host or device pointer
                              depending on the entry point.  May be NULL for components the output colourspace
                              does not need (worker.rs:59). */
    uint64_t n_i16;        /* number of i16 in the plane                                                    */
    int32_t qt[64];        /* quantisation table, natural order (headers.rs:533-543)                        */
    uint32_t h_samp;       /* Components::horizontal_sample                                                 */
    uint32_t v_samp;       /* Components::vertical_sample                                                   */
    uint32_t width_stride; /* Components::width_stride = h_samp * mcu_x * 8 (headers.rs:338)                */
    uint32_t reserved;
} zj_component;

#define ZJ_FLAG_PROGRESSIVE 1u /* strips come from mcu_prog.rs:188-233 (zip stops silently) instead of
                                  mcu.rs:225-369 (chunks.next().unwrap()) -- only matters when the
                                  over-allocated output runs out of strips, see DESIGN.md                   */
#define ZJ_FLAG_ISLOW 2u       /* not in the reference: ZJ_VARIANT_SPEC with libjpeg-turbo's islow IDCT as step 1
                                  (the statement is above, next to ZJ_VARIANT_SPEC's)                        */

typedef struct zj_image {
    uint32_t width, height; /* ImageInfo::width/height (decoder.rs:652-668)                                 */
    uint32_t n_comp;        /* 1 (GRAYSCALE in) or 3 (YCbCr in) = input_colorspace.num_components()         */
    uint32_t out_cs;        /* zj_colorspace: ZuneJpegOptions::out_colorspace                               */
    uint32_t variant;       /* zj_variant                                                                   */
    uint32_t flags;         /* ZJ_FLAG_*                                                                    */
    zj_component comp[3];   /* comp[0] = Y and carries the maximum sampling factors (decoder.rs:609-646)    */
} zj_image;

/* ------------------------------------------------------------- GPU path  */

/* Number of CUDA devices visible (0 when there is none; never fails). */
ZJ_API int zj_gpu_device_count(void);

/* Bytes the reference's decode_buffer returns for this image: width*height*out_components
 * (mcu.rs:375-379); ceil(width / d) * ceil(height / d) * out_components for a DCT-scaled image.  Returns 0 on a bad descriptor. */
ZJ_API size_t zj_output_size(const zj_image *img);

/* Validate a descriptor exactly as the GPU entry points do, without touching a device. */
ZJ_API int zj_validate_image(const zj_image *img);

/* Replaces every worker::post_process call of `n` images (worker.rs:32-85).
 * HOST entry point: imgs[i].comp[*].coeff and out[i] are host pointers (pinned memory from
 * zj_gpu_pinned_alloc makes the copies asynchronous); the call stages H2D, launches, copies D2H and
 * returns after `stream` has drained.  out[i] receives exactly zj_output_size(&imgs[i]) bytes; bytes the
 * reference leaves untouched in its zero-initialised Vec (mcu.rs:222) are written as 0. */
ZJ_API int zj_gpu_reconstruct(int device, void *stream, const zj_image *imgs, size_t n,
                              uint8_t *const *out, const size_t *out_len);

/* The same call in two halves, for callers that have host work to do meanwhile (mcu.rs:230-369 entropy-decodes strip k+1
 * while its pool post-processes strip k): _submit queues the uploads, kernels and downloads and returns; the planes and the
 * outputs must stay untouched until _finish(pending) has returned, which waits (the thread sleeps, it does not spin),
 * releases `pending` and reports the status of the whole call.  A failed _submit leaves nothing to finish. */
typedef struct zj_pending zj_pending;
ZJ_API int zj_gpu_reconstruct_submit(int device, void *stream, const zj_image *imgs, size_t n,
                                     uint8_t *const *out, const size_t *out_len, zj_pending **pending);
ZJ_API int zj_gpu_reconstruct_finish(zj_pending *pending);

/* Several devices of one box (north_star: "batches of images (and, for single huge images, restart-interval strips) are
 * partitioned across the GPUs with independent streams, no NCCL: the work shards with no reduction").  n >= n_dev: contiguous
 * image ranges, one per device (zj_partition).  n < n_dev: every image is cut into contiguous STRIP ranges, one per device
 * (zj_image_strip_range): worker::post_process (src/worker.rs:32-85) is called per strip and every rule in it is local to
 * that strip, so a device needs only its strips' coefficient rows and writes only its rows.  One host thread per device
 * drives zj_gpu_reconstruct on that device's streams.  Host pointers, as zj_gpu_reconstruct. */
ZJ_API int zj_gpu_reconstruct_multi(const int *devices, size_t n_dev, const zj_image *imgs, size_t n,
                                    uint8_t *const *out, const size_t *out_len);
/* [begin, end) of part `part` when n_items are cut into n_parts contiguous, balanced ranges (sizes differ by at most one). */
ZJ_API void zj_partition(size_t n_items, size_t n_parts, size_t part, size_t *begin, size_t *end);
/* Strips [strip_begin, strip_end) of `img` as an image of their own: *sub = the descriptor (planes advanced to the first
 * strip, height = the range's rows; the range that ends at the last strip also owns the rows below it), *out_offset /
 * *out_bytes = where its pixels live inside the whole image's output.  *n_strips = strips of the whole image (pass sub,
 * out_offset, out_bytes = NULL to query only that).  Reconstructing every range of a partition gives exactly the bytes of
 * reconstructing the whole image.  ZJ_ERR_UNSUPPORTED: this image cannot be cut (its strip count was limited by the
 * reference's output-capacity rule, mcu_prog.rs:206-209, or it is a ZJ_VARIANT_SPEC image). */
ZJ_API int zj_image_strip_range(const zj_image *img, uint32_t strip_begin, uint32_t strip_end, zj_image *sub,
                                size_t *out_offset, size_t *out_bytes, uint32_t *n_strips);

/* DEVICE entry point: coefficient planes and outputs already live in the memory of `device`.
 * Asynchronous on `stream` (a cudaStream_t, NULL = legacy default stream); no host<->device pixel traffic.
 * Device coefficient planes must start on a 16-byte boundary (ZJ_ERR_INVALID_ARG otherwise; cudaMalloc'ed memory
 * always does); outputs may have any alignment (4-byte aligned outputs take the fastest kernel). */
ZJ_API int zj_gpu_reconstruct_device(int device, void *stream, const zj_image *imgs, size_t n,
                                     uint8_t *const *out_dev, const size_t *out_len);

/* A reusable plan for a fixed batch of device-resident images: descriptors, strip/tile work lists and qt
 * tables are uploaded once; zj_batch_run only launches kernels (CUDA-graph friendly). */
typedef struct zj_batch zj_batch;
ZJ_API int zj_batch_create(int device, const zj_image *imgs, size_t n, uint8_t *const *out_dev,
                           const size_t *out_len, zj_batch **plan);
ZJ_API int zj_batch_run(zj_batch *plan, void *stream);
/* kernels launched by one zj_batch_run (for accounting) */
ZJ_API int zj_batch_launches(const zj_batch *plan);
/* algorithmic bytes one zj_batch_run moves: coefficient bytes read + output bytes written */
ZJ_API uint64_t zj_batch_algorithmic_bytes(const zj_batch *plan);
ZJ_API void zj_batch_destroy(zj_batch *plan);

/* ---------------------------------------------------- device-side consumers (SURVEY.md 8(f).4) */
/* What a GPU consumer of the pixels reads, produced without leaving the device.  The reference's writers stop at
 * interleaved u8 (the per-colourspace dispatch of src/worker.rs:113-133, stores of src/color_convert/scalar.rs:52-169);
 * this descriptor extends them.  Every value is a function of the EXACT u8 the reference writes:
 *   u8:            the byte itself; at half size (a + b + c + d + 2) >> 2 over the 2x2 box (odd last row / column dropped)
 *   f32:           (float(u8) - mean[c]) * inv_std[c]    -- two IEEE fp32 operations (subtract, then multiply), no FMA;
 *                  at half size the first operand is float(a + b + c + d) * 0.25f
 *   f16:           the f32 value rounded to nearest even
 * The default descriptor (zj_output_desc_default: HWC, u8, full size, all channels) is the reference's output unchanged. */
typedef enum zj_layout { ZJ_LAYOUT_HWC = 0, ZJ_LAYOUT_CHW = 1 } zj_layout;
typedef enum zj_dtype { ZJ_DTYPE_U8 = 0, ZJ_DTYPE_F16 = 1, ZJ_DTYPE_F32 = 2 } zj_dtype;
typedef struct zj_output_desc {
    uint32_t layout;      /* zj_layout                                                                          */
    uint32_t dtype;       /* zj_dtype                                                                           */
    uint32_t scale_log2;  /* 0 = full size, 1 = 2x2 box average to (width / 2) x (height / 2)                    */
    uint32_t channels;    /* 0 = every byte of the colourspace's pixel; 3 = drop the 4th byte of RGBA / RGBX    */
    float mean[4];        /* per channel, in u8 units (ignored for u8 output)                                   */
    float inv_std[4];
} zj_output_desc;
ZJ_API void zj_output_desc_default(zj_output_desc *d);
/* 1 when `d` asks for nothing but the reference's bytes */
ZJ_API int zj_output_desc_is_default(const zj_output_desc *d);
/* bytes / width / height / channels of image `img` under descriptor `d` (0 on a bad descriptor) */
ZJ_API size_t zj_consumer_output_size(const zj_image *img, const zj_output_desc *d);
ZJ_API int zj_consumer_output_shape(const zj_image *img, const zj_output_desc *d, uint32_t *out_w, uint32_t *out_h, uint32_t *out_c);
/* The consumer alone: `src_dev` = width*height*nc interleaved u8 in device memory (nc = 1, 3 or 4) -> dst_dev.  Asynchronous on `stream`. */
ZJ_API int zj_gpu_convert_device(int device, void *stream, const uint8_t *src_dev, uint32_t width, uint32_t height, uint32_t nc,
                                 const zj_output_desc *d, void *dst_dev, size_t dst_len);
/* zj_gpu_reconstruct_device followed by the consumer: out_dev[i] receives zj_consumer_output_size(&imgs[i], d) bytes.  The
 * interleaved u8 intermediate lives in a stream-ordered scratch buffer and is produced and consumed in sub-batches of at most
 * ZJ_CONSUMER_CHUNK_MB megabytes (default 1024).  Returns after `stream` has drained. */
ZJ_API int zj_gpu_reconstruct_device_ex(int device, void *stream, const zj_image *imgs, size_t n, const zj_output_desc *d,
                                        void *const *out_dev, const size_t *out_len);

/* ---------------------------------------------------- cropped, resized batch tensors (DESIGN.md section 4.5.1) */
/* What a model reads: one N x OC x OH x OW (CHW) or N x OH x OW x OC (HWC) tensor, slot i at i * zj_resize_slot_size bytes,
 * each slot a crop of image i resized to out_w x out_h, in the type / layout / channels / normalisation of a zj_output_desc
 * (scale_log2 must be 0).  torchvision's resized_crop: crop first, then resize; neighbours are clamped to the crop and pixels
 * outside it never contribute.  p[r][c][ch] = the u8 the reference writes at crop row r, column c; every fp32 operation is
 * one IEEE round-to-nearest operation, in the order written, no FMA:
 *   ZJ_FILTER_AREA      adaptive average pooling: output row i covers crop rows [i*h/OH, ceil((i+1)*h/OH)), columns alike;
 *                       s = exact integer sum of the window's bytes, n = its pixel count.  u8: (s + n/2) / n (integer);
 *                       float: v = float(s) / float(n).  At exactly half size this is the scale_log2 = 1 consumer.
 *   ZJ_FILTER_BILINEAR  torch interpolate(mode="bilinear", align_corners=False, antialias=False): sx = float(w) / float(OW),
 *                       fx = max((float(j) + 0.5f) * sx - 0.5f, 0), c0 = min(int(fx), w - 1), c1 = min(c0 + 1, w - 1),
 *                       ax = fx - float(c0), bx = 1 - ax; rows alike (sy, r0, r1, ay, by).  top = bx*p[r0][c0] + ax*p[r0][c1],
 *                       bot = bx*p[r1][c0] + ax*p[r1][c1], v = by*top + ay*bot.  u8: v rounded to nearest even, clamped to [0, 255].
 *   float outputs       (v - mean[c]) * inv_std[c]; f16 = that value rounded to nearest even.
 * OC = nc, or 3 when channels = 3 and nc = 4; every image of a call must have the same OC.
 *
 * Pillow's Image.resize (DESIGN.md section 4.5.2): ZJ_FILTER_PIL_BILINEAR and ZJ_FILTER_PIL_BICUBIC (16 + Pillow's Resampling
 * number) give Pillow's bytes, and with short_side the result of torchvision's Resize(S) + CenterCrop on a PIL image.  Each
 * channel is independent; for nc = 4 this is Pillow's "RGBX" result, and channels = 3 then gives Pillow's "RGB".
 *   1. Resized size.  short_side = 0: (RW, RH) = (OW, OH), top = left = 0 (RandomResizedCrop, Resize((h, w))).  short_side =
 *      S > 0: short = min(w, h), long = max(w, h), new_long = (int)((double)(S * long) / (double)short), (RW, RH) = (S,
 *      new_long) if w <= h, else (new_long, S); top = round_half_even((RH - OH) / 2.0), left likewise.  RW < OW, RH < OH
 *      (torchvision would pad), RW > 65535 or RH > 65535: ZJ_ERR_INVALID_ARG.
 *   2. Coefficients per axis (in = crop size, out = RW or RH, i = index of the full resized axis), IEEE double in the order
 *      written, no FMA: support0 = 1 (bilinear) or 2 (bicubic); scale = (double)in / out, fs = max(scale, 1.0),
 *      support = support0 * fs, center = (i + 0.5) * scale, xmin = max((int)(center - support + 0.5), 0),
 *      xmax = min((int)(center + support + 0.5), in) - xmin; for x < xmax: k[x] = f(((x + xmin) - center + 0.5) * (1.0 / fs)),
 *      summed in order as ww; k[x] /= ww when ww != 0; kk[x] = (int)(k[x] * 2^22 + 0.5), or (int)(-0.5 + k[x] * 2^22) when
 *      k[x] < 0.  f: bilinear 1 - |x| on |x| < 1; bicubic (a = -0.5) ((a + 2)|x| - (a + 3))x^2 + 1 on |x| < 1,
 *      (((|x| - 5)|x| + 8)|x| - 4)a on |x| < 2; 0 elsewhere.
 *   3. A horizontal pass, then a vertical pass over its u8 result: each value clip8(2^21 + sum(p * kk)) in int32, clip8(s) =
 *      clamp(s >> 22, 0, 255).  (An axis that keeps its size has weights 1, 0, ...: running its pass equals skipping it.)
 *   4. The slot holds rows [top, top + OH) x columns [left, left + OW) of that u8 result u; float outputs are
 *      (float(u) - mean[c]) * inv_std[c]. */
typedef struct zj_roi { uint32_t x, y, w, h; } zj_roi;                      /* w, h >= 1, x + w <= width, y + h <= height */
/* out_w, out_h 1..65535.  reserved = 0 for AREA and BILINEAR; short_side for the PIL filters (0 = resize straight to out_w x out_h) */
typedef struct zj_resize {
    uint32_t out_w, out_h, filter;
    union { uint32_t reserved; uint32_t short_side; };
} zj_resize;
enum { ZJ_FILTER_AREA = 0, ZJ_FILTER_BILINEAR = 1, ZJ_FILTER_PIL_BILINEAR = 18, ZJ_FILTER_PIL_BICUBIC = 19 };
/* bytes of one slot for images of nc bytes per pixel (0 on a bad descriptor) */
ZJ_API size_t zj_resize_slot_size(const zj_output_desc *d, const zj_resize *r, uint32_t nc);
/* The smallest strip range (zj_image_strip_range) whose rows cover [row_begin, row_end), as a virtual image *sub; *sub_row0 =
 * the row of row_begin inside it.  The range that reaches the last strip also owns the rows below it, which the reference never
 * writes.  A range too short to be planned as an image of its own (the output-capacity rule of mcu.rs:198-209 refuses a last
 * strip of a few rows on its own) starts at earlier strips; an image the strip rule cannot cut (ZJ_ERR_UNSUPPORTED there) is
 * returned whole, *sub_row0 = row_begin. */
ZJ_API int zj_image_rows(const zj_image *img, uint32_t row_begin, uint32_t row_end, zj_image *sub, uint32_t *sub_row0);
/* The resize alone over width*height*nc interleaved u8 in device memory (width, height <= 65535; any alignment: no byte
 * outside those width*height*nc is read): crop `roi` (NULL = the whole image) into the dst_dev slot.  Asynchronous on `stream`. */
ZJ_API int zj_gpu_resize_device(int device, void *stream, const uint8_t *src_dev, uint32_t width, uint32_t height, uint32_t nc,
                                const zj_roi *roi, const zj_output_desc *d, const zj_resize *r, void *dst_dev, size_t dst_len);
/* Device coefficient planes in, one batch tensor out (out_len >= n slots).  Only the strips that hold rois[i]'s rows
 * (zj_image_rows) are reconstructed, into a stream-ordered u8 scratch buffer, in sub-batches of at most ZJ_CONSUMER_CHUNK_MB
 * megabytes as zj_gpu_reconstruct_device_ex does; rois = NULL: whole images.  Returns after `stream` has drained. */
ZJ_API int zj_gpu_reconstruct_device_resized(int device, void *stream, const zj_image *imgs, size_t n, const zj_roi *rois,
                                             const zj_output_desc *d, const zj_resize *r, void *out_dev, size_t out_len);

/* Memory helpers so a non-CUDA host language can stage buffers without linking the CUDA runtime. */
ZJ_API int zj_gpu_pinned_alloc(size_t bytes, void **p);
ZJ_API int zj_gpu_pinned_free(void *p);
ZJ_API int zj_gpu_device_alloc(int device, size_t bytes, void **p);
ZJ_API int zj_gpu_device_free(int device, void *p);
ZJ_API int zj_gpu_memcpy_h2d(int device, void *stream, void *dst_dev, const void *src_host, size_t bytes);
ZJ_API int zj_gpu_memcpy_d2h(int device, void *stream, void *dst_host, const void *src_dev, size_t bytes);
ZJ_API int zj_gpu_memset(int device, void *stream, void *dst_dev, int value, size_t bytes);
ZJ_API int zj_gpu_stream_create(int device, void **stream);
ZJ_API int zj_gpu_stream_destroy(int device, void *stream);
ZJ_API int zj_gpu_stream_synchronize(int device, void *stream);
/* CUDA-event timing on `stream` (events see only the stream they are recorded on). */
ZJ_API int zj_gpu_event_create(int device, void **event);
ZJ_API int zj_gpu_event_record(int device, void *event, void *stream);
ZJ_API int zj_gpu_event_elapsed_ms(int device, void *start, void *stop, float *ms);
ZJ_API int zj_gpu_event_destroy(int device, void *event);

ZJ_API const char *zj_gpu_strerror(int status);
ZJ_API const char *zj_gpu_last_cuda_error(void);
/* number of kernel launches this library has issued in this process (monotonic) */
ZJ_API uint64_t zj_gpu_launch_count(void);

/* ------------------------------------------------- host front-end (C++)  */
/* The reference's host stage -- headers (src/headers.rs, src/marker.rs, src/decoder.rs:239-411) and entropy
 * decode (src/bitstream.rs, src/huffman.rs, src/mcu.rs:253-351, src/mcu_prog.rs:49-129,249-430) -- stays on
 * the CPU.  There is no Rust toolchain in this build environment, so it is restated in C++ here; in a Rust
 * deployment these symbols are not needed (INTEGRATION.md). */

typedef struct zj_options {       /* ZuneJpegOptions (src/options.rs:6-40), same defaults */
    uint32_t use_unsafe;          /* 1; ZJ_USE_SPEC_OUTPUT (not in the reference): ZJ_VARIANT_SPEC output, and the host stage
                                     decodes every MCU row with Q9-Q11 off, whatever zj_host_set_quirks says;
                                     ZJ_USE_LIBJPEG_OUTPUT: the same, and the images carry ZJ_FLAG_ISLOW;
                                     ZJ_USE_LIBJPEG_OUTPUT | k << 4, k = 1..3: the same, decoded at 1/2^k (ZJ_FLAG_SCALE_*);
                                     any of these three | ZJ_USE_EXIF_ORIENTATION: the same, oriented (ZJ_FLAG_ORIENT_*) */
    uint32_t out_colorspace;      /* ZJ_CS_RGB                                           */
    uint32_t num_threads;         /* 4                                                   */
    uint32_t max_width;           /* 16384                                               */
    uint32_t max_height;          /* 16384                                               */
    uint32_t max_scans;           /* 64                                                  */
    uint32_t strict_mode;         /* 0                                                   */
    int32_t device;               /* CUDA ordinal used by zj_decoder_decode_buffer (0)   */
} zj_options;

/* DecodeErrors variants (src/errors.rs:16-43) */
typedef enum zj_decode_error_kind {
    ZJ_DE_NONE = 0,
    ZJ_DE_FORMAT = 1,
    ZJ_DE_FORMAT_STATIC = 2,
    ZJ_DE_ILLEGAL_MAGIC_BYTES = 3,
    ZJ_DE_HUFFMAN_DECODE = 4,
    ZJ_DE_ZERO_ERROR = 5,
    ZJ_DE_DQT_ERROR = 6,
    ZJ_DE_SOS_ERROR = 7,
    ZJ_DE_SOF_ERROR = 8,
    ZJ_DE_UNSUPPORTED = 9,
    ZJ_DE_MCU_ERROR = 10,
    ZJ_DE_EXHAUSTED_DATA = 11,
    ZJ_DE_LARGE_DIMENSIONS = 12,
    ZJ_DE_GPU = 13 /* not in the reference: the GPU stage failed, message = zj_gpu_strerror */
} zj_decode_error_kind;

typedef struct zj_image_info {    /* ImageInfo (src/decoder.rs:652-668) */
    uint16_t width, height;
    uint8_t pixel_density;
    uint8_t sof;                  /* SOFMarkers ordinal (src/misc.rs): 0 BaselineDct, 2 ProgressiveDctHuffman */
    uint16_t x_density, y_density;
    uint8_t components;
    uint8_t valid;                /* 0 until headers were parsed (Decoder::info() -> None, decoder.rs:210)    */
} zj_image_info;

typedef struct zj_decoder zj_decoder;

ZJ_API void zj_options_default(zj_options *o);
ZJ_API zj_decoder *zj_decoder_new(const zj_options *o);                /* Decoder::new_with_options           */
ZJ_API void zj_decoder_free(zj_decoder *d);
ZJ_API int zj_decoder_read_headers(zj_decoder *d, const uint8_t *buf, size_t len); /* Decoder::read_headers  */
ZJ_API int zj_decoder_info(const zj_decoder *d, zj_image_info *info);  /* Decoder::info                       */
ZJ_API uint32_t zj_decoder_out_colorspace(const zj_decoder *d);        /* Decoder::get_output_colorspace      */
/* The EXIF orientation o (1-8) of the last zj_decoder_read_headers / decode, whatever the options: 1 before headers were read
 * or when the file has none (the rules are next to ZJ_FLAG_ORIENT_SHIFT).  Callers size outputs and draw crops with it. */
ZJ_API uint32_t zj_decoder_orientation(const zj_decoder *d);
/* Host stage only: headers + entropy decode into coefficient planes owned by the decoder (pinned when a
 * device is present).  `img` is filled with a descriptor pointing at them (valid until the next call). */
ZJ_API int zj_decoder_decode_coefficients(zj_decoder *d, const uint8_t *buf, size_t len, zj_image *img);
/* Baseline scans with restart markers (DRI) are entropy-decoded by up to `num_threads` host threads, one restart interval
 * per thread at a time (src/mcu.rs:253-351 and 386-418 run per interval); the result is kept only when every interval ended
 * exactly where the next one starts, otherwise the scan is redone by the reference's sequential loop, so the planes are
 * always what that loop produces.  Returns how many intervals the last decode ran side by side (0 = sequential loop). */
ZJ_API size_t zj_decoder_entropy_segments(const zj_decoder *d);
/* Decoder::decode_buffer: host stage, then zj_gpu_reconstruct.  *out is malloc'd (zj_buffer_free). */
ZJ_API int zj_decoder_decode_buffer(zj_decoder *d, const uint8_t *buf, size_t len, uint8_t **out,
                                    size_t *out_len);
ZJ_API void zj_buffer_free(uint8_t *p);
/* decode_into of later zune-jpeg releases: the same, into the caller's buffer of out_cap bytes (pinned memory from
 * zj_gpu_pinned_alloc makes every copy asynchronous); *out_len = bytes written.  Baseline images of >= 4 MP run as a strip
 * pipeline the way the reference's driver does (src/mcu.rs:230-369 entropy-decodes strip k+1 while its pool post-processes
 * strip k): finished strip ranges (zj_image_strip_range) are uploaded, reconstructed and downloaded while the host --
 * sequentially, or with its restart intervals side by side -- is still entropy-decoding the rest of the image. */
ZJ_API int zj_decoder_decode_into(zj_decoder *d, const uint8_t *buf, size_t len, uint8_t *out, size_t out_cap,
                                  size_t *out_len);
/* Batch front door (the reference has none: it parallelises the strips of ONE image, mcu.rs:230-369): n JPEGs are
 * decoded by `o->num_threads` host threads (0 = one per hardware thread), one image per thread at a time; each thread
 * runs the host stage, hands its planes to zj_gpu_reconstruct_submit and starts on its next image (a second set of planes)
 * while the GPU works, so entropy decoding overlaps transfer and reconstruction of this thread's and the others' images.  out[i] non-NULL on entry = caller buffer of out_len[i] bytes (pinned memory copies
 * fastest); NULL = malloc'ed here (zj_buffer_free).  status[i] = per-image zj_status; returns the number of failed
 * images (0 = all decoded) or a negative zj_status for invalid arguments. */
ZJ_API int zj_decode_batch(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                           uint8_t **out, size_t *out_len, int *status);
/* The DecodeErrors of image i of the LAST batch call made by the calling thread (any of the zj_decode_batch* front doors):
 * the variant (zj_decode_error_kind) and Display text Decoder::decode_buffer would have reported for that input
 * (src/errors.rs:16-113); ZJ_DE_NONE / "" for images that decoded.  Valid until the thread's next batch call. */
ZJ_API int zj_batch_error_kind(size_t i);
ZJ_API const char *zj_batch_error(size_t i);
/* zj_decode_batch keeps its workers' decoders (pinned coefficient planes sized for the largest image seen, two per host
 * thread) for the next call; this frees them. */
/* zj_decode_batch over several devices of one box: contiguous image ranges, one per device, each range decoded by its own
 * share of the host threads (o->num_threads / n_dev each; o->device is ignored) and reconstructed on its device.  With
 * fewer images than devices every image is entropy-decoded by all host threads (restart intervals side by side) and its
 * strips are spread over the devices (zj_gpu_reconstruct_multi). */
ZJ_API int zj_decode_batch_multi(const zj_options *o, const int *devices, size_t n_dev, const uint8_t *const *bufs,
                                 const size_t *lens, size_t n, uint8_t **out, size_t *out_len, int *status);
ZJ_API void zj_release_host_caches(void);
/* Device-side state kept between calls, and its release.  zj_gpu_reconstruct[_submit] keeps, per host thread that called it,
 * its staging streams and up to three device staging buffers (256 MB sub-batches by default); zj_decode_batch_gpu[_device]
 * keeps two slots of device staging memory (>= 1 GB each once used, up to the 4 / 8 GB sub-batch budget; a slot that a call
 * grew beyond ZJ_RETAIN_MB megabytes is freed when that call ends -- default 16384, i.e. never: re-allocating a 6.7 GB slot
 * was measured at up to 119 ms per call), their streams and small pinned blocks.  zj_release_device_caches frees all of
 * it except what a thread is using at that moment (it waits for a zj_decode_batch_gpu call in flight); the next call
 * allocates again.  Call it when the process wants its HBM back, e.g. a data loader that shares the GPU with a training job. */
ZJ_API void zj_release_device_caches(void);
/* The same call with the entropy stage on the GPU too, for the JPEGs that allow it: baseline scans with restart markers (DRI)
 * whose every interval ends the way the reference's sequential loop (src/mcu.rs:253-351, 386-418) ends it.  Their files are
 * uploaded instead of their coefficient planes, one GPU thread per restart interval runs the reference's bit reader and MCU
 * loop (src/bitstream.rs:159-402) into device planes, which are reconstructed in place.  All other images (no DRI,
 * progressive, header errors, an interval that ends differently) take the zj_decode_batch route, so pixels, statuses and
 * errors are those of zj_decode_batch.  *n_gpu_entropy (may be NULL) = images whose entropy stage ran on the GPU. */
ZJ_API int zj_decode_batch_gpu(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                               uint8_t **out, size_t *out_len, int *status, size_t *n_gpu_entropy);
/* ... and with the pixels left in device memory (no PCIe download at all: what is uploaded is the JPEG file): out_dev[i] is a
 * device buffer of out_len[i] >= width*height*components bytes (sizes: zj_decoder_read_headers + zj_decoder_info); images
 * that take the host route are uploaded after decoding.  The call returns when all pixels are in place. */
ZJ_API int zj_decode_batch_gpu_device(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                                      uint8_t *const *out_dev, size_t *out_len, int *status, size_t *n_gpu_entropy);
/* ... and handed to a device-side consumer (zj_output_desc above): out_dev[i] receives zj_consumer_output_size bytes in the
 * layout / type / scale of `d` (sizes before decoding: zj_decoder_read_headers + zj_decoder_info give width, height and
 * components; out_len[i] is checked).  On return out_len[i] = bytes written. */
ZJ_API int zj_decode_batch_gpu_device_ex(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                                         const zj_output_desc *d, void *const *out_dev, size_t *out_len, int *status,
                                         size_t *n_gpu_entropy);
/* ... and cropped and resized into one batch tensor (zj_gpu_reconstruct_device_resized above; out_len >= n slots, the slot size
 * from the OC that o->out_colorspace gives).  Whole images are decoded; statuses and zj_batch_error* are those of
 * zj_decode_batch, and a decoded image whose roi does not fit it (known only after its headers) or whose OC differs gets
 * ZJ_ERR_INVALID_ARG.  The slot of a failed image is left untouched.  rois = NULL: whole images. */
ZJ_API int zj_decode_batch_gpu_device_resized(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                                              const zj_roi *rois, const zj_output_desc *d, const zj_resize *r, void *out_dev,
                                              size_t out_len, int *status, size_t *n_gpu_entropy);
/* TEST-ONLY switches for three bugs of the reference's host stage that this library reproduces by default so that its
 * coefficient planes are the reference's (DESIGN.md section 2).  A cleared bit makes the cited lines behave like libjpeg:
 *   Q9  src/huffman.rs:249-252   fast-AC entry `(k << 10) + ...` is an i16: |k| >= 32 loses its top bits
 *   Q10 src/bitstream.rs:278-281 decode_dc refills only below 16 buffered bits but may consume 27: the reader under-runs
 *   Q11 src/mcu.rs:337-342       the MCU loop breaks on a PREFETCHED EOI: trailing components of the last MCU stay zero
 * Process-wide; takes effect for decodes started afterwards (a ZJ_USE_SPEC_OUTPUT decode runs with every bit cleared, whatever
 * is set here).  With any bit cleared the GPU entropy route (zj_decode_batch_gpu*) sends every image through the host stage.
 * tests/test_quirks.py is the only caller. */
enum { ZJ_QUIRK_Q9_FAST_AC_I16 = 1u, ZJ_QUIRK_Q10_DC_REFILL = 2u, ZJ_QUIRK_Q11_EOI_BREAK = 4u, ZJ_QUIRK_ALL = 7u };
ZJ_API void zj_host_set_quirks(uint32_t mask);
ZJ_API uint32_t zj_host_get_quirks(void);
ZJ_API int zj_decoder_error_kind(const zj_decoder *d);                 /* zj_decode_error_kind                */
ZJ_API const char *zj_decoder_error(const zj_decoder *d);              /* Display text of the DecodeErrors    */

#ifdef __cplusplus
}
#endif
#endif /* ZUNE_JPEG_B200_H */
