// zj_device.h -- descriptors shared by the host-side planner (zj_capi.cu) and the kernels (zj_kernels.cu), and the
// declarations of the library's functions that one source file calls in another.
//
// Vocabulary follows the reference: an image is cut into MCU-row *strips* (the unit of
// worker::post_process, reference src/worker.rs:32; geometry src/mcu.rs:139-226, src/mcu_prog.rs:132-203);
// a strip is cut into *tiles* of TM MCU columns, one CTA per tile.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/zune_jpeg_b200.h"

namespace zj {

enum Mode : int { MODE_NONE = 0, MODE_H = 1, MODE_V = 2, MODE_HV = 3 };  // SubSampRatios, components.rs:130
enum OutKind : int {
    OUT_RGB = 0,   // YCbCr -> RGB | "RGBA" | "RGBX": the 3-byte conv16 + row-tail rule (worker.rs:143-251)
    OUT_YCC = 1,   // YCbCr -> YCbCr interleave (color_convert/scalar.rs:119-169)
    OUT_GRAY = 2,  // (YCbCr | GRAYSCALE) -> GRAYSCALE (color_convert/scalar.rs:91-114)
    OUT_ZERO = 3   // every other pair: nothing is written (worker.rs:131-132)
};

// MCU columns per tile, chosen so that one CTA of ZJ_THREADS threads has about one 8x8 block per thread
// (including the chroma halo blocks):                 blocks / MCU column        + halo
//   (per 128 threads) NONE: 3 blocks -> TM 40 -> 120  H: 8 -> TM 15 -> 120 + 8
//   V:    4 blocks  -> TM 32 -> 128                   HV: 12 -> TM 10 -> 120 + 8 (+4 in tile 0)
constexpr int ZJ_THREADS = 256;
constexpr int ZJ_MINBLOCKS = 3;  // CTAs per SM the register allocation is capped for
constexpr int ZJ_SLOW_CAP = 192;  // edge units per tile queued for the generic path
// tile widths scale with the CTA size (128 threads: 40 / 15 / 32 / 10)
constexpr int TM_NONE = 40 * ZJ_THREADS / 128, TM_H = 15 * ZJ_THREADS / 128, TM_V = 32 * ZJ_THREADS / 128, TM_HV = 10 * ZJ_THREADS / 128, TM_GRAY = 128;

// The fast kernel (X86 variant): 256 threads = 128 producers (IDCT, two 8x8 blocks per thread and strip) + 128
// consumers (up-sampling / colour / stores, two 16-sample units per thread and strip).
constexpr int ZF_THREADS = 256, ZF_PRODUCERS = 128, ZF_CONSUMERS = 128;
constexpr int ZF_MINBLOCKS = 3;
constexpr int ZF_DEFAULT_SPC = 40;      // target strips per CTA (see strips_per_cta)
// unit columns (16 luma samples) per tile: 2 * ZF_CONSUMERS / row groups per strip
constexpr int ZF_XU_GRAY = 32;                  // luma-only fast kernel: 512-sample tiles
// (4:2:2: 15 instead of 16 -- the strip-tile's block list, 2 x 30 luma + 2 x 2 x 15 chroma + 8 halo blocks, is then exactly
// 128 = one IDCT pass of the four producer warps; with 16 it is 136 and the producers' critical path a second pass)
constexpr int ZF_XU_NONE = 2 * ZF_CONSUMERS / 8, ZF_XU_H = 15, ZF_XU_V = 2 * ZF_CONSUMERS / 8, ZF_XU_HV = 2 * ZF_CONSUMERS / 16;

struct DevImage {
    const int16_t *coeff[3];  // device pointers, whole-image planes
    uint8_t *out;             // device pointer, width*height*nc bytes
    uint32_t qtw[3][32];      // quantisation tables packed for dp2a: word k = q[2k] | q[2k+1] << 24
    uint32_t width, height;
    uint32_t nc;              // output bytes per pixel
    uint32_t out_kind;        // OutKind
    uint32_t mcu_x;           // MCU columns (headers.rs:316)
    uint32_t n_strips;        // strips the reference processes (Q1: may not cover the image)
    uint32_t n_tiles;         // tiles per strip
    uint32_t Wp;              // luma plane row width = comp[0].width_stride
    uint32_t W;               // chroma plane row width = comp[1].width_stride (0 if no chroma)
    uint32_t stride;          // output row stride in bytes = width*nc
    // colour writer constants (worker.rs:171,221-223; SURVEY A.5)
    uint32_t n_norm;          // samples [0, n_norm) of a row are written at byte 3*s ("normal" chunks)
    uint32_t P;               // 3*n_norm for RGB; bytes >= P not covered by the tail stay zero
    uint32_t T;               // tail chunk (samples Wp-16..Wp-1) lands at bytes [T, T+48); 0xffffffff = none
    uint32_t small_width;     // width < 16: temp-buffer path (worker.rs:158-163,176-198)
    uint32_t hv_avx;          // HV + X86 + chroma strip >= 500 samples -> AVX2 closed form
    uint32_t gray_rows_ok;    // Q7 resolved: 1 = plain row copy is what the reference does
    uint32_t gray_brows;      // luma-only output: block rows of the Y plane the reference processes
    uint32_t tile_q, tile_r;  // tile t covers MCU columns (fast kernel: 16-sample unit columns) [t*q + min(t,r), ...): the first r tiles are one wider
    uint32_t chroma_wh;       // DCT-scaled images: the real chroma size dw | dh << 16 (width, height, stride: the scaled output's;
                              // n_strips: MCU rows)
    uint64_t magic_w;         // ceil(2^40 / W): idx / W == (idx * magic_w) >> 40 for idx < 2^20
};

// MCU columns per tile of scaled_kernel (DCT-scaled images), by mode: about one block per thread in phase 1
constexpr int TS_NONE = 80, TS_H = 60, TS_V = 32, TS_HV = 42;
// The scale k of a zj_image (ZJ_FLAG_SCALE_*), and the size of its output (output_dims): width x height, or ceil(width / 2^k) x
// ceil(height / 2^k) for a DCT-scaled image, with the two swapped by orientations 5-8.  Everything downstream of reconstruction
// sees this size.
inline uint32_t image_scale(const zj_image *img) { return (img->flags & ZJ_FLAG_SCALE_MASK) >> ZJ_FLAG_SCALE_SHIFT; }
// The EXIF orientation code o - 1 of a zj_image (ZJ_FLAG_ORIENT_*): 0 = none; 4-7 (o = 5-8) swap width and height
inline uint32_t image_orient(const zj_image *img) { return (img->flags & ZJ_FLAG_ORIENT_MASK) >> ZJ_FLAG_ORIENT_SHIFT; }
// The reconstructed image before orientation: the size the kernels write (and the oriented image's stored frame)
inline void stored_dims(const zj_image *img, uint32_t *w, uint32_t *h)
{
    const uint32_t k = image_scale(img), m = (1u << k) - 1;
    *w = (uint32_t)(((uint64_t)img->width + m) >> k);
    *h = (uint32_t)(((uint64_t)img->height + m) >> k);
}
inline void output_dims(const zj_image *img, uint32_t *w, uint32_t *h)
{
    if (image_orient(img) >= 4) stored_dims(img, h, w);
    else stored_dims(img, w, h);
}

// Pillow's Transpose for orientation code t = o - 1 (ZJ_FLAG_ORIENT_*), as a map of stored pixel (x, y) of a w x h image to the
// output: mirror x (x -> w-1-x), mirror y, then swap the axes.
inline __host__ __device__ bool orient_flip_x(uint32_t t) { return t == 1 || t == 2 || t == 6 || t == 7; }
inline __host__ __device__ bool orient_flip_y(uint32_t t) { return t == 2 || t == 3 || t == 5 || t == 6; }
inline __host__ __device__ bool orient_swap(uint32_t t) { return t >= 4; }

// One image of an orient launch (zj_consumer.cu): a w x h region of interleaved u8 pixels (row pitch `pitch` bytes, starting at
// `src`) goes through the transform of orientation code `orient` into `dst`, a tightly packed image of w x h (or h x w) pixels.
struct OrientImage {
    const uint8_t *src;
    uint8_t *dst;
    uint32_t pitch;
    uint32_t w, h;
    uint32_t orient;
    uint32_t nc;                  // bytes per pixel (the launch's)
};

// A four-component (CMYK / YCCK) image: what zj_image cannot carry -- the fourth component and the colour model the host stage
// decided (DESIGN.md section 4.6.4).  Passed next to a zj_image with n_comp = 4; not part of the C ABI.
struct Extra4 {
    zj_component k;           // the fourth component in SOF order
    uint32_t jpeg_cs;         // ZJ_CS_CMYK or ZJ_CS_YCCK
};

// One image of a raster_kernel launch (ZJ_VARIANT_SPEC): four-component input, or three components with sampling factors other
// than luma (1|2) x (1|2) and chroma 1 x 1.  The planes are raster planes of mcu_x h_z x mcu_y v_z blocks.  Only that kernel reads
// it, so DevImage -- and the code of every other kernel -- stays as it is.
enum RasterKind : uint32_t {
    RASTER_OUT_RGB = 0,    // RGB, RGBA, RGBX
    RASTER_OUT_GRAY = 1,   // GRAYSCALE
    RASTER_OUT_RAW = 2     // the colour model's own samples: CMYK (four components), YCbCr (three)
};
enum RasterModel : uint32_t { RASTER_YCC = 0, RASTER_CMYK = 1, RASTER_YCCK = 2 };   // the colour model of the components
constexpr int TC_PIXELS = 128;   // output columns per raster_kernel tile (at most)
struct RasterImage {
    const int16_t *coeff[4];  // device pointers, whole-image planes in SOF order
    uint8_t *out;             // W' x H' x nc bytes (the stored frame)
    uint32_t qtw[4][32];      // as DevImage::qtw
    uint32_t bpr[4];          // blocks per plane row (width_stride / 8)
    uint32_t h[4], v[4];      // sampling factors (1..4)
    uint32_t ss[4];           // block size in samples (rule 1'')
    uint32_t dw[4], dh[4];    // real component sizes (rule 3'')
    uint32_t ratio[4];        // up-sampling ratios rh | rv << 8: rh = hmax s0 / (h ss), rv = vmax s0 / (v ss) (1..4 each)
    uint32_t width, height;   // W' x H'
    uint32_t nc, kind, model; // output bytes per pixel, RasterKind, RasterModel
    uint32_t hmax, vmax, mcu_x, mcu_y, tile_mcus, n_tiles;
};
// Three-component factors that take raster_kernel (spec output): every factor 1..4, and not luma (1|2) x (1|2) with chroma 1 x 1,
// which the fused kernels take
inline bool raster_factors(const zj_component (&c)[3])
{
    for (int z = 0; z < 3; z++)
        if (c[z].h_samp < 1 || c[z].h_samp > 4 || c[z].v_samp < 1 || c[z].v_samp > 4) return false;
    const bool luma = c[0].h_samp <= 2 && c[0].v_samp <= 2;
    return !(luma && c[1].h_samp == 1 && c[1].v_samp == 1 && c[2].h_samp == 1 && c[2].v_samp == 1);
}
// Block size in samples of a component with factors (h, v) when the largest are (hmax, vmax) and the smallest block is s0 (rule
// 1'', libjpeg-turbo jdmaster.c jpeg_core_output_dimensions)
inline uint32_t block_size(uint32_t hmax, uint32_t vmax, uint32_t h, uint32_t v, uint32_t s0)
{
    uint32_t ss = s0;
    while (ss < 8 && (hmax * s0) % (2 * h * ss) == 0 && (vmax * s0) % (2 * v * ss) == 0) ss *= 2;
    return ss;
}

// Host-side launch plan entry: one kernel launch per (mode, variant, IDCT, out-kind class) group.
struct LaunchGroup {
    int mode, variant, gray;  // gray = luma-only kernel
    int fast;                 // reconstruct_fast_kernel (X86 variant, aligned output)
    int islow;                // ZJ_FLAG_ISLOW (SPEC variant only): libjpeg-turbo's islow IDCT
    int scale;                // ZJ_FLAG_SCALE_* (SPEC | ISLOW only): 1/2^scale DCT-scaled decode, scaled_kernel
    int raster;               // 3 or 4: raster_kernel over RasterImage records of that many components (first / count index those)
    uint32_t first, count;    // images [first, first+count) of the sorted device array
    uint32_t max_tiles, max_strips;
};

// One image of a consumer launch (zj_consumer.cu): interleaved u8 pixels in, the layout / type / scale of zj_output_desc out.
struct ConvImage {
    const uint8_t *src;           // u8, interleaved, width * height * nc
    void *dst;
    uint32_t width, height, nc;   // source geometry
    uint32_t ow, oh, oc;          // output geometry (oc = channels written)
};

// One image of a resize launch (zj_consumer.cu): a crop of interleaved u8 pixels in, one slot of the batch tensor out.  The
// output size, layout, type and channels are the launch's.
struct ResizeImage {
    const uint8_t *src;           // byte 0 of the crop's pixel (0, first): first = 0, or PilGeometry::y0 for the PIL filters
    const uint8_t *lo, *hi;       // the source image's bytes: no load reaches outside [lo, hi)
    void *dst;                    // the image's slot
    uint32_t pitch;               // bytes per source row (width * nc)
    uint32_t w, h;                // crop size in pixels
    float sx, sy;                 // bilinear scales float(w) / float(out_w), float(h) / float(out_h) (one IEEE division each)
};

// Kernel launches: zj_kernels.cu (reconstruction), zj_consumer.cu (consumer, resize)
cudaError_t launch_group(const DevImage *d_images, const LaunchGroup &g, cudaStream_t stream);
cudaError_t launch_raster(const RasterImage *d_images, const LaunchGroup &g, cudaStream_t stream);
cudaError_t launch_convert(const ConvImage *d_images, uint32_t count, uint32_t nc, uint32_t max_ow, uint32_t max_oh, const zj_output_desc &d, cudaStream_t s);
cudaError_t launch_resize(const ResizeImage *d_images, uint32_t count, uint32_t nc, const zj_output_desc &d, const zj_resize &r, cudaStream_t s);
// images [0, count) (count <= 65535) of nc bytes per pixel; max_w x max_h covers every region
cudaError_t launch_orient(const OrientImage *d_images, uint32_t count, uint32_t nc, uint32_t max_w, uint32_t max_h, cudaStream_t s);

// The PIL filters (header rules 1 and 2) for a crop of w x h: the resized size, the window's offset in it, and the crop rows
// [y0, y1) the window's vertical taps read.  ZJ_ERR_INVALID_ARG when the resized size breaks rule 1.
inline bool pil_filter(uint32_t filter) { return filter == ZJ_FILTER_PIL_BILINEAR || filter == ZJ_FILTER_PIL_BICUBIC; }
struct PilGeometry { uint32_t rw, rh, left, top, y0, y1; };
int pil_geometry(const zj_resize &r, uint32_t w, uint32_t h, PilGeometry *g);
// The PIL resize of images host[0, count) (count <= 65535, one nc): coefficient tables, horizontal and vertical passes, with
// their scratch from the stream-ordered pool of `device`.  *launches += the kernels launched.  Asynchronous on `s`.
cudaError_t launch_pil_resize(const ResizeImage *host, uint32_t count, uint32_t nc, const zj_output_desc &d, const zj_resize &r,
                              int device, cudaStream_t s, int *launches);

// ---- zj_capi.cu for zj_host_decoder.cpp (hidden symbols, not part of the C ABI)
int num_components(uint32_t cs);   // output bytes per pixel of colourspace cs (ColorSpace::num_components); 0 = not a colourspace
// bytes the consumer writes for a width x height image of nc bytes per pixel; 0 = a bad descriptor or nc
size_t convert_size(uint32_t width, uint32_t height, uint32_t nc, const zj_output_desc *d);
// *crop = the crop `roi` of a width x height image of nc bytes per pixel (NULL = the whole image), into a batch tensor of
// slot_nc-byte source pixels; ZJ_ERR_INVALID_ARG when it does not fit the image, the image's channel count is not the slots' or
// (PIL filters) its resized size breaks rule 1
int resize_admit(const zj_output_desc *d, const zj_resize *r, uint32_t slot_nc, const zj_roi *roi, uint32_t width, uint32_t height,
                 uint32_t nc, zj_roi *crop);
// device memory from this library's stream-ordered pool of `device`, allocated / freed in the order of `stream`
int scratch_alloc(void **p, size_t bytes, int device, void *stream);
void scratch_free(void *p, void *stream);

// One decoded image in device memory: the input of the second pass of the JPEG-bytes route
struct U8Image {
    const uint8_t *src;           // u8, interleaved, width * height * nc
    uint32_t width, height, nc;
    zj_roi crop;                  // resize_many: the crop
    void *dst;                    // convert_many: the image's output; resize_many: its slot
};
// the consumer / the resize over n decoded images, one launch per run of equal pixel formats; asynchronous on `stream`
int convert_many(int device, void *stream, const U8Image *imgs, size_t n, const zj_output_desc *d);
int resize_many(int device, void *stream, const U8Image *imgs, size_t n, const zj_output_desc *d, const zj_resize *r);

// zj_gpu_reconstruct_submit with an optional Extra4 per image (ext = NULL, or ext[i] read only where imgs[i].n_comp = 4): the
// JPEG-bytes routes reach four-component images through it.  zj_gpu_reconstruct_submit passes NULL, so the planes-in entry
// points keep refusing n_comp = 4.
int reconstruct_submit4(int device, void *stream, const zj_image *imgs, const Extra4 *ext, size_t n, uint8_t *const *out,
                        const size_t *out_len, zj_pending **pending);
// zj_validate_image of such an image, *out_size = zj_output_size (ext is read only when img->n_comp = 4)
int validate_image4(const zj_image *img, const Extra4 *ext, size_t *out_size);

void release_stream_caches();   // the idle staging streams and buffers of zj_gpu_reconstruct_submit
void trim_pools();              // the stream-ordered pools' cached memory back to the driver

}  // namespace zj
