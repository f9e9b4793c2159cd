// zj_capi.cu -- the C ABI of include/zune_jpeg_b200.h: descriptor validation, strip/tile planning, device
// memory plumbing and kernel launches.  No CPU fallback lives here: without a CUDA device every compute
// entry point returns ZJ_ERR_NO_DEVICE.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <mutex>
#include <new>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/zune_jpeg_b200.h"
#include "zj_device.h"

using namespace zj;

static thread_local char g_cuda_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

static int cuda_fail(cudaError_t e, const char *what)
{
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
    if (e == cudaErrorMemoryAllocation) return ZJ_ERR_OOM;
    return ZJ_ERR_CUDA;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(e_, #call); } while (0)

int zj::num_components(uint32_t cs)  // ColorSpace::num_components, reference src/misc.rs:108-118
{
    switch (cs) {
    case ZJ_CS_RGB: case ZJ_CS_YCBCR: return 3;
    case ZJ_CS_CMYK: case ZJ_CS_YCCK: case ZJ_CS_RGBA: case ZJ_CS_RGBX: return 4;
    case ZJ_CS_GRAYSCALE: return 1;
    default: return 0;
    }
}

// --------------------------------------------------------------------------------------------- planning
struct Plan {
    int mode, variant, gray, zero_only, fast;
    int islow;         // ZJ_FLAG_ISLOW: the kernels' IDCT is libjpeg-turbo's islow
    int scale;         // ZJ_FLAG_SCALE_*: DCT-scaled decode to 1/2^scale (scaled_kernel)
    int orient;        // ZJ_FLAG_ORIENT_*: the orientation code o - 1 (0 = none), applied by a second pass (orient_kernel)
    uint32_t n_strips, rows, ncomp_used;
    size_t chunk[3];   // i16 per strip per component
    size_t out_size;
    DevImage dev;      // pointers filled by the caller
    uint32_t grid_tiles, grid_strips;   // launch extents (grid_strips: strips as the kernel counts them)
};

// Strip geometry of reference src/mcu.rs:139-226 (baseline) / src/mcu_prog.rs:132-203 (progressive) and the
// colour-writer constants of src/worker.rs:143-251.
static int plan_image(const zj_image *img, Plan *pl, const void *out = nullptr)
{
    if (!img) return ZJ_ERR_INVALID_ARG;
    if (img->n_comp != 1 && img->n_comp != 3) return ZJ_ERR_INVALID_ARG;
    if (img->width == 0 || img->height == 0 || img->width > 65535 || img->height > 65535) return ZJ_ERR_INVALID_ARG;
    const int nc = num_components(img->out_cs);
    if (nc == 0) return ZJ_ERR_INVALID_ARG;
    if (img->variant != ZJ_VARIANT_X86 && img->variant != ZJ_VARIANT_SCALAR && img->variant != ZJ_VARIANT_SPEC) return ZJ_ERR_INVALID_ARG;
    const bool spec = img->variant == ZJ_VARIANT_SPEC;
    const bool islow = (img->flags & ZJ_FLAG_ISLOW) != 0;   // spec output with libjpeg-turbo's IDCT: every rule below as for spec
    if (islow && !spec) return ZJ_ERR_INVALID_ARG;
    const uint32_t scale = image_scale(img);                 // DCT-scaled: spec | islow planes, reconstructed by scaled_kernel
    if (scale && !islow) return ZJ_ERR_INVALID_ARG;
    const uint32_t orient = image_orient(img);               // oriented: spec planes, reconstructed as such, then orient_kernel
    if (orient && !spec) return ZJ_ERR_INVALID_ARG;
    const uint32_t h = img->comp[0].h_samp, v = img->comp[0].v_samp;
    if (img->n_comp == 1 && (h != 1 || v != 1)) return ZJ_ERR_UNSUPPORTED;  // mcu.rs:171-196 resets these before the path
    for (uint32_t z = 1; z < img->n_comp; z++)
        if (img->comp[z].h_samp != 1 || img->comp[z].v_samp != 1) return ZJ_ERR_UNSUPPORTED;  // decoder.rs:634-643
    int mode;
    if (h == 1 && v == 1) mode = MODE_NONE;
    else if (h == 2 && v == 1) mode = MODE_H;
    else if (h == 1 && v == 2) mode = MODE_V;
    else if (h == 2 && v == 2) mode = MODE_HV;
    else return ZJ_ERR_UNSUPPORTED;  // decoder.rs:512-519

    const uint32_t w = img->width, hh = img->height;
    const uint32_t mcu_x = (w + 8 * h - 1) / (8 * h), mcu_y = (hh + 8 * v - 1) / (8 * v);  // headers.rs:316-318
    for (uint32_t z = 0; z < img->n_comp; z++) {
        if (img->comp[z].width_stride != img->comp[z].h_samp * mcu_x * 8) return ZJ_ERR_INVALID_ARG;  // headers.rs:338
        for (int k = 0; k < 64; k++)
            if (img->comp[z].qt[k] < 0 || img->comp[z].qt[k] > 255) return ZJ_ERR_INVALID_ARG;  // 8-bit tables only, headers.rs:156-173
    }
    memset(pl, 0, sizeof(*pl));
    pl->mode = mode;
    pl->variant = (int)img->variant;
    pl->islow = islow;
    pl->scale = (int)scale;
    pl->orient = (int)orient;
    uint32_t n_strips, ybr, cbr;
    switch (mode) {
    case MODE_H: n_strips = mcu_y / 2; ybr = 2; cbr = 2; break;   // mcu.rs:147-154 -- Q1: odd MCU row dropped
    case MODE_HV: n_strips = mcu_y / 2; ybr = 4; cbr = 2; break;  // mcu.rs:155-159
    case MODE_V: n_strips = mcu_y; ybr = 2; cbr = 1; break;       // mcu.rs:160-163
    default: n_strips = (hh + 7) / 8; ybr = 1; cbr = 1; break;    // mcu.rs:164-169
    }
    if (spec && (mode == MODE_H || mode == MODE_HV)) n_strips = (mcu_y + 1) / 2;   // every MCU row
    const uint32_t rows = 8 * h * v;
    const size_t out_chunk = (size_t)w * nc * rows;               // mcu.rs:226
    const size_t capacity = (size_t)(uint16_t)(w + 8) * (size_t)(uint16_t)(hh + 8);  // mcu.rs:198 (u16 add)
    const size_t extra = (mode != MODE_NONE ? 128u : 0u) * (size_t)hh * nc;           // mcu.rs:207
    const size_t avail = (capacity * nc + extra) / out_chunk;
    if (n_strips > avail && !spec) {
        if (img->flags & ZJ_FLAG_PROGRESSIVE) n_strips = (uint32_t)avail;  // mcu_prog.rs:206-209, zip stops
        else return ZJ_ERR_REF_PANIC;                                      // mcu.rs:354, chunks.next().unwrap()
    }
    pl->n_strips = n_strips;
    pl->grid_strips = n_strips;
    pl->rows = rows;
    uint32_t ow, oh;   // the kernels write the stored frame; the orient pass turns it into output_dims
    stored_dims(img, &ow, &oh);
    pl->out_size = (size_t)ow * oh * nc;
    pl->chunk[0] = (size_t)ybr * h * mcu_x * 64;
    pl->chunk[1] = pl->chunk[2] = (size_t)cbr * mcu_x * 64;

    const uint32_t in_cs = img->n_comp == 1 ? ZJ_CS_GRAYSCALE : ZJ_CS_YCBCR;
    const uint32_t oc = img->out_cs;
    uint32_t kind;
    if (oc == ZJ_CS_GRAYSCALE) kind = OUT_GRAY;                                       // worker.rs:115-118
    else if (in_cs == ZJ_CS_YCBCR && oc == ZJ_CS_YCBCR) kind = OUT_YCC;               // worker.rs:120-123
    else if (in_cs == ZJ_CS_YCBCR && (oc == ZJ_CS_RGB || oc == ZJ_CS_RGBA || oc == ZJ_CS_RGBX)) kind = OUT_RGB;  // :125-129
    else kind = OUT_ZERO;                                                             // worker.rs:131-132
    if (spec && kind == OUT_ZERO) {   // one-component input keeps RGB / RGBA / RGBX; every other pair has no stated output
        if (in_cs != ZJ_CS_GRAYSCALE || (oc != ZJ_CS_RGB && oc != ZJ_CS_RGBA && oc != ZJ_CS_RGBX)) return ZJ_ERR_UNSUPPORTED;
        kind = OUT_RGB;
    }
    pl->gray = kind == OUT_GRAY;
    pl->zero_only = kind == OUT_ZERO;
    pl->ncomp_used = kind == OUT_GRAY ? 1u : (kind == OUT_ZERO ? 0u : img->n_comp);  // min(in, out) comps are IDCT'd; unused results are dropped

    DevImage &d = pl->dev;
    d.width = w; d.height = hh; d.nc = (uint32_t)nc; d.out_kind = kind;
    d.mcu_x = mcu_x; d.n_strips = n_strips;
    d.Wp = img->comp[0].width_stride;
    d.W = img->n_comp == 3 ? img->comp[1].width_stride : 0;
    d.stride = w * (uint32_t)nc;
    d.T = 0xffffffffu;
    d.small_width = 0;
    d.hv_avx = (mode == MODE_HV && img->variant == ZJ_VARIANT_X86 && (size_t)16 * d.W >= 500) ? 1u : 0u;  // upsampler/avx2.rs:16
    for (uint32_t z = 0; z < img->n_comp; z++)
        for (int k = 0; k < 32; k++)
            d.qtw[z][k] = (uint32_t)img->comp[z].qt[2 * k] | ((uint32_t)img->comp[z].qt[2 * k + 1] << 24);

    if (scale) {
        // scaled_kernel, for every output colourspace (GRAYSCALE: the luma plane): one MCU row x TS MCU columns per CTA
        d.width = ow; d.height = oh; d.stride = ow * (uint32_t)nc;
        d.n_strips = mcu_y;
        // the real chroma size (rules 1'' and 3''): 4:2:0 chroma blocks are 2 s0 samples wide, every other chroma block s0
        const uint64_t ss = (8u >> scale) * (mode == MODE_HV ? 2u : 1u);
        d.chroma_wh = (uint32_t)((w * ss + 8 * h - 1) / (8 * h)) | (uint32_t)((hh * ss + 8 * v - 1) / (8 * v)) << 16;
        const int tsv[4] = {TS_NONE, TS_H, TS_V, TS_HV};
        d.n_tiles = (mcu_x + tsv[mode] - 1) / tsv[mode];
        pl->grid_tiles = d.n_tiles;
        pl->grid_strips = mcu_y;
        return ZJ_OK;
    }
    if (kind == OUT_GRAY) {
        // ycbcr_to_grayscale (color_convert/scalar.rs:97-112): width_mcu = len / width must equal the strip's row
        // count, otherwise the chunking overruns the strip's output slice and the reference panics (Q7).
        const size_t len = (size_t)rows * d.Wp;
        if (n_strips > 0 && len / w != rows && !spec) return ZJ_ERR_REF_PANIC;   // (no strip, no call, no panic: the output stays zero)
        d.gray_rows_ok = 1;
        d.gray_brows = n_strips * (rows / 8);
        // X86 variant (and SPEC, whose grey output is the X86 luma plane): producer / consumer kernel over pairs of block rows;
        // SCALAR (unclamped DC-only samples) and SPEC | ISLOW (the islow luma plane): gray_kernel
        pl->fast = img->variant != ZJ_VARIANT_SCALAR && !islow && !getenv("ZJ_NO_FAST");
        if (pl->fast) {
            const uint32_t ucols = (d.Wp + 15) / 16;
            d.n_tiles = (ucols + ZF_XU_GRAY - 1) / ZF_XU_GRAY;
            d.tile_q = ucols / d.n_tiles;
            d.tile_r = ucols % d.n_tiles;
            pl->grid_strips = (d.gray_brows + 1) / 2;
        } else {
            d.n_tiles = (d.Wp / 8 + ZJ_THREADS - 1) / ZJ_THREADS;
        }
        pl->grid_tiles = d.n_tiles;
    } else if (spec) {
        // spec_kernel: tiles of exactly TM MCU columns, so that every tile starts on a 16-pixel boundary
        const int tmv[4] = {TM_NONE, TM_H, TM_V, TM_HV};
        d.n_tiles = (mcu_x + tmv[mode] - 1) / tmv[mode];
        d.tile_q = tmv[mode];
        pl->grid_tiles = d.n_tiles;
        return ZJ_OK;
    } else if (kind == OUT_YCC) {
        d.n_norm = w; d.P = 3 * w;
    } else if (kind == OUT_RGB) {
        if (w < 16) {
            if (d.Wp > 16) return ZJ_ERR_REF_PANIC;  // copy_from_slice into [0;16], worker.rs:183
            d.small_width = 1;
        } else {
            const uint32_t E = d.Wp / 16 > 0 ? d.Wp / 16 - 1 : 0;  // worker.rs:171
            d.n_norm = 16 * E;
            d.P = 48 * E;
            if (d.P > d.stride) return ZJ_ERR_REF_PANIC;
            const uint32_t room = d.stride - d.P;
            const uint32_t diff = room < 64 ? 64 - room : 0;       // worker.rs:221
            d.T = d.P > diff ? d.P - diff : 0;                     // worker.rs:223
            if (d.T + 48 > d.stride) return ZJ_ERR_REF_PANIC;
        }
    }
    if (kind != OUT_GRAY) {
        // the fast kernel covers the X86 variant with word-aligned rows; everything else runs the generic kernel
        pl->fast = img->variant == ZJ_VARIANT_X86 && (kind == OUT_RGB || kind == OUT_YCC) && !d.small_width && (d.stride & 3u) == 0 &&
                   (mode != MODE_HV || d.hv_avx) && (reinterpret_cast<uintptr_t>(out) & 3) == 0 && !getenv("ZJ_NO_FAST");
        if (pl->fast) {
            const uint32_t xuv[4] = {ZF_XU_NONE, ZF_XU_H, ZF_XU_V, ZF_XU_HV};
            const uint32_t ucols = (d.Wp + 15) / 16;            // 16-sample unit columns
            d.n_tiles = (ucols + xuv[mode] - 1) / xuv[mode];
            d.tile_q = ucols / d.n_tiles;
            d.tile_r = ucols % d.n_tiles;
        } else {
            const int tmv[4] = {TM_NONE, TM_H, TM_V, TM_HV};
            d.n_tiles = (mcu_x + tmv[mode] - 1) / tmv[mode];
            d.tile_q = mcu_x / d.n_tiles;
            d.tile_r = mcu_x % d.n_tiles;
        }
        pl->grid_tiles = d.n_tiles;
        d.magic_w = d.W ? (((uint64_t)1 << 40) + d.W - 1) / d.W : 0;
    }
    return ZJ_OK;
}

static int check_buffers(const zj_image *img, const Plan &pl, const void *out, size_t out_len)
{
    for (uint32_t z = 0; z < pl.ncomp_used; z++) {
        if (!img->comp[z].coeff) return ZJ_ERR_INVALID_ARG;
        if (img->comp[z].n_i16 < (uint64_t)pl.n_strips * pl.chunk[z]) return ZJ_ERR_SHORT_PLANE;
    }
    if (!out) return ZJ_ERR_INVALID_ARG;
    if (out_len < pl.out_size) return ZJ_ERR_SHORT_OUTPUT;
    return ZJ_OK;
}

// device-resident planes are read with 128-bit accesses: every plane must start on a 16-byte boundary
static int check_device_alignment(const zj_image *img, const Plan &pl)
{
    for (uint32_t z = 0; z < pl.ncomp_used; z++)
        if (reinterpret_cast<uintptr_t>(img->comp[z].coeff) & 15) return ZJ_ERR_INVALID_ARG;
    return ZJ_OK;
}

// ------------------------------------------------------------------------------------------------ batches
struct OrientRun { uint32_t first, count, nc, max_w, max_h; };   // one orient_kernel launch over d_orient[first, first + count)
struct zj_batch {
    int device;
    std::vector<LaunchGroup> groups;
    std::vector<std::pair<uint8_t *, size_t>> zero_only;  // outputs that are just memset (worker.rs:131-132)
    DevImage *d_images;
    size_t n_images;
    // oriented images (ZJ_FLAG_ORIENT_*): reconstructed into `scratch`, owned by the batch, then oriented into their outputs
    std::vector<OrientRun> orient_runs;
    OrientImage *d_orient;
    uint8_t *scratch;
    uint64_t algo_bytes;
    cudaStream_t pool_stream;   // non-null + pooled: descriptors come from the stream-ordered pool of this stream
    bool pooled;
};

// Stream-ordered allocations of this library (descriptor arrays, the consumers' scratch) come from a PRIVATE memory pool per
// device whose release threshold keeps its memory across synchronisations -- by default a pool returns everything to the driver
// at every synchronisation, which would re-map the staging memory on each call.  The process's default pool is left alone
// (other cudaMallocAsync users of the host application keep the behaviour they configured).
static cudaMemPool_t g_pool[64] = {};
static std::mutex g_pool_mu;
static cudaMemPool_t device_pool(int device)
{
    if (device < 0 || device >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(g_pool_mu);
    if (!g_pool[device]) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        cudaMemPool_t pool = nullptr;
        if (cudaMemPoolCreate(&pool, &props) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            g_pool[device] = pool;
        } else cudaGetLastError();
    }
    return g_pool[device];
}
// cudaMallocAsync from the private pool (falls back to the default pool if it could not be created)
static cudaError_t pool_alloc(void **p, size_t bytes, int device, cudaStream_t s)
{
    cudaMemPool_t pool = device_pool(device);
    return pool ? cudaMallocFromPoolAsync(p, bytes, pool, s) : cudaMallocAsync(p, bytes, s);
}
// gives the pool's cached memory back to the driver (zj_release_device_caches)
void zj::trim_pools()
{
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (int d = 0; d < 64; d++) if (g_pool[d]) cudaMemPoolTrimTo(g_pool[d], 0);
    cudaGetLastError();
}

static int set_device(int device)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return ZJ_ERR_NO_DEVICE; }
    if (device < 0 || device >= n) return ZJ_ERR_NO_DEVICE;
    CU(cudaSetDevice(device));
    return ZJ_OK;
}

extern "C" {

int zj_gpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

size_t zj_output_size(const zj_image *img)
{
    Plan pl;
    int rc = plan_image(img, &pl);
    if (rc != ZJ_OK && rc != ZJ_ERR_REF_PANIC) return 0;
    uint32_t w, h;
    output_dims(img, &w, &h);
    return (size_t)w * h * num_components(img->out_cs);
}

int zj_validate_image(const zj_image *img)
{
    Plan pl;
    int rc = plan_image(img, &pl);
    if (rc != ZJ_OK) return rc;
    for (uint32_t z = 0; z < pl.ncomp_used; z++)
        if (img->comp[z].n_i16 < (uint64_t)pl.n_strips * pl.chunk[z]) return ZJ_ERR_SHORT_PLANE;
    return ZJ_OK;
}

// `pooled`: allocate / upload the descriptors in stream order on `ps` (no device-wide synchronisation: cudaMalloc and
// above all cudaFree serialise every thread that feeds the device, which is what zj_decode_batch's workers are)
// `regions` (may be NULL): for an oriented image with regions[i].w != 0, only that rectangle of its stored frame is oriented, and
// out_dev[i] receives it (regions[i].w * regions[i].h * nc bytes, in the displayed frame)
static int batch_create_impl(int device, const zj_image *imgs, size_t n, uint8_t *const *out_dev, const size_t *out_len, zj_batch **plan,
                             bool pooled, cudaStream_t ps, const zj_roi *regions = nullptr);

int zj_batch_create(int device, const zj_image *imgs, size_t n, uint8_t *const *out_dev, const size_t *out_len, zj_batch **plan)
{
    return batch_create_impl(device, imgs, n, out_dev, out_len, plan, false, nullptr);
}

// device memory for the batch's own arrays: from the stream-ordered pool on `ps` (pooled) or cudaMalloc
static cudaError_t batch_alloc(void **p, size_t bytes, bool pooled, int device, cudaStream_t ps)
{
    return pooled ? pool_alloc(p, bytes, device, ps) : cudaMalloc(p, bytes);
}
static void batch_free(void *p, bool pooled, cudaStream_t ps)
{
    if (!p) return;
    if (pooled) cudaFreeAsync(p, ps); else cudaFree(p);
}

static int batch_create_impl(int device, const zj_image *imgs, size_t n, uint8_t *const *out_dev, const size_t *out_len, zj_batch **plan,
                             bool pooled, cudaStream_t ps, const zj_roi *regions)
{
    if (!plan) return ZJ_ERR_INVALID_ARG;
    *plan = nullptr;
    if ((!imgs || !out_dev || !out_len) && n) return ZJ_ERR_INVALID_ARG;
    int rc = set_device(device);
    if (rc) return rc;
    std::vector<Plan> plans(n);
    std::vector<OrientImage> orient;      // the oriented images' second pass, src = their offset into the scratch buffer for now
    size_t scratch_bytes = 0;
    for (size_t i = 0; i < n; i++) {
        rc = plan_image(&imgs[i], &plans[i], out_dev[i]);
        if (rc) return rc;
        const bool region = plans[i].orient && regions && regions[i].w;
        rc = check_buffers(&imgs[i], plans[i], out_dev[i], region ? SIZE_MAX : out_len[i]);
        if (rc) return rc;
        rc = check_device_alignment(&imgs[i], plans[i]);
        if (rc) return rc;
        for (int z = 0; z < 3; z++) plans[i].dev.coeff[z] = (uint32_t)z < plans[i].ncomp_used ? imgs[i].comp[z].coeff : nullptr;
        plans[i].dev.out = out_dev[i];
        if (plans[i].orient) {
            OrientImage oi{};
            const uint32_t nc = plans[i].dev.nc;
            uint32_t w, h;
            stored_dims(&imgs[i], &w, &h);
            const zj_roi r = region ? regions[i] : zj_roi{0, 0, w, h};
            if ((uint64_t)r.x + r.w > w || (uint64_t)r.y + r.h > h || r.h == 0) return ZJ_ERR_INVALID_ARG;
            if (out_len[i] < (size_t)r.w * r.h * nc) return ZJ_ERR_SHORT_OUTPUT;
            oi.src = reinterpret_cast<const uint8_t *>(scratch_bytes + (size_t)r.y * w * nc + (size_t)r.x * nc);
            oi.dst = out_dev[i];
            oi.pitch = w * nc;
            oi.w = r.w; oi.h = r.h;
            oi.orient = (uint32_t)plans[i].orient;
            oi.nc = nc;
            orient.push_back(oi);
            plans[i].dev.out = reinterpret_cast<uint8_t *>(scratch_bytes);
            scratch_bytes += (plans[i].out_size + 255) & ~(size_t)255;
        }
    }
    zj_batch *b = new zj_batch();
    b->device = device;
    b->d_images = nullptr;
    b->n_images = 0;
    b->algo_bytes = 0;
    b->d_orient = nullptr;
    b->scratch = nullptr;
    b->pooled = pooled;
    b->pool_stream = ps;
    if (scratch_bytes) {
        cudaError_t e = batch_alloc((void **)&b->scratch, scratch_bytes, pooled, device, ps);
        if (e != cudaSuccess) { delete b; return cuda_fail(e, "cudaMalloc(orientation scratch)"); }
        for (size_t i = 0; i < n; i++)
            if (plans[i].orient) plans[i].dev.out = b->scratch + reinterpret_cast<uintptr_t>(plans[i].dev.out);
        for (OrientImage &oi : orient) oi.src = b->scratch + reinterpret_cast<uintptr_t>(oi.src);
        // one launch per bytes-per-pixel class
        std::stable_sort(orient.begin(), orient.end(), [](const OrientImage &a, const OrientImage &c) { return a.nc < c.nc; });
    }
    // group by kernel: (scale, gray, fast, mode, variant, IDCT); stable so images keep their relative order
    std::vector<size_t> order;
    for (size_t i = 0; i < n; i++) {
        if (plans[i].zero_only) b->zero_only.push_back({out_dev[i], plans[i].out_size});
        else order.push_back(i);
        b->algo_bytes += plans[i].out_size;
        for (uint32_t z = 0; z < plans[i].ncomp_used; z++) b->algo_bytes += (uint64_t)plans[i].n_strips * plans[i].chunk[z] * 2;
    }
    auto key = [&](size_t i) {
        return plans[i].scale * 128 + plans[i].gray * 64 + plans[i].fast * 32 + plans[i].mode * 8 + plans[i].islow * 4 + plans[i].variant;
    };
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t c) { return key(a) < key(c); });
    std::vector<DevImage> host(order.size());
    for (size_t k = 0; k < order.size(); k++) host[k] = plans[order[k]].dev;
    for (size_t k = 0; k < order.size();) {
        size_t e = k;
        LaunchGroup g{};
        g.gray = plans[order[k]].gray; g.mode = plans[order[k]].mode; g.variant = plans[order[k]].variant; g.fast = plans[order[k]].fast;
        g.islow = plans[order[k]].islow;
        g.scale = plans[order[k]].scale;
        g.first = (uint32_t)k;
        while (e < order.size() && key(order[e]) == key(order[k]) && e - k < 65535) {
            g.max_tiles = std::max(g.max_tiles, plans[order[e]].grid_tiles);
            g.max_strips = std::max(g.max_strips, plans[order[e]].grid_strips);
            e++;
        }
        g.count = (uint32_t)(e - k);
        b->groups.push_back(g);
        k = e;
    }
    for (size_t k = 0; k < orient.size();) {
        OrientRun run{(uint32_t)k, 0, orient[k].nc, 0, 0};
        for (; k < orient.size() && orient[k].nc == run.nc && run.count < 65535; k++, run.count++) {
            run.max_w = std::max(run.max_w, orient[k].w);
            run.max_h = std::max(run.max_h, orient[k].h);
        }
        b->orient_runs.push_back(run);
    }
    // (pageable sources: the async copies return once the data sits in the driver's staging buffer)
    auto upload = [&](void **dst, const void *src, size_t bytes, const char *what) -> int {
        cudaError_t e = batch_alloc(dst, bytes, pooled, device, ps);
        if (e != cudaSuccess) { *dst = nullptr; return cuda_fail(e, what); }
        e = pooled ? cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ps) : cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
        return e == cudaSuccess ? ZJ_OK : cuda_fail(e, what);
    };
    if (!host.empty()) {
        rc = upload((void **)&b->d_images, host.data(), host.size() * sizeof(DevImage), "cudaMemcpy(descriptors)");
        b->n_images = host.size();
    }
    if (rc == ZJ_OK && !orient.empty()) rc = upload((void **)&b->d_orient, orient.data(), orient.size() * sizeof(OrientImage), "cudaMemcpy(orientation descriptors)");
    if (rc != ZJ_OK) { zj_batch_destroy(b); return rc; }
    *plan = b;
    return ZJ_OK;
}

int zj_batch_run(zj_batch *b, void *stream)
{
    if (!b) return ZJ_ERR_INVALID_ARG;
    int rc = set_device(b->device);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    for (auto &z : b->zero_only) CU(cudaMemsetAsync(z.first, 0, z.second, s));
    for (auto &g : b->groups) {
        CU(launch_group(b->d_images, g, s));
        g_launches.fetch_add(1);
    }
    for (const OrientRun &r : b->orient_runs) {
        CU(launch_orient(b->d_orient + r.first, r.count, r.nc, r.max_w, r.max_h, s));
        g_launches.fetch_add(1);
    }
    return ZJ_OK;
}

int zj_batch_launches(const zj_batch *b) { return b ? (int)(b->groups.size() + b->orient_runs.size()) : 0; }
uint64_t zj_batch_algorithmic_bytes(const zj_batch *b) { return b ? b->algo_bytes : 0; }

void zj_batch_destroy(zj_batch *b)
{
    if (!b) return;
    if (b->d_images || b->d_orient || b->scratch) {
        cudaSetDevice(b->device);
        batch_free(b->d_images, b->pooled, b->pool_stream);
        batch_free(b->d_orient, b->pooled, b->pool_stream);
        batch_free(b->scratch, b->pooled, b->pool_stream);
    }
    delete b;
}

int zj_gpu_reconstruct_device(int device, void *stream, const zj_image *imgs, size_t n, uint8_t *const *out_dev, const size_t *out_len)
{
    zj_batch *b = nullptr;
    int rc = zj_batch_create(device, imgs, n, out_dev, out_len, &b);
    if (rc) return rc;
    rc = zj_batch_run(b, stream);
    // the descriptor array must outlive the kernels
    if (rc == ZJ_OK) { cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream); if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize"); }
    zj_batch_destroy(b);
    return rc;
}

}  // extern "C"

// ------------------------------------------------------------------------------------- device-side consumers
// (The header gives the zj_* functions below their C linkage; the templates this part shares cannot have it.)
void zj_output_desc_default(zj_output_desc *d)
{
    if (!d) return;
    memset(d, 0, sizeof(*d));
    for (int c = 0; c < 4; c++) d->inv_std[c] = 1.0f;
}

static int desc_check(const zj_output_desc *d)
{
    if (!d || d->layout > ZJ_LAYOUT_CHW || d->dtype > ZJ_DTYPE_F32 || d->scale_log2 > 1 || (d->channels != 0 && d->channels != 3)) return ZJ_ERR_INVALID_ARG;
    return ZJ_OK;
}

int zj_output_desc_is_default(const zj_output_desc *d)
{
    return d && d->layout == ZJ_LAYOUT_HWC && d->dtype == ZJ_DTYPE_U8 && d->scale_log2 == 0 && d->channels == 0;
}

static size_t dtype_size(uint32_t dt) { return dt == ZJ_DTYPE_U8 ? 1 : (dt == ZJ_DTYPE_F16 ? 2 : 4); }

// channels written per pixel of nc source bytes (channels = 3 drops the fourth byte)
static uint32_t out_channels(const zj_output_desc *d, uint32_t nc) { return (d->channels == 3 && nc == 4) ? 3u : nc; }

static int conv_shape(uint32_t width, uint32_t height, uint32_t nc, const zj_output_desc *d, uint32_t *ow, uint32_t *oh, uint32_t *oc)
{
    int rc = desc_check(d);
    if (rc) return rc;
    if (nc != 1 && nc != 3 && nc != 4) return ZJ_ERR_INVALID_ARG;
    *ow = width >> d->scale_log2;
    *oh = height >> d->scale_log2;
    *oc = out_channels(d, nc);
    return ZJ_OK;
}

size_t zj::convert_size(uint32_t width, uint32_t height, uint32_t nc, const zj_output_desc *d)
{
    uint32_t ow, oh, oc;
    return conv_shape(width, height, nc, d, &ow, &oh, &oc) == ZJ_OK ? (size_t)ow * oh * oc * dtype_size(d->dtype) : 0;
}

int zj_consumer_output_shape(const zj_image *img, const zj_output_desc *d, uint32_t *out_w, uint32_t *out_h, uint32_t *out_c)
{
    if (!img || !out_w || !out_h || !out_c) return ZJ_ERR_INVALID_ARG;
    uint32_t w, h;
    output_dims(img, &w, &h);
    return conv_shape(w, h, (uint32_t)num_components(img->out_cs), d, out_w, out_h, out_c);
}

size_t zj_consumer_output_size(const zj_image *img, const zj_output_desc *d)
{
    if (!img || zj_output_size(img) == 0) return 0;
    uint32_t w, h;
    output_dims(img, &w, &h);
    return convert_size(w, h, (uint32_t)num_components(img->out_cs), d);
}

// One launch of the second pass (the consumer for ConvImage, the resize for ResizeImage) per run of consecutive images with the
// same bytes per pixel, at most 65535 images each: the image index is gridDim.z.  dev / host: the same descriptors in device /
// host memory, nc[i]: image i's bytes per pixel, r: the resize's parameters.
template <class Img>
static int launch_runs(const Img *dev, const Img *host, const uint32_t *nc, size_t n, const zj_output_desc &d, const zj_resize *r, cudaStream_t s)
{
    constexpr bool convert = std::is_same<Img, ConvImage>::value;
    for (size_t k = 0, k1 = 0; k < n; k = k1) {
        uint32_t mw = 0, mh = 0;   // the consumer's grid covers the run's largest output
        for (k1 = k; k1 < n && nc[k1] == nc[k] && k1 - k < 65535; k1++)
            if constexpr (convert) { mw = std::max(mw, host[k1].ow); mh = std::max(mh, host[k1].oh); }
        cudaError_t e;
        if constexpr (convert) {
            if (!mw || !mh) continue;   // nothing to write (half size of images one pixel wide or high)
            e = launch_convert(dev + k, (uint32_t)(k1 - k), nc[k], mw, mh, d, s);
        } else if (pil_filter(r->filter)) {
            int device = 0, launches = 0;
            e = cudaGetDevice(&device);
            if (e == cudaSuccess) e = launch_pil_resize(host + k, (uint32_t)(k1 - k), nc[k], d, *r, device, s, &launches);
            g_launches.fetch_add(launches);
            if (e != cudaSuccess) return cuda_fail(e, "PIL resize launch");
            continue;
        } else {
            e = launch_resize(dev + k, (uint32_t)(k1 - k), nc[k], d, *r, s);
        }
        g_launches.fetch_add(1);
        if (e != cudaSuccess) return cuda_fail(e, convert ? "consumer launch" : "resize launch");
    }
    return ZJ_OK;
}

// Copies the descriptors host[0, n) into a stream-ordered pool allocation, calls use(that copy) and frees it, all in the order of s
template <class Img, class Use>
static int with_device_copy(const Img *host, size_t n, int device, cudaStream_t s, Use use)
{
    Img *dev = nullptr;
    CU(pool_alloc((void **)&dev, n * sizeof(Img), device, s));
    // (pageable source: the async copy returns once the data sits in the driver's staging buffer)
    const cudaError_t e = cudaMemcpyAsync(dev, host, n * sizeof(Img), cudaMemcpyHostToDevice, s);
    const int rc = e == cudaSuccess ? use(static_cast<const Img *>(dev)) : cuda_fail(e, "cudaMemcpyAsync(descriptors)");
    cudaFreeAsync(dev, s);
    return rc;
}

// The second pass over n images whose u8 pixels are already in device memory
template <class Img>
static int run_pass(int device, cudaStream_t s, const Img *host, const uint32_t *nc, size_t n, const zj_output_desc &d, const zj_resize *r)
{
    return with_device_copy(host, n, device, s, [&](const Img *dev) { return launch_runs(dev, host, nc, n, d, r, s); });
}

int zj_gpu_convert_device(int device, void *stream, const uint8_t *src_dev, uint32_t width, uint32_t height, uint32_t nc,
                          const zj_output_desc *d, void *dst_dev, size_t dst_len)
{
    ConvImage ci{};
    int rc = conv_shape(width, height, nc, d, &ci.ow, &ci.oh, &ci.oc);
    if (rc) return rc;
    if (!src_dev || !dst_dev) return ZJ_ERR_INVALID_ARG;
    if (dst_len < convert_size(width, height, nc, d)) return ZJ_ERR_SHORT_OUTPUT;
    rc = set_device(device);
    if (rc) return rc;
    if (ci.ow == 0 || ci.oh == 0) return ZJ_OK;
    ci.src = src_dev; ci.dst = dst_dev; ci.width = width; ci.height = height; ci.nc = nc;
    return run_pass(device, (cudaStream_t)stream, &ci, &nc, 1, *d, nullptr);
}

// Sub-batch budget of the u8 intermediate (scratch memory of the call).  Measured on 128 4K images (profiles/README.md):
// sub-batches small enough to stay in the 126 MB L2 between the two kernels (48 MB: 245 GP/s) lose more to under-filled
// launches than the cache saves; 320 MB: 292 GP/s, the whole batch at once: 320 GP/s.  1 GB keeps the launches large and the
// scratch bounded.
static size_t consumer_chunk_bytes()
{
    static const size_t v = [] {
        const char *e = getenv("ZJ_CONSUMER_CHUNK_MB");
        long mb = e ? atol(e) : 1024;
        if (mb < 1) mb = 1;
        return (size_t)mb << 20;
    }();
    return v;
}

// Sub-batches of consecutive images whose u8 intermediates, and the scratch their zj_batch allocates for them (oriented images),
// fit consumer_chunk_bytes() together (at least one image each)
struct ConsumerChunk { size_t first, count, bytes, charged; };
// places image i's intermediate of `bytes` bytes in the last sub-batch or a new one, charging `extra` more bytes to its budget;
// returns its offset in the scratch buffer
static size_t chunk_place(std::vector<ConsumerChunk> &chunks, size_t i, size_t bytes, size_t extra = 0)
{
    const size_t padded = (bytes + 255) & ~(size_t)255, charge = padded + ((extra + 255) & ~(size_t)255);
    if (chunks.empty() || chunks.back().charged + charge > consumer_chunk_bytes()) chunks.push_back({i, 0, 0, 0});
    const size_t off = chunks.back().bytes;
    chunks.back().bytes += padded;
    chunks.back().charged += charge;
    chunks.back().count++;
    return off;
}

// Frees the scratch an oriented image's batch reconstructs into, in the order of the pooled batch's stream: once its launches
// are queued, the next sub-batch may take its place
static void batch_drop_scratch(zj_batch *b)
{
    if (b && b->scratch && b->pooled) { cudaFreeAsync(b->scratch, b->pool_stream); b->scratch = nullptr; }
}

// The planes route of the second pass: subs[i] is reconstructed into u8_size[i] bytes of a stream-ordered scratch buffer, in
// sub-batches that take turns in it, and each sub-batch is followed by the pass over its images.  build(i, image i's u8
// pixels) gives image i's descriptor; the descriptors are uploaded once.  regions (may be NULL): the rectangles of oriented images
// that are oriented into their u8_size[i] bytes (batch_create_impl).  Returns after `s` has drained.
template <class Build>
static int reconstruct_then(int device, cudaStream_t s, const zj_image *subs, const std::vector<size_t> &u8_size, const uint32_t *nc,
                            const zj_output_desc &d, const zj_resize *r, Build build, const zj_roi *regions = nullptr)
{
    using Img = decltype(build(0, nullptr));
    const size_t n = u8_size.size();
    std::vector<ConsumerChunk> chunks;
    std::vector<size_t> u8_off(n);
    size_t scratch_bytes = 0;
    for (size_t i = 0; i < n; i++) {
        // (an oriented image is reconstructed whole into its batch's own scratch, then oriented into its u8_size[i] bytes)
        u8_off[i] = chunk_place(chunks, i, u8_size[i], image_orient(&subs[i]) ? zj_output_size(&subs[i]) : 0);
        scratch_bytes = std::max(scratch_bytes, chunks.back().bytes);
    }
    uint8_t *scratch = nullptr;
    CU(pool_alloc((void **)&scratch, scratch_bytes, device, s));
    std::vector<Img> host(n);
    for (size_t i = 0; i < n; i++) host[i] = build(i, scratch + u8_off[i]);
    const int rc = with_device_copy(host.data(), n, device, s, [&](const Img *dev) {
        int rc = ZJ_OK;
        std::vector<zj_batch *> batches;
        for (size_t c = 0; c < chunks.size() && rc == ZJ_OK; c++) {
            const ConsumerChunk &ch = chunks[c];
            std::vector<uint8_t *> outs(ch.count);
            for (size_t k = 0; k < ch.count; k++) outs[k] = scratch + u8_off[ch.first + k];
            zj_batch *b = nullptr;
            rc = batch_create_impl(device, subs + ch.first, ch.count, outs.data(), u8_size.data() + ch.first, &b, true, s,
                                   regions ? regions + ch.first : nullptr);
            if (rc) break;
            batches.push_back(b);
            rc = zj_batch_run(b, s);
            batch_drop_scratch(b);
            if (rc == ZJ_OK) rc = launch_runs(dev + ch.first, host.data() + ch.first, nc + ch.first, ch.count, d, r, s);
        }
        // the descriptor arrays and the scratch must outlive the kernels
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess && rc == ZJ_OK) rc = cuda_fail(e, "cudaStreamSynchronize");
        for (zj_batch *b : batches) zj_batch_destroy(b);
        return rc;
    });
    cudaFreeAsync(scratch, s);
    return rc;
}

int zj_gpu_reconstruct_device_ex(int device, void *stream, const zj_image *imgs, size_t n, const zj_output_desc *d,
                                 void *const *out_dev, const size_t *out_len)
{
    int rc = desc_check(d);
    if (rc) return rc;
    if (zj_output_desc_is_default(d)) return zj_gpu_reconstruct_device(device, stream, imgs, n, reinterpret_cast<uint8_t *const *>(out_dev), out_len);
    if ((!imgs || !out_dev || !out_len) && n) return ZJ_ERR_INVALID_ARG;
    rc = set_device(device);
    if (rc) return rc;
    std::vector<ConvImage> conv(n);
    std::vector<uint32_t> nc(n);
    std::vector<size_t> u8_size(n);
    for (size_t i = 0; i < n; i++) {
        u8_size[i] = zj_output_size(&imgs[i]);
        if (u8_size[i] == 0) { rc = zj_validate_image(&imgs[i]); return rc ? rc : (int)ZJ_ERR_INVALID_ARG; }
        ConvImage &ci = conv[i];
        output_dims(&imgs[i], &ci.width, &ci.height);
        ci.nc = nc[i] = (uint32_t)num_components(imgs[i].out_cs);
        rc = conv_shape(ci.width, ci.height, ci.nc, d, &ci.ow, &ci.oh, &ci.oc);
        if (rc) return rc;
        if (!out_dev[i]) return ZJ_ERR_INVALID_ARG;
        if (out_len[i] < convert_size(ci.width, ci.height, ci.nc, d)) return ZJ_ERR_SHORT_OUTPUT;
        ci.dst = out_dev[i];
    }
    if (n == 0) return ZJ_OK;
    return reconstruct_then(device, (cudaStream_t)stream, imgs, u8_size, nc.data(), *d, nullptr, [&](size_t i, const uint8_t *u8) {
        conv[i].src = u8;
        return conv[i];
    });
}

// ------------------------------------------------------------------------------------- cropped, resized batch tensors
static int resize_check(const zj_output_desc *d, const zj_resize *r)
{
    int rc = desc_check(d);
    if (rc) return rc;
    // (sizes up to 65535, as for images: the kernels' window products fit 32 bits)
    if (d->scale_log2 != 0 || !r || r->out_w == 0 || r->out_h == 0 || r->out_w > 65535 || r->out_h > 65535)
        return ZJ_ERR_INVALID_ARG;
    if (!pil_filter(r->filter) && (r->filter > ZJ_FILTER_BILINEAR || r->reserved != 0)) return ZJ_ERR_INVALID_ARG;
    return ZJ_OK;
}

size_t zj_resize_slot_size(const zj_output_desc *d, const zj_resize *r, uint32_t nc)
{
    if (resize_check(d, r) != ZJ_OK || (nc != 1 && nc != 3 && nc != 4)) return 0;
    return (size_t)r->out_w * r->out_h * out_channels(d, nc) * dtype_size(d->dtype);
}

// *out = the crop of a width x height image that `roi` names (NULL = the whole image)
static int roi_resolve(const zj_roi *roi, uint32_t width, uint32_t height, zj_roi *out)
{
    if (!roi) { *out = {0, 0, width, height}; return ZJ_OK; }
    if (roi->w == 0 || roi->h == 0 || (uint64_t)roi->x + roi->w > width || (uint64_t)roi->y + roi->h > height) return ZJ_ERR_INVALID_ARG;
    *out = *roi;
    return ZJ_OK;
}

int zj::resize_admit(const zj_output_desc *d, const zj_resize *r, uint32_t slot_nc, const zj_roi *roi, uint32_t width, uint32_t height,
                     uint32_t nc, zj_roi *crop)
{
    if (out_channels(d, nc) != out_channels(d, slot_nc)) return ZJ_ERR_INVALID_ARG;   // one tensor: one channel count
    int rc = roi_resolve(roi, width, height, crop);
    PilGeometry g;
    if (rc == ZJ_OK && pil_filter(r->filter)) rc = pil_geometry(*r, crop->w, crop->h, &g);
    return rc;
}

// The crop rows [*first, *end) the resize reads: all of them, or (PIL filters) the rows of the window's vertical taps
static void crop_rows(const zj_resize &r, const zj_roi &crop, uint32_t *first, uint32_t *end)
{
    PilGeometry g;
    if (pil_filter(r.filter) && pil_geometry(r, crop.w, crop.h, &g) == ZJ_OK) { *first = g.y0; *end = g.y1; }
    else { *first = 0; *end = crop.h; }
}

// src: the width x height (rows of it) u8 image the crop lies in, from its row `row0` on; row0 is the row of the crop's first
// row the resize reads (crop_rows)
static ResizeImage resize_image(const uint8_t *src, uint32_t width, uint32_t height, uint32_t nc, uint32_t row0, const zj_roi &roi, void *dst,
                                const zj_resize &r)
{
    ResizeImage ri{};
    ri.pitch = width * nc;
    ri.lo = src;
    ri.hi = src + (size_t)height * ri.pitch;
    ri.src = src + (size_t)row0 * ri.pitch + (size_t)roi.x * nc;
    ri.dst = dst;
    ri.w = roi.w; ri.h = roi.h;
    ri.sx = (float)roi.w / (float)r.out_w;   // IEEE single-precision division, as the kernel's other operations
    ri.sy = (float)roi.h / (float)r.out_h;
    return ri;
}

int zj_image_rows(const zj_image *img, uint32_t row_begin, uint32_t row_end, zj_image *sub, uint32_t *sub_row0)
{
    Plan pl;
    int rc = plan_image(img, &pl);
    if (rc) return rc;
    uint32_t w, h;
    output_dims(img, &w, &h);
    if (!sub || !sub_row0 || row_begin >= row_end || row_end > h) return ZJ_ERR_INVALID_ARG;
    // strips [s0, s1): the strips the rows fall in; rows at or below the last strip belong to the range that ends with it
    const uint32_t ns = pl.n_strips;
    const uint32_t s0 = ns ? std::min(row_begin / pl.rows, ns - 1) : 0;
    const uint32_t s1 = ns ? std::min((row_end + pl.rows - 1) / pl.rows, ns) : 0;
    // A virtual image is planned like any image, so the output-capacity rule (mcu.rs:198-209) applies to it on its own: a short
    // range at the bottom (one row of a last strip) can be refused where the whole image is not.  Such a range starts at earlier
    // strips instead; an image that cannot be cut at all (ZJ_ERR_UNSUPPORTED) is returned whole.
    for (uint32_t b = s0;; b--) {
        rc = zj_image_strip_range(img, b, s1, sub, nullptr, nullptr, nullptr);
        if (rc == ZJ_OK) { *sub_row0 = row_begin - b * pl.rows; return ZJ_OK; }
        if (rc == ZJ_ERR_UNSUPPORTED || (rc == ZJ_ERR_REF_PANIC && b == 0)) break;
        if (rc != ZJ_ERR_REF_PANIC) return rc;
    }
    *sub = *img;
    *sub_row0 = row_begin;
    return ZJ_OK;
}

int zj_gpu_resize_device(int device, void *stream, const uint8_t *src_dev, uint32_t width, uint32_t height, uint32_t nc, const zj_roi *roi,
                         const zj_output_desc *d, const zj_resize *r, void *dst_dev, size_t dst_len)
{
    const size_t slot = zj_resize_slot_size(d, r, nc);
    if (slot == 0 || width == 0 || height == 0 || width > 65535 || height > 65535 || !src_dev || !dst_dev) return ZJ_ERR_INVALID_ARG;
    zj_roi crop;
    int rc = resize_admit(d, r, nc, roi, width, height, nc, &crop);
    if (rc) return rc;
    if (dst_len < slot) return ZJ_ERR_SHORT_OUTPUT;
    rc = set_device(device);
    if (rc) return rc;
    uint32_t first, end;
    crop_rows(*r, crop, &first, &end);
    const ResizeImage ri = resize_image(src_dev, width, height, nc, crop.y + first, crop, dst_dev, *r);
    return run_pass(device, (cudaStream_t)stream, &ri, &nc, 1, *d, r);
}

int zj_gpu_reconstruct_device_resized(int device, void *stream, const zj_image *imgs, size_t n, const zj_roi *rois, const zj_output_desc *d,
                                      const zj_resize *r, void *out_dev, size_t out_len)
{
    int rc = resize_check(d, r);
    if (rc) return rc;
    if ((!imgs || !out_dev) && n) return ZJ_ERR_INVALID_ARG;
    // per image: the crop, the strips that hold the rows the resize reads and the size of their u8 pixels.  Of an oriented image
    // only the rectangle that those rows and the crop's columns come from is oriented, into a buffer of its own: region[i].
    std::vector<zj_image> subs(n);
    std::vector<zj_roi> crops(n), region(n, zj_roi{0, 0, 0, 0});
    std::vector<uint32_t> row0(n), nc(n), width(n);
    std::vector<size_t> u8_size(n);
    for (size_t i = 0; i < n; i++) {
        if (zj_output_size(&imgs[i]) == 0) { rc = zj_validate_image(&imgs[i]); return rc ? rc : (int)ZJ_ERR_INVALID_ARG; }
        nc[i] = (uint32_t)num_components(imgs[i].out_cs);
        uint32_t height;
        output_dims(&imgs[i], &width[i], &height);
        rc = resize_admit(d, r, nc[0], rois ? &rois[i] : nullptr, width[i], height, nc[i], &crops[i]);
        if (rc) return rc;
        uint32_t first, end;
        crop_rows(*r, crops[i], &first, &end);
        if (const uint32_t t = image_orient(&imgs[i])) {
            uint32_t sw, sh;
            stored_dims(&imgs[i], &sw, &sh);
            // displayed columns [crop.x, crop.x + crop.w) x rows [crop.y + first, crop.y + end): back through the swap and the mirrors
            uint32_t xa = crops[i].x, xb = crops[i].x + crops[i].w, ya = crops[i].y + first, yb = crops[i].y + end;
            if (orient_swap(t)) { std::swap(xa, ya); std::swap(xb, yb); }
            if (orient_flip_x(t)) { const uint32_t a = sw - xb; xb = sw - xa; xa = a; }
            if (orient_flip_y(t)) { const uint32_t a = sh - yb; yb = sh - ya; ya = a; }
            region[i] = zj_roi{xa, ya, xb - xa, yb - ya};
            subs[i] = imgs[i];
            width[i] = crops[i].w;       // the buffer holds the crop's columns ...
            row0[i] = 0;                 // ... and its rows [first, end)
            crops[i].x = 0;
            u8_size[i] = (size_t)region[i].w * region[i].h * nc[i];
            continue;
        }
        rc = zj_image_rows(&imgs[i], crops[i].y + first, crops[i].y + end, &subs[i], &row0[i]);
        if (rc) return rc;
        u8_size[i] = zj_output_size(&subs[i]);
        if (u8_size[i] == 0) { rc = zj_validate_image(&subs[i]); return rc ? rc : (int)ZJ_ERR_INVALID_ARG; }
    }
    const size_t slot = n ? zj_resize_slot_size(d, r, nc[0]) : 0;
    if (n && out_len / slot < n) return ZJ_ERR_SHORT_OUTPUT;
    rc = set_device(device);
    if (rc) return rc;
    if (n == 0) return ZJ_OK;
    return reconstruct_then(device, (cudaStream_t)stream, subs.data(), u8_size, nc.data(), *d, r, [&](size_t i, const uint8_t *u8) {
        uint32_t sub_w, sub_h;
        output_dims(&subs[i], &sub_w, &sub_h);
        if (region[i].w) sub_h = (uint32_t)(u8_size[i] / ((size_t)width[i] * nc[i]));
        return resize_image(u8, width[i], sub_h, nc[i], row0[i], crops[i], static_cast<uint8_t *>(out_dev) + i * slot, *r);
    }, region.data());
}

// ------------------------------------------------------------------------------------- the JPEG-bytes route's second pass
int zj::scratch_alloc(void **p, size_t bytes, int device, void *stream)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(pool_alloc(p, bytes, device, (cudaStream_t)stream));
    return ZJ_OK;
}
void zj::scratch_free(void *p, void *stream) { if (p) cudaFreeAsync(p, (cudaStream_t)stream); }

int zj::convert_many(int device, void *stream, const U8Image *imgs, size_t n, const zj_output_desc *d)
{
    int rc = desc_check(d);
    if (rc) return rc;
    rc = set_device(device);
    if (rc) return rc;
    if (n == 0) return ZJ_OK;
    std::vector<ConvImage> conv(n);
    std::vector<uint32_t> nc(n);
    for (size_t i = 0; i < n; i++) {
        ConvImage &ci = conv[i];
        ci.src = imgs[i].src; ci.dst = imgs[i].dst; ci.width = imgs[i].width; ci.height = imgs[i].height; ci.nc = nc[i] = imgs[i].nc;
        rc = conv_shape(ci.width, ci.height, ci.nc, d, &ci.ow, &ci.oh, &ci.oc);
        if (rc) return rc;
    }
    return run_pass(device, (cudaStream_t)stream, conv.data(), nc.data(), n, *d, nullptr);
}

// (the crops, channel counts and resized sizes were admitted by the caller: resize_admit)
int zj::resize_many(int device, void *stream, const U8Image *imgs, size_t n, const zj_output_desc *d, const zj_resize *r)
{
    int rc = resize_check(d, r);
    if (rc) return rc;
    rc = set_device(device);
    if (rc) return rc;
    if (n == 0) return ZJ_OK;
    std::vector<ResizeImage> ri(n);
    std::vector<uint32_t> nc(n);
    for (size_t i = 0; i < n; i++) {
        nc[i] = imgs[i].nc;
        uint32_t first, end;
        crop_rows(*r, imgs[i].crop, &first, &end);
        ri[i] = resize_image(imgs[i].src, imgs[i].width, imgs[i].height, nc[i], imgs[i].crop.y + first, imgs[i].crop, imgs[i].dst, *r);
    }
    return run_pass(device, (cudaStream_t)stream, ri.data(), nc.data(), n, *d, r);
}

// Staging state of zj_gpu_reconstruct_submit, leased per host thread (see there); the idle ones are what
// zj_release_device_caches frees.
constexpr int ZJ_NS = 3;   // staging streams per device: the sub-batches of a call take turns on them
struct StreamCache {
    cudaStream_t s[64][ZJ_NS] = {};
    uint8_t *buf[64][ZJ_NS] = {};
    size_t cap[64][ZJ_NS] = {};
};
struct CachePool {
    std::mutex mu;
    std::vector<StreamCache *> idle;
};
static CachePool g_stream_pool;

// frees the streams and device staging buffers of every cache no thread holds (the exported entry point is
// zj_release_device_caches in zj_host_decoder.cpp)
void zj::release_stream_caches()
{
    std::vector<StreamCache *> drop;
    {
        std::lock_guard<std::mutex> lock(g_stream_pool.mu);
        drop.swap(g_stream_pool.idle);
    }
    int prev = -1;
    cudaGetDevice(&prev);
    for (StreamCache *c : drop) {
        for (int dev = 0; dev < 64; dev++) {
            bool any = false;
            for (int k = 0; k < ZJ_NS; k++) any = any || c->s[dev][k] || c->buf[dev][k];
            if (!any || cudaSetDevice(dev) != cudaSuccess) continue;
            for (int k = 0; k < ZJ_NS; k++) {
                if (c->s[dev][k]) cudaStreamSynchronize(c->s[dev][k]);
                if (c->buf[dev][k]) cudaFree(c->buf[dev][k]);
                if (c->s[dev][k]) cudaStreamDestroy(c->s[dev][k]);
            }
        }
        delete c;
    }
    if (prev >= 0) cudaSetDevice(prev);
    cudaGetLastError();
}

extern "C" {

// Host entry point: stage planes H2D, run, copy pixels D2H.  Images are processed in sub-batches on internal streams so
// that the copies of one sub-batch overlap the kernels of the other.  Split in two halves: zj_gpu_reconstruct_submit queues
// everything and returns while the GPU works (the caller's planes and outputs stay in use), zj_gpu_reconstruct_finish waits
// and releases the per-call state; zj_gpu_reconstruct = both.
struct zj_pending {
    int device = 0;
    int ns = 0;
    cudaStream_t st[ZJ_NS] = {};
    cudaStream_t user = nullptr;
    cudaEvent_t done[ZJ_NS] = {};
    std::vector<zj_batch *> batches;
};

int zj_gpu_reconstruct_finish(zj_pending *p)
{
    if (!p) return ZJ_ERR_INVALID_ARG;
    int rc = set_device(p->device);
    for (int k = 0; k < p->ns && rc == ZJ_OK; k++) {
        // a blocking-sync event: the host thread sleeps instead of spinning, its core is free for another thread's Huffman work
        cudaError_t e = p->done[k] ? cudaEventSynchronize(p->done[k]) : cudaStreamSynchronize(p->st[k]);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventSynchronize");
    }
    for (int k = 0; k < p->ns; k++) if (p->done[k]) cudaEventDestroy(p->done[k]);
    for (zj_batch *b : p->batches) zj_batch_destroy(b);
    // (user == NULL is the legacy default stream: synchronising it would serialise this thread against every blocking stream
    // of the process, and nothing of this call was queued on it -- the internal streams were waited for above)
    if (rc == ZJ_OK && p->user) { cudaError_t e = cudaStreamSynchronize(p->user); if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize(user)"); }
    delete p;
    return rc;
}

int zj_gpu_reconstruct_submit(int device, void *stream, const zj_image *imgs, size_t n, uint8_t *const *out, const size_t *out_len, zj_pending **pending)
{
    if (!pending) return ZJ_ERR_INVALID_ARG;
    *pending = nullptr;
    if ((!imgs || !out || !out_len) && n) return ZJ_ERR_INVALID_ARG;
    int rc = set_device(device);
    if (rc) return rc;
    std::vector<Plan> plans(n);
    for (size_t i = 0; i < n; i++) {
        rc = plan_image(&imgs[i], &plans[i]);
        if (rc) return rc;
        rc = check_buffers(&imgs[i], plans[i], out[i], out_len[i]);
        if (rc) return rc;
    }
    static const bool trace = getenv("ZJ_SUBMIT_TRACE") != nullptr;
    auto now_ms = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_in = trace ? now_ms() : 0;
    auto lap = [&](const char *what) { if (trace) fprintf(stderr, "[zj submit] %-22s +%.3f ms\n", what, now_ms() - t_in); };
    cudaStream_t user = (cudaStream_t)stream;
    cudaStream_t st[ZJ_NS];
    // the staging streams are created once per host thread and device and reused: creating / destroying streams takes
    // driver-wide locks, which hurts when many threads call in (zj_decode_batch)
    // ... and so is the device staging buffer of every stream (grown on demand, reused in stream order): memory that the
    // stream-ordered pool hands from one stream to another makes the second stream wait for the first one's work, which
    // serialises the upload of one sub-batch behind the download of the previous one
    struct Lease {
        StreamCache *c = nullptr;
        ~Lease()
        {
            if (!c) return;
            std::lock_guard<std::mutex> lock(g_stream_pool.mu);
            g_stream_pool.idle.push_back(c);
        }
    };
    thread_local Lease lease;
    if (!lease.c) {
        std::lock_guard<std::mutex> lock(g_stream_pool.mu);
        if (!g_stream_pool.idle.empty()) { lease.c = g_stream_pool.idle.back(); g_stream_pool.idle.pop_back(); }
    }
    if (!lease.c) lease.c = new (std::nothrow) StreamCache;
    if (!lease.c) return ZJ_ERR_OOM;
    StreamCache &cache = *lease.c;
    if (device >= 64) return ZJ_ERR_NO_DEVICE;
    for (int k = 0; k < ZJ_NS; k++) {
        if (!cache.s[device][k]) CU(cudaStreamCreateWithFlags(&cache.s[device][k], cudaStreamNonBlocking));
        st[k] = cache.s[device][k];
    }
    // everything issued on `user` before this call must be visible
    cudaEvent_t ev_in;
    CU(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
    CU(cudaEventRecord(ev_in, user));
    for (int k = 0; k < ZJ_NS; k++) CU(cudaStreamWaitEvent(st[k], ev_in, 0));
    cudaEventDestroy(ev_in);   // (released once the recorded work has completed)
    lap("streams + entry event");

    zj_pending *pd = new (std::nothrow) zj_pending;
    if (!pd) return ZJ_ERR_OOM;
    pd->device = device;
    pd->ns = ZJ_NS;
    pd->user = user;
    for (int k = 0; k < ZJ_NS; k++) pd->st[k] = st[k];

    const size_t budget = (size_t)256 << 20;  // device staging per sub-batch
    size_t i = 0;
    int which = 0;
    rc = ZJ_OK;
    while (i < n && rc == ZJ_OK) {
        size_t j = i, bytes = 0, charged = 0;   // staging bytes; those plus the batch's own scratch for oriented images
        while (j < n) {
            size_t need = plans[j].out_size, coef = 0;
            for (uint32_t z = 0; z < plans[j].ncomp_used; z++) coef += (size_t)plans[j].n_strips * plans[j].chunk[z] * 2;
            need += coef + coef / 8 + 4096;      // (planes uploaded as one span may carry the gaps between them)
            const size_t orient_scratch = plans[j].orient ? plans[j].out_size + 256 : 0;
            // (the first sub-batch is a small one: kernels and downloads start after 1/8 of the usual upload)
            if (j > i && charged + need + orient_scratch > (i == 0 ? budget / 8 : budget)) break;
            bytes += need + 4 * 256;
            charged += need + 4 * 256 + orient_scratch;
            j++;
        }
        const int slot = which;                   // stream s and its staging buffer
        cudaStream_t s = st[slot];
        which = (which + 1) % ZJ_NS;
        cudaError_t e = cudaSuccess;
        if (cache.cap[device][slot] < bytes) {
            if (cache.buf[device][slot]) {
                cudaStreamSynchronize(s);
                cudaFree(cache.buf[device][slot]); cache.buf[device][slot] = nullptr; cache.cap[device][slot] = 0;
            }
            e = cudaMalloc((void **)&cache.buf[device][slot], bytes + bytes / 8);
            if (e != cudaSuccess) { cache.buf[device][slot] = nullptr; rc = cuda_fail(e, "cudaMalloc(staging)"); break; }
            cache.cap[device][slot] = bytes + bytes / 8;
        }
        lap("staging buffer");
        uint8_t *pool = cache.buf[device][slot];
        std::vector<zj_image> dimgs(imgs + i, imgs + j);
        std::vector<uint8_t *> douts(j - i);
        std::vector<size_t> dlens(j - i);
        size_t off = 0;
        auto take = [&](size_t nbytes) { uint8_t *p = pool + off; off += (nbytes + 255) & ~(size_t)255; return p; };
        // device addresses first, then the descriptors, then the copies: the descriptor upload comes from pageable memory, and such a
        // copy first waits for everything queued on its stream -- behind the plane uploads it would hold the host back until they
        // are done, and nothing of the next sub-batch could be queued meanwhile
        // Planes that follow each other in host memory (the host stage keeps an image's planes in one block) keep their
        // relative positions on the device and go up as ONE copy: a 4 MB chroma plane alone reaches 44 GB/s over PCIe, the
        // 25 MB of a whole 4K image 49.
        std::vector<size_t> span(j - i, 0);     // bytes of the merged copy (0 = one copy per plane)
        for (size_t k = i; k < j; k++) {
            const uint32_t nz = plans[k].ncomp_used;
            size_t nbz[3] = {0, 0, 0}, rel[3] = {0, 0, 0}, sum = 0;
            bool merge = nz > 1;
            for (uint32_t z = 0; z < nz; z++) { nbz[z] = (size_t)plans[k].n_strips * plans[k].chunk[z] * 2; sum += nbz[z]; }
            for (uint32_t z = 0; z < nz; z++) {
                const uintptr_t a0 = reinterpret_cast<uintptr_t>(imgs[k].comp[0].coeff), az = reinterpret_cast<uintptr_t>(imgs[k].comp[z].coeff);
                if (az < a0) { merge = false; break; }
                rel[z] = az - a0;
                if ((rel[z] & 15) || (z > 0 && rel[z] < rel[z - 1] + nbz[z - 1])) { merge = false; break; }
            }
            const size_t total = merge ? rel[nz - 1] + nbz[nz - 1] : 0;
            if (merge && total <= sum + sum / 8 + 4096) {
                uint8_t *base = take(total);
                for (uint32_t z = 0; z < nz; z++) dimgs[k - i].comp[z].coeff = (const int16_t *)(base + rel[z]);
                span[k - i] = total;
            } else {
                for (uint32_t z = 0; z < nz; z++) dimgs[k - i].comp[z].coeff = (const int16_t *)take(nbz[z]);
            }
            douts[k - i] = take(plans[k].out_size);
            dlens[k - i] = plans[k].out_size;
        }
        zj_batch *b = nullptr;
        rc = batch_create_impl(device, dimgs.data(), dimgs.size(), douts.data(), dlens.data(), &b, true, s);
        if (rc != ZJ_OK) break;
        for (size_t k = i; k < j && rc == ZJ_OK; k++) {
            if (span[k - i]) {
                e = cudaMemcpyAsync((void *)dimgs[k - i].comp[0].coeff, imgs[k].comp[0].coeff, span[k - i], cudaMemcpyHostToDevice, s);
                if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync(H2D)");
                continue;
            }
            for (uint32_t z = 0; z < plans[k].ncomp_used; z++) {
                const size_t nb = (size_t)plans[k].n_strips * plans[k].chunk[z] * 2;
                e = cudaMemcpyAsync((void *)dimgs[k - i].comp[z].coeff, imgs[k].comp[z].coeff, nb, cudaMemcpyHostToDevice, s);
                if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemcpyAsync(H2D)"); break; }
            }
        }
        if (rc != ZJ_OK) { zj_batch_destroy(b); break; }
        lap("descriptors + uploads");
        pd->batches.push_back(b);
        rc = zj_batch_run(b, s);
        batch_drop_scratch(b);
        if (rc != ZJ_OK) break;
        for (size_t k = i; k < j; k++) {
            e = cudaMemcpyAsync(out[k], douts[k - i], plans[k].out_size, cudaMemcpyDeviceToHost, s);
            if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemcpyAsync(D2H)"); break; }
        }
        lap("kernels + downloads");
        i = j;
    }
    if (rc == ZJ_OK) {
        for (int k = 0; k < ZJ_NS; k++) {
            if (cudaEventCreateWithFlags(&pd->done[k], cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) { pd->done[k] = nullptr; cudaGetLastError(); continue; }
            if (cudaEventRecord(pd->done[k], st[k]) != cudaSuccess) { cudaEventDestroy(pd->done[k]); pd->done[k] = nullptr; cudaGetLastError(); }
        }
        *pending = pd;
        return ZJ_OK;
    }
    const int rc_submit = rc;
    zj_gpu_reconstruct_finish(pd);   // waits for what was queued, releases the descriptors
    return rc_submit;
}

// ------------------------------------------------------------------------------------------ several devices
// The path shards with no exchange step (SURVEY.md 8(e)): images are independent, and so are the strips of one image --
// every rule of worker::post_process is local to the strip it is called for (worker.rs:32-85 sees one strip's coefficients
// and one strip's output rows).  So a batch is cut into contiguous image ranges, one per device, and a batch with fewer
// images than devices is cut inside the images: contiguous STRIP ranges, each a "virtual image" whose planes start at the
// range's first strip and whose output starts at the range's first row.  One host thread per device runs its share through
// zj_gpu_reconstruct on that device's own streams; nothing is exchanged between devices.
void zj_partition(size_t n_items, size_t n_parts, size_t part, size_t *begin, size_t *end)
{
    size_t lo = 0, hi = 0;
    if (n_parts && part < n_parts) {
        const size_t base = n_items / n_parts, rem = n_items % n_parts;
        lo = part * base + std::min(part, rem);
        hi = lo + base + (part < rem ? 1 : 0);
    }
    if (begin) *begin = lo;
    if (end) *end = hi;
}

int zj_image_strip_range(const zj_image *img, uint32_t strip_begin, uint32_t strip_end, zj_image *sub, size_t *out_offset, size_t *out_bytes,
                         uint32_t *n_strips)
{
    Plan pl;
    int rc = plan_image(img, &pl);
    if (rc) return rc;
    if (n_strips) *n_strips = pl.n_strips;
    if (!sub && !out_offset && !out_bytes) return ZJ_OK;           // a query for the strip count
    if (img->variant == ZJ_VARIANT_SPEC) return ZJ_ERR_UNSUPPORTED;  // its rows need chroma context from neighbouring strips
    if (strip_begin > strip_end || strip_end > pl.n_strips) return ZJ_ERR_INVALID_ARG;
    const size_t row_bytes = (size_t)img->width * num_components(img->out_cs);
    // the range that holds the last strip also owns the rows below it; an image without strips is one (empty) range at 0
    const bool last = strip_end == pl.n_strips && (strip_begin < strip_end || pl.n_strips == 0);
    if (strip_begin == strip_end && !last) {
        if (out_offset) *out_offset = 0;
        if (out_bytes) *out_bytes = 0;
        if (sub) { *sub = *img; sub->height = 0; }
        return ZJ_OK;
    }
    const uint64_t row0 = (uint64_t)strip_begin * pl.rows;
    if (row0 > img->height) return ZJ_ERR_INVALID_ARG;
    // the last range also owns the rows below the last strip (a partial strip, and the rows the reference never writes: Q1)
    const uint32_t h = last ? img->height - (uint32_t)row0 : (strip_end - strip_begin) * pl.rows;
    if (!last && row0 + h > img->height) return ZJ_ERR_INVALID_ARG;

    if (out_offset) *out_offset = (size_t)row0 * row_bytes;
    if (out_bytes) *out_bytes = (size_t)h * row_bytes;
    if (sub) {
        *sub = *img;
        sub->height = h;
        for (uint32_t z = 0; z < img->n_comp; z++) {
            const uint64_t skip = (uint64_t)strip_begin * pl.chunk[z];
            if (img->comp[z].coeff) sub->comp[z].coeff = img->comp[z].coeff + skip;
            sub->comp[z].n_i16 = img->comp[z].n_i16 > skip ? img->comp[z].n_i16 - skip : 0;
        }
        if (h == 0) return ZJ_OK;
        // the virtual image must plan to exactly the strips of the range (it does unless the whole image's strip count was
        // cut by the reference's output-capacity rule, mcu_prog.rs:206-209 -- widths next to 65535 only)
        Plan ps;
        rc = plan_image(sub, &ps);
        if (rc) return rc;
        if (ps.n_strips != strip_end - strip_begin) return ZJ_ERR_UNSUPPORTED;
    }
    return ZJ_OK;
}

int zj_gpu_reconstruct_multi(const int *devices, size_t n_dev, const zj_image *imgs, size_t n, uint8_t *const *out, const size_t *out_len)
{
    if (!devices || n_dev == 0 || ((!imgs || !out || !out_len) && n)) return ZJ_ERR_INVALID_ARG;
    if (n == 0) return ZJ_OK;
    // per device: a list of (virtual) images with their output slices
    struct Share { std::vector<zj_image> imgs; std::vector<uint8_t *> out; std::vector<size_t> len; int rc = ZJ_OK; };
    std::vector<Share> share(n_dev);
    bool by_strips = n < n_dev;
    if (by_strips) {
        for (size_t i = 0; i < n && by_strips; i++) {
            uint32_t ns = 0;
            int rc = zj_image_strip_range(&imgs[i], 0, 0, nullptr, nullptr, nullptr, &ns);
            if (rc) return rc;
            if (!out[i]) return ZJ_ERR_INVALID_ARG;
            if (out_len[i] < zj_output_size(&imgs[i])) return ZJ_ERR_SHORT_OUTPUT;
            std::vector<Share> trial(n_dev);
            for (size_t k = 0; k < n_dev; k++) {
                size_t s0, s1;
                zj_partition(ns, n_dev, k, &s0, &s1);
                if (s0 == s1 && !(ns == 0 && k == 0)) continue;   // (an image without strips: its never-written rows go to the first device)
                zj_image sub;
                size_t off = 0, bytes = 0;
                rc = zj_image_strip_range(&imgs[i], (uint32_t)s0, (uint32_t)s1, &sub, &off, &bytes, nullptr);
                if (rc == ZJ_ERR_UNSUPPORTED) { by_strips = false; break; }   // cannot be cut: whole images per device instead
                if (rc) return rc;
                if (bytes == 0) continue;
                share[k].imgs.push_back(sub); share[k].out.push_back(out[i] + off); share[k].len.push_back(bytes);
            }
        }
        if (!by_strips) for (auto &sh : share) { sh.imgs.clear(); sh.out.clear(); sh.len.clear(); }
    }
    if (!by_strips) {
        for (size_t k = 0; k < n_dev; k++) {
            size_t lo, hi;
            zj_partition(n, n_dev, k, &lo, &hi);
            share[k].imgs.assign(imgs + lo, imgs + hi);
            share[k].out.assign(out + lo, out + hi);
            share[k].len.assign(out_len + lo, out_len + hi);
        }
    }
    auto run = [&](size_t k) {
        Share &sh = share[k];
        if (sh.imgs.empty()) return;
        try { sh.rc = zj_gpu_reconstruct(devices[k], nullptr, sh.imgs.data(), sh.imgs.size(), sh.out.data(), sh.len.data()); }
        catch (...) { sh.rc = ZJ_ERR_OOM; }
    };
    std::vector<std::thread> pool;
    for (size_t k = 1; k < n_dev; k++) {
        try { pool.emplace_back(run, k); } catch (...) { run(k); }
    }
    run(0);
    for (auto &t : pool) t.join();
    for (size_t k = 0; k < n_dev; k++) if (share[k].rc != ZJ_OK) return share[k].rc;
    return ZJ_OK;
}

int zj_gpu_reconstruct(int device, void *stream, const zj_image *imgs, size_t n, uint8_t *const *out, const size_t *out_len)
{
    zj_pending *pd = nullptr;
    int rc = zj_gpu_reconstruct_submit(device, stream, imgs, n, out, out_len, &pd);
    if (rc != ZJ_OK) return rc;
    return zj_gpu_reconstruct_finish(pd);
}

// ------------------------------------------------------------------------------------- memory helpers
int zj_gpu_pinned_alloc(size_t bytes, void **p)
{
    if (!p) return ZJ_ERR_INVALID_ARG;
    *p = nullptr;
    if (zj_gpu_device_count() == 0) return ZJ_ERR_NO_DEVICE;
    CU(cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocPortable));
    return ZJ_OK;
}
int zj_gpu_pinned_free(void *p) { if (p) CU(cudaFreeHost(p)); return ZJ_OK; }
int zj_gpu_device_alloc(int device, size_t bytes, void **p)
{
    if (!p) return ZJ_ERR_INVALID_ARG;
    *p = nullptr;
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaMalloc(p, bytes ? bytes : 1));
    return ZJ_OK;
}
int zj_gpu_device_free(int device, void *p)
{
    int rc = set_device(device);
    if (rc) return rc;
    if (p) CU(cudaFree(p));
    return ZJ_OK;
}
int zj_gpu_memcpy_h2d(int device, void *stream, void *dst, const void *src, size_t bytes)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return ZJ_OK;
}
int zj_gpu_memcpy_d2h(int device, void *stream, void *dst, const void *src, size_t bytes)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return ZJ_OK;
}
int zj_gpu_memset(int device, void *stream, void *dst, int value, size_t bytes)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaMemsetAsync(dst, value, bytes, (cudaStream_t)stream));
    return ZJ_OK;
}
int zj_gpu_stream_create(int device, void **stream)
{
    if (!stream) return ZJ_ERR_INVALID_ARG;
    int rc = set_device(device);
    if (rc) return rc;
    cudaStream_t s;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *stream = (void *)s;
    return ZJ_OK;
}
int zj_gpu_stream_destroy(int device, void *stream)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaStreamDestroy((cudaStream_t)stream));
    return ZJ_OK;
}
int zj_gpu_stream_synchronize(int device, void *stream)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return ZJ_OK;
}
int zj_gpu_event_create(int device, void **event)
{
    if (!event) return ZJ_ERR_INVALID_ARG;
    int rc = set_device(device);
    if (rc) return rc;
    cudaEvent_t e;
    CU(cudaEventCreate(&e));
    *event = (void *)e;
    return ZJ_OK;
}
int zj_gpu_event_record(int device, void *event, void *stream)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaEventRecord((cudaEvent_t)event, (cudaStream_t)stream));
    return ZJ_OK;
}
int zj_gpu_event_elapsed_ms(int device, void *start, void *stop, float *ms)
{
    if (!ms) return ZJ_ERR_INVALID_ARG;
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaEventSynchronize((cudaEvent_t)stop));
    CU(cudaEventElapsedTime(ms, (cudaEvent_t)start, (cudaEvent_t)stop));
    return ZJ_OK;
}
int zj_gpu_event_destroy(int device, void *event)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(cudaEventDestroy((cudaEvent_t)event));
    return ZJ_OK;
}

const char *zj_gpu_strerror(int status)
{
    switch (status) {
    case ZJ_OK: return "ok";
    case ZJ_ERR_INVALID_ARG: return "invalid argument or inconsistent image descriptor";
    case ZJ_ERR_UNSUPPORTED: return "Unknown down-sampling method, cannot continue";  // decoder.rs:512-519
    case ZJ_ERR_SHORT_PLANE: return "coefficient plane smaller than the strips it must feed";
    case ZJ_ERR_SHORT_OUTPUT: return "output buffer smaller than width*height*components";
    case ZJ_ERR_REF_PANIC: return "the reference decoder panics on this geometry";
    case ZJ_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    case ZJ_ERR_CUDA: return "CUDA runtime error (see zj_gpu_last_cuda_error)";
    case ZJ_ERR_OOM: return "out of device or pinned memory";
    case ZJ_ERR_DECODE: return "JPEG header / entropy decode error (see zj_decoder_error)";
    default: return "unknown status";
    }
}
const char *zj_gpu_last_cuda_error(void) { return g_cuda_err; }
uint64_t zj_gpu_launch_count(void) { return g_launches.load(); }

}  // extern "C"
