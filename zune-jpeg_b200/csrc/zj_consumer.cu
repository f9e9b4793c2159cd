// zj_consumer.cu -- device-side consumers of the reconstructed pixels (SURVEY.md 8(f).4): the pixels the fused kernels
// wrote (u8, interleaved, exactly the bytes of the reference's decode_buffer) are turned into what a GPU consumer reads --
// planar (CHW) or interleaved (HWC) u8 / f16 / f32, per-channel `(x - mean) * inv_std`, optionally a 2x2 box down-scale,
// optionally without the alpha / padding byte of "RGBA" / "RGBX" -- without leaving the device.  The reference's writers
// that this extends are the per-colourspace dispatch of src/worker.rs:113-133 and the interleaving stores of
// src/color_convert/scalar.rs:52-169: every value here is a function of those writers' exact u8 results, so the u8 / HWC /
// full-size descriptor stays bit-identical to the reference and the other descriptors are specified (and tested) as
//     f = (float(u8) - mean[c]) * inv_std[c]                 (two IEEE fp32 operations, no fused multiply-add)
//     u8 at half size = (a + b + c + d + 2) >> 2,  f at half size = (float(a + b + c + d) * 0.25f - mean[c]) * inv_std[c]
//     f16 = round-to-nearest-even of the fp32 value
// applied to the oracle's bytes.
//
// One thread produces 8 consecutive output pixels of one row (all channels): its inputs are 8 * nc (or 2 rows of 16 * nc)
// contiguous bytes, read as 32-bit words when the row allows it, and its outputs are 16-byte stores when the row allows it.
// HBM-bound: 3 B/px in + 6 B/px out for RGB -> f16 (measured: 6.3 TB/s of the 6.5 TB/s copy bandwidth).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "../../include/zune_jpeg_b200.h"
#include "zj_device.h"

namespace zj {

struct ConvParams {
    float mean[4], inv_std[4];
};

typedef unsigned int u32;

template <typename T> __device__ __forceinline__ T cvt(float f);
template <> __device__ __forceinline__ float cvt<float>(float f) { return f; }
template <> __device__ __forceinline__ uint8_t cvt<uint8_t>(float) { return 0; }   // (never taken: u8 outputs do not go through floats)
template <> __device__ __forceinline__ __half cvt<__half>(float f) { return __float2half_rn(f); }

// 8 elements of type T to `p`: one or two 16-byte stores when `vec`, element stores otherwise (n = valid elements)
template <typename T>
__device__ __forceinline__ void store8(T *p, const T (&v)[8], const int n, const bool vec)
{
    if (vec && n == 8) {
        if (sizeof(T) == 1) {
            uint2 w;
            memcpy(&w, v, 8);
            *reinterpret_cast<uint2 *>(p) = w;
        } else if (sizeof(T) == 2) {
            uint4 w;
            memcpy(&w, v, 16);
            *reinterpret_cast<uint4 *>(p) = w;
        } else {
            uint4 w0, w1;
            memcpy(&w0, v, 16);
            memcpy(&w1, reinterpret_cast<const char *>(v) + 16, 16);
            reinterpret_cast<uint4 *>(p)[0] = w0;
            reinterpret_cast<uint4 *>(p)[1] = w1;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++)
            if (i < n) p[i] = v[i];
    }
}

// NB contiguous bytes from `p` into words (little endian): aligned 32-bit loads when possible
template <int NW>
__device__ __forceinline__ void load_bytes(const uint8_t *p, const int nbytes, u32 (&w)[NW])
{
    if ((reinterpret_cast<uintptr_t>(p) & 3) == 0 && nbytes == NW * 4) {
#pragma unroll
        for (int k = 0; k < NW; k++) w[k] = __ldg(reinterpret_cast<const u32 *>(p) + k);
    } else {
#pragma unroll
        for (int k = 0; k < NW; k++) {
            u32 v = 0;
#pragma unroll
            for (int b = 0; b < 4; b++)
                if (4 * k + b < nbytes) v |= (u32)__ldg(p + 4 * k + b) << (8 * b);
            w[k] = v;
        }
    }
}
template <int NW> __device__ __forceinline__ u32 byte_at(const u32 (&w)[NW], const int k) { return (w[k >> 2] >> (8 * (k & 3))) & 0xffu; }

// T: output element (uint8_t, __half, float); CHW: planar output; HALF: 2x2 box down-scale; NC: source bytes per pixel;
// OC: channels written (NC, or 3 of 4)
template <typename T, bool CHW, bool HALF, int NC, int OC>
__global__ void __launch_bounds__(256) convert_kernel(const ConvImage *__restrict__ images, const ConvParams prm)
{
    const ConvImage im = images[blockIdx.z];
    const u32 y = blockIdx.y;
    if (y >= im.oh) return;
    const u32 x0 = 8u * (blockIdx.x * 256u + threadIdx.x);
    if (x0 >= im.ow) return;
    const int n = (int)min(8u, im.ow - x0);
    constexpr int S = HALF ? 2 : 1;
    constexpr int NW = 8 * S * NC / 4;   // words per source row segment
    u32 sum[8][NC];                      // per output pixel and channel: the u8 (or the sum of the four)
    {
        const size_t srow = (size_t)im.width * NC;
        const uint8_t *p = im.src + (size_t)(S * y) * srow + (size_t)(S * x0) * NC;
        u32 w[NW];
        load_bytes<NW>(p, n * S * NC, w);
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int c = 0; c < NC; c++)
                sum[i][c] = HALF ? byte_at<NW>(w, (2 * i) * NC + c) + byte_at<NW>(w, (2 * i + 1) * NC + c) : byte_at<NW>(w, i * NC + c);
        if (HALF) {
            load_bytes<NW>(p + srow, n * S * NC, w);
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int c = 0; c < NC; c++) sum[i][c] += byte_at<NW>(w, (2 * i) * NC + c) + byte_at<NW>(w, (2 * i + 1) * NC + c);
        }
    }
    T *const dst = reinterpret_cast<T *>(im.dst);
    const size_t plane = (size_t)im.ow * im.oh;
    if (CHW) {
#pragma unroll
        for (int c = 0; c < OC; c++) {
            T v[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (sizeof(T) == 1) v[i] = (T)(HALF ? (sum[i][c] + 2u) >> 2 : sum[i][c]);
                else {
                    const float f = HALF ? __fmul_rn((float)sum[i][c], 0.25f) : (float)sum[i][c];
                    v[i] = cvt<T>(__fmul_rn(__fsub_rn(f, prm.mean[c]), prm.inv_std[c]));
                }
            }
            T *q = dst + (size_t)c * plane + (size_t)y * im.ow + x0;
            store8<T>(q, v, n, (reinterpret_cast<uintptr_t>(q) & 15) == 0);
        }
    } else {
        // interleaved: 8 * OC consecutive elements, stored in OC groups of 8
        T *q = dst + ((size_t)y * im.ow + x0) * OC;
        const bool vec = (reinterpret_cast<uintptr_t>(q) & 15) == 0 && n == 8;
#pragma unroll
        for (int g = 0; g < OC; g++) {
            T v[8];
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const int px = (8 * g + e) / OC, ch = (8 * g + e) % OC;   // compile-time after unrolling
                const u32 s = sum[px][ch];
                if (sizeof(T) == 1) v[e] = (T)(HALF ? (s + 2u) >> 2 : s);
                else {
                    const float f = HALF ? __fmul_rn((float)s, 0.25f) : (float)s;
                    v[e] = cvt<T>(__fmul_rn(__fsub_rn(f, prm.mean[ch]), prm.inv_std[ch]));
                }
            }
            const int left = n * OC - 8 * g;   // valid elements of this group
            if (left <= 0) break;
            store8<T>(q + 8 * g, v, left < 8 ? left : 8, vec);
        }
    }
}

template <typename T, bool CHW, bool HALF>
static cudaError_t launch_nc(const ConvImage *d_images, uint32_t nc, uint32_t oc, dim3 grid, const ConvParams &prm, cudaStream_t s)
{
    if (nc == 1) convert_kernel<T, CHW, HALF, 1, 1><<<grid, 256, 0, s>>>(d_images, prm);
    else if (nc == 3) convert_kernel<T, CHW, HALF, 3, 3><<<grid, 256, 0, s>>>(d_images, prm);
    else if (oc == 3) convert_kernel<T, CHW, HALF, 4, 3><<<grid, 256, 0, s>>>(d_images, prm);
    else convert_kernel<T, CHW, HALF, 4, 4><<<grid, 256, 0, s>>>(d_images, prm);
    return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_t(const ConvImage *d_images, uint32_t nc, uint32_t oc, bool chw, bool half, dim3 grid, const ConvParams &prm, cudaStream_t s)
{
    if (chw) return half ? launch_nc<T, true, true>(d_images, nc, oc, grid, prm, s) : launch_nc<T, true, false>(d_images, nc, oc, grid, prm, s);
    return half ? launch_nc<T, false, true>(d_images, nc, oc, grid, prm, s) : launch_nc<T, false, false>(d_images, nc, oc, grid, prm, s);
}

// images [0, count) of d_images share nc; max_ow / max_oh bound the grid
cudaError_t launch_convert(const ConvImage *d_images, uint32_t count, uint32_t nc, uint32_t max_ow, uint32_t max_oh, const zj_output_desc &d, cudaStream_t s)
{
    ConvParams prm;
    for (int c = 0; c < 4; c++) { prm.mean[c] = d.mean[c]; prm.inv_std[c] = d.inv_std[c]; }
    dim3 grid((max_ow + 8 * 256 - 1) / (8 * 256), max_oh, count);
    const bool chw = d.layout == ZJ_LAYOUT_CHW, half = d.scale_log2 == 1;
    const uint32_t oc = (d.channels == 3 && nc == 4) ? 3u : nc;
    switch (d.dtype) {
    case ZJ_DTYPE_U8: return launch_t<uint8_t>(d_images, nc, oc, chw, half, grid, prm, s);
    case ZJ_DTYPE_F16: return launch_t<__half>(d_images, nc, oc, chw, half, grid, prm, s);
    default: return launch_t<float>(d_images, nc, oc, chw, half, grid, prm, s);
    }
}

// ------------------------------------------------------------------------------------------------------ resize
// A crop of each image's u8 pixels resized to one out_w x out_h slot of a batch tensor (zj_gpu_resize_device and the
// *_resized entry points; the specification is the header's, DESIGN.md section 4.5.1).  Every value is a function of the u8
// bytes of the crop alone: neighbours are clamped to the crop and pixels outside it never contribute.
//   ZJ_FILTER_AREA      output row i covers crop rows [floor(i*h/OH), ceil((i+1)*h/OH)), columns alike; s = exact sum of the
//                       window's bytes, n = its pixel count; u8 = (s + n/2) / n, float = float(s) / float(n)
//   ZJ_FILTER_BILINEAR  torch interpolate(bilinear, align_corners=False, antialias=False) in the stated fp32 order;
//                       u8 = round-to-nearest-even of the value, clamped to [0, 255]
// then (v - mean[c]) * inv_std[c] for floats, every fp32 operation a single IEEE round-to-nearest one (no FMA).

struct ResizeParams {
    float mean[4], inv_std[4];
    uint32_t ow, oh;
};

constexpr int RZ_ROWS = 8;   // output rows per CTA: one warp each (256 threads)

template <typename T> __device__ __forceinline__ u32 to_bits(T v);
template <> __device__ __forceinline__ u32 to_bits<uint8_t>(uint8_t v) { return v; }
template <> __device__ __forceinline__ u32 to_bits<__half>(__half v) { return __half_as_ushort(v); }
template <> __device__ __forceinline__ u32 to_bits<float>(float v) { return __float_as_uint(v); }
template <typename T> __device__ __forceinline__ T from_bits(u32 b);
template <> __device__ __forceinline__ uint8_t from_bits<uint8_t>(u32 b) { return (uint8_t)b; }
template <> __device__ __forceinline__ __half from_bits<__half>(u32 b) { return __ushort_as_half((unsigned short)b); }
template <> __device__ __forceinline__ float from_bits<float>(u32 b) { return __uint_as_float(b); }

// 8 consecutive output pixels (n valid) of output row y, all OC channels, into the slot: per plane (CHW) or as 8 * OC
// interleaved elements (HWC); 16-byte stores where the address allows them (store8)
template <typename T, bool CHW, int OC>
__device__ __forceinline__ void store_px8(T *dst, const ResizeParams &prm, u32 y, u32 x0, int n, const T (&v)[8][OC])
{
    if (CHW) {
        const size_t plane = (size_t)prm.ow * prm.oh;
#pragma unroll
        for (int c = 0; c < OC; c++) {
            T u[8];
#pragma unroll
            for (int e = 0; e < 8; e++) u[e] = v[e][c];
            T *q = dst + (size_t)c * plane + (size_t)y * prm.ow + x0;
            store8<T>(q, u, n, (reinterpret_cast<uintptr_t>(q) & 15) == 0);
        }
    } else {
        T *q = dst + ((size_t)y * prm.ow + x0) * OC;
        const bool vec = (reinterpret_cast<uintptr_t>(q) & 15) == 0 && n == 8;
#pragma unroll
        for (int g = 0; g < OC; g++) {
            T u[8];
#pragma unroll
            for (int e = 0; e < 8; e++) u[e] = v[(8 * g + e) / OC][(8 * g + e) % OC];
            const int left = n * OC - 8 * g;
            if (left <= 0) break;
            store8<T>(q + 8 * g, u, left < 8 ? left : 8, vec);
        }
    }
}

template <typename T> __device__ __forceinline__ T normalise(float v, float mean, float inv_std)
{
    return cvt<T>(__fmul_rn(__fsub_rn(v, mean), inv_std));
}

// dp4a mask of the bytes of channel c in a word whose byte 0 belongs to channel ph
template <int NC> __device__ __forceinline__ u32 chan_mask(int ph, int c)
{
    if (NC == 1) return 0x01010101u;
    int k = c - ph;
    if (k < 0) k += NC;
    if (NC == 4) return 1u << (8 * k);
    return k == 0 ? 0x01000001u : 1u << (8 * k);   // NC == 3: bytes k and k + 3
}

// (s + n/2) / n for s <= 255 * n, without a 64-bit division: a float estimate (off by less than 0.001) corrected by one step
__device__ __forceinline__ u32 div_round(uint64_t s, u32 n)
{
    const uint64_t t = s + n / 2;
    u32 q = (u32)__fdividef(__ull2float_rn(t), __uint2float_rn(n));
    if ((uint64_t)q * n > t) q--;
    else if ((uint64_t)(q + 1) * n <= t) q++;
    return q;
}

// Sums the bytes [b, e) of one window row per channel into acc: the aligned words from a = b & ~3 on, one dp4a per word and
// channel against m[c] (the channel's bytes of the word) and keep (the bytes inside [b, e)).  INSIDE: every word lies in the source
// image; otherwise a word that does not is assembled from the window's bytes by byte loads, so no load leaves the image.
template <int NC, int OC, bool INSIDE>
__device__ __forceinline__ void area_span(uintptr_t a, const uintptr_t b, const uintptr_t e, u32 (&m)[OC], u32 (&acc)[OC])
{
    for (; a < e; a += 4) {
        u32 keep = 0xffffffffu;
        if (a < b) keep = 0xffffffffu << (8 * (u32)(b - a));
        if (a + 4 > e) keep &= 0xffffffffu >> (8 * (u32)(a + 4 - e));
        u32 wd;
        if (INSIDE || (a >= b && a + 4 <= e)) wd = __ldg(reinterpret_cast<const u32 *>(a));
        else {
            wd = 0;
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (a + k >= b && a + k < e) wd |= (u32)__ldg(reinterpret_cast<const uint8_t *>(a + k)) << (8 * k);
        }
#pragma unroll
        for (int c = 0; c < OC; c++) acc[c] = __dp4a(wd, m[c] & keep, acc[c]);
        if (NC == 3) {   // the next word starts one channel later
            u32 t[OC];
#pragma unroll
            for (int c = 0; c < OC; c++) t[c] = m[c];
#pragma unroll
            for (int c = 0; c < OC; c++) m[c] = t[(c + 2) % 3];
        }
    }
}

// ZJ_FILTER_AREA.  A warp owns 32 consecutive output columns of one output row, a lane one column: in every source row of the
// window the warp reads one contiguous span, each lane its own window's bytes as the aligned 32-bit words that hold them, summed
// per channel by one dp4a against a byte mask (bytes outside the window or of another channel weigh 0).  No load reaches outside
// the source image: the one or two words that would are read byte by byte.  Groups of 8 lanes then hand their values to one
// lane, which stores 8 pixels.
template <typename T, bool CHW, int NC, int OC>
__global__ void __launch_bounds__(256) resize_area_kernel(const ResizeImage *__restrict__ images, const ResizeParams prm)
{
    const ResizeImage im = images[blockIdx.z];
    const u32 lane = threadIdx.x & 31;
    const u32 i = blockIdx.y * RZ_ROWS + (threadIdx.x >> 5);
    if (i >= prm.oh) return;   // (warp-uniform: the shuffles below see every lane of a warp that gets there)
    const u32 j = blockIdx.x * 32u + lane;
    const bool live = j < prm.ow;
    // (crop and output sizes are at most 65535: the products fit 32 bits)
    const u32 r0 = i * im.h / prm.oh, r1 = ((i + 1) * im.h + prm.oh - 1) / prm.oh;
    const u32 c0 = live ? j * im.w / prm.ow : 0u;
    const u32 c1 = live ? ((j + 1) * im.w + prm.ow - 1) / prm.ow : 0u;
    uint64_t sum[OC];
#pragma unroll
    for (int c = 0; c < OC; c++) sum[c] = 0;
    const uintptr_t lo = reinterpret_cast<uintptr_t>(im.lo), hi = reinterpret_cast<uintptr_t>(im.hi);
    const uint8_t *row = im.src + (size_t)r0 * im.pitch;
    for (u32 r = r0; r < r1; r++, row += im.pitch) {
        const uintptr_t b = reinterpret_cast<uintptr_t>(row) + (size_t)c0 * NC, e = reinterpret_cast<uintptr_t>(row) + (size_t)c1 * NC;
        uintptr_t a = b & ~(uintptr_t)3;
        // channel of the first word's byte 0 (the crop starts on a pixel)
        const int ph = (int)(((long long)c0 * NC - (long long)(b - a)) % NC + NC) % NC;
        u32 m[OC];
#pragma unroll
        for (int c = 0; c < OC; c++) m[c] = chan_mask<NC>(ph, c);
        u32 acc[OC];
#pragma unroll
        for (int c = 0; c < OC; c++) acc[c] = 0;
        // every aligned word of the span lies inside the source image (all rows but the image's first and last, at most)
        if (a >= lo && ((e + 3) & ~(uintptr_t)3) <= hi) area_span<NC, OC, true>(a, b, e, m, acc);
        else area_span<NC, OC, false>(a, b, e, m, acc);
#pragma unroll
        for (int c = 0; c < OC; c++) sum[c] += acc[c];
    }
    const u32 n = (r1 - r0) * (c1 - c0);
    u32 bits[OC];
#pragma unroll
    for (int c = 0; c < OC; c++) {
        if (!live) bits[c] = 0;
        else if (sizeof(T) == 1) bits[c] = div_round(sum[c], n);
        else bits[c] = to_bits<T>(normalise<T>(__fdiv_rn(__ull2float_rn(sum[c]), __uint2float_rn(n)), prm.mean[c], prm.inv_std[c]));
    }
    T v[8][OC];
    if (sizeof(T) == 1) {   // u8: the OC channels of a pixel travel in one word
        u32 packed = 0;
#pragma unroll
        for (int c = 0; c < OC; c++) packed |= bits[c] << (8 * c);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const u32 p = __shfl_sync(0xffffffffu, packed, (lane & ~7u) + k);
#pragma unroll
            for (int c = 0; c < OC; c++) v[k][c] = from_bits<T>((p >> (8 * c)) & 0xffu);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; k++)
#pragma unroll
            for (int c = 0; c < OC; c++) v[k][c] = from_bits<T>(__shfl_sync(0xffffffffu, bits[c], (lane & ~7u) + k));
    }
    const u32 x0 = j;   // for the storing lanes (lane % 8 == 0)
    if ((lane & 7) == 0 && x0 < prm.ow)
        store_px8<T, CHW, OC>(reinterpret_cast<T *>(im.dst), prm, i, x0, (int)min(8u, prm.ow - x0), v);
}

// source index, weights of output index j (crop size n_in, scale s = float(n_in) / float(n_out)) -- the exact fp32 sequence
// of the specification
__device__ __forceinline__ void bilinear_coord(u32 j, u32 n_in, float s, int &i0, float &a, float &b)
{
    float f = __fsub_rn(__fmul_rn(__fadd_rn(__uint2float_rn(j), 0.5f), s), 0.5f);
    if (f < 0.0f) f = 0.0f;
    i0 = min((int)f, (int)n_in - 1);
    a = __fsub_rn(f, (float)i0);
    b = __fsub_rn(1.0f, a);
}

// ZJ_FILTER_BILINEAR.  A CTA covers 256 output columns x 8 output rows of one image; their coordinate tables are built once in
// shared memory.  A thread produces 8 consecutive output pixels of a row: four byte loads per pixel and channel.
template <typename T, bool CHW, int NC, int OC>
__global__ void __launch_bounds__(256) resize_bilinear_kernel(const ResizeImage *__restrict__ images, const ResizeParams prm)
{
    __shared__ int s_c0[256];
    __shared__ float s_ax[256], s_bx[256];
    __shared__ int s_r0[RZ_ROWS];
    __shared__ float s_ay[RZ_ROWS], s_by[RZ_ROWS];
    const ResizeImage im = images[blockIdx.z];
    const u32 jt = blockIdx.x * 256u, it = blockIdx.y * RZ_ROWS;
    const u32 t = threadIdx.x;
    if (jt + t < prm.ow) bilinear_coord(jt + t, im.w, im.sx, s_c0[t], s_ax[t], s_bx[t]);
    if (t < RZ_ROWS && it + t < prm.oh) bilinear_coord(it + t, im.h, im.sy, s_r0[t], s_ay[t], s_by[t]);
    __syncthreads();
    const u32 ly = t >> 5, xl = 8u * (t & 31);
    const u32 y = it + ly, x0 = jt + xl;
    if (y >= prm.oh || x0 >= prm.ow) return;
    const int n = (int)min(8u, prm.ow - x0);
    const int r0 = s_r0[ly], r1 = min(r0 + 1, (int)im.h - 1);
    const float ay = s_ay[ly], by = s_by[ly];
    const uint8_t *p0 = im.src + (size_t)r0 * im.pitch, *p1 = im.src + (size_t)r1 * im.pitch;
    T v[8][OC];
#pragma unroll
    for (int e = 0; e < 8; e++) {
        const int k = xl + min(e, n - 1);   // (columns past the row's end repeat the last one; they are not stored)
        const int c0 = s_c0[k], c1 = min(c0 + 1, (int)im.w - 1);
        const float ax = s_ax[k], bx = s_bx[k];
#pragma unroll
        for (int c = 0; c < OC; c++) {
            const float p00 = __ldg(p0 + c0 * NC + c), p01 = __ldg(p0 + c1 * NC + c);
            const float p10 = __ldg(p1 + c0 * NC + c), p11 = __ldg(p1 + c1 * NC + c);
            const float top = __fadd_rn(__fmul_rn(bx, p00), __fmul_rn(ax, p01));
            const float bot = __fadd_rn(__fmul_rn(bx, p10), __fmul_rn(ax, p11));
            const float val = __fadd_rn(__fmul_rn(by, top), __fmul_rn(ay, bot));
            if (sizeof(T) == 1) v[e][c] = (T)min(max(__float2int_rn(val), 0), 255);
            else v[e][c] = normalise<T>(val, prm.mean[c], prm.inv_std[c]);
        }
    }
    store_px8<T, CHW, OC>(reinterpret_cast<T *>(im.dst), prm, y, x0, n, v);
}

template <typename T, bool CHW, int NC, int OC>
static void launch_resize_k(const ResizeImage *d_images, uint32_t count, bool area, const ResizeParams &prm, cudaStream_t s)
{
    const uint32_t gy = (prm.oh + RZ_ROWS - 1) / RZ_ROWS;
    if (area) resize_area_kernel<T, CHW, NC, OC><<<dim3((prm.ow + 31) / 32, gy, count), 256, 0, s>>>(d_images, prm);
    else resize_bilinear_kernel<T, CHW, NC, OC><<<dim3((prm.ow + 255) / 256, gy, count), 256, 0, s>>>(d_images, prm);
}

template <typename T, bool CHW>
static void launch_resize_nc(const ResizeImage *d_images, uint32_t count, uint32_t nc, uint32_t oc, bool area, const ResizeParams &prm, cudaStream_t s)
{
    if (nc == 1) launch_resize_k<T, CHW, 1, 1>(d_images, count, area, prm, s);
    else if (nc == 3) launch_resize_k<T, CHW, 3, 3>(d_images, count, area, prm, s);
    else if (oc == 3) launch_resize_k<T, CHW, 4, 3>(d_images, count, area, prm, s);
    else launch_resize_k<T, CHW, 4, 4>(d_images, count, area, prm, s);
}

template <typename T>
static void launch_resize_t(const ResizeImage *d_images, uint32_t count, uint32_t nc, uint32_t oc, bool chw, bool area, const ResizeParams &prm, cudaStream_t s)
{
    if (chw) launch_resize_nc<T, true>(d_images, count, nc, oc, area, prm, s);
    else launch_resize_nc<T, false>(d_images, count, nc, oc, area, prm, s);
}

// images [0, count) of d_images (count <= 65535) share nc; the descriptors were checked by the caller
cudaError_t launch_resize(const ResizeImage *d_images, uint32_t count, uint32_t nc, const zj_output_desc &d, const zj_resize &r, cudaStream_t s)
{
    ResizeParams prm;
    for (int c = 0; c < 4; c++) { prm.mean[c] = d.mean[c]; prm.inv_std[c] = d.inv_std[c]; }
    prm.ow = r.out_w;
    prm.oh = r.out_h;
    const bool chw = d.layout == ZJ_LAYOUT_CHW, area = r.filter == ZJ_FILTER_AREA;
    const uint32_t oc = (d.channels == 3 && nc == 4) ? 3u : nc;
    switch (d.dtype) {
    case ZJ_DTYPE_U8: launch_resize_t<uint8_t>(d_images, count, nc, oc, chw, area, prm, s); break;
    case ZJ_DTYPE_F16: launch_resize_t<__half>(d_images, count, nc, oc, chw, area, prm, s); break;
    default: launch_resize_t<float>(d_images, count, nc, oc, chw, area, prm, s); break;
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------ Pillow's resize
// ZJ_FILTER_PIL_BILINEAR / _BICUBIC (the header's rules 1-4, DESIGN.md section 4.5.2), structured as Pillow's Resample.c: a
// table kernel builds each image's integer weights for the window's columns and rows, a horizontal pass writes a u8
// intermediate of the rows the vertical taps read x the window's columns, and a vertical pass writes the slot.

// Double operations of the coefficient rule, each one IEEE round-to-nearest operation: on the device through the intrinsics
// (nvcc contracts a * b + c into an FMA otherwise), on the host through a volatile product, which no compiler can fuse.
__host__ __device__ __forceinline__ double pil_add(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ __forceinline__ double pil_mul(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    volatile double p = a * b;
    return p;
#endif
}
__host__ __device__ __forceinline__ double pil_div(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    volatile double q = a / b;
    return q;
#endif
}

// One output index i of an axis resized from n_in to n_out: the first tap, the tap count, the centre and 1 / fs (rule 2)
struct PilSpan { int xmin, count; double center, ss; };
__host__ __device__ __forceinline__ PilSpan pil_span(uint32_t i, uint32_t n_in, uint32_t n_out, double support0)
{
    const double scale = pil_div((double)n_in, (double)n_out);
    const double fs = scale > 1.0 ? scale : 1.0;
    const double support = pil_mul(support0, fs);
    PilSpan sp;
    sp.center = pil_mul(pil_add((double)i, 0.5), scale);
    sp.xmin = (int)pil_add(pil_add(sp.center, -support), 0.5);
    if (sp.xmin < 0) sp.xmin = 0;
    int xmax = (int)pil_add(pil_add(sp.center, support), 0.5);
    if (xmax > (int)n_in) xmax = (int)n_in;
    sp.count = xmax - sp.xmin;
    sp.ss = pil_div(1.0, fs);
    return sp;
}

static double pil_support0(uint32_t filter) { return filter == ZJ_FILTER_PIL_BICUBIC ? 2.0 : 1.0; }

int pil_geometry(const zj_resize &r, uint32_t w, uint32_t h, PilGeometry *g)
{
    uint64_t rw = r.out_w, rh = r.out_h, left = 0, top = 0;
    if (r.short_side) {
        const uint64_t s = r.short_side, sh = std::min(w, h), lg = std::max(w, h);
        const uint64_t nl = (uint64_t)((double)(s * lg) / (double)sh);   // (one IEEE division, then truncation)
        rw = w <= h ? s : nl;
        rh = w <= h ? nl : s;
        if (rw < r.out_w || rh < r.out_h || rw > 65535 || rh > 65535) return ZJ_ERR_INVALID_ARG;
        // round_half_even((R - out) / 2.0)
        const uint64_t dx = rw - r.out_w, dy = rh - r.out_h;
        left = dx / 2 + ((dx & 1) && ((dx / 2) & 1));
        top = dy / 2 + ((dy & 1) && ((dy / 2) & 1));
    }
    g->rw = (uint32_t)rw; g->rh = (uint32_t)rh; g->left = (uint32_t)left; g->top = (uint32_t)top;
    // the taps' first rows grow with the output row, and so do their ends: the window's first and last rows bound them
    const double s0 = pil_support0(r.filter);
    const PilSpan a = pil_span(g->top, h, g->rh, s0), b = pil_span(g->top + r.out_h - 1, h, g->rh, s0);
    g->y0 = (uint32_t)a.xmin;
    g->y1 = (uint32_t)(b.xmin + b.count);
    return ZJ_OK;
}

// One image of the PIL launches.  tab: the horizontal table (n = out_w entries: xmin[n], count[n], then kk[x][n] for x < ksh),
// then at tab_v the vertical one (n = out_h, ksv), xmin relative to the crop; tmp: rows x tpitch u8, crop rows [y0, y0 + rows)
// x the window's columns, OC bytes per pixel.
struct PilImage {
    const uint8_t *src;           // byte 0 of the crop's pixel (0, y0)
    uint8_t *tmp;
    void *dst;
    int *tab;
    uint32_t pitch, w, h;         // source row bytes, crop size
    uint32_t rw, rh, left, top;   // resized size, window offset
    uint32_t y0, rows;
    uint32_t ksh, ksv, tab_v;
};
struct PilParams {
    uint32_t filter, tpitch;
};

__device__ __forceinline__ double pil_f(double x, bool bicubic)
{
    if (x < 0.0) x = -x;
    if (!bicubic) return x < 1.0 ? __dadd_rn(1.0, -x) : 0.0;
    const double a = -0.5;
    if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dadd_rn(__dmul_rn(a + 2.0, x), -(a + 3.0)), x), x), 1.0);
    if (x < 2.0) return __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(x, -5.0), x), 8.0), x), -4.0), a);
    return 0.0;
}

// One thread per window index and axis (blockIdx.y: 0 = columns, 1 = rows): rule 2's weights, the filter evaluated twice (the
// sum, then the normalised values) rather than stored
__global__ void __launch_bounds__(256) pil_table_kernel(const PilImage *__restrict__ images, const ResizeParams prm, const PilParams pp)
{
    const PilImage im = images[blockIdx.z];
    const bool vert = blockIdx.y == 1;
    const u32 n = vert ? prm.oh : prm.ow;
    const u32 i = blockIdx.x * 256u + threadIdx.x;
    if (i >= n) return;
    const bool bicubic = pp.filter == ZJ_FILTER_PIL_BICUBIC;
    const PilSpan sp = pil_span(i + (vert ? im.top : im.left), vert ? im.h : im.w, vert ? im.rh : im.rw, bicubic ? 2.0 : 1.0);
    int *tab = im.tab + (vert ? im.tab_v : 0u);
    tab[i] = sp.xmin;
    tab[n + i] = sp.count;
    double ww = 0.0;
    for (int x = 0; x < sp.count; x++) ww = __dadd_rn(ww, pil_f(__dmul_rn(__dadd_rn(__dadd_rn((double)(x + sp.xmin), -sp.center), 0.5), sp.ss), bicubic));
    int *kk = tab + 2 * n + i;
    for (int x = 0; x < sp.count; x++) {
        double k = pil_f(__dmul_rn(__dadd_rn(__dadd_rn((double)(x + sp.xmin), -sp.center), 0.5), sp.ss), bicubic);
        if (ww != 0.0) k = __ddiv_rn(k, ww);
        kk[(size_t)x * n] = k < 0.0 ? (int)__dadd_rn(-0.5, __dmul_rn(k, 4194304.0)) : (int)__dadd_rn(0.5, __dmul_rn(k, 4194304.0));
    }
}

__device__ __forceinline__ u32 clip8(int s) { return (u32)min(max(s >> 22, 0), 255); }

constexpr int PIL_HROWS = 4;   // rows per thread of the horizontal pass: each weight is loaded once for them

// Horizontal pass: a warp owns 32 consecutive window columns of PIL_HROWS intermediate rows (8 warps: 32 rows), a lane one
// column: per tap one weight (the lanes' weights are consecutive words) and NC bytes per row.  Every byte read lies in the crop.
template <int NC, int OC>
__global__ void __launch_bounds__(256) pil_horizontal_kernel(const PilImage *__restrict__ images, const ResizeParams prm, const PilParams pp)
{
    const PilImage im = images[blockIdx.z];
    const u32 j = blockIdx.x * 32u + (threadIdx.x & 31);
    const u32 r0 = (blockIdx.y * 8u + (threadIdx.x >> 5)) * PIL_HROWS;
    if (j >= prm.ow || r0 >= im.rows) return;
    const int nr = (int)min((u32)PIL_HROWS, im.rows - r0);
    const int xmin = im.tab[j], count = im.tab[prm.ow + j];
    const int *kk = im.tab + 2 * prm.ow + j;
    const uint8_t *row[PIL_HROWS];
#pragma unroll
    for (int r = 0; r < PIL_HROWS; r++) row[r] = im.src + (size_t)(r0 + min(r, nr - 1)) * im.pitch + (size_t)xmin * NC;   // (rows past the last repeat it)
    int acc[PIL_HROWS][OC];
#pragma unroll
    for (int r = 0; r < PIL_HROWS; r++)
#pragma unroll
        for (int c = 0; c < OC; c++) acc[r][c] = 1 << 21;
    const bool words = NC == 4 && (reinterpret_cast<uintptr_t>(im.src) & 3) == 0;   // (pitch = 4 * width: every pixel aligned)
    for (int x = 0; x < count; x++) {
        const int k = __ldg(kk + (size_t)x * prm.ow);
#pragma unroll
        for (int r = 0; r < PIL_HROWS; r++) {
            const uint8_t *p = row[r] + x * NC;
            if (NC == 4 && words) {
                const u32 wd = __ldg(reinterpret_cast<const u32 *>(p));
#pragma unroll
                for (int c = 0; c < OC; c++) acc[r][c] += (int)((wd >> (8 * c)) & 0xffu) * k;
            } else {
#pragma unroll
                for (int c = 0; c < OC; c++) acc[r][c] += (int)__ldg(p + c) * k;
            }
        }
    }
    uint8_t *t = im.tmp + (size_t)r0 * pp.tpitch + (size_t)j * OC;
#pragma unroll
    for (int r = 0; r < PIL_HROWS; r++)
        if (r < nr)
#pragma unroll
            for (int c = 0; c < OC; c++) t[(size_t)r * pp.tpitch + c] = (uint8_t)clip8(acc[r][c]);
}

// Vertical pass: a thread produces 8 consecutive pixels of one slot row (8 warps: 8 rows), reading 8 * OC intermediate bytes
// per tap as OC 8-byte words (tpitch and the window columns are multiples of 8 pixels), and stores them as the resize does.
template <typename T, bool CHW, int OC>
__global__ void __launch_bounds__(256) pil_vertical_kernel(const PilImage *__restrict__ images, const ResizeParams prm, const PilParams pp)
{
    const PilImage im = images[blockIdx.z];
    const u32 i = blockIdx.y * RZ_ROWS + (threadIdx.x >> 5);
    const u32 x0 = 8u * (blockIdx.x * 32u + (threadIdx.x & 31));
    if (i >= prm.oh || x0 >= prm.ow) return;
    const int *tv = im.tab + im.tab_v;
    const int ymin = tv[i] - (int)im.y0, count = tv[prm.oh + i];
    const int *kk = tv + 2 * prm.oh + i;
    int acc[8][OC];
#pragma unroll
    for (int e = 0; e < 8; e++)
#pragma unroll
        for (int c = 0; c < OC; c++) acc[e][c] = 1 << 21;
    const uint8_t *q = im.tmp + (size_t)ymin * pp.tpitch + (size_t)x0 * OC;
    for (int y = 0; y < count; y++, q += pp.tpitch) {
        const int k = __ldg(kk + (size_t)y * prm.oh);
        uint2 wd[OC];
#pragma unroll
        for (int g = 0; g < OC; g++) wd[g] = __ldg(reinterpret_cast<const uint2 *>(q) + g);
#pragma unroll
        for (int b = 0; b < 8 * OC; b++) {
            const u32 word = (b & 7) < 4 ? wd[b >> 3].x : wd[b >> 3].y;
            acc[b / OC][b % OC] += (int)((word >> (8 * (b & 3))) & 0xffu) * k;
        }
    }
    T v[8][OC];
#pragma unroll
    for (int e = 0; e < 8; e++)
#pragma unroll
        for (int c = 0; c < OC; c++) {
            const u32 u = clip8(acc[e][c]);
            v[e][c] = sizeof(T) == 1 ? (T)u : normalise<T>((float)u, prm.mean[c], prm.inv_std[c]);
        }
    store_px8<T, CHW, OC>(reinterpret_cast<T *>(im.dst), prm, i, x0, (int)min(8u, prm.ow - x0), v);
}

template <typename T, bool CHW>
static void launch_pil_vertical(const PilImage *d, uint32_t count, uint32_t oc, const ResizeParams &prm, const PilParams &pp, cudaStream_t s)
{
    const dim3 grid((prm.ow + 255) / 256, (prm.oh + RZ_ROWS - 1) / RZ_ROWS, count);
    if (oc == 1) pil_vertical_kernel<T, CHW, 1><<<grid, 256, 0, s>>>(d, prm, pp);
    else if (oc == 3) pil_vertical_kernel<T, CHW, 3><<<grid, 256, 0, s>>>(d, prm, pp);
    else pil_vertical_kernel<T, CHW, 4><<<grid, 256, 0, s>>>(d, prm, pp);
}

template <typename T>
static void launch_pil_vertical_t(const PilImage *d, uint32_t count, uint32_t oc, bool chw, const ResizeParams &prm, const PilParams &pp, cudaStream_t s)
{
    if (chw) launch_pil_vertical<T, true>(d, count, oc, prm, pp, s);
    else launch_pil_vertical<T, false>(d, count, oc, prm, pp, s);
}

// Intermediate and table bytes per launch of the passes: a run whose images need more is cut into sub-batches that take turns
// in one scratch buffer (at least one image each)
constexpr size_t PIL_CHUNK_BYTES = (size_t)1 << 30;

cudaError_t launch_pil_resize(const ResizeImage *host, uint32_t count, uint32_t nc, const zj_output_desc &d, const zj_resize &r,
                              int device, cudaStream_t s, int *launches)
{
    ResizeParams prm;
    for (int c = 0; c < 4; c++) { prm.mean[c] = d.mean[c]; prm.inv_std[c] = d.inv_std[c]; }
    prm.ow = r.out_w;
    prm.oh = r.out_h;
    const uint32_t oc = (d.channels == 3 && nc == 4) ? 3u : nc;
    PilParams pp;
    pp.filter = r.filter;
    pp.tpitch = ((r.out_w + 7u) & ~7u) * oc;
    const double s0 = pil_support0(r.filter);
    auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
    // per image: geometry, table strides (at most 2 * ceil(support) + 1 taps, as Pillow's), and its table + intermediate bytes
    std::vector<PilImage> im(count);
    std::vector<size_t> off(count);
    struct Chunk { uint32_t first, count, max_rows; size_t bytes; };
    std::vector<Chunk> chunks;
    size_t scratch = 0;
    for (uint32_t k = 0; k < count; k++) {
        const ResizeImage &ri = host[k];
        PilGeometry g;
        if (pil_geometry(r, ri.w, ri.h, &g) != ZJ_OK) return cudaErrorInvalidValue;   // (never: the callers admitted the crops)
        PilImage &p = im[k];
        p.src = ri.src; p.dst = ri.dst; p.pitch = ri.pitch; p.w = ri.w; p.h = ri.h;
        p.rw = g.rw; p.rh = g.rh; p.left = g.left; p.top = g.top; p.y0 = g.y0; p.rows = g.y1 - g.y0;
        auto ksize = [&](uint32_t n_in, uint32_t n_out) {
            const double sup = pil_mul(s0, std::max(pil_div((double)n_in, (double)n_out), 1.0));
            return 2u * (uint32_t)std::ceil(sup) + 1u;
        };
        p.ksh = ksize(ri.w, g.rw);
        p.ksv = ksize(ri.h, g.rh);
        p.tab_v = (uint32_t)(align((size_t)r.out_w * (2 + p.ksh) * 4) / 4);
        const size_t tab_bytes = align(((size_t)p.tab_v + (size_t)r.out_h * (2 + p.ksv)) * 4);
        const size_t bytes = tab_bytes + align((size_t)p.rows * pp.tpitch);
        if (chunks.empty() || chunks.back().bytes + bytes > PIL_CHUNK_BYTES) chunks.push_back({k, 0, 0, 0});
        Chunk &ch = chunks.back();
        off[k] = ch.bytes;
        ch.bytes += bytes;
        ch.count++;
        ch.max_rows = std::max(ch.max_rows, p.rows);
        scratch = std::max(scratch, ch.bytes);
    }
    const size_t desc_bytes = align(count * sizeof(PilImage));
    uint8_t *buf = nullptr;
    if (scratch_alloc((void **)&buf, desc_bytes + scratch, device, s) != ZJ_OK) return cudaErrorMemoryAllocation;
    uint8_t *const work = buf + desc_bytes;
    for (uint32_t k = 0; k < count; k++) {
        im[k].tab = reinterpret_cast<int *>(work + off[k]);
        im[k].tmp = work + off[k] + align(((size_t)im[k].tab_v + (size_t)r.out_h * (2 + im[k].ksv)) * 4);
    }
    PilImage *dev = reinterpret_cast<PilImage *>(buf);
    // (pageable source: the async copy returns once the data sits in the driver's staging buffer)
    cudaError_t e = cudaMemcpyAsync(dev, im.data(), count * sizeof(PilImage), cudaMemcpyHostToDevice, s);
    // the sub-batches take turns in the scratch buffer, in the order of s
    for (size_t c = 0; c < chunks.size() && e == cudaSuccess; c++) {
        const Chunk &ch = chunks[c];
        const PilImage *di = dev + ch.first;
        pil_table_kernel<<<dim3((std::max(r.out_w, r.out_h) + 255) / 256, 2, ch.count), 256, 0, s>>>(di, prm, pp);
        const dim3 gh((r.out_w + 31) / 32, (ch.max_rows + 8 * PIL_HROWS - 1) / (8 * PIL_HROWS), ch.count);
        if (nc == 1) pil_horizontal_kernel<1, 1><<<gh, 256, 0, s>>>(di, prm, pp);
        else if (nc == 3) pil_horizontal_kernel<3, 3><<<gh, 256, 0, s>>>(di, prm, pp);
        else if (oc == 3) pil_horizontal_kernel<4, 3><<<gh, 256, 0, s>>>(di, prm, pp);
        else pil_horizontal_kernel<4, 4><<<gh, 256, 0, s>>>(di, prm, pp);
        const bool chw = d.layout == ZJ_LAYOUT_CHW;
        switch (d.dtype) {
        case ZJ_DTYPE_U8: launch_pil_vertical_t<uint8_t>(di, ch.count, oc, chw, prm, pp, s); break;
        case ZJ_DTYPE_F16: launch_pil_vertical_t<__half>(di, ch.count, oc, chw, prm, pp, s); break;
        default: launch_pil_vertical_t<float>(di, ch.count, oc, chw, prm, pp, s); break;
        }
        *launches += 3;
        e = cudaGetLastError();
    }
    scratch_free(buf, s);
    return e;
}

// ------------------------------------------------------------------------------------------------------ orientation
// The EXIF orientation pass (DESIGN.md section 4.6.3): Pillow's Transpose of a region of u8 pixels, each pixel's NC bytes moving
// together.  One CTA moves one OT x OT source tile through shared memory, so that the loads run along source rows and the
// stores along destination rows: aligned 32-bit words wherever the word lies inside the row segment, bytes at its unaligned
// ends.  No byte outside the source region is read, none outside the destination written.  Each thread issues all its loads
// before its first shared store, so that a CTA has its whole tile in flight.
constexpr int OT = 64;   // tile side in pixels

template <int NC>
__global__ void __launch_bounds__(256) orient_kernel(const OrientImage *__restrict__ images)
{
    // words per shared row: a row segment of OT * NC bytes starting at any offset mod 4 (odd, so that the column reads of the
    // transposing orientations spread over the banks)
    constexpr int P = (OT * NC + 3) / 4 + 1;
    constexpr int NW = (OT * P + 255) / 256;   // word slots per thread and phase
    __shared__ u32 tile[OT * P];
    const OrientImage im = images[blockIdx.z];
    const u32 x0 = blockIdx.x * OT, y0 = blockIdx.y * OT;
    if (x0 >= im.w || y0 >= im.h) return;
    const u32 tw = min((u32)OT, im.w - x0), th = min((u32)OT, im.h - y0);
    // tile row r holds source row y0 + r, pixels [x0, x0 + tw): its byte b at shared byte 4 P r + (offset of the row mod 4) + b
    const uint8_t *const src = im.src + (size_t)y0 * im.pitch + (size_t)x0 * NC;
    const u32 src_a = (u32)reinterpret_cast<uintptr_t>(src);
    {
        const int nb = (int)(tw * NC);
        u32 v[NW];
#pragma unroll
        for (int q = 0; q < NW; q++) {
            const u32 i = threadIdx.x + 256u * q, r = i / P, k = i - r * P;
            v[q] = 0;
            const int mis = (int)((src_a + r * im.pitch) & 3u), lo = 4 * (int)k - mis;   // the word's first byte in the row segment
            if (r >= th || lo >= nb) continue;
            const uint8_t *row = src + (size_t)r * im.pitch;
            if (lo >= 0 && lo + 4 <= nb) {
                v[q] = __ldg(reinterpret_cast<const u32 *>(row + lo));
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++)
                    if (lo + j >= 0 && lo + j < nb) v[q] |= (u32)__ldg(row + lo + j) << (8 * j);
            }
        }
#pragma unroll
        for (int q = 0; q < NW; q++) {
            const u32 i = threadIdx.x + 256u * q;
            if (i < th * P) tile[i] = v[q];
        }
    }
    __syncthreads();
    const uint8_t *const sb = reinterpret_cast<const uint8_t *>(tile);
    const bool fx = orient_flip_x(im.orient), fy = orient_flip_y(im.orient), sw = orient_swap(im.orient);
    // the tile's place in the destination: mirrored x' / y' ranges, axes swapped
    const u32 xm0 = fx ? im.w - x0 - tw : x0, ym0 = fy ? im.h - y0 - th : y0;
    const u32 dx0 = sw ? ym0 : xm0, dy0 = sw ? xm0 : ym0, dtw = sw ? th : tw, dth = sw ? tw : th;
    const u32 dpitch = (sw ? im.h : im.w) * NC;
    uint8_t *const dst = im.dst + (size_t)dy0 * dpitch + (size_t)dx0 * NC;
    const u32 dst_a = (u32)reinterpret_cast<uintptr_t>(dst);
    const int nb = (int)(dtw * NC);
#pragma unroll
    for (int q = 0; q < NW; q++) {
        const u32 i = threadIdx.x + 256u * q, r = i / P, k = i - r * P;
        const int mis = (int)((dst_a + r * dpitch) & 3u), lo = 4 * (int)k - mis;
        if (r >= dth || lo >= nb) continue;
        // the shared bytes of destination pixel p of row r: its local (x', y'), mirrored back to the source tile
        auto pixel = [&](u32 p) {
            const u32 xl = sw ? r : p, yl = sw ? p : r;
            const u32 sx = fx ? tw - 1 - xl : xl, sy = fy ? th - 1 - yl : yl;
            return sb + 4 * P * sy + ((src_a + sy * im.pitch) & 3u) + sx * NC;
        };
        const u32 b0 = (u32)max(lo, 0);
        u32 p = b0 / NC, c = b0 - p * NC;   // the word's first byte in the row: pixel p, channel c
        const uint8_t *px = pixel(p);
        u32 v = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int b = lo + j;
            if (b < 0 || b >= nb) continue;
            v |= (u32)px[c] << (8 * j);
            if (++c == NC && b + 1 < nb) { c = 0; px = pixel(++p); }
        }
        uint8_t *row = dst + (size_t)r * dpitch;
        if (lo >= 0 && lo + 4 <= nb) {
            *reinterpret_cast<u32 *>(row + lo) = v;
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (lo + j >= 0 && lo + j < nb) row[lo + j] = (uint8_t)(v >> (8 * j));
        }
    }
}

cudaError_t launch_orient(const OrientImage *d_images, uint32_t count, uint32_t nc, uint32_t max_w, uint32_t max_h, cudaStream_t s)
{
    const dim3 grid((max_w + OT - 1) / OT, (max_h + OT - 1) / OT, count);
    if (nc == 1) orient_kernel<1><<<grid, 256, 0, s>>>(d_images);
    else if (nc == 3) orient_kernel<3><<<grid, 256, 0, s>>>(d_images);
    else orient_kernel<4><<<grid, 256, 0, s>>>(d_images);
    return cudaGetLastError();
}

}  // namespace zj
