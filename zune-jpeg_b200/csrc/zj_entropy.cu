// zj_entropy.cu -- baseline Huffman entropy decode of restart intervals on the GPU (SURVEY 8(f).1, "or on-GPU").
//
// One thread per restart interval.  A thread is the reference's sequential decoder confined to its interval: the bit
// reader of src/bitstream.rs (64-bit buffer refilled 32 bits at a time, 0xFF00 un-stuffing, "marker seen" state with its
// faked zero bits, rotate-based get_bits: :159-261, :394-402), decode_mcu_block with the fast-AC table (:314-373, Q9 and
// Q10 included -- they live in the tables and in the refill thresholds, both reproduced as written), and the MCU loop of
// src/mcu.rs:253-351 with the restart bookkeeping of :386-418 (Q8: the countdown ticks once per component).  Coefficients
// go straight into the zeroed device planes (raster block order, natural coefficient order: the layout the
// reconstruction kernels read).
//
// An interval is accepted (status 0) only if the reset of handle_rst fired exactly after the last component of its last
// MCU, with the reader standing where the next interval was assumed to start, and nothing else the sequential loop
// reacts to was met before (an early reset, EOI, another marker, a decode error, a block outside its strip).  If every
// interval of an image is accepted, the sequential loop would have gone through exactly the same states; otherwise the
// host stage decodes the image (zj_host_decoder.cpp), so the planes are always what the reference's loop produces.
//
// Work per thread is bit-serial and divergent by nature (this is the "branchy" stage); what the GPU offers is tens of
// thousands of intervals in flight at once -- a batch of 64 8192x8192 images is 32768 independent intervals -- and no
// PCIe upload of coefficient planes (201 MB per such image; its JPEG file is 12 MB).
#include <cuda_runtime.h>
#include <stdlib.h>
#include <stdint.h>

#include "zj_entropy.h"

namespace zj {

typedef unsigned long long u64;
typedef uint32_t u32;

__constant__ uint8_t c_unzigzag[80] = {  // src/misc.rs:30-41 (16 entries of padding)
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63,
    63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63};

enum { MK_NONE = 0, MK_RST = 1, MK_EOI = 2 };

struct Reader {                    // BitStream + Cursor of one interval
    const uint8_t *data;
    u32 len, pos;
    u64 buffer, aligned;
    u32 bits_left;
    int marker;                    // MK_*; has_marker == (marker != MK_NONE)
    bool bad;                      // something the interval-local decode cannot stand for: the host stage takes over

    __device__ __forceinline__ u32 read_u8_or_zero() { const u32 v = pos < len ? (u32)__ldg(data + pos) : 0u; pos++; return v; }

    // bitstream.rs:159-261
    __device__ __forceinline__ void refill()
    {
        if (bits_left > 32 && marker == MK_NONE) return;
        if (marker != MK_NONE) { bits_left = 63; return; }   // fake zero bits after a marker (:254-258)
        refill_body();
    }
    __device__ __forceinline__ void refill_body()
    {
        const u32 position = pos;
        if (position + 4 < len) {
            const u32 msb = ((u32)__ldg(data + position) << 24) | ((u32)__ldg(data + position + 1) << 16) | ((u32)__ldg(data + position + 2) << 8) | (u32)__ldg(data + position + 3);
            const u32 v = msb ^ 0xFFFFFFFFu;   // has_byte(msb, 255), :705-717
            if ((~((((v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | v) | 0x7F7F7F7Fu)) == 0) {
                pos = position + 4;
                bits_left += 32;
                buffer = (buffer << 32) | msb;
                aligned = buffer << (64 - bits_left);
                return;
            }
        }
        for (int k = 0; k < 4; k++) {
            const u32 byte = read_u8_or_zero();
            buffer = (buffer << 8) | byte;
            bits_left += 8;
            if (byte == 0xff) {
                u32 next = read_u8_or_zero();
                if (next != 0x00) {
                    while (next == 0xFF) next = read_u8_or_zero();
                    if (next != 0x00) {
                        buffer >>= 8;
                        bits_left -= 8;
                        if (bits_left != 0) aligned = buffer << (64 - bits_left);
                        if (next >= 0xD0 && next <= 0xD7) marker = MK_RST;
                        else if (next == 0xD9) marker = MK_EOI;
                        else { marker = MK_EOI; bad = true; }   // any other marker (or an unknown one) ends the interval-local decode
                        return;
                    }
                }
            }
        }
        aligned = buffer << (64 - bits_left);
    }
    __device__ __forceinline__ int peek9() const { return (int)(aligned >> 55); }
    __device__ __forceinline__ int peek16() const { return (int)(aligned >> 48); }
    __device__ __forceinline__ void drop_bits(u32 n)
    {
        bits_left = bits_left > n ? bits_left - n : 0;
        aligned = n >= 64 ? 0 : aligned << n;
    }
    __device__ __forceinline__ int get_bits(u32 n)   // :394-402 (a rotate, not a shift)
    {
        const u64 mask = (1ull << n) - 1;
        const u32 r = n & 63;
        aligned = r ? (aligned << r) | (aligned >> (64 - r)) : aligned;
        const int bits = (int)(aligned & mask);
        bits_left = bits_left > n ? bits_left - n : 0;
        return bits;
    }
    __device__ __forceinline__ void reset() { bits_left = 0; marker = MK_NONE; buffer = 0; aligned = 0; }   // :673-680
};

__device__ __forceinline__ int huff_extend(int x, int s)   // bitstream.rs:685-689
{
    return x + (((x - (1 << (s - 1))) >> 31) & (int)(((u32)-1 << s) + 1));
}

// decode_huff! macro, bitstream.rs:49-90
__device__ __forceinline__ void decode_huff(Reader &r, int &symbol, const EntTable &t)
{
    int code_length = symbol >> 9;
    symbol &= 511;
    if (code_length > 9) {
        symbol = r.peek16();
        while (code_length < 17) {
            if (symbol < t.maxcode[code_length]) break;
            code_length++;
        }
        if (code_length == 17) { r.bad = true; return; }   // "Bad Huffman Code"
        symbol >>= (16 - code_length);
        symbol = t.values[(symbol + t.offset[code_length]) & 0xFF];
    }
    r.drop_bits((u32)code_length);
}

// decode_mcu_block, bitstream.rs:314-373; block == nullptr: the component is not output, its coefficients are dropped
__device__ __forceinline__ void decode_block(Reader &r, const EntTable &dc, const EntTable &ac, const uint8_t *__restrict__ unzigzag, int16_t *__restrict__ block, int &pred)
{
    // decode_dc, :272-297 (refills only below 16 buffered bits, Q10)
    if (r.bits_left < 16) r.refill();
    int symbol = dc.lookup[r.peek9()];
    decode_huff(r, symbol, dc);
    if (r.bad) return;
    if (symbol != 0) { const int rr = r.get_bits((u32)symbol); symbol = huff_extend(rr, symbol); }
    pred = (int)((u32)pred + (u32)symbol);
    if (block) block[0] = (int16_t)pred;
    u32 pos = 1;
    while (pos < 64) {
        r.refill();
        if (r.bad) return;
        symbol = r.peek9();
        const int fast_ac = (int)ac.ac_lookup[symbol];
        if (fast_ac != 0) {
            pos += (u32)((fast_ac >> 4) & 63);
            if (block) block[unzigzag[pos < 63 ? pos : 63] & 63] = (int16_t)(fast_ac >> 10);
            r.drop_bits((u32)(fast_ac & 15));
            pos += 1;
        } else {
            symbol = ac.lookup[symbol];
            decode_huff(r, symbol, ac);
            if (r.bad) return;
            int rr = symbol >> 4;
            symbol &= 15;
            if (symbol != 0) {
                pos += (u32)rr;
                rr = r.get_bits((u32)symbol);
                symbol = huff_extend(rr, symbol);
                if (block) block[unzigzag[pos & 63] & 63] = (int16_t)symbol;
                pos += 1;
            } else if (rr != 15) {
                return;
            } else {
                pos += 16;
            }
        }
    }
}

template <int ENT_LANES>
__global__ void __launch_bounds__(ENT_THREADS) entropy_kernel(const EntImage *__restrict__ images)
{
    __shared__ EntTable sT[6];
    __shared__ uint8_t sZ[80];   // (threads index it with different positions: a constant-bank access would be serialised)
    const EntImage &im = images[blockIdx.y];
    constexpr u32 ENT_SEGS = ENT_THREADS / 32 * ENT_LANES;   // intervals per CTA
    if (blockIdx.x * ENT_SEGS >= im.n_seg) return;
    {   // the image's tables: [dc, ac] per component
        const u32 words = (u32)(sizeof(EntTable) / 4) * 2u * im.ncomp;
        const u32 *src = reinterpret_cast<const u32 *>(im.tables);
        u32 *dst = reinterpret_cast<u32 *>(sT);
        for (u32 i = threadIdx.x; i < words; i += ENT_THREADS) dst[i] = src[i];
    }
    for (u32 i = threadIdx.x; i < 80; i += ENT_THREADS) sZ[i] = c_unzigzag[i];
    __syncthreads();
    if ((threadIdx.x & 31u) >= (u32)ENT_LANES) return;
    const u32 k = blockIdx.x * ENT_SEGS + (threadIdx.x >> 5) * ENT_LANES + (threadIdx.x & 31u);
    if (k >= im.n_seg) return;

    Reader r;
    r.data = im.data; r.len = im.len; r.pos = im.seg_start[k];
    r.buffer = 0; r.aligned = 0; r.bits_left = 0; r.marker = MK_NONE; r.bad = false;
    int dc0 = 0, dc1 = 0, dc2 = 0;   // predictors (kept in registers: no dynamically indexed array)
    u32 todo = im.restart_interval;
    const u32 first = k * im.per_seg, last = min(im.total_mcus, first + im.per_seg);
    const bool must_reset = k + 1 < im.n_seg;
    const u32 per_strip = im.bias * im.mcu_w, ncomp = im.ncomp;
    bool ok = true, was_reset = false;

    for (u32 m = first; m < last && ok && !was_reset; m++) {
        const u32 strip = m / per_strip, v = (m - strip * per_strip) / im.mcu_w, j = m - strip * per_strip - v * im.mcu_w;
        for (u32 pos = 0; pos < ncomp; pos++) {
            const EntTable &dc = sT[2 * pos], &ac = sT[2 * pos + 1];
            const u32 hs = im.h_samp[pos], vs = im.v_samp[pos], is_y = im.is_y[pos];
            int16_t *plane = im.plane[pos];
            for (u32 v_samp = 0; v_samp < vs && ok; v_samp++) {
                for (u32 h_samp = 0; h_samp < hs && ok; h_samp++) {
                    int16_t *block = nullptr;
                    if (plane) {
                        // mcu.rs:293-312
                        const u32 y_offset = is_y * v * (im.hv_width_stride + (im.hv_width_stride * (vs - 1)));
                        const u32 another_stride = im.is_hv ? im.hv_width_stride * v_samp : im.width_stride * v_samp;
                        const u32 yet_another_stride = (im.is_hv && !is_y) ? (im.width_stride >> 2) * v : 0u;
                        const u32 start = (j * 64 * hs) + (h_samp * 64) + another_stride + y_offset + yet_another_stride;
                        if (start + 64 > im.strip_len[pos]) { ok = false; break; }   // the reference panics here (mcu.rs:314)
                        block = plane + (size_t)strip * im.strip_len[pos] + start;
                    }
                    int pred = pos == 0 ? dc0 : (pos == 1 ? dc1 : dc2);
                    decode_block(r, dc, ac, sZ, block, pred);
                    if (pos == 0) dc0 = pred; else if (pos == 1) dc1 = pred; else dc2 = pred;
                    if (r.bad) ok = false;
                }
            }
            if (!ok) break;
            todo = todo - 1;           // once per COMPONENT (Q8)
            if (todo == 0) {           // handle_rst, mcu.rs:386-418
                todo = im.restart_interval;
                if (r.marker == MK_RST) {
                    r.reset();
                    dc0 = dc1 = dc2 = 0;
                    if (m + 1 == last && pos + 1 == ncomp) was_reset = true;
                    else ok = false;   // a reset in the middle of the interval
                    break;
                }
            }
            if (r.marker != MK_NONE) {   // mcu.rs:337-348
                if (r.marker == MK_EOI) {
                    if (must_reset) ok = false;
                    break;
                }
                continue;                // RSTn met ahead of the countdown: keep going on faked zero bits
            }
        }
    }
    if (ok && must_reset && (!was_reset || r.pos != im.seg_start[k + 1])) ok = false;
    im.status[k] = ok ? 0 : 1;
}

template <int LANES>
static int launch_lanes(const EntImage *d_images, uint32_t n_images, uint32_t max_seg, cudaStream_t s)
{
    constexpr uint32_t SEGS = ENT_THREADS / 32 * LANES;
    dim3 grid((max_seg + SEGS - 1) / SEGS, n_images);
    entropy_kernel<LANES><<<grid, ENT_THREADS, 0, s>>>(d_images);
    return (int)cudaGetLastError();
}

int launch_entropy(const EntImage *d_images, uint32_t n_images, uint32_t max_seg, void *stream)
{
    if (n_images == 0 || max_seg == 0) return 0;
    const uint64_t intervals = (uint64_t)n_images * max_seg;          // (an upper bound: images of one launch may differ)
    cudaStream_t s = (cudaStream_t)stream;
    if (intervals < 12000) return launch_lanes<8>(d_images, n_images, max_seg, s);
    if (intervals < 24000) return launch_lanes<16>(d_images, n_images, max_seg, s);
    return launch_lanes<32>(d_images, n_images, max_seg, s);
}

}  // namespace zj
