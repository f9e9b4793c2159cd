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

// decode_mcu_block, bitstream.rs:314-373; block == nullptr: the component is not output, its coefficients are dropped.
// SPEC: Q10 off (the DC refill happens whenever <= 32 bits are buffered, as before every AC symbol)
template <bool SPEC>
__device__ __forceinline__ void decode_block(Reader &r, const EntTable &dc, const EntTable &ac, const uint8_t *__restrict__ unzigzag, int16_t *__restrict__ block, int &pred)
{
    // decode_dc, :272-297 (refills only below 16 buffered bits, Q10)
    if (SPEC || r.bits_left < 16) r.refill();
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

// SPEC: the loop of a spec decode (Q10 and Q11 off); the acceptance rule and the Q8 bookkeeping are the same
template <int ENT_LANES, bool SPEC>
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
                    decode_block<SPEC>(r, dc, ac, sZ, block, pred);
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
                    if (!SPEC) break;      // Q11; spec: finish the MCU on the bits already buffered
                    continue;
                }
                continue;                // RSTn met ahead of the countdown: keep going on faked zero bits
            }
        }
    }
    if (ok && must_reset && (!was_reset || r.pos != im.seg_start[k + 1])) ok = false;
    im.status[k] = ok ? 0 : 1;
}

template <int LANES>
static int launch_lanes(const EntImage *d_images, uint32_t n_images, uint32_t max_seg, cudaStream_t s, bool spec)
{
    constexpr uint32_t SEGS = ENT_THREADS / 32 * LANES;
    dim3 grid((max_seg + SEGS - 1) / SEGS, n_images);
    if (spec) entropy_kernel<LANES, true><<<grid, ENT_THREADS, 0, s>>>(d_images);
    else entropy_kernel<LANES, false><<<grid, ENT_THREADS, 0, s>>>(d_images);
    return (int)cudaGetLastError();
}

int launch_entropy(const EntImage *d_images, uint32_t n_images, uint32_t max_seg, void *stream, bool spec)
{
    if (n_images == 0 || max_seg == 0) return 0;
    const uint64_t intervals = (uint64_t)n_images * max_seg;          // (an upper bound: images of one launch may differ)
    cudaStream_t s = (cudaStream_t)stream;
    if (intervals < 12000) return launch_lanes<8>(d_images, n_images, max_seg, s, spec);
    if (intervals < 24000) return launch_lanes<16>(d_images, n_images, max_seg, s, spec);
    return launch_lanes<32>(d_images, n_images, max_seg, s, spec);
}

// ================================================================ scans without restart markers (spec and libjpeg output)
// Phases per sub-batch, all on one stream: SYNC_ROUNDS launches of sync_round_kernel, then accept_kernel, write_kernel and
// dc_kernel.  The de-stuffing (FF 00 -> FF, fill bytes dropped) is done by the host stage while it looks for the scan's end.
//
// Bounds: a decode runs only while its position is below its end (<= nbits) and refills only when <= 32 bits are buffered, so
// the highest word it loads is (pos + 32) / 32 <= nbits / 32 + 1, inside the >= 8 zero bytes after the data.  Table reads are
// indexed by 9-bit peeks, code lengths 1..17 and `& 0xFF`; coefficient positions are checked <= 63 before a store.  Stores
// happen only in write_kernel and dc_kernel, from the states accept_kernel verified, at block indices below the total, after
// the addressing check of mcu.rs:293-312 (start + 64 <= strip_len).  State words and counters are indexed by the thread's own
// subsequence k < n_sub, its predecessor k - 1, or the round r < SYNC_ROUNDS.

struct SyncBits {          // a bit reader over the de-stuffed scan: the next nb (>= 33 after refill) bits sit at the top of buf
    const uint32_t *w;
    u64 buf, pos;
    u32 nb, wi;
    __device__ __forceinline__ u32 word(u32 i) const { return __byte_perm(__ldg(w + i), 0, 0x0123); }
    __device__ __forceinline__ void init(const uint32_t *words, u64 p)
    {
        w = words; pos = p;
        wi = (u32)(p >> 5);
        buf = ((u64)word(wi) << 32) | word(wi + 1);
        wi += 2;
        const u32 s = (u32)(p & 31);
        buf <<= s;
        nb = 64 - s;
    }
    __device__ __forceinline__ void refill() { if (nb <= 32) { buf |= (u64)word(wi++) << (32 - nb); nb += 32; } }
    __device__ __forceinline__ u32 peek(u32 n) const { return (u32)(buf >> (64 - n)); }
    __device__ __forceinline__ void drop(u32 n) { buf <<= n; nb -= n; pos += n; }
    __device__ __forceinline__ int get(u32 n) { const int v = (int)peek(n); drop(n); return v; }
};

// decode_huff! (bitstream.rs:49-90) on SyncBits: the symbol, or -1 for a code the table does not hold
__device__ __forceinline__ int sync_huff(SyncBits &b, const EntTable &t, int symbol)
{
    int code_length = symbol >> 9;
    symbol &= 511;
    if (code_length > 9) {
        symbol = (int)b.peek(16);
        while (code_length < 17) {
            if (symbol < t.maxcode[code_length]) break;
            code_length++;
        }
        if (code_length == 17) return -1;
        symbol >>= (16 - code_length);
        symbol = t.values[(symbol + t.offset[code_length]) & 0xFF];
    }
    b.drop((u32)code_length);
    return symbol;
}

__device__ __forceinline__ u64 sync_state(u64 pos, u32 slot, u32 coef) { return pos << 16 | slot << 8 | coef; }

// mcu.rs:293-312 for global block g: its coefficients, nullptr when its component is not output; ok = false when the
// reference would index outside the strip
__device__ __forceinline__ int16_t *sync_block(const SyncImage &im, u32 g, bool &ok)
{
    const u32 m = g / im.bpm, slot = g - m * im.bpm;
    const u32 pos = im.slot_comp[slot], v_samp = im.slot_v[slot], h_samp = im.slot_h[slot];
    int16_t *plane = im.plane[pos];
    if (!plane) return nullptr;
    const u32 per_strip = im.bias * im.mcu_w;
    const u32 strip = m / per_strip, v = (m - strip * per_strip) / im.mcu_w, j = m - strip * per_strip - v * im.mcu_w;
    const u32 hs = im.h_samp[pos], vs = im.v_samp[pos], is_y = im.is_y[pos];
    const u32 y_offset = is_y * v * (im.hv_width_stride + (im.hv_width_stride * (vs - 1)));
    const u32 another_stride = im.is_hv ? im.hv_width_stride * v_samp : im.width_stride * v_samp;
    const u32 yet_another_stride = (im.is_hv && !is_y) ? (im.width_stride >> 2) * v : 0u;
    const u32 start = (j * 64 * hs) + (h_samp * 64) + another_stride + y_offset + yet_another_stride;
    if (start + 64 > im.strip_len[pos]) { ok = false; return nullptr; }
    return plane + (size_t)strip * im.strip_len[pos] + start;
}

// The host stage's decode_mcu_block (bitstream.rs:314-373 with Q9-Q11 off), one symbol at a time, from state (pos, slot,
// coef) over the symbols that start below `end`.  Returns the exit state, or SYNC_INVALID on a code the table does not hold,
// a non-zero coefficient past index 63 or a symbol that ends beyond nbits; `blocks` = blocks completed before that.
// WRITE: g0 = global index of the block in progress at the entry; coefficients and DC differences are stored for blocks
// below `total`, and the decode stops at block `total`; ok = false when an addressing check fails.
template <bool WRITE>
__device__ u64 sync_decode(const SyncImage &im, const EntTable *T, const uint8_t *Z, u64 pos, u32 slot, u32 coef, u64 end,
                           u32 &blocks, u32 g0, u32 total, bool &ok)
{
    blocks = 0;
    if (pos >= end) return sync_state(pos, slot, coef);
    SyncBits b;
    b.init(im.bits, pos);
    int16_t *blk = nullptr;
    if (WRITE) { if (g0 >= total) return sync_state(pos, slot, coef); blk = sync_block(im, g0, ok); }
    while (b.pos < end) {
        if (WRITE && !ok) break;
        const u32 comp = im.slot_comp[slot];
        const EntTable &dc = T[2 * comp], &ac = T[2 * comp + 1];
        b.refill();
        if (coef == 0) {
            int s = sync_huff(b, dc, dc.lookup[b.peek(9)]);
            if (s < 0) return SYNC_INVALID;
            int v = 0;
            if (s != 0) v = huff_extend(b.get((u32)s), s);
            if (WRITE) im.dc[g0 + blocks] = (int16_t)v;
            coef = 1;
        } else {
            const int fast_ac = (int)ac.ac_lookup[b.peek(9)];
            if (fast_ac != 0) {
                coef += (u32)((fast_ac >> 4) & 63);
                const int v = fast_ac >> 10;
                if (v != 0) {
                    if (coef > 63) return SYNC_INVALID;
                    if (WRITE && blk) blk[Z[coef] & 63] = (int16_t)v;
                }
                b.drop((u32)(fast_ac & 15));
                coef += 1;
            } else {
                int s = sync_huff(b, ac, ac.lookup[b.peek(9)]);
                if (s < 0) return SYNC_INVALID;
                const u32 rr = (u32)s >> 4;
                s &= 15;
                if (s != 0) {
                    coef += rr;
                    if (coef > 63) return SYNC_INVALID;
                    const int v = huff_extend(b.get((u32)s), s);
                    if (WRITE && blk) blk[Z[coef] & 63] = (int16_t)v;
                    coef += 1;
                } else if (rr != 15) {
                    coef = 64;
                } else {
                    coef += 16;
                }
            }
        }
        if (b.pos > im.nbits) return SYNC_INVALID;
        if (coef >= 64) {
            blocks++;
            coef = 0;
            slot = slot + 1 == im.bpm ? 0 : slot + 1;
            if (WRITE) {
                if (g0 + blocks >= total) break;
                blk = sync_block(im, g0 + blocks, ok);
            }
        }
    }
    return sync_state(b.pos, slot, coef);
}

__device__ __forceinline__ void sync_tables(const SyncImage &im, EntTable *sT, uint8_t *sZ)
{
    const u32 words = (u32)(sizeof(EntTable) / 4) * 2u * (u32)(im.slot_comp[im.bpm - 1] + 1);
    const u32 *src = reinterpret_cast<const u32 *>(im.tables);
    u32 *dst = reinterpret_cast<u32 *>(sT);
    for (u32 i = threadIdx.x; i < words; i += SYNC_THREADS) dst[i] = src[i];
    for (u32 i = threadIdx.x; i < 80; i += SYNC_THREADS) sZ[i] = c_unzigzag[i];
    __syncthreads();
}

__device__ __forceinline__ u64 sync_end(const SyncImage &im, u32 k)
{
    return k + 1 == im.n_sub ? im.nbits : (u64)(k + 1) * SYNC_BITS;
}

// Round r: subsequence k's entry is its predecessor's exit of round r - 1 (round 0, or an invalid exit: the guess
// (k * SYNC_BITS, slot 0, coefficient 0)); subsequence 0 always starts at the scan start.  A subsequence decodes only when its
// entry differs from the one its last decode used.  A round in which no subsequence decodes is the fixpoint: both exit
// buffers then hold the same states, and later rounds return at once.
__global__ void __launch_bounds__(SYNC_THREADS) sync_round_kernel(const SyncImage *__restrict__ images, u32 r)
{
    __shared__ EntTable sT[6];
    __shared__ uint8_t sZ[80];
    const SyncImage &im = images[blockIdx.y];
    if (blockIdx.x * SYNC_THREADS >= im.n_sub) return;
    if (r >= 2 && im.changed[r - 1] == 0) return;
    sync_tables(im, sT, sZ);
    const u32 k = blockIdx.x * SYNC_THREADS + threadIdx.x;
    if (k >= im.n_sub) return;
    u64 entry = sync_state((u64)k * SYNC_BITS, 0, 0);
    if (k > 0 && r > 0) {
        const u64 e = im.exit[(r - 1) & 1][k - 1];
        if (e != SYNC_INVALID) entry = e;
    }
    if (r > 0 && entry == im.used[k]) { im.exit[r & 1][k] = im.exit[(r - 1) & 1][k]; return; }
    im.used[k] = entry;
    u32 blocks;
    bool ok = true;
    im.exit[r & 1][k] = sync_decode<false>(im, sT, sZ, entry >> 16, (u32)(entry >> 8) & 255, (u32)entry & 255, sync_end(im, k), blocks, 0, 0, ok);
    im.count[k] = blocks;
    atomicAdd(&im.changed[r], 1u);
}

// One CTA per image: takes the image when the rounds reached the fixpoint and the decode from the true entries completes
// total_mcus * bpm blocks before its first error (or without one); count[k] becomes subsequence k's first global block index.
__global__ void __launch_bounds__(1024) accept_kernel(const SyncImage *__restrict__ images)
{
    __shared__ u32 s_sum[1024];
    __shared__ u32 s_err;
    const SyncImage &im = images[blockIdx.x];
    bool settled = false;
    for (u32 r = 1; r < SYNC_ROUNDS; r++) settled = settled || im.changed[r] == 0;
    if (!settled) { if (threadIdx.x == 0) *im.status = 1; return; }
    if (threadIdx.x == 0) s_err = 0xFFFFFFFFu;
    const u32 n = im.n_sub, per = (n + 1023) / 1024;
    const u32 k0 = min(n, threadIdx.x * per), k1 = min(n, k0 + per);
    u32 sum = 0;
    for (u32 k = k0; k < k1; k++) sum += im.count[k];
    s_sum[threadIdx.x] = sum;
    __syncthreads();
    for (u32 d = 1; d < 1024; d <<= 1) {          // inclusive scan of the chunk sums
        const u32 v = threadIdx.x >= d ? s_sum[threadIdx.x - d] : 0u;
        __syncthreads();
        s_sum[threadIdx.x] += v;
        __syncthreads();
    }
    u32 base = s_sum[threadIdx.x] - sum;
    for (u32 k = k0; k < k1; k++) {
        const u32 c = im.count[k];
        im.count[k] = base;
        if (im.exit[0][k] == SYNC_INVALID) atomicMin(&s_err, k);
        base += c;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const u32 total = im.total_mcus * im.bpm;
        u64 reached;
        if (s_err != 0xFFFFFFFFu) {
            // the block in progress at the first error: the next subsequence's base (the scan total behind the last one)
            const u32 kb = s_err;
            reached = kb + 1 < n ? (u64)im.count[kb + 1] : (u64)s_sum[1023];
        } else {
            reached = s_sum[1023];
        }
        *im.status = reached >= total ? 0 : 1;
    }
}

// Subsequence k decodes again from its verified entry and stores the AC coefficients and DC differences of its blocks
__global__ void __launch_bounds__(SYNC_THREADS) write_kernel(const SyncImage *__restrict__ images)
{
    __shared__ EntTable sT[6];
    __shared__ uint8_t sZ[80];
    __shared__ uint8_t s_status;
    const SyncImage &im = images[blockIdx.y];
    if (blockIdx.x * SYNC_THREADS >= im.n_sub) return;
    // (other CTAs of the image may set the status while this one runs: one read per CTA, published by the barrier)
    if (threadIdx.x == 0) s_status = *im.status;
    sync_tables(im, sT, sZ);
    if (s_status != 0) return;
    const u32 k = blockIdx.x * SYNC_THREADS + threadIdx.x;
    if (k >= im.n_sub) return;
    const u32 total = im.total_mcus * im.bpm, g0 = im.count[k];
    if (g0 >= total) return;
    const u64 entry = k == 0 ? 0ull : im.exit[0][k - 1];
    if (entry == SYNC_INVALID) return;   // (not reached: subsequences behind an error start at or past block total)
    u32 blocks;
    bool ok = true;
    sync_decode<true>(im, sT, sZ, entry >> 16, (u32)(entry >> 8) & 255, (u32)entry & 255, sync_end(im, k), blocks, g0, total, ok);
    if (!ok) *im.status = 1;
}

// One CTA per image: the DC predictors, a wrapping 32-bit prefix sum of the differences per component in block order,
// stored as (int16_t)pred the way decode_dc does
__global__ void __launch_bounds__(1024) dc_kernel(const SyncImage *__restrict__ images)
{
    __shared__ u32 s_sum[3][1024];
    const SyncImage &im = images[blockIdx.x];
    if (*im.status != 0) return;
    const u32 mcus = im.total_mcus, per = (mcus + 1023) / 1024, bpm = im.bpm;
    const u32 m0 = min(mcus, threadIdx.x * per), m1 = min(mcus, m0 + per);
    u32 sum[3] = {0, 0, 0};
    for (u32 m = m0; m < m1; m++)
        for (u32 s = 0; s < bpm; s++) {
            const u32 c = im.slot_comp[s];
            const u32 d = (u32)(int)im.dc[m * bpm + s];
            sum[0] += c == 0 ? d : 0u; sum[1] += c == 1 ? d : 0u; sum[2] += c == 2 ? d : 0u;
        }
    for (int c = 0; c < 3; c++) s_sum[c][threadIdx.x] = sum[c];
    __syncthreads();
    for (u32 d = 1; d < 1024; d <<= 1) {
        u32 v[3];
        for (int c = 0; c < 3; c++) v[c] = threadIdx.x >= d ? s_sum[c][threadIdx.x - d] : 0u;
        __syncthreads();
        for (int c = 0; c < 3; c++) s_sum[c][threadIdx.x] += v[c];
        __syncthreads();
    }
    u32 pred[3];
    for (int c = 0; c < 3; c++) pred[c] = s_sum[c][threadIdx.x] - sum[c];
    for (u32 m = m0; m < m1; m++)
        for (u32 s = 0; s < bpm; s++) {
            const u32 c = im.slot_comp[s];
            const u32 d = (u32)(int)im.dc[m * bpm + s];
            u32 p = c == 0 ? pred[0] : (c == 1 ? pred[1] : pred[2]);
            p += d;
            if (c == 0) pred[0] = p; else if (c == 1) pred[1] = p; else pred[2] = p;
            bool ok = true;
            int16_t *blk = sync_block(im, m * bpm + s, ok);   // (checked by write_kernel: every block below the total was visited)
            if (blk) blk[0] = (int16_t)p;
        }
}

int launch_sync_phase(const SyncImage *d_images, uint32_t n_images, uint32_t max_sub, void *stream, int phase)
{
    if (n_images == 0 || max_sub == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const dim3 grid((max_sub + SYNC_THREADS - 1) / SYNC_THREADS, n_images);
    if (phase == SYNC_PHASE_ROUNDS)
        for (u32 r = 0; r < SYNC_ROUNDS; r++) sync_round_kernel<<<grid, SYNC_THREADS, 0, s>>>(d_images, r);
    else if (phase == SYNC_PHASE_ACCEPT) accept_kernel<<<n_images, 1024, 0, s>>>(d_images);
    else if (phase == SYNC_PHASE_WRITE) write_kernel<<<grid, SYNC_THREADS, 0, s>>>(d_images);
    else dc_kernel<<<n_images, 1024, 0, s>>>(d_images);
    return (int)cudaGetLastError();
}

// ================================================================ progressive scans (spec and libjpeg output)
// DESIGN.md section 5.6.  Reads are bounded as in the baseline decode: a decode stops once a read ends beyond nbits and loads at
// most one word past (pos + 32) / 32 <= nbits / 32 + 1, inside the >= 8 zero bytes behind the scan.  Stores go to blocks
// whose addressing check passed (prog_block), at zig-zag positions <= se <= 63, from verified states only: first scans store in
// their write pass once the accept kernel set `ok`, refinements store as they go and turn the image down on any error, so
// whatever they stored is never used.

// the host stage's block of scan block g (mcu_prog.rs:304 / :408 address rules), nullptr when that check fails
__device__ __forceinline__ int16_t *prog_block(const ProgScan &sc, u32 g)
{
    u32 z, x, y;
    if (sc.nslot > 1) {
        const u32 m = g / sc.nslot, s = g - m * sc.nslot, i = m / sc.mcu_x, j = m - i * sc.mcu_x;
        z = sc.slot_z[s];
        x = j * sc.hs[z] + sc.slot_h[s];
        y = i * sc.vs[z] + sc.slot_v[s];
    } else {
        z = sc.slot_z[0];
        y = g / sc.mw;
        x = g - y * sc.mw;
    }
    const u64 at = 64ull * ((u64)y * sc.bw[z] + x);
    if (at + 64 > sc.plane_len[z]) return nullptr;
    return sc.plane[z] + at;
}

// One symbol at a time of a first scan (DC first: decode_prog_dc_first, AC first: decode_mcu_ac_first with the host loop's
// EOB-run skip), from state (pos, slot, coef) over the symbols that start below `end`, as sync_decode does.  An EOB symbol
// completes its block and EOBRUN - 1 more.  SYNC_INVALID additionally on a non-zero coefficient past se.
// WRITE: stores DC differences / AC values (value << al) of blocks below total and stops there; *last = the start of the
// symbol that reached total; ok = false on a failed addressing check.
template <bool WRITE>
__device__ u64 prog_decode(const ProgScan &sc, const EntTable *T, const uint8_t *Z, u64 pos, u32 slot, u32 coef, u64 end,
                           u32 &blocks, u32 g0, bool &ok, u64 *last)
{
    blocks = 0;
    if (pos >= end) return sync_state(pos, slot, coef);
    SyncBits b;
    b.init(sc.bits, pos);
    const bool dc = sc.kind == PROG_DC_FIRST;
    const u32 ss = sc.ss, se = sc.se, al = sc.al;
    int16_t *blk = nullptr;
    if (WRITE) {
        if (g0 >= sc.total) return sync_state(pos, slot, coef);
        blk = prog_block(sc, g0);
        if (!blk) { ok = false; return sync_state(pos, slot, coef); }
    }
    while (b.pos < end) {
        const u64 start = b.pos;
        b.refill();
        u32 done = 0;
        if (dc) {
            const EntTable &t = T[sc.slot_t[slot]];
            const int s = sync_huff(b, t, t.lookup[b.peek(9)]);
            if (s < 0) return SYNC_INVALID;
            int v = 0;
            if (s != 0) v = huff_extend(b.get((u32)s), s);
            if (WRITE) sc.dc[g0 + blocks] = (int16_t)v;
            done = 1;
        } else {
            const EntTable &t = T[0];
            const int fast_ac = (int)t.ac_lookup[b.peek(9)];
            if (fast_ac != 0) {   // (progressive tables: only entries with a value)
                coef += (u32)((fast_ac >> 4) & 63);
                if (coef > se) return SYNC_INVALID;
                if (WRITE) blk[Z[coef] & 63] = (int16_t)((u32)(fast_ac >> 10) << al);
                b.drop((u32)(fast_ac & 15));
                coef += 1;
            } else {
                int s = sync_huff(b, t, t.lookup[b.peek(9)]);
                if (s < 0) return SYNC_INVALID;
                const u32 rr = (u32)s >> 4;
                s &= 15;
                if (s != 0) {
                    coef += rr;
                    if (coef > se) return SYNC_INVALID;
                    const int v = huff_extend(b.get((u32)s), s);
                    if (WRITE) blk[Z[coef] & 63] = (int16_t)((u32)v << al);
                    coef += 1;
                } else if (rr != 15) {
                    done = (1u << rr) + (rr ? (u32)b.get(rr) : 0u);   // EOBRUN blocks, this one included
                } else {
                    coef += 16;
                }
            }
            if (done == 0 && coef > se) done = 1;
        }
        if (b.pos > sc.nbits) return SYNC_INVALID;
        if (done) {
            blocks += done;
            coef = dc ? 0 : ss;
            slot = dc && slot + 1 < sc.nslot ? slot + 1 : 0;
            if (WRITE) {
                if (g0 + blocks >= sc.total) { *last = start; break; }
                blk = prog_block(sc, g0 + blocks);
                if (!blk) { ok = false; break; }
            }
        }
    }
    return sync_state(b.pos, slot, coef);
}

__device__ __forceinline__ void prog_tables(const ProgScan &sc, EntTable *sT, uint8_t *sZ, u32 nthreads)
{
    const u32 words = (u32)(sizeof(EntTable) / 4) * (sc.kind == PROG_DC_FIRST ? (u32)sc.slot_t[sc.nslot - 1] + 1 : 1u);
    const u32 *src = reinterpret_cast<const u32 *>(sc.tables);
    u32 *dst = reinterpret_cast<u32 *>(sT);
    for (u32 i = threadIdx.x; i < words; i += nthreads) dst[i] = src[i];
    for (u32 i = threadIdx.x; i < 80; i += nthreads) sZ[i] = c_unzigzag[i];
    __syncthreads();
}

__device__ __forceinline__ u64 prog_end(const ProgScan &sc, u32 k) { return k + 1 == sc.n_sub ? sc.nbits : (u64)(k + 1) * SYNC_BITS; }
__device__ __forceinline__ u32 prog_coef0(const ProgScan &sc) { return sc.kind == PROG_DC_FIRST ? 0u : sc.ss; }

// sync_round_kernel over first scans: blockIdx.y = scan; the guess of subsequence k is (k * SYNC_BITS, slot 0, first coefficient)
__global__ void __launch_bounds__(SYNC_THREADS) prog_round_kernel(const ProgScan *__restrict__ scans, u32 r)
{
    __shared__ EntTable sT[3];
    __shared__ uint8_t sZ[80];
    const ProgScan &sc = scans[blockIdx.y];
    if (blockIdx.x * SYNC_THREADS >= sc.n_sub) return;
    if (r >= 2 && sc.changed[r - 1] == 0) return;
    prog_tables(sc, sT, sZ, SYNC_THREADS);
    const u32 k = blockIdx.x * SYNC_THREADS + threadIdx.x;
    if (k >= sc.n_sub) return;
    u64 entry = sync_state((u64)k * SYNC_BITS, 0, prog_coef0(sc));
    if (k > 0 && r > 0) {
        const u64 e = sc.exit[(r - 1) & 1][k - 1];
        if (e != SYNC_INVALID) entry = e;
    }
    if (r > 0 && entry == sc.used[k]) { sc.exit[r & 1][k] = sc.exit[(r - 1) & 1][k]; return; }
    sc.used[k] = entry;
    u32 blocks;
    bool ok = true;
    sc.exit[r & 1][k] = prog_decode<false>(sc, sT, sZ, entry >> 16, (u32)(entry >> 8) & 255, (u32)entry & 255, prog_end(sc, k), blocks, 0, ok, nullptr);
    sc.count[k] = blocks;
    atomicAdd(&sc.changed[r], 1u);
}

// accept_kernel over first scans (one CTA per scan): ok = settled and total blocks reached before the first error
__global__ void __launch_bounds__(1024) prog_accept_kernel(const ProgScan *__restrict__ scans)
{
    __shared__ u32 s_sum[1024];
    __shared__ u32 s_err;
    const ProgScan &sc = scans[blockIdx.x];
    bool settled = false;
    for (u32 r = 1; r < PROG_ROUNDS; r++) settled = settled || sc.changed[r] == 0;
    if (!settled) { if (threadIdx.x == 0) { *sc.ok = 0; *sc.status |= PROG_DOWN_FIRST; } return; }
    if (threadIdx.x == 0) s_err = 0xFFFFFFFFu;
    // (EOB runs let counts grow past any bound: sums saturate at total, an associative operation, so every base below the
    // total is exact and the others say "at or past the total")
    const u32 n = sc.n_sub, per = (n + 1023) / 1024, total = sc.total;
    const u32 k0 = min(n, threadIdx.x * per), k1 = min(n, k0 + per);
    u32 sum = 0;
    for (u32 k = k0; k < k1; k++) sum = min(total, sum + min(total, sc.count[k]));
    s_sum[threadIdx.x] = sum;
    __syncthreads();
    for (u32 d = 1; d < 1024; d <<= 1) {
        const u32 v = threadIdx.x >= d ? s_sum[threadIdx.x - d] : 0u;
        __syncthreads();
        s_sum[threadIdx.x] = min(total, s_sum[threadIdx.x] + v);
        __syncthreads();
    }
    u32 base = threadIdx.x ? s_sum[threadIdx.x - 1] : 0u;
    for (u32 k = k0; k < k1; k++) {
        const u32 c = min(total, sc.count[k]);
        sc.count[k] = base;
        if (sc.exit[0][k] == SYNC_INVALID) atomicMin(&s_err, k);
        base = min(total, base + c);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const u64 reached = s_err != 0xFFFFFFFFu ? (s_err + 1 < n ? (u64)sc.count[s_err + 1] : (u64)s_sum[1023]) : (u64)s_sum[1023];
        const bool ok = reached >= sc.total;
        *sc.ok = ok ? 1 : 0;
        if (!ok) *sc.status |= PROG_DOWN_FIRST;
    }
}

// write_kernel over first scans; the thread that reaches the last block checks the file's first scan for the marker rule
__global__ void __launch_bounds__(SYNC_THREADS) prog_write_kernel(const ProgScan *__restrict__ scans)
{
    __shared__ EntTable sT[3];
    __shared__ uint8_t sZ[80];
    __shared__ uint8_t s_ok;
    const ProgScan &sc = scans[blockIdx.y];
    if (blockIdx.x * SYNC_THREADS >= sc.n_sub) return;
    if (threadIdx.x == 0) s_ok = *sc.ok;
    prog_tables(sc, sT, sZ, SYNC_THREADS);
    if (s_ok == 0) return;
    const u32 k = blockIdx.x * SYNC_THREADS + threadIdx.x;
    if (k >= sc.n_sub) return;
    const u32 g0 = sc.count[k];
    if (g0 >= sc.total) return;
    const u64 entry = k == 0 ? sync_state(0, 0, prog_coef0(sc)) : sc.exit[0][k - 1];
    if (entry == SYNC_INVALID) return;   // (not reached: subsequences behind an error start at or past block total)
    u32 blocks;
    bool ok = true;
    u64 last = ~0ull;
    prog_decode<true>(sc, sT, sZ, entry >> 16, (u32)(entry >> 8) & 255, (u32)entry & 255, prog_end(sc, k), blocks, g0, ok, &last);
    if (!ok) *sc.status |= PROG_DOWN_ADDRESS;
    if (sc.marker_check && last != ~0ull) {
        // decode_progressive wants the marker behind the first scan met by its bit reader (has_marker): the reader fetches 32
        // bits when <= 32 are buffered, before every symbol, so at the last symbol (start c) it has fetched 32 bits (c = 0) or
        // the least multiple of 32 >= c + 33 -- and it met the marker when that is more than the scan holds
        const u64 fetched = last == 0 ? 32 : (last + 33 + 31) / 32 * 32;
        if (fetched <= sc.nbits) *sc.status |= PROG_DOWN_MARKER;
    }
}

// dc_kernel over DC first scans: the predictor of each scan component, a wrapping 32-bit prefix sum in block order, stored
// as decode_prog_dc_first stores it, (int16)((uint16)pred << al)
__global__ void __launch_bounds__(1024) prog_dc_kernel(const ProgScan *__restrict__ scans)
{
    __shared__ u32 s_sum[3][1024];
    const ProgScan &sc = scans[blockIdx.x];
    if (sc.kind != PROG_DC_FIRST || *sc.ok == 0) return;
    const u32 bpm = sc.nslot, mcus = sc.total / bpm, per = (mcus + 1023) / 1024;
    const u32 m0 = min(mcus, threadIdx.x * per), m1 = min(mcus, m0 + per);
    u32 sum[3] = {0, 0, 0};
    for (u32 m = m0; m < m1; m++)
        for (u32 s = 0; s < bpm; s++) {
            const u32 c = sc.slot_t[s], d = (u32)(int)sc.dc[m * bpm + s];
            sum[0] += c == 0 ? d : 0u; sum[1] += c == 1 ? d : 0u; sum[2] += c == 2 ? d : 0u;
        }
    for (int c = 0; c < 3; c++) s_sum[c][threadIdx.x] = sum[c];
    __syncthreads();
    for (u32 d = 1; d < 1024; d <<= 1) {
        u32 v[3];
        for (int c = 0; c < 3; c++) v[c] = threadIdx.x >= d ? s_sum[c][threadIdx.x - d] : 0u;
        __syncthreads();
        for (int c = 0; c < 3; c++) s_sum[c][threadIdx.x] += v[c];
        __syncthreads();
    }
    u32 pred[3];
    for (int c = 0; c < 3; c++) pred[c] = s_sum[c][threadIdx.x] - sum[c];
    for (u32 m = m0; m < m1; m++)
        for (u32 s = 0; s < bpm; s++) {
            const u32 c = sc.slot_t[s];
            u32 p = (c == 0 ? pred[0] : (c == 1 ? pred[1] : pred[2])) + (u32)(int)sc.dc[m * bpm + s];
            if (c == 0) pred[0] = p; else if (c == 1) pred[1] = p; else pred[2] = p;
            int16_t *blk = prog_block(sc, m * bpm + s);   // (checked by the write kernel: every block below the total was visited)
            if (blk) blk[0] = (int16_t)(p << sc.al);
        }
}

// DC refinement (decode_prog_dc_refine): bit g of the scan belongs to block g; blockIdx.y = scan of the launch's ordinal, so
// no two threads of a launch touch one coefficient
__global__ void __launch_bounds__(256) prog_dc_refine_kernel(const ProgScan *__restrict__ scans)
{
    const ProgScan &sc = scans[blockIdx.y];
    const u32 g = blockIdx.x * 256 + threadIdx.x;
    if (g == 0 && sc.nbits < sc.total) *sc.status |= PROG_DOWN_DC_REFINE;
    if (g >= sc.total || (u64)g >= sc.nbits) return;
    if (((__ldg(sc.bits + (g >> 5)) >> ((g & 24) + (7 - (g & 7)))) & 1u) == 0) return;   // (bytes in file order, MSB first)
    int16_t *blk = prog_block(sc, g);
    if (!blk) { *sc.status |= PROG_DOWN_ADDRESS; return; }
    blk[0] = (int16_t)((uint16_t)blk[0] + (uint16_t)(1u << sc.al));
}

// Per block of an AC refinement chain's component: bit k set when the coefficient at zig-zag position k is non-zero
__global__ void __launch_bounds__(256) prog_mask_kernel(const ProgScan *__restrict__ scans, const ProgChain *__restrict__ chains)
{
    __shared__ uint8_t sZ[64];
    const ProgScan &sc = scans[chains[blockIdx.y].first];
    const u32 z = sc.slot_z[0], n = sc.plane_len[z] / 64;
    if (threadIdx.x < 64) sZ[threadIdx.x] = c_unzigzag[threadIdx.x];
    __syncthreads();
    const u32 b = blockIdx.x * 256 + threadIdx.x;
    if (b >= n) return;
    const int16_t *blk = sc.plane[z] + (u64)b * 64;
    u64 m = 0;
    for (u32 k = 0; k < 64; k++) m |= (u64)(blk[sZ[k]] != 0) << k;
    sc.mask[b] = m;
}

// the correction bits of the non-zero coefficients in `nz` (zig-zag bit mask), one bit each in zig-zag order: the mask of those
// whose bit is 1
__device__ __forceinline__ u64 prog_corrections(SyncBits &b, u64 nz)
{
    u64 out = 0;
    while (nz) {
        const u32 c = min((u32)__popcll(nz), 32u);
        b.refill();
        const u32 v = (u32)b.get(c);
        for (u32 q = 0; q < c; q++) {
            const u32 k = (u32)__ffsll((long long)nz) - 1;
            nz &= nz - 1;
            if ((v >> (c - 1 - q)) & 1u) out |= 1ull << k;
        }
    }
    return out;
}

__device__ __forceinline__ u64 prog_from(u32 k) { return k >= 64 ? 0ull : ~0ull << k; }

// One AC refinement scan: decode_mcu_ac_refine with the host's eob_run bookkeeping.  Its symbols and bit counts depend only on
// the bits and on which coefficients are non-zero, so the walk reads the masks and records per block what the host stage would
// change; prog_apply_kernel changes it.  (A coefficient the scan places is never visited again by the same scan, so corrections
// only touch coefficients that were non-zero before it.)  All 32 lanes run the walk in step; blocks that start inside an EOB
// run read one correction bit per non-zero coefficient of the band and nothing else, so the warp takes 32 of them at a time:
// a prefix sum of their bit counts gives each lane where its bits start.  Lane 0 stores what the serial part records.
// False when the image must be turned down: a code no table holds, a symbol with s != 1, a zero run past the band end, a read
// beyond the data or a failed addressing check.  (A lane reads at most 12 bytes past the data: inside the image's buffer.)
__device__ bool prog_refine_scan(const ProgScan &scan, const EntTable &T)
{
    const u32 lane = threadIdx.x & 31;
    const u32 z = scan.slot_z[0], ss = scan.ss, se = scan.se, mw = scan.mw, total = scan.total, bw = scan.bw[z];
    const u64 plane_len = scan.plane_len[z], nbits = scan.nbits;
    uint64_t *const mask = scan.mask, *const rec = scan.rec;
    const uint32_t *const words = scan.bits;
    const u64 band = prog_from(ss) & (~0ull >> (63 - se));
    SyncBits b;
    b.init(words, 0);
    u32 eob = 0;
    for (u32 g = 0; g < total;) {
        if (eob > 0) {   // ---- up to 32 blocks inside the run, one per lane
            const u32 n = min(min(eob, 32u), total - g), gl = g + lane;
            const u32 i = gl / mw, j = gl - (gl / mw) * mw;
            const u64 at = 64ull * ((u64)i * bw + j);
            const bool mine = lane < n;
            if (__any_sync(~0u, mine && at + 64 > plane_len)) return false;
            const u64 m = mine ? mask[at >> 6] : 0ull;
            const u64 nz = (m >> 1) ? m & band : 0ull;
            const u32 c = (u32)__popcll(nz);
            u32 incl = c;
            for (u32 d = 1; d < 32; d <<= 1) { const u32 v = __shfl_up_sync(~0u, incl, d); if (lane >= d) incl += v; }
            const u32 sum = __shfl_sync(~0u, incl, 31);
            const u64 p0 = b.pos + incl - c;
            if (b.pos + sum > nbits) return false;
            if (mine) {
                u64 corr = 0;
                if (c) {
                    const u32 w = (u32)(p0 >> 5), off = (u32)(p0 & 31);
                    const u64 hi = ((u64)b.word(w) << 32) | b.word(w + 1);
                    const u64 win = off ? (hi << off) | (b.word(w + 2) >> (32 - off)) : hi;   // the 64 bits from p0
                    u64 left = nz;
                    for (u32 q = 0; left; q++, left &= left - 1)
                        if ((win >> (63 - q)) & 1) corr |= left & (~left + 1);
                }
                uint64_t *r = rec + 3 * (at >> 6);
                r[0] = corr; r[1] = 0; r[2] = 0;
            }
            b.init(words, b.pos + sum);
            eob -= n;
            g += n;
            continue;
        }
        // ---- a block that starts with a symbol (the same on every lane)
        const u32 i = g / mw, j = g - i * mw;
        const u64 at = 64ull * ((u64)i * bw + j);
        if (at + 64 > plane_len) return false;
        u64 m = mask[at >> 6];
        const u64 m0 = m;
        u64 corr = 0, placed = 0, neg = 0;
        u32 k = ss;
        for (;;) {
            b.refill();
            int s = sync_huff(b, T, T.lookup[b.peek(9)]);
            if (s < 0) return false;
            const u32 rr = (u32)s >> 4;
            s &= 15;
            if (s == 0 && rr != 15) {
                eob = (1u << rr) + (rr ? (u32)b.get(rr) : 0u);
                break;
            }
            bool minus = false;
            if (s != 0) {
                if (s != 1) return false;
                minus = b.get(1) == 0;
            }
            // the (rr + 1)-th zero coefficient at or after k: the corrections of the non-zero ones before it come first
            u64 zeros = ~m & band & prog_from(k);
            if ((u32)__popcll(zeros) <= rr) return false;
            for (u32 q = 0; q < rr; q++) zeros &= zeros - 1;
            const u32 pz = (u32)__ffsll((long long)zeros) - 1;
            corr |= prog_corrections(b, m & prog_from(k) & ((1ull << pz) - 1));
            if (b.pos > nbits) return false;
            if (s != 0) { placed |= 1ull << pz; neg |= (u64)minus << pz; m |= 1ull << pz; }
            k = pz + 1;
            if (k > se) break;
        }
        if (b.pos > nbits) return false;
        if (eob > 0) {
            if (m >> 1) corr |= prog_corrections(b, m & band & prog_from(k));
            if (b.pos > nbits) return false;
            eob--;
        }
        if (lane == 0) {
            uint64_t *r = rec + 3 * (at >> 6);
            r[0] = corr; r[1] = placed; r[2] = neg;
            if (m != m0) mask[at >> 6] = m;
        }
        __syncwarp();
        g++;
    }
    return true;
}

// One warp per (image, component): its AC refinement scans in file order
__global__ void __launch_bounds__(32) prog_refine_kernel(const ProgScan *__restrict__ scans, const ProgChain *__restrict__ chains)
{
    __shared__ EntTable sT;
    __shared__ uint8_t sZ[80];
    const ProgChain ch = chains[blockIdx.x];
    for (u32 q = 0; q < ch.count; q++) {
        const ProgScan &sc = scans[ch.first + q];
        __syncthreads();
        prog_tables(sc, &sT, sZ, 32);
        if (!prog_refine_scan(sc, sT)) {
            if (threadIdx.x == 0) *sc.status |= PROG_DOWN_AC_REFINE;
            return;
        }
    }
}

// The records of a chain's scans applied to its planes in scan order, one thread per block: a correction adds 2^al away from
// zero when that bit is clear (decode_mcu_ac_refine), a placed coefficient becomes +-2^al
__global__ void __launch_bounds__(256) prog_apply_kernel(const ProgScan *__restrict__ scans, const ProgChain *__restrict__ chains)
{
    __shared__ uint8_t sZ[64];
    const ProgChain ch = chains[blockIdx.y];
    const ProgScan &s0 = scans[ch.first];
    const u32 z = s0.slot_z[0], n = s0.plane_len[z] / 64;
    if (threadIdx.x < 64) sZ[threadIdx.x] = c_unzigzag[threadIdx.x];
    __syncthreads();
    const u32 bl = blockIdx.x * 256 + threadIdx.x;
    if (bl >= n || *s0.status != 0) return;
    const u32 y = bl / s0.bw[z], x = bl - y * s0.bw[z];
    int16_t *blk = s0.plane[z] + (u64)bl * 64;
    for (u32 q = 0; q < ch.count; q++) {
        const ProgScan &sc = scans[ch.first + q];
        if (x >= sc.mw || (u64)y * sc.mw + x >= sc.total) continue;   // not a block of the scan
        const uint64_t *r = sc.rec + 3 * (u64)bl;
        const int p1 = 1 << sc.al;
        for (u64 c = r[0]; c; c &= c - 1) {
            int16_t &v = blk[sZ[__ffsll((long long)c) - 1] & 63];
            if ((v & p1) == 0) v = (int16_t)(v >= 0 ? v + p1 : v - p1);
        }
        const u64 neg = r[2];
        for (u64 c = r[1]; c; c &= c - 1) {
            const u32 k = (u32)__ffsll((long long)c) - 1;
            blk[sZ[k] & 63] = (int16_t)((neg >> k) & 1 ? -p1 : p1);
        }
    }
}

int launch_prog_phase(const ProgScan *d_scans, uint32_t n_first, uint32_t max_sub, const uint32_t *dc_ref, uint32_t n_dc_ord,
                      uint32_t max_dc_blocks, const ProgChain *d_chains, uint32_t n_chain, uint32_t max_blocks, void *stream, int phase)
{
    cudaStream_t s = (cudaStream_t)stream;
    const dim3 grid((max_sub + SYNC_THREADS - 1) / SYNC_THREADS, n_first);
    if (phase <= PROG_PHASE_DC && (n_first == 0 || max_sub == 0)) return 0;
    if (phase == PROG_PHASE_ROUNDS)
        for (u32 r = 0; r < PROG_ROUNDS; r++) prog_round_kernel<<<grid, SYNC_THREADS, 0, s>>>(d_scans, r);
    else if (phase == PROG_PHASE_ACCEPT) prog_accept_kernel<<<n_first, 1024, 0, s>>>(d_scans);
    else if (phase == PROG_PHASE_WRITE) prog_write_kernel<<<grid, SYNC_THREADS, 0, s>>>(d_scans);
    else if (phase == PROG_PHASE_DC) prog_dc_kernel<<<n_first, 1024, 0, s>>>(d_scans);
    else if (phase == PROG_PHASE_DC_REFINE) {
        for (u32 r = 0; r < n_dc_ord && max_dc_blocks; r++)
            prog_dc_refine_kernel<<<dim3((max_dc_blocks + 255) / 256, dc_ref[r + 1] - dc_ref[r]), 256, 0, s>>>(d_scans + dc_ref[r]);
    } else if (phase == PROG_PHASE_MASK) {
        if (n_chain && max_blocks) prog_mask_kernel<<<dim3((max_blocks + 255) / 256, n_chain), 256, 0, s>>>(d_scans, d_chains);
    } else if (phase == PROG_PHASE_AC_REFINE) {
        if (n_chain) prog_refine_kernel<<<n_chain, 32, 0, s>>>(d_scans, d_chains);
    } else if (n_chain && max_blocks) prog_apply_kernel<<<dim3((max_blocks + 255) / 256, n_chain), 256, 0, s>>>(d_scans, d_chains);
    return (int)cudaGetLastError();
}

}  // namespace zj
