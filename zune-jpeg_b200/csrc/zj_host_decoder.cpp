// zj_host_decoder.cpp -- the HOST stage in front of the GPU path: JPEG headers and Huffman entropy decode
// into whole-image i16 coefficient planes, plus the `Decoder` object of the reference's public API.
//
// In a Rust deployment this stage is the reference's own code (src/headers.rs, src/marker.rs, src/huffman.rs,
// src/bitstream.rs, src/mcu.rs, src/mcu_prog.rs) and only the GPU entry points are bound (INTEGRATION.md).
// There is no Rust toolchain in this build environment, so the stage is restated here in C++ with the same
// observable behaviour: same marker loop, same table construction, same bit-reader state machine (including
// what happens after a marker is met inside a scan), same restart bookkeeping (SURVEY Q8), same errors.
// The branchy bit-serial work stays on the CPU by design; everything after it runs in zj_kernels.cu.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <functional>
#include <new>
#include <string>
#include <thread>
#include <atomic>
#include <mutex>
#include <vector>

#include "../../include/zune_jpeg_b200.h"
#include "zj_device.h"
#include "zj_entropy.h"

// Worker threads pull their work from a shared counter, so a pool that could not be grown (std::system_error: thread limit)
// just runs with fewer threads -- the calling thread always works too.  Nothing may unwind through the C ABI.
template <typename Pool, typename Fn>
static bool spawn(Pool &pool, Fn &fn)
{
    try { pool.emplace_back(std::ref(fn)); return true; }
    catch (...) { return false; }
}

namespace {

// ------------------------------------------------------------------------------------------------ errors
struct DecodeError {  // DecodeErrors, reference src/errors.rs:16-43
    int kind;
    std::string msg;
};
#define FAIL(k, m) throw DecodeError{(k), (m)}

static std::string fmt(const char *f, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, f);
    vsnprintf(buf, sizeof(buf), f, ap);
    va_end(ap);
    return std::string(buf);
}
static const char *IO_EOF = "Error decoding an image:\n failed to fill whole buffer";  // From<io::Error>, errors.rs:120-126

// ------------------------------------------------------------------------------------------------ markers
enum MarkerKind { M_SOF, M_DHT, M_DAC, M_RST, M_SOI, M_EOI, M_SOS, M_DQT, M_DNL, M_DRI, M_APP, M_COM };
struct Marker { int kind; int n; bool operator==(const Marker &o) const { return kind == o.kind && n == o.n; } };

static bool marker_from_u8(uint8_t b, Marker *m)  // Marker::from_u8, src/marker.rs:48-78
{
    switch (b) {
    case 0xFE: *m = {M_COM, 0}; return true;
    case 0xC0: *m = {M_SOF, 0}; return true;
    case 0xC2: *m = {M_SOF, 2}; return true;
    case 0xC4: *m = {M_DHT, 0}; return true;
    case 0xCC: *m = {M_DAC, 0}; return true;
    case 0xD8: *m = {M_SOI, 0}; return true;
    case 0xD9: *m = {M_EOI, 0}; return true;
    case 0xDA: *m = {M_SOS, 0}; return true;
    case 0xDB: *m = {M_DQT, 0}; return true;
    case 0xDC: *m = {M_DNL, 0}; return true;
    case 0xDD: *m = {M_DRI, 0}; return true;
    case 0xE0: *m = {M_APP, 0}; return true;
    case 0xE1: *m = {M_APP, 1}; return true;
    case 0xEE: *m = {M_APP, 14}; return true;
    default:
        if (b >= 0xD0 && b <= 0xD7) { *m = {M_RST, b - 0xD0}; return true; }
        return false;
    }
}
static std::string marker_debug(const Marker &m)  // #[derive(Debug)]
{
    switch (m.kind) {
    case M_SOF: return fmt("SOF(%d)", m.n);
    case M_DHT: return "DHT";
    case M_DAC: return "DAC";
    case M_RST: return fmt("RST(%d)", m.n);
    case M_SOI: return "SOI";
    case M_EOI: return "EOI";
    case M_SOS: return "SOS";
    case M_DQT: return "DQT";
    case M_DNL: return "DNL";
    case M_DRI: return "DRI";
    case M_APP: return fmt("APP(%d)", m.n);
    default: return "COM";
    }
}

static const uint8_t UN_ZIGZAG[80] = {  // src/misc.rs:30-41 (16 entries of padding)
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63,
    63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63};

// ------------------------------------------------------------------------------------------------ cursor
struct Cursor {  // std::io::Cursor<Vec<u8>> as the reference uses it
    const uint8_t *data;
    size_t len;
    size_t pos;
    uint8_t read_byte()  // misc::read_byte, src/misc.rs:268-278
    {
        if (pos >= len) FAIL(ZJ_DE_FORMAT, IO_EOF);
        return data[pos++];
    }
    uint16_t read_u16_be()  // misc::read_u16_be, src/misc.rs:281-296: a short read is ExhaustedData
    {
        size_t avail = pos < len ? len - pos : 0;
        if (avail < 2) { pos += avail; FAIL(ZJ_DE_EXHAUSTED_DATA, ""); }
        uint16_t v = (uint16_t)((data[pos] << 8) | data[pos + 1]);
        pos += 2;
        return v;
    }
    void read_exact(uint8_t *dst, size_t n, int kind, const std::string &msg)
    {
        size_t avail = pos < len ? len - pos : 0;
        if (avail < n) { pos = len; FAIL(kind, msg); }
        memcpy(dst, data + pos, n);
        pos += n;
    }
    void consume(size_t n) { pos += n; }
    uint64_t read_u8_or_zero()  // bitstream.rs:696-703
    {
        uint64_t v = pos < len ? data[pos] : 0;
        pos++;
        return v;
    }
};

// ------------------------------------------------------------------------------------------------ Huffman
constexpr int HUFF_LOOKAHEAD = 9;  // src/huffman.rs:9

// Host-stage quirks of the reference (DESIGN.md section 2), reproduced by default.  zj_host_set_quirks() clears bits for
// TESTS ONLY: with a bit cleared the corresponding lines behave the way libjpeg does, which is how tests/test_quirks.py
// shows that each deviation from libjpeg on the reference's own fixtures comes from exactly the cited lines.  Every decode takes
// its mask from here when it starts (zj_decoder::quirks); a spec-output decode (ZJ_USE_SPEC_OUTPUT or ZJ_USE_LIBJPEG_OUTPUT)
// runs with none of them.
static std::atomic<uint32_t> g_quirks{ZJ_QUIRK_ALL};

struct HuffmanTable {  // src/huffman.rs:14-41
    int32_t maxcode[18];
    int32_t offset[18];
    int32_t lookup[1 << HUFF_LOOKAHEAD];
    int16_t ac_lookup[1 << HUFF_LOOKAHEAD];
    bool has_ac_lookup;
    uint8_t bits[17];
    uint8_t values[256];
    bool present;
};

// HuffmanTable::new + make_derived_table, src/huffman.rs:45-276
static void build_huffman(HuffmanTable &p, const uint8_t codes[17], const uint8_t values[256], bool is_dc, bool is_progressive, bool q9)
{
    const int32_t too_long = (HUFF_LOOKAHEAD + 1) << HUFF_LOOKAHEAD;
    memset(p.maxcode, 0, sizeof(p.maxcode));
    memset(p.offset, 0, sizeof(p.offset));
    for (int i = 0; i < (1 << HUFF_LOOKAHEAD); i++) p.lookup[i] = too_long;
    memcpy(p.bits, codes, 17);
    memcpy(p.values, values, 256);
    p.has_ac_lookup = false;
    p.present = true;

    uint8_t huff_size[257] = {0};
    uint32_t huff_code[257] = {0};
    size_t k = 0;
    for (int l = 1; l <= 16; l++)
        for (int i = p.bits[l]; i != 0; i--) huff_size[k++] = (uint8_t)l;  // figure C.1
    huff_size[k] = 0;
    const size_t num_symbols = k;
    uint32_t code = 0;
    int32_t si = huff_size[0];
    k = 0;
    while (huff_size[k] != 0) {  // figure C.2
        while ((int32_t)huff_size[k] == si) { huff_code[k] = code; code++; k++; }
        p.maxcode[si] = (int32_t)(code << (16 - si));
        if ((int32_t)code >= (1 << si)) FAIL(ZJ_DE_HUFFMAN_DECODE, "Bad Huffman Table");
        code <<= 1;
        si++;
    }
    k = 0;
    for (int l = 0; l <= 16; l++) {  // figure F.15
        if (p.bits[l] == 0) p.maxcode[l] = -1;
        else { p.offset[l] = (int32_t)k - (int32_t)huff_code[k]; k += p.bits[l]; }
    }
    p.offset[17] = 0;
    p.maxcode[17] = 0x000FFFFF;
    k = 0;
    for (int l = 1; l <= HUFF_LOOKAHEAD; l++) {
        for (int i = 1; i <= (int)p.bits[l]; i++) {
            size_t look_bits = (size_t)huff_code[k] << (HUFF_LOOKAHEAD - l);
            for (int c = 0; c < (1 << (HUFF_LOOKAHEAD - l)); c++) { p.lookup[look_bits] = (l << HUFF_LOOKAHEAD) | p.values[k]; look_bits++; }
            k++;
        }
    }
    if (!is_dc) {  // fast AC table: decode + receive_extend in one lookup (huffman.rs:180-257)
        int16_t fast[1 << HUFF_LOOKAHEAD];
        for (int i = 0; i < (1 << HUFF_LOOKAHEAD); i++) fast[i] = 255;
        for (size_t i = 0; i < num_symbols; i++) {
            const int s = huff_size[i];
            if (s <= HUFF_LOOKAHEAD) {
                const size_t c = (size_t)(huff_code[i] << (HUFF_LOOKAHEAD - s)), m = (size_t)1 << (HUFF_LOOKAHEAD - s);
                for (size_t j = 0; j < m; j++) fast[c + j] = (int16_t)i;
            }
        }
        for (int i = 0; i < (1 << HUFF_LOOKAHEAD); i++) {
            p.ac_lookup[i] = 0;
            const int16_t fast_v = fast[i];
            if (fast_v < 255) {
                const uint8_t rs = p.values[fast_v];
                const int16_t run = (rs >> 4) & 15, mag_bits = rs & 15, len = huff_size[fast_v];
                if (mag_bits == 0 && !is_progressive) {
                    const int16_t new_run = run == 0 ? 63 : run;
                    p.ac_lookup[i] = (int16_t)((new_run << 4) + len);
                } else if (mag_bits != 0 && (len + mag_bits) <= HUFF_LOOKAHEAD) {
                    int16_t kk = (int16_t)((((int16_t)i << len) & ((1 << HUFF_LOOKAHEAD) - 1)) >> (HUFF_LOOKAHEAD - mag_bits));
                    const int16_t m = (int16_t)(1 << (mag_bits - 1));
                    if (kk < m) kk = (int16_t)(kk + (int16_t)((int16_t)(~0u << mag_bits) + 1));
                    // Q9 (huffman.rs:249-252): the entry is an i16, so `k << 10` keeps only 6 bits of k: |k| >= 32 decodes wrong.
                    // Quirk off: such values stay out of the fast table and take the general path below it.
                    const int16_t lim = q9 ? 128 : 32;
                    if (kk >= -lim && kk <= lim - 1) p.ac_lookup[i] = (int16_t)((kk << 10) + (run << 4) + (len + mag_bits));
                }
            }
        }
        p.has_ac_lookup = true;
    }
    if (is_dc)
        for (size_t i = 0; i < num_symbols; i++)
            if (p.values[i] > 15) FAIL(ZJ_DE_HUFFMAN_DECODE, "Bad Huffman Table");
}

// ------------------------------------------------------------------------------------------------ bit reader
struct BitStream {  // src/bitstream.rs:94-114
    uint64_t buffer = 0, aligned_buffer = 0;
    uint8_t bits_left = 0;
    bool has_marker = false;
    Marker marker{};
    uint8_t successive_high = 0, successive_low = 0, spec_start = 0, spec_end = 0;
    int32_t eob_run = 0;
    bool q10 = true;   // Q10: decode_dc refills only below 16 buffered bits (bitstream.rs:278-281); set from zj_decoder::quirks

    static bool has_byte_ff(uint32_t b)  // has_byte(b, 255), bitstream.rs:705-717
    {
        const uint32_t v = b ^ 0xFFFFFFFFu;
        return (~((((v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | v) | 0x7F7F7F7Fu)) != 0;
    }
    // bitstream.rs:159-261
    // (the test that decides whether anything happens is kept inline in front of the out-of-line body: it is evaluated once
    // per Huffman symbol and is false for most of them)
    inline __attribute__((always_inline)) void refill(Cursor &r)
    {
        if (__builtin_expect(bits_left > 32 && !has_marker, 1)) return;
        refill_body(r);
    }
    __attribute__((noinline)) void refill_body(Cursor &r)
    {
        if (bits_left <= 32 && !has_marker) {
            const size_t position = r.pos;
            if (position + 4 < r.len) {
                const uint32_t msb = ((uint32_t)r.data[position] << 24) | ((uint32_t)r.data[position + 1] << 16) |
                                     ((uint32_t)r.data[position + 2] << 8) | r.data[position + 3];
                if (!has_byte_ff(msb)) {
                    r.pos = position + 4;
                    bits_left += 32;
                    buffer <<= 32;
                    buffer |= msb;
                    aligned_buffer = buffer << (64 - bits_left);
                    return;
                }
            }
            for (int k = 0; k < 4; k++) {
                const uint64_t byte = r.read_u8_or_zero();
                buffer = (buffer << 8) | byte;
                bits_left += 8;
                if (byte == 0xff) {
                    uint64_t next = r.read_u8_or_zero();
                    if (next != 0x00) {
                        while (next == 0xFF) next = r.read_u8_or_zero();
                        if (next != 0x00) {
                            buffer >>= 8;
                            bits_left -= 8;
                            if (bits_left != 0) aligned_buffer = buffer << (64 - bits_left);
                            Marker m;
                            if (!marker_from_u8((uint8_t)next, &m)) FAIL(ZJ_DE_FORMAT, fmt("Unknown marker 0xFF%llX", (unsigned long long)next));
                            marker = m;
                            has_marker = true;
                            return;
                        }
                    }
                }
            }
            aligned_buffer = buffer << (64 - bits_left);
        } else if (has_marker) {
            bits_left = 63;  // fake zero bits after a marker, bitstream.rs:254-258
        }
    }
    template <int N> int32_t peek_bits() const { return (int32_t)(aligned_buffer >> (64 - N)); }
    void drop_bits(uint8_t n)
    {
        bits_left = bits_left > n ? bits_left - n : 0;
        aligned_buffer = n >= 64 ? 0 : aligned_buffer << n;
    }
    int32_t get_bits(uint8_t n)  // bitstream.rs:394-402 (a rotate, not a shift)
    {
        const uint64_t mask = (1ull << n) - 1;
        const unsigned r = n & 63;
        aligned_buffer = r ? (aligned_buffer << r) | (aligned_buffer >> (64 - r)) : aligned_buffer;
        const int32_t bits = (int32_t)(aligned_buffer & mask);
        bits_left = bits_left > n ? bits_left - n : 0;
        return bits;
    }
    uint8_t get_bit() { const uint8_t k = (uint8_t)(aligned_buffer >> 63); drop_bits(1); return k; }
    static int32_t huff_extend(int32_t x, int32_t s)  // bitstream.rs:685-689
    {
        return x + (((x - (1 << (s - 1))) >> 31) & (int32_t)(((uint32_t)-1 << s) + 1));
    }
    // decode_huff! macro, bitstream.rs:49-90
    void decode_huff(int32_t &symbol, const HuffmanTable &t)
    {
        int32_t code_length = symbol >> HUFF_LOOKAHEAD;
        symbol &= (1 << HUFF_LOOKAHEAD) - 1;
        if (code_length > HUFF_LOOKAHEAD) {
            symbol = peek_bits<16>();
            while (code_length < 17) {
                if (symbol < t.maxcode[code_length]) break;
                code_length++;
            }
            if (code_length == 17) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("Bad Huffman Code 0x%X, corrupt JPEG", (unsigned)symbol));
            symbol >>= (16 - code_length);
            symbol = t.values[(symbol + t.offset[code_length]) & 0xFF];
        }
        drop_bits((uint8_t)code_length);
    }
    void decode_dc(Cursor &r, const HuffmanTable &dc, int32_t &pred)  // bitstream.rs:272-297
    {
        // Q10: a DC code (<= 16 bits) plus its magnitude bits (<= 11) can need 27 bits, but the refill happens only below 16:
        // the reader under-runs and mis-syncs.  Quirk off: refill like the AC loop does (whenever <= 32 bits are buffered).
        if (bits_left < 16 || !q10) refill(r);
        int32_t symbol = dc.lookup[peek_bits<HUFF_LOOKAHEAD>()];
        decode_huff(symbol, dc);
        if (symbol != 0) { const int32_t rr = get_bits((uint8_t)symbol); symbol = huff_extend(rr, symbol); }
        pred = (int32_t)((uint32_t)pred + (uint32_t)symbol);
    }
    // bitstream.rs:314-373
    void decode_mcu_block(Cursor &r, const HuffmanTable &dc, const HuffmanTable &ac, int16_t *block, int32_t &pred)
    {
        size_t pos = 1;
        decode_dc(r, dc, pred);
        block[0] = (int16_t)pred;
        while (pos < 64) {
            refill(r);
            int32_t symbol = peek_bits<HUFF_LOOKAHEAD>();
            const int16_t fast_ac = ac.ac_lookup[symbol];
            symbol = ac.lookup[symbol];
            if (fast_ac != 0) {
                pos += (size_t)((fast_ac >> 4) & 63);
                block[UN_ZIGZAG[std::min<size_t>(pos, 63)] & 63] = (int16_t)(fast_ac >> 10);
                drop_bits((uint8_t)(fast_ac & 15));
                pos += 1;
            } else {
                decode_huff(symbol, ac);
                int32_t rr = symbol >> 4;
                symbol &= 15;
                if (symbol != 0) {
                    pos += (size_t)rr;
                    rr = get_bits((uint8_t)symbol);
                    symbol = huff_extend(rr, symbol);
                    block[UN_ZIGZAG[pos & 63] & 63] = (int16_t)symbol;
                    pos += 1;
                } else if (rr != 15) {
                    return;
                } else {
                    pos += 16;
                }
            }
        }
    }
    void decode_prog_dc_first(Cursor &r, const HuffmanTable &dc, int16_t *block, int32_t &pred)  // bitstream.rs:407-415
    {
        decode_dc(r, dc, pred);
        *block = (int16_t)((uint16_t)(int16_t)pred * (uint16_t)(1u << successive_low));
    }
    void decode_prog_dc_refine(Cursor &r, int16_t *block)  // bitstream.rs:417-433
    {
        if (bits_left < 1) refill(r);
        if (get_bit() == 1) *block = (int16_t)((uint16_t)*block + (uint16_t)(1u << successive_low));
    }
    // bitstream.rs:443-506
    void decode_mcu_ac_first(Cursor &r, const HuffmanTable &ac, int16_t *block)
    {
        const int shift = successive_low;
        size_t k = spec_start;
        for (;;) {
            refill(r);
            int32_t symbol = peek_bits<HUFF_LOOKAHEAD>();
            const int16_t fac = ac.ac_lookup[symbol];
            symbol = ac.lookup[symbol];
            if (fac != 0) {
                k += (size_t)((fac >> 4) & 63);
                block[UN_ZIGZAG[std::min<size_t>(k, 63)] & 63] = (int16_t)((uint16_t)(int16_t)(fac >> 10) * (uint16_t)(1u << shift));
                drop_bits((uint8_t)(fac & 15));
                k += 1;
            } else {
                decode_huff(symbol, ac);
                int32_t rr = symbol >> 4;
                symbol &= 15;
                if (symbol != 0) {
                    k += (size_t)rr;
                    rr = get_bits((uint8_t)symbol);
                    symbol = huff_extend(rr, symbol);
                    block[UN_ZIGZAG[k & 63] & 63] = (int16_t)((uint16_t)(int16_t)symbol * (uint16_t)(1u << shift));
                    k += 1;
                } else {
                    if (rr != 15) {
                        eob_run = 1 << rr;
                        eob_run += get_bits((uint8_t)rr);
                        eob_run -= 1;
                        break;
                    }
                    k += 16;
                }
            }
            if (k > spec_end) break;
        }
    }
    // bitstream.rs:507-658
    void decode_mcu_ac_refine(Cursor &r, const HuffmanTable &table, int16_t *block)
    {
        const int16_t bit = (int16_t)(1 << successive_low);
        uint8_t k = spec_start;
        if (eob_run == 0) {
            for (;;) {
                refill(r);
                int32_t symbol = table.lookup[peek_bits<HUFF_LOOKAHEAD>()];
                decode_huff(symbol, table);
                int32_t rr = symbol >> 4;
                symbol &= 15;
                if (symbol == 0) {
                    if (rr != 15) {
                        eob_run = 1 << rr;
                        eob_run += get_bits((uint8_t)rr);
                        break;
                    }
                } else {
                    if (symbol != 1) FAIL(ZJ_DE_HUFFMAN_DECODE, "Bad Huffman code, corrupt JPEG?");
                    symbol = get_bit() == 1 ? (int32_t)bit : (int32_t)-bit;
                }
                while (k <= spec_end) {
                    int16_t *coefficient = &block[UN_ZIGZAG[k & 63] & 63];
                    if (*coefficient != 0) {
                        if (get_bit() == 1 && (*coefficient & bit) == 0) {
                            if (*coefficient >= 0) *coefficient = (int16_t)(*coefficient + bit);
                            else *coefficient = (int16_t)(*coefficient - bit);
                        }
                        if (bits_left < 1) refill(r);
                    } else {
                        rr -= 1;
                        if (rr < 0) break;
                    }
                    k += 1;
                }
                if (symbol != 0) block[UN_ZIGZAG[k & 63] & 63] = (int16_t)symbol;
                k += 1;
                if (k > spec_end) break;
            }
        }
        if (eob_run > 0) {
            bool any = false;
            for (int i = 1; i < 64; i++) if (block[i] != 0) { any = true; break; }
            if (any) {
                refill(r);
                while (k <= spec_end) {
                    int16_t *coefficient = &block[UN_ZIGZAG[k & 63] & 63];
                    if (*coefficient != 0 && get_bit() == 1) {
                        if ((*coefficient & bit) == 0) {
                            if (*coefficient >= 0) *coefficient = (int16_t)(*coefficient + bit);
                            else *coefficient = (int16_t)(*coefficient - bit);
                        }
                    }
                    if (bits_left < 1) refill(r);
                    k += 1;
                }
            }
            eob_run -= 1;
        }
    }
    void update_progressive_params(uint8_t ah, uint8_t al, uint8_t ss, uint8_t se) { successive_high = ah; successive_low = al; spec_start = ss; spec_end = se; }
    void reset() { bits_left = 0; has_marker = false; buffer = 0; aligned_buffer = 0; eob_run = 0; }  // bitstream.rs:673-680
};

// ------------------------------------------------------------------------------------------------ decoder
enum ComponentID { ID_Y, ID_CB, ID_CR };
static const char *comp_debug(int id) { return id == ID_Y ? "Y" : (id == ID_CB ? "Cb" : "Cr"); }
enum SubSamp { SS_NONE, SS_H, SS_V, SS_HV };

struct Component {  // src/components.rs:18-43
    int component_id;
    size_t vertical_sample, horizontal_sample, dc_huff_table, ac_huff_table;
    uint8_t quantization_table_number;
    int32_t quantization_table[64];
    int32_t dc_pred;
    size_t width_stride;
    uint8_t id;
};

// The three coefficient planes of an image live in ONE block (pinned when a device is present), each plane on a 256-byte
// boundary: zj_gpu_reconstruct uploads planes that follow each other in host memory with a single copy (three copies of
// 16.6 + 4.1 + 4.1 MB for a 4K 4:2:0 image run at 44 GB/s over PCIe, one of 24.9 MB at 49).
struct PlaneBuf { int16_t *p = nullptr; };
struct PlaneBlock {
    int16_t *base = nullptr;
    size_t cap = 0;   // i16
    bool pinned = false;
    void release()
    {
        if (!base) return;
        if (pinned) cudaFreeHost(base); else free(base);
        base = nullptr; cap = 0;
    }
    // planes[z].p for plane_len[z] i16 each (0 = no plane); zeroed on request
    void ensure(PlaneBuf (&planes)[3], const size_t (&plane_len)[3], bool want_pinned, bool zero)
    {
        size_t off[3], total = 0;
        for (int z = 0; z < 3; z++) { off[z] = total; total += (plane_len[z] + 127) & ~(size_t)127; }
        if (total > cap) {
            release();
            const size_t want = total + total / 8 + 128;
            if (want_pinned && cudaHostAlloc((void **)&base, want * 2, cudaHostAllocPortable) == cudaSuccess) pinned = true;
            else { cudaGetLastError(); base = (int16_t *)aligned_alloc(256, (want * 2 + 255) & ~(size_t)255); pinned = false; }
            if (!base) { cap = 0; FAIL(ZJ_DE_FORMAT, "out of memory for coefficient planes"); }
            cap = want;
        }
        for (int z = 0; z < 3; z++) {
            planes[z].p = plane_len[z] ? base + off[z] : nullptr;
            if (zero && plane_len[z]) memset(planes[z].p, 0, plane_len[z] * 2);
        }
    }
};

}  // namespace

// Progress of the baseline entropy stage, strip by strip (SURVEY 8(f).2: the reference entropy-decodes strip k+1 while its
// thread pool post-processes strip k, mcu.rs:230-369 / 356-368).  `begin` is called once the planes exist and the descriptor is
// final, `progress(n)` whenever strips [0, n) of every plane are complete and will not be touched again, `restart` when the
// planes are about to be decoded again from the start (the interval-parallel form was turned down).
struct StripSink {
    virtual void begin(const zj_image &img, size_t n_strips) = 0;
    virtual void progress(size_t strips_done) = 0;
    virtual void restart() = 0;
    virtual ~StripSink() {}
};

// ------------------------------------------------------------------------------------------------ EXIF orientation
// The APP1 segments before the first SOS that carry metadata (the statement is next to ZJ_FLAG_ORIENT_SHIFT in the header).
// They point into the caller's buffer, which outlives the header parse they are read in.
struct OrientSource {
    struct Span { const uint8_t *p; size_t n; };
    std::vector<Span> exif;        // the EXIF bytes: the first Exif APP1 payload, then each later one's bytes after its header
    size_t exif_len = 0;
    Span xmp{nullptr, 0};          // the last XMP APP1 segment's bytes after its 29-byte header

    void clear() { exif.clear(); exif_len = 0; xmp = {nullptr, 0}; }   // (keeps the span list's capacity for the next file)

    // n bytes at offset `off` of the EXIF bytes; false when they are not all there
    bool read(size_t off, size_t n, uint8_t *dst) const
    {
        if (off > exif_len || n > exif_len - off) return false;
        for (size_t k = 0; k < exif.size() && n; k++) {
            if (off >= exif[k].n) { off -= exif[k].n; continue; }
            const size_t m = std::min(n, exif[k].n - off);
            memcpy(dst, exif[k].p + off, m);
            dst += m; n -= m; off = 0;
        }
        return n == 0;
    }
    // Pillow's Image.getexif() orientation, then exif_transpose's choice: 2-8, or 1 for no transform
    uint32_t orientation() const
    {
        static const uint8_t EXIF_HDR[6] = {'E', 'x', 'i', 'f', 0, 0};
        size_t base = 0;   // Exif.load strips every leading "Exif\0\0"
        for (uint8_t h[6]; read(base, 6, h) && memcmp(h, EXIF_HDR, 6) == 0;) base += 6;
        long v = -1;       // the tag's value; -1 = IFD0 has no tag 0x0112
        if (base < exif_len) {
            uint8_t hd[8];
            if (!read(base, 8, hd)) return 1;   // (Pillow raises on a short or unknown TIFF header; its orientation is then 1)
            const bool le = memcmp(hd, "II*\0", 4) == 0;
            if (!le && memcmp(hd, "MM\0*", 4) != 0) return 1;
            auto u16 = [le](const uint8_t *b) { return le ? (uint32_t)(b[0] | b[1] << 8) : (uint32_t)(b[0] << 8 | b[1]); };
            auto u32 = [le](const uint8_t *b) { return le ? (uint32_t)b[0] | (uint32_t)b[1] << 8 | (uint32_t)b[2] << 16 | (uint32_t)b[3] << 24
                                                          : (uint32_t)b[0] << 24 | (uint32_t)b[1] << 16 | (uint32_t)b[2] << 8 | (uint32_t)b[3]; };
            const size_t tiff_len = exif_len - base;
            const size_t ifd = u32(hd + 4);
            uint8_t cnt[2];
            // IFD0 as ImageFileDirectory_v2.load reads it: entries up to the first one that cannot be read whole (its bytes, or
            // the data it points at), skipping unknown types and empty values; a later entry of a tag replaces an earlier one
            if (ifd <= tiff_len && read(base + ifd, 2, cnt)) {
                static const uint8_t unit[14] = {0, 1, 1, 2, 4, 8, 1, 1, 2, 4, 8, 4, 8, 4};   // TIFF type -> bytes per value
                const uint32_t n = u16(cnt);
                for (uint32_t k = 0; k < n; k++) {
                    uint8_t e[12];
                    if (!read(base + ifd + 2 + 12 * (size_t)k, 12, e)) break;
                    const uint32_t typ = u16(e + 2), count = u32(e + 4);
                    if (typ == 0 || typ >= 14) continue;
                    const uint64_t size = (uint64_t)count * unit[typ];
                    if (size == 0) continue;
                    uint8_t val[4];
                    const uint8_t *vp = e + 8;
                    if (size > 4) {
                        const uint64_t off = u32(e + 8);
                        if (off + size > tiff_len) break;
                        if (u16(e) == 0x0112 && !read(base + off, 4, val)) break;
                        vp = val;
                    }
                    if (u16(e) != 0x0112) continue;
                    // SHORT / LONG and their signed forms: the first value (Pillow keeps it when the count is not 1); any other
                    // type: a value that is not an orientation
                    if (typ == 3) v = u16(vp);
                    else if (typ == 8) v = (int16_t)u16(vp);
                    else if (typ == 4) v = u32(vp);
                    else if (typ == 9) v = (int32_t)u32(vp);
                    else v = 0;
                }
            }
        }
        if (v < 0 && xmp.p) {
            // the first match of tiff:Orientation(="|>)([0-9])
            static const char KEY[] = "tiff:Orientation";
            const size_t kl = sizeof(KEY) - 1;
            for (size_t at = 0; at + kl + 2 <= xmp.n;) {
                const uint8_t *f = (const uint8_t *)memmem(xmp.p + at, xmp.n - at, KEY, kl);
                if (!f) break;
                const size_t q = (size_t)(f - xmp.p) + kl;
                if (q + 1 < xmp.n && xmp.p[q] == '=' && xmp.p[q + 1] == '"' && q + 2 < xmp.n && xmp.p[q + 2] >= '0' && xmp.p[q + 2] <= '9') { v = xmp.p[q + 2] - '0'; break; }
                if (q + 1 < xmp.n && xmp.p[q] == '>' && xmp.p[q + 1] >= '0' && xmp.p[q + 1] <= '9') { v = xmp.p[q + 1] - '0'; break; }
                at = (size_t)(f - xmp.p) + 1;
            }
        }
        return v >= 2 && v <= 8 ? (uint32_t)v : 1u;
    }
};

struct zj_decoder {  // Decoder, reference src/decoder.rs:60-121
    StripSink *sink = nullptr;   // set for the duration of one zj_decoder_decode_into call
    zj_options options;
    zj_image_info info{};
    bool qt_present[4] = {false, false, false, false};
    int32_t qt_tables[4][64];
    HuffmanTable dc_tables[4], ac_tables[4];
    std::vector<Component> components;
    size_t h_max = 1, v_max = 1, mcu_width = 0, mcu_height = 0, mcu_x = 0, mcu_y = 0;
    bool interleaved = false;
    int sub_sample_ratio = SS_NONE;
    uint32_t input_colorspace = ZJ_CS_YCBCR;
    bool is_progressive = false;
    uint8_t spec_start = 0, spec_end = 0, succ_high = 0, succ_low = 0, num_scans = 0;
    size_t z_order[4] = {0, 0, 0, 0};
    size_t restart_interval = 0, todo = 0x7fffffff;
    // error of the last call
    int err_kind = ZJ_DE_NONE;
    std::string err_msg, err_display;
    // coefficient planes (reused across calls)
    PlaneBuf planes[3];
    PlaneBlock plane_block;
    size_t plane_len[3] = {0, 0, 0};
    bool have_device = false;
    // restart-interval-parallel entropy decode: threads to use (0 = options.num_threads) and how many intervals the last
    // decode ran side by side (0 = the sequential loop)
    size_t entropy_threads = 0, last_entropy_segments = 0;
    // EXIF orientation: the metadata segments met before the first SOS, and the orientation they give (1 until that SOS)
    OrientSource orient_src;
    bool before_sos = true;
    uint32_t orientation = 1;

    explicit zj_decoder(const zj_options &o) : options(o)
    {
        for (auto &t : dc_tables) t.present = false;
        for (auto &t : ac_tables) t.present = false;
        int n = 0;
        have_device = cudaGetDeviceCount(&n) == cudaSuccess && n > 0;
        if (!have_device) cudaGetLastError();
    }
    ~zj_decoder() { plane_block.release(); }

    void reset_state()  // a fresh Decoder::default(options) for every call, keeping the plane buffers
    {
        quirks = spec() ? 0u : g_quirks.load();
        const uint32_t keep_cs = user_out_cs;
        options.out_colorspace = keep_cs;
        info = zj_image_info{};
        for (bool &b : qt_present) b = false;
        for (auto &t : dc_tables) t.present = false;
        for (auto &t : ac_tables) t.present = false;
        components.clear();
        h_max = v_max = 1;
        mcu_width = mcu_height = mcu_x = mcu_y = 0;
        interleaved = false;
        sub_sample_ratio = SS_NONE;
        input_colorspace = ZJ_CS_YCBCR;
        is_progressive = false;
        spec_start = spec_end = succ_high = succ_low = num_scans = 0;
        for (auto &z : z_order) z = 0;
        restart_interval = 0;
        todo = 0x7fffffff;
        orient_src.clear();
        before_sos = true;
        orientation = 1;
    }
    uint32_t user_out_cs = ZJ_CS_RGB;
    uint32_t quirks = ZJ_QUIRK_ALL;   // the host-stage quirks of this decode (g_quirks when it started; none for spec output)
    bool quirk(uint32_t bit) const { return (quirks & bit) != 0; }
    // spec output, with either IDCT and at any scale: the host stage is the same for all, only the descriptor's ZJ_FLAG_ISLOW and
    // ZJ_FLAG_SCALE_* differ
    bool spec() const { return use() == ZJ_USE_SPEC_OUTPUT || libjpeg(); }
    bool libjpeg() const { return use() == ZJ_USE_LIBJPEG_OUTPUT || scale() != 0; }
    // ZJ_USE_LIBJPEG_OUTPUT | k << 4, k = 1..3: the DCT-scaled decode to 1/2^k (every other value keeps its meaning)
    static uint32_t scale_of(uint32_t u)
    {
        const uint32_t k = u >> 4;
        return (u & 15u) == ZJ_USE_LIBJPEG_OUTPUT && k >= 1 && k <= 3 ? k : 0;
    }
    uint32_t scale() const { return scale_of(use()); }
    // ZJ_USE_EXIF_ORIENTATION ORed into a spec, libjpeg or scaled value: that value, oriented; every other value keeps its meaning
    bool exif_orientation() const
    {
        const uint32_t u = options.use_unsafe & ~(uint32_t)ZJ_USE_EXIF_ORIENTATION;
        return (options.use_unsafe & ZJ_USE_EXIF_ORIENTATION) && (u == ZJ_USE_SPEC_OUTPUT || u == ZJ_USE_LIBJPEG_OUTPUT || scale_of(u) != 0);
    }
    uint32_t use() const { return exif_orientation() ? options.use_unsafe & ~(uint32_t)ZJ_USE_EXIF_ORIENTATION : options.use_unsafe; }
    // a one-component image: GRAYSCALE output (headers.rs:278-285, mcu.rs:171-196), except that spec output keeps RGB / RGBA / RGBX
    void gray_input_out_cs()
    {
        const uint32_t cs = options.out_colorspace;
        if (!(spec() && (cs == ZJ_CS_RGB || cs == ZJ_CS_RGBA || cs == ZJ_CS_RGBX))) options.out_colorspace = ZJ_CS_GRAYSCALE;
    }

    static size_t out_components(uint32_t cs)
    {
        switch (cs) {
        case ZJ_CS_RGB: case ZJ_CS_YCBCR: return 3;
        case ZJ_CS_GRAYSCALE: return 1;
        default: return 4;
        }
    }
    size_t in_components() const { return input_colorspace == ZJ_CS_GRAYSCALE ? 1 : 3; }

    // ---------------------------------------------------------------- headers (src/headers.rs)
    void parse_huffman(Cursor &buf)  // headers.rs:18-121
    {
        size_t avail = buf.pos < buf.len ? buf.len - buf.pos : 0;
        if (avail < 2) { buf.pos += avail; FAIL(ZJ_DE_FORMAT_STATIC, "Could not read Huffman length from image"); }
        const uint16_t l = buf.read_u16_be();
        if (l < 2) FAIL(ZJ_DE_FORMAT_STATIC, "Invalid Huffman length in image");
        int32_t dht_length = (int32_t)l - 2;
        while (dht_length > 16) {
            const uint8_t ht_info = buf.read_byte();
            const uint8_t dc_or_ac = (ht_info >> 4) & 0xF;
            const size_t index = ht_info & 0xF;
            uint8_t num_symbols[17] = {0};
            if (index >= 4) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("Invalid DHT index %zu, expected between 0 and 3", index));
            if (dc_or_ac > 1) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("Invalid DHT position %u, should be 0 or 1", (unsigned)dc_or_ac));
            buf.read_exact(num_symbols + 1, 16, ZJ_DE_HUFFMAN_DECODE, "Could not read bytes into the buffer");
            dht_length -= 1 + 16;
            int32_t symbols_sum = 0;
            for (int i = 0; i < 17; i++) symbols_sum += num_symbols[i];
            if (symbols_sum > 256) FAIL(ZJ_DE_HUFFMAN_DECODE, "Encountered Huffman table with excessive length in DHT");
            if (symbols_sum > dht_length)
                FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("Excessive Huffman table of length %d found when header length is %d", symbols_sum, dht_length));
            dht_length -= symbols_sum;
            uint8_t symbols[256] = {0};
            buf.read_exact(symbols, (size_t)symbols_sum, ZJ_DE_FORMAT, "Could not read symbols into the buffer\nfailed to fill whole buffer");
            if (dc_or_ac == 0) build_huffman(dc_tables[index], num_symbols, symbols, true, is_progressive, quirk(ZJ_QUIRK_Q9_FAST_AC_I16));
            else build_huffman(ac_tables[index], num_symbols, symbols, false, is_progressive, quirk(ZJ_QUIRK_Q9_FAST_AC_I16));
        }
        if (dht_length > 0) FAIL(ZJ_DE_HUFFMAN_DECODE, "Bogus Huffman table definition");
    }
    void parse_dqt(Cursor &buf)  // headers.rs:125-196
    {
        uint16_t l;
        try { l = buf.read_u16_be(); } catch (DecodeError &) { FAIL(ZJ_DE_FORMAT, "Could not read  DQT length Exhausted data in the image"); }
        if (l < 2) FAIL(ZJ_DE_DQT_ERROR, "Invalid DQT length. Length should be greater than 2");
        uint16_t qt_length = (uint16_t)(l - 2);
        while (qt_length > 0) {
            const uint8_t qt_info = buf.read_byte();
            const size_t precision = qt_info >> 4, table_position = qt_info & 0x0f;
            const size_t precision_value = 64 * (precision + 1);
            if ((uint16_t)(precision_value + 1) > qt_length)
                FAIL(ZJ_DE_DQT_ERROR, fmt("Invalid QT table bytes left :%u. Too small to construct a valid qt table which should be %zu long", (unsigned)qt_length, precision_value + 1));
            int32_t table[64];
            if (precision == 0) {
                uint8_t qv[64];
                buf.read_exact(qv, 64, ZJ_DE_FORMAT, "Could not read symbols into the buffer\nfailed to fill whole buffer");
                qt_length = (uint16_t)(qt_length - (uint16_t)precision_value - 1);
                for (int i = 0; i < 64; i++) table[UN_ZIGZAG[i]] = qv[i];  // un_zig_zag, headers.rs:533-543
            } else if (precision == 1) {
                FAIL(ZJ_DE_DQT_ERROR, "Support for 16 bit quantization table is not complete");
            } else {
                FAIL(ZJ_DE_DQT_ERROR, fmt("Expected QT precision value of either 0 or 1, found %zu", precision));
            }
            if (table_position >= 4) FAIL(ZJ_DE_DQT_ERROR, fmt("Too large table position for QT :%zu, expected between 0 and 3", table_position));
            memcpy(qt_tables[table_position], table, sizeof(table));
            qt_present[table_position] = true;
        }
    }
    void parse_start_of_frame(Cursor &buf, int sof)  // headers.rs:200-347
    {
        uint16_t length;
        try { length = buf.read_u16_be(); } catch (DecodeError &) { FAIL(ZJ_DE_FORMAT, "Cannot read SOF length, exhausted data"); }
        const uint8_t dt_precision = buf.read_byte();
        if (dt_precision != 8)
            FAIL(ZJ_DE_SOF_ERROR, fmt("The library can only parse 8-bit images, the image has %u bits of precision", (unsigned)dt_precision));
        info.pixel_density = dt_precision;
        uint16_t img_height, img_width;
        try { img_height = buf.read_u16_be(); } catch (DecodeError &) { FAIL(ZJ_DE_FORMAT, "Cannot read image height, exhausted data"); }
        info.height = img_height;
        try { img_width = buf.read_u16_be(); } catch (DecodeError &) { FAIL(ZJ_DE_FORMAT, "Cannot read image width, exhausted data"); }
        info.width = img_width;
        info.valid = 1;
        if (img_width > (uint16_t)options.max_width)
            FAIL(ZJ_DE_FORMAT, fmt("Image width %u greater than width limit %u. If use `set_limits` if you want to support huge images", (unsigned)img_width, (unsigned)(uint16_t)options.max_width));
        if (img_height > (uint16_t)options.max_height)
            FAIL(ZJ_DE_FORMAT, fmt("Image height %u greater than height limit %u. If use `set_limits` if you want to support huge images", (unsigned)img_height, (unsigned)(uint16_t)options.max_height));
        if (img_width == 0 || img_height == 0) FAIL(ZJ_DE_ZERO_ERROR, "");
        const uint8_t num_components = buf.read_byte();
        if (num_components == 0) FAIL(ZJ_DE_SOF_ERROR, "Number of components cannot be zero.");
        const uint16_t expected = (uint16_t)(8 + 3 * (uint16_t)num_components);
        if (length != expected)
            FAIL(ZJ_DE_SOF_ERROR, fmt("Length of start of frame differs from expected %u,value is %u", (unsigned)expected, (unsigned)length));
        if (num_components == 1) { input_colorspace = ZJ_CS_GRAYSCALE; gray_input_out_cs(); }
        info.components = num_components;
        std::vector<Component> comps;
        for (int i = 0; i < num_components; i++) {
            uint8_t a[3];
            buf.read_exact(a, 3, ZJ_DE_FORMAT, "Could not read component data\nfailed to fill whole buffer");
            Component c{};  // Components::from, components.rs:49-114
            if (a[0] == 1) c.component_id = ID_Y;
            else if (a[0] == 2) c.component_id = ID_CB;
            else if (a[0] == 3) c.component_id = ID_CR;
            else FAIL(ZJ_DE_FORMAT, fmt("Unknown component id found,%u, expected value between 1 and 3\nNote I and Q components are not supported yet", (unsigned)a[0]));
            c.horizontal_sample = a[1] >> 4;
            c.vertical_sample = a[1] & 0x0f;
            c.quantization_table_number = a[2];
            if (a[2] >= 4) FAIL(ZJ_DE_FORMAT, fmt("Too large quantization number :%u, expected value between 0 and 4", (unsigned)a[2]));
            auto pow2 = [](size_t x) { return x != 0 && (x & (x - 1)) == 0; };
            if (!pow2(c.horizontal_sample)) FAIL(ZJ_DE_FORMAT, fmt("Horizontal sample is not a power of two(%zu) cannot decode", c.horizontal_sample));
            if (!pow2(c.vertical_sample)) FAIL(ZJ_DE_FORMAT, fmt("Vertical sub-sample is not power of two(%zu) cannot decode", c.vertical_sample));
            c.width_stride = c.horizontal_sample;
            c.id = a[0];
            comps.push_back(c);
        }
        info.sof = (uint8_t)sof;
        for (auto &c : comps) {  // headers.rs:306-339 (h_max / mcu_x evolve component by component)
            h_max = std::max(h_max, c.horizontal_sample);
            v_max = std::max(v_max, c.vertical_sample);
            mcu_width = h_max * 8;
            mcu_height = v_max * 8;
            mcu_x = ((size_t)info.width + mcu_width - 1) / mcu_width;
            mcu_y = ((size_t)info.height + mcu_height - 1) / mcu_height;
            if (h_max != 1 || v_max != 1) interleaved = true;
            if (!qt_present[c.quantization_table_number])
                FAIL(ZJ_DE_DQT_ERROR, fmt("No quantization table for component %s", comp_debug(c.component_id)));
            memcpy(c.quantization_table, qt_tables[c.quantization_table_number], sizeof(c.quantization_table));
            c.width_stride *= mcu_x * 8;
        }
        for (bool &b : qt_present) b = false;  // headers.rs:343
        components = comps;
    }
    void parse_sos(Cursor &buf)  // headers.rs:350-463
    {
        const uint16_t ls = buf.read_u16_be();
        const uint8_t ns = buf.read_byte();
        bool seen[4] = {false, false, false, false};
        num_scans = ns;
        if (ls != 6 + 2 * (uint16_t)ns) FAIL(ZJ_DE_SOS_ERROR, "Bad SOS length,corrupt jpeg");
        if (!(ns >= 1 && ns < 4))
            FAIL(ZJ_DE_SOS_ERROR, fmt("Number of components in start of scan should be less than 3 but more than 0. Found %u", (unsigned)ns));
        if (info.components == 0) FAIL(ZJ_DE_SOF_ERROR, "Number of components cannot be zero.");
        for (int i = 0; i < ns; i++) {
            const uint8_t id = buf.read_byte();
            if ((size_t)id > components.size())
                FAIL(ZJ_DE_SOF_ERROR, fmt("Too large component ID %u, expected value between 0 and %zu", (unsigned)id, components.size()));
            if (id >= 4) FAIL(ZJ_DE_SOF_ERROR, fmt("Too large component ID %u, expected value between 0 and %zu", (unsigned)id, components.size()));
            if (seen[id]) FAIL(ZJ_DE_SOF_ERROR, fmt("Duplicate ID %u seen twice in the same component", (unsigned)id));
            seen[id] = true;
            const uint8_t y = buf.read_byte();
            uint8_t j = 0;
            while (j < info.components) {
                if (components[j].id == id) break;
                j++;
            }
            if (j == info.components)
                FAIL(ZJ_DE_SOF_ERROR, fmt("Invalid component id %u, expected a value between 0 and %zu", (unsigned)id, components.size()));
            components[j].dc_huff_table = (y >> 4) & 0xF;
            components[j].ac_huff_table = y & 0xF;
            z_order[i] = j;
        }
        spec_start = buf.read_byte() & 63;
        spec_end = buf.read_byte() & 63;
        const uint8_t bit_approx = buf.read_byte();
        succ_high = bit_approx >> 4;
        if (succ_high > 13) FAIL(ZJ_DE_SOF_ERROR, fmt("Invalid Ah parameter %u, range should be 0-13", (unsigned)succ_low));
        succ_low = bit_approx & 0xF;
        if (succ_low > 13) FAIL(ZJ_DE_SOF_ERROR, fmt("Invalid Al parameter %u, range should be 0-13", (unsigned)succ_low));
    }
    void skip_segment(Cursor &buf, const char *msg_fmt)
    {
        const uint16_t length = buf.read_u16_be();
        if (length < 2) FAIL(ZJ_DE_FORMAT, fmt(msg_fmt, (unsigned)length));
        buf.consume((size_t)length - 2);
    }
    void parse_marker_inner(const Marker &m, Cursor &buf)  // decoder.rs:304-411
    {
        switch (m.kind) {
        case M_SOF:
            if (m.n == 2) is_progressive = true;
            parse_start_of_frame(buf, m.n == 0 ? 0 : 2);
            break;
        case M_DQT: parse_dqt(buf); break;
        case M_DHT: parse_huffman(buf); break;
        case M_SOS:
            if (before_sos) { before_sos = false; orientation = orient_src.orientation(); }
            parse_sos(buf);
            break;
        case M_EOI: FAIL(ZJ_DE_FORMAT, "Premature End of image");
        case M_DAC: case M_DNL:
            FAIL(ZJ_DE_FORMAT, fmt("Parsing of the following header `%s` is not supported,cannot continue", marker_debug(m).c_str()));
        case M_DRI:
            if (buf.read_u16_be() != 4) FAIL(ZJ_DE_FORMAT, "Bad DRI length, Corrupt JPEG");
            restart_interval = buf.read_u16_be();
            todo = restart_interval;
            break;
        case M_APP:
            if (m.n == 1 && before_sos) {
                const size_t start = buf.pos + 2;
                skip_segment(buf, "Found a marker with invalid length:%u\n");
                note_app1(buf.data + start, std::min(buf.pos, buf.len) - std::min(start, buf.len));
                break;
            }
            skip_segment(buf, "Found a marker with invalid length:%u\n");
            break;
        default: skip_segment(buf, "Found a marker with invalid length:%u\n"); break;
        }
    }
    // an APP1 segment's payload before the first SOS: EXIF or XMP (JpegImagePlugin.py APP())
    void note_app1(const uint8_t *p, size_t n)
    {
        static const char XMP[] = "http://ns.adobe.com/xap/1.0/";   // (29 bytes with its NUL)
        OrientSource &o = orient_src;
        if (n >= 6 && memcmp(p, "Exif\0\0", 6) == 0) {
            const size_t skip = o.exif.empty() ? 0 : 6;
            o.exif.push_back({p + skip, n - skip});
            o.exif_len += n - skip;
        } else if (n >= sizeof(XMP) && memcmp(p, XMP, sizeof(XMP)) == 0) {
            o.xmp = {p + sizeof(XMP), n - sizeof(XMP)};
        }
    }
    void decode_headers_internal(Cursor &buf)  // decoder.rs:239-303
    {
        const uint16_t magic = buf.read_u16_be();
        uint8_t last_byte = 0;
        size_t bytes_before_marker = 0;
        if (magic != 0xffd8) FAIL(ZJ_DE_ILLEGAL_MAGIC_BYTES, fmt("%u", (unsigned)magic));
        for (;;) {
            const uint8_t m = buf.read_byte();
            if (last_byte == 0xFF) {
                Marker mk;
                bytes_before_marker = 0;
                if (marker_from_u8(m, &mk)) {
                    parse_marker_inner(mk, buf);
                    if (mk.kind == M_SOS) return;
                } else {
                    skip_segment(buf, "Found a marker with invalid length : %u");
                }
            }
            last_byte = m;
            bytes_before_marker += 1;
            if (options.strict_mode && bytes_before_marker > 3) FAIL(ZJ_DE_FORMAT_STATIC, "[strict-mode]: Extra bytes between headers");
        }
    }

    // ---------------------------------------------------------------- checks (decoder.rs:468-523,609-646; mcu.rs:74-116)
    void check_component_dimensions()
    {
        const Component *y = nullptr;
        for (auto &c : components) if (c.component_id == ID_Y) { y = &c; break; }
        if (!y) FAIL(ZJ_DE_FORMAT_STATIC, "Could not find Y component for the image");
        const size_t cbcr = y->width_stride / h_max;
        for (auto &c : components) {
            if (c.component_id == ID_Y) continue;
            if (c.width_stride != cbcr)
                FAIL(ZJ_DE_FORMAT, fmt("Invalid image width and height stride for component %s, expected %zu, but found %zu", comp_debug(c.component_id), cbcr, c.width_stride));
            if (c.horizontal_sample != 1 || c.vertical_sample != 1)
                FAIL(ZJ_DE_FORMAT, fmt("Invalid component sample for component %s, expected (1,1), found (%zu,%zu)", comp_debug(c.component_id), c.vertical_sample, c.horizontal_sample));
        }
    }
    void check_tables()
    {
        for (size_t i = 0; i < in_components() && i < components.size(); i++) {
            const Component &c = components[i];
            if (c.dc_huff_table >= 4) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("No Huffman DC table for component %s ", comp_debug(c.component_id)));
            if (!dc_tables[c.dc_huff_table].present) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("No DC table for component %s", comp_debug(c.component_id)));
            if (c.ac_huff_table >= 4) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("No Huffman AC table for component %s ", comp_debug(c.component_id)));
            if (!ac_tables[c.ac_huff_table].present) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("No AC table for component %s", comp_debug(c.component_id)));
        }
    }
    void set_upsampling()
    {
        if (h_max == v_max && h_max == 1) return;
        if (h_max == 2 && v_max == 1) sub_sample_ratio = SS_H;
        else if (h_max == 1 && v_max == 2) sub_sample_ratio = SS_V;
        else if (h_max == 2 && v_max == 2) sub_sample_ratio = SS_HV;
        else FAIL(ZJ_DE_FORMAT, "Unknown down-sampling method, cannot continue");
    }
    void handle_rst(BitStream &stream)  // mcu.rs:386-418
    {
        todo = restart_interval;
        if (stream.has_marker) {
            if (stream.marker.kind == M_RST) {
                stream.reset();
                for (auto &c : components) c.dc_pred = 0;
            } else if (stream.marker.kind == M_EOI) {
            } else {
                FAIL(ZJ_DE_MCU_ERROR, fmt("Marker %s found in bitstream, possibly corrupt jpeg", marker_debug(stream.marker).c_str()));
            }
        }
    }

    // ---------------------------------------------------------------- baseline entropy stage (mcu.rs:127-351)
    // State the MCU loop of mcu.rs:253-351 carries from block to block.  The sequential decode owns one for the whole
    // scan; the restart-interval-parallel decode gives every interval its own.
    struct ScanState {
        BitStream stream;
        int32_t dc_pred[3] = {0, 0, 0};
        size_t todo = 0;
    };
    struct BaselineGeom {
        size_t mcu_w = 0, mcu_h = 0, bias = 1, width_stride = 0, hv_width_stride = 0, out_nc = 0, ncomp = 0;
        size_t total = 0;   // MCUs the scan decodes
        bool is_hv = false, zero_per_strip = false;
        size_t strip_len[3] = {0, 0, 0};
    };
    struct SegmentAbnormal {};   // the interval did not end the way a conformant one does: redo the scan sequentially

    // The MCU loop over MCUs [first, last) in (strip, v, j) order.
    //   SEGMENT == false: the reference's loop as written (first = 0, last = all): handle_rst / marker handling of
    //                     mcu.rs:323-348, 386-418.
    //   SEGMENT == true : one restart interval decoded on its own.  The same state machine, but it must end with the
    //                     reset of handle_rst exactly after the last component of MCU last-1 (returns true; `must_reset`
    //                     says whether that is required) and must not meet anything else the sequential loop would
    //                     react to (an earlier reset, EOI before the end, another marker): those throw SegmentAbnormal
    //                     and the caller falls back to the sequential loop, which then reproduces whatever the reference
    //                     does with such a stream (SURVEY Q8).
    template <bool SEGMENT>
    bool baseline_mcus(Cursor &reader, ScanState &st, const BaselineGeom &g, const size_t first, const size_t last, const bool must_reset)
    {
        int16_t tmp[64];
        BitStream &stream = st.stream;
        const size_t per_strip = g.bias * g.mcu_w;
        for (size_t m = first; m < last; m++) {
            const size_t strip = m / per_strip, v = (m - strip * per_strip) / g.mcu_w, j = m - strip * per_strip - v * g.mcu_w;
            if (!SEGMENT && sink && strip > 0 && m == strip * per_strip) sink->progress(strip);
            if (!SEGMENT && g.zero_per_strip && m == strip * per_strip) {
                // the planes start out zeroed (mcu.rs:238-250 allocates fresh zeroed strip buffers): done strip by strip right
                // before the strip is decoded, so the blocks are still in cache when the coefficients are written
                for (size_t pos = 0; pos < 3; pos++)
                    if (g.strip_len[pos]) memset(planes[pos].p + strip * g.strip_len[pos], 0, g.strip_len[pos] * 2);
            }
            for (size_t pos = 0; pos < g.ncomp; pos++) {
                const Component &component = components[pos];
                const HuffmanTable &dc_table = dc_tables[component.dc_huff_table & 3];
                if (!dc_table.present) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("No DC table for component %s", comp_debug(component.component_id)));
                const HuffmanTable &ac_table = ac_tables[component.ac_huff_table & 3];
                if (!ac_table.present) FAIL(ZJ_DE_HUFFMAN_DECODE, fmt("No AC table for component %s", comp_debug(component.component_id)));
                for (size_t v_samp = 0; v_samp < component.vertical_sample; v_samp++) {
                    for (size_t h_samp = 0; h_samp < component.horizontal_sample; h_samp++) {
                        if (std::min(g.out_nc - 1, pos) == pos) {
                            // mcu.rs:293-312
                            const size_t is_y = component.component_id == ID_Y ? 1 : 0;
                            const size_t y_offset = is_y * v * (g.hv_width_stride + (g.hv_width_stride * (component.vertical_sample - 1)));
                            const size_t another_stride = (g.width_stride * v_samp * (g.is_hv ? 0 : 1)) + g.hv_width_stride * v_samp * (g.is_hv ? 1 : 0);
                            const size_t yet_another_stride = (g.is_hv ? 1 : 0) * (g.width_stride >> 2) * v * (component.component_id != ID_Y ? 1 : 0);
                            const size_t start = (j * 64 * component.horizontal_sample) + (h_samp * 64) + another_stride + y_offset + yet_another_stride;
                            if (start + 64 > g.strip_len[pos]) FAIL(ZJ_DE_GPU, "the reference decoder panics here (block index out of range, mcu.rs:314)");
                            stream.decode_mcu_block(reader, dc_table, ac_table, planes[pos].p + strip * g.strip_len[pos] + start, st.dc_pred[pos]);
                        } else {
                            stream.decode_mcu_block(reader, dc_table, ac_table, tmp, st.dc_pred[pos]);
                        }
                    }
                }
                st.todo = st.todo - 1;  // wrapping_sub, once per COMPONENT (Q8)
                if (st.todo == 0) {     // handle_rst, mcu.rs:386-418
                    st.todo = restart_interval;
                    if (stream.has_marker) {
                        if (stream.marker.kind == M_RST) {
                            stream.reset();
                            for (int32_t &p : st.dc_pred) p = 0;
                            if (SEGMENT) {
                                if (m + 1 == last && pos + 1 == g.ncomp) return true;
                                throw SegmentAbnormal{};   // a reset in the middle of the interval
                            }
                        } else if (stream.marker.kind == M_EOI) {
                        } else {
                            FAIL(ZJ_DE_MCU_ERROR, fmt("Marker %s found in bitstream, possibly corrupt jpeg", marker_debug(stream.marker).c_str()));
                        }
                    }
                }
                if (stream.has_marker) {  // mcu.rs:337-348
                    if (stream.marker.kind == M_EOI) {
                        if (SEGMENT && must_reset) throw SegmentAbnormal{};
                        // Q11 (mcu.rs:337-342): the reader PREFETCHES, so EOI is usually "seen" while the last MCU still has
                        // components to decode from buffered bits; the break drops them.  Quirk off: finish the MCU.
                        if (quirk(ZJ_QUIRK_Q11_EOI_BREAK)) break;
                        continue;
                    }
                    if (stream.marker.kind == M_RST) continue;
                    if (SEGMENT) throw SegmentAbnormal{};
                    parse_marker_inner(stream.marker, reader);
                }
            }
        }
        if (SEGMENT && must_reset) throw SegmentAbnormal{};   // the interval ended without the reader having met its RSTn
        return false;
    }

    // Ends of the RSTn markers of the scan that starts at `from` (index of the byte after 0xFF [0xFF..] 0xDn, i.e. where the
    // bit reader stands after bitstream.rs:200-215 met it).  Stops at the first marker that is not RSTn.
    static void find_restart_markers(const Cursor &reader, size_t from, size_t want, std::vector<size_t> &ends)
    {
        const uint8_t *d = reader.data;
        const size_t n = reader.len;
        size_t p = from;
        while (p < n && ends.size() < want) {
            const uint8_t *f = (const uint8_t *)memchr(d + p, 0xFF, n - p);
            if (!f) break;
            p = (size_t)(f - d) + 1;
            while (p < n && d[p] == 0xFF) p++;
            if (p >= n) break;
            const uint8_t b = d[p++];
            if (b == 0x00) continue;
            if (b >= 0xD0 && b <= 0xD7) { ends.push_back(p); continue; }
            break;
        }
    }

    // Restart-interval-parallel form of the loop (SURVEY 8(f).1): with DRI present every interval starts from a known
    // state (fresh bit reader right after its RSTn, predictors 0, countdown = DRI), so `threads` host threads decode
    // different intervals side by side, each with the reference's own state machine, straight into the planes.  It is only
    // kept when EVERY interval ended exactly where the next one was assumed to start (same MCU, same byte); then the
    // sequential loop would have gone through the very same states.  Anything else returns false with the planes dirty.
    bool baseline_parallel(const Cursor &reader0, const ScanState &st0, const BaselineGeom &g, size_t threads)
    {
        const size_t total = g.total;
        // a conformant stream has DRI MCUs per interval = DRI * ncomp ticks of the countdown (Q8: it ticks once per
        // component), so it fires ncomp times per interval and only the last firing, at the interval's end, meets the marker
        const size_t per_seg = restart_interval;
        if (per_seg == 0 || total <= per_seg) return false;
        const size_t n_seg = (total + per_seg - 1) / per_seg;
        std::vector<size_t> ends;
        ends.reserve(n_seg);
        find_restart_markers(reader0, reader0.pos, n_seg - 1, ends);
        if (ends.size() < n_seg - 1) return false;
        if (threads > n_seg) threads = n_seg;
        std::atomic<size_t> next{0};
        std::atomic<bool> bad{false};
        // strips complete so far = the prefix of finished intervals (intervals are claimed in order, so the prefix keeps up)
        std::mutex prefix_mu;
        std::vector<uint8_t> seg_done(sink ? n_seg : 0, 0);
        size_t prefix = 0, told = 0;
        const size_t per_strip = g.bias * g.mcu_w;
        auto finished = [&](size_t k) {
            if (!sink) return;
            std::lock_guard<std::mutex> lock(prefix_mu);
            seg_done[k] = 1;
            while (prefix < n_seg && seg_done[prefix]) prefix++;
            if (bad.load(std::memory_order_relaxed)) return;
            const size_t strips = std::min(total, prefix * per_seg) / per_strip;
            if (strips > told && strips < g.mcu_h) { told = strips; sink->progress(strips); }   // (the last strip is reported by the caller)
        };
        auto work = [&]() {
            for (;;) {
                const size_t k = next.fetch_add(1);
                if (k >= n_seg || bad.load(std::memory_order_relaxed)) return;
                Cursor rd = reader0;
                ScanState st;
                if (k == 0) st = st0;
                else { rd.pos = ends[k - 1]; st.todo = restart_interval; st.stream.q10 = quirk(ZJ_QUIRK_Q10_DC_REFILL); }
                const size_t first = k * per_seg, last = std::min(total, first + per_seg);
                const bool must_reset = k + 1 < n_seg;
                try {
                    const bool was_reset = baseline_mcus<true>(rd, st, g, first, last, must_reset);
                    if (must_reset && (!was_reset || rd.pos != ends[k])) bad = true;
                    else finished(k);
                } catch (SegmentAbnormal &) { bad = true; }
                catch (...) { bad = true; }   // a DecodeError: the sequential loop will raise it at the right place
            }
        };
        std::vector<std::thread> pool;
        for (size_t t = 1; t < threads; t++) if (!spawn(pool, work)) break;
        work();
        for (auto &t : pool) t.join();
        if (bad) return false;
        last_entropy_segments = n_seg;
        return true;
    }

    // Everything decode_baseline settles before its MCU loop (mcu.rs:139-250): checks, strip geometry, plane sizes.
    void baseline_setup(BaselineGeom &g)
    {
        check_component_dimensions();
        check_tables();
        if (components.size() < in_components()) FAIL(ZJ_DE_FORMAT, "missing components");
        size_t mcu_w, mcu_h, bias = 1;
        if (interleaved) {
            set_upsampling();
            // Q1: strips of two MCU rows, an odd last MCU row is dropped; spec output decodes it, in a half-empty last strip
            const size_t strips2 = spec() ? (mcu_y + 1) / 2 : mcu_y / 2;
            if (sub_sample_ratio == SS_H) { mcu_w = mcu_x * 2; mcu_h = strips2; }
            else if (sub_sample_ratio == SS_HV) { mcu_w = mcu_x; mcu_h = strips2; bias = 2; }
            else { mcu_w = mcu_x; mcu_h = mcu_y; }
        } else {
            mcu_w = ((size_t)info.width + 7) / 8;
            mcu_h = ((size_t)info.height + 7) / 8;
        }
        if (input_colorspace == ZJ_CS_GRAYSCALE && interleaved) {  // mcu.rs:171-196
            if (options.strict_mode) FAIL(ZJ_DE_FORMAT_STATIC, "[strict-mode]: Grayscale image with down-sampled component.");
            mcu_w = ((size_t)info.width + 7) / 8;
            h_max = 1;
            gray_input_out_cs();
            v_max = 1;
            sub_sample_ratio = SS_NONE;
            components[0].vertical_sample = 1;
            components[0].width_stride = mcu_w * 8;
            components[0].horizontal_sample = 1;
            mcu_h = ((size_t)info.height + 7) / 8;
            bias = 1;
        }
        const size_t component_capacity = mcu_w * 64;
        g.mcu_w = mcu_w; g.mcu_h = mcu_h; g.bias = bias;
        g.total = mcu_w * mcu_h * bias;
        if (spec() && (sub_sample_ratio == SS_H || sub_sample_ratio == SS_HV)) g.total = mcu_x * mcu_y;
        g.is_hv = sub_sample_ratio == SS_HV;
        g.out_nc = out_components(options.out_colorspace);
        g.ncomp = in_components();
        g.width_stride = (component_capacity * components[0].vertical_sample * components[0].horizontal_sample * bias) >> 1;
        g.hv_width_stride = g.width_stride >> 1;
        // the reference's output Vec must have one chunk per strip, or chunks.next().unwrap() panics (mcu.rs:354)
        if (!spec()) {
            const size_t capacity = (size_t)(uint16_t)(info.width + 8) * (size_t)(uint16_t)(info.height + 8);
            const size_t extra = (interleaved ? 128u : 0u) * (size_t)info.height * g.out_nc;
            const size_t chunk = (size_t)info.width * g.out_nc * 8 * h_max * v_max;
            if (mcu_h > (capacity * g.out_nc + extra) / chunk) FAIL(ZJ_DE_GPU, "the reference decoder panics on this geometry (output chunks exhausted, mcu.rs:354)");
        }
        // whole-image planes: strip s of component z lives at s * strip_len[z] (== mcu_prog.rs layout)
        for (size_t pos = 0; pos < 3; pos++) { plane_len[pos] = 0; g.strip_len[pos] = 0; }
        for (size_t pos = 0; pos < components.size() && pos < 3; pos++) {
            if (std::min(g.out_nc - 1, pos) == pos) {  // mcu.rs:244
                g.strip_len[pos] = component_capacity * components[pos].vertical_sample * components[pos].horizontal_sample * bias;
                plane_len[pos] = g.strip_len[pos] * mcu_h;
            }
        }
    }

    void decode_baseline(Cursor &reader)
    {
        BaselineGeom g;
        baseline_setup(g);
        last_entropy_segments = 0;
        size_t threads = entropy_threads ? entropy_threads : (options.num_threads ? options.num_threads : std::thread::hardware_concurrency());
        if (threads == 0) threads = 1;
        const size_t total = g.total;
        plane_block.ensure(planes, plane_len, have_device, false);
        // zeroing all planes at once, for the interval-parallel form (whose intervals start anywhere inside a strip): split over
        // the threads too -- 200 MB of planes of an 8192^2 image take as long to clear as to entropy-decode on 8 threads
        auto zero_planes = [&]() {
            const size_t CH = (size_t)1 << 20;   // bytes per piece
            std::vector<std::pair<char *, size_t>> pieces;
            for (size_t pos = 0; pos < 3; pos++)
                for (size_t o = 0; o < plane_len[pos] * 2; o += CH) pieces.emplace_back((char *)planes[pos].p + o, std::min(CH, plane_len[pos] * 2 - o));
            std::atomic<size_t> next{0};
            auto work = [&]() { for (size_t i; (i = next.fetch_add(1)) < pieces.size();) memset(pieces[i].first, 0, pieces[i].second); };
            std::vector<std::thread> pool;
            for (size_t t = 1; t < threads && t < pieces.size(); t++) if (!spawn(pool, work)) break;
            work();
            for (auto &t : pool) t.join();
        };
        if (sink) {
            zj_image img;
            fill_descriptor(&img);
            sink->begin(img, g.mcu_h);
        }
        ScanState st;
        st.stream.q10 = quirk(ZJ_QUIRK_Q10_DC_REFILL);
        for (size_t pos = 0; pos < g.ncomp && pos < 3; pos++) st.dc_pred[pos] = components[pos].dc_pred;
        st.todo = todo;
        // worth the thread start-up only for scans of some size (about 0.1 ms of Huffman work per 4096 blocks)
        if (threads > 1 && restart_interval > 0 && todo == restart_interval && total >= 2 * restart_interval &&
            reader.len - std::min(reader.len, reader.pos) >= (size_t)64 * 1024) {
            zero_planes();
            if (baseline_parallel(reader, st, g, threads)) return;
            // some interval did not end like a conformant one: the reference's loop decides what comes out
            if (sink) sink->restart();
        }
        g.zero_per_strip = true;
        baseline_mcus<false>(reader, st, g, 0, total, false);
        for (size_t pos = 0; pos < g.ncomp && pos < 3; pos++) components[pos].dc_pred = st.dc_pred[pos];
        todo = st.todo;
    }

    // ---------------------------------------------------------------- GPU form of the baseline entropy stage (zj_entropy.cu)
    struct GpuPrep {
        BaselineGeom g;
        std::vector<uint32_t> seg_start;   // reader position at the start of every restart interval (+ one unused entry)
        size_t n_seg = 0, total = 0;
    };
    // Headers are parsed (reader stands at the first entropy-coded byte).  True when the scan can be handed to the GPU: a
    // baseline scan with restart markers in the state the interval-parallel forms start from.  Everything else -- and every
    // error -- is left to the host stage, which then reports exactly what the reference reports.
    bool gpu_entropy_prepare(const Cursor &reader, GpuPrep &pp)
    {
        if (is_progressive || restart_interval == 0 || todo != restart_interval) return false;
        if (quirks != ZJ_QUIRK_ALL) return false;   // the GPU form carries the quirks as written; test switches and spec output -> host stage
        if (reader.len >= 0xFFFFFFF0ull) return false;
        try { baseline_setup(pp.g); } catch (DecodeError &) { return false; }
        const BaselineGeom &g = pp.g;
        for (size_t pos = 0; pos < g.ncomp; pos++) {
            const Component &c = components[pos];
            if (c.dc_pred != 0 || !dc_tables[c.dc_huff_table & 3].present || !ac_tables[c.ac_huff_table & 3].present) return false;
            if (g.strip_len[pos] > 0x7FFFFFFFull || plane_len[pos] > ((size_t)1 << 40)) return false;
        }
        pp.total = g.total;
        if (pp.total <= restart_interval || pp.total > 0x7FFFFFFFull) return false;
        pp.n_seg = (pp.total + restart_interval - 1) / restart_interval;
        std::vector<size_t> ends;
        ends.reserve(pp.n_seg);
        find_restart_markers(reader, reader.pos, pp.n_seg - 1, ends);
        if (ends.size() < pp.n_seg - 1) return false;
        pp.seg_start.resize(pp.n_seg + 1);
        pp.seg_start[0] = (uint32_t)reader.pos;
        for (size_t k = 1; k < pp.n_seg; k++) pp.seg_start[k] = (uint32_t)ends[k - 1];
        pp.seg_start[pp.n_seg] = 0;
        return true;
    }
    void gpu_entropy_tables(zj::EntTable *t) const   // [dc, ac] per component
    {
        for (size_t pos = 0; pos < in_components(); pos++) {
            const HuffmanTable *src[2] = {&dc_tables[components[pos].dc_huff_table & 3], &ac_tables[components[pos].ac_huff_table & 3]};
            for (int k = 0; k < 2; k++) {
                zj::EntTable &d = t[2 * pos + k];
                memcpy(d.lookup, src[k]->lookup, sizeof(d.lookup));
                memcpy(d.ac_lookup, src[k]->ac_lookup, sizeof(d.ac_lookup));
                memcpy(d.maxcode, src[k]->maxcode, sizeof(d.maxcode));
                memcpy(d.offset, src[k]->offset, sizeof(d.offset));
                memcpy(d.values, src[k]->values, sizeof(d.values));
            }
        }
    }

    // ---------------------------------------------------------------- progressive entropy stage (mcu_prog.rs)
    bool get_marker(Cursor &reader, BitStream &stream, Marker *out)  // mcu_prog.rs:436-473
    {
        if (stream.has_marker) { stream.has_marker = false; *out = stream.marker; return true; }
        for (;;) {
            if (reader.pos >= reader.len) return false;
            const uint8_t marker = reader.data[reader.pos++];
            if (marker == 255) {
                if (reader.pos >= reader.len) return false;
                uint8_t r = reader.data[reader.pos++];
                while (r == 0xFF) {
                    if (reader.pos >= reader.len) return false;
                    r = reader.data[reader.pos++];
                }
                if (r != 0) return marker_from_u8(r, out);
                if (reader.pos >= reader.len) return false;
            }
        }
    }
    void parse_entropy_coded_data(Cursor &reader, BitStream &stream)  // mcu_prog.rs:249-430
    {
        check_component_dimensions();
        stream.reset();
        for (auto &c : components) c.dc_pred = 0;
        if ((size_t)num_scans > in_components())
            FAIL(ZJ_DE_FORMAT, fmt("Number of scans %u cannot be greater than number of components, %zu", (unsigned)num_scans, in_components()));
        if (num_scans == 1) {
            if (spec_end != 0 && spec_start == 0) FAIL(ZJ_DE_HUFFMAN_DECODE, "Can't merge DC and AC corrupt jpeg");
            const size_t k = z_order[0];
            if (k >= components.size()) FAIL(ZJ_DE_FORMAT, fmt("Cannot find component %zu, corrupt image", k));
            size_t mw, mh;
            if (components[k].component_id == ID_Y || !interleaved) { mw = ((size_t)info.width + 7) / 8; mh = ((size_t)info.height + 7) / 8; }
            else { mw = mcu_x; mh = mcu_y; }
            size_t i = 0, j = 0;
            while (i < mh) {
                while (j < mw) {
                    const size_t start = 64 * (j + i * (components[k].width_stride / 8));
                    if (i >= mh) break;
                    if (k >= 3 || start + 64 > plane_len[k]) FAIL(ZJ_DE_GPU, "the reference decoder panics here (block index out of range, mcu_prog.rs:304)");
                    int16_t *data = planes[k].p + start;
                    if (spec_start == 0) {
                        const size_t pos = components[k].dc_huff_table & 3;
                        if (!dc_tables[pos].present) FAIL(ZJ_DE_FORMAT, fmt("Huffman table at index  %zu not initialized", pos));
                        if (succ_high == 0) stream.decode_prog_dc_first(reader, dc_tables[pos], data, components[k].dc_pred);
                        else stream.decode_prog_dc_refine(reader, data);
                    } else {
                        const size_t pos = components[k].ac_huff_table;
                        if (pos >= 4) FAIL(ZJ_DE_FORMAT, fmt("No huffman table for component:%zu", pos));
                        if (!ac_tables[pos].present) FAIL(ZJ_DE_FORMAT, fmt("Huffman table at index  %zu not initialized", pos));
                        if (succ_high == 0) {
                            if (stream.eob_run > 0) {  // skip whole blocks, mcu_prog.rs:336-351
                                i += (j + (size_t)stream.eob_run - 1) / mw;
                                j = (j + (size_t)stream.eob_run - 1) % mw;
                                stream.eob_run = 0;
                            } else {
                                stream.decode_mcu_ac_first(reader, ac_tables[pos], data);
                            }
                        } else {
                            stream.decode_mcu_ac_refine(reader, ac_tables[pos], data);
                        }
                    }
                    j += 1;
                    todo -= 1;
                    if (todo == 0) handle_rst(stream);
                }
                j = 0;
                i += 1;
            }
        } else {
            if (spec_end != 0) FAIL(ZJ_DE_HUFFMAN_DECODE, "Can't merge dc and AC corrupt jpeg");
            for (size_t i = 0; i < mcu_y; i++) {
                for (size_t j = 0; j < mcu_x; j++) {
                    for (size_t k = 0; k < num_scans; k++) {
                        const size_t n = z_order[k];
                        if (n >= components.size()) FAIL(ZJ_DE_FORMAT, fmt("Cannot find component %zu, corrupt image", n));
                        Component &component = components[n];
                        if (component.dc_huff_table >= 4) FAIL(ZJ_DE_FORMAT, fmt("No huffman table for component:%zu", component.dc_huff_table));
                        const HuffmanTable &huff_table = dc_tables[component.dc_huff_table];
                        if (!huff_table.present) FAIL(ZJ_DE_FORMAT, fmt("Huffman table at index  %zu not initialized", component.dc_huff_table));
                        for (size_t v_samp = 0; v_samp < component.vertical_sample; v_samp++) {
                            for (size_t h_samp = 0; h_samp < component.horizontal_sample; h_samp++) {
                                const size_t x2 = j * component.horizontal_sample + h_samp;
                                const size_t y2 = i * component.vertical_sample + v_samp;
                                const size_t position = 64 * (x2 + y2 * component.width_stride / 8);
                                if (n >= 3 || position >= plane_len[n]) FAIL(ZJ_DE_GPU, "the reference decoder panics here (block index out of range, mcu_prog.rs:408)");
                                int16_t *data = planes[n].p + position;
                                if (succ_high == 0) stream.decode_prog_dc_first(reader, huff_table, data, component.dc_pred);
                                else stream.decode_prog_dc_refine(reader, data);
                            }
                        }
                        todo = todo - 1;
                        if (todo == 0) handle_rst(stream);
                    }
                }
            }
        }
    }
    void decode_progressive(Cursor &reader)  // mcu_prog.rs:49-129 (+ the geometry half of finish_progressive_decoding)
    {
        check_component_dimensions();
        size_t mw, mh;
        if (interleaved) { mw = mcu_x; mh = mcu_y; } else { mw = ((size_t)info.width + 7) / 8; mh = ((size_t)info.height + 7) / 8; }
        if (spec() && interleaved && h_max == 2) mh += mh & 1;   // 4:2:2 / 4:2:0 spec output reads whole strips of two MCU rows
        mw *= 64;
        if (components.size() < in_components()) FAIL(ZJ_DE_FORMAT, "missing components");
        for (size_t i = 0; i < 3; i++) plane_len[i] = 0;
        for (size_t i = 0; i < in_components(); i++) plane_len[i] = mw * components[i].vertical_sample * components[i].horizontal_sample * mh;
        plane_block.ensure(planes, plane_len, have_device, true);
        size_t seen_scans = 1;
        BitStream stream;
        stream.q10 = quirk(ZJ_QUIRK_Q10_DC_REFILL);
        stream.update_progressive_params(succ_high, succ_low, spec_start, spec_end);
        parse_entropy_coded_data(reader, stream);
        if (!stream.has_marker) FAIL(ZJ_DE_FORMAT_STATIC, "Marker missing where expected");
        Marker marker = stream.marker;
        stream.has_marker = false;
        while (!(marker.kind == M_EOI)) {
            if (marker.kind == M_DHT) {
                parse_huffman(reader);
            } else if (marker.kind == M_SOS) {
                parse_sos(reader);
                stream.update_progressive_params(succ_high, succ_low, spec_start, spec_end);
                parse_entropy_coded_data(reader, stream);
                if (!get_marker(reader, stream, &marker)) FAIL(ZJ_DE_FORMAT_STATIC, "Marker missing where expected");
                seen_scans += 1;
                if (seen_scans > options.max_scans) FAIL(ZJ_DE_FORMAT, fmt("Too many scans, exceeded limit of %u", (unsigned)options.max_scans));
                stream.reset();
                continue;
            } else {
                break;
            }
            if (!get_marker(reader, stream, &marker)) FAIL(ZJ_DE_FORMAT_STATIC, "Marker missing where expected");
        }
        // finish_progressive_decoding, mcu_prog.rs:132-168
        set_upsampling();
        if (input_colorspace == ZJ_CS_GRAYSCALE && interleaved) {
            if (options.strict_mode) FAIL(ZJ_DE_FORMAT_STATIC, "[strict-mode]: Grayscale image with down-sampled component.");
            // mcu_prog.rs:161-167 sets horizontal_sample = mcu_width ("not tested" per its own comment); the IDCT
            // then indexes past its chunk and panics (idct get_mut(..).unwrap()).
            FAIL(ZJ_DE_GPU, "the reference decoder panics on progressive grayscale images with a down-sampled component");
        }
    }

    // ---------------------------------------------------------------- host stage driver
    void fill_descriptor(zj_image *img)
    {
        memset(img, 0, sizeof(*img));
        img->width = info.width;
        img->height = info.height;
        img->n_comp = (uint32_t)in_components();
        img->out_cs = options.out_colorspace;
        img->variant = spec() ? ZJ_VARIANT_SPEC : (options.use_unsafe ? ZJ_VARIANT_X86 : ZJ_VARIANT_SCALAR);
        img->flags = (is_progressive ? ZJ_FLAG_PROGRESSIVE : 0) | (libjpeg() ? ZJ_FLAG_ISLOW : 0) | scale() << ZJ_FLAG_SCALE_SHIFT |
                     (exif_orientation() ? (orientation - 1) << ZJ_FLAG_ORIENT_SHIFT : 0);
        for (size_t z = 0; z < in_components(); z++) {
            zj_component &c = img->comp[z];
            c.coeff = plane_len[z] ? planes[z].p : nullptr;
            c.n_i16 = plane_len[z];
            memcpy(c.qt, components[z].quantization_table, sizeof(c.qt));
            c.h_samp = (uint32_t)components[z].horizontal_sample;
            c.v_samp = (uint32_t)components[z].vertical_sample;
            c.width_stride = (uint32_t)components[z].width_stride;
        }
    }
    void host_stage(const uint8_t *buf, size_t len, zj_image *img)  // decode_internal, decoder.rs:420-434
    {
        reset_state();
        Cursor cur{buf, len, 0};
        decode_headers_internal(cur);
        if (is_progressive) decode_progressive(cur);
        else decode_baseline(cur);
        fill_descriptor(img);
    }
    void set_error(const DecodeError &e)
    {
        err_kind = e.kind;
        err_msg = e.msg;
        switch (e.kind) {  // Display, errors.rs:77-113
        case ZJ_DE_FORMAT: err_display = e.msg; break;
        case ZJ_DE_FORMAT_STATIC: err_display = "\"" + e.msg + "\""; break;
        case ZJ_DE_HUFFMAN_DECODE: err_display = "Error decoding huffman tables.Reason:" + e.msg; break;
        case ZJ_DE_ZERO_ERROR: err_display = "Image width or height is set to zero, cannot continue"; break;
        case ZJ_DE_DQT_ERROR: err_display = "Error parsing DQT segment. Reason:" + e.msg; break;
        case ZJ_DE_SOS_ERROR: err_display = "Error parsing SOS Segment. Reason:" + e.msg; break;
        case ZJ_DE_SOF_ERROR: err_display = "Error parsing SOF segment. Reason:" + e.msg; break;
        case ZJ_DE_ILLEGAL_MAGIC_BYTES: err_display = "Error parsing image. Illegal start bytes:" + e.msg; break;
        case ZJ_DE_MCU_ERROR: err_display = "Error in decoding MCU. Reason " + e.msg; break;
        case ZJ_DE_EXHAUSTED_DATA: err_display = "Exhausted data in the image"; break;
        default: err_display = e.msg; break;
        }
    }
    void clear_error() { err_kind = ZJ_DE_NONE; err_msg.clear(); err_display.clear(); }
};

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

ZJ_API void zj_options_default(zj_options *o)  // ZuneJpegOptions::default, src/options.rs:23-39
{
    if (!o) return;
    o->use_unsafe = 1;
    o->out_colorspace = ZJ_CS_RGB;
    o->num_threads = 4;
    o->max_width = 1 << 14;
    o->max_height = 1 << 14;
    o->max_scans = 64;
    o->strict_mode = 0;
    o->device = 0;
}

ZJ_API zj_decoder *zj_decoder_new(const zj_options *o)
{
    zj_options opt;
    if (o) opt = *o; else zj_options_default(&opt);
    zj_decoder *d = new (std::nothrow) zj_decoder(opt);
    if (d) d->user_out_cs = opt.out_colorspace;
    return d;
}
ZJ_API void zj_decoder_free(zj_decoder *d) { delete d; }

ZJ_API int zj_decoder_read_headers(zj_decoder *d, const uint8_t *buf, size_t len)
{
    if (!d || (!buf && len)) return ZJ_ERR_INVALID_ARG;
    d->clear_error();
    try {
        d->reset_state();
        Cursor cur{buf, len, 0};
        d->decode_headers_internal(cur);
    } catch (DecodeError &e) { d->set_error(e); return ZJ_ERR_DECODE; }
    catch (const std::bad_alloc &) { return ZJ_ERR_OOM; }       // nothing may unwind through the C ABI
    catch (...) { return ZJ_ERR_DECODE; }
    return ZJ_OK;
}
ZJ_API int zj_decoder_info(const zj_decoder *d, zj_image_info *info)
{
    if (!d || !info) return ZJ_ERR_INVALID_ARG;
    *info = d->info;
    return ZJ_OK;
}
ZJ_API uint32_t zj_decoder_out_colorspace(const zj_decoder *d) { return d ? d->options.out_colorspace : 0; }
ZJ_API uint32_t zj_decoder_orientation(const zj_decoder *d) { return d ? d->orientation : 1; }

ZJ_API int zj_decoder_decode_coefficients(zj_decoder *d, const uint8_t *buf, size_t len, zj_image *img)
{
    if (!d || (!buf && len) || !img) return ZJ_ERR_INVALID_ARG;
    d->clear_error();
    try { d->host_stage(buf, len, img); } catch (DecodeError &e) { d->set_error(e); return ZJ_ERR_DECODE; }
    catch (const std::bad_alloc &) { return ZJ_ERR_OOM; }
    catch (...) { return ZJ_ERR_DECODE; }
    return ZJ_OK;
}

// Strip pipeline of ONE image (SURVEY 8(f).2, mcu.rs:230-369): finished strip ranges are uploaded, reconstructed and downloaded
// while the host is still entropy-decoding the rest of the same image.  Ranges are the virtual images of zj_image_strip_range,
// queued with zj_gpu_reconstruct_submit on the calling thread's cached streams; one finish per range at the end.
struct PipeSink : StripSink {
    int device = 0;
    uint8_t *out = nullptr;
    size_t out_cap = 0;
    zj_image img{};
    size_t n_strips = 0, step = 0, submitted = 0;
    std::vector<zj_pending *> pend;
    std::mutex mu;
    int rc = ZJ_OK;
    bool active = false;
    void begin(const zj_image &im, size_t ns) override
    {
        img = im;
        uint32_t plan_strips = 0;
        // only when the image plans, has as many strips as the host stage counts, and is worth cutting
        if (zj_image_strip_range(&img, 0, 0, nullptr, nullptr, nullptr, &plan_strips) != ZJ_OK || plan_strips != ns) return;
        zj_image whole;
        size_t off = 0, bytes = 0;
        if (zj_image_strip_range(&img, 0, (uint32_t)ns, &whole, &off, &bytes, nullptr) != ZJ_OK) return;   // cannot be cut
        if (zj_output_size(&img) == 0 || zj_output_size(&img) > out_cap) return;
        // a pageable destination makes every download a blocking, staged copy on the thread that queues it (2 GB/s): such
        // callers get the one-shot path, whose single download at least waits for nothing else
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, out) != cudaSuccess || at.type != cudaMemoryTypeHost) { cudaGetLastError(); return; }
        static const size_t ranges = [] { const char *e = getenv("ZJ_STRIP_RANGES"); long v = e ? atol(e) : 16; return (size_t)(v < 1 ? 1 : v); }();
        static const size_t min_px = [] { const char *e = getenv("ZJ_STRIP_PIPE_MIN_MP"); double v = e ? atof(e) : 4.0; return (size_t)(v * 1e6); }();
        if (ranges < 2 || (size_t)img.width * img.height < min_px || ns < 2 * ranges) return;
        n_strips = ns;
        step = (ns + ranges - 1) / ranges;
        active = true;
        t_begin = now_ms();
    }
    static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
    double t_begin = 0;
    void submit_range(size_t s0, size_t s1)
    {
        static const bool trace = getenv("ZJ_PIPE_TRACE") != nullptr;
        const double t0 = trace ? now_ms() : 0;
        zj_image sub;
        size_t off = 0, bytes = 0;
        int r = zj_image_strip_range(&img, (uint32_t)s0, (uint32_t)s1, &sub, &off, &bytes, nullptr);
        if (r == ZJ_OK && bytes) {
            uint8_t *o = out + off;
            zj_pending *pd = nullptr;
            r = zj_gpu_reconstruct_submit(device, nullptr, &sub, 1, &o, &bytes, &pd);
            if (r == ZJ_OK) pend.push_back(pd);
        }
        if (r != ZJ_OK && rc == ZJ_OK) rc = r;
        if (trace) fprintf(stderr, "[zj pipe] strips [%zu, %zu) queued at %.2f ms, submit took %.2f ms (rc %d)\n", s0, s1, t0 - t_begin, now_ms() - t0, r);
    }
    void progress(size_t done) override
    {
        if (!active) return;
        std::lock_guard<std::mutex> lock(mu);
        while (rc == ZJ_OK && submitted + step <= done && submitted + step < n_strips) {
            submit_range(submitted, submitted + step);
            submitted += step;
        }
    }
    int drain()
    {
        int r = rc;
        for (zj_pending *pd : pend) { const int f = zj_gpu_reconstruct_finish(pd); if (f != ZJ_OK && r == ZJ_OK) r = f; }
        pend.clear();
        return r;
    }
    void restart() override
    {
        if (!active) return;
        std::lock_guard<std::mutex> lock(mu);
        drain();            // (copies of the first attempt may still be reading the planes)
        rc = ZJ_OK;
        submitted = 0;
    }
    // the entropy stage is done: the remaining strips (and the rows below them), then wait for everything
    int finish()
    {
        std::lock_guard<std::mutex> lock(mu);
        if (rc == ZJ_OK) submit_range(submitted, n_strips);
        submitted = n_strips;
        const int r = drain();
        if (getenv("ZJ_PIPE_TRACE")) fprintf(stderr, "[zj pipe] drained at %.2f ms\n", now_ms() - t_begin);
        return r;
    }
    ~PipeSink() override { drain(); }
};

// decode_into of later zune-jpeg releases (BASELINE north_star names `decode()/decode_into()`): the pixels go into the caller's
// buffer (pinned memory makes every copy asynchronous).  Baseline images of some size run the strip pipeline above.
ZJ_API int zj_decoder_decode_into(zj_decoder *d, const uint8_t *buf, size_t len, uint8_t *out, size_t out_cap, size_t *out_len)
{
    if (!d || (!buf && len) || !out || !out_len) return ZJ_ERR_INVALID_ARG;
    *out_len = 0;
    PipeSink ps;
    ps.device = d->options.device;
    ps.out = out;
    ps.out_cap = out_cap;
    zj_image img;
    d->sink = d->have_device ? &ps : nullptr;
    const bool trace = getenv("ZJ_PIPE_TRACE") != nullptr;
    const double t_call = trace ? PipeSink::now_ms() : 0;
    int rc = zj_decoder_decode_coefficients(d, buf, len, &img);
    d->sink = nullptr;
    if (trace) fprintf(stderr, "[zj pipe] host stage returned after %.2f ms (begin was at +%.2f ms)\n", PipeSink::now_ms() - t_call, ps.t_begin - t_call);
    if (rc) return rc;          // (~PipeSink waits for whatever was queued)
    const size_t n = zj_output_size(&img);
    rc = zj_validate_image(&img);
    if (rc == ZJ_OK && n == 0) rc = ZJ_ERR_INVALID_ARG;
    if (rc == ZJ_OK && n > out_cap) rc = ZJ_ERR_SHORT_OUTPUT;
    if (rc == ZJ_OK) rc = ps.active ? ps.finish() : zj_gpu_reconstruct(d->options.device, nullptr, &img, 1, &out, &n);
    if (rc != ZJ_OK) {
        std::string m = zj_gpu_strerror(rc);
        if (rc == ZJ_ERR_CUDA || rc == ZJ_ERR_OOM) m += std::string(" -- ") + zj_gpu_last_cuda_error();
        d->set_error(DecodeError{rc == ZJ_ERR_UNSUPPORTED ? ZJ_DE_FORMAT : ZJ_DE_GPU, m});
        return rc;
    }
    *out_len = n;
    return ZJ_OK;
}

ZJ_API int zj_decoder_decode_buffer(zj_decoder *d, const uint8_t *buf, size_t len, uint8_t **out, size_t *out_len)
{
    if (!d || (!buf && len) || !out || !out_len) return ZJ_ERR_INVALID_ARG;
    *out = nullptr;
    *out_len = 0;
    // the size comes from the headers (mcu.rs:375-379: width * height * out components); they are parsed again by the decode
    int rc = zj_decoder_read_headers(d, buf, len);
    if (rc) return rc;
    const size_t cap = (size_t)d->info.width * d->info.height * zj::num_components(d->options.out_colorspace);
    uint8_t *o = (uint8_t *)malloc(cap ? cap : 1);
    if (!o) return ZJ_ERR_OOM;
    size_t n = 0;
    rc = zj_decoder_decode_into(d, buf, len, o, cap, &n);
    if (rc != ZJ_OK) { free(o); return rc; }
    *out = o;
    *out_len = n;
    return ZJ_OK;
}
ZJ_API void zj_buffer_free(uint8_t *p) { free(p); }

// decoders (with their pinned coefficient planes) kept between zj_decode_batch calls; zj_release_host_caches frees them
static std::mutex g_idle_mu;
static std::vector<zj_decoder *> g_idle;
ZJ_API void zj_release_host_caches(void)
{
    std::vector<zj_decoder *> drop;
    {
        std::lock_guard<std::mutex> lock(g_idle_mu);
        drop.swap(g_idle);
    }
    for (zj_decoder *d : drop) zj_decoder_free(d);
}

// Batch front door.  The reference decodes one image per Decoder and parallelises the strips of that image
// (scoped_threadpool, mcu.rs:230-369); with the pixel path on the GPU the host threads are free to run the branchy
// stage of DIFFERENT images side by side: every worker owns a decoder (its pinned coefficient planes are reused from
// image to image), entropy-decodes one image, hands the planes to zj_gpu_reconstruct on its own streams and moves on,
// so the Huffman stage of some images overlaps transfer and reconstruction of others.
// DecodeErrors of the images of the last batch call of this thread (zj_batch_error_kind / zj_batch_error): the batch front
// doors report a per-image zj_status; the variant and Display text the reference's Decoder would have returned live here.
struct BatchErr { int kind = ZJ_DE_NONE; std::string msg; };
static thread_local std::vector<BatchErr> t_batch_err;
static void note_gpu_error(BatchErr *e, int rc)
{
    if (!e || rc == ZJ_OK) return;
    e->kind = rc == ZJ_ERR_UNSUPPORTED ? ZJ_DE_FORMAT : ZJ_DE_GPU;
    e->msg = zj_gpu_strerror(rc);
}
static int decode_batch_impl(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                             uint8_t **out, size_t *out_len, int *status, BatchErr *errs);

ZJ_API int zj_decode_batch(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                           uint8_t **out, size_t *out_len, int *status)
{
    try { t_batch_err.assign(n, BatchErr{}); } catch (...) { return ZJ_ERR_OOM; }
    return decode_batch_impl(o, bufs, lens, n, out, out_len, status, t_batch_err.data());
}
ZJ_API int zj_batch_error_kind(size_t i) { return i < t_batch_err.size() ? t_batch_err[i].kind : (int)ZJ_DE_NONE; }
ZJ_API const char *zj_batch_error(size_t i) { return i < t_batch_err.size() ? t_batch_err[i].msg.c_str() : ""; }

static int decode_batch_impl(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                             uint8_t **out, size_t *out_len, int *status, BatchErr *errs)
{
    if ((!bufs || !lens || !out || !out_len || !status) && n) return ZJ_ERR_INVALID_ARG;
    zj_options opt;
    if (o) opt = *o; else zj_options_default(&opt);
    size_t nthreads = opt.num_threads ? opt.num_threads : std::thread::hardware_concurrency();
    if (nthreads == 0) nthreads = 1;
    const size_t per_image_threads = n ? std::max<size_t>(1, nthreads / n) : 1;
    if (nthreads > n) nthreads = n;
    std::atomic<size_t> next{0};
    std::atomic<int> failed{0};
    // decoders (with their pinned coefficient planes) are kept between calls: page-locking and releasing 25 MB per
    // image and thread costs more than decoding it, and both serialise in the driver
    std::mutex &idle_mu = g_idle_mu;
    std::vector<zj_decoder *> &idle = g_idle;
    auto take_decoder = [&]() -> zj_decoder * {
        zj_decoder *d = nullptr;
        {
            std::lock_guard<std::mutex> lock(idle_mu);
            if (!idle.empty()) { d = idle.back(); idle.pop_back(); }
        }
        if (d) { d->options = opt; d->user_out_cs = opt.out_colorspace; d->clear_error(); }
        else d = zj_decoder_new(&opt);
        if (d) d->entropy_threads = per_image_threads;   // the host threads left over when there are fewer images than threads
        return d;
    };
    auto give_back = [&](zj_decoder *d) {
        if (!d) return;
        {
            std::lock_guard<std::mutex> lock(idle_mu);
            if (idle.size() < 512) { idle.push_back(d); return; }
        }
        zj_decoder_free(d);
    };
    // A worker alternates between two decoders (two sets of pinned planes): while the GPU uploads, reconstructs and
    // downloads image i from the planes of one, the thread entropy-decodes its next image into the planes of the other.
    auto worker = [&]() {
        zj_decoder *dec[2] = {take_decoder(), nullptr};
        struct InFlight { zj_pending *pd = nullptr; size_t i = 0; uint8_t *dst = nullptr; size_t need = 0; bool mine = false; } fl;
        auto settle = [&]() {   // wait for the image in flight and publish its result
            if (!fl.pd) return;
            const int rc = zj_gpu_reconstruct_finish(fl.pd);
            fl.pd = nullptr;
            if (rc == ZJ_OK) { out[fl.i] = fl.dst; out_len[fl.i] = fl.need; }
            else { if (fl.mine) free(fl.dst); if (fl.mine || !out[fl.i]) out[fl.i] = nullptr; out_len[fl.i] = 0; failed++; note_gpu_error(errs ? errs + fl.i : nullptr, rc); }
            status[fl.i] = rc;
        };
        int cur = 0;
        for (;;) {
            const size_t i = next.fetch_add(1);
            if (i >= n) break;
            if (!dec[cur]) dec[cur] = take_decoder();
            zj_decoder *d = dec[cur];
            if (!d) { status[i] = ZJ_ERR_OOM; out_len[i] = 0; failed++; note_gpu_error(errs ? errs + i : nullptr, ZJ_ERR_OOM); continue; }
            zj_image img;
            int rc = (!bufs[i] && lens[i]) ? ZJ_ERR_INVALID_ARG : zj_decoder_decode_coefficients(d, bufs[i], lens[i], &img);
            if (rc == ZJ_ERR_DECODE && errs) { errs[i].kind = d->err_kind; errs[i].msg = d->err_display; }   // the reference's DecodeErrors
            size_t need = 0;
            if (rc == ZJ_OK) {
                need = zj_output_size(&img);
                rc = zj_validate_image(&img);
                if (rc == ZJ_OK && need == 0) rc = ZJ_ERR_INVALID_ARG;
            }
            uint8_t *dst = out[i];
            bool mine = false;
            if (rc == ZJ_OK) {
                if (dst) { if (out_len[i] < need) rc = ZJ_ERR_SHORT_OUTPUT; }
                else { dst = (uint8_t *)malloc(need); mine = true; if (!dst) rc = ZJ_ERR_OOM; }
            }
            settle();   // the previous image (its planes are the ones this thread decodes into next)
            zj_pending *pd = nullptr;
            if (rc == ZJ_OK) rc = zj_gpu_reconstruct_submit(opt.device, nullptr, &img, 1, &dst, &need, &pd);
            if (rc == ZJ_OK) {
                fl.pd = pd; fl.i = i; fl.dst = dst; fl.need = need; fl.mine = mine;
                cur ^= 1;
            } else {
                if (mine) free(dst);
                if (mine || !out[i]) out[i] = nullptr;
                out_len[i] = 0;
                failed++;
                status[i] = rc;
                if (rc != ZJ_ERR_DECODE) note_gpu_error(errs ? errs + i : nullptr, rc);
            }
        }
        settle();
        give_back(dec[0]);
        give_back(dec[1]);
    };
    std::vector<std::thread> pool;
    for (size_t t = 1; t < nthreads; t++) if (!spawn(pool, worker)) break;
    if (n) worker();
    for (auto &t : pool) t.join();
    return failed.load();
}
// zj_decode_batch over several devices (contiguous image ranges, no exchange between devices; DESIGN.md section 6)
ZJ_API int zj_decode_batch_multi(const zj_options *o, const int *devices, size_t n_dev, const uint8_t *const *bufs,
                                 const size_t *lens, size_t n, uint8_t **out, size_t *out_len, int *status)
{
    if (!devices || n_dev == 0 || ((!bufs || !lens || !out || !out_len || !status) && n)) return ZJ_ERR_INVALID_ARG;
    zj_options opt;
    if (o) opt = *o; else zj_options_default(&opt);
    size_t nthreads = opt.num_threads ? opt.num_threads : std::thread::hardware_concurrency();
    if (nthreads == 0) nthreads = 1;
    if (n >= n_dev) {
        std::vector<int> rcs(n_dev, 0);
        auto run = [&](size_t k) {
            size_t lo, hi;
            zj_partition(n, n_dev, k, &lo, &hi);
            if (lo == hi) return;
            zj_options ok = opt;
            ok.device = devices[k];
            ok.num_threads = (uint32_t)std::max<size_t>(1, nthreads / n_dev);
            cudaSetDevice(devices[k]);
            rcs[k] = zj_decode_batch(&ok, bufs + lo, lens + lo, hi - lo, out + lo, out_len + lo, status + lo);
        };
        std::vector<std::thread> pool;
        for (size_t k = 1; k < n_dev; k++) {
            try { pool.emplace_back(run, k); } catch (...) { run(k); }
        }
        run(0);
        for (auto &t : pool) t.join();
        int failed = 0;
        for (int rc : rcs) { if (rc < 0) return rc; failed += rc; }
        return failed;
    }
    // fewer images than devices: one image at a time, all host threads on its restart intervals, its strips over the devices
    int failed = 0;
    opt.num_threads = (uint32_t)nthreads;
    opt.device = devices[0];
    for (size_t i = 0; i < n; i++) {
        zj_decoder *d = zj_decoder_new(&opt);
        zj_image img;
        int rc = !d ? (int)ZJ_ERR_OOM : ((!bufs[i] && lens[i]) ? (int)ZJ_ERR_INVALID_ARG : zj_decoder_decode_coefficients(d, bufs[i], lens[i], &img));
        size_t need = 0;
        if (rc == ZJ_OK) { need = zj_output_size(&img); rc = zj_validate_image(&img); if (rc == ZJ_OK && need == 0) rc = ZJ_ERR_INVALID_ARG; }
        uint8_t *dst = out[i];
        bool mine = false;
        if (rc == ZJ_OK) {
            if (dst) { if (out_len[i] < need) rc = ZJ_ERR_SHORT_OUTPUT; }
            else { dst = (uint8_t *)malloc(need); mine = true; if (!dst) rc = ZJ_ERR_OOM; }
        }
        if (rc == ZJ_OK) rc = zj_gpu_reconstruct_multi(devices, n_dev, &img, 1, &dst, &need);
        if (rc == ZJ_OK) { out[i] = dst; out_len[i] = need; }
        else { if (mine) free(dst); if (mine || !out[i]) out[i] = nullptr; out_len[i] = 0; failed++; }
        status[i] = rc;
        if (d) zj_decoder_free(d);
    }
    return failed;
}

// ---- state zj_decode_batch_gpu[_device] keeps between calls: two slots of device staging memory (at least 1 GB each once
// used, grown to the sub-batch budget), their streams and pinned descriptor / status blocks.  zj_release_device_caches frees
// them; a buffer larger than ZJ_RETAIN_MB (default 16384: never, in practice) is freed when the call that grew it ends.
struct GpuSlot {
    cudaStream_t s = nullptr; uint8_t *mem = nullptr; size_t cap = 0;
    std::vector<zj_batch *> batches;          // reconstruction launch plans whose kernels may still be running
    std::vector<size_t> take, idx;            // images of the sub-batch in stage 1 / images whose pixels are on their way
    std::vector<zj::EntImage> eimg;
    std::vector<uint8_t *> pix;
    std::vector<size_t> st_off;
    uint8_t *meta_host = nullptr, *st_host = nullptr;   // pinned: descriptors + tables + interval starts up, statuses down
    size_t meta_cap = 0, st_cap = 0;
    bool staged = false;
    void release()      // stream, device staging memory and the pinned descriptor / status blocks
    {
        if (mem) cudaFree(mem);
        if (s) cudaStreamDestroy(s);
        if (meta_host) cudaFreeHost(meta_host);
        if (st_host) cudaFreeHost(st_host);
        *this = GpuSlot{};
    }
};
struct GpuSlotCache { GpuSlot slot[2]; int device = -1; };
static std::mutex g_slot_mu;
static GpuSlotCache g_slot_cache;
static size_t slot_retain_bytes()
{
    // (default 16 GB: above any sub-batch budget, i.e. the slots are kept until zj_release_device_caches.  Re-allocating a
    // 6.7 GB slot was measured at up to 119 ms per call -- four times the call itself)
    static const size_t v = [] { const char *e = getenv("ZJ_RETAIN_MB"); long mb = e ? atol(e) : 16384; return (size_t)(mb < 0 ? 0 : mb) << 20; }();
    return v;
}
ZJ_API void zj_release_device_caches(void)
{
    {
        std::lock_guard<std::mutex> lock(g_slot_mu);     // (waits for a zj_decode_batch_gpu call in flight)
        if (g_slot_cache.device >= 0 && cudaSetDevice(g_slot_cache.device) == cudaSuccess)
            for (auto &sl : g_slot_cache.slot) sl.release();
        g_slot_cache.device = -1;
        cudaGetLastError();
    }
    zj::release_stream_caches();
    zj::trim_pools();
}

// Batch front door with the entropy stage on the GPU as well (zj_entropy.cu) for the JPEGs that allow it: baseline scans
// with restart markers whose every interval ends the way the reference's sequential loop ends it.  Those upload their FILE
// (not their coefficient planes: 12 MB instead of 201 MB for an 8192x8192 image), are entropy-decoded one restart interval per
// GPU thread into device planes, reconstructed in place and downloaded.  Every other image -- no DRI, progressive, a header
// error, one interval that ends differently -- goes through zj_decode_batch (host stage), so results and errors are the
// same as there.
static int decode_batch_gpu_impl(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                                 uint8_t **out, size_t *out_len, int *status, size_t *n_gpu_entropy, const bool dev_out)
{
    if (n_gpu_entropy) *n_gpu_entropy = 0;
    if ((!bufs || !lens || !out || !out_len || !status) && n) return ZJ_ERR_INVALID_ARG;
    zj_options opt;
    if (o) opt = *o; else zj_options_default(&opt);
    size_t nthreads = opt.num_threads ? opt.num_threads : std::thread::hardware_concurrency();
    if (nthreads == 0) nthreads = 1;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= opt.device) {
        cudaGetLastError();
        return dev_out ? (int)ZJ_ERR_NO_DEVICE : zj_decode_batch(o, bufs, lens, n, out, out_len, status);
    }

    const bool trace = getenv("ZJ_GPU_ENTROPY_TRACE") != nullptr;   // phase times on stderr (adds synchronisation)
    auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_mark = now();
    auto lap = [&](const char *what, cudaStream_t s) {
        if (!trace) return;
        if (s) cudaStreamSynchronize(s);
        const double t = now();
        fprintf(stderr, "[zj_decode_batch_gpu] %-28s %8.2f ms\n", what, t - t_mark);
        t_mark = t;
    };
    // ---- headers + restart-marker scan of every image on the host threads
    struct Item { zj_decoder *d = nullptr; zj_decoder::GpuPrep pp; bool gpu = false; size_t need = 0; zj_image img; };
    std::vector<Item> items(n);
    {
        std::atomic<size_t> next{0};
        auto work = [&]() {
            for (size_t i; (i = next.fetch_add(1)) < n;) {
                Item &it = items[i];
                if (!bufs[i] || lens[i] == 0) continue;
                it.d = zj_decoder_new(&opt);
                if (!it.d) continue;
                try {
                    it.d->reset_state();
                    Cursor cur{bufs[i], lens[i], 0};
                    it.d->decode_headers_internal(cur);
                    it.gpu = it.d->gpu_entropy_prepare(cur, it.pp);
                    if (it.gpu) {
                        it.d->fill_descriptor(&it.img);
                        it.need = zj_output_size(&it.img);
                        if (it.need == 0 || (out[i] && out_len[i] < it.need) || (dev_out && !out[i])) it.gpu = false;   // the host path reports it
                        for (uint32_t z = 0; z < it.img.n_comp; z++) it.img.comp[z].coeff = it.img.comp[z].n_i16 ? (const int16_t *)16 : nullptr;
                        if (it.gpu && zj_validate_image(&it.img) != ZJ_OK) it.gpu = false;
                    }
                } catch (DecodeError &) { it.gpu = false; }
            }
        };
        std::vector<std::thread> pool;
        for (size_t t = 1; t < std::min(nthreads, n); t++) if (!spawn(pool, work)) break;
        if (n) work();
        for (auto &t : pool) t.join();
    }

    lap("headers + marker scan", nullptr);
    std::vector<BatchErr> batch_errs(n);
    // ---- the host route (zj_decode_batch) for a list of images.  Those that cannot use the GPU entropy stage at all (no DRI,
    // progressive, header errors) start on it right away, on the host threads, while the GPU works on the others.
    auto run_host = [&](const std::vector<size_t> &rest) -> int {
        if (rest.empty()) return 0;
        std::vector<const uint8_t *> b2(rest.size());
        std::vector<size_t> l2(rest.size()), ol2(rest.size());
        std::vector<uint8_t *> o2(rest.size());
        std::vector<int> s2(rest.size(), 0);
        for (size_t t = 0; t < rest.size(); t++) {
            b2[t] = bufs[rest[t]]; l2[t] = lens[rest[t]];
            o2[t] = dev_out ? nullptr : out[rest[t]];          // device outputs: decoded into host memory first, then uploaded
            ol2[t] = dev_out ? 0 : out_len[rest[t]];
        }
        std::vector<BatchErr> e2(rest.size());
        int f = decode_batch_impl(&opt, b2.data(), l2.data(), rest.size(), o2.data(), ol2.data(), s2.data(), e2.data());
        if (f < 0) return f;
        for (size_t t = 0; t < rest.size(); t++) {
            const size_t i = rest[t];
            batch_errs[i] = e2[t];
            if (!dev_out) { out[i] = o2[t]; out_len[i] = ol2[t]; status[i] = s2[t]; continue; }
            int rc = s2[t];
            if (rc == ZJ_OK) {
                if (!out[i]) rc = ZJ_ERR_INVALID_ARG;
                else if (out_len[i] < ol2[t]) rc = ZJ_ERR_SHORT_OUTPUT;
                else if (cudaMemcpy(out[i], o2[t], ol2[t], cudaMemcpyHostToDevice) != cudaSuccess) { cudaGetLastError(); rc = ZJ_ERR_CUDA; }
                if (rc != ZJ_OK) f++;
            }
            free(o2[t]);
            out_len[i] = rc == ZJ_OK ? ol2[t] : 0;
            status[i] = rc;
        }
        return f;
    };
    std::vector<char> is_early(n, 0);
    std::vector<size_t> early_list;
    for (size_t i = 0; i < n; i++) if (!items[i].gpu) { is_early[i] = 1; early_list.push_back(i); }
    int early_rc = 0;
    std::thread early;
    if (!early_list.empty()) {
        try { early = std::thread([&]() { cudaSetDevice(opt.device); early_rc = run_host(early_list); }); }
        catch (...) { early_rc = run_host(early_list); }      // no thread to be had: do it here, before the GPU phase
    }
    // ---- GPU: sub-batches of as many images as fit the staging budget, two slots in flight.  Stage 1 of sub-batch b (upload,
    // clear the planes, entropy kernel, status download) is queued before the host waits for the statuses of sub-batch b-1 and
    // queues its stage 2 (reconstruction, pixel download), so the two streams keep the GPU and both PCIe directions busy.
    std::vector<char> on_gpu(n, 0);
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    auto footprint = [&](const Item &it, size_t len) {
        size_t b = al(len + 8) + al(sizeof(zj::EntImage)) + al(6 * sizeof(zj::EntTable)) + al((it.pp.n_seg + 1) * 4) + al(it.pp.n_seg) + 1024 + (dev_out ? 0 : al(it.need));
        for (int z = 0; z < 3; z++) b += al(it.d->plane_len[z] * 2);
        return b;
    };
    const char *env_mb = getenv("ZJ_GPU_ENTROPY_BUDGET_MB");
    const size_t budget = (size_t)(env_mb ? std::max(64, atoi(env_mb)) : (dev_out ? 8192 : 4096)) << 20;   // host outputs: smaller sub-batches, so that the download of one overlaps the kernels of the next (2 GB and 8 GB measured slower)
    auto pinned_grow = [](uint8_t *&p, size_t &cap, size_t need) -> bool {
        if (cap >= need) return true;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        const size_t want = need + need / 2 + 4096;
        if (cudaHostAlloc((void **)&p, want, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); p = nullptr; return false; }
        cap = want;
        return true;
    };
    // the two slots' streams and device memory are kept between calls (allocating and freeing gigabytes costs 3-13 ms per
    // call and synchronises the device); one call at a time uses them, a concurrent call works with slots of its own
    GpuSlotCache own;
    std::unique_lock<std::mutex> cache_lock(g_slot_mu, std::try_to_lock);
    GpuSlotCache &sc = cache_lock.owns_lock() ? g_slot_cache : own;
    bool cuda_ok = cudaSetDevice(opt.device) == cudaSuccess;
    if (cuda_ok && sc.device != opt.device) {
        for (auto &sl : sc.slot) sl.release();
        sc.device = opt.device;
    }
    GpuSlot *slot = sc.slot;
    for (int k = 0; k < 2 && cuda_ok; k++)
        if (!slot[k].s) cuda_ok = cudaStreamCreateWithFlags(&slot[k].s, cudaStreamNonBlocking) == cudaSuccess;
    std::vector<uint8_t *> malloced(n, nullptr);
    auto drain = [&](GpuSlot &sl) {   // wait for the slot's downloads, publish its images
        if (sl.idx.empty() && sl.batches.empty()) return;
        const bool ok = cudaStreamSynchronize(sl.s) == cudaSuccess;
        if (!ok) cudaGetLastError();
        for (zj_batch *b : sl.batches) zj_batch_destroy(b);
        sl.batches.clear();
        for (size_t i : sl.idx) if (on_gpu[i] == 1) on_gpu[i] = ok ? 2 : 0;
        sl.idx.clear();
    };
    size_t i0 = 0;
    // stage 1: false when there is nothing (left) to queue
    auto stage1 = [&](GpuSlot &sl) -> bool {
        sl.staged = false;
        sl.take.clear();
        size_t bytes = 0, i1 = i0;
        while (i1 < n) {
            const Item &it = items[i1];
            if (it.gpu) {
                const size_t f = footprint(it, lens[i1]);
                if (!sl.take.empty() && bytes + f > budget) break;
                bytes += f;
                sl.take.push_back(i1);
            }
            i1++;
        }
        i0 = i1;
        if (sl.take.empty()) return false;
        if (sl.cap < bytes) {
            if (sl.mem) cudaFree(sl.mem);
            sl.mem = nullptr; sl.cap = 0;
            // (a first small batch reserves 1 GB so that the next ones need no new allocation)
            size_t want = std::max(bytes, std::min(budget, (size_t)1 << 30));
            if (cudaMalloc((void **)&sl.mem, want) != cudaSuccess) {
                cudaGetLastError();
                want = bytes;
                if (cudaMalloc((void **)&sl.mem, want) != cudaSuccess) { cudaGetLastError(); sl.mem = nullptr; sl.take.clear(); return true; }   // host path
            }
            sl.cap = want;
        }
        lap("take + cudaMalloc", nullptr);
        const std::vector<size_t> &take = sl.take;
        size_t off = 0;
        auto carve = [&](size_t nb) { uint8_t *p = sl.mem + off; off += al(nb); return p; };
        // planes of the whole sub-batch first, contiguous: one memset
        sl.eimg.assign(take.size(), zj::EntImage{});
        for (size_t t = 0; t < take.size(); t++) {
            const Item &it = items[take[t]];
            for (int z = 0; z < 3; z++) sl.eimg[t].plane[z] = it.d->plane_len[z] ? (int16_t *)carve(it.d->plane_len[z] * 2) : nullptr;
        }
        bool ok = cudaMemsetAsync(sl.mem, 0, off, sl.s) == cudaSuccess;
        lap("memset planes", sl.s);
        // descriptors, Huffman tables and interval starts of the sub-batch travel as ONE pinned block, the statuses come back as one
        sl.pix.assign(take.size(), nullptr);
        sl.st_off.assign(take.size(), 0);
        size_t st_total = 0, seg_words = 0;
        for (size_t t = 0; t < take.size(); t++) { sl.st_off[t] = st_total; st_total += items[take[t]].pp.n_seg; seg_words += items[take[t]].pp.n_seg + 1; }
        const size_t off_tab = al(take.size() * sizeof(zj::EntImage)), off_seg = off_tab + al(6 * take.size() * sizeof(zj::EntTable));
        const size_t meta_bytes = off_seg + al(seg_words * 4);
        ok = ok && pinned_grow(sl.meta_host, sl.meta_cap, meta_bytes) && pinned_grow(sl.st_host, sl.st_cap, st_total);
        uint8_t *d_meta = carve(meta_bytes), *d_status = carve(st_total);
        uint32_t max_seg = 0;
        size_t seg_at = 0;
        for (size_t t = 0; t < take.size() && ok; t++) {
            const size_t i = take[t];
            Item &it = items[i];
            zj::EntImage &e = sl.eimg[t];
            const zj_decoder::BaselineGeom &g = it.pp.g;
            uint8_t *d_data = carve(lens[i] + 8);
            it.d->gpu_entropy_tables(reinterpret_cast<zj::EntTable *>(sl.meta_host + off_tab) + 6 * t);
            memcpy(sl.meta_host + off_seg + seg_at * 4, it.pp.seg_start.data(), (it.pp.n_seg + 1) * 4);
            sl.pix[t] = dev_out ? out[i] : carve(it.need);
            e.data = d_data; e.len = (uint32_t)lens[i];
            e.seg_start = reinterpret_cast<const uint32_t *>(d_meta + off_seg) + seg_at;
            e.status = d_status + sl.st_off[t];
            e.tables = reinterpret_cast<const zj::EntTable *>(d_meta + off_tab) + 6 * t;
            seg_at += it.pp.n_seg + 1;
            e.n_seg = (uint32_t)it.pp.n_seg; e.per_seg = (uint32_t)it.d->restart_interval; e.total_mcus = (uint32_t)it.pp.total;
            e.restart_interval = (uint32_t)it.d->restart_interval;
            e.mcu_w = (uint32_t)g.mcu_w; e.bias = (uint32_t)g.bias; e.ncomp = (uint32_t)g.ncomp; e.is_hv = g.is_hv ? 1u : 0u;
            e.width_stride = (uint32_t)g.width_stride; e.hv_width_stride = (uint32_t)g.hv_width_stride;
            for (int z = 0; z < 3; z++) {
                e.strip_len[z] = (uint32_t)g.strip_len[z];
                const bool have = (size_t)z < g.ncomp;
                e.h_samp[z] = have ? (uint32_t)it.d->components[z].horizontal_sample : 0u;
                e.v_samp[z] = have ? (uint32_t)it.d->components[z].vertical_sample : 0u;
                e.is_y[z] = have && it.d->components[z].component_id == ID_Y ? 1u : 0u;
            }
            max_seg = std::max(max_seg, e.n_seg);
        }
        if (ok) memcpy(sl.meta_host, sl.eimg.data(), take.size() * sizeof(zj::EntImage));
        ok = ok && off <= sl.cap && cudaMemcpyAsync(d_meta, sl.meta_host, meta_bytes, cudaMemcpyHostToDevice, sl.s) == cudaSuccess;
        // files + entropy kernel (behind the cleared planes and the descriptors), then the statuses come back
        for (size_t t = 0; t < take.size() && ok; t++)
            ok = cudaMemcpyAsync(const_cast<uint8_t *>(sl.eimg[t].data), bufs[take[t]], lens[take[t]], cudaMemcpyHostToDevice, sl.s) == cudaSuccess;
        ok = ok && zj::launch_entropy(reinterpret_cast<const zj::EntImage *>(d_meta), (uint32_t)take.size(), max_seg, sl.s) == 0;
        ok = ok && (st_total == 0 || cudaMemcpyAsync(sl.st_host, d_status, st_total, cudaMemcpyDeviceToHost, sl.s) == cudaSuccess);
        lap("files + entropy kernels", sl.s);
        if (!ok) cudaGetLastError();
        sl.staged = ok;   // (not staged: nothing is published, these images go through the host path)
        return true;
    };
    // stage 2: the statuses are in; accepted images are reconstructed from their device planes and downloaded
    auto stage2 = [&](GpuSlot &sl) {
        if (!sl.staged) return;
        sl.staged = false;
        if (cudaStreamSynchronize(sl.s) != cudaSuccess) { cudaGetLastError(); return; }
        std::vector<zj_image> dimgs;
        std::vector<uint8_t *> douts;
        std::vector<size_t> dlens, who;
        for (size_t t = 0; t < sl.take.size(); t++) {
            const size_t i = sl.take[t];
            Item &it = items[i];
            bool all = true;
            for (size_t k = 0; k < it.pp.n_seg; k++) all = all && sl.st_host[sl.st_off[t] + k] == 0;
            if (!all) continue;
            zj_image di = it.img;
            for (uint32_t z = 0; z < di.n_comp; z++) di.comp[z].coeff = sl.eimg[t].plane[z];
            dimgs.push_back(di); douts.push_back(sl.pix[t]); dlens.push_back(it.need); who.push_back(i);
        }
        if (dimgs.empty()) return;
        zj_batch *b = nullptr;
        int rc = zj_batch_create(opt.device, dimgs.data(), dimgs.size(), douts.data(), dlens.data(), &b);
        if (rc == ZJ_OK) { sl.batches.push_back(b); rc = zj_batch_run(b, sl.s); }
        for (size_t t = 0; t < who.size() && rc == ZJ_OK; t++) {
            const size_t i = who[t];
            if (!dev_out) {
                uint8_t *dst = out[i];
                if (!dst) { dst = (uint8_t *)malloc(items[i].need); malloced[i] = dst; }
                if (!dst) continue;
                if (cudaMemcpyAsync(dst, douts[t], dlens[t], cudaMemcpyDeviceToHost, sl.s) != cudaSuccess) { cudaGetLastError(); continue; }
            }
            on_gpu[i] = 1;
            sl.idx.push_back(i);
        }
        lap("status + reconstruct (+ d2h)", trace ? sl.s : nullptr);
    };
    if (cuda_ok) {
        int cur = 0;
        bool more = true;
        while (more) {
            GpuSlot &sl = slot[cur];
            drain(sl);
            more = stage1(sl);
            stage2(slot[cur ^ 1]);   // (measured: queueing it before stage 1 instead is no faster, and slower with small sub-batches)
            cur ^= 1;
        }
        stage2(slot[0]);
        stage2(slot[1]);
    }
    for (int k = 0; k < 2; k++) {
        drain(slot[k]);
        slot[k].take.clear();
        if (&sc == &own) slot[k].release();
        else if (slot[k].cap > slot_retain_bytes()) {      // a buffer that grew past the retention cap goes back to the driver
            cudaFree(slot[k].mem);
            slot[k].mem = nullptr; slot[k].cap = 0;
        }
    }
    if (cache_lock.owns_lock()) cache_lock.unlock();
    size_t n_gpu = 0;
    int failed = 0;
    std::vector<size_t> rest;
    for (size_t i = 0; i < n; i++) {
        if (items[i].d) { zj_decoder_free(items[i].d); items[i].d = nullptr; }
        if (on_gpu[i] == 2) {
            n_gpu++;
            status[i] = ZJ_OK;
            if (malloced[i]) out[i] = malloced[i];
            out_len[i] = items[i].need;
        } else {
            if (malloced[i]) { free(malloced[i]); malloced[i] = nullptr; }
            if (!is_early[i]) rest.push_back(i);
        }
    }
    if (n_gpu_entropy) *n_gpu_entropy = n_gpu;
    // ---- the images the GPU turned down: the host stage
    if (early.joinable()) early.join();
    if (early_rc < 0) return early_rc;
    failed += early_rc;
    const int late_rc = run_host(rest);
    if (late_rc < 0) return late_rc;
    failed += late_rc;
    for (size_t i = 0; i < n; i++) if (status[i] != ZJ_OK && batch_errs[i].kind == ZJ_DE_NONE) note_gpu_error(&batch_errs[i], status[i]);
    t_batch_err.swap(batch_errs);
    return failed;
}

ZJ_API int zj_decode_batch_gpu(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                               uint8_t **out, size_t *out_len, int *status, size_t *n_gpu_entropy)
{
    return decode_batch_gpu_impl(o, bufs, lens, n, out, out_len, status, n_gpu_entropy, false);
}
ZJ_API int zj_decode_batch_gpu_device(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                                      uint8_t *const *out_dev, size_t *out_len, int *status, size_t *n_gpu_entropy)
{
    return decode_batch_gpu_impl(o, bufs, lens, n, const_cast<uint8_t **>(out_dev), out_len, status, n_gpu_entropy, true);
}

// The first pass of the device-output calls with a second pass: every image decoded into a stream-ordered u8 scratch buffer
// (zj_decode_batch_gpu_device), then second_pass(img, failed) over img[i] = image i's geometry and pixels.  second_pass checks
// each decoded image, counts the images it turns down in `failed`, queues its launches and returns their status.  Returns
// zj_decode_batch's result with those images added, or a negative zj_status; the pixels are in place on return.
static int decode_then(const zj_options &opt, const uint8_t *const *bufs, const size_t *lens, size_t n, int *status, size_t *n_gpu_entropy,
                       const std::function<int(std::vector<zj::U8Image> &, int &)> &second_pass)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= opt.device) { cudaGetLastError(); return ZJ_ERR_NO_DEVICE; }
    if (cudaSetDevice(opt.device) != cudaSuccess) { cudaGetLastError(); return ZJ_ERR_NO_DEVICE; }
    // geometry of every image from its headers: the u8 intermediate is sized before decoding
    std::vector<zj::U8Image> img(n);
    std::vector<size_t> off(n), len(n);
    std::vector<bool> parsed(n);
    size_t total = 0;
    for (size_t i = 0; i < n; i++) {
        zj_decoder *dd = zj_decoder_new(&opt);
        zj_image_info info;
        if (dd && zj_decoder_read_headers(dd, bufs[i], lens[i]) == ZJ_OK && zj_decoder_info(dd, &info) == ZJ_OK && info.valid) {
            // (the output's size: a DCT-scaled decode gives ceil(width / 2^k) x ceil(height / 2^k), as output_dims states)
            const uint32_t k = dd->scale(), m = (1u << k) - 1;
            img[i].width = (info.width + m) >> k; img[i].height = (info.height + m) >> k;
            if (dd->exif_orientation() && dd->orientation >= 5) std::swap(img[i].width, img[i].height);   // (orientations 5-8)
            img[i].nc = (uint32_t)zj::num_components(zj_decoder_out_colorspace(dd));
            len[i] = (size_t)img[i].width * img[i].height * img[i].nc;
            off[i] = total;
            total += (len[i] + 255) & ~(size_t)255;
            parsed[i] = true;
        }
        if (dd) zj_decoder_free(dd);
    }
    uint8_t *scratch = nullptr;
    if (total) { const int arc = zj::scratch_alloc((void **)&scratch, total, opt.device, nullptr); if (arc != ZJ_OK) return arc; }
    std::vector<uint8_t *> mid(n);
    // (images whose headers do not parse get a dummy one-byte slot: the decode call reports their error)
    for (size_t i = 0; i < n; i++) { mid[i] = parsed[i] ? scratch + off[i] : scratch; img[i].src = mid[i]; }
    int failed = zj_decode_batch_gpu_device(&opt, bufs, lens, n, mid.data(), len.data(), status, n_gpu_entropy);
    if (failed >= 0) {
        int crc = second_pass(img, failed);
        if (crc == ZJ_OK && cudaStreamSynchronize(nullptr) != cudaSuccess) { cudaGetLastError(); crc = ZJ_ERR_CUDA; }
        if (crc != ZJ_OK) failed = crc;
    }
    zj::scratch_free(scratch, nullptr);
    return failed;
}

// The device-output call with a consumer descriptor: the pixels are reconstructed into a stream-ordered u8 scratch buffer and
// converted from there (zj_consumer.cu); with the default descriptor this IS zj_decode_batch_gpu_device.
ZJ_API int zj_decode_batch_gpu_device_ex(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                                         const zj_output_desc *d, void *const *out_dev, size_t *out_len, int *status,
                                         size_t *n_gpu_entropy)
{
    if (!d) return ZJ_ERR_INVALID_ARG;
    if (zj_output_desc_is_default(d))
        return zj_decode_batch_gpu_device(o, bufs, lens, n, reinterpret_cast<uint8_t *const *>(out_dev), out_len, status, n_gpu_entropy);
    if ((!bufs || !lens || !out_dev || !out_len || !status) && n) return ZJ_ERR_INVALID_ARG;
    zj_options opt;
    if (o) opt = *o; else zj_options_default(&opt);
    return decode_then(opt, bufs, lens, n, status, n_gpu_entropy, [&](std::vector<zj::U8Image> &img, int &failed) {
        // every decoded image through the consumer: one launch per run of equal pixel formats
        std::vector<zj::U8Image> conv;
        for (size_t i = 0; i < n; i++) {
            if (status[i] != ZJ_OK) { out_len[i] = 0; continue; }
            const size_t need = zj::convert_size(img[i].width, img[i].height, img[i].nc, d);
            if (!out_dev[i]) { status[i] = ZJ_ERR_INVALID_ARG; failed++; out_len[i] = 0; continue; }
            if (out_len[i] < need) { status[i] = ZJ_ERR_SHORT_OUTPUT; failed++; out_len[i] = 0; continue; }
            out_len[i] = need;
            img[i].dst = out_dev[i];
            conv.push_back(img[i]);
        }
        return zj::convert_many(opt.device, nullptr, conv.data(), conv.size(), d);
    });
}

// The batch-tensor call: whole images decoded into a stream-ordered u8 scratch buffer (as zj_decode_batch_gpu_device_ex does),
// then each decoded image's crop resized into its slot (zj_consumer.cu).
ZJ_API int zj_decode_batch_gpu_device_resized(const zj_options *o, const uint8_t *const *bufs, const size_t *lens, size_t n,
                                              const zj_roi *rois, const zj_output_desc *d, const zj_resize *r, void *out_dev,
                                              size_t out_len, int *status, size_t *n_gpu_entropy)
{
    if ((!bufs || !lens || !out_dev || !status) && n) return ZJ_ERR_INVALID_ARG;
    zj_options opt;
    if (o) opt = *o; else zj_options_default(&opt);
    // every slot has the channel count the options' colourspace gives
    const uint32_t nc_opt = (uint32_t)zj::num_components(opt.out_colorspace);
    const size_t slot = zj_resize_slot_size(d, r, nc_opt);
    if (slot == 0) return ZJ_ERR_INVALID_ARG;
    if (n && out_len / slot < n) return ZJ_ERR_SHORT_OUTPUT;
    return decode_then(opt, bufs, lens, n, status, n_gpu_entropy, [&](std::vector<zj::U8Image> &img, int &failed) {
        // every decoded image whose crop fits it and whose channel count is the slots' through the resize
        std::vector<zj::U8Image> admitted;
        for (size_t i = 0; i < n; i++) {
            if (status[i] != ZJ_OK) continue;
            if (zj::resize_admit(d, r, nc_opt, rois ? &rois[i] : nullptr, img[i].width, img[i].height, img[i].nc, &img[i].crop) != ZJ_OK) {
                status[i] = ZJ_ERR_INVALID_ARG; failed++; continue;
            }
            img[i].dst = static_cast<uint8_t *>(out_dev) + i * slot;
            admitted.push_back(img[i]);
        }
        return zj::resize_many(opt.device, nullptr, admitted.data(), admitted.size(), d, r);
    });
}

ZJ_API void zj_host_set_quirks(uint32_t mask) { g_quirks.store(mask & ZJ_QUIRK_ALL); }
ZJ_API uint32_t zj_host_get_quirks(void) { return g_quirks.load(); }
ZJ_API size_t zj_decoder_entropy_segments(const zj_decoder *d) { return d ? d->last_entropy_segments : 0; }
ZJ_API int zj_decoder_error_kind(const zj_decoder *d) { return d ? d->err_kind : ZJ_DE_NONE; }
ZJ_API const char *zj_decoder_error(const zj_decoder *d) { return d ? d->err_display.c_str() : ""; }

}  // extern "C"
