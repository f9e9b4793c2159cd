// zj_entropy.h -- descriptors of the GPU form of the baseline entropy stage (zj_entropy.cu), filled by the host
// front-end (zj_host_decoder.cpp).
//
// Scope: baseline scans with restart markers (DRI), and (spec and libjpeg output only) baseline scans without them, below.
// Every restart interval starts from a known state (fresh bit
// reader right behind its RSTn, predictors 0, countdown = DRI), so one GPU thread per interval runs the reference's MCU
// loop (src/mcu.rs:253-351, handle_rst :386-418) with the reference's bit reader (src/bitstream.rs:159-402) and writes
// coefficients straight into the device planes the reconstruction kernels read.  An interval that does not end exactly
// the way the sequential loop would end it is reported, and the image goes through the host stage instead.
#pragma once
#include <stdint.h>

namespace zj {

struct EntTable {          // HuffmanTable, src/huffman.rs:14-41 (the members the decode loop reads)
    int32_t lookup[512];
    int16_t ac_lookup[512];
    int32_t maxcode[18];
    int32_t offset[18];
    uint8_t values[256];
};

struct EntImage {
    const uint8_t *data;          // the whole JPEG file (device)
    uint32_t len;                 // its length (the reader's bounds, bitstream.rs:696-703)
    const uint32_t *seg_start;    // n_seg + 1 entries: reader position at the start of interval k; entry n_seg is unused
    uint8_t *status;              // n_seg entries, written by the kernel: 0 = ended like the sequential loop ends it
    const EntTable *tables;       // 2 * ncomp entries: [dc, ac] of component 0, 1, 2
    int16_t *plane[3];            // whole-image planes (zeroed before the launch); nullptr = component not output (mcu.rs:244)
    uint32_t n_seg, per_seg, total_mcus, restart_interval;
    uint32_t mcu_w, bias, ncomp, is_hv;
    uint32_t width_stride, hv_width_stride;
    uint32_t strip_len[3];
    uint32_t h_samp[3], v_samp[3], is_y[3];
};

// One thread per restart interval, LANES of them per warp (the other lanes leave at once).  The lanes of a warp sit in
// different branches of the symbol loop and a warp step costs what all the branches it holds cost together, so fewer intervals
// per warp means shorter steps and more warps to hide the dependent table / byte loads behind -- as long as the GPU has warp
// slots to spare.  Measured (JPEG bytes -> pixels in HBM, 4K 4:2:0, 135 intervals per image): 32 images 29.0 / 13.5 / 8.9 / 12.1 ms
// with 32 / 16 / 8 / 4 lanes, 256 images 27.2 / 30.1 / 30.7 / 33.4 ms: launch_entropy picks 8, 16 or 32 by the number of
// intervals of the launch.  grid = (ceil(max n_seg / intervals per CTA), images)
constexpr int ENT_THREADS = 256;                         // threads per CTA
// spec: the libjpeg form of the loop (spec and libjpeg output, zj_decoder::quirks == 0): the DC refill whenever <= 32 bits are
// buffered (Q10 off) and no break on a prefetched EOI (Q11 off); the tables come without Q9 from the host stage
int launch_entropy(const EntImage *d_images, uint32_t n_images, uint32_t max_seg, void *stream, bool spec = false);

// ---- scans without restart markers, spec and libjpeg output only (zj_entropy.cu, DESIGN.md section 5.5)
// With Q9-Q11 off the host stage's symbols are a pure function of the de-stuffed bit sequence, so a decode that starts at a
// code boundary in the right (block slot, coefficient index) state goes on exactly as the sequential loop does.  The bits are
// cut into subsequences of SYNC_BITS; each thread decodes one from an entry state and records its exit state (the state at the
// first symbol that starts at or beyond the subsequence's end), rounds take the predecessor's exit as the next entry until a
// round changes nothing; at that fixpoint every entry is the sequential decoder's state at that bit.
constexpr uint32_t SYNC_BITS = 1024;       // bits per subsequence
constexpr uint32_t SYNC_ROUNDS = 24;       // sync rounds launched per sub-batch; an image not settled by then is turned down
constexpr int SYNC_THREADS = 256;
constexpr uint64_t SYNC_INVALID = ~0ull;   // exit state of a decode that met an error (its count says how many blocks it completed)

struct SyncImage {
    const uint32_t *bits;         // de-stuffed scan, big-endian bytes, followed by >= 8 zero bytes (reads past nbits stay inside)
    uint64_t nbits;
    const EntTable *tables;       // 2 * ncomp entries: [dc, ac] of component 0, 1, 2
    int16_t *plane[3];            // zeroed whole-image planes; nullptr = component not output
    uint64_t *exit[2];            // n_sub states each (pos << 16 | slot << 8 | coef), by round parity
    uint64_t *used;               // n_sub: the entry state the subsequence's last decode started from
    uint32_t *count;              // n_sub: blocks that decode completed; then (accept kernel) the first global block index
    uint32_t *changed;            // SYNC_ROUNDS counters, zeroed: decodes run in round r
    int16_t *dc;                  // total blocks: DC differences in block order
    uint8_t *status;              // one byte, written by the accept kernel: 0 = take the planes, 1 = host stage
    uint32_t n_sub, total_mcus, bpm;
    uint32_t mcu_w, bias, is_hv, width_stride, hv_width_stride;
    uint32_t strip_len[3], h_samp[3], v_samp[3], is_y[3];
    uint8_t slot_comp[8], slot_v[8], slot_h[8];   // block slot of the MCU -> component, v_samp, h_samp (bpm <= 6)
};
// Queues one phase of the decode of n_images images on `stream` (the phases in this order: SYNC_ROUNDS round launches, accept,
// write, DC); returns a cudaError_t.
enum { SYNC_PHASE_ROUNDS = 0, SYNC_PHASE_ACCEPT = 1, SYNC_PHASE_WRITE = 2, SYNC_PHASE_DC = 3 };
int launch_sync_phase(const SyncImage *d_images, uint32_t n_images, uint32_t max_sub, void *stream, int phase);

// ---- progressive scans, spec and libjpeg output only (zj_entropy.cu, DESIGN.md section 5.6)
// Every scan of the image is decoded from its own de-stuffed bits into the zeroed whole-image planes of the host stage's
// progressive loops (mcu_prog.rs).  Phases, each over all scans of its kind in the sub-batch: (1) first scans (DC first, AC
// first), self-synchronising like the baseline decode; (2) DC refinements, one bit per block; (3) AC refinements, one thread per
// (image, component) walking that component's refinement scans in file order over non-zero masks, recording per block what
// changes, then applied to the planes one thread per block.  The host stage only hands over files whose scan
// script allows this order (every first scan of a component before its refinements of the same kind, first scans of a
// component on disjoint coefficients).
// sync rounds launched for first scans (a round after the fixpoint returns at once): their EOB runs let a wrong guess stay
// consistent for longer than a baseline scan does, and files needing more than SYNC_ROUNDS were found
constexpr uint32_t PROG_ROUNDS = 64;
enum { PROG_DC_FIRST = 0, PROG_DC_REFINE = 1, PROG_AC_FIRST = 2, PROG_AC_REFINE = 3 };
enum { PROG_DOWN_FIRST = 1, PROG_DOWN_ADDRESS = 2, PROG_DOWN_MARKER = 4, PROG_DOWN_DC_REFINE = 8, PROG_DOWN_AC_REFINE = 16 };
struct ProgScan {
    const uint32_t *bits;         // de-stuffed scan, big-endian bytes, followed by >= 8 zero bytes
    uint64_t nbits;
    const EntTable *tables;       // DC first: the DC table of each scan component; AC scans: the AC table
    int16_t *plane[3];            // the image's zeroed whole-image planes (raster block order)
    uint64_t *mask;               // AC refinement: per block of its component, the non-zero coefficients (zig-zag bit order)
    uint64_t *rec;                // AC refinement: per block of its component, 3 masks (zig-zag bit order) -- coefficients whose
                                  // correction bit is 1, coefficients the scan places, those of them that are negative
    uint64_t *exit[2];            // first scans: n_sub states (pos << 16 | slot << 8 | coef) by round parity
    uint64_t *used;               // first scans: n_sub entries
    uint32_t *count;              // first scans: n_sub
    uint32_t *changed;            // first scans: PROG_ROUNDS counters, zeroed
    int16_t *dc;                  // DC first: total DC differences in block order
    uint8_t *ok;                  // first scans: written by the accept kernel, 1 = its states are verified
    uint8_t *status;              // the image's status byte (shared by its scans): non-zero = turned down, PROG_DOWN_* bits say
                                  // by which phase (racing phases may keep only one of several)
    uint32_t plane_len[3], bw[3];  // i16 per plane; blocks per plane row
    uint32_t hs[3], vs[3];        // sampling factors per component
    uint32_t n_sub, total;        // subsequences (first scans); blocks of the scan (MCUs x blocks per MCU when interleaved)
    uint32_t kind, ss, se, al;
    uint32_t nslot, mw, mcu_x;    // blocks per MCU (1: non-interleaved, raster over mw blocks per row); MCUs per row
    uint32_t marker_check;        // the file's first scan: the host stage needs its bit reader to have met the marker behind it
    uint8_t slot_z[8], slot_t[8], slot_h[8], slot_v[8];   // block slot -> component, table, h / v offset in the MCU
};
struct ProgChain { uint32_t first, count; };   // AC refinement scans [first, first + count) of one (image, component)
// Queues the phases on `stream`: scans [0, n_first) are first scans (max_sub: the most subsequences of one), dc_ref[r] ..
// dc_ref[r + 1] the DC refinements of ordinal r (r < n_dc_ord), chains the AC refinement chains (max_blocks: the most blocks of
// a chain's plane).  phase: PROG_PHASE_*; returns a cudaError_t.
enum { PROG_PHASE_ROUNDS = 0, PROG_PHASE_ACCEPT = 1, PROG_PHASE_WRITE = 2, PROG_PHASE_DC = 3, PROG_PHASE_DC_REFINE = 4,
       PROG_PHASE_MASK = 5, PROG_PHASE_AC_REFINE = 6, PROG_PHASE_AC_APPLY = 7, PROG_PHASES = 8 };
int launch_prog_phase(const ProgScan *d_scans, uint32_t n_first, uint32_t max_sub, const uint32_t *dc_ref, uint32_t n_dc_ord,
                      uint32_t max_dc_blocks, const ProgChain *d_chains, uint32_t n_chain, uint32_t max_blocks, void *stream, int phase);

}  // namespace zj
