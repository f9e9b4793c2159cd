// zj_kernels.cu -- sm_100a kernels for the post-entropy path of zune-jpeg (reference src/worker.rs:32-251).
//
// One fused kernel per (sub-sampling mode, CPU variant mirrored): a CTA owns one TILE of one STRIP and does
//   phase 1: dequantise + 8x8 integer IDCT + level shift + clamp, one thread per 8x8 block, the whole block in
//            registers (no transposes: pass A walks rows, pass B walks columns of the same register file);
//            results go to shared-memory sample planes (u8 for the X86 variant, i16 for SCALAR) together with
//            the chroma halo blocks the strip-flat up-samplers reach into;
//   phase 2: chroma up-sampling (the reference's as-written closed forms, SURVEY.md Appendix A.4) +
//            YCbCr->RGB / YCbCr interleave + the row writer of worker.rs:143-251 (row-tail rule, zero bytes).
// Bytes the reference never writes are written as zero here, so the output needs no memset.
//
// Everything is integer and must be bit-exact against oracle/ (tests/test_gpu_parity.py).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "zj_device.h"

#define ZF_LIKELY(x) __builtin_expect(!!(x), 1)
#define ZF_UNLIKELY(x) __builtin_expect(!!(x), 0)

namespace zj {

typedef uint32_t u32;

// ------------------------------------------------------------------------------------------------ IDCT
// 1-D 8-point kernel: reference src/idct/scalar.rs:79-166 == src/idct/avx2.rs:251-331.  All arithmetic is
// in Z/2^32 (u32), the final shift is arithmetic.
// The butterfly is written as the 43 operations it needs (27 multiply-adds / adds of the even and odd parts + 16 for the final
// sums and shifts) with the multiply-adds pinned as `mad.lo` -- the reference's plain expression form compiled to 50 (the
// rounding bias as four separate adds, the products of p3 / p4 formed once and added twice).  Regrouping is exact: all of it is
// arithmetic in Z/2^32 (tests/test_idct_regroup.py checks it against the reference's literal order).
template <int K> __device__ __forceinline__ u32 madk(u32 a, u32 c) { u32 d; asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "n"(K), "r"(c)); return d; }

template <int SH>
__device__ __forceinline__ void idct8(u32 &s0, u32 &s1, u32 &s2, u32 &s3, u32 &s4, u32 &s5, u32 &s6, u32 &s7, const u32 bias)
{
    const u32 p1 = (s2 + s6) * 2217u;
    const u32 t2 = madk<-7567>(s6, p1), t3 = madk<3135>(s2, p1);
    const u32 v = (s0 << 12) + bias;
    const u32 t0 = madk<4096>(s4, v), t1 = madk<-4096>(s4, v);
    const u32 x0 = t0 + t3, x3 = t0 - t3, x1 = t1 + t2, x2 = t1 - t2;
    const u32 p3 = s7 + s3, p4 = s5 + s1, q1 = s7 + s1, q2 = s5 + s3;
    const u32 p5 = (p3 + p4) * 4816u;
    const u32 r1 = madk<-3685>(q1, p5), r2 = madk<-10497>(q2, p5);
    const u32 a = madk<1223>(s7, madk<-8034>(p3, r1));
    const u32 c = madk<12586>(s3, madk<-8034>(p3, r2));
    const u32 b = madk<8410>(s5, madk<-1597>(p4, r2));
    const u32 d = madk<6149>(s1, madk<-1597>(p4, r1));
    s0 = (u32)((int)(x0 + d) >> SH);
    s1 = (u32)((int)(x1 + c) >> SH);
    s2 = (u32)((int)(x2 + b) >> SH);
    s3 = (u32)((int)(x3 + a) >> SH);
    s4 = (u32)((int)(x3 - a) >> SH);
    s5 = (u32)((int)(x2 - b) >> SH);
    s6 = (u32)((int)(x1 - c) >> SH);
    s7 = (u32)((int)(x0 - d) >> SH);
}


// The same 1-D kernel with s4 = s5 = s6 = s7 = 0 folded in (identical results, fewer operations): used when a whole
// warp's blocks have nothing outside the top-left 4x4 (99.8 % of the chroma blocks of a quality-90 photo).
template <int SH>
__device__ __forceinline__ void idct8_lo4(u32 &s0, u32 &s1, u32 &s2, u32 &s3, u32 &s4, u32 &s5, u32 &s6, u32 &s7, const u32 bias)
{
    // 29 operations: every intermediate is a two-term combination of (s0, s2) or (s1, s3) with the constants summed up front
    const u32 t0 = (s0 << 12) + bias;
    const u32 x0 = madk<2217 + 3135>(s2, t0), x3 = madk<-(2217 + 3135)>(s2, t0), x1 = madk<2217>(s2, t0), x2 = madk<-2217>(s2, t0);
    const u32 c48 = s3 * 4816u, d48 = s1 * 4816u;
    const u32 dd = madk<6149 - 3685 + 4816 - 1597>(s1, c48);            // d * 6149 + q1 + p4
    const u32 cc = madk<12586 - 10497 + 4816 - 8034>(s3, d48);          // c * 12586 + q2 + p3
    const u32 bb = madk<4816 - 10497>(s3, s1 * (u32)(4816 - 1597));     // q2 + p4
    const u32 aa = madk<4816 - 3685>(s1, s3 * (u32)(4816 - 8034));      // q1 + p3
    s0 = (u32)((int)(x0 + dd) >> SH);
    s1 = (u32)((int)(x1 + cc) >> SH);
    s2 = (u32)((int)(x2 + bb) >> SH);
    s3 = (u32)((int)(x3 + aa) >> SH);
    s4 = (u32)((int)(x3 - aa) >> SH);
    s5 = (u32)((int)(x2 - bb) >> SH);
    s6 = (u32)((int)(x1 - cc) >> SH);
    s7 = (u32)((int)(x0 - dd) >> SH);
}

// The same 1-D kernel with s6 = s7 = 0 folded in: the column pass of blocks whose rows 6 and 7 are zero
// (99 % of the luma blocks of a quality-90 photo).
template <int SH>
__device__ __forceinline__ void idct8_lo6(u32 &s0, u32 &s1, u32 &s2, u32 &s3, u32 &s4, u32 &s5, u32 &s6, u32 &s7, const u32 bias)
{
    // 35 operations
    const u32 v = (s0 << 12) + bias;
    const u32 t0 = madk<4096>(s4, v), t1 = madk<-4096>(s4, v);
    const u32 x0 = madk<2217 + 3135>(s2, t0), x3 = madk<-(2217 + 3135)>(s2, t0), x1 = madk<2217>(s2, t1), x2 = madk<-2217>(s2, t1);
    const u32 p4 = s5 + s1, q2 = s5 + s3;          // a = s7 = 0: p3 = c, q1 = d
    const u32 p5 = (s3 + p4) * 4816u;
    const u32 r1 = madk<-3685>(s1, p5), r2 = madk<-10497>(q2, p5);
    const u32 aa = madk<-8034>(s3, r1);
    const u32 cc = madk<12586 - 8034>(s3, r2);
    const u32 bb = madk<8410>(s5, madk<-1597>(p4, r2));
    const u32 dd = madk<6149>(s1, madk<-1597>(p4, r1));
    s0 = (u32)((int)(x0 + dd) >> SH);
    s1 = (u32)((int)(x1 + cc) >> SH);
    s2 = (u32)((int)(x2 + bb) >> SH);
    s3 = (u32)((int)(x3 + aa) >> SH);
    s4 = (u32)((int)(x3 - aa) >> SH);
    s5 = (u32)((int)(x2 - bb) >> SH);
    s6 = (u32)((int)(x1 - cc) >> SH);
    s7 = (u32)((int)(x0 - dd) >> SH);
}

// x / n for 0 <= x, 1 <= n <= 1024 without an integer divide: (x + 0.5) / n is at least 0.5/n away from an integer,
// far more than the error of the float reciprocal, so truncation is exact
__device__ __forceinline__ int div_small(int x, float rcp_n) { return (int)(((float)x + 0.5f) * rcp_n); }

__device__ __forceinline__ u32 clamp255(u32 v) { return (u32)max(min((int)v, 255), 0); }

// s16x2 . u8 dot products (IDP.2A): unpack + dequantise one coefficient in a single instruction.
__device__ __forceinline__ u32 dp2a_lo(u32 a, u32 b) { u32 d; asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0)); return d; }
__device__ __forceinline__ u32 dp2a_hi(u32 a, u32 b) { u32 d; asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0)); return d; }

// I2IP.U8.S32.SAT: d = (c << 16) | sat_u8(a) << 8 | sat_u8(b) -- clamp to [0,255] and pack two values per instruction
__device__ __forceinline__ u32 pack_sat2(int hi, int lo, u32 upper) { u32 d; asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(hi), "r"(lo), "r"(upper)); return d; }
// v[] are UNCLAMPED i32 results; the clamp of idct/avx2.rs:402-413 happens in the saturating pack
__device__ __forceinline__ void store_row(uint8_t *dst, const u32 v[8])
{
    uint2 w;
    w.x = pack_sat2((int)v[1], (int)v[0], pack_sat2((int)v[3], (int)v[2], 0u));
    w.y = pack_sat2((int)v[5], (int)v[4], pack_sat2((int)v[7], (int)v[6], 0u));
    *reinterpret_cast<uint2 *>(dst) = w;
}
template <bool CLAMP = true>
__device__ __forceinline__ void store_row(int16_t *dst, const u32 vin[8])
{
    u32 v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = CLAMP ? clamp255(vin[k]) : vin[k];
    uint4 w;
    w.x = (v[0] & 0xffffu) | (v[1] << 16);
    w.y = (v[2] & 0xffffu) | (v[3] << 16);
    w.z = (v[4] & 0xffffu) | (v[5] << 16);
    w.w = (v[6] & 0xffffu) | (v[7] << 16);
    *reinterpret_cast<uint4 *>(dst) = w;
}

// DC-only rows: X86 already clamped the value (the saturating pack is a no-op), SCALAR must stay unclamped
__device__ __forceinline__ void store_dc_row(uint8_t *dst, const u32 v[8]) { store_row(dst, v); }
__device__ __forceinline__ void store_dc_row(int16_t *dst, const u32 v[8]) { store_row<false>(dst, v); }

// Dequantise + 2-D IDCT + level shift + clamp of one block; rows written to dst[r*dst_stride + 0..7].
//   VARIANT 0 (X86):    pass A along rows, pass B down columns, DC-only value clamped   (idct/avx2.rs:64-398)
//   VARIANT 1 (SCALAR): pass A down columns, pass B along rows, DC-only value NOT clamped (idct/scalar.rs:19-282)
// qtw: 32 words, word k = q[2k] | q[2k+1] << 24 (natural order).  dst rows must be 8 samples-aligned.
// 128-bit loads of one block's 64 coefficients (read once: non-coherent path); lanes without a block get zeros
__device__ __forceinline__ void load_block(const bool active, const int16_t *__restrict__ src, int4 (&raw)[8])
{
    const int4 *p = reinterpret_cast<const int4 *>(src);
#pragma unroll
    for (int r = 0; r < 8; r++) raw[r] = active ? __ldg(p + r) : make_int4(0, 0, 0, 0);
}

// `active` lanes own a block; every lane of the warp must call this (warp votes pick the sparse code paths).
template <int VARIANT, typename ST>
__device__ __forceinline__ void idct_block(const bool active, const int4 (&raw)[8], const u32 *__restrict__ qtw, ST *__restrict__ dst, int dst_stride)
{

    u32 rowor[8], col47 = 0;
    rowor[0] = ((u32)raw[0].x & 0xffff0000u) | (u32)raw[0].y | (u32)raw[0].z | (u32)raw[0].w;
#pragma unroll
    for (int r = 1; r < 8; r++) rowor[r] = (u32)raw[r].x | (u32)raw[r].y | (u32)raw[r].z | (u32)raw[r].w;
#pragma unroll
    for (int r = 0; r < 8; r++) col47 |= (u32)raw[r].z | (u32)raw[r].w;
    const u32 r45 = rowor[4] | rowor[5], r67 = rowor[6] | rowor[7];
    const u32 acc = rowor[0] | rowor[1] | rowor[2] | rowor[3] | r45 | r67;
    // warp-uniform sparsity classes (a zero row / column transforms to exact zeros, so skipping it changes nothing)
    const bool any_r67 = __any_sync(0xffffffffu, r67 != 0);
    const bool any_r47 = __any_sync(0xffffffffu, (r45 | r67) != 0);
    const bool any_c47 = __any_sync(0xffffffffu, col47 != 0);
    if (!active) return;

    if (acc == 0) {
        // all 63 AC coefficients zero: ((c0 as i16).wrapping_mul(q0 as i16) >> 3) + 128 in i16
        // (avx2.rs:159-167 clamps, scalar.rs:45-48 does not)
        int dc = (int)(int16_t)((u32)raw[0].x & 0xffffu);
        int q0 = (int)(int16_t)(qtw[0] & 0xffu);
        int v = (int)(int16_t)(dc * q0);
        v = (int)(int16_t)((v >> 3) + 128);
        if (VARIANT == 0) v = max(min(v, 255), 0);
        u32 vv[8];
#pragma unroll
        for (int k = 0; k < 8; k++) vv[k] = (u32)v;
#pragma unroll
        for (int r = 0; r < 8; r++) store_dc_row(dst + r * dst_stride, vv);
        return;
    }

    u32 a[64];
    const u32 SCALE_BITS = 512u + 65536u + (128u << 17);
    auto dequant_row = [&](int r, int nwords) {
        const u32 w[4] = {(u32)raw[r].x, (u32)raw[r].y, (u32)raw[r].z, (u32)raw[r].w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (k < nwords) {
                const u32 q = qtw[r * 4 + k];
                a[r * 8 + 2 * k] = dp2a_lo(w[k], q);
                a[r * 8 + 2 * k + 1] = dp2a_hi(w[k], q);
            } else {
                a[r * 8 + 2 * k] = 0;
                a[r * 8 + 2 * k + 1] = 0;
            }
        }
    };
    if (VARIANT == 0) {
        if (!any_r47 && !any_c47) {
            // top-left 4x4 only: 4 row transforms and 8 column transforms, each with 4 inputs
#pragma unroll
            for (int r = 0; r < 4; r++) {
                dequant_row(r, 2);
                idct8_lo4<10>(a[r * 8], a[r * 8 + 1], a[r * 8 + 2], a[r * 8 + 3], a[r * 8 + 4], a[r * 8 + 5], a[r * 8 + 6], a[r * 8 + 7], 512u);
            }
#pragma unroll
            for (int c = 0; c < 8; c++)
                idct8_lo4<17>(a[c], a[8 + c], a[16 + c], a[24 + c], a[32 + c], a[40 + c], a[48 + c], a[56 + c], SCALE_BITS);
        } else {
#pragma unroll
            for (int r = 0; r < 6; r++) {
                dequant_row(r, 4);
                idct8<10>(a[r * 8], a[r * 8 + 1], a[r * 8 + 2], a[r * 8 + 3], a[r * 8 + 4], a[r * 8 + 5], a[r * 8 + 6], a[r * 8 + 7], 512u);
            }
            if (any_r67) {
#pragma unroll
                for (int r = 6; r < 8; r++) {
                    dequant_row(r, 4);
                    idct8<10>(a[r * 8], a[r * 8 + 1], a[r * 8 + 2], a[r * 8 + 3], a[r * 8 + 4], a[r * 8 + 5], a[r * 8 + 6], a[r * 8 + 7], 512u);
                }
            } else {
#pragma unroll
                for (int k = 48; k < 64; k++) a[k] = 0;   // (0 * c + 512) >> 10 == 0
            }
#pragma unroll
            for (int c = 0; c < 8; c++)
                idct8<17>(a[c], a[8 + c], a[16 + c], a[24 + c], a[32 + c], a[40 + c], a[48 + c], a[56 + c], SCALE_BITS);
        }
    } else {
#pragma unroll
        for (int r = 0; r < 8; r++) dequant_row(r, 4);
#pragma unroll
        for (int c = 0; c < 8; c++)
            idct8<10>(a[c], a[8 + c], a[16 + c], a[24 + c], a[32 + c], a[40 + c], a[48 + c], a[56 + c], 512u);
#pragma unroll
        for (int r = 0; r < 8; r++)
            idct8<17>(a[r * 8], a[r * 8 + 1], a[r * 8 + 2], a[r * 8 + 3], a[r * 8 + 4], a[r * 8 + 5], a[r * 8 + 6], a[r * 8 + 7], SCALE_BITS);
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {
        u32 vv[8];
#pragma unroll
        for (int k = 0; k < 8; k++) vv[k] = a[r * 8 + k];
        store_row(dst + r * dst_stride, vv);  // clamps
    }
}

// ------------------------------------------------------------------------------------------------ islow IDCT
constexpr int IDCT_X86 = 0, IDCT_ISLOW = 2;   // spec_kernel's IDCT parameter (gray_kernel's VARIANT: 1 is SCALAR's)
// libjpeg-turbo's jpeg_idct_islow (jidctint.c): step 1 of ZJ_FLAG_ISLOW images (the statement is in include/zune_jpeg_b200.h).
// All arithmetic is in Z/2^32, as in the X86 IDCT.  One 1-D pass: CONST_BITS 13, 12 multiplies; the DESCALE rounding comes in as
// `bias`.  Pass 1 (columns) ends in DESCALE(x, 11).  Pass 2 (rows) ends in range_limit[v], v = DESCALE(x, 18) & 1023 = bits
// 18-27 of x + 2^17: the table is v + 128 for v in [0, 511] and v - 896 for [512, 1023], each clamped to [0, 255], i.e. v read as
// a signed 10-bit value, plus 128, clamped (store_row's saturating pack clamps).
template <bool ROWS>
__device__ __forceinline__ void islow8(u32 &s0, u32 &s1, u32 &s2, u32 &s3, u32 &s4, u32 &s5, u32 &s6, u32 &s7, const u32 bias)
{
    // even part
    const u32 z1 = (s2 + s6) * 4433u;                                        // FIX_0_541196100
    const u32 t2 = madk<-15137>(s6, z1), t3 = madk<6270>(s2, z1);           // FIX_1_847759065, FIX_0_765366865
    const u32 t0 = madk<8192>(s0 + s4, bias), t1 = madk<8192>(s0 - s4, bias);
    const u32 x0 = t0 + t3, x3 = t0 - t3, x1 = t1 + t2, x2 = t1 - t2;         // tmp10, tmp13, tmp11, tmp12
    // odd part: z1 = s7 + s1, z2 = s5 + s3, z3 = s7 + s3, z4 = s5 + s1
    const u32 z3 = s7 + s3, z4 = s5 + s1;
    const u32 z5 = (z3 + z4) * 9633u;                                        // FIX_1_175875602
    const u32 p1 = (s7 + s1) * (u32)-7373, p2 = (s5 + s3) * (u32)-20995;   // FIX_0_899976223, FIX_2_562915447
    const u32 r3 = madk<-16069>(z3, z5), r4 = madk<-3196>(z4, z5);          // FIX_1_961570560, FIX_0_390180644
    const u32 a = madk<2446>(s7, p1 + r3);                                   // tmp0, FIX_0_298631336
    const u32 b = madk<16819>(s5, p2 + r4);                                  // tmp1, FIX_2_053119869
    const u32 c = madk<25172>(s3, p2 + r3);                                  // tmp2, FIX_3_072711026
    const u32 d = madk<12299>(s1, p1 + r4);                                  // tmp3, FIX_1_501321110
    const u32 o[8] = {x0 + d, x1 + c, x2 + b, x3 + a, x3 - a, x2 - b, x1 - c, x0 - d};
    u32 *const s[8] = {&s0, &s1, &s2, &s3, &s4, &s5, &s6, &s7};
#pragma unroll
    for (int k = 0; k < 8; k++) *s[k] = ROWS ? (u32)(((int)(o[k] << 4) >> 22) + 128) : (u32)((int)o[k] >> 11);
}

// Dequantise + islow IDCT of one block, u8 rows written to dst[r*dst_stride + 0..7]; fits load_block like idct_block, and every
// lane of the warp must call it.  The zero-AC shortcuts of jidctint.c: a block whose AC is all zero has one sample value; the
// row shortcut of pass 2 equals the full pass and is not taken; the column shortcut of pass 1 equals the full pass unless the
// dequantised DC is 2^18 or more in magnitude, so it is applied after the full pass, only in warps where such a DC occurs.
// Warp-uniform sparsity classes fold zero inputs out of the passes, as in idct_block: top-left 4x4 only, rows 6-7 zero, full.
__device__ __forceinline__ void idct_islow_block(const bool active, const int4 (&raw)[8], const u32 *__restrict__ qtw, uint8_t *__restrict__ dst, int dst_stride)
{
    u32 rowor[8], col47 = 0, cor[4] = {0u, 0u, 0u, 0u};
    rowor[0] = ((u32)raw[0].x & 0xffff0000u) | (u32)raw[0].y | (u32)raw[0].z | (u32)raw[0].w;
#pragma unroll
    for (int r = 1; r < 8; r++) {
        rowor[r] = (u32)raw[r].x | (u32)raw[r].y | (u32)raw[r].z | (u32)raw[r].w;
        cor[0] |= (u32)raw[r].x; cor[1] |= (u32)raw[r].y; cor[2] |= (u32)raw[r].z; cor[3] |= (u32)raw[r].w;
    }
#pragma unroll
    for (int r = 0; r < 8; r++) col47 |= (u32)raw[r].z | (u32)raw[r].w;
    u32 dcol = 0;   // bit c: column c has no coefficient in rows 1-7 (jidctint.c's pass-1 shortcut)
#pragma unroll
    for (int c = 0; c < 8; c++) dcol |= (((c & 1) ? cor[c >> 1] >> 16 : cor[c >> 1] & 0xffffu) == 0 ? 1u : 0u) << c;
    const u32 r45 = rowor[4] | rowor[5], r67 = rowor[6] | rowor[7];
    const u32 acc = rowor[0] | rowor[1] | rowor[2] | rowor[3] | r45 | r67;
    const bool any_r67 = __any_sync(0xffffffffu, r67 != 0);
    const bool any_r47 = __any_sync(0xffffffffu, (r45 | r67) != 0);
    const bool any_c47 = __any_sync(0xffffffffu, col47 != 0);
    if (!active) return;

    if (acc == 0) {
        // every column takes the pass-1 shortcut, every row the pass-2 one: range_limit[DESCALE(DC * q << 2, 5) & 1023]
        const int z = (int)(int16_t)((u32)raw[0].x & 0xffffu) * (int)(qtw[0] & 0xffu);
        const u32 v = (u32)(((int)((u32)((z * 4 + 16) >> 5) << 22) >> 22) + 128);
        u32 vv[8];
#pragma unroll
        for (int k = 0; k < 8; k++) vv[k] = v;
#pragma unroll
        for (int r = 0; r < 8; r++) store_row(dst + r * dst_stride, vv);   // clamps
        return;
    }

    u32 a[64];
    auto dequant_row = [&](int r, int nwords) {
        const u32 w[4] = {(u32)raw[r].x, (u32)raw[r].y, (u32)raw[r].z, (u32)raw[r].w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (k < nwords) {
                const u32 q = qtw[r * 4 + k];
                a[r * 8 + 2 * k] = dp2a_lo(w[k], q);
                a[r * 8 + 2 * k + 1] = dp2a_hi(w[k], q);
            } else {
                a[r * 8 + 2 * k] = 0;
                a[r * 8 + 2 * k + 1] = 0;
            }
        }
    };
    // pass 1 down columns [0, ncols); a column without AC whose DC wraps gets the shortcut value DC << 2 instead
    auto pass1 = [&](int ncols, bool fix) {
#pragma unroll
        for (int c = 0; c < 8; c++) {
            if (c >= ncols) continue;
            const u32 dc = a[c];
            islow8<false>(a[c], a[8 + c], a[16 + c], a[24 + c], a[32 + c], a[40 + c], a[48 + c], a[56 + c], 1u << 10);
            if (fix && ((dcol >> c) & 1u)) {
#pragma unroll
                for (int r = 0; r < 8; r++) a[r * 8 + c] = dc << 2;
            }
        }
    };
    // some dequantised DC of row 0 has |value| >= 2^18 (vote of the lanes still here: the outcome only decides who runs the
    // exact per-lane fix-up of pass1)
    auto big_dc = [&]() {
        u32 o = 0;
#pragma unroll
        for (int c = 0; c < 8; c++) o |= a[c] + (1u << 18);
        return __any_sync(__activemask(), dcol != 0 && o >= (1u << 19));
    };
    // pass 2 along the rows, and the stores
    auto pass2 = [&]() {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            islow8<true>(a[r * 8], a[r * 8 + 1], a[r * 8 + 2], a[r * 8 + 3], a[r * 8 + 4], a[r * 8 + 5], a[r * 8 + 6], a[r * 8 + 7], 1u << 17);
            u32 vv[8];
#pragma unroll
            for (int k = 0; k < 8; k++) vv[k] = a[r * 8 + k];
            store_row(dst + r * dst_stride, vv);   // clamps: range_limit
        }
    };
    // each class runs its own copy of the passes, so that the zeros it knows of fold away
    if (!any_r47 && !any_c47) {
#pragma unroll
        for (int r = 0; r < 8; r++) dequant_row(r, r < 4 ? 2 : 0);
        pass1(4, big_dc());
#pragma unroll
        for (int r = 0; r < 8; r++)
#pragma unroll
            for (int c = 4; c < 8; c++) a[r * 8 + c] = 0;   // all-zero columns: 0 by either form of pass 1
        pass2();
    } else {
#pragma unroll
        for (int r = 0; r < 6; r++) dequant_row(r, 4);
        const bool fix = big_dc();
        if (any_r67) {
            dequant_row(6, 4);
            dequant_row(7, 4);
            pass1(8, fix);
        } else {
            dequant_row(6, 0);
            dequant_row(7, 0);
            pass1(8, fix);
        }
        pass2();
    }
}

// ------------------------------------------------------------------------------------------------ reduced IDCTs
// libjpeg-turbo's jidctred.c: step 2'' of DCT-scaled images (the statement is in include/zune_jpeg_b200.h), in Z/2^32 as islow8.
// A block of S x S samples (S = 4: jpeg_idct_4x4, 2: jpeg_idct_2x2, 1: jpeg_idct_1x1) fits load_block's registers: load_rows<S>
// reads only the rows the transform uses (S = 1: the DC's 32-byte sector), and idct_reduced<S> needs no warp vote.
template <int S>
__device__ __forceinline__ bool row_used(int r) { return S == 4 ? r != 4 : (S == 2 ? (r < 2 || (r & 1)) : r == 0); }

template <int S>
__device__ __forceinline__ void load_rows(const bool active, const int16_t *__restrict__ src, int4 (&raw)[8])
{
    const int4 *p = reinterpret_cast<const int4 *>(src);
#pragma unroll
    for (int r = 0; r < 8; r++) raw[r] = active && row_used<S>(r) ? __ldg(p + r) : make_int4(0, 0, 0, 0);
}

// coefficient and dequantised value at row r, column c (compile-time after unrolling)
__device__ __forceinline__ int coef_at(const int4 (&raw)[8], int r, int c)
{
    const int k = c >> 1;
    const u32 w = (u32)(k == 0 ? raw[r].x : k == 1 ? raw[r].y : k == 2 ? raw[r].z : raw[r].w);
    return (c & 1) ? (int)w >> 16 : (int)(int16_t)(w & 0xffffu);
}
__device__ __forceinline__ u32 dequant_at(const int4 (&raw)[8], const u32 *__restrict__ qtw, int r, int c)
{
    const u32 w = qtw[(r * 8 + c) >> 1];
    return (u32)coef_at(raw, r, c) * ((c & 1) ? w >> 24 : w & 0xffu);
}
// range_limit[DESCALE(x, N) & 1023]: bits N..N+9 of x + 2^(N-1) read as a signed 10-bit value, plus 128, clamped
template <int N>
__device__ __forceinline__ u32 descale_limit(u32 x) { return clamp255((u32)(((int)((x + (1u << (N - 1))) << (22 - N)) >> 22) + 128)); }

// one 1-D pass of jpeg_idct_4x4 (inputs 0-3, 5-7) and of jpeg_idct_2x2 (inputs 0, 1, 3, 5, 7), before the DESCALE
__device__ __forceinline__ void red4(u32 v0, u32 v1, u32 v2, u32 v3, u32 v5, u32 v6, u32 v7, u32 o[4])
{
    const u32 t0 = v0 << 14;                                                              // << (CONST_BITS + 1)
    const u32 t2 = v2 * 15137u + v6 * (u32)-6270;                                         // FIX_1_847759065, -FIX_0_765366865
    const u32 t10 = t0 + t2, t12 = t0 - t2;
    const u32 a = v7 * (u32)-1730 + v5 * 11893u + v3 * (u32)-17799 + v1 * 8697u;         // tmp0
    const u32 b = v7 * (u32)-4176 + v5 * (u32)-4926 + v3 * 7373u + v1 * 20995u;          // tmp2
    o[0] = t10 + b; o[1] = t12 + a; o[2] = t12 - a; o[3] = t10 - b;
}
__device__ __forceinline__ void red2(u32 v0, u32 v1, u32 v3, u32 v5, u32 v7, u32 o[2])
{
    const u32 t10 = v0 << 15;                                                             // << (CONST_BITS + 2)
    const u32 t0 = v7 * (u32)-5906 + v5 * 6967u + v3 * (u32)-10426 + v1 * 29692u;
    o[0] = t10 + t0; o[1] = t10 - t0;
}

// Dequantise + reduced IDCT of one block into dst[r * dst_stride + c], r, c < S (S = 4, 2, 1); called by lanes that own a block
template <int S>
__device__ __forceinline__ void idct_reduced(const int4 (&raw)[8], const u32 *__restrict__ qtw, uint8_t *__restrict__ dst, int dst_stride)
{
    if constexpr (S == 1) {
        dst[0] = (uint8_t)descale_limit<3>(dequant_at(raw, qtw, 0, 0));
    } else if constexpr (S == 2) {
        u32 ws[2][8];
#pragma unroll
        for (int c = 0; c < 8; c++) {
            if (!row_used<2>(c)) continue;   // columns 2, 4, 6: never read by pass 2
            if ((coef_at(raw, 1, c) | coef_at(raw, 3, c) | coef_at(raw, 5, c) | coef_at(raw, 7, c)) == 0) {
                ws[0][c] = ws[1][c] = dequant_at(raw, qtw, 0, c) << 2;
            } else {
                u32 o[2];
                red2(dequant_at(raw, qtw, 0, c), dequant_at(raw, qtw, 1, c), dequant_at(raw, qtw, 3, c), dequant_at(raw, qtw, 5, c),
                     dequant_at(raw, qtw, 7, c), o);
                ws[0][c] = (u32)((int)(o[0] + (1u << 12)) >> 13);
                ws[1][c] = (u32)((int)(o[1] + (1u << 12)) >> 13);
            }
        }
#pragma unroll
        for (int r = 0; r < 2; r++) {
            const u32 *w = ws[r];
            uint8_t *d = dst + r * dst_stride;
            if ((w[1] | w[3] | w[5] | w[7]) == 0) {
                d[0] = d[1] = (uint8_t)descale_limit<5>(w[0]);
            } else {
                u32 o[2];
                red2(w[0], w[1], w[3], w[5], w[7], o);
                d[0] = (uint8_t)descale_limit<20>(o[0]);
                d[1] = (uint8_t)descale_limit<20>(o[1]);
            }
        }
    } else {
        static_assert(S == 4, "reduced IDCT sizes: 4, 2, 1");
        u32 ws[4][8];
#pragma unroll
        for (int c = 0; c < 8; c++) {
            if (c == 4) continue;            // column 4: never read by pass 2
            if ((coef_at(raw, 1, c) | coef_at(raw, 2, c) | coef_at(raw, 3, c) | coef_at(raw, 5, c) | coef_at(raw, 6, c) | coef_at(raw, 7, c)) == 0) {
                ws[0][c] = ws[1][c] = ws[2][c] = ws[3][c] = dequant_at(raw, qtw, 0, c) << 2;
            } else {
                u32 o[4];
                red4(dequant_at(raw, qtw, 0, c), dequant_at(raw, qtw, 1, c), dequant_at(raw, qtw, 2, c), dequant_at(raw, qtw, 3, c),
                     dequant_at(raw, qtw, 5, c), dequant_at(raw, qtw, 6, c), dequant_at(raw, qtw, 7, c), o);
#pragma unroll
                for (int r = 0; r < 4; r++) ws[r][c] = (u32)((int)(o[r] + (1u << 11)) >> 12);
            }
        }
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const u32 *w = ws[r];
            u32 v[4];
            if ((w[1] | w[2] | w[3] | w[5] | w[6] | w[7]) == 0) {
                v[0] = v[1] = v[2] = v[3] = descale_limit<5>(w[0]);
            } else {
                u32 o[4];
                red4(w[0], w[1], w[2], w[3], w[5], w[6], w[7], o);
#pragma unroll
                for (int k = 0; k < 4; k++) v[k] = descale_limit<19>(o[k]);
            }
            *reinterpret_cast<u32 *>(dst + r * dst_stride) = v[0] | v[1] << 8 | v[2] << 16 | v[3] << 24;
        }
    }
}

// The IDCT of the fast kernel's producers (X86 variant, u8 planes), written as two short loops instead of one long
// unrolled body so that it stays resident in the instruction cache next to the consumers' code:
//   row pass:    row r of the block is read from the thread's staging slot (16-byte chunk r at sl ^ (r << 4)),
//                dequantised and transformed; the eight 32-bit results go to the thread's scratch column (chunk k at
//                sc + k * 16 * ZF_PRODUCERS: chunks 2r and 2r+1).  Rows that are zero in every block of the warp are
//                skipped (a zero row transforms to exact zeros), rows without anything in columns 4-7 use the 4-input form;
//   column pass: two groups of four columns, each read back as one 128-bit word per row, transformed, clamped and
//                stored as four bytes per row.
// Identical results to idct_block<0>: same 1-D kernels, same order (rows, then columns), same DC-only shortcut.
__device__ __forceinline__ void lds128(u32 addr, u32 &a, u32 &b, u32 &c, u32 &d) { asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr)); }
__device__ __forceinline__ void sts128(u32 addr, u32 a, u32 b, u32 c, u32 d) { asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory"); }

// one row of the row pass: dequantise (IDP.2A: s16 x u8) + 1-D transform, results to scratch chunks k, k+1
__device__ __forceinline__ void row_pass(const bool any, const bool anyhi, const u32 w0, const u32 w1, const u32 w2, const u32 w3,
                                         const uint4 q, const u32 out)
{
    constexpr u32 CH = 16u * ZF_PRODUCERS;   // bytes between scratch chunks
    if (!any) {                              // zero in every block of the warp: a zero row transforms to exact zeros
        sts128(out, 0u, 0u, 0u, 0u);
        sts128(out + CH, 0u, 0u, 0u, 0u);
        return;
    }
    u32 s0 = dp2a_lo(w0, q.x), s1 = dp2a_hi(w0, q.x), s2 = dp2a_lo(w1, q.y), s3 = dp2a_hi(w1, q.y), s4 = 0, s5 = 0, s6 = 0, s7 = 0;
    if (anyhi) {
        s4 = dp2a_lo(w2, q.z); s5 = dp2a_hi(w2, q.z); s6 = dp2a_lo(w3, q.w); s7 = dp2a_hi(w3, q.w);
        idct8<10>(s0, s1, s2, s3, s4, s5, s6, s7, 512u);
    } else {
        idct8_lo4<10>(s0, s1, s2, s3, s4, s5, s6, s7, 512u);   // nothing in columns 4-7
    }
    sts128(out, s0, s1, s2, s3);
    sts128(out + CH, s4, s5, s6, s7);
}

// four columns of the column pass: NIN input rows (the rest are zero in every block of the warp)
template <int NIN>
__device__ __forceinline__ void col_pass(const bool active, const bool dconly, const u32 dcword, const u32 in, uint8_t *__restrict__ out, const int stride)
{
    constexpr u32 CH = 16u * ZF_PRODUCERS;
    const u32 SCALE_BITS = 512u + 65536u + (128u << 17);
    u32 a[8][4];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        if (r < NIN) lds128(in + (u32)(2 * r) * CH, a[r][0], a[r][1], a[r][2], a[r][3]);
        else a[r][0] = a[r][1] = a[r][2] = a[r][3] = 0;
    }
#pragma unroll
    for (int c = 0; c < 4; c++) {
        if (NIN == 4) idct8_lo4<17>(a[0][c], a[1][c], a[2][c], a[3][c], a[4][c], a[5][c], a[6][c], a[7][c], SCALE_BITS);
        else if (NIN == 6) idct8_lo6<17>(a[0][c], a[1][c], a[2][c], a[3][c], a[4][c], a[5][c], a[6][c], a[7][c], SCALE_BITS);
        else idct8<17>(a[0][c], a[1][c], a[2][c], a[3][c], a[4][c], a[5][c], a[6][c], a[7][c], SCALE_BITS);
    }
    if (!active) return;
    if (ZF_UNLIKELY(dconly)) {
#pragma unroll
        for (int r = 0; r < 8; r++) *reinterpret_cast<u32 *>(out + r * stride) = dcword;
    } else {
#pragma unroll
        for (int r = 0; r < 8; r++)
            *reinterpret_cast<u32 *>(out + r * stride) = pack_sat2((int)a[r][1], (int)a[r][0], pack_sat2((int)a[r][3], (int)a[r][2], 0u));   // clamps
    }
}

// UNROLL: 1 = the row-pair loop stays rolled (4:2:0 / 4:4:0: the consumers' hot code leaves no room in the 32 KB instruction
// cache for more); 4 = unrolled (everything that depends on the row pair becomes static: +7 % on 4:2:2, +10 % luma-only)
template <int UNROLL, bool LO6, typename AfterRows>
__device__ __forceinline__ void idct_rolled(const bool active, const u32 sl, const u32 sc, const u32 *__restrict__ qtw, uint8_t *__restrict__ dst, const int dst_stride,
                                            AfterRows after_rows)
{
    constexpr u32 CH = 16u * ZF_PRODUCERS;
    // Row pairs are visited from the bottom (rows 6-7) to the top (rows 0-1): the first word of the LAST visited pair is then
    // the one that holds the DC coefficient and is simply what `carry` is left with -- no per-iteration selects.  acc collects
    // everything except that word's low half (all 63 AC coefficients); nz collects, one bit per pair, which pairs were
    // transformed (warp-uniform: bit 3 = rows 6-7 ... bit 0 = rows 0-1).
    u32 acc = 0, carry = 0, nz = 0;
#pragma unroll UNROLL
    for (int i = 96; i >= 0; i -= 32) {        // i = 32 * row pair: byte offset in the slot and in the table, 1/256 of the scratch offset
        u32 a0, a1, a2, a3, b0, b1, b2, b3;
        const u32 pa = sl ^ (u32)i;
        lds128(pa, a0, a1, a2, a3);
        lds128(pa ^ 16u, b0, b1, b2, b3);
        const u32 hi = a2 | a3 | b2 | b3, rest = a1 | b0 | b1 | hi;
        acc |= carry | rest;
        carry = a0;
        nz <<= 1;
        const u32 o = sc + (u32)i * (CH / 8u);
        // the pair is skipped when it is zero in every block of the warp (a zero row transforms to exact zeros) ...
        if (!__any_sync(0xffffffffu, (a0 | rest) != 0)) {
            if (i < 64) {                      // (rows 4-7: zeroed below, and only if the column pass will read them)
#pragma unroll
                for (int k = 0; k < 4; k++) sts128(o + (u32)k * CH, 0u, 0u, 0u, 0u);
            }
            continue;
        }
        nz |= 1u;
        // ... and uses the 4-input form when nothing sits in columns 4-7
        const bool anyhi = __any_sync(0xffffffffu, hi != 0);
        const uint4 qa = *reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(qtw) + i), qb = *reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(qtw) + i + 16);
        u32 s0 = dp2a_lo(a0, qa.x), s1 = dp2a_hi(a0, qa.x), s2 = dp2a_lo(a1, qa.y), s3 = dp2a_hi(a1, qa.y), s4 = 0, s5 = 0, s6 = 0, s7 = 0;
        u32 t0 = dp2a_lo(b0, qb.x), t1 = dp2a_hi(b0, qb.x), t2 = dp2a_lo(b1, qb.y), t3 = dp2a_hi(b1, qb.y), t4 = 0, t5 = 0, t6 = 0, t7 = 0;
        if (anyhi) {
            s4 = dp2a_lo(a2, qa.z); s5 = dp2a_hi(a2, qa.z); s6 = dp2a_lo(a3, qa.w); s7 = dp2a_hi(a3, qa.w);
            t4 = dp2a_lo(b2, qb.z); t5 = dp2a_hi(b2, qb.z); t6 = dp2a_lo(b3, qb.w); t7 = dp2a_hi(b3, qb.w);
            idct8<10>(s0, s1, s2, s3, s4, s5, s6, s7, 512u);
            idct8<10>(t0, t1, t2, t3, t4, t5, t6, t7, 512u);
        } else {
            idct8_lo4<10>(s0, s1, s2, s3, s4, s5, s6, s7, 512u);
            idct8_lo4<10>(t0, t1, t2, t3, t4, t5, t6, t7, 512u);
        }
        sts128(o, s0, s1, s2, s3);
        sts128(o + CH, s4, s5, s6, s7);
        sts128(o + 2 * CH, t0, t1, t2, t3);
        sts128(o + 3 * CH, t4, t5, t6, t7);
    }
    acc |= carry & 0xffff0000u;
    const u32 dc0 = carry;
    const bool rows45 = (nz & 4u) != 0, rows67 = (nz & 8u) != 0;
    const bool rows47 = rows45 || rows67;
    if (rows47 && !(rows45 && rows67) && !(LO6 && rows45)) {       // the 8-input column pass reads rows 4-7: zero the pair that was skipped
        const u32 o = sc + (u32)(rows45 ? 12 : 8) * CH;
#pragma unroll
        for (int k = 0; k < 4; k++) sts128(o + (u32)k * CH, 0u, 0u, 0u, 0u);
    }
    __syncwarp();
    after_rows();                             // every lane of the warp is done with its staging slot
    // all 63 AC coefficients zero: ((c0 as i16).wrapping_mul(q0 as i16) >> 3) + 128 in i16, clamped (avx2.rs:159-167) --
    // not what the full transform gives (Q3), so it is a per-block decision
    const bool dconly = acc == 0;
    const int dc = (int)(int16_t)(dc0 & 0xffffu), q0 = (int)(int16_t)(qtw[0] & 0xffu);
    int v = (int)(int16_t)(dc * q0);
    v = (int)(int16_t)((v >> 3) + 128);
    const u32 dcword = (u32)max(min(v, 255), 0) * 0x01010101u;
    if (!rows47) {                            // rows 4-7 are zero in every block of the warp
#pragma unroll 1
        for (int g = 0; g < 2; g++) col_pass<4>(active, dconly, dcword, sc + (u32)g * CH, dst + 4 * g, dst_stride);
    } else {
        if (LO6 && !rows67) {                 // rows 6-7 are zero in every block of the warp (five luma jobs in six of a quality-90 photo)
#pragma unroll 1
            for (int g = 0; g < 2; g++) col_pass<6>(active, dconly, dcword, sc + (u32)g * CH, dst + 4 * g, dst_stride);
        } else {
#pragma unroll 1
            for (int g = 0; g < 2; g++) col_pass<8>(active, dconly, dcword, sc + (u32)g * CH, dst + 4 * g, dst_stride);
        }
    }
}

// ------------------------------------------------------------------------------------------- tile geometry
template <int MODE> struct ModeTraits;
template <> struct ModeTraits<MODE_NONE> { static constexpr int H = 1, V = 1, YBR = 1, CBR = 1, TM = TM_NONE, HALO = 0; };
template <> struct ModeTraits<MODE_H>    { static constexpr int H = 2, V = 1, YBR = 2, CBR = 2, TM = TM_H,    HALO = 1; };
template <> struct ModeTraits<MODE_V>    { static constexpr int H = 1, V = 2, YBR = 2, CBR = 1, TM = TM_V,    HALO = 0; };
template <> struct ModeTraits<MODE_HV>   { static constexpr int H = 2, V = 2, YBR = 4, CBR = 2, TM = TM_HV,   HALO = 1; };

// Chroma samples of the strip as the reference's up-samplers see them: a FLAT array of CROWS*W samples
// (row-major).  In shared memory a row holds [left halo block | tile columns | right halo block | special
// block]; the halo blocks wrap around the image (the flat filters run across row ends, SURVEY Q4a).
template <typename ST>
struct ChromaView {
    const ST *base;  // smem plane of one component
    int W;           // chroma row width in the image
    int n;           // CROWS * W
    int c0, c1;      // tile column range [c0, c1)
    int lhb, rhb, spb;  // block columns held in the left / right / special halo slots (-1 = none)
    int cs;          // smem row stride (samples)
    unsigned long long magic_w;  // ceil(2^40 / W)
    __device__ __noinline__ int at(int row, int col) const   // the leaf every generic sample fetch goes through stays a call (code size)
    {
        int lc;
        if (col >= c0 && col < c1) lc = 8 + (col - c0);
        else if ((col >> 3) == lhb) lc = col & 7;
        else if ((col >> 3) == rhb) lc = 8 + (c1 - c0) + (col & 7);
        else lc = 16 + (c1 - c0) + (col & 7);  // special slot (col >> 3 == spb)
        return (int)base[row * cs + lc];
    }
    __device__ __forceinline__ int flat(int idx) const
    {
        const int row = (int)(((unsigned long long)(unsigned)idx * magic_w) >> 40);  // idx / W without a divide
        return at(row, idx - row * W);
    }
    // `.get(i).unwrap_or(&0)` of upsampler/avx2.rs:264-270
    __device__ __forceinline__ int flat_or0(int idx) const { return (idx >= 0 && idx < n) ? flat(idx) : 0; }
};

__device__ __forceinline__ int T3(int a, int b) { return (3 * a + b + 2) >> 2; }  // (3a + b + 2) >> 2

// ---- H, flat strip of n = 16*W samples, output index o in [0, 2n)        (upsampler/scalar.rs:5-60, sse.rs:24-134)
template <int VARIANT, typename ST>
__device__ int up_h(const ChromaView<ST> &v, int o)
{
    const int n = v.n;
    const int i = o >> 1;
    if (VARIANT == 0 && o >= 2 * n - 8) {  // Q4b: the SSE tail
        const int il = n - 4;
        switch (o - (2 * n - 8)) {
        case 0: return T3(v.flat(il), v.flat(il - 1));
        case 1: return T3(v.flat(il), v.flat(il + 1));
        case 2: return T3(v.flat(il + 1), v.flat(il));
        case 3: return v.flat(il + 1);
        case 4: return v.flat(il + 2);
        case 5: return T3(v.flat(il + 2), v.flat(il + 1));
        case 6: return T3(v.flat(il + 2), v.flat(il + 3));
        default: return v.flat(il + 3);
        }
    }
    if (o == 0) return v.flat(0);
    if (o == 1) return T3(v.flat(0), v.flat(1));
    if (VARIANT == 1) {
        if (o == 2 * n - 2) return T3(v.flat(n - 2), v.flat(n - 1));  // sic, scalar.rs:55
        if (o == 2 * n - 1) return v.flat(n - 1);
    }
    return (o & 1) ? T3(v.flat(i), v.flat(i + 1)) : T3(v.flat(i), v.flat(i - 1));
}

// ---- V, 8 rows in, 16 rows out, no neighbour-strip context (upsampler/scalar.rs:64-147, Q4c)
template <typename ST>
__device__ int up_v(const ChromaView<ST> &v, int yl, int x)
{
    if (yl < 2) return v.at(0, x);
    if (yl >= 14) return v.at(7, x);
    const int k = yl >> 1;
    const int a = v.at(k, x), b = v.at(k + 1, x);
    return (yl & 1) ? T3(b, a) : T3(a, b);
}

// ---- HV scalar = H(V(in)) with V seeing 8 double-rows of S = 2W samples (upsampler/scalar.rs:148-166, Q4d)
template <typename ST>
__device__ int hv_vo(const ChromaView<ST> &v, int f)
{
    const int S = 2 * v.W;
    const int d = (int)(((unsigned long long)(unsigned)f * v.magic_w) >> 40) >> 1, i = f - d * S, k = d >> 1;  // f / (2W)
    if (d < 2) return v.flat(i);
    if (d >= 14) return v.flat(7 * S + i);
    const int a = v.flat(k * S + i), b = v.flat((k + 1) * S + i);
    return (d & 1) ? T3(b, a) : T3(a, b);
}
template <typename ST>
__device__ int up_hv_scalar(const ChromaView<ST> &v, int o)
{
    const int n2 = 2 * v.n;  // length of the V output
    const int i = o >> 1;
    if (o == 0) return hv_vo(v, 0);
    if (o == 1) return T3(hv_vo(v, 0), hv_vo(v, 1));
    if (o == 2 * n2 - 2) return T3(hv_vo(v, n2 - 2), hv_vo(v, n2 - 1));
    if (o == 2 * n2 - 1) return hv_vo(v, n2 - 1);
    return (o & 1) ? T3(hv_vo(v, i), hv_vo(v, i + 1)) : T3(hv_vo(v, i), hv_vo(v, i - 1));
}

// ---- HV AVX2 closed form (upsampler/avx2.rs:29-342; SURVEY A.4 Q4e/f/g)
template <typename ST>
__device__ int up_hv_avx(const ChromaView<ST> &v, int o)
{
    const int S = v.n >> 3;  // input double-row length = 2W
    const int L = 2 * S;     // output double-row length
    const int d2 = (int)(((unsigned long long)(unsigned)o * v.magic_w) >> 40) >> 2;  // o / (4W)
    int e = o - d2 * L;
    const int j = d2 >> 1, far = d2 & 1;
    const int sj = (j == 0 || j == 7) ? 0 : S;
    if (far && e == 0) e = 1;  // avx2.rs:330
    int i = e >> 1;
    const int odd = e & 1;
    if (i >= S - 16) {  // last 32 outputs of the double-row: raw input shifted 17 samples left (avx2.rs:277-307,332-338)
        int k = i - (S - 16);
        if (k == 15) k = 14;
        const int c = (j + 1) * S - 33 + k + (far ? sj : 0);
        return odd ? T3(v.flat(c), v.flat(c + 1)) : T3(v.flat(c), v.flat(c - 1));
    }
    const int bj = j * S;
    auto R = [&](int ii) {
        const int a = v.flat(bj + ii), b = v.flat(bj + ii + sj);
        return far ? T3(b, a) : T3(a, b);
    };
    const int lane = i & 15, t = i >> 4;
    int m;
    if (!odd) {
        if (lane != 0) m = R(i - 1);
        else if (t >= 1) { const int p = bj + 16 * t; m = (3 * (v.flat_or0(p) + v.flat_or0(p + sj) + 2)) >> 2; }
        else if (j == 0) m = v.flat(0);
        else { const int p = bj - 16, s = (j - 1 == 0) ? 0 : S; m = (3 * (v.flat_or0(p) + v.flat_or0(p + s) + 2)) >> 2; }
    } else {
        if (lane != 15) m = R(i + 1);
        else if (t >= 1) { const int p = bj + 16 * t + 16; m = (3 * (v.flat_or0(p) + v.flat_or0(p + sj) + 2)) >> 2; }
        else if (j == 0) m = v.flat(16);
        else { const int p = bj, s = (j - 1 == 0) ? 0 : S; m = (3 * (v.flat_or0(p) + v.flat_or0(p + s) + 2)) >> 2; }
    }
    return T3(R(i), m);
}

// One up-sampled chroma value at strip row yl, luma column x (generic, per-sample path).
template <int MODE, int VARIANT, typename ST>
__device__ __forceinline__ int chroma_at(const ChromaView<ST> &v, int yl, int x, int Wp, int hv_avx)
{
    if (MODE == MODE_NONE) return v.at(yl, x);
    if (MODE == MODE_V) return up_v(v, yl, x);
    const int o = yl * Wp + x;
    if (MODE == MODE_H) return up_h<VARIANT>(v, o);
    if (VARIANT == 0 && hv_avx) return up_hv_avx(v, o);
    return up_hv_scalar(v, o);
}

// conv16 per pixel: color_convert/scalar.rs:66-85 == avx.rs:123-192 (wrapping i16)
__device__ __forceinline__ void ycc_to_rgb(int y, int cb, int cr, u32 &r, u32 &g, u32 &b)
{
    const int cbb = (int)(int16_t)(cb - 128), crr = (int)(int16_t)(cr - 128);
    const int rr = (int)(int16_t)(y + ((int)(int16_t)(45 * crr) >> 5));
    const int gg = (int)(int16_t)(y - ((int)(int16_t)((int)(int16_t)(11 * cbb) + (int)(int16_t)(23 * crr)) >> 5));
    const int bb = (int)(int16_t)(y + ((int)(int16_t)(113 * cbb) >> 6));
    r = (u32)max(min(rr, 255), 0);
    g = (u32)max(min(gg, 255), 0);
    b = (u32)max(min(bb, 255), 0);
}


// ------------------------------------------------------------------------- generic (edge) path
// Every quirk of the reference, any variant, one sample at a time; only edge units of a tile come here.
// slow_pixel used to be kept out of line.  With that call inside a consumer warp, compute-sanitizer's synccheck reported
// divergent threads at the next named barrier (results and racecheck were clean); inlined -- only its leaf ChromaView::at
// stays a call, which keeps the hot loop of the kernel small enough for the instruction cache -- memcheck, racecheck and
// synccheck are all clean and the headline config is no slower (tools/sanitize_cases.py).
template <typename ST>
struct SlowCtx {
    ChromaView<ST> cv[2];
    const ST *sY;
    uint8_t *out;
    int twy, X0, Wp, hv_avx;
    u32 y_base, height, stride, n_norm, T, width, nc;
    bool ycc;
};

template <int MODE, int VARIANT, typename ST>
__device__ __forceinline__ void slow_pixel(const SlowCtx<ST> &c, int yl, int x)  // x = tile-local luma column
{
    const u32 y = c.y_base + yl;
    if (y >= c.height) return;                 // rows past the image are truncated (mcu.rs:375)
    uint8_t *row = c.out + (size_t)y * c.stride;
    const u32 T = c.T;
    const int s = c.X0 + x;                    // sample (luma column) in the padded row
    const bool normal = (u32)s < c.n_norm;
    const bool tail = (T != 0xffffffffu) && s >= c.Wp - 16;
    if (!normal && !tail) return;
    const int yy = (int)c.sY[yl * c.twy + x];
    const int cb = chroma_at<MODE, VARIANT, ST>(c.cv[0], yl, s, c.Wp, c.hv_avx);
    const int cr = chroma_at<MODE, VARIANT, ST>(c.cv[1], yl, s, c.Wp, c.hv_avx);
    u32 px[3];
    if (c.ycc) { px[0] = (u32)yy & 0xff; px[1] = (u32)cb & 0xff; px[2] = (u32)cr & 0xff; }  // `as u8`
    else ycc_to_rgb(yy, cb, cr, px[0], px[1], px[2]);
    if (normal) {
#pragma unroll
        for (int ch = 0; ch < 3; ch++) { const u32 b = 3 * s + ch; if (!(b >= T && b < T + 48)) row[b] = (uint8_t)px[ch]; }
    }
    if (tail) {
#pragma unroll
        for (int ch = 0; ch < 3; ch++) row[T + 3 * (s - (c.Wp - 16)) + ch] = (uint8_t)px[ch];
    }
}

// width < 16: the first 16 samples (zero-padded past Wp) are converted into a 16*nc-byte temp and its first
// width*nc bytes are copied out (worker.rs:176-198).  A single tile covers the row.
template <int MODE, int VARIANT, typename ST>
__device__ __forceinline__ void slow_small_width(const SlowCtx<ST> &c, int rows, int tid)
{
    const u32 rowbytes = c.width * c.nc;
    for (int u = tid; u < rows * 16; u += ZJ_THREADS) {
        const int yl = u >> 4, s = u & 15;
        const u32 y = c.y_base + yl;
        if (y >= c.height) continue;
        int yy = 0, cb = 0, cr = 0;
        if (s < c.Wp) {
            yy = (int)c.sY[yl * c.twy + s];
            cb = chroma_at<MODE, VARIANT, ST>(c.cv[0], yl, s, c.Wp, c.hv_avx);
            cr = chroma_at<MODE, VARIANT, ST>(c.cv[1], yl, s, c.Wp, c.hv_avx);
        }
        u32 px[3];
        ycc_to_rgb(yy, cb, cr, px[0], px[1], px[2]);
        uint8_t *row = c.out + (size_t)y * c.stride;
#pragma unroll
        for (int ch = 0; ch < 3; ch++) { const u32 b = 3 * s + ch; if (b < rowbytes) row[b] = (uint8_t)px[ch]; }
        if (s == 0) for (u32 b = 48; b < rowbytes; b++) row[b] = 0;
    }
}

// ------------------------------------------------------------------------------------ packed fast path
// Interior units (everything but the image / strip / AVX2-vector edge cases listed at the call site) are
// computed 8 pixels at a time on 16x2 lane pairs: VIADD.16x2 / VIMNMX.S16x2.RELU clamp two lanes per
// instruction, IDP.2A evaluates 3a+b+2 of the triangle filter in one instruction, PRMT does all byte traffic.
// Only for the X86 variant (its samples are clamped to [0,255] and live as bytes in shared memory).
__device__ __forceinline__ u32 prmt(u32 a, u32 b, u32 s) { return __byte_perm(a, b, s); }
__device__ __forceinline__ u32 lanes01(u32 w) { return prmt(w, 0u, 0x4140u); }  // bytes 0,1 -> 16-bit lanes
__device__ __forceinline__ u32 lanes23(u32 w) { return prmt(w, 0u, 0x4342u); }  // bytes 2,3 -> 16-bit lanes
__device__ __forceinline__ u32 vadd2(u32 a, u32 b) { u32 d; asm("add.s16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ u32 maxu2(u32 a, u32 b) { u32 d; asm("max.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ u32 minu2(u32 a, u32 b) { u32 d; asm("min.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ u32 minrelu2(u32 a, u32 b) { u32 d; asm("min.relu.s16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ u32 dp2a_u(u32 a, u32 b, u32 c) { u32 d; asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
// T(a,b) = (3a + b + 2) >> 2 on both lanes (values <= 255, so no lane overflows)
__device__ __forceinline__ u32 T2(u32 a, u32 b) { return ((a * 3u + b + 0x00020002u) >> 2) & 0x00ff00ffu; }

// Horizontal x2 triangle filter of four samples R0..R3 with neighbours R(-1), R4:
//   out[2i] = T(R[i], R[i-1]), out[2i+1] = T(R[i], R[i+1])    (upsampler/scalar.rs:30-42 == avx2.rs:178-197)
// h = (R(-1), R4), a = (R0, R1), b = (R2, R3) as lane pairs; o[k] = (out[2k], out[2k+1]) as lane pairs.
__device__ __forceinline__ void hfilter8(u32 h, u32 a, u32 b, u32 o[4])
{
    const u32 W13 = 0x0301u, W31 = 0x0103u;                                  // lane0*1 + lane1*3 / lane0*3 + lane1*1
    const u32 qm1 = prmt(h, a, 0x5410u);                                      // (R(-1), R0)
    const u32 q1 = prmt(a, b, 0x5432u);                                       // (R1, R2)
    const u32 q3 = prmt(b, h, 0x7632u);                                       // (R3, R4)
    const u32 o0 = dp2a_u(qm1, W13, 2u), o1 = dp2a_u(a, W31, 2u), o2 = dp2a_u(a, W13, 2u), o3 = dp2a_u(q1, W31, 2u);
    const u32 o4 = dp2a_u(q1, W13, 2u), o5 = dp2a_u(b, W31, 2u), o6 = dp2a_u(b, W13, 2u), o7 = dp2a_u(q3, W31, 2u);
    // pack two results into lanes, shift both at once, mask off the bits that crossed the lane boundary
    // (results reach 287 when a mis-scaled lane-0/15 neighbour is involved, hence 9-bit lanes)
    o[0] = ((o0 + (o1 << 16)) >> 2) & 0x01ff01ffu;
    o[1] = ((o2 + (o3 << 16)) >> 2) & 0x01ff01ffu;
    o[2] = ((o4 + (o5 << 16)) >> 2) & 0x01ff01ffu;
    o[3] = ((o6 + (o7 << 16)) >> 2) & 0x01ff01ffu;
}

// conv16 on lane pairs (color_convert/avx.rs:123-192), exact for y in [0,255], cb/cr in [0,287]:
//   r = clamp(y + ((45*(cr-128)) >> 5))           = clamp((32y + 45cr - 5760) >> 5)
//   g = clamp(y - ((11*(cb-128)+23*(cr-128)) >> 5)) = clamp((32y - 11cb - 23cr + 4352 + 31) >> 5)   [-floor(t/32) = floor((31-t)/32)]
//   b = clamp(y + ((113*(cb-128)) >> 6))          = clamp((64y + 113cb - 14464) >> 6)
// clamping before the shift (to 255*32+31 / 255*64+63) equals clamping after it.  Results: bytes 0 and 2.
__device__ __forceinline__ void convert_pair(u32 y, u32 cb, u32 cr, u32 &r, u32 &g, u32 &b)
{
    const u32 y32 = y << 5;
    r = minrelu2(vadd2(cr * 45u + y32, 0xE980E980u), 0x1FFF1FFFu) >> 5;                          // -5760
    g = minrelu2(vadd2(y32 + 0x331F331Fu - cb * 11u - cr * 23u, 0xDE00DE00u), 0x1FFF1FFFu) >> 5;  // +13087, then -8704
    // 64y + 113cb reaches 48751 (> i16 range), so this channel is clamped as unsigned lanes: [14464, 30847] - 14464
    b = (minu2(maxu2(cb * 113u + (y32 << 1), 0x38803880u), 0x787F787Fu) - 0x38803880u) >> 6;
}

// The same with the results left in bytes 1 and 3: the final `>> 5` / `>> 6` (a shift: ALU pipe, the busier one in the
// consumers) becomes `* 8` / `* 4` on lanes that are already clamped to 13 / 14 bits (a multiply: FMA pipe), and the byte
// interleave picks bytes 1 and 3 instead of 0 and 2.  The blue channel is clamped from above as unsigned lanes first
// (64y + 113cb reaches 48751), then shifted down by 14464 and clamped at zero as signed lanes: one instruction fewer.
// Every channel is biased so that ONE lane constant (k = -16384, kept in a register by the caller) brings it back: the biases
// ride on immediates of 32-bit adds (all lanes stay inside [0, 65535], so the lanes never carry into each other).  Red and
// green share y32g = 32y + 20767 (one LEA; 20767 = 16384 + 4352 + 31); red's lane constant takes the difference back
// (kr = -5760 - 20767, the lane-wise add wraps mod 2^16 and the true result lies in [-5760, 15315]).
__device__ __forceinline__ void convert_pair_hi(u32 y, u32 cb, u32 cr, u32 &r, u32 &g, u32 &b, const u32 k, const u32 kr)
{
    const u32 y32g = y * 32u + 0x511F511Fu;
    r = minrelu2(vadd2(cr * 45u + y32g, kr), 0x1FFF1FFFu) * 8u;
    g = minrelu2(vadd2(y32g - cb * 11u - cr * 23u, k), 0x1FFF1FFFu) * 8u;
    b = minrelu2(vadd2(minu2(cb * 113u + y * 64u + 0x07800780u, 0x7FFF7FFFu), k), 0x3FFF3FFFu) * 4u;   // +1920 = 16384 - 14464
}

// 8 pixels -> 24 interleaved bytes.  c0/c1/c2 hold channel pairs with the values in bytes 0 and 2.
__device__ __forceinline__ void pack24(const u32 c0[4], const u32 c1[4], const u32 c2[4], u32 w[6])
{
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const u32 rg0 = prmt(c0[2 * h], c1[2 * h], 0x6240u);          // [R0 G0 R1 G1]
        const u32 rg1 = prmt(c0[2 * h + 1], c1[2 * h + 1], 0x6240u);  // [R2 G2 R3 G3]
        w[3 * h] = prmt(rg0, c2[2 * h], 0x2410u);                      // [R0 G0 B0 R1]
        w[3 * h + 1] = prmt(prmt(rg0, c2[2 * h], 0x0063u), rg1, 0x5410u);  // [G1 B1 R2 G2]
        w[3 * h + 2] = prmt(rg1, c2[2 * h + 1], 0x6324u);              // [B2 R3 G3 B3]
    }
}

__device__ __forceinline__ void emit8(uint8_t *dst, const u32 y[4], const u32 cb[4], const u32 cr[4], bool ycc, int nwords)
{
    u32 w[6];
    if (ycc) {
        pack24(y, cb, cr, w);  // `as u8` interleave (color_convert/scalar.rs:152-161)
    } else {
        u32 r[4], g[4], b[4];
#pragma unroll
        for (int k = 0; k < 4; k++) convert_pair(y[k], cb[k], cr[k], r[k], g[k], b[k]);
        pack24(r, g, b, w);
    }
    if (nwords == 6 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
        uint2 *d = reinterpret_cast<uint2 *>(dst);
        d[0] = make_uint2(w[0], w[1]); d[1] = make_uint2(w[2], w[3]); d[2] = make_uint2(w[4], w[5]);
    } else {
        u32 *d = reinterpret_cast<u32 *>(dst);
#pragma unroll
        for (int k = 0; k < 6; k++) if (k < nwords) d[k] = w[k];
    }
}

__device__ __forceinline__ void load_y8(const uint8_t *p, u32 y[4])
{
    const uint2 v = *reinterpret_cast<const uint2 *>(p);
    y[0] = lanes01(v.x); y[1] = lanes23(v.x); y[2] = lanes01(v.y); y[3] = lanes23(v.y);
}

// --------------------------------------------------------------------------------------- the fused kernel
// grid = (tiles, strips [+1 when rows are dropped], images of this launch group); block = ZJ_THREADS.
template <int MODE, int VARIANT>
__global__ void __launch_bounds__(ZJ_THREADS, ZJ_MINBLOCKS)
reconstruct_kernel(const DevImage *__restrict__ images)
{
    typedef ModeTraits<MODE> MT;
    typedef typename std::conditional<VARIANT == 0, uint8_t, int16_t>::type ST;
    constexpr int ROWS = 8 * MT::H * MT::V;   // output rows per strip (mcu.rs:226)
    constexpr int YROWS = 8 * MT::YBR;        // == ROWS
    constexpr int CROWS = 8 * MT::CBR;
    constexpr int TWY = 8 * MT::H * MT::TM;   // luma tile width (samples)
    constexpr int TWC = 8 * MT::TM;           // chroma tile width
    constexpr int CS = TWC + 24;              // chroma smem row: halo | tile | halo | special
    static_assert(YROWS == ROWS, "luma rows");
    static_assert(MT::YBR * MT::H * MT::TM + 2 * (MT::CBR * MT::TM + (MT::HALO ? 3 * MT::CBR : 0)) <= ZJ_THREADS, "one 8x8 block per thread");

    __shared__ __align__(16) ST sY[YROWS * TWY];
    __shared__ __align__(16) ST sC[2][CROWS * CS];
    __shared__ u32 sQ[3][32];
    __shared__ int sSlowN;
    __shared__ unsigned short sSlow[ZJ_SLOW_CAP];  // edge units left to the generic path (row group << 8 | x unit)

    const DevImage &im = images[blockIdx.z];
    const u32 tile = blockIdx.x, strip = blockIdx.y;
    if (tile >= im.n_tiles) return;
    const int tid = threadIdx.x;
    const u32 stride = im.stride;
    uint8_t *__restrict__ out = im.out;

    // rows below the last processed strip stay zero in the reference (Q1 dropped MCU row, mcu.rs:154,158)
    if (strip >= im.n_strips) {
        if (strip > im.n_strips) return;
        const size_t lo = (size_t)im.n_strips * ROWS * stride, hi = (size_t)im.height * stride;
        if (lo >= hi) return;
        const size_t span = hi - lo, per = (span + im.n_tiles - 1) / im.n_tiles;
        size_t b0 = lo + (size_t)tile * per, b1 = b0 + per;
        if (b1 > hi) b1 = hi;
        for (size_t b = b0 + tid; b < b1; b += ZJ_THREADS) out[b] = 0;
        return;
    }

    // tile -> MCU column range, spread evenly (first tile_r tiles one column wider) so every tile keeps >= TM/2 columns
    const int mcu_x = (int)im.mcu_x, nt = (int)im.n_tiles;
    const int m0 = (int)(tile * im.tile_q + min(tile, im.tile_r)), m1 = (int)((tile + 1) * im.tile_q + min(tile + 1, im.tile_r));
    const int tm = m1 - m0;                      // MCU columns in this tile (<= TM)
    const int Wp = (int)im.Wp, W = (int)im.W;
    const int ybpr = MT::H * mcu_x;              // luma blocks per block-row of the plane

    // ---------------------------------------------------------------- phase 1: IDCT into shared planes
    const int lhb = (MT::HALO && mcu_x > 0) ? (m0 == 0 ? mcu_x - 1 : m0 - 1) : -1;  // wraps: flat filters cross row ends
    const int rhb = MT::HALO ? (m1 == mcu_x ? 0 : m1) : -1;
    // AVX2 HV: lane-0 neighbour of the first vector of a double-row is a stale value taken 16 samples before
    // the end of the previous double-row (Q4f) -> tile 0 also needs block column mcu_x-2
    const int spb = (MODE == MODE_HV && VARIANT == 0 && im.hv_avx && m0 == 0 && nt > 1) ? mcu_x - 2 : -1;
    {
        const int nY = MT::YBR * MT::H * tm;
        const int nC = MT::CBR * tm;                  // per chroma component
        const int nHalo = MT::HALO ? MT::CBR : 0;     // per side per component
        const int nSp = spb >= 0 ? MT::CBR : 0;
        const int total = nY + 2 * (nC + 2 * nHalo + nSp);
        const int per = nC + 2 * nHalo + nSp;
        const float r_htm = __frcp_rn((float)(MT::H * tm)), r_tm = __frcp_rn((float)tm);
        {
            // total <= ZJ_THREADS (one block per thread); lanes without a block still take part in the warp votes
            const int b = tid;
            const bool active = b < total;
            const int16_t *src = nullptr;
            const u32 *qt = sQ[0];
            ST *dst = sY;
            int dstride = TWY;
            if (!active) {
            } else if (b < nY) {
                const int br = div_small(b, r_htm), bc = b - br * (MT::H * tm);
                const size_t blk = ((size_t)strip * MT::YBR + br) * ybpr + (size_t)MT::H * m0 + bc;
                src = im.coeff[0] + blk * 64; qt = sQ[0]; dst = sY + br * 8 * TWY + bc * 8; dstride = TWY;
            } else {
                int c = b - nY;
                const int comp = c >= per ? 1 : 0;
                c -= comp * per;
                int br, gcol, lcol;  // block row, global block column, smem column
                if (c < nC) { br = div_small(c, r_tm); const int bc = c - br * tm; gcol = m0 + bc; lcol = 8 + bc * 8; }
                else if (c < nC + nHalo) { br = c - nC; gcol = lhb; lcol = 0; }
                else if (c < nC + 2 * nHalo) { br = c - nC - nHalo; gcol = rhb; lcol = 8 + tm * 8; }
                else { br = c - nC - 2 * nHalo; gcol = spb; lcol = 16 + tm * 8; }
                const size_t blk = ((size_t)strip * MT::CBR + br) * mcu_x + gcol;
                src = im.coeff[1 + comp] + blk * 64; qt = sQ[1 + comp]; dst = sC[comp] + br * 8 * CS + lcol; dstride = CS;
            }
            // issue the coefficient loads first; the table copy and the barrier below overlap their latency
            int4 raw[8];
            load_block(active, src, raw);
            for (int k = tid; k < 96; k += ZJ_THREADS) sQ[k >> 5][k & 31] = im.qtw[k >> 5][k & 31];
            if (tid == 0) sSlowN = 0;
            __syncthreads();
            idct_block<VARIANT, ST>(active, raw, qt, dst, dstride);  // the only call site: one copy of the unrolled IDCT
        }
    }
    __syncthreads();

    // ---------------------------------------------------------------- phase 2: up-sample, convert, write
    const int X0 = m0 * 8 * MT::H;           // first luma column of the tile
    const int tw = tm * 8 * MT::H;           // luma columns in the tile
    const bool last_tile = (tile + 1 == (u32)nt);
    const u32 y_base = strip * ROWS;
    const u32 n_norm = im.n_norm, T = im.T, P = im.P;
    const bool ycc = im.out_kind == OUT_YCC;
    const int hv_avx = (int)im.hv_avx;
    // context of the generic path: built only by the CTAs that need it (edge tiles, SCALAR variant, ...)
    auto make_ctx = [&](SlowCtx<ST> &sc) {
#pragma unroll
        for (int c = 0; c < 2; c++) {
            sc.cv[c].base = sC[c]; sc.cv[c].W = W; sc.cv[c].n = CROWS * W;
            sc.cv[c].c0 = m0 * 8; sc.cv[c].c1 = m1 * 8; sc.cv[c].lhb = lhb; sc.cv[c].rhb = rhb; sc.cv[c].spb = spb; sc.cv[c].cs = CS; sc.cv[c].magic_w = im.magic_w;
        }
        sc.sY = sY; sc.twy = TWY; sc.X0 = X0; sc.Wp = Wp; sc.hv_avx = hv_avx; sc.y_base = y_base; sc.height = im.height;
        sc.stride = stride; sc.n_norm = n_norm; sc.T = T; sc.ycc = ycc; sc.out = out; sc.width = im.width; sc.nc = im.nc;
    };

    if (im.small_width) {
        SlowCtx<ST> sc;
        make_ctx(sc);
        slow_small_width<MODE, VARIANT, ST>(sc, ROWS, tid);
        return;
    }

    // A unit is 8 luma columns of one output row (NONE, H) or of the two rows that share their chroma inputs
    // (V: rows 2k,2k+1; HV: rows 4j+p and 4j+p+2, the near and far results of chroma row 2j+p).
    constexpr int RPU = (MODE == MODE_V || MODE == MODE_HV) ? 2 : 1;   // rows per unit
    constexpr int NRU = ROWS / RPU;                                    // row groups per strip
    const int xunits = tw >> 3;
    const bool fast_ok = (VARIANT == 0) && ((stride & 3u) == 0) && ((reinterpret_cast<uintptr_t>(out) & 3) == 0) && (MODE != MODE_HV || hv_avx);
    // thread -> fixed x unit, loop over row groups: everything that depends only on the column is hoisted
    const float r_xu = __frcp_rn((float)xunits);
    const int rpp = div_small(ZJ_THREADS, r_xu);   // row groups per pass
    const int r0 = div_small(tid, r_xu), xu = tid - r0 * xunits;
    const int xl = xu << 3;
    const int xs = X0 + xl;                        // first sample of the unit in the padded row
    const int cc0 = xs >> 1;                       // first chroma column (H, HV)
    // Where the unit's 24 bytes go in the output row (worker.rs:201-246, SURVEY A.5):
    //   samples < n_norm ("normal" 16-sample chunks) sit at byte 3*s, except bytes the tail chunk overwrites;
    //   samples >= Wp-16 (the tail chunk) sit at T + 3*(s - (Wp-16));  anything else is never written.
    int dst_off = 3 * xs;
    int nwords = 6;                                // words of the unit to store; 0 = nothing; -1 = leave to the generic path
    if ((u32)(xs + 8) <= n_norm) {
        if ((u32)(3 * xs + 24) > T && (u32)(3 * xs) < T + 48) {        // overlaps the tail chunk's bytes [T, T+48)
            const int keep = (int)T - 3 * xs;                            // bytes before T survive
            nwords = (keep > 0 && (keep & 3) == 0 && (u32)(3 * xs + 24) <= T + 48) ? (keep >> 2) : (keep <= 0 && (u32)(3 * xs + 24) <= T + 48 ? 0 : -1);
        }
    } else if (T != 0xffffffffu && xs >= Wp - 16) {
        dst_off = (int)T + 3 * (xs - (Wp - 16));
    } else if ((u32)xs >= n_norm && (T == 0xffffffffu || xs + 8 <= Wp - 16)) {
        nwords = 0;                                                      // e.g. the 8 samples between the last chunk and the tail when Wp % 16 == 8
    } else {
        nwords = -1;
    }
    if ((dst_off & 3) != 0) nwords = nwords > 0 ? -1 : nwords;
    // chroma window cc0-1 .. cc0+4: the flat filters run across image-row ends (Q4a), so the first / last unit of a
    // row takes its outer neighbour from the previous / next chroma row, which is what the wrapped halo blocks hold
    const bool first_x = (MODE == MODE_H || MODE == MODE_HV) && cc0 == 0;
    const bool last_x = (MODE == MODE_H || MODE == MODE_HV) && cc0 + 4 == W;
    for (int rg = r0; fast_ok && r0 < rpp && rg < NRU; rg += rpp) {
        int yl0, yl1;                              // strip rows of the unit
        if (MODE == MODE_V) { yl0 = 2 * rg; yl1 = yl0 + 1; }
        else if (MODE == MODE_HV) { yl0 = 4 * (rg >> 1) + (rg & 1); yl1 = yl0 + 2; }
        else { yl0 = rg; yl1 = rg; }
        bool fast = nwords >= 0;
        int l0 = 0;
        bool hv_tail = false;
        if (MODE == MODE_H) {
            // strip start (out[0], out[1] edge rule) and strip end (scalar.rs:46-57 / the SSE tail Q4b) stay generic
            fast = fast && !(first_x && rg == 0) && !(last_x && rg == NRU - 1);
        }
        if (MODE == MODE_HV) {
            const int p = rg & 1;
            l0 = (p * W + cc0) & 15;               // AVX2 lane of the unit's first sample
            hv_tail = p == 1 && cc0 + 4 > W - 16;  // last 32 outputs of an odd row: raw input shifted 17 samples left (Q4g)
            // generic only when the raw tail of a narrow last tile reaches outside it, or for images too narrow for the
            // first-vector rule below
            fast = fast && !(hv_tail && W - 36 < m0 * 8) && !(p == 0 && cc0 < 16 && W < 48);
        }
        if (nwords == 0 && fast) continue;         // nothing of this unit is ever written
        if (!fast) {
            // edge unit: queue it; all threads share the queued samples after the loop (a warp that ran the
            // generic code inline would serialise ~10^4 instructions behind one or two active lanes)
            const int slot = atomicAdd(&sSlowN, 1);
            if (slot < ZJ_SLOW_CAP) sSlow[slot] = (unsigned short)((rg << 8) | xu);  // (overflow: whole tile redone below)
            continue;
        }
        if constexpr (VARIANT == 0) {
            u32 cb0[4], cr0[4], cb1[4], cr1[4];    // chroma lane pairs of row 0 / row 1 of the unit
#pragma unroll
            for (int c = 0; c < 2; c++) {
                u32 *o0 = c == 0 ? cb0 : cr0, *o1 = c == 0 ? cb1 : cr1;
                const uint8_t *base = reinterpret_cast<const uint8_t *>(sC[c]);
                if (MODE == MODE_NONE) {
                    const uint2 v = *reinterpret_cast<const uint2 *>(base + yl0 * CS + 8 + xl);
                    o0[0] = lanes01(v.x); o0[1] = lanes23(v.x); o0[2] = lanes01(v.y); o0[3] = lanes23(v.y);
                } else if (MODE == MODE_V) {
                    // rows 2k, 2k+1 <- T(r_k, r_k+1), T(r_k+1, r_k); first and last pair replicate (scalar.rs:64-147)
                    const int ka = rg == 0 ? 0 : (rg == 7 ? 7 : rg), kb = rg == 0 ? 0 : (rg == 7 ? 7 : rg + 1);
                    const uint2 va = *reinterpret_cast<const uint2 *>(base + ka * CS + 8 + xl);
                    const uint2 vb = *reinterpret_cast<const uint2 *>(base + kb * CS + 8 + xl);
                    const u32 a[4] = {lanes01(va.x), lanes23(va.x), lanes01(va.y), lanes23(va.y)};
                    const u32 b[4] = {lanes01(vb.x), lanes23(vb.x), lanes01(vb.y), lanes23(vb.y)};
#pragma unroll
                    for (int k = 0; k < 4; k++) { o0[k] = T2(a[k], b[k]); o1[k] = T2(b[k], a[k]); }
                } else {
                    const int lc = 8 + (cc0 - m0 * 8);  // smem column of cc0 (multiple of 4)
                    // outer neighbours of the first / last unit of a row live one chroma row up / down (flat array)
                    const int off0 = (first_x && (MODE == MODE_H || (rg & 1))) ? -CS : 0, off2 = last_x ? CS : 0;
                    if (MODE == MODE_H) {
                        const uint8_t *pa = base + yl0 * CS + lc;
                        const u32 w0 = *reinterpret_cast<const u32 *>(pa - 4 + off0), w1 = *reinterpret_cast<const u32 *>(pa), w2 = *reinterpret_cast<const u32 *>(pa + 4 + off2);
                        hfilter8(prmt(w0, w2, 0x0403u) & 0x00ff00ffu, lanes01(w1), lanes23(w1), o0);
                    } else if (hv_tail) {
                        // out[O+2k] = T(in[c], in[c-1]), out[O+2k+1] = T(in[c], in[c+1]), c = (row end) - 33 + k: no vertical
                        // blend, raw row 2j+1 for the near row and row 2j+3 for the far row; k = 15 repeats k = 14
                        // (upsampler/avx2.rs:277-307,332-338)
                        const int j = rg >> 1, ra = 2 * j + 1, rb = (j == 0 || j == 7) ? ra : ra + 2;
                        const int q = (cc0 - (W - 16)) >> 2;                  // which 8 of the 32 outputs
                        const int lq = 8 + (W - 36 + 4 * q - m0 * 8);         // smem column of c - 3 for k = 4q (multiple of 4)
                        const u32 *pa = reinterpret_cast<const u32 *>(base + ra * CS + lq);
                        const u32 *pb = reinterpret_cast<const u32 *>(base + rb * CS + lq);
                        const u32 a0 = pa[0], a1 = pa[1], b0 = pb[0], b1 = pb[1];
                        hfilter8(prmt(a0, a1, 0x0702u) & 0x00ff00ffu, prmt(a0, a1, 0x0403u) & 0x00ff00ffu, prmt(a1, 0u, 0x4241u), o0);
                        hfilter8(prmt(b0, b1, 0x0702u) & 0x00ff00ffu, prmt(b0, b1, 0x0403u) & 0x00ff00ffu, prmt(b1, 0u, 0x4241u), o1);
                        if (q == 3) { o0[3] = o0[2]; o1[3] = o1[2]; }
                    } else {
                        // chroma row 2j+p blended with row 2j+p+2 (same row for the first / last double-row)
                        const int j = rg >> 1, ra = 2 * j + (rg & 1), rb = (j == 0 || j == 7) ? ra : ra + 2;
                        const uint8_t *pa = base + ra * CS + lc, *pb = base + rb * CS + lc;
                        const u32 a0 = *reinterpret_cast<const u32 *>(pa - 4 + off0), a1 = *reinterpret_cast<const u32 *>(pa), a2 = *reinterpret_cast<const u32 *>(pa + 4 + off2);
                        const u32 b0 = *reinterpret_cast<const u32 *>(pb - 4 + off0), b1 = *reinterpret_cast<const u32 *>(pb), b2 = *reinterpret_cast<const u32 *>(pb + 4 + off2);
                        const u32 Aa = lanes01(a1), Ab = lanes23(a1), Ah = prmt(a0, a2, 0x0403u) & 0x00ff00ffu;
                        const u32 Ba = lanes01(b1), Bb = lanes23(b1), Bh = prmt(b0, b2, 0x0403u) & 0x00ff00ffu;
                        u32 Nh = T2(Ah, Bh), Fh = T2(Bh, Ah);
                        // lane 0: the "previous" value is 3*(in+in'+2)>>2 of the vector's OWN first element (Q4e);
                        // lane 15: the "next" value is the same expression on the next vector's first element
                        const u32 pv = (3u * ((Aa & 0xffffu) + (Ba & 0xffffu) + 2u)) >> 2;
                        const u32 pf = ((3u * ((Ah >> 16) + (Bh >> 16) + 2u)) >> 2) << 16;
                        u32 pv2 = pv, pf2 = pf;
                        if ((rg & 1) == 0 && cc0 < 16) {
                            // first vector of a double-row (t = 0): its lane-0 / lane-15 neighbours are whatever the loop
                            // left behind (upsampler/avx2.rs:67-68,264-270; Q4f): for j = 0 the raw in[0] / in[16], for
                            // j >= 1 the values computed 16 samples before the end of double-row j-1 with ITS stride
                            if (j == 0) {
                                pv2 = Aa & 0xffffu;
                                pf2 = Ah & 0xffff0000u;
                            } else {
                                const int spc0 = (m0 == 0 && nt > 1) ? 16 + tm * 8 : 8 + (W - 16 - m0 * 8);  // smem column of chroma col W-16
                                const int rp = 2 * j - 1, rq = (j == 1) ? rp : rp + 2;                          // partner row: stride of double-row j-1
                                const u32 x0 = base[rp * CS + spc0], x1 = base[rq * CS + spc0];
                                pv2 = (3u * (x0 + x1 + 2u)) >> 2;
                                const int c0s = 8 - m0 * 8;                                                     // smem column of chroma col 0 (tile 0)
                                const u32 y0 = base[2 * j * CS + c0s], y1 = (j == 1) ? y0 : (j == 7 ? 0u : (u32)base[(2 * j + 2) * CS + c0s]);
                                pf2 = ((3u * (y0 + y1 + 2u)) >> 2) << 16;
                            }
                        }
                        const u32 keep = (l0 == 0 ? 0xffff0000u : 0xffffffffu) & (l0 == 12 ? 0x0000ffffu : 0xffffffffu);
                        const u32 ins = (l0 == 0 ? pv2 : 0u) | (l0 == 12 ? pf2 : 0u);
                        Nh = (Nh & keep) | ins;
                        Fh = (Fh & keep) | ins;
                        hfilter8(Nh, T2(Aa, Ba), T2(Ab, Bb), o0);
                        hfilter8(Fh, T2(Ba, Aa), T2(Bb, Ab), o1);
                        if ((rg & 1) == 0 && cc0 == 0) o1[0] = (o1[0] >> 16) * 0x00010001u;  // far rows: out[0] = out[1] (avx2.rs:330)
                    }
                }
            }
            const uint8_t *ybase = reinterpret_cast<const uint8_t *>(sY);
            u32 yv[4];
            if (y_base + yl0 < im.height) {
                load_y8(ybase + yl0 * TWY + xl, yv);
                emit8(out + (size_t)(y_base + yl0) * stride + dst_off, yv, cb0, cr0, ycc, nwords);
            }
            if (RPU == 2 && y_base + yl1 < im.height) {
                load_y8(ybase + yl1 * TWY + xl, yv);
                emit8(out + (size_t)(y_base + yl1) * stride + dst_off, yv, cb1, cr1, ycc, nwords);
            }
        }
    }
    __syncthreads();
    const int nslow = sSlowN;
    if (!fast_ok || nslow > ZJ_SLOW_CAP) {
        // SCALAR variant (i16 samples, unclamped DC-only values), odd strides, tiny 4:2:0 images (or a queue
        // overflow): every sample takes the generic path, one sample per thread
        SlowCtx<ST> sc;
        make_ctx(sc);
        for (int u = tid; u < ROWS * tw; u += ZJ_THREADS) {
            const int yl = u / tw;
            slow_pixel<MODE, VARIANT, ST>(sc, yl, u - yl * tw);
        }
    } else if (nslow > 0) {
        SlowCtx<ST> sc;
        make_ctx(sc);
        for (int t = tid; t < nslow * 8 * RPU; t += ZJ_THREADS) {
            const int e = sSlow[t / (8 * RPU)], r = (t >> 3) % RPU, k = t & 7;
            const int rg = e >> 8, xl2 = (e & 0xff) << 3;
            int yl;
            if (MODE == MODE_V) yl = 2 * rg + r;
            else if (MODE == MODE_HV) yl = 4 * (rg >> 1) + (rg & 1) + 2 * r;
            else yl = rg;
            slow_pixel<MODE, VARIANT, ST>(sc, yl, xl2 + k);
        }
    }
    // bytes of the row nobody writes: [P, stride) minus the tail chunk (Q5: 16 zero bytes; Q6: the w "alpha" bytes)
    if (last_tile) {
        const u32 nz = stride > P ? stride - P : 0;
        for (u32 u = tid; u < (u32)ROWS * nz; u += ZJ_THREADS) {
            const u32 yl = u / nz, b = P + (u - yl * nz);
            const u32 y = y_base + yl;
            if (y < im.height && !(b >= T && b < T + 48)) out[(size_t)y * stride + b] = 0;
        }
    }
}

// =========================================================================== the fast kernel (X86 variant)
// Same arithmetic as above, organised as a producer / consumer pipeline inside one CTA of 256 threads that owns one
// tile column of `spc` consecutive strips:
//   * warps 0-3 (producers) run the IDCT: two passes of one 8x8 block per thread fill the strip's sample planes in
//     shared memory (double-buffered);
//   * warps 4-7 (consumers) turn the planes into pixels: every thread produces two UNITS per strip, a unit being 16
//     luma columns (one conv16 chunk of the reference, color_convert/avx.rs:67-107) of one output row (NONE, H) or
//     of the two rows that share their chroma inputs (V, HV).
// The two halves meet only at named barriers (full / empty per buffer), so the integer-multiply-heavy IDCT of strip
// s+1 overlaps the byte-shuffling colour stage of strip s on every SM sub-partition.  Everything that depends only
// on the thread's position in the tile -- block pointers, the row writer's placement rule, the AVX2 lane of the unit,
// neighbour offsets -- is computed once, before the strip loop.  Units the packed code does not cover are queued
// once and handled per sample by the generic path (slow_pixel) in every strip.
template <int MODE> struct FastTraits {
    static constexpr int H = (MODE == MODE_H || MODE == MODE_HV) ? 2 : 1, V = (MODE == MODE_V || MODE == MODE_HV) ? 2 : 1;
    static constexpr int ROWS = 8 * H * V;            // output rows per strip (mcu.rs:226)
    static constexpr int YBR = H * V, CBR = H;        // block rows per strip: luma / chroma (SURVEY A.1 table)
    static constexpr int CROWS = 8 * CBR;
    static constexpr int RPU = V;                     // rows per unit
    static constexpr int NRG = ROWS / RPU;            // row groups per strip
    static constexpr int XU = MODE == MODE_H ? ZF_XU_H : 2 * ZF_CONSUMERS / NRG;   // unit columns per tile (two units per consumer thread; 4:2:2: see zj_device.h)
    static_assert(XU * NRG <= 2 * ZF_CONSUMERS, "two units per consumer thread");
    static constexpr int TWY = 16 * XU;               // luma samples per tile row
    static constexpr int TWC = TWY / H;               // chroma samples per tile row
    static constexpr int YB = TWY / 8, CB = TWC / 8;  // blocks per block row of the tile
    static constexpr int CS = TWC + 24;               // chroma smem row: left halo | tile | right halo | special
    static constexpr int NSLOT = MODE == MODE_H ? 2 : (MODE == MODE_HV ? 3 : 0);  // halo block columns per chroma plane
    // a 6-input column pass for jobs whose rows 6-7 are zero in every block of the warp: pays where the row-pair loop is rolled or
    // the strip is short (4:2:0 +1.1 %, 4:2:2 +0.6 %); with the unrolled loops of 4:4:4 / luma-only its code costs more than it saves
    static constexpr bool LO6 = MODE == MODE_HV || MODE == MODE_H;
    // row-pair loop of the IDCT: unrolled where the instruction cache has room for it (measured per mode); 4:2:0 / 4:4:0 stay
    // rolled, their consumers' hot code leaves no room in the 32 KB instruction cache for more (see idct_rolled)
    static constexpr int IDCT_UNROLL = (MODE == MODE_HV || MODE == MODE_V) ? 1 : 4;
    static constexpr int NY = YBR * YB, NC = CBR * CB, PER = NC + NSLOT * CBR;
    static constexpr int YBYTES = ROWS * TWY, CBYTES = CROWS * CS, BUF = YBYTES + 2 * CBYTES;  // one buffer of sample planes
    static_assert(NY + 2 * PER <= 2 * ZF_PRODUCERS, "two 8x8 blocks per producer thread");
    // block rows of 32 / 16 blocks are staged by cooperative, fully coalesced copies of whole runs; any other width packs the
    // list densely (a job of 32 consecutive entries then spans several runs and planes) and every lane copies its own block
    static constexpr bool DENSE = (YB % 16) != 0;
    static_assert(BUF % 16 == 0 && YBYTES % 16 == 0 && CBYTES % 8 == 0, "plane alignment");
};

// n = T(a, b), f = T(b, a) on both lanes, sharing a + b + 2:  3a + b + 2 = (a + b + 2) + 2a
__device__ __forceinline__ void T2pair(u32 a, u32 b, u32 &n, u32 &f)
{
    const u32 s = a + b + 0x00020002u;
    n = ((s + 2u * a) >> 2) & 0x00ff00ffu;
    f = ((s + 2u * b) >> 2) & 0x00ff00ffu;
}
// 4:2:0 packed path: the vertical blend hands 4 * T(a, b) to the horizontal filter instead of T(a, b), and the `>> 2` of the
// blend becomes part of the filter's own shift --
//   (3 * 4N + 4L + 8) >> 4  ==  (3N + L + 2) >> 2      (exact: everything is a multiple of 4)
// which takes two shifts out of every T2pair.  Lanes stay below 3 * 1536 + 1536 + 8 = 6152.
__device__ __forceinline__ void T2pair_s(u32 a, u32 b, u32 &n, u32 &f)
{
    const u32 s = a + b + 0x00020002u;
    n = (s + 2u * a) & 0xFFFCFFFCu;
    f = (s + 2u * b) & 0xFFFCFFFCu;
}
__device__ __forceinline__ u32 evens(u32 w) { return prmt(w, 0u, 0x4240u); }  // bytes 0,2 -> 16-bit lanes
__device__ __forceinline__ u32 odds(u32 w) { return prmt(w, 0u, 0x4341u); }   // bytes 1,3 -> 16-bit lanes

// named barriers (id 0 is __syncthreads); count = every thread of the CTA: one half arrives, the other half waits
// (bar.sync / bar.arrive are warp-aligned instructions: the warp is re-converged first -- the generic per-sample path and
// the zero-fill loops leave lanes of a consumer warp at different places)
__device__ __forceinline__ void bar_sync(int id) { __syncwarp(); asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(ZF_THREADS) : "memory"); }
__device__ __forceinline__ void bar_sync_consumers(int id) { __syncwarp(); asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(ZF_CONSUMERS) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id) { __syncwarp(); asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(ZF_THREADS) : "memory"); }

// Horizontal x2 triangle filter of eight samples R0..R7 (r[k] = (R2k, R2k+1) as lane pairs) with outer neighbours
// h = (R(-1), R8):  out[2i] = T(R[i], R[i-1]), out[2i+1] = T(R[i], R[i+1])  (upsampler/scalar.rs:30-42 == avx2.rs:178-197)
// Results as E[k] = (out[4k], out[4k+2]), O[k] = (out[4k+1], out[4k+3]); lanes are 9 bits wide because a mis-scaled
// lane-0/15 neighbour (Q4e) can push a result to 287.
__device__ __forceinline__ void hfilter16(u32 h, const u32 r[4], u32 E[4], u32 O[4])
{
    u32 L[5];
    L[0] = prmt(h, r[0], 0x5410u);       // (R(-1), R0)
    L[1] = prmt(r[0], r[1], 0x5432u);    // (R1, R2)
    L[2] = prmt(r[1], r[2], 0x5432u);
    L[3] = prmt(r[2], r[3], 0x5432u);
    L[4] = prmt(r[3], h, 0x7632u);       // (R7, R8)
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u32 p3 = r[k] * 3u + 0x00020002u;
        E[k] = ((p3 + L[k]) >> 2) & 0x01ff01ffu;
        O[k] = ((p3 + L[k + 1]) >> 2) & 0x01ff01ffu;
    }
}

// the same filter on inputs scaled by 4 (r[k], h = 4 * sample, see T2pair_s); results are the unscaled ones of hfilter16
__device__ __forceinline__ void hfilter16_s(u32 h, const u32 r[4], u32 E[4], u32 O[4])
{
    u32 L[5];
    L[0] = prmt(h, r[0], 0x5410u);
    L[1] = prmt(r[0], r[1], 0x5432u);
    L[2] = prmt(r[1], r[2], 0x5432u);
    L[3] = prmt(r[2], r[3], 0x5432u);
    L[4] = prmt(r[3], h, 0x7632u);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u32 p3 = r[k] * 3u + 0x00080008u;
        E[k] = ((p3 + L[k]) >> 4) & 0x01ff01ffu;
        O[k] = ((p3 + L[k + 1]) >> 4) & 0x01ff01ffu;
    }
}

// 16 pixels of one row -> 48 interleaved bytes.  yw: the 16 luma bytes; cbE/cbO/crE/crO: chroma in the E/O
// arrangement of hfilter16.  nw = number of leading 32-bit words to store (12, or fewer when the row's tail chunk
// overwrites the rest, worker.rs:221-246); vec = 16-byte stores are aligned.
__device__ __forceinline__ void emit16(uint8_t *dst, const u32 yw[4], const u32 cbE[4], const u32 cbO[4], const u32 crE[4], const u32 crO[4],
                                       const bool ycc, const int nw, const bool vec, const u32 sel, const u32 kk, const u32 kr = 0u)
{
    // sel: byte selector of the first interleave step (the channel values sit in bytes 1 and 3 after convert_pair_hi, in bytes
    // 0 and 2 otherwise); kk: the lane constant of convert_pair_hi -- both held in registers by the caller
    u32 w[12];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u32 yE = evens(yw[k]), yO = odds(yw[k]);
        u32 c0E, c1E, c2E, c0O, c1O, c2O;
        if (ycc) {  // `as u8` interleave (color_convert/scalar.rs:152-161)
            c0E = yE; c1E = cbE[k]; c2E = crE[k]; c0O = yO; c1O = cbO[k]; c2O = crO[k];
        } else {
            convert_pair_hi(yE, cbE[k], crE[k], c0E, c1E, c2E, kk, kr);
            convert_pair_hi(yO, cbO[k], crO[k], c0O, c1O, c2O, kk, kr);
        }
        const u32 rgE = prmt(c0E, c1E, sel);   // [R0 G0 R2 G2]
        const u32 brO = prmt(c2E, c0O, sel);   // [B0 R1 B2 R3]
        const u32 gbO = prmt(c1O, c2O, sel);   // [G1 B1 G3 B3]
        w[3 * k] = prmt(rgE, brO, 0x5410u);        // [R0 G0 B0 R1]
        w[3 * k + 1] = prmt(gbO, rgE, 0x7610u);    // [G1 B1 R2 G2]
        w[3 * k + 2] = prmt(brO, gbO, 0x7632u);    // [B2 R3 G3 B3]
    }
    if (ZF_LIKELY(vec && nw == 12)) {
        uint4 *d = reinterpret_cast<uint4 *>(dst);
        d[0] = make_uint4(w[0], w[1], w[2], w[3]); d[1] = make_uint4(w[4], w[5], w[6], w[7]); d[2] = make_uint4(w[8], w[9], w[10], w[11]);
    } else if (vec && nw == 8) {
        uint4 *d = reinterpret_cast<uint4 *>(dst);
        d[0] = make_uint4(w[0], w[1], w[2], w[3]); d[1] = make_uint4(w[4], w[5], w[6], w[7]);
    } else {
        u32 *d = reinterpret_cast<u32 *>(dst);
#pragma unroll
        for (int k = 0; k < 12; k++) if (k < nw) d[k] = w[k];
    }
}

__device__ __forceinline__ void load16(const uint8_t *p, const bool a16, u32 w[4])
{
    if (a16) { const uint4 v = *reinterpret_cast<const uint4 *>(p); w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; }
    else { const uint2 v0 = *reinterpret_cast<const uint2 *>(p), v1 = *reinterpret_cast<const uint2 *>(p + 8); w[0] = v0.x; w[1] = v0.y; w[2] = v1.x; w[3] = v1.y; }
}

constexpr int ZF_NB = 2;   // plane buffers in flight
enum { BAR_FULL = 1, BAR_EMPTY = 3, BAR_QUEUE = 5 };  // + buffer index (BAR_QUEUE + 1: the producers' own barrier)

template <int MODE>
__global__ void __launch_bounds__(ZF_THREADS, ZF_MINBLOCKS)
reconstruct_fast_kernel(const DevImage *__restrict__ images, const int spc)
{
    typedef FastTraits<MODE> FT;
    typedef uint8_t ST;
    constexpr int ROWS = FT::ROWS, TWY = FT::TWY, CS = FT::CS, NRG = FT::NRG, XU = FT::XU, RPU = FT::RPU;
    constexpr bool HALO = FT::NSLOT > 0;

    extern __shared__ __align__(128) uint8_t sDynAll[];  // [staging slots ZF_PRODUCERS * 128 B | row-pass scratch ZF_PRODUCERS * 256 B | ZF_NB plane buffers of [Y | Cb | Cr]]
    ST *const sPlanes = sDynAll + 3 * ZF_PRODUCERS * 128 + 128;   // (+ one all-zero slot)
    __shared__ __align__(16) u32 sQ[3][32];
    __shared__ int sSlowN;
    __shared__ unsigned short sSlow[ZJ_SLOW_CAP];      // units left to the generic path (row group << 8 | tile column / 8)

    const DevImage &im = images[blockIdx.z];
    const u32 tile = blockIdx.x;
    if (tile >= im.n_tiles) return;
    const int tid = threadIdx.x;
    const u32 stride = im.stride;
    uint8_t *__restrict__ out = im.out;
    const u32 n_strips = im.n_strips;
    const u32 s_begin = blockIdx.y * (u32)spc;

    // rows below the last processed strip stay zero in the reference (Q1 dropped MCU row, mcu.rs:154,158):
    // written by the first row of CTAs past the image's strips
    if (s_begin >= n_strips) {
        if (s_begin >= n_strips + (u32)spc) return;
        const size_t lo = (size_t)n_strips * ROWS * stride, hi = (size_t)im.height * stride;
        if (lo >= hi) return;
        const size_t span = hi - lo, per = (span + im.n_tiles - 1) / im.n_tiles;
        size_t b0 = lo + (size_t)tile * per, b1 = b0 + per;
        if (b1 > hi) b1 = hi;
        for (size_t b = b0 + tid; b < b1; b += ZF_THREADS) out[b] = 0;
        return;
    }
    const int n_it = (int)(min(s_begin + (u32)spc, n_strips) - s_begin);   // strips of this CTA

    // tile -> unit columns [u0, u1) (16 luma samples each), spread evenly: the first tile_r tiles are one wider
    const int nt = (int)im.n_tiles;
    const int u0 = (int)(tile * im.tile_q + min(tile, im.tile_r)), u1 = (int)((tile + 1) * im.tile_q + min(tile + 1, im.tile_r));
    const int Wp = (int)im.Wp, W = (int)im.W, mcu_x = (int)im.mcu_x;
    const int X0 = 16 * u0;                                        // first luma column of the tile
    const int yb0 = 2 * u0, nyb = min(2 * u1, Wp >> 3) - yb0;      // luma block columns of the tile
    const int cb0 = FT::H == 2 ? u0 : yb0, ncb = FT::H == 2 ? u1 - u0 : nyb;  // chroma block columns
    // halo block columns wrap around the image: the flat filters run across row ends (Q4a); tile 0 of the AVX2 HV
    // form also needs block column mcu_x-2 for the stale first-vector neighbours (Q4f)
    const int lhb = HALO ? (cb0 == 0 ? mcu_x - 1 : cb0 - 1) : -1;
    const int rhb = HALO ? (cb0 + ncb == mcu_x ? 0 : cb0 + ncb) : -1;
    const int spb = (MODE == MODE_HV && tile == 0 && nt > 1) ? mcu_x - 2 : -1;
    const u32 n_norm = im.n_norm, T = im.T, P = im.P;

    for (int k = tid; k < 96; k += ZF_THREADS) sQ[k >> 5][k & 31] = im.qtw[k >> 5][k & 31];
    if (tid == 0) sSlowN = 0;
    __syncthreads();

    const bool producer = tid < ZF_PRODUCERS;
    const int rtid = producer ? tid : tid - ZF_PRODUCERS;
    if (producer) {
        // ================================================================= producers: dequantise + IDCT
        // Blocks rtid and rtid + ZF_PRODUCERS of the tile's list [Y | Cb tile | Cr tile | Cb halo | Cr halo]: every warp
        // owns 32 consecutive entries = one or two contiguous runs of blocks in global memory (or up to 32 lone halo
        // blocks).  The warp copies its runs with fully coalesced cp.async into its 32 staging slots (128 bytes each,
        // 16-byte chunks XOR-swizzled by the slot number so that the per-thread 128-bit reads are conflict-free),
        // one strip ahead of the arithmetic.
        constexpr int NHB = FT::NSLOT * FT::CBR;                  // halo blocks per chroma plane
        // Which of the four producer jobs a hardware warp takes is rotated with the CTA index: the jobs are not equally heavy
        // (in 4:2:0 two warps carry a luma AND a chroma pass), warp w always runs on SM sub-partition w mod 4, and the three
        // resident CTAs of an SM would otherwise pile their heavy warps onto the same two sub-partitions.
        const int lane = tid & 31, wq = ((rtid >> 5) + (int)(blockIdx.x + blockIdx.y + blockIdx.z)) & 3;
        const int ybpr = Wp >> 3;
        // block index -> plane, block row, global block column (-1: none), smem column
        auto decode = [&](int b, int &comp, int &br, int &gcol, int &lcol) {
            if (b < FT::NY) { comp = 0; br = b / FT::YB; const int bc = b % FT::YB; gcol = bc < nyb ? yb0 + bc : -1; lcol = bc * 8; }
            else if (b < FT::NY + 2 * FT::NC) {
                int c = b - FT::NY; comp = 1 + c / FT::NC; c %= FT::NC;
                br = c / FT::CB; const int bc = c % FT::CB; gcol = bc < ncb ? cb0 + bc : -1; lcol = 8 + bc * 8;
            } else {
                int hx = b - FT::NY - 2 * FT::NC; comp = 1 + hx / (NHB > 0 ? NHB : 1); hx %= (NHB > 0 ? NHB : 1);
                const int slot = hx / FT::CBR; br = hx % FT::CBR;
                gcol = slot == 0 ? lhb : (slot == 1 ? rhb : spb);
                lcol = slot == 0 ? 0 : (slot == 1 ? 8 + ncb * 8 : 16 + ncb * 8);
                if (NHB == 0 || comp > 2) { comp = 1; gcol = -1; }
            }
        };
        auto block_ptr = [&](int comp, int br, int gcol) -> const int16_t * {
            return comp == 0 ? im.coeff[0] + (((size_t)s_begin * FT::YBR + br) * ybpr + gcol) * 64
                             : im.coeff[comp] + (((size_t)s_begin * FT::CBR + br) * mcu_x + gcol) * 64;
        };
        const u32 stepY = (u32)(FT::YBR * ybpr * 64), stepC = (u32)(FT::CBR * mcu_x * 64);   // i16 per strip
        // One staging job = the 32 consecutive list entries [B0, B0 + 32) of a warp: where this lane's block of the job goes (pk),
        // how the warp copies the job's runs (g0 / g1 lane pointers at the CTA's first strip, jm).
        //   pk: bits 0-15 byte offset in the plane buffer, 16 active, 17 chroma, 18-19 table, 20 left halo block (nothing reads it;
        //       the compiler schedules the setup differently without it, so it goes with the next change that re-measures the kernel)
        //   jm: bits 0-7 chunk k of the cooperative copy is inside the run, bit 8 the lane copies its own (lone) block
        auto setup_job = [&](const int B0, u32 &pkj, const int16_t *&g0, const int16_t *&g1, u32 &jmj) {
            int comp, br, gcol, lcol;
            decode(B0 + lane, comp, br, gcol, lcol);
            const bool active = gcol >= 0;
            pkj = (comp == 0 ? (u32)(br * 8 * TWY + lcol) : (u32)(FT::YBYTES + (comp - 1) * FT::CBYTES + br * 8 * CS + lcol)) |
                  (active ? 0x10000u : 0u) | (comp ? 0x20000u : 0u) | ((u32)comp << 18) |
                  ((comp != 0 && lcol == 0) ? 0x100000u : 0u);   // bit 20: see pk above
            const int lsub = lane >> 3, lch = lane & 7;
            g0 = g1 = im.coeff[0];
            int mode = 0, lim0 = 0, lim1 = 0;   // mode: 0 none, 1 one run of 32, 2 two runs of 16, 3 lone blocks
            if (FT::DENSE) {
                if (active) { mode = 3; g0 = block_ptr(comp, br, gcol); }
            } else if (B0 < FT::NY + 2 * FT::NC) {
                int c0, b0r, gg0, l0;
                decode(B0, c0, b0r, gg0, l0);
                const bool isY = B0 < FT::NY;
                const int bpr = isY ? FT::YB : FT::CB;           // blocks per tile block row
                const int col0 = isY ? (B0 % FT::YB) : ((B0 - FT::NY) % FT::NC) % FT::CB;
                const int have = (isY ? nyb : ncb) - col0;       // valid blocks from col0 on
                const int first = (isY ? yb0 : cb0) + col0;
                if (bpr >= 32) { mode = 1; lim0 = min(max(have, 0), 32) - lsub; g0 = block_ptr(c0, b0r, first) + lsub * 64 + lch * 8; }
                else {
                    mode = 2; lim0 = lim1 = min(max(have, 0), 16) - lsub;
                    g0 = block_ptr(c0, b0r, first) + lsub * 64 + lch * 8;
                    g1 = block_ptr(c0, b0r + 1, first) + lsub * 64 + lch * 8;
                }
            } else if (active) { mode = 3; g0 = block_ptr(comp, br, gcol); }
            u32 m = 0;
            for (int k = 0; k < 8; k++) {
                const bool second = mode == 2 && k >= 4;
                if ((mode == 1 || mode == 2) && 4 * (second ? k - 4 : k) < (second ? lim1 : lim0)) m |= 1u << k;
            }
            if (mode == 3) m = 0x100u;
            if (mode == 2) g1 -= 4 * 256;           // chunk k of run 1 is at g1 + (k - 4) * 256
            else g1 = g0;
            jmj = m;
        };
        const u32 stage0 = (u32)__cvta_generic_to_shared(sDynAll) + (u32)(wq * 32) * 128u;     // the warp's slots of pass 0 (pass 1: + 16 KB)
        const u32 d_even = stage0 + (u32)(lane >> 3) * 128u + (u32)(((lane & 7) ^ (lane >> 3)) * 16);
        const u32 d_odd = stage0 + (u32)(lane >> 3) * 128u + (u32)(((lane & 7) ^ ((lane >> 3) + 4)) * 16);
        const u32 slx = (stage0 + (u32)lane * 128u) | (u32)((lane & 7) * 16);              // own slot, chunk r at slx ^ (r << 4)
        const u32 scr = (u32)__cvta_generic_to_shared(sDynAll) + ZF_PRODUCERS * 128u + (u32)rtid * 16u;   // scratch column of the row pass
        // threads without a block in a pass read an all-zero slot instead (their own slot may hold the other pass's block)
        const u32 zslot = ((u32)__cvta_generic_to_shared(sDynAll) + 3u * ZF_PRODUCERS * 128u) | (u32)((lane & 7) * 16);
        if (rtid < 8) sts128(zslot - (u32)((lane & 7) * 16) + (u32)rtid * 16u, 0u, 0u, 0u, 0u);
        asm volatile("bar.sync %0, %1;" ::"r"((int)BAR_QUEUE + 1), "n"(ZF_PRODUCERS) : "memory");   // producers only
        // (these four are a few integer operations each from the lane index; made opaque so that they are kept instead of
        // being recomputed in every pass)
        asm volatile("" : "+r"(const_cast<u32 &>(d_even)), "+r"(const_cast<u32 &>(d_odd)), "+r"(const_cast<u32 &>(slx)), "+r"(const_cast<u32 &>(scr)));
        auto issue = [&](const int16_t *g0, const int16_t *g1, const u32 m) {
            if (ZF_LIKELY(m == 0xffu)) {   // a full job: no per-chunk predicates
#pragma unroll
                for (int k = 0; k < 8; k++)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(((k & 1) ? d_odd : d_even) + k * 512u), "l"((k < 4 ? g0 : g1) + k * 256) : "memory");
            } else if (m & 0x100u) {
#pragma unroll
                for (int r = 0; r < 8; r++)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(slx ^ (u32)(r << 4)), "l"(g0 + r * 8) : "memory");
            } else {
#pragma unroll
                for (int k = 0; k < 8; k++)
                    if (m & (1u << k))
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(((k & 1) ? d_odd : d_even) + k * 512u), "l"((k < 4 ? g0 : g1) + k * 256) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        // this thread's own two blocks / this warp's staging jobs
        u32 pk[2], jm[2];
        const int16_t *q0[2], *q1[2];    // lane pointers into run 0 / run 1 (lone blocks: the lane's own block)
#pragma unroll
        for (int ps = 0; ps < 2; ps++) {
            // pass 0: job wq.  Pass 1: the jobs after the first four, handed out so that a warp whose pass-0 job is a (cheap)
            // chroma job gets one first -- without sub-sampling warps 0,1 transform luma and 2,3 take Cb, then Cr; in 4:2:2 the
            // lone halo job goes to a chroma warp.  (4:2:0 / 4:4:0: all four pass-0 jobs are luma, order is irrelevant.)
            const int jw = ps == 0 ? wq : ((wq + ((MODE == MODE_NONE || MODE == MODE_H) ? 2 : 0)) & 3);
            setup_job(ps * ZF_PRODUCERS + jw * 32, pk[ps], q0[ps], q1[ps], jm[ps]);
        }
        // loop-carried state
        const int16_t *qa0 = q0[0], *qb0 = q1[0], *qa1 = q0[1], *qb1 = q1[1];
        const u32 pk0 = pk[0], pk1 = pk[1], jm0 = jm[0], jm1 = jm[1];
        // per-strip step of the copy pointers: by the plane of the warp's blocks (dense lists: of the lane's own block)
        const u32 st0 = FT::DENSE ? ((pk0 & 0x20000u) ? stepC : stepY) : ((wq * 32 < FT::NY) ? stepY : stepC);
        const u32 st1 = FT::DENSE ? ((pk1 & 0x20000u) ? stepC : stepY) : ((ZF_PRODUCERS + wq * 32 < FT::NY) ? stepY : stepC);
        // one staging slot per thread: the copy of the next pass is issued as soon as the row pass has drained the slot
        // and lands while the column pass runs
        const bool work0 = __any_sync(0xffffffffu, (pk0 & 0x10000u) != 0), work1 = __any_sync(0xffffffffu, (pk1 & 0x10000u) != 0);   // any block in the warp
        issue(qa0, qb0, jm0);
        qa0 += st0; qb0 += st0;
        int buf = 0;
        for (int it = 0; it < n_it; it++) {
            ST *planes = sPlanes + buf * FT::BUF;
#pragma unroll 1
            for (int ps = 0; ps < 2; ps++) {
                // A warp without a pass-1 job (4:2:2: every warp -- the strip-tile's list is exactly one pass) copies its NEXT
                // strip's job as soon as the row pass of pass 0 has drained the slot, and skips pass 1: issued from pass 1 the copy
                // had no lead at all -- the warp waited for it at the top of the next strip (10 % of all stall samples of the
                // 1080p 4:2:2 config sat on that wait).
                if (ps == 1 && !work1) break;
                const u32 pkk = ps ? pk1 : pk0;
                const bool active = (pkk & 0x10000u) != 0;
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
                if (ps == 0 && it >= ZF_NB) bar_sync(BAR_EMPTY + buf);   // the consumers are done with this buffer
                // the copy issued from this pass: the warp's pass-1 job of this strip, or its pass-0 job of the next strip
                // (one call site: the copy code exists once in the loop)
                auto refill = [&]() {
                    const bool nxt = ps || !work1;           // the next strip's pass-0 job
                    issue(nxt ? qa0 : qa1, nxt ? qb0 : qb1, nxt ? (it + 1 < n_it ? jm0 : 0u) : jm1);
                    if (nxt) { qa0 += st0; qb0 += st0; } else { qa1 += st1; qb1 += st1; }
                };
                if (ps ? work1 : work0) idct_rolled<FT::IDCT_UNROLL, FT::LO6>(active, active ? slx : zslot, scr, sQ[(pkk >> 18) & 3u], planes + (pkk & 0xffffu), (pkk & 0x20000u) ? CS : TWY, refill);
                else refill();
            }
            bar_arrive(BAR_FULL + buf);
            buf = buf + 1 == ZF_NB ? 0 : buf + 1;
        }
        return;
    }

    // ===================================================================== consumers: up-sample, convert, write
    const int tc = rtid;
    const int xu = tc % XU, rgA = tc / XU;                // this thread's units: (xu, rgA) and (xu, rgA + NRG/2)
    const bool ycc = im.out_kind == OUT_YCC;
    u32 esel = !ycc ? 0x7351u : 0x6240u, ekk = 0xC000C000u ^ ((u32)spc >> 30);   // (spc < 2^30: a constant ptxas cannot see)
    asm volatile("" : "+r"(esel), "+r"(ekk));   // (opaque: kept in registers instead of being rematerialised in front of every use)
    u32 ekr = 0x98619861u ^ ((u32)spc >> 30);
    asm volatile("" : "+r"(ekr));
    int xs = X0 + 16 * xu;                                // first sample of the unit in the padded row
    // Where the unit's 48 bytes go (worker.rs:201-246, SURVEY A.5): samples < n_norm ("normal" 16-sample chunks) sit at
    // byte 3*s, except bytes the tail chunk overwrites; the tail chunk (samples Wp-16..Wp-1) sits at T; the rest is never written
    int kind = 0;                                         // 0 = nothing to write, 1 = packed path, 2 = generic path
    int dst_off = 3 * xs, nw = 12;
    if (u0 + xu < u1 && rgA < NRG / 2) {                   // (XU * NRG / 2 may be smaller than the consumer count: those threads idle)
        if ((u32)(xs + 16) <= n_norm) {
            kind = 1;
            if (T != 0xffffffffu && (u32)(3 * xs + 48) > T && (u32)(3 * xs) < T + 48) {   // overlaps the tail chunk's bytes [T, T+48)
                const int keep = (int)T - 3 * xs;                                        // bytes before T survive
                if ((u32)(3 * xs + 48) > T + 48) kind = 2;
                else if (keep <= 0) kind = 0;
                else if ((keep & 3) == 0) nw = keep >> 2;
                else kind = 2;
            }
        } else if (T != 0xffffffffu && (u0 + xu) == ((Wp - 16) >> 4)) {
            kind = 1; xs = Wp - 16; dst_off = (int)T;
        } else if ((u32)xs < n_norm) {
            kind = 2;                                                                     // partially inside [0, n_norm): YCbCr output, width % 16 != 0
        }
    }
    if (kind == 1 && (dst_off & 3) != 0) kind = 2;
    const bool vec = ((stride & 15u) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0) && ((dst_off & 15) == 0) && ((nw & 3) == 0);
    const int xl = xs - X0;                               // tile-local luma column
    const bool y16 = (xl & 15) == 0;
    const int cc0 = FT::H == 2 ? xs >> 1 : xs;            // first chroma column
    const int lc = 8 + (cc0 - cb0 * 8);                   // its smem column
    const bool first_x = HALO && cc0 == 0, last_x = HALO && cc0 + 8 == W;
    // per-unit state of the two halves; the second unit sits ROWS/2 output rows (CROWS/2 chroma rows) below the first
    int kindA = kind, kindB = kind;
    int off0 = 0, off2 = 0;                               // row offsets of the outer neighbours (flat filters, Q4a)
    bool sel0 = false, firstvec = false, hv_tail = false;
    const int pbit = rgA & 1;                             // HV: row parity inside the double-row
    if (MODE == MODE_H) {
        off0 = first_x ? -CS : 0; off2 = last_x ? CS : 0;
        // the strip's first unit (out[0] = in[0], sse.rs:24-30) and last unit (the SSE tail, Q4b) are patched in place below
    } else if (MODE == MODE_HV) {
        off0 = (first_x && pbit) ? -CS : 0; off2 = last_x ? CS : 0;
        sel0 = (((pbit ? W : 0) + cc0) & 15) == 0;        // unit starts an AVX2 vector (else it ends one)
        firstvec = pbit == 0 && cc0 < 16;                 // vector t = 0 of the double-row (Q4f)
        hv_tail = pbit == 1 && cc0 + 16 >= W;             // last 32 outputs of the double-row (Q4g)
        if (kind == 1 && hv_tail && W - 36 - cb0 * 8 < (cb0 == 0 ? 0 : -8)) kindA = kindB = 2;  // raw tail reaches left of the tile's halo (or wraps a row)
        if (kind == 1 && firstvec && W < 48) kindA = kindB = 2;
    }
#pragma unroll
    for (int h = 0; h < 2; h++)
        if ((h ? kindB : kindA) == 2) {
            const int slot = atomicAdd(&sSlowN, 1);
            if (slot < ZJ_SLOW_CAP) sSlow[slot] = (unsigned short)(((rgA + h * (NRG / 2)) << 8) | (xl >> 3));
        }
    bar_sync_consumers(BAR_QUEUE);   // the queue is complete (consumer warps only)
    const int nslow = sSlowN;

    // bytes of a row nobody writes: [P, stride) minus the tail chunk [T, T+48) (Q5: 16 zero bytes; Q6: the w "alpha"
    // bytes) = [z0, stride); every tile zeroes its share, with the widest stores the alignment allows
    const u32 z0 = (T != 0xffffffffu && T + 48 > P) ? T + 48 : P;
    const u32 zlen = stride > z0 ? stride - z0 : 0;
    const int zg = (((z0 | stride) & 15u) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) ? 16 : ((((z0 | stride) & 3u) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0) ? 4 : 1);
    const u32 zper = ((zlen / zg + nt - 1) / nt) * zg;             // bytes per tile (multiple of the store size)
    const u32 zb0 = min(z0 + tile * zper, stride), zb1 = min(zb0 + zper, stride);
    const int zcnt = (int)((zb1 - zb0) / zg);                     // stores per row for this tile
    const int zrpp = (zcnt > 0 && zcnt < ZF_CONSUMERS) ? ZF_CONSUMERS / zcnt : 1;           // rows covered per pass of the consumer threads
    const int zr0 = (zcnt > 0 && zcnt < ZF_CONSUMERS) ? (tc / zcnt < zrpp ? tc / zcnt : ROWS) : 0;
    const int zk0 = (zcnt > 0 && zcnt < ZF_CONSUMERS) ? tc % zcnt : tc;

    int buf = 0;
    for (int it = 0; it < n_it; it++) {
        const ST *planes = sPlanes + buf * FT::BUF;
        const u32 y_base = (s_begin + it) * ROWS;
        bar_sync(BAR_FULL + buf);
#pragma unroll 1
        for (int h = 0; h < 2; h++) {
            if ((h ? kindB : kindA) != 1) continue;
            const int rg = rgA + h * (NRG / 2);
            int yl0, yl1, ra, rb;                                     // rows of the unit inside the strip; chroma rows blended
            if (MODE == MODE_V) { yl0 = 2 * rg; yl1 = yl0 + 1; ra = rg; rb = (rg == 0 || rg == 7) ? rg : rg + 1; }   // scalar.rs:64-147 (Q4c)
            else if (MODE == MODE_HV) { const int j = rg >> 1; yl0 = 4 * j + pbit; yl1 = yl0 + 2; ra = 2 * j + pbit; rb = (j == 0 || j == 7) ? ra : ra + 2; }  // (Q4d)
            else { yl0 = rg; yl1 = rg; ra = rg; rb = rg; }
            u32 E0[2][4], O0[2][4], E1[2][4], O1[2][4];   // [cb|cr] chroma of row 0 / row 1 of the unit, E/O arrangement
#pragma unroll
            for (int c = 0; c < 2; c++) {
                const uint8_t *base = planes + FT::YBYTES + c * FT::CBYTES;
                if (MODE == MODE_NONE) {
                    u32 w[4];
                    load16(base + ra * CS + lc, false, w);
#pragma unroll
                    for (int k = 0; k < 4; k++) { E0[c][k] = evens(w[k]); O0[c][k] = odds(w[k]); }
                } else if (MODE == MODE_V) {
                    u32 a[4], b[4];
                    load16(base + ra * CS + lc, false, a);
                    load16(base + rb * CS + lc, false, b);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const u32 aE = evens(a[k]), aO = odds(a[k]), bE = evens(b[k]), bO = odds(b[k]);
                        T2pair(aE, bE, E0[c][k], E1[c][k]);                // rows 2k, 2k+1 <- T(r_k, r_k+1), T(r_k+1, r_k)
                        T2pair(aO, bO, O0[c][k], O1[c][k]);
                    }
                } else if (MODE == MODE_H) {
                    const uint8_t *pa = base + ra * CS + lc;
                    const uint2 a = *reinterpret_cast<const uint2 *>(pa);
                    const bool hstart = first_x && rg == 0, hend = last_x && rg == NRG - 1;
                    // strip start: out[0] = in[0] = T(in[0], in[0]) -- the left neighbour is the sample itself; no row above to read
                    const u32 left = hstart ? (a.x & 0xffu) : (u32)pa[off0 - 1], right = hend ? 0u : (u32)pa[off2 + 8];
                    const u32 r[4] = {lanes01(a.x), lanes23(a.x), lanes01(a.y), lanes23(a.y)};
                    hfilter16(left | (right << 16), r, E0[c], O0[c]);
                    if (ZF_UNLIKELY(hend)) {
                        // the last eight outputs of the strip, as upsample_horizontal_sse leaves them (sse.rs:117-131, Q4b), R = in[n-8..n-1]:
                        //   out[8..15] = T(R4,R3), T(R4,R5), T(R5,R4), R5, R6, T(R6,R5), T(R6,R7), R7
                        // against the regular T(R4,R3), T(R4,R5), T(R5,R4), T(R5,R6), T(R6,R5), T(R6,R7), T(R7,R6), T(R7,R8)
                        const u32 e3 = E0[c][3], o3 = O0[c][3];                       // (out12, out14), (out13, out15) regular
                        O0[c][2] = prmt(O0[c][2], r[2], 0x7610u);                     // out11 = R5
                        E0[c][3] = prmt(r[3], o3, 0x5410u);                           // (R6, T(R6,R7))
                        O0[c][3] = prmt(e3, r[3], 0x7610u);                           // (T(R6,R5), R7)
                    }
                } else if (ZF_LIKELY(!hv_tail)) {
                    const uint8_t *pa = base + ra * CS + lc, *pb = base + rb * CS + lc;
                    const uint2 a = *reinterpret_cast<const uint2 *>(pa), b = *reinterpret_cast<const uint2 *>(pb);
                    const u32 aL = pa[off0 - 1], aR = pa[off2 + 8], bL = pb[off0 - 1], bR = pb[off2 + 8];
                    const u32 A[4] = {lanes01(a.x), lanes23(a.x), lanes01(a.y), lanes23(a.y)};
                    const u32 B[4] = {lanes01(b.x), lanes23(b.x), lanes01(b.y), lanes23(b.y)};
                    const u32 Ah = aL | (aR << 16), Bh = bL | (bR << 16);
                    u32 N[4], F[4];
                    u32 Nh, Fh;
#pragma unroll
                    for (int k = 0; k < 4; k++) T2pair_s(A[k], B[k], N[k], F[k]);
                    T2pair_s(Ah, Bh, Nh, Fh);
                    // AVX2 form: lane 0 of a vector takes 3*(in+in'+2)>>2 of its OWN first element as "previous" value,
                    // lane 15 the same expression of the next vector's first element as "next" value (Q4e)
                    u32 pv = (3u * ((sel0 ? (a.x & 0xffu) + (b.x & 0xffu) : aR + bR) + 2u)) >> 2;
                    if (ZF_UNLIKELY(firstvec)) {
                        // vector t = 0: the neighbours are whatever the loop left behind (avx2.rs:67-68,264-270; Q4f): for
                        // j = 0 the raw in[0] / in[16], for j >= 1 the values computed 16 samples before the end of
                        // double-row j-1 (lane 0) and at the start of double-row j (lane 15), both with the stride of j-1
                        const int j = rg >> 1;
                        if (j == 0) pv = sel0 ? (a.x & 0xffu) : aR;
                        else if (sel0) {
                            const int spc0 = nt > 1 ? 16 + ncb * 8 : 8 + (W - 16);                 // smem column of chroma column W-16
                            const int rp = 2 * j - 1, rq = (j == 1) ? rp : rp + 2;
                            pv = (3u * ((u32)base[rp * CS + spc0] + (u32)base[rq * CS + spc0] + 2u)) >> 2;
                        } else {
                            const u32 y0 = base[2 * j * CS + 8], y1 = (j == 1) ? y0 : (j == 7 ? 0u : (u32)base[(2 * j + 2) * CS + 8]);
                            pv = (3u * (y0 + y1 + 2u)) >> 2;
                        }
                    }
                    pv = pv * 4u;                                          // (<= 4 * 384: one lane)
                    const u32 keep = sel0 ? 0xffff0000u : 0x0000ffffu, ins = sel0 ? pv : pv << 16;
                    Nh = (Nh & keep) | ins;
                    Fh = (Fh & keep) | ins;
                    hfilter16_s(Nh, N, E0[c], O0[c]);
                    hfilter16_s(Fh, F, E1[c], O1[c]);
                    if (firstvec && cc0 == 0) E1[c][0] = prmt(E1[c][0], O1[c][0], 0x3254u);   // far rows: out[0] = out[1] (avx2.rs:330)
                } else {
                    // last 32 outputs of the double-row: out[O+2k] = T(in[c], in[c-1]), out[O+2k+1] = T(in[c], in[c+1]),
                    // c = (row end) - 33 + k: raw row 2j+1 (near) / 2j+3 (far), no vertical blend; k = 15 repeats k = 14
                    // (upsampler/avx2.rs:277-307,332-338; Q4g)
                    const int q = (cc0 - (W - 16)) >> 3;                      // which half of the 32 outputs
                    const int lq = 8 + (W - 36 + 8 * q - cb0 * 8);            // smem column of c - 3 for k = 8q (multiple of 4)
#pragma unroll
                    for (int f = 0; f < 2; f++) {
                        const u32 *pw = reinterpret_cast<const u32 *>(base + (f ? rb : ra) * CS + lq);
                        const u32 w0 = pw[0], w1 = pw[1], w2 = pw[2];
                        const u32 r[4] = {prmt(w0, w1, 0x0403u) & 0x00ff00ffu, prmt(w1, 0u, 0x4241u), prmt(w1, w2, 0x0403u) & 0x00ff00ffu, prmt(w2, 0u, 0x4241u)};
                        const u32 hh = prmt(w0, w2, 0x0702u) & 0x00ff00ffu;
                        u32 *E = f ? E1[c] : E0[c], *O = f ? O1[c] : O0[c];
                        hfilter16(hh, r, E, O);
                        if (q == 1) { E[3] = prmt(E[3], 0u, 0x1010u); O[3] = prmt(O[3], 0u, 0x1010u); }
                    }
                }
            }
            if (y_base + yl0 < im.height) {
                u32 yw[4];
                load16(planes + yl0 * TWY + xl, FT::H == 2 || y16, yw);
                emit16(out + (size_t)(y_base + yl0) * stride + dst_off, yw, E0[0], O0[0], E0[1], O0[1], ycc, nw, vec, esel, ekk, ekr);
            }
            if (RPU == 2 && y_base + yl1 < im.height) {
                u32 yw[4];
                load16(planes + yl1 * TWY + xl, FT::H == 2 || y16, yw);
                emit16(out + (size_t)(y_base + yl1) * stride + dst_off, yw, E1[0], O1[0], E1[1], O1[1], ycc, nw, vec, esel, ekk, ekr);
            }
        }
        if (ZF_UNLIKELY(nslow > 0)) {
            SlowCtx<ST> sc;
#pragma unroll
            for (int c = 0; c < 2; c++) {
                sc.cv[c].base = planes + FT::YBYTES + c * FT::CBYTES; sc.cv[c].W = W; sc.cv[c].n = FT::CROWS * W;
                sc.cv[c].c0 = cb0 * 8; sc.cv[c].c1 = (cb0 + ncb) * 8; sc.cv[c].lhb = lhb; sc.cv[c].rhb = rhb; sc.cv[c].spb = spb; sc.cv[c].cs = CS; sc.cv[c].magic_w = im.magic_w;
            }
            sc.sY = planes; sc.twy = TWY; sc.X0 = X0; sc.Wp = Wp; sc.hv_avx = (int)im.hv_avx; sc.y_base = y_base; sc.height = im.height;
            sc.stride = stride; sc.n_norm = n_norm; sc.T = T; sc.ycc = ycc; sc.out = out; sc.width = im.width; sc.nc = im.nc;
            if (nslow > ZJ_SLOW_CAP) {
                const int tw = nyb * 8;
                // (every lane makes the same number of trips, so the warps arrive at the barriers below in one piece)
                for (int u0s = 0; u0s < ROWS * tw; u0s += ZF_CONSUMERS) {
                    const int u = u0s + tc;
                    if (u < ROWS * tw) { const int yl = u / tw; slow_pixel<MODE, 0, ST>(sc, yl, u - yl * tw); }
                }
            } else {
                const int total = nslow * 16 * RPU;
                for (int t0s = 0; t0s < total; t0s += ZF_CONSUMERS) {
                    const int t = t0s + tc;
                    if (t < total) {
                        const int e = sSlow[t / (16 * RPU)], r = (t >> 4) % RPU, k = t & 15;
                        const int g = e >> 8, xl2 = (e & 0xff) << 3;
                        int yl;
                        if (MODE == MODE_V) yl = 2 * g + r;
                        else if (MODE == MODE_HV) yl = 4 * (g >> 1) + (g & 1) + 2 * r;
                        else yl = g;
                        if (xl2 + k < nyb * 8) slow_pixel<MODE, 0, ST>(sc, yl, xl2 + k);
                    }
                }
            }
            __syncwarp();
        }
        if (it + ZF_NB < n_it) bar_arrive(BAR_EMPTY + buf);          // the producers may refill this buffer
        buf = buf + 1 == ZF_NB ? 0 : buf + 1;
        if (ZF_UNLIKELY(zcnt > 0)) {
            // thread -> (row zr0 + i * zrpp, store zk0 + j * ZF_CONSUMERS): no divisions inside the strip loop
            for (int yl = zr0; yl < ROWS; yl += zrpp) {
                const u32 y = y_base + (u32)yl;
                if (y >= im.height) break;
                uint8_t *zrow = out + (size_t)y * stride + zb0;
                for (int k = zk0; k < zcnt; k += ZF_CONSUMERS) {
                    uint8_t *z = zrow + (size_t)k * zg;
                    if (zg == 16) *reinterpret_cast<uint4 *>(z) = make_uint4(0u, 0u, 0u, 0u);
                    else if (zg == 4) *reinterpret_cast<u32 *>(z) = 0u;
                    else *z = 0;
                }
            }
            __syncwarp();
        }
    }
}

// ------------------------------------------------------------------------------------- luma-only kernel
// (YCbCr | GRAYSCALE) -> GRAYSCALE: IDCT of the Y plane only (worker.rs:59,115-118), `as u8` row copy
// (color_convert/scalar.rs:91-114; Q7 is resolved on the host: geometries where the reference panics are
// rejected before launch).  grid = (ceil(blocks per block-row / 128), block-rows + 1, images).
// VARIANT: the IDCT -- 0 = X86, 1 = SCALAR, IDCT_ISLOW = the islow luma plane of ZJ_FLAG_ISLOW images (whose rows all lie in
// the image's strips, so the reference's geometry rules are no-ops here).
template <int VARIANT>
__global__ void __launch_bounds__(ZJ_THREADS)
gray_kernel(const DevImage *__restrict__ images, int rows_per_strip)
{
    typedef typename std::conditional<VARIANT == 1, int16_t, uint8_t>::type ST;
    __shared__ __align__(16) ST sT[ZJ_THREADS][64 + 8];  // one block per thread, padded
    __shared__ u32 sQ[32];
    const DevImage &im = images[blockIdx.z];
    const int tid = threadIdx.x;
    const int ybpr = (int)(im.Wp >> 3);
    const u32 brows = im.n_strips * (u32)(rows_per_strip >> 3);  // block rows the reference processes
    const u32 br = blockIdx.y;
    uint8_t *__restrict__ out = im.out;
    if (br >= brows) {
        if (br > brows) return;
        const size_t lo = (size_t)brows * 8 * im.stride, hi = (size_t)im.height * im.stride;
        if (lo >= hi) return;
        const size_t span = hi - lo, per = (span + gridDim.x - 1) / gridDim.x;
        size_t b0 = lo + (size_t)blockIdx.x * per, b1 = b0 + per;
        if (b1 > hi) b1 = hi;
        for (size_t b = b0 + tid; b < b1; b += ZJ_THREADS) out[b] = 0;
        return;
    }
    if (tid < 32) sQ[tid] = im.qtw[0][tid];
    __syncthreads();
    const int bc = blockIdx.x * ZJ_THREADS + tid;
    const bool active = bc < ybpr;
    const size_t blk = (size_t)br * ybpr + (active ? bc : 0);
    int4 raw[8];
    load_block(active, im.coeff[0] + blk * 64, raw);
    if constexpr (VARIANT == IDCT_ISLOW) idct_islow_block(active, raw, sQ, &sT[tid][0], 8);
    else idct_block<VARIANT, ST>(active, raw, sQ, &sT[tid][0], 8);
    if (!active) return;
    const u32 x0 = (u32)bc * 8;
#pragma unroll 1
    for (int r = 0; r < 8; r++) {
        const u32 y = br * 8 + r;
        if (y >= im.height) break;
        uint8_t *row = out + (size_t)y * im.stride;
        for (int k = 0; k < 8; k++)
            if (x0 + k < im.width) row[x0 + k] = (uint8_t)((u32)sT[tid][r * 8 + k] & 0xff);
    }
}

// ------------------------------------------------------------------------------------- spec-correct kernel
// ZJ_VARIANT_SPEC (the statement is in include/zune_jpeg_b200.h): every row of the image, libjpeg's integer "fancy"
// up-sampling with every neighbour index clamped to the real chroma size, JFIF colour, opaque alpha.  No quirk of the reference
// applies, so the rows of a strip need chroma from the strips above and below and the tiles are simply TM MCU columns wide.
// grid = (tiles, strips, images); block = ZJ_THREADS.
//   phase 1: IDCT of the tile's luma and chroma blocks and of the chroma context the filters reach -- one block column on each
//            side (H, HV) and one block row above and below (V, HV), where it lies inside the real chroma size -- into shared
//            sample planes; IDCT_X86: the X86 IDCT (idct_block<0>), IDCT_ISLOW (ZJ_FLAG_ISLOW): idct_islow_block;
//   phase 2: one thread = 16 consecutive pixels of one row, stored as 16-byte words where the row's address allows it.
__device__ __forceinline__ void jfif_rgb(int y, int cb, int cr, u32 &r, u32 &g, u32 &b)  // jdcolor.c, 16-bit fixed point
{
    cb -= 128;
    cr -= 128;
    r = clamp255((u32)(y + ((91881 * cr + 32768) >> 16)));
    g = clamp255((u32)(y + ((-22554 * cb - 46802 * cr + 32768) >> 16)));
    b = clamp255((u32)(y + ((116130 * cb + 32768) >> 16)));
}

// (two CTAs per SM: at three, the 80-register cap makes the 16-pixel units of phase 2 spill)
template <int MODE, int IDCT>
__global__ void __launch_bounds__(ZJ_THREADS, 2)
spec_kernel(const DevImage *__restrict__ images)
{
    typedef ModeTraits<MODE> MT;
    constexpr int ROWS = 8 * MT::H * MT::V;   // luma rows per strip
    constexpr int CROWS = 8 * MT::CBR;        // chroma rows per strip
    constexpr int TWY = 8 * MT::H * MT::TM;   // luma tile width
    constexpr int PC = MT::H == 2 ? 8 : 0;    // context columns on each side of the chroma tile
    constexpr int PR = MT::V == 2 ? 8 : 0;    // context rows above and below it
    constexpr int CS = 8 * MT::TM + 2 * PC;   // chroma smem row
    constexpr int UPR = TWY / 16;             // 16-pixel units per row
    static_assert(TWY % 16 == 0 && CS % 16 == 0, "16-byte units");
    __shared__ __align__(16) uint8_t sY[ROWS * TWY];
    __shared__ __align__(16) uint8_t sC[2][(CROWS + 2 * PR) * CS];
    __shared__ u32 sQ[3][32];

    const DevImage &im = images[blockIdx.z];
    const int tile = (int)blockIdx.x, strip = (int)blockIdx.y;
    if (tile >= (int)im.n_tiles || strip >= (int)im.n_strips) return;
    const int tid = threadIdx.x;
    const int mcu_x = (int)im.mcu_x, width = (int)im.width, height = (int)im.height;
    const int m0 = tile * MT::TM, m1 = min(m0 + MT::TM, mcu_x), tm = m1 - m0;
    const bool color = im.W != 0;                                                  // 0: one-component input
    const int cw = (width + MT::H - 1) / MT::H, ch = (height + MT::V - 1) / MT::V;  // real chroma size
    // chroma block rows [rb0, rb1) and block columns [cb0, cb1) of this CTA, context included
    const int rb0 = strip * MT::CBR - ((PR && strip > 0) ? 1 : 0);
    const int rb1 = (strip + 1) * MT::CBR + ((PR && (strip + 1) * CROWS < ch) ? 1 : 0);
    const int cb0 = m0 - ((PC && m0 > 0) ? 1 : 0);
    const int cb1 = m1 + ((PC && m1 * 8 < cw) ? 1 : 0);
    const int ccols = cb1 - cb0;
    const int nY = MT::YBR * MT::H * tm, nC = color ? (rb1 - rb0) * ccols : 0;
    const int total = nY + 2 * nC;
    const int ybpr = MT::H * mcu_x;
    const float r_htm = __frcp_rn((float)(MT::H * tm)), r_cc = __frcp_rn((float)ccols);
    for (int k = tid; k < 96; k += ZJ_THREADS) sQ[k >> 5][k & 31] = im.qtw[k >> 5][k & 31];
    __syncthreads();

    // ---------------------------------------------------------------- phase 1
    for (int b0 = 0; b0 < total; b0 += ZJ_THREADS) {   // CTA-uniform trip count: every lane takes part in the warp votes
        const int b = b0 + tid;
        const bool active = b < total;
        const int16_t *src = nullptr;
        const u32 *qt = sQ[0];
        uint8_t *dst = sY;
        int dstride = TWY;
        if (!active) {
        } else if (b < nY) {
            const int br = div_small(b, r_htm), bc = b - br * (MT::H * tm);
            src = im.coeff[0] + (((size_t)strip * MT::YBR + br) * ybpr + (size_t)MT::H * m0 + bc) * 64;
            dst = sY + br * 8 * TWY + bc * 8;
        } else {
            int c = b - nY;
            const int comp = c >= nC ? 1 : 0;
            c -= comp * nC;
            const int r = div_small(c, r_cc), k = c - r * ccols;
            const int br = rb0 + r, bc = cb0 + k;
            src = im.coeff[1 + comp] + ((size_t)br * mcu_x + bc) * 64;
            qt = sQ[1 + comp];
            dst = sC[comp] + ((br - strip * MT::CBR) * 8 + PR) * CS + (bc - m0) * 8 + PC;
            dstride = CS;
        }
        int4 raw[8];
        load_block(active, src, raw);
        if constexpr (IDCT == IDCT_ISLOW) idct_islow_block(active, raw, qt, dst, dstride);
        else idct_block<0, uint8_t>(active, raw, qt, dst, dstride);
    }
    __syncthreads();

    // ---------------------------------------------------------------- phase 2
    const int nc = (int)im.nc;
    const bool ycc = im.out_kind == OUT_YCC;
    const int xt = 8 * MT::H * m0;              // first luma column of the tile
    const int ct0 = 8 * m0 - PC;                // chroma column of smem column 0
    const int cr0 = strip * CROWS - PR;         // chroma row of smem row 0
    for (int u = tid; u < ROWS * UPR; u += ZJ_THREADS) {
        const int yl = u / UPR, ux = u - yl * UPR;
        const int y = strip * ROWS + yl, x0 = xt + 16 * ux;
        if (y >= height || x0 >= width) continue;
        const int npx = min(16, width - x0);
        const uint4 yv = *reinterpret_cast<const uint4 *>(sY + yl * TWY + 16 * ux);
        const u32 yw[4] = {yv.x, yv.y, yv.z, yv.w};
        // chroma rows: j, and for V / HV the vertical neighbour jn (j - 1 for even rows, j + 1 for odd ones)
        int j = y, jn = y;
        if (MT::V == 2) { j = y >> 1; jn = (y & 1) ? min(j + 1, ch - 1) : max(j - 1, 0); }
        // H / HV: s[t] = the (column-summed) chroma sample at column clamp(x0 / 2 - 1 + t), t = 0..9
        int s[2][10];
        u32 cv[2][4];
        if (color) {
#pragma unroll
            for (int comp = 0; comp < 2; comp++) {
                const uint8_t *ra = sC[comp] + (j - cr0) * CS - ct0, *rn = sC[comp] + (jn - cr0) * CS - ct0;
                if (MT::H == 2) {
#pragma unroll
                    for (int t = 0; t < 10; t++) {
                        const int ci = min(max((x0 >> 1) - 1 + t, 0), cw - 1);
                        s[comp][t] = MT::V == 2 ? 3 * (int)ra[ci] + (int)rn[ci] : (int)ra[ci];
                    }
                } else {
                    const uint4 a = *reinterpret_cast<const uint4 *>(ra + x0);
                    cv[comp][0] = a.x; cv[comp][1] = a.y; cv[comp][2] = a.z; cv[comp][3] = a.w;
                    if (MT::V == 2) {
                        const uint4 n = *reinterpret_cast<const uint4 *>(rn + x0);
                        const u32 nw[4] = {n.x, n.y, n.z, n.w};
                        const u32 bias = (y & 1) ? 2u : 1u;
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            u32 o = 0;
#pragma unroll
                            for (int e = 0; e < 4; e++) {
                                const u32 av = (cv[comp][q] >> (8 * e)) & 0xffu, nv = (nw[q] >> (8 * e)) & 0xffu;
                                o |= ((3u * av + nv + bias) >> 2) << (8 * e);
                            }
                            cv[comp][q] = o;
                        }
                    }
                }
            }
        }
        u32 w[16];
#pragma unroll
        for (int k = 0; k < 16; k++) w[k] = 0;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const int yy = (int)((yw[k >> 2] >> (8 * (k & 3))) & 0xffu);
            int cb = yy, cr = yy;
            if (color) {
                if (MT::H == 2) {
                    const int t = (k >> 1) + 1;   // s index of this pixel's chroma column
                    if (MT::V == 2) {
                        cb = (k & 1) ? (3 * s[0][t] + s[0][t + 1] + 7) >> 4 : (3 * s[0][t] + s[0][t - 1] + 8) >> 4;
                        cr = (k & 1) ? (3 * s[1][t] + s[1][t + 1] + 7) >> 4 : (3 * s[1][t] + s[1][t - 1] + 8) >> 4;
                    } else {
                        cb = (k & 1) ? (3 * s[0][t] + s[0][t + 1] + 2) >> 2 : (3 * s[0][t] + s[0][t - 1] + 1) >> 2;
                        cr = (k & 1) ? (3 * s[1][t] + s[1][t + 1] + 2) >> 2 : (3 * s[1][t] + s[1][t - 1] + 1) >> 2;
                    }
                } else {
                    cb = (int)((cv[0][k >> 2] >> (8 * (k & 3))) & 0xffu);
                    cr = (int)((cv[1][k >> 2] >> (8 * (k & 3))) & 0xffu);
                }
            }
            u32 p0 = (u32)yy, p1 = (u32)cb, p2 = (u32)cr;
            if (color && !ycc) jfif_rgb(yy, cb, cr, p0, p1, p2);
            if (nc == 4) {
                w[k] = p0 | (p1 << 8) | (p2 << 16) | 0xff000000u;
            } else {
                const u32 px[3] = {p0, p1, p2};
#pragma unroll
                for (int c = 0; c < 3; c++) w[(3 * k + c) >> 2] |= px[c] << (8 * ((3 * k + c) & 3));
            }
        }
        uint8_t *d = im.out + ((size_t)y * width + x0) * nc;
        const int nbytes = npx * nc, nw = 4 * nc;   // bytes of this unit, words of a whole unit
        const uintptr_t a = reinterpret_cast<uintptr_t>(d);
        if (npx == 16 && (a & 15) == 0) {
            uint4 *d4 = reinterpret_cast<uint4 *>(d);
            d4[0] = make_uint4(w[0], w[1], w[2], w[3]);
            d4[1] = make_uint4(w[4], w[5], w[6], w[7]);
            d4[2] = make_uint4(w[8], w[9], w[10], w[11]);
            if (nc == 4) d4[3] = make_uint4(w[12], w[13], w[14], w[15]);
        } else if ((a & 3) == 0) {
            u32 *dw = reinterpret_cast<u32 *>(d);
#pragma unroll
            for (int k = 0; k < 16; k++) if (k < nw && 4 * k + 4 <= nbytes) dw[k] = w[k];
#pragma unroll
            for (int k = 0; k < 16; k++)
                if (k < nw && 4 * k < nbytes && 4 * k + 4 > nbytes)
                    for (int e = 0; e < 3; e++) if (4 * k + e < nbytes) d[4 * k + e] = (uint8_t)(w[k] >> (8 * e));
        } else {
#pragma unroll
            for (int k = 0; k < 64; k++) if (k < nbytes) d[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
        }
    }
}

// ------------------------------------------------------------------------------------- DCT-scaled kernel
// ZJ_VARIANT_SPEC | ZJ_FLAG_ISLOW with ZJ_FLAG_SCALE_* = LOG2D (the statement is in include/zune_jpeg_b200.h): every block becomes
// S0 = 8 >> LOG2D (luma) or SC (chroma: 2 S0 for 4:2:0, else S0) samples a side, so one MCU is H S0 x V S0 output pixels and carries
// one SC x SC chroma block.  4:4:4 and 4:2:0 chroma then needs no up-sampling, 4:2:2 is up-sampled along rows and 4:4:0 down
// columns -- with libjpeg's fancy filters when S0 > 1 (4:2:2: and the chroma is wider than 2), by repetition otherwise.
// grid = (tiles of TS MCU columns, MCU rows, images); block = ZJ_THREADS; one kernel for every output colourspace.
//   phase 1: the tile's luma blocks, then its chroma blocks and the context the fancy filters reach (one block column on each side
//            for 4:2:2, one block row above and below for 4:4:0, where it holds real chroma samples), into shared sample planes;
//            SC = 8 (4:2:0 at 1/2) is the islow IDCT of step 1', whose warp votes need the loop's CTA-uniform trip count;
//   phase 2: one thread per output pixel: up-sampling, JFIF colour, alpha.
template <int MODE, int LOG2D>
__global__ void __launch_bounds__(ZJ_THREADS, ZJ_MINBLOCKS)
scaled_kernel(const DevImage *__restrict__ images)
{
    static_assert(LOG2D >= 1 && LOG2D <= 3, "scales 1/2, 1/4, 1/8");
    typedef ModeTraits<MODE> MT;
    constexpr int S0 = 8 >> LOG2D;
    constexpr int SC = MODE == MODE_HV ? 2 * S0 : S0;
    constexpr int TS = MODE == MODE_NONE ? TS_NONE : (MODE == MODE_H ? TS_H : (MODE == MODE_V ? TS_V : TS_HV));
    constexpr bool FANCY = S0 > 1;
    constexpr int PC = MODE == MODE_H && FANCY ? SC : 0;   // context columns on each side of the chroma tile
    constexpr int PR = MODE == MODE_V && FANCY ? SC : 0;   // context rows above and below it
    constexpr int YW = TS * MT::H * S0, YR = MT::V * S0;   // luma tile
    constexpr int CW = TS * SC + 2 * PC, CR = SC + 2 * PR; // chroma tile
    __shared__ __align__(16) uint8_t sY[YR * YW];
    __shared__ __align__(16) uint8_t sC[2][CR * CW];
    __shared__ u32 sQ[3][32];

    const DevImage &im = images[blockIdx.z];
    const int tile = (int)blockIdx.x, my = (int)blockIdx.y;
    if (tile >= (int)im.n_tiles || my >= (int)im.n_strips) return;
    const int tid = threadIdx.x;
    const int mcu_x = (int)im.mcu_x, width = (int)im.width, height = (int)im.height;
    const int m0 = tile * TS, m1 = min(m0 + TS, mcu_x), tm = m1 - m0;
    const bool color = im.W != 0 && im.out_kind != OUT_GRAY;          // luma only: one-component input or GRAYSCALE output
    const int dw = (int)(im.chroma_wh & 0xffffu), dh = (int)(im.chroma_wh >> 16);
    for (int k = tid; k < 96; k += ZJ_THREADS) sQ[k >> 5][k & 31] = im.qtw[k >> 5][k & 31];
    __syncthreads();

    // ---------------------------------------------------------------- phase 1
    // S x S samples of the block at src into dst (S = 8: every lane of the warp must call it)
    auto transform = [&](auto size, const bool active, const int16_t *src, const u32 *qt, uint8_t *dst, int dstride) {
        constexpr int S = decltype(size)::value;
        int4 raw[8];
        if constexpr (S == 8) {
            load_block(active, src, raw);
            idct_islow_block(active, raw, qt, dst, dstride);
        } else {
            load_rows<S>(active, src, raw);
            if (active) idct_reduced<S>(raw, qt, dst, dstride);
        }
    };
    const int ybpr = MT::H * mcu_x, ycols = MT::H * tm, nY = MT::V * ycols;
    for (int b = tid; b < nY; b += ZJ_THREADS) {
        const int br = b / ycols, bc = b - br * ycols;
        transform(std::integral_constant<int, S0>(), true, im.coeff[0] + ((size_t)(my * MT::V + br) * ybpr + MT::H * m0 + bc) * 64, sQ[0],
                  sY + br * S0 * YW + bc * S0, YW);
    }
    if (color) {
        // chroma block rows [rb0, rb1) and block columns [cb0, cb1), context included
        const int rb0 = my - (PR && my > 0 ? 1 : 0), rb1 = my + 1 + (PR && (my + 1) * SC < dh ? 1 : 0);
        const int cb0 = m0 - (PC && m0 > 0 ? 1 : 0), cb1 = m1 + (PC && m1 * SC < dw ? 1 : 0);
        const int ccols = cb1 - cb0, nC = (rb1 - rb0) * ccols;
        for (int b0 = 0; b0 < 2 * nC; b0 += ZJ_THREADS) {   // CTA-uniform trip count
            const int b = b0 + tid;
            const bool active = b < 2 * nC;
            const int comp = active && b >= nC ? 1 : 0, c = active ? b - comp * nC : 0;
            const int br = rb0 + c / ccols, bc = cb0 + c % ccols;
            transform(std::integral_constant<int, SC>(), active, im.coeff[1 + comp] + ((size_t)br * mcu_x + bc) * 64, sQ[1 + comp],
                      sC[comp] + ((br - my) * SC + PR) * CW + (bc - m0) * SC + PC, CW);
        }
    }
    __syncthreads();

    // ---------------------------------------------------------------- phase 2
    const int nc = (int)im.nc;
    const bool ycc = im.out_kind == OUT_YCC;
    const int x_t = m0 * MT::H * S0, y_t = my * YR;   // first output column / row of the tile
    for (int u = tid; u < YR * YW; u += ZJ_THREADS) {
        const int yl = u / YW, xl = u - yl * YW;
        const int y = y_t + yl, x = x_t + xl;
        if (y >= height || x >= width) continue;
        const int yy = sY[yl * YW + xl];
        u32 p[3] = {(u32)yy, (u32)yy, (u32)yy};
        if (color) {
            int cc[2];
#pragma unroll
            for (int comp = 0; comp < 2; comp++) {
                const uint8_t *s = sC[comp];
                if (MODE == MODE_H) {
                    // chroma column i of the image is smem column i - (m0 SC - PC); the row is the pixel's
                    const uint8_t *row = s + yl * CW - (m0 * SC - PC);
                    const int i = x >> 1;
                    if (FANCY && dw > 2) cc[comp] = (x & 1) ? (3 * row[i] + row[min(i + 1, dw - 1)] + 2) >> 2 : (3 * row[i] + row[max(i - 1, 0)] + 1) >> 2;
                    else cc[comp] = row[i];
                } else if (MODE == MODE_V) {
                    // chroma row j of the image is smem row j - (my SC - PR); the column is the pixel's
                    const uint8_t *col = s + xl - (my * SC - PR) * CW;
                    const int j = y >> 1;
                    if (FANCY) cc[comp] = (y & 1) ? (3 * col[j * CW] + col[min(j + 1, dh - 1) * CW] + 2) >> 2 : (3 * col[j * CW] + col[max(j - 1, 0) * CW] + 1) >> 2;
                    else cc[comp] = col[j * CW];
                } else {
                    cc[comp] = s[yl * CW + xl];
                }
            }
            p[1] = (u32)cc[0]; p[2] = (u32)cc[1];
            if (!ycc) jfif_rgb(yy, cc[0], cc[1], p[0], p[1], p[2]);
        }
        uint8_t *d = im.out + ((size_t)y * width + x) * nc;
        d[0] = (uint8_t)p[0];
        if (nc >= 3) { d[1] = (uint8_t)p[1]; d[2] = (uint8_t)p[2]; }
        if (nc == 4) d[3] = 255;
    }
}

// ------------------------------------------------------------------------------------- per-component kernel
// Images whose components each take their own way (the statements are in include/zune_jpeg_b200.h next to
// zj_decoder_jpeg_colorspace): CMYK / YCCK input (NC = 4), and YCbCr input with sampling factors outside the fused kernels'
// sets (NC = 3).  Each component has its own factors (1..4), block size ss_z (S0 = 8 >> LOG2D, 2 S0 or 4 S0) and integer
// up-sampling ratio (rh_z, rv_z), each 1..4.
// grid = (tiles of tile_mcus MCU columns = at most TC_PIXELS output columns, MCU rows, images); block = ZJ_THREADS.
//   phase 1: every component's blocks of the tile, plus one context block on each side along an axis it is up-sampled on, into a
//            shared plane per component whose sample (j, i) sits at row j - (first row - 8), column i - (first column - 8);
//            blocks of ss = 8 (IDCT: X86 or islow, with warp votes) run in a CTA-uniform loop of their own, reduced ones after;
//   phase 2: one thread per output pixel: up-sampling per component, then JFIF colour (NC = 3) or YCCK -> CMYK and Pillow's
//            CMYK;I -> RGB (NC = 4), output.
__device__ __forceinline__ u32 cmyk_channel(u32 x, u32 nk)   // Convert.c cmyk2rgb: nk - MULDIV255(x, nk)
{
    const u32 t = x * nk + 128;
    return nk - (((t >> 8) + t) >> 8);
}
__device__ __forceinline__ int div_ratio(int x, int r) { return r == 3 ? x / 3 : x >> (r >> 1); }   // x / r, r = 1..4

template <int IDCT, int LOG2D, int NC>
__global__ void __launch_bounds__(ZJ_THREADS, 2)
raster_kernel(const RasterImage *__restrict__ images)
{
    static_assert(LOG2D == 0 || IDCT == IDCT_ISLOW, "DCT scaling is libjpeg output only");
    static_assert(NC == 3 || NC == 4, "three or four components");
    constexpr int S0 = 8 >> LOG2D;
    constexpr bool FANCY = S0 > 1;
    // shared plane: 8 + TC_PIXELS + 8 columns; 8 rows above, then an MCU row of up to 32 rows (ratio 1), or up to 16 rows and 8 of
    // context below (ratio 2; ratios 3 and 4 need less)
    constexpr int PS = 144, PR = 40;
    __shared__ __align__(16) uint8_t sP[NC][PR * PS];
    __shared__ u32 sQ[NC][32];

    const RasterImage &im = images[blockIdx.z];
    const int tile = (int)blockIdx.x, my = (int)blockIdx.y;
    if (tile >= (int)im.n_tiles || my >= (int)im.mcu_y) return;
    const int tid = threadIdx.x;
    const int m0 = tile * (int)im.tile_mcus, m1 = min(m0 + (int)im.tile_mcus, (int)im.mcu_x);
    for (int k = tid; k < 32 * NC; k += ZJ_THREADS) sQ[k >> 5][k & 31] = im.qtw[k >> 5][k & 31];

    // block rows [rb0, rb1) x columns [cb0, cb1) of each component, context included; its plane origin (c0, r0) in samples
    int rb0[NC], cb0[NC], ncol[NC], nblk[NC], c0[NC], r0[NC];
#pragma unroll
    for (int z = 0; z < NC; z++) {
        const int h = (int)im.h[z], v = (int)im.v[z], ss = (int)im.ss[z];
        const bool uh = (im.ratio[z] & 255u) > 1, uv = im.ratio[z] > 255u;   // up-sampled along x / y
        const int a0 = m0 * h, a1 = m1 * h, b0 = my * v, b1 = (my + 1) * v;
        cb0[z] = a0 - (uh && a0 > 0 ? 1 : 0);
        const int cb1 = a1 + (uh && a1 * ss < (int)im.dw[z] ? 1 : 0);
        rb0[z] = b0 - (uv && b0 > 0 ? 1 : 0);
        const int rb1 = b1 + (uv && b1 * ss < (int)im.dh[z] ? 1 : 0);
        ncol[z] = cb1 - cb0[z];
        nblk[z] = ncol[z] * (rb1 - rb0[z]);
        c0[z] = a0 * ss - 8;
        r0[z] = b0 * ss - 8;
    }
    __syncthreads();

    // ---------------------------------------------------------------- phase 1
    // block b of the components whose block size is (full) 8 or (!full) smaller: component, source and destination (src stays
    // NULL past the last block)
    auto locate = [&](const bool full, int b, int &z, const int16_t *&src, uint8_t *&dst) {
#pragma unroll
        for (int k = 0; k < NC; k++) {
            if (src || ((int)im.ss[k] == 8) != full) continue;
            if (b >= nblk[k]) { b -= nblk[k]; continue; }
            const int ss = (int)im.ss[k];
            const int br = rb0[k] + b / ncol[k], bc = cb0[k] + b % ncol[k];
            src = im.coeff[k] + ((size_t)br * im.bpr[k] + bc) * 64;
            dst = sP[k] + (br * ss - r0[k]) * PS + (bc * ss - c0[k]);
            z = k;
        }
    };
    int n_full = 0, n_red = 0;
#pragma unroll
    for (int k = 0; k < NC; k++) (im.ss[k] == 8 ? n_full : n_red) += nblk[k];
    for (int b0 = 0; b0 < n_full; b0 += ZJ_THREADS) {   // CTA-uniform trip count: every lane takes part in the warp votes
        int z = 0;
        const int16_t *src = nullptr;
        uint8_t *dst = sP[0];
        if (b0 + tid < n_full) locate(true, b0 + tid, z, src, dst);
        const bool active = src != nullptr;
        int4 raw[8];
        load_block(active, src, raw);
        if constexpr (IDCT == IDCT_ISLOW) idct_islow_block(active, raw, sQ[active ? z : 0], dst, PS);
        else idct_block<0, uint8_t>(active, raw, sQ[active ? z : 0], dst, PS);
    }
    if constexpr (S0 < 8) {
        for (int b = tid; b < n_red; b += ZJ_THREADS) {
            int z = 0;
            const int16_t *src = nullptr;
            uint8_t *dst = nullptr;
            locate(false, b, z, src, dst);
            int4 raw[8];
            const int ss = (int)im.ss[z];   // S0, 2 S0 or 4 S0, below 8
            if (ss == S0) {
                load_rows<S0>(true, src, raw);
                idct_reduced<S0>(raw, sQ[z], dst, PS);
            } else if constexpr (2 * S0 < 8) {
                if (ss == 2 * S0) {
                    load_rows<2 * S0>(true, src, raw);
                    idct_reduced<2 * S0>(raw, sQ[z], dst, PS);
                } else if constexpr (4 * S0 < 8) {
                    load_rows<4 * S0>(true, src, raw);
                    idct_reduced<4 * S0>(raw, sQ[z], dst, PS);
                }
            }
        }
    }
    __syncthreads();

    // ---------------------------------------------------------------- phase 2
    const int width = (int)im.width, height = (int)im.height, nc = (int)im.nc;
    const int mw = (int)im.hmax * S0, mh = (int)im.vmax * S0;   // output pixels per MCU
    const int tw = (m1 - m0) * mw;
    for (int u = tid; u < tw * mh; u += ZJ_THREADS) {
        const int yl = u / tw, xl = u - yl * tw;
        const int x = m0 * mw + xl, y = my * mh + yl;
        if (x >= width || y >= height) continue;
        u32 s[NC];
#pragma unroll
        for (int z = 0; z < NC; z++) {
            const int dw = (int)im.dw[z], dh = (int)im.dh[z], rh = (int)(im.ratio[z] & 255u), rv = (int)(im.ratio[z] >> 8);
            const uint8_t *p = sP[z];
            const int i = div_ratio(x, rh), j = div_ratio(y, rv);
            auto at = [&](int jj, int ii) { return (int)p[(jj - r0[z]) * PS + (ii - c0[z])]; };
            int val;
            if (rh == 2 && rv == 2 && FANCY && dw > 2) {         // HV: s[i] = 3 c[j][i] + c[j'][i]
                const int jn = (y & 1) ? min(j + 1, dh - 1) : max(j - 1, 0);
                const int in = (x & 1) ? min(i + 1, dw - 1) : max(i - 1, 0);
                const int si = 3 * at(j, i) + at(jn, i), sn = 3 * at(j, in) + at(jn, in);
                val = (x & 1) ? (3 * si + sn + 7) >> 4 : (3 * si + sn + 8) >> 4;
            } else if (rh == 2 && rv == 1 && FANCY && dw > 2) {  // H
                const int in = (x & 1) ? min(i + 1, dw - 1) : max(i - 1, 0);
                val = (3 * at(j, i) + at(j, in) + 1 + (x & 1)) >> 2;
            } else if (rh == 1 && rv == 2 && FANCY) {            // V
                const int jn = (y & 1) ? min(j + 1, dh - 1) : max(j - 1, 0);
                val = (3 * at(j, i) + at(jn, i) + 1 + (y & 1)) >> 2;
            } else {                                             // no up-sampling, or rh x rv repetition
                val = at(j, i);
            }
            s[z] = (u32)val;
        }
        uint8_t *d = im.out + ((size_t)y * width + x) * nc;
        if constexpr (NC == 3) {
            if (im.kind == RASTER_OUT_GRAY) {   // the Y plane
                d[0] = (uint8_t)s[0];
                continue;
            }
            if (im.kind == RASTER_OUT_RAW) {    // YCbCr
                d[0] = (uint8_t)s[0]; d[1] = (uint8_t)s[1]; d[2] = (uint8_t)s[2];
                continue;
            }
            u32 r, g, b;
            jfif_rgb((int)s[0], (int)s[1], (int)s[2], r, g, b);
            d[0] = (uint8_t)r; d[1] = (uint8_t)g; d[2] = (uint8_t)b;
            if (nc == 4) d[3] = 255;
        } else {
            // Pillow's CMYK;I bytes: YCCK -> libjpeg's CMYK (255 - (Y + chroma term), clamped) inverted is the JFIF RGB of (Y, Cb, Cr)
            u32 c, m, ye;
            if (im.model == RASTER_YCCK) jfif_rgb((int)s[0], (int)s[1], (int)s[2], c, m, ye);
            else { c = 255 - s[0]; m = 255 - s[1]; ye = 255 - s[2]; }
            const u32 nk = s[3];
            if (im.kind == RASTER_OUT_RAW) {    // CMYK
                d[0] = (uint8_t)c; d[1] = (uint8_t)m; d[2] = (uint8_t)ye; d[3] = (uint8_t)(255 - nk);
                continue;
            }
            const u32 r = cmyk_channel(c, nk), g = cmyk_channel(m, nk), b = cmyk_channel(ye, nk);
            if (im.kind == RASTER_OUT_GRAY) {
                d[0] = (uint8_t)((19595 * r + 38470 * g + 7471 * b + 32768) >> 16);
                continue;
            }
            d[0] = (uint8_t)r; d[1] = (uint8_t)g; d[2] = (uint8_t)b;
            if (nc == 4) d[3] = 255;
        }
    }
}

template <int NC>
static void launch_raster_nc(dim3 grid, const RasterImage *p, const LaunchGroup &g, cudaStream_t stream)
{
    if (!g.islow) raster_kernel<IDCT_X86, 0, NC><<<grid, ZJ_THREADS, 0, stream>>>(p);
    else if (g.scale == 0) raster_kernel<IDCT_ISLOW, 0, NC><<<grid, ZJ_THREADS, 0, stream>>>(p);
    else if (g.scale == 1) raster_kernel<IDCT_ISLOW, 1, NC><<<grid, ZJ_THREADS, 0, stream>>>(p);
    else if (g.scale == 2) raster_kernel<IDCT_ISLOW, 2, NC><<<grid, ZJ_THREADS, 0, stream>>>(p);
    else raster_kernel<IDCT_ISLOW, 3, NC><<<grid, ZJ_THREADS, 0, stream>>>(p);
}

cudaError_t launch_raster(const RasterImage *d_images, const LaunchGroup &g, cudaStream_t stream)
{
    dim3 grid(g.max_tiles, g.max_strips, g.count);   // max_strips: MCU rows
    const RasterImage *p = d_images + g.first;
    if (g.raster == 4) launch_raster_nc<4>(grid, p, g, stream);
    else launch_raster_nc<3>(grid, p, g, stream);
    return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------- host launchers
template <int MODE>
static cudaError_t launch_spec(const DevImage *d_images, const LaunchGroup &g, cudaStream_t stream)
{
    dim3 grid(g.max_tiles, g.max_strips, g.count);
    if (g.islow) spec_kernel<MODE, IDCT_ISLOW><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first);
    else spec_kernel<MODE, IDCT_X86><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first);
    return cudaGetLastError();
}

template <int MODE>
static cudaError_t launch_scaled(const DevImage *d_images, const LaunchGroup &g, cudaStream_t stream)
{
    dim3 grid(g.max_tiles, g.max_strips, g.count);   // max_strips: MCU rows
    if (g.scale == 1) scaled_kernel<MODE, 1><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first);
    else if (g.scale == 2) scaled_kernel<MODE, 2><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first);
    else scaled_kernel<MODE, 3><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first);
    return cudaGetLastError();
}

template <int MODE, int VARIANT>
static cudaError_t launch_reconstruct(const DevImage *d_images, const LaunchGroup &g, cudaStream_t stream)
{
    dim3 grid(g.max_tiles, g.max_strips + 1, g.count);
    reconstruct_kernel<MODE, VARIANT><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------- luma-only kernel, fast variant
// (YCbCr | GRAYSCALE) -> GRAYSCALE for the X86 variant, built from the same parts as reconstruct_fast_kernel: four
// producer warps stage coefficients with cp.async and run the rolled IDCT into double-buffered sample planes, four
// consumer warps copy the planes out in 16-byte row segments.  A CTA owns one tile column (up to 512 samples) of `spc`
// consecutive "strips" of TWO luma block rows (16 image rows; 128 blocks = one IDCT pass).  The plane is just a raster of
// blocks here -- the reference's strip geometry only decides how many block rows exist (DevImage::gray_brows).
constexpr int ZG_TW = 512, ZG_ROWS = 16, ZG_BUF = ZG_TW * ZG_ROWS;   // tile width, rows per strip, bytes per plane buffer

__global__ void __launch_bounds__(ZF_THREADS, 3)
gray_fast_kernel(const DevImage *__restrict__ images, const int spc)
{
    extern __shared__ __align__(128) uint8_t sDynAll[];  // [staging 16 KB | scratch 32 KB | zero slot | 2 plane buffers]
    uint8_t *const sPlanes = sDynAll + 3 * ZF_PRODUCERS * 128 + 128;
    __shared__ __align__(16) u32 sQ[32];

    const DevImage &im = images[blockIdx.z];
    const u32 tile = blockIdx.x;
    if (tile >= im.n_tiles) return;
    const int tid = threadIdx.x;
    const u32 stride = im.stride, width = im.width, height = im.height;
    uint8_t *__restrict__ out = im.out;
    const u32 brows = im.gray_brows;                       // luma block rows the reference processes
    const u32 n_strips = (brows + 1) / 2;
    const u32 s_begin = blockIdx.y * (u32)spc;
    if (s_begin >= n_strips) {
        // rows below the processed block rows stay zero (Q1); written by the first row of CTAs past the image's strips
        if (s_begin >= n_strips + (u32)spc) return;
        const size_t lo = (size_t)min(brows * 8u, height) * stride, hi = (size_t)height * stride;
        if (lo >= hi) return;
        const size_t span = hi - lo, per = (span + im.n_tiles - 1) / im.n_tiles;
        size_t b0 = lo + (size_t)tile * per, b1 = b0 + per;
        if (b1 > hi) b1 = hi;
        for (size_t b = b0 + tid; b < b1; b += ZF_THREADS) out[b] = 0;
        return;
    }
    const int n_it = (int)(min(s_begin + (u32)spc, n_strips) - s_begin);
    const int u0 = (int)(tile * im.tile_q + min(tile, im.tile_r)), u1 = (int)((tile + 1) * im.tile_q + min(tile + 1, im.tile_r));
    const int Wp = (int)im.Wp, ybpr = Wp >> 3;
    const int X0 = 16 * u0, yb0 = 2 * u0, nyb = min(2 * u1, ybpr) - yb0;   // luma block columns of the tile
    if (tid < 32) sQ[tid] = im.qtw[0][tid];
    __syncthreads();

    if (tid < ZF_PRODUCERS) {
        const int lane = tid & 31, wq = tid >> 5;
        const int br = wq >> 1, bc0 = (wq & 1) * 32;         // the warp's block row inside the strip, first block column
        const bool active = bc0 + lane < nyb;
        const bool work = bc0 < nyb;
        const u32 dsto = (u32)(br * 8 * ZG_TW + (bc0 + lane) * 8);
        const u32 step = (u32)(2 * ybpr * 64);                // i16 per strip
        const int16_t *q0 = im.coeff[0] + (((size_t)s_begin * 2 + br) * ybpr + yb0 + bc0) * 64 + (lane >> 3) * 64 + (lane & 7) * 8;
        u32 jm = 0;                                            // bit k: chunk k of the cooperative copy is inside the run
        for (int k = 0; k < 8; k++) if (4 * k + (lane >> 3) < min(max(nyb - bc0, 0), 32)) jm |= 1u << k;
        const u32 stage0 = (u32)__cvta_generic_to_shared(sDynAll) + (u32)(wq * 32) * 128u;
        const u32 d_even = stage0 + (u32)(lane >> 3) * 128u + (u32)(((lane & 7) ^ (lane >> 3)) * 16);
        const u32 d_odd = stage0 + (u32)(lane >> 3) * 128u + (u32)(((lane & 7) ^ ((lane >> 3) + 4)) * 16);
        const u32 slx = (stage0 + (u32)lane * 128u) | (u32)((lane & 7) * 16);
        const u32 scr = (u32)__cvta_generic_to_shared(sDynAll) + ZF_PRODUCERS * 128u + (u32)tid * 16u;
        const u32 zslot = ((u32)__cvta_generic_to_shared(sDynAll) + 3u * ZF_PRODUCERS * 128u) | (u32)((lane & 7) * 16);
        if (tid < 8) sts128(zslot - (u32)((lane & 7) * 16) + (u32)tid * 16u, 0u, 0u, 0u, 0u);
        asm volatile("bar.sync %0, %1;" ::"r"(6), "n"(ZF_PRODUCERS) : "memory");   // producers only
        auto issue = [&](const int16_t *g, const bool valid) {
            if (valid) {
#pragma unroll
                for (int k = 0; k < 8; k++)
                    if (jm & (1u << k))
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(((k & 1) ? d_odd : d_even) + k * 512u), "l"(g + k * 256) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        // the last strip of an image with an odd number of block rows has no second block row: nothing to read there
        auto row_exists = [&](int it) { return (s_begin + (u32)it) * 2 + (u32)br < brows; };
        issue(q0, row_exists(0));
        q0 += step;
        for (int it = 0; it < n_it; it++) {
            uint8_t *planes = sPlanes + (it & 1) * ZG_BUF;
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncwarp();
            if (it >= 2) bar_sync(BAR_EMPTY + (it & 1));
            auto refill = [&]() {
                if (it + 1 < n_it) { issue(q0, row_exists(it + 1)); q0 += step; }
            };
            if (work && row_exists(it)) idct_rolled<4, false>(active, active ? slx : zslot, scr, sQ, planes + dsto, ZG_TW, refill);
            else refill();
            bar_arrive(BAR_FULL + (it & 1));
        }
        return;
    }

    // consumers: four 16-sample units per thread and strip (rows rg, rg+4, rg+8, rg+12 of the strip)
    const int tc = tid - ZF_PRODUCERS;
    const int xu = tc & 31, rgA = tc >> 5;
    const int xs = X0 + 16 * xu, xl = 16 * xu;
    const int npx = (u0 + xu < u1) ? min(max((int)width - xs, 0), 16) : 0;     // samples of the unit inside the image row
    const bool vec = npx == 16 && (stride & 15u) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    const bool words = npx == 16 && (stride & 3u) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0;
    for (int it = 0; it < n_it; it++) {
        const uint8_t *planes = sPlanes + (it & 1) * ZG_BUF;
        const u32 y_base = (s_begin + (u32)it) * ZG_ROWS;
        bar_sync(BAR_FULL + (it & 1));
        if (npx > 0) {
#pragma unroll
            for (int h = 0; h < 4; h++) {
                const int rg = rgA + 4 * h;
                const u32 y = y_base + (u32)rg;
                if (y >= height) continue;
                uint4 v = make_uint4(0u, 0u, 0u, 0u);
                if (y < brows * 8u) v = *reinterpret_cast<const uint4 *>(planes + rg * ZG_TW + xl);   // `as u8` row copy (scalar.rs:91-114)
                uint8_t *d = out + (size_t)y * stride + xs;
                if (vec) *reinterpret_cast<uint4 *>(d) = v;
                else if (words) { u32 *dw = reinterpret_cast<u32 *>(d); dw[0] = v.x; dw[1] = v.y; dw[2] = v.z; dw[3] = v.w; }
                else {
                    const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 16; k++) if (k < npx) d[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
                }
            }
        }
        if (it + 2 < n_it) bar_arrive(BAR_EMPTY + (it & 1));
    }
}

// Strips per CTA of the fast kernels.  A CTA pays one pipeline fill / drain per strip range, so ranges should be long
// (about ZF_DEFAULT_SPC strips, equal parts of the image); but the launch must still offer a few CTAs per resident slot
// (3 per SM), so small batches are cut finer.  ZJ_SPC in the environment overrides.
static int strips_per_cta(const LaunchGroup &g)
{
    static int forced = -1, slots = 0;
    if (forced < 0) {
        const char *e = getenv("ZJ_SPC");
        forced = e ? (atoi(e) < 1 ? 1 : atoi(e)) : 0;
    }
    if (forced) return forced;
    if (slots == 0) {
        int dev = 0, sms = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        slots = 3 * sms;
    }
    const long S = g.max_strips > 0 ? (long)g.max_strips : 1;
    long parts = (S + ZF_DEFAULT_SPC - 1) / ZF_DEFAULT_SPC;
    const long columns = (long)g.max_tiles * (long)g.count;
    while (columns * parts < 2L * slots && S / parts > 4) parts++;
    return (int)((S + parts - 1) / parts);
}

template <int MODE>
static cudaError_t launch_fast(const DevImage *d_images, const LaunchGroup &g, cudaStream_t stream)
{
    const int spc = strips_per_cta(g);
    dim3 grid(g.max_tiles, (g.max_strips + spc - 1) / spc + 1, g.count);
    typedef FastTraits<MODE> FT;
    constexpr size_t smem = 3 * ZF_PRODUCERS * 128 + 128 + (size_t)ZF_NB * FT::BUF;
    static bool configured[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(reconstruct_fast_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    reconstruct_fast_kernel<MODE><<<grid, ZF_THREADS, smem, stream>>>(d_images + g.first, spc);
    return cudaGetLastError();
}

static cudaError_t launch_gray_fast(const DevImage *d_images, const LaunchGroup &g, cudaStream_t stream)
{
    const int spc = strips_per_cta(g);
    dim3 grid(g.max_tiles, (g.max_strips + spc - 1) / spc + 1, g.count);   // max_strips: pairs of block rows
    constexpr size_t smem = 3 * ZF_PRODUCERS * 128 + 128 + 2 * ZG_BUF;
    static bool configured[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(gray_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    gray_fast_kernel<<<grid, ZF_THREADS, smem, stream>>>(d_images + g.first, spc);
    return cudaGetLastError();
}

cudaError_t launch_group(const DevImage *d_images, const LaunchGroup &g, cudaStream_t stream)
{
    if (g.scale) {
        switch (g.mode) {
        case MODE_NONE: return launch_scaled<MODE_NONE>(d_images, g, stream);
        case MODE_H: return launch_scaled<MODE_H>(d_images, g, stream);
        case MODE_V: return launch_scaled<MODE_V>(d_images, g, stream);
        default: return launch_scaled<MODE_HV>(d_images, g, stream);
        }
    }
    if (g.gray && g.fast) return launch_gray_fast(d_images, g, stream);
    if (g.variant == ZJ_VARIANT_SPEC && !g.gray) {
        switch (g.mode) {
        case MODE_NONE: return launch_spec<MODE_NONE>(d_images, g, stream);
        case MODE_H: return launch_spec<MODE_H>(d_images, g, stream);
        case MODE_V: return launch_spec<MODE_V>(d_images, g, stream);
        default: return launch_spec<MODE_HV>(d_images, g, stream);
        }
    }
    if (g.fast) {
        switch (g.mode) {
        case MODE_NONE: return launch_fast<MODE_NONE>(d_images, g, stream);
        case MODE_H: return launch_fast<MODE_H>(d_images, g, stream);
        case MODE_V: return launch_fast<MODE_V>(d_images, g, stream);
        default: return launch_fast<MODE_HV>(d_images, g, stream);
        }
    }
    if (g.gray) {
        const int rows = g.mode == MODE_NONE ? 8 : (g.mode == MODE_HV ? 32 : 16);
        dim3 grid(g.max_tiles, g.max_strips * (rows >> 3) + 1, g.count);
        if (g.islow) gray_kernel<IDCT_ISLOW><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first, rows);
        else if (g.variant != ZJ_VARIANT_SCALAR) gray_kernel<0><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first, rows);   // X86 or SPEC
        else gray_kernel<1><<<grid, ZJ_THREADS, 0, stream>>>(d_images + g.first, rows);
        return cudaGetLastError();
    }
    switch (g.mode * 2 + g.variant) {
    case MODE_NONE * 2 + 0: return launch_reconstruct<MODE_NONE, 0>(d_images, g, stream);
    case MODE_NONE * 2 + 1: return launch_reconstruct<MODE_NONE, 1>(d_images, g, stream);
    case MODE_H * 2 + 0: return launch_reconstruct<MODE_H, 0>(d_images, g, stream);
    case MODE_H * 2 + 1: return launch_reconstruct<MODE_H, 1>(d_images, g, stream);
    case MODE_V * 2 + 0: return launch_reconstruct<MODE_V, 0>(d_images, g, stream);
    case MODE_V * 2 + 1: return launch_reconstruct<MODE_V, 1>(d_images, g, stream);
    case MODE_HV * 2 + 0: return launch_reconstruct<MODE_HV, 0>(d_images, g, stream);
    default: return launch_reconstruct<MODE_HV, 1>(d_images, g, stream);
    }
}

}  // namespace zj
