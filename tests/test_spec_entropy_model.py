"""A pure-Python model of the self-synchronising entropy decode of zj_entropy.cu (DESIGN.md section 5.5): de-stuff, sync
rounds to the fixpoint, count + exclusive scan, write, DC prefix sum.  It must give the host stage's spec planes exactly
(Decoder.decode_coefficients with spec output), with subsequences of 32-256 bits so that every file has many boundaries and
some need more than one round, and it must turn down what the GPU form turns down."""
import io

import numpy as np
import pytest

import jpeg_util
from zune_jpeg_b200.decoder import Decoder, ZuneJpegOptions

UNZIGZAG = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
            35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]
INVALID = None


class Table:
    """build_huffman of zj_host_decoder.cpp (huffman.rs) without Q9: lookup, fast-AC table, maxcode, offset, values"""

    def __init__(self, counts, values, is_dc):
        self.values = list(values) + [0] * (256 - len(values))
        self.lookup = [10 << 9] * 512
        self.maxcode, self.offset = [0] * 18, [0] * 18
        size = [l for l in range(1, 17) for _ in range(counts[l - 1])]
        code, k, si = [0] * len(size), 0, size[0] if size else 0
        c = 0
        while k < len(size):
            while k < len(size) and size[k] == si:
                code[k] = c
                c += 1
                k += 1
            self.maxcode[si] = c << (16 - si)
            c <<= 1
            si += 1
        k = 0
        for l in range(17):
            n = counts[l - 1] if l else 0
            if n == 0:
                self.maxcode[l] = -1
            else:
                self.offset[l] = k - code[k]
                k += n
        self.maxcode[17] = 0x000FFFFF
        for i, (s, cd) in enumerate(zip(size, code)):
            if s <= 9:
                for j in range(1 << (9 - s)):
                    self.lookup[(cd << (9 - s)) + j] = (s << 9) | self.values[i]
        self.ac = [0] * 512
        if not is_dc:
            fast = [255] * 512
            for i, (s, cd) in enumerate(zip(size, code)):
                if s <= 9:
                    for j in range(1 << (9 - s)):
                        fast[(cd << (9 - s)) + j] = i
            for i in range(512):
                if fast[i] == 255:
                    continue
                rs = self.values[fast[i]]
                run, mag, ln = rs >> 4, rs & 15, size[fast[i]]
                if mag == 0:
                    self.ac[i] = ((run or 63) << 4) + ln
                elif ln + mag <= 9:
                    kk = ((i << ln) & 511) >> (9 - mag)
                    if kk < (1 << (mag - 1)):
                        kk += (-1 << mag) + 1
                    if -32 <= kk <= 31:
                        self.ac[i] = (kk << 10) + (run << 4) + ln + mag


def extend(x, s):
    return x - (1 << s) + 1 if x < (1 << (s - 1)) else x


class Jpeg:
    """headers of a baseline file (what the spec branch of gpu_entropy_prepare needs) and the host stage's plane geometry"""

    def __init__(self, data):
        self.data, p = data, 2
        dc, ac, self.dri = {}, {}, 0
        while True:
            assert data[p] == 0xFF
            m, ln = data[p + 1], int.from_bytes(data[p + 2:p + 4], "big")
            seg = data[p + 4:p + 2 + ln]
            if m == 0xC0:
                self.h, self.w, nc = int.from_bytes(seg[1:3], "big"), int.from_bytes(seg[3:5], "big"), seg[5]
                self.comps = [(seg[6 + 3 * i], seg[7 + 3 * i] >> 4, seg[7 + 3 * i] & 15) for i in range(nc)]
            elif m == 0xC4:
                q = 0
                while q < len(seg):
                    tc, th, counts = seg[q] >> 4, seg[q] & 15, list(seg[q + 1:q + 17])
                    vals = seg[q + 17:q + 17 + sum(counts)]
                    (ac if tc else dc)[th] = Table(counts, vals, not tc)
                    q += 17 + sum(counts)
            elif m == 0xDD:
                self.dri = int.from_bytes(seg[0:2], "big")
            elif m == 0xDA:
                sel = {seg[1 + 2 * i]: seg[2 + 2 * i] for i in range(seg[0])}
                self.tables = [(dc[sel[cid] >> 4], ac[sel[cid] & 15]) for cid, _, _ in self.comps]
                self.scan = p + 2 + ln
                break
            p += 2 + ln
        hm, vm = max(c[1] for c in self.comps), max(c[2] for c in self.comps)
        mcu_x, mcu_y = -(-self.w // (8 * hm)), -(-self.h // (8 * vm))
        self.bias, self.is_hv = 1, hm == 2 and vm == 2
        if hm != 1 or vm != 1:
            strips2 = (mcu_y + 1) // 2
            self.mcu_w, self.mcu_h = (mcu_x * 2, strips2) if (hm, vm) == (2, 1) else ((mcu_x, strips2) if self.is_hv else (mcu_x, mcu_y))
            self.bias = 2 if self.is_hv else 1
        else:
            self.mcu_w, self.mcu_h = -(-self.w // 8), -(-self.h // 8)
        self.total = mcu_x * mcu_y if (hm, vm) in ((2, 1), (2, 2)) else self.mcu_w * self.mcu_h * self.bias
        cap = self.mcu_w * 64
        y = self.comps[0]
        self.width_stride = (cap * y[1] * y[2] * self.bias) >> 1
        self.hv_stride = self.width_stride >> 1
        self.strip_len = [cap * c[1] * c[2] * self.bias for c in self.comps]
        self.slots = [(z, v, h) for z, c in enumerate(self.comps) for v in range(c[2]) for h in range(c[1])]

    def block(self, g):
        """mcu.rs:293-312 for global block g: (component, offset) or None when the reference would index outside the strip"""
        bpm = len(self.slots)
        m, (z, vs_, hs_) = g // bpm, self.slots[g % bpm]
        _, hs, vs = self.comps[z]
        per_strip = self.bias * self.mcu_w
        strip, v = m // per_strip, (m % per_strip) // self.mcu_w
        j = m - strip * per_strip - v * self.mcu_w
        is_y = 1 if self.comps[z][0] == 1 else 0
        start = (j * 64 * hs + hs_ * 64 + (self.hv_stride if self.is_hv else self.width_stride) * vs_ +
                 is_y * v * (self.hv_stride * vs) + ((self.width_stride >> 2) * v if self.is_hv and not is_y else 0))
        if start + 64 > self.strip_len[z]:
            return None
        return z, strip * self.strip_len[z] + start


def destuff(data, p):
    """phase 1: the scan as the bit reader sees it; None unless the first marker behind it is EOI"""
    out = bytearray()
    while p < len(data):
        b = data[p]
        p += 1
        if b != 0xFF:
            out.append(b)
            continue
        while p < len(data) and data[p] == 0xFF:
            p += 1
        if p >= len(data):
            return None
        nxt = data[p]
        p += 1
        if nxt == 0x00:
            out.append(0xFF)
            continue
        return bytes(out) if nxt == 0xD9 else None
    return None


class Bits:
    def __init__(self, b):
        self.n = len(b) * 8
        self.v = int.from_bytes(b + bytes(8), "big")
        self.top = self.n + 64

    def peek(self, pos, k):
        return (self.v >> (self.top - pos - k)) & ((1 << k) - 1)


def huff(bits, pos, t, sym):
    """decode_huff!: (symbol, new pos) or None"""
    ln = sym >> 9
    sym &= 511
    if ln > 9:
        s16 = bits.peek(pos, 16)
        while ln < 17 and not s16 < t.maxcode[ln]:
            ln += 1
        if ln == 17:
            return None
        sym = t.values[((s16 >> (16 - ln)) + t.offset[ln]) & 0xFF]
    return sym, pos + ln


def decode(j, bits, state, end, write=None):
    """sync_decode: from state (pos, slot, coef) over the symbols that start below `end`; returns (exit or INVALID, blocks).
    write = (g0, total, planes, dc): store coefficients / DC differences of blocks below total, stop at total."""
    pos, slot, coef = state
    bpm, blocks = len(j.slots), 0
    cur = None
    if write:
        g0, total, planes, dcd = write
        if g0 >= total:
            return state, 0
        cur = j.block(g0)
    while pos < end:
        z = j.slots[slot][0]
        dc, ac = j.tables[z]
        if coef == 0:
            r = huff(bits, pos, dc, dc.lookup[bits.peek(pos, 9)])
            if r is None:
                return INVALID, blocks
            s, pos = r
            v = extend(bits.peek(pos, s), s) if s else 0
            pos += s
            if write:
                dcd[g0 + blocks] = v
            coef = 1
        else:
            f = ac.ac[bits.peek(pos, 9)]
            if f:
                coef += (f >> 4) & 63
                v = f >> 10
                if v:
                    if coef > 63:
                        return INVALID, blocks
                    if write and cur:
                        planes[cur[0]][cur[1] + UNZIGZAG[coef]] = v
                pos += f & 15
                coef += 1
            else:
                r = huff(bits, pos, ac, ac.lookup[bits.peek(pos, 9)])
                if r is None:
                    return INVALID, blocks
                s, pos = r
                rr, s = s >> 4, s & 15
                if s:
                    coef += rr
                    if coef > 63:
                        return INVALID, blocks
                    v = extend(bits.peek(pos, s), s)
                    pos += s
                    if write and cur:
                        planes[cur[0]][cur[1] + UNZIGZAG[coef]] = v
                    coef += 1
                elif rr != 15:
                    coef = 64
                else:
                    coef += 16
        if pos > bits.n:
            return INVALID, blocks
        if coef >= 64:
            blocks, coef, slot = blocks + 1, 0, (slot + 1) % bpm
            if write:
                if g0 + blocks >= total:
                    break
                cur = j.block(g0 + blocks)
                if cur is None:
                    raise AddressError
    return (pos, slot, coef), blocks


class AddressError(Exception):
    pass


def model(data, S, max_rounds=None):
    """phases 1-5; (planes, rounds) or (None, reason).  max_rounds None: n_sub + 2, which always reaches the fixpoint (after
    round r the entries of subsequences 0..r are true)"""
    j = Jpeg(data)
    if j.dri:
        return None, "dri"
    scan = destuff(data, j.scan)
    if not scan:
        return None, "no EOI behind the scan"
    bits = Bits(scan)
    n = -(-bits.n // S)
    ends = [min(bits.n, (k + 1) * S) for k in range(n)]
    ends[-1] = bits.n
    guess = [(k * S, 0, 0) for k in range(n)]
    used, exits, counts = [None] * n, [None] * n, [0] * n
    rounds = 0
    for r in range(max_rounds or n + 2):                                    # phase 2: sync rounds
        prev, changed = list(exits), 0
        for k in range(n):
            e = guess[k] if (k == 0 or r == 0 or prev[k - 1] is INVALID) else prev[k - 1]
            if r > 0 and e == used[k]:
                continue
            used[k] = e
            exits[k], counts[k] = decode(j, bits, e, ends[k])
            changed += 1
        rounds = r + 1
        if r > 0 and changed == 0:
            break
    else:
        return None, "not settled"
    base = [0] * n                                                 # phase 3: exclusive scan
    for k in range(1, n):
        base[k] = base[k - 1] + counts[k - 1]
    total = j.total * len(j.slots)
    err = next((k for k in range(n) if exits[k] is INVALID), None)
    reached = base[err] + counts[err] if err is not None else base[-1] + counts[-1]
    if reached < total:
        return None, "fewer blocks than the frame holds"
    planes = [np.zeros(j.strip_len[z] * j.mcu_h, np.int64) for z in range(len(j.comps))]
    dcd = [0] * total
    try:                                                           # phase 4: write
        for k in range(n):
            entry = (0, 0, 0) if k == 0 else exits[k - 1]
            if base[k] >= total or entry is INVALID:
                continue
            if j.block(base[k]) is None:
                raise AddressError
            decode(j, bits, entry, ends[k], (base[k], total, planes, dcd))
    except AddressError:
        return None, "addressing"
    pred = [0] * len(j.comps)                                      # phase 5: DC, wrapping 32-bit, stored as int16
    for g in range(total):
        z = j.slots[g % len(j.slots)][0]
        pred[z] = (pred[z] + dcd[g]) & 0xFFFFFFFF
        at = j.block(g)
        planes[z][at[1]] = (pred[z] ^ 0x8000) & 0xFFFF
        planes[z][at[1]] -= 0x8000
    return [p.astype(np.int16) for p in planes], rounds


def _enc(seed, w, h, sub, q, optimize=False, gray=False):
    im = jpeg_util.smooth_image(seed, w, h, gray, noise=12)
    bio = io.BytesIO()
    kw = dict(quality=q, optimize=optimize)
    if not gray:
        kw["subsampling"] = jpeg_util.SUBSAMPLING[sub]
    im.save(bio, "JPEG", **kw)
    return bio.getvalue()


def _host(data):
    _, planes = Decoder.new_with_options(ZuneJpegOptions().set_spec_output(True)).decode_coefficients(data)
    return planes


CASES = [(sub, q, opt, w, h) for sub in ("420", "422", "444", "gray") for (q, opt) in ((50, False), (75, True), (90, False), (100, False), (95, True))
         for (w, h) in ((1, 1), (13, 7), (33, 17), (99, 70))]


@pytest.mark.parametrize("sub,q,opt,w,h", CASES)
def test_model_equals_the_host_stage(sub, q, opt, w, h):
    data = _enc(len(CASES) + w * 7 + h + q, w, h, sub if sub != "gray" else "444", q, opt, gray=sub == "gray")
    want = _host(data)
    for S in (32, 96, 256):
        got, rounds = model(data, S)
        assert got is not None, rounds
        assert len(got) == len(want) and all(np.array_equal(a, b) for a, b in zip(got, want)), (S, rounds)


def test_some_files_need_more_than_one_round():
    rounds = []
    for k, sub in enumerate(("420", "422", "444")):
        data = _enc(500 + k, 99, 70, sub, 90)
        for S in (32, 64, 128):
            got, r = model(data, S)
            assert got is not None and all(np.array_equal(a, b) for a, b in zip(got, _host(data)))
            rounds.append(r)
    # round 0 decodes from guesses, round 1 from their exits; a third decode round means some entry changed twice
    assert max(rounds) >= 3, rounds


def _scan_body(data):
    sos = data.index(b"\xff\xda")
    return sos + 2 + int.from_bytes(data[sos + 2:sos + 4], "big")


def test_model_turns_down_what_the_host_route_must_take():
    base = _enc(600, 99, 70, "420", 90)
    body = _scan_body(base)
    assert model(base, 64)[0] is not None
    assert model(base[:-200], 64) == (None, "no EOI behind the scan")                       # truncated
    ones = bytearray(base)
    ones[body + 100:body + 108] = b"\xff\x00" * 4                                           # 32 one bits: no code holds them
    assert model(bytes(ones), 64)[0] is None
    stray = bytearray(base)
    stray[body + 50:body + 52] = b"\xff\xc4"
    assert model(bytes(stray), 64) == (None, "no EOI behind the scan")                      # stray marker
    rst = bytearray(base)
    rst[body + 50:body + 52] = b"\xff\xd2"
    assert model(bytes(rst), 64) == (None, "no EOI behind the scan")                        # RSTn without DRI
    short = base[:body + (len(base) - body) // 2] + b"\xff\xd9"
    if short[-3] == 0xFF:
        short = short[:-3] + short[-2:]
    assert model(short, 64) == (None, "fewer blocks than the frame holds")                 # data ends mid-scan
    # a bound below what the subsequences need: turned down
    assert model(base, 32, max_rounds=2) == (None, "not settled")
    # a flipped bit decodes to garbage or is turned down; what is taken equals the host stage
    for p in range(body + 10, len(base) - 20, 97):
        flip = bytearray(base)
        flip[p] ^= 0x10
        if flip[p] == 0xFF or flip[p - 1] == 0xFF:
            continue
        got, why = model(bytes(flip), 64)
        if got is not None:
            assert all(np.array_equal(a, b) for a, b in zip(got, _host(bytes(flip))))
