"""GPU entropy decoding of progressive spec and libjpeg output (ZJ_USE_GPU_PROGRESSIVE, DESIGN.md section 5.6).

On the CPU: the ABI, and a pure-Python model of the four phases of zj_entropy.cu -- first scans decoded self-synchronising
(rounds, accept, write, DC prefix), DC refinements, AC refinement chains over non-zero masks, one status per image -- that must
give the host stage's progressive planes exactly and turn down what the GPU form turns down.  On the GPU: every result bit for
bit against the host route (the same options without the bit) and, where that matches Pillow, against Pillow."""
import ctypes as C
import io
import os
import subprocess
import sys

import numpy as np
import pytest
from PIL import Image, ImageOps

import jpeg_util
from test_spec_entropy_model import INVALID, UNZIGZAG, AddressError, Bits, Table, extend, huff
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, Decoder, DecodeErrors, ZuneJpegOptions, decode_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DC_FIRST, DC_REFINE, AC_FIRST, AC_REFINE = range(4)


def s16(x):
    return ((x + 0x8000) & 0xFFFF) - 0x8000


def prog_table(counts, vals, is_dc):
    """build_huffman after SOF2: the fast-AC table keeps only entries with a value"""
    t = Table(counts, vals, is_dc)
    t.ac = [f if f >> 10 else 0 for f in t.ac]
    return t


class Scan:
    pass


class TurnDown(Exception):
    pass


def walk(data, max_scans=64):
    """the host stage's progressive branch of gpu_entropy_prepare: the frame and its scans, or TurnDown(reason)"""
    p, dc, ac, f = 2, {}, {}, Scan()
    f.dri = 0

    def dht(seg):
        q = 0
        while q < len(seg):
            tc, th, counts = seg[q] >> 4, seg[q] & 15, list(seg[q + 1:q + 17])
            (ac if tc else dc)[th] = prog_table(counts, seg[q + 17:q + 17 + sum(counts)], not tc)
            q += 17 + sum(counts)

    while True:
        if p + 4 > len(data) or data[p] != 0xFF:
            raise TurnDown("header")
        m, ln = data[p + 1], int.from_bytes(data[p + 2:p + 4], "big")
        seg = data[p + 4:p + 2 + ln]
        if m == 0xC2:
            f.h, f.w, nc = int.from_bytes(seg[1:3], "big"), int.from_bytes(seg[3:5], "big"), seg[5]
            f.comps = [(seg[6 + 3 * i], seg[7 + 3 * i] >> 4, seg[7 + 3 * i] & 15) for i in range(nc)]
        elif m == 0xC4:
            dht(seg)
        elif m == 0xDD:
            f.dri = int.from_bytes(seg[0:2], "big")
        elif m == 0xDA:
            break
        p += 2 + ln
    if f.dri:
        raise TurnDown("dri")
    nc = len(f.comps)
    hm, vm = max(c[1] for c in f.comps), max(c[2] for c in f.comps)
    f.mcu_x, f.mcu_y = -(-f.w // (8 * hm)), -(-f.h // (8 * vm))
    ilv = hm != 1 or vm != 1
    if nc == 1 and ilv:
        raise TurnDown("gray with a down-sampled component")
    f.H, f.V = [c[1] for c in f.comps], [c[2] for c in f.comps]
    f.bw = [c[1] * f.mcu_x for c in f.comps]
    mw, mh = (f.mcu_x, f.mcu_y) if ilv else (-(-f.w // 8), -(-f.h // 8))
    if ilv and hm == 2:
        mh += mh & 1
    f.plane_len = [mw * 64 * c[1] * c[2] * mh for c in f.comps]
    scans, cov, dref, aref = [], [0] * nc, [False] * nc, [False] * nc
    while True:
        ln = int.from_bytes(data[p + 2:p + 4], "big")
        seg = data[p + 4:p + 2 + ln]
        ns = seg[0]
        sel = [(next(i for i, c in enumerate(f.comps) if c[0] == seg[1 + 2 * k]), seg[2 + 2 * k]) for k in range(ns)]
        sc = Scan()
        sc.ss, sc.se, ah, sc.al = seg[1 + 2 * ns], seg[2 + 2 * ns], seg[3 + 2 * ns] >> 4, seg[3 + 2 * ns] & 15
        dcs = ns > 1 or sc.ss == 0
        sc.kind = (DC_FIRST if ah == 0 else DC_REFINE) if dcs else (AC_FIRST if ah == 0 else AC_REFINE)
        if not scans and ah:
            raise TurnDown("first scan is a refinement")
        if ns == 1:
            if sc.ss == 0 and sc.se != 0:
                raise TurnDown("DC and AC merged")
            z = sel[0][0]
            sc.mw, bh = (-(-f.w // 8), -(-f.h // 8)) if (f.comps[z][0] == 1 or not ilv) else (f.mcu_x, f.mcu_y)
            sc.total, sc.slots = sc.mw * bh, [(z, 0, 0, 0)]
            sc.tables = [] if sc.kind == DC_REFINE else [dc[sel[0][1] >> 4 & 3] if dcs else ac[sel[0][1] & 15]]
            if not dcs and sc.ss > sc.se:
                raise TurnDown("band")
        else:
            if sc.se != 0:
                raise TurnDown("DC and AC merged")
            sc.slots = [(z, t, h, v) for t, (z, _) in enumerate(sel) for v in range(f.V[z]) for h in range(f.H[z])]
            sc.tables = [dc[s >> 4] for _, s in sel] if sc.kind == DC_FIRST else []
            sc.total = f.mcu_x * f.mcu_y * len(sc.slots)
        for z, _ in sel:
            band = 1 if dcs else ((1 << (sc.se + 1)) - 1) & ~((1 << sc.ss) - 1)
            if sc.kind in (DC_FIRST, AC_FIRST):
                if (dref if dcs else aref)[z] or cov[z] & band:
                    raise TurnDown("order")
                cov[z] |= band
            else:
                (dref if dcs else aref)[z] = True
        p += 2 + ln
        body, p, code = destuff(data, p)
        sc.bits, sc.nbits = Bits(body), len(body) * 8
        if sc.nbits == 0:
            raise TurnDown("empty scan")
        scans.append(sc)
        if len(scans) > max_scans:
            raise TurnDown("too many scans")
        while code == 0xC4:                       # DHT, then get_marker
            ln = int.from_bytes(data[p:p + 2], "big")
            dht(data[p + 2:p + ln])
            p, code = next_marker(data, p + ln)
        if code == 0xD9:
            return f, scans
        if code != 0xDA:
            raise TurnDown("marker %02X between scans" % code)
        p -= 2


def destuff(data, p):
    """destuff_scan: (bytes, position behind the marker, marker code)"""
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
            break
        nxt = data[p]
        p += 1
        if nxt == 0x00:
            out.append(0xFF)
            continue
        return bytes(out), p, nxt
    raise TurnDown("no marker behind a scan")


def next_marker(data, p):
    """get_marker: the next FF xx with xx not 00 / FF"""
    while p + 1 < len(data):
        if data[p] == 0xFF:
            q = p + 1
            while q < len(data) and data[q] == 0xFF:
                q += 1
            if q < len(data) and data[q] != 0:
                return q + 1, data[q]
            p = q + 1
        else:
            p += 1
    raise TurnDown("no marker")


def block(f, sc, g):
    """prog_block: (component, offset) or None when the host stage's address check fails"""
    if len(sc.slots) > 1:
        m, s = divmod(g, len(sc.slots))
        i, j = divmod(m, f.mcu_x)
        z, _, h, v = sc.slots[s]
        x, y = j * f.H[z] + h, i * f.V[z] + v
    else:
        z = sc.slots[0][0]
        y, x = divmod(g, sc.mw)
    at = 64 * (y * f.bw[z] + x)
    return (z, at) if at + 64 <= f.plane_len[z] else None


def first_decode(f, sc, state, end, write=None):
    """prog_decode: (exit or INVALID, blocks, start of the symbol that reached the total)"""
    pos, slot, coef = state
    bits, blocks, last, cur = sc.bits, 0, None, None
    if pos >= end:
        return state, 0, None
    if write:
        g0, planes, dcd = write
        if g0 >= sc.total:
            return state, 0, None
        cur = block(f, sc, g0)
        if cur is None:
            raise AddressError
    while pos < end:
        start, done = pos, 0
        if sc.kind == DC_FIRST:
            t = sc.tables[sc.slots[slot][1]]
            r = huff(bits, pos, t, t.lookup[bits.peek(pos, 9)])
            if r is None:
                return INVALID, blocks, None
            s, pos = r
            v = extend(bits.peek(pos, s), s) if s else 0
            pos += s
            if write:
                dcd[g0 + blocks] = v
            done = 1
        else:
            t = sc.tables[0]
            fa = t.ac[bits.peek(pos, 9)]
            if fa:
                coef += (fa >> 4) & 63
                if coef > sc.se:
                    return INVALID, blocks, None
                if write:
                    planes[cur[0]][cur[1] + UNZIGZAG[coef]] = s16((fa >> 10) << sc.al)
                pos += fa & 15
                coef += 1
            else:
                r = huff(bits, pos, t, t.lookup[bits.peek(pos, 9)])
                if r is None:
                    return INVALID, blocks, None
                s, pos = r
                rr, s = s >> 4, s & 15
                if s:
                    coef += rr
                    if coef > sc.se:
                        return INVALID, blocks, None
                    v = extend(bits.peek(pos, s), s)
                    pos += s
                    if write:
                        planes[cur[0]][cur[1] + UNZIGZAG[coef]] = s16(v << sc.al)
                    coef += 1
                elif rr != 15:
                    done = (1 << rr) + (bits.peek(pos, rr) if rr else 0)
                    pos += rr
                else:
                    coef += 16
            if not done and coef > sc.se:
                done = 1
        if pos > sc.nbits:
            return INVALID, blocks, None
        if done:
            blocks += done
            coef = 0 if sc.kind == DC_FIRST else sc.ss
            slot = (slot + 1) % len(sc.slots) if sc.kind == DC_FIRST else 0
            if write:
                if g0 + blocks >= sc.total:
                    last = start
                    break
                cur = block(f, sc, g0 + blocks)
                if cur is None:
                    raise AddressError
    return (pos, slot, coef), blocks, last


def first_scan(f, sc, S, max_rounds, planes, is_file_first):
    """phase 1 for one scan: rounds, accept, write, DC prefix; returns the rounds it took"""
    n = -(-sc.nbits // S)
    ends = [min(sc.nbits, (k + 1) * S) for k in range(n)]
    ends[-1] = sc.nbits
    c0 = 0 if sc.kind == DC_FIRST else sc.ss
    used, exits, counts = [None] * n, [None] * n, [0] * n
    for r in range(max_rounds or n + 2):
        prev, changed = list(exits), 0
        for k in range(n):
            e = (k * S, 0, c0) if (k == 0 or r == 0 or prev[k - 1] is INVALID) else prev[k - 1]
            if r > 0 and e == used[k]:
                continue
            used[k] = e
            exits[k], counts[k], _ = first_decode(f, sc, e, ends[k])
            changed += 1
        rounds = r + 1
        if r > 0 and changed == 0:
            break
    else:
        raise TurnDown("not settled")
    base = [0] * n
    for k in range(1, n):
        base[k] = base[k - 1] + counts[k - 1]
    err = next((k for k in range(n) if exits[k] is INVALID), None)
    reached = base[err] + counts[err] if err is not None else base[-1] + counts[-1]
    if reached < sc.total:
        raise TurnDown("fewer blocks than the scan holds")
    dcd = [0] * sc.total
    last = None
    try:
        for k in range(n):
            entry = (0, 0, c0) if k == 0 else exits[k - 1]
            if base[k] >= sc.total or entry is INVALID:
                continue
            _, _, lk = first_decode(f, sc, entry, ends[k], (base[k], planes, dcd))
            last = lk if lk is not None else last
    except AddressError:
        raise TurnDown("addressing")
    if is_file_first and last is not None:
        fetched = 32 if last == 0 else -(-(last + 33) // 32) * 32
        if fetched <= sc.nbits:
            raise TurnDown("marker not met by the first scan's reader")
    if sc.kind == DC_FIRST:
        pred = [0] * 3
        for g in range(sc.total):
            t = sc.slots[g % len(sc.slots)][1]
            pred[t] = (pred[t] + dcd[g]) & 0xFFFFFFFF
            z, at = block(f, sc, g)
            planes[z][at] = s16((pred[t] & 0xFFFF) << sc.al)
    return rounds


def refine_scan(f, sc, masks):
    """prog_refine_scan: decode_mcu_ac_refine against the non-zero masks; {offset: (corrected, placed, negative)} per block"""
    bits, pos, z = sc.bits, 0, sc.slots[0][0]
    t, eob, mask, rec = sc.tables[0], 0, masks[z], {}

    def corrections(ks, pos):
        return sum(1 << q for i, q in enumerate(ks) if bits.peek(pos + i, 1)), pos + len(ks)

    for g in range(sc.total):
        y, x = divmod(g, sc.mw)
        at = 64 * (y * f.bw[z] + x)
        if at + 64 > f.plane_len[z]:
            raise TurnDown("addressing")
        m, k, corr, placed, neg = mask[at // 64], sc.ss, 0, 0, 0
        if eob == 0:
            while True:
                r = huff(bits, pos, t, t.lookup[bits.peek(pos, 9)])
                if r is None:
                    raise TurnDown("invalid code")
                s, pos = r
                rr, s = s >> 4, s & 15
                if s == 0 and rr != 15:
                    eob = (1 << rr) + (bits.peek(pos, rr) if rr else 0)
                    pos += rr
                    break
                minus = False
                if s:
                    if s != 1:
                        raise TurnDown("refinement magnitude")
                    minus = not bits.peek(pos, 1)
                    pos += 1
                zeros = [q for q in range(k, sc.se + 1) if not (m >> q) & 1]
                if len(zeros) <= rr:
                    raise TurnDown("zero run past the band")
                pz = zeros[rr]
                c, pos = corrections([q for q in range(k, pz) if (m >> q) & 1], pos)
                corr |= c
                if pos > sc.nbits:
                    raise TurnDown("beyond the data")
                if s:
                    placed, neg, m = placed | 1 << pz, neg | minus << pz, m | 1 << pz
                k = pz + 1
                if k > sc.se:
                    break
            if pos > sc.nbits:
                raise TurnDown("beyond the data")
        if eob > 0:
            if m >> 1:
                c, pos = corrections([q for q in range(k, sc.se + 1) if (m >> q) & 1], pos)
                corr |= c
            if pos > sc.nbits:
                raise TurnDown("beyond the data")
            eob -= 1
        rec[at] = (corr, placed, neg)
        mask[at // 64] = m
    return rec


def apply(plane, al, rec):
    """prog_apply_kernel: corrections add 2^al away from zero where that bit is clear, placed coefficients become +-2^al"""
    p1 = 1 << al
    for at, (corr, placed, neg) in rec.items():
        for q in range(64):
            x = plane[at + UNZIGZAG[q]]
            if (corr >> q) & 1 and x & p1 == 0:
                plane[at + UNZIGZAG[q]] = s16(x + p1 if x >= 0 else x - p1)
            if (placed >> q) & 1:
                plane[at + UNZIGZAG[q]] = -p1 if (neg >> q) & 1 else p1


def model(data, S, max_rounds=None, max_scans=64):
    """phases 1-4 (status: any TurnDown); (planes, max rounds of a first scan) or (None, reason)"""
    try:
        f, scans = walk(data, max_scans)
        planes = [[0] * n for n in f.plane_len]
        rounds = 0
        for i, sc in enumerate(scans):                                           # phase 1
            if sc.kind in (DC_FIRST, AC_FIRST):
                rounds = max(rounds, first_scan(f, sc, S, max_rounds, planes, i == 0))
        for sc in scans:                                                         # phase 2
            if sc.kind == DC_REFINE:
                if sc.nbits < sc.total:
                    raise TurnDown("DC refinement shorter than its blocks")
                for g in range(sc.total):
                    if sc.bits.peek(g, 1):
                        b = block(f, sc, g)
                        if b is None:
                            raise TurnDown("addressing")
                        planes[b[0]][b[1]] = s16(planes[b[0]][b[1]] + (1 << sc.al))
        masks = [[sum(1 << k for k in range(64) if p[64 * b + UNZIGZAG[k]] != 0) for b in range(len(p) // 64)] for p in planes]
        for z in range(len(planes)):                                             # phase 3, one chain per component
            recs = [(sc.al, refine_scan(f, sc, masks)) for sc in scans if sc.kind == AC_REFINE and sc.slots[0][0] == z]
            for al, rec in recs:                                                 # ... then applied in scan order
                apply(planes[z], al, rec)
    except TurnDown as e:
        return None, str(e)
    return [np.array(p, np.int16) for p in planes], rounds


# ---------------------------------------------------------------------------------------------------- files
def _enc(seed, w, h, sub="420", q=90, optimize=False, gray=False, noise=12, **kw):
    im = jpeg_util.smooth_image(seed, w, h, gray, noise=noise)
    bio = io.BytesIO()
    args = dict(quality=q, optimize=optimize, progressive=True)
    args.update(kw)
    if not gray:
        args["subsampling"] = jpeg_util.SUBSAMPLING[sub]
    im.save(bio, "JPEG", **args)
    return bio.getvalue()


def _libjpeg(bit=False, cs=ColorSpace.RGB):
    o = ZuneJpegOptions().set_out_colorspace(cs).set_libjpeg_output(True).set_gpu_entropy(True)
    return o.set_gpu_progressive(True) if bit else o


def _host(data):
    _, planes = Decoder.new_with_options(ZuneJpegOptions().set_libjpeg_output(True)).decode_coefficients(data)
    return planes


def _same(got, want):
    return len(got) == len(want) and all(np.array_equal(np.asarray(a).ravel(), np.asarray(b).ravel()) for a, b in zip(got, want))


CASES = [(sub, q, opt, w, h) for sub in ("420", "422", "444", "gray") for (q, opt) in ((50, False), (75, True), (90, False), (100, False), (95, True))
         for (w, h) in ((1, 1), (13, 7), (33, 17), (99, 70))]


def _case_file(sub, q, opt, w, h):
    return _enc(len(CASES) + w * 7 + h + q, w, h, sub if sub != "gray" else "444", q, opt, gray=sub == "gray")


def _units(data):
    """(header, [scan units]): a unit is the DHT segments in front of one SOS, the SOS and its entropy-coded data"""
    p = data.index(b"\xff\xda")
    s, starts = 2, []   # the segments from SOI to the first SOS: the header ends before the DHT run in front of that SOS
    while s < p:
        starts.append(s)
        s += 2 + int.from_bytes(data[s + 2:s + 4], "big")
    head_end = p
    for st in reversed(starts):
        if data[st + 1] != 0xC4:
            break
        head_end = st
    head, rest, units, cur = data[:head_end], data[head_end:-2], [], 0
    while cur < len(rest):
        u = cur
        while rest[cur + 1] == 0xC4:
            cur += 2 + int.from_bytes(rest[cur + 2:cur + 4], "big")
        assert rest[cur + 1] == 0xDA
        cur += 2 + int.from_bytes(rest[cur + 2:cur + 4], "big")
        while cur < len(rest) and not (rest[cur] == 0xFF and rest[cur + 1] not in (0x00, 0xFF) and not 0xD0 <= rest[cur + 1] <= 0xD7):
            cur += 1
        units.append(rest[u:cur])
    return head, units


def _splice(data, order):
    head, units = _units(data)
    body = b"".join(units[k] for k in order)
    return head + body + b"\xff\xd9"


# ---------------------------------------------------------------------------------------------------- ABI (CPU)
def test_abi_value_and_options_size():
    assert _ffi.USE_GPU_PROGRESSIVE == 0x400
    assert C.sizeof(_ffi.ZjOptions) == 32
    header = open(os.path.join(ROOT, "include", "zune_jpeg_b200.h")).read()
    assert "ZJ_USE_GPU_PROGRESSIVE = 0x400" in header


def test_options_builder_needs_gpu_entropy():
    with pytest.raises(ValueError):
        ZuneJpegOptions().set_libjpeg_output(True).set_gpu_progressive(True)._raw()
    with pytest.raises(ValueError):
        ZuneJpegOptions().set_gpu_entropy(True).set_gpu_progressive(True)._raw()
    o = ZuneJpegOptions().set_libjpeg_output(True).set_scale_denom(2).set_exif_orientation(True).set_gpu_entropy(True).set_gpu_progressive(True)
    assert o.get_gpu_progressive() and o._raw().use_unsafe == _ffi.USE_LIBJPEG_OUTPUT | 1 << _ffi.USE_SCALE_SHIFT | 0x100 | 0x200 | 0x400
    assert ZuneJpegOptions().set_spec_output(True).set_gpu_entropy(True).set_gpu_progressive(True)._raw().use_unsafe == _ffi.USE_SPEC_OUTPUT | 0x600


@pytest.mark.parametrize("spec", [False, True])
def test_coefficients_ignore_the_bit(spec):
    data = _enc(3, 61, 45, "420", 85)
    o = ZuneJpegOptions().set_spec_output(True) if spec else ZuneJpegOptions().set_libjpeg_output(True)
    ia, pa = Decoder.new_with_options(o).decode_coefficients(data)
    ib, pb = Decoder.new_with_options(o.set_gpu_entropy(True).set_gpu_progressive(True)).decode_coefficients(data)
    assert (ia.width, ia.height, ia.flags) == (ib.width, ib.height, ib.flags) and _same(pa, pb)


# ---------------------------------------------------------------------------------------------------- model (CPU)
@pytest.mark.parametrize("sub,q,opt,w,h", CASES)
def test_model_equals_the_host_stage(sub, q, opt, w, h):
    data = _case_file(sub, q, opt, w, h)
    want = _host(data)
    for S in (32, 96, 256):
        got, rounds = model(data, S)
        assert got is not None, rounds
        assert _same(got, want), (S, rounds)


def test_every_scan_carries_its_tables_and_some_files_need_more_than_one_round():
    data = _enc(500, 99, 70, "420", 90)
    head, units = _units(data)
    assert len(units) == 10 and all(b"\xff\xc4" in u for k, u in enumerate(units) if k != 6)   # DHT before each scan with codes
    rounds = []
    for k, sub in enumerate(("420", "422", "444")):
        data = _enc(500 + k, 99, 70, sub, 90)
        for S in (32, 64, 128):
            got, r = model(data, S)
            assert got is not None and _same(got, _host(data))
            rounds.append(r)
    assert max(rounds) >= 3, rounds


# libjpeg's simple progression for YCbCr: 0 DC first, 1 Y AC 1-5, 2 Cr AC, 3 Cb AC, 4 Y AC 6-63, 5 Y AC refine, 6 DC refine,
# 7 Cr AC refine, 8 Cb AC refine, 9 Y AC refine
SPLICED = [[0, 6, 1, 2, 3, 4, 5, 7, 8, 9],      # DC refinement before the AC first scans
           [0, 1, 2, 3, 4, 7, 8, 5, 6, 9],      # chroma refinements before the luma ones
           [0, 2, 3, 7, 8, 1, 4, 5, 9, 6]]      # a component's whole AC script at once, the DC refinement last


@pytest.mark.parametrize("order", SPLICED)
def test_model_equals_the_host_on_other_scan_orders(order):
    for k, sub in enumerate(("420", "444")):
        data = _splice(_enc(700 + k, 99, 70, sub, 90), order)
        got, why = model(data, 64)
        assert got is not None, why
        assert _same(got, _host(data))


def test_model_turns_down_what_the_host_route_must_take():
    base = _enc(600, 99, 70, "420", 90)
    assert model(base, 64)[0] is not None
    assert model(_splice(base, [0, 1, 2, 3, 5, 4, 6, 7, 8, 9]), 64) == (None, "order")        # AC first after a refinement
    head, units = _units(base)
    dri = head + b"\xff\xdd\x00\x04\x00\x05" + b"".join(units) + b"\xff\xd9"
    assert model(dri, 64) == (None, "dri")
    for seg in (b"\xff\xfe\x00\x04hi", b"\xff\xe1\x00\x04hi"):                              # COM / APP1 between scans
        assert model(head + units[0] + seg + b"".join(units[1:]) + b"\xff\xd9", 64)[1] == "marker %02X between scans" % seg[1]
    assert model(base[:-200], 64)[0] is None                                                 # truncated
    sos = base.index(b"\xff\xda")
    body = sos + 2 + int.from_bytes(base[sos + 2:sos + 4], "big")
    ones = bytearray(base)
    ones[body + 20:body + 28] = b"\xff\x00" * 4                                              # 32 one bits in the DC first scan
    assert model(bytes(ones), 64)[0] is None
    cut = head + b"".join(units[:9]) + units[9][:len(units[9]) // 2] + b"\xff\xd9"           # data ends mid-scan
    got, why = model(cut, 64)
    assert got is None, why
    assert model(base, 64, max_scans=5) == (None, "too many scans")
    assert model(base, 32, max_rounds=2) == (None, "not settled")
    # flipped bits: what is taken equals the host stage
    for p in range(body + 10, len(base) - 20, 211):
        flip = bytearray(base)
        flip[p] ^= 0x10
        if flip[p] == 0xFF or flip[p - 1] == 0xFF or base[p] == 0xFF:
            continue
        got, why = model(bytes(flip), 64)
        if got is not None:
            assert _same(got, _host(bytes(flip)))


# ---------------------------------------------------------------------------------------------------- GPU
def _pillow(data, gray=False):
    return np.asarray(Image.open(io.BytesIO(data)).convert("L" if gray else "RGB"))


def _both(files, opts_bit, opts_plain, **kw):
    s1, s0 = {}, {}
    got = decode_batch(files, opts_bit, threads=4, gpu_entropy=True, stats=s1, **kw)
    want = decode_batch(files, opts_plain, threads=4, gpu_entropy=True, stats=s0, **kw)
    return got, want, s1["gpu_entropy"], s0["gpu_entropy"]


def _corpus():
    return [_case_file(*c) for c in CASES]


@pytest.mark.gpu
def test_corpus_equals_the_host_route_and_pillow():
    files = _corpus() + [_splice(_enc(700, 99, 70, "420", 90), o) for o in SPLICED]
    got, want, n1, n0 = _both(files, _libjpeg(True), _libjpeg(False))
    assert n0 == 0 and n1 == len(files)
    assert [g == w for g, w in zip(got, want)] == [True] * len(files)
    assert [g == _pillow(d).tobytes() for g, d in zip(got, files)] == [True] * len(files)
    spec = ZuneJpegOptions().set_spec_output(True).set_gpu_entropy(True)
    got, want, n1, _ = _both(files, spec.set_gpu_progressive(True), spec)
    assert n1 == len(files) and got == want


@pytest.mark.gpu
def test_scaled_oriented_and_large():
    files = [_enc(7, 8192, 8192, "420", 90, noise=4), _enc(8, 1000, 700, "420", 95, optimize=True)]
    got, want, n1, _ = _both(files, _libjpeg(True), _libjpeg(False))
    assert n1 == 2 and got == want
    for d in (2, 4, 8):
        o = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True).set_scale_denom(d).set_gpu_entropy(True)
        got, want, n1, _ = _both(files[1:], o.set_gpu_progressive(True), o)
        assert n1 == 1 and got == want
    im = jpeg_util.smooth_image(9, 203, 101)
    ex = im.getexif()
    ex[0x0112] = 6
    bio = io.BytesIO()
    im.save(bio, "JPEG", quality=90, exif=ex.tobytes(), progressive=True)
    data = bio.getvalue()
    o = ZuneJpegOptions().set_libjpeg_output(True).set_exif_orientation(True).set_gpu_entropy(True)
    got, want, n1, _ = _both([data], o.set_gpu_progressive(True), o)
    assert n1 == 1 and got == want
    assert got[0] == np.asarray(ImageOps.exif_transpose(Image.open(io.BytesIO(data))).convert("RGB")).tobytes()


def _damaged_progressive():
    base = _enc(20, 200, 150, "420", 90)
    head, units = _units(base)
    sos = base.index(b"\xff\xda")
    body = sos + 2 + int.from_bytes(base[sos + 2:sos + 4], "big")
    ones = bytearray(base)
    ones[body + 20:body + 28] = b"\xff\x00" * 4
    return [base[:len(base) - 700],                                                        # truncated, no EOI
            bytes(ones),                                                                   # a code no table holds
            head + b"".join(units[:9]) + units[9][:len(units[9]) // 2] + b"\xff\xd9",      # data ends mid-scan
            head + units[0] + b"\xff\xfe\x00\x04hi" + b"".join(units[1:]) + b"\xff\xd9",    # COM between scans
            _splice(base, [0, 1, 2, 3, 5, 4, 6, 7, 8, 9]),                                  # AC first after a refinement
            _enc(21, 200, 150, "420", 90, restart_marker_rows=1)]                          # DRI


@pytest.mark.gpu
def test_mixed_and_damaged_files_give_the_host_results():
    base = [_enc(30, 120, 90, "420", 90, progressive=False), _enc(31, 120, 90, "420", 90, progressive=False, restart_marker_rows=1)]
    prog = [_enc(32, 120, 90, "420", 90), _enc(33, 97, 61, "444", 80, optimize=True), _enc(34, 64, 40, gray=True)]
    cmyk = Image.fromarray(np.random.default_rng(1).integers(0, 255, (40, 48, 4), np.uint8), "CMYK")
    bio = io.BytesIO()
    cmyk.save(bio, "JPEG", quality=90, progressive=True)
    other = [bio.getvalue(), b"\xff\xd8\xff\xc2\x00\x05"]
    damaged = _damaged_progressive()
    files = base + prog + other + damaged
    got, want, n1, n0 = _both(files, _libjpeg(True), _libjpeg(False))
    assert n0 == 2 and n1 == 5
    for d in damaged:
        s = {}
        decode_batch([d], _libjpeg(True), threads=4, gpu_entropy=True, stats=s)
        assert s["gpu_entropy"] == 0
    for g, w in zip(got, want):
        if isinstance(w, DecodeErrors):
            assert isinstance(g, DecodeErrors) and str(g) == str(w) and g.args == w.args
        else:
            assert g == w


@pytest.mark.gpu
def test_device_out_and_resized_equal_the_host_route():
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import decode_batch_resized
    files = [_enc(40, 640, 362, "420", 90), _enc(41, 333, 250, "422", 95, optimize=True), _enc(42, 500, 301, "444", 85)]
    pil = [_pillow(d) for d in files]
    for desc in (None, gpu.OutputDesc("CHW", "f16", False, 0, (0.0,) * 4, (1.0,) * 4)):
        res = []
        for bit in (True, False):
            es = 1 if desc is None else 2
            outs = [gpu.DeviceBuffer(p.size * es) for p in pil]
            stats = {}
            r = decode_batch(files, _libjpeg(bit), threads=4, device_out=[(o.ptr, o.nbytes) for o in outs], desc=desc, stats=stats)
            assert r == [o.nbytes for o in outs]
            assert stats["gpu_entropy"] == (len(files) if bit else 0)
            res.append([o.download().tobytes() for o in outs])
        assert res[0] == res[1]
        if desc is None:
            assert res[0] == [p.tobytes() for p in pil]
    rz = gpu.Resize((224, 224), "pil_bicubic", short_side=256)
    outs = []
    for bit in (True, False):
        stats = {}
        out, errs = decode_batch_resized(files, rz, None, None, _libjpeg(bit), threads=4, stats=stats)
        assert errs == [None] * len(files) and stats["gpu_entropy"] == (len(files) if bit else 0)
        outs.append(out.download())
    assert outs[0].tobytes() == outs[1].tobytes()
    from torchvision.transforms import InterpolationMode, v2
    tv = v2.Compose([v2.Resize(256, interpolation=InterpolationMode.BICUBIC), v2.CenterCrop(224)])
    for k, p in enumerate(pil):
        assert outs[0][k].tobytes() == np.asarray(tv(Image.fromarray(p))).tobytes(), k


@pytest.mark.gpu
def test_small_budget_covers_several_sub_batches():
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "from test_progressive_entropy_model import _corpus, _enc, _libjpeg\n"
            "from zune_jpeg_b200.decoder import decode_batch\n"
            "files = [_enc(60 + k, 1200, 900, '420', 90) for k in range(24)] + _corpus()[:16]\n"
            "s = {}\n"
            "a = decode_batch(files, _libjpeg(True), threads=4, gpu_entropy=True, stats=s)\n"
            "b = decode_batch(files, _libjpeg(False), threads=4)\n"
            "assert a == b and s['gpu_entropy'] == len(files), s\n"
            "print('ok')\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, ZJ_GPU_ENTROPY_BUDGET_MB="64")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]
