"""Sequential restatement of what cv2.imdecode(buf, IMREAD_COLOR) does to a baseline JPEG (OpenCV 4.13 with
libjpeg-turbo 3.1: ISLOW integer IDCT, fancy upsampling, table-driven YCbCr -> BGR), plus a model of the device
decoder's self-synchronising parallel Huffman decode (Weissenberger & Schmidt, ICPP 2018).

Everything here is integer arithmetic on numpy / Python ints; tests/test_oracle_jpeg.py pins it bit for bit against
cv2.imdecode.  The supported set is that of frcnn_jpeg_inspect (include/frcnn_b200.h)."""
import struct

import numpy as np

NATURAL = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                    7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38,
                    31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63], np.int64)
LUMA_SAMPLING = {(1, 1), (2, 1), (1, 2), (2, 2), (4, 1)}      # (h, v) of component 0; chroma must be 1x1


class Unsupported(Exception):
    pass


class Invalid(Exception):
    pass


def _exif_orientation(p):
    """Orientation tag of an Exif APP1 payload (after 'Exif\\0\\0'), 1 when absent; Unsupported when unreadable."""
    if len(p) < 8 or p[:2] not in (b"II", b"MM"):
        raise Unsupported("unreadable EXIF")
    e = "<" if p[:2] == b"II" else ">"
    off = struct.unpack(e + "I", p[4:8])[0]
    if off + 2 > len(p):
        raise Unsupported("unreadable EXIF")
    n = struct.unpack(e + "H", p[off:off + 2])[0]
    for i in range(n):
        q = off + 2 + 12 * i
        if q + 12 > len(p):
            raise Unsupported("unreadable EXIF")
        tag, typ, cnt = struct.unpack(e + "HHI", p[q:q + 8])
        if tag == 0x0112:
            return struct.unpack(e + "H", p[q + 8:q + 10])[0] if typ == 3 else 1
    return 1


def parse(data):
    """Header of a baseline file up to its scan -> dict; raises Unsupported / Invalid (rules of frcnn_jpeg_inspect)."""
    d = bytes(data)
    n = len(d)
    if n < 4 or d[0] != 0xFF or d[1] != 0xD8:
        raise Invalid("no SOI")
    pos, jfif, adobe, frame, dri = 2, False, None, None, 0
    qt, ht = {}, {}
    while True:
        if pos >= n or d[pos] != 0xFF:
            raise Invalid("marker expected")
        while pos < n and d[pos] == 0xFF:
            pos += 1
        if pos >= n:
            raise Invalid("truncated")
        m = d[pos]
        pos += 1
        if m in (0x01,) or 0xD0 <= m <= 0xD9:
            raise Invalid("unexpected marker %02x" % m)
        if pos + 2 > n:
            raise Invalid("truncated")
        ln = (d[pos] << 8) | d[pos + 1]
        if ln < 2 or pos + ln > n:
            raise Invalid("segment length")
        seg = d[pos + 2:pos + ln]
        pos += ln
        if m in (0xC0, 0xC1):
            if frame is not None or len(seg) < 6:
                raise Invalid("SOF")
            prec, h, w, nc = seg[0], (seg[1] << 8) | seg[2], (seg[3] << 8) | seg[4], seg[5]
            if prec != 8:
                raise Unsupported("precision %d" % prec)
            if len(seg) != 6 + 3 * nc:
                raise Invalid("SOF length")
            if nc not in (1, 3):
                raise Unsupported("%d components" % nc)
            if h == 0 or w == 0:
                raise Invalid("zero dimension")
            comps = []
            for c in range(nc):
                cid, hv, tq = seg[6 + 3 * c:9 + 3 * c]
                if not (1 <= hv >> 4 <= 4 and 1 <= hv & 15 <= 4) or tq > 3:
                    raise Invalid("SOF component")
                comps.append(dict(id=cid, h=hv >> 4, v=hv & 15, tq=tq))
            frame = dict(height=h, width=w, comps=comps)
        elif 0xC2 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC) or m in (0xC8, 0xCC):
            raise Unsupported("SOF%d / arithmetic" % (m - 0xC0))
        elif m == 0xC4:
            q = 0
            while q < len(seg):
                if q + 17 > len(seg):
                    raise Invalid("DHT")
                tc, th = seg[q] >> 4, seg[q] & 15
                if tc > 1 or th > 3:
                    raise Invalid("DHT class / id")
                counts = list(seg[q + 1:q + 17])
                tot = sum(counts)
                if tot > 256 or q + 17 + tot > len(seg):
                    raise Invalid("DHT")
                code = 0
                for ln in range(16):                       # canonical codes must fit their lengths
                    code += counts[ln]
                    if code > 1 << (ln + 1):
                        raise Invalid("DHT code lengths")
                    code <<= 1
                if tc == 0 and any(v > 15 for v in seg[q + 17:q + 17 + tot]):
                    raise Invalid("DC category above 15")
                ht[(tc, th)] = (counts, list(seg[q + 17:q + 17 + tot]))
                q += 17 + tot
        elif m == 0xDB:
            q = 0
            while q < len(seg):
                pq, tq = seg[q] >> 4, seg[q] & 15
                if pq > 1 or tq > 3 or q + 1 + 64 * (pq + 1) > len(seg):
                    raise Invalid("DQT")
                vals = seg[q + 1:q + 1 + 64 * (pq + 1)]
                zz = [vals[i] for i in range(64)] if pq == 0 else [(vals[2 * i] << 8) | vals[2 * i + 1] for i in range(64)]
                tab = np.zeros(64, np.int64)
                tab[NATURAL] = zz
                qt[tq] = tab
                q += 1 + 64 * (pq + 1)
        elif m == 0xDD:
            if len(seg) != 2:
                raise Invalid("DRI")
            dri = (seg[0] << 8) | seg[1]
        elif m == 0xDC:
            raise Unsupported("DNL")
        elif m == 0xE0:
            if len(seg) >= 14 and seg[:5] == b"JFIF\0":
                jfif = True
        elif m == 0xE1:
            if seg[:6] == b"Exif\0\0" and _exif_orientation(seg[6:]) not in (0, 1):
                raise Unsupported("EXIF orientation")
        elif m == 0xEE:
            if len(seg) >= 12 and seg[:5] == b"Adobe":
                adobe = seg[11]
        elif m == 0xDA:
            if frame is None:
                raise Invalid("SOS before SOF")
            if len(seg) < 1 or len(seg) != 4 + 2 * seg[0]:
                raise Invalid("SOS length")
            ns = seg[0]
            comps = frame["comps"]
            if ns != len(comps):
                raise Unsupported("multi-scan")
            for i in range(ns):
                cid, t = seg[1 + 2 * i], seg[2 + 2 * i]
                c = next((c for c in comps if c["id"] == cid), None)
                if c is None or comps.index(c) != i:
                    raise Invalid("scan component")
                c["td"], c["ta"] = t >> 4, t & 15
                if (0, c["td"]) not in ht or (1, c["ta"]) not in ht:
                    raise Invalid("undefined Huffman table")
                if c["tq"] not in qt:
                    raise Invalid("undefined quantisation table")
            ss, se, ahal = seg[1 + 2 * ns:4 + 2 * ns]
            if ss != 0 or se != 63 or ahal != 0:
                raise Unsupported("not sequential")
            if len(comps) == 3:
                rgb = (not jfif) and (adobe == 0 if adobe is not None else [c["id"] for c in comps] == [82, 71, 66])
                if rgb:
                    raise Unsupported("RGB / Adobe transform 0")
                if (comps[1]["h"], comps[1]["v"], comps[2]["h"], comps[2]["v"]) != (1, 1, 1, 1) or \
                        (comps[0]["h"], comps[0]["v"]) not in LUMA_SAMPLING:
                    raise Unsupported("sampling")
            frame.update(qt=qt, ht=ht, dri=dri, scan=pos)
            return frame


def geometry(f):
    """libjpeg's per-component geometry (jdinput.c initial_setup / per_scan_setup)."""
    comps, W, H = f["comps"], f["width"], f["height"]
    hm, vm = max(c["h"] for c in comps), max(c["v"] for c in comps)
    for c in comps:
        c["dw"] = -(-W * c["h"] // hm)
        c["dh"] = -(-H * c["v"] // vm)
        c["wb"] = -(-W * c["h"] // (hm * 8))
        c["hb"] = -(-H * c["v"] // (vm * 8))
    if len(comps) == 1:
        c = comps[0]
        mcux, mcuy, layout = c["wb"], c["hb"], [(0, 0, 0)]
        c["pw"], c["ph"] = c["wb"], c["hb"]               # plane extent in blocks
    else:
        mcux, mcuy = -(-W // (8 * hm)), -(-H // (8 * vm))
        layout = [(ci, y, x) for ci, c in enumerate(comps) for y in range(c["v"]) for x in range(c["h"])]
        for c in comps:
            c["pw"], c["ph"] = mcux * c["h"], mcuy * c["v"]
    return dict(hm=hm, vm=vm, mcux=mcux, mcuy=mcuy, layout=layout)


def segments(data, start):
    """Entropy-coded data from `start`: stuffed zeros dropped, split at RSTn -> list of interval byte strings."""
    d, out, cur, i, n = data, [], bytearray(), start, len(data)
    while i < n:
        b = d[i]
        if b != 0xFF:
            cur.append(b)
            i += 1
            continue
        j = i + 1
        while j < n and d[j] == 0xFF:
            j += 1
        if j >= n:
            break
        if d[j] == 0x00:
            cur.append(0xFF)
            i = j + 1
        elif 0xD0 <= d[j] <= 0xD7:
            out.append(bytes(cur))
            cur = bytearray()
            i = j + 1
        else:
            break
    out.append(bytes(cur))
    return out


class CorruptData(Exception):
    pass


def _lookup(counts, vals):
    """canonical Huffman code -> {(length, code): value}"""
    tab, code, k = {}, 0, 0
    for ln in range(1, 17):
        for _ in range(counts[ln - 1]):
            tab[(ln, code)] = vals[k]
            code += 1
            k += 1
        code <<= 1
    return tab


class _Bits:
    def __init__(self, data):
        self.v = int.from_bytes(data, "big") if data else 0
        self.n = 8 * len(data)

    def get(self, pos, k):
        """k bits at pos, zero-filled past the end (like libjpeg when it meets a marker)."""
        if k == 0:
            return 0
        if pos + k <= self.n:
            return (self.v >> (self.n - pos - k)) & ((1 << k) - 1)
        have = max(self.n - pos, 0)
        top = (self.v & ((1 << have) - 1)) if have else 0
        return top << (k - have)


def _extend(x, s):
    return x - (1 << s) + 1 if s and x < (1 << (s - 1)) else x


def _symbol(bits, pos, tab):
    code = 0
    for ln in range(1, 17):
        code = (code << 1) | bits.get(pos + ln - 1, 1)
        if (ln, code) in tab:
            return tab[(ln, code)], ln
    raise CorruptData("code not in table at bit %d" % pos)


class Decoder:
    """Huffman decoding of one image; a state is (bit position, block in MCU, coefficient index)."""

    def __init__(self, f, g):
        self.f, self.g = f, g
        comps = f["comps"]
        self.dc = [_lookup(*f["ht"][(0, c["td"])]) for c in comps]
        self.ac = [_lookup(*f["ht"][(1, c["ta"])]) for c in comps]
        self.blk_comp = [ci for ci, _, _ in g["layout"]]
        self.bpm = len(g["layout"])
        self.max_code_len = max(max((ln for ln, _ in t), default=0) for t in self.dc + self.ac)

    def run(self, bits, state, stop_bit, max_blocks=None, sink=None):
        """Decode symbols from `state` while the position is below `stop_bit` (and fewer than `max_blocks` blocks have
        ended).  A symbol that would reach past the stream's last bit is not decoded: the run stops before it.  Returns
        (state, blocks ended).  sink(block_number, k, value) receives every coefficient (k = 0: the DC difference).
        Raises CorruptData on a code missing from its table or a coefficient index past 63."""
        pos, blk, k = state
        nblk = 0
        while pos < stop_bit and (max_blocks is None or nblk < max_blocks):
            comp = self.blk_comp[blk]
            try:
                s, ln = _symbol(bits, pos, self.dc[comp] if k == 0 else self.ac[comp])
            except CorruptData:
                if bits.n - pos < 16:           # the 16-bit window reaches past the data: padding, not a code
                    break
                raise
            r, s = (0, s) if k == 0 else (s >> 4, s & 15)
            if k == 0 and s > 15:
                raise CorruptData("DC category %d" % s)
            if pos + ln + s > bits.n:
                break
            v = _extend(bits.get(pos + ln, s), s)
            if k == 0:
                if sink:
                    sink(nblk, 0, v)
                k = 1
            elif s:
                k += r
                if k > 63:
                    raise CorruptData("coefficient index past 63")
                if sink:
                    sink(nblk, k, v)
                k += 1
            elif r == 15:
                k += 16
                if k > 64:
                    raise CorruptData("coefficient index past 63")
            else:
                k = 64
            pos += ln + s
            if k >= 64:
                k, blk, nblk = 0, (blk + 1) % self.bpm, nblk + 1
        return (pos, blk, k), nblk


def decode_coefficients(data, f=None):
    """Sequential decode: quantised coefficients (blocks, 64) int64 in natural order, blocks in MCU order, DC absolute."""
    f = f or parse(data)
    g = geometry(f)
    dec = Decoder(f, g)
    ivs = segments(bytes(data), f["scan"])
    n_mcu = g["mcux"] * g["mcuy"]
    ri = f["dri"] or n_mcu
    n_iv = -(-n_mcu // ri)
    coef = np.zeros((n_mcu * dec.bpm, 64), np.int64)
    base = 0
    for iv in range(n_iv):
        if iv >= len(ivs):
            raise CorruptData("missing restart interval")
        bits = _Bits(ivs[iv])
        want = min(ri, n_mcu - iv * ri) * dec.bpm

        def sink(b, k, v, base=base):
            coef[base + b, NATURAL[k]] = v
        _, got = dec.run(bits, (0, 0, 0), bits.n, want, sink)
        if got != want:
            raise CorruptData("interval %d ended after %d of %d blocks" % (iv, got, want))
        base += want
    _dc_prefix(coef, dec, ri)
    return coef, f, g


def _dc_prefix(coef, dec, ri):
    """DC differences -> absolute DC per component, predictors reset at every restart interval."""
    per_iv = ri * dec.bpm
    pred = [0, 0, 0]
    for b in range(coef.shape[0]):
        if b % per_iv == 0:
            pred = [0, 0, 0]
        c = dec.blk_comp[b % dec.bpm]
        pred[c] += int(coef[b, 0])
        coef[b, 0] = np.int16(np.int64(pred[c]).astype(np.int16))


def sync_decode(data, sub_bits, f=None):
    """The device decoder's Huffman stage: every interval is cut into `sub_bits`-bit subsequences; each is decoded from
    a guessed state (its first bit, block 0, coefficient 0; exact for an interval's first), then subsequence j is
    re-decoded from the exit state of j-1 whenever that changed (from its own guess again when j-1's chain met corrupt
    data, so that a wrong guess's error never travels along the stream), until no exit state changes.  At that fixed point
    every exit state is the sequential one (induction from the interval starts).  An exclusive scan of the block
    counts places each subsequence's blocks, the DC sums per subsequence place the DC predictors, and a final pass
    writes the coefficients.  Returns the same array as decode_coefficients."""
    f = f or parse(data)
    g = geometry(f)
    dec = Decoder(f, g)
    ivs = segments(bytes(data), f["scan"])
    n_mcu = g["mcux"] * g["mcuy"]
    ri = f["dri"] or n_mcu
    n_iv = -(-n_mcu // ri)
    coef = np.zeros((n_mcu * dec.bpm, 64), np.int64)
    for iv in range(n_iv):
        bits = _Bits(ivs[iv])
        want = min(ri, n_mcu - iv * ri) * dec.bpm
        n_sub = max(-(-bits.n // sub_bits), 1)
        ends = [min((j + 1) * sub_bits, bits.n) for j in range(n_sub)]

        def d(entry, j):
            if entry is None:                     # the predecessor met corrupt data: start from this one's guess
                entry = (j * sub_bits, 0, 0)
            try:
                return dec.run(bits, entry, ends[j])
            except CorruptData:
                return None, 0                   # a chain that meets corrupt data (a wrong guess, or a bad file)
        res = [d((0, 0, 0) if j == 0 else (j * sub_bits, 0, 0), j) for j in range(n_sub)]
        changed = [True] * n_sub
        while any(changed):
            new, now = list(res), [False] * n_sub
            for j in range(1, n_sub):
                if changed[j - 1]:
                    new[j] = d(res[j - 1][0], j)
                    now[j] = new[j][0] != res[j][0]
            res, changed = new, now
        if any(r[0] is None for r in res):
            raise CorruptData("interval %d: corrupt entropy data" % iv)
        counts = [r[1] for r in res]
        if sum(counts) < want:
            raise CorruptData("interval %d: %d of %d blocks" % (iv, sum(counts), want))
        start = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(int)
        base = iv * ri * dec.bpm
        for j in range(n_sub):
            if start[j] >= want:
                break

            def sink(b, k, v, j=j):
                coef[base + start[j] + b, NATURAL[k]] = v
            dec.run(bits, (0, 0, 0) if j == 0 else res[j - 1][0], ends[j], None, sink)
    _dc_prefix(coef, dec, ri)
    return coef


# ---- sample reconstruction: jidctint.c, jdsample.c, jdcolor.c ----------------------------------------------------------
_C = dict(c0298=2446, c0390=3196, c0541=4433, c0765=6270, c0899=7373, c1175=9633, c1501=12299, c1847=15137,
          c1961=16069, c2053=16819, c2562=20995, c3072=25172)


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _idct_1d(v, pass1):
    """one 8-point pass of jpeg_idct_islow on the last axis (int64 arrays); pass1 descales by CONST_BITS-PASS1_BITS"""
    c = _C
    z2, z3 = v[..., 2], v[..., 6]
    z1 = (z2 + z3) * c["c0541"]
    tmp2 = z1 + z3 * -c["c1847"]
    tmp3 = z1 + z2 * c["c0765"]
    tmp0 = (v[..., 0] + v[..., 4]) << 13
    tmp1 = (v[..., 0] - v[..., 4]) << 13
    tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    t0, t1, t2, t3 = v[..., 7], v[..., 5], v[..., 3], v[..., 1]
    z1, z2, z3, z4 = t0 + t3, t1 + t2, t0 + t2, t1 + t3
    z5 = (z3 + z4) * c["c1175"]
    t0, t1, t2, t3 = t0 * c["c0298"], t1 * c["c2053"], t2 * c["c3072"], t3 * c["c1501"]
    z1, z2, z3, z4 = z1 * -c["c0899"], z2 * -c["c2562"], z3 * -c["c1961"], z4 * -c["c0390"]
    z3, z4 = z3 + z5, z4 + z5
    t0, t1, t2, t3 = t0 + z1 + z3, t1 + z2 + z4, t2 + z2 + z3, t3 + z1 + z4
    n = 11 if pass1 else 18
    out = [tmp10 + t3, tmp11 + t2, tmp12 + t1, tmp13 + t0, tmp13 - t0, tmp12 - t1, tmp11 - t2, tmp10 - t3]
    return np.stack([_descale(o, n) for o in out], axis=-1)


def _range_limit(x):
    """libjpeg's post-IDCT range_limit[x & 1023]"""
    s = ((x + 512) & 1023) - 512
    return np.clip(s + 128, 0, 255)


def idct_islow(blocks, qtab):
    """(n, 64) quantised coefficients (natural order) -> (n, 8, 8) samples, bit-exact jpeg_idct_islow."""
    x = (blocks.astype(np.int64) * qtab[None].astype(np.int64)).reshape(-1, 8, 8)
    x = x.astype(np.int16).astype(np.int64)
    # pass 1 on columns; an all-zero AC column gives dc << PASS1_BITS, which the general formula reproduces
    ws = _idct_1d(np.swapaxes(x, 1, 2), True)                    # [n, col, row]
    ws = np.swapaxes(ws, 1, 2)                                   # [n, row, col]
    out = _idct_1d(ws, False)
    return _range_limit(out).astype(np.uint8)


def planes(coef, f, g):
    """IDCT every block into per-component sample planes of (ph*8, pw*8)."""
    comps = f["comps"]
    bpm = len(g["layout"])
    out = [np.zeros((c["ph"] * 8, c["pw"] * 8), np.uint8) for c in comps]
    samples = [None] * len(comps)
    for ci, c in enumerate(comps):
        idx = [i for i, (cc, _, _) in enumerate(g["layout"]) if cc == ci]
        sel = np.concatenate([np.arange(i, coef.shape[0], bpm) for i in idx]) if bpm > 1 else np.arange(coef.shape[0])
        samples[ci] = idct_islow(coef[sel], f["qt"][c["tq"]])
        k = 0
        for i in idx:
            _, yy, xx = g["layout"][i]
            for m in range(g["mcux"] * g["mcuy"]):
                my, mx = divmod(m, g["mcux"])
                by, bx = (my * c["v"] + yy, mx * c["h"] + xx) if bpm > 1 else (my, mx)
                out[ci][by * 8:by * 8 + 8, bx * 8:bx * 8 + 8] = samples[ci][k]
                k += 1
    return out


def upsample(plane, c, g, W, H):
    """jdsample.c: full size, h2v1 / h2v2 fancy (replication when downsampled_width <= 2), h1v2 fancy, int_upsample."""
    hx, vx = g["hm"] // c["h"], g["vm"] // c["v"]
    dw, dh = c["dw"], c["dh"]
    p = plane.astype(np.int64)
    if (hx, vx) == (1, 1):
        return plane[:H, :W]
    if (hx, vx) == (4, 1) or (hx in (2,) and dw <= 2 and vx in (1, 2)):
        out = np.repeat(np.repeat(p, hx, axis=1), vx, axis=0)
        return out[:H, :W].astype(np.uint8)
    rows = np.arange(p.shape[0])
    if vx == 2:
        up = p[np.clip(rows - 1, 0, dh - 1)]
        dn = p[np.clip(rows + 1, 0, dh - 1)]
        cs = np.empty((2 * p.shape[0], p.shape[1]), np.int64)
        cs[0::2] = 3 * p + up
        cs[1::2] = 3 * p + dn
    else:
        cs = p
    if hx == 1:                                                      # h1v2
        bias = np.tile(np.array([1, 2])[:, None], (p.shape[0], 1))
        return ((cs + bias) >> 2)[:H, :W].astype(np.uint8)
    cols = np.arange(dw)
    left, right = cs[:, np.maximum(cols - 1, 0)], cs[:, np.minimum(cols + 1, dw - 1)]
    mid = cs[:, :dw]
    out = np.empty((cs.shape[0], 2 * dw), np.int64)
    if vx == 1:                                                      # h2v1
        out[:, 0::2] = (3 * mid + left + 1) >> 2
        out[:, 1::2] = (3 * mid + right + 2) >> 2
    else:                                                            # h2v2
        out[:, 0::2] = (3 * mid + left + 8) >> 4
        out[:, 1::2] = (3 * mid + right + 7) >> 4
    return out[:H, :W].astype(np.uint8)


def ycc_to_bgr(y, cb, cr):
    """jdcolor.c ycc_rgb_convert with its SCALEBITS-16 tables, written B, G, R."""
    x = np.arange(256, dtype=np.int64) - 128
    one_half = 1 << 15
    cr_r = (91881 * x + one_half) >> 16
    cb_b = (116130 * x + one_half) >> 16
    cr_g = -46802 * x
    cb_g = -22554 * x + one_half
    y = y.astype(np.int64)
    r = np.clip(y + cr_r[cr], 0, 255)
    g = np.clip(y + ((cb_g[cb] + cr_g[cr]) >> 16), 0, 255)
    b = np.clip(y + cb_b[cb], 0, 255)
    return np.stack([b, g, r], axis=-1).astype(np.uint8)


def decode(data):
    """cv2.imdecode(data, IMREAD_COLOR) for a supported baseline file: (H, W, 3) uint8 BGR."""
    coef, f, g = decode_coefficients(data)
    W, H = f["width"], f["height"]
    pl = planes(coef, f, g)
    ups = [upsample(p, c, g, W, H) for p, c in zip(pl, f["comps"])]
    if len(ups) == 1:
        return np.repeat(ups[0][:, :, None], 3, axis=2)
    return ycc_to_bgr(*ups)


def code_lengths(data):
    """Every Huffman code length the scan uses (for tests that need codes longer than the device's fast table)."""
    f = parse(data)
    g = geometry(f)
    dec = Decoder(f, g)
    used = set()
    orig = _symbol

    def spy(bits, pos, tab):
        v, ln = orig(bits, pos, tab)
        used.add(ln)
        return v, ln
    globals()["_symbol"] = spy
    try:
        decode_coefficients(data, f)
    finally:
        globals()["_symbol"] = orig
    return used
