"""The FLAC output format (``artspeech_b200/audio.py``, ``as_flac_encode``) restated in Python / numpy from its
definition, and a separately written FLAC reader.

``encode`` follows the docstring step by step: exact int64 autocorrelation, the fp64 Levinson recursion in the stated
order (Python floats are IEEE doubles and never fuse a multiply into an add), the precision-12 quantisation with error
feedback, every candidate's exact bit count, and the bit packing.  ``decode`` reads a stream the way RFC 9639 defines
it, checks the sync code, both CRCs, the STREAMINFO fields and the streamable-subset limits, and fails loudly on
anything it does not handle."""
from __future__ import annotations

import math

import numpy as np

BLOCK = 4096
MAX_LPC = 8
PRECISION = 12
MAX_PORDER = 8
MAX_RICE = 14
RATE_CODES = {8000: 0b0100, 16000: 0b0101, 22050: 0b0110, 24000: 0b0111, 32000: 0b1000, 44100: 0b1001,
              48000: 0b1010}
FIXED_COEFS = ((), (1,), (2, -1), (3, -3, 1), (4, -6, 4, -1))


def bound(n: int) -> int:
    """The largest file of ``n`` samples: ``42 + 2 n + 18 ceil(n / 4096)`` bytes."""
    return 42 + 2 * n + 18 * (-(-n // BLOCK))


# ---- CRCs --------------------------------------------------------------------------------------------------------
def _table(poly, width):
    top, mask = 1 << (width - 1), (1 << width) - 1
    out = []
    for b in range(256):
        c = b << (width - 8)
        for _ in range(8):
            c = ((c << 1) ^ poly) & mask if c & top else (c << 1) & mask
        out.append(c)
    return out


_T8, _T16 = _table(0x07, 8), _table(0x8005, 16)


def crc8(data) -> int:
    """CRC-8, polynomial 0x07, initial value 0, MSB first (CRC-8/SMBUS)."""
    c = 0
    for b in bytes(data):
        c = _T8[c ^ b]
    return c


def crc16(data) -> int:
    """CRC-16, polynomial 0x8005, initial value 0, MSB first (CRC-16/UMTS)."""
    c = 0
    t = _T16
    for b in bytes(data):
        c = ((c << 8) & 0xFFFF) ^ t[(c >> 8) ^ b]
    return c


# ---- bit writer --------------------------------------------------------------------------------------------------
class _Bits:
    """MSB-first bit string kept as a list of numpy 0/1 arrays."""

    def __init__(self):
        self.parts = []
        self.n = 0

    def put(self, value: int, nbits: int):
        if nbits:
            v = int(value) & ((1 << nbits) - 1)
            self.parts.append(np.array([(v >> (nbits - 1 - i)) & 1 for i in range(nbits)], dtype=np.uint8))
            self.n += nbits

    def put_array(self, values, nbits: int):
        """Each of ``values`` (int64) as an ``nbits``-bit two's complement field."""
        v = np.asarray(values, dtype=np.int64) & ((1 << nbits) - 1)
        sh = np.arange(nbits - 1, -1, -1, dtype=np.int64)
        self.parts.append(((v[:, None] >> sh[None, :]) & 1).astype(np.uint8).reshape(-1))
        self.n += nbits * v.size

    def put_rice(self, u, k: int):
        """Rice codes of the non-negative ``u`` with parameter ``k``: ``u >> k`` zeros, a one, the ``k`` low bits."""
        u = np.asarray(u, dtype=np.int64)
        q = u >> k
        ln = q + 1 + k
        start = np.concatenate([[0], np.cumsum(ln)[:-1]]) if u.size else np.zeros(0, np.int64)
        bits = np.zeros(int(ln.sum()), dtype=np.uint8)
        bits[start + q] = 1
        for j in range(k):
            bits[start + q + 1 + j] = (u >> (k - 1 - j)) & 1
        self.parts.append(bits)
        self.n += bits.size

    def tobytes(self) -> bytes:
        bits = np.concatenate(self.parts) if self.parts else np.zeros(0, np.uint8)
        return np.packbits(bits).tobytes()        # zero-padded to a byte boundary


# ---- the encoder -------------------------------------------------------------------------------------------------
def utf8_number(v: int) -> bytes:
    """FLAC's UTF-8-style coding of a frame number (``v < 2^31``)."""
    if v < 0x80:
        return bytes([v])
    for nb, lim in ((2, 0x800), (3, 0x10000), (4, 0x200000), (5, 0x4000000), (6, 0x80000000)):
        if v < lim:
            out = [0x80 | ((v >> (6 * i)) & 0x3F) for i in range(nb - 1)][::-1]
            lead = ((0xFF << (8 - nb)) & 0xFF) | (v >> (6 * (nb - 1)))
            return bytes([lead] + out)
    raise ValueError(f"frame number {v} does not fit")


def frame_header(f: int, bs: int, rate: int) -> bytes:
    code = 0b1100 if bs == BLOCK else 0b0111
    rc = RATE_CODES.get(rate, 0b1101)
    h = bytes([0xFF, 0xF8, (code << 4) | rc, 0b0000_100_0]) + utf8_number(f)
    if code == 0b0111:
        h += (bs - 1).to_bytes(2, "big")
    if rc == 0b1101:
        h += rate.to_bytes(2, "big")
    return h + bytes([crc8(h)])


def autocorrelation(x) -> list:
    """``R[l] = sum_{i=l}^{bs-1} x[i] x[i-l]``, l = 0..8, exact (Python integers)."""
    x = np.asarray(x, dtype=np.int64)
    return [int(np.dot(x[l:], x[:max(0, x.size - l)])) for l in range(MAX_LPC + 1)]


def levinson(R) -> list:
    """The predictor of every order the recursion reaches: ``[a_1 .. a_m]`` (fp64) for m = 1, 2, ..."""
    R = [float(v) for v in R]
    E = R[0]
    a = [0.0] * (MAX_LPC + 1)
    out = []
    for m in range(1, MAX_LPC + 1):
        if not E > 0.0:
            break
        acc = R[m]
        for j in range(1, m):
            acc = acc - a[j] * R[m - j]
        k = acc / E
        if not math.isfinite(k):
            break
        old = a[:]
        for j in range(1, m):
            a[j] = old[j] - k * old[m - j]
        a[m] = k
        E = E * (1.0 - k * k)
        out.append(a[1:m + 1])
    return out


def llround(v: float) -> int:
    """C's ``llround``: nearest integer, halves away from zero."""
    t = math.trunc(v)
    if abs(v - t) >= 0.5:
        t += 1 if v > 0 else -1
    return int(t)


def quantize(a):
    """``(q, shift)`` of the fp64 predictor ``a`` at precision 12, or None when it is not a candidate."""
    if not all(math.isfinite(v) for v in a):
        return None
    cmax = max(abs(v) for v in a)
    _, e = math.frexp(cmax)
    shift = PRECISION - 1 - e
    if shift < 0:
        return None
    shift = min(shift, 15)
    scale = float(2 ** shift)
    err, q = 0.0, []
    for v in a:
        err += v * scale
        qi = min(max(llround(err), -(1 << (PRECISION - 1))), (1 << (PRECISION - 1)) - 1)
        err -= qi
        q.append(qi)
    return q, shift


def residual(x, coefs, shift):
    """``r[i] = x[i] - ((sum_j c_j x[i-j]) >> shift)`` for i >= order, int64."""
    x = np.asarray(x, dtype=np.int64)
    p = len(coefs)
    acc = np.zeros(x.size - p, dtype=np.int64)
    for j, c in enumerate(coefs, start=1):
        acc += int(c) * x[p - j:x.size - j]
    return x[p:] - (acc >> shift)


def zigzag(r):
    return np.where(r >= 0, 2 * r, -2 * r - 1)


def rice_plan(u, bs: int, order: int):
    """``(bits, porder, ks)``: the cheapest partition order and per-partition parameters of the residual ``u`` (the
    ``bs - order`` zigzag values), ``bits`` counting the method and order fields."""
    v = np.zeros(bs, dtype=np.int64)                      # block positions; the warm-up samples count nothing
    v[order:] = u
    ks_all = np.arange(MAX_RICE + 1, dtype=np.int64)
    omax = 0
    while omax < MAX_PORDER and bs % (2 << omax) == 0:
        omax += 1
    # sum_{i in partition} (u_i >> k) at the finest order, then pairs of partitions summed up the tree
    level = {omax: (v[:, None] >> ks_all[None, :]).reshape(1 << omax, bs >> omax, -1).sum(1)}
    for o in range(omax - 1, -1, -1):
        level[o] = level[o + 1].reshape(1 << o, 2, -1).sum(1)
    best = None
    for o in range(omax + 1):
        if (bs >> o) <= order:
            continue
        m = bs >> o
        cnt = np.full(1 << o, m, dtype=np.int64)
        cnt[0] -= order
        cost = level[o] + cnt[:, None] * (1 + ks_all[None, :])
        ks = np.argmin(cost, axis=1)                       # the first minimum: ties go to the smaller k
        bits = 2 + 4 + int((4 + cost[np.arange(1 << o), ks]).sum())
        if best is None or bits < best[0]:
            best = (bits, o, [int(k) for k in ks])
    return best


def subframe_choice(x):
    """The chosen subframe of one block: ``(bits, kind, order, extra)`` with kind in constant / fixed / lpc /
    verbatim; ``extra`` is ``(q, shift, porder, ks)`` for the predictors."""
    x = np.asarray(x, dtype=np.int64)
    bs = x.size
    cands = []
    if np.all(x == x[0]):
        cands.append((8 + 16, "constant", 0, None))
    for order in range(5):
        if bs > order:
            r = residual(x, FIXED_COEFS[order], 0)
            if np.all(np.abs(r) < 2 ** 31):
                bits, po, ks = rice_plan(zigzag(r), bs, order)
                cands.append((8 + 16 * order + bits, "fixed", order, (FIXED_COEFS[order], 0, po, ks)))
    for a in levinson(autocorrelation(x)):
        p = len(a)
        qs = quantize(a)
        if bs <= p or qs is None:
            continue
        q, shift = qs
        r = residual(x, q, shift)
        if np.all(np.abs(r) < 2 ** 31):
            bits, po, ks = rice_plan(zigzag(r), bs, p)
            cands.append((8 + 16 * p + 4 + 5 + PRECISION * p + bits, "lpc", p, (q, shift, po, ks)))
    cands.append((8 + 16 * bs, "verbatim", 0, None))
    return min(cands, key=lambda c: c[0])              # min keeps the first of equal sizes


def encode_frame(x, f: int, rate: int):
    """``(frame bytes, kind, order)`` of block ``f``."""
    x = np.asarray(x, dtype=np.int64)
    bs = x.size
    bits, kind, order, extra = subframe_choice(x)
    w = _Bits()
    w.put(0, 1)
    if kind == "constant":
        w.put(0b000000, 6); w.put(0, 1); w.put(int(x[0]), 16)
    elif kind == "verbatim":
        w.put(0b000001, 6); w.put(0, 1); w.put_array(x, 16)
    else:
        coefs, shift, po, ks = extra
        w.put((0b001000 | order) if kind == "fixed" else (0b100000 | (order - 1)), 6)
        w.put(0, 1)
        w.put_array(x[:order], 16)
        if kind == "lpc":
            w.put(PRECISION - 1, 4); w.put(shift, 5); w.put_array(coefs, PRECISION)
        u = zigzag(residual(x, coefs, shift))
        w.put(0b00, 2); w.put(po, 4)
        m = bs >> po
        for p, k in enumerate(ks):
            w.put(k, 4)
            w.put_rice(u[max(0, p * m - order):(p + 1) * m - order], k)
    assert w.n == bits, (w.n, bits, kind, order)
    frame = frame_header(f, bs, rate) + w.tobytes()
    return frame + crc16(frame).to_bytes(2, "big"), kind, order


def streaminfo(n: int, rate: int, min_frame: int, max_frame: int) -> bytes:
    si = (BLOCK << 16 | BLOCK).to_bytes(4, "big") + min_frame.to_bytes(3, "big") + max_frame.to_bytes(3, "big")
    si += ((rate << 44) | (0 << 41) | (15 << 36) | n).to_bytes(8, "big") + bytes(16)
    return b"fLaC" + bytes([0x80, 0, 0, 34]) + si


def encode(x, rate: int, stats=None) -> bytes:
    """The FLAC file of the int16 samples ``x`` at ``rate`` Hz.  ``stats``: an optional dict counting the chosen
    ``(kind, order)`` subframes."""
    x = np.asarray(x, dtype=np.int64)
    n = x.size
    frames = []
    for f in range(-(-n // BLOCK)):
        fr, kind, order = encode_frame(x[f * BLOCK:(f + 1) * BLOCK], f, rate)
        frames.append(fr)
        if stats is not None:
            stats[(kind, order)] = stats.get((kind, order), 0) + 1
    sizes = [len(fr) for fr in frames]
    out = streaminfo(n, rate, min(sizes, default=0), max(sizes, default=0)) + b"".join(frames)
    assert len(out) <= bound(n)
    return out


# ---- the reader --------------------------------------------------------------------------------------------------
class DecodeError(ValueError):
    pass


class _Reader:
    def __init__(self, data: bytes):
        self.data = data
        self.bits = np.unpackbits(np.frombuffer(data, dtype=np.uint8)).astype(np.int64)
        nb = self.bits.size
        # next set bit at or after each position (for unary codes), and 32-bit windows (for fixed-width fields)
        idx = np.where(self.bits == 1, np.arange(nb), nb)
        self.next_one = np.minimum.accumulate(idx[::-1])[::-1] if nb else idx
        pad = np.concatenate([self.bits, np.zeros(32, np.int64)])
        win = np.zeros(nb, dtype=np.int64)
        for j in range(32):
            win = (win << 1) | pad[j:j + nb]
        self.win = win
        self.pos = 0

    def read(self, nbits: int) -> int:
        if nbits == 0:
            return 0
        if self.pos + nbits > self.bits.size:
            raise DecodeError("unexpected end of stream")
        v = 0
        p = self.pos
        while nbits > 32:
            v = (v << 32) | int(self.win[p]); p += 32; nbits -= 32
        v = (v << nbits) | (int(self.win[p]) >> (32 - nbits))
        self.pos = p + nbits
        return v

    def read_signed(self, nbits: int) -> int:
        v = self.read(nbits)
        return v - (1 << nbits) if v >> (nbits - 1) else v

    def align(self):
        self.pos = (self.pos + 7) // 8 * 8

    def read_rice(self, count: int, k: int) -> np.ndarray:
        out = np.empty(count, dtype=np.int64)
        nxt, win, nb = self.next_one, self.win, self.bits.size
        p = self.pos
        for i in range(count):
            if p >= nb:
                raise DecodeError("unexpected end of stream in a residual")
            o = int(nxt[p])
            if o >= nb or o + 1 + k > nb:
                raise DecodeError("unexpected end of stream in a residual")
            low = (int(win[o + 1]) >> (32 - k)) if k else 0
            out[i] = ((o - p) << k) | low
            p = o + 1 + k
        self.pos = p
        return out


def _read_utf8(r: _Reader) -> int:
    b0 = r.read(8)
    if b0 < 0x80:
        return b0
    n = 0
    while b0 & (0x80 >> n):
        n += 1
    if n < 2 or n > 6:
        raise DecodeError(f"bad coded number lead byte {b0:#x}")
    v = b0 & (0xFF >> (n + 1))
    for _ in range(n - 1):
        c = r.read(8)
        if c & 0xC0 != 0x80:
            raise DecodeError("bad coded number continuation byte")
        v = (v << 6) | (c & 0x3F)
    return v


def _unzig(u):
    return np.where(u & 1, -(u >> 1) - 1, u >> 1)


def _predict(warm, coefs, shift, res):
    """Samples from warm-up samples, predictor coefficients (for x[i-1], x[i-2], ...) and residuals."""
    p = len(coefs)
    x = np.zeros(p + res.size, dtype=np.int64)
    x[:p] = warm
    c = [int(v) for v in coefs]
    xs = x.tolist()
    rs = res.tolist()
    for i in range(p, len(xs)):
        s = 0
        for j in range(p):
            s += c[j] * xs[i - 1 - j]
        xs[i] = rs[i - p] + (s >> shift)
    return np.array(xs, dtype=np.int64)


def _subframe(r: _Reader, bs: int, info: dict):
    if r.read(1):
        raise DecodeError("subframe padding bit set")
    t = r.read(6)
    if r.read(1):
        raise DecodeError("wasted-bits flag: not produced by this encoder")
    if t == 0:
        info["kinds"].append(("constant", 0))
        return np.full(bs, r.read_signed(16), dtype=np.int64)
    if t == 1:
        info["kinds"].append(("verbatim", 0))
        return np.array([r.read_signed(16) for _ in range(bs)], dtype=np.int64)
    if 8 <= t <= 12:
        order = t - 8
        warm = [r.read_signed(16) for _ in range(order)]
        coefs, shift = [(), (1,), (2, -1), (3, -3, 1), (4, -6, 4, -1)][order], 0
        info["kinds"].append(("fixed", order))
    elif t >= 32:
        order = t - 31
        warm = [r.read_signed(16) for _ in range(order)]
        prec = r.read(4) + 1
        if prec == 16:
            raise DecodeError("invalid LPC precision")
        shift = r.read_signed(5)
        if shift < 0:
            raise DecodeError("negative LPC shift")
        coefs = [r.read_signed(prec) for _ in range(order)]
        info["kinds"].append(("lpc", order))
        if order > 12:
            raise DecodeError("LPC order above the streamable subset's 12")
    else:
        raise DecodeError(f"reserved subframe type {t}")
    method = r.read(2)
    if method != 0:
        raise DecodeError(f"residual coding method {method}: not produced by this encoder")
    po = r.read(4)
    if po > 8:
        raise DecodeError("partition order above the streamable subset's 8")
    if bs % (1 << po) or (bs >> po) < order:
        raise DecodeError("partition order does not fit the block")
    res = []
    for p in range(1 << po):
        k = r.read(4)
        if k == 15:
            raise DecodeError("escaped partition: not produced by this encoder")
        cnt = (bs >> po) - (order if p == 0 else 0)
        res.append(r.read_rice(cnt, k))
    res = _unzig(np.concatenate(res)) if res else np.zeros(0, np.int64)
    return _predict(warm, coefs, shift, res)


def decode(data: bytes, info: dict = None):
    """``(samples int16, sample_rate)`` of a FLAC file of one 16-bit channel.  ``info``: an optional dict that
    receives the STREAMINFO fields, the frame sizes and the subframe kinds."""
    info = {} if info is None else info
    info["kinds"], info["frame_sizes"] = [], []
    data = bytes(data)
    if data[:4] != b"fLaC":
        raise DecodeError("no fLaC marker")
    if data[4] != 0x80 or int.from_bytes(data[5:8], "big") != 34:
        raise DecodeError("expected one STREAMINFO block, flagged last, of 34 bytes")
    si = int.from_bytes(data[8:42], "big")
    f = lambda shift, bits: (si >> shift) & ((1 << bits) - 1)
    min_bs, max_bs = f(256, 16), f(240, 16)
    min_fr, max_fr = f(216, 24), f(192, 24)
    rate, chans, bps, total, md5 = f(172, 20), f(169, 3) + 1, f(164, 5) + 1, f(128, 36), f(0, 128)
    info.update(min_block=min_bs, max_block=max_bs, min_frame=min_fr, max_frame=max_fr, rate=rate,
                channels=chans, bits=bps, total=total, md5=md5)
    if chans != 1 or bps != 16:
        raise DecodeError(f"{chans} channels of {bps} bits: only mono 16-bit is read")
    if min_bs < 16 or max_bs < min_bs or max_bs > (4608 if rate <= 48000 else 16384):
        raise DecodeError(f"block sizes {min_bs}..{max_bs} outside the streamable subset")
    if rate == 0 or rate > 655350:
        raise DecodeError(f"sample rate {rate}")
    out, pos, fnum = [], 42, 0
    while pos < len(data):
        r = _Reader(data[pos:pos + 15 + 2 * max_bs + 4])
        if r.read(15) != 0b111111111111100 or r.read(1) != 0:
            raise DecodeError(f"frame {fnum}: bad sync code or blocking strategy")
        bcode, rcode = r.read(4), r.read(4)
        if r.read(4) != 0 or r.read(3) != 0b100 or r.read(1) != 0:
            raise DecodeError(f"frame {fnum}: not one 16-bit channel")
        num = _read_utf8(r)
        if num != fnum:
            raise DecodeError(f"frame number {num}, expected {fnum}")
        if bcode == 0b0110:
            bs = r.read(8) + 1
        elif bcode == 0b0111:
            bs = r.read(16) + 1
        elif bcode >= 0b1000:
            bs = 256 << (bcode - 8)
        elif bcode == 0b0001:
            bs = 192
        elif 2 <= bcode <= 5:
            bs = 576 << (bcode - 2)
        else:
            raise DecodeError(f"frame {fnum}: reserved block-size code")
        table = {0b0100: 8000, 0b0101: 16000, 0b0110: 22050, 0b0111: 24000, 0b1000: 32000, 0b1001: 44100,
                 0b1010: 48000, 0b1011: 96000, 0b0001: 88200, 0b0010: 176400, 0b0011: 192000}
        if rcode in table:
            fr_rate = table[rcode]
        elif rcode == 0b1100:
            fr_rate = r.read(8) * 1000
        elif rcode == 0b1101:
            fr_rate = r.read(16)
        elif rcode == 0b1110:
            fr_rate = r.read(16) * 10
        else:
            raise DecodeError(f"frame {fnum}: sample-rate code {rcode:#06b} (the subset needs it in the header)")
        if fr_rate != rate:
            raise DecodeError(f"frame {fnum}: rate {fr_rate} differs from STREAMINFO's {rate}")
        hlen = r.pos // 8
        if r.read(8) != crc8(data[pos:pos + hlen]):
            raise DecodeError(f"frame {fnum}: header CRC-8 mismatch")
        if bs > max_bs or (bs < min_bs and total - max_bs * fnum > bs):
            raise DecodeError(f"frame {fnum}: block size {bs} outside STREAMINFO's range")
        x = _subframe(r, bs, info)
        r.align()
        end = r.pos // 8
        if end + 2 > len(data) - pos or r.read(16) != crc16(data[pos:pos + end]):
            raise DecodeError(f"frame {fnum}: CRC-16 mismatch")
        if x.min(initial=0) < -32768 or x.max(initial=0) > 32767:
            raise DecodeError(f"frame {fnum}: samples outside 16 bits")
        info["frame_sizes"].append(end + 2)
        out.append(x)
        pos += end + 2
        fnum += 1
    sizes = info["frame_sizes"]
    if sizes and (min(sizes) != min_fr or max(sizes) != max_fr):
        raise DecodeError(f"frame sizes {min(sizes)}..{max(sizes)}, STREAMINFO says {min_fr}..{max_fr}")
    if not sizes and (min_fr or max_fr):
        raise DecodeError("frame sizes given for a stream without frames")
    x = np.concatenate(out) if out else np.zeros(0, np.int64)
    if x.size != total:
        raise DecodeError(f"{x.size} samples, STREAMINFO says {total}")
    return x.astype(np.int16), rate


def encode_model(x, lens, sample_rate):
    """Torch model of ``ops.flac_encode`` (CPU): ``(uint8 [B, bound(S)], int64 [B])``."""
    import torch
    B, S = x.shape
    out = torch.zeros(B, bound(S), dtype=torch.uint8)
    nbytes = torch.zeros(B, dtype=torch.int64)
    for b in range(B):
        n = S if lens is None else min(max(int(lens[b]), 0), S)
        f = encode(x[b, :n].numpy(), int(sample_rate))
        out[b, :len(f)] = torch.frombuffer(bytearray(f), dtype=torch.uint8)
        nbytes[b] = len(f)
    return out, nbytes
