"""FLAC (RFC 9639) test encoder and reference decoder, pure Python / numpy.  Test infrastructure only: the product never
imports it.

``encode`` writes a stream whose every coding decision can be forced per frame (``FramePlan`` / ``SubPlan``): blocking
strategy, block-size / sample-rate / sample-size header codes, channel assignment, subframe type (CONSTANT, VERBATIM,
FIXED 0-4, LPC 1-32 with coefficient precision 1-15), wasted bits, residual coding method, partition order and escaped
partitions (width 0 included).  ``decode`` is a separate, sequential reader of the same format that checks every CRC and
reserved value; it shares no code with the encoder beyond the two CRC functions, which the tests pin to their published
check values.
"""
import hashlib
import struct
from dataclasses import dataclass, field

import numpy

# ----------------------------------------------------------------------------------------------------------- CRCs

def crc8(data, crc=0):
    """CRC-8, polynomial x^8 + x^2 + x + 1 (0x07), initial value 0, not reflected (RFC 9639 section 9.1.8)."""
    for b in data:
        crc ^= b
        for _ in range(8):
            crc = ((crc << 1) ^ 0x07) & 0xFF if crc & 0x80 else (crc << 1) & 0xFF
    return crc


def crc16(data, crc=0):
    """CRC-16, polynomial x^16 + x^15 + x^2 + 1 (0x8005), initial value 0, not reflected (section 9.3)."""
    for b in data:
        crc ^= b << 8
        for _ in range(8):
            crc = ((crc << 1) ^ 0x8005) & 0xFFFF if crc & 0x8000 else (crc << 1) & 0xFFFF
    return crc


# -------------------------------------------------------------------------------------------------------- encoder

COMMON_BLOCK_SIZES = {192: 1, 576: 2, 1152: 3, 2304: 4, 4608: 5, 256: 8, 512: 9, 1024: 10, 2048: 11, 4096: 12, 8192: 13,
                      16384: 14, 32768: 15}
TABLE_RATES = {88200: 1, 176400: 2, 192000: 3, 8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10, 96000: 11}
SAMPLE_SIZE_CODES = {8: 1, 12: 2, 16: 4, 20: 5, 24: 6}
ASSIGN = {"independent": None, "left_side": 8, "side_right": 9, "mid_side": 10}


@dataclass
class SubPlan:
    kind: str = "auto"           # auto | constant | verbatim | fixed | lpc ("auto": constant when the block is, else lpc)
    order: int = 2               # FIXED 0-4, LPC 1-32
    precision: int = 12          # LPC coefficient precision 1-15
    method: int = 0              # residual coding method 0 (4-bit parameters) or 1 (5-bit)
    porder: int = 0              # partition order 0-15 (lowered until the block allows it)
    escape: tuple = ()           # partitions written escaped (raw, width may be 0)
    wasted: bool = True          # use wasted bits when every sample has trailing zeros


@dataclass
class FramePlan:
    assign: str = "independent"
    bs_code: str = "auto"        # auto (common code when there is one) | 8 | 16 (explicit size)
    rate_code: str = "streaminfo"  # streaminfo | table | khz | hz | 10hz
    size_code: str = "streaminfo"  # streaminfo | explicit
    subs: list = field(default_factory=list)   # SubPlan per channel (default SubPlan() when missing)


class BitWriter:
    def __init__(self):
        self.parts = []
        self.n = 0

    def put(self, v, n):
        if n:
            self.parts.append(format(v & ((1 << n) - 1), "0%db" % n))
            self.n += n

    def unary(self, q):
        self.parts.append("0" * q + "1")
        self.n += q + 1

    def pad(self):
        self.put(0, (-self.n) % 8)

    def bytes(self):
        assert self.n % 8 == 0
        s = "".join(self.parts)
        return int(s, 2).to_bytes(len(s) // 8, "big") if s else b""


def utf8_number(v):
    if v < 0x80:
        return bytes([v])
    for n in range(2, 8):
        if v < 1 << (5 * n + 1):
            break
    out = [0x80 | ((v >> (6 * i)) & 0x3F) for i in range(n - 2, -1, -1)]
    first = ((0xFF << (8 - n)) & 0xFF) | (v >> (6 * (n - 1)))
    return bytes([first] + out)


def _signed_width(x):
    """bits of the narrowest two's complement field holding every value of x (0 when all are zero)"""
    if not numpy.any(x):
        return 0
    lo, hi = int(x.min()), int(x.max())
    w = 1
    while not (-(1 << (w - 1)) <= lo and hi < (1 << (w - 1))):
        w += 1
    return w


def _residual(w, res, bs, order, sp):
    method = sp.method
    porder = sp.porder
    while porder > 0 and (bs % (1 << porder) or (bs >> porder) < order):
        porder -= 1
    w.put(method, 2)
    w.put(porder, 4)
    esc = 31 if method else 15
    psize = bs >> porder
    u_all = numpy.where(res >= 0, res.astype(numpy.int64) * 2, -res.astype(numpy.int64) * 2 - 1)
    start = 0
    for p in range(1 << porder):
        n = psize - (order if p == 0 else 0)
        r, u = res[start:start + n], u_all[start:start + n]
        start += n
        if p in sp.escape:
            width = _signed_width(r)
            w.put(esc, 4 + method)
            w.put(width, 5)
            for v in r.tolist():
                w.put(v, width)
            continue
        best = min(range(esc), key=lambda k: n * (k + 1) + int((u >> k).sum()))
        w.put(best, 4 + method)
        for v in u.tolist():
            w.unary(v >> best)
            w.put(v, best)


def _lpc_coefs(x, order, precision):
    """least-squares predictor of x, quantised to `precision` bits with a non-negative shift"""
    n = x.shape[0]
    A = numpy.stack([x[order - j - 1:n - j - 1] for j in range(order)], axis=1).astype(numpy.float64)
    c = numpy.linalg.lstsq(A, x[order:].astype(numpy.float64), rcond=None)[0] if n > order else numpy.zeros(order)
    cmax = float(numpy.abs(c).max()) if order else 0.0
    shift = 15
    lim = (1 << (precision - 1)) - 1
    while shift > 0 and cmax * (1 << shift) > lim:
        shift -= 1
    q = numpy.clip(numpy.round(c * (1 << shift)), -lim - 1, lim).astype(numpy.int64)
    return q, shift


def predict(x, coefs, shift):
    """prediction of x[order:] with coefs[j] applied to the sample j + 1 back (exact, int64)"""
    order = len(coefs)
    n = x.shape[0]
    acc = numpy.zeros(n - order, dtype=numpy.int64)
    for j, c in enumerate(coefs):
        acc += int(c) * x[order - j - 1:n - j - 1].astype(numpy.int64)
    return acc >> shift


FIXED_COEFS = [[], [1], [2, -1], [3, -3, 1], [4, -6, 4, -1]]


def _subframe(w, x, sbps, sp):
    x = x.astype(numpy.int64)
    bs = x.shape[0]
    kind = sp.kind
    if kind == "auto":
        kind = "constant" if numpy.all(x == x[0]) else "lpc"
    if kind == "constant" and not numpy.all(x == x[0]):
        kind = "verbatim"
    wasted = 0
    if sp.wasted and numpy.any(x) and kind != "constant":
        while wasted < sbps - 1 and not numpy.any(x & ((1 << (wasted + 1)) - 1)):
            wasted += 1
    x = x >> wasted
    sbps -= wasted
    order = min(sp.order, bs) if kind in ("fixed", "lpc") else 0
    if kind == "lpc" and order == 0:
        kind = "verbatim"
    code = {"constant": 0, "verbatim": 1}.get(kind, 8 + order if kind == "fixed" else 31 + order)
    w.put(0, 1)
    w.put(code, 6)
    if wasted:
        w.put(1, 1)
        w.unary(wasted - 1)
    else:
        w.put(0, 1)
    if kind == "constant":
        w.put(int(x[0]), sbps)
        return
    if kind == "verbatim":
        for v in x.tolist():
            w.put(v, sbps)
        return
    for v in x[:order].tolist():
        w.put(v, sbps)
    if kind == "fixed":
        coefs, shift = FIXED_COEFS[order], 0
    else:
        coefs, shift = _lpc_coefs(x, order, sp.precision)
        w.put(sp.precision - 1, 4)
        w.put(shift, 5)
        for c in coefs.tolist():
            w.put(c, sp.precision)
    res = x[order:] - predict(x, coefs, shift)
    if numpy.abs(res).max(initial=0) >= 1 << 30:
        raise OverflowError("residual does not fit 32 bits")
    _residual(w, res, bs, order, sp)


def _subframe_safe(w, x, sbps, sp):
    """an ill-conditioned least-squares fit can give a residual outside 32 bits: such a block falls back to FIXED"""
    trial = BitWriter()
    try:
        _subframe(trial, x, sbps, sp)
    except OverflowError:
        trial = BitWriter()
        _subframe(trial, x, sbps, SubPlan(kind="fixed", order=min(sp.order, 2), method=sp.method, porder=sp.porder))
    w.parts += trial.parts
    w.n += trial.n


def _frame(pcm, first, index, rate, bps, variable, plan):
    bs, nch = pcm.shape
    hdr = bytearray([0xFF, 0xF8 | int(variable)])
    tail = b""
    if plan.bs_code == "auto" and bs in COMMON_BLOCK_SIZES:
        bcode = COMMON_BLOCK_SIZES[bs]
    elif plan.bs_code == "16" or bs > 256:
        bcode, tail = 7, struct.pack(">H", bs - 1)
    else:
        bcode, tail = 6, bytes([bs - 1])
    rc, rtail = 0, b""
    if plan.rate_code == "table" and rate in TABLE_RATES:
        rc = TABLE_RATES[rate]
    elif plan.rate_code == "khz" and rate % 1000 == 0 and rate // 1000 < 256:
        rc, rtail = 12, bytes([rate // 1000])
    elif plan.rate_code == "hz" and rate < 65536:
        rc, rtail = 13, struct.pack(">H", rate)
    elif plan.rate_code == "10hz" and rate % 10 == 0 and rate // 10 < 65536:
        rc, rtail = 14, struct.pack(">H", rate // 10)
    assign = ASSIGN[plan.assign] if nch == 2 else None
    hdr.append((bcode << 4) | rc)
    ss = SAMPLE_SIZE_CODES.get(bps, 0) if plan.size_code == "explicit" else 0
    hdr.append(((nch - 1 if assign is None else assign) << 4) | (ss << 1))
    hdr += utf8_number(first if variable else index) + tail + rtail
    hdr.append(crc8(hdr))
    left, right = (pcm[:, 0].astype(numpy.int64), pcm[:, 1].astype(numpy.int64)) if nch == 2 else (None, None)
    if assign == 8:
        chans, extra = [left, left - right], [0, 1]
    elif assign == 9:
        chans, extra = [left - right, right], [1, 0]
    elif assign == 10:
        chans, extra = [(left + right) >> 1, left - right], [0, 1]
    else:
        chans, extra = [pcm[:, c] for c in range(nch)], [0] * nch
    w = BitWriter()
    for c in range(nch):
        _subframe_safe(w, chans[c], bps + extra[c], plan.subs[c] if c < len(plan.subs) else SubPlan())
    w.pad()
    body = bytes(hdr) + w.bytes()
    return body + struct.pack(">H", crc16(body))


def pcm_md5(pcm, bps):
    nb = (bps + 7) // 8
    x = pcm.astype(numpy.int64).reshape(-1) & ((1 << (8 * nb)) - 1)
    raw = numpy.stack([(x >> (8 * i)) & 0xFF for i in range(nb)], axis=1).astype(numpy.uint8)
    return hashlib.md5(raw.tobytes()).digest()


def encode(pcm, rate, bps, blocksize=4096, variable=False, blocksizes=None, plan=None, extra_blocks=(), id3=None,
           streaminfo_bs=None):
    """pcm (n, channels) ints -> FLAC stream bytes.  ``blocksizes``: explicit block sizes (variable blocking, or fixed
    with a short last block); ``plan(frame_index) -> FramePlan``; ``extra_blocks``: (type, payload) metadata blocks after
    STREAMINFO; ``id3``: an ID3v2 tag payload to put in front."""
    pcm = numpy.asarray(pcm, dtype=numpy.int64)
    if pcm.ndim == 1:
        pcm = pcm[:, None]
    n, nch = pcm.shape
    if blocksizes is None:
        blocksizes = [blocksize] * (n // blocksize) + ([n % blocksize] if n % blocksize else [])
    assert sum(blocksizes) == n and all(b > 0 for b in blocksizes)
    frames, first = [], 0
    for k, bs in enumerate(blocksizes):
        fp = plan(k) if plan else FramePlan()
        frames.append(_frame(pcm[first:first + bs], first, k, rate, bps, variable, fp))
        first += bs
    body = blocksizes[:-1] if len(blocksizes) > 1 else blocksizes
    min_bs, max_bs = streaminfo_bs or (min(body), max(blocksizes))
    sizes = [len(f) for f in frames]
    si = BitWriter()
    si.put(min_bs, 16); si.put(max_bs, 16); si.put(min(sizes), 24); si.put(max(sizes), 24)
    si.put(rate, 20); si.put(nch - 1, 3); si.put(bps - 1, 5); si.put(n, 36)
    blocks = [(0, si.bytes() + pcm_md5(pcm, bps))] + list(extra_blocks)
    out = bytearray()
    if id3 is not None:
        size = len(id3)
        out += b"ID3\x04\x00\x00" + bytes([(size >> 21) & 0x7F, (size >> 14) & 0x7F, (size >> 7) & 0x7F, size & 0x7F]) + id3
    out += b"fLaC"
    for i, (t, payload) in enumerate(blocks):
        out.append((0x80 if i == len(blocks) - 1 else 0) | t)
        out += len(payload).to_bytes(3, "big") + payload
    for f in frames:
        out += f
    return bytes(out)


# -------------------------------------------------------------------------------------------------------- decoder

class _Bits:
    def __init__(self, data, pos):
        self.d = data
        self.bit = pos * 8

    def read(self, n):
        if n == 0:
            return 0
        i, off = self.bit >> 3, self.bit & 7
        nbytes = (off + n + 7) // 8
        if i + nbytes > len(self.d):
            raise ValueError("truncated frame")
        v = int.from_bytes(self.d[i:i + nbytes], "big")
        self.bit += n
        return (v >> (nbytes * 8 - off - n)) & ((1 << n) - 1)

    def sread(self, n):
        v = self.read(n)
        return v - (1 << n) if n and v >> (n - 1) else v

    def unary(self):
        q = 0
        while self.read(1) == 0:
            q += 1
        return q

    @property
    def byte(self):
        return self.bit >> 3


def read_metadata(data):
    """-> (streaminfo dict, offset of the first frame)"""
    p = 0
    if data[:3] == b"ID3":
        size = (data[6] << 21) | (data[7] << 14) | (data[8] << 7) | data[9]
        p = 10 + size + (10 if data[5] & 0x10 else 0)
    if data[p:p + 4] != b"fLaC":
        raise ValueError("not a FLAC stream")
    p += 4
    info, last = None, False
    while not last:
        last, t, n = data[p] >> 7, data[p] & 0x7F, int.from_bytes(data[p + 1:p + 4], "big")
        if t == 0:
            b = _Bits(data, p + 4)
            info = dict(min_bs=b.read(16), max_bs=b.read(16), min_frame=b.read(24), max_frame=b.read(24), rate=b.read(20),
                        channels=b.read(3) + 1, bps=b.read(5) + 1, total=b.read(36), md5=bytes(data[p + 22:p + 38]))
        p += 4 + n
    if info is None:
        raise ValueError("no STREAMINFO")
    return info, p


def decode(data):
    """FLAC bytes -> (streaminfo dict, int64 samples (total, channels)).  Frames are read one after the other from the
    end of the metadata; every CRC, reserved value and frame number is checked.  info["frame_offsets"]: where each
    frame starts."""
    data = bytes(data)
    info, p = read_metadata(data)
    out, total, index = [], 0, 0
    info["frame_offsets"] = []
    while total < info["total"]:
        info["frame_offsets"].append(p)
        b = _Bits(data, p)
        sync = b.read(15)
        if sync != 0x7FFC:
            raise ValueError("lost sync at byte %d" % p)
        variable = b.read(1)
        bcode, rcode, acode, scode, reserved = b.read(4), b.read(4), b.read(4), b.read(3), b.read(1)
        if reserved or bcode == 0 or rcode == 15 or acode > 10 or scode in (3, 7):
            raise ValueError("reserved header value")
        lead = b.read(8)
        ones = 0
        while ones < 8 and lead & (0x80 >> ones):
            ones += 1
        if ones == 1 or ones == 8 or (not variable and ones == 7):
            raise ValueError("bad coded number")
        nbytes = max(ones, 1)
        num = lead & (0x7F >> ones) if ones else lead
        for _ in range(nbytes - 1):
            c = b.read(8)
            if c >> 6 != 2:
                raise ValueError("bad coded number")
            num = (num << 6) | (c & 0x3F)
        if bcode == 1: bs = 192
        elif bcode <= 5: bs = 576 << (bcode - 2)
        elif bcode == 6: bs = b.read(8) + 1
        elif bcode == 7: bs = b.read(16) + 1
        else: bs = 256 << (bcode - 8)
        if rcode == 12: b.read(8)
        elif rcode in (13, 14): b.read(16)
        if b.read(8) != crc8(data[p:b.byte - 1]):
            raise ValueError("header CRC-8 mismatch at byte %d" % p)
        if num != (total if variable else index):
            raise ValueError("frame number out of sequence")
        bps = info["bps"] if scode == 0 else {1: 8, 2: 12, 4: 16, 5: 20, 6: 24}[scode]
        nch = acode + 1 if acode <= 7 else 2
        chans = []
        for c in range(nch):
            side = (acode == 8 and c == 1) or (acode == 9 and c == 0) or (acode == 10 and c == 1)
            chans.append(_ref_subframe(b, bs, bps + side))
        if b.bit & 7:
            if b.read(8 - (b.bit & 7)):
                raise ValueError("nonzero padding")
        end = b.byte
        if b.read(16) != crc16(data[p:end]):
            raise ValueError("frame CRC-16 mismatch at byte %d" % p)
        if acode == 8:
            chans[1] = chans[0] - chans[1]
        elif acode == 9:
            chans[0] = chans[0] + chans[1]
        elif acode == 10:
            mid, side = chans
            mid = (mid << 1) | (side & 1)
            chans = [(mid + side) >> 1, (mid - side) >> 1]
        out.append(numpy.stack(chans, axis=1))
        total += bs
        index += 1
        p = end + 2
    if total != info["total"]:
        raise ValueError("block sizes do not sum to the total")
    return info, numpy.concatenate(out) if out else numpy.zeros((0, info["channels"]), numpy.int64)


def _ref_subframe(b, bs, sbps):
    if b.read(1):
        raise ValueError("subframe padding bit set")
    t = b.read(6)
    wasted = b.unary() + 1 if b.read(1) else 0
    sbps -= wasted
    x = numpy.zeros(bs, dtype=numpy.int64)
    if t == 0:
        x[:] = b.sread(sbps)
    elif t == 1:
        for i in range(bs):
            x[i] = b.sread(sbps)
    elif 8 <= t <= 12 or t >= 32:
        order = t - 8 if t <= 12 else t - 31
        for i in range(order):
            x[i] = b.sread(sbps)
        if t <= 12:
            coefs, shift = FIXED_COEFS[order], 0
        else:
            prec = b.read(4) + 1
            if prec == 16:
                raise ValueError("invalid coefficient precision")
            shift = b.sread(5)
            if shift < 0:
                raise ValueError("negative LPC shift")
            coefs = [b.sread(prec) for _ in range(order)]
        method = b.read(2)
        if method > 1:
            raise ValueError("reserved residual coding method")
        porder = b.read(4)
        pbits, esc = (5, 31) if method else (4, 15)
        res = []
        for part in range(1 << porder):
            n = (bs >> porder) - (order if part == 0 else 0)
            k = b.read(pbits)
            if k == esc:
                width = b.read(5)
                res += [b.sread(width) for _ in range(n)]
            else:
                for _ in range(n):
                    u = (b.unary() << k) | b.read(k)
                    res.append((u >> 1) ^ -(u & 1))
        for i in range(order, bs):
            s = 0
            for j, c in enumerate(coefs):
                s += c * int(x[i - j - 1])
            x[i] = res[i - order] + (s >> shift)
    else:
        raise ValueError("reserved subframe type %d" % t)
    return x << wasted


# ------------------------------------------------------------------------------------------------- test material

def synth_pcm(rng, n, nch, bps, wasted=0, constant_run=False):
    """speech-like ints: a few decaying tones, noise and a random walk, optionally with a silent / DC stretch and with
    `wasted` low bits zero"""
    t = numpy.arange(n)
    lim = (1 << (bps - 1)) - 1
    chans = []
    base = numpy.zeros(n)
    for _ in range(3):
        base += rng.uniform(0.05, 0.3) * numpy.sin(2 * numpy.pi * rng.uniform(80, 3000) / 16000 * t + rng.uniform(0, 6))
    for c in range(nch):
        x = base * rng.uniform(0.5, 1.0) + 0.02 * rng.standard_normal(n) + 0.001 * numpy.cumsum(rng.standard_normal(n))
        x = numpy.clip(numpy.round(x * lim), -lim - 1, lim).astype(numpy.int64)
        if constant_run and n > 64:
            a = int(rng.integers(0, n // 2))
            x[a:a + n // 3] = int(rng.integers(-3, 4))
        if wasted:
            x = (x >> wasted) << wasted
        chans.append(x)
    return numpy.stack(chans, axis=1)


def random_plan(rng, nch, max_order=32, tools=None):
    """FramePlan factory drawing every coding tool at random (``tools`` restricts the subframe kinds)"""
    kinds = tools or ["auto", "constant", "verbatim", "fixed", "lpc"]

    def plan(k):
        subs = []
        for _ in range(nch):
            kind = kinds[int(rng.integers(len(kinds)))]
            order = int(rng.integers(0, 5)) if kind == "fixed" else int(rng.integers(1, max_order + 1))
            porder = int(rng.integers(0, 9)) if rng.random() < 0.8 else 15
            esc = tuple(int(e) for e in rng.integers(0, 1 << min(porder, 3), size=int(rng.integers(0, 3))))
            subs.append(SubPlan(kind=kind, order=order, precision=int(rng.integers(1, 16)), method=int(rng.integers(2)),
                                porder=porder, escape=esc, wasted=bool(rng.random() < 0.8)))
        assign = ["independent", "left_side", "side_right", "mid_side"][int(rng.integers(4))] if nch == 2 else "independent"
        return FramePlan(assign=assign, bs_code=["auto", "8", "16"][int(rng.integers(3))],
                         rate_code=["streaminfo", "table", "khz", "hz", "10hz"][int(rng.integers(5))],
                         size_code=["streaminfo", "explicit"][int(rng.integers(2))], subs=subs)
    return plan


def matrix_case(i, seed=0):
    """The i-th file of the tool matrix: cycles bps 8/12/16/20/24, 1-8 channels, fixed and variable blocking, a short
    last frame, one-frame files of fewer than 16 samples, silent stretches and wasted bits.  -> (bytes, pcm, rate, bps)"""
    rng = numpy.random.default_rng(seed * 100003 + i)
    bps = (8, 12, 16, 20, 24)[i % 5]
    nch = (1, 2, 2, 1, 3, 2, 4, 5, 6, 7, 8)[i % 11]
    rate = (16000, 8000, 44100, 48000, 22050, 11025)[i % 6]
    variable = (i // 3) % 2 == 1
    if i % 13 == 7:
        n = int(rng.integers(1, 16))                                 # one frame of fewer than 16 samples
        blocksizes = [n]
    elif variable:
        n = int(rng.integers(300, 3000))
        blocksizes, left = [], n
        while left:
            b = min(left, int(rng.integers(16, 700)))
            blocksizes.append(b)
            left -= b
    else:
        bs = (192, 256, 576, 1024, 4096, 300, 1152)[i % 7]
        n = int(rng.integers(bs // 2, 3 * bs + 1)) if bs < 3000 else int(rng.integers(bs + 1, 2 * bs))
        blocksizes = None
    wasted = int(rng.integers(1, 4)) if i % 4 == 1 and bps > 8 else 0
    pcm = synth_pcm(rng, n, nch, bps, wasted=wasted, constant_run=i % 3 == 0)
    blocksize = (192, 256, 576, 1024, 4096, 300, 1152)[i % 7]
    data = encode(pcm, rate, bps, blocksize=blocksize, variable=variable, blocksizes=blocksizes,
                  plan=random_plan(rng, nch), streaminfo_bs=(blocksize, blocksize) if not variable and blocksizes is None else None)
    return data, pcm, rate, bps
