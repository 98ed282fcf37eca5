"""A BGZF image whose literal/length code does not fit the inflate kernel's second-level tables, so that every code longer than
the primary table is resolved by the canonical walk (range limits and index offsets in the stream's global scratch).

The dynamic Huffman block is written by hand: six literals get codes of 2..7 bits, the other 260 symbols of the literal/length
alphabet 9-bit codes.  With an 8-bit primary table the 9-bit codes fill 130 table prefixes, two codes each; every prefix needs a
sub-table of the minimum 8 entries, 1040 in all, more than the 1016 the sub-table area holds.  (Test infrastructure.)"""
import random
import struct
import zlib

SHORT = {ord("A"): 2, ord("C"): 3, ord("G"): 4, ord("T"): 5, ord("N"): 6, ord("\n"): 7}
HLIT, HDIST = 266, 4
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
LBITS, SUB_CAPACITY = 8, 1016   # FASTF_TPS_LBITS, FASTF_TPS_LITSUB_U16 (bgzf_inflate_tps.cuh)


class _Bits:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def put(self, v, n):   # n bits of v, least significant first
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, c, n):   # a Huffman code, most significant bit first
        self.put(int(format(c, "0%db" % n)[::-1], 2), n)

    def flush(self):
        if self.n:
            self.out.append(self.acc & 255)
        self.acc, self.n = 0, 0
        return bytes(self.out)


def _canonical(lengths):
    """RFC 1951 3.2.2: symbol -> (code, length)"""
    bl_count = [0] * 16
    for l in lengths:
        if l:
            bl_count[l] += 1
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + bl_count[b - 1]) << 1
        nxt[b] = code
    codes = {}
    for s, l in enumerate(lengths):
        if l:
            codes[s] = (nxt[l], l)
            nxt[l] += 1
    return codes


def lit_lengths():
    return [SHORT.get(s, 9) for s in range(HLIT)]


def subtable_entries(lengths, tbits=LBITS):
    """entries the kernel's second-level tables would need for this code (sub-table per table prefix, at least 8 entries)"""
    longest = {}
    for sym, (c, l) in _canonical(lengths).items():
        if l > tbits:
            p = c >> (l - tbits)
            longest[p] = max(longest.get(p, 0), l - tbits)
    return sum(8 if b < 3 else 1 << b for b in longest.values())


def deflate_walk_block(payload):
    """one final dynamic-Huffman deflate block, literals only, with the code of lit_lengths()"""
    lit = lit_lengths()
    dist = [2] * HDIST
    cl = {9: 2, 2: 3, 3: 3, 4: 3, 5: 3, 6: 3, 7: 3}   # code-length code: complete (1/4 + 6/8)
    cl_lengths = [cl.get(s, 0) for s in range(19)]
    hclen = max(i for i, s in enumerate(CL_ORDER) if cl_lengths[s]) + 1
    w = _Bits()
    w.put(1, 1)
    w.put(2, 2)
    w.put(HLIT - 257, 5)
    w.put(HDIST - 1, 5)
    w.put(hclen - 4, 4)
    for s in CL_ORDER[:hclen]:
        w.put(cl_lengths[s], 3)
    clc = _canonical(cl_lengths)
    for l in lit + dist:
        w.code(*clc[l])
    lc = _canonical(lit)
    for b in payload:
        w.code(*lc[b])
    w.code(*lc[256])
    return w.flush()


def bgzf_block(raw, payload):
    bsize = 18 + len(raw) + 8
    hdr = bytes([0x1F, 0x8B, 8, 4, 0, 0, 0, 0, 0, 0xFF, 6, 0, ord("B"), ord("C"), 2, 0]) + struct.pack("<H", bsize - 1)
    return hdr + raw + struct.pack("<II", zlib.crc32(payload) & 0xFFFFFFFF, len(payload))


def image(seed=5, nblocks=3, size=12000):
    """(BGZF bytes, inflated bytes): walk-only blocks between ordinary zlib blocks, then the BGZF end-of-file block"""
    rng = random.Random(seed)
    common = [b for b in range(256) if b not in SHORT]
    img, want = bytearray(), bytearray()
    for k in range(nblocks):
        # mostly 9-bit literals (walks), some short ones so that literal runs of every length occur
        p = bytes(rng.choice(common) if rng.random() < 0.8 else rng.choice(list(SHORT)) for _ in range(size + 517 * k))
        raw = deflate_walk_block(p)
        assert zlib.decompress(raw, -15) == p
        img += bgzf_block(raw, p)
        want += p
        q = bytes(rng.choice(b"ACGTN\t\n0123") for _ in range(5000))
        zc = zlib.compressobj(6, zlib.DEFLATED, -15)
        img += bgzf_block(zc.compress(q) + zc.flush(), q)
        want += q
    img += bgzf_block(zlib.compressobj(6, zlib.DEFLATED, -15).flush(), b"")
    return bytes(img), bytes(want)
