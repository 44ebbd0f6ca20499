"""Greedy LZ4 block encoder, one sequential definition -- the specification of K7 (a0_k7_lz4_encode).

Test infrastructure only.  K7 must produce exactly these bytes (tests/test_gpu_lz4_encode.py), and
the output is an ordinary python-lz4 block, so ``oracle.lz4_block.decode``, K6a (a0_ex_decode) and
the system liblz4 all read it (tests/test_lz4_encode_oracle.py).

The parse:

* a table of 4096 entries holds, for each hash, the last position inserted (all entries start at 0);
  ``h(p) = (read32le(p) * 2654435761 mod 2^32) >> 20``;
* at every position p (step 1) the candidate c = table[h(p)] is read and p is inserted; c counts when
  c < p, p - c <= 65535 (the format's offset limit) and the 4 bytes at c and p are equal;
* no match starts within the last 12 bytes (p + 12 <= n) and the last 5 bytes are literals, so a
  match is extended forward (only) while its end e < n - 5;
* after a match [p, e) the position e - 2 is inserted and the search resumes at e.

If the python-lz4 block (4-byte little-endian size + block) is not shorter than the input, the input
itself is returned: K6a takes a blob of exactly the decoded size as uncompressed.
"""

HASH_LOG = 12
MIN_MATCH = 4
LAST_LITERALS = 5
MF_LIMIT = 12
MAX_OFFSET = 65535


def hash4(word):
    return ((word * 2654435761) & 0xFFFFFFFF) >> (32 - HASH_LOG)


def _length(extra, out):
    while extra >= 255:
        out.append(255)
        extra -= 255
    out.append(extra)


def _sequence(out, lit, off, ml):
    ll = len(lit)
    tok = (min(ll, 15) << 4) | (0 if ml is None else min(ml - MIN_MATCH, 15))
    out.append(tok)
    if ll >= 15:
        _length(ll - 15, out)
    out += lit
    if ml is None:
        return
    out += bytes((off & 255, off >> 8))
    if ml - MIN_MATCH >= 15:
        _length(ml - MIN_MATCH - 15, out)


def encode_block(data):
    """The raw LZ4 block of the greedy parse (no size prefix)."""
    data = bytes(data)
    n = len(data)
    table = [0] * (1 << HASH_LOG)
    rd = lambda p: int.from_bytes(data[p:p + 4], "little")
    out = bytearray()
    anchor = p = 0
    while p + MF_LIMIT <= n:
        h = hash4(rd(p))
        c = table[h]
        table[h] = p
        if c < p and p - c <= MAX_OFFSET and data[c:c + 4] == data[p:p + 4]:
            off = p - c
            e = p + MIN_MATCH
            while e < n - LAST_LITERALS and data[e] == data[e - off]:
                e += 1
            _sequence(out, data[anchor:p], off, e - p)
            table[hash4(rd(e - 2))] = e - 2
            anchor = p = e
        else:
            p += 1
    _sequence(out, data[anchor:], None, None)
    return bytes(out)


def encode_greedy(data):
    """python-lz4 blob of ``data`` (the decoded size as 4 bytes little-endian, then the block), or
    ``data`` itself when that blob would not be shorter."""
    data = bytes(data)
    blob = len(data).to_bytes(4, "little") + encode_block(data)
    return blob if len(blob) < len(data) else data
