"""BGZF writer for the tests (htslib's bgzip format, written with stdlib zlib): gzip members with a `BC` extra subfield holding
BSIZE (member size - 1), raw DEFLATE data, CRC32 and ISIZE, and the 28-byte end-of-file member.  Controls what the device
decoder has to meet: level 0 (stored) .. 9, the Z_FIXED / Z_HUFFMAN_ONLY / Z_RLE strategies, sync flushes inside a member
(several blocks, empty stored blocks) and member sizes from 1 byte to 65,280 bytes."""
from __future__ import annotations

import gzip
import struct
import zlib

EOF_MEMBER = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
MAX_TEXT = 65280        # bgzip's largest text per member: even stored, the member stays within 64 KiB


def deflate(text: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, sync_every: int = 0) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    if not sync_every:
        return co.compress(text) + co.flush()
    out = []
    for p in range(0, len(text), sync_every):
        out.append(co.compress(text[p:p + sync_every]))
        out.append(co.flush(zlib.Z_SYNC_FLUSH))      # ends the block, then an empty stored block
    out.append(co.flush())
    return b"".join(out)


def member(text: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, sync_every: int = 0, data: bytes | None = None,
           crc: int | None = None, isize: int | None = None) -> bytes:
    """One BGZF member of `text`; `data`, `crc`, `isize` replace the computed DEFLATE data / trailer fields (corrupt members)."""
    d = deflate(text, level, strategy, sync_every) if data is None else data
    bsize = 12 + 6 + len(d) + 8 - 1
    assert bsize < 65536, "member larger than 64 KiB"
    head = struct.pack("<BBBBIBBH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6) + b"BC" + struct.pack("<HH", 2, bsize)
    return head + d + struct.pack("<II", zlib.crc32(text) if crc is None else crc, len(text) if isize is None else isize)


def split(text: bytes, sizes=MAX_TEXT) -> list[bytes]:
    """text cut into member texts: `sizes` is one size or a sequence used cyclically"""
    sizes = [sizes] if isinstance(sizes, int) else list(sizes)
    out, p, i = [], 0, 0
    while p < len(text):
        n = max(1, min(MAX_TEXT, sizes[i % len(sizes)]))
        out.append(text[p:p + n])
        p += n
        i += 1
    return out


def write(text: bytes, sizes=MAX_TEXT, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, sync_every: int = 0, eof: bool = True,
          plain_from: int | None = None) -> bytes:
    """text as BGZF; members from index `plain_from` on are ordinary gzip members without the BC field"""
    parts = []
    for i, t in enumerate(split(text, sizes)):
        if plain_from is not None and i >= plain_from:
            parts.append(gzip.compress(t, compresslevel=level if level else 1, mtime=0))
        else:
            parts.append(member(t, level, strategy, sync_every))
    if eof:
        parts.append(EOF_MEMBER)
    return b"".join(parts)


def members(blob: bytes) -> list[tuple[int, int]]:
    """(offset, size) of every BGZF member of blob, from the BSIZE fields"""
    out, p = [], 0
    while p < len(blob):
        xlen = struct.unpack_from("<H", blob, p + 10)[0]
        q, size = p + 12, None
        while q < p + 12 + xlen:
            slen = struct.unpack_from("<H", blob, q + 2)[0]
            if blob[q:q + 2] == b"BC" and slen == 2:
                size = struct.unpack_from("<H", blob, q + 4)[0] + 1
            q += 4 + slen
        assert size is not None, "not a BGZF member"
        out.append((p, size))
        p += size
    return out
