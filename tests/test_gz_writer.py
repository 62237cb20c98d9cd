"""The gzip crafting helper (tests/gz.py) on the CPU: its members are what Python's gzip module and zlib's gzread read, and the
gzread oracle reports the errors the device path must report."""
import gzip
import zlib

import gz


def test_members_read_back():
    text = b"@r1\nACGT\n+\nIIII\n" * 5000
    for blob in (gz.member(text), gz.member(text, 1, fname=b"a.fq", comment=b"c", extra=b"XY\x02\x00ab", hcrc=True),
                 gz.stream(text, 9, flush_every=7000), gz.stream(text, 6, flush_every=5000, flush=zlib.Z_FULL_FLUSH),
                 gz.member(segments=[(text[:30000], 6, 0), (text[30000:], 0, 0)])):
        assert gzip.decompress(blob) == text
        assert gz.gzread(blob) == (text, True)


def test_segment_starts_are_block_starts():
    a, b = b"ACGT" * 3000, b"TTGCA" * 2000
    data, starts = gz.deflate([(a, 6, 0), (b, 6, 0)])
    assert starts[0] == 0 and zlib.decompressobj(-15).decompress(data[starts[1]:]) == b


def test_gzread_oracle_errors():
    m = gz.member(b"A" * 1000)
    assert gz.gzread(m + b"hello world") == (b"A" * 1000, True)           # trailing garbage is ignored
    assert gz.gzread(m + b"\0" * 100) == (b"A" * 1000, True)
    assert not gz.gzread(m[:-3])[1]                                      # truncated trailer
    assert not gz.gzread(m + b"\x1f\x8bjunkjunk")[1]                      # magic followed by junk
    bad = bytearray(m)
    bad[-8] ^= 1
    assert not gz.gzread(bytes(bad))[1]                                  # CRC
    assert gz.gzread(gz.member(b"") + m) == (b"A" * 1000, True)          # an empty member
