"""Ordinary gzip crafted for the device inflate tests (sage2_b200/csrc/gunzip.cu): members written segment by segment with
Python's zlib, so that the tests know where DEFLATE blocks start, and zlib's own gzread (libz.so.1 through ctypes) as the
oracle -- the reference reads its input through kseq + gzread."""
import ctypes
import os
import struct
import tempfile
import zlib

_z = ctypes.CDLL("libz.so.1")
_z.gzopen.restype = ctypes.c_void_p
_z.gzopen.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
_z.gzread.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint]
_z.gzclose.argtypes = [ctypes.c_void_p]


def gzread(blob: bytes):
    """(text, ok): what zlib's gzread returns for the file `blob`; ok = False when it reported an error (-1) or stopped with a
    truncated stream (Z_BUF_ERROR: the partial text without an error return)."""
    fd, path = tempfile.mkstemp(suffix=".gz")
    try:
        os.write(fd, blob)
        os.close(fd)
        f = _z.gzopen(path.encode(), b"rb")
        buf = ctypes.create_string_buffer(1 << 16)
        out = []
        while True:
            n = _z.gzread(f, buf, 1 << 16)
            if n <= 0:
                break
            out.append(buf.raw[:n])
        err = ctypes.c_int(0)
        _z.gzerror.restype = ctypes.c_char_p
        _z.gzerror.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int)]
        _z.gzerror(f, ctypes.byref(err))
        _z.gzclose(f)
        return b"".join(out), n == 0 and err.value == 0
    finally:
        os.unlink(path)


def header(fname: bytes = None, comment: bytes = None, extra: bytes = None, hcrc: bool = False, mtime: int = 0) -> bytes:
    flg = (8 if fname is not None else 0) | (16 if comment is not None else 0) | (4 if extra is not None else 0) | (2 if hcrc else 0)
    h = b"\x1f\x8b\x08" + bytes([flg]) + struct.pack("<I", mtime) + b"\x00\x03"
    if extra is not None:
        h += struct.pack("<H", len(extra)) + extra
    if fname is not None:
        h += fname + b"\0"
    if comment is not None:
        h += comment + b"\0"
    if hcrc:
        h += struct.pack("<H", zlib.crc32(h) & 0xFFFF)
    return h


def deflate(segments, flush=zlib.Z_SYNC_FLUSH):
    """Raw DEFLATE of the segments [(text, level, strategy)], each by a compressor of its own (no match crosses a segment) and
    ended by `flush` (byte-aligned), the last one finished.  Returns (data, starts): starts[i] = the byte where segment i's first
    block begins."""
    out, starts = b"", []
    for i, (text, level, strategy) in enumerate(segments):
        starts.append(len(out))
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
        out += c.compress(text) + c.flush(zlib.Z_FINISH if i == len(segments) - 1 else flush)
    return out, starts


def member(text: bytes = None, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, segments=None, flush=zlib.Z_SYNC_FLUSH,
           **hdr) -> bytes:
    """One gzip member of `text` (or of the segments of deflate())"""
    segments = segments or [(text, level, strategy)]
    whole = b"".join(s[0] for s in segments)
    data, _ = deflate(segments, flush)
    return header(**hdr) + data + struct.pack("<II", zlib.crc32(whole), len(whole) & 0xFFFFFFFF)


def stream(text: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, flush_every: int = 0, flush=zlib.Z_SYNC_FLUSH) -> bytes:
    """One member written by one compressor, flushed every `flush_every` bytes of text (0: never)"""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    data = b""
    step = flush_every or max(1, len(text))
    for i in range(0, len(text), step):
        data += c.compress(text[i:i + step])
        if flush_every:
            data += c.flush(flush)
    data += c.flush(zlib.Z_FINISH)
    return header() + data + struct.pack("<II", zlib.crc32(text), len(text) & 0xFFFFFFFF)
