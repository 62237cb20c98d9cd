"""GFA 1.0 of an overlap graph, independent of the CUDA writer (sage2gpu_write_gfa, include/sage2gpu.h).

write_gfa  the GFA bytes from the text of a `.reads` file and a `.graph3` file (what the reference's saveReadsInFile /
           saveOverlapGraphInFile write): "H\tVN:Z:1.0\n", one S line per read in id order, then one L line per undirected
           edge in `.graph3` order -- the record (a, b, type, delta) with a < b, its twin skipped -- with overlap
           n = len(b) - delta and the orientations of TYPE_ORIENTATION.
validate   checks a GFA of that form on its own: the header; S ids 1..U contiguous, LN = sequence length, sequences over
           ACGT; every L names existing segments, has k <= n <= min(len a, len b) and is an exact overlap: the last n bases
           of a in orientation oa equal the first n bases of b in orientation ob.  Raises GfaError.
"""
from __future__ import annotations

import contextlib
import io

# edge type of .graph3 (SURVEY 8 A8) -> (oa, ob)
TYPE_ORIENTATION = {
    3: (b"+", b"+"),     # fwd b prefix on fwd a suffix
    2: (b"+", b"-"),     # rc b prefix on fwd a suffix
    0: (b"-", b"-"),     # fwd b suffix on fwd a prefix
    1: (b"-", b"+"),     # rc b suffix on fwd a prefix
}

HEADER = b"H\tVN:Z:1.0\n"
_RC = bytes.maketrans(b"ACGT", b"TGCA")


class GfaError(ValueError):
    pass


def _open(src, mode="rb"):
    """A path opened (and closed on exit), or a file object used as it is (left open)."""
    if isinstance(src, (str, bytes)) or hasattr(src, "__fspath__"):
        return open(src, mode)
    return contextlib.nullcontext(src)


def write_gfa(reads_src, graph3_src, out) -> None:
    """reads_src / graph3_src: paths or binary file objects; out: a path or a binary file object."""
    with _open(out, "wb") as fo:
        fo.write(HEADER)
        lengths = [0]
        with _open(reads_src) as fr:
            U = int(fr.readline())
            buf = []
            for i in range(1, U + 1):
                freq, ln, fwd, _ = fr.readline().rstrip(b"\n").split(b"\t")
                lengths.append(int(ln))
                buf.append(b"S\t%d\t%s\tLN:i:%s\tRC:i:%s\n" % (i, fwd, ln, freq))
                if len(buf) >= 65536:
                    fo.write(b"".join(buf))
                    buf = []
            fo.write(b"".join(buf))
        with _open(graph3_src) as fg:
            for _ in range(3):              # genomeSize, numberOfReads, averageReadLength
                fg.readline()
            buf = []
            for line in fg:
                if line == b"\n":
                    continue
                f = line.split(b"\t")
                a, b = int(f[0]), int(f[1])
                if a >= b:                  # the twin record of an edge already written
                    continue
                oa, ob = TYPE_ORIENTATION[int(f[2])]
                buf.append(b"L\t%d\t%s\t%d\t%s\t%dM\n" % (a, oa, b, ob, lengths[b] - int(f[4])))
                if len(buf) >= 65536:
                    fo.write(b"".join(buf))
                    buf = []
            fo.write(b"".join(buf))


def write_gfa_bytes(reads_src, graph3_src) -> bytes:
    out = io.BytesIO()
    write_gfa(reads_src, graph3_src, out)
    return out.getvalue()


def _oriented(seq: bytes, o: bytes) -> bytes:
    return seq if o == b"+" else seq.translate(_RC)[::-1]


def validate(src, k: int) -> dict:
    """src: bytes, a path or a binary file object.  Returns {"segments": U, "links": E}; raises GfaError at the first fault."""
    with (io.BytesIO(src) if isinstance(src, (bytes, bytearray)) else _open(src)) as f:
        if f.readline() != HEADER:
            raise GfaError("line 1: not the header H\\tVN:Z:1.0")
        seqs = [b""]                         # 1-based
        links = 0
        lineno = 1
        for line in f:
            lineno += 1
            if not line.endswith(b"\n"):
                raise GfaError(f"line {lineno}: no line end")
            x = line[:-1].split(b"\t")
            if x[0] == b"S":
                if links:
                    raise GfaError(f"line {lineno}: S line after the L lines")
                if len(x) != 5 or not x[3].startswith(b"LN:i:") or not x[4].startswith(b"RC:i:"):
                    raise GfaError(f"line {lineno}: S line has not the fields id, sequence, LN:i, RC:i")
                if x[1] != b"%d" % len(seqs):
                    raise GfaError(f"line {lineno}: segment id {x[1]!r}, expected {len(seqs)}")
                s = x[2]
                if not s or s.translate(None, b"ACGT"):
                    raise GfaError(f"line {lineno}: sequence not over ACGT")
                if int(x[3][5:]) != len(s):
                    raise GfaError(f"line {lineno}: LN {x[3][5:]!r} != sequence length {len(s)}")
                if not x[4][5:].isdigit():
                    raise GfaError(f"line {lineno}: RC {x[4][5:]!r} is not a count")
                seqs.append(s)
            elif x[0] == b"L":
                if len(x) != 6 or not x[5].endswith(b"M"):
                    raise GfaError(f"line {lineno}: L line has not the fields a, oa, b, ob, <n>M")
                a, oa, b, ob, n = int(x[1]), x[2], int(x[3]), x[4], int(x[5][:-1])
                if not (1 <= a < len(seqs)) or not (1 <= b < len(seqs)):
                    raise GfaError(f"line {lineno}: link to a missing segment ({a}, {b})")
                if oa not in (b"+", b"-") or ob not in (b"+", b"-"):
                    raise GfaError(f"line {lineno}: bad orientation")
                sa, sb = seqs[a], seqs[b]
                if not (k <= n <= min(len(sa), len(sb))):
                    raise GfaError(f"line {lineno}: overlap {n} outside [{k}, {min(len(sa), len(sb))}]")
                if _oriented(sa, oa)[len(sa) - n:] != _oriented(sb, ob)[:n]:
                    raise GfaError(f"line {lineno}: {a}{oa.decode()} {b}{ob.decode()} is not an exact overlap of {n} bases")
                links += 1
            else:
                raise GfaError(f"line {lineno}: unexpected record type {x[0]!r}")
        return {"segments": len(seqs) - 1, "links": links}
