"""Ordinary gzip inflated on the device (sage2_b200/csrc/gunzip.cu): sage2gpu_inflate_gzip equals zlib's gzread byte for
byte, block starts found on the device split a piece into ranges decoded at once (false candidates rejected), data that
gzread rejects gives SAGE2GPU_ERR_FORMAT naming the compressed offset and leaves the context usable, pieces carry their state
across contexts, and `sage2gpu` on gzip input writes the same files as on the plain text."""
import hashlib
import json
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import datasets
import gz
import long_datasets
from sage2_b200 import api, synth

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "golden.json")))
BIG = json.load(open(os.path.join(HERE, "golden", "golden_big.json")))
BIN = os.path.join(os.path.dirname(api.LIB_PATH), "sage2gpu")
STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "huffman": zlib.Z_HUFFMAN_ONLY, "rle": zlib.Z_RLE,
              "fixed": zlib.Z_FIXED}


@pytest.fixture(scope="module")
def gpu():
    g = api.Sage2Gpu(0)
    yield g
    g.close()


def _text(kind: str, n: int = 4000, seed: int = 9) -> bytes:
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        s = bytes(rng.choice(list(b"ACGTN"), p=[0.3, 0.2, 0.2, 0.29, 0.01], size=int(rng.integers(50, 300))).astype(np.uint8))
        if kind == "fastq":
            q = bytes(rng.integers(33, 75, size=len(s)).astype(np.uint8))
            out.append(b"@read%d/1 lane=3\n%s\n+\n%s\n" % (i, s, q))
        else:
            out.append(b">read%d\n%s\n" % (i, s))
    return b"".join(out)


def _same(gpu, blob):
    want, ok = gz.gzread(blob)
    assert ok
    got, ms, ranges, confirmed, rejected = gpu.inflate_gzip(blob)
    assert got == want
    assert 1 <= confirmed <= ranges and rejected < ranges
    return confirmed, rejected


@pytest.mark.parametrize("kind", ["fastq", "fasta"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_levels_equal_gzread(gpu, kind, level):
    _same(gpu, gz.stream(_text(kind, 20000), level))


@pytest.mark.parametrize("strategy", sorted(STRATEGIES))
def test_strategies_equal_gzread(gpu, strategy):
    _same(gpu, gz.stream(_text("fastq", 12000), 6, STRATEGIES[strategy]))


@pytest.mark.parametrize("flush", [zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH])
def test_flushes_equal_gzread(gpu, flush):
    _same(gpu, gz.stream(_text("fastq", 12000), 6, flush_every=7777, flush=flush))


def test_incompressible_runs_and_far_matches(gpu):
    rng = np.random.default_rng(3)
    noise = bytes(rng.integers(0, 256, size=300000).astype(np.uint8))
    _same(gpu, gz.stream(noise, 6))
    _same(gpu, gz.stream(b"A" * 3000000 + b"C" * 700001, 9))                # distance 1, length 258 throughout
    # a block that starts right where a 32 KiB stretch repeats: every match of the range that starts there reaches 32768 back
    acgt = bytes(rng.choice(list(b"ACGT"), size=96 * 1024).astype(np.uint8))
    rep = acgt[-32768:]
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    data = c.compress(acgt) + c.flush(zlib.Z_SYNC_FLUSH) + c.compress(rep * 3) + c.flush(zlib.Z_FINISH)
    text = acgt + rep * 3
    blob = gz.header() + data + struct.pack("<II", zlib.crc32(text), len(text))
    confirmed, _ = _same(gpu, blob)
    assert confirmed > 1


def test_members_headers_empty_members_and_trailing_bytes(gpu):
    a, b = _text("fastq", 3000, 1), _text("fasta", 2000, 2)
    blob = (gz.member(a, 6, fname=b"a.fastq") + gz.member(b"", 6) + gz.member(b, 1, comment=b"two", extra=b"XY\x03\x00abc", hcrc=True)
            + gz.member(b"", 9, fname=b"", hcrc=True) + gz.member(a[:5000], 9))
    for tail in (b"", b"\0" * 777, b"not a gzip member, ignored", b"\x1f"):
        _same(gpu, blob + tail)


def test_level6_fastq_runs_in_parallel(gpu):
    text = _text("fastq", 25000, 5)
    assert len(text) >= 4 << 20
    confirmed, _ = _same(gpu, gz.stream(text, 6))
    assert confirmed > 1


def test_false_block_starts_are_rejected(gpu):
    # stored blocks full of a dynamic-block header: every chunk that falls inside them finds a candidate there
    text = _text("fastq", 6000, 7)
    hdr = gz.deflate([(text[:20000], 6, 0)])[0][:256]
    fake = hdr * 4000
    blob = gz.header() + gz.deflate([(text[:200000], 6, 0), (fake, 0, 0), (text[200000:], 6, 0)])[0]
    whole = text[:200000] + fake + text[200000:]
    blob += struct.pack("<II", zlib.crc32(whole), len(whole))
    _, rejected = _same(gpu, blob)
    assert rejected >= 1


def _corrupt():
    """case -> (gzip bytes, compressed offset the error names)"""
    a, b = _text("fastq", 600, 11), _text("fastq", 30, 12)
    H = len(gz.header())
    data, starts = gz.deflate([(a, 6, 0), (b, 6, 0)])
    blk2 = H + starts[1]
    good = gz.header() + data + struct.pack("<II", zlib.crc32(a + b), len(a + b))
    out = {}
    x = bytearray(good); x[-8] ^= 1; out["crc"] = (bytes(x), 0)
    x = bytearray(good); x[-4] ^= 1; out["isize"] = (bytes(x), 0)
    x = bytearray(good); x[blk2] |= 0b110; out["type3"] = (bytes(x), blk2)
    # a later block with an over-subscribed code-length code: BFINAL, BTYPE 2, HLIT 0, HDIST 0, HCLEN 15, 19 lengths of 1
    bits = [1, 0, 1] + [0] * 10 + [1, 1, 1, 1] + [1, 0, 0] * 19
    bits += [0] * (-len(bits) % 8)
    over = bytes(sum(bit << i for i, bit in enumerate(bits[j:j + 8])) for j in range(0, len(bits), 8))
    out["oversubscribed"] = (gz.header() + data[:starts[1]] + over + b"\0" * 64 + struct.pack("<II", 0, 0), blk2)
    sdata, sstarts = gz.deflate([(a, 6, 0), (b, 0, 0)])
    x = bytearray(gz.header() + sdata + struct.pack("<II", zlib.crc32(a + b), len(a + b)))
    x[H + sstarts[1] + 3] ^= 0xFF                                             # NLEN
    out["stored_len"] = (bytes(x), H + sstarts[1])
    out["truncated_block"] = (good[:blk2 + (len(data) - starts[1]) // 2], blk2)
    out["truncated_trailer"] = (good[:-3], 0)
    m2 = gz.member(b, 6, fname=b"second")
    out["truncated_header"] = (good + m2[:12], len(good))
    out["magic_junk"] = (good + b"\x1f\x8bjunkjunkjunk", len(good))
    # the second member's first match reaches back into the first member: fixed block, 'A', then length 3 distance 5
    bits = [1, 1, 0]
    def code(c, n):
        bits.extend((c >> i) & 1 for i in reversed(range(n)))
    code(0x30 + ord("A"), 8)
    code(1, 7)                                                               # length 3 (symbol 257)
    code(4, 5)                                                               # distance 5-6 (code 4, one extra bit 0)
    bits.append(0)
    code(0, 7)                                                               # end of block
    bits += [0] * (-len(bits) % 8)
    blk = bytes(sum(bit << i for i, bit in enumerate(bits[j:j + 8])) for j in range(0, len(bits), 8))
    out["distance"] = (good + gz.header() + blk + struct.pack("<II", 0, 4), len(good) + H)
    return out


@pytest.mark.parametrize("case", sorted(_corrupt()))
def test_corrupt_streams_fail_with_their_offset(gpu, case):
    blob, off = _corrupt()[case]
    assert not gz.gzread(blob)[1]
    with pytest.raises(api.Sage2GpuError) as e:
        gpu.inflate_gzip(blob)
    assert e.value.code == api.ERR_FORMAT and e.value.bad_offset == off, str(e.value)
    g = api.Sage2Gpu(0)
    try:
        g.load_begin(31)
        st = api.GzipState()
        with pytest.raises(api.Sage2GpuError) as e:
            g.load_append_gzip(b"", blob, True, st, 1 << 20)
        assert e.value.bad_offset == off and st.offset == 0 and g.load_count() == 0
        text = _text("fastq", 500, 4)
        r = g.load_append_gzip(b"", gz.member(text), True, api.GzipState(), 1 << 20)   # the context is still usable
        assert r["n_records"] == 500 and g.load_count() == 500
    finally:
        g.close()
    _same(gpu, gz.member(b"still fine"))


def _stream_pieces(blob: bytes, feed: int = 20000, bound: int = 65536):
    """blob through load_append_gzip in pieces of `feed` compressed bytes (more while a piece holds no complete block), text
    bound `bound`, alternating between two contexts: (pieces, text consumed, records, records held by the contexts)"""
    ctxs = [api.Sage2Gpu(0), api.Sage2Gpu(0)]
    try:
        for c in ctxs:
            c.load_begin(31)
        st, pre, marker, pos, i, n_rec, used, f = api.GzipState(), b"", 0, 0, 0, 0, 0, feed
        while not st.done:
            chunk = blob[pos:pos + f]
            r = ctxs[i % 2].load_append_gzip(pre, chunk, pos + len(chunk) == len(blob), st, bound, marker)
            pos += r["in_consumed"]
            f = f * 2 if r["in_consumed"] == 0 else feed
            pre, marker = r["rest"], r["marker"]
            n_rec += r["n_records"]
            used += r["consumed"]
            i += 1
        assert pos == len(blob) and pre == b""
        return i, used, n_rec, sum(c.load_count() for c in ctxs)
    finally:
        for c in ctxs:
            c.close()


def test_streaming_pieces_alternate_between_contexts():
    text = _text("fastq", 9000, 21)
    head = text[:text.index(b"\n@read", 100000) + 1]
    blob = gz.member(segments=[(text[:700000], 6, 0), (text[700000:], 1, 0)], fname=b"x") + gz.member(head, 9)
    pieces, used, n_rec, held = _stream_pieces(blob)
    assert pieces > 10 and used == len(text) + len(head)
    assert n_rec == 9000 + head.count(b"@read") == held


@pytest.mark.parametrize("case", ["level0", "stored_segment"])
def test_streaming_stored_blocks_across_pieces(case):
    # stored blocks longer than what is left of a piece: the piece stops at the block's start, the next one decodes it
    text = _text("fastq", 3000, 23)
    if case == "level0":
        blob = gz.stream(text, 0)
    else:
        cut = text.index(b"\n@read", len(text) // 3) + 1
        blob = gz.member(segments=[(text[:cut], 6, 0), (text[cut:2 * cut], 0, 0), (text[2 * cut:], 6, 0)])
    assert gz.gzread(blob) == (text, True)
    pieces, used, n_rec, held = _stream_pieces(blob, feed=30000, bound=1 << 20)
    assert pieces > 4 and used == len(text) and n_rec == 3000 == held


def _md5(p):
    return hashlib.md5(open(p, "rb").read()).hexdigest()


def _cli(args, out, env=None, check=True):
    r = subprocess.run([BIN, *args, "-o", str(out), "-p", "g", "-M", "3"], capture_output=True, text=True,
                       env=dict(os.environ, **(env or {})))
    if not check:
        return r
    assert r.returncode == 0, r.stderr
    return _md5(out / "g.reads"), _md5(out / "g.graph3"), open(out / "g.log").read()


def _fasta(path, reads):
    with open(path, "wb") as f:
        for i, s in enumerate(synth.to_list(reads)):
            f.write(b">r%d\n%s\n" % (i, bytes(s)))


def _gz_file(src, dst, level=6):
    dst.write_bytes(gz.stream(src.read_bytes(), level))
    return dst


@pytest.mark.parametrize("name", ["mixed", "cfg1", "f504"])
def test_cli_gzip_fastq_and_fasta(name, tmp_path):
    if name in long_datasets.LONG_DATASETS:
        reads, k = long_datasets.get(name)
    else:
        reads, k = datasets.get(name) if name in datasets.DATASETS else synth.config(name)
    fq, fa = tmp_path / "a.fastq", tmp_path / "a.fa"
    synth.write_fastq(str(fq), reads)
    _fasta(fa, reads)
    want = (GOLD[name]["reads_md5"], GOLD[name]["graph3_md5"]) if name in GOLD else _cli(["-f", str(fq), "-k", str(k)], tmp_path / "p")[:2]
    for src in (fq, fa):
        r, g, log = _cli(["-f", str(_gz_file(src, tmp_path / (src.name + ".gz"))), "-k", str(k)], tmp_path / ("o_" + src.name))
        assert (r, g) == want
        if name == "mixed":       # irregular records: the whole file goes to the sequential parser, as the plain text does
            assert "at text offset 0; the rest of the file continues on the sequential parser" in log
        else:
            assert "Records split on the device: yes; gzip text inflated on the device" in log


def test_cli_gzip_mate_files_of_unequal_length(tmp_path):
    reads, k = datasets.get("rep")
    lst = synth.to_list(reads)
    a, b = lst[0::2], lst[1::2][:-700]
    synth.write_fastq(str(tmp_path / "m1.fastq"), a)
    synth.write_fastq(str(tmp_path / "m2.fastq"), b)
    for m in ("m1", "m2"):
        _gz_file(tmp_path / f"{m}.fastq", tmp_path / f"{m}.fastq.gz")
    (tmp_path / "in.list").write_text(f"f1={tmp_path}/m1.fastq.gz\nf2={tmp_path}/m2.fastq.gz\n")
    kept = a[:min(len(a), len(b) + 1)] + b[:min(len(b), len(a))]
    synth.write_fastq(str(tmp_path / "kept.fastq"), kept)
    got = _cli(["-l", str(tmp_path / "in.list"), "-k", str(k)], tmp_path / "o", env={"SAGE2GPU_UPLOAD_PIECE_BYTES": "65536"})
    want = _cli(["-f", str(tmp_path / "kept.fastq"), "-k", str(k)], tmp_path / "w")
    assert got[:2] == want[:2] and "gzip text inflated on the device" in got[2]


@pytest.mark.parametrize("layout", ["replicated", "sharded"])
def test_cli_gzip_pieces_straddle_contexts(layout, tmp_path):
    reads, k = synth.config("cfg1")
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    z = _gz_file(fq, tmp_path / "a.fastq.gz")
    env = {"SAGE2GPU_UPLOAD_PIECE_BYTES": "65536", "SAGE2GPU_TABLE_LAYOUT": layout}
    for devs in ("0,0", "0,0,0"):
        r, g, log = _cli(["-f", str(z), "-k", str(k), "--devices", devs], tmp_path / ("o" + devs.replace(",", "_")), env=env)
        assert (r, g) == (GOLD["cfg1"]["reads_md5"], GOLD["cfg1"]["graph3_md5"]), devs
        assert "gzip text inflated on the device" in log


def test_cli_gzip_multiline_fasta_falls_back(tmp_path):
    reads, k = synth.config("cfg1")
    lst = synth.to_list(reads)
    half = len(lst) // 2
    regular = b"".join(b">r%d\n%s\n" % (i, s) for i, s in enumerate(lst[:half]))
    multi = b"".join(b">r%d\n%s\n%s\n" % (i, s[:60], s[60:]) for i, s in enumerate(lst[half:]))
    (tmp_path / "ml.fa.gz").write_bytes(gz.stream(regular + multi, 6))
    r, g, log = _cli(["-f", str(tmp_path / "ml.fa.gz"), "-k", str(k)], tmp_path / "o", env={"SAGE2GPU_UPLOAD_PIECE_BYTES": str(1 << 20)})
    assert (r, g) == (GOLD["cfg1"]["reads_md5"], GOLD["cfg1"]["graph3_md5"])
    assert "gzip text inflated on the device" in log and "not in the regular" in log


def test_cli_gzip_level0_larger_than_a_piece(tmp_path):
    reads, k = synth.config("cfg1")
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    z = _gz_file(fq, tmp_path / "a.fastq.gz", level=0)
    assert z.stat().st_size > 4 << 20
    r, g, log = _cli(["-f", str(z), "-k", str(k)], tmp_path / "o", env={"SAGE2GPU_UPLOAD_PIECE_BYTES": str(1 << 18)})
    assert (r, g) == (GOLD["cfg1"]["reads_md5"], GOLD["cfg1"]["graph3_md5"])
    assert "gzip text inflated on the device" in log and "sequential parser" not in log


def test_cli_corrupt_gzip_fails_loudly(tmp_path):
    reads, k = datasets.get("mixed")
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    good = gz.stream(fq.read_bytes(), 6)
    bad = bytearray(good)
    bad[-8] ^= 1
    (tmp_path / "bad.fastq.gz").write_bytes(bytes(bad))
    r = _cli(["-f", str(tmp_path / "bad.fastq.gz"), "-k", str(k)], tmp_path / "o", check=False)
    assert r.returncode != 0
    assert "compressed offset 0" in r.stderr and "FORMAT" in r.stderr
    assert not os.path.exists(tmp_path / "o" / "g.graph3")


def test_cli_gzip_cfg2_full_size(tmp_path):
    reads, k = synth.config("cfg2")
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    (tmp_path / "a.fastq.gz").write_bytes(gz.stream(fq.read_bytes(), 1))
    fq.unlink()
    r, g, log = _cli(["-f", str(tmp_path / "a.fastq.gz"), "-k", str(k)], tmp_path / "o")
    assert (r, g) == (BIG["cfg2"]["reads_md5"], BIG["cfg2"]["graph3_md5"])
    assert "gzip text inflated on the device" in log
