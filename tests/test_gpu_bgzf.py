"""BGZF inflated on the device (sage2_b200/csrc/inflate.cu): sage2gpu_inflate_bgzf equals zlib byte for byte, a member that
breaks a DEFLATE / gzip rule gives SAGE2GPU_ERR_FORMAT naming it and leaves the context usable, and `sage2gpu` on BGZF input
writes the same files as on the plain text."""
import gzip
import hashlib
import json
import os
import subprocess
import zlib

import numpy as np
import pytest

import bgzf
import datasets
import long_datasets
from sage2_b200 import api, synth

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "golden.json")))
BIG = json.load(open(os.path.join(HERE, "golden", "golden_big.json")))
BIN = os.path.join(os.path.dirname(api.LIB_PATH), "sage2gpu")
STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "fixed": zlib.Z_FIXED, "huffman": zlib.Z_HUFFMAN_ONLY, "rle": zlib.Z_RLE}


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


class Bits:
    """DEFLATE bit writer: fields LSB first, Huffman codes MSB first"""
    def __init__(self):
        self.b = []

    def put(self, v, n):
        self.b += [(v >> i) & 1 for i in range(n)]

    def code(self, c, n):
        self.b += [(c >> i) & 1 for i in reversed(range(n))]

    def align(self):
        self.b += [0] * (-len(self.b) % 8)

    def raw(self, data):
        self.align()
        for x in data:
            self.put(x, 8)

    def bytes(self):
        self.align()
        return bytes(sum(self.b[i + j] << j for j in range(8)) for i in range(0, len(self.b), 8))


def _fixed_lit(bw, s):
    if s < 144:
        bw.code(0x30 + s, 8)
    elif s < 256:
        bw.code(0x190 + s - 144, 9)
    elif s < 280:
        bw.code(s - 256, 7)
    else:
        bw.code(0xC0 + s - 280, 8)


@pytest.mark.parametrize("kind", ["fastq", "fasta"])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
@pytest.mark.parametrize("strategy", sorted(STRATEGIES))
def test_inflate_equals_zlib(gpu, kind, level, strategy):
    text = _text(kind)
    for sizes, sync in ((bgzf.MAX_TEXT, 0), ([1, 2, 300, 65280, 4099], 0), (30000, 2500)):
        blob = bgzf.write(text, sizes, level, STRATEGIES[strategy], sync)
        got, _ = gpu.inflate_bgzf(blob)
        assert got == text, (sizes, sync)


def test_inflate_incompressible_runs_and_far_distances(gpu):
    rng = np.random.default_rng(1)
    rnd = rng.integers(0, 256, size=300_000).astype(np.uint8).tobytes()
    for level in (0, 6, 9):
        assert gpu.inflate_bgzf(bgzf.write(rnd, level=level))[0] == rnd
    runs = b"A" * 70000 + b"AC" * 9000 + b"ACGTTGCA" * 5000          # length-258 matches, distance 1 and short overlapping copies
    assert gpu.inflate_bgzf(bgzf.write(runs, level=9))[0] == runs
    # a distance of 32,768 (zlib's deflate never emits one): 32 KiB stored, then a length-258 match at distance 32768
    head = rng.integers(0, 256, size=32768).astype(np.uint8).tobytes()
    bw = Bits()
    bw.put(0, 1); bw.put(0, 2); bw.align(); bw.put(32768, 16); bw.put(32768 ^ 0xFFFF, 16); bw.raw(head)
    bw.put(1, 1); bw.put(1, 2)
    for _ in range(3):
        _fixed_lit(bw, 285); bw.code(29, 5); bw.put(8191, 13)
    _fixed_lit(bw, 256)
    data = bw.bytes()
    want = head + (head * 2)[:3 * 258]
    assert zlib.decompress(data, -15) == want
    assert gpu.inflate_bgzf(bgzf.member(want, data=data) + bgzf.EOF_MEMBER)[0] == want


def _corrupt_members():
    """name -> a member that breaks one rule"""
    t = _text("fastq", 300, seed=3)
    good = bgzf.deflate(t)
    out = {"crc": bgzf.member(t, crc=zlib.crc32(t) ^ 0x10), "isize": bgzf.member(t, isize=len(t) + 1),
           "isize_short": bgzf.member(t, isize=len(t) - 1)}
    bw = Bits()                                   # dynamic block: 19 code-length codes of length 1 (over-subscribed)
    bw.put(1, 1); bw.put(2, 2); bw.put(0, 5); bw.put(0, 5); bw.put(15, 4)
    for _ in range(19):
        bw.put(1, 3)
    out["oversubscribed"] = bgzf.member(b"x" * 10, data=bw.bytes() + b"\0" * 8)
    bw = Bits()                                   # fixed block: a match of distance 1 as the first symbol
    bw.put(1, 1); bw.put(1, 2); _fixed_lit(bw, 257); bw.code(0, 5); _fixed_lit(bw, 256)
    out["distance"] = bgzf.member(b"xxx", data=bw.bytes())
    out["block_type_3"] = bgzf.member(b"x", data=b"\x07\x00")
    out["stored_nlen"] = bgzf.member(b"hello", data=b"\x01\x05\x00\x05\x00hello")
    out["truncated"] = bgzf.member(t, data=good[:-6])
    return out


@pytest.mark.parametrize("case", ["crc", "isize", "isize_short", "oversubscribed", "distance", "block_type_3", "stored_nlen", "truncated",
                                  "bsize_past_end"])
def test_corrupt_member_names_it_and_context_stays_usable(gpu, case):
    recs = _text("fastq", 900, seed=4)
    ok = [bgzf.member(x) for x in bgzf.split(recs, 20000)]
    if case == "bsize_past_end":
        blob, bad = b"".join(ok)[:-5], len(ok) - 1
    else:
        blob, bad = b"".join(ok[:2]) + _corrupt_members()[case] + b"".join(ok[2:]), 2
    with pytest.raises(api.Sage2GpuError) as e:
        gpu.inflate_bgzf(blob, text_capacity=1 << 22)
    assert e.value.code == api.ERR_FORMAT and e.value.bad_member == bad, str(e.value)
    gpu.load_begin(20)
    first = gpu.load_append_bgzf(b"", b"".join(ok[:1]), False)
    n0 = gpu.load_count()
    assert n0 == first["n_records"] > 0
    with pytest.raises(api.Sage2GpuError) as e:
        gpu.load_append_bgzf(first["rest"], blob, True, marker=first["marker"])
    assert e.value.code == api.ERR_FORMAT and e.value.bad_member == bad
    assert f"member {bad} " in str(e.value)
    assert gpu.load_count() == n0                 # nothing appended
    r = gpu.load_append_bgzf(first["rest"], b"".join(ok[1:]) + bgzf.EOF_MEMBER, True, marker=first["marker"])
    assert n0 + r["n_records"] == gpu.load_count() == 900 and r["rest"] == b""


def test_pieces_carry_the_rest_between_contexts(gpu):
    """A piece's unfinished record comes back to the host and goes in front of the next piece, on another context."""
    recs = _text("fastq", 2000, seed=8)
    mem = [bgzf.member(x) for x in bgzf.split(recs, [777, 5000, 1])] + [bgzf.EOF_MEMBER]
    other = api.Sage2Gpu(0)
    try:
        ctx = [gpu, other]
        for g in ctx:
            g.load_begin(20)
        rest, marker, total = b"", 0, 0
        for i in range(0, len(mem), 7):
            r = ctx[(i // 7) % 2].load_append_bgzf(rest, b"".join(mem[i:i + 7]), i + 7 >= len(mem), marker=marker)
            rest, marker, total = r["rest"], r["marker"], total + r["n_records"]
        assert total == 2000 == gpu.load_count() + other.load_count() and rest == b""
    finally:
        other.close()


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


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


def _bgzf_file(src, dst, **kw):
    dst.write_bytes(bgzf.write(src.read_bytes(), **kw))
    return dst


@pytest.mark.parametrize("name", ["mixed", "cfg1", "f504"])
def test_cli_bgzf_fastq_and_fasta(name, tmp_path):
    if name in long_datasets.LONG_DATASETS:
        reads, k = long_datasets.get(name)
    else:
        reads, k = datasets.get(name) if name in datasets.DATASETS else synth.config(name)
    fq, fa = tmp_path / "a.fastq", tmp_path / "a.fa"
    synth.write_fastq(str(fq), reads)
    _fasta(fa, reads)
    want = (GOLD[name]["reads_md5"], GOLD[name]["graph3_md5"]) if name in GOLD else _cli(["-f", str(fq), "-k", str(k)], tmp_path / "p")[:2]
    for src in (fq, fa):
        bz = _bgzf_file(src, tmp_path / (src.name + ".gz"), sizes=[65280, 3001, 40000])
        r, g, log = _cli(["-f", str(bz), "-k", str(k)], tmp_path / ("o_" + src.name))
        assert (r, g) == want
        if name == "mixed":       # irregular records: the whole file goes to the sequential parser, as the plain text does
            assert "at compressed offset 0; the rest of the file continues on the sequential parser" in log
        else:
            assert "BGZF text inflated on the device" in log and "sequential parser (host zlib)" not in log


def test_cli_bgzf_mate_files_of_unequal_length(tmp_path):
    reads, k = datasets.get("rep")
    lst = synth.to_list(reads)
    a, b = lst[0::2], lst[1::2][:-700]
    synth.write_fastq(str(tmp_path / "m1.fastq"), a)
    synth.write_fastq(str(tmp_path / "m2.fastq"), b)
    for m in ("m1", "m2"):
        _bgzf_file(tmp_path / f"{m}.fastq", tmp_path / f"{m}.fastq.gz", sizes=9000)
    (tmp_path / "in.list").write_text(f"f1={tmp_path}/m1.fastq.gz\nf2={tmp_path}/m2.fastq.gz\n")
    kept = a[:min(len(a), len(b) + 1)] + b[:min(len(b), len(a))]
    synth.write_fastq(str(tmp_path / "kept.fastq"), kept)
    got = _cli(["-l", str(tmp_path / "in.list"), "-k", str(k)], tmp_path / "o", env={"SAGE2GPU_UPLOAD_PIECE_BYTES": "65536"})
    want = _cli(["-f", str(tmp_path / "kept.fastq"), "-k", str(k)], tmp_path / "w")
    assert got[:2] == want[:2] and "BGZF text inflated on the device" in got[2]


@pytest.mark.parametrize("layout", ["replicated", "sharded"])
def test_cli_bgzf_pieces_straddle_contexts(layout, tmp_path):
    reads, k = datasets.get("mixed")
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    bz = _bgzf_file(fq, tmp_path / "a.fastq.gz", sizes=[10007, 65280, 333])
    env = {"SAGE2GPU_UPLOAD_PIECE_BYTES": "65536", "SAGE2GPU_TABLE_LAYOUT": layout}
    for devs in ("0,0", "0,0,0"):
        r, g, log = _cli(["-f", str(bz), "-k", str(k), "--devices", devs], tmp_path / ("o" + devs.replace(",", "_")), env=env)
        assert (r, g) == (GOLD["mixed"]["reads_md5"], GOLD["mixed"]["graph3_md5"]), devs
        assert "BGZF text inflated on the device" in log


def test_cli_bgzf_falls_back_mid_file(tmp_path):
    reads, k = synth.config("cfg1")
    lst = synth.to_list(reads)
    gold = (GOLD["cfg1"]["reads_md5"], GOLD["cfg1"]["graph3_md5"])
    half = len(lst) // 2
    regular = b"".join(b">r%d\n%s\n" % (i, s) for i, s in enumerate(lst[:half]))
    multi = b"".join(b">r%d\n%s\n%s\n" % (i, s[:60], s[60:]) for i, s in enumerate(lst[half:]))
    # later members hold multi-line FASTA: the device splits the first pieces, the host parser the rest
    (tmp_path / "ml.fa.gz").write_bytes(bgzf.write(regular + multi))
    env = {"SAGE2GPU_UPLOAD_PIECE_BYTES": str(1 << 20)}
    r, g, log = _cli(["-f", str(tmp_path / "ml.fa.gz"), "-k", str(k)], tmp_path / "o1", env=env)
    assert (r, g) == gold
    assert "BGZF text inflated on the device" in log and "not in the regular" in log
    # later members are ordinary gzip members without the BC field
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    n_members = len(bgzf.split(fq.read_bytes()))
    (tmp_path / "nobc.fastq.gz").write_bytes(bgzf.write(fq.read_bytes(), plain_from=n_members * 2 // 3))
    r, g, log = _cli(["-f", str(tmp_path / "nobc.fastq.gz"), "-k", str(k)], tmp_path / "o2", env=env)
    assert (r, g) == gold
    assert "BGZF text inflated on the device" in log and "without a BC field" in log


@pytest.mark.parametrize("case", ["crc", "distance", "truncated"])
def test_cli_corrupt_member_fails_loudly(case, tmp_path):
    reads, k = datasets.get("mixed")
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    ok = [bgzf.member(x) for x in bgzf.split(fq.read_bytes(), 20000)]
    off = sum(len(m) for m in ok[:3])
    (tmp_path / "bad.fastq.gz").write_bytes(b"".join(ok[:3]) + _corrupt_members()[case] + b"".join(ok[3:]) + bgzf.EOF_MEMBER)
    r = _cli(["-f", str(tmp_path / "bad.fastq.gz"), "-k", str(k)], tmp_path / "o", check=False)
    assert r.returncode != 0
    assert f"compressed offset {off}" in r.stderr and "FORMAT" in r.stderr
    assert not os.path.exists(tmp_path / "o" / "g.graph3")


def test_cli_bgzf_cfg2_full_size(tmp_path):
    reads, k = synth.config("cfg2")
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    text = fq.read_bytes()
    fq.unlink()
    (tmp_path / "a.fastq.gz").write_bytes(b"".join(bgzf.member(x, 1) for x in bgzf.split(text)) + bgzf.EOF_MEMBER)
    r, g, log = _cli(["-f", str(tmp_path / "a.fastq.gz"), "-k", str(k)], tmp_path / "o")
    assert (r, g) == (BIG["cfg2"]["reads_md5"], BIG["cfg2"]["graph3_md5"])
    assert "BGZF text inflated on the device" in log
