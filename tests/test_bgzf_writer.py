"""CPU checks of the BGZF writer the GPU tests use (tests/bgzf.py): every file it writes reads back through Python's gzip, its
members state their own sizes, and the host program's sequential parser (--parse-only) reads a BGZF file exactly as the plain
file."""
import gzip
import json
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import bgzf
from sage2_b200 import api, synth

BIN = os.path.join(os.path.dirname(api.LIB_PATH), "sage2gpu")

STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "fixed": zlib.Z_FIXED, "huffman": zlib.Z_HUFFMAN_ONLY, "rle": zlib.Z_RLE}


def _fastq(n=3000, seed=5):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        s = bytes(rng.choice(list(b"ACGT"), size=int(rng.integers(60, 200))).astype(np.uint8))
        out.append(b"@r%d\n%s\n+\n%s\n" % (i, s, b"I" * len(s)))
    return b"".join(out)


@pytest.mark.parametrize("level", [0, 1, 6, 9])
@pytest.mark.parametrize("strategy", sorted(STRATEGIES))
def test_members_read_back_through_gzip(level, strategy):
    text = _fastq()
    for sizes, sync in ((bgzf.MAX_TEXT, 0), ([1, 7, 4096, 65280, 333], 0), (20000, 3000)):
        blob = bgzf.write(text, sizes, level, STRATEGIES[strategy], sync)
        assert gzip.decompress(blob) == text
        mem = bgzf.members(blob)
        assert sum(s for _, s in mem) == len(blob)
        assert blob[mem[-1][0]:] == bgzf.EOF_MEMBER
        for off, size in mem:
            assert size <= 65536
            assert struct.unpack_from("<I", blob, off + size - 4)[0] <= bgzf.MAX_TEXT


def test_sync_flush_makes_several_blocks_and_empty_stored_blocks():
    d = bgzf.deflate(b"ACGT" * 5000, 6, zlib.Z_DEFAULT_STRATEGY, 1000)
    assert d.count(b"\x00\x00\xff\xff") >= 5        # LEN 0 / NLEN 0xFFFF of the empty stored blocks
    assert zlib.decompress(d, -15) == b"ACGT" * 5000


def test_parse_only_reads_bgzf_as_the_plain_file(tmp_path):
    if not os.path.exists(BIN):
        api.build_library()
    reads = [bytes(r) for r in synth.to_list(synth.config("cfg1")[0][:20000])]
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    bz = tmp_path / "a.fastq.gz"
    bz.write_bytes(bgzf.write(fq.read_bytes(), [65280, 1000, 17]))

    def run(p):
        r = subprocess.run([BIN, "-f", str(p), "-k", "20", "--parse-only"], capture_output=True, text=True, check=True)
        return json.loads(r.stdout)

    assert run(bz) == run(fq)
    assert run(fq)["reads"] == len(reads)
