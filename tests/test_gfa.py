"""CPU tests of tests/gfa.py, the reference writer and validator of the GFA that sage2gpu_write_gfa writes on the device.

The validator checks every L line as an exact sequence overlap in its stated orientations, so the writer passing it on the
reference's own `.reads` / `.graph3` pins the mapping of SAGE2's edge types to GFA orientations."""
import gzip
import itertools
import os
import subprocess

import pytest

import datasets
import gfa
import long_datasets
from oracle import oracle
from sage2_b200 import api, synth

HERE = os.path.dirname(os.path.abspath(__file__))


def _mixed_gfa() -> bytes:
    return gfa.write_gfa_bytes(gzip.open(os.path.join(HERE, "golden", "mixed.reads.gz")),
                               gzip.open(os.path.join(HERE, "golden", "mixed.graph3.gz")))


def test_reference_mixed_files_give_a_valid_gfa():
    """The reference's committed output for `mixed` (k = 45): every one of its 15,254 edges is an exact overlap."""
    text = _mixed_gfa()
    assert gfa.validate(text, 45) == {"segments": 15409, "links": 15254}
    lines = text.split(b"\n")
    assert lines[0] == b"H\tVN:Z:1.0" and lines[1].startswith(b"S\t1\t") and lines[-1] == b""
    # two edges of different types between one pair of reads are two L lines
    pairs = [tuple(l.split(b"\t")[1:4:2]) for l in lines if l.startswith(b"L\t")]
    assert len(set(pairs)) == 15254 - 125


def test_every_other_type_mapping_is_rejected():
    """Only the documented table makes the reference's edges exact overlaps: each of the 23 other assignments of the four
    orientation pairs to the four types fails the validator."""
    orig = dict(gfa.TYPE_ORIENTATION)
    pairs = list(orig.values())
    rejected = 0
    try:
        for perm in itertools.permutations(pairs):
            table = dict(zip(sorted(orig), perm))
            if table == orig:
                continue
            gfa.TYPE_ORIENTATION.clear()
            gfa.TYPE_ORIENTATION.update(table)
            with pytest.raises(gfa.GfaError):
                gfa.validate(_mixed_gfa(), 45)
            rejected += 1
    finally:
        gfa.TYPE_ORIENTATION.clear()
        gfa.TYPE_ORIENTATION.update(orig)
    assert rejected == 23


def _oracle_gfa(reads, k, tmp_path) -> bytes:
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    o.write_reads(str(tmp_path / "o.reads"))
    o.write_graph3(str(tmp_path / "o.graph3"))
    text = gfa.write_gfa_bytes(str(tmp_path / "o.reads"), str(tmp_path / "o.graph3"))
    assert gfa.validate(text, k) == {"segments": o.U, "links": o.n_edges}
    return text


@pytest.mark.parametrize("name", list(datasets.DATASETS))
def test_oracle_files_give_a_valid_gfa(name, tmp_path):
    reads, k = datasets.get(name)
    text = _oracle_gfa(reads, k, tmp_path)
    if name == "empty":
        assert text == gfa.HEADER


@pytest.mark.parametrize("name", list(long_datasets.LONG_DATASETS))
def test_oracle_files_of_long_reads_give_a_valid_gfa(name, tmp_path):
    reads, k = long_datasets.get(name)
    _oracle_gfa(reads, k, tmp_path)


def _first_link(text: bytes):
    lines = text.split(b"\n")
    i = next(j for j, l in enumerate(lines) if l.startswith(b"L\t"))
    return lines, i, lines[i].split(b"\t")


def test_validator_rejects_a_flipped_orientation():
    lines, i, f = _first_link(_mixed_gfa())
    f[4] = b"-" if f[4] == b"+" else b"+"
    lines[i] = b"\t".join(f)
    with pytest.raises(gfa.GfaError, match="not an exact overlap"):
        gfa.validate(b"\n".join(lines), 45)


def test_validator_rejects_an_overlap_off_by_one():
    for delta in (1, -1):
        lines, i, f = _first_link(_mixed_gfa())
        f[5] = b"%dM" % (int(f[5][:-1]) + delta)
        lines[i] = b"\t".join(f)
        with pytest.raises(gfa.GfaError, match="not an exact overlap"):
            gfa.validate(b"\n".join(lines), 45)


def test_validator_rejects_a_link_to_a_missing_segment():
    lines, i, f = _first_link(_mixed_gfa())
    f[3] = b"15410"
    lines[i] = b"\t".join(f)
    with pytest.raises(gfa.GfaError, match="missing segment"):
        gfa.validate(b"\n".join(lines), 45)


def test_validator_rejects_broken_segments():
    lines = _mixed_gfa().split(b"\n")
    for bad in (lines[1].replace(b"\t1\t", b"\t2\t", 1),            # ids not 1..U
                lines[1].replace(b"LN:i:100", b"LN:i:99"),          # LN != sequence length
                lines[1].replace(b"AAAA", b"AANA", 1)):             # not over ACGT
        with pytest.raises(gfa.GfaError):
            gfa.validate(b"\n".join([lines[0], bad] + lines[2:]), 45)
    with pytest.raises(gfa.GfaError, match="header"):
        gfa.validate(b"\n".join(lines[1:]), 45)


@pytest.mark.parametrize("steps", [["-M", "2"], ["-M", "1"], ["-m", "4"], ["-m", "5", "-M", "7"]])
def test_cli_gfa_without_step_3_is_refused_before_any_work(steps, tmp_path):
    """`sage2gpu --gfa` writes the graph of step 3: with -M < 3 or -m >= 4 it exits non-zero at once -- no device is opened
    (so this runs without one), no output directory is made, no file is written."""
    binary = os.path.join(os.path.dirname(api.LIB_PATH), "sage2gpu")
    if not os.path.exists(binary):
        api.build_library()
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), datasets.get("single")[0])
    out = tmp_path / "out"
    p = subprocess.run([binary, "-f", str(fq), "-k", "40", "-o", str(out), "-p", "g", "--gfa", *steps],
                       capture_output=True, text=True)
    assert p.returncode != 0
    assert "--gfa" in p.stderr
    assert not out.exists()
