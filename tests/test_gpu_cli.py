"""GPU tests of the C++ host program: `sage2gpu -f <fastq> -k K -M 3` must write the same bytes as the
unmodified reference's `SAGE2 -s -M 3` (md5s in tests/golden/golden.json, fixtures for `mixed`), and the
reference's own steps 4-7 continued from our files must give byte-identical contig / scaffold FASTA."""
import gzip
import hashlib
import json
import os
import subprocess

import pytest

import datasets
from oracle import oracle
from sage2_b200 import api, synth

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "golden.json")))
BIN = os.path.join(os.path.dirname(api.LIB_PATH), "sage2gpu")


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


def _get(name):
    return datasets.get(name) if name in datasets.DATASETS else synth.config(name)


@pytest.mark.parametrize("name", ["mixed", "rep", "varlen_err", "k70", "cfg1", "cfg4mini"])
def test_cli_files_byte_identical_to_reference(name, tmp_path):
    reads, k = _get(name)
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    out = tmp_path / "out"
    subprocess.run([BIN, "-f", str(fq), "-k", str(k), "-o", str(out), "-p", "g", "-M", "3"], check=True)
    assert _md5(out / "g.reads") == GOLD[name]["reads_md5"]
    assert _md5(out / "g.graph3") == GOLD[name]["graph3_md5"]
    if name == "mixed":      # the complete files the reference wrote are committed fixtures
        for ext in (".reads", ".graph3"):
            want = gzip.open(os.path.join(HERE, "golden", "mixed" + ext + ".gz"), "rb").read()
            assert open(out / ("g" + ext), "rb").read() == want
    log = open(out / "g.log").read()
    assert f"Number of unique reads: {GOLD[name]['unique_reads']}" in log


def test_cli_list_input_two_mate_files(tmp_path):
    reads, k = _get("rep")
    lst = synth.to_list(reads)
    for mate in (0, 1):
        synth.write_fastq(str(tmp_path / f"m{mate + 1}.fastq"), lst[mate::2])
    (tmp_path / "in.list").write_text(f"f1={tmp_path}/m1.fastq\nf2={tmp_path}/m2.fastq\n")
    out = tmp_path / "out"
    subprocess.run([BIN, "-l", str(tmp_path / "in.list"), "-k", str(k), "-o", str(out), "-p", "g", "-M", "3"], check=True)
    assert _md5(out / "g.reads") == GOLD["rep"]["reads_md5"]
    assert _md5(out / "g.graph3") == GOLD["rep"]["graph3_md5"]


@pytest.mark.skipif(not os.access(oracle.REF_SAGE2, os.X_OK), reason="the compiled reference did not travel (oracle/_ref/SAGE2)")
def test_downstream_fasta_identical_through_reference_steps_4_to_7(tmp_path):
    """north_star: byte-identical contig and scaffold FASTA downstream.  Both arms restart at step 4 (the
    reference's restart path differs from its straight-through path, SURVEY.md section 5)."""
    reads, k = _get("cfg4mini")
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    ours, ref = tmp_path / "ours", tmp_path / "ref"
    env = dict(os.environ, OMP_NUM_THREADS="1")
    subprocess.run([BIN, "-f", str(fq), "-k", str(k), "-o", str(ours), "-p", "g", "--reference", oracle.REF_SAGE2], check=True, env=env)
    subprocess.run([oracle.REF_SAGE2, "-f", str(fq), "-k", str(k), "-o", str(ref), "-p", "g", "-s", "-M", "3"], check=True, env=env,
                   stdout=subprocess.DEVNULL)
    subprocess.run([oracle.REF_SAGE2, "-f", str(fq), "-k", str(k), "-o", str(ref), "-p", "g", "-m", "4"], check=True, env=env,
                   stdout=subprocess.DEVNULL)
    for ext in (".reads", ".graph3"):
        assert _md5(ours / ("g" + ext)) == _md5(ref / ("g" + ext))
    fastas = sorted(f for f in os.listdir(ref) if f.endswith(".fasta"))
    assert fastas, "the reference wrote no FASTA"
    for f in fastas:
        assert open(ours / f, "rb").read() == open(ref / f, "rb").read(), f


def _run_cli(args, out):
    subprocess.run([BIN, *args, "-o", str(out), "-p", "g", "-M", "3"], check=True)
    return _md5(out / "g.reads"), _md5(out / "g.graph3"), open(out / "g.log").read()


def test_device_record_splitting_and_sequential_fallback(tmp_path):
    """The same reads as regular FASTQ (records split on the device), 2-line FASTA, gzip, multi-line FASTA
    (sequential parser) and a FASTQ whose irregular record sits in a later 32 MB piece (device first, then the
    sequential parser from that point on): identical files every time."""
    reads, k = _get("cfg1")                       # 400,000 reads, 88 MB of FASTQ: three pieces
    gold = (GOLD["cfg1"]["reads_md5"], GOLD["cfg1"]["graph3_md5"])
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    r, g, log = _run_cli(["-f", str(fq), "-k", str(k)], tmp_path / "o1")
    assert (r, g) == gold and "Records split on the device: yes" in log

    lst = synth.to_list(reads)
    fa = tmp_path / "a.fa"
    with open(fa, "wb") as f:
        for i, s in enumerate(lst):
            f.write(b">r%d\n%s\n" % (i, s))
    r, g, log = _run_cli(["-f", str(fa), "-k", str(k)], tmp_path / "o2")
    assert (r, g) == gold and "Records split on the device: yes" in log

    gz = tmp_path / "a.fastq.gz"
    with gzip.open(gz, "wb", compresslevel=1) as f:
        f.write(open(fq, "rb").read())
    r, g, log = _run_cli(["-f", str(gz), "-k", str(k)], tmp_path / "o3")
    assert (r, g) == gold and "Records split on the device: yes" in log

    ml = tmp_path / "multi.fa"
    with open(ml, "wb") as f:
        for i, s in enumerate(lst):
            f.write(b">r%d\n%s\n%s\n" % (i, s[:60], s[60:]))
    r, g, log = _run_cli(["-f", str(ml), "-k", str(k)], tmp_path / "o4")
    assert (r, g) == gold and "Records split on the device: no" in log

    mixed = tmp_path / "mixed.fastq"
    with open(mixed, "wb") as f:
        for i, s in enumerate(lst):
            if i == 250_000:          # ~55 MB into the file: a record with its sequence and quality on two lines each
                f.write(b"@r%d\n%s\n%s\n+\n%s\n%s\n" % (i, s[:50], s[50:], b"I" * 50, b"I" * (len(s) - 50)))
            else:
                f.write(b"@r%d\n%s\n+\n%s\n" % (i, s, b"I" * len(s)))
    r, g, log = _run_cli(["-f", str(mixed), "-k", str(k)], tmp_path / "o5")
    assert (r, g) == gold and "Records split on the device: yes" in log


def test_two_mate_files_of_unequal_length(tmp_path):
    """The reference alternates the mate files and stops when one ends (inputReader.cpp:26-49)."""
    reads, k = _get("rep")
    lst = synth.to_list(reads)
    m1, m2 = lst[0::2], lst[1::2]
    for name, (a, b) in {"long1": (m1, m2[:-700]), "long2": (m1[:-500], m2)}.items():
        synth.write_fastq(str(tmp_path / f"{name}_1.fastq"), a)
        synth.write_fastq(str(tmp_path / f"{name}_2.fastq"), b)
        (tmp_path / f"{name}.list").write_text(f"f1={tmp_path}/{name}_1.fastq\nf2={tmp_path}/{name}_2.fastq\n")
        n1, n2 = len(a), len(b)
        kept = a[:min(n1, n2 + 1)] + b[:min(n2, n1)]
        synth.write_fastq(str(tmp_path / f"{name}_expected.fastq"), kept)
        got = _run_cli(["-l", str(tmp_path / f"{name}.list"), "-k", str(k)], tmp_path / f"{name}_o")
        want = _run_cli(["-f", str(tmp_path / f"{name}_expected.fastq"), "-k", str(k)], tmp_path / f"{name}_w")
        assert got[:2] == want[:2]
        assert f"Good reads: {len(kept)}" in got[2].replace(",", "")


def _devices_args():
    import torch
    out = [("0,0", "two contexts on one GPU"), ("0,0,0", "three contexts on one GPU")]
    if torch.cuda.device_count() >= 2:
        out.append(("0,1", "two GPUs"))
    if torch.cuda.device_count() >= 4:
        out.append(("0-3", "four GPUs"))
    return out


@pytest.mark.parametrize("name", ["mixed", "rep", "varlen_err", "hicopy", "cfg1"])
def test_cli_several_devices_byte_identical_to_reference(name, tmp_path):
    """`sage2gpu --devices LIST`: ONE process, one context per listed device, every stage partitioned, peer copies between
    the stages (no NCCL, no Python).  Same bytes as the unmodified reference, from the first and from the last context."""
    reads, k = _get(name)
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    for devs, _ in _devices_args():
        out = tmp_path / ("out_" + devs.replace(",", "_"))
        subprocess.run([BIN, "-f", str(fq), "-k", str(k), "-o", str(out), "-p", "g", "-M", "3", "--devices", devs], check=True)
        assert _md5(out / "g.reads") == GOLD[name]["reads_md5"], devs
        assert _md5(out / "g.graph3") == GOLD[name]["graph3_md5"], devs
        log = open(out / "g.log").read()
        assert f"Number of unique reads: {GOLD[name]['unique_reads']}" in log
