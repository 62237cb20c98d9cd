"""GPU tests of the restart from a saved `.reads` file (ReadLoader::loadReadsFromFile, readLoader.cpp:289; `sage2gpu -m 2 / -m 3`).

The file the reference's saveReadsInFile writes (here the oracle's, or the reference's own for `mixed`) is parsed and checked on
the device; steps 2-3 from it must give the bytes a straight run gives.  Every rule of the grammar broken once must fail with
SAGE2GPU_ERR_FORMAT naming the right line, through the C ABI and through the host program."""
import gzip
import hashlib
import json
import os
import re
import subprocess

import numpy as np
import pytest

import datasets
import long_datasets
from oracle import oracle
from sage2_b200 import api, synth
from test_gpu_cli import BIN, _devices_args
from test_gpu_read_organisation import CASES

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "golden.json")))
GOLD_BIG = json.load(open(os.path.join(HERE, "golden", "golden_big.json")))
DEVICES = [d for d, _ in _devices_args()]
NO_INPUT = "/nonexistent/input.fastq"        # -f stays required; a restart must not open it


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


def _get(name):
    return datasets.get(name) if name in datasets.DATASETS else synth.config(name)


def _oracle_files(reads, k, d, prefix="o"):
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    o.write_reads(str(d / f"{prefix}.reads"))
    o.write_graph3(str(d / f"{prefix}.graph3"))
    return o


def _restart(path, k, out_dir, tag="g"):
    """load_saved_reads -> table -> graph; returns the context and the paths of its two files."""
    gpu = api.Sage2Gpu(0)
    gpu.load_saved_reads(str(path), k)
    gpu.build_hash_table()
    gpu.build_overlap_graph()
    gpu.write_reads(str(out_dir / f"{tag}.reads"))
    gpu.write_graph3(str(out_dir / f"{tag}.graph3"))
    return gpu, out_dir / f"{tag}.reads", out_dir / f"{tag}.graph3"


def _cli(args, out, env=None, check=True):
    e = dict(os.environ, **(env or {}))
    p = subprocess.run([BIN, *args, "-o", str(out), "-M", "3"], env=e, capture_output=True, text=True)
    if check:
        assert p.returncode == 0, p.stderr
    return p


# ---- 1. the C ABI on every data set --------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", list(datasets.DATASETS))
def test_api_restart_equals_oracle(name, tmp_path, monkeypatch):
    reads, k = datasets.get(name)
    o = _oracle_files(reads, k, tmp_path)
    b, off = synth.concat(reads)
    straight = api.Sage2Gpu(0)
    straight.run_steps123(b, off, k)
    want_digest = straight.digest()
    for build in ("bucketed", "direct"):
        monkeypatch.setenv("SAGE2GPU_TABLE_BUILD", build)
        for fast in (0, 1):
            gpu = api.Sage2Gpu(0)
            gpu.set_option("fast_scan", fast)
            gpu.load_saved_reads(str(tmp_path / "o.reads"), k)
            c = gpu.counters()
            assert (c["unique_reads"], c["good_reads"], c["total_reads"], c["avg_len"]) == (o.U, o.N, o.N, o.avg_len), (build, fast)
            gpu.build_hash_table()
            gpu.build_overlap_graph()
            tag = f"{build}{fast}"
            gpu.write_reads(str(tmp_path / f"{tag}.reads"))
            gpu.write_graph3(str(tmp_path / f"{tag}.graph3"))
            assert open(tmp_path / f"{tag}.reads", "rb").read() == open(tmp_path / "o.reads", "rb").read(), (build, fast)
            assert open(tmp_path / f"{tag}.graph3", "rb").read() == open(tmp_path / "o.graph3", "rb").read(), (build, fast)
            assert gpu.digest() == want_digest, (build, fast)
            gpu.close()


def test_read_loader_load_reads_from_file(tmp_path):
    reads, k = datasets.get("rep")
    o = _oracle_files(reads, k, tmp_path)
    loader = api.ReadLoader(k)
    loader.loadReadsFromFile(str(tmp_path / "o.reads"))
    assert (loader.numberOfReads, loader.numberOfUniqueReads, loader.averageReadLength) == (o.N, o.U, o.avg_len)
    assert loader.totalBP == int(np.sum(o.frequency[1:].astype(np.int64) * o.length[1:]))
    table = api.HashTable(k, loader)
    table.hashPrefixesAndSuffix()
    graph = api.EconomyGraph(k, table)
    graph.buildInitialOverlapGraph()
    graph.saveOverlapGraphInFile(str(tmp_path / "g.graph3"))
    assert _md5(tmp_path / "g.graph3") == _md5(tmp_path / "o.graph3")


def test_slices_over_three_contexts_equal_one(tmp_path):
    """The slice calls by hand: three contexts parse a third of the body each, pack at the common stride, all-gather; the
    order check then runs over the complete reads."""
    import torch
    reads, k = long_datasets.get("short_in_wide")
    _oracle_files(reads, k, tmp_path)
    path = str(tmp_path / "o.reads")
    world = 3
    gpus = [api.Sage2Gpu(0) for _ in range(world)]
    U, body = gpus[0].saved_reads_info(path)
    sl = [g.saved_reads_slice(path, k, body * r // world, body * (r + 1) // world) for r, g in enumerate(gpus)]
    assert sum(s["n_lines"] for s in sl) == U and min(s["n_lines"] for s in sl) > 0
    ml = max(s["max_read_length"] for s in sl)
    packs = [g.saved_reads_pack(r, world, ml) for r, g in enumerate(gpus)]
    uloc = [p["unique_local"] for p in packs]
    lay = [g.reads_gather_layout(uloc) for g in gpus]
    from test_gpu_cli_devices import _gather_blocks
    _gather_blocks([x["records"] for x in lay], uloc, lay[0]["stride"])
    _gather_blocks([x["lengths"] for x in lay], uloc, 1, "<i2")
    _gather_blocks([x["frequencies"] for x in lay], uloc, 1, "<i2")
    torch.cuda.synchronize()
    good, bp = sum(p["good_reads"] for p in packs), sum(p["total_bp"] for p in packs)
    for g in gpus:
        g.reads_gather_finish()
        g.saved_reads_finish(U, good, bp)
        g.build_hash_table()
        g.build_overlap_graph()
        g.write_graph3(str(tmp_path / "s.graph3"))
        assert _md5(tmp_path / "s.graph3") == _md5(tmp_path / "o.graph3")


# ---- 2. the reference's own file ------------------------------------------------------------------------------------------

def test_reference_reads_file_gives_reference_graph(tmp_path):
    out = tmp_path / "out"
    out.mkdir()
    (out / "g.reads").write_bytes(gzip.open(os.path.join(HERE, "golden", "mixed.reads.gz"), "rb").read())
    _cli(["-f", NO_INPUT, "-k", str(GOLD["mixed"]["k"]), "-p", "g", "-m", "2"], out)
    assert (out / "g.graph3").read_bytes() == gzip.open(os.path.join(HERE, "golden", "mixed.graph3.gz"), "rb").read()


# ---- 3. the host program --------------------------------------------------------------------------------------------------

def _golden_reads(name, d):
    """<d>/g.reads with the reference's bytes (the straight GPU run writes them; checked against golden.json)."""
    reads, k = _get(name)
    b, off = synth.concat(reads)
    gpu = api.Sage2Gpu(0)
    gpu.load_reads(b, off, k)
    d.mkdir(exist_ok=True)
    gpu.write_reads(str(d / "g.reads"))
    gpu.close()
    assert _md5(d / "g.reads") == GOLD[name]["reads_md5"]
    return reads, k


@pytest.mark.parametrize("name", ["mixed", "rep", "varlen_err", "hicopy", "cfg1"])
def test_cli_restart_byte_identical_to_reference(name, tmp_path):
    out = tmp_path / "out"
    reads, k = _golden_reads(name, out)
    for step in ("2", "3"):
        p = _cli(["-f", NO_INPUT, "-k", str(k), "-p", "g", "-m", step], out)
        assert _md5(out / "g.graph3") == GOLD[name]["graph3_md5"], step
        assert _md5(out / "g.reads") == GOLD[name]["reads_md5"], step
        log = open(out / "g.log").read()
        assert f"Restart at step {step}: the reads are loaded from {out}/g.reads" in log
        assert f"Number of unique reads: {GOLD[name]['unique_reads']}" in log
        assert "g.reads is the file this restart loaded: not rewritten" in log
        assert ("-m 3 runs as -m 2" in log) == (step == "3")
        (out / "g.graph3").unlink()
    # another prefix continues from g.reads and writes its own copy of it
    _cli(["-f", NO_INPUT, "-k", str(k), "-p", "other", "-i", "g", "-m", "2"], out)
    assert (out / "other.reads").read_bytes() == (out / "g.reads").read_bytes()
    assert _md5(out / "other.graph3") == GOLD[name]["graph3_md5"]
    if name == "mixed":      # without a .reads file: step 1 from the input files
        fq = tmp_path / "in.fastq"
        synth.write_fastq(str(fq), reads)
        fresh = tmp_path / "fresh"
        _cli(["-f", str(fq), "-k", str(k), "-p", "g", "-m", "2"], fresh)
        assert _md5(fresh / "g.reads") == GOLD[name]["reads_md5"] and _md5(fresh / "g.graph3") == GOLD[name]["graph3_md5"]
        log = open(fresh / "g.log").read()
        assert f"NOTE: {fresh}/g.reads does not exist: -m 2 runs step 1 from the input files" in log
        assert "Restart at step" not in log


# ---- 4. k sweep -------------------------------------------------------------------------------------------------------------

def test_k_sweep_from_one_reads_file(tmp_path):
    """Fixed-length reads organised once at k = 50, restarted at k = 63: the oracle's straight run at k = 63.  A restart at
    k >= the read length fails and writes no .graph3."""
    reads, _ = datasets.get("clean")        # 100-base reads
    _oracle_files(reads, 50, tmp_path, "k50")
    _oracle_files(reads, 63, tmp_path, "k63")
    _, r, g = _restart(tmp_path / "k50.reads", 63, tmp_path)
    assert g.read_bytes() == (tmp_path / "k63.graph3").read_bytes()
    assert r.read_bytes() == (tmp_path / "k50.reads").read_bytes()
    gpu = api.Sage2Gpu(0)
    with pytest.raises(api.Sage2GpuError) as e:
        gpu.load_saved_reads(str(tmp_path / "k50.reads"), 100)
    assert e.value.code == api.ERR_FORMAT and "line 2: the read is not longer than -k (100)" in str(e.value)
    out = tmp_path / "cli"
    out.mkdir()
    (out / "g.reads").write_bytes((tmp_path / "k50.reads").read_bytes())
    p = _cli(["-f", NO_INPUT, "-k", "100", "-p", "g", "-m", "2"], out, check=False)
    assert p.returncode != 0 and "line 2: the read is not longer than -k (100)" in p.stderr
    assert not (out / "g.graph3").exists()


# ---- 5. long reads ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["f56", "v248", "hicopy250", "v505", "f1016", "short_in_wide"])
def test_long_reads_restart_equals_oracle(name, tmp_path):
    reads, k = long_datasets.get(name)
    _oracle_files(reads, k, tmp_path)
    gpu, r, g = _restart(tmp_path / "o.reads", k, tmp_path)
    assert gpu.counters()["record_words"] == long_datasets.SW[name]
    assert r.read_bytes() == (tmp_path / "o.reads").read_bytes()
    assert g.read_bytes() == (tmp_path / "o.graph3").read_bytes()


# ---- 6. several contexts ------------------------------------------------------------------------------------------------------

def _parsed(log):
    return [int(x) for x in re.search(r"Lines parsed per context:([ 0-9]+)", log).group(1).split()]


@pytest.mark.parametrize("layout", ["replicated", "sharded"])
def test_cli_restart_on_several_contexts(layout, tmp_path):
    env = {"SAGE2GPU_TABLE_LAYOUT": layout}
    for name in ("mixed", "cfg1"):
        src = tmp_path / name
        _, k = _golden_reads(name, src)
        for devs in DEVICES:
            out = tmp_path / f"{name}_{devs.replace(',', '_')}"
            out.mkdir()
            (out / "g.reads").write_bytes((src / "g.reads").read_bytes())
            piece = {"SAGE2GPU_UPLOAD_PIECE_BYTES": "65536"} if name == "mixed" else {}
            _cli(["-f", NO_INPUT, "-k", str(k), "-p", "g", "-m", "2", "--devices", devs], out, dict(env, **piece))
            assert _md5(out / "g.graph3") == GOLD[name]["graph3_md5"], devs
            log = open(out / "g.log").read()
            got = _parsed(log)
            assert len(got) == (4 if devs == "0-3" else len(devs.split(","))) and min(got) > 0 and sum(got) == GOLD[name]["unique_reads"], got
            assert f"Number of unique reads: {GOLD[name]['unique_reads']}" in log
            assert f"Table layout: {layout} (SAGE2GPU_TABLE_LAYOUT)" in log
    # fewer lines than contexts
    reads, k = datasets.get("single")
    src = tmp_path / "single"
    src.mkdir()
    _oracle_files(reads, k, src)
    for devs in DEVICES:
        out = tmp_path / f"single_{devs.replace(',', '_')}"
        out.mkdir()
        (out / "g.reads").write_bytes((src / "o.reads").read_bytes())
        _cli(["-f", NO_INPUT, "-k", str(k), "-p", "g", "-m", "3", "--devices", devs], out, env)
        assert (out / "g.graph3").read_bytes() == (src / "o.graph3").read_bytes(), devs
        assert sum(_parsed(open(out / "g.log").read())) == 1


# ---- 7. malformed files ---------------------------------------------------------------------------------------------------------

def _lines(path):
    return open(path, "rb").read().split(b"\n")[:-1]


def _join(lines):
    return b"\n".join(lines) + b"\n"


def _swap(lines, i):
    lines = list(lines)
    lines[i], lines[i + 1] = lines[i + 1], lines[i]
    return lines


def _mutations(base):
    """(name, file bytes, the line the error must name, words of the rule); base = the lines of a valid file (0 = the count)."""
    L = list(base)
    U = len(L) - 1
    i = 10                               # file line i + 1
    f, n, F, R = L[i].split(b"\t")
    pal = next(j for j in range(1, U + 1) if L[j].split(b"\t")[2] != L[j].split(b"\t")[3])
    pf, pn, pF, pR = L[pal].split(b"\t")
    out = [
        ("freq_leading_zero", L[:i] + [b"0" + L[i]] + L[i + 1:], i + 1, "FREQ"),
        ("freq_too_big", L[:i] + [b"\t".join([b"65536", n, F, R])] + L[i + 1:], i + 1, "FREQ"),
        ("len_mismatch", L[:i] + [b"\t".join([f, str(int(n) + 1).encode(), F, R])] + L[i + 1:], i + 1, "|F| = |R| = LEN"),
        ("len_zero", L[:i] + [b"\t".join([f, b"0", F, R])] + L[i + 1:], i + 1, "LEN"),
        ("lower_case", L[:i] + [b"\t".join([f, n, F.lower(), R])] + L[i + 1:], i + 1, "F contains"),
        ("n_base", L[:i] + [b"\t".join([f, n, F[:5] + b"N" + F[6:], R])] + L[i + 1:], i + 1, "F contains"),
        ("carriage_return", L[:i] + [L[i] + b"\r"] + L[i + 1:], i + 1, "|F| = |R| = LEN"),
        ("not_revcomp", L[:i] + [b"\t".join([f, n, F, R[:7] + (b"A" if R[7:8] != b"A" else b"C") + R[8:]])] + L[i + 1:], i + 1,
         "reverse complement"),
        ("not_canonical", L[:pal] + [b"\t".join([pf, pn, pR, pF])] + L[pal + 1:], pal + 1, "canonical"),
        ("too_long", L[:i] + [b"\t".join([b"1", b"1017", b"A" * 1017, b"T" * 1017])] + L[i + 1:], i + 1, "longer than 1016"),
        ("swapped_pair", _swap(L, i), i + 2, "increasing order"),
        ("duplicate_line", L[:i + 1] + [L[i]] + L[i + 1:], i + 2, "increasing order"),
        ("extra_line", [str(U - 1).encode()] + L[1:], U + 1, "more reads than"),
        ("missing_line", [str(U + 1).encode()] + L[1:], U + 2, "the file ends after"),
        ("bad_count", [b"0" + L[0]] + L[1:], 1, "first line"),
    ]
    out = [(name, _join(ls), line, rule) for name, ls, line, rule in out]
    whole = _join(L)
    cut = whole.rfind(b"\n", 0, len(whole) - 1) + 40
    out.append(("truncated", whole[:cut], U + 1, "truncated"))
    out.append(("gzip", gzip.compress(whole), 1, "gzip"))
    return out


def test_malformed_files_fail_naming_the_line(tmp_path):
    reads, k = datasets.get("rep")
    _oracle_files(reads, k, tmp_path)
    base = _lines(tmp_path / "o.reads")
    for name, data, line, rule in _mutations(base):
        d = tmp_path / name
        d.mkdir()
        (d / "g.reads").write_bytes(data)
        for piece in ("65536", None):          # many pieces per context, and one
            env = {"SAGE2GPU_UPLOAD_PIECE_BYTES": piece} if piece else {}
            os.environ.update(env)
            try:
                gpu = api.Sage2Gpu(0)
                with pytest.raises(api.Sage2GpuError) as e:
                    gpu.load_saved_reads(str(d / "g.reads"), k)
                assert e.value.code == api.ERR_FORMAT, (name, str(e.value))
                assert f"line {line}: " in str(e.value) and rule in str(e.value), (name, str(e.value))
                # nothing is loaded
                with pytest.raises(api.Sage2GpuError):
                    gpu.build_hash_table()
                gpu.close()
            finally:
                os.environ.pop("SAGE2GPU_UPLOAD_PIECE_BYTES", None)
        for devs in [None] + DEVICES[:1]:
            args = ["-f", NO_INPUT, "-k", str(k), "-p", "g", "-m", "2"] + (["--devices", devs] if devs else [])
            p = _cli(args, d, check=False)
            assert p.returncode != 0, (name, devs)
            assert f"line {line}: " in p.stderr and rule in p.stderr and p.stderr.startswith("FORMAT"), (name, devs, p.stderr)
            assert not (d / "g.graph3").exists(), (name, devs)
            assert f"line {line}: " in open(d / "g.log").read()


def test_swapped_pair_across_two_contexts(tmp_path):
    """The last line of context 0's slice and the first of context 1's swapped: each slice alone is in order."""
    reads, k = datasets.get("rep")
    _oracle_files(reads, k, tmp_path)
    L = _lines(tmp_path / "o.reads")
    body = sum(len(x) + 1 for x in L[1:])
    starts = np.cumsum([0] + [len(x) + 1 for x in L[1:]])      # byte offset of body line j (file line j + 2)
    a = int(np.searchsorted(starts, body // 2, side="left")) - 1  # the line that holds byte body // 2 - 1: last of slice 0
    if len(L[a + 1]) != len(L[a + 2]):                         # a swap of equal lengths keeps the boundary where it is
        pytest.fail("pick another data set: the lines at the boundary differ in length")
    swapped = _swap(L, a + 1)
    d = tmp_path / "cli"
    d.mkdir()
    (d / "g.reads").write_bytes(_join(swapped))
    p = _cli(["-f", NO_INPUT, "-k", str(k), "-p", "g", "-m", "2", "--devices", "0,0"], d, check=False)
    assert p.returncode != 0 and f"line {a + 3}: " in p.stderr and "increasing order" in p.stderr, p.stderr
    assert not (d / "g.graph3").exists()


# ---- 8. frequency wrap -----------------------------------------------------------------------------------------------------------

def test_frequency_wrap_is_documented_limit(tmp_path):
    """A read of 70,000 copies is saved with FREQ 70,000 mod 65,536: the edges equal the oracle's, numberOfReads in the .graph3
    header is the sum of the wrapped frequencies (a straight run counts every copy)."""
    reads, k = CASES["freq_wrap"]()
    o = _oracle_files(reads, k, tmp_path)
    gpu, _, g = _restart(tmp_path / "o.reads", k, tmp_path)
    e = gpu.edges()
    assert len(e) == o.n_edges
    for f in ("from", "to", "type", "delta", "delta_twin"):
        np.testing.assert_array_equal(e[f], o.edges[f])
    freq = o.frequency[1:].astype(np.int64)
    bp = int(np.sum(freq * o.length[1:]))
    head = g.read_bytes().split(b"\n")[:3]
    assert int(head[1]) == int(freq.sum()) < o.N
    assert int(head[2]) == bp // int(freq.sum())
    assert (o.frequency == 70_000 % 65_536).any()


# ---- 9. full size -------------------------------------------------------------------------------------------------------------

def test_cfg2_restart_gives_the_reference_graph(tmp_path):
    reads, k = synth.config_cached("cfg2")
    b, off = synth.concat(reads)
    gpu = api.Sage2Gpu(0)
    gpu.load_reads(b, off, k)
    gpu.write_reads(str(tmp_path / "g.reads"))
    gpu.close()
    assert _md5(tmp_path / "g.reads") == GOLD_BIG["cfg2"]["reads_md5"]
    _, _, g = _restart(tmp_path / "g.reads", k, tmp_path, "r")
    assert _md5(g) == GOLD_BIG["cfg2"]["graph3_md5"]
