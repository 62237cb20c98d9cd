"""GPU tests of the GFA 1.0 writer (sage2gpu_write_gfa, `sage2gpu --gfa`): the bytes the device formats must be, byte for
byte, what the independent Python writer of tests/gfa.py makes from the `.reads` / `.graph3` of the same graph, and what
it makes passes the validator there (every L line an exact overlap in its stated orientations)."""
import gzip
import hashlib
import json
import os
import shutil
import subprocess

import pytest

import datasets
import gfa
import long_datasets
from oracle import oracle
from sage2_b200 import api, synth
from test_gpu_cli import BIN

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "golden.json")))
BIG = json.load(open(os.path.join(HERE, "golden", "golden_big.json")))

# csrc/format.cu: S and L lines go to the file in batches of at most this many bytes of text, sized for the widest line
BATCH_BYTES = 1 << 28


def _md5_file(path):
    h = hashlib.md5()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 22), b""):
            h.update(blk)
    return h.hexdigest()


def _get(name):
    if name in datasets.DATASETS:
        return datasets.get(name)
    if name in long_datasets.LONG_DATASETS:
        return long_datasets.get(name)
    return synth.config(name)


# ---- 1. the C ABI against the Python writer on the oracle's files ---------------------------------------------------------

@pytest.mark.parametrize("name", list(datasets.DATASETS) + list(long_datasets.LONG_DATASETS))
def test_write_gfa_equals_python_writer_on_oracle_files(name, tmp_path):
    reads, k = _get(name)
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    o.write_reads(str(tmp_path / "o.reads"))
    o.write_graph3(str(tmp_path / "o.graph3"))
    want = gfa.write_gfa_bytes(str(tmp_path / "o.reads"), str(tmp_path / "o.graph3"))
    gpu = api.Sage2Gpu(0)
    gpu.run_steps123(b, off, k)
    gpu.write_gfa(str(tmp_path / "g.gfa"))
    assert (tmp_path / "g.gfa").read_bytes() == want


def test_write_gfa_before_the_graph_is_a_state_error(tmp_path):
    reads, k = datasets.get("rep")
    b, off = synth.concat(reads)
    gpu = api.Sage2Gpu(0)
    with pytest.raises(api.Sage2GpuError) as e:            # nothing loaded
        gpu.write_gfa(str(tmp_path / "a.gfa"))
    assert e.value.code == api.ERR_STATE and "no overlap graph" in str(e.value)
    gpu.load_reads(b, off, k)
    gpu.build_hash_table()
    with pytest.raises(api.Sage2GpuError) as e:            # reads and table, no graph yet
        gpu.write_gfa(str(tmp_path / "a.gfa"))
    assert e.value.code == api.ERR_STATE
    assert not (tmp_path / "a.gfa").exists()
    gpu.build_overlap_graph()
    with pytest.raises(api.Sage2GpuError) as e:            # a directory that does not exist
        gpu.write_gfa(str(tmp_path / "no" / "such" / "dir" / "a.gfa"))
    assert e.value.code == api.ERR_IO
    gpu.write_gfa(str(tmp_path / "a.gfa"))
    gfa.validate(str(tmp_path / "a.gfa"), k)


# ---- 2. full size: batch seams ----------------------------------------------------------------------------------------------

def _full_size(name, tmp_path):
    """`.reads` / `.graph3` with the reference's md5s, and the `.gfa` of the same context equal to the Python writer's output
    from them and valid.  Returns the counters and the longest read."""
    reads, k = synth.config_cached(name)
    b, off = synth.concat(reads)
    max_len = int((off[1:] - off[:-1]).max())
    del reads
    gpu = api.Sage2Gpu(0)
    gpu.run_steps123(b, off, k)
    del b, off
    for ext, write in ((".reads", gpu.write_reads), (".graph3", gpu.write_graph3), (".gfa", gpu.write_gfa)):
        write(str(tmp_path / ("g" + ext)))
    c = gpu.counters()
    gpu.close()
    assert _md5_file(tmp_path / "g.reads") == BIG[name]["reads_md5"]
    assert _md5_file(tmp_path / "g.graph3") == BIG[name]["graph3_md5"]
    gfa.write_gfa(str(tmp_path / "g.reads"), str(tmp_path / "g.graph3"), str(tmp_path / "p.gfa"))
    os.remove(tmp_path / "g.graph3")
    assert _md5_file(tmp_path / "g.gfa") == _md5_file(tmp_path / "p.gfa")
    os.remove(tmp_path / "p.gfa")
    os.remove(tmp_path / "g.reads")
    assert gfa.validate(str(tmp_path / "g.gfa"), k) == {"segments": c["unique_reads"], "links": c["n_edges"]}
    return c, max_len


def test_cfg2_full_size_gfa(tmp_path):
    c, max_len = _full_size("cfg2", tmp_path)
    # the S lines cross at least one batch seam
    assert c["unique_reads"] > BATCH_BYTES // (max_len + 35)


@pytest.mark.skipif(not os.environ.get("SAGE2_TEST_CFG4_FILES") or "cfg4" not in BIG,
                    reason="cfg4 files: opt in with SAGE2_TEST_CFG4_FILES=1")
def test_cfg4_full_size_gfa(tmp_path):
    c, _ = _full_size("cfg4", tmp_path)
    # the L lines cross several batch seams
    assert c["n_edges"] > 3 * (BATCH_BYTES // 34)


# ---- 3. the host program ----------------------------------------------------------------------------------------------------

def _cli(args, out, env=None):
    e = dict(os.environ, **(env or {}))
    p = subprocess.run([BIN, *args, "-o", str(out), "-p", "g", "-M", "3"], env=e, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    return out


def _files(out):
    return (out / "g.reads").read_bytes(), (out / "g.graph3").read_bytes()


@pytest.mark.parametrize("name", ["mixed", "rep", "varlen_err", "cfg1"])
def test_cli_gfa(name, tmp_path):
    reads, k = _get(name)
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    args = ["-f", str(fq), "-k", str(k)]
    plain = _files(_cli(args, tmp_path / "plain"))
    assert not (tmp_path / "plain" / "g.gfa").exists()
    runs = {
        "one context": _cli(args + ["--gfa"], tmp_path / "one"),
        "--devices 0,0 replicated": _cli(args + ["--gfa", "--devices", "0,0"], tmp_path / "rep",
                                         {"SAGE2GPU_TABLE_LAYOUT": "replicated"}),
        "--devices 0,0 sharded": _cli(args + ["--gfa", "--devices", "0,0"], tmp_path / "shard",
                                      {"SAGE2GPU_TABLE_LAYOUT": "sharded"}),
    }
    # -m 2: restart from the .reads the plain run wrote
    (tmp_path / "restart").mkdir()
    shutil.copy(tmp_path / "plain" / "g.reads", tmp_path / "restart" / "g.reads")
    runs["-m 2 restart"] = _cli(["-f", "/nonexistent/input.fastq", "-k", str(k), "-m", "2", "--gfa"], tmp_path / "restart")
    want = gfa.write_gfa_bytes(str(tmp_path / "plain" / "g.reads"), str(tmp_path / "plain" / "g.graph3"))
    for how, out in runs.items():
        assert _files(out) == plain, how                  # the flag changes no other file
        got = (out / "g.gfa").read_bytes()
        assert got == gfa.write_gfa_bytes(str(out / "g.reads"), str(out / "g.graph3")), how
        assert got == want, how
        assert "Function saveGfa in " in (out / "g.log").read_text(), how
    assert tuple(hashlib.md5(x).hexdigest() for x in plain) == (GOLD[name]["reads_md5"], GOLD[name]["graph3_md5"])
    if name == "mixed":      # the reference's committed files give the same GFA
        ref = gfa.write_gfa_bytes(gzip.open(os.path.join(HERE, "golden", "mixed.reads.gz")),
                                  gzip.open(os.path.join(HERE, "golden", "mixed.graph3.gz")))
        assert want == ref
