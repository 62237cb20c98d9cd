"""GPU tests of `sage2gpu --devices LIST`: the input spread over the contexts as it is read, and the table layout the program
picks (replicated on every context, or sharded by key hash with the window probes routed through peer-memory mailboxes).
Whatever the layout and however the input was spread, `.reads` and `.graph3` must be the bytes the reference writes
(md5s in tests/golden/golden.json) or, for sets without goldens, the oracle's files."""
import gzip
import hashlib
import json
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import datasets
import long_datasets
from oracle import oracle
from sage2_b200 import api, synth
from test_gpu_cli import BIN, _devices_args

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "golden.json")))
DEVICES = [d for d, _ in _devices_args()]
LAYOUTS = ["replicated", "sharded"]


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


def _get(name):
    return datasets.get(name) if name in datasets.DATASETS else synth.config(name)


def _run(args, out, devs, layout=None, **env):
    e = dict(os.environ, **{k: str(v) for k, v in env.items()})
    if layout:
        e["SAGE2GPU_TABLE_LAYOUT"] = layout
    subprocess.run([BIN, *args, "-o", str(out), "-p", "g", "-M", "3", "--devices", devs], check=True, env=e)
    return _md5(out / "g.reads"), _md5(out / "g.graph3"), open(out / "g.log").read()


def _received(log):
    return [int(x) for x in re.search(r"Reads received per context:([ 0-9]+)", log).group(1).split()]


def _gold(name):
    return GOLD[name]["reads_md5"], GOLD[name]["graph3_md5"]


@pytest.mark.parametrize("name", ["mixed", "rep", "varlen_err", "hicopy", "cfg1"])
def test_sharded_layout_byte_identical_to_reference(name, tmp_path):
    reads, k = _get(name)
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    for devs in DEVICES:
        r, g, log = _run(["-f", str(fq), "-k", str(k)], tmp_path / devs.replace(",", "_"), devs, "sharded")
        assert (r, g) == _gold(name), devs
        assert "Table layout: sharded (SAGE2GPU_TABLE_LAYOUT)" in log
        assert f"Number of unique reads: {GOLD[name]['unique_reads']}" in log
        assert re.search(r"Size of hash table: \d+ slots, \d+ distinct keys \(sum over the shards\)", log)


@pytest.mark.parametrize("name", ["mixed", "rep", "varlen_err", "hicopy"])
def test_small_pieces_reach_every_context(name, tmp_path):
    """Sets smaller than one 32 MB piece, dealt out in 64 KB pieces: every context receives reads and packs its part, in
    the layout the program picks; the reference's bytes."""
    reads, k = _get(name)
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    for devs in DEVICES:
        r, g, log = _run(["-f", str(fq), "-k", str(k)], tmp_path / devs.replace(",", "_"), devs, SAGE2GPU_UPLOAD_PIECE_BYTES=65536)
        assert (r, g) == _gold(name), devs
        got = _received(log)
        assert len(got) == (4 if devs == "0-3" else len(devs.split(","))) and min(got) > 0, (devs, got)
        assert f"Number of unique reads: {GOLD[name]['unique_reads']}" in log


def test_sharded_layout_grows_the_mailboxes_for_the_phase_c_list(tmp_path):
    """An error-rich set sends many reads to phase C; with routed batches of 64 reads the list batch is far larger than the
    mailboxes, which must grow for it."""
    reads, k = _get("err")
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    for devs in DEVICES:
        r, g, log = _run(["-f", str(fq), "-k", str(k)], tmp_path / devs.replace(",", "_"), devs, "sharded", SAGE2GPU_ROUTE_BATCH_READS=64)
        assert (r, g) == _gold("err"), devs
        assert "routed batches of 64 reads" in log
        listed = int(re.search(r"list batch of the reads left for phase C: (\d+) reads", log).group(1))
        assert listed > 64
        assert f"Total reads left to explore: {listed}" in log


@pytest.mark.parametrize("layout", LAYOUTS)
def test_distributed_ingest_device_parser_gzip_and_sequential_parser(layout, tmp_path):
    """cfg1 (88 MB of FASTQ: three 32 MB pieces; 16 MB pieces for four contexts) as regular FASTQ, gzip and multi-line FASTA
    (sequential parser, smaller chunks so that they reach every context): golden bytes, and every context received reads."""
    reads, k = _get("cfg1")
    lst = synth.to_list(reads)
    fq = tmp_path / "a.fastq"
    synth.write_fastq(str(fq), reads)
    gz = tmp_path / "a.fastq.gz"
    with gzip.open(gz, "wb", compresslevel=1) as f:
        f.write(open(fq, "rb").read())
    ml = tmp_path / "multi.fa"
    with open(ml, "wb") as f:
        for i, s in enumerate(lst):
            f.write(b">r%d\n%s\n%s\n" % (i, s[:60], s[60:]))
    for devs in DEVICES:
        G = len(devs.split(",")) if "-" not in devs else 4
        pieces = {} if G <= 3 else {"SAGE2GPU_UPLOAD_PIECE_BYTES": 16 << 20}        # three 32 MB pieces leave a fourth context empty
        for path, env, split in ((fq, pieces, "yes"), (gz, pieces, "yes"), (ml, {"SAGE2GPU_UPLOAD_PIECE_BYTES": 4 << 20}, "no")):
            out = tmp_path / f"{path.name}_{devs.replace(',', '_')}"
            r, g, log = _run(["-f", str(path), "-k", str(k)], out, devs, layout, **env)
            assert (r, g) == _gold("cfg1"), (path.name, devs)
            assert f"Records split on the device: {split}" in log
            got = _received(log)
            assert len(got) == G and min(got) > 0 and sum(got) == len(lst), (path.name, devs, got)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_distributed_ingest_two_mate_files_of_unequal_length(layout, tmp_path):
    """The reference stops a two-file data set when one file ends (inputReader.cpp:26-49).  With 64 KB pieces file 1 is spread
    over every context, and its surplus must leave the contexts that hold its LAST records."""
    reads, k = _get("rep")
    lst = synth.to_list(reads)
    m1, m2 = lst[0::2], lst[1::2]
    for name, (a, b) in {"long1": (m1, m2[:-700]), "long2": (m1[:-500], m2)}.items():
        synth.write_fastq(str(tmp_path / f"{name}_1.fastq"), a)
        synth.write_fastq(str(tmp_path / f"{name}_2.fastq"), b)
        (tmp_path / f"{name}.list").write_text(f"f1={tmp_path}/{name}_1.fastq\nf2={tmp_path}/{name}_2.fastq\n")
        one = subprocess.run([BIN, "-l", str(tmp_path / f"{name}.list"), "-k", str(k), "-o", str(tmp_path / f"{name}_one"), "-p", "g", "-M", "3"],
                             check=True)
        want = (_md5(tmp_path / f"{name}_one" / "g.reads"), _md5(tmp_path / f"{name}_one" / "g.graph3"))
        kept = min(len(a), len(b) + 1) + min(len(b), len(a))
        for devs in DEVICES:
            r, g, log = _run(["-l", str(tmp_path / f"{name}.list"), "-k", str(k)], tmp_path / f"{name}_{devs.replace(',', '_')}", devs, layout,
                             SAGE2GPU_UPLOAD_PIECE_BYTES=65536)
            assert (r, g) == want, (name, devs)
            got = _received(log)
            assert min(got) > 0 and sum(got) == kept, (name, devs, got)
            assert f"Good reads: {kept}" in log.replace(",", "")


@pytest.mark.parametrize("layout", LAYOUTS)
def test_distributed_ingest_widest_reads_in_one_context(layout, tmp_path):
    """short_in_wide with its reads of 400-1016 bases at the head of the file and 64 KB pieces: only the first context sees
    them, the others must still pack at their stride (32 words).  Equal to the oracle's files."""
    reads, k = long_datasets.get("short_in_wide")
    lst = synth.to_list(reads)
    lst = sorted(lst, key=len, reverse=True)[:9] + sorted(lst, key=len, reverse=True)[9:]
    assert len(lst[8]) >= 400 and max(len(s) for s in lst[9:]) <= 150
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), lst)
    b, off = synth.concat(lst)
    o = oracle.OracleRun(b, off, k)
    o.write_reads(str(tmp_path / "o.reads"))
    o.write_graph3(str(tmp_path / "o.graph3"))
    want = (_md5(tmp_path / "o.reads"), _md5(tmp_path / "o.graph3"))
    for devs in DEVICES:
        r, g, log = _run(["-f", str(fq), "-k", str(k)], tmp_path / devs.replace(",", "_"), devs, layout, SAGE2GPU_UPLOAD_PIECE_BYTES=65536)
        assert (r, g) == want, devs
        got = _received(log)
        assert min(got) > 0, got


def test_small_set_picks_the_replicated_layout(tmp_path):
    reads, k = _get("rep")
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    env = {k_: v for k_, v in os.environ.items() if k_ != "SAGE2GPU_TABLE_LAYOUT"}
    out = tmp_path / "out"
    subprocess.run([BIN, "-f", str(fq), "-k", str(k), "-o", str(out), "-p", "g", "-M", "3", "--devices", "0,0"], check=True, env=env)
    assert (_md5(out / "g.reads"), _md5(out / "g.graph3")) == _gold("rep")
    log = open(out / "g.log").read()
    assert "Table layout: replicated. Per context: replicated table" in log
    assert re.search(r"GPU 0: replicated table \+ reserve of its contexts \d+ bytes, free \d+ bytes: fits", log)
    assert "The replicated table fits on every GPU." in log


# ---- the C ABI underneath ----------------------------------------------------------------------------------------------

def test_streamed_upload_over_three_contexts_packs_at_the_longest_read():
    """Three contexts on one GPU each receive part of one streamed upload (the widest reads all in one of them), agree on the
    longest read, pack their slices at its stride, all-gather and organise: the oracle's reads and edges."""
    reads, k = long_datasets.get("short_in_wide")
    lst = sorted(synth.to_list(reads), key=len, reverse=True)
    b, off = synth.concat(lst)
    o = oracle.OracleRun(b, off, k)
    world = 3
    gpus = [api.Sage2Gpu(0) for _ in range(world)]
    cut = [0, 9, len(lst) // 2, len(lst)]          # the 9 reads of 400-1016 bases go to context 0 only
    for r, g in enumerate(gpus):
        g.load_begin(k)
        for c0 in range(cut[r], cut[r + 1], 1000):        # several chunks per context
            c1 = min(cut[r + 1], c0 + 1000)
            cb, co = synth.concat(lst[c0:c1])
            g.load_append(cb, co)
    lens = [g.load_max_length() for g in gpus]
    assert lens[0] == max(len(s) for s in lst) and max(lens[1:]) <= 150
    slices = [g.load_finish_slice(max(lens)) for g in gpus]
    assert [s["n_reads"] for s in slices] == [cut[r + 1] - cut[r] for r in range(world)]
    assert len({s["record_words"] for s in slices}) == 1 and slices[0]["record_words"] == long_datasets.SW["short_in_wide"]
    counts = [s["n_reads"] for s in slices]
    sw = slices[0]["record_words"]
    lay = [g.raw_gather_layout(r, world, counts) for r, g in enumerate(gpus)]
    views = [torch.as_tensor(_Dev(lay[r]["records"], lay[r]["total"] * sw), device="cuda:0") for r in range(world)]
    offs = np.cumsum([0] + counts) * sw
    for q in range(world):
        blk = views[q][offs[q]:offs[q + 1]].clone()
        for r in range(world):
            if r != q:
                views[r][offs[q]:offs[q + 1]] = blk
    torch.cuda.synchronize()
    good, bp = sum(s["good_reads"] for s in slices), sum(s["total_bp"] for s in slices)
    for g in gpus:
        g.raw_gather_finish(sum(counts), good, bp)
    # organising the whole gathered set on every context (world 1 each) must give the oracle's read set
    for g in gpus:
        g.organize_partition(0, 1)
        g.build_hash_table()
        g.build_overlap_graph()
        r = g.reads()
        np.testing.assert_array_equal(r["length"], o.length[1:])
        np.testing.assert_array_equal(r["frequency"], o.frequency[1:])
        np.testing.assert_array_equal(r["fwd"], o.fwd)
        e = g.edges()
        assert len(e) == o.n_edges
        for f in ("from", "to", "type", "delta", "delta_twin"):
            np.testing.assert_array_equal(e[f], o.edges[f])


def _gather_blocks(ptrs, counts, words, typestr="<i8"):
    """In memory, between contexts on GPU 0: block q (counts[q] * words elements) of every context's array from context q."""
    total = sum(counts) * words
    views = [torch.as_tensor(_Dev(p, total, typestr), device="cuda:0") for p in ptrs]
    offs = np.cumsum([0] + list(counts)) * words
    for q in range(len(ptrs)):
        blk = views[q][offs[q]:offs[q + 1]].clone()
        for r in range(len(ptrs)):
            if r != q:
                views[r][offs[q]:offs[q + 1]] = blk
    torch.cuda.synchronize()


def test_low_memory_switched_on_after_the_gather_releases_the_input():
    """The sharded layout is chosen after the reads are gathered: switching low_memory on then must release the packed
    input, the packed slice and the local unique run at once (the stages that would have released them are over)."""
    reads, k = synth.config("cfg1")
    b, off = synth.concat(reads)
    n = len(off) - 1
    world, cut = 2, [0, n // 2, n]
    gpus = [api.Sage2Gpu(0) for _ in range(world)]
    keep = []
    info = []
    for r, g in enumerate(gpus):
        sb, so = b[off[cut[r]]:off[cut[r + 1]]], off[cut[r]:cut[r + 1] + 1] - off[cut[r]]
        keep.append((sb, so))
        info.append(g.pack_slice(sb.ctypes.data, so.ctypes.data, cut[r + 1] - cut[r], k, False, int(np.diff(off).max())))
    counts = [cut[r + 1] - cut[r] for r in range(world)]
    sw = info[0]["record_words"]
    lay = [g.raw_gather_layout(r, world, counts) for r, g in enumerate(gpus)]
    _gather_blocks([x["records"] for x in lay], counts, sw)
    for g in gpus:
        g.raw_gather_finish(n, sum(x["good_reads"] for x in info), sum(x["total_bp"] for x in info))
    uloc = [g.organize_partition(r, world) for r, g in enumerate(gpus)]
    rl = [g.reads_gather_layout(uloc) for g in gpus]
    stride = rl[0]["stride"]
    _gather_blocks([x["records"] for x in rl], uloc, stride)
    _gather_blocks([x["lengths"] for x in rl], uloc, 1, "<i2")
    _gather_blocks([x["frequencies"] for x in rl], uloc, 1, "<i2")
    for g in gpus:
        g.reads_gather_finish()
    before = gpus[0].table_bytes(world)["device_free"]
    for g in gpus:
        g.set_option("low_memory", 1)
    after = gpus[0].table_bytes(world)["device_free"]
    packed = 8 * sw * n          # the joint packed records, held by each of the two contexts
    assert after - before >= world * packed, (before, after, packed)
    # the contexts still build the sharded table and the graph from the replicated reads
    o = oracle.OracleRun(b, off, k)
    from sage2_b200 import multi
    for r, g in enumerate(gpus):
        g.build_hash_table_shard(r, world)
    multi.run_local([multi.sharded_graph_steps(g, r, world, multi.device_view_fn(torch.device("cuda", 0))) for r, g in enumerate(gpus)])
    for g in gpus:
        assert len(g.edges()) == o.n_edges


class _Dev:
    def __init__(self, ptr, n, typestr="<i8"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


@pytest.mark.parametrize("name,world", [("rep", 1), ("varlen_err", 2), ("hicopy", 3)])
def test_table_bytes_match_the_built_tables(name, world):
    """sage2gpu_table_bytes: slot bytes equal what the build allocates, entry bytes bound what it fills, in both layouts."""
    reads, k = datasets.get(name)
    b, off = synth.concat(reads)
    for layout in LAYOUTS:
        gpus = [api.Sage2Gpu(0) for _ in range(world)]
        for r, g in enumerate(gpus):
            g.load_reads(b, off, k)
        sizes = [g.table_bytes(world) for g in gpus]
        assert all(s["device_free"] > 0 for s in sizes)
        if layout == "sharded":
            for r, g in enumerate(gpus):
                g.build_hash_table_shard(r, world)
                info = g.table_shard_info()
                assert sizes[r]["sharded_slots"] == 8 * info["slots"]
                assert sizes[r]["sharded_entries"] >= 4 * info["entries"]
        else:
            for r, g in enumerate(gpus):
                g.build_hash_table_part(r, world) if world > 1 else g.build_hash_table()
            infos = [g.table_shard_info() for g in gpus]
            if world > 1:
                ec = [i["entries"] for i in infos]
                lay = [g.table_gather_layout(ec) for g in gpus]
                for g in gpus:       # the slot and entry arrays stay ungathered: only the sizes are compared here
                    g.table_gather_finish(ec, [i["distinct"] for i in infos], [i["over"] for i in infos])
                infos = [g.table_shard_info() for g in gpus]
            for r, g in enumerate(gpus):
                assert sizes[r]["replicated_slots"] == 8 * infos[r]["slots"]
                assert sizes[r]["replicated_entries"] >= 4 * infos[r]["entries"]
        for g in gpus:
            g.close()
