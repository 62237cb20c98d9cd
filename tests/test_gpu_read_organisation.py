"""GPU parity of the read organisation (sort, dedupe, F / RC records) and of the table build on inputs made to reach
their rarer paths: tie runs of equal leading bases just below and above the in-kernel limit and far above it, exact
duplicates past the uint16_t frequency wrap, keys shared by many reads (runs of entries and masked keys), and keys
crowded into one home sector of the slot index.  Every case runs with both table builds and with the reads organised
over two contexts (key-range partitioned), against the oracle."""
import numpy as np
import pytest
import torch

from oracle import oracle
from sage2_b200 import api, multi, synth
from test_gpu_parity import _compare, _run_gpu

pytestmark = pytest.mark.gpu

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
# csrc/reads.cu: runs of more than kTieLimit reads with equal leading bases leave tie_fix_kernel for refine_long_runs; the
# leading bases compared are 16 for inputs of up to 134 M reads
TIE_LIMIT, SORT_BASES = 32, 16


def _seq(rng, n):
    return ACGT[rng.integers(0, 4, size=n)].tobytes()


def _fwd(rng, n):
    """n bases starting and ending with A: the read is smaller than its reverse complement, so it is stored as it is and its
    leading bases stay the ones written here."""
    return b"A" + _seq(rng, n - 2) + b"A"


def _tie_runs(run_sizes, seed):
    rng = np.random.default_rng(seed)
    g = synth.random_genome(30_000, seed)
    reads = synth.to_list(synth.paired_reads(g, 100, 20, seed=seed + 1, mu=300, sigma=20))
    for size in run_sizes:
        head = b"A" + _seq(rng, SORT_BASES - 1)
        members = [head + _fwd(rng, 100 - SORT_BASES) for _ in range(size)]
        members += [members[int(i)] for i in rng.integers(0, size, size=size // 4)]      # duplicates inside the run
        rng.shuffle(members)
        reads += members
    return reads


def _near_limit():
    return _tie_runs([TIE_LIMIT - 1, TIE_LIMIT, TIE_LIMIT + 1, TIE_LIMIT + 2, TIE_LIMIT + 8] * 20, 101), 45


def _far_above_limit():
    return _tie_runs([3000, 700, 2 * TIE_LIMIT + 1], 111), 45


def _freq_wrap():
    rng = np.random.default_rng(121)
    g = synth.random_genome(20_000, 122)
    reads = synth.to_list(synth.paired_reads(g, 100, 20, seed=123, mu=300, sigma=20))
    hot = _fwd(rng, 100)
    reads += [hot] * 70_000
    warm = _fwd(rng, 100)
    reads += [warm] * 65_536
    rng.shuffle(reads)
    return reads, 45


def _shared_keys(k):
    """Reads that share their first and last h = min(k, 64) bases with different middles: all of one key's entries but the
    first meet its slot taken (the table build's second round); groups of 40 (a run of entries) and of 400 (a masked key)."""
    rng = np.random.default_rng(131 + k)
    h = min(k, 64)
    g = synth.random_genome(30_000, 132)
    reads = synth.to_list(synth.paired_reads(g, 120, 20, seed=133, mu=300, sigma=20))
    for size in (40, 40, 400, 3):
        pre, suf = b"A" + _seq(rng, h - 1), _seq(rng, h - 1) + b"A"
        reads += [pre + _seq(rng, 22) + suf for _ in range(size)]
    return reads, k


def _mix64(x):
    x = x ^ (x >> np.uint64(33))
    x = x * np.uint64(0xFF51AFD7ED558CCD)
    x = x ^ (x >> np.uint64(33))
    x = x * np.uint64(0xC4CEB9FE1A85EC53)
    return x ^ (x >> np.uint64(33))


def _crowded_sector():
    """All reads distinct, h = 32; the prefix keys of 24 of them share one home sector of the slot index (4 slots), so they
    probe on into the following sectors."""
    rng = np.random.default_rng(141)
    k, L, n = 32, 90, 3000
    nsec = max(256, (4 * n + 2 * n + 3) // 4)           # csrc/table.cu, one context: 4 keys per read, load factor <= 2/3
    cand = rng.integers(0, 1 << 62, size=400_000, dtype=np.uint64)      # the 31 bases after the leading A
    with np.errstate(over="ignore"):
        v1 = cand                                        # 'A' + 31 bases as a 64-bit big-endian 2-bit integer: A = 0
        hsh = _mix64(v1 ^ _mix64(np.uint64(0x9E3779B97F4A7C15)))
        hi, lo = hsh >> np.uint64(32), hsh & np.uint64(0xFFFFFFFF)
        sec = (hi * np.uint64(nsec) + ((lo * np.uint64(nsec)) >> np.uint64(32))) >> np.uint64(32)
    target = np.bincount(sec.astype(np.int64), minlength=nsec).argmax()
    picked = cand[sec == target][:24]
    assert len(picked) >= 12
    reads = []
    for v in picked:
        bases = bytes(ACGT[(int(v) >> (2 * (30 - i))) & 3] for i in range(31))
        reads.append(b"A" + bases + _fwd(rng, L - 32))
    while len(reads) < n:
        reads.append(_fwd(rng, L))
    return reads, k


CASES = {
    "near_limit": _near_limit, "far_above_limit": _far_above_limit, "freq_wrap": _freq_wrap,
    "shared_keys_k45": lambda: _shared_keys(45), "shared_keys_k31": lambda: _shared_keys(31), "shared_keys_k70": lambda: _shared_keys(70),
    "crowded_sector": _crowded_sector,
}


@pytest.mark.parametrize("build", ["bucketed", "direct"])
@pytest.mark.parametrize("name", list(CASES))
def test_one_context_equals_oracle(name, build, monkeypatch):
    monkeypatch.setenv("SAGE2GPU_TABLE_BUILD", build)
    reads, k = CASES[name]()
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    loader, _ = _run_gpu(reads, k)
    _compare(o, loader.gpu)
    if name == "freq_wrap":
        assert (loader.gpu.reads()["frequency"] == 70_000 % 65_536).any()


@pytest.mark.parametrize("build", ["bucketed", "direct"])
@pytest.mark.parametrize("name", list(CASES))
def test_two_contexts_partitioned_equal_oracle(name, build, monkeypatch):
    monkeypatch.setenv("SAGE2GPU_TABLE_BUILD", build)
    reads, k = CASES[name]()
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    dev = torch.device("cuda", 0)
    tb, to = torch.from_numpy(b).to(dev), torch.from_numpy(off).to(dev)
    torch.cuda.synchronize()
    gpus = [api.Sage2Gpu(0) for _ in range(2)]
    multi.run_local([multi.partitioned_graph_steps(g, r, 2, multi.device_view_fn(dev), tb.data_ptr(), to.data_ptr(), len(off) - 1, k, True)
                     for r, g in enumerate(gpus)])
    for g in gpus:
        c = g.counters()
        assert c["unique_reads"] == o.U and c["distinct_keys"] == o.distinct_keys and c["keys_over_threshold"] == o.keys_over_threshold
        r = g.reads()
        np.testing.assert_array_equal(r["length"], o.length[1:])
        np.testing.assert_array_equal(r["frequency"], o.frequency[1:])
        np.testing.assert_array_equal(r["fwd"], o.fwd)
        np.testing.assert_array_equal(r["rc"], o.rc)
        e = g.edges()
        assert len(e) == o.n_edges
        for f in ("from", "to", "type", "delta", "delta_twin"):
            np.testing.assert_array_equal(e[f], o.edges[f])
