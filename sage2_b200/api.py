"""Python host side of libsage2gpu (ctypes over the C ABI in include/sage2gpu.h).

`Sage2Gpu` is the thin handle; `ReadLoader`, `HashTable` and `EconomyGraph` mirror the reference's
step-1..3 classes and method names (inputReader/readLoader.h:32-56, economyGraph/hashTable.h:20-44,
economyGraph/economyGraph.h:32-54) so that the parity tests read like a reference driver
(main.cpp:37-132).  There is no CPU fallback: if libsage2gpu.so is missing or no CUDA device is
present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsage2gpu.so")


class Sage2GpuError(RuntimeError):
    """`code` = the library's return code (include/sage2gpu.h: 5 = SAGE2GPU_ERR_FORMAT), `bad_line` = the line a format error names,
    `bad_member` = the index of the BGZF member that failed a check (-1: none), `bad_offset` = the compressed offset of the gzip
    member or block that failed a check (-1: none)."""
    code = 0
    bad_line = 0
    bad_member = -1
    bad_offset = -1


ERR_FORMAT = 5
ERR_STATE = 3
ERR_IO = 4


class GzipState(C.Structure):
    """sage2gpu_gzip_state: where a piece of a gzip stream continues (all zeros before the first piece)."""
    _fields_ = [("offset", C.c_uint64), ("member_offset", C.c_uint64), ("member_bytes", C.c_uint64), ("bit", C.c_uint32),
                ("in_member", C.c_uint32), ("crc", C.c_uint32), ("window_bytes", C.c_uint32), ("done", C.c_uint32),
                ("reserved", C.c_uint32), ("window", C.c_uint8 * 32768)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "total_reads", "good_reads", "unique_reads", "total_bp", "avg_len",
        "hash_len", "distinct_keys", "keys_over_threshold", "table_capacity",
        "contained_ext", "contained_size", "left_to_explore",
        "edges_phase_b", "candidates_c", "edges_inserted_c", "transitive_removed",
        "n_edges", "compare_calls", "window_probes", "slow_path_reads", "record_words", "probe_restarts", "phase_c_on_device",
        "fast_path_reads")]


class Timers(C.Structure):
    _fields_ = [(n, C.c_float) for n in (
        "ingest", "sort_reads", "build_table", "phase_a", "phase_b", "phase_c_dev", "phase_c_host",
        "sort_edges", "total", "phase_a_kernel")]


EDGE_DT = np.dtype([("from", "<u8"), ("to", "<u8"), ("type", "<u4"), ("delta", "<u4"),
                    ("delta_twin", "<u4"), ("reserved", "<u4")])

EXPORTS = ["sage2gpu_create", "sage2gpu_destroy", "sage2gpu_last_error", "sage2gpu_load_reads",
           "sage2gpu_load_begin", "sage2gpu_load_append", "sage2gpu_load_append_text", "sage2gpu_load_count", "sage2gpu_load_remove",
           "sage2gpu_load_finish", "sage2gpu_host_alloc", "sage2gpu_host_free",
           "sage2gpu_load_reads_device", "sage2gpu_build_hash_table", "sage2gpu_build_overlap_graph",
           "sage2gpu_phase_a_partition", "sage2gpu_phase_a_buffers", "sage2gpu_finish_graph",
           "sage2gpu_run_steps123", "sage2gpu_get_counters", "sage2gpu_get_timers", "sage2gpu_reads_bytes",
           "sage2gpu_get_reads", "sage2gpu_get_extensions", "sage2gpu_get_edges", "sage2gpu_get_edges_packed", "sage2gpu_write_reads",
           "sage2gpu_write_graph3", "sage2gpu_kernel_launches", "sage2gpu_stream", "sage2gpu_measure_gather",
           "sage2gpu_build_hash_table_shard", "sage2gpu_phase_a_sharded_begin", "sage2gpu_route_begin", "sage2gpu_shard_answer",
           "sage2gpu_route_finish", "sage2gpu_phase_a_routed", "sage2gpu_phase_a_sharded_end", "sage2gpu_phase_b",
           "sage2gpu_map_reads", "sage2gpu_mailbox_create", "sage2gpu_mailbox_open", "sage2gpu_route_post", "sage2gpu_answer_post",
           "sage2gpu_route_collect", "sage2gpu_mailbox_barrier", "sage2gpu_digest", "sage2gpu_set_option",
           "sage2gpu_load_reads_partition", "sage2gpu_reads_gather_layout", "sage2gpu_reads_gather_finish",
           "sage2gpu_table_shard_info", "sage2gpu_table_gather_layout", "sage2gpu_table_gather_finish",
           "sage2gpu_pack_slice", "sage2gpu_raw_gather_layout", "sage2gpu_raw_gather_finish", "sage2gpu_organize_partition",
           "sage2gpu_synth_reads", "sage2gpu_build_hash_table_part", "sage2gpu_load_finish_packed", "sage2gpu_peer_copy",
           "sage2gpu_phase_a_import", "sage2gpu_load_max_length", "sage2gpu_load_finish_slice", "sage2gpu_table_bytes",
           "sage2gpu_load_saved_reads", "sage2gpu_saved_reads_info", "sage2gpu_saved_reads_slice", "sage2gpu_saved_reads_pack",
           "sage2gpu_saved_reads_finish", "sage2gpu_table_view", "sage2gpu_load_append_bgzf", "sage2gpu_inflate_bgzf",
           "sage2gpu_load_append_gzip", "sage2gpu_inflate_gzip", "sage2gpu_write_gfa"]

_lib = None


def build_library(force: bool = False) -> None:
    """Compile libsage2gpu.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    args = ["make", "-C", os.path.join(HERE, "csrc"), "-j8"]
    if force:
        subprocess.check_call(args + ["clean"], stdout=subprocess.DEVNULL)
    subprocess.check_call(args, stdout=subprocess.DEVNULL)


def load_library():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Sage2GpuError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        vp, i64, u64p = C.c_void_p, C.c_int64, C.POINTER(C.c_uint64)
        lib.sage2gpu_create.argtypes = [C.POINTER(vp), C.c_int]
        lib.sage2gpu_destroy.argtypes = [vp]
        lib.sage2gpu_destroy.restype = None
        lib.sage2gpu_last_error.argtypes = [vp]
        lib.sage2gpu_last_error.restype = C.c_char_p
        lib.sage2gpu_load_reads.argtypes = [vp, vp, vp, i64, C.c_int]
        lib.sage2gpu_load_reads_device.argtypes = [vp, vp, vp, i64, C.c_int]
        lib.sage2gpu_load_begin.argtypes = [vp, C.c_int]
        lib.sage2gpu_load_append.argtypes = [vp, vp, vp, i64]
        lib.sage2gpu_load_append_text.argtypes = [vp, vp, C.c_uint64, C.c_int, C.POINTER(C.c_int), C.c_uint64, u64p, u64p]
        lib.sage2gpu_load_append_bgzf.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, C.c_int, C.POINTER(C.c_int), C.c_uint64, u64p, u64p,
                                                  vp, C.c_uint64, u64p, C.POINTER(i64)]
        lib.sage2gpu_inflate_bgzf.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, u64p, C.POINTER(i64), C.POINTER(C.c_float)]
        lib.sage2gpu_load_append_gzip.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, C.c_int, C.c_uint64, C.POINTER(GzipState),
                                                  C.POINTER(C.c_int), C.c_uint64, u64p, u64p, vp, C.c_uint64, u64p, u64p, C.POINTER(i64)]
        lib.sage2gpu_inflate_gzip.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, u64p, C.POINTER(i64), C.POINTER(C.c_float), u64p, u64p,
                                              u64p]
        lib.sage2gpu_load_count.argtypes = [vp, u64p]
        lib.sage2gpu_load_remove.argtypes = [vp, C.c_uint64, C.c_uint64]
        lib.sage2gpu_load_finish.argtypes = [vp]
        lib.sage2gpu_load_max_length.argtypes = [vp, C.POINTER(C.c_int)]
        lib.sage2gpu_load_finish_slice.argtypes = [vp, C.c_int, u64p, u64p, u64p, u64p]
        lib.sage2gpu_table_bytes.argtypes = [vp, C.c_int, u64p, u64p, u64p, u64p, u64p]
        lib.sage2gpu_load_saved_reads.argtypes = [vp, C.c_char_p, C.c_int]
        lib.sage2gpu_saved_reads_info.argtypes = [vp, C.c_char_p, u64p, u64p]
        lib.sage2gpu_saved_reads_slice.argtypes = [vp, C.c_char_p, C.c_int, C.c_uint64, C.c_uint64, u64p, C.POINTER(C.c_int), u64p]
        lib.sage2gpu_saved_reads_pack.argtypes = [vp, C.c_int, C.c_int, C.c_int, u64p, u64p, u64p]
        lib.sage2gpu_saved_reads_finish.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64, u64p]
        lib.sage2gpu_host_alloc.argtypes = [C.c_uint64]
        lib.sage2gpu_host_alloc.restype = vp
        lib.sage2gpu_host_free.argtypes = [vp]
        lib.sage2gpu_host_free.restype = None
        lib.sage2gpu_build_hash_table.argtypes = [vp]
        lib.sage2gpu_build_overlap_graph.argtypes = [vp]
        lib.sage2gpu_phase_a_partition.argtypes = [vp, C.c_int, C.c_int]
        lib.sage2gpu_phase_a_buffers.argtypes = [vp] + [C.POINTER(vp)] * 4 + [u64p, u64p]
        lib.sage2gpu_finish_graph.argtypes = [vp]
        lib.sage2gpu_table_view.argtypes = [vp, C.POINTER(vp), u64p, C.POINTER(vp), u64p, u64p, u64p]
        lib.sage2gpu_build_hash_table_shard.argtypes = [vp, C.c_int, C.c_int]
        lib.sage2gpu_phase_a_sharded_begin.argtypes = [vp, C.c_int, C.c_int, u64p, u64p]
        lib.sage2gpu_route_begin.argtypes = [vp, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.POINTER(vp), u64p, u64p]
        lib.sage2gpu_shard_answer.argtypes = [vp, vp, u64p, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(vp), u64p]
        lib.sage2gpu_route_finish.argtypes = [vp, vp, vp, u64p]
        lib.sage2gpu_phase_a_routed.argtypes = [vp, u64p]
        lib.sage2gpu_phase_a_sharded_end.argtypes = [vp]
        lib.sage2gpu_phase_b.argtypes = [vp]
        lib.sage2gpu_mailbox_create.argtypes = [vp, C.c_int, C.c_int, C.c_uint64, vp, C.POINTER(vp)]
        lib.sage2gpu_mailbox_open.argtypes = [vp, C.c_int, vp, vp]
        lib.sage2gpu_route_post.argtypes = [vp, C.c_int, C.c_uint64, C.c_uint64, C.c_int, u64p, u64p]
        lib.sage2gpu_answer_post.argtypes = [vp, C.c_int, u64p]
        lib.sage2gpu_route_collect.argtypes = [vp]
        lib.sage2gpu_mailbox_barrier.argtypes = [vp]
        lib.sage2gpu_map_reads.argtypes = [vp, vp, vp, i64, C.c_int, vp, vp, C.POINTER(C.c_float)]
        lib.sage2gpu_run_steps123.argtypes = [vp, vp, vp, i64, C.c_int]
        lib.sage2gpu_get_counters.argtypes = [vp, C.POINTER(Counters)]
        lib.sage2gpu_get_timers.argtypes = [vp, C.POINTER(Timers)]
        lib.sage2gpu_reads_bytes.argtypes = [vp, u64p]
        lib.sage2gpu_get_reads.argtypes = [vp, vp, vp, vp, vp, vp]
        lib.sage2gpu_get_extensions.argtypes = [vp, vp, vp, vp]
        lib.sage2gpu_get_edges.argtypes = [vp, vp, C.c_uint64, u64p]
        lib.sage2gpu_get_edges_packed.argtypes = [vp, vp, C.c_uint64, u64p]
        lib.sage2gpu_write_reads.argtypes = [vp, C.c_char_p]
        lib.sage2gpu_write_graph3.argtypes = [vp, C.c_char_p]
        lib.sage2gpu_write_gfa.argtypes = [vp, C.c_char_p]
        lib.sage2gpu_measure_gather.argtypes = [vp, C.c_uint64, C.c_int, C.c_uint64, C.c_int, C.POINTER(C.c_double)]
        lib.sage2gpu_load_reads_partition.argtypes = [vp, vp, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, u64p]
        lib.sage2gpu_pack_slice.argtypes = [vp, vp, vp, i64, C.c_int, C.c_int, C.c_int, u64p, u64p, u64p]
        lib.sage2gpu_raw_gather_layout.argtypes = [vp, C.c_int, C.c_int, u64p, C.POINTER(vp), u64p, u64p]
        lib.sage2gpu_raw_gather_finish.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64]
        lib.sage2gpu_organize_partition.argtypes = [vp, C.c_int, C.c_int, u64p]
        lib.sage2gpu_synth_reads.argtypes = [vp, vp, vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_float, C.c_float, C.c_uint64]
        lib.sage2gpu_reads_gather_layout.argtypes = [vp, u64p, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), u64p, u64p, u64p]
        lib.sage2gpu_reads_gather_finish.argtypes = [vp]
        lib.sage2gpu_build_hash_table_part.argtypes = [vp, C.c_int, C.c_int]
        lib.sage2gpu_table_shard_info.argtypes = [vp, u64p, u64p, u64p, u64p]
        lib.sage2gpu_table_gather_layout.argtypes = [vp, u64p, C.POINTER(vp), C.POINTER(vp), u64p, u64p]
        lib.sage2gpu_table_gather_finish.argtypes = [vp, u64p, u64p, u64p]
        lib.sage2gpu_digest.argtypes = [vp, u64p, u64p]
        lib.sage2gpu_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
        lib.sage2gpu_stream.argtypes = [vp]
        lib.sage2gpu_stream.restype = vp
        lib.sage2gpu_kernel_launches.argtypes = []
        lib.sage2gpu_kernel_launches.restype = C.c_uint64
        _lib = lib
    return _lib


def kernel_launches() -> int:
    """CUDA kernels launched by libsage2gpu in this process so far."""
    return int(load_library().sage2gpu_kernel_launches())


class Sage2Gpu:
    """One libsage2gpu context = one GPU."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        self._h = C.c_void_p()
        rc = self._lib.sage2gpu_create(C.byref(self._h), device)
        if rc != 0:
            raise Sage2GpuError(f"sage2gpu_create(device={device}) failed with code {rc}: no usable CUDA device "
                                "(libsage2gpu has no CPU fallback)")
        self._keep = None

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.sage2gpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str, bad_line: int = 0):
        if rc != 0:
            msg = self._lib.sage2gpu_last_error(self._h)
            err = Sage2GpuError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
            err.code, err.bad_line = rc, int(bad_line)
            raise err

    # ---- steps --------------------------------------------------------------------------------
    def load_reads(self, bases: np.ndarray, offsets: np.ndarray, min_overlap: int):
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self._keep = (bases, offsets)
        self._check(self._lib.sage2gpu_load_reads(self._h, bases.ctypes.data, offsets.ctypes.data,
                                                  len(offsets) - 1, int(min_overlap)), "load_reads")

    def load_reads_ptr(self, bases_ptr: int, offsets_ptr: int, n_reads: int, min_overlap: int, device: bool):
        fn = self._lib.sage2gpu_load_reads_device if device else self._lib.sage2gpu_load_reads
        self._check(fn(self._h, bases_ptr, offsets_ptr, int(n_reads), int(min_overlap)), "load_reads")

    def load_reads_chunked(self, bases: np.ndarray, offsets: np.ndarray, min_overlap: int, reads_per_chunk: int):
        """Streamed upload (sage2gpu_load_begin/_append/_finish); same result as load_reads."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self._keep = (bases, offsets)
        n = len(offsets) - 1
        self._check(self._lib.sage2gpu_load_begin(self._h, int(min_overlap)), "load_begin")
        for r0 in range(0, n, reads_per_chunk):
            r1 = min(n, r0 + reads_per_chunk)
            self._check(self._lib.sage2gpu_load_append(self._h, bases.ctypes.data, offsets[r0:r1 + 1].ctypes.data, r1 - r0),
                        "load_append")
        self._check(self._lib.sage2gpu_load_finish(self._h), "load_finish")

    def load_begin(self, min_overlap: int):
        self._check(self._lib.sage2gpu_load_begin(self._h, int(min_overlap)), "load_begin")

    def inflate_bgzf(self, data: bytes, text_capacity: int = -1):
        """The BGZF members of `data` inflated on the device: (text bytes, kernel ms).  A member that fails a check raises
        Sage2GpuError with code ERR_FORMAT and `bad_member` = its index."""
        src = np.frombuffer(bytes(data), np.uint8)
        n_out, bad, ms = C.c_uint64(), C.c_int64(-1), C.c_float()
        if text_capacity < 0:       # sizing: ISIZE sums come from the headers, nothing is inflated for a 0-byte buffer
            self._lib.sage2gpu_inflate_bgzf(self._h, src.ctypes.data, len(src), None, 0, C.byref(n_out), C.byref(bad), None)
            text_capacity = n_out.value
        out = np.empty(max(1, text_capacity), np.uint8)
        rc = self._lib.sage2gpu_inflate_bgzf(self._h, src.ctypes.data, len(src), out.ctypes.data, text_capacity, C.byref(n_out),
                                             C.byref(bad), C.byref(ms))
        self._check_bgzf(rc, "inflate_bgzf", bad.value)
        return out[:n_out.value].tobytes(), float(ms.value)

    def load_append_bgzf(self, prefix: bytes, data: bytes, is_final: bool, marker: int = 0, max_records: int = (1 << 64) - 1,
                         rest_capacity: int = 1 << 26):
        """One piece of whole BGZF members after the host text `prefix` (sage2gpu_load_append_bgzf).  Returns a dict with
        marker, consumed, n_records and rest (the text the next piece takes as its prefix)."""
        pre = np.frombuffer(bytes(prefix) or b"\0", np.uint8)
        src = np.frombuffer(bytes(data) or b"\0", np.uint8)
        rest = np.empty(max(1, rest_capacity), np.uint8)
        mk, used, nrec, nrest, bad = C.c_int(marker), C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_int64(-1)
        rc = self._lib.sage2gpu_load_append_bgzf(self._h, pre.ctypes.data, len(prefix), src.ctypes.data, len(data), int(bool(is_final)),
                                                 C.byref(mk), max_records, C.byref(used), C.byref(nrec), rest.ctypes.data, rest_capacity,
                                                 C.byref(nrest), C.byref(bad))
        self._check_bgzf(rc, "load_append_bgzf", bad.value)
        return {"marker": mk.value, "consumed": used.value, "n_records": nrec.value,
                "rest": rest[:min(nrest.value, rest_capacity)].tobytes()}

    def inflate_gzip(self, data: bytes, text_capacity: int = -1):
        """A whole gzip stream inflated on the device (sage2gpu_inflate_gzip): (text bytes, kernel ms, ranges decoded, ranges
        confirmed, candidates rejected).  Data that fails a check raises Sage2GpuError with code ERR_FORMAT and `bad_offset` =
        the compressed offset of the member or block."""
        src = np.frombuffer(bytes(data) or b"\0", np.uint8)
        cap = text_capacity if text_capacity >= 0 else 4 * len(data) + (1 << 20)
        while True:
            out = np.empty(max(1, cap), np.uint8)
            n_out, bad, ms, nr, conf, rej = C.c_uint64(), C.c_int64(-1), C.c_float(), C.c_uint64(), C.c_uint64(), C.c_uint64()
            rc = self._lib.sage2gpu_inflate_gzip(self._h, src.ctypes.data, len(data), out.ctypes.data, cap, C.byref(n_out), C.byref(bad),
                                                 C.byref(ms), C.byref(nr), C.byref(conf), C.byref(rej))
            if rc == ERR_STATE and text_capacity < 0 and b"smaller than the text" in (self._lib.sage2gpu_last_error(self._h) or b""):
                cap *= 4
                continue
            self._check_gzip(rc, "inflate_gzip", bad.value)
            return out[:n_out.value].tobytes(), float(ms.value), nr.value, conf.value, rej.value

    def load_append_gzip(self, prefix: bytes, data: bytes, is_final: bool, state: "GzipState", text_bound: int, marker: int = 0,
                         max_records: int = (1 << 64) - 1, rest_capacity: int = 1 << 26):
        """One piece of a gzip stream after the host text `prefix` (sage2gpu_load_append_gzip): `data` = the compressed bytes from
        state.offset on, `state` moves to where the next piece starts.  Returns a dict with marker, consumed, n_records, rest and
        in_consumed (compressed bytes the state moved past)."""
        pre = np.frombuffer(bytes(prefix) or b"\0", np.uint8)
        src = np.frombuffer(bytes(data) or b"\0", np.uint8)
        rest = np.empty(max(1, rest_capacity), np.uint8)
        mk, used, nrec, nrest, nin, bad = C.c_int(marker), C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_int64(-1)
        rc = self._lib.sage2gpu_load_append_gzip(self._h, pre.ctypes.data, len(prefix), src.ctypes.data, len(data), int(bool(is_final)),
                                                 text_bound, C.byref(state), C.byref(mk), max_records, C.byref(used), C.byref(nrec),
                                                 rest.ctypes.data, rest_capacity, C.byref(nrest), C.byref(nin), C.byref(bad))
        self._check_gzip(rc, "load_append_gzip", bad.value)
        return {"marker": mk.value, "consumed": used.value, "n_records": nrec.value,
                "rest": rest[:min(nrest.value, rest_capacity)].tobytes(), "in_consumed": nin.value}

    def _check_gzip(self, rc: int, what: str, bad_offset: int):
        try:
            self._check(rc, what)
        except Sage2GpuError as e:
            e.bad_offset = int(bad_offset)
            raise

    def _check_bgzf(self, rc: int, what: str, bad_member: int):
        try:
            self._check(rc, what)
        except Sage2GpuError as e:
            e.bad_member = int(bad_member)
            raise

    def load_count(self) -> int:
        n = C.c_uint64()
        self._check(self._lib.sage2gpu_load_count(self._h, C.byref(n)), "load_count")
        return n.value

    def load_append(self, bases: np.ndarray, offsets: np.ndarray):
        """One chunk of a streamed upload: read r = bases[offsets[r], offsets[r+1]).  The buffers are kept alive until the
        next call on this context (the library may still be copying them)."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self._keep = (bases, offsets)
        self._check(self._lib.sage2gpu_load_append(self._h, bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1), "load_append")

    # ---- restart from a saved .reads file (ReadLoader::loadReadsFromFile, readLoader.cpp:289) ---------------------------
    def load_saved_reads(self, path: str, min_overlap: int):
        """The reads of a saved .reads file (what write_reads / the reference's saveReadsInFile write), parsed and checked on the
        device.  A file that breaks the grammar raises Sage2GpuError with code ERR_FORMAT; the message names the line."""
        self._check(self._lib.sage2gpu_load_saved_reads(self._h, path.encode(), int(min_overlap)), "load_saved_reads")

    def saved_reads_info(self, path: str) -> tuple:
        """(U of the first line, bytes of the body)."""
        u, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_saved_reads_info(self._h, path.encode(), C.byref(u), C.byref(b)), "saved_reads_info")
        return int(u.value), int(b.value)

    def saved_reads_slice(self, path: str, min_overlap: int, byte_begin: int, byte_end: int) -> dict:
        """The lines whose first byte lies in [byte_begin, byte_end) of the body; on a format error `bad_line` counts from the
        slice's first line."""
        n, m, bad = C.c_uint64(), C.c_int(), C.c_uint64()
        rc = self._lib.sage2gpu_saved_reads_slice(self._h, path.encode(), int(min_overlap), int(byte_begin), int(byte_end), C.byref(n),
                                                  C.byref(m), C.byref(bad))
        self._check(rc, "saved_reads_slice", bad.value)
        return {"n_lines": int(n.value), "max_read_length": int(m.value)}

    def saved_reads_pack(self, rank: int, world: int, max_read_length: int) -> dict:
        u, g, b = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_saved_reads_pack(self._h, int(rank), int(world), int(max_read_length), C.byref(u), C.byref(g), C.byref(b)),
                    "saved_reads_pack")
        return {"unique_local": int(u.value), "good_reads": int(g.value), "total_bp": int(b.value)}

    def saved_reads_finish(self, n_reads: int, good_reads: int, total_bp: int):
        bad = C.c_uint64()
        rc = self._lib.sage2gpu_saved_reads_finish(self._h, int(n_reads), int(good_reads), int(total_bp), C.byref(bad))
        self._check(rc, "saved_reads_finish", bad.value)

    def load_max_length(self) -> int:
        """Longest read appended since load_begin (nothing is packed)."""
        m = C.c_int()
        self._check(self._lib.sage2gpu_load_max_length(self._h, C.byref(m)), "load_max_length")
        return int(m.value)

    def load_finish_slice(self, max_read_length: int) -> dict:
        """The streamed upload packed as this context's slice, at the stride of the read set's longest read (as pack_slice)."""
        n, g, b, w = (C.c_uint64() for _ in range(4))
        self._check(self._lib.sage2gpu_load_finish_slice(self._h, int(max_read_length), C.byref(n), C.byref(g), C.byref(b), C.byref(w)),
                    "load_finish_slice")
        return {"n_reads": int(n.value), "good_reads": int(g.value), "total_bp": int(b.value), "record_words": int(w.value)}

    def table_bytes(self, world: int) -> dict:
        """Bytes of the table this context would hold with `world` contexts, replicated or sharded (slots exact, entries an
        upper bound), and the free memory of its GPU."""
        v = [C.c_uint64() for _ in range(5)]
        self._check(self._lib.sage2gpu_table_bytes(self._h, int(world), *(C.byref(x) for x in v)), "table_bytes")
        return {"replicated_slots": int(v[0].value), "replicated_entries": int(v[1].value), "sharded_slots": int(v[2].value),
                "sharded_entries": int(v[3].value), "device_free": int(v[4].value)}

    def build_hash_table(self):
        self._check(self._lib.sage2gpu_build_hash_table(self._h), "build_hash_table")

    def build_overlap_graph(self):
        self._check(self._lib.sage2gpu_build_overlap_graph(self._h), "build_overlap_graph")

    def phase_a_partition(self, rank: int, world: int):
        self._check(self._lib.sage2gpu_phase_a_partition(self._h, int(rank), int(world)), "phase_a_partition")

    def phase_a_buffers(self) -> dict:
        """Device pointers of the phase-A arrays (length world*chunk) for the multi-GPU exchange."""
        p = [C.c_void_p() for _ in range(4)]
        chunk, U = C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_phase_a_buffers(self._h, *(C.byref(x) for x in p), C.byref(chunk), C.byref(U)),
                    "phase_a_buffers")
        return {"right": p[0].value or 0, "left": p[1].value or 0, "over_limit": p[2].value or 0,
                "contained_by": p[3].value or 0, "chunk": int(chunk.value), "unique_reads": int(U.value)}

    def finish_graph(self):
        self._check(self._lib.sage2gpu_finish_graph(self._h), "finish_graph")

    def table_view(self) -> dict:
        """Device pointers and sizes of the table this context holds: "slots" (uint64 x n_slots, `shards` shards of
        sectors_per_shard sectors of 4 slots) and "entries" (uint32 x n_entries)."""
        ps, pe = C.c_void_p(), C.c_void_p()
        v = [C.c_uint64() for _ in range(4)]
        self._check(self._lib.sage2gpu_table_view(self._h, C.byref(ps), C.byref(v[0]), C.byref(pe), C.byref(v[1]), C.byref(v[2]), C.byref(v[3])),
                    "table_view")
        return {"slots": ps.value or 0, "n_slots": int(v[0].value), "entries": pe.value or 0, "n_entries": int(v[1].value),
                "sectors_per_shard": int(v[2].value), "shards": int(v[3].value)}

    # ---- several GPUs, every stage partitioned (include/sage2gpu.h) --------------------------------------------
    def load_reads_partition(self, bases_ptr: int, offsets_ptr: int, n_reads: int, min_overlap: int, device: bool, rank: int, world: int) -> int:
        """organizeReads for this rank's key range; returns its number of unique reads."""
        u = C.c_uint64()
        self._check(self._lib.sage2gpu_load_reads_partition(self._h, bases_ptr, offsets_ptr, int(n_reads), int(min_overlap), int(bool(device)),
                                                            int(rank), int(world), C.byref(u)), "load_reads_partition")
        return int(u.value)

    def pack_slice(self, bases_ptr: int, offsets_ptr: int, n_reads: int, min_overlap: int, device: bool, max_read_length: int) -> dict:
        g, b, w = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_pack_slice(self._h, bases_ptr, offsets_ptr, int(n_reads), int(min_overlap), int(bool(device)),
                                                  int(max_read_length), C.byref(g), C.byref(b), C.byref(w)), "pack_slice")
        return {"good_reads": int(g.value), "total_bp": int(b.value), "record_words": int(w.value)}

    def raw_gather_layout(self, rank: int, world: int, counts) -> dict:
        cs = (C.c_uint64 * len(counts))(*[int(x) for x in counts])
        p = C.c_void_p()
        first, total = C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_raw_gather_layout(self._h, int(rank), int(world), cs, C.byref(p), C.byref(first), C.byref(total)),
                    "raw_gather_layout")
        return {"records": p.value or 0, "first": int(first.value), "total": int(total.value)}

    def raw_gather_finish(self, total_reads: int, good_reads: int, total_bp: int):
        self._check(self._lib.sage2gpu_raw_gather_finish(self._h, int(total_reads), int(good_reads), int(total_bp)), "raw_gather_finish")

    def organize_partition(self, rank: int, world: int) -> int:
        u = C.c_uint64()
        self._check(self._lib.sage2gpu_organize_partition(self._h, int(rank), int(world), C.byref(u)), "organize_partition")
        return int(u.value)

    def synth_reads(self, bases_ptr: int, offsets_ptr: int, first_pair: int, n_pairs: int, genome_bp: int, read_length: int,
                    insert_mean: float = 450.0, insert_sd: float = 30.0, seed: int = 1):
        self._check(self._lib.sage2gpu_synth_reads(self._h, bases_ptr, offsets_ptr, int(first_pair), int(n_pairs), int(genome_bp), int(read_length),
                                                   float(insert_mean), float(insert_sd), int(seed)), "synth_reads")

    def reads_gather_layout(self, counts) -> dict:
        cs = (C.c_uint64 * len(counts))(*[int(x) for x in counts])
        p = [C.c_void_p() for _ in range(3)]
        first, total, stride = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_reads_gather_layout(self._h, cs, *(C.byref(x) for x in p), C.byref(first), C.byref(total), C.byref(stride)),
                    "reads_gather_layout")
        return {"records": p[0].value or 0, "lengths": p[1].value or 0, "frequencies": p[2].value or 0, "first": int(first.value),
                "total": int(total.value), "stride": int(stride.value), "counts": [int(x) for x in counts]}

    def reads_gather_finish(self):
        self._check(self._lib.sage2gpu_reads_gather_finish(self._h), "reads_gather_finish")

    def build_hash_table_part(self, rank: int, world: int):
        self._check(self._lib.sage2gpu_build_hash_table_part(self._h, int(rank), int(world)), "build_hash_table_part")

    def table_shard_info(self) -> dict:
        v = [C.c_uint64() for _ in range(4)]
        self._check(self._lib.sage2gpu_table_shard_info(self._h, *(C.byref(x) for x in v)), "table_shard_info")
        return {"slots": int(v[0].value), "entries": int(v[1].value), "distinct": int(v[2].value), "over": int(v[3].value)}

    def table_gather_layout(self, entry_counts) -> dict:
        cs = (C.c_uint64 * len(entry_counts))(*[int(x) for x in entry_counts])
        ps, pe = C.c_void_p(), C.c_void_p()
        sps, ef = C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_table_gather_layout(self._h, cs, C.byref(ps), C.byref(pe), C.byref(sps), C.byref(ef)), "table_gather_layout")
        return {"slots": ps.value or 0, "entries": pe.value or 0, "slots_per_shard": int(sps.value), "entries_first": int(ef.value)}

    def table_gather_finish(self, entry_counts, distinct, over):
        mk = lambda a: (C.c_uint64 * len(a))(*[int(x) for x in a])
        self._check(self._lib.sage2gpu_table_gather_finish(self._h, mk(entry_counts), mk(distinct), mk(over)), "table_gather_finish")

    # ---- sharded table (include/sage2gpu.h, "The table sharded by key hash") ----------------------------------
    def build_hash_table_shard(self, rank: int, world: int):
        self._check(self._lib.sage2gpu_build_hash_table_shard(self._h, int(rank), int(world)), "build_hash_table_shard")

    def phase_a_sharded_begin(self, rank: int, world: int) -> tuple:
        """(first, count): this rank's slice of the unique reads (0-based indices)."""
        first, count = C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_phase_a_sharded_begin(self._h, int(rank), int(world), C.byref(first), C.byref(count)),
                    "phase_a_sharded_begin")
        return int(first.value), int(count.value)

    def route_begin(self, what: int, first: int, count: int, exact: bool, world: int) -> dict:
        """-> {"ptr": device pointer of the query streams, "counts": queries per owner, "words": uint64 per query,
        "n_reads": reads in the batch}."""
        q = C.c_void_p()
        counts = (C.c_uint64 * world)()
        n = C.c_uint64()
        self._check(self._lib.sage2gpu_route_begin(self._h, int(what), int(first), int(count), int(bool(exact)), int(world),
                                                   C.byref(q), counts, C.byref(n)), "route_begin")
        return {"ptr": q.value or 0, "counts": [int(x) for x in counts], "words": 2 if exact else 1, "n_reads": int(n.value)}

    def shard_answer(self, queries_ptr: int, counts_per_source, exact: bool, world: int) -> dict:
        """-> {"resp": device pointer (uint64 per query), "entries": device pointer (uint32), "entry_counts": per source}."""
        cps = (C.c_uint64 * world)(*[int(x) for x in counts_per_source])
        resp, ent = C.c_void_p(), C.c_void_p()
        ecnt = (C.c_uint64 * world)()
        self._check(self._lib.sage2gpu_shard_answer(self._h, queries_ptr or None, cps, int(bool(exact)), int(world), C.byref(resp),
                                                    C.byref(ent), ecnt), "shard_answer")
        return {"resp": resp.value or 0, "entries": ent.value or 0, "entry_counts": [int(x) for x in ecnt]}

    def route_finish(self, resp_ptr: int, entries_ptr: int, entry_counts):
        ec = (C.c_uint64 * len(entry_counts))(*[int(x) for x in entry_counts])
        self._check(self._lib.sage2gpu_route_finish(self._h, resp_ptr or None, entries_ptr or None, ec), "route_finish")

    # ---- the same exchange over peer memory (mailboxes) ------------------------------------------------------------
    def mailbox_create(self, rank: int, world: int, max_reads_per_batch: int) -> dict:
        """-> {"handle": the 64-byte CUDA IPC handle (bytes), "ptr": the mailbox's device pointer (same-process peers)}."""
        h = (C.c_char * 64)()
        p = C.c_void_p()
        self._check(self._lib.sage2gpu_mailbox_create(self._h, int(rank), int(world), int(max_reads_per_batch), h, C.byref(p)), "mailbox_create")
        self.mailbox_batch_reads = int(max_reads_per_batch)
        return {"handle": bytes(h.raw), "ptr": p.value or 0}

    def mailbox_open(self, peer_rank: int, handle: bytes | None = None, ptr: int = 0):
        self._check(self._lib.sage2gpu_mailbox_open(self._h, int(peer_rank), handle if handle else None, ptr or None), "mailbox_open")

    def route_post(self, what: int, first: int, count: int, exact: bool) -> tuple:
        """-> (reads in the batch, bytes stored into other ranks' mailboxes)."""
        n, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_route_post(self._h, int(what), int(first), int(count), int(bool(exact)), C.byref(n), C.byref(b)), "route_post")
        return int(n.value), int(b.value)

    def answer_post(self, exact: bool) -> int:
        b = C.c_uint64()
        self._check(self._lib.sage2gpu_answer_post(self._h, int(bool(exact)), C.byref(b)), "answer_post")
        return int(b.value)

    def mailbox_barrier(self):
        self._check(self._lib.sage2gpu_mailbox_barrier(self._h), "mailbox_barrier")

    def route_collect(self):
        self._check(self._lib.sage2gpu_route_collect(self._h), "route_collect")

    def phase_a_routed(self) -> int:
        n = C.c_uint64()
        self._check(self._lib.sage2gpu_phase_a_routed(self._h, C.byref(n)), "phase_a_routed")
        return int(n.value)

    def phase_a_sharded_end(self):
        self._check(self._lib.sage2gpu_phase_a_sharded_end(self._h), "phase_a_sharded_end")

    def phase_b(self):
        self._check(self._lib.sage2gpu_phase_b(self._h), "phase_b")

    def map_reads(self, bases: np.ndarray, offsets: np.ndarray):
        """getIdOfRead of every read (readLoader.cpp:319-353): (signed ids int64, isGoodRead uint8, kernel ms)."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n = len(offsets) - 1
        ids, good, ms = np.zeros(n, np.int64), np.zeros(n, np.uint8), C.c_float()
        self._check(self._lib.sage2gpu_map_reads(self._h, bases.ctypes.data, offsets.ctypes.data, n, 0, ids.ctypes.data,
                                                 good.ctypes.data, C.byref(ms)), "map_reads")
        return ids, good, float(ms.value)

    def map_reads_ptr(self, bases_ptr: int, offsets_ptr: int, n: int, ids_ptr: int, good_ptr: int, device: bool) -> float:
        ms = C.c_float()
        self._check(self._lib.sage2gpu_map_reads(self._h, bases_ptr, offsets_ptr, int(n), int(bool(device)), ids_ptr, good_ptr or None,
                                                 C.byref(ms)), "map_reads")
        return float(ms.value)

    def run_steps123(self, bases, offsets, min_overlap: int):
        self.load_reads(bases, offsets, min_overlap)
        self.build_hash_table()
        self.build_overlap_graph()

    def measure_gather(self, footprint_bytes: int, granule_bytes: int = 32, n_loads: int = 1 << 28, mode: int = 0) -> float:
        """GB/s of random `granule_bytes` gathers over `footprint_bytes` (the random-sector roofline)."""
        g = C.c_double()
        self._check(self._lib.sage2gpu_measure_gather(self._h, int(footprint_bytes), int(granule_bytes), int(n_loads),
                                                      int(mode), C.byref(g)), "measure_gather")
        return float(g.value)

    def stream_ptr(self) -> int:
        """cudaStream_t of this context (e.g. for torch.cuda.ExternalStream)."""
        return int(self._lib.sage2gpu_stream(self._h) or 0)

    # ---- results ------------------------------------------------------------------------------
    def counters(self) -> dict:
        c = Counters()
        self._check(self._lib.sage2gpu_get_counters(self._h, C.byref(c)), "get_counters")
        return {n: int(getattr(c, n)) for n, _ in Counters._fields_}

    def timers(self) -> dict:
        t = Timers()
        self._check(self._lib.sage2gpu_get_timers(self._h, C.byref(t)), "get_timers")
        return {n: float(getattr(t, n)) for n, _ in Timers._fields_}

    def reads(self) -> dict:
        U = self.counters()["unique_reads"]
        nb = C.c_uint64()
        self._check(self._lib.sage2gpu_reads_bytes(self._h, C.byref(nb)), "reads_bytes")
        out = dict(length=np.zeros(U, np.uint16), frequency=np.zeros(U, np.uint16),
                   byte_off=np.zeros(U + 1, np.uint64), fwd=np.zeros(nb.value, np.uint8), rc=np.zeros(nb.value, np.uint8))
        self._check(self._lib.sage2gpu_get_reads(self._h, out["length"].ctypes.data, out["frequency"].ctypes.data,
                                                 out["byte_off"].ctypes.data, out["fwd"].ctypes.data,
                                                 out["rc"].ctypes.data), "get_reads")
        return out

    def extensions(self) -> dict:
        U = self.counters()["unique_reads"]
        out = dict(right=np.zeros(U, np.uint64), left=np.zeros(U, np.uint64), explored=np.zeros(U, np.uint8))
        self._check(self._lib.sage2gpu_get_extensions(self._h, out["right"].ctypes.data, out["left"].ctypes.data,
                                                      out["explored"].ctypes.data), "get_extensions")
        return out

    def edges(self) -> np.ndarray:
        n = C.c_uint64()
        self._check(self._lib.sage2gpu_get_edges(self._h, None, 0, C.byref(n)), "get_edges")
        out = np.zeros(n.value, dtype=EDGE_DT)
        if n.value:
            self._check(self._lib.sage2gpu_get_edges(self._h, out.ctypes.data, n.value, C.byref(n)), "get_edges")
        return out

    def edges_packed_into(self, out_ptr: int, capacity: int) -> int:
        """Raw (w0, w1) edge words straight into a caller buffer (e.g. pinned); returns the edge count."""
        n = C.c_uint64()
        self._check(self._lib.sage2gpu_get_edges_packed(self._h, out_ptr, int(capacity), C.byref(n)), "get_edges_packed")
        return int(n.value)

    def digest(self, reads: bool = True, edges: bool = True) -> dict:
        """Order-sensitive digests of the resident reads / edge list (definitions: tests/digest.py)."""
        r, e = C.c_uint64(), C.c_uint64()
        self._check(self._lib.sage2gpu_digest(self._h, C.byref(r) if reads else None, C.byref(e) if edges else None), "digest")
        return {"reads": int(r.value) if reads else None, "edges": int(e.value) if edges else None}

    def set_option(self, name: str, value: int):
        self._check(self._lib.sage2gpu_set_option(self._h, name.encode(), int(value)), "set_option")

    def write_reads(self, path: str):
        self._check(self._lib.sage2gpu_write_reads(self._h, path.encode()), "write_reads")

    def write_graph3(self, path: str):
        self._check(self._lib.sage2gpu_write_graph3(self._h, path.encode()), "write_graph3")

    def write_gfa(self, path: str):
        """The reads and the overlap graph as GFA 1.0 (one S line per read, one L line per edge; include/sage2gpu.h), formatted
        on the device.  Sage2GpuError with code ERR_STATE before build_overlap_graph, ERR_IO when the file cannot be written."""
        self._check(self._lib.sage2gpu_write_gfa(self._h, path.encode()), "write_gfa")


# ---- mirrors of the reference's step 1-3 classes (main.cpp:37-132) ---------------------------------

class ReadLoader:
    """inputReader/readLoader.h:32-56."""

    def __init__(self, minOvlp: int, device: int = 0):
        self.minOverlap = int(minOvlp)
        self.gpu = Sage2Gpu(device)
        self.numberOfReads = self.numberOfUniqueReads = self.totalBP = 0
        self._pending = None

    def readDatasetInBytes(self, reads):
        """`reads`: list[bytes] / (N,L) uint8 array of sequences (the FASTQ parse is the caller's)."""
        from . import synth
        self._pending = synth.concat(reads)

    def organizeReads(self):
        bases, offsets = self._pending
        self.gpu.load_reads(bases, offsets, self.minOverlap)
        c = self.gpu.counters()
        self.numberOfReads, self.numberOfUniqueReads, self.totalBP = c["good_reads"], c["unique_reads"], c["total_bp"]
        self.averageReadLength = c["avg_len"]

    def saveReadsInFile(self, path: str):
        self.gpu.write_reads(path)

    def loadReadsFromFile(self, path: str):
        """readLoader.cpp:289: the reads of a saved .reads file (SAGE2 -m 2 / -m 3) instead of readDatasetInBytes + organizeReads.
        numberOfReads is the sum of the file's frequencies (each a uint16_t count, wrapped at 65,536 copies)."""
        self.gpu.load_saved_reads(path, self.minOverlap)
        c = self.gpu.counters()
        self.numberOfReads, self.numberOfUniqueReads, self.totalBP = c["good_reads"], c["unique_reads"], c["total_bp"]
        self.averageReadLength = c["avg_len"]

    def getIdOfRead(self, reads):
        """readLoader.cpp:319-353 for a batch: signed ids (0 = absent; bad reads, which step 6 never looks up, give 0)."""
        from . import synth
        b, off = synth.concat(reads)
        return self.gpu.map_reads(b, off)[0]


class HashTable:
    """economyGraph/hashTable.h:20-44."""

    def __init__(self, minOvlp: int, loader: ReadLoader):
        self.minOverlap, self.loaderObj = int(minOvlp), loader

    def hashPrefixesAndSuffix(self):
        self.loaderObj.gpu.build_hash_table()
        c = self.loaderObj.gpu.counters()
        self.hashStringLength, self.sizeOfHashTable = c["hash_len"], c["table_capacity"]


class EconomyGraph:
    """economyGraph/economyGraph.h:32-54; the three calls of main.cpp:109-114 map onto one device pass."""

    def __init__(self, minOvlp: int, hash1: HashTable):
        self.minOverlap, self.hashObj, self.loaderObj = int(minOvlp), hash1, hash1.loaderObj
        self._built = False

    def buildInitialOverlapGraph(self):
        self.loaderObj.gpu.build_overlap_graph()
        self._built = True

    def buildOverlapGraphEconomy(self):
        if not self._built:
            raise Sage2GpuError("buildInitialOverlapGraph must run first (main.cpp:109-111)")

    def sortEconomyGraph(self):
        if not self._built:
            raise Sage2GpuError("buildInitialOverlapGraph must run first")

    def saveOverlapGraphInFile(self, path: str):
        """OverlapGraph::convertGraph + saveOverlapGraphInFile (overlapGraph.cpp:84-115,338-369)."""
        self.loaderObj.gpu.write_graph3(path)
