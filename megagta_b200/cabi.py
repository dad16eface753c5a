"""ctypes binding of libmgta_cuda.so (include/mgta_cuda.h).  There is no fallback: if the library is
missing or no CUDA device is present, loading / context creation raises."""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libmgta_cuda.so")
NUM_BUCKETS = 65536


class MgtaError(RuntimeError):
    pass


class Opts(ctypes.Structure):
    _fields_ = [("kmer_k", ctypes.c_int32), ("min_count", ctypes.c_int32), ("need_mercy", ctypes.c_int32),
                ("device", ctypes.c_int32), ("rank", ctypes.c_int32), ("world", ctypes.c_int32),
                ("hbm_budget_bytes", ctypes.c_int64), ("stream", ctypes.c_void_p),
                ("sort_items_cap", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class StageStats(ctypes.Structure):
    _fields_ = [("n_items", ctypes.c_uint64), ("n_batches", ctypes.c_uint64), ("n_launches", ctypes.c_uint64),
                ("n_giants", ctypes.c_uint64), ("out_bytes", ctypes.c_uint64), ("n_edges", ctypes.c_uint64),
                ("ms_total", ctypes.c_float), ("ms_hist", ctypes.c_float), ("ms_extract", ctypes.c_float),
                ("ms_partition", ctypes.c_float), ("ms_sort_emit", ctypes.c_float),
                ("key_words", ctypes.c_int32), ("item_words", ctypes.c_int32), ("sort_cap", ctypes.c_int32),
                ("msd_levels", ctypes.c_int32), ("ms_nodes", ctypes.c_float), ("reserved", ctypes.c_int32),
                ("n_node_ops", ctypes.c_uint64), ("n_tip_items", ctypes.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class Collective(ctypes.Structure):
    """mgta_collective: the exchange the library asks the caller to run among the shards (include/mgta_cuda.h)"""
    _fields_ = [("op", ctypes.c_int32), ("reserved", ctypes.c_int32), ("send", ctypes.c_void_p), ("recv", ctypes.c_void_p),
                ("bytes", ctypes.c_uint64)]


COLL_NONE, COLL_ALL_TO_ALL, COLL_ALL_GATHER, COLL_ALL_REDUCE_SUM_U32, COLL_ALL_REDUCE_SUM_U64 = 0, 1, 2, 3, 4

SINK = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p,
                        ctypes.c_uint64, ctypes.POINTER(ctypes.c_int64))

EXPORTS = ["mgta_ctx_create", "mgta_ctx_destroy", "mgta_last_error", "mgta_set_reads", "mgta_set_reads_async", "mgta_alloc_reads",
           "mgta_reads_device_buffers", "mgta_stage1_histogram",
           "mgta_stage2_histogram", "mgta_stage1", "mgta_solid_device_buffer", "mgta_get_is_solid", "mgta_set_is_solid",
           "mgta_get_mercy_candidates", "mgta_get_num_mercy", "mgta_stage2", "mgta_shard_range", "mgta_get_stats", "mgta_words_per_key",
           "mgta_abi_version", "mgta_sharded_begin", "mgta_sharded_step", "mgta_sharded_result",
           "mgta_sdbg_create", "mgta_sdbg_destroy", "mgta_sdbg_last_error", "mgta_sdbg_append", "mgta_sdbg_sink", "mgta_sdbg_finish",
           "mgta_sdbg_header", "mgta_sdbg_array", "mgta_sdbg_copy", "mgta_stage2_into_sdbg", "mgta_pack_reads", "mgta_tools_last_error", "mgta_find_seeds"]

# include/mgta_sdbg_query.h: kept apart from EXPORTS, which mirrors include/mgta_cuda.h
QUERY_EXPORTS = ["mgta_sdbg_query_row_bytes", "mgta_sdbg_query"]
(SQ_LOOKUP, SQ_LABEL, SQ_FORWARD, SQ_BACKWARD, SQ_OUTDEGREE, SQ_INDEGREE, SQ_OUTGOING, SQ_INCOMING, SQ_MULTIPLICITY,
 SQ_REVCOMP) = range(1, 11)
# include/mgta_sdbg_unitig.h
UNITIG_EXPORTS = ["mgta_sdbg_unitigs", "mgta_sdbg_unitig_copy"]
UNITIG_CYCLE, UNITIG_SELF_RC = 1, 2
# include/mgta_sdbg_unitig_graph.h
UNITIG_GRAPH_EXPORTS = ["mgta_sdbg_unitig_links", "mgta_sdbg_unitig_link_copy"]


class SdbgHeader(ctypes.Structure):
    """mgta_sdbg_header_t"""
    _fields_ = [("size", ctypes.c_int64), ("kmer_k", ctypes.c_int32), ("words_per_tip_label", ctypes.c_int32),
                ("num_tips", ctypes.c_int64), ("num_large_mul", ctypes.c_int64), ("f", ctypes.c_int64 * 6), ("rank_f", ctypes.c_int64 * 6),
                ("w_freq", ctypes.c_int64 * 9), ("last_ones", ctypes.c_int64), ("tip_ones", ctypes.c_int64),
                ("n_minor", ctypes.c_int64), ("n_major", ctypes.c_int64)]


(SDBG_W, SDBG_LAST, SDBG_IS_TIP, SDBG_INVALID, SDBG_IS_MULTI_1, SDBG_EDGE_MULTI, SDBG_LARGE_EDGE, SDBG_LARGE_VALUE,
 SDBG_TIP_SEQ) = range(9)
(SDBG_W_MINOR, SDBG_W_MAJOR, SDBG_W_SELECT, SDBG_LAST_MINOR, SDBG_LAST_MAJOR, SDBG_LAST_SELECT, SDBG_TIP_MINOR,
 SDBG_TIP_MAJOR) = range(16, 24)

_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MgtaError("%s not built (run `python -c 'import __graft_entry__ as g; g.build()'`)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        lib.mgta_last_error.restype = ctypes.c_char_p
        lib.mgta_last_error.argtypes = [ctypes.c_void_p]
        lib.mgta_ctx_create.argtypes = [ctypes.POINTER(Opts), ctypes.POINTER(ctypes.c_void_p)]
        lib.mgta_ctx_destroy.argtypes = [ctypes.c_void_p]
        lib.mgta_ctx_destroy.restype = None
        lib.mgta_set_reads.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                       ctypes.c_uint64, ctypes.c_int32]
        lib.mgta_set_reads_async.argtypes = lib.mgta_set_reads.argtypes
        lib.mgta_alloc_reads.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64,
                                         ctypes.c_int32]
        lib.mgta_reads_device_buffers.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
                                                  ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_void_p),
                                                  ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_stage1_histogram.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        lib.mgta_stage2_histogram.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        lib.mgta_stage1.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        lib.mgta_solid_device_buffer.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
                                                 ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_get_is_solid.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
        lib.mgta_set_is_solid.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
        lib.mgta_get_mercy_candidates.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                                  ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_get_num_mercy.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_stage2.argtypes = [ctypes.c_void_p, SINK, ctypes.c_void_p, ctypes.c_void_p]
        lib.mgta_shard_range.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
        lib.mgta_get_stats.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(StageStats)]
        lib.mgta_sharded_begin.argtypes = [ctypes.c_void_p, ctypes.c_int, SINK, ctypes.c_void_p]
        lib.mgta_sharded_step.argtypes = [ctypes.c_void_p, ctypes.POINTER(Collective)]
        lib.mgta_sharded_result.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        lib.mgta_sdbg_create.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]
        lib.mgta_sdbg_destroy.argtypes = [ctypes.c_void_p]
        lib.mgta_sdbg_destroy.restype = None
        lib.mgta_sdbg_last_error.argtypes = [ctypes.c_void_p]
        lib.mgta_sdbg_last_error.restype = ctypes.c_char_p
        lib.mgta_sdbg_append.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]
        lib.mgta_sdbg_finish.argtypes = [ctypes.c_void_p]
        lib.mgta_sdbg_header.argtypes = [ctypes.c_void_p, ctypes.POINTER(SdbgHeader)]
        lib.mgta_sdbg_array.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                        ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_sdbg_copy.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64]
        lib.mgta_stage2_into_sdbg.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        lib.mgta_pack_reads.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64]
        lib.mgta_tools_last_error.restype = ctypes.c_char_p
        lib.mgta_find_seeds.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64,
                                        ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                        ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_sdbg_sink.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]
        lib.mgta_words_per_key.argtypes = [ctypes.c_int, ctypes.c_int]
        lib.mgta_sdbg_query_row_bytes.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_sdbg_query.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64]
        lib.mgta_sdbg_unitigs.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_uint64)]
        lib.mgta_sdbg_unitig_copy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64]
        lib.mgta_sdbg_unitig_links.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]
        lib.mgta_sdbg_unitig_link_copy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
        _lib = lib
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class Context:
    """One GPU / one lv1-bucket shard.  Thin object wrapper over the C ABI."""

    def __init__(self, k, min_count=2, need_mercy=False, device=0, rank=0, world=1, hbm_budget_bytes=0, stream=None,
                 sort_items_cap=0):
        self.lib = load()
        self.opts = Opts(k, min_count, int(need_mercy), device, rank, world, hbm_budget_bytes, stream, sort_items_cap, 0)
        self.h = ctypes.c_void_p()
        rc = self.lib.mgta_ctx_create(ctypes.byref(self.opts), ctypes.byref(self.h))
        if rc != 0:
            raise MgtaError("mgta_ctx_create: %s" % self.lib.mgta_last_error(None).decode())
        self.k, self.m = k, min_count
        self._reads = None

    def _check(self, rc, what):
        if rc != 0:
            raise MgtaError("%s failed (%d): %s" % (what, rc, self.lib.mgta_last_error(self.h).decode()))

    def close(self):
        if self.h:
            self.lib.mgta_ctx_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_reads(self, seq, start, n_short=None, max_len=None):
        seq = np.ascontiguousarray(seq, dtype=np.uint32)
        start = np.ascontiguousarray(start, dtype=np.uint64)
        n = len(start) - 1
        n_short = n if n_short is None else n_short
        if max_len is None:
            lens = np.diff(start[:n_short + 1].astype(np.int64))
            max_len = int(lens.max()) if len(lens) else 0
        self._reads = (seq, start)
        self.n_short, self.max_len = n_short, max_len
        self._check(self.lib.mgta_set_reads(self.h, _p(seq), len(seq), _p(start), n, n_short, max_len), "mgta_set_reads")

    def set_reads_async(self, seq_ptr, n_words, start_ptr, n_reads, n_short, max_len):
        """asynchronous upload from PINNED host memory given by address (the caller keeps the buffers alive and unchanged
        until the next stage / histogram call has returned); mgta_stage1 pipelines the extraction behind the copy"""
        self.n_short, self.max_len = n_short, max_len
        self._check(self.lib.mgta_set_reads_async(self.h, seq_ptr, n_words, start_ptr, n_reads, n_short, max_len),
                    "mgta_set_reads_async")

    def alloc_reads(self, n_words, n_reads, n_short, total_bases, max_len):
        self.n_short, self.max_len = n_short, max_len
        self._check(self.lib.mgta_alloc_reads(self.h, n_words, n_reads, n_short, total_bases, max_len), "mgta_alloc_reads")

    def reads_device_buffers(self):
        a, an, b, bn = ctypes.c_void_p(), ctypes.c_uint64(), ctypes.c_void_p(), ctypes.c_uint64()
        self._check(self.lib.mgta_reads_device_buffers(self.h, ctypes.byref(a), ctypes.byref(an), ctypes.byref(b),
                                                       ctypes.byref(bn)), "mgta_reads_device_buffers")
        return (a.value, an.value), (b.value, bn.value)

    def histogram(self, stage):
        h = np.zeros(NUM_BUCKETS, dtype=np.int64)
        fn = self.lib.mgta_stage1_histogram if stage == 1 else self.lib.mgta_stage2_histogram
        self._check(fn(self.h, _p(h)), "mgta_stage%d_histogram" % stage)
        return h

    def stage1(self):
        ec = np.zeros(NUM_BUCKETS, dtype=np.int64)
        self._check(self.lib.mgta_stage1(self.h, _p(ec)), "mgta_stage1")
        return ec

    def get_is_solid(self):
        n = (max(0, self.max_len - self.k) * self.n_short + 7) // 8
        buf = np.zeros(n + 8, dtype=np.uint8)
        self._check(self.lib.mgta_get_is_solid(self.h, _p(buf), len(buf)), "mgta_get_is_solid")
        return buf

    def set_is_solid(self, buf):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        self._check(self.lib.mgta_set_is_solid(self.h, _p(buf), len(buf)), "mgta_set_is_solid")

    def solid_device_buffer(self):
        p, n = ctypes.c_void_p(), ctypes.c_uint64()
        self._check(self.lib.mgta_solid_device_buffer(self.h, ctypes.byref(p), ctypes.byref(n)), "mgta_solid_device_buffer")
        return p.value, n.value

    def mercy_candidates(self):
        n = ctypes.c_uint64()
        self._check(self.lib.mgta_get_mercy_candidates(self.h, None, 0, ctypes.byref(n)), "mgta_get_mercy_candidates")
        out = np.empty(n.value, dtype=np.uint64)
        if n.value:
            self._check(self.lib.mgta_get_mercy_candidates(self.h, _p(out), n.value, ctypes.byref(n)),
                        "mgta_get_mercy_candidates")
        return out

    def num_mercy(self):
        n = ctypes.c_uint64()
        self._check(self.lib.mgta_get_num_mercy(self.h, ctypes.byref(n)), "mgta_get_num_mercy")
        return n.value

    def stage2(self, collect=True):
        """-> (stream bytes, meta int64[65536,3], totals int64[10]).
        collect=True   copy every delivery into one Python bytes object (tests, file writers)
        collect="count" the library still copies records + table to pinned host memory each batch, the sink only
                       counts them (bench e2e: no extra Python-side memcpy); stream is returned as its length
        collect=False  records stay on the device (sink = NULL)"""
        parts = []
        nbytes_total = [0]
        meta = np.zeros((NUM_BUCKETS, 3), dtype=np.int64)

        failed = []

        def sink(user, b0, b1, ptr, nbytes, mptr):
            try:
                if nbytes and collect is True:
                    for o in range(0, nbytes, 1 << 30):      # ctypes.string_at takes a C int size: slices of 1 GiB
                        parts.append(ctypes.string_at(ptr + o, min(1 << 30, nbytes - o)))
                nbytes_total[0] += nbytes
                meta[b0:b1] = np.ctypeslib.as_array(mptr, shape=((b1 - b0) * 3,)).reshape(b1 - b0, 3)
                return 0
            except BaseException as e:                       # ctypes would print and swallow it: abort the stage instead
                failed.append(e)
                return -1

        cb = SINK(sink) if collect else ctypes.cast(None, SINK)
        totals = np.zeros(10, dtype=np.int64)
        rc = self.lib.mgta_stage2(self.h, cb, None, _p(totals))
        if failed:
            raise failed[0]
        self._check(rc, "mgta_stage2")
        return (b"".join(parts) if collect is True else nbytes_total[0]), meta, totals

    # ---- sharded build (world > 1): the library walks the protocol, the caller runs the collectives it asks for
    def sharded_begin(self, stage, collect=True):
        """collect: as in stage2() (stage 2 only)"""
        self._sh = {"stage": stage, "collect": collect, "parts": [], "nbytes": 0, "meta": np.zeros((NUM_BUCKETS, 3), dtype=np.int64)}
        sh = self._sh

        def sink(user, b0, b1, ptr, nbytes, mptr):
            try:
                if nbytes and collect is True:
                    for o in range(0, nbytes, 1 << 30):      # ctypes.string_at takes a C int size: slices of 1 GiB
                        sh["parts"].append(ctypes.string_at(ptr + o, min(1 << 30, nbytes - o)))
                sh["nbytes"] += nbytes
                sh["meta"][b0:b1] = np.ctypeslib.as_array(mptr, shape=((b1 - b0) * 3,)).reshape(b1 - b0, 3)
                return 0
            except BaseException as e:                       # ctypes would print and swallow it: abort the stage instead
                sh["failed"] = e
                return -1

        sh["cb"] = SINK(sink) if (collect and stage == 2) else ctypes.cast(None, SINK)      # kept alive until the result is read
        self._check(self.lib.mgta_sharded_begin(self.h, stage, sh["cb"], None), "mgta_sharded_begin")

    def sharded_step(self):
        """-> Collective to run among the shards on this context's stream, or None when the stage has finished"""
        c = Collective()
        rc = self.lib.mgta_sharded_step(self.h, ctypes.byref(c))
        if self._sh.get("failed") is not None:
            raise self._sh["failed"]
        self._check(rc, "mgta_sharded_step")
        return None if c.op == COLL_NONE else c

    def sharded_result(self):
        """stage 1 -> edge_counting int64[65536] of the whole graph; stage 2 -> (stream | byte count, meta, totals) of this shard"""
        sh = self._sh
        if sh["stage"] == 1:
            ec = np.zeros(NUM_BUCKETS, dtype=np.int64)
            self._check(self.lib.mgta_sharded_result(self.h, _p(ec), None), "mgta_sharded_result")
            return ec
        totals = np.zeros(10, dtype=np.int64)
        self._check(self.lib.mgta_sharded_result(self.h, None, _p(totals)), "mgta_sharded_result")
        return (b"".join(sh["parts"]) if sh["collect"] is True else sh["nbytes"]), sh["meta"], totals

    def sharded(self, stage, run_collective, collect=True):
        """One whole stage: run_collective(Collective) executes an exchange among the shards (see shards.TorchComm)."""
        self.sharded_begin(stage, collect)
        while True:
            c = self.sharded_step()
            if c is None:
                return self.sharded_result()
            run_collective(c)

    def shard_range(self):
        a, b = ctypes.c_int32(), ctypes.c_int32()
        self._check(self.lib.mgta_shard_range(self.h, ctypes.byref(a), ctypes.byref(b)), "mgta_shard_range")
        return a.value, b.value

    def stats(self, stage):
        s = StageStats()
        self._check(self.lib.mgta_get_stats(self.h, stage, ctypes.byref(s)), "mgta_get_stats")
        return s.as_dict()


class Sdbg:
    """The in-memory succinct de Bruijn graph (SuccinctDBG::LoadFromMultiFile + rank/select tables) built on the device:
    thin wrapper over mgta_sdbg_* (include/mgta_cuda.h)."""

    def __init__(self, k, need_multiplicity=True, device=0, stream=None):
        self.lib = load()
        self.h = ctypes.c_void_p()
        rc = self.lib.mgta_sdbg_create(device, stream, k, int(need_multiplicity), ctypes.byref(self.h))
        if rc != 0:
            raise MgtaError("mgta_sdbg_create failed (%d): no CUDA device? (there is no CPU fallback)" % rc)
        self.need_multiplicity = bool(need_multiplicity)
        self.k, self.device = k, device

    def _check(self, rc, what):
        if rc != 0:
            raise MgtaError("%s failed (%d): %s" % (what, rc, self.lib.mgta_sdbg_last_error(self.h).decode()))

    def close(self):
        if self.h:
            self.lib.mgta_sdbg_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def append(self, b0, b1, stream_bytes, meta):
        """records of buckets [b0, b1) (bytes-like, host) + their int64[b1 - b0, 3] table"""
        meta = np.ascontiguousarray(meta, dtype=np.int64)
        buf = np.frombuffer(stream_bytes, dtype=np.uint8) if len(stream_bytes) else np.zeros(0, np.uint8)
        self._check(self.lib.mgta_sdbg_append(self.h, b0, b1, _p(buf) if len(buf) else None, len(buf), _p(meta)), "mgta_sdbg_append")

    def from_files(self, prefix, delivery_bytes=1 << 29):
        """the graph files <prefix>.sdbg_info / .sdbg.<i> (what SuccinctDBG::LoadFromMultiFile reads, succinct_dbg.cpp:595-723):
        the bucket ranges of the files are put back into bucket order (the reference's writer threads scatter them) and
        handed over in deliveries of about delivery_bytes"""
        from . import sdbg_io
        hdr, rows = sdbg_io.read_info(prefix)
        wpt = hdr["words_per_tip_label"]
        files = [np.memmap("%s.sdbg.%d" % (prefix, i), dtype=np.uint8, mode="r") if os.path.getsize("%s.sdbg.%d" % (prefix, i)) else
                 np.zeros(0, np.uint8) for i in range(hdr["num_threads"])]
        nb = hdr["num_buckets"]
        size = rows[:, 3] * 2 + rows[:, 5] * 2 + rows[:, 4] * 4 * wpt
        b0, parts, acc = 0, [], 0
        for b in range(nb):
            if rows[b, 1] != -1:
                parts.append(files[int(rows[b, 1])][int(rows[b, 2]):int(rows[b, 2]) + int(size[b])])
                acc += int(size[b])
            if acc >= delivery_bytes or b == nb - 1:
                self.append(b0, b + 1, np.concatenate(parts).tobytes() if parts else b"", rows[b0:b + 1, 3:6])
                b0, parts, acc = b + 1, [], 0
        return hdr

    def from_stage2(self, ctx):
        """stage 2 of `ctx` straight into the builder (records parsed in HBM) -> totals int64[10]"""
        totals = np.zeros(10, dtype=np.int64)
        rc = self.lib.mgta_stage2_into_sdbg(ctx.h, self.h, _p(totals))
        if rc != 0:
            raise MgtaError("mgta_stage2_into_sdbg failed (%d): %s" % (rc, self.lib.mgta_last_error(ctx.h).decode()))
        return totals

    def finish(self):
        self._check(self.lib.mgta_sdbg_finish(self.h), "mgta_sdbg_finish")
        return self.header()

    def header(self):
        h = SdbgHeader()
        self._check(self.lib.mgta_sdbg_header(self.h, ctypes.byref(h)), "mgta_sdbg_header")
        return h

    def array(self, which, c=0, dtype=np.uint8):
        p, n = ctypes.c_void_p(), ctypes.c_uint64()
        self._check(self.lib.mgta_sdbg_array(self.h, which, c, ctypes.byref(p), ctypes.byref(n)), "mgta_sdbg_array")
        out = np.zeros(n.value, dtype=np.uint8)
        self._check(self.lib.mgta_sdbg_copy(self.h, which, c, _p(out), n.value), "mgta_sdbg_copy")
        return out.view(dtype)

    # ---- navigation queries (include/mgta_sdbg_query.h) ------------------------------------------------------------
    def query(self, op, x):
        """runs `op` (SQ_*) on every row of x: packed k-mers (uint32 [n, words]) for SQ_LOOKUP, edge ids (int64 [n]) for
        the others.  x is a numpy array or a CUDA torch tensor, and the result is of the same kind (for a tensor it stays
        on the device): int64 [n], int64 [n, 4] for SQ_OUTGOING / SQ_INCOMING, uint32 [n, words + 1] for SQ_LABEL
        (int32 for a tensor; the last column is 1 for a tip node)."""
        in_row, out_row = ctypes.c_uint64(), ctypes.c_uint64()
        self._check(self.lib.mgta_sdbg_query_row_bytes(self.h, op, ctypes.byref(in_row), ctypes.byref(out_row)), "mgta_sdbg_query_row_bytes")
        wpt = (2 * self.k + 31) // 32
        cols = {SQ_LABEL: wpt + 1, SQ_OUTGOING: 4, SQ_INCOMING: 4}.get(op, 1)
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, dtype=np.uint32 if op == SQ_LOOKUP else np.int64)
            n = x.nbytes // in_row.value
            if n * in_row.value != x.nbytes:
                raise ValueError("input of %d bytes is not a whole number of %d-byte rows" % (x.nbytes, in_row.value))
            out = np.empty((n, cols), dtype=np.uint32 if op == SQ_LABEL else np.int64)
            self._check(self.lib.mgta_sdbg_query(self.h, op, _p(x) if n else None, n, _p(out) if n else None, out.nbytes), "mgta_sdbg_query")
        else:
            import torch
            if not x.is_cuda or x.device.index != self.device:
                raise ValueError("a tensor input must live on cuda:%d, the graph's device" % self.device)
            x = x.contiguous()
            if x.element_size() * x.numel() % in_row.value:
                raise ValueError("input of %d bytes is not a whole number of %d-byte rows" % (x.element_size() * x.numel(), in_row.value))
            n = x.element_size() * x.numel() // in_row.value
            out = torch.empty((n, cols), dtype=torch.int32 if op == SQ_LABEL else torch.int64, device=x.device)
            torch.cuda.current_stream(x.device).synchronize()      # x is written on torch's stream, the query runs on the graph's
            self._check(self.lib.mgta_sdbg_query(self.h, op, x.data_ptr() if n else None, n, out.data_ptr() if n else None,
                                                 out.numel() * 8 if op != SQ_LABEL else out.numel() * 4), "mgta_sdbg_query")
        return out if cols > 1 else out.reshape(-1)

    def lookup(self, kmers):
        """packed k-mers -> the last edge of each node, or -1"""
        return self.query(SQ_LOOKUP, kmers)

    def label(self, edges):
        return self.query(SQ_LABEL, edges)

    def forward(self, edges):
        return self.query(SQ_FORWARD, edges)

    def backward(self, edges):
        return self.query(SQ_BACKWARD, edges)

    def outdegree(self, edges):
        return self.query(SQ_OUTDEGREE, edges)

    def indegree(self, edges):
        return self.query(SQ_INDEGREE, edges)

    def outgoing(self, edges):
        return self.query(SQ_OUTGOING, edges)

    def incoming(self, edges):
        return self.query(SQ_INCOMING, edges)

    def multiplicity(self, edges):
        return self.query(SQ_MULTIPLICITY, edges)

    def revcomp(self, edges):
        return self.query(SQ_REVCOMP, edges)

    # ---- unitigs (include/mgta_sdbg_unitig.h) ------------------------------------------------------------------------
    def unitigs(self, device=False):
        """the maximal non-branching paths of the graph, one of every reverse-complement pair -> (rows int64 [U, 6]:
        first_edge, last_edge, n_edges, seq_offset, mult_sum, flags (UNITIG_CYCLE | UNITIG_SELF_RC); seq uint8 [chars]:
        the ASCII sequences in row order).  numpy arrays, or CUDA tensors on the graph's device when device=True."""
        n_rows, n_chars = ctypes.c_int64(), ctypes.c_uint64()
        self._check(self.lib.mgta_sdbg_unitigs(self.h, ctypes.byref(n_rows), ctypes.byref(n_chars)), "mgta_sdbg_unitigs")
        U, C = n_rows.value, n_chars.value
        if device:
            import torch
            rows = torch.empty((U, 6), dtype=torch.int64, device="cuda:%d" % self.device)
            seq = torch.empty(C, dtype=torch.uint8, device=rows.device)
            torch.cuda.current_stream(rows.device).synchronize()     # the copy runs on the graph's stream
            rp, sp = rows.data_ptr(), seq.data_ptr()
        else:
            rows, seq = np.empty((U, 6), np.int64), np.empty(C, np.uint8)
            rp, sp = rows.ctypes.data, seq.ctypes.data
        self._check(self.lib.mgta_sdbg_unitig_copy(self.h, rp if U else None, U * 48, sp if C else None, C), "mgta_sdbg_unitig_copy")
        return rows, seq

    # ---- the unitig graph (include/mgta_sdbg_unitig_graph.h) ----------------------------------------------------------
    def unitig_links(self, device=False):
        """the links between the rows of the last unitigs() call -> int64 [L, 2] (from, to), sorted: oriented unitigs
        o = 2 * row (its sequence) or 2 * row + 1 (the reverse complement), one link of every twin pair, overlap k.
        numpy, or a CUDA tensor on the graph's device when device=True."""
        n = ctypes.c_int64()
        self._check(self.lib.mgta_sdbg_unitig_links(self.h, ctypes.byref(n)), "mgta_sdbg_unitig_links")
        L = n.value
        if device:
            import torch
            links = torch.empty((L, 2), dtype=torch.int64, device="cuda:%d" % self.device)
            torch.cuda.current_stream(links.device).synchronize()    # the copy runs on the graph's stream
            p = links.data_ptr()
        else:
            links = np.empty((L, 2), np.int64)
            p = links.ctypes.data
        self._check(self.lib.mgta_sdbg_unitig_link_copy(self.h, p if L else None, L * 16), "mgta_sdbg_unitig_link_copy")
        return links


def pack_kmers(kmers, k):
    """ACGT strings of length k -> uint32 [n, ceil(2k / 32)]: the first character in bits 31..30 of word 0, unused low bits 0"""
    wpt = (2 * k + 31) // 32
    if any(len(s) != k for s in kmers):
        raise ValueError("every k-mer must have %d characters" % k)
    codes = np.frombuffer("".join(kmers).encode(), dtype=np.uint8).reshape(len(kmers), k)
    lut = np.full(256, 255, np.uint8)
    lut[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4, dtype=np.uint8)
    c = lut[codes].astype(np.uint32)
    if (c == 255).any():
        raise ValueError("k-mers are over ACGT")
    c = np.concatenate([c, np.zeros((len(kmers), wpt * 16 - k), np.uint32)], axis=1).reshape(len(kmers), wpt, 16)
    return (c << (2 * np.arange(15, -1, -1, dtype=np.uint32))).sum(axis=2, dtype=np.uint32)


def unpack_kmers(words, k):
    """uint32 [n, >= ceil(2k / 32)] (LABEL rows may carry their tip column) -> ACGT strings of length k"""
    w = np.asarray(words, dtype=np.uint32)[:, :(2 * k + 31) // 32]
    c = (w[:, :, None] >> (2 * np.arange(15, -1, -1, dtype=np.uint32))) & 3
    s = np.frombuffer(b"ACGT", np.uint8)[c.reshape(len(w), -1)[:, :k]]
    return [r.tobytes().decode() for r in s]


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def unitig_strings(rows, seq):
    """rows and sequence of Sdbg.unitigs (numpy or torch) -> the ACGT string of every row"""
    rows, seq = _host(rows), _host(seq)
    ends = np.append(rows[1:, 3], len(seq)) if len(rows) else np.zeros(0, np.int64)
    b = seq.tobytes()
    return [b[o:e].decode() for o, e in zip(rows[:, 3].tolist(), ends.tolist())]


def write_unitigs_fasta(path, rows, seq, min_len=0):
    """the unitigs as plain FASTA (usable as the next k's `buildgraph --assist_seq`), those of at least min_len
    characters: >unitig_<row> len=<chars> edges=<n> multi=<mult_sum / n, or na> flags=<flags>"""
    rows = _host(rows)
    with open(path, "w") as f:
        for i, s in enumerate(unitig_strings(rows, seq)):
            if len(s) < min_len:
                continue
            n, mult, flags = int(rows[i, 2]), int(rows[i, 4]), int(rows[i, 5])
            f.write(">unitig_%d len=%d edges=%d multi=%s flags=%d\n%s\n" % (i, len(s), n, "%.2f" % (mult / n) if mult >= 0 else "na", flags, s))


def write_unitigs_gfa(path, rows, seq, links, k):
    """the unitig graph as GFA 1.0 (Bandage and other GFA tools): one S line per row, named as in write_unitigs_fasta,
    with KC:i:<mult_sum> when multiplicities are known, and one L line per link of Sdbg.unitig_links (+ for an even
    oriented id, - for an odd one) with an overlap of k characters"""
    rows, links = _host(rows), _host(links)
    with open(path, "w") as f:
        f.write("H\tVN:Z:1.0\n")
        for i, s in enumerate(unitig_strings(rows, seq)):
            mult = int(rows[i, 4])
            f.write("S\tunitig_%d\t%s\tLN:i:%d%s\n" % (i, s, len(s), "\tKC:i:%d" % mult if mult >= 0 else ""))
        for a, b in links.tolist():
            f.write("L\tunitig_%d\t%s\tunitig_%d\t%s\t%dM\n" % (a // 2, "-" if a & 1 else "+", b // 2, "-" if b & 1 else "+", k))


def pack_reads(seqs, device=0):
    """ASCII sequences (list of bytes) -> the <X>.bin records `megagta buildlib` writes for them (np.uint32): mgta_pack_reads"""
    lib = load()
    bases = np.frombuffer(b"".join(seqs), dtype=np.uint8) if seqs else np.zeros(0, np.uint8)
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs], dtype=np.uint64)
    words = int(sum(1 + (len(s) + 15) // 16 for s in seqs))
    out = np.zeros(words, dtype=np.uint32)
    rc = lib.mgta_pack_reads(device, _p(bases) if len(bases) else None, _p(off), len(seqs), _p(out), words)
    if rc != 0:
        raise MgtaError("mgta_pack_reads failed (%d): %s" % (rc, lib.mgta_tools_last_error().decode()))
    return out
