"""ctypes binding of libgaml_b200.so (include/gaml_b200.h) + a thin `ProbCalculator` mirror.

This module is plumbing for tests and bench.py: the product is the C ABI. It never touches oracle/.
`ProbCalculator.calc_prob(paths)` has the meaning of the reference's
`ProbCalculator::CalcProb(paths, zeros, total_len)` (prob_calculator.h:63-109): same statefulness, same
outputs. The library has no CPU fallback; creating a context without a B200 raises GamlError.
"""
from __future__ import annotations

import ctypes as C
import itertools
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .workload import ALN_DTYPE, KIND_PACBIO, KIND_PAIRED, PB_DTYPE, ReadSetSpec, Workload

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgaml_b200.so")

INT32_MIN = -(2 ** 31)
PARTIAL_DOUBLES = 5   # GAML_PARTIAL_DOUBLES


class GamlError(RuntimeError):
    pass


class ReadsetConfig(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("mismatch_prob", C.c_double),
                ("match_prob", C.c_double), ("insert_mean", C.c_double), ("insert_std", C.c_double),
                ("min_prob_per_base", C.c_double), ("min_prob_start", C.c_double), ("weight", C.c_double),
                ("penalty_constant", C.c_double), ("step", C.c_double)]


class Result(C.Structure):
    _fields_ = [("prob", C.c_double), ("total_len", C.c_int32), ("n_sets", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("evals", C.c_int64), ("last_records_gathered", C.c_int64),
                ("last_reads_scanned", C.c_int64), ("last_algorithmic_bytes", C.c_int64),
                ("last_h2d_bytes", C.c_int64), ("last_d2h_bytes", C.c_int64), ("last_device_ms", C.c_double),
                ("last_score_kernel_ms", C.c_double), ("last_was_full", C.c_int32),
                ("last_overflow_reads", C.c_int32), ("last_prepare_host_us", C.c_double),
                ("last_launch_host_us", C.c_double), ("last_finish_host_us", C.c_double),
                ("last_scratch_placements", C.c_int64), ("last_multi_items", C.c_int64),
                ("fast_change_evals", C.c_int64), ("delta_only_evals", C.c_int64), ("cache_appends", C.c_int64),
                ("cache_rebuilds", C.c_int64), ("full_reuse_evals", C.c_int64), ("full_patch_evals", C.c_int64),
                ("last_batch_cov_events", C.c_int64), ("last_batch_cov_segments", C.c_int64),
                ("last_batch_cov_exported", C.c_int64)]


EXPORTS = ["gaml_ctx_create", "gaml_ctx_destroy", "gaml_last_error", "gaml_ctx_stream", "gaml_set_graph",
           "gaml_add_readset", "gaml_cache_insert", "gaml_cache_insert_pacbio", "gaml_cache_contains",
           "gaml_cache_commit", "gaml_calc_prob", "gaml_calc_prob_partial", "gaml_combine_partials", "gaml_combine_partials_raw",
           "gaml_eval_prepare", "gaml_eval_launch", "gaml_eval_finish", "gaml_reset_state", "gaml_read_values",
           "gaml_calc_prob_batch", "gaml_calc_prob_batch_partial",
           "gaml_get_stats", "gaml_set_profiling", "gaml_read_timeline", "gaml_set_result_exchange",
           "gaml_eval_finish_gathered", "gaml_calc_prob_gathered", "gaml_cache_save", "gaml_cache_load",
           "gaml_pacbio_alignment_logprob", "gaml_peer_exchange_create", "gaml_peer_exchange_open", "gaml_peer_exchange_close",
           "gaml_nccl_unique_id", "gaml_nccl_exchange_init", "gaml_calc_prob_batch_gathered",
           "gaml_penalty_export", "gaml_penalty_import", "gaml_calc_prob_batch_shard", "gaml_batch_penalty_export",
           "gaml_batch_penalty_import", "gaml_combine_batch_partials"]

_lib = None


def load_library() -> C.CDLL:
    """Loads the in-tree CUDA library; fails loudly if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GamlError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(LIB_PATH)
    vp, i32p, i64p, dp = C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_double)
    lib.gaml_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.gaml_ctx_destroy.argtypes = [vp]
    lib.gaml_ctx_destroy.restype = None
    lib.gaml_last_error.argtypes = [vp]
    lib.gaml_last_error.restype = C.c_char_p
    lib.gaml_ctx_stream.argtypes = [vp]
    lib.gaml_ctx_stream.restype = vp
    lib.gaml_set_graph.argtypes = [vp, C.c_int32, i32p, i32p]
    lib.gaml_add_readset.argtypes = [vp, C.POINTER(ReadsetConfig), C.c_int64, C.c_int64, C.c_int64, i32p, i32p,
                                     C.c_int32, C.c_int32]
    lib.gaml_cache_insert.argtypes = [vp, C.c_int, C.c_int, i32p, C.c_int32, vp, C.c_int64, C.c_int32]
    lib.gaml_cache_insert_pacbio.argtypes = [vp, C.c_int, i32p, C.c_int32, vp, C.c_int64]
    lib.gaml_cache_contains.argtypes = [vp, C.c_int, C.c_int, i32p, C.c_int32]
    lib.gaml_cache_commit.argtypes = [vp]
    lib.gaml_calc_prob.argtypes = [vp, i32p, i64p, C.c_int32, C.POINTER(Result), i32p]
    lib.gaml_calc_prob_partial.argtypes = [vp, i32p, i64p, C.c_int32, dp, i32p]
    lib.gaml_combine_partials.argtypes = [vp, dp, C.c_int32, C.c_int32, C.POINTER(Result), i32p]
    lib.gaml_combine_partials_raw.argtypes = [dp, C.c_int32, C.c_int32, i32p, i64p, dp, C.c_int32, C.POINTER(Result), i32p]
    lib.gaml_calc_prob_batch.argtypes = [vp, C.c_int32, i32p, i64p, i32p, i64p, i64p, dp, i32p, i32p]
    lib.gaml_calc_prob_batch_partial.argtypes = [vp, C.c_int32, i32p, i64p, i32p, i64p, i64p, dp, i32p]
    lib.gaml_eval_prepare.argtypes = [vp, i32p, i64p, C.c_int32]
    lib.gaml_eval_launch.argtypes = [vp]
    lib.gaml_eval_finish.argtypes = [vp, dp, i32p]
    lib.gaml_reset_state.argtypes = [vp]
    lib.gaml_read_values.argtypes = [vp, C.c_int, dp, C.c_int64]
    lib.gaml_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.gaml_set_profiling.argtypes = [vp, C.c_int32]
    lib.gaml_read_timeline.argtypes = [vp, C.POINTER(C.c_double), C.c_int32]
    u8p, i64p_, i32p_ = C.POINTER(C.c_uint8), C.POINTER(C.c_int64), C.POINTER(C.c_int32)
    lib.gaml_pacbio_alignment_logprob.argtypes = [vp, C.c_double, C.c_double, C.c_int32, C.c_int64, u8p, i64p_, u8p, i64p_, i32p_,
                                                  i32p_, u8p, i64p_, C.POINTER(C.c_double)]
    lib.gaml_cache_save.argtypes = [vp, C.c_int, C.c_char_p]
    lib.gaml_cache_load.argtypes = [vp, C.c_int, C.c_char_p]
    lib.gaml_set_result_exchange.argtypes = [vp, vp, C.c_int64, C.c_int32, C.c_int32]
    lib.gaml_eval_finish_gathered.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    lib.gaml_calc_prob_gathered.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.c_int32, C.POINTER(C.c_double),
                                            C.POINTER(C.c_int32)]
    lib.gaml_calc_prob_batch_gathered.argtypes = [vp, C.c_int32, i32p, i64p, i32p, i64p, i64p, dp, i32p, i32p]
    lib.gaml_penalty_export.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64), C.c_int64, C.POINTER(C.c_int64)]
    lib.gaml_penalty_import.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64), C.c_int64]
    lib.gaml_calc_prob_batch_shard.argtypes = [vp, C.c_int32, i32p, i64p, i32p, i64p, i64p, dp, i32p]
    lib.gaml_batch_penalty_export.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64), C.c_int64, C.POINTER(C.c_int64)]
    lib.gaml_batch_penalty_import.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64), C.c_int64]
    lib.gaml_combine_batch_partials.argtypes = [vp, dp, C.c_int32, C.c_int32, dp, i32p]
    lib.gaml_peer_exchange_create.argtypes = [vp, C.c_int32, C.c_int32, vp, C.POINTER(vp)]
    lib.gaml_peer_exchange_open.argtypes = [vp, vp, C.POINTER(vp)]
    lib.gaml_peer_exchange_close.argtypes = [vp]
    lib.gaml_nccl_unique_id.argtypes = [vp]
    lib.gaml_nccl_exchange_init.argtypes = [vp, vp, C.c_int32, C.c_int32]
    for name in EXPORTS:
        if name not in ("gaml_ctx_destroy", "gaml_last_error", "gaml_ctx_stream"):
            getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int32)


def _p32(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def flatten_walks(walks: Sequence[Sequence[int]]) -> Tuple[np.ndarray, np.ndarray]:
    """vector<vector<int>> -> (concatenated node ids, n_walks+1 offsets), the C ABI's walk layout."""
    offs = np.zeros(len(walks) + 1, dtype=np.int64)
    if len(walks):
        np.cumsum(np.fromiter(map(len, walks), dtype=np.int64, count=len(walks)), out=offs[1:])
    total = int(offs[-1])
    nodes = np.fromiter(itertools.chain.from_iterable(walks), dtype=np.int32, count=total) if total else np.zeros(1, np.int32)
    return nodes, offs


class FlatWalks:
    """Walks in the C ABI's layout with their ctypes pointers made once (what a C++ caller simply holds): keeps
    the Python plumbing out of timed loops."""
    __slots__ = ("nodes", "offs", "n", "p_nodes", "p_offs")

    def __init__(self, walks=None, nodes=None, offs=None):
        if walks is not None:
            nodes, offs = flatten_walks(walks)
        self.nodes, self.offs = nodes, offs
        self.n = len(offs) - 1
        self.p_nodes = nodes.ctypes.data_as(C.POINTER(C.c_int32))
        self.p_offs = offs.ctypes.data_as(C.POINTER(C.c_int64))


class ProbCalculator:
    """Mirror of the reference's `ProbCalculator` over the C ABI (one context, one CUDA stream)."""

    def __init__(self, node_len, normalize_map=None, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.gaml_ctx_create(device, C.byref(h))
        if rc != 0:
            raise GamlError(f"gaml_ctx_create failed ({rc}): {self.lib.gaml_last_error(None).decode()}")
        self.h = h
        nl = _i32(node_len)
        nm = _i32(normalize_map) if normalize_map is not None else None
        self._check(self.lib.gaml_set_graph(self.h, len(nl), _p32(nl), _p32(nm) if nm is not None else None))
        self.sets: List[dict] = []

    # -- plumbing --
    def _check(self, rc: int) -> int:
        if rc < 0:
            raise GamlError(f"gaml_b200 error {rc}: {self.lib.gaml_last_error(self.h).decode()}")
        return rc

    def close(self):
        if getattr(self, "h", None):
            try:
                self.clear_result_exchange()
            except Exception:
                pass
            self.lib.gaml_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self) -> int:
        return int(self.lib.gaml_ctx_stream(self.h) or 0)

    # -- read sets / cache --
    def add_readset(self, spec: ReadSetSpec, shard: Optional[Tuple[int, int]] = None,
                    max_read_len: Optional[Sequence[int]] = None, lens_are_local: bool = False) -> int:
        lo, hi = shard if shard is not None else (0, spec.n_reads)
        cfg = ReadsetConfig(kind=spec.kind, mismatch_prob=spec.mismatch_prob, match_prob=spec.match_prob,
                            insert_mean=spec.insert_mean, insert_std=spec.insert_std,
                            min_prob_per_base=spec.min_prob_per_base, min_prob_start=spec.min_prob_start,
                            weight=spec.weight, penalty_constant=spec.penalty_constant, step=spec.step)
        lens = [_i32(rl if lens_are_local else rl[lo:hi]) for rl in spec.read_len]
        if max_read_len is None:
            max_read_len = [int(rl.max()) if len(rl) else 0 for rl in spec.read_len]
        l2 = _p32(lens[1]) if spec.kind == KIND_PAIRED else None
        m2 = int(max_read_len[1]) if spec.kind == KIND_PAIRED else -1
        sid = self._check(self.lib.gaml_add_readset(self.h, C.byref(cfg), spec.n_reads, lo, hi, _p32(lens[0]), l2,
                                                    int(max_read_len[0]), m2))
        self.sets.append({"spec": spec, "lo": lo, "hi": hi})
        return sid

    def cache_insert(self, set_id: int, mate: int, key: Sequence[int], records: np.ndarray,
                     key_max_position: int = INT32_MIN) -> None:
        k = _i32(key)
        spec = self.sets[set_id]["spec"]
        if spec.kind == KIND_PACBIO:
            r = np.ascontiguousarray(records, dtype=PB_DTYPE)
            self._check(self.lib.gaml_cache_insert_pacbio(self.h, set_id, _p32(k), len(k), r.ctypes.data, len(r)))
        else:
            r = np.ascontiguousarray(records, dtype=ALN_DTYPE)
            self._check(self.lib.gaml_cache_insert(self.h, set_id, mate, _p32(k), len(k), r.ctypes.data, len(r),
                                                   key_max_position))

    def prepared_insert(self, set_id: int, mate: int, key: Sequence[int], records: np.ndarray, key_max_position: int = INT32_MIN):
        """cache_insert of a short-read key with the array conversions and ctypes pointers made up front: returns a callable
        that performs just the C call (what a C++ caller's gaml_cache_insert costs) — for timed loops."""
        k = _i32(key)
        r = np.ascontiguousarray(records, dtype=ALN_DTYPE)
        pk, nk, pr, nr = _p32(k), len(k), r.ctypes.data, len(r)
        fn, h, check = self.lib.gaml_cache_insert, self.h, self._check

        def run(_keep=(k, r)):
            check(fn(h, set_id, mate, pk, nk, pr, nr, key_max_position))
        return run

    def cache_contains(self, set_id: int, mate: int, key: Sequence[int]) -> bool:
        k = _i32(key)
        return bool(self._check(self.lib.gaml_cache_contains(self.h, set_id, mate, _p32(k), len(k))))

    def commit(self) -> None:
        self._check(self.lib.gaml_cache_commit(self.h))

    @classmethod
    def from_workload(cls, wl: Workload, device: int = 0, shard_of=None) -> "ProbCalculator":
        """Loads every read set and injected cache of a workload. shard_of=(rank, world) keeps the
        contiguous read-id block of that rank for each set (SURVEY §8e)."""
        pc = cls(wl.node_len, wl.normalize_map, device)
        for spec in wl.sets:
            shard = None
            if shard_of is not None:
                rank, world = shard_of
                per = (spec.n_reads + world - 1) // world
                shard = (min(rank * per, spec.n_reads), min((rank + 1) * per, spec.n_reads))
            sid = pc.add_readset(spec, shard)
            for mate, cache in enumerate(spec.caches):
                for key, recs in cache.items():
                    pc.cache_insert(sid, mate, key, recs)
        pc.commit()
        return pc

    # -- scoring --
    def calc_prob(self, paths: Sequence[Sequence[int]]):
        """-> (prob, zeros [(floored, n_reads)] per set, total_len)."""
        nodes, offs = flatten_walks(paths)
        res = Result()
        zeros = np.zeros(2 * max(len(self.sets), 1), dtype=np.int32)
        self._check(self.lib.gaml_calc_prob(self.h, _p32(nodes), offs.ctypes.data_as(C.POINTER(C.c_int64)),
                                            len(paths), C.byref(res), _p32(zeros)))
        z = [(int(zeros[2 * i]), int(zeros[2 * i + 1])) for i in range(len(self.sets))]
        return res.prob, z, res.total_len

    def _io_buffers(self):
        n = PARTIAL_DOUBLES * max(len(self.sets), 1)
        io = getattr(self, "_io", None)
        if io is None or io[0].size != n:
            part = np.zeros(n, dtype=np.float64)
            tl = C.c_int32()
            zeros = np.zeros(2 * max(len(self.sets), 1), dtype=np.int32)
            io = self._io = (part, part.ctypes.data_as(C.POINTER(C.c_double)), tl, C.byref(tl), Result(), zeros, _p32(zeros))
        return io

    def calc_prob_partial_flat(self, nodes, offs: Optional[np.ndarray] = None):
        """gaml_calc_prob_partial on walks already in the C ABI's layout (what a C++ caller passes): a FlatWalks, or
        the (nodes, offsets) arrays."""
        fw = nodes if isinstance(nodes, FlatWalks) else FlatWalks(nodes=nodes, offs=offs)
        part, p_part, tl, p_tl = self._io_buffers()[:4]
        rc = self.lib.gaml_calc_prob_partial(self.h, fw.p_nodes, fw.p_offs, fw.n, p_part, p_tl)
        if rc < 0:
            self._check(rc)
        return part.copy(), tl.value

    def calc_prob_partial(self, paths: Sequence[Sequence[int]]):
        nodes, offs = flatten_walks(paths)
        part = np.zeros(PARTIAL_DOUBLES * max(len(self.sets), 1), dtype=np.float64)
        tl = C.c_int32()
        self._check(self.lib.gaml_calc_prob_partial(self.h, _p32(nodes), offs.ctypes.data_as(C.POINTER(C.c_int64)),
                                                    len(paths), part.ctypes.data_as(C.POINTER(C.c_double)),
                                                    C.byref(tl)))
        return part, tl.value

    def combine(self, gathered: np.ndarray, n_shards: int, total_len: int):
        res, zeros, p_zeros = self._io_buffers()[4:]
        gb = getattr(self, "_gbuf", None)
        if gb is None or gb[0].size != gathered.size:
            buf = np.zeros(gathered.size, dtype=np.float64)
            gb = self._gbuf = (buf, buf.ctypes.data_as(C.POINTER(C.c_double)))
        gb[0][:] = gathered.reshape(-1)
        rc = self.lib.gaml_combine_partials(self.h, gb[1], n_shards, total_len, C.byref(res), p_zeros)
        if rc < 0:
            self._check(rc)
        z = [(int(zeros[2 * i]), int(zeros[2 * i + 1])) for i in range(len(self.sets))]
        return res.prob, z, res.total_len

    def prepare(self, paths):
        nodes, offs = flatten_walks(paths)
        self._check(self.lib.gaml_eval_prepare(self.h, _p32(nodes), offs.ctypes.data_as(C.POINTER(C.c_int64)),
                                               len(paths)))

    def launch(self):
        self._check(self.lib.gaml_eval_launch(self.h))

    def finish(self):
        part = np.zeros(PARTIAL_DOUBLES * max(len(self.sets), 1), dtype=np.float64)
        tl = C.c_int32()
        self._check(self.lib.gaml_eval_finish(self.h, part.ctypes.data_as(C.POINTER(C.c_double)), C.byref(tl)))
        return part, tl.value

    @staticmethod
    def pack_candidates(candidates):
        """list of (erased base-walk indices, added walks) -> the flat host arrays of gaml_calc_prob_batch."""
        n = len(candidates)
        er_off = np.zeros(n + 1, dtype=np.int64)
        ca_off = np.zeros(n + 1, dtype=np.int64)
        er, added = [], []
        for i, (e, a) in enumerate(candidates):
            er.extend(int(x) for x in e)
            added.extend(a)
            er_off[i + 1] = len(er)
            ca_off[i + 1] = len(added)
        nodes, w_off = flatten_walks(added)
        return n, _i32(er if er else [0]), er_off, nodes, w_off, ca_off

    def calc_prob_batch_partial_packed(self, packed):
        """gaml_calc_prob_batch_partial on pre-packed host arrays -> (partials [n, sets, PARTIAL_DOUBLES], total_lens [n])."""
        n, er_a, er_off, nodes, w_off, ca_off = packed
        ns = max(len(self.sets), 1)
        part = np.zeros(n * ns * PARTIAL_DOUBLES, dtype=np.float64)
        tls = np.zeros(n, dtype=np.int32)
        i64p = C.POINTER(C.c_int64)
        self._check(self.lib.gaml_calc_prob_batch_partial(self.h, n, _p32(er_a), er_off.ctypes.data_as(i64p), _p32(nodes),
                                                          w_off.ctypes.data_as(i64p), ca_off.ctypes.data_as(i64p),
                                                          part.ctypes.data_as(C.POINTER(C.c_double)), _p32(tls)))
        return part.reshape(n, ns, PARTIAL_DOUBLES), tls

    def calc_prob_batch_packed(self, packed):
        """gaml_calc_prob_batch (scores combined in the library) on pre-packed host arrays -> (probs [n], total_lens [n])."""
        n, er_a, er_off, nodes, w_off, ca_off = packed
        probs = np.zeros(n, dtype=np.float64)
        tls = np.zeros(n, dtype=np.int32)
        zeros = np.zeros(n * 2 * max(len(self.sets), 1), dtype=np.int32)
        i64p = C.POINTER(C.c_int64)
        self._check(self.lib.gaml_calc_prob_batch(self.h, n, _p32(er_a), er_off.ctypes.data_as(i64p), _p32(nodes),
                                                  w_off.ctypes.data_as(i64p), ca_off.ctypes.data_as(i64p),
                                                  probs.ctypes.data_as(C.POINTER(C.c_double)), _p32(tls), _p32(zeros)))
        return probs, tls

    def calc_prob_batch_gathered_packed(self, packed):
        """gaml_calc_prob_batch_gathered: every rank's shard, one all-reduce, exact combine -> (probs [n], total_lens [n])."""
        n, er_a, er_off, nodes, w_off, ca_off = packed
        probs = np.zeros(n, dtype=np.float64)
        tls = np.zeros(n, dtype=np.int32)
        zeros = np.zeros(n * 2 * max(len(self.sets), 1), dtype=np.int32)
        i64p = C.POINTER(C.c_int64)
        self._check(self.lib.gaml_calc_prob_batch_gathered(self.h, n, _p32(er_a), er_off.ctypes.data_as(i64p), _p32(nodes),
                                                           w_off.ctypes.data_as(i64p), ca_off.ctypes.data_as(i64p),
                                                           probs.ctypes.data_as(C.POINTER(C.c_double)), _p32(tls), _p32(zeros)))
        return probs, tls

    def calc_prob_batch_shard_packed(self, packed):
        """gaml_calc_prob_batch_shard: this shard's partials of every candidate (penalised sets included; their coverage waits
        for batch_penalty_export / _import) -> (partials [n, sets, PARTIAL_DOUBLES], total_lens [n])."""
        n, er_a, er_off, nodes, w_off, ca_off = packed
        ns = max(len(self.sets), 1)
        part = np.zeros(n * ns * PARTIAL_DOUBLES, dtype=np.float64)
        tls = np.zeros(n, dtype=np.int32)
        i64p = C.POINTER(C.c_int64)
        self._check(self.lib.gaml_calc_prob_batch_shard(self.h, n, _p32(er_a), er_off.ctypes.data_as(i64p), _p32(nodes),
                                                        w_off.ctypes.data_as(i64p), ca_off.ctypes.data_as(i64p),
                                                        part.ctypes.data_as(C.POINTER(C.c_double)), _p32(tls)))
        return part.reshape(n, ns, PARTIAL_DOUBLES), tls

    def batch_penalty_export(self, set_id: int) -> np.ndarray:
        """gaml_batch_penalty_export: this shard's thinned coverage keys of the pending shard batch (uint64)."""
        n = C.c_int64(0)
        rc = self.lib.gaml_batch_penalty_export(self.h, set_id, None, 0, C.byref(n))
        if rc < 0 and n.value == 0:
            self._check(rc)
        out = np.zeros(max(n.value, 1), dtype=np.uint64)
        self._check(self.lib.gaml_batch_penalty_export(self.h, set_id, out.ctypes.data_as(C.POINTER(C.c_uint64)), n.value,
                                                       C.byref(n)))
        return out[:n.value]

    def batch_penalty_import(self, set_id: int, all_keys: np.ndarray) -> None:
        """gaml_batch_penalty_import: the concatenation of every shard's exported keys (this shard's included)."""
        a = np.ascontiguousarray(all_keys, dtype=np.uint64)
        p = a.ctypes.data_as(C.POINTER(C.c_uint64)) if len(a) else None
        self._check(self.lib.gaml_batch_penalty_import(self.h, set_id, p, len(a)))

    def combine_batch_partials(self, gathered: np.ndarray):
        """gaml_combine_batch_partials: gathered [n_shards, n, sets, PARTIAL_DOUBLES] -> (probs [n], zeros [n, sets, 2])."""
        g = np.ascontiguousarray(gathered, dtype=np.float64)
        ns = max(len(self.sets), 1)
        n_shards, n = g.shape[0], g.shape[1]
        probs = np.zeros(n, dtype=np.float64)
        zeros = np.zeros(n * 2 * ns, dtype=np.int32)
        self._check(self.lib.gaml_combine_batch_partials(self.h, g.ctypes.data_as(C.POINTER(C.c_double)), n_shards, n,
                                                         probs.ctypes.data_as(C.POINTER(C.c_double)), _p32(zeros)))
        return probs, zeros.reshape(n, ns, 2)

    def calc_prob_batch(self, candidates):
        """candidates: list of (erased base-walk indices, added walks). -> (probs [n], total_lens [n], zeros [n][sets]).
        Paired sets only; a penalised set is scored with each candidate's own coverage-gap bad bases."""
        n = len(candidates)
        er_off = np.zeros(n + 1, dtype=np.int64)
        ca_off = np.zeros(n + 1, dtype=np.int64)
        er, added = [], []
        for i, (e, a) in enumerate(candidates):
            er.extend(int(x) for x in e)
            added.extend(a)
            er_off[i + 1] = len(er)
            ca_off[i + 1] = len(added)
        er_a = _i32(er if er else [0])
        nodes, w_off = flatten_walks(added)
        probs = np.zeros(n, dtype=np.float64)
        tls = np.zeros(n, dtype=np.int32)
        zeros = np.zeros(n * 2 * max(len(self.sets), 1), dtype=np.int32)
        i64p = C.POINTER(C.c_int64)
        self._check(self.lib.gaml_calc_prob_batch(self.h, n, _p32(er_a), er_off.ctypes.data_as(i64p), _p32(nodes),
                                                  w_off.ctypes.data_as(i64p), ca_off.ctypes.data_as(i64p),
                                                  probs.ctypes.data_as(C.POINTER(C.c_double)), _p32(tls), _p32(zeros)))
        return probs, tls, zeros.reshape(n, max(len(self.sets), 1), 2)

    def reset_state(self):
        self._check(self.lib.gaml_reset_state(self.h))

    def read_values(self, set_id: int) -> np.ndarray:
        n = self.sets[set_id]["hi"] - self.sets[set_id]["lo"]
        out = np.zeros(max(n, 1), dtype=np.float64)
        self._check(self.lib.gaml_read_values(self.h, set_id, out.ctypes.data_as(C.POINTER(C.c_double)), n))
        return out[:n]

    def set_result_exchange(self, shm_buf, rank: int, world: int) -> None:
        """shm_buf: a writable buffer over a host shared-memory segment every rank has mapped (dist.ResultExchange)."""
        self._exch_keep = shm_buf
        addr = C.addressof(C.c_char.from_buffer(shm_buf))
        self._check(self.lib.gaml_set_result_exchange(self.h, C.c_void_p(addr), len(shm_buf), rank, world))
        self._exch_world = world
        ns = max(len(self.sets), 1)
        g = np.zeros(world * ns * PARTIAL_DOUBLES, dtype=np.float64)
        self._gath = (g, g.ctypes.data_as(C.POINTER(C.c_double)))

    def _gather_buffers(self, world: int) -> None:
        self._exch_world = world
        ns = max(len(self.sets), 1)
        g = np.zeros(world * ns * PARTIAL_DOUBLES, dtype=np.float64)
        self._gath = (g, g.ctypes.data_as(C.POINTER(C.c_double)))

    def peer_exchange_create(self, rank: int, world: int):
        """gaml_peer_exchange_create -> (this rank's cudaIpcMemHandle_t as 64 bytes, its device pointer)."""
        handle = (C.c_char * 64)()
        ptr = C.c_void_p()
        self._check(self.lib.gaml_peer_exchange_create(self.h, rank, world, C.cast(handle, C.c_void_p), C.byref(ptr)))
        return bytes(handle), ptr.value

    def peer_exchange_open(self, handles: Optional[Sequence[bytes]] = None, local_ptrs: Optional[Sequence[Optional[int]]] = None) -> None:
        """handles: every rank's 64-byte IPC handle (rank order); local_ptrs: device pointers of contexts in THIS process."""
        world = len(handles) if handles is not None else len(local_ptrs)
        hb = b"".join(handles) if handles is not None else None
        arr = None
        if local_ptrs is not None:
            arr = (C.c_void_p * world)(*[C.c_void_p(p) if p else C.c_void_p() for p in local_ptrs])
        self._check(self.lib.gaml_peer_exchange_open(self.h, hb, arr))
        self._gather_buffers(world)

    def peer_exchange_close(self) -> None:
        self._check(self.lib.gaml_peer_exchange_close(self.h))

    def nccl_exchange_init(self, unique_id: Optional[bytes], rank: int, world: int) -> None:
        """gaml_nccl_exchange_init: unique_id = 128 bytes from nccl_unique_id() of ONE rank, broadcast to all (None detaches)."""
        self._check(self.lib.gaml_nccl_exchange_init(self.h, unique_id, rank, world))
        if unique_id is not None:
            self._gather_buffers(world)

    def penalty_export(self, set_id: int) -> np.ndarray:
        """gaml_penalty_export: this shard's coverage events of the last evaluation (uint64 words)."""
        n = C.c_int64(0)
        rc = self.lib.gaml_penalty_export(self.h, set_id, None, 0, C.byref(n))
        if rc < 0 and n.value == 0:
            self._check(rc)
        out = np.zeros(max(n.value, 1), dtype=np.uint64)
        self._check(self.lib.gaml_penalty_export(self.h, set_id, out.ctypes.data_as(C.POINTER(C.c_uint64)), n.value, C.byref(n)))
        return out[:n.value]

    def penalty_import(self, set_id: int, all_events: np.ndarray) -> None:
        """gaml_penalty_import: the concatenation of every shard's events (this shard's included)."""
        a = np.ascontiguousarray(all_events, dtype=np.uint64)
        p = a.ctypes.data_as(C.POINTER(C.c_uint64)) if len(a) else None
        self._check(self.lib.gaml_penalty_import(self.h, set_id, p, len(a)))

    def clear_result_exchange(self) -> None:
        if getattr(self, "_exch_keep", None) is not None:
            self._check(self.lib.gaml_set_result_exchange(self.h, None, 0, 0, 1))
            self._exch_keep = None

    def calc_prob_gathered_flat(self, fw: "FlatWalks"):
        """gaml_calc_prob_gathered: this rank's evaluation, then every rank's partials ([world, sets, PARTIAL_DOUBLES])."""
        g, p_g = self._gath
        tl, p_tl = self._io_buffers()[2:4]
        rc = self.lib.gaml_calc_prob_gathered(self.h, fw.p_nodes, fw.p_offs, fw.n, p_g, p_tl)
        if rc < 0:
            self._check(rc)
        return g.reshape(self._exch_world, -1), tl.value

    def pacbio_alignment_logprob(self, alns, match_prob: float, mismatch_prob: float, band: int = 2) -> np.ndarray:
        """gaml_pacbio_alignment_logprob over a list of alnprob.Alignment."""
        from . import alnprob
        return self.pacbio_alignment_logprob_flat(alnprob.flatten(alns), match_prob, mismatch_prob, band)

    def pacbio_alignment_logprob_flat(self, flat, match_prob: float, mismatch_prob: float, band: int = 2) -> np.ndarray:
        """The same on arrays already in the C ABI's layout (alnprob.flatten)."""
        s1, s1_off, s2, s2_off, posstart, op_len, op_chr, op_off = flat
        n_alns = len(posstart)
        out = np.zeros(n_alns, dtype=np.float64)
        u8p, i64p = C.POINTER(C.c_uint8), C.POINTER(C.c_int64)
        def u8(a):
            a = np.ascontiguousarray(a if len(a) else np.zeros(1, np.uint8))
            return a, a.ctypes.data_as(u8p)
        k1, p1 = u8(s1)
        k2, p2 = u8(s2)
        k3, p3 = u8(op_chr)
        ol = np.ascontiguousarray(op_len if len(op_len) else np.zeros(1, np.int32))
        self._check(self.lib.gaml_pacbio_alignment_logprob(self.h, match_prob, mismatch_prob, band, n_alns, p1,
                                                           s1_off.ctypes.data_as(i64p), p2, s2_off.ctypes.data_as(i64p),
                                                           _p32(posstart if len(posstart) else np.zeros(1, np.int32)), _p32(ol), p3,
                                                           op_off.ctypes.data_as(i64p), out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def cache_save(self, set_id: int, path: str) -> None:
        self._check(self.lib.gaml_cache_save(self.h, set_id, path.encode()))

    def cache_load(self, set_id: int, path: str) -> None:
        self._check(self.lib.gaml_cache_load(self.h, set_id, path.encode()))

    def finish_gathered(self):
        g, p_g = self._gath
        tl, p_tl = self._io_buffers()[2:4]
        self._check(self.lib.gaml_eval_finish_gathered(self.h, p_g, p_tl))
        return g.reshape(self._exch_world, -1).copy(), tl.value

    def set_profiling(self, level) -> None:
        """0 off (default); 1 events around the evaluation (stats().last_device_ms); 2 + per-set events around the
        streaming kernels (stats().last_score_kernel_ms); 3 device globaltimer stamps per kernel (read_timeline)."""
        self._check(self.lib.gaml_set_profiling(self.h, int(level)))

    def read_timeline(self) -> dict:
        out = np.zeros(12, dtype=np.float64)
        self._check(self.lib.gaml_read_timeline(self.h, out.ctypes.data_as(C.POINTER(C.c_double)), 12))
        names = ["apply_slots", "tier1", "tier2", "many_placement", "delta_or_multi", "total"]
        return {n: (float(out[2 * i]), float(out[2 * i + 1])) for i, n in enumerate(names) if out[2 * i] >= 0}

    def stats(self) -> Stats:
        s = Stats()
        self._check(self.lib.gaml_get_stats(self.h, C.byref(s)))
        return s


def nccl_unique_id() -> bytes:
    """128-byte ncclUniqueId for gaml_nccl_exchange_init (call on one rank, broadcast)."""
    buf = (C.c_char * 128)()
    rc = load_library().gaml_nccl_unique_id(C.cast(buf, C.c_void_p))
    if rc < 0:
        raise GamlError(f"gaml_nccl_unique_id failed ({rc}): {load_library().gaml_last_error(None).decode()}")
    return bytes(buf)


def combine_partials_raw(gathered: np.ndarray, kinds: Sequence[int], n_reads_total: Sequence[int],
                         weights: Sequence[float], total_len: int):
    """Context-free combine of all-gathered shard partials ([n_shards, n_sets, PARTIAL_DOUBLES]) -> (prob, zeros, total_len)."""
    lib = load_library()
    g = np.ascontiguousarray(gathered, dtype=np.float64).reshape(-1, len(kinds), PARTIAL_DOUBLES)
    k = _i32(kinds)
    n = np.ascontiguousarray(n_reads_total, dtype=np.int64)
    w = np.ascontiguousarray(weights, dtype=np.float64)
    res = Result()
    zeros = np.zeros(2 * max(len(kinds), 1), dtype=np.int32)
    rc = lib.gaml_combine_partials_raw(g.ctypes.data_as(C.POINTER(C.c_double)), g.shape[0], len(kinds), _p32(k),
                                       n.ctypes.data_as(C.POINTER(C.c_int64)), w.ctypes.data_as(C.POINTER(C.c_double)),
                                       total_len, C.byref(res), _p32(zeros))
    if rc != 0:
        raise GamlError(f"gaml_combine_partials_raw failed ({rc})")
    return res.prob, [(int(zeros[2 * i]), int(zeros[2 * i + 1])) for i in range(len(kinds))], res.total_len
