"""CPU tests of everything around the kernels: the C ABI surface, the workload files, the synthetic cache
builder's key rules, and the world_size-2 sharded combine over gloo. No compute call needs a GPU here."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from gaml_b200 import api, dist, synth, workload


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "gaml_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(gaml_[a-z_0-9]+)\s*\(", hdr)))
    assert len(declared) >= 18
    lib = api.load_library()
    for name in declared:
        assert hasattr(lib, name), name
    assert sorted(api.EXPORTS) == declared


def test_struct_layouts_match_header():
    assert C.sizeof(api.ReadsetConfig) == 8 + 9 * 8
    assert C.sizeof(api.Result) == 16
    assert workload.ALN_DTYPE.itemsize == 16 and workload.PB_DTYPE.itemsize == 24


def test_no_cpu_fallback_without_gpu():
    """Run in a child process that sees no CUDA device, so that the no-GPU failure mode is checked on GPU machines too."""
    code = ("import sys; sys.path.insert(0, {root!r})\n"
            "from gaml_b200 import api\n"
            "try:\n"
            "    api.ProbCalculator([100, 100])\n"
            "except api.GamlError as e:\n"
            "    print('GamlError:', e)\n").format(root=ROOT)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                         text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.startswith("GamlError:") and "no CPU fallback" in out.stdout, out.stdout


def test_combine_raw_is_pure_host_arithmetic():
    # two shards, one paired + one pacbio set; partial = {integer part, 2^-40 units, floored, -inf terms, nan terms}
    half = float(2 ** 39)
    g = np.array([[[-101.0, half, 3.0, 0, 0], [-50.0, 0.0, 1.0, 0, 0]], [[-200.0, half, 4.0, 0, 0], [-25.0, 0.0, 0.0, 0, 0]]])
    prob, zeros, tl = api.combine_partials_raw(g, [1, 2], [10, 5], [1.0, 0.5], 1000)
    assert zeros == [(7, 10), (1, 5)] and tl == 1000
    expect = (-300.0 / 10) * 1.0 + ((-75.0 / 5) - np.log(2000.0)) * 0.5      # -101 + .5 - 200 + .5 = -300
    assert prob == pytest.approx(expect, rel=1e-15)
    # total_len == 0 is replaced by 1 (graph.cc:3067-3069)
    prob0, _, _ = api.combine_partials_raw(g[:1], [1, 2], [10, 5], [1.0, 0.5], 0)
    assert prob0 == pytest.approx((-100.5 / 10) + ((-50.0 / 5) - np.log(2.0)) * 0.5, rel=1e-15)
    # a -inf term (log 0) makes the set's score -inf, like the reference's running sum would
    g[0, 0, 3] = 1
    assert api.combine_partials_raw(g, [1, 2], [10, 5], [1.0, 0.5], 1000)[0] == -np.inf
    # exactness: shard order and grouping cannot change the result
    rng = np.random.default_rng(0)
    parts = np.zeros((8, 1, 5))
    parts[:, 0, 0] = -rng.integers(10 ** 6, 10 ** 8, size=8)
    parts[:, 0, 1] = rng.integers(0, 2 ** 40, size=8)
    a = api.combine_partials_raw(parts, [1], [10 ** 6], [1.0], 5)[0]
    b = api.combine_partials_raw(parts[::-1], [1], [10 ** 6], [1.0], 5)[0]
    merged = parts.reshape(4, 2, 1, 5).sum(axis=1)      # pre-adding pairs of shards is exact too (integers < 2^53)
    c = api.combine_partials_raw(merged, [1], [10 ** 6], [1.0], 5)[0]
    assert a == b == c


def test_workload_roundtrip(tmp_path):
    wl = synth.mixed_workload(6, 3000, 200, 30, n_single=100, n_evals=5, seed=5, pacbio_len=2500)
    p = str(tmp_path / "w.wl")
    workload.write_workload(p, wl)
    back = workload.read_workload(p)
    assert back.evals == wl.evals
    assert np.array_equal(back.node_len, wl.node_len)
    for a, b in zip(wl.sets, back.sets):
        assert a.kind == b.kind and a.n_reads == b.n_reads
        for ca, cb in zip(a.caches, b.caches):
            assert list(ca.keys()) == list(cb.keys())
            for k in ca:
                assert np.array_equal(ca[k], cb[k])


def test_window_key_rule():
    node_len = np.array([1000, 1000, 100, 100, 150, 150, 80, 80, 5000, 5000], dtype=np.int32)
    ctg = [0, 2, 4, 6, 8]
    # node 0: following 100 + 150 = 250 <= 300, + 80 = 330 > 300 -> stop after node 6 (graph.cc:555-561)
    assert synth.window_key(ctg, 0, node_len) == (0, 2, 4, 6)
    assert synth.window_key(ctg, 3, node_len) == (6, 8)
    assert synth.window_key(ctg, 4, node_len) == (8,)
    keys = synth.short_keys_for_walks([ctg], node_len, with_single_node=True)
    assert (0,) in keys and (8,) in keys and (2,) not in keys      # single-node key only when len > 300
    assert synth.split_contigs([0, -5, 2, 4, -7]) == [[0], [2, 4], []]


def test_pacbio_key_rule():
    node_len = np.array([3000, 3000, 2, 2, 2500, 2500], dtype=np.int32)
    nmap = np.arange(6, dtype=np.int32)
    keys = synth.pacbio_keys_for_walks([[0, 2, 4]], node_len, nmap, max_read_len=1000)
    # from node 0: [0], [0,2] (2 <= 1000), [0,2,4] (2502 > 1000 -> pushed, then break) (graph.cc:2440-2453)
    assert keys == [(0,), (0, 2), (0, 2, 4), (2,), (2, 4), (4,)]


def test_synthetic_cache_positions_are_sorted_and_cropped():
    wl = synth.paired_workload(6, 2000, 500, n_evals=6, seed=3)
    for cache in wl.sets[0].caches:
        for key, recs in cache.items():
            if len(recs) == 0:
                continue
            order = np.lexsort((recs["read_id"], recs["position"]))
            assert np.array_equal(order, np.arange(len(recs)))          # Aligment::operator<
            if len(key) > 1 and wl.node_len[key[0]] > synth.K_MIN_SUBPATH:
                assert recs["position"].min() >= wl.node_len[key[0]] - synth.K_MIN_SUBPATH + 1   # graph.cc:849-851


def test_shard_bounds_cover_all_reads():
    for n in (0, 1, 7, 1000, 1001):
        for world in (1, 2, 3, 8):
            b = [dist.shard_bounds(n, r, world) for r in range(world)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))


WORKER = r'''
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch, torch.distributed as dist
from gaml_b200 import api, workload
from gaml_b200.dist import shard_bounds, allgather_partials
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
wl = workload.read_workload({wl!r}); ref = workload.read_results({res!r})
spec = wl.sets[0]
ok = True
for e, r in enumerate(ref):
    p = r.per_read[0]
    lo, hi = shard_bounds(spec.n_reads, rank, world)
    L = r.total_len if r.total_len else 1
    thr = np.exp(spec.min_prob_start + spec.min_prob_per_base * (spec.read_len[0][lo:hi] + spec.read_len[1][lo:hi]))
    v = p[lo:hi] / (2 * L)
    fl = v < thr
    terms = np.log(np.where(fl, thr, v))
    X = sum(int(x) for x in np.rint(terms * 2.0 ** 40))          # exact integer sum in units of 2^-40
    part = np.array([float(X >> 40), float(X & (2 ** 40 - 1)), float(fl.sum()), 0.0, 0.0])
    g = allgather_partials(part)
    assert g.shape == (world, 5)
    prob, zeros, tl = api.combine_partials_raw(g, [1], [spec.n_reads], [spec.weight], r.total_len)
    ok &= zeros == r.zeros and abs(prob - r.score) <= 1e-12 * abs(r.score)
dist.barrier()
sys.stdout.write("RANK%d_%s\n" % (rank, "OK" if ok else "FAIL")); sys.stdout.flush()
sys.exit(0 if ok else 1)
'''


def test_world_size_2_sharded_combine_gloo(tmp_path):
    """N>1 host path on CPU: each rank reduces its read-id block of the reference's per-read values
    (golden fixture), partials are all-gathered over gloo and combined through the C ABI."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT, wl=os.path.join(GOLDEN, "synth_paired.wl"),
                                    res=os.path.join(GOLDEN, "synth_paired.ref.res")))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29517", str(script)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "RANK0_OK" in out.stdout and "RANK1_OK" in out.stdout


def test_fast_get_changes_equals_the_reference_container():
    """tests/cpp/test_walk_changes.cc: the diff-based GetChanges (walk_set.h) against the reference's algorithm on the
    real std::unordered_multiset over 18 000 random evaluations (CPU only)."""
    import __graft_entry__ as entry
    entry.build()
    out = subprocess.run([entry.CHANGES_TEST_BIN], capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.startswith("OK"), out.stdout


def test_dropin_list_bookkeeping():
    """tests/cpp/test_flat_paths.cc: the drop-in ProbCalculator's flat walk lists (integration/flat_paths.h) — alignment with
    the previous call's list and the multiset difference handed to gaml_calc_prob_batch — over 12 000 random candidate
    lists (CPU only)."""
    import __graft_entry__ as entry
    entry.build()
    out = subprocess.run([entry.FLAT_TEST_BIN], capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.startswith("OK"), out.stdout
