"""The end of a paired full evaluation's chain (B200). Replayed as a CUDA graph, the chain ends with the streaming kernel;
when that kernel listed reads for the many-placement pass it publishes a pending line, and the owning host runs the
pass on demand before it takes the final line. A set that listed reads keeps the pass in its chain from then on."""
import mmap
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import GOLDEN
from gaml_b200 import api, synth, workload

pytestmark = pytest.mark.gpu

REL_TOTAL = 1e-9


def _full_eval(pc, walks):
    """One evaluation through prepare / launch / finish: (partials, total_len, kernels launched by launch + finish,
    kernels launched by launch alone)."""
    pc.prepare(walks)
    l0 = pc.stats().kernel_launches
    pc.launch()
    l1 = pc.stats().kernel_launches
    part, tl = pc.finish()
    return part, tl, pc.stats().kernel_launches - l0, l1 - l0


def test_listed_reads_take_the_on_demand_pass_and_match_the_golden():
    wl = workload.read_workload(os.path.join(GOLDEN, "hand_paired.wl"))
    ref = workload.read_results(os.path.join(GOLDEN, "hand_paired.ref.res"))
    pc = api.ProbCalculator.from_workload(wl)
    # fresh context: the chain ends with the streaming kernel, which lists reads -> pending line -> pass on demand
    part1, tl1, n1, chain1 = _full_eval(pc, wl.evals[0])
    st = pc.stats()
    assert st.last_was_full == 1 and st.last_overflow_reads > 0
    assert n1 == chain1 + 1   # the chain had no many-placement pass: finish() launched it
    assert np.array_equal(pc.read_values(0), ref[0].per_read[0])
    prob, zeros, tl = pc.combine(part1[None, :], 1, tl1)
    assert tl == ref[0].total_len and zeros == ref[0].zeros
    assert abs(prob - ref[0].score) <= REL_TOTAL * abs(ref[0].score)
    # the set listed reads: its next full evaluation has the pass in the chain — the same kernels, the same result
    pc.reset_state()
    part2, tl2, n2, chain2 = _full_eval(pc, wl.evals[0])
    assert pc.stats().last_overflow_reads == st.last_overflow_reads
    assert chain2 == n2 == n1 and tl2 == tl1 and np.array_equal(part2, part1)
    assert np.array_equal(pc.read_values(0), ref[0].per_read[0])
    # and the rest of the trajectory (incremental evaluations on top of that state) still matches bit for bit
    for e in range(1, len(wl.evals)):
        prob, zeros, tl = pc.calc_prob(wl.evals[e])
        assert tl == ref[e].total_len and zeros == ref[e].zeros, e
        assert abs(prob - ref[e].score) <= REL_TOTAL * abs(ref[e].score), e
        assert np.array_equal(pc.read_values(0), ref[e].per_read[0]), e
    pc.close()


def test_on_demand_pass_equals_the_pass_in_the_chain(monkeypatch):
    """Direct launches (no graphs) always end with the many-placement pass: the partials are identical."""
    wl = workload.read_workload(os.path.join(GOLDEN, "hand_paired.wl"))
    graph = api.ProbCalculator.from_workload(wl)
    monkeypatch.setenv("GAML_B200_NO_GRAPHS", "1")
    direct = api.ProbCalculator.from_workload(wl)
    monkeypatch.delenv("GAML_B200_NO_GRAPHS")
    a, ta, _, _ = _full_eval(graph, wl.evals[0])
    b, tb, _, _ = _full_eval(direct, wl.evals[0])
    assert ta == tb and np.array_equal(a, b)
    assert np.array_equal(graph.read_values(0), direct.read_values(0))
    graph.close()
    direct.close()


def test_chain_without_listed_reads_ends_with_the_streaming_kernel():
    wl = synth.paired_workload(46, 10000, 200_000, n_evals=2, seed=11)
    pc = api.ProbCalculator.from_workload(wl)
    ref = api.ProbCalculator.from_workload(wl)
    ref.set_profiling(2)   # the profiled chain keeps the trailing pass
    _, _, n, chain = _full_eval(pc, wl.evals[0])
    st = pc.stats()
    assert st.last_overflow_reads == 0
    # apply_slots, [multi pass], streaming kernel
    assert n == chain == 2 + (st.last_multi_items > 0), (n, chain, st.last_multi_items)
    _, _, n_ref, _ = _full_eval(ref, wl.evals[0])
    assert n_ref == n + 1
    assert np.array_equal(pc.read_values(0), ref.read_values(0))
    pc.close()
    ref.close()


def test_host_exchange_with_a_pending_shard_matches_the_unsharded_result():
    """Two read-id shards as two contexts sharing one result-exchange segment, each finished on its own thread (as its
    own process would): a shard that publishes a pending line runs its pass, and the other waits for the final line."""
    wl = workload.read_workload(os.path.join(GOLDEN, "hand_paired.wl"))
    whole = api.ProbCalculator.from_workload(wl)
    seg = mmap.mmap(-1, max(2 * 2 * 8 * 64, mmap.PAGESIZE))
    ranks = []
    for rk in range(2):
        pc = api.ProbCalculator.from_workload(wl, shard_of=(rk, 2))
        pc.set_result_exchange(seg, rk, 2)
        ranks.append(pc)
    listed = []
    with ThreadPoolExecutor(2) as pool:
        for e, walks in enumerate(wl.evals):
            ref = whole.calc_prob(walks)
            for pc in ranks:
                pc.prepare(walks)
                pc.launch()
            outs = []
            for g, tl in pool.map(lambda pc: pc.finish_gathered(), ranks):
                outs.append(ranks[0].combine(g, 2, tl))
            if e == 0:
                listed = [pc.stats().last_overflow_reads for pc in ranks]
            assert outs[0] == outs[1], e
            assert outs[0] == ref, (e, outs[0], ref)   # exact integer partial sums: bit-identical for any sharding
    assert sum(listed) > 0, listed   # a shard went through the pending line
    for pc in ranks:
        pc.close()
    whole.close()
