"""Batched candidate evaluation (gaml_calc_prob_batch) of paired read sets with a coverage-gap penalty (B200).

Every candidate's score must be the double a sequential gaml_calc_prob of its walk set returns after the same history:
tp - bad_bases_c * penalty_constant, where bad_bases_c is the state's bad bases minus the erased walks' and plus the added
walks' own sweeps over the current cache (graph.cc:1938, 1946, 1988).
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from gaml_b200 import api, synth, workload

pytestmark = pytest.mark.gpu

REL_TOTAL = 1e-9
PENALTY, STEP = 0.00007, 300.0 - 30.0   # gaml.cc:860: step = insert_mean - penalty_step


def _delta(base, cand):
    """(indices of base walks not in cand, walks of cand not in base) as a multiset difference."""
    from collections import Counter
    need = Counter(tuple(w) for w in cand)
    erased = []
    for i, w in enumerate(base):
        if need[tuple(w)] > 0:
            need[tuple(w)] -= 1
        else:
            erased.append(i)
    have = Counter(tuple(w) for w in base)
    added = []
    for w in cand:
        if have[tuple(w)] > 0:
            have[tuple(w)] -= 1
        else:
            added.append(list(w))
    return erased, added


def _penalised(wl):
    wl.sets[0].penalty_constant = PENALTY
    wl.sets[0].step = STEP
    return wl


def _walks_of(base, cand):
    erased, added = cand
    gone = set(erased)
    return [list(w) for k, w in enumerate(base) if k not in gone] + [list(w) for w in added]


def _shaped_candidates(base):
    """One candidate of every shape the penalty bookkeeping has to get right, on the first walks of `base`."""
    multi = [i for i, w in enumerate(base) if sum(1 for x in w if x >= 0) >= 2]
    i, j = (multi + [0, 1])[:2] if multi else (0, 1)
    if i == j:
        j = (i + 1) % len(base)
    flip = lambda w: [(x ^ 1) if x >= 0 else x for x in reversed(w)]
    cands = [
        ([i, j], [list(base[i]) + [-150] + list(base[j])]),   # join with a gap: a contig start inside the walk
        ([i], [flip(base[i])]),                               # reverse-complement flip
        ([j], []),                                            # only erases
        ([], [list(base[i])]),                                # only adds (a second copy of a walk)
        ([], []),                                             # the base itself
    ]
    if multi:
        w = base[multi[0]]
        cut = next(t for t in range(1, len(w)) if w[t] >= 0 and w[t - 1] >= 0) if any(
            w[t] >= 0 and w[t - 1] >= 0 for t in range(1, len(w))) else None
        if cut is not None:
            cands.append(([multi[0]], [list(w[:cut]), list(w[cut:])]))                       # split
        k = (multi[0] + 1) % len(base)
        a, b = list(w[:1]) + list(base[k][1:]), list(base[k][:1]) + list(w[1:])
        if all(x and x[0] >= 0 and x[-1] >= 0 for x in (a, b)):
            cands.append(([multi[0], k], [a, b]))                                            # tail swap
    return cands


def _sequential(wl, history, walks):
    pc = api.ProbCalculator.from_workload(wl)
    for h in history:
        pc.calc_prob(h)
    out = pc.calc_prob(walks)
    pc.close()
    return out


def _check_batch(wl, n_hist, n_random, seed, oracle=None):
    """Batch = the workload's remaining evaluations as deltas + shaped + random candidates; each must equal, bit for bit,
    a fresh context's sequential evaluation after the same history. Returns (cands, penalised probs, unpenalised probs)."""
    import bench
    history = wl.evals[:n_hist]
    base = history[-1]
    shaped = _shaped_candidates(base)
    assert len(shaped) == 7   # every shape, split and tail swap included: the base has walks of several nodes
    cands = [_delta(base, c) for c in wl.evals[n_hist:]] + shaped + bench.make_candidates(base, n_random, np.random.default_rng(seed))
    assert any(not a for _, a in cands) and any(not e for e, _ in cands)
    assert any(any(x < 0 for w in a for x in w) for _, a in cands)   # gaps inside added walks

    wl.sets[0].penalty_constant = 0.0
    plain = api.ProbCalculator.from_workload(wl)
    _penalised(wl)
    pc = api.ProbCalculator.from_workload(wl)
    for walks in history:
        last = pc.calc_prob(walks)
        plain.calc_prob(walks)
    state_before = pc.read_values(0).copy()
    probs, tls, zeros = pc.calc_prob_batch(cands)
    st = pc.stats()
    assert st.last_batch_cov_segments == sum(len(e) + len(a) for e, a in cands)
    assert st.last_batch_cov_events > 0
    assert np.array_equal(pc.read_values(0), state_before)   # stateless
    assert pc.calc_prob(base) == last                          # and the next evaluation is unaffected
    plain_probs, plain_tls, _ = plain.calc_prob_batch(cands)
    pc.close()
    plain.close()
    assert np.array_equal(tls, plain_tls)
    for i, cand in enumerate(cands):
        p, z, tl = _sequential(wl, history, _walks_of(base, cand))
        assert probs[i] == p, (i, cand[0], probs[i], p)       # bit-identical
        assert int(tls[i]) == tl and (int(zeros[i, 0, 0]), int(zeros[i, 0, 1])) == z[0], i
    if oracle is not None:
        for i in (0, len(cands) // 2, len(cands) - 1):
            small = workload.Workload(node_len=wl.node_len, normalize_map=wl.normalize_map, sets=wl.sets,
                                      evals=history + [_walks_of(base, cands[i])])
            ref = oracle(small, f"batchpen{i}", dump=False)
            assert abs(probs[i] - ref[-1].score) <= REL_TOTAL * abs(ref[-1].score), (i, probs[i], ref[-1].score)
            assert int(tls[i]) == ref[-1].total_len and int(zeros[i, 0, 0]) == ref[-1].zeros[0][0]
    return cands, probs, plain_probs


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_penalised_batch_equals_sequential_evaluation(seed, oracle):
    """Sparse coverage, penalised: every candidate bit-identical to sequential evaluation, the batch stateless, three
    candidates against the oracle. The penalty must really act, and per candidate: the penalised minus the unpenalised
    scores are not one constant offset."""
    wl = synth.paired_workload(14, 2500, 400, n_evals=40, seed=seed)
    _, probs, plain = _check_batch(wl, 20, 48, seed, oracle)
    diff = probs - plain
    assert np.any(diff != 0)
    assert len(set(diff.tolist())) > 1


def test_penalised_batch_with_repeat_keys_and_scratch_reads():
    """The repeat-rich workload: keys that occur several times in a candidate's walks and reads with many placements
    take the general replay and the scratch path of the batch, which must emit the same coverage events."""
    wl = synth.paired_workload(14, 2500, 6000, n_evals=26, seed=77)
    _check_batch(wl, 8, 32, 77)


def test_c4_shape_penalised_batch_of_1024_candidates():
    """Config 4's shape with a penalty: 1024 candidates in one batch, a sample bit-identical to sequential evaluation."""
    import bench
    wl = _penalised(synth.paired_workload(10000, 10000, 1_200_000, n_evals=22, seed=44))
    history = wl.evals[:6]
    base = history[-1]
    pc = api.ProbCalculator.from_workload(wl)
    for walks in history:
        last = pc.calc_prob(walks)
    cands = bench.make_candidates(base, 1024, np.random.default_rng(5))
    probs, tls, zeros = pc.calc_prob_batch(cands)
    assert pc.calc_prob(base) == last
    pc.close()
    for i in (0, 1, 17, 300, 511, 777, 1023):
        p, z, tl = _sequential(wl, history, _walks_of(base, cands[i]))
        assert probs[i] == p, (i, probs[i], p)
        assert int(tls[i]) == tl and (int(zeros[i, 0, 0]), int(zeros[i, 0, 1])) == z[0]


def test_partial_batch_of_a_penalised_set_is_refused():
    """The _partial form carries no bad bases (gaml_combine_partials would apply the base state's): it stays refused."""
    wl = _penalised(synth.paired_workload(14, 2500, 400, n_evals=4, seed=0))
    pc = api.ProbCalculator.from_workload(wl)
    pc.calc_prob(wl.evals[0])
    packed = pc.pack_candidates([_delta(wl.evals[0], wl.evals[1])])
    with pytest.raises(api.GamlError, match=r"error -4:.*no bad bases"):
        pc.calc_prob_batch_partial_packed(packed)
    pc.close()


def test_reference_batched_driver_with_a_penalty_is_identical(tmp_path):
    """The reference's own annealing driver over the CUDA library, plain and with the moves' candidate lists in device
    batches, on a penalised paired set: both traces identical to the pure reference's, which the penalty changes."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not all(os.path.exists(os.path.join(ref_dir, b)) for b in ("gaml_ref", "gaml_gpu", "gaml_gpu_batched")):
        pytest.skip("oracle/_ref/gaml_ref + gaml_gpu + gaml_gpu_batched not prebuilt")
    script = os.path.join(ROOT, "tools", "run_e2e.sh")
    # 1000 pairs over ~105 kbp: coverage gaps longer than the step, so the penalty changes the accept / reject decisions
    env = dict(os.environ, E2E_KINDS="paired", E2E_READS="1000")
    plain = subprocess.run(["bash", script, str(tmp_path / "plain"), "200"], capture_output=True, text=True, timeout=600, env=env)
    assert plain.returncode == 0, plain.stdout + plain.stderr
    env["E2E_PENALTY"] = "0.0001 30"
    out = subprocess.run(["bash", script, str(tmp_path / "pen"), "200"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("IDENTICAL TRAJECTORY") == 2, out.stdout
    with open(tmp_path / "plain" / "paired.ref.log") as a, open(tmp_path / "pen" / "paired.ref.log") as b:
        assert a.read() != b.read()
