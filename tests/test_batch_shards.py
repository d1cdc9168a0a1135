"""Candidate batches with a coverage-gap penalty on read-id shards (gaml_calc_prob_batch_shard) (B200).

Every shard scores its reads of every candidate and keeps a thinned set of its coverage events; the union of all shards'
thinned events is imported on every shard, and the combined probs must be bit-identical to gaml_calc_prob_batch on an
unsharded context with the same history.
"""
import dataclasses
import os
import pickle
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from gaml_b200 import api, synth

pytestmark = pytest.mark.gpu

PENALTY, STEP = 0.00007, 300.0 - 30.0   # gaml.cc:860: step = insert_mean - penalty_step
ERR_STATE = r"error -6:"


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


def _penalised(wl, step=STEP):
    wl.sets[0].penalty_constant = PENALTY
    wl.sets[0].step = step
    return wl


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


def _pen_sets(wl):
    return [s for s, spec in enumerate(wl.sets) if spec.penalty_constant != 0]


def _evaluate(shards, walks, pen_sets):
    """One stateful evaluation over the shards, the shard penalty exchanged (gaml_penalty_export / _import)."""
    parts = [pc.calc_prob_partial(walks) for pc in shards]
    if len(shards) > 1:
        for s in pen_sets:
            union = np.concatenate([pc.penalty_export(s) for pc in shards])
            for pc in shards:
                pc.penalty_import(s, union)
    return shards[0].combine(np.stack([p for p, _ in parts]), len(shards), parts[0][1])


def _shard_batch(shards, packed, pen_sets):
    """The whole protocol in one process: shard batch, exports concatenated, import and combine on every shard."""
    outs = [pc.calc_prob_batch_shard_packed(packed) for pc in shards]
    for s in pen_sets:
        union = np.concatenate([pc.batch_penalty_export(s) for pc in shards])
        for pc in shards:
            pc.batch_penalty_import(s, union)
    g = np.stack([part for part, _ in outs])
    return outs, [pc.combine_batch_partials(g) for pc in shards]


def _candidates(wl, n_hist, n_random, seed):
    import bench
    history = wl.evals[:n_hist]
    base = history[-1]
    cands = [_delta(base, c) for c in wl.evals[n_hist:]] + _shaped_candidates(base) + \
        bench.make_candidates(base, n_random, np.random.default_rng(seed))
    return history, base, cands


def _unsharded(wl, history, cands):
    whole = api.ProbCalculator.from_workload(wl)
    for walks in history:
        whole.calc_prob(walks)
    probs, tls, zeros = whole.calc_prob_batch(cands)
    whole.close()
    return probs, tls, zeros


def _check_shards(wl, history, cands, n_shards, ref):
    """Every shard's probs, zeros and total lengths equal the unsharded batch's bit for bit; returns the shards (open)."""
    pen = _pen_sets(wl)
    shards = [api.ProbCalculator.from_workload(wl, shard_of=(r, n_shards)) for r in range(n_shards)]
    for walks in history:
        _evaluate(shards, walks, pen)
    outs, res = _shard_batch(shards, api.ProbCalculator.pack_candidates(cands), pen)
    ref_probs, ref_tls, ref_zeros = ref
    for (_, tls), (probs, zeros) in zip(outs, res):
        assert np.array_equal(tls, ref_tls)
        assert np.array_equal(zeros, ref_zeros)
        bad = np.flatnonzero(probs != ref_probs)
        assert len(bad) == 0, (n_shards, bad[:8], probs[bad[:8]], ref_probs[bad[:8]])
    return shards


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_shard_batch_equals_the_unsharded_penalised_batch(seed):
    """Sparse coverage, penalised, on 1, 2 and 3 shards: bit-identical to the unsharded batch; the penalty acts per candidate."""
    wl = synth.paired_workload(14, 2500, 400, n_evals=40, seed=seed)
    history, _, cands = _candidates(wl, 20, 48, seed)
    plain_probs = _unsharded(wl, history, cands)[0]
    ref = _unsharded(_penalised(wl), history, cands)
    diff = ref[0] - plain_probs
    assert np.any(diff != 0) and len(set(diff.tolist())) > 1
    for n in (1, 2, 3):
        for pc in _check_shards(wl, history, cands, n, ref):
            assert pc.stats().last_batch_cov_segments == sum(len(e) + len(a) for e, a in cands)
            pc.close()


def test_shard_batch_with_repeat_keys_and_scratch_reads():
    """The repeat-rich workload: the general replay and the scratch path of the batch emit the events on each shard."""
    wl = _penalised(synth.paired_workload(14, 2500, 6000, n_evals=26, seed=77))
    history, _, cands = _candidates(wl, 8, 32, 77)
    for pc in _check_shards(wl, history, cands, 2, _unsharded(wl, history, cands)):
        pc.close()


def test_c4_shape_shard_batch_exports_few_keys():
    """Config 4's shape, 1024 candidates on 2 shards: bit-identical, fewer keys exported than emitted, and each export
    strictly increasing with at most two keys per (segment, step-wide bucket)."""
    import bench
    wl = _penalised(synth.paired_workload(10000, 10000, 1_200_000, n_evals=22, seed=44))
    history = wl.evals[:6]
    cands = bench.make_candidates(history[-1], 1024, np.random.default_rng(5))
    ref = _unsharded(wl, history, cands)
    shards = _check_shards(wl, history, cands, 2, ref)
    w = int(np.floor(STEP)) + 1
    for pc in shards:
        st = pc.stats()
        assert 0 < st.last_batch_cov_exported < st.last_batch_cov_events
        keys = pc.batch_penalty_export(0)
        assert len(keys) == st.last_batch_cov_exported
        assert np.all(keys[1:] > keys[:-1])
        seg = keys >> np.uint64(33)
        u = (keys >> np.uint64(1)) & np.uint64(0xFFFFFFFF)
        assert np.all(keys & np.uint64(1) == 1)
        _, counts = np.unique(np.stack([seg, u // np.uint64(w)]), axis=1, return_counts=True)
        assert counts.max() <= 2
        pc.close()


def test_negative_step_removes_duplicates_only():
    """A penalty step above the insert mean makes `step` negative: the shards only drop duplicate keys. Still exact."""
    wl = _penalised(synth.paired_workload(14, 2500, 400, n_evals=40, seed=0), step=-30.0)
    history, _, cands = _candidates(wl, 20, 48, 0)
    for pc in _check_shards(wl, history, cands, 2, _unsharded(wl, history, cands)):
        pc.close()


def test_penalised_and_unpenalised_sets_in_one_shard_batch():
    """Two paired sets, one penalised: the unpenalised set's partials equal gaml_calc_prob_batch_partial's, the probs
    the unsharded batch's, and the unpenalised set has nothing to export."""
    wl = _penalised(synth.paired_workload(14, 2500, 400, n_evals=40, seed=1))
    wl.sets.append(dataclasses.replace(wl.sets[0], penalty_constant=0.0))
    history, _, cands = _candidates(wl, 20, 24, 1)
    shards = _check_shards(wl, history, cands, 2, _unsharded(wl, history, cands))
    packed = api.ProbCalculator.pack_candidates(cands)
    for r, pc in enumerate(shards):
        with pytest.raises(api.GamlError, match=ERR_STATE):
            pc.batch_penalty_export(1)
        part, _ = pc.calc_prob_batch_shard_packed(packed)
        alone_wl = dataclasses.replace(wl, sets=[wl.sets[1]])
        alone = api.ProbCalculator.from_workload(alone_wl, shard_of=(r, 2))
        for walks in history:
            alone.calc_prob_partial(walks)
        ref_part, _ = alone.calc_prob_batch_partial_packed(packed)
        assert np.array_equal(part[:, 1, :], ref_part[:, 0, :])
        alone.close()
        pc.close()


def test_shard_batch_is_stateless():
    wl = _penalised(synth.paired_workload(14, 2500, 400, n_evals=40, seed=2))
    history, base, cands = _candidates(wl, 20, 24, 2)
    shards = [api.ProbCalculator.from_workload(wl, shard_of=(r, 2)) for r in range(2)]
    for walks in history:
        last = _evaluate(shards, walks, [0])
    before = [pc.read_values(0).copy() for pc in shards]
    packed = api.ProbCalculator.pack_candidates(cands)
    outs = [pc.calc_prob_batch_shard_packed(packed) for pc in shards]
    assert all(np.array_equal(pc.read_values(0), v) for pc, v in zip(shards, before))
    union = np.concatenate([pc.batch_penalty_export(0) for pc in shards])
    for pc in shards:
        pc.batch_penalty_import(0, union)
    assert all(np.array_equal(pc.read_values(0), v) for pc, v in zip(shards, before))
    g = np.stack([part for part, _ in outs])
    assert np.array_equal(shards[0].combine_batch_partials(g)[0], shards[1].combine_batch_partials(g)[0])
    assert _evaluate(shards, base, [0]) == last
    for pc in shards:
        pc.close()


def test_shard_batch_state_errors():
    wl = _penalised(synth.paired_workload(14, 2500, 400, n_evals=40, seed=0))
    history, base, cands = _candidates(wl, 10, 8, 0)
    shards = [api.ProbCalculator.from_workload(wl, shard_of=(r, 2)) for r in range(2)]
    for walks in history:
        _evaluate(shards, walks, [0])
    packed = api.ProbCalculator.pack_candidates(cands)
    with pytest.raises(api.GamlError, match=ERR_STATE):
        shards[0].combine_batch_partials(np.zeros((2, len(cands), 1, api.PARTIAL_DOUBLES)))   # no batch yet
    outs = [pc.calc_prob_batch_shard_packed(packed) for pc in shards]
    g = np.stack([part for part, _ in outs])
    with pytest.raises(api.GamlError, match=ERR_STATE + ".*not imported"):
        shards[0].combine_batch_partials(g)                                                    # before the import
    union = np.concatenate([pc.batch_penalty_export(0) for pc in shards])
    shards[0].batch_penalty_import(0, union)
    with pytest.raises(api.GamlError, match=ERR_STATE + ".*n_cand"):
        shards[0].combine_batch_partials(g[:, :-1])
    shards[0].combine_batch_partials(g)
    _evaluate(shards, base, [0])                          # a later evaluation drops the pending batch
    for call in (lambda pc: pc.batch_penalty_export(0), lambda pc: pc.batch_penalty_import(0, union),
                 lambda pc: pc.combine_batch_partials(g)):
        with pytest.raises(api.GamlError, match=ERR_STATE):
            call(shards[0])
    for pc in shards:                                     # an evaluation whose shard penalty is still pending
        pc.calc_prob_partial(base)
    with pytest.raises(api.GamlError, match=ERR_STATE + ".*gaml_penalty_import"):
        shards[0].calc_prob_batch_shard_packed(packed)
    for pc in shards:
        pc.close()


CHILD = r"""
import pickle
import sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, sys.argv[5])
from gaml_b200 import api, dist as gdist, synth
rank, world, port, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
wl = synth.paired_workload(14, 2500, 400, n_evals=40, seed=0)
wl.sets[0].penalty_constant, wl.sets[0].step = %r, %r
pc = api.ProbCalculator.from_workload(wl, shard_of=(rank, world))
for walks in wl.evals[:20]:
    part, tl = pc.calc_prob_partial(walks)
    pc.penalty_import(0, gdist.allgather_keys(pc.penalty_export(0)))
    g = gdist.allgather_partials(part)
    pc.combine(g, world, tl)
with open(out + ".cands.pkl", "rb") as f:
    packed = api.ProbCalculator.pack_candidates(pickle.load(f))
probs, tls, zeros = gdist.sharded_calc_prob_batch(pc, packed)
np.save(out + f".{rank}.npy", probs)
pc.close()
dist.destroy_process_group()
""" % (PENALTY, STEP)


def test_two_processes_over_gloo(tmp_path):
    """dist.sharded_calc_prob_batch over torch.distributed (gloo), one shard context per process on the same GPU."""
    wl = _penalised(synth.paired_workload(14, 2500, 400, n_evals=40, seed=0))
    history, _, cands = _candidates(wl, 20, 24, 0)
    ref_probs = _unsharded(wl, history, cands)[0]
    out = str(tmp_path / "probs")
    with open(out + ".cands.pkl", "wb") as f:
        pickle.dump(cands, f)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    env = dict(os.environ, PYTHONPATH=ROOT)
    procs = [subprocess.Popen([sys.executable, "-c", CHILD, str(r), "2", str(port), out, ROOT], cwd=ROOT, env=env,
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    logs = []
    try:
        for p in procs:
            logs.append(p.communicate(timeout=600)[0])
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.wait()
    assert all(p.returncode == 0 for p in procs), logs
    for r in range(2):
        assert np.array_equal(np.load(out + f".{r}.npy"), ref_probs)
