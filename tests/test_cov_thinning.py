"""Exactness of the coverage-event thinning of shard candidate batches (gaml_calc_prob_batch_shard), on the CPU.

Each shard keeps, of its sorted covered-position keys, only the first and last distinct position of every bucket
(segment, u // w), u = (uint32)(pos ^ 2^31), w = floor(step) + 1 (w = 1 for a negative step). The sweep of the contig
starts plus the union of every shard's kept keys must give each segment the same bad bases as the sweep of all raw
events. Both the sweep (kernels.cu coverage_sweep_kernel) and the rule (coverage_thin_kernel) are restated here.
"""
import math

import numpy as np
import pytest


def key(seg, pos, covered):
    """cov_key: seg << 33 | (pos ^ 2^31) << 1 | type bit (1: covered position, 0: contig start)."""
    return (int(seg) << 33) | ((int(pos) + 2 ** 31) << 1) | int(covered)


def decode(k):
    return k >> 33, ((k >> 1) & 0xFFFFFFFF) - 2 ** 31, k & 1


def sweep(keys, cs, step, min_from_start):
    """coverage_sweep_kernel over the sorted keys -> {segment: bad bases}. cs: segment -> ascending contig starts."""
    keys = sorted(keys)
    bad = {}
    for i, k in enumerate(keys):
        seg, pos, covered = decode(k)
        if not covered:
            continue
        prev_pos, prev_type = 0, -1
        if i > 0:
            ps, pp, pc = decode(keys[i - 1])
            if ps == seg:
                prev_pos, prev_type = pp, (3 if pc else 1)
        last_begin = 0
        for c in cs.get(seg, []):
            if c <= pos:
                last_begin = c
            else:
                break
        if pos - prev_pos > step and prev_type in (3, -1) and pos - last_begin > min_from_start:
            bad[seg] = bad.get(seg, 0) + pos - prev_pos
    return bad


def bucket_width(step):
    """0 stands for one bucket per segment (floor(step) + 1 >= 2^32)."""
    if not step >= 0:
        return 1
    return 0 if step >= 4294967295.0 else math.floor(step) + 1


def thin(keys, step):
    """One shard's export: the first and last distinct key of every (segment, u // w) bucket, ascending."""
    w = bucket_width(step)
    d = sorted(set(keys))
    b = [(k >> 33, (((k >> 1) & 0xFFFFFFFF) // w) if w else 0) for k in d]
    return [k for i, k in enumerate(d) if i == 0 or b[i - 1] != b[i] or i + 1 == len(d) or b[i + 1] != b[i]]


def naive_thin(keys, step):
    """The WRONG rule: drop a position whose two neighbours are within `step` of each other."""
    d = sorted(set(keys))
    pos = [decode(k)[1] for k in d]
    return [k for i, k in enumerate(d) if i == 0 or i + 1 == len(d) or pos[i + 1] - pos[i - 1] > step]


def same_sums(a, b):
    return all(a.get(s, 0) == b.get(s, 0) for s in set(a) | set(b))


def random_case(rng):
    n_seg = int(rng.integers(1, 6))
    cs = {s: sorted(set(rng.integers(-200, 4000, rng.integers(0, 3)).tolist())) for s in range(n_seg)}
    events = []
    for s in range(n_seg):
        if rng.random() < 0.5:   # dense clusters: gaps mostly below the step, a few above
            for centre in rng.integers(-300, 5000, rng.integers(1, 5)):
                events += [(s, int(p)) for p in centre + rng.integers(0, 400, rng.integers(1, 60))]
        else:                    # sparse: gaps around and above the step
            events += [(s, int(p)) for p in rng.integers(-300, 5000, rng.integers(0, 25))]
    keys = [key(s, p, 1) for s, p in events]
    keys += [keys[int(i)] for i in rng.integers(0, max(len(keys), 1), rng.integers(0, len(keys) + 1))] if keys else []
    type1 = [key(s, p, 0) for s in cs for p in cs[s]]
    return cs, type1, keys


@pytest.mark.parametrize("step", [0.0, 0.5, 270.0, 270.9, -5.0, 1e7])
def test_thinned_union_sweeps_like_the_raw_events(step):
    rng = np.random.default_rng(int(abs(step) * 10) + 11)
    thinned_any = False
    for _ in range(60):
        cs, type1, keys = random_case(rng)
        mfs = float(rng.choice([0.0, 150.0, 500.0]))
        raw = sweep(type1 + keys, cs, step, mfs)
        n_shards = int(rng.integers(1, 5))
        owner = rng.integers(0, n_shards, len(keys))
        union = list(type1)
        for r in range(n_shards):
            kept = thin([k for k, o in zip(keys, owner) if o == r], step)
            assert kept == sorted(kept) and len(set(kept)) == len(kept)   # ascending, one copy of a key
            w = bucket_width(step)
            buckets = [(k >> 33, (((k >> 1) & 0xFFFFFFFF) // w) if w else 0) for k in kept]
            assert max([buckets.count(b) for b in buckets] + [0]) <= 2
            union += kept
        thinned_any |= len(union) - len(type1) < len(set(keys))
        assert same_sums(sweep(union, cs, step, mfs), raw), (step, mfs, n_shards)
    if bucket_width(step) != 1:
        assert thinned_any   # the rule really dropped distinct positions


def test_a_dropped_pair_of_neighbours_would_open_a_gap():
    """0, 8, 10, 18 with step 10: each inner point has neighbours within the step, but dropping both leaves a gap of 18.
    The neighbour rule gets this wrong (so the comparison above can see such an error); the bucket rule does not."""
    keys = [key(0, p, 1) for p in (0, 8, 10, 18)]
    raw = sweep(keys, {}, 10.0, 0.0)
    assert raw.get(0, 0) == 0
    assert sweep(naive_thin(keys, 10.0), {}, 10.0, 0.0) == {0: 18}
    assert same_sums(sweep(thin(keys, 10.0), {}, 10.0, 0.0), raw)


def test_negative_step_removes_duplicates_only():
    keys = [key(1, p, 1) for p in (5, 5, 6, 9, 9, 9, 40)]
    assert thin(keys, -3.0) == sorted(set(keys))
    raw = sweep(keys, {}, -3.0, 0.0)    # a duplicate "adds" its gap of 0
    assert raw == sweep(thin(keys, -3.0), {}, -3.0, 0.0) == {1: 40}
