#!/usr/bin/env python
"""Cost of the coverage-gap penalty in a candidate batch (gaml_calc_prob_batch) on one GPU.

Two contexts over the same workload (BASELINE config 2, or one eighth of config 4 with --kind c4shard), one without and
one with a penalty on the paired set, both after the same incremental history. The same 1024 candidates
(bench.make_candidates) are scored by both, alternating, several times. Then the penalised context's sequential
alternative — calc_prob(candidate) and calc_prob(base) for each of a sample of candidates — scaled to the batch size.
With --shards N, the penalised set is also split into N read-id shard contexts on the same GPU, run one after the other
(gaml_calc_prob_batch_shard, the thinned coverage keys exported and imported, gaml_combine_batch_partials): per shard its
call and device time and its emitted events against its exported keys, the import and combine times, and every prob
checked against the unsharded penalised batch.
Last, one profiled batch of each (torch.profiler, CUDA kernels) for the per-kernel split of the added time.
JSON lines go to stdout and to <out>/batch_penalty_<kind>.jsonl (--out; a new temporary directory by default).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def spread(xs):
    xs = sorted(xs)
    return {"median": float(np.median(xs)), "min": xs[0], "max": xs[-1], "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kind", choices=["c2", "c4shard"], default="c2")
    ap.add_argument("--evals", type=int, default=10, help="evaluations of the incremental history")
    ap.add_argument("--candidates", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sequential-sample", type=int, default=16)
    ap.add_argument("--penalty", type=float, default=0.00007)
    ap.add_argument("--step", type=float, default=300.0 - 30.0)
    ap.add_argument("--out", default=None, help="output directory (default: a new temporary directory)")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--shards", type=int, default=0, help="also run the penalised batch on N read-id shard contexts")
    args = ap.parse_args()
    if args.out is None:
        args.out = tempfile.mkdtemp(prefix="batch_penalty_")
    os.makedirs(args.out, exist_ok=True)
    out_path = os.path.join(args.out, f"batch_penalty_{args.kind}.jsonl")
    out = open(out_path, "w")
    print(f"writing {out_path}", file=sys.stderr, flush=True)

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    emit({"what": "gpu", "kind": args.kind, "nvidia_smi": gpu_info()})
    wl, shard = bench.make_workload(1, 0, args.evals, kind=args.kind)
    plain, _, _ = bench.load_calculator(wl, shard, 0)
    wl.sets[0].penalty_constant = args.penalty
    wl.sets[0].step = args.step
    pen, _, _ = bench.load_calculator(wl, shard, 0)
    for walks in wl.evals:
        plain.calc_prob(walks)
        last = pen.calc_prob(walks)
    base = wl.evals[-1]
    cands = bench.make_candidates(base, args.candidates, np.random.default_rng(123))
    packed = plain.pack_candidates(cands)

    def one(pc):
        l0 = pc.stats().kernel_launches
        t0 = time.perf_counter()
        probs, _ = pc.calc_prob_batch_packed(packed)
        wall = (time.perf_counter() - t0) * 1e3
        st = pc.stats()
        return probs, {"wall_ms": wall, "library_call_ms": st.last_prepare_host_us * 1e-3, "device_ms": st.last_device_ms,
                       "launches": int(st.kernel_launches - l0), "events": int(st.last_batch_cov_events),
                       "segments": int(st.last_batch_cov_segments), "touched_mate1_records": int(st.last_records_gathered)}

    one(plain)   # warm-up of every shape the timed loop uses
    one(pen)
    runs = {"plain": [], "penalised": []}
    for _ in range(args.reps):
        p_plain, r = one(plain)
        runs["plain"].append(r)
        p_pen, r = one(pen)
        runs["penalised"].append(r)
    assert pen.calc_prob(base) == last   # stateless
    summary = {}
    for name, rs in runs.items():
        summary[name] = {k: spread([r[k] for r in rs]) for k in ("wall_ms", "library_call_ms", "device_ms")}
        summary[name].update({k: rs[-1][k] for k in ("launches", "events", "segments", "touched_mate1_records")})
        emit({"what": "batch", "context": name, "candidates": len(cands), **summary[name]})
    diff = np.asarray(p_pen) - np.asarray(p_plain)
    emit({"what": "penalty_effect", "candidates_changed": int(np.count_nonzero(diff)), "distinct_offsets": len(set(diff.tolist()))})

    # the sequential alternative on the penalised context: evaluate the candidate, then go back to the base
    rng = np.random.default_rng(7)
    sample = rng.choice(len(cands), size=min(args.sequential_sample, len(cands)), replace=False)
    seq_ms = []
    for i in sample:
        erased, added = cands[int(i)]
        gone = set(erased)
        walks = [w for k, w in enumerate(base) if k not in gone] + [list(w) for w in added]
        t0 = time.perf_counter()
        p, _, _ = pen.calc_prob(walks)
        pen.calc_prob(base)
        seq_ms.append((time.perf_counter() - t0) * 1e3)
        assert p == p_pen[int(i)], (int(i), p, p_pen[int(i)])   # the batch's score, bit for bit
    seq = spread(seq_ms)
    scaled = seq["median"] * len(cands)
    emit({"what": "sequential", "sample": len(sample), "ms_per_candidate_there_and_back": seq,
          "scaled_ms_per_batch": scaled,
          "speedup_batch_vs_sequential": scaled / summary["penalised"]["wall_ms"]["median"],
          "penalised_over_plain_library_call": summary["penalised"]["library_call_ms"]["median"] / summary["plain"]["library_call_ms"]["median"],
          "penalised_over_plain_wall": summary["penalised"]["wall_ms"]["median"] / summary["plain"]["wall_ms"]["median"]})

    if args.shards:
        sharded_leg(args, wl, base, packed, np.asarray(p_pen), summary["penalised"], emit)

    if not args.no_profile:   # a run of its own: per-kernel device time of one batch of each context
        import torch
        from torch.profiler import ProfilerActivity, profile
        for name, pc in (("plain", plain), ("penalised", pen)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                pc.calc_prob_batch_packed(packed)
                torch.cuda.synchronize()
            per = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    key = ev.name if len(ev.name) < 120 else ev.name[:117] + "..."
                    t, n = per.get(key, (0.0, 0))
                    per[key] = (t + ev.device_time_total / 1e3, n + 1)
            emit({"what": "profile", "context": name,
                  "kernels_ms": {k: round(v[0], 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1][0])},
                  "counts": {k: v[1] for k, v in per.items()}})
    plain.close()
    pen.close()
    out.close()


def sharded_leg(args, wl, base, packed, ref_probs, unsharded, emit):
    """The penalised batch over args.shards read-id shard contexts of one GPU, run one after the other. A multi-GPU job
    runs the shards side by side, so besides the sum the record gives the slowest shard of each step (the collectives
    that move the keys and partials between GPUs are not part of it)."""
    from gaml_b200 import api
    n = args.shards
    shards = [api.ProbCalculator.from_workload(wl, shard_of=(r, n)) for r in range(n)]

    def evaluate(walks):
        parts = [pc.calc_prob_partial(walks) for pc in shards]
        if n > 1:
            union = np.concatenate([pc.penalty_export(0) for pc in shards])
            for pc in shards:
                pc.penalty_import(0, union)
        return shards[0].combine(np.stack([p for p, _ in parts]), n, parts[0][1])

    for walks in wl.evals:
        evaluate(walks)

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        return r, (time.perf_counter() - t0) * 1e3

    def once():
        rec = {k: [] for k in ("call_ms", "library_call_ms", "device_ms", "events", "exported", "export_ms", "import_ms",
                               "combine_ms")}
        parts = []
        for pc in shards:
            (part, _), ms = timed(lambda: pc.calc_prob_batch_shard_packed(packed))
            st = pc.stats()
            parts.append(part)
            rec["call_ms"].append(ms)
            rec["library_call_ms"].append(st.last_prepare_host_us * 1e-3)
            rec["device_ms"].append(st.last_device_ms)
            rec["events"].append(int(st.last_batch_cov_events))
            rec["exported"].append(int(st.last_batch_cov_exported))
        keys = []
        for pc in shards:
            k, ms = timed(lambda: pc.batch_penalty_export(0))
            keys.append(k)
            rec["export_ms"].append(ms)
        union = np.concatenate(keys)
        for pc in shards:
            rec["import_ms"].append(timed(lambda: pc.batch_penalty_import(0, union))[1])
        g = np.stack(parts)
        probs = None
        for pc in shards:
            (probs, _), ms = timed(lambda: pc.combine_batch_partials(g))
            rec["combine_ms"].append(ms)
        return probs, rec

    once()   # warm-up
    recs = []
    for _ in range(args.reps):
        probs, rec = once()
        bad = np.flatnonzero(probs != ref_probs)
        assert len(bad) == 0, ("sharded probs differ from the unsharded batch", bad[:8])
        recs.append(rec)
    per_shard = [{k: spread([r[k][i] for r in recs]) for k in ("call_ms", "library_call_ms", "device_ms")} |
                 {"events": recs[-1]["events"][i], "exported": recs[-1]["exported"][i]} for i in range(n)]
    for i, ps in enumerate(per_shard):
        emit({"what": "shard_batch", "n_shards": n, "shard": i, **ps,
              "exported_over_events": ps["exported"] / max(ps["events"], 1)})
    steps = ("call_ms", "export_ms", "import_ms", "combine_ms")
    slowest = {k: spread([max(r[k]) for r in recs]) for k in steps}
    total = spread([sum(sum(r[k]) for k in steps) for r in recs])
    critical = spread([sum(max(r[k]) for k in steps) for r in recs])
    emit({"what": "sharded_batch", "n_shards": n, "candidates": len(ref_probs), "slowest_shard": slowest,
          "sum_over_shards_ms": total, "slowest_shard_path_ms": critical,
          "unsharded_penalised_wall_ms": unsharded["wall_ms"], "unsharded_penalised_library_call_ms": unsharded["library_call_ms"],
          "events": sum(recs[-1]["events"]), "exported": sum(recs[-1]["exported"]), "probs_bit_identical": True})
    for pc in shards:
        pc.close()


if __name__ == "__main__":
    main()
