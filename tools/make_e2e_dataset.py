#!/usr/bin/env python
"""Synthetic end-to-end dataset for the reference's own `gaml` driver (BASELINE config 1 style):
a Velvet-style LastGraph with real node sequences, FASTQ reads sampled from the genome, and a config file.
Both oracle/_ref/gaml_ref (pure reference) and oracle/_ref/gaml_gpu (reference Optimize + moves over the CUDA
ProbCalculator, integration/prob_calculator.h) run on it; tools/compare_traces.py diffs their annealing traces.

LastGraph as LoadGraph consumes it (graph.cc:52-106): first line "<n>\\t...", per node a header line, the
forward sequence and the twin's sequence; "ARC\\t<src>\\t<dst>\\t..." with signed 1-based node ids. The twin
sequence is the exact reverse complement, so walking a path backwards spells the reverse complement.
"""
import argparse
import os

import numpy as np

COMP = str.maketrans("ACGT", "TGCA")


def revcomp(s: str) -> str:
    return s.translate(COMP)[::-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--kind", choices=["single", "paired"], default="single")
    ap.add_argument("--n-unique", type=int, default=10)
    ap.add_argument("--unique-len", type=int, default=10000)
    ap.add_argument("--n-reads", type=int, default=50000)
    ap.add_argument("--iterations", type=int, default=500)
    ap.add_argument("--seed", type=int, default=7)
    # coverage-gap penalty of the paired set (PrepareReadSetFromConfig, gaml.cc:783-872: the paired sweep's step is
    # insert_mean - penalty_step); both omitted: no penalty keys, the reference's defaults
    ap.add_argument("--penalty-constant", type=float, default=None)
    ap.add_argument("--penalty-step", type=float, default=None)
    args = ap.parse_args()
    os.makedirs(args.outdir, exist_ok=True)
    rng = np.random.default_rng(args.seed)

    def randseq(n):
        return "".join(np.array(list("ACGT"))[rng.integers(0, 4, size=n)])

    lens = (args.unique_len * (1 + 0.2 * (2 * rng.random(args.n_unique) - 1))).astype(int)
    nodes = [randseq(int(n)) for n in lens]
    n_rep = 3
    reps = [randseq(400) for _ in range(n_rep)]
    nodes += reps
    units = list(range(args.n_unique))
    slots = rng.choice(args.n_unique - 1, size=2 * n_rep, replace=False)
    for i, b in sorted(((i, int(b) + 1) for i, b in enumerate(slots)), key=lambda t: -t[1]):
        units.insert(b, args.n_unique + i // 2)
    genome = "".join(nodes[u] for u in units)

    with open(os.path.join(args.outdir, "LastGraph"), "w") as f:
        f.write(f"{len(nodes)}\t0\t31\t1\n")
        for i, s in enumerate(nodes):
            f.write(f"NODE\t{i + 1}\t{len(s)}\t0\t0\t0\t0\n{s}\n{revcomp(s)}\n")
        seen = set()
        for a, b in zip(units[:-1], units[1:]):
            if (a, b) not in seen:
                seen.add((a, b))
                f.write(f"ARC\t{a + 1}\t{b + 1}\t1\n")

    def mutate(s):
        a = np.array(list(s))
        m = rng.random(len(a)) < 0.01
        a[m] = np.array(list("ACGT"))[rng.integers(0, 4, size=int(m.sum()))]
        return "".join(a)

    def fastq(path, reads):
        with open(path, "w") as f:
            for i, s in enumerate(reads):
                f.write(f"@r{i}\n{s}\n+\n{'I' * len(s)}\n")

    cfg = [f"graph={args.outdir}/LastGraph", f"max_iterations={args.iterations}", f"output_prefix={args.outdir}/out", ""]
    if args.kind == "single":
        reads = []
        for _ in range(args.n_reads):
            p = int(rng.integers(0, len(genome) - 100))
            s = genome[p:p + 100]
            reads.append(mutate(revcomp(s) if rng.random() < 0.5 else s))
        fastq(os.path.join(args.outdir, "reads.fastq"), reads)
        cfg += ["[rs]", "type=single", f"filename={args.outdir}/reads.fastq", f"cache_prefix={args.outdir}/nocache"]
    else:
        r1, r2 = [], []
        for _ in range(args.n_reads):
            ins = max(200, int(round(rng.normal(300, 30))))
            p = int(rng.integers(0, len(genome) - ins))
            frag = genome[p:p + ins]
            if rng.random() < 0.5:
                frag = revcomp(frag)
            r1.append(mutate(frag[:100]))
            r2.append(mutate(revcomp(frag[-100:])))
        fastq(os.path.join(args.outdir, "reads_1.fastq"), r1)
        fastq(os.path.join(args.outdir, "reads_2.fastq"), r2)
        cfg += ["[rs]", "type=paired", f"filename1={args.outdir}/reads_1.fastq", f"filename2={args.outdir}/reads_2.fastq",
                "insert_mean=300", "insert_std=30", f"cache_prefix={args.outdir}/nocache"]
        if args.penalty_constant is not None:
            cfg.append(f"penalty_constant={args.penalty_constant:g}")
        if args.penalty_step is not None:
            cfg.append(f"penalty_step={args.penalty_step:g}")
    with open(os.path.join(args.outdir, "gaml.cfg"), "w") as f:
        f.write("\n".join(cfg) + "\n")
    print(f"genome {len(genome)} bp, {len(nodes)} nodes, {args.n_reads} {args.kind} reads -> {args.outdir}")


if __name__ == "__main__":
    main()
