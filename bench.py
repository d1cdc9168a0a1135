#!/usr/bin/env python
"""bench.py — alignments scored/s of the GAML assembly-likelihood path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA path through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU path (oracle/_ref)
  python bench.py ... --dump-outputs DIR                   also write the last timed step's results to DIR/*.npy

A step = one full log-likelihood evaluation (`ProbCalculator::CalcProb` on a fresh ScoringState,
prob_calculator.h:63-109).
  N = 1: BASELINE config 2 — synthetic 4.6 Mbp genome, 2 M innie read pairs 2x100 bp, insert 300+-30, injected cache.
  N > 1: BASELINE config 4 — the 100 Mbp / 10 000-node genome with 6.25 M read pairs (one eighth of the 50 M) per GPU,
         sharded by read id: N = 8 is the whole of config 4, N = 2 / 4 the same genome at a quarter / half of the coverage
         (weak scaling: the per-GPU shard is fixed).
Every rank scores its shard; the ranks' 64-byte result lines are exchanged by the evaluation's own kernels over NVLink
peer memory (--exchange peer), a host shared-memory segment the kernels write into (host, the default: the fastest end to
end in the A/B on the 8-GPU box, profiles/r02_exchange_ab.md) or one ncclAllReduce (nccl), and every rank combines them exactly.

One JSON line on stdout (rank 0). `value` is device time with all inputs resident in HBM — CUDA events around each
evaluation's kernel chain on the library's stream (with --exchange peer the chain ends with the kernel that has received
every rank's line); `value_incl_exchange` is the wall clock from the chain's submission until the rank holds every rank's
result line; L2 flushed between steps, all ranks released together after the flush. `e2e` is the same metric through gaml_calc_prob_partial / gaml_calc_prob_gathered with host buffers in and out,
wall clock. `roofline` is the dominant kernel of this rank against the measured HBM copy peak. The incremental (delta)
evaluations of the annealing loop are reported beside it as `sa_iters_per_s`.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

C2 = dict(n_unique=460, unique_len=10000, n_pairs=2_000_000)
WORKLOAD_NAME = ("C2: synthetic 4.6 Mbp genome (460 x ~10 kbp nodes + 3 repeat nodes x2), 2M innie read pairs 2x100 bp, "
                 "insert 300+-30, edit distance 0-2, 10% of mates with a second alignment; one walk per long node")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


C4 = dict(n_unique=10000, unique_len=10000, n_pairs=50_000_000)


def make_workload(world: int, rank: int, n_evals: int, scale: float = 1.0, kind: str = "c2"):
    """Config 2 per GPU: the genome and read set grow with `world`, each rank generates only its shard.
    kind="c4shard": BASELINE config 4 (100 Mbp, 50 M pairs) as ONE of eight read-id shards per GPU — rank r of
    `world` GPUs holds shard r (so --gpus 8 is the whole of config 4, --gpus 1 is one eighth of it)."""
    from gaml_b200 import synth
    if kind == "c4shard":
        per = C4["n_pairs"] // 8
        lo, hi = rank * per, (rank + 1) * per
        wl = synth.paired_workload(C4["n_unique"], C4["unique_len"], per * world, n_evals=n_evals, seed=44, read_lo=lo, read_hi=hi)
        return wl, (lo, hi)
    n_pairs_total = int(C2["n_pairs"] * scale) * world
    per = (n_pairs_total + world - 1) // world
    lo, hi = rank * per, min((rank + 1) * per, n_pairs_total)
    wl = synth.paired_workload(int(C2["n_unique"] * scale) * world, C2["unique_len"], n_pairs_total, n_evals=n_evals,
                               seed=42, read_lo=lo, read_hi=hi)
    return wl, (lo, hi)


def load_calculator(wl, shard, device, world=1, torch_dev=None):
    """Builds the context from a (possibly shard-only) workload. The skip rule (graph.cc:577-596) needs each
    key's largest position over ALL reads, so with several ranks the per-key maxima of the shards are
    MAX-all-reduced first (keys are enumerated identically on every rank)."""
    from gaml_b200 import api
    pc = api.ProbCalculator(wl.node_len, wl.normalize_map, device)
    spec = wl.sets[0]
    lo, hi = shard
    sid = pc.add_readset(spec, shard=(lo, hi), max_read_len=[int(spec.read_len[0].max()), int(spec.read_len[1].max())],
                         lens_are_local=True)
    key_max = {}
    if world > 1:
        import torch
        import torch.distributed as dist
        flat = [int(recs["position"].max()) if len(recs) else api.INT32_MIN for cache in spec.caches for recs in cache.values()]
        t = torch.tensor(flat, dtype=torch.int64, device=torch_dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        it = iter(t.cpu().tolist())
        for mate, cache in enumerate(spec.caches):
            for key in cache:
                key_max[(mate, key)] = int(next(it))
    t0 = time.perf_counter()
    nbytes = 0
    for mate, cache in enumerate(spec.caches):
        for key, recs in cache.items():
            pc.cache_insert(sid, mate, key, recs, key_max.get((mate, key), api.INT32_MIN))
            nbytes += recs.nbytes
    pc.commit()
    return pc, time.perf_counter() - t0, nbytes


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.rows = []
        self.proc = None
        self.device = device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)   # a run that fails before stop() must not leave the poller running
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t0 = time.time()
        while not self.rows and time.time() - t0 < 5.0:   # nvidia-smi needs a second to come up on an 8-GPU box
            time.sleep(0.05)
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_READ_VALUES_MAX = 1 << 21   # every read of config 2 (2 M pairs); a larger shard is sampled


def dump_outputs(out_dir: str, pc, gathered, total_len: int, world: int) -> None:
    """Writes what the timed evaluation returned in its last step, as float64 .npy files: the partial sums of every rank
    (`partials`), their exact combination (`prob`, `floored` = [set][floored reads, reads], `total_len`) and the per-read
    values of this rank's first read set (`read_values`; for a set of more than DUMP_READ_VALUES_MAX reads a fixed, seeded
    sample of them, whose read indices go to `read_index`)."""
    os.makedirs(out_dir, exist_ok=True)
    prob, zeros, tl = pc.combine(gathered, world, total_len)
    arrays = {"partials": gathered, "prob": [prob], "floored": zeros, "total_len": [tl]}
    values = pc.read_values(0)
    if len(values) > DUMP_READ_VALUES_MAX:
        idx = np.sort(np.random.default_rng(0).choice(len(values), DUMP_READ_VALUES_MAX, replace=False))
        values = values[idx]
        arrays["read_index"] = idx
    arrays["read_values"] = values
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------
def shard_workload(wl, lo, hi):
    """Workload restricted to reads [lo,hi) with ids shifted to 0 — what one CPU process scores."""
    from gaml_b200.workload import ReadSetSpec, Workload
    spec = wl.sets[0]
    caches = []
    for cache in spec.caches:
        c = {}
        for k, recs in cache.items():
            m = (recs["read_id"] >= lo) & (recs["read_id"] < hi)
            r = recs[m].copy()
            r["read_id"] -= lo
            c[k] = r
        caches.append(c)
    s2 = ReadSetSpec(kind=spec.kind, n_reads=hi - lo, read_len=[rl[lo:hi] for rl in spec.read_len], caches=caches,
                     mismatch_prob=spec.mismatch_prob, match_prob=spec.match_prob, insert_mean=spec.insert_mean,
                     insert_std=spec.insert_std, min_prob_per_base=spec.min_prob_per_base,
                     min_prob_start=spec.min_prob_start, weight=spec.weight, step=spec.step)
    return Workload(node_len=wl.node_len, normalize_map=wl.normalize_map, sets=[s2], evals=[wl.evals[0]])


def cpu_binary():
    ref = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
    if os.path.exists(ref):
        return ref, "reference"
    import __graft_entry__ as entry
    entry.build()
    return os.path.join(ROOT, "oracle", "gaml_oracle"), "port"


def run_cpu(wl, n_procs: int, repeats: int, tmp: str):
    """n_procs independent processes of the reference's single-threaded scorer, each on a contiguous
    read-id block; returns per-repeat wall (max over processes) and the alignments scored per repeat."""
    from gaml_b200 import workload
    binary, kind = cpu_binary()
    n = wl.sets[0].n_reads
    per = (n + n_procs - 1) // n_procs
    procs, outs, aligns = [], [], 0
    for p in range(n_procs):
        lo, hi = p * per, min((p + 1) * per, n)
        if hi <= lo:
            continue
        sw = shard_workload(wl, lo, hi)
        aligns += sw.sets[0].n_records()
        wp, rp = os.path.join(tmp, f"cpu{p}.wl"), os.path.join(tmp, f"cpu{p}.res")
        workload.write_workload(wp, sw)
        outs.append(rp)
        procs.append((binary, wp, rp))
    running = [subprocess.Popen([b, wp, rp, "0", str(repeats)], cwd=tmp, stdout=subprocess.DEVNULL,
                                stderr=subprocess.DEVNULL) for b, wp, rp in procs]
    for r in running:
        if r.wait() != 0:
            raise RuntimeError("CPU scorer failed")
    secs = np.array([[e.seconds for e in workload.read_results(rp)] for rp in outs])   # [procs, repeats]
    return secs.max(axis=0), aligns, kind


def workload_kind(args, world: int) -> str:
    return args.workload if args.workload != "auto" else ("c2" if world == 1 else "c4shard")


def config_for(kind: str, world: int, scale: float = 1.0) -> dict:
    """The `config` object of the JSON line — identical for both arms."""
    if kind == "c2":
        name = WORKLOAD_NAME + (f" — per GPU; {world} GPUs hold {world}x the genome and reads, sharded by read id" if world > 1 else "")
        pairs = int(C2["n_pairs"] * scale) * world
    else:
        name = (f"C4: synthetic 100 Mbp genome (10000 x ~10 kbp nodes + 3 repeat nodes x2), innie read pairs 2x100 bp, insert 300+-30, "
                f"edit distance 0-2, 10% of mates with a second alignment; one walk per long node; {C4['n_pairs'] // 8} read pairs "
                f"(1/8 of config 4's 50 M) per GPU, sharded by read id over {world} GPU(s)" + (" = the whole of config 4" if world == 8 else ""))
        pairs = (C4["n_pairs"] // 8) * world
    return {"workload": name, "step": "one full logL evaluation (CalcProb on a fresh ScoringState)", "read_pairs": pairs,
            "parallelism": f"read-id shards x{world}" if world > 1 else "one GPU"}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    n_procs = max(1, min(cores, 64))
    kind = workload_kind(args, world)
    # the job's workload is `world` shards; the CPU scores shard 0 of it as the bounded sample (a rate, not a total)
    wl, (lo, hi) = make_workload(world, 0, 1, scale=args.scale, kind=kind)
    assert lo == 0
    wl.sets[0].n_reads = hi - lo     # rank 0's shard holds reads [0, hi): read ids and the length arrays are already local
    with tempfile.TemporaryDirectory() as tmp:
        per_step, aligns, kind_cpu = run_cpu(wl, n_procs, args.steps + args.warmup, tmp)
    timed = per_step[args.warmup:]
    total = float(timed.sum())
    value = aligns * len(timed) / total
    line = {
        "impl": "reference", "metric": "alignments_scored_per_s", "value": value, "unit": "alignments/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(timed),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_for(kind, world, args.scale),
        "alignments_per_step": aligns,
        "cpu_baseline": {"value": value, "unit": "alignments/s", "cores": n_procs, "kind": kind_cpu,
                         "sample": (f"one GPU's shard of the workload ({wl.sets[0].n_reads} read pairs) split into {n_procs} contiguous read-id "
                                    f"blocks, one single-threaded reference process per block, {len(timed)} timed full evaluations each; "
                                    "step time = slowest process; the rate stands for the whole job (the CPU's cores are busy either way)")},
        "e2e": {"value": value, "unit": "alignments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def ncu_traffic(kind: str):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture of THIS workload, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kind, {}).get("paired_stream_kernel_dram_bytes_per_launch")
        except Exception:
            return None
    return None


def make_candidates(base, n, rng):
    """BASELINE config 5's mix: 40 % extend, 30 % interchange, 30 % disconnect, each on 1-2 walks of `base`."""
    cands = []
    multi = [i for i, w in enumerate(base) if sum(1 for x in w if x >= 0) >= 2]
    for _ in range(n):
        u = rng.random()
        if u < 0.4 or not multi:                                   # extend: join two walks (sometimes with a gap)
            i, j = (int(x) for x in rng.choice(len(base), size=2, replace=False))
            mid = [-int(rng.integers(1, 400))] if rng.random() < 0.3 else []
            cands.append(([i, j], [list(base[i]) + mid + list(base[j])]))
        elif u < 0.7:                                              # interchange: swap the tails of two walks
            i = multi[int(rng.integers(len(multi)))]
            j = int(rng.integers(len(base)))
            if j == i:
                j = (j + 1) % len(base)
            ci = int(rng.integers(1, len(base[i])))
            cj = int(rng.integers(0, len(base[j]) + 1))
            a, b = list(base[i][:ci]) + list(base[j][cj:]), list(base[j][:cj]) + list(base[i][ci:])
            ok = all(w and w[0] >= 0 and w[-1] >= 0 for w in (a, b))
            cands.append(([i, j], [a, b]) if ok else ([i], [[(x ^ 1) if x >= 0 else x for x in reversed(base[i])]]))
        else:                                                      # disconnect: split one walk
            i = multi[int(rng.integers(len(multi)))]
            nodes_pos = [t for t in range(1, len(base[i])) if base[i][t] >= 0 and base[i][t - 1] >= 0]
            if not nodes_pos:
                cands.append(([i], [[(x ^ 1) if x >= 0 else x for x in reversed(base[i])]]))
            else:
                cut = nodes_pos[int(rng.integers(len(nodes_pos)))]
                cands.append(([i], [list(base[i][:cut]), list(base[i][cut:])]))
    return cands


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gaml_b200", choices=["gaml_b200", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the c2 workload (debug only; 1.0 = config 2)")
    ap.add_argument("--delta-steps", type=int, default=200)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the C1 / C3 legs")
    ap.add_argument("--no-dropin", action="store_true", help="skip the drop-in ProbCalculator leg (oracle/_ref/gpu_harness)")
    ap.add_argument("--workload", default="auto", choices=["auto", "c2", "c4shard"],
                    help="auto (default): config 2 on one GPU, one eighth of config 4 per GPU on several")
    ap.add_argument("--batch", type=int, default=1024, help="candidate moves per gaml_calc_prob_batch launch (0 = skip)")
    ap.add_argument("--exchange", default="host", choices=["peer", "host", "nccl"],
                    help="how the ranks' result lines meet (N > 1): host shared memory written by the kernels (default: the fastest end to "
                         "end on the 8-GPU box, profiles/r02_exchange_ab.md), NVLink peer memory, ncclAllReduce")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed evaluation to DIR/<name>.npy, so that two builds can be compared "
                         "output for output: all ranks' partial sums and their combination, rank 0's per-read values of its "
                         "first read set (CUDA arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "gaml_b200":
        ap.error("--dump-outputs needs --impl gaml_b200: the reference arm reports timings only")
    args.warmup = max(args.warmup, 3) if args.impl == "gaml_b200" else args.warmup

    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    from gaml_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: anything a library prints there meanwhile (NCCL's version banner) goes to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the scoring path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    kind = workload_kind(args, world)
    t_gen = time.perf_counter()
    n_evals = 2 + args.delta_steps
    wl, shard = make_workload(world, rank, n_evals, scale=args.scale, kind=kind)
    t_gen = time.perf_counter() - t_gen
    pc, t_upload, cache_bytes = load_calculator(wl, shard, local_rank, world, dev)
    log(f"[rank {rank}] workload {kind} generated in {t_gen:.1f}s; cache of {cache_bytes / 1e6:.1f} MB inserted+CSR built in {t_upload:.2f}s")
    walks0 = wl.evals[0]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    flush_view = flush.view(torch.int32)
    flush_sink = torch.zeros((), dtype=torch.int64, device=dev)

    exchange_name = None
    if world > 1:
        from gaml_b200 import dist as gdist
        if args.exchange != "nccl":
            gdist.NcclExchange(rank, world).attach(pc)   # the communicator also serves the candidate batches; attached first:
                                                         # a kernel-fused exchange attached after it takes over the result lines
        if args.exchange == "peer":
            gdist.PeerExchange(rank, world).attach(pc)
            exchange_name = ("NVLink peer memory: the block that completes a read set stores its 64-byte result line into every rank's "
                             "exchange buffer; the chain's last kernel waits for all ranks' lines (inside the timed region)")
        elif args.exchange == "nccl":
            gdist.NcclExchange(rank, world).attach(pc)
            exchange_name = "one ncclAllReduce(sum, fp64) of the ranks' result lines per evaluation on the library's stream"
        else:
            gdist.ResultExchange(rank, world).attach(pc)
            exchange_name = "host shared-memory segment written by the kernels' last blocks, read by every rank's host"
    flat0 = api.FlatWalks(walks0)

    def flush_l2():
        flush.fill_(1)            # write > L2 ...
        flush_sink.copy_(flush_view.sum())   # ... then read it back so L2 is left holding CLEAN foreign lines
        torch.cuda.synchronize()

    sync_t = torch.zeros(1, dtype=torch.int64, device=dev) if world > 1 else None

    def rendezvous():
        """All ranks leave together AFTER their own flush: a step's clock never contains another rank's flush. A barrier
        alone releases the ranks tens of microseconds apart (more than the exchange costs), so rank 0 then names an instant
        0.3 ms ahead on the node's monotonic clock and every rank spins until it."""
        if world > 1:
            dist.barrier()
            if rank == 0:
                sync_t[0] = time.monotonic_ns() + 300_000
            dist.broadcast(sync_t, 0)
            t_start = int(sync_t.item())
            while time.monotonic_ns() < t_start:
                pass

    def finish_all():
        if world > 1:
            g, tl = pc.finish_gathered()
            return g, tl
        part, tl = pc.finish()
        return part[None, :], tl

    def full_step_device():
        """One full evaluation, inputs resident: (device ms of the evaluation's chain incl. the exchange, ms of the
        dominant kernel, gathered partials, total_len)."""
        pc.reset_state()
        pc.prepare(walks0)
        flush_l2()
        rendezvous()
        t0 = time.perf_counter()
        pc.launch()
        g, tl = finish_all()
        wall = time.perf_counter() - t0
        st = pc.stats()
        return st.last_device_ms, st.last_score_kernel_ms, g, tl, wall

    def eval_all_ranks(fw):
        """One evaluation through the C ABI, all ranks' partials combined: (prob, zeros, total_len)."""
        if world > 1:
            g, tl = pc.calc_prob_gathered_flat(fw)
            return pc.combine(g, world, tl)
        part, tl = pc.calc_prob_partial_flat(fw)
        return pc.combine(part[None, :], 1, tl)   # the C ABI's walk layout: host int32 ids + int64 offsets (what a C++ caller holds)

    # e2e alternates between the start walk set and the one a single annealing move later: every step is a full evaluation of
    # a walk list that differs from the one evaluated before it, so the library flattens it and uploads its slot tables
    # each time (an unchanged list would find its tables on the device already: reported separately as e2e_same_walks)
    alts = []
    for w in wl.evals[1:]:   # (a scripted move can be a no-op: take lists that differ from the start list and from each other)
        if w != walks0 and all(w != a for a in alts):
            alts.append(w)
        if len(alts) == 3:
            break
    if not alts:
        raise RuntimeError("the workload's trajectory never leaves the start walks: e2e needs a second walk set")
    e2e_cycle = [flat0] + [api.FlatWalks(a) for a in alts]

    def full_step_e2e(fw=None):
        """(wall seconds of the C-ABI call incl. the exchange + combine, result); reset, L2 flush and the rendezvous are outside."""
        pc.reset_state()
        flush_l2()
        rendezvous()
        t0 = time.perf_counter()
        res = eval_all_ranks(fw if fw is not None else flat0)
        return time.perf_counter() - t0, res

    # ---- value: device-resident inputs, CUDA events, L2 flushed between steps ----
    pc.set_profiling(1)   # two events around each evaluation, nodes of its CUDA graph
    for _ in range(args.warmup):
        full_step_device()
    sampler = ClockSampler(local_rank)
    launches0 = pc.stats().kernel_launches
    barrier()
    import gc
    gc.disable()              # no collector pauses inside the timed loops (every rank waits for the slowest one)
    if rank == 0:             # one nvidia-smi poller per job, not per rank
        sampler.start()
    dev_ms, wall_ms = 0.0, 0.0
    for _ in range(args.steps):
        d, _k, g_full, tl, wall = full_step_device()
        dev_ms += max_over_ranks(d) if world > 1 else d   # per step: the slowest rank's chain
        wall_ms += 1e3 * max_over_ranks(wall)             # launch -> every rank's result line received, slowest rank
    barrier()
    st = pc.stats()
    launches = st.kernel_launches - launches0
    a_local, bytes_local = st.last_records_gathered, st.last_algorithmic_bytes
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pc, g_full, tl, world)
    # roofline timing of the streaming pass: the same steps again with the library's per-kernel events switched on
    # (an event between two kernels serialises them, so the chained launches of the timed region above are given up
    # at the two boundaries of the streaming pass; the kernels themselves are identical)
    pc.set_profiling(2)
    full_step_device()
    ker_ms, ker_list = 0.0, []
    for _ in range(args.steps):
        ker_list.append(full_step_device()[1])
        ker_ms += ker_list[-1]
    ker_list.sort()
    # device timeline of one more step: globaltimer stamps at each kernel's first block start / last block end
    # (no events, chain and graph intact) — shows how the kernels of an evaluation overlap
    pc.set_profiling(3)
    full_step_device()
    full_step_device()
    timeline = {k: [round(a, 2), round(b, 2)] for k, (a, b) in pc.read_timeline().items()}
    pc.set_profiling(0)
    st = pc.stats()
    full_overflow_reads = {"multi_pass_items": int(st.last_multi_items), "many_placement_pass_reads": int(st.last_overflow_reads),
                           "scratch_placements": int(st.last_scratch_placements)}
    a_total = sum_over_ranks(float(a_local))

    # ---- e2e: host walks in, host result out, wall clock, exchange included ----
    n_cyc = len(e2e_cycle)
    for k in range(-(-args.warmup // n_cyc) * n_cyc):
        full_step_e2e(e2e_cycle[k % n_cyc])
    barrier()
    e2e_s, e2e_aln, h2d, h2d_max, prep_full_us = 0.0, 0.0, 0, 0, 0.0
    st0 = pc.stats()
    for k in range(args.steps):
        dt, (prob_k, zeros_k, tl_k) = full_step_e2e(e2e_cycle[k % n_cyc])
        e2e_s += max_over_ranks(dt)
        st = pc.stats()
        e2e_aln += float(st.last_records_gathered)
        h2d += int(st.last_h2d_bytes)
        h2d_max = max(h2d_max, int(st.last_h2d_bytes))
        prep_full_us += st.last_prepare_host_us / args.steps
        if k % n_cyc == 0:
            prob, zeros, tl_full = prob_k, zeros_k, tl_k
    st1 = pc.stats()
    e2e_how = {"walk_lists_cycled": n_cyc, "patched": int(st1.full_patch_evals - st0.full_patch_evals),
               "tables_resident": int(st1.full_reuse_evals - st0.full_reuse_evals),
               "all_walks_flattened": args.steps - int(st1.full_patch_evals - st0.full_patch_evals) - int(st1.full_reuse_evals - st0.full_reuse_evals)}
    h2d = h2d // max(args.steps, 1)
    barrier()
    e2e_aln = sum_over_ranks(e2e_aln)
    d2h = pc.stats().last_d2h_bytes
    # the same walk set over and over (what `value` evaluates): its slot tables are on the device already
    same_s = 0.0
    full_step_e2e(flat0)
    for _ in range(max(args.steps // 2, 1)):
        dt, _res = full_step_e2e(flat0)
        same_s += max_over_ranks(dt)
    same_steps = max(args.steps // 2, 1)
    barrier()
    # a list unrelated to the one on the device (the start list reversed, alternating with the start list): no alignment
    # between consecutive lists, every walk is flattened and all slot updates are uploaded
    flat_rev = api.FlatWalks(list(reversed(walks0)))
    cold_s, cold_h2d, cold_steps = 0.0, 0, max(args.steps // 4, 2)
    for k in range(cold_steps + 2):
        dt, _res = full_step_e2e(flat0 if k & 1 else flat_rev)
        if k >= 2:
            cold_s += max_over_ranks(dt)
            cold_h2d = max(cold_h2d, int(pc.stats().last_h2d_bytes))
    cold_info = {"value": a_total * cold_steps / cold_s, "unit": "alignments/s", "ms_per_step": 1e3 * cold_s / cold_steps,
                 "h2d_bytes_per_step": cold_h2d,
                 "note": "the start list and its reverse in turn: consecutive lists do not align, all walks are flattened on the host"}
    full_step_e2e(flat0)
    barrier()
    clocks = sampler.stop()

    # ---- incremental evaluations of the annealing loop (delta kernel + O(R) pass), ranks in lockstep ----
    pc.reset_state()
    full_step_e2e()
    seq = wl.evals[1:1 + args.delta_steps]
    seq_flat = [api.FlatWalks(w) for w in seq]
    barrier()
    only0 = pc.stats().delta_only_evals
    t0 = time.perf_counter()
    slow_evals = []
    for k_eval, nodes_offs in enumerate(seq_flat):
        t_e = time.perf_counter()
        eval_all_ranks(nodes_offs)
        if time.perf_counter() - t_e > 1e-3:
            s_ = pc.stats()
            slow_evals.append((k_eval, round((time.perf_counter() - t_e) * 1e3, 2), round(s_.last_prepare_host_us), round(s_.last_launch_host_us),
                               round(s_.last_finish_host_us), int(s_.last_was_full)))
    barrier()
    delta_s = max_over_ranks(time.perf_counter() - t0)
    if slow_evals:
        log(f"[rank {rank}] incremental evaluations over 1 ms (index, ms, prepare/launch/finish us, full): {slow_evals[:8]}")
    delta_only = pc.stats().delta_only_evals - only0
    # the same trajectory once more, untimed, reading the library's per-evaluation device time and counters
    pc.reset_state()
    full_step_e2e()
    pc.set_profiling(1)
    delta_dev_ms, touched, delta_bytes, prep_us = 0.0, 0, 0, 0.0
    for nodes_offs in seq_flat:
        eval_all_ranks(nodes_offs)
        s2 = pc.stats()
        delta_dev_ms += s2.last_device_ms
        touched += s2.last_records_gathered
        delta_bytes += s2.last_algorithmic_bytes
        prep_us += s2.last_prepare_host_us
    pc.set_profiling(0)

    # ---- BASELINE config 5: 1024 candidate moves scored per launch against the current state (stateless) ----
    base = seq[-1] if seq else walks0
    batch_info = None
    if args.batch > 0:
        cands = make_candidates(base, args.batch, np.random.default_rng(123))
        packed = pc.pack_candidates(cands)

        def run_batch():
            if world == 1:   # one GPU: the library combines (gaml_calc_prob_batch), as a host caller would use it
                return list(pc.calc_prob_batch_packed(packed)[0])
            return list(pc.calc_prob_batch_gathered_packed(packed)[0])   # one all-reduce of all candidates' partials inside the library
        run_batch()
        launches_b0 = pc.stats().kernel_launches
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            batch_probs = run_batch()
        barrier()
        batch_s = max_over_ranks(time.perf_counter() - t0) / 3
        stb = pc.stats()
        batch_info = {"candidates_per_launch": args.batch, "ms_per_batch": 1e3 * batch_s, "candidates_per_s": args.batch / batch_s,
                      "device_ms_per_batch": stb.last_device_ms, "library_call_ms": stb.last_prepare_host_us * 1e-3,
                      "touched_mate1_records": int(stb.last_records_gathered),
                      "mix": "40% extend / 30% interchange / 30% disconnect on the walk set reached after the incremental run",
                      "kernel_launches_per_batch": int((pc.stats().kernel_launches - launches_b0) / 3),
                      "best_candidate_prob": float(max(batch_probs)),
                      "note": "gaml_calc_prob_batch (N=1) / gaml_calc_prob_batch_gathered (N>1: one ncclAllReduce of all candidates' exact partials inside the library): "
                              "host arrays in, scores out, wall clock; each score is bit-identical to a sequential gaml_calc_prob of that candidate"}

    peak, peak_src = measured_peak()
    achieved = bytes_local / (ker_ms / args.steps * 1e-3) / 1e9
    cfg = config_for(kind, world, args.scale)
    line = {
        "metric": "alignments_scored_per_s", "value": a_total * args.steps / (dev_ms * 1e-3), "unit": "alignments/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "alignments_per_step": int(a_total),
        "value_incl_exchange": {"value": a_total * args.steps / (wall_ms * 1e-3), "unit": "alignments/s", "ms_per_step": wall_ms / args.steps,
                                "note": "inputs resident as for `value`; wall clock from the kernel chain's submission until THIS rank holds every rank's "
                                        "result line (N > 1) / its own (N = 1), max over ranks: device time + launch + the exchange"},
        "measurement": {"l2": "flushed between steps (256 MiB write, then read back so L2 holds clean foreign lines)",
                        "timing": "CUDA events around each evaluation's kernel chain (nodes of its CUDA graph on the library stream); N > 1: all ranks "
                                  "released together after their flush, the chain ends with the exchange's gather kernel, per step the max over ranks",
                        "exchange": exchange_name},
        "roofline": {"bound": "hbm", "kernel": "paired_stream_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": ncu_traffic(kind), "peak_source": peak_src, "per": "GPU (rank 0's shard)",
                     "algorithmic_bytes_per_launch": int(bytes_local), "kernel_ms": ker_ms / args.steps, "kernel_ms_median": ker_list[len(ker_list) // 2], "kernel_ms_min": ker_list[0], "kernel_ms_max": ker_list[-1],
                     "timing": f"CUDA events around the streaming kernel (rare shapes + tier 1 + tier 2, one launch) on the library stream, {args.steps} extra "
                               "steps after the timed region with gaml_set_profiling 2, L2 flushed between steps"},
        "e2e": {"value": e2e_aln / e2e_s, "unit": "alignments/s", "h2d_bytes_per_step": int(h2d), "h2d_bytes_max": int(h2d_max), "full_evaluations": e2e_how,
                "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_s / args.steps, "host_prepare_us": prep_full_us,
                "note": "gaml_calc_prob_partial (N=1) / gaml_calc_prob_gathered (N>1, the exchange included) + exact combine: host walk arrays in, "
                        "score out, wall clock per step (max over ranks), L2 flushed between steps, ranks released together after the flush; the "
                        "steps cycle through walk lists one to three annealing moves apart, so every step's list differs from the one evaluated before "
                        "it; the library keeps the slot tables of one BASE list on the device and builds + uploads only the updates of the "
                        "keys the changed walks look up (h2d_bytes_per_step = mean, full_evaluations = how each step was prepared); a list "
                        "unrelated to the resident one flattens every walk: e2e_cold_list; the alignment cache is resident state like the "
                        "reference's aligment_cache_"},
        "e2e_cold_list": cold_info,
        "e2e_same_walks": {"value": a_total * same_steps / same_s, "unit": "alignments/s", "ms_per_step": 1e3 * same_s / same_steps,
                           "note": "the same call on the walk set evaluated last (a fresh ScoringState over unchanged walks): the set's slot tables "
                                   "are still on the device, nothing is flattened or uploaded"},
        "gpu_launches": int(launches),
        "device_timeline_us": timeline,
        "ordered_paths_per_full_eval": full_overflow_reads,
        "clocks": clocks,
        "sa_iters_per_s": len(seq) / delta_s,
        "incremental": {"evals": len(seq), "e2e_ms_per_eval": 1e3 * delta_s / max(len(seq), 1),
                        "device_ms_per_eval": delta_dev_ms / max(len(seq), 1), "touched_alignments_per_eval": touched / max(len(seq), 1),
                        "algorithmic_bytes_per_eval": delta_bytes / max(len(seq), 1), "host_prepare_us_per_eval": prep_us / max(len(seq), 1),
                        "evals_without_O(R)_pass": int(delta_only),
                        "note": "each evaluation = gaml_calc_prob_partial / gaml_calc_prob_gathered on host walk arrays (+ combine), wall clock, ranks in "
                                "lockstep; an evaluation whose total length equals the previous one's swaps the touched reads' terms in the exact "
                                "running total instead of re-summing all reads"},
        "batch": batch_info,
        "cache_upload": {"seconds": t_upload, "bytes": int(cache_bytes)},
        "result": {"prob": prob, "total_len": tl_full, "floored": zeros[0][0]},
    }

    # ---- cache growth (SURVEY §7.3 "the arena must support append"): the same trajectory on a context that starts with the
    #      keys of the first walk set only and is handed each new window when a walk first needs it (what the annealing loop's
    #      on-demand aligner does, graph.cc:1967-1968) — insert + evaluate timed together ----
    if rank == 0 and world == 1 and args.delta_steps > 0:
        from gaml_b200 import synth
        spec = wl.sets[0]
        pc2 = api.ProbCalculator(wl.node_len, wl.normalize_map, local_rank)
        sid2 = pc2.add_readset(spec)
        have = [set(), set()]

        def missing_keys(walks):
            out = []
            for k in synth.short_keys_for_walks(walks, wl.node_len, with_single_node=True):
                for m in range(2):
                    if k not in have[m] and k in spec.caches[m]:
                        have[m].add(k)
                        out.append((m, k, spec.caches[m][k]))
            return out
        for m, k, recs in missing_keys(walks0):
            pc2.cache_insert(sid2, m, k, recs)
        pc2.calc_prob_partial_flat(flat0)
        grow_us, warm_us, new_keys, new_recs = [], [], 0, 0
        for fw, walks in zip(seq_flat, seq):
            todo = missing_keys(walks)
            inserts = [pc2.prepared_insert(sid2, m, k, recs) for m, k, recs in todo]   # (array conversions outside the clock)
            t0 = time.perf_counter()
            for ins in inserts:
                ins()
            part2, _tl2 = pc2.calc_prob_partial_flat(fw)
            dt = (time.perf_counter() - t0) * 1e6
            (grow_us if todo else warm_us).append(dt)
            new_keys += len(todo)
            new_recs += sum(len(r) for _, _, r in todo)
        st2 = pc2.stats()
        line["append"] = {"evals_inserting_keys": len(grow_us), "us_per_eval_inserting": float(np.median(grow_us)) if grow_us else None,
                          "mean_us_inserting": float(np.mean(grow_us)) if grow_us else None,
                          "us_per_eval_warm": float(np.median(warm_us)) if warm_us else None, "keys_inserted": new_keys, "records_inserted": new_recs,
                          "cache_appends": int(st2.cache_appends), "cache_rebuilds": int(st2.cache_rebuilds),
                          "same_partials_as_preloaded_context": bool(np.array_equal(part2, pc.calc_prob_partial_flat(seq_flat[-1])[0])) if seq_flat else None,
                          "note": "gaml_cache_insert of the windows a walk set needs for the first time + gaml_calc_prob_partial, wall clock, median; "
                                  "the records go to the arena tail, the affected reads' rows are relocated and the reads scored by the appendix phase"}
        pc2.close()

    # ---- the drop-in boundary: ProbCalculator::CalcProb of integration/prob_calculator.h, driven by the reference's
    #      cache-injection harness compiled against it (oracle/_ref/gpu_harness), on the same incremental trajectory ----
    gpu_harness = os.path.join(ROOT, "oracle", "_ref", "gpu_harness")
    if rank == 0 and world == 1 and not args.no_dropin and os.path.exists(gpu_harness):
        from gaml_b200 import workload as wlmod
        n_drop = min(len(wl.evals), 1 + min(args.delta_steps, 100))
        sub = wlmod.Workload(node_len=wl.node_len, normalize_map=wl.normalize_map, sets=wl.sets, evals=wl.evals[:n_drop])
        try:
            with tempfile.TemporaryDirectory() as tmp:
                wp, rp = os.path.join(tmp, "dropin.wl"), os.path.join(tmp, "dropin.res")
                wlmod.write_workload(wp, sub)
                t0 = time.perf_counter()
                subprocess.run([gpu_harness, wp, rp, "0", "2"], check=True, cwd=tmp, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                               timeout=600)
                log(f"drop-in leg took {time.perf_counter() - t0:.1f}s")
                res = wlmod.read_results(rp)
            # second repeat: a fresh ProbCalculator over host caches that are complete — its first call mirrors the cache
            # (excluded), the following ones are warm incremental CalcProb calls
            warm = np.array([r.seconds for r in res[n_drop + 1:]]) * 1e6
            ok = all(abs(a.score - b.score) <= 1e-9 * abs(b.score) for a, b in zip(res[:n_drop], res[n_drop:]))
            line["dropin"] = {"dropin_us_per_calcprob": float(np.median(warm)), "mean_us": float(warm.mean()), "calls": int(len(warm)),
                              "p10_us": float(np.percentile(warm, 10)), "p90_us": float(np.percentile(warm, 90)),
                              "c_abi_e2e_us_per_eval": 1e3 * line["incremental"]["e2e_ms_per_eval"],
                              "c_abi_us_per_eval_inserting_keys": (line.get("append") or {}).get("us_per_eval_inserting"),
                              "repeat_scores_agree": bool(ok),
                              "what_is_compared": "the harness's ProbCalculator starts with an empty device cache, so most of its calls also "
                                                  "upload the windows of the move's new walks (a cache append) - the C-ABI figure for that is "
                                                  "c_abi_us_per_eval_inserting_keys; calls whose walks need no new window are the p10 and compare "
                                                  "with c_abi_e2e_us_per_eval",
                              "note": "ProbCalculator::CalcProb(paths, zeros, total_len) of integration/prob_calculator.h (vector<vector<int>> in, "
                                      "score out), timed inside oracle/_ref/gpu_harness around each call on the incremental trajectory; median"}
        except Exception as exc:   # the boundary leg never takes the bench line down
            line["dropin"] = {"error": str(exc)[:200]}

    # ---- the other single-GPU configurations of BASELINE.json (C1: single-end reads, C3: paired + PacBio), full evaluations
    #      through the C ABI with host walk arrays (the parity tests score the same workloads against the oracle) ----
    if rank == 0 and world == 1 and not args.no_other_configs and kind == "c2":
        from gaml_b200 import synth
        others = {}
        specs = (("c1", "C1: 100 kbp genome, 50 k single-end 100 bp reads", lambda: synth.single_workload(10, 10000, 50_000, n_evals=4, seed=7)),
                 ("c3", "C3: config 2's 2 M read pairs (weight 1.0) + 46 k PacBio-like 10 kbp reads (weight 0.5)",
                  lambda: synth.mixed_workload(460, 10000, int(2_000_000 * args.scale), int(46_000 * args.scale), n_evals=4, seed=42, pacbio_len=10000)))
        for name, desc, make in specs:
            try:
                t0 = time.perf_counter()
                wlo = make()
                pco = api.ProbCalculator.from_workload(wlo, device=local_rank)
                fws = [api.FlatWalks(w) for w in wlo.evals]
                pco.set_profiling(1)
                for fw in fws:                      # warm-up: every list once (graphs, buffers)
                    pco.reset_state()
                    pco.calc_prob_partial_flat(fw)
                n_o, wall_o, dev_o, rec_o = max(args.steps, 4), 0.0, 0.0, 0
                for k in range(n_o):
                    pco.reset_state()
                    flush_l2()
                    t1 = time.perf_counter()
                    pco.calc_prob_partial_flat(fws[k % len(fws)])
                    wall_o += time.perf_counter() - t1
                    sto = pco.stats()
                    dev_o += sto.last_device_ms
                    rec_o += int(sto.last_records_gathered)
                others[name] = {"workload": desc, "alignments_per_eval": rec_o // n_o, "e2e_ms_per_eval": 1e3 * wall_o / n_o,
                                "device_ms_per_eval": dev_o / n_o, "e2e_alignments_per_s": rec_o / wall_o,
                                "read_sets": [int(sp.kind) for sp in wlo.sets], "setup_s": round(time.perf_counter() - t0 - wall_o, 1)}
                pco.close()
            except Exception as exc:
                others[name] = {"error": str(exc)[:200]}
        others["note"] = ("full evaluations (fresh ScoringState) cycling through the workload's walk lists, gaml_calc_prob_partial with host "
                          "walk arrays, wall clock, L2 flushed between evaluations; read_sets: 0 single, 1 paired, 2 PacBio")
        line["other_configs"] = others

    if rank == 0 and not args.no_cpu_baseline and world == 1:
        # bounded CPU sample on the box's host: the reference's own scorer, 1 core, the whole workload, a few full evaluations
        with tempfile.TemporaryDirectory() as tmp:
            t0 = time.perf_counter()
            per_step, aligns, kind_cpu = run_cpu(wl, 1, 5, tmp)
            log(f"cpu baseline ({kind_cpu}) took {time.perf_counter() - t0:.1f}s")
        line["cpu_baseline"] = {"value": aligns * len(per_step) / float(per_step.sum()), "unit": "alignments/s", "cores": 1,
                                "kind": kind_cpu, "sample": f"whole {kind} workload, 5 full evaluations on one core (the reference is single-threaded)"}
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    pc.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
