"""Per-chromosome Fit-Hi-C on BASELINE config 3's genome (23 hg19 chromosomes @5kb, all pairs within 10 Mb), generated on the
device as bench.py does, in three forms:

  (a) distributed.ChromosomePass: every chromosome's fit in one launch, every chromosome's q-values in one step;
  (b) the loop the authors' workflow implies: one single-chromosome GenomePass per chromosome, each run to completion;
  (c) the genome-wide GenomePass (one fit, one ranking over the genome), for reference.

Prints one JSON line: the card and its power limit, ms per step, per-stage device times and launches per step of each form,
and whether (a) equals (b) bit for bit (p, q and the fit of every chromosome).

    python tools/bench_per_chromosome.py [--steps 5] [--warmup 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

STAGES = ["hist", "fit", "pvalues", "bh"]


def _card():
    import torch
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        limit = "unknown (%r)" % e
    return {"name": torch.cuda.get_device_name(0), "power_limit": limit}


def _stages(marks):
    out, prev = {}, "start"
    for n in STAGES:
        if n in marks:
            out[n] = marks[prev].elapsed_time(marks[n])
            prev = n
    return out


def _add(acc, d, scale=1.0):
    for k, v in d.items():
        acc[k] = acc.get(k, 0.0) + v * scale


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    import bench
    from blueberry_b200.distributed import ChromosomePass, GenomePass
    from blueberry_b200.engine import PassEngine
    if not torch.cuda.is_available():
        raise SystemExit("bench_per_chromosome.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": _card(), "workload": bench.WORKLOADS["cfg3"]["name"], "steps": args.steps}
    W = bench.Workload(bench.WORKLOADS["cfg3"], 1, 0, dev)
    R, K = W.R, W.max_dist

    def engines():
        es = []
        for c in W.chroms:
            e = PassEngine(R, bench.N_BINS, 0, K, W.bins[c], dev)
            e.set_fragments([W.bins[c]], [(W.bins[c] - 1) * R])
            e.set_bias(W.eng.bias)
            es.append(e)
        return es

    def timed(step, launches):
        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        n0 = launches()
        step()
        per_step = launches() - n0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / args.steps, per_step

    # (a) one ChromosomePass
    cp = ChromosomePass(engines(), W.shards, q_values=True)
    ms, n = timed(lambda: cp.run(), lambda: cp.launches)
    acc = {}
    for _ in range(args.steps):
        marks = {}
        cp.enqueue(cp.n_tests, marks=marks)
        cp.finish()
        _add(acc, _stages(marks), 1.0 / args.steps)
    out["a_batched"] = {"ms_per_step": ms, "launches_per_step": n, "stages_ms": acc}

    # (b) the loop of single-chromosome passes, each to completion (a host synchronisation per chromosome)
    singles = []
    for e, sh in zip(engines(), W.shards):
        gp = GenomePass(e, group=False, q_values=True)
        gp.attach([sh])
        singles.append(gp)

    def loop():
        for gp in singles:
            gp.run()
    ms, n = timed(loop, lambda: sum(gp.eng.launches for gp in singles))
    acc, fit_ms = {}, [0.0] * len(singles)
    for _ in range(args.steps):
        for i, gp in enumerate(singles):
            marks = {}
            gp.enqueue(marks=marks)
            gp.finish()
            st = _stages(marks)
            _add(acc, st, 1.0 / args.steps)
            fit_ms[i] += st["fit"] / args.steps
    out["b_loop"] = {"ms_per_step": ms, "launches_per_step": n, "stages_ms": acc,
                     "slowest_single_fit_ms": max(fit_ms), "slowest_single_fit_chrom": fit_ms.index(max(fit_ms))}

    # (a) against (b), bit for bit
    cp.run()
    for gp in singles:
        gp.run()
    same = True
    for i, gp in enumerate(singles):
        same &= torch.equal(cp.chrom_p(i).view(torch.int64), gp.shard_p(0).view(torch.int64))
        same &= torch.equal(cp.chrom_q(i).view(torch.int64), gp.shard_q(0).view(torch.int64))
        fa = bytes(cp.engs[i].fit_result.cpu().numpy().tobytes())
        fb = bytes(gp.eng.fit_result.cpu().numpy().tobytes())
        same &= fa[:72] == fb[:72] and fa[184:] == fb[184:]           # all but the SM cycle counters
    out["a_equals_b_bitwise"] = bool(same)
    out["rows"] = int(sum(sh.n for sh in W.shards))
    del singles, cp
    torch.cuda.empty_cache()

    # (c) the genome-wide pass
    gp = GenomePass(W.eng, group=False, q_values=True)
    gp.attach(W.shards)
    ms, n = timed(lambda: gp.run(), lambda: W.eng.launches)
    acc = {}
    for _ in range(args.steps):
        marks = {}
        gp.enqueue(marks=marks)
        gp.finish()
        _add(acc, _stages(marks), 1.0 / args.steps)
    out["c_genome_wide"] = {"ms_per_step": ms, "launches_per_step": n, "stages_ms": acc}
    out["fit_stage_a_over_c"] = out["a_batched"]["stages_ms"]["fit"] / out["c_genome_wide"]["stages_ms"]["fit"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
