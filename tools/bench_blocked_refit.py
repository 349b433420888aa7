"""The two-pass workload (BASELINE config 4's method: pass 1, the rows with p <= 1 / possibleIntraInRangeCount left out of the
statistics, refit, every record scored again) in row blocks from host memory on one GPU: distributed.BlockedPass(refit=True).
Records are generated on the device as bench.py does and copied to pinned host columns; results land in host float64 columns.

  --leg a: BASELINE config 4 (chr1 @ 1 kb, 2 Mb cap: 496.75e6 records), which also fits resident:
           (a) the resident two-pass device step, records already on the device (both passes settled on their s first);
           (b) BlockedPass(refit=True) at the default block_rows, every block resident, p_first_out given;
           (c) as (b), with nothing resident (all three sweeps from the host).
           Checks: (b) and (c) equal (a) bit for bit - p_first, p, q, the tables after pass 2, the spline and both fits.
  --leg d: a genome-wide 1 kb two-pass that the resident two-pass refuses: the largest prefix of config 5's chromosome list the
           host can hold, past 2^32 rows if possible (p_first_out omitted when only that gets there), otherwise past the
           resident two-pass' memory estimate.  Checks: a 1e6-row p sample against scipy's bdtrc (the oracle's scoring) with
           pass 2's S and spline; q of every row below the saturation bucket against a host BH over exactly those rows, bit
           for bit, every other non-NaN q = 1.0.

Per leg: ms per pass (median), GB in / out, host unpack time, launches, peak device memory, the pass-1 outliers.  Prints one
JSON line (with the card's name and power limit) and writes it to --out when given.

    python tools/bench_blocked_refit.py --leg a|d [--steps 5] [--warmup 2] [--out file.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import bench_blocked_pass as bbp          # noqa: E402  (the card, the host, the records and the engine of config 5; host BH)


def _fit_cmp(raw):
    raw = bytes(raw)
    return raw[:72] + raw[184:]


def _blocked_timed(bp, eng, shards, p_out, q_out, p1_out, steps, warmup):
    """Run bp `warmup + steps` times; per-pass ms, unpack ms, launches per pass, peak device GB over the run."""
    import numpy as np
    import torch
    dev = bp.device
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    l0 = eng.launches
    t_all, unpack, fit = [], [], None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        fit = bp.run(shards, p_out, q_out, p_first_out=p1_out)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        print("pass %d: %.0f ms" % (i, ms), file=sys.stderr, flush=True)
        if i >= warmup:
            t_all.append(ms)
            unpack.append(bp.host_unpack_s * 1e3)
    return fit, {"block_rows": bp.block_rows, "blocks": len(bp.blocks), "resident_blocks": int(sum(bp.resident)),
                 "ms_per_pass": t_all, "ms_median": float(np.median(t_all)), "gb_in": round(bp.bytes_in / 1e9, 3),
                 "gb_out": round(bp.bytes_out / 1e9, 3), "host_unpack_ms": unpack,
                 "launches_per_pass": (eng.launches - l0) // (warmup + steps),
                 "peak_device_gb": round((torch.cuda.max_memory_allocated(dev) - base) / 1e9, 2)}


def leg_a(args, dev):
    import numpy as np
    import torch
    import bench
    from blueberry_b200.distributed import BlockedPass, GenomePass
    from blueberry_b200.fithic import _in_range_possible
    W = bench.Workload(bench.WORKLOADS["cfg4"], 1, 0, dev)
    eng = W.eng
    n = W.starts[-1] + W.sizes[-1]
    thr = 1.0 / _in_range_possible(eng.possible.cpu().numpy(), W.R, eng.min_dist, eng.max_dist)
    out = {"workload": bench.WORKLOADS["cfg4"]["name"], "records": n, "p_outlier": thr, "legs": {}}

    # ---- (a) resident: both passes settle first, then the timed steps run with the settled s
    gp1 = GenomePass(eng, group=False, q_values=False)
    gp1.attach(W.shards)
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(W.shards)
    fit1 = gp1.run()
    fit2 = gp.run(exclude=(gp1.p, thr))
    s = (gp1._smoothing, gp._smoothing)

    def step_a():
        gp1.enqueue(smoothing=s[0])
        gp.enqueue(smoothing=s[1], exclude=(gp1.p, thr))

    for _ in range(args.warmup):
        step_a()
    torch.cuda.synchronize()
    eng.launches = 0
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    t = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step_a()
        e1.record()
        e1.synchronize()
        t.append(e0.elapsed_time(e1))
    ref = {"p_first": [gp1.shard_p(i).cpu().numpy() for i in range(len(W.shards))],
           "p": [gp.shard_p(i).cpu().numpy() for i in range(len(W.shards))],
           "q": [gp.shard_q(i).cpu().numpy() for i in range(len(W.shards))],
           "obs": eng.obs_sum.cpu().numpy(), "totals": eng.totals.cpu().numpy(), "sy": eng.spline_y.cpu().numpy(),
           "fit1": _fit_cmp(bytes(fit1)), "fit2": _fit_cmp(bytes(fit2))}
    outliers = int(sum((p <= thr).sum() for p in ref["p_first"]))
    out["legs"]["a_resident_two_pass"] = {"ms_per_pass": t, "ms_median": float(np.median(t)), "gb_in": 0.0, "gb_out": 0.0,
                                          "host_unpack_ms": None, "launches_per_pass": eng.launches // args.steps,
                                          "peak_device_gb_above_records_and_passes": round((torch.cuda.max_memory_allocated(dev) - base) / 1e9, 2),
                                          "device_gb_records_and_passes": round(base / 1e9, 2), "outliers": outliers,
                                          "fit_s": [fit1.smoothing, fit2.smoothing]}

    # ---- records to pinned host columns; the device copies and the resident passes go
    shards = []
    for a, m, c in zip(W.starts, W.sizes, W.chroms):
        shards.append((c,) + tuple(x[a:a + m].cpu().pin_memory() for x in (W.mid1, W.mid2, W.count)))
    del gp1, gp
    W.mid1 = W.mid2 = W.count = None
    W.shards = []
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    p_out = [torch.empty(int(sh[1].numel()), dtype=torch.float64).pin_memory() for sh in shards]
    q_out = [torch.empty(int(sh[1].numel()), dtype=torch.float64).pin_memory() for sh in shards]
    p1_out = [torch.empty(int(sh[1].numel()), dtype=torch.float64).pin_memory() for sh in shards]

    def bits_equal(a, b):
        return bool(np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64)))

    for name, kw in (("b_blocked_all_resident", {}), ("c_blocked_nothing_resident", {"resident_bytes": 0})):
        bp = BlockedPass(eng, q_values=True, refit=True, **kw)
        fit, res = _blocked_timed(bp, eng, shards, p_out, q_out, p1_out, args.steps, args.warmup)
        res["outliers"] = int(sum((p.numpy() <= thr).sum() for p in p1_out))
        res["bit_identical_to_a"] = {
            "p_first": all(bits_equal(x.numpy(), y) for x, y in zip(p1_out, ref["p_first"])),
            "p": all(bits_equal(x.numpy(), y) for x, y in zip(p_out, ref["p"])),
            "q": all(bits_equal(x.numpy(), y) for x, y in zip(q_out, ref["q"])),
            "tables": bool(np.array_equal(eng.obs_sum.cpu().numpy(), ref["obs"]) and np.array_equal(eng.totals.cpu().numpy(), ref["totals"])),
            "spline_y": bits_equal(eng.spline_y.cpu().numpy(), ref["sy"]),
            "fit_first": _fit_cmp(bytes(bp.fit_first)) == ref["fit1"],
            "fit": _fit_cmp(bytes(fit)) == ref["fit2"]}
        res["all_bit_identical"] = all(res["bit_identical_to_a"].values())
        out["legs"][name] = res
        print(json.dumps({name: res}), file=sys.stderr, flush=True)
        del bp
        torch.cuda.empty_cache()
    return out


def leg_d(args, dev):
    import numpy as np
    import torch
    import bench
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import BlockedPass, resident_pass_bytes
    lib = _lib.load()
    wl = bench.WORKLOADS["cfg5"]
    R, K = wl["R"], wl["max_dist"] // wl["R"]
    host = bbp._host()
    free, total = torch.cuda.mem_get_info(dev)
    chroms_all = list(wl["chroms"])
    sizes_all = [int(lib.bbk_synth_n_pairs(-(-bench.HG19[c] // R), K)) for c in chroms_all]
    budget = host["mem_available_gb"] * 1e9 * 0.6          # records + results pinned, the rest for the process and the checks

    def prefix(per_record):
        k = len(chroms_all)
        while k > 1 and sum(sizes_all[:k]) * per_record > budget:
            k -= 1
        return k

    estimate_rows = next((r for r in range(1, 1 << 36, 1 << 26) if resident_pass_bytes(r, True, refit=True) + (1 << 30) > free), None)
    k36, k28 = prefix(36), prefix(28)
    if sum(sizes_all[:k36]) >= (1 << 32):
        k, with_first, scope = k36, True, "past 2^32 rows, p_first_out given (36 B a record: records, p, q, p_first)"
    elif sum(sizes_all[:k28]) >= (1 << 32):
        k, with_first, scope = k28, False, "past 2^32 rows; p_first_out omitted so that the host holds it (28 B a record: records, p, q)"
    else:
        k, with_first, scope = k36, True, "below 2^32 rows; past the resident two-pass' memory estimate (36 B a record)"
    chroms, sizes = chroms_all[:k], sizes_all[:k]
    if k < len(chroms_all):
        scope = "the largest prefix of the chromosome list the host can hold, " + scope
    out = {"workload": wl["name"] + ", two passes", "host": host, "chromosomes": [c + 1 for c in chroms], "records": sum(sizes),
           "above_2_32_rows": sum(sizes) >= (1 << 32), "p_first_out": with_first, "scope": scope,
           "device_free_gb": round(free / 1e9, 1),
           "resident_two_pass_estimate_gb": round(resident_pass_bytes(sum(sizes), True, refit=True) / 1e9, 1),
           "resident_two_pass_refused": sum(sizes) >= (1 << 32) or resident_pass_bytes(sum(sizes), True, refit=True) + (1 << 30) > free}
    if estimate_rows:
        out["resident_two_pass_largest_rows_estimate"] = estimate_rows
    if not out["resident_two_pass_refused"]:
        out["error"] = "the host cannot hold a prefix that the resident two-pass refuses"
        return out
    print(json.dumps(out), file=sys.stderr, flush=True)
    t0 = time.perf_counter()
    shards, bias_host = bbp._synth_host(wl, chroms, dev)
    p_out = [torch.empty(n, dtype=torch.float64).pin_memory() for n in sizes]
    q_out = [torch.empty(n, dtype=torch.float64).pin_memory() for n in sizes]
    p1_out = [torch.empty(n, dtype=torch.float64).pin_memory() for n in sizes] if with_first else None
    out["setup_s"] = round(time.perf_counter() - t0, 1)
    eng = bbp._engine(wl, chroms, bias_host, dev)
    # table 1 from one single pass (untimed): the rows table 2 leaves out are the pass-1 outliers
    BlockedPass(eng, q_values=False).run(shards, p_out)
    intra_first = int(eng.totals[3].item())                 # observedIntraAllCount
    bp = BlockedPass(eng, q_values=True, refit=True)
    steps = args.steps
    if args.max_passes:
        steps = max(1, min(steps, args.max_passes - args.warmup))
    fit, res = _blocked_timed(bp, eng, shards, p_out, q_out, p1_out, steps, args.warmup)
    out.update(res)
    ms = res["ms_median"]
    out.update({"link_in_gb_per_s_over_pass": round(bp.bytes_in / 1e9 / (ms / 1e3), 1),
                "link_out_gb_per_s_over_pass": round(bp.bytes_out / 1e9 / (ms / 1e3), 1),
                "S_first": int(bp.fit_first.S), "S": int(fit.S), "candidates": bp.n_candidates, "p_outlier": bp.p_outlier})
    out["outliers"] = intra_first - int(eng.totals[3].item())
    out["outliers_note"] = "observedIntraAllCount of table 1 (one single pass) minus that of table 2"
    if with_first:
        out["outliers_from_p_first"] = int(sum((p.numpy() <= bp.p_outlier).sum() for p in p1_out))
    # checks: a p sample against the oracle's scoring (scipy bdtrc) with pass 2's S and spline, q against a host BH
    from oracle import fithic_oracle as fo
    i_sh = int(np.argmax(sizes))
    c = chroms[i_sh]
    n = sizes[i_sh]
    sel = np.arange(0, n, max(1, n // 1_000_000))
    m1, m2, cn = (shards[i_sh][j].numpy()[sel] for j in (1, 2, 3))
    pg = p_out[i_sh].numpy()[sel]
    sy = eng.spline_y[:fit.L].cpu().numpy()
    tab = np.where((bias_host[c] < 0.5) | (bias_host[c] > 2), -1.0, bias_host[c])
    b1, b2 = tab[(m1 - R // 2) // R], tab[(m2 - R // 2) // R]
    pr, scored, keep = fo.score_pairs(m1, m2, cn, int(fit.S), fit.k0, sy, R, 0, wl["max_dist"], b1, b2)
    kk = keep & (pr > 1e-290) & (pg <= 1)
    out["p_sample_rows"] = int(len(sel))
    out["p_sample_keep_equal"] = bool(np.array_equal(pg <= 1, keep))
    out["p_sample_max_dlog10p_vs_scipy"] = float(np.abs(np.log10(pg[kk]) - np.log10(pr[kk])).max()) if kk.any() else 0.0
    print(json.dumps(out), file=sys.stderr, flush=True)
    t0 = time.perf_counter()
    ok, ok_rest, n_below = bbp._host_bh([x.numpy() for x in p_out], [x.numpy() for x in q_out], bp.tau_key)
    out.update({"q_below_saturation_rows": n_below, "q_below_saturation_bit_identical_host_bh": ok,
                "q_other_rows_all_one": ok_rest, "check_s": round(time.perf_counter() - t0, 1)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--leg", choices=["a", "d"], required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--max-passes", type=int, default=0, help="--leg d: at most this many passes, warm-up included (0: no cap)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_blocked_refit needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"tool": "tools/bench_blocked_refit.py", "card": bbp._card(), "steps": args.steps, "warmup": args.warmup}
    res["leg_" + args.leg] = leg_a(args, dev) if args.leg == "a" else leg_d(args, dev)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
