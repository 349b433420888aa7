"""The genome-wide pass in row blocks from host memory (distributed.BlockedPass) on one GPU.  Records are generated on the
device as bench.py does (bbk_synth_contacts_range) and copied to pinned host columns; results land in host float64 columns.

  --leg a: BASELINE config 3 (1.17e9 records), which also fits resident: the resident GenomePass step against BlockedPass at the
           default block_rows, at a small block_rows, and with nothing resident (both sweeps from the host).  Per leg: ms per
           pass, GB in / out, launches, peak device memory, and whether p / q of every row equal the resident pass bit for bit.
  --leg b: BASELINE config 5 (23 chromosomes at 1 kb, 2 Mb cap: 6.03e9 records, past 2^32 rows) genome-wide on one GPU, which
           the resident pass refuses.  When the host cannot hold the 168 GB of records and results, the largest prefix of the
           chromosome list it can hold that still has more than 2^32 rows.  Reports ms per pass, the resident blocks, link
           rates, host unpack time, peak device memory, the host's cores and memory, and checks: a 1e6-row p sample against
           scipy's bdtrc (the oracle's scoring), q of every row below the saturation bucket against a host BH over exactly
           those rows (sorted, forward running max, N = non-NaN rows) bit for bit, every other non-NaN q = 1.0.

Prints one JSON line (with the card's name and power limit) and writes it to --out when given.

    python tools/bench_blocked_pass.py --leg a|b [--steps 5] [--warmup 2] [--out file.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _card():
    import torch
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        limit = "unknown (%r)" % e
    return {"name": torch.cuda.get_device_name(0), "power_limit": limit}


def _host():
    mem = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    avail = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_AVPHYS_PAGES")
    return {"cores": os.cpu_count(), "mem_gb": round(mem / 1e9, 1), "mem_available_gb": round(avail / 1e9, 1)}


def _synth_host(wl, chroms, dev, chunk=1 << 27):
    """Records of these chromosomes (bench.py's generator, seeds and biases) as pinned int32 host columns, one shard each."""
    import numpy as np
    import torch
    import bench
    from blueberry_b200 import _lib
    lib = _lib.load()
    R, K = wl["R"], wl["max_dist"] // wl["R"]
    bufs = [torch.empty(chunk, dtype=torch.int32, device=dev) for _ in range(3)]
    shards, bias_host = [], {}
    for c in chroms:
        nb = -(-bench.HG19[c] // R)
        n = int(lib.bbk_synth_n_pairs(nb, K))
        rng = np.random.default_rng(bench.SEED + 7919 * (c + 1))
        bias_host[c] = np.exp(rng.normal(0.0, 0.25, size=nb))
        bdev = torch.from_numpy(bias_host[c]).to(dev)
        cols = [torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(3)]
        for a in range(0, n, chunk):
            m = min(chunk, n - a)
            _lib.check(lib.bbk_synth_contacts_range(nb, K, R, wl["depth"], bench.DECAY, bench.SEED + 1000003 * c, _lib.ptr(bdev), a, m,
                                                    _lib.ptr(bufs[0]), _lib.ptr(bufs[1]), _lib.ptr(bufs[2]), _lib.stream_ptr()), "synth")
            for h, d in zip(cols, bufs):
                h[a:a + m].copy_(d[:m])
        shards.append((c, cols[0], cols[1], cols[2]))
    return shards, bias_host


def _engine(wl, chroms, bias_host, dev):
    import numpy as np
    import bench
    from blueberry_b200.engine import BiasTables, PassEngine
    R = wl["R"]
    bins = [-(-bench.HG19[c] // R) for c in chroms]
    eng = PassEngine(R, bench.N_BINS, 0, wl["max_dist"], max(bins), dev)
    eng.set_fragments(bins, [(nb - 1) * R for nb in bins])
    tabs = [np.where((bias_host[c] < 0.5) | (bias_host[c] > 2), -1.0, bias_host[c]) for c in chroms]
    eng.set_bias(BiasTables(tabs, [R // 2] * len(bins), dev))
    return eng


def _timed(fn, steps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t.append((time.perf_counter() - t0) * 1e3)
    return t


def leg_a(args, dev):
    import numpy as np
    import torch
    import bench
    from blueberry_b200.distributed import BlockedPass, GenomePass
    from blueberry_b200.engine import Shard
    wl = bench.WORKLOADS["cfg3"]
    chroms = list(wl["chroms"])
    shards, bias_host = _synth_host(wl, chroms, dev)
    n_rec = sum(int(s[1].numel()) for s in shards)
    out = {"workload": wl["name"], "records": n_rec, "legs": {}}
    # resident: the records on the device, GenomePass
    eng = _engine(wl, chroms, bias_host, dev)
    dshards = [Shard(*(t.to(dev) for t in s[1:]), chrom=s[0]) for s in shards]
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(dshards)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    l0 = eng.launches
    t = _timed(lambda: gp.run(), args.steps, args.warmup)
    out["legs"]["resident_genome_pass"] = {"ms_per_pass": t, "ms_median": float(np.median(t)),
                                           "launches_per_pass": (eng.launches - l0) // (args.steps + args.warmup),
                                           "peak_device_gb_above_records": round((torch.cuda.max_memory_allocated(dev) - base) / 1e9, 2),
                                           "records_device_gb": round(12 * n_rec / 1e9, 2)}
    p_out = [torch.empty(int(s[1].numel()), dtype=torch.float64).pin_memory() for s in shards]
    q_out = [torch.empty(int(s[1].numel()), dtype=torch.float64).pin_memory() for s in shards]
    for name, kw in (("blocked_default", {}), ("blocked_small_blocks", {"block_rows": 1 << 22}),
                     ("blocked_nothing_resident", {"resident_bytes": 0})):
        e2 = _engine(wl, chroms, bias_host, dev)
        bp = BlockedPass(e2, q_values=True, **kw)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        l0 = e2.launches
        t = _timed(lambda: bp.run(shards, p_out, q_out), args.steps, args.warmup)
        same = all(torch.equal(gp.shard_p(i).view(torch.int64), p_out[i].to(dev).view(torch.int64)) and
                   torch.equal(gp.shard_q(i).view(torch.int64), q_out[i].to(dev).view(torch.int64)) for i in range(len(shards)))
        same = same and torch.equal(eng.obs_sum, e2.obs_sum) and torch.equal(eng.totals, e2.totals) and \
            torch.equal(eng.spline_y, e2.spline_y) and torch.equal(eng.fit_result[:72], e2.fit_result[:72]) and \
            torch.equal(eng.fit_result[184:], e2.fit_result[184:])
        out["legs"][name] = {"block_rows": bp.block_rows, "blocks": len(bp.blocks), "resident_blocks": int(sum(bp.resident)),
                             "ms_per_pass": t, "ms_median": float(np.median(t)), "gb_in": round(bp.bytes_in / 1e9, 3),
                             "gb_out": round(bp.bytes_out / 1e9, 3), "host_unpack_ms": round(bp.host_unpack_s * 1e3, 1),
                             "launches_per_pass": (e2.launches - l0) // (args.steps + args.warmup),
                             "peak_device_gb": round((torch.cuda.max_memory_allocated(dev) - base) / 1e9, 2),
                             "bit_identical_to_resident": bool(same)}
        del bp, e2
    return out


def _host_bh(ps, qs, tau_key, chunk=1 << 26):
    """q of the rows below the saturation bucket against the reference's BH over exactly those rows (N = the non-NaN rows);
    every other non-NaN q 1.0.  Column by column in chunks: only the rows below the bucket are gathered."""
    import numpy as np
    tau = np.uint64(tau_key)
    n_valid, sel_p, sel_q, ok_rest = 0, [], [], True
    for p, q in zip(ps, qs):
        for a in range(0, len(p), chunk):
            pc, qc = p[a:a + chunk], q[a:a + chunk]
            valid = ~np.isnan(pc)
            n_valid += int(valid.sum())
            below = valid & (pc != 1.0) & ((pc.view(np.uint64) | np.uint64(1 << 63)) < tau)
            sel_p.append(pc[below])
            sel_q.append(qc[below])
            ok_rest = ok_rest and bool((qc[valid & ~below & (pc != 1.0)] == 1.0).all())
    ps_, qs_ = np.concatenate(sel_p), np.concatenate(sel_q)
    order = np.argsort(ps_, kind="stable")
    srt = ps_[order]
    rank = np.searchsorted(srt, srt, side="left") + 1
    qv = np.maximum.accumulate(np.minimum((srt * float(n_valid)) / rank.astype(np.float64), 1.0))
    want = np.empty_like(qv)
    want[order] = qv
    return bool(np.array_equal(want.view(np.uint64), qs_.view(np.uint64))), ok_rest, int(len(ps_))


def leg_b(args, dev):
    import numpy as np
    import torch
    import bench
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import BlockedPass
    lib = _lib.load()
    wl = bench.WORKLOADS["cfg5"]
    R, K = wl["R"], wl["max_dist"] // wl["R"]
    host = _host()
    chroms = list(wl["chroms"])
    sizes = [int(lib.bbk_synth_n_pairs(-(-bench.HG19[c] // R), K)) for c in chroms]
    print("host: %s" % host, file=sys.stderr, flush=True)
    budget = host["mem_available_gb"] * 1e9 * 0.6          # records + p + q pinned, the rest for the process and the checks
    note = "the whole configuration"
    while sum(sizes) * 28 > budget and len(chroms) > 1:
        chroms, sizes = chroms[:-1], sizes[:-1]
        note = "the largest prefix of the chromosome list the host can hold (28 B a record: records, p, q)"
    out = {"workload": wl["name"], "host": host, "chromosomes": [c + 1 for c in chroms], "records": sum(sizes),
           "above_2_32_rows": sum(sizes) >= (1 << 32), "scope": note}
    if sum(sizes) < (1 << 32):
        out["error"] = "the host cannot hold a prefix of more than 2^32 records"
        return out
    t0 = time.perf_counter()
    shards, bias_host = _synth_host(wl, chroms, dev)
    print("records on the host: %d chromosomes, %d records" % (len(chroms), sum(sizes)), file=sys.stderr, flush=True)
    p_out = [torch.empty(n, dtype=torch.float64).pin_memory() for n in sizes]
    q_out = [torch.empty(n, dtype=torch.float64).pin_memory() for n in sizes]
    out["setup_s"] = round(time.perf_counter() - t0, 1)
    eng = _engine(wl, chroms, bias_host, dev)
    bp = BlockedPass(eng, q_values=True)
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    steps, warm = args.steps, args.warmup
    t_all, unpack, fit = [], [], None
    l0 = eng.launches
    for i in range(warm + steps):
        t0 = time.perf_counter()
        fit = bp.run(shards, p_out, q_out)
        torch.cuda.synchronize()
        print("pass %d: %.0f ms" % (i, (time.perf_counter() - t0) * 1e3), file=sys.stderr, flush=True)
        if i >= warm:
            t_all.append((time.perf_counter() - t0) * 1e3)
            unpack.append(bp.host_unpack_s * 1e3)
        if time.perf_counter() - t0 > 60 and i >= warm:
            break                       # a pass of a minute: fewer steps
    ms = float(np.median(t_all))
    out.update({"block_rows": bp.block_rows, "blocks": len(bp.blocks), "resident_blocks": [int(k) for k, r in enumerate(bp.resident) if r],
                "ms_per_pass": t_all, "ms_median": ms, "gb_in": round(bp.bytes_in / 1e9, 2), "gb_out": round(bp.bytes_out / 1e9, 2),
                "link_in_gb_per_s_over_pass": round(bp.bytes_in / 1e9 / (ms / 1e3), 1),
                "link_out_gb_per_s_over_pass": round(bp.bytes_out / 1e9 / (ms / 1e3), 1),
                "host_unpack_ms": unpack, "peak_device_gb": round((torch.cuda.max_memory_allocated(dev) - base) / 1e9, 2),
                "launches_per_pass": (eng.launches - l0) // (warm + len(t_all)), "S": int(fit.S), "candidates": bp.n_candidates})
    # checks: a p sample against the oracle's scoring (scipy bdtrc), q against a host BH
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
    ok, ok_rest, n_below = _host_bh([x.numpy() for x in p_out], [x.numpy() for x in q_out], bp.tau_key)
    out.update({"q_below_saturation_rows": n_below, "q_below_saturation_bit_identical_host_bh": ok,
                "q_other_rows_all_one": ok_rest, "check_s": round(time.perf_counter() - t0, 1)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--leg", choices=["a", "b"], required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_blocked_pass needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": _card()}
    res["leg_" + args.leg] = leg_a(args, dev) if args.leg == "a" else leg_b(args, dev)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
