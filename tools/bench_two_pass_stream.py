"""The two-pass workload (BASELINE config 4: chr1 @ 1 kb, all pairs within 2 Mb, zeros kept, biases; pass 1, the outliers with
p <= 1 / possibleIntraInRangeCount left out of the statistics, refit, every record scored again) end to end from host memory.
The records are generated on the device as bench.py does and copied to host memory.  Legs, each after warm-up:

  (a) the device-resident step bench.py times: gp1.enqueue(); gp.enqueue(exclude=(gp1.p, threshold));
  (b) HostStream(GenomePass, refit=True): pinned int32 columns in, dense p, q and p_first out (two sets of host outputs);
  (c) as (b), with packed results (submit_packed: p / q of the refit pass);
  (d) as (c), fed PackedRecords packed once before the timed loop;
  (e) FitHiC.fit_transform_arrays(refit=True, q_values=True) on pageable numpy columns, one call per step;
  (f) the single-pass HostStream(GenomePass, packed=True) over the same records, for comparison.

Both passes first settle on the reference's own s (GenomePass.run), and every leg runs with those values, so that all of them
compute the same thing.  Prints one JSON line: the card and its power limit, per leg ms/step, host-to-device and
device-to-host bytes per step, launches per step, the peak allocated device memory from the leg's construction on, and
whether the last pass of (b)-(d) and (e)'s outputs equal (a)'s device columns bit for bit.

    python tools/bench_two_pass_stream.py [--steps 5] [--warmup 2] [--dropin-calls 2]
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


def _card():
    import torch
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        limit = "unknown (%r)" % e
    return {"name": torch.cuda.get_device_name(0), "power_limit": limit}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--dropin-calls", type=int, default=2)
    args = ap.parse_args()
    if args.steps < 1 or args.dropin_calls < 1:
        ap.error("--steps and --dropin-calls must be at least 1")
    import numpy as np
    import torch
    import bench
    from blueberry_b200 import synth
    from blueberry_b200.distributed import GenomePass, HostStream, pack_records
    from blueberry_b200.fithic import FitHiC, _in_range_possible
    if not torch.cuda.is_available():
        raise SystemExit("bench_two_pass_stream.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": _card(), "workload": bench.WORKLOADS["cfg4"]["name"], "steps": args.steps, "warmup": args.warmup}
    W = bench.Workload(bench.WORKLOADS["cfg4"], 1, 0, dev)
    eng = W.eng
    n = W.starts[-1] + W.sizes[-1]
    thr = 1.0 / _in_range_possible(eng.possible.cpu().numpy(), W.R, eng.min_dist, eng.max_dist)
    out["rows"] = n
    out["threshold"] = {"p_outlier": thr, "equals_bench_py": thr == 1.0 / float(W.possible_in_range)}

    def bits(a):
        return np.ascontiguousarray(a).view(np.uint64)

    def same(a, b):
        return bool(np.array_equal(bits(a), bits(b)))

    # ---- (a) resident records; both passes settle first, then the timed steps run with the settled s
    torch.cuda.reset_peak_memory_stats(dev)
    gp1 = GenomePass(eng, group=False, q_values=False)
    gp1.attach(W.shards)
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(W.shards)
    gp1.run()
    gp.run(exclude=(gp1.p, thr))
    s = (gp1._smoothing, gp._smoothing)
    out["settled_smoothing"] = s

    def step_a():
        gp1.enqueue(smoothing=s[0])
        gp.enqueue(smoothing=s[1], exclude=(gp1.p, thr))

    for _ in range(args.warmup):
        step_a()
    torch.cuda.synchronize()
    eng.launches = 0
    step_a()
    launches_a = eng.launches
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_a()
    e1.record()
    torch.cuda.synchronize()
    out["a_device_resident"] = {"ms_per_step": e0.elapsed_time(e1) / args.steps, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                                "launches_per_step": launches_a,
                                "peak_alloc_gib_from_construction_incl_resident_records": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
    ref = {"p_first": gp1.shard_p(0).cpu().numpy(), "p": gp.shard_p(0).cpu().numpy(), "q": gp.shard_q(0).cpu().numpy()}
    out["outliers"] = int((ref["p_first"] <= thr).sum())

    h_in = [torch.empty(W.rows, dtype=torch.int32).pin_memory() for _ in range(3)]
    for h, d in zip(h_in, (W.mid1, W.mid2, W.count)):
        h.copy_(d)
    del gp1, gp
    W.mid1 = W.mid2 = W.count = None
    W.shards = []
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    cols_np = [h.numpy()[:n] for h in h_in]
    rec = pack_records([tuple(cols_np)])
    out["packed_records"] = {"bytes": rec.nbytes, "bytes_per_record": rec.nbytes / n}
    p_out, q_out = np.empty(W.rows, dtype=np.float64), np.empty(W.rows, dtype=np.float64)

    def stream_leg(feed, h2d, refit=True, packed=False, dense_outs=None):
        torch.cuda.reset_peak_memory_stats(dev)
        hs = HostStream(GenomePass(eng, group=False, q_values=True), W.sizes, W.chroms, slots=2, packed=packed, refit=refit)
        outs = [hs.packed_buffers() for _ in range(2)] if packed else dense_outs
        for _ in range(args.warmup):
            feed(hs, outs[hs.submitted % 2])
        hs.drain()
        torch.cuda.synchronize()
        hs.gp.launches = 0
        feed(hs, outs[hs.submitted % 2])
        hs.drain()
        launches = hs.gp.launches
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):          # the last value lists leave the device in drain(): inside the timed region
            feed(hs, outs[hs.submitted % 2])
        hs.drain()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        k = hs.submitted - 1
        last = outs[k % 2]
        fit_bytes = hs.slots[0].h_fit.numel() * (2 if refit else 1)
        res = {"ms_per_step": ms, "h2d_bytes_per_step": h2d, "launches_per_step": launches,
               "peak_alloc_gib_from_stream_construction": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
        if packed:
            p, q = last.dense(p_out, q_out)
            res["d2h_bytes_per_step"] = last.nbytes() + fit_bytes
            if refit:
                res["refit_pass_equals_a"] = same(p[:n], ref["p"]) and same(q[:n], ref["q"])
        else:
            h_p1, h_p, h_q = last
            res["d2h_bytes_per_step"] = 24 * n + fit_bytes
            res["refit_pass_equals_a"] = same(h_p.numpy()[:n], ref["p"]) and same(h_q.numpy()[:n], ref["q"])
            res["p_first_equals_a"] = same(h_p1.numpy()[:n], ref["p_first"])
        if refit:
            res["fit_s"] = (hs.fit_of(k, first=True).smoothing, hs.fit_of(k).smoothing)
        del hs, outs, last
        torch.cuda.empty_cache()
        return res

    def dense_feed(hs, o):
        hs.submit(h_in[0], h_in[1], h_in[2], o[1], o[2], h_p_first=o[0], smoothing=s)

    dense_outs = [[torch.empty(W.rows, dtype=torch.float64).pin_memory() for _ in range(3)] for _ in range(2)]
    out["b_dense_pinned_columns"] = stream_leg(dense_feed, 12 * n, dense_outs=dense_outs)
    del dense_outs
    out["c_packed_results"] = stream_leg(lambda hs, o: hs.submit_packed(h_in[0], h_in[1], h_in[2], o, smoothing=s), 12 * n, packed=True)
    out["d_packed_results_packed_records"] = stream_leg(lambda hs, o: hs.submit_packed(rec, out=o, smoothing=s), rec.nbytes, packed=True)
    out["f_single_pass_packed"] = stream_leg(lambda hs, o: hs.submit_packed(h_in[0], h_in[1], h_in[2], o), 12 * n, refit=False,
                                             packed=True)

    # ---- (e) the drop-in call on pageable numpy columns (chr1 / chr2 None: one chromosome)
    cols_np = [c.copy() for c in cols_np]
    del h_in
    rec = None
    nb = W.bins[0]
    fc, fm = synth.make_fragments([nb], W.R)
    model = FitHiC("cfg4", W.R, n_bins=bench.N_BINS, max_dist=W.max_dist, min_dist=0)
    bias = (np.zeros(nb, dtype=np.int32), fm, W.bias_host[0])
    torch.cuda.reset_peak_memory_stats(dev)
    times = []
    for _ in range(args.dropin_calls):
        t0 = time.perf_counter()
        o = model.fit_transform_arrays(None, cols_np[0], None, cols_np[1], cols_np[2], fc, fm, bias=bias, refit=True, q_values=True)
        times.append((time.perf_counter() - t0) * 1e3)
    out["e_fit_transform_arrays_refit"] = {
        "ms_per_call": times, "h2d_bytes_per_step": 12 * n,
        "d2h_bytes_per_step_note": "p_first dense (8 B/row) + p / q packed as in (c) + the fit tables",
        "d2h_bytes_per_step": 8 * n + out["c_packed_results"]["d2h_bytes_per_step"],
        "launches_per_step": int(o.gpu_launches), "peak_alloc_gib_from_first_call": torch.cuda.max_memory_allocated(dev) / 2 ** 30,
        "equals_a": same(o.p_first, ref["p_first"]) and same(o.p, ref["p"]) and same(o.q, ref["q"]),
        "fit_s": o.fit.smoothing}
    a = out["a_device_resident"]["ms_per_step"]
    out["summary"] = {
        "ms_per_step": {k: out[k]["ms_per_step"] for k in ("a_device_resident", "b_dense_pinned_columns", "c_packed_results",
                                                          "d_packed_results_packed_records", "f_single_pass_packed")},
        "e_ms_per_call_min": min(times), "d_over_b": out["d_packed_results_packed_records"]["ms_per_step"] / out["b_dense_pinned_columns"]["ms_per_step"],
        "b_over_a": out["b_dense_pinned_columns"]["ms_per_step"] / a,
        "all_equal_a": all(out[k].get("refit_pass_equals_a", True) and out[k].get("p_first_equals_a", True) for k in
                           ("b_dense_pinned_columns", "c_packed_results", "d_packed_results_packed_records")) and
                       out["e_fit_transform_arrays_refit"]["equals_a"]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
