"""Packed contact records over the host link (distributed.PackedRecords, bbkio_pack_records -> bbk_unpack_records) on BASELINE
config 3's genome (23 hg19 chromosomes @5kb, all pairs within 10 Mb, zeros kept), generated on the device as bench.py does and
copied to host memory.  Every leg streams the genome-wide pass through HostStream(GenomePass, packed=True), two device slots:

  (e)  records from pre-filled pinned int32 columns (bench.py's e2e leg);
  (e') each step first copies pageable numpy columns into the pinned columns with bbkio_copy_bytes (what a numpy caller pays);
  (f)  PackedRecords packed once before the timed loop;
  (g)  each step packs from the same pageable numpy columns (pass k + 1 is packed on the host while pass k runs);
  (d)  / (d-f): the per-chromosome ChromosomePass stream from pinned columns / from PackedRecords packed once.

Prints one JSON line: the card and its power limit, the host's cores and CPU model, per leg ms/step, H2D bytes per step and
the peak device memory from the stream's construction on; the packed size per row; the packing rate in GB/s of int32 input;
and whether the last result of (e), (e'), (f) and (g) (and of (d) and (d-f)) is bit-identical (p, q and fit).

    python tools/bench_packed_records.py [--steps 5] [--warmup 2]
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


def _cpu():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"cores": os.cpu_count(), "affinity": len(os.sched_getaffinity(0)), "model": model}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import numpy as np
    import torch
    import bench
    from blueberry_b200 import _io
    from blueberry_b200.distributed import ChromosomePass, GenomePass, HostStream, pack_records
    from blueberry_b200.engine import PassEngine
    if not torch.cuda.is_available():
        raise SystemExit("bench_packed_records.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": _card(), "host": _cpu(), "workload": bench.WORKLOADS["cfg3"]["name"], "steps": args.steps}
    W = bench.Workload(bench.WORKLOADS["cfg3"], 1, 0, dev)
    R, K = W.R, W.max_dist
    in_rows = W.starts[-1] + W.sizes[-1]
    h_in = [torch.empty(W.rows, dtype=torch.int32).pin_memory() for _ in range(3)]
    for h, d in zip(h_in, (W.mid1, W.mid2, W.count)):
        h.copy_(d)
    pageable = [h.numpy().copy() for h in h_in]                # what a numpy caller holds
    engines = []
    for c in W.chroms:
        e = PassEngine(R, bench.N_BINS, 0, K, W.bins[c], dev)
        e.set_fragments([W.bins[c]], [(W.bins[c] - 1) * R])
        e.set_bias(W.eng.bias)
        engines.append(e)
    cp = ChromosomePass(engines, W.shards, q_values=True)       # built on the genome's sizes; the streams attach their slots
    cp.shards, cp.p, cp.q = [], None, None
    shards_np = [tuple(c[a:a + n] for c in pageable) for a, n in zip(W.starts, W.sizes)]
    W.mid1 = W.mid2 = W.count = None
    W.shards = []
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    out["rows"] = {"records": int(sum(W.sizes)), "layout": int(in_rows)}

    # packing alone: int32 input bytes over host time, all cores and one core
    rec = pack_records(shards_np)
    t0 = time.perf_counter()
    for _ in range(3):
        pack_records(shards_np, out=rec)
    pack_s = (time.perf_counter() - t0) / 3
    t0 = time.perf_counter()
    pack_records(shards_np, out=rec, threads=1)
    pack1_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    for _ in range(3):
        for dst, src in zip(h_in, pageable):
            _io.copy_bytes(dst.data_ptr(), src.ctypes.data, 4 * in_rows)
    copy_s = (time.perf_counter() - t0) / 3
    out["packed"] = {"bytes": rec.nbytes, "bytes_per_record": rec.nbytes / sum(W.sizes), "bytes_per_layout_row": rec.nbytes / in_rows,
                     "bound_bytes": _io.pack_records_bound(in_rows)}
    out["host_rates"] = {"pack_s": pack_s, "pack_gbps_int32_in": 12 * sum(W.sizes) / pack_s / 1e9,
                         "pack_s_one_thread": pack1_s, "pack_gbps_one_thread": 12 * sum(W.sizes) / pack1_s / 1e9,
                         "copy_bytes_s": copy_s, "copy_bytes_gbps": 12 * in_rows / copy_s / 1e9}

    recs = [rec, pack_records(shards_np)]          # (g) alternates two PackedRecords; (f) sends recs[0] every step
    p_out = np.empty(max(in_rows, 4), dtype=np.float64)
    q_out = np.empty(max(in_rows, 4), dtype=np.float64)
    ref = {}

    def stream_leg(pas, feed, h2d_bytes, key):
        torch.cuda.reset_peak_memory_stats(dev)
        hs = HostStream(pas, W.sizes, W.chroms, slots=2, packed=True)
        outs = [hs.packed_buffers() for _ in range(2)]

        def step():
            feed(hs, outs[hs.submitted % 2])

        for _ in range(args.warmup):
            step()
        hs.drain()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):          # the last value lists leave the device in drain(): inside the timed region
            step()
        hs.drain()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        peak = torch.cuda.max_memory_allocated(dev)
        last = outs[(hs.submitted - 1) % 2]
        fits = hs.fit_of(hs.submitted - 1)
        fits = fits if isinstance(fits, list) else [fits]
        fit_bytes = [bytes(f)[:72] + bytes(f)[184:] for f in fits]           # all but the SM cycle counters
        p, q = last.dense(p_out, q_out)
        res = {"ms_per_step": ms, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": last.nbytes() + hs.slots[0].h_fit.numel(),
               "peak_alloc_gib_from_stream_construction": peak / 2 ** 30}
        if key not in ref:
            ref[key] = (p.copy(), q.copy(), fit_bytes)
        else:
            rp, rq, rf = ref[key]
            res["bit_identical_to_first_leg"] = bool(np.array_equal(p.view(np.uint64), rp.view(np.uint64)) and
                                                     np.array_equal(q.view(np.uint64), rq.view(np.uint64)) and fit_bytes == rf)
        del hs, outs, last
        pas.shards, pas.p, pas.q = [], None, None               # the pass lets go of the stream's slots
        torch.cuda.empty_cache()
        return res

    def from_pinned(hs, o):
        hs.submit_packed(h_in[0], h_in[1], h_in[2], o)

    staging = [h_in, [torch.empty(W.rows, dtype=torch.int32).pin_memory() for _ in range(3)]]

    def from_numpy_copied(hs, o):
        j = hs.submitted % 2
        hs.slots[j].in_ready.synchronize()          # the slot's previous records (from staging[j]) have crossed the link
        for dst, src in zip(staging[j], pageable):
            _io.copy_bytes(dst.data_ptr(), src.ctypes.data, 4 * in_rows)
        hs.submit_packed(staging[j][0], staging[j][1], staging[j][2], o)

    def from_packed_once(hs, o):
        hs.submit_packed(recs[0], out=o)

    def from_numpy_packed(hs, o):
        j = hs.submitted % 2
        hs.slots[j].in_ready.synchronize()          # recs[j] has crossed the link: refill it for this pass
        pack_records(shards_np, out=recs[j])
        hs.submit_packed(recs[j], out=o)

    gp = GenomePass(W.eng, group=False, q_values=True)
    out["e_pinned_columns"] = stream_leg(gp, from_pinned, 12 * in_rows, "genome")
    out["e1_numpy_copied_to_pinned"] = stream_leg(gp, from_numpy_copied, 12 * in_rows, "genome")
    out["f_packed_once"] = stream_leg(gp, from_packed_once, recs[0].nbytes, "genome")
    out["g_packed_each_step"] = stream_leg(gp, from_numpy_packed, recs[0].nbytes, "genome")
    del gp
    torch.cuda.empty_cache()

    out["d_chromosome_pinned_columns"] = stream_leg(cp, from_pinned, 12 * in_rows, "chromosome")
    out["d_f_chromosome_packed_once"] = stream_leg(cp, from_packed_once, recs[0].nbytes, "chromosome")
    e, f = out["e_pinned_columns"]["ms_per_step"], out["f_packed_once"]["ms_per_step"]
    out["summary"] = {"f_over_e": f / e, "g_over_e1": out["g_packed_each_step"]["ms_per_step"] / out["e1_numpy_copied_to_pinned"]["ms_per_step"],
                      "d_f_over_d": out["d_f_chromosome_packed_once"]["ms_per_step"] / out["d_chromosome_pinned_columns"]["ms_per_step"],
                      "all_bit_identical": all(out[k].get("bit_identical_to_first_leg", True) for k in
                                               ("e1_numpy_copied_to_pinned", "f_packed_once", "g_packed_each_step",
                                                "d_f_chromosome_packed_once"))}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
