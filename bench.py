#!/usr/bin/env python
"""bench.py - Fit-Hi-C contact pairs/sec on B200 (BASELINE.json's metric), one JSON line on stdout.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU arm (oracle port on the host cores)

Default workload (config.workload): BASELINE config 3 - the 23 hg19 chromosomes at 5 kb (607,271 bins), every pair within
10 Mb (1,169,126,271 records, zeros kept), ICE-style biases, synthetic counts generated on the device - the configuration
the metric is quoted on ("at 1/2/4/8 B200").  The SAME genome is scored at every N (strong scaling): the records are
cut into N equal pieces along the chromosomes (distributed.plan_shards: whole chromosomes, a chromosome that straddles
a cut is split into row blocks), through the public multi-GPU entry point distributed.GenomePass: K1 per shard ->
all-reduce of the distance table (NCCL) -> fit -> K4 (one streaming kernel per shard + the patch pass over the deferred
rows) -> genome-wide Benjamini-Hochberg q-values (histogram all-reduce + one fixed-capacity all-gather).
With --gpus 8 the line also carries BASELINE config 5 (genome-wide 1 kb, 2 Mb cap, 6,029,643,315 records) as
cfg5_ms_per_step / cfg5_frac.  Other workloads: --workload cfg2 (chr1 @ 5 kb), cfg4 (chr1 @ 1 kb, two passes), cfg5.
A "step" is one whole pass over the resident records; ms_per_step / value are one pass on its own.  two_passes_in_flight
(one GPU by default, --overlap on elsewhere) is the throughput when independent passes alternate on two streams.
--dump-outputs DIR writes what the last timed step computed (rank 0's rows) as float64 .npy files, so that two builds can be
compared output for output: the inputs are generated from fixed seeds and are the same in every run with the same arguments.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_BINS = 100
DECAY = 1.08
SEED = 20161108
BYTES_PER_PAIR = 48          # 12 (K1 read) + 20 (K4 read+write) + 16 (K5 read+write), BASELINE.md section 2
K4_BYTES_PER_PAIR = 20
DUMP_ROWS = 1 << 20          # --dump-outputs: records of the seeded sample (at most 32 MiB: row, keep, p, q)

HG19 = [249250621, 243199373, 198022430, 191154276, 180915260, 171115067, 159138663, 146364022, 141213431, 135534747,
        135006516, 133851895, 115169878, 107349540, 102531392, 90354753, 81195210, 78077248, 59128983, 63025520, 48129895,
        51304566, 155270560]

# depth = Poisson mean of a d = 0 pair with unit bias, chosen so that S stays below 2^31 (the reference's bdtrc takes a C int)
WORKLOADS = {
    "cfg2": dict(R=5000, max_dist=10_000_000, depth=600.0, chroms=[0], two_pass=False,
                 name="cfg2: chr1@5kb, all pairs within 10 Mb"),
    "cfg3": dict(R=5000, max_dist=10_000_000, depth=450.0, chroms=list(range(23)), two_pass=False,
                 name="cfg3: 23 hg19 chromosomes @5kb, all intra-chromosomal pairs within 10 Mb, sharded by chromosome"),
    "cfg4": dict(R=1000, max_dist=2_000_000, depth=60.0, chroms=[0], two_pass=True,
                 name="cfg4: chr1@1kb, all pairs within 2 Mb, two passes (refit after outlier removal)"),
    "cfg5": dict(R=1000, max_dist=2_000_000, depth=25.0, chroms=list(range(23)), two_pass=False,
                 name="cfg5: 23 hg19 chromosomes @1kb, all intra-chromosomal pairs within 2 Mb, band-sharded"),
}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _true_reference():
    """The unmodified reference timed end to end (gz text in / out, one core) in the build container by
    tools/time_true_reference.py - /root/reference does not exist on the GPU box, so this is a committed measurement."""
    path = os.path.join(ROOT, "profiles", "true_reference_timing.json")
    try:
        with open(path) as fh:
            return json.load(fh)
    except Exception:
        return None


def _k4_sources_sha():
    h = hashlib.sha256()
    for f in ("pvalue.cu", "pvalue_tiles.inl"):
        with open(os.path.join(ROOT, "blueberry_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def _k4_traffic(workload, n_gpus):
    """dram__bytes_read.sum + dram__bytes_write.sum of the K4 kernels from the committed ncu --set full capture of THIS
    workload and THESE kernel sources (profiles/k4_traffic.json); None when there is no capture or the sources changed."""
    path = os.path.join(ROOT, "profiles", "k4_traffic.json")
    if not os.path.exists(path):
        return None
    try:
        with open(path) as fh:
            for rec in json.load(fh):
                if rec.get("workload") == workload and rec.get("n_gpus") == n_gpus and rec.get("sources_sha16") == _k4_sources_sha():
                    return rec.get("dram_bytes")
    except Exception:
        return None
    return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons; started before the warm-up (nvidia-smi takes ~100 ms to come up),
    reduced over the samples whose timestamp falls inside the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.t0 = self.t1 = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in self.tmp.read().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), [nm for nm, v in zip(names, f[3:7]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        os.unlink(self.tmp.name)
        inside = [r for r in rows if self.t0 is not None and self.t0 - 0.005 <= r[0] <= self.t1 + 0.005]
        use = inside if inside else rows[-20:]
        if use:
            out["sm_mhz"] = statistics.median(r[1] for r in use)
            out["sm_max_mhz"] = max(r[2] for r in use)
            out["reasons"] = sorted(set(x for r in use for x in r[3]))
            out["samples"] = len(use)
            out["window"] = "timed region" if inside else "last samples under load (timed region shorter than the sampling period)"
        return out


# =================================================================================================
# CPU arm: the oracle port of the reference path on the host cores
# =================================================================================================
def _cpu_block(args):
    """One bounded sample: a chromosome-shaped block (nb bins, all pairs within max_dist) through the whole
    reference path restated in oracle/fithic_oracle.py: histogram, binning, spline, scoring, BH."""
    nb, seed, repeat, R, max_dist, depth = args
    import numpy as np
    from blueberry_b200 import synth
    from oracle import fithic_oracle as fo
    bias = synth.make_bias([nb], seed)
    fc, fm = synth.make_fragments([nb], R)
    c = synth.make_contacts([nb], R, max_dist, depth, seed, bias)
    bd, _ = fo.read_bias_arrays(np.zeros(nb, dtype=np.int64), fm, bias[0])
    t0 = time.perf_counter()
    for _ in range(repeat):
        res = fo.fithic_arrays(fc, fm, None, c["mid1"], None, c["mid2"], c["count"], R, N_BINS, 0, max_dist, bias=bd)
        keep = res.keep
        fo.benjamini_hochberg_correction(res.p[keep], int(keep.sum()))
    return len(c["count"]) * repeat, time.perf_counter() - t0


def cpu_baseline(cores, wl, nb=3000, repeat=1):
    """pairs/s of the oracle port on `cores` host processes (each gets its own block)."""
    import multiprocessing as mp
    jobs = [(nb, SEED + 101 * i, repeat, wl["R"], wl["max_dist"], wl["depth"]) for i in range(cores)]
    t0 = time.perf_counter()
    if cores == 1:
        res = [_cpu_block(jobs[0])]
        wall = res[0][1]
    else:
        with mp.get_context("spawn").Pool(cores) as pool:
            res = pool.map(_cpu_block, jobs)
        wall = max(r[1] for r in res)              # slowest worker's compute time (generation excluded)
    pairs = sum(r[0] for r in res)
    return pairs / wall, pairs, wall, time.perf_counter() - t0


def run_reference_arm(args, out_fd):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    cores = min(os.cpu_count() or 1, 64)
    nb = 2600 if wl["R"] == 5000 else 4200
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_baseline(cores, wl, nb=nb)
    vals, per_step = [], []
    for _ in range(args.steps):
        v, pairs, wall, _ = cpu_baseline(cores, wl, nb=nb)
        vals.append(v); per_step.append(wall)
    value = statistics.mean(vals)
    K = wl["max_dist"] // wl["R"]
    sample = "%d blocks/step of %d bins (all pairs within %d bp at %d bp, ~%.1fM records each), one per core" % (
        cores, nb, wl["max_dist"], wl["R"], ((K + 1) * nb - K * (K + 1) // 2) / 1e6)
    line = {
        "impl": "reference", "metric": "fithic_contact_pairs_per_sec", "value": value, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(per_step),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"] + " (bounded sample per step)", "resolution": wl["R"],
                   "n_bins": N_BINS, "max_dist": wl["max_dist"]},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample,
                         "true_reference": _true_reference(),
                         "note": "oracle/fithic_oracle.py (numpy / scipy restatement of fithic.py, ~100x faster than the reference's "
                                 "per-line Python; the unmodified reference itself needs /root/reference, absent on the GPU box - "
                                 "its rate, timed in the build container, is in DESIGN.md section 5)"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(out_fd, line)


# =================================================================================================
# GPU arm
# =================================================================================================
class Workload(object):
    """This rank's share of a synthetic genome, resident on the device, plus the genome-wide tables every rank holds."""

    def __init__(self, wl, world, rank, dev, pieces=None, share_of=None):
        import numpy as np
        import torch
        from blueberry_b200 import _lib
        from blueberry_b200.distributed import layout_rows, plan_shards
        from blueberry_b200.engine import BiasTables, PassEngine, Shard
        lib = _lib.load()
        R, K = wl["R"], wl["max_dist"] // wl["R"]
        self.R, self.K, self.max_dist = R, K, wl["max_dist"]
        chrom_list = list(wl["chroms"])
        if share_of:
            # a single-GPU stand-in for a larger box: the genome of this run is what `world` of `share_of` GPUs would hold as
            # WHOLE chromosomes (longest-processing-time packing), so that possible pairs, S and the spline stay consistent
            pairs_all = [int(lib.bbk_synth_n_pairs(-(-HG19[c] // R), K)) for c in chrom_list]
            lpt = plan_shards(pairs_all, share_of, mode="lpt")
            chrom_list = [chrom_list[c] for c in sorted(c for r in range(world) for (c, _, _) in lpt[r])]
        self.chrom_list = chrom_list
        self.bins = [-(-HG19[c] // R) for c in chrom_list]
        self.pairs = [int(lib.bbk_synth_n_pairs(nb, K)) for nb in self.bins]
        plan = plan_shards(self.pairs, world)
        mine = plan[rank]
        self.P_total = sum(n for r in range(world) for (_, _, n) in plan[r])
        self.sizes = [n for (_, _, n) in mine]
        self.chroms = [c for (c, _, _) in mine]
        starts, rows = layout_rows(self.sizes)
        self.starts, self.rows = starts, max(rows, 4)
        self.P_local = sum(self.sizes)
        self.mid1, self.mid2, self.count = (torch.zeros(self.rows, dtype=torch.int32, device=dev) for _ in range(3))
        bias_host = []
        for ci, nb in enumerate(self.bins):
            rng = np.random.default_rng(SEED + 7919 * (chrom_list[ci] + 1))
            bias_host.append(np.exp(rng.normal(0.0, 0.25, size=nb)))
        self.bias_host = bias_host
        for (c, first, n), off in zip(mine, starts):
            bdev = torch.from_numpy(bias_host[c]).to(dev)
            _lib.check(lib.bbk_synth_contacts_range(self.bins[c], K, R, wl["depth"], DECAY, SEED + 1000003 * chrom_list[c], _lib.ptr(bdev), first, n,
                                                    ctypes_ptr(self.mid1, off), ctypes_ptr(self.mid2, off), ctypes_ptr(self.count, off),
                                                    _lib.stream_ptr()), "bbk_synth_contacts_range")
            torch.cuda.synchronize()
        self.shards = [Shard(self.mid1[a:a + n], self.mid2[a:a + n], self.count[a:a + n], chrom=c)
                       for a, n, c in zip(starts, self.sizes, self.chroms)]
        self.nkeys = max(self.bins)                      # maxPossibleGenomicDist / R + 1 (fithic.py:300-303)
        self.eng = PassEngine(R, N_BINS, 0, self.max_dist, self.nkeys, dev)
        self.eng.set_fragments(self.bins, [(nb - 1) * R for nb in self.bins])
        tabs = [np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias_host]       # read_bias_file, fithic.py:147-149
        self.eng.set_bias(BiasTables(tabs, [R // 2] * len(self.bins), dev))
        self.possible_in_range = sum(nb * K - K * (K + 1) // 2 for nb in self.bins)   # d = R .. K*R


def ctypes_ptr(t, offset_elems=0):
    import ctypes
    return ctypes.c_void_p(t.data_ptr() + offset_elems * t.element_size())


def _parity_bits(W, gp, fit, dev, world):
    """Checks carried in the JSON line: (1) K1's table and S against torch.index_add_ over the same records (all-reduced),
    bit-exact; (2) a strided 1e6-record sample of p against the oracle's scoring (scipy bdtrc) with the device's spline."""
    import numpy as np
    import torch
    import torch.distributed as dist
    out = {}
    eng = W.eng
    tab = torch.zeros(W.nkeys, dtype=torch.int64, device=dev)
    S = torch.zeros(1, dtype=torch.int64, device=dev)
    for sh in W.shards:
        if sh.n == 0:
            continue
        d = (sh.mid2 - sh.mid1).to(torch.int64)
        ok = (d > 0) & (d <= W.max_dist)                                   # fithic.py:256-257 (min_dist = 0: d > 0)
        S += sh.count[ok].sum(dtype=torch.int64)
        key = ok & (d % W.R == 0) & (d // W.R < W.nkeys)
        tab.index_add_(0, (d[key] // W.R), sh.count[key].to(torch.int64))
        del d, ok, key
    if world > 1:
        dist.all_reduce(tab)
        dist.all_reduce(S)
    out["hist_equal_index_add"] = bool(torch.equal(tab, eng.obs_sum)) and int(S.item()) == int(eng.totals[0].item())
    # p sample vs the oracle
    try:
        from oracle import fithic_oracle as fo
        i_sh = max(range(len(W.shards)), key=lambda i: W.shards[i].n) if W.shards else None
        if i_sh is not None and W.shards[i_sh].n:
            sh = W.shards[i_sh]
            stride = max(1, sh.n // 1_000_000)
            sel = torch.arange(0, sh.n, stride, device=dev)
            m1, m2, cn = (t[sel].cpu().numpy() for t in (sh.mid1, sh.mid2, sh.count))
            pg = gp.shard_p(i_sh)[sel].cpu().numpy()
            sy = eng.spline_y[:fit.L].cpu().numpy()
            tabb = np.where((W.bias_host[sh.chrom] < 0.5) | (W.bias_host[sh.chrom] > 2), -1.0, W.bias_host[sh.chrom])
            b1, b2 = tabb[(m1 - W.R // 2) // W.R], tabb[(m2 - W.R // 2) // W.R]
            pr, scored, keep = fo.score_pairs(m1, m2, cn, int(fit.S), fit.k0, sy, W.R, 0, W.max_dist, b1, b2)
            same_keep = bool(np.array_equal(pg <= 1, keep))
            kk = keep & (pr > 1e-290) & (pg <= 1)
            err = float(np.abs(np.log10(pg[kk]) - np.log10(pr[kk])).max()) if kk.any() else 0.0
            out["p_sample_rows"] = int(len(sel))
            out["p_sample_keep_equal"] = same_keep
            out["p_sample_max_dlog10p_vs_scipy"] = err
            out["S"] = int(fit.S)
    except Exception as e:                                                     # the oracle is a checker, never a dependency
        out["p_sample_error"] = repr(e)
    return out


def _measure(args, wl_name, world, rank, dev, full, out):
    """Times one workload; fills `out` (dict).  full: also stages, e2e, parity (the headline workload)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from blueberry_b200.distributed import GenomePass, HostStream
    from blueberry_b200.engine import PassEngine

    wl = WORKLOADS[wl_name]
    share_of = None
    if wl_name == "cfg5" and world < 8:
        share_of = 8                                     # one GPU cannot hold the genome at 1 kb: `world` of 8 pieces
    W = Workload(wl, world, rank, dev, share_of=share_of)
    gp = GenomePass(W.eng, q_values=True)
    gp.attach(W.shards)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    two_pass = wl["two_pass"]
    if two_pass:
        # config 4: pass 1 (p only) -> statistics without the outliers -> refit -> every record scored again, with q-values
        gp1 = GenomePass(W.eng, q_values=False)
        gp1.attach(W.shards)
        p_outlier = 1.0 / float(W.possible_in_range)

        def step():
            gp1.enqueue()
            gp.enqueue(exclude=(gp1.p, p_outlier))
    else:
        def step():
            gp.enqueue()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    barrier()
    fit = gp.finish()                                           # raises for a failed fit; settles the gather capacity
    W.eng.launches = 0
    step()
    launches_per_step = W.eng.launches
    barrier()

    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) if (rank == 0 and full) else None
    if sampler:
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.mark_start()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    if sampler:
        sampler.mark_end()
    ms = e0.elapsed_time(e1)
    tms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_per_step = float(tms.item()) / args.steps
    out["clocks"] = sampler.stop() if sampler else None
    if full and rank == 0 and args.dump_outputs:
        _dump_outputs(args.dump_outputs, W, gp)
    out["ms_per_step"] = ms_per_step
    out["P_total"], out["P_local"] = W.P_total, W.P_local
    out["value"] = W.P_total / (ms_per_step * 1e-3)
    peak, peak_src = _peaks()
    bpp = 104 if two_pass else BYTES_PER_PAIR
    out["whole_pass_frac"] = bpp * W.P_total / (ms_per_step * 1e-3) / 1e9 / (peak * world)
    out["launches_per_step"] = launches_per_step
    out["workload_name"] = wl["name"] + (" (stand-in for an 8-GPU box: the %d whole chromosomes %d of 8 GPUs would hold, %s)" % (len(W.chrom_list), world, ",".join(str(c + 1) for c in W.chrom_list)) if share_of else "")
    out["W"], out["gp"], out["fit"] = W, gp, fit
    if not full or two_pass:
        if two_pass:
            out["stages_ms"] = None
        return

    # ---- per-stage device times (separate instrumented steps; CUDA events on the streams the kernels run on)
    names = ["hist", "allreduce", "fit", "pvalues", "bh"]
    acc = dict((n, 0.0) for n in names)
    reps = min(args.steps, 5)
    for _ in range(reps):
        marks = {}
        gp.enqueue(marks=marks)
        torch.cuda.synchronize()
        prev = "start"
        for n in names:
            if n in marks:
                acc[n] += marks[prev].elapsed_time(marks[n]) / reps
                prev = n
    # the K4 kernels alone, back to back on one stream (what the roofline object is computed from)
    k4a = k4b = 0.0
    if gp.listed:
        from blueberry_b200 import _lib
        import ctypes
        eng, lib = W.eng, W.eng.lib
        bias = ctypes.byref(eng.bias.struct) if eng.bias is not None else None
        flags = _lib.ptr(eng.bias.flags) if eng.bias is not None else None
        for _ in range(reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            st = _lib.stream_ptr()
            _lib.check(lib.bbk_score_begin(_lib.ptr(gp.score_state), _lib.ptr(eng.p_hist), st), "bbk_score_begin")
            _lib.check(lib.bbk_score_guard(_lib.ptr(eng.fit_result), _lib.ptr(eng.spline_y), _lib.ptr(gp.score_state), st), "bbk_score_guard")
            ev[0].record()
            live = [(sh, off) for sh, off in zip(gp.shards, gp.offsets) if sh.n]
            for (sh, off), st_i in zip(live, eng.fan_out(len(live))):
                _lib.check(lib.bbk_score_pairs(_lib.ptr(sh.mid1), _lib.ptr(sh.mid2), _lib.ptr(sh.count), sh.n, sh.chrom, eng.R,
                                               eng.min_dist, eng.max_dist, _lib.ptr(eng.fit_result), _lib.ptr(eng.spline_y), bias, flags,
                                               off, _lib.ptr(gp.p), _lib.ptr(gp.q), _lib.ptr(eng.p_hist), ctypes.byref(gp.cands),
                                               ctypes.byref(gp.deferred), _lib.ptr(gp.score_state), st_i), "bbk_score_pairs")
            eng.fan_in()
            ev[1].record()
            _lib.check(lib.bbk_score_deferred(ctypes.byref(gp.deferred), _lib.ptr(eng.fit_result), _lib.ptr(gp.p), _lib.ptr(gp.q),
                                              _lib.ptr(eng.p_hist), ctypes.byref(gp.cands), _lib.ptr(gp.score_state), st), "bbk_score_deferred")
            ev[2].record()
            torch.cuda.synchronize()
            k4a += ev[0].elapsed_time(ev[1]) / reps
            k4b += ev[1].elapsed_time(ev[2]) / reps
        gp.enqueue()                                     # leave a complete pass behind (q-values included)
        torch.cuda.synchronize()
    score = _score_state(gp)
    out["stages_ms"] = acc
    out["k4_alone_ms"] = {"score_tiles_kernel": k4a, "score_deferred_kernel": k4b}
    out["work_list"] = {"deferred_rows": int(score.n_list), "candidates_p_lt_2^-5": int(score.n_cand), "exact_mode": int(score.exact)}
    tmax = torch.tensor([k4a + k4b, acc["hist"], acc["bh"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    k4_ms = float(tmax[0].item())
    k4_gbs = K4_BYTES_PER_PAIR * W.P_total / world / (k4_ms * 1e-3) / 1e9 if k4_ms > 0 else 0.0
    out["roofline"] = {
        "bound": "hbm", "kernel": "K4 = score_tiles_kernel (one launch per shard) + score_deferred_kernel (per GPU, timed back to back on one stream)",
        "achieved": k4_gbs, "peak": peak, "unit": "GB/s", "frac": k4_gbs / peak,
        "traffic": _k4_traffic(wl_name, world), "peak_source": peak_src,
        "algorithmic_bytes_per_launch": K4_BYTES_PER_PAIR * W.P_total // world,
        "traffic_note": "K4 also writes the 8 B/pair of q that the byte table books under K5 (28 B/pair moved for 20 algorithmic); "
                        "traffic is null unless profiles/k4_traffic.json holds a capture of these sources",
        "whole_pass_frac": out["whole_pass_frac"],
        "stage_gbs_per_gpu": {"hist (12 B/pair)": 12 * W.P_local / (acc["hist"] * 1e-3) / 1e9 if acc["hist"] > 0 else None,
                              "score_tiles (12 B/pair in + 16 B/pair of p, q out)": 28 * W.P_local / (k4a * 1e-3) / 1e9 if k4a > 0 else None},
    }
    out["parity"] = _parity_bits(W, gp, fit, dev, world)

    # ---- throughput with TWO passes in flight (a second engine + GenomePass on a second stream, passes alternate): the
    # one-CTA fit and the launch-bound q-value step of one pass run beside the streaming kernels of the other, and K1 (DRAM-bound)
    # shares the SMs with K4 (issue-bound).  Reported beside the headline, which stays the time of one pass on its own.
    # (N > 1: only on request, --overlap on - the second lane gets its own process group, i.e. its own NCCL communicator, so that
    # its collectives do not queue behind the first lane's.)
    if args.overlap == "on" or (args.overlap == "auto" and world == 1):
        try:
            eng2 = PassEngine(W.R, N_BINS, 0, W.max_dist, W.nkeys, dev)
            eng2.set_fragments(W.bins, [(nb - 1) * W.R for nb in W.bins])
            eng2.set_bias(W.eng.bias)
            group2 = dist.new_group(list(range(world))) if world > 1 else None
            gp2 = GenomePass(eng2, group=group2, q_values=True, gather_capacity=gp.gather_cap)
            gp2.attach(W.shards)
            lanes = [(gp, torch.cuda.Stream(dev)), (gp2, torch.cuda.Stream(dev))]
            main = torch.cuda.current_stream(dev)

            def run_overlapped(k):
                for _, s in lanes:
                    s.wait_stream(main)
                for i in range(k):
                    g, s = lanes[i & 1]
                    with torch.cuda.stream(s):
                        g.enqueue()
                for _, s in lanes:
                    main.wait_stream(s)

            run_overlapped(4)
            barrier()
            with torch.cuda.stream(lanes[1][1]):
                gp2.finish()                                 # settles its lists / gather capacity (collective at N > 1)
            barrier()
            o_steps = max(2, args.steps) & ~1
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            f0.record()
            run_overlapped(o_steps)
            f1.record()
            barrier()
            tms = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            o_ms = float(tms.item()) / o_steps
            same = bool(torch.equal(gp.p[:gp.rows].view(torch.int64), gp2.p[:gp2.rows].view(torch.int64))) and \
                bool(torch.equal(gp.q[:gp.rows].view(torch.int64), gp2.q[:gp2.rows].view(torch.int64)))
            out["two_passes_in_flight"] = {"ms_per_pass": o_ms, "value": W.P_total / (o_ms * 1e-3), "unit": "pairs/s", "passes": o_steps,
                                           "whole_pass_frac": bpp * W.P_total / (o_ms * 1e-3) / 1e9 / (peak * world),
                                           "both_lanes_bit_identical": same,
                                           "note": "throughput over independent passes (e.g. successive samples), two at a time on two streams; "
                                                   "the headline ms_per_step is one pass on its own"}
            del gp2, eng2, lanes
            torch.cuda.empty_cache()
            gp.enqueue()
            torch.cuda.synchronize()
        except Exception as e:                                                 # an extra: never fatal for the line
            out["two_passes_in_flight"] = {"error": repr(e)}

    # ---- end to end (1): host (pinned) tables in, p and q back to the host, every step, through distributed.HostStream.
    # The results cross the host link packed (two bits per row + the values that are not 1.0 / NaN, bbk_pack_scores); the dense
    # float64 columns are rebuilt on the host OUTSIDE the timed region and compared with the device's columns bit for bit.
    h_in = [torch.empty(W.rows, dtype=torch.int32).pin_memory() for _ in range(3)]
    for h, d in zip(h_in, (W.mid1, W.mid2, W.count)):
        h.copy_(d)
    torch.cuda.synchronize()
    W.mid1 = W.mid2 = W.count = None                     # the stream's device slots take their place (memory)
    W.shards = []
    gp.shards, gp.p, gp.q = [], None, None
    torch.cuda.empty_cache()
    pipe = HostStream(gp, W.sizes, W.chroms, slots=2, packed=True)
    outs = [pipe.packed_buffers() for _ in range(2)]
    e2e_steps = max(2, min(args.steps, 10 if W.P_local < 200_000_000 else 6))
    for k in range(2):
        pipe.submit_packed(h_in[0], h_in[1], h_in[2], outs[k % 2])
    pipe.drain(); torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        pipe.submit_packed(h_in[0], h_in[1], h_in[2], outs[k % 2])
    pipe.drain(); torch.cuda.synchronize()
    resub = 0
    for k in range(pipe.submitted - 2, pipe.submitted):
        if PassEngine.reference_smoothing(pipe.fit_of(k)) is not None:
            resub += 1
    wall = time.perf_counter() - t0
    barrier()
    tms = torch.tensor([wall * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    e2e_ms = float(tms.item()) / e2e_steps
    last = outs[(e2e_steps - 1) % 2]
    d2h = torch.tensor([float(last.nbytes() + int(W.eng.fit_result.numel()))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(d2h)
    t1 = time.perf_counter()
    h_p, h_q = last.dense()
    unpack_s = time.perf_counter() - t1
    slot = pipe.slots[(pipe.submitted - 1) % 2]
    same = bool(np.array_equal(h_p.view(np.uint64), slot.p.cpu().numpy().view(np.uint64))) and \
        bool(np.array_equal(h_q.view(np.uint64), slot.q.cpu().numpy().view(np.uint64)))
    out["emitted_rows_rank0"] = int((h_p <= 1).sum())
    out["q_le_0.01_rank0"] = int((h_q <= 0.01).sum())
    out["e2e"] = {"value": W.P_total / (e2e_ms * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": 12 * W.rows * world,
                  "d2h_bytes_per_step": int(d2h.item()),
                  "steps": e2e_steps, "ms_per_step": e2e_ms,
                  "mode": "distributed.HostStream(packed=True): pinned host tables in; p and q back as two bits per row + the values that are not "
                          "1.0 / NaN (lossless), pipelined across steps (2 device slots)",
                  "dense_bytes_per_step": 16 * W.rows * world, "packed_values_rank0": {"p": last.n_p, "q": last.n_q, "overflow": last.overflow},
                  "unpacked_equals_device_columns_rank0": same, "host_unpack_s_rank0_untimed": unpack_s,
                  "fit_checked_passes": 2, "smoothing_resubmits": resub}
    del pipe, h_in, outs, last, h_p, h_q
    out["parity"]["e2e_unpacked_equals_device_columns"] = same

    # ---- end to end (2): the drop-in array call users make, FitHiC.fit_transform_arrays (numpy in, numpy out), on chr1 of
    # the same genome (one process; rank 0 only) - staging, the pass, and the copy back of p / q and all the tables
    if rank == 0 and not args.no_dropin:
        from blueberry_b200.fithic import FitHiC
        c0 = 0
        nb, K, R = W.bins[c0], W.K, W.R
        from blueberry_b200 import _lib
        lib = W.eng.lib
        n = int(lib.bbk_synth_n_pairs(nb, K))
        n = min(n, 100_000_000)
        cols = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(3)]
        bdev = torch.from_numpy(W.bias_host[c0]).to(dev)
        _lib.check(lib.bbk_synth_contacts_range(nb, K, R, wl["depth"], DECAY, SEED + 1000003 * c0, _lib.ptr(bdev), 0, n,
                                                _lib.ptr(cols[0]), _lib.ptr(cols[1]), _lib.ptr(cols[2]), _lib.stream_ptr()), "synth")
        m1, m2, cn = (c.cpu().numpy() for c in cols)
        del cols
        fm = (np.arange(nb, dtype=np.int64) * R + R // 2)
        fc = np.zeros(nb, dtype=np.int32)
        model = FitHiC("bench", R, n_bins=N_BINS, max_dist=W.max_dist)
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            res = model.fit_transform_arrays(None, m1, None, m2, cn, fc, fm, bias=(fc, fm, W.bias_host[c0]), q_values=True)
            times.append(time.perf_counter() - t0)
        best = min(times[1:])
        out["e2e_dropin"] = {"call": "FitHiC.fit_transform_arrays(numpy columns) -> numpy p, q", "workload": "chr1 of the same genome",
                             "pairs": n, "ms_per_call": 1e3 * best, "value": n / best, "unit": "pairs/s", "n_gpus": 1,
                             "h2d_bytes": 12 * n, "result_bytes_dense": 16 * n,
                             "note": "numpy (pageable) columns in, numpy p / q / keep out; the results cross the link packed and are unpacked by all host cores",
                             "kept_rows": int(res.keep.sum())}


def _score_state(gp):
    from blueberry_b200 import _lib
    return _lib.ScoreState.from_buffer_copy(gp.score_state.cpu().numpy().tobytes())


def _dump_outputs(path, W, gp):
    """What a caller of GenomePass holds after the last timed step, as float64 .npy files under `path`: for a fixed, seeded
    sample of this rank's records (row = the record's index in shard order) keep = (p <= 1) and the p and q of the kept
    ones (a record that is not scored or is dropped holds NaN, fithic.py:431-434), the distance table and totals K1 left,
    the fit's bins and spline, and the fit's scalars."""
    import numpy as np
    import torch
    eng = W.eng
    fit = eng.read_fit()
    sizes = [sh.n for sh in gp.shards]
    starts = np.cumsum([0] + sizes)
    n = int(starts[-1])
    rows = np.unique(np.random.default_rng(SEED).integers(0, n, DUMP_ROWS)) if n else np.zeros(0, dtype=np.int64)
    shard = np.searchsorted(starts, rows, side="right") - 1
    idx = torch.from_numpy(np.asarray(gp.offsets, dtype=np.int64)[shard] + rows - starts[shard]).to(eng.device)
    p, q = gp.p[idx].cpu().numpy(), gp.q[idx].cpu().numpy()
    keep = p <= 1
    arrays = {
        "row": rows, "keep": keep, "p": p[keep], "q": q[keep], "observed": eng.obs_sum, "totals": eng.totals,
        "x": eng.x[:fit.n_out], "y": eng.y[:fit.n_out], "spline_y": eng.spline_y[:fit.L],
        "fit": np.array([fit.S, fit.k0, fit.L, fit.n_out, fit.n_knots, fit.min_x, fit.max_x, fit.residual, fit.smoothing]),
    }
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


def run_ours(args, out_fd):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    main = {}
    _measure(args, args.workload, world, rank, dev, True, main)
    W, gp, fit = main.pop("W"), main.pop("gp"), main.pop("fit")
    wl = WORKLOADS[args.workload]
    totals = W.eng.totals.cpu().numpy()
    n_knots = int(fit.n_knots)
    fit_cycles = dict(zip(["stage+boundaries", "bin_stats", "spline_search", "grid_eval", "pava+residual", "total"],
                          [int(v) for v in fit.phase_cycles]))
    sizes_gb = 12 * W.P_local / 1e9
    del W, gp
    torch.cuda.empty_cache()

    extra = {}
    if world == 8 and args.workload == "cfg3" and not args.no_cfg5:
        c5 = {}
        _measure(args, "cfg5", world, rank, dev, False, c5)
        extra = {"cfg5_ms_per_step": c5["ms_per_step"], "cfg5_frac": c5["whole_pass_frac"], "cfg5_pairs": c5["P_total"],
                 "cfg5_pairs_per_sec": c5["value"],
                 "cfg5_note": "BASELINE config 5 on the same 8 GPUs right after the headline workload: genome-wide 1 kb, 2 Mb cap, band-sharded; "
                              "frac = 48 B x pairs / (time x 8 x peak); north_star target >= 0.60"}
        c5.pop("W"); c5.pop("gp"); c5.pop("fit")
        torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, pairs, wall_c, _ = cpu_baseline(1, wl, nb=4500)
        cpu = {"value": v, "unit": "pairs/s", "cores": 1, "kind": "port", "true_reference": _true_reference(),
               "sample": "one %d-bin block of the same workload (%.1fM records): histogram, binning, spline, bdtrc scoring, BH; "
                         "oracle/fithic_oracle.py on 1 of %d host cores, %.1f s" % (4500, pairs / 1e6, os.cpu_count() or 1, wall_c)}

    if rank == 0:
        line = {
            "metric": "fithic_contact_pairs_per_sec", "value": main["value"], "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if args.workload != "cfg5" or world >= 8 else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": main["workload_name"], "pairs_total": main["P_total"], "pairs_rank0": main["P_local"],
                       "resolution": wl["R"], "max_dist": wl["max_dist"], "n_bins": N_BINS, "biases": True,
                       "entry_point": "blueberry_b200.distributed.GenomePass" + (" (two passes: enqueue(), then enqueue(exclude=(p_first, 1/possibleIntraInRangeCount)))" if wl["two_pass"] else ""),
                       "sharding": "distributed.plan_shards: equal record counts, whole chromosomes, row blocks where a chromosome straddles a cut",
                       "q_values": "genome-wide (histogram all-reduce + fixed-capacity candidate all-gather, no host round trip)" if world > 1 else "genome-wide (one rank)",
                       "l2": "inputs (%.2f GB on rank 0) exceed the 126 MB L2" % sizes_gb,
                       "bytes_per_pair": 104 if wl["two_pass"] else BYTES_PER_PAIR, "S": int(totals[0]), "spline_knots": n_knots,
                       "emitted_rows_rank0": main.get("emitted_rows_rank0"), "q_le_0.01_rank0": main.get("q_le_0.01_rank0")},
            "stages_ms": main.get("stages_ms"),
            "k4_alone_ms": main.get("k4_alone_ms"),
            "work_list": main.get("work_list"),
            "fit_phase_cycles": fit_cycles,
            "roofline": main.get("roofline") or {"bound": "hbm", "whole_pass_frac": main["whole_pass_frac"]},
            "whole_pass_frac": main["whole_pass_frac"],
            "parity": main.get("parity"),
            "cpu_baseline": cpu,
            "e2e": main.get("e2e"),
            "e2e_dropin": main.get("e2e_dropin"),
            "two_passes_in_flight": main.get("two_passes_in_flight"),
            "gpu_launches": main["launches_per_step"] * args.steps,
            "clocks": main.get("clocks"),
        }
        line.update(extra)
        _emit(out_fd, line)
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """Keep stdout for the ONE JSON line: libraries (NCCL prints its version banner there) get stderr instead."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit(saved_fd, line):
    sys.stdout.flush()
    os.write(saved_fd, (json.dumps(line) + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-dropin", action="store_true", help="skip the fit_transform_arrays end-to-end leg")
    ap.add_argument("--no-cfg5", action="store_true", help="--gpus 8: skip the extra BASELINE config 5 measurement")
    ap.add_argument("--overlap", default="auto", choices=["auto", "on", "off"],
                    help="the two-passes-in-flight throughput measurement: auto = on one GPU only")
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS),
                    help="cfg3 (default: the configuration the metric is quoted on), cfg2, cfg4 (two passes) or cfg5")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write keep / p / q (a seeded sample of rank 0's records) and the fit of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU pass (--impl ours)")
    out_fd = _claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args, out_fd)
    else:
        run_ours(args, out_fd)


if __name__ == "__main__":
    main()
