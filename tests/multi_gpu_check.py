"""Run under torchrun on N GPUs (driven by tests/test_gpu_genome_pass.py, or by hand): the public multi-GPU pass
(distributed.GenomePass over distributed.plan_shards pieces - chromosomes split across ranks) against the
single-process CPU oracle on ALL records: all-reduced distance table and S, p per rank, genome-wide q bit for bit.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 tests/multi_gpu_check.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.dup2(2, 1)
    dist.init_process_group("nccl", device_id=dev)
    from blueberry_b200 import synth
    from blueberry_b200.distributed import GenomePass, plan_shards
    from blueberry_b200.engine import BiasTables, PassEngine, Shard
    from oracle import fithic_oracle as fo

    R, bins, max_dist = 10000, [420, 380, 300, 260, 150, 90], 2_000_000
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, 4)
    c = synth.make_contacts(bins, R, max_dist, 90.0, 23, bias)                 # same on every rank (seeded)
    pairs = [int((c["chrom"] == i).sum()) for i in range(len(bins))]
    starts = np.concatenate([[0], np.cumsum(pairs)])
    plan = plan_shards(pairs, world)
    t32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
    shards, rows = [], []
    for (ci, first, n) in plan[rank]:
        a = int(starts[ci]) + first
        shards.append(Shard(t32(c["mid1"][a:a + n]), t32(c["mid2"][a:a + n]), t32(c["count"][a:a + n]), chrom=ci))
        rows.append(np.arange(a, a + n))
    rows = np.concatenate(rows) if rows else np.zeros(0, dtype=np.int64)
    bc = np.concatenate([np.full(b, i) for i, b in enumerate(bins)])
    bd, _ = fo.read_bias_arrays(bc, fm, np.concatenate(bias))
    ok = True
    # the streaming K4 with its candidate list, then the direct kernel (max_dist + R = 2^31 is beyond the streaming K4's
    # 31-bit distances) with a select pass over p: both go through the same fixed-capacity all-gather
    for pass_max_dist, listed in ((max_dist, True), (2 ** 31 - R, False)):
        eng = PassEngine(R, 100, 0, pass_max_dist, max(bins), dev)
        eng.set_fragments(bins, [(b - 1) * R for b in bins])
        eng.set_bias(BiasTables([np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias], [R // 2] * len(bins), dev))
        # a deliberately small gather capacity: the first pass overflows it, finish() grows it and repeats
        gp = GenomePass(eng, q_values=True, gather_capacity=256)
        gp.attach(shards)
        ok &= gp.listed == listed
        fit = gp.run()
        grown = gp.gather_cap
        p = np.concatenate([gp.shard_p(i).cpu().numpy() for i in range(len(shards))]) if shards else np.zeros(0)
        q = np.concatenate([gp.shard_q(i).cpu().numpy() for i in range(len(shards))]) if shards else np.zeros(0)

        # single-process oracle on ALL records
        ref = fo.fithic_arrays(fc, fm, c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], R, 100, 0, pass_max_dist, bias=bd)
        ok &= np.array_equal(eng.obs_sum.cpu().numpy(), ref.contacts.observed) and int(fit.S) == ref.contacts.S
        t = eng.totals.cpu().numpy()
        ok &= int(t[6]) == ref.contacts.min_obs_dist and int(t[7]) == ref.contacts.max_obs_dist and int(t[1]) == ref.contacts.intra_in_range_count
        ok &= np.array_equal(eng.spline_y[:fit.L].cpu().numpy(), ref.spline_y)
        keep_ref = ref.keep[rows]
        ok &= np.array_equal(p <= 1, keep_ref)
        kk = keep_ref & (ref.p[rows] > 0)
        err = float(np.abs(np.log10(p[kk]) - np.log10(ref.p[rows][kk])).max()) if kk.any() else 0.0
        ok &= err <= 1e-6
        # genome-wide q: every rank's p gathered, ranked together by the oracle; this rank's rows must match bit for bit
        sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([len(p)], dtype=torch.int64, device=dev))
        sizes = [int(s.item()) for s in sizes]
        cap = max(max(sizes), 1)
        buf = torch.full((cap,), float("nan"), dtype=torch.float64, device=dev)
        buf[:len(p)] = torch.from_numpy(p).to(dev)
        allp = [torch.empty(cap, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(allp, buf)
        p_all = np.concatenate([a[:s].cpu().numpy() for a, s in zip(allp, sizes)])
        valid = ~np.isnan(p_all)
        q_ref_all = np.full(len(p_all), np.nan)
        q_ref_all[valid] = fo.benjamini_hochberg_correction(p_all[valid], int(valid.sum()))
        off = sum(sizes[:rank])
        mine = q_ref_all[off:off + len(p)]
        same = np.array_equal(np.isnan(q), np.isnan(mine)) and np.array_equal(q[~np.isnan(q)], mine[~np.isnan(mine)])
        ok &= same
        ok &= grown > 256                                                      # the overflow path was exercised
        if rank == 0:
            sys.stderr.write("multi_gpu_check world=%d listed=%s: records/rank %s, gather capacity 256 -> %d, max |dlog10 p| %.3g, "
                             "q identical %s\n" % (world, listed, sizes, grown, err, same))
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        sys.stderr.write("multi_gpu_check world=%d -> %s\n" % (world, "OK" if flag.item() else "FAILED"))
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
