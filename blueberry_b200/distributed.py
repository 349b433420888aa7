"""The Fit-Hi-C significance pass over many shards and many GPUs (the path BASELINE.json's north_star names:
"pairs are sharded by chromosome, or by diagonal band within large chromosomes, across the GPUs of a single box").

One process per GPU.  Every rank holds some shards (whole chromosomes, or row blocks of a chromosome that straddles a
cut); what the reference keeps in ONE global table and ONE global S (fithic.py:110-133: one mainDic, one
observedIntraInRangeSum) is made global by a single integer all-reduce after K1; the fit is then replicated
bit-identically on every rank, scoring is local, and the q-values are ranked genome-wide (the reference's q-value step
gathers the p-values of all chromosomes, utils.py:31-90 -> blueberry.pyx:40-75) through an all-reduce of the 4096-bucket
p histogram and one fixed-capacity all-gather of the few candidate keys.  Nothing between the first and the last kernel
of a pass touches the host.

    K1 per shard -> [all-reduce] -> fit (one CTA) -> guard -> K4 per shard (one streaming pass over bulk-staged tiles)
    -> K4 patch pass over the deferred rows -> K5 q-values (local, or genome-wide across ranks)

GenomePass is that sequence; plan_shards / shard_rows decide who holds what.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .engine import PassEngine, Shard


def _world(group=None):
    """(world size, rank) of `group`; None = the default group when torch.distributed is initialised; False = this
    process alone whatever is initialised."""
    import torch.distributed as dist
    if group is False:
        return 1, 0
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group), dist.get_rank(group)
    return 1, 0


def plan_shards(pairs_per_chrom, world, mode="balanced", align=4):
    """Who holds which records.  pairs_per_chrom[c] = number of records of chromosome c (in its own order).

    mode "balanced": the chromosomes, laid end to end, are cut into `world` pieces of equal record count (to `align`
    records); a chromosome that straddles a cut is split into row blocks (no halo: pairs are independent once the
    distance table is global), so at most world-1 chromosomes are split.
    mode "lpt": whole chromosomes only, longest-processing-time bin packing (sharding.lpt_assign).
    Returns plan[rank] = [(chrom, first_record, n_records), ...]."""
    pairs = [int(x) for x in pairs_per_chrom]
    if mode == "lpt":
        from .sharding import lpt_assign
        owner = lpt_assign(pairs, world)
        return [[(c, 0, pairs[c]) for c in range(len(pairs)) if owner[c] == r and pairs[c] > 0] for r in range(world)]
    if mode != "balanced":
        raise ValueError("mode must be 'balanced' or 'lpt'")
    total = sum(pairs)
    cuts = [min(total, (total * r // world + align - 1) // align * align) for r in range(world)] + [total]
    plan = [[] for _ in range(world)]
    start = 0
    for c, n in enumerate(pairs):
        for r in range(world):
            lo, hi = max(cuts[r], start), min(cuts[r + 1], start + n)
            if hi > lo:
                plan[r].append((c, lo - start, hi - lo))
        start += n
    return plan


def shard_rows(n_rows, world, rank, align=4):
    """Rows [lo, hi) of an arbitrary record table that rank `rank` takes: equal contiguous slices (records are
    independent; for chromosome-sorted input this is sharding by chromosome with band splits at the cuts)."""
    lo = min(n_rows, (n_rows * rank // world + align - 1) // align * align)
    hi = n_rows if rank == world - 1 else min(n_rows, (n_rows * (rank + 1) // world + align - 1) // align * align)
    return lo, hi


def layout_rows(sizes):
    """Rank-local row layout of shards held back to back: (starts, total rows); every start is a multiple of 4 rows, so
    that every shard's columns stay 16-byte aligned."""
    starts, off = [], 0
    for n in sizes:
        starts.append(off)
        off += (int(n) + 3) & ~3
    return starts, off


class GenomePass(object):
    """One pass over the shards attached to this rank, genome-wide statistics and q-values across the ranks of `group`.

    engine: a PassEngine carrying the tables every rank shares (possible pairs, bias tables) - set_fragments / set_bias
    must have been called with the WHOLE genome's fragments / biases on every rank.
    """

    def __init__(self, engine, group=None, q_values=True, gather_capacity=1 << 17):
        self.eng = engine
        self.lib = engine.lib
        self.device = engine.device
        self.world, self.rank = _world(group)
        self.group = None if group is False else group
        self.q_values = bool(q_values)
        self.gather_cap = int(gather_capacity)
        R = engine.R
        # the streaming K4 needs every in-range distance (and distance + R) to fit 31 bits; otherwise the direct kernel runs
        self.listed = 0 <= engine.min_dist <= engine.max_dist and engine.max_dist + R < (1 << 31) and R >= 2
        self._range_ok = self.listed
        self.shards = []
        self.offsets = []
        self.rows = 0
        self.p = self.q = None
        dev = self.device
        self.score_state = torch.zeros(ctypes.sizeof(_lib.ScoreState), dtype=torch.uint8, device=dev)
        self.bh_state = torch.zeros(4, dtype=torch.int64, device=dev)
        self.q_ones = torch.zeros(2, dtype=torch.float64, device=dev)
        self.gather_overflow = torch.zeros(1, dtype=torch.int32, device=dev)
        self.force_exact = False        # tests: raise BbkScoreState.exact whatever the guard says
        self._host = torch.zeros(engine.fit_result.numel() + self.score_state.numel() + 8, dtype=torch.uint8).pin_memory()
        self.n_tests = -1

    # ------------------------------------------------------------------ buffers
    def attach(self, shards, p=None, q=None, list_capacity=None, cand_capacity=None):
        """Shards of this rank (engine.Shard).  Row r of shard i is row offsets[i] + r of the rank-local p / q buffers
        (offsets are multiples of 4; the few padding rows in between hold NaN).  p / q: optional caller buffers of
        at least `rows` float64 (16-byte aligned)."""
        dev = self.device
        self.shards = list(shards)
        self.offsets, self.rows = layout_rows([sh.n for sh in self.shards])
        if self.rows >= (1 << 32):
            raise ValueError("more than 2^32 records on one rank")
        m = max(self.rows, 4)
        self.p = p if p is not None else torch.empty(m, dtype=torch.float64, device=dev)
        self.q = (q if q is not None else torch.empty(m, dtype=torch.float64, device=dev)) if self.q_values else None
        for sh, o in zip(self.shards, self.offsets):
            if sh.n & 3:
                self.p[o + sh.n:o + ((sh.n + 3) & ~3)] = float("nan")
                if self.q is not None:
                    self.q[o + sh.n:o + ((sh.n + 3) & ~3)] = float("nan")
        # shards with chromosome columns (mixed rows) go through the direct kernel
        mixed = any(sh.chr1 is not None for sh in self.shards)
        if mixed and self.world > 1:
            raise ValueError("multi-GPU passes take one-chromosome shards (no chromosome columns)")
        self.listed = self._range_ok and not mixed and not (self.eng.bias is not None and self.eng.bias.step == 1)
        if self.listed:
            # rows the streaming pass defers (large counts, significant rows): a few per cent; an overflow repeats the pass
            cap = int(list_capacity) if list_capacity else min(m, max(1 << 20, m // 4))
            have = getattr(self, "deferred", None)
            if have is None or have.capacity < cap or list_capacity:
                self.l_row = torch.empty(cap, dtype=torch.int32, device=dev)
                self.l_cnt = torch.empty(cap, dtype=torch.int32, device=dev)
                self.l_prior = torch.empty(cap, dtype=torch.float64, device=dev)
                self.deferred = _lib.DeferredList(self.l_row.data_ptr(), self.l_cnt.data_ptr(), self.l_prior.data_ptr(), cap)
            ccap = int(cand_capacity) if cand_capacity else min(m, max(1 << 20, m // 16))
            if getattr(self, "cands", None) is None or self.cands.capacity < ccap or cand_capacity:
                self.c_keys = torch.empty(ccap, dtype=torch.int64, device=dev)
                self.c_rows = torch.empty(ccap, dtype=torch.int32, device=dev)
                self.cands = _lib.Candidates(self.c_keys.data_ptr(), self.c_rows.data_ptr(), ccap)
        if self.q_values:
            if self.world == 1:
                need = int(self.lib.bbk_bh_workspace_bytes(m))
                if getattr(self, "bh_ws", None) is None or self.bh_ws.numel() < need:
                    self.bh_ws = torch.empty(need, dtype=torch.uint8, device=dev)
            elif getattr(self, "sel_ws", None) is None:
                self.sel_ws = torch.empty(int(self.lib.bbk_bh_workspace_bytes(0)), dtype=torch.uint8, device=dev)
                self._alloc_gather()
        return self

    def _alloc_gather(self):
        dev, cap = self.device, self.gather_cap
        self.send = torch.zeros(cap + 1, dtype=torch.int64, device=dev)
        self.send_idx = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
        self.recv = torch.empty(self.world * (cap + 1), dtype=torch.int64, device=dev)
        self.gat_ws = torch.empty(int(self.lib.bbk_bh_gathered_workspace_bytes(self.world, cap)), dtype=torch.uint8, device=dev)

    def shard_p(self, i):
        return self.p[self.offsets[i]:self.offsets[i] + self.shards[i].n]

    def shard_q(self, i):
        return self.q[self.offsets[i]:self.offsets[i] + self.shards[i].n]

    # ------------------------------------------------------------------ the pass
    def _score(self, st, want_q=True):
        """K4: the guard, one streaming pass per shard, the patch pass over the deferred rows."""
        eng, lib = self.eng, self.lib
        bias = ctypes.byref(eng.bias.struct) if eng.bias is not None else None
        flags = _lib.ptr(eng.bias.flags) if eng.bias is not None else None
        hist = _lib.ptr(eng.p_hist) if want_q else None
        cands = ctypes.byref(self.cands) if want_q else None
        q = _lib.ptr(self.q) if want_q else None
        _lib.check(lib.bbk_score_guard(_lib.ptr(eng.fit_result), _lib.ptr(eng.spline_y), _lib.ptr(self.score_state), st), "bbk_score_guard")
        eng.launches += 1
        if self.force_exact:
            self.score_state[24:28] = torch.tensor([1, 0, 0, 0], dtype=torch.uint8, device=self.device)     # BbkScoreState.exact
        live = [(sh, off) for sh, off in zip(self.shards, self.offsets) if sh.n]
        for (sh, off), st_i in zip(live, eng.fan_out(len(live))):
            _lib.check(lib.bbk_score_pairs(_lib.ptr(sh.mid1), _lib.ptr(sh.mid2), _lib.ptr(sh.count), sh.n, sh.chrom, eng.R,
                                           eng.min_dist, eng.max_dist, _lib.ptr(eng.fit_result), _lib.ptr(eng.spline_y), bias, flags,
                                           off, _lib.ptr(self.p), q, hist, cands, ctypes.byref(self.deferred),
                                           _lib.ptr(self.score_state), st_i), "bbk_score_pairs")
            eng.launches += 1
        eng.fan_in()
        _lib.check(lib.bbk_score_deferred(ctypes.byref(self.deferred), _lib.ptr(eng.fit_result), _lib.ptr(self.p), q, hist, cands,
                                          _lib.ptr(self.score_state), st), "bbk_score_deferred")
        eng.launches += 1

    def enqueue(self, n_tests=-1, smoothing=None, marks=None, exclude=None):
        """Enqueue the whole pass on the current stream; no host synchronisation.
        marks (optional dict): filled with CUDA events at the stage boundaries (name -> event recorded AFTER that stage),
        for per-stage timing.
        exclude (optional): (p_first, p_outlier) - the refit pass of BASELINE config 4: the statistics (K1) skip the records
        whose first-pass p (p_first: a buffer laid out like this pass' p) is <= p_outlier, then EVERY record is scored with
        the refitted S and spline (definition in include/bbk.h, bbk_hist_pairs_excluding)."""
        import torch.distributed as dist
        eng, lib = self.eng, self.lib
        main = torch.cuda.current_stream(self.device)
        st = _lib.stream_ptr(main)

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(main)
                marks[name] = ev

        self.n_tests = int(n_tests)
        self._smoothing = smoothing
        want_q = self.q_values
        mark("start")
        if self.listed:
            _lib.check(lib.bbk_score_begin(_lib.ptr(self.score_state), _lib.ptr(eng.p_hist) if want_q else None, st), "bbk_score_begin")
            eng.launches += 1
        elif want_q:
            eng.p_hist.zero_()
            eng.launches += 1
        if exclude is not None:
            p_first, p_outlier = exclude
            eng.hist_excluding(self.shards, [p_first[o:o + sh.n] for sh, o in zip(self.shards, self.offsets)], p_outlier)
        else:
            eng.hist(self.shards)
        self._exclude = exclude
        mark("hist")
        if self.world > 1:
            eng.allreduce_stats(self.group)
        mark("allreduce")
        eng.fit(smoothing)
        mark("fit")
        if self.listed:
            self._score(st, want_q)
        else:
            for i, sh in enumerate(self.shards):
                if sh.n:
                    eng.pvalues(sh, self.shard_p(i), with_hist=want_q)
        mark("pvalues")
        if want_q and not (self.rows == 0 and self.world == 1):
            self._qvalues(st)
        mark("bh")

    def _qvalues(self, st):
        import torch.distributed as dist
        eng, lib = self.eng, self.lib
        m = self.rows
        if self.world == 1:
            if self.listed:
                _lib.check(lib.bbk_bh_qvalues_listed(_lib.ptr(self.p), m, self.n_tests, _lib.ptr(eng.p_hist), _lib.ptr(self.q),
                                                     ctypes.byref(self.cands), _lib.ptr(self.score_state), _lib.ptr(self.bh_ws),
                                                     self.bh_ws.numel(), st), "bbk_bh_qvalues_listed")
                eng.launches += 6          # init, threshold, candidate filter, compact (returns at once), rank, ones fix
            else:
                _lib.check(lib.bbk_bh_qvalues(_lib.ptr(self.p), m, self.n_tests, _lib.BH_UNSORTED, _lib.ptr(eng.p_hist), _lib.ptr(self.q),
                                              None, _lib.ptr(self.bh_ws), self.bh_ws.numel(), st), "bbk_bh_qvalues")
                eng.launches += 5          # init, threshold, compact, rank (one cooperative launch), ones fix
            return
        # genome-wide: global histogram -> common saturation bucket -> candidates below it -> one fixed-capacity all-gather
        dist.all_reduce(eng.p_hist, op=dist.ReduceOp.SUM, group=self.group)
        cap = self.gather_cap
        keys = ctypes.c_void_p(self.send.data_ptr() + 8)
        if self.listed:
            _lib.check(lib.bbk_bh_select_listed(_lib.ptr(self.p), m, self.n_tests, _lib.ptr(eng.p_hist), _lib.ptr(self.q),
                                                ctypes.byref(self.cands), _lib.ptr(self.score_state), keys, _lib.ptr(self.send_idx), cap,
                                                _lib.ptr(self.bh_state), _lib.ptr(self.sel_ws), self.sel_ws.numel(), st), "bbk_bh_select_listed")
        else:
            _lib.check(lib.bbk_bh_select(_lib.ptr(self.p), m, self.n_tests, _lib.ptr(eng.p_hist), _lib.ptr(self.q), keys,
                                         _lib.ptr(self.send_idx), cap, _lib.ptr(self.bh_state), _lib.ptr(self.sel_ws), self.sel_ws.numel(),
                                         st), "bbk_bh_select")
        _lib.check(lib.bbk_bh_pack_count(_lib.ptr(self.bh_state), _lib.ptr(self.send), st), "bbk_bh_pack_count")
        dist.all_gather_into_tensor(self.recv, self.send, group=self.group)
        _lib.check(lib.bbk_bh_rank_gathered_padded(_lib.ptr(self.recv), self.world, cap, self.rank, _lib.ptr(self.bh_state),
                                                   _lib.ptr(self.send_idx), _lib.ptr(self.q), _lib.ptr(self.q_ones),
                                                   _lib.ptr(self.gather_overflow), _lib.ptr(self.gat_ws), self.gat_ws.numel(), st),
                   "bbk_bh_rank_gathered_padded")
        _lib.check(lib.bbk_bh_fix_ones_dev(_lib.ptr(self.p), m, _lib.ptr(self.q_ones), _lib.ptr(self.q), st), "bbk_bh_fix_ones_dev")
        # init, threshold, [candidate filter], compact, export, pack | prepare, compact, rank, export, scatter | ones fix
        eng.launches += 12 if self.listed else 11

    def read_state(self):
        """(FitResult bytes, ScoreState, gather overflow) after ONE synchronisation."""
        nf, ns = self.eng.fit_result.numel(), self.score_state.numel()
        self._host[:nf].copy_(self.eng.fit_result, non_blocking=True)
        self._host[nf:nf + ns].copy_(self.score_state, non_blocking=True)
        self._host[nf + ns:nf + ns + 4].copy_(self.gather_overflow.view(torch.uint8), non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        raw = self._host.numpy().tobytes()
        score = _lib.ScoreState.from_buffer_copy(raw[nf:nf + ns])
        ov = int(np.frombuffer(raw[nf + ns:nf + ns + 4], dtype=np.int32)[0])
        return raw[:nf], score, ov

    def finish(self):
        """Wait for the pass and make it final: raises what the reference would raise for a failed fit; repeats the pass
        when the reference's own smoothing factor differs from the kernel's (engine.reference_smoothing), when the work
        list was too small, or when the candidate all-gather overflowed its capacity (grown for the next passes too).
        Returns the FitResult."""
        import torch.distributed as dist
        for _ in range(6):
            raw, score, ov = self.read_state()
            if _lib.FitResult.from_buffer_copy(raw).status == _lib.FIT_TOO_MANY_BINS and self.eng.grow_bins():
                self.enqueue(self.n_tests, smoothing=self._smoothing, exclude=getattr(self, "_exclude", None))      # more bins than the default buffers hold: one per key
                continue
            fit = PassEngine.decode_fit(raw)
            again = False
            s_ref = PassEngine.reference_smoothing(fit)          # None once the pass ran with the reference's own s
            if s_ref is not None:
                self._smoothing, again = s_ref, True
            if self.listed and score.overflow:
                self.attach(self.shards, self.p, self.q, list_capacity=max(self.rows, 4))
                again = True
            if self.world > 1 and self.q_values:
                flags = torch.tensor([ov, 1 if again else 0, self.rows], dtype=torch.int64, device=self.device)
                dist.all_reduce(flags, op=dist.ReduceOp.MAX, group=self.group)
                ov_any, again, max_rows = int(flags[0].item()), bool(int(flags[1].item())), int(flags[2].item())
                if ov_any:
                    # ov_any = the largest candidate count of any rank: the next power of two with a quarter of headroom (the
                    # all-gather moves the whole capacity, so it should fit, not dwarf, what is sent)
                    need = max(int(ov_any * 1.25), 2 * self.gather_cap)
                    self.gather_cap = max(4, min(1 << (need - 1).bit_length(), max_rows))
                    self.gather_overflow.zero_()
                    self._alloc_gather()
                    again = True
            if not again:
                self.last_score = score
                return fit
            self.enqueue(self.n_tests, smoothing=self._smoothing, exclude=getattr(self, "_exclude", None))
        raise _lib.BbkError("the pass did not settle after 6 attempts")

    def run(self, n_tests=-1, smoothing=None, exclude=None):
        self.enqueue(n_tests, smoothing, exclude=exclude)
        return self.finish()


class ChromosomePass(object):
    """Fit-Hi-C once per chromosome, every chromosome in one pass on this GPU: the authors' workflow (one run per chromosome,
    datatypes.pyx:26) without one fit launch, one q-value step and one host synchronisation per chromosome.

    engines[i]: the PassEngine of chromosome i, set up with that chromosome's fragments only (its own possible pairs, distance
    table, fit buffers and histogram); every engine has the same resolution / n_bins / distance limits and the same bias
    tables (or none).  shards[i]: its records, one compact Shard (chrom = its id).  Chromosome i's result equals a GenomePass
    over engines[i] and shards[i] alone, bit for bit.  Streaming K4 only: the conditions of GenomePass.listed must hold.

        per chromosome (three streams): K1              ->  ONE bbk_fit_batched
        ->  per chromosome (three streams): guard, streaming K4, patch pass  ->  ONE bbk_bh_qvalues_segmented
    """

    def __init__(self, engines, shards, q_values=True, list_capacity=None, cand_capacity=None):
        if len(engines) != len(shards) or not engines:
            raise ValueError("one engine per shard, at least one")
        self.engs, self.shards = list(engines), list(shards)
        e0 = self.engs[0]
        self.lib, self.device = e0.lib, e0.device
        for e in self.engs:
            if (e.R, e.n_bins, e.min_dist, e.max_dist, e.bias) != (e0.R, e0.n_bins, e0.min_dist, e0.max_dist, e0.bias):
                raise ValueError("every chromosome's engine needs the same resolution, n_bins, distance limits and bias tables")
        if not (0 <= e0.min_dist <= e0.max_dist and e0.max_dist + e0.R < (1 << 31) and e0.R >= 2) or \
                (e0.bias is not None and e0.bias.step == 1):
            raise ValueError("ChromosomePass runs the streaming K4 only (GenomePass.listed)")
        if any(sh.chr1 is not None for sh in self.shards):
            raise ValueError("ChromosomePass takes one-chromosome shards (no chromosome columns)")
        self.q_values = bool(q_values)
        n = len(self.engs)
        dev = self.device
        self.offsets, self.rows = layout_rows([sh.n for sh in self.shards])
        if self.rows >= (1 << 32):
            raise ValueError("more than 2^32 records on one GPU")
        m = max(self.rows, 4)
        self.p = torch.full((m,), float("nan"), dtype=torch.float64, device=dev)
        self.q = torch.full((m,), float("nan"), dtype=torch.float64, device=dev) if self.q_values else None
        ns = ctypes.sizeof(_lib.ScoreState)
        self.score_state = torch.zeros(n * ns, dtype=torch.uint8, device=dev)
        self.p_hist = torch.zeros(n * _lib.PHIST_LEN, dtype=torch.int64, device=dev)
        self.lists = [None] * n
        self.cands = [None] * n
        for i, sh in enumerate(self.shards):
            mi = max((sh.n + 3) & ~3, 4)
            self._alloc_list(i, int(list_capacity) if list_capacity else min(mi, max(1 << 20, mi // 4)))
            if self.q_values:
                cc = int(cand_capacity) if cand_capacity else min(mi, max(1 << 20, mi // 16))
                keys = torch.empty(cc, dtype=torch.int64, device=dev)
                rows = torch.empty(cc, dtype=torch.int32, device=dev)
                self.cands[i] = (keys, rows, _lib.Candidates(keys.data_ptr(), rows.data_ptr(), cc))
        if self.q_values:
            self.seg_off = torch.tensor(self.offsets + [self.rows], dtype=torch.int64, device=dev)
            segs = (_lib.BhSegment * n)()
            for i in range(n):
                segs[i].d_p_hist = self.p_hist[i * _lib.PHIST_LEN:].data_ptr()
                segs[i].d_state = self.score_state[i * ns:].data_ptr()
                segs[i].cands = self.cands[i][2]
                segs[i].n_tests = -1
            self._segs_host = segs
            self.segs = torch.zeros(ctypes.sizeof(segs), dtype=torch.uint8, device=dev)
            self.bh_ws = torch.empty(int(self.lib.bbk_bh_segmented_workspace_bytes(m, n)), dtype=torch.uint8, device=dev)
            self.n_tests = None
        self.problems = torch.zeros(n * ctypes.sizeof(_lib.FitProblem), dtype=torch.uint8, device=dev)
        self._set_problems()
        self.smoothing = [None] * n
        nf = e0.fit_result.numel()
        self._host = torch.zeros(n * (nf + ns), dtype=torch.uint8).pin_memory()
        self._sides = [torch.cuda.Stream(dev) for _ in range(2)]
        self._ev = [torch.cuda.Event() for _ in range(3)]
        self.launches = 0

    def _alloc_list(self, i, cap):
        dev = self.device
        row = torch.empty(cap, dtype=torch.int32, device=dev)
        cnt = torch.empty(cap, dtype=torch.int32, device=dev)
        prior = torch.empty(cap, dtype=torch.float64, device=dev)
        self.lists[i] = (row, cnt, prior, _lib.DeferredList(row.data_ptr(), cnt.data_ptr(), prior.data_ptr(), cap))

    def _set_problems(self):
        """The device array of fit descriptors (again after grow_bins has replaced an engine's buffers)."""
        probs = (_lib.FitProblem * len(self.engs))()
        for pr, e in zip(probs, self.engs):
            pr.d_possible, pr.d_obs_sum, pr.d_totals = e.possible.data_ptr(), e.obs_sum.data_ptr(), e.totals.data_ptr()
            pr.d_result, pr.d_x, pr.d_y, pr.d_bin_of_key = e.fit_result.data_ptr(), e.x.data_ptr(), e.y.data_ptr(), e.bin_of_key.data_ptr()
            pr.d_spline_y, pr.d_spline_raw = e.spline_y.data_ptr(), e.spline_raw.data_ptr()
            pr.d_knots, pr.d_coefs = e.knots.data_ptr(), e.coefs.data_ptr()
            pr.d_workspace, pr.workspace_bytes = e.fit_ws.data_ptr(), e.fit_ws.numel()
            pr.nkeys, pr.max_bins = e.nkeys, e.max_bins
        self.problems.copy_(torch.frombuffer(bytearray(bytes(probs)), dtype=torch.uint8))

    def chrom_p(self, i):
        return self.p[self.offsets[i]:self.offsets[i] + self.shards[i].n]

    def chrom_q(self, i):
        return self.q[self.offsets[i]:self.offsets[i] + self.shards[i].n]

    def _lanes(self, main):
        """Stream pointers of three lanes (main and two side streams that start after what main holds so far)."""
        self._ev[0].record(main)
        for sd in self._sides:
            sd.wait_event(self._ev[0])
        return [_lib.stream_ptr(x) for x in [main] + self._sides]

    def _join(self, main):
        for sd, ev in zip(self._sides, self._ev[1:]):
            ev.record(sd)
            main.wait_event(ev)

    def enqueue(self, n_tests=None, marks=None):
        """Enqueue the whole pass on the current stream; no host synchronisation.  n_tests: None (every chromosome's N is its
        number of emitted rows) or one value per chromosome (-1 = that default).  marks: as GenomePass.enqueue."""
        lib, R = self.lib, self.engs[0]
        main = torch.cuda.current_stream(self.device)
        st = _lib.stream_ptr(main)
        ns = ctypes.sizeof(_lib.ScoreState)

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(main)
                marks[name] = ev

        want_q = self.q_values
        if want_q:
            nt = [-1] * len(self.engs) if n_tests is None else [int(x) for x in n_tests]
            if nt != self.n_tests:
                for i, v in enumerate(nt):
                    self._segs_host[i].n_tests = v
                self.segs.copy_(torch.frombuffer(bytearray(bytes(self._segs_host)), dtype=torch.uint8))
                self.n_tests = nt
        mark("start")
        self.score_state.zero_()
        self.launches += 1
        if want_q:
            self.p_hist.zero_()
            self.launches += 1
        lanes = self._lanes(main)
        for i, (e, sh) in enumerate(zip(self.engs, self.shards)):
            li = lanes[i % 3]
            _lib.check(lib.bbk_hist_init(_lib.ptr(e.obs_sum), e.nkeys, _lib.ptr(e.totals), li), "bbk_hist_init")
            _lib.check(lib.bbk_hist_pairs(None, None, _lib.ptr(sh.mid1), _lib.ptr(sh.mid2), _lib.ptr(sh.count), sh.n, e.R, e.min_dist,
                                          e.max_dist, e.nkeys, _lib.ptr(e.obs_sum), _lib.ptr(e.totals), li), "bbk_hist_pairs")
            self.launches += 2
        self._join(main)
        mark("hist")
        for i, e in enumerate(self.engs):
            if self.smoothing[i] is not None:         # this chromosome gets the reference's own s (PassEngine.reference_smoothing)
                req = _lib.FitResult()
                req.status = _lib.FIT_S_GIVEN
                req.smoothing = float(self.smoothing[i])
                e.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8))
        _lib.check(lib.bbk_fit_batched(_lib.ptr(self.problems), len(self.engs), R.n_bins, R.R, R.min_dist, R.max_dist, st),
                   "bbk_fit_batched")
        self.launches += 1
        mark("fit")
        lanes = self._lanes(main)
        for i, (e, sh) in enumerate(zip(self.engs, self.shards)):
            li = lanes[i % 3]
            state = ctypes.c_void_p(self.score_state.data_ptr() + i * ns)
            hist = ctypes.c_void_p(self.p_hist.data_ptr() + i * 8 * _lib.PHIST_LEN) if want_q else None
            cands = ctypes.byref(self.cands[i][2]) if want_q else None
            q = _lib.ptr(self.q) if want_q else None
            bias = ctypes.byref(e.bias.struct) if e.bias is not None else None
            flags = _lib.ptr(e.bias.flags) if e.bias is not None else None
            deferred = ctypes.byref(self.lists[i][3])
            _lib.check(lib.bbk_score_guard(_lib.ptr(e.fit_result), _lib.ptr(e.spline_y), state, li), "bbk_score_guard")
            self.launches += 1
            if sh.n:
                _lib.check(lib.bbk_score_pairs(_lib.ptr(sh.mid1), _lib.ptr(sh.mid2), _lib.ptr(sh.count), sh.n, sh.chrom, e.R, e.min_dist,
                                               e.max_dist, _lib.ptr(e.fit_result), _lib.ptr(e.spline_y), bias, flags, self.offsets[i],
                                               _lib.ptr(self.p), q, hist, cands, deferred, state, li), "bbk_score_pairs")
                self.launches += 1
            _lib.check(lib.bbk_score_deferred(deferred, _lib.ptr(e.fit_result), _lib.ptr(self.p), q, hist, cands, state, li),
                       "bbk_score_deferred")
            self.launches += 1
        self._join(main)
        mark("pvalues")
        if want_q and self.rows:
            _lib.check(lib.bbk_bh_qvalues_segmented(_lib.ptr(self.p), self.rows, _lib.ptr(self.seg_off), _lib.ptr(self.segs),
                                                    len(self.engs), _lib.ptr(self.q), _lib.ptr(self.bh_ws), self.bh_ws.numel(), st),
                       "bbk_bh_qvalues_segmented")
            self.launches += 5          # threshold, candidate filter, pass over p (returns at once), rank, ones fix
        mark("bh")

    def read_state(self):
        """[(FitResult bytes, ScoreState)] of every chromosome after ONE synchronisation."""
        nf, ns, n = self.engs[0].fit_result.numel(), ctypes.sizeof(_lib.ScoreState), len(self.engs)
        for i, e in enumerate(self.engs):
            self._host[i * nf:(i + 1) * nf].copy_(e.fit_result, non_blocking=True)
        self._host[n * nf:].copy_(self.score_state, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        raw = self._host.numpy().tobytes()
        return [(raw[i * nf:(i + 1) * nf], _lib.ScoreState.from_buffer_copy(raw[n * nf + i * ns:n * nf + (i + 1) * ns]))
                for i in range(n)]

    def finish(self):
        """Wait for the pass and make it final, chromosome by chromosome as GenomePass.finish does: a chromosome with more bins
        than its buffers hold gets room for one per key, one whose s is not the reference's own gets that s, one whose deferred
        list overflowed gets a list as long as its rows, and the pass repeats (at most 6 times; the other chromosomes come out
        the same, every stage being deterministic).  A failed fit raises what the reference would raise for that chromosome
        alone, naming it; chromosomes are checked in ascending order.  Returns the FitResults."""
        for _ in range(6):
            state = self.read_state()
            grown = [i for i, (raw, _) in enumerate(state)
                     if _lib.FitResult.from_buffer_copy(raw).status == _lib.FIT_TOO_MANY_BINS and self.engs[i].grow_bins()]
            if grown:
                self._set_problems()
                self.enqueue(self.n_tests if self.q_values else None)
                continue
            fits, again = [], False
            for i in sorted(range(len(self.engs)), key=lambda j: self.shards[j].chrom):
                raw, score = state[i]
                try:
                    fit = PassEngine.decode_fit(raw)
                except Exception as e:
                    from .fithic import naming_chromosome
                    raise naming_chromosome(e, self.shards[i].chrom)
                s_ref = PassEngine.reference_smoothing(fit)
                if s_ref is not None:
                    self.smoothing[i], again = s_ref, True
                if score.overflow:
                    self._alloc_list(i, max((self.shards[i].n + 3) & ~3, 4))
                    again = True
            if not again:
                self.last_state = state
                return [PassEngine.decode_fit(raw) for raw, _ in state]
            self.enqueue(self.n_tests if self.q_values else None)
        raise _lib.BbkError("the per-chromosome pass did not settle after 6 attempts")

    def run(self, n_tests=None):
        self.enqueue(n_tests)
        return self.finish()


class HostStream(object):
    """Successive passes streamed from pinned host memory through one GenomePass (the end-to-end call of this rank).

    A pass cannot start scoring before all of its records are on the device (S and the spline need the whole distance
    table, fithic.py:110-133), so inside one pass the inbound and the outbound copies never overlap; across passes they do:
    `slots` device copies of the record columns and of p / q, three streams (in, run, out) and per-slot events.  The host
    table is three contiguous pinned int32 columns holding this rank's shards back to back (shard i = rows
    starts[i] .. starts[i] + sizes[i], starts = layout_rows(sizes): every start a multiple of 4); p / q come back as pinned
    float64 columns over the same rows.  Nothing here synchronises the host: call drain() (or wait on the event submit() returns) before reading."""

    class _Slot(object):
        pass

    def __init__(self, genome_pass, sizes, chroms, slots=2, packed=False, cap_p=None, cap_q=None):
        """sizes / chroms: records and chromosome of every shard; the slots hold layout_rows(sizes) rows.
        packed: results cross the host link as two bits per row + the values that are not 1.0 / NaN (bbk_pack_scores);
        submit_packed() returns a PackedScores whose dense() rebuilds the float64 columns bit for bit.  cap_p / cap_q: rows
        the packed value lists can hold (default rows / 2 and rows / 16; a pass that needs more comes back dense)."""
        self.gp = genome_pass
        self.sizes, self.chroms = [int(x) for x in sizes], [int(x) for x in chroms]
        self.starts, rows = layout_rows(self.sizes)
        self.rows = max(rows, 4)
        self.packed = bool(packed)
        dev = genome_pass.device
        self.slots = []
        for _ in range(int(slots)):
            s = HostStream._Slot()
            s.mid1, s.mid2, s.count = (torch.empty(self.rows, dtype=torch.int32, device=dev) for _ in range(3))
            s.p = torch.full((self.rows,), float("nan"), dtype=torch.float64, device=dev)
            s.q = torch.full((self.rows,), float("nan"), dtype=torch.float64, device=dev) if genome_pass.q_values else None
            s.shards = self._shards(s, self.starts, self.sizes)
            s.in_ready, s.run_done, s.out_done, s.counts_ready = (torch.cuda.Event() for _ in range(4))
            s.fit = torch.zeros_like(genome_pass.eng.fit_result)
            s.h_fit = torch.zeros(genome_pass.eng.fit_result.numel(), dtype=torch.uint8).pin_memory()
            if self.packed:
                s.pack = DevicePack(self.rows, dev, genome_pass.q_values, cap_p, cap_q)
                s.h_pack_state = torch.zeros(ctypes.sizeof(_lib.PackState), dtype=torch.uint8).pin_memory()
            s.index = -1
            self.slots.append(s)
        # Nothing here synchronises, so nothing would see BbkScoreState.overflow: the deferred list has a place for every row
        # of a slot (and later attaches keep it, being no larger).
        genome_pass.attach(s.shards, s.p, s.q, list_capacity=self.rows)
        self.s_in, self.s_run, self.s_out = (torch.cuda.Stream(dev) for _ in range(3))
        self.s_run.wait_stream(torch.cuda.current_stream(dev))
        self.submitted = 0
        self._pending = None

    def _shards(self, s, starts, sizes):
        return [Shard(s.mid1[a:a + n], s.mid2[a:a + n], s.count[a:a + n], chrom=c) for a, n, c in zip(starts, sizes, self.chroms)]

    def _run(self, h_mid1, h_mid2, h_count, h_out, n_tests, sizes, q_values, pack=False):
        """What submit() and submit_packed() share: check the host columns, copy the records into the next slot (stream in)
        and run the pass there (stream run), packing p / q after it when `pack`.  Returns (slot, rows the pass covers)."""
        s = self.slots[self.submitted % len(self.slots)]
        sizes = self.sizes if sizes is None else [int(x) for x in sizes]
        starts, rows = layout_rows(sizes)
        if len(sizes) != len(self.chroms) or rows > self.rows:
            raise ValueError("sizes must give one shard per chromosome of the stream and fit its %d rows" % self.rows)
        n = starts[-1] + sizes[-1] if sizes else 0
        for t in (h_mid1, h_mid2, h_count) + h_out:
            if t is not None and (not t.is_pinned() or t.numel() < n):
                raise ValueError("host columns must be pinned and hold at least %d rows" % n)
        if q_values and s.q is None:
            raise ValueError("the stream's GenomePass was made with q_values=False")
        shards = s.shards if sizes is self.sizes else self._shards(s, starts, sizes)
        self.submitted += 1
        s.index = self.submitted - 1
        self.s_in.wait_event(s.run_done)        # the pass that last read this slot's records has finished
        with torch.cuda.stream(self.s_in):
            s.mid1[:n].copy_(h_mid1[:n], non_blocking=True)
            s.mid2[:n].copy_(h_mid2[:n], non_blocking=True)
            s.count[:n].copy_(h_count[:n], non_blocking=True)
            s.in_ready.record()
        # the previous packed pass' value lists: their sizes are on the host by now (or soon); their copies overlap these inbound ones
        self._finalize_pending()
        self.s_run.wait_event(s.in_ready)
        self.s_run.wait_event(s.out_done)       # this slot's previous p / q have left the device
        gp = self.gp
        with torch.cuda.stream(self.s_run):
            keep_q, gp.q_values = gp.q_values, q_values
            gp.attach(shards, s.p, s.q)
            gp.enqueue(n_tests)
            gp.q_values = keep_q
            s.fit.copy_(gp.eng.fit_result, non_blocking=True)
            if pack:
                s.pack.pack(s.p, s.q, self.s_run)
                gp.eng.launches += 2
            s.run_done.record()
        return s, n

    def submit(self, h_mid1, h_mid2, h_count, h_p, h_q=None, n_tests=-1, sizes=None):
        """Enqueue one pass over the host table; returns the event that fires when p (and q) are on the host.
        sizes: this pass' shard sizes, one per chromosome of the stream (default: the sizes it was made with); their
        layout_rows total must fit the slots.  The host columns hold at least the rows the pass covers (up to the end of its
        last shard), and exactly those rows come back.  Without h_q the pass skips the q-value step; at N > 1 that step is
        collective, so every rank must pass or omit h_q alike."""
        s, n = self._run(h_mid1, h_mid2, h_count, (h_p, h_q), n_tests, sizes, h_q is not None)
        self.s_out.wait_event(s.run_done)
        with torch.cuda.stream(self.s_out):
            h_p[:n].copy_(s.p[:n], non_blocking=True)
            if h_q is not None:
                h_q[:n].copy_(s.q[:n], non_blocking=True)
            s.h_fit.copy_(s.fit, non_blocking=True)
            s.out_done.record()
        return s.out_done

    # ------------------------------------------------------------------ packed results
    def submit_packed(self, h_mid1, h_mid2, h_count, out, n_tests=-1):
        """Like submit(), but p / q come back packed into `out` (a PackedScores made by packed_buffers()).  The sizes of the two
        value lists are only known once the pass has run, so their copies are issued lazily: by the NEXT submission (after
        it has put its own inbound copies on the wire) or by drain().  Returns `out`; out.done fires when it is complete."""
        if not self.packed:
            raise ValueError("this stream was not created with packed=True")
        s, _ = self._run(h_mid1, h_mid2, h_count, (), n_tests, None, self.gp.q_values, pack=True)
        self.s_out.wait_event(s.run_done)
        with torch.cuda.stream(self.s_out):
            s.h_pack_state.copy_(s.pack.state, non_blocking=True)
            s.counts_ready.record()
            out.codes.copy_(s.pack.codes, non_blocking=True)
            out.chunks.copy_(s.pack.chunks, non_blocking=True)
            s.h_fit.copy_(s.fit, non_blocking=True)
        out.rows, out.want_q = self.rows, s.q is not None
        out.done = None
        self._pending = (s, out)
        return out

    def _finalize_pending(self):
        if self._pending is None:
            return
        s, out = self._pending
        self._pending = None
        s.counts_ready.synchronize()
        st = _lib.PackState.from_buffer_copy(s.h_pack_state.numpy().tobytes())
        out.n_p, out.n_q, out.overflow = int(st.n_p), int(st.n_q), bool(st.overflow)
        with torch.cuda.stream(self.s_out):
            if out.overflow:                                     # more values than the lists hold: this pass comes back dense
                out.dense_p = torch.empty(self.rows, dtype=torch.float64).pin_memory()
                out.dense_p.copy_(s.p, non_blocking=True)
                if s.q is not None:
                    out.dense_q = torch.empty(self.rows, dtype=torch.float64).pin_memory()
                    out.dense_q.copy_(s.q, non_blocking=True)
            else:
                if out.n_p:
                    out.vals_p[:out.n_p].copy_(s.pack.vals_p[:out.n_p], non_blocking=True)
                if out.n_q and s.pack.vals_q is not None:
                    out.vals_q[:out.n_q].copy_(s.pack.vals_q[:out.n_q], non_blocking=True)
            s.out_done.record()
        out.done = s.out_done

    def packed_buffers(self):
        """Pinned host buffers for one packed result."""
        pk = self.slots[0].pack
        return PackedScores(self.rows, pk.codes.numel(), pk.chunks.numel() // 24, pk.cap_p, pk.cap_q)

    def fit_of(self, index):
        """Fit result of submission `index` once its outputs are on the host (raises the reference's exception for a failed
        fit); PassEngine.reference_smoothing(result) tells whether that pass must be repeated with the reference's own s.
        Only the last `slots` submissions are held."""
        s = self.slots[int(index) % len(self.slots)]
        if s.index != int(index):
            raise KeyError("submission %d is no longer (or not yet) held by the stream" % int(index))
        s.out_done.synchronize()
        return PassEngine.decode_fit(s.h_fit.numpy().tobytes())

    def drain(self):
        self._finalize_pending()
        self.s_out.synchronize()


class DevicePack(object):
    """Device buffers of one pass' p / q columns in the form that crosses the host link (bbk_pack_scores): the code words,
    the chunk table, the p and q value lists and the pack state.  cap_p / cap_q: values the lists hold (default rows / 2 and
    rows / 16, at least 1024); a pass with more raises PackState.overflow, and the caller decides what comes back instead."""

    def __init__(self, rows, device, want_q, cap_p=None, cap_q=None):
        self.lib = _lib.load()
        self.rows = int(rows)
        self.cap_p = int(cap_p) if cap_p else max(self.rows // 2, 1024)
        self.cap_q = (int(cap_q) if cap_q else max(self.rows // 16, 1024)) if want_q else 0
        self.codes = torch.empty(int(self.lib.bbk_pack_code_words(self.rows)), dtype=torch.int32, device=device)
        self.chunks = torch.empty(int(self.lib.bbk_pack_chunks(self.rows)) * 24, dtype=torch.uint8, device=device)
        self.vals_p = torch.empty(self.cap_p, dtype=torch.float64, device=device)
        self.vals_q = torch.empty(self.cap_q, dtype=torch.float64, device=device) if want_q else None
        self.state = torch.zeros(ctypes.sizeof(_lib.PackState), dtype=torch.uint8, device=device)

    def pack(self, p, q, stream=None):
        """bbk_pack_scores over the first `rows` rows of p and q (None without q-values); two launches on `stream`."""
        _lib.check(self.lib.bbk_pack_scores(_lib.ptr(p), _lib.ptr(q), self.rows, _lib.ptr(self.codes), _lib.ptr(self.chunks),
                                            _lib.ptr(self.vals_p), self.cap_p, _lib.ptr(self.vals_q), self.cap_q, _lib.ptr(self.state),
                                            _lib.stream_ptr(stream)), "bbk_pack_scores")


class PackedScores(object):
    """One pass' p / q columns as they cross the host link (bbk_pack_scores): two bits per row, a chunk table and the values
    that are not 1.0 / NaN, in pinned host memory.  dense() rebuilds the float64 columns bit for bit (libbbkio, all cores)."""

    def __init__(self, rows, n_words, n_chunks, cap_p, cap_q):
        self.rows = int(rows)
        self.codes = torch.empty(n_words, dtype=torch.int32).pin_memory()
        self.chunks = torch.empty(n_chunks * 24, dtype=torch.uint8).pin_memory()
        self.vals_p = torch.empty(max(cap_p, 1), dtype=torch.float64).pin_memory()
        self.vals_q = torch.empty(max(cap_q, 1), dtype=torch.float64).pin_memory() if cap_q else None
        self.n_p = self.n_q = 0
        self.overflow = False
        self.want_q = cap_q > 0
        self.dense_p = self.dense_q = None
        self.done = None

    def nbytes(self):
        """Bytes that crossed the link for this result."""
        if self.overflow:
            return 8 * self.rows * (2 if self.dense_q is not None else 1) + self.codes.numel() * 4 + self.chunks.numel()
        return self.codes.numel() * 4 + self.chunks.numel() + 8 * (self.n_p + self.n_q)

    def dense(self, p_out=None, q_out=None, threads=0):
        """(p, q) as dense numpy float64 columns (q None without q-values)."""
        from . import _io
        if self.done is None:
            raise RuntimeError("the result is not complete yet: call HostStream.drain() (or submit the next pass) first")
        self.done.synchronize()
        if self.overflow:
            return self.dense_p.numpy(), (self.dense_q.numpy() if self.dense_q is not None else None)
        return _io.unpack_scores(self.codes.numpy(), self.chunks.numpy(), self.vals_p.numpy(),
                                 self.vals_q.numpy() if self.vals_q is not None else None, self.rows, p_out, q_out, threads,
                                 want_q=self.want_q)
