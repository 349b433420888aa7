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

from . import _io, _lib
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

    @property
    def launches(self):
        """Kernel launches counted so far (the engine's counter)."""
        return self.eng.launches

    @launches.setter
    def launches(self, n):
        self.eng.launches = n

    def fit_results(self):
        """The device BbkFitResult a pass leaves, as a list of one (HostStream copies it with each pass)."""
        return [self.eng.fit_result]

    def decode_fits(self, raw):
        """fit_results() bytes -> FitResult; raises what the reference would raise for a failed fit."""
        return PassEngine.decode_fit(raw)

    # ------------------------------------------------------------------ buffers
    def check_sizes(self, sizes):
        """Raise ValueError unless shards of these sizes can be attached."""
        if layout_rows(sizes)[1] >= (1 << 32):
            raise ValueError("more than 2^32 records on one rank")

    def attach(self, shards, p=None, q=None, list_capacity=None, cand_capacity=None):
        """Shards of this rank (engine.Shard).  Row r of shard i is row offsets[i] + r of the rank-local p / q buffers
        (offsets are multiples of 4; the few padding rows in between hold NaN).  p / q: optional caller buffers of
        at least `rows` float64 (16-byte aligned)."""
        dev = self.device
        self.shards = list(shards)
        self.check_sizes([sh.n for sh in self.shards])
        self.offsets, self.rows = layout_rows([sh.n for sh in self.shards])
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
        """shards: the most records each chromosome can have; a later attach() may give any chromosome fewer (0 included)."""
        if len(engines) != len(shards) or not engines:
            raise ValueError("one engine per shard, at least one")
        self.engs = list(engines)
        e0 = self.engs[0]
        self.lib, self.device = e0.lib, e0.device
        for e in self.engs:
            if (e.R, e.n_bins, e.min_dist, e.max_dist, e.bias) != (e0.R, e0.n_bins, e0.min_dist, e0.max_dist, e0.bias):
                raise ValueError("every chromosome's engine needs the same resolution, n_bins, distance limits and bias tables")
        if not (0 <= e0.min_dist <= e0.max_dist and e0.max_dist + e0.R < (1 << 31) and e0.R >= 2) or \
                (e0.bias is not None and e0.bias.step == 1):
            raise ValueError("ChromosomePass runs the streaming K4 only (GenomePass.listed)")
        self.q_values = bool(q_values)
        n = len(self.engs)
        dev = self.device
        self.chroms = [sh.chrom for sh in shards]
        self.max_sizes = [sh.n for sh in shards]
        self.check_sizes(self.max_sizes)
        ns = ctypes.sizeof(_lib.ScoreState)
        self.score_state = torch.zeros(n * ns, dtype=torch.uint8, device=dev)
        self.p_hist = torch.zeros(n * _lib.PHIST_LEN, dtype=torch.int64, device=dev)
        self.shards, self.offsets, self.rows = [], [], 0
        self.p = self.q = None
        self.lists = [None] * n
        self.cands = [None] * n
        self.n_tests = None
        if self.q_values:
            self.seg_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            self._seg_layout = None
            self._segs_host = (_lib.BhSegment * n)()
            for i in range(n):
                self._segs_host[i].d_p_hist = self.p_hist[i * _lib.PHIST_LEN:].data_ptr()
                self._segs_host[i].d_state = self.score_state[i * ns:].data_ptr()
            self.segs = torch.zeros(ctypes.sizeof(self._segs_host), dtype=torch.uint8, device=dev)
            self._segs_nt = None                # the n_tests values self.segs holds (None: not uploaded yet)
        self.problems = torch.zeros(n * ctypes.sizeof(_lib.FitProblem), dtype=torch.uint8, device=dev)
        self._set_problems()
        self.smoothing = [None] * n
        nf = e0.fit_result.numel()
        self._host = torch.zeros(n * (nf + ns), dtype=torch.uint8).pin_memory()
        self._sides = [torch.cuda.Stream(dev) for _ in range(2)]
        self._ev = [torch.cuda.Event() for _ in range(3)]
        self.launches = 0
        self.attach(shards, list_capacity=list_capacity, cand_capacity=cand_capacity)

    def check_sizes(self, sizes):
        """Raise ValueError unless shards of these sizes can be attached: one per chromosome, none larger than it was built with."""
        if len(sizes) != len(self.engs):
            raise ValueError("one shard per chromosome of the pass (%d), got %d" % (len(self.engs), len(sizes)))
        for c, n, most in zip(self.chroms, sizes, self.max_sizes):
            if not 0 <= int(n) <= most:
                raise ValueError("chromosome %d: %d rows, more than the %d the pass was built with" % (c, int(n), most))
        if layout_rows(sizes)[1] >= (1 << 32):
            raise ValueError("more than 2^32 records on one GPU")

    def attach(self, shards, p=None, q=None, list_capacity=None, cand_capacity=None):
        """Point the pass at other records (one compact Shard per chromosome, in the order and with the ids it was built with,
        none larger than then) and other p / q buffers of at least `rows` float64 (laid out by layout_rows; the padding rows
        between chromosomes are set to NaN), keeping the engines, the bias tables and the fit and q-value descriptors.
        list_capacity / cand_capacity: given, every chromosome's deferred / candidate list is made anew with that many places
        (at most its built size, which no pass can exceed: such a deferred list cannot overflow); omitted, the lists already
        attached are kept (the first attach makes them at their default sizes, from the built sizes)."""
        shards = list(shards)
        self.check_sizes([sh.n for sh in shards])
        if any(sh.chr1 is not None for sh in shards):
            raise ValueError("ChromosomePass takes one-chromosome shards (no chromosome columns)")
        if [sh.chrom for sh in shards] != self.chroms:
            raise ValueError("the shards' chromosome ids differ from the pass' %s" % self.chroms)
        dev = self.device
        self.shards = shards
        self.offsets, self.rows = layout_rows([sh.n for sh in shards])
        m = max(self.rows, 4)
        for t in (p, q):
            if t is not None and t.numel() < m:
                raise ValueError("p / q buffers need at least %d rows" % m)
        self.p = p if p is not None else torch.full((m,), float("nan"), dtype=torch.float64, device=dev)
        self.q = (q if q is not None else torch.full((m,), float("nan"), dtype=torch.float64, device=dev)) if self.q_values else None
        for sh, o in zip(self.shards, self.offsets):
            if sh.n & 3:
                self.p[o + sh.n:o + ((sh.n + 3) & ~3)] = float("nan")
                if self.q is not None:
                    self.q[o + sh.n:o + ((sh.n + 3) & ~3)] = float("nan")
        for i, most in enumerate(self.max_sizes):
            mi = max((most + 3) & ~3, 4)
            if list_capacity or self.lists[i] is None:
                self._alloc_list(i, min(mi, int(list_capacity)) if list_capacity else min(mi, max(1 << 20, mi // 4)))
            if self.q_values and (cand_capacity or self.cands[i] is None):
                cc = min(mi, int(cand_capacity)) if cand_capacity else min(mi, max(1 << 20, mi // 16))
                keys = torch.empty(cc, dtype=torch.int64, device=dev)
                rows = torch.empty(cc, dtype=torch.int32, device=dev)
                self.cands[i] = (keys, rows, _lib.Candidates(keys.data_ptr(), rows.data_ptr(), cc))
                self._segs_host[i].cands = self.cands[i][2]
                self._segs_nt = None
        if self.q_values:
            layout = self.offsets + [self.rows]
            if layout != self._seg_layout:
                # non_blocking: a pageable source is staged at once, and the stream is not synchronised
                self.seg_off.copy_(torch.tensor(layout, dtype=torch.int64), non_blocking=True)
                self._seg_layout = layout
            need = int(self.lib.bbk_bh_segmented_workspace_bytes(m, len(self.engs)))
            if getattr(self, "bh_ws", None) is None or self.bh_ws.numel() < need:
                self.bh_ws = torch.empty(need, dtype=torch.uint8, device=dev)
        return self

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
        """Enqueue the whole pass on the current stream; no host synchronisation.  n_tests: None or -1 (every chromosome's N is
        its number of emitted rows) or one value per chromosome (-1 = that default).  marks: as GenomePass.enqueue.
        Chromosome i's fit takes s = smoothing[i] when that is set (finish() sets it to PassEngine.reference_smoothing of the
        chromosome's fit; a caller that streams passes sets it itself and submits the pass again)."""
        lib, R = self.lib, self.engs[0]
        main = torch.cuda.current_stream(self.device)
        st = _lib.stream_ptr(main)
        ns = ctypes.sizeof(_lib.ScoreState)

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(main)
                marks[name] = ev

        if n_tests is None or (np.ndim(n_tests) == 0 and int(n_tests) == -1):
            nt = [-1] * len(self.engs)
        else:
            nt = [int(x) for x in n_tests]
            if len(nt) != len(self.engs):
                raise ValueError("n_tests: one value per chromosome (%d), got %d" % (len(self.engs), len(nt)))
        self.n_tests = nt
        want_q = self.q_values
        if want_q and nt != self._segs_nt:
            for i, v in enumerate(nt):
                self._segs_host[i].n_tests = v
            self.segs.copy_(torch.frombuffer(bytearray(bytes(self._segs_host)), dtype=torch.uint8), non_blocking=True)
            self._segs_nt = nt
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
                e.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8), non_blocking=True)
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
            fits = self.decode_fits(b"".join(raw for raw, _ in state))
            again = False
            for i, (fit, (_, score)) in enumerate(zip(fits, state)):
                s_ref = PassEngine.reference_smoothing(fit)
                if s_ref is not None:
                    self.smoothing[i], again = s_ref, True
                if score.overflow:
                    self._alloc_list(i, max((self.shards[i].n + 3) & ~3, 4))
                    again = True
            if not again:
                self.last_state = state
                return fits
            self.enqueue(self.n_tests if self.q_values else None)
        raise _lib.BbkError("the per-chromosome pass did not settle after 6 attempts")

    def run(self, n_tests=None):
        self.enqueue(n_tests)
        return self.finish()

    def fit_results(self):
        """The device BbkFitResult of every chromosome, in the pass' order (HostStream copies them with each pass)."""
        return [e.fit_result for e in self.engs]

    def decode_fits(self, raw):
        """fit_results() bytes back to back -> [FitResult], in the pass' order.  A failed fit raises what the reference would
        raise for that chromosome alone, naming it (fithic.naming_chromosome); the lowest failing id wins."""
        nf = len(raw) // len(self.engs)
        for i in sorted(range(len(self.engs)), key=lambda j: self.chroms[j]):
            try:
                PassEngine.decode_fit(raw[i * nf:(i + 1) * nf])
            except Exception as e:
                from .fithic import naming_chromosome
                raise naming_chromosome(e, self.chroms[i])
        return [PassEngine.decode_fit(raw[i * nf:(i + 1) * nf]) for i in range(len(self.engs))]


class HostStream(object):
    """Successive passes streamed from pinned host memory through one GenomePass or ChromosomePass (the end-to-end call of
    this rank).

    A pass cannot start scoring before all of its records are on the device (S and the spline need the whole distance
    table, fithic.py:110-133), so inside one pass the inbound and the outbound copies never overlap; across passes they do:
    `slots` device copies of the record columns and of p / q, three streams (in, run, out) and per-slot events.  The host
    table is three contiguous pinned int32 columns holding this rank's shards back to back (shard i = rows
    starts[i] .. starts[i] + sizes[i], starts = layout_rows(sizes): every start a multiple of 4); p / q come back as pinned
    float64 columns over the same rows.  Nothing here synchronises the host: call drain() (or wait on the event submit() returns) before reading.

    With a ChromosomePass every shard is one chromosome (chroms = its ids, in its order; sizes at most those it was built
    with), each gets its own fit and q-values, and fit_of(k) returns one FitResult per chromosome.

    With refit=True (a GenomePass on one GPU) every submission is the two-pass workload of BASELINE config 4, as
    fit_transform_arrays(refit=True) runs it: pass 1 without q-values into the slot's p_first, then the refit pass that leaves
    the rows with p_first <= 1 / possibleIntraInRangeCount out of the statistics and scores every row again, both on the run
    stream with no host synchronisation in between.  fit_of(k, first=True) is pass 1's fit."""

    class _Slot(object):
        pass

    def __init__(self, genome_pass, sizes, chroms, slots=2, packed=False, cap_p=None, cap_q=None, cap_in=None, refit=False):
        """genome_pass: a GenomePass or a ChromosomePass.  sizes / chroms: records and chromosome of every shard; the slots hold
        layout_rows(sizes) rows.  packed: results cross the host link as two bits per row + the values that are not 1.0 / NaN
        (bbk_pack_scores); submit_packed() returns a PackedScores whose dense() rebuilds the float64 columns bit for bit, over
        the slot's rows (the padding rows between shards hold NaN; shard i is rows starts[i] .. starts[i] + sizes[i]).
        cap_p / cap_q: rows the packed value lists can hold (default rows / 2 and rows / 16; a pass that needs more comes back
        dense).
        cap_in: bytes of the one device buffer that packed records (PackedRecords) cross into, shared by all slots; default
        bbkio_pack_records_bound of the slots' rows, the most any pass can need.  It is allocated by the first submission of
        packed records.
        refit: run every submission as two passes (class docstring).  The outlier threshold depends on the fragments alone, so
        it is computed here, once, as fit_transform_arrays(refit=True) computes it; possibleIntraInRangeCount <= 0 raises
        ZeroDivisionError.  A ChromosomePass, or a GenomePass across ranks, raises NotImplementedError."""
        self.refit = bool(refit)
        if self.refit:
            if not isinstance(genome_pass, GenomePass):
                raise NotImplementedError("refit=True streams a GenomePass; per_chromosome=True does not take refit=True")
            if genome_pass.world > 1:
                raise NotImplementedError("refit=True runs on one GPU")
            from .fithic import _in_range_possible
            eng = genome_pass.eng
            in_rng = _in_range_possible(eng.possible.cpu().numpy(), eng.R, eng.min_dist, eng.max_dist)
            if in_rng <= 0:
                raise ZeroDivisionError("float division by zero (possibleIntraInRangeCount == 0)")
            self.p_outlier = 1.0 / in_rng
        self.gp = genome_pass
        self.sizes, self.chroms = [int(x) for x in sizes], [int(x) for x in chroms]
        self.starts, rows = layout_rows(self.sizes)
        self.rows = max(rows, 4)
        self.packed = bool(packed)
        dev = genome_pass.device
        nf = sum(f.numel() for f in genome_pass.fit_results())
        self.slots = []
        for _ in range(int(slots)):
            s = HostStream._Slot()
            s.mid1, s.mid2, s.count = (torch.empty(self.rows, dtype=torch.int32, device=dev) for _ in range(3))
            s.p = torch.full((self.rows,), float("nan"), dtype=torch.float64, device=dev)
            s.q = torch.full((self.rows,), float("nan"), dtype=torch.float64, device=dev) if genome_pass.q_values else None
            s.shards = self._shards(s, self.starts, self.sizes)
            s.in_ready, s.run_done, s.out_done, s.counts_ready = (torch.cuda.Event() for _ in range(4))
            s.fit = torch.zeros(nf, dtype=torch.uint8, device=dev)
            s.h_fit = torch.zeros(nf, dtype=torch.uint8).pin_memory()
            if self.refit:
                s.p_first = torch.full((self.rows,), float("nan"), dtype=torch.float64, device=dev)
                s.fit_first = torch.zeros(nf, dtype=torch.uint8, device=dev)
                s.h_fit_first = torch.zeros(nf, dtype=torch.uint8).pin_memory()
            if self.packed:
                s.pack = DevicePack(self.rows, dev, genome_pass.q_values, cap_p, cap_q)
                s.h_pack_state = torch.zeros(ctypes.sizeof(_lib.PackState), dtype=torch.uint8).pin_memory()
            s.index = -1
            self.slots.append(s)
        # Nothing here synchronises, so nothing would see BbkScoreState.overflow: the deferred list has a place for every row
        # of a slot (and later attaches keep it, being no larger).  A ChromosomePass caps each chromosome's list at the rows it
        # was built with, which no pass can exceed.
        genome_pass.attach(s.shards, s.p, s.q, list_capacity=self.rows)
        self.s_in, self.s_run, self.s_out = (torch.cuda.Stream(dev) for _ in range(3))
        self.s_run.wait_stream(torch.cuda.current_stream(dev))
        self.submitted = 0
        self._pending = None
        self.cap_in = int(cap_in) if cap_in is not None else _io.pack_records_bound(layout_rows(self.sizes)[1])
        self.d_in = None

    def _shards(self, s, starts, sizes):
        return [Shard(s.mid1[a:a + n], s.mid2[a:a + n], s.count[a:a + n], chrom=c) for a, n, c in zip(starts, sizes, self.chroms)]

    def _smoothing(self, smoothing):
        """smoothing= of a submission, checked: (s_first, s_second) with refit, else one s (None: the kernel's own)."""
        if isinstance(self.gp, ChromosomePass):
            if smoothing is not None:
                raise ValueError("a ChromosomePass stream takes chromosome i's s from pass.smoothing[i], not smoothing=")
            return None
        if not self.refit:
            return None if smoothing is None else float(smoothing)
        if smoothing is None:
            return None, None
        if isinstance(smoothing, (str, bytes)) or np.ndim(smoothing) != 1 or len(smoothing) != 2:
            raise ValueError("a refit stream takes smoothing=(s_first, s_second), each None or a float")
        return tuple(None if v is None else float(v) for v in smoothing)

    def _run(self, h_mid1, h_mid2, h_count, h_out, n_tests, sizes, q_values, pack=False, smoothing=None):
        """What submit() and submit_packed() share: check the host columns (or the packed records in h_mid1), copy the records
        into the next slot (stream in; packed records are decoded there into the slot's columns) and run the pass there
        (stream run; with refit, pass 1 into the slot's p_first, its fit copied aside, then the refit pass), packing p / q
        after it when `pack`.  Returns (slot, rows the pass covers)."""
        smoothing = self._smoothing(smoothing)
        s = self.slots[self.submitted % len(self.slots)]
        sizes = self.sizes if sizes is None else [int(x) for x in sizes]
        starts, rows = layout_rows(sizes)
        if len(sizes) != len(self.chroms) or rows > self.rows:
            raise ValueError("sizes must give one shard per chromosome of the stream and fit its %d rows" % self.rows)
        n = starts[-1] + sizes[-1] if sizes else 0
        rec = h_mid1 if isinstance(h_mid1, PackedRecords) else None
        if rec is not None:
            if h_mid2 is not None or h_count is not None:
                raise ValueError("pass either packed records or the three host columns")
            if rec.rows != rows or rec.sizes != sizes:
                raise ValueError("the packed records have layout %s (%d rows); this pass has %s (%d rows)" % (rec.sizes, rec.rows, sizes, rows))
            if rec.nbytes > self.cap_in:
                raise ValueError("the packed records take %d bytes; the stream's inbound buffer holds %d (cap_in)" % (rec.nbytes, self.cap_in))
            rec.check()
        cols = (h_mid1, h_mid2, h_count) if rec is None else ()
        for t in cols + h_out:
            if t is not None and (not t.is_pinned() or t.numel() < n):
                raise ValueError("host columns must be pinned and hold at least %d rows" % n)
        if q_values and s.q is None:
            raise ValueError("the stream's pass was made with q_values=False")
        self.gp.check_sizes(sizes)
        shards = s.shards if sizes is self.sizes else self._shards(s, starts, sizes)
        if rec is not None and self.d_in is None:
            with torch.cuda.stream(self.s_in):
                self.d_in = torch.empty(max(self.cap_in, 16), dtype=torch.uint8, device=s.mid1.device)
        self.submitted += 1
        s.index = self.submitted - 1
        self.s_in.wait_event(s.run_done)        # the pass that last read this slot's records has finished
        with torch.cuda.stream(self.s_in):
            if rec is None:
                s.mid1[:n].copy_(h_mid1[:n], non_blocking=True)
                s.mid2[:n].copy_(h_mid2[:n], non_blocking=True)
                s.count[:n].copy_(h_count[:n], non_blocking=True)
            else:
                # one inbound buffer: the next pass' copy queues behind this decode on the same stream
                self.d_in[:rec.nbytes].copy_(rec.buf[:rec.nbytes], non_blocking=True)
                _decode_records(self.d_in, rec.nbytes, rec.rows, s.mid1, s.mid2, s.count, self.s_in)
                self.gp.launches += 1
            s.in_ready.record()
        # the previous packed pass' value lists: their sizes are on the host by now (or soon); their copies overlap these inbound ones
        self._finalize_pending()
        self.s_run.wait_event(s.in_ready)
        self.s_run.wait_event(s.out_done)       # this slot's previous p / q have left the device
        gp = self.gp
        with torch.cuda.stream(self.s_run):
            keep_q = gp.q_values
            try:
                if self.refit:
                    # one pass object for both passes: they share its deferred list, which has a place for every slot row
                    gp.q_values = False
                    gp.attach(shards, s.p_first, None)
                    gp.enqueue(-1, smoothing=smoothing[0])
                    s.fit_first.copy_(gp.eng.fit_result, non_blocking=True)
                    gp.q_values = q_values
                    gp.attach(shards, s.p, s.q)
                    gp.enqueue(n_tests, smoothing=smoothing[1], exclude=(s.p_first, self.p_outlier))
                else:
                    gp.q_values = q_values
                    gp.attach(shards, s.p, s.q)
                    if isinstance(gp, ChromosomePass):
                        gp.enqueue(n_tests)
                    else:
                        gp.enqueue(n_tests, smoothing=smoothing)
            finally:
                gp.q_values = keep_q
            o = 0
            for f in gp.fit_results():
                s.fit[o:o + f.numel()].copy_(f, non_blocking=True)
                o += f.numel()
            if pack:
                s.pack.pack(s.p, s.q, self.s_run)
                gp.launches += 2
            s.run_done.record()
        return s, n

    def submit(self, h_mid1, h_mid2=None, h_count=None, h_p=None, h_q=None, n_tests=-1, sizes=None, h_p_first=None, smoothing=None):
        """Enqueue one pass over the host table; returns the event that fires when p (and q) are on the host.
        sizes: this pass' shard sizes, one per chromosome of the stream (default: the sizes it was made with); their
        layout_rows total must fit the slots.  The host columns hold at least the rows the pass covers (up to the end of its
        last shard), and exactly those rows come back.  Without h_q the pass skips the q-value step; at N > 1 that step is
        collective, so every rank must pass or omit h_q alike.
        h_mid1 may instead be a PackedRecords of exactly this pass' sizes (h_mid2 / h_count omitted): submit(rec, h_p=..,
        h_q=..).  It is validated on the host, crosses the link as it is and is decoded into the slot on the device; a layout
        that differs from the pass', more bytes than cap_in, or a buffer that fails validation raise ValueError before
        anything is copied.  Like h_p, the PackedRecords may be refilled once the returned event has fired.
        smoothing: the s a GenomePass stream's fit takes (None: the kernel's min(y) * min(y)); a pass whose fit_of(k) gives
        PassEngine.reference_smoothing(fit) != None is submitted again with that value to equal GenomePass.run.  With refit,
        a pair (s_first, s_second) for the two passes, each None or a float: settle s_first by fit_of(k, first=True), then
        s_second by fit_of(k), as fit_transform_arrays(refit=True) does.  A ChromosomePass stream takes pass.smoothing[i]
        instead, and smoothing= raises ValueError there.
        h_p_first (refit only): an optional pinned float64 column that receives pass 1's p over the same rows as h_p."""
        if h_p is None:
            raise ValueError("submit needs h_p")
        if h_p_first is not None and not self.refit:
            raise ValueError("h_p_first needs a stream made with refit=True")
        s, n = self._run(h_mid1, h_mid2, h_count, (h_p, h_q, h_p_first), n_tests, sizes, h_q is not None, smoothing=smoothing)
        self.s_out.wait_event(s.run_done)
        with torch.cuda.stream(self.s_out):
            h_p[:n].copy_(s.p[:n], non_blocking=True)
            if h_q is not None:
                h_q[:n].copy_(s.q[:n], non_blocking=True)
            if h_p_first is not None:
                h_p_first[:n].copy_(s.p_first[:n], non_blocking=True)
            self._fits_out(s)
            s.out_done.record()
        return s.out_done

    def _fits_out(self, s):
        s.h_fit.copy_(s.fit, non_blocking=True)
        if self.refit:
            s.h_fit_first.copy_(s.fit_first, non_blocking=True)

    # ------------------------------------------------------------------ packed results
    def submit_packed(self, h_mid1, h_mid2=None, h_count=None, out=None, n_tests=-1, smoothing=None):
        """Like submit(), but p / q come back packed into `out` (a PackedScores made by packed_buffers()).  The sizes of the two
        value lists are only known once the pass has run, so their copies are issued lazily: by the NEXT submission (after
        it has put its own inbound copies on the wire) or by drain().  Returns `out`; out.done fires when it is complete.
        h_mid1 may be a PackedRecords of the stream's sizes, as in submit(): submit_packed(rec, out=out); it may be refilled
        once out.done has fired.  smoothing: as in submit().  With refit, `out` holds the refit pass' p / q; pass 1's p does
        not come back (its fit does: fit_of(k, first=True))."""
        if out is None:
            raise ValueError("submit_packed needs out (packed_buffers())")
        if not self.packed:
            raise ValueError("this stream was not created with packed=True")
        s, _ = self._run(h_mid1, h_mid2, h_count, (), n_tests, None, self.gp.q_values, pack=True, smoothing=smoothing)
        self.s_out.wait_event(s.run_done)
        with torch.cuda.stream(self.s_out):
            s.h_pack_state.copy_(s.pack.state, non_blocking=True)
            s.counts_ready.record()
            out.codes.copy_(s.pack.codes, non_blocking=True)
            out.chunks.copy_(s.pack.chunks, non_blocking=True)
            self._fits_out(s)
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

    def fit_of(self, index, first=False):
        """Fit result of submission `index` once its outputs are on the host (raises the reference's exception for a failed
        fit); PassEngine.reference_smoothing(result) tells whether that pass must be repeated with the reference's own s
        (submit(..., smoothing=...)).
        With a ChromosomePass: one FitResult per chromosome, in its order; a failed fit raises for the lowest failing id,
        naming it, and a chromosome is repeated with its own s by setting pass.smoothing[i] and submitting again.
        With refit: the refit pass' fit, after raising pass 1's exception if pass 1 failed (what fit_transform_arrays(refit=True)
        raises first); first=True: pass 1's fit.
        Only the last `slots` submissions are held."""
        if first and not self.refit:
            raise ValueError("first=True needs a stream made with refit=True")
        s = self.slots[int(index) % len(self.slots)]
        if s.index != int(index):
            raise KeyError("submission %d is no longer (or not yet) held by the stream" % int(index))
        s.out_done.synchronize()
        if self.refit:
            fit1 = self.gp.decode_fits(s.h_fit_first.numpy().tobytes())
            if first:
                return fit1
        return self.gp.decode_fits(s.h_fit.numpy().tobytes())

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


def _decode_records(d_buf, nbytes, rows, mid1, mid2, count, stream):
    """bbk_unpack_records on `stream`: packed records already on the device (validated on the host by the caller, as
    bbkio_check_records) into the first `rows` rows of three int32 columns."""
    _lib.check(_lib.load().bbk_unpack_records(_lib.ptr(d_buf), int(nbytes), int(rows), _lib.ptr(mid1), _lib.ptr(mid2), _lib.ptr(count),
                                              _lib.stream_ptr(stream)), "bbk_unpack_records")


class PackedRecords(object):
    """The contact records of one pass packed for the host link (include/bbk.h, BbkRecHeader: a frame-of-reference code per
    4096 rows, ~3 B/row on Hi-C records against 12 B/row of int32 columns) in a pinned uint8 buffer.  rows / sizes: the pass
    layout (layout_rows(sizes)); nbytes: bytes of buf in use.  Made and refilled by pack_records()."""

    def __init__(self, capacity):
        self.buf = torch.empty(max(int(capacity), 32), dtype=torch.uint8).pin_memory()
        self.rows, self.sizes, self.nbytes = 0, [], 0

    def check(self):
        """Raise ValueError unless buf holds valid packed records of `rows` rows (bbkio_check_records)."""
        _io.check_records(self.buf.data_ptr(), self.nbytes, self.rows)

    def to_device(self, device=None):
        """Validate on the host, copy once and decode on the device (current stream; asynchronous): returns (mid1, mid2, count),
        int32 tensors of `rows` rows in the pass layout (padding rows between shards are 0).  buf may be refilled once the
        current stream has passed this call."""
        self.check()
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        with torch.cuda.device(dev):
            d_buf = torch.empty(max(self.nbytes, 16), dtype=torch.uint8, device=dev)
            d_buf[:self.nbytes].copy_(self.buf[:self.nbytes], non_blocking=True)
            cols = [torch.empty(max(self.rows, 4), dtype=torch.int32, device=dev) for _ in range(3)]
            _decode_records(d_buf, self.nbytes, self.rows, cols[0], cols[1], cols[2], torch.cuda.current_stream(dev))
        return tuple(c[:self.rows] for c in cols)


def pack_records(shards, out=None, threads=0):
    """Pack the records of one pass for the host link: shards = [(mid1, mid2, count), ...], int32 host columns (numpy arrays or
    CPU tensors, any memory) laid out as layout_rows gives, without assembling padded columns first.  All host cores
    (threads <= 0), two phases over 4096-row chunks; the bytes do not depend on the thread count.  out: a PackedRecords to
    refill (ValueError when its buffer is too small), or None for a new one sized for the worst case.  Returns it."""
    sizes = [len(sh[0]) for sh in shards]
    rows = layout_rows(sizes)[1]
    if out is None:
        out = PackedRecords(_io.pack_records_bound(rows))
    out.rows, out.sizes, out.nbytes = 0, [], 0
    nbytes = _io.pack_records(shards, out.buf.data_ptr(), out.buf.numel(), threads)
    out.rows, out.sizes, out.nbytes = rows, sizes, nbytes
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# One genome-wide pass larger than the device: row blocks streamed from host memory
# ---------------------------------------------------------------------------------------------------------------------------
BLOCK_ALIGN = _lib.PACK_CHUNK       # every piece starts on a packed-results chunk: its rows unpack straight into the shard's output
_SMALL_P_KEY = int(np.array([0.03125]).view(np.uint64)[0]) | (1 << 63)      # bbk_key_of(BBK_SMALL_P)


def plan_blocks(sizes, block_rows, align=BLOCK_ALIGN):
    """Cut shards of these sizes, laid end to end, into row blocks of at most `block_rows` rows.  A block is a list of
    pieces (shard, first row of the shard, rows, device row); every piece starts on a multiple of `align` in the block's
    device buffers (so of 4, as in layout_rows), the rows between pieces are padding, and a block's device rows
    (block_device_rows) are at most block_rows rounded up to `align`.  A shard is cut wherever a block fills up (records
    are independent).  Empty shards get no piece.  Returns the list of blocks."""
    block_rows, align = int(block_rows), int(align)
    if align <= 0 or align & 3:
        raise ValueError("align must be a positive multiple of 4")
    if block_rows < 1 or (block_rows + align - 1) // align * align >= (1 << 32):
        raise ValueError("block_rows must be positive and, rounded up to %d, below 2^32; got %d" % (align, block_rows))
    blocks, cur, used = [], [], 0
    for s, n in enumerate(sizes):
        n = int(n)
        if n < 0:
            raise ValueError("shard %d has a negative size" % s)
        first = 0
        while first < n:
            take = min(n - first, block_rows - used)
            cur.append((s, first, take, used))
            used = (used + take + align - 1) // align * align
            first += take
            if used >= block_rows:
                blocks.append(cur)
                cur, used = [], 0
    if cur:
        blocks.append(cur)
    return blocks


def block_device_rows(block, align=BLOCK_ALIGN):
    """Device rows of one block of plan_blocks: its last piece's end, rounded up to `align`."""
    _, _, n, off = block[-1]
    return (off + n + align - 1) // align * align


def resident_pass_bytes(rows, q_values=True, refit=False):
    """Device bytes of a resident genome-wide pass over `rows` layout rows (GenomePass, streaming K4): 12 B of records, 8 B of
    p (and 8 B of q), the deferred list (rows / 4 x 16 B) and the candidate list (rows / 16 x 12 B), plus the q-value
    workspace of one GPU (bbk_bh_workspace_bytes: 24 B a row).  refit: the two-pass workload of fit_transform_arrays(refit=True),
    whose pass 1 holds its own p, deferred list and candidate list while the refit pass runs."""
    rows = int(rows)
    per = 12 + 8 + 16 / 4 + 12 / 16 + ((8 + 24) if q_values else 0) + ((8 + 16 / 4 + 12 / 16) if refit else 0)
    return int(rows * per)


def needs_blocked_pass(rows, free_bytes, q_values=True, margin=1 << 30, refit=False):
    """Whether a genome-wide pass over `rows` layout rows cannot run resident on one GPU with `free_bytes` of free device
    memory (torch.cuda.mem_get_info): 2^32 rows or more, or more bytes than are free after a margin.  refit: the two-pass
    workload (resident_pass_bytes)."""
    return int(rows) >= (1 << 32) or resident_pass_bytes(rows, q_values, refit) + int(margin) > int(free_bytes)


def _host_f64(a, n, what):
    """A float64 host output column of exactly n rows as a numpy view (numpy array or CPU tensor)."""
    if isinstance(a, torch.Tensor):
        if a.is_cuda or a.dtype != torch.float64 or not a.is_contiguous():
            raise ValueError("%s: contiguous float64 host columns (numpy or CPU tensors)" % what)
        a = a.numpy()
    if not isinstance(a, np.ndarray) or a.dtype != np.float64 or a.ndim != 1 or not a.flags.c_contiguous or not a.flags.writeable:
        raise ValueError("%s: contiguous, writable float64 host columns" % what)
    if a.shape[0] != n:
        raise ValueError("%s: the column has %d rows, its shard %d" % (what, a.shape[0], n))
    return a


def _host_rows(a, what):
    """Rows of a host record column (numpy array of integers or a CPU tensor)."""
    if isinstance(a, torch.Tensor):
        if a.is_cuda:
            raise ValueError("%s: host columns (numpy or CPU tensors), not device tensors" % what)
        return int(a.shape[0]) if a.dim() == 1 else -1
    a = np.asarray(a)
    if a.ndim != 1 or a.dtype.kind not in "iu":
        raise ValueError("%s: one-dimensional integer columns" % what)
    return int(a.shape[0])


class BlockedPass(object):
    """One genome-wide Fit-Hi-C pass on one GPU over records held in host memory, in row blocks, so that a pass larger than
    the device (BASELINE config 5: 6.03e9 records, past 2^32 rows and ~197 GB resident) runs, with the same bits as
    GenomePass(engine, group=False).run over the same shards held resident.

        sweep 1: K1 per piece, block after block, into one table  ->  fit, settled with ONE synchronisation (more bins, the
        reference's own s, a failed fit raising before any p exists)  ->  sweep 2: per block guard, streaming K4, patch pass,
        results packed and unpacked into the caller's columns by all host cores  ->  q-values: every block's candidates
        selected against the genome-wide histogram, as ranks would be, ranked together ONCE (bbk_bh_rank_gathered_all) and
        scattered on the host  [-> a third sweep over p from the host when the candidate lists do not cover every candidate]

    Blocks whose records fit `resident_bytes` stay on the device between the sweeps; the others are sent again.  The inbound
    copy of block k + 1 overlaps the kernels of block k, which overlap the outbound copy of block k - 1.
    engine: a PassEngine over the whole genome (set_fragments / set_bias as for GenomePass), with the streaming K4's
    conditions (GenomePass.listed): 0 <= min_dist <= max_dist, max_dist + resolution < 2^31, resolution >= 2, no bias table
    of step 1.  Otherwise ValueError.

    refit=True runs the two-pass workload of BASELINE config 4 (fit_transform_arrays(refit=True)) with the same bits as the
    resident two-pass (GenomePass(q_values=False).run, then GenomePass.run(exclude=(p_first, p_outlier)) on the same engine):

        sweep 1: K1 into table 1  ->  fit 1, settled (fit_first)  ->  sweep 2: per block pass 1's scores into the block's p
        slot, then K1 over the block's rows whose pass-1 p is not <= p_outlier into table 2 (the engine's tables, refilled:
        pass-1 scoring reads only the fit and the spline)  [-> pass 1's p packed into p_first_out]  ->  fit 2, settled  ->
        sweep 3 and the q-values as above

    Pass 1's p never crosses the link for the refit itself; the records of the blocks that are not resident cross it once
    per sweep.  The outlier threshold p_outlier = 1 / possibleIntraInRangeCount depends on the fragments alone and is
    computed here, as fit_transform_arrays(refit=True) computes it; a count <= 0 raises ZeroDivisionError before any device
    work."""

    def __init__(self, engine, q_values=True, block_rows=1 << 27, resident_bytes=None, cand_capacity=None, refit=False):
        e = engine
        if not (0 <= e.min_dist <= e.max_dist and e.max_dist + e.R < (1 << 31) and e.R >= 2) or \
                (e.bias is not None and e.bias.step == 1):
            raise ValueError("BlockedPass runs the streaming K4 only (the conditions of GenomePass.listed)")
        plan_blocks([], block_rows)                       # checks block_rows
        self.eng, self.lib, self.device = e, e.lib, e.device
        self.q_values = bool(q_values)
        self.block_rows = int(block_rows)
        self.resident_bytes = None if resident_bytes is None else int(resident_bytes)
        self.cand_capacity = None if cand_capacity is None else max(int(cand_capacity), 1)
        self.refit = bool(refit)
        self.p_outlier = None
        if self.refit:
            from .fithic import _in_range_possible
            in_rng = _in_range_possible(e.possible.cpu().numpy(), e.R, e.min_dist, e.max_dist)
            if in_rng <= 0:
                raise ZeroDivisionError("float division by zero (possibleIntraInRangeCount == 0)")
            self.p_outlier = 1.0 / in_rng
        self.force_exact = False        # tests: raise BbkScoreState.exact whatever the guard says
        self.blocks, self.resident = [], []
        self.fit_first = None
        self.bytes_in = self.bytes_out = 0
        self.host_unpack_s = 0.0

    @property
    def launches(self):
        """Kernel launches counted so far (the engine's counter)."""
        return self.eng.launches

    @launches.setter
    def launches(self, n):
        self.eng.launches = n

    # ------------------------------------------------------------------ checks
    def check(self, shards, p_out, q_out=None, p_first_out=None):
        """Raise ValueError unless the arguments of run() are complete; returns (sizes, p columns, q columns)."""
        return self._check(shards, p_out, q_out, p_first_out)[:3]

    def _check(self, shards, p_out, q_out, p_first_out):
        shards = list(shards)
        sizes, ps, qs, p1s = [], [], [], None
        if p_out is None or len(p_out) != len(shards):
            raise ValueError("p_out: one column per shard")
        if self.q_values and (q_out is None or len(q_out) != len(shards)):
            raise ValueError("q_out: one column per shard (the pass was made with q_values=True)")
        if not self.q_values and q_out is not None:
            raise ValueError("q_out given, but the pass was made with q_values=False")
        if p_first_out is not None:
            if not self.refit:
                raise ValueError("p_first_out needs a pass made with refit=True")
            if len(p_first_out) != len(shards):
                raise ValueError("p_first_out: one column per shard")
            p1s = []
        for i, sh in enumerate(shards):
            if len(sh) != 4:
                raise ValueError("shard %d: (chrom, mid1, mid2, count); BlockedPass takes one-chromosome shards" % i)
            n = _host_rows(sh[1], "shard %d" % i)
            if n < 0 or _host_rows(sh[2], "shard %d" % i) != n or _host_rows(sh[3], "shard %d" % i) != n:
                raise ValueError("shard %d: the columns differ in length" % i)
            sizes.append(n)
            ps.append(_host_f64(p_out[i], n, "p_out[%d]" % i))
            qs.append(_host_f64(q_out[i], n, "q_out[%d]" % i) if self.q_values else None)
            if p1s is not None:
                p1s.append(_host_f64(p_first_out[i], n, "p_first_out[%d]" % i))
        blocks = plan_blocks(sizes, self.block_rows)
        cc = self._cand_cap(blocks)
        if len(blocks) * cc >= (1 << 32):
            raise ValueError("%d blocks of %d candidate places reach 2^32: use larger blocks" % (len(blocks), cc))
        return sizes, ps, qs, p1s

    def _cand_cap(self, blocks):
        if self.cand_capacity:
            return self.cand_capacity
        most = max([block_device_rows(b) for b in blocks] + [4])
        return min(most, max(1 << 20, self.block_rows // 16))

    # ------------------------------------------------------------------ helpers
    def _copy_piece(self, dst, col, lo, n):
        """Rows [lo, lo + n) of a host column into the device view dst (current stream)."""
        if isinstance(col, torch.Tensor) and col.dtype == torch.int32 and col.is_pinned():
            dst.copy_(col[lo:lo + n], non_blocking=True)
        else:
            from .fithic import _to_device_i32
            dst.copy_(_to_device_i32(col, self.device, lo, lo + n), non_blocking=True)
        self.bytes_in += 4 * n

    def _records_in(self, k, cols, stream, ready):
        """The pieces of block k into its record columns, on `stream`; `ready` fires when they are there."""
        with torch.cuda.stream(stream):
            for (s, lo, n, off) in self.blocks[k]:
                for dst, j in zip(cols, (1, 2, 3)):
                    self._copy_piece(dst[off:off + n], self._shards[s][j], lo, n)
            ready.record(stream)

    def _pieces(self, k, cols):
        return [(self._shards[s][0], Shard(cols[0][off:off + n], cols[1][off:off + n], cols[2][off:off + n], chrom=self._shards[s][0]), off)
                for (s, lo, n, off) in self.blocks[k]]

    def _nan_padding(self, k, p, q):
        """Padding rows of block k (between its pieces and up to its device rows) = NaN in p / q (the pack sees them as empty)."""
        blk = self.blocks[k]
        ends = [off + n for (_, _, n, off) in blk]
        starts = [off for (_, _, _, off) in blk[1:]] + [block_device_rows(blk)]
        for a, b in zip(ends, starts):
            if b > a:
                p[a:b] = float("nan")
                if q is not None:
                    q[a:b] = float("nan")
                self.eng.launches += 1 if q is None else 2

    # ------------------------------------------------------------------ the pass
    def run(self, shards, p_out, q_out=None, n_tests=-1, marks=None, p_first_out=None):
        """Run the pass.  shards: [(chrom, mid1, mid2, count)], host columns (numpy integer arrays, or CPU tensors; pinned int32
        tensors go by one asynchronous copy each).  p_out / q_out: one float64 host column per shard, exactly as long as it
        (numpy arrays or CPU tensors); q_out only with q_values.  n_tests: N of the q-values (-1: the number of non-NaN p); with
        refit, of the refit pass.  marks (optional dict): CUDA events recorded after each stage ("start", "hist", "fit",
        "pvalues", "bh"; with refit also "hist_first" and "fit_first" after sweep 1 and fit 1, and "hist" after sweep 2).
        Returns the FitResult (with refit: the refit pass', pass 1's is fit_first); a failed fit raises what GenomePass.run
        raises, before any p of its pass is computed and with p_out / q_out untouched.
        p_first_out (refit only): one float64 host column per shard, like p_out, that receives pass 1's p.  It is written
        during sweep 2, so it already holds pass 1's p when the refit pass' fit fails."""
        sizes, ps, qs, p1s = self._check(shards, p_out, q_out, p_first_out)
        eng, lib, dev = self.eng, self.lib, self.device
        self._shards = [tuple(sh) for sh in shards]
        self.blocks = plan_blocks(sizes, self.block_rows)
        self.bytes_in = self.bytes_out = 0
        self.host_unpack_s = 0.0
        self.fit_first = None
        nb = len(self.blocks)
        dev_rows = [block_device_rows(b) for b in self.blocks]
        main = torch.cuda.current_stream(dev)
        st = _lib.stream_ptr(main)

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(main)
                marks[name] = ev

        mark("start")
        # the working set (sized by block_rows), then the records of as many blocks as the budget holds, in order
        br = self.block_rows
        ns = ctypes.sizeof(_lib.ScoreState)
        self.score_state = torch.zeros(max(nb, 1) * ns, dtype=torch.uint8, device=dev)
        self._h_state = torch.zeros(max(nb, 1) * ns, dtype=torch.uint8).pin_memory()
        slot_rows = max(dev_rows + [4])
        pq = [(torch.empty(slot_rows, dtype=torch.float64, device=dev),
               torch.empty(slot_rows, dtype=torch.float64, device=dev) if self.q_values else None) for _ in range(min(nb, 2))]
        packs = [DevicePack(slot_rows, dev, self.q_values) for _ in range(len(pq))]
        h_packs = [PackedScores(slot_rows, pk.codes.numel(), pk.chunks.numel() // 24, pk.cap_p, pk.cap_q) for pk in packs]
        h_pack_state = [torch.zeros(ctypes.sizeof(_lib.PackState), dtype=torch.uint8).pin_memory() for _ in packs]
        l_cap = slot_rows                                  # the deferred list has a place for every row of a block: no overflow
        l_row = torch.empty(l_cap, dtype=torch.int32, device=dev)
        l_cnt = torch.empty(l_cap, dtype=torch.int32, device=dev)
        l_prior = torch.empty(l_cap, dtype=torch.float64, device=dev)
        deferred = _lib.DeferredList(l_row.data_ptr(), l_cnt.data_ptr(), l_prior.data_ptr(), l_cap)
        ccap = self._cand_cap(self.blocks)
        cands = []
        if self.q_values:
            for _ in range(nb):
                keys = torch.empty(ccap, dtype=torch.int64, device=dev)
                rows = torch.empty(ccap, dtype=torch.int32, device=dev)
                cands.append((keys, rows, _lib.Candidates(keys.data_ptr(), rows.data_ptr(), ccap)))
        slot_bytes = 12 * slot_rows
        budget = self.resident_bytes
        if budget is None:
            free, total = torch.cuda.mem_get_info(dev)
            budget = free - max(1 << 30, total // 50) - 2 * slot_bytes
        self.resident, used = [], 0
        for r in dev_rows:
            keep = used + 12 * r <= budget
            self.resident.append(keep)
            used += 12 * r if keep else 0
        # resident blocks get their own columns; the others share two slots
        cols = [tuple(torch.empty(r, dtype=torch.int32, device=dev) for _ in range(3)) if keep else None
                for r, keep in zip(dev_rows, self.resident)]
        slots = [tuple(torch.empty(slot_rows, dtype=torch.int32, device=dev) for _ in range(3)) for _ in range(2)] \
            if not all(self.resident) else []
        far = [k for k in range(nb) if not self.resident[k]]         # blocks sent again in each later sweep, in turn through the two slots
        slot_of = {k: i & 1 for i, k in enumerate(far)}
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        s_in.wait_stream(main)
        s_out.wait_stream(main)
        in_ready = [torch.cuda.Event() for _ in range(nb)]
        slot_free = [torch.cuda.Event() for _ in range(2)]

        def block_cols(k):
            return cols[k] if self.resident[k] else slots[slot_of[k]]

        def send(k):
            if not self.resident[k]:
                s_in.wait_event(slot_free[slot_of[k]])        # the kernels that last read this slot have finished
            self._records_in(k, block_cols(k), s_in, in_ready[k])

        def sweep():
            """The blocks in order, each once its records are on the device: the resident ones are, the others are sent again
            through the two slots, the next one while this one's kernels run."""
            if far:
                send(far[0])
            for k in range(nb):
                if not self.resident[k]:
                    i = far.index(k)
                    if i + 1 < len(far):
                        send(far[i + 1])                      # into the other slot, while block k is scored
                    main.wait_event(in_ready[k])
                yield k

        def records_done(k):
            if not self.resident[k]:
                slot_free[slot_of[k]].record(main)

        bias = ctypes.byref(eng.bias.struct) if eng.bias is not None else None
        flags = _lib.ptr(eng.bias.flags) if eng.bias is not None else None

        def score(k, p, q, hist, cand):
            """K4 of block k into the device columns p / q: score state k, the guard, the streaming pass per piece, the patch
            pass.  Returns the pieces."""
            state = ctypes.c_void_p(self.score_state.data_ptr() + k * ns)
            _lib.check(lib.bbk_score_begin(state, hist if k == 0 else None, st), "bbk_score_begin")
            _lib.check(lib.bbk_score_guard(_lib.ptr(eng.fit_result), _lib.ptr(eng.spline_y), state, st), "bbk_score_guard")
            eng.launches += 2
            if self.force_exact:
                self.score_state[k * ns + 24:k * ns + 28] = torch.tensor([1, 0, 0, 0], dtype=torch.uint8, device=dev)
            c = ctypes.byref(cand) if cand is not None else None
            pieces = self._pieces(k, block_cols(k))
            for (_, sh, off), st_i in zip(pieces, eng.fan_out(len(pieces))):
                _lib.check(lib.bbk_score_pairs(_lib.ptr(sh.mid1), _lib.ptr(sh.mid2), _lib.ptr(sh.count), sh.n, sh.chrom, eng.R, eng.min_dist,
                                               eng.max_dist, _lib.ptr(eng.fit_result), _lib.ptr(eng.spline_y), bias, flags, off,
                                               _lib.ptr(p), _lib.ptr(q), hist, c, ctypes.byref(deferred), state,
                                               st_i), "bbk_score_pairs")
                eng.launches += 1
            eng.fan_in()
            _lib.check(lib.bbk_score_deferred(ctypes.byref(deferred), _lib.ptr(eng.fit_result), _lib.ptr(p), _lib.ptr(q),
                                              hist, c, state, st), "bbk_score_deferred")
            eng.launches += 1
            return pieces

        run_done = [torch.cuda.Event() for _ in range(2)]
        counts_ready = [torch.cuda.Event() for _ in range(2)]
        out_free = [torch.cuda.Event() for _ in range(2)]
        pending = []

        def send_back(k, j, p, q, p_cols, q_cols, with_state):
            """Block k's results in slot j packed on the device and sent to the host; the previous block's are unpacked into
            p_cols / q_cols meanwhile.  with_state: block k's score state comes back too."""
            pk = packs[j]
            pk.rows = dev_rows[k]
            pk.pack(p, q, main)
            eng.launches += 2
            run_done[j].record(main)
            s_out.wait_event(run_done[j])
            hp = h_packs[j]
            with torch.cuda.stream(s_out):
                h_pack_state[j].copy_(pk.state, non_blocking=True)
                if with_state:
                    self._h_state[k * ns:(k + 1) * ns].copy_(self.score_state[k * ns:(k + 1) * ns], non_blocking=True)
                nw, nc = int(lib.bbk_pack_code_words(dev_rows[k])), int(lib.bbk_pack_chunks(dev_rows[k])) * 24
                hp.codes[:nw].copy_(pk.codes[:nw], non_blocking=True)
                hp.chunks[:nc].copy_(pk.chunks[:nc], non_blocking=True)
                self.bytes_out += 4 * nw + nc
                counts_ready[j].record(s_out)
            if pending:
                self._unpack(*pending.pop())
            pending.append((k, j, p, q, pk, hp, h_pack_state[j], counts_ready[j], out_free[j], s_out, p_cols, q_cols))

        def drain():
            if pending:
                self._unpack(*pending.pop())
            s_out.synchronize()

        # ---- sweep 1: K1 into one table
        _lib.check(lib.bbk_hist_init(_lib.ptr(eng.obs_sum), eng.nkeys, _lib.ptr(eng.totals), st), "bbk_hist_init")
        eng.launches += 1
        if nb:
            send(0)
        for k in range(nb):
            if k + 1 < nb:
                send(k + 1)
            main.wait_event(in_ready[k])
            for _, sh, _ in self._pieces(k, block_cols(k)):
                _lib.check(lib.bbk_hist_pairs(None, None, _lib.ptr(sh.mid1), _lib.ptr(sh.mid2), _lib.ptr(sh.count), sh.n, eng.R, eng.min_dist,
                                              eng.max_dist, eng.nkeys, _lib.ptr(eng.obs_sum), _lib.ptr(eng.totals), st), "bbk_hist_pairs")
                eng.launches += 1
            records_done(k)

        if self.refit:
            mark("hist_first")
            self.fit_first = self._settle_fit()                  # pass 1's fit: raises before any p exists
            mark("fit_first")
            # ---- sweep 2: pass 1's p per block into its p slot, then K1 into table 2 over the rows that are not outliers
            _lib.check(lib.bbk_hist_init(_lib.ptr(eng.obs_sum), eng.nkeys, _lib.ptr(eng.totals), st), "bbk_hist_init")
            eng.launches += 1
            for k in sweep():
                j = k & 1
                p = pq[j][0]
                main.wait_event(out_free[j])              # this slot's previous pass-1 p has left the device
                if p1s is not None:
                    self._nan_padding(k, p, None)
                pieces = score(k, p, None, None, None)
                for _, sh, off in pieces:
                    _lib.check(lib.bbk_hist_pairs_excluding(None, None, _lib.ptr(sh.mid1), _lib.ptr(sh.mid2), _lib.ptr(sh.count),
                                                             _lib.ptr(p[off:off + sh.n]), self.p_outlier, sh.n, eng.R, eng.min_dist,
                                                             eng.max_dist, eng.nkeys, _lib.ptr(eng.obs_sum), _lib.ptr(eng.totals), st),
                               "bbk_hist_pairs_excluding")
                    eng.launches += 1
                records_done(k)
                if p1s is not None:
                    send_back(k, j, p, None, p1s, None, False)
            drain()
        mark("hist")

        # ---- the fit, settled on the host once
        fit = self._settle_fit()
        mark("fit")

        # ---- the scoring sweep: block after block; results packed, unpacked into the caller's columns by the host
        want_q = self.q_values
        hist = _lib.ptr(eng.p_hist) if want_q else None
        if nb == 0 and want_q:
            eng.p_hist.zero_()
            eng.launches += 1
        for k in sweep():
            j = k & 1
            p, q = pq[j]
            main.wait_event(out_free[j])                  # this slot's previous results have left the device
            self._nan_padding(k, p, q)
            score(k, p, q, hist, cands[k][2] if want_q else None)
            records_done(k)
            send_back(k, j, p, q, ps, qs, True)
        drain()
        mark("pvalues")
        states = [_lib.ScoreState.from_buffer_copy(self._h_state.numpy().tobytes()[k * ns:(k + 1) * ns]) for k in range(nb)]
        if any(s.overflow for s in states):
            raise _lib.BbkError("a block's deferred list overflowed")     # it has a place for every row: cannot happen
        self.last_states = states
        # the records are not needed any more: the q-value step gets their memory
        cols = slots = packs = pq = None
        if want_q and nb:
            self._qvalues(int(n_tests), states, cands, ps, qs, dev_rows)
        mark("bh")
        return fit

    def _settle_fit(self, smoothing=None):
        eng = self.eng
        host = torch.zeros(eng.fit_result.numel(), dtype=torch.uint8).pin_memory()
        for _ in range(6):
            eng.fit(smoothing)
            host.copy_(eng.fit_result, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            raw = host.numpy().tobytes()
            if _lib.FitResult.from_buffer_copy(raw).status == _lib.FIT_TOO_MANY_BINS and eng.grow_bins():
                continue                                          # more bins than the default buffers hold: one per key
            fit = PassEngine.decode_fit(raw)                      # raises what the reference would raise
            s_ref = PassEngine.reference_smoothing(fit)
            if s_ref is None:
                return fit
            smoothing = s_ref
        raise _lib.BbkError("the fit did not settle after 6 attempts")

    def _unpack(self, k, j, p, q, pk, hp, h_state, counts_ready, out_free, s_out, ps, qs):
        """Block k's packed results (slot j) into the caller's columns: the value lists follow once their sizes are known, then
        every piece is unpacked by all host cores straight into its shard's rows."""
        import time
        counts_ready.synchronize()
        pst = _lib.PackState.from_buffer_copy(h_state.numpy().tobytes())
        blk = self.blocks[k]
        with torch.cuda.stream(s_out):
            if pst.overflow:                      # more values than the lists hold: the columns come back dense, piece by piece
                for (s, lo, n, off) in blk:
                    torch.from_numpy(ps[s][lo:lo + n]).copy_(p[off:off + n])
                    if q is not None:
                        torch.from_numpy(qs[s][lo:lo + n]).copy_(q[off:off + n])
                    self.bytes_out += 8 * n * (2 if q is not None else 1)
                out_free.record(s_out)
                return
            n_p, n_q = int(pst.n_p), int(pst.n_q)
            if n_p:
                hp.vals_p[:n_p].copy_(pk.vals_p[:n_p], non_blocking=True)
            if n_q and pk.vals_q is not None:
                hp.vals_q[:n_q].copy_(pk.vals_q[:n_q], non_blocking=True)
            self.bytes_out += 8 * (n_p + n_q)
            out_free.record(s_out)
        out_free.synchronize()
        t0 = time.perf_counter()
        codes, chunks = hp.codes.numpy(), hp.chunks.numpy()
        vp, vq = hp.vals_p.numpy(), (hp.vals_q.numpy() if hp.vals_q is not None else None)
        for (s, lo, n, off) in blk:
            _io.unpack_scores(codes[off // 16:], chunks[off // _lib.PACK_CHUNK * 24:], vp, vq, n, ps[s][lo:lo + n],
                              qs[s][lo:lo + n] if q is not None else None, want_q=q is not None)
        self.host_unpack_s += time.perf_counter() - t0

    # ------------------------------------------------------------------ q-values across blocks
    def _qvalues(self, n_tests, states, cands, ps, qs, dev_rows):
        """The genome-wide q-value step with the blocks as ranks: candidates selected per block against the global histogram,
        ranked together once, scattered into q_out through the piece map; the p == 1.0 group fixed on the host when its q is
        below 1.  The candidate lists cover every candidate unless the saturation bucket is at or above 2^-5 or a list
        overflowed: then a third sweep selects from p itself, uploaded from p_out."""
        eng, lib, dev = self.eng, self.lib, self.device
        nb = len(self.blocks)
        ns = ctypes.sizeof(_lib.ScoreState)
        st = _lib.stream_ptr()
        self.sel_ws = torch.empty(int(lib.bbk_bh_workspace_bytes(0)), dtype=torch.uint8, device=dev)
        listed = not any(s.cand_overflow for s in states)
        cap = max([int(s.n_cand) for s in states] + [1])
        scratch = None
        for _ in range(4):
            if nb * cap >= (1 << 32):
                raise _lib.BbkError("%d blocks of %d q-value candidates reach 2^32: use larger blocks" % (nb, cap))
            recv = torch.zeros(nb * (cap + 1), dtype=torch.int64, device=dev)
            idx = torch.empty(nb * cap, dtype=torch.int32, device=dev)
            bh_state = torch.zeros(4 * nb, dtype=torch.int64, device=dev)
            q_all = torch.empty(nb * cap, dtype=torch.float64, device=dev)
            q_ones = torch.zeros(2, dtype=torch.float64, device=dev)
            overflow = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = torch.empty(int(lib.bbk_bh_gathered_workspace_bytes(nb, cap)), dtype=torch.uint8, device=dev)
            if scratch is None:
                rows = max(dev_rows)
                scratch = (torch.empty(rows, dtype=torch.float64, device=dev), torch.empty(rows, dtype=torch.float64, device=dev))
            sp, sq = scratch
            for k in range(nb):
                keys = ctypes.c_void_p(recv.data_ptr() + 8 * (k * (cap + 1) + 1))
                kidx = ctypes.c_void_p(idx.data_ptr() + 4 * k * cap)
                kst = ctypes.c_void_p(bh_state.data_ptr() + 32 * k)
                m = dev_rows[k]
                if listed:
                    # p / q are read only when the list does not cover every candidate: that result is discarded below
                    _lib.check(lib.bbk_bh_select_listed(_lib.ptr(sp), m, n_tests, _lib.ptr(eng.p_hist), _lib.ptr(sq), ctypes.byref(cands[k][2]),
                                                        ctypes.c_void_p(self.score_state.data_ptr() + k * ns), keys, kidx, cap, kst,
                                                        _lib.ptr(self.sel_ws), self.sel_ws.numel(), st), "bbk_bh_select_listed")
                    eng.launches += 5           # init, threshold, candidate filter, compact (returns at once), export
                else:
                    self._p_in(k, sp, ps)
                    _lib.check(lib.bbk_bh_select(_lib.ptr(sp), m, n_tests, _lib.ptr(eng.p_hist), _lib.ptr(sq), keys, kidx, cap, kst,
                                                 _lib.ptr(self.sel_ws), self.sel_ws.numel(), st), "bbk_bh_select")
                    eng.launches += 4           # init, threshold, compact, export
                _lib.check(lib.bbk_bh_pack_count(kst, ctypes.c_void_p(recv.data_ptr() + 8 * k * (cap + 1)), st), "bbk_bh_pack_count")
                eng.launches += 1
            _lib.check(lib.bbk_bh_rank_gathered_all(_lib.ptr(recv), nb, cap, _lib.ptr(bh_state), _lib.ptr(q_all), _lib.ptr(q_ones),
                                                    _lib.ptr(overflow), _lib.ptr(ws), ws.numel(), st), "bbk_bh_rank_gathered_all")
            eng.launches += 4                   # prepare, compact, rank, export
            h_state = bh_state.cpu().numpy().view(np.uint64).reshape(nb, 4)
            ov = int(overflow.item())
            if listed and int(h_state[0, 1]) > _SMALL_P_KEY:
                listed = False                  # saturation at or above 2^-5: the lists miss candidates
                continue
            if ov:
                cap = ov                        # the largest block count: every block fits now
                continue
            break
        else:
            raise _lib.BbkError("the q-value step did not settle")
        counts = h_state[:, 0].astype(np.int64)
        self.tau_key, self.n_candidates = int(h_state[0, 1]), int(counts.sum())       # for a caller's checks
        h_q, h_idx = q_all.cpu().numpy(), idx.cpu().numpy().view(np.uint32)
        h_ones = q_ones.cpu().numpy()
        for k, blk in enumerate(self.blocks):
            n = int(counts[k])
            if not n:
                continue
            rows = h_idx[k * cap:k * cap + n].astype(np.int64)
            vals = h_q[k * cap:k * cap + n]
            offs = np.array([off for (_, _, _, off) in blk], dtype=np.int64)
            which = np.searchsorted(offs, rows, side="right") - 1
            for i, (s, lo, pn, off) in enumerate(blk):
                sel = which == i
                if sel.any():
                    qs[s][lo + rows[sel] - off] = vals[sel]
        if h_ones[1] != 0.0:                    # q of the p == 1.0 group is below 1 (N below the number of emitted rows)
            self._fix_ones(ps, qs, float(h_ones[0]))

    def _p_in(self, k, sp, ps):
        """Block k's p from the caller's columns into the device column sp (padding rows NaN), for the pass over p."""
        blk = self.blocks[k]
        self._nan_padding(k, sp, None)
        for (s, lo, n, off) in blk:
            sp[off:off + n].copy_(torch.from_numpy(ps[s][lo:lo + n]), non_blocking=True)
            self.bytes_in += 8 * n

    @staticmethod
    def _fix_ones(ps, qs, q_ones, chunk=1 << 24):
        """q = q_ones wherever p == 1.0, by all host cores (numpy releases the GIL in both calls)."""
        import os
        from concurrent.futures import ThreadPoolExecutor
        jobs = [(p, q, a) for p, q in zip(ps, qs) for a in range(0, len(p), chunk)]

        def one(job):
            p, q, a = job
            np.copyto(q[a:a + chunk], q_ones, where=p[a:a + chunk] == 1.0)

        with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
            list(ex.map(one, jobs))
