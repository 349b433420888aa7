"""Device-side stages of one Fit-Hi-C significance pass (the reference's fithic(), fithic.py:110-133); distributed.GenomePass
enqueues them.

    K1 hist_pairs  ->  [allreduce of the distance table across ranks]  ->  K2/K3 fit (one CTA)
    ->  K4 pvalues  ->  K5 Benjamini-Hochberg q-values (opt-in; the reference writes -1, fithic.py:435)

Everything between the first and last kernel is enqueued on one CUDA stream with no host
synchronisation; S, the spline range and the candidate count of the q-value step stay on the device.
PyTorch is used for device memory, streams and torch.distributed only.
"""
import ctypes

import numpy as np
import torch

from . import _lib


def reduce_distance_stats(obs_sum, totals, group=None):
    """All-reduce K1's outputs across ranks, in place: per-distance sums and the six sum-type totals are
    added, minObservedGenomicDist / maxObservedGenomicDist take min / max (fithic.py:258-259).  Integer
    reductions are independent of the reduction order, so every rank ends with bit-identical tables and
    the fit that follows is replicated deterministically.  No-op without an initialised process group."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    # two collectives: one SUM over [obs_sum | the six sum-type totals], one MAX over [-min, max]
    nk = obs_sum.numel()
    pack = torch.cat([obs_sum, totals[:6]])
    ext = torch.stack([-totals[6], totals[7]])
    dist.all_reduce(pack, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(ext, op=dist.ReduceOp.MAX, group=group)
    obs_sum.copy_(pack[:nk])
    totals[:6] = pack[nk:]
    totals[6] = -ext[0]
    totals[7] = ext[1]


MAX_WORLD = 64          # ranks the packed statistics buffer has min / max slots for


class Shard(object):
    """Contact records of one shard (a chromosome or a diagonal band), as int32 CUDA tensors.

    chr1/chr2 may be None: every record is on chromosome `chrom` (the compact 12 B/pair layout).
    """

    def __init__(self, mid1, mid2, count, chr1=None, chr2=None, chrom=0):
        for t in (mid1, mid2, count, chr1, chr2):
            if t is not None:
                if t.dtype != torch.int32 or not t.is_cuda or not t.is_contiguous():
                    raise ValueError("shard columns must be contiguous int32 CUDA tensors")
        if (chr1 is None) != (chr2 is None):
            raise ValueError("chr1 and chr2 must both be given or both be None")
        self.mid1, self.mid2, self.count, self.chr1, self.chr2 = mid1, mid2, count, chr1, chr2
        self.chrom = int(chrom)
        self.n = int(mid1.numel())
        if mid2.numel() != self.n or count.numel() != self.n:
            raise ValueError("shard columns differ in length")


class BiasTables(object):
    """Dense per-chromosome bias tables on the device (biasDic of fithic.py:136-158).

    values[c]: float64 array over the grid mid0[c] + i*resolution; NaN = locus absent (lookup gives 1.0).
    Out-of-range biases must already be mapped to -1 (read_bias_file does that, fithic.py:147-149).
    """

    def __init__(self, values, mid0, device, step=0):
        """step: distance between neighbouring entries of every table; 0 = the resolution of the pass."""
        self.n_chrom = len(values)
        self.step = int(step)
        base = np.zeros(self.n_chrom + 1, dtype=np.int64)
        for c, v in enumerate(values):
            base[c + 1] = base[c] + len(v)
        flat = np.concatenate([np.asarray(v, dtype=np.float64) for v in values]) if self.n_chrom else np.zeros(0)
        self.bias = torch.from_numpy(flat).to(device)
        self.chrom_base = torch.from_numpy(base).to(device)
        self.mid0 = torch.from_numpy(np.asarray(mid0, dtype=np.int64)).to(device)
        self.struct = _lib.BiasTable(self.bias.data_ptr(), self.chrom_base.data_ptr(), self.mid0.data_ptr(), self.n_chrom, self.step)
        # one flag bit per entry (value < 0 or > 4) for bbk_score_pairs: count <= 0 rows look at two bits, not two values
        lib = _lib.load()
        n = int(self.bias.numel())
        self.flags = torch.zeros(int(lib.bbk_bias_flags_bytes(n)) // 4, dtype=torch.int32, device=device)
        if n:
            with torch.cuda.device(self.bias.device):
                _lib.check(lib.bbk_bias_flags(_lib.ptr(self.bias), n, _lib.ptr(self.flags), _lib.stream_ptr()), "bbk_bias_flags")


class PassEngine(object):
    """Buffers + kernel sequence for one pass over a set of shards resident on this GPU."""

    def __init__(self, resolution, n_bins, min_dist, max_dist, nkeys, device=None, max_bins=None):
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.R = int(resolution)
        self.n_bins = int(n_bins)
        self.min_dist = int(min_dist)
        self.max_dist = int(max_dist)
        self.nkeys = int(nkeys)
        if self.nkeys <= 0:
            raise ValueError("the fragment list gives no genomic distances (nkeys == 0)")
        # more than n_bins bins can come out (fithic.py:208); every distance could close one
        self.max_bins = int(max_bins) if max_bins else max(4, min(self.nkeys, max(4 * self.n_bins, 512)))
        dev = self.device
        self.possible = torch.zeros(self.nkeys, dtype=torch.int64, device=dev)
        # K1's whole output is ONE buffer [obs_sum | totals | 2 x MAX_WORLD slots for the min / max observed distance],
        # so that one SUM all-reduce makes it genome-wide (bbk_stats_pack / bbk_stats_unpack)
        self.stats = torch.zeros(self.nkeys + 8 + 2 * MAX_WORLD, dtype=torch.int64, device=dev)
        self.obs_sum = self.stats[:self.nkeys]
        self.totals = self.stats[self.nkeys:self.nkeys + 8]
        self.fit_result = torch.zeros(ctypes.sizeof(_lib.FitResult), dtype=torch.uint8, device=dev)
        self.x = torch.zeros(self.max_bins, dtype=torch.float64, device=dev)
        self.y = torch.zeros(self.max_bins, dtype=torch.float64, device=dev)
        self.bin_of_key = torch.zeros(self.nkeys, dtype=torch.int32, device=dev)
        self.spline_y = torch.zeros(self.nkeys, dtype=torch.float64, device=dev)
        self.spline_raw = torch.zeros(self.nkeys, dtype=torch.float64, device=dev)
        self.knots = torch.zeros(self.max_bins + 4, dtype=torch.float64, device=dev)
        self.coefs = torch.zeros(self.max_bins + 4, dtype=torch.float64, device=dev)
        ws = int(self.lib.bbk_fit_workspace_bytes(self.max_bins, self.nkeys))
        self.fit_ws = torch.zeros(ws, dtype=torch.uint8, device=dev)
        self.p_hist = torch.zeros(_lib.PHIST_LEN, dtype=torch.int64, device=dev)
        self.bias = None
        self.bh_ws = None
        self.launches = 0

    def grow_bins(self):
        """Room for one bin per distance key (the most fithic.py:188-209 can emit: once S - total reaches 0 every remaining key
        closes a bin).  Returns False when the buffers already have that size."""
        if self.max_bins >= self.nkeys:
            return False
        dev = self.device
        self.max_bins = max(4, self.nkeys)
        self.x = torch.zeros(self.max_bins, dtype=torch.float64, device=dev)
        self.y = torch.zeros(self.max_bins, dtype=torch.float64, device=dev)
        self.knots = torch.zeros(self.max_bins + 4, dtype=torch.float64, device=dev)
        self.coefs = torch.zeros(self.max_bins + 4, dtype=torch.float64, device=dev)
        self.fit_ws = torch.zeros(int(self.lib.bbk_fit_workspace_bytes(self.max_bins, self.nkeys)), dtype=torch.uint8, device=dev)
        return True

    # ------------------------------------------------------------------ setup
    def set_fragments(self, n_frags, max_frag):
        """possible[] from per-chromosome fragment counts (fithic.py:302-311)."""
        nf = torch.tensor(list(n_frags), dtype=torch.int64, device=self.device)
        mf = torch.tensor(list(max_frag), dtype=torch.int64, device=self.device)
        _lib.check(self.lib.bbk_possible_pairs(_lib.ptr(nf), _lib.ptr(mf), len(n_frags), self.R, self.nkeys,
                                               _lib.ptr(self.possible), _lib.stream_ptr()), "bbk_possible_pairs")
        self.launches += 1

    def set_bias(self, tables):
        self.bias = tables

    # ------------------------------------------------------------------ stages
    def fan_out(self, n_jobs):
        """Stream pointers for n_jobs independent per-shard launches of one stage: the current stream and two side streams in
        turn, so that the tail of one shard's persistent kernel overlaps the head of the next (23 chromosomes = 23 tails
        otherwise).  Call fan_in() after the launches."""
        main = torch.cuda.current_stream(self.device)
        if n_jobs <= 1:
            self._fan = None
            return [_lib.stream_ptr(main)] * max(n_jobs, 1)
        if getattr(self, "_sides", None) is None:
            self._sides = [torch.cuda.Stream(self.device) for _ in range(2)]
            self._fan_ev = [torch.cuda.Event() for _ in range(3)]
        self._fan_ev[0].record(main)
        for sd in self._sides:
            sd.wait_event(self._fan_ev[0])
        lanes = [main] + self._sides
        self._fan = main
        return [_lib.stream_ptr(lanes[i % 3]) for i in range(n_jobs)]

    def fan_in(self):
        if getattr(self, "_fan", None) is None:
            return
        for sd, ev in zip(self._sides, self._fan_ev[1:]):
            ev.record(sd)
            self._fan.wait_event(ev)
        self._fan = None

    def hist(self, shards):
        st = _lib.stream_ptr()
        _lib.check(self.lib.bbk_hist_init(_lib.ptr(self.obs_sum), self.nkeys, _lib.ptr(self.totals), st), "bbk_hist_init")
        self.launches += 1
        live = [sh for sh in shards if sh.n]
        for sh, st_i in zip(live, self.fan_out(len(live))):
            _lib.check(self.lib.bbk_hist_pairs(_lib.ptr(sh.chr1), _lib.ptr(sh.chr2), _lib.ptr(sh.mid1), _lib.ptr(sh.mid2),
                                               _lib.ptr(sh.count), sh.n, self.R, self.min_dist, self.max_dist, self.nkeys,
                                               _lib.ptr(self.obs_sum), _lib.ptr(self.totals), st_i), "bbk_hist_pairs")
            self.launches += 1
        self.fan_in()

    def hist_excluding(self, shards, p_list, p_outlier):
        """Second-pass histogram: K1 over the records whose first-pass p is NOT <= p_outlier."""
        st = _lib.stream_ptr()
        _lib.check(self.lib.bbk_hist_init(_lib.ptr(self.obs_sum), self.nkeys, _lib.ptr(self.totals), st), "bbk_hist_init")
        self.launches += 1
        for sh, p in zip(shards, p_list):
            if sh.n == 0:
                continue
            _lib.check(self.lib.bbk_hist_pairs_excluding(_lib.ptr(sh.chr1), _lib.ptr(sh.chr2), _lib.ptr(sh.mid1), _lib.ptr(sh.mid2),
                                                         _lib.ptr(sh.count), _lib.ptr(p), float(p_outlier), sh.n, self.R,
                                                         self.min_dist, self.max_dist, self.nkeys, _lib.ptr(self.obs_sum),
                                                         _lib.ptr(self.totals), st), "bbk_hist_pairs_excluding")
            self.launches += 1

    def allreduce_stats(self, group=None):
        """Sum the distance table and totals over ranks (integers: order-free, bit-exact): one collective on the packed
        buffer, the min / max observed distance travelling in per-rank slots (two one-warp kernels around it)."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return
        world = dist.get_world_size(group)
        if world == 1:
            return
        if world > MAX_WORLD:
            reduce_distance_stats(self.obs_sum, self.totals, group)
            return
        rank, st = dist.get_rank(group), _lib.stream_ptr()
        ext = self.stats[self.nkeys + 8:]
        _lib.check(self.lib.bbk_stats_pack(_lib.ptr(self.totals), _lib.ptr(ext), world, rank, st), "bbk_stats_pack")
        dist.all_reduce(self.stats[:self.nkeys + 8 + 2 * world], op=dist.ReduceOp.SUM, group=group)
        _lib.check(self.lib.bbk_stats_unpack(_lib.ptr(self.totals), _lib.ptr(ext), world, st), "bbk_stats_unpack")
        self.launches += 2

    def fit(self, smoothing=None):
        """K2b + K3.  smoothing: the spline's s when the caller wants to give it (see reference_smoothing); by default the
        kernel uses min(y) * min(y)."""
        if smoothing is not None:
            req = _lib.FitResult()
            req.status = _lib.FIT_S_GIVEN
            req.smoothing = float(smoothing)
            self.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8))
        _lib.check(self.lib.bbk_fit(_lib.ptr(self.possible), _lib.ptr(self.obs_sum), self.nkeys, _lib.ptr(self.totals),
                                    self.n_bins, self.R, self.min_dist, self.max_dist, self.max_bins,
                                    _lib.ptr(self.fit_result), _lib.ptr(self.x), _lib.ptr(self.y), _lib.ptr(self.bin_of_key),
                                    _lib.ptr(self.spline_y), _lib.ptr(self.spline_raw), _lib.ptr(self.knots),
                                    _lib.ptr(self.coefs), _lib.ptr(self.fit_ws), self.fit_ws.numel(), _lib.stream_ptr()),
                   "bbk_fit")
        self.launches += 1

    def _bh_workspace(self, m):
        need = int(self.lib.bbk_bh_workspace_bytes(int(m)))
        if self.bh_ws is None or self.bh_ws.numel() < need:
            self.bh_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self.bh_ws

    def pvalues(self, shard, p_out, with_hist=False):
        """K4.  with_hist: also fill self.p_hist (zero it first)."""
        bias = ctypes.byref(self.bias.struct) if self.bias is not None else None
        _lib.check(self.lib.bbk_pvalues(_lib.ptr(shard.chr1), _lib.ptr(shard.chr2), _lib.ptr(shard.mid1), _lib.ptr(shard.mid2),
                                        _lib.ptr(shard.count), shard.n, shard.chrom, self.R, self.min_dist, self.max_dist,
                                        _lib.ptr(self.fit_result), _lib.ptr(self.spline_y), bias, _lib.ptr(p_out),
                                        _lib.ptr(self.p_hist) if with_hist else None, _lib.stream_ptr()), "bbk_pvalues")
        self.launches += 1

    def qvalues(self, p, q, n_tests=-1):
        """K5 over p, with the histogram K4 left in self.p_hist."""
        m = int(p.numel())
        ws = self._bh_workspace(m)
        _lib.check(self.lib.bbk_bh_qvalues(_lib.ptr(p), m, int(n_tests), _lib.BH_UNSORTED, _lib.ptr(self.p_hist), _lib.ptr(q), None,
                                           _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "bbk_bh_qvalues")
        self.launches += 5       # init, threshold, compact, rank (one cooperative launch), ones fix

    # ------------------------------------------------------------------ results
    @staticmethod
    def reference_smoothing(fit):
        """s exactly as the reference computes it, `min(y)**2` on Python floats (fithic.py:340): that is libm's pow(ymin, 2.0),
        which is one ulp away from the correctly rounded ymin*ymin the kernel computes for about 0.09 % of inputs (glibc 2.39).
        Returns None when the kernel's s (fit.smoothing) already equals it, else the value to pass to fit(smoothing=...).
        min(y) comes back inside the fit result (BbkFitResult.y_min)."""
        if fit.n_out <= 0:
            return None
        s_ref = float(fit.y_min) ** 2
        return None if s_ref == fit.smoothing else s_ref

    @staticmethod
    def decode_fit(raw):
        """BbkFitResult bytes -> FitResult; raises what the reference would raise for a failed fit."""
        res = _lib.FitResult.from_buffer_copy(raw)
        err = _lib.FIT_STATUS.get(res.status, (RuntimeError, "fit stage failed with status %d" % res.status))
        if err is not None:
            raise err[0](err[1])
        return res

    def read_fit(self):
        """Copy the fit status back (synchronises) and raise what the reference would raise."""
        return self.decode_fit(self.fit_result.cpu().numpy().tobytes())


class HostPipeline(object):
    """Successive single-shard passes (one library each, a distributed.GenomePass on this GPU alone) streamed from pinned
    host memory.

    A pass cannot start scoring before all of its records are on the device (S and the spline need the whole
    distance table, fithic.py:110-133), so inside one pass the inbound and the outbound copies never overlap.
    Across passes they do: while library k is being scored and its p/q travel back, library k+1 is already
    arriving.  `slots` device copies of the record columns and of p/q make that legal; three streams (in, run,
    out) and per-slot events order them.  Nothing here synchronises the host; call drain() (or wait on the event
    submit() returns) before reading the host outputs.
    """

    class _Slot(object):
        pass

    def __init__(self, engine, max_pairs, chrom=0, slots=2):
        from .distributed import GenomePass
        self.eng = engine
        self.chrom = int(chrom)
        self.max_pairs = int(max_pairs)
        dev = engine.device
        rows = max((self.max_pairs + 3) & ~3, 4)          # GenomePass.attach: a shard's p / q rows in whole groups of 4
        self.slots = []
        for _ in range(int(slots)):
            s = HostPipeline._Slot()
            s.mid1, s.mid2, s.count = (torch.empty(self.max_pairs, dtype=torch.int32, device=dev) for _ in range(3))
            s.p, s.q = (torch.empty(rows, dtype=torch.float64, device=dev) for _ in range(2))
            s.in_ready, s.run_done, s.out_done = (torch.cuda.Event() for _ in range(3))
            s.fit = torch.zeros_like(engine.fit_result)                      # this pass' BbkFitResult (the engine's is overwritten by the next pass)
            s.h_fit = torch.zeros(engine.fit_result.numel(), dtype=torch.uint8).pin_memory()
            s.index = -1
            self.slots.append(s)
        # Nothing here synchronises, so nothing would see BbkScoreState.overflow: the deferred list has a place for every row
        # of a slot (and later attaches keep it, being no larger).
        self.gp = GenomePass(engine, group=False)
        self.gp.attach([Shard(s.mid1, s.mid2, s.count, chrom=self.chrom)], s.p, s.q, list_capacity=rows)
        self.s_in, self.s_run, self.s_out = (torch.cuda.Stream(dev) for _ in range(3))
        self.s_run.wait_stream(torch.cuda.current_stream(dev))      # the engine's tables were filled there
        self.submitted = 0

    def submit(self, h_mid1, h_mid2, h_count, h_p, h_q=None, n_tests=-1):
        """Enqueue one pass: pinned int32 host columns in, p (and q when h_q is given) back into pinned float64
        host buffers.  Returns the event that fires when the outputs are on the host."""
        n = int(h_mid1.numel())
        if n > self.max_pairs or h_mid2.numel() != n or h_count.numel() != n or h_p.numel() != n:
            raise ValueError("library larger than the pipeline's slots, or columns differ in length")
        for t in (h_mid1, h_mid2, h_count, h_p, h_q):
            if t is not None and not t.is_pinned():
                raise ValueError("host buffers must be pinned (torch.Tensor.pin_memory)")
        s = self.slots[self.submitted % len(self.slots)]
        self.submitted += 1
        self.s_in.wait_event(s.run_done)        # the pass that last read this slot's records has finished
        with torch.cuda.stream(self.s_in):
            s.mid1[:n].copy_(h_mid1, non_blocking=True)
            s.mid2[:n].copy_(h_mid2, non_blocking=True)
            s.count[:n].copy_(h_count, non_blocking=True)
            s.in_ready.record()
        self.s_run.wait_event(s.in_ready)
        self.s_run.wait_event(s.out_done)       # this slot's previous p/q have left the device
        with torch.cuda.stream(self.s_run):
            self.gp.q_values = h_q is not None
            self.gp.attach([Shard(s.mid1[:n], s.mid2[:n], s.count[:n], chrom=self.chrom)], s.p, s.q)
            self.gp.enqueue(n_tests)
            s.fit.copy_(self.eng.fit_result, non_blocking=True)
            s.run_done.record()
        self.s_out.wait_event(s.run_done)
        with torch.cuda.stream(self.s_out):
            h_p.copy_(s.p[:n], non_blocking=True)
            if h_q is not None:
                h_q.copy_(s.q[:n], non_blocking=True)
            s.h_fit.copy_(s.fit, non_blocking=True)
            s.out_done.record()
        s.index = self.submitted - 1
        return s.out_done

    def fit_of(self, index):
        """Fit result of submission `index` (0-based), once its outputs are on the host: raises what the reference would
        raise for that library (ZeroDivisionError, ...), else returns the FitResult - PassEngine.reference_smoothing(result)
        then tells whether the pass has to be submitted again with the reference's own s.  Only the last `slots`
        submissions are kept."""
        s = self.slots[int(index) % len(self.slots)]
        if s.index != int(index):
            raise KeyError("submission %d is no longer (or not yet) held by the pipeline" % int(index))
        s.out_done.synchronize()
        return PassEngine.decode_fit(s.h_fit.numpy().tobytes())

    def drain(self):
        self.s_out.synchronize()
