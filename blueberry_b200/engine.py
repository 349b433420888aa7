"""Device-side stages of one Fit-Hi-C significance pass (the reference's fithic(), fithic.py:110-133): the tables a pass
shares (Shard, BiasTables, PassEngine's possible pairs, distance table and fit buffers) and the launches of its stages.
distributed.GenomePass enqueues them and adds the streaming K4 and K5, the Benjamini-Hochberg q-values (opt-in; the
reference writes -1, fithic.py:435).

    K1 hist_pairs  ->  [allreduce of the distance table across ranks]  ->  K2/K3 fit (one CTA)  ->  K4 pvalues (direct)

Nothing here synchronises the host except read_fit(): S and the spline range stay on the device.
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
            # non_blocking: a pageable source is staged at once, and the stream (HostStream's run stream) is not synchronised
            self.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8), non_blocking=True)
        _lib.check(self.lib.bbk_fit(_lib.ptr(self.possible), _lib.ptr(self.obs_sum), self.nkeys, _lib.ptr(self.totals),
                                    self.n_bins, self.R, self.min_dist, self.max_dist, self.max_bins,
                                    _lib.ptr(self.fit_result), _lib.ptr(self.x), _lib.ptr(self.y), _lib.ptr(self.bin_of_key),
                                    _lib.ptr(self.spline_y), _lib.ptr(self.spline_raw), _lib.ptr(self.knots),
                                    _lib.ptr(self.coefs), _lib.ptr(self.fit_ws), self.fit_ws.numel(), _lib.stream_ptr()),
                   "bbk_fit")
        self.launches += 1

    def pvalues(self, shard, p_out, with_hist=False):
        """K4.  with_hist: also fill self.p_hist (zero it first)."""
        bias = ctypes.byref(self.bias.struct) if self.bias is not None else None
        _lib.check(self.lib.bbk_pvalues(_lib.ptr(shard.chr1), _lib.ptr(shard.chr2), _lib.ptr(shard.mid1), _lib.ptr(shard.mid2),
                                        _lib.ptr(shard.count), shard.n, shard.chrom, self.R, self.min_dist, self.max_dist,
                                        _lib.ptr(self.fit_result), _lib.ptr(self.spline_y), bias, _lib.ptr(p_out),
                                        _lib.ptr(self.p_hist) if with_hist else None, _lib.stream_ptr()), "bbk_pvalues")
        self.launches += 1

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
