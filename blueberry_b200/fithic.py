"""Drop-in for blueberry/fithic.py - same names, argument order, files and return types - with the
work done by the sm_100a kernels of libbbk.so.

Reference entry points mirrored here (paths relative to the reference root):
    FitHiC(libname, resolution, n_bins=100, n_passes=2, max_dist=-1, min_dist=-1)   fithic.py:49-83
    FitHiC.fit_transform(interactions, fragments, biases="none", verbose=False)      fithic.py:85-108
    fithic(libname, resolution, n_bins, min_dist, max_dist, n_passes, interactions, frags, biases, verbose)  :110
    generate_FragPairs / read_bias_file / read_interactions / calculate_probabilities / fit_spline
    in_range_check(interactionDistance, min_dist, max_dist)                           fithic.py:445
    benjamini_hochberg_correction(p_values, num_total_tests)                          fithic.py:466

Added (the reference parses gzip text line by line; that is not GPU work):
    FitHiC.fit_transform_arrays(...) -> PassOutput      records in / p (and q) out as arrays

Deliberate deviations (SURVEY.md section 0): the reference keeps all totals in module globals that
are never reset (fithic.py:25-42), so a second call in one process accumulates onto the first; here
every generate_FragPairs starts from the initial values (fresh-process semantics).  The module
attributes of the same names are still updated after each stage.  n_passes is accepted and ignored,
as in the reference (fithic.py:121-133 runs one pass).  No PNG is drawn.

There is no CPU fallback: without libbbk.so and a CUDA device these functions raise.
"""
import gzip
import sys

import numpy as np
import torch

from . import _io, _lib
from .engine import BiasTables, PassEngine, Shard

# ---- module globals of the reference (fithic.py:25-45), refreshed by the stage functions ----
possibleIntraInRangeCount = 0
observedIntraInRangeCount = 0
observedIntraInRangeSum = 0
possibleIntraAllCount = 0
observedIntraAllCount = 0
observedIntraAllSum = 0
possibleInterAllCount = 0
observedInterAllCount = 0
observedInterAllSum = 0
baselineIntraChrProb = 0
interChrProb = 0
minObservedGenomicDist = 500000000
maxObservedGenomicDist = 0
maxPossibleGenomicDist = 0
distScaling = 10000.0

_this = sys.modules[__name__]


def _device():
    if not torch.cuda.is_available():
        raise _lib.BbkError("blueberry_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def in_range_check(interactionDistance, min_dist, max_dist):
    """fithic.py:445-449."""
    if (min_dist == -1 or (min_dist > -1 and interactionDistance > min_dist)) and \
            (max_dist == -1 or (max_dist > -1 and interactionDistance <= max_dist)):
        return True
    return False


# =================================================================================================
# text ingest (host): the reference's three gzip formats -> arrays
# =================================================================================================
class _ChromIds(object):
    """Chromosome name -> small integer id (order of first appearance)."""

    def __init__(self):
        self.ids = {}
        self.names = []

    def encode(self, names):
        uniq, inv = np.unique(np.asarray(names, dtype=object), return_inverse=True)
        lut = np.empty(len(uniq), dtype=np.int32)
        for i, u in enumerate(uniq):
            if u not in self.ids:
                self.ids[u] = len(self.names)
                self.names.append(u)
            lut[i] = self.ids[u]
        return lut[inv]


def _read_table(path, ncols):
    import pandas as pd
    # whitespace split like str.split() (fithic.py:143,245,288); too few columns -> ValueError like the unpack
    df = pd.read_csv(path, sep=r"\s+", header=None, compression="gzip", dtype=str, engine="c")
    if df.shape[1] < ncols:
        raise ValueError("not enough values to unpack (expected %d, got %d)" % (ncols, df.shape[1]))
    return df


def _parse_fragments(path, chroms):
    df = _read_table(path, 2)                                  # fithic.py:288: first two columns
    return chroms.encode(df[0].values), df[1].values.astype(np.int64)


def _parse_interactions(path, chroms):
    """fithic.py:243-247 on the whole file, by the native reader (libbbkio.so, include/bbk_io.h)."""
    from . import _io
    names, c1, m1, c2, m2, cnt = _io.read_interactions(path)
    lut = chroms.encode(names) if names else np.zeros(0, dtype=np.int32)
    return lut[c1], m1, lut[c2], m2, cnt


# =================================================================================================
# fragments -> possible pairs (host bookkeeping, device table)
# =================================================================================================
class _FragInfo(object):
    __slots__ = ("n_frags", "max_frag", "n_total", "max_possible", "nkeys", "possible_inter_all", "possible_intra_all")


def _frag_info(frag_chrom, frag_mid, resolution):
    """Per-chromosome fragment counts and the derived totals (fithic.py:284-318)."""
    R = int(resolution)
    frag_chrom = np.asarray(frag_chrom)
    frag_mid = np.asarray(frag_mid, dtype=np.int64)
    info = _FragInfo()
    info.n_frags, info.max_frag = [], []
    n_total, max_possible = 0, 0                               # module global starts at 0 (:42)
    # allFragsDic[chr] is a dict keyed by mid: duplicates collapse (:289-291)
    key = frag_chrom.astype(np.int64) * (1 << 40) + (frag_mid + (1 << 39))
    uniq = np.unique(key)
    uc = (uniq >> 40).astype(np.int64)
    um = (uniq & ((1 << 40) - 1)) - (1 << 39)
    for c in np.unique(uc):
        sel = um[uc == c]
        n = int(sel.size)
        mf = int(sel.max()) - R // 2                           # :298 (py2 integer division)
        info.n_frags.append(n)
        info.max_frag.append(mf)
        n_total += n
        max_possible = max(max_possible, mf)                   # :300
    inter, intra = 0, 0
    for n in info.n_frags:
        inter += n * (n_total - n)                             # :313
        intra += (n * (n + 1)) // 2                            # :314
    info.n_total = n_total
    info.max_possible = max_possible
    info.nkeys = len(range(0, max_possible + 1, R))            # :302
    info.possible_inter_all = inter // 2                       # :316
    info.possible_intra_all = intra
    return info


MAX_BIAS_ENTRIES = 1 << 27          # dense bias tables: at most 1 GiB of float64


def _bias_tables(bias_dic, resolution, device, n_chrom_hint=0):
    """biasDic {chrom id: {mid: bias}} -> dense device tables on the grid mid0 + i*step.  Loci on the fragment grid (the usual
    bias file) give step = resolution; any other set of loci is put on the coarsest grid that holds them all (the gcd of their
    offsets and the resolution), so that biasDic[chr][mid] (fithic.py:418-425) finds exactly the loci of the file."""
    R = int(resolution)
    n_chrom = max([n_chrom_hint] + [c + 1 for c in bias_dic])
    per_chrom, step = [], R
    for c in range(n_chrom):
        sub = bias_dic.get(c)
        if not sub:
            per_chrom.append(None)
            continue
        if isinstance(sub, tuple):                               # (mids, values) arrays, first occurrences only
            mids, vals = sub
        else:
            mids = np.fromiter(sub.keys(), dtype=np.int64, count=len(sub))
            vals = np.fromiter(sub.values(), dtype=np.float64, count=len(sub))
        # a NaN bias makes the reference's prior NaN and the row is dropped (fithic.py:431-434); NaN is the table's "no such
        # locus" mark, so such a value is stored as +inf: the prior comes out as +-inf or NaN and the row is dropped all the same
        vals = np.where(np.isnan(vals), np.inf, vals)
        m0 = int(mids.min())
        off = mids - m0
        step = int(np.gcd.reduce(np.concatenate([[step], off[off > 0]]))) if (off > 0).any() else step
        per_chrom.append((m0, off, vals))
    total = sum(int(off.max() // step) + 1 for (m0, off, vals) in (x for x in per_chrom if x is not None))
    if total > MAX_BIAS_ENTRIES:
        raise NotImplementedError("the bias loci only share a %d-bp grid: the dense device bias tables would need %d entries "
                                  "(limit %d)" % (step, total, MAX_BIAS_ENTRIES))
    values, mid0 = [], []
    for x in per_chrom:
        if x is None:
            values.append(np.zeros(0))
            mid0.append(0)
            continue
        m0, off, vals = x
        tab = np.full(int(off.max() // step) + 1, np.nan)
        tab[off // step] = vals
        values.append(tab)
        mid0.append(m0)
    return BiasTables(values, mid0, device, step=0 if step == R else step)


# =================================================================================================
# the array entry point
# =================================================================================================
class PassOutput(object):
    """Everything one pass produces, as numpy arrays / Python scalars."""
    __slots__ = ("p", "q", "keep", "x", "y", "spline_x", "spline_y", "spline_y_raw", "residual", "possible",
                 "observed", "bin_of_key", "totals", "frag", "fit", "gpu_launches", "p_first", "rows")


def _pad16(n):
    return (n + 1) & ~1          # float64 slices must stay 16-byte aligned


_STAGE_BYTES = 64 << 20
_stage = {}


def _staging(dev):
    """Two pinned staging buffers per device (allocated once): chunk k+1 is converted / copied into one of them by the
    host while the DMA of chunk k from the other is still running."""
    key = str(dev)
    if key not in _stage:
        _stage[key] = ([torch.empty(_STAGE_BYTES, dtype=torch.uint8).pin_memory() for _ in range(2)],
                       [torch.cuda.Event() for _ in range(2)])
    return _stage[key]


def _to_device_i32(a, dev, lo=0, hi=None):
    """Rows [lo, hi) of an integer column -> int32 CUDA tensor.  Pinned int32 torch tensors go by one asynchronous DMA;
    numpy / pageable input is staged through pinned memory in chunks (conversion to int32 and the DMA overlap).  Values that
    do not fit int32 raise OverflowError (checked per chunk, only for inputs wider than 32 bits)."""
    if isinstance(a, torch.Tensor):
        t = a[lo:hi]
        if t.is_cuda:
            return t.to(dev, dtype=torch.int32).contiguous()
        if t.dtype == torch.int32 and t.is_pinned():
            return t.to(dev, non_blocking=True)
        a, lo, hi = t.numpy(), 0, None
    a = np.asarray(a)
    a = a[lo:hi]
    if a.dtype.kind not in "iu":
        a = a.astype(np.int64)
    n = int(a.shape[0])
    out = torch.empty(max(n, 1), dtype=torch.int32, device=dev)[:n]
    if n == 0:
        return out
    wide = a.dtype.itemsize > 4 or a.dtype == np.uint32
    bufs, evs = _staging(dev)
    per = _STAGE_BYTES // 4
    stream = torch.cuda.current_stream(dev)
    for k, start in enumerate(range(0, n, per)):
        stop = min(n, start + per)
        chunk = a[start:stop]
        if wide and chunk.size and (chunk.min() < -2**31 or chunk.max() >= 2**31):
            raise OverflowError("coordinates / counts must fit in int32 on the device")
        buf, ev = bufs[k & 1], evs[k & 1]
        if k >= 2:
            ev.synchronize()                                   # the DMA that last read this buffer has finished
        h = buf[:4 * (stop - start)].view(torch.int32)
        if chunk.dtype == np.int32 and chunk.flags.c_contiguous:
            _io.copy_bytes(h.data_ptr(), chunk.ctypes.data, 4 * (stop - start))     # all cores: one thread's memcpy is half the link
        else:
            np.copyto(h.numpy(), chunk, casting="unsafe")
        out[start:stop].copy_(h, non_blocking=True)
        ev.record(stream)
    for ev in evs:
        ev.synchronize()
    return out


def _rows_to_shards(chr1, mid1, chr2, mid2, count, lo, hi, dev, max_runs=64):
    """Rows [lo, hi) of the record table as device shards.  Input sorted by chromosome (the usual case, and what the
    authors' per-chromosome files are, datatypes.pyx:26) falls into a few runs of intra-chromosomal rows: each run is a
    shard in the compact 12 B/pair layout, as a view (row order is kept, so p / q line up with the input).  Anything
    else - inter-chromosomal rows, interleaved chromosomes - is one shard with chromosome columns."""
    m1, m2, cn = (_to_device_i32(a, dev, lo, hi) for a in (mid1, mid2, count))
    n = int(m1.numel())
    if chr1 is None:
        return [Shard(m1, m2, cn, chrom=0)]
    c1 = np.asarray(chr1)[lo:hi]
    c2 = np.asarray(chr2)[lo:hi]
    if n == 0:
        return [Shard(m1, m2, cn, chrom=0)]
    if np.array_equal(c1, c2):
        cuts = np.flatnonzero(c1[1:] != c1[:-1]) + 1
        # a run must start on a 16-byte boundary to be a view: 4-record alignment of every cut
        if len(cuts) < max_runs and not (cuts & 3).any():
            bounds = [0] + cuts.tolist() + [n]
            return [Shard(m1[a:b], m2[a:b], cn[a:b], chrom=int(c1[a])) for a, b in zip(bounds[:-1], bounds[1:])]
        if len(cuts) == 0:
            return [Shard(m1, m2, cn, chrom=int(c1[0]))]
        if len(cuts) < max_runs:
            # unaligned cuts: give every run its own (aligned) copy on the device
            bounds = [0] + cuts.tolist() + [n]
            return [Shard(m1[a:b].clone(), m2[a:b].clone(), cn[a:b].clone(), chrom=int(c1[a])) for a, b in zip(bounds[:-1], bounds[1:])]
    return [Shard(m1, m2, cn, _to_device_i32(c1, dev), _to_device_i32(c2, dev))]


_out_pinned = {}


def _pinned_cache(dev, name, nbytes):
    """A pinned host buffer of at least nbytes, kept per device and purpose (pinning memory costs more than the copy)."""
    key = (str(dev), name)
    buf = _out_pinned.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8).pin_memory()
        _out_pinned[key] = buf
    return buf


def _scores_to_host(p_rows, q_rows, dev):
    """The pass' p / q columns as numpy arrays, plus keep = (p <= 1): packed on the device (bbk_pack_scores: two bits per row +
    the values that are not 1.0 / NaN), moved through pinned buffers that are allocated once, unpacked by all host cores."""
    from .distributed import DevicePack
    n = int(p_rows.numel())
    p = np.empty(n, dtype=np.float64)
    q = np.empty(n, dtype=np.float64) if q_rows is not None else None
    keep = np.empty(n, dtype=np.bool_)
    if n == 0:
        return p, q, keep
    if p_rows.data_ptr() & 15 or (q_rows is not None and q_rows.data_ptr() & 15):
        p_rows = p_rows.clone()
        q_rows = q_rows.clone() if q_rows is not None else None
    for caps in ((None, None), (n, n)):          # on overflow: every row carries a value, lists as long as the columns
        pk = DevicePack(n, dev, q_rows is not None, *caps)
        pk.pack(p_rows, q_rows)
        ps = _lib.PackState.from_buffer_copy(pk.state.cpu().numpy().tobytes())
        if not ps.overflow:
            break
    n_p, n_q = int(ps.n_p), int(ps.n_q)
    words, nch = pk.codes.numel(), pk.chunks.numel() // 24
    h_codes = _pinned_cache(dev, "codes", 4 * words)[:4 * words].view(torch.int32)
    h_chunks = _pinned_cache(dev, "chunks", 24 * nch)[:24 * nch]
    h_vp = _pinned_cache(dev, "vals_p", 8 * max(n_p, 1))[:8 * max(n_p, 1)].view(torch.float64)
    h_vq = _pinned_cache(dev, "vals_q", 8 * max(n_q, 1))[:8 * max(n_q, 1)].view(torch.float64)
    h_codes.copy_(pk.codes, non_blocking=True)
    h_chunks.copy_(pk.chunks, non_blocking=True)
    if n_p:
        h_vp[:n_p].copy_(pk.vals_p[:n_p], non_blocking=True)
    if n_q:
        h_vq[:n_q].copy_(pk.vals_q[:n_q], non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    _io.unpack_scores(h_codes.numpy(), h_chunks.numpy(), h_vp.numpy(), h_vq.numpy() if q_rows is not None else None, n, p, q,
                      want_q=q_rows is not None, keep_out=keep.view(np.uint8))
    return p, q, keep


def _to_host(t):
    """Device tensor -> numpy through pinned memory (asynchronous; synchronise before reading)."""
    h = torch.empty(t.shape, dtype=t.dtype).pin_memory()
    h.copy_(t, non_blocking=True)
    return h


def _in_range_possible(possible, resolution, min_dist, max_dist):
    d = np.arange(len(possible), dtype=np.int64) * int(resolution)
    ok = np.ones(len(possible), bool)
    ok &= (d > min_dist) if min_dist > -1 else (np.full(len(possible), min_dist == -1))
    ok &= (d <= max_dist) if max_dist > -1 else (np.full(len(possible), max_dist == -1))
    return int(sum(int(v) for v in np.asarray(possible)[ok]))


def _run_pass(resolution, n_bins, min_dist, max_dist, frag_chrom, frag_mid, chr1, mid1, chr2, mid2, count,
              bias_dic=None, want_q=False, n_tests=None, keep_device=False, refit=False, group=None):
    from .distributed import GenomePass, _world, shard_rows
    dev = _device()
    info = _frag_info(frag_chrom, frag_mid, resolution)
    eng = PassEngine(resolution, n_bins, min_dist, max_dist, info.nkeys, dev)
    eng.set_fragments(info.n_frags, info.max_frag)
    if bias_dic:
        eng.set_bias(_bias_tables(bias_dic, resolution, dev))
    group = False if group is None else (None if group is True else group)      # None: this GPU alone; True: the default group
    world, rank = _world(group)
    n_rows = int(len(mid1))
    lo, hi = shard_rows(n_rows, world, rank)
    nt = -1 if n_tests is None else int(n_tests)
    first = None
    if refit:
        if world > 1:
            raise NotImplementedError("refit=True runs on one GPU")
        same = chr1 is None or (np.asarray(chr1) == np.asarray(chr2)).all() and np.unique(np.asarray(chr1)).size <= 1
        if same:
            chrom = int(np.asarray(chr1).flat[0]) if chr1 is not None and len(chr1) else 0
            shard = Shard(_to_device_i32(mid1, dev), _to_device_i32(mid2, dev), _to_device_i32(count, dev), chrom=chrom)
        else:
            shard = Shard(_to_device_i32(mid1, dev), _to_device_i32(mid2, dev), _to_device_i32(count, dev),
                          _to_device_i32(chr1, dev), _to_device_i32(chr2, dev))
        # pass 1 without q-values, then the refit on the non-outliers scores every record again.  (GenomePass.finish repeats a
        # pass with the reference's own s when the kernel's min(y) * min(y) is not libm's min(y)**2: one ulp off for ~0.09 % of inputs.)
        gp1 = GenomePass(eng, group=False, q_values=False)
        gp1.attach([shard])
        gp1.run()
        in_rng = _in_range_possible(eng.possible.cpu().numpy(), resolution, min_dist, max_dist)
        if in_rng <= 0:
            raise ZeroDivisionError("float division by zero (possibleIntraInRangeCount == 0)")
        gp2 = GenomePass(eng, group=False, q_values=want_q)
        gp2.attach([shard])
        fit = gp2.run(n_tests=nt, exclude=(gp1.p, 1.0 / in_rng))      # raises what the reference would raise
        first = gp1.shard_p(0)
        p_rows, q_rows = gp2.shard_p(0), (gp2.shard_q(0) if want_q else None)
    else:
        gp = GenomePass(eng, group=group, q_values=want_q)
        shards = _rows_to_shards(chr1, mid1, chr2, mid2, count, lo, hi, dev)
        gp.attach(shards)
        fit = gp.run(n_tests=nt)                                # raises what the reference would raise
        if len(shards) == 1:
            p_rows, q_rows = gp.shard_p(0), (gp.shard_q(0) if want_q else None)
        else:                                                   # drop the alignment padding between the runs
            p_rows = torch.cat([gp.shard_p(i) for i in range(len(shards))])
            q_rows = torch.cat([gp.shard_q(i) for i in range(len(shards))]) if want_q else None

    out = _pass_output(eng, fit, info, resolution, min_dist, max_dist, p_rows, q_rows if want_q else None, first, dev)
    out.rows = (lo, hi)
    return out


def _pass_output(eng, fit, info, resolution, min_dist, max_dist, p_rows, q_rows, first, dev):
    """PassOutput of one finished pass: the engine's tables and fit, p / q / keep of the given rows."""
    out = PassOutput()
    out.fit = fit
    out.frag = info
    host = {"x": _to_host(eng.x[:fit.n_out]), "y": _to_host(eng.y[:fit.n_out]),
            "spline_y": _to_host(eng.spline_y[:fit.L]), "spline_raw": _to_host(eng.spline_raw[:fit.L]),
            "possible": _to_host(eng.possible), "observed": _to_host(eng.obs_sum), "bin_of_key": _to_host(eng.bin_of_key),
            "totals": _to_host(eng.totals), "first": _to_host(first) if first is not None else None}
    out.p, out.q, out.keep = _scores_to_host(p_rows, q_rows, dev)    # keep: fithic.py:434 (NaN = not scored or dropped)
    torch.cuda.current_stream(dev).synchronize()
    out.x = host["x"].numpy()
    out.y = host["y"].numpy()
    out.spline_x = (np.arange(fit.L, dtype=np.int64) + fit.k0) * int(resolution)
    out.spline_y = host["spline_y"].numpy()
    out.spline_y_raw = host["spline_raw"].numpy()
    out.residual = float(fit.residual)
    out.possible = host["possible"].numpy()
    out.observed = host["observed"].numpy()
    out.bin_of_key = host["bin_of_key"].numpy()
    t = host["totals"].numpy()
    out.totals = {
        "observedIntraInRangeSum": int(t[0]), "observedIntraInRangeCount": int(t[1]),
        "observedIntraAllSum": int(t[2]), "observedIntraAllCount": int(t[3]),
        "observedInterAllSum": int(t[4]), "observedInterAllCount": int(t[5]),
        "minObservedGenomicDist": int(t[6]), "maxObservedGenomicDist": int(t[7]),
        "maxPossibleGenomicDist": info.max_possible,
        "possibleIntraAllCount": info.possible_intra_all, "possibleInterAllCount": info.possible_inter_all,
        "possibleIntraInRangeCount": _in_range_possible(out.possible, resolution, min_dist, max_dist),
    }
    out.gpu_launches = eng.launches
    out.p_first = host["first"].numpy() if first is not None else None
    return out


def split_chromosomes(chr1, chr2, frag_chrom, n_tests=None, refit=False, group=None):
    """The argument checks and the input split of fit_transform_arrays(per_chromosome=True), on the host alone.

    Returns [(chrom, lo, hi, frag_rows, n_tests_c)] in ascending chromosome order: the chromosome's rows are rows [lo, hi)
    of the record table, its fragments are frag_rows (indices into frag_chrom) and n_tests_c its N (None: its own number of
    emitted rows).  n_tests: None, one value for every chromosome, or a mapping {chrom: n} (a chromosome it does not name
    gets None).  Raises ValueError for inter-chromosomal rows or a chromosome whose rows are not contiguous, and
    NotImplementedError for refit=True or a process group."""
    if group is not None:
        raise NotImplementedError("per_chromosome=True runs on one GPU (group must be None)")
    if refit:
        raise NotImplementedError("per_chromosome=True does not take refit=True")
    if chr1 is None or chr2 is None:
        raise ValueError("per_chromosome=True needs the chromosome columns chr1 and chr2")
    c1, c2 = np.asarray(chr1), np.asarray(chr2)
    if c1.shape != c2.shape or c1.ndim != 1:
        raise ValueError("chr1 and chr2 must be one-dimensional and of the same length")
    bad = np.flatnonzero(c1 != c2)
    if bad.size:
        raise ValueError("per_chromosome=True takes intra-chromosomal rows only; row %d has chr1 %d and chr2 %d"
                         % (bad[0], c1[bad[0]], c2[bad[0]]))
    n = int(c1.size)
    if n == 0:
        return []
    cuts = np.flatnonzero(c1[1:] != c1[:-1]) + 1
    starts = np.concatenate([[0], cuts]).astype(np.int64)
    ends = np.concatenate([cuts, [n]]).astype(np.int64)
    ids = c1[starts].astype(np.int64)
    uniq, cnt = np.unique(ids, return_counts=True)
    if (cnt > 1).any():
        raise ValueError("the rows of chromosome %d are not contiguous: per_chromosome=True needs every chromosome's rows "
                         "in one block" % uniq[cnt > 1][0])
    fc = np.asarray(frag_chrom)
    mapping = hasattr(n_tests, "keys")
    if mapping:
        n_tests = {int(k): v for k, v in n_tests.items()}
    plan = []
    for j in np.argsort(ids, kind="stable"):
        c = int(ids[j])
        nt = n_tests.get(c) if mapping else n_tests
        plan.append((c, int(starts[j]), int(ends[j]), np.flatnonzero(fc == c), None if nt is None else int(nt)))
    return plan


def naming_chromosome(e, chrom):
    """An exception of the type of e whose message starts with the chromosome it is about (e itself when its type does not
    take a message); .chrom holds the id."""
    try:
        err = type(e)("chromosome %d: %s" % (chrom, e))
    except Exception:
        err = e
    err.chrom = int(chrom)
    return err


def _own_bias_step(sub, resolution):
    """The grid step _bias_tables would give a chromosome's bias loci on their own."""
    mids = np.asarray(sub[0], dtype=np.int64)
    off = mids - mids.min()
    R = int(resolution)
    return int(np.gcd.reduce(np.concatenate([[R], off[off > 0]]))) if (off > 0).any() else R


def _run_per_chromosome(resolution, n_bins, min_dist, max_dist, frag_chrom, frag_mid, chr1, mid1, chr2, mid2, count, bias,
                        want_q, n_tests, refit, group):
    """fit_transform_arrays(per_chromosome=True): {chrom: PassOutput}, each equal to the call for that chromosome alone.
    Chromosomes go through one distributed.ChromosomePass when the streaming K4 applies to them (the distance limits allow it
    and their bias loci lie on the fragment grid, as they would alone); the others, and every chromosome when the limits do
    not allow it, through single calls."""
    from .distributed import ChromosomePass
    plan = split_chromosomes(chr1, chr2, frag_chrom, n_tests, refit, group)
    if not plan:
        return {}
    R = int(resolution)
    fc, fm = np.asarray(frag_chrom), np.asarray(frag_mid)
    c1, c2 = np.asarray(chr1), np.asarray(chr2)
    bias_all = _bias_dict_from_arrays(*bias) if bias is not None else {}

    def bias_of(c):
        return {c: bias_all[c]} if c in bias_all else None

    def single(c, lo, hi, fsel, nt):
        out = _run_pass(R, n_bins, min_dist, max_dist, fc[fsel], fm[fsel], c1[lo:hi], mid1[lo:hi], c2[lo:hi], mid2[lo:hi],
                        count[lo:hi], bias_of(c), want_q=want_q, n_tests=nt)
        out.rows = (lo, hi)
        return out

    listed = 0 <= min_dist <= max_dist and max_dist + R < (1 << 31) and R >= 2
    batch = [x for x in plan if listed and len(x[3]) and (x[0] not in bias_all or _own_bias_step(bias_all[x[0]], R) == R)]
    out, failed = {}, None
    if batch:
        dev = _device()
        tables = None
        if any(x[0] in bias_all for x in batch):
            try:
                tables = _bias_tables({x[0]: bias_all[x[0]] for x in batch if x[0] in bias_all}, R, dev)
            except NotImplementedError:              # together the tables are too large: one chromosome at a time
                batch = []
    if batch:
        engines, shards, infos = [], [], []
        for c, lo, hi, fsel, nt in batch:
            info = _frag_info(fc[fsel], fm[fsel], R)
            eng = PassEngine(R, n_bins, min_dist, max_dist, info.nkeys, dev)
            eng.set_fragments(info.n_frags, info.max_frag)
            if tables is not None:
                eng.set_bias(tables)
            cols = []
            for a in (mid1, mid2, count):
                t = _to_device_i32(a, dev, lo, hi)
                cols.append(t.clone() if t.data_ptr() & 15 else t)     # the streaming K4 reads 16-byte aligned columns
            engines.append(eng)
            shards.append(Shard(*cols, chrom=c))
            infos.append(info)
        cp = ChromosomePass(engines, shards, q_values=want_q)
        try:
            fits = cp.run([-1 if x[4] is None else x[4] for x in batch])
        except Exception as e:
            if getattr(e, "chrom", None) is None:
                raise
            failed = (e.chrom, e)
        else:
            launches = cp.launches + sum(e.launches for e in engines)
            for i, (c, lo, hi, fsel, nt) in enumerate(batch):
                o = _pass_output(engines[i], fits[i], infos[i], R, min_dist, max_dist, cp.chrom_p(i),
                                 cp.chrom_q(i) if want_q else None, None, dev)
                o.rows = (lo, hi)
                o.gpu_launches = launches
                out[c] = o
    in_batch = set(x[0] for x in batch)
    for c, lo, hi, fsel, nt in plan:
        if c in in_batch:
            continue
        if failed is not None and c > failed[0]:
            break
        try:
            out[c] = single(c, lo, hi, fsel, nt)
        except Exception as e:
            raise naming_chromosome(e, c)
    if failed is not None:
        raise failed[1]
    return {c: out[c] for c, _, _, _, _ in plan}


class FitHiC(object):
    """Fit-Hi-C transformer object (fithic.py:49-108) - same constructor, same fit_transform."""

    def __init__(self, libname, resolution, n_bins=100, n_passes=2, max_dist=-1, min_dist=-1):
        self.libname = libname
        self.resolution = resolution
        self.n_bins = n_bins
        self.n_passes = n_passes
        self.max_dist = max_dist if max_dist != -1 else 10000000     # fithic.py:82
        self.min_dist = min_dist if min_dist != -1 else 0            # fithic.py:83

    def fit_transform(self, interactions, fragments, biases="none", verbose=False):
        """Paths in, files out, returns None - exactly fithic.py:85-108."""
        fithic(self.libname, self.resolution, self.n_bins, self.min_dist, self.max_dist, self.n_passes,
               interactions, fragments, biases, verbose)

    def fit_transform_arrays(self, chr1, mid1, chr2, mid2, count, frag_chrom, frag_mid, bias=None,
                             q_values=False, n_tests=None, refit=False, group=None, per_chromosome=False):
        """The same pass on in-memory records.

        chr1/chr2: integer chromosome ids per record (None: all records on one chromosome).
        bias: None or (bias_chrom, bias_mid, bias_value) arrays in file order (fithic.py:143).
        q_values: also compute Benjamini-Hochberg q-values over the emitted rows (the reference
        writes the literal -1, fithic.py:435); n_tests defaults to the number of emitted rows.
        refit: second pass (BASELINE config 4).  The reference accepts n_passes and never uses it
        (fithic.py:121-133); with refit=True the rows of pass 1 with p <= 1/possibleIntraInRangeCount are
        left out of the statistics, the bins and spline are refitted with the reference's own stage
        semantics and every record is scored again (p_first keeps the pass-1 values).
        group: under torch.distributed (one process per GPU, every rank passing the SAME arrays) rank r scores rows
        shard_rows(n, world, r) of the table - PassOutput.rows says which, p / q / keep cover those rows only; the
        distance table, S, the bins and the spline are genome-wide (one all-reduce), and so are the q-values
        (distributed.GenomePass).  group=True: the default process group; or any ProcessGroup; None = this GPU alone.
        per_chromosome: Fit-Hi-C once per chromosome, as the authors ran it (one run per chromosome, datatypes.pyx:26).
        Returns {chrom id: PassOutput}; out[c] equals this call on c's rows, c's fragments and c's bias rows alone (every
        field but gpu_launches, which counts the whole pass), and out[c].rows is the range of c's rows in the input.
        n_tests may then also be a mapping {chrom: n}.  Every chromosome's rows must be one contiguous block and
        intra-chromosomal (else ValueError); refit and group are not supported (NotImplementedError).  With the streaming
        K4 (0 <= min_dist <= max_dist, max_dist + resolution < 2^31) every chromosome's fit runs in one launch and the
        q-values in one step (distributed.ChromosomePass); otherwise it is the loop of single calls.  A chromosome whose
        call alone would raise makes this call raise the same exception type, naming the chromosome (lowest id first).
        """
        if per_chromosome:
            return _run_per_chromosome(self.resolution, self.n_bins, self.min_dist, self.max_dist, frag_chrom, frag_mid, chr1,
                                       mid1, chr2, mid2, count, bias, q_values, n_tests, refit, group)
        bias_dic = None
        if bias is not None:
            bias_dic = _bias_dict_from_arrays(*bias)
        return _run_pass(self.resolution, self.n_bins, self.min_dist, self.max_dist, frag_chrom, frag_mid,
                         chr1, mid1, chr2, mid2, count, bias_dic, want_q=q_values, n_tests=n_tests, refit=refit, group=group)


def _bias_dict_from_arrays(bias_chrom, bias_mid, bias_val):
    """read_bias_file on arrays: out-of-[0.5,2] -> -1 (:147-149), first occurrence wins (:153-154)."""
    bias_chrom = np.asarray(bias_chrom)
    bias_mid = np.asarray(bias_mid, dtype=np.int64)
    v = np.asarray(bias_val, dtype=np.float64).copy()
    v[(v < 0.5) | (v > 2)] = -1.0
    out = {}
    key = bias_chrom.astype(np.int64) * (1 << 40) + (bias_mid + (1 << 39))
    _, first = np.unique(key, return_index=True)
    first = np.sort(first)
    ch = bias_chrom[first].astype(np.int64)
    for c in np.unique(ch):
        sel = first[ch == c]
        out[int(c)] = (bias_mid[sel], v[sel])                    # arrays instead of a dict per chromosome (_bias_tables takes both)
    return out


# =================================================================================================
# the path-based pass and the reference's stage functions
# =================================================================================================
class _Session(object):
    """State the reference keeps in module globals between its stage functions."""
    chroms = None
    frag = None
    frag_arrays = None
    contacts = None
    result = None


_session = _Session()


def _publish(**kw):
    for k, v in kw.items():
        setattr(_this, k, v)


def read_bias_file(infilename, verbose):
    """fithic.py:136-158 -> {chr name: {mid: bias}}."""
    if verbose:
        sys.stderr.write("\n\nReading ICE biases. \n")
    df = _read_table(infilename, 3)
    if df.shape[1] != 3:
        raise ValueError("too many values to unpack (expected 3)")
    names = df[0].values
    mids = df[1].values.astype(np.int64)
    vals = df[2].values.astype(np.float64)
    bad = (vals < 0.5) | (vals > 2)
    vals = np.where(bad, -1.0, vals)
    biases = {}
    for c, m, b in zip(names, mids, vals):
        sub = biases.setdefault(c, {})
        if int(m) not in sub:
            sub[int(m)] = -1 if b == -1.0 else float(b)
    if verbose:
        print("Out of " + str(len(df)) + " loci " + str(int(bad.sum())) + " were discarded with biases not in range [0.5 2]\n\n")
    return biases


def generate_FragPairs(infilename, resolution, min_dist, max_dist, verbose):
    """fithic.py:272-332 -> mainDic {distance: [possible pairs, 0]}."""
    if verbose:
        print("\nEnumerating all possible intra-chromosomal fragment pairs in-range\n")
        print("------------------------------------------------------------------------------------\n")
    _session.chroms = _ChromIds()
    fc, fm = _parse_fragments(infilename, _session.chroms)
    info = _frag_info(fc, fm, resolution)
    _session.frag = info
    _session.frag_arrays = (fc, fm)
    dev = _device()
    eng = PassEngine(resolution, 100, min_dist, max_dist, info.nkeys, dev)
    eng.set_fragments(info.n_frags, info.max_frag)
    possible = eng.possible.cpu().numpy()
    in_rng = sum(int(v) for k, v in enumerate(possible) if in_range_check(k * resolution, min_dist, max_dist))
    _publish(maxPossibleGenomicDist=info.max_possible, possibleIntraAllCount=info.possible_intra_all,
             possibleInterAllCount=info.possible_inter_all, possibleIntraInRangeCount=in_rng,
             interChrProb=(1.0 / info.possible_inter_all if info.possible_inter_all > 0 else 0),
             baselineIntraChrProb=1.0 / info.possible_intra_all,
             observedIntraInRangeCount=0, observedIntraInRangeSum=0, observedIntraAllCount=0, observedIntraAllSum=0,
             observedInterAllCount=0, observedInterAllSum=0, minObservedGenomicDist=500000000, maxObservedGenomicDist=0)
    if verbose:
        print("Number of all fragments= " + str(info.n_total) + "\t resolution= " + str(resolution))
        print("Possible, Intra-chr in range: pairs= " + str(in_rng))
        print("Possible, Intra-chr all: pairs= " + str(info.possible_intra_all))
        print("Possible, Inter-chr all: pairs= " + str(info.possible_inter_all))
        print("Desired genomic distance range	[%d %d]" % (min_dist, max_dist) + "\n")
        print("Range of possible genomic distances	[0	%d]" % (info.max_possible) + "\n")
    return {int(k) * int(resolution): [int(v), 0] for k, v in enumerate(possible)}


def _main_dic_tables(mainDic, resolution):
    keys = sorted(mainDic)
    R = int(resolution)
    if keys != [k * R for k in range(len(keys))]:
        raise ValueError("mainDic keys must be 0, R, 2R, ... as generate_FragPairs builds them")
    return (np.array([mainDic[k][0] for k in keys], dtype=np.int64),
            np.array([mainDic[k][1] for k in keys], dtype=np.int64))


def read_interactions(mainDic, infile, min_dist, max_dist, verbose):
    """fithic.py:229-270: adds the contact counts per distance to mainDic (K1 on the device)."""
    if verbose:
        print("\nReading all the contact counts\n")
        print("------------------------------------------------------------------------------------\n")
    if _session.chroms is None:
        _session.chroms = _ChromIds()
    c1, m1, c2, m2, cnt = _parse_interactions(infile, _session.chroms)
    _session.contacts = (c1, m1, c2, m2, cnt)
    resolution = sorted(mainDic)[1] if len(mainDic) > 1 else 1
    dev = _device()
    eng = PassEngine(resolution, 100, min_dist, max_dist, len(mainDic), dev)
    t32 = lambda a: _to_device_i32(a, dev)                       # range-checked: OverflowError instead of a silent wrap
    eng.hist([Shard(t32(m1), t32(m2), t32(cnt), t32(c1), t32(c2))])
    obs = eng.obs_sum.cpu().numpy()
    t = eng.totals.cpu().numpy()
    for k, key in enumerate(sorted(mainDic)):
        mainDic[key][1] += int(obs[k])
    _publish(observedIntraInRangeSum=_this.observedIntraInRangeSum + int(t[0]),
             observedIntraInRangeCount=_this.observedIntraInRangeCount + int(t[1]),
             observedIntraAllSum=_this.observedIntraAllSum + int(t[2]),
             observedIntraAllCount=_this.observedIntraAllCount + int(t[3]),
             observedInterAllSum=_this.observedInterAllSum + int(t[4]),
             observedInterAllCount=_this.observedInterAllCount + int(t[5]),
             minObservedGenomicDist=min(_this.minObservedGenomicDist, int(t[6])),
             maxObservedGenomicDist=max(_this.maxObservedGenomicDist, int(t[7])))
    if verbose:
        print("Observed, Intra-chr in range: pairs= " + str(_this.observedIntraInRangeCount) + "\t totalCount= " + str(_this.observedIntraInRangeSum))
        print("Observed, Intra-chr all: pairs= " + str(_this.observedIntraAllCount) + "\t totalCount= " + str(_this.observedIntraAllSum))
        print("Observed, Inter-chr all: pairs= " + str(_this.observedInterAllCount) + "\t totalCount= " + str(_this.observedInterAllSum))
        print("Range of observed genomic distances [%d %d]" % (_this.minObservedGenomicDist, _this.maxObservedGenomicDist) + "\n")
    return mainDic


def _fit_from_tables(possible, observed, S, n_bins, resolution, min_dist, max_dist):
    dev = _device()
    eng = PassEngine(resolution, n_bins, min_dist, max_dist, len(possible), dev)
    eng.possible.copy_(torch.from_numpy(possible))
    eng.obs_sum.copy_(torch.from_numpy(observed))
    eng.totals.zero_()
    eng.totals[0] = int(S)
    eng.fit()
    return eng


def calculate_probabilities(mainDic, n_bins, resolution, min_dist, max_dist, filename, verbose):
    """fithic.py:160-227 -> (x, y, yerr) lists.  Like the reference it opens (and never writes)
    `filename + '.res<R>.txt'`."""
    if verbose:
        print("\nCalculating probability means and standard deviations by equal-occupancy binning of contact counts\n")
        print("------------------------------------------------------------------------------------\n")
    open(filename + '.res' + str(resolution) + '.txt', 'w').close()        # fithic.py:164
    possible, observed = _main_dic_tables(mainDic, resolution)
    S = _this.observedIntraInRangeSum
    if verbose:
        print("observed intra-chr read counts in range\t" + repr(S) + ",\tdesired number of contacts per bin\t" +
              repr(S // n_bins) + ",\tnumber of bins\t" + repr(n_bins) + "\n")
    eng = _fit_from_tables(possible, observed, S, n_bins, resolution, min_dist, max_dist)
    raw = _lib.FitResult.from_buffer_copy(eng.fit_result.cpu().numpy().tobytes())
    if raw.status in (-11, -13, -14):                         # binning errors; spline errors belong to fit_spline
        err = _lib.FIT_STATUS[raw.status]
        raise err[0](err[1])
    n = raw.n_out
    x = eng.x[:n].cpu().numpy().tolist()
    y = eng.y[:n].cpu().numpy().tolist()
    return x, y, [0.0] * n


def fit_spline(mainDic, x, y, yerr, infilename, outfilename, biasDic, resolution, min_dist, max_dist, verbose):
    """fithic.py:334-437: spline + antitonic fit on (x, y), then score every record of `infilename`
    and write `<outfilename>.res<R>.significances.txt.gz`.  Returns (splineX, newSplineY, residual)."""
    if verbose:
        print("\nFit a univariate spline to the probability means\n")
        print("------------------------------------------------------------------------------------\n")
    dev = _device()
    lib = _lib.load()
    nkeys = len(mainDic)
    m = len(x)
    if m < 4:
        raise ValueError("m > k must hold")
    eng = PassEngine(resolution, max(m, 4), min_dist, max_dist, nkeys, dev, max_bins=max(m, 4))
    xs = torch.tensor(list(x), dtype=torch.float64, device=dev)
    ys = torch.tensor(list(y), dtype=torch.float64, device=dev)
    ws_bytes = int(lib.bbk_fit_workspace_bytes(max(m, 4), nkeys)) + 16 * m + 64
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=dev)
    req = _lib.FitResult()                                      # s exactly as fithic.py:340 computes it, on Python floats
    req.status = _lib.FIT_S_GIVEN
    req.smoothing = float(min(list(y)) ** 2)
    eng.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8))
    _lib.check(lib.bbk_fit_from_bins(_lib.ptr(xs), _lib.ptr(ys), m, nkeys, int(resolution), _lib.ptr(eng.fit_result),
                                     _lib.ptr(eng.spline_y), _lib.ptr(eng.spline_raw), _lib.ptr(eng.knots),
                                     _lib.ptr(eng.coefs), _lib.ptr(ws), ws_bytes, _lib.stream_ptr()), "bbk_fit_from_bins")
    # the scoring kernel reads S from the fit record
    S = int(_this.observedIntraInRangeSum)
    fit = eng.read_fit()
    fit.S = S
    eng.fit_result.copy_(torch.frombuffer(bytearray(bytes(fit)), dtype=torch.uint8))
    splineX = [(fit.k0 + i) * int(resolution) for i in range(fit.L)]
    newSplineY = eng.spline_y[:fit.L].cpu().numpy().tolist()
    residual = float(fit.residual)

    if verbose:
        print("lower bound on mid-range distances  " + repr(min_dist) + ", upper bound on mid-range distances  " + repr(max_dist) + "\n")
    chroms = _session.chroms if _session.chroms is not None else _ChromIds()
    c1, m1, c2, m2, cnt = _parse_interactions(infilename, chroms)
    if len(biasDic) > 0:
        ids = {chroms.ids[name]: sub for name, sub in biasDic.items() if name in chroms.ids}
        eng.set_bias(_bias_tables(ids, resolution, dev, n_chrom_hint=len(chroms.names)))
    t32 = lambda a: _to_device_i32(a, dev)
    shard = Shard(t32(m1), t32(m2), t32(cnt), t32(c1), t32(c2))
    p = torch.empty(_pad16(shard.n), dtype=torch.float64, device=dev)[:shard.n]
    eng.pvalues(shard, p)
    pv = p.cpu().numpy()
    _write_significances('{}.res{}.significances.txt.gz'.format(outfilename, resolution), chroms, c1, m1, c2, m2, cnt, pv, None)
    _session.result = (pv,)
    return splineX, newSplineY, residual


def _write_significances(path, chroms, c1, m1, c2, m2, cnt, p, q):
    """fithic.py:410-435: header + one row per record with p_val <= 1; q column is the literal -1
    unless q-values were asked for.  Formatted and compressed by all host cores (libbbkio.so, include/bbk_io.h)."""
    from . import _io
    _io.write_significances(path, list(chroms.names), c1, m1, c2, m2, cnt, p, q)


def fithic(libname, resolution, n_bins, min_dist, max_dist, n_passes, interactions, frags, biases, verbose,
           q_values=False):
    """fithic.py:110-133: one pass (n_passes is ignored, as in the reference), files in / files out."""
    chroms = _ChromIds()
    fc, fm = _parse_fragments(frags, chroms)
    bias_dic = None
    if biases != 'none':
        named = read_bias_file(biases, verbose)
        for name in named:
            chroms.encode([name])
        bias_dic = {chroms.ids[name]: sub for name, sub in named.items()}
    c1, m1, c2, m2, cnt = _parse_interactions(interactions, chroms)
    if verbose:
        print("\n\t\tSPLINE FIT PASS 1 (spline-1) \n")
    open(libname + ".fithic_pass1" + '.res' + str(resolution) + '.txt', 'w').close()          # fithic.py:164
    out = _run_pass(resolution, n_bins, min_dist, max_dist, fc, fm, c1, m1, c2, m2, cnt, bias_dic, want_q=q_values)
    _publish(**out.totals)
    _write_significances('{}.res{}.significances.txt.gz'.format(libname + ".spline_pass1", resolution),
                         chroms, c1, m1, c2, m2, cnt, out.p, out.q)
    if verbose:
        print("\nExecution of fit-hic completed successfully. \n\n")
    return


def benjamini_hochberg_correction(p_values, num_total_tests):
    """fithic.py:466-487: unsorted p in, q in input order out, as a list."""
    dev = _device()
    lib = _lib.load()
    p = torch.tensor(np.asarray(p_values, dtype=np.float64), device=dev)
    m = p.numel()
    if m == 0:
        return []
    pp = torch.empty(_pad16(m), dtype=torch.float64, device=dev)[:m].copy_(p)
    q = torch.empty(_pad16(m), dtype=torch.float64, device=dev)[:m]
    ws = torch.empty(int(lib.bbk_bh_workspace_bytes(m)), dtype=torch.uint8, device=dev)
    _lib.check(lib.bbk_bh_qvalues(_lib.ptr(pp), m, int(num_total_tests), _lib.BH_UNSORTED, None, _lib.ptr(q), None,
                                  _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "bbk_bh_qvalues")
    return q.cpu().numpy().tolist()
