"""GPU tests of per-chromosome passes streamed from pinned host memory: distributed.HostStream over a ChromosomePass.

Every streamed pass is compared, bit for bit, with a freshly built ChromosomePass run on the same records: p and q of every
chromosome, and every chromosome's fit result apart from its SM cycle counters.
"""
import struct

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R, N_BINS = 5000, 100


def _fit_cmp(raw):
    """The bytes of a BbkFitResult that a fit defines, without the SM cycle counters (as tools/bench_per_chromosome.py)."""
    raw = bytes(raw)
    return raw[:72] + raw[184:]


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).tobytes() if a.size else b""


class _Genome(object):
    pass


def _genome(seed, bins, max_dist, with_bias=True):
    """Chromosomes with non-consecutive ids in no particular order; bias tables on every other chromosome (the others have
    all loci absent)."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.engine import BiasTables
    rng = np.random.default_rng(seed)
    g = _Genome()
    g.dev = torch.device("cuda", 0)
    g.bins, g.max_dist = list(bins), int(max_dist)
    g.ids = [int(x) for x in rng.permutation(np.arange(len(bins)) * 2 + 1)]
    g.bias = synth.make_bias(g.bins, seed, sigma=0.3)
    g.tables = None
    if with_bias:
        vals = [np.zeros(0)] * (max(g.ids) + 1)
        for i, (c, b) in enumerate(zip(g.ids, g.bias)):
            vals[c] = np.where((b < 0.5) | (b > 2), -1.0, b) if i % 2 == 0 else np.full(len(b), np.nan)
        g.tables = BiasTables(vals, [R // 2] * len(vals), g.dev)
    return g


def _engines(g, extra=()):
    from blueberry_b200.engine import PassEngine
    es = []
    for nb in list(g.bins) + list(extra):
        e = PassEngine(R, N_BINS, 0, g.max_dist, nb, g.dev)
        e.set_fragments([nb], [(nb - 1) * R])
        e.set_bias(g.tables)
        es.append(e)
    return es


def _sample(g, seed, depth):
    """[(mid1, mid2, count)] per chromosome (every pair within max_dist, zeros included, so the rows are the same in every
    sample and only the counts differ)."""
    from blueberry_b200 import synth
    c = synth.make_contacts(g.bins, R, g.max_dist, depth, seed, g.bias)
    return [tuple(c[k][c["chrom"] == i] for k in ("mid1", "mid2", "count")) for i in range(len(g.bins))]


def _host_table(cols, sizes):
    """Pinned int32 columns holding chromosome i's first sizes[i] rows at layout_rows(sizes)[0][i]."""
    import torch
    from blueberry_b200.distributed import layout_rows
    starts, rows = layout_rows(sizes)
    h = [torch.zeros(max(rows, 4), dtype=torch.int32).pin_memory() for _ in range(3)]
    for col, a, n in zip(cols, starts, sizes):
        for t, v in zip(h, col):
            t[a:a + n] = torch.from_numpy(np.ascontiguousarray(v[:n], dtype=np.int32))
    return h


def _shards(g, cols, sizes, ids):
    import torch
    from blueberry_b200.engine import Shard
    return [Shard(*(torch.from_numpy(np.ascontiguousarray(v[:n], dtype=np.int32)).to(g.dev) for v in col), chrom=c)
            for col, n, c in zip(cols, sizes, ids)]


class _Ref(object):
    pass


def _reference(g, cols, sizes, q_values=True, n_tests=None, smoothing=None, finish=True, engines=None, ids=None):
    """A fresh ChromosomePass on the records: run() (or the pass alone, finish=False).  Returns its p / q bits per chromosome,
    its fit-result bytes per chromosome, the exception run() raised and the smoothing list it ended with."""
    import torch
    from blueberry_b200.distributed import ChromosomePass
    cp = ChromosomePass(engines if engines is not None else _engines(g), _shards(g, cols, sizes, ids or g.ids), q_values=q_values)
    if smoothing is not None:
        cp.smoothing = list(smoothing)
    ref = _Ref()
    ref.err = None
    if finish:
        try:
            cp.run(n_tests)
        except Exception as e:
            ref.err = e
    else:
        cp.enqueue(n_tests)
    torch.cuda.synchronize()
    ref.p = [_bits(cp.chrom_p(i).cpu().numpy()) for i in range(len(sizes))]
    ref.q = [_bits(cp.chrom_q(i).cpu().numpy()) for i in range(len(sizes))] if q_values else None
    ref.raws = [bytes(e.fit_result.cpu().numpy().tobytes()) for e in cp.engs]
    ref.smoothing = list(cp.smoothing)
    ref.state = cp.last_state if finish and ref.err is None else None
    return ref


def _assert_fits(hs, k, ref):
    """fit_of(k) against the reference: the same FitResults, or the same exception naming the same chromosome (and the same
    bytes for every chromosome whose fit did not fail)."""
    if ref.err is None:
        fits = hs.fit_of(k)
        assert len(fits) == len(ref.raws)
        assert [_fit_cmp(bytes(f)) for f in fits] == [_fit_cmp(r) for r in ref.raws]
        return fits
    with pytest.raises(type(ref.err)) as ei:
        hs.fit_of(k)
    assert str(ei.value) == str(ref.err) and ei.value.chrom == ref.err.chrom
    raw = hs.slots[k % len(hs.slots)].h_fit.numpy().tobytes()
    nf = len(raw) // len(ref.raws)
    for i, r in enumerate(ref.raws):
        got = raw[i * nf:(i + 1) * nf]
        ok = struct.unpack_from("i", r)[0] == 0
        assert (_fit_cmp(got) if ok else got[:4]) == (_fit_cmp(r) if ok else r[:4]), "chromosome %d" % i
    return None


def _assert_columns(p, q, sizes, ref):
    from blueberry_b200.distributed import layout_rows
    starts, _ = layout_rows(sizes)
    for i, (a, n) in enumerate(zip(starts, sizes)):
        assert _bits(p[a:a + n]) == ref.p[i], "p of chromosome %d" % i
        if q is not None:
            assert _bits(q[a:a + n]) == ref.q[i], "q of chromosome %d" % i


@pytest.fixture(scope="module")
def genome():
    """Five chromosomes, five samples of different depths (one with its own N per chromosome), their references."""
    g = _genome(7, [310, 180, 260, 400, 225], 60 * R)
    g.sizes = [len(c[0]) for c in _sample(g, 0, 10.0)]
    g.samples = [_sample(g, 100 + k, d) for k, d in enumerate((12.0, 40.0, 6.0, 90.0, 25.0))]
    g.n_tests = [None, None, None, [50, -1, 7000, -1, 300], -1]
    g.refs = [_reference(g, s, g.sizes, n_tests=nt) for s, nt in zip(g.samples, g.n_tests)]
    g.hosts = [_host_table(s, g.sizes) for s in g.samples]
    return g


def _stream(g, **kw):
    from blueberry_b200.distributed import ChromosomePass, HostStream
    cp = ChromosomePass(_engines(g), _shards(g, g.samples[0], g.sizes, g.ids), q_values=True)
    return cp, HostStream(cp, g.sizes, g.ids, **kw)


def _pinned(n):
    import torch
    return torch.empty(max(n, 4), dtype=torch.float64).pin_memory()


def test_dense_stream_equals_chromosome_pass_run(genome):
    """Five samples through two slots (two passes in flight): every pass equals ChromosomePass.run, and fit_of(k) its fits."""
    import torch
    g = genome
    cp, hs = _stream(g, slots=2)
    outs = []
    for k, (h, ref, nt) in enumerate(zip(g.hosts, g.refs, g.n_tests)):
        cp.smoothing = list(ref.smoothing)        # a chromosome the reference repeated with its own s is submitted with it
        h_p, h_q = _pinned(len(h[0])), _pinned(len(h[0]))
        hs.submit(h[0], h[1], h[2], h_p, h_q, n_tests=nt)
        outs.append((h_p, h_q))
        if k:                                     # pass k - 1, while pass k is in flight
            _assert_fits(hs, k - 1, g.refs[k - 1])
            _assert_columns(outs[k - 1][0].numpy(), outs[k - 1][1].numpy(), g.sizes, g.refs[k - 1])
    hs.drain()
    k = len(g.refs) - 1
    fits = _assert_fits(hs, k, g.refs[k])
    assert len(fits) == len(g.ids) and all(f.S > 0 for f in fits)
    _assert_columns(outs[k][0].numpy(), outs[k][1].numpy(), g.sizes, g.refs[k])
    assert g.refs[0].p[0] != g.refs[1].p[0]
    with pytest.raises(KeyError):
        hs.fit_of(0)
    torch.cuda.synchronize()


def test_packed_stream_equals_dense_stream(genome):
    """The same samples with packed results: dense() gives the slot layout (padding rows NaN) with every chromosome equal to
    the reference; value lists too small for one pass bring that pass back dense, still equal."""
    from blueberry_b200.distributed import layout_rows
    g = genome
    starts, rows = layout_rows(g.sizes)
    real = np.zeros(max(rows, 4), bool)
    for a, n in zip(starts, g.sizes):
        real[a:a + n] = True
    assert not real.all()                         # there is padding between chromosomes
    # value lists with room for every row: these small samples have far more q below 1 than the default rows / 16
    cp, hs = _stream(g, slots=2, packed=True, cap_p=rows, cap_q=rows)
    outs = [hs.packed_buffers() for _ in g.samples]
    for h, o, ref, nt in zip(g.hosts, outs, g.refs, g.n_tests):
        cp.smoothing = list(ref.smoothing)
        hs.submit_packed(h[0], h[1], h[2], o, n_tests=nt)
    hs.drain()
    for o, ref in zip(outs, g.refs):
        assert not o.overflow
        p, q = o.dense()
        assert len(p) == hs.rows
        _assert_columns(p, q, g.sizes, ref)
        assert np.isnan(p[~real]).all() and np.isnan(q[~real]).all()
    for k in (len(outs) - 2, len(outs) - 1):
        _assert_fits(hs, k, g.refs[k])
    cp, small = _stream(g, slots=2, packed=True, cap_p=8, cap_q=8)
    cp.smoothing = list(g.refs[1].smoothing)
    o = small.submit_packed(g.hosts[1][0], g.hosts[1][1], g.hosts[1][2], small.packed_buffers())
    small.drain()
    assert o.overflow
    p, q = o.dense()
    _assert_columns(p, q, g.sizes, g.refs[1])
    assert np.isnan(p[~real]).all()
    _assert_fits(small, 0, g.refs[1])


def test_smaller_sizes_with_empty_and_one_row_chromosomes(genome):
    """sizes= below the built sizes, one chromosome at 0 rows and one at 1 row, equal to a ChromosomePass built on those rows;
    a size above a chromosome's built size raises ValueError before anything is copied or submitted."""
    import torch
    g = genome
    cp, hs = _stream(g, slots=2)
    smp = g.samples[1]
    cols, sizes = [], []
    for i, (m1, m2, c) in enumerate(smp):
        if i == 1:
            cols.append((m1[:0], m2[:0], c[:0]))                          # 0 rows
        elif i == 3:
            j = int(np.flatnonzero(m2 - m1 == 3 * R)[0])                  # 1 in-range row
            cols.append((m1[j:j + 1], m2[j:j + 1], np.array([5], dtype=np.int32)))
        else:
            n = [len(m1) // 2 + 1, 0, len(m1) - 3, 0, 1001][i]
            cols.append((m1[:n], m2[:n], c[:n]))
        sizes.append(len(cols[-1][0]))
    assert sizes[1] == 0 and sizes[3] == 1 and all(a <= b for a, b in zip(sizes, g.sizes))
    h = _host_table(cols, sizes)
    h_p, h_q = _pinned(len(h[0])), _pinned(len(h[0]))
    too_big = list(g.sizes)
    too_big[2] += 1
    too_big[0] -= 4                                                       # the slot would still hold them all
    hb =_host_table([(np.resize(m1, n), np.resize(m2, n), np.resize(c, n)) for (m1, m2, c), n in zip(smp, too_big)], too_big)
    big_p, big_q = _pinned(len(hb[0])), _pinned(len(hb[0]))
    with pytest.raises(ValueError, match="chromosome %d" % g.ids[2]):
        hs.submit(hb[0], hb[1], hb[2], big_p, big_q, sizes=too_big)
    assert hs.submitted == 0
    ref = _reference(g, cols, sizes)
    assert ref.err is not None                                            # the empty chromosome (or the one-row one) fails
    hs.submit(h[0], h[1], h[2], h_p, h_q, sizes=sizes)
    hs.drain()
    _assert_columns(h_p.numpy(), h_q.numpy(), sizes, ref)
    _assert_fits(hs, 0, ref)
    # the built sizes again, after the small pass: equal to the reference
    cp.smoothing = list(g.refs[2].smoothing)
    h_p, h_q = _pinned(hs.rows), _pinned(hs.rows)
    hs.submit(g.hosts[2][0], g.hosts[2][1], g.hosts[2][2], h_p, h_q)
    hs.drain()
    _assert_columns(h_p.numpy(), h_q.numpy(), g.sizes, g.refs[2])
    _assert_fits(hs, 1, g.refs[2])
    torch.cuda.synchronize()


def test_submit_without_q_leaves_q_alone(genome):
    """Without h_q the pass skips the segmented q-value step: p equals a q_values=False ChromosomePass and the slot's q keeps
    what the slot's previous pass left there."""
    g = genome
    cp, hs = _stream(g, slots=2)
    outs = []
    for k in (0, 1):
        cp.smoothing = list(g.refs[k].smoothing)
        h = g.hosts[k]
        outs.append((_pinned(hs.rows), _pinned(hs.rows)))
        hs.submit(h[0], h[1], h[2], outs[k][0], outs[k][1])
    hs.drain()
    q_before = hs.slots[0].q.cpu().numpy().copy()
    ref = _reference(g, g.samples[2], g.sizes, q_values=False)
    cp.smoothing = list(ref.smoothing)
    h = g.hosts[2]
    h_p = _pinned(hs.rows)
    hs.submit(h[0], h[1], h[2], h_p)
    hs.drain()
    assert cp.q_values
    _assert_columns(h_p.numpy(), None, g.sizes, ref)
    _assert_fits(hs, 2, ref)
    assert _bits(hs.slots[0].q.cpu().numpy()) == _bits(q_before)
    _assert_columns(outs[0][0].numpy(), outs[0][1].numpy(), g.sizes, g.refs[0])


def test_deferred_lists_hold_every_row_and_candidate_lists_overflow():
    """One chromosome of more than 2^20 rows, nearly all deferred (counts above 64 go to the patch pass), streamed next to
    ordinary chromosomes: the stream gives each chromosome a deferred list as long as its rows, so nothing overflows unseen,
    and p / q equal ChromosomePass.run (which repeats the pass with a larger list).  Then a pass whose candidate lists are
    too small for the q-values: the segmented step falls back on the device and the result is the same."""
    import ctypes
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import ChromosomePass, HostStream
    lib = _lib.load()
    K = 100
    g = _genome(3, [300, 220, 260], K * R, with_bias=False)
    nb = 20050
    n = int(lib.bbk_synth_n_pairs(nb, K))
    assert n > 1 << 20
    big = [torch.empty(n, dtype=torch.int32, device=g.dev) for _ in range(3)]
    _lib.check(lib.bbk_synth_contacts(nb, K, R, 20000.0, 1.08, 3, None, _lib.ptr(big[0]), _lib.ptr(big[1]), _lib.ptr(big[2]),
                                      _lib.stream_ptr()), "synth")
    cols = _sample(g, 9, 30.0)
    cols.insert(1, tuple(t.cpu().numpy() for t in big))
    ids = g.ids[:1] + [2 * len(g.bins) + 1] + g.ids[1:]                  # the big chromosome gets an id of its own
    sizes = [len(c[0]) for c in cols]

    def engines():
        es = _engines(g, extra=[nb])
        return es[:1] + es[-1:] + es[1:-1]
    ref = _reference(g, cols, sizes, engines=engines(), ids=ids)
    assert ref.err is None
    assert ref.state[1][1].n_list > max(1 << 20, n // 4)                # more than a default-size list holds
    h = _host_table(cols, sizes)
    for cand_capacity in (None, 64):
        cp = ChromosomePass(engines(), _shards(g, cols, sizes, ids), q_values=True, cand_capacity=cand_capacity)
        hs = HostStream(cp, sizes, ids, slots=2)
        assert [l[3].capacity for l in cp.lists] == [(s + 3) & ~3 for s in sizes]
        cp.smoothing = list(ref.smoothing)
        h_p, h_q = _pinned(hs.rows), _pinned(hs.rows)
        hs.submit(h[0], h[1], h[2], h_p, h_q)
        hs.drain()
        _assert_columns(h_p.numpy(), h_q.numpy(), sizes, ref)
        _assert_fits(hs, 0, ref)
        raw = cp.score_state.cpu().numpy().tobytes()
        ns = ctypes.sizeof(_lib.ScoreState)
        states = [_lib.ScoreState.from_buffer_copy(raw[i * ns:(i + 1) * ns]) for i in range(len(sizes))]
        assert not any(s.overflow for s in states)
        if cand_capacity:
            assert any(s.cand_overflow for s in states)


def test_failed_fit_names_the_lowest_chromosome_and_smoothing_resubmission(genome):
    """Chromosomes whose counts are all zero: fit_of(k) raises ZeroDivisionError naming the lowest such id, as run() does.
    Then a chromosome resubmitted with pass.smoothing[i] set equals a ChromosomePass pass with the same smoothing[i]."""
    g = genome
    cp, hs = _stream(g, slots=2)
    order = sorted(range(len(g.ids)), key=lambda i: g.ids[i])
    zero = [order[3], order[1]]
    cols = [(m1, m2, np.zeros_like(c) if i in zero else c) for i, (m1, m2, c) in enumerate(g.samples[0])]
    ref = _reference(g, cols, g.sizes)
    assert isinstance(ref.err, ZeroDivisionError) and ref.err.chrom == g.ids[order[1]]
    h = _host_table(cols, g.sizes)
    h_p, h_q = _pinned(hs.rows), _pinned(hs.rows)
    hs.submit(h[0], h[1], h[2], h_p, h_q)
    hs.drain()
    with pytest.raises(ZeroDivisionError, match="chromosome %d:" % g.ids[order[1]]):
        hs.fit_of(0)
    _assert_fits(hs, 0, ref)
    _assert_columns(h_p.numpy(), h_q.numpy(), g.sizes, ref)
    # resubmission with a chromosome's s given
    cp.smoothing = list(g.refs[0].smoothing)
    hs.submit(g.hosts[0][0], g.hosts[0][1], g.hosts[0][2], h_p, h_q)
    hs.drain()
    fits = _assert_fits(hs, 1, g.refs[0])
    i = order[2]
    smoothing = list(g.refs[0].smoothing)
    smoothing[i] = fits[i].smoothing * 1.5
    ref = _reference(g, g.samples[0], g.sizes, smoothing=smoothing, finish=False)
    cp.smoothing = list(smoothing)
    hs.submit(g.hosts[0][0], g.hosts[0][1], g.hosts[0][2], h_p, h_q)
    hs.drain()
    fits2 = _assert_fits(hs, 2, ref)
    assert fits2[i].smoothing == smoothing[i] and _fit_cmp(bytes(fits2[i])) != _fit_cmp(bytes(fits[i]))
    _assert_columns(h_p.numpy(), h_q.numpy(), g.sizes, ref)
    assert ref.p[i] != g.refs[0].p[i]                                     # the given s changed that chromosome's p
