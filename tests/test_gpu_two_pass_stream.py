"""GPU tests of the two-pass stream, distributed.HostStream(GenomePass, ..., refit=True) (BASELINE config 4 from host memory),
and of smoothing= on GenomePass streams.

Every streamed submission is compared with the sequence fit_transform_arrays(refit=True) runs on the same engine and records:
pass 1 without q-values, the outlier threshold 1 / possibleIntraInRangeCount, the refit pass with exclude=(p_first, threshold),
each pass settled on its s.  p_first, p and q are compared by bit pattern over the rows the records cover, and both fit results
byte for byte (all but the SM cycle counters)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R = 5000


def _fit_cmp(raw):
    """The bytes of a BbkFitResult that a fit defines, without the SM cycle counters."""
    raw = bytes(raw)
    return raw[:72] + raw[184:]


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _pinned(n, fill=7.0):
    import torch
    return torch.full((max(n, 4),), fill, dtype=torch.float64).pin_memory()


def _threshold(eng):
    from blueberry_b200.fithic import _in_range_possible
    return 1.0 / _in_range_possible(eng.possible.cpu().numpy(), eng.R, eng.min_dist, eng.max_dist)


def _pass(gp, n_tests, smoothing, exclude, settle):
    if settle:
        return bytes(gp.run(n_tests, smoothing=smoothing, exclude=exclude))
    gp.enqueue(n_tests, smoothing=smoothing, exclude=exclude)          # this s and no other (run() would go on to the reference's)
    raw, score, _ = gp.read_state()
    assert score.overflow == 0
    return raw


def _serial(eng, shards, smoothing=(None, None), want_q=True, n_tests=-1, settle=True):
    """fit_transform_arrays(refit=True)'s two passes on `eng` and `shards`, each a GenomePass of its own.  settle: each pass
    settles on the reference's own s as GenomePass.run does (smoothing then gives the first s tried); otherwise each pass runs
    once with the s given.  Returns a dict: p_first / p / q (numpy, layout rows), fit1 / fit2 (bytes), s (the s each pass
    ended with, None = the kernel's own), thr, the two passes."""
    from blueberry_b200.distributed import GenomePass, layout_rows
    rows = max(layout_rows([sh.n for sh in shards])[1], 4)
    thr = _threshold(eng)
    cap = None if settle else rows
    gp1 = GenomePass(eng, group=False, q_values=False)
    gp1.attach(shards, list_capacity=cap)
    fit1 = _pass(gp1, -1, smoothing[0], None, settle)
    gp2 = GenomePass(eng, group=False, q_values=want_q)
    gp2.attach(shards, list_capacity=cap)
    fit2 = _pass(gp2, n_tests, smoothing[1], (gp1.p, thr), settle)
    return {"p_first": gp1.p.cpu().numpy()[:rows], "p": gp2.p.cpu().numpy()[:rows],
            "q": gp2.q.cpu().numpy()[:rows] if want_q else None, "fit1": fit1, "fit2": fit2,
            "s": (gp1._smoothing, gp2._smoothing), "thr": thr, "passes": (gp1, gp2)}


def _check(ref, real, p_first=None, p=None, q=None):
    """The streamed columns (numpy over the same rows as ref's) on the real rows, bit for bit."""
    for got, key in ((p_first, "p_first"), (p, "p"), (q, "q")):
        if got is not None:
            assert _same_bits(got[:len(real)][real], ref[key][:len(real)][real]), key


# ------------------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def synth():
    """One chromosome of 6000 bins @ 5 kb, all pairs within 2 Mb, with biases; five libraries of ragged sizes (odd and even)
    generated on the device (bbk_synth_contacts), as device columns."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.engine import BiasTables, PassEngine
    lib = _lib.load()
    dev = torch.device("cuda:0")
    nb, K = 6000, 400
    P = int(lib.bbk_synth_n_pairs(nb, K))
    rng = np.random.default_rng(5)
    bias_host = np.exp(rng.normal(0.0, 0.25, size=nb))
    bias_dev = torch.from_numpy(bias_host).to(dev)
    eng = PassEngine(R, 100, 0, K * R, nb, dev)
    eng.set_fragments([nb], [(nb - 1) * R])
    eng.set_bias(BiasTables([np.where((bias_host < 0.5) | (bias_host > 2), -1.0, bias_host)], [R // 2], dev))
    libs = []
    for i in range(5):
        cols = [torch.empty(P, dtype=torch.int32, device=dev) for _ in range(3)]
        _lib.check(lib.bbk_synth_contacts(nb, K, R, 40.0 + 25 * i, 1.08, 100 + i, _lib.ptr(bias_dev), _lib.ptr(cols[0]),
                                          _lib.ptr(cols[1]), _lib.ptr(cols[2]), _lib.stream_ptr()), "synth")
        n = P - 1000 * i - (i & 1)
        libs.append([c[:n].contiguous() for c in cols])
    torch.cuda.synchronize()
    return eng, P, libs


def _shard(cols):
    from blueberry_b200.engine import Shard
    return Shard(*cols)


def _host(cols):
    return [c.cpu().pin_memory() for c in cols]


def _genome(seed, bins, max_dist, depth, dev):
    """Per-chromosome numpy columns of a small genome (synth.make_contacts, zeros kept) and its GenomePass engine, with biases."""
    from blueberry_b200 import synth
    from blueberry_b200.engine import BiasTables, PassEngine
    bias = synth.make_bias(bins, seed, sigma=0.3)
    c = synth.make_contacts(bins, R, max_dist, depth, seed, bias)
    shards = [tuple(np.ascontiguousarray(c[k][c["chrom"] == i]) for k in ("mid1", "mid2", "count")) for i in range(len(bins))]
    eng = PassEngine(R, 100, 0, max_dist, max(bins), dev)
    eng.set_fragments(bins, [(b - 1) * R for b in bins])
    eng.set_bias(BiasTables([np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias], [R // 2] * len(bins), dev))
    return shards, bias, eng


def _layout_host(shards):
    """Pinned int32 host columns of the pass layout and the mask of the real rows."""
    import torch
    from blueberry_b200.distributed import layout_rows
    starts, rows = layout_rows([len(s[0]) for s in shards])
    h = [torch.zeros(max(rows, 4), dtype=torch.int32).pin_memory() for _ in range(3)]
    real = np.zeros(max(rows, 4), bool)
    for a, s in zip(starts, shards):
        for j in range(3):
            h[j][a:a + len(s[j])] = torch.from_numpy(s[j])
        real[a:a + len(s[0])] = True
    return h, real


# ------------------------------------------------------------------------------------------------------------ 1. dense
def test_dense_stream_equals_serial_two_pass(synth):
    """Five libraries through two slots, each with its settled (s1, s2); then a pass without h_q (the slot's q is left
    alone), a pass without h_p_first, and fit_of of an evicted submission."""
    import torch
    from blueberry_b200.distributed import GenomePass, HostStream
    eng, P, libs = synth
    refs = [_serial(eng, [_shard(cols)]) for cols in libs]
    hosts = [_host(cols) for cols in libs]
    hs = HostStream(GenomePass(eng, group=False), [P], [0], slots=2, refit=True)
    outs = []
    for cols, ref in zip(hosts, refs):
        n = cols[0].numel()
        h = [_pinned(n) for _ in range(3)]
        hs.submit(cols[0], cols[1], cols[2], h[1], h[2], sizes=[n], h_p_first=h[0], smoothing=ref["s"])
        outs.append(h)
    hs.drain()
    for (h_p1, h_p, h_q), ref, cols in zip(outs, refs, hosts):
        n = cols[0].numel()
        real = np.ones(n, bool)
        _check(ref, real, h_p1.numpy(), h_p.numpy(), h_q.numpy())
        assert int((ref["p_first"][:n] <= ref["thr"]).sum()) > 0      # pass 2 left outliers out
        assert not _same_bits(ref["p_first"][:n], ref["p"][:n])
    for k in (3, 4):
        assert _fit_cmp(hs.fit_of(k, first=True)) == _fit_cmp(refs[k]["fit1"])
        assert _fit_cmp(hs.fit_of(k)) == _fit_cmp(refs[k]["fit2"])
    assert _fit_cmp(refs[3]["fit1"]) != _fit_cmp(refs[3]["fit2"])
    for first in (False, True):
        with pytest.raises(KeyError):
            hs.fit_of(0, first=first)

    # without h_q: no q-value step, and the slot's q (pass 3's) is left alone
    slot = hs.slots[hs.submitted % 2]
    q_before = slot.q.clone()
    n = hosts[1][0].numel()
    ref = _serial(eng, [_shard(libs[1])], want_q=False)
    h_p1, h_p = _pinned(n), _pinned(n)
    hs.submit(hosts[1][0], hosts[1][1], hosts[1][2], h_p, sizes=[n], h_p_first=h_p1, smoothing=ref["s"]).synchronize()
    _check(ref, np.ones(n, bool), h_p1.numpy(), h_p.numpy())
    assert torch.equal(slot.q.view(torch.int64), q_before.view(torch.int64))
    assert _fit_cmp(hs.fit_of(hs.submitted - 1)) == _fit_cmp(ref["fit2"])
    # without h_p_first
    n = hosts[2][0].numel()
    h_p, h_q = _pinned(n), _pinned(n)
    hs.submit(hosts[2][0], hosts[2][1], hosts[2][2], h_p, h_q, sizes=[n], smoothing=refs[2]["s"]).synchronize()
    _check(refs[2], np.ones(n, bool), p=h_p.numpy(), q=h_q.numpy())
    assert _fit_cmp(hs.fit_of(hs.submitted - 1, first=True)) == _fit_cmp(refs[2]["fit1"])


def test_dense_stream_three_shards():
    """A GenomePass of three chromosomes: exclude= slices p_first by the shards' offsets in the slot."""
    import torch
    from blueberry_b200.distributed import GenomePass, HostStream
    from blueberry_b200.engine import Shard
    dev = torch.device("cuda", 0)
    bins = [700, 41, 650]
    shards, _, eng = _genome(4, bins, 300 * R, 80.0, dev)
    sizes = [len(s[0]) for s in shards]
    assert any(n & 3 for n in sizes)
    ref = _serial(eng, [Shard(*(torch.from_numpy(c).to(dev) for c in s), chrom=i) for i, s in enumerate(shards)])
    h, real = _layout_host(shards)
    hs = HostStream(GenomePass(eng, group=False), sizes, [0, 1, 2], slots=2, refit=True)
    n = len(real)
    h_p1, h_p, h_q = _pinned(n), _pinned(n), _pinned(n)
    hs.submit(h[0], h[1], h[2], h_p, h_q, h_p_first=h_p1, smoothing=ref["s"]).synchronize()
    _check(ref, real, h_p1.numpy(), h_p.numpy(), h_q.numpy())
    assert _fit_cmp(hs.fit_of(0, first=True)) == _fit_cmp(ref["fit1"])
    assert _fit_cmp(hs.fit_of(0)) == _fit_cmp(ref["fit2"])
    assert int((ref["p_first"][real] <= ref["thr"]).sum()) > 0


# ------------------------------------------------------------------------------------------------------------ 2. drop-in
def test_config4_shape_equals_fit_transform_arrays_refit():
    """BASELINE config 4's shape (1 kb, 2 Mb cap, 4000 bins, depth 60, biases): the stream, settling s1 and s2 by resubmission
    as a caller does, equals fit_transform_arrays(refit=True, q_values=True) bit for bit."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.distributed import GenomePass, HostStream
    from blueberry_b200.engine import PassEngine
    from blueberry_b200.fithic import FitHiC, _bias_dict_from_arrays, _bias_tables, _frag_info
    dev = torch.device("cuda", 0)
    R1, bins, max_dist = 1000, [4000], 2_000_000
    fc, fm = synth.make_fragments(bins, R1)
    bias = synth.make_bias(bins, 4)
    c = synth.make_contacts(bins, R1, max_dist, 60.0, 404, bias)
    barr = (np.zeros(bins[0], dtype=np.int32), fm.copy(), bias[0])
    model = FitHiC("unused", R1, n_bins=100, max_dist=max_dist, min_dist=0)
    out = model.fit_transform_arrays(c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], fc, fm, bias=barr, refit=True,
                                     q_values=True)
    info = _frag_info(fc, fm, R1)
    eng = PassEngine(R1, model.n_bins, model.min_dist, model.max_dist, info.nkeys, dev)
    eng.set_fragments(info.n_frags, info.max_frag)
    eng.set_bias(_bias_tables(_bias_dict_from_arrays(*barr), R1, dev))
    n = len(c["count"])
    h = [torch.from_numpy(np.ascontiguousarray(c[k], dtype=np.int32)).pin_memory() for k in ("mid1", "mid2", "count")]
    hs = HostStream(GenomePass(eng, group=False), [n], [0], slots=2, refit=True)
    h_p1, h_p, h_q = _pinned(n), _pinned(n), _pinned(n)
    s = [None, None]
    for _ in range(3):                                 # the caller's loop: pass 1's s first, then the refit's
        hs.submit(h[0], h[1], h[2], h_p, h_q, h_p_first=h_p1, smoothing=tuple(s)).synchronize()
        k = hs.submitted - 1
        s1 = PassEngine.reference_smoothing(hs.fit_of(k, first=True))
        s2 = PassEngine.reference_smoothing(hs.fit_of(k)) if s1 is None else None
        if s1 is None and s2 is None:
            break
        s[0 if s1 is not None else 1] = s1 if s1 is not None else s2
    assert _same_bits(h_p1.numpy()[:n], out.p_first)
    assert _same_bits(h_p.numpy()[:n], out.p)
    assert _same_bits(h_q.numpy()[:n], out.q)
    assert _fit_cmp(hs.fit_of(k)) == _fit_cmp(out.fit)
    assert int((out.p_first <= 1.0 / out.totals["possibleIntraInRangeCount"]).sum()) > 0
    assert hs.p_outlier == 1.0 / out.totals["possibleIntraInRangeCount"]


# ------------------------------------------------------------------------------------------------------------ 3. packed
def test_packed_stream_equals_dense_stream(synth):
    """submit_packed with refit: the same p / q as the dense stream, with value lists that hold the pass, with lists that
    overflow (the pass comes back dense), and fed PackedRecords instead of columns."""
    from blueberry_b200.distributed import GenomePass, HostStream, pack_records
    eng, P, libs = synth
    cols = libs[1]
    n = cols[0].numel()
    ref = _serial(eng, [_shard(cols)])
    h = _host(cols)
    dense = HostStream(GenomePass(eng, group=False), [n], [0], slots=2, refit=True)
    h_p, h_q = _pinned(n), _pinned(n)
    dense.submit(h[0], h[1], h[2], h_p, h_q, smoothing=ref["s"]).synchronize()
    _check(ref, np.ones(n, bool), p=h_p.numpy(), q=h_q.numpy())
    want = (h_p.numpy()[:n].copy(), h_q.numpy()[:n].copy(), _fit_cmp(dense.fit_of(0, first=True)), _fit_cmp(dense.fit_of(0)))
    rec = pack_records([tuple(c.numpy() for c in h)])
    for caps, feed in (((None, None), "columns"), ((8, 8), "columns"), ((None, None), "records")):
        hs = HostStream(GenomePass(eng, group=False), [n], [0], slots=2, packed=True, cap_p=caps[0], cap_q=caps[1], refit=True)
        outs = []
        for _ in range(3):                             # three passes through two slots
            o = hs.packed_buffers()
            if feed == "records":
                hs.submit_packed(rec, out=o, smoothing=ref["s"])
            else:
                hs.submit_packed(h[0], h[1], h[2], o, smoothing=ref["s"])
            outs.append(o)
        hs.drain()
        for k, o in enumerate(outs):
            assert o.overflow == (caps[0] == 8)
            p, q = o.dense()
            assert _same_bits(p[:n], want[0]) and _same_bits(q[:n], want[1]), (caps, feed, k)
        assert (_fit_cmp(hs.fit_of(2, first=True)), _fit_cmp(hs.fit_of(2))) == want[2:]


# ------------------------------------------------------------------------------------------------------------ 4. failures
def test_failed_pass_and_rejected_streams(synth):
    import torch
    from blueberry_b200.distributed import ChromosomePass, GenomePass, HostStream
    from blueberry_b200.engine import BiasTables, PassEngine, Shard
    eng, P, libs = synth
    dev = eng.device
    hs = HostStream(GenomePass(eng, group=False), [P], [0], slots=2, refit=True)
    h = _host(libs[0])
    n = h[0].numel()
    zero = torch.zeros(n, dtype=torch.int32).pin_memory()
    h_p, h_q, h_p1 = _pinned(n), _pinned(n), _pinned(n)
    hs.submit(h[0], h[1], zero, h_p, h_q, sizes=[n], h_p_first=h_p1)
    with pytest.raises(ZeroDivisionError):             # S == 0 in pass 1 (fithic.py:216)
        hs.fit_of(0)
    with pytest.raises(ZeroDivisionError):
        hs.fit_of(0, first=True)
    ref = _serial(eng, [_shard(libs[2])])               # the next submission is not affected
    h2 = _host(libs[2])
    n2 = h2[0].numel()
    hs.submit(h2[0], h2[1], h2[2], h_p, h_q, sizes=[n2], h_p_first=h_p1, smoothing=ref["s"]).synchronize()
    _check(ref, np.ones(n2, bool), h_p1.numpy(), h_p.numpy(), h_q.numpy())
    assert _fit_cmp(hs.fit_of(1)) == _fit_cmp(ref["fit2"])
    # argument checks, before anything is queued
    for kw in ({"smoothing": 1.0}, {"smoothing": (1.0,)}, {"smoothing": (1.0, 2.0, 3.0)}):
        with pytest.raises(ValueError):
            hs.submit(h2[0], h2[1], h2[2], h_p, sizes=[n2], **kw)
    assert hs.submitted == 2
    single = HostStream(GenomePass(eng, group=False), [P], [0], slots=2)
    with pytest.raises(ValueError):
        single.submit(h2[0], h2[1], h2[2], h_p, sizes=[n2], h_p_first=h_p1)
    with pytest.raises(ValueError):
        single.fit_of(0, first=True)
    assert single.submitted == 0

    # a fragment set without a single in-range pair: the threshold divides by zero, as refit=True does
    lone = PassEngine(R, 100, 0, 10 * R, 1, dev)
    lone.set_fragments([1, 1], [0, 0])
    with pytest.raises(ZeroDivisionError):
        HostStream(GenomePass(lone, group=False), [16], [0], slots=2, refit=True)
    # refit across ranks
    gp = GenomePass(eng, group=False)
    gp.world = 2
    with pytest.raises(NotImplementedError):
        HostStream(gp, [P], [0], slots=2, refit=True)

    # ChromosomePass: no refit, and no smoothing= (it takes pass.smoothing[i])
    bins = [300, 200]
    shards, bias, _ = _genome(7, bins, 100 * R, 40.0, dev)
    tables = BiasTables([np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias], [R // 2] * len(bins), dev)
    engines = []
    for nb in bins:
        e = PassEngine(R, 100, 0, 100 * R, nb, dev)
        e.set_fragments([nb], [(nb - 1) * R])
        e.set_bias(tables)
        engines.append(e)
    cp = ChromosomePass(engines, [Shard(*(torch.from_numpy(c).to(dev) for c in s), chrom=i) for i, s in enumerate(shards)])
    sizes = [len(s[0]) for s in shards]
    with pytest.raises(NotImplementedError):
        HostStream(cp, sizes, [0, 1], slots=2, refit=True)
    chs = HostStream(cp, sizes, [0, 1], slots=2)
    hc, real = _layout_host(shards)
    h_p = _pinned(len(real))
    with pytest.raises(ValueError):
        chs.submit(hc[0], hc[1], hc[2], h_p, smoothing=1.0)
    assert chs.submitted == 0
    chs.submit(hc[0], hc[1], hc[2], h_p).synchronize()  # None is accepted
    assert len(chs.fit_of(0)) == 2


# ------------------------------------------------------------------------------------------------------------ 5. given s
def test_resubmission_with_a_given_s(synth):
    """smoothing= reaches the fit: a single-pass stream with 1.5 s equals GenomePass's pass with that s, and a refit stream
    with (1.5 s1, None) and (None, 1.5 s2) equals the serial passes with the same values.  (GenomePass.run would go on to the
    reference's own s, so the reference passes run once with the s given.)"""
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import GenomePass, HostStream
    eng, P, libs = synth
    cols = libs[3]
    n = cols[0].numel()
    h = _host(cols)
    real = np.ones(n, bool)

    gp = GenomePass(eng, group=False)
    gp.attach([_shard(cols)])
    x = 1.5 * gp.run().smoothing
    gp = GenomePass(eng, group=False)
    gp.attach([_shard(cols)], list_capacity=max(n, 4))
    gp.enqueue(smoothing=x)
    raw, score, _ = gp.read_state()
    assert score.overflow == 0
    want_p, want_q = gp.p.cpu().numpy(), gp.q.cpu().numpy()
    hs = HostStream(GenomePass(eng, group=False), [n], [0], slots=2)
    h_p, h_q = _pinned(n), _pinned(n)
    hs.submit(h[0], h[1], h[2], h_p, h_q, smoothing=x).synchronize()
    assert _same_bits(h_p.numpy()[:n], want_p[:n]) and _same_bits(h_q.numpy()[:n], want_q[:n])
    assert _fit_cmp(hs.fit_of(0)) == _fit_cmp(raw) and hs.fit_of(0).smoothing == x

    base = _serial(eng, [_shard(cols)])
    s1 = _lib.FitResult.from_buffer_copy(base["fit1"]).smoothing
    s2 = _lib.FitResult.from_buffer_copy(base["fit2"]).smoothing
    hs = HostStream(GenomePass(eng, group=False), [n], [0], slots=2, refit=True)
    for pair in ((1.5 * s1, None), (None, 1.5 * s2)):
        ref = _serial(eng, [_shard(cols)], smoothing=pair, settle=False)
        h_p1, h_p, h_q = _pinned(n), _pinned(n), _pinned(n)
        hs.submit(h[0], h[1], h[2], h_p, h_q, h_p_first=h_p1, smoothing=pair).synchronize()
        _check(ref, real, h_p1.numpy(), h_p.numpy(), h_q.numpy())
        k = hs.submitted - 1
        f1, f2 = hs.fit_of(k, first=True), hs.fit_of(k)
        assert (_fit_cmp(f1), _fit_cmp(f2)) == (_fit_cmp(ref["fit1"]), _fit_cmp(ref["fit2"]))
        assert [f.smoothing for f, v in zip((f1, f2), pair) if v is not None] == [v for v in pair if v is not None]
    assert not _same_bits(ref["p"], base["p"])


# ------------------------------------------------------------------------------------------------------------ 6. deferred
def test_two_pass_stream_deferred_list_holds_every_row():
    """A slot of more than 2^20 rows, nearly all deferred by the streaming K4 in both passes: the one deferred list the two
    passes share has a place for every row, and both passes equal the serial ones (which repeat a pass whose list overflowed)."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import GenomePass, HostStream
    from blueberry_b200.engine import PassEngine
    lib = _lib.load()
    dev = torch.device("cuda:0")
    nb, K = 20050, 100
    n = int(lib.bbk_synth_n_pairs(nb, K))
    assert n > 1 << 20
    cols = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(3)]
    _lib.check(lib.bbk_synth_contacts(nb, K, R, 20000.0, 1.08, 3, None, _lib.ptr(cols[0]), _lib.ptr(cols[1]), _lib.ptr(cols[2]),
                                      _lib.stream_ptr()), "synth")
    eng = PassEngine(R, 100, 0, K * R, nb, dev)
    eng.set_fragments([nb], [(nb - 1) * R])
    ref = _serial(eng, [_shard(cols)])
    for gp in ref["passes"]:
        assert gp.listed and gp.last_score.n_list > max(1 << 20, n // 4)     # more than a default-size list holds
    h = _host(cols)
    hs = HostStream(GenomePass(eng, group=False), [n], [0], slots=2, refit=True)
    h_p1, h_p, h_q = _pinned(n), _pinned(n), _pinned(n)
    hs.submit(h[0], h[1], h[2], h_p, h_q, h_p_first=h_p1, smoothing=ref["s"])
    hs.drain()
    _check(ref, np.ones(n, bool), h_p1.numpy(), h_p.numpy(), h_q.numpy())
    assert _fit_cmp(hs.fit_of(0, first=True)) == _fit_cmp(ref["fit1"]) and _fit_cmp(hs.fit_of(0)) == _fit_cmp(ref["fit2"])
