"""GPU tests of packed contact records (include/bbk.h, BbkRecHeader): PackedRecords.to_device against the columns they were
packed from, and distributed.HostStream fed PackedRecords against the same stream fed the int32 columns, bit for bit (p, q
and fit results, dense and packed results, GenomePass and ChromosomePass).  Every buffer that reaches the device has passed
bbkio_check_records on the host first."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R, N_BINS = 5000, 100
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).tobytes() if a.size else b""


def _fit_cmp(raw):
    """The bytes of a BbkFitResult that a fit defines, without the SM cycle counters."""
    raw = bytes(raw)
    return raw[:72] + raw[184:]


def _fits(x):
    return [_fit_cmp(bytes(f)) for f in (x if isinstance(x, list) else [x])]


def _expected(shards):
    from blueberry_b200.distributed import layout_rows
    starts, rows = layout_rows([len(s[0]) for s in shards])
    cols = [np.zeros(rows, dtype=np.int32) for _ in range(3)]
    for a, sh in zip(starts, shards):
        for j in range(3):
            cols[j][a:a + len(sh[j])] = sh[j]
    return cols


def _host_cases():
    rng = np.random.default_rng(11)

    def row_major(n, K=2000):
        i = np.arange(n, dtype=np.int64)
        m1 = (i // (K + 1)) * R + R // 2
        return (m1.astype(np.int32), (m1 + (i % (K + 1)) * R).astype(np.int32), rng.poisson(3.0, n).astype(np.int32))

    def full(n):
        return tuple(rng.integers(I32_MIN, I32_MAX, n, endpoint=True, dtype=np.int64).astype(np.int32) for _ in range(3))

    cases = [[row_major(n)] for n in (0, 1, 3, 4095, 4096, 4097, 3 * 4096 + 5)]
    cases.append([row_major(n) for n in (5, 0, 4093, 1, 6000, 3)])
    n = 5000
    cases.append([(np.zeros(n, np.int32),) * 3])
    cases.append([(np.full(n, I32_MIN, np.int32), np.full(n, I32_MAX, np.int32), np.full(n, I32_MAX, np.int32))])
    cases.append([(np.full(n, I32_MAX, np.int32), np.full(n, I32_MIN, np.int32), np.full(n, I32_MIN, np.int32))])
    cases.append([(np.resize(np.array([I32_MIN, I32_MAX, 0, 0], np.int32), n), np.resize(np.array([I32_MAX, I32_MIN, 0, 1], np.int32), n),
                   np.resize(np.array([I32_MIN, I32_MAX, 7, 0], np.int32), n))])          # a 33-bit e
    cases.append([full(9001), full(4096), full(3)])
    return cases


def test_to_device_equals_the_packed_columns():
    import torch
    from blueberry_b200.distributed import pack_records
    dev = torch.device("cuda", 0)
    for shards in _host_cases():
        rec = pack_records(shards)
        got = rec.to_device(dev)
        want = _expected(shards)
        torch.cuda.synchronize()
        for g, w in zip(got, want):
            assert g.numel() == w.size
            assert np.array_equal(g.cpu().numpy(), w)


def test_to_device_on_a_large_row_major_block():
    """5e7 rows of BASELINE config 2's shape (chr1 @ 5 kb, all pairs within 10 Mb, zeros kept), generated on the device."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import pack_records
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    n, nb, K = 50_000_000, 49851, 2000
    cols = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(3)]
    _lib.check(lib.bbk_synth_contacts_range(nb, K, R, 25.0, 1.08, 17, None, 0, n, _lib.ptr(cols[0]), _lib.ptr(cols[1]), _lib.ptr(cols[2]),
                                            _lib.stream_ptr()), "synth")
    host = [c.cpu().numpy() for c in cols]
    rec = pack_records([tuple(host)])
    assert rec.nbytes < 4 * n
    got = rec.to_device(dev)
    for g, c in zip(got, cols):
        assert torch.equal(g, c)


# ---------------------------------------------------------------------------------------------------------------- HostStream
def _genome(seed, bins, max_dist, depth):
    """Per-chromosome (mid1, mid2, count) numpy columns, every pair within max_dist (zeros kept), and per-chromosome biases."""
    from blueberry_b200 import synth
    bias = synth.make_bias(bins, seed, sigma=0.3)
    c = synth.make_contacts(bins, R, max_dist, depth, seed, bias)
    return [tuple(np.ascontiguousarray(c[k][c["chrom"] == i]) for k in ("mid1", "mid2", "count")) for i in range(len(bins))], bias


def _genome_engine(bins, max_dist, bias, dev):
    from blueberry_b200.engine import BiasTables, PassEngine
    eng = PassEngine(R, N_BINS, 0, max_dist, max(bins), dev)
    eng.set_fragments(bins, [(b - 1) * R for b in bins])
    eng.set_bias(BiasTables([np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias], [R // 2] * len(bins), dev))
    return eng


def _chrom_engines(bins, max_dist, bias, dev):
    from blueberry_b200.engine import BiasTables, PassEngine
    tables = BiasTables([np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias], [R // 2] * len(bins), dev)
    es = []
    for nb in bins:
        e = PassEngine(R, N_BINS, 0, max_dist, nb, dev)
        e.set_fragments([nb], [(nb - 1) * R])
        e.set_bias(tables)
        es.append(e)
    return es


def _pinned(shards, rows):
    """Pinned int32 host columns of the pass layout (what a caller of the column form fills)."""
    import torch
    cols = _expected(shards)
    h = [torch.zeros(max(rows, 4), dtype=torch.int32).pin_memory() for _ in range(3)]
    for t, c in zip(h, cols):
        t[:c.size] = torch.from_numpy(c)
    return h


def _dense_pair(hs, shards, sizes=None, with_q=True, rec=None):
    """One pass fed columns, then the same records fed packed, both with dense results: (p, q, fits) of each."""
    import torch
    from blueberry_b200.distributed import layout_rows, pack_records
    starts, rows = layout_rows([len(s[0]) for s in shards])
    n = max(rows, 4)
    out = []
    for packed in (False, True):
        h_p = torch.full((n,), 7.0, dtype=torch.float64).pin_memory()
        h_q = torch.full((n,), 7.0, dtype=torch.float64).pin_memory() if with_q else None
        if packed:
            rec = pack_records(shards, out=rec)
            ev = hs.submit(rec, h_p=h_p, h_q=h_q, sizes=sizes)
        else:
            h = _pinned(shards, rows)
            ev = hs.submit(h[0], h[1], h[2], h_p, h_q, sizes=sizes)
        ev.synchronize()
        k = hs.submitted - 1
        real = np.zeros(n, bool)
        for a, s in zip(starts, shards):
            real[a:a + len(s[0])] = True
        p = h_p.numpy()[real].copy()
        q = h_q.numpy()[real].copy() if with_q else None
        out.append((_bits(p), _bits(q) if with_q else None, _fits(hs.fit_of(k))))
    return out, rec


def _packed_pair(hs, shards):
    """The same with packed results: (p, q, fits) fed columns, then fed PackedRecords."""
    from blueberry_b200.distributed import layout_rows, pack_records
    rows = layout_rows([len(s[0]) for s in shards])[1]
    out = []
    for packed in (False, True):
        o = hs.packed_buffers()
        if packed:
            hs.submit_packed(pack_records(shards), out=o)
        else:
            h = _pinned(shards, rows)
            hs.submit_packed(h[0], h[1], h[2], o)
        hs.drain()
        p, q = o.dense()
        out.append((_bits(p), _bits(q) if q is not None else None, _fits(hs.fit_of(hs.submitted - 1))))
    return out


def test_host_stream_genome_pass_one_shard():
    import torch
    from blueberry_b200.distributed import GenomePass, HostStream
    dev = torch.device("cuda", 0)
    bins = [900]
    shards, bias = _genome(3, bins, 400 * R, 60.0)
    eng = _genome_engine(bins, 400 * R, bias, dev)
    sizes = [len(s[0]) for s in shards]
    hs = HostStream(GenomePass(eng, group=False), sizes, [0], slots=2)
    (a, b), _ = _dense_pair(hs, shards)
    assert a == b
    hs = HostStream(GenomePass(eng, group=False), sizes, [0], slots=2, packed=True)
    a, b = _packed_pair(hs, shards)
    assert a == b


def test_host_stream_genome_pass_several_shards_smaller_passes_and_an_empty_shard():
    import torch
    from blueberry_b200.distributed import GenomePass, HostStream
    dev = torch.device("cuda", 0)
    bins = [700, 500, 40, 650]
    shards, bias = _genome(4, bins, 300 * R, 80.0)
    eng = _genome_engine(bins, 300 * R, bias, dev)
    full = [len(s[0]) for s in shards]
    chroms = list(range(len(bins)))
    hs = HostStream(GenomePass(eng, group=False), full, chroms, slots=2)
    (a, b), rec = _dense_pair(hs, shards)
    assert a == b
    # smaller passes through sizes=: ragged cuts, one chromosome without records
    for cut in ([full[0] - 3, 0, full[2], full[3] - 1001], [5, full[1] - 2, 0, 17]):
        part = [tuple(c[:n] for c in s) for s, n in zip(shards, cut)]
        (a, b), rec = _dense_pair(hs, part, sizes=cut, rec=rec)
        assert a == b
    hs = HostStream(GenomePass(eng, group=False), full, chroms, slots=2, packed=True)
    a, b = _packed_pair(hs, shards)
    assert a == b


def test_host_stream_chromosome_pass_with_q_values():
    import torch
    from blueberry_b200.distributed import ChromosomePass, HostStream
    from blueberry_b200.engine import Shard
    dev = torch.device("cuda", 0)
    bins = [600, 450, 300]
    shards, bias = _genome(5, bins, 250 * R, 70.0)
    chroms = [0, 1, 2]
    sizes = [len(s[0]) for s in shards]

    def cpass():
        es = _chrom_engines(bins, 250 * R, bias, dev)
        return ChromosomePass(es, [Shard(*(torch.from_numpy(c).to(dev) for c in s), chrom=i) for s, i in zip(shards, chroms)])

    hs = HostStream(cpass(), sizes, chroms, slots=2)
    (a, b), _ = _dense_pair(hs, shards)
    assert a == b and len(a[2]) == 3
    hs = HostStream(cpass(), sizes, chroms, slots=2, packed=True)
    a, b = _packed_pair(hs, shards)
    assert a == b


def test_host_stream_alternating_packed_records_and_a_pass_without_q():
    """Four submissions alternating two PackedRecords of different records (two slots, one inbound buffer), then a pass
    without h_q: each equals the column-fed pass over the same records."""
    import torch
    from blueberry_b200.distributed import GenomePass, HostStream, layout_rows, pack_records
    dev = torch.device("cuda", 0)
    bins = [800]
    libs = []
    for seed, depth in ((6, 50.0), (7, 90.0)):
        shards, bias = _genome(seed, bins, 300 * R, depth)
        libs.append(shards)
    eng = _genome_engine(bins, 300 * R, bias, dev)
    sizes = [len(libs[0][0][0])]
    rows = max(layout_rows(sizes)[1], 4)
    hs = HostStream(GenomePass(eng, group=False), sizes, [0], slots=2)
    want = []
    for shards in libs:
        h = _pinned(shards, rows)
        h_p, h_q = (torch.empty(rows, dtype=torch.float64).pin_memory() for _ in range(2))
        hs.submit(h[0], h[1], h[2], h_p, h_q).synchronize()
        want.append((_bits(h_p.numpy()[:sizes[0]]), _bits(h_q.numpy()[:sizes[0]]), _fits(hs.fit_of(hs.submitted - 1))))
    assert want[0][0] != want[1][0]
    recs = [pack_records(s) for s in libs]
    outs = []
    for k in range(4):
        h_p, h_q = (torch.empty(rows, dtype=torch.float64).pin_memory() for _ in range(2))
        outs.append((h_p, h_q, hs.submit(recs[k % 2], h_p=h_p, h_q=h_q), hs.submitted - 1))
    for k, (h_p, h_q, ev, idx) in enumerate(outs):
        ev.synchronize()
        got = (_bits(h_p.numpy()[:sizes[0]]), _bits(h_q.numpy()[:sizes[0]]))
        assert got == want[k % 2][:2], "submission %d" % k
        if k >= 2:
            assert _fits(hs.fit_of(idx)) == want[k % 2][2]
    # without h_q: the pass skips the q-value step; p equals the column-fed pass without h_q
    (a, b), _ = _dense_pair(hs, libs[1], with_q=False, rec=recs[0])
    assert a == b and a[0] == want[1][0]


def test_host_stream_rejects_bad_packed_records_before_any_copy():
    import torch
    from blueberry_b200.distributed import GenomePass, HostStream, PackedRecords, pack_records
    dev = torch.device("cuda", 0)
    bins = [300]
    shards, bias = _genome(8, bins, 100 * R, 40.0)
    eng = _genome_engine(bins, 100 * R, bias, dev)
    n = len(shards[0][0])
    h_p = torch.empty(n + 4, dtype=torch.float64).pin_memory()
    rec = pack_records(shards)
    hs = HostStream(GenomePass(eng, group=False), [n], [0], slots=2, cap_in=rec.nbytes - 16)

    def rejected(r, **kw):
        before = hs.submitted
        with pytest.raises(ValueError):
            hs.submit(r, h_p=h_p, **kw)
        assert hs.submitted == before and hs.d_in is None          # no pass queued, no buffer allocated or copied into

    rejected(rec)                                                    # more bytes than cap_in
    hs = HostStream(GenomePass(eng, group=False), [n], [0], slots=2)
    other = pack_records([tuple(c[:n - 8] for c in shards[0])])
    rejected(other)                                                  # another layout
    rejected(rec, sizes=[n - 8])                                     # the pass' sizes= differ from the records'
    bad = pack_records(shards, out=PackedRecords(rec.buf.numel()))
    bad.buf[0] ^= 0xFF                                               # fails validation (magic)
    rejected(bad)
    trunc = pack_records(shards)
    trunc.nbytes -= 1                                                # truncated
    rejected(trunc)
    with pytest.raises(ValueError):
        bad.to_device(dev)
    with pytest.raises(ValueError):
        pack_records(shards, out=PackedRecords(64))                  # too small to refill
    hs.submit(rec, h_p=h_p).synchronize()                            # the stream still works
    assert hs.submitted == 1
