"""GPU tests of the genome-wide pass in row blocks from host memory (distributed.BlockedPass): every case equals a resident
GenomePass(engine, group=False).run over the same shards, bit for bit - p and q of every row, K1's tables and totals, bins,
spline and spline_raw, the BbkFitResult without its SM cycle counters - whatever the block size and the residency budget;
plus bbk_bh_rank_gathered_all against bbk_bh_rank_gathered_padded, the oracle, and fit_transform_arrays on the blocked path."""
import numpy as np
import pytest

from helpers import log10_close

pytestmark = pytest.mark.gpu


def _fit_cmp(raw):
    raw = bytes(raw)
    return raw[:72] + raw[184:]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _genome(bins, R=10000, max_dist=2_000_000, depth=150.0, seed=31, bias_on=(0,), zero_rows=True):
    from blueberry_b200 import synth
    bias = synth.make_bias(bins, seed)
    for c in range(len(bins)):
        if c not in bias_on:
            bias[c] = np.ones(bins[c])
    c = synth.make_contacts(bins, R, max_dist, depth, seed, bias, keep_zeros=zero_rows)
    shards = []
    for k in range(len(bins)):
        sel = c["chrom"] == k
        shards.append((k, c["mid1"][sel].copy(), c["mid2"][sel].copy(), c["count"][sel].copy()))
    return dict(bins=bins, R=R, max_dist=max_dist, bias=bias, shards=shards, contacts=c)


def _engine(g, dev, n_bins=100, max_bins=None):
    from blueberry_b200.engine import BiasTables, PassEngine
    bins, R = g["bins"], g["R"]
    eng = PassEngine(R, n_bins, 0, g["max_dist"], max(bins), dev, max_bins=max_bins)
    eng.set_fragments(bins, [(b - 1) * R for b in bins])
    tabs = [np.where((b < 0.5) | (b > 2), -1.0, b) for b in g["bias"]]
    eng.set_bias(BiasTables(tabs, [R // 2] * len(bins), dev))
    return eng


def _state(eng, fit):
    return dict(obs=eng.obs_sum.cpu().numpy(), totals=eng.totals.cpu().numpy(), x=eng.x[:fit.n_out].cpu().numpy(),
                y=eng.y[:fit.n_out].cpu().numpy(), sy=eng.spline_y[:fit.L].cpu().numpy(), sr=eng.spline_raw[:fit.L].cpu().numpy(),
                fit=_fit_cmp(eng.fit_result.cpu().numpy().tobytes()))


def _resident(g, dev, q_values=True, n_tests=-1, force_exact=False, **ekw):
    import torch
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import Shard
    eng = _engine(g, dev, **ekw)
    gp = GenomePass(eng, group=False, q_values=q_values)
    gp.force_exact = force_exact
    gp.attach([Shard(*(torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev) for a in sh[1:]), chrom=sh[0]) for sh in g["shards"]])
    fit = gp.run(n_tests=n_tests)
    p = [gp.shard_p(i).cpu().numpy() for i in range(len(g["shards"]))]
    q = [gp.shard_q(i).cpu().numpy() for i in range(len(g["shards"]))] if q_values else None
    return fit, p, q, _state(eng, fit)


def _blocked(g, dev, q_values=True, n_tests=-1, force_exact=False, block_rows=1 << 27, resident_bytes=None, pinned=False,
             cand_capacity=None, **ekw):
    import torch
    from blueberry_b200.distributed import BlockedPass
    eng = _engine(g, dev, **ekw)
    bp = BlockedPass(eng, q_values=q_values, block_rows=block_rows, resident_bytes=resident_bytes, cand_capacity=cand_capacity)
    bp.force_exact = force_exact
    shards = g["shards"]
    if pinned:
        shards = [(c,) + tuple(torch.from_numpy(a).pin_memory() for a in sh) for c, *sh in shards]
        p = [torch.full((len(sh[1]),), -7.0, dtype=torch.float64).pin_memory() for sh in shards]
        q = [torch.full((len(sh[1]),), -7.0, dtype=torch.float64).pin_memory() for sh in shards] if q_values else None
    else:
        p = [np.full(len(sh[1]), -7.0) for sh in shards]
        q = [np.full(len(sh[1]), -7.0) for sh in shards] if q_values else None
    fit = bp.run(shards, p, q, n_tests=n_tests)
    p = [np.asarray(x) for x in p]
    q = [np.asarray(x) for x in q] if q_values else None
    return fit, p, q, _state(eng, fit), bp


def _assert_same(ref, got, q_values=True):
    fit_r, p_r, q_r, st_r = ref
    fit_b, p_b, q_b, st_b = got[:4]
    for k in st_r:
        if k == "fit":
            assert st_r[k] == st_b[k], "fit results differ"
        else:
            assert np.array_equal(_bits(st_r[k]) if st_r[k].dtype == np.float64 else st_r[k],
                                  _bits(st_b[k]) if st_b[k].dtype == np.float64 else st_b[k]), k
    for i in range(len(p_r)):
        assert np.array_equal(_bits(p_r[i]), _bits(p_b[i])), "p of shard %d" % i
        if q_values:
            assert np.array_equal(_bits(q_r[i]), _bits(q_b[i])), "q of shard %d" % i


@pytest.fixture(scope="module")
def dev():
    import torch
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def g3():
    return _genome([420, 300, 180], bias_on=(0, 2))


@pytest.fixture(scope="module")
def ref3(g3, dev):
    return _resident(g3, dev)


@pytest.mark.parametrize("block_rows", [1 << 27, 4096, 3 * 4096, 12_345, 5_003, 1 << 15])
def test_block_sizes(g3, ref3, dev, block_rows):
    got = _blocked(g3, dev, block_rows=block_rows)
    _assert_same(ref3, got)
    nb = len(got[4].blocks)
    assert nb == 1 if block_rows == 1 << 27 else nb > 1
    if block_rows in (12_345, 5_003):     # chromosomes cut inside, at rows that are not multiples of 4
        assert any(lo % 4 for b in got[4].blocks for (_, lo, _, _) in b)


@pytest.mark.parametrize("budget", ["all", "none", "half"])
def test_residency_budgets(g3, ref3, dev, budget):
    total = sum(len(sh[1]) for sh in g3["shards"]) * 12
    rb = {"all": None, "none": 0, "half": total // 2}[budget]
    got = _blocked(g3, dev, block_rows=8 * 4096, resident_bytes=rb)
    _assert_same(ref3, got)
    res = got[4].resident
    assert all(res) if budget == "all" else (not any(res) if budget == "none" else (any(res) and not all(res)))


def test_without_q_values(g3, dev):
    ref = _resident(g3, dev, q_values=False)
    _assert_same(ref, _blocked(g3, dev, q_values=False, block_rows=5 * 4096, resident_bytes=0), q_values=False)


@pytest.mark.parametrize("n_tests", [25, 10 ** 7, 40_000])
def test_n_tests(g3, dev, n_tests):
    ref = _resident(g3, dev, n_tests=n_tests)
    _assert_same(ref, _blocked(g3, dev, n_tests=n_tests, block_rows=9 * 4096, resident_bytes=50_000))
    if n_tests == 25:               # the fallback sweep over p, and q of the p == 1.0 rows below 1
        p, q = np.concatenate(ref[1]), np.concatenate(ref[2])
        assert (q[p == 1.0] < 1.0).all()


def test_candidate_lists_overflow(g3, ref3, dev):
    got = _blocked(g3, dev, block_rows=6 * 4096, cand_capacity=16)
    assert any(s.cand_overflow for s in got[4].last_states)
    _assert_same(ref3, got)


def test_exact_mode(g3, dev):
    ref = _resident(g3, dev, force_exact=True)
    _assert_same(ref, _blocked(g3, dev, force_exact=True, block_rows=7 * 4096))


def test_fit_wants_more_bins(g3, dev):
    ref = _resident(g3, dev, max_bins=4)
    got = _blocked(g3, dev, max_bins=4, block_rows=7 * 4096)
    assert ref[0].n_out > 4
    _assert_same(ref, got)


def test_fit_settled_on_reference_s(g3, dev, monkeypatch):
    from blueberry_b200.engine import PassEngine
    given = set()

    def ref_s(fit):                    # a reference s that differs from the kernel's once, as libm's pow does for ~0.09 % of inputs
        if fit.n_out <= 0 or fit.smoothing in given:
            return None
        s = fit.smoothing * 1.25
        given.add(s)
        return s

    monkeypatch.setattr(PassEngine, "reference_smoothing", staticmethod(ref_s))
    ref = _resident(g3, dev)
    got = _blocked(g3, dev, block_rows=7 * 4096, resident_bytes=0)
    assert ref[0].smoothing in given
    _assert_same(ref, got)


def test_all_zero_counts_raise_and_leave_outputs(dev):
    g = _genome([200, 150], bias_on=())
    g["shards"] = [(c, m1, m2, np.zeros_like(cn)) for c, m1, m2, cn in g["shards"]]
    with pytest.raises(ZeroDivisionError):
        _resident(g, dev)
    from blueberry_b200.distributed import BlockedPass
    bp = BlockedPass(_engine(g, dev), block_rows=4096)
    p = [np.full(len(sh[1]), -7.0) for sh in g["shards"]]
    q = [np.full(len(sh[1]), -7.0) for sh in g["shards"]]
    with pytest.raises(ZeroDivisionError):
        bp.run(g["shards"], p, q)
    assert all((x == -7.0).all() for x in p + q)


def test_pinned_inputs_and_outputs(g3, ref3, dev):
    _assert_same(ref3, _blocked(g3, dev, block_rows=11 * 4096, pinned=True, resident_bytes=100_000))


def test_genomes_of_one_to_five_chromosomes(dev):
    for bins, bias_on, zeros in (([350], (0,), True), ([260, 90, 400, 31, 150], (1, 3), False), ([500, 2], (), True)):
        g = _genome(bins, bias_on=bias_on, zero_rows=zeros, seed=len(bins) + 3)
        ref = _resident(g, dev)
        for br, rb in ((1 << 27, None), (4096, 0), (13 * 4096, 200_000)):
            _assert_same(ref, _blocked(g, dev, block_rows=br, resident_bytes=rb))


def test_config2_shape(dev):
    """BASELINE config 2's shape (5 kb, 10 Mb cap, a 5000-bin chromosome = 8.0e6 records) in blocks of 2^20 rows."""
    g = _genome([5000], R=5000, max_dist=10_000_000, depth=600.0, seed=5, bias_on=(0,))
    ref = _resident(g, dev)
    got = _blocked(g, dev, block_rows=1 << 20, resident_bytes=40 << 20)
    assert len(got[4].blocks) == 8 and any(got[4].resident) and not all(got[4].resident)
    _assert_same(ref, got)


def test_against_oracle_and_reference_q(dev):
    from oracle import fithic_oracle as fo
    g = _genome([420, 300, 180], bias_on=(0, 1, 2), seed=31)
    fit, p, q, st, bp = _blocked(g, dev, block_rows=5 * 4096, resident_bytes=0)
    p, q = np.concatenate(p), np.concatenate(q)
    c, bins, R = g["contacts"], g["bins"], g["R"]
    from blueberry_b200 import synth
    fc, fm = synth.make_fragments(bins, R)
    bc = np.concatenate([np.full(b, i) for i, b in enumerate(bins)])
    bd, _ = fo.read_bias_arrays(bc, fm, np.concatenate(g["bias"]))
    ref = fo.fithic_arrays(fc, fm, c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], R, 100, 0, g["max_dist"], bias=bd)
    assert np.array_equal(st["obs"], ref.contacts.observed) and int(fit.S) == ref.contacts.S
    assert np.array_equal(st["sy"], ref.spline_y)
    assert np.array_equal(p <= 1, ref.keep)
    sel = ref.keep & (ref.p > 0)
    ok, nbad = log10_close(p[sel], ref.p[sel], 1e-6)
    assert ok, nbad
    keep = ref.keep
    assert np.array_equal(q[keep], fo.benjamini_hochberg_correction(p[keep], int(keep.sum())))
    ok, nbad = log10_close(q[keep], fo.benjamini_hochberg_correction(ref.p[keep], int(keep.sum())), 1e-6)
    assert ok, nbad


def test_fit_transform_arrays_on_the_blocked_path(dev, monkeypatch):
    from blueberry_b200 import fithic, synth
    bins, R, max_dist = [300, 200, 120], 10000, 1_500_000
    bias = synth.make_bias(bins, 1)
    fc, fm = synth.make_fragments(bins, R)
    c = synth.make_contacts(bins, R, max_dist, 120.0, 11, bias)
    bc = np.concatenate([np.full(b, i, dtype=np.int32) for i, b in enumerate(bins)])
    model = fithic.FitHiC("blocked", R, n_bins=100, max_dist=max_dist, min_dist=0)

    def call(blocked, **kw):
        seen = []

        def route(rows, want_q, d):
            seen.append(rows)
            return blocked
        monkeypatch.setattr(fithic, "use_blocked_pass", route)
        out = model.fit_transform_arrays(c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], fc, fm,
                                         bias=(bc, fm, np.concatenate(bias)), **kw)
        assert seen
        return out

    for kw in (dict(q_values=True), dict(q_values=False), dict(q_values=True, n_tests=25)):
        a, b = call(False, **kw), call(True, **kw)
        for f in type(a).__slots__:
            if f == "gpu_launches":
                continue
            va, vb = getattr(a, f, None), getattr(b, f, None)
            if f == "fit":
                assert _fit_cmp(bytes(va)) == _fit_cmp(bytes(vb))
            elif isinstance(va, np.ndarray):
                assert va.dtype == vb.dtype and np.array_equal(va.view(np.uint8), vb.view(np.uint8)), f
            elif f == "frag":
                assert type(va) is type(vb)
            else:
                assert va == vb, f


def test_rank_gathered_all_equals_per_rank_padded(dev):
    import torch
    from blueberry_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(4)
    world, cap = 5, 3000
    counts = [3000, 0, 1234, 2999, 17]
    recv = np.zeros(world * (cap + 1), dtype=np.uint64)
    for r, n in enumerate(counts):
        p = rng.random(n) * 0.03
        p[: n // 7] = p[0] if n else 0.0              # ties across blocks
        recv[r * (cap + 1)] = n
        recv[r * (cap + 1) + 1:r * (cap + 1) + 1 + n] = p.view(np.uint64) | np.uint64(1 << 63)
    tau = int(np.array([0.03125]).view(np.uint64)[0]) | (1 << 63)
    state = torch.tensor(np.array([counts[0], tau, 40_000, 5], dtype=np.uint64).view(np.int64), device=dev)
    d_recv = torch.from_numpy(recv.view(np.int64)).to(dev)
    ws = torch.empty(int(lib.bbk_bh_gathered_workspace_bytes(world, cap)), dtype=torch.uint8, device=dev)
    st = _lib.stream_ptr()
    q_all = torch.full((world * cap,), -3.0, dtype=torch.float64, device=dev)
    ones_a = torch.zeros(2, dtype=torch.float64, device=dev)
    ov_a = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(lib.bbk_bh_rank_gathered_all(_lib.ptr(d_recv), world, cap, _lib.ptr(state), _lib.ptr(q_all), _lib.ptr(ones_a), _lib.ptr(ov_a),
                                            _lib.ptr(ws), ws.numel(), st), "bbk_bh_rank_gathered_all")
    idx = torch.arange(cap, dtype=torch.int32, device=dev)
    qa = q_all.cpu().numpy()
    for r in range(world):
        q_r = torch.full((cap,), -5.0, dtype=torch.float64, device=dev)
        ones = torch.zeros(2, dtype=torch.float64, device=dev)
        ov = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.bbk_bh_rank_gathered_padded(_lib.ptr(d_recv), world, cap, r, _lib.ptr(state), _lib.ptr(idx), _lib.ptr(q_r),
                                                   _lib.ptr(ones), _lib.ptr(ov), _lib.ptr(ws), ws.numel(), st), "padded")
        n = counts[r]
        assert np.array_equal(_bits(q_r.cpu().numpy()[:n]), _bits(qa[r * cap:r * cap + n]))
        assert (qa[r * cap + n:(r + 1) * cap] == -3.0).all()
        assert np.array_equal(_bits(ones.cpu().numpy()), _bits(ones_a.cpu().numpy()))
        assert int(ov.item()) == int(ov_a.item()) == 0
    with pytest.raises(_lib.BbkError):
        _lib.check(lib.bbk_bh_rank_gathered_all(_lib.ptr(d_recv), 2, 1 << 31, _lib.ptr(state), _lib.ptr(q_all), _lib.ptr(ones_a),
                                                _lib.ptr(ov_a), _lib.ptr(ws), ws.numel(), st), "bbk_bh_rank_gathered_all")
