"""GPU tests: (1) the path-based drop-in (gzip text in, significances.txt.gz out, stage functions) against the
golden outputs of the reference; (2) size-independent properties at BASELINE's full config-2 size."""
import gzip
import os

import numpy as np
import pytest

from helpers import load_golden, log10_close

pytestmark = pytest.mark.gpu


def _write_inputs(tmp, g):
    def name(c):
        return "chr%d" % (int(c) + 1)
    inter = os.path.join(tmp, "interactions.gz")
    frags = os.path.join(tmp, "fragments.gz")
    with gzip.open(inter, "wt") as fh:
        for a, b, c, d, e in zip(g["chr1"], g["mid1"], g["chr2"], g["mid2"], g["count"]):
            fh.write("%s\t%d\t%s\t%d\t%d\n" % (name(a), b, name(c), d, e))
    with gzip.open(frags, "wt") as fh:
        for c, m in zip(g["frag_chrom"], g["frag_mid"]):
            fh.write("%s\t%d\t0\t0\t0\n" % (name(c), m))
    bias = "none"
    if bool(g["has_bias"]):
        bias = os.path.join(tmp, "biases.gz")
        with gzip.open(bias, "wt") as fh:
            for c, m, b in zip(g["bias_chrom"], g["bias_mid"], g["bias_val"]):
                fh.write("%s\t%d\t%r\n" % (name(c), m, float(b)))
    return inter, frags, bias


def _parse(path):
    rows = []
    with gzip.open(path, "rt") as fh:
        header = fh.readline()
        for line in fh:
            rows.append(line.rstrip("\n").split("\t"))
    return header, rows


@pytest.mark.parametrize("name", ["pass_bias_dense", "pass_messy"])
def test_fit_transform_files_match_reference_output(name, tmp_path):
    from blueberry_b200.fithic import FitHiC
    g = load_golden(name)
    inter, frags, bias = _write_inputs(str(tmp_path), g)
    R = int(g["resolution"])
    lib = os.path.join(str(tmp_path), "lib")
    model = FitHiC(lib, R, n_bins=int(g["n_bins"]), max_dist=int(g["max_dist_arg"]), min_dist=int(g["min_dist_arg"]))
    assert model.fit_transform(inter, frags, bias) is None                    # fithic.py:85-108 returns None
    assert os.path.exists("%s.fithic_pass1.res%d.txt" % (lib, R))             # opened, never written (fithic.py:164)
    header, rows = _parse("%s.spline_pass1.res%d.significances.txt.gz" % (lib, R))
    assert header == "chr1\tfragmentMid1\tchr2\tfragmentMid2\tcontactCount\tp-value\tq-value\n"   # fithic.py:411
    assert len(rows) == len(g["ref_out_p"])
    assert [int(r[1]) for r in rows] == g["ref_out_mid1"].tolist()
    assert [int(r[3]) for r in rows] == g["ref_out_mid2"].tolist()
    assert [int(r[4]) for r in rows] == g["ref_out_count"].tolist()
    assert [r[0] for r in rows] == ["chr%d" % (c + 1) for c in g["ref_out_chr1"]]
    assert all(r[6] == "-1" for r in rows)                                     # fithic.py:435
    ok, nbad = log10_close(np.array([float(r[5]) for r in rows]), g["ref_out_p"], 1e-6)
    assert ok, nbad


def test_stage_functions_drop_in(tmp_path):
    """generate_FragPairs -> read_interactions -> calculate_probabilities -> fit_spline, as fithic() chains them."""
    from blueberry_b200 import fithic as f
    g = load_golden("pass_bias_dense")
    inter, frags, bias = _write_inputs(str(tmp_path), g)
    R, lo, hi = int(g["resolution"]), int(g["ref_min_dist"]), int(g["ref_max_dist"])
    main = f.generate_FragPairs(frags, R, lo, hi, False)
    assert sorted(main) == [k * R for k in range(len(g["ref_possible"]))]
    assert [main[k][0] for k in sorted(main)] == g["ref_possible"].tolist()
    assert f.possibleIntraInRangeCount == int(g["ref_possible_intra_in_range"])
    bias_dic = f.read_bias_file(bias, False)
    main = f.read_interactions(main, inter, lo, hi, False)
    assert [main[k][1] for k in sorted(main)] == g["ref_observed"].tolist()
    assert f.observedIntraInRangeSum == int(g["ref_S"])
    x, y, yerr = f.calculate_probabilities(main, int(g["n_bins"]), R, lo, hi, os.path.join(str(tmp_path), "l.fithic_pass1"), False)
    assert x == g["ref_x"].tolist() and y == g["ref_y"].tolist() and yerr == [0.0] * len(x)
    sx, sy, residual = f.fit_spline(main, x, y, yerr, inter, os.path.join(str(tmp_path), "l.spline_pass1"), bias_dic, R, lo, hi, False)
    assert sx == g["ref_spline_x"].tolist()
    assert np.allclose(sy, g["ref_spline_y"], rtol=1e-12, atol=0)
    header, rows = _parse(os.path.join(str(tmp_path), "l.spline_pass1.res%d.significances.txt.gz" % R))
    assert len(rows) == len(g["ref_out_p"])
    ok, nbad = log10_close(np.array([float(r[5]) for r in rows]), g["ref_out_p"], 1e-6)
    assert ok, nbad


def test_full_size_properties_config2_genome_pass():
    """BASELINE config 2 (chr1 @ 5 kb, 97,750,851 records) generated on the device: properties that need no oracle."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import BiasTables, PassEngine, Shard
    lib = _lib.load()
    dev = torch.device("cuda:0")
    R, nb, K, max_dist = 5000, 49851, 2000, 10_000_000
    P = int(lib.bbk_synth_n_pairs(nb, K))
    assert P == 97750851
    rng = np.random.default_rng(5)
    bias_host = np.exp(rng.normal(0.0, 0.25, size=nb))
    bias_dev = torch.from_numpy(bias_host).to(dev)
    mid1 = torch.empty(P, dtype=torch.int32, device=dev)
    mid2 = torch.empty(P, dtype=torch.int32, device=dev)
    count = torch.empty(P, dtype=torch.int32, device=dev)
    _lib.check(lib.bbk_synth_contacts(nb, K, R, 600.0, 1.08, 99, _lib.ptr(bias_dev), _lib.ptr(mid1), _lib.ptr(mid2),
                                      _lib.ptr(count), _lib.stream_ptr()), "synth")
    eng = PassEngine(R, 100, 0, max_dist, nb, dev)
    eng.set_fragments([nb], [(nb - 1) * R])
    eng.set_bias(BiasTables([np.where((bias_host < 0.5) | (bias_host > 2), -1.0, bias_host)], [R // 2], dev))
    gp = GenomePass(eng, group=False)
    gp.attach([Shard(mid1, mid2, count)])
    gp.run()
    p, q = gp.shard_p(0), gp.shard_q(0)
    fit = eng.read_fit()
    d = (mid2 - mid1).long()
    # K1: a checksum of checksums - the table must hold exactly the in-range counts, distance by distance
    in_range = (d > 0) & (d <= max_dist)
    S = int(count[in_range].long().sum().item())
    assert int(eng.totals[0].item()) == S == fit.S
    assert int(eng.obs_sum.sum().item()) == S
    ref_hist = torch.zeros(nb, dtype=torch.int64, device=dev).index_add_(0, (d[in_range] // R), count[in_range].long())
    assert torch.equal(ref_hist, eng.obs_sum)
    assert int(eng.totals[1].item()) == int(in_range.sum().item())
    assert int(eng.totals[3].item()) == P and int(eng.totals[2].item()) == int(count.long().sum().item())
    assert (int(eng.totals[6].item()), int(eng.totals[7].item())) == (R, max_dist)
    # K2a: closed form
    k = torch.arange(nb, device=dev)
    assert torch.equal(eng.possible, nb - k)
    # K3: the fitted prior is positive and non-increasing over the grid
    sy = eng.spline_y[:fit.L]
    assert bool((sy > 0).all()) and bool((sy[1:] <= sy[:-1]).all())
    # K4: zero counts -> exactly 1 (or NaN when a bias is discarded); everything else in (0, 1]; more contacts
    # at the same prior never give a larger p
    ok_bias = torch.from_numpy((bias_host >= 0.5) & (bias_host <= 2)).to(dev)
    i1 = (mid1 - R // 2) // R
    i2 = (mid2 - R // 2) // R
    # a discarded bias is -1 (fithic.py:147-149): exactly one of the two makes the prior negative and the row is
    # dropped (:434); two of them multiply to +1 and the row is scored - as in the reference
    valid = ok_bias[i1] == ok_bias[i2]
    assert bool(torch.isnan(p[~valid]).all()) and not bool(torch.isnan(p[valid]).any())
    assert bool((p[valid & (count == 0)] == 1.0).all())
    pv = p[valid]
    assert bool(((pv >= 0) & (pv <= 1)).all())
    # K5: q is NaN exactly where p is, q >= p, and sorting by p sorts q (forward running max)
    assert torch.equal(torch.isnan(q), torch.isnan(p))
    qv = q[valid]
    assert bool((qv >= pv).all()) and bool((qv <= 1).all())
    n_valid = int(valid.sum().item())
    cand = pv < 1e-3
    ps, order = torch.sort(pv[cand])
    qs = qv[cand][order]
    assert bool((qs[1:] >= qs[:-1]).all())
    # exact BH on the smallest 10^5 p-values (ranks below any saturation point are exact ranks)
    top = min(100000, ps.numel())
    ps_h, qs_h = ps[:top].cpu().numpy(), qs[:top].cpu().numpy()
    bh = np.maximum.accumulate(np.minimum(ps_h * n_valid / np.arange(1, top + 1), 1))
    # ties share the first tie's value: compare through the oracle's tie-aware formulation
    first = np.searchsorted(ps_h, ps_h, side="left")
    bh_t = np.maximum.accumulate(np.minimum(ps_h * n_valid / (first + 1), 1))
    assert np.array_equal(qs_h, bh_t) or np.array_equal(qs_h, bh)


def test_config1_full_size_against_oracle():
    """BASELINE config 1 in full (chr21 @ 10 kb, 4,813 bins, no effective distance cap, 11,584,891 records):
    the device pass against the CPU oracle on identical records (generated on the device, copied to the host)."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.fithic import FitHiC
    from blueberry_b200 import synth
    from oracle import fithic_oracle as fo
    lib = _lib.load()
    dev = torch.device("cuda:0")
    R, nb = 10000, 4813
    K = nb - 1
    max_dist = 48_130_000
    P = int(lib.bbk_synth_n_pairs(nb, K))
    assert P == 11584891
    rng = np.random.default_rng(21)
    bias_host = np.exp(rng.normal(0.0, 0.25, size=nb))
    bias_dev = torch.from_numpy(bias_host).to(dev)
    mid1 = torch.empty(P, dtype=torch.int32, device=dev)
    mid2 = torch.empty(P, dtype=torch.int32, device=dev)
    count = torch.empty(P, dtype=torch.int32, device=dev)
    _lib.check(lib.bbk_synth_contacts(nb, K, R, 3000.0, 1.08, 2021, _lib.ptr(bias_dev), _lib.ptr(mid1), _lib.ptr(mid2),
                                      _lib.ptr(count), _lib.stream_ptr()), "synth")
    m1, m2, c = mid1.cpu().numpy(), mid2.cpu().numpy(), count.cpu().numpy()
    fc, fm = synth.make_fragments([nb], R)
    bc = np.zeros(nb, dtype=np.int32)
    model = FitHiC("cfg1", R, n_bins=100, max_dist=max_dist)
    out = model.fit_transform_arrays(None, m1, None, m2, c, fc, fm, bias=(bc, fm, bias_host), q_values=True)
    bd, _ = fo.read_bias_arrays(bc, fm, bias_host)
    ref = fo.fithic_arrays(fc, fm, None, m1, None, m2, c, R, 100, model.min_dist, model.max_dist, bias=bd)
    assert np.array_equal(out.possible, ref.frag.possible)
    assert np.array_equal(out.observed, ref.contacts.observed)
    assert out.totals["observedIntraInRangeSum"] == ref.contacts.S < 2 ** 31
    assert np.array_equal(out.bin_of_key, ref.bin_of_key)
    assert np.array_equal(out.x, np.array(ref.x)) and np.array_equal(out.y, np.array(ref.y))
    assert out.spline_x[0] == ref.k0 * R and len(out.spline_y) == len(ref.spline_y)
    assert np.array_equal(out.spline_y, ref.spline_y)
    assert np.array_equal(out.keep, ref.keep)
    k = ref.keep & (ref.p >= 1e-300)
    err = np.abs(np.log10(out.p[k]) - np.log10(ref.p[k]))
    print("config 1: S=%d, %d rows kept, max |dlog10 p| vs oracle %.3g (p99 %.3g)" % (ref.contacts.S, int(ref.keep.sum()), err.max(), np.percentile(err, 99)))
    assert err.max() <= 1e-5
    assert (out.p[ref.keep & (ref.p < 1e-300)] <= 1e-299).all()
    qref = fo.benjamini_hochberg_correction(out.p[out.keep], int(out.keep.sum()))
    assert np.array_equal(out.q[out.keep], qref)


def test_nan_and_odd_bias_values_follow_the_reference():
    """A bias file may hold anything float() parses: `nan` passes read_bias_file's range test (fithic.py:147-149) and makes the
    prior NaN, so every row touching that locus is dropped (fithic.py:431-434) - also next to a discarded (-1) locus and for
    zero counts; `inf` is > 2 and becomes -1.  The dense device table marks missing loci with NaN, so these must not be
    mistaken for missing ones."""
    from blueberry_b200 import synth
    from blueberry_b200.fithic import FitHiC
    from oracle import fithic_oracle as fo
    R, bins, max_dist = 10000, [260], 1_200_000
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, 4, sigma=0.3)[0]
    bias[[7, 50, 51, 200]] = np.nan
    bias[[60, 120]] = np.inf
    bias[90] = 0.1                                              # discarded: -1
    c = synth.make_contacts(bins, R, max_dist, 200.0, 9, [np.where(np.isfinite(bias), bias, 1.0)])
    bc = np.zeros(bins[0], dtype=np.int32)
    keep_idx = np.r_[0:30, 31:bins[0]]                          # one locus missing from the file altogether
    model = FitHiC("nanbias", R, max_dist=max_dist)
    out = model.fit_transform_arrays(None, c["mid1"], None, c["mid2"], c["count"], fc, fm, bias=(bc[keep_idx], fm[keep_idx], bias[keep_idx]), q_values=True)
    bd, _ = fo.read_bias_arrays(bc[keep_idx], fm[keep_idx], bias[keep_idx])
    ref = fo.fithic_arrays(fc, fm, None, c["mid1"], None, c["mid2"], c["count"], R, 100, model.min_dist, model.max_dist, bias=bd)
    assert np.array_equal(out.keep, ref.keep)
    touched = np.isin(c["mid1"], fm[[7, 50, 51, 200]]) | np.isin(c["mid2"], fm[[7, 50, 51, 200]])
    assert touched.any() and not out.keep[touched].any()
    k = ref.keep & (ref.p > 0)
    assert np.abs(np.log10(out.p[k]) - np.log10(ref.p[k])).max() <= 1e-6


@pytest.mark.parametrize("shift", [2500, 1234])
def test_bias_loci_off_the_fragment_grid(shift):
    """The reference takes ANY bias file: biasDic[chr][mid] is an exact-key lookup (fithic.py:418-425).  Loci that are not on the
    fragments' grid put the dense device tables on the coarsest grid that holds them all; rows whose mids hit such a locus get
    its bias, rows on the vacated grid positions get 1.0 - through the streaming K4 and through the general kernel."""
    from blueberry_b200 import synth
    from blueberry_b200.fithic import FitHiC
    from oracle import fithic_oracle as fo
    R, bins, max_dist = 10000, [240], 1_000_000
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, 6, sigma=0.3)[0]
    c = synth.make_contacts(bins, R, max_dist, 150.0, 13, [bias])
    bm = fm.copy()
    moved = np.array([5, 40, 41, 130, 239])
    bm[moved] += shift                                          # these loci are NOT where the fragments are
    m1, m2 = c["mid1"].copy(), c["mid2"].copy()
    rng = np.random.default_rng(shift)
    for j in moved:                                             # some rows sit exactly on the moved loci, the others keep the vacated mids
        hit = np.flatnonzero(c["mid2"] == fm[j])
        take = hit[rng.random(len(hit)) < 0.5]
        m2[take] = bm[j]
    bc = np.zeros(bins[0], dtype=np.int32)
    model = FitHiC("offgrid", R, max_dist=max_dist)
    bd, _ = fo.read_bias_arrays(bc, bm, bias)
    ref = fo.fithic_arrays(fc, fm, None, m1, None, m2, c["count"], R, 100, model.min_dist, model.max_dist, bias=bd)
    for chrom_cols in (False, True):                            # compact shard (streaming K4) / chromosome columns (general kernel)
        ch = np.zeros(len(m1), dtype=np.int32) if chrom_cols else None
        if chrom_cols:
            ch2 = ch.copy()
            out = model.fit_transform_arrays(ch, m1, ch2, m2, c["count"], fc, fm, bias=(bc, bm, bias), q_values=True)
        else:
            out = model.fit_transform_arrays(None, m1, None, m2, c["count"], fc, fm, bias=(bc, bm, bias), q_values=True)
        assert np.array_equal(out.keep, ref.keep)
        k = ref.keep & (ref.p > 0)
        assert np.abs(np.log10(out.p[k]) - np.log10(ref.p[k])).max() <= 1e-6
    assert len(np.unique(ref.p[np.isin(m2, bm[moved])])) > 1    # the moved loci were really used


def test_decimate_matches_reference_golden_and_oracle(tmp_path):
    """K7 (bbk_decimate through FithicContactMap.decimate) against the golden output of the reference's own method
    (tests/golden/decimate.npz), bit for bit including the order-dependent sum and product, then against the oracle on
    larger inputs: unsorted files, exact duplicates, one giant group, a single row, an empty map."""
    from blueberry_b200.datatypes import FithicContactMap
    from oracle import datatypes_oracle as do
    g = load_golden("decimate")
    cm = FithicContactMap.from_arrays(g["map_in"], resolution=1000)
    cm.decimate(5000)
    assert cm.resolution == 5000
    assert np.array_equal(cm.map, g["ref_5000"])
    assert np.array_equal(cm.regions, np.union1d(g["ref_5000"][:, 0], g["ref_5000"][:, 1]))
    cm.decimate(25000)
    assert np.array_equal(cm.map, g["ref_25000_of_5000"])
    assert np.array_equal(cm.contacts(), do.contacts(g["ref_25000_of_5000"]))
    rng = np.random.default_rng(31)
    for n, span, shuffle in ((200000, 3000, True), (150001, 40, False), (1, 5, False), (70000, 1, True)):
        m1 = rng.integers(0, span, n) * 1000 + 500
        m2 = m1 + rng.integers(0, max(span // 10, 1), n) * 1000
        mp = np.stack([m1, m2, rng.integers(0, 40, n), rng.random(n) ** 2, np.minimum(rng.random(n) * 2, 1.0)], axis=1).astype(np.float64)
        if not shuffle:
            mp = mp[np.lexsort((mp[:, 1], mp[:, 0]))]
        cm = FithicContactMap.from_arrays(mp)
        cm.decimate(5000)
        assert np.array_equal(cm.map, do.decimate(mp, 5000)), (n, span)
    empty = FithicContactMap.from_arrays(np.zeros((0, 5)))
    empty.decimate(5000)
    assert empty.map.shape == (0, 5)
    with pytest.raises(ValueError):
        FithicContactMap.from_arrays(np.array([[1e12, 5.0, 1, 0.5, 0.5]])).decimate(5000)
    # the reader: a file written by the pass's own writer
    from blueberry_b200 import _io
    path = str(tmp_path / "x.significances.txt.gz")
    mp = g["map_in"]
    _io.write_significances(path, ["chr1"], None, mp[:, 0].astype(np.int64), None, mp[:, 1].astype(np.int64), mp[:, 2].astype(np.int64),
                            mp[:, 3], mp[:, 4])
    cm = FithicContactMap(path, resolution=1000)
    # pandas' default float parser (what datatypes.pyx:314 uses) is not round-trip exact (relative error up to ~1e-12 on
    # 17-digit decimals): the integer columns are exact, and the file itself is exact under float_precision='round_trip'
    assert np.array_equal(cm.map[:, :3], mp[:, :3])
    assert np.allclose(cm.map[:, 3:], mp[:, 3:], rtol=1e-11, atol=0.0)
    import pandas
    exact = pandas.read_csv(path, sep="\t", usecols=[1, 3, 4, 5, 6], engine='c', dtype='float64', float_precision='round_trip').values
    assert np.array_equal(exact, mp)
    assert cm.to_matrix('count', n_bins=600).sum() > 0


def test_contact_map_band_records_match_compiled_reference(tmp_path):
    """K8 (band ingest + normalize) against the golden matrices of the reference's ContactMap (compiled verbatim):
    the records scattered into a zero matrix ARE the reference's matrix, before and after normalize()."""
    from blueberry_b200.datatypes import ContactMap
    g = load_golden("contact_map")
    R = int(g["resolution"])
    cm = ContactMap((g["pos1"], g["pos2"], g["count"]), g["kr_norm"], g["kr_expected"], resolution=R)
    assert cm.n_bins == int(g["ref_n_bins"])
    assert np.array_equal(cm.to_dense(), g["ref_matrix"])
    assert np.array_equal(cm.regions, g["ref_regions"])
    cm.normalize()
    assert np.array_equal(cm.to_dense(), g["ref_normalized"])
    # from files, like the reference reads them
    raw, krp, kep = str(tmp_path / "c.RAWobserved"), str(tmp_path / "c.KRnorm"), str(tmp_path / "c.KRexpected")
    with open(raw, "w") as fh:
        for a, b, c in zip(g["pos1"], g["pos2"], g["count"]):
            fh.write("%r\t%r\t%r\n" % (float(a), float(b), float(c)))
    np.savetxt(krp, g["kr_norm"]); np.savetxt(kep, g["kr_expected"])
    cm2 = ContactMap(raw, krp, kep, resolution=R)
    cm2.normalize()
    assert np.allclose(cm2.to_dense(), g["ref_normalized"], rtol=1e-12, atol=0)      # savetxt's %.18e text round trip
    kr = g["kr_norm"].copy()
    kr[int(np.nanargmax(kr))] = 0.0
    bad = ContactMap((g["pos1"], g["pos2"], g["count"]), kr, g["kr_expected"], resolution=R)
    with pytest.raises(ZeroDivisionError):
        bad.normalize()
    with pytest.raises(IndexError):
        ContactMap((g["pos1"] + 10 ** 7, g["pos2"], g["count"]), g["kr_norm"], g["kr_expected"], resolution=R)
