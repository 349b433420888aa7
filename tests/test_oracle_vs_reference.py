"""The oracle against the original blueberry sources executed live.  They are not part of this repository: point
BLUEBERRY_REFERENCE at a checkout to run these; without one they skip.  tests/test_oracle_golden.py checks the same
functions against outputs of the original stored under tests/golden/."""
import numpy as np
import pytest

from oracle import ref_loader

pytestmark = pytest.mark.skipif(not ref_loader.reference_available(), reason="no checkout of the original blueberry sources (BLUEBERRY_REFERENCE)")


def test_live_reference_small_pass():
    from blueberry_b200 import synth
    from oracle import run_reference as rr, fithic_oracle as fo
    R, bins = 20000, [150, 90]
    bias = synth.make_bias(bins, 3)
    fc, fm = synth.make_fragments(bins, R)
    c = synth.make_contacts(bins, R, 1_000_000, 40.0, 9, bias)
    bc = np.concatenate([np.full(b, i) for i, b in enumerate(bins)])
    ref = rr.run_reference_pass(fc, fm, c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], R,
                                n_bins=50, max_dist=1_000_000, bias=(bc, fm, np.concatenate(bias)))
    bd, _ = fo.read_bias_arrays(bc, fm, np.concatenate(bias))
    o = fo.fithic_arrays(fc, fm, c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], R, 50,
                         ref["min_dist"], ref["max_dist"], bias=bd)
    assert np.array_equal(o.frag.possible, ref["possible"])
    assert np.array_equal(o.contacts.observed, ref["observed"])
    assert np.array_equal(np.array(o.y), ref["y"]) and np.array_equal(np.array(o.x), ref["x"])
    assert np.array_equal(o.spline_y, ref["spline_y"])
    assert np.array_equal(o.p[o.keep], ref["out"]["p"])


def test_live_reference_cython_helpers():
    from oracle import fithic_oracle as fo
    cy = ref_loader.load_reference_cython()
    rng = np.random.default_rng(0)
    p = np.sort(rng.random(500))
    assert np.array_equal(np.asarray(cy.benjamini_hochberg(p, 777)), fo.benjamini_hochberg_sorted(p, 777))
    reg = np.sort(rng.choice(10**6, 800, replace=False)).astype(np.float64) * 37
    assert cy.count_band_regions(reg) == fo.count_band_regions(reg)


def test_live_reference_decimate():
    """The restatement of FithicContactMap.decimate against the reference's own method body, executed here."""
    import numpy as np
    from oracle import datatypes_oracle as do, run_reference
    rng = np.random.default_rng(23)
    n = 3000
    m1 = rng.integers(0, 300, n) * 1000 + 500
    m2 = m1 + rng.integers(0, 40, n) * 1000
    mp = np.stack([m1, m2, rng.integers(0, 30, n), rng.random(n) ** 3, rng.random(n)], axis=1).astype(np.float64)
    for r in (2000, 5000, 25000):
        assert np.array_equal(run_reference.run_reference_decimate(mp, r), do.decimate(mp, r))


def test_live_reference_contact_map():
    """The dense ContactMap restatement against the reference class itself (compiled verbatim into oracle/_ref)."""
    import numpy as np
    from oracle import datatypes_oracle as do, run_reference
    rng = np.random.default_rng(41)
    nb, R = 30, 10000
    kr = rng.random(nb) + 0.5
    kr[[2, 11]] = np.nan
    ke = rng.random(nb) * 20 + 1
    b1 = rng.integers(0, nb + 1, 200)
    b2 = np.minimum(b1 + rng.integers(0, 8, 200), nb)
    cnt = rng.integers(1, 90, 200).astype(np.float64)
    before, after, regions, n_bins = run_reference.run_reference_contact_map(b1 * R, b2 * R, cnt, kr, ke, R)
    m, reg = do.contact_map_dense(b1 * R, b2 * R, cnt, n_bins, R)
    assert n_bins == nb and np.array_equal(m, before) and np.array_equal(reg, regions)
    assert np.array_equal(do.normalize_dense(m, kr, ke, n_bins), after)


def test_live_reference_extract_contacts():
    """utils.extract_contacts executed from the reference's own source (two print statements edited) on a file read by the
    reference's own FithicContactMap, against the oracle's restatement on the table as that class read it."""
    from oracle import run_reference as rr, datatypes_oracle as do
    rng = np.random.default_rng(77)
    n = 1500
    m1 = rng.integers(0, 2500, n) * 5000 + 2500
    m2 = m1 + rng.integers(0, 2300, n) * 5000
    mp = np.stack([m1, m2, rng.integers(1, 40, n), rng.random(n) ** 5, np.full(n, -1.0)], axis=1).astype(np.float64)
    rr.write_reference_significances(mp, 5, 5000)
    held = rr.reference_map_as_read(5, 5000)
    got, band = rr.run_reference_extract_contacts(5, 5000, alpha=0.1, n_regions=True)
    assert np.array_equal(do.extract_contacts(held, 5, 0.1), got)
    assert do.count_band_regions(do.regions(held)) == band
    assert np.array_equal(do.extract_contacts(held, 5), rr.run_reference_extract_contacts(5, 5000))

