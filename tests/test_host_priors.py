"""Host-side samplers, companion priors and stellar relations against fixtures produced by the
reference's own priors.py / funcs.py (oracle/gen_golden.py).  Bit-exact: identical draws are the
premise of every downstream parity check."""
import numpy as np
import pytest

from triceratops_b200 import funcs, priors


@pytest.fixture(scope="module")
def g(golden):
    return golden("samplers.npz")


@pytest.mark.parametrize("M", [1.3, 1.0, 0.811, 0.3, 0.25, 0.08])
def test_mass_ratio_samplers(g, M):
    assert np.array_equal(priors.sample_q(g["x"].copy(), M), g["q/%g" % M])
    assert np.array_equal(priors.sample_q_companion(g["x"].copy(), M), g["qc/%g" % M])


def test_planet_radius_inclination_periastron(g):
    assert np.array_equal(priors.sample_rp(g["x"].copy(), g["Ms"], False), g["rp/mixed"])
    assert np.array_equal(priors.sample_rp(g["x"].copy(), g["Ms"], True), g["rp/flat"])
    assert np.array_equal(priors.sample_inc(g["x"].copy()), g["inc"])
    assert np.array_equal(priors.sample_w(g["x"].copy()), g["w"])


@pytest.mark.parametrize("tag,planet,P", [("planet", True, 3.0), ("eb_short", False, 3.0),
                                          ("eb_long", False, 20.0)])
def test_eccentricities_consume_the_global_rng_like_the_reference(g, tag, planet, P):
    np.random.seed(6)
    assert np.array_equal(priors.sample_ecc(g["x"], planet, P), g["ecc/" + tag])


def test_stellar_and_flux_relations(g):
    n = g["m"].size
    rad, teff = funcs.stellar_relations(g["m"], np.full(n, 0.9), np.full(n, 5000.))
    assert np.array_equal(rad, g["rad"]) and np.array_equal(teff, g["teff"])
    for filt in ("TESS", "J", "H", "K"):
        assert np.array_equal(funcs.flux_relation(g["m"], filt), g["flux/" + filt])
    assert np.array_equal(funcs.flux_relation(g["m"], "Vis"), g["flux/TESS"])


def test_companion_priors(g, contrast_file):
    sep, con = funcs.file_to_contrast_curve(contrast_file)
    with np.errstate(divide="ignore"):
        for M in (1.3, 0.811):
            assert np.array_equal(priors.lnprior_bound_TP(M, 8.16, g["dm"], sep, con),
                                  g["bound_TP/%g" % M])
            assert np.array_equal(priors.lnprior_bound_EB(M, 8.16, g["dm"], sep, con),
                                  g["bound_EB/%g" % M])
            assert np.array_equal(
                priors.lnprior_bound_TP(M, np.nan, g["dm"], np.array([2.2]), np.array([1.0])),
                g["bound_TP_nocc/%g" % M])
        assert np.array_equal(priors.lnprior_background(1234, g["dm"], sep, con), g["background"])


def test_background_prior_is_natural_log(contrast_file):
    """Known answer of the reference's tests/test_background_prior_log_base.py:32-56."""
    sep, con = funcs.file_to_contrast_curve(contrast_file)
    dm = np.array([0.5, 2.0, 5.0])
    want = np.log((500 / 0.1) * (1 / 3600) ** 2 * np.interp(dm, con, sep) ** 2)
    np.testing.assert_allclose(priors.lnprior_background(500, dm, sep, con), want, rtol=0, atol=0)


def test_trilegal_reader(g, trilegal_file):
    got = funcs.trilegal_results(trilegal_file, 10.7307)
    for k, v in zip(("Tmags", "Masses", "loggs", "Teffs", "Zs", "Jmags", "Hmags", "Kmags"), got):
        assert np.array_equal(v, g["trilegal/" + k])


def test_renorm_flux():
    f, e = funcs.renorm_flux(np.array([1.0, 0.99]), 0.001, 0.5)
    np.testing.assert_allclose(f, [1.0, 0.98])
    assert e == 0.002


def test_trilegal_table_is_cached_per_file_version(tmp_path, trilegal_file):
    """The saved TRILEGAL table is parsed once per (path, mtime, size); a rewritten file is read
    again."""
    import os
    import shutil
    from triceratops_b200 import funcs
    path = str(tmp_path / "tri.csv")
    shutil.copy(trilegal_file, path)
    a = funcs.trilegal_results(path, 10.0)
    assert funcs._read_trilegal(path) is funcs._read_trilegal(path)
    b = funcs.trilegal_results(path, 10.0)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    lines = open(path).read().splitlines()
    with open(path, "w") as fh:                 # drop ten stars, keep header and trailer rows
        fh.write("\n".join(lines[:1] + lines[11:]) + "\n")
    st = os.stat(path)
    os.utime(path, ns=(st.st_atime_ns, st.st_mtime_ns + 1_000_000))
    c = funcs.trilegal_results(path, -99.0)
    full = funcs.trilegal_results(trilegal_file, -99.0)
    assert c[0].size == full[0].size - 10


@pytest.mark.parametrize("mission", ["TESS", "Kepler"])
def test_dense_ldc_table_holds_the_rounded_lookup_of_every_node(mission):
    """The device sampler's (Teff, logg) table at each tabulated Z: every grid node's entry is
    what at_Z_rounded returns for that node, and there is no other entry."""
    from triceratops_b200._ldc import grid_for
    grid = grid_for(mission)
    for Z in np.unique(grid.Zs):
        at_Z = grid.Zs == Z
        T, logg = grid.Teffs[at_Z].astype(float), grid.loggs[at_Z]
        u1, u2 = grid.at_Z_rounded(Z, T, logg, 10000)
        tab1, tab2 = grid.dense_table(Z)
        it, ig = ((T - 3500) // 250).astype(int), np.round((logg - 3.5) / 0.5).astype(int)
        assert np.array_equal(tab1[it, ig], u1) and np.array_equal(tab2[it, ig], u2)
        assert np.isfinite(tab1).sum() == np.isfinite(tab2).sum() == at_Z.sum()
