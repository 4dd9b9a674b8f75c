"""The oracle against the reference on seeded random problems other than those of test_oracle_golden.py: the reference's
outputs, and the exact inputs it was given, are frozen in tests/golden/oracle_vs_ref.npz
(tests/golden/make_golden_live.py executes the reference through oracle/ref_shim.py to produce them)."""
import numpy as np
import pytest

from oracle import gp_oracle as O
from tests.helpers import load


@pytest.fixture(scope="module")
def g():
    return load("oracle_vs_ref")


@pytest.mark.parametrize("kind", ["SE", "ARDSE", "Matern32", "Matern52"])
def test_kernels_and_logprob(g, kind):
    comp, cand, vals, ls = (g["k_%s_%s" % (kind, k)] for k in ("comp", "cand", "vals", "ls"))
    np.testing.assert_allclose(O.kernel(kind, ls, comp), g["k_%s_self" % kind], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(O.kernel(kind, ls, comp, cand), g["k_%s_cross" % kind], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(O.gp_logprob(kind, 0.1, 2e-3, 1.3, ls, comp, vals), g["k_%s_logprob" % kind], rtol=1e-11)


def test_compute_ei_with_and_without_pending(g):
    comp, cand, vals = g["ei_comp"], g["ei_cand"], g["ei_vals"]
    h = (float(g["ei_mean"]), float(g["ei_noise"]), float(g["ei_amp2"]), g["ei_ls"])
    np.testing.assert_allclose(O.compute_ei("Matern52", h, comp, np.zeros((0, comp.shape[1])), cand, vals),
                               g["ei_nopend"], rtol=1e-9, atol=1e-14)
    np.testing.assert_allclose(O.compute_ei("Matern52", h, comp, g["ei_pend"], cand, vals, g["ei_normals"]),
                               g["ei_withpend"], rtol=1e-9, atol=1e-14)


def test_sobol_and_optimize_hypers(g):
    from oracle import sobol_oracle as SO
    assert np.array_equal(SO.i4_sobol_generate(6, 50, 2), g["sobol_6x50_skip2"])
    m, noise, amp2, ls = O.gp_optimize_hypers("Matern52", g["mll_comp"], g["mll_vals"])
    np.testing.assert_allclose([m, noise, amp2], [g["mll_mean"], g["mll_noise"], g["mll_amp2"]], rtol=1e-6)
    np.testing.assert_allclose(ls, g["mll_ls"], rtol=1e-6)
