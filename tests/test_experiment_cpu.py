"""Host-side caller of the imputation path (rpsmf_b200/experiment.py) on the CPU: the random stream, the mask
generator and the result record must reproduce the reference's published run (PM25, 30 %, seed 123, repeat 0:
ExperimentImpute/output/LondonAir_PM25_30_{rPSMF,PSMF}.json).  The fit itself is injected: here the oracle."""

import numpy as np
import pytest

from conftest import load_golden
from oracle import psmf_oracle as po
from rpsmf_b200 import experiment as ex


def _oracle_fit(robust):
    def rpsmf(Y, C, X, d, n, r, M, Mmiss, V, Q0, R0, P, lambda0, sig, Iter, YorigInt, Einit):
        Ep, Ef, ib, *_ = po.impute_fit(Y, C, X, M, Mmiss, V, Q0, float(R0[0, 0]), P, lambda0, float(sig), Iter, YorigInt, Einit, True)
        return Ep, Ef, np.zeros((1, Iter + 1)), ib

    def psmf(Y, C, X, d, n, r, M, Mmiss, lam, V, Q, R, P, sig, Iter, YorgInt, Einit):
        Ep, Ef, ib, *_ = po.impute_fit(Y, C, X, M, Mmiss, V, Q, float(R[0, 0]), P, 1.8, float(sig), Iter, YorgInt, Einit, False)
        return Ep, Ef, np.zeros((1, Iter + 1)), ib

    return rpsmf if robust else psmf


@pytest.mark.parametrize("method", ["rPSMF", "PSMF"])
def test_published_run_is_reproduced(method):
    g = load_golden("impute_pm25_30")
    out = ex.run_impute_experiment(g["Yorig"], method, int(g["pct"]), seed=123, repeats=1, fit=_oracle_fit(method == "rPSMF"))
    hy, hc, hx = [str(h) for h in g["rep0_hashes"]]
    assert out["hashes"] == dict(Y=[hy], C=[hc], X=[hx])           # inputs regenerated bit for bit
    pub = g["rep0_%s_published" % method]                           # error_predict, error_full, inside_sig
    assert abs(out["results"]["error_predict"][0] - pub[0]) / pub[0] < 1e-10
    assert abs(out["results"]["error_full"][0] - pub[1]) / pub[1] < 1e-10
    assert abs(out["results"]["inside_sig"][0] - pub[2]) < 1e-12
    assert out["method"] == method and out["seed"] == 123 and out["missing_percentage"] == 30
    assert 0.30 <= out["missing_ratio"] < 0.32
    assert ("lambda0" in out["parameters"]) == (method == "rPSMF")


def test_prepare_missing_mask_and_stream():
    g = load_golden("impute_pm25_30")
    np.random.seed(123)
    Ymiss = np.copy(g["Yorig"])
    ratio, Mmiss = ex.prepare_missing(Ymiss, 0.30)
    assert np.array_equal(Mmiss, g["rep0_Mmiss"])
    assert np.array_equal(np.isnan(Ymiss), np.isnan(g["Yorig"]) | (Mmiss == 1))
    d, r = g["rep0_C0"].shape
    assert np.array_equal(np.random.rand(d, r), g["rep0_C0"])       # the stream continues exactly where the reference's does
    assert np.array_equal(np.random.rand(r, g["Yorig"].shape[1]), g["rep0_X0"])
    # segments never wrap and never touch column 0
    assert Mmiss[:, 0].sum() == 0


def test_argument_checks():
    with pytest.raises(ValueError):
        ex.run_impute_experiment(np.zeros((3, 50)), "BPMF", 30, seed=1, fit=lambda *a: None)
    with pytest.raises(TypeError):
        ex.run_impute_experiment(np.zeros((3, 50)), "PSMF", 30, seed=1, fit=lambda *a: None, rank=4)


def test_published_pinning_summary():
    """tests/golden/pin_published.py replayed all 18 published result files whose input CSVs ship with the
    reference (3 datasets x 3 percentages x 2 methods): inputs of all 100 repeats by hash, results of the first
    repeats through the oracle.  The summary it wrote is committed; one file (PM2.5, 20 %, PSMF) is replayed here
    from the stored data set (LondonAir_PM25.csv, kept in impute_pm25_30.npz) against its stored published results."""
    import json
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    s = json.load(open(os.path.join(here, "golden", "published_pinning.json")))
    assert len(s["files"]) == 18 and s["all_hashes_match"]
    assert all(f["repeats_hashed"] == 100 and f["repeats_fitted"] >= 2 for f in s["files"])
    # end-of-fit scalars of the d x d reference against the O(d r^2) oracle: 17 files <= 1.3e-11, sp500 40 % rPSMF 1.25e-9
    assert s["max_rel_err_error_predict"] < 2e-9 and s["max_rel_err_error_full"] < 2e-9
    assert s["max_abs_err_inside_sig"] == 0.0
    pub = json.load(open(os.path.join(here, "golden", "published_results.json")))["files"]["LondonAir_PM25_20_PSMF"]
    Yorig = load_golden("impute_pm25_30")["Yorig"]
    out = ex.run_impute_experiment(Yorig, "PSMF", 20, seed=pub["seed"], repeats=1, fit=_oracle_fit(False))
    assert out["hashes"]["Y"][0] == pub["hashes"]["Y"][0]
    assert abs(out["results"]["error_full"][0] - pub["results"]["error_full"][0]) / pub["results"]["error_full"][0] < 1e-9
