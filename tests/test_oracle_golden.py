"""CPU: the oracle against the committed fixtures.  Hybrid fixtures were produced by the reference's own
src/hybrid_system.py; ALS / tower fixtures are oracle-minted (parity unpinned, see headers)."""
import json
import os

import numpy as np
import pytest

from oracle import als_oracle, c_oracle, hybrid_oracle, towers_oracle

G = os.path.join(os.path.dirname(__file__), "golden")


def hybrid_cases():
    return json.load(open(os.path.join(G, "hybrid_reference_cases.json")))["cases"]


@pytest.mark.parametrize("case", hybrid_cases(), ids=lambda c: c["name"])
def test_hybrid_oracle_matches_reference_fixture(case):
    als, tt = np.array(case["als"]), np.array(case["tt"])
    a_f1, t_f1 = case["als_f1_in"] or 0.0, case["tt_f1_in"] or 0.0
    if case["actual"] is not None:   # hybrid_system.py:104-105: F1 from the two score lists
        actual = {int(k): v for k, v in case["actual"].items()}
        a_f1 = hybrid_oracle.compute_f1_score(actual, dict(enumerate(als)))
        t_f1 = hybrid_oracle.compute_f1_score(actual, dict(enumerate(tt)))
        assert [a_f1, t_f1] == pytest.approx(case["f1_after"], abs=1e-12)
    blend = hybrid_oracle.adaptive_fusion_dense(als, tt, a_f1, t_f1)
    idx, sc = hybrid_oracle.topk_desc(blend, case["top_k"])
    assert list(idx) == case["out_items"]
    # reference blends an fp64 ALS column with an fp32 tower column: agree to fp32 resolution
    assert np.allclose(sc, case["out_scores"], rtol=0, atol=2e-7)


def test_f1_known_answers_of_the_reference():
    """compute_f1_score (src/als_model.py:171-177) returned these for the same inputs (SURVEY.md Appendix C):
    F1@2 of {1, 2, 9} against {1, 2, 3} is 0.8, and an empty set of actual ratings scores 0."""
    assert hybrid_oracle.compute_f1_score({1: 5, 2: 4, 3: 3}, {1: .9, 2: .8, 9: .7, 3: .1}, k=2) == pytest.approx(0.8)
    assert hybrid_oracle.compute_f1_score({}, {1: 1.0}) == 0


def test_minmax_semantics_match_sklearn():
    from sklearn.preprocessing import MinMaxScaler
    rng = np.random.default_rng(0)
    for x in (rng.normal(size=50), np.full(7, 3.0), np.array([2.0]), np.array([-1.0, 1.0])):
        ref = MinMaxScaler().fit_transform(x.reshape(-1, 1)).ravel()
        assert np.allclose(hybrid_oracle.minmax(x), ref, atol=1e-15)


def test_als_oracle_fixtures_and_restatements_agree():
    z = np.load(os.path.join(G, "als_oracle_cases.npz"))
    for imp in (0, 1):
        X, Y = als_oracle.als_fit(z["tiny_u"], z["tiny_i"], z["tiny_r"], 3, 3, 2, 3, 0.1, z["tiny_X0"],
                                  implicit=bool(imp), alpha=2.0)
        assert np.array_equal(X, z[f"tiny_imp{imp}_X"]) or np.allclose(X, z[f"tiny_imp{imp}_X"], atol=1e-6)
        assert np.allclose(Y, z[f"tiny_imp{imp}_Y"], atol=1e-6)
    u, i, r = z["mid_u"], z["mid_i"], z["mid_r"]
    X, Y = als_oracle.als_fit(u, i, r, 200, 150, 10, 10, 0.1, z["mid_X0"], half_step=c_oracle.als_half_step)
    assert np.allclose(X, z["mid_X"], atol=2e-5) and np.allclose(Y, z["mid_Y"], atol=2e-5)
    assert als_oracle.rmse(X, Y, u, i, r) == pytest.approx(float(z["mid_rmse"]), abs=1e-6)
    Xi, Yi = als_oracle.als_fit(u, i, z["mid_r_implicit"], 200, 150, 10, 5, 0.05, z["mid_X0"], implicit=True,
                                alpha=40.0, half_step=c_oracle.als_half_step)
    assert np.allclose(Xi, z["mid_Xi"], atol=2e-5) and np.allclose(Yi, z["mid_Yi"], atol=2e-5)


def test_als_half_step_satisfies_normal_equations():
    """Known-answer property: the solved row satisfies (sum y y^T + lambda n I) x = sum r y."""
    rng = np.random.default_rng(4)
    U, I, k, nnz, lam = 60, 40, 6, 500, 0.3
    u, i = rng.integers(0, U, nnz), rng.integers(0, I, nnz)
    r = rng.uniform(0.5, 5, nnz).astype(np.float32)
    X = als_oracle.init_factors(U, k, 0)
    rp, ci, v = als_oracle.coo_to_csr(i, u, r, I)
    Y = als_oracle.als_half_step_loops(rp, ci, v, X, lam)
    for j in range(I):
        lo, hi = rp[j], rp[j + 1]
        if hi == lo:
            assert not Y[j].any()
            continue
        Gm = X[ci[lo:hi]].astype(np.float64)
        A = Gm.T @ Gm + lam * (hi - lo) * np.eye(k)
        assert np.allclose(A @ Y[j], v[lo:hi].astype(np.float64) @ Gm, atol=1e-4)
    # explicit closed form on a 1-rating row: x = r y / (|y|^2 + lambda)
    rp1, ci1, v1 = np.array([0, 1]), np.array([3], np.int32), np.array([4.0], np.float32)
    y = X[3].astype(np.float64)
    x = als_oracle.als_half_step_loops(rp1, ci1, v1, X, lam)[0]
    assert np.allclose(x, 4.0 * y / (y @ y + lam), atol=1e-6)


def test_item_half_step_runs_first():
    """Initial item factors must not matter (Spark's loop starts with the item half-step)."""
    z = np.load(os.path.join(G, "als_oracle_cases.npz"))
    ir, ic, iv = als_oracle.coo_to_csr(z["tiny_i"], z["tiny_u"], z["tiny_r"], 3)
    Y1 = als_oracle.als_half_step(ir, ic, iv, z["tiny_X0"], 0.1)
    X, Y = als_oracle.als_fit(z["tiny_u"], z["tiny_i"], z["tiny_r"], 3, 3, 2, 1, 0.1, z["tiny_X0"])
    ur, uc, uv = als_oracle.coo_to_csr(z["tiny_u"], z["tiny_i"], z["tiny_r"], 3)
    assert np.array_equal(X, als_oracle.als_half_step(ur, uc, uv, Y1, 0.1))


def test_tower_oracle_fixture_and_layer_norm():
    z = np.load(os.path.join(G, "tower_oracle_case.npz"))
    w = {k[2:]: z[k] for k in z.files if k.startswith("w_")}
    num = towers_oracle.scale_numeric(z["raw"], z["scale"], z["offset"])
    iv = towers_oracle.item_tower(w, z["ids"], z["manu"], z["cat"], num)
    assert np.allclose(iv, z["item_vecs"], atol=1e-6)
    assert np.allclose(towers_oracle.user_tower(w, np.arange(60)), z["user_vecs"], atol=1e-6)
    import torch
    x = torch.randn(5, 50, dtype=torch.float64)
    g, b = torch.rand(50, dtype=torch.float64), torch.rand(50, dtype=torch.float64)
    ref = torch.nn.functional.layer_norm(x, (50,), g, b, 1e-3).numpy()
    got = towers_oracle.layer_norm(x.numpy().astype(np.float32), g.numpy().astype(np.float32), b.numpy().astype(np.float32))
    assert np.allclose(got, ref, atol=1e-5)


def test_c_hybrid_topk_matches_numpy_oracle():
    rng = np.random.default_rng(11)
    Ua, Ia = rng.normal(size=(9, 12)).astype(np.float32), rng.normal(size=(70, 12)).astype(np.float32)
    Ut, It = rng.normal(size=(9, 5)).astype(np.float32), rng.normal(size=(70, 5)).astype(np.float32)
    i1, s1 = hybrid_oracle.hybrid_topk_dense(Ua, Ia, Ut, It, 0.8, 0.2, 10)
    i2, s2 = c_oracle.hybrid_topk(Ua, Ia, Ut, It, 0.8, 0.2, 10)
    assert np.allclose(s1, s2, atol=1e-5)
    assert (i1 == i2).mean() > 0.95
