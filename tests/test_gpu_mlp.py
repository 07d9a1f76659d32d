"""One-hidden-layer ReLU networks (scikit-learn MLPClassifier / MLPRegressor) on the GPU against the CPU oracle given the
scikit-learn callable itself.  Tolerance: 1e-5 relative to the largest |phi| of the instance; additivity to 1e-8.  The test
networks are trained briefly from scikit-learn's initialisation, so their weights are moderate and no score saturates the
oracle's float64 1 - p."""
import warnings

import numpy as np
import pytest

from conftest import make_problem, rel_err

pytestmark = pytest.mark.gpu
sklearn = pytest.importorskip("sklearn")
from sklearn.exceptions import ConvergenceWarning  # noqa: E402
from sklearn.neural_network import MLPClassifier, MLPRegressor  # noqa: E402

TOL = 1e-5
KERNELS = ["simt", "auto"]


def _fit(est, X, y):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", ConvergenceWarning)
        return est.fit(X, y)


def mlp_problem(kind="binary", seed=0, n=12, N=16, widths=(1, 1, 3, 2, 1, 2), H=24, weights=False, constant_groups=(),
                n_out=2):
    """make_problem's data and groups with a fitted network in place of the linear classifier."""
    prob = make_problem(seed=seed, n=n, N=N, widths=widths, weights=weights, constant_groups=constant_groups)
    rng = np.random.default_rng(seed + 100)
    D = prob["X"].shape[1]
    Xt = rng.standard_normal((400, D))
    u = rng.standard_normal((D, 3))
    s = np.tanh(Xt @ u) + 0.3 * rng.standard_normal((400, 3))
    if kind == "binary":
        model = _fit(MLPClassifier(hidden_layer_sizes=(H,), max_iter=40, random_state=seed), Xt, (s[:, 0] > 0).astype(int))
        prob["predict"] = model.predict_proba
    elif kind == "softmax":
        model = _fit(MLPClassifier(hidden_layer_sizes=(H,), max_iter=40, random_state=seed), Xt, np.argmax(s, axis=1))
        prob["predict"] = model.predict_proba
    else:
        y = s[:, 0] if n_out == 1 else s[:, :n_out]
        model = _fit(MLPRegressor(hidden_layer_sizes=(H,), max_iter=40, random_state=seed), Xt, y)
        prob["predict"] = model.predict
    prob["model"] = model
    return prob


def _dd(mod, prob):
    args = (prob["groups"],) + ((prob["weights"],) if prob["weights"] is not None else ())
    return mod.DenseData(prob["bg"], prob["group_names"], *args)


def _oracle(prob, link):
    from oracle import shap_kernel_oracle as o
    return o.KernelExplainerOracle(prob["predict"], _dd(o, prob), link=link, record_plans=True)


def _engine(prob, link, **kw):
    from distributedkernelshap_b200 import data
    from distributedkernelshap_b200.engine import GpuKernelExplainer
    return GpuKernelExplainer(prob["predict"], _dd(data, prob), link=link, **kw)


def _as_list(x):
    return x if isinstance(x, list) else [x]


def _compare(got, want, tol=TOL):
    got, want = _as_list(got), _as_list(want)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.shape == w.shape
        assert rel_err(g, w) < tol, rel_err(g, w)


def _oracle_fed(orc, X, plan_of, nsamples, l1_reg=False):
    """Per-instance oracle run on the given plans; plan_of(i) -> (Z dense, w).  Returns [C][n, G] (or [n, G])."""
    rows = [orc.explain(X[i:i + 1], plan=plan_of(i), nsamples=nsamples, l1_reg=l1_reg) for i in range(X.shape[0])]
    phi = np.stack(rows)                                  # [n, G, C] or [n, G]
    return [phi[:, :, c] for c in range(phi.shape[2])] if phi.ndim == 3 else phi


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("link", ["logit", "identity"])
def test_full_enumeration_matches_oracle(link, kernel):
    prob = mlp_problem(seed=1, n=16, N=12)
    orc, eng = _oracle(prob, link), _engine(prob, link, kernel=kernel)
    want = orc.shap_values(prob["X"], nsamples=10000, l1_reg=False)
    got = eng.shap_values(prob["X"], nsamples=10000, l1_reg=False)
    _compare(got, want)
    np.testing.assert_allclose(eng.expected_value, orc.expected_value, rtol=1e-12)
    fx = prob["predict"](prob["X"])
    for c in range(2):
        total = (np.log(fx[:, c] / (1 - fx[:, c])) if link == "logit" else fx[:, c]) - eng.expected_value[c]
        np.testing.assert_allclose(got[c].sum(axis=1), total, rtol=1e-8, atol=1e-8)
    np.testing.assert_array_equal(got[0], -got[1])


@pytest.mark.parametrize("nsamples", [300, 2048])
def test_shared_plan_matches_oracle_and_the_kernels_agree(nsamples):
    """M = 12 groups that all vary: 'auto' takes the shared-plan MLP kernel, 'simt' the general one."""
    from distributedkernelshap_b200.plan import build_plan
    prob = mlp_problem(seed=4, n=10, N=25, widths=(1,) * 6 + (3, 2, 2, 1, 5, 1), H=40)
    orc = _oracle(prob, "logit")
    got = {}
    for kernel in KERNELS:
        np.random.seed(11)
        eng = _engine(prob, "logit", kernel=kernel)
        got[kernel] = eng.shap_values(prob["X"], nsamples=nsamples, l1_reg=False)
    M, _ = eng.varying(prob["X"])
    assert np.all(M == 12)
    np.random.seed(11)
    plan = build_plan(12, nsamples)
    want = _oracle_fed(orc, prob["X"], lambda i: (plan.dense(), plan.weights), nsamples)
    for kernel in KERNELS:
        _compare(got[kernel], want)
    assert rel_err(got["auto"][1], got["simt"][1]) < 1e-6


@pytest.mark.parametrize("kernel", KERNELS)
def test_caller_supplied_per_instance_plans(kernel):
    prob = mlp_problem(seed=3, n=12, N=16, widths=(1, 1, 1, 1, 3, 2, 1, 2, 1, 4, 1, 1))
    orc, eng = _oracle(prob, "logit"), _engine(prob, "logit", kernel=kernel)
    np.random.seed(0)
    want = orc.shap_values(prob["X"], nsamples=500, l1_reg=False)
    plans = [(Z, w) for (_, Z, w) in orc.plans]
    got = eng.shap_values(prob["X"], nsamples=500, l1_reg=False, plans=plans)
    _compare(got, want)


def test_device_drawn_per_instance_plans():
    prob = mlp_problem(seed=6, n=10, N=16, widths=(1, 1, 1, 1, 3, 2, 1, 2, 1, 4, 1, 1))
    orc = _oracle(prob, "logit")
    eng = _engine(prob, "logit", seed=3, plan_mode="per_instance")
    got = eng.shap_values(prob["X"], nsamples=600, l1_reg=False)
    zb, w = eng.instance_plans()
    M, _ = eng.varying(prob["X"])
    from distributedkernelshap_b200.plan import resolve_nsamples

    def plan_of(i):
        S = resolve_nsamples(int(M[i]), 600)[0]
        k = np.arange(int(M[i]), dtype=np.uint64)
        return ((zb[i, :S, None] >> k[None, :]) & np.uint64(1)).astype(np.uint8), w[i, :S]
    _compare(got, _oracle_fed(orc, prob["X"], plan_of, 600))


@pytest.mark.parametrize("kernel", KERNELS)
def test_weighted_background_and_constant_groups(kernel):
    prob = mlp_problem(seed=5, n=10, N=9, widths=(1, 2, 1, 3, 1, 1), weights=True, constant_groups=(1, 3))
    orc, eng = _oracle(prob, "logit"), _engine(prob, "logit", kernel=kernel)
    want = orc.shap_values(prob["X"], nsamples=100, l1_reg=False)
    got = eng.shap_values(prob["X"], nsamples=100, l1_reg=False)
    _compare(got, want)
    assert np.all(got[1][:, 1] == 0) and np.all(got[1][:, 3] == 0)      # non-varying groups get exactly 0


@pytest.mark.parametrize("kernel", KERNELS)
def test_degenerate_M(kernel):
    prob = mlp_problem(seed=15, n=6, N=8, widths=(1, 2, 1, 3, 1))
    X = prob["X"]
    prob["bg"][:] = prob["bg"][0]                        # constant background: a group varies iff x differs from it
    X[1] = prob["bg"][0]                                 # M = 0
    X[2] = prob["bg"][0]; X[2, 0] += 1.0                 # M = 1
    orc, eng = _oracle(prob, "logit"), _engine(prob, "logit", kernel=kernel)
    want = orc.shap_values(X, nsamples=100, l1_reg=False)
    got = eng.shap_values(X, nsamples=100, l1_reg=False)
    _compare(got, want)
    M, _ = eng.varying(X)
    assert M[1] == 0 and M[2] == 1
    assert np.all(got[1][1] == 0)


@pytest.mark.parametrize("N", [1, 200])
def test_background_sizes(N):
    from distributedkernelshap_b200.plan import build_plan
    prob = mlp_problem(seed=7, n=6, N=N, widths=(1,) * 9, H=32)
    orc = _oracle(prob, "logit")
    np.random.seed(2)
    eng = _engine(prob, "logit")
    got = eng.shap_values(prob["X"], nsamples=200, l1_reg=False)
    M, _ = eng.varying(prob["X"])
    assert np.all(M == 9)
    np.random.seed(2)
    plan = build_plan(9, 200)
    _compare(got, _oracle_fed(orc, prob["X"], lambda i: (plan.dense(), plan.weights), 200))


@pytest.mark.parametrize("kernel", KERNELS)
def test_softmax_head(kernel):
    prob = mlp_problem(kind="softmax", seed=8, n=8, N=14)
    orc, eng = _oracle(prob, "logit"), _engine(prob, "logit", kernel=kernel)
    want = orc.shap_values(prob["X"], nsamples=10000, l1_reg=False)
    got = eng.shap_values(prob["X"], nsamples=10000, l1_reg=False)
    assert len(got) == 3
    _compare(got, want)
    np.testing.assert_allclose(eng.expected_value, orc.expected_value, rtol=1e-12)


@pytest.mark.parametrize("n_out", [1, 2])
@pytest.mark.parametrize("kernel", KERNELS)
def test_regressor(n_out, kernel):
    prob = mlp_problem(kind="regressor", seed=9, n=8, N=14, n_out=n_out)
    orc, eng = _oracle(prob, "identity"), _engine(prob, "identity", kernel=kernel)
    want = orc.shap_values(prob["X"], nsamples=10000, l1_reg=False)
    got = eng.shap_values(prob["X"], nsamples=10000, l1_reg=False)
    assert eng.vector_out == (n_out == 2)
    _compare(got, want)
    np.testing.assert_allclose(eng.expected_value, orc.expected_value, rtol=1e-12)


@pytest.mark.parametrize("l1_reg", ["auto", "aic", "num_features(5)"])
def test_l1_selection_on_the_shared_plan_kernel(l1_reg):
    from distributedkernelshap_b200.plan import build_plan
    prob = mlp_problem(seed=10, n=6, N=20, widths=(1,) * 16, H=32)
    orc = _oracle(prob, "logit")
    np.random.seed(4)
    eng = _engine(prob, "logit", kernel="shared")
    got = eng.shap_values(prob["X"], nsamples=300, l1_reg=l1_reg)
    np.random.seed(4)
    plan = build_plan(16, 300)
    want = _oracle_fed(orc, prob["X"], lambda i: (plan.dense(), plan.weights), 300, l1_reg=l1_reg)
    np.testing.assert_array_equal(got[1] != 0, want[1] != 0)
    if l1_reg.startswith("num_features"):
        assert np.all((want[1] != 0).sum(axis=1) <= 5)
    _compare(got, want)


def test_kernelshap_end_to_end_on_adult_shaped_data():
    from distributedkernelshap_b200.datasets import adult_like
    from distributedkernelshap_b200.explainers.kernel_shap import KernelShap
    from oracle.shap_kernel_oracle import DenseData, KernelExplainerOracle
    d = adult_like(n_explain=48)
    rng = np.random.default_rng(0)
    Xt = np.concatenate([d["background"], d["X_explain"]])
    y = (Xt[:, :4] @ rng.standard_normal(4) + Xt[:, 4:] @ rng.normal(0, 0.5, Xt.shape[1] - 4) > 0).astype(int)
    mlp = _fit(MLPClassifier(hidden_layer_sizes=(100,), max_iter=30, random_state=0), Xt, y)
    ks = KernelShap(mlp.predict_proba, link="logit", feature_names=d["group_names"], seed=0)
    ks.fit(d["background"], groups=d["groups"], group_names=d["group_names"])
    exp = ks.explain(d["X_explain"], silent=True, nsamples=2048, l1_reg=False)
    p = mlp.predict_proba(d["X_explain"])
    np.testing.assert_allclose(exp.raw["raw_prediction"], np.log(p / (1 - p)), rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(exp.shap_values[1].sum(1) + exp.expected_value[1], exp.raw["raw_prediction"][:, 1],
                               rtol=1e-8, atol=1e-8)
    M, _ = ks._explainer.varying(d["X_explain"])
    orc = KernelExplainerOracle(mlp.predict_proba, DenseData(d["background"], d["group_names"], d["groups"]), link="logit")
    worst = 0.0
    for i in range(0, 48, 6):
        plan = ks._explainer.shared_plan(int(M[i]), 2048)
        phi = orc.explain(d["X_explain"][i:i + 1], plan=(plan.dense(), plan.weights), nsamples=2048, l1_reg=False)
        worst = max(worst, rel_err(exp.shap_values[1][i], phi[:, 1]))
    assert worst < TOL, worst


def test_device_resident_calls_replay_bit_identically():
    import torch
    prob = mlp_problem(seed=11, n=40, N=14, widths=(1, 2, 1, 1, 3, 1, 1, 2))
    eng = _engine(prob, "logit")
    want = eng.shap_values(prob["X"], nsamples=120, l1_reg=False)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        eng.set_stream(stream.cuda_stream)
        X_dev = torch.from_numpy(prob["X"]).cuda()
        phi = torch.zeros((2, 40, 8), dtype=torch.float64, device="cuda")
        for _ in range(4):
            eng.explain_device(X_dev.data_ptr(), 40, phi.data_ptr(), nsamples=120)
        eng.check_status()
        assert eng.graph_launches() >= 2
        np.testing.assert_array_equal(phi[1].cpu().numpy(), want[1])
        np.testing.assert_array_equal(phi[0].cpu().numpy(), want[0])


def test_device_side_refusals():
    from distributedkernelshap_b200 import _cabi
    from distributedkernelshap_b200.engine import GpuKernelExplainer
    prob = mlp_problem(seed=12, n=4, N=10)
    with pytest.raises(NotImplementedError, match="tcgen05"):
        _engine(prob, "logit", kernel="tcgen05")
    eng = _engine(prob, "logit")
    with pytest.raises(NotImplementedError, match="tcgen05"):
        eng.set_kernel("tcgen05")
    wide = mlp_problem(seed=13, n=2, N=6, widths=(1,) * 65, H=8)
    with pytest.raises(_cabi.DksError, match="64 groups"):
        _engine(wide, "logit")
    model = prob["model"]

    class Liar:
        coefs_ = model.coefs_
        intercepts_ = model.intercepts_
        activation = "relu"
        out_activation_ = "logistic"
        classes_ = model.classes_

        def predict_proba(self, X):
            return model.predict_proba(X) ** 2
    with pytest.raises(ValueError, match="network"):
        GpuKernelExplainer(Liar().predict_proba, prob["bg"])
