"""One-hidden-layer ReLU networks on the host side: extraction from fitted scikit-learn MLPs, the NumPy forward of the
spec, refusals and spec validation.  No GPU here."""
import warnings

import numpy as np
import pytest

from distributedkernelshap_b200.predictors import (LinearModelSpec, LinearSoftmaxClassifier, MLPModelSpec,
                                                   extract_model_spec)

sklearn = pytest.importorskip("sklearn")
from sklearn.exceptions import ConvergenceWarning  # noqa: E402
from sklearn.neural_network import MLPClassifier, MLPRegressor  # noqa: E402


def _data(n=120, D=6, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, D))
    return rng, X


def _fit(est, X, y):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", ConvergenceWarning)
        return est.fit(X, y)


def test_binary_classifier_extraction_matches_sklearn():
    rng, X = _data()
    y = (X[:, 0] + X[:, 1] * X[:, 2] > 0).astype(int)
    clf = _fit(MLPClassifier(hidden_layer_sizes=(16,), max_iter=60, random_state=0), X, y)
    spec = extract_model_spec(clf.predict_proba)
    assert isinstance(spec, MLPModelSpec)
    assert spec.activation == "binary_logistic" and spec.kappa == 1.0 and spec.n_outputs == 2
    assert spec.W1.shape == (16, 6) and spec.W2.shape == (1, 16)
    np.testing.assert_allclose(spec(X), clf.predict_proba(X), rtol=0, atol=1e-12)


def test_multiclass_classifier_extraction_matches_sklearn():
    rng, X = _data(seed=1)
    y = np.argmax(X[:, :3], axis=1)
    clf = _fit(MLPClassifier(hidden_layer_sizes=(20,), max_iter=60, random_state=1), X, y)
    spec = extract_model_spec(clf.predict_proba)
    assert spec.activation == "softmax" and spec.n_outputs == 3 and not spec.scalar_out
    np.testing.assert_allclose(spec(X), clf.predict_proba(X), rtol=0, atol=1e-12)


@pytest.mark.parametrize("n_out", [1, 2])
def test_regressor_extraction_matches_sklearn(n_out):
    rng, X = _data(seed=2)
    y = X[:, :n_out] * 2.0 + np.maximum(X[:, 1:1 + n_out], 0)
    reg = _fit(MLPRegressor(hidden_layer_sizes=(12,), max_iter=60, random_state=2), X, y[:, 0] if n_out == 1 else y)
    spec = extract_model_spec(reg.predict)
    assert spec.activation == "identity" and spec.scalar_out == (n_out == 1) and spec.n_outputs == n_out
    got, want = spec(X), reg.predict(X)
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)


def test_spec_passes_through_and_linear_models_are_unchanged():
    spec = MLPModelSpec(np.ones((3, 2)), np.zeros(3), np.ones((1, 3)), [0.5], "binary_logistic")
    assert extract_model_spec(spec) is spec
    clf = LinearSoftmaxClassifier(np.ones((1, 4)), [0.1])
    lin = extract_model_spec(clf.predict_proba)
    assert isinstance(lin, LinearModelSpec) and lin.kappa == 2.0
    with pytest.raises(TypeError):
        extract_model_spec(lambda X: X)


def test_spec_forward_is_relu_then_head():
    rng = np.random.default_rng(3)
    W1, b1, W2, b2 = rng.standard_normal((5, 4)), rng.standard_normal(5), rng.standard_normal((2, 5)), rng.standard_normal(2)
    X = rng.standard_normal((7, 4))
    h = np.maximum(X @ W1.T + b1, 0)
    np.testing.assert_allclose(MLPModelSpec(W1, b1, W2, b2, "identity")(X), h @ W2.T + b2, rtol=1e-14)
    z = h @ W2[:1].T + b2[:1]
    p = MLPModelSpec(W1, b1, W2[:1], b2[:1], "binary_logistic")(X)
    np.testing.assert_allclose(p[:, 1], 1 / (1 + np.exp(-z[:, 0])), rtol=1e-13)
    np.testing.assert_allclose(p.sum(axis=1), 1.0, rtol=1e-15)


def test_refusals():
    rng, X = _data(seed=4)
    y = (X[:, 0] > 0).astype(int)
    deep = _fit(MLPClassifier(hidden_layer_sizes=(8, 8), max_iter=20, random_state=0), X, y)
    with pytest.raises(NotImplementedError, match="hidden layers"):
        extract_model_spec(deep.predict_proba)
    for act in ("tanh", "logistic", "identity"):
        m = _fit(MLPClassifier(hidden_layer_sizes=(8,), activation=act, max_iter=20, random_state=0), X, y)
        with pytest.raises(NotImplementedError, match="ReLU"):
            extract_model_spec(m.predict_proba)
    wide = _fit(MLPClassifier(hidden_layer_sizes=(129,), max_iter=5, random_state=0), X, y)
    with pytest.raises(NotImplementedError, match="128"):
        extract_model_spec(wide.predict_proba)
    ok = _fit(MLPClassifier(hidden_layer_sizes=(8,), max_iter=20, random_state=0), X, y)
    with pytest.raises(TypeError, match="labels"):
        extract_model_spec(ok.predict)
    multilabel = _fit(MLPClassifier(hidden_layer_sizes=(8,), max_iter=20, random_state=0), X,
                      np.c_[y, 1 - y, (X[:, 1] > 0).astype(int)])
    with pytest.raises(NotImplementedError, match="multilabel"):
        extract_model_spec(multilabel.predict_proba)
    ymany = (np.arange(len(X)) % 9)
    many = _fit(MLPClassifier(hidden_layer_sizes=(8,), max_iter=5, random_state=0), X, ymany)
    with pytest.raises(NotImplementedError, match="at most 8"):
        extract_model_spec(many.predict_proba)
    reg = _fit(MLPRegressor(hidden_layer_sizes=(8,), max_iter=5, random_state=0), X, np.tile(X[:, :1], (1, 9)))
    with pytest.raises(NotImplementedError, match="at most 8"):
        extract_model_spec(reg.predict)


def test_spec_validation():
    W1, b1 = np.ones((3, 2)), np.zeros(3)
    with pytest.raises(ValueError, match="b1"):
        MLPModelSpec(W1, np.zeros(2), np.ones((1, 3)), [0.0], "identity")
    with pytest.raises(ValueError, match="hidden layer has 3"):
        MLPModelSpec(W1, b1, np.ones((1, 4)), [0.0], "identity")
    with pytest.raises(ValueError, match="b2"):
        MLPModelSpec(W1, b1, np.ones((2, 3)), [0.0], "identity")
    with pytest.raises(ValueError, match="unknown activation"):
        MLPModelSpec(W1, b1, np.ones((1, 3)), [0.0], "tanh")
    with pytest.raises(ValueError, match="single output"):
        MLPModelSpec(W1, b1, np.ones((2, 3)), [0.0, 0.0], "binary_logistic")
    with pytest.raises(ValueError, match="two output"):
        MLPModelSpec(W1, b1, np.ones((1, 3)), [0.0], "softmax")
