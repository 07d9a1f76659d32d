"""The model side of the hot path: linear scores (or one hidden layer of ReLU units) followed by a probability head.

The reference passes an opaque Python callable (``clf.predict_proba`` of a scikit-learn
``LogisticRegression(multi_class='multinomial')``, benchmarks/ray_pool.py:34, scripts/fit_adult_model.py:27-32).
CUDA kernels cannot call Python, so the engine needs the callable's parameters.  ``extract_linear_spec``
recovers them from the bound method's owner and ``GpuKernelExplainer`` checks the recovered model against the
callable on the background rows before trusting it; anything else raises (there is no CPU fallback)."""
import numpy as np

from . import _cabi


class LinearModelSpec:
    """``z = X W^T + b`` then a head.  ``W`` is [R, D], ``b`` [R].

    activation: 'identity' (outputs z), 'binary_logistic' (R == 1; outputs [1 - s, s], s = sigmoid(kappa z)),
    'softmax' (outputs softmax(z), R = C >= 2).  ``scalar_out``: the callable returns a 1-D array."""

    def __init__(self, W, b, activation, kappa=1.0, scalar_out=False):
        self.W = np.ascontiguousarray(np.atleast_2d(np.asarray(W, dtype=np.float64)))
        self.b = np.ascontiguousarray(np.atleast_1d(np.asarray(b, dtype=np.float64)))
        if self.W.shape[0] != self.b.shape[0]:
            raise ValueError(f"W has {self.W.shape[0]} rows but b has {self.b.shape[0]} entries")
        if activation not in ("identity", "binary_logistic", "softmax"):
            raise ValueError(f"unknown activation {activation!r}")
        if activation == "binary_logistic" and self.W.shape[0] != 1:
            raise ValueError("binary_logistic needs a single score row")
        self.activation = activation
        self.kappa = float(kappa)
        self.scalar_out = bool(scalar_out)

    @property
    def act_code(self):
        return {"identity": _cabi.ACT_IDENTITY, "binary_logistic": _cabi.ACT_BINARY_LOGISTIC,
                "softmax": _cabi.ACT_SOFTMAX}[self.activation]

    @property
    def n_outputs(self):
        return 2 if self.activation == "binary_logistic" else self.W.shape[0]

    def __call__(self, X):
        """NumPy evaluation with scikit-learn's conventions (used on the host by build_explanation and tests)."""
        X = np.asarray(X, dtype=np.float64)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        z = X @ self.W.T + self.b
        if self.activation == "identity":
            return z[:, 0] if self.scalar_out else z
        if self.activation == "binary_logistic":
            t = self.kappa * z[:, 0]
            scores = np.c_[-t / 2.0, t / 2.0]
        else:
            scores = z
        scores = scores - scores.max(axis=1, keepdims=True)
        e = np.exp(scores)
        return e / e.sum(axis=1, keepdims=True)


class LinearSoftmaxClassifier:
    """Minimal stand-in for the fitted scikit-learn 0.23 ``LogisticRegression(multi_class='multinomial')`` the
    reference pickles (scripts/fit_adult_model.py:27-32): ``coef_`` [1, D] / ``intercept_`` [1] for two classes
    with ``predict_proba = softmax([-z, z])`` (so p1 = sigmoid(2 z)), or [C, D] / [C] with a plain softmax."""

    def __init__(self, coef, intercept, multi_class="multinomial"):
        self.coef_ = np.atleast_2d(np.asarray(coef, dtype=np.float64))
        self.intercept_ = np.atleast_1d(np.asarray(intercept, dtype=np.float64))
        self.multi_class = multi_class
        self.classes_ = np.arange(2 if self.coef_.shape[0] == 1 else self.coef_.shape[0])

    def dks_linear_spec(self):
        if self.coef_.shape[0] == 1:
            return LinearModelSpec(self.coef_, self.intercept_, "binary_logistic",
                                   kappa=2.0 if self.multi_class == "multinomial" else 1.0)
        if self.multi_class != "multinomial":
            raise NotImplementedError("one-vs-rest multi-class heads are not supported")
        return LinearModelSpec(self.coef_, self.intercept_, "softmax")

    def decision_function(self, X):
        z = np.asarray(X, dtype=np.float64) @ self.coef_.T + self.intercept_
        return z[:, 0] if z.shape[1] == 1 else z

    def predict_proba(self, X):
        return self.dks_linear_spec()(X)

    def predict(self, X):
        return self.classes_[np.argmax(self.predict_proba(X), axis=1)]


def extract_linear_spec(predictor):
    """Recover ``LinearModelSpec`` from what the reference hands to ``KernelShap`` (a callable).

    Accepts: a ``LinearModelSpec``; any object/bound method whose owner offers ``dks_linear_spec()``; bound
    ``predict_proba`` / ``decision_function`` / ``predict`` of scikit-learn linear models (``coef_``/``intercept_``).
    Raises ``TypeError`` for everything else."""
    if isinstance(predictor, LinearModelSpec):
        return predictor
    owner = getattr(predictor, "__self__", None)
    method = getattr(predictor, "__name__", None)
    if owner is None and hasattr(predictor, "dks_linear_spec"):
        return predictor.dks_linear_spec()
    if owner is None:
        raise TypeError("predictor must be a bound method of a linear model (e.g. clf.predict_proba) or a "
                        "LinearModelSpec: the CUDA engine cannot call an opaque Python function and has no CPU fallback")
    if hasattr(owner, "dks_linear_spec") and method == "predict_proba":
        return owner.dks_linear_spec()
    if not (hasattr(owner, "coef_") and hasattr(owner, "intercept_")):
        raise TypeError(f"{type(owner).__name__} exposes no coef_/intercept_: only linear models are supported")
    coef = np.atleast_2d(np.asarray(owner.coef_, dtype=np.float64))
    intercept = np.atleast_1d(np.asarray(owner.intercept_, dtype=np.float64))
    if method == "predict_proba":
        if coef.shape[0] == 1:
            mc = getattr(owner, "multi_class", "auto")
            # scikit-learn >= 1.5 binary problems: sigmoid(z); 0.23 'multinomial' binary: softmax([-z, z])
            kappa = 2.0 if mc == "multinomial" else 1.0
            return LinearModelSpec(coef, intercept, "binary_logistic", kappa=kappa)
        if getattr(owner, "multi_class", "multinomial") == "ovr":
            raise NotImplementedError("one-vs-rest multi-class heads are not supported")
        return LinearModelSpec(coef, intercept, "softmax")
    if method in ("decision_function", "predict", "_decision_function"):
        if method == "predict" and hasattr(owner, "classes_"):
            raise TypeError("classifier.predict returns labels, which KernelSHAP cannot explain; pass predict_proba")
        return LinearModelSpec(coef, intercept, "identity", scalar_out=coef.shape[0] == 1)
    raise TypeError(f"unsupported predictor method {method!r}")


MLP_MAX_HIDDEN = 128
MLP_MAX_OUTPUTS = 8


class MLPModelSpec:
    """One hidden layer of ReLU units, then a head: ``h = relu(X W1^T + b1)``, ``z = h W2^T + b2``.  ``W1`` is [H, D],
    ``b1`` [H], ``W2`` [R, H], ``b2`` [R]; ``activation`` / ``kappa`` / ``scalar_out`` as in ``LinearModelSpec``
    ('binary_logistic' is scikit-learn's logistic output unit with kappa = 1: outputs [1 - s, s])."""

    def __init__(self, W1, b1, W2, b2, activation, kappa=1.0, scalar_out=False):
        self.W1 = np.ascontiguousarray(np.atleast_2d(np.asarray(W1, dtype=np.float64)))
        self.b1 = np.ascontiguousarray(np.atleast_1d(np.asarray(b1, dtype=np.float64)))
        self.W2 = np.ascontiguousarray(np.atleast_2d(np.asarray(W2, dtype=np.float64)))
        self.b2 = np.ascontiguousarray(np.atleast_1d(np.asarray(b2, dtype=np.float64)))
        H, R = self.W1.shape[0], self.W2.shape[0]
        if self.b1.shape != (H,):
            raise ValueError(f"W1 has {H} rows but b1 has {self.b1.shape[0]} entries")
        if self.W2.shape[1] != H:
            raise ValueError(f"W2 has {self.W2.shape[1]} columns but the hidden layer has {H} units")
        if self.b2.shape != (R,):
            raise ValueError(f"W2 has {R} rows but b2 has {self.b2.shape[0]} entries")
        if activation not in ("identity", "binary_logistic", "softmax"):
            raise ValueError(f"unknown activation {activation!r}")
        if activation == "binary_logistic" and R != 1:
            raise ValueError("binary_logistic needs a single output unit")
        if activation == "softmax" and R < 2:
            raise ValueError("softmax needs at least two output units")
        if H > MLP_MAX_HIDDEN:
            raise NotImplementedError(f"{H} hidden units: the CUDA engine handles at most {MLP_MAX_HIDDEN}")
        if R > MLP_MAX_OUTPUTS:
            raise NotImplementedError(f"{R} output units: the CUDA engine handles at most {MLP_MAX_OUTPUTS}")
        self.activation = activation
        self.kappa = float(kappa)
        self.scalar_out = bool(scalar_out)

    act_code = LinearModelSpec.act_code

    @property
    def n_outputs(self):
        return 2 if self.activation == "binary_logistic" else self.W2.shape[0]

    @property
    def n_features(self):
        return self.W1.shape[1]

    def __call__(self, X):
        """NumPy float64 forward with scikit-learn's conventions."""
        X = np.asarray(X, dtype=np.float64)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        h = np.maximum(X @ self.W1.T + self.b1, 0.0)
        return LinearModelSpec(self.W2, self.b2, self.activation, self.kappa, self.scalar_out)(h)


def _mlp_spec_from_sklearn(owner, method):
    """``MLPClassifier.predict_proba`` / ``MLPRegressor.predict`` of a fitted one-hidden-layer ReLU network."""
    coefs, intercepts = owner.coefs_, owner.intercepts_
    if len(coefs) != 2:
        raise NotImplementedError(f"{type(owner).__name__} has {len(coefs) - 1} hidden layers: the CUDA engine explains "
                                  "networks of one hidden layer")
    if owner.activation != "relu":
        raise NotImplementedError(f"hidden activation {owner.activation!r}: the CUDA engine explains ReLU networks only")
    out = owner.out_activation_
    W1, b1 = np.asarray(coefs[0], dtype=np.float64).T, intercepts[0]
    W2, b2 = np.asarray(coefs[1], dtype=np.float64).T, intercepts[1]
    if hasattr(owner, "classes_"):
        if method != "predict_proba":
            raise TypeError("classifier.predict returns labels, which KernelSHAP cannot explain; pass predict_proba")
        if out == "logistic" and W2.shape[0] == 1:
            return MLPModelSpec(W1, b1, W2, b2, "binary_logistic", kappa=1.0)
        if out == "softmax":
            return MLPModelSpec(W1, b1, W2, b2, "softmax")
        raise NotImplementedError(f"{type(owner).__name__} with {W2.shape[0]} {out} outputs (multilabel): only binary "
                                  "and multi-class heads are supported")
    if method != "predict":
        raise TypeError(f"unsupported predictor method {method!r}")
    if out != "identity":
        raise NotImplementedError(f"regression output activation {out!r} is not supported")
    return MLPModelSpec(W1, b1, W2, b2, "identity", scalar_out=W2.shape[0] == 1)


def _is_sklearn_mlp(owner):
    return all(hasattr(owner, a) for a in ("coefs_", "intercepts_", "activation", "out_activation_"))


def extract_model_spec(predictor):
    """What the engine calls: an ``MLPModelSpec`` for an ``MLPModelSpec`` or a bound ``predict_proba`` / ``predict`` of a
    fitted scikit-learn ``MLPClassifier`` / ``MLPRegressor``; ``extract_linear_spec(predictor)`` for everything else."""
    if isinstance(predictor, MLPModelSpec):
        return predictor
    owner = getattr(predictor, "__self__", None)
    if owner is not None and _is_sklearn_mlp(owner):
        return _mlp_spec_from_sklearn(owner, getattr(predictor, "__name__", None))
    return extract_linear_spec(predictor)
