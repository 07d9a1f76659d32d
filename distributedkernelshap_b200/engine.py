"""``GpuKernelExplainer``: the object that sits in ``KernelShap._explainer``.

In the reference that slot holds ``KernelExplainerWrapper`` (explainers/kernel_shap.py:217-261), a subclass of
``shap.KernelExplainer``; ``KernelShap`` only needs ``get_explanation(X, **kwargs)``, ``.expected_value`` and
``.vector_out`` from it (kernel_shap.py:789-790, :880-887).  This class keeps that constructor shape
``(predictor, background_data, link=..., seed=...)`` and those members, and runs the per-instance hot path
(varying groups -> coalition plan -> mask/impute -> predict -> background mean -> link -> constrained WLS) in
CUDA through the C ABI of ``include/dks.h``.  No CPU fallback: without ``libdks.so`` and a B200 it raises.
"""
import ctypes as C
import logging

import numpy as np

from . import _cabi
from .data import DenseData, convert_to_data, convert_to_link
from .plan import build_plan, l1_tables, pack_dense_plan, projection, resolve_nsamples, sampling_info
from .predictors import MLPModelSpec, extract_model_spec

logger = logging.getLogger(__name__)

MODEL_CHECK_RTOL = 1e-9
MAX_ROWS_PER_CALL = 65536     # rows per C-ABI call: bounds the engine's per-call workspace (n x S x 8 B on the fast path)


def refuse_partial_sets_beyond_64_groups(G, hist):
    """Multi-word coalition rows (more than 64 groups) exist on the shared-plan path only, which takes the instances whose
    groups ALL vary.  ``hist[M]`` = instances with M varying groups: anything below G is refused here, before plans (and,
    beyond 128 groups, their projections) are built for sizes no kernel would evaluate -- the library reports the same
    condition as status 3 (unsupported)."""
    if G <= 64:
        return
    partial = [M for M in range(0, G) if hist[M] > 0]
    if partial:
        raise NotImplementedError(
            f"{int(sum(hist[M] for M in partial))} instance(s) have a partial varying set (M in {partial[:8]}"
            f"{'...' if len(partial) > 8 else ''} of {G} groups): more than 64 groups run on the shared-plan path, which "
            "needs every group to vary (unsupported otherwise)")


class GpuKernelExplainer:
    """CUDA KernelSHAP explainer with the interface of ``shap.KernelExplainer`` / ``KernelExplainerWrapper``.

    Parameters
    ----------
    model
        What the reference passes as ``predictor``: a bound ``predict_proba`` / ``decision_function`` of a linear
        model, ``predict_proba`` / ``predict`` of a one-hidden-layer ReLU ``MLPClassifier`` / ``MLPRegressor``, or a
        ``LinearModelSpec`` / ``MLPModelSpec`` (see ``predictors.extract_model_spec``).
    data
        Background data: array, DataFrame or ``DenseData`` (groups and weights honoured).
    link
        ``'identity'`` or ``'logit'``.
    seed
        As in ``KernelExplainerWrapper.__init__`` (kernel_shap.py:225-228): seeds the global legacy NumPy stream the
        sampled part of the coalition plans is drawn from.
    device
        CUDA device ordinal (default: ``LOCAL_RANK`` under torchrun, else 0).
    """

    def __init__(self, model, data, link="identity", seed=None, device=None, kernel="auto", plan_mode="shared", **kwargs):
        if kwargs:
            raise TypeError(f"unexpected keyword arguments {sorted(kwargs)}")
        if plan_mode not in ("shared", "per_instance"):
            raise ValueError("plan_mode must be 'shared' or 'per_instance'")
        if seed is not None:
            np.random.seed(seed)           # the reference's constructor side effect (kernel_shap.py:225-228)
        self.seed = None if seed is None else int(seed)
        self.plan_mode = plan_mode
        self.plan_seed = 0 if seed is None else int(seed) & 0xFFFFFFFFFFFFFFFF
        self.lib = _cabi.load()
        self.link = convert_to_link(link)
        self.model_callable = model
        self.spec = extract_model_spec(model)
        self.is_mlp = isinstance(self.spec, MLPModelSpec)
        self.data = convert_to_data(data)
        if self.data.transposed:
            raise NotImplementedError("transposed DenseData (group sizes matching axis 0) is not supported")
        bg = np.ascontiguousarray(np.asarray(self.data.data, dtype=np.float64))
        if bg.ndim != 2:
            raise TypeError("background data must be two-dimensional")
        self.N, self.P = bg.shape
        n_cols = (self.spec.W1 if self.is_mlp else self.spec.W).shape[1]
        if n_cols != self.P:
            raise ValueError(f"model expects {n_cols} columns, background has {self.P}")
        if self.N > 100:
            logger.warning("Using %d background data samples could cause slower run times. Consider using "
                           "shap.sample(data, K) or shap.kmeans(data, K) to summarize the background as K samples.",
                           self.N)
        if device is None:
            import os
            device = int(os.environ.get("LOCAL_RANK", "0"))
        self.device = int(device)

        self._ctx = C.c_void_p()
        _cabi.check(self.lib.dks_create(C.byref(self._ctx), self.device))
        weights = np.ascontiguousarray(self.data.weights, dtype=np.float64)
        _cabi.check(self.lib.dks_set_background(self._ctx, _cabi.ptr(bg), self.N, self.P, _cabi.ptr(weights)))
        offsets = np.zeros(self.data.groups_size + 1, dtype=np.int32)
        offsets[1:] = np.cumsum([len(g) for g in self.data.groups])
        cols = np.ascontiguousarray(np.concatenate([np.asarray(g, dtype=np.int32) for g in self.data.groups]), dtype=np.int32)
        _cabi.check(self.lib.dks_set_groups(self._ctx, _cabi.ptr(offsets), _cabi.ptr(cols), self.data.groups_size))
        if self.is_mlp:
            sp = self.spec
            _cabi.check(self.lib.dks_set_mlp_model(self._ctx, _cabi.ptr(sp.W1), _cabi.ptr(sp.b1), sp.W1.shape[0], _cabi.ptr(sp.W2),
                                                   _cabi.ptr(sp.b2), sp.W2.shape[0], sp.act_code, sp.kappa, int(sp.scalar_out)))
        else:
            _cabi.check(self.lib.dks_set_model(self._ctx, _cabi.ptr(self.spec.W), _cabi.ptr(self.spec.b), self.spec.W.shape[0],
                                               self.spec.act_code, self.spec.kappa, int(self.spec.scalar_out)))
        link_code = _cabi.LINK_LOGIT if str(self.link) == "logit" else _cabi.LINK_IDENTITY
        _cabi.check(self.lib.dks_set_link(self._ctx, link_code))
        self.set_kernel(kernel)
        _cabi.check(self.lib.dks_set_plan_mode(self._ctx, 1 if plan_mode == "per_instance" else 0, self.plan_seed))
        _cabi.check(self.lib.dks_fit(self._ctx))

        self.D = self.spec.n_outputs
        fnull = np.zeros(self.D)
        expected = np.zeros(self.D)
        _cabi.check(self.lib.dks_get_fnull(self._ctx, _cabi.ptr(fnull), _cabi.ptr(expected)))
        self.vector_out = not self.spec.scalar_out
        self.fnull = fnull
        self.expected_value = expected if self.vector_out else float(expected[0])
        self._nsamples_req = None
        self._plan_cache = {}
        self._l1_uploaded = {}
        self._l1_state = (0, 0, 0)
        self._link_fx_parts = []
        self._last_rows = 0
        self._check_model_against_callable(bg)

    # ------------------------------------------------------------------------------------------------------
    def _check_model_against_callable(self, bg):
        """The extracted model must reproduce the user's callable on the background rows (GPU float64 forward)."""
        if not callable(self.model_callable):
            return
        want = np.asarray(self.model_callable(bg), dtype=np.float64).reshape(self.N, -1)
        got = self.predict(bg)
        if want.shape != got.shape or not np.allclose(got, want, rtol=1e-7, atol=1e-9, equal_nan=True):
            raise ValueError(f"the {'network' if self.is_mlp else 'linear model'} extracted from `predictor` does not "
                             "reproduce predictor(background): "
                             "refusing to explain a different function (max abs diff "
                             f"{np.max(np.abs(got - want)) if want.shape == got.shape else 'shape mismatch'})")

    def predict(self, X):
        """Model outputs [n, C] computed on the GPU in float64."""
        X = np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64)))
        out = np.zeros((X.shape[0], self.D))
        _cabi.check(self.lib.dks_predict_host(self._ctx, _cabi.ptr(X), X.shape[0], _cabi.ptr(out)))
        return out

    def set_kernel(self, kernel):
        code = {"auto": _cabi.KERNEL_AUTO, "simt": _cabi.KERNEL_SIMT, "tcgen05": _cabi.KERNEL_TCGEN05,
                "shared": _cabi.KERNEL_SHARED}[kernel]
        if kernel == "tcgen05" and getattr(self, "is_mlp", False):
            raise NotImplementedError("the tcgen05 kernel evaluates linear models only; networks run on 'auto', 'shared' "
                                      "or 'simt'")
        _cabi.check(self.lib.dks_set_kernel(self._ctx, code))
        self.kernel = kernel

    def set_option(self, name, value):
        """Tuning knob of the C library (``dks_set_option``): 'fused', 'fused_ni', 'fused_warps', 'fused_batch',
        'push_in_kernel', 'graph', 'graph_timing', 'wide_gemm', 'wide_acache'."""
        _cabi.check(self.lib.dks_set_option(self._ctx, str(name).encode(), int(value)))

    # ------------------------------------------------------------------------------------------------------
    def _set_nsamples(self, nsamples):
        req = 0 if nsamples in ("auto", None) else int(nsamples)
        if req != self._nsamples_req:
            _cabi.check(self.lib.dks_set_nsamples(self._ctx, req))
            self._nsamples_req = req

    def _l1_guard(self, l1_reg, nsamples, hist=None):
        """Upstream's ``solve`` runs an l1 feature selection before the constrained WLS when ``l1_reg`` is 'aic' / 'bic' /
        'num_features(k)', or under 'auto' when fewer than 20% of the coalition space is evaluated.  Without ``hist``:
        whether the M histogram is needed to decide.  With it: ``(mode, k, others_plain)`` for ``dks_set_l1`` -- the
        selection runs on the shared-plan path (csrc/dks_l1.cuh) for the instances whose groups all vary; what that path
        does not cover is refused, never silently solved without the selection."""
        if l1_reg in (False, 0):
            return False if hist is None else (0, 0, 0)
        G = self.data.groups_size
        explicit = None
        if l1_reg in ("aic", "bic"):
            explicit = (1 if l1_reg == "aic" else 2, 0)
        elif isinstance(l1_reg, str) and l1_reg.startswith("num_features("):
            explicit = (3, int(l1_reg[len("num_features("):-1]))
        elif l1_reg != "auto":
            raise NotImplementedError(f"l1_reg={l1_reg!r}: a fixed Lasso strength is not implemented in the CUDA engine; "
                                      "use 'auto', 'aic', 'bic', 'num_features(k)' or False")

        def needs(M):
            if explicit is not None:
                return True
            S, max_s = resolve_nsamples(M, nsamples)
            return S / max_s < 0.2
        if hist is None:
            return explicit is not None or any(needs(M) for M in range(2, G + 1))
        present = [M for M in range(2, G + 1) if hist[M] > 0]
        wanting = [M for M in present if needs(M)]
        if not wanting:
            return (0, 0, 0)
        if max(wanting) > 128:
            raise NotImplementedError(
                f"l1_reg={l1_reg!r} selects features among {max(wanting)} varying groups; the CUDA engine's LARS path covers at "
                "most 128 groups -- pass l1_reg=False for the plain constrained WLS (or 'num_features(k)' on a narrower "
                "grouping)")
        partial = [M for M in wanting if M != G]
        if partial:
            raise NotImplementedError(
                f"l1_reg={l1_reg!r} selects features for instances with M in {partial} varying groups (a partial varying "
                "set); the CUDA engine runs the selection for instances whose groups all vary only -- pass l1_reg=False")
        if self.plan_mode != "shared":
            raise NotImplementedError("l1 feature selection runs with plan_mode='shared' only")
        if self.spec.act_code != _cabi.ACT_BINARY_LOGISTIC or not np.allclose(self.data.weights, self.data.weights[0]):
            raise NotImplementedError("l1 feature selection needs the binary-logistic head and uniform background weights "
                                      "(the shared-plan path)")
        mode, k = explicit if explicit is not None else (1, 0)
        return (mode, k, 1 if len(present) > 1 else 0)

    def _apply_l1(self, l1_reg, nsamples, hist):
        """Uploads the l1 tables of the G-group plan when the call needs them and tells the library the mode."""
        mode, k, others_plain = (0, 0, 0) if l1_reg in (False, 0) else self._l1_guard(l1_reg, nsamples, hist)
        if mode:
            G = self.data.groups_size
            S, _ = resolve_nsamples(G, nsamples)
            if self._l1_uploaded.get(G) != S:
                self._ensure_shared_plans(hist, nsamples)
                t = l1_tables(self.shared_plan(G, nsamples))
                sqab = np.ascontiguousarray(t["sqa"] + t["sqb"])
                _cabi.check(self.lib.dks_set_l1_tables(
                    self._ctx, G, _cabi.ptr(t["gram_raw"]), _cabi.ptr(t["gram_norm"]), _cabi.ptr(t["colsum"]),
                    _cabi.ptr(t["scale"]), _cabi.ptr(t["bz"]), _cabi.ptr(t["gram_w"]), _cabi.ptr(t["b"]), _cabi.ptr(sqab),
                    t["sum_b"], t["sum_sqb"], t["n_aug"]))
                self._l1_uploaded[G] = S
        if (mode, k, others_plain) != self._l1_state:
            _cabi.check(self.lib.dks_set_l1(self._ctx, mode, k, others_plain))
            self._l1_state = (mode, k, others_plain)

    def shared_plan(self, M, nsamples="auto"):
        """The coalition plan every instance with ``M`` varying groups shares under ``plan_mode='shared'`` (also the
        source of the enumerated prefix of device-drawn plans).  With a ``seed`` the sampled part comes from a private
        ``RandomState`` keyed by (seed, M, rows): the same plan on every worker, thread and rank whatever the order in
        which they meet the M values.  Without a seed it is drawn from the global legacy stream at first use, like the
        reference's unseeded explainer."""
        S, _ = resolve_nsamples(M, nsamples)
        cached = self._plan_cache.get((M, S))
        if cached is not None:
            return cached
        rng = None
        if self.seed is not None:
            rng = np.random.RandomState((self.seed * 1000003 + 7919 * M + S) & 0xFFFFFFFF)
        plan = build_plan(M, nsamples, rng=rng)
        self._plan_cache[(M, S)] = plan         # what was uploaded is what this accessor reports
        return plan

    def _ensure_shared_plans(self, hist, nsamples):
        refuse_partial_sets_beyond_64_groups(self.data.groups_size, hist)
        for M in range(2, self.data.groups_size + 1):
            if hist[M] == 0:
                continue
            present = C.c_int(0)
            _cabi.check(self.lib.dks_has_shared_plan(self._ctx, M, C.byref(present)))
            if present.value:
                continue
            plan = self.shared_plan(M, nsamples)
            _cabi.check(self.lib.dks_set_shared_plan(self._ctx, M, plan.S, _cabi.ptr(plan.zbits), _cabi.ptr(plan.weights)))
            if M > 128:
                # sixteen-word rows: the (M-1) x (M-1) normal matrix is factored here, once per plan, in float64
                pt, dvec = projection(plan)
                _cabi.check(self.lib.dks_set_plan_projection(self._ctx, M, _cabi.ptr(pt), _cabi.ptr(dvec)))
            nfixed, n_full, n_paired, cdf, weight_left = sampling_info(plan)
            if len(cdf) > 32:
                if self.plan_mode == "per_instance":
                    raise NotImplementedError(f"per-instance device plans support at most 32 sampled subset sizes (M={M})")
                continue
            _cabi.check(self.lib.dks_set_plan_sampling(self._ctx, M, nfixed, n_full, n_paired, len(cdf),
                                                       _cabi.ptr(cdf) if len(cdf) else None, weight_left))

    def m_histogram(self):
        hist = np.zeros(self.data.groups_size + 1, dtype=np.int32)
        _cabi.check(self.lib.dks_get_m_histogram(self._ctx, _cabi.ptr(hist)))
        return hist

    def varying(self, X):
        """(M [n], bit-mask [n]) of ``KernelExplainer.varying_groups`` for every row of X (GPU)."""
        X = np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64)))
        _cabi.check(self.lib.dks_prepare_host(self._ctx, _cabi.ptr(X), X.shape[0]))
        M = np.zeros(X.shape[0], dtype=np.int32)
        mask = np.zeros(X.shape[0], dtype=np.uint64)
        _cabi.check(self.lib.dks_get_varying(self._ctx, _cabi.ptr(M), _cabi.ptr(mask)))
        return M, mask

    # ------------------------------------------------------------------------------------------------------
    def shap_values(self, X, **kwargs):
        """``KernelExplainer.shap_values``: list of C arrays [n, groups] (vector output) or one array.

        kwargs: ``nsamples`` ('auto' | int), ``l1_reg`` ('auto' | False | 0), ``silent`` (ignored), and
        ``plans`` = per-instance coalition plans ``[(Z [S_i, M_i] | zbits [S_i], w [S_i]) | None, ...]`` evaluated
        instead of the engine's own shared plans (this is how tests give the oracle and the GPU identical inputs)."""
        nsamples = kwargs.pop("nsamples", "auto")
        l1_reg = kwargs.pop("l1_reg", "auto")
        plans = kwargs.pop("plans", None)
        row_offset = int(kwargs.pop("row_offset", 0))
        kwargs.pop("silent", None)
        if kwargs:
            raise TypeError(f"unexpected keyword arguments {sorted(kwargs)}")
        try:
            import pandas as pd
            if isinstance(X, (pd.DataFrame, pd.Series)):
                X = X.values
        except ImportError:  # pragma: no cover
            pass
        try:
            from scipy import sparse
            if sparse.issparse(X):
                X = X.toarray()
        except ImportError:  # pragma: no cover
            pass
        X = np.asarray(X, dtype=np.float64)
        single = X.ndim == 1
        if single:
            X = X.reshape(1, -1)
        assert X.ndim == 2, "Instance must have 1 or 2 dimensions!"
        if X.shape[1] != self.P:
            raise ValueError(f"X has {X.shape[1]} columns, background has {self.P}")
        X = np.ascontiguousarray(X)
        n, G = X.shape[0], self.data.groups_size
        if n == 0:                              # nothing to explain: empty arrays of the right shape (the C ABI wants n > 0)
            self._last_rows = 0
            empty = np.zeros((self.D, 0, G))
            return [empty[c] for c in range(self.D)] if self.vector_out else empty[0]
        self._set_nsamples(nsamples)
        need_hist = self._l1_guard(l1_reg, nsamples)

        if n > MAX_ROWS_PER_CALL:     # large inputs go through in row chunks (results are independent per row)
            parts, fx_parts = [], []
            for lo in range(0, n, MAX_ROWS_PER_CALL):
                hi = min(n, lo + MAX_ROWS_PER_CALL)
                sub = dict(nsamples=nsamples, l1_reg=l1_reg, row_offset=row_offset + lo)
                if plans is not None:
                    sub["plans"] = plans[lo:hi]
                part = self.shap_values(X[lo:hi], **sub)
                fx_parts.append(self.link_predictions().reshape(hi - lo, -1))
                parts.append(part if isinstance(part, list) else [part])
            merged = [np.concatenate([pt[c] for pt in parts], axis=0) for c in range(len(parts[0]))]
            self._link_fx_parts = fx_parts
            self._last_rows = n
            return merged if self.vector_out else merged[0]

        phi = np.empty((self.D, n, G))      # the device writes every entry (zeros for groups that do not vary)
        self._link_fx_parts = []
        if self.plan_mode == "per_instance":
            # the device draws each row's plan from (seed, global row index): tell it where this block starts
            _cabi.check(self.lib.dks_set_row_offset(self._ctx, row_offset))
        if plans is not None:
            if G > 64:
                raise NotImplementedError("caller-supplied per-instance plans need at most 64 groups (multi-word coalition "
                                          "rows exist on the shared-plan path only)")
            zb, w, stride = self._pack_external_plans(plans, n, nsamples)
            if need_hist:
                _cabi.check(self.lib.dks_prepare_host(self._ctx, _cabi.ptr(X), n))
                if self._l1_guard(l1_reg, nsamples, self.m_histogram())[0]:
                    raise NotImplementedError("l1 feature selection runs on the engine's shared plans, not on "
                                              "caller-supplied per-instance plans -- pass l1_reg=False")
            self._apply_l1(False, nsamples, None)
            _cabi.check(self.lib.dks_explain_host(self._ctx, _cabi.ptr(X), n, _cabi.ptr(phi), _cabi.ptr(zb), _cabi.ptr(w),
                                                  stride))
        else:
            if need_hist:
                _cabi.check(self.lib.dks_prepare_host(self._ctx, _cabi.ptr(X), n))
                hist = self.m_histogram()
                self._ensure_shared_plans(hist, nsamples)
                self._apply_l1(l1_reg, nsamples, hist)
            else:
                self._apply_l1(False, nsamples, None)
            rc = self.lib.dks_explain_host(self._ctx, _cabi.ptr(X), n, _cabi.ptr(phi), None, None, 0)
            if rc == _cabi.DKS_ERR_PLAN_MISSING:
                # first call (or a new M): build the missing plans from the M histogram and run again
                self._ensure_shared_plans(self.m_histogram(), nsamples)
                rc = self.lib.dks_explain_host(self._ctx, _cabi.ptr(X), n, _cabi.ptr(phi), None, None, 0)
            _cabi.check(rc)

        self._last_rows = n
        if not self.vector_out:
            return phi[0, 0] if single else phi[0]
        if single:
            return [phi[c, 0] for c in range(self.D)]
        return [phi[c] for c in range(self.D)]

    def link_predictions(self):
        """``link(f(x))`` of the rows of the last ``shap_values`` call, ``[n, C]`` (``[n]`` for scalar-output models):
        stage 1 of the explain call computes it on the device, so ``KernelShap.build_explanation`` does not have to run
        the predictor over ``X`` again for ``raw_prediction`` (kernel_shap.py:949)."""
        if self._link_fx_parts:                 # the call went through in row chunks
            out = np.concatenate(self._link_fx_parts, axis=0)
        elif self._last_rows == 0:
            return None
        else:
            out = np.zeros((self._last_rows, self.D))
            rc = self.lib.dks_get_link_fx(self._ctx, _cabi.ptr(out), self._last_rows)
            if rc == _cabi.DKS_ERR_INVALID:     # another call (varying(), explain_device()) ran stage 1 since
                return None
            _cabi.check(rc)
        return out if self.vector_out else out[:, 0]

    def summarise(self, n, segments=None, want_sums=False):
        """``KernelShap.build_explanation`` post-processing on the device, off the phi of the last host-path
        ``shap_values`` call over ``n`` rows (kernel_shap.py:36-109, :112-207, :952-956): mean |phi| per output and
        aggregated (``mean_abs`` [C + 1, Gp]), their descending order (``order``), the arg-max class of the raw prediction
        (``argmax`` [n]) and, with ``segments`` (offsets of consecutive groups to add up: ``sum_categories``), the summed
        shap values (``phi_sum`` [C, n, Gp]).  Returns None when the last call is not resident (row chunks, other calls)."""
        if n != self._last_rows or self._link_fx_parts:
            return None
        G = self.data.groups_size
        seg = None if segments is None else np.ascontiguousarray(segments, dtype=np.int32)
        Gp = G if seg is None else len(seg) - 1
        mean_abs = np.zeros((self.D + 1, Gp))
        order = np.zeros((self.D + 1, Gp), dtype=np.int32)
        argmax = np.zeros(n, dtype=np.int32)
        phi_sum = np.zeros((self.D, n, Gp)) if (want_sums and seg is not None) else None
        rc = self.lib.dks_summarise_host(self._ctx, n, _cabi.ptr(seg), Gp, _cabi.ptr(phi_sum), _cabi.ptr(mean_abs),
                                         _cabi.ptr(order), _cabi.ptr(argmax))
        if rc == _cabi.DKS_ERR_INVALID:
            return None
        _cabi.check(rc)
        return {"mean_abs": mean_abs, "order": order, "argmax": argmax, "phi_sum": phi_sum}

    def instance_plans(self):
        """Plans the device drew in the last ``plan_mode='per_instance'`` call: ``(zbits uint64[n, stride],
        w float64[n, stride])`` -- rows past an instance's S are zero.  For audits and tests."""
        n, stride = C.c_int(0), C.c_int(0)
        _cabi.check(self.lib.dks_get_instance_plans(self._ctx, None, None, C.byref(n), C.byref(stride)))
        zb = np.zeros((n.value, stride.value), dtype=np.uint64)
        w = np.zeros((n.value, stride.value), dtype=np.float64)
        if n.value:
            _cabi.check(self.lib.dks_get_instance_plans(self._ctx, _cabi.ptr(zb), _cabi.ptr(w), C.byref(n), C.byref(stride)))
        return zb, w

    def _pack_external_plans(self, plans, n, nsamples):
        if len(plans) != n:
            raise ValueError(f"got {len(plans)} plans for {n} instances")
        stride = max([len(p[1]) for p in plans if p is not None and p[1] is not None] + [2])
        zb = np.zeros((n, stride), dtype=np.uint64)
        w = np.zeros((n, stride), dtype=np.float64)
        for i, p in enumerate(plans):
            if p is None or p[1] is None:
                continue
            Z, wi = p[-2], np.asarray(p[-1], dtype=np.float64)
            Z = np.asarray(Z)
            bits = pack_dense_plan(Z) if Z.ndim == 2 else Z.astype(np.uint64)
            zb[i, :len(bits)] = bits
            w[i, :len(wi)] = wi
        return zb, w, stride

    # ---- device-resident API (torch tensors appear only as raw pointers) ---------------------------------------
    def set_stream(self, cuda_stream_ptr):
        """Enqueue the engine's work on the given ``cudaStream_t`` (e.g. ``torch.cuda.current_stream().cuda_stream``)."""
        _cabi.check(self.lib.dks_set_stream(self._ctx, C.c_void_p(int(cuda_stream_ptr))))

    def explain_device(self, X_dev_ptr, n, phi_dev_ptr, nsamples="auto"):
        """Asynchronously explain ``n`` rows resident in device memory (float64 [n, D] at ``X_dev_ptr``) into the device
        buffer ``phi_dev_ptr`` (float64 [C, n, G]) using the shared plans already on the device.  Call ``check_status()``
        after synchronising to learn about missing plans / numerical failures."""
        self._set_nsamples(nsamples)
        self._apply_l1(False, nsamples, None)             # the device-resident call is the plain constrained WLS
        _cabi.check(self.lib.dks_run_dev(self._ctx, C.c_void_p(int(X_dev_ptr)), int(n), C.c_void_p(int(phi_dev_ptr))))

    def explain_block_to_device(self, X, nsamples="auto", l1_reg="auto", row_offset=0, silent=None):
        """Explain host rows ``X`` and leave the shap values ON THE DEVICE: returns a float64 CUDA tensor ``[C, n, G]``
        (torch owns the buffers; the engine sees raw pointers).  Used by the SPMD path of ``DistributedExplainer`` so that
        the all-gather runs on what the solve wrote, without a host round trip.  Zero rows give an empty tensor."""
        import torch
        X = np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64)))
        n, G = X.shape[0], self.data.groups_size
        dev = torch.device("cuda", self.device)
        phi = torch.empty((self.D, n, G), dtype=torch.float64, device=dev)
        if n == 0:
            return phi
        if X.shape[1] != self.P:
            raise ValueError(f"X has {X.shape[1]} columns, background has {self.P}")
        self._set_nsamples(nsamples)
        need_hist = self._l1_guard(l1_reg, nsamples)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev)
            if getattr(self, "_block_stream", None) != stream.cuda_stream:
                self.set_stream(stream.cuda_stream)
                self._block_stream = stream.cuda_stream
            X_dev = torch.from_numpy(X).to(dev, non_blocking=True)
            if self.plan_mode == "per_instance":
                _cabi.check(self.lib.dks_set_row_offset(self._ctx, int(row_offset)))
            if need_hist:
                _cabi.check(self.lib.dks_prepare_dev(self._ctx, C.c_void_p(X_dev.data_ptr()), n))
                hist = self.m_histogram()
                self._ensure_shared_plans(hist, nsamples)
                self._apply_l1(l1_reg, nsamples, hist)
            else:
                self._apply_l1(False, nsamples, None)
            for attempt in range(2):
                _cabi.check(self.lib.dks_run_dev(self._ctx, C.c_void_p(X_dev.data_ptr()), n, C.c_void_p(phi.data_ptr())))
                detail = C.c_int(0)
                rc = self.lib.dks_last_status(self._ctx, C.byref(detail))            # synchronises the stream
                if rc == _cabi.DKS_ERR_PLAN_MISSING and attempt == 0:
                    self._ensure_shared_plans(self.m_histogram(), nsamples)       # first call / new M: build and rerun
                    continue
                _cabi.check(rc)
                break
        self._last_rows = 0                     # link_predictions() refers to host-path calls only
        return phi

    def set_peers(self, world, rank, gathered_ptrs, slab_doubles):
        """Multi-GPU push all-gather: ``gathered_ptrs[r]`` = device address (mapped in this process) of rank r's gathered
        ``[world, C, n, G]`` buffer; after every ``explain_device`` this rank's phi is stored into slab ``rank`` of every
        peer's buffer by the engine's own kernel.  ``world <= 1`` switches it off."""
        if world <= 1:
            _cabi.check(self.lib.dks_set_peers(self._ctx, 0, 0, None, 0))
            return
        ptrs = np.asarray([int(p) for p in gathered_ptrs], dtype=np.uint64)
        _cabi.check(self.lib.dks_set_peers(self._ctx, int(world), int(rank), _cabi.ptr(ptrs), int(slab_doubles)))

    def set_peer_flags(self, flag_ptrs):
        """Multi-GPU: ``flag_ptrs[r]`` = device address (mapped here) of rank r's zero-initialised ``uint64[world]`` flag
        array.  Every ``explain_device`` then ends with the engine's own cross-GPU signal / wait, so the gathered buffer is
        complete when the stream reaches the next operation.  ``None`` switches it off."""
        if flag_ptrs is None:
            _cabi.check(self.lib.dks_set_peer_flags(self._ctx, None))
            return
        ptrs = np.asarray([int(p) for p in flag_ptrs], dtype=np.uint64)
        _cabi.check(self.lib.dks_set_peer_flags(self._ctx, _cabi.ptr(ptrs)))

    def graph_launches(self):
        """How many ``explain_device`` calls were replayed as one CUDA-graph launch."""
        cnt = C.c_int64(0)
        _cabi.check(self.lib.dks_graph_launches(self._ctx, C.byref(cnt)))
        return cnt.value

    def check_status(self):
        """Synchronise the engine's stream and raise if the last explain reported a problem."""
        detail = C.c_int(0)
        _cabi.check(self.lib.dks_last_status(self._ctx, C.byref(detail)))

    # ---- KernelExplainerWrapper members (kernel_shap.py:231-261) ---------------------------------------------
    def get_explanation(self, X, **kwargs):
        """Accepts an array, or a ``(batch_index, batch)`` tuple when called from a distributed context."""
        if isinstance(X, tuple):
            batch_idx, batch = X
            return batch_idx, self.shap_values(batch, **kwargs)
        return self.shap_values(X, **kwargs)

    def return_attribute(self, name):
        return self.__getattribute__(name)

    # ---- introspection used by bench.py / tests -----------------------------------------------------------------
    def kernel_launches(self):
        v = C.c_int64(0)
        _cabi.check(self.lib.dks_kernel_launches(self._ctx, C.byref(v)))
        return int(v.value)

    def last_timings_ms(self):
        out = np.zeros(3, dtype=np.float32)
        _cabi.check(self.lib.dks_last_timings(self._ctx, _cabi.ptr(out)))
        return {"prepare": float(out[0]), "coalitions": float(out[1]), "total": float(out[2])}

    def debug_scores(self, X, instance, nsamples="auto"):
        """Raw accumulator tile of the tcgen05 kernel for one instance: float32 [S_cap, Npad] of scaled masked scores
        ``-kappa*log2(e) * score(s, j)`` (tests only)."""
        _cabi.check(self.lib.dks_debug_score_dump(self._ctx, int(instance)))
        try:
            self.shap_values(X, nsamples=nsamples, l1_reg=False)
            buf = np.zeros(1 << 22, dtype=np.float32)
            rows, cols = C.c_int(0), C.c_int(0)
            _cabi.check(self.lib.dks_debug_get_scores(self._ctx, _cabi.ptr(buf), buf.size, C.byref(rows), C.byref(cols)))
        finally:
            _cabi.check(self.lib.dks_debug_score_dump(self._ctx, -1))
        return buf[:rows.value * cols.value].reshape(rows.value, cols.value).copy()

    def debug_timeline(self, X, nsamples="auto"):
        """clock64 timeline [6, 256] of CTA 0 of the tcgen05 kernel (see ``dks_debug_get_timeline``); tests/tuning only."""
        self.shap_values(X, nsamples=nsamples, l1_reg=False)          # plans uploaded, steady state
        _cabi.check(self.lib.dks_debug_score_dump(self._ctx, 0))
        try:
            self.shap_values(X, nsamples=nsamples, l1_reg=False)
            buf = np.zeros((6, 256), dtype=np.float32)
            _cabi.check(self.lib.dks_debug_get_timeline(self._ctx, _cabi.ptr(buf)))
        finally:
            _cabi.check(self.lib.dks_debug_score_dump(self._ctx, -1))
        return buf

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.dks_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # pragma: no cover
            pass
