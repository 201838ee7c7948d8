"""
Host-side mirror of the reference's `t_SVGP` (reference src/models/tsvgp.py:117-304) for the one hot path this package
implements: `natgrad_step`, `elbo`, `predict_f` over `DenseSites (lambda_1, lambda_2_sqrt)`.

The GPflow kernel, likelihood and inducing-variable objects are used unchanged: only the attributes the reference path
reads are touched (duck-typed; `.numpy()` is honoured):
    kernel      SquaredExponential / RBF / Matern12 / Matern32 / Matern52 : .variance, .lengthscales (scalar, [D] or [1, D]);
                SharedIndependent (.kernel, .output_dim) ; SeparateIndependent (.kernels, one per latent)
    likelihood  Gaussian (.variance) | Bernoulli (inv_probit link) | StudentT (.scale, .df)   [+ .num_gauss_hermite_points]
                | Softmax | HeteroskedasticTFPConditional (distribution_class Normal, scale_transform Exp / Softplus)
    inducing    InducingPoints (.Z) or an ndarray [M, D]
    mean_function  None / Zero, or a callable evaluated on the host
All arithmetic runs in libtsvgp.so on the GPU (float64); tensors cross through DLPack + ctypes.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_tensor

DEFAULT_N_GH = 20  # gpflow.likelihoods.ScalarLikelihood default (GPflow 2.2.1)


def _value(p):
    if hasattr(p, "numpy"):
        p = p.numpy()
    return np.asarray(p, dtype=np.float64)


def _kernel_spec(kernel, num_latent_gps=None):
    """(kind, variance, lengthscales) of one kernel; a list of them, one per latent, for SeparateIndependent."""
    name = type(kernel).__name__
    if name == "SharedIndependent":   # gpflow.kernels.SharedIndependent(kernel, output_dim): one kernel for every latent
        if num_latent_gps is not None and int(kernel.output_dim) != int(num_latent_gps):
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, f"SharedIndependent output_dim {kernel.output_dim} != num_latent_gps {num_latent_gps}")
        return _kernel_spec(kernel.kernel)
    if name == "SeparateIndependent":   # gpflow.kernels.SeparateIndependent(kernels): one kernel per latent
        specs = [_kernel_spec(k) for k in kernel.kernels]
        if num_latent_gps is not None and len(specs) != int(num_latent_gps):
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, f"SeparateIndependent has {len(specs)} kernels, num_latent_gps is {num_latent_gps}")
        return specs
    if name in ("SquaredExponential", "RBF"):
        kind = _lib.KERNEL_SE
    elif name == "Matern52":
        kind = _lib.KERNEL_MATERN52
    elif name == "Matern32":
        kind = _lib.KERNEL_MATERN32
    elif name == "Matern12":
        kind = _lib.KERNEL_MATERN12
    else:
        raise NotImplementedError(f"kernel {name}: the B200 path implements SquaredExponential, Matern12, Matern32 and Matern52")
    active = getattr(kernel, "active_dims", None)
    if active is not None and not (isinstance(active, slice) and active == slice(None, None, None)):
        raise NotImplementedError("active_dims other than all dimensions")
    ls = np.atleast_1d(_value(kernel.lengthscales)).reshape(-1)
    return kind, float(_value(kernel.variance)), ls


def _likelihood_spec(lik):
    name = type(lik).__name__
    n_gh = int(getattr(lik, "num_gauss_hermite_points", DEFAULT_N_GH))
    if name == "Gaussian":
        return _lib.LIK_GAUSSIAN, float(_value(lik.variance)), 0.0, 0
    if name == "Bernoulli":
        link = getattr(lik, "invlink", None)
        if link is not None and getattr(link, "__name__", "inv_probit") != "inv_probit":
            raise NotImplementedError("Bernoulli: only the inv_probit link is implemented")
        return _lib.LIK_BERNOULLI_PROBIT, 0.0, 0.0, n_gh
    if name == "StudentT":
        return _lib.LIK_STUDENT_T, float(_value(lik.scale)), float(_value(lik.df)), n_gh
    if name == "Softmax":   # gpflow.likelihoods.Softmax(num_classes): MonteCarloLikelihood, num_monte_carlo_points = 100
        return _lib.LIK_SOFTMAX, float(lik.num_classes), 0.0, int(getattr(lik, "num_monte_carlo_points", 100))
    if name == "HeteroskedasticTFPConditional":   # 2 latents (loc, scale), NDiagGHQuadrature(2, n_gh)
        dist = getattr(getattr(lik, "distribution_class", None), "__name__", None)
        transform = type(getattr(lik, "scale_transform", None)).__name__
        if dist != "Normal":
            raise NotImplementedError(f"HeteroskedasticTFPConditional: distribution_class {dist}; the B200 path implements Normal")
        if transform not in ("Exp", "Softplus"):
            raise NotImplementedError(f"HeteroskedasticTFPConditional: scale_transform {transform}; the B200 path implements Exp and Softplus")
        return _lib.LIK_HETEROSKEDASTIC, 0.0 if transform == "Exp" else 1.0, 0.0, _n_gh(lik)
    raise NotImplementedError(f"likelihood {name}: the B200 path implements Gaussian, Bernoulli (probit), StudentT, Softmax and "
                              "HeteroskedasticTFPConditional")


def _n_gh(lik):
    """Gauss-Hermite points per axis: likelihood.quadrature.n_gh, else num_gauss_hermite_points, else GPflow's default 20."""
    q = getattr(lik, "quadrature", None)
    if q is not None and hasattr(q, "n_gh"):
        return int(q.n_gh)
    return int(getattr(lik, "num_gauss_hermite_points", DEFAULT_N_GH))


def _coupled(lik):
    """The likelihood couples the latents of a point: Y is [N, 1] whatever num_latent_gps is."""
    return type(lik).__name__ in ("Softmax", "HeteroskedasticTFPConditional")


def _separate(kernel):
    return type(kernel).__name__ == "SeparateIndependent"


class DenseSites:
    """reference src/sites.py:43-80 — a view of the device-resident sites of one model."""

    def __init__(self, model):
        self._model = model

    @property
    def lambda_1(self):
        return self._model.lambda_1

    @property
    def lambda_2_sqrt(self):
        return self._model.lambda_2_sqrt

    @property
    def lambda_2(self):
        return self._model.lambda_2


class t_SVGP:
    """Drop-in for the reference `t_SVGP` on the natgrad / elbo / predict_f path.

    `num_latent_gps = L > 1` (shared kernel and inducing points, one site pair per latent; reference tsvgp.py:276-281, its
    Bernoulli fixture with L = 2 at tests/models/test_tsvgp.py:45-88, the Softmax classifier of docs/notebooks/mnist.py:117-122)
    lives in ONE device context: one Kuu / Kuu + jitter I chain and one Kuf slab per launch serve all latents, the variance
    product, the weighted SYRK and the site update run per latent.  `Y` is [N, L] for likelihoods whose terms are independent
    over the latent axis (Gaussian, Bernoulli, StudentT) and [N, 1] class labels for `Softmax`."""

    def __init__(self, kernel, likelihood, inducing_variable, *, mean_function=None, num_latent_gps=1, lambda_1=None,
                 lambda_2_sqrt=None, num_data=None, force=False, device=0):
        self._lib = _lib.load()
        self.kernel = kernel
        self.likelihood = likelihood
        self.inducing_variable = inducing_variable
        self.mean_function = mean_function
        self.num_data = num_data
        self.whiten = False
        self.force = force
        self.name = "t_svgp"
        if lambda_2_sqrt is not None:
            lambda_2_sqrt = np.asarray(lambda_2_sqrt, dtype=np.float64)
            assert lambda_2_sqrt.ndim == 3  # tsvgp.py:182
            num_latent_gps = lambda_2_sqrt.shape[0]
        self.num_latent_gps = L = int(num_latent_gps)
        if L > 1 and mean_function is not None and type(mean_function).__name__ != "Zero":
            raise NotImplementedError("mean_function with num_latent_gps > 1")
        ctx = C.c_void_p()
        rc = self._lib.tsvgp_create(C.byref(ctx), int(device))
        if rc != _lib.OK:
            msg = self._lib.tsvgp_last_error(None)
            raise _lib.TsvgpError(rc, msg.decode() if msg else "tsvgp_create failed")
        self._ctx = ctx
        self.world_size, self.rank = 1, 0
        self._kernel_key = self._lik_key = self._z_key = None
        self._resident = None  # (N_local, keepalive) of the data set by set_data
        if L > 1:
            self._check(self._lib.tsvgp_set_num_latent(self._ctx, L))
        self._sync_objects()
        if lambda_1 is not None or lambda_2_sqrt is not None:
            self.assign_sites(lambda_1, lambda_2_sqrt)

    # ---- lifetime ------------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.tsvgp_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        _lib.raise_for(self._lib, self._ctx, rc)

    def set_option(self, name, value):
        self._check(self._lib.tsvgp_set_option(self._ctx, name.encode(), float(value)))

    # ---- model objects -> device (re-read on every call: GPflow parameters are mutable) ---------------------------
    def _Z(self):
        iv = self.inducing_variable
        if hasattr(iv, "inducing_variables"):   # SharedIndependentInducingVariables: one Z shared by the L latents (tsvgp.py:249-254)
            iv = iv.inducing_variables[0]
        return _value(iv.Z if hasattr(iv, "Z") else iv)

    def _mean_fn(self, X):
        mf = self.mean_function
        if mf is None or type(mf).__name__ == "Zero":
            return None
        return np.ascontiguousarray(_value(mf(X)).reshape(X.shape[0], -1)[:, 0])

    def _sync_objects(self):
        spec = _kernel_spec(self.kernel, self.num_latent_gps)
        if isinstance(spec, list):   # one kernel per latent: the key holds every latent's parameters
            key = tuple((kind, var, ls.tobytes()) for kind, var, ls in spec)
            if key != self._kernel_key:
                kinds = np.array([k for k, _, _ in spec], dtype=np.int32)
                var = np.array([v for _, v, _ in spec], dtype=np.float64)
                ls = np.ascontiguousarray(np.concatenate([l for _, _, l in spec]), dtype=np.float64)
                nls = np.array([l.size for _, _, l in spec], dtype=np.int32)
                self._check(self._lib.tsvgp_set_kernels(self._ctx, kinds.ctypes.data, var.ctypes.data_as(_lib._dp),
                                                        ls.ctypes.data_as(_lib._dp), nls.ctypes.data))
                self._kernel_key = key
        else:
            kind, var, ls = spec
            key = (kind, var, ls.tobytes())
            if key != self._kernel_key:
                self._check(self._lib.tsvgp_set_kernel(self._ctx, kind, var, ls.ctypes.data_as(_lib._dp), ls.size))
                self._kernel_key = key
        lk = _likelihood_spec(self.likelihood)
        if lk != self._lik_key:
            gx = gw = None
            if lk[3] > 0:
                x, w = np.polynomial.hermite.hermgauss(lk[3])
                gx, gw = x.ctypes.data_as(_lib._dp), w.ctypes.data_as(_lib._dp)
            self._check(self._lib.tsvgp_set_likelihood(self._ctx, lk[0], lk[1], lk[2], lk[3], gx, gw))
            self._lik_key = lk
        Z = np.ascontiguousarray(self._Z())
        if Z.ndim != 2:
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, "inducing inputs must be [M, D]")
        mz = self._mean_fn(Z)
        zkey = (Z.shape, Z.tobytes(), None if mz is None else mz.tobytes())
        if zkey != self._z_key:
            self._check(self._lib.tsvgp_set_inducing(self._ctx, Z.ctypes.data, Z.shape[0], Z.shape[1], None if mz is None else mz.ctypes.data))
            self._z_key = zkey
        self._M, self._D = Z.shape

    @property
    def num_inducing(self):
        return self._M

    # ---- DenseSites state (sites.py:43-80; tsvgp.py:187-200) --------------------------------------------------------
    @property
    def sites(self):
        return DenseSites(self)

    @property
    def lambda_1(self):
        out = np.empty((self._M, self.num_latent_gps))
        self._check(self._lib.tsvgp_get_sites(self._ctx, out.ctypes.data, None))
        return out

    @property
    def lambda_2_sqrt(self):
        out = np.empty((self.num_latent_gps, self._M, self._M))
        self._check(self._lib.tsvgp_get_sites(self._ctx, None, out.ctypes.data))
        return out

    @property
    def lambda_2(self):
        out = np.empty((self.num_latent_gps, self._M, self._M))
        self._check(self._lib.tsvgp_get_lambda_2(self._ctx, out.ctypes.data))
        return out

    def assign_sites(self, lambda_1=None, lambda_2_sqrt=None):
        """`lambda_1.assign(...)` / `lambda_2_sqrt.assign(...)` of the reference (tsvgp.py:302-303): [M, L] and [L, M, M]."""
        L = self.num_latent_gps
        l1 = l2 = None
        if lambda_1 is not None:
            l1 = np.ascontiguousarray(np.asarray(lambda_1, dtype=np.float64).reshape(-1, L))
            if l1.shape[0] != self._M:
                raise _lib.InvalidArgumentError(_lib.ERR_INVALID, f"lambda_1 must be [{self._M}, {L}]")
        if lambda_2_sqrt is not None:
            l2 = np.ascontiguousarray(np.asarray(lambda_2_sqrt, dtype=np.float64).reshape(-1, self._M, self._M))
            if l2.shape[0] != L:
                raise _lib.InvalidArgumentError(_lib.ERR_INVALID, f"lambda_2_sqrt must be [{L}, {self._M}, {self._M}]")
        self._check(self._lib.tsvgp_set_sites(self._ctx, None if l1 is None else l1.ctypes.data, None if l2 is None else l2.ctypes.data))

    def get_mean_chol_cov_inducing_posterior(self):
        """tsvgp.py:202-212 -> (m_q [M, 1], chol_S [1, M, M])."""
        self._sync_objects()
        m = np.empty((self._M, self.num_latent_gps))
        cs = np.empty((self.num_latent_gps, self._M, self._M))
        self._check(self._lib.tsvgp_posterior(self._ctx, m.ctypes.data, cs.ctypes.data))
        return m, cs

    # ---- data -----------------------------------------------------------------------------------------------------
    def set_data(self, data):
        """Make (X [N, D], Y [N, 1]) — this rank's rows of the minibatch — resident on the GPU.  Host arrays are copied
        (H2D); device tensors (DLPack) are aliased and must stay alive and unchanged until the next set_data."""
        X, Y = data
        tx, ty = as_tensor(X, "X", self), as_tensor(Y, "Y", self)
        if len(tx.shape) != 2:
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, "X must be [N, D]")
        N, D = tx.shape
        ny = int(np.prod(ty.shape))
        ycols = 1 if _coupled(self.likelihood) else self.num_latent_gps
        if ny != N * ycols:
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, f"Y must be [N, {ycols}] with N = {N}, got {ty.shape}")
        mean_x = None
        if self._mean_fn(np.zeros((1, D))) is not None:
            if tx.on_device:
                raise NotImplementedError("a non-zero mean_function needs host-resident X")
            mean_x = self._mean_fn(np.asarray(X, dtype=np.float64))
        self._check(self._lib.tsvgp_set_data(self._ctx, tx.ptr, ty.ptr, N, D, None if mean_x is None else mean_x.ctypes.data))
        self._resident = (N, (tx, ty, mean_x))
        return N

    def stage_data(self, data):
        if self.num_latent_gps > 1 and not _coupled(self.likelihood):
            raise NotImplementedError("stage_data with num_latent_gps > 1: use set_data")
        """Start copying the NEXT minibatch to the GPU on a copy stream while the current step computes (use pinned host
        arrays, `tsvgp_b200.pinned_empty`, for a truly asynchronous copy); `commit_staged()` makes it resident."""
        X, Y = data
        tx, ty = as_tensor(X, "X", self), as_tensor(Y, "Y", self)
        N, D = tx.shape
        if int(np.prod(ty.shape)) != N:
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, "Y must be [N, 1]")
        if self._mean_fn(np.zeros((1, D))) is not None:
            raise NotImplementedError("stage_data with a non-zero mean_function")
        self._check(self._lib.tsvgp_stage_data(self._ctx, tx.ptr, ty.ptr, N, D, None))
        self._staged = (N, (tx, ty))
        return N

    def commit_staged(self):
        self._check(self._lib.tsvgp_commit_staged(self._ctx))
        self._resident = (self._staged[0], self._staged[1] + (None,))
        self._staged = None
        return self._resident[0]

    def _scale(self, n_local, global_minibatch_size):
        n = n_local if global_minibatch_size is None else int(global_minibatch_size)
        if global_minibatch_size is None and self.world_size > 1:
            raise ValueError("sharded over ranks: pass global_minibatch_size (rows summed over all ranks)")
        return float(self.num_data) / float(n) if self.num_data is not None else 1.0  # tsvgp.py:89-94, 286-291

    def _ingest(self, data):
        if data is not None:
            return self.set_data(data)
        if self._resident is None:
            raise _lib.TsvgpError(_lib.ERR_STATE, "no data: pass data=(X, Y) or call set_data first")
        return self._resident[0]

    # ---- the path ---------------------------------------------------------------------------------------------------
    def natgrad_step(self, data=None, lr=0.1, jitter=1e-9, *, global_minibatch_size=None, return_elbo=False):
        """tsvgp.py:234-304.  Mutates lambda_1 / lambda_2_sqrt (on the device).  `data=None` reuses the resident data.
        Raises NonPositiveVarianceError, sites unchanged, when a predictive variance of the minibatch is not positive.  The
        Gaussian update does not read the variances and forms none per point: it raises when a point of X or its predictive mean is
        not finite and, with return_elbo, when the sum of the variances (from the step's statistics) is not positive."""
        self._sync_objects()
        n = self._ingest(data)
        out = C.c_double()
        self._check(self._lib.tsvgp_natgrad_step(self._ctx, float(lr), float(jitter), self._scale(n, global_minibatch_size),
                                                 C.byref(out) if return_elbo else None))
        return out.value if return_elbo else None

    def elbo(self, data=None, *, global_minibatch_size=None):
        """tsvgp.py:79-95."""
        self._sync_objects()
        n = self._ingest(data)
        out = C.c_double()
        self._check(self._lib.tsvgp_elbo(self._ctx, self._scale(n, global_minibatch_size), C.byref(out)))
        return out.value

    def elbo_and_grad(self, data=None, *, global_minibatch_size=None):
        """M-step objective and its gradient with the sites held fixed (what the reference gets from TensorFlow autodiff of
        `elbo` / `training_loss_closure`; tsvgp.py:72-95, tests/models/test_tsvgp.py:168-188).
        -> (elbo, {"variance", "lengthscales" (shape of kernel.lengthscales), "Z" [M, D], "likelihood"}), gradients w.r.t. the
        constrained parameter values (chain your own positive transform); "likelihood" is d/d variance (Gaussian),
        d/d scale (StudentT) or None (Bernoulli, Softmax).  Softmax: one Monte-Carlo draw per call, the one `elbo` would use
        next (or the draws fixed by `set_mc_epsilon`)."""
        if _separate(self.kernel):
            raise NotImplementedError("elbo_and_grad with SeparateIndependent kernels")
        if type(self.likelihood).__name__ == "HeteroskedasticTFPConditional":
            raise NotImplementedError("elbo_and_grad with the heteroskedastic likelihood")
        self._sync_objects()
        if self._mean_fn(np.zeros((1, self._D))) is not None:
            raise NotImplementedError("elbo_and_grad with a non-zero mean_function")
        n = self._ingest(data)
        kernel = self.kernel.kernel if type(self.kernel).__name__ == "SharedIndependent" else self.kernel
        kind, _, ls = _kernel_spec(kernel)
        e, dv, dl = C.c_double(), C.c_double(), C.c_double()
        dls, dZ = np.empty(ls.size), np.empty((self._M, self._D))
        self._check(self._lib.tsvgp_elbo_grad(self._ctx, self._scale(n, global_minibatch_size), C.byref(e), C.byref(dv),
                                              dls.ctypes.data, dZ.ctypes.data, C.byref(dl)))
        lik = _likelihood_spec(self.likelihood)[0]
        return e.value, {"variance": dv.value, "lengthscales": dls.reshape(np.shape(_value(kernel.lengthscales)) or ()),
                         "Z": dZ, "likelihood": None if lik in (_lib.LIK_BERNOULLI_PROBIT, _lib.LIK_SOFTMAX) else dl.value}

    def maximum_log_likelihood_objective(self, data=None):  # tsvgp.py:72-77
        return self.elbo(data)

    def training_loss(self, data=None):
        return -self.elbo(data)

    def prior_kl(self):
        """tsvgp.py:65-70."""
        self._sync_objects()
        out = C.c_double()
        self._check(self._lib.tsvgp_prior_kl(self._ctx, C.byref(out)))
        return out.value

    def _query(self, Xnew):
        """Xnew [N, D] (host array or DLPack device tensor, aliased) -> (tensor, N, D, mean_function(Xnew) [N] or None)."""
        self._sync_objects()
        tx = as_tensor(Xnew, "Xnew", self)
        if len(tx.shape) != 2:
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, "Xnew must be [N, D]")
        N, D = tx.shape
        mean_x = None
        if self._mean_fn(np.zeros((1, D))) is not None:
            mean_x = self._mean_fn(np.asarray(Xnew, dtype=np.float64))
        return tx, N, D, mean_x

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        """tsvgp.py:97-114 -> (mean [N, L], var [N, L]); raises if any variance is <= 0 (:113).
        full_cov=True -> (mean [N, L], cov [L, N, N]), GPflow's layouts; only the diagonal of cov is checked for positivity."""
        if full_output_cov:
            raise NotImplementedError("full_output_cov: never exercised on this path by the reference")
        tx, N, D, mean_x = self._query(Xnew)
        L = self.num_latent_gps
        mx = None if mean_x is None else mean_x.ctypes.data
        if full_cov:
            if N == 0:
                return np.empty((0, L)), np.empty((L, 0, 0))
            mean, cov = np.empty((N, L)), np.empty((L, N, N))
            self._check(self._lib.tsvgp_predict_f_full_cov(self._ctx, tx.ptr, N, D, mx, mean.ctypes.data, cov.ctypes.data))
            return mean, cov
        if N == 0:   # an empty query returns empty moments, as the reference's conditional does
            return np.empty((0, L)), np.empty((0, L))
        mean, var = np.empty((N, L)), np.empty((N, L))
        self._check(self._lib.tsvgp_predict_f(self._ctx, tx.ptr, N, D, mx, mean.ctypes.data, var.ctypes.data))
        return mean, var

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, *, epsilon=None):
        """GPModel.predict_f_samples -> [S, N, L], or [N, L] when num_samples is None.
        full_cov=True: mean + chol(cov_l + 1e-6 I) eps per latent (gpflow sample_mvn); False: mean + sqrt(var) eps.
        `epsilon [S, N, L]` fixes the standard-normal draws (as `set_mc_epsilon` does for Softmax); otherwise they come from the
        library's Philox generator, option "sample_seed", a new draw per call."""
        if full_output_cov:
            raise NotImplementedError("full_output_cov: never exercised on this path by the reference")
        tx, N, D, mean_x = self._query(Xnew)
        L = self.num_latent_gps
        S = 1 if num_samples is None else int(num_samples)
        if S < 1:
            raise _lib.InvalidArgumentError(_lib.ERR_INVALID, "num_samples must be >= 1")
        eps = None
        if epsilon is not None:
            eps = as_tensor(epsilon, "epsilon", self)
            if tuple(eps.shape) != (S, N, L):
                raise _lib.InvalidArgumentError(_lib.ERR_INVALID, f"epsilon must be [{S}, {N}, {L}], got {tuple(eps.shape)}")
        out = np.empty((S, N, L))
        if N > 0:
            self._check(self._lib.tsvgp_predict_f_samples(self._ctx, tx.ptr, N, D, None if mean_x is None else mean_x.ctypes.data,
                                                          S, int(bool(full_cov)), None if eps is None else eps.ptr, out.ctypes.data))
        return out[0] if num_samples is None else out

    def set_mc_epsilon(self, epsilon):
        """Softmax likelihood: fix the Monte-Carlo draws to `epsilon [S, N, L]` (GPflow's `epsilon` argument of
        MonteCarloLikelihood.variational_expectations) for every pass over exactly N points; None returns to the generator."""
        if epsilon is None:
            self._check(self._lib.tsvgp_set_mc_epsilon(self._ctx, None, 0, 0, 0))
            return
        self._sync_objects()
        e = np.ascontiguousarray(epsilon, dtype=np.float64)
        S, N, L = e.shape
        self._check(self._lib.tsvgp_set_mc_epsilon(self._ctx, e.ctypes.data, S, N, L))

    # ---- inherited GPModel surface built on predict_f (used by the reference's callers: experiments/uci_regression.py:114,142,
    # 145,251).  O(N) host arithmetic on the GPU's predict_f output; GPflow 2.2.1 likelihood semantics [GPflow-recalled]:
    # Gaussian closed forms; Bernoulli(inv_probit) analytic mean; Student-t / generic via 20-point Gauss-Hermite. -------------
    def _gh(self):
        x, w = np.polynomial.hermite.hermgauss(_n_gh(self.likelihood))
        return x * np.sqrt(2.0), w / np.sqrt(np.pi)

    def _hetero_grid(self, Xnew):
        """HeteroskedasticTFPConditional: predict_f's marginals on the NDiagGHQuadrature grid -> (loc F0 [N, n, 1],
        scale T(F1) [N, 1, n], log weights [1, n, n]) over the n x n nodes."""
        mu, var = self.predict_f(Xnew)
        z, w = self._gh()
        F0 = (mu[:, 0:1] + np.sqrt(var[:, 0:1]) * z)[:, :, None]
        F1 = (mu[:, 1:2] + np.sqrt(var[:, 1:2]) * z)[:, None, :]
        scale = np.exp(F1) if type(self.likelihood.scale_transform).__name__ == "Exp" else np.logaddexp(0.0, F1)
        return F0, scale, np.log(w)[None, :, None] + np.log(w)[None, None, :]

    def predict_y(self, Xnew, full_cov=False, full_output_cov=False):
        """GPModel.predict_y -> likelihood.predict_mean_and_var(f_mean, f_var)."""
        from math import erf
        if full_cov or full_output_cov:   # as GPflow 2.2.1's likelihoods: only the marginals are propagated
            raise NotImplementedError("predict_y with full_cov / full_output_cov")
        name = type(self.likelihood).__name__
        if name == "HeteroskedasticTFPConditional":   # QuadratureLikelihood: E[loc], E[scale^2 + loc^2] - E[loc]^2  -> [N, 1]
            F0, scale, logw = self._hetero_grid(Xnew)
            W = np.exp(logw)
            Ey = np.sum(W * F0, axis=(1, 2))
            Ey2 = np.sum(W * (np.square(scale) + np.square(F0)), axis=(1, 2))
            return Ey[:, None], (Ey2 - np.square(Ey))[:, None]
        mu, var = self.predict_f(Xnew)
        if name == "Gaussian":
            return mu, var + float(_value(self.likelihood.variance))
        if name == "Bernoulli":
            p = 0.5 * (1.0 + np.vectorize(erf)(mu / np.sqrt(1.0 + var) / np.sqrt(2.0))) * (1 - 2e-3) + 1e-3
            return p, p - np.square(p)
        sc, df = float(_value(self.likelihood.scale)), float(_value(self.likelihood.df))   # StudentT: E[y|f] = f, Var[y|f] = scale^2 df/(df-2)
        return mu, var + sc * sc * df / (df - 2.0)

    def predict_log_density(self, data, full_cov=False, full_output_cov=False):
        """GPModel.predict_log_density -> log int p(y | f) q(f) df per point, [N]."""
        from math import lgamma
        if full_cov or full_output_cov:
            raise NotImplementedError("predict_log_density with full_cov / full_output_cov")
        X, Y = data
        Y = np.asarray(Y, dtype=np.float64)
        name = type(self.likelihood).__name__
        if name == "HeteroskedasticTFPConditional":   # log sum_ij w_i w_j Normal(F0_i, T(F1_j)).pdf(y)  -> [N]
            from scipy.special import logsumexp
            F0, scale, logw = self._hetero_grid(X)
            y = Y.reshape(-1, 1, 1)
            logp = -0.5 * np.log(2 * np.pi) - np.log(scale) - 0.5 * np.square((y - F0) / scale)
            return logsumexp(logp + logw, axis=(1, 2))
        mu, var = self.predict_f(X)
        if name == "Gaussian":
            v = var + float(_value(self.likelihood.variance))
            return np.sum(-0.5 * (np.log(2 * np.pi) + np.log(v) + np.square(Y - mu) / v), axis=-1)
        if name == "Bernoulli":
            p, _ = self.predict_y(X)
            return np.sum(np.log(np.where(Y == 1, p, 1 - p)), axis=-1)
        z, w = self._gh()
        sc, df = float(_value(self.likelihood.scale)), float(_value(self.likelihood.df))
        F = mu[..., None] + np.sqrt(var)[..., None] * z
        const = lgamma((df + 1) * 0.5) - lgamma(df * 0.5) - 0.5 * (np.log(sc * sc) + np.log(df) + np.log(np.pi))
        logp = const - 0.5 * (df + 1) * np.log1p(np.square((Y[..., None] - F) / sc) / df) + np.log(w)
        mx = logp.max(axis=-1, keepdims=True)
        return np.sum(mx[..., 0] + np.log(np.sum(np.exp(logp - mx), axis=-1)), axis=-1)

    def training_loss_closure(self, data=None):
        """GPModel.training_loss_closure: a zero-argument callable returning -ELBO on `data`."""
        return lambda: self.training_loss(data)

    # ---- multi-GPU: one model (context) per rank ------------------------------------------------------------------------
    def init_comm(self, world_size, rank, unique_id: bytes):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(self._lib.tsvgp_comm_init(self._ctx, int(world_size), int(rank), buf))
        self.world_size, self.rank = int(world_size), int(rank)

    def timings(self):
        """CUDA-event milliseconds of the last natgrad_step (see tsvgp_get_timings)."""
        buf = (C.c_double * 10)()
        self._check(self._lib.tsvgp_get_timings(self._ctx, buf, 10))
        keys = ["total", "prepare", "stream", "allreduce", "dense", "slabs", "launches", "route", "cond_est", "chain_role"]
        return {k: buf[i] for i, k in enumerate(keys)}

    def kernel_profile(self):
        """Per-kernel-class CUDA-event totals of the last natgrad_step run with option profile=1: {class: (ms, launches)}."""
        buf = (C.c_double * 12)()
        self._check(self._lib.tsvgp_get_kernel_profile(self._ctx, buf, 12))
        names = ["kuf", "variance_gemm", "point_stats", "whiten_gemm", "syrk", "kuf_g"]
        return {k: (buf[2 * i], int(buf[2 * i + 1])) for i, k in enumerate(names)}

    def timer_start(self):
        self._check(self._lib.tsvgp_timer_start(self._ctx))

    def timer_stop(self):
        ms = C.c_double()
        self._check(self._lib.tsvgp_timer_stop(self._ctx, C.byref(ms)))
        return ms.value

    def device_array(self, host_array):
        """Upload a host array into GPU memory owned by the returned handle (usable as X / Y in set_data)."""
        return _lib.DeviceArray(self, host_array)

    def sync(self):
        self._check(self._lib.tsvgp_sync(self._ctx))


class MultiLatent_t_SVGP(t_SVGP):
    """Kept as a name for `t_SVGP(..., num_latent_gps = L > 1)`: since round 2 the L latents live in ONE device context (see t_SVGP)."""


class t_SVGP_white(t_SVGP):
    """Drop-in for the reference's whitened sibling `t_SVGP_white` (src/models/tsvgp_white.py:23-246): sites
    t(u) with natural parameters (lambda_1, Lambda_2) in the K-scaled parameterisation, Lambda_2 a full symmetric matrix
    (`lambda_2 [1, M, M]`, default 1e-10 I), updated without any factorisation:
        lambda_1 <- (1-lr) lambda_1 + lr s K (G1 - 2 G2 mZ) ;  Lambda_2 <- (1-lr) Lambda_2 - 2 lr s K G2 K.
    Same constructor / natgrad_step / elbo / predict_f / prior_kl / get_mean_chol_cov_inducing_posterior surface
    (+ `predict_f_extra_data`; any num_latent_gps with Gaussian / Bernoulli / StudentT; `elbo_and_grad` is not built for this
    parameterisation)."""

    def __init__(self, kernel, likelihood, inducing_variable, *, mean_function=None, num_latent_gps=1, lambda_1=None,
                 lambda_2=None, num_data=None, device=0):
        if lambda_2 is not None:
            lambda_2 = np.asarray(lambda_2, dtype=np.float64)
            assert lambda_2.ndim == 3  # tsvgp_white.py:87
            num_latent_gps = lambda_2.shape[0]
        if _coupled(likelihood):
            raise NotImplementedError(f"t_SVGP_white with the {type(likelihood).__name__} likelihood")
        if _separate(kernel):
            raise NotImplementedError("t_SVGP_white with SeparateIndependent kernels")
        super().__init__(kernel, likelihood, inducing_variable, mean_function=mean_function, num_latent_gps=num_latent_gps,
                         num_data=num_data, device=device)
        self.name = "t_svgp_white"
        self.set_option("white", 1)
        if lambda_1 is not None or lambda_2 is not None:
            self.assign_sites(lambda_1, lambda_2)

    @property
    def lambda_2_sqrt(self):
        raise AttributeError("t_SVGP_white stores lambda_2 itself (src/models/tsvgp_white.py:91-97)")

    def assign_sites(self, lambda_1=None, lambda_2=None):
        """`lambda_1 [M, L]`, `lambda_2 [L, M, M]` (full symmetric matrices, tsvgp_white.py:79-89)."""
        super().assign_sites(lambda_1, lambda_2)

    def elbo_and_grad(self, data=None, *, global_minibatch_size=None):
        raise NotImplementedError("elbo_and_grad for t_SVGP_white")

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        if full_cov:   # the reference's whitened conditional computes the diagonal only (tsvgp_white.py:122-132)
            raise NotImplementedError("full_cov for t_SVGP_white")
        return super().predict_f(Xnew, full_cov, full_output_cov)

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, *, epsilon=None):
        if full_cov:
            raise NotImplementedError("full_cov for t_SVGP_white: pass full_cov=False")
        return super().predict_f_samples(Xnew, num_samples, False, full_output_cov, epsilon=epsilon)

    def natgrad_step(self, data=None, lr=0.1, jitter=1e-9, *, global_minibatch_size=None, return_elbo=False):
        """tsvgp_white.py:215-246.  The reference accepts `jitter` but never forwards it: compute_data_natural_params is called
        without it (:228) and factors Kuu + 1e-9 I whatever the caller passed — reproduced here."""
        return super().natgrad_step(data, lr, 1e-9, global_minibatch_size=global_minibatch_size, return_elbo=return_elbo)

    def predict_f_extra_data(self, Xnew, extra_data, jitter=1e-6):
        """tsvgp_white.py:134-158: predictions at Xnew after conditioning the current sites on `extra_data` (the sites themselves
        are left unchanged; `extra_data` becomes the resident minibatch)."""
        self._sync_objects()
        self.set_data(extra_data)
        tx = as_tensor(Xnew, "Xnew", self)
        N, D = tx.shape
        if self._mean_fn(np.zeros((1, D))) is not None:
            raise NotImplementedError("predict_f_extra_data with a non-zero mean_function")
        mean, var = np.empty((N, self.num_latent_gps)), np.empty((N, self.num_latent_gps))
        self._check(self._lib.tsvgp_predict_f_extra_data(self._ctx, tx.ptr, N, D, None, float(jitter), mean.ctypes.data, var.ctypes.data))
        return mean, var


def stream_minibatches(model, batches):
    """Input pipeline: iterate `batches` (an iterable of (X, Y) host arrays, ideally pinned) so that batch i + 1 is being copied
    to the GPU while the caller's loop body works on batch i.  Yields the number of rows of the now-resident minibatch:

        for n in stream_minibatches(model, loader):
            model.natgrad_step(lr=0.5)          # data=None: the resident minibatch
    """
    it = iter(batches)
    try:
        model.stage_data(next(it))
    except StopIteration:
        return
    while True:
        n = model.commit_staged()
        try:
            model.stage_data(next(it))
            more = True
        except StopIteration:
            more = False
        yield n
        if not more:
            return


def comm_unique_id() -> bytes:
    """ncclGetUniqueId — call on rank 0 and send the 128 bytes to the other ranks."""
    lib = _lib.load()
    buf = C.create_string_buffer(128)
    rc = lib.tsvgp_comm_unique_id(buf)
    if rc != _lib.OK:
        raise _lib.TsvgpError(rc, "NCCL is not available")
    return buf.raw


def shard_rows(n_rows, world_size, rank, weights=None):
    """Contiguous row ranges of the minibatch (SURVEY §8e): rank r owns rows [lo, hi).  Near-equal by default; with `weights`
    (one relative share per rank, e.g. from `balance_weights`) the inner boundaries fall on multiples of 128 rows at the
    cumulative shares."""
    n_rows, world_size = int(n_rows), int(world_size)
    if weights is None:
        base, rem = divmod(n_rows, world_size)
        lo = rank * base + min(rank, rem)
        return lo, lo + base + (1 if rank < rem else 0)
    w = np.asarray(weights, dtype=np.float64)
    if w.shape != (world_size,) or not np.all(w > 0):
        raise ValueError("weights must be one positive share per rank")
    cum = np.concatenate([[0.0], np.cumsum(w / w.sum())])
    bounds = [min(n_rows, int(round(c * n_rows / 128.0)) * 128) for c in cum]
    bounds[0], bounds[-1] = 0, n_rows
    for r in range(1, world_size + 1):          # every rank keeps at least one row
        bounds[r] = max(bounds[r], bounds[r - 1] + 1)
    if bounds[-1] != n_rows:
        raise ValueError("too few rows for this many ranks")
    return bounds[rank], bounds[rank + 1]


def balance_weights(prepare_ms, stream_ms, rows, roles, max_skew=0.1):
    """Row shares that let every rank finish its streaming pass at the same time when the ranks do different things in front of
    it (option "split_chains": rank 0 builds the posterior factors alone, rank 1 runs the K9 chain underneath early slabs, the
    others only early slabs, see DESIGN §5).  Inputs, one entry per rank, from the last step(s) with the current shares:
    timings()["prepare"], timings()["stream"], the rank's row count, timings()["chain_role"].
    Model: prepare_r + stream_r = o_r + rows_r / rate, with ONE streaming rate (rows per ms, measured on the ranks whose stream
    phase is streaming only: role 1, no early slabs) and a per-rank offset o_r (the chain in front of the pass on rank 0, next to
    nothing on the others, whose early slabs fill the wait).  The shares solve  o_r + rows_r / rate = T  for all r  with
    sum rows_r = N, and are clipped to 1 +- max_skew of the mean.  All roles 0 (no split): equal shares."""
    prep, stream, rows, roles = (np.asarray(a, dtype=np.float64) for a in (prepare_ms, stream_ms, rows, roles))
    W = rows.size
    if not np.any(roles != 0):
        return np.full(W, 1.0 / W)
    pure = roles == 1
    if not np.any(pure):
        pure = np.ones(W, dtype=bool)
    rate = np.sum(rows[pure]) / np.sum(stream[pure])
    off = prep + stream - rows / rate
    T = (np.sum(rows) / rate + np.sum(off)) / W
    new_rows = np.maximum(rate * (T - off), 1.0)
    w = new_rows / np.sum(new_rows)
    w = np.clip(w, (1.0 - max_skew) / W, (1.0 + max_skew) / W)
    return w / np.sum(w)
