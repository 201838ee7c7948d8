"""
Variational EM around the B200 path, as the reference's callers run it (experiments/uci_regression.py:112-146,
docs/notebooks/mnist.py:161-189): per iteration `n_e_steps` natural-gradient steps on the sites (E-step, `natgrad_step`), then
`n_m_steps` Adam steps on the hyperparameters with the sites held fixed (M-step).  The reference differentiates `-elbo` with
TensorFlow through GPflow's softplus-constrained Parameters; here the gradient comes from `t_SVGP.elbo_and_grad` (constrained
values) and is chained through a log transform: d/d log(theta) = theta * d/d theta.
"""
import numpy as np

from .model import _value


def _assign(obj, name, value):
    cur = getattr(obj, name)
    if hasattr(cur, "assign"):           # gpflow.Parameter / tf.Variable
        cur.assign(value)
    else:
        setattr(obj, name, value if np.ndim(value) else float(value))


class _Adam:
    def __init__(self, lr, b1=0.9, b2=0.999, eps=1e-8):
        self.lr, self.b1, self.b2, self.eps, self.t, self.m, self.v = lr, b1, b2, eps, 0, {}, {}

    def step(self, name, x, grad):      # ascent on the ELBO
        g = np.asarray(grad, dtype=np.float64)
        m = self.m[name] = self.b1 * self.m.get(name, 0.0) + (1 - self.b1) * g
        v = self.v[name] = self.b2 * self.v.get(name, 0.0) + (1 - self.b2) * g * g
        mh, vh = m / (1 - self.b1 ** self.t), v / (1 - self.b2 ** self.t)
        return x + self.lr * mh / (np.sqrt(vh) + self.eps)


def fit(model, data, n_iters=10, n_e_steps=8, n_m_steps=20, lr_natgrad=1.0, lr_adam=0.1, train_Z=False, callback=None):
    """Run variational EM on `data = (X, Y)` (kept resident on the GPU).  Mutates model.kernel (the wrapped kernel of a
    SharedIndependent) / model.likelihood
    (and model.inducing_variable when train_Z) in place; returns the ELBO trace (one value per M-step evaluation)."""
    if type(model.kernel).__name__ == "SeparateIndependent":
        raise NotImplementedError("vem.fit with SeparateIndependent kernels: elbo_and_grad is not built for them")
    kernel = model.kernel.kernel if type(model.kernel).__name__ == "SharedIndependent" else model.kernel   # the shared kernel
    model.set_data(data)
    adam = _Adam(lr_adam)
    lik_name = type(model.likelihood).__name__
    lik_attr = {"Gaussian": "variance", "StudentT": "scale"}.get(lik_name)
    trace = []
    for it in range(n_iters):
        for _ in range(n_e_steps):                                   # E-step: uci_regression.py:120-122
            model.natgrad_step(lr=lr_natgrad)
        for _ in range(n_m_steps):                                   # M-step: uci_regression.py:124-126 (Adam on -elbo)
            elbo, g = model.elbo_and_grad()
            trace.append(elbo)
            adam.t += 1
            var = float(_value(kernel.variance))
            ls = _value(kernel.lengthscales)
            _assign(kernel, "variance", float(np.exp(adam.step("log_var", np.log(var), var * g["variance"]))))
            new_ls = np.exp(adam.step("log_ls", np.log(ls), ls * np.reshape(g["lengthscales"], np.shape(ls))))
            _assign(kernel, "lengthscales", new_ls if np.ndim(ls) else float(new_ls))
            if lik_attr is not None:
                th = float(_value(getattr(model.likelihood, lik_attr)))
                _assign(model.likelihood, lik_attr, float(np.exp(adam.step("log_lik", np.log(th), th * g["likelihood"]))))
            if train_Z:
                iv = model.inducing_variable
                Z = _value(iv.Z if hasattr(iv, "Z") else iv)
                Znew = adam.step("Z", Z, g["Z"])
                if hasattr(iv, "Z"):
                    _assign(iv, "Z", Znew)
                else:
                    model.inducing_variable = Znew
        if callback is not None:
            callback(it, trace[-1] if trace else None, model)
    return trace
