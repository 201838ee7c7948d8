"""
Attribute-only stand-ins for the GPflow objects the path reads (GPflow 2.2.1 is not installable in this image).  They
carry NO arithmetic: class names and attribute names are GPflow's, so `t_SVGP` treats them exactly like the real objects.
"""
import numpy as np


class SquaredExponential:
    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = float(variance)
        self.lengthscales = np.asarray(lengthscales, dtype=np.float64)


RBF = SquaredExponential


class Matern52:
    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = float(variance)
        self.lengthscales = np.asarray(lengthscales, dtype=np.float64)


class Matern12:
    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = float(variance)
        self.lengthscales = np.asarray(lengthscales, dtype=np.float64)


class Matern32:
    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = float(variance)
        self.lengthscales = np.asarray(lengthscales, dtype=np.float64)


class SharedIndependent:
    """gpflow.kernels.SharedIndependent(kernel, output_dim): one kernel for every latent GP."""

    def __init__(self, kernel, output_dim):
        self.kernel = kernel
        self.output_dim = int(output_dim)


class SeparateIndependent:
    """gpflow.kernels.SeparateIndependent(kernels): one kernel per latent GP."""

    def __init__(self, kernels):
        self.kernels = list(kernels)


class Gaussian:
    def __init__(self, variance=1.0):
        self.variance = float(variance)


class Bernoulli:
    pass


class StudentT:
    def __init__(self, scale=1.0, df=3.0):
        self.scale = float(scale)
        self.df = float(df)


class Softmax:
    """gpflow.likelihoods.Softmax(num_classes): a MonteCarloLikelihood with num_monte_carlo_points = 100."""

    def __init__(self, num_classes, num_monte_carlo_points=100):
        self.num_classes = int(num_classes)
        self.num_monte_carlo_points = int(num_monte_carlo_points)


class Normal:
    """tfp.distributions.Normal: only the class name is read."""


class Exp:
    """tfp.bijectors.Exp: only the class name is read."""


class Softplus:
    """tfp.bijectors.Softplus: only the class name is read."""


class NDiagGHQuadrature:
    def __init__(self, dim, n_gh):
        self.dim = int(dim)
        self.n_gh = int(n_gh)


class HeteroskedasticTFPConditional:
    """gpflow.likelihoods.HeteroskedasticTFPConditional(distribution_class, scale_transform): two latent GPs, loc and
    scale = scale_transform(f_1); quadrature NDiagGHQuadrature(latent_dim, num_gauss_hermite_points)."""

    def __init__(self, distribution_class=Normal, scale_transform=None, num_gauss_hermite_points=20):
        self.distribution_class = distribution_class
        self.scale_transform = Exp() if scale_transform is None else scale_transform
        self.latent_dim = 2
        self.quadrature = NDiagGHQuadrature(self.latent_dim, num_gauss_hermite_points)


class InducingPoints:
    def __init__(self, Z):
        self.Z = np.array(Z, dtype=np.float64)

    @property
    def num_inducing(self):
        return self.Z.shape[0]


class SharedIndependentInducingVariables:
    """gpflow.inducing_variables.SharedIndependentInducingVariables(InducingPoints(Z)): `.inducing_variables[0].Z` is what
    the reference reads (src/models/tsvgp.py:249-254)."""

    def __init__(self, inducing_variable):
        self.inducing_variables = [inducing_variable]
