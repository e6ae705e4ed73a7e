"""Named weak forms with fused CUDA kernels.

Each object is an ordinary callable with the reference's form signature
`form(basis, *args) -> integrand tensor`, so it also runs through the generic
(integrand -> quad_reduce -> scatter) path and can be checked against it.  When handed to
`integrate_bilinear_form` / `integrate_linear_form` directly, the basis dispatches to the
fused kernel instead and no integrand is materialised.

Forms covered (SURVEY.md section 8(a) row a15):
  Stiffness / Mass / StiffnessMass   examples/example_weak.py:78-81, tests/test_assembly.py:68-73
  Load(source)                       tests/test_assembly.py:79-84
  WeakResidual(source)               examples/example_weak.py:64-75, example_patches.py:102-113,
                                     example_fracture_vpinns.py:104-113
  H1Error(exact, exact_grad)         examples/example_weak.py:113-124

Coefficients: `Stiffness(kappa)`, `Mass(c)` and `StiffnessMass(kappa, c)` take numbers, callables of the quadrature
points or tensors broadcastable to `(*lead, n_q, 1, 1)` (DESIGN.md section 8(g)), so `-div(kappa grad u) + c u = f`
assembles without an integrand.  The VPINN residual of `-div(kappa grad u) = f` needs no new kernel: pass
`kappa_q * grad u_NN` as the gradient to `WeakResidual`.
"""

from __future__ import annotations

import math
from typing import Callable, Optional

import torch

from . import _lib


class Source:
    """Right-hand side f: analytic kinds are evaluated inside the kernels."""

    kind = _lib.TFEM_SRC_NONE
    params = (0.0, 0.0, 0.0, 0.0)

    def __call__(self, points: torch.Tensor) -> torch.Tensor:  # (...,d) -> (...,1)
        return torch.zeros_like(points[..., :1])


class ConstSource(Source):
    kind = _lib.TFEM_SRC_CONST

    def __init__(self, value: float = 1.0):
        self.params = (float(value), 0.0, 0.0, 0.0)

    def __call__(self, points):
        return torch.full_like(points[..., :1], self.params[0])


class SinSinSource(Source):
    """f = amplitude * sin(wx x) sin(wy y); defaults give 2 pi^2 sin(pi x) sin(pi y)."""

    kind = _lib.TFEM_SRC_SINSIN

    def __init__(self, amplitude: float = 2.0 * math.pi**2, wx: float = math.pi, wy: float = math.pi):
        self.params = (float(amplitude), float(wx), float(wy), 0.0)

    def __call__(self, points):
        a, wx, wy, _ = self.params
        return a * torch.sin(wx * points[..., 0:1]) * torch.sin(wy * points[..., 1:2])


class SampledSource(Source):
    """f given by a Python callable of the quadrature points, sampled with torch (f_q array)."""

    kind = _lib.TFEM_SRC_SAMPLED

    def __init__(self, function: Callable[[torch.Tensor], torch.Tensor]):
        self.function = function
        self._samples = None  # (key, values at a basis' quadrature points), filled by AbstractBasis._sampled_source

    def refresh(self):
        """Forget cached samples (for a callable whose values change between calls)."""
        self._samples = None

    def __call__(self, points):
        return self.function(points)


def as_source(source) -> Source:
    if source is None:
        return Source()
    if isinstance(source, Source):
        return source
    if callable(source):
        return SampledSource(source)
    return ConstSource(float(source))


def _coefficient(value):
    """A number stays a float (the constant-coefficient kernels); a tensor is kept as given; a callable of the
    quadrature points is wrapped in a `SampledSource`, whose samples the basis caches like a sampled right-hand side."""
    if isinstance(value, torch.Tensor) and value.dim() > 0:
        return value
    if callable(value):
        return SampledSource(value)
    return float(value)


def _is_zero(coefficient) -> bool:
    return isinstance(coefficient, float) and coefficient == 0.0


class FusedBilinear:
    """alpha * grad(u).grad(v) + beta * u v.

    `alpha` and `beta` each take a number, a callable of the quadrature points returning `(..., 1)` values, or a
    tensor broadcastable to `(*lead, n_q, 1, 1)` (`lead` = the basis' element batch shape: `(N, 1, 1, 1)` per element,
    `(N, n_q, 1, 1)` per quadrature point, `(F, 1, 1, 1, 1)` per fracture).  Field coefficients run on the two-pass
    path (`tfem_tri_p1_weighted_local_forms`); number coefficients keep the constant-coefficient kernels."""

    def __init__(self, alpha=0.0, beta=0.0):
        self.alpha, self.beta = _coefficient(alpha), _coefficient(beta)

    @property
    def has_field(self) -> bool:
        """True when alpha or beta is a callable or tensor field rather than a number."""
        return not (isinstance(self.alpha, float) and isinstance(self.beta, float))

    def refresh(self):
        """Forget the cached samples of callable coefficients (for callables whose values change between calls)."""
        for c in (self.alpha, self.beta):
            if isinstance(c, SampledSource):
                c.refresh()

    def __call__(self, basis):
        alpha, beta = (c(basis.integration_points) if isinstance(c, SampledSource) else c for c in (self.alpha, self.beta))
        out = None
        if not _is_zero(alpha):
            out = alpha * (basis.v_grad @ basis.v_grad.mT)
        if not _is_zero(beta):
            mass = beta * (basis.v @ basis.v.mT)
            out = mass if out is None else out + mass
        if out is None:
            out = 0.0 * (basis.v @ basis.v.mT)
        return out


class Stiffness(FusedBilinear):
    def __init__(self, alpha=1.0):
        super().__init__(alpha, 0.0)


class Mass(FusedBilinear):
    def __init__(self, beta=1.0):
        super().__init__(0.0, beta)


class StiffnessMass(FusedBilinear):
    def __init__(self, alpha=1.0, beta=1.0):
        super().__init__(alpha, beta)


class Load:
    """f(x_q) * v."""

    def __init__(self, source=None):
        self.source = as_source(source if source is not None else SinSinSource())

    def __call__(self, basis):
        return self.source(basis.integration_points) * basis.v


class WeakResidual:
    """f v - grad(v) . grad(u):  `basis.integrate_linear_form(WeakResidual(f), gradient)`.

    `gradient` is a callable evaluated at `basis.integration_points` (e.g.
    `neural_network.gradient`) or the tensor of its values `(..., N, q, 1, d)`."""

    def __init__(self, source=None):
        self.source = as_source(source if source is not None else SinSinSource())

    @staticmethod
    def field(basis, gradient) -> torch.Tensor:
        return gradient(basis.integration_points) if callable(gradient) else gradient

    def __call__(self, basis, gradient):
        grad = self.field(basis, gradient)
        return self.source(basis.integration_points) * basis.v - basis.v_grad @ grad.mT


class H1Error:
    """(u_ex - u)^2 + |grad u_ex - grad u|^2 of examples/example_weak.py:113-124:
    `basis.integrate_functional(H1Error(exact, exact_grad), neural_network, neural_network.gradient)`.

    `exact(points) -> (..., 1)` and `exact_grad(points) -> (..., d)` are sampled once per basis (the points do not
    move); `u` / `gradient` are callables of the points or tensors of their values."""

    def __init__(self, exact: Callable[[torch.Tensor], torch.Tensor], exact_grad: Callable[[torch.Tensor], torch.Tensor]):
        self.exact, self.exact_grad = exact, exact_grad
        self._samples = None

    def refresh(self):
        self._samples = None

    @staticmethod
    def field(basis, value) -> torch.Tensor:
        return value(basis.integration_points) if callable(value) else value

    def __call__(self, basis, u, gradient):
        points = basis.integration_points
        diff = self.exact(points) - self.field(basis, u)
        diff_grad = self.exact_grad(points) - self.field(basis, gradient)
        return diff**2 + (diff_grad**2).sum(-1, keepdim=True)


class Jump:
    """h_E ((grad u+ . n) + (grad u- . (-n)))^2 of examples/example_jump.py:75-87.

    `edges_basis.integrate_functional(Jump(grad_edges), n_E, h_E)` with `grad_edges` the
    `(..., N_E, 2, 1, 1, d)` tensor returned by `basis.interpolate(edges_basis, u)[1]`."""

    def __init__(self, grad_edges: Optional[torch.Tensor] = None):
        self.grad_edges = grad_edges

    def __call__(self, basis, normal, size, grad_edges=None):
        g = self.grad_edges if grad_edges is None else grad_edges
        plus, minus = torch.unbind(g, dim=-4)
        return size * ((plus * normal).sum(-1, keepdim=True) + (minus * -normal).sum(-1, keepdim=True)) ** 2
