"""Risk measures of the Bellman backup (include/sdp_b200.h, SdpRisk).

`MeanCVaR(alpha, weight)` replaces the expectation over the perturbation nodes by
`(1 - weight) * E[v] + weight * CVaR_alpha[v]`, the CVaR being the mean of the upper
`1 - alpha` tail of the node values.  Nested in every backup, it is the mean-CVaR objective
of risk-averse storage and hydro control.  `weight = 0` is the expectation.
"""
import math

from . import _cabi
from .tabulate import joint_proba

__all__ = ["MeanCVaR"]


class MeanCVaR(object):
    """Nested mean-CVaR risk measure: 0 <= alpha < 1, 0 <= weight <= 1."""
    __slots__ = ("alpha", "weight")

    def __init__(self, alpha, weight):
        alpha, weight = float(alpha), float(weight)
        if not (0.0 <= alpha < 1.0):
            raise ValueError("MeanCVaR: alpha must be in [0, 1), got %r" % alpha)
        if not (0.0 <= weight <= 1.0):
            raise ValueError("MeanCVaR: weight must be in [0, 1], got %r" % weight)
        object.__setattr__(self, "alpha", alpha)
        object.__setattr__(self, "weight", weight)

    def __setattr__(self, name, value):
        raise AttributeError("MeanCVaR is immutable")

    def __repr__(self):
        return "MeanCVaR(alpha=%r, weight=%r)" % (self.alpha, self.weight)

    def __eq__(self, other):
        return isinstance(other, MeanCVaR) and (self.alpha, self.weight) == (other.alpha, other.weight)

    def __hash__(self):
        return hash((MeanCVaR, self.alpha, self.weight))

    def constants(self):
        """(inv_beta, beta, w_mean, w_cvar), computed once in fp64 as the kernels expect"""
        beta = 1.0 - self.alpha
        return 1.0 / beta, beta, 1.0 - self.weight, self.weight

    def c_struct(self):
        r = _cabi.SdpRisk()
        r.inv_beta, r.beta, r.w_mean, r.w_cvar = self.constants()
        return r


def check_risk(risk, perturb_proba):
    """The SdpRisk of `risk` (None for None) after checking it and the node probabilities it
    will weigh: a MeanCVaR, finite non-negative probabilities, at most RISK_MAX_W nodes."""
    if risk is None:
        return None
    if not isinstance(risk, MeanCVaR):
        raise TypeError("risk must be None or a MeanCVaR, got %s" % type(risk).__name__)
    p = joint_proba(perturb_proba)
    W = p.size
    if W > _cabi.RISK_MAX_W:
        raise ValueError("risk: W = %d perturbation nodes, the risk kernels support at most %d"
                         % (W, _cabi.RISK_MAX_W))
    if not all(math.isfinite(x) and x >= 0.0 for x in p.tolist()):
        raise ValueError("risk: the perturbation probabilities must be finite and >= 0")
    return risk.c_struct()
